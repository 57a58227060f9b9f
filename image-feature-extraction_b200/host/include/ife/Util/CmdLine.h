// Small command-line parser with the surface of the TCLAP subset the reference tools use
// (ValueArg / MultiArg with a short flag, a long name, a required bit and a default):
// `-i path`, `--image path`, `--image=path`, repeated flags for MultiArg, `-h/--help`,
// `--version`.  Parse errors print "PARSE ERROR" with the offending argument and make the
// tool exit with EXIT_FAILURE, as TCLAP's default handler does.  An argument with nargs > 1
// takes that many values after its flag (`-s 0.7 0.7 2.5`).
#ifndef IFE_B200_CMDLINE_H
#define IFE_B200_CMDLINE_H
#include <cstdlib>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

namespace ife {

class CmdLine {
public:
  struct Arg {
    std::string flag, name, desc, type;
    bool required, multi;
    std::vector<std::string> values;
    bool set = false;
    int nargs = 1;
  };
  CmdLine(const std::string& message, const std::string& version) : m_Message(message), m_Version(version) {}

  Arg& add(const std::string& flag, const std::string& name, const std::string& desc, bool required,
           const std::string& def, const std::string& type, bool multi = false) {
    m_Args.push_back(Arg{flag, name, desc, type, required, multi, {}, false});
    if (!multi && !required) m_Args.back().values.push_back(def);
    return m_Args.back();
  }
  const Arg& get(const std::string& name) const {
    for (const Arg& a : m_Args) if (a.name == name) return a;
    throw std::logic_error("unknown argument " + name);
  }
  std::string value(const std::string& name) const { return get(name).values.empty() ? std::string() : get(name).values.back(); }
  const std::vector<std::string>& values(const std::string& name) const { return get(name).values; }

  // returns false (after printing) when the program should exit; *exit_code says how
  bool parse(int argc, char** argv, int* exit_code) {
    m_Prog = argc > 0 ? argv[0] : "tool";
    for (int i = 1; i < argc; ++i) {
      std::string tok = argv[i], val;
      bool has_val = false;
      if (tok == "-h" || tok == "--help") { usage(std::cout); *exit_code = EXIT_SUCCESS; return false; }
      if (tok == "--version") { std::cout << m_Prog << "  version: " << m_Version << std::endl; *exit_code = EXIT_SUCCESS; return false; }
      Arg* arg = nullptr;
      if (tok.rfind("--", 0) == 0) {
        const size_t eq = tok.find('=');
        const std::string name = tok.substr(2, eq == std::string::npos ? std::string::npos : eq - 2);
        if (eq != std::string::npos) { val = tok.substr(eq + 1); has_val = true; }
        for (Arg& a : m_Args) if (a.name == name) arg = &a;
      } else if (tok.size() >= 2 && tok[0] == '-') {
        for (Arg& a : m_Args) if (a.flag == tok.substr(1, 1)) arg = &a;
        if (arg && tok.size() > 2) { val = tok.substr(2); has_val = true; }
      }
      if (!arg) return error("Couldn't find match for argument", tok, exit_code);
      if (!has_val) {
        if (i + 1 >= argc) return error("Missing a value for this argument!", tok, exit_code);
        val = argv[++i];
      }
      if (arg->set && !arg->multi) return error("Argument already set!", tok, exit_code);
      if (!arg->multi) arg->values.clear();
      arg->values.push_back(val);
      for (int k = 1; k < arg->nargs; ++k) {
        if (i + 1 >= argc) return error("This argument takes " + std::to_string(arg->nargs) + " values!", tok, exit_code);
        arg->values.push_back(argv[++i]);
      }
      arg->set = true;
    }
    for (const Arg& a : m_Args)
      if (a.required && !a.set) return error("Required argument missing: " + a.name, "", exit_code);
    return true;
  }

  template <typename T>
  static bool convert(const std::string& s, T* out) {
    std::istringstream is(s);
    is >> *out;
    return !is.fail() && is.eof();
  }
  static bool to_bool(const std::string& s, bool* out) {
    if (s == "1" || s == "true" || s == "True" || s == "TRUE") { *out = true; return true; }
    if (s == "0" || s == "false" || s == "False" || s == "FALSE") { *out = false; return true; }
    return false;
  }
  bool error(const std::string& what, const std::string& arg, int* exit_code) const {
    std::cerr << "PARSE ERROR:";
    if (!arg.empty()) std::cerr << " Argument: " << arg;
    std::cerr << std::endl << "             " << what << std::endl << std::endl;
    usage(std::cerr);
    *exit_code = EXIT_FAILURE;
    return false;
  }
  void usage(std::ostream& os) const {
    os << "USAGE:" << std::endl << "   " << m_Prog;
    for (const Arg& a : m_Args) {
      std::string one = "-" + a.flag;
      for (int k = 0; k < a.nargs; ++k) one += " <" + a.type + ">";
      os << " " << (a.required ? one : "[" + one + "]") << (a.multi ? " ..." : "");
    }
    os << " [--version] [-h]" << std::endl << std::endl << "Where:" << std::endl;
    for (const Arg& a : m_Args)
      os << "   -" << a.flag << " <" << a.type << ">,  --" << a.name << " <" << a.type << ">"
         << (a.multi ? "  (accepted multiple times)" : "") << std::endl
         << "     " << (a.required ? "(required)  " : "") << a.desc << std::endl;
    os << std::endl << "   " << m_Message << std::endl;
  }

private:
  std::string m_Message, m_Version, m_Prog;
  std::vector<Arg> m_Args;
};

}  // namespace ife
#endif
