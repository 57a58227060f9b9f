// Resample -i in.nii[.gz] -o out.nii[.gz] -s sx sy sz [-n/--nearest bool] [-d/--default value]
// Puts a scan (linear interpolation, float in and out) or a mask / label image (nearest neighbour,
// read as unsigned short, labels above 255 refused, written as uint8 -- the mask type the other
// tools read) on a new voxel spacing, so that ROIs cut in voxels cover the same tissue volume on
// every scanner.  Origin and orientation are kept; the output header carries the new spacing.
// Semantics: itk::ResampleImageFilter with an identity transform (ife_cuda_resample,
// include/ife_cuda.h; DESIGN.md "Resampling").  The flags follow this project's tools and are not
// those of the reference's tools/Resample.cxx.
#include <cmath>
#include <cstdlib>
#include <iostream>
#include <string>
#include <vector>

#include "ife/Context.h"
#include "ife/IO/NiftiIO.h"
#include "ife/Util/CmdLine.h"

const std::string VERSION("0.1");

template <typename T>
void ResampleAndWrite(const std::string& path, const void* in, const ife::Geometry& g, const ife::Geometry& og,
                      int interp, double defaultValue) {
  ife::Image<T> out;
  out.SetGeometry(og);
  out.Allocate();
  int outDims[3];
  ife::CudaContext& c = ife::CudaContext::Instance();
  c.Check(ife_cuda_resample(c.Handle(), in, out.GetBufferPointer(), (int)sizeof(T), g.size.data(), g.spacing.data(),
                            og.spacing.data(), interp, defaultValue, outDims, IFE_MEM_HOST));
  ife::nifti::Write(path, out);
}

int main(int argc, char* argv[]) {
  ife::CmdLine cmd("Resample an image to a new voxel spacing.", VERSION);
  cmd.add("i", "input", "Path to input image.", true, "", "path");
  cmd.add("o", "output", "Path to output image.", true, "", "path");
  cmd.add("s", "spacing", "Output voxel spacing sx sy sz (physical units of the input).", true, "", "double").nargs = 3;
  cmd.add("n", "nearest", "Nearest-neighbour interpolation for masks / label images (uint8 output).", false, "0", "boolean");
  cmd.add("d", "default", "Value of output voxels outside the input.", false, "0", "double");
  int rc;
  if (!cmd.parse(argc, argv, &rc)) return rc;
  const std::string inPath(cmd.value("input")), outPath(cmd.value("output"));
  double spacing[3];
  for (int d = 0; d < 3; ++d) {
    const std::string& s = cmd.values("spacing")[d];
    if (!ife::CmdLine::convert(s, &spacing[d]) || !(spacing[d] > 0.0) || !std::isfinite(spacing[d])) {
      cmd.error("Spacing must be a positive number, not '" + s + "'", "-s", &rc);
      return rc;
    }
  }
  bool nearest = false;
  if (!ife::CmdLine::to_bool(cmd.value("nearest"), &nearest)) {
    cmd.error("Couldn't read argument value from string '" + cmd.value("nearest") + "'", "-n", &rc);
    return rc;
  }
  double defaultValue = 0.0;
  if (!ife::CmdLine::convert(cmd.value("default"), &defaultValue) ||
      (nearest && !(defaultValue >= 0.0 && defaultValue <= 255.0 && defaultValue == std::floor(defaultValue)))) {
    cmd.error("Default value must be a number (in nearest mode an integer in [0, 255]), not '" + cmd.value("default") + "'",
              "-d", &rc);
    return rc;
  }

  try {
    ife::Geometry g;
    std::vector<unsigned char> labels;
    ife::Image<float>::Pointer image;
    const void* in;
    if (nearest) {
      auto mask16 = ife::nifti::Read<unsigned short>(inPath);
      g = mask16->GetGeometry();
      labels.resize(g.voxels());
      const unsigned short* p = mask16->GetBufferPointer();
      for (size_t i = 0; i < labels.size(); ++i) {
        if (p[i] > 255) throw std::runtime_error("label " + std::to_string(p[i]) + " does not fit the uint8 output of nearest mode");
        labels[i] = (unsigned char)p[i];
      }
      in = labels.data();
    } else {
      image = ife::nifti::Read<float>(inPath);
      g = image->GetGeometry();
      in = image->GetBufferPointer();
    }
    const int elemBytes = nearest ? 1 : 4;
    const int interp = nearest ? IFE_INTERP_NEAREST : IFE_INTERP_LINEAR;
    int outDims[3];   // the size query needs no device
    const int rcq = ife_cuda_resample(nullptr, in, nullptr, elemBytes, g.size.data(), g.spacing.data(), spacing, interp,
                                      defaultValue, outDims, IFE_MEM_HOST);
    if (rcq != IFE_OK) throw ife::ExceptionObject(rcq, "cannot resample this image to the requested spacing");
    ife::Geometry og = g;   // origin and the source header (orientation) stay
    og.size = {{outDims[0], outDims[1], outDims[2]}};
    og.spacing = {{spacing[0], spacing[1], spacing[2]}};
    std::cout << "Resampling " << g.size[0] << "x" << g.size[1] << "x" << g.size[2] << " -> " << outDims[0] << "x"
              << outDims[1] << "x" << outDims[2] << (nearest ? " (nearest)" : " (linear)") << std::endl;
    if (nearest) ResampleAndWrite<unsigned char>(outPath, in, g, og, interp, defaultValue);
    else ResampleAndWrite<float>(outPath, in, g, og, interp, defaultValue);
  } catch (std::exception& e) {
    std::cerr << "Failed to process." << std::endl
              << "Input: " << inPath << std::endl
              << "Output: " << outPath << std::endl
              << "ExceptionObject: " << e.what() << std::endl;
    return EXIT_FAILURE;
  }
  return EXIT_SUCCESS;
}
