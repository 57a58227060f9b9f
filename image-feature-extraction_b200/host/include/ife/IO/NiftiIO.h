// NIfTI-1 single-file (.nii / .nii.gz) reader and writer: what the tools read and write
// through itk::ImageFileReader / ImageFileWriter in the reference (OUT_FILE_TYPE ".nii.gz",
// tools/ExtractFeatures.cxx:15).  Voxel data are cast to the requested pixel type on read
// (scl_slope / scl_inter applied as ITK's NIfTI IO does); spacing comes from pixdim.  The
// source header travels with the image so that outputs keep the input's orientation.
#ifndef IFE_B200_NIFTI_IO_H
#define IFE_B200_NIFTI_IO_H
#include <zlib.h>

#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <future>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "ife/Image.h"

namespace ife {
namespace nifti {

enum { DT_UINT8 = 2, DT_INT16 = 4, DT_INT32 = 8, DT_FLOAT32 = 16, DT_FLOAT64 = 64, DT_INT8 = 256,
       DT_UINT16 = 512, DT_UINT32 = 768 };

inline void swap_bytes(void* p, size_t size, size_t count) {
  unsigned char* b = static_cast<unsigned char*>(p);
  for (size_t i = 0; i < count; ++i, b += size)
    for (size_t j = 0; j < size / 2; ++j) std::swap(b[j], b[size - 1 - j]);
}

template <typename T> T rd(const std::vector<unsigned char>& h, size_t off, bool swapped) {
  T v;
  std::memcpy(&v, h.data() + off, sizeof(T));
  if (swapped) swap_bytes(&v, sizeof(T), 1);
  return v;
}
template <typename T> void wr(std::vector<unsigned char>& h, size_t off, T v) { std::memcpy(h.data() + off, &v, sizeof(T)); }

inline bool ends_with(const std::string& s, const std::string& e) {
  return s.size() >= e.size() && s.compare(s.size() - e.size(), e.size(), e) == 0;
}

// IFE_IO_THREADS in the environment sets the thread count of the reader's conversion and of the
// .nii.gz writer (default: the hardware's, at most 32).
inline int io_threads(size_t pieces) {
  int t = (int)std::thread::hardware_concurrency();
  if (const char* e = std::getenv("IFE_IO_THREADS")) t = std::atoi(e);
  t = std::max(1, std::min(t, 32));
  return (int)std::min<size_t>((size_t)t, std::max<size_t>(pieces, 1));
}


template <typename TOut, typename TIn>
void convert_range(const unsigned char* raw, bool swapped, bool scale, double slope, double inter, TOut* out, size_t a, size_t b) {
  for (size_t i = a; i < b; ++i) {
    TIn v;
    std::memcpy(&v, raw + i * sizeof(TIn), sizeof(TIn));
    if (swapped) swap_bytes(&v, sizeof(TIn), 1);
    out[i] = scale ? static_cast<TOut>((double)v * slope + inter) : static_cast<TOut>(v);
  }
}

// raw voxels -> pixel type, on all cores (a 512x512x400 scan is 105 M voxels)
template <typename TOut, typename TIn>
void convert(const unsigned char* raw, bool swapped, double slope, double inter, TOut* out, size_t n) {
  const bool scale = slope != 0.0 && !(slope == 1.0 && inter == 0.0);
  const int n_threads = io_threads(n >> 22);
  if (n_threads <= 1) { convert_range<TOut, TIn>(raw, swapped, scale, slope, inter, out, 0, n); return; }
  std::vector<std::thread> pool;
  const size_t per = (n + n_threads - 1) / n_threads;
  for (int t = 0; t < n_threads; ++t)
    pool.emplace_back([=] { convert_range<TOut, TIn>(raw, swapped, scale, slope, inter, out, std::min(n, t * per), std::min(n, (t + 1) * per)); });
  for (auto& t : pool) t.join();
}

// seconds spent inside Read() / Write() so far in this process (the tools print them under IFE_TIMING)
inline double& read_seconds() { static double s = 0.0; return s; }
inline double& write_seconds() { static double s = 0.0; return s; }
struct ScopedSeconds {
  double& acc;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  explicit ScopedSeconds(double& a) : acc(a) {}
  ~ScopedSeconds() {
    static std::mutex mu;   // files are read concurrently (ReadPair)
    std::lock_guard<std::mutex> lk(mu);
    acc += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  }
};

template <typename T>
typename Image<T>::Pointer Read(const std::string& path) {
  ScopedSeconds clock(read_seconds());
  gzFile f = gzopen(path.c_str(), "rb");
  if (!f) throw std::runtime_error("cannot open '" + path + "'");
  std::vector<unsigned char> hdr(352, 0);
  if (gzread(f, hdr.data(), 348) != 348) { gzclose(f); throw std::runtime_error("'" + path + "': short NIfTI header"); }
  int sizeof_hdr;
  std::memcpy(&sizeof_hdr, hdr.data(), 4);
  bool swapped = false;
  if (sizeof_hdr != 348) {
    swap_bytes(&sizeof_hdr, 4, 1);
    if (sizeof_hdr != 348) { gzclose(f); throw std::runtime_error("'" + path + "' is not a NIfTI-1 file"); }
    swapped = true;
  }
  if (std::memcmp(hdr.data() + 344, "n+1", 3) != 0) { gzclose(f); throw std::runtime_error("'" + path + "': only single-file NIfTI-1 (n+1) is supported"); }
  const int ndim = rd<int16_t>(hdr, 40, swapped);
  int dims[3] = {1, 1, 1};
  for (int d = 0; d < 3 && d < ndim; ++d) dims[d] = rd<int16_t>(hdr, 42 + 2 * d, swapped);
  for (int d = 3; d < ndim && d < 7; ++d)
    if (rd<int16_t>(hdr, 42 + 2 * d, swapped) > 1) { gzclose(f); throw std::runtime_error("'" + path + "': more than 3 dimensions"); }
  const int datatype = rd<int16_t>(hdr, 70, swapped);
  const float vox_offset = rd<float>(hdr, 108, swapped);
  const double slope = rd<float>(hdr, 112, swapped), inter = rd<float>(hdr, 116, swapped);
  auto img = Image<T>::New();
  Geometry g;
  g.size = {{dims[0], dims[1], dims[2]}};
  for (int d = 0; d < 3; ++d) {
    const double p = std::fabs((double)rd<float>(hdr, 76 + 4 * (d + 1), swapped));
    g.spacing[d] = p > 0 ? p : 1.0;
  }
  g.origin = {{(double)rd<float>(hdr, 268, swapped), (double)rd<float>(hdr, 272, swapped), (double)rd<float>(hdr, 276, swapped)}};
  if (!swapped) g.nifti_header.assign(hdr.begin(), hdr.begin() + 348);
  img->SetGeometry(g);
  img->Allocate();
  size_t bpv;
  switch (datatype) {
    case DT_UINT8: case DT_INT8: bpv = 1; break;
    case DT_INT16: case DT_UINT16: bpv = 2; break;
    case DT_INT32: case DT_UINT32: case DT_FLOAT32: bpv = 4; break;
    case DT_FLOAT64: bpv = 8; break;
    default: gzclose(f); throw std::runtime_error("'" + path + "': unsupported NIfTI datatype " + std::to_string(datatype));
  }
  const long skip = (long)(vox_offset > 348 ? vox_offset : 352) - 348;
  std::vector<unsigned char> junk(skip > 0 ? skip : 1);
  if (skip > 0 && gzread(f, junk.data(), (unsigned)skip) != skip) { gzclose(f); throw std::runtime_error("'" + path + "': truncated"); }
  const size_t n = g.voxels();
  const size_t raw_bytes = n * bpv;
  std::unique_ptr<unsigned char[]> raw_store(new unsigned char[raw_bytes ? raw_bytes : 1]);   // not zero-filled
  const unsigned char* raw = raw_store.get();
  size_t got = 0;
  while (got < raw_bytes) {
    const unsigned want = (unsigned)std::min<size_t>(raw_bytes - got, 1u << 30);
    const int r = gzread(f, raw_store.get() + got, want);
    if (r <= 0) break;
    got += (size_t)r;
  }
  gzclose(f);
  if (got != raw_bytes) throw std::runtime_error("'" + path + "': truncated voxel data");
  T* out = img->GetBufferPointer();
  switch (datatype) {
    case DT_UINT8: convert<T, uint8_t>(raw, swapped, slope, inter, out, n); break;
    case DT_INT8: convert<T, int8_t>(raw, swapped, slope, inter, out, n); break;
    case DT_INT16: convert<T, int16_t>(raw, swapped, slope, inter, out, n); break;
    case DT_UINT16: convert<T, uint16_t>(raw, swapped, slope, inter, out, n); break;
    case DT_INT32: convert<T, int32_t>(raw, swapped, slope, inter, out, n); break;
    case DT_UINT32: convert<T, uint32_t>(raw, swapped, slope, inter, out, n); break;
    case DT_FLOAT32: convert<T, float>(raw, swapped, slope, inter, out, n); break;
    case DT_FLOAT64: convert<T, double>(raw, swapped, slope, inter, out, n); break;
  }
  return img;
}

// Two files at once (a scan and its mask): inflating a .nii.gz is one serial zlib stream per file, so
// the second file is read on its own thread.  An error in the first file is the one reported.
template <typename T1, typename T2>
std::pair<typename Image<T1>::Pointer, typename Image<T2>::Pointer> ReadPair(const std::string& path1, const std::string& path2) {
  auto second = std::async(std::launch::async, [&path2]() { return Read<T2>(path2); });
  typename Image<T1>::Pointer first = Read<T1>(path1);   // throws: `second`'s destructor waits for the thread
  return std::make_pair(first, second.get());
}

// One gzip member written by several threads (the way pigz does it): the payload is cut into
// 8 MB pieces, every piece is deflated on its own as a raw stream that ends on a byte boundary
// (Z_FULL_FLUSH; the last one with Z_FINISH), the pieces are written in order behind one gzip
// header, and the CRC-32 of the whole is combined from the pieces'.  Any gzip reader sees an
// ordinary .gz file.  The 32 feature volumes of one ExtractFeatures run are 13 GB of floats:
// with one zlib stream the tool spent 75 s writing them and 0.4 s computing them.
inline void gz_write_parallel(const std::string& path, const unsigned char* head, size_t head_bytes,
                              const unsigned char* data, size_t bytes) {
  const size_t kPiece = (size_t)8 << 20;
  // piece 0 carries the NIfTI header in front of its share of the data
  const size_t n_pieces = std::max<size_t>((bytes + kPiece - 1) / kPiece, 1);
  const int n_threads = io_threads(n_pieces);
  struct Piece { std::vector<unsigned char> z; uLong crc = 0; size_t raw = 0; bool ready = false; bool failed = false; };
  std::vector<Piece> pieces(n_pieces);
  std::mutex mu;
  std::condition_variable cv;
  std::atomic<size_t> next(0);
  size_t written = 0;   // pieces already on disk (guarded by mu): bounds the compressed data held in memory
  bool abort_all = false;

  auto work = [&]() {
    for (;;) {
      const size_t i = next.fetch_add(1);
      if (i >= n_pieces) return;
      {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return abort_all || i < written + 2 * (size_t)n_threads; });
        if (abort_all) return;
      }
      const size_t off = i * kPiece, len = std::min(kPiece, bytes - std::min(bytes, off));
      const bool last = i + 1 == n_pieces;
      Piece& P = pieces[i];
      z_stream zs;
      std::memset(&zs, 0, sizeof(zs));
      bool ok = deflateInit2(&zs, 1, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) == Z_OK;
      if (ok) {
        const size_t head_here = i == 0 ? head_bytes : 0;
        P.z.resize(deflateBound(&zs, (uLong)(len + head_here)) + 64);
        zs.next_out = P.z.data();
        zs.avail_out = (uInt)P.z.size();
        uLong crc = crc32(0L, Z_NULL, 0);
        if (head_here) {
          crc = crc32(crc, head, (uInt)head_here);
          zs.next_in = const_cast<unsigned char*>(head);
          zs.avail_in = (uInt)head_here;
          ok = deflate(&zs, Z_NO_FLUSH) == Z_OK && zs.avail_in == 0;
        }
        if (ok) {
          crc = crc32(crc, data + off, (uInt)len);
          zs.next_in = const_cast<unsigned char*>(data + off);
          zs.avail_in = (uInt)len;
          const int r = deflate(&zs, last ? Z_FINISH : Z_FULL_FLUSH);
          ok = (last ? r == Z_STREAM_END : r == Z_OK) && zs.avail_in == 0 && zs.avail_out > 0;
        }
        P.z.resize(ok ? (size_t)zs.total_out : 0);
        P.crc = crc;
        P.raw = len + head_here;
        deflateEnd(&zs);   // Z_DATA_ERROR for the unfinished pieces is expected
      }
      std::lock_guard<std::mutex> lk(mu);
      P.failed = !ok;
      P.ready = true;
      cv.notify_all();
    }
  };

  FILE* f = std::fopen(path.c_str(), "wb");
  if (!f) throw std::runtime_error("cannot write '" + path + "'");
  std::vector<std::thread> pool;
  for (int t = 0; t < n_threads; ++t) pool.emplace_back(work);
  static const unsigned char gz_head[10] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 4, 3};   // deflate, no name, no time, fastest, unix
  bool ok = std::fwrite(gz_head, 1, 10, f) == 10;
  uLong crc = crc32(0L, Z_NULL, 0);
  size_t total = 0;
  for (size_t i = 0; i < n_pieces; ++i) {
    Piece* P = &pieces[i];
    {
      std::unique_lock<std::mutex> lk(mu);
      cv.wait(lk, [&] { return P->ready; });
    }
    ok = ok && !P->failed && std::fwrite(P->z.data(), 1, P->z.size(), f) == P->z.size();
    crc = crc32_combine(crc, P->crc, (z_off_t)P->raw);
    total += P->raw;
    std::vector<unsigned char>().swap(P->z);
    std::lock_guard<std::mutex> lk(mu);
    written = i + 1;
    if (!ok) abort_all = true;
    cv.notify_all();
    if (!ok) break;
  }
  for (auto& t : pool) t.join();
  unsigned char tail[8];
  for (int b = 0; b < 4; ++b) {
    tail[b] = (unsigned char)((crc >> (8 * b)) & 0xff);
    tail[4 + b] = (unsigned char)(((uint64_t)total >> (8 * b)) & 0xff);
  }
  ok = ok && std::fwrite(tail, 1, 8, f) == 8;
  ok = (std::fclose(f) == 0) && ok;
  if (!ok) {
    std::remove(path.c_str());
    throw std::runtime_error("error writing '" + path + "'");
  }
}

template <typename T> struct DataType;
template <> struct DataType<float> { static const int16_t code = DT_FLOAT32; };
template <> struct DataType<unsigned char> { static const int16_t code = DT_UINT8; };
template <> struct DataType<short> { static const int16_t code = DT_INT16; };
template <> struct DataType<unsigned short> { static const int16_t code = DT_UINT16; };

template <typename T>
void Write(const std::string& path, const Geometry& g, const T* data) {
  ScopedSeconds clock(write_seconds());
  std::vector<unsigned char> hdr(352, 0);
  if (g.nifti_header.size() == 348) {
    std::copy(g.nifti_header.begin(), g.nifti_header.end(), hdr.begin());
    // a spacing that differs from the one Read() took from the header (resampling) replaces pixdim
    // and scales the sform's column of that axis; the qform takes its scale from pixdim itself
    for (int d = 0; d < 3; ++d) {
      const double p = std::fabs((double)rd<float>(hdr, 76 + 4 * (d + 1), false));
      const double was = p > 0 ? p : 1.0;
      if (g.spacing[d] == was) continue;
      wr<float>(hdr, 76 + 4 * (d + 1), (float)g.spacing[d]);
      for (int r = 0; r < 3; ++r) {
        const size_t off = 280 + 16 * r + 4 * d;   // srow_x / srow_y / srow_z, column d
        wr<float>(hdr, off, (float)(rd<float>(hdr, off, false) * (g.spacing[d] / was)));
      }
    }
  }
  wr<int32_t>(hdr, 0, 348);
  int16_t dim[8] = {3, (int16_t)g.size[0], (int16_t)g.size[1], (int16_t)g.size[2], 1, 1, 1, 1};
  std::memcpy(hdr.data() + 40, dim, sizeof(dim));
  wr<int16_t>(hdr, 70, DataType<T>::code);
  wr<int16_t>(hdr, 72, (int16_t)(8 * sizeof(T)));
  if (g.nifti_header.size() != 348) {
    float pixdim[8] = {1, (float)g.spacing[0], (float)g.spacing[1], (float)g.spacing[2], 0, 0, 0, 0};
    std::memcpy(hdr.data() + 76, pixdim, sizeof(pixdim));
    wr<int16_t>(hdr, 254, 1);  // sform_code: scanner coordinates, axis-aligned
    float sx[4] = {(float)g.spacing[0], 0, 0, (float)g.origin[0]};
    float sy[4] = {0, (float)g.spacing[1], 0, (float)g.origin[1]};
    float sz[4] = {0, 0, (float)g.spacing[2], (float)g.origin[2]};
    std::memcpy(hdr.data() + 280, sx, 16);
    std::memcpy(hdr.data() + 296, sy, 16);
    std::memcpy(hdr.data() + 312, sz, 16);
    hdr[123] = 2;  // xyzt_units: millimetres
  }
  wr<float>(hdr, 108, 352.0f);
  wr<float>(hdr, 112, 1.0f);   // scl_slope
  wr<float>(hdr, 116, 0.0f);   // scl_inter
  std::memcpy(hdr.data() + 344, "n+1", 4);
  const size_t bytes = g.voxels() * sizeof(T);
  if (ends_with(path, ".gz")) {
    gz_write_parallel(path, hdr.data(), 352, reinterpret_cast<const unsigned char*>(data), bytes);
  } else {
    FILE* f = std::fopen(path.c_str(), "wb");
    if (!f) throw std::runtime_error("cannot write '" + path + "'");
    bool ok = std::fwrite(hdr.data(), 1, 352, f) == 352 && std::fwrite(data, 1, bytes, f) == bytes;
    ok = (std::fclose(f) == 0) && ok;
    if (!ok) throw std::runtime_error("error writing '" + path + "'");
  }
}

template <typename T>
void Write(const std::string& path, const Image<T>& img) { Write(path, img.GetGeometry(), img.GetBufferPointer()); }

}  // namespace nifti
}  // namespace ife
#endif
