// Signed Euclidean distance map of a uint8 mask: itk::SignedMaurerDistanceMapImageFilter as recalled,
// and the probability-weighted mean of that map (the expected distance).  ife_cuda_signed_distance_map
// and ife_cuda_expected_signed_distance in ife_cuda.cu validate the arguments; the semantics are
// stated once in include/ife_cuda.h and DESIGN.md ("Signed distance maps"), and restated on the CPU in
// tests/distance_ref.py.
//
// An exact separable transform in three line passes:
//   x pass  one warp per row: the contour flag (sdm_is_contour) from the 3x3 neighbour rows, then the
//           distance |dx| to the nearest contour voxel of the row by a forward max-scan and a backward
//           min-scan of contour positions.  Out: int16 |dx| per voxel, kSdmNone when the row has none.
//   y pass  one thread per (x, z) line, x-adjacent lines in one warp (every load and store coalesced):
//           the lower envelope of the parabolas f(q) + sy^2 (y - q)^2 over the line's sites
//           (Felzenszwalb-Huttenlocher), then one sweep that reads each voxel's winning site off the
//           envelope.  Out: the winner's offsets (|dx|, |dy|) as 2 x int16 per voxel.
//   z pass  the same along z over the (x, y) lines; the winner's D is recomputed from its integer
//           offsets in the fixed operation order below, signed with the mask, and written as float
//           (or, for the expected distance, weighted and summed without writing the map).
// The envelope's site stack lives in global memory (workspace b0), entry k of line L at
// [k * n_lines + L], so the lanes of a warp touching the same depth touch consecutive words.
//
// D(v) = fl(fl(fl((dx sx)^2) + fl((dy sy)^2)) + fl((dz sz)^2)), each square fl(t * t) of t = fl(d * s):
// every operation one rounded double operation.  Rounding is monotone, so the minimum over the
// separable passes is the minimum over all contour voxels; with a unit spacing every value is an
// integer and the envelope's decisions are exact.
#pragma once
#include <cfloat>
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

namespace ife {

constexpr int kSdmMaxAxis = 32767;          // offsets and stack positions are int16
constexpr int16_t kSdmNone = 0x7fff;        // no contour voxel on the line (largest offset is 32766)
constexpr int kSdmRowsPerBlock = 8;         // x pass: one warp per row
constexpr int kSdmLineThreads = 256;        // y / z passes: one thread per line
constexpr int kSdmReduceThreads = 256;      // expected distance: final reduction block

// One block's (or the whole volume's) share of the expected distance.
struct SdmPartial {
  double swd;     // sum of weight * distance
  double sw;      // sum of weight
  int bad_weight; // weights that are negative or not finite
  int no_site;    // voxels with no contour voxel anywhere (the center mask has no contour)
};

struct SdmArgs {
  int nx, ny, nz;
  double s[3];               // spacing
  const uint8_t* mask;
  int16_t* gx;               // x pass out / y pass in
  uint32_t* gxy;             // y pass out / z pass in: |dx| | |dy| << 16
  void* stack;               // envelope stacks (uint32 entries in the y pass, uint64 in the z pass)
  float* out;                // the map (z pass, map mode)
  int inside_positive, squared;
  // expected distance (z pass, sum mode)
  const float* weight;
  const uint8_t* region;     // null: every voxel
  SdmPartial* partial;       // one per block of the z pass
};

// The contour rule: an object voxel with a background voxel among its 26 neighbours inside the image
// (voxels outside the image are not background).  tests/distance_ref.py `contour` is its CPU twin.
__device__ __forceinline__ bool sdm_is_contour(const uint8_t* __restrict__ m, int x, int y, int z, int nx, int ny,
                                               int nz) {
  const size_t nxy = (size_t)nx * ny;
  if (m[(size_t)z * nxy + (size_t)y * nx + x] == 0) return false;
  for (int dz = -1; dz <= 1; ++dz) {
    const int zz = z + dz;
    if (zz < 0 || zz >= nz) continue;
    for (int dy = -1; dy <= 1; ++dy) {
      const int yy = y + dy;
      if (yy < 0 || yy >= ny) continue;
      const uint8_t* row = m + (size_t)zz * nxy + (size_t)yy * nx;
      for (int dx = -1; dx <= 1; ++dx) {
        const int xx = x + dx;
        if (xx >= 0 && xx < nx && __ldg(row + xx) == 0) return true;
      }
    }
  }
  return false;
}

__device__ __forceinline__ double sdm_sq(int d, double s) {
  const double t = __dmul_rn((double)d, s);
  return __dmul_rn(t, t);
}

// x pass: one warp per (y, z) row, 32 voxels per step.
__global__ void __launch_bounds__(32 * kSdmRowsPerBlock)
sdm_pass_x(const SdmArgs A) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kSdmRowsPerBlock + (threadIdx.x >> 5);
  if (row >= (long long)A.ny * A.nz) return;   // whole warps leave together
  const int y = (int)(row % A.ny), z = (int)(row / A.ny);
  const int nx = A.nx;
  int16_t* g = A.gx + (size_t)row * nx;
  // forward: distance to the nearest contour voxel at or left of x
  int last = -1;
  for (int x0 = 0; x0 < nx; x0 += 32) {
    const int x = x0 + lane;
    const bool c = x < nx && sdm_is_contour(A.mask, x, y, z, nx, A.ny, A.nz);
    int p = c ? x : last;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int q = __shfl_up_sync(0xffffffffu, p, o);
      if (lane >= o) p = max(p, q);
    }
    if (x < nx) g[x] = p < 0 ? kSdmNone : (int16_t)(x - p);
    last = __shfl_sync(0xffffffffu, p, 31);
  }
  __syncwarp();
  // backward: nearest contour voxel at or right of x (a contour voxel is where the left distance is 0)
  int next = 0x7fffffff;
  for (int x0 = (nx - 1) / 32 * 32; x0 >= 0; x0 -= 32) {
    const int x = x0 + lane;
    const int16_t left = x < nx ? g[x] : kSdmNone;
    int p = left == 0 ? x : next;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int q = __shfl_down_sync(0xffffffffu, p, o);
      if (lane + o < 32) p = min(p, q);
    }
    if (x < nx && p != 0x7fffffff) {
      const int right = p - x;
      if (left == kSdmNone || right < left) g[x] = (int16_t)right;
    }
    next = __shfl_sync(0xffffffffu, p, 0);
  }
}

// The y and z passes share one kernel: the line geometry, the carried value and the stack entry differ.
//   Z == false: lines (x, z) along y; a site carries |dx| (int16); f = fl((dx sx)^2).
//   Z == true : lines (x, y) along z; a site carries |dx| | |dy| << 16; f = fl(fl((dx sx)^2) + fl((dy sy)^2)).
template <bool Z>
struct SdmLine {
  typedef typename std::conditional<Z, uint32_t, int16_t>::type In;
  typedef typename std::conditional<Z, unsigned long long, uint32_t>::type Entry;   // position | value << 16
  static __device__ __forceinline__ bool site(In v) { return (int16_t)(v & 0xffff) != kSdmNone; }
  static __device__ __forceinline__ double f(In v, const double* s) {
    if (Z) return __dadd_rn(sdm_sq((int)(v & 0xffff), s[0]), sdm_sq((int)(v >> 16), s[1]));
    return sdm_sq((int)v, s[0]);
  }
  static __device__ __forceinline__ Entry pack(int q, In v) { return (Entry)q | ((Entry)(Z ? (uint32_t)v : (uint16_t)v) << 16); }
  static __device__ __forceinline__ int pos(Entry e) { return (int)(e & 0xffff); }
  static __device__ __forceinline__ In val(Entry e) { return (In)(e >> 16); }
};

// Abscissa num / den (den > 0) where the parabola of site r (r > q) starts to lie below the one of
// site q.  It is compared by cross-multiplication, not divided: with a unit spacing num and den are
// integers, every product stays below 2^53 for axes of up to kSdmMaxAxis voxels, and each decision of
// the envelope is exact.
struct SdmSep {
  double num, den;
};
__device__ __forceinline__ SdmSep sdm_sep(int q, double fq, int r, double fr, double w) {
  return SdmSep{__dadd_rn(__dsub_rn(fr, fq), __dmul_rn(w, (double)(r * r - q * q))), __dmul_rn(2.0 * w, (double)(r - q))};
}
__device__ __forceinline__ bool sdm_after(const SdmSep& a, const SdmSep& b) {   // a > b
  return __dmul_rn(a.num, b.den) > __dmul_rn(b.num, a.den);
}

// SUM: the expected distance's z pass -- weight the signed distance instead of writing it.
template <bool Z, bool SUM>
__global__ void __launch_bounds__(kSdmLineThreads)
sdm_pass_line(const SdmArgs A) {
  typedef SdmLine<Z> L;
  typedef typename L::In In;
  typedef typename L::Entry Entry;
  const int nx = A.nx, n = Z ? A.nz : A.ny;
  const size_t n_lines = (size_t)nx * (Z ? A.ny : A.nz);
  const size_t line = (size_t)blockIdx.x * kSdmLineThreads + threadIdx.x;
  const bool active = line < n_lines;
  const size_t x = line % nx, o = line / nx;   // o: z (y pass) or y (z pass)
  const size_t stride = Z ? (size_t)nx * A.ny : (size_t)nx;
  const size_t start = Z ? o * nx + x : o * (size_t)nx * A.ny + x;
  const In* in = Z ? reinterpret_cast<const In*>(A.gxy) : reinterpret_cast<const In*>(A.gx);
  Entry* stack = static_cast<Entry*>(A.stack);
  const double w = Z ? __dmul_rn(A.s[2], A.s[2]) : __dmul_rn(A.s[1], A.s[1]);
  double swd = 0.0, sw = 0.0;
  int bad = 0, none = 0;
  if (active) {
    // lower envelope: stack[0..k) of sites, top (vt, ft) and the one below it (vs, fs) in registers;
    // zt is where the top's parabola starts to be the lowest
    int k = 0, vt = 0, vs = 0;
    double ft = 0.0, fs = 0.0;
    SdmSep zt{0.0, 1.0};
    for (int q = 0; q < n; ++q) {
      const In c = in[start + (size_t)q * stride];
      if (!L::site(c)) continue;
      const double fq = L::f(c, A.s);
      SdmSep sq{0.0, 1.0};
      while (k > 0) {
        sq = sdm_sep(vt, ft, q, fq, w);
        if (k == 1 || sdm_after(sq, zt)) break;
        --k;                                   // the top is nowhere the lowest: pop it
        vt = vs; ft = fs;
        if (k > 1) {
          const Entry e = stack[(size_t)(k - 2) * n_lines + line];
          vs = L::pos(e); fs = L::f(L::val(e), A.s);
          zt = sdm_sep(vs, fs, vt, ft, w);
        }
      }
      if (k > 0) { vs = vt; fs = ft; zt = sq; }
      stack[(size_t)k * n_lines + line] = L::pack(q, c);
      vt = q; ft = fq;
      ++k;
    }
    // sweep: each voxel takes the envelope's site at its position
    int j = 0, v0 = 0, v1 = 0;
    In c0 = (In)kSdmNone, c1 = 0;
    double f0 = 0.0, f1 = 0.0;
    SdmSep b{0.0, 1.0};   // where site j + 1 takes over
    if (k > 0) {
      const Entry e = stack[line];
      v0 = L::pos(e); c0 = L::val(e); f0 = L::f(c0, A.s);
    }
    if (k > 1) {
      const Entry e = stack[n_lines + line];
      v1 = L::pos(e); c1 = L::val(e); f1 = L::f(c1, A.s);
      b = sdm_sep(v0, f0, v1, f1, w);
    }
    for (int y = 0; y < n; ++y) {
      while (j + 1 < k && b.num < __dmul_rn((double)y, b.den)) {
        ++j;
        v0 = v1; c0 = c1; f0 = f1;
        if (j + 1 < k) {
          const Entry e = stack[(size_t)(j + 1) * n_lines + line];
          v1 = L::pos(e); c1 = L::val(e); f1 = L::f(c1, A.s);
          b = sdm_sep(v0, f0, v1, f1, w);
        }
      }
      const size_t i = start + (size_t)y * stride;
      const int d = abs(y - v0);
      if (!Z) {
        A.gxy[i] = k == 0 ? (uint32_t)(uint16_t)kSdmNone : (uint32_t)(uint16_t)c0 | ((uint32_t)d << 16);
        continue;
      }
      float v = FLT_MAX;
      if (k > 0) {
        const double D = __dadd_rn(f0, sdm_sq(d, A.s[2]));
        v = A.squared ? __double2float_rn(D) : __double2float_rn(__dsqrt_rn(D));
      }
      const bool obj = A.mask[i] != 0;
      if ((A.inside_positive ? !obj : obj) && v != 0.0f) v = -v;
      if (!SUM) {
        A.out[i] = v;
      } else if (!A.region || A.region[i] != 0) {
        const float wt = A.weight[i];
        if (!(wt >= 0.0f) || wt == INFINITY) ++bad;
        none += k == 0;
        swd = __dadd_rn(swd, __dmul_rn((double)wt, (double)v));
        sw = __dadd_rn(sw, (double)wt);
      }
    }
  }
  if (SUM) {
    // fixed-order block reduction: thread t's sums, then a tree over the block
    __shared__ SdmPartial red[kSdmLineThreads];
    red[threadIdx.x] = SdmPartial{swd, sw, bad, none};
    __syncthreads();
    for (int h = kSdmLineThreads / 2; h > 0; h >>= 1) {
      if ((int)threadIdx.x < h) {
        SdmPartial& a = red[threadIdx.x];
        const SdmPartial& c = red[threadIdx.x + h];
        a.swd = __dadd_rn(a.swd, c.swd);
        a.sw = __dadd_rn(a.sw, c.sw);
        a.bad_weight += c.bad_weight;
        a.no_site += c.no_site;
      }
      __syncthreads();
    }
    if (threadIdx.x == 0) A.partial[blockIdx.x] = red[0];
  }
}

// The blocks' partials in one block, in a fixed order: thread t sums partials t, t + 256, ... in turn,
// then a tree.  out[0] is the whole volume's.
__global__ void __launch_bounds__(kSdmReduceThreads)
sdm_reduce_partials(const SdmPartial* __restrict__ partial, int n, SdmPartial* out) {
  __shared__ SdmPartial red[kSdmReduceThreads];
  SdmPartial a{0.0, 0.0, 0, 0};
  for (int i = threadIdx.x; i < n; i += kSdmReduceThreads) {
    const SdmPartial c = partial[i];
    a.swd = __dadd_rn(a.swd, c.swd);
    a.sw = __dadd_rn(a.sw, c.sw);
    a.bad_weight += c.bad_weight;
    a.no_site += c.no_site;
  }
  red[threadIdx.x] = a;
  __syncthreads();
  for (int h = kSdmReduceThreads / 2; h > 0; h >>= 1) {
    if ((int)threadIdx.x < h) {
      SdmPartial& p = red[threadIdx.x];
      const SdmPartial& c = red[threadIdx.x + h];
      p.swd = __dadd_rn(p.swd, c.swd);
      p.sw = __dadd_rn(p.sw, c.sw);
      p.bad_weight += c.bad_weight;
      p.no_site += c.no_site;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0];
}

}  // namespace ife
