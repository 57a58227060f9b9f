// Resampling onto a new voxel spacing: itk::ResampleImageFilter with an identity transform, the
// output origin equal to the input's, and LinearInterpolateImageFunction (float) or
// NearestNeighborInterpolateImageFunction (float or uint8).  ife_cuda_resample in ife_cuda.cu
// validates the arguments and sizes the output; the semantics are restated once, with every
// constant named, in DESIGN.md ("Resampling") and in the CPU reference tests/resample_ref.py.
//
// Output-stationary: a thread owns four x-adjacent output voxels of one row.  The continuous
// index of every axis is computed in double with explicitly rounded operations, so the result
// is the reference's bit for bit:
//   c = (i * s'_d) * (1 / s_d)        (1 / s_d comes from the host; c = i when s'_d == s_d)
//   inside  <=>  -0.5 <= c < n_d - 0.5 on every axis, else the default value
//   linear : b = max(floor(c), 0), w = c - b (0 when not positive), upper = min(b + 1, n_d - 1);
//            nested lerps a + (b - a) * w along x (4), y (2), z (1), rounded to float once
//   nearest: min(floor(c + 0.5), n_d - 1)
// PRECONDITION (linear): the input is finite.  a + (b - a) * 0 == a is what makes the lerp
// equal to ITK's early-return branches for w == 0; an Inf or NaN neighbour with weight 0 turns it
// into NaN.
// The eight (four for nearest) neighbours are gathered through L1; an input plane is reused by
// every output plane that falls between it and the next, so upsampling in z reads it from L2.
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

namespace ife {

enum { RS_LINEAR = 0, RS_NEAREST_F32 = 1, RS_NEAREST_U8 = 2 };

constexpr int kRsBX = 32, kRsBY = 8, kRsV = 4;   // block 32x8 threads, four x-voxels per thread
// four resident blocks: up to 64 registers, which the linear kernel needs to keep the 32 gathers of a
// thread in flight without spilling (left to itself ptxas stops at 40 and spills)
constexpr int kRsMinBlocks = 4;

struct ResampleArgs {
  const void* in;
  void* out;
  int n[3];          // input nx, ny, nz
  int m[3];          // output nx, ny, nz
  double so[3];      // output spacing
  double inv[3];     // 1 / input spacing
  int ident[3];      // output spacing == input spacing: c = i exactly
  float def_f32;
  uint8_t def_u8;
};

struct RsAxis {
  int b0, b1;   // lower / upper neighbour (nearest: b0 only)
  double w;     // weight of b1 (linear)
  bool inside;
};

template <bool NEAREST>
__device__ __forceinline__ RsAxis rs_axis(int i, double so, double inv, int ident, int n) {
  const double c = ident ? (double)i : __dmul_rn(__dmul_rn((double)i, so), inv);
  RsAxis a;
  a.inside = c >= -0.5 && c < (double)n - 0.5;
  if (NEAREST) {
    a.b0 = min(max((int)floor(__dadd_rn(c, 0.5)), 0), n - 1);
    a.b1 = a.b0;
    a.w = 0.0;
  } else {
    a.b0 = min(max((int)floor(c), 0), n - 1);
    const double t = __dsub_rn(c, (double)a.b0);
    a.w = t > 0.0 ? t : 0.0;
    a.b1 = min(a.b0 + 1, n - 1);
  }
  return a;
}

__device__ __forceinline__ double rs_lerp(double a, double b, double w) {
  return __dadd_rn(a, __dmul_rn(__dsub_rn(b, a), w));
}

// VEC: the output row length is a multiple of 4 and the output 16-byte (uint8: 4-byte) aligned, so
// every thread's four voxels go out in one store; otherwise each voxel below m[0] is stored alone.
template <int MODE, bool VEC>
__global__ void __launch_bounds__(kRsBX * kRsBY, kRsMinBlocks)
resample_kernel(const ResampleArgs A) {
  typedef typename std::conditional<MODE == RS_NEAREST_U8, uint8_t, float>::type T;
  constexpr bool NEAREST = MODE != RS_LINEAR;
  const int x0 = (blockIdx.x * kRsBX + threadIdx.x) * kRsV;
  const int y = blockIdx.y * kRsBY + threadIdx.y;
  const int z = blockIdx.z;
  if (x0 >= A.m[0] || y >= A.m[1]) return;
  const RsAxis az = rs_axis<NEAREST>(z, A.so[2], A.inv[2], A.ident[2], A.n[2]);
  const RsAxis ay = rs_axis<NEAREST>(y, A.so[1], A.inv[1], A.ident[1], A.n[1]);
  const T* __restrict__ in = static_cast<const T*>(A.in);
  const size_t nx = (size_t)A.n[0], nxy = nx * (size_t)A.n[1];
  // rows (y0,z0), (y1,z0), (y0,z1), (y1,z1)
  const T* r00 = in + (size_t)az.b0 * nxy + (size_t)ay.b0 * nx;
  const T* r10 = in + (size_t)az.b0 * nxy + (size_t)ay.b1 * nx;
  const T* r01 = in + (size_t)az.b1 * nxy + (size_t)ay.b0 * nx;
  const T* r11 = in + (size_t)az.b1 * nxy + (size_t)ay.b1 * nx;
  const bool row_inside = az.inside && ay.inside;
  const T def = MODE == RS_NEAREST_U8 ? (T)A.def_u8 : (T)A.def_f32;
  T v[kRsV];
#pragma unroll
  for (int k = 0; k < kRsV; ++k) {
    const int x = x0 + k;
    const RsAxis ax = rs_axis<NEAREST>(x, A.so[0], A.inv[0], A.ident[0], A.n[0]);
    if (!(row_inside && ax.inside) || x >= A.m[0]) {
      v[k] = def;
    } else if constexpr (NEAREST) {
      v[k] = __ldg(r00 + ax.b0);
    } else {
      const double c00 = rs_lerp((double)__ldg(r00 + ax.b0), (double)__ldg(r00 + ax.b1), ax.w);
      const double c10 = rs_lerp((double)__ldg(r10 + ax.b0), (double)__ldg(r10 + ax.b1), ax.w);
      const double c01 = rs_lerp((double)__ldg(r01 + ax.b0), (double)__ldg(r01 + ax.b1), ax.w);
      const double c11 = rs_lerp((double)__ldg(r11 + ax.b0), (double)__ldg(r11 + ax.b1), ax.w);
      const double cy0 = rs_lerp(c00, c10, ay.w);
      const double cy1 = rs_lerp(c01, c11, ay.w);
      v[k] = (T)(float)rs_lerp(cy0, cy1, az.w);
    }
  }
  T* out = static_cast<T*>(A.out) + ((size_t)z * A.m[1] + y) * (size_t)A.m[0] + x0;
  if constexpr (VEC) {
    if constexpr (MODE == RS_NEAREST_U8)
      *reinterpret_cast<uchar4*>(out) = make_uchar4(v[0], v[1], v[2], v[3]);
    else
      *reinterpret_cast<float4*>(out) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int k = 0; k < kRsV; ++k)
      if (x0 + k < A.m[0]) out[k] = v[k];
  }
}

}  // namespace ife
