// libife_cuda.so -- host side of the C ABI declared in include/ife_cuda.h: context,
// device workspace, coefficient set-up and kernel orchestration.  No CPU fallback: every
// entry point fails with IFE_E_CUDA when no device is usable.
#include "ife_cuda.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <sys/mman.h>

#include <cuda_runtime.h>

#include "distance_map.cuh"
#include "eigen_features.cuh"
#include "features_march.cuh"
#include "features_march4.cuh"
#include "recursive_gaussian.cuh"
#include "iir_tma.cuh"
#include "radix_sort.cuh"
#include "resample.cuh"
#include "support_box.cuh"
#include "ife_ctx.h"

namespace ife {

int fail(ife_cuda_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->error = buf;
  return code;
}

#define IFE_CUDA_TRY(ctx, expr)                                                              \
  do {                                                                                       \
    cudaError_t e_ = (expr);                                                                 \
    if (e_ != cudaSuccess)                                                                   \
      return ife::fail(ctx, e_ == cudaErrorMemoryAllocation ? IFE_E_NOMEM : IFE_E_CUDA,      \
                       "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__,     \
                       __LINE__);                                                            \
  } while (0)

#define IFE_TRY(expr)          \
  do {                         \
    int rc_ = (expr);          \
    if (rc_ != IFE_OK) return rc_; \
  } while (0)

ProfScope::ProfScope(ife_cuda_ctx* c, int kind) : ctx(c) {
  if (!c->profiling) return;
  if (c->prof_used + 2 > c->prof_events.size()) {
    for (int i = 0; i < 2; ++i) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) return;
      c->prof_events.push_back(e);
    }
  }
  cudaEventRecord(c->prof_events[c->prof_used], c->stream());
  end = c->prof_events[c->prof_used + 1];
  c->prof_used += 2;
  c->prof_kinds.push_back(kind);
}
ProfScope::~ProfScope() {
  if (end) cudaEventRecord(end, ctx->stream());
}

int DeviceBuffer::reserve(ife_cuda_ctx* ctx, size_t want) {
  if (want <= bytes) return IFE_OK;
  if (ptr) {
    // every stream of the context may still be reading the old allocation (copy stream: D2H of
    // the previous scale / halo exchange; high-priority stream: option overlap_scales)
    IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->main_stream()));
    if (ctx->alt_stream) IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->alt_stream));
    if (ctx->copy_stream) IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
    if (ctx->hp_stream) IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->hp_stream));
    IFE_CUDA_TRY(ctx, cudaFree(ptr));
    ptr = nullptr;
    bytes = 0;
  }
  IFE_CUDA_TRY(ctx, cudaMalloc(&ptr, want));
  bytes = want;
  return IFE_OK;
}

void DeviceBuffer::release() {
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  bytes = 0;
}

// ---------------------------------------------------------------------------------------
// Coefficients of ITK's zero-order recursive Gaussian (Deriche 4th order with the
// Farneback-Westin parameter set), unit DC gain, symmetric anticausal part, constant-
// extension boundary terms.  sigma is physical; the recursion runs on samples.
// Replaces RecursiveGaussianImageFilter::SetUp as reached from
// include/ife/Filters/NormalizedGaussianConvolutionImageFilter.hxx:51-55.
// ---------------------------------------------------------------------------------------
GaussCoef make_gauss_coef(double sigma, double spacing) {
  const double sd = spacing < 1e-8 ? sigma : sigma / spacing;
  const double a[2] = {1.3530, -0.3531}, b[2] = {1.8151, 0.0902};
  const double w[2] = {0.6681, 2.0787}, l[2] = {-1.3932, -1.3732};
  double sn[2], cs[2], ex[2];
  for (int i = 0; i < 2; ++i) {
    sn[i] = std::sin(w[i] / sd);
    cs[i] = std::cos(w[i] / sd);
    ex[i] = std::exp(l[i] / sd);
  }
  GaussCoef c;
  double* D = c.D;  // D[0] = D1 ...
  D[3] = ex[0] * ex[0] * ex[1] * ex[1];
  D[2] = -2 * cs[0] * ex[0] * ex[1] * ex[1];
  D[2] += -2 * cs[1] * ex[1] * ex[0] * ex[0];
  D[1] = 4 * cs[1] * cs[0] * ex[0] * ex[1];
  D[1] += ex[0] * ex[0] + ex[1] * ex[1];
  D[0] = -2 * (ex[1] * cs[1] + ex[0] * cs[0]);
  const double SD = 1.0 + D[0] + D[1] + D[2] + D[3];

  double* N = c.N;
  N[0] = a[0] + a[1];
  N[1] = ex[1] * (b[1] * sn[1] - (a[1] + 2 * a[0]) * cs[1]);
  N[1] += ex[0] * (b[0] * sn[0] - (a[0] + 2 * a[1]) * cs[0]);
  N[2] = (a[0] + a[1]) * cs[1] * cs[0];
  N[2] -= b[0] * cs[1] * sn[0] + b[1] * cs[0] * sn[1];
  N[2] *= 2 * ex[0] * ex[1];
  N[2] += a[1] * ex[0] * ex[0] + a[0] * ex[1] * ex[1];
  N[3] = ex[1] * ex[0] * ex[0] * (b[1] * sn[1] - a[1] * cs[1]);
  N[3] += ex[0] * ex[1] * ex[1] * (b[0] * sn[0] - a[0] * cs[0]);
  const double SN0 = N[0] + N[1] + N[2] + N[3];
  const double alpha0 = 2 * SN0 / SD - N[0];
  for (int i = 0; i < 4; ++i) N[i] *= 1.0 / alpha0;

  c.M[0] = N[1] - D[0] * N[0];
  c.M[1] = N[2] - D[1] * N[0];
  c.M[2] = N[3] - D[2] * N[0];
  c.M[3] = -D[3] * N[0];
  const double SN = N[0] + N[1] + N[2] + N[3];
  const double SM = c.M[0] + c.M[1] + c.M[2] + c.M[3];
  for (int i = 0; i < 4; ++i) {
    c.BN[i] = D[i] * SN / SD;
    c.BM[i] = D[i] * SM / SD;
  }
  return c;
}

StencilCoef make_stencil_coef(const double spacing[3]) {
  StencilCoef s;
  for (int d = 0; d < 3; ++d) {
    const double inv = 1.0 / spacing[d];
    s.d1[d] = (double)(float)(0.5 * inv);
    s.d2a[d] = (double)(float)(1.0 * inv);
    s.d2b[d] = (double)(float)(-2.0 * inv);
    s.g1[d] = 0.5 * inv;
  }
  return s;
}

// ---------------------------------------------------------------------------------------
// Recursive Gaussian passes
// ---------------------------------------------------------------------------------------
constexpr int kChunk = 16;
#ifndef IFE_XWARPS
#define IFE_XWARPS 4
#endif
constexpr int kXWarps = IFE_XWARPS;

size_t ckpt_bytes(int nf, int n, size_t n_lines) {
  const int n_chunks = (n + kChunk - 1) / kChunk;
  return (size_t)std::max(n_chunks - 1, 0) * nf * 4 * n_lines * sizeof(double);
}

size_t ckpt_bytes_volume(int nf, int nx, int ny, int nz) {
  // lines padded to whole tiles of 32 (the tensor-map kernels checkpoint every lane of a tile)
  // one field: two stacks of ceil(rows / 2) rows each (smooth_volume), i.e. up to one row more
  const size_t px = (size_t)(nx + 31) / 32 * 32, py = (size_t)(ny + 31) / 32 * 32;
  const size_t ry = (size_t)ny + (nf == 1), rz = (size_t)nz + (nf == 1);
  const size_t a = ckpt_bytes(nf, nz, px * ry);
  const size_t b = ckpt_bytes(nf, nx, py * rz);
  const size_t c = ckpt_bytes(nf, ny, px * rz);
  return std::max(a, std::max(b, c));
}

// ---------------------------------------------------------------------------------------
// Tensor-map (TMA) passes: iir_tma.cuh.  cuTensorMapEncodeTiled comes from the driver through
// the runtime's entry-point query, so the library does not link libcuda.
// ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// 3-D view, x fastest: dims in elements, strides of dims 1 and 2 in bytes
int make_map3(ife_cuda_ctx* ctx, CUtensorMap* m, const void* base, bool u8, long long d0, long long d1, long long d2,
              long long stride1_bytes, long long stride2_bytes, int b0, int b1, int b2, bool swizzle64) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return fail(ctx, IFE_E_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  const cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
  const cuuint64_t strides[2] = {(cuuint64_t)stride1_bytes, (cuuint64_t)stride2_bytes};
  const cuuint32_t box[3] = {(cuuint32_t)b0, (cuuint32_t)b1, (cuuint32_t)b2};
  const cuuint32_t es[3] = {1, 1, 1};
  const CUresult r = fn(m, u8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                        const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ctx, IFE_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return IFE_OK;
}

#ifndef IFE_TMA_MINB_S
#define IFE_TMA_MINB_S 12    // resident 64-thread blocks per SM the strided passes' registers are cut for
#endif
#ifndef IFE_TMA_MINB_Z
#define IFE_TMA_MINB_Z 11    // z pass: 20.2 KB of shared memory per block (two roles + the tile of ones)
#endif
#ifndef IFE_TMA_MINB_ZF
#define IFE_TMA_MINB_ZF 9    // z pass with a float certainty: 25.3 KB of shared memory per block
#endif
#ifndef IFE_TMA_MINB_X
#define IFE_TMA_MINB_X 8
#endif

template <int AXIS, int INMODE, bool DIVIDE, int MASKMODE = 0>
int launch_tma_pass(ife_cuda_ctx* ctx, const GaussCoef& C, const CUtensorMap& i0, const CUtensorMap& i1,
                    const CUtensorMap& o0, const CUtensorMap& o1, const TmaArgs& A, dim3 grid) {
  constexpr int MINB = AXIS == AX_X ? IFE_TMA_MINB_X
                                    : (INMODE == IN_IMG_U8 ? IFE_TMA_MINB_Z : (INMODE == IN_IMG_F32 ? IFE_TMA_MINB_ZF : IFE_TMA_MINB_S));
  constexpr size_t smem_need = (INMODE == IN_IMG_U8    ? kRegionImgU8 + kRegionU8 + kOnesTile
                                : INMODE == IN_IMG_F32 ? kRegionImgF32 + kRegionF32 + kOnesTile
                                                       : 2 * (AXIS == AX_X ? kRegionX : kRegionF32)) + kTmaBarBytes;
  // The x pass (three staging slots per warp, TMA-latency-sensitive) is measurably faster with seven
  // blocks per SM than with the eight its shared memory allows (0.544 vs 0.555 ms): where more than
  // seven would fit (233472 B per SM, 1 KB of it reserved per block), the shared-memory request is
  // padded so that exactly seven do.
  constexpr bool seven = AXIS == AX_X && 233472 / (smem_need + 1024) > 7;
  constexpr size_t smem = seven ? std::max<size_t>(smem_need, (233472 / 7 - 1024) / 128 * 128) : smem_need;
  if (ctx->arith == IFE_ARITH_FMA) {
    auto kern = iir_tma_kernel<AXIS, INMODE, DIVIDE, true, MINB, MASKMODE>;
    IFE_CUDA_TRY(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, 64, smem, ctx->stream()>>>(C, i0, i1, o0, o1, A);
  } else {
    auto kern = iir_tma_kernel<AXIS, INMODE, DIVIDE, false, MINB, MASKMODE>;
    IFE_CUDA_TRY(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, 64, smem, ctx->stream()>>>(C, i0, i1, o0, o1, A);
  }
  ctx->launches++;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  return IFE_OK;
}

// Can the two-field smoothing of an nx x ny x nzb volume take the tensor-map kernels?
bool tma_passes_usable(const ife_cuda_ctx* ctx, const float* in0, const void* cert, bool cert_is_u8, const float* out0,
                       int nx, int ny, int nzb, const uint8_t* outmask_u8, const float* outmask_f32) {
  if (!ctx->use_tma || !cert) return false;
  // row pitch of 16 bytes for every map: nx % 16 for the uint8 certainty, nx % 4 for a float one; grid.y
  if (nx % (cert_is_u8 ? 16 : 4) != 0 || ny >= 65536 || nzb >= 65536) return false;
  auto al = [](const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; };
  return al(in0) && al(cert) && al(out0) && encode_tiled_fn() != nullptr;
}

// ... and the one-field smoothing (plain Gaussian)?  Rows of 16-byte multiples for the maps' strides.
bool tma_gaussian_usable(const ife_cuda_ctx* ctx, const float* in0, const void* cert, const float* out0, int nx, int ny,
                         int nzb, const uint8_t* outmask_u8, const float* outmask_f32) {
  if (!ctx->use_tma || cert || outmask_u8 || outmask_f32) return false;
  if (nx % 4 != 0 || ny >= 2 * 65535 || nzb >= 2 * 65535) return false;
  auto al = [](const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; };
  return al(in0) && al(out0) && encode_tiled_fn() != nullptr;
}

template <int NF, int INMODE, bool DIVIDE>
int launch_strided(ife_cuda_ctx* ctx, const GaussCoef& C, const PassArgs& A) {
  const unsigned grid = (unsigned)((A.n_lines + 127) / 128);
  ProfScope prof(ctx, A.stride == (long long)A.na && A.sb == 0 ? K_PASS_Z : K_PASS_Y);
  if (ctx->arith == IFE_ARITH_FMA)
    gauss_pass_strided<NF, INMODE, DIVIDE, kChunk, true><<<grid, 128, 0, ctx->stream()>>>(C, A);
  else
    gauss_pass_strided<NF, INMODE, DIVIDE, kChunk, false><<<grid, 128, 0, ctx->stream()>>>(C, A);
  ctx->launches++;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  return IFE_OK;
}

template <int NF>
int launch_x(ife_cuda_ctx* ctx, const GaussCoef& C, const PassArgs& A) {
  const long long lines_per_block = 32LL * kXWarps;
  const unsigned grid = (unsigned)((A.n_lines + lines_per_block - 1) / lines_per_block);
  ProfScope prof(ctx, K_PASS_X);
  if (ctx->arith == IFE_ARITH_FMA)
    gauss_pass_x<NF, kChunk, true, kXWarps><<<grid, 32 * kXWarps, 0, ctx->stream()>>>(C, A);
  else
    gauss_pass_x<NF, kChunk, false, kXWarps><<<grid, 32 * kXWarps, 0, ctx->stream()>>>(C, A);
  ctx->launches++;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  return IFE_OK;
}

// Smooth `nzb` planes of nx*ny.  Pass order z, x, y as SmoothingRecursiveGaussianImageFilter.
//   nf == 1: out0 = G(in0)                                       (in1 unused)
//   nf == 2: fields (in0*c, c) with c = in1 (u8 or f32); result = G(in0*c)/G(c) -> out0
// The z pass runs over all nzb planes; the x and y passes (which do not couple planes) only
// over planes [keep0, keep1), and out0 / outmask_* hold exactly those planes (a z-slab
// keeps its owned planes +-1 and drops the warm-up halo after the z pass).
// Scratch: ws.a0,a1,b0,b1 and ws.ckpt must already be large enough.
int smooth_volume(ife_cuda_ctx* ctx, const float* in0, const void* cert, bool cert_is_u8,
                  float* out0, int nx, int ny, int nzb, int keep0, int keep1,
                  const double spacing[3], double sigma, const uint8_t* outmask_u8,
                  const float* outmask_f32, const int* box = nullptr) {
  if (nx < 4 || ny < 4 || nzb < 4)
    return fail(ctx, IFE_E_TOO_SMALL,
                "recursive Gaussian needs at least 4 samples per axis (got %d x %d x %d)", nx, ny,
                nzb);
  if (!(sigma > 0.0)) return fail(ctx, IFE_E_INVALID, "sigma must be positive (got %g)", sigma);
  if (keep0 < 0 || keep1 > nzb || keep0 >= keep1) return fail(ctx, IFE_E_INVALID, "bad plane range");
  // Support box (masked paths, plan_masked): nothing outside it is ever read, so the z
  // pass only keeps the box's planes (below them the causal sweep alone runs, above them the
  // anticausal one), the x pass runs the rows of those planes, and the y pass the columns
  // (x, z) that cross the box, restricted to its y range.  Columns come in whole warps of 32.
  int kz0 = keep0, kz1 = keep1, kx0 = 0, kx1 = nx, ky0 = 0, ky1 = ny;
  if (box) {
    kz0 = std::max(keep0, box[4]); kz1 = std::min(keep1, box[5]);
    ky0 = box[2]; ky1 = box[3];
    if (nx % 32 == 0) { kx0 = box[0] / 32 * 32; kx1 = (box[1] + 31) / 32 * 32; }
    if (kz0 >= kz1 || ky0 >= ky1 || box[0] >= box[1]) return IFE_OK;   // no voxel is wanted
  }
  const int nf = cert ? 2 : 1;
  Workspace& ws = ctx->ws;
  const GaussCoef cz = make_gauss_coef(sigma, spacing[2]);
  const GaussCoef cx = make_gauss_coef(sigma, spacing[0]);
  const GaussCoef cy = make_gauss_coef(sigma, spacing[1]);
  float* a0 = (float*)ws.a0.ptr;
  float* a1 = (float*)ws.a1.ptr;
  float* b0 = (float*)ws.b0.ptr;
  float* b1 = (float*)ws.b1.ptr;

  if (tma_passes_usable(ctx, in0, cert, cert_is_u8, out0, nx, ny, nzb, outmask_u8, outmask_f32)) {
    // tensor-map staged passes (iir_tma.cuh): same windows, same results bit for bit
    const long long plane = (long long)nx * ny;
    const int nzk = kz1 - kz0;
    const size_t koff = (size_t)kz0 * plane, boff = (size_t)(kz0 - keep0) * plane;
    CUtensorMap mi0, mi1, mo0, mo1;
    TmaArgs T;
    std::memset(&T, 0, sizeof(T));
    T.ckpt = (double*)ws.ckpt.ptr;
    {   // z pass: lanes along x, block y = row, samples along z; the multiply c*T is fused into the loads
      IFE_TRY(make_map3(ctx, &mi0, in0, false, nx, ny, nzb, 4LL * nx, 4 * plane, 32, 1, kTRows, false));
      if (cert_is_u8) IFE_TRY(make_map3(ctx, &mi1, cert, true, nx, ny, nzb, nx, plane, 32, 1, kTRows, false));
      else IFE_TRY(make_map3(ctx, &mi1, cert, false, nx, ny, nzb, 4LL * nx, 4 * plane, 32, 1, kTRows, false));
      IFE_TRY(make_map3(ctx, &mo0, a0, false, nx, ny, nzb, 4LL * nx, 4 * plane, 32, 1, kTL, false));
      IFE_TRY(make_map3(ctx, &mo1, a1, false, nx, ny, nzb, 4LL * nx, 4 * plane, 32, 1, kTL, false));
      T.in0 = in0; T.in1 = cert;
      T.s_lane = 1; T.s_bx = 32; T.s_by = nx; T.s_n = plane; T.lanes_total = nx;
      T.n = nzb; T.out_lo = kz0; T.out_hi = kz1; T.rows1 = ny;
      ProfScope prof(ctx, K_PASS_Z);
      if (cert_is_u8) IFE_TRY((launch_tma_pass<AX_Z, IN_IMG_U8, false>(ctx, cz, mi0, mi1, mo0, mo1, T, dim3((nx + 31) / 32, ny))));
      else IFE_TRY((launch_tma_pass<AX_Z, IN_IMG_F32, false>(ctx, cz, mi0, mi1, mo0, mo1, T, dim3((nx + 31) / 32, ny))));
    }
    {   // x pass: lanes along y (one line each), block y = plane, samples along x
      IFE_TRY(make_map3(ctx, &mi0, a0 + koff, false, nx, ny, nzk, 4LL * nx, 4 * plane, kXRow, 32, 1, false));
      IFE_TRY(make_map3(ctx, &mi1, a1 + koff, false, nx, ny, nzk, 4LL * nx, 4 * plane, kXRow, 32, 1, false));
      IFE_TRY(make_map3(ctx, &mo0, b0 + boff, false, nx, ny, nzk, 4LL * nx, 4 * plane, kTL, 32, 1, true));
      IFE_TRY(make_map3(ctx, &mo1, b1 + boff, false, nx, ny, nzk, 4LL * nx, 4 * plane, kTL, 32, 1, true));
      T.in0 = a0 + koff; T.in1 = a1 + koff;
      T.s_lane = nx; T.s_bx = 32LL * nx; T.s_by = plane; T.s_n = 1; T.lanes_total = ny;
      T.n = nx; T.out_lo = 0; T.out_hi = nx; T.rows1 = nzk;
      ProfScope prof(ctx, K_PASS_X);
      IFE_TRY((launch_tma_pass<AX_X, IN_FIELDS, false>(ctx, cx, mi0, mi1, mo0, mo1, T, dim3((ny + 31) / 32, nzk))));
    }
    {   // y pass: lanes along x in [kx0, kx1), block y = plane, samples along y; the divide is fused into the stores
      const size_t yoff = boff + (size_t)kx0;
      const int wx = kx1 - kx0;
      IFE_TRY(make_map3(ctx, &mi0, b0 + yoff, false, wx, ny, nzk, 4LL * nx, 4 * plane, 32, kTRows, 1, false));
      IFE_TRY(make_map3(ctx, &mi1, b1 + yoff, false, wx, ny, nzk, 4LL * nx, 4 * plane, 32, kTRows, 1, false));
      IFE_TRY(make_map3(ctx, &mo0, out0 + yoff, false, wx, ny, nzk, 4LL * nx, 4 * plane, 32, kTL, 1, false));
      T.in0 = b0 + yoff; T.in1 = b1 + yoff;
      T.s_lane = 1; T.s_bx = 32; T.s_by = plane; T.s_n = nx; T.lanes_total = wx;
      T.n = ny; T.out_lo = ky0; T.out_hi = ky1; T.rows1 = nzk;
      ProfScope prof(ctx, K_PASS_Y);
      const dim3 gy((wx + 31) / 32, nzk);
      if (outmask_u8) {
        T.mask = outmask_u8 + yoff;
        IFE_TRY((launch_tma_pass<AX_Y, IN_FIELDS, true, 1>(ctx, cy, mi0, mi1, mo0, mo0, T, gy)));
      } else if (outmask_f32) {
        T.mask = outmask_f32 + yoff;
        IFE_TRY((launch_tma_pass<AX_Y, IN_FIELDS, true, 2>(ctx, cy, mi0, mi1, mo0, mo0, T, gy)));
      } else {
        IFE_TRY((launch_tma_pass<AX_Y, IN_FIELDS, true>(ctx, cy, mi0, mi1, mo0, mo0, T, gy)));
      }
    }
    return IFE_OK;
  }

  if (tma_gaussian_usable(ctx, in0, cert, out0, nx, ny, nzb, outmask_u8, outmask_f32)) {
    // One field (the plain smoothing Gaussian) through the same kernels: the second warp of a block,
    // which carries field c in the normalized convolution, takes a second stack of rows instead --
    // the upper half of the y rows in the z pass, the upper half of the planes in the x and y passes.
    // Its tensor maps are views of that half, so the kernels see two independent "fields".
    const long long plane = (long long)nx * ny;
    const int nzk = kz1 - kz0;
    const size_t koff = (size_t)kz0 * plane, boff = (size_t)(kz0 - keep0) * plane;
    CUtensorMap mi0, mi1, mo0, mo1;
    TmaArgs T;
    std::memset(&T, 0, sizeof(T));
    T.ckpt = (double*)ws.ckpt.ptr;
    {   // z pass: rows [0, h) and [h, ny)
      const int h = (ny + 1) / 2, h1 = ny - h;   // h1 >= 2
      const size_t off1 = (size_t)h * nx;
      IFE_TRY(make_map3(ctx, &mi0, in0, false, nx, h, nzb, 4LL * nx, 4 * plane, 32, 1, kTRows, false));
      IFE_TRY(make_map3(ctx, &mi1, in0 + off1, false, nx, h1, nzb, 4LL * nx, 4 * plane, 32, 1, kTRows, false));
      IFE_TRY(make_map3(ctx, &mo0, a0, false, nx, h, nzb, 4LL * nx, 4 * plane, 32, 1, kTL, false));
      IFE_TRY(make_map3(ctx, &mo1, a0 + off1, false, nx, h1, nzb, 4LL * nx, 4 * plane, 32, 1, kTL, false));
      T.in0 = in0; T.in1 = in0 + off1;
      T.s_lane = 1; T.s_bx = 32; T.s_by = nx; T.s_n = plane; T.lanes_total = nx;
      T.n = nzb; T.out_lo = kz0; T.out_hi = kz1; T.rows1 = h1;
      ProfScope prof(ctx, K_PASS_Z);
      IFE_TRY((launch_tma_pass<AX_Z, IN_FIELDS, false>(ctx, cz, mi0, mi1, mo0, mo1, T, dim3((nx + 31) / 32, h))));
    }
    const int h = (nzk + 1) / 2, h1 = nzk - h;   // x and y passes: planes [0, h) and [h, nzk) of the kept range
    const int m1 = std::max(h1, 1);              // a map needs a non-empty extent even when nobody uses it
    const size_t off1 = (size_t)h * plane;
    {   // x pass
      IFE_TRY(make_map3(ctx, &mi0, a0 + koff, false, nx, ny, h, 4LL * nx, 4 * plane, kXRow, 32, 1, false));
      IFE_TRY(make_map3(ctx, &mi1, a0 + koff + off1, false, nx, ny, m1, 4LL * nx, 4 * plane, kXRow, 32, 1, false));
      IFE_TRY(make_map3(ctx, &mo0, b0 + boff, false, nx, ny, h, 4LL * nx, 4 * plane, kTL, 32, 1, true));
      IFE_TRY(make_map3(ctx, &mo1, b0 + boff + off1, false, nx, ny, m1, 4LL * nx, 4 * plane, kTL, 32, 1, true));
      T.in0 = a0 + koff; T.in1 = a0 + koff + off1;
      T.s_lane = nx; T.s_bx = 32LL * nx; T.s_by = plane; T.s_n = 1; T.lanes_total = ny;
      T.n = nx; T.out_lo = 0; T.out_hi = nx; T.rows1 = h1;
      ProfScope prof(ctx, K_PASS_X);
      IFE_TRY((launch_tma_pass<AX_X, IN_FIELDS, false>(ctx, cx, mi0, mi1, mo0, mo1, T, dim3((ny + 31) / 32, h))));
    }
    {   // y pass, straight into the result
      IFE_TRY(make_map3(ctx, &mi0, b0 + boff, false, nx, ny, h, 4LL * nx, 4 * plane, 32, kTRows, 1, false));
      IFE_TRY(make_map3(ctx, &mi1, b0 + boff + off1, false, nx, ny, m1, 4LL * nx, 4 * plane, 32, kTRows, 1, false));
      IFE_TRY(make_map3(ctx, &mo0, out0 + boff, false, nx, ny, h, 4LL * nx, 4 * plane, 32, kTL, 1, false));
      IFE_TRY(make_map3(ctx, &mo1, out0 + boff + off1, false, nx, ny, m1, 4LL * nx, 4 * plane, 32, kTL, 1, false));
      T.in0 = b0 + boff; T.in1 = b0 + boff + off1;
      T.s_lane = 1; T.s_bx = 32; T.s_by = plane; T.s_n = nx; T.lanes_total = nx;
      T.n = ny; T.out_lo = ky0; T.out_hi = ky1; T.rows1 = h1;
      ProfScope prof(ctx, K_PASS_Y);
      IFE_TRY((launch_tma_pass<AX_Y, IN_FIELDS, false>(ctx, cy, mi0, mi1, mo0, mo1, T, dim3((nx + 31) / 32, h))));
    }
    return IFE_OK;
  }

  // Plain register-staged kernels (any layout): the same lines as above, each swept whole; the
  // samples outside the windows that they also write are never read.
  PassArgs A;
  std::memset(&A, 0, sizeof(A));
  A.ckpt = (double*)ws.ckpt.ptr;

  // z pass: lines = nx*ny columns, contiguous across the plane
  A.in0 = in0; A.in1 = cert; A.out0 = a0; A.out1 = a1;
  A.n = nzb; A.stride = (long long)nx * ny; A.na = nx * ny > 0 ? nx * ny : 1; A.sb = 0;
  A.n_lines = (long long)nx * ny;
  if (nf == 1) IFE_TRY((launch_strided<1, IN_FIELDS, false>(ctx, cz, A)));
  else if (cert_is_u8) IFE_TRY((launch_strided<2, IN_IMG_U8, false>(ctx, cz, A)));
  else IFE_TRY((launch_strided<2, IN_IMG_F32, false>(ctx, cz, A)));

  // x pass: lines = ny*nzk rows, contiguous (b0/b1/out0 hold planes [keep0, keep1): plane kz0
  // sits at offset kz0 - keep0)
  const int nzk = kz1 - kz0;
  const size_t plane = (size_t)nx * ny;
  const size_t koff = (size_t)kz0 * plane, boff = (size_t)(kz0 - keep0) * plane;
  A.in0 = a0 + koff; A.in1 = a1 + koff; A.out0 = b0 + boff; A.out1 = b1 + boff;
  A.n = nx; A.stride = 1; A.na = 1; A.sb = 0; A.n_lines = (long long)ny * nzk;
  if (nf == 1) IFE_TRY((launch_x<1>(ctx, cx, A)));
  else IFE_TRY((launch_x<2>(ctx, cx, A)));

  // y pass: lines indexed (x, z) with x in [kx0, kx1); base = x + z*nx*ny; stride nx
  const size_t yoff = boff + (size_t)kx0;
  A.in0 = b0 + yoff; A.in1 = b1 + yoff; A.out0 = out0 + yoff; A.out1 = nullptr;
  A.n = ny; A.stride = nx; A.na = kx1 - kx0; A.sb = (long long)plane; A.n_lines = (long long)(kx1 - kx0) * nzk;
  A.mask_u8 = outmask_u8 ? outmask_u8 + yoff : nullptr;
  A.mask_f32 = outmask_f32 ? outmask_f32 + yoff : nullptr;
  if (nf == 1) IFE_TRY((launch_strided<1, IN_FIELDS, false>(ctx, cy, A)));
  else IFE_TRY((launch_strided<2, IN_FIELDS, true>(ctx, cy, A)));
  return IFE_OK;
}

// Support box of a mask (see support_box.cuh).  Three steps so that a batch can run the
// reduction on its copy stream right behind the upload of the mask:
//   support_box_usable  option on and the layout allows the 16-byte scan (else the passes run
//                       everywhere);
//   launch_support_box  reduction kernel + read-back of the six extents into pinned slot
//                       `slot` (0 or 1), on stream `st`;
//   finish_support_box  after `st` got there: box = {x0,x1,y0,y1,z0,z1}, half-open, clipped to
//                       the bounding box of an ROI list (host array of n_roi x {x,y,z,sx,sy,sz})
//                       when there is one, grown by the stencil reach of one voxel; all zero
//                       when no voxel is wanted.
bool support_box_usable(const ife_cuda_ctx* ctx, const uint8_t* d_mask, int nx, int ny, int nz) {
  return ctx->use_box && d_mask && nx % 16 == 0 && reinterpret_cast<uintptr_t>(d_mask) % 16 == 0 &&
         (long long)ny * nz < (1LL << 31);
}

int launch_support_box(ife_cuda_ctx* ctx, const uint8_t* d_mask, int nx, int ny, int nz,
                       cudaStream_t st, int slot) {
  IFE_TRY(ctx->ws.box.reserve(ctx, 12 * sizeof(int)));
  if (!ctx->box_host)
    IFE_CUDA_TRY(ctx, cudaHostAlloc((void**)&ctx->box_host, 12 * sizeof(int), cudaHostAllocDefault));
  int* raw = (int*)ctx->ws.box.ptr + 6 * slot;
  IFE_CUDA_TRY(ctx, cudaMemsetAsync(raw, 0, 6 * sizeof(int), st));
  const unsigned n_rows = (unsigned)((long long)ny * nz);
  const unsigned grid = (unsigned)std::min<long long>(((long long)n_rows + 31) / 32, 8LL * ctx->sm_count);
  mask_box_kernel<<<grid, 256, 0, st>>>(d_mask, nx, ny, n_rows, raw);
  ctx->launches++;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->box_host + 6 * slot, raw, 6 * sizeof(int), cudaMemcpyDeviceToHost, st));
  return IFE_OK;
}

void finish_support_box(const ife_cuda_ctx* ctx, int slot, int nx, int ny, int nz, const int* rois,
                        int n_roi, int box[6]) {
  const int* h = ctx->box_host + 6 * slot;
  const int n[3] = {nx, ny, nz};
  int lo[3], hi[3];
  bool empty = false;
  for (int d = 0; d < 3; ++d) {
    lo[d] = kBoxBig - h[2 * d];
    hi[d] = h[2 * d + 1];
  }
  if (n_roi > 0 && rois) {
    for (int d = 0; d < 3; ++d) {
      int rlo = n[d], rhi = 0;
      for (int r = 0; r < n_roi; ++r) {
        rlo = std::min(rlo, rois[6 * r + d]);
        rhi = std::max(rhi, rois[6 * r + d] + rois[6 * r + 3 + d]);
      }
      lo[d] = std::max(lo[d], rlo);
      hi[d] = std::min(hi[d], rhi);
    }
  }
  for (int d = 0; d < 3; ++d) empty = empty || lo[d] >= hi[d];
  for (int d = 0; d < 3; ++d) {
    box[2 * d] = empty ? 0 : std::max(lo[d] - 1, 0);
    box[2 * d + 1] = empty ? 0 : std::min(hi[d] + 1, n[d]);
  }
}

// ---------------------------------------------------------------------------------------
// Masked smoothing.  With a mask c in {0, != 0} both fields of the normalized convolution, c*T
// and c, are EXACT zeros outside the mask's bounding box.  The recursion of a line that has
// only seen zeros is in the zero state, and ITK's boundary rule (the first sample extended to
// infinity) starts a line whose first sample is zero in that same state.  So smoothing the
// bounding box grown by one voxel as if it were the whole image -- a dense copy of it -- gives
// the same bits inside it as smoothing the whole image, for all three passes, at a cost
// proportional to the box instead of the volume.  (Where the box touches the image border
// the first sample is the image's own: the same rule either way.)  An ROI list shrinks what
// is needed further but not what is zero: there the box of the mask is cropped and the
// ROI-clipped box windows the passes inside the crop (smooth_volume's `box`).
// ---------------------------------------------------------------------------------------
struct MaskedPlan {
  bool have_box = false;   // the support box is known (else: smooth everything)
  bool empty = false;      // no voxel is wanted
  bool cropped = false;    // the passes run on a cropped copy
  int box[6];              // wanted region, full coordinates (ROI-clipped, grown by one voxel)
  int org[3], cdim[3];     // crop origin / size
  int cbox[6];             // `box` in crop coordinates
  bool window = false;     // cbox is much smaller than the crop: window the passes with it
  const float* img = nullptr;      // what the passes read: the cropped copies or the caller's
  const uint8_t* mask = nullptr;
};

// widen [lo, hi) to at least 4 samples inside [0, n) and, where there is room, to a multiple
// of the chunk length (whole chunks at both ends of a line take the interleaved loop); the
// added samples are zeros like everything else outside the mask's box
inline void widen4(int& lo, int& hi, int n) {
  while (hi - lo < 4 && hi < n) ++hi;
  while (hi - lo < 4 && lo > 0) --lo;
  while ((hi - lo) % kChunk != 0 && hi < n) ++hi;
  while ((hi - lo) % kChunk != 0 && lo > 0) --lo;
}

// After the extents of slot `slot` are on the host.  Launches the crop on the context's stream.
int plan_masked(ife_cuda_ctx* ctx, bool have_box, int slot, const float* d_img, const uint8_t* d_mask,
                int nx, int ny, int nz, const int* rois, int n_roi, MaskedPlan* P) {
  *P = MaskedPlan();
  P->img = d_img; P->mask = d_mask;
  P->have_box = have_box;
  ctx->work_dims[0] = nx; ctx->work_dims[1] = ny; ctx->work_dims[2] = nz;
  if (!have_box) return IFE_OK;
  int mbox[6];
  finish_support_box(ctx, slot, nx, ny, nz, nullptr, 0, mbox);
  finish_support_box(ctx, slot, nx, ny, nz, rois, n_roi, P->box);
  P->empty = P->box[0] >= P->box[1];
  if (P->empty) return IFE_OK;
  if (nx % 32 != 0 || reinterpret_cast<uintptr_t>(d_img) % 16 != 0) return IFE_OK;
  int lo[3] = {mbox[0] / 32 * 32, mbox[2], mbox[4]};
  int hi[3] = {std::min(nx, (mbox[1] + 31) / 32 * 32), mbox[3], mbox[5]};
  widen4(lo[1], hi[1], ny);
  widen4(lo[2], hi[2], nz);
  const long long nc = (long long)(hi[0] - lo[0]) * (hi[1] - lo[1]) * (hi[2] - lo[2]);
  if ((double)nc > 0.85 * (double)nx * ny * nz) return IFE_OK;   // not worth the copy
  for (int d = 0; d < 3; ++d) { P->org[d] = lo[d]; P->cdim[d] = hi[d] - lo[d]; }
  for (int d = 0; d < 3; ++d) {
    P->cbox[2 * d] = std::max(P->box[2 * d] - lo[d], 0);
    P->cbox[2 * d + 1] = std::min(P->box[2 * d + 1] - lo[d], P->cdim[d]);
  }
  const long long nb = (long long)(P->cbox[1] - P->cbox[0]) * (P->cbox[3] - P->cbox[2]) * (P->cbox[5] - P->cbox[4]);
  P->window = n_roi > 0 && (double)nb < 0.8 * (double)nc;
  Workspace& ws = ctx->ws;
  IFE_TRY(ws.crop_img.reserve(ctx, (size_t)nc * sizeof(float)));
  IFE_TRY(ws.crop_mask.reserve(ctx, (size_t)nc));
  IFE_TRY(ws.crop_blur.reserve(ctx, (size_t)nc * sizeof(float)));
  const long long n4 = nc / 4;
  const unsigned grid = (unsigned)std::min<long long>((n4 + 255) / 256, 16LL * ctx->sm_count);
  crop_box_kernel<<<grid, 256, 0, ctx->stream()>>>(d_img, d_mask, (float*)ws.crop_img.ptr, (uint8_t*)ws.crop_mask.ptr,
                                                   nx, ny, lo[0], lo[1], lo[2], P->cdim[0], P->cdim[1], n4);
  ctx->launches++;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  P->cropped = true;
  for (int d = 0; d < 3; ++d) ctx->work_dims[d] = P->cdim[d];
  P->img = (const float*)ws.crop_img.ptr;
  P->mask = (const uint8_t*)ws.crop_mask.ptr;
  return IFE_OK;
}

// The same for one scan on the context's stream: the support box's reduction, one wait for its
// extents, then the plan.
int plan_masked(ife_cuda_ctx* ctx, const float* d_img, const uint8_t* d_mask, int nx, int ny, int nz,
                const int* rois, int n_roi, MaskedPlan* P) {
  const bool have_box = support_box_usable(ctx, d_mask, nx, ny, nz);
  if (have_box) {
    IFE_TRY(launch_support_box(ctx, d_mask, nx, ny, nz, ctx->stream(), 0));
    IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream()));
  }
  return plan_masked(ctx, have_box, 0, d_img, d_mask, nx, ny, nz, rois, n_roi, P);
}

// Upload a scan's ROI list to d_rois on the context's stream.  With a crop the list is moved into
// crop coordinates and clipped to the crop (in-mask voxels all lie inside it) in `moved`, which
// must outlive the copy.
int upload_rois(ife_cuda_ctx* ctx, const MaskedPlan& P, const int* rois, int n_roi, int* d_rois,
                std::vector<int>* moved) {
  if (n_roi == 0) return IFE_OK;
  if (P.cropped) {
    moved->assign((size_t)n_roi * 6, 0);
    for (int i = 0; i < n_roi; ++i) {
      int lo[3], hi[3];
      bool empty = false;
      for (int d = 0; d < 3; ++d) {
        lo[d] = std::max(rois[6 * i + d] - P.org[d], 0);
        hi[d] = std::min(rois[6 * i + d] + rois[6 * i + 3 + d] - P.org[d], P.cdim[d]);
        empty = empty || lo[d] >= hi[d];
      }
      for (int d = 0; d < 3; ++d) {
        (*moved)[6 * i + d] = empty ? 0 : lo[d];
        (*moved)[6 * i + 3 + d] = empty ? 0 : hi[d] - lo[d];
      }
    }
    rois = moved->data();
  }
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(d_rois, rois, (size_t)n_roi * 6 * sizeof(int), cudaMemcpyHostToDevice,
                                    ctx->stream()));
  return IFE_OK;
}

// blur (full layout) <- normalized Gaussian of (img, mask) at `sigma`, valid wherever P.box says
// (uncrop = false: the result stays in ws.crop_blur, crop layout -- histogram-only callers run the
// fused kernel on the crop as well)
int smooth_masked(ife_cuda_ctx* ctx, const MaskedPlan& P, const float* d_img, const uint8_t* d_mask,
                  float* blur, int nx, int ny, int nz, const double spacing[3], double sigma,
                  bool uncrop = true) {
  if (P.have_box && P.empty) return IFE_OK;
  if (!P.cropped)
    return smooth_volume(ctx, d_img, d_mask, true, blur, nx, ny, nz, 0, nz, spacing, sigma, nullptr, nullptr,
                         P.have_box ? P.box : nullptr);
  float* cblur = (float*)ctx->ws.crop_blur.ptr;
  IFE_TRY(smooth_volume(ctx, P.img, P.mask, true, cblur, P.cdim[0], P.cdim[1], P.cdim[2], 0, P.cdim[2], spacing,
                        sigma, nullptr, nullptr, P.window ? P.cbox : nullptr));
  if (!uncrop) return IFE_OK;
  const long long n4 = (long long)P.cdim[0] * P.cdim[1] * P.cdim[2] / 4;
  const unsigned grid = (unsigned)std::min<long long>((n4 + 255) / 256, 16LL * ctx->sm_count);
  uncrop_kernel<<<grid, 256, 0, ctx->stream()>>>(cblur, blur, nx, ny, P.org[0], P.org[1], P.org[2], P.cdim[0],
                                                 P.cdim[1], n4);
  ctx->launches++;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  return IFE_OK;
}

int reserve_smoothing(ife_cuda_ctx* ctx, int nf, int nx, int ny, int nzb) {
  Workspace& ws = ctx->ws;
  const size_t vol = (size_t)nx * ny * nzb * sizeof(float);
  IFE_TRY(ws.a0.reserve(ctx, vol));
  IFE_TRY(ws.b0.reserve(ctx, vol));
  if (nf == 2) {
    IFE_TRY(ws.a1.reserve(ctx, vol));
    IFE_TRY(ws.b1.reserve(ctx, vol));
  }
  IFE_TRY(ws.ckpt.reserve(ctx, std::max<size_t>(ckpt_bytes_volume(nf, nx, ny, nzb), 8)));
  return IFE_OK;
}

// ---------------------------------------------------------------------------------------
// Fused feature kernel launch
// ---------------------------------------------------------------------------------------
template <int MODE, bool HIST>
void launch_features_t(bool unit, dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                       const StencilCoef& S, const FeatArgs& A, int zchunk) {
  constexpr int NFEAT = MODE == 0 ? 8 : ((MODE == 1 || MODE == 3) ? 6 : 1);
  bool all = true, none = true;
  for (int k = 0; k < NFEAT; ++k) { all = all && A.out[k] != nullptr; none = none && A.out[k] == nullptr; }
  if (zchunk < 0) {   // four voxels per thread (features_march4.cuh); grid / block were sized for it
    zchunk = -zchunk;
    auto go = [&](void (*kern)(StencilCoef, FeatArgs, int)) {
      if (smem > 30 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      kern<<<grid, block, smem, st>>>(S, A, zchunk);
    };
    if (HIST && none && unit) go(features_march4_kernel<MODE, HIST, true, HIST ? 2 : 0>);   // histograms only
    else if (all && unit) go(features_march4_kernel<MODE, HIST, true, 1>);
    else if (unit) go(features_march4_kernel<MODE, HIST, true, 0>);
    else go(features_march4_kernel<MODE, HIST, false, 0>);
    return;
  }
  if (zchunk > 0) {   // z-marching kernel (everything but ROI-list histograms)
    auto go = [&](void (*kern)(StencilCoef, FeatArgs, int)) {
      if (smem > 40 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      kern<<<grid, block, smem, st>>>(S, A, zchunk);
    };
    if (HIST && none && unit) go(features_march_kernel<MODE, HIST, true, HIST ? 2 : 0>);   // histograms only
    else if (all && unit) go(features_march_kernel<MODE, HIST, true, 1>);
    else if (unit) go(features_march_kernel<MODE, HIST, true, 0>);
    else go(features_march_kernel<MODE, HIST, false, 0>);
    return;
  }
  constexpr int BM = MODE == 3 ? 1 : MODE;   // the raw Hessian only exists in the z-march kernel (checked by the caller)
  if (all && unit) features_kernel<BM, HIST, true, true><<<grid, block, smem, st>>>(S, A);
  else if (unit) features_kernel<BM, HIST, true, false><<<grid, block, smem, st>>>(S, A);
  else features_kernel<BM, HIST, false, false><<<grid, block, smem, st>>>(S, A);
}

// shared memory of the z-march kernel's histogram sink: padded edge rows + private counter columns
inline size_t march_hist_smem(int nfeat, int n_edges) {
  return (size_t)nfeat * ((size_t)hist_edge_pitch(n_edges) * sizeof(float) +
                          (size_t)(n_edges + 1) * (kMX * kMY));   // one byte per (bin, thread)
}
inline bool march_hist_fits(int nfeat, int n_edges) { return march_hist_smem(nfeat, n_edges) <= 96 * 1024; }

int launch_features(ife_cuda_ctx* ctx, int mode, const StencilCoef& S, const FeatArgs& A,
                    bool unit_spacing) {
  const bool hist = A.hist.edges != nullptr;
  const int nfeat = mode == 0 ? 8 : ((mode == 1 || mode == 3) ? 6 : 1);
  const int nzo = A.zb1 - A.zb0;
  if (nzo <= 0 || A.nx <= 0 || A.ny <= 0) return IFE_OK;
  dim3 block(kTX, kTY, 1);
  dim3 grid((A.nx + kTX - 1) / kTX, (A.ny + kTY - 1) / kTY, (nzo + kTZ - 1) / kTZ);
  // ROI-list histograms keep the brick kernel (bricks that touch no ROI exit at once);
  // everything else marches 32x8 columns in z, in chunks sized for >= ~8 waves of blocks
  int zchunk = 0;
  if (!(hist && A.hist.n_roi > 0) && !A.mask_f32 && (long long)A.nx * A.ny < (1LL << 28)) {
    block = dim3(kMX, kMY, 1);
    grid.x = (A.nx + kMX - 1) / kMX;
    grid.y = (A.ny + kMY - 1) / kMY;
    const long long cols = (long long)grid.x * grid.y;
    const long long want = (8LL * (1024 / (kMX * kMY)) * ctx->sm_count + cols - 1) / cols;   // chunks per column
    zchunk = (int)std::max<long long>(16, (nzo + want - 1) / want);
    zchunk = std::min(zchunk, nzo);
    zchunk = (int)std::min<long long>(zchunk, (1LL << 31) / ((long long)A.nx * A.ny) - 2);   // 32-bit offsets
    grid.z = (nzo + zchunk - 1) / zchunk;
  }
  if (grid.y > 65535 || grid.z > 65535) return fail(ctx, IFE_E_INVALID, "volume too large for the launch grid");
  if (mode == 3 && zchunk == 0) return fail(ctx, IFE_E_INVALID, "raw Hessian output needs planes below 2^28 voxels");
  // brick kernel: edge rows as given + uint32 counters; march kernel: rows padded to a power
  // of two + one private 8-bit counter column per thread (falls back to the brick kernel when
  // that does not fit)
  size_t smem = 0;
  if (hist && zchunk > 0) {
    smem = march_hist_smem(nfeat, A.hist.n_edges);
    if (!march_hist_fits(nfeat, A.hist.n_edges)) {
      zchunk = 0;
      block = dim3(kTX, kTY, 1);
      grid = dim3((A.nx + kTX - 1) / kTX, (A.ny + kTY - 1) / kTY, (nzo + kTZ - 1) / kTZ);
    } else if (zchunk > 255) {
      zchunk = 255;    // 8-bit private counters: a thread must not see more than 255 voxels
      grid.z = (nzo + zchunk - 1) / zchunk;
    }
  }
  if (hist && zchunk == 0)
    smem = (size_t)nfeat * (A.hist.n_edges * sizeof(float) + (A.hist.n_edges + 1) * sizeof(uint32_t));
  if (zchunk == 0 && smem > 30 * 1024)
    return fail(ctx, IFE_E_INVALID, "too many histogram edges (%d) for shared memory", A.hist.n_edges);
  // four voxels per thread when the layout allows 16-byte staging and stores
  if (zchunk > 0 && ctx->use_march4 && (A.nx & 3) == 0) {
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    bool ok = al16(A.vol) && (!A.mask_u8 || (reinterpret_cast<uintptr_t>(A.mask_u8) & 3) == 0) &&
              (!A.hist.packed || al16(A.hist.packed));
    for (int k = 0; k < nfeat; ++k) ok = ok && al16(A.out[k]);
    if (ok) {
      block = dim3(kQX, kQY, 1);
      grid.x = (A.nx + kQW - 1) / kQW;
      grid.y = (A.ny + kQY - 1) / kQY;
      const long long cols = (long long)grid.x * grid.y;
      const long long want = (8LL * 4 * ctx->sm_count + cols - 1) / cols;   // chunks per column for ~8 waves of blocks
      int zc = (int)std::max<long long>(16, (nzo + want - 1) / want);
      zc = std::min(zc, nzo);
      if (hist) zc = std::min(zc, 63);   // 8-bit private counters: four voxels per plane and thread
      grid.z = (nzo + zc - 1) / zc;
      zchunk = -zc;
    }
  }
  cudaStream_t st = ctx->stream();
  ProfScope prof(ctx, mode == 2 ? K_OTHER : K_FEATURES);
  if (mode == 0) {
    if (hist) launch_features_t<0, true>(unit_spacing, grid, block, smem, st, S, A, zchunk);
    else launch_features_t<0, false>(unit_spacing, grid, block, 0, st, S, A, zchunk);
  } else if (mode == 1) {
    if (hist) launch_features_t<1, true>(unit_spacing, grid, block, smem, st, S, A, zchunk);
    else launch_features_t<1, false>(unit_spacing, grid, block, 0, st, S, A, zchunk);
  } else if (mode == 3) {
    if (hist) return fail(ctx, IFE_E_INVALID, "raw Hessian output has no histogram sink");
    launch_features_t<3, false>(unit_spacing, grid, block, 0, st, S, A, zchunk);
  } else {
    if (hist) launch_features_t<2, true>(unit_spacing, grid, block, smem, st, S, A, zchunk);
    else launch_features_t<2, false>(unit_spacing, grid, block, 0, st, S, A, zchunk);
  }
  ctx->launches++;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  return IFE_OK;
}

inline bool is_unit_spacing(const double spacing[3]) {
  return spacing[0] == 1.0 && spacing[1] == 1.0 && spacing[2] == 1.0;
}

// ROI lists longer than this take the packed-bin path (one block per ROI)
constexpr int kManyRois = 192;

// The histograms of one scan (ife_cuda_emphysema_histograms and each scan of _histograms_batch):
// per scale the normalized convolution of the plan's volume and the fused kernel's histogram sink,
// on the crop when there is one, since no feature volume leaves the call.  d_edges:
// [n_sigma*8][n_edges]; d_rois: the scan's ROI list in the plan's frame (upload_rois); d_counts:
// [max(n_roi,1)][n_sigma*8][n_edges+1], zeroed.  Of the workspace only the smoothing buffers and
// ws.packed are touched: a batch keeps its upload and count slots in ws.in_*, ws.out[*], ws.counts.
int bin_masked_scan(ife_cuda_ctx* ctx, const MaskedPlan& P, const float* d_img, const uint8_t* d_mask,
                    int nx, int ny, int nz, const double spacing[3], const double* sigmas, int n_sigma,
                    const float* d_edges, int n_edges, const int* d_rois, int n_roi, uint32_t* d_counts) {
  if (P.have_box && P.empty) return IFE_OK;   // no voxel is wanted
  // Many ROIs (MakeBagDense, large MakeBag runs): the per-voxel search through the ROI list of
  // the brick kernel does not scale, so the fused kernel leaves packed bin indices and one
  // block per ROI counts its box (roi_hist_packed_kernel).
  const bool many_rois = n_roi > kManyRois && n_edges <= 253 && march_hist_fits(8, n_edges) &&
                         (long long)nx * ny < (1LL << 28);
  if (many_rois) IFE_TRY(ctx->ws.packed.reserve(ctx, (size_t)nx * ny * nz * sizeof(unsigned long long)));
  const int fx = P.cropped ? P.cdim[0] : nx, fy = P.cropped ? P.cdim[1] : ny, fz = P.cropped ? P.cdim[2] : nz;
  const int nb = n_edges + 1;
  const StencilCoef S = make_stencil_coef(spacing);
  float* blur = P.cropped ? (float*)ctx->ws.crop_blur.ptr : (float*)ctx->ws.blur.ptr;
  for (int s = 0; s < n_sigma; ++s) {
    IFE_TRY(smooth_masked(ctx, P, d_img, d_mask, blur, nx, ny, nz, spacing, sigmas[s], false));
    FeatArgs A;
    std::memset(&A, 0, sizeof(A));
    A.vol = blur; A.mask_u8 = P.mask;
    A.nx = fx; A.ny = fy; A.nzb = fz; A.zb0 = 0; A.zb1 = fz;
    A.hist.edges = d_edges + (size_t)s * 8 * n_edges;
    A.hist.counts = d_counts + (size_t)s * 8 * nb;
    A.hist.n_edges = n_edges;
    A.hist.stride_roi = (long long)n_sigma * 8 * nb;
    if (many_rois) {
      A.hist.packed = (unsigned long long*)ctx->ws.packed.ptr;
      IFE_TRY(launch_features(ctx, 0, S, A, is_unit_spacing(spacing)));
      ProfScope prof(ctx, K_OTHER);
      roi_hist_packed_kernel<<<(unsigned)n_roi, 256, (size_t)8 * nb * sizeof(uint32_t), ctx->stream()>>>(
          A.hist.packed, fx, fy, d_rois, nb, A.hist.counts, A.hist.stride_roi);
      ctx->launches++;
      IFE_CUDA_TRY(ctx, cudaGetLastError());
    } else {
      A.hist.rois = d_rois; A.hist.n_roi = n_roi;
      IFE_TRY(launch_features(ctx, 0, S, A, is_unit_spacing(spacing)));
    }
  }
  return IFE_OK;
}

int check_dims(ife_cuda_ctx* ctx, const int dims[3], const double spacing[3]) {
  if (!dims || !spacing) return fail(ctx, IFE_E_INVALID, "dims/spacing must not be null");
  for (int d = 0; d < 3; ++d) {
    if (dims[d] <= 0) return fail(ctx, IFE_E_INVALID, "dims[%d] = %d must be positive", d, dims[d]);
    if (!(spacing[d] > 0.0))
      return fail(ctx, IFE_E_INVALID, "spacing[%d] = %g must be positive", d, spacing[d]);
  }
  return IFE_OK;
}

// Every box of an ROI list (host, n_roi x {x0,y0,z0,sx,sy,sz}) is non-empty and inside the image.
int check_rois(ife_cuda_ctx* ctx, const int* rois, int n_roi, const int dims[3]) {
  for (int r = 0; r < n_roi; ++r) {
    const int* b = rois + 6 * r;
    if (b[0] < 0 || b[1] < 0 || b[2] < 0 || b[3] <= 0 || b[4] <= 0 || b[5] <= 0 ||
        b[0] + b[3] > dims[0] || b[1] + b[4] > dims[1] || b[2] + b[5] > dims[2])
      return fail(ctx, IFE_E_INVALID, "ROI %d is not inside the image", r);
  }
  return IFE_OK;
}

// Stage a host array on the device (or pass a device pointer through).
template <typename T>
int stage_in(ife_cuda_ctx* ctx, DeviceBuffer& buf, const T* src, size_t count, int mem,
             const T** dev) {
  if (!src) { *dev = nullptr; return IFE_OK; }
  if (mem == IFE_MEM_DEVICE) { *dev = src; return IFE_OK; }
  IFE_TRY(buf.reserve(ctx, count * sizeof(T)));
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(buf.ptr, src, count * sizeof(T), cudaMemcpyHostToDevice,
                                    ctx->stream()));
  *dev = (const T*)buf.ptr;
  return IFE_OK;
}

// Where the kernels write an output of `count` elements: with IFE_MEM_HOST the workspace buffer
// `buf`, which finish_out copies to the caller's `dst`; else `dst` itself.
template <typename T>
int stage_out(ife_cuda_ctx* ctx, DeviceBuffer& buf, T* dst, size_t count, int mem, T** dev) {
  *dev = dst;
  if (mem != IFE_MEM_HOST) return IFE_OK;
  IFE_TRY(buf.reserve(ctx, count * sizeof(T)));
  *dev = (T*)buf.ptr;
  return IFE_OK;
}

// With IFE_MEM_HOST: copy a staged output back on the context's stream and wait for it.
template <typename T>
int finish_out(ife_cuda_ctx* ctx, T* dst, const T* dev, size_t count, int mem) {
  if (mem != IFE_MEM_HOST) return IFE_OK;
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(dst, dev, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream()));
  IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream()));
  return IFE_OK;
}

// int16 -> float on the device (exact).  Option "host_image_i16": the HOST image pointers of the
// ife_cuda_emphysema_* calls point to int16 voxels -- CT's type on disk, which the reference's tools
// widen to float on the host while reading (tools/ExtractFeatures.cxx:90-96) -- so a scan's upload
// is 2 bytes per voxel instead of 4.
__global__ void widen_i16_kernel(const short* __restrict__ in, float* __restrict__ out, size_t n) {
  const size_t i4 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 + 3 < n) {
    const short4 v = *reinterpret_cast<const short4*>(in + i4);
    *reinterpret_cast<float4*>(out + i4) = make_float4((float)v.x, (float)v.y, (float)v.z, (float)v.w);
  } else {
    for (size_t i = i4; i < n; ++i) out[i] = (float)in[i];
  }
}

// upload + widen on stream `st` into `dst` (n floats), through `tmp` (n int16)
int upload_image_i16(ife_cuda_ctx* ctx, const void* host_i16, void* tmp, float* dst, size_t n, cudaStream_t st) {
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(tmp, host_i16, n * sizeof(short), cudaMemcpyHostToDevice, st));
  const unsigned grid = (unsigned)((n / 4 + 256) / 256);
  widen_i16_kernel<<<grid, 256, 0, st>>>((const short*)tmp, dst, n);
  ctx->launches++;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  return IFE_OK;
}

// the image of an ife_cuda_emphysema_* call: float, or int16 on the host with option "host_image_i16"
int stage_image(ife_cuda_ctx* ctx, const float* image, size_t n, int mem, const float** dev) {
  if (mem == IFE_MEM_DEVICE || !ctx->host_image_i16) return stage_in(ctx, ctx->ws.in_img, image, n, mem, dev);
  IFE_TRY(ctx->ws.in_img.reserve(ctx, n * sizeof(float)));
  IFE_TRY(ctx->ws.in_i16.reserve(ctx, 2 * ((n + 3) & ~(size_t)3) * sizeof(short)));
  IFE_TRY(upload_image_i16(ctx, image, ctx->ws.in_i16.ptr, (float*)ctx->ws.in_img.ptr, n, ctx->stream()));
  *dev = (const float*)ctx->ws.in_img.ptr;
  return IFE_OK;
}

}  // namespace ife

using namespace ife;

// =======================================================================================
// C ABI
// =======================================================================================
extern "C" {

int ife_cuda_abi_version(void) { return IFE_CUDA_ABI_VERSION; }

int ife_cuda_create(int device, ife_cuda_ctx** out) {
  if (!out) return IFE_E_INVALID;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) return IFE_E_CUDA;
  ife_cuda_ctx* ctx = new ife_cuda_ctx();
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return IFE_E_CUDA;
  }
  cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
  for (auto& ev : ctx->events) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  for (auto& ev : ctx->ov_events) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  {
    int least = 0, greatest = 0;
    cudaDeviceGetStreamPriorityRange(&least, &greatest);
    cudaStreamCreateWithPriority(&ctx->hp_stream, cudaStreamNonBlocking, greatest);
  }
  *out = ctx;
  return IFE_OK;
}

void ife_cuda_destroy(ife_cuda_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  ife_cuda_comm_destroy(ctx);
  ctx->ws.release_all();
  if (ctx->box_host) cudaFreeHost(ctx->box_host);
  for (auto& ev : ctx->events) if (ev) cudaEventDestroy(ev);
  for (auto& ev : ctx->ov_events) if (ev) cudaEventDestroy(ev);
  if (ctx->hp_stream) cudaStreamDestroy(ctx->hp_stream);
  for (auto& ev : ctx->prof_events) cudaEventDestroy(ev);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
}

const char* ife_cuda_last_error(const ife_cuda_ctx* ctx) {
  return ctx ? ctx->error.c_str() : "null context";
}

// Page-locked host memory.  cudaHostAlloc costs 0.48 s per GB on the B200 boxes (the driver faults
// and zeroes 4 KB pages on one core): 6 s for the 13.4 GB of feature volumes one ExtractFeatures run
// holds, against 0.3 s of GPU work.  Large blocks are therefore mapped anonymously with transparent huge
// pages, faulted in by all cores, and registered with the driver: 0.043 s per GB, the same 57 GB/s of
// D2H rate (profiles/micro/pin_alloc.cu).  Anything that fails falls back to cudaHostAlloc.
namespace {
struct MappedBlock { void* base; size_t len; };
std::mutex g_mapped_mu;
std::map<void*, MappedBlock> g_mapped;   // user pointer -> mapping
constexpr size_t kHugePage = (size_t)2 << 20;

void* host_alloc_mapped(size_t bytes) {
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {   // nothing to register with
    cudaGetLastError();
    return nullptr;
  }
  const auto t_begin = std::chrono::steady_clock::now();
  const size_t len = (bytes + 2 * kHugePage - 1) / kHugePage * kHugePage;   // room to align the start to 2 MB
  void* base = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
  if (base == MAP_FAILED) return nullptr;
  char* p = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(base) + kHugePage - 1) / kHugePage * kHugePage);
  madvise(p, bytes, MADV_HUGEPAGE);   // advisory: without it the touch below just faults 4 KB pages
  int n_threads = (int)std::thread::hardware_concurrency();
  n_threads = std::max(1, std::min(n_threads, std::min(32, (int)(bytes / (64u << 20)) + 1)));
  const size_t per = (bytes / n_threads + 4095) / 4096 * 4096;
  std::vector<std::thread> pool;
  for (int t = 0; t < n_threads; ++t)
    pool.emplace_back([=] {
      const size_t a = (size_t)t * per, b = std::min(bytes, a + per);
      for (size_t i = a; i < b; i += 4096) reinterpret_cast<volatile char*>(p)[i] = 0;
    });
  for (auto& t : pool) t.join();
  const auto t_touch = std::chrono::steady_clock::now();
  const cudaError_t reg = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
  if (std::getenv("IFE_ALLOC_TRACE"))
    std::fprintf(stderr, "[ife] host_alloc %zu MB: map + touch (%d threads) %.3f s, register %.3f s (%s)\n", bytes >> 20, n_threads,
                 std::chrono::duration<double>(t_touch - t_begin).count(),
                 std::chrono::duration<double>(std::chrono::steady_clock::now() - t_touch).count(), cudaGetErrorString(reg));
  if (reg != cudaSuccess) {
    cudaGetLastError();
    munmap(base, len);
    return nullptr;
  }
  std::lock_guard<std::mutex> lk(g_mapped_mu);
  g_mapped[p] = MappedBlock{base, len};
  return p;
}
}  // namespace

int ife_cuda_host_alloc(size_t bytes, void** ptr) {
  if (!ptr) return IFE_E_INVALID;
  *ptr = nullptr;
  if (bytes == 0) return IFE_OK;
  if (bytes >= ((size_t)32 << 20) && !std::getenv("IFE_NO_MAPPED_HOST_ALLOC")) {
    *ptr = host_alloc_mapped(bytes);
    if (*ptr) return IFE_OK;
  }
  if (cudaHostAlloc(ptr, bytes, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();   // not sticky: the caller falls back to pageable memory
    *ptr = nullptr;
    return IFE_E_CUDA;
  }
  return IFE_OK;
}

void ife_cuda_host_free(void* ptr) {
  if (!ptr) return;
  MappedBlock blk{nullptr, 0};
  {
    std::lock_guard<std::mutex> lk(g_mapped_mu);
    auto it = g_mapped.find(ptr);
    if (it != g_mapped.end()) { blk = it->second; g_mapped.erase(it); }
  }
  if (blk.base) {
    cudaHostUnregister(ptr);
    munmap(blk.base, blk.len);
  } else {
    cudaFreeHost(ptr);
  }
}

int ife_cuda_set_stream(ife_cuda_ctx* ctx, void* s) {
  if (!ctx) return IFE_E_INVALID;
  ctx->user_stream = (cudaStream_t)s;
  ctx->use_user_stream = s != nullptr;
  return IFE_OK;
}

int ife_cuda_set_arith(ife_cuda_ctx* ctx, int mode) {
  if (!ctx) return IFE_E_INVALID;
  if (mode != IFE_ARITH_PLAIN && mode != IFE_ARITH_FMA)
    return fail(ctx, IFE_E_INVALID, "unknown arithmetic mode %d", mode);
  ctx->arith = mode;
  return IFE_OK;
}

int ife_cuda_get_arith(const ife_cuda_ctx* ctx) { return ctx ? ctx->arith : IFE_E_INVALID; }

int ife_cuda_synchronize(ife_cuda_ctx* ctx) {
  if (!ctx) return IFE_E_INVALID;
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream()));
  IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
  return IFE_OK;
}

uint64_t ife_cuda_launch_count(const ife_cuda_ctx* ctx) { return ctx ? ctx->launches : 0; }

int ife_cuda_last_work_dims(const ife_cuda_ctx* ctx, int dims[3]) {
  if (!ctx || !dims) return IFE_E_INVALID;
  for (int d = 0; d < 3; ++d) dims[d] = ctx->work_dims[d];
  return IFE_OK;
}

int ife_cuda_set_option(ife_cuda_ctx* ctx, const char* name, int value) {
  if (!ctx || !name) return IFE_E_INVALID;
  if (std::strcmp(name, "tma_passes") == 0) { ctx->use_tma = value != 0; return IFE_OK; }
  if (std::strcmp(name, "march4") == 0) { ctx->use_march4 = value != 0; return IFE_OK; }
  if (std::strcmp(name, "host_image_i16") == 0) { ctx->host_image_i16 = value != 0; return IFE_OK; }
  if (std::strcmp(name, "support_box") == 0) { ctx->use_box = value != 0; return IFE_OK; }
  if (std::strcmp(name, "overlap_scales") == 0) { ctx->overlap_scales = value != 0; return IFE_OK; }
  return fail(ctx, IFE_E_INVALID, "unknown option '%s'", name);
}

int ife_cuda_profile_enable(ife_cuda_ctx* ctx, int on) {
  if (!ctx) return IFE_E_INVALID;
  ctx->profiling = on != 0;
  ctx->prof_used = 0;
  ctx->prof_kinds.clear();
  return IFE_OK;
}

int ife_cuda_profile_read(ife_cuda_ctx* ctx, double ms[IFE_PROFILE_KINDS],
                          uint64_t launches[IFE_PROFILE_KINDS]) {
  if (!ctx || !ms || !launches) return IFE_E_INVALID;
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream()));
  for (int k = 0; k < IFE_PROFILE_KINDS; ++k) { ms[k] = 0.0; launches[k] = 0; }
  for (size_t i = 0; i < ctx->prof_kinds.size(); ++i) {
    float t = 0.f;
    IFE_CUDA_TRY(ctx, cudaEventElapsedTime(&t, ctx->prof_events[2 * i], ctx->prof_events[2 * i + 1]));
    ms[ctx->prof_kinds[i]] += t;
    launches[ctx->prof_kinds[i]]++;
  }
  ctx->prof_used = 0;
  ctx->prof_kinds.clear();
  return IFE_OK;
}

int ife_cuda_reserve(ife_cuda_ctx* ctx, const int dims[3], int n_outputs) {
  if (!ctx || !dims) return IFE_E_INVALID;
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  IFE_TRY(reserve_smoothing(ctx, 2, dims[0], dims[1], dims[2]));
  IFE_TRY(ctx->ws.blur.reserve(ctx, n * sizeof(float)));
  if (n_outputs > 0) {
    IFE_TRY(ctx->ws.in_img.reserve(ctx, n * sizeof(float)));
    IFE_TRY(ctx->ws.in_mask.reserve(ctx, n * sizeof(float)));
    IFE_TRY(ctx->ws.out[0].reserve(ctx, n * sizeof(float) * n_outputs));
    if (n_outputs >= 8) IFE_TRY(ctx->ws.out[1].reserve(ctx, n * sizeof(float) * n_outputs));
  }
  return IFE_OK;
}

int ife_cuda_gaussian(ife_cuda_ctx* ctx, const float* in, float* out, const int dims[3],
                      const double spacing[3], double sigma, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!in || !out) return fail(ctx, IFE_E_INVALID, "null image pointer");
  IFE_TRY(check_dims(ctx, dims, spacing));
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  IFE_TRY(reserve_smoothing(ctx, 1, dims[0], dims[1], dims[2]));
  const float* d_in;
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, in, n, mem, &d_in));
  float* d_out;
  IFE_TRY(stage_out(ctx, ctx->ws.out[0], out, n, mem, &d_out));
  IFE_TRY(smooth_volume(ctx, d_in, nullptr, false, d_out, dims[0], dims[1], dims[2], 0, dims[2], spacing,
                        sigma, nullptr, nullptr));
  return finish_out(ctx, out, d_out, n, mem);
}

int ife_cuda_normalized_gaussian(ife_cuda_ctx* ctx, const float* image, const float* cert_f32,
                                 const uint8_t* cert_u8, float* out, const int dims[3],
                                 const double spacing[3], double sigma, int mask_output, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!image || !out) return fail(ctx, IFE_E_INVALID, "null image pointer");
  if ((cert_f32 == nullptr) == (cert_u8 == nullptr))
    return fail(ctx, IFE_E_INVALID, "exactly one of certainty_f32 / certainty_u8 must be given");
  IFE_TRY(check_dims(ctx, dims, spacing));
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  IFE_TRY(reserve_smoothing(ctx, 2, dims[0], dims[1], dims[2]));
  const float* d_img;
  const float* d_cf = nullptr;
  const uint8_t* d_cu = nullptr;
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, image, n, mem, &d_img));
  if (cert_f32) IFE_TRY(stage_in(ctx, ctx->ws.in_mask, cert_f32, n, mem, &d_cf));
  else IFE_TRY(stage_in(ctx, ctx->ws.in_mask, cert_u8, n, mem, &d_cu));
  float* d_out;
  IFE_TRY(stage_out(ctx, ctx->ws.out[0], out, n, mem, &d_out));
  const void* cert = cert_f32 ? (const void*)d_cf : (const void*)d_cu;
  IFE_TRY(smooth_volume(ctx, d_img, cert, cert_u8 != nullptr, d_out, dims[0], dims[1], dims[2],
                        0, dims[2], spacing, sigma, mask_output ? d_cu : nullptr,
                        mask_output ? d_cf : nullptr));
  return finish_out(ctx, out, d_out, n, mem);
}

int ife_cuda_gradient_magnitude(ife_cuda_ctx* ctx, const float* in, const float* mask_f32,
                                const uint8_t* mask_u8, float* out, const int dims[3],
                                const double spacing[3], int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!in || !out) return fail(ctx, IFE_E_INVALID, "null image pointer");
  IFE_TRY(check_dims(ctx, dims, spacing));
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  const float* d_in;
  const float* d_mf = nullptr;
  const uint8_t* d_mu = nullptr;
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, in, n, mem, &d_in));
  if (mask_f32) IFE_TRY(stage_in(ctx, ctx->ws.in_mask, mask_f32, n, mem, &d_mf));
  else if (mask_u8) IFE_TRY(stage_in(ctx, ctx->ws.in_mask, mask_u8, n, mem, &d_mu));
  float* d_out;
  IFE_TRY(stage_out(ctx, ctx->ws.out[0], out, n, mem, &d_out));
  FeatArgs A;
  std::memset(&A, 0, sizeof(A));
  A.vol = d_in; A.mask_u8 = d_mu; A.mask_f32 = d_mf; A.out[0] = d_out;
  A.nx = dims[0]; A.ny = dims[1]; A.nzb = dims[2]; A.zb0 = 0; A.zb1 = dims[2];
  IFE_TRY(launch_features(ctx, 2, make_stencil_coef(spacing), A, is_unit_spacing(spacing)));
  return finish_out(ctx, out, d_out, n, mem);
}

int ife_cuda_hessian_eigen_features(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                    float* out6, const int dims[3], const double spacing[3],
                                    double sigma, int flags, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!image || !out6) return fail(ctx, IFE_E_INVALID, "null image pointer");
  IFE_TRY(check_dims(ctx, dims, spacing));
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  const float* d_img;
  const uint8_t* d_mask;
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, image, n, mem, &d_img));
  IFE_TRY(stage_in(ctx, ctx->ws.in_mask, mask, n, mem, &d_mask));
  const float* src = d_img;
  if (sigma > 0.0) {
    IFE_TRY(reserve_smoothing(ctx, 1, dims[0], dims[1], dims[2]));
    IFE_TRY(ctx->ws.blur.reserve(ctx, n * sizeof(float)));
    IFE_TRY(smooth_volume(ctx, d_img, nullptr, false, (float*)ctx->ws.blur.ptr, dims[0], dims[1],
                          dims[2], 0, dims[2], spacing, sigma, nullptr, nullptr));
    src = (const float*)ctx->ws.blur.ptr;
  }
  float* d_out;
  IFE_TRY(stage_out(ctx, ctx->ws.out[0], out6, 6 * n, mem, &d_out));
  FeatArgs A;
  std::memset(&A, 0, sizeof(A));
  A.vol = src; A.mask_u8 = d_mask;
  for (int k = 0; k < 6; ++k) A.out[k] = d_out + (size_t)k * n;
  A.nx = dims[0]; A.ny = dims[1]; A.nzb = dims[2]; A.zb0 = 0; A.zb1 = dims[2];
  A.dy_bug = (flags & IFE_FDHF_TOOL_DY_BUG) ? 1 : 0;
  IFE_TRY(launch_features(ctx, 1, make_stencil_coef(spacing), A, is_unit_spacing(spacing)));
  return finish_out(ctx, out6, d_out, 6 * n, mem);
}

int ife_cuda_hessian(ife_cuda_ctx* ctx, const float* image, float* out6, const int dims[3],
                     const double spacing[3], int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!image || !out6) return fail(ctx, IFE_E_INVALID, "null image pointer");
  IFE_TRY(check_dims(ctx, dims, spacing));
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  const float* d_img;
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, image, n, mem, &d_img));
  float* d_out;
  IFE_TRY(stage_out(ctx, ctx->ws.out[0], out6, 6 * n, mem, &d_out));
  FeatArgs A;
  std::memset(&A, 0, sizeof(A));
  A.vol = d_img;
  for (int k = 0; k < 6; ++k) A.out[k] = d_out + (size_t)k * n;
  A.nx = dims[0]; A.ny = dims[1]; A.nzb = dims[2]; A.zb0 = 0; A.zb1 = dims[2];
  IFE_TRY(launch_features(ctx, 3, make_stencil_coef(spacing), A, is_unit_spacing(spacing)));
  return finish_out(ctx, out6, d_out, 6 * n, mem);
}

int ife_cuda_emphysema_features(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                float* out, const int dims[3], const double spacing[3],
                                const double* sigmas, int n_sigma, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!image || !mask || !out) return fail(ctx, IFE_E_INVALID, "null image/mask/out pointer");
  if (!sigmas || n_sigma <= 0) return fail(ctx, IFE_E_INVALID, "need at least one scale");
  IFE_TRY(check_dims(ctx, dims, spacing));
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int nx = dims[0], ny = dims[1], nz = dims[2];
  const size_t n = (size_t)nx * ny * nz;
  IFE_TRY(reserve_smoothing(ctx, 2, nx, ny, nz));
  IFE_TRY(ctx->ws.blur.reserve(ctx, n * sizeof(float)));
  const float* d_img;
  const uint8_t* d_mask;
  IFE_TRY(stage_image(ctx, image, n, mem, &d_img));
  IFE_TRY(stage_in(ctx, ctx->ws.in_mask, mask, n, mem, &d_mask));
  if (mem == IFE_MEM_HOST) {
    // two staging buffers so that the D2H copy of scale s overlaps the kernels of scale s+1
    IFE_TRY(ctx->ws.out[0].reserve(ctx, 8 * n * sizeof(float)));
    if (n_sigma > 1) IFE_TRY(ctx->ws.out[1].reserve(ctx, 8 * n * sizeof(float)));
  }
  const StencilCoef S = make_stencil_coef(spacing);
  MaskedPlan plan;    // all eight outputs are masked: smooth only what in-mask voxels can see
  IFE_TRY(plan_masked(ctx, d_img, d_mask, nx, ny, nz, nullptr, 0, &plan));
  // Option "overlap_scales" (device-resident calls with several scales): the Gaussian passes run
  // on the context's high-priority stream one scale ahead of the fused feature kernel, which
  // stays on the main stream and fills the issue slots the FP64-latency-bound passes leave
  // idle; two blur buffers, events ov_events[1+b] (blur b written) / [3+b] (blur b consumed).
  const bool overlap = ctx->overlap_scales && mem == IFE_MEM_DEVICE && n_sigma > 1 && ctx->hp_stream;
  if (overlap) {
    IFE_TRY(ctx->ws.blur2.reserve(ctx, n * sizeof(float)));
    IFE_CUDA_TRY(ctx, cudaEventRecord(ctx->ov_events[0], ctx->main_stream()));
    IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->hp_stream, ctx->ov_events[0], 0));
  }
  for (int s = 0; s < n_sigma; ++s) {
    float* blur = (float*)(overlap && (s & 1) ? ctx->ws.blur2.ptr : ctx->ws.blur.ptr);
    float* d_out = mem == IFE_MEM_HOST ? (float*)ctx->ws.out[s & 1].ptr : out + (size_t)s * 8 * n;
    if (mem == IFE_MEM_HOST && s >= 2)  // the staging buffer must have been drained
      IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream(), ctx->events[2 + (s & 1)], 0));
    if (overlap) {
      if (s >= 2) IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->hp_stream, ctx->ov_events[3 + (s & 1)], 0));
      ctx->alt_stream = ctx->hp_stream;
    }
    const int rc_smooth = smooth_masked(ctx, plan, d_img, d_mask, blur, nx, ny, nz, spacing, sigmas[s]);
    ctx->alt_stream = nullptr;
    IFE_TRY(rc_smooth);
    if (overlap) {
      IFE_CUDA_TRY(ctx, cudaEventRecord(ctx->ov_events[1 + (s & 1)], ctx->hp_stream));
      IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->main_stream(), ctx->ov_events[1 + (s & 1)], 0));
    }
    FeatArgs A;
    std::memset(&A, 0, sizeof(A));
    A.vol = blur; A.mask_u8 = d_mask;
    for (int k = 0; k < 8; ++k) A.out[k] = d_out + (size_t)k * n;
    A.nx = nx; A.ny = ny; A.nzb = nz; A.zb0 = 0; A.zb1 = nz;
    IFE_TRY(launch_features(ctx, 0, S, A, is_unit_spacing(spacing)));
    if (overlap) IFE_CUDA_TRY(ctx, cudaEventRecord(ctx->ov_events[3 + (s & 1)], ctx->main_stream()));
    if (mem == IFE_MEM_HOST) {
      IFE_CUDA_TRY(ctx, cudaEventRecord(ctx->events[s & 1], ctx->stream()));
      IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->events[s & 1], 0));
      IFE_CUDA_TRY(ctx, cudaMemcpyAsync(out + (size_t)s * 8 * n, d_out, 8 * n * sizeof(float),
                                        cudaMemcpyDeviceToHost, ctx->copy_stream));
      IFE_CUDA_TRY(ctx, cudaEventRecord(ctx->events[2 + (s & 1)], ctx->copy_stream));
    }
  }
  if (mem == IFE_MEM_HOST) {
    IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
    IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream()));
  }
  return IFE_OK;
}

int ife_cuda_emphysema_histograms(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                  const int dims[3], const double spacing[3], const double* sigmas,
                                  int n_sigma, const float* edges, int n_edges, const int* rois,
                                  int n_roi, uint32_t* counts, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!image || !mask || !counts || !edges) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  if (!sigmas || n_sigma <= 0) return fail(ctx, IFE_E_INVALID, "need at least one scale");
  if (n_edges <= 0) return fail(ctx, IFE_E_INVALID, "need at least one histogram edge");
  if (n_roi < 0 || (n_roi > 0 && !rois)) return fail(ctx, IFE_E_INVALID, "bad ROI list");
  IFE_TRY(check_dims(ctx, dims, spacing));
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int nx = dims[0], ny = dims[1], nz = dims[2];
  const size_t n = (size_t)nx * ny * nz;
  IFE_TRY(check_rois(ctx, rois, n_roi, dims));
  IFE_TRY(reserve_smoothing(ctx, 2, nx, ny, nz));
  IFE_TRY(ctx->ws.blur.reserve(ctx, n * sizeof(float)));
  const float* d_img;
  const uint8_t* d_mask;
  IFE_TRY(stage_image(ctx, image, n, mem, &d_img));
  IFE_TRY(stage_in(ctx, ctx->ws.in_mask, mask, n, mem, &d_mask));

  const int rows = n_sigma * 8, R = std::max(n_roi, 1);
  const size_t n_counts = (size_t)R * rows * (n_edges + 1);
  // parameter arrays are host pointers; counts follows `mem`
  IFE_TRY(ctx->ws.edges.reserve(ctx, (size_t)rows * n_edges * sizeof(float)));
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws.edges.ptr, edges, (size_t)rows * n_edges * sizeof(float),
                                    cudaMemcpyHostToDevice, ctx->stream()));
  int* d_rois = nullptr;
  if (n_roi > 0) {   // uploaded below, once the crop frame is known
    IFE_TRY(ctx->ws.rois.reserve(ctx, (size_t)n_roi * 6 * sizeof(int)));
    d_rois = (int*)ctx->ws.rois.ptr;
  }
  uint32_t* d_counts;
  IFE_TRY(stage_out(ctx, ctx->ws.counts, counts, n_counts, mem, &d_counts));
  IFE_CUDA_TRY(ctx, cudaMemsetAsync(d_counts, 0, n_counts * sizeof(uint32_t), ctx->stream()));
  MaskedPlan plan;    // only in-mask voxels (inside some ROI, when there are ROIs) are binned
  IFE_TRY(plan_masked(ctx, d_img, d_mask, nx, ny, nz, rois, n_roi, &plan));
  {
    std::vector<int> moved;
    IFE_TRY(upload_rois(ctx, plan, rois, n_roi, d_rois, &moved));
    if (!moved.empty()) IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream()));   // `moved` is about to go
  }
  IFE_TRY(bin_masked_scan(ctx, plan, d_img, d_mask, nx, ny, nz, spacing, sigmas, n_sigma,
                          (const float*)ctx->ws.edges.ptr, n_edges, d_rois, n_roi, d_counts));
  return finish_out(ctx, counts, d_counts, n_counts, mem);
}

int ife_cuda_emphysema_histograms_batch(ife_cuda_ctx* ctx, int n_scans, const float* const* images,
                                        const uint8_t* const* masks, const int dims[3],
                                        const double spacing[3], const double* sigmas, int n_sigma,
                                        const float* edges, int n_edges, const int* rois, int n_roi,
                                        uint32_t* counts) {
  if (!ctx) return IFE_E_INVALID;
  if (n_scans <= 0) return IFE_OK;
  if (!images || !masks || !counts || !edges) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  if (!sigmas || n_sigma <= 0) return fail(ctx, IFE_E_INVALID, "need at least one scale");
  if (n_edges <= 0) return fail(ctx, IFE_E_INVALID, "need at least one histogram edge");
  if (n_roi < 0 || (n_roi > 0 && !rois)) return fail(ctx, IFE_E_INVALID, "bad ROI list");
  IFE_TRY(check_dims(ctx, dims, spacing));
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int nx = dims[0], ny = dims[1], nz = dims[2];
  const size_t n = (size_t)nx * ny * nz;
  for (int i = 0; i < n_scans; ++i) {
    if (!images[i] || !masks[i]) return fail(ctx, IFE_E_INVALID, "scan %d: null image or mask", i);
    if (check_rois(ctx, rois + (size_t)i * n_roi * 6, n_roi, dims) != IFE_OK)
      return fail(ctx, IFE_E_INVALID, "scan %d: %s", i, ctx->error.c_str());
  }
  Workspace& ws = ctx->ws;
  IFE_TRY(reserve_smoothing(ctx, 2, nx, ny, nz));
  IFE_TRY(ws.blur.reserve(ctx, n * sizeof(float)));
  // two upload slots: the H2D copy of scan i+1 (copy stream) runs behind the kernels of scan i
  DeviceBuffer* img_slot[2] = {&ws.in_img, &ws.out[0]};
  DeviceBuffer* mask_slot[2] = {&ws.in_mask, &ws.out[1]};
  for (int k = 0; k < 2; ++k) {
    IFE_TRY(img_slot[k]->reserve(ctx, n * sizeof(float)));
    IFE_TRY(mask_slot[k]->reserve(ctx, n));
  }
  if (ctx->host_image_i16) IFE_TRY(ws.in_i16.reserve(ctx, 2 * ((n + 3) & ~(size_t)3) * sizeof(short)));
  const int rows = n_sigma * 8, R = std::max(n_roi, 1);
  const size_t n_counts = (size_t)R * rows * (n_edges + 1);
  IFE_TRY(ws.edges.reserve(ctx, (size_t)rows * n_edges * sizeof(float)));
  IFE_TRY(ws.counts.reserve(ctx, 2 * n_counts * sizeof(uint32_t)));
  int* d_rois = nullptr;   // each scan's list, uploaded on the context's stream right before its kernels
  if (n_roi > 0) {
    IFE_TRY(ws.rois.reserve(ctx, (size_t)n_roi * 6 * sizeof(int)));
    d_rois = (int*)ws.rois.ptr;
  }
  cudaStream_t st = ctx->stream(), cp = ctx->copy_stream;
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ws.edges.ptr, edges, (size_t)rows * n_edges * sizeof(float),
                                    cudaMemcpyHostToDevice, st));
  const bool use_box = support_box_usable(ctx, (const uint8_t*)mask_slot[0]->ptr, nx, ny, nz) &&
                       support_box_usable(ctx, (const uint8_t*)mask_slot[1]->ptr, nx, ny, nz);
  // events[0..1]: upload of slot k done; events[2..3]: kernels reading slot k done
  auto upload = [&](int i) -> int {
    const int k = i & 1;
    if (i >= 2) IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(cp, ctx->events[2 + k], 0));
    if (ctx->host_image_i16)
      IFE_TRY(upload_image_i16(ctx, images[i], (short*)ws.in_i16.ptr + (size_t)k * ((n + 3) & ~(size_t)3), (float*)img_slot[k]->ptr, n, cp));
    else
      IFE_CUDA_TRY(ctx, cudaMemcpyAsync(img_slot[k]->ptr, images[i], n * sizeof(float), cudaMemcpyHostToDevice, cp));
    IFE_CUDA_TRY(ctx, cudaMemcpyAsync(mask_slot[k]->ptr, masks[i], n, cudaMemcpyHostToDevice, cp));
    // the mask's support box is reduced right behind its upload, so the host never has to
    // wait for the kernels of the scan before
    if (use_box) IFE_TRY(launch_support_box(ctx, (const uint8_t*)mask_slot[k]->ptr, nx, ny, nz, cp, k));
    IFE_CUDA_TRY(ctx, cudaEventRecord(ctx->events[k], cp));
    return IFE_OK;
  };
  IFE_TRY(upload(0));
  std::vector<std::vector<int>> moved((size_t)n_scans);   // alive until the copies have run
  for (int i = 0; i < n_scans; ++i) {
    const int k = i & 1;
    if (i + 1 < n_scans) IFE_TRY(upload(i + 1));
    IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->events[k], 0));
    const float* d_img = (const float*)img_slot[k]->ptr;
    const uint8_t* d_mask = (const uint8_t*)mask_slot[k]->ptr;
    uint32_t* d_counts = (uint32_t*)ws.counts.ptr + (size_t)k * n_counts;
    IFE_CUDA_TRY(ctx, cudaMemsetAsync(d_counts, 0, n_counts * sizeof(uint32_t), st));
    if (use_box) IFE_CUDA_TRY(ctx, cudaEventSynchronize(ctx->events[k]));   // upload i and its box are in
    MaskedPlan plan;
    const int* scan_rois = n_roi > 0 ? rois + (size_t)i * n_roi * 6 : nullptr;
    IFE_TRY(plan_masked(ctx, use_box, k, d_img, d_mask, nx, ny, nz, scan_rois, n_roi, &plan));
    IFE_TRY(upload_rois(ctx, plan, scan_rois, n_roi, d_rois, &moved[i]));
    IFE_TRY(bin_masked_scan(ctx, plan, d_img, d_mask, nx, ny, nz, spacing, sigmas, n_sigma,
                            (const float*)ws.edges.ptr, n_edges, d_rois, n_roi, d_counts));
    IFE_CUDA_TRY(ctx, cudaEventRecord(ctx->events[2 + k], st));
    IFE_CUDA_TRY(ctx, cudaMemcpyAsync(counts + (size_t)i * n_counts, d_counts, n_counts * sizeof(uint32_t),
                                      cudaMemcpyDeviceToHost, st));
  }
  IFE_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  IFE_CUDA_TRY(ctx, cudaStreamSynchronize(cp));
  return IFE_OK;
}

int ife_cuda_histogram(ife_cuda_ctx* ctx, const float* values, size_t n, const float* edges,
                       int n_edges, uint32_t* counts, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!edges || !counts || (n > 0 && !values)) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  if (n_edges <= 0) return fail(ctx, IFE_E_INVALID, "need at least one histogram edge");
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t smem = n_edges * sizeof(float) + (n_edges + 1) * sizeof(uint32_t);
  if (smem > 48 * 1024) return fail(ctx, IFE_E_INVALID, "too many histogram edges (%d)", n_edges);
  const float* d_vals = nullptr;
  if (n > 0) IFE_TRY(stage_in(ctx, ctx->ws.in_img, values, n, mem, &d_vals));
  IFE_TRY(ctx->ws.edges.reserve(ctx, n_edges * sizeof(float)));
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws.edges.ptr, edges, n_edges * sizeof(float),
                                    cudaMemcpyHostToDevice, ctx->stream()));
  uint32_t* d_counts;
  IFE_TRY(stage_out(ctx, ctx->ws.counts, counts, n_edges + 1, mem, &d_counts));
  IFE_CUDA_TRY(ctx, cudaMemsetAsync(d_counts, 0, (n_edges + 1) * sizeof(uint32_t), ctx->stream()));
  if (n > 0) {
    const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx->sm_count * 16);
    histogram_kernel<<<grid, 256, smem, ctx->stream()>>>(d_vals, n, (const float*)ctx->ws.edges.ptr,
                                                         n_edges, d_counts);
    ctx->launches++;
    IFE_CUDA_TRY(ctx, cudaGetLastError());
  }
  return finish_out(ctx, counts, d_counts, n_edges + 1, mem);
}

int ife_cuda_intensity_roi_histograms(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                      const int dims[3], const float* edges, int n_edges,
                                      const int* rois, int n_roi, uint32_t* counts, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!image || !mask || !edges || !counts) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  if (n_edges <= 0) return fail(ctx, IFE_E_INVALID, "need at least one histogram edge");
  if (n_roi < 0 || (n_roi > 0 && !rois)) return fail(ctx, IFE_E_INVALID, "bad ROI list");
  const double unit[3] = {1.0, 1.0, 1.0};
  IFE_TRY(check_dims(ctx, dims, unit));
  if (n_roi == 0) return IFE_OK;
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int nx = dims[0], ny = dims[1], nz = dims[2];
  const size_t n = (size_t)nx * ny * nz;
  IFE_TRY(check_rois(ctx, rois, n_roi, dims));
  const size_t smem = n_edges * sizeof(float) + (n_edges + 1) * sizeof(uint32_t);
  if (smem > 48 * 1024) return fail(ctx, IFE_E_INVALID, "too many histogram edges (%d)", n_edges);
  const float* d_img;
  const uint8_t* d_mask;
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, image, n, mem, &d_img));
  IFE_TRY(stage_in(ctx, ctx->ws.in_mask, mask, n, mem, &d_mask));
  IFE_TRY(ctx->ws.edges.reserve(ctx, n_edges * sizeof(float)));
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws.edges.ptr, edges, n_edges * sizeof(float),
                                    cudaMemcpyHostToDevice, ctx->stream()));
  IFE_TRY(ctx->ws.rois.reserve(ctx, (size_t)n_roi * 6 * sizeof(int)));
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws.rois.ptr, rois, (size_t)n_roi * 6 * sizeof(int),
                                    cudaMemcpyHostToDevice, ctx->stream()));
  const size_t n_counts = (size_t)n_roi * (n_edges + 1);
  uint32_t* d_counts;
  IFE_TRY(stage_out(ctx, ctx->ws.counts, counts, n_counts, mem, &d_counts));
  {
    ProfScope prof(ctx, K_OTHER);
    roi_intensity_hist_kernel<<<(unsigned)n_roi, 256, smem, ctx->stream()>>>(
        d_img, d_mask, nx, ny, (const int*)ctx->ws.rois.ptr, (const float*)ctx->ws.edges.ptr, n_edges, d_counts);
    ctx->launches++;
    IFE_CUDA_TRY(ctx, cudaGetLastError());
  }
  return finish_out(ctx, counts, d_counts, n_counts, mem);
}

int ife_cuda_resample(ife_cuda_ctx* ctx, const void* in, void* out, int elem_bytes, const int dims[3],
                      const double spacing[3], const double out_spacing[3], int interp, double default_value,
                      int out_dims[3], int mem) {
  if (!ctx && out) return IFE_E_INVALID;   // a size query needs no context (nor a device)
  if (!in || !out_dims || !out_spacing) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  if (interp != IFE_INTERP_LINEAR && interp != IFE_INTERP_NEAREST)
    return fail(ctx, IFE_E_INVALID, "unknown interpolator %d", interp);
  if (elem_bytes != 4 && elem_bytes != 1) return fail(ctx, IFE_E_INVALID, "elem_bytes must be 4 (float) or 1 (uint8)");
  if (interp == IFE_INTERP_LINEAR && elem_bytes != 4)
    return fail(ctx, IFE_E_INVALID, "linear interpolation takes float voxels only");
  if (elem_bytes == 1 && !(default_value >= 0.0 && default_value <= 255.0 && default_value == std::floor(default_value)))
    return fail(ctx, IFE_E_INVALID, "default value %g is not a uint8 value", default_value);
  IFE_TRY(check_dims(ctx, dims, spacing));
  int m[3];
  for (int d = 0; d < 3; ++d) {
    if (!std::isfinite(spacing[d])) return fail(ctx, IFE_E_INVALID, "spacing[%d] is not finite", d);
    if (!(out_spacing[d] > 0.0) || !std::isfinite(out_spacing[d]))
      return fail(ctx, IFE_E_INVALID, "out_spacing[%d] = %g must be positive and finite", d, out_spacing[d]);
    // n' = max(1, floor(n * s / s' + 0.5)), in double
    const double want = std::floor((double)dims[d] * spacing[d] / out_spacing[d] + 0.5);
    if (!(want <= 2147483647.0)) return fail(ctx, IFE_E_INVALID, "output axis %d would have %g voxels", d, want);
    m[d] = std::max(1, (int)want);
  }
  const size_t n_in = (size_t)dims[0] * dims[1] * dims[2], n_out = (size_t)m[0] * m[1] * m[2];
  if (m[1] > 65535 * kRsBY || m[2] > 65535) return fail(ctx, IFE_E_INVALID, "output grid %d x %d x %d is too large", m[0], m[1], m[2]);
  for (int d = 0; d < 3; ++d) out_dims[d] = m[d];
  if (!out) return IFE_OK;
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const uint8_t* d_in;
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, static_cast<const uint8_t*>(in), n_in * elem_bytes, mem, &d_in));
  uint8_t* d_out;
  IFE_TRY(stage_out(ctx, ctx->ws.out[0], static_cast<uint8_t*>(out), n_out * elem_bytes, mem, &d_out));
  ResampleArgs A;
  std::memset(&A, 0, sizeof(A));
  A.in = d_in;
  A.out = d_out;
  for (int d = 0; d < 3; ++d) {
    A.n[d] = dims[d];
    A.m[d] = m[d];
    A.so[d] = out_spacing[d];
    A.inv[d] = 1.0 / spacing[d];
    A.ident[d] = out_spacing[d] == spacing[d];
  }
  A.def_f32 = (float)default_value;
  A.def_u8 = elem_bytes == 1 ? (uint8_t)default_value : 0;
  const int mode = interp == IFE_INTERP_LINEAR ? RS_LINEAR : elem_bytes == 4 ? RS_NEAREST_F32 : RS_NEAREST_U8;
  const bool vec = m[0] % kRsV == 0 && reinterpret_cast<uintptr_t>(d_out) % (kRsV * elem_bytes) == 0;
  const dim3 block(kRsBX, kRsBY), grid((unsigned)((m[0] + kRsBX * kRsV - 1) / (kRsBX * kRsV)),
                                       (unsigned)((m[1] + kRsBY - 1) / kRsBY), (unsigned)m[2]);
  {
    ProfScope prof(ctx, K_OTHER);
    cudaStream_t st = ctx->stream();
    switch (mode * 2 + (vec ? 1 : 0)) {
      case 0: resample_kernel<RS_LINEAR, false><<<grid, block, 0, st>>>(A); break;
      case 1: resample_kernel<RS_LINEAR, true><<<grid, block, 0, st>>>(A); break;
      case 2: resample_kernel<RS_NEAREST_F32, false><<<grid, block, 0, st>>>(A); break;
      case 3: resample_kernel<RS_NEAREST_F32, true><<<grid, block, 0, st>>>(A); break;
      case 4: resample_kernel<RS_NEAREST_U8, false><<<grid, block, 0, st>>>(A); break;
      default: resample_kernel<RS_NEAREST_U8, true><<<grid, block, 0, st>>>(A); break;
    }
    ctx->launches++;
    IFE_CUDA_TRY(ctx, cudaGetLastError());
  }
  return finish_out(ctx, static_cast<uint8_t*>(out), d_out, n_out * elem_bytes, mem);
}

// The three passes of a signed distance map (csrc/distance_map.cuh) on the context's stream.  With
// A.partial set the z pass sums the weighted map into per-block partials instead of writing it.
static int signed_distance_passes(ife_cuda_ctx* ctx, SdmArgs& A) {
  const size_t n = (size_t)A.nx * A.ny * A.nz;
  IFE_TRY(ctx->ws.a0.reserve(ctx, n * sizeof(int16_t)));
  IFE_TRY(ctx->ws.a1.reserve(ctx, n * sizeof(uint32_t)));
  IFE_TRY(ctx->ws.b0.reserve(ctx, n * sizeof(unsigned long long)));
  A.gx = (int16_t*)ctx->ws.a0.ptr;
  A.gxy = (uint32_t*)ctx->ws.a1.ptr;
  A.stack = ctx->ws.b0.ptr;
  cudaStream_t st = ctx->stream();
  const unsigned rows = (unsigned)(((size_t)A.ny * A.nz + kSdmRowsPerBlock - 1) / kSdmRowsPerBlock);
  const unsigned lines_y = (unsigned)(((size_t)A.nx * A.nz + kSdmLineThreads - 1) / kSdmLineThreads);
  const unsigned lines_z = (unsigned)(((size_t)A.nx * A.ny + kSdmLineThreads - 1) / kSdmLineThreads);
  {
    ProfScope prof(ctx, K_OTHER);
    sdm_pass_x<<<rows, 32 * kSdmRowsPerBlock, 0, st>>>(A);
  }
  {
    ProfScope prof(ctx, K_OTHER);
    sdm_pass_line<false, false><<<lines_y, kSdmLineThreads, 0, st>>>(A);
  }
  {
    ProfScope prof(ctx, K_OTHER);
    if (A.partial) sdm_pass_line<true, true><<<lines_z, kSdmLineThreads, 0, st>>>(A);
    else sdm_pass_line<true, false><<<lines_z, kSdmLineThreads, 0, st>>>(A);
  }
  ctx->launches += 3;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  return IFE_OK;
}

// Arguments shared by the two distance entry points.
static int check_distance_args(ife_cuda_ctx* ctx, const int dims[3], const double spacing[3], int flags, int allowed) {
  if (flags & ~allowed) return fail(ctx, IFE_E_INVALID, "unknown flag bits 0x%x", flags & ~allowed);
  IFE_TRY(check_dims(ctx, dims, spacing));
  for (int d = 0; d < 3; ++d) {
    if (!std::isfinite(spacing[d])) return fail(ctx, IFE_E_INVALID, "spacing[%d] is not finite", d);
    if (dims[d] > kSdmMaxAxis)
      return fail(ctx, IFE_E_INVALID, "dims[%d] = %d: a distance map takes axes of up to %d voxels", d, dims[d], kSdmMaxAxis);
  }
  return IFE_OK;
}

static SdmArgs distance_args(const int dims[3], const double spacing[3], const uint8_t* d_mask, int flags) {
  SdmArgs A;
  std::memset(&A, 0, sizeof(A));
  A.nx = dims[0];
  A.ny = dims[1];
  A.nz = dims[2];
  for (int d = 0; d < 3; ++d) A.s[d] = spacing[d];
  A.mask = d_mask;
  A.inside_positive = (flags & IFE_SDM_INSIDE_POSITIVE) != 0;
  A.squared = (flags & IFE_SDM_SQUARED) != 0;
  return A;
}

int ife_cuda_signed_distance_map(ife_cuda_ctx* ctx, const uint8_t* mask, float* out, const int dims[3],
                                 const double spacing[3], int flags, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!mask || !out) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  IFE_TRY(check_distance_args(ctx, dims, spacing, flags, IFE_SDM_INSIDE_POSITIVE | IFE_SDM_SQUARED));
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const uint8_t* d_mask;
  IFE_TRY(stage_in(ctx, ctx->ws.in_mask, mask, n, mem, &d_mask));
  float* d_out;
  IFE_TRY(stage_out(ctx, ctx->ws.out[0], out, n, mem, &d_out));
  SdmArgs A = distance_args(dims, spacing, d_mask, flags);
  A.out = d_out;
  IFE_TRY(signed_distance_passes(ctx, A));
  return finish_out(ctx, out, d_out, n, mem);
}

int ife_cuda_expected_signed_distance(ife_cuda_ctx* ctx, const uint8_t* center, const float* weight,
                                      const uint8_t* region, const int dims[3], const double spacing[3],
                                      int flags, double* result, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!center || !weight || !result) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  IFE_TRY(check_distance_args(ctx, dims, spacing, flags, IFE_SDM_INSIDE_POSITIVE));
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const uint8_t *d_center, *d_region;
  const float* d_weight;
  IFE_TRY(stage_in(ctx, ctx->ws.in_mask, center, n, mem, &d_center));
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, weight, n, mem, &d_weight));
  IFE_TRY(stage_in(ctx, ctx->ws.out[0], region, n, mem, &d_region));   // this call writes no volume
  SdmArgs A = distance_args(dims, spacing, d_center, flags);
  A.weight = d_weight;
  A.region = d_region;
  // the z pass's per-block partials and their sum go where the x pass's output was
  const int n_blocks = (int)(((size_t)dims[0] * dims[1] + kSdmLineThreads - 1) / kSdmLineThreads);
  IFE_TRY(ctx->ws.a0.reserve(ctx, std::max(n * sizeof(int16_t), (n_blocks + 1) * sizeof(SdmPartial))));
  SdmPartial* partial = (SdmPartial*)ctx->ws.a0.ptr;
  A.partial = partial;
  IFE_TRY(signed_distance_passes(ctx, A));
  if (!ctx->box_host)
    IFE_CUDA_TRY(ctx, cudaHostAlloc((void**)&ctx->box_host, 12 * sizeof(int), cudaHostAllocDefault));
  static_assert(sizeof(SdmPartial) <= 12 * sizeof(int), "the sums come back through box_host");
  cudaStream_t st = ctx->stream();
  {
    ProfScope prof(ctx, K_OTHER);
    sdm_reduce_partials<<<1, kSdmReduceThreads, 0, st>>>(partial, n_blocks, partial + n_blocks);
    ctx->launches++;
    IFE_CUDA_TRY(ctx, cudaGetLastError());
  }
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->box_host, partial + n_blocks, sizeof(SdmPartial), cudaMemcpyDeviceToHost, st));
  IFE_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  SdmPartial S;
  std::memcpy(&S, ctx->box_host, sizeof(S));
  if (S.no_site) return fail(ctx, IFE_E_INVALID, "the center mask has no contour voxel");
  if (S.bad_weight) return fail(ctx, IFE_E_INVALID, "%d weights are negative or not finite", S.bad_weight);
  if (!(S.sw > 0.0)) return fail(ctx, IFE_E_INVALID, "the weights sum to %g", S.sw);
  *result = S.swd / S.sw;
  return IFE_OK;
}

// In-place device sort of n floats at d_data (csrc/radix_sort.cuh): 8 passes of count / scan / scatter
// between d_data and a scratch buffer; after an even number of passes the result is back in d_data.
static int radix_sort_device(ife_cuda_ctx* ctx, float* d_data, size_t n) {
  const unsigned n_tiles = (unsigned)((n + kRsTile - 1) / kRsTile);
  IFE_TRY(ctx->ws.out[1].reserve(ctx, n * sizeof(uint32_t)));
  IFE_TRY(ctx->ws.counts.reserve(ctx, (size_t)kRsBins * n_tiles * sizeof(uint32_t)));
  uint32_t* a = reinterpret_cast<uint32_t*>(d_data);
  uint32_t* b = (uint32_t*)ctx->ws.out[1].ptr;
  uint32_t* cnt = (uint32_t*)ctx->ws.counts.ptr;
  cudaStream_t st = ctx->stream();
  const unsigned g = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx->sm_count * 16);
  rs_to_keys_kernel<<<g, 256, 0, st>>>(a, n);
  for (int pass = 0; pass < 8; ++pass) {
    rs_count_kernel<<<n_tiles, kRsThreads, 0, st>>>(a, n, 4 * pass, cnt, n_tiles);
    rs_scan_kernel<<<1, 1024, 0, st>>>(cnt, (size_t)kRsBins * n_tiles);
    rs_scatter_kernel<<<n_tiles, kRsThreads, 0, st>>>(a, b, n, 4 * pass, cnt, n_tiles);
    std::swap(a, b);
  }
  rs_from_keys_kernel<<<g, 256, 0, st>>>(a, n);   // a == d_data again
  ctx->launches += 26;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  return IFE_OK;
}

int ife_cuda_sort_f32(ife_cuda_ctx* ctx, float* data, size_t n, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (n == 0) return IFE_OK;
  if (!data) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  if (n > (size_t)0x7fffffff) return fail(ctx, IFE_E_INVALID, "too many samples for one sort (%zu)", n);
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const float* d_in_c;
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, (const float*)data, n, mem, &d_in_c));
  float* d_in = const_cast<float*>(d_in_c);
  IFE_TRY(radix_sort_device(ctx, d_in, n));
  return finish_out(ctx, data, d_in, n, mem);
}

// The compaction sink of the bin-edge determination: features on the device, only the sampled
// voxels' values leave it.
int ife_cuda_emphysema_feature_samples(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                       const uint8_t* select, const long long* index, size_t n_index,
                                       const int dims[3], const double spacing[3], const double* sigmas,
                                       int n_sigma, int sorted, float* out, size_t* n_out, int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (!image || !mask || !sigmas || n_sigma <= 0 || !n_out) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  if ((select != nullptr) == (index != nullptr)) return fail(ctx, IFE_E_INVALID, "give either a selection mask or an index list");
  IFE_TRY(check_dims(ctx, dims, spacing));
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int nx = dims[0], ny = dims[1], nz = dims[2];
  const size_t n = (size_t)nx * ny * nz;
  cudaStream_t st = ctx->stream();
  const float* d_img;
  const uint8_t* d_mask;
  IFE_TRY(stage_image(ctx, image, n, mem, &d_img));
  IFE_TRY(stage_in(ctx, ctx->ws.in_mask, mask, n, mem, &d_mask));
  // which voxels: selection flags -> per-tile counts -> offsets (host prefix over a few thousand
  // integers); or an explicit index list
  const unsigned n_tiles = (unsigned)((n + kCsTile - 1) / kCsTile);
  const uint8_t* d_sel = nullptr;
  const long long* d_idx = nullptr;
  size_t n_sel = n_index;
  if (select) {
    if (mem == IFE_MEM_HOST) {
      IFE_TRY(ctx->ws.slab_mask.reserve(ctx, n));
      IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws.slab_mask.ptr, select, n, cudaMemcpyHostToDevice, st));
      d_sel = (const uint8_t*)ctx->ws.slab_mask.ptr;
    } else {
      d_sel = select;
    }
    IFE_TRY(ctx->ws.counts.reserve(ctx, (size_t)n_tiles * sizeof(uint32_t)));
    IFE_TRY(ctx->ws.rois.reserve(ctx, (size_t)n_tiles * sizeof(uint64_t)));
    cs_count_kernel<<<n_tiles, kCsThreads, 0, st>>>(d_sel, n, (uint32_t*)ctx->ws.counts.ptr);
    ctx->launches++;
    std::vector<uint32_t> cnt(n_tiles);
    IFE_CUDA_TRY(ctx, cudaMemcpyAsync(cnt.data(), ctx->ws.counts.ptr, (size_t)n_tiles * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    IFE_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    std::vector<uint64_t> off(n_tiles);
    uint64_t run = 0;
    for (unsigned t = 0; t < n_tiles; ++t) { off[t] = run; run += cnt[t]; }
    n_sel = (size_t)run;
    IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws.rois.ptr, off.data(), (size_t)n_tiles * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    IFE_CUDA_TRY(ctx, cudaStreamSynchronize(st));   // `off` leaves scope
  } else {
    for (size_t j = 0; j < n_index && mem == IFE_MEM_HOST; ++j)
      if (index[j] < 0 || (size_t)index[j] >= n) return fail(ctx, IFE_E_INVALID, "sample index %zu out of range", j);
    if (mem == IFE_MEM_HOST) {
      IFE_TRY(ctx->ws.rois.reserve(ctx, std::max<size_t>(n_index, 1) * sizeof(long long)));
      IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws.rois.ptr, index, n_index * sizeof(long long), cudaMemcpyHostToDevice, st));
      d_idx = (const long long*)ctx->ws.rois.ptr;
    } else {
      d_idx = index;
    }
  }
  *n_out = n_sel;
  if (n_sel == 0 || !out) return IFE_OK;   // out == null: the caller only asked how many
  if (n_sel > (size_t)0x7fffffff) return fail(ctx, IFE_E_INVALID, "too many samples (%zu)", n_sel);

  IFE_TRY(reserve_smoothing(ctx, 2, nx, ny, nz));
  IFE_TRY(ctx->ws.blur.reserve(ctx, n * sizeof(float)));
  IFE_TRY(ctx->ws.out[0].reserve(ctx, 8 * n * sizeof(float)));
  MaskedPlan plan;
  IFE_TRY(plan_masked(ctx, d_img, d_mask, nx, ny, nz, nullptr, 0, &plan));
  const size_t rows_bytes = (size_t)8 * n_sel * sizeof(float);
  float* d_rows = out;
  if (mem == IFE_MEM_HOST) {
    IFE_TRY(ctx->ws.packed.reserve(ctx, rows_bytes));
    d_rows = (float*)ctx->ws.packed.ptr;
  }
  float* blur = (float*)ctx->ws.blur.ptr;
  float* feats = (float*)ctx->ws.out[0].ptr;
  const StencilCoef S = make_stencil_coef(spacing);
  for (int s = 0; s < n_sigma; ++s) {
    IFE_TRY(smooth_masked(ctx, plan, d_img, d_mask, blur, nx, ny, nz, spacing, sigmas[s]));
    FeatArgs A;
    std::memset(&A, 0, sizeof(A));
    A.vol = blur; A.mask_u8 = d_mask;
    for (int k = 0; k < 8; ++k) A.out[k] = feats + (size_t)k * n;
    A.nx = nx; A.ny = ny; A.nzb = nz; A.zb0 = 0; A.zb1 = nz;
    IFE_TRY(launch_features(ctx, 0, S, A, is_unit_spacing(spacing)));
    float* rows = mem == IFE_MEM_HOST ? d_rows : out + (size_t)s * 8 * n_sel;
    if (d_sel) {
      cs_gather_kernel<<<n_tiles, kCsThreads, 0, st>>>(d_sel, n, (const uint64_t*)ctx->ws.rois.ptr, feats, n, 8, rows, n_sel);
    } else {
      const unsigned g = (unsigned)std::min<size_t>((n_sel + 255) / 256, (size_t)ctx->sm_count * 16);
      cs_gather_index_kernel<<<g, 256, 0, st>>>(d_idx, n_sel, feats, n, 8, rows, n_sel);
    }
    ctx->launches++;
    IFE_CUDA_TRY(ctx, cudaGetLastError());
    if (sorted)
      for (int k = 0; k < 8; ++k) IFE_TRY(radix_sort_device(ctx, rows + (size_t)k * n_sel, n_sel));
    if (mem == IFE_MEM_HOST) {
      IFE_CUDA_TRY(ctx, cudaMemcpyAsync(out + (size_t)s * 8 * n_sel, rows, rows_bytes, cudaMemcpyDeviceToHost, st));
      IFE_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
  }
  return IFE_OK;
}

int ife_cuda_eigen_features_batch(ife_cuda_ctx* ctx, const float* A6, float* out6, size_t n,
                                  int mem) {
  if (!ctx) return IFE_E_INVALID;
  if (n == 0) return IFE_OK;
  if (!A6 || !out6) return fail(ctx, IFE_E_INVALID, "null pointer argument");
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const float* d_in;
  IFE_TRY(stage_in(ctx, ctx->ws.in_img, A6, 6 * n, mem, &d_in));
  float* d_out;
  IFE_TRY(stage_out(ctx, ctx->ws.out[0], out6, 6 * n, mem, &d_out));
  eigen_features_batch_lean_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream()>>>(d_in, d_out, n);
  ctx->launches++;
  IFE_CUDA_TRY(ctx, cudaGetLastError());
  return finish_out(ctx, out6, d_out, 6 * n, mem);
}

}  // extern "C"

#include "slab.cuh"
