// Recursive (IIR) Gaussian line passes for sm_100a.
//
// Replaces itk::RecursiveGaussianImageFilter as cascaded by
// itk::SmoothingRecursiveGaussianImageFilter, which is what the reference smooths with
// (include/ife/Filters/NormalizedGaussianConvolutionImageFilter.h:72, .hxx:51-55).  The
// filter is a 4th-order Deriche recursion: out = causal(x) + anticausal(x), each a
// 4-tap feed-forward plus 4-tap feedback recurrence run in double along one image axis,
// the result stored as float.  To be bit-identical with the CPU path the recurrence is
// evaluated in the same association and (per context) either with separately rounded
// multiplies/adds or with the fused chain a -mfma build of the same source produces.
//
// GPU formulation.  One thread owns one line.  The anticausal half needs the line's
// future, so a line is swept twice:
//   phase A  forward over the whole line, causal recurrence only; every L samples the
//            four feedback values are saved as a checkpoint (32 B per field per chunk);
//   phase B  backward over chunks of L samples: reload the chunk, replay the causal
//            recurrence from its checkpoint into registers, run the anticausal
//            recurrence backward through the chunk (its state carried from the chunk
//            after), emit float(causal + anticausal).
// Nothing but the input (twice), the output (once) and the checkpoints touches HBM; no
// full-precision intermediate volume exists.  Lines along y and z are strided in memory
// with x across the threads of a warp, so every load/store is a 128-byte coalesced row
// (gauss_pass_strided).  Lines along x are contiguous; there a warp owns 32 adjacent
// lines and moves [32 lines] x [L samples] tiles through shared memory so that global
// traffic stays coalesced while each lane walks its own line (gauss_pass_x).
//
// The multiply of normalized convolution (c*T) is fused into the loads of the first pass
// and its divide (G(cT)/G(c), with ITK's zero-divisor rule) into the stores of the last.
#pragma once
#include <cfloat>
#include <cstdint>
#include <cuda_runtime.h>

#include "fdiv.cuh"

namespace ife {

// N0..N3 feed-forward (causal), D1..D4 feedback, M1..M4 feed-forward (anticausal),
// BN/BM boundary feedback coefficients (edge value extended to infinity).
struct GaussCoef {
  double N[4], D[4], M[4], BN[4], BM[4];
};

enum InMode { IN_FIELDS = 0, IN_IMG_U8 = 1, IN_IMG_F32 = 2 };

template <bool FMA>
__device__ __forceinline__ double dot4(double a0, double c0, double a1, double c1, double a2,
                                       double c2, double a3, double c3) {
  if (FMA) {
    double t = __dmul_rn(a0, c0);
    t = __fma_rn(a1, c1, t);
    t = __fma_rn(a2, c2, t);
    t = __fma_rn(a3, c3, t);
    return t;
  } else {
    double t = __dadd_rn(__dmul_rn(a0, c0), __dmul_rn(a1, c1));
    t = __dadd_rn(t, __dmul_rn(a2, c2));
    t = __dadd_rn(t, __dmul_rn(a3, c3));
    return t;
  }
}

// State of one direction of the recurrence for one field: h[k] = output k+1 samples
// behind (causal) / ahead (anticausal); x[k] likewise for the input.
struct Rec {
  double h0, h1, h2, h3;
  double x0, x1, x2, x3;  // causal uses x0..x2 (x[i-1..i-3]); anticausal x0..x3 (x[p+1..p+4])
};

// Feedback coefficients in use: D1..D4 in the interior, BN/BM for taps that still refer to
// the virtual constant extension beyond the line end.
struct Fb {
  double c0, c1, c2, c3;
};

__device__ __forceinline__ Fb fb_select(const double (&D)[4], const double (&B)[4], int done) {
  Fb f;
  f.c0 = done >= 1 ? D[0] : B[0];
  f.c1 = done >= 2 ? D[1] : B[1];
  f.c2 = done >= 3 ? D[2] : B[2];
  f.c3 = done >= 4 ? D[3] : B[3];
  return f;
}

template <bool FMA>
__device__ __forceinline__ double causal_step(const GaussCoef& C, const Fb& fb, Rec& s, double xi) {
  const double n = dot4<FMA>(xi, C.N[0], s.x0, C.N[1], s.x1, C.N[2], s.x2, C.N[3]);
  const double d = dot4<FMA>(s.h0, fb.c0, s.h1, fb.c1, s.h2, fb.c2, s.h3, fb.c3);
  const double y = __dsub_rn(n, d);
  s.x2 = s.x1; s.x1 = s.x0; s.x0 = xi;
  s.h3 = s.h2; s.h2 = s.h1; s.h1 = s.h0; s.h0 = y;
  return y;
}

// anticausal output at position p from x[p+1..p+4], w[p+1..p+4]; then x[p] is shifted in
template <bool FMA>
__device__ __forceinline__ double anti_step(const GaussCoef& C, const Fb& fb, Rec& s, double xp) {
  const double n = dot4<FMA>(s.x0, C.M[0], s.x1, C.M[1], s.x2, C.M[2], s.x3, C.M[3]);
  const double d = dot4<FMA>(s.h0, fb.c0, s.h1, fb.c1, s.h2, fb.c2, s.h3, fb.c3);
  const double w = __dsub_rn(n, d);
  s.x3 = s.x2; s.x2 = s.x1; s.x1 = s.x0; s.x0 = xp;
  s.h3 = s.h2; s.h2 = s.h1; s.h1 = s.h0; s.h0 = w;
  return w;
}

__device__ __forceinline__ void rec_fill(Rec& s, double v) {
  s.h0 = s.h1 = s.h2 = s.h3 = v;
  s.x0 = s.x1 = s.x2 = s.x3 = v;
}

// Checkpoints: ckpt[((chunk-1)*NF + f)*4 + k][line] doubles, line fastest (coalesced).
template <int NF>
__device__ __forceinline__ size_t ckpt_index(int chunk, int f, int k, size_t n_lines, size_t line) {
  return ((size_t)((chunk - 1) * NF + f) * 4 + k) * n_lines + line;
}

// ---------------------------------------------------------------------------------------
// Chunk processing, generic over where the samples come from (SRC: void(int j, double(&)[NF]))
// and where the results go (SINK: void(int j, const float(&)[NF])).
//
// forward_chunk  : phase A, advance the causal recurrence over one chunk.
// backward_chunk : phase B, replay causal from `cs` (state at i0) into registers, then run
//                  the anticausal recurrence backward from `as` (state at i0+len) and emit
//                  float(causal + anticausal).
// GENERIC = false is the hot path: a full chunk (len == L) strictly inside the line, no
// predicates and constant feedback coefficients, so the fully unrolled body is nothing but
// the recurrence.  GENERIC = true handles the first chunk (boundary coefficients), the
// last chunk(s) and partial chunks.
// ---------------------------------------------------------------------------------------
template <int NF, int L, bool FMA, bool GENERIC, int UNROLL = L, typename SRC>
__device__ __forceinline__ void forward_chunk(const GaussCoef& C, const SRC& src, int i0, int len,
                                              Rec (&cs)[NF]) {
  Fb fb = fb_select(C.D, C.BN, 4);
#pragma unroll UNROLL
  for (int j = 0; j < L; ++j) {
    if (!GENERIC || j < len) {
      if (GENERIC) fb = fb_select(C.D, C.BN, i0 + j);
      double v[NF];
      src(j, v);
#pragma unroll
      for (int f = 0; f < NF; ++f) causal_step<FMA>(C, fb, cs[f], v[f]);
    }
  }
}

// Where the replayed causal values of a chunk wait for the anticausal sweep: registers
// (RegYB) here, a per-warp buffer in shared memory in the tensor-map kernels (iir_tma.cuh).
template <int NF, int L>
struct RegYB {
  double v[NF][L];
  __device__ __forceinline__ void set(int f, int j, double x) { v[f][j] = x; }
  __device__ __forceinline__ double get(int f, int j) const { return v[f][j]; }
};

template <int NF, int L, bool FMA, bool GENERIC, int UNROLL = L, typename SRC, typename SINK, typename YB>
__device__ __forceinline__ void backward_chunk(const GaussCoef& C, const SRC& src, const SINK& sink,
                                               int i0, int len, int n, Rec (&cs)[NF],
                                               Rec (&as)[NF], YB& yb) {
  if (!GENERIC) {
    // Hot path.  The causal replay (forward through the chunk, from the checkpoint) and the
    // anticausal recurrence (backward, from the state the chunk after left) are independent
    // until their sum, so they run in the same loop from opposite ends: 2*NF independent
    // dependency chains per thread instead of NF, which is what keeps the FP64 pipe busy at
    // the few warps per SM the recurrence's registers allow.  In the first half both
    // results are parked in yb (the slot of the other direction is still free); in the
    // second half each new value meets its parked partner and the sample is emitted.
    static_assert(L % 2 == 0, "chunk length must be even");
    const Fb fc = fb_select(C.D, C.BN, 4);
    const Fb fa = fb_select(C.D, C.BM, 4);
    constexpr int U2 = UNROLL >= L ? L / 2 : UNROLL;
#pragma unroll U2
    for (int t = 0; t < L / 2; ++t) {
      const int jc = t, ja = L - 1 - t;
      double vc[NF], va[NF];
      src(jc, vc);
      src(ja, va);
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        yb.set(f, jc, causal_step<FMA>(C, fc, cs[f], vc[f]));
        yb.set(f, ja, anti_step<FMA>(C, fa, as[f], va[f]));
      }
    }
#pragma unroll U2
    for (int t = L / 2; t < L; ++t) {
      const int jc = t, ja = L - 1 - t;
      double vc[NF], va[NF];
      src(jc, vc);
      src(ja, va);
      float oc[NF], oa[NF];
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        const double y = causal_step<FMA>(C, fc, cs[f], vc[f]);
        const double w = anti_step<FMA>(C, fa, as[f], va[f]);
        oc[f] = (float)__dadd_rn(y, yb.get(f, jc));      // parked anticausal value of jc
        oa[f] = (float)__dadd_rn(yb.get(f, ja), w);      // parked causal value of ja
      }
      sink(jc, oc);
      sink(ja, oa);
    }
    return;
  }
  {
    Fb fb = fb_select(C.D, C.BN, 4);
#pragma unroll UNROLL
    for (int j = 0; j < L; ++j) {
      if (!GENERIC || j < len) {
        if (GENERIC) fb = fb_select(C.D, C.BN, i0 + j);
        double v[NF];
        src(j, v);
#pragma unroll
        for (int f = 0; f < NF; ++f) yb.set(f, j, causal_step<FMA>(C, fb, cs[f], v[f]));
      }
    }
  }
  {
    Fb fb = fb_select(C.D, C.BM, 4);
#pragma unroll UNROLL
    for (int j = L - 1; j >= 0; --j) {
      if (!GENERIC || j < len) {
        if (GENERIC) fb = fb_select(C.D, C.BM, n - 1 - (i0 + j));
        double v[NF];
        src(j, v);
        float o[NF];
#pragma unroll
        for (int f = 0; f < NF; ++f) {
          const double w = anti_step<FMA>(C, fb, as[f], v[f]);
          o[f] = (float)__dadd_rn(yb.get(f, j), w);
        }
        sink(j, o);
      }
    }
  }
}

template <int NF, int L, bool FMA, bool GENERIC, typename SRC, typename SINK>
__device__ __forceinline__ void backward_chunk(const GaussCoef& C, const SRC& src, const SINK& sink,
                                               int i0, int len, int n, Rec (&cs)[NF],
                                               Rec (&as)[NF]) {
  RegYB<NF, L> yb;
  backward_chunk<NF, L, FMA, GENERIC, L>(C, src, sink, i0, len, n, cs, as, yb);
}

// anticausal recurrence only (no output): used above the wanted output range, where a
// z-slab's warm-up halo only has to deliver the recursion state at the slab's upper edge
template <int NF, int L, bool FMA, bool GENERIC, typename SRC>
__device__ __forceinline__ void anti_chunk(const GaussCoef& C, const SRC& src, int i0, int len, int n,
                                           Rec (&as)[NF]) {
  Fb fb = fb_select(C.D, C.BM, 4);
#pragma unroll
  for (int j = L - 1; j >= 0; --j) {
    if (!GENERIC || j < len) {
      if (GENERIC) fb = fb_select(C.D, C.BM, n - 1 - (i0 + j));
      double v[NF];
      src(j, v);
#pragma unroll
      for (int f = 0; f < NF; ++f) anti_step<FMA>(C, fb, as[f], v[f]);
    }
  }
}

// chunk [i0, i0+len) of a line of n samples can take the hot path
template <int L>
__device__ __forceinline__ bool chunk_is_interior(int i0, int len, int n) {
  return len == L && i0 >= 4 && i0 + len + 3 <= n - 1;
}

// register-array source / sink (samples of the chunk already in registers)
template <int NF, int L>
struct RegSrc {
  const float (&xs)[NF][L];
  __device__ __forceinline__ void operator()(int j, double (&v)[NF]) const {
#pragma unroll
    for (int f = 0; f < NF; ++f) v[f] = (double)xs[f][j];
  }
};
template <int NF, int L>
struct RegSink {
  float (&xs)[NF][L];
  __device__ __forceinline__ void operator()(int j, const float (&o)[NF]) const {
#pragma unroll
    for (int f = 0; f < NF; ++f) xs[f][j] = o[f];
  }
};

// itk::DivideImageFilter functor: b != 0 ? a/b : NumericTraits<float>::max()
__device__ __forceinline__ float itk_divide(float a, float b) {
  if (b == 0.0f) return FLT_MAX;
  // far from the mask both G(cT) and G(c) are tiny, down to denormals: scale both by 2^80
  // (exact, the quotient is unchanged), twice if need be, so that they too take the
  // branch-free division instead of the compiler's slow path
  float as = a, bs = b;
  if (fabsf(bs) < 0x1p-40f && fabsf(as) < 0x1p40f) { as *= 0x1p80f; bs *= 0x1p80f; }
  if (fabsf(bs) < 0x1p-40f && fabsf(as) < 0x1p40f) { as *= 0x1p80f; bs *= 0x1p80f; }
  const float mb = fabsf(bs);
  if (mb > 0x1p-40f && mb < 0x1p40f && div_safe_num(as)) return div_with_rcp(as, bs, __frcp_rn(bs));
  return __fdiv_rn(a, b);
}

struct PassArgs {
  const float* in0;     // field 0 (or the image T when INMODE != IN_FIELDS)
  const void* in1;      // field 1 (float), or certainty (uint8 / float) when INMODE != IN_FIELDS
  float* out0;
  float* out1;          // unused when DIVIDE or NF == 1
  const uint8_t* mask_u8;   // DIVIDE only: optional MaskImageFilter on the quotient
  const float* mask_f32;    //   "
  double* ckpt;
  int n;                // samples per line
  long long stride;    // element stride between consecutive samples of a line
  int na;               // lines are indexed l = a + na*b, base = a + b*sb  (strided pass)
  long long sb;
  long long n_lines;
};

template <int NF, int INMODE>
__device__ __forceinline__ void load_sample(const PassArgs& A, size_t idx, float (&v)[NF]) {
  if (INMODE == IN_FIELDS) {
    v[0] = __ldg(A.in0 + idx);
    if (NF == 2) v[NF - 1] = __ldg(reinterpret_cast<const float*>(A.in1) + idx);
  } else {
    const float t = __ldg(A.in0 + idx);
    float c;
    if (INMODE == IN_IMG_U8) c = (float)__ldg(reinterpret_cast<const uint8_t*>(A.in1) + idx);
    else c = __ldg(reinterpret_cast<const float*>(A.in1) + idx);
    v[0] = __fmul_rn(t, c);  // itk::MultiplyImageFilter (NormalizedGaussian...hxx:48-49)
    v[NF - 1] = c;
  }
}

// ---------------------------------------------------------------------------------------
// Lines strided in memory (y and z passes): thread <-> line, x across the warp.
// ---------------------------------------------------------------------------------------
template <int NF, int INMODE, bool DIVIDE, int L, bool FMA>
__global__ void __launch_bounds__(128)
gauss_pass_strided(const __grid_constant__ GaussCoef C, const __grid_constant__ PassArgs A) {
  const long long line = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (line >= A.n_lines) return;
  const size_t base = (size_t)(line % A.na) + (size_t)(line / A.na) * (size_t)A.sb;
  const size_t st = (size_t)A.stride;
  const int n = A.n;
  const int n_chunks = (n + L - 1) / L;

  float xs[NF][L];
  Rec cs[NF];

  // ---- phase A: causal sweep, checkpoint at every chunk start ----
  for (int k = 0; k < n_chunks; ++k) {
    const int i0 = k * L;
    const int len = min(L, n - i0);
#pragma unroll
    for (int j = 0; j < L; ++j) {
      if (j < len) {
        float v[NF];
        load_sample<NF, INMODE>(A, base + (size_t)(i0 + j) * st, v);
#pragma unroll
        for (int f = 0; f < NF; ++f) xs[f][j] = v[f];
      }
    }
    if (k == 0) {
#pragma unroll
      for (int f = 0; f < NF; ++f) rec_fill(cs[f], (double)xs[f][0]);
    } else {
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        A.ckpt[ckpt_index<NF>(k, f, 0, A.n_lines, line)] = cs[f].h0;
        A.ckpt[ckpt_index<NF>(k, f, 1, A.n_lines, line)] = cs[f].h1;
        A.ckpt[ckpt_index<NF>(k, f, 2, A.n_lines, line)] = cs[f].h2;
        A.ckpt[ckpt_index<NF>(k, f, 3, A.n_lines, line)] = cs[f].h3;
      }
    }
    {
      const RegSrc<NF, L> src{xs};
      if (len == L && i0 >= 4) forward_chunk<NF, L, FMA, false>(C, src, i0, len, cs);
      else forward_chunk<NF, L, FMA, true>(C, src, i0, len, cs);
    }
  }

  // ---- phase B: backward over chunks ----
  Rec as[NF];
  // the last chunk is still in xs; its last sample is the edge value
  {
    const int len_last = n - (n_chunks - 1) * L;
    float vlast[NF];
#pragma unroll
    for (int f = 0; f < NF; ++f) vlast[f] = xs[f][0];
#pragma unroll
    for (int j = 1; j < L; ++j)
      if (j < len_last) {
#pragma unroll
        for (int f = 0; f < NF; ++f) vlast[f] = xs[f][j];
      }
#pragma unroll
    for (int f = 0; f < NF; ++f) rec_fill(as[f], (double)vlast[f]);
  }
  for (int k = n_chunks - 1; k >= 0; --k) {
    const int i0 = k * L;
    const int len = min(L, n - i0);
    if (k != n_chunks - 1) {
#pragma unroll
      for (int j = 0; j < L; ++j) {
        float v[NF];
        load_sample<NF, INMODE>(A, base + (size_t)(i0 + j) * st, v);
#pragma unroll
        for (int f = 0; f < NF; ++f) xs[f][j] = v[f];
      }
    }
    if (k == 0) {
#pragma unroll
      for (int f = 0; f < NF; ++f) rec_fill(cs[f], (double)xs[f][0]);
    } else {
      float v1[NF], v2[NF], v3[NF];
      load_sample<NF, INMODE>(A, base + (size_t)(i0 - 1) * st, v1);
      load_sample<NF, INMODE>(A, base + (size_t)(i0 - 2) * st, v2);
      load_sample<NF, INMODE>(A, base + (size_t)(i0 - 3) * st, v3);
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        cs[f].h0 = A.ckpt[ckpt_index<NF>(k, f, 0, A.n_lines, line)];
        cs[f].h1 = A.ckpt[ckpt_index<NF>(k, f, 1, A.n_lines, line)];
        cs[f].h2 = A.ckpt[ckpt_index<NF>(k, f, 2, A.n_lines, line)];
        cs[f].h3 = A.ckpt[ckpt_index<NF>(k, f, 3, A.n_lines, line)];
        cs[f].x0 = (double)v1[f];
        cs[f].x1 = (double)v2[f];
        cs[f].x2 = (double)v3[f];
        cs[f].x3 = 0.0;
      }
    }
    {
      // the sink overwrites xs[.][j] only after the anticausal step has consumed it
      const RegSrc<NF, L> src{xs};
      const RegSink<NF, L> sink{xs};
      if (chunk_is_interior<L>(i0, len, n)) backward_chunk<NF, L, FMA, false>(C, src, sink, i0, len, n, cs, as);
      else backward_chunk<NF, L, FMA, true>(C, src, sink, i0, len, n, cs, as);
    }
#pragma unroll
    for (int j = 0; j < L; ++j) {
      if (j < len) {
        const size_t idx = base + (size_t)(i0 + j) * st;
        if (DIVIDE) {
          float q = itk_divide(xs[0][j], xs[NF - 1][j]);
          if (A.mask_u8) q = __ldg(A.mask_u8 + idx) != 0 ? q : 0.0f;
          if (A.mask_f32) q = __ldg(A.mask_f32 + idx) != 0.0f ? q : 0.0f;
          A.out0[idx] = q;
        } else {
          A.out0[idx] = xs[0][j];
          if (NF == 2) A.out1[idx] = xs[NF - 1][j];
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// Lines contiguous in memory (x pass): a warp owns 32 adjacent lines; [32 lines][L samples]
// tiles are staged through shared memory (row pitch 34 floats: conflict-free both for the
// coalesced side, lanes = 2 lines x 16 samples, and for the per-line side, lane = line).
// ---------------------------------------------------------------------------------------
constexpr int kTilePitch = 34;

template <int NF, int L>
struct XTile {
  float v[NF][L][kTilePitch];
};

template <int NF, int L>
__device__ __forceinline__ void xtile_load(const PassArgs& A, XTile<NF, L>& T, long long line0,
                                           int i0, int len, int lane, float (&xs)[NF][L]) {
  static_assert(L == 16, "tile mapping assumes 16 samples per chunk");
  const int j = lane & 15;
#pragma unroll
  for (int m = 0; m < 16; ++m) {
    const int ll = 2 * m + (lane >> 4);
    const long long gl = line0 + ll;
    if (gl < A.n_lines && j < len) {
      const size_t idx = (size_t)gl * (size_t)A.n + (size_t)(i0 + j);
      T.v[0][j][ll] = __ldg(A.in0 + idx);
      if (NF == 2) T.v[NF - 1][j][ll] = __ldg(reinterpret_cast<const float*>(A.in1) + idx);
    }
  }
  __syncwarp();
#pragma unroll
  for (int f = 0; f < NF; ++f)
#pragma unroll
    for (int jj = 0; jj < L; ++jj) xs[f][jj] = T.v[f][jj][lane];
  __syncwarp();
}

template <int NF, int L>
__device__ __forceinline__ void xtile_store(const PassArgs& A, XTile<NF, L>& T, long long line0,
                                            int i0, int len, int lane, const float (&xs)[NF][L]) {
#pragma unroll
  for (int f = 0; f < NF; ++f)
#pragma unroll
    for (int jj = 0; jj < L; ++jj) T.v[f][jj][lane] = xs[f][jj];
  __syncwarp();
  const int j = lane & 15;
#pragma unroll
  for (int m = 0; m < 16; ++m) {
    const int ll = 2 * m + (lane >> 4);
    const long long gl = line0 + ll;
    if (gl < A.n_lines && j < len) {
      const size_t idx = (size_t)gl * (size_t)A.n + (size_t)(i0 + j);
      A.out0[idx] = T.v[0][j][ll];
      if (NF == 2) A.out1[idx] = T.v[NF - 1][j][ll];
    }
  }
  __syncwarp();
}

template <int NF, int L, bool FMA, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
gauss_pass_x(const __grid_constant__ GaussCoef C, const __grid_constant__ PassArgs A) {
  __shared__ XTile<NF, L> tiles[WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long line0 = ((long long)blockIdx.x * WARPS + warp) * 32;
  if (line0 >= A.n_lines) return;
  XTile<NF, L>& T = tiles[warp];
  const long long line = line0 + lane;
  const bool active = line < A.n_lines;
  const long long cl = active ? line : A.n_lines - 1;  // inactive lanes shadow a valid line
  const int n = A.n;
  const int n_chunks = (n + L - 1) / L;

  float xs[NF][L];
  Rec cs[NF];

  for (int k = 0; k < n_chunks; ++k) {
    const int i0 = k * L;
    const int len = min(L, n - i0);
    xtile_load<NF, L>(A, T, line0, i0, len, lane, xs);
    if (k == 0) {
#pragma unroll
      for (int f = 0; f < NF; ++f) rec_fill(cs[f], (double)xs[f][0]);
    } else if (active) {
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        A.ckpt[ckpt_index<NF>(k, f, 0, A.n_lines, line)] = cs[f].h0;
        A.ckpt[ckpt_index<NF>(k, f, 1, A.n_lines, line)] = cs[f].h1;
        A.ckpt[ckpt_index<NF>(k, f, 2, A.n_lines, line)] = cs[f].h2;
        A.ckpt[ckpt_index<NF>(k, f, 3, A.n_lines, line)] = cs[f].h3;
      }
    }
    {
      const RegSrc<NF, L> src{xs};
      if (len == L && i0 >= 4) forward_chunk<NF, L, FMA, false>(C, src, i0, len, cs);
      else forward_chunk<NF, L, FMA, true>(C, src, i0, len, cs);
    }
  }

  Rec as[NF];
  {
    const int len_last = n - (n_chunks - 1) * L;
    float vlast[NF];
#pragma unroll
    for (int f = 0; f < NF; ++f) vlast[f] = xs[f][0];
#pragma unroll
    for (int j = 1; j < L; ++j)
      if (j < len_last) {
#pragma unroll
        for (int f = 0; f < NF; ++f) vlast[f] = xs[f][j];
      }
#pragma unroll
    for (int f = 0; f < NF; ++f) rec_fill(as[f], (double)vlast[f]);
  }
  for (int k = n_chunks - 1; k >= 0; --k) {
    const int i0 = k * L;
    const int len = min(L, n - i0);
    if (k != n_chunks - 1) xtile_load<NF, L>(A, T, line0, i0, len, lane, xs);
    if (k == 0) {
#pragma unroll
      for (int f = 0; f < NF; ++f) rec_fill(cs[f], (double)xs[f][0]);
    } else {
      const size_t hb = (size_t)cl * (size_t)n + (size_t)i0;
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        const float* src = f == 0 ? A.in0 : reinterpret_cast<const float*>(A.in1);
        cs[f].h0 = A.ckpt[ckpt_index<NF>(k, f, 0, A.n_lines, cl)];
        cs[f].h1 = A.ckpt[ckpt_index<NF>(k, f, 1, A.n_lines, cl)];
        cs[f].h2 = A.ckpt[ckpt_index<NF>(k, f, 2, A.n_lines, cl)];
        cs[f].h3 = A.ckpt[ckpt_index<NF>(k, f, 3, A.n_lines, cl)];
        cs[f].x0 = (double)__ldg(src + hb - 1);
        cs[f].x1 = (double)__ldg(src + hb - 2);
        cs[f].x2 = (double)__ldg(src + hb - 3);
        cs[f].x3 = 0.0;
      }
    }
    {
      // the sink overwrites xs[.][j] only after the anticausal step has consumed it
      const RegSrc<NF, L> src{xs};
      const RegSink<NF, L> sink{xs};
      if (chunk_is_interior<L>(i0, len, n)) backward_chunk<NF, L, FMA, false>(C, src, sink, i0, len, n, cs, as);
      else backward_chunk<NF, L, FMA, true>(C, src, sink, i0, len, n, cs, as);
    }
    xtile_store<NF, L>(A, T, line0, i0, len, lane, xs);
  }
}

}  // namespace ife
