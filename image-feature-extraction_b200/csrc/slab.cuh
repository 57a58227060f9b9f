// Multi-GPU z-slab path: halo exchange over NCCL send/recv, per-rank pipeline on
// slab+halo, histogram all-reduce.  Included by ife_cuda.cu (single translation unit).
//
// The reference has nothing distributed (single process, whole volume in host RAM,
// `UpdateLargestPossibleRegion()` everywhere: tools/ExtractFeatures.cxx:142); this is the
// B200 answer to volumes that want more than one GPU.  The volume is cut into contiguous
// z-slabs (z is the slowest index, so a slab is one contiguous block).  The only stage
// that couples planes beyond +-1 is the z pass of the recursive Gaussian, an IIR whose
// response to a wrong start state decays as exp(-1.37 d/sigma): each rank therefore
// receives H = ceil(halo_factor*sigma_max/spacing_z)+5 raw planes from its z neighbours
// ONCE per call (image 4 B/voxel + mask 1 B/voxel, grouped ncclSend/ncclRecv over
// NVLink), runs the z pass on slab+halo, and everything after it on slab+-1 planes.
// Global volume edges use the filter's own boundary rule, so a 1-rank run is identical to
// the single-GPU entry point.
//
// NCCL is bound lazily with dlopen so that single-GPU users need no NCCL at all.
#pragma once
#include <dlfcn.h>
#include <nccl.h>

namespace ife {

struct NcclApi {
  void* handle = nullptr;
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclSend) Send = nullptr;
  decltype(&ncclRecv) Recv = nullptr;
  decltype(&ncclAllReduce) AllReduce = nullptr;
  decltype(&ncclGroupStart) GroupStart = nullptr;
  decltype(&ncclGroupEnd) GroupEnd = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  bool ok = false;
};

inline NcclApi& nccl_api() {
  static NcclApi api;
  if (api.handle) return api;
  // a process that already loaded an NCCL (e.g. torch's bundled one) gets that one
  api.handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!api.handle) api.handle = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!api.handle) return api;
#define IFE_NCCL_SYM(name) api.name = (decltype(api.name))dlsym(api.handle, "nccl" #name)
  IFE_NCCL_SYM(GetUniqueId);
  IFE_NCCL_SYM(CommInitRank);
  IFE_NCCL_SYM(CommDestroy);
  IFE_NCCL_SYM(Send);
  IFE_NCCL_SYM(Recv);
  IFE_NCCL_SYM(AllReduce);
  IFE_NCCL_SYM(GroupStart);
  IFE_NCCL_SYM(GroupEnd);
  IFE_NCCL_SYM(GetErrorString);
#undef IFE_NCCL_SYM
  api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.Send && api.Recv &&
           api.AllReduce && api.GroupStart && api.GroupEnd && api.GetErrorString;
  return api;
}

#define IFE_NCCL_TRY(ctx, expr)                                                           \
  do {                                                                                    \
    ncclResult_t r_ = (expr);                                                             \
    if (r_ != ncclSuccess)                                                                \
      return ife::fail(ctx, IFE_E_COMM, "%s failed: %s", #expr, nccl_api().GetErrorString(r_)); \
  } while (0)

inline void slab_range(int nz, int n_ranks, int rank, int* z0, int* z1) {
  *z0 = (int)((long long)nz * rank / n_ranks);
  *z1 = (int)((long long)nz * (rank + 1) / n_ranks);
}

}  // namespace ife

extern "C" {

int ife_cuda_comm_unique_id(ife_cuda_ctx* ctx, uint8_t id[IFE_COMM_ID_BYTES]) {
  if (!ctx || !id) return IFE_E_INVALID;
  ife::NcclApi& api = ife::nccl_api();
  if (!api.ok) return ife::fail(ctx, IFE_E_COMM, "libnccl.so.2 could not be loaded");
  static_assert(sizeof(ncclUniqueId) == IFE_COMM_ID_BYTES, "NCCL unique id size");
  ncclUniqueId uid;
  IFE_NCCL_TRY(ctx, api.GetUniqueId(&uid));
  std::memcpy(id, &uid, sizeof(uid));
  return IFE_OK;
}

int ife_cuda_comm_init(ife_cuda_ctx* ctx, const uint8_t id[IFE_COMM_ID_BYTES], int n_ranks,
                       int rank) {
  if (!ctx || !id) return IFE_E_INVALID;
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks)
    return ife::fail(ctx, IFE_E_INVALID, "bad rank %d of %d", rank, n_ranks);
  ife::NcclApi& api = ife::nccl_api();
  if (!api.ok) return ife::fail(ctx, IFE_E_COMM, "libnccl.so.2 could not be loaded");
  if (ctx->nccl_comm) ife_cuda_comm_destroy(ctx);
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  ncclUniqueId uid;
  std::memcpy(&uid, id, sizeof(uid));
  ncclComm_t comm;
  IFE_NCCL_TRY(ctx, api.CommInitRank(&comm, n_ranks, uid, rank));
  ctx->nccl_comm = comm;
  ctx->n_ranks = n_ranks;
  ctx->rank = rank;
  return IFE_OK;
}

int ife_cuda_comm_destroy(ife_cuda_ctx* ctx) {
  if (!ctx) return IFE_E_INVALID;
  if (ctx->nccl_comm) {
    ife::nccl_api().CommDestroy((ncclComm_t)ctx->nccl_comm);
    ctx->nccl_comm = nullptr;
  }
  ctx->n_ranks = 1;
  ctx->rank = 0;
  return IFE_OK;
}

void ife_cuda_slab_range(int nz_global, int n_ranks, int rank, int* z0, int* z1) {
  ife::slab_range(nz_global, n_ranks, rank, z0, z1);
}

int ife_cuda_slab_halo(double sigma, double spacing_z, double halo_factor) {
  if (!(halo_factor > 0.0)) halo_factor = 12.0;
  return (int)std::ceil(halo_factor * sigma / spacing_z) + 4 + 1;
}

// Per-rank compute on a buffer that already holds the owned planes plus halo: device
// pointers bimg/bmask cover global planes [bz0, bz1); the rank owns [z0, z1).
static int slab_compute(ife_cuda_ctx* ctx, const float* bimg, const uint8_t* bmask, int bz0, int bz1,
                        int z0, int z1, float* out, const int global_dims[3],
                        const double spacing[3], const double* sigmas, int n_sigma,
                        const float* edges, int n_edges, uint32_t* counts, double halo_factor,
                        int mem, uint32_t** d_counts_out, cudaEvent_t far_ready = nullptr,
                        int near_h = 0) {
  using namespace ife;
  cudaStream_t st = ctx->stream();
  bool far_waited = far_ready == nullptr;
  Workspace& ws = ctx->ws;
  const int nx = global_dims[0], ny = global_dims[1], nz = global_dims[2];
  const size_t plane = (size_t)nx * ny;
  const int nzo = z1 - z0, nzb = bz1 - bz0;
  const size_t n_own = plane * nzo;
  const int fz0 = std::max(0, z0 - 1), fz1 = std::min(nz, z1 + 1);  // planes the stencil reads
  const int nzf = fz1 - fz0;
  IFE_TRY(reserve_smoothing(ctx, 2, nx, ny, nzb));
  IFE_TRY(ws.blur.reserve(ctx, plane * nzf * sizeof(float)));
  const int rows = n_sigma * 8, nb = n_edges + 1;
  uint32_t* d_counts = nullptr;
  if (edges) {
    IFE_TRY(ws.edges.reserve(ctx, (size_t)rows * n_edges * sizeof(float)));
    IFE_CUDA_TRY(ctx, cudaMemcpyAsync(ws.edges.ptr, edges, (size_t)rows * n_edges * sizeof(float),
                                      cudaMemcpyHostToDevice, st));
    IFE_TRY(stage_out(ctx, ws.counts, counts, (size_t)rows * nb, mem, &d_counts));
    IFE_CUDA_TRY(ctx, cudaMemsetAsync(d_counts, 0, (size_t)rows * nb * sizeof(uint32_t), st));
  }
  if (d_counts_out) *d_counts_out = d_counts;
  if (out && mem == IFE_MEM_HOST) IFE_TRY(ws.out[0].reserve(ctx, 8 * n_own * sizeof(float)));

  const StencilCoef S = make_stencil_coef(spacing);
  for (int s = 0; s < n_sigma; ++s) {
    // z-pass extent at this scale: the warm-up halo shrinks with sigma
    const int H = ife_cuda_slab_halo(sigmas[s], spacing[2], halo_factor);
    if (!far_waited && H > near_h) {   // first scale that reads planes of the second exchange group
      IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(st, far_ready, 0));
      far_waited = true;
    }
    const int sz0 = std::max(bz0, z0 - H), sz1 = std::min(bz1, z1 + H);
    float* blur = (float*)ws.blur.ptr;
    IFE_TRY(smooth_volume(ctx, bimg + plane * (sz0 - bz0), bmask + plane * (sz0 - bz0), true, blur, nx,
                          ny, sz1 - sz0, fz0 - sz0, fz1 - sz0, spacing, sigmas[s], nullptr, nullptr));
    FeatArgs A;
    std::memset(&A, 0, sizeof(A));
    A.vol = blur;
    A.mask_u8 = bmask + plane * (fz0 - bz0);
    A.nx = nx; A.ny = ny; A.nzb = nzf; A.zb0 = z0 - fz0; A.zb1 = A.zb0 + nzo; A.z_global0 = fz0;
    float* d_out = nullptr;
    if (out) {
      d_out = mem == IFE_MEM_HOST ? (float*)ws.out[0].ptr : out + (size_t)s * 8 * n_own;
      for (int k = 0; k < 8; ++k) A.out[k] = d_out + (size_t)k * n_own;
    }
    if (edges) {
      A.hist.edges = (const float*)ws.edges.ptr + (size_t)s * 8 * n_edges;
      A.hist.counts = d_counts + (size_t)s * 8 * nb;
      A.hist.n_edges = n_edges;
      A.hist.n_roi = 0;
      A.hist.stride_roi = (long long)rows * nb;
    }
    IFE_TRY(launch_features(ctx, 0, S, A, is_unit_spacing(spacing)));
    if (out && mem == IFE_MEM_HOST)
      IFE_CUDA_TRY(ctx, cudaMemcpyAsync(out + (size_t)s * 8 * n_own, d_out, 8 * n_own * sizeof(float),
                                        cudaMemcpyDeviceToHost, st));
  }
  if (!far_waited) IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(st, far_ready, 0));
  return IFE_OK;
}

static int slab_check_args(ife_cuda_ctx* ctx, const float* image, float* out, const int global_dims[3],
                           const double spacing[3], const double* sigmas, int n_sigma,
                           const float* edges, int n_edges, uint32_t* counts) {
  using namespace ife;
  if (!image) return fail(ctx, IFE_E_INVALID, "null image pointer");
  if (!out && !edges) return fail(ctx, IFE_E_INVALID, "nothing to compute: out and edges both null");
  if (edges && (!counts || n_edges <= 0)) return fail(ctx, IFE_E_INVALID, "bad histogram arguments");
  if (!sigmas || n_sigma <= 0) return fail(ctx, IFE_E_INVALID, "need at least one scale");
  return check_dims(ctx, global_dims, spacing);
}

int ife_cuda_slab_emphysema_features_local(ife_cuda_ctx* ctx, const float* image_ext,
                                           const uint8_t* mask_ext, int ext_z0, int ext_nz,
                                           int own_z0, int own_nz, float* out,
                                           const int global_dims[3], const double spacing[3],
                                           const double* sigmas, int n_sigma, const float* edges,
                                           int n_edges, uint32_t* counts, double halo_factor,
                                           int mem) {
  using namespace ife;
  if (!ctx) return IFE_E_INVALID;
  IFE_TRY(slab_check_args(ctx, image_ext, out, global_dims, spacing, sigmas, n_sigma, edges, n_edges, counts));
  const int nz = global_dims[2];
  if (own_nz <= 0 || own_z0 < 0 || own_z0 + own_nz > nz || ext_z0 < 0 || ext_z0 + ext_nz > nz ||
      ext_z0 > own_z0 || ext_z0 + ext_nz < own_z0 + own_nz)
    return fail(ctx, IFE_E_INVALID, "bad slab ranges");
  // the buffer must reach one plane past the slab (central differences) unless at a global edge
  if ((own_z0 > 0 && ext_z0 > own_z0 - 1) || (own_z0 + own_nz < nz && ext_z0 + ext_nz < own_z0 + own_nz + 1))
    return fail(ctx, IFE_E_INVALID, "halo must cover at least one plane on every interior side");
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t plane = (size_t)global_dims[0] * global_dims[1];
  const float* d_img;
  const uint8_t* d_mask;
  IFE_TRY(stage_in(ctx, ctx->ws.slab_img, image_ext, plane * ext_nz, mem, &d_img));
  if (mask_ext) {
    IFE_TRY(stage_in(ctx, ctx->ws.slab_mask, mask_ext, plane * ext_nz, mem, &d_mask));
  } else {
    IFE_TRY(ctx->ws.slab_mask.reserve(ctx, plane * ext_nz));
    IFE_CUDA_TRY(ctx, cudaMemsetAsync(ctx->ws.slab_mask.ptr, 1, plane * ext_nz, ctx->stream()));
    d_mask = (const uint8_t*)ctx->ws.slab_mask.ptr;
  }
  uint32_t* d_counts = nullptr;
  IFE_TRY(slab_compute(ctx, d_img, d_mask, ext_z0, ext_z0 + ext_nz, own_z0, own_z0 + own_nz, out,
                       global_dims, spacing, sigmas, n_sigma, edges, n_edges, counts, halo_factor, mem,
                       &d_counts));
  // the wait also covers the per-scale copies of `out` that slab_compute enqueued
  if (edges) return finish_out(ctx, counts, d_counts, (size_t)n_sigma * 8 * (n_edges + 1), mem);
  if (mem == IFE_MEM_HOST) IFE_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream()));
  return IFE_OK;
}

int ife_cuda_slab_emphysema_features(ife_cuda_ctx* ctx, const float* image_slab,
                                     const uint8_t* mask_slab, float* out,
                                     const int global_dims[3], const double spacing[3],
                                     const double* sigmas, int n_sigma, const float* edges,
                                     int n_edges, uint32_t* counts, double halo_factor, int mem) {
  using namespace ife;
  if (!ctx) return IFE_E_INVALID;
  IFE_TRY(slab_check_args(ctx, image_slab, out, global_dims, spacing, sigmas, n_sigma, edges, n_edges, counts));
  const int P = ctx->n_ranks, me = ctx->rank;
  if (P > 1 && !ctx->nccl_comm) return fail(ctx, IFE_E_COMM, "communicator not initialised");
  IFE_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  NcclApi& api = nccl_api();
  ncclComm_t comm = (ncclComm_t)ctx->nccl_comm;
  cudaStream_t st = ctx->stream();

  const int nx = global_dims[0], ny = global_dims[1], nz = global_dims[2];
  const size_t plane = (size_t)nx * ny;
  int z0, z1;
  slab_range(nz, P, me, &z0, &z1);
  const int nzo = z1 - z0;
  if (nzo <= 0) return fail(ctx, IFE_E_INVALID, "rank %d owns no planes (nz=%d, ranks=%d)", me, nz, P);
  double smax = 0.0;
  for (int s = 0; s < n_sigma; ++s) smax = std::max(smax, sigmas[s]);
  const int Hmax = ife_cuda_slab_halo(smax, spacing[2], halo_factor);
  const int bz0 = std::max(0, z0 - Hmax), bz1 = std::min(nz, z1 + Hmax);
  const int nzb = bz1 - bz0;
  const size_t n_own = plane * nzo;

  // ---- slab + halo buffers ----
  Workspace& ws = ctx->ws;
  IFE_TRY(ws.slab_img.reserve(ctx, plane * nzb * sizeof(float)));
  IFE_TRY(ws.slab_mask.reserve(ctx, plane * nzb));
  float* bimg = (float*)ws.slab_img.ptr;
  uint8_t* bmask = (uint8_t*)ws.slab_mask.ptr;
  cudaStream_t cs = ctx->copy_stream;
  cudaEvent_t ev_own = ctx->events[0], ev_near = ctx->events[1], ev_far = ctx->events[2], ev_done = ctx->events[3];
  // kernels of the previous call may still read the halo planes the receives overwrite
  IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(cs, ev_done, 0));
  const cudaMemcpyKind kin = mem == IFE_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  IFE_CUDA_TRY(ctx, cudaMemcpyAsync(bimg + plane * (z0 - bz0), image_slab, n_own * sizeof(float), kin, st));
  if (mask_slab)
    IFE_CUDA_TRY(ctx, cudaMemcpyAsync(bmask + plane * (z0 - bz0), mask_slab, n_own, kin, st));
  else
    IFE_CUDA_TRY(ctx, cudaMemsetAsync(bmask + plane * (z0 - bz0), 1, n_own, st));

  // ---- halo exchange on the copy stream, in two groups: the planes the first scale needs
  // (its halo is the smallest when scales ascend), then the rest, which arrives behind the
  // kernels of the first scale.  Device-resident slabs are sent straight from the caller's
  // buffers, so the exchange does not wait for the copy into the slab+halo buffer either.
  cudaEvent_t far_ready = nullptr;
  int near_h = Hmax;
  if (P > 1) {
    const bool own_src = mem == IFE_MEM_DEVICE && mask_slab != nullptr;
    const float* simg = own_src ? image_slab : bimg + plane * (z0 - bz0);
    const uint8_t* smask = own_src ? mask_slab : bmask + plane * (z0 - bz0);
    if (!own_src) {
      IFE_CUDA_TRY(ctx, cudaEventRecord(ev_own, st));
      IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(cs, ev_own, 0));
    }
    near_h = std::min(Hmax, ife_cuda_slab_halo(sigmas[0], spacing[2], halo_factor));
    // planes at distance (hlo, hhi] outside each slab travel in one grouped call
    auto exchange = [&](int hlo, int hhi) -> int {
      IFE_NCCL_TRY(ctx, api.GroupStart());
      for (int r = 0; r < P; ++r) {
        if (r == me) continue;
        int rz0, rz1;
        slab_range(nz, P, r, &rz0, &rz1);
        const bool above = rz0 >= z1;   // r's slab lies above mine (slabs are ordered)
        // planes I need from r
        int n0 = above ? std::max(z1 + hlo, rz0) : std::max(std::max(0, z0 - hhi), rz0);
        int n1 = above ? std::min(std::min(nz, z1 + hhi), rz1) : std::min(z0 - hlo, rz1);
        if (n0 < n1) {
          IFE_NCCL_TRY(ctx, api.Recv(bimg + plane * (n0 - bz0), plane * (n1 - n0), ncclFloat, r, comm, cs));
          IFE_NCCL_TRY(ctx, api.Recv(bmask + plane * (n0 - bz0), plane * (n1 - n0), ncclUint8, r, comm, cs));
        }
        // planes r needs from me: I am below r exactly when r is above me
        int s0 = above ? std::max(std::max(0, rz0 - hhi), z0) : std::max(rz1 + hlo, z0);
        int s1 = above ? std::min(rz0 - hlo, z1) : std::min(std::min(nz, rz1 + hhi), z1);
        if (s0 < s1) {
          IFE_NCCL_TRY(ctx, api.Send(simg + plane * (s0 - z0), plane * (s1 - s0), ncclFloat, r, comm, cs));
          IFE_NCCL_TRY(ctx, api.Send(smask + plane * (s0 - z0), plane * (s1 - s0), ncclUint8, r, comm, cs));
        }
      }
      IFE_NCCL_TRY(ctx, api.GroupEnd());
      return IFE_OK;
    };
    IFE_TRY(exchange(0, near_h));
    IFE_CUDA_TRY(ctx, cudaEventRecord(ev_near, cs));
    if (near_h < Hmax) {
      IFE_TRY(exchange(near_h, Hmax));
      IFE_CUDA_TRY(ctx, cudaEventRecord(ev_far, cs));
      far_ready = ev_far;
    }
    {
      // profiling kind 5: how long the main stream sits in this wait = the exposed part of the
      // first exchange group (the second group hides behind the kernels of the first scale)
      ProfScope prof(ctx, K_EXCHANGE);
      IFE_CUDA_TRY(ctx, cudaStreamWaitEvent(st, ev_near, 0));
    }
  }

  uint32_t* d_counts = nullptr;
  IFE_TRY(slab_compute(ctx, bimg, bmask, bz0, bz1, z0, z1, out, global_dims, spacing, sigmas, n_sigma,
                       edges, n_edges, counts, halo_factor, mem, &d_counts, far_ready, near_h));

  // ---- combine the per-rank histograms ----
  if (edges) {
    const size_t n_counts = (size_t)n_sigma * 8 * (n_edges + 1);
    if (P > 1)
      IFE_NCCL_TRY(ctx, api.AllReduce(d_counts, d_counts, n_counts, ncclUint32, ncclSum, comm, st));
    if (mem == IFE_MEM_HOST)
      IFE_CUDA_TRY(ctx, cudaMemcpyAsync(counts, d_counts, n_counts * sizeof(uint32_t),
                                        cudaMemcpyDeviceToHost, st));
  }
  // recorded AFTER the all-reduce: the next call's exchange (copy stream) waits on it, so the
  // communicator never has operations in flight on two streams at once, and the halo planes are
  // not overwritten while this call's kernels still read them
  IFE_CUDA_TRY(ctx, cudaEventRecord(ev_done, st));
  if (mem == IFE_MEM_HOST) IFE_CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return IFE_OK;
}

}  // extern "C"
