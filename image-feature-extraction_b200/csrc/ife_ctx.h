// Internal: the per-GPU context behind the opaque ife_cuda_ctx of include/ife_cuda.h.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include <cuda_runtime.h>

struct ife_cuda_ctx;

namespace ife {

// Grow-only device allocation owned by a context.
struct DeviceBuffer {
  void* ptr = nullptr;
  size_t bytes = 0;
  int reserve(ife_cuda_ctx* ctx, size_t want);
  void release();
};

struct Workspace {
  DeviceBuffer a0, a1, b0, b1;  // float volumes between the z, x and y passes (two fields)
  DeviceBuffer blur, blur2;     // smoothed volume fed to the fused feature kernel (blur2: option overlap_scales)
  DeviceBuffer ckpt;            // recursion checkpoints (double)
  DeviceBuffer in_img, in_mask; // staging for IFE_MEM_HOST inputs
  DeviceBuffer in_i16;          // int16 images on their way to float (option "host_image_i16"; two slots)
  DeviceBuffer out[2];          // staging for IFE_MEM_HOST outputs (double-buffered per scale)
  DeviceBuffer edges, rois, counts;
  DeviceBuffer packed;          // eight bin indices per voxel (many-ROI histogram path)
  DeviceBuffer slab_img, slab_mask;  // slab + halo planes (multi-GPU)
  DeviceBuffer box;             // raw extents[6] of the output mask (support_box.cuh)
  DeviceBuffer crop_img, crop_mask, crop_blur;   // the mask's bounding box as a dense volume (smooth_masked)
  void release_all() {
    DeviceBuffer* all[] = {&a0, &a1, &b0, &b1, &blur, &ckpt, &in_img, &in_mask, &out[0], &out[1],
                           &edges, &rois, &counts, &packed, &slab_img, &slab_mask, &box, &blur2, &crop_img, &crop_mask, &crop_blur, &in_i16};
    for (DeviceBuffer* b : all) b->release();
  }
};

int fail(ife_cuda_ctx* ctx, int code, const char* fmt, ...);

// kernel kinds for ife_cuda_profile_read
enum { K_PASS_Z = 0, K_PASS_X = 1, K_PASS_Y = 2, K_FEATURES = 3, K_OTHER = 4, K_EXCHANGE = 5, K_NUM = 6 };

// RAII: records a CUDA event before and after a kernel launch when profiling is on
struct ProfScope {
  ife_cuda_ctx* ctx;
  cudaEvent_t end = nullptr;
  ProfScope(ife_cuda_ctx* c, int kind);
  ~ProfScope();
};

}  // namespace ife

struct ife_cuda_ctx {
  int device = 0;
  int sm_count = 148;
  int arith = 1;  // IFE_ARITH_FMA
  cudaStream_t own_stream = nullptr;
  cudaStream_t copy_stream = nullptr;
  cudaStream_t hp_stream = nullptr;    // highest priority: the Gaussian passes of option "overlap_scales"
  cudaStream_t alt_stream = nullptr;   // when set, launches go here instead of the main stream
  cudaStream_t user_stream = nullptr;
  bool use_user_stream = false;
  cudaEvent_t events[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ov_events[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // overlap_scales: input ready, blur[0..1] written, blur[0..1] consumed
  uint64_t launches = 0;
  bool use_tma = true;     // tensor-map staged, field-per-warp Gaussian passes where the layout allows (option "tma_passes")
  bool use_march4 = true;  // fused feature kernel with four voxels per thread where the layout allows (option "march4")
  bool host_image_i16 = false;   // host image pointers of the ife_cuda_emphysema_* calls are int16 (option "host_image_i16")
  bool use_box = true;     // masked paths smooth only the mask's support box (option "support_box")
  int* box_host = nullptr; // pinned: the mask extents (or an expected distance's sums) come back here once per call
  bool overlap_scales = false;   // option "overlap_scales": features of scale s run beside the passes of scale s+1
  std::string error;
  ife::Workspace ws;
  // optional per-kernel timing (ife_cuda_profile_*): event pairs around every launch
  bool profiling = false;
  std::vector<cudaEvent_t> prof_events;  // 2 per launch: begin, end
  std::vector<int> prof_kinds;
  size_t prof_used = 0;                  // events handed out since the last read
  // NCCL (resolved lazily with dlopen; see slab.cu)
  void* nccl_comm = nullptr;
  int n_ranks = 1;
  int rank = 0;
  // what the last masked call's passes actually ran on (the crop of the mask's box, or the volume)
  int work_dims[3] = {0, 0, 0};

  cudaStream_t main_stream() const { return use_user_stream ? user_stream : own_stream; }
  cudaStream_t stream() const { return alt_stream ? alt_stream : main_stream(); }
};
