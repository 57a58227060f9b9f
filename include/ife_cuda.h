/* ife_cuda.h -- C ABI of libife_cuda.so, the B200 (sm_100a) implementation of the dense
 * per-voxel hot path of orting/image-feature-extraction:
 *
 *   multi-scale (recursive) Gaussian smoothing / masked normalized convolution
 *   -> finite-difference Hessian + gradient magnitude -> closed-form symmetric 3x3
 *   eigenvalues -> eigenvalue features -> optional mask -> optional DenseHistogram binning.
 *
 * The reference has no FFI of its own: its surface for this path is a set of C++ ITK
 * filter classes and functors plus four command-line tools.  Each entry point below names
 * the reference interface it replaces (paths relative to the reference checkout); the C++
 * facades in image-feature-extraction_b200/host/include/ife/ keep the reference's class
 * and method names and call these functions, and INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - volumes are float32, x fastest: idx = x + nx*(y + ny*z); dims = {nx,ny,nz};
 *     spacing = {sx,sy,sz} in physical units (sigma is physical, as in ITK);
 *   - masks are uint8 (itk::Image<unsigned char,3>, tools/ExtractFeatures.cxx:82) unless
 *     an argument says float (the tools that read the mask/certainty as float);
 *   - multi-component results are SoA planes: out[k*nx*ny*nz + idx];
 *   - `mem` says where EVERY data pointer of the call lives: IFE_MEM_HOST (the library
 *     stages through its own device buffers; the call returns when the outputs are in the
 *     host buffers) or IFE_MEM_DEVICE (pointers are device pointers on the context's
 *     device; work is enqueued on the context's stream and the call returns without
 *     synchronising);  small parameter arrays (dims, spacing, sigmas, edges, rois) are
 *     always host pointers;
 *   - every function returns 0 on success or a negative IFE_E_* code; the message is
 *     kept per context (ife_cuda_last_error).  No exception crosses this boundary;
 *   - a context is bound to one device and one stream and is NOT thread-safe; use one
 *     context per host thread / GPU.  Outputs must not alias inputs.
 *   - there is no CPU fallback: without a CUDA device every call fails with IFE_E_CUDA.
 */
#ifndef IFE_CUDA_H
#define IFE_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IFE_CUDA_ABI_VERSION 1

typedef struct ife_cuda_ctx ife_cuda_ctx;

enum { IFE_MEM_HOST = 0, IFE_MEM_DEVICE = 1 };

enum {
  IFE_OK = 0,
  IFE_E_INVALID = -1,   /* bad argument (null pointer, non-positive size, ...) */
  IFE_E_TOO_SMALL = -2, /* an axis has < 4 samples: ITK's recursive Gaussian throws */
  IFE_E_CUDA = -3,      /* CUDA runtime / driver failure (message has the CUDA error) */
  IFE_E_NOMEM = -4,     /* device allocation failed */
  IFE_E_COMM = -5       /* NCCL failure or communicator not initialised */
};

/* Arithmetic of the recursive Gaussian's line recursion (double precision either way):
 * PLAIN rounds every multiply and add separately, left to right, as ITK's source reads
 * when built without FMA contraction; FMA contracts each left-to-right sum of products
 * into multiply + fused multiply-adds the way `g++ -O2 -mfma` does.  Both are bit-exact
 * against the oracle run in the same mode. */
enum { IFE_ARITH_PLAIN = 0, IFE_ARITH_FMA = 1 };

/* Number of per-voxel features of ImageToEmphysemaFeaturesFilter
 * (include/ife/Filters/ImageToEmphysemaFeaturesFilter.h:62 `numFeatures = 8`), in the
 * order [GaussianBlur, GradientMagnitude, Eigenvalue1..3, LaplacianOfGaussian,
 * GaussianCurvature, FrobeniusNorm] (tools/ExtractFeatures.cxx:126-130). */
#define IFE_NUM_FEATURES 8
/* Features of EigenvalueFeaturesFunctor (include/ife/Numerics/EigenvalueFeaturesFunctor.h:
 * 20-31): [e1, e2, e3, e1+e2+e3, e1*e2*e3, sqrt(e1^2+e2^2+e3^2)]. */
#define IFE_NUM_EIGEN_FEATURES 6

/* ---- context ------------------------------------------------------------------- */
int ife_cuda_abi_version(void);
int ife_cuda_create(int device, ife_cuda_ctx** ctx);
void ife_cuda_destroy(ife_cuda_ctx* ctx);
const char* ife_cuda_last_error(const ife_cuda_ctx* ctx);
/* Page-locked host memory for the buffers handed to IFE_MEM_HOST calls: the library's
 * host<->device copies of such a buffer run at full PCIe rate and overlap with the kernels
 * (a pageable buffer is staged by the driver, synchronously).  No context needed; fails with
 * IFE_E_CUDA without a device (callers then fall back to malloc).  The C++ facades allocate every
 * image this way (host/include/ife/Image.h).  Blocks of 32 MB and more are anonymous huge-page
 * mappings faulted in by all cores and registered with the driver (0.05 s per GB instead of
 * cudaHostAlloc's 0.4-0.5); IFE_NO_MAPPED_HOST_ALLOC in the environment forces cudaHostAlloc,
 * IFE_ALLOC_TRACE prints the time of every large allocation to stderr.  Free with
 * ife_cuda_host_free only. */
int ife_cuda_host_alloc(size_t bytes, void** ptr);
void ife_cuda_host_free(void* ptr);
/* Use an existing cudaStream_t (e.g. a framework's current stream) instead of the
 * context's own; pass NULL to go back to the context's stream. */
int ife_cuda_set_stream(ife_cuda_ctx* ctx, void* cuda_stream);
int ife_cuda_set_arith(ife_cuda_ctx* ctx, int arith_mode);
int ife_cuda_get_arith(const ife_cuda_ctx* ctx);
int ife_cuda_synchronize(ife_cuda_ctx* ctx);
/* Pre-size the context's device workspace for volumes of `dims` (optional; the workspace
 * otherwise grows on first use).  n_outputs = how many float output volumes the largest
 * IFE_MEM_HOST call will stage (0 when only device pointers are used). */
int ife_cuda_reserve(ife_cuda_ctx* ctx, const int dims[3], int n_outputs);
/* Kernel launches issued by this context since creation (bench.py's gpu_launches). */
uint64_t ife_cuda_launch_count(const ife_cuda_ctx* ctx);
/* Dimensions of the volume the Gaussian passes of the last masked call
 * (ife_cuda_emphysema_features / _histograms / _histograms_batch) actually ran on: the dense crop
 * of the mask's support box (option "support_box"), or the full dims when no crop was taken.
 * For benchmarks that report bytes moved per kernel. */
int ife_cuda_last_work_dims(const ife_cuda_ctx* ctx, int dims[3]);

/* Tuning / debugging switches.  "support_box" (default 1): the calls whose every result is masked
 * (ife_cuda_emphysema_features / _histograms / _histograms_batch) smooth only what an in-mask
 * voxel can see -- the mask's bounding box grown by the one-voxel stencil reach, smoothed as a
 * dense cropped copy (outside the mask both fields of the normalized convolution are exact
 * zeros, so the crop gives the same bits), and inside it only the ROI list's bounding box when
 * there is one; the box is reduced on the device and read back once per call, which makes
 * these calls wait for the stream once.  0 smooths the whole volume (same results bit for bit --
 * PRECONDITION: the image is finite.  The identity rests on c*T being an exact zero wherever the
 * mask c is zero; a NaN or Inf voxel OUTSIDE the mask's box gives 0*NaN = NaN, which the
 * reference (and option value 0) propagates along the whole IIR line into in-mask voxels while
 * the cropped path never sees it.  CT volumes are integer-valued; callers with non-finite
 * padding must clear it or switch the option off).
 * "tma_passes" (default 1): normalized convolution with a uint8 certainty on volumes with
 * nx % 16 == 0, or with a float certainty and nx % 4 == 0 (with or without output mask), and the plain
 * Gaussian with nx % 4 == 0 run the tensor-map staged, field-per-warp pass kernels
 * (csrc/iir_tma.cuh); 0 selects the plain register-staged kernels, which every other layout
 * runs (same results bit for bit).
 * "march4" (default 1): the fused feature kernel owns four x-adjacent voxels per thread when
 * nx % 4 == 0 and the pointers are 16-byte aligned (csrc/features_march4.cuh); 0 selects the
 * one-voxel-per-thread kernel (same results bit for bit).
 * "host_image_i16" (default 0): the HOST image pointers handed to ife_cuda_emphysema_features /
 * _histograms / _histograms_batch / _feature_samples point to int16 voxels (cast the pointer) -- CT's
 * type on disk, which the reference's tools widen to float on the host while reading
 * (tools/ExtractFeatures.cxx:90-96).  The library uploads 2 bytes per voxel and widens on the device
 * (exact); a batch of scans whose kernels take less time than a float upload becomes kernel-bound.
 * Device pointers are always float.
 * "overlap_scales" (default 0): device-resident ife_cuda_emphysema_features calls with several
 * scales run the Gaussian passes one scale ahead on a high-priority stream of the context,
 * beside the fused feature kernel of the scale before (two blur buffers); same results bit
 * for bit, +2..4 % throughput measured, per-kernel timings then overlap. */
int ife_cuda_set_option(ife_cuda_ctx* ctx, const char* name, int value);

/* Optional per-kernel timing for benchmarks: while enabled, every kernel launch of the
 * context is bracketed by CUDA events on the launching stream.  ife_cuda_profile_read
 * synchronises, returns the summed device time (ms) and launch count per kernel kind since
 * the last read, and resets.  Kinds: 0 = Gaussian z pass, 1 = x pass, 2 = y pass,
 * 3 = fused Hessian/eigen/feature(/histogram) kernel, 4 = other, 5 = not a kernel: the time
 * the main stream of ife_cuda_slab_emphysema_features waited for the first halo exchange group
 * (the exposed part of the exchange). */
#define IFE_PROFILE_KINDS 6
int ife_cuda_profile_enable(ife_cuda_ctx* ctx, int on);
int ife_cuda_profile_read(ife_cuda_ctx* ctx, double ms[IFE_PROFILE_KINDS],
                          uint64_t launches[IFE_PROFILE_KINDS]);

/* ---- per-stage entry points ------------------------------------------------------ */

/* itk::SmoothingRecursiveGaussianImageFilter<float image> as the reference uses it
 * (include/ife/Filters/NormalizedGaussianConvolutionImageFilter.h:72): three recursive
 * (IIR, Deriche 4th order) passes z, x, y in double, float storage between passes. */
int ife_cuda_gaussian(ife_cuda_ctx* ctx, const float* in, float* out, const int dims[3],
                      const double spacing[3], double sigma, int mem);

/* itk::NormalizedGaussianConvolutionImageFilter::GenerateData
 * (include/ife/Filters/NormalizedGaussianConvolutionImageFilter.hxx:37-63):
 * out = G(c*T)/G(c).  Exactly one of certainty_f32 / certainty_u8 is non-null (the
 * MaskedNormalizedConvolution tool reads the certainty as float, tools/
 * MaskedNormalizedConvolution.cxx:129-139; ImageToEmphysemaFeaturesFilter casts a uint8
 * mask, .hxx:21).  mask_output != 0 applies itk::MaskImageFilter with the certainty as
 * mask (tools/MaskedNormalizedConvolution.cxx:156-159, the tool's -m flag). */
int ife_cuda_normalized_gaussian(ife_cuda_ctx* ctx, const float* image,
                                 const float* certainty_f32, const uint8_t* certainty_u8,
                                 float* out, const int dims[3], const double spacing[3],
                                 double sigma, int mask_output, int mem);

/* itk::GradientMagnitudeImageFilter followed by itk::MaskImageFilter
 * (tools/FiniteDifference_GradientFeatures.cxx:105-113).  Either mask may be null. */
int ife_cuda_gradient_magnitude(ife_cuda_ctx* ctx, const float* in, const float* mask_f32,
                                const uint8_t* mask_u8, float* out, const int dims[3],
                                const double spacing[3], int mem);

/* itk::Hessian3DImageFilter + EigenvalueFeaturesFunctor with the mask rule of
 * tools/FiniteDifference_HessianFeatures.cxx:209-229 (mask == 0 -> six zeros), fused:
 * the Hessian is never written to memory.  sigma > 0 first smooths with ife_cuda_gaussian
 * (BASELINE.json configs[0]); sigma <= 0 is the tool as shipped (no smoothing).
 * out6 = 6 SoA planes [eig1, eig2, eig3, LoG, Curvature, Frobenius].  mask may be null.
 * flags: IFE_FDHF_TOOL_DY_BUG reproduces the tool's `dyFilter->SetDirection(0)`
 * (tools/FiniteDifference_HessianFeatures.cxx:153-156). */
#define IFE_FDHF_TOOL_DY_BUG 1
int ife_cuda_hessian_eigen_features(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                    float* out6, const int dims[3], const double spacing[3],
                                    double sigma, int flags, int mem);

/* itk::Hessian3DImageFilter itself (include/ife/Filters/Hessian3DImageFilter.hxx:11-60): the six
 * central-difference stencils on the image as given (no smoothing, no mask), cross terms as two
 * chained first-order DerivativeImageFilters (the intermediate is rounded to float), every
 * stage scaled once by 1/spacing[direction], ZeroFluxNeumann (index-clamped) edges.
 * out6 = 6 SoA planes in the filter's component order [Dxx, Dxy, Dxz, Dyy, Dyz, Dzz]
 * (Hessian3DImageFilter.hxx:53-59). */
int ife_cuda_hessian(ife_cuda_ctx* ctx, const float* image, float* out6, const int dims[3],
                     const double spacing[3], int mem);

/* itk::ImageToEmphysemaFeaturesFilter for a list of scales
 * (include/ife/Filters/ImageToEmphysemaFeaturesFilter.hxx:94-121, looped over sigma as
 * tools/ExtractFeatures.cxx:132-154 does): out = [n_sigma][8] SoA planes. */
int ife_cuda_emphysema_features(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                float* out, const int dims[3], const double spacing[3],
                                const double* sigmas, int n_sigma, int mem);

/* The same features binned without ever writing them: the insert loop of
 * tools/MakeBag.cxx:425-470 over DenseHistogram<float>
 * (include/ife/Statistics/DenseHistogram.h:47-53; bin = number of edges < value).
 *   edges  : [n_sigma*8][n_edges] float, sorted per row (one row per scale and feature,
 *            features organised by scale as MakeBag.cxx:451-453);
 *   rois   : [n_roi][6] int {x0,y0,z0,sx,sy,sz}, or n_roi == 0 for one ROI = whole volume;
 *   counts : [max(n_roi,1)][n_sigma*8][n_edges+1] uint32, overwritten (host or device
 *            per `mem`).
 * Only voxels with mask != 0 are inserted. */
int ife_cuda_emphysema_histograms(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                  const int dims[3], const double spacing[3],
                                  const double* sigmas, int n_sigma, const float* edges,
                                  int n_edges, const int* rois, int n_roi, uint32_t* counts,
                                  int mem);

/* A batch of scans of identical size (BASELINE.json configs[4]: "batch of scans, full
 * multi-scale feature + histogram bagging pipeline"): ife_cuda_emphysema_histograms for
 * n_scans host-resident scans, with the upload of scan i+1 overlapped with the kernels of
 * scan i (pinned host memory makes the overlap real).  images / masks: arrays of n_scans
 * host pointers; rois: [n_scans][n_roi][6] (each scan its own ROIs) or NULL with
 * n_roi == 0; counts: [n_scans][max(n_roi,1)][n_sigma*8][n_edges+1], host.  One scan per
 * GPU is the multi-GPU sharding of this workload: one context and one call per GPU. */
int ife_cuda_emphysema_histograms_batch(ife_cuda_ctx* ctx, int n_scans, const float* const* images,
                                        const uint8_t* const* masks, const int dims[3],
                                        const double spacing[3], const double* sigmas, int n_sigma,
                                        const float* edges, int n_edges, const int* rois, int n_roi,
                                        uint32_t* counts);

/* DenseHistogram<float>::insert over an array (include/ife/Statistics/DenseHistogram.h:
 * 47-53): counts[n_edges+1] is overwritten. */
int ife_cuda_histogram(ife_cuda_ctx* ctx, const float* values, size_t n, const float* edges,
                       int n_edges, uint32_t* counts, int mem);

/* tools/MakeBagOnlyIntensity.cxx:352-391: for every ROI box {x0,y0,z0,sx,sy,sz} the
 * intensities of its in-mask voxels (mask != 0) are inserted into ONE DenseHistogram<float>
 * with the given edges.  rois: host int[n_roi][6]; edges: host float[n_edges];
 * counts: uint32[n_roi][n_edges+1] (overwritten), host or device per `mem`, like image / mask. */
int ife_cuda_intensity_roi_histograms(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                      const int dims[3], const float* edges, int n_edges,
                                      const int* rois, int n_roi, uint32_t* counts, int mem);

/* Resampling onto a new voxel spacing: itk::ResampleImageFilter with an identity transform and the
 * output origin equal to the input's (the reference's Resample tool, which is not part of the port
 * otherwise; DESIGN.md "Resampling" restates the semantics and lists where they differ from ITK).
 *   out_dims[d] = max(1, floor(dims[d] * spacing[d] / out_spacing[d] + 0.5)) in double; out_dims is
 *   always written, and out == NULL only queries it (in must still be given; ctx may then be NULL,
 *   so the query works without a device);
 *   continuous index c = (i * out_spacing[d]) * (1 / spacing[d]), c = i where the spacings are equal;
 *   outside -0.5 <= c < dims[d] - 0.5 on any axis the voxel is default_value;
 *   IFE_INTERP_LINEAR: LinearInterpolateImageFunction, float voxels only (elem_bytes 4).
 *     PRECONDITION: the input is finite (a zero-weight Inf or NaN neighbour would poison the lerp);
 *   IFE_INTERP_NEAREST: NearestNeighborInterpolateImageFunction, index floor(c + 0.5); float or uint8
 *     voxels (elem_bytes 4 or 1; for uint8 default_value must be an integer in [0, 255]).
 * in and out have the layout and `mem` of every volume of this ABI (x fastest, dims = {nx,ny,nz}).
 * IFE_E_INVALID for a null in, a non-positive or non-finite spacing, linear with elem_bytes 1, or an
 * unknown interp. */
#define IFE_INTERP_LINEAR 0
#define IFE_INTERP_NEAREST 1
int ife_cuda_resample(ife_cuda_ctx* ctx, const void* in, void* out, int elem_bytes,
                      const int dims[3], const double spacing[3], const double out_spacing[3],
                      int interp, double default_value, int out_dims[3], int mem);

/* Ascending in-place sort of n floats: the `std::sort` of the feature samples in
 * tools/DetermineHistogramBinEdges_MultiScaleEigenvalueFeatures.cxx:282-283.  A radix sort of
 * this library's own (csrc/radix_sort.cuh: 4-bit digits, count / scan / stable scatter; no
 * CUB); the equal-frequency edge walk of DetermineEdgesForEqualizedHistogram.h then runs on
 * the host, it touches O(bins * log n) samples. */
int ife_cuda_sort_f32(ife_cuda_ctx* ctx, float* data, size_t n, int mem);

/* The sampling loop of tools/DetermineHistogramBinEdges_MultiScaleEigenvalueFeatures.cxx:171-264
 * with the feature volumes never leaving the device ("compaction sink"): for every scale the 8
 * features of ImageToEmphysemaFeaturesFilter are computed on the device and only the sampled
 * voxels' values are kept, as dense rows out[s][k][j], j < *n_out.
 *   select != NULL: uint8 flags per voxel; the selected voxels in voxel-index order (the "all
 *                   foreground voxels" mode, -S 0); index must be NULL;
 *   index  != NULL: n_index voxel indices (x + nx*(y + ny*z)), repeats allowed, order kept (the
 *                   random sampling mode); select must be NULL.
 * sorted != 0 additionally sorts every row ascending on the device (ife_cuda_sort_f32's kernels),
 * which is what the edge walk wants.  out == NULL only counts (*n_out). */
int ife_cuda_emphysema_feature_samples(ife_cuda_ctx* ctx, const float* image, const uint8_t* mask,
                                       const uint8_t* select, const long long* index, size_t n_index,
                                       const int dims[3], const double spacing[3], const double* sigmas,
                                       int n_sigma, int sorted, float* out, size_t* n_out, int mem);

/* EigenvalueFeaturesFunctor<float> (and through it Symmetric3x3EigenvalueSolver<float>,
 * include/ife/Numerics/Symmetric3x3EigenvalueSolver.h:33-132) over n interleaved
 * matrices A6 = [A11,A12,A13,A22,A23,A33]; out6 interleaved. */
int ife_cuda_eigen_features_batch(ife_cuda_ctx* ctx, const float* A6, float* out6, size_t n,
                                  int mem);

/* ---- multi-GPU: z-slab partitioned volumes (one process / context per GPU) --------- */

/* NCCL unique id (128 bytes) created on rank 0 and passed to every rank by the caller
 * (any out-of-band channel: torch.distributed store, MPI, a file). */
#define IFE_COMM_ID_BYTES 128
int ife_cuda_comm_unique_id(ife_cuda_ctx* ctx, uint8_t id[IFE_COMM_ID_BYTES]);
int ife_cuda_comm_init(ife_cuda_ctx* ctx, const uint8_t id[IFE_COMM_ID_BYTES], int n_ranks,
                       int rank);
int ife_cuda_comm_destroy(ife_cuda_ctx* ctx);

/* Planes [z0, z1) of a global volume of global_dims owned by this rank when the volume is
 * cut into n_ranks contiguous z-slabs. */
void ife_cuda_slab_range(int nz_global, int n_ranks, int rank, int* z0, int* z1);
/* Halo planes per side needed at scale sigma: ceil(halo_factor*sigma/spacing_z) + 4 warm-up
 * planes for the z recursion + 1 for the z central difference. */
int ife_cuda_slab_halo(double sigma, double spacing_z, double halo_factor);

/* ImageToEmphysemaFeaturesFilter on this rank's z-slab of a larger volume.  image_slab /
 * mask_slab hold ONLY the owned planes [z0,z1); halo planes are exchanged with the z
 * neighbours with ncclSend/ncclRecv over NVLink, once per call, sized for the largest
 * sigma.  out = [n_sigma][8] SoA planes of the owned slab (may be null when only
 * histograms are wanted).  When edges != null the owned voxels are binned and the
 * per-rank counts are summed over ranks with ncclAllReduce; every rank receives the
 * global counts [n_sigma*8][n_edges+1].  mask_slab may be null (all inside -> plain
 * Gaussian instead of normalized convolution is NOT implied: a null mask means certainty 1
 * everywhere).  halo_factor <= 0 selects the default (12).
 * ACCURACY: the recursive Gaussian has an infinite impulse response, so a slab result equals
 * the whole-volume result bit for bit only when the halo reaches the volume's ends (e.g.
 * halo_factor >= nz / sigma_min).  A finite halo starts the z recursion from the edge-extension
 * state halo(sigma) planes away; the start-state error decays as exp(-1.37 d / sigma), i.e.
 * below 1e-7 of the local contrast at the default 12 sigma.  Measured on 1024^3 at 2 ranks
 * (bench.py, "slab" leg, parity block): 9e-5 of the output values differ from the single-GPU
 * result in their last bits, 3e-7 of the voxels by more than 1e-4 * max|lambda|, no change of
 * eigenvalue ordering; at halo_factor 8 those fractions are 5e-3 and 5e-5.  Histogram counts
 * move by the same few voxels near bin edges. */
int ife_cuda_slab_emphysema_features(ife_cuda_ctx* ctx, const float* image_slab,
                                     const uint8_t* mask_slab, float* out,
                                     const int global_dims[3], const double spacing[3],
                                     const double* sigmas, int n_sigma, const float* edges,
                                     int n_edges, uint32_t* counts, double halo_factor,
                                     int mem);

/* The per-rank half of the call above without any communication: image_ext / mask_ext hold
 * global planes [ext_z0, ext_z0+ext_nz), which must contain the owned planes
 * [own_z0, own_z0+own_nz) plus whatever halo the caller has (at least one plane on every
 * side that is not a global edge; the z recursion warms up over min(available, halo(sigma))
 * planes).  counts are this slab's own (not reduced).  Lets a caller with its own transport
 * (MPI, host staging, a single GPU walking over slabs of a volume larger than its memory)
 * use the slab pipeline. */
int ife_cuda_slab_emphysema_features_local(ife_cuda_ctx* ctx, const float* image_ext,
                                           const uint8_t* mask_ext, int ext_z0, int ext_nz,
                                           int own_z0, int own_nz, float* out,
                                           const int global_dims[3], const double spacing[3],
                                           const double* sigmas, int n_sigma, const float* edges,
                                           int n_edges, uint32_t* counts, double halo_factor,
                                           int mem);

#ifdef __cplusplus
}
#endif
#endif /* IFE_CUDA_H */
