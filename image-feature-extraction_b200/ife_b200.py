"""ctypes binding of libife_cuda.so (include/ife_cuda.h) for the tests, bench.py and Python
callers.  Thin on purpose: every function maps 1:1 onto a C-ABI entry point; numpy arrays
are passed as host pointers (IFE_MEM_HOST), torch CUDA tensors / raw integers as device
pointers (IFE_MEM_DEVICE).

There is NO CPU fallback: if the shared library is missing or no CUDA device is usable the
constructors raise.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IFE_CUDA_LIB") or os.path.join(_HERE, "lib", "libife_cuda.so")
HEADER_PATH = os.path.normpath(os.path.join(_HERE, "..", "include", "ife_cuda.h"))

MEM_HOST, MEM_DEVICE = 0, 1
INTERP_LINEAR, INTERP_NEAREST = 0, 1
ARITH_PLAIN, ARITH_FMA = 0, 1
FDHF_TOOL_DY_BUG = 1
NUM_FEATURES = 8
COMM_ID_BYTES = 128
FEATURE_NAMES = ["GaussianBlur", "GradientMagnitude", "Eigenvalue1", "Eigenvalue2", "Eigenvalue3",
                 "LaplacianOfGaussian", "GaussianCurvature", "FrobeniusNorm"]
ERRORS = {0: "IFE_OK", -1: "IFE_E_INVALID", -2: "IFE_E_TOO_SMALL", -3: "IFE_E_CUDA",
          -4: "IFE_E_NOMEM", -5: "IFE_E_COMM"}


class IfeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s: %s" % (ERRORS.get(code, code), msg))
        self.code = code


_lib = None


def load_library():
    """dlopen the in-tree libife_cuda.so; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            "%s is missing: build it with `make -C image-feature-extraction_b200` "
            "(or __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i, d, sz = C.c_void_p, C.c_int, C.c_double, C.c_size_t
    ip, dp = C.POINTER(C.c_int), C.POINTER(C.c_double)
    L.ife_cuda_abi_version.restype = i
    L.ife_cuda_create.argtypes = [i, C.POINTER(vp)]
    L.ife_cuda_destroy.argtypes = [vp]
    L.ife_cuda_destroy.restype = None
    L.ife_cuda_last_error.argtypes = [vp]
    L.ife_cuda_last_error.restype = C.c_char_p
    L.ife_cuda_set_stream.argtypes = [vp, vp]
    L.ife_cuda_set_arith.argtypes = [vp, i]
    L.ife_cuda_get_arith.argtypes = [vp]
    L.ife_cuda_synchronize.argtypes = [vp]
    L.ife_cuda_reserve.argtypes = [vp, ip, i]
    L.ife_cuda_launch_count.argtypes = [vp]
    L.ife_cuda_launch_count.restype = C.c_uint64
    L.ife_cuda_last_work_dims.argtypes = [vp, ip]
    L.ife_cuda_set_option.argtypes = [vp, C.c_char_p, i]
    L.ife_cuda_profile_enable.argtypes = [vp, i]
    L.ife_cuda_profile_read.argtypes = [vp, dp, C.POINTER(C.c_uint64)]
    L.ife_cuda_gaussian.argtypes = [vp, vp, vp, ip, dp, d, i]
    L.ife_cuda_normalized_gaussian.argtypes = [vp, vp, vp, vp, vp, ip, dp, d, i, i]
    L.ife_cuda_gradient_magnitude.argtypes = [vp, vp, vp, vp, vp, ip, dp, i]
    L.ife_cuda_hessian_eigen_features.argtypes = [vp, vp, vp, vp, ip, dp, d, i, i]
    L.ife_cuda_hessian.argtypes = [vp, vp, vp, ip, dp, i]
    L.ife_cuda_emphysema_features.argtypes = [vp, vp, vp, vp, ip, dp, dp, i, i]
    L.ife_cuda_emphysema_histograms.argtypes = [vp, vp, vp, ip, dp, dp, i, vp, i, vp, i, vp, i]
    L.ife_cuda_emphysema_histograms_batch.argtypes = [vp, i, vp, vp, ip, dp, dp, i, vp, i, vp, i, vp]
    L.ife_cuda_histogram.argtypes = [vp, vp, sz, vp, i, vp, i]
    L.ife_cuda_intensity_roi_histograms.argtypes = [vp, vp, vp, ip, vp, i, vp, i, vp, i]
    L.ife_cuda_eigen_features_batch.argtypes = [vp, vp, vp, sz, i]
    L.ife_cuda_sort_f32.argtypes = [vp, vp, sz, i]
    L.ife_cuda_resample.argtypes = [vp, vp, vp, i, ip, dp, dp, i, d, ip, i]
    L.ife_cuda_emphysema_feature_samples.argtypes = [vp, vp, vp, vp, vp, sz, ip, dp, dp, i, i, vp, C.POINTER(sz), i]
    L.ife_cuda_host_alloc.argtypes = [sz, C.POINTER(C.c_void_p)]
    L.ife_cuda_host_free.argtypes = [vp]
    L.ife_cuda_host_free.restype = None
    L.ife_cuda_comm_unique_id.argtypes = [vp, vp]
    L.ife_cuda_comm_init.argtypes = [vp, vp, i, i]
    L.ife_cuda_comm_destroy.argtypes = [vp]
    L.ife_cuda_slab_range.argtypes = [i, i, i, ip, ip]
    L.ife_cuda_slab_range.restype = None
    L.ife_cuda_slab_halo.argtypes = [d, d, d]
    L.ife_cuda_slab_emphysema_features.argtypes = [vp, vp, vp, vp, ip, dp, dp, i, vp, i, vp, d, i]
    L.ife_cuda_slab_emphysema_features_local.argtypes = [vp, vp, vp, i, i, i, i, vp, ip, dp, dp, i, vp, i,
                                                         vp, d, i]
    _lib = L
    return L


def declared_symbols():
    """Every function name include/ife_cuda.h declares (for the export test)."""
    import re
    text = open(HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ife_cuda_[a-z0-9_]+)\s*\(", text)))


def slab_range(nz, n_ranks, rank):
    """Planes [z0, z1) owned by `rank` (pure host arithmetic; same rule as the library)."""
    return nz * rank // n_ranks, nz * (rank + 1) // n_ranks


def slab_halo(sigma, spacing_z=1.0, halo_factor=12.0):
    import math
    return int(math.ceil(halo_factor * sigma / spacing_z)) + 5


def resampled_dims(dims, spacing, out_spacing):
    """(nx, ny, nz) of ife_cuda_resample's output grid: max(1, floor(n * s / s' + 0.5)) per axis in
    double, the library's rule (pure host arithmetic, for sizing device buffers)."""
    import math
    return tuple(max(1, int(math.floor(int(n) * float(s) / float(so) + 0.5)))
                 for n, s, so in zip(dims, spacing, out_spacing))


def _i3(dims):
    return (C.c_int * 3)(*[int(v) for v in dims])


def _d3(sp):
    return (C.c_double * 3)(*[float(v) for v in (sp if sp is not None else (1.0, 1.0, 1.0))])


def _dn(vals):
    vals = [float(v) for v in vals]
    return (C.c_double * len(vals))(*vals)


def _ptr(a):
    """host numpy array -> void*; None -> NULL; int -> itself (device pointer)."""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


def _dims_of(vol):
    nz, ny, nx = vol.shape
    return (nx, ny, nz)


class Context:
    """One ife_cuda_ctx: bound to one device and one stream; not thread-safe."""

    def __init__(self, device=0, arith=ARITH_FMA):
        self.L = load_library()
        h = C.c_void_p()
        rc = self.L.ife_cuda_create(device, C.byref(h))
        if rc != 0:
            raise IfeError(rc, "ife_cuda_create(device=%d) failed: no usable CUDA device "
                               "(there is no CPU fallback)" % device)
        self.h = h
        self.set_arith(arith)
        # A/B switches for the profiling scripts: IFE_CUDA_OPTIONS="march4=0,tma_passes=0"
        for kv in filter(None, os.environ.get("IFE_CUDA_OPTIONS", "").split(",")):
            name, _, val = kv.partition("=")
            self.set_option(name.strip(), int(val or 1))

    def close(self):
        if getattr(self, "h", None):
            self.L.ife_cuda_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise IfeError(rc, self.L.ife_cuda_last_error(self.h).decode())

    # ---- context control
    def set_arith(self, mode):
        self._check(self.L.ife_cuda_set_arith(self.h, mode))

    def set_stream(self, cuda_stream_handle):
        self._check(self.L.ife_cuda_set_stream(self.h, C.c_void_p(cuda_stream_handle or 0)))

    def set_option(self, name, value):
        self._check(self.L.ife_cuda_set_option(self.h, name.encode(), int(value)))

    def synchronize(self):
        self._check(self.L.ife_cuda_synchronize(self.h))

    def reserve(self, dims, n_outputs=0):
        self._check(self.L.ife_cuda_reserve(self.h, _i3(dims), n_outputs))

    def launch_count(self):
        return int(self.L.ife_cuda_launch_count(self.h))

    def last_work_dims(self):
        """(nx, ny, nz) the Gaussian passes of the last masked call ran on (crop or full volume)."""
        d = (C.c_int * 3)()
        self._check(self.L.ife_cuda_last_work_dims(self.h, d))
        return tuple(int(v) for v in d)

    PROFILE_KINDS = ["gauss_pass_z", "gauss_pass_x", "gauss_pass_y", "features_fused", "other",
                     "exchange_wait"]

    def profile_enable(self, on=True):
        self._check(self.L.ife_cuda_profile_enable(self.h, int(on)))

    def profile_read(self):
        """-> {kind: (total_ms, launches)} since the last read (synchronises)."""
        ms = (C.c_double * len(self.PROFILE_KINDS))()
        n = (C.c_uint64 * len(self.PROFILE_KINDS))()
        self._check(self.L.ife_cuda_profile_read(self.h, ms, n))
        return {k: (ms[j], int(n[j])) for j, k in enumerate(self.PROFILE_KINDS)}

    # ---- host-array conveniences (IFE_MEM_HOST); volumes are (nz, ny, nx) numpy arrays
    def gaussian(self, vol, sigma, spacing=None):
        vol = np.ascontiguousarray(vol, np.float32)
        out = np.empty_like(vol)
        self._check(self.L.ife_cuda_gaussian(self.h, _ptr(vol), _ptr(out), _i3(_dims_of(vol)),
                                             _d3(spacing), sigma, MEM_HOST))
        return out

    def normalized_gaussian(self, img, certainty, sigma, spacing=None, mask_output=False):
        img = np.ascontiguousarray(img, np.float32)
        out = np.empty_like(img)
        cf = cu = None
        if certainty.dtype == np.uint8:
            cu = np.ascontiguousarray(certainty)
        else:
            cf = np.ascontiguousarray(certainty, np.float32)
        self._check(self.L.ife_cuda_normalized_gaussian(
            self.h, _ptr(img), _ptr(cf), _ptr(cu), _ptr(out), _i3(_dims_of(img)), _d3(spacing),
            sigma, int(mask_output), MEM_HOST))
        return out

    def gradient_magnitude(self, vol, mask=None, spacing=None):
        vol = np.ascontiguousarray(vol, np.float32)
        out = np.empty_like(vol)
        mf = mu = None
        if mask is not None:
            if mask.dtype == np.uint8:
                mu = np.ascontiguousarray(mask)
            else:
                mf = np.ascontiguousarray(mask, np.float32)
        self._check(self.L.ife_cuda_gradient_magnitude(
            self.h, _ptr(vol), _ptr(mf), _ptr(mu), _ptr(out), _i3(_dims_of(vol)), _d3(spacing),
            MEM_HOST))
        return out

    def hessian(self, img, spacing=None):
        """itk::Hessian3DImageFilter: -> (6, nz, ny, nx) planes [Dxx, Dxy, Dxz, Dyy, Dyz, Dzz]."""
        img = np.ascontiguousarray(img, np.float32)
        out = np.empty((6,) + img.shape, np.float32)
        self._check(self.L.ife_cuda_hessian(self.h, _ptr(img), _ptr(out), _i3(_dims_of(img)), _d3(spacing), MEM_HOST))
        return out

    def hessian_eigen_features(self, img, mask=None, sigma=0.0, spacing=None, flags=0):
        img = np.ascontiguousarray(img, np.float32)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        out = np.empty((6,) + img.shape, np.float32)
        self._check(self.L.ife_cuda_hessian_eigen_features(
            self.h, _ptr(img), _ptr(m), _ptr(out), _i3(_dims_of(img)), _d3(spacing), sigma, flags,
            MEM_HOST))
        return out

    def emphysema_features(self, img, mask, sigmas, spacing=None, out=None, _raw_image=False):
        # _raw_image: pass the image buffer as it is (int16 with option "host_image_i16")
        img = np.ascontiguousarray(img) if _raw_image else np.ascontiguousarray(img, np.float32)
        mask = np.ascontiguousarray(mask, np.uint8)
        sigmas = list(sigmas)
        if out is None:
            out = np.empty((len(sigmas), 8) + img.shape, np.float32)
        self._check(self.L.ife_cuda_emphysema_features(
            self.h, _ptr(img), _ptr(mask), _ptr(out), _i3(_dims_of(img)), _d3(spacing),
            _dn(sigmas), len(sigmas), MEM_HOST))
        return out

    def emphysema_histograms(self, img, mask, sigmas, edges, rois=None, spacing=None, _raw_image=False):
        img = np.ascontiguousarray(img) if _raw_image else np.ascontiguousarray(img, np.float32)
        mask = np.ascontiguousarray(mask, np.uint8)
        sigmas = list(sigmas)
        edges = np.ascontiguousarray(edges, np.float32).reshape(len(sigmas) * 8, -1)
        r = None if rois is None else np.ascontiguousarray(rois, np.int32).reshape(-1, 6)
        R = 1 if r is None else r.shape[0]
        counts = np.zeros((R, len(sigmas) * 8, edges.shape[1] + 1), np.uint32)
        self._check(self.L.ife_cuda_emphysema_histograms(
            self.h, _ptr(img), _ptr(mask), _i3(_dims_of(img)), _d3(spacing), _dn(sigmas),
            len(sigmas), _ptr(edges), edges.shape[1], _ptr(r), 0 if r is None else R,
            _ptr(counts), MEM_HOST))
        return counts

    def emphysema_histograms_batch(self, images, masks, sigmas, edges, rois=None, spacing=None, _raw_image=False):
        """images / masks: lists of equally shaped (nz, ny, nx) host arrays (pinned memory makes
        the upload overlap real); rois: (n_scans, R, 6) or None -> counts (n_scans, R|1, S*8, E+1)"""
        images = [np.ascontiguousarray(a) if _raw_image else np.ascontiguousarray(a, np.float32) for a in images]
        masks = [np.ascontiguousarray(m, np.uint8) for m in masks]
        n = len(images)
        sigmas = list(sigmas)
        edges = np.ascontiguousarray(edges, np.float32).reshape(len(sigmas) * 8, -1)
        r = None if rois is None else np.ascontiguousarray(rois, np.int32).reshape(n, -1, 6)
        R = 1 if r is None else r.shape[1]
        counts = np.zeros((n, R, len(sigmas) * 8, edges.shape[1] + 1), np.uint32)
        ip_ = (C.c_void_p * n)(*[a.ctypes.data for a in images])
        mp_ = (C.c_void_p * n)(*[m.ctypes.data for m in masks])
        self._check(self.L.ife_cuda_emphysema_histograms_batch(
            self.h, n, ip_, mp_, _i3(_dims_of(images[0])), _d3(spacing), _dn(sigmas), len(sigmas),
            _ptr(edges), edges.shape[1], _ptr(r), 0 if r is None else R, _ptr(counts)))
        return counts

    def histogram(self, values, edges):
        values = np.ascontiguousarray(values, np.float32).ravel()
        edges = np.ascontiguousarray(edges, np.float32)
        counts = np.zeros(edges.size + 1, np.uint32)
        self._check(self.L.ife_cuda_histogram(self.h, _ptr(values) if values.size else None,
                                              values.size, _ptr(edges), edges.size, _ptr(counts),
                                              MEM_HOST))
        return counts

    def intensity_roi_histograms(self, image, mask, edges, rois):
        """-> counts (n_roi, n_edges+1): MakeBagOnlyIntensity's per-ROI intensity histograms"""
        image = np.ascontiguousarray(image, np.float32)
        mask = np.ascontiguousarray(mask, np.uint8)
        edges = np.ascontiguousarray(edges, np.float32).ravel()
        r = np.ascontiguousarray(rois, np.int32).reshape(-1, 6)
        counts = np.zeros((len(r), edges.size + 1), np.uint32)
        self._check(self.L.ife_cuda_intensity_roi_histograms(
            self.h, _ptr(image), _ptr(mask), _i3(_dims_of(image)), _ptr(edges), edges.size,
            _ptr(r) if len(r) else None, len(r), _ptr(counts), MEM_HOST))
        return counts

    def sort(self, values):
        v = np.array(values, np.float32).ravel()
        self._check(self.L.ife_cuda_sort_f32(self.h, _ptr(v) if v.size else None, v.size, MEM_HOST))
        return v

    def feature_samples(self, img, mask, sigmas, select=None, index=None, sort=False, spacing=None):
        """The 8 features at the selected voxels only: -> (n_sigma, 8, n_selected) rows, in voxel
        order (select: uint8 flags) or list order (index: voxel indices), optionally sorted."""
        img = np.ascontiguousarray(img, np.float32)
        m = np.ascontiguousarray(mask, np.uint8)
        sigmas = list(sigmas)
        sel = None if select is None else np.ascontiguousarray(select, np.uint8)
        idx = None if index is None else np.ascontiguousarray(index, np.int64)
        n_idx = 0 if idx is None else idx.size
        n_out = C.c_size_t(0)
        args = (self.h, _ptr(img), _ptr(m), _ptr(sel), _ptr(idx), n_idx, _i3(_dims_of(img)), _d3(spacing),
                _dn(sigmas), len(sigmas), 1 if sort else 0)
        self._check(self.L.ife_cuda_emphysema_feature_samples(*args, None, C.byref(n_out), MEM_HOST))
        out = np.empty((len(sigmas), 8, n_out.value), np.float32)
        if n_out.value:
            self._check(self.L.ife_cuda_emphysema_feature_samples(*args, _ptr(out), C.byref(n_out), MEM_HOST))
        return out

    def resample(self, vol, spacing, out_spacing, nearest=False, default=0.0):
        """(nz, ny, nx) float32 or uint8 volume at voxel spacing (sx, sy, sz) -> the volume resampled
        to out_spacing (linear: float32 only; nearest: float32 or uint8, the type is kept)."""
        vol = np.ascontiguousarray(vol)
        if vol.dtype not in (np.float32, np.uint8):
            raise TypeError("resample takes float32 or uint8 volumes, not %s" % vol.dtype)
        od = (C.c_int * 3)()
        args = (_i3(_dims_of(vol)), _d3(spacing), _d3(out_spacing), INTERP_NEAREST if nearest else INTERP_LINEAR,
                float(default), od, MEM_HOST)
        self._check(self.L.ife_cuda_resample(self.h, _ptr(vol), None, vol.dtype.itemsize, *args))  # sizes only
        out = np.empty((od[2], od[1], od[0]), vol.dtype)
        self._check(self.L.ife_cuda_resample(self.h, _ptr(vol), _ptr(out), vol.dtype.itemsize, *args))
        return out

    def eigen_features_batch(self, A6):
        A6 = np.ascontiguousarray(A6, np.float32).reshape(-1, 6)
        out = np.empty_like(A6)
        self._check(self.L.ife_cuda_eigen_features_batch(self.h, _ptr(A6), _ptr(out), A6.shape[0],
                                                         MEM_HOST))
        return out

    # ---- raw device-pointer calls (IFE_MEM_DEVICE); pointers are ints (tensor.data_ptr())
    def emphysema_features_dev(self, img_ptr, mask_ptr, out_ptr, dims, sigmas, spacing=None):
        sigmas = list(sigmas)
        self._check(self.L.ife_cuda_emphysema_features(
            self.h, _ptr(img_ptr), _ptr(mask_ptr), _ptr(out_ptr), _i3(dims), _d3(spacing),
            _dn(sigmas), len(sigmas), MEM_DEVICE))

    def emphysema_histograms_dev(self, img_ptr, mask_ptr, counts_ptr, dims, sigmas, edges,
                                 rois=None, spacing=None):
        sigmas = list(sigmas)
        edges = np.ascontiguousarray(edges, np.float32).reshape(len(sigmas) * 8, -1)
        r = None if rois is None else np.ascontiguousarray(rois, np.int32).reshape(-1, 6)
        self._check(self.L.ife_cuda_emphysema_histograms(
            self.h, _ptr(img_ptr), _ptr(mask_ptr), _i3(dims), _d3(spacing), _dn(sigmas),
            len(sigmas), _ptr(edges), edges.shape[1], _ptr(r), 0 if r is None else r.shape[0],
            _ptr(counts_ptr), MEM_DEVICE))

    def gaussian_dev(self, img_ptr, out_ptr, dims, sigma, spacing=None):
        self._check(self.L.ife_cuda_gaussian(self.h, _ptr(img_ptr), _ptr(out_ptr), _i3(dims), _d3(spacing),
                                             sigma, MEM_DEVICE))

    def normalized_gaussian_dev(self, img_ptr, cert_f32_ptr, out_ptr, dims, sigma, spacing=None, mask_output=False):
        self._check(self.L.ife_cuda_normalized_gaussian(self.h, _ptr(img_ptr), _ptr(cert_f32_ptr), None, _ptr(out_ptr),
                                                        _i3(dims), _d3(spacing), sigma, int(mask_output), MEM_DEVICE))

    def resample_dev(self, in_ptr, out_ptr, dims, spacing, out_spacing, elem_bytes=4, nearest=False,
                     default=0.0):
        """Device-pointer resample (enqueued on the context's stream) -> out_dims (nx, ny, nz);
        out_ptr=None only computes out_dims."""
        od = (C.c_int * 3)()
        self._check(self.L.ife_cuda_resample(
            self.h, _ptr(in_ptr), _ptr(out_ptr), elem_bytes, _i3(dims), _d3(spacing), _d3(out_spacing),
            INTERP_NEAREST if nearest else INTERP_LINEAR, float(default), od, MEM_DEVICE))
        return tuple(int(v) for v in od)

    def hessian_eigen_features_dev(self, img_ptr, mask_ptr, out_ptr, dims, sigma, spacing=None,
                                   flags=0):
        self._check(self.L.ife_cuda_hessian_eigen_features(
            self.h, _ptr(img_ptr), _ptr(mask_ptr), _ptr(out_ptr), _i3(dims), _d3(spacing), sigma,
            flags, MEM_DEVICE))

    # ---- multi-GPU
    def comm_unique_id(self):
        buf = (C.c_uint8 * COMM_ID_BYTES)()
        self._check(self.L.ife_cuda_comm_unique_id(self.h, buf))
        return bytes(buf)

    def comm_init(self, uid, n_ranks, rank):
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(uid)
        self._check(self.L.ife_cuda_comm_init(self.h, buf, n_ranks, rank))

    def comm_destroy(self):
        self._check(self.L.ife_cuda_comm_destroy(self.h))

    def slab_emphysema_features(self, img_slab, mask_slab, global_dims, sigmas, spacing=None,
                                edges=None, want_features=True, halo_factor=0.0):
        """Host-array form: img_slab (nzo, ny, nx) are the planes this rank owns."""
        img_slab = np.ascontiguousarray(img_slab, np.float32)
        m = None if mask_slab is None else np.ascontiguousarray(mask_slab, np.uint8)
        sigmas = list(sigmas)
        out = np.empty((len(sigmas), 8) + img_slab.shape, np.float32) if want_features else None
        e = counts = None
        n_edges = 0
        if edges is not None:
            e = np.ascontiguousarray(edges, np.float32).reshape(len(sigmas) * 8, -1)
            n_edges = e.shape[1]
            counts = np.zeros((len(sigmas) * 8, n_edges + 1), np.uint32)
        self._check(self.L.ife_cuda_slab_emphysema_features(
            self.h, _ptr(img_slab), _ptr(m), _ptr(out), _i3(global_dims), _d3(spacing),
            _dn(sigmas), len(sigmas), _ptr(e), n_edges, _ptr(counts), halo_factor, MEM_HOST))
        return out, counts

    def slab_emphysema_features_local(self, img_ext, mask_ext, ext_z0, own_z0, own_nz, global_dims,
                                      sigmas, spacing=None, edges=None, want_features=True,
                                      halo_factor=0.0):
        """No communication: img_ext (ext_nz, ny, nx) holds global planes from ext_z0 on."""
        img_ext = np.ascontiguousarray(img_ext, np.float32)
        m = None if mask_ext is None else np.ascontiguousarray(mask_ext, np.uint8)
        sigmas = list(sigmas)
        shape = (own_nz,) + img_ext.shape[1:]
        out = np.empty((len(sigmas), 8) + shape, np.float32) if want_features else None
        e = counts = None
        n_edges = 0
        if edges is not None:
            e = np.ascontiguousarray(edges, np.float32).reshape(len(sigmas) * 8, -1)
            n_edges = e.shape[1]
            counts = np.zeros((len(sigmas) * 8, n_edges + 1), np.uint32)
        self._check(self.L.ife_cuda_slab_emphysema_features_local(
            self.h, _ptr(img_ext), _ptr(m), ext_z0, img_ext.shape[0], own_z0, own_nz, _ptr(out),
            _i3(global_dims), _d3(spacing), _dn(sigmas), len(sigmas), _ptr(e), n_edges, _ptr(counts),
            halo_factor, MEM_HOST))
        return out, counts

    def slab_emphysema_features_dev(self, img_ptr, mask_ptr, out_ptr, global_dims, sigmas,
                                    spacing=None, edges=None, counts_ptr=None, halo_factor=0.0):
        sigmas = list(sigmas)
        e = None
        n_edges = 0
        if edges is not None:
            e = np.ascontiguousarray(edges, np.float32).reshape(len(sigmas) * 8, -1)
            n_edges = e.shape[1]
        self._check(self.L.ife_cuda_slab_emphysema_features(
            self.h, _ptr(img_ptr), _ptr(mask_ptr), _ptr(out_ptr), _i3(global_dims), _d3(spacing),
            _dn(sigmas), len(sigmas), _ptr(e), n_edges, _ptr(counts_ptr), halo_factor, MEM_DEVICE))
