"""Every kernel variant the C ABI selects, each asserted by the kernels that actually ran.

The library chooses its kernels from layout facts of each call: nx % 4 / 16 / 32, the 16-byte
(or 4-byte) alignment of every pointer, the mask's support box, the number of histogram edges
and the number of ROIs.  Host-pointer calls always hand the kernels the library's own aligned
workspace buffers, so the alignment fallbacks only run for device pointers (IFE_MEM_DEVICE, the
path framework callers take).  These tests
  A. record which kernels a call launched (torch.profiler, CUDA activities);
  B. call every IFE_MEM_DEVICE entry point at 16-byte-aligned and at offset pointers and require
     the host call's result, asserting which variant each layout selects;
  C. run the support-box windows on the full volume (no crop) against the same call without a
     box and against the oracle;
  D. put histogram values exactly on edges for every binning implementation;
  E. fill the 8-bit private counters of both z-marching kernels to their caps.
"""
import ctypes as C
import json
import re

import numpy as np
import pytest

import ife_b200
import synth
from ife_b200 import MEM_DEVICE, _d3, _dn, _i3
from test_gpu_parity import assert_eigen_parity, bits_equal, mismatch_report

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


# ------------------------------------------------------------------------------ A: which kernels ran
_KERNEL = re.compile(r"\bife::(\w+)[<(]")
_trace_no = [0]


def ran(ctx, tmp_path, fn):
    """Run fn() under torch.profiler (CUDA activities), ending with ctx.synchronize().
    -> (fn's result, set of the library's kernel names that ran, e.g. {"iir_tma_kernel"})."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        result = fn()
        ctx.synchronize()
    _trace_no[0] += 1
    path = tmp_path / ("trace%d.json" % _trace_no[0])
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    names = set()
    for e in events:
        if str(e.get("cat", "")).lower() == "kernel":
            m = _KERNEL.search(e.get("name", ""))
            if m:
                names.add(m.group(1))
    return result, names


def test_profiler_records_library_kernels(ctx, tmp_path):
    vol = synth.ct_like((16, 32, 64), seed=1, n_blobs=3)
    out, names = ran(ctx, tmp_path, lambda: ctx.gaussian(vol, 1.0))
    assert "iir_tma_kernel" in names, "no library kernel in the trace: %s" % sorted(names)
    assert "gauss_pass_x" not in names and "gauss_pass_strided" not in names
    assert np.isfinite(out).all()


# ------------------------------------------------------------------------------ device buffers
def dev(a, off=0):
    """Device copy of numpy array `a` whose data pointer sits `off` bytes past an allocation start
    (the caching allocator's blocks are at least 512-byte aligned)."""
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    if off == 0:
        return t
    k = off // t.element_size()
    assert k * t.element_size() == off
    buf = torch.empty(t.numel() + k, dtype=t.dtype, device="cuda")
    v = buf[k:k + t.numel()].view(t.shape)
    v.copy_(t)
    return v


def dev_out(shape, dtype, off=0):
    fill = float("nan") if dtype == torch.float32 else (0x5A if dtype == torch.uint8 else 0x5A5A5A5A)
    return dev(torch.full(shape, fill, dtype=dtype).numpy(), off)


def P(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def dims_of(shape):
    return _i3((shape[2], shape[1], shape[0]))


SP = _d3(None)
NXS = (64, 48, 36, 37)
# byte offsets of (float inputs, uint8 inputs, outputs); 0 = 16-byte aligned
LAYOUTS = [(0, 0, 0), (4, 0, 0), (0, 1, 0), (0, 4, 0), (0, 0, 4), (4, 1, 4), (4, 4, 4)]


def blob(shape, c, r):
    zz, yy, xx = np.ogrid[:shape[0], :shape[1], :shape[2]]
    d = sum(((g - ci) / ri) ** 2 for g, ci, ri in zip((zz, yy, xx), c, r))
    return (d <= 1).astype(np.uint8)


def scan(nx, seed=0):
    """(16, 48, nx) CT-like image, a blob mask well inside (labels 1 and 2), its support box a
    crop when nx % 32 == 0."""
    shape = (16, 48, nx)
    img = synth.ct_like(shape, seed=100 + nx + seed, n_blobs=6)
    m = blob(shape, (8, 15, 0.55 * nx), (5, 8, 0.27 * nx))
    m[:, :, : nx // 2] *= 2
    return img, m


def same(got, want, what):
    got = got.cpu().numpy() if hasattr(got, "cpu") else got
    assert got.shape == want.shape, what
    if got.dtype.kind == "f":
        n, worst = mismatch_report(got, want)
        assert n == 0, "%s: %d values differ from the host call (max %.3g)" % (what, n, worst)
    else:
        assert np.array_equal(got, want), "%s: counts differ from the host call" % what


def al(off):
    return off % 16 == 0


def masked_variants(names, nx, fo, uo, what):
    """The support box / crop / pass family / features kernel rules of a masked call whose kernels
    read the context's blur buffer (aligned) and the caller's uint8 mask at offset uo."""
    box = nx % 16 == 0 and al(uo)
    assert ("mask_box_kernel" in names) == box, what
    # scan()'s mask is cropped whenever the layout allows a crop
    assert ("crop_box_kernel" in names) == (box and nx % 32 == 0 and al(fo)), what
    cropped = "crop_box_kernel" in names
    tma = cropped or (nx % 16 == 0 and al(fo) and al(uo))
    assert ("iir_tma_kernel" in names) == tma, what
    if not tma:
        assert {"gauss_pass_x", "gauss_pass_strided"} <= names, what
    return cropped


def march_variant(names, march4, what):
    if march4:
        assert "features_march4_kernel" in names and "features_march_kernel" not in names, what
    else:
        assert "features_march_kernel" in names and "features_march4_kernel" not in names, what
    assert "features_kernel" not in names, what


# ------------------------------------------------------------------------------ B: device pointers
def test_gaussian_device_layouts(ctx, oracle, tmp_path):
    for nx in NXS:
        img, _ = scan(nx)
        host = ctx.gaussian(img, 1.3)
        assert mismatch_report(host, oracle.smoothing_recursive_gaussian(img, 1.3, arith=1))[0] == 0
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_in, d_out = dev(img, fo), dev_out(img.shape, torch.float32, oo)
            _, names = ran(ctx, tmp_path, lambda: ctx._check(ctx.L.ife_cuda_gaussian(
                ctx.h, P(d_in), P(d_out), dims_of(img.shape), SP, 1.3, MEM_DEVICE)))
            same(d_out, host, what)
            tma = nx % 4 == 0 and al(fo) and al(oo)
            assert ("iir_tma_kernel" in names) == tma, what
            assert tma or "gauss_pass_x" in names, what


@pytest.mark.parametrize("cert", ["u8", "f32"])
@pytest.mark.parametrize("mask_output", [0, 1])
def test_normalized_gaussian_device_layouts(ctx, oracle, tmp_path, cert, mask_output):
    for nx in NXS:
        img, m = scan(nx)
        if cert == "u8":
            c = m
        else:
            c = np.random.default_rng(nx).uniform(0.1, 1, m.shape).astype(np.float32) * (m != 0)
        host = ctx.normalized_gaussian(img, c, 1.2, mask_output=bool(mask_output))
        ref = oracle.normalized_gaussian(img, c.astype(np.float32), 1.2, arith=1)
        if mask_output:
            ref = np.where(c != 0, ref, np.float32(0))
        assert mismatch_report(host, ref)[0] == 0
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_img, d_out = dev(img, fo), dev_out(img.shape, torch.float32, oo)
            d_cu = dev(c, uo) if cert == "u8" else None
            d_cf = dev(c, fo) if cert == "f32" else None
            _, names = ran(ctx, tmp_path, lambda: ctx._check(ctx.L.ife_cuda_normalized_gaussian(
                ctx.h, P(d_img), P(d_cf), P(d_cu), P(d_out), dims_of(img.shape), SP, 1.2, mask_output,
                MEM_DEVICE)))
            same(d_out, host, what)
            cert_ok = (nx % 16 == 0 and al(uo)) if cert == "u8" else (nx % 4 == 0 and al(fo))
            tma = cert_ok and al(fo) and al(oo)
            assert ("iir_tma_kernel" in names) == tma, what
            assert tma or "gauss_pass_x" in names, what


@pytest.mark.parametrize("mask", [None, "u8", "f32"])
def test_gradient_magnitude_device_layouts(ctx, tmp_path, mask):
    for nx in NXS:
        img, m = scan(nx)
        mk = None if mask is None else (m if mask == "u8" else m.astype(np.float32))
        host = ctx.gradient_magnitude(img, mk)
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_img, d_out = dev(img, fo), dev_out(img.shape, torch.float32, oo)
            d_mu = dev(mk, uo) if mask == "u8" else None
            d_mf = dev(mk, fo) if mask == "f32" else None
            _, names = ran(ctx, tmp_path, lambda: ctx._check(ctx.L.ife_cuda_gradient_magnitude(
                ctx.h, P(d_img), P(d_mf), P(d_mu), P(d_out), dims_of(img.shape), SP, MEM_DEVICE)))
            same(d_out, host, what)
            if mask == "f32":
                assert "features_kernel" in names, what
                assert not names & {"features_march_kernel", "features_march4_kernel"}, what
            else:
                m4 = nx % 4 == 0 and al(fo) and al(oo) and (mask is None or uo % 4 == 0)
                march_variant(names, m4, what)


def test_hessian_device_layouts(ctx, tmp_path):
    for nx in NXS:
        img, _ = scan(nx)
        host = ctx.hessian(img)
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_img, d_out = dev(img, fo), dev_out((6,) + img.shape, torch.float32, oo)
            _, names = ran(ctx, tmp_path, lambda: ctx._check(ctx.L.ife_cuda_hessian(
                ctx.h, P(d_img), P(d_out), dims_of(img.shape), SP, MEM_DEVICE)))
            same(d_out, host, what)
            march_variant(names, nx % 4 == 0 and al(fo) and al(oo), what)


@pytest.mark.parametrize("sigma", [0.0, 1.2])
def test_hessian_eigen_features_device_layouts(ctx, tmp_path, sigma):
    for nx in NXS:
        img, m = scan(nx)
        host = ctx.hessian_eigen_features(img, m, sigma=sigma)
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_img, d_m = dev(img, fo), dev(m, uo)
            d_out = dev_out((6,) + img.shape, torch.float32, oo)
            _, names = ran(ctx, tmp_path, lambda: ctx._check(ctx.L.ife_cuda_hessian_eigen_features(
                ctx.h, P(d_img), P(d_m), P(d_out), dims_of(img.shape), SP, sigma, 0, MEM_DEVICE)))
            same(d_out, host, what)
            vol_ok = sigma > 0 or al(fo)          # with sigma > 0 the stencil reads the blur buffer
            march_variant(names, nx % 4 == 0 and vol_ok and uo % 4 == 0 and al(oo), what)
            if sigma > 0:
                assert ("iir_tma_kernel" in names) == (nx % 4 == 0 and al(fo)), what


@pytest.mark.parametrize("sigmas", [[1.0], [0.6, 1.2, 2.4]])
def test_emphysema_features_device_layouts(ctx, oracle, tmp_path, sigmas):
    for nx in NXS:
        img, m = scan(nx)
        dims = (nx, img.shape[1], img.shape[0])
        host = ctx.emphysema_features(img, m, sigmas)
        if len(sigmas) == 1:           # the variants below all equal the host call: tie it to the oracle
            ref = oracle.emphysema_features(img, m, sigmas[0], arith=1)
            assert mismatch_report(host[0, :2], ref[:2])[0] == 0
            assert_eigen_parity(np.moveaxis(host[0, 2:], 0, -1), np.moveaxis(ref[2:], 0, -1), "nx=%d" % nx)
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_img, d_m = dev(img, fo), dev(m, uo)
            d_out = dev_out((len(sigmas), 8) + img.shape, torch.float32, oo)
            _, names = ran(ctx, tmp_path, lambda: ctx._check(ctx.L.ife_cuda_emphysema_features(
                ctx.h, P(d_img), P(d_m), P(d_out), dims_of(img.shape), SP, _dn(sigmas), len(sigmas),
                MEM_DEVICE)))
            same(d_out, host, what)
            cropped = masked_variants(names, nx, fo, uo, what)
            if not cropped:
                assert ctx.last_work_dims() == dims, what
            march_variant(names, nx % 4 == 0 and uo % 4 == 0 and al(oo), what)
            if nx == 64 and (fo, uo, oo) == (4, 0, 0):    # box windows on the full volume, plain passes
                assert {"mask_box_kernel", "gauss_pass_x", "gauss_pass_strided"} <= names
                assert "crop_box_kernel" not in names and "iir_tma_kernel" not in names


@pytest.mark.parametrize("kind", ["none", "six", "many"])
def test_emphysema_histograms_device_layouts(ctx, tmp_path, kind):
    for nx in NXS:
        img, m = scan(nx)
        F = ctx.emphysema_features(img, m, [0.6, 1.2])
        edges = np.stack([synth.equalized_edges(F[s, k][m != 0], 12) for s in range(2) for k in range(8)])
        rois = None
        if kind == "six":
            rois = synth.random_rois(m, 6, (7, 5, 3), seed=nx)
        elif kind == "many":
            rois = np.ascontiguousarray(synth.dense_rois(m, (5, 3, 3))[::2])
            assert len(rois) > 192
        host = ctx.emphysema_histograms(img, m, [0.6, 1.2], edges, rois)
        assert host.sum() > 0
        n_roi = 0 if rois is None else len(rois)
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_img, d_m = dev(img, fo), dev(m, uo)
            d_c = dev_out(host.shape, torch.int32, oo)
            _, names = ran(ctx, tmp_path, lambda: ctx._check(ctx.L.ife_cuda_emphysema_histograms(
                ctx.h, P(d_img), P(d_m), dims_of(img.shape), SP, _dn([0.6, 1.2]), 2, edges.ctypes.data_as(C.c_void_p),
                edges.shape[1], None if rois is None else rois.ctypes.data_as(C.c_void_p), n_roi, P(d_c),
                MEM_DEVICE)))
            same(d_c.cpu().numpy().view(np.uint32), host, what)
            cropped = masked_variants(names, nx, fo, uo, what)
            if kind == "six":
                assert "features_kernel" in names, what
            else:
                # the fused kernel reads the blur buffer and, on a crop, the cropped mask
                march_variant(names, nx % 4 == 0 and (cropped or uo % 4 == 0), what)
            assert ("roi_hist_packed_kernel" in names) == (kind == "many"), what


def test_flat_and_intensity_histograms_device_layouts(ctx, tmp_path):
    for nx in NXS:
        img, m = scan(nx)
        img = np.round(img / 16).astype(np.float32)
        edges = np.arange(-60, 40, 3, dtype=np.float32)
        rois = np.concatenate([synth.random_rois(m, 40, (9, 7, 5), seed=nx), [[0, 0, 0, nx, 48, 16]]]).astype(np.int32)
        h_flat = ctx.histogram(img, edges)
        h_roi = ctx.intensity_roi_histograms(img, m, edges, rois)
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_img, d_m = dev(img, fo), dev(m, uo)
            d_c = dev_out(h_flat.shape, torch.int32, oo)
            d_r = dev_out(h_roi.shape, torch.int32, oo)
            ep = edges.ctypes.data_as(C.c_void_p)
            _, names = ran(ctx, tmp_path, lambda: (
                ctx._check(ctx.L.ife_cuda_histogram(ctx.h, P(d_img), img.size, ep, edges.size, P(d_c), MEM_DEVICE)),
                ctx._check(ctx.L.ife_cuda_intensity_roi_histograms(
                    ctx.h, P(d_img), P(d_m), dims_of(img.shape), ep, edges.size, rois.ctypes.data_as(C.c_void_p),
                    len(rois), P(d_r), MEM_DEVICE))))
            same(d_c.cpu().numpy().view(np.uint32), h_flat, what)
            same(d_r.cpu().numpy().view(np.uint32), h_roi, what)
            assert {"histogram_kernel", "roi_intensity_hist_kernel"} <= names, what


def test_sort_and_eigen_batch_device_layouts(ctx):
    rng = np.random.default_rng(9)
    v = rng.normal(0, 50, 10_007).astype(np.float32)
    v[::13] = 0.0
    v[::17] = -0.0
    v[::11] = 3.25
    host_sorted = ctx.sort(v)
    A6 = synth.special_matrices(5003, seed=4)
    host_eig = ctx.eigen_features_batch(A6)
    for fo, _, oo in LAYOUTS:
        d = dev(v, fo)
        torch.cuda.synchronize()
        ctx._check(ctx.L.ife_cuda_sort_f32(ctx.h, P(d), v.size, MEM_DEVICE))
        ctx.synchronize()
        assert np.array_equal(d.cpu().numpy().view(np.uint32), host_sorted.view(np.uint32)), (fo, oo)
        d_a, d_o = dev(A6, fo), dev_out(A6.shape, torch.float32, oo)
        torch.cuda.synchronize()
        ctx._check(ctx.L.ife_cuda_eigen_features_batch(ctx.h, P(d_a), P(d_o), A6.shape[0], MEM_DEVICE))
        ctx.synchronize()
        same(d_o, host_eig, (fo, oo))


@pytest.mark.parametrize("how", ["select", "index"])
def test_feature_samples_device_layouts(ctx, tmp_path, how):
    sigmas = [0.6, 2.4]
    for nx in NXS:
        img, m = scan(nx)
        rng = np.random.default_rng(nx)
        sel = ((m != 0) & (rng.uniform(0, 1, m.shape) < 0.5)).astype(np.uint8)
        idx = rng.integers(0, img.size, 3001).astype(np.int64)
        host = ctx.feature_samples(img, m, sigmas, select=sel) if how == "select" else \
            ctx.feature_samples(img, m, sigmas, index=idx)
        n_sel = host.shape[2]
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_img, d_m = dev(img, fo), dev(m, uo)
            d_sel = dev(sel, uo) if how == "select" else None
            d_idx = dev(idx) if how == "index" else None       # int64 list: natural alignment
            d_out = dev_out(host.shape, torch.float32, oo)
            n_out = C.c_size_t(0)
            _, names = ran(ctx, tmp_path, lambda: ctx._check(ctx.L.ife_cuda_emphysema_feature_samples(
                ctx.h, P(d_img), P(d_m), P(d_sel), P(d_idx), 0 if d_idx is None else idx.size,
                dims_of(img.shape), SP, _dn(sigmas), 2, 0, P(d_out), C.byref(n_out), MEM_DEVICE)))
            assert n_out.value == n_sel, what
            same(d_out, host, what)
            masked_variants(names, nx, fo, uo, what)


def test_slab_local_device_layouts(ctx, tmp_path):
    sigmas = [0.6, 1.2]
    for nx in NXS:
        img, m = scan(nx)
        gdims = (nx, img.shape[1], img.shape[0])
        F = ctx.emphysema_features(img, m, sigmas)
        edges = np.stack([synth.equalized_edges(F[s, k][m != 0], 10) for s in range(2) for k in range(8)])
        e0, e1, z0, z1 = 1, 15, 4, 12
        h_out, h_cnt = ctx.slab_emphysema_features_local(img[e0:e1], m[e0:e1], e0, z0, z1 - z0, gdims, sigmas,
                                                         edges=edges)
        for fo, uo, oo in LAYOUTS:
            what = "nx=%d layout=%s" % (nx, (fo, uo, oo))
            d_img, d_m = dev(img[e0:e1], fo), dev(m[e0:e1], uo)
            d_out = dev_out(h_out.shape, torch.float32, oo)
            d_c = dev_out(h_cnt.shape, torch.int32, oo)
            _, names = ran(ctx, tmp_path, lambda: ctx._check(ctx.L.ife_cuda_slab_emphysema_features_local(
                ctx.h, P(d_img), P(d_m), e0, e1 - e0, z0, z1 - z0, P(d_out), _i3(gdims), SP, _dn(sigmas), 2,
                edges.ctypes.data_as(C.c_void_p), edges.shape[1], P(d_c), 0.0, MEM_DEVICE)))
            same(d_out, h_out, what)
            same(d_c.cpu().numpy().view(np.uint32), h_cnt, what)
            march_variant(names, nx % 4 == 0 and uo % 4 == 0 and al(oo), what)
            assert ("iir_tma_kernel" in names) == (nx % 16 == 0 and al(fo) and al(uo)), what


def test_resample_device_layouts(ctx):
    for nx in NXS:
        img, m = scan(nx)
        sp, osp = (0.8, 0.9, 1.5), (0.7, 1.1, 1.0)       # output rows of 73/55/41/42 voxels
        for vol, nearest in ((img, False), (img, True), (m, True)):
            host = ctx.resample(vol, sp, osp, nearest=nearest)
            eb = vol.dtype.itemsize
            for fo, uo, oo in ((0, 0, 0), (4, 1, 4), (0, 4, 4), (4, 0, 0), (0, 0, 4)):
                io = fo if eb == 4 else uo
                d_in = dev(vol, io)
                d_out = dev_out(host.shape, torch.float32 if eb == 4 else torch.uint8, oo if eb == 4 else uo)
                od = ctx.resample_dev(d_in.data_ptr(), None, (nx, 48, 16), sp, osp, eb, nearest)
                assert od == (host.shape[2], host.shape[1], host.shape[0])
                torch.cuda.synchronize()
                ctx.resample_dev(d_in.data_ptr(), d_out.data_ptr(), (nx, 48, 16), sp, osp, eb, nearest)
                ctx.synchronize()
                got = d_out.cpu().numpy()
                assert np.array_equal(got.view(np.uint8), host.view(np.uint8)), (nx, nearest, eb, fo, uo, oo)
        # output rows of 64 voxels: the 16-byte store path at +0 and its fallback at +4 B
        out4 = (0.8 * nx / 64, 0.9, 1.5)
        host = ctx.resample(img, sp, out4)
        assert host.shape[2] == 64
        for oo in (0, 4):
            d_in, d_out = dev(img), dev_out(host.shape, torch.float32, oo)
            torch.cuda.synchronize()
            ctx.resample_dev(d_in.data_ptr(), d_out.data_ptr(), (nx, 48, 16), sp, out4)
            ctx.synchronize()
            same(d_out, host, "resample nx=%d out +%d B" % (nx, oo))


def test_calls_on_a_caller_stream(ctx):
    """Routed to a torch stream: device calls and then a torch op on that stream that reads their
    output, with no synchronisation of the context in between."""
    img, m = scan(64)
    sigmas = [0.6, 1.2]
    ref = ctx.emphysema_features(img, m, sigmas)
    ref_g = ctx.gaussian(img, 2.0)
    d_img, d_m = dev(img, 4), dev(m, 1)
    out = torch.empty((2, 8) + img.shape, dtype=torch.float32, device="cuda")
    g = torch.empty(img.shape, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    ctx.set_stream(s.cuda_stream)
    try:
        with torch.cuda.stream(s):
            ctx._check(ctx.L.ife_cuda_emphysema_features(ctx.h, P(d_img), P(d_m), P(out), dims_of(img.shape), SP,
                                                         _dn(sigmas), 2, MEM_DEVICE))
            ctx.gaussian_dev(d_img.data_ptr(), g.data_ptr(), (64, 48, 16), 2.0)
            res = out * 1.0
            res_g = g + 0.0
            got, got_g = res.cpu().numpy(), res_g.cpu().numpy()
    finally:
        ctx.set_stream(None)
    assert bits_equal(got, ref)
    assert bits_equal(got_g, ref_g)


# ------------------------------------------------------------------------------ C: box windows, no crop
def _case_c(name):
    """The tensor-map passes write whole chunks of 16 samples (iir_tma.cuh: chunks [k_lo, kA) with
    kA = ceil(out_hi / 16)), so a y window that ends one row short only shows when the box ends one
    row past a chunk boundary: the boxes below end at y = 33 (C1, mask rows 14..31) and y = 17
    (C2, ROI rows up to 15), and the stencil of the last wanted row reads the first row of a chunk
    that only the full window writes."""
    rng = np.random.default_rng(7)
    if name == "c1":       # nx % 16 == 0, nx % 32 != 0: no crop, z and y windows, tensor-map u8 passes
        shape = (24, 40, 80)
        mask = blob(shape, (12, 22.5, 41), (6, 9, 15))
        rois2 = np.array([[30, 14, 9, 9, 7, 5], [40, 18, 12, 11, 9, 6]], np.int32)
        y_end = int(np.nonzero(mask.any((0, 2)))[0].max()) + 1
    else:                  # nx = 256: the crop would be 87.5 % of the volume; y pass x window [32, 256)
        shape = (24, 32, 256)
        mask = np.zeros(shape, np.uint8)
        mask[:, :, 40:250] = rng.uniform(0, 1, (24, 32, 210)) < 0.7
        mask[:, :, 120:170] = 1
        rois2 = np.array([[100, 5, 4, 9, 7, 5], [104, 8, 9, 8, 8, 6]], np.int32)    # narrow in x
        y_end = int((rois2[:, 1] + rois2[:, 4]).max())
    assert (y_end + 1) % 16 == 1, y_end      # the box's y end (grown by one row) is 16 m + 1
    img = synth.ct_like(shape, seed=71, n_blobs=10)
    return shape, img, mask, rois2


def _pollute_blur(ctx, shape):
    """Overwrite the context's blur buffer with unrelated values: a windowed call must not rely on
    what a previous full-volume call left outside its windows."""
    noise = np.random.default_rng(3).normal(0, 300, shape).astype(np.float32)
    ctx.hessian_eigen_features(noise, None, sigma=1.0)


def _without_box(ctx, fn):
    ctx.set_option("support_box", 0)
    try:
        return fn()
    finally:
        ctx.set_option("support_box", 1)


@pytest.mark.parametrize("case", ["c1", "c2", "c3"])
def test_box_windows_without_a_crop(ctx, oracle, tmp_path, case):
    shape, img, mask, rois2 = _case_c("c2" if case == "c3" else case)
    dims = (shape[2], shape[1], shape[0])
    sigmas = [0.6, 2.4]
    if case == "c3":
        ctx.set_option("tma_passes", 0)
    try:
        def windowed(fn):
            _pollute_blur(ctx, shape)
            out, names = ran(ctx, tmp_path, fn)
            assert ctx.last_work_dims() == dims
            assert "mask_box_kernel" in names and "crop_box_kernel" not in names, sorted(names)
            if case == "c3":
                assert "iir_tma_kernel" not in names and {"gauss_pass_x", "gauss_pass_strided"} <= names
            else:
                assert "iir_tma_kernel" in names
            _pollute_blur(ctx, shape)
            return out

        out = windowed(lambda: ctx.emphysema_features(img, mask, sigmas))
        full = _without_box(ctx, lambda: ctx.emphysema_features(img, mask, sigmas))
        assert bits_equal(out, full)
        assert np.all(out[:, :, mask == 0] == 0)
        for s, sigma in enumerate(sigmas):
            ref = oracle.emphysema_features(img, mask, sigma, arith=1)
            assert mismatch_report(out[s, 0], ref[0])[0] == 0, "blur sigma=%g" % sigma
            assert mismatch_report(out[s, 1], ref[1])[0] == 0, "gradient sigma=%g" % sigma
            assert_eigen_parity(np.moveaxis(out[s, 2:], 0, -1), np.moveaxis(ref[2:], 0, -1), "sigma=%g" % sigma)

        edges = np.stack([synth.equalized_edges(out[s, k][mask != 0], 12) for s in range(2) for k in range(8)])
        many = synth.dense_rois(mask[:, :, :], (3, 3, 3))
        many = many[(many[:, 0] >= rois2[:, 0].min()) & (many[:, 0] < rois2[:, 0].max() + 4)][::3]
        assert len(many) > 192
        for rois in (None, rois2, many):
            got = windowed(lambda: ctx.emphysema_histograms(img, mask, sigmas, edges, rois))
            ref = _without_box(ctx, lambda: ctx.emphysema_histograms(img, mask, sigmas, edges, rois))
            assert np.array_equal(got, ref) and got.sum() > 0
        img2 = synth.ct_like(shape, seed=72, n_blobs=10)
        roisb = np.stack([rois2, rois2 + np.array([2, 1, 1, 0, 0, 0], np.int32)])
        for rb in (None, roisb):
            got = windowed(lambda: ctx.emphysema_histograms_batch([img, img2], [mask, mask], sigmas, edges, rb))
            ref = _without_box(ctx, lambda: ctx.emphysema_histograms_batch([img, img2], [mask, mask], sigmas,
                                                                            edges, rb))
            assert np.array_equal(got, ref) and got.sum() > 0
    finally:
        ctx.set_option("tma_passes", 1)


# ------------------------------------------------------------------------------ D: values on edges
def bins_of(row, v):
    """bin = number of edges < value (NaN: 0), the DenseHistogram rule"""
    b = np.searchsorted(row, v, side="left")
    b[np.isnan(v)] = 0
    return b


def tie_edges(F, mask, n_edges):
    """Per feature row: n_edges values that occur in F[k][mask != 0], sorted, one of them twice."""
    rows = []
    for k in range(F.shape[0]):
        u = np.unique(F[k][mask != 0])
        u = u[np.isfinite(u)]
        assert len(u) >= n_edges, (k, len(u))
        pick = u[np.round(np.linspace(0, len(u) - 1, n_edges - 1)).astype(int)]
        rows.append(np.sort(np.concatenate([pick, pick[len(pick) // 2: len(pick) // 2 + 1]])))
    return np.stack(rows).astype(np.float32)


def ref_counts(F, mask, edges, rois=None):
    """(R or 1, rows, E+1) counts of the in-mask voxels (of each ROI box)"""
    nz, ny, nx = mask.shape
    boxes = [(0, 0, 0, nx, ny, nz)] if rois is None else rois
    out = np.zeros((len(boxes), F.shape[0], edges.shape[1] + 1), np.uint32)
    for r, (x, y, z, sx, sy, sz) in enumerate(boxes):
        sel = mask[z:z + sz, y:y + sy, x:x + sx] != 0
        for k in range(F.shape[0]):
            v = F[k, z:z + sz, y:y + sy, x:x + sx][sel]
            out[r, k] = np.bincount(bins_of(edges[k], v), minlength=edges.shape[1] + 1)
    return out


D_SHAPE = (24, 40, 64)


@pytest.fixture(scope="module")
def d_scan(ctx):
    img = synth.ct_like(D_SHAPE, seed=55, n_blobs=10)
    mask = synth.lung_mask(D_SHAPE)
    F = ctx.emphysema_features(img, mask, [1.2])[0]
    return img, mask, F


def _hist(ctx, tmp_path, d_scan, n_edges, rois=None):
    img, mask, F = d_scan
    edges = tie_edges(F, mask, n_edges)
    got, names = ran(ctx, tmp_path, lambda: ctx.emphysema_histograms(img, mask, [1.2], edges, rois))
    want = ref_counts(F, mask, edges, rois)
    assert np.array_equal(got, want), "n_edges=%d: %d counts differ" % (n_edges, int((got != want).sum()))
    return names


@pytest.mark.parametrize("n_edges", [12, 40, 80])
def test_ties_march4_sink(ctx, tmp_path, d_scan, n_edges):
    names = _hist(ctx, tmp_path, d_scan, n_edges)
    march_variant(names, True, n_edges)


@pytest.mark.parametrize("n_edges", [40, 80])
def test_ties_march_sink(ctx, tmp_path, d_scan, n_edges):
    ctx.set_option("march4", 0)
    try:
        names = _hist(ctx, tmp_path, d_scan, n_edges)
    finally:
        ctx.set_option("march4", 1)
    march_variant(names, False, n_edges)


@pytest.mark.parametrize("n_edges", [120, 479])
def test_ties_brick_sink(ctx, tmp_path, d_scan, n_edges):
    img, mask, F = d_scan
    rois = synth.random_rois(mask, 6, (11, 9, 7), seed=4)
    names = _hist(ctx, tmp_path, d_scan, n_edges, rois)
    assert "features_kernel" in names and "roi_hist_packed_kernel" not in names
    names = _hist(ctx, tmp_path, d_scan, n_edges)      # no ROIs: too many edges for the march sink
    assert "features_kernel" in names
    with pytest.raises(ife_b200.IfeError) as e:
        ctx.emphysema_histograms(img, mask, [1.2], tie_edges(F, mask, 480), rois)
    assert e.value.code == -1


def test_ties_brick_sink_crowded_roi_list(ctx, tmp_path, d_scan):
    """150 near-identical boxes: more ROIs touch one brick than its list holds (96), so the
    brick walks the whole list."""
    img, mask, F = d_scan
    base = np.array([20, 12, 8, 12, 10, 8], np.int32)
    rois = np.stack([base + np.array([i % 3, (i // 3) % 2, (i // 6) % 2, 0, 0, 0], np.int32) for i in range(150)])
    names = _hist(ctx, tmp_path, d_scan, 40, rois)
    assert "features_kernel" in names


@pytest.mark.parametrize("n_edges", [40, 91, 92])
def test_ties_packed_sink(ctx, tmp_path, d_scan, n_edges):
    img, mask, F = d_scan
    rois = synth.dense_rois(mask, (5, 3, 3))[::7]
    assert len(rois) > 192
    names = _hist(ctx, tmp_path, d_scan, n_edges, rois)
    if n_edges <= 91:
        assert "roi_hist_packed_kernel" in names and "features_kernel" not in names
    else:
        assert "features_kernel" in names and "roi_hist_packed_kernel" not in names


def _intensity_case():
    shape = (20, 24, 40)
    nz, ny, nx = shape
    rng = np.random.default_rng(12)
    img = rng.integers(-3100, 3101, shape).astype(np.float32)
    r = rng.uniform(0, 1, shape)
    img[r < 0.4] = rng.integers(-35, 36, int((r < 0.4).sum()))
    img[(r >= 0.4) & (r < 0.5)] = 0.0
    img[(r >= 0.5) & (r < 0.6)] = -0.0
    mask = rng.integers(0, 3, shape).astype(np.uint8)
    rois = [[0, 0, 0, nx, ny, nz]]
    rois += [[x, y, z, 1, 1, 1] for z in (0, nz - 1) for y in (0, ny - 1) for x in (0, nx - 1)]
    rois += [[0, 3, 4, 5, 6, 7], [nx - 5, 3, 4, 5, 6, 7], [3, 0, 4, 5, 6, 7], [3, ny - 6, 4, 5, 6, 7],
             [3, 4, 0, 5, 6, 7], [3, 4, nz - 7, 5, 6, 7]]
    rois += [[2, 3, 1, 35, 4, 3]]                                 # sx > 32, sy * sz > 8
    sx, sy, sz = rng.integers(1, 16, 1000), rng.integers(1, 12, 1000), rng.integers(1, 10, 1000)
    rois += np.stack([rng.integers(0, nx - sx + 1), rng.integers(0, ny - sy + 1), rng.integers(0, nz - sz + 1),
                      sx, sy, sz], 1).tolist()
    return img, mask, np.array(rois, np.int32)


@pytest.mark.parametrize("n_edges", [1, 63, 6143])
def test_ties_intensity_and_flat_histograms(ctx, n_edges):
    img, mask, rois = _intensity_case()
    lo = -(n_edges // 2)
    row = np.arange(lo, lo + n_edges, dtype=np.float32)
    assert 0.0 in row
    neg = row.copy()
    neg[row == 0] = -0.0                                          # -0.0 as an edge
    assert np.signbit(neg[neg == 0]).all()
    for edges in (row, neg):
        got = ctx.intensity_roi_histograms(img, mask, edges, rois)
        for r, (x, y, z, sx, sy, sz) in enumerate(rois):
            v = img[z:z + sz, y:y + sy, x:x + sx][mask[z:z + sz, y:y + sy, x:x + sx] != 0]
            want = np.bincount(bins_of(edges, v), minlength=n_edges + 1)
            assert np.array_equal(got[r], want), "ROI %d %s" % (r, rois[r])
        for v in (img.ravel(), img.ravel()[:1], img.ravel()[:1001], img.ravel()[7:7 + 4099]):
            want = np.bincount(bins_of(edges, v), minlength=n_edges + 1)
            assert np.array_equal(ctx.histogram(v, edges), want), (n_edges, v.size)


def test_histogram_edge_limit(ctx):
    img, mask, rois = _intensity_case()
    edges = np.arange(6144, dtype=np.float32)
    for call in (lambda: ctx.intensity_roi_histograms(img, mask, edges, rois[:3]),
                 lambda: ctx.histogram(img, edges)):
        with pytest.raises(ife_b200.IfeError) as e:
            call()
        assert e.value.code == -1


# ------------------------------------------------------------------------------ E: full counters
def march4_zchunk(nx, ny, nz, sm_count):
    """launch_features (csrc/ife_cuda.cu), four voxels per thread: planes per block before the
    63-plane cap of the 8-bit private counters."""
    cols = -(-nx // 128) * -(-ny // 4)
    want = -(-8 * 4 * sm_count // cols)
    return min(max(16, -(-nz // want)), nz)


def march_zchunk(nx, ny, nz, sm_count):
    """launch_features, one voxel per thread: planes per block before the 255 cap."""
    cols = -(-nx // 32) * -(-ny // 4)
    want = -(-8 * (1024 // 128) * sm_count // cols)
    zc = min(max(16, -(-nz // want)), nz)
    return min(zc, (1 << 31) // (nx * ny) - 2)


@pytest.mark.parametrize("which", ["march4", "march"])
def test_private_counters_at_their_caps(tmp_path, which):
    """A flat image in an all-ones mask: every voxel lands in bin 1 of every row.  Were a private
    8-bit counter to see 256 voxels, the row would come out short by a multiple of 256."""
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    if which == "march4":
        nz, ny, nx = 640, 512, 512
        assert march4_zchunk(nx, ny, nz, sm) > 63          # the cap binds
    else:
        nz, ny, nx = 256, 1184, 1024
        assert march_zchunk(nx, ny, nz, sm) > 255
    n = nz * ny * nx
    img = torch.full((nz, ny, nx), -800.0, dtype=torch.float32, device="cuda")
    mask = torch.ones((nz, ny, nx), dtype=torch.uint8, device="cuda")
    counts = torch.zeros((1, 8, 3), dtype=torch.int32, device="cuda")
    edges = np.array([[-801.0, -799.0]] + [[-1.0, 1.0]] * 7, np.float32)
    torch.cuda.synchronize()
    c = ife_b200.Context(0)
    try:
        if which == "march":
            c.set_option("march4", 0)
        _, names = ran(c, tmp_path, lambda: c.emphysema_histograms_dev(
            img.data_ptr(), mask.data_ptr(), counts.data_ptr(), (nx, ny, nz), [1.0], edges))
        got = counts.cpu().numpy().view(np.uint32)
    finally:
        c.close()
    march_variant(names, which == "march4", which)
    assert np.all(got[0, :, 1] == n), "bin 1 holds %s of %d voxels" % (got[0, :, 1].tolist(), n)
    assert np.all(got[0, :, 0] == 0) and np.all(got[0, :, 2] == 0)
