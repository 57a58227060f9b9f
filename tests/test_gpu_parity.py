"""GPU parity tests: the CUDA path, called through the C ABI with host buffers, against the
CPU oracle on the same seeded inputs.

Bar (BASELINE.json north_star): eigenvalues within 1e-4 * max|lambda| per voxel with the
same ordering; histogram counts exact except for voxels within that tolerance of an edge.
What is asserted here is stronger: every stage is BIT-IDENTICAL to the oracle run in the
same arithmetic mode, except that the solver's double-precision acos/cos are polynomial
kernels within ~1 ulp of glibc's instead of glibc itself, which after narrowing to float may
flip the last bit of an eigenvalue for a vanishing fraction of voxels (<= MISMATCH_FRAC,
each still within TOL; currently none is observed).
"""
import numpy as np
import pytest

import synth

pytestmark = pytest.mark.gpu

TOL = 1e-4            # relative to max|lambda| per voxel (north_star)
MISMATCH_FRAC = 2e-5  # allowed fraction of last-bit differences (libm vs the polynomial acos/cos)


def bits_equal(a, b):
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def mismatch_report(gpu, ref):
    """(#elements that differ, max |diff|) with NaN == NaN and -0 == +0."""
    neq = ~((gpu == ref) | (np.isnan(gpu) & np.isnan(ref)))
    n = int(neq.sum())
    return n, (float(np.max(np.abs(gpu[neq].astype(np.float64) - ref[neq]))) if n else 0.0)


def assert_eigen_parity(gpu6, ref6, what):
    """gpu6/ref6: (..., 6) features [e1,e2,e3,LoG,Curv,Frob]."""
    g = gpu6.reshape(-1, 6); r = ref6.reshape(-1, 6)
    finite = np.isfinite(r).all(1)
    assert np.array_equal(np.isnan(g), np.isnan(r)), what
    neq_rows = (~((g == r) | (np.isnan(g) & np.isnan(r)))).any(1)
    frac = neq_rows.mean()
    assert frac <= MISMATCH_FRAC, "%s: %.3g of voxels differ" % (what, frac)
    rows = neq_rows & finite
    if rows.any():
        lam = np.abs(r[rows, :3]).max(1)
        err = np.abs(g[rows, :3].astype(np.float64) - r[rows, :3]).max(1)
        assert np.all(err <= TOL * lam), "%s: eigenvalue error beyond 1e-4*max|lambda|" % what


# ------------------------------------------------------------------------------ solver
def test_solver_batch_matches_reference_golden(ctx):
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "solver_ref.npz"))
    out = ctx.eigen_features_batch(g["A6"])
    assert_eigen_parity(out, g["features_f32"], "golden")
    # diagonal / tie cases never touch a transcendental: exactly equal
    diag = (g["A6"][:, [1, 2, 4]] == 0).all(1)
    assert bits_equal(out[diag], g["features_f32"][diag])


def test_solver_batch_matches_oracle_2M(ctx, oracle):
    A = synth.special_matrices(2_000_000, seed=21)
    out = ctx.eigen_features_batch(A)
    ref = oracle.features_f32(A)
    assert_eigen_parity(out, ref, "2M sweep")
    n, _ = mismatch_report(out, ref)
    print("solver sweep: %d of %d values differ from the oracle" % (n, out.size))
    # the reference's own known answers (test/Symmetric3x3EigenvalueSolverTest.cxx:48-90)
    kat = np.array([[1, 0, 0, 1, 0, 1], [1, 0, 0, 2, 0, 3], [-1, 0, 0, -2, 0, -3], [1, 0, 0, -2, 0, 3],
                    [0.27, 0.92, 0.58, 0.24, 0.75, 0.04], [599, 860, -835, -941, 817, -207]], np.float32)
    exp = np.array([[1, 1, 1], [3, 2, 1], [-3, -2, -1], [3, -2, 1],
                    [1.70680634, -0.7205504, -0.43625594], [-2005.21004566, 1183.41690727, 272.79313839]])
    got = ctx.eigen_features_batch(kat)[:, :3]
    assert np.allclose(got, exp, rtol=2e-6, atol=1e-6)
    assert ctx.eigen_features_batch(np.zeros((0, 6), np.float32)).shape == (0, 6)


# ------------------------------------------------------------------------------ smoothing
@pytest.mark.parametrize("arith", [0, 1])
@pytest.mark.parametrize("shape,sigma", [((40, 48, 64), 1.0), ((4, 4, 4), 0.6), ((5, 17, 33), 2.4),
                                         ((37, 16, 130), 4.8), ((19, 21, 23), 1.2)])
def test_gaussian_bit_exact(ctx, oracle, arith, shape, sigma):
    vol = synth.ct_like(shape, seed=2, n_blobs=6)
    ctx.set_arith(arith)
    try:
        out = ctx.gaussian(vol, sigma)
    finally:
        ctx.set_arith(1)
    ref = oracle.smoothing_recursive_gaussian(vol, sigma, arith=arith)
    n, worst = mismatch_report(out, ref)
    assert n == 0, "%d voxels differ (max %.3g)" % (n, worst)


def test_gaussian_anisotropic_and_errors(ctx, oracle):
    import ife_b200
    vol = synth.ct_like((20, 24, 28), seed=5, n_blobs=4)
    sp = (0.7, 0.7, 2.5)
    assert bits_equal(ctx.gaussian(vol, 2.0, spacing=sp),
                      oracle.smoothing_recursive_gaussian(vol, 2.0, spacing=sp, arith=1))
    with pytest.raises(ife_b200.IfeError) as e:
        ctx.gaussian(vol[:3], 1.0)          # ITK throws for < 4 samples per line
    assert e.value.code == -2
    with pytest.raises(ife_b200.IfeError) as e:
        ctx.gaussian(vol, 0.0)
    assert e.value.code == -1


@pytest.mark.parametrize("arith", [0, 1])
def test_normalized_gaussian_bit_exact(ctx, oracle, arith):
    shape = (36, 40, 44)
    img = synth.ct_like(shape, seed=7, n_blobs=8)
    m8 = synth.clamp01(synth.lung_mask(shape))
    ctx.set_arith(arith)
    try:
        out_u8 = ctx.normalized_gaussian(img, m8, 1.2)
        cert = np.random.default_rng(0).uniform(0, 1, shape).astype(np.float32)
        cert[m8 == 0] = 0
        out_f = ctx.normalized_gaussian(img, cert, 2.4)
        out_fm = ctx.normalized_gaussian(img, cert, 2.4, mask_output=True)
    finally:
        ctx.set_arith(1)
    ref_u8 = oracle.normalized_gaussian(img, m8.astype(np.float32), 1.2, arith=arith)
    ref_f = oracle.normalized_gaussian(img, cert, 2.4, arith=arith)
    assert mismatch_report(out_u8, ref_u8)[0] == 0
    assert mismatch_report(out_f, ref_f)[0] == 0
    assert mismatch_report(out_fm, np.where(cert != 0, ref_f, np.float32(0)))[0] == 0


@pytest.mark.parametrize("arith", [0, 1])
def test_tensor_map_passes_bit_exact(ctx, oracle, arith):
    """The tensor-map staged, field-per-warp passes (csrc/iir_tma.cuh; taken when nx % 16 == 0
    with a uint8 certainty) against the plain register-staged passes and the oracle: whole tiles, ragged
    tiles in every direction (nx, ny not multiples of 32, lines that are not whole chunks),
    lines shorter than one chunk, the smallest volume ITK accepts."""
    shapes = [((40, 64, 96), 1.2), ((37, 45, 48), 2.4), ((4, 4, 16), 0.6), ((5, 6, 32), 1.0),
              ((16, 16, 16), 4.8), ((33, 32, 64), 0.6), ((19, 70, 80), 1.0), ((130, 20, 16), 4.8)]
    ctx.set_arith(arith)
    try:
        for shape, sigma in shapes:      # shape = (nz, ny, nx)
            img = synth.ct_like(shape, seed=sum(shape), n_blobs=6)
            m8 = synth.clamp01(synth.lung_mask(shape))
            if min(shape) < 8:
                m8 = (np.random.default_rng(3).uniform(0, 1, shape) < 0.7).astype(np.uint8)
            got = ctx.normalized_gaussian(img, m8, sigma)
            ctx.set_option("tma_passes", 0)
            try:
                old = ctx.normalized_gaussian(img, m8, sigma)
            finally:
                ctx.set_option("tma_passes", 1)
            n, worst = mismatch_report(got, old)
            assert n == 0, "%s sigma=%g: %d values differ from the plain passes (max %g)" % (shape, sigma, n, worst)
            if np.prod(shape) < 200_000:
                ref = oracle.normalized_gaussian(img, m8.astype(np.float32), sigma, arith=arith)
                assert mismatch_report(got, ref)[0] == 0, "%s sigma=%g vs oracle" % (shape, sigma)
        # mask values other than 0/1 (the filter casts, it does not clamp)
        shape = (24, 40, 64)
        img = synth.ct_like(shape, seed=5, n_blobs=5)
        m8 = np.random.default_rng(4).integers(0, 4, shape).astype(np.uint8)
        got = ctx.normalized_gaussian(img, m8, 1.5)
        assert mismatch_report(got, oracle.normalized_gaussian(img, m8.astype(np.float32), 1.5, arith=arith))[0] == 0
    finally:
        ctx.set_arith(1)


@pytest.mark.parametrize("arith", [1, 0])
def test_tensor_map_plain_gaussian_bit_exact(ctx, oracle, arith):
    """One field through the tensor-map kernels (nx % 4 == 0): the second warp of a block takes a
    second stack of rows (upper half of y in the z pass, upper half of the planes in the x and y
    passes).  Odd row / plane counts (the halves differ by one), ragged tiles, short lines."""
    shapes = [((40, 64, 96), 1.2), ((37, 45, 48), 2.4), ((4, 4, 16), 0.6), ((5, 7, 32), 1.0), ((16, 16, 16), 4.8),
              ((33, 31, 64), 0.6), ((19, 70, 84), 1.0), ((130, 21, 20), 4.8), ((9, 5, 4), 0.6)]
    ctx.set_arith(arith)
    try:
        for shape, sigma in shapes:      # shape = (nz, ny, nx)
            img = synth.ct_like(shape, seed=sum(shape) + 1, n_blobs=6)
            got = ctx.gaussian(img, sigma)
            ctx.set_option("tma_passes", 0)
            try:
                old = ctx.gaussian(img, sigma)
            finally:
                ctx.set_option("tma_passes", 1)
            n, worst = mismatch_report(got, old)
            assert n == 0, "%s sigma=%g: %d values differ from the plain passes (max %g)" % (shape, sigma, n, worst)
            if np.prod(shape) < 200_000:
                ref = oracle.smoothing_recursive_gaussian(img, sigma, arith=arith)
                assert mismatch_report(got, ref)[0] == 0, "%s sigma=%g vs oracle" % (shape, sigma)
        # anisotropic spacing, and the consumer of the plain Gaussian: Hessian eigen features at sigma > 0
        shape = (21, 40, 64)
        img = synth.ct_like(shape, seed=8, n_blobs=5)
        sp = (0.7, 0.7, 1.3)
        assert mismatch_report(ctx.gaussian(img, 1.1, spacing=sp), oracle.smoothing_recursive_gaussian(img, 1.1, spacing=sp, arith=arith))[0] == 0
    finally:
        ctx.set_arith(1)


@pytest.mark.parametrize("arith", [1, 0])
def test_tensor_map_float_certainty_bit_exact(ctx, oracle, arith):
    """NormalizedGaussianConvolutionImageFilter's own signature, (float T, float c) -> float, through the
    tensor-map kernels (nx % 4 == 0, no output mask): fractional certainties, zero certainties, ragged tiles."""
    shapes = [((40, 64, 96), 1.2), ((37, 45, 48), 2.4), ((4, 4, 16), 0.6), ((5, 7, 36), 1.0), ((33, 31, 20), 0.6),
              ((19, 70, 84), 4.8)]
    ctx.set_arith(arith)
    try:
        for shape, sigma in shapes:      # shape = (nz, ny, nx)
            img = synth.ct_like(shape, seed=sum(shape) + 2, n_blobs=6)
            rng = np.random.default_rng(sum(shape))
            cert = rng.uniform(0, 1, shape).astype(np.float32)
            cert[rng.uniform(0, 1, shape) < 0.3] = 0.0
            got = ctx.normalized_gaussian(img, cert, sigma)
            ctx.set_option("tma_passes", 0)
            try:
                old = ctx.normalized_gaussian(img, cert, sigma)
            finally:
                ctx.set_option("tma_passes", 1)
            n, worst = mismatch_report(got, old)
            assert n == 0, "%s sigma=%g: %d values differ from the plain passes (max %g)" % (shape, sigma, n, worst)
            if np.prod(shape) < 200_000:
                ref = oracle.normalized_gaussian(img, cert, sigma, arith=arith)
                assert mismatch_report(got, ref)[0] == 0, "%s sigma=%g vs oracle" % (shape, sigma)
        # the output mask (the tool's -m flag) is applied where the y pass divides: same answer as masking
        # afterwards and as the plain kernels, float and uint8 certainty, ragged tiles
        for shape in ((24, 40, 64), (21, 37, 48), (9, 50, 16)):
            img = synth.ct_like(shape, seed=9, n_blobs=5)
            for cert in ((np.random.default_rng(6).uniform(0, 1, shape) < 0.6).astype(np.float32),
                         (np.random.default_rng(7).uniform(0, 1, shape) < 0.5).astype(np.uint8)):
                plain = ctx.normalized_gaussian(img, cert, 1.5)
                masked = ctx.normalized_gaussian(img, cert, 1.5, mask_output=True)
                assert bits_equal(masked, np.where(cert != 0, plain, np.float32(0)))
                ctx.set_option("tma_passes", 0)
                try:
                    assert bits_equal(masked, ctx.normalized_gaussian(img, cert, 1.5, mask_output=True))
                finally:
                    ctx.set_option("tma_passes", 1)
    finally:
        ctx.set_arith(1)


def test_normalized_gaussian_zero_divisor_rule(ctx, oracle):
    # certainty identically zero -> G(c) == 0 -> itk::DivideImageFilter yields float max
    img = synth.ct_like((8, 8, 8), seed=1, n_blobs=2)
    zero = np.zeros((8, 8, 8), np.uint8)
    out = ctx.normalized_gaussian(img, zero, 1.0)
    assert np.all(out == np.finfo(np.float32).max)
    assert bits_equal(out, oracle.normalized_gaussian(img, zero.astype(np.float32), 1.0, arith=1))


# ------------------------------------------------------------------------------ stencils
def test_gradient_magnitude_bit_exact(ctx, oracle):
    shape = (21, 33, 47)
    img = synth.ct_like(shape, seed=8, n_blobs=5)
    assert bits_equal(ctx.gradient_magnitude(img), oracle.gradient_magnitude(img))
    m = synth.lung_mask(shape).astype(np.float32)      # the tool reads the mask as float
    assert bits_equal(ctx.gradient_magnitude(img, m), oracle.fd_gradient_features(img, m))
    sp = (0.8, 1.25, 3.0)
    assert bits_equal(ctx.gradient_magnitude(img, spacing=sp), oracle.gradient_magnitude(img, spacing=sp))


def test_hessian_six_components_bit_exact(ctx, oracle):
    """itk::Hessian3DImageFilter on its own (ife_cuda_hessian): the six stencil outputs
    [Dxx, Dxy, Dxz, Dyy, Dyz, Dzz] (Hessian3DImageFilter.hxx:53-59) against oracle.hessian6, unit
    and anisotropic spacing, ragged sizes, the clamped edge planes included."""
    for shape, sp, seed in (((20, 24, 32), None, 3), ((9, 13, 37), None, 4), ((16, 40, 64), (0.7, 0.8, 2.5), 5),
                            ((4, 4, 4), None, 6), ((5, 7, 3), (1.0, 2.0, 0.5), 7)):
        vol = synth.ct_like(shape, seed=seed, n_blobs=5)
        got = ctx.hessian(vol, spacing=sp)
        ref = np.moveaxis(oracle.hessian6(vol, spacing=sp), -1, 0)
        assert got.shape == ref.shape
        n, worst = mismatch_report(got, ref)
        assert n == 0, "%s spacing %s: %d Hessian entries differ (max %g)" % (shape, sp, n, worst)
        # the edge planes are where ZeroFluxNeumann matters: spot-check them explicitly
        for ax in (1, 2, 3):
            assert bits_equal(np.take(got, [0, -1], axis=ax), np.take(ref, [0, -1], axis=ax))
    # the eigen features of ife_cuda_hessian_eigen_features are the functor applied to this output
    vol = synth.ct_like((12, 16, 32), seed=9, n_blobs=4)
    H = ctx.hessian(vol)
    feats = ctx.eigen_features_batch(np.ascontiguousarray(np.moveaxis(H, 0, -1).reshape(-1, 6)))
    fused = np.moveaxis(ctx.hessian_eigen_features(vol), 0, -1).reshape(-1, 6)
    assert bits_equal(feats, fused)


def test_fd_hessian_features_tool_semantics(ctx, oracle):
    import ife_b200
    shape = (30, 34, 38)
    img = synth.ct_like(shape, seed=9, n_blobs=6)
    mask = synth.lung_mask(shape)          # labels {0,1,2}: the tool tests mask == 0
    out = ctx.hessian_eigen_features(img, mask)
    ref = oracle.fd_hessian_features(img, mask)
    assert np.all(out[:, mask == 0] == 0)
    assert_eigen_parity(np.moveaxis(out, 0, -1), np.moveaxis(ref, 0, -1), "fdhf")
    out = ctx.hessian_eigen_features(img, None, flags=ife_b200.FDHF_TOOL_DY_BUG)
    ref = oracle.fd_hessian_features(img, None, fdhf_tool_bug=True)
    assert_eigen_parity(np.moveaxis(out, 0, -1), np.moveaxis(ref, 0, -1), "fdhf dy-bug")
    sp = (0.6, 0.6, 1.5)
    out = ctx.hessian_eigen_features(img, mask, spacing=sp)
    ref = oracle.fd_hessian_features(img, mask, spacing=sp)
    assert_eigen_parity(np.moveaxis(out, 0, -1), np.moveaxis(ref, 0, -1), "fdhf anisotropic")
    # a constant image has an exactly zero Hessian: diagonal branch, all features 0
    flat = np.full(shape, -1000.0, np.float32)
    assert np.all(ctx.hessian_eigen_features(flat) == 0)


def test_config0_128cube_sigma1(ctx, oracle):
    """BASELINE.json configs[0]: FiniteDifference_HessianFeatures on a synthetic 128^3 float
    volume, single sigma = 1.0 (smooth with the library Gaussian, then the tool)."""
    shape = (128, 128, 128)
    img = synth.ct_like(shape, seed=1)
    out = ctx.hessian_eigen_features(img, None, sigma=1.0)
    ref = oracle.fd_hessian_features(img, None, sigma=1.0, arith=1)
    assert_eigen_parity(np.moveaxis(out, 0, -1), np.moveaxis(ref, 0, -1), "config 0")
    n, worst = mismatch_report(out, ref)
    print("config0: %d of %d output values differ from the oracle (max abs %.3g)" % (n, out.size, worst))
    e = out[:3].reshape(3, -1)
    tol = 1e-5 * np.abs(e).max(0)
    assert np.all(np.abs(e[0]) >= np.abs(e[1]) - tol) and np.all(np.abs(e[1]) >= np.abs(e[2]) - tol)


# ------------------------------------------------------------------------------ full feature stack
@pytest.mark.parametrize("arith", [0, 1])
def test_emphysema_features_multiscale(ctx, oracle, arith):
    shape = (48, 56, 72)
    sigmas = [0.6, 1.2, 2.4, 4.8]
    img = synth.ct_like(shape, seed=10, n_blobs=12)
    mask = synth.clamp01(synth.lung_mask(shape))
    ctx.set_arith(arith)
    try:
        out = ctx.emphysema_features(img, mask, sigmas)
    finally:
        ctx.set_arith(1)
    assert out.shape == (4, 8) + shape
    for s, sigma in enumerate(sigmas):
        ref = oracle.emphysema_features(img, mask, sigma, arith=arith)
        assert np.all(out[s][:, mask == 0] == 0)
        assert mismatch_report(out[s, 0], ref[0])[0] == 0, "blur sigma=%g" % sigma
        assert mismatch_report(out[s, 1], ref[1])[0] == 0, "gradient magnitude sigma=%g" % sigma
        assert_eigen_parity(np.moveaxis(out[s, 2:], 0, -1), np.moveaxis(ref[2:], 0, -1),
                            "eigen features sigma=%g" % sigma)


def test_emphysema_features_ragged_and_all_ones_mask(ctx, oracle):
    shape = (7, 13, 35)
    img = synth.ct_like(shape, seed=12, n_blobs=3)
    ones = np.ones(shape, np.uint8)
    out = ctx.emphysema_features(img, ones, [1.0])[0]
    ref = oracle.emphysema_features(img, ones, 1.0, arith=1)
    assert mismatch_report(out[:2], ref[:2])[0] == 0
    assert_eigen_parity(np.moveaxis(out[2:], 0, -1), np.moveaxis(ref[2:], 0, -1), "ragged")
    none = np.zeros(shape, np.uint8)
    assert np.all(ctx.emphysema_features(img, none, [1.0]) == 0)


def test_emphysema_features_anisotropic_spacing(ctx, oracle):
    """Real CT is anisotropic (sigma is in mm, ImageToEmphysemaFeaturesFilter.h:57): the whole
    stack -- three passes with per-axis sigma/spacing, the general-spacing branch of the fused
    kernel, the histogram sink -- against the oracle at spacing (0.7, 0.7, 2.5), with the
    support box on (nx % 32 == 0) and off (ragged nx)."""
    sp = (0.7, 0.7, 2.5)
    for shape, seed in (((24, 64, 96), 51), ((20, 37, 45), 52)):
        img = synth.ct_like(shape, seed=seed, n_blobs=8)
        mask = synth.clamp01(synth.lung_mask(shape))
        for sigma in (1.0, 2.4):
            out = ctx.emphysema_features(img, mask, [sigma], spacing=sp)[0]
            ref = oracle.emphysema_features(img, mask, sigma, spacing=sp, arith=1)
            assert np.all(out[:, mask == 0] == 0)
            assert mismatch_report(out[:2], ref[:2])[0] == 0, "blur / gradient magnitude %s sigma=%g" % (shape, sigma)
            assert_eigen_parity(np.moveaxis(out[2:], 0, -1), np.moveaxis(ref[2:], 0, -1),
                                "anisotropic %s sigma=%g" % (shape, sigma))
        feats = oracle.emphysema_features(img, mask, 1.0, spacing=sp, arith=1)
        edges = np.stack([synth.equalized_edges(feats[k][mask != 0], 12) for k in range(8)])
        got = ctx.emphysema_histograms(img, mask, [1.0], edges, spacing=sp)
        ref_counts = oracle.features_histograms(feats, mask, edges)
        assert np.abs(got.astype(np.int64) - ref_counts.astype(np.int64)).sum() <= 2


def test_support_box_is_invisible_to_both_pass_families(ctx, oracle):
    """Masked paths smooth only the mask's bounding box grown by the stencil reach (lines that
    miss it are skipped, the sweeps along a line stop at it).  No result may change: the same
    call with the option off, the same call through the plain pass kernels instead of the
    tensor-map ones, and the oracle give identical outputs; an empty mask and a mask touching
    the volume corner work too."""
    shape = (40, 64, 96)                      # nz, ny, nx: every pass takes its tensor-map kernel
    sigmas = [0.6, 2.4]
    img = synth.ct_like(shape, seed=31, n_blobs=10)
    zz, yy, xx = np.ogrid[:shape[0], :shape[1], :shape[2]]
    blob = (((zz - 27) / 6.0) ** 2 + ((yy - 20) / 9.0) ** 2 + ((xx - 70) / 11.0) ** 2 <= 1).astype(np.uint8)
    corner = np.zeros(shape, np.uint8); corner[:3, :2, :5] = 1; corner[-1, -1, -1] = 1
    for mask in (blob, corner):
        out = ctx.emphysema_features(img, mask, sigmas)
        ctx.set_option("support_box", 0)
        try:
            full = ctx.emphysema_features(img, mask, sigmas)
        finally:
            ctx.set_option("support_box", 1)
        assert bits_equal(out, full)
        assert np.all(out[:, :, mask == 0] == 0)
    for s, sigma in enumerate(sigmas):        # `out` is the corner mask's result
        ref = oracle.emphysema_features(img, corner, sigma, arith=1)
        assert mismatch_report(out[s, :2], ref[:2])[0] == 0
        assert_eigen_parity(np.moveaxis(out[s, 2:], 0, -1), np.moveaxis(ref[2:], 0, -1), "box sigma=%g" % sigma)
    assert np.all(ctx.emphysema_features(img, np.zeros(shape, np.uint8), sigmas) == 0)
    ctx.set_option("tma_passes", 0)           # the plain pass kernels take the same windows
    try:
        assert bits_equal(ctx.emphysema_features(img, corner, sigmas), out)
    finally:
        ctx.set_option("tma_passes", 1)
    # histograms: the box is also clipped to the ROI list's bounding box
    edges = _edges_for(oracle, img, blob, sigmas, 12)
    rois = np.array([[60, 12, 22, 9, 7, 5], [72, 20, 26, 11, 9, 6]], np.int32)   # x,y,z,sx,sy,sz
    for r in (None, rois):
        got = ctx.emphysema_histograms(img, blob, sigmas, edges, r)
        ctx.set_option("support_box", 0)
        try:
            full = ctx.emphysema_histograms(img, blob, sigmas, edges, r)
        finally:
            ctx.set_option("support_box", 1)
        assert np.array_equal(got, full)
    assert got.sum() > 0
    many = synth.dense_rois(blob, (7, 5, 3))[::3]          # > 192 ROIs: packed-bin path, on the crop
    assert len(many) > 192
    got = ctx.emphysema_histograms(img, blob, sigmas, edges, many)
    ctx.set_option("support_box", 0)
    try:
        full = ctx.emphysema_histograms(img, blob, sigmas, edges, many)
    finally:
        ctx.set_option("support_box", 1)
    assert np.array_equal(got, full) and got.sum() > 0
    roisb = np.stack([rois, rois + np.array([3, 2, 1, 0, 0, 0], np.int32)])
    bothr = ctx.emphysema_histograms_batch([img, img], [blob, blob], sigmas, edges, roisb)
    assert np.array_equal(bothr[0], ctx.emphysema_histograms(img, blob, sigmas, edges, roisb[0]))
    assert np.array_equal(bothr[1], ctx.emphysema_histograms(img, blob, sigmas, edges, roisb[1]))
    both = ctx.emphysema_histograms_batch([img, img], [blob, corner], sigmas, edges)
    assert np.array_equal(both[0], ctx.emphysema_histograms(img, blob, sigmas, edges))
    assert np.array_equal(both[1], ctx.emphysema_histograms(img, corner, sigmas, edges))


def test_support_box_finite_input_precondition(ctx):
    """include/ife_cuda.h documents the one way option "support_box" can change a result: a NaN
    voxel OUTSIDE the mask's box.  The full-volume path multiplies it by the zero certainty
    (0 * NaN = NaN) and the recursion carries it into the mask, as the reference would; the
    cropped path never reads it and gives the result of the image with that voxel cleared."""
    shape = (40, 64, 96)
    img = synth.ct_like(shape, seed=33, n_blobs=8)
    zz, yy, xx = np.ogrid[:shape[0], :shape[1], :shape[2]]
    mask = (((zz - 20) / 6.0) ** 2 + ((yy - 30) / 9.0) ** 2 + ((xx - 40) / 11.0) ** 2 <= 1).astype(np.uint8)
    bad = img.copy()
    bad[20, 30, 90] = np.nan                     # same row as the blob's centre, far outside its box
    clean = img.copy()
    clean[20, 30, 90] = 0.0
    with_box = ctx.emphysema_features(bad, mask, [1.2])
    assert np.isfinite(with_box).all() and bits_equal(with_box, ctx.emphysema_features(clean, mask, [1.2]))
    ctx.set_option("support_box", 0)
    try:
        full = ctx.emphysema_features(bad, mask, [1.2])
    finally:
        ctx.set_option("support_box", 1)
    assert np.isnan(full[0, 0][mask != 0]).any()  # the reference's behaviour: the NaN reaches in-mask voxels


def test_overlap_scales_same_results(ctx):
    """Option overlap_scales (device-resident calls): the Gaussian passes run one scale ahead
    on a second stream, the feature kernel of the scale before beside them, two blur buffers
    and events in between.  Same bits as the serial schedule, call after call."""
    torch = pytest.importorskip("torch")
    shape = (40, 64, 96)
    sigmas = [0.6, 1.2, 2.4, 4.8, 1.0]
    img = torch.from_numpy(synth.ct_like(shape, seed=41, n_blobs=10)).cuda()
    mask = torch.from_numpy(synth.clamp01(synth.lung_mask(shape))).cuda()
    dims = (shape[2], shape[1], shape[0])
    ref = torch.empty((len(sigmas), 8) + shape, dtype=torch.float32, device="cuda")
    out = torch.full_like(ref, float("nan"))
    torch.cuda.synchronize()          # the context runs on its own (non-blocking) stream
    ctx.emphysema_features_dev(img.data_ptr(), mask.data_ptr(), ref.data_ptr(), dims, sigmas)
    ctx.synchronize()
    ctx.set_option("overlap_scales", 1)
    try:
        for _ in range(3):     # back to back: the second call must not overtake the first one's readers
            ctx.emphysema_features_dev(img.data_ptr(), mask.data_ptr(), out.data_ptr(), dims, sigmas)
        ctx.synchronize()
    finally:
        ctx.set_option("overlap_scales", 0)
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int32), ref.view(torch.int32))


# ------------------------------------------------------------------------------ histograms
def test_histogram_flat_array(ctx, oracle):
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "hist_ref.npz"))
    assert np.array_equal(ctx.histogram(g["values"], g["edges"]), g["counts"])
    # test/DenseHistogramTest.cxx:10-31
    vals = [-1, 0, 0.5, 1, 1.5, 2.1, 2.6, 2.9, 3.2, 3.5, 4.2, 4.6, 5, 6, 7, 8, 9, 10]
    assert ctx.histogram(vals, [1, 2.5, 3.0, 4.7, 6.2, 8.3]).tolist() == [4, 2, 2, 4, 2, 2, 2]
    assert ctx.histogram(np.zeros(0, np.float32), [0.0, 1.0]).tolist() == [0, 0, 0]
    rng = np.random.default_rng(4)
    v = rng.standard_normal(3_000_001).astype(np.float32)
    e = np.sort(rng.standard_normal(40)).astype(np.float32)
    assert np.array_equal(ctx.histogram(v, e), oracle.hist_f32(e, v)[0])
    # heavy contention: every value in one bin
    assert ctx.histogram(np.full(1_000_000, 0.25, np.float32), e).sum() == 1_000_000


def _edges_for(oracle, img, mask, sigmas, n_edges=40):
    rows = []
    for sigma in sigmas:
        f = oracle.emphysema_features(img, mask, sigma, arith=1)
        for k in range(8):
            rows.append(synth.equalized_edges(f[k][mask != 0], n_edges))
    return np.stack(rows)


def test_emphysema_histograms_whole_mask_and_rois(ctx, oracle):
    shape = (40, 48, 56)
    sigmas = [0.6, 2.4]
    img = synth.ct_like(shape, seed=13, n_blobs=10)
    mask = synth.clamp01(synth.lung_mask(shape))
    edges = _edges_for(oracle, img, mask, sigmas)
    feats = np.concatenate([oracle.emphysema_features(img, mask, s, arith=1) for s in sigmas])
    ref = oracle.features_histograms(feats, mask, edges)
    got = ctx.emphysema_histograms(img, mask, sigmas, edges)
    assert got.shape == ref.shape == (1, 16, 41)
    assert np.all(got.sum(2) == mask.sum())          # every in-mask voxel lands in exactly one bin
    diff = np.abs(got.astype(np.int64) - ref.astype(np.int64)).sum()
    # eigen features may differ in the last bit for <= MISMATCH_FRAC of voxels; such a voxel
    # changes bin only if it sits on an edge
    assert diff <= 2 * max(1, int(MISMATCH_FRAC * mask.sum() * 12)), diff
    assert np.array_equal(got[0, [0, 1, 8, 9]], ref[0, [0, 1, 8, 9]])   # blur/gradient rows exact
    rois = synth.random_rois(mask, 6, (11, 9, 7), seed=3)
    ref = oracle.features_histograms(feats, mask, edges, rois)
    got = ctx.emphysema_histograms(img, mask, sigmas, edges, rois)
    assert got.shape == ref.shape == (6, 16, 41)
    assert np.abs(got.astype(np.int64) - ref.astype(np.int64)).sum() <= 2


def test_many_rois_one_block_per_roi(ctx, oracle):
    """MakeBagDense semantics: one ROI per in-mask voxel.  More than 192 ROIs switch to packed
    bin indices + one block per ROI; the counts must equal the oracle's per-ROI insert loop and
    the small-list path."""
    shape = (18, 22, 28)
    sigmas = [0.6, 1.2]
    img = synth.ct_like(shape, seed=23, n_blobs=5)
    mask = synth.clamp01(synth.lung_mask(shape))
    edges = _edges_for(oracle, img, mask, sigmas, 12)
    rois = synth.dense_rois(mask, (7, 5, 3))
    assert len(rois) > 400
    got = ctx.emphysema_histograms(img, mask, sigmas, edges, rois)
    assert got.shape == (len(rois), 16, 13)
    small = np.concatenate([ctx.emphysema_histograms(img, mask, sigmas, edges, rois[i:i + 150])
                            for i in range(0, len(rois), 150)])
    assert np.array_equal(got, small)
    feats = np.concatenate([oracle.emphysema_features(img, mask, s, arith=1) for s in sigmas])
    pick = np.arange(0, len(rois), 7)
    ref = oracle.features_histograms(feats, mask, edges, rois[pick])
    assert np.abs(got[pick].astype(np.int64) - ref.astype(np.int64)).sum() <= 4
    assert np.array_equal(got[pick][:, [0, 1, 8, 9]], ref[:, [0, 1, 8, 9]])     # blur/gradient rows exact
    # every ROI row sums to the number of in-mask voxels of its box
    x0, y0, z0, sx, sy, sz = rois[len(rois) // 2]
    assert np.all(got[len(rois) // 2].sum(1) == (mask[z0:z0 + sz, y0:y0 + sy, x0:x0 + sx] != 0).sum())


def test_histograms_many_edges_take_the_atomic_kernel(ctx):
    """200 edges per row do not fit the private-counter columns of the z-march kernel: the call
    falls back to the brick kernel (shared-memory atomics) and must give the same counts as
    binning the feature volumes with searchsorted."""
    shape = (20, 24, 36)
    img = synth.ct_like(shape, seed=21, n_blobs=4)
    mask = synth.clamp01(synth.lung_mask(shape))
    feats = ctx.emphysema_features(img, mask, [1.2])[0]
    inside = mask != 0
    for n_edges in (200, 63, 64, 3):
        edges = np.stack([synth.equalized_edges(feats[k][inside], n_edges) for k in range(8)])
        counts = ctx.emphysema_histograms(img, mask, [1.2], edges)[0]
        for k in range(8):
            ref = np.bincount(np.searchsorted(edges[k], feats[k][inside], side="left"), minlength=n_edges + 1)
            assert np.array_equal(counts[k], ref), (n_edges, k)


def test_histograms_batch_equals_one_call_per_scan(ctx):
    shape = (24, 32, 40)
    sigmas = [0.6, 1.2]
    imgs = [synth.ct_like(shape, seed=80 + i, n_blobs=5) for i in range(3)]
    mask = synth.clamp01(synth.lung_mask(shape))
    edges = np.tile(np.linspace(-60, 60, 12, dtype=np.float32), (16, 1))
    rois = np.stack([synth.random_rois(mask, 4, (9, 7, 5), seed=i) for i in range(3)])
    one = np.stack([ctx.emphysema_histograms(im, mask, sigmas, edges) for im in imgs])
    assert np.array_equal(ctx.emphysema_histograms_batch(imgs, [mask] * 3, sigmas, edges), one)
    one = np.stack([ctx.emphysema_histograms(im, mask, sigmas, edges, rois[i]) for i, im in enumerate(imgs)])
    assert np.array_equal(ctx.emphysema_histograms_batch(imgs, [mask] * 3, sigmas, edges, rois), one)


def test_radix_sort_and_compaction_sink(ctx):
    """The step before binning (DetermineHistogramBinEdges_MultiScaleEigenvalueFeatures.cxx:171-296):
    the library's own radix sort against numpy (ties, negatives, zeros of both signs, infinities,
    sizes around the tile boundaries) and the compaction sink -- the features at the selected
    voxels only -- against the full feature volumes."""
    rng = np.random.default_rng(17)
    for n in (1, 2, 255, 2048, 2049, 4097, 100_003, 1_500_000):
        v = rng.normal(0, 50, n).astype(np.float32)
        v[rng.integers(0, n, max(1, n // 7))] = np.float32(3.25)          # ties
        v[rng.integers(0, n, max(1, n // 50))] = np.float32(0.0)
        v[rng.integers(0, n, max(1, n // 60))] = np.float32(-0.0)
        if n > 100:
            v[:3] = [np.inf, -np.inf, np.float32(1e-42)]                   # infinities, a denormal
        got = ctx.sort(v.copy())
        ref = np.sort(v)
        assert np.array_equal(got, ref), "n=%d" % n                        # -0.0 == 0.0 under array_equal, as under std::sort
    shape = (24, 40, 64)
    img = synth.ct_like(shape, seed=61, n_blobs=8)
    mask = synth.clamp01(synth.lung_mask(shape))
    sigmas = [0.6, 2.4]
    full = ctx.emphysema_features(img, mask, sigmas)
    fg = (mask != 0) & (rng.uniform(0, 1, shape) < 0.6)                   # a subset of the foreground
    rows = ctx.feature_samples(img, mask, sigmas, select=fg.astype(np.uint8))
    assert rows.shape == (2, 8, int(fg.sum()))
    assert bits_equal(rows, full[:, :, fg])                               # voxel order = C order of the flags
    srt = ctx.feature_samples(img, mask, sigmas, select=fg.astype(np.uint8), sort=True)
    assert bits_equal(srt, np.sort(full[:, :, fg], axis=2))
    idx = rng.integers(0, img.size, 5000)                                  # random sampling with repeats
    rows = ctx.feature_samples(img, mask, sigmas, index=idx)
    assert bits_equal(rows, full.reshape(2, 8, -1)[:, :, idx])
    assert ctx.feature_samples(img, mask, sigmas, select=np.zeros(shape, np.uint8)).shape == (2, 8, 0)


def test_workspace_growth_between_host_calls(oracle):
    """The grow-only workspace is reallocated while copies of the previous call may still be in
    flight on the context's copy stream (IFE_MEM_HOST multi-scale calls download scale s while scale
    s+1 computes): a small multi-scale call followed at once by larger ones, on a FRESH context, must
    give each call its own correct result."""
    import ife_b200
    c = ife_b200.Context(0)
    try:
        sig = [0.6, 1.2, 2.4]
        outs, refs = [], []
        for shape, seed in (((12, 16, 32), 1), ((24, 40, 64), 2), ((20, 24, 48), 3), ((40, 64, 96), 4)):
            img = synth.ct_like(shape, seed=70 + seed, n_blobs=5)
            mask = synth.clamp01(synth.lung_mask(shape))
            outs.append(c.emphysema_features(img, mask, sig))          # host pointers, no sync in between but the call's own
            refs.append((img, mask))
        for out, (img, mask) in zip(outs, refs):
            ref = np.stack([oracle.emphysema_features(img, mask, s, arith=1) for s in sig])
            assert mismatch_report(out[:, :2], ref[:, :2])[0] == 0
            assert_eigen_parity(np.moveaxis(out[:, 2:], 1, -1), np.moveaxis(ref[:, 2:], 1, -1), "growth")
    finally:
        c.close()


def test_int16_host_images(ctx):
    """Option host_image_i16: the host image pointer is int16 (CT's type on disk); the upload is 2
    bytes per voxel and the widening to float happens on the device.  Same results as the float
    upload of the same values, for the feature volumes, the histograms and a batch (odd voxel
    counts included: the second upload slot of a batch must stay aligned)."""
    for shape in ((24, 40, 64), (9, 13, 37)):
        img16 = np.round(synth.ct_like(shape, seed=81, n_blobs=6)).astype(np.int16)
        imgf = img16.astype(np.float32)
        mask = synth.clamp01(synth.lung_mask(shape))
        sig = [0.6, 2.4]
        ref = ctx.emphysema_features(imgf, mask, sig)
        edges = np.stack([synth.equalized_edges(ref[s, k][mask != 0], 12) for s in range(2) for k in range(8)])
        ref_counts = ctx.emphysema_histograms(imgf, mask, sig, edges)
        ref_batch = ctx.emphysema_histograms_batch([imgf, imgf[::-1].copy(), imgf], [mask, mask[::-1].copy(), mask], sig, edges)
        ctx.set_option("host_image_i16", 1)
        try:
            as_f32_ptr = img16.view(np.int16)          # the binding passes the buffer's address; dtype is not checked by the C ABI
            got = ctx.emphysema_features(as_f32_ptr, mask, sig, _raw_image=True)
            got_counts = ctx.emphysema_histograms(as_f32_ptr, mask, sig, edges, _raw_image=True)
            got_batch = ctx.emphysema_histograms_batch([img16, img16[::-1].copy(), img16], [mask, mask[::-1].copy(), mask], sig, edges, _raw_image=True)
        finally:
            ctx.set_option("host_image_i16", 0)
        assert bits_equal(got, ref)
        assert np.array_equal(got_counts, ref_counts)
        assert np.array_equal(got_batch, ref_batch)


def test_bad_arguments_are_rejected(ctx):
    import ctypes
    import ife_b200
    L = ctx.L
    d = (ctypes.c_int * 3)(8, 8, 8)
    sp = (ctypes.c_double * 3)(1, 1, 1)
    buf = np.zeros((8, 8, 8), np.float32)
    p = buf.ctypes.data_as(ctypes.c_void_p)
    assert L.ife_cuda_gaussian(ctx.h, None, p, d, sp, 1.0, 0) == -1
    assert L.ife_cuda_gaussian(None, p, p, d, sp, 1.0, 0) == -1
    bad = (ctypes.c_int * 3)(8, 0, 8)
    assert L.ife_cuda_gaussian(ctx.h, p, p, bad, sp, 1.0, 0) == -1
    assert b"dims" in L.ife_cuda_last_error(ctx.h)
    with pytest.raises(ife_b200.IfeError):
        ctx.emphysema_histograms(buf, np.ones((8, 8, 8), np.uint8), [1.0], np.zeros((8, 4), np.float32),
                                 rois=[[0, 0, 0, 9, 1, 1]])


# ------------------------------------------------------------------------------ full size
def test_full_size_invariants_512x512x400(ctx):
    """BASELINE.json configs[1] size; checked through size-independent properties."""
    shape = (400, 512, 512)
    rng = np.random.default_rng(2)
    coarse = rng.standard_normal((26, 33, 33)).astype(np.float32)
    import torch
    img = torch.nn.functional.interpolate(torch.from_numpy(coarse)[None, None], size=shape,
                                          mode="trilinear", align_corners=True)[0, 0].numpy()
    img = np.ascontiguousarray(img * 300 - 800 + rng.standard_normal(shape).astype(np.float32) * 20)
    mask = synth.clamp01(synth.lung_mask(shape))
    out = ctx.emphysema_features(img, mask, [1.2])[0]
    inside = mask != 0
    assert np.all(out[:, ~inside] == 0)
    e = out[2:5][:, inside]
    assert np.isfinite(out).all()
    tol = 1e-5 * np.abs(e).max(0)
    assert np.all(np.abs(e[0]) >= np.abs(e[1]) - tol) and np.all(np.abs(e[1]) >= np.abs(e[2]) - tol)
    assert np.array_equal(out[5][inside], (e[0] + e[1]) + e[2])                 # LoG
    assert np.array_equal(out[6][inside], (e[0] * e[1]) * e[2])                 # curvature
    assert np.array_equal(out[7][inside], np.sqrt((e[0] * e[0] + e[1] * e[1]) + e[2] * e[2]))
    # trace of the Hessian == 7-point Laplacian of the blur, up to float rounding
    b = out[0]
    z, y, x = 200, 256, 150
    assert inside[z, y, x]
    lap = (b[z, y, x - 1] + b[z, y, x + 1] + b[z, y - 1, x] + b[z, y + 1, x] + b[z - 1, y, x] +
           b[z + 1, y, x] - 6.0 * b[z, y, x])
    if inside[z - 1:z + 2, y - 1:y + 2, x - 1:x + 2].all():
        assert abs(out[5][z, y, x] - lap) <= 1e-3 * max(1.0, abs(lap))
    # the support box (on by default) changes nothing at full size either
    ctx.set_option("support_box", 0)
    try:
        full = ctx.emphysema_features(img, mask, [1.2])[0]
    finally:
        ctx.set_option("support_box", 1)
    assert bits_equal(out, full)
    del full
    # histograms of the same run: row sums == number of in-mask voxels
    edges = np.stack([synth.equalized_edges(out[k][inside][::97], 40) for k in range(8)])
    counts = ctx.emphysema_histograms(img, mask, [1.2], edges)
    assert np.all(counts.sum(2) == inside.sum())
    for k in (0, 1, 2, 7):
        ref = np.bincount(np.searchsorted(edges[k], out[k][inside], side="left"), minlength=41)
        assert np.array_equal(counts[0, k], ref)


def test_full_size_plain_gaussian_512x512x400(ctx):
    """The one-field smoothing at BASELINE's full size through size-independent properties: both kernel
    families agree bit for bit, a constant stays constant (unit DC gain, edge extension), the result is
    the true Gaussian to the accuracy of the 4th-order recursive approximation, and an odd plane count
    (the second warp's stack of planes is one shorter) changes nothing."""
    import scipy.ndimage
    shape = (399, 512, 512)
    rng = np.random.default_rng(5)
    img = np.ascontiguousarray(rng.standard_normal(shape).astype(np.float32) * 50 - 500)
    img[200:230, 100:400, 50:300] += 400.0
    got = ctx.gaussian(img, 2.4)
    ctx.set_option("tma_passes", 0)
    try:
        old = ctx.gaussian(img, 2.4)
    finally:
        ctx.set_option("tma_passes", 1)
    assert bits_equal(got, old)
    del old
    assert np.isfinite(got).all()
    sub = (slice(150, 280), slice(60, 200), slice(20, 120))       # interior block, far from the volume's faces
    ref = scipy.ndimage.gaussian_filter(img[100:330, 10:250, 0:170].astype(np.float64), 2.4, mode="nearest", truncate=8.0)
    dev = np.abs(got[sub] - ref[50:180, 50:190, 20:120]).max()
    assert dev < 0.02 * 400.0, dev                                 # Deriche-type approximation error, not rounding
    const = np.full((64, 512, 512), 7.25, np.float32)
    assert np.abs(ctx.gaussian(const, 4.8) - 7.25).max() < 1e-5


# ------------------------------------------------------------------------------ z-slabs (one GPU)
def test_slab_single_rank_equals_whole_volume(ctx):
    shape = (40, 36, 44)
    img = synth.ct_like(shape, seed=14, n_blobs=8)
    mask = synth.clamp01(synth.lung_mask(shape))
    sigmas = [0.6, 2.4]
    whole = ctx.emphysema_features(img, mask, sigmas)
    edges = np.stack([synth.equalized_edges(whole[s, k][mask != 0], 20) for s in range(2) for k in range(8)])
    out, counts = ctx.slab_emphysema_features(img, mask, (44, 36, 40), sigmas, edges=edges)
    assert bits_equal(out, whole)
    assert np.array_equal(counts, ctx.emphysema_histograms(img, mask, sigmas, edges)[0])


@pytest.mark.parametrize("halo_factor,exact", [(0.0, False), (1000.0, True)])
def test_slab_local_pipeline_matches_whole_volume(ctx, halo_factor, exact):
    """Walk a volume slab by slab with ife_cuda_slab_emphysema_features_local (no NCCL): with a
    halo that reaches the volume ends the result is bit-identical; with the default halo
    (12 sigma + 5 planes) the truncated warm-up of the z recursion may move a blur value by
    an ulp, which the eigenvalues see at <= 1e-4 * max|lambda| (asserted)."""
    import ife_b200
    shape = (96, 40, 48)
    nz = shape[0]
    img = synth.ct_like(shape, seed=15, n_blobs=20)
    mask = synth.clamp01(synth.lung_mask(shape))
    sigmas = [0.6, 1.2]
    whole = ctx.emphysema_features(img, mask, sigmas)
    edges = np.stack([synth.equalized_edges(whole[s, k][mask != 0], 20) for s in range(2) for k in range(8)])
    whole_counts = ctx.emphysema_histograms(img, mask, sigmas, edges)[0]
    parts, total = [], np.zeros_like(whole_counts)
    P = 3
    for r in range(P):
        z0, z1 = ife_b200.slab_range(nz, P, r)
        H = ife_b200.slab_halo(max(sigmas), 1.0, halo_factor if halo_factor > 0 else 12.0)
        e0, e1 = max(0, z0 - H), min(nz, z1 + H)
        out, counts = ctx.slab_emphysema_features_local(img[e0:e1], mask[e0:e1], e0, z0, z1 - z0,
                                                        (shape[2], shape[1], nz), sigmas, edges=edges,
                                                        halo_factor=halo_factor)
        parts.append(out)
        total += counts
    got = np.concatenate(parts, axis=2)
    assert got.shape == whole.shape
    if exact:
        assert bits_equal(got, whole)
        assert np.array_equal(total, whole_counts)
    else:
        n, worst = mismatch_report(got, whole)
        print("default halo: %d of %d values differ from the whole-volume run (max abs %.3g)" % (n, got.size, worst))
        assert np.all(total.sum(1) == mask.sum())
        blur_err = np.abs(got[:, 0].astype(np.float64) - whole[:, 0])
        assert blur_err.max() <= 2.5e-4            # a few float ulps at ~1000 HU
        lam = np.abs(whole[:, 2:5]).max(1)
        err = np.abs(got[:, 2:5].astype(np.float64) - whole[:, 2:5]).max(1)
        assert np.mean(err > TOL * lam + 1e-3) < 1e-3
