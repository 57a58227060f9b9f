"""CPU tests: pin the oracle (oracle/liboracle.so) against the reference's own known-answer
tests, the committed golden fixtures generated from the reference headers, and -- when the
prebuilt oracle/_ref is present -- the reference headers themselves, bit for bit."""
import os

import numpy as np
import pytest

import synth

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def bits_equal(a, b):
    """bitwise equality of float arrays, NaN == NaN, -0 == +0"""
    a = np.asarray(a); b = np.asarray(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


# ---- test/Symmetric3x3EigenvalueSolverTest.cxx:48-90 (solver instantiated with double) ----
KATS = [
    ([1, 0, 0, 1, 0, 1], [1, 1, 1]),                       # Identity
    ([1, 0, 0, 2, 0, 3], [3, 2, 1]),                       # DiagonalPos
    ([-1, 0, 0, -2, 0, -3], [-3, -2, -1]),                 # DiagonalNeg
    ([1, 0, 0, -2, 0, 3], [3, -2, 1]),                     # DiagonalPosNeg
    ([0.27, 0.92, 0.58, 0.24, 0.75, 0.04], [1.70680634, -0.7205504, -0.43625594]),   # RandomsSmallNums
    ([599, 860, -835, -941, 817, -207], [-2005.21004566, 1183.41690727, 272.79313839]),  # RandomsBigNums
]


def float_ulps(a, b):
    a = np.float32(a).view(np.int32).astype(np.int64)
    b = np.float32(b).view(np.int32).astype(np.int64)
    a = np.where(a < 0, np.int64(-2 ** 31) - a, a)
    b = np.where(b < 0, np.int64(-2 ** 31) - b, b)
    return np.abs(a - b)


@pytest.mark.parametrize("A,expected", KATS)
def test_solver_known_answers_f64(oracle, A, expected):
    ev = oracle.eig_f64(A)[0]
    # EXPECT_FLOAT_EQ: within 4 ULPs after narrowing to float
    assert np.all(float_ulps(ev, expected) <= 4)


def test_solver_ones_near_zero(oracle):
    ev = oracle.eig_f64([1, 1, 1, 1, 1, 1])[0]   # EXPECT_NEAR(.., 1e-15)
    assert np.allclose(ev, [3, 0, 0], rtol=0, atol=1e-15)


def test_solver_float_known_answers(oracle):
    for A, expected in KATS:
        ev = oracle.eig_f32(A)[0]
        assert np.allclose(ev, expected, rtol=2e-6, atol=1e-6)


def test_solver_golden_fixture(oracle):
    g = np.load(os.path.join(GOLDEN, "solver_ref.npz"))
    assert bits_equal(oracle.features_f32(g["A6"]), g["features_f32"])
    assert bits_equal(oracle.eig_f32(g["A6"]), g["eig_f32"])
    assert bits_equal(oracle.eig_f64(g["A6"].astype(np.float64)), g["eig_f64"])


def test_solver_ordering_and_features(oracle):
    A = synth.special_matrices(20000, seed=5)
    f = oracle.features_f32(A)
    e = f[:, :3]
    ok = ~np.isnan(e).any(1)
    # |e0| >= |e1| >= |e2| up to float rounding (exactly degenerate pairs may tie either way)
    tol = 1e-5 * np.abs(e[ok]).max(1)
    assert np.all(np.abs(e[ok, 0]) >= np.abs(e[ok, 1]) - tol)
    assert np.all(np.abs(e[ok, 1]) >= np.abs(e[ok, 2]) - tol)
    assert bits_equal(f[:, 3], (e[:, 0] + e[:, 1]) + e[:, 2])
    assert bits_equal(f[:, 4], (e[:, 0] * e[:, 1]) * e[:, 2])
    assert bits_equal(f[:, 5], np.sqrt((e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2]))
    # against numpy's symmetric eigensolver (double), sorted by magnitude
    M = np.zeros((A.shape[0], 3, 3))
    M[:, 0, 0], M[:, 0, 1], M[:, 0, 2], M[:, 1, 1], M[:, 1, 2], M[:, 2, 2] = A.T.astype(np.float64)
    M[:, 1, 0], M[:, 2, 0], M[:, 2, 1] = M[:, 0, 1], M[:, 0, 2], M[:, 1, 2]
    w = np.linalg.eigvalsh(M)
    w = np.take_along_axis(w, np.argsort(-np.abs(w), axis=1), axis=1)
    ed = oracle.eig_f64(A.astype(np.float64))
    scale = np.abs(w).max(1, keepdims=True) + 1e-300
    assert np.max(np.abs(np.sort(ed, 1) - np.sort(w, 1)) / scale) < 1e-6


def test_ref_matches_restatement_bit_for_bit(oracle):
    """The restatement against the reference: its stored outputs always, its headers
    themselves (oracle/_ref) on 200k more matrices where that library has been built."""
    # ref_functor_volume_f32 (oracle/ref_glue.cpp) is the reference functor per voxel and six
    # zeros outside the mask, so the stored functor outputs give the volume the reference
    # returns for the stored matrices read as an interleaved Hessian volume
    g = np.load(os.path.join(GOLDEN, "solver_ref.npz"))
    m = (np.arange(g["A6"].shape[0]) % 3 != 0).astype(np.uint8)
    want = np.where(m[:, None] != 0, g["features_f32"], np.float32(0))
    assert bits_equal(oracle.functor_volume(g["A6"], m, threads=2), want)
    assert bits_equal(oracle.functor_volume(g["A6"], threads=2), g["features_f32"])
    if not oracle.ref_available():
        return
    R = oracle.Ref()
    assert R.math_overload_is_double()
    A = synth.special_matrices(200000, seed=9)
    assert bits_equal(oracle.features_f32(A), R.features_f32(A))
    assert bits_equal(oracle.eig_f64(A.astype(np.float64)), R.eig_f64(A.astype(np.float64)))
    h = np.random.default_rng(2).standard_normal((5000, 6)).astype(np.float32)
    m = (np.arange(5000) % 3 != 0).astype(np.uint8)
    assert bits_equal(oracle.functor_volume(h, m, threads=2), R.functor_volume(h, m, threads=2))


# ---- test/DenseHistogramTest.cxx:10-55 ----
HVALS = [-1, 0, 0.5, 1, 1.5, 2.1, 2.6, 2.9, 3.2, 3.5, 4.2, 4.6, 5, 6, 7, 8, 9, 10]
HEDGES = [1, 2.5, 3.0, 4.7, 6.2, 8.3]


def test_histogram_known_answers(oracle):
    counts, freqs = oracle.hist_f32(HEDGES, HVALS)
    assert counts.tolist() == [4, 2, 2, 4, 2, 2, 2]
    exp = (np.array([4, 2, 2, 4, 2, 2, 2], np.float64) / 18).astype(np.float32)
    assert np.all(float_ulps(freqs, exp) <= 4)


def test_histogram_nan_and_edges(oracle):
    counts, _ = oracle.hist_f32(HEDGES, [np.nan, 1.0, 2.5, 8.3, np.inf, -np.inf])
    # NaN -> bin 0; a value equal to an edge belongs to the bin left of it
    assert counts.tolist() == [3, 1, 0, 0, 0, 1, 1]


def test_histogram_golden_fixture(oracle):
    g = np.load(os.path.join(GOLDEN, "hist_ref.npz"))
    counts, freqs = oracle.hist_f32(g["edges"], g["values"])
    assert np.array_equal(counts, g["counts"]) and bits_equal(freqs, g["freqs"])
    assert counts.sum() == g["values"].size


# ---- test/DetermineEdgesForEqualizedHistogramTest.cxx:30-120 ----
def test_edges_known_answers(oracle):
    assert oracle.determine_edges(np.arange(1, 10.0), 3).tolist() == [4, 7]
    assert oracle.determine_edges(np.ones(8), 2).tolist() == [1]
    assert oracle.determine_edges([1, 1, 1, 1, 1, 2, 2, 3, 3, 3], 3).tolist() == [2, 3]
    with pytest.raises(IndexError):
        oracle.determine_edges(np.arange(1, 10.0), 10)


def test_edges_properties(oracle):
    rng = np.random.default_rng(0)
    s = np.sort(rng.uniform(-10, 10, 1000))
    e = oracle.determine_edges(s, 50)
    assert np.all(np.diff(e) > 0)
    s = np.unique(s)
    s = s[: s.size - s.size % 50]
    e = oracle.determine_edges(s, 50)
    assert np.all(np.diff(np.searchsorted(s, e)) == s.size // 50)


def test_edges_golden_fixture(oracle):
    g = np.load(os.path.join(GOLDEN, "edges_ref.npz"))
    for name in ("normal41", "dups7", "zeros10", "dups41"):
        e = oracle.determine_edges(g[name + "_samples"], int(g[name + "_nbins"]))
        assert bits_equal(e, g[name + "_edges"]), name


# ---- restated ITK stages: self-consistency (parity unpinned, see oracle_itk.cpp) ----
@pytest.mark.parametrize("sigma", [0.6, 1.0, 2.4, 4.8])
def test_gaussian_impulse_response(oracle, sigma):
    c = oracle.gaussian_coefficients(sigma)
    n = 401
    x = np.zeros(n); x[n // 2] = 1
    h = oracle.gaussian_line(c, x)
    assert abs(h.sum() - 1) < 1e-9                      # unit DC gain
    assert np.max(np.abs(h - h[::-1])) < 1e-12          # symmetric
    k = np.arange(n) - n // 2
    g = np.exp(-k ** 2 / (2 * sigma ** 2)); g /= g.sum()
    assert np.max(np.abs(h - g)) < 4e-3 * g.max() + 2e-3
    # constant line stays constant (edge extension)
    assert np.max(np.abs(oracle.gaussian_line(c, np.full(50, 7.25)) - 7.25)) < 1e-12
    # FMA arithmetic differs from PLAIN only at rounding level
    assert np.max(np.abs(oracle.gaussian_line(c, x, 1) - h)) < 1e-15


def test_gaussian_volume_is_separable_composition(oracle):
    vol = synth.ct_like((12, 10, 14), seed=3, n_blobs=5)
    out = oracle.smoothing_recursive_gaussian(vol, 1.3, threads=2)
    # z, then x, then y with float storage in between
    c = oracle.gaussian_coefficients(1.3)
    t = vol.astype(np.float64)
    t = np.apply_along_axis(lambda l: oracle.gaussian_line(c, l), 0, t).astype(np.float32).astype(np.float64)
    t = np.apply_along_axis(lambda l: oracle.gaussian_line(c, l), 2, t).astype(np.float32).astype(np.float64)
    t = np.apply_along_axis(lambda l: oracle.gaussian_line(c, l), 1, t).astype(np.float32)
    assert bits_equal(out, t)
    with pytest.raises(ValueError):
        oracle.smoothing_recursive_gaussian(vol[:3], 1.0)


def test_gaussian_anisotropic_spacing(oracle):
    vol = synth.ct_like((10, 12, 9), seed=4, n_blobs=4)
    a = oracle.smoothing_recursive_gaussian(vol, 2.0, spacing=(2.0, 2.0, 2.0), threads=1)
    b = oracle.smoothing_recursive_gaussian(vol, 1.0, spacing=(1.0, 1.0, 1.0), threads=1)
    assert bits_equal(a, b)  # sigma is physical: sigma/spacing is what the recursion sees


def test_derivative_stencils(oracle):
    z, y, x = np.meshgrid(np.arange(6.0), np.arange(7.0), np.arange(8.0), indexing="ij")
    vol = (x * x + 3 * x * y + 0.5 * z * z + 2 * y * z).astype(np.float32)
    d2x = oracle.derivative(vol, 0, 2)
    assert np.all(d2x[:, :, 1:-1] == 2)
    assert np.all(d2x[:, :, 0] == vol[:, :, 1] - vol[:, :, 0])      # clamped edge
    dx = oracle.derivative(vol, 0, 1)
    assert np.allclose(dx[:, :, 1:-1], (2 * x + 3 * y)[:, :, 1:-1])
    dxy = oracle.derivative(dx, 1, 1)
    assert np.allclose(dxy[:, 1:-1, 1:-1], 3)
    h = oracle.hessian6(vol)
    assert np.allclose(h[1:-1, 1:-1, 1:-1], [2, 3, 0, 0, 2, 1])
    # spacing scales every stage once (the ITK quirk: second order is /spacing, not /spacing^2)
    assert np.allclose(oracle.derivative(vol, 0, 2, spacing=(2, 1, 1)), d2x / 2)
    gm = oracle.gradient_magnitude(vol)
    g = np.sqrt((2 * x + 3 * y) ** 2 + (3 * x + 2 * z) ** 2 + (z + 2 * y) ** 2)
    assert np.allclose(gm[1:-1, 1:-1, 1:-1], g[1:-1, 1:-1, 1:-1], rtol=1e-6)


def test_emphysema_features_composition(oracle):
    shape = (16, 18, 20)
    img = synth.ct_like(shape, seed=6, n_blobs=6)
    mask = synth.clamp01(synth.lung_mask(shape))
    assert 0 < mask.sum() < mask.size
    f = oracle.emphysema_features(img, mask, 1.2, threads=2)
    assert f.shape == (8,) + shape
    assert np.all(f[:, mask == 0] == 0)
    blur = oracle.normalized_gaussian(img, mask.astype(np.float32), 1.2, threads=2)
    assert bits_equal(f[0][mask != 0], blur[mask != 0])
    hess = oracle.hessian6(blur)
    feat = oracle.functor_volume(hess)
    for k in range(6):
        assert bits_equal(f[2 + k][mask != 0], feat[..., k][mask != 0])
    assert bits_equal(f[1][mask != 0], oracle.gradient_magnitude(blur)[mask != 0])
    # all-ones certainty: normalized convolution == plain smoothing up to the division
    ones = np.ones(shape, np.float32)
    nb = oracle.normalized_gaussian(img, ones, 1.2, threads=2)
    pb = oracle.smoothing_recursive_gaussian(img, 1.2, threads=2)
    assert np.max(np.abs(nb - pb)) < 1e-3


def test_features_histograms_rois(oracle):
    shape = (12, 14, 16)
    rng = np.random.default_rng(1)
    feats = rng.standard_normal((8,) + shape).astype(np.float32)
    mask = (rng.uniform(size=shape) > 0.4).astype(np.uint8)
    edges = np.sort(rng.standard_normal((8, 10)).astype(np.float32), axis=1)
    whole = oracle.features_histograms(feats, mask, edges)
    assert whole.shape == (1, 8, 11) and np.all(whole.sum(2) == mask.sum())
    for k in range(8):
        c, _ = oracle.hist_f32(edges[k], feats[k][mask != 0])
        assert np.array_equal(c, whole[0, k])
    rois = np.array([[0, 0, 0, 5, 5, 5], [3, 2, 1, 7, 6, 5]], np.int32)
    per = oracle.features_histograms(feats, mask, edges, rois)
    sub = mask[1:6, 2:8, 3:10]
    assert np.all(per[1].sum(1) == sub.sum())
