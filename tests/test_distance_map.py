"""Signed distance maps and the expected distance (ife_cuda_signed_distance_map /
ife_cuda_expected_signed_distance, Context.signed_distance_map / expected_distance, the C++ facades and
the SignedDistanceMap / ExpectedDistance tools) against the CPU reference tests/distance_ref.py."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import distance_ref as R
import ife_b200
import nifti_util
import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "image-feature-extraction_b200")
BIN = os.path.join(PKG, "bin")
ANISO = (0.7, 0.7, 2.5)
FLAGS = [(False, False), (True, False), (False, True), (True, True)]   # (inside_positive, squared)


def run(tool, *args):
    return subprocess.run([os.path.join(BIN, tool)] + list(args), capture_output=True, text=True, timeout=600)


def _ball(shape, centers, radii):
    z, y, x = np.indices(shape, dtype=np.float64)
    m = np.zeros(shape, np.uint8)
    for (cz, cy, cx), r in zip(centers, radii):
        m[(z - cz) ** 2 + (y - cy) ** 2 + (x - cx) ** 2 <= r * r] = 1
    return m


def make_mask(kind, shape):
    nz, ny, nx = shape
    if kind == "blob":
        rng = np.random.default_rng(91)
        c = rng.uniform(0, 1, (4, 3)) * np.array(shape)
        return _ball(shape, c, rng.uniform(2, 0.4 * max(shape), 4))
    if kind == "lung":
        return synth.lung_mask(shape)                       # labels {0, 1, 2}: object is != 0
    if kind == "tubes_plates":
        m = np.zeros(shape, np.uint8)
        m[:, ny // 3, :] = 3                                # a one-voxel plate: every voxel is contour
        m[:, 2 * ny // 3: 2 * ny // 3 + 2, nx // 2: nx // 2 + 2] = 1   # a tube along z
        m[nz // 2, :, max(0, nx // 4 - 1): nx // 4 + 1] = 1             # a tube along y
        return m
    if kind == "single":
        m = np.zeros(shape, np.uint8)
        m[nz // 2, ny // 3, nx - 1 - nx // 4] = 1
        return m
    if kind == "every_face":
        m = np.ones(shape, np.uint8)
        m[tuple(slice(s // 4, s - s // 4) if s > 2 else slice(0, 0) for s in shape)] = 0
        m[0, 0, 0] = 0
        return m
    if kind == "empty":
        return np.zeros(shape, np.uint8)
    if kind == "full":
        return np.full(shape, 7, np.uint8)
    raise ValueError(kind)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _ulps(a, b):
    """float32 ulp distance of equal-signed maps."""
    ia = _bits(np.abs(a)).astype(np.int64)
    ib = _bits(np.abs(b)).astype(np.int64)
    return np.abs(ia - ib)


# ---- CPU ------------------------------------------------------------------------------------

def test_contour_single_voxel_and_plate():
    m = np.zeros((5, 6, 7), np.uint8)
    m[2, 3, 4] = 1
    c = R.contour(m)
    assert c.sum() == 1 and c[2, 3, 4]
    p = np.zeros((5, 6, 7), np.uint8)
    p[:, 2, :] = 9                                          # one voxel thick, touching four faces
    assert np.array_equal(R.contour(p), p != 0)


def test_contour_border_faces_are_not_contour():
    m = np.ones((6, 7, 8), np.uint8)
    assert not R.contour(m).any()                           # the image border is no contour
    m[3, 3, 3] = 0                                          # one background voxel inside
    c = R.contour(m)
    want = np.zeros_like(c)
    want[2:5, 2:5, 2:5] = True
    want[3, 3, 3] = False
    assert np.array_equal(c, want)
    h = np.zeros((6, 7, 8), np.uint8)
    h[:, :, :4] = 1                                         # half the image, touching five faces
    c = R.contour(h)
    assert np.array_equal(np.argwhere(c)[:, 2], np.full(6 * 7, 3))


def test_brute_force_and_scipy_agree():
    cases = [((13, 17, 19), "blob"), ((15, 22, 26), "lung"), ((9, 14, 11), "tubes_plates")]
    for shape, kind in cases:
        m = make_mask(kind, shape)
        for sp in ((1.0, 1.0, 1.0), ANISO, (0.68359375, 0.9, 1.25)):
            b, s = R.squared_brute(m, sp), R.squared_scipy(m, sp)
            for ip, sq in FLAGS:
                rb, rs = R.signed(m, b, ip, sq), R.signed(m, s, ip, sq)
                if sp == (1.0, 1.0, 1.0):
                    assert np.array_equal(_bits(rb), _bits(rs)), (kind, sp)
                else:
                    assert np.array_equal(np.signbit(rb), np.signbit(rs))
                    assert _ulps(rb, rs).max() <= 1, (kind, sp)
    assert R.squared_brute(np.zeros((3, 4, 5), np.uint8)) is None
    assert R.squared_brute(np.ones((3, 4, 5), np.uint8)) is None


def test_library_rejects_a_null_context():
    L = ife_b200.load_library()
    m = np.zeros(8, np.uint8)
    out = np.zeros(8, np.float32)
    res = ctypes.c_double()
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    assert L.ife_cuda_signed_distance_map(None, vp(m), vp(out), ife_b200._i3((2, 2, 2)), ife_b200._d3(None), 0,
                                          ife_b200.MEM_HOST) == -1
    assert L.ife_cuda_expected_signed_distance(None, vp(m), vp(out), None, ife_b200._i3((2, 2, 2)), ife_b200._d3(None),
                                               0, ctypes.byref(res), ife_b200.MEM_HOST) == -1


def test_cli_surface_and_bad_arguments(tmp_path):
    p = run("SignedDistanceMap", "--help")
    assert p.returncode == 0
    for flag in ("-i <", "-o <", "-p <", "-q <", "-b <", "--inside-positive", "--squared", "--background"):
        assert flag in p.stdout
    p = run("ExpectedDistance", "--help")
    assert p.returncode == 0
    for flag in ("-c <", "-w <", "-m <", "-p <"):
        assert flag in p.stdout
    assert run("SignedDistanceMap", "--version").stdout.strip().endswith("version: 0.1")
    d = str(tmp_path)
    nifti_util.write(d + "/m.nii", np.zeros((3, 4, 5), np.uint8))
    io = ["-i", d + "/m.nii", "-o", d + "/o.nii"]
    for args in ([], ["-i", d + "/m.nii"], io + ["-p", "maybe"], io + ["-q", "2"], io + ["-b", "-1"],
                 io + ["-b", "70000"], io + ["-b", "x"], io + ["--bogus", "1"]):
        p = run("SignedDistanceMap", *args)
        assert p.returncode == 1 and "PARSE ERROR" in p.stderr, args
    for args in ([], ["-c", d + "/m.nii"], ["-c", d + "/m.nii", "-w", d + "/m.nii", "-p", "maybe"],
                 ["-c", d + "/m.nii", "-w", d + "/m.nii", "--bogus", "1"]):
        p = run("ExpectedDistance", *args)
        assert p.returncode == 1 and "PARSE ERROR" in p.stderr, args
    assert not os.path.exists(d + "/o.nii")


# ---- GPU ------------------------------------------------------------------------------------

GPU_CASES = [((23, 29, 37), k) for k in ("blob", "lung", "tubes_plates", "single", "every_face", "empty", "full")] + \
            [((7, 64, 5), "lung"), ((7, 64, 5), "blob"), ((9, 11, 1), "blob"), ((9, 11, 1), "every_face"),
             ((6, 1, 10), "blob"), ((1, 13, 12), "lung")]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,kind", GPU_CASES)
@pytest.mark.parametrize("spacing", [(1.0, 1.0, 1.0), ANISO])
def test_gpu_equals_brute_force(ctx, shape, kind, spacing):
    m = make_mask(kind, shape)
    D = R.squared_brute(m, spacing)
    for ip, sq in FLAGS:
        got = ctx.signed_distance_map(m, spacing, inside_positive=ip, squared=sq)
        want = R.signed(m, D, ip, sq)
        assert np.array_equal(_bits(got), _bits(want)), (kind, spacing, ip, sq, int((got != want).sum()))
    if kind in ("empty", "full"):
        got = ctx.signed_distance_map(m, spacing)
        assert np.all(np.abs(got) == R.FLT_MAX)
        assert np.all(np.signbit(got) == (kind == "full"))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(96, 128, 128), (400, 512, 512)])
def test_gpu_equals_scipy_on_the_lung_mask(ctx, shape):
    m = synth.lung_mask(shape)
    got = ctx.signed_distance_map(m)
    assert np.array_equal(_bits(got), _bits(R.signed(m, R.squared_scipy(m))))
    got = ctx.signed_distance_map(m, ANISO)
    want = R.signed(m, R.squared_scipy(m, ANISO))
    assert np.array_equal(np.signbit(got), np.signbit(want))
    u = _ulps(got, want)
    diff = np.flatnonzero(u)
    print("lung %s at %s: %d voxels differ from scipy by 1 float ulp" % (shape, ANISO, diff.size))
    assert u.max() <= 1
    # scipy picked another nearest contour voxel whose D rounds differently: the GPU's is the minimum
    if diff.size:
        pick = diff[:: max(1, diff.size // 64)]
        D = R.squared_brute(m, ANISO, chunk=8, voxels=pick)
        assert np.array_equal(_bits(np.abs(got.ravel()[pick])), _bits(np.sqrt(D).astype(np.float32)))


@pytest.mark.gpu
def test_gpu_device_pointers_equal_host_path(ctx):
    import torch
    shape = (21, 30, 41)
    m = synth.lung_mask(shape)
    dims = shape[::-1]
    d_m = torch.from_numpy(m).cuda()
    buf = torch.zeros(m.size + 1, dtype=torch.float32, device="cuda")
    for ip, sq in FLAGS:
        want = ctx.signed_distance_map(m, ANISO, inside_positive=ip, squared=sq)
        for off in (0, 1):                                  # the output 4 bytes past a 16-byte boundary
            torch.cuda.synchronize()
            ctx.signed_distance_map_dev(d_m.data_ptr(), buf.data_ptr() + 4 * off, dims, ANISO, ip, sq)
            ctx.synchronize()
            got = buf[off:off + m.size].cpu().numpy().reshape(shape)
            assert np.array_equal(_bits(got), _bits(want)), (ip, sq, off)


@pytest.mark.gpu
def test_gpu_launches_are_counted(ctx):
    m = make_mask("blob", (8, 9, 10))
    n0 = ctx.launch_count()
    ctx.signed_distance_map(m)
    assert ctx.launch_count() == n0 + 3
    ctx.expected_distance(m, np.ones(m.shape, np.float32))
    assert ctx.launch_count() == n0 + 7


@pytest.mark.gpu
def test_gpu_rejects_bad_arguments(ctx):
    L = ctx.L
    m = np.zeros(8, np.uint8)
    m[0] = 1
    out = np.zeros(8, np.float32)
    res = ctypes.c_double()
    vp = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)

    def sdm(mask=m, o=out, dims=(2, 2, 2), sp=(1, 1, 1), flags=0):
        return L.ife_cuda_signed_distance_map(ctx.h, vp(mask), vp(o), ife_b200._i3(dims), ife_b200._d3(sp), flags,
                                              ife_b200.MEM_HOST)

    def exp(center=m, w=out + 1, region=None, sp=(1, 1, 1), flags=0):
        return L.ife_cuda_expected_signed_distance(ctx.h, vp(center), vp(w), vp(region), ife_b200._i3((2, 2, 2)),
                                                   ife_b200._d3(sp), flags, ctypes.byref(res), ife_b200.MEM_HOST)
    assert sdm() == 0 and sdm(flags=3) == 0 and exp() == 0 and exp(flags=1) == 0
    for bad in (dict(mask=None), dict(o=None), dict(flags=4), dict(flags=-1), dict(sp=(0, 1, 1)),
                dict(sp=(1, float("nan"), 1)), dict(sp=(1, 1, float("inf"))), dict(dims=(32768, 1, 1)),
                dict(dims=(1, 0, 1))):
        assert sdm(**bad) == -1, bad                       # IFE_E_INVALID
    for bad in (dict(center=None), dict(w=None), dict(flags=2), dict(sp=(1, -1, 1))):
        assert exp(**bad) == -1, bad


def _weights(shape, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.0, 1.0, shape).astype(np.float32)


@pytest.mark.gpu
def test_gpu_expected_distance(ctx):
    shape = (23, 40, 37)
    center = make_mask("lung", shape)
    w = _weights(shape, 92)
    region = make_mask("blob", shape)
    for sp in ((1.0, 1.0, 1.0), ANISO):
        for ip in (False, True):
            dmap = ctx.signed_distance_map(center, sp, inside_positive=ip)
            for reg in (None, region):
                e = ctx.expected_distance(center, w, reg, sp, inside_positive=ip)
                assert e == pytest.approx(R.expected(dmap, w, reg), rel=1e-12, abs=0)
                again = ctx.expected_distance(center, w, reg, sp, inside_positive=ip)
                assert np.float64(e).view(np.uint64) == np.float64(again).view(np.uint64)
    # weights outside the region do not enter the sum
    w2 = w.copy()
    w2[region == 0] = np.nan
    assert ctx.expected_distance(center, w2, region) == ctx.expected_distance(center, w, region)


@pytest.mark.gpu
def test_gpu_expected_distance_rejects(ctx):
    shape = (10, 12, 14)
    center = make_mask("blob", shape)
    w = _weights(shape, 93)
    for bad_w in (np.zeros(shape, np.float32), np.where(center != 0, w, -0.5).astype(np.float32)):
        with pytest.raises(ife_b200.IfeError) as e:
            ctx.expected_distance(center, bad_w)
        assert e.value.code == -1
    for v in (np.nan, np.inf):
        bad_w = w.copy()
        bad_w[3, 4, 5] = v
        with pytest.raises(ife_b200.IfeError) as e:
            ctx.expected_distance(center, bad_w)
        assert e.value.code == -1
    with pytest.raises(ife_b200.IfeError) as e:                # no weight inside the region
        ctx.expected_distance(center, w, np.zeros(shape, np.uint8))
    assert e.value.code == -1
    for contourless in (np.zeros(shape, np.uint8), np.ones(shape, np.uint8)):
        with pytest.raises(ife_b200.IfeError) as e:
            ctx.expected_distance(contourless, w)
        assert e.value.code == -1 and "contour" in str(e.value)


@pytest.mark.gpu
def test_signed_distance_map_tool(ctx, tmp_path):
    d = str(tmp_path)
    shape = (14, 24, 28)
    sp = tuple(float(np.float32(v)) for v in ANISO)
    lab = synth.lung_mask(shape).astype(np.uint16)
    lab[0, 0, :5] = 300                                         # labels above 255 are object too
    nifti_util.write(d + "/mask.nii.gz", lab, sp)
    obj = (lab != 0).astype(np.uint8)
    for args, ip, sq in (([], False, False), (["-p", "1"], True, False), (["-q", "true"], False, True),
                         (["--inside-positive=true", "--squared=1"], True, True)):
        p = run("SignedDistanceMap", "-i", d + "/mask.nii.gz", "-o", d + "/sdm.nii.gz", *args)
        assert p.returncode == 0, p.stderr
        got, pix = nifti_util.read(d + "/sdm.nii.gz")
        assert got.dtype == np.float32 and pix == sp
        assert np.array_equal(_bits(got), _bits(ctx.signed_distance_map(obj, sp, inside_positive=ip, squared=sq)))
    p = run("SignedDistanceMap", "-i", d + "/mask.nii.gz", "-o", d + "/sdm2.nii", "-b", "2")
    assert p.returncode == 0, p.stderr
    got, _ = nifti_util.read(d + "/sdm2.nii")
    assert np.array_equal(_bits(got), _bits(ctx.signed_distance_map((lab != 2).astype(np.uint8), sp)))
    p = run("SignedDistanceMap", "-i", d + "/missing.nii", "-o", d + "/x.nii")
    assert p.returncode == 1 and "Failed to process." in p.stderr


@pytest.mark.gpu
def test_expected_distance_tool(ctx, tmp_path):
    d = str(tmp_path)
    shape = (14, 24, 28)
    sp = tuple(float(np.float32(v)) for v in ANISO)
    center = synth.lung_mask(shape).astype(np.uint16)
    w = _weights(shape, 94)
    region = make_mask("blob", shape).astype(np.uint16) * 5
    nifti_util.write(d + "/c.nii.gz", center, sp)
    nifti_util.write(d + "/w.nii.gz", w, sp)
    nifti_util.write(d + "/r.nii", region, sp)
    c8, r8 = (center != 0).astype(np.uint8), (region != 0).astype(np.uint8)
    for extra, reg, ip in (([], None, False), (["-m", d + "/r.nii"], r8, False), (["-m", d + "/r.nii", "-p", "1"], r8, True)):
        p = run("ExpectedDistance", "-c", d + "/c.nii.gz", "-w", d + "/w.nii.gz", *extra)
        assert p.returncode == 0, p.stderr
        assert p.stdout.strip() == "%.17g" % ctx.expected_distance(c8, w, reg, sp, inside_positive=ip)
    nifti_util.write(d + "/w_other.nii", w, (0.7, 0.7, 2.0))      # another spacing
    nifti_util.write(d + "/r_small.nii", region[:, :, :-1])
    for extra in (["-w", d + "/w_other.nii"], ["-w", d + "/w.nii.gz", "-m", d + "/r_small.nii"]):
        p = run("ExpectedDistance", "-c", d + "/c.nii.gz", *extra)
        assert p.returncode == 1 and "geometries differ" in p.stderr, extra
    p = run("ExpectedDistance", "-c", d + "/w_other.nii", "-w", d + "/w_other.nii")   # weights as a mask: no
    assert p.returncode == 1 and "Failed to process." in p.stderr                   # background, no contour


_FACADE_SRC = r"""
#include <cstdio>
#include "itkSignedMaurerDistanceMapImageFilter.h"
#include "ife/IO/NiftiIO.h"
#include "ife/Statistics/ExpectedDistanceFromCenterToInterestPoint.h"
int main(int argc, char** argv) {
  auto m = ife::nifti::Read<unsigned char>(argv[1]);
  auto f = itk::SignedMaurerDistanceMapImageFilter<itk::Image<unsigned char, 3>, itk::Image<float, 3> >::New();
  if (!f->GetSquaredDistance() || f->GetInsideIsPositive() || !f->GetUseImageSpacing()) return 2;
  f->SetInput(m.get());
  f->Update();
  ife::nifti::Write(argv[2], *f->GetOutput());
  f->SetUseImageSpacing(false);
  f->SetSquaredDistance(false);
  f->Update();
  ife::nifti::Write(argv[3], *f->GetOutput());
  auto w = ife::nifti::Read<float>(argv[4]);
  std::printf("%.17g\n", ife::ExpectedDistanceFromCenterToInterestPoint(*m, *w));
  return 0;
}
"""


@pytest.mark.gpu
def test_cpp_facade_defaults(ctx, tmp_path):
    d = str(tmp_path)
    src = tmp_path / "f.cxx"
    src.write_text(_FACADE_SRC)
    exe = str(tmp_path / "f")
    r = subprocess.run(["g++", "-std=c++14", "-I", os.path.join(PKG, "host", "include"),
                        "-I", os.path.join(PKG, "host", "include", "itk_compat"), "-I", os.path.join(ROOT, "include"),
                        str(src), "-o", exe, "-L", os.path.join(PKG, "lib"), "-life_cuda", "-lz", "-pthread",
                        "-Wl,-rpath," + os.path.join(PKG, "lib")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    shape = (12, 20, 22)
    sp = tuple(float(np.float32(v)) for v in ANISO)
    m = (synth.lung_mask(shape) != 0).astype(np.uint8)
    w = _weights(shape, 95)
    nifti_util.write(d + "/m.nii", m, sp)
    nifti_util.write(d + "/w.nii", w, sp)
    r = subprocess.run([exe, d + "/m.nii", d + "/sq.nii", d + "/unit.nii", d + "/w.nii"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    sq, _ = nifti_util.read(d + "/sq.nii")
    unit, _ = nifti_util.read(d + "/unit.nii")
    assert np.array_equal(_bits(sq), _bits(ctx.signed_distance_map(m, sp, squared=True)))
    assert np.array_equal(_bits(unit), _bits(ctx.signed_distance_map(m)))
    assert r.stdout.strip() == "%.17g" % ctx.expected_distance(m, w, spacing=sp)
