"""Resampling onto a new voxel spacing (ife_cuda_resample, Context.resample / resample_dev, the
Resample tool, NIfTI headers with a new spacing) against the CPU reference tests/resample_ref.py."""
import ctypes
import os
import struct
import subprocess

import numpy as np
import pytest

import ife_b200
import nifti_util
import resample_ref as R
import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "image-feature-extraction_b200")
BIN = os.path.join(PKG, "bin")


def run(tool, *args):
    return subprocess.run([os.path.join(BIN, tool)] + list(args), capture_output=True, text=True, timeout=600)


def _coords(shape_in, spacing, out_spacing):
    """Continuous indices (z, y, x) of every output voxel, as 1-D arrays per axis."""
    nz, ny, nx = shape_in
    mx, my, mz = R.output_dims((nx, ny, nz), spacing, out_spacing)
    ax = []
    for m, s, so in ((mz, spacing[2], out_spacing[2]), (my, spacing[1], out_spacing[1]), (mx, spacing[0], out_spacing[0])):
        i = np.arange(m, dtype=np.float64)
        ax.append(i if so == s else (i * so) * (1.0 / s))
    return ax


# ---- CPU ------------------------------------------------------------------------------------

def test_reference_linear_agrees_with_scipy_at_interior_points():
    from scipy import ndimage
    shape = (14, 17, 19)
    vol = synth.ct_like(shape, seed=81, n_blobs=5)
    sp, osp = (0.7, 0.9, 2.5), (0.45, 1.3, 0.8)
    got = R.resample(vol, sp, osp)
    cz, cy, cx = _coords(shape, sp, osp)
    Z, Y, X = np.meshgrid(cz, cy, cx, indexing="ij")
    want = ndimage.map_coordinates(vol.astype(np.float64), [Z, Y, X], order=1, mode="nearest")
    interior = (Z <= shape[0] - 1) & (Y <= shape[1] - 1) & (X <= shape[2] - 1)
    assert interior.mean() > 0.8
    np.testing.assert_allclose(got[interior], want[interior], rtol=1e-6, atol=1e-6 * np.abs(vol).max())


def test_reference_nearest_agrees_with_index_rounding():
    shape = (9, 12, 11)
    lab = synth.lung_mask(shape)
    for sp, osp in (((0.7, 0.7, 2.5), (0.7, 0.7, 0.7)), ((1.0, 0.5, 1.5), (0.3, 1.7, 1.5))):
        got = R.resample(lab, sp, osp, nearest=True, default=9)
        cz, cy, cx = _coords(shape, sp, osp)
        idx = [np.minimum((c + 0.5).astype(np.int64), n - 1) for c, n in zip((cz, cy, cx), shape)]
        ins = [(c >= -0.5) & (c < n - 0.5) for c, n in zip((cz, cy, cx), shape)]
        want = lab[np.ix_(*idx)]
        inside = ins[0][:, None, None] & ins[1][None, :, None] & ins[2][None, None, :]
        want = np.where(inside, want, np.uint8(9))
        assert got.dtype == np.uint8 and np.array_equal(got, want)


def test_size_rule_binding_reference_and_library_agree():
    L = ife_b200.load_library()
    vol = np.zeros(1, np.float32)
    cases = [((512, 512, 160), (0.7, 0.7, 2.5), (0.7, 0.7, 0.7)),
             ((5, 7, 3), (1.0, 1.0, 1.0), (3.0, 0.3, 7.0)),
             ((33, 1, 2), (0.68359375, 1.0, 1.25), (0.5, 1.0, 0.625)),
             ((10, 10, 10), (1.0, 1.0, 1.0), (0.8, 1.0 / 0.3, 4.0))]   # x: 12.5 -> 13, z: 2.5 -> 3
    for dims, sp, osp in cases:
        od = (ctypes.c_int * 3)()
        # the size query takes no context, so it runs without a device
        rc = L.ife_cuda_resample(None, vol.ctypes.data_as(ctypes.c_void_p), None, 4, ife_b200._i3(dims),
                                 ife_b200._d3(sp), ife_b200._d3(osp), ife_b200.INTERP_LINEAR, 0.0, od, ife_b200.MEM_HOST)
        assert rc == 0
        assert tuple(od) == ife_b200.resampled_dims(dims, sp, osp) == R.output_dims(dims, sp, osp)
    assert ife_b200.resampled_dims((10, 10, 10), (1, 1, 1), (0.8, 1.0, 4.0)) == (13, 10, 3)


def test_library_rejects_bad_arguments():
    L = ife_b200.load_library()
    vol = np.zeros(8, np.float32)
    vp = vol.ctypes.data_as(ctypes.c_void_p)
    od = (ctypes.c_int * 3)()

    def q(ptr=vp, elem=4, sp=(1, 1, 1), osp=(1, 1, 1), interp=0, default=0.0):
        return L.ife_cuda_resample(None, ptr, None, elem, ife_b200._i3((2, 2, 2)), ife_b200._d3(sp), ife_b200._d3(osp),
                                   interp, default, od, ife_b200.MEM_HOST)
    assert q() == 0 and q(elem=1, interp=1) == 0 and q(elem=4, interp=1) == 0
    for bad in (dict(ptr=None), dict(sp=(0, 1, 1)), dict(sp=(1, -1, 1)), dict(osp=(1, 1, 0)),
                dict(osp=(1, float("nan"), 1)), dict(osp=(float("inf"), 1, 1)), dict(sp=(1, 1, float("inf"))),
                dict(elem=1, interp=0), dict(elem=2, interp=1), dict(interp=2),
                dict(elem=1, interp=1, default=256.0), dict(elem=1, interp=1, default=1.5)):
        assert q(**bad) == -1, bad                                   # IFE_E_INVALID
    # a real call needs a context
    assert L.ife_cuda_resample(None, vp, vp, 4, ife_b200._i3((2, 2, 2)), ife_b200._d3((1, 1, 1)),
                               ife_b200._d3((1, 1, 1)), 0, 0.0, od, ife_b200.MEM_HOST) == -1


def test_cli_surface_and_bad_arguments(tmp_path):
    p = run("Resample", "--help")
    assert p.returncode == 0 and "-s <double> <double> <double>" in p.stdout
    for flag in ("-i <", "-o <", "-n <", "-d <"):
        assert flag in p.stdout
    assert run("Resample", "--version").stdout.strip().endswith("version: 0.1")
    d = str(tmp_path)
    nifti_util.write(d + "/img.nii", np.zeros((3, 4, 5), np.float32))
    for args in ([], ["-i", d + "/img.nii", "-o", d + "/o.nii"],                     # -s missing
                 ["-i", d + "/img.nii", "-o", d + "/o.nii", "-s", "0.7", "0.7"],     # two values
                 ["-i", d + "/img.nii", "-o", d + "/o.nii", "-s", "0.7", "0", "1"],
                 ["-i", d + "/img.nii", "-o", d + "/o.nii", "-s", "0.7", "-1", "1"],
                 ["-i", d + "/img.nii", "-o", d + "/o.nii", "-s", "0.7", "nan", "1"],
                 ["-i", d + "/img.nii", "-o", d + "/o.nii", "-s", "0.7", "x", "1"],
                 ["-i", d + "/img.nii", "-o", d + "/o.nii", "-s", "1", "1", "1", "-n", "maybe"],
                 ["-i", d + "/img.nii", "-o", d + "/o.nii", "-s", "1", "1", "1", "-d", "abc"],
                 ["-i", d + "/img.nii", "-o", d + "/o.nii", "-s", "1", "1", "1", "-n", "1", "-d", "300"],
                 ["-i", d + "/img.nii", "-o", d + "/o.nii", "-s", "1", "1", "1", "--bogus", "1"]):
        p = run("Resample", *args)
        assert p.returncode == 1 and "PARSE ERROR" in p.stderr, args
    p = run("Resample", "-i", d + "/missing.nii", "-o", d + "/o.nii", "-s", "1", "1", "1")
    assert p.returncode == 1 and "Failed to process." in p.stderr


def test_cli_nearest_refuses_labels_above_255(tmp_path):
    d = str(tmp_path)
    lab = np.zeros((3, 4, 5), np.uint16)
    lab[1, 2, 3] = 256
    nifti_util.write(d + "/lab.nii.gz", lab)
    p = run("Resample", "-i", d + "/lab.nii.gz", "-o", d + "/o.nii.gz", "-s", "1", "1", "1", "--nearest", "true")
    assert p.returncode == 1 and "label 256" in p.stderr and not os.path.exists(d + "/o.nii.gz")


_WRITE_SRC = r"""
#include <cstdlib>
#include "ife/IO/NiftiIO.h"
int main(int argc, char** argv) {
  auto img = ife::nifti::Read<float>(argv[1]);
  ife::Geometry g = img->GetGeometry();
  for (int d = 0; d < 3; ++d) g.spacing[d] = std::atof(argv[3 + d]);
  ife::nifti::Write(argv[2], g, img->GetBufferPointer());
  return 0;
}
"""


def _header(path):
    import gzip
    raw = (gzip.open if path.endswith(".gz") else open)(path, "rb").read()
    return raw[:348]


def test_header_carrying_image_written_with_new_spacing(tmp_path):
    """NiftiIO Write: a spacing that differs from the source header's pixdim replaces it and scales the
    sform column of that axis; origin (sform offsets, qoffset) and every other byte stay.  With the
    header's own spacing the header is written back unchanged, as every other tool does."""
    d = str(tmp_path)
    src = tmp_path / "w.cxx"
    src.write_text(_WRITE_SRC)
    exe = str(tmp_path / "w")
    r = subprocess.run(["g++", "-std=c++14", "-I", os.path.join(PKG, "host", "include"), "-I", os.path.join(ROOT, "include"),
                        str(src), "-o", exe, "-L", os.path.join(PKG, "lib"), "-life_cuda", "-lz", "-pthread",
                        "-Wl,-rpath," + os.path.join(PKG, "lib")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    sp = (0.75, 0.75, 2.5)
    nifti_util.write(d + "/in.nii", np.arange(60, dtype=np.float32).reshape(3, 4, 5), sp)
    h = bytearray(open(d + "/in.nii", "rb").read())
    struct.pack_into("<h", h, 252, 1)                                  # qform_code
    struct.pack_into("<3f", h, 268, -120.5, 33.25, -7.0)               # qoffset
    struct.pack_into("<4f", h, 280, -0.75, 0.0, 0.0, 190.5)            # srow_x: x runs right to left
    struct.pack_into("<4f", h, 296, 0.0, 0.75, 0.0, -12.0)
    struct.pack_into("<4f", h, 312, 0.0, 0.0, 2.5, -300.25)
    open(d + "/in.nii", "wb").write(bytes(h))

    r = subprocess.run([exe, d + "/in.nii", d + "/same.nii.gz"] + [repr(v) for v in sp], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert _header(d + "/same.nii.gz") == bytes(h[:348])

    new = (0.5, 0.75, 0.625)
    r = subprocess.run([exe, d + "/in.nii", d + "/new.nii"] + [repr(v) for v in new], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = _header(d + "/new.nii")
    _, pix = nifti_util.read(d + "/new.nii")
    assert pix == tuple(float(np.float32(v)) for v in new)
    assert struct.unpack_from("<3f", out, 268) == struct.unpack_from("<3f", h, 268)
    assert struct.unpack_from("<4f", out, 280) == (float(np.float32(-0.5)), 0.0, 0.0, 190.5)
    assert struct.unpack_from("<4f", out, 296) == (0.0, 0.75, 0.0, -12.0)
    assert struct.unpack_from("<4f", out, 312) == (0.0, 0.0, 0.625, -300.25)
    changed = [i for i in range(348) if out[i] != h[i]]
    assert all(80 <= i < 92 or 280 <= i < 328 for i in changed), changed


# ---- GPU ------------------------------------------------------------------------------------

def _same(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,sp,osp", [
    ((40, 48, 64), (0.7, 0.7, 2.5), (0.7, 0.7, 0.7)),          # anisotropic -> isotropic, nx' % 4 == 0
    ((13, 21, 30), (0.8, 0.6, 1.25), (0.57, 0.9, 0.4)),       # up x, down y, up z; nx' = 42
    ((17, 19, 23), (1.0, 1.0, 1.0), (2.7, 0.35, 1.6)),         # down x, up y, down z
    ((9, 10, 11), (0.6836, 0.6836, 1.0), (0.5, 0.5, 0.5)),     # ragged nx' = 15
])
def test_gpu_equals_reference_bit_for_bit(ctx, shape, sp, osp):
    img = synth.ct_like(shape, seed=82, n_blobs=6)
    lab = synth.lung_mask(shape)
    got = ctx.resample(img, sp, osp)
    assert _same(got, R.resample(img, sp, osp))
    assert _same(ctx.resample(img, sp, osp, nearest=True), R.resample(img, sp, osp, nearest=True))
    assert _same(ctx.resample(lab, sp, osp, nearest=True), R.resample(lab, sp, osp, nearest=True))
    nx, ny, nz = ife_b200.resampled_dims(shape[::-1], sp, osp)
    assert got.shape == (nz, ny, nx)


@pytest.mark.gpu
def test_gpu_ct_like_anisotropic_to_isotropic(ctx):
    shape = (40, 96, 100)
    sp, osp = (0.7, 0.7, 2.5), (0.7, 0.7, 0.7)
    img = synth.ct_like(shape, seed=83)
    lab = synth.lung_mask(shape)
    out = ctx.resample(img, sp, osp)
    assert out.shape == (143, 96, 100)
    assert _same(out, R.resample(img, sp, osp))
    m = ctx.resample(lab, sp, osp, nearest=True)
    assert _same(m, R.resample(lab, sp, osp, nearest=True))
    assert set(np.unique(m)) == {0, 1, 2}


@pytest.mark.gpu
def test_gpu_border_and_outside_voxels_take_the_default(ctx):
    shape = (6, 7, 9)
    img = synth.ct_like(shape, seed=84, n_blobs=3)
    lab = synth.lung_mask(shape)
    sp, osp = (1.0, 1.0, 1.0), (0.3, 0.45, 0.2)
    cz, cy, cx = _coords(shape, sp, osp)
    assert ((cx > shape[2] - 1) & (cx < shape[2] - 0.5)).any()       # half-voxel border: inside, clamped
    assert (cx >= shape[2] - 0.5).any() and (cz >= shape[0] - 0.5).any()  # beyond: default
    for default in (0.0, -1024.5):
        got = ctx.resample(img, sp, osp, default=default)
        ref = R.resample(img, sp, osp, default=default)
        assert _same(got, ref)
        assert (got[:, :, -1] == np.float32(default)).all()
    for default in (0, 7):
        got = ctx.resample(lab, sp, osp, nearest=True, default=default)
        assert _same(got, R.resample(lab, sp, osp, nearest=True, default=default))
        assert (got[-1] == default).all()


@pytest.mark.gpu
def test_gpu_equal_spacing_is_the_identity(ctx):
    shape = (11, 13, 18)
    img = synth.ct_like(shape, seed=85, n_blobs=4)
    img[3, 4, 5:9] = 0.0              # zeros next to large values: an ulp off an integer index would show
    lab = synth.lung_mask(shape)
    for sp in ((0.7, 0.7, 2.5), (0.68359375, 0.3, 1.1)):
        assert _same(ctx.resample(img, sp, sp), img)
        assert _same(ctx.resample(img, sp, sp, nearest=True), img)
        assert _same(ctx.resample(lab, sp, sp, nearest=True), lab)


@pytest.mark.gpu
def test_gpu_device_pointers_equal_host_path(ctx):
    import torch
    shape = (20, 30, 41)
    sp, osp = (0.7, 0.7, 2.5), (0.7, 0.7, 0.7)
    img = synth.ct_like(shape, seed=86, n_blobs=5)
    lab = synth.lung_mask(shape)
    for vol, nearest in ((img, False), (img, True), (lab, True)):
        dims = vol.shape[::-1]
        nx, ny, nz = ife_b200.resampled_dims(dims, sp, osp)
        d_in = torch.from_numpy(vol).cuda()
        d_out = torch.empty((nz, ny, nx), dtype=d_in.dtype, device="cuda")
        torch.cuda.synchronize()
        od = ctx.resample_dev(d_in.data_ptr(), d_out.data_ptr(), dims, sp, osp, elem_bytes=vol.itemsize,
                              nearest=nearest, default=3)
        ctx.synchronize()
        assert od == (nx, ny, nz)
        assert _same(d_out.cpu().numpy(), ctx.resample(vol, sp, osp, nearest=nearest, default=3))


@pytest.mark.gpu
def test_gpu_launches_are_counted(ctx):
    vol = np.ones((4, 5, 6), np.float32)
    n0 = ctx.launch_count()
    ctx.resample(vol, (1, 1, 1), (0.5, 0.5, 0.5))
    assert ctx.launch_count() == n0 + 1


@pytest.mark.gpu
def test_resample_tool_then_extract_features_against_reference_chain(tmp_path, oracle):
    from test_host_tools import _eig_close
    shape = (14, 24, 28)
    sp = tuple(float(np.float32(v)) for v in (0.8, 0.8, 2.0))   # pixdim is float32 on disk
    img = synth.ct_like(shape, seed=87, n_blobs=6)
    lab = synth.lung_mask(shape)
    d = str(tmp_path)
    nifti_util.write(d + "/img.nii.gz", img.astype(np.int16), sp)      # CT is int16 on disk
    nifti_util.write(d + "/mask.nii.gz", lab, sp)
    imgf = img.astype(np.int16).astype(np.float32)
    osp = (0.8, 0.8, 0.8)
    p = run("Resample", "-i", d + "/img.nii.gz", "-o", d + "/img_r.nii.gz", "-s", "0.8", "0.8", "0.8")
    assert p.returncode == 0, p.stderr
    p = run("Resample", "-i", d + "/mask.nii.gz", "-o", d + "/mask_r.nii.gz", "-s", "0.8", "0.8", "0.8", "-n", "1")
    assert p.returncode == 0, p.stderr

    ref_img = R.resample(imgf, sp, osp)
    ref_lab = R.resample(lab, sp, osp, nearest=True)
    got_img, pix = nifti_util.read(d + "/img_r.nii.gz")
    got_lab, pix_m = nifti_util.read(d + "/mask_r.nii.gz")
    nx, ny, nz = ife_b200.resampled_dims(shape[::-1], sp, osp)
    assert got_img.shape == got_lab.shape == (nz, ny, nx) == ref_img.shape
    assert pix == pix_m == tuple(float(np.float32(v)) for v in osp)
    assert got_lab.dtype == np.uint8 and _same(got_lab, ref_lab)
    assert _same(got_img, ref_img)

    p = run("ExtractFeatures", "-i", d + "/img_r.nii.gz", "-m", d + "/mask_r.nii.gz", "-o", d + "/feat", "-s", "1.2")
    assert p.returncode == 0, p.stderr
    ref = oracle.emphysema_features(ref_img, synth.clamp01(ref_lab), float(np.float32(1.2)), spacing=pix, arith=1)
    for k, nm in enumerate(oracle.FEATURE_NAMES8):
        got, _ = nifti_util.read("%s/feat_scale_1.200000%s.nii.gz" % (d, nm))
        assert (np.array_equal(got, ref[k]) if k < 2 else _eig_close(got, ref[k])), nm
