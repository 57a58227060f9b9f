"""CPU reference of ife_cuda_resample: itk::ResampleImageFilter with an identity transform, the
output origin equal to the input's, LinearInterpolateImageFunction (RealType double) or
NearestNeighborInterpolateImageFunction.  The tests compare the GPU against it bit for bit.

Every step is one NumPy ufunc on float64 arrays, i.e. one IEEE-754 operation rounded once; there
is no contraction into fused multiply-adds, so this restatement computes what the kernel's
explicitly rounded __dmul_rn / __dadd_rn / __dsub_rn compute.

Constants and rules (DESIGN.md "Resampling"):
  n'_d = max(1, floor(n_d * s_d / s'_d + 0.5))                         OUTPUT_SIZE_ROUNDING = 0.5
  c_d  = (i_d * s'_d) * (1 / s_d); c_d = i_d when s'_d == s_d
  inside <=> -0.5 <= c_d < n_d - 0.5 on every axis                     BUFFER_HALF_VOXEL = 0.5
  linear : b = max(floor(c), 0), w = c - b if > 0 else 0, upper = min(b + 1, n - 1),
           lerp(a, b, w) = a + (b - a) * w along x, then y, then z, one rounding to float32
  nearest: min(floor(c + 0.5), n - 1)                                  NEAREST_ROUNDING = 0.5
"""
import math

import numpy as np

OUTPUT_SIZE_ROUNDING = 0.5
BUFFER_HALF_VOXEL = 0.5
NEAREST_ROUNDING = 0.5


def output_dims(dims, spacing, out_spacing):
    """(nx, ny, nz) of the output grid."""
    return tuple(max(1, int(math.floor(float(n) * float(s) / float(so) + OUTPUT_SIZE_ROUNDING)))
                 for n, s, so in zip(dims, spacing, out_spacing))


def _axis(n, m, s, so, nearest):
    i = np.arange(m, dtype=np.float64)
    c = i if so == s else (i * np.float64(so)) * np.float64(1.0 / s)
    inside = (c >= -BUFFER_HALF_VOXEL) & (c < np.float64(n) - BUFFER_HALF_VOXEL)
    if nearest:
        b0 = np.minimum(np.maximum(np.floor(c + NEAREST_ROUNDING), 0), n - 1).astype(np.int64)
        return b0, b0, None, inside
    b0 = np.minimum(np.maximum(np.floor(c), 0), n - 1).astype(np.int64)
    t = c - b0.astype(np.float64)
    w = np.where(t > 0, t, 0.0)
    b1 = np.minimum(b0 + 1, n - 1)
    return b0, b1, w, inside


def _lerp(a, b, w):
    return a + (b - a) * w


def resample(vol, spacing, out_spacing, nearest=False, default=0.0):
    """vol: (nz, ny, nx) float32 (linear or nearest) or uint8 (nearest); spacing / out_spacing
    (sx, sy, sz) -> (nz', ny', nx') volume of the same dtype."""
    vol = np.ascontiguousarray(vol)
    if not nearest and vol.dtype != np.float32:
        raise TypeError("linear interpolation takes float32 volumes")
    nz, ny, nx = vol.shape
    mx, my, mz = output_dims((nx, ny, nz), spacing, out_spacing)
    x0, x1, wx, ix = _axis(nx, mx, float(spacing[0]), float(out_spacing[0]), nearest)
    y0, y1, wy, iy = _axis(ny, my, float(spacing[1]), float(out_spacing[1]), nearest)
    z0, z1, wz, iz = _axis(nz, mz, float(spacing[2]), float(out_spacing[2]), nearest)
    inside = iz[:, None, None] & iy[None, :, None] & ix[None, None, :]
    if nearest:
        out = vol[np.ix_(z0, y0, x0)]
    else:
        v = vol.astype(np.float64)
        wx, wy, wz = wx[None, None, :], wy[None, :, None], wz[:, None, None]
        c00 = _lerp(v[np.ix_(z0, y0, x0)], v[np.ix_(z0, y0, x1)], wx)
        c10 = _lerp(v[np.ix_(z0, y1, x0)], v[np.ix_(z0, y1, x1)], wx)
        c01 = _lerp(v[np.ix_(z1, y0, x0)], v[np.ix_(z1, y0, x1)], wx)
        c11 = _lerp(v[np.ix_(z1, y1, x0)], v[np.ix_(z1, y1, x1)], wx)
        out = _lerp(_lerp(c00, c10, wy), _lerp(c01, c11, wy), wz).astype(np.float32)
    return np.where(inside, out, np.asarray(default).astype(vol.dtype)).astype(vol.dtype)
