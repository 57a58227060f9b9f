"""CPU reference of the signed distance map (ife_cuda_signed_distance_map) and the expected distance
(ife_cuda_expected_signed_distance).  Volumes are (nz, ny, nx); spacing is (sx, sy, sz).

D(v) = min over contour voxels c of fl(fl(fl((dx*sx)^2) + fl((dy*sy)^2)) + fl((dz*sz)^2)), each square
t * t of t = d * s, every numpy float64 operation one rounded IEEE operation in this order."""
import math

import numpy as np

FLT_MAX = np.float32(np.finfo(np.float32).max)


def contour(mask):
    """Object voxels (mask != 0) with a background voxel among their 26 neighbours inside the image;
    voxels outside the image are not background."""
    obj = np.asarray(mask) != 0
    bg = np.pad(~obj, 1, constant_values=False)
    near = np.zeros_like(obj)
    nz, ny, nx = obj.shape
    for dz in range(3):
        for dy in range(3):
            for dx in range(3):
                near |= bg[dz:dz + nz, dy:dy + ny, dx:dx + nx]
    return obj & near


def _d(dx, dy, dz, spacing):
    sx, sy, sz = (float(s) for s in spacing)
    tx, ty, tz = dx * sx, dy * sy, dz * sz
    return (tx * tx + ty * ty) + tz * tz


def squared_brute(mask, spacing=(1.0, 1.0, 1.0), chunk=2048, voxels=None):
    """D at every voxel (or at the flat indices `voxels`) by a minimum over all contour voxels;
    None when there is no contour voxel."""
    c = np.argwhere(contour(mask)).astype(np.float64)
    if len(c) == 0:
        return None
    shape = np.asarray(mask).shape
    idx = np.arange(int(np.prod(shape))) if voxels is None else np.asarray(voxels)
    out = np.empty(idx.size, np.float64)
    for a in range(0, idx.size, chunk):
        z, y, x = (v.astype(np.float64) for v in np.unravel_index(idx[a:a + chunk], shape))
        D = _d(x[:, None] - c[None, :, 2], y[:, None] - c[None, :, 1], z[:, None] - c[None, :, 0], spacing)
        out[a:a + chunk] = D.min(1)
    return out.reshape(shape) if voxels is None else out


def squared_scipy(mask, spacing=(1.0, 1.0, 1.0)):
    """D from the nearest contour voxel scipy's exact EDT picks, recomputed in the order above (for
    volumes too large for the brute force)."""
    from scipy import ndimage
    cont = contour(mask)
    if not cont.any():
        return None
    sx, sy, sz = spacing
    iz, iy, ix = ndimage.distance_transform_edt(~cont, sampling=(sz, sy, sx), return_distances=False,
                                                return_indices=True)
    z, y, x = np.indices(cont.shape, dtype=np.int32)
    return _d((x - ix).astype(np.float64), (y - iy).astype(np.float64), (z - iz).astype(np.float64), spacing)


def signed(mask, D, inside_positive=False, squared=False):
    """The float32 map from D (None: no contour voxel anywhere)."""
    obj = np.asarray(mask) != 0
    if D is None:
        v = np.full(obj.shape, FLT_MAX, np.float32)
    else:
        v = (D if squared else np.sqrt(D)).astype(np.float32)
    neg = ~obj if inside_positive else obj
    return np.where(neg & (v != 0), -v, v).astype(np.float32)


def signed_distance_map(mask, spacing=(1.0, 1.0, 1.0), inside_positive=False, squared=False):
    return signed(mask, squared_brute(mask, spacing), inside_positive, squared)


def expected(dist_map, weight, region=None):
    """sum w * d / sum w with math.fsum (correctly rounded sums) over region != 0."""
    sel = np.ones(dist_map.shape, bool) if region is None else np.asarray(region) != 0
    w = np.asarray(weight, np.float64)[sel]
    d = np.asarray(dist_map, np.float64)[sel]
    return math.fsum(w * d) / math.fsum(w)
