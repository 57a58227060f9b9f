"""ife_cuda_emphysema_histograms and ife_cuda_emphysema_histograms_batch bin each scan through the
same per-scan path: a batch must give the counts of one call per scan, with the same kernel
launches, for every ROI-list regime (none, a short list searched per voxel, more than 192 ROIs
counted one block per ROI).  All three ROI-taking entry points reject a box outside the image."""
import numpy as np
import pytest

import ife_b200
import synth

pytestmark = pytest.mark.gpu

SHAPE = (24, 40, 64)       # nx % 32 == 0 and a lung mask well inside: the passes run on a crop
SIGMAS = [0.6, 1.2]


def _scans():
    imgs = [synth.ct_like(SHAPE, seed=90 + i, n_blobs=6) for i in range(3)]
    mask = synth.clamp01(synth.lung_mask(SHAPE))
    masks = [mask, np.roll(mask, 3, axis=2), np.roll(mask, -2, axis=1)]
    return imgs, masks


def _roi_lists(masks, kind):
    if kind == "none":
        return None
    if kind == "few":
        return np.stack([synth.random_rois(m, 150, (9, 7, 5), seed=i) for i, m in enumerate(masks)])
    dense = [synth.dense_rois(m, (7, 5, 3))[i::4] for i, m in enumerate(masks)]
    n = min(len(d) for d in dense)
    assert n > 192
    return np.stack([d[:n] for d in dense])


@pytest.mark.parametrize("kind", ["none", "few", "many"])
def test_batch_equals_single_calls_with_the_same_launches(ctx, kind):
    imgs, masks = _scans()
    rois = _roi_lists(masks, kind)
    edges = np.tile(np.linspace(-60, 60, 12, dtype=np.float32), (len(SIGMAS) * 8, 1))
    ctx.emphysema_histograms_batch(imgs, masks, SIGMAS, edges, rois)    # workspace grown, kernels loaded
    one, launches = [], 0
    for i in range(3):
        l0 = ctx.launch_count()
        one.append(ctx.emphysema_histograms(imgs[i], masks[i], SIGMAS, edges, None if rois is None else rois[i]))
        launches += ctx.launch_count() - l0
        assert ctx.last_work_dims() != (SHAPE[2], SHAPE[1], SHAPE[0])    # the crop was taken
    l0 = ctx.launch_count()
    batch = ctx.emphysema_histograms_batch(imgs, masks, SIGMAS, edges, rois)
    assert ctx.launch_count() - l0 == launches
    assert np.array_equal(batch, np.stack(one))
    assert batch.sum() > 0


@pytest.mark.parametrize("bad", [[0, 0, 0, 9, 1, 1], [-1, 0, 0, 2, 2, 2], [0, 0, 7, 1, 1, 2], [1, 1, 1, 0, 1, 1]])
def test_roi_outside_the_image_is_rejected_by_every_entry_point(ctx, bad):
    shape = (8, 8, 8)
    img = np.zeros(shape, np.float32)
    mask = np.ones(shape, np.uint8)
    rois = np.array([[1, 1, 1, 2, 2, 2], bad], np.int32)
    edges = np.zeros((8, 4), np.float32)
    with pytest.raises(ife_b200.IfeError, match="ROI 1 is not inside the image") as e:
        ctx.emphysema_histograms(img, mask, [1.0], edges, rois)
    assert e.value.code == -1
    with pytest.raises(ife_b200.IfeError, match="scan 1: ROI 1 is not inside the image") as e:
        ctx.emphysema_histograms_batch([img, img], [mask, mask], [1.0], edges, np.stack([rois[[0, 0]], rois]))
    assert e.value.code == -1
    with pytest.raises(ife_b200.IfeError, match="ROI 1 is not inside the image") as e:
        ctx.intensity_roi_histograms(img, mask, edges[0], rois)
    assert e.value.code == -1
