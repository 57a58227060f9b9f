"""Per-kernel CUDA-event times of the normalized convolution with a FLOAT certainty image (the reference
filter's own signature) at 512x512x400, tensor-map passes on and off.
Usage: python profiles/exp_normconv_f32.py [sigma]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "image-feature-extraction_b200"))
sys.path.insert(0, ROOT)
import torch
import bench
import ife_b200

sigma = float(sys.argv[1]) if len(sys.argv) > 1 else 1.2
dev = torch.device("cuda", 0)
ctx = ife_b200.Context(0)
nx, ny, nz = bench.DIMS
img, mask = bench.synth_scan_torch(torch, dev, 100, "lung")
cert = mask.to(torch.float32) * 0.75 + 0.125
out = torch.empty((nz, ny, nx), dtype=torch.float32, device=dev)
ref = None
for tma in (1, 0):
    ctx.set_option("tma_passes", tma)
    fn = lambda: ctx.normalized_gaussian_dev(img.data_ptr(), cert.data_ptr(), out.data_ptr(), bench.DIMS, sigma)
    for it in range(3):
        fn()
    ctx.synchronize()
    ctx.profile_enable(True)
    ctx.profile_read()
    for it in range(8):
        fn()
    r = ctx.profile_read()
    ctx.profile_enable(False)
    t = {k: round(v[0] / max(v[1], 1), 4) for k, v in r.items() if v[1] and k != "other"}
    cur = out.clone()
    same = None if ref is None else bool(torch.equal(cur, ref))
    ref = cur
    print("normalized convolution, float certainty, sigma", sigma, "tma" if tma else "plain", t, "sum_passes",
          round(sum(v for k, v in t.items() if "pass" in k), 4), "identical to previous:", same, flush=True)
ctx.close()
