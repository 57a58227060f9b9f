"""Per-kernel CUDA-event times of the plain smoothing Gaussian (one field) and of the sigma > 0
Hessian eigen features at 512x512x400, tensor-map passes on and off.
Usage: python profiles/exp_gaussian.py [sigma]"""
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
img, _ = bench.synth_scan_torch(torch, dev, 100, "ones")
out = torch.empty((nz, ny, nx), dtype=torch.float32, device=dev)
ref = None
for tma in (1, 0):
    ctx.set_option("tma_passes", tma)
    fn = lambda: ctx.gaussian_dev(img.data_ptr(), out.data_ptr(), bench.DIMS, sigma)
    for it in range(3):
        fn()
    ctx.synchronize()
    ctx.profile_enable(True)
    ctx.profile_read()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for it in range(8):
        fn()
    r = ctx.profile_read()
    ctx.profile_enable(False)
    t = {k: round(v[0] / max(v[1], 1), 4) for k, v in r.items() if v[1] and k != "other"}
    cur = out.clone()
    same = None if ref is None else bool(torch.equal(cur, ref))
    ref = cur
    print("gaussian sigma", sigma, "tma" if tma else "plain", t, "sum_passes",
          round(sum(v for k, v in t.items() if "pass" in k), 4), "identical to previous:", same, flush=True)
ctx.close()
