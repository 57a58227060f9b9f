"""Per-kernel CUDA-event times of the extract workload at full size (512x512x400), one scale,
all-ones and lung masks, for the tensor-map passes on and off.
Usage: [IFE_CUDA_LIB=...] python profiles/exp_passes.py [sigma]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "image-feature-extraction_b200"))
sys.path.insert(0, ROOT)
import torch
import bench
import ife_b200

sig = [float(sys.argv[1])] if len(sys.argv) > 1 else [1.2]
dev = torch.device("cuda", 0)
ctx = ife_b200.Context(0)
nx, ny, nz = bench.DIMS
out = torch.empty((1, 8, nz, ny, nx), dtype=torch.float32, device=dev)
for mask_kind in ("ones", "lung"):
    img, mask = bench.synth_scan_torch(torch, dev, 100, mask_kind)
    ref = None
    for tma in (1, 0):
        try:
            ctx.set_option("tma_passes", tma)
        except Exception:
            if tma == 0:
                continue
        fn = lambda: ctx.emphysema_features_dev(img.data_ptr(), mask.data_ptr(), out.data_ptr(), bench.DIMS, sig)
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
        cur = out[0, 0].clone()
        same = None if ref is None else bool(torch.equal(cur, ref))
        ref = cur
        print(os.path.basename(os.environ.get("IFE_CUDA_LIB", "product")), mask_kind, "tma" if tma else "plain", t,
              "sum_passes", round(sum(v for k, v in t.items() if "pass" in k), 4), "blur identical to previous:", same, flush=True)
ctx.close()
