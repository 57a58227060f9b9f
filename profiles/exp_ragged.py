"""Per-pass CUDA-event times of the Gaussian passes on layouts the tensor-map kernels cannot take
(nx not a multiple of 16 with a uint8 certainty, nx not a multiple of 4 for one field), where
the plain register-staged kernels run: normalized convolution with a uint8 mask on 500x500x400
and the plain Gaussian on 510x512x400, device-resident, sigma 1.2.  Prints ms per launch of each
pass for several repeats, and a sha256 of each result so that two builds can be compared.
Usage: [IFE_CUDA_LIB=...] python profiles/exp_ragged.py [repeats]"""
import hashlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "image-feature-extraction_b200"))
import torch
import ife_b200

repeats = int(sys.argv[1]) if len(sys.argv) > 1 else 5
dev = torch.device("cuda", 0)
ctx = ife_b200.Context(0)
g = torch.Generator(device=dev).manual_seed(7)
tag = os.environ.get("IFE_CUDA_LIB", "in-tree")


def run(name, dims, fn, out):
    for _ in range(3):
        fn()
    ctx.synchronize()
    for r in range(repeats):
        ctx.profile_enable(True)
        ctx.profile_read()
        for _ in range(10):
            fn()
        t = ctx.profile_read()
        ctx.profile_enable(False)
        per = {k[len("gauss_pass_"):]: round(v[0] / v[1], 4) for k, v in t.items() if k.startswith("gauss_pass") and v[1]}
        print(tag, name, "x".join(map(str, dims)), "repeat", r, per, "sum", round(sum(per.values()), 4), flush=True)
    print(tag, name, "sha256", hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest(), flush=True)


nx, ny, nz = 500, 500, 400
img = torch.randn((nz, ny, nx), generator=g, device=dev) * 300 - 500
mask = (torch.rand((nz, ny, nx), generator=g, device=dev) < 0.7).to(torch.uint8)
out = torch.empty_like(img)
L = ctx.L
run("normalized_gaussian_u8", (nx, ny, nz),
    lambda: ctx._check(L.ife_cuda_normalized_gaussian(ctx.h, img.data_ptr(), None, mask.data_ptr(), out.data_ptr(),
                                                      ife_b200._i3((nx, ny, nz)), ife_b200._d3(None), 1.2, 0,
                                                      ife_b200.MEM_DEVICE)),
    out)
del img, mask, out

nx, ny, nz = 510, 512, 400
img = torch.randn((nz, ny, nx), generator=g, device=dev) * 300 - 500
out = torch.empty_like(img)
run("gaussian", (nx, ny, nz), lambda: ctx.gaussian_dev(img.data_ptr(), out.data_ptr(), (nx, ny, nz), 1.2), out)
ctx.close()
