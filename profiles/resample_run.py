"""Timing of ife_cuda_resample on a B200: a 512x512x160 scan at (0.7, 0.7, 2.5) mm resampled to 0.7 mm
isotropic (output 512x512x571), linear on float, nearest on float and on a uint8 mask.  Device-resident
(torch tensors, IFE_MEM_DEVICE), warm, timed with CUDA events on the context's stream over many calls.
The input (168 MB as float) is larger than the 126 MB L2, and every call writes 600 MB (float), so
no call finds its input left in L2 by the one before.
Reports ms per call, output Gvoxel/s, and the share of the HBM bound computed from the algorithmic
bytes (4 N_in + 4 N_out for float, N_in + N_out for uint8) at the data sheet's 7.7 TB/s, with the card
name and power limit read in the same run.
Usage: python profiles/resample_run.py [out.json]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "image-feature-extraction_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import ife_b200
import synth

HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU
DIMS = (512, 512, 160)            # nx, ny, nz
SPACING, OUT_SPACING = (0.7, 0.7, 2.5), (0.7, 0.7, 0.7)
WARMUP, ITERS = 5, 30


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return torch.cuda.get_device_name(0), q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    dev = torch.device("cuda", 0)
    ctx = ife_b200.Context(0)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    nx, ny, nz = DIMS
    # one 64-plane slab of the synthetic scan tiled in z (a full-size synth volume takes minutes on the host)
    slab = synth.ct_like((64, ny, nx), seed=11, n_blobs=60)
    img = torch.from_numpy(np.ascontiguousarray(np.concatenate([slab, slab[::-1], slab], 0)[:nz])).to(dev)
    mslab = synth.lung_mask((64, ny, nx))
    mask = torch.from_numpy(np.ascontiguousarray(np.concatenate([mslab, mslab[::-1], mslab], 0)[:nz])).to(dev)
    mx, my, mz = ife_b200.resampled_dims(DIMS, SPACING, OUT_SPACING)
    n_in, n_out = nx * ny * nz, mx * my * mz
    name, smi = card()
    results = {"card": name, "nvidia_smi_name_power_limit_max_sm_clock": smi, "in_dims": DIMS, "out_dims": (mx, my, mz),
               "spacing": SPACING, "out_spacing": OUT_SPACING, "iters": ITERS, "modes": {}}
    for mode, src, nearest in (("linear_f32", img, False), ("nearest_f32", img, True), ("nearest_u8", mask, True)):
        out = torch.empty((mz, my, mx), dtype=src.dtype, device=dev)
        eb = src.element_size()

        def call():
            ctx.resample_dev(src.data_ptr(), out.data_ptr(), DIMS, SPACING, OUT_SPACING, elem_bytes=eb, nearest=nearest)

        for _ in range(WARMUP):
            call()
        torch.cuda.synchronize()
        ctx.profile_enable(True)
        ctx.profile_read()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(ITERS):
            call()
        t1.record()
        torch.cuda.synchronize()
        kern_ms, launches = ctx.profile_read()["other"]
        ctx.profile_enable(False)
        ms = t0.elapsed_time(t1) / ITERS
        bytes_alg = eb * (n_in + n_out)
        results["modes"][mode] = {
            "ms_per_call": round(ms, 4),
            "kernel_ms_per_call": round(kern_ms / max(launches, 1), 4),
            "out_gvoxel_per_s": round(n_out / (ms * 1e-3) / 1e9, 2),
            "algorithmic_bytes": bytes_alg,
            "achieved_tb_per_s": round(bytes_alg / (ms * 1e-3) / 1e12, 3),
            "share_of_hbm_bound": round(bytes_alg / HBM_BYTES_PER_S / (ms * 1e-3), 3),
        }
        del out
    # the timed outputs must be the host path's (same kernels, staged copies): spot-check one mode
    chk = torch.empty((mz, my, mx), dtype=torch.float32, device=dev)
    ctx.resample_dev(img.data_ptr(), chk.data_ptr(), DIMS, SPACING, OUT_SPACING)
    host = ctx.resample(img.cpu().numpy(), SPACING, OUT_SPACING)
    torch.cuda.synchronize()
    results["device_equals_host_path"] = bool(np.array_equal(chk.cpu().numpy().view(np.uint32), host.view(np.uint32)))
    ctx.set_stream(None)
    ctx.close()
    line = json.dumps(results)
    print(line)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
