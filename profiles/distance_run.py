"""Timing of ife_cuda_signed_distance_map and ife_cuda_expected_signed_distance on a B200: the
512x512x400 lung mask of tests/synth.py at unit spacing and at (0.7, 0.7, 2.5) mm.  Device-resident
(torch tensors, IFE_MEM_DEVICE for the map), warm, timed with CUDA events on the context's stream over
many calls; the device time of the calls' kernels from ife_cuda_profile_read (every kernel of these
calls is kind "other") in a separate profiled loop.  The mask (105 MB) and the map (419 MB) together exceed the
126 MB L2, so no call finds its input left in L2 by the one before.
Bytes: the compulsory 5 B/voxel (1 B of mask in, 4 B of float map out; the expected distance instead
reads 1 B of mask and 4 B of weight) over ms per call, against the data sheet's 7.7 TB/s.  The
intermediates' bytes are reported separately: the x pass writes 2 B/voxel, the y pass reads them and
writes 4 B of offsets plus 4 B of stack entries per site and reads the stack back, the z pass reads the
offsets and writes and reads 8 B of stack entries per site (at most; a site popped early is read once).
The CPU comparison is scipy.ndimage.distance_transform_edt on the same mask on the host cores.
The card name and power limit are read in the same run.
Usage: python profiles/distance_run.py [out.json]"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "image-feature-extraction_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import distance_ref
import ife_b200
import synth

HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU
SHAPE = (400, 512, 512)           # nz, ny, nx
SPACINGS = [(1.0, 1.0, 1.0), (0.7, 0.7, 2.5)]
WARMUP, ITERS = 3, 20


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return torch.cuda.get_device_name(0), q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def timed(ctx, call):
    for _ in range(WARMUP):
        call()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(ITERS):
        call()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / ITERS
    ctx.profile_enable(True)
    ctx.profile_read()
    for _ in range(ITERS):
        call()
    kern_ms, launches = ctx.profile_read()["other"]
    ctx.profile_enable(False)
    return ms, kern_ms / ITERS, launches // ITERS


def main():
    dev = torch.device("cuda", 0)
    ctx = ife_b200.Context(0)
    # a stream of its own: the legacy default stream's handle is 0, which ife_cuda_set_stream reads as
    # "the context's own stream", and the events below would then time nothing
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    mask_np = synth.lung_mask(SHAPE)
    n = mask_np.size
    mask = torch.from_numpy(mask_np).to(dev)
    out = torch.empty(SHAPE, dtype=torch.float32, device=dev)
    weight_np = np.random.default_rng(5).uniform(0, 1, SHAPE).astype(np.float32)
    dims = SHAPE[::-1]
    name, smi = card()
    n_contour = int(distance_ref.contour(mask_np).sum())
    results = {"card": name, "nvidia_smi_name_power_limit_max_sm_clock": smi, "dims": dims,
               "contour_voxels": n_contour, "iters": ITERS, "runs": []}
    compulsory = 5 * n
    intermediates = {"x_pass_write": 2 * n, "y_pass": 2 * n + 4 * n + 2 * 4 * n, "z_pass_at_most": 4 * n + 2 * 8 * n}
    results["intermediate_bytes_per_call"] = intermediates
    for sp in SPACINGS:
        ms, kern_ms, launches = timed(ctx, lambda: ctx.signed_distance_map_dev(mask.data_ptr(), out.data_ptr(), dims, sp))
        # the expected distance takes host arrays (IFE_MEM_HOST) and waits for its scalar: its time
        # includes the 525 MB upload of mask and weight
        t = time.perf_counter()
        e = ctx.expected_distance(mask_np, weight_np, spacing=sp)
        e_ms = (time.perf_counter() - t) * 1e3
        _, e_kern_ms, e_launches = timed(ctx, lambda: ctx.expected_distance(mask_np, weight_np, spacing=sp))
        t = time.perf_counter()
        distance_ref.squared_scipy(mask_np, sp)
        cpu_s = time.perf_counter() - t
        results["runs"].append({
            "spacing": sp,
            "map_ms_per_call": round(ms, 3),
            "map_kernel_ms_per_call": round(kern_ms, 3),
            "map_launches_per_call": launches,
            "map_compulsory_tb_per_s": round(compulsory / (ms * 1e-3) / 1e12, 3),
            "map_share_of_hbm_bound": round(compulsory / HBM_BYTES_PER_S / (ms * 1e-3), 3),
            "expected_distance": e,
            "expected_host_call_ms": round(e_ms, 2),
            "expected_kernel_ms_per_call": round(e_kern_ms, 3),
            "expected_launches_per_call": e_launches,
            "scipy_edt_with_indices_s": round(cpu_s, 2),
            "host_cores": os.cpu_count(),
        })
        print(json.dumps(results["runs"][-1]), flush=True)
    ctx.set_stream(None)
    ctx.close()
    line = json.dumps(results)
    print(line)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
