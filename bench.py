#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json metric: Gvoxel/s, multi-scale Hessian eigen
features, 512^2 x 400 CT; % HBM peak).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                  [--workload extract|hist|slab] [--mask ones|lung] [--arith fma|plain]
                  [--rois N] [--no-box] [--overlap] [--no-e2e] [--no-cpu-baseline]
                  [--no-hist] [--no-slab] [--slab-size S] [--slab-steps K] [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic scan: ImageToEmphysemaFeaturesFilter
semantics (masked normalized convolution -> gradient magnitude -> fused Hessian/eigen
features -> mask) at sigma in {0.6, 1.2, 2.4, 4.8}, eight float feature volumes written per
scale (tools/ExtractFeatures.cxx semantics, BASELINE.json configs[1]).  Units = voxel-scales
(nx*ny*nz*|sigma|).  N > 1: one process per GPU (torchrun), one scan per GPU, no data-path
collective (weak scaling).  That is the HEADLINE (`metric`, `value`, `roofline`, `e2e`,
`cpu_baseline`).  The same JSON line carries two more measured legs:

  "hist": BASELINE.json configs[2] / [4] -- the same features binned into DenseHistograms
          instead of written (MakeBag semantics), lung-shaped mask, 40 equalized edges per
          (scale, feature): whole-mask histograms and 50 fixed-seed 41^3 ROIs, device-resident and
          end to end (one call and a batch of 8 scans), with an ORACLE parity block on a
          64-plane sample that contains the mask boundary;
  "slab": BASELINE.json configs[3] -- ONE 1024^3 volume cut into z-slabs over the N ranks
          through ife_cuda_slab_emphysema_features with feature volumes AND histograms on (NCCL
          halo send/recv + histogram all-reduce; strong scaling), with a parity block against the
          single-GPU entry point run on the whole volume on every rank.

`--workload hist|slab` make that leg the headline of a focused run (profiles/ scripts).

Prints ONE JSON line (rank 0).  `value` is device-resident throughput (CUDA events on the
launching stream, max over ranks); `e2e` goes through the C ABI with pinned HOST buffers, H2D
and D2H inside the timed region; `roofline` is the dominant kernel's algorithmic bytes / its
measured launch time against MEASURED_PEAKS.json; `cpu_baseline` is the CPU oracle timed on
this box's host cores on a bounded sample of the same workload.  Every timed loop runs
--steps K steps (the slab leg: --slab-steps when given; a step of the hist leg's batch
sub-legs is one call of 8 scans).

--dump-outputs DIR (rank 0) writes, right after each leg's timed steps, what its last step
returned to the caller, so that two builds can be compared output for output on the same
seeded inputs:
  extract_features.npy        float32 (n_sigma, 8, DUMP_VOXELS)  the feature volumes at
                              DUMP_VOXELS voxel positions drawn with a fixed seed
  hist_edges.npy              float32 (n_sigma*8, 40)  the edges the hist leg bins with (derived
                              from the scan's features by the library under test)
  hist_whole_mask_counts.npy  float64 (1, n_sigma*8, 41)
  hist_rois_counts.npy        float64 (min(rois, DUMP_ROIS), n_sigma*8, 41)  the first ROIs' counts
  slab_features.npy           float32 (scales in the last call, 8, DUMP_VOXELS) of rank 0's slab
  slab_edges.npy              float32 (n_sigma*8, 40)  like hist_edges, from the first 64 planes
  slab_counts.npy             float64 (n_sigma*8, 41)
At most 2 x 4 x 8 x DUMP_VOXELS x 4 B = 32 MB of samples plus 11 MB of counts.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True       # the benchmark writes nothing into the (possibly read-only) tree
sys.path.insert(0, os.path.join(ROOT, "image-feature-extraction_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

SIGMAS = [0.6, 1.2, 2.4, 4.8]
DIMS = (512, 512, 400)               # nx, ny, nz
METRIC = "Gvoxel/s multi-scale Hessian eigen features, 512^2x400 CT"
# algorithmic bytes per voxel-scale per kernel (SURVEY.md section 8d, pipeline P2 = 78 B):
#   z pass r(4 img + 1 mask) w8 | x pass r8 w8 | y pass r8 w4 (divide fused) | fused r(4+1) w32
ALGO_BYTES = {"gauss_pass_z": 13, "gauss_pass_x": 16, "gauss_pass_y": 12, "features_fused": 37}
ALGO_BYTES_HIST = {"gauss_pass_z": 13, "gauss_pass_x": 16, "gauss_pass_y": 12, "features_fused": 5}
# what limits each kernel according to the ncu captures under profiles/ (HBM is < 60 % busy in
# all of them): the passes by FP64-pipe issue + dependent-chain latency, the fused kernel by
# instruction issue
BOUND_NCU = {"gauss_pass_z": "issue+fp64", "gauss_pass_x": "hbm+fp64", "gauss_pass_y": "issue+fp64", "features_fused": "issue"}
CPU_SAMPLE_NZ = 64                   # CPU arms (cpu_baseline, --impl reference): 512 x 512 x 64, all four scales
CPU_SAMPLE = "%dx%dx%d sub-volume x %d scales" % (DIMS[0], DIMS[1], CPU_SAMPLE_NZ, len(SIGMAS))
HIST_SAMPLE_Z0 = 32                  # hist parity sample: planes [32, 96) -- the lung mask starts at z = 50
N_EDGES = 40
DUMP_VOXELS = 1 << 17                # --dump-outputs: voxel positions sampled from each feature stack
DUMP_ROIS = 1000                     # --dump-outputs: ROI histograms written at most
WORKLOAD = ("ExtractFeatures multi-scale eigen features (8 masked feature volumes per scale) on one "
            "512x512x400 float CT-like scan per GPU, sigma{0.6,1.2,2.4,4.8}; the CPU arms (cpu_baseline, "
            "--impl reference) time a bounded sample of it per step: " + CPU_SAMPLE)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6553.3, "B200 device-copy bandwidth of BASELINE.md (no MEASURED_PEAKS.json)"


def traffic_for(workload, kernel):
    """dram bytes per launch from an `ncu --set full` capture, keyed by workload/kernel
    (profiles/traffic.json); None when that instantiation was not captured."""
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(tp):
        return None
    return json.load(open(tp)).get(workload, {}).get(kernel)


class ClockSampler:
    """Streams nvidia-smi clocks / throttle reasons (one process, -lms 100) while the timed
    region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread = index, [], None, None

    def _loop(self):
        for line in self.proc.stdout:
            cells = [c.strip() for c in line.strip().split(",")]
            if len(cells) >= 6:
                self.rows.append((time.perf_counter(), cells))

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()
        t0 = time.perf_counter()
        while not self.rows and time.perf_counter() - t0 < 3.0:   # wait for the first sample
            time.sleep(0.01)
        self.t_begin = time.perf_counter()

    def stop(self):
        t_end = time.perf_counter()
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=3)
            except Exception:
                self.proc.kill()
        rows = [c for (t, c) in self.rows if getattr(self, "t_begin", 0) <= t <= t_end + 0.15] or [c for (_, c) in self.rows]
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def synth_volume_torch(torch, device, seed, shape, z_range=None):
    """CT-like volume generated on the device (same recipe as tests/synth.py in spirit: smooth
    structures + tube + plate + noise).  shape = (nz, ny, nx); z_range = (z0, z1) builds only
    those planes of the same global volume (noise seeded per plane, so slabs agree)."""
    nz, ny, nx = shape
    z0, z1 = z_range or (0, nz)
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    coarse = torch.randn((1, 1, nz // 16 + 1, ny // 16 + 1, nx // 16 + 1), generator=g, device=device)
    if z_range is None:
        img = torch.nn.functional.interpolate(coarse, size=(nz, ny, nx), mode="trilinear", align_corners=True)[0, 0]
    else:   # the same trilinear interpolation, evaluated plane range by plane range
        img = torch.empty((z1 - z0, ny, nx), dtype=torch.float32, device=device)
        ys = torch.linspace(-1, 1, ny, device=device)
        xs = torch.linspace(-1, 1, nx, device=device)
        for a in range(z0, z1, 32):
            b = min(a + 32, z1)
            zs = torch.linspace(-1, 1, nz, device=device)[a:b]
            zz, yy, xx = torch.meshgrid(zs, ys, xs, indexing="ij")
            grid = torch.stack((xx, yy, zz), dim=-1)[None]
            img[a - z0:b - z0] = torch.nn.functional.grid_sample(coarse, grid, mode="bilinear", align_corners=True)[0, 0]
            del grid, zz, yy, xx
    img = img * 300.0 - 800.0
    y = torch.arange(ny, device=device, dtype=torch.float32)[None, :, None]
    x = torch.arange(nx, device=device, dtype=torch.float32)[None, None, :]
    img += 500.0 * torch.exp(-((y - ny * 0.37) ** 2 + (x - nx * 0.61) ** 2) / 8.0)
    img += 300.0 * torch.exp(-((y - ny * 0.7) ** 2) / 4.5)
    for a in range(z0, z1, 64):     # noise: one generator state per 64-plane block of the global volume
        b = min(a + 64, z1)
        gb = torch.Generator(device=device)
        gb.manual_seed(seed * 100003 + a // 64)
        blk = torch.randn((64, ny, nx), generator=gb, device=device)
        img[a - z0:b - z0] += 30.0 * blk[a % 64:a % 64 + (b - a)]
        del blk
    return img.contiguous()


def synth_scan_torch(torch, device, seed, mask_kind):
    """One 512x512x400 scan and a lung-shaped or all-ones mask."""
    nx, ny, nz = DIMS
    img = synth_volume_torch(torch, device, seed, (nz, ny, nx))
    if mask_kind == "ones":
        mask = torch.ones((nz, ny, nx), dtype=torch.uint8, device=device)
    else:
        import synth
        mask = torch.from_numpy(synth.clamp01(synth.lung_mask((nz, ny, nx)))).to(device)
    return img, mask


def equalized_edges_from_scan(torch, ctx, img, mask, n_edges, dims=None):
    """40 equal-frequency edges per (scale, feature), as MakeBag gets them from
    DetermineHistogramBinEdges_MultiScaleEigenvalueFeatures: quantiles of a 2 M-voxel sample of
    the in-mask feature values of this scan (set-up, outside the timed region)."""
    import numpy as np
    nx, ny, nz = dims or DIMS
    dev = img.device
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    inside = torch.nonzero(mask.reshape(-1), as_tuple=False).reshape(-1)
    pick = inside[torch.randint(0, inside.numel(), (2_000_000,), generator=g, device=dev)]
    q = torch.linspace(0.0, 1.0, n_edges + 2, device=dev, dtype=torch.float64)[1:-1]
    feats = torch.empty((1, 8, nz, ny, nx), dtype=torch.float32, device=dev)
    rows = []
    for s in SIGMAS:
        ctx.emphysema_features_dev(img.data_ptr(), mask.data_ptr(), feats.data_ptr(), (nx, ny, nz), [s])
        ctx.synchronize()
        for k in range(8):
            v = torch.sort(feats[0, k].reshape(-1)[pick].to(torch.float64)).values
            rows.append(v[(q * (v.numel() - 1)).long()].to(torch.float32))
        torch.cuda.synchronize()   # torch's stream has read `feats` before the library (own stream) overwrites it
    del feats
    edges = torch.stack(rows).cpu().numpy()
    # strictly increasing rows keep every bin meaningful even where a feature saturates
    for r in edges:
        for j in range(1, len(r)):
            if not r[j] > r[j - 1]:
                r[j] = np.nextafter(r[j - 1], np.float32(np.inf))
    return np.ascontiguousarray(edges, np.float32)


def cpu_sample_inputs(mask_kind, seed=2):
    """The bounded sample both CPU arms run: 512 x 512 x 64 planes, numpy."""
    import numpy as np
    import synth
    nx, ny, _ = DIMS
    shape = (CPU_SAMPLE_NZ, ny, nx)
    img = synth.ct_like(shape, seed=seed, n_blobs=64)
    mask = (np.ones(shape, np.uint8) if mask_kind == "ones"
            else synth.clamp01(synth.lung_mask((400, ny, nx)))[HIST_SAMPLE_Z0:HIST_SAMPLE_Z0 + CPU_SAMPLE_NZ])
    return img, np.ascontiguousarray(mask)


def run_reference(args, out_stream):
    """--impl reference: the reference's CPU path (oracle port + the reference's own functor
    header; ITK itself cannot be built in this image) on this box's host cores.  Same metric,
    config and arithmetic mode as the GPU arm; each step is the bounded sample the GPU arm's
    cpu_baseline uses (512x512x64 planes x 4 scales)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    O.build()
    cores = os.cpu_count() or 1
    img, mask = cpu_sample_inputs(args.mask)
    units = img.size * len(SIGMAS)
    oarith = O.ARITH_FMA if args.arith == "fma" else O.ARITH_PLAIN

    def step():
        for s in SIGMAS:
            O.emphysema_features_reference_arm(img, mask, s, arith=oarith, threads=cores)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    val = units / dt / 1e9
    out_stream.emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Gvoxel/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64 recursion / f32 stencil+solver",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "mask": args.mask, "arith": args.arith,
                   "parallelism": "1 scan per GPU, no data-path collective",
                   "l2": "inputs (525 MB/scan) and every intermediate are larger than the 126 MB L2; no flush needed"},
        "cpu_baseline": {"value": val, "unit": "Gvoxel/s", "cores": cores,
                         "kind": "port", "reference_functor_compiled": bool(O.ref_available()),
                         "sample": CPU_SAMPLE + " per step (ITK stages restated; per-voxel functor = reference header)"},
        "e2e": {"value": val, "unit": "Gvoxel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def feature_parity(np, gpu, ref, arith):
    """SURVEY.md section 8d parity metrics for (n_sigma, 8, nz, ny, nx) feature stacks."""
    same = (gpu == ref) | (np.isnan(gpu) & np.isnan(ref))
    lam_ref, lam_gpu = ref[:, 2:5], gpu[:, 2:5]
    scale = np.abs(lam_ref).max(1)
    err = np.abs(lam_gpu.astype(np.float64) - lam_ref).max(1)
    rel = np.where(scale > 0, err / np.where(scale > 0, scale, 1), 0.0)
    order_ok = (np.abs(lam_gpu[:, 0]) >= np.abs(lam_gpu[:, 1])) & (np.abs(lam_gpu[:, 1]) >= np.abs(lam_gpu[:, 2]))
    order_ref = (np.abs(lam_ref[:, 0]) >= np.abs(lam_ref[:, 1])) & (np.abs(lam_ref[:, 1]) >= np.abs(lam_ref[:, 2]))
    return {"values_compared": int(ref.size), "values_differing": int((~same).sum()),
            "eig_max_rel_err": float(rel.max()), "eig_p99_rel_err": float(np.percentile(rel, 99)),
            "eig_frac_gt_1e-4": float((rel > 1e-4).mean()),
            "ordering_mismatches_vs_oracle": int((order_ok != order_ref).sum()), "arith": arith}


def cpu_baseline(ctx, arith):
    """Times the CPU oracle on the bounded sample and, with the oracle's output in hand, reports
    the parity of the CUDA path on that same sample, plus the reference's own build-flag noise
    floor: what changes between a PLAIN and an FMA build of the same CPU code."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle as O
    import synth
    O.build()
    cores = os.cpu_count() or 1
    img, mask = cpu_sample_inputs("ones")
    oarith = O.ARITH_FMA if arith == "fma" else O.ARITH_PLAIN
    ref = []
    t0 = time.perf_counter()
    for s in SIGMAS:
        ref.append(O.emphysema_features_reference_arm(img, mask, s, arith=oarith, threads=cores))
    dt = time.perf_counter() - t0
    ref = np.stack(ref)
    gpu = ctx.emphysema_features(img, mask, SIGMAS)
    parity = feature_parity(np, gpu, ref, arith)
    parity["sample_voxel_scales"] = int(img.size * len(SIGMAS))
    parity["note"] = ("GPU vs CPU oracle (same arithmetic mode) on the cpu_baseline sample; "
                      "bit-identical when values_differing == 0")
    # build-flag noise floor of the reference itself: oracle PLAIN vs oracle FMA, same inputs
    other = np.stack([O.emphysema_features_reference_arm(img, mask, s, arith=O.ARITH_PLAIN if arith == "fma" else O.ARITH_FMA,
                                                         threads=cores) for s in SIGMAS])
    noise = feature_parity(np, other, ref, "plain-vs-fma")
    edges = np.stack([synth.equalized_edges(ref[s, k].reshape(-1), N_EDGES) for s in range(len(SIGMAS)) for k in range(8)])
    shp = (-1,) + ref.shape[2:]
    ca = O.features_histograms(ref.reshape(shp), mask, edges)
    cb = O.features_histograms(other.reshape(shp), mask, edges)
    noise["hist_sum_abs_dcount"] = int(np.abs(ca.astype(np.int64) - cb.astype(np.int64)).sum())
    noise["hist_inserts"] = int(ca.sum())
    noise["note"] = ("CPU oracle built PLAIN vs built FMA (what -mfma changes in the reference's own output): the "
                     "floor below which bit-exactness buys nothing")
    parity["reference_build_flag_noise"] = noise
    return {"value": img.size * len(SIGMAS) / dt / 1e9, "unit": "Gvoxel/s", "cores": cores,
            "kind": "port", "reference_functor_compiled": bool(O.ref_available()),
            "sample": CPU_SAMPLE + ", %.1f s of CPU work (ITK stages restated; per-voxel functor = reference header)" % dt}, parity


class QuietStdout:
    """Routes fd 1 to stderr while the benchmark runs (NCCL and friends print banners on
    stdout) so that the JSON line is the ONLY thing this process writes to stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, line):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        print(line, flush=True)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def bind_to_gpu_numa_node(index):
    """CPU affinity of this process := the CPUs NVML reports as local to GPU `index`.
    Returns a short description for the JSON line (or why nothing was done)."""
    if os.environ.get("IFE_BENCH_NO_BIND"):
        return "off (IFE_BENCH_NO_BIND)"
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].strip().isdigit() else index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = (cpus & allowed) or allowed
        os.sched_setaffinity(0, cpus)
        return "NUMA-local to GPU %d: %d CPUs" % (phys, len(cpus))
    except Exception as e:      # no NVML, restricted container: stay where we are
        return "unchanged (%s)" % type(e).__name__


class Env:
    """Everything a leg needs: torch, the process group, the context and its stream."""

    def __init__(self, args):
        import torch
        import ife_b200
        self.torch, self.ife = torch, ife_b200
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback "
                             "(use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        # run on the CPUs next to this GPU's PCIe root, so that the page-locked host buffers of the
        # e2e legs are first-touched on the local NUMA node (every rank otherwise lands on node 0)
        self.affinity = bind_to_gpu_numa_node(self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self.warmup = max(args.warmup, 3)
        self.ctx = ife_b200.Context(self.local_rank, arith=ife_b200.ARITH_FMA if args.arith == "fma" else ife_b200.ARITH_PLAIN)
        self.stream = torch.cuda.Stream(device=self.dev)
        self.ctx.set_stream(self.stream.cuda_stream)
        if args.no_box:
            self.ctx.set_option("support_box", 0)
        if args.overlap:
            self.ctx.set_option("overlap_scales", 1)
        self.peak, self.peak_src = measured_peaks()

    def max_over_ranks(self, v):
        if not self.dist:
            return float(v)
        t = self.torch.tensor([v], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v):
        if not self.dist:
            return float(v)
        t = self.torch.tensor([v], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, step, steps, warmup, clocks=False):
        """W untimed steps, then K steps between CUDA events on the launching stream, bracketed by
        barrier + synchronize on both sides -> (ms total, max over ranks; launches; per-kind
        profile of rank-local launches; clocks on rank 0)."""
        torch, ctx = self.torch, self.ctx
        with torch.cuda.stream(self.stream):
            for _ in range(warmup):
                step()
            torch.cuda.synchronize()
            sampler = ClockSampler(self.local_rank) if clocks and self.rank == 0 else None
            if sampler:
                sampler.start()          # before the barrier: its start-up must not skew the ranks
            self.barrier()
            ctx.profile_enable(True)
            l0 = ctx.launch_count()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(self.stream)
            for _ in range(steps):
                step()
            ev1.record(self.stream)
            torch.cuda.synchronize()
            self.barrier()
            ms = ev0.elapsed_time(ev1)
            launches = ctx.launch_count() - l0
            prof = ctx.profile_read()
            ctx.profile_enable(False)
            clk = sampler.stop() if sampler else None
        return self.max_over_ranks(ms), launches, prof, clk


def kernel_table(env, prof, algo, voxels_per_launch, ms_total, workload_key):
    """Per-kernel CUDA-event time -> achieved algorithmic GB/s and fraction of the HBM peak."""
    kinds = {k: v for k, v in prof.items() if v[1] > 0 and k in algo}
    table = {}
    for k, (tms, cnt) in kinds.items():
        gbs = algo[k] * voxels_per_launch / (tms / cnt * 1e-3) / 1e9
        table[k] = {"ms_per_launch": tms / cnt, "launches": cnt, "algo_bytes_per_voxel": algo[k],
                    "achieved_gbs": gbs, "frac": gbs / env.peak, "share_of_step": tms / ms_total,
                    "bound_ncu": BOUND_NCU.get(k), "traffic": traffic_for(workload_key, k)}
    return table


def dump_output(env, name, arr):
    """--dump-outputs: DIR/<name>.npy from rank 0.  arr: numpy, or a device tensor of counts."""
    if not env.args.dump_outputs or env.rank != 0:
        return
    import numpy as np
    if not isinstance(arr, np.ndarray):
        arr = arr.to(env.torch.float64).cpu().numpy()
    os.makedirs(env.args.dump_outputs, exist_ok=True)
    np.save(os.path.join(env.args.dump_outputs, name + ".npy"), arr)


def dump_feature_sample(env, name, feats):
    """--dump-outputs: (S, 8, nz, ny, nx) device features -> (S, 8, DUMP_VOXELS) float32 at voxel
    positions drawn with a fixed seed (the same positions for every build and run)."""
    if not env.args.dump_outputs or env.rank != 0:
        return
    import numpy as np
    nvox = feats[0, 0].numel()
    idx = np.sort(np.random.default_rng(0).choice(nvox, size=min(DUMP_VOXELS, nvox), replace=False))
    pick = env.torch.from_numpy(idx).to(feats.device)
    dump_output(env, name, feats.reshape(feats.shape[:2] + (nvox,))[:, :, pick].cpu().numpy())


# ------------------------------------------------------------------------------------------
# headline leg: ExtractFeatures semantics, one scan per GPU
# ------------------------------------------------------------------------------------------
def leg_extract(env, img, mask):
    import ctypes as C
    torch, ctx, args = env.torch, env.ctx, env.args
    nx, ny, nz = DIMS
    n = nx * ny * nz
    units = n * len(SIGMAS)
    out = torch.empty((len(SIGMAS), 8, nz, ny, nx), dtype=torch.float32, device=env.dev)
    torch.cuda.synchronize()

    def step():
        ctx.emphysema_features_dev(img.data_ptr(), mask.data_ptr(), out.data_ptr(), DIMS, SIGMAS)

    ms, launches, prof, clocks = env.timed(step, args.steps, env.warmup, clocks=True)
    dump_feature_sample(env, "extract_features", out)     # before the other arithmetic mode overwrites `out`
    ms_per_step = ms / args.steps
    value = env.world * units / (ms_per_step * 1e-3) / 1e9
    wd = ctx.last_work_dims()
    nwork = wd[0] * wd[1] * wd[2]
    table = kernel_table(env, prof, ALGO_BYTES, n, ms, "extract_" + args.mask)
    for k in ("gauss_pass_z", "gauss_pass_x", "gauss_pass_y"):      # the passes run on the crop when there is one
        if k in table and nwork != n:
            table[k]["frac_of_bytes_moved"] = table[k]["frac"] * nwork / n
    dom = max(table, key=lambda k: table[k]["ms_per_launch"] * table[k]["launches"])
    pipe_b = sum(ALGO_BYTES.values())
    roofline = {"bound": "hbm", "kernel": dom, "achieved": table[dom]["achieved_gbs"], "peak": env.peak,
                "unit": "GB/s", "frac": table[dom]["frac"], "traffic": table[dom]["traffic"],
                "peak_source": env.peak_src, "limiter_ncu": BOUND_NCU.get(dom), "kernels": table,
                "note": "bound = the roofline the fraction is taken against (the path's minimum bytes over the measured "
                        "HBM copy bandwidth); limiter_ncu = what ncu shows the kernel waiting on",
                "pipeline": {"algo_bytes_per_voxel_scale": pipe_b,
                             "achieved_gbs": pipe_b * units / (ms_per_step * 1e-3) / 1e9,
                             "frac": pipe_b * units / (ms_per_step * 1e-3) / 1e9 / env.peak}}
    # the other arithmetic mode of the recursion (the reference built without / with FMA contraction:
    # a stock x86-64 build is PLAIN), a short device-resident measurement for the record
    other = None
    if env.world == 1:
        alt = env.ife.ARITH_PLAIN if args.arith == "fma" else env.ife.ARITH_FMA
        ctx.set_arith(alt)
        try:
            ms_o, _, _, _ = env.timed(step, args.steps, 2, clocks=False)
        finally:
            ctx.set_arith(env.ife.ARITH_FMA if args.arith == "fma" else env.ife.ARITH_PLAIN)
        other = {"arith": "plain" if args.arith == "fma" else "fma", "ms_per_step": ms_o / args.steps,
                 "value": units / (ms_o / args.steps * 1e-3) / 1e9, "unit": "Gvoxel/s",
                 "note": "same workload, device-resident, the recursion's other arithmetic mode (bit-exact against the oracle in that mode)"}
    e2e = None
    if not args.no_e2e:
        h_img = torch.empty((nz, ny, nx), dtype=torch.float32, pin_memory=True).copy_(img)
        h_mask = torch.empty((nz, ny, nx), dtype=torch.uint8, pin_memory=True).copy_(mask)
        del out
        torch.cuda.empty_cache()
        h_out = torch.empty((len(SIGMAS), 8, nz, ny, nx), dtype=torch.float32, pin_memory=True)
        dims_c, sp_c = (C.c_int * 3)(*DIMS), (C.c_double * 3)(1, 1, 1)
        sig_c = (C.c_double * len(SIGMAS))(*SIGMAS)

        def e2e_step():
            ctx._check(ctx.L.ife_cuda_emphysema_features(ctx.h, C.c_void_p(h_img.data_ptr()), C.c_void_p(h_mask.data_ptr()),
                                                         C.c_void_p(h_out.data_ptr()), dims_c, sp_c, sig_c, len(SIGMAS),
                                                         env.ife.MEM_HOST))
        e_steps = args.steps
        for _ in range(2):
            e2e_step()
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            e2e_step()          # synchronous: returns when the outputs are in host memory
        torch.cuda.synchronize()
        dt = env.max_over_ranks((time.perf_counter() - t0) / e_steps)
        e2e = {"value": env.world * units / dt / 1e9, "unit": "Gvoxel/s", "ms_per_step": dt * 1e3, "steps": e_steps,
               "h2d_bytes_per_step": int(h_img.numel() * 4 + h_mask.numel()), "d2h_bytes_per_step": int(h_out.numel() * 4),
               "api": "ife_cuda_emphysema_features(..., IFE_MEM_HOST) with pinned host buffers"}
        del h_out, h_img, h_mask
    else:
        del out
    torch.cuda.empty_cache()
    return {"value": value, "ms_per_step": ms_per_step, "roofline": roofline, "e2e": e2e,
            "launches": launches, "clocks": clocks, "other_arith": other}


# ------------------------------------------------------------------------------------------
# hist leg: MakeBag semantics (configs[2] and [4]), lung mask
# ------------------------------------------------------------------------------------------
def hist_parity_vs_oracle(env):
    """GPU histograms (whole mask and 50 ROIs) against the CPU oracle on a 64-plane sample of the
    lung-masked scan that contains the mask boundary (planes 32..96; the mask starts at z = 50)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle as O
    import synth
    O.build()
    cores = os.cpu_count() or 1
    img, mask = cpu_sample_inputs("lung", seed=3)
    oarith = O.ARITH_FMA if env.args.arith == "fma" else O.ARITH_PLAIN
    ref = np.stack([O.emphysema_features_reference_arm(img, mask, s, arith=oarith, threads=cores) for s in SIGMAS])
    inside = mask != 0
    edges = np.stack([synth.equalized_edges(ref[s, k][inside], N_EDGES) for s in range(len(SIGMAS)) for k in range(8)])
    feats = ref.reshape((-1,) + ref.shape[2:])
    rois = synth.random_rois(mask, 50, (41, 41, 41), seed=7)
    ref_whole = O.features_histograms(feats, mask, edges)
    ref_rois = O.features_histograms(feats, mask, edges, rois)
    gpu = env.ctx.emphysema_features(img, mask, SIGMAS)
    g_whole = env.ctx.emphysema_histograms(img, mask, SIGMAS, edges)
    g_rois = env.ctx.emphysema_histograms(img, mask, SIGMAS, edges, rois)
    par = feature_parity(np, gpu, ref, env.args.arith)
    par.update({
        "sample": "%dx%dx%d planes [%d, %d) of the lung-masked volume (mask boundary inside), all %d scales" %
                  (DIMS[0], DIMS[1], CPU_SAMPLE_NZ, HIST_SAMPLE_Z0, HIST_SAMPLE_Z0 + CPU_SAMPLE_NZ, len(SIGMAS)),
        "mask_voxels": int(inside.sum()),
        "whole_mask_inserts": int(ref_whole.sum()),
        "whole_mask_sum_abs_dcount": int(np.abs(g_whole.astype(np.int64) - ref_whole.astype(np.int64)).sum()),
        "roi_inserts": int(ref_rois.sum()),
        "roi_sum_abs_dcount": int(np.abs(g_rois.astype(np.int64) - ref_rois.astype(np.int64)).sum()),
        "note": "GPU histograms vs DenseHistogram inserts of the CPU oracle's features, %d equalized edges per "
                "(scale, feature); bit-exact when both sums are 0" % N_EDGES})
    return par


def leg_hist(env, mask_kind="lung", n_rois=50, headline=False):
    import ctypes as C
    import numpy as np
    import synth
    torch, ctx, args = env.torch, env.ctx, env.args
    nx, ny, nz = DIMS
    n = nx * ny * nz
    units = n * len(SIGMAS)
    img, mask = synth_scan_torch(torch, env.dev, 100 + env.rank, mask_kind)
    edges = equalized_edges_from_scan(torch, ctx, img, mask, N_EDGES)
    mask_np = mask.cpu().numpy()
    mask_frac = float(mask_np.mean())
    rois = synth.random_rois(mask_np, n_rois, (41, 41, 41), seed=7) if n_rois > 0 else None
    counts = torch.zeros((1, len(SIGMAS) * 8, N_EDGES + 1), dtype=torch.int32, device=env.dev)
    counts_r = torch.zeros((max(n_rois, 1), len(SIGMAS) * 8, N_EDGES + 1), dtype=torch.int32, device=env.dev)
    torch.cuda.synchronize()
    res = {"config": {"workload": "MakeBag-style: ImageToEmphysemaFeaturesFilter features binned into DenseHistograms, no feature "
                                  "volume written; one 512x512x400 scan per GPU, sigma{0.6,1.2,2.4,4.8}, %d equalized edges per "
                                  "(scale, feature)" % N_EDGES, "mask": mask_kind, "mask_fill": mask_frac, "arith": args.arith,
                      "scaling": "weak"}}

    def run(name, step, roi_count):
        ms, launches, prof, _ = env.timed(step, args.steps, env.warmup)
        ms_per_step = ms / args.steps
        wd = ctx.last_work_dims()
        nwork = wd[0] * wd[1] * wd[2]
        table = kernel_table(env, prof, ALGO_BYTES_HIST, n, ms, "hist_%s%s" % (mask_kind, "_rois" if roi_count else ""))
        for k in table:       # every kernel of a histogram-only call runs on the crop
            table[k]["frac_of_bytes_moved"] = table[k]["frac"] * nwork / n
        pipe_b = sum(ALGO_BYTES_HIST.values())
        gbs = pipe_b * units / (ms_per_step * 1e-3) / 1e9
        res[name] = {"value": env.world * units / (ms_per_step * 1e-3) / 1e9, "unit": "Gvoxel/s", "ms_per_step": ms_per_step,
                     "steps": args.steps, "gpu_launches": launches, "rois": roi_count,
                     "work_dims": list(wd), "work_fraction_of_volume": nwork / n,
                     "roofline": {"algo_bytes_per_voxel_scale": pipe_b,
                                  "full_volume_equivalent_frac": gbs / env.peak,
                                  "frac_of_bytes_moved": gbs * nwork / n / env.peak,
                                  "peak": env.peak, "unit": "GB/s", "kernels": table,
                                  "note": "full_volume_equivalent = the work the reference does (whole volume) over this time: a "
                                          "work-equivalent rate, not an HBM fraction; frac_of_bytes_moved counts only the crop of "
                                          "the mask's box the kernels really process"}}

    run("whole_mask", lambda: ctx.emphysema_histograms_dev(img.data_ptr(), mask.data_ptr(), counts.data_ptr(), DIMS,
                                                           SIGMAS, edges, None), 0)
    if n_rois > 0:
        run("rois", lambda: ctx.emphysema_histograms_dev(img.data_ptr(), mask.data_ptr(), counts_r.data_ptr(), DIMS,
                                                         SIGMAS, edges, rois), n_rois)
    # invariant at full size: every row of the whole-mask histogram holds every in-mask voxel once
    row_sums = counts[0].to(torch.int64).sum(1)
    res["whole_mask"]["row_sums_equal_mask_voxels"] = bool((row_sums == int(mask_np.sum())).all().item())
    dump_output(env, "hist_edges", edges)
    dump_output(env, "hist_whole_mask_counts", counts)
    if n_rois > 0:
        dump_output(env, "hist_rois_counts", counts_r[:DUMP_ROIS])

    if not args.no_e2e:
        h_img = torch.empty((nz, ny, nx), dtype=torch.float32, pin_memory=True).copy_(img)
        h_mask = torch.empty((nz, ny, nx), dtype=torch.uint8, pin_memory=True).copy_(mask)
        h_counts = np.zeros((1, len(SIGMAS) * 8, N_EDGES + 1), np.uint32)
        dims_c, sp_c = (C.c_int * 3)(*DIMS), (C.c_double * 3)(1, 1, 1)
        sig_c = (C.c_double * len(SIGMAS))(*SIGMAS)

        def e2e_step():
            ctx._check(ctx.L.ife_cuda_emphysema_histograms(ctx.h, C.c_void_p(h_img.data_ptr()), C.c_void_p(h_mask.data_ptr()),
                                                           dims_c, sp_c, sig_c, len(SIGMAS), edges.ctypes.data_as(C.c_void_p),
                                                           N_EDGES, None, 0, h_counts.ctypes.data_as(C.c_void_p), env.ife.MEM_HOST))
        e_steps = args.steps
        for _ in range(2):
            e2e_step()
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            e2e_step()
        torch.cuda.synchronize()
        dt = env.max_over_ranks((time.perf_counter() - t0) / e_steps)
        e2e = {"value": env.world * units / dt / 1e9, "unit": "Gvoxel/s", "ms_per_step": dt * 1e3, "steps": e_steps,
               "h2d_bytes_per_step": int(h_img.numel() * 4 + h_mask.numel()), "d2h_bytes_per_step": int(h_counts.nbytes),
               "api": "ife_cuda_emphysema_histograms(..., IFE_MEM_HOST) with pinned host buffers"}
        # BASELINE.json configs[4] on this GPU: a batch of host-resident scans through
        # ife_cuda_emphysema_histograms_batch (upload of scan i+1 behind the kernels of scan i)
        nb = 8                               # configs[4]: 64 scans over 8 GPUs = 8 scans per GPU
        imgs, masks = [h_img.numpy()] * nb, [h_mask.numpy()] * nb     # the same pinned scan nb times: identical traffic
        ctx.emphysema_histograms_batch(imgs, masks, SIGMAS, edges, None)
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):       # one step = one call of nb scans
            ctx.emphysema_histograms_batch(imgs, masks, SIGMAS, edges, None)
        dtb = env.max_over_ranks((time.perf_counter() - t0) / (nb * args.steps))
        e2e["batch"] = {"value": env.world * units / dtb / 1e9, "unit": "Gvoxel/s", "ms_per_scan": dtb * 1e3,
                        "scans_per_call": nb, "steps": args.steps, "api": "ife_cuda_emphysema_histograms_batch (host scans, uploads overlapped)"}
        # the same batch with the scans as int16 on the host (CT's type on disk; option
        # "host_image_i16": 2 bytes per voxel up, widened on the device) -- the synthetic scan is
        # rounded to integers for this sub-leg, so its histograms are those of the rounded scan
        h_i16 = torch.empty((nz, ny, nx), dtype=torch.int16, pin_memory=True).copy_(img.round().to(torch.int16))
        ctx.set_option("host_image_i16", 1)
        try:
            imgs16 = [h_i16.numpy()] * nb
            ctx.emphysema_histograms_batch(imgs16, masks, SIGMAS, edges, None, _raw_image=True)
            env.barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                ctx.emphysema_histograms_batch(imgs16, masks, SIGMAS, edges, None, _raw_image=True)
            dt16 = env.max_over_ranks((time.perf_counter() - t0) / (nb * args.steps))
        finally:
            ctx.set_option("host_image_i16", 0)
        e2e["batch_int16_upload"] = {"value": env.world * units / dt16 / 1e9, "unit": "Gvoxel/s", "ms_per_scan": dt16 * 1e3,
                                     "scans_per_call": nb, "steps": args.steps, "h2d_bytes_per_scan": int(h_i16.numel() * 2 + h_mask.numel()),
                                     "api": "ife_cuda_emphysema_histograms_batch, option host_image_i16"}
        res["e2e"] = e2e
        del h_img, h_mask, h_i16
    del img, mask, counts, counts_r
    torch.cuda.empty_cache()
    if env.rank == 0 and env.world == 1 and not args.no_cpu_baseline:
        res["parity"] = hist_parity_vs_oracle(env)
    return res


# ------------------------------------------------------------------------------------------
# slab leg: one 1024^3 volume in z-slabs (configs[3]); NCCL halo exchange + histogram all-reduce
# ------------------------------------------------------------------------------------------
def slab_parity(torch, a, b):
    """a (slab path), b (single-GPU entry point): (8, nz, ny, nx) device tensors of the same planes."""
    n_diff = frac_bad = order_mis = 0
    max_rel = 0.0
    nzp = a.shape[1]
    for z in range(0, nzp, 8):
        pa, pb = a[:, z:z + 8], b[:, z:z + 8]
        same = (pa == pb) | (torch.isnan(pa) & torch.isnan(pb))
        n_diff += int((~same).sum().item())
        la, lb = pa[2:5].double(), pb[2:5].double()
        scale = lb.abs().amax(0)
        err = (la - lb).abs().amax(0)
        rel = torch.where(scale > 0, err / torch.where(scale > 0, scale, torch.ones_like(scale)), (err > 0).double() * 1e30)
        frac_bad += int((rel > 1e-4).sum().item())
        max_rel = max(max_rel, float(rel.max().item()))
        oa = (la[0].abs() >= la[1].abs()) & (la[1].abs() >= la[2].abs())
        ob = (lb[0].abs() >= lb[1].abs()) & (lb[1].abs() >= lb[2].abs())
        order_mis += int((oa != ob).sum().item())
    return n_diff, frac_bad, order_mis, max_rel


def leg_slab(env):
    import numpy as np
    torch, ctx, args, ife = env.torch, env.ctx, env.args, env.ife
    world, rank, dev = env.world, env.rank, env.dev
    size = args.slab_size
    gd = (size, size, size)
    plane = size * size
    z0, z1 = ife.slab_range(size, world, rank)
    nzo = z1 - z0
    n_own = nzo * plane
    steps = args.slab_steps or args.steps
    # every rank builds the whole volume: its own planes feed the slab path, all of them the
    # single-GPU reference of the parity block
    full = synth_volume_torch(torch, dev, 4, (size, size, size), z_range=(0, size))
    full_mask = torch.ones((size, size, size), dtype=torch.uint8, device=dev)
    img = full[z0:z1]
    mask = full_mask[z0:z1]
    # histogram edges: equalized on the first 64 planes (set-up)
    sub = min(64, size)
    edges = equalized_edges_from_scan(torch, ctx, full[:sub].contiguous(), full_mask[:sub].contiguous(), N_EDGES,
                                      dims=(size, size, sub))
    if world > 1:   # one set of edges for every rank (MakeBag reads them from one file): rank 0's
        box = [edges if rank == 0 else None]
        env.dist.broadcast_object_list(box, src=0)
        edges = box[0]
    rows, nb = len(SIGMAS) * 8, N_EDGES + 1
    per_scale = 8 * n_own * 4 * len(SIGMAS) > 60e9    # one scale's outputs at a time when all four would not fit
    out = torch.empty(((1 if per_scale else len(SIGMAS)), 8, nzo, size, size), dtype=torch.float32, device=dev)
    counts = torch.zeros((rows, nb), dtype=torch.int32, device=dev)
    if world > 1:
        uid = [ctx.comm_unique_id() if rank == 0 else None]
        env.dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], world, rank)
    torch.cuda.synchronize()

    def run_once(halo_factor=0.0):
        if per_scale:
            for si, s in enumerate(SIGMAS):
                ctx.slab_emphysema_features_dev(img.data_ptr(), mask.data_ptr(), out.data_ptr(), gd, [s],
                                                edges=edges[8 * si:8 * si + 8], counts_ptr=counts[8 * si:].data_ptr(),
                                                halo_factor=halo_factor)
        else:
            ctx.slab_emphysema_features_dev(img.data_ptr(), mask.data_ptr(), out.data_ptr(), gd, SIGMAS,
                                            edges=edges, counts_ptr=counts.data_ptr(), halo_factor=halo_factor)

    ms, launches, prof, clocks = env.timed(run_once, steps, env.warmup, clocks=True)
    dump_feature_sample(env, "slab_features", out)        # before the parity block reuses `out`
    dump_output(env, "slab_edges", edges)
    dump_output(env, "slab_counts", counts)
    ms_per_step = ms / steps
    units = size ** 3 * len(SIGMAS)
    value = units / (ms_per_step * 1e-3) / 1e9
    exch_ms = env.max_over_ranks(prof.get("exchange_wait", (0.0, 0))[0] / steps)
    # bytes this rank receives per step (image 4 B + mask 1 B per halo voxel); one exchange per call
    def recv_planes(H):
        return min(H, z0) + min(H, size - z1)
    if world == 1:
        recv = 0
    elif per_scale:
        recv = sum(recv_planes(ife.slab_halo(s, 1.0, args.halo_factor)) for s in SIGMAS) * plane * 5
    else:
        recv = recv_planes(ife.slab_halo(max(SIGMAS), 1.0, args.halo_factor)) * plane * 5
    exchanged = env.sum_over_ranks(recv)
    pipe_b = 78
    res = {"metric": METRIC.replace("512^2x400 CT", "%d^3 volume, z-slabs" % size), "value": value, "unit": "Gvoxel/s",
           "n_gpus": world, "steps": steps, "warmup": env.warmup, "ms_per_step": ms_per_step, "scaling": "strong",
           "config": {"workload": "one %d^3 float volume cut into %d z-slabs through ife_cuda_slab_emphysema_features, "
                                  "sigma{0.6,1.2,2.4,4.8}, 8 masked feature volumes per scale AND %d-edge histograms "
                                  "(ncclSend/ncclRecv halo exchange + ncclAllReduce of the counts)" % (size, world, N_EDGES),
                      "mask": "ones", "arith": args.arith, "halo_factor": args.halo_factor,
                      "halo_planes_per_side_largest_scale": ife.slab_halo(max(SIGMAS), 1.0, args.halo_factor),
                      "outputs": "one scale per call (4 exchanges per step)" if per_scale else "all scales in one call (1 exchange per step)"},
           "exchanged_bytes_per_step": int(exchanged), "exchange_exposed_ms_per_step": exch_ms,
           "allreduce_counters": rows * nb, "gpu_launches": launches, "clocks": clocks,
           "roofline": {"bound": "hbm", "kernel": "pipeline", "achieved": pipe_b * units / (ms_per_step * 1e-3) / 1e9 / world,
                        "peak": env.peak, "unit": "GB/s", "frac": pipe_b * units / (ms_per_step * 1e-3) / 1e9 / world / env.peak,
                        "note": "per-GPU algorithmic bytes (78 B/voxel-scale) over the step time"}}

    # ---- parity against the single-GPU entry point on the whole volume (every rank, own planes) ----
    if not args.no_slab_parity:
        ref = torch.empty((1, 8, size, size, size), dtype=torch.float32, device=dev)
        ref_counts = torch.zeros((1, rows, nb), dtype=torch.int32, device=dev)
        ctx.emphysema_histograms_dev(full.data_ptr(), full_mask.data_ptr(), ref_counts.data_ptr(), gd, SIGMAS, edges, None)
        torch.cuda.synchronize()
        factors = sorted(set([8.0, 10.0, args.halo_factor])) if world > 1 else [args.halo_factor]
        sweep = {}
        one = out
        for f in factors:
            tot = {"values_differing": 0, "voxels_eig_err_gt_1e-4": 0, "ordering_mismatches": 0, "eig_max_rel_err": 0.0,
                   "hist_sum_abs_dcount": 0}
            cnt = torch.zeros((rows, nb), dtype=torch.int32, device=dev)
            for si, s in enumerate(SIGMAS):
                ctx.emphysema_features_dev(full.data_ptr(), full_mask.data_ptr(), ref.data_ptr(), gd, [s])
                # all four scales in the call so that the halo is the one the timed path uses; keep scale si
                if per_scale:
                    ctx.slab_emphysema_features_dev(img.data_ptr(), mask.data_ptr(), one.data_ptr(), gd, [s],
                                                    edges=edges[8 * si:8 * si + 8], counts_ptr=cnt[8 * si:].data_ptr(), halo_factor=f)
                    got = one[0]
                else:
                    if si == 0:
                        ctx.slab_emphysema_features_dev(img.data_ptr(), mask.data_ptr(), out.data_ptr(), gd, SIGMAS,
                                                        edges=edges, counts_ptr=cnt.data_ptr(), halo_factor=f)
                    got = out[si]
                torch.cuda.synchronize()
                nd, nbad, nord, mrel = slab_parity(torch, got, ref[0, :, z0:z1])
                tot["values_differing"] += nd
                tot["voxels_eig_err_gt_1e-4"] += nbad
                tot["ordering_mismatches"] += nord
                tot["eig_max_rel_err"] = max(tot["eig_max_rel_err"], mrel)
            tot["hist_sum_abs_dcount"] = int((cnt.to(torch.int64) - ref_counts[0].to(torch.int64)).abs().sum().item())
            for k in ("values_differing", "voxels_eig_err_gt_1e-4", "ordering_mismatches"):
                tot[k] = int(env.sum_over_ranks(tot[k]))
            tot["eig_max_rel_err"] = env.max_over_ranks(tot["eig_max_rel_err"])
            tot["frac_voxels_eig_err_gt_1e-4"] = tot["voxels_eig_err_gt_1e-4"] / float(units)
            tot["halo_planes_per_side_largest_scale"] = ife.slab_halo(max(SIGMAS), 1.0, f)
            sweep["halo_factor_%g" % f] = tot
        res["parity"] = dict(sweep["halo_factor_%g" % args.halo_factor])
        res["parity"]["voxel_scales_compared"] = int(units)
        res["parity"]["values_compared"] = int(units * 8)
        res["parity"]["hist_inserts"] = int(units * 8)
        res["parity"]["note"] = ("slab path on %d rank(s) vs ife_cuda_emphysema_features / _histograms on the whole %d^3 volume "
                                 "(every rank compares the planes it owns; sums over ranks)" % (world, size))
        res["parity_vs_halo_factor"] = sweep
        del ref, ref_counts
    del full, full_mask, out, counts
    torch.cuda.empty_cache()
    return res


def main():
    with QuietStdout() as out:
        _main(out)


def _main(out_stream):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="extract", choices=["extract", "hist", "slab"])
    ap.add_argument("--mask", default="ones", choices=["ones", "lung"])
    ap.add_argument("--arith", default="fma", choices=["fma", "plain"])
    ap.add_argument("--slab-size", type=int, default=1024)
    ap.add_argument("--slab-steps", type=int, default=None, help="slab leg: timed steps (default: --steps)")
    ap.add_argument("--halo-factor", type=float, default=12.0)
    ap.add_argument("--rois", type=int, default=50, help="hist leg: bin into N fixed-seed 41^3 ROIs (MakeBag) besides the whole mask")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-hist", action="store_true", help="skip the hist leg")
    ap.add_argument("--no-slab", action="store_true", help="skip the slab leg")
    ap.add_argument("--no-slab-parity", action="store_true")
    ap.add_argument("--no-box", action="store_true", help="A/B: smooth the whole volume even where the mask cannot see it")
    ap.add_argument("--overlap", action="store_true", help="option overlap_scales: features of scale s beside the passes of scale s+1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what each leg's last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or (args.slab_steps is not None and args.slab_steps < 1):
        ap.error("--steps and --slab-steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; --impl reference has none")
    if args.impl == "reference":
        if "--steps" not in " ".join(sys.argv):
            args.steps = 3                   # ~4 s of CPU work per step
        return run_reference(args, out_stream)

    env = Env(args)
    torch = env.torch
    base = {"metric": METRIC, "unit": "Gvoxel/s", "n_gpus": env.world, "steps": args.steps, "warmup": env.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 recursion / f32 stencil+solver", "data": "synthetic"}
    line = None
    if args.workload == "slab":            # focused run: the slab leg as the headline
        s = leg_slab(env)
        line = dict(base, **{k: s[k] for k in ("metric", "value", "ms_per_step", "steps", "scaling", "config", "roofline",
                                               "gpu_launches", "clocks")})
        line.update({"e2e": None, "cpu_baseline": None, "slab": s})
    elif args.workload == "hist":          # focused run: the hist leg as the headline
        h = leg_hist(env, args.mask, args.rois)
        key = "rois" if args.rois > 0 and "rois" in h else "whole_mask"
        line = dict(base, value=h[key]["value"], ms_per_step=h[key]["ms_per_step"], config=h["config"],
                    roofline=h[key]["roofline"], gpu_launches=h[key]["gpu_launches"], e2e=h.get("e2e"),
                    cpu_baseline=None, parity=h.get("parity"), hist=h, clocks=None)
    else:
        img, mask = synth_scan_torch(torch, env.dev, 100 + env.rank, args.mask)
        x = leg_extract(env, img, mask)
        cpu = parity = None
        if env.rank == 0 and env.world == 1 and not args.no_cpu_baseline:
            cpu, parity = cpu_baseline(env.ctx, args.arith)
        del img, mask
        torch.cuda.empty_cache()
        line = dict(base, value=x["value"], ms_per_step=x["ms_per_step"],
                    config={"workload": WORKLOAD, "mask": args.mask, "arith": args.arith,
                            "parallelism": "1 scan per GPU, no data-path collective",
                            "cpu_affinity": env.affinity,
                            "l2": "inputs (525 MB/scan) and every intermediate are larger than the 126 MB L2; no flush needed"},
                    roofline=x["roofline"], e2e=x["e2e"], cpu_baseline=cpu, parity=parity,
                    gpu_launches=x["launches"], clocks=x["clocks"], other_arith=x["other_arith"])
        if not args.no_hist:
            line["hist"] = leg_hist(env, "lung", args.rois)
        if not args.no_slab:
            line["slab"] = leg_slab(env)
    if env.rank == 0:
        out_stream.emit(json.dumps(line))
    env.ctx.close()
    if env.dist:
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()
