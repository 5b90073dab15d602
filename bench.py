#!/usr/bin/env python
"""bench.py -- headline benchmark of the HiPR-FISH spectral-segmentation front end on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path

Metric (BASELINE.json): neighbor2d Mpix/s at 2048^2 x 95 channels.  A step is one pass of the
hot path (channel sum -> /max -> edge pad -> 9x11 line profiles -> F1 epilogue, i.e.
syn/..._measurement.py:105-124 without the skimage denoise) over one synthetic 2048x2048x95
float32 field of view per GPU (BASELINE config 2; with N GPUs each rank has its own FOVs -- config
3's FOV sharding, no collective, weak scaling).  The per-cell mean-spectrum reduction
(syn/..._measurement.py:167-172) is timed in a second region and reported as cells/s.

value      : device-resident throughput, CUDA events around exactly K steps, max over ranks.
e2e        : the same pipeline through the C ABI's host-buffer entry point
             (hipr_neighbor2d_host): pinned host cube -> H2D -> kernels -> D2H score, every step.
roofline   : the dominant kernel (channel sum, K1), 384 B/pixel algorithmic (SURVEY.md 8d),
             its launches timed with CUDA events inside the timed region.
cpu_baseline: the compiled reference Cython (oracle/_ref) + the scripts' numpy blocks, one core,
             on a bounded crop of the same FOV.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "hiprfish-image-analysis_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

H = W = 2048
C = 95
BYTES_PER_PIXEL = 4 * C + 4          # SURVEY.md 8d: read the cube once, write the score map
METRIC = "neighbor2d Mpix/s at 2048x2048x95ch"
WORKLOAD = "c2: one synthetic 2048x2048x95 float32 FOV per GPU per step (FOV-sharded, BASELINE config 2/3)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pool", type=int, default=2, help="resident FOVs per GPU that the steps rotate over")
    ap.add_argument("--e2e-steps", type=int, default=0, help="host-buffer steps (0: min(steps, 10))")
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="side of the CPU crop (0: the whole 2048^2 FOV for the cpu_baseline leg; for --impl reference a "
                         "side chosen from a calibration pass so that the K timed steps take about --cpu-budget seconds)")
    ap.add_argument("--cpu-budget", type=float, default=90.0, help="target seconds of the --impl reference timed region")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the timings of the rows either side of the hot path")
    ap.add_argument("--streams", type=int, default=2,
                    help="CUDA streams consecutive (independent) FOVs alternate over; 2 lets FOV i+1's channel sum "
                         "run under FOV i's stencil")
    ap.add_argument("--path", default="pipeline", choices=["pipeline", "fused", "two-kernel"],
                    help="pipeline: hipr_neighbor2d, one C-ABI call per FOV = channel sum + fixed-point stencil "
                         "(default); fused: one launch per FOV (fused2d.cu); two-kernel: the same two kernels as "
                         "separate calls with the global range")
    ap.add_argument("--bands", type=int, default=0)
    ap.add_argument("--graph", action="store_true", help="replay each FOV's pipeline as a captured CUDA graph")
    ap.add_argument("--workload", default="fov", choices=["fov", "mosaic", "zstack"],
                    help="fov (default, the headline): one 2048^2 FOV per GPU per step; mosaic: BASELINE config 5, one "
                         "stitched mosaic split into row slabs across the ranks with an NCCL halo exchange")
    ap.add_argument("--mosaic-side", type=int, default=16384)
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="mosaic halo / range exchange: this library's kernels over NVLink peer memory, or NCCL send/recv + all-reduce")
    ap.add_argument("--zstack", default="1024x1024x64", help="X x Y x Z of the --workload zstack volume (BASELINE config 4)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--workload fov only: after the timed steps, write what the last timed step returned on rank 0 "
                         "(other ranks write nothing) to DIR: score.npy (2048x2048 float32 score map) and, except for "
                         "--path fused, channel_sum.npy (2048x2048 float64 channel sums) and channel_sum_max_min.npy "
                         "(their global max and min), so that two builds can be compared output for output (the "
                         "inputs are seeded: the same arguments give the same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "fov"):
        ap.error("--dump-outputs writes the headline workload's outputs: it needs --impl b200 --workload fov")
    return args


# ------------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py touches oracle/)
# ------------------------------------------------------------------------------------------------

def _lp2d():
    from oracle import load_ref, hipr_oracle
    ref = load_ref("neighbor2d")
    if ref is not None:
        return ref.line_profile_2d_v2, "reference"
    return hipr_oracle.line_profile_2d_v2, "port"


def cpu_single_core(cube_np):
    """The reference path on one core (it is single-threaded): returns seconds."""
    from oracle import hipr_oracle
    lp, kind = _lp2d()
    t0 = time.perf_counter()
    score = hipr_oracle.neighbor2d_score(cube_np, "F1", lp_func=lp)
    return time.perf_counter() - t0, kind, score


def parity_stats(got, want, rtol=1e-5, atol=5e-7):
    """Deviation of a float32 result from the float64 reference: the counts are what the gates in tests/ assert on
    windows, here over the whole array."""
    import numpy as np
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    err = np.abs(got - want)
    nz = want != 0
    return {"n": int(want.size), "max_abs": float(err.max()), "max_rel": float((err[nz] / np.abs(want[nz])).max()),
            "n_outside_rtol1e-5_atol0": int((err > rtol * np.abs(want)).sum()),
            "n_outside_gate": int((err > atol + rtol * np.abs(want)).sum()),
            "gate": "rtol %g, atol %g (the gate of tests/)" % (rtol, atol),
            "nan_mismatch": int((np.isnan(got) != np.isnan(want)).sum())}


_G = {}


def _band_sum(args):
    r0, r1 = args
    import numpy as np
    return np.sum(_G["cube"][r0:r1], axis=2)


def _band_score(args):
    from oracle import hipr_oracle
    padded_band, = args
    lp, _ = _lp2d()
    return hipr_oracle.epilogue_F1(lp(padded_band, 11, 9))


def reference_step(pool, cube_np, nproc):
    """One pass of the reference path over `cube_np` with `nproc` worker processes over row bands
    (the reference's own parallelism is `snakemake -j` over independent images; bands of one image
    with a 5-row halo compute exactly the same thing)."""
    import numpy as np
    Hs = cube_np.shape[0]
    edges = np.linspace(0, Hs, nproc + 1).astype(int)
    bands = [(int(a), int(b)) for a, b in zip(edges[:-1], edges[1:]) if b > a]
    sums = pool.map(_band_sum, bands)
    s = np.concatenate(sums, axis=0)
    s = s / np.max(s)
    padded = np.pad(s, 5, mode="edge").astype(np.float64)
    parts = pool.map(_band_score, [(padded[a:b + 10],) for a, b in bands])
    return np.concatenate(parts, axis=0)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import numpy as np
    import torch
    from hipr_b200 import synth
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[k] = "1"          # as syn/Snakefile:13-14
    cores = len(os.sched_getaffinity(0))
    _, kind = _lp2d()
    ctx = mp.get_context("fork")
    side = args.cpu_sample
    if side <= 0:
        # bounded sample: calibrate on a 512^2 crop, then pick the crop side (multiple of 64, at most the
        # whole 2048^2 FOV) whose K timed steps fit --cpu-budget seconds
        cal = synth.make_fov(512, 512, C, fov_index=0)[0].numpy()
        _G["cube"] = cal
        nproc = max(1, min(cores, 512 // 32))
        with ctx.Pool(nproc) as pool:
            reference_step(pool, cal, nproc)
            t0 = time.perf_counter()
            reference_step(pool, cal, nproc)
            rate = 512 * 512 / (time.perf_counter() - t0)
        side = int((rate * args.cpu_budget / max(args.steps + max(args.warmup, 1), 1)) ** 0.5) // 64 * 64
        side = max(256, min(H, side))
    cube = synth.make_fov(side, side, C, fov_index=0)[0].numpy()
    _G["cube"] = cube
    nproc = max(1, min(cores, side // 32))
    with ctx.Pool(nproc) as pool:
        for _ in range(max(args.warmup, 1)):
            reference_step(pool, cube, nproc)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            reference_step(pool, cube, nproc)
        dt = time.perf_counter() - t0
    mpix_s = side * side * args.steps / dt / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": mpix_s, "unit": "Mpix/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "flavour": "F1", "patch_size": 11, "phi_range": 9},
        "cpu_baseline": {"value": mpix_s, "unit": "Mpix/s", "cores": nproc, "kind": kind,
                         "sample": "%dx%dx%d crop of FOV 0 per step, %d worker processes over row bands"
                                   % (side, side, C, nproc)},
        "e2e": {"value": mpix_s, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------

class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample(self):
        if self.nv is None:
            return
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for bit, name in self.REASONS.items():
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self._stop_evt.is_set():
            self.sample()
            time.sleep(0.001)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def bind_to_gpu_cpus(index):
    """Pins this process to the CPUs NVML reports as local to GPU `index` (its NUMA node), so that the pinned
    host buffers of the end-to-end leg are allocated next to the GPU's PCIe root port.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        allowed = os.sched_getaffinity(0)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        ideal = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1}
        cpus = ideal & allowed
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "%d of %d allowed cpus" % (len(cpus), len(allowed))
    except Exception as exc:      # NVML or the cpuset may not allow it: run unbound
        return "unbound (%s)" % type(exc).__name__
    return "unbound"


def measure_next_rows(cube, labels, with_cpu):
    """The rows either side of the hot path (SURVEY.md 8f), device-resident, each beside its CPU restatement
    timed on a bounded crop: registration paste + flat field + sum (K0), flat-field channel sum, NL-means
    denoise, the denoised chain, per-cell geometry, paint by label.  Extra information, not the headline."""
    import numpy as np
    import torch
    from hipr_b200 import ops

    def gpu_ms(fn, n=10):
        for _ in range(2):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    npix = cube.shape[0] * cube.shape[1]
    edges = (0, 32, 55, 75, 89, 95)
    stacks = [cube[:, :, a:b].contiguous() for a, b in zip(edges[:-1], edges[1:])]
    shifts = [(0, 0), (3, -2), (-4, 5), (1, 1), (-1, -7)]
    cal = torch.rand(cube.shape, device=cube.device) + 0.5
    s64 = ops.channel_sum(cube, None, normalize=True, dtype=torch.float64)
    L = int(ops.label_max(labels).item())
    lut = torch.rand((L + 1, 3), device=cube.device, dtype=torch.float64)
    out = {}
    t = gpu_ms(lambda: ops.register_stacks(stacks, shifts))
    out["register_stacks"] = {"ms": t, "gb_s": npix * 768 / t / 1e6, "bytes_per_px": 768}
    t = gpu_ms(lambda: ops.register_stacks(stacks, shifts, cal))
    out["register_stacks_flat_field"] = {"ms": t, "gb_s": npix * 1148 / t / 1e6, "bytes_per_px": 1148}
    t = gpu_ms(lambda: ops.channel_sum(cube, cal, normalize=False, dtype=torch.float64, return_max=True))
    out["channel_sum_flat_field"] = {"ms": t, "gb_s": npix * 768 / t / 1e6, "bytes_per_px": 768}
    t = gpu_ms(lambda: ops.denoise_nl_means(s64, h=0.02), n=5)
    out["denoise_nl_means"] = {"ms": t, "mpix_s": npix / t / 1e3}
    # the z-stack caller's denoise (bio-ana:454, h = 0.03) on a 128 x 132 x 54 volume: 12,167 shifts x 216-voxel windows
    vol3 = (0.5 + 0.05 * torch.rand((128, 132, 54), device=cube.device, dtype=torch.float64))
    t = gpu_ms(lambda: ops.denoise_nl_means(vol3, h=0.03), n=2)
    out["denoise_nl_means_3d"] = {"ms": t, "shape": [128, 132, 54], "mvox_s": vol3.numel() / t / 1e3,
                                  "g_voxel_shifts_s": vol3.numel() * 12167 / t / 1e6}
    del vol3
    t = gpu_ms(lambda: ops.neighbor2d_score(cube, "F1", denoise_h=0.02), n=5)
    out["chain_sum_denoise_score"] = {"ms": t, "mpix_s": npix / t / 1e3}
    host = ops.pinned_empty(tuple(cube.shape), np.float32)
    torch.from_numpy(host).copy_(cube.cpu())
    score_host = ops.pinned_empty(tuple(cube.shape[:2]), np.float32)
    ops.neighbor2d_score_host(host, "F1", out=score_host, denoise_h=0.02)
    t0 = time.perf_counter()
    for _ in range(3):
        ops.neighbor2d_score_host(host, "F1", out=score_host, denoise_h=0.02)
    out["e2e_chain_with_denoise"] = {"ms": 1e3 * (time.perf_counter() - t0) / 3, "mpix_s": npix / ((time.perf_counter() - t0) / 3) / 1e6,
                                     "api": "hipr_neighbor2d_host_denoise (pinned host cube -> score, lines 105-124 in full)"}
    # the same flow over a batch of FOVs: FOV i + 1 crosses PCIe while FOV i is denoised, scored and read back
    nb = 4
    ops.neighbor2d_score_host_batch([host] * 2, "F1", denoise_h=0.02, out=[score_host] * 2)
    t0 = time.perf_counter()
    ops.neighbor2d_score_host_batch([host] * nb, "F1", denoise_h=0.02, out=[score_host] * nb)
    tb = 1e3 * (time.perf_counter() - t0) / nb
    out["e2e_chain_with_denoise_batch"] = {"ms_per_fov": tb, "mpix_s": npix / tb / 1e3, "fovs": nb,
                                           "api": "hipr_neighbor2d_host_batch (pinned host cubes -> scores; denoise + stencil of FOV i under the upload of FOV i + 1)"}
    del host
    # a1, the strict drop-in: the literal (H, W, 9, 11) float64 gather of line_profile_2d_v2 (792 B written + 8 read per
    # pixel).  Device-resident against the HBM write roofline, and numpy -> numpy through hipr_line_profile_2d_host
    # (3.3 GB of output per 2048^2 image: the call is the PCIe time of the result)
    pad64 = torch.nn.functional.pad(s64[None, None], (5, 5, 5, 5), mode="replicate")[0, 0].contiguous()
    t = gpu_ms(lambda: ops.line_profile_2d(pad64, 11, 9), n=5)
    out["dropin_line_profile_2d_v2"] = {"ms": t, "gb_s": npix * 800 / t / 1e6, "bytes_per_px": 800}
    pad_np = pad64.cpu().numpy()
    del pad64
    try:                                        # 3.3 GB of page-locked memory: skipped, not fatal, where the host refuses it
        lp_host = ops.line_profile_2d_host(pad_np, 11, 9, pinned=True)
        t0 = time.perf_counter()
        for _ in range(2):
            ops.line_profile_2d_host(pad_np, 11, 9, out=lp_host)
        t = 1e3 * (time.perf_counter() - t0) / 2
        out["dropin_line_profile_2d_v2"].update({"host_ms_pinned_out": t, "host_gb_s": lp_host.nbytes / t / 1e6,
                                                 "api": "hipr_line_profile_2d_host (numpy float64 in, page-locked float64 out)"})
        del lp_host
    except (RuntimeError, MemoryError) as exc:
        out["dropin_line_profile_2d_v2"]["host_error"] = str(exc)[:200]
    if with_cpu:
        lp_page = np.empty((cube.shape[0], cube.shape[1], 9, 11), dtype=np.float64)
        lp_page.fill(0.0)                                      # fault the pages in outside the timed call
        t0 = time.perf_counter()
        ops.line_profile_2d_host(pad_np, 11, 9, out=lp_page)
        out["dropin_line_profile_2d_v2"]["host_ms_pageable_out"] = 1e3 * (time.perf_counter() - t0)
        del lp_page
    del pad_np
    score = ops.neighbor2d_pipeline(cube, "F1")[0]
    t = gpu_ms(lambda: ops.kmeans_threshold(score, 2), n=5)
    km = ops.kmeans_threshold(score, 2)
    out["kmeans_threshold_k2"] = {"ms": t, "n_iter": km.n_iter, "centers": [float(v) for v in km.cluster_centers_],
                                  "note": "KMeans(2, random_state=0) on the 2048^2 score map incl. labels + mask + result readback"}
    t = gpu_ms(lambda: ops.kmeans_threshold(score, 3), n=5)
    out["kmeans_threshold_k3"] = {"ms": t, "n_iter": ops.kmeans_threshold(score, 3).n_iter}
    t = gpu_ms(lambda: ops.cell_geometry(labels, L))
    out["cell_geometry"] = {"ms": t, "cells": L}
    t = gpu_ms(lambda: ops.paint_labels(labels, lut, L))
    out["paint_labels_rgb"] = {"ms": t, "gb_s": npix * (labels.element_size() + 24) / t / 1e6}
    if with_cpu:
        from oracle import hipr_oracle
        n = 512
        crop = [st[:n, :n].cpu().numpy() for st in stacks]
        t0 = time.perf_counter()
        hipr_oracle.register_stacks(crop, shifts, cal[:n, :n].cpu().numpy())
        out["register_stacks_flat_field"]["cpu_ms_scaled"] = 1e3 * (time.perf_counter() - t0) * npix / (n * n)
        m = 160
        t0 = time.perf_counter()
        hipr_oracle.denoise_nl_means_2d(s64[:m, :m].cpu().numpy(), h=0.02)
        out["denoise_nl_means"]["cpu_ms_scaled"] = 1e3 * (time.perf_counter() - t0) * npix / (m * m)
        out["denoise_nl_means"]["cpu_note"] = "numpy restatement of skimage's fast mode on a %dx%d crop, scaled by pixels" % (m, m)
        try:
            s_np = score.cpu().numpy()
            t0 = time.perf_counter()
            c_sk, l_sk, m_sk, it_sk, _ = hipr_oracle.kmeans1d_sklearn(s_np, 2)
            out["kmeans_threshold_k2"]["cpu_ms"] = 1e3 * (time.perf_counter() - t0)
            out["kmeans_threshold_k2"]["parity"] = {
                "oracle": "scikit-learn KMeans on the same float32 score map (whole FOV)",
                "max_abs_center_diff": float(np.max(np.abs(c_sk - km.cluster_centers_))), "n_iter_equal": it_sk == km.n_iter,
                "labels_differing": int((km.labels.cpu().numpy() != l_sk).sum()),
                "mask_differing": int((km.mask.cpu().numpy() != m_sk).sum())}
        except ImportError:
            pass
        lab_np = labels[:n, :n].cpu().numpy()
        t0 = time.perf_counter()
        hipr_oracle.cell_geometry(lab_np)
        out["cell_geometry"]["cpu_ms_scaled"] = 1e3 * (time.perf_counter() - t0) * npix / (n * n)
    return out


# ------------------------------------------------------------------------------------------------
# the CUDA arm
# ------------------------------------------------------------------------------------------------

def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import hipr_b200
    from hipr_b200 import ops, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_cpus(local)       # before any pinned allocation: host buffers land on the GPU's NUMA node
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lib = hipr_b200.lib()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback")

    # resident inputs: `pool` FOVs per GPU, FOV index = rank + world * i (config 3's sharding)
    pool = [synth.make_fov(H, W, C, fov_index=rank + world * i, device=dev) for i in range(args.pool)]
    cubes = [p[0] for p in pool]
    labels = [p[1] for p in pool]
    max_labels = [int(ops.label_max(l).item()) for l in labels]
    npix = H * W

    streams = [torch.cuda.Stream(device=dev) for _ in range(args.streams)] if args.streams > 1 else None

    def step(i, ev=None):
        """One FOV through the timed path: (score, float64 channel sums, MaxKey of the sums); the fused path returns
        the score alone, (score, None, None)."""
        cube = cubes[i % len(cubes)]
        st = streams[i % len(streams)] if streams else torch.cuda.current_stream()
        with torch.cuda.stream(st):
            if args.path == "pipeline":
                return ops.neighbor2d_pipeline(cube, "F1", bands=args.bands)
            if args.path == "fused":
                if ev:
                    ev[0].record(st)
                out = ops.neighbor2d_fused(cube, "F1")
                if ev:
                    ev[1].record(st)
                return out, None, None
            if ev:
                ev[0].record(st)
            s, mk = ops.channel_sum(cube, None, normalize=False, dtype=torch.float64, return_max=True)
            if ev:
                ev[1].record(st)
            out = ops.lne2d_fixed(s, "F1", 11, 9, padded=False, range_keys=mk)
        return out, s, mk

    def fork():
        if streams:
            for st in streams:
                st.wait_stream(torch.cuda.current_stream())

    def join():
        if streams:
            for st in streams:
                torch.cuda.current_stream().wait_stream(st)

    # ---- headline timed region ------------------------------------------------------------------
    for i in range(max(args.warmup, 3)):
        step(i)
    if args.graph:
        # one captured graph per resident FOV: the banded pipeline's ~20 stream operations become
        # a single launch (the pipeline forks to a side stream and joins, which capture follows)
        torch.cuda.synchronize()
        graphs, graph_out = [], []
        for j in range(len(cubes)):
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                graph_out.append(step(j))
            graphs.append(gr)
        eager_step = step

        def step(i, ev=None):          # noqa: F811
            if ev:
                ev[0].record()
            graphs[i % len(graphs)].replay()
            if ev:
                ev[1].record()
            return graph_out[i % len(graphs)]
        for i in range(3):
            step(i)
    # hold the clocks up: ~0.25 s more of the same work before the timed region (untimed)
    t_end = time.perf_counter() + 0.25
    while time.perf_counter() < t_end:
        step(0)
        torch.cuda.synchronize()
    k1_events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    barrier()
    launches0 = lib.hipr_launch_count()
    sampler.start()
    e0.record()
    fork()
    for i in range(args.steps):
        last = step(i, k1_events[i])
    join()
    e1.record()
    barrier()
    clocks = sampler.stop()
    launches = lib.hipr_launch_count() - launches0
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        score, s, mk = last
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "score.npy"), score.cpu().numpy().astype(np.float32))
        if s is not None:
            np.save(os.path.join(args.dump_outputs, "channel_sum.npy"), s.cpu().numpy().astype(np.float64))
            np.save(os.path.join(args.dump_outputs, "channel_sum_max_min.npy"),
                    torch.cat(mk.values()).cpu().numpy().astype(np.float64))
    del last

    # ---- roofline region: the dominant kernel (channel sum) launched alone, K times ---------------
    # (inside the headline region its launches share the SMs with the other stream's stencil, so a
    # per-launch duration taken there would include that overlap)
    def k1_step(i):
        return ops.channel_sum(cubes[i % len(cubes)], None, normalize=False, dtype=torch.float64, return_max=True)

    for i in range(3):
        k1_step(i)
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    r0.record()
    for i in range(args.steps):
        k1_step(i)
    r1.record()
    barrier()
    k1_ms = r0.elapsed_time(r1) / args.steps
    if args.path == "fused":
        k1_ms = sum(a.elapsed_time(b) for a, b in k1_events) / args.steps

    # ---- per-cell spectra region ----------------------------------------------------------------
    # reset + accumulate + finalize (compaction of the present labels, means, row-max normalisation) per step, straight
    # through the C ABI with pre-bound arguments; on the synthetic FOV (25 % foreground) and on a dense label image
    # (biofilm-like: 94 % foreground, 16 x 16-pixel cells)
    vp = ctypes.c_void_p

    def cell_region(cube_t, labels_t, steps_n):
        mlab = int(ops.label_max(labels_t).item())
        sums = torch.empty((mlab + 1, C), dtype=torch.float64, device=dev)
        cnts = torch.empty(mlab + 1, dtype=torch.int32, device=dev)
        n_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        lab_o = torch.empty(mlab, dtype=torch.int64, device=dev)
        area_o = torch.empty(mlab, dtype=torch.int64, device=dev)
        avg_o = torch.empty((mlab, C), dtype=torch.float64, device=dev)
        norm_o = torch.empty((mlab, C), dtype=torch.float64, device=dev)
        a = (vp(cube_t.data_ptr()), vp(labels_t.data_ptr()), labels_t.element_size(), npix, W, C, mlab, vp(sums.data_ptr()),
             vp(cnts.data_ptr()))
        fin = (vp(sums.data_ptr()), vp(cnts.data_ptr()), mlab, C, vp(n_dev.data_ptr()), vp(lab_o.data_ptr()),
               vp(area_o.data_ptr()), vp(avg_o.data_ptr()), vp(norm_o.data_ptr()))

        def one():
            st = vp(torch.cuda.current_stream().cuda_stream)
            lib.hipr_cell_spectra_reset(a[7], a[8], mlab, C, st)
            rc = lib.hipr_cell_spectra_accumulate(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], None, st)
            rc = rc or lib.hipr_cell_spectra_finalize(*fin, st)
            if rc:
                raise RuntimeError("hipr_cell_spectra_*: %d" % rc)

        def acc_only():
            st = vp(torch.cuda.current_stream().cuda_stream)
            lib.hipr_cell_spectra_reset(a[7], a[8], mlab, C, st)
            lib.hipr_cell_spectra_accumulate(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], None, st)

        out = []
        for fn in (one, acc_only):
            for _ in range(3):
                fn()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            c0.record()
            for _ in range(steps_n):
                fn()
            c1.record()
            barrier()
            out.append(c0.elapsed_time(c1) / steps_n)
        fgf = float((labels_t > 0).float().mean().item())
        return out[0], out[1], int(n_dev.item()), fgf

    cell_ms_step, cell_acc_ms, n_cells0, fg_frac = cell_region(cubes[0], labels[0], args.steps)
    cell_ms = cell_ms_step * args.steps
    cells_per_step = n_cells0
    yy = torch.arange(H, device=dev)[:, None]
    xx = torch.arange(W, device=dev)[None, :]
    dense = ((yy // 16) * (W // 16) + (xx // 16) + 1).to(torch.int32)
    dense = torch.where(((yy % 16) == 0) & ((xx % 4) == 0), torch.zeros_like(dense), dense).contiguous()   # thin background seams
    dense_ms, dense_acc_ms, dense_cells, dense_fg = cell_region(cubes[0], dense, min(args.steps, 50))
    del dense

    # ---- end to end through the host-buffer C ABI -----------------------------------------------
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    host = ops.pinned_empty((H, W, C), np.float32)
    torch.from_numpy(host).copy_(cubes[0].cpu())
    score_host = ops.pinned_empty((H, W), np.float32)
    for _ in range(2):
        ops.neighbor2d_score_host(host, "F1", out=score_host)
    barrier()
    e2e_dev_ms = 0.0
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ops.neighbor2d_score_host(host, "F1", out=score_host)
        e2e_dev_ms += lib.hipr_host_last_elapsed_ms()
    torch.cuda.synchronize()
    e2e_wall_ms = 1e3 * (time.perf_counter() - t0)
    score_check = float(score_host.mean())
    host_api_score = score_host.copy()
    # per-cell spectra end to end: pinned host cube + host label image -> cell table on the host
    labels_host = labels[0].cpu().numpy()
    ops.cell_spectra_host(host, labels_host)
    barrier()
    t0 = time.perf_counter()
    cell_e2e_steps = 3
    for _ in range(cell_e2e_steps):
        cell_tab = ops.cell_spectra_host(host, labels_host)
    cell_e2e_ms = 1e3 * (time.perf_counter() - t0) / cell_e2e_steps
    cell_e2e_n = int(cell_tab[0].size)
    # the scripts' real flow (syn/..._measurement.py:161-173): score map, (watershed on the host), per-cell spectra of the
    # SAME cube: one upload through the handle API instead of two
    with ops.Fov(host) as fov:
        fov.score("F1", out=score_host)
        fov.cell_spectra(labels_host)
    barrier()
    flow_steps = 5
    t0 = time.perf_counter()
    for _ in range(flow_steps):
        with ops.Fov(host) as fov:
            fov.score("F1", out=score_host)
            flow_tab = fov.cell_spectra(labels_host)
    flow_ms = 1e3 * (time.perf_counter() - t0) / flow_steps
    flow_equal = bool(np.array_equal(score_host, host_api_score) and np.array_equal(flow_tab[0], cell_tab[0])
                      and np.array_equal(flow_tab[1], cell_tab[1]) and np.allclose(flow_tab[2], cell_tab[2], rtol=1e-12, atol=0))
    # plain host-to-device ceiling: the same number of bytes from page-locked memory with one cudaMemcpyAsync, every
    # rank at once (what the box's PCIe / host memory system delivers to N GPUs simultaneously)
    pin = torch.empty(H * W * C, dtype=torch.float32).pin_memory()
    dst = torch.empty(H * W * C, dtype=torch.float32, device=dev)
    dst.copy_(pin, non_blocking=True)
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    h0.record()
    for _ in range(5):
        dst.copy_(pin, non_blocking=True)
    h1.record()
    barrier()
    h2d_ms = h0.elapsed_time(h1) / 5
    del pin, dst
    # the same FOV as the uint16 counts a detector delivers (value = count / 65535 in float32, bioformats' rescale)
    raw = ops.pinned_empty((H, W, C), np.uint16)
    cmax = float(cubes[0].max())
    torch.from_numpy(raw.view(np.int16)).copy_((cubes[0] * (0.9 * 65535.0 / cmax)).round().to(torch.int32).cpu().to(torch.int16))
    for _ in range(2):
        ops.neighbor2d_score_host_raw(raw, 65535.0, "F1", out=score_host)
    barrier()
    raw_dev_ms = 0.0
    for _ in range(e2e_steps):
        ops.neighbor2d_score_host_raw(raw, 65535.0, "F1", out=score_host)
        raw_dev_ms += lib.hipr_host_last_elapsed_ms()
    torch.cuda.synchronize()
    del raw

    # ---- reduce over ranks (max time) -----------------------------------------------------------
    t = torch.tensor([ms, cell_ms, e2e_dev_ms, e2e_wall_ms, k1_ms, raw_dev_ms, cell_e2e_ms, flow_ms, h2d_ms, cell_acc_ms, dense_ms,
                      dense_acc_ms], dtype=torch.float64, device=dev)
    cnt = torch.tensor([launches, cells_per_step], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    ms, cell_ms, e2e_dev_ms, e2e_wall_ms, k1_ms, raw_dev_ms, cell_e2e_ms, flow_ms, h2d_ms, cell_acc_ms, dense_ms, dense_acc_ms = \
        [float(x) for x in t.tolist()]
    launches, cells_all = int(cnt[0].item()), float(cnt[1].item())

    # ---- the other configurations, recorded in the same line -----------------------------------
    # c5 (needs >= 2 ranks): the split mosaic with this library's peer-memory exchange; c4 (1 rank): the z-stack
    zstack = mosaic = None
    if not args.no_extras:
        if world > 1:
            mosaic = measure_mosaic(args, dev, rank, world, 2048, args.mosaic_side, min(args.steps, 20), hbm_peak=hbm_peak)
        else:
            zstack = measure_zstack(args, dev, rank, world, min(args.steps, 10), hbm_peak, with_cpu=not args.no_cpu)
    if rank == 0:
        value = world * npix * args.steps / (ms * 1e-3) / 1e6
        k1_gbs = npix * BYTES_PER_PIXEL / (k1_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:
            import hashlib
            tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
            traffic = tj["chansum_bytes_per_launch"]
            sha = hashlib.sha256(open(os.path.join(PKG, "csrc", "chansum.cu"), "rb").read()).hexdigest()
            traffic_src = {"capture": tj.get("source"), "round": tj.get("round"),
                           "how": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this kernel "
                                  "(profiles/), not re-measured in this run",
                           "kernel_source_unchanged_since_capture": tj.get("chansum_cu_sha256") == sha}
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "flavour": "F1", "patch_size": 11, "phi_range": 9},
            "impl_detail": {"path": args.path, "streams": args.streams,
                            "l2": "inputs larger than L2 (1.59 GB cube per step, %d FOVs in rotation)" % len(cubes),
                            "arithmetic": "float64 channel sums, 31-bit fixed-point stencil, float32 score"},
            "pipeline_frac_of_hbm_peak": value / world * 1e6 * BYTES_PER_PIXEL / 1e9 / hbm_peak,
            "roofline": {"bound": "hbm", "kernel": "fused2d_kernel" if args.path == "fused" else "chansum_bulk_kernel",
                         "how": "this kernel launched alone K times between two CUDA events, same inputs",
                         "share_of_serial_step": k1_ms / (ms / args.steps) if args.streams == 1 else None,
                         "share_of_step": min(1.0, k1_ms / (ms / args.steps)),
                         "share_note": "two streams: the stencil of FOV i runs under the channel sum of FOV i+1, so the step is "
                                       "~one channel sum; ncu's serialised launch list and --streams 1 give the serial share "
                                       "(profiles/r02_summary.md)" if args.streams > 1 else "streams=1: serial step",
                         "achieved": k1_gbs, "peak": hbm_peak,
                         "unit": "GB/s", "frac": k1_gbs / hbm_peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": npix * BYTES_PER_PIXEL, "ms_per_launch": k1_ms},
            "e2e": {"value": world * npix * e2e_steps / (e2e_dev_ms * 1e-3) / 1e6, "unit": "Mpix/s",
                    "h2d_bytes_per_step": npix * C * 4, "d2h_bytes_per_step": npix * 4, "steps": e2e_steps,
                    "ms_per_step": e2e_dev_ms / e2e_steps, "wall_ms_per_step": e2e_wall_ms / e2e_steps,
                    "api": "hipr_neighbor2d_host (C ABI, pinned host buffers)", "score_mean": score_check,
                    "host_numa_binding": numa,
                    "h2d_ceiling": {"gb_s_per_gpu": npix * C * 4 / (h2d_ms * 1e-3) / 1e9, "ms": h2d_ms,
                                    "how": "plain cudaMemcpyAsync of the same %d bytes from page-locked memory, all %d ranks at once, "
                                           "max over ranks" % (npix * C * 4, world)},
                    "frac_of_h2d_ceiling": h2d_ms / (e2e_dev_ms / e2e_steps)},
            "e2e_flow": {"ms_per_fov": flow_ms, "mpix_per_s": world * npix / (flow_ms * 1e-3) / 1e6,
                         "api": "hipr_fov_upload -> hipr_fov_score -> hipr_fov_cell_spectra -> hipr_fov_release: ONE upload of the "
                                "cube for the score map and the per-cell spectra (wall clock, incl. device allocation)",
                         "two_uploads_ms": e2e_dev_ms / e2e_steps + cell_e2e_ms, "equals_separate_calls": flow_equal,
                         "h2d_bytes_per_fov": npix * C * 4 + npix * labels[0].element_size()},
            "e2e_raw_u16": {"value": world * npix * e2e_steps / (raw_dev_ms * 1e-3) / 1e6, "unit": "Mpix/s",
                            "h2d_bytes_per_step": npix * C * 2, "d2h_bytes_per_step": npix * 4,
                            "ms_per_step": raw_dev_ms / e2e_steps,
                            "api": "hipr_neighbor2d_host_raw: the FOV as the detector's uint16 counts, rescaled on the "
                                   "GPU exactly as bioformats does on the host (half the PCIe bytes, same score)"},
            "cell_spectra": {"cells_per_s": cells_all * args.steps / (cell_ms * 1e-3),
                             "mpix_per_s": world * npix * args.steps / (cell_ms * 1e-3) / 1e6,
                             "ms_per_step": cell_ms / args.steps, "cells_per_fov": cells_all / world,
                             "foreground_fraction": fg_frac,
                             "e2e": {"cells_per_s": world * cell_e2e_n / (cell_e2e_ms * 1e-3), "ms_per_step": cell_e2e_ms,
                                     "h2d_bytes_per_step": npix * C * 4 + npix * labels[0].element_size(),
                                     "api": "hipr_cell_spectra_host (pinned host cube + label image -> cell table, wall clock)"},
                             "timed": "reset + accumulate + finalize (compaction, means, row-max normalisation) per step",
                             "accumulate_ms": cell_acc_ms,
                             "fetched_bytes_per_step": int(npix * (fg_frac * 4 * C + labels[0].element_size())),
                             "fetched_gbs": npix * (fg_frac * 4 * C + labels[0].element_size()) / (cell_acc_ms * 1e-3) / 1e9,
                             "frac_of_hbm_peak_on_fetched_bytes": npix * (fg_frac * 4 * C + labels[0].element_size()) / (cell_acc_ms * 1e-3) / 1e9 / hbm_peak,
                             "note": "background pixels' channel vectors are never fetched; the roofline is taken on the "
                                     "bytes the kernel has to fetch (foreground pixels' vectors + the label image)",
                             "dense_labels": {"foreground_fraction": dense_fg, "cells": dense_cells, "ms_per_step": dense_ms,
                                              "accumulate_ms": dense_acc_ms,
                                              "fetched_gbs": npix * (dense_fg * 4 * C + 4) / (dense_acc_ms * 1e-3) / 1e9,
                                              "frac_of_hbm_peak_on_fetched_bytes": npix * (dense_fg * 4 * C + 4) / (dense_acc_ms * 1e-3) / 1e9 / hbm_peak,
                                              "cells_per_s": dense_cells / (dense_ms * 1e-3)}},
            "gpu_launches": launches, "clocks": clocks,
        }
        if world == 1 and not args.no_extras:
            try:
                line["next_rows"] = measure_next_rows(cubes[0], labels[0], not args.no_cpu)
            except Exception as exc:        # auxiliary measurements must never cost the headline line
                line["next_rows"] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:300])}
        if not args.no_cpu and world == 1:
            side = args.cpu_sample or H
            crop = cubes[0][:side, :side].cpu().numpy()
            for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
                os.environ[k] = "1"
            sec, kind, want = cpu_single_core(crop)
            if side == H:
                # the oracle just scored the step's whole FOV: compare, do not throw it away
                from oracle import hipr_oracle
                dev_score = ops.neighbor2d_pipeline(cubes[0], "F1")[0].cpu().numpy()
                par = {"score_device": parity_stats(dev_score, want), "score_host_api": parity_stats(host_api_score, want),
                       "device_equals_host_api_bitwise": bool(np.array_equal(dev_score, host_api_score)),
                       "reference": "oracle/_ref line_profile_2d_v2 + the scripts' numpy blocks in float64, whole 2048^2 FOV"
                                    if kind == "reference" else "oracle port, whole FOV"}
                wl, wa, wavg, wnorm = hipr_oracle.cell_spectra(labels_host, crop)
                gl, ga, gavg, gnorm = cell_tab
                same = bool(np.array_equal(gl, wl) and np.array_equal(ga, wa))
                par["cell_spectra"] = {"labels_and_areas_equal": same, "n_cells": int(wl.size),
                                       "max_rel_mean": float(np.max(np.abs(gavg - wavg) / np.abs(wavg))) if same else None,
                                       "max_rel_norm": float(np.max(np.abs(gnorm - wnorm) / np.maximum(np.abs(wnorm), 1e-300))) if same else None,
                                       "gate": "labels / pixel counts bit-exact, means rtol 1e-5"}
                line["parity"] = par
            line["cpu_baseline"] = {"value": side * side / sec / 1e6, "unit": "Mpix/s", "cores": 1, "kind": kind,
                                    "sample": "%dx%dx%d crop of the step's FOV, single process (the reference is "
                                              "single-threaded), %.1f s" % (side, side, C, sec),
                                    "host_cores_available": len(os.sched_getaffinity(0))}
        if zstack is not None:
            line["zstack"] = zstack
        if mosaic is not None:
            line["mosaic"] = mosaic
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_mosaic(args, dev, rank, world, rows, width, steps, exchanges=("p2p", "p2p_inorder", "nccl"), hbm_peak=6554.2):
    """BASELINE config 5 on the ranks of an initialised NCCL job: a stitched (rows * world) x width x 95 mosaic cut into
    row slabs, one per rank.  Per step: channel sum of the slab -> 5-row halo exchange of the sum image (+ max / min) ->
    fixed-point stencil on the extended slab; then per-cell spectra reduced to rank 0.  Exchange kinds:
      p2p          this library's push / wait kernels over NVLink peer memory, row-banded so that stencil and exchange
                   run under the channel sum (hipr_mosaic_p2p_score);
      p2p_inorder  the same kernels, sum -> exchange -> stencil in order (bit-identical to nccl);
      nccl         batch_isend_irecv + all_reduce.
    Returns the dict on rank 0 (None elsewhere)."""
    import torch
    import torch.distributed as dist
    from hipr_b200 import sharding, synth

    height = rows * world
    r0 = rank * rows
    labels_full, L = synth.make_labels(height, width, seed=4321, device=dev)
    labels = labels_full[r0:r0 + rows].contiguous()
    del labels_full
    cube = torch.empty((rows, width, C), dtype=torch.float32, device=dev)
    for a in range(0, rows, 256):        # generated in 256-row pieces to bound peak memory
        b = min(a + 256, rows)
        cube[a:b] = synth.make_cube(b - a, width, C, seed=1234 + r0 + a, device=dev, labels=labels[a:b])
    slab = sharding.MosaicSlab()
    p2p = sharding.P2PMosaicSlab(rows, width)
    bands = args.bands if args.bands else 16     # 16 k wide slabs: 8 bands -> 2.31 ms, 16 -> 2.23 ms (round 1)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    runners = {"p2p": lambda: p2p.score(cube, "F1", bands=bands), "p2p_inorder": lambda: p2p.score(cube, "F1"),
               "nccl": lambda: slab.score(cube, "F1")}
    out = {}
    for kind in exchanges:
        run = runners[kind]
        for _ in range(3):
            score = run()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            score = run()
        e1.record()
        barrier()
        p2p.check_peers()
        t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        chk = score.double().sum().reshape(1)
        nan = torch.isnan(score).sum().reshape(1).double()
        dist.all_reduce(chk)
        dist.all_reduce(nan)
        out[kind] = {"ms_per_step": float(t.item()), "score_checksum": float(chk.item()), "nan_pixels": int(nan.item())}
    for _ in range(2):
        slab.cell_spectra(cube, labels, L, root=0)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    c0.record()
    for _ in range(steps):
        cells = slab.cell_spectra(cube, labels, L, root=0)      # one table, on rank 0 (reduce, not all-reduce)
    c1.record()
    barrier()
    t = torch.tensor([c0.elapsed_time(c1) / steps], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    cms = float(t.item())
    p2p.close()
    del cube, labels
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    npix = height * width
    best = exchanges[0]
    ms = out[best]["ms_per_step"]
    res = {"workload": "c5: %dx%dx%d mosaic, %d row slabs of %d rows (the 16384^2 mosaic at 8 GPUs; the same slab per GPU "
                       "at smaller N)" % (height, width, C, world, rows),
           "flavour": "F1", "steps": steps, "exchange": best, "row_bands": bands,
           "ms_per_step": ms, "mpix_per_s": npix / (ms * 1e-3) / 1e6,
           "frac_of_hbm_peak_per_gpu": rows * width * BYTES_PER_PIXEL / (ms * 1e-3) / 1e9 / hbm_peak,
           "halo_bytes_per_neighbour": 5 * width * 8, "by_exchange": out,
           "cell_spectra": {"cells": int(cells[0].numel()), "ms_per_step": cms, "cells_per_s": int(cells[0].numel()) / (cms * 1e-3),
                            "reduce_to_rank0_bytes": (L + 1) * (C * 8 + 4)}}
    if "p2p_inorder" in out and "nccl" in out:
        res["checksum_equal_p2p_inorder_nccl"] = out["p2p_inorder"]["score_checksum"] == out["nccl"]["score_checksum"]
    return res


def run_mosaic(args):
    """--workload mosaic: config 5 alone (extra line, not the headline metric)."""
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world < 2:
        raise SystemExit("--workload mosaic needs torchrun with >= 2 ranks")
    dist.init_process_group("nccl", device_id=dev)
    side = args.mosaic_side
    kinds = ("p2p", "p2p_inorder", "nccl") if args.exchange == "p2p" else ("nccl",)
    res = measure_mosaic(args, dev, rank, world, side // world, side, args.steps, kinds)
    if rank == 0:
        print(json.dumps({"metric": "mosaic neighbor2d Mpix/s (row slabs + 5-row halo exchange over NVLink)",
                          "value": res["mpix_per_s"], "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
                          "ms_per_step": res["ms_per_step"], "scaling": "strong", "config": {"workload": res["workload"]},
                          "mosaic": res}), flush=True)
    dist.destroy_process_group()


def measure_zstack(args, dev, rank, world, steps, hbm_peak, with_cpu=True):
    """BASELINE config 4: one X x Y x Z x 95 z-stack through the 72-direction 3-D stencil, the
    `generate_3d_segmentation_memory_efficient` chain (bio/..._analysis.py:807-817): channel sum -> /max ->
    edge pad -> line_profile_memory_efficient_v2 -> mean * (1 - qcv) over the 72 directions.  With N ranks every
    rank has its own z-stack (independent volumes, no collective).  Returns the dict on rank 0."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import hipr_b200
    from hipr_b200 import ops, synth

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    X, Y, Z = [int(v) for v in args.zstack.lower().split("x")]
    n_stacks = 2 if args.streams > 1 else 1           # resident z-stacks the steps rotate over
    cubes = []
    for k in range(n_stacks):
        cube = torch.empty((X, Y, Z, C), dtype=torch.float32, device=dev)
        full = synth.make_volume_cube(X, 8, Z, C, seed=99 + rank + 1000 * k, device=dev)   # periodic in y with period 8 planes
        for y in range(0, Y, 8):                                                            # + fresh noise per slab
            n = min(8, Y - y)
            cube[:, y:y + n] = full[:, :n] + 0.01 * torch.rand((X, n, Z, 1), device=dev)
        del full
        cubes.append(cube)
    cube = cubes[0]
    nvox = X * Y * Z
    lib = hipr_b200.lib()
    zstreams = [torch.cuda.Stream(device=dev) for _ in range(2)] if n_stacks > 1 else None
    counter = [0]

    def step():
        # independent z-stacks alternate between two streams: the channel sum of stack i+1 (HBM-bound) runs beside the
        # stencil of stack i (ALU-bound)
        i = counter[0]
        counter[0] += 1
        if zstreams is None:
            return ops.neighbor3d_score(cube, "ME2")
        with torch.cuda.stream(zstreams[i % 2]):
            return ops.neighbor3d_score(cubes[i % n_stacks], "ME2")

    def fork():
        if zstreams:
            for st in zstreams:
                st.wait_stream(torch.cuda.current_stream())

    def join():
        if zstreams:
            for st in zstreams:
                torch.cuda.current_stream().wait_stream(st)

    def k1():
        return ops.channel_sum(cube, None, normalize=False, dtype=torch.float64, return_max=True)

    fork()
    for _ in range(4):
        score = step()
    join()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = lib.hipr_launch_count()
    e0.record()
    fork()
    for _ in range(steps):
        score = step()
    join()
    e1.record()
    barrier()
    launches = lib.hipr_launch_count() - l0
    ms = e0.elapsed_time(e1) / steps
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s64, mk = k1()
    barrier()
    r0.record()
    for _ in range(steps):
        k1()
    r1.record()
    barrier()
    k1_ms = r0.elapsed_time(r1) / steps
    # the stencil alone, on the resident sum volume
    ops.lne3d_fixed(s64, "ME2", maxkey=mk)
    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    q0.record()
    for _ in range(steps):
        ops.lne3d_fixed(s64, "ME2", maxkey=mk)
    q1.record()
    barrier()
    k4_ms = q0.elapsed_time(q1) / steps
    t = torch.tensor([ms, k1_ms, k4_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, k1_ms, k4_ms = [float(v) for v in t.tolist()]
    res = None
    if rank == 0:
        res = {"metric": "neighbor (3-D) Mvox/s at %dx%dx%dx95ch" % (X, Y, Z), "value": world * nvox / (ms * 1e-3) / 1e6,
               "unit": "Mvox/s", "n_gpus": world, "steps": steps, "warmup": 3, "ms_per_step": ms,
               "higher_is_better": True, "scaling": "weak", "dtype": "f32", "data": "synthetic",
               "config": {"workload": "c4: %dx%dx%dx95 float32 z-stack per GPU, (11, 9, 9) stencil, epilogue ME2" % (X, Y, Z)},
               "impl_detail": {"arithmetic": "float64 channel sums, 31-bit fixed-point stencil, float32 score",
                               "streams": 2 if zstreams else 1, "resident_stacks": n_stacks,
                               "l2": "inputs larger than L2 (%.1f GB cube per step)" % (nvox * C * 4 / 1e9)},
               "pipeline_frac_of_hbm_peak": nvox * BYTES_PER_PIXEL / (ms * 1e-3) / 1e9 / hbm_peak,
               "roofline": {"bound": "hbm", "kernel": "chansum_bulk_kernel", "achieved": nvox * BYTES_PER_PIXEL / (k1_ms * 1e-3) / 1e9,
                            "peak": hbm_peak, "unit": "GB/s", "frac": nvox * BYTES_PER_PIXEL / (k1_ms * 1e-3) / 1e9 / hbm_peak,
                            "ms_per_launch": k1_ms, "traffic": None},
               "stencil": {"kernel": "lne3d_q_kernel", "ms_per_launch": k4_ms, "mvox_per_s": nvox / (k4_ms * 1e-3) / 1e6,
                           "bound": "ALU pipe (min / max issue), not HBM: 12 B per voxel"},
               "gpu_launches": launches, "score_mean": float(score.mean())}
        if with_cpu and world == 1:
            # the reference's own 3-D chain on a 32^3 sub-volume (it runs at a few thousand voxels per second), and the
            # same sub-volume through the CUDA path: parity on what the CPU can finish
            from oracle import hipr_oracle, load_ref
            ref = load_ref("neighbor")
            me2 = ref.line_profile_memory_efficient_v2 if ref is not None else hipr_oracle.line_profile_memory_efficient_v2
            n = 32
            sub = cube[:n, :n, :n].contiguous()
            sub_np = sub.cpu().numpy()
            t0 = time.perf_counter()
            sm = np.sum(sub_np.astype(np.float64), axis=3)     # the scripts' arrays are float64 (np.zeros + paste)
            sm = sm / np.max(sm)
            dirs = np.asarray(me2(np.pad(sm, 5, mode="edge").astype(np.float64), 11, 9, 9))
            want = hipr_oracle.epilogue_F2_dirs(dirs)
            sec = time.perf_counter() - t0
            res["cpu_baseline"] = {"value": n ** 3 / sec / 1e6, "unit": "Mvox/s", "cores": 1,
                                   "kind": "reference" if ref is not None else "port",
                                   "sample": "%d^3 sub-volume through line_profile_memory_efficient_v2 + numpy epilogue, %.1f s" % (n, sec)}
            res["parity"] = parity_stats(ops.neighbor3d_score(sub, "ME2").cpu().numpy(), want)
    del cube, cubes
    torch.cuda.empty_cache()
    return res


def run_zstack(args):
    """--workload zstack: config 4 alone (extra line, not the headline metric)."""
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    hbm_peak = 6554.2
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    res = measure_zstack(args, dev, rank, world, args.steps, hbm_peak, with_cpu=not args.no_cpu)
    if rank == 0:
        print(json.dumps(res), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "mosaic":
        run_mosaic(args)
    elif args.workload == "zstack":
        run_zstack(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
