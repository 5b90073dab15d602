"""Times K9 (excitation_shifts: float64 channel sums + FFT cross-correlations, csrc/xcorr2d.cu) on seeded 2048^2 FOVs
in the 95-channel (32, 23, 20, 14, 6) and 63-channel (23, 20, 14, 6) layouts and prints one JSON line:
  - ms per FOV for the whole call, its channel sums alone and the FFT work (the difference), by CUDA events over
    --reps calls after warm-up; achieved GB/s against algorithmic bytes (sums: 4 B per channel read + 8 written per
    image and pixel; each 2-D complex128 FFT: 64 B/px, n forward + n - 1 inverse) and the fraction of the
    device-to-device copy rate measured in the same run;
  - the chain stacks -> shifts -> K0 -> score against K0 -> score with the shifts given;
  - the numpy oracle on one FOV on this host's CPU (--no-cpu skips it);
  - the card name and power limit (nvidia-smi query).
The working set (~1 GB per FOV) is far larger than L2.  python tools/time_shifts.py [--reps N] [--size S] [--no-cpu]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "hiprfish-image-analysis_b200"), os.path.join(ROOT, "tests")]
import numpy as np
import torch

import hipr_b200
from hipr_b200 import lib, synth
import shift_oracle

LAYOUTS = {"95": (32, 23, 20, 14, 6), "63": (23, 20, 14, 6)}
OFFSETS = [(0, 0), (2, -3), (-11, 7), (5, 0), (-1, 24)]


def events_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        idx = torch.cuda.current_device()
        name, power = [s.strip() for s in out[idx].split(",")]
        return name, power
    except Exception as e:                         # the query is informative only
        return torch.cuda.get_device_name(), "unknown (%s)" % type(e).__name__


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--no-cpu", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_shifts.py needs a CUDA device")
    H = W = args.size
    npix = H * W
    stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)   # noqa: E731

    big = torch.empty(1 << 28, dtype=torch.uint8, device="cuda")
    big2 = torch.empty_like(big)
    copy_ms = events_ms(lambda: big2.copy_(big), args.reps)
    copy_gbs = 2 * big.numel() / copy_ms / 1e6
    del big, big2

    result = {"size": [H, W], "reps": args.reps, "copy_GBps": round(copy_gbs, 1)}
    for name, chans in LAYOUTS.items():
        n = len(chans)
        offsets = OFFSETS[:n]
        m = max(max(abs(a), abs(b)) for a, b in offsets)
        cube, labels, _ = synth.make_fov(H + 2 * m, W + 2 * m, sum(chans), fov_index=7, device="cuda")
        cube += 0.1 * (labels > 0)[..., None]
        edges = np.cumsum((0,) + chans)
        stacks = [cube[m + a:m + a + H, m + b:m + b + W, edges[e]:edges[e + 1]].contiguous()
                  for e, (a, b) in enumerate(offsets)]
        del cube, labels
        shifts = hipr_b200.excitation_shifts(stacks, transform=None)
        found = bool(np.array_equal(shifts, np.asarray(offsets, dtype=np.float64)))

        need = lib().hipr_xcorr2d_workspace_bytes(H, W, n)
        work = torch.empty(need, dtype=torch.uint8, device="cuda")
        out = torch.empty((n, 2), dtype=torch.float64, device="cuda")
        sums = torch.empty((n, H, W), dtype=torch.float64, device="cuda")
        ptrs = (C.c_void_p * n)(*[s.data_ptr() for s in stacks])
        chans_np = np.asarray(chans, dtype=np.int32)

        def call():
            rc = lib().hipr_excitation_shifts(ptrs, chans_np.ctypes.data_as(C.c_void_p), n, H, W, 1, 1.0,
                                              C.c_void_p(work.data_ptr()), need, C.c_void_p(out.data_ptr()), stream())
            assert rc == 0, rc

        def sums_only():
            for e in range(n):
                rc = lib().hipr_chansum(C.c_void_p(stacks[e].data_ptr()), None, npix, chans[e],
                                        C.c_void_p(sums[e].data_ptr()), 1, None, stream())
                assert rc == 0, rc

        total_ms = events_ms(call, args.reps)
        sums_ms = events_ms(sums_only, args.reps)
        fft_ms = total_ms - sums_ms
        sum_bytes = npix * (4 * sum(chans) + 8 * n)
        fft_bytes = npix * 64 * (2 * n - 1)
        chain_est = events_ms(lambda: hipr_b200.neighbor2d_score_from_stacks(stacks, shifts="estimate",
                                                                              return_cube=False), args.reps)
        chain_given = events_ms(lambda: hipr_b200.neighbor2d_score_from_stacks(stacks, shifts=shifts,
                                                                                return_cube=False), args.reps)
        r = {
            "stacks": n, "channels": sum(chans), "offsets_found": found,
            "shifts_ms": round(total_ms, 3), "sums_ms": round(sums_ms, 3), "fft_ms": round(fft_ms, 3),
            "sums_GBps": round(sum_bytes / sums_ms / 1e6, 1), "fft_GBps": round(fft_bytes / fft_ms / 1e6, 1),
            "sums_frac_copy": round(sum_bytes / sums_ms / 1e6 / copy_gbs, 3),
            "fft_frac_copy": round(fft_bytes / fft_ms / 1e6 / copy_gbs, 3),
            "chain_estimate_ms": round(chain_est, 3), "chain_given_shifts_ms": round(chain_given, 3),
        }
        if not args.no_cpu:
            host = [s.cpu().numpy() for s in stacks]
            t0 = time.perf_counter()
            want = shift_oracle.excitation_shifts(host, "log", 1.0)
            r["numpy_oracle_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
            r["oracle_equal"] = bool(np.array_equal(want, hipr_b200.excitation_shifts(stacks, "log", 1.0)))
        result["layout_" + name] = r
        del stacks, work, sums
        torch.cuda.empty_cache()
    result["device"], result["power_limit"] = card()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
