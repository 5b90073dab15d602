"""Times K12 (binary morphology, csrc/morphology.cu) with CUDA events after warm-up, next to scipy.ndimage on one host
core in the same run, and checks every timed result against scipy.

  python tools/time_morphology.py [--reps N] [--json PATH]

Inputs: the 2048^2 synthetic capsule mask (synth.make_labels > 0) under binary_opening with the cross, disk(2) and
disk(5) and under binary_erosion with disk(3) and iterations=2; 2048^2 noise at p = 0.5 under binary_opening with the
cross; a 1024 x 1024 x 64 smoothed-noise volume under binary_opening with the 6-neighbour cross and ball(3).

"pass" is one hipr_binary_morphology pass (one launch) on preallocated buffers; "operator" is the public call with its
allocations.  A pass reads and writes one byte per pixel, so its traffic is 2 x npix bytes; the share of the HBM rate
is that over the pass time and 7.7 TB/s.  A 2048^2 working set (4 MB in, 4 MB out) stays in the 126 MB L2 between
repetitions, so its share is a nominal figure; the volume's (64 MB in, 64 MB out) is at the size of L2."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "hiprfish-image-analysis_b200")]
import numpy as np  # noqa: E402
import scipy.ndimage as ndi  # noqa: E402
import torch  # noqa: E402

import hipr_b200  # noqa: E402
from hipr_b200 import ops, synth  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name()


def device_ms(fn, reps):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def host_ms(fn, reps=3):
    best = float("inf")
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t)
    return best * 1e3


def disk(r):
    y, x = np.mgrid[-r:r + 1, -r:r + 1]
    return x * x + y * y <= r * r


def ball(r):
    z, y, x = np.mgrid[-r:r + 1, -r:r + 1, -r:r + 1]
    return x * x + y * y + z * z <= r * r


def pass_call(mask_dev, structure, dilate):
    """One hipr_binary_morphology pass on preallocated buffers: one launch and nothing else."""
    dims = (mask_dev.dim(),) + tuple(mask_dev.shape) + (1,) * (3 - mask_dev.dim())
    s = ops._structure(structure, mask_dev.dim())
    sdims = s.shape + (1,) * (3 - s.ndim)
    raw = mask_dev.view(torch.uint8)
    out = torch.empty_like(raw)
    lib = hipr_b200.lib()

    def run():
        ops.check(lib.hipr_binary_morphology(C.c_void_p(raw.data_ptr()), *dims, s.ctypes.data_as(C.c_void_p), *sdims,
                                             int(dilate), 0, 1, None, 0, C.c_void_p(out.data_ptr()), ops._stream()),
                  "binary_morphology")
    return run, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    torch.set_num_threads(1)
    rng = np.random.default_rng(0)
    lab, _ = synth.make_labels(2048, 2048)
    capsules = (lab > 0).numpy()
    noise = rng.random((2048, 2048)) < 0.5
    volume = ndi.gaussian_filter(rng.random((1024, 1024, 64), dtype=np.float32), 2) > 0.5
    cross2, cross3 = ndi.generate_binary_structure(2, 1), ndi.generate_binary_structure(3, 1)
    cases = [("capsules 2048^2", capsules, "opening", "cross", cross2, 1),
             ("capsules 2048^2", capsules, "opening", "disk(2)", disk(2), 1),
             ("capsules 2048^2", capsules, "opening", "disk(5)", disk(5), 1),
             ("capsules 2048^2", capsules, "erosion", "disk(3)", disk(3), 2),
             ("noise p=0.5 2048^2", noise, "opening", "cross", cross2, 1),
             ("smoothed noise 1024x1024x64", volume, "opening", "6-cross", cross3, 1),
             ("smoothed noise 1024x1024x64", volume, "opening", "ball(3)", ball(3), 1)]
    rows = []
    print("card, power limit:", card())
    for name, mask, op, sname, st, it in cases:
        dev = torch.from_numpy(mask).cuda()
        big = mask.size > 2 ** 22
        reps = max(5, args.reps // 5) if big else args.reps
        f = getattr(hipr_b200, "binary_" + op)
        ref = getattr(ndi, "binary_" + op)
        passes = it * (2 if op in ("opening", "closing") else 1)
        run_e, _ = pass_call(dev, st, False)
        run_d, _ = pass_call(dev, st, True)
        ero_ms = device_ms(run_e, reps)
        dil_ms = device_ms(run_d, reps)
        op_ms = device_ms(lambda: f(dev, st, it), reps)
        want = ref(mask, st, it)
        ok = bool(np.array_equal(f(dev, st, it).cpu().numpy(), want))
        cpu = host_ms(lambda: ref(mask, st, it), 1 if big else 3)
        pass_ms = (ero_ms + dil_ms) / 2
        share = 2 * mask.size / (pass_ms * 1e-3) / HBM_BYTES_PER_S
        rows.append(dict(op=op, input=name, structure=sname, members=int(np.count_nonzero(st)),
                         runs=int(ops._structure_runs(ops._structure(st, mask.ndim)).shape[0]), iterations=it,
                         erosion_pass_ms=round(ero_ms, 4), dilation_pass_ms=round(dil_ms, 4),
                         operator_ms=round(op_ms, 4), passes=passes, scipy_ms=round(cpu, 2),
                         pass_hbm_share=round(share, 3), exact=ok))
        print("%-8s %-28s %-8s it %d  pass: erosion %.4f ms dilation %.4f ms (%.2f of HBM)  operator %.4f ms "
              "(%d passes)  scipy %.1f ms  exact %s" % (op, name, sname, it, ero_ms, dil_ms, share, op_ms, passes,
                                                         cpu, ok))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(dict(card=card(), rows=rows), f, indent=1)
    if not all(r["exact"] for r in rows):
        sys.exit("a timed result differs from scipy")


if __name__ == "__main__":
    main()
