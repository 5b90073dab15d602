"""Times K10 (connected-component labelling, csrc/label.cu) and the operators built on it with CUDA events after
warm-up, next to scipy.ndimage on one host core in the same run, and checks every timed result against scipy.

  python tools/time_label.py [--reps N] [--json PATH]

Inputs: the 2048^2 synthetic capsule mask (synth.make_labels), 2048^2 noise at the percolation threshold of 4- and
8-connectivity, the 2048^2 one-pixel serpentine, and a 1024 x 1024 x 64 volume (smoothed noise, 26-connectivity).
A 2048^2 working set (mask 4 MB, parent array 16 MB, labels 16 MB) stays in the 126 MB L2 between repetitions;
the volume's (64 + 256 + 256 MB) does not."""
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


def label_call(mask_dev, conn):
    """hipr_label on preallocated buffers: the five launches and nothing else."""
    dims = (mask_dev.dim(),) + tuple(mask_dev.shape) + (1,) * (3 - mask_dev.dim())
    ws = hipr_b200.lib().hipr_label_workspace_bytes(*dims)
    work = torch.empty(ws, dtype=torch.uint8, device="cuda")
    out = torch.empty(mask_dev.shape, dtype=torch.int32, device="cuda")
    n = torch.empty(1, dtype=torch.int64, device="cuda")
    raw = mask_dev.view(torch.uint8)
    lib = hipr_b200.lib()

    def run():
        ops.check(lib.hipr_label(C.c_void_p(raw.data_ptr()), 4, 0, *dims, conn, C.c_void_p(work.data_ptr()), ws,
                                 C.c_void_p(out.data_ptr()), 4, C.c_void_p(n.data_ptr()), ops._stream()), "label")
    return run, out, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    torch.set_num_threads(1)
    rng = np.random.default_rng(0)
    lab, _ = synth.make_labels(2048, 2048)
    capsules = (lab > 0).numpy()
    snake = np.zeros((2048, 2048), bool)
    snake[0::2] = True
    snake[1::4, -1] = True
    snake[3::4, 0] = True
    volume = ndi.uniform_filter(rng.random((1024, 1024, 64), dtype=np.float32), 3) > 0.55
    cases = [("capsules 2048^2", capsules, 1), ("capsules 2048^2", capsules, 2),
             ("noise p=0.593 2048^2", rng.random((2048, 2048)) < 0.593, 1),
             ("noise p=0.407 2048^2", rng.random((2048, 2048)) < 0.407, 2),
             ("serpentine 2048^2", snake, 1),
             ("smoothed noise 1024x1024x64", volume, 3)]
    rows = []
    print("card, power limit:", card())
    for name, mask, conn in cases:
        st = ndi.generate_binary_structure(mask.ndim, conn)
        want, wn = ndi.label(mask, st)
        dev = torch.from_numpy(mask).cuda()
        run, out, n = label_call(dev, conn)
        reps = args.reps if mask.size <= 2 ** 22 else max(5, args.reps // 5)
        ms = device_ms(run, reps)
        run()
        ok = int(n.item()) == wn and np.array_equal(out.cpu().numpy(), want)
        op_ms = device_ms(lambda: hipr_b200.label(dev, conn), reps)
        cpu = host_ms(lambda: ndi.label(mask, st))
        rows.append(dict(op="label", input=name, connectivity=conn, components=int(wn), device_ms=round(ms, 4),
                         operator_ms=round(op_ms, 4), scipy_ms=round(cpu, 2), exact=ok))
        print("label %-28s conn %d  n %8d  hipr_label %.3f ms  label() %.3f ms  scipy %.1f ms  exact %s"
              % (name, conn, wn, ms, op_ms, cpu, ok))
    for name, mask in (("capsules 2048^2", capsules), ("smoothed noise 1024x1024x64", volume)):
        dev = torch.from_numpy(mask).cuda()
        reps = args.reps if mask.size <= 2 ** 22 else max(5, args.reps // 5)
        for op, fn, ref in (
                ("binary_fill_holes", lambda: hipr_b200.binary_fill_holes(dev), lambda: ndi.binary_fill_holes(mask)),
                ("remove_small_objects", lambda: hipr_b200.remove_small_objects(dev, 64),
                 lambda: _rso(mask, 64)),
                ("clear_border", lambda: hipr_b200.clear_border(dev), None)):
            ms = device_ms(fn, reps)
            got = fn().cpu().numpy()
            cpu, ok = None, None
            if ref is not None:
                cpu = host_ms(ref, 1 if mask.size > 2 ** 22 else 3)
                ok = bool(np.array_equal(got, ref()))
            rows.append(dict(op=op, input=name, operator_ms=round(ms, 4),
                             scipy_ms=None if cpu is None else round(cpu, 2), exact=ok))
            print("%-20s %-28s operator %.3f ms  scipy %s  exact %s"
                  % (op, name, ms, "-" if cpu is None else "%.1f ms" % cpu, ok))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(dict(card=card(), rows=rows), f, indent=1)


def _rso(mask, min_size):
    lab, _ = ndi.label(mask)
    sizes = np.bincount(lab.ravel())
    out = mask.copy()
    out[sizes[lab] < min_size] = False
    return out


if __name__ == "__main__":
    main()
