"""Times K11 (the marker watershed, csrc/watershed.cu) with CUDA events after warm-up, and reports per case the
rounds of its three phases, the tile visits and an upper bound on the bytes each round moves.

  python tools/time_watershed.py [--reps N] [--json PATH]

Cases: the 2048^2 synthetic FOV chain (negated F1 score map as the landscape, markers from the brightest fifth of the
k-means mask, the filled and cleaned mask as the watershed mask), a 2048^2 noise landscape with 2,000 random markers,
a constant 2048^2 plateau with 2,000 random markers, the 2048^2 one-pixel serpentine with one marker (the worst case:
the flood crosses the image 1,024 times), and a 1024 x 1024 x 64 noise volume with 20,000 markers at connectivity 3.
Each 2-D working set (image, markers, 16 B of workspace per pixel: under 110 MB) stays in the 126 MB L2 between
repetitions; the volume's (1.3 GB) does not.  The 2-D results are checked against the Python rule
(tests/watershed_oracle.py), whose run time is printed as the restatement time; scikit-image's own flood is not
installed here, so no speed-up over it is claimed."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "hiprfish-image-analysis_b200"), os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import hipr_b200  # noqa: E402
from hipr_b200 import ops, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name()


def device_ms(fn, reps, warmup=2):
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


def watershed_call(image, markers, mask, conn):
    """hipr_watershed on preallocated buffers: the memset and the one launch, no NaN check, no status read."""
    lib = hipr_b200.lib()
    dims = (image.dim(),) + tuple(image.shape) + (1,) * (3 - image.dim())
    code = 1 if image.dtype == torch.float64 else 0
    ws = lib.hipr_watershed_workspace_bytes(*dims, code, markers.element_size())
    work = torch.empty(ws, dtype=torch.uint8, device="cuda")
    out = torch.empty_like(markers)
    status = torch.zeros(8, dtype=torch.int64, device="cuda")
    m = None if mask is None else C.c_void_p(mask.view(torch.uint8).data_ptr())

    def run():
        ops.check(lib.hipr_watershed(C.c_void_p(image.data_ptr()), code, C.c_void_p(markers.data_ptr()),
                                     markers.element_size(), m, *dims, conn, C.c_void_p(work.data_ptr()), ws,
                                     C.c_void_p(out.data_ptr()), C.c_void_p(status.data_ptr()), ops._stream()),
                  "watershed")
    return run, out, status


def bytes_per_visit(image, markers, mask):
    """Upper bound per tile visit: the halo'd tile of the phase's words, the per-pixel inputs, the write-back."""
    if image.dim() == 2:
        t = min(64, image.shape[0]) * min(64, image.shape[1])
        halo = (min(64, image.shape[0]) + 2) * (min(64, image.shape[1]) + 2)
    else:
        e = [min(16, s) for s in image.shape]
        t, halo = e[0] * e[1] * e[2], (e[0] + 2) * (e[1] + 2) * (e[2] + 2)
    inputs = image.element_size() + markers.element_size() + (0 if mask is None else 1)
    return (halo * 8 + t * (inputs + 8), halo * 4 + t * 8, halo * 8 + t * 12)


def random_markers(rng, shape, n):
    m = np.zeros(shape, np.int32)
    m.ravel()[rng.choice(m.size, n, replace=False)] = np.arange(1, n + 1)
    return m


def serpentine(H, W):
    m = np.zeros((H, W), bool)
    m[::2] = True
    for r in range(1, H, 2):
        m[r, W - 1 if (r // 2) % 2 == 0 else 0] = True
    return m


def chain_case():
    cube, _, _ = synth.make_fov(2048, 2048, 95, fov_index=3)
    score = ops.neighbor2d_score(cube.cuda(), "F1")
    kept = ops.remove_small_objects(ops.binary_fill_holes(ops.kmeans_threshold(score, 2).mask), 20)
    thr = torch.quantile(score[kept].float()[::7], 0.8)
    markers = ops.label(ops.remove_small_objects(kept & (score >= thr), 4), connectivity=1)
    return (-score).contiguous(), markers, kept


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default=None)
    ap.add_argument("--no-check", action="store_true", help="skip the Python restatement")
    args = ap.parse_args()
    import watershed_oracle as wo
    rng = np.random.default_rng(0)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    cases = [("fov chain 2048^2", chain_case, 1, args.reps),
             ("noise 2048^2", lambda: (cu(rng.random((2048, 2048)).astype(np.float32)),
                                       cu(random_markers(rng, (2048, 2048), 2000)), None), 1, args.reps),
             ("plateau 2048^2", lambda: (cu(np.full((2048, 2048), 0.5, np.float32)),
                                         cu(random_markers(rng, (2048, 2048), 2000)), None), 1, args.reps),
             ("serpentine 2048^2", lambda: (cu(rng.random((2048, 2048)).astype(np.float32)),
                                            cu(np.pad(np.ones((1, 1), np.int32), ((0, 2047), (0, 2047)))),
                                            cu(serpentine(2048, 2048))), 1, 1),
             ("volume 1024x1024x64 c3", lambda: (torch.rand(1024, 1024, 64, device="cuda"),
                                                 cu(random_markers(rng, (1024, 1024, 64), 20000)), None), 3, 3)]
    print("card, power limit:", card())
    rows = []
    for name, make, conn, reps in cases:
        image, markers, mask = make()
        run, out, status = watershed_call(image, markers, mask, conn)
        ms = device_ms(run, reps, warmup=1 if reps == 1 else 2)
        st = status.cpu().numpy()
        assert st[0] == 0, st
        rounds = int(st[1:4].sum())
        visit_bytes = bytes_per_visit(image, markers, mask)
        moved = sum(int(v) * b for v, b in zip(st[4:7], visit_bytes))
        row = dict(case=name, ms=round(ms, 3), rounds=[int(x) for x in st[1:4]], tile_visits=[int(x) for x in st[4:7]],
                   ctas=int(st[7]), mb_per_round=round(moved / max(rounds, 1) / 1e6, 2))
        if image.dim() == 2 and not args.no_check:
            t = time.perf_counter()
            want = wo.watershed_rule(image.cpu().numpy(), markers.cpu().numpy(), conn,
                                     None if mask is None else mask.cpu().numpy())
            row["restatement_s"] = round(time.perf_counter() - t, 1)
            row["equal_to_rule"] = bool(np.array_equal(out.cpu().numpy(), want))
        rows.append(row)
        print(json.dumps(row), flush=True)
        del image, markers, mask, out
        torch.cuda.empty_cache()
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(dict(card=card(), rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
