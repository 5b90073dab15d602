"""Outputs of the fixed-point stencils (csrc/lne2d_q.cu, csrc/lne3d.cu, csrc/fused2d.cu) and of the registration paste
(csrc/register.cu) on seeded inputs at the benchmark's sizes, for comparing two builds of libhipr_b200.so bit for bit.
Dump once per library, each in its own process, then compare:

    python tools/fixed_point_outputs.py dump A.npz [--lib path/to/libhipr_b200.so]
    python tools/fixed_point_outputs.py dump B.npz --lib other/libhipr_b200.so
    python tools/fixed_point_outputs.py compare A.npz B.npz
"""
import argparse
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hiprfish-image-analysis_b200"))


def dump(path, lib_path):
    import torch
    from hipr_b200 import _lib
    if lib_path:
        _lib.LIB_PATH = os.path.abspath(lib_path)
    import hipr_b200
    from hipr_b200 import ops, synth, tables
    torch.cuda.set_device(0)
    out = {}
    dev = "cuda"

    def put(name, t):
        out[name] = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)

    # 2-D: one synthetic 2048 x 2048 x 95 field of view, its channel sums through the stencil entry point
    cube, _, _ = synth.make_fov(2048, 2048, 95, fov_index=0)
    cube = cube.to(dev)
    score, s, _ = ops.neighbor2d_pipeline(cube, "F1")
    put("pipeline_F1_score", score)
    put("pipeline_F1_sum", s)
    for fl in ("F1", "F2"):
        sc, ss, _ = ops.neighbor2d_fused(cube, fl, return_sum=True)
        put("fused_%s_score" % fl, sc)
        put("fused_%s_sum" % fl, ss)
    pinned = np.ascontiguousarray(tables.line_table_2d(11, 9), dtype=np.int32)
    other = np.ascontiguousarray(pinned[:, ::-1, :])     # same lines, samples reversed: not the baked table
    for dt in (torch.float64, torch.float32):
        img = s.to(dt).contiguous()
        keys = ops.image_range(img)
        for fl in ("F1", "F2", "F3"):
            for rng in ("local", "global"):
                if rng == "local" and fl == "F3":
                    continue
                for tname, tab in (("baked", pinned), ("table", other)):
                    o = torch.empty((2048, 2048), dtype=torch.float32, device=dev)
                    ops.check(_lib.lib().hipr_lne2d_q(
                        C.c_void_p(img.data_ptr()), 2048, 2048, 2048, 0, ops._DT[dt], 11, 9,
                        tab.ctypes.data_as(C.c_void_p), _lib.FLAVOURS[fl], keys.ptr() if rng == "global" else None,
                        C.c_void_p(o.data_ptr()), None), "hipr_lne2d_q")
                    put("lne2d_%s_%s_%s_%s" % (str(dt)[6:], fl, rng, tname), o)
    # 3-D: a seeded smooth volume at the z-stack benchmark's size, and a smaller one for the per-direction output
    g = torch.Generator(device=dev).manual_seed(11)

    def volume(X, Y, Z):
        v = torch.rand((1, 1, X, Y, Z), generator=g, device=dev, dtype=torch.float64)
        v = torch.nn.functional.avg_pool3d(v, 5, stride=1, padding=2)[0, 0]
        return (v + 0.05 * torch.rand((X, Y, Z), generator=g, device=dev, dtype=torch.float64)).contiguous()

    vol = volume(1024, 1024, 64)
    mk = ops.image_range(vol)
    for fl in ("F2", "F3", "ME2"):
        put("lne3d_%s" % fl, ops.lne3d_fixed(vol, fl, maxkey=mk))
    small = volume(128, 128, 64)
    put("lne3d_dirs", ops.lne3d_fixed(small, "ME2", maxkey=ops.image_range(small), dirs_only=True))
    del vol, small
    # registration paste, 95- and 63-channel layouts, with and without a flat field
    for chans in ((32, 23, 20, 14, 6), (23, 20, 14, 6)):
        shifts = [(0, 0), (3, -2), (-4, 1), (2, 5), (-1, -3)][:len(chans)]
        stacks = [torch.rand((2048, 2048, c), generator=g, device=dev) + 0.1 for c in chans]
        cal = torch.rand((2048, 2048, sum(chans)), generator=g, device=dev) + 0.5
        for cname, cc in (("plain", None), ("flat", cal)):
            rc, rs, rk = hipr_b200.register_stacks(stacks, shifts, cc)
            put("register_%d_%s_cube" % (sum(chans), cname), rc)
            put("register_%d_%s_sum" % (sum(chans), cname), rs)
        del stacks, cal
    torch.cuda.synchronize()
    np.savez(path, **out)
    print("dumped %d arrays from %s" % (len(out), _lib.LIB_PATH))


def compare(a_path, b_path):
    a, b = np.load(a_path), np.load(b_path)
    bad = sorted(set(a.files) ^ set(b.files))
    for k in sorted(set(a.files) & set(b.files)):
        same = np.array_equal(a[k], b[k], equal_nan=True) and a[k].dtype == b[k].dtype
        print("%-40s %-14s %s" % (k, "x".join(map(str, a[k].shape)), "equal" if same else "DIFFERENT"))
        if not same:
            bad.append(k)
    print("%d arrays, %d differ" % (len(a.files), len(bad)))
    return 1 if bad else 0


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    sub = ap.add_subparsers(dest="cmd", required=True)
    d = sub.add_parser("dump")
    d.add_argument("out")
    d.add_argument("--lib", default=None)
    c = sub.add_parser("compare")
    c.add_argument("a")
    c.add_argument("b")
    args = ap.parse_args()
    if args.cmd == "dump":
        dump(args.out, args.lib)
    else:
        sys.exit(compare(args.a, args.b))
