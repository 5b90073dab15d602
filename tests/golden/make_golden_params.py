"""Generates tests/golden/oracle_params_vectors.npz: the oracle's line profiles at the non-default parameter sets of
tests/test_oracle.py, on the same seeded inputs as its compiled-reference comparisons.

These are outputs of the oracle (oracle/hipr_oracle.py), frozen so that a clean checkout notices when they change.
Where oracle/_ref is built (oracle/build_ref.py), this script first asserts that the compiled original gives the
same arrays, so the file is then also a record of the original's outputs.

    python tests/golden/make_golden_params.py
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import hipr_oracle as O, load_ref  # noqa: E402

PARAMS_2D = [(11, 9), (7, 5), (11, 4), (15, 9), (11, 12), (5, 3), (13, 16)]
PARAMS_3D = [(11, 9, 9), (7, 5, 4), (9, 6, 7), (5, 3, 3)]


def input_2d(P, R):
    return np.random.default_rng(P * 100 + R).random((P + 12, P + 16))


def input_3d(params):
    P = params[0]
    a = np.random.default_rng(sum(params)).random((P + 10, P + 4, P + 3))
    return a, a[:P + 2, :P + 2, :P + 1]


def key(params):
    return "_".join(str(p) for p in params)


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def main():
    r2, r3 = load_ref("neighbor2d"), load_ref("neighbor")
    out = {}
    for P, R in PARAMS_2D:
        a = input_2d(P, R)
        lp = O.line_profile_2d_v2(a, P, R)
        if r2 is not None:
            assert np.array_equal(r2.line_profile_2d_v2(a, P, R), lp)
        out["lp2d_sha256_" + key((P, R))] = sha(lp)
    for params in PARAMS_3D:
        a, small = input_3d(params)
        lp = O.line_profile_v2(a, *params)
        me2 = O.line_profile_memory_efficient_v2(small, *params)
        v3 = O.line_profile_memory_efficient_v3(a, *params)
        if r3 is not None:
            assert np.array_equal(r3.line_profile_v2(a, *params), lp)
            assert np.array_equal(r3.line_profile_memory_efficient_v2(small, *params), me2)
            ok = ~np.isnan(v3)
            assert np.array_equal(r3.line_profile_memory_efficient_v3(a, *params)[ok], v3[ok])
        out["lp3d_sha256_" + key(params)] = sha(lp)
        out["me2_3d_" + key(params)] = me2
        out["v3_" + key(params)] = v3
    path = os.path.join(HERE, "oracle_params_vectors.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes;",
          "checked against the compiled original" if r2 is not None and r3 is not None else "oracle/_ref not built")


if __name__ == "__main__":
    main()
