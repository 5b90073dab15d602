"""The exact references of tests/cell_exact_oracle.py checked on the CPU: against oracle.cell_geometry, against the
exactness argument the GPU tests rest on, and the argument checks of the host entry point that come before any
library call."""
import math
from fractions import Fraction

import numpy as np
import pytest

import cell_exact_oracle as X


@pytest.mark.parametrize("H,W,drop", [(160, 200, 0.0), (97, 131, 0.2)])
def test_exact_geometry_matches_numpy_oracle(oracle, H, W, drop):
    from hipr_b200 import synth
    labels, _ = synth.make_labels(H, W, seed=H + W, drop_fraction=drop)
    seg = labels.numpy()
    wl, wa, wg = oracle.cell_geometry(seg)
    lab, rows = X.exact_geometry(seg)
    assert np.array_equal(lab, wl)
    assert np.array_equal([g["area"] for g in rows], wa)
    got = X.geometry_table(rows)
    np.testing.assert_allclose(got[:, :5], wg[:, :5], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(got[:, 6:], wg[:, 6:], rtol=1e-12, atol=1e-9)
    d = np.abs(got[:, 5] - wg[:, 5])
    assert np.all(np.minimum(d, np.pi - d) < 1e-9)


def test_exact_geometry_special_shapes():
    """Lines have l2 == 0 exactly; squares, plus and X shapes have mu20 == mu02 and take the +-pi/4 branch."""
    seg, kinds = X.lines()
    lab, rows = X.exact_geometry(seg)
    assert list(lab) == sorted(kinds)
    for k, g in zip(lab, rows):
        assert g["l2"] == 0 and g["minor_axis_length"] == 0 and g["eccentricity"] == 1
        want = {"h": math.pi / 2, "v": 0.0, "d": -math.pi / 4, "a": math.pi / 4}[kinds[k]]
        assert float(g["orientation"]) == want
        assert float(g["major_axis_length"]) == pytest.approx(4 * math.sqrt(float(g["a"] + g["c"])), rel=1e-15)
    lab, rows = X.exact_geometry(X.round_shapes())
    assert len(rows) == 16
    for g in rows:
        assert g["mu20"] == g["mu02"] and g["mu11"] == 0 and float(g["orientation"]) == math.pi / 4
        assert abs(g["l1"] - g["l2"]) <= g["l1"] * X.Decimal("1e-50")


def test_decimal_atan2_against_math():
    rng = np.random.default_rng(0)
    for y, x in rng.normal(size=(200, 2)) * np.exp(rng.uniform(-5, 5, (200, 1))):
        got = float(X.atan2_decimal(X._dec(Fraction(y)), X._dec(Fraction(x))))
        assert got == pytest.approx(math.atan2(y, x), rel=4e-16, abs=1e-300)
    assert float(X.pi_decimal()) == math.pi
    assert str(X.pi_decimal())[:52] == "3.14159265358979323846264338327950288419716939937510"


def test_exact_moments_integers():
    seg = np.zeros((5, 7), np.int64)
    seg[1, 2] = seg[3, 6] = 4
    seg[0, :] = 9
    seg[4, 4] = -2
    mom = X.exact_moments(seg)
    assert mom == {4: (2, 4, 8, 10, 40, 20), 9: (7, 0, 21, 0, 91, 0)}
    assert X.exact_moments(seg, max_label=5) == {4: mom[4]}


@pytest.mark.parametrize("name", sorted(X.SPECTRA_LAYOUTS))
@pytest.mark.parametrize("scale_exp", [-12, 110, -149])
def test_float32_run_sums_are_exact_on_dyadic_cubes(oracle, name, scale_exp):
    """The kernel's run walk, restated with float32 run sums, gives float64 totals equal to the float64 bincount:
    on dyadic cubes the GPU table has one exact answer."""
    shape = (37, 41)
    lab = X.SPECTRA_LAYOUTS[name](shape, 5)
    cube = X.dyadic_cube(shape, 7, seed=11, scale_exp=scale_exp)
    run_lab, run_n, s32, s64 = X.float32_run_sums(cube, lab)
    assert np.array_equal(s32.astype(np.float64), s64)
    if run_lab.size == 0:
        return
    sums = np.zeros((int(run_lab.max()) + 1, 7))
    counts = np.zeros(int(run_lab.max()) + 1, np.int64)
    np.add.at(sums, run_lab, s32.astype(np.float64))
    np.add.at(counts, run_lab, run_n)
    wl, wa, wavg, _ = oracle.cell_spectra(lab, cube)
    assert np.array_equal(counts[wl], wa)
    assert np.array_equal(sums[wl] / counts[wl][:, None], wavg)


def test_float32_run_sums_worst_case_and_negative_control():
    """Full-scale counts in full 32-pixel runs stay exact; general float32 data does not (the exactness is a
    property of the data the tests choose, not of any 32-term float32 sum)."""
    lab = np.ones((4, 64), np.int64)
    for e in (-12, 110, -149):
        cube = np.full((4, 64, 3), np.ldexp(np.float32(4095), e), np.float32)
        _, n, s32, s64 = X.float32_run_sums(cube, lab)
        assert np.all(n == 32) and np.array_equal(s32.astype(np.float64), s64)
        assert np.all(np.isfinite(s32)) and np.all(s32 > 0)
    cube = X.wide_range_cube((4, 64), 3, seed=1)
    _, _, s32, s64 = X.float32_run_sums(cube, lab)
    assert not np.array_equal(s32.astype(np.float64), s64)


def test_layouts_hit_the_kernel_branches():
    """The layouts hold what their names promise."""
    g = X.group_fill((33 * 32,), 0).reshape(-1, 32)
    assert [int((row > 0).sum()) for row in g] == list(range(33))
    r = (X.run_lengths((20000,)).ravel() > 0).astype(np.int8)
    edges = np.flatnonzero(np.diff(np.r_[1, r, 1]))
    assert set(range(1, 34)) <= set((edges[1::2] - edges[0::2]).tolist())          # every background gap 1..33
    s = X.sparse_ids((4000,), 0)
    assert set(np.unique(s[s > 0]).tolist()) == set(X.CHUNK_EDGE_IDS)
    c = X.checkerboard((3, 5, 7))
    assert np.all(np.diff(c.ravel())[np.arange(c.size - 1) % 7 != 6] != 0)
    assert (X.negative_labels((50, 50), 0) < 0).any()


def test_cell_spectra_host_rejects_a_transposed_label_image():
    """A (H, W, C) cube with a (W, H) label image has the right number of pixels and the wrong pairing: refused
    before any library call (so also without a device)."""
    import hipr_b200
    cube = np.zeros((5, 7, 3), np.float32)
    with pytest.raises(ValueError, match=r"\(5, 7, 3\).*\(7, 5\)"):
        hipr_b200.cell_spectra_host(cube, np.zeros((7, 5), np.int32))
    with pytest.raises(ValueError):
        hipr_b200.cell_spectra_host(cube, np.zeros(35, np.int32))
