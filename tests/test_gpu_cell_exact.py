"""The per-cell stage against exact references (tests/cell_exact_oracle.py): mean spectra bit for bit on dyadic
cubes through all three entry points, error-bounded on general float32 data, numpy's semantics on non-finite input,
the overflow counter of the C ABI; geometry bit for bit where the kernel's integer moments make it exact and within
bounds derived from the eigenproblem's conditioning elsewhere; paint for every table dtype."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest

import cell_exact_oracle as X

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -52
CHANNELS = [1, 31, 32, 33, 64, 65, 96, 97, 127, 128, 129, 255, 256, 257, 300]   # CK = 1..4 and 128-channel passes


def _cu(t, a):
    return t.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(table):
    return tuple(x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x) for x in table)


def _assert_same_table(got, want):
    """Labels and areas equal; avgint and avgint_norm equal value for value (NaN where the reference has NaN)."""
    gl, ga, gavg, gnorm = _host(got)
    wl, wa, wavg, wnorm = _host(want)
    assert gl.dtype == np.int64 and ga.dtype == np.int64
    assert np.array_equal(gl, wl) and np.array_equal(ga, wa)
    assert gavg.shape == wavg.shape and gnorm.shape == wnorm.shape
    assert np.array_equal(gavg, wavg, equal_nan=True)
    assert np.array_equal(gnorm, wnorm, equal_nan=True)


def _spectra_case(torch, oracle, lab, cube, label_dtype=np.int32, max_label=None):
    import hipr_b200
    lab = lab.astype(label_dtype)
    got = hipr_b200.cell_spectra(_cu(torch, cube), _cu(torch, lab), max_label)
    ref = lab if max_label is None else np.where(lab > max_label, 0, lab)
    want = oracle.cell_spectra(ref, cube)
    _assert_same_table(got, want)
    return got


# ---------------------------------------------------------------------------------------------------------------
# spectra, bit for bit on dyadic cubes
# ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("C", [33, 130])
@pytest.mark.parametrize("label_dtype", [np.int32, np.int64])
@pytest.mark.parametrize("layout", sorted(X.SPECTRA_LAYOUTS))
def test_spectra_layouts_bit_exact(torch_cuda, oracle, layout, label_dtype, C):
    shape = (61, 67)
    lab = X.SPECTRA_LAYOUTS[layout](shape, C)
    _spectra_case(torch_cuda, oracle, lab, X.dyadic_cube(shape, C, seed=C + 1), label_dtype)


@pytest.mark.parametrize("scale_exp", [-12, 110, -149])
@pytest.mark.parametrize("C", CHANNELS)
def test_spectra_channel_counts_and_scales_bit_exact(torch_cuda, oracle, C, scale_exp):
    shape = (37, 53)
    lab = X.group_fill(shape, C)
    lab[:3] = X.run_lengths((3, 53), C)
    cube = X.dyadic_cube(shape, C, seed=C, scale_exp=scale_exp)
    _spectra_case(torch_cuda, oracle, lab, cube, np.int64 if C % 2 else np.int32)


@pytest.mark.parametrize("shape", [(1,), (31,), (32,), (33,), (1023,), (1025,), (1, 1), (3, 11), (31, 33), (33, 31),
                                   (7, 147), (5, 7, 9), (3, 33, 31), (2, 1, 1025)])
@pytest.mark.parametrize("label_dtype", [np.int32, np.int64])
def test_spectra_sizes_bit_exact(torch_cuda, oracle, shape, label_dtype):
    n = int(np.prod(shape))
    lab = X.random_runs(shape, n, low=0, high=5, max_run=9)
    if n == 1:
        lab[...] = 2
    _spectra_case(torch_cuda, oracle, lab, X.dyadic_cube(shape, 65, seed=n), label_dtype)


@pytest.mark.parametrize("layout", ["checkerboard", "recurring", "group_fill", "run_lengths"])
def test_spectra_volumes_bit_exact(torch_cuda, oracle, layout):
    shape = (6, 17, 23)
    lab = X.SPECTRA_LAYOUTS[layout](shape, 3)
    _spectra_case(torch_cuda, oracle, lab, X.dyadic_cube(shape, 97, seed=4), np.int64)


@pytest.mark.parametrize("shape,cuts", [((70, 45), (1, 2, 19, 20, 33, 34, 69)),
                                        ((9, 13, 7), (1, 2, 5, 8))])
@pytest.mark.parametrize("C", [65, 129])
def test_spectra_slabs_accumulate_bit_exact(torch_cuda, oracle, shape, cuts, C):
    """Slabs cut at rows that are not multiples of 32 (one-row slabs among them) accumulated into one table: the
    same table as one call, equal to the reference."""
    import hipr_b200
    t = torch_cuda
    lab = X.random_runs(shape, 7, low=-1, high=9, max_run=13).astype(np.int32)
    cube = X.dyadic_cube(shape, C, seed=8)
    c, l = _cu(t, cube), _cu(t, lab)
    L = int(lab.max())
    sums = counts = None
    for r0, r1 in zip((0,) + cuts, cuts + (shape[0],)):
        sums, counts = hipr_b200.cell_spectra_accumulate(c[r0:r1], l[r0:r1], L, sums, counts)
    got = hipr_b200.cell_spectra_finalize(sums, counts)
    _assert_same_table(got, oracle.cell_spectra(lab, cube))
    _assert_same_table(got, hipr_b200.cell_spectra(c, l))


def test_spectra_three_entry_points_agree_bit_for_bit(torch_cuda, oracle):
    """cell_spectra, slab accumulation and the host entry point (a 200 x 256 x 257 cube: three 96-row bands) give
    one table, the reference's, and the same table again on a second run."""
    import hipr_b200
    t = torch_cuda
    shape, Cn = (200, 256), 257
    lab = X.random_runs(shape, 21, low=0, high=40, max_run=60)
    lab[50:53] = X.recurring((3, 256))
    lab[120:122] = X.sparse_ids((2, 256), 1)
    lab = lab.astype(np.int32)
    cube = X.dyadic_cube(shape, Cn, seed=22)
    want = oracle.cell_spectra(lab, cube)
    c, l = _cu(t, cube), _cu(t, lab)
    dev = hipr_b200.cell_spectra(c, l)
    _assert_same_table(dev, want)
    _assert_same_table(hipr_b200.cell_spectra(c, l), dev)
    sums = counts = None
    for r0, r1 in ((0, 1), (1, 95), (95, 96), (96, 161), (161, 200)):
        sums, counts = hipr_b200.cell_spectra_accumulate(c[r0:r1], l[r0:r1], int(lab.max()), sums, counts)
    _assert_same_table(hipr_b200.cell_spectra_finalize(sums, counts), want)
    host = hipr_b200.cell_spectra_host(cube, lab)
    _assert_same_table(host, want)
    _assert_same_table(hipr_b200.cell_spectra_host(cube, lab.astype(np.int64)), host)


# ---------------------------------------------------------------------------------------------------------------
# spectra on general float32 data, non-finite input, explicit max_label, the overflow counter, shape checks
# ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", ["random_runs", "recurring", "checkerboard"])
@pytest.mark.parametrize("C", [33, 130])
def test_spectra_general_float32_within_the_run_sum_bound(torch_cuda, layout, C):
    """|avg - exact| <= 32 * 2**-24 * mean|x| + 2**-52 * |exact|: float32 run sums of at most 32 pixels, exact
    float64 totals up to rounding, one division.  The exact mean from math.fsum per cell and channel."""
    import hipr_b200
    shape = (24, 29)
    lab = X.SPECTRA_LAYOUTS[layout](shape, 2).astype(np.int32)
    cube = X.wide_range_cube(shape, C, seed=C)
    labels, area, avg, _ = _host(hipr_b200.cell_spectra(_cu(torch_cuda, cube), _cu(torch_cuda, lab)))
    flat, vals = lab.reshape(-1), cube.reshape(-1, C).astype(np.float64)
    assert np.array_equal(labels, np.unique(flat[flat > 0]))
    for i, k in enumerate(labels):
        v = vals[flat == k]
        assert area[i] == v.shape[0]
        for ch in range(C):
            exact = Fraction(math.fsum(v[:, ch])) / v.shape[0]
            bound = 32 * 2.0 ** -24 * float(np.abs(v[:, ch]).mean()) + EPS * abs(float(exact))
            assert abs(Fraction(avg[i, ch]) - exact) <= Fraction(bound), (k, ch)


def test_spectra_non_finite_input_follows_numpy(torch_cuda, oracle):
    """NaN in one channel of one pixel: NaN mean there and a NaN avgint_norm row; +inf and -inf in one cell (in one
    run and in two groups): NaN; a lone inf: inf (and inf / inf = NaN in its avgint_norm row)."""
    shape, Cn = (8, 64), 40
    lab = np.zeros(shape, np.int32)
    lab[0, 2:30] = 1
    lab[1, :] = 2
    lab[2, 5:9] = 3
    lab[3, 0:64] = 4
    lab[5, 3:20] = 5
    cube = X.dyadic_cube(shape, Cn, seed=3)
    cube[0, 7, 4] = np.nan
    cube[1, 3, 6], cube[1, 40, 6] = np.inf, -np.inf         # cell 2: two groups -> inf + -inf in float64
    cube[3, 10, 9], cube[3, 11, 9] = np.inf, -np.inf        # cell 4: one run -> NaN in float32
    cube[2, 6, 11] = np.inf                                 # cell 3: lone inf
    cube[5, 4, 12] = -np.inf
    labels, _, avg, norm = _spectra_case(torch_cuda, oracle, lab, cube)
    avg, norm = avg.cpu().numpy(), norm.cpu().numpy()
    assert np.isnan(avg[0, 4]) and np.isnan(norm[0]).all() and np.isfinite(np.delete(avg[0], 4)).all()
    assert np.isnan(avg[1, 6]) and np.isnan(avg[3, 9]) and np.isnan(norm[1]).all() and np.isnan(norm[3]).all()
    assert avg[2, 11] == np.inf and np.isnan(norm[2, 11]) and (np.delete(norm[2], 11) == 0).all()
    assert avg[4, 12] == -np.inf and np.isfinite(norm[4, :12]).all()


@pytest.mark.parametrize("label_dtype", [np.int32, np.int64])
def test_spectra_labels_above_max_label_are_background(torch_cuda, oracle, label_dtype):
    shape = (45, 77)
    lab = X.random_runs(shape, 5, low=-4, high=60, max_run=11)
    cube = X.dyadic_cube(shape, 97, seed=6)
    for k in (1, 17, 31, 58):
        labels, area, _, _ = _host(_spectra_case(torch_cuda, oracle, lab, cube, label_dtype, max_label=k))
        assert labels.max() <= k and area.sum() == ((lab > 0) & (lab <= k)).sum()


@pytest.mark.parametrize("Cn", [95, 300])
@pytest.mark.parametrize("label_dtype", [np.int32, np.int64])
def test_overflow_counter_counts_each_pixel_once(torch_cuda, oracle, Cn, label_dtype):
    """hipr_cell_spectra_accumulate's overflow_dev counts the pixels with label > max_label once, whatever the
    number of 128-channel passes; those pixels are not accumulated."""
    import hipr_b200
    t = torch_cuda
    shape, max_label = (51, 83), 25
    lab = X.random_runs(shape, Cn, low=-2, high=41, max_run=7).astype(label_dtype)
    cube = X.dyadic_cube(shape, Cn, seed=Cn)
    c, l = _cu(t, cube), _cu(t, lab)
    sums = t.zeros((max_label + 1, Cn), dtype=t.float64, device="cuda")
    counts = t.zeros(max_label + 1, dtype=t.int32, device="cuda")
    ovf = t.zeros(1, dtype=t.int32, device="cuda")
    stream = C.c_void_p(t.cuda.current_stream().cuda_stream)
    for _ in range(2):       # the counter is added to, like the sums
        assert hipr_b200.lib().hipr_cell_spectra_accumulate(
            C.c_void_p(c.data_ptr()), C.c_void_p(l.data_ptr()), lab.itemsize, lab.size, shape[1], Cn, max_label,
            C.c_void_p(sums.data_ptr()), C.c_void_p(counts.data_ptr()), C.c_void_p(ovf.data_ptr()), stream) == 0
    t.cuda.synchronize()
    assert int(ovf.item()) == 2 * int((lab > max_label).sum()) > 0
    ref = np.where(lab > max_label, 0, lab)
    wl, wa, wavg, wnorm = oracle.cell_spectra(ref, cube)
    _assert_same_table(hipr_b200.cell_spectra_finalize(sums / 2, t.div(counts, 2, rounding_mode="floor")),
                       (wl, wa, wavg, wnorm))


def test_spectra_refuse_a_label_image_shaped_unlike_the_cube(torch_cuda):
    import hipr_b200
    t = torch_cuda
    cube = t.zeros((6, 10, 3), device="cuda")
    for bad in ((10, 6), (60,), (6, 10, 1), (2, 3, 10)):
        with pytest.raises(ValueError, match=r"\(6, 10, 3\)"):
            hipr_b200.cell_spectra(cube, t.ones(bad, dtype=t.int32, device="cuda"), 1)
        with pytest.raises(ValueError):
            hipr_b200.cell_spectra_accumulate(cube, t.ones(bad, dtype=t.int32, device="cuda"), 1)
    with pytest.raises(ValueError):
        hipr_b200.cell_spectra_host(np.zeros((6, 10, 3), np.float32), np.ones((10, 6), np.int32))


# ---------------------------------------------------------------------------------------------------------------
# geometry
# ---------------------------------------------------------------------------------------------------------------

def _ulps(got, exact):
    """|got - exact| in units of the spacing of float(exact) (exact: Fraction)."""
    f = float(exact)
    return abs(Fraction(got) - exact) / Fraction(np.spacing(abs(f))) if f != 0 else (0 if got == 0 else math.inf)


def _check_geometry(torch, seg, max_label=None, label_dtype=np.int32):
    """cell_geometry against exact_geometry; -> (device table, exact rows)."""
    import hipr_b200
    lab, area, geom = _host(hipr_b200.cell_geometry(_cu(torch, seg.astype(label_dtype)), max_label))
    wl, rows = X.exact_geometry(seg, max_label)
    assert np.array_equal(lab, wl)
    assert np.array_equal(area, [g["area"] for g in rows])
    for i, g in enumerate(rows):
        # integer numerators below 2**53: one correctly rounded division, bit for bit; above: within one ulp
        for col, key, num in ((0, "centroid_row", "sr"), (1, "centroid_col", "sc"),
                              (6, "mu20", "a2"), (7, "mu02", "c2"), (8, "mu11", "b2")):
            exact = g[key]
            if abs(g[num]) < 2 ** 53:
                assert geom[i, col] == float(exact), (lab[i], key, geom[i, col], float(exact))
            else:
                assert _ulps(geom[i, col], exact) <= 1, (lab[i], key)
        l1, l2 = g["l1"], g["l2"]
        maj, minr, ecc, ori = (float(x) for x in geom[i, 2:6])
        # major axis: relative 16 eps
        assert abs(X.Decimal(maj) - g["major_axis_length"]) <= X.Decimal(16 * EPS) * g["major_axis_length"]
        # |l2_dev - l2| <= 16 eps l1, through the minor axis (l2_dev = (minor / 4)^2, exactly) and 1 - ecc^2
        l2_dev = (X.Decimal(minr) / 4) ** 2
        assert abs(l2_dev - l2) <= X.Decimal(16 * EPS) * l1, (lab[i], minr)
        if l1 > 0:
            assert abs((1 - X.Decimal(ecc) ** 2) - l2 / l1) <= X.Decimal(16 * EPS), (lab[i], ecc)
        else:
            assert ecc == 0.0
        # orientation modulo pi: exact +-pi/4 where a == c, else within 16 eps l1 / (l1 - l2) (+ atan2's rounding)
        if g["a"] == g["c"]:
            assert ori == float(g["orientation"]), (lab[i], ori)
        else:
            d = abs(X.Decimal(ori) - g["orientation"]) % X.pi_decimal()
            d = min(d, X.pi_decimal() - d)
            assert d <= X.Decimal(16 * EPS) * (l1 / (l1 - l2) + 1), (lab[i], ori, float(g["orientation"]))
    return (lab, area, geom), rows


@pytest.mark.parametrize("shape,origin,label_dtype", [((290, 333), (0, 0), np.int32),
                                                       ((60300, 131), (60000, 5), np.int64),
                                                       ((210, 65013), (3, 64700), np.int32),
                                                       ((1000, 13), (0, 0), np.int64)])
def test_geometry_rods_exact(torch_cuda, shape, origin, label_dtype):
    """Rods at angles over [0, pi), near the origin, at rows ~60000, at columns ~65000, and on a 13-pixel-wide
    image (every 32-pixel strip of the moments kernel spans three rows)."""
    box = 40 if shape[1] > 13 else 12
    seg = X.rods(shape, seed=shape[0], origin=origin, box=box,
                 half_len=(4, 14) if box == 40 else (1, 3), radius=(1.0, 4.0) if box == 40 else (1.0, 2.5))
    _, rows = _check_geometry(torch_cuda, seg, label_dtype=label_dtype)
    assert len(rows) >= 6


def test_geometry_lines_are_exact(torch_cuda):
    """One-pixel lines: l2 == 0 exactly, so minor_axis_length == 0.0 and eccentricity == 1.0; horizontal pi/2,
    vertical 0, diagonal -pi/4, anti-diagonal +pi/4."""
    seg, kinds = X.lines()
    (lab, _, geom), _ = _check_geometry(torch_cuda, seg)
    assert np.all(geom[:, 3] == 0.0) and np.all(geom[:, 4] == 1.0)
    want = {"h": math.pi / 2, "v": 0.0, "d": -math.pi / 4, "a": math.pi / 4}
    assert np.array_equal(geom[:, 5], [want[kinds[k]] for k in lab])


def test_geometry_round_shapes_take_the_quarter_pi_branch(torch_cuda):
    """Single pixels, squares, plus and X shapes: mu20 == mu02 exactly, orientation exactly pi/4; a single pixel
    has zero axes and eccentricity 0."""
    seg = X.round_shapes()
    (lab, area, geom), rows = _check_geometry(torch_cuda, seg)
    assert np.all(geom[:, 6] == geom[:, 7]) and np.all(geom[:, 8] == 0.0)
    assert np.all(geom[:, 5] == math.pi / 4)
    one = area == 1
    assert one.sum() == 4 and np.all(geom[one, 2:5] == 0.0)


@pytest.mark.parametrize("shape", [(2048, 2048), (1, 65536), (65536, 1)])
def test_geometry_one_label_covering_the_image(torch_cuda, shape):
    """Numerators above 2**53: the central moments within one ulp of the exact value."""
    seg = np.ones(shape, np.int32)
    (_, area, geom), rows = _check_geometry(torch_cuda, seg)
    assert area[0] == seg.size
    assert max(abs(rows[0]["a2"]), abs(rows[0]["c2"])) >= 2 ** 53


def test_geometry_ignores_labels_outside_one_to_max_label(torch_cuda):
    rng = np.random.default_rng(9)
    seg = X.rods((200, 243), seed=4)
    noise = rng.random(seg.shape) < 0.02
    seg[noise & (seg == 0)] = -rng.integers(1, 5, int((noise & (seg == 0)).sum()))
    L = int(seg.max())
    for k in (L, L // 2, 1):
        (lab, _, _), _ = _check_geometry(torch_cuda, seg, max_label=k, label_dtype=np.int64)
        assert lab.size and lab.max() <= k


# ---------------------------------------------------------------------------------------------------------------
# paint
# ---------------------------------------------------------------------------------------------------------------

def _table(rng, rows, K, dtype):
    shape = (rows,) if K is None else (rows, K)
    if dtype == np.bool_:
        return rng.random(shape) < 0.5
    if np.issubdtype(dtype, np.integer):
        info = np.iinfo(dtype)
        return rng.integers(info.min, info.max, shape, dtype=dtype, endpoint=True)
    return (rng.standard_normal(shape) * 1e3).astype(dtype)


@pytest.mark.parametrize("K", [None, 1, 3, 5])
@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.int32, np.int64, np.uint8, np.bool_])
@pytest.mark.parametrize("label_dtype", [np.int32, np.int64])
def test_paint_every_table_dtype(torch_cuda, dtype, K, label_dtype):
    """out = values[where((lab < 0) | (lab > max_label), 0, lab)], with the default max_label (the table's last
    row) and with an explicit max_label below it."""
    import hipr_b200
    rng = np.random.default_rng(K or 0)
    L = 57
    lab = X.random_runs((37, 71), 1, low=-3, high=L + 9, max_run=5).astype(label_dtype)
    values = _table(rng, L + 1, K, dtype)
    for max_label in (None, L - 20, 0):
        got = hipr_b200.paint_labels(_cu(torch_cuda, lab), _cu(torch_cuda, values), max_label).cpu().numpy()
        m = L if max_label is None else max_label
        want = values[np.where((lab < 0) | (lab > m), 0, lab)]
        assert got.dtype == want.dtype and got.shape == want.shape
        assert np.array_equal(got, want)
