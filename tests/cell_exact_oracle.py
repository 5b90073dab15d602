"""Exact references for the per-cell stage (csrc/cell_spectra.cu, csrc/cell_geometry.cu) and the label layouts
where its kernels branch.  numpy and the standard library only: no torch, no GPU.

Spectra.  cell_accumulate_kernel sums a run of equal labels in float32 registers, flushes it into float64 sums at
every label change and at the end of each 32-pixel group (a run never holds more than 32 pixels), and
cell_rows_kernel divides once by the integer pixel count.  On cubes of values k * 2**e with integer 0 <= k < 4096
(`dyadic_cube`: 12-bit counts over their full scale) a run sum is below 32 * 4096 * 2**e on a 2**e grid -- 17
significant bits, exact in float32 -- and every float64 total is exact while a cell has fewer than 2**41 pixels.  The
mean is then one correctly rounded division, the same one oracle.cell_spectra's float64 bincount makes, so the
device's table must equal it bit for bit, whatever order the atomics land in.  That holds for every power of two e
that keeps a 32-pixel sum finite in float32: e = 110 (sums below 2**127) and e = -149 (subnormal values; the library
is built without flush-to-zero) included.  `float32_run_sums` restates the kernel's run walk on the CPU, so the
argument can be checked without a device.

Geometry.  cell_geometry_kernel forms, from 64-bit integer raw moments, the centroid as (double) m1 / n and the
central moments as (double)(n * sum(x y) - sum(x) sum(y)) / n from 128-bit integers.  While those integers are below
2**53 each value is one correctly rounded division and equals float(Fraction(...)) exactly; above, it is within one
ulp.  `exact_geometry` gives those values as Fractions, and the eigenvalues, axis lengths, eccentricity and
orientation of the kernel's formulas in 50-digit decimal arithmetic.
"""
import decimal
from decimal import Decimal
from fractions import Fraction

import numpy as np

GROUP = 32               # pixels of one warp's group in cell_accumulate_kernel
COMPACT_CHUNK = 1024     # labels per step of cell_compact_kernel's scan
DIGITS = 50

_CTX = decimal.Context(prec=DIGITS + 10)


# --------------------------------------------------------------------------------------------------------------
# data
# --------------------------------------------------------------------------------------------------------------

def dyadic_cube(shape, C, seed, scale_exp=-12):
    """float32 array shape + (C,) of values k * 2**scale_exp, k uniform in [0, 4096)."""
    k = np.random.default_rng(seed).integers(0, 4096, tuple(shape) + (C,))
    cube = np.ldexp(k.astype(np.float64), scale_exp).astype(np.float32)
    assert np.array_equal(cube.astype(np.float64), np.ldexp(k.astype(np.float64), scale_exp))   # representable
    return cube


def wide_range_cube(shape, C, seed):
    """float32 array shape + (C,) of mixed-sign values with magnitudes spread over 2**-20 ... 2**20."""
    rng = np.random.default_rng(seed)
    mant = rng.uniform(1.0, 2.0, tuple(shape) + (C,))
    sign = rng.choice([-1.0, 1.0], tuple(shape) + (C,))
    return np.ldexp(sign * mant, rng.integers(-20, 20, tuple(shape) + (C,))).astype(np.float32)


# --------------------------------------------------------------------------------------------------------------
# label layouts where the spectra kernels branch (flat layouts: the accumulator walks the label image as a flat
# array, so each of these is built along the flat index and reshaped to any shape)
# --------------------------------------------------------------------------------------------------------------

def _flat(shape):
    return int(np.prod(shape, dtype=np.int64))


def checkerboard(shape, seed=0):
    """Two labels alternating at every pixel along every axis: a label change at every pixel."""
    idx = np.indices(shape).sum(axis=0)
    return (idx % 2 + 1).astype(np.int64)


def stripes(shape, seed=0):
    """One-pixel stripes along the fastest axis, one label per column; with an odd row length the label changes
    drift against the 32-pixel groups from row to row."""
    return (np.indices(shape)[-1] + 1).astype(np.int64)


def run_lengths(shape, seed=0):
    """Runs of every length 1..70 separated by background gaps of 0..33 pixels.  Runs come in pairs of one label,
    so a label also resumes after a gap inside a group (the kernel keeps the run open across background)."""
    n = _flat(shape)
    out = np.zeros(n, np.int64)
    p, i = 0, seed
    while p < n:
        length, gap = i % 70 + 1, i % 34
        out[p:p + length] = (i // 2) % 37 + 1
        p += length + gap
        i += 1
    return out.reshape(shape)


def group_fill(shape, seed=0):
    """32-pixel groups holding exactly k = 0..32 foreground pixels at random positions (k = group index mod 33),
    labels drawn from 1..5."""
    n = _flat(shape)
    rng = np.random.default_rng(seed)
    out = np.zeros(n, np.int64)
    for g in range((n + GROUP - 1) // GROUP):
        width = min(GROUP, n - g * GROUP)
        k = min(g % (GROUP + 1), width)
        pos = g * GROUP + rng.choice(width, k, replace=False)
        out[pos] = rng.integers(1, 6, k)
    return out.reshape(shape)


def recurring(shape, seed=0):
    """label = (p * 7919) % 13 + 1: every pixel foreground, 13 cells each recurring in many separated runs."""
    return ((np.arange(_flat(shape), dtype=np.int64) * 7919) % 13 + 1).reshape(shape)


CHUNK_EDGE_IDS = (1, 1023, 1024, 1025, 2047, 2048, 2049, (1 << 20) + 1)


def sparse_ids(shape, seed=0):
    """Runs of the ids at the edges of cell_compact_kernel's 1024-label chunks (the largest just above 2**20),
    in random order and lengths, between background gaps."""
    n = _flat(shape)
    rng = np.random.default_rng(seed)
    out = np.zeros(n, np.int64)
    p = 0
    while p < n:
        length = int(rng.integers(1, 40))
        out[p:p + length] = CHUNK_EDGE_IDS[int(rng.integers(0, len(CHUNK_EDGE_IDS)))]
        p += length + int(rng.integers(0, 5))
    return out.reshape(shape)


def negative_labels(shape, seed=0):
    """Runs of labels in -3..5: negative labels are background."""
    return random_runs(shape, seed, low=-3, high=6)


def whole(shape, seed=0):
    """One label covering the whole image."""
    return np.full(shape, 3, np.int64)


def random_runs(shape, seed=0, low=0, high=7, max_run=40):
    """Runs of random lengths 1..max_run with random labels in [low, high) (0 and below: background)."""
    n = _flat(shape)
    rng = np.random.default_rng(seed)
    lengths = rng.integers(1, max_run + 1, n + 1)
    ends = np.cumsum(lengths)
    k = int(np.searchsorted(ends, n)) + 1
    return np.repeat(rng.integers(low, high, k), lengths[:k])[:n].astype(np.int64).reshape(shape)


SPECTRA_LAYOUTS = {f.__name__: f for f in (checkerboard, stripes, run_lengths, group_fill, recurring, sparse_ids,
                                           negative_labels, whole, random_runs)}


def float32_run_sums(cube, labels, max_label=None):
    """cell_accumulate_kernel's walk on the CPU: the foreground pixels (0 < label <= max_label) of each 32-pixel
    group, split into runs of equal labels, each summed sequentially in float32.
    -> (run labels (m,), run pixel counts (m,), float32 run sums (m, C), float64 run sums (m, C))."""
    C = cube.shape[-1]
    lab = np.asarray(labels).reshape(-1).astype(np.int64)
    vals = np.asarray(cube, np.float32).reshape(-1, C)
    fg = lab > 0
    if max_label is not None:
        fg &= lab <= max_label
    idx = np.flatnonzero(fg)
    if idx.size == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros((0, C), np.float32), np.zeros((0, C))
    lab_fg, grp = lab[idx], idx // GROUP
    starts = np.flatnonzero(np.r_[True, (lab_fg[1:] != lab_fg[:-1]) | (grp[1:] != grp[:-1])])
    counts = np.diff(np.r_[starts, idx.size])
    assert counts.max() <= GROUP
    s32 = np.zeros((starts.size, C), np.float32)
    s64 = np.zeros((starts.size, C), np.float64)
    for j in range(int(counts.max())):
        live = counts > j
        v = vals[idx[starts[live] + j]]
        s32[live] += v                      # float32 + float32 -> float32, pixel by pixel as the kernel adds
        s64[live] += v.astype(np.float64)
    return lab_fg[starts], counts, s32, s64


# --------------------------------------------------------------------------------------------------------------
# geometry
# --------------------------------------------------------------------------------------------------------------

def exact_moments(seg, max_label=None):
    """{label: (n, sum r, sum c, sum r^2, sum c^2, sum r c)} as Python integers, for every label with
    0 < label <= max_label of the 2-D label image."""
    seg = np.asarray(seg)
    keep = seg > 0
    if max_label is not None:
        keep &= seg <= max_label
    r, c = np.nonzero(keep)
    if r.size == 0:
        return {}
    lab = seg[r, c].astype(np.int64)
    order = np.argsort(lab, kind="stable")
    lab, r, c = lab[order], r[order].astype(np.int64), c[order].astype(np.int64)
    # int64 partial sums: exact while n * max(coordinate)^2 < 2**63
    assert r.size * max(int(r.max()), int(c.max()), 1) ** 2 < 2 ** 63
    starts = np.flatnonzero(np.r_[True, lab[1:] != lab[:-1]])
    sums = [np.add.reduceat(x, starts) for x in (np.ones_like(r), r, c, r * r, c * c, r * c)]
    return {int(lab[s]): tuple(int(x[i]) for x in sums) for i, s in enumerate(starts)}


def _dec(q):
    """Fraction -> Decimal in the working context."""
    return _CTX.divide(Decimal(q.numerator), Decimal(q.denominator))


def _atan_small(x):
    """atan(x) for 0 <= x <= 1 by argument halving and the Taylor series."""
    halvings = 0
    while x > Decimal("0.05"):
        x = _CTX.divide(x, _CTX.add(1, _CTX.sqrt(_CTX.add(1, _CTX.multiply(x, x)))))
        halvings += 1
    eps = Decimal(10) ** -(_CTX.prec + 2)
    total, term, x2, n = Decimal(0), x, _CTX.multiply(x, x), 0
    while _CTX.abs(term) > eps:
        t = _CTX.divide(term, 2 * n + 1)
        total = _CTX.add(total, t) if n % 2 == 0 else _CTX.subtract(total, t)
        term = _CTX.multiply(term, x2)
        n += 1
    return _CTX.multiply(total, 2 ** halvings)


_PI = None


def pi_decimal():
    global _PI
    if _PI is None:   # Machin: pi = 16 atan(1/5) - 4 atan(1/239)
        _PI = _CTX.subtract(_CTX.multiply(16, _atan_small(_CTX.divide(1, 5))),
                            _CTX.multiply(4, _atan_small(_CTX.divide(1, 239))))
    return _PI


def atan2_decimal(y, x):
    """atan2 in decimal arithmetic, with C's conventions: atan2(0, x < 0) = +pi, atan2(0, 0) = 0."""
    pi = pi_decimal()
    half_pi = _CTX.divide(pi, 2)
    if x == 0:
        return half_pi if y > 0 else (_CTX.minus(half_pi) if y < 0 else Decimal(0))
    ay, ax = _CTX.abs(y), _CTX.abs(x)
    t = _atan_small(_CTX.divide(ay, ax)) if ay <= ax else _CTX.subtract(half_pi, _atan_small(_CTX.divide(ax, ay)))
    if x < 0:
        t = _CTX.subtract(pi, t)
    return _CTX.minus(t) if y < 0 else t


def geometry_from_moments(m):
    """One label's raw moments (n, sr, sc, srr, scc, src) -> dict of exact values: centroid and central moments as
    Fractions, the integer numerators of those (sr, sc; a2, c2, b2 = n * mu), the covariance a, b, c, and l1 >= l2, major / minor axis length,
    eccentricity and orientation as Decimals, by the formulas of cell_geometry_kernel and oracle.cell_geometry."""
    n, sr, sc, srr, scc, src = m
    a2, c2, b2 = n * srr - sr * sr, n * scc - sc * sc, n * src - sr * sc
    g = {"area": n, "sr": sr, "sc": sc, "a2": a2, "c2": c2, "b2": b2,
         "centroid_row": Fraction(sr, n), "centroid_col": Fraction(sc, n),
         "mu20": Fraction(a2, n), "mu02": Fraction(c2, n), "mu11": Fraction(b2, n)}
    a, c, b = Fraction(a2, n * n), Fraction(c2, n * n), Fraction(b2, n * n)     # covariance of (row, col)
    g.update(a=a, b=b, c=c)
    tr = a + c
    root = _CTX.sqrt(_dec((a - c) ** 2 + 4 * b * b))
    l1 = _CTX.divide(_CTX.add(_dec(tr), root), 2)
    # l2 = (tr - root) / 2 = 2 (a c - b^2) / (tr + root): no cancellation, and exactly 0 for a line (a c == b^2)
    det = a * c - b * b
    l2 = _CTX.divide(_CTX.multiply(2, _dec(det)), _CTX.add(_dec(tr), root)) if tr > 0 else Decimal(0)
    g.update(l1=l1, l2=_CTX.max(l2, Decimal(0)))
    g["major_axis_length"] = _CTX.multiply(4, _CTX.sqrt(l1))
    g["minor_axis_length"] = _CTX.multiply(4, _CTX.sqrt(g["l2"]))
    g["eccentricity"] = Decimal(0) if l1 == 0 else _CTX.sqrt(_CTX.subtract(1, _CTX.divide(g["l2"], l1)))
    # 'rc' orientation: a == c -> -pi/4 if mu11 > 0 else pi/4, else 0.5 atan2(2 b, a - c)
    quarter = _CTX.divide(pi_decimal(), 4)
    g["orientation"] = ((_CTX.minus(quarter) if b > 0 else quarter) if a == c
                        else _CTX.divide(atan2_decimal(_dec(2 * b), _dec(a - c)), 2))
    return g


def exact_geometry(seg, max_label=None):
    """-> (labels int64 (n,), [geometry_from_moments dict per label]), labels ascending, 0 < label <= max_label."""
    mom = exact_moments(seg, max_label)
    labels = sorted(mom)
    return np.array(labels, np.int64), [geometry_from_moments(mom[k]) for k in labels]


GEOMETRY_COLUMNS = ("centroid_row", "centroid_col", "major_axis_length", "minor_axis_length", "eccentricity",
                    "orientation", "mu20", "mu02", "mu11")


def geometry_table(rows):
    """exact_geometry's rows -> float64 (n, 9) in the column order of hipr_b200.cell_geometry, each entry the
    exact value rounded once."""
    return np.array([[float(g[k]) for k in GEOMETRY_COLUMNS] for g in rows], np.float64).reshape(-1, 9)


# --------------------------------------------------------------------------------------------------------------
# geometry layouts (2-D)
# --------------------------------------------------------------------------------------------------------------

def rods(shape, seed=0, origin=(0, 0), box=40, half_len=(4, 14), radius=(1.0, 4.0)):
    """Capsules ("rods", the domain's cells) at angles spread over [0, pi), one per box x box tile of the region
    starting at `origin`; label = tile index + 1."""
    H, W = shape
    rng = np.random.default_rng(seed)
    out = np.zeros(shape, np.int64)
    r0, c0 = origin
    ny, nx = (H - r0) // box, (W - c0) // box
    yy, xx = np.mgrid[0:box, 0:box].astype(np.float64)
    for i in range(ny * nx):
        ty, tx = divmod(i, nx)
        ang = np.pi * i / max(ny * nx, 1) + rng.uniform(0, 0.05)
        hl, rad = rng.uniform(*half_len), rng.uniform(*radius)
        cy, cx = box / 2 + rng.uniform(-2, 2), box / 2 + rng.uniform(-2, 2)
        u = (xx - cx) * np.cos(ang) + (yy - cy) * np.sin(ang)
        v = -(xx - cx) * np.sin(ang) + (yy - cy) * np.cos(ang)
        du = np.maximum(np.abs(u) - hl, 0.0)
        inside = (du * du + v * v) <= rad * rad
        inside[0, :] = inside[-1, :] = inside[:, 0] = inside[:, -1] = False
        tile = out[r0 + ty * box: r0 + (ty + 1) * box, c0 + tx * box: c0 + (tx + 1) * box]
        tile[inside] = i + 1
    return out


LINE_LENGTHS = (2, 3, 5, 8, 13, 21, 34)


def lines(seed=0):
    """One-pixel lines -- horizontal, vertical, diagonal and anti-diagonal, of lengths 2..34 -- each in its own 36 x 36
    box of a 149 x 257 image (odd width: the moments kernel's 32-pixel strips wrap mid-row).
    -> (labels, {label: kind}), kind in "hvda"."""
    out = np.zeros((4 * 36 + 5, 7 * 36 + 5), np.int64)
    kinds = {}
    for k, kind in enumerate("hvda"):
        for i, length in enumerate(LINE_LENGTHS):
            lab = 1 + k * len(LINE_LENGTHS) + i
            r0, c0 = 3 + 36 * k, 2 + 36 * i
            t = np.arange(length)
            rr, cc = {"h": (r0 + 0 * t, c0 + t), "v": (r0 + t, c0 + 0 * t), "d": (r0 + t, c0 + t),
                      "a": (r0 + t, c0 + length - 1 - t)}[kind]
            out[rr, cc] = lab
            kinds[lab] = kind
    return out, kinds


def round_shapes(shape=(60, 75), seed=0):
    """Single pixels, squares and plus shapes: mu20 == mu02 (the a == c branch of the orientation)."""
    out = np.zeros(shape, np.int64)
    lab = 0
    for i in range(4):
        lab += 1
        out[2 + 3 * i, 2] = lab                                   # single pixel
        k = i + 2
        lab += 1
        out[2 + 14 * i: 2 + 14 * i + k, 8: 8 + k] = lab           # k x k square
        lab += 1
        r, c, arm = 6 + 14 * i, 30, i + 1                          # plus with arms of length arm
        out[r - arm: r + arm + 1, c] = lab
        out[r, c - arm: c + arm + 1] = lab
        lab += 1
        d = np.arange(2 * i + 3)                                   # an X: mu20 == mu02, mu11 == 0
        out[2 + 14 * i + d, 50 + d] = lab
        out[2 + 14 * i + d, 50 + 2 * i + 2 - d] = lab
    return out
