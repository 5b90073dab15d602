"""The flat-field divide (syn/..._measurement.py:104) and the raw-count rescale, checked where division code goes
wrong: every float32 divisor significand, every numerator significand, the exponent edges of the K0 fast quotient,
zero / denormal / infinite / NaN operands, and every channel position of the flat-field sums.

Three hand-written forms are covered:
  * the K0 cube quotient (csrc/register.cu): `div_rn_fast` on the aligned tiles of the compiled layouts,
    `__fdiv_rn` elsewhere -- required to equal numpy's IEEE float32 quotient bit for bit on every route;
  * the flat-field channel sums of K1 and K0 (`sum_channels_div`, csrc/hipr_common.cuh) -- each term within
    TERM_RTOL of numpy's float64 quotient, non-finite sums equal to numpy's;
  * the raw-count rescale of K1 (`raw_value`) -- bit-identical to u.astype(float32) / float32(scale).

Every reference is numpy.  Quotients are compared as uint32 bit patterns (signed zeros count), NaN by position
only.  The generators are plain functions so that the CPU tests at the top can check that they produce what the GPU
tests claim to cover."""
import numpy as np
import pytest

CHANS95 = (32, 23, 20, 14, 6)      # the reference's five excitations: 95 channels
CHANS63 = (23, 20, 14, 6)          # without the 405 nm excitation: 63 channels
NSIG = 1 << 23                     # float32 significands

# exponent fields around the K0 fast quotient's range test (ev - 67u < 121u, i.e. fields 67..187 = [2^-60, 2^61)),
# plus zero / denormal (0), the smallest and largest normal binades and inf / NaN (255)
EDGE_FIELDS = (0, 1, 66, 67, 68, 186, 187, 188, 253, 254, 255)

# numerators paired with every divisor significand in [1, 2): 1, 2 - 2^-23, 1 + 2^-23, 1.5 and three powers of two
SWEEP_NUMERATORS = np.array([1.0, 2 - 2.0 ** -23, 1 + 2.0 ** -23, 1.5, 2.0 ** -3, 2.0 ** 3, 2.0 ** 59], np.float32)
# divisors paired with every numerator significand in [1, 2)
SWEEP_DIVISORS = np.array([2 - 2.0 ** -23, 1 + 2.0 ** -23, 1.5, 3.0, 1 - 2.0 ** -24], np.float32)
N_RANDOM = 3                       # random partners per significand, on top of the structured ones

# Flat-field sums, per term: v * r0 is exact in float64; the correction v*r0 * (e + e^2) carries four float32
# roundings (e, e + e^2, v * r0, the fma into the accumulator), each <= 2^-24 relative, on a quantity <= 2^-23 of the
# term (rcp.approx is within 1 ulp); the float64 total and numpy's own quotient add 2^-53 each.
TERM_RTOL = 2.0 ** -45 + 2.0 ** -52          # 2.86e-14
SUM_RTOL = 1e-13                             # whole-pixel sums of positive terms (as test_gpu_register.py)


def _f32(bits):
    return np.asarray(bits, dtype=np.uint32).view(np.float32)


def _u32(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def _random_floats(rng, shape, fields, negative=False):
    """float32 values with random significands and exponent fields drawn from `fields` (inclusive range)."""
    e = rng.integers(fields[0], fields[1] + 1, size=shape, dtype=np.uint32)
    bits = (e << np.uint32(23)) | rng.integers(0, NSIG, size=shape, dtype=np.uint32)
    if negative:
        bits |= rng.integers(0, 2, size=shape, dtype=np.uint32) << np.uint32(31)
    return _f32(bits)


def _all_significands(field=127):
    return _f32(np.uint32(field << 23) | np.arange(NSIG, dtype=np.uint32))


# ---- generators -----------------------------------------------------------------------------------------------------
def divisor_sweep(seed=1):
    """(v, w) flat float32: all 2^23 divisor significands in [1, 2), each against SWEEP_NUMERATORS and N_RANDOM
    random numerators with exponent fields 67..187 (the fast quotient's range)."""
    rng = np.random.default_rng(seed)
    w = _all_significands()
    v = np.empty((len(SWEEP_NUMERATORS) + N_RANDOM, NSIG), np.float32)
    v[:len(SWEEP_NUMERATORS)] = SWEEP_NUMERATORS[:, None]
    v[len(SWEEP_NUMERATORS):] = _random_floats(rng, (N_RANDOM, NSIG), (67, 187), negative=True)
    return v.ravel(), np.tile(w, v.shape[0])


def numerator_sweep(seed=2):
    """(v, w) flat float32: all 2^23 numerator significands in [1, 2), each against SWEEP_DIVISORS and N_RANDOM random
    divisors with exponent fields 67..187."""
    rng = np.random.default_rng(seed)
    v = _all_significands()
    w = np.empty((len(SWEEP_DIVISORS) + N_RANDOM, NSIG), np.float32)
    w[:len(SWEEP_DIVISORS)] = SWEEP_DIVISORS[:, None]
    w[len(SWEEP_DIVISORS):] = _random_floats(rng, (N_RANDOM, NSIG), (67, 187), negative=True)
    return np.tile(v, w.shape[0]), w.ravel()


def exponent_edges(per_class=64, seed=3):
    """(v, w) flat float32: the full cross product of EDGE_FIELDS for both operands and all four sign pairs,
    `per_class` values each.  The first value of a class has significand 0 (zero, a power of two, inf), the second
    all ones; the rest are random (denormals in field 0, NaN in field 255)."""
    rng = np.random.default_rng(seed)
    fv, fw, sv, sw, k = np.meshgrid(np.array(EDGE_FIELDS, np.uint32), np.array(EDGE_FIELDS, np.uint32),
                                    np.array([0, 1], np.uint32), np.array([0, 1], np.uint32),
                                    np.arange(per_class), indexing="ij")

    def sig(shape):
        m = rng.integers(1, NSIG, size=shape, dtype=np.uint32)
        m[..., 0] = 0
        m[..., 1] = NSIG - 1
        return m

    v = (sv << np.uint32(31)) | (fv << np.uint32(23)) | sig(k.shape)
    w = (sw << np.uint32(31)) | (fw << np.uint32(23)) | sig(k.shape)
    return _f32(v.ravel()), _f32(w.ravel())


def term_positions(npix, C):
    """Channel of pixel p's single non-zero numerator: p mod C, so consecutive pixels walk every channel."""
    return np.arange(npix) % C


def term_divisor_sweep(seed=4):
    """(v, w) per pixel for the one-term sums: every divisor significand in [1, 2) with a random numerator in [1, 2)."""
    rng = np.random.default_rng(seed)
    return _random_floats(rng, NSIG, (127, 127)), _all_significands()


def wide_range_cube(H, W, C, seed=5):
    """(v, w) (H, W, C) positive: numerators with a per-pixel binade 2^-126 .. 2^125, row 1 denormal;
    divisors in [0.5, 1.5)."""
    rng = np.random.default_rng(seed)
    k = rng.integers(-126, 126, size=(H, W, 1))
    k[0, :2, 0] = (-126, 125)
    v = (rng.random((H, W, C)) + 1.0) * np.exp2(k.astype(np.float64))
    v = v.astype(np.float32)
    v[1] = _random_floats(rng, (W, C), (0, 0))           # denormal numerators only
    w = (0.5 + rng.random((H, W, C))).astype(np.float32)
    return v, w


# (numerator, divisor) pairs whose float64 quotient is not finite, or whose float32 intermediates are not
# (the kernels' exact float64 fallback), or whose divisor the float32 reciprocal flushes
NONFINITE_CASES = [
    (1.5, 0.0), (-1.5, 0.0), (1.5, -0.0), (0.0, 0.0),                   # inf, -inf, -inf, NaN
    (1.0, 1e-40), (1.0, float(_f32(1))), (-2.0, float(_f32(0x80000005))),  # denormal divisors: finite in float64
    (1.0, np.inf), (np.inf, np.inf), (np.inf, 1.0), (-np.inf, 2.0),     # 0, NaN, inf, -inf
    (1.0, np.nan), (np.nan, 1.0),                                       # NaN
    (2.0 ** 127, 0.75), (2.0 ** 127, 0.5), (3e38, 1e-3),                # v * r0 overflows float32
    (1e-40, 1.0), (float(_f32(1)), 1.5),                                # denormal numerators
]


def nonfinite_cube(npix, C, seed=6):
    """(v, w) (npix, C): random positive terms, except channel p mod C of pixel p, which takes
    NONFINITE_CASES[(p // C) mod len(NONFINITE_CASES)], so that every case meets every channel position."""
    rng = np.random.default_rng(seed)
    v = (0.5 + rng.random((npix, C))).astype(np.float32)
    w = (0.5 + rng.random((npix, C))).astype(np.float32)
    p = np.arange(npix)
    case = (p // C) % len(NONFINITE_CASES)
    cases = np.array(NONFINITE_CASES, np.float32)
    v[p, p % C] = cases[case, 0]
    w[p, p % C] = cases[case, 1]
    return v, w


def flushed_divisor_cube(npix, C, seed=7):
    """(v, w) (npix, C) positive, channel p mod C of pixel p holding a divisor above 2^126 (exponent fields
    253 / 254, significand non-zero) under a numerator in [2^100, 2^127)."""
    rng = np.random.default_rng(seed)
    v = (0.5 + rng.random((npix, C))).astype(np.float32)
    w = (0.5 + rng.random((npix, C))).astype(np.float32)
    p = np.arange(npix)
    big = _f32(((253 + p % 2) << 23).astype(np.uint32) | rng.integers(1, NSIG, size=npix, dtype=np.uint32))
    v[p, p % C] = _random_floats(rng, npix, (227, 253))          # the term stays visible in the sum
    w[p, p % C] = big
    return v, w


RANGE_KINDS = ("nan", "nan_inf", "inf", "all_nan")


def range_cube(kind, npix, C, seed=8):
    """(npix, C) float32 whose channel sums contain NaN and / or +inf at a few pixels (all NaN for "all_nan")."""
    rng = np.random.default_rng(seed)
    v = rng.random((npix, C), dtype=np.float32)
    if kind == "all_nan":
        v[:, 7] = np.nan
    if kind in ("nan", "nan_inf"):
        v[[3, npix // 2, npix - 1], [0, 50, C - 1]] = np.nan
    if kind in ("inf", "nan_inf"):
        v[[5, npix - 2], [1, C - 2]] = np.inf
    return v


def range_reference(sums):
    """The range rule of DESIGN.md section 2: max / min skip NaN (np.nanmax / np.nanmin); -inf / +inf when every sum
    is NaN.  normalize divides by that max: finite / inf = 0, inf / inf = NaN, NaN stays NaN."""
    finite_or_inf = sums[~np.isnan(sums)]
    vmax = finite_or_inf.max() if finite_or_inf.size else -np.inf
    vmin = finite_or_inf.min() if finite_or_inf.size else np.inf
    with np.errstate(invalid="ignore", divide="ignore"):
        return vmax, vmin, sums / vmax


RAW_SCALES = (65535.0, 4095.0, 255.0, 1.0, 3.0, 65536.0)


def raw_counts_cube(bits, C, extra=37):
    """(n, C) raw counts, one non-zero sample per pixel: pixel p holds count p (mod 2^bits) at channel p mod C;
    2^bits pixels plus `extra` (a ragged remainder after the 128-pixel chunks)."""
    n = (1 << bits) + extra
    p = np.arange(n)
    u = np.zeros((n, C), np.uint16 if bits > 8 else np.uint8)
    u[p, p % C] = p % (1 << bits)
    return u


# ---- CPU: the generators cover what the GPU tests claim -------------------------------------------------------------
def test_divisor_sweep_covers_every_significand():
    v, w = divisor_sweep()
    n = len(SWEEP_NUMERATORS) + N_RANDOM
    assert v.shape == w.shape == (n * NSIG,)
    wb = _u32(w).reshape(n, NSIG)
    for row in wb:                                                     # each numerator meets every significand
        assert np.array_equal(row & 0x7fffff, np.arange(NSIG)) and np.all(row >> 23 == 127)
    vb = _u32(v).reshape(n, NSIG)
    assert np.array_equal(vb[:len(SWEEP_NUMERATORS), 0], _u32(SWEEP_NUMERATORS))
    assert _u32(SWEEP_NUMERATORS)[1] == 0x3fffffff and _u32(SWEEP_NUMERATORS)[2] == 0x3f800001
    fields = (vb[len(SWEEP_NUMERATORS):] >> 23) & 0xff
    assert fields.min() == 67 and fields.max() == 187 and np.any(vb[len(SWEEP_NUMERATORS):] >> 31)
    # the case that motivated the sweep: 1 / (2 - 2^-23) is just above a rounding midpoint
    assert _u32(np.float32(1.0) / _f32(0x3fffffff)) == 0x3f000001


def test_numerator_sweep_covers_every_significand():
    v, w = numerator_sweep()
    n = len(SWEEP_DIVISORS) + N_RANDOM
    vb = _u32(v).reshape(n, NSIG)
    for row in vb:
        assert np.array_equal(row & 0x7fffff, np.arange(NSIG)) and np.all(row >> 23 == 127)
    wb = _u32(w).reshape(n, NSIG)
    assert np.array_equal(wb[:len(SWEEP_DIVISORS), 0], _u32(SWEEP_DIVISORS))
    assert _u32(SWEEP_DIVISORS)[4] == 0x3f7fffff                       # 1 - 2^-24
    fields = (wb[len(SWEEP_DIVISORS):] >> 23) & 0xff
    assert fields.min() == 67 and fields.max() == 187


def test_exponent_edges_cover_both_sides_of_the_fast_range():
    v, w = exponent_edges()
    vb, wb = _u32(v), _u32(w)
    fv, fw = (vb >> 23) & 0xff, (wb >> 23) & 0xff
    pairs = set(zip(fv.tolist(), fw.tolist()))
    assert pairs == {(a, b) for a in EDGE_FIELDS for b in EDGE_FIELDS}          # the full cross product
    for lo, hi in ((66, 67), (187, 188)):                                          # both sides of each boundary
        assert {lo, hi} <= set(fv.tolist()) and {lo, hi} <= set(fw.tolist())
    for b in (vb, wb):
        x = _f32(b)
        assert np.any(x == 0) and np.any(np.signbit(x) & (x == 0))                # +0 and -0
        assert np.any((b & 0x7f800000) == 0) and np.any(((b & 0x7f800000) == 0) & ((b & 0x7fffff) != 0))   # denormals
        assert np.any(np.isposinf(x)) and np.any(np.isneginf(x)) and np.any(np.isnan(x))
    with np.errstate(all="ignore"):
        q = v / w
    qb = _u32(q)
    assert np.any(np.isnan(q)) and np.any(np.isposinf(q)) and np.any(np.isneginf(q))
    assert np.any(qb == 0x80000000) and np.any(qb == 0)
    # pairs inside the fast range and pairs that leave it on each side
    fast = (fv - 67 < 121) & (fw - 67 < 121)
    assert fast.any() and (~fast).any()


def test_one_term_generators():
    v, w = term_divisor_sweep()
    assert np.array_equal(_u32(w) & 0x7fffff, np.arange(NSIG))
    assert np.all((_u32(v) >> 23) == 127)
    for C in (95, 63):
        for npix in (1 << 20, 1 << 12):
            assert np.array_equal(np.unique(term_positions(npix, C)), np.arange(C))


def test_wide_range_generator():
    v, w = wide_range_cube(16, 64, 95)
    e = (_u32(v) >> 23) & 0xff
    assert e.min() == 0 and e.max() == 252 and np.all(e[1] == 0) and np.all(v >= 0)
    assert {1, 252} <= set(e[0, :2].ravel().tolist())                  # the binades 2^-126 and 2^125
    assert np.all((w >= 0.5) & (w < 1.5))


def test_nonfinite_generator_reaches_every_case_and_position():
    C, npix = 95, 64 * 96
    v, w = nonfinite_cube(npix, C)
    p = np.arange(npix)
    seen = set(zip(((p // C) % len(NONFINITE_CASES)).tolist(), (p % C).tolist()))
    assert seen == {(k, c) for k in range(len(NONFINITE_CASES)) for c in range(C)}
    with np.errstate(all="ignore"):
        want = (v.astype(np.float64) / w.astype(np.float64)).sum(axis=1)
        pf = v * (np.float32(1) / w)                                     # the float32 product v * r0
        q = v.astype(np.float64) / w
    assert np.any(np.isposinf(want)) and np.any(np.isneginf(want)) and np.any(np.isnan(want)) and np.any(np.isfinite(want))
    assert np.any(np.isinf(pf) & np.isfinite(q))                         # v * r0 overflows, the quotient does not
    assert np.any((w != 0) & (np.abs(w) < np.finfo(np.float32).tiny))      # denormal divisors
    assert np.any((v != 0) & (np.abs(v) < np.finfo(np.float32).tiny))      # denormal numerators
    v, w = flushed_divisor_cube(1024, C)
    fw = (_u32(w) >> 23) & 0xff
    assert set(fw[p[:1024], p[:1024] % C].tolist()) == {253, 254} and np.all(w[p[:1024], p[:1024] % C] > 2.0 ** 126)


def test_range_generator():
    for kind in RANGE_KINDS:
        s = range_cube(kind, 640, 95).astype(np.float64).sum(axis=1)
        vmax, vmin, norm = range_reference(s)
        assert np.any(np.isnan(s)) == (kind != "inf")
        assert np.any(np.isposinf(s)) == (kind in ("inf", "nan_inf"))
        if kind == "all_nan":
            assert np.all(np.isnan(s)) and vmax == -np.inf and vmin == np.inf
        elif "inf" in kind:
            assert vmax == np.inf and np.any(norm == 0) and np.isnan(norm[np.isposinf(s)]).all()


@pytest.mark.parametrize("bits", [16, 8])
def test_raw_counts_generator(bits):
    u = raw_counts_cube(bits, 95)
    assert np.array_equal(np.sort(u.max(axis=1)[:1 << bits]), np.arange(1 << bits))
    assert np.all(np.count_nonzero(u, axis=1) <= 1) and u.shape[0] % 128 != 0


# ---- GPU ------------------------------------------------------------------------------------------------------------
# The K0 routes a flat-field quotient can take.  W = 1088 = 17 tiles of 64 pixels and W * C % 4 == 0, so every tile
# of the compiled layouts is on the fast path (div_rn_fast); the general kernel, an unaligned flat field (base
# 4 mod 16 bytes) and the ragged last tile of W = 1100 use __fdiv_rn.
K0_ROUTES = {
    "fixed95": dict(chans=CHANS95, W=1088, generic=False, offset=0),
    "fixed63": dict(chans=CHANS63, W=1088, generic=False, offset=0),
    "generic": dict(chans=CHANS95, W=1088, generic=True, offset=0),
    "unaligned_flat_field": dict(chans=CHANS95, W=1088, generic=False, offset=1),
    "ragged": dict(chans=CHANS95, W=1100, generic=False, offset=0),
}


def _set_generic(monkeypatch, on):
    if on:
        monkeypatch.setenv("HIPR_REGISTER_GENERIC", "1")
    else:
        monkeypatch.delenv("HIPR_REGISTER_GENERIC", raising=False)


def _k0_quotients(torch, monkeypatch, vf, wf, route, return_sums=False):
    """K0 on the flat pairs (vf, wf) (float32 CUDA tensors), zero shifts: the registered cube is the stacked v,
    so cube.ravel()[i] is K0's vf[i] / wf[i].  The pairs are padded with 1 / 1 to whole rows of the route's width."""
    import hipr_b200
    r = K0_ROUTES[route]
    C, W, N = sum(r["chans"]), r["W"], vf.numel()
    H = -(-N // (W * C))
    v = torch.ones(H * W * C, dtype=torch.float32, device="cuda")
    v[:N] = vf
    wbuf = torch.ones(H * W * C + r["offset"], dtype=torch.float32, device="cuda")
    wbuf[r["offset"]:r["offset"] + N] = wf
    w = wbuf[r["offset"]:].view(H, W, C)
    assert (w.data_ptr() % 16 != 0) == (r["offset"] != 0)
    v = v.view(H, W, C)
    edges = np.cumsum((0,) + r["chans"])
    stacks = [v[:, :, a:b].contiguous() for a, b in zip(edges[:-1], edges[1:])]
    del v
    _set_generic(monkeypatch, r["generic"])
    try:
        cube, s, mk = hipr_b200.register_stacks(stacks, None, calibration=w, return_cube=not return_sums)
    finally:
        _set_generic(monkeypatch, False)
    torch.cuda.synchronize()
    return (s, mk) if return_sums else cube.view(-1)[:N]


def _bit_diff(torch, got, want):
    """Indices where two float32 CUDA tensors differ as bit patterns (NaN compared by position only)."""
    bad = (got.view(torch.int32) != want.view(torch.int32)) & ~(torch.isnan(got) & torch.isnan(want))
    return torch.nonzero(bad).flatten()


def _report(torch, idx, vf, wf, got, want, limit=8):
    i = idx[:limit]
    rows = zip(vf[i].view(torch.int32).tolist(), wf[i].view(torch.int32).tolist(),
               got[i].view(torch.int32).tolist(), want[i].view(torch.int32).tolist())
    return "%d differ; first (v, w, got, want) bits: %s" % (
        idx.numel(), ", ".join("(%08x, %08x, %08x, %08x)" % tuple(x & 0xffffffff for x in t) for t in rows))


def _check_k0_routes(torch, monkeypatch, v, w):
    """Every K0 route equals numpy's float32 quotient bit for bit, and the routes equal each other."""
    with np.errstate(all="ignore"):
        want = torch.from_numpy(v / w).cuda()
    vf, wf = torch.from_numpy(v).cuda(), torch.from_numpy(w).cuda()
    failures, first = {}, None
    for route in K0_ROUTES:
        got = _k0_quotients(torch, monkeypatch, vf, wf, route)
        idx = _bit_diff(torch, got, want)
        if idx.numel():
            failures[route] = _report(torch, idx, vf, wf, got, want)
        if first is None:
            first = got.clone()
        elif not torch.equal(got.view(torch.int32), first.view(torch.int32)):
            failures[route + " vs " + next(iter(K0_ROUTES))] = _report(torch, _bit_diff(torch, got, first), vf, wf, got, first)
        del got
    assert not failures, failures


@pytest.mark.gpu
def test_k0_quotient_every_divisor_significand(torch_cuda, monkeypatch):
    """All 2^23 divisor significands x 10 numerators (83.9 M pairs, one call of 812 x 1088 x 95 per route)."""
    _check_k0_routes(torch_cuda, monkeypatch, *divisor_sweep())


@pytest.mark.gpu
def test_k0_quotient_every_numerator_significand(torch_cuda, monkeypatch):
    """All 2^23 numerator significands x 8 divisors (67.1 M pairs)."""
    _check_k0_routes(torch_cuda, monkeypatch, *numerator_sweep())


@pytest.mark.gpu
def test_k0_quotient_exponent_edges(torch_cuda, monkeypatch):
    """Both operands over the exponent fields either side of the fast quotient's range, zeros, denormals, inf, NaN."""
    _check_k0_routes(torch_cuda, monkeypatch, *exponent_edges())


def _one_term_dev(torch, v, w, C, offset=0, extra=0):
    """(npix + extra, C) CUDA cube and flat field: pixel p holds v[p] / w[p] at channel p mod C and 0 / 1 elsewhere
    (the `extra` pixels are 0 / 1).  offset > 0 starts both at `offset` floats into their buffers."""
    npix = v.numel()
    n = (npix + extra) * C
    cb = torch.zeros(n + offset, dtype=torch.float32, device="cuda")
    wb = torch.ones(n + offset, dtype=torch.float32, device="cuda")
    cube, cal = cb[offset:].view(npix + extra, C), wb[offset:].view(npix + extra, C)
    p = torch.arange(npix, device="cuda")
    cube[p, p % C] = v
    cal[p, p % C] = w
    return cube, cal


def _term_errors(got, want):
    return np.abs(got - want) / np.abs(want)


@pytest.mark.gpu
def test_flat_field_sum_terms_every_divisor_significand(torch_cuda, monkeypatch):
    """One non-zero term per pixel, at every channel position in turn: the pixel's sum is that term's quotient.
    All 2^23 divisor significands, within TERM_RTOL of numpy's float64 quotient through K1 (bulk path, two threads
    per pixel) and K0 (fixed layout and general kernel, four threads per pixel)."""
    import hipr_b200
    torch = torch_cuda
    v, w = term_divisor_sweep()
    want = v.astype(np.float64) / w.astype(np.float64)
    C, chunk = 95, 1 << 20
    worst = {}
    for k in range(0, NSIG, chunk):
        vd, wd = torch.from_numpy(v[k:k + chunk]).cuda(), torch.from_numpy(w[k:k + chunk]).cuda()
        cube, cal = _one_term_dev(torch, vd, wd, C)
        got = {"K1": hipr_b200.channel_sum(cube, cal, normalize=False, dtype=torch.float64)}
        stacks = [cube[:, a:b].contiguous().view(1024, chunk // 1024, b - a)
                  for a, b in zip(np.cumsum((0,) + CHANS95)[:-1], np.cumsum(CHANS95))]
        cal3 = cal.view(1024, chunk // 1024, C)
        for name, generic in (("K0 fixed", False), ("K0 general", True)):
            _set_generic(monkeypatch, generic)
            got[name] = hipr_b200.register_stacks(stacks, None, calibration=cal3, return_cube=False)[1].view(-1)
        _set_generic(monkeypatch, False)
        for name, g in got.items():
            err = _term_errors(g.cpu().numpy(), want[k:k + chunk])
            worst[name] = max(worst.get(name, 0.0), float(err.max()))
        del cube, cal, stacks, cal3, got
    assert all(e <= TERM_RTOL for e in worst.values()), (worst, TERM_RTOL)


def _k1_routes(torch, v, w):
    """K1 flat-field sums of (npix, C) host arrays through the bulk path (16-byte aligned, whole 64-pixel chunks
    plus a ragged remainder for the warp kernel) and through the warp kernel alone (bases 4 bytes off)."""
    import hipr_b200
    out = {}
    for name, off in (("K1 bulk + tail", 0), ("K1 unaligned", 1)):
        n = v.size
        cb = torch.empty(n + off, dtype=torch.float32, device="cuda")
        wb = torch.empty(n + off, dtype=torch.float32, device="cuda")
        cb[off:] = torch.from_numpy(v.ravel()).cuda()
        wb[off:] = torch.from_numpy(w.ravel()).cuda()
        cube, cal = cb[off:].view(v.shape), wb[off:].view(w.shape)
        out[name] = hipr_b200.channel_sum(cube, cal, normalize=False, dtype=torch.float64, return_max=True)
    return out


def _k0_sum_routes(torch, monkeypatch, v, w):
    """K0 flat-field sums of (H, W, 95) host arrays: fixed layout and general kernel."""
    import hipr_b200
    edges = np.cumsum((0,) + CHANS95)
    stacks = [torch.from_numpy(np.ascontiguousarray(v[:, :, a:b])).cuda() for a, b in zip(edges[:-1], edges[1:])]
    cal = torch.from_numpy(w).cuda()
    out = {}
    for name, generic in (("K0 fixed", False), ("K0 general", True)):
        _set_generic(monkeypatch, generic)
        _, s, mk = hipr_b200.register_stacks(stacks, None, calibration=cal, return_cube=False)
        out[name] = (s, mk)
    _set_generic(monkeypatch, False)
    return out


def _check_sums(got, want, rtol, what):
    """Finite sums within rtol of numpy's; non-finite ones equal (NaN by position, infinities with their sign)."""
    fin = np.isfinite(want)
    bad_nf = ~fin & ~((np.isnan(want) & np.isnan(got)) | (want == got))
    assert not bad_nf.any(), "%s: %d non-finite sums differ, first at %s: got %r want %r" % (
        what, bad_nf.sum(), np.argwhere(bad_nf)[0], got[bad_nf][0], want[bad_nf][0])
    with np.errstate(all="ignore"):
        err = np.where(want == 0, np.where(got == 0, 0.0, np.inf), np.abs(got - want) / np.abs(want))
        err = np.where(fin, err, 0.0)
    bad = fin & ~(err <= rtol)
    assert not bad.any(), "%s: %d sums outside rtol %g, worst %.3g at %s (got %r want %r)" % (
        what, bad.sum(), rtol, np.nanmax(np.where(bad, err, 0)), np.argwhere(bad)[0], got[bad][0], want[bad][0])


def _check_range(got_s, mk, what):
    vmax, vmin, _ = range_reference(got_s)
    gmax, gmin = (float(x) for x in mk.values())
    assert gmax == vmax and gmin == vmin, (what, gmax, gmin, vmax, vmin)


@pytest.mark.gpu
def test_flat_field_sums_wide_range(torch_cuda, monkeypatch):
    """Positive numerators with per-pixel binades 2^-126 .. 2^125 and a row of denormal numerators: whole-pixel sums
    within SUM_RTOL of numpy's float64 sums on every K1 and K0 route."""
    torch = torch_cuda
    H, W = 96, 192
    v, w = wide_range_cube(H, W, 95)
    want = (v.astype(np.float64) / w.astype(np.float64)).sum(axis=-1)
    # the K1 calls leave out the last 5 pixels: a ragged remainder after the 64-pixel chunks
    got = dict(_k1_routes(torch, v.reshape(-1, 95)[:-5], w.reshape(-1, 95)[:-5]))
    got.update(_k0_sum_routes(torch, monkeypatch, v, w))
    for name, (s, mk) in got.items():
        s = s.cpu().numpy().ravel()
        _check_sums(s, want.ravel()[:s.size], SUM_RTOL, name)
        _check_range(s, mk, name)


@pytest.mark.gpu
def test_flat_field_sums_nonfinite(torch_cuda, monkeypatch):
    """Zero, denormal, infinite and NaN divisors, infinite / NaN / denormal numerators and numerators whose float32
    product v * r0 overflows, each at every channel position: sums equal numpy's where numpy's are not finite
    (the exact float64 fallback of each half pixel in K1 and each quarter in K0), within SUM_RTOL elsewhere."""
    torch = torch_cuda
    C, H, W = 95, 64, 96
    v, w = nonfinite_cube(H * W, C)
    with np.errstate(all="ignore"):
        want = (v.astype(np.float64) / w.astype(np.float64)).sum(axis=-1)
    got = dict(_k1_routes(torch, v[:-7], w[:-7]))
    got.update(_k0_sum_routes(torch, monkeypatch, v.reshape(H, W, C), w.reshape(H, W, C)))
    for name, (s, mk) in got.items():
        s = s.cpu().numpy().ravel()
        _check_sums(s, want[:s.size], SUM_RTOL, name)
        _check_range(s, mk, name)


@pytest.mark.gpu
def test_flat_field_sums_flush_divisors_above_2_126(torch_cuda, monkeypatch):
    """Documented deviation (hipr_common.cuh, DESIGN.md section 3 K1): a divisor above 2^126 has its float32
    reciprocal flushed to zero, so on the K1 bulk path and in K0 its term counts as 0.  The K1 warp kernel divides in
    float64 and keeps the term."""
    torch = torch_cuda
    C, H, W = 95, 64, 96
    v, w = flushed_divisor_cube(H * W, C)
    q = v.astype(np.float64) / w.astype(np.float64)
    p = np.arange(H * W)
    exact = q.sum(axis=-1)
    q[p, p % C] = 0.0
    flushed = q.sum(axis=-1)
    assert np.all(flushed < exact)
    k1 = _k1_routes(torch, v, w)
    _check_sums(k1["K1 bulk + tail"][0].cpu().numpy(), flushed, SUM_RTOL, "K1 bulk")
    _check_sums(k1["K1 unaligned"][0].cpu().numpy(), exact, SUM_RTOL, "K1 warp kernel")
    for name, (s, _) in _k0_sum_routes(torch, monkeypatch, v.reshape(H, W, C), w.reshape(H, W, C)).items():
        _check_sums(s.cpu().numpy().ravel(), flushed, SUM_RTOL, name)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", RANGE_KINDS)
def test_range_keys_with_nonfinite_sums(torch_cuda, monkeypatch, kind):
    """The max / min keys skip NaN sums (DESIGN.md section 2) on every entry point: K1 bulk and warp kernel,
    K0 fixed layout and general kernel, without and with a flat field; normalize=True divides by that max."""
    import hipr_b200
    torch = torch_cuda
    C, H, W = 95, 40, 128
    v = range_cube(kind, H * W, C)
    want = v.astype(np.float64).sum(axis=-1)
    vmax, vmin, want_norm = range_reference(want)
    ones = np.ones_like(v)
    runs = {}
    for flat in (False, True):
        for name, off in (("K1 bulk", 0), ("K1 unaligned", 1)):
            buf = torch.empty(v.size + off, dtype=torch.float32, device="cuda")
            buf[off:] = torch.from_numpy(v.ravel()).cuda()
            cube = buf[off:].view(H * W, C)
            cal = torch.ones_like(cube) if flat else None
            s, mk = hipr_b200.channel_sum(cube, cal, normalize=False, dtype=torch.float64, return_max=True)
            norm = hipr_b200.channel_sum(cube, cal, normalize=True, dtype=torch.float64)
            runs["%s%s" % (name, " flat" if flat else "")] = (s, mk, norm)
        edges = np.cumsum((0,) + CHANS95)
        stacks = [torch.from_numpy(np.ascontiguousarray(v.reshape(H, W, C)[:, :, a:b])).cuda()
                  for a, b in zip(edges[:-1], edges[1:])]
        for name, generic in (("K0 fixed", False), ("K0 general", True)):
            _set_generic(monkeypatch, generic)
            _, s, mk = hipr_b200.register_stacks(stacks, None, calibration=torch.from_numpy(ones).cuda().view(H, W, C)
                                                 if flat else None, return_cube=False)
            runs["%s%s" % (name, " flat" if flat else "")] = (s, mk, None)
        _set_generic(monkeypatch, False)
    for name, (s, mk, norm) in runs.items():
        s = s.cpu().numpy().ravel()
        _check_sums(s, want, 1e-14, name)
        gmax, gmin = (float(x) for x in mk.values())
        assert gmax == vmax and gmin == vmin, (name, gmax, gmin, vmax, vmin)
        if norm is not None:
            _check_sums(norm.cpu().numpy().ravel(), want_norm, 2e-14, name + " normalize")


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [16, 8])
@pytest.mark.parametrize("scale", RAW_SCALES)
def test_raw_counts_every_count(torch_cuda, bits, scale):
    """Every uint16 / uint8 count, one per pixel at every channel position: the float64 sum is that sample's
    float32(count) / float32(scale), bit for bit, through the bulk path + ragged tail and through the warp kernel
    alone (a base 2 bytes off 16)."""
    import hipr_b200
    torch = torch_cuda
    C = 95
    u = raw_counts_cube(bits, C)
    want = (u.astype(np.float32) / np.float32(scale)).astype(np.float64).sum(axis=1)
    tdt = torch.int16 if bits > 8 else torch.uint8
    for off in (0, 1):
        buf = torch.zeros(u.size + off, dtype=tdt, device="cuda")
        buf[off:] = torch.from_numpy(u.ravel().view(np.int16) if bits > 8 else u.ravel()).cuda()
        got, mk = hipr_b200.channel_sum_raw(buf[off:].view(u.shape), scale, return_max=True)
        got = got.cpu().numpy()
        bad = got.view(np.uint64) != want.view(np.uint64)
        assert not bad.any(), (off, int(bad.sum()), u[bad].max(axis=1)[:8], got[bad][:8], want[bad][:8])
        assert float(mk.value()) == want.max()
