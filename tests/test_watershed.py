"""CPU checks of the marker watershed (K11): the rule of tests/watershed_oracle.py against the heap restatement of
scikit-image's flood on tie-free inputs, against the three relaxations of the kernel's design on any input, hand-built
tie cases, and the argument checks of ops.watershed and the C entry points (no device call)."""
import ctypes as C

import numpy as np
import pytest

import watershed_oracle as wo


# ---- a second formulation: the kernel's three minimum relaxations, Jacobi sweeps in numpy until nothing changes ----

def _shifted(a, ndim, connectivity, fill):
    """For every neighbour offset: the padded array read at that offset, cut to the image."""
    p = np.pad(a, 1, constant_values=fill)
    out = []
    for d in wo.offsets(ndim, connectivity):
        out.append(p[tuple(slice(1 + k, s - 1 + k) for k, s in zip(d, p.shape))])
    return out


def relax_rule(image, markers, connectivity=1, mask=None):
    image = np.asarray(image, np.float64) + 0.0
    inside = np.ones(image.shape, bool) if mask is None else np.asarray(mask).astype(bool)
    markers = np.asarray(markers) * inside
    is_m = markers != 0
    nd = image.ndim
    # phase 1: L = max(v, min L over neighbours), markers fixed at v
    L = np.where(is_m, image, np.inf)
    while True:
        ml = np.min(_shifted(L, nd, connectivity, np.inf), axis=0)
        new = np.where(is_m, image, np.where(inside, np.maximum(image, ml), np.inf))
        if np.array_equal(new, L):
            break
        L = new
    reached = np.isfinite(L)
    # phase 2: candidates = neighbours of minimal L; markers 0, entries 1, else 1 + min d over candidates
    sl = _shifted(L, nd, connectivity, np.inf)
    ml = np.min(sl, axis=0)
    cand = [s == ml for s in sl]
    entry = reached & ~is_m & (L > ml)
    fixed = is_m | entry | ~reached
    big = np.iinfo(np.int64).max // 4
    D = np.where(is_m, 0, np.where(entry, 1, big))
    while True:
        sd = _shifted(D, nd, connectivity, big)
        md = np.min([np.where(c, s, big) for c, s in zip(cand, sd)], axis=0)
        new = np.where(fixed, D, np.minimum(D, md + 1))
        if np.array_equal(new, D):
            break
        D = new
    # phase 3: parents = candidates of minimal d; label = min label over the parents
    sd = _shifted(D, nd, connectivity, big)
    md = np.min([np.where(c, s, big) for c, s in zip(cand, sd)], axis=0)
    par = [c & (s == md) for c, s in zip(cand, sd)]
    lab = np.where(is_m, markers.astype(np.int64), big)
    while True:
        sl3 = _shifted(lab, nd, connectivity, big)
        mlab = np.min([np.where(p, s, big) for p, s in zip(par, sl3)], axis=0)
        new = np.where(is_m | ~reached, lab, np.minimum(lab, mlab))
        if np.array_equal(new, lab):
            break
        lab = new
    return np.where(reached, lab, 0).astype(markers.dtype)


# ---- inputs ------------------------------------------------------------------------------------------------------

def random_case(shape, seed, values="continuous", n_markers=6, masked=True, dtype=np.int32):
    rng = np.random.default_rng(seed)
    if values == "continuous":
        image = rng.standard_normal(shape)
    elif values == "uint8":
        image = rng.integers(0, 6, shape).astype(np.float64)
    else:                                                               # plateaus: blocks of equal value
        image = np.kron(rng.integers(0, 3, tuple((s + 3) // 4 for s in shape)), np.ones((4,) * len(shape)))
        image = image[tuple(slice(0, s) for s in shape)].astype(np.float64)
    markers = np.zeros(shape, dtype)
    npix = int(np.prod(shape))
    idx = rng.choice(npix, size=min(n_markers, npix), replace=False)
    markers.ravel()[idx] = rng.permutation(np.r_[np.arange(1, len(idx) // 2 + 1), -np.arange(1, len(idx) - len(idx) // 2 + 1)])
    mask = rng.random(shape) < 0.8 if masked else None
    return image, markers, mask


CASES = [((23, 31), 1), ((23, 31), 2), ((1, 40), 1), ((40, 1), 2), ((9, 10, 11), 1), ((9, 10, 11), 2),
         ((9, 10, 11), 3), ((1, 12, 13), 3), ((14, 1, 1), 3)]


@pytest.mark.parametrize("shape,conn", CASES)
def test_rule_equals_heap_without_ties(shape, conn):
    checked = 0
    for seed in range(12):
        image, markers, mask = random_case(shape, 1000 * conn + seed, masked=seed % 3 != 0,
                                           dtype=np.int64 if seed % 2 else np.int32)
        heap = wo.watershed_heap(image, markers, conn, mask)
        assert not heap.tied.any()                                    # continuous values: no tie decides a pixel
        rule = wo.watershed_rule(image, markers, conn, mask)
        assert rule.dtype == markers.dtype
        assert np.array_equal(rule, heap.labels)
        checked += 1
        if mask is not None:
            assert not heap.labels[~mask].any()                       # outside the mask (markers there dropped)
    assert checked == 12


def test_rule_equals_heap_with_unreachable_regions_and_markers_outside_the_mask():
    rng = np.random.default_rng(5)
    image = rng.random((30, 30))
    mask = np.ones((30, 30), bool)
    mask[:, 14:16] = False                                            # two halves, markers only in the left one
    markers = np.zeros((30, 30), np.int32)
    markers[3, 3], markers[20, 9], markers[10, 15] = 4, -2, 7         # (10, 15) lies outside the mask
    heap = wo.watershed_heap(image, markers, 1, mask)
    assert not heap.tied.any()
    rule = wo.watershed_rule(image, markers, 1, mask)
    assert np.array_equal(rule, heap.labels)
    assert not rule[:, 14:].any() and set(np.unique(rule[:, :14])) == {-2, 4}


@pytest.mark.parametrize("values", ["continuous", "uint8", "plateau"])
@pytest.mark.parametrize("shape,conn", CASES)
def test_rule_equals_the_three_relaxations(shape, conn, values):
    for seed in range(6):
        image, markers, mask = random_case(shape, 7 * seed + conn, values, n_markers=2 + seed,
                                           masked=seed % 2 == 1)
        if seed == 5:
            markers[...] = 0                                          # no markers at all
        got = wo.watershed_rule(image, markers, conn, mask)
        assert np.array_equal(got, relax_rule(image, markers, conn, mask)), (values, seed)


def test_levels_order_the_pops_and_popper_is_a_neighbour():
    image, markers, mask = random_case((20, 24), 3, "uint8", n_markers=5)
    heap = wo.watershed_heap(image, markers, 2, mask)
    lab = heap.labels.ravel()
    for p in np.flatnonzero(heap.popper.ravel() >= 0):
        q = heap.popper.ravel()[p]
        a, b = np.unravel_index(p, image.shape), np.unravel_index(q, image.shape)
        assert max(abs(i - j) for i, j in zip(a, b)) == 1
        assert lab[p] == lab[q]
        assert heap.level.ravel()[p] >= heap.level.ravel()[q]


# ---- hand-built ties --------------------------------------------------------------------------------------------

def test_plateau_between_two_markers_is_split_by_age_in_the_heap():
    # marker 2 (value 0) on the left, marker 1 (value 0.5) on the right, a plateau of 1s between them.  The heap pops
    # the left marker first, so (0, 1) gets the smaller age and its pop labels the middle pixel 2.  The rule prefers
    # the smaller label among the two equal keys (1, 1, .).
    image = np.array([[0.0, 1.0, 1.0, 1.0, 0.5]])
    markers = np.array([[2, 0, 0, 0, 1]], np.int32)
    heap = wo.watershed_heap(image, markers)
    assert heap.labels.tolist() == [[2, 2, 2, 1, 1]]
    assert heap.tied.tolist() == [[False, False, True, False, False]]
    assert heap.popper.tolist() == [[-1, 0, 1, 4, -1]]
    assert heap.level.tolist() == [[0.0, 1.0, 1.0, 1.0, 0.5]]
    assert wo.watershed_rule(image, markers).tolist() == [[2, 2, 1, 1, 1]]
    assert relax_rule(image, markers).tolist() == [[2, 2, 1, 1, 1]]


def test_equal_valued_markers():
    image = np.zeros((1, 3))
    markers = np.array([[3, 0, 1]], np.int64)
    heap = wo.watershed_heap(image, markers)
    assert heap.labels.tolist() == [[3, 3, 1]]                        # index order of the equal markers
    assert heap.tied.tolist() == [[False, True, False]]
    assert wo.watershed_rule(image, markers).tolist() == [[3, 1, 1]]  # the smaller label


def test_signed_zeros_are_one_level():
    image = np.array([[-0.0, 0.0, 0.0]])
    markers = np.array([[2, 0, 1]], np.int32)
    heap = wo.watershed_heap(image, markers)
    assert heap.tied.tolist() == [[False, True, False]]               # -0.0 == +0.0 for the heap
    assert heap.labels.tolist() == [[2, 2, 1]]
    assert wo.watershed_rule(image, markers).tolist() == [[2, 1, 1]]  # not -0.0 < +0.0, which would give 2
    assert relax_rule(image, markers).tolist() == [[2, 1, 1]]


def test_a_marker_prefers_itself_then_fewer_hops():
    # on one plateau, (0, 3) is 3 hops from marker 1 and 2 from marker 5: fewer hops win over the smaller label
    image = np.zeros((1, 6))
    markers = np.array([[1, 0, 0, 0, 0, 5]], np.int32)
    assert wo.watershed_rule(image, markers).tolist() == [[1, 1, 1, 5, 5, 5]]
    assert relax_rule(image, markers).tolist() == [[1, 1, 1, 5, 5, 5]]


# ---- ops.watershed refuses CPU tensors and bad arguments -----------------------------------------------------------

def test_watershed_has_no_cpu_path():
    import torch
    import hipr_b200
    img = torch.zeros(8, 8)
    mk = torch.zeros(8, 8, dtype=torch.int32)
    with pytest.raises(ValueError, match="no CPU path"):
        hipr_b200.watershed(img, mk)
    with pytest.raises(TypeError):
        hipr_b200.watershed(np.zeros((8, 8)), np.zeros((8, 8), np.int32))


def test_watershed_argument_checks(monkeypatch):
    """The Python-side checks run before any device call: a CUDA-looking tensor is faked so they can be reached
    without a GPU."""
    import torch
    import hipr_b200
    from hipr_b200 import ops

    monkeypatch.setattr(ops, "_dev", lambda t, name, dtypes=(): (_ for _ in ()).throw(TypeError(name))
                        if t.dtype not in dtypes else t)
    img = torch.zeros(8, 9)
    mk = torch.zeros(8, 9, dtype=torch.int32)
    with pytest.raises(TypeError, match="image"):
        hipr_b200.watershed(img.half(), mk)
    with pytest.raises(TypeError, match="markers"):
        hipr_b200.watershed(img, mk.float())
    with pytest.raises(TypeError, match="markers"):
        hipr_b200.watershed(img, mk.to(torch.int16))
    with pytest.raises(TypeError, match="mask"):
        hipr_b200.watershed(img, mk, mask=torch.zeros(8, 9, dtype=torch.int32))
    with pytest.raises(ValueError, match="differ in shape"):
        hipr_b200.watershed(img, torch.zeros(9, 8, dtype=torch.int32))
    with pytest.raises(ValueError, match="differ in shape"):
        hipr_b200.watershed(img, mk, mask=torch.zeros(8, 8, dtype=torch.bool))
    with pytest.raises(ValueError, match="2-D image or a 3-D volume"):
        hipr_b200.watershed(torch.zeros(9), torch.zeros(9, dtype=torch.int32))
    with pytest.raises(ValueError, match="2-D image or a 3-D volume"):
        hipr_b200.watershed(torch.zeros(2, 2, 2, 2), torch.zeros(2, 2, 2, 2, dtype=torch.int32))
    with pytest.raises(ValueError, match="empty"):
        hipr_b200.watershed(torch.zeros(0, 4), torch.zeros(0, 4, dtype=torch.int32))
    with pytest.raises(ValueError, match="connectivity"):
        hipr_b200.watershed(img, mk, connectivity=3)
    with pytest.raises(ValueError, match="connectivity"):
        hipr_b200.watershed(torch.zeros(3, 4, 5), torch.zeros(3, 4, 5, dtype=torch.int32), connectivity=0)
    with pytest.raises(TypeError, match="connectivity"):
        hipr_b200.watershed(img, mk, connectivity=1.5)


def test_watershed_entry_points_argument_checks():
    import hipr_b200
    lib = hipr_b200.lib()
    buf = (C.c_char * 64)()
    p = C.cast(buf, C.c_void_p)
    # control block, 6 dirty flags per 64 x 64 tile, 8-byte level / label words, 4-byte hop and neighbour-mask words
    assert lib.hipr_watershed_workspace_bytes(2, 2048, 2048, 0, 0, 4) == 256 + 1024 * 24 + 2048 * 2048 * 16
    assert lib.hipr_watershed_workspace_bytes(3, 3, 5, 7, 1, 8) == 256 + 256 + 1024 + 2 * 512   # 105 pixels
    assert lib.hipr_watershed_workspace_bytes(3, 1024, 1024, 2048, 0, 4) == -7   # 2^31 pixels: HIPR_E_RANGE
    assert lib.hipr_watershed_workspace_bytes(2, 46341, 46341, 0, 0, 4) == -7
    assert lib.hipr_watershed_workspace_bytes(4, 2, 2, 2, 0, 4) == -1
    assert lib.hipr_watershed_workspace_bytes(2, 0, 5, 0, 0, 4) == -1
    assert lib.hipr_watershed_workspace_bytes(2, 4, 4, 0, 2, 4) == -2            # integer image
    assert lib.hipr_watershed_workspace_bytes(2, 4, 4, 0, 0, 2) == -2            # int16 markers
    ws = lib.hipr_watershed_workspace_bytes(2, 4, 4, 0, 0, 4)
    args = [p, 0, p, 4, None, 2, 4, 4, 0, 1, p, ws, p, p, None]
    for k in (0, 2, 10, 12, 13):                                                  # null pointers
        bad = list(args)
        bad[k] = None
        assert lib.hipr_watershed(*bad) == -1
    for k, v, code in ((9, 3, -1), (9, 0, -1), (5, 4, -1), (1, 3, -2), (3, 2, -2), (11, ws - 1, -7)):
        bad = list(args)
        bad[k] = v
        assert lib.hipr_watershed(*bad) == code, (k, v)
