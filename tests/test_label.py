"""CPU checks of the connected-component operators (K10): restatements in tests/label_oracle.py against a brute-force
union-find, and the argument checks of the device operators and the C entry points (no device call)."""
import ctypes as C
import itertools

import numpy as np
import pytest

import label_oracle

SHAPES = [(1, 1), (1, 17), (17, 1), (9, 13), (24, 31), (1, 7, 9), (5, 6, 1), (6, 7, 8)]


def _offsets(ndim, connectivity):
    return [d for d in itertools.product((-1, 0, 1), repeat=ndim) if 0 < sum(map(abs, d)) <= connectivity]


def brute_label(image, connectivity, mask):
    """Union-find over pixels: neighbours at city-block distance <= connectivity (one step per axis) join when
    both are non-zero (mask) or equal and non-zero; components numbered by first pixel in raster order."""
    image = np.asarray(image)
    flat = image.ravel()
    parent = list(range(flat.size))

    def find(a):
        while parent[a] != a:
            a = parent[a]
        return a

    for p in np.ndindex(image.shape):
        if image[p] == 0:
            continue
        for d in _offsets(image.ndim, connectivity):
            q = tuple(a + b for a, b in zip(p, d))
            if all(0 <= c < s for c, s in zip(q, image.shape)) and image[q] != 0 and (mask or image[q] == image[p]):
                ra, rb = find(np.ravel_multi_index(p, image.shape)), find(np.ravel_multi_index(q, image.shape))
                parent[max(ra, rb)] = min(ra, rb)
    out = np.zeros(flat.size, np.int32)
    names = {}
    for i in range(flat.size):
        if flat[i] != 0:
            out[i] = names.setdefault(find(i), len(names) + 1)
    return out.reshape(image.shape), len(names)


def _inputs(shape, seed):
    rng = np.random.default_rng(seed)
    yield rng.random(shape) < 0.45                                       # mask
    yield rng.integers(-2, 3, shape).astype(np.int32)                    # touching regions, negative values too
    blocks = np.kron(rng.integers(0, 4, (shape[0] // 2 + 1,) + shape[1:]), np.ones((2,) + (1,) * (len(shape) - 1)))
    yield blocks[:shape[0]].astype(np.int64)                             # larger equal-valued regions that touch


@pytest.mark.parametrize("shape", SHAPES)
def test_restatement_matches_brute_force_union_find(shape):
    for conn in range(1, len(shape) + 1):
        for k, image in enumerate(_inputs(shape, seed=len(shape) * 100 + sum(shape))):
            if image.dtype == bool:
                got, n = label_oracle.label_mask(image, conn)
            else:
                got, n = label_oracle.label_image(image, conn)
            want, wn = brute_label(image, conn, mask=image.dtype == bool)
            assert n == wn and np.array_equal(got, want), (shape, conn, k)


def test_label_image_separates_touching_values():
    image = np.array([[1, 1, 2, 2],
                      [1, 3, 3, 2],
                      [0, 3, -1, -1],
                      [5, 0, -1, 7]], np.int32)
    lab, n = label_oracle.label_image(image, 1)
    assert n == 6
    assert np.array_equal(lab, [[1, 1, 2, 2], [1, 3, 3, 2], [0, 3, 4, 4], [5, 0, 4, 6]])
    lab2, n2 = label_oracle.label_image(image, 2)                    # diagonal neighbours all differ in value
    assert n2 == 6 and np.array_equal(lab2, lab)


def _brute_clear_border(image, buffer_size, bgval):
    lab, n = brute_label(image, image.ndim, mask=image.dtype == bool)
    edge = set()
    for p in np.ndindex(image.shape):
        if any(c <= buffer_size or c >= s - 1 - buffer_size for c, s in zip(p, image.shape)):
            edge.add(lab[p])
    out = image.copy()
    for p in np.ndindex(image.shape):
        if lab[p] in edge:
            out[p] = bgval
    return out


@pytest.mark.parametrize("shape", [(12, 15), (7, 8, 9), (1, 9)])
def test_clear_border_restatement(shape):
    for k, image in enumerate(_inputs(shape, seed=7)):
        for buffer_size in range(0, min(shape)):
            for bgval in (0, 9):
                if image.dtype == bool and bgval:
                    continue
                got = label_oracle.clear_border(image, buffer_size, bgval)
                assert np.array_equal(got, _brute_clear_border(image, buffer_size, bgval)), (k, buffer_size, bgval)
    with pytest.raises(ValueError, match="buffer size"):
        label_oracle.clear_border(np.zeros(shape, np.int32), min(shape))


def test_clear_border_sets_touching_background_to_bgval():
    image = np.zeros((6, 6), np.int32)
    image[2:4, 2:4] = 3
    out = label_oracle.clear_border(image, 0, 5)
    assert (out[image == 0] == 5).all() and (out[2:4, 2:4] == 3).all()


@pytest.mark.parametrize("shape", [(20, 23), (6, 7, 8)])
def test_remove_small_objects_restatement(shape):
    rng = np.random.default_rng(3)
    mask = rng.random(shape) < 0.4
    labels = rng.integers(0, 40, shape).astype(np.int64)
    for min_size in (0, 1, 2, 3, 5, 12):
        for conn in range(1, len(shape) + 1):
            lab, n = brute_label(mask, conn, mask=True)
            sizes = np.bincount(lab.ravel(), minlength=n + 1)
            want = mask & (sizes[lab] >= min_size)
            assert np.array_equal(label_oracle.remove_small_objects_mask(mask, min_size, conn), want)
        want = np.where(np.bincount(labels.ravel())[labels] >= min_size, labels, 0) if min_size else labels
        assert np.array_equal(label_oracle.remove_small_objects_labels(labels, min_size), want)
    with pytest.raises(ValueError):
        label_oracle.remove_small_objects_labels(labels - 1, 3)


def test_relabel_sequential_restatement():
    labels = np.array([[0, 5, 5], [9, 0, 2], [9, 9, 40]], np.int32)
    out, fw, inv = label_oracle.relabel_sequential(labels, offset=3)
    assert np.array_equal(out, [[0, 4, 4], [5, 0, 3], [5, 5, 6]])
    assert fw.shape == (41,) and fw[5] == 4 and fw[40] == 6 and fw[0] == 0 and fw[7] == 0
    assert np.array_equal(inv, [0, 0, 0, 2, 5, 9, 40])
    assert np.array_equal(fw[labels], out) and np.array_equal(inv[out], labels)
    with pytest.raises(ValueError):
        label_oracle.relabel_sequential(labels, 0)
    with pytest.raises(ValueError):
        label_oracle.relabel_sequential(labels - 1)


def test_fill_holes_is_background_components_off_the_edge():
    rng = np.random.default_rng(11)
    for shape in ((40, 37), (9, 10, 11)):
        for conn in range(1, len(shape) + 1):
            mask = rng.random(shape) < 0.55
            bg, n = brute_label(~mask, conn, mask=True)
            edge = np.zeros(n + 1, bool)
            for p in np.ndindex(shape):
                if any(c == 0 or c == s - 1 for c, s in zip(p, shape)):
                    edge[bg[p]] = True
            want = mask | ((bg > 0) & ~edge[bg])
            assert np.array_equal(label_oracle.binary_fill_holes(mask, conn), want)


# ---- the device operators refuse CPU tensors and bad arguments ----------------------------------------------------

def _ops():
    import torch
    import hipr_b200
    return torch, hipr_b200


def test_label_operators_have_no_cpu_path():
    torch, h = _ops()
    m = torch.zeros(8, 8, dtype=torch.bool)
    lab = torch.zeros(8, 8, dtype=torch.int32)
    for call in (lambda: h.label(m), lambda: h.remove_small_objects(m), lambda: h.binary_fill_holes(m),
                 lambda: h.clear_border(lab), lambda: h.relabel_sequential(lab),
                 lambda: h.paint_labels(lab, torch.zeros(3, dtype=torch.int64))):
        with pytest.raises(ValueError, match="no CPU path"):
            call()
    with pytest.raises(TypeError):
        h.label(np.zeros((8, 8), bool))


def test_label_operator_argument_checks(monkeypatch):
    """The Python-side checks run before any device call: a CUDA-looking tensor is faked so they can be reached
    without a GPU."""
    torch, h = _ops()
    from hipr_b200 import ops

    monkeypatch.setattr(ops, "_dev", lambda t, name, dtypes=(): (_ for _ in ()).throw(TypeError(name))
                        if t.dtype not in dtypes else t)
    m2 = torch.zeros(8, 9, dtype=torch.bool)
    m3 = torch.zeros(4, 5, 6, dtype=torch.bool)
    with pytest.raises(ValueError, match="connectivity"):
        h.label(m2, connectivity=3)
    with pytest.raises(ValueError, match="connectivity"):
        h.label(m3, connectivity=0)
    with pytest.raises(TypeError, match="connectivity"):
        h.label(m3, connectivity=1.5)
    with pytest.raises(TypeError, match="dtype"):
        h.label(m2, dtype=torch.float32)
    with pytest.raises(ValueError, match="2-D image or a 3-D volume"):
        h.label(torch.zeros(9, dtype=torch.bool))
    with pytest.raises(ValueError, match="2-D image or a 3-D volume"):
        h.binary_fill_holes(torch.zeros(2, 3, 4, 5, dtype=torch.bool))
    with pytest.raises(ValueError, match="empty"):
        h.label(torch.zeros(0, 4, dtype=torch.bool))
    with pytest.raises(TypeError):
        h.label(torch.zeros(4, 4))                                        # float: not a mask or label image
    with pytest.raises(TypeError):
        h.remove_small_objects(torch.zeros(4, 4, dtype=torch.uint8))
    with pytest.raises(ValueError, match="buffer size"):
        h.clear_border(torch.zeros(8, 9, dtype=torch.int32), buffer_size=8)
    with pytest.raises(ValueError, match="buffer_size"):
        h.clear_border(torch.zeros(8, 9, dtype=torch.int32), buffer_size=-1)
    with pytest.raises(ValueError, match="bgval"):
        h.clear_border(torch.zeros(8, 9, dtype=torch.int32), bgval=2 ** 31)
    with pytest.raises(ValueError, match="Offset"):
        h.relabel_sequential(torch.zeros(8, 9, dtype=torch.int32), offset=0)
    with pytest.raises(TypeError):
        h.relabel_sequential(m2)


def test_label_entry_points_argument_checks():
    import hipr_b200
    lib = hipr_b200.lib()
    buf = (C.c_char * 64)()
    p = C.cast(buf, C.c_void_p)
    # parent array (int32 per pixel) + one int32 per 4096-pixel chunk, each rounded up to 256 bytes
    assert lib.hipr_label_workspace_bytes(2, 2048, 2048, 0) == 2048 * 2048 * 4 + 1024 * 4
    assert lib.hipr_label_workspace_bytes(3, 3, 5, 7) == 512 + 256
    assert lib.hipr_label_workspace_bytes(3, 1024, 1024, 2048) == -7       # 2^31 pixels: HIPR_E_RANGE
    assert lib.hipr_label_workspace_bytes(2, 46341, 46341, 0) == -7
    assert lib.hipr_label_workspace_bytes(4, 2, 2, 2) == -1
    assert lib.hipr_label_workspace_bytes(2, 0, 5, 0) == -1
    ws = lib.hipr_label_workspace_bytes(2, 4, 4, 0)
    assert lib.hipr_label(None, 4, 0, 2, 4, 4, 0, 1, p, ws, p, 4, p, None) == -1
    assert lib.hipr_label(p, 4, 0, 2, 4, 4, 0, 3, p, ws, p, 4, p, None) == -1             # connectivity > ndim
    assert lib.hipr_label(p, 4, 0, 3, 4, 4, 4, 0, p, ws, p, 4, p, None) == -1             # connectivity 0
    assert lib.hipr_label(p, 0, 0, 2, 4, 4, 0, 1, p, ws, p, 4, p, None) == -2             # float image
    assert lib.hipr_label(p, 4, 0, 2, 4, 4, 0, 1, p, ws, p, 2, p, None) == -2             # int16 labels
    assert lib.hipr_label(p, 4, 0, 2, 4, 4, 0, 1, p, ws - 4, p, 4, p, None) == -7         # workspace too small
    assert lib.hipr_label_counts(None, 4, 2, 4, 4, 0, -1, 3, p, None, None) == -1
    assert lib.hipr_label_counts(p, 2, 2, 4, 4, 0, -1, 3, p, None, None) == -2
    assert lib.hipr_label_counts(p, 4, 2, 4, 4, 0, -1, -1, p, None, None) == -1
    assert lib.hipr_label_clear(p, 0, p, 16, p, 0, p, None) == -2
    assert lib.hipr_label_clear(p, 4, p, 0, p, 0, p, None) == -1
    assert lib.hipr_paint_labels(p, 4, 16, p, 1, 3, 5, p, None) == -2                    # unknown value dtype
