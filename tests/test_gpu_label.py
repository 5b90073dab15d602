"""Connected-component operators (K10, csrc/label.cu) on the GPU: labels and counts bit-identical to scipy.ndimage
(masks) and the restatement of scikit-image in tests/label_oracle.py (label images), on random, percolating, adversarial,
degenerate and full-size inputs; the operators built on the labelling; determinism; and the whole segmentation
back end from the k-means mask to the per-cell spectra."""
import ctypes as C

import numpy as np
import pytest

import label_oracle

pytestmark = pytest.mark.gpu

def _cuda(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _want_label(image, conn):
    image = np.asarray(image)
    if image.dtype in (np.bool_, np.uint8):
        return label_oracle.label_mask(image, conn)
    return label_oracle.label_image(image, conn)


def _check_label(torch, h, image, conn=None, dtype=None):
    dtype = dtype or torch.int32
    got, n = h.label(_cuda(torch, image), connectivity=conn, return_num=True, dtype=dtype)
    want, wn = _want_label(image, conn)
    assert got.dtype == dtype
    assert n == wn, (n, wn)
    assert np.array_equal(got.cpu().numpy(), want)
    return n


@pytest.fixture(scope="module")
def h(torch_cuda):
    import hipr_b200
    return hipr_b200


# ---- exactness on random inputs ---------------------------------------------------------------------------------

SMALL = [(1, 1), (1, 700), (700, 1), (33, 65), (100, 37), (257, 129), (1, 1, 1), (1, 40, 50), (40, 50, 1),
         (3, 70, 33), (17, 9, 40), (33, 31, 65)]


@pytest.mark.parametrize("shape", SMALL)
def test_label_random_all_dtypes_and_connectivities(torch_cuda, h, shape):
    rng = np.random.default_rng(sum(shape))
    mask = rng.random(shape) < 0.5
    values = rng.integers(-2, 4, shape)
    for conn in range(1, len(shape) + 1):
        _check_label(torch_cuda, h, mask, conn)
        _check_label(torch_cuda, h, mask.astype(np.uint8) * rng.integers(1, 255, shape).astype(np.uint8),
                     conn)
        _check_label(torch_cuda, h, values.astype(np.int32), conn)
        _check_label(torch_cuda, h, values.astype(np.int64), conn, dtype=torch_cuda.int64)
        _check_label(torch_cuda, h, (values * 1_000_000_007).astype(np.int64), conn)


def test_label_default_connectivity_is_full(torch_cuda, h):
    rng = np.random.default_rng(5)
    for shape in ((64, 80), (12, 20, 24)):
        mask = rng.random(shape) < 0.3
        assert np.array_equal(h.label(_cuda(torch_cuda, mask)).cpu().numpy(), label_oracle.label_mask(mask, len(shape))[0])


# ---- percolation: single components span the image ----------------------------------------------------------------

@pytest.mark.parametrize("shape,conn,p", [((2048, 2048), 1, 0.59), ((2048, 2048), 2, 0.41),
                                          ((192, 256, 256), 1, 0.31), ((192, 256, 256), 2, 0.14),
                                          ((192, 256, 256), 3, 0.10)])
def test_label_percolation(torch_cuda, h, shape, conn, p):
    import scipy.ndimage as ndi
    mask = np.random.default_rng(conn * 7 + len(shape)).random(shape) < p
    n = _check_label(torch_cuda, h, mask, conn)
    want, _ = label_oracle.label_mask(mask, conn)
    big = np.argmax(np.bincount(want.ravel())[1:]) + 1
    extent = [s.stop - s.start for s in ndi.find_objects((want == big).astype(np.int32))[0]]
    assert n > 1000 and max(extent) >= max(shape) // 2          # many clusters, and one that spans the image


# ---- adversarial shapes -------------------------------------------------------------------------------------------

def serpentine(H, W):
    """A one-pixel-wide path through every other row, joined at alternating ends: one 4-connected component."""
    s = np.zeros((H, W), bool)
    s[0::2] = True
    s[1::4, W - 1] = True
    s[3::4, 0] = True
    return s


def test_label_serpentine(torch_cuda, h):
    s = serpentine(2048, 2048)
    for conn in (1, 2):
        assert _check_label(torch_cuda, h, s, conn) == 1
    vol = np.zeros((8, 129, 130), bool)                        # the same path through a volume, plane after plane
    vol[:, 0::2] = True
    vol[:, 1::4, -1] = True
    vol[:, 3::4, 0] = True
    vol[1::2, -1, 0] = False
    for conn in (1, 2, 3):
        _check_label(torch_cuda, h, vol, conn)


def test_label_u_and_comb(torch_cuda, h):
    """Components whose first pixel lies to the right of, and in a later tile than, most of their pixels."""
    img = np.zeros((700, 700), np.int32)
    img[280:300, 3:680] = 1                                     # U: bar at the bottom ...
    img[150:300, 3:6] = 1                                       # ... short left arm
    img[5:300, 660:680] = 1                                     # ... tall right arm holds the first pixel
    for k, c in enumerate(range(20, 640, 37)):                  # comb: teeth rising from a bar, tallest last
        img[660 - 20 * k:690, c:c + 3] = 2
    img[680:690, 20:640] = 2
    img[100:110, 100:110] = 2                                   # same value, not connected
    for conn in (1, 2):
        assert _check_label(torch_cuda, h, img, conn) == 3
        assert _check_label(torch_cuda, h, img != 0, conn) == 3
    vol = np.zeros((40, 50, 60), bool)
    vol[35, :, :] = True
    vol[:, 45, 50:] = True
    vol[2:36, 10, 3] = True
    for conn in (1, 2, 3):
        assert _check_label(torch_cuda, h, vol, conn) == 1


def test_label_checkerboard(torch_cuda, h):
    board = (np.add.outer(np.arange(2048), np.arange(2048)) % 2 == 0)
    assert _check_label(torch_cuda, h, board, 1) == 2048 * 2048 // 2
    assert _check_label(torch_cuda, h, board, 2) == 1
    vol = (np.indices((32, 64, 64)).sum(0) % 2 == 0)
    assert _check_label(torch_cuda, h, vol, 1) == vol.sum()
    assert _check_label(torch_cuda, h, vol, 2) == 1


# ---- edge cases ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape", [(1, 1), (1, 5000), (5000, 1), (31, 33), (513, 515), (7, 1, 9), (5, 33, 1),
                                   (1, 1, 77), (9, 17, 33)])
def test_label_edge_cases(torch_cuda, h, shape):
    for conn in range(1, len(shape) + 1):
        assert _check_label(torch_cuda, h, np.zeros(shape, bool), conn) == 0
        assert _check_label(torch_cuda, h, np.ones(shape, bool), conn) == 1
        assert _check_label(torch_cuda, h, np.full(shape, -3, np.int64), conn) == 1
        corners = np.zeros(shape, np.int32)
        for c in np.ndindex(*([2] * len(shape))):
            corners[tuple(-1 if b else 0 for b in c)] = 7
        _check_label(torch_cuda, h, corners, conn)


# ---- realistic sizes ----------------------------------------------------------------------------------------------

def test_label_synthetic_fov_and_volume(torch_cuda, h):
    from hipr_b200 import synth
    lab, _ = synth.make_labels(2048, 2048)
    mask = (lab > 0).numpy()
    for conn in (1, 2):
        assert _check_label(torch_cuda, h, mask, conn) > 3000
    _check_label(torch_cuda, h, lab.numpy(), 1)
    import scipy.ndimage as ndi
    rng = np.random.default_rng(2)
    vol = ndi.uniform_filter(rng.random((1024, 1024, 64), dtype=np.float32), 3) > 0.55
    _check_label(torch_cuda, h, vol, 3)


# ---- outputs, inputs, views ---------------------------------------------------------------------------------------

def test_label_views_and_output_dtypes(torch_cuda, h):
    rng = np.random.default_rng(9)
    base = rng.integers(0, 3, (300, 400)).astype(np.int64)
    t = _cuda(torch_cuda, base)
    for view, ref in ((t[::2, 1:], base[::2, 1:]), (t.T, base.T), (t[5:200, 7:300:3], base[5:200, 7:300:3])):
        assert not view.is_contiguous()
        for dtype in (torch_cuda.int32, torch_cuda.int64):
            got, n = h.label(view, connectivity=1, return_num=True, dtype=dtype)
            want, wn = label_oracle.label_image(ref, 1)
            assert n == wn and got.dtype == dtype and np.array_equal(got.cpu().numpy(), want)
            got = h.label(view != 0, connectivity=2, dtype=dtype)
            assert np.array_equal(got.cpu().numpy(), label_oracle.label_mask(ref != 0, 2)[0])


# ---- determinism and the workspace --------------------------------------------------------------------------------

def test_label_deterministic_and_independent_of_workspace(torch_cuda, h):
    torch = torch_cuda
    from hipr_b200 import ops
    lib = h.lib()
    mask = np.random.default_rng(4).random((1024, 1536)) < 0.59
    m = _cuda(torch, mask).view(torch.uint8)
    want, wn = label_oracle.label_mask(mask, 1)
    ws = lib.hipr_label_workspace_bytes(2, 1024, 1536, 0)
    results = []
    for fill in (None, 0x00, 0xFF, 0x80, "random"):
        work = torch.empty(ws, dtype=torch.uint8, device="cuda")
        if fill == "random":
            work.random_(0, 256)
        elif fill is not None:
            work.fill_(fill)
        out = torch.full((1024, 1536), -5, dtype=torch.int32, device="cuda")
        n = torch.full((1,), -5, dtype=torch.int64, device="cuda")
        ops.check(lib.hipr_label(C.c_void_p(m.data_ptr()), 4, 0, 2, 1024, 1536, 0, 1, C.c_void_p(work.data_ptr()),
                                 ws, C.c_void_p(out.data_ptr()), 4, C.c_void_p(n.data_ptr()),
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)), "label")
        results.append((out.cpu().numpy(), int(n.item())))
    for out, n in results:
        assert n == wn and np.array_equal(out, want)


def test_label_launches_and_no_host_copy(torch_cuda, h):
    """Five launches whatever the image holds, and no device-to-host copy unless return_num."""
    torch = torch_cuda
    from torch.profiler import ProfilerActivity, profile
    lib = h.lib()
    noise = _cuda(torch, np.random.default_rng(1).random((2048, 2048)) < 0.59)
    snake = _cuda(torch, serpentine(2048, 2048))
    counts = {}
    for name, img in (("noise", noise), ("serpentine", snake)):
        h.label(img)                                           # warm-up
        torch.cuda.synchronize()
        before = lib.hipr_launch_count()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            h.label(img)
            torch.cuda.synchronize()
        counts[name] = lib.hipr_launch_count() - before
        names = [e.name for e in prof.events()]
        assert not any("DtoH" in n or "Device -> Host" in n for n in names), names
        k10 = [n for n in names if any(k in n for k in ("tile_union", "border_union", "flatten_kernel",
                                                       "chunk_scan", "write_labels"))]
        assert len(k10) == 5, k10
    assert counts == {"noise": 5, "serpentine": 5}


# ---- the operators built on the labelling -------------------------------------------------------------------------

@pytest.mark.parametrize("shape", [(257, 300), (1, 900), (20, 33, 40)])
def test_remove_small_objects(torch_cuda, h, shape):
    rng = np.random.default_rng(6)
    mask = rng.random(shape) < 0.45
    for conn in range(1, len(shape) + 1):
        for min_size in (0, 1, 2, 5, 64):
            got = h.remove_small_objects(_cuda(torch_cuda, mask), min_size, conn)
            assert got.dtype == torch_cuda.bool
            assert np.array_equal(got.cpu().numpy(), label_oracle.remove_small_objects_mask(mask, min_size, conn))
    labels = label_oracle.label_mask(mask, 1)[0]
    for dt in (np.int32, np.int64):
        lab = (labels * 3).astype(dt)                           # gaps in the numbering
        for min_size in (1, 3, 10):
            got = h.remove_small_objects(_cuda(torch_cuda, lab), min_size)
            assert got.dtype == _cuda(torch_cuda, lab).dtype
            assert np.array_equal(got.cpu().numpy(), label_oracle.remove_small_objects_labels(lab, min_size))
        with pytest.raises(ValueError, match="negative"):
            h.remove_small_objects(_cuda(torch_cuda, lab - 1), 3)


@pytest.mark.parametrize("shape", [(512, 480), (1, 50), (50, 1), (24, 40, 36)])
def test_binary_fill_holes(torch_cuda, h, shape):
    rng = np.random.default_rng(8)
    for p in (0.3, 0.55, 0.7):
        mask = rng.random(shape) < p
        for conn in range(1, len(shape) + 1):
            for m in (mask, mask.astype(np.uint8)):
                got = h.binary_fill_holes(_cuda(torch_cuda, m), conn)
                assert got.dtype == torch_cuda.bool
                assert np.array_equal(got.cpu().numpy(), label_oracle.binary_fill_holes(m, conn))
    from hipr_b200 import synth
    lab, _ = synth.make_labels(2048, 2048)
    ring = (lab > 0).numpy() & ~np.isin(np.arange(lab.numel()).reshape(lab.shape) % 7, (0,))
    assert np.array_equal(h.binary_fill_holes(_cuda(torch_cuda, ring)).cpu().numpy(), label_oracle.binary_fill_holes(ring))


@pytest.mark.parametrize("shape", [(300, 257), (1, 40), (20, 25, 30)])
def test_clear_border(torch_cuda, h, shape):
    rng = np.random.default_rng(10)
    mask = rng.random(shape) < 0.35
    labels = label_oracle.label_mask(mask, 1)[0]
    for image in (mask, mask.astype(np.uint8), labels.astype(np.int32), (labels % 5).astype(np.int64) - 1):
        for buffer_size in sorted(b for b in {0, 1, 3, min(shape) - 1} if b < min(shape)):
            for bgval in ((0,) if image.dtype == bool else (0, 7)):
                got = h.clear_border(_cuda(torch_cuda, image), buffer_size, bgval)
                want = label_oracle.clear_border(image, buffer_size, bgval)
                assert got.dtype == _cuda(torch_cuda, image).dtype
                assert np.array_equal(got.cpu().numpy(), want), (image.dtype, buffer_size, bgval)
    with pytest.raises(ValueError, match="buffer size"):
        h.clear_border(_cuda(torch_cuda, labels), min(shape))


def test_relabel_sequential(torch_cuda, h):
    rng = np.random.default_rng(12)
    base = rng.integers(0, 50, (200, 300)) * 1000
    base[base == 7000] = 0
    for dt in (np.int32, np.int64):
        for offset in (1, 3, 1000):
            lab = base.astype(dt)
            got, fw, inv = h.relabel_sequential(_cuda(torch_cuda, lab), offset)
            want, wfw, winv = label_oracle.relabel_sequential(lab, offset)
            assert got.dtype == _cuda(torch_cuda, want).dtype
            for a, b in ((got, want), (fw, wfw), (inv, winv)):
                assert np.array_equal(a.cpu().numpy(), b)
    vol = rng.integers(0, 4, (10, 20, 30)).astype(np.int64) * 5
    got, fw, inv = h.relabel_sequential(_cuda(torch_cuda, vol))
    assert all(np.array_equal(a.cpu().numpy(), b) for a, b in zip((got, fw, inv), label_oracle.relabel_sequential(vol)))
    two = np.array([[0, 9], [5, 0]], np.int32)                 # offset + n - 1 beyond int32: int64 result
    got, _, _ = h.relabel_sequential(_cuda(torch_cuda, two), 2 ** 31 - 2)
    assert got.dtype == torch_cuda.int32 and got.cpu().numpy().tolist() == [[0, 2 ** 31 - 1], [2 ** 31 - 2, 0]]
    got, _, _ = h.relabel_sequential(_cuda(torch_cuda, two), 2 ** 31 - 1)
    assert got.dtype == torch_cuda.int64 and got.cpu().numpy().tolist() == [[0, 2 ** 31], [2 ** 31 - 1, 0]]
    with pytest.raises(ValueError, match="negative"):
        h.relabel_sequential(_cuda(torch_cuda, np.array([[0, -1]], np.int32)))


# ---- the whole back end on the device ----------------------------------------------------------------------------

def test_segmentation_chain_stays_on_device(torch_cuda, h):
    """score map -> k-means mask -> fill holes -> remove small objects -> label -> clear border -> relabel ->
    per-cell spectra and geometry, on the device; the same chain on the host from the same mask."""
    torch = torch_cuda
    from hipr_b200 import synth
    cube, _, _ = synth.make_fov(512, 640, 95, fov_index=2)
    cube_d = cube.cuda()
    score = h.neighbor2d_score(cube_d, "F1")
    mask = h.kmeans_threshold(score, 2).mask
    filled = h.binary_fill_holes(mask)
    kept = h.remove_small_objects(filled, 20)
    lab = h.label(kept, connectivity=1)
    cleared = h.clear_border(lab)
    seg, fw, inv = h.relabel_sequential(cleared)
    spec = h.cell_spectra(cube_d, seg)
    geom = h.cell_geometry(seg)

    m = mask.cpu().numpy()
    assert 0.05 < m.mean() < 0.95
    w = label_oracle.binary_fill_holes(m)
    w = label_oracle.remove_small_objects_mask(w, 20, 1)
    w, _ = label_oracle.label_mask(w, 1)
    w = label_oracle.clear_border(w)
    wseg, _, _ = label_oracle.relabel_sequential(w)
    assert np.array_equal(seg.cpu().numpy(), wseg)
    assert wseg.max() > 20
    host = h.cell_spectra_host(cube.numpy(), wseg)             # float64 atomics: sums agree to rounding
    assert np.array_equal(spec[0].cpu().numpy(), host[0]) and np.array_equal(spec[1].cpu().numpy(), host[1])
    for a, b in zip(spec[2:], host[2:]):
        np.testing.assert_allclose(a.cpu().numpy(), b, rtol=1e-12)
    hgeom = h.cell_geometry(_cuda(torch, wseg))
    for a, b in zip(geom, hgeom):
        assert torch.equal(a, b)
