"""The marker watershed (K11, csrc/watershed.cu) on the GPU: bit-identical to the rule of tests/watershed_oracle.py on
every input (tied, signed zeros, infinities, degenerate shapes, views), to the heap restatement of scikit-image wherever
no pixel is tie-decided; the serpentine worst case; workspace independence, determinism, launches and copies; the
device-label form of Fov.cell_spectra; and the whole segmentation chain from the score map to the per-cell spectra."""
import ctypes as C

import numpy as np
import pytest

import label_oracle
import watershed_oracle as wo

pytestmark = pytest.mark.gpu


def _cuda(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def h(torch_cuda):
    import hipr_b200
    return hipr_b200


def _check(torch, h, image, markers, conn, mask=None, tag=""):
    """Device result == rule bit for bit; == heap where the heap has no tie-decided pixel (else print the count)."""
    got = h.watershed(_cuda(torch, image), _cuda(torch, markers), conn, None if mask is None else _cuda(torch, mask))
    assert got.dtype == _cuda(torch, markers).dtype
    got = got.cpu().numpy()
    want = wo.watershed_rule(image, markers, conn, mask)
    assert np.array_equal(got, want), (tag, int((got != want).sum()))
    heap = wo.watershed_heap(image, markers, conn, mask)
    if not heap.tied.any():
        assert np.array_equal(got, heap.labels), tag
    else:
        print("%s: %d tie-decided pixels, %d labels differ from the heap" % (tag, heap.tied.sum(),
                                                                             (got != heap.labels).sum()))
    return got


def _markers(rng, shape, n, dtype):
    m = np.zeros(shape, dtype)
    idx = rng.choice(m.size, size=min(n, m.size), replace=False)
    m.ravel()[idx] = rng.integers(-5, 40, len(idx))
    m.ravel()[idx[m.ravel()[idx] == 0]] = 3
    return m


def _images(rng, shape):
    yield "continuous", rng.standard_normal(shape)
    yield "uint8", np.floor(rng.random(shape) * 256) / 255.0                 # quantised: plateaus everywhere
    yield "constant", np.full(shape, 0.25)                                   # one big plateau
    z = rng.choice([-0.0, 0.0, 1.0, np.inf, -np.inf], size=shape)            # signed zeros and infinities
    yield "zeros_infs", z


SHAPES = [((96, 130), (1, 2)), ((1, 300), (1, 2)), ((300, 1), (1, 2)), ((1, 1), (1, 2)), ((70, 64), (1, 2)),
          ((20, 33, 40), (1, 2, 3)), ((1, 40, 50), (1, 2, 3)), ((40, 3, 1), (1, 2, 3)), ((2, 2, 2), (1, 2, 3))]


@pytest.mark.parametrize("shape,conns", SHAPES)
def test_watershed_matches_rule(torch_cuda, h, shape, conns):
    rng = np.random.default_rng(sum(shape))
    for conn in conns:
        for k, (kind, image) in enumerate(_images(rng, shape)):
            for dt in (np.float32, np.float64):
                mdt = np.int32 if (k + conn) % 2 else np.int64
                markers = _markers(rng, shape, max(1, int(np.prod(shape)) // 200), mdt)
                mask = (rng.random(shape) < 0.85) if (k + conn) % 3 else None
                _check(torch_cuda, h, image.astype(dt), markers, conn, mask, "%s %s %s c%d" % (shape, kind, dt.__name__, conn))


def test_watershed_no_markers_and_all_markers(torch_cuda, h):
    rng = np.random.default_rng(4)
    image = rng.random((50, 70)).astype(np.float32)
    mask = rng.random((50, 70)) < 0.7
    torch = torch_cuda
    assert not h.watershed(_cuda(torch, image), _cuda(torch, np.zeros((50, 70), np.int32))).any()
    full = rng.integers(1, 9, (50, 70)).astype(np.int64) * rng.choice([-1, 1], (50, 70))
    assert np.array_equal(h.watershed(_cuda(torch, image), _cuda(torch, full)).cpu().numpy(), full)
    got = h.watershed(_cuda(torch, image), _cuda(torch, full), mask=_cuda(torch, mask)).cpu().numpy()
    assert np.array_equal(got, full * mask)                                  # markers outside the mask are dropped


def test_watershed_integer_images_and_uint8_mask(torch_cuda, h):
    torch = torch_cuda
    rng = np.random.default_rng(9)
    raw = rng.integers(0, 5000, (60, 80))
    markers = _markers(rng, (60, 80), 20, np.int32)
    mask = (rng.random((60, 80)) < 0.8).astype(np.uint8)
    want = wo.watershed_rule(raw.astype(np.float64), markers, 2, mask)
    for dt in (torch.uint8, torch.uint16, torch.int32):
        img = torch.from_numpy(raw % 256 if dt == torch.uint8 else raw).to(dt).cuda()
        w = want if dt != torch.uint8 else wo.watershed_rule((raw % 256).astype(np.float64), markers, 2, mask)
        got = h.watershed(img, _cuda(torch, markers), 2, _cuda(torch, mask))
        assert np.array_equal(got.cpu().numpy(), w), dt


def test_watershed_views(torch_cuda, h):
    torch = torch_cuda
    rng = np.random.default_rng(13)
    big = rng.standard_normal((80, 90, 7))
    mk = _markers(rng, (80, 90, 7), 60, np.int64)
    mask = rng.random((80, 90, 7)) < 0.8
    bt, mt, kt = _cuda(torch, big), _cuda(torch, mk), _cuda(torch, mask)
    for sl in ((slice(None), slice(None), 3), (slice(5, 70, 2), slice(None), 1), (slice(None), 4, slice(None))):
        got = h.watershed(bt[sl], mt[sl], 2, kt[sl]).cpu().numpy()
        assert np.array_equal(got, wo.watershed_rule(big[sl], mk[sl], 2, mask[sl]))
    t = (slice(None), slice(None), slice(None))
    got = h.watershed(bt[t].transpose(1, 2), mt[t].transpose(1, 2), 3).cpu().numpy()      # (80, 7, 90), strided
    assert np.array_equal(got, wo.watershed_rule(big.transpose(0, 2, 1), mk.transpose(0, 2, 1), 3))


def serpentine(H, W):
    """One-pixel corridor: every other row open, joined alternately at the right and the left end."""
    m = np.zeros((H, W), bool)
    m[::2] = True
    for r in range(1, H, 2):
        m[r, W - 1 if (r // 2) % 2 == 0 else 0] = True
    return m


def test_watershed_serpentine(torch_cuda, h):
    torch = torch_cuda
    from hipr_b200 import ops
    rng = np.random.default_rng(17)
    mask = serpentine(512, 512)
    image = rng.random((512, 512)).astype(np.float32)
    markers = np.zeros((512, 512), np.int32)
    markers[0, 0] = 7
    out, status = ops._watershed(_cuda(torch, image), _cuda(torch, markers), 1, _cuda(torch, mask))
    st = status.cpu().numpy()
    print("serpentine 512^2: rounds per phase %s, tile visits %s, CTAs %d" % (st[1:4], st[4:7], st[7]))
    assert st[0] == 0
    assert np.array_equal(out.cpu().numpy(), np.where(mask, 7, 0))


def _raw_watershed(torch, h, image, markers, work, conn=1):
    from hipr_b200 import ops
    lib = h.lib()
    out = torch.full_like(markers, -9)
    status = torch.full((8,), -9, dtype=torch.int64, device="cuda")
    ops.check(lib.hipr_watershed(C.c_void_p(image.data_ptr()), 1 if image.dtype == torch.float64 else 0,
                                 C.c_void_p(markers.data_ptr()), markers.element_size(), None, 2, image.shape[0],
                                 image.shape[1], 0, conn, C.c_void_p(work.data_ptr()), work.numel(),
                                 C.c_void_p(out.data_ptr()), C.c_void_p(status.data_ptr()),
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)), "watershed")
    return out, status


def test_watershed_workspace_and_determinism(torch_cuda, h):
    torch = torch_cuda
    rng = np.random.default_rng(21)
    image = _cuda(torch, np.floor(rng.random((700, 900)) * 16))              # heavily tied
    markers = _cuda(torch, _markers(rng, (700, 900), 300, np.int32))
    ws = h.lib().hipr_watershed_workspace_bytes(2, 700, 900, 0, 1, 4)
    results = []
    for fill in (0x00, 0xFF, 0x5A, None):
        work = torch.empty(ws, dtype=torch.uint8, device="cuda")
        if fill is None:
            work.copy_(torch.randint(0, 256, (ws,), dtype=torch.uint8, device="cuda"))
        else:
            work.fill_(fill)
        out, status = _raw_watershed(torch, h, image, markers, work, 2)
        assert int(status[0]) == 0
        results.append(out.cpu().numpy())
    want = wo.watershed_rule(image.cpu().numpy(), markers.cpu().numpy(), 2)
    for r in results:
        assert np.array_equal(r, want)


def test_watershed_rejects_nan(torch_cuda, h):
    torch = torch_cuda
    image = torch.zeros(20, 30, device="cuda")
    image[5, 5] = float("nan")
    markers = torch.zeros(20, 30, dtype=torch.int32, device="cuda")
    markers[0, 0] = 1
    with pytest.raises(ValueError, match="NaN"):
        h.watershed(image, markers)
    mask = torch.ones(20, 30, dtype=torch.bool, device="cuda")
    mask[5, 5] = False
    got = h.watershed(image, markers, mask=mask)                             # NaN outside the mask is harmless
    assert int(got.sum()) == 20 * 30 - 1


def test_watershed_launches_and_copies(torch_cuda, h):
    """One launch whatever the image holds; the only device-to-host copies are the NaN check and the status."""
    torch = torch_cuda
    from torch.profiler import ProfilerActivity, profile
    lib = h.lib()
    rng = np.random.default_rng(23)
    noise = (_cuda(torch, rng.random((1024, 1024)).astype(np.float32)), _cuda(torch, _markers(rng, (1024, 1024), 500, np.int32)), None)
    snake = (_cuda(torch, rng.random((256, 256)).astype(np.float32)),
             _cuda(torch, np.pad(np.ones((1, 1), np.int32), ((0, 255), (0, 255)))), _cuda(torch, serpentine(256, 256)))
    counts = {}
    for name, (img, mk, mask) in (("noise", noise), ("serpentine", snake)):
        h.watershed(img, mk, mask=mask)
        torch.cuda.synchronize()
        before = lib.hipr_launch_count()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            h.watershed(img, mk, mask=mask)
            torch.cuda.synchronize()
        counts[name] = lib.hipr_launch_count() - before
        names = [e.name for e in prof.events()]
        d2h = [n for n in names if "DtoH" in n or "Device -> Host" in n]
        assert len(d2h) <= 2, d2h
        assert sum("watershed_kernel" in n for n in names) == 1
    assert counts == {"noise": 1, "serpentine": 1}


def test_fov_cell_spectra_device_labels(torch_cuda, h):
    torch = torch_cuda
    from hipr_b200 import synth
    cube, _, _ = synth.make_fov(256, 320, 40, fov_index=1)
    lab, _ = synth.make_labels(256, 320)
    with h.Fov(cube.numpy()) as fov:
        for dt in (np.int32, np.int64):
            lab_np = lab.numpy().astype(dt)
            a = fov.cell_spectra(lab_np)
            b = fov.cell_spectra(_cuda(torch, lab_np))
            assert len(a[0]) > 10
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
            for x, y in zip(a[2:], b[2:]):                                   # float64 atomics: agree to rounding
                np.testing.assert_allclose(y, x, rtol=1e-12)
                print("device labels vs numpy labels: max |diff| %.3g" % np.max(np.abs(x - y)))
        empty = fov.cell_spectra(torch.zeros(256, 320, dtype=torch.int32, device="cuda"))
        assert all(len(t) == 0 for t in empty)
        with pytest.raises(ValueError, match="labels must be"):
            fov.cell_spectra(torch.zeros(256, 321, dtype=torch.int32, device="cuda"))
        with pytest.raises(TypeError):
            fov.cell_spectra(torch.zeros(256, 320, dtype=torch.float32, device="cuda"))


def test_segmentation_chain_with_watershed(torch_cuda, h):
    """2048^2 FOV: score -> k-means mask -> fill holes -> remove small objects -> label markers -> watershed on the
    negated score -> clear border -> relabel -> Fov.cell_spectra with device labels; the same chain on the host
    through the oracles from the same score map and mask."""
    import time
    torch = torch_cuda
    from hipr_b200 import synth
    cube, _, _ = synth.make_fov(2048, 2048, 95, fov_index=3)
    with h.Fov(cube.numpy()) as fov:
        cube_d = cube.cuda()
        score = h.neighbor2d_score(cube_d, "F1")
        del cube_d
        mask = h.kmeans_threshold(score, 2).mask
        filled = h.binary_fill_holes(mask)
        kept = h.remove_small_objects(filled, 20)
        thr = torch.quantile(score[kept].float()[::7], 0.8)
        seeds = h.remove_small_objects(kept & (score >= thr), 4)
        markers = h.label(seeds, connectivity=1)
        seg = h.watershed(-score, markers, 1, kept)
        seg, _, _ = h.relabel_sequential(h.clear_border(seg))
        spec = fov.cell_spectra(seg)

        s, m = score.cpu().numpy(), mask.cpu().numpy()
        k = label_oracle.remove_small_objects_mask(label_oracle.binary_fill_holes(m), 20, 1)
        sd = label_oracle.remove_small_objects_mask(k & (s >= float(thr)), 4, 1)
        wm, n_markers = label_oracle.label_mask(sd, 1)
        t0 = time.perf_counter()
        w = wo.watershed_rule(-s, wm, 1, k)
        print("2048^2 chain: %d markers; restatement time %.1f s" % (n_markers, time.perf_counter() - t0))
        wseg, _, _ = label_oracle.relabel_sequential(label_oracle.clear_border(w))
        assert np.array_equal(seg.cpu().numpy(), wseg)
        assert wseg.max() > 50
        host = fov.cell_spectra(wseg)
    assert np.array_equal(spec[0], host[0]) and np.array_equal(spec[1], host[1])
    for a, b in zip(spec[2:], host[2:]):
        np.testing.assert_allclose(a, b, rtol=1e-5)
