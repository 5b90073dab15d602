"""Binary morphology (K12, csrc/morphology.cu) on the GPU: binary_erosion, binary_dilation, binary_opening and
binary_closing bit-identical to scipy.ndimage across operations, border values, iterations, structures, shapes around
the 32-bit word edges, contents and full-size inputs; argument checks; workspace independence and determinism; the
launch count; and the segmentation chain from the k-means mask to the label image."""
import ctypes as C

import numpy as np
import pytest
import scipy.ndimage as ndi

import label_oracle

pytestmark = pytest.mark.gpu

OPS = ("erosion", "dilation", "opening", "closing")


@pytest.fixture(scope="module")
def h(torch_cuda):
    import hipr_b200
    return hipr_b200


def _cuda(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# scikit-image is not installed: its footprints disk(r) and ball(r) are x^2 + y^2 (+ z^2) <= r^2
def disk(r):
    y, x = np.mgrid[-r:r + 1, -r:r + 1]
    return x * x + y * y <= r * r


def ball(r):
    z, y, x = np.mgrid[-r:r + 1, -r:r + 1, -r:r + 1]
    return x * x + y * y + z * z <= r * r


def _want(op, mask, structure, iterations, border_value):
    """scipy.ndimage's answer.  brute_force=True: scipy 1.18.1's default path for iterations > 1 corrupts memory when
    the image is smaller than the structure along an axis; brute_force repeats the single pass, which scipy defines
    to give the same result."""
    mask = np.asarray(mask) != 0
    if structure is None:
        structure = ndi.generate_binary_structure(mask.ndim, 1)
    f = getattr(ndi, "binary_" + op)
    return f(mask, structure, iterations, border_value=border_value, brute_force=True)


def _check(torch, h, mask, structure=None, op="erosion", iterations=1, border_value=0, dev=None):
    dev = _cuda(torch, mask) if dev is None else dev
    got = getattr(h, "binary_" + op)(dev, structure, iterations, border_value)
    assert got.dtype == torch.bool and tuple(got.shape) == tuple(np.shape(mask)) and got.device == dev.device
    want = _want(op, mask, structure, iterations, border_value)
    ok = np.array_equal(got.cpu().numpy(), want)
    assert ok, (op, np.shape(mask), None if structure is None else np.shape(structure), iterations, border_value,
                int((got.cpu().numpy() != want).sum()))


@pytest.mark.parametrize("op", OPS)
def test_operations_border_values_and_iterations(torch_cuda, h, op):
    rng = np.random.default_rng(1)
    m2 = rng.random((100, 95)) < 0.5
    m3 = rng.random((17, 9, 40)) < 0.5
    for b in (0, 1):
        for it in (1, 2, 5):
            _check(torch_cuda, h, m2, None, op, it, b)
            _check(torch_cuda, h, m2, disk(2), op, it, b)
            _check(torch_cuda, h, m3, None, op, it, b)
            _check(torch_cuda, h, m3, ball(1), op, it, b)


def _asymmetric(rng, shape):
    s = rng.random(shape) < 0.5
    s.flat[rng.integers(s.size)] = True
    return s


def _structures_2d():
    rng = np.random.default_rng(7)
    out = [ndi.generate_binary_structure(2, c) for c in (1, 2)]
    out += [np.ones((k, k), bool) for k in (3, 5, 9)]
    out += [disk(r) for r in range(1, 16)]
    out += [np.ones((1, k), bool) for k in (3, 7, 31)] + [np.ones((k, 1), bool) for k in (3, 7, 31)]
    out += [np.ones((1, 1), bool), np.zeros((3, 3), bool), np.zeros((1, 1), bool)]
    out += [_asymmetric(rng, s) for s in [(3, 3), (3, 5), (5, 3), (7, 7), (1, 9), (9, 1), (11, 5)]]
    out += [np.ones((31, 31), bool), _asymmetric(rng, (31, 31)), _asymmetric(rng, (31, 3))]   # the largest extent
    return out


def _structures_3d():
    rng = np.random.default_rng(8)
    out = [ndi.generate_binary_structure(3, c) for c in (1, 2, 3)]
    out += [np.ones((k, k, k), bool) for k in (3, 5)]
    out += [ball(r) for r in range(1, 8)]
    for k in (3, 9):
        out += [np.ones((k, 1, 1), bool), np.ones((1, k, 1), bool), np.ones((1, 1, k), bool)]
    out += [np.ones((1, 1, 1), bool), np.zeros((3, 3, 3), bool)]
    out += [_asymmetric(rng, s) for s in [(3, 3, 3), (1, 3, 5), (5, 3, 1), (3, 5, 7)]]
    out += [np.ones((31, 1, 1), bool), np.ones((1, 31, 1), bool), np.ones((1, 1, 31), bool),
            _asymmetric(rng, (3, 31, 5))]                                                          # the largest extent
    return out


def test_structures_2d(torch_cuda, h):
    rng = np.random.default_rng(2)
    masks = [rng.random((70, 97)) < p for p in (0.3, 0.8)]
    for s in _structures_2d():
        for m in masks:
            for op in ("erosion", "dilation"):
                for b in (0, 1):
                    _check(torch_cuda, h, m, s, op, 1, b)
        _check(torch_cuda, h, masks[0], s, "opening", 2, 0)
        _check(torch_cuda, h, masks[1], s, "closing", 2, 1)


def test_structures_3d(torch_cuda, h):
    rng = np.random.default_rng(3)
    masks = [rng.random((19, 23, 45)) < p for p in (0.3, 0.8)]
    for s in _structures_3d():
        for m in masks:
            for op in ("erosion", "dilation"):
                for b in (0, 1):
                    _check(torch_cuda, h, m, s, op, 1, b)
        _check(torch_cuda, h, masks[0], s, "opening", 2, 1)
        _check(torch_cuda, h, masks[1], s, "closing", 2, 0)


def test_largest_cube(torch_cuda, h):
    """31 x 31 x 31, the largest extent along every axis at once, on a volume smaller than it along two axes."""
    m = np.random.default_rng(12).random((6, 40, 9)) < 0.9
    for op in ("erosion", "dilation"):
        for b in (0, 1):
            _check(torch_cuda, h, m, np.ones((31, 31, 31), bool), op, 1, b)


def test_structure_as_cpu_tensor_and_values(torch_cuda, h):
    m = np.random.default_rng(4).random((40, 70)) < 0.5
    s = np.array([[0, 3, 0], [1, 1, 0], [0, 0, -2]], np.int64)
    _check(torch_cuda, h, m, torch_cuda.from_numpy(s), "dilation", 2, 1)
    _check(torch_cuda, h, m, s.astype(np.float32), "erosion", 1, 0)
    got = h.binary_erosion(_cuda(torch_cuda, m), torch_cuda.from_numpy(s), border_value=7)   # non-zero counts as 1
    assert np.array_equal(got.cpu().numpy(), _want("erosion", m, s, 1, 1))


@pytest.mark.parametrize("shape", [(1, 1), (1, 200), (200, 1), (1, 1, 90), (1, 90, 1), (90, 1, 1),
                                   (20, 31), (20, 32), (20, 33), (20, 63), (20, 64), (20, 65), (20, 95),
                                   (3, 70, 33), (17, 9, 40), (5, 4, 95), (2, 3, 64)])
def test_shapes(torch_cuda, h, shape):
    rng = np.random.default_rng(sum(shape))
    m = rng.random(shape) < 0.6
    big = disk(5) if len(shape) == 2 else ball(3)          # radius above some of these extents
    for s in (None, big):
        for op in OPS:
            for b in (0, 1):
                for it in (1, 2):
                    _check(torch_cuda, h, m, s, op, it, b)


def test_contents(torch_cuda, h):
    torch = torch_cuda
    rng = np.random.default_rng(5)
    for shape, s in (((150, 77), disk(3)), ((13, 30, 70), ball(2))):
        for p in (0.1, 0.5, 0.9):
            m = rng.random(shape) < p
            for op in OPS:
                _check(torch, h, m, s, op, 2, 0)
                _check(torch, h, m, None, op, 1, 1)
        for m in (np.zeros(shape, bool), np.ones(shape, bool)):         # the border value alone decides the edge
            for op in OPS:
                for b in (0, 1):
                    _check(torch, h, m, s, op, 1, b)
                    _check(torch, h, m, None, op, 3, b)
        vals = rng.integers(0, 256, shape).astype(np.uint8)
        vals[rng.random(shape) < 0.4] = 0
        for op in OPS:
            _check(torch, h, vals, s, op, 1, 0)
    m = rng.random((64, 96)) < 0.5
    dev = _cuda(torch, m)
    _check(torch, h, m.T, disk(2), "opening", 1, 0, dev=dev.t())                  # a transpose
    _check(torch, h, m[3::2, 1::3], None, "closing", 2, 1, dev=dev[3::2, 1::3])   # a strided slice
    m3 = rng.random((10, 20, 40)) < 0.5
    dev3 = _cuda(torch, m3)
    _check(torch, h, m3.transpose(2, 0, 1), ball(1), "dilation", 2, 1, dev=dev3.permute(2, 0, 1))
    u8 = (rng.integers(0, 4, (50, 70)) * 60).astype(np.uint8)
    du8 = _cuda(torch, u8)
    _check(torch, h, u8[:, ::2], disk(1), "erosion", 1, 1, dev=du8[:, ::2])


def test_full_size(torch_cuda, h):
    torch = torch_cuda
    from hipr_b200 import synth
    labels, _ = synth.make_labels(2048, 2048)
    m = labels.numpy() > 0
    dev = _cuda(torch, m)
    for s in (None, disk(5)):
        _check(torch, h, m, s, "opening", 1, 0, dev=dev)
        _check(torch, h, m, s, "erosion", 2, 1, dev=dev)
    rng = np.random.default_rng(9)
    v = ndi.gaussian_filter(rng.random((1024, 1024, 64)).astype(np.float32), 2) > 0.5
    dv = _cuda(torch, v)
    _check(torch, h, v, None, "opening", 1, 0, dev=dv)
    _check(torch, h, v, ball(2), "opening", 1, 0, dev=dv)


def test_mask_arguments(torch_cuda, h):
    torch = torch_cuda
    for f in (h.binary_erosion, h.binary_dilation, h.binary_opening, h.binary_closing):
        with pytest.raises(TypeError, match="mask: unsupported dtype"):
            f(torch.zeros(8, 8, device="cuda"))
        with pytest.raises(TypeError, match="mask: unsupported dtype"):
            f(torch.zeros(8, 8, dtype=torch.int32, device="cuda"))
        with pytest.raises(ValueError, match="2-D image or a 3-D volume"):
            f(torch.zeros(8, dtype=torch.bool, device="cuda"))
        with pytest.raises(ValueError, match="2-D image or a 3-D volume"):
            f(torch.zeros(2, 3, 4, 5, dtype=torch.bool, device="cuda"))
        with pytest.raises(ValueError, match="mask is empty"):
            f(torch.zeros(0, 5, dtype=torch.bool, device="cuda"))
        with pytest.raises(ValueError, match="no CPU path"):
            f(torch.zeros(8, 8, dtype=torch.bool))
        with pytest.raises(RuntimeError, match="structure and input must have same dimensionality"):
            f(torch.zeros(8, 8, dtype=torch.bool, device="cuda"), np.ones((3, 3, 3)))
        with pytest.raises(ValueError, match="iterations must be >= 1"):
            f(torch.zeros(8, 8, dtype=torch.bool, device="cuda"), iterations=0)


def test_workspace_contents_do_not_matter_and_calls_repeat(torch_cuda, h):
    torch = torch_cuda
    lib = h.lib()
    m = np.random.default_rng(10).random((300, 250)) < 0.5
    dev = _cuda(torch, m).view(torch.uint8)
    s = np.ascontiguousarray(disk(4).astype(np.uint8))
    want = _want("dilation", m, s, 3, 1)
    ws = lib.hipr_morphology_workspace_bytes(2, 300, 250, 1, 3)
    assert ws >= 300 * 250
    outs = []
    for fill in (0x00, 0xFF, 0x00, 0xFF):
        work = torch.full((ws,), fill, dtype=torch.uint8, device="cuda")
        out = torch.full(m.shape, 0xAB, dtype=torch.uint8, device="cuda")
        assert lib.hipr_binary_morphology(C.c_void_p(dev.data_ptr()), 2, 300, 250, 1, s.ctypes.data_as(C.c_void_p),
                                          9, 9, 1, 1, 1, 3, C.c_void_p(work.data_ptr()), ws,
                                          C.c_void_p(out.data_ptr()), None) == 0
        outs.append(out.cpu().numpy())
    for o in outs:
        assert np.array_equal(o, want.astype(np.uint8))
    # a workspace one byte short is refused before anything is launched
    assert lib.hipr_binary_morphology(C.c_void_p(dev.data_ptr()), 2, 300, 250, 1, s.ctypes.data_as(C.c_void_p),
                                      9, 9, 1, 1, 1, 3, C.c_void_p(work.data_ptr()), ws - 1,
                                      C.c_void_p(out.data_ptr()), None) == -7
    first = h.binary_closing(_cuda(torch, m), disk(3), 2)
    for _ in range(3):
        assert torch.equal(h.binary_closing(_cuda(torch, m), disk(3), 2), first)


def test_launches_and_no_host_copy(torch_cuda, h):
    """One launch per pass: iterations per erosion or dilation, twice that for opening and closing; no device-to-host
    copy."""
    torch = torch_cuda
    from torch.profiler import ProfilerActivity, profile
    lib = h.lib()
    m = _cuda(torch, np.random.default_rng(11).random((2048, 2048)) < 0.5)
    cases = (("erosion", 1, 1), ("dilation", 3, 3), ("opening", 2, 4), ("closing", 5, 10))
    for op, it, launches in cases:
        f = getattr(h, "binary_" + op)
        f(m, disk(2), it)                                       # warm-up
        torch.cuda.synchronize()
        before = lib.hipr_launch_count()
        f(m, disk(2), it)
        assert lib.hipr_launch_count() - before == launches, op
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:  # one profiling cycle for all four operators
        for op, it, _ in cases:
            getattr(h, "binary_" + op)(m, disk(2), it)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert not any("DtoH" in n or "Device -> Host" in n for n in names), names
    # the exact count is hipr_launch_count's above: after earlier profiling in the same process, CUPTI can drop a
    # kernel record while it requests an activity buffer, so the trace bounds the count only from above
    kernels = [n for n in names if "morphology_kernel" in n]
    assert 0 < len(kernels) <= sum(c[2] for c in cases), (len(kernels), sorted(set(names)))


def test_segmentation_chain_with_opening(torch_cuda, h):
    """2048^2 FOV: score -> k-means mask -> binary_opening -> remove_small_objects -> binary_fill_holes -> label, and
    the same chain on the host (scipy.ndimage.binary_opening, tests/label_oracle.py) from the same mask."""
    torch = torch_cuda
    from hipr_b200 import synth
    cube, _, _ = synth.make_fov(2048, 2048, 95, fov_index=3)
    score = h.neighbor2d_score(cube.cuda(), "F1")
    mask = h.kmeans_threshold(score, 2).mask
    for s in (None, disk(1)):
        opened = h.binary_opening(mask, s)
        kept = h.remove_small_objects(opened, 20)
        filled = h.binary_fill_holes(kept)
        lab, n = h.label(filled, connectivity=1, return_num=True)

        m = mask.cpu().numpy()
        o = ndi.binary_opening(m, s)
        assert np.array_equal(opened.cpu().numpy(), o)
        want, wn = label_oracle.label_mask(
            label_oracle.binary_fill_holes(label_oracle.remove_small_objects_mask(o, 20, 1)), 1)
        assert n == wn and wn > 0
        assert np.array_equal(lab.cpu().numpy(), want)
