"""GPU parity of the registration-shift kernels (csrc/xcorr2d.cu) against the numpy restatement of
skimage.feature.register_translation (tests/shift_oracle.py: register_translation, excitation_shifts)."""
import ctypes as C

import numpy as np
import pytest

import shift_oracle
from test_shifts import CHANS, WINDOW_CASES, shifted_stacks

pytestmark = pytest.mark.gpu


def _images(shape, seed, roll=(0, 0)):
    rng = np.random.default_rng(seed)
    src = rng.random(shape)
    src[: shape[0] // 3, : shape[1] // 5] += 1.0                      # one dominant structure: a clear peak
    target = np.roll(src, roll, axis=(0, 1)) + 0.05 * rng.random(shape)
    return src, target


def _gap(acc):
    top = np.partition(acc.ravel(), -2)[-2:]
    return (top[1] - top[0]) / top[1]


@pytest.mark.parametrize("shape", [(16, 16), (32, 64), (64, 8192), (8192, 64), (256, 1024), (2048, 2048)])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_correlation_map_matches_numpy(torch_cuda, shape, dtype):
    import hipr_b200
    src, target = _images(shape, sum(shape), roll=(shape[0] // 7, -(shape[1] // 9)))
    src, target = src.astype(dtype), target.astype(dtype)
    want_shift, want_acc = shift_oracle.register_translation(src, target, return_correlation=True)
    shift, corr = hipr_b200.register_translation(torch_cuda.from_numpy(src).cuda(), torch_cuda.from_numpy(target).cuda(),
                                                 return_correlation=True)
    acc = corr.cpu().numpy()
    assert corr.dtype == torch_cuda.float64 and acc.shape == shape
    assert np.max(np.abs(acc - want_acc)) <= 1e-11 * want_acc.max()
    assert _gap(want_acc) > 1e-9
    assert isinstance(shift, np.ndarray) and shift.dtype == np.float64 and shift.shape == (2,)
    assert np.array_equal(shift, want_shift)


@pytest.mark.parametrize("shape,rolls", [
    ((8, 8), [(0, 0), (1, -1), (3, 3), (4, 4), (5, -4), (-3, 2)]),
    ((2, 4), [(0, 1), (1, 2), (1, 3)]),
    ((64, 32), [(31, 15), (32, 16), (33, 17), (-31, -15), (0, 16), (63, 31)]),
    ((128, 512), [(7, -200), (64, 256), (-64, -256), (65, 257), (1, 1)]),
    ((4096, 16), [(2047, 7), (2048, 8), (-2047, -7), (3, 0)]),
])
def test_register_translation_equals_oracle(torch_cuda, shape, rolls):
    import hipr_b200
    for k, roll in enumerate(rolls):
        src, target = _images(shape, 100 + k, roll)
        want, acc = shift_oracle.register_translation(src, target, return_correlation=True)
        assert _gap(acc) > 1e-9, roll
        got = hipr_b200.register_translation(torch_cuda.from_numpy(src).cuda(), torch_cuda.from_numpy(target).cuda())
        assert np.array_equal(got, want), (roll, got, want)


@pytest.mark.parametrize("transform,eps", [(None, 0.0), ("log", 1.0), ("log", 0.0)])
@pytest.mark.parametrize("case", range(len(WINDOW_CASES)))
def test_excitation_shifts_equal_oracle(torch_cuda, transform, eps, case):
    import hipr_b200
    H, W, offsets, chans, fov = WINDOW_CASES[case]
    stacks = shifted_stacks(H, W, offsets, chans, fov)
    want = shift_oracle.excitation_shifts(stacks, transform, eps)
    got = hipr_b200.excitation_shifts([torch_cuda.from_numpy(s).cuda() for s in stacks], transform=transform, eps=eps)
    assert got.dtype == np.float64 and got.shape == (len(stacks), 2)
    assert np.array_equal(got, want)
    assert np.array_equal(got[0], [0.0, 0.0])
    if eps > 0 or transform is None:                  # see test_shifts.WINDOW_CASES for log with eps = 0
        assert np.array_equal(got, np.asarray(offsets, dtype=np.float64))


def test_excitation_shifts_full_size(torch_cuda):
    """One 2048 x 2048 x 95 field of view in the reference's five-excitation layout."""
    import hipr_b200
    offsets = [(0, 0), (2, -3), (-11, 7), (5, 0), (-1, 24)]
    stacks = shifted_stacks(2048, 2048, offsets, CHANS, 4)
    dev = [torch_cuda.from_numpy(s).cuda() for s in stacks]
    for transform, eps in ((None, 0.0), ("log", 1.0)):
        got = hipr_b200.excitation_shifts(dev, transform=transform, eps=eps)
        assert np.array_equal(got, shift_oracle.excitation_shifts(stacks, transform, eps))
        assert np.array_equal(got, np.asarray(offsets, dtype=np.float64))


def test_edge_semantics_on_device(torch_cuda):
    import hipr_b200
    t = torch_cuda
    const = t.full((32, 64), 3.5, dtype=t.float64, device="cuda")
    shift, corr = hipr_b200.register_translation(const, const, return_correlation=True)
    assert np.array_equal(shift, [0.0, 0.0])                                 # every |cc| equal: lowest index
    assert t.unique(corr).numel() == 1
    rng = np.random.default_rng(3)
    base = rng.random((32, 32, 4), dtype=np.float32) + 0.5
    stacks = [base, np.ascontiguousarray(np.roll(base[:, :, :3], (4, -3), axis=(0, 1)))]
    stacks[1][5, 6, :] = 0.0                                                  # log(0) = -inf: NaN everywhere
    dev = [t.from_numpy(s).cuda() for s in stacks]
    assert np.array_equal(hipr_b200.excitation_shifts(dev, "log", 0.0), [[0, 0], [0, 0]])
    assert np.array_equal(hipr_b200.excitation_shifts(dev, "log", 1e-3), [[0, 0], [-4, 3]])
    img = rng.random((16, 8))
    for roll, want in (((8, 4), [8.0, 4.0]), ((9, 5), [7.0, 3.0]), ((7, 3), [-7.0, -3.0])):
        got = hipr_b200.register_translation(t.from_numpy(img).cuda(), t.from_numpy(np.roll(img, roll, axis=(0, 1))).cuda())
        assert np.array_equal(got, want), roll
    one = hipr_b200.excitation_shifts([dev[0]])
    assert np.array_equal(one, [[0.0, 0.0]])


def test_score_from_stacks_with_estimated_shifts(torch_cuda):
    import hipr_b200
    offsets = [(0, 0), (1, -2), (-3, 0), (0, 4), (2, 2)]
    stacks = shifted_stacks(128, 128, offsets, CHANS, 5)
    dev = [torch_cuda.from_numpy(s).cuda() for s in stacks]
    shifts = shift_oracle.excitation_shifts(stacks)
    score, cube, s64, _ = hipr_b200.neighbor2d_score_from_stacks(dev, shifts="estimate")
    want_score, want_cube, want_s64, _ = hipr_b200.neighbor2d_score_from_stacks(dev, shifts=shifts)
    assert torch_cuda.equal(score, want_score) and torch_cuda.equal(cube, want_cube) and torch_cuda.equal(s64, want_s64)
    cube2, s2, _ = hipr_b200.register_stacks(dev, shifts="estimate")
    assert torch_cuda.equal(cube2, want_cube) and torch_cuda.equal(s2, want_s64)


def test_side_stream_and_repeatability(torch_cuda):
    import hipr_b200
    t = torch_cuda
    H, W, offsets, chans, fov = WINDOW_CASES[3]
    stacks = shifted_stacks(H, W, offsets, chans, fov)
    want = shift_oracle.excitation_shifts(stacks, None)
    side = t.cuda.Stream()
    with t.cuda.stream(side):
        dev = [t.from_numpy(s).to("cuda", non_blocking=False) for s in stacks]
        a = hipr_b200.excitation_shifts(dev, transform=None)
        b = hipr_b200.excitation_shifts(dev, transform=None)
        src, target = _images((256, 128), 7, (5, -9))
        s1, c1 = hipr_b200.register_translation(t.from_numpy(src).cuda(), t.from_numpy(target).cuda(), True)
        s2, c2 = hipr_b200.register_translation(t.from_numpy(src).cuda(), t.from_numpy(target).cuda(), True)
    assert np.array_equal(a, want) and np.array_equal(a, b)
    assert np.array_equal(s1, s2) and t.equal(c1, c2) and np.array_equal(s1, [-5.0, 9.0])


def test_argument_errors(torch_cuda):
    import hipr_b200
    from hipr_b200 import lib
    t = torch_cuda
    a = t.zeros((48, 64), dtype=t.float64, device="cuda")
    with pytest.raises(ValueError, match="power of two"):
        hipr_b200.register_translation(a, a)
    with pytest.raises(ValueError, match="power of two"):
        hipr_b200.excitation_shifts([t.zeros((64, 100, 3), device="cuda")])
    with pytest.raises(ValueError, match="power of two"):
        hipr_b200.neighbor2d_score_from_stacks([t.zeros((40, 64, 3), device="cuda")] * 2, shifts="estimate")
    b = t.zeros((64, 64), dtype=t.float64, device="cuda")
    with pytest.raises(ValueError):
        hipr_b200.register_translation(b, t.zeros((64, 32), dtype=t.float64, device="cuda"))
    with pytest.raises(TypeError):
        hipr_b200.register_translation(b, b.float())
    with pytest.raises(TypeError):
        hipr_b200.register_translation(b.int(), b.int())
    with pytest.raises(ValueError):
        hipr_b200.excitation_shifts([t.zeros((64, 64, 3), device="cuda"), t.zeros((64, 32, 3), device="cuda")])
    with pytest.raises(TypeError):
        hipr_b200.excitation_shifts([t.zeros((64, 64, 3), dtype=t.float64, device="cuda")])
    with pytest.raises(ValueError):
        hipr_b200.excitation_shifts([])
    with pytest.raises(ValueError):
        hipr_b200.excitation_shifts([t.zeros((64, 64, 3), device="cuda")], transform="log10")
    with pytest.raises(ValueError):
        hipr_b200.register_stacks([t.zeros((64, 64, 3), device="cuda")], shifts="guess")
    # the C ABI directly: a workspace one byte short, and an unsupported size
    need = lib().hipr_xcorr2d_workspace_bytes(64, 64, 2)
    work = t.empty(need, dtype=t.uint8, device="cuda")
    out = t.empty(2, dtype=t.float64, device="cuda")
    stream = C.c_void_p(t.cuda.current_stream().cuda_stream)
    args = (C.c_void_p(b.data_ptr()), C.c_void_p(b.data_ptr()), 1, 64, 64, C.c_void_p(work.data_ptr()))
    assert lib().hipr_register_translation_2d(*args, need - 1, C.c_void_p(out.data_ptr()), None, stream) == -7
    assert lib().hipr_register_translation_2d(*args, need, C.c_void_p(out.data_ptr()), None, stream) == 0
    assert lib().hipr_register_translation_2d(C.c_void_p(b.data_ptr()), C.c_void_p(b.data_ptr()), 1, 64, 48,
                                              C.c_void_p(work.data_ptr()), need, C.c_void_p(out.data_ptr()), None,
                                              stream) == -9
    st = t.zeros((64, 64, 3), device="cuda")
    ptrs = (C.c_void_p * 2)(st.data_ptr(), st.data_ptr())
    chans = np.array([3, 3], dtype=np.int32)
    need2 = lib().hipr_xcorr2d_workspace_bytes(64, 64, 2)
    assert lib().hipr_excitation_shifts(ptrs, chans.ctypes.data_as(C.c_void_p), 2, 64, 64, 1, 0.0,
                                        C.c_void_p(work.data_ptr()), need2 - 256, C.c_void_p(out.data_ptr()), stream) == -7
    t.cuda.synchronize()
