"""CPU checks of the registration-shift oracle (register_translation, excitation_shifts) and of the host side of
the device operators that reproduce it (csrc/xcorr2d.cu).  No device call is made here."""
import numpy as np
import pytest

import shift_oracle

CHANS = (32, 23, 20, 14, 6)


def brute_force_correlation(src, target):
    """|cc| of the circular cross-correlation without an FFT: cc[dr, dc] = sum_z src[z + (dr, dc)] * target[z]."""
    H, W = src.shape
    cc = np.empty((H, W))
    for dr in range(H):
        for dc in range(W):
            cc[dr, dc] = np.sum(np.roll(src, (-dr, -dc), axis=(0, 1)) * target)
    return np.abs(cc)


def shifted_stacks(H, W, offsets, chans=CHANS, fov_index=0):
    """Excitation stacks cut from one synthetic FOV at windows displaced by `offsets` (row, col) from the first:
    stack e sees the scene at (r + offsets[e][0], c + offsets[e][1]), so register_translation(sum_0, sum_e) must
    find offsets[e] (a non-circular shift: the windows overlap only in part).  Every cell also carries 0.1 per
    channel, so that it shows in every excitation (the synthetic barcodes leave many cells dark in some)."""
    from hipr_b200 import synth
    m = max(max(abs(a), abs(b)) for a, b in offsets)
    cube, labels, _ = synth.make_fov(H + 2 * m, W + 2 * m, sum(chans), fov_index=fov_index)
    cube = cube.numpy() + np.float32(0.1) * (labels.numpy() > 0)[..., None]
    edges = np.cumsum((0,) + tuple(chans))
    return [np.ascontiguousarray(cube[m + a:m + a + H, m + b:m + b + W, edges[e]:edges[e + 1]])
            for e, (a, b) in enumerate(offsets)]


@pytest.mark.parametrize("shape", [(8, 8), (12, 20), (16, 32), (1, 16)])
def test_oracle_equals_brute_force_correlation(shape):
    rng = np.random.default_rng(sum(shape))
    src = rng.random(shape)
    target = np.roll(src, (shape[0] // 3, -(shape[1] // 4)), axis=(0, 1)) + 0.1 * rng.random(shape)
    shift, acc = shift_oracle.register_translation(src, target, return_correlation=True)
    want = brute_force_correlation(src, target)
    np.testing.assert_allclose(acc, want, rtol=0, atol=1e-12 * want.max())
    peak = np.array(np.unravel_index(np.argmax(want), shape), dtype=np.float64)
    for ax, n in enumerate(shape):
        if peak[ax] > n // 2:
            peak[ax] -= n
        if n == 1:
            peak[ax] = 0
    assert np.array_equal(shift, peak)
    # the circular roll by (k, l) is found as (-k, -l), wrapped
    assert np.array_equal(shift_oracle.register_translation(src, np.roll(src, (1, 2), axis=(0, 1))),
                          [-1.0 if shape[0] > 1 else 0.0, -2.0])


# Known offsets the plain (unwindowed) cross-correlation recovers on these scenes.  Two limits of the algorithm
# itself, seen with the oracle: offsets near half the frame (overlap of half the window or less) lock onto the
# periodic cell grid, and log(sum) with eps = 0 is negative on the dim 6-channel excitation's background, which
# turns the correlation's sign over most of the frame; eps = 1 keeps the log positive.
WINDOW_CASES = [
    (64, 64, [(0, 0), (3, -5), (-7, 0), (0, 8), (-8, 6)], CHANS, 0),
    (128, 64, [(0, 0), (-9, 2), (17, -7), (13, 8), (-1, -1)], CHANS, 1),
    (32, 128, [(0, 0), (-4, 2), (3, -16), (4, 11)], CHANS[1:], 2),
    (256, 256, [(0, 0), (2, -3), (-31, 20), (25, -9), (1, 40)], CHANS, 3),
]


@pytest.mark.parametrize("transform,eps", [(None, 0.0), ("log", 1.0)])
@pytest.mark.parametrize("case", range(len(WINDOW_CASES)))
def test_oracle_recovers_window_offsets(transform, eps, case):
    H, W, offsets, chans, fov = WINDOW_CASES[case]
    got = shift_oracle.excitation_shifts(shifted_stacks(H, W, offsets, chans, fov), transform=transform, eps=eps)
    assert got.dtype == np.float64 and got.shape == (len(offsets), 2)
    assert np.array_equal(got, np.asarray(offsets, dtype=np.float64))


def test_oracle_edge_semantics():
    const = np.full((16, 16), 3.5)
    assert np.array_equal(shift_oracle.register_translation(const, const), [0.0, 0.0])        # all ties: lowest index
    rng = np.random.default_rng(1)
    base = rng.random((32, 32, 4), dtype=np.float32) + 0.5
    stacks = [base, np.ascontiguousarray(np.roll(base[:, :, :3], (4, -3), axis=(0, 1)))]
    assert np.array_equal(shift_oracle.excitation_shifts(stacks, "log"), [[0, 0], [-4, 3]])
    stacks[1][5, 6, :] = 0.0                                                             # log(0) = -inf -> NaN cc
    assert np.array_equal(shift_oracle.excitation_shifts(stacks, "log", eps=0.0), [[0, 0], [0, 0]])
    assert np.array_equal(shift_oracle.excitation_shifts(stacks, "log", eps=1e-3), [[0, 0], [-4, 3]])
    img = rng.random((16, 8))
    assert np.array_equal(shift_oracle.register_translation(img, np.roll(img, (8, 4), axis=(0, 1))), [8.0, 4.0])   # n / 2
    assert np.array_equal(shift_oracle.register_translation(img, np.roll(img, (9, 5), axis=(0, 1))), [7.0, 3.0])
    line = rng.random((1, 16))
    assert np.array_equal(shift_oracle.register_translation(line, np.roll(line, 3, axis=1)), [0.0, -3.0])
    with pytest.raises(ValueError):
        shift_oracle.register_translation(img, img.T)


def test_workspace_size_rules():
    import hipr_b200
    ws = hipr_b200.lib().hipr_xcorr2d_workspace_bytes
    a = ws(2048, 2048, 5)
    assert a >= 5 * 2048 * 2048 * 24                      # float64 sums + complex128 spectra
    assert ws(2048, 2048, 2) < a and ws(2048, 1024, 5) < a
    assert ws(2, 2, 2) > 0 and ws(8192, 8192, 1) > 0 and ws(2, 8192, 8) > 0
    for H, W in [(2048, 2000), (1, 16), (16, 1), (0, 16), (16384, 16), (-4, 4), (96, 64), (64, 3)]:
        assert ws(H, W, 2) < 0, (H, W)
    assert ws(16, 16, 0) < 0 and ws(16, 16, 9) < 0


def test_operators_refuse_cpu_tensors():
    torch = pytest.importorskip("torch")
    import hipr_b200
    img = torch.zeros((16, 16), dtype=torch.float64)
    with pytest.raises(ValueError, match="no CPU path"):
        hipr_b200.register_translation(img, img)
    with pytest.raises(ValueError, match="no CPU path"):
        hipr_b200.excitation_shifts([torch.zeros((16, 16, 3))])
    with pytest.raises(ValueError, match="no CPU path"):
        hipr_b200.register_stacks([torch.zeros((16, 16, 3))], shifts="estimate")
