"""GPU parity, 3-D path (bio/neighbor.pyx) against the oracle."""
import hashlib
import os

import numpy as np
import pytest

from conftest import smooth_image

pytestmark = pytest.mark.gpu
RTOL, ATOL_F32, ATOL_F64 = 1e-5, 2e-6, 1e-12
GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors.npz"))


def _cuda(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _golden_padded_volume():
    """The padded input the reference stencils were run on for tests/golden/reference_vectors.npz."""
    vol = GOLD["vol3d"]
    return np.pad(vol / vol.max(), 5, mode="edge")


@pytest.mark.parametrize("shape,params", [((3, 4, 5), (11, 9, 9)), ((9, 8, 33), (11, 9, 9)), ((6, 5, 7), (7, 5, 4)),
                                           ((4, 4, 4), (5, 3, 3)), ((5, 6, 4), (9, 6, 7))])
def test_line_profile_v2_bit_exact(torch_cuda, oracle, shape, params):
    import neighbor
    P = params[0]
    a = np.random.default_rng(1).random(tuple(s + P - 1 for s in shape))
    got = neighbor.line_profile_v2(a, *params)
    want = oracle.line_profile_v2(a, *params)
    assert got.shape == want.shape and got.dtype == np.float64
    assert np.array_equal(got, want)


def test_line_profile_v2_vs_compiled_reference(torch_cuda):
    """Against the output of the unmodified reference stencil, stored in tests/golden/reference_vectors.npz."""
    import neighbor
    lp = neighbor.line_profile_v2(_golden_padded_volume(), 11, 9, 9)
    assert hashlib.sha256(lp.tobytes()).digest() == GOLD["lp3d_sha256"].tobytes()


@pytest.mark.parametrize("shape,params", [((9, 10, 40), (11, 9, 9)), ((4, 3, 5), (11, 9, 9)), ((6, 5, 7), (7, 5, 4)),
                                           ((5, 6, 4), (9, 6, 7))])
def test_memory_efficient_v2(torch_cuda, oracle, shape, params):
    import neighbor
    P = params[0]
    a = smooth_image(tuple(s + P - 1 for s in shape), 3).astype(np.float64)
    got = neighbor.line_profile_memory_efficient_v2(a, *params)
    want = oracle.line_profile_memory_efficient_v2(a, *params)
    assert got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-15)


def test_memory_efficient_v2_vs_compiled_reference(torch_cuda):
    import neighbor
    got = neighbor.line_profile_memory_efficient_v2(_golden_padded_volume(), 11, 9, 9)
    np.testing.assert_allclose(got, GOLD["me2_3d"], rtol=1e-12, atol=1e-15)


def test_memory_efficient_v2_host_bands(torch_cuda):
    """hipr_lne3d_dirs_host: several bands of x-planes, pageable / page-locked / caller's output, all bit-identical to
    the device operator on the whole volume (which the tests above hold against the oracle and the compiled reference)."""
    import hipr_b200
    a = smooth_image((50, 70, 60), 9).astype(np.float64)          # (40, 60, 50, 72) float64 = 69 MB: 3 bands
    want = hipr_b200.lne3d_dirs(_cuda(torch_cuda, a), 11, 9, 9, padded=True).cpu().numpy()
    got = hipr_b200.lne3d_dirs_host(a, 11, 9, 9)
    assert got.shape == (40, 60, 50, 72) and np.array_equal(got, want)
    assert np.array_equal(hipr_b200.lne3d_dirs_host(a, 11, 9, 9, pinned=True), want)
    out = np.full(want.shape, -1.0)
    assert hipr_b200.lne3d_dirs_host(a, 11, 9, 9, out=out) is out and np.array_equal(out, want)
    with pytest.raises(TypeError):
        hipr_b200.lne3d_dirs_host(a.astype(np.float32), 11, 9, 9)


def test_line_profile_v2_host_bands(torch_cuda):
    """hipr_line_profile_3d_host: several bands of x-planes (6,336 B per voxel), bit-identical to the device operator."""
    import hipr_b200
    a = smooth_image((34, 40, 42), 12).astype(np.float64)          # (24, 30, 32, 72, 11) float64 = 146 MB: 5 bands
    want = hipr_b200.line_profile_3d(_cuda(torch_cuda, a), 11, 9, 9).cpu().numpy()
    got = hipr_b200.line_profile_3d_host(a, 11, 9, 9)
    assert got.shape == (24, 30, 32, 72, 11) and np.array_equal(got, want)
    assert np.array_equal(hipr_b200.line_profile_3d_host(a, 11, 9, 9, pinned=True), want)


def test_memory_efficient_v2_flat_lines_clamped(torch_cuda, oracle):
    import neighbor
    a = np.full((15, 15, 15), 0.5)
    a[7, 7, 7] = 0.5 + 1e-9
    got = neighbor.line_profile_memory_efficient_v2(a, 11, 9, 9)
    want = oracle.line_profile_memory_efficient_v2(a, 11, 9, 9)
    assert not np.isnan(got).any()
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-15)


@pytest.mark.parametrize("flavour", ["F2", "F3", "ME2"])
@pytest.mark.parametrize("dtype_name", ["float32", "float64"])
def test_lne3d(torch_cuda, oracle, flavour, dtype_name):
    import hipr_b200
    vol = smooth_image((12, 17, 40), 5)
    v = vol.astype(np.float64) if dtype_name == "float64" else vol
    got = hipr_b200.lne3d(_cuda(torch_cuda, v), flavour).cpu().numpy()
    want = oracle.lne3d(vol.astype(np.float64), flavour)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_F64 if dtype_name == "float64" else ATOL_F32)


@pytest.mark.parametrize("flavour", ["F2", "F3", "ME2"])
def test_lne3d_generic_parameters(torch_cuda, oracle, flavour):
    import hipr_b200
    vol = smooth_image((9, 8, 11), 6).astype(np.float64)
    got = hipr_b200.lne3d(_cuda(torch_cuda, vol), flavour, 7, 5, 4).cpu().numpy()
    want = oracle.lne3d(vol, flavour, 7, 5, 4)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_F64)


def test_memory_efficient_v3(torch_cuda, oracle):
    """v3 reads outside its patch (flat addressing).  On a smooth volume: equal to the oracle, NaN exactly where
    the reference's read leaves the buffer.  On the input of tests/golden/reference_vectors.npz: equal to the
    compiled reference's stored output on the first 6 rows, whose reads stay in the buffer."""
    import neighbor
    a = smooth_image((24, 15, 14), 7).astype(np.float64)
    got = neighbor.line_profile_memory_efficient_v3(a, 11, 9, 9)
    want = oracle.line_profile_memory_efficient_v3(a, 11, 9, 9)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-12, equal_nan=True)
    assert (~np.isnan(got)).any()          # the comparison above is not over NaN alone
    got = neighbor.line_profile_memory_efficient_v3(GOLD["v3_in"], 11, 9, 9)[:6]
    assert not np.isnan(got).any()
    np.testing.assert_allclose(got, GOLD["v3_out"], rtol=1e-9, atol=1e-12)


def test_neighbor3d_score_pipeline(torch_cuda, oracle):
    import hipr_b200
    from hipr_b200 import synth
    cube = synth.make_volume_cube(10, 12, 36, 95, seed=5)
    got = hipr_b200.neighbor3d_score(cube.cuda(), "ME2", dtype=torch_cuda.float64).cpu().numpy()
    s, _ = oracle.prologue(cube.numpy())
    want = oracle.lne3d(s / s.max(), "ME2")
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL_F64)


def test_dead_functions_fail_like_the_reference(torch_cuda):
    import neighbor
    with pytest.raises(ValueError, match="Buffer dtype mismatch"):
        neighbor.neighbor_average(np.zeros((30, 30, 30), np.float32), 11)
    with pytest.raises(ValueError, match="Buffer dtype mismatch"):
        neighbor.line_profile(np.zeros((12, 12, 12)), 11, 9, 9)


@pytest.mark.parametrize("flavour", ["F2", "F3", "ME2"])
@pytest.mark.parametrize("shape", [(3, 4, 5), (12, 17, 40), (9, 8, 33)])
def test_lne3d_fixed_point(torch_cuda, oracle, flavour, shape):
    """Fixed-point 3-D stencil on a float64 (already normalised) volume against the float64 oracle."""
    import hipr_b200
    vol = smooth_image(shape, 31).astype(np.float64) + 0.1
    vol /= vol.max()
    got = hipr_b200.lne3d_fixed(_cuda(torch_cuda, vol), flavour).cpu().numpy()
    want = oracle.lne3d(vol, flavour)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=5e-7, equal_nan=True)


def test_lne3d_fixed_point_dirs_and_pipeline(torch_cuda, oracle):
    import hipr_b200
    from hipr_b200 import synth
    vol = smooth_image((16, 15, 44), 32).astype(np.float64)
    vol /= vol.max()
    vp = np.pad(vol, 5, mode="edge")
    got = hipr_b200.lne3d_fixed(_cuda(torch_cuda, vp), "ME2", padded=True, dirs_only=True).cpu().numpy()
    want = oracle.line_profile_memory_efficient_v2(vp, 11, 9, 9)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=5e-7)
    cube = synth.make_volume_cube(10, 12, 36, 95, seed=6)
    s, _ = oracle.prologue(cube.numpy())
    for fl in ("ME2", "F2", "F3"):
        got = hipr_b200.neighbor3d_score(cube.cuda(), fl).cpu().numpy()
        assert got.dtype == np.float32
        np.testing.assert_allclose(got, oracle.lne3d(s / s.max(), fl), rtol=RTOL, atol=5e-7)
    assert hipr_b200.lne3d_fixed(_cuda(torch_cuda, vol), "ME2", 7, 5, 4) is None


@pytest.mark.parametrize("flavour", ["ME2", "F2", "F3"])
def test_neighbor3d_host_entry_point(torch_cuda, oracle, flavour):
    """hipr_neighbor3d_host: numpy z-stack cube in, numpy score volume out == the device-resident pipeline, bit for
    bit, and the oracle within the gate."""
    import hipr_b200
    from hipr_b200 import synth
    cube = synth.make_volume_cube(20, 24, 40, 95, seed=3).numpy()
    got = hipr_b200.neighbor3d_score_host(cube, flavour)
    dev = hipr_b200.neighbor3d_score(torch_cuda.from_numpy(cube).cuda(), flavour).cpu().numpy()
    assert np.array_equal(got, dev)
    s = cube.astype(np.float64).sum(axis=3)
    want = oracle.lne3d(s / s.max(), flavour)
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=5e-7)
    with pytest.raises(ValueError):
        hipr_b200.neighbor3d_score_host(cube[0], flavour)


@pytest.mark.parametrize("flavour", ["ME2", "F2", "F3"])
def test_score3d_strict_relative_parity(torch_cuda, oracle, flavour):
    """1e-5 RELATIVE, no absolute term (north_star's gate as written), on a z-stack cube through the default
    fixed-point pipeline: voxels the grid cannot resolve are recomputed in float64 (lne3d_refine_kernel); a batch of
    two stacks (two streams) gives the same volumes."""
    import hipr_b200
    from hipr_b200 import synth
    cube = synth.make_volume_cube(24, 20, 40, 95, seed=11)
    cube = cube + 0.01 * torch_cuda.rand((24, 20, 40, 1), generator=torch_cuda.Generator().manual_seed(3))
    s = cube.numpy().astype(np.float64).sum(axis=3)
    want = oracle.lne3d(s / s.max(), flavour)
    got = hipr_b200.neighbor3d_score(cube.cuda(), flavour)
    assert bool((got >= 0).all() | torch_cuda.isnan(got).any()), "a refinement sentinel survived"
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-5, atol=0, equal_nan=True)
    both = hipr_b200.neighbor3d_score(torch_cuda.stack([cube, cube * 0.5]).cuda(), flavour)
    assert torch_cuda.equal(both[0], got)
    np.testing.assert_allclose(both[1].cpu().numpy(), want, rtol=1e-5, atol=0, equal_nan=True)


def test_dirs3d_strict_relative_parity(torch_cuda, oracle):
    """line_profile_memory_efficient_v2's (X, Y, Z, 72) output from the fixed-point stencil: every value within 1e-5
    relative (values the grid cannot resolve are recomputed in float64, lne3d_refine_dirs_kernel)."""
    import hipr_b200
    vol = smooth_image((14, 13, 38), 33).astype(np.float64) + 0.05
    vol /= vol.max()
    vp = np.pad(vol, 5, mode="edge")
    got = hipr_b200.lne3d_fixed(_cuda(torch_cuda, vp), "ME2", padded=True, dirs_only=True).cpu().numpy()
    want = oracle.line_profile_memory_efficient_v2(vp, 11, 9, 9)
    assert (got >= 0).all()
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=0)
