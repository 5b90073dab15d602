"""Binary morphology (K12) without a device: the default structure, the run table the kernel is given, and the checks
of the structure and of `iterations` (classes and messages as scipy.ndimage's where scipy has them)."""
import numpy as np
import pytest
import scipy.ndimage as ndi


@pytest.fixture(scope="module")
def ops():
    from hipr_b200 import ops
    return ops


def _disk(r):
    y, x = np.mgrid[-r:r + 1, -r:r + 1]
    return (x * x + y * y <= r * r).astype(np.uint8)


def _ball(r):
    z, y, x = np.mgrid[-r:r + 1, -r:r + 1, -r:r + 1]
    return (x * x + y * y + z * z <= r * r).astype(np.uint8)


def _rebuild(runs, shape):
    """The structure a run table describes."""
    s3 = (1,) * (3 - len(shape)) + tuple(shape)
    out = np.zeros(s3, dtype=np.uint8)
    c = [n // 2 for n in s3]
    for d0, d1, a, b in runs:
        out[d0 + c[0], d1 + c[1], a + c[2]:b + c[2] + 1] = 1
    return out.reshape(shape)


@pytest.mark.parametrize("ndim", [2, 3])
def test_default_structure_is_scipys_cross(ops, ndim):
    s = ops._structure(None, ndim)
    assert s.dtype == np.uint8 and s.flags.c_contiguous
    assert np.array_equal(s, ndi.generate_binary_structure(ndim, 1))


def _structures():
    rng = np.random.default_rng(12)
    out = [_disk(r) for r in range(1, 16)] + [_ball(r) for r in (1, 2, 3, 7, 15)]
    out += [ndi.generate_binary_structure(n, c).astype(np.uint8) for n in (2, 3) for c in range(1, n + 1)]
    out += [np.ones((31, 31), np.uint8), np.ones((31, 31, 31), np.uint8), np.zeros((3, 3), np.uint8),
            np.ones((1, 1), np.uint8), np.ones((1, 31), np.uint8), np.ones((31, 1, 1), np.uint8)]
    for shape in [(3, 5), (7, 1), (31, 31), (1, 31), (5, 3, 7), (9, 9, 9), (1, 1, 31)]:
        for p in (0.3, 0.5, 0.8):
            out.append((rng.random(shape) < p).astype(np.uint8))
    return out


def test_run_table_reconstructs_the_structure(ops):
    for s in _structures():
        runs = ops._structure_runs(ops._structure(s, s.ndim))
        assert runs.dtype == np.int32 and runs.shape[1] == 4
        assert np.array_equal(_rebuild(runs, s.shape), s), s.shape
        # maximal runs: two runs of one row never touch
        for (r0, r1, _, b), (q0, q1, a, _) in zip(runs[:-1], runs[1:]):
            assert (r0, r1) != (q0, q1) or a > b + 1


def test_run_table_of_a_disk_has_one_run_per_row(ops):
    runs = ops._structure_runs(ops._structure(_disk(5), 2))
    assert runs.tolist() == [[0, dy, -w, w] for dy, w in zip(range(-5, 6), (0, 3, 4, 4, 4, 5, 4, 4, 4, 3, 0))]


def test_structure_values_and_host_types(ops):
    import torch
    s = np.array([[0, 2, 0], [-1, 1, 0], [0, 0, 0.5]])
    want = (s != 0).astype(np.uint8)
    assert np.array_equal(ops._structure(s, 2), want)
    assert np.array_equal(ops._structure(torch.from_numpy(s), 2), want)
    assert np.array_equal(ops._structure(s.tolist(), 2), want)
    assert np.array_equal(ops._structure(np.asfortranarray(_ball(2))[:, ::-1], 3), _ball(2)[:, ::-1])


def test_structure_dimensionality(ops):
    with pytest.raises(RuntimeError, match="structure and input must have same dimensionality"):
        ops._structure(np.ones((3, 3)), 3)
    with pytest.raises(RuntimeError, match="structure and input must have same dimensionality"):
        ops._structure(np.ones((3, 3, 3)), 2)
    with pytest.raises(RuntimeError, match="structure and input must have same dimensionality"):
        ops._structure(np.ones(3), 2)


@pytest.mark.parametrize("shape", [(2, 3), (3, 4), (3, 3, 2), (0, 3), (32, 1)])
def test_structure_even_extents(ops, shape):
    with pytest.raises(ValueError, match="odd"):
        ops._structure(np.ones(shape), len(shape))


@pytest.mark.parametrize("shape", [(33, 1), (1, 33), (3, 3, 33), (33, 33)])
def test_structure_extents_over_the_limit(ops, shape):
    with pytest.raises(ValueError, match="at most 31"):
        ops._structure(np.ones(shape), len(shape))


def test_structure_runs_over_the_limit(ops):
    checker = np.indices((31, 31, 31)).sum(axis=0) % 2      # 31 * 31 rows of 15 or 16 runs
    with pytest.raises(ValueError, match="more than 1000 runs"):
        ops._structure(checker, 3)
    assert ops._structure(np.ones((31, 31, 31)), 3).shape == (31, 31, 31)   # 961 runs: accepted


def test_iterations(ops):
    assert ops._iterations(1) == 1 and ops._iterations(np.int64(5)) == 5
    for bad in (0, -1):
        with pytest.raises(ValueError, match="iterations must be >= 1"):
            ops._iterations(bad)
    for bad in (1.5, 1.0, "2", True, None):
        with pytest.raises(TypeError, match="iterations must be an integer"):
            ops._iterations(bad)


def test_limits_match_the_header(ops):
    import os
    from conftest import ROOT
    text = open(os.path.join(ROOT, "include", "hipr_b200.h")).read()
    assert "#define HIPR_MORPH_MAX_EXTENT %d" % ops.MORPHOLOGY_MAX_EXTENT in text
    assert "#define HIPR_MORPH_MAX_RUNS   %d" % ops.MORPHOLOGY_MAX_RUNS in text


def test_workspace_bytes_and_argument_checks(ops):
    lib = ops.lib()
    assert lib.hipr_morphology_workspace_bytes(2, 2048, 2048, 1, 1) == 0
    assert lib.hipr_morphology_workspace_bytes(2, 2048, 2048, 1, 2) == 2048 * 2048
    assert lib.hipr_morphology_workspace_bytes(3, 3, 70, 33, 5) == 7168           # 6930 rounded up to 256
    assert lib.hipr_morphology_workspace_bytes(3, 2048, 1024, 1024, 2) == -7      # 2^31 pixels: HIPR_E_RANGE
    assert lib.hipr_morphology_workspace_bytes(2, 4, 4, 1, 0) == -1
    assert lib.hipr_morphology_workspace_bytes(4, 4, 4, 4, 1) == -1
    s = np.ones((3, 3), np.uint8)
    sp = s.ctypes.data
    assert lib.hipr_binary_morphology(None, 2, 8, 8, 1, sp, 3, 3, 1, 0, 0, 1, None, 0, None, None) == -1
    assert lib.hipr_morphology_runs(None, 1, 3, 3, None, 0) == -1
    assert lib.hipr_morphology_runs(sp, 1, 3, 2, None, 0) == -1
    assert lib.hipr_morphology_runs(sp, 1, 3, 33, None, 0) == -7
    assert lib.hipr_morphology_runs(sp, 1, 3, 3, None, 0) == 3                    # count only
