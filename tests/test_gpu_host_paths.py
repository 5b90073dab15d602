"""The host-array entry points share one band upload, one call scope, one 2-D score tail and one cell-table layout
(csrc/host_api.cu).  These tests pin the behaviour those shared pieces carry: the band ring across the FOVs of a
batch and across pinned and pageable inputs, general stencil parameters and F3 on every 2-D host path, 3-D and
per-cell bands that wrap the ring, an argument error found after the upload was enqueued, and the device timing."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-5
ATOL_F32 = 2e-6      # float64 stencil, float32 score
ATOL_FIXED = 5e-7    # fixed-point stencil


def _pinned(a):
    import hipr_b200
    p = hipr_b200.pinned_empty(a.shape, a.dtype)
    p[...] = a
    return p


@pytest.mark.parametrize("denoise_h", [None, 0.02])
def test_batch_ring_carries_over_fovs(torch_cuda, denoise_h):
    """Six FOVs of two bands each (160 rows of 1024 x 95 float32; 86 rows per 32 MiB band): the three ring slots
    do not line up with the FOVs, so each FOV starts on a different slot.  Pinned and pageable cubes alternate
    irregularly.  Every score is bit-identical to the single-FOV entry point."""
    import hipr_b200
    from hipr_b200 import synth
    cubes = [synth.make_fov(160, 1024, 95, fov_index=20 + i)[0].numpy() for i in range(6)]
    mixed = [_pinned(c) if pin else c for c, pin in zip(cubes, (False, True, True, False, True, False))]
    want = [hipr_b200.neighbor2d_score_host(c, "F1", denoise_h=denoise_h) for c in cubes]
    got = hipr_b200.neighbor2d_score_host_batch(mixed, "F1", denoise_h=denoise_h)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


@pytest.mark.parametrize("params", [(7, 5), (11, 9)])
def test_f3_and_general_parameters_agree_across_host_paths(torch_cuda, oracle, params):
    """F3 (global range) at the pipelines' (11, 9) table (fixed-point stencil) and at (7, 5) (float64 stencil):
    the single-FOV, batch and Fov-handle paths give the same bits, within the gate of the oracle."""
    import hipr_b200
    from hipr_b200 import synth
    P, R = params
    cubes = [synth.make_fov(96, 160, 95, fov_index=30 + i)[0].numpy() for i in range(3)]
    single = [hipr_b200.neighbor2d_score_host(c, "F3", patch_size=P, phi_range=R) for c in cubes]
    batch = hipr_b200.neighbor2d_score_host_batch(cubes, "F3", patch_size=P, phi_range=R)
    for c, s, b in zip(cubes, single, batch):
        assert np.array_equal(s, b)
        with hipr_b200.Fov(c) as fov:
            assert np.array_equal(fov.score("F3", patch_size=P, phi_range=R), s)
        if params == (11, 9):
            np.testing.assert_allclose(s, oracle.neighbor2d_score(c, "F3"), rtol=RTOL, atol=ATOL_FIXED)
        else:
            total = c.astype(np.float64).sum(axis=2)
            np.testing.assert_allclose(s, oracle.lne2d(total / total.max(), "F3", P, R), rtol=RTOL, atol=ATOL_F32)


def test_neighbor3d_host_bands_pageable_and_pinned(torch_cuda):
    """A 112 x 64 x 40 x 95 float32 z-stack (109 MB, four bands of 34 x-planes: the ring wraps): pageable and
    page-locked input give the same bits as each other and as the device-resident pipeline."""
    import hipr_b200
    from hipr_b200 import synth
    cube = synth.make_volume_cube(112, 64, 40, 95, seed=5).numpy()
    pageable = hipr_b200.neighbor3d_score_host(cube, "ME2")
    pinned = hipr_b200.neighbor3d_score_host(_pinned(cube), "ME2")
    dev = hipr_b200.neighbor3d_score(torch_cuda.from_numpy(cube).cuda(), "ME2").cpu().numpy()
    assert np.array_equal(pageable, pinned)
    assert np.array_equal(pageable, dev)


def test_cell_spectra_host_over_several_bands(torch_cuda, oracle):
    """A 512 x 512 x 95 cube streams in four bands of whole 32-row tiles: pageable and page-locked input give the
    same table as the Fov handle (one pass over the resident cube), bit for bit, with the oracle's labels and areas."""
    import hipr_b200
    from hipr_b200 import synth
    cube, labels, _ = synth.make_fov(512, 512, 95, fov_index=11)
    cube, labels = cube.numpy(), labels.numpy()
    pageable = hipr_b200.cell_spectra_host(cube, labels)
    pinned = hipr_b200.cell_spectra_host(_pinned(cube), labels)
    with hipr_b200.Fov(cube) as fov:
        resident = fov.cell_spectra(labels)
    for a, b, c in zip(pageable, pinned, resident):
        assert np.array_equal(a, b) and np.array_equal(a, c)
    wl, wa, _, _ = oracle.cell_spectra(labels, cube)
    assert np.array_equal(pageable[0], wl) and np.array_equal(pageable[1], wa)


def test_error_after_enqueue_leaves_the_workspace_usable(torch_cuda):
    """An unknown flavour code is found by the stencil, after the cube was uploaded and summed: the call returns the
    flavour error, and the next valid call on the same workspace returns the right score."""
    import hipr_b200
    from hipr_b200 import synth, tables
    from hipr_b200._lib import lib
    cube = synth.make_fov(64, 96, 95, fov_index=12)[0].numpy()
    want = hipr_b200.neighbor2d_score_host(cube, "F1")
    tab = np.ascontiguousarray(tables.line_table_2d(11, 9), dtype=np.int32)
    score = np.empty((64, 96), np.float32)
    code = lib().hipr_neighbor2d_host(cube.ctypes.data_as(C.c_void_p), 64, 96, 95, 11, 9,
                                      tab.ctypes.data_as(C.c_void_p), 99, score.ctypes.data_as(C.c_void_p), None)
    assert code == -5                                   # HIPR_E_FLAVOUR
    assert np.array_equal(hipr_b200.neighbor2d_score_host(cube, "F1"), want)


def test_host_entry_points_record_their_device_time(torch_cuda):
    """hipr_host_last_elapsed_ms() is positive after every timed host entry point; cell_spectra_host is not timed
    and leaves the previous call's value."""
    import hipr_b200
    from hipr_b200 import synth
    from hipr_b200._lib import lib
    cube, labels, _ = synth.make_fov(64, 96, 95, fov_index=13)
    cube, labels = cube.numpy(), labels.numpy()
    vol = synth.make_volume_cube(12, 14, 16, 95, seed=6).numpy()
    pad2 = np.pad(np.random.default_rng(0).random((20, 24)), 5, mode="edge")
    pad3 = np.pad(np.random.default_rng(1).random((6, 7, 8)), 5, mode="edge")
    raw = np.clip(np.round(cube * 40000.0), 0, 65535).astype(np.uint16)
    fov = hipr_b200.Fov(cube)
    calls = [
        lambda: None,                                   # hipr_fov_upload, above
        lambda: hipr_b200.neighbor2d_score_host(cube, "F1"),
        lambda: hipr_b200.neighbor2d_score_host(cube, "F1", denoise_h=0.02),
        lambda: hipr_b200.neighbor2d_score_host_raw(raw, 65535.0, "F1"),
        lambda: hipr_b200.neighbor2d_score_host_batch([cube, cube], "F1"),
        lambda: hipr_b200.neighbor3d_score_host(vol, "ME2"),
        lambda: hipr_b200.neighbor3d_score_host(vol, "ME2", denoise_h=0.03, denoise_distance=3),
        lambda: hipr_b200.line_profile_2d_host(pad2, 11, 9),
        lambda: hipr_b200.line_profile_3d_host(pad3, 11, 9, 9),
        lambda: hipr_b200.lne3d_dirs_host(pad3, 11, 9, 9),
        lambda: fov.score("F1"),
        lambda: fov.cell_spectra(labels),
    ]
    try:
        for call in calls:
            call()
            assert lib().hipr_host_last_elapsed_ms() > 0.0
        before = lib().hipr_host_last_elapsed_ms()
        hipr_b200.cell_spectra_host(cube, labels)
        assert lib().hipr_host_last_elapsed_ms() == before
    finally:
        fov.close()
