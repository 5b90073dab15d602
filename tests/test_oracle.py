"""The oracle is pinned: against the compiled, unmodified reference (oracle/_ref) where it is built,
and against golden vectors generated from it (tests/golden/make_golden.py) everywhere."""
import hashlib
import os

import numpy as np
import pytest

from conftest import smooth_image

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.npz"))
SHA_2D = "b1278799e8f5fd61d163437987943d3b2d104245e493df6dab5f2072335dbb3d"      # SURVEY.md section 4
SHA_3D = "13bca0604962da5b1568581024e69ea5f4079c9ad9b04745a4beec04a8d93040"


def test_tables_match_survey_hashes_and_golden(oracle):
    t2 = oracle.line_table_2d(11, 9).transpose(2, 0, 1)
    t3 = oracle.line_table_3d(11, 9, 9).transpose(2, 0, 1)
    assert hashlib.sha256((t2 - 5).astype(np.int64).tobytes()).hexdigest() == SHA_2D
    assert hashlib.sha256((t3 - 5).astype(np.int64).tobytes()).hexdigest() == SHA_3D
    assert np.array_equal(t2, GOLD["table2d_11_9"])
    assert np.array_equal(t3, GOLD["table3d_11_9_9"])
    # SURVEY.md: phi3 and phi6 are not mirror images (np.round of 2.5000000000000004 vs -2.4999999999999996)
    assert (t2[3, 0] - 5).tolist() == [-3, -4] and (t2[6, 0] - 5).tolist() == [2, -4]
    assert all((t2[:, 5] == 5).ravel()) and all((t3[:, 5] == 5).ravel())     # centre sample is the pixel itself
    assert len({tuple(p) for p in (t2 - 5).reshape(-1, 2)}) == 64             # 64 distinct footprint pixels
    assert len({tuple(p) for p in (t3 - 5).reshape(-1, 3)}) == 355
    assert len({tuple(map(tuple, d)) for d in t3}) == 66                      # 66 of 72 lines distinct


def test_golden_2d(oracle):
    img = GOLD["img2d"]
    padded = np.pad(img / img.max(), 5, mode="edge")
    lp = oracle.line_profile_2d_v2(padded, 11, 9)
    assert hashlib.sha256(lp.tobytes()).digest() == GOLD["lp2d_sha256"].tobytes()
    assert np.array_equal(lp[:3, :4], GOLD["lp2d_corner"])
    for f in ("F1", "F2", "F3"):
        assert np.array_equal(oracle.EPILOGUES[f](lp), GOLD["score2d_" + f], equal_nan=True)
        assert np.array_equal(oracle.lne2d(img / img.max(), f), GOLD["score2d_" + f], equal_nan=True)


def test_golden_3d(oracle):
    vol = GOLD["vol3d"]
    vp = np.pad(vol / vol.max(), 5, mode="edge")
    lp5 = oracle.line_profile_v2(vp, 11, 9, 9)
    assert hashlib.sha256(lp5.tobytes()).digest() == GOLD["lp3d_sha256"].tobytes()
    assert np.array_equal(oracle.line_profile_memory_efficient_v2(vp, 11, 9, 9), GOLD["me2_3d"])
    assert np.array_equal(oracle.lne3d(vol / vol.max(), "ME2"), GOLD["score3d_ME2"])
    assert np.array_equal(oracle.lne3d(vol / vol.max(), "F2"), GOLD["score3d_F2"])
    assert np.array_equal(oracle.lne3d(vol / vol.max(), "F3"), GOLD["score3d_F3"])
    got = oracle.line_profile_memory_efficient_v3(GOLD["v3_in"], 11, 9, 9)[:6]
    assert not np.isnan(got).any()
    assert np.array_equal(got, GOLD["v3_out"])


def test_golden_pipeline_and_cells(oracle):
    cube, lab = GOLD["cube"], GOLD["labels"]
    assert np.array_equal(oracle.neighbor2d_score(cube, "F1"), GOLD["cube_score_F1"])
    l, a, avg, norm = oracle.cell_spectra(lab, cube)
    assert np.array_equal(l, GOLD["cell_labels"]) and np.array_equal(a, GOLD["cell_area"])
    assert np.array_equal(avg, GOLD["cell_avgint"]) and np.array_equal(norm, GOLD["cell_avgint_norm"])
    assert l.tolist() == [3, 7, 12]


@pytest.mark.parametrize("params", [(11, 9), (7, 5), (11, 4), (15, 9), (11, 12), (5, 3), (13, 16)])
def test_line_profile_2d_vs_compiled_reference(oracle, ref2d, params):
    P, R = params
    a = np.random.default_rng(P * 100 + R).random((P + 12, P + 16))
    assert np.array_equal(ref2d.line_profile_2d_v2(a, P, R), oracle.line_profile_2d_v2(a, P, R))


@pytest.mark.parametrize("params", [(11, 9, 9), (7, 5, 4), (9, 6, 7), (5, 3, 3)])
def test_3d_vs_compiled_reference(oracle, ref3d, params):
    P = params[0]
    a = np.random.default_rng(sum(params)).random((P + 10, P + 4, P + 3))
    assert np.array_equal(ref3d.line_profile_v2(a, *params), oracle.line_profile_v2(a, *params))
    small = a[:P + 2, :P + 2, :P + 1]                       # the reference's me_v2 runs at ~3 kvox/s
    assert np.array_equal(ref3d.line_profile_memory_efficient_v2(small, *params),
                          oracle.line_profile_memory_efficient_v2(small, *params))
    got = oracle.line_profile_memory_efficient_v3(a, *params)
    ok = ~np.isnan(got)
    assert ok.any()
    assert np.array_equal(ref3d.line_profile_memory_efficient_v3(a, *params)[ok], got[ok])


PARAMS = np.load(os.path.join(os.path.dirname(__file__), "golden", "oracle_params_vectors.npz"))


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest()


@pytest.mark.parametrize("params", [(11, 9), (7, 5), (11, 4), (15, 9), (11, 12), (5, 3), (13, 16)])
def test_line_profile_2d_frozen_at_other_parameters(oracle, params):
    """The inputs of test_line_profile_2d_vs_compiled_reference against the oracle's frozen output
    (tests/golden/make_golden_params.py): runs without oracle/_ref, so a change of the oracle at
    non-default parameters is caught in a clean checkout too."""
    P, R = params
    a = np.random.default_rng(P * 100 + R).random((P + 12, P + 16))
    assert _sha(oracle.line_profile_2d_v2(a, P, R)) == PARAMS["lp2d_sha256_%d_%d" % params].tobytes()


@pytest.mark.parametrize("params", [(11, 9, 9), (7, 5, 4), (9, 6, 7), (5, 3, 3)])
def test_3d_frozen_at_other_parameters(oracle, params):
    """The inputs of test_3d_vs_compiled_reference against the oracle's frozen outputs
    (tests/golden/make_golden_params.py)."""
    P = params[0]
    k = "%d_%d_%d" % params
    a = np.random.default_rng(sum(params)).random((P + 10, P + 4, P + 3))
    assert _sha(oracle.line_profile_v2(a, *params)) == PARAMS["lp3d_sha256_" + k].tobytes()
    small = a[:P + 2, :P + 2, :P + 1]
    assert np.array_equal(oracle.line_profile_memory_efficient_v2(small, *params), PARAMS["me2_3d_" + k])
    got = oracle.line_profile_memory_efficient_v3(a, *params)
    assert (~np.isnan(got)).any()
    assert np.array_equal(got, PARAMS["v3_" + k], equal_nan=True)


def test_identities_from_the_survey(oracle):
    """me_v2 == (v2[..., 5] - min) / max(max - min, 1e-8); percentiles of 9 values are order
    statistics 2 and 6; of 72 values they are lerps at 17.75 / 53.25."""
    a = smooth_image((15, 14, 16), 1).astype(np.float64)
    lp = oracle.line_profile_v2(a, 11, 9, 9)
    mn, mx = lp.min(-1), lp.max(-1)
    assert np.array_equal(oracle.line_profile_memory_efficient_v2(a, 11, 9, 9), (lp[..., 5] - mn) / np.maximum(mx - mn, 1e-8))
    v = np.random.default_rng(0).random((50, 9))
    s = np.sort(v, axis=1)
    assert np.array_equal(np.percentile(v, 25, axis=1), s[:, 2]) and np.array_equal(np.percentile(v, 75, axis=1), s[:, 6])
    v = np.random.default_rng(1).random((50, 72))
    s = np.sort(v, axis=1)
    assert np.array_equal(np.percentile(v, 25, axis=1), s[:, 18] - (s[:, 18] - s[:, 17]) * 0.25)
    assert np.array_equal(np.percentile(v, 75, axis=1), s[:, 53] + (s[:, 54] - s[:, 53]) * 0.25)


def test_cell_spectra_matches_scipy_ndimage(oracle):
    """regionprops(...).mean_intensity is the per-label arithmetic mean: cross-check with scipy."""
    from scipy import ndimage
    rng = np.random.default_rng(5)
    lab = (rng.integers(0, 40, (60, 70)) * (rng.random((60, 70)) > 0.4)).astype(np.int64)
    lab[lab == 17] = 0                                   # a missing id: rows are the labels present
    img = rng.random((60, 70, 12))
    labels, area, avg, norm = oracle.cell_spectra(lab, img)
    assert labels.tolist() == sorted(set(np.unique(lab)) - {0}) and 17 not in labels
    assert np.array_equal(area, ndimage.sum_labels(np.ones_like(lab), lab, labels).astype(np.int64))
    for k in range(12):
        np.testing.assert_allclose(avg[:, k], ndimage.mean(img[:, :, k], lab, labels), rtol=1e-13)
    np.testing.assert_allclose(norm, avg / avg.max(axis=1)[:, None])


def test_reference_errors(ref2d, ref3d):
    with pytest.raises(ValueError, match="Buffer dtype mismatch"):
        ref2d.line_profile_2d_v2(np.zeros((12, 12), np.float32), 11, 9)
    with pytest.raises(ValueError, match="Buffer dtype mismatch"):
        ref3d.neighbor_average(np.zeros((30, 30, 30), np.float32), 11)


def test_register_stacks_is_a_shifted_paste(oracle):
    """oracle.register_stacks (syn/..._measurement.py:86-105) == out[r, c] = in[r - sr, c - sc], zero outside."""
    rng = np.random.default_rng(0)
    H, W = 13, 13
    stacks = [rng.random((H, W, c)) for c in (3, 2, 4)]
    shifts = [(0, 0), (2.7, -3.2), (-5, 1)]
    cube, s = oracle.register_stacks(stacks, shifts)
    want = np.zeros((H, W, 9))
    off = 0
    for a, (sr, sc) in zip(stacks, shifts):
        sr, sc = int(sr), int(sc)
        for r in range(H):
            for c in range(W):
                if 0 <= r - sr < H and 0 <= c - sc < W:
                    want[r, c, off:off + a.shape[2]] = a[r - sr, c - sc]
        off += a.shape[2]
    assert np.array_equal(cube, want)
    assert np.array_equal(s, want.sum(axis=2))
    cal = 0.5 + rng.random((H, W, 9))
    cube2, s2 = oracle.register_stacks(stacks, shifts, cal)
    assert np.array_equal(cube2, want / cal) and np.array_equal(s2, (want / cal).sum(axis=2))


def _nlm_image(shape, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:shape[0], 0:shape[1]]
    img = (np.sin(yy / 5.0) ** 2 + np.cos(xx / 7.0) ** 2) / 2 + 0.03 * rng.random(shape)
    return img / img.max()


@pytest.mark.parametrize("h,d", [(0.02, 11), (0.1, 11), (0.03, 4)])
def test_nlm_restatement_equals_direct_formulation(oracle, h, d):
    """PARITY UNPINNED (scikit-image absent): the loop-for-loop restatement of skimage's fast NL-means
    (integral images, symmetric accumulation) equals the estimator written pixel by pixel."""
    img = _nlm_image((31, 29), 1)
    a = oracle.denoise_nl_means_2d(img, patch_distance=d, h=h)
    b = oracle.denoise_nl_means_2d_direct(img, patch_distance=d, h=h)
    np.testing.assert_allclose(a, b, rtol=1e-12)


def test_nlm_properties(oracle):
    img = _nlm_image((40, 36), 2)
    out = oracle.denoise_nl_means_2d(img, h=0.02)
    assert out.shape == img.shape and out.min() >= img.min() - 1e-12 and out.max() <= img.max() + 1e-12   # convex weights
    flat = np.full((24, 24), 0.3)
    np.testing.assert_allclose(oracle.denoise_nl_means_2d(flat, h=0.02), flat, rtol=1e-13)
    # a tiny h keeps only the zero shift (every other patch is further than the cutoff): identity
    np.testing.assert_allclose(oracle.denoise_nl_means_2d(img, h=1e-4), img, rtol=1e-14)
    # even patch sizes are made odd, as skimage does
    assert np.array_equal(oracle.denoise_nl_means_2d(img, patch_size=6, h=0.05), oracle.denoise_nl_means_2d(img, patch_size=7, h=0.05))


def test_cell_geometry_known_shapes(oracle):
    """The regionprops restatement on shapes with closed-form moments."""
    seg = np.zeros((30, 40), dtype=np.int64)
    seg[5:9, 10:30] = 3            # 4 x 20 rectangle
    lab, area, g = oracle.cell_geometry(seg)
    assert lab.tolist() == [3] and area.tolist() == [80]
    np.testing.assert_allclose(g[0, :2], [6.5, 19.5])
    # variances of a discrete uniform: (n^2 - 1) / 12
    np.testing.assert_allclose(g[0, 2], 4 * np.sqrt((20 ** 2 - 1) / 12.0))
    np.testing.assert_allclose(g[0, 3], 4 * np.sqrt((4 ** 2 - 1) / 12.0))
    np.testing.assert_allclose(abs(g[0, 5]), np.pi / 2)      # long axis along the columns ('rc' convention)
    painted = oracle.paint_labels(seg, np.array([0.0, 1.0, 2.0, 7.5]))
    assert painted[6, 12] == 7.5 and painted[0, 0] == 0.0 and painted.sum() == 80 * 7.5


def test_oracle_next_rows_match_frozen_vectors(oracle):
    """tests/golden/next_rows_vectors.npz (make_golden_next.py): the restatements have not drifted."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "next_rows_vectors.npz"))
    cube, ssum = oracle.register_stacks([g["reg_stack0"], g["reg_stack1"], g["reg_stack2"]], g["reg_shifts"], g["reg_calibration"])
    assert np.array_equal(cube, g["reg_cube"]) and np.array_equal(ssum, g["reg_sum"])
    np.testing.assert_allclose(oracle.denoise_nl_means_2d(g["nlm_in"], h=0.02), g["nlm_out_h002"], rtol=1e-13)
    np.testing.assert_allclose(oracle.denoise_nl_means_2d(g["nlm_in"], h=0.1), g["nlm_out_h01"], rtol=1e-13)
    lab, area, geom = oracle.cell_geometry(g["geo_seg"])
    assert np.array_equal(lab, g["geo_labels"]) and np.array_equal(area, g["geo_area"])
    np.testing.assert_allclose(geom, g["geo_geometry"], rtol=1e-13, atol=1e-13)
    assert np.array_equal(oracle.paint_labels(g["geo_seg"], g["paint_values"]), g["paint_out"])


@pytest.mark.parametrize("h,d", [(0.05, 2), (0.03, 3)])
def test_nlm3d_restatement_equals_direct_formulation(oracle, h, d):
    """The loop-for-loop restatement of skimage's _fast_nl_means_denoising_3d (integral images, symmetric
    accumulation) against the voxel-by-voxel form the CUDA kernel evaluates."""
    rng = np.random.default_rng(7)
    x, y, z = np.meshgrid(np.arange(9), np.arange(10), np.arange(11), indexing="ij")
    vol = 0.5 + 0.3 * np.sin(x / 2.0 + y / 3.0) * np.cos(z / 2.5) + 0.02 * rng.standard_normal((9, 10, 11))
    a = oracle.denoise_nl_means_3d(vol, patch_distance=d, h=h)
    b = oracle.denoise_nl_means_3d_direct(vol, patch_distance=d, h=h)
    np.testing.assert_allclose(a, b, rtol=1e-12)
    flat = np.full((9, 10, 11), 0.25)
    np.testing.assert_allclose(oracle.denoise_nl_means_3d(flat, patch_distance=d, h=h), flat, rtol=1e-13)


def test_nlm3d_golden_vectors_present():
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "nlm3d_vectors.npz"))
    assert g["nlm3d_in"].shape == g["nlm3d_out_h003"].shape == (17, 18, 40)
    assert np.all(np.isfinite(g["nlm3d_out_h003"])) and np.abs(g["nlm3d_out_h003"] - g["nlm3d_in"]).max() < 0.2
