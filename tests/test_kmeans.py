"""1-D k-means thresholding (SURVEY.md 8f rank 3).  Oracle = scikit-learn's KMeans itself (1.9.0 in this image),
frozen in tests/golden/kmeans_vectors.npz; oracle.kmeans1d is the numpy restatement of what scikit-learn does in
one dimension, which is what the CUDA kernel reproduces."""
import hashlib
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden_kmeans import CASES, case_image, kmeans_case  # noqa: E402

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "kmeans_vectors.npz"))


def _sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


@pytest.mark.parametrize("i", range(len(CASES)))
def test_restatement_matches_golden_sklearn(oracle, i):
    seed, k, n_init, tr, eps, pos = CASES[i]
    img = case_image(seed)
    assert np.array_equal(_sha(img), GOLD["case%d_img_sha256" % i])
    cen, labels, mask, n_iter, inertia = oracle.kmeans1d(img, k, 0, n_init, tr, eps, pos)
    np.testing.assert_allclose(cen, GOLD["case%d_centers" % i], rtol=0, atol=1e-12)
    assert n_iter == int(GOLD["case%d_n_iter" % i])
    assert np.array_equal(_sha(labels.astype(np.int32)), GOLD["case%d_labels_sha256" % i])
    assert int(mask.sum()) == int(GOLD["case%d_mask_sum" % i])
    np.testing.assert_allclose(inertia, float(GOLD["case%d_inertia" % i]), rtol=1e-10)


def test_restatement_matches_installed_sklearn(oracle):
    """Against scikit-learn itself where it is installed (any version whose k-means++ / Lloyd agree with 1.9)."""
    sklearn = pytest.importorskip("sklearn")
    if tuple(int(v) for v in sklearn.__version__.split(".")[:2]) < (1, 4):
        pytest.skip("n_init='auto' semantics need scikit-learn >= 1.4")
    rng = np.random.default_rng(5)
    for trial, k in enumerate((2, 3, 2, 3)):
        n = 60000
        a = np.concatenate([rng.normal(0.1, 0.05, n), rng.normal(0.6 + 0.1 * trial, 0.1, n // 3), rng.normal(1.5, 0.2, n // 5)])
        rng.shuffle(a)
        a = a.astype(np.float32).reshape(-1, 250)
        c1, l1, m1, it1, in1 = oracle.kmeans1d_sklearn(a, k)
        c2, l2, m2, it2, in2 = oracle.kmeans1d(a, k)
        np.testing.assert_allclose(c2, c1, rtol=0, atol=1e-12)
        assert it1 == it2 and np.array_equal(l1, l2) and np.array_equal(m1, m2)


def test_mask_orientation_is_the_brighter_cluster(oracle):
    img = kmeans_case(11)
    cen, labels, mask, _, _ = oracle.kmeans1d(img, 2)
    bright = int(np.argmax(cen))
    assert np.array_equal(mask, labels == bright)
    # the scripts' own orientation code, verbatim (syn/..._measurement.py:126-135)
    image_final = img.astype(np.float64)
    image0 = image_final * (labels == 0)
    image1 = image_final * (labels == 1)
    i0 = np.average(image0[image0 > 0])
    i1 = np.average(image1[image1 > 0])
    want = (labels == 1) if i0 < i1 else (labels == 0)
    assert np.array_equal(mask, want)


# ---- CUDA ----------------------------------------------------------------------------------------------------

def _threshold_band(cen, x, delta):
    """Samples within `delta` of a boundary between two neighbouring centres (where a 1e-12 difference in the centres
    could legitimately flip a label)."""
    c = np.sort(cen)
    mids = (c[:-1] + c[1:]) / 2
    return np.min(np.abs(x[..., None] - mids), axis=-1) < delta


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(CASES)))
def test_gpu_kmeans_matches_sklearn_golden(torch_cuda, oracle, i):
    import hipr_b200
    seed, k, n_init, tr, eps, pos = CASES[i]
    img = case_image(seed)
    res = hipr_b200.kmeans_threshold(torch_cuda.from_numpy(img).cuda(), k, 0, n_init, tr, eps, pos)
    want_c = GOLD["case%d_centers" % i]
    np.testing.assert_allclose(res.cluster_centers_, want_c, rtol=0, atol=1e-9)      # the bar is 1e-6
    assert res.n_iter == int(GOLD["case%d_n_iter" % i])
    np.testing.assert_allclose(res.inertia, float(GOLD["case%d_inertia" % i]), rtol=1e-9)
    _, want_labels, want_mask, _, _ = oracle.kmeans1d(img, k, 0, n_init, tr, eps, pos)
    got_labels = res.labels.cpu().numpy()
    assert np.array_equal(_sha(want_labels.astype(np.int32)), GOLD["case%d_labels_sha256" % i])
    differ = got_labels != want_labels
    # identical everywhere; a label may only differ within 1e-9 of a threshold (none does on these cases)
    x = oracle._kmeans_samples(img, tr, eps, False)[2].reshape(img.shape) if tr else img.astype(np.float64)
    assert not (differ & ~_threshold_band(want_c, x, 1e-9)).any()
    assert int(differ.sum()) == 0
    assert np.array_equal(res.mask.cpu().numpy(), want_mask)
    assert int(res.counts.sum()) == res.n_samples == int((img > 0).sum() if pos else img.size)


@pytest.mark.gpu
def test_gpu_kmeans_on_a_score_map(torch_cuda, oracle):
    """The call of syn/..._measurement.py:125 on the real thing: the F1 score map of a synthetic FOV (float32 on the
    device, float64 for scikit-learn), full 512 x 512, plus the float64-input path."""
    pytest.importorskip("sklearn")
    import hipr_b200
    from hipr_b200 import synth
    cube, _, _ = synth.make_fov(512, 512, 95, fov_index=3)
    score = hipr_b200.neighbor2d_score(cube.cuda(), "F1")
    s_np = score.cpu().numpy()
    for k in (2, 3):
        want_c, want_l, want_m, want_it, _ = oracle.kmeans1d_sklearn(s_np, k)
        for t in (score, score.double()):
            res = hipr_b200.kmeans_threshold(t, k)
            np.testing.assert_allclose(res.cluster_centers_, want_c, rtol=0, atol=1e-9)
            assert res.n_iter == want_it
            assert np.array_equal(res.labels.cpu().numpy(), want_l)
            assert np.array_equal(res.mask.cpu().numpy(), want_m)
    # log of the sum image, as eco/..._measurement.py:72-73
    s = hipr_b200.channel_sum(cube.cuda(), normalize=False, dtype=torch_cuda.float64)
    want_c, want_l, want_m, want_it, _ = oracle.kmeans1d_sklearn(s.cpu().numpy(), 2, transform="log", eps=1e-2)
    res = hipr_b200.kmeans_threshold(s, 2, transform="log", eps=1e-2)
    np.testing.assert_allclose(res.cluster_centers_, want_c, rtol=0, atol=1e-9)
    assert np.array_equal(res.labels.cpu().numpy(), want_l) and res.n_iter == want_it


@pytest.mark.gpu
def test_gpu_kmeans_rejects_bad_input(torch_cuda):
    import hipr_b200
    x = torch_cuda.rand(64, 64, device="cuda")
    with pytest.raises(ValueError):
        hipr_b200.kmeans_threshold(x.cpu(), 2)                       # no CPU path
    bad = x.clone()
    bad[3, 4] = float("nan")
    with pytest.raises(ValueError):
        hipr_b200.kmeans_threshold(bad, 2)                           # scikit-learn raises on NaN as well
    with pytest.raises(ValueError):
        hipr_b200.kmeans_threshold(torch_cuda.zeros(8, 8, device="cuda"), 2, positive_only=True)   # no samples
    with pytest.raises(ValueError):
        hipr_b200.kmeans_threshold(x, 9)                             # k <= 8
