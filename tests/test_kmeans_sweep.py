"""Sweeps of the 1-D k-means row (K8) beyond the frozen golden cases of test_kmeans.py.

CPU: the numpy restatement oracle.kmeans1d against scikit-learn itself on seeded data of four kinds (continuous,
8-bit quantised, 12-bit counts with zeros, six levels), k = 2..8, n_init 1 / 3 / 10, positive_only and the log
transforms.  Where a clustering runs empty (more clusters than distinct values) scikit-learn relocates the cluster and
warns; the restatement, like the kernel, raises instead.

GPU: the CUDA kernel against scikit-learn (where installed) and against the restatement (always), at the sizes, grid
shapes, dtypes, parameters and output options where a kernel of this structure can go wrong, and with its workspace
pre-filled with different byte patterns."""
import ctypes as C
import math
import os
import sys
import warnings

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden_kmeans import kmeans_case  # noqa: E402

from conftest import smooth_image  # noqa: E402

EMPTY = "a cluster ran empty"          # the kernel's and the restatement's RuntimeError
KM_THREADS = 512                       # kmeans1d.cu: one CTA takes a chunk of a multiple of 512 samples


def _sklearn():
    sklearn = pytest.importorskip("sklearn")
    if tuple(int(v) for v in sklearn.__version__.split(".")[:2]) < (1, 4):
        pytest.skip("n_init semantics need scikit-learn >= 1.4")
    import sklearn.cluster  # noqa: F401  (loads scikit-learn's OpenMP runtime before its threads are limited)
    from threadpoolctl import threadpool_limits
    return threadpool_limits


def _have_sklearn():
    try:
        _sklearn()
    except pytest.skip.Exception:
        return False
    return True


def _max_n_init(k):
    """The largest n_init hipr_kmeans1d_uniforms accepts: 256 draws, 1 + (2 + int(log k)) * (k - 1) per initialisation."""
    return 256 // (1 + (2 + int(math.log(k))) * (k - 1))


def _fit_sklearn(oracle, img, k, n_init=1, transform=None, eps=0.0, positive_only=False, max_iter=300, tol=1e-4):
    """scikit-learn's answer on one thread, or EMPTY where it warns that it found fewer distinct clusters than k."""
    from sklearn.exceptions import ConvergenceWarning
    with _sklearn()(1), warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        out = oracle.kmeans1d_sklearn(img, k, 0, n_init, transform, eps, positive_only, max_iter=max_iter, tol=tol)
    if any(issubclass(w.category, ConvergenceWarning) and "distinct clusters" in str(w.message) for w in caught):
        return EMPTY
    return out


def _fit_restatement(oracle, img, k, n_init=1, transform=None, eps=0.0, positive_only=False, max_iter=300, tol=1e-4):
    try:
        return oracle.kmeans1d(img, k, 0, n_init, transform, eps, positive_only, max_iter=max_iter, tol=tol)
    except RuntimeError as exc:
        assert EMPTY in str(exc)
        return EMPTY


# ---- CPU: the restatement against scikit-learn -----------------------------------------------------------------

def sweep_data(kind, rng):
    """Non-negative float32 vectors of 200..20,000 samples."""
    n = int(rng.integers(200, 20000))
    if kind == "continuous":
        a = np.abs(np.concatenate([rng.normal(0.15, 0.05, n), rng.normal(0.55, 0.1, n // 3), rng.normal(0.9, 0.08, n // 6)]))
    elif kind == "8bit":
        a = np.concatenate([rng.normal(0.2, 0.08, n), rng.normal(0.6, 0.1, n // 4)])
        a = np.clip(np.round(a * 255), 0, 255) / 255
    elif kind == "12bit_zeros":
        a = np.concatenate([np.zeros(n // 4), rng.gamma(2.0, 150.0, n), rng.normal(2500, 400, n // 5)])
        a = np.clip(np.round(a), 0, 4095)
    else:
        assert kind == "levels6"
        a = rng.integers(0, 6, n) / 5.0
    rng.shuffle(a)
    return a.astype(np.float32)


@pytest.mark.parametrize("kind", ["continuous", "8bit", "12bit_zeros", "levels6"])
def test_restatement_sweep_matches_sklearn(oracle, kind):
    """k = 2..8 x n_init 1 / 3 / 10 (capped at what the kernel accepts) x positive_only, the transform cycling through
    none, log10(x + 1e-3) and ln(x + 1e-2): centres within 1e-12 of the data's scale, labels identical, same n_iter,
    and the restatement raises exactly where scikit-learn warns about fewer distinct clusters."""
    _sklearn()
    transforms = [(None, 0.0), ("log10", 1e-3), ("log", 1e-2)]
    rng = np.random.default_rng(["continuous", "8bit", "12bit_zeros", "levels6"].index(kind))
    case, raised, worst = 0, 0, 0.0
    for k in range(2, 9):
        for n_init in sorted({min(n, _max_n_init(k)) for n in (1, 3, 10)}):
            for pos in (False, True):
                tr, eps = transforms[case % 3]
                case += 1
                a = sweep_data(kind, rng)
                what = "%s k=%d n_init=%d positive_only=%s transform=%s n=%d" % (kind, k, n_init, pos, tr, a.size)
                want = _fit_sklearn(oracle, a, k, n_init, tr, eps, pos)
                got = _fit_restatement(oracle, a, k, n_init, tr, eps, pos)
                if want is EMPTY or got is EMPTY:
                    assert want is got, what + ": scikit-learn found fewer distinct clusters xor the restatement raised"
                    raised += 1
                    continue
                scale = max(1.0, float(np.abs(oracle._kmeans_samples(a, tr, eps, pos)[2]).max()))
                d = float(np.abs(got[0] - want[0]).max())
                worst = max(worst, d / scale)
                assert d <= 1e-12 * scale, what + ": centres differ by %g" % d
                assert got[3] == want[3], what
                assert np.array_equal(got[1], want[1]), what + ": %d labels differ" % int((got[1] != want[1]).sum())
                assert np.array_equal(got[2], want[2]), what
    if kind == "levels6":
        assert raised > 0                # k = 7 and 8 on six levels: the empty-cluster path was taken
    print("%s: %d cases, %d empty-cluster raises, largest centre difference %.3g of the scale" % (kind, case, raised, worst))


# ---- GPU: the kernel against scikit-learn and the restatement ---------------------------------------------------

def mixture(shape, rng, modes=8):
    """Positive values from `modes` separated normal modes of unequal weights (k up to 8 is meaningful)."""
    n = int(np.prod(shape))
    w = rng.random(modes) + 0.2
    which = rng.choice(modes, n, p=w / w.sum())
    return np.abs(np.linspace(0.1, 0.9, modes)[which] + rng.normal(0, 0.04, n)).reshape(shape).astype(np.float32)


def _threshold_band(cen, x, delta):
    c = np.sort(cen)
    mids = (c[:-1] + c[1:]) / 2
    return np.min(np.abs(x[..., None] - mids), axis=-1) < delta


def _samples(oracle, img, transform, eps, positive_only):
    """Per-pixel sample value (transformed) and the valid mask, image shaped."""
    with np.errstate(divide="ignore", invalid="ignore"):
        x = oracle._kmeans_samples(img, transform, eps, False)[2].reshape(img.shape)
    valid = (img > 0) if positive_only else np.ones(img.shape, dtype=bool)
    return x, valid


def _compare(res, want, who, img, x, valid, fill_label, return_labels, return_mask):
    cen, labels, mask, n_iter, inertia = want
    d = float(np.abs(res.cluster_centers_ - cen).max())
    assert d <= 1e-9, "%s: centres differ by %g" % (who, d)
    assert res.n_iter == n_iter, who
    np.testing.assert_allclose(res.inertia, inertia, rtol=1e-9, err_msg=who)
    assert int(res.counts.sum()) == res.n_samples == int(valid.sum()), who
    band = valid & _threshold_band(cen, np.where(valid, x, 0.0), 1e-9)
    n_band = 0
    if return_labels:
        got = res.labels.cpu().numpy()
        assert got.shape == img.shape
        differ = got != np.where(valid, labels, fill_label)
        assert not (differ & ~band).any(), "%s: %d labels differ outside the 1e-9 band" % (who, int((differ & ~band).sum()))
        n_band = int(differ.sum())
    else:
        assert res.labels is None
    if return_mask:
        got = res.mask.cpu().numpy()
        assert got.dtype == np.bool_ and got.shape == img.shape
        assert not ((got != mask) & ~band).any(), who
    else:
        assert res.mask is None
    if n_band:
        warnings.warn("%s: %d labels differ within 1e-9 of a threshold between centres" % (who, n_band))
    return d, n_band


def run_case(torch, oracle, img, k, n_init=1, transform=None, eps=0.0, positive_only=False, max_iter=300, tol=1e-4,
             fill_label=0, return_labels=True, return_mask=True, view=None):
    """The kernel on `img` (or on view(tensor of img), a non-contiguous view) against every reference available."""
    import hipr_b200
    t = torch.from_numpy(np.ascontiguousarray(img)).cuda()
    if view is not None:
        t = view(t)
        assert not t.is_contiguous()
        img = t.cpu().numpy()
    args = (k, n_init, transform, eps, positive_only)
    refs = {"restatement": _fit_restatement(oracle, img, *args, max_iter=max_iter, tol=tol)}
    if _have_sklearn():
        refs["scikit-learn"] = _fit_sklearn(oracle, img, *args, max_iter=max_iter, tol=tol)
    call = lambda: hipr_b200.kmeans_threshold(t, k, 0, n_init, transform, eps, positive_only, max_iter=max_iter,  # noqa: E731
                                              tol=tol, return_labels=return_labels, return_mask=return_mask,
                                              fill_label=fill_label)
    if any(w is EMPTY for w in refs.values()):
        assert all(w is EMPTY for w in refs.values()), "the references disagree on an empty cluster"
        with pytest.raises(RuntimeError, match=EMPTY):
            call()
        print("k=%d n_init=%d: every reference and the kernel report an empty cluster" % (k, n_init))
        return None
    res = call()
    x, valid = _samples(oracle, img, transform, eps, positive_only)
    for who, want in refs.items():
        d, n_band = _compare(res, want, who, img, x, valid, fill_label, return_labels, return_mask)
        print("shape=%s dtype=%s k=%d n_init=%d vs %s: max |centre diff| %.3g, labels in the band %d"
              % (img.shape, img.dtype, k, n_init, who, d, n_band))
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(2, 9))
def test_gpu_smallest_sizes(torch_cuda, oracle, k):
    """n = k (k distinct values) is the smallest legal size; n = k - 1 raises like scikit-learn.

    On k evenly spaced values several k-means++ candidates tie exactly in potential (removing either end of a
    symmetric gap).  scikit-learn breaks such a tie by the rounding of its ||x||^2 - 2 x c + ||c||^2 distances and BLAS
    sums, which neither the kernel nor the restatement reproduces (k = 7 here picks a different seed order): there the
    kernel is held to the restatement exactly and to scikit-learn as a partition (same centres in sorted order, same
    mask)."""
    import hipr_b200
    rng = np.random.default_rng(k)
    a = (0.05 + 0.9 * rng.random(k)).astype(np.float32)
    res = run_case(torch_cuda, oracle, a, k)
    assert sorted(res.counts.tolist()) == [1] * k
    tied = rng.permutation(np.linspace(0.05, 0.95, k)).astype(np.float32)
    res = hipr_b200.kmeans_threshold(torch_cuda.from_numpy(tied).cuda(), k)
    cen, labels, mask, n_iter, _ = oracle.kmeans1d(tied, k)
    assert np.array_equal(res.cluster_centers_, cen) and res.n_iter == n_iter
    assert np.array_equal(res.labels.cpu().numpy(), labels) and np.array_equal(res.mask.cpu().numpy(), mask)
    if _have_sklearn():
        sk = _fit_sklearn(oracle, tied, k)
        np.testing.assert_allclose(np.sort(res.cluster_centers_), np.sort(sk[0]), rtol=0, atol=1e-9)
        assert np.array_equal(res.mask.cpu().numpy(), sk[2])
    with pytest.raises(ValueError, match="n_samples=%d should be >= n_clusters=%d" % (k - 1, k)):
        hipr_b200.kmeans_threshold(torch_cuda.from_numpy(a[:k - 1]).cuda(), k)
    if _have_sklearn():
        with pytest.raises(ValueError):
            oracle.kmeans1d_sklearn(a[:k - 1], k)


SIZES = {"n31": 31, "n511": 511, "n513": 513, "n4113": 4096 + 17}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SIZES))
@pytest.mark.parametrize("k", [2, 3, 5])
def test_gpu_odd_sizes(torch_cuda, oracle, name, k):
    """Sizes below, at and just past one CTA's 512-sample chunk, and a chunk that ends inside a warp."""
    run_case(torch_cuda, oracle, mixture((SIZES[name],), np.random.default_rng(SIZES[name] + k), modes=k), k, n_init=3)


@pytest.mark.gpu
@pytest.mark.parametrize("grid", ["1", "2", "147", "sms", "2sms"])
def test_gpu_grid_shapes(torch_cuda, oracle, grid):
    """hipr_kmeans1d launches min(SMs x resident CTAs per SM, ceil(n / 512)) CTAs.  The kernel's 126 registers x 512
    threads leave room for one CTA per SM on sm_100a, so the full grid is the SM count (148 on a B200).  Sizes whose
    grid is 1, 2, 147 CTAs and the full grid, each with a last CTA that ends inside a warp (n = grid x 512 - 17);
    "2sms" gives the full grid with 1024-sample chunks."""
    sms = torch_cuda.cuda.get_device_properties(0).multi_processor_count
    g = {"sms": sms, "2sms": 2 * sms}.get(grid) or int(grid)
    n = g * KM_THREADS - 17
    img = mixture((n,), np.random.default_rng(g), modes=3)
    for k in (2, 3):
        run_case(torch_cuda, oracle, img, k, n_init=3)


@pytest.mark.gpu
def test_gpu_full_size_score_map_and_volume(torch_cuda, oracle):
    """One full 2048 x 2048 score-map-like image (k = 3) and a 64 x 256 x 256 z-stack volume (k = 2, log10), both
    reaching the full grid; n_init = 1 keeps scikit-learn at about 2 s a fit."""
    run_case(torch_cuda, oracle, kmeans_case(21, (2048, 2048)), 3)
    vol = smooth_image((64, 256, 256), 5, noise=0.2)
    run_case(torch_cuda, oracle, vol, 2, transform="log10", eps=1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(2, 9))
def test_gpu_k_and_n_init(torch_cuda, oracle, k):
    """k = 2..8 with n_init 1, 3, 10 and the largest the kernel accepts; one more raises a clear ValueError."""
    import hipr_b200
    img = mixture((100, 200), np.random.default_rng(100 + k))
    top = _max_n_init(k)
    assert hipr_b200.lib().hipr_kmeans1d_uniforms(k, top) > 0 > hipr_b200.lib().hipr_kmeans1d_uniforms(k, top + 1)
    for n_init in sorted({1, 3, min(10, top), top}):
        run_case(torch_cuda, oracle, img, k, n_init=n_init)
    with pytest.raises(ValueError, match="n_init=%d is too large for k=%d" % (top + 1, k)):
        hipr_b200.kmeans_threshold(torch_cuda.from_numpy(img).cuda(), k, n_init=top + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3])
def test_gpu_float64_not_float32_representable(torch_cuda, oracle, k):
    rng = np.random.default_rng(7 + k)
    img = mixture((120, 130), rng).astype(np.float64) + 1e-9 * rng.random((120, 130))
    assert not np.array_equal(img, img.astype(np.float32).astype(np.float64))
    run_case(torch_cuda, oracle, img, k, n_init=3)
    run_case(torch_cuda, oracle, img, k, transform="log", eps=1e-6, positive_only=True)


@pytest.mark.gpu
@pytest.mark.parametrize("transform,eps,positive_only", [("log10", 1e-3, False), ("log10", 1e-3, True), ("log", 1e-2, False),
                                                         ("log", 1e-2, True), ("log10", 0.0, True), ("log", 0.0, True)])
def test_gpu_transforms_on_counts(torch_cuda, oracle, transform, eps, positive_only):
    """12-bit counts with zeros; eps = 0 only with positive_only (test_gpu_log_of_zero_raises: the zeros raise)."""
    rng = np.random.default_rng(3)
    img = np.clip(np.round(rng.gamma(1.5, 300.0, (150, 170))), 0, 4095).astype(np.float32)
    img[rng.random(img.shape) < 0.2] = 0.0
    for k in (2, 3):
        run_case(torch_cuda, oracle, img, k, n_init=3, transform=transform, eps=eps, positive_only=positive_only)


@pytest.mark.gpu
@pytest.mark.parametrize("transform", ["log10", "log"])
def test_gpu_log_of_zero_raises(torch_cuda, oracle, transform):
    import hipr_b200
    img = kmeans_case(3)
    assert (img == 0).any()
    with pytest.raises(ValueError, match="NaN or infinity"):
        hipr_b200.kmeans_threshold(torch_cuda.from_numpy(img).cuda(), 2, transform=transform, eps=0.0)
    if _have_sklearn():
        with pytest.raises(ValueError), np.errstate(divide="ignore"):
            oracle.kmeans1d_sklearn(img, 2, transform=transform, eps=0.0)


def _positive_layout(layout, rng):
    """(64, 512) images (64 CTAs of one 512-sample row each) whose zeros leave whole warps or CTAs without a valid
    sample."""
    img = mixture((64, 512), rng, modes=3)
    if layout == "first_rows_zero":          # CTAs 0 and 1 (and so warp 0 of block 0) have no valid sample
        img[:2] = 0.0
    elif layout == "first_warp_zero":        # block 0 has valid samples, its warp 0 none
        img[0, :32] = 0.0
    elif layout == "trailing_ctas_zero":
        img[40:] = 0.0
    elif layout == "one_cta":                # every valid sample in CTA 40
        keep = img[40].copy()
        img[:] = 0.0
        img[40] = keep
    else:
        assert layout == "scattered_zeros"
        img[rng.random(img.shape) < 0.5] = 0.0
    return img


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["first_rows_zero", "first_warp_zero", "trailing_ctas_zero", "one_cta", "scattered_zeros"])
def test_gpu_positive_only_layouts(torch_cuda, oracle, layout):
    img = _positive_layout(layout, np.random.default_rng(11))
    for k in (2, 3):
        run_case(torch_cuda, oracle, img, k, n_init=3, positive_only=True)


def _two_levels_background_first(rng):
    """Zero first row, then two positive levels: with k = 3 the first two seeds cover every valid value, so the third
    seed's target is 0, and warp 0 of block 0 holds no valid sample."""
    img = np.where(rng.random((32, 512)) < 0.5, 0.25, 0.75).astype(np.float32)
    img[0] = 0.0
    return img


@pytest.mark.gpu
def test_gpu_more_clusters_than_levels_raises(torch_cuda, oracle):
    """Where a cluster runs empty scikit-learn relocates it and warns; the kernel and the restatement both raise."""
    img = _two_levels_background_first(np.random.default_rng(1))
    assert run_case(torch_cuda, oracle, img, 3, n_init=3, positive_only=True) is None
    levels = (np.random.default_rng(2).integers(0, 6, 5000) / 5.0).astype(np.float32)
    assert run_case(torch_cuda, oracle, levels, 8) is None


@pytest.mark.gpu
@pytest.mark.parametrize("max_iter,tol", [(1, 1e-4), (2, 1e-4), (300, 0.0)])
@pytest.mark.parametrize("k", [2, 3])
def test_gpu_iteration_control(torch_cuda, oracle, max_iter, tol, k):
    """max_iter = 1 and 2 stop before convergence: the labels are those of the final centres, as scikit-learn reruns
    its assignment step; tol = 0 stops only on unchanged labels or a zero shift."""
    img = kmeans_case(30 + k)
    for n_init in (1, 3):
        res = run_case(torch_cuda, oracle, img, k, n_init=n_init, max_iter=max_iter, tol=tol)
        assert res.n_iter <= max_iter


@pytest.mark.gpu
@pytest.mark.parametrize("fill_label", [0, 7, -1])
def test_gpu_fill_label(torch_cuda, oracle, fill_label):
    img = kmeans_case(40)
    run_case(torch_cuda, oracle, img, 3, positive_only=True, fill_label=fill_label)


@pytest.mark.gpu
@pytest.mark.parametrize("return_labels,return_mask", [(False, True), (True, False), (False, False)])
def test_gpu_optional_outputs(torch_cuda, oracle, return_labels, return_mask):
    run_case(torch_cuda, oracle, kmeans_case(41), 2, n_init=3, return_labels=return_labels, return_mask=return_mask)


@pytest.mark.gpu
@pytest.mark.parametrize("view", ["transpose", "strided"])
def test_gpu_non_contiguous_view(torch_cuda, oracle, view):
    f = {"transpose": lambda t: t.t(), "strided": lambda t: t[::2, 1::3]}[view]
    run_case(torch_cuda, oracle, kmeans_case(42), 2, view=f)
    run_case(torch_cuda, oracle, kmeans_case(43), 3, positive_only=True, view=f)


# ---- GPU: results must not depend on what the workspace held -----------------------------------------------------

def _raw_call(torch, img, k, n_init, positive_only, work, pattern, fill_work=True):
    """hipr_kmeans1d through the C ABI with every output (and the workspace, if fill_work) pre-filled with `pattern`."""
    import hipr_b200
    from hipr_b200 import ops
    lib = hipr_b200.lib()
    x = torch.from_numpy(np.ascontiguousarray(img)).cuda()
    u = np.ascontiguousarray(np.random.RandomState(0).random_sample(lib.hipr_kmeans1d_uniforms(k, n_init)))
    labels = torch.empty(x.shape, dtype=torch.int32, device="cuda")
    mask = torch.empty(x.shape, dtype=torch.uint8, device="cuda")
    res = torch.empty(32, dtype=torch.float64, device="cuda")
    for t in (labels, mask, res) + ((work,) if fill_work else ()):
        t.view(torch.uint8).fill_(pattern)
    torch.cuda.synchronize()
    code = lib.hipr_kmeans1d(C.c_void_p(x.data_ptr()), ops.F32, x.numel(), 0, 0.0, int(positive_only), k, n_init,
                             u.ctypes.data_as(C.c_void_p), 300, 1e-4, C.c_void_p(work.data_ptr()),
                             C.c_void_p(labels.data_ptr()), 0, C.c_void_p(mask.data_ptr()), C.c_void_p(res.data_ptr()),
                             ops._stream())
    assert code == 0
    torch.cuda.synchronize()
    return res.cpu().numpy(), labels.cpu().numpy(), mask.cpu().numpy()


@pytest.mark.gpu
def test_gpu_result_independent_of_workspace_contents(torch_cuda):
    """Status, result, labels and mask are bit-identical whether the workspace held 0x3F or 0x7F bytes: on a normal
    case, on the zero-target seeding of _two_levels_background_first (k = 3), and on a second call that reuses the
    workspace of a call on a different input."""
    import hipr_b200
    nbytes = int(hipr_b200.lib().hipr_kmeans1d_workspace_bytes())
    cases = [(kmeans_case(1), 2, 3, False), (_two_levels_background_first(np.random.default_rng(1)), 3, 1, True),
             (_positive_layout("first_rows_zero", np.random.default_rng(5)), 3, 3, True)]
    for img, k, n_init, pos in cases:
        runs = []
        for pattern in (0x3F, 0x7F):
            work = torch_cuda.empty(nbytes, dtype=torch_cuda.uint8, device="cuda")
            runs.append(_raw_call(torch_cuda, img, k, n_init, pos, work, pattern))
        (r0, l0, m0), (r1, l1, m1) = runs
        assert np.array_equal(r0.view(np.uint64), r1.view(np.uint64)), "result depends on the workspace: %s / %s" % (r0[:8], r1[:8])
        if r0[0] == 0:
            assert np.array_equal(l0, l1) and np.array_equal(m0, m1)
    # two calls in a row on one workspace, the second on a different input, against a fresh workspace
    work = torch_cuda.empty(nbytes, dtype=torch_cuda.uint8, device="cuda")
    first, second = cases[0], cases[2]
    _raw_call(torch_cuda, first[0], first[1], first[2], first[3], work, 0x3F)
    again = _raw_call(torch_cuda, second[0], second[1], second[2], second[3], work, 0x7F, fill_work=False)
    fresh = _raw_call(torch_cuda, second[0], second[1], second[2], second[3],
                      torch_cuda.empty(nbytes, dtype=torch_cuda.uint8, device="cuda"), 0x3F)
    assert np.array_equal(again[0].view(np.uint64), fresh[0].view(np.uint64))
    assert np.array_equal(again[1], fresh[1]) and np.array_equal(again[2], fresh[2])
