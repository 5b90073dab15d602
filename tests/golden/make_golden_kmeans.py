"""Freezes scikit-learn's answers for the 1-D k-means row (SURVEY.md 8f rank 3) so that the pin also holds where
scikit-learn is a different version: inputs are regenerated from seeds, the outputs of
sklearn.cluster.KMeans (version recorded) are stored.

    python tests/golden/make_golden_kmeans.py
"""
import hashlib
import os
import sys

import numpy as np
import sklearn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import hipr_oracle as O  # noqa: E402


def kmeans_case(seed, shape=(96, 128)):
    """A score-map-like image: dark background, bright cells, a few exact zeros; float32 representable."""
    rng = np.random.default_rng(seed)
    img = rng.normal(0.12, 0.04, shape)
    yy, xx = np.mgrid[:shape[0], :shape[1]]
    for _ in range(12):
        cy, cx = rng.integers(8, shape[0] - 8), rng.integers(8, shape[1] - 8)
        img += (0.45 + 0.25 * rng.random()) * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * (3 + 3 * rng.random()) ** 2))
    img = np.clip(img, 0, None)
    img[rng.random(shape) < 0.02] = 0.0
    return img.astype(np.float32)


def levels6_vector():
    """19,918 float32 values on the six levels {0, 0.2, ..., 1.0}, as quantised counts give.  With positive_only, k = 2
    and n_init = 3 the third initialisation has centre-ordered cluster sizes (6584, 9977) against the first's (9977,
    6584) and a lower inertia, so scikit-learn takes it: comparing sorted sizes would call the two the same clustering.
    The draws before the vector replay the seeded sweep that found it, so that it is the same vector."""
    rng = np.random.default_rng(0)
    for t in range(3):
        n = int(rng.integers(200, 40000))
        rng.normal(size=n)
        rng.normal(size=n // 3) if t < 2 else rng.random(n)
    return (rng.integers(0, 6, int(rng.integers(200, 40000))) / 5.0).astype(np.float32)


def case_image(seed):
    return levels6_vector() if seed == "levels6" else kmeans_case(seed)


CASES = [  # (seed, k, n_init, transform, eps, positive_only)
    (1, 2, 1, None, 0.0, False),
    (2, 3, 1, None, 0.0, False),
    (3, 2, 1, "log10", 1e-8, False),
    (4, 2, 1, "log", 1e-2, False),
    (5, 2, 1, None, 0.0, True),
    (6, 3, 1, None, 0.0, True),
    (7, 2, 3, None, 0.0, False),
    ("levels6", 2, 3, None, 0.0, True),
    ("levels6", 2, 10, None, 0.0, True),
    ("levels6", 3, 10, None, 0.0, True),
]


def main():
    """Cases already in the archive keep their stored values: scikit-learn's OpenMP reductions change the last bits of
    centres and inertia with the thread count, so a rerun is only checked against them (labels, mask, n_iter exact,
    centres 1e-12, inertia rtol 1e-10)."""
    path = os.path.join(HERE, "kmeans_vectors.npz")
    old = dict(np.load(path)) if os.path.exists(path) else {}
    out = {"sklearn_version": np.array(sklearn.__version__)}
    for i, (seed, k, n_init, tr, eps, pos) in enumerate(CASES):
        img = case_image(seed)
        cen, labels, mask, n_iter, inertia = O.kmeans1d_sklearn(img, k, 0, n_init, tr, eps, pos)
        new = {"case%d_centers" % i: cen,
               "case%d_n_iter" % i: np.array(n_iter),
               "case%d_inertia" % i: np.array(inertia),
               "case%d_labels_sha256" % i: np.frombuffer(hashlib.sha256(labels.astype(np.int32).tobytes()).digest(), dtype=np.uint8),
               "case%d_mask_sum" % i: np.array(int(mask.sum())),
               "case%d_img_sha256" % i: np.frombuffer(hashlib.sha256(img.tobytes()).digest(), dtype=np.uint8)}
        if "case%d_centers" % i in old:
            for key, v in new.items():
                if key.endswith("_centers"):
                    np.testing.assert_allclose(v, old[key], rtol=0, atol=1e-12, err_msg=key)
                elif key.endswith("_inertia"):
                    np.testing.assert_allclose(v, old[key], rtol=1e-10, err_msg=key)
                else:
                    assert np.array_equal(v, old[key]), key
                new[key] = old[key]
        out.update(new)
    np.savez_compressed(path, **out)
    print("wrote kmeans_vectors.npz with", len(CASES), "cases, scikit-learn", sklearn.__version__)


if __name__ == "__main__":
    main()
