"""Pure Python / numpy references for the marker watershed (K11, csrc/watershed.cu).  Test infrastructure only.

scikit-image is not installed and the reference pins no version of it: PARITY UNPINNED.

watershed_heap  a loop-for-loop restatement of scikit-image's non-compact flood
                (skimage/segmentation/_watershed_cy.pyx, watershed_raveled with compactness 0, no watershed line): the
                markers (markers * mask) are pushed at age 0, and a popped pixel labels every unlabelled in-mask
                neighbour with its own label and pushes it with the next age.  The heap is keyed by (value, age, index):
                the index only orders equal-valued markers at age 0, where scikit-image's own heap layout decides.
                Also returns each pixel's popper, its level (the running maximum of the popped values when it was
                popped) and the tie-decided pixels (two neighbours of minimal level with different final labels).
watershed_rule  the deterministic rule the device computes (DESIGN.md K11), by the same heap loop keyed by
                K = (L, d, label): a pixel's key is f(K(q), p) of the first neighbour q popped, where
                f((L, d, l), p) = (L, d + 1, l) if v(p) <= L else (v(p), 1, l).

Both take an image (float), markers (int, any non-zero value is a marker), a connectivity 1 .. ndim and an optional
boolean mask, in 2-D or 3-D, and return labels of the markers' dtype (0 outside the mask and where no marker reaches).
A 2048 x 2048 image takes tens of seconds on one core.
"""
import heapq
import itertools
from collections import namedtuple

import numpy as np

HeapResult = namedtuple("HeapResult", "labels popper level tied")


def offsets(ndim, connectivity):
    """scipy's generate_binary_structure(ndim, connectivity) without the centre."""
    return [d for d in itertools.product((-1, 0, 1), repeat=ndim) if 0 < sum(map(abs, d)) <= connectivity]


def _prepare(image, markers, connectivity, mask):
    image = np.asarray(image)
    markers = np.asarray(markers)
    if image.shape != markers.shape or image.ndim not in (2, 3):
        raise ValueError("image and markers must be 2-D or 3-D arrays of one shape")
    if not 1 <= connectivity <= image.ndim:
        raise ValueError("connectivity must be in [1, ndim]")
    inside = np.ones(image.shape, bool) if mask is None else np.asarray(mask).astype(bool)
    markers = markers * inside                                    # scikit-image's _validate_inputs
    pshape = tuple(s + 2 for s in image.shape)
    strides = np.cumprod((1,) + pshape[::-1][:-1])[::-1]
    offs = [int(np.dot(d, strides)) for d in offsets(image.ndim, connectivity)]
    core = tuple(slice(1, -1) for _ in pshape)
    val = np.zeros(pshape)
    val[core] = image.astype(np.float64) + 0.0                    # -0.0 + 0.0 = +0.0; the heap's == treats them alike
    lab = np.zeros(pshape, np.int64)
    lab[core] = markers
    inm = np.zeros(pshape, bool)
    inm[core] = inside
    return val.ravel().tolist(), lab.ravel().tolist(), inm.ravel().tolist(), offs, pshape, core, markers.dtype


def _unpad(flat, pshape, core, dtype):
    return np.asarray(flat).reshape(pshape)[core].astype(dtype)


def watershed_heap(image, markers, connectivity=1, mask=None):
    """-> HeapResult(labels, popper (flat image index of the pixel whose pop labelled it, -1 for markers and
    unlabelled pixels), level (float64; inf where unlabelled), tied (bool))."""
    val, lab, inm, offs, pshape, core, dtype = _prepare(image, markers, connectivity, mask)
    n = len(val)
    popper = [-1] * n
    level = [np.inf] * n
    heap = [(val[i], 0, i) for i in range(n) if lab[i] != 0]
    heapq.heapify(heap)
    age = 1
    run = -np.inf
    while heap:
        v, _, i = heapq.heappop(heap)
        run = v if v > run else run
        level[i] = run
        li = lab[i]
        for o in offs:
            j = i + o
            if not inm[j] or lab[j] != 0:
                continue
            lab[j] = li
            popper[j] = i
            heapq.heappush(heap, (val[j], age, j))
            age += 1
    labels = _unpad(lab, pshape, core, dtype)
    lev = _unpad(level, pshape, core, np.float64)
    # popper as a flat index of the unpadded image
    pop = np.asarray(popper).reshape(pshape)
    coords = np.unravel_index(np.where(pop >= 0, pop, 0), pshape)
    flat = np.ravel_multi_index(tuple(c - 1 for c in coords), labels.shape, mode="clip")
    flat = np.where(pop >= 0, flat, -1)[core]
    markers = np.asarray(markers) * (np.ones(labels.shape, bool) if mask is None else np.asarray(mask).astype(bool))
    return HeapResult(labels, flat, lev, tie_decided(labels, lev, markers != 0, connectivity))


def tie_decided(labels, level, is_marker, connectivity):
    """Non-marker labelled pixels with two neighbours of minimal level (among the labelled neighbours) whose labels
    differ."""
    labels = np.asarray(labels)
    lev = np.pad(np.asarray(level, np.float64), 1, constant_values=np.inf)
    lab = np.pad(labels.astype(np.int64), 1)
    core = tuple(slice(1, -1) for _ in lev.shape)
    shifted = []
    for d in offsets(labels.ndim, connectivity):
        sl = tuple(slice(1 + k, s - 1 + k) for k, s in zip(d, lev.shape))
        shifted.append((lev[sl], lab[sl]))
    ml = np.min([s[0] for s in shifted], axis=0)
    big = np.iinfo(np.int64).max
    lo = np.min([np.where(s[0] == ml, s[1], big) for s in shifted], axis=0)
    hi = np.max([np.where(s[0] == ml, s[1], -big) for s in shifted], axis=0)
    return np.isfinite(lev[core]) & ~np.asarray(is_marker) & np.isfinite(ml) & (lo != hi)


def watershed_rule(image, markers, connectivity=1, mask=None):
    """The device's rule, by the heap loop keyed by K = (L, d, label)."""
    val, lab, inm, offs, pshape, core, dtype = _prepare(image, markers, connectivity, mask)
    n = len(val)
    heap = [(val[i], 0, lab[i], i) for i in range(n) if lab[i] != 0]
    heapq.heapify(heap)
    while heap:
        L, d, li, i = heapq.heappop(heap)
        for o in offs:
            j = i + o
            if not inm[j] or lab[j] != 0:
                continue
            lab[j] = li
            vj = val[j]
            heapq.heappush(heap, (L, d + 1, li, j) if vj <= L else (vj, 1, li, j))
    return _unpad(lab, pshape, core, dtype)
