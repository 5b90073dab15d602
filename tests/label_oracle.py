"""numpy / scipy reference for the connected-component operators (csrc/label.cu, K10): label, remove_small_objects,
binary_fill_holes, clear_border and relabel_sequential, the segmentation back end between the k-means mask and the label
image (syn/..._measurement.py:125-158, eco/..._measurement.py:73-127, bio/..._analysis.py:367-419, 463-501).  The checker
in tests/test_label.py and tests/test_gpu_label.py; never imported by the product.  TEST
INFRASTRUCTURE ONLY.

The binary operators are thin wrappers around scipy.ndimage (pinned: 1.18.1 is installed), which numbers components in
raster order of their first pixel.  The label-image operators restate scikit-image, which is absent here and which the
reference does not pin: PARITY UNPINNED for those.
"""
import numpy as np


def _structure(ndim, connectivity):
    import scipy.ndimage as ndi
    return ndi.generate_binary_structure(ndim, ndim if connectivity is None else connectivity)


def label_mask(mask, connectivity=None):
    """scipy.ndimage.label(mask != 0, generate_binary_structure(ndim, connectivity)) -> (int32 labels, n)."""
    import scipy.ndimage as ndi
    mask = np.asarray(mask) != 0
    lab, n = ndi.label(mask, _structure(mask.ndim, connectivity))
    return lab.astype(np.int32), int(n)


def label_image(image, connectivity=None):
    """skimage.measure.label(image, background=0, connectivity) for an integer label image
    (skimage/measure/_ccomp.pyx: union-find over equal-valued non-zero neighbours, root = smallest raster index,
    then numbered in raster order).  PARITY UNPINNED.  Restated as the connected components
    (scipy.sparse.csgraph) of the graph whose edges join equal, non-zero neighbours under the structure of
    `connectivity`, renumbered by first pixel -> (int32 labels, n)."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    image = np.asarray(image)
    st = _structure(image.ndim, connectivity)
    idx = np.arange(image.size).reshape(image.shape)
    rows, cols = [idx.ravel()], [idx.ravel()]
    centre = np.array(st.shape) // 2
    for off in np.argwhere(st) - centre:
        if tuple(off) <= (0,) * image.ndim:
            continue                                        # each pair once, and not the centre
        a = tuple(slice(max(0, -o), image.shape[d] - max(0, o)) for d, o in enumerate(off))
        b = tuple(slice(max(0, o), image.shape[d] - max(0, -o)) for d, o in enumerate(off))
        join = (image[a] == image[b]) & (image[a] != 0)
        rows.append(idx[a][join])
        cols.append(idx[b][join])
    r, c = np.concatenate(rows), np.concatenate(cols)
    graph = coo_matrix((np.ones(r.size, np.int8), (r, c)), shape=(image.size, image.size))
    _, comp = connected_components(graph, directed=False)
    flat = image.ravel()
    fg = np.flatnonzero(flat != 0)
    first = np.unique(comp[fg], return_index=True)[1]       # first pixel of each component, in raster order
    ids = comp[fg][np.sort(first)]
    remap = np.zeros(comp.max() + 1, np.int64)
    remap[ids] = np.arange(1, ids.size + 1)
    out = np.zeros(image.size, np.int32)
    out[fg] = remap[comp[fg]]
    return out.reshape(image.shape), int(ids.size)


def remove_small_objects_mask(mask, min_size=64, connectivity=1):
    """skimage.morphology.remove_small_objects for a bool input: scipy.ndimage.label with the structure of
    `connectivity`, components of fewer than min_size pixels removed (scikit-image's own recipe with scipy)."""
    mask = np.asarray(mask, bool)
    if min_size == 0:
        return mask.copy()
    lab, _ = label_mask(mask, connectivity)
    sizes = np.bincount(lab.ravel())
    out = mask.copy()
    out[sizes[lab] < min_size] = False
    return out


def remove_small_objects_labels(labels, min_size=64):
    """skimage.morphology.remove_small_objects for an integer input (skimage/morphology/misc.py): the labels are
    the components, sizes = np.bincount(labels.ravel()) (ValueError for a negative label), labels of fewer than
    min_size pixels set to 0.  PARITY UNPINNED."""
    labels = np.asarray(labels)
    if min_size == 0:
        return labels.copy()
    sizes = np.bincount(labels.ravel())
    out = labels.copy()
    out[sizes[labels] < min_size] = 0
    return out


def binary_fill_holes(mask, connectivity=1):
    """scipy.ndimage.binary_fill_holes(mask, generate_binary_structure(ndim, connectivity))."""
    import scipy.ndimage as ndi
    mask = np.asarray(mask) != 0
    return ndi.binary_fill_holes(mask, _structure(mask.ndim, connectivity))


def clear_border(labels, buffer_size=0, bgval=0):
    """skimage.segmentation.clear_border(labels, buffer_size, bgval) (skimage/segmentation/_clear_border.py):
    a band of buffer_size + 1 pixels along every edge; the image relabelled with label(labels, background=0) at
    full connectivity; every component (the background, label 0, included) with a pixel in the band set to bgval.
    PARITY UNPINNED."""
    image = np.asarray(labels)
    if any(buffer_size >= s for s in image.shape):
        raise ValueError("buffer size may not be greater than labels size")
    out = image.copy()
    borders = np.zeros(image.shape, bool)
    ext = buffer_size + 1
    for d in range(image.ndim):
        sl = [slice(None)] * image.ndim
        sl[d] = slice(ext)
        borders[tuple(sl)] = True
        sl[d] = slice(-ext, None)
        borders[tuple(sl)] = True
    if image.dtype == bool or image.dtype == np.uint8:
        lab, n = label_mask(image, image.ndim)
    else:
        lab, n = label_image(image, image.ndim)
    touched = np.isin(np.arange(n + 1), np.unique(lab[borders]))
    out[touched[lab]] = bgval
    return out


def relabel_sequential(labels, offset=1):
    """skimage.segmentation.relabel_sequential(labels, offset) in its array form (scikit-image <= 0.17 returned
    these arrays; later versions wrap them in ArrayMap): -> (relabelled, forward_map (max + 1,), inverse_map
    (offset + n,)).  PARITY UNPINNED."""
    labels = np.asarray(labels)
    if offset <= 0:
        raise ValueError("Offset must be strictly positive.")
    if labels.min() < 0:
        raise ValueError("Cannot relabel array that contains negative values.")
    present = np.unique(labels)
    present = present[present != 0]
    n = len(present)
    out_dtype = labels.dtype if offset + n - 1 <= np.iinfo(labels.dtype).max else np.int64
    forward = np.zeros(int(labels.max()) + 1, out_dtype)
    forward[present] = np.arange(offset, offset + n)
    inverse = np.zeros(offset + n, labels.dtype)
    inverse[offset:] = present
    return forward[labels], forward, inverse
