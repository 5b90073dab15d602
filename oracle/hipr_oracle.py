"""CPU oracle for the HiPR-FISH spectral-segmentation front end.  TEST INFRASTRUCTURE ONLY.

This module is a numpy restatement of the reference algorithm; it is the checker, never the
product.  Only tests/, __graft_entry__.smoke() and bench.py's CPU legs import it.  The product
(hiprfish-image-analysis_b200/) never does and has no CPU fallback.

Parity status: PINNED.  The reference ships no tests or golden vectors (SURVEY.md §4), but
its native stencils compile here unmodified (oracle/build_ref.py -> oracle/_ref/), and
tests/test_oracle.py checks every function below against that compiled reference;
tests/golden/ freezes vectors generated from it (tests/golden/make_golden.py) so the pin
also holds on the GPU box where /root/reference is absent.  The per-cell reduction follows
scikit-image's regionprops (third-party, NOT vendored in the reference, version not pinned
anywhere in the reference; era skimage 0.14-0.15): for that one function parity is pinned only
on its published definition (arithmetic mean over label==L pixels, ascending present labels)
and cross-checked against scipy.ndimage.mean.

Paths are relative to /root/reference:
  eco/ = hiprfish-image-analysis-ecoli/        bio/ = hiprfish-image-analysis-biofilm/
  syn/ = hiprfish-image-analysis-synthetic-community/
"""
import numpy as np

# --------------------------------------------------------------------------------------------
# Offset tables
# --------------------------------------------------------------------------------------------

def _fill_line(tab, col, steps, half):
    """Fill tab[:, :, col] for one direction.

    `steps` = the rounded end-point offsets of the half line (one per axis).  Follows
    eco/neighbor2d.pyx:36-55 (2-D) and bio/neighbor.pyx:147-170 (3-D, same construction with a
    third axis): the longest axis decides how many distinct samples the line has; shorter lines
    are centred and their two end samples replicated.
    """
    P = tab.shape[0]
    steps = np.asarray(steps, dtype=np.int64)
    longest = steps[np.argmax(np.abs(steps))]
    sgn = np.sign(steps)
    n = int(2 * abs(longest) + 1)
    first = int((P - n) / 2) if n < P else 0
    for li in range(n):
        for ax in range(len(steps)):
            h = sgn[ax] * li * (2 * abs(steps[ax]) + 1) / n          # true division
            tab[li + first, ax, col] = int(np.sign(h) * np.floor(np.abs(h)) + half - steps[ax])
    if n < P:
        for li in range(first):
            tab[li, :, col] = tab[first, :, col]
        for li in range(first):
            tab[li + n + first, :, col] = tab[n + first - 1, :, col]


def line_table_2d(patch_size, phi_range):
    """(P, 2, R) int64 patch coordinates, eco/neighbor2d.pyx:32-55."""
    half = int((patch_size - 1) / 2)
    tab = np.zeros((patch_size, 2, phi_range), dtype=np.int64)
    for phi in range(phi_range):
        a = int(np.round(half * np.cos(phi * np.pi / phi_range)))
        b = int(np.round(half * np.sin(phi * np.pi / phi_range)))
        _fill_line(tab, phi, (a, b), half)
    return tab


def line_table_3d(patch_size, theta_range, phi_range):
    """(P, 3, (theta_range-1)*phi_range) int64, bio/neighbor.pyx:141-170 (v2 and me_v2)."""
    half = int((patch_size - 1) / 2)
    tab = np.zeros((patch_size, 3, (theta_range - 1) * phi_range), dtype=np.int64)
    for theta in range(1, theta_range):
        for phi in range(phi_range):
            col = (theta - 1) * phi_range + phi
            st = np.sin(theta * np.pi / theta_range)
            a = int(np.round(half * np.cos(phi * np.pi / phi_range) * st))
            b = int(np.round(half * np.sin(phi * np.pi / phi_range) * st))
            c = int(np.round(half * np.cos(theta * np.pi / theta_range)))
            _fill_line(tab, col, (a, b, c), half)
    return tab


def line_table_3d_v3(patch_size, theta_range, phi_range):
    """(P, 3, T) int64 table of line_profile_memory_efficient_v3, bio/neighbor.pyx:301-324.

    Differs from line_table_3d: short lines use np.round of the signed fraction (:313-315);
    full-length lines use np.floor of sign*li*(2*step+1)/n with the SIGNED step (:322-324).
    """
    half = int((patch_size - 1) / 2)
    T = (theta_range - 1) * phi_range
    tab = np.zeros((patch_size, 3, T), dtype=np.int64)
    for theta in range(1, theta_range):
        for phi in range(phi_range):
            col = (theta - 1) * phi_range + phi
            st = np.sin(theta * np.pi / theta_range)
            steps = np.array([int(np.round(half * np.cos(phi * np.pi / phi_range) * st)),
                              int(np.round(half * np.sin(phi * np.pi / phi_range) * st)),
                              int(np.round(half * np.cos(theta * np.pi / theta_range)))], dtype=np.int64)
            longest = steps[np.argmax(np.abs(steps))]
            sgn = np.sign(steps)
            n = int(2 * abs(longest) + 1)
            if n < patch_size:
                first = int((patch_size - n) / 2)
                for li in range(n):
                    for ax in range(3):
                        tab[li + first, ax, col] = int(np.round(sgn[ax] * li * (2 * abs(steps[ax]) + 1) / n)
                                                       + half - steps[ax])
                for li in range(first):
                    tab[li, :, col] = tab[first, :, col]
                for li in range(first):
                    tab[li + n + first, :, col] = tab[n + first - 1, :, col]
            else:
                for li in range(n):
                    for ax in range(3):
                        tab[li, ax, col] = int(np.floor(sgn[ax] * li * (2 * steps[ax] + 1) / n)
                                               + half - steps[ax])
    return tab


# --------------------------------------------------------------------------------------------
# Stencils (vectorised restatements of the native hot loops)
# --------------------------------------------------------------------------------------------

def line_profile_2d_v2(image_padded, patch_size, phi_range):
    """eco/neighbor2d.pyx:8-64: lp[i,j,t,li] = image_padded[i+tab[li,0,t], j+tab[li,1,t]]."""
    a = np.asarray(image_padded)
    if a.dtype != np.float64:
        raise ValueError("Buffer dtype mismatch, expected 'double' but got '%s'" % a.dtype)
    if a.ndim != 2:
        raise ValueError("Buffer has wrong number of dimensions (expected 2, got %d)" % a.ndim)
    tab = line_table_2d(patch_size, phi_range)
    H = a.shape[0] - (patch_size - 1)
    W = a.shape[1] - (patch_size - 1)
    out = np.zeros((H, W, phi_range, patch_size), dtype=np.float64)
    for t in range(phi_range):
        for li in range(patch_size):
            di, dj = tab[li, 0, t], tab[li, 1, t]
            out[:, :, t, li] = a[di:di + H, dj:dj + W]
    return out


def _gather3d(a, tab, patch_size):
    X = a.shape[0] - (patch_size - 1)
    Y = a.shape[1] - (patch_size - 1)
    Z = a.shape[2] - (patch_size - 1)
    T = tab.shape[2]
    out = np.zeros((X, Y, Z, T, patch_size), dtype=np.float64)
    for t in range(T):
        for li in range(patch_size):
            di, dj, dk = tab[li, :, t]
            out[:, :, :, t, li] = a[di:di + X, dj:dj + Y, dk:dk + Z]
    return out


def _gather3d_flat(a, tab, patch_size):
    """Gather for the v3 table, whose entries reach 18 for (11,9,9): the reference indexes an
    11^3 memoryview slice with them, bounds checks off (bio/neighbor.pyx:265-267,328-334), i.e.
    it reads image_padded's buffer at the flat address.  In-buffer addresses are reproduced
    exactly; an address past the end of the buffer (undefined behaviour in the reference)
    yields NaN here."""
    a = np.ascontiguousarray(a)
    Xp, Yp, Zp = a.shape
    X, Y, Z = Xp - (patch_size - 1), Yp - (patch_size - 1), Zp - (patch_size - 1)
    T = tab.shape[2]
    flat = np.concatenate([a.reshape(-1), [np.nan]])
    i, j, k = np.meshgrid(np.arange(X), np.arange(Y), np.arange(Z), indexing="ij")
    out = np.zeros((X, Y, Z, T, patch_size), dtype=np.float64)
    for t in range(T):
        for li in range(patch_size):
            di, dj, dk = tab[li, :, t]
            idx = ((i + di) * Yp + (j + dj)) * Zp + (k + dk)
            idx = np.where((idx >= 0) & (idx < a.size), idx, a.size)
            out[:, :, :, t, li] = flat[idx]
    return out


def _check3d(a):
    if a.dtype != np.float64:
        raise ValueError("Buffer dtype mismatch, expected 'double' but got '%s'" % a.dtype)
    if a.ndim != 3:
        raise ValueError("Buffer has wrong number of dimensions (expected 3, got %d)" % a.ndim)


def line_profile_v2(image_padded, patch_size, theta_range, phi_range):
    """bio/neighbor.pyx:115-181: 5-D literal gather (X,Y,Z,T,P)."""
    a = np.asarray(image_padded)
    _check3d(a)
    return _gather3d(a, line_table_3d(patch_size, theta_range, phi_range), patch_size)


def line_profile_memory_efficient_v2(image_padded, patch_size, theta_range, phi_range):
    """bio/neighbor.pyx:186-263: per direction (centre-min)/max(max-min,1e-8) -> (X,Y,Z,T)."""
    a = np.asarray(image_padded)
    _check3d(a)
    lp = _gather3d(a, line_table_3d(patch_size, theta_range, phi_range), patch_size)
    mn = lp.min(axis=4)
    rng = np.maximum(lp.max(axis=4) - mn, 1e-8)
    return (lp[..., int((patch_size - 1) / 2)] - mn) / rng


def line_profile_memory_efficient_v3(image_padded, patch_size, theta_range, phi_range):
    """bio/neighbor.pyx:268-349: v3 table, then avg*(p25-p75)/(p25+p75+1e-8) per voxel (:342-348)."""
    a = np.asarray(image_padded)
    _check3d(a)
    lp = _gather3d_flat(a, line_table_3d_v3(patch_size, theta_range, phi_range), patch_size)
    mn = lp.min(axis=4)
    rng = np.maximum(lp.max(axis=4) - mn, 1e-8)
    e = (lp[..., int((patch_size - 1) / 2)] - mn) / rng
    T = e.shape[3]
    avg = np.zeros(e.shape[:3])
    for t in range(T):                       # sequential accumulation order of :343-345
        avg += e[..., t]
    avg /= T
    uq = np.percentile(e, 25, axis=3)        # names swapped in the reference (:346-347)
    lq = np.percentile(e, 75, axis=3)
    return avg * (uq - lq) / (uq + lq + 1e-8)


# --------------------------------------------------------------------------------------------
# Prologue / epilogue (numpy blocks of the measurement scripts)
# --------------------------------------------------------------------------------------------

def prologue(cube, calibration=None, normalize=True, pad=5, sum_axes=None):
    """syn/...measurement.py:102-109 without the skimage NLM denoise.

    cube (..., C) -> channel sum over the last axis (or `sum_axes`, bio/...:451) -> /max ->
    edge pad -> float64.  Returns (sum_image, padded_float64).
    """
    x = np.asarray(cube, dtype=np.float64)
    if calibration is not None:
        x = x / np.asarray(calibration, dtype=np.float64)
    s = np.sum(x, axis=(x.ndim - 1) if sum_axes is None else sum_axes)
    sn = s / np.max(s) if normalize else s
    return s, np.pad(sn, pad, mode="edge").astype(np.float64)


def register_stacks(image_stack, shift_vectors, calibration_image=None):
    """Registration paste, channel stack, flat field, channel sum:
    syn/hiprfish_imaging_multispecies_spectral_image_measurement.py:86-105 (test infrastructure).
    shift_vectors: per stack (row, col), truncated with int() as at :89-90.  The reference uses
    image_stack[0].shape[0] for both axes (:87, square images); here rows use H and columns W, the same
    thing on square images.  Returns (image_channel (H, W, C) float64, image_registered_sum (H, W))."""
    image_registered = [np.zeros(image.shape) for image in image_stack]
    H, W = image_stack[0].shape[:2]
    for i in range(len(image_stack)):
        shift_row = int(shift_vectors[i][0])
        shift_col = int(shift_vectors[i][1])
        original_row_min = int(np.maximum(0, shift_row))
        original_row_max = int(H + np.minimum(0, shift_row))
        original_col_min = int(np.maximum(0, shift_col))
        original_col_max = int(W + np.minimum(0, shift_col))
        registered_row_min = int(-np.minimum(0, shift_row))
        registered_row_max = int(H - np.maximum(0, shift_row))
        registered_col_min = int(-np.minimum(0, shift_col))
        registered_col_max = int(W - np.maximum(0, shift_col))
        image_registered[i][original_row_min: original_row_max, original_col_min: original_col_max, :] = \
            image_stack[i][registered_row_min: registered_row_max, registered_col_min: registered_col_max, :]
    image_channel = np.dstack(image_registered)
    if calibration_image is not None:
        image_channel = image_channel / calibration_image
    return image_channel, np.sum(image_channel, axis=2)


NLM_DISTANCE_CUTOFF = 5.0


def denoise_nl_means_2d(image, patch_size=7, patch_distance=11, h=0.1, sigma=0.0):
    """skimage.restoration.denoise_nl_means(image, h=h) for a 2-D grayscale image with the defaults the
    scripts use (fast_mode=True, patch_size=7, patch_distance=11, sigma=0):
    syn/hiprfish_imaging_multispecies_spectral_image_measurement.py:108 (h = 0.02),
    bio/hiprfish_imaging_biofilm_analysis.py:350, 592, 668, 725, 989.

    PARITY UNPINNED: scikit-image is a third-party dependency that the reference neither vendors nor pins
    (era 0.14-0.15) and it is not installed here.  This restates the published algorithm of
    skimage/restoration/_nl_means_denoising.pyx::_fast_nl_means_denoising_2d (Darbon et al. 2008, integral
    images of squared differences, one per patch shift), loop for loop:
      * reflect padding by offset + d + 1, offset = patch_size // 2;
      * for every shift (t_row in [-d, d], t_col in [0, d]): integral image of (padded - shifted)^2 - 2 sigma^2;
        patch distance from its four corners at +-offset (a 2*offset square, NOT patch_size: a quirk of
        the implementation), clipped at 0 and divided by h^2 * patch_size^2;
      * weight = alpha * exp(-distance) unless distance > 5, alpha = 0.5 on the t_col = 0, t_row != 0
        column (visited from both sides); accumulated symmetrically into both pixels of the pair (so the
        zero shift counts twice);
      * result / weights, cropped.
    Vectorised over pixels (numpy), one shift at a time.  Test infrastructure only."""
    image = np.asarray(image, dtype=np.float64)
    if image.ndim != 2:
        raise ValueError("2-D grayscale images only")
    s = int(patch_size)
    if s % 2 == 0:
        s += 1
    d = int(patch_distance)
    offset = s // 2
    pad_size = offset + d + 1
    padded = np.pad(image, pad_size, mode="reflect")
    n_row, n_col = padded.shape
    result = np.zeros_like(padded)
    weights = np.zeros_like(padded)
    h2s2 = h * h * s * s            # n_channels = 1
    var = 2.0 * sigma * sigma
    for t_row in range(-d, d + 1):
        row_start = max(offset, offset - t_row)
        row_end = min(n_row - offset, n_row - offset - t_row)
        for t_col in range(0, d + 1):
            alpha = 0.5 if (t_col == 0 and t_row != 0) else 1.0
            # _integral_image_2d
            integral = np.zeros_like(padded)
            ra, rb = max(1, -t_row), min(n_row, n_row - t_row)
            ca, cb = 1, n_col - t_col
            diff = (padded[ra:rb, ca:cb] - padded[ra + t_row:rb + t_row, ca + t_col:cb + t_col]) ** 2 - var
            integral[ra:rb, ca:cb] = np.cumsum(np.cumsum(diff, axis=0), axis=1)
            # inner loops on pixel coordinates
            col_start, col_end = offset, n_col - offset - t_col
            R = slice(row_start, row_end)
            Cs = slice(col_start, col_end)
            dist = (integral[row_start + offset:row_end + offset, col_start + offset:col_end + offset]
                    + integral[row_start - offset:row_end - offset, col_start - offset:col_end - offset]
                    - integral[row_start - offset:row_end - offset, col_start + offset:col_end + offset]
                    - integral[row_start + offset:row_end + offset, col_start - offset:col_end - offset])
            dist = np.maximum(dist, 0.0) / h2s2
            w = np.where(dist > NLM_DISTANCE_CUTOFF, 0.0, alpha * np.exp(-dist))
            Rs = slice(row_start + t_row, row_end + t_row)
            Css = slice(col_start + t_col, col_end + t_col)
            weights[R, Cs] += w
            weights[Rs, Css] += w
            result[R, Cs] += w * padded[Rs, Css]
            result[Rs, Css] += w * padded[R, Cs]
    out = result[pad_size:-pad_size, pad_size:-pad_size] / weights[pad_size:-pad_size, pad_size:-pad_size]
    return out


def denoise_nl_means_2d_direct(image, patch_size=7, patch_distance=11, h=0.1):
    """The same estimator written pixel by pixel (no integral images, no symmetric accumulation): for every
    pixel p and every shift t in [-d, d]^2, weight = exp(-max(sum over the 2*offset window of
    (v[u] - v[u + t])^2, 0) / (h^2 s^2)) if that distance is <= 5, the zero shift counted twice.  Used to
    check the restatement above against an independent formulation (tests/test_oracle.py); O(N d^2 s^2)."""
    image = np.asarray(image, dtype=np.float64)
    s = int(patch_size) | 1
    d = int(patch_distance)
    offset = s // 2
    pad = offset + d + 1
    v = np.pad(image, pad, mode="reflect")
    H, W = image.shape
    h2s2 = h * h * s * s
    acc_w = np.zeros((H, W))
    acc_v = np.zeros((H, W))
    lo, hi = -offset + 1, offset        # window rows / cols p + lo .. p + hi
    for tr in range(-d, d + 1):
        for tc in range(-d, d + 1):
            a = v[pad + lo: pad + H + hi, pad + lo: pad + W + hi]
            b = v[pad + lo + tr: pad + H + hi + tr, pad + lo + tc: pad + W + hi + tc]
            D = (a - b) ** 2                                  # (H + 2*offset - 1, W + 2*offset - 1)
            box = np.zeros((H, W))
            n = hi - lo + 1
            for i in range(n):
                for j in range(n):
                    box += D[i:i + H, j:j + W]
            dist = np.maximum(box, 0.0) / h2s2
            w = np.where(dist > NLM_DISTANCE_CUTOFF, 0.0, np.exp(-dist))
            if tr == 0 and tc == 0:
                w = 2.0 * w
            acc_w += w
            acc_v += w * v[pad + tr: pad + tr + H, pad + tc: pad + tc + W]
    return acc_v / acc_w


def denoise_nl_means_3d(image, patch_size=7, patch_distance=11, h=0.1, sigma=0.0):
    """skimage.restoration.denoise_nl_means(volume, h=h) for a 3-D grayscale volume (multichannel=False, fast mode),
    as the z-stack caller uses it: bio/hiprfish_imaging_biofilm_analysis.py:454 (h = 0.03).

    PARITY UNPINNED, twice over: scikit-image is neither vendored nor pinned by the reference and is not installed
    here; and its era matters -- scikit-image <= 0.14 treats a 3-D array with multichannel=None as a 2-D image with
    Z channels (deprecation warning), 0.15+ as a volume.  This restates the published algorithm of
    skimage/restoration/_nl_means_denoising.pyx::_fast_nl_means_denoising_3d (the volume reading), loop for loop:
      * reflect padding by offset + d + 1;
      * for every shift (t_pln, t_row in [-d, d], t_col in [0, d]): 3-D integral image of (padded - shifted)^2
        - 2 sigma^2, patch distance by inclusion-exclusion over its eight corners at +-offset (a 2*offset cube),
        clipped at 0 and divided by h^2 * patch_size^3;
      * weight = alpha * exp(-distance) unless distance > 5, alpha = 0.5 on the t_col = 0 plane except the zero
        shift; accumulated symmetrically into both voxels of the pair;
      * result / weights, cropped.
    Vectorised over voxels, one shift at a time ((2d + 1)^2 (d + 1) shifts: minutes for d = 11 on a 20^3 volume).
    Test infrastructure only."""
    image = np.asarray(image, dtype=np.float64)
    if image.ndim != 3:
        raise ValueError("3-D grayscale volumes only")
    s = int(patch_size)
    if s % 2 == 0:
        s += 1
    d = int(patch_distance)
    o = s // 2
    pad_size = o + d + 1
    padded = np.pad(image, pad_size, mode="reflect")
    n_pln, n_row, n_col = padded.shape
    result = np.zeros_like(padded)
    weights = np.zeros_like(padded)
    h2s3 = h * h * s * s * s
    var = 2.0 * sigma * sigma
    for t_pln in range(-d, d + 1):
        p0, p1 = max(o, o - t_pln), min(n_pln - o, n_pln - o - t_pln)
        pa, pb = max(1, -t_pln), min(n_pln, n_pln - t_pln)
        for t_row in range(-d, d + 1):
            r0, r1 = max(o, o - t_row), min(n_row - o, n_row - o - t_row)
            ra, rb = max(1, -t_row), min(n_row, n_row - t_row)
            for t_col in range(0, d + 1):
                alpha = 0.5 if (t_col == 0 and (t_pln != 0 or t_row != 0)) else 1.0
                c0, c1 = o, n_col - o - t_col
                ca, cb = 1, n_col - t_col
                integral = np.zeros_like(padded)
                diff = (padded[pa:pb, ra:rb, ca:cb] - padded[pa + t_pln:pb + t_pln, ra + t_row:rb + t_row, ca + t_col:cb + t_col]) ** 2 - var
                integral[pa:pb, ra:rb, ca:cb] = np.cumsum(np.cumsum(np.cumsum(diff, axis=0), axis=1), axis=2)

                def I(dp, dr, dc):
                    return integral[p0 + dp:p1 + dp, r0 + dr:r1 + dr, c0 + dc:c1 + dc]
                dist = (I(o, o, o) - I(-o, o, o) - I(o, -o, o) - I(o, o, -o)
                        + I(-o, -o, o) + I(-o, o, -o) + I(o, -o, -o) - I(-o, -o, -o))
                dist = np.maximum(dist, 0.0) / h2s3
                w = np.where(dist > NLM_DISTANCE_CUTOFF, 0.0, alpha * np.exp(-dist))
                A = (slice(p0, p1), slice(r0, r1), slice(c0, c1))
                B = (slice(p0 + t_pln, p1 + t_pln), slice(r0 + t_row, r1 + t_row), slice(c0 + t_col, c1 + t_col))
                weights[A] += w
                weights[B] += w
                result[A] += w * padded[B]
                result[B] += w * padded[A]
    c = slice(pad_size, -pad_size)
    return result[c, c, c] / weights[c, c, c]


def denoise_nl_means_3d_direct(image, patch_size=7, patch_distance=11, h=0.1):
    """The same estimator voxel by voxel (no integral images, no symmetric accumulation): for every voxel p and every
    shift t in [-d, d]^3, weight = exp(-max(sum over the 2*offset cube p - offset + 1 .. p + offset of
    (v[u] - v[u + t])^2, 0) / (h^2 s^3)) if that distance is <= 5, the zero shift counted twice.  This is the form the
    CUDA kernel evaluates; used to check the restatement above against an independent formulation."""
    image = np.asarray(image, dtype=np.float64)
    s = int(patch_size) | 1
    d = int(patch_distance)
    o = s // 2
    pad = o + d + 1
    v = np.pad(image, pad, mode="reflect")
    X, Y, Z = image.shape
    h2s3 = h * h * s * s * s
    acc_w = np.zeros((X, Y, Z))
    acc_v = np.zeros((X, Y, Z))
    lo, n = -o + 1, 2 * o
    a = v[pad + lo: pad + X + o, pad + lo: pad + Y + o, pad + lo: pad + Z + o]
    for tx in range(-d, d + 1):
        for ty in range(-d, d + 1):
            for tz in range(-d, d + 1):
                b = v[pad + lo + tx: pad + X + o + tx, pad + lo + ty: pad + Y + o + ty, pad + lo + tz: pad + Z + o + tz]
                D = (a - b) ** 2
                box = np.zeros((X, Y, Z))
                for i in range(n):
                    for j in range(n):
                        for k in range(n):
                            box += D[i:i + X, j:j + Y, k:k + Z]
                dist = np.maximum(box, 0.0) / h2s3
                w = np.where(dist > NLM_DISTANCE_CUTOFF, 0.0, np.exp(-dist))
                if tx == 0 and ty == 0 and tz == 0:
                    w = 2.0 * w
                acc_w += w
                acc_v += w * v[pad + tx: pad + tx + X, pad + ty: pad + ty + Y, pad + tz: pad + tz + Z]
    return acc_v / acc_w


def _mean_quartiles(rnc, axis):
    m = np.average(rnc, axis=axis)
    with np.errstate(invalid="ignore"):
        lq = np.percentile(rnc, 25, axis=axis)
        uq = np.percentile(rnc, 75, axis=axis)
    return m, lq, uq


def epilogue_F1(lp):
    """syn/...measurement.py:111-124 (= bio/...:353-366, 595-608).  lp (..., R, P) -> (...)."""
    with np.errstate(invalid="ignore", divide="ignore"):
        lp = np.nan_to_num(lp)
        mn = np.min(lp, axis=-1)
        mx = np.max(lp, axis=-1) - mn
        rel = (lp - mn[..., None]) / mx[..., None]
        rnc = rel[..., int((lp.shape[-1] - 1) / 2)]
        m, lq, uq = _mean_quartiles(rnc, rnc.ndim - 1)
        qcv = np.zeros(uq.shape)
        pre = (uq - lq) / (uq + lq + 1e-8)
        qcv[uq > 0] = pre[uq > 0]
        return m * (1 - qcv)


def epilogue_F2(lp):
    """bio/...:905-917 (and :671-683, 728-740, 995-1007 in 2-D): nan_to_num on qcv, no epsilon."""
    with np.errstate(invalid="ignore", divide="ignore"):
        lp = np.nan_to_num(lp)
        mn = np.min(lp, axis=-1)
        mx = np.max(lp, axis=-1) - mn
        rel = (lp - mn[..., None]) / mx[..., None]
        rnc = rel[..., int((lp.shape[-1] - 1) / 2)]
        return epilogue_F2_dirs(rnc)


def epilogue_F2_dirs(rnc):
    """bio/...:457-462 and :812-817: the F2 reduction applied to the me_v2 output (..., T)."""
    with np.errstate(invalid="ignore", divide="ignore"):
        m, lq, uq = _mean_quartiles(rnc, rnc.ndim - 1)
        qcv = np.nan_to_num((uq - lq) / (uq + lq))
        return m * (1 - qcv)


def epilogue_F3(lp):
    """bio/...:1114-1125: +1e-8 on the line range and on uq+lq, no nan_to_num."""
    with np.errstate(invalid="ignore", divide="ignore"):
        mn = np.min(lp, axis=-1)
        mx = np.max(lp, axis=-1) - mn
        rel = (lp - mn[..., None]) / (mx[..., None] + 1e-8)
        rnc = rel[..., int((lp.shape[-1] - 1) / 2)]
        m, lq, uq = _mean_quartiles(rnc, rnc.ndim - 1)
        qcv = (uq - lq) / (uq + lq + 1e-8)
        return m * (1 - qcv)


EPILOGUES = {"F1": epilogue_F1, "F2": epilogue_F2, "F3": epilogue_F3}


def lne2d(image, flavour="F1", patch_size=11, phi_range=9, lp_func=None):
    """pad(5,'edge') -> line_profile_2d_v2 -> epilogue; image is the (normalised) sum image."""
    half = int((patch_size - 1) / 2)
    padded = np.pad(np.asarray(image, dtype=np.float64), half, mode="edge")
    lp = (lp_func or line_profile_2d_v2)(padded, patch_size, phi_range)
    return EPILOGUES[flavour](lp)


def lne3d(volume, flavour="F2", patch_size=11, theta_range=9, phi_range=9, lp_func=None, me_func=None):
    """3-D score map.  'F2'/'F3': line_profile_v2 + epilogue (bio/...:904-917, 1112-1125);
    'ME2': line_profile_memory_efficient_v2 + F2 reduction (bio/...:811-817)."""
    half = int((patch_size - 1) / 2)
    padded = np.pad(np.asarray(volume, dtype=np.float64), half, mode="edge")
    if flavour == "ME2":
        e = (me_func or line_profile_memory_efficient_v2)(padded, patch_size, theta_range, phi_range)
        return epilogue_F2_dirs(e)
    lp = (lp_func or line_profile_v2)(padded, patch_size, theta_range, phi_range)
    return EPILOGUES[flavour](lp)


# --------------------------------------------------------------------------------------------
# Per-cell mean spectra
# --------------------------------------------------------------------------------------------

def cell_spectra(seg, img):
    """syn/...measurement.py:167-172 (= eco/...:151-157, ref/...:177-183, bio/...:1214-1220).

    skimage.measure.regionprops(seg, intensity_image=img[..., k]).mean_intensity for every
    channel: the float64 arithmetic mean of img over the pixels of each label, regions in
    ascending order of the labels present, label 0 (background) and negative labels ignored.
    Returns (labels int64 (n,), area int64 (n,), avgint float64 (n, C), avgint_norm (n, C)).
    """
    seg = np.asarray(seg)
    img = np.asarray(img)
    C = img.shape[-1]
    flat = seg.reshape(-1).astype(np.int64)
    vals = img.reshape(-1, C).astype(np.float64)
    keep = flat > 0
    flat, vals = flat[keep], vals[keep]
    if flat.size == 0:
        z = np.zeros((0, C))
        return np.zeros(0, np.int64), np.zeros(0, np.int64), z, z.copy()
    area_all = np.bincount(flat)
    labels = np.nonzero(area_all)[0]
    area = area_all[labels]
    avg = np.empty((labels.size, C), dtype=np.float64)
    for k in range(C):
        avg[:, k] = np.bincount(flat, weights=vals[:, k], minlength=area_all.size)[labels] / area
    with np.errstate(invalid="ignore", divide="ignore"):
        norm = avg / np.max(avg, axis=1)[:, None]
    return labels.astype(np.int64), area.astype(np.int64), avg, norm


# --------------------------------------------------------------------------------------------
# Whole 2-D path, as the reference runs it (used by bench.py's CPU legs)
# --------------------------------------------------------------------------------------------

def neighbor2d_score(cube, flavour="F1", calibration=None, lp_func=None):
    """cube (H,W,C) -> image_final (H,W): prologue (no NLM) + stencil + epilogue."""
    _, padded = prologue(cube, calibration=calibration)
    lp = (lp_func or line_profile_2d_v2)(padded, 11, 9)
    return EPILOGUES[flavour](lp)


def cell_geometry(seg):
    """regionprops(seg) geometry (test infrastructure): for every label present, ascending: label, area,
    and [centroid_row, centroid_col, major_axis_length, minor_axis_length, eccentricity, orientation, mu20,
    mu02, mu11], following scikit-image's _regionprops.py: centroid = mean of the pixel coordinates; inertia
    tensor [[mu02, -mu11], [-mu11, mu20]] / area from the central moments; its eigenvalues l1 >= l2 (clipped at
    0) give 4 sqrt(l1), 4 sqrt(l2), sqrt(1 - l2 / l1); orientation in the 'rc' convention of scikit-image >= 0.16.
    PARITY UNPINNED for orientation (the reference's scikit-image version is not pinned and the convention
    changed in 0.16); the other properties are version independent.  Consumers:
    syn/hiprfish_imaging_classify_spectra.py:38-46, bio/hiprfish_imaging_biofilm_analysis.py:1232-1240."""
    seg = np.asarray(seg)
    labs = np.unique(seg[seg > 0])
    geom = np.zeros((labs.size, 9))
    area = np.zeros(labs.size, dtype=np.int64)
    for i, L in enumerate(labs):
        rc = np.argwhere(seg == L).astype(np.float64)
        area[i] = rc.shape[0]
        cen = rc.mean(axis=0)
        d = rc - cen
        mu20, mu02, mu11 = (d[:, 0] ** 2).sum(), (d[:, 1] ** 2).sum(), (d[:, 0] * d[:, 1]).sum()
        T = np.array([[mu02, -mu11], [-mu11, mu20]]) / area[i]
        ev = np.clip(np.sort(np.linalg.eigvalsh(T))[::-1], 0, None)
        l1, l2 = ev
        a, b, c = T[0, 0], T[0, 1], T[1, 1]
        if a - c == 0:
            orient = -np.pi / 4 if b < 0 else np.pi / 4
        else:
            orient = 0.5 * np.arctan2(-2 * b, c - a)
        geom[i] = [cen[0], cen[1], 4 * np.sqrt(l1), 4 * np.sqrt(l2), 0.0 if l1 == 0 else np.sqrt(1 - l2 / l1), orient,
                   mu20, mu02, mu11]
    return labs.astype(np.int64), area, geom


def paint_labels(seg, values):
    """image[seg == label] = values[label] for every label (eco/hiprfish_imaging_image_classification.py:64-70,
    bio/hiprfish_imaging_biofilm_analysis.py:1247-1257), values[0] = background."""
    seg = np.asarray(seg)
    values = np.asarray(values)
    out = np.empty(seg.shape + values.shape[1:], dtype=values.dtype)
    out[...] = values[0]
    for L in np.unique(seg[seg > 0]):
        out[seg == L] = values[L]
    return out


# --------------------------------------------------------------------------------------------
# 1-D k-means thresholding (SURVEY.md 8f rank 3)
# --------------------------------------------------------------------------------------------

def _kmeans_samples(image, transform=None, eps=0.0, positive_only=False):
    img = np.asarray(image, dtype=np.float64)
    valid = (img > 0) if positive_only else np.ones(img.shape, dtype=bool)
    x = img[valid]
    if transform == "log10":
        x = np.log10(x + eps)
    elif transform == "log":
        x = np.log(x + eps)
    return img, valid, x


def _kmeans_finish(img, valid, labels_valid, k, fill_label=0):
    """Full-size label image, and the scripts' orientation: the cluster with the largest mean of its positive image
    values is the foreground (syn/..._measurement.py:126-135: `image0 = image_final*(seg == 0)`,
    `i0 = np.average(image0[image0 > 0])`, `if i0 < i1: mask = seg == 1`; np.argmax([i0, i1, i2]) at bio/...:471)."""
    labels = np.full(img.shape, fill_label, dtype=np.int32)
    labels[valid] = labels_valid
    pm = np.full(k, -np.inf)
    for j in range(k):
        sel = valid & (labels == j) & (img > 0)
        if sel.any():
            pm[j] = img[sel].mean()
    bright = int(np.argmax(pm))
    return labels, valid & (labels == bright), pm, bright


def kmeans1d_sklearn(image, n_clusters=2, random_state=0, n_init=1, transform=None, eps=0.0, positive_only=False,
                     max_iter=300, tol=1e-4):
    """THE pinned oracle of this row: scikit-learn itself (1.9.0 in this image), called as the scripts call it:
    KMeans(n_clusters = k, random_state = 0).fit_predict(x.reshape(-1, 1))  (syn/..._measurement.py:125, 141;
    bio/..._analysis.py:367, 384, 463, 819, 830; eco/..._measurement.py:73, 85).  n_init=1 is scikit-learn >= 1.4's
    'auto' for k-means++; the reference's era used 10.
    Returns (cluster_centers_ (k,), labels (image shape, int32), foreground mask, n_iter, inertia)."""
    from sklearn.cluster import KMeans
    img, valid, x = _kmeans_samples(image, transform, eps, positive_only)
    km = KMeans(n_clusters=n_clusters, random_state=random_state, n_init=n_init, max_iter=max_iter,
                tol=tol).fit(x.reshape(-1, 1))
    labels, mask, _, _ = _kmeans_finish(img, valid, km.labels_, n_clusters)
    return km.cluster_centers_.ravel().copy(), labels, mask, int(km.n_iter_), float(km.inertia_)


def kmeans1d(image, n_clusters=2, random_state=0, n_init=1, transform=None, eps=0.0, positive_only=False, max_iter=300,
             tol=1e-4):
    """numpy restatement of what scikit-learn 1.9.0's KMeans does on one feature (sklearn/cluster/_kmeans.py:
    fit -> _kmeans_plusplus -> _kmeans_single_lloyd), checked label for label against kmeans1d_sklearn in
    tests/test_kmeans.py and tests/test_kmeans_sweep.py.  It documents exactly what the CUDA kernel reproduces:
      * X is centred by its mean; tol_abs = tol * var(X);
      * seeding: first seed = sample floor(u0 * n) (RandomState.choice with uniform p); every further seed: `trials`
        = 2 + int(log(k)) candidates at searchsorted(cumsum(closest_dist_sq), u * current_pot), keep the one with the
        smallest new potential (a target of 0, once the seeds cover every distinct value, picks the first sample);
      * Lloyd: label = argmin_j(c_j^2 - 2 x c_j) (first minimum), centres = cluster means; stop when the labels did not
        change (in 1-D: the cluster sizes) or sum((c_new - c_old)^2) <= tol_abs; labels are then those of the final centres;
      * a Lloyd step that leaves a cluster empty raises RuntimeError (scikit-learn relocates the cluster and warns
        that fewer distinct clusters than n_clusters were found; neither is reproduced);
      * best of n_init by inertia (first wins ties), and only when the clustering differs from the best so far: in 1-D
        a clustering is identified by its cluster sizes in centre order (scikit-learn's _is_same_clustering).
    Returns like kmeans1d_sklearn."""
    img, valid, x = _kmeans_samples(image, transform, eps, positive_only)
    k, n = int(n_clusters), x.size
    trials = 2 + int(np.log(k))
    u = np.random.RandomState(random_state).random_sample(n_init * (1 + trials * (k - 1)))
    mean = x.mean()
    xc = x - mean
    tol_abs = np.var(x) * tol
    best, ui = None, 0
    for _ in range(n_init):
        cid = min(int(np.floor(u[ui] * n)), n - 1)
        ui += 1
        centers = [xc[cid]]
        closest = (xc - centers[0]) ** 2
        pot = closest.sum()
        for _c in range(1, k):
            r = u[ui:ui + trials] * pot
            ui += trials
            cand = np.clip(np.searchsorted(np.cumsum(closest), r), None, n - 1)
            d = np.minimum(closest[None, :], (xc[None, :] - xc[cand][:, None]) ** 2)
            pots = d.sum(axis=1)
            b = int(np.argmin(pots))
            pot, closest = pots[b], d[b]
            centers.append(xc[cand[b]])
        centers = np.array(centers)
        counts_old = None
        for it in range(max_iter):
            lab = np.argmin(centers[None, :] ** 2 - 2 * xc[:, None] * centers[None, :], axis=1)
            counts = np.bincount(lab, minlength=k)
            if not counts.all():
                raise RuntimeError("a cluster ran empty during Lloyd iterations (scikit-learn would relocate it; not reproduced)")
            new = np.bincount(lab, weights=xc, minlength=k) / counts
            shift = ((new - centers) ** 2).sum()
            centers = new
            if counts_old is not None and np.array_equal(counts, counts_old):
                break
            if shift <= tol_abs:
                break
            counts_old = counts
        lab = np.argmin(centers[None, :] ** 2 - 2 * xc[:, None] * centers[None, :], axis=1)
        inertia = float(((xc - centers[lab]) ** 2).sum())
        sizes = np.bincount(lab, minlength=k)[np.argsort(centers)]
        if best is None or (inertia < best[0] and not np.array_equal(sizes, best[4])):
            best = (inertia, centers + mean, lab, it + 1, sizes)
    labels, mask, _, _ = _kmeans_finish(img, valid, best[2], k)
    return best[1], labels, mask, best[3], best[0]
