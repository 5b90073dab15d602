"""numpy restatement of the registration-shift step the scripts take from scikit-image (syn/..._measurement.py:83-85):
register_translation and the per-excitation excitation_shifts built on it.  The checker of csrc/xcorr2d.cu (K9) in
tests/test_shifts.py, tests/test_gpu_shifts.py and tools/time_shifts.py; never imported by the product.  TEST
INFRASTRUCTURE ONLY."""
import numpy as np


def register_translation(src_image, target_image, return_correlation=False):
    """skimage.feature.register_translation(src_image, target_image)[0] with the defaults the scripts use
    (upsample_factor=1, space="real"): syn/hiprfish_imaging_multispecies_spectral_image_measurement.py:83-85.

    PARITY UNPINNED: scikit-image is a third-party dependency that the reference neither vendors nor pins
    (era 0.14-0.15) and it is not installed here.  This restates
    skimage/feature/register_translation.py::register_translation up to its integer shift (the lines before
    `if upsample_factor > 1`): float64 FFTs, the cross-power spectrum src_freq * target_freq.conj(), the argmax
    of its inverse's magnitude (numpy's: a NaN beats any number, ties go to the lowest flat index), midpoints
    np.fix(n / 2), shifts above the midpoint minus the axis length, and 0 on axes of length 1.  The error and
    phasediff outputs are not restated.  With return_correlation also returns |cc|.  Test infrastructure only."""
    src = np.asarray(src_image, dtype=np.float64)
    target = np.asarray(target_image, dtype=np.float64)
    if src.shape != target.shape:
        raise ValueError("Error: images must be same size for register_translation")
    shape = src.shape
    cc = np.fft.ifftn(np.fft.fftn(src) * np.fft.fftn(target).conj())
    acc = np.abs(cc)
    maxima = np.unravel_index(np.argmax(acc), shape)
    midpoints = np.array([np.fix(axis_size / 2) for axis_size in shape])
    shifts = np.array(maxima, dtype=np.float64)
    shifts[shifts > midpoints] -= np.array(shape)[shifts > midpoints]
    shifts[np.array(shape) == 1] = 0
    return (shifts, acc) if return_correlation else shifts


def excitation_shifts(image_stack, transform="log", eps=0.0):
    """The shift vectors the scripts hand the registration paste, syn/..._measurement.py:83-85: per excitation
    stack the channel sum (taken in float64, as register_stacks' sums), T(sum) = log(sum + eps) (transform="log";
    the reading of the scripts this project assumes, not confirmed against them) or the sum itself (None), then
    (0, 0) for the first stack and register_translation(T(sum_0), T(sum_e)) for the others.

    PARITY UNPINNED, as register_translation.  Returns (n, 2) float64.  Test infrastructure only."""
    if transform not in (None, "log"):
        raise ValueError("transform must be None or 'log'")
    sums = [np.sum(np.asarray(s, dtype=np.float64), axis=2) for s in image_stack]
    with np.errstate(divide="ignore", invalid="ignore"):
        images = [np.log(s + eps) if transform == "log" else s for s in sums]
        out = np.zeros((len(images), 2))
        for e in range(1, len(images)):
            out[e] = register_translation(images[0], images[e])
    return out
