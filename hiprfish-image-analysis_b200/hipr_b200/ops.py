"""Device-resident operators: torch CUDA tensors in, torch CUDA tensors out, stream-ordered on
torch's current stream.  torch is used for device memory and streams only; every kernel that
runs here is one of libhipr_b200's.  No CPU fallback: CPU tensors are rejected.

Reference blocks replaced (paths relative to the reference repository):
  register_stacks   syn/hiprfish_imaging_multispecies_spectral_image_measurement.py:86-105
  excitation_shifts syn/hiprfish_imaging_multispecies_spectral_image_measurement.py:83-85 (register_translation)
  channel_sum       syn/hiprfish_imaging_multispecies_spectral_image_measurement.py:105-106
  lne2d             eco/neighbor2d.pyx:56-63 + syn/...measurement.py:109-124 (F1), bio F2 / F3
  neighbor2d_score  syn/...measurement.py:105-124 without the skimage denoise
  line_profile_2d   eco/neighbor2d.pyx:8-64
  line_profile_3d   bio/neighbor.pyx:115-181
  lne3d_dirs        bio/neighbor.pyx:186-263
  lne3d             bio/neighbor.pyx + bio/hiprfish_imaging_biofilm_analysis.py:812-817, 905-917, 1114-1125
  cell_spectra      syn/...measurement.py:167-172
  label, remove_small_objects, binary_fill_holes, clear_border, relabel_sequential, watershed,
  binary_erosion, binary_dilation, binary_opening, binary_closing
                    the segmentation back end, syn/...measurement.py:125-158, eco/...measurement.py:44-127,
                    bio/...analysis.py:367-419, 463-501
"""
import ctypes as C

import numpy as np
import torch

from . import tables
from ._lib import F32, F64, FLAVOURS, I32, I64, U8, HiprError, check, lib

# the ABI's dtype code of each torch dtype an entry point may take (bool is stored as one byte, like uint8)
_ABI = {torch.float32: F32, torch.float64: F64, torch.int32: I32, torch.int64: I64, torch.uint8: U8, torch.bool: U8}
_LABEL_DTYPES = (torch.bool, torch.uint8, torch.int32, torch.int64)
UNSUPPORTED = -9
HIPR_E_RANGE = -7


def _stream():
    return torch.cuda.current_stream().cuda_stream


_PLAIN = {int, float, bool, type(None)}


def _arg(a):
    """One argument of a libhipr_b200 call: tensors and numpy arrays by their data pointer, a MaxKey by its keys, a
    list or tuple of them as an array of pointers; anything else (numbers, None, C.byref(...)) as it is."""
    # isinstance(a, torch.Tensor) is slow when false: it comes last, after the exact type and the other classes
    if type(a) is torch.Tensor:
        return a.data_ptr()
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if isinstance(a, MaxKey):
        return a.key.data_ptr()
    if isinstance(a, (list, tuple)):
        return (C.c_void_p * len(a))(*[_arg(x) for x in a])
    if isinstance(a, torch.Tensor):
        return a.data_ptr()
    return a


def _call(name, *args, what=None, ok=()):
    """lib().hipr_<name>(*args), its return code checked under the prefix `what` (default: name); the codes in `ok`
    are returned instead of raised."""
    # numbers and None, most of the arguments, pass without a call of _arg
    code = getattr(lib(), "hipr_" + name)(*[a if type(a) in _PLAIN else _arg(a) for a in args])
    if code not in ok:
        check(code, what or name)
    return code


def _launch(name, device, *args, what=None, ok=()):
    """_call of a device entry point on `device`, stream-ordered on torch's current stream."""
    with torch.cuda.device(device):
        return _call(name, *args, _stream(), what=what, ok=ok)


def _workspace(name, device, *size_args, what=None, errors=None):
    """The uint8 device workspace hipr_<name>(*size_args) asks for.  A negative answer raises ValueError(errors[code])
    where the caller names the code, and goes through check (prefix `what`, default: name) otherwise."""
    need = int(getattr(lib(), "hipr_" + name)(*size_args))
    if need < 0:
        if errors and need in errors:
            raise ValueError(errors[need])
        check(need, what or name)
    return torch.empty(need, dtype=torch.uint8, device=device)


def _dev(t, name, dtypes=(torch.float32, torch.float64)):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor on a CUDA device" % name)
    if not t.is_cuda:
        raise ValueError("%s must live on a CUDA device (there is no CPU path)" % name)
    if t.dtype not in dtypes:
        raise TypeError("%s: unsupported dtype %s" % (name, t.dtype))
    return t.contiguous()


def _dims(t, name):
    """(ndim, d0, d1, d2) of a 2-D image or a 3-D volume (d2 = 1 for an image), as the segmentation entry points take
    it; ValueError for another rank or an empty tensor."""
    if t.dim() not in (2, 3):
        raise ValueError("%s must be a 2-D image or a 3-D volume, got shape %s" % (name, tuple(t.shape)))
    if t.numel() == 0:
        raise ValueError("%s is empty" % name)
    return (t.dim(),) + tuple(t.shape) + (1,) * (3 - t.dim())


def _same(a, b, names):
    """ValueError unless tensor a (called names[0]) has the shape and device of b (names[1])."""
    if a.shape != b.shape:
        raise ValueError("%s %s and %s %s differ in shape" % (names[0], tuple(a.shape), names[1], tuple(b.shape)))
    if a.device != b.device:
        raise ValueError("%s and %s are on different devices" % (names[1], names[0]))


def _out_dims(shape, P, padded, what):
    """Output shape of a stencil with P-sample lines: the input's shape, or with padded=True the shape of the image
    inside its (P - 1) / 2 border.  ValueError when that is empty."""
    dims = tuple(d - P + 1 for d in shape) if padded else tuple(shape)
    if min(dims) < 1:
        raise ValueError("%s smaller than the patch" % what)
    return dims


_CUBE_AXES = {3: "(H, W, C)", 4: "(X, Y, Z, C)"}


def _host_cube(a, ndim=None, dtypes=(np.float32,), name="cube"):
    """A numpy entry point's input as a C-contiguous array: TypeError for another dtype, ValueError (ndim given) for
    another rank."""
    a = np.ascontiguousarray(a)
    if a.dtype not in dtypes:
        raise TypeError("%s must be %s, got %s" % (name, " or ".join(np.dtype(d).name for d in dtypes), a.dtype))
    if ndim is not None and a.ndim != ndim:
        raise ValueError("cube must be %s" % _CUBE_AXES[ndim])
    return a


def _flavour(f):
    try:
        return FLAVOURS[f]
    except KeyError:
        raise ValueError("unknown flavour %r (one of %s)" % (f, sorted(FLAVOURS)))


class MaxKey:
    """Two device scalars: max and min of an image as order-preserving keys (see hipr_b200.h)."""

    def __init__(self, device):
        # filled (and reset) by hipr_chansum / hipr_image_range; no torch kernel on the hot path
        self.key = torch.empty(2, dtype=torch.int64, device=device)

    def value(self):
        out = torch.empty(1, dtype=torch.float64, device=self.key.device)
        _launch("maxkey_decode", self.key.device, self, out)
        return out

    def values(self):
        """(max, min) as 1-element float64 device tensors."""
        out = torch.empty(2, dtype=torch.float64, device=self.key.device)
        _launch("range_decode", self.key.device, self, out)
        return out[0:1], out[1:2]

    @classmethod
    def from_values(cls, vmax, vmin):
        mm = torch.cat([vmax.reshape(1), vmin.reshape(1)]).to(torch.float64).contiguous()
        mk = cls(mm.device)
        _launch("range_encode", mm.device, mm, mk)
        return mk


def channel_sum(cube, calibration=None, normalize=True, dtype=torch.float32, return_max=False):
    """cube (..., C) float32 -> (...) sum over the last axis, divided by its global max when
    `normalize` (image_registered_sum / np.max(...)).  Accumulation is float64."""
    cube = _dev(cube, "cube", (torch.float32,))
    if cube.dim() < 2:
        raise ValueError("cube must have at least 2 dimensions (..., C)")
    Cn = cube.shape[-1]
    npix = cube.numel() // Cn
    if calibration is not None:
        calibration = _dev(calibration, "calibration", (torch.float32,))
        if calibration.shape != cube.shape:
            calibration = calibration.expand_as(cube).contiguous()
    out = torch.empty(cube.shape[:-1], dtype=dtype, device=cube.device)
    mk = MaxKey(cube.device) if (normalize or return_max) else None
    _launch("chansum", cube.device, cube, calibration, npix, Cn, out, _ABI[dtype], mk, what="channel_sum")
    if normalize:
        _launch("normalize", cube.device, out, _ABI[dtype], npix, mk)
    return (out, mk) if return_max else out


def channel_sum_raw(cube, scale, return_max=False):
    """cube (..., C) of raw detector counts (torch.uint8 / uint16 / int16 bit pattern of uint16) -> float64
    channel sums of float32(count) / float32(scale), the values bioformats' rescale hands the scripts."""
    if not isinstance(cube, torch.Tensor) or not cube.is_cuda:
        raise ValueError("cube must be a CUDA tensor (there is no CPU path)")
    if cube.dtype not in (torch.uint8, torch.uint16, torch.int16):
        raise TypeError("raw cube must be uint8 or uint16, got %s" % cube.dtype)
    cube = cube.contiguous()
    Cn = cube.shape[-1]
    npix = cube.numel() // Cn
    out = torch.empty(cube.shape[:-1], dtype=torch.float64, device=cube.device)
    mk = MaxKey(cube.device)
    _launch("chansum_raw", cube.device, cube, cube.element_size(), float(scale), npix, Cn, out, mk,
            what="channel_sum_raw")
    return (out, mk) if return_max else out


def register_stacks(stacks, shifts=None, calibration=None, return_cube=True):
    """Registration paste + np.dstack + flat-field divide + channel sum in one pass (csrc/register.cu).

    stacks: list of (H, W, c_e) float32 CUDA tensors, one per excitation; shifts: per stack (row, col)
    integer shifts as the scripts derive them from register_translation (int(shift_vector)), None = no
    shift, "estimate" = excitation_shifts(stacks) first (one synchronisation); calibration: None or a
    (H, W, C) float32 divisor.  Returns (cube (H, W, C) float32 or None, channel sums (H, W) float64, MaxKey)."""
    stacks = [_dev(s, "stack %d" % i, (torch.float32,)) for i, s in enumerate(stacks)]
    if not stacks:
        raise ValueError("need at least one excitation stack")
    H, W = stacks[0].shape[:2]
    for s in stacks:
        if s.dim() != 3 or tuple(s.shape[:2]) != (H, W):
            raise ValueError("every stack must be (H, W, c_e) with the same H, W")
    n = len(stacks)
    if shifts is None:
        shifts = [(0, 0)] * n
    elif isinstance(shifts, str):
        if shifts != "estimate":
            raise ValueError("shifts must be None, 'estimate' or one (row, col) per stack")
        shifts = excitation_shifts(stacks)
    if len(shifts) != n:
        raise ValueError("one (row, col) shift per stack")
    chans = np.asarray([s.shape[2] for s in stacks], dtype=np.int32)
    srow = np.asarray([int(v[0]) for v in shifts], dtype=np.int32)     # int(): truncation, as the scripts do
    scol = np.asarray([int(v[1]) for v in shifts], dtype=np.int32)
    Cn = int(chans.sum())
    dev = stacks[0].device
    if calibration is not None:
        calibration = _dev(calibration, "calibration", (torch.float32,))
        if tuple(calibration.shape) != (H, W, Cn):
            calibration = calibration.expand(H, W, Cn).contiguous()
    cube = torch.empty((H, W, Cn), dtype=torch.float32, device=dev) if return_cube else None
    s64 = torch.empty((H, W), dtype=torch.float64, device=dev)
    mk = MaxKey(dev)
    _launch("register_stacks", dev, stacks, chans, srow, scol, n, H, W, calibration, cube, s64, mk)
    return cube, s64, mk


def neighbor2d_score_from_stacks(stacks, shifts=None, calibration=None, flavour="F1", return_cube=True):
    """syn/..._measurement.py:86-124 without the skimage calls: excitation stacks -> registered cube,
    channel sums, score map (fixed-point stencil); shifts as register_stacks ("estimate": estimated from the
    stacks with excitation_shifts).  Returns (score, cube, sums, MaxKey)."""
    cube, s64, mk = register_stacks(stacks, shifts, calibration, return_cube)
    score = lne2d_fixed(s64, flavour, 11, 9, padded=False, range_keys=mk)
    return score, cube, s64, mk


def _xcorr_workspace(H, W, n, device):
    return _workspace("xcorr2d_workspace_bytes", device, int(H), int(W), int(n), errors={
        UNSUPPORTED: "image height and width must each be a power of two in [2, 8192], got (%d, %d)" % (H, W)})


def register_translation(src, target, return_correlation=False):
    """skimage.feature.register_translation(src, target)[0] (upsample_factor=1, space="real") on the device, as
    syn/...measurement.py:83-85 calls it: the peak of |ifftn(fftn(src) * conj(fftn(target)))| in float64 FFTs
    (csrc/xcorr2d.cu), numpy's argmax order, indices above n // 2 wrapped to negative shifts.
    src, target: (H, W) float32 / float64 CUDA tensors of the same shape and dtype, H and W powers of two in
    [2, 8192].  Returns the (row, col) shift as a numpy (2,) float64 array (synchronises once); with
    return_correlation also the (H, W) float64 |cc| tensor."""
    src = _dev(src, "src")
    target = _dev(target, "target")
    if src.dim() != 2 or src.shape != target.shape:
        raise ValueError("src and target must be 2-D images of the same shape")
    if src.dtype != target.dtype:
        raise TypeError("src and target must have the same dtype, got %s and %s" % (src.dtype, target.dtype))
    if src.device != target.device:
        raise ValueError("src and target must be on the same device")
    H, W = src.shape
    dev = src.device
    work = _xcorr_workspace(H, W, 2, dev)
    shift = torch.empty(2, dtype=torch.float64, device=dev)
    corr = torch.empty((H, W), dtype=torch.float64, device=dev) if return_correlation else None
    _launch("register_translation_2d", dev, src, target, _ABI[src.dtype], H, W, work, work.numel(), shift, corr,
            what="register_translation")
    out = shift.cpu().numpy()
    return (out, corr) if return_correlation else out


SHIFT_TRANSFORMS = {None: 0, "log": 1}


def excitation_shifts(stacks, transform="log", eps=0.0):
    """The scripts' registration shifts (syn/...measurement.py:83-85) on the device: per excitation stack the float64
    channel sum, transformed (transform="log": ln(sum + eps); None: the sum itself), then
    register_translation(T(sum_0), T(sum_e)) for every e >= 1; row 0 is (0, 0).  The default "log" is a reading of
    the scripts that has not been confirmed against them.  stacks: list of (H, W, c_e) float32 CUDA tensors (the
    register_stacks input), H and W powers of two in [2, 8192].  Returns a numpy (n, 2) float64 array (synchronises
    once)."""
    if transform not in SHIFT_TRANSFORMS:
        raise ValueError("transform must be None or 'log'")
    stacks = [_dev(s, "stack %d" % i, (torch.float32,)) for i, s in enumerate(stacks)]
    if not stacks:
        raise ValueError("need at least one excitation stack")
    H, W = stacks[0].shape[:2]
    for s in stacks:
        if s.dim() != 3 or tuple(s.shape[:2]) != (H, W) or s.device != stacks[0].device:
            raise ValueError("every stack must be (H, W, c_e) with the same H, W, on the same device")
    n = len(stacks)
    if n > 8:
        raise ValueError("at most 8 excitation stacks")
    dev = stacks[0].device
    work = _xcorr_workspace(H, W, n, dev)
    shifts = torch.empty((n, 2), dtype=torch.float64, device=dev)
    chans = np.asarray([s.shape[2] for s in stacks], dtype=np.int32)
    _launch("excitation_shifts", dev, stacks, chans, n, H, W, SHIFT_TRANSFORMS[transform], float(eps), work,
            work.numel(), shifts)
    return shifts.cpu().numpy()


def denoise_nl_means(image, patch_size=7, patch_distance=11, h=0.1):
    """skimage.restoration.denoise_nl_means(image, h=h) for a 2-D image (fast mode, sigma 0), as
    syn/...measurement.py:108 calls it on the normalised sum image, or for a 3-D volume as bio/...analysis.py:454
    calls it on a z-stack.  (H, W) / (X, Y, Z) float32 / float64 CUDA tensor -> same dtype.  csrc/nlm2d.cu,
    csrc/nlm3d.cu; patch_size 7, patch_distance <= 15."""
    image = _dev(image, "image")
    if image.dim() == 3:
        # a z-stack volume (bio/...analysis.py:454, h = 0.03): csrc/nlm3d.cu
        X, Y, Z = image.shape
        work = _workspace("denoise_nl_means_3d_workspace", image.device, X, Y, Z, int(patch_distance),
                          errors={-1: "patch_distance must be in [0, 15]"})
        out = torch.empty_like(image)
        _launch("denoise_nl_means_3d", image.device, image, X, Y, Z, _ABI[image.dtype], int(patch_size),
                int(patch_distance), float(h), out, work, work.numel())
        return out
    if image.dim() != 2:
        raise ValueError("image must be 2-D or 3-D, got %d-D" % image.dim())
    Hh, Ww = image.shape
    out = torch.empty_like(image)
    _launch("denoise_nl_means_2d", image.device, image, Hh, Ww, _ABI[image.dtype], int(patch_size), int(patch_distance),
            float(h), out, what="denoise_nl_means")
    return out


def lne2d(image, flavour="F1", patch_size=11, phi_range=9, padded=False, maxkey=None):
    """Score map ("local neighbourhood enhancement") of a 2-D image.

    image: (H, W) when padded=False (border samples clamp to the edge, = np.pad(mode='edge')),
    or the already padded (H+P-1, W+P-1) image when padded=True.  maxkey: optional MaxKey from
    channel_sum(normalize=False, return_max=True); samples are divided by the max on load."""
    image = _dev(image, "image")
    if image.dim() != 2:
        raise ValueError("image must be 2-D, got %d-D" % image.dim())
    tab = tables.line_table_2d(patch_size, phi_range)
    P = tab.shape[1]
    Hs, Ws = image.shape
    out = torch.empty(_out_dims(image.shape, P, padded, "image"), dtype=image.dtype, device=image.device)
    _launch("lne2d", image.device, image, Hs, Ws, Ws, int(bool(padded)), _ABI[image.dtype], P, tab.shape[0], tab,
            _flavour(flavour), maxkey, out)
    return out


def image_range(image):
    """MaxKey (max and min keys) of any float image, for lne2d_fixed."""
    image = _dev(image, "image")
    mk = MaxKey(image.device)
    _launch("image_range", image.device, image, _ABI[image.dtype], image.numel(), mk)
    return mk


def lne2d_fixed(image, flavour="F1", patch_size=11, phi_range=9, padded=False, range_keys=None):
    """lne2d on a 31-bit fixed-point copy of the image (csrc/lne2d_q.cu): min, max and differences
    along each line are exact, so a float64 image keeps its precision at float32 speed.  The
    implied normalisation is image / max(image).  (11, 9) only; float32 score out."""
    image = _dev(image, "image")
    if image.dim() != 2:
        raise ValueError("image must be 2-D, got %d-D" % image.dim())
    tab = tables.line_table_2d(patch_size, phi_range)
    if tab.shape[:2] != (9, 11):
        raise ValueError("the fixed-point stencil exists for patch_size=11, phi_range=9 only; use lne2d")
    if range_keys is None and _flavour(flavour) not in (1, 2):
        range_keys = image_range(image)      # F3 scales its epsilon by the global range
    # F1 / F2 with no keys: every 32x32 tile is quantised with its own min / max (finest resolution)
    Hs, Ws = image.shape
    out = torch.empty(_out_dims(image.shape, 11, padded, "image"), dtype=torch.float32, device=image.device)
    _launch("lne2d_q", image.device, image, Hs, Ws, Ws, int(bool(padded)), _ABI[image.dtype], 11, 9, tab,
            _flavour(flavour), range_keys, out, what="lne2d_fixed")
    return out


_SIDE = {}


def _side_streams(device, n=2):
    key = (device.index if device.index is not None else torch.cuda.current_device(), n)
    if key not in _SIDE:
        _SIDE[key] = [torch.cuda.Stream(device=device) for _ in range(n)]
    return _SIDE[key]


def _over_side_streams(batch, fn):
    """fn(item) for each item of a batch, alternating between two side streams (so that one item's HBM-bound channel
    sum runs beside the previous item's stencil) and joined on the caller's stream; -> the results stacked (each
    part of a tuple result stacked on its own)."""
    cur = torch.cuda.current_stream(batch.device)
    side = _side_streams(batch.device)
    for st in side:
        st.wait_stream(cur)
    res = []
    for i, item in enumerate(batch):
        with torch.cuda.stream(side[i % len(side)]):
            res.append(fn(item))
    for st in side:
        cur.wait_stream(st)
    for r in res:
        for t in (r if isinstance(r, tuple) else (r,)):
            t.record_stream(cur)
    if res and isinstance(res[0], tuple):
        return tuple(torch.stack(part) for part in zip(*res))
    return torch.stack(res)


def neighbor2d_fused(cube, flavour="F1", patch_size=11, phi_range=9, return_sum=False):
    """cube (H, W, C) float32 -> float32 score in ONE launch (csrc/fused2d.cu).  Returns None when
    the request is outside the fused kernel's envelope (the caller then uses the two-kernel
    path).  With return_sum: (score, float64 channel sums, MaxKey)."""
    cube = _dev(cube, "cube", (torch.float32,))
    if cube.dim() != 3:
        raise ValueError("cube must be (H, W, C)")
    H, W, Cn = cube.shape
    tab = tables.line_table_2d(patch_size, phi_range)
    score = torch.empty((H, W), dtype=torch.float32, device=cube.device)
    s = torch.empty((H, W), dtype=torch.float64, device=cube.device) if return_sum else None
    mk = MaxKey(cube.device) if return_sum else None
    if _launch("neighbor2d_fused", cube.device, cube, H, W, Cn, tab.shape[1], tab.shape[0], tab, _flavour(flavour),
               score, s, mk, ok=(UNSUPPORTED,)) == UNSUPPORTED:
        return None
    return (score, s, mk) if return_sum else score


def neighbor2d_pipeline(cube, flavour="F1", patch_size=11, phi_range=9, bands=0):
    """cube (H, W, C) float32 -> (score float32, channel sums float64, MaxKey) through
    hipr_neighbor2d: channel sum and fixed-point stencil overlapped band by band (csrc/pipeline2d.cu).
    Returns None for parameters outside (11, 9)."""
    cube = _dev(cube, "cube", (torch.float32,))
    if cube.dim() != 3:
        raise ValueError("cube must be (H, W, C)")
    H, W, Cn = cube.shape
    tab = tables.line_table_2d(patch_size, phi_range)
    score = torch.empty((H, W), dtype=torch.float32, device=cube.device)
    s = torch.empty((H, W), dtype=torch.float64, device=cube.device)
    mk = MaxKey(cube.device)
    if _launch("neighbor2d", cube.device, cube, H, W, Cn, tab.shape[1], tab.shape[0], tab, _flavour(flavour), score, s,
               mk, int(bands), ok=(UNSUPPORTED,)) == UNSUPPORTED:
        return None
    return score, s, mk


def neighbor2d_score(cube, flavour="F1", calibration=None, patch_size=11, phi_range=9, dtype=None,
                     return_sum=False, denoise_h=None):
    """cube (H, W, C) or (N, H, W, C) float32 -> score map(s) (H, W) / (N, H, W).

    channel sum -> /max -> [NL-means denoise] -> edge pad -> line profiles -> epilogue, FOV by FOV (each
    FOV has its own max).  dtype=None (default): float64 channel sums feed the fixed-point stencil
    (lne2d_fixed; float32 score).  dtype=torch.float32 / float64: the sum image is stored in that
    type and the floating-point stencil of that type runs, dividing by the max on load.
    denoise_h: None, or the `h` of skimage.restoration.denoise_nl_means applied to the normalised sum
    image before the stencil (0.02 at syn/...measurement.py:108): the whole chain stays on the device."""
    cube = _dev(cube, "cube", (torch.float32,))
    if denoise_h is not None and cube.dim() == 3:
        s = channel_sum(cube, calibration, normalize=True, dtype=torch.float64)
        den = denoise_nl_means(s, h=denoise_h)
        # the denoised image is smooth: its 11-sample lines span ~1e-4 of a tile's range, below what the
        # 31-bit fixed-point stencil resolves to 1e-5 (measured 5e-6), so the float64 stencil runs here
        # (0.25 ms at 2048^2, next to ~9 ms of denoising)
        score = lne2d(den if dtype in (None, torch.float64) else den.to(dtype), flavour, patch_size, phi_range)
        return (score, den) if return_sum else score
    if cube.dim() == 4:
        # independent FOVs, each with its own max
        return _over_side_streams(cube, lambda c: neighbor2d_score(c, flavour, calibration, patch_size, phi_range,
                                                                   dtype, return_sum, denoise_h))
    if cube.dim() != 3:
        raise ValueError("cube must be (H, W, C) or (N, H, W, C)")
    if dtype is None and calibration is None:
        res = neighbor2d_pipeline(cube, flavour, patch_size, phi_range)
        if res is not None:
            score, s, mk = res
            if not return_sum:
                return score
            sn = torch.empty(s.shape, dtype=torch.float32, device=s.device)
            _launch("normalize_cast", cube.device, s, s.numel(), mk, sn)
            return score, sn
    fixed = dtype is None and tables.line_table_2d(patch_size, phi_range).shape[:2] == (9, 11)
    if dtype is None:
        dtype = torch.float64
    s, mk = channel_sum(cube, calibration, normalize=False, dtype=dtype, return_max=True)
    if fixed:
        score = lne2d_fixed(s, flavour, patch_size, phi_range, padded=False, range_keys=mk)
    else:
        score = lne2d(s, flavour, patch_size, phi_range, padded=False, maxkey=mk)
    if return_sum:
        _launch("normalize", cube.device, s, _ABI[dtype], s.numel(), mk)
        return score, s
    return score


def line_profile_2d(image_padded, patch_size, phi_range):
    """Literal gather: (Hp, Wp) -> (Hp-P+1, Wp-P+1, phi_range, P), same dtype."""
    image_padded = _dev(image_padded, "image_padded")
    if image_padded.dim() != 2:
        raise ValueError("Buffer has wrong number of dimensions (expected 2, got %d)" % image_padded.dim())
    tab = tables.line_table_2d(patch_size, phi_range)
    R, P = tab.shape[0], tab.shape[1]
    Hp, Wp = image_padded.shape
    out = torch.empty(_out_dims(image_padded.shape, P, True, "image") + (R, P), dtype=image_padded.dtype,
                      device=image_padded.device)
    _launch("line_profile_2d", image_padded.device, image_padded, Hp, Wp, _ABI[image_padded.dtype], P, R, tab, out)
    return out


def _host_gather(name, image_padded, ndim, table_args, what, per_sample, out, pinned):
    """The host gathers, hipr_<name>: a padded float64 image / volume in; out: the caller's C-contiguous float64
    array, or a new one (backed by page-locked memory with pinned=True) of the unpadded shape + (n_dirs,) and, with
    per_sample, + (P,)."""
    a = np.ascontiguousarray(image_padded)
    if a.dtype != np.float64:
        raise TypeError("image_padded must be float64, got %s" % a.dtype)
    if a.ndim != ndim:
        raise ValueError("Buffer has wrong number of dimensions (expected %d, got %d)" % (ndim, a.ndim))
    tab = (tables.line_table_2d if ndim == 2 else tables.line_table_3d)(*table_args)
    R, P = tab.shape[0], tab.shape[1]
    shape = _out_dims(a.shape, P, True, what) + ((R, P) if per_sample else (R,))
    if out is None:
        out = torch.empty(shape, dtype=torch.float64, pin_memory=True).numpy() if pinned else np.empty(shape, dtype=np.float64)
    elif out.shape != shape or out.dtype != np.float64 or not out.flags.c_contiguous:
        raise ValueError("out must be a C-contiguous float64 array of shape %s" % (shape,))
    _call(name, a, *a.shape, P, R, tab, out)
    return out


def line_profile_2d_host(image_padded, patch_size, phi_range, out=None, pinned=False):
    """numpy float64 (Hp, Wp) -> numpy float64 (Hp-P+1, Wp-P+1, phi_range, P) through hipr_line_profile_2d_host: the
    gather runs in row bands on the device under the device -> host copy of the previous bands.  out: a caller's
    array (page-locked or not); pinned=True returns an array backed by page-locked memory (torch's caching host
    allocator), which the copy reaches at the PCIe rate without the staging ring."""
    return _host_gather("line_profile_2d_host", image_padded, 2, (patch_size, phi_range), "image", True, out, pinned)


def _vol(volume, name):
    volume = _dev(volume, name)
    if volume.dim() != 3:
        raise ValueError("Buffer has wrong number of dimensions (expected 3, got %d)" % volume.dim())
    return volume


def line_profile_3d(volume_padded, patch_size, theta_range, phi_range):
    """Literal 5-D gather: (Xp, Yp, Zp) -> (X, Y, Z, (theta_range-1)*phi_range, P)."""
    v = _vol(volume_padded, "image_padded")
    tab = tables.line_table_3d(patch_size, theta_range, phi_range)
    T, P = tab.shape[0], tab.shape[1]
    out = torch.empty(_out_dims(v.shape, P, True, "volume") + (T, P), dtype=v.dtype, device=v.device)
    _launch("line_profile_3d", v.device, v, *v.shape, _ABI[v.dtype], P, T, tab, out)
    return out


def lne3d_dirs(volume, patch_size=11, theta_range=9, phi_range=9, padded=True, maxkey=None):
    """line_profile_memory_efficient_v2: per-direction relative centre value, (X, Y, Z, T)."""
    v = _vol(volume, "image_padded")
    tab = tables.line_table_3d(patch_size, theta_range, phi_range)
    T, P = tab.shape[0], tab.shape[1]
    out = torch.empty(_out_dims(v.shape, P, padded, "volume") + (T,), dtype=v.dtype, device=v.device)
    _launch("lne3d_dirs", v.device, v, *v.shape, int(bool(padded)), _ABI[v.dtype], P, T, tab, maxkey, out)
    return out


def lne3d_dirs_host(volume_padded, patch_size=11, theta_range=9, phi_range=9, out=None, pinned=False):
    """numpy float64 (Xp, Yp, Zp) -> numpy float64 (X, Y, Z, T) through hipr_lne3d_dirs_host
    (line_profile_memory_efficient_v2 for host arrays: bands of x-planes under the device -> host copy)."""
    return _host_gather("lne3d_dirs_host", volume_padded, 3, (patch_size, theta_range, phi_range), "volume", False,
                        out, pinned)


def line_profile_3d_host(volume_padded, patch_size=11, theta_range=9, phi_range=9, out=None, pinned=False):
    """numpy float64 (Xp, Yp, Zp) -> numpy float64 (X, Y, Z, T, P) through hipr_line_profile_3d_host
    (line_profile_v2 for host arrays: bands of x-planes under the device -> host copy)."""
    return _host_gather("line_profile_3d_host", volume_padded, 3, (patch_size, theta_range, phi_range), "volume", True,
                        out, pinned)


def lne3d(volume, flavour="F2", patch_size=11, theta_range=9, phi_range=9, padded=False, maxkey=None):
    """3-D score map (X, Y, Z).  flavour 'F2' / 'F3' / 'ME2', or 'V3' (needs padded=True)."""
    v = _vol(volume, "volume")
    if flavour == "V3":
        tab = tables.line_table_3d_v3(patch_size, theta_range, phi_range)
    else:
        tab = tables.line_table_3d(patch_size, theta_range, phi_range)
    T, P = tab.shape[0], tab.shape[1]
    out = torch.empty(_out_dims(v.shape, P, padded, "volume"), dtype=v.dtype, device=v.device)
    _launch("lne3d", v.device, v, *v.shape, int(bool(padded)), _ABI[v.dtype], P, T, tab, _flavour(flavour), maxkey, out)
    return out


def lne3d_fixed(volume, flavour="ME2", patch_size=11, theta_range=9, phi_range=9, padded=False, maxkey=None,
                dirs_only=False):
    """lne3d / lne3d_dirs on a 31-bit fixed-point copy of the volume (brick-local range, exact
    differences; csrc/lne3d.cu).  float32 out.  maxkey scales the 1e-8 epsilons of F3 / ME2 (None: the
    volume is already normalised).  Returns None outside (11, 9, 9)."""
    v = _vol(volume, "volume")
    tab = tables.line_table_3d(patch_size, theta_range, phi_range)
    T, P = tab.shape[0], tab.shape[1]
    out = torch.empty(_out_dims(v.shape, P, padded, "volume") + ((T,) if dirs_only else ()), dtype=torch.float32,
                      device=v.device)
    if _launch("lne3d_q", v.device, v, *v.shape, int(bool(padded)), _ABI[v.dtype], P, T, tab, _flavour(flavour),
               int(bool(dirs_only)), maxkey, out, what="lne3d_fixed", ok=(UNSUPPORTED,)) == UNSUPPORTED:
        return None
    return out


def neighbor3d_score(cube, flavour="ME2", patch_size=11, theta_range=9, phi_range=9, dtype=None, denoise_h=None,
                     denoise_distance=11):
    """cube (X, Y, Z, C) float32 -> score volume (X, Y, Z): channel sum -> /max -> edge pad ->
    3-D line profiles -> epilogue (bio/...analysis.py:807-817 for 'ME2').  dtype=None: float64 sums +
    fixed-point stencil (float32 score); torch.float32 / float64: floating-point stencil of that type.
    A batch (N, X, Y, Z, C) of independent z-stacks alternates between two streams, so that the channel sum of
    stack i+1 (HBM-bound) runs beside the stencil of stack i (ALU-bound); returns (N, X, Y, Z).
    denoise_h: with the NL-means denoise of bio/...analysis.py:454 (h = 0.03 there) between the normalisation and the
    stencil (csrc/nlm3d.cu, float64 stencil after it)."""
    cube = _dev(cube, "cube", (torch.float32,))
    if cube.dim() == 5:
        return _over_side_streams(cube, lambda c: neighbor3d_score(c, flavour, patch_size, theta_range, phi_range,
                                                                   dtype, denoise_h, denoise_distance))
    if cube.dim() != 4:
        raise ValueError("cube must be (X, Y, Z, C) or (N, X, Y, Z, C)")
    if denoise_h is not None:
        # bio/...analysis.py:452-462 in full: sum -> /max -> denoise_nl_means(h) -> edge pad -> me_v2 -> epilogue; the
        # denoised volume is too smooth for the fixed-point grid (as in 2-D): float64 stencil
        s = channel_sum(cube, None, normalize=True, dtype=torch.float64)
        den = denoise_nl_means(s, patch_distance=denoise_distance, h=denoise_h)
        return lne3d(den, flavour, patch_size, theta_range, phi_range, padded=False)
    s, mk = channel_sum(cube, None, normalize=False, dtype=dtype or torch.float64, return_max=True)
    if dtype is None:
        res = lne3d_fixed(s, flavour, patch_size, theta_range, phi_range, padded=False, maxkey=mk)
        if res is not None:
            return res
    return lne3d(s, flavour, patch_size, theta_range, phi_range, padded=False, maxkey=mk)


# ---------------------------------------------------------------------------------------------
# per-cell spectra
# ---------------------------------------------------------------------------------------------

def label_max(labels):
    labels = _dev(labels, "labels", (torch.int32, torch.int64))
    out = torch.empty(1, dtype=torch.int64, device=labels.device)
    _launch("label_max", labels.device, labels, labels.element_size(), labels.numel(), out)
    return out


def _cell_sums(device, cube, labels, Cn, max_label, sums=None, counts=None):
    """hipr_cell_spectra_accumulate of a cube (a tensor, or the device pointer of a resident one) over a contiguous
    label image into sums / counts; None: a new zeroed table (hipr_cell_spectra_reset) on `device`."""
    if sums is None:
        sums = torch.empty((max_label + 1, Cn), dtype=torch.float64, device=device)
        counts = torch.empty(max_label + 1, dtype=torch.int32, device=device)
        _launch("cell_spectra_reset", device, sums, counts, max_label, Cn)
    _launch("cell_spectra_accumulate", device, cube, labels, labels.element_size(), labels.numel(),
            labels.shape[-1] if labels.dim() > 1 else 0, Cn, max_label, sums, counts, None)
    return sums, counts


def cell_spectra_accumulate(cube, labels, max_label, sums=None, counts=None):
    """Adds this (slab of a) label image's per-label channel sums and pixel counts into
    sums (max_label+1, C) float64 / counts (max_label+1) int32 (allocated zeroed if None)."""
    cube = _dev(cube, "cube", (torch.float32,))
    labels = _dev(labels, "labels", (torch.int32, torch.int64))
    Cn = cube.shape[-1]
    # pixel p of the label image pairs with cube row p: a transposed label image has the right size, the wrong pairing
    if tuple(cube.shape[:-1]) != tuple(labels.shape):
        raise ValueError("cube %s and labels %s do not match: the cube must be labels.shape + (C,)"
                         % (tuple(cube.shape), tuple(labels.shape)))
    max_label = int(max_label)
    if (sums is None) != (counts is None):
        raise ValueError("pass both sums and counts (to keep accumulating) or neither")
    return _cell_sums(cube.device, cube, labels, Cn, max_label, sums, counts)


def cell_spectra_finalize(sums, counts):
    """-> (labels int64 (n,), area int64 (n,), avgint float64 (n, C), avgint_norm float64 (n, C)),
    rows in ascending order of the labels present.  Synchronises once to learn n."""
    max_label, Cn = sums.shape[0] - 1, sums.shape[1]
    dev = sums.device
    cap = max(max_label, 1)
    n_cells = torch.zeros(1, dtype=torch.int32, device=dev)
    labels = torch.empty(cap, dtype=torch.int64, device=dev)
    area = torch.empty(cap, dtype=torch.int64, device=dev)
    avg = torch.empty((cap, Cn), dtype=torch.float64, device=dev)
    norm = torch.empty((cap, Cn), dtype=torch.float64, device=dev)
    _launch("cell_spectra_finalize", dev, sums, counts, max_label, Cn, n_cells, labels, area, avg, norm)
    n = int(n_cells.item())
    return labels[:n], area[:n], avg[:n], norm[:n]


def cell_spectra(cube, labels, max_label=None):
    """regionprops-equivalent per-cell mean spectra of cube (..., C) over the label image."""
    if max_label is None:
        max_label = int(label_max(labels).item())
    sums, counts = cell_spectra_accumulate(cube, labels, max_label)
    return cell_spectra_finalize(sums, counts)


GEOMETRY_COLUMNS = ("centroid_row", "centroid_col", "major_axis_length", "minor_axis_length", "eccentricity",
                    "orientation", "mu20", "mu02", "mu11")


def cell_geometry(labels, max_label=None):
    """regionprops(segmentation) geometry of a 2-D label image: -> (labels int64 (n,), area int64 (n,),
    geometry float64 (n, 9) with columns GEOMETRY_COLUMNS), rows in ascending order of the labels present
    (syn/hiprfish_imaging_classify_spectra.py:38-46).  Integer raw moments on the device are exact."""
    labels = _dev(labels, "labels", (torch.int32, torch.int64))
    if labels.dim() != 2:
        raise ValueError("labels must be a 2-D label image")
    if max_label is None:
        max_label = int(label_max(labels).item())
    max_label = int(max_label)
    dev = labels.device
    Hh, Ww = labels.shape
    cap = max(max_label, 1)
    mom = torch.empty((max_label + 1, 6), dtype=torch.int64, device=dev)
    scratch = torch.empty(max_label + 1, dtype=torch.int32, device=dev)
    n_cells = torch.zeros(1, dtype=torch.int32, device=dev)
    lab = torch.empty(cap, dtype=torch.int64, device=dev)
    area = torch.empty(cap, dtype=torch.int64, device=dev)
    geom = torch.empty((cap, 9), dtype=torch.float64, device=dev)
    _launch("cell_moments", dev, labels, labels.element_size(), Hh, Ww, max_label, mom)
    _launch("cell_geometry_finalize", dev, mom, max_label, scratch, n_cells, lab, area, geom)
    n = int(n_cells.item())
    return lab[:n], area[:n], geom[:n]


def orientation_xy(geometry):
    """Orientation column in the 'xy' coordinate convention of scikit-image <= 0.15 (regionprops' default before
    0.16, the era the reference's cpython-35 artefacts point to): -0.5 * atan2(2 mu11, var_col - var_row), from the
    central moments cell_geometry returns (columns mu20 = row variance, mu02 = column variance, mu11).  cell_geometry's
    own `orientation` column follows the 'rc' convention of scikit-image >= 0.16.  Neither is pinned by the reference
    (no version file, scikit-image not installed here): PARITY UNPINNED, see INTEGRATION.md.  geometry: the (n, 9)
    table (torch tensor or numpy array) -> (n,) of the same kind."""
    if isinstance(geometry, torch.Tensor):
        mu20, mu02, mu11 = geometry[:, 6], geometry[:, 7], geometry[:, 8]
        return -0.5 * torch.atan2(2.0 * mu11, mu02 - mu20)
    g = np.asarray(geometry)
    return -0.5 * np.arctan2(2.0 * g[:, 8], g[:, 7] - g[:, 6])


def paint_labels(labels, values, max_label=None):
    """out[p] = values[labels[p]]: the `image[segmentation == label] = value` loops of
    eco/hiprfish_imaging_image_classification.py:64-70 / bio/...analysis.py:1247-1257 as one gather.
    values: (max_label + 1,) or (max_label + 1, K) float32 / float64 (or int32 / int64 / uint8 / bool lookup
    tables), row 0 = background."""
    labels = _dev(labels, "labels", (torch.int32, torch.int64))
    values = _dev(values, "values", (torch.float32, torch.float64, torch.int32, torch.int64, torch.uint8, torch.bool))
    squeeze = values.dim() == 1
    v2 = values.reshape(values.shape[0], -1)
    if max_label is None:
        max_label = v2.shape[0] - 1
    if v2.shape[0] < max_label + 1:
        raise ValueError("values needs max_label + 1 rows")
    K = v2.shape[1]
    out = torch.empty(tuple(labels.shape) + (() if squeeze else (K,)), dtype=values.dtype, device=labels.device)
    _launch("paint_labels", labels.device, labels, labels.element_size(), labels.numel(), v2, K, int(max_label),
            _ABI[values.dtype], out)
    return out


# ---------------------------------------------------------------------------------------------
# connected components (K10, csrc/label.cu)
# Per-pixel work runs in libhipr_b200's kernels.  The per-label tables between them (n + 1 or max_label + 1
# entries: which components to keep, the new numbering) are built with torch on the device.
# ---------------------------------------------------------------------------------------------

def _label_input(image, name, dtypes=_LABEL_DTYPES):
    """-> (contiguous tensor, with bool viewed as uint8; dtype code; (ndim, d0, d1, d2))."""
    image = _dev(image, name, dtypes)
    dims = _dims(image, name)
    raw = image.view(torch.uint8) if image.dtype == torch.bool else image
    return raw, _ABI[image.dtype], dims


def _connectivity(connectivity, ndim):
    if connectivity is None:
        return ndim
    if isinstance(connectivity, bool) or not isinstance(connectivity, (int, np.integer)):
        raise TypeError("connectivity must be an integer")
    if not 1 <= connectivity <= ndim:
        raise ValueError("connectivity must be in [1, %d], got %d" % (ndim, connectivity))
    return int(connectivity)


def _label(raw, code, dims, connectivity, invert=False, dtype=torch.int32):
    """Labels and the component count n (a 1-element int64 device tensor); no synchronisation."""
    dev = raw.device
    work = _workspace("label_workspace_bytes", dev, *dims, what="label (an image of 2^31 pixels or more)")
    out = torch.empty(raw.shape, dtype=dtype, device=dev)
    n = torch.empty(1, dtype=torch.int64, device=dev)
    _launch("label", dev, raw, code, int(invert), *dims, connectivity, work, work.numel(), out, out.element_size(), n)
    return out, n


def _label_counts(labels, dims, max_label, border=-1):
    """np.bincount(labels, minlength=max_label + 1) as int32 (border >= 0: only the pixels within `border` of an
    edge), and the number of labels outside [0, max_label]."""
    dev = labels.device
    counts = torch.empty(max_label + 1, dtype=torch.int32, device=dev)
    over = torch.empty(1, dtype=torch.int32, device=dev)
    _launch("label_counts", dev, labels, labels.element_size(), *dims, int(border), int(max_label), counts, over)
    return counts, over


def label(image, connectivity=None, return_num=False, dtype=torch.int32):
    """skimage.measure.label(image, background=0, connectivity=connectivity) on the device.

    image: 2-D (H, W) or 3-D (X, Y, Z) CUDA tensor.  bool / uint8 is a mask (non-zero is foreground, as
    scipy.ndimage.label); int32 / int64 is a label image whose neighbours connect when their values are equal and
    non-zero.  connectivity 1 .. ndim (default ndim): 4 / 8 neighbours in 2-D, 6 / 18 / 26 in 3-D.  Components are
    numbered 1 .. n in raster order of their first pixel.  -> labels of `dtype` (int32 or int64), and n when
    return_num (the only case that synchronises)."""
    if dtype not in (torch.int32, torch.int64):
        raise TypeError("dtype must be torch.int32 or torch.int64")
    raw, code, dims = _label_input(image, "image")
    out, n = _label(raw, code, dims, _connectivity(connectivity, dims[0]), dtype=dtype)
    return (out, int(n.item())) if return_num else out


def remove_small_objects(ar, min_size=64, connectivity=1):
    """skimage.morphology.remove_small_objects(ar, min_size, connectivity) on the device.

    bool ar: components (scipy.ndimage.label with that connectivity) of fewer than min_size pixels become False;
    the result is bool.  int32 / int64 ar: a label image whose labels are the components as they are (np.bincount
    sizes, connectivity unused); labels of fewer than min_size pixels become 0, the dtype is kept, and a negative
    label raises ValueError as np.bincount does.  Synchronises once (bool) or twice (labels)."""
    raw, code, dims = _label_input(ar, "ar", (torch.bool, torch.int32, torch.int64))
    conn = _connectivity(connectivity, dims[0])
    min_size = int(min_size)
    if min_size == 0:
        return ar.clone()
    if ar.dtype == torch.bool:
        lab, n = _label(raw, code, dims, conn)
        counts, _ = _label_counts(lab, dims, int(n.item()))
        keep = (counts >= min_size).to(torch.uint8)
        keep[0] = 0
        return paint_labels(lab, keep).view(torch.bool)
    max_label = int(label_max(raw).item())
    counts, over = _label_counts(raw, dims, max_label)
    if int(over.item()):
        raise ValueError("remove_small_objects: negative labels (np.bincount: 'list' argument must have no negative "
                         "elements)")
    lut = torch.arange(max_label + 1, dtype=ar.dtype, device=raw.device) * (counts >= min_size).to(ar.dtype)
    return paint_labels(raw, lut)


def binary_fill_holes(mask, connectivity=1):
    """scipy.ndimage.binary_fill_holes(mask, generate_binary_structure(ndim, connectivity)) on the device: the
    background components (at that connectivity) that touch no edge of the image are filled.  mask: bool / uint8
    (or int32 / int64, non-zero is foreground) 2-D or 3-D CUDA tensor -> bool.  Synchronises once."""
    raw, code, dims = _label_input(mask, "mask")
    lab, n = _label(raw, code, dims, _connectivity(connectivity, dims[0]), invert=True)
    on_edge, _ = _label_counts(lab, dims, int(n.item()), border=0)
    fill = (on_edge == 0).to(torch.uint8)
    fill[0] = 1                                        # label 0: the mask's own foreground
    return paint_labels(lab, fill).view(torch.bool)


def clear_border(labels, buffer_size=0, bgval=0):
    """skimage.segmentation.clear_border(labels, buffer_size, bgval) on the device.

    The image is relabelled with label(labels, background=0) at full connectivity; every component with a pixel
    within buffer_size of an edge is set to bgval, all other pixels keep their values.  The background is itself a
    component there: when a zero lies in that band, every zero becomes bgval.  labels: bool / uint8 / int32 / int64,
    2-D or 3-D; the result has its dtype.  ValueError if buffer_size >= a dimension.  Synchronises once."""
    raw, code, dims = _label_input(labels, "labels")
    buffer_size = int(buffer_size)
    if buffer_size < 0:
        raise ValueError("buffer_size must be >= 0")
    if any(buffer_size >= s for s in labels.shape):
        raise ValueError("buffer size may not be greater than labels size")
    bgval = int(bool(bgval)) if labels.dtype == torch.bool else int(bgval)
    info = torch.iinfo(raw.dtype)
    if not info.min <= bgval <= info.max:
        raise ValueError("bgval %d does not fit %s" % (bgval, raw.dtype))
    lab, n = _label(raw, code, dims, dims[0])
    on_edge, _ = _label_counts(lab, dims, int(n.item()), border=buffer_size)
    out = torch.empty_like(raw)
    _launch("label_clear", raw.device, raw, code, lab, raw.numel(), on_edge, bgval, out, what="clear_border")
    return out.view(torch.bool) if labels.dtype == torch.bool else out


def relabel_sequential(labels, offset=1):
    """skimage.segmentation.relabel_sequential(labels, offset) on the device: the non-zero labels present, in
    ascending order, become offset, offset + 1, ...; 0 stays 0.  labels: int32 / int64 -> (relabelled,
    forward_map (max_label + 1,), inverse_map (offset + n,)), with forward_map[old] = new and inverse_map[new] = old
    (the arrays behind scikit-image's ArrayMap).  The result keeps the input dtype unless the largest new label
    needs int64.  ValueError for offset < 1 or a negative label.  Synchronises twice."""
    raw, code, dims = _label_input(labels, "labels", (torch.int32, torch.int64))
    if isinstance(offset, bool) or not isinstance(offset, (int, np.integer)) or offset < 1:
        raise ValueError("Offset must be strictly positive.")
    offset = int(offset)
    max_label = int(label_max(raw).item())
    counts, over = _label_counts(raw, dims, max_label)
    if int(over.item()):
        raise ValueError("Cannot relabel array that contains negative values.")
    present = torch.nonzero(counts[1:]).flatten() + 1
    n = present.numel()
    out_dtype = raw.dtype if offset + n - 1 <= torch.iinfo(raw.dtype).max else torch.int64
    forward = torch.zeros(max_label + 1, dtype=out_dtype, device=raw.device)
    forward[present] = torch.arange(offset, offset + n, dtype=out_dtype, device=raw.device)
    inverse = torch.zeros(offset + n, dtype=raw.dtype, device=raw.device)
    inverse[offset:] = present.to(raw.dtype)
    return paint_labels(raw, forward), forward, inverse


# ---------------------------------------------------------------------------------------------
# marker watershed (K11, csrc/watershed.cu)
# ---------------------------------------------------------------------------------------------

# integer images become the float type that holds every value exactly
_WS_EXACT = {torch.uint8: torch.float32, torch.uint16: torch.float32, torch.int32: torch.float64}


def _watershed(image, markers, connectivity=1, mask=None):
    """watershed's checks and launch -> (labels, status): status is the kernel's 8 int64 status words on the device
    (hipr_b200.h: status, rounds and tile visits per phase, CTAs).  Synchronises once, for the NaN check."""
    image = _dev(image, "image", (torch.float32, torch.float64) + tuple(_WS_EXACT))
    markers = _dev(markers, "markers", (torch.int32, torch.int64))
    dims = _dims(image, "image")          # markers and mask: the image's shape
    _same(markers, image, ("markers", "image"))
    if mask is not None:
        mask = _dev(mask, "mask", (torch.bool, torch.uint8))
        _same(mask, image, ("mask", "image"))
        mask = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    conn = _connectivity(connectivity, image.dim())
    if image.dtype in _WS_EXACT:
        image = image.to(_WS_EXACT[image.dtype])
    else:
        nan = torch.isnan(image) if mask is None else torch.isnan(image) & (mask != 0)
        if bool(nan.any()):
            raise ValueError("image has NaN inside the mask: the flooding order is undefined there")
    code, lb = _ABI[image.dtype], markers.element_size()
    dev = image.device
    work = _workspace("watershed_workspace_bytes", dev, *dims, code, lb,
                      what="watershed (an image of 2^31 pixels or more)")
    out = torch.empty_like(markers)
    status = torch.empty(8, dtype=torch.int64, device=dev)
    _launch("watershed", dev, image, code, markers, lb, mask, *dims, conn, work, work.numel(), out, status)
    return out, status


def watershed(image, markers, connectivity=1, mask=None):
    """skimage.segmentation.watershed(image, markers, connectivity=connectivity, mask=mask) on the device.

    image: 2-D (H, W) or 3-D (X, Y, Z) CUDA tensor, float32 / float64 (uint8, uint16 and int32 are converted to a float
    type that holds them exactly).  markers: int32 / int64 of the same shape; every non-zero value is a marker,
    negative ones too; markers outside the mask are dropped.  mask: None or bool / uint8.  connectivity 1 .. ndim.
    -> labels with the markers' dtype: 0 outside the mask and where no marker reaches.

    Equal to scikit-image's heap flood wherever no pixel is tie-decided (two neighbours of minimal level with
    different labels); at ties it follows the deterministic rule of DESIGN.md K11 (markers first, then fewer hops
    within the level, then the smaller label) instead of scikit-image's age order.  ValueError for NaN inside the
    mask.  Synchronises twice: the NaN check and the status read."""
    out, status = _watershed(image, markers, connectivity, mask)
    st = int(status[0].item())
    if st:
        raise HiprError("watershed: phase %d did not converge within its round cap" % st)
    return out


# ---------------------------------------------------------------------------------------------
# binary morphology (K12, csrc/morphology.cu)
# ---------------------------------------------------------------------------------------------

MORPHOLOGY_MAX_EXTENT = 31     # HIPR_MORPH_MAX_EXTENT: disk(15), ball(15)
MORPHOLOGY_MAX_RUNS = 1000     # HIPR_MORPH_MAX_RUNS


def _structure(structure, ndim):
    """-> the structure as a C-contiguous uint8 numpy array of `ndim` axes (1 = member), checked as scipy checks it
    plus this kernel's limits.  None: generate_binary_structure(ndim, 1), built here (the product imports no scipy)."""
    if structure is None:
        idx = np.indices((3,) * ndim)
        return np.ascontiguousarray((np.abs(idx - 1).sum(axis=0) <= 1).astype(np.uint8))
    s = np.asarray(structure) != 0
    if s.ndim != ndim:
        raise RuntimeError("structure and input must have same dimensionality")
    if any(n % 2 == 0 for n in s.shape):
        raise ValueError("structure extents must be odd, got shape %s (an even extent needs scipy's origin shift, "
                         "which is not offered)" % (s.shape,))
    if max(s.shape) > MORPHOLOGY_MAX_EXTENT:
        raise ValueError("structure extents must be at most %d, got shape %s" % (MORPHOLOGY_MAX_EXTENT, s.shape))
    s = np.ascontiguousarray(s.astype(np.uint8))
    if _structure_runs(s).shape[0] > MORPHOLOGY_MAX_RUNS:
        raise ValueError("structure has more than %d runs of members along its last axis (the kernel's limit)"
                         % MORPHOLOGY_MAX_RUNS)
    return s


def _structure_runs(s):
    """The kernel's run table of a checked structure: (n, 4) int32 rows (d0, d1, first d2, last d2) of offsets from the
    centre, one per maximal run of members along the last axis; a 2-D structure has d0 = 0."""
    s3 = s.reshape((1,) * (3 - s.ndim) + s.shape)
    ptr = s3.ctypes.data_as(C.c_void_p)
    n = lib().hipr_morphology_runs(ptr, *s3.shape, None, 0)
    check(min(n, 0), "structure")
    runs = np.empty((n, 4), dtype=np.int32)
    check(min(lib().hipr_morphology_runs(ptr, *s3.shape, runs.ctypes.data_as(C.c_void_p), n), 0), "structure")
    return runs


def _iterations(iterations):
    if isinstance(iterations, bool) or not isinstance(iterations, (int, np.integer)):
        raise TypeError("iterations must be an integer")
    if iterations < 1:
        raise ValueError("iterations must be >= 1 (scipy's iterations < 1, repeat until nothing changes, is not "
                         "offered), got %d" % iterations)
    return int(iterations)


def _morphology(mask, structure, iterations, border_value, dilate):
    raw, _, dims = _label_input(mask, "mask", (torch.bool, torch.uint8))
    s = _structure(structure, dims[0])
    iterations = _iterations(iterations)
    dev = raw.device
    work = _workspace("morphology_workspace_bytes", dev, *dims, iterations,
                      what="binary morphology (an image of 2^31 pixels or more)")
    out = torch.empty(raw.shape, dtype=torch.uint8, device=dev)
    _launch("binary_morphology", dev, raw, *dims, s, *(s.shape + (1,) * (3 - s.ndim)), int(dilate),
            1 if border_value else 0, iterations, work, work.numel(), out,
            what="binary_dilation" if dilate else "binary_erosion")
    return out.view(torch.bool)


def binary_erosion(mask, structure=None, iterations=1, border_value=0):
    """scipy.ndimage.binary_erosion(mask, structure, iterations, border_value=border_value) on the device, bit for bit.

    mask: bool / uint8 CUDA tensor, 2-D (H, W) or 3-D (X, Y, Z), non-zero is True.  structure: None (the cross,
    generate_binary_structure(ndim, 1)) or a host array-like (numpy, CPU tensor) of ndim axes, non-zero is a member;
    every extent odd and at most 31.  out[p] = AND over members o of mask[p + o], with every pixel outside the image
    equal to border_value (non-zero counts as 1), repeated `iterations` (>= 1) times.  -> a new bool tensor.  One launch
    per pass; no host synchronisation and no device-to-host copy."""
    return _morphology(mask, structure, iterations, border_value, False)


def binary_dilation(mask, structure=None, iterations=1, border_value=0):
    """scipy.ndimage.binary_dilation(mask, structure, iterations, border_value=border_value) on the device, bit for
    bit: out[p] = OR over members o of mask[p - o] (the structure reflected), repeated `iterations` times.  Arguments,
    result and cost as binary_erosion; no host synchronisation and no device-to-host copy."""
    return _morphology(mask, structure, iterations, border_value, True)


def binary_opening(mask, structure=None, iterations=1, border_value=0):
    """scipy.ndimage.binary_opening(mask, structure, iterations, border_value=border_value) on the device, bit for bit:
    binary_erosion `iterations` times, then binary_dilation `iterations` times, both with border_value.  2 x iterations
    launches; no host synchronisation and no device-to-host copy."""
    return binary_dilation(binary_erosion(mask, structure, iterations, border_value), structure, iterations,
                           border_value)


def binary_closing(mask, structure=None, iterations=1, border_value=0):
    """scipy.ndimage.binary_closing(mask, structure, iterations, border_value=border_value) on the device, bit for bit:
    binary_dilation `iterations` times, then binary_erosion `iterations` times, both with border_value (so with the
    default 0 the closing erodes from the image edge, as scipy's does).  2 x iterations launches; no host
    synchronisation and no device-to-host copy."""
    return binary_erosion(binary_dilation(mask, structure, iterations, border_value), structure, iterations,
                          border_value)


# ---------------------------------------------------------------------------------------------
# 1-D k-means thresholding
# ---------------------------------------------------------------------------------------------

KMEANS_TRANSFORMS = {None: 0, "none": 0, "log10": 1, "log": 2}


class KMeans1DResult:
    """cluster_centers_ (k,), counts (k,), positive_means (k,), labels (int32 tensor, image shape) or None, mask
    (bool tensor: the brightest cluster) or None, n_iter, inertia, bright (label of the brightest cluster),
    n_samples, best_init."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def kmeans_threshold(image, n_clusters=2, random_state=0, n_init=1, transform=None, eps=0.0, positive_only=False,
                     max_iter=300, tol=1e-4, return_labels=True, return_mask=True, fill_label=0):
    """KMeans(n_clusters, random_state=random_state).fit_predict(f(image).reshape(-1, 1)) of scikit-learn 1.9 on the
    device, plus the scripts' mask orientation (syn/...measurement.py:125-137): f = identity, log10(image + eps)
    (transform='log10') or ln(image + eps) ('log'); positive_only: cluster image[image > 0] only, the other pixels
    get fill_label / mask 0 (bio/...analysis.py:819).  image: float32 / float64 CUDA tensor of any shape.
    Synchronises once (to read the 32-double result)."""
    image = _dev(image, "image")
    k = int(n_clusters)
    if not isinstance(random_state, (int, np.integer)):
        raise TypeError("random_state must be an integer seed (the reference passes 0)")
    nu = lib().hipr_kmeans1d_uniforms(k, int(n_init))
    if nu == -7:                                     # HIPR_E_RANGE: KM_MAXU = 256 seeding draws in the kernel
        raise ValueError("kmeans_threshold: n_init=%d is too large for k=%d: the kernel holds 256 seeding draws, %d per "
                         "initialisation" % (int(n_init), k, lib().hipr_kmeans1d_uniforms(k, 1)))
    check(nu if nu < 0 else 0, "kmeans_threshold")
    # scikit-learn's draws, in its order: RandomState(seed).choice (one double) then uniform(size=trials) per seed
    u = np.ascontiguousarray(np.random.RandomState(int(random_state)).random_sample(nu), dtype=np.float64)
    try:
        tcode = KMEANS_TRANSFORMS[transform]
    except KeyError:
        raise ValueError("transform must be None, 'log10' or 'log'")
    dev = image.device
    work = _workspace("kmeans1d_workspace_bytes", dev)
    labels = torch.empty(image.shape, dtype=torch.int32, device=dev) if return_labels else None
    mask = torch.empty(image.shape, dtype=torch.uint8, device=dev) if return_mask else None
    res = torch.empty(32, dtype=torch.float64, device=dev)
    _launch("kmeans1d", dev, image, _ABI[image.dtype], image.numel(), tcode, float(eps), int(bool(positive_only)), k,
            int(n_init), u, int(max_iter), float(tol), work, labels, int(fill_label), mask, res,
            what="kmeans_threshold")
    r = res.cpu().numpy()
    status = int(r[0])
    if status == 2:
        raise ValueError("Input X contains NaN or infinity.")          # scikit-learn's check_array message
    if status == 4:
        raise ValueError("n_samples=%d should be >= n_clusters=%d." % (int(r[1]), k))
    if status == 3:
        raise RuntimeError("a cluster ran empty during Lloyd iterations (scikit-learn would relocate it; not reproduced)")
    return KMeans1DResult(cluster_centers_=r[8:8 + k].copy(), counts=r[16:16 + k].astype(np.int64),
                          positive_means=r[24:24 + k].copy(), labels=labels, mask=mask.view(torch.bool) if mask is not None else None,
                          n_iter=int(r[4]), inertia=float(r[5]), bright=int(r[7]), n_samples=int(r[1]), best_init=int(r[6]))


# ---------------------------------------------------------------------------------------------
# host-buffer (numpy) entry points: copies happen inside the library
# ---------------------------------------------------------------------------------------------

def pinned_empty(shape, dtype=np.float32):
    """numpy array backed by page-locked memory from hipr_host_alloc (freed with the array)."""
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    _call("host_alloc", C.byref(p), max(nbytes, 1))

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                lib().hipr_host_free(self.ptr)
            except Exception:
                pass

    buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
    buf._hipr_owner = _Owner(p)
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def neighbor2d_score_host(cube, flavour="F1", patch_size=11, phi_range=9, return_sum=False, out=None, denoise_h=None):
    """numpy (H, W, C) float32 -> numpy (H, W) float32 score map, through hipr_neighbor2d_host (denoise_h: with the
    NL-means denoise of syn/...measurement.py:108 in the chain, hipr_neighbor2d_host_denoise)."""
    cube = _host_cube(cube, 3)
    H, W, Cn = cube.shape
    tab = tables.line_table_2d(patch_size, phi_range)
    score = out if out is not None else np.empty((H, W), dtype=np.float32)
    s = np.empty((H, W), dtype=np.float32) if return_sum else None
    name, denoise = ("neighbor2d_host", ()) if denoise_h is None else ("neighbor2d_host_denoise", (float(denoise_h),))
    _call(name, cube, H, W, Cn, tab.shape[1], tab.shape[0], tab, _flavour(flavour), *denoise, score, s)
    return (score, s) if return_sum else score


def neighbor2d_score_host_batch(cubes, flavour="F1", patch_size=11, phi_range=9, denoise_h=None, out=None):
    """A list of numpy (H, W, C) float32 cubes -> list of numpy (H, W) float32 score maps through
    hipr_neighbor2d_host_batch: FOV i + 1 crosses PCIe while FOV i is denoised (denoise_h), scored and read back."""
    cubes = [_host_cube(c) for c in cubes]
    if not cubes:
        raise ValueError("empty batch")
    H, W, Cn = cubes[0].shape
    for c in cubes:
        if c.shape != (H, W, Cn):
            raise ValueError("every cube of a batch must have the same (H, W, C)")
    n = len(cubes)
    tab = tables.line_table_2d(patch_size, phi_range)
    scores = out if out is not None else [np.empty((H, W), dtype=np.float32) for _ in range(n)]
    if len(scores) != n:
        raise ValueError("one output array per cube")
    _call("neighbor2d_host_batch", cubes, n, H, W, Cn, tab.shape[1], tab.shape[0], tab, _flavour(flavour),
          float(denoise_h) if denoise_h else 0.0, scores)
    return scores


def neighbor3d_score_host(cube, flavour="ME2", patch_size=11, theta_range=9, phi_range=9, out=None, denoise_h=None,
                          denoise_distance=11):
    """numpy (X, Y, Z, C) float32 -> numpy (X, Y, Z) float32 score volume, through hipr_neighbor3d_host
    (bio/...analysis.py:807-817 for 'ME2'); denoise_h: with the 3-D NL-means of bio/...analysis.py:454 in the chain
    (hipr_neighbor3d_host_denoise)."""
    cube = _host_cube(cube, 4)
    X, Y, Z, Cn = cube.shape
    tab = tables.line_table_3d(patch_size, theta_range, phi_range)
    score = out if out is not None else np.empty((X, Y, Z), dtype=np.float32)
    name, denoise = (("neighbor3d_host", ()) if denoise_h is None else
                     ("neighbor3d_host_denoise", (float(denoise_h), int(denoise_distance))))
    _call(name, cube, X, Y, Z, Cn, tab.shape[1], tab.shape[0], tab, _flavour(flavour), *denoise, score)
    return score


def neighbor2d_score_host_raw(cube, scale, flavour="F1", patch_size=11, phi_range=9, out=None):
    """numpy (H, W, C) uint16 / uint8 raw counts -> numpy (H, W) float32 score map, the score of the cube
    bioformats' rescale would produce (count / scale in float32), through hipr_neighbor2d_host_raw."""
    cube = _host_cube(cube, 3, (np.uint8, np.uint16), "raw cube")
    H, W, Cn = cube.shape
    tab = tables.line_table_2d(patch_size, phi_range)
    score = out if out is not None else np.empty((H, W), dtype=np.float32)
    _call("neighbor2d_host_raw", cube, cube.itemsize, float(scale), H, W, Cn, tab.shape[1], tab.shape[0], tab,
          _flavour(flavour), score, None)
    return score


def cell_spectra_host(cube, labels):
    """numpy cube (..., C) float32 + integer label image -> (labels, area, avgint, avgint_norm)."""
    cube = _host_cube(cube)
    labels = _host_cube(labels, None, (np.int32, np.int64), "labels")
    Cn = cube.shape[-1]
    if cube.shape[:-1] != labels.shape:
        raise ValueError("cube %s and labels %s do not match: the cube must be labels.shape + (C,)"
                         % (cube.shape, labels.shape))
    cols = labels.shape[-1] if labels.ndim > 1 else 0

    def fill(cap, n, *table):
        return _call("cell_spectra_host", cube, labels, labels.itemsize, labels.size, cols, Cn, cap, n, *table,
                     ok=(HIPR_E_RANGE,))

    def fetch(cap, n, *table):
        # the table is still on the device: fetch it (no second pass over the cube)
        return _call("cell_spectra_host_fetch", cap, *table, what="cell_spectra_host")

    return _cell_table(Cn, "cell_spectra_host", fill, fetch)


def _cell_rows(k, Cn):
    """A host cell table of k rows: labels, area, avgint, avgint_norm."""
    return np.empty(k, np.int64), np.empty(k, np.int64), np.empty((k, Cn), np.float64), np.empty((k, Cn), np.float64)


def _cell_table(Cn, what, fill, refill):
    """(labels, area, avgint, avgint_norm) from a host entry point: fill(cap, n, *table) writes up to cap rows and the
    number of cells to n; when they do not fit (HIPR_E_RANGE with n > cap), refill(cap, n, *table) writes them again
    to a table of cap = n rows."""
    n, cap = C.c_int64(0), 4096
    table = _cell_rows(cap, Cn)
    code = fill(cap, C.byref(n), *table)
    if code == HIPR_E_RANGE and n.value > cap:
        cap = int(n.value)
        table = _cell_rows(cap, Cn)
        code = refill(cap, C.byref(n), *table)
    check(code, what)
    k = int(n.value)
    return tuple(a[:k] for a in table)


class Fov:
    """One upload of a field of view for both steps of `measure_biofilm_images_no_reference`
    (syn/...measurement.py:161-173): the (H, W, C) float32 numpy cube is streamed to the current CUDA device once and
    stays resident; `score()` is lines 105-124 (without the denoise), `cell_spectra(segmentation)` lines 167-172.

        with hipr_b200.Fov(image_registered) as fov:
            image_final = fov.score("F1")
            ...                                  # k-means mask, label, watershed, clear_border on the device
            labels, area, avgint, avgint_norm = fov.cell_spectra(image_seg)   # image_seg: a CUDA tensor
    """

    def __init__(self, cube):
        cube = _host_cube(cube, 3)
        self.shape = cube.shape
        # hipr_fov_upload uses the current device (needed only to check device labels against it)
        self._device = torch.cuda.current_device() if torch.cuda.is_available() else None
        h = C.c_void_p()
        _call("fov_upload", cube, *cube.shape, C.byref(h))
        self._h = h

    def _handle(self):
        if self._h is None:
            raise ValueError("this field of view has been released")
        return self._h

    def score(self, flavour="F1", patch_size=11, phi_range=9, return_sum=False, out=None):
        H, W, _ = self.shape
        tab = tables.line_table_2d(patch_size, phi_range)
        score = out if out is not None else np.empty((H, W), dtype=np.float32)
        s = np.empty((H, W), dtype=np.float32) if return_sum else None
        _call("fov_score", self._handle(), tab.shape[1], tab.shape[0], tab, _flavour(flavour), score, s)
        return (score, s) if return_sum else score

    def cell_spectra(self, labels):
        """-> (labels, area, avgint, avgint_norm) numpy arrays, rows in ascending label order.  labels: the (H, W)
        int32 / int64 label image, as a numpy array (uploaded) or as a CUDA tensor on the handle's device (read in
        place, stream-ordered on torch's current stream: a label image from `watershed` never leaves the device)."""
        if isinstance(labels, torch.Tensor):
            return self._cell_spectra_device(labels)
        labels = _host_cube(labels, None, (np.int32, np.int64), "labels")
        H, W, Cn = self.shape
        if labels.shape != (H, W):
            raise ValueError("labels must be (%d, %d)" % (H, W))

        def fill(cap, n, *table):
            return _call("fov_cell_spectra", self._handle(), labels, labels.itemsize, cap, n, *table,
                         ok=(HIPR_E_RANGE,))

        # the cube is resident: the second call is one pass over it, no upload
        return _cell_table(Cn, "fov_cell_spectra", fill, fill)

    def _cell_spectra_device(self, labels):
        labels = _dev(labels, "labels", (torch.int32, torch.int64))
        H, W, Cn = self.shape
        if tuple(labels.shape) != (H, W):
            raise ValueError("labels must be (%d, %d)" % (H, W))
        if labels.device.index != self._device:
            raise ValueError("labels live on cuda:%d, this field of view on cuda:%d" % (labels.device.index,
                                                                                       self._device))
        cube = self.device_arrays()[0]
        max_label = int(label_max(labels).item())
        if max_label <= 0:
            return _cell_rows(0, Cn)
        sums, counts = _cell_sums(labels.device, cube, labels, Cn, max_label)
        return tuple(t.cpu().numpy() for t in cell_spectra_finalize(sums, counts))

    def device_arrays(self):
        """(cube, channel sums, range keys) device pointers as ints, for callers that continue on the device."""
        a, b, c = C.c_void_p(), C.c_void_p(), C.c_void_p()
        _call("fov_device_arrays", self._handle(), C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def close(self):
        if self._h is not None:
            lib().hipr_fov_release(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
