"""Tensor-level operators: CUDA torch tensors in, CUDA torch tensors out.

Each function checks its arguments, allocates outputs / scratch with torch (the C ABI never
allocates), and enqueues the kernels of ``libcamlin_b200.so`` on torch's current CUDA stream.
The main ones are also registered as PyTorch custom ops (``torch.ops.camera_linearity.*``) at
the bottom of this file.  There is no CPU implementation: a CPU tensor raises.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import HdrMergeArgs, IcrfProblem, check

Tensor = torch.Tensor


# ------------------------------------------------------------------------------------- helpers
def _require_cuda(*tensors: Optional[Tensor]) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"expected a torch.Tensor, got {type(t)}")
        if not t.is_cuda:
            raise RuntimeError("camera_linearity_b200 operators run on CUDA tensors only "
                               "(no CPU fallback); move the data to the GPU first")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("all tensors must live on the same CUDA device")
    if dev is None:
        raise RuntimeError("no CUDA tensor given")
    return dev


def _first_cuda_device(obj) -> Optional[torch.device]:
    if isinstance(obj, torch.Tensor):
        return obj.device if obj.is_cuda else None
    if isinstance(obj, (list, tuple)):
        for item in obj:
            dev = _first_cuda_device(item)
            if dev is not None:
                return dev
    return None


def _on_device(fn):
    """Run an operator with the device of its tensors current: the library launches on the CURRENT device and on
    ``torch.cuda.current_stream()``, so tensors living on cuda:N while another device is current would otherwise be
    handed to the wrong device's stream (and the per-device queries -- SM count, occupancy, function attributes --
    would describe the wrong GPU)."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = None
        for a in list(args) + list(kwargs.values()):
            dev = _first_cuda_device(a)
            if dev is not None:
                break
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper


def _ptr(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _f64c(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float64:
        t = t.to(torch.float64)
    return t.contiguous()


def _dn_view(t: Tensor) -> Tuple[Tensor, int]:
    """Integer image -> (contiguous tensor whose bytes are uint8/uint16 DNs, bytes per DN)."""
    if t.dtype == torch.uint8:
        return t.contiguous(), 1
    if t.dtype in (torch.uint16, torch.int16):
        return t.contiguous(), 2
    raise TypeError(f"digital-number images must be uint8 or uint16, got {t.dtype}")


def _lut_pair(icrf: Tensor, icrf_diff: Optional[Tensor], channels: int):
    icrf = _f64c(icrf)
    if icrf.ndim == 1:
        icrf = icrf.reshape(-1, 1)
    if icrf.ndim != 2 or icrf.shape[1] != channels:
        raise ValueError(f"ICRF must have shape (BITS, {channels}); got {tuple(icrf.shape)}")
    if icrf_diff is not None:
        icrf_diff = _f64c(icrf_diff)
        if icrf_diff.ndim == 1:
            icrf_diff = icrf_diff.reshape(-1, 1)
        if icrf_diff.shape != icrf.shape:
            raise ValueError("ICRF_diff must have the same shape as ICRF")
    return icrf, icrf_diff


# ------------------------------------------------------------------------------------- K1
@_on_device
def linearize(val: Tensor, std: Optional[Tensor], icrf: Tensor, icrf_diff: Optional[Tensor] = None,
              max_dn: float = 255.0, return_bins: bool = False):
    """``out[..., c] = ICRF[bin(val[..., c]), c]`` (+ ``ICRF_diff[bin] * std``); K1 of DESIGN.md.

    val: integer DN image (uint8 / uint16) or floating image in [0, 1]; the last dimension is the
    channel axis and must match the ICRF's second dimension (a 1-D ICRF = one channel).
    """
    _require_cuda(val, std, icrf, icrf_diff)
    lib = _lib.load()
    channels = 1 if icrf.ndim == 1 else int(icrf.shape[1])
    if val.ndim == 0 or (channels > 1 and val.shape[-1] != channels):
        raise ValueError(f"last dimension of val {tuple(val.shape)} must equal the ICRF channel count {channels}")
    lut, dlut = _lut_pair(icrf, icrf_diff, channels)
    bits = int(lut.shape[0])
    use_std = std is not None and dlut is not None
    std_c = _f64c(std) if use_std else None
    if use_std and std_c.shape != val.shape:
        raise ValueError("Value and std shapes must match.")
    n = val.numel()
    out_val = torch.empty(val.shape, dtype=torch.float64, device=val.device)
    out_std = torch.empty_like(out_val) if use_std else None
    bins = None
    if val.dtype.is_floating_point:
        v = _f64c(val)
        if return_bins:
            bins = torch.empty(val.shape, dtype=torch.int16, device=val.device)
        check(lib.cl_linearize_f64(_ptr(v), float(max_dn), _ptr(std_c), _ptr(lut),
                                   _ptr(dlut) if use_std else None, _ptr(out_val), _ptr(out_std),
                                   _ptr(bins), n, channels, bits, _stream()), "cl_linearize_f64")
    else:
        v, dn_bytes = _dn_view(val)
        check(lib.cl_linearize_dn(_ptr(v), dn_bytes, _ptr(std_c), _ptr(lut),
                                  _ptr(dlut) if use_std else None, _ptr(out_val), _ptr(out_std), n,
                                  channels, bits, _stream()), "cl_linearize_dn")
        if return_bins:
            bins = v
    if return_bins:
        return out_val, out_std, bins
    return out_val, out_std


# ------------------------------------------------------------------------------------- K2
@_on_device
def flat_roi_means(flat: Tensor, flat_std: Tensor, roi: Tuple[int, int, int, int],
                   max_dn: float = 255.0) -> Tensor:
    """ROI means ``[m_0..m_{C-1}, ms_0..ms_{C-1}]`` of a flat field (measurand.py:561-583)."""
    _require_cuda(flat, flat_std)
    lib = _lib.load()
    if flat.ndim != 3:
        raise ValueError("flat field must be (H, W, C)")
    h, w, c = (int(s) for s in flat.shape)
    if flat.dtype.is_floating_point:
        f, fbytes = _f64c(flat), 8
    else:
        f, fbytes = _dn_view(flat)
    fs = _f64c(flat_std)
    out = torch.empty(2 * c, dtype=torch.float64, device=flat.device)
    ws_bytes = lib.cl_flat_roi_means_workspace_bytes(h, w, c)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=flat.device)
    r0, r1, c0, c1 = (int(x) for x in roi)
    check(lib.cl_flat_roi_means(_ptr(f), fbytes, float(max_dn), _ptr(fs), h, w, c, r0, r1, c0, c1,
                                _ptr(out), _ptr(ws), ws_bytes, _stream()), "cl_flat_roi_means")
    return out


@_on_device
def hdr_merge(dn: Sequence[Tensor], std: Optional[Sequence[Optional[Tensor]]],
              exposures: Sequence[float], icrf: Tensor, icrf_diff: Tensor, *,
              std_lut: Optional[Tensor] = None,
              darks: Optional[Sequence[Optional[Tensor]]] = None,
              dark_scales: Optional[Sequence[float]] = None, dark_threshold: float = 0.0,
              median_kernel: int = 3, flat: Optional[Tensor] = None,
              flat_std: Optional[Tensor] = None, flat_means: Optional[Tensor] = None,
              algo: int = 0, out: Optional[Tuple[Tensor, Tensor]] = None,
              workspace: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """Fused weighted HDR merge of N exposures (K2 of DESIGN.md); returns (radiance, std).

    dn[k]: (H, W, C) uint8/uint16 exposures in ascending exposure order; std[k]: float64
    uncertainty images (an entry may be None when ``std_lut`` is given); darks[k]: the dark frame
    selected for exposure k or None; flat / flat_std / flat_means: optional flat-field epilogue.
    """
    n = len(dn)
    if n < 1 or n > _lib.CL_MAX_EXPOSURES:
        raise ValueError(f"hdr_merge supports 1..{_lib.CL_MAX_EXPOSURES} exposures, got {n}")
    if len(exposures) != n:
        raise ValueError("one exposure time per image is required")
    _require_cuda(*dn, icrf, icrf_diff, std_lut, flat, flat_std, flat_means)
    lib = _lib.load()
    first, dn_bytes = _dn_view(dn[0])
    if first.ndim != 3:
        raise ValueError("exposures must be (H, W, C) images")
    h, w, c = (int(s) for s in first.shape)
    keep: List[Tensor] = []            # keeps converted tensors alive until the launch is enqueued

    def _img(t: Tensor) -> Tensor:
        v, b = _dn_view(t)
        if b != dn_bytes or tuple(v.shape) != (h, w, c):
            raise ValueError("all exposures / dark frames must share dtype and shape")
        keep.append(v)
        return v

    dn_c = [_img(t) for t in dn]
    lut, dlut = _lut_pair(icrf, icrf_diff, c)
    if dlut is None:
        raise ValueError("ICRF_diff is required for the merge")
    bits = int(lut.shape[0])
    std_c: List[Optional[Tensor]] = []
    for k in range(n):
        s = None if std is None else std[k]
        if s is None:
            if std_lut is None:
                raise ValueError(f"exposure {k} has no uncertainty image and no std_lut was given")
            std_c.append(None)
        else:
            _require_cuda(s)
            s = _f64c(s)
            if tuple(s.shape) != (h, w, c):
                raise ValueError("Value and std shapes must match.")
            keep.append(s)
            std_c.append(s)
    sl = None
    if std_lut is not None:
        sl, _ = _lut_pair(std_lut, None, c)
        if sl.shape[0] != bits:
            raise ValueError("std_lut must have as many rows as the ICRF")
    dark_c: List[Optional[Tensor]] = [None] * n
    if darks is not None:
        if len(darks) != n:
            raise ValueError("darks must have one entry (or None) per exposure")
        for k, d in enumerate(darks):
            if d is not None:
                _require_cuda(d)
                dark_c[k] = _img(d)
    scales = [1.0] * n if dark_scales is None else [float(x) for x in dark_scales]

    args = HdrMergeArgs()
    args.n_exposures, args.height, args.width, args.channels = n, h, w, c
    args.dn_bytes, args.bits = dn_bytes, bits
    dn_arr = (C.c_void_p * n)(*[t.data_ptr() for t in dn_c])
    std_arr = (C.c_void_p * n)(*[_ptr(t) for t in std_c])
    dark_arr = (C.c_void_p * n)(*[_ptr(t) for t in dark_c])
    t_arr = (C.c_double * n)(*[float(x) for x in exposures])
    sc_arr = (C.c_double * n)(*scales)
    args.dn = C.cast(dn_arr, C.POINTER(C.c_void_p))
    args.std = C.cast(std_arr, C.POINTER(C.c_void_p))
    args.dark = C.cast(dark_arr, C.POINTER(C.c_void_p))
    args.exposure_s = C.cast(t_arr, C.POINTER(C.c_double))
    args.dark_scale = C.cast(sc_arr, C.POINTER(C.c_double))
    args.lut, args.dlut, args.std_lut = _ptr(lut), _ptr(dlut), _ptr(sl)
    args.dark_threshold = float(dark_threshold)
    args.median_kernel = int(median_kernel)
    fv = fs = fm = None
    if flat is not None:
        if flat_std is None or flat_means is None:
            raise ValueError("flat-field correction needs flat, flat_std and flat_means")
        if flat.dtype.is_floating_point:
            fv, fbytes = _f64c(flat), 8
        else:
            fv, fbytes = _dn_view(flat)
        fs, fm = _f64c(flat_std), _f64c(flat_means)
        if tuple(fv.shape) != (h, w, c) or tuple(fs.shape) != (h, w, c) or fm.numel() != 2 * c:
            raise ValueError("flat field shapes must match the exposures; flat_means must be (2C,)")
        args.flat_bytes = fbytes
        args.flat, args.flat_std, args.flat_means = _ptr(fv), _ptr(fs), _ptr(fm)
    else:
        args.flat_bytes = 0
    if out is None:
        out_val = torch.empty((h, w, c), dtype=torch.float64, device=first.device)
        out_std = torch.empty_like(out_val)
    else:
        out_val, out_std = out
        _require_cuda(out_val, out_std)
        for o in (out_val, out_std):
            if o.dtype != torch.float64 or tuple(o.shape) != (h, w, c) or not o.is_contiguous():
                raise ValueError("out tensors must be contiguous float64 (H, W, C)")
    args.out_val, args.out_std = _ptr(out_val), _ptr(out_std)
    args.algo = int(algo)
    ws_bytes = lib.cl_hdr_merge_workspace_bytes(C.byref(args))
    ws = workspace
    if ws_bytes and (ws is None or ws.numel() * ws.element_size() < ws_bytes):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=first.device)
    check(lib.cl_hdr_merge(C.byref(args), _ptr(ws) if ws_bytes else None, ws_bytes, _stream()),
          "cl_hdr_merge")
    return out_val, out_std


@_on_device
def gaussian_weight(val: Tensor) -> Tuple[Tensor, Tensor]:
    """``apply_gaussian_weight`` (measurand.py:606-618): returns (w, dw)."""
    _require_cuda(val)
    lib = _lib.load()
    v = _f64c(val)
    w = torch.empty_like(v)
    dw = torch.empty_like(v)
    check(lib.cl_gaussian_weight(_ptr(v), _ptr(w), _ptr(dw), v.numel(), _stream()), "cl_gaussian_weight")
    return w, dw


@_on_device
def bad_pixel_filter(val: Tensor, std: Optional[Tensor], dark_val: Tensor, threshold: float,
                     kernel: int) -> Tuple[Tensor, Optional[Tensor]]:
    """``filter_larger_than_by_map`` (measurand.py:543-557) on float64 (H, W, C) images."""
    _require_cuda(val, std, dark_val)
    lib = _lib.load()
    if val.ndim != 3:
        raise ValueError("bad_pixel_filter expects (H, W, C) images")
    v, s, d = _f64c(val), _f64c(std), _f64c(dark_val)
    if d.shape != v.shape:
        d = d.expand_as(v).contiguous()
    h, w, c = (int(x) for x in v.shape)
    out_v = torch.empty_like(v)
    out_s = torch.empty_like(v) if s is not None else None
    check(lib.cl_bad_pixel_filter(_ptr(v), _ptr(s), _ptr(d), float(threshold), int(kernel), h, w, c,
                                  _ptr(out_v), _ptr(out_s), _stream()), "cl_bad_pixel_filter")
    return out_v, out_s


@_on_device
def flat_field_normalize(val: Tensor, std: Tensor, flat_val: Tensor, flat_std: Tensor,
                         flat_means: Tensor) -> Tuple[Tensor, Tensor]:
    """``normalize_by_map`` (measurand.py:559-604) given the ROI means."""
    _require_cuda(val, std, flat_val, flat_std, flat_means)
    lib = _lib.load()
    v, s, fv, fs, fm = (_f64c(t) for t in (val, std, flat_val, flat_std, flat_means))
    c = int(v.shape[-1])
    out_v, out_s = torch.empty_like(v), torch.empty_like(v)
    check(lib.cl_flat_field_normalize(_ptr(v), _ptr(s), _ptr(fv), _ptr(fs), _ptr(fm), v.numel(), c,
                                      _ptr(out_v), _ptr(out_s), _stream()), "cl_flat_field_normalize")
    return out_v, out_s


# ------------------------------------------------------------------------------------- K3
WELFORD_U16_MAX_FRAMES = 65536     # the stack form's limit for uint16 frames (DESIGN.md, K3); beyond: streaming form
_U16_TABLE_ROWS = 65536


def _welford_frames(frames: Tensor) -> Tensor:
    if frames.dtype not in (torch.uint8, torch.uint16) or frames.ndim < 2:
        raise TypeError("frames must be a uint8 or uint16 tensor (F, ...)")
    return frames.contiguous()


def _welford_table(icrf: Optional[Tensor], channels: int, wide: bool) -> Tuple[Optional[Tensor], int]:
    """The ICRF as a contiguous float64 (rows, C) table and its row count; a uint16 stack takes up to 65536 rows."""
    if icrf is None:
        return None, 0
    lut, _ = _lut_pair(icrf, None, channels)
    rows = int(lut.shape[0])
    if wide and not 1 <= rows <= _U16_TABLE_ROWS:
        raise ValueError(f"an ICRF for uint16 frames has 1 ... 65536 rows, got {rows}")
    return lut, rows


def _dn_out_of_range() -> IndexError:
    return IndexError("a frame's digital number has no row in the ICRF (index out of bounds, as NumPy raises)")


@_on_device
def welford_update(frames: Tensor, mean: Tensor, m2: Tensor, count0: int,
                   icrf: Optional[Tensor] = None, max_dn: float = 255.0) -> int:
    """Fold ``frames`` (F, H, W, C) uint8 or uint16 into the running (mean, m2) state in place -- the
    reference's sequential recurrence (video_processing.py:205-208), bit-identical float64.  With uint16 frames and
    an ICRF shorter than 65536 rows, a DN without a row raises IndexError before the state changes."""
    _require_cuda(frames, mean, m2, icrf)
    lib = _lib.load()
    fr = _welford_frames(frames)
    wide = fr.dtype == torch.uint16
    f = int(fr.shape[0])
    n = fr[0].numel() if f else mean.numel()
    c = int(fr.shape[-1])
    for s in (mean, m2):
        if s.dtype != torch.float64 or not s.is_contiguous() or s.numel() != n:
            raise ValueError("mean / m2 must be contiguous float64 with one element per sample")
    lut, rows = _welford_table(icrf, c, wide)
    if not wide:
        check(lib.cl_welford_update(_ptr(fr), f, n, c, _ptr(lut), float(max_dn), _ptr(mean), _ptr(m2),
                                    int(count0), _stream()), "cl_welford_update")
        return count0 + f
    if lut is not None and rows < _U16_TABLE_ROWS and fr.numel() and _max_dn(fr) >= rows:
        raise _dn_out_of_range()
    check(lib.cl_welford_update_u16(_ptr(fr), f, n, c, _ptr(lut), rows, float(max_dn), _ptr(mean), _ptr(m2),
                                    int(count0), _stream()), "cl_welford_update_u16")
    return count0 + f


@_on_device
def welford_finalize(mean: Tensor, m2: Optional[Tensor], count: int, max_dn: float = 255.0,
                     dtype: torch.dtype = torch.uint8):
    """Returns (sem float64 or None, quantised mean) -- video_processing.py:210-215 with repair R9.  The quantised
    mean is ``np.around(mean * max_dn).astype(dtype)``: ``dtype`` torch.uint8 (8-bit frames) or torch.uint16 (16-bit
    frames, the R9 extension of DESIGN.md section 3)."""
    _require_cuda(mean, m2)
    if dtype not in (torch.uint8, torch.uint16):
        raise TypeError(f"the quantised mean is uint8 or uint16, not {dtype}")
    lib = _lib.load()
    n = mean.numel()
    sem = torch.empty_like(mean) if m2 is not None else None
    mean_q = torch.empty(mean.shape, dtype=dtype, device=mean.device)
    fn = lib.cl_welford_finalize_u16 if dtype == torch.uint16 else lib.cl_welford_finalize
    check(fn(_ptr(mean), _ptr(m2), int(count), n, float(max_dn), _ptr(sem), _ptr(mean_q), _stream()),
          "cl_welford_finalize_u16" if dtype == torch.uint16 else "cl_welford_finalize")
    return sem, mean_q


@_on_device
def welford_stack(frames: Tensor, icrf: Optional[Tensor] = None, max_dn: float = 255.0,
                  workspace: Optional[Tensor] = None):
    """Mean / SEM / quantised mean of a resident frame stack (F, H, W, C) uint8 or uint16 (K3 of DESIGN.md).  The
    quantised mean has the frames' dtype.  uint16 stacks of more than WELFORD_U16_MAX_FRAMES frames raise
    CamlinError (CL_ERR_UNSUPPORTED): ``video_processing.welford_stack`` takes the streaming form for them."""
    _require_cuda(frames, icrf)
    lib = _lib.load()
    fr = _welford_frames(frames)
    wide = fr.dtype == torch.uint16
    f = int(fr.shape[0])
    if f < 1:
        raise ValueError("at least one frame is required")
    shape = tuple(fr.shape[1:])
    n = fr[0].numel()
    c = int(fr.shape[-1])
    lut, rows = _welford_table(icrf, c, wide)
    mean = torch.empty(shape, dtype=torch.float64, device=fr.device)
    sem = torch.empty_like(mean)
    mean_q = torch.empty(shape, dtype=fr.dtype, device=fr.device)
    ws_bytes = lib.cl_welford_stack_workspace_bytes(f, n)
    ws = workspace
    if ws is None or ws.numel() * ws.element_size() < ws_bytes:
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=fr.device)
    if not wide:
        check(lib.cl_welford_stack(_ptr(fr), f, n, c, _ptr(lut), float(max_dn), _ptr(mean), _ptr(sem),
                                   _ptr(mean_q), _ptr(ws), ws_bytes, _stream()), "cl_welford_stack")
        return mean, sem, mean_q
    check(lib.cl_welford_stack_u16(_ptr(fr), f, n, c, _ptr(lut), rows, float(max_dn), _ptr(mean), _ptr(sem),
                                   _ptr(mean_q), _ptr(ws), ws_bytes, _stream()), "cl_welford_stack_u16")
    # a table shorter than 65536 rows: the kernel flags DNs without a row in the workspace header's second word
    if lut is not None and rows < _U16_TABLE_ROWS and n and bool(ws.reshape(-1).view(torch.uint8)[4:8].any()):
        raise _dn_out_of_range()
    return mean, sem, mean_q


# ------------------------------------------------------------------------------------- K4
def _plan_device(fn):
    """Method flavour of ``_on_device`` for objects that carry ``self.device``."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        dev = self.device
        if dev.index is None or dev.index == torch.cuda.current_device():
            return fn(self, *args, **kwargs)
        with torch.cuda.device(dev):
            return fn(self, *args, **kwargs)
    return wrapper


def _max_dn(dn: Tensor) -> int:
    """Largest sample of a uint8 / uint16 tensor (torch has no max for uint16: widened to int32 first, never viewed
    as int16, which would turn 32768..65535 negative)."""
    return int(dn.max()) if dn.dtype == torch.uint8 else int(dn.to(torch.int32).max())


class IcrfEnergyPlan:
    """Device-resident state of one calibration problem (one colour channel): pixel samples,
    PCA basis, scratch.  ``partial()`` and ``finalize()`` map onto the C ABI calls so that a
    multi-GPU driver can all-reduce the pair sums in between (parallel.py).  uint8 stacks take curves of up to 256
    points, uint16 stacks (16- / 12-bit cameras) up to 65536 through the ``_u16`` entry points."""

    def __init__(self, dn_stack: Tensor, std_stack: Optional[Tensor], exposures, mean_icrf,
                 pca_basis: Tensor, lower: int, upper: int, use_mean_icrf: bool, n_candidates: int):
        dev = _require_cuda(dn_stack, std_stack, pca_basis)
        self.device = dev
        self.lib = _lib.load()
        if dn_stack.dtype not in (torch.uint8, torch.uint16):
            raise TypeError("the calibration value stack must be uint8 or uint16 "
                            "(ICRF_calibration_exposure.py:191 indexes the curve with it)")
        self.wide = dn_stack.dtype == torch.uint16          # 16-bit (or 12-bit) camera: the _u16 entry points
        if dn_stack.ndim != 3:
            raise ValueError("image_stack must be a 3D CuPy array with shape (X, Y, N).")
        n_exp = int(dn_stack.shape[2])
        exposures = np.asarray(exposures, dtype=np.float64)
        if exposures.ndim != 1 or exposures.size != n_exp:
            raise ValueError("exposure_values must be a 1D CuPy array matching the third dimension of image_stack.")
        if not 2 <= n_exp <= _lib.CL_MAX_PAIR_EXPOSURES:
            raise ValueError(f"2..{_lib.CL_MAX_PAIR_EXPOSURES} exposures are supported, got {n_exp}")
        self.dn = dn_stack.contiguous().reshape(-1, n_exp)
        self.n_pixels = int(self.dn.shape[0])
        self.std = None
        if std_stack is not None:
            if std_stack.shape != dn_stack.shape:
                raise ValueError("Value and std shapes must match.")
            self.std = _f64c(std_stack).reshape(-1, n_exp)
        self.pca = _f64c(pca_basis)
        self.datapoints = int(self.pca.shape[0])
        self.n_pc = int(self.pca.shape[1])
        self.mean = None if mean_icrf is None else _f64c(torch.as_tensor(mean_icrf, device=dev))
        if self.n_pixels and _max_dn(self.dn) >= self.datapoints:
            raise IndexError("digital numbers exceed the curve length")
        self.exposures = (C.c_double * n_exp)(*exposures.tolist())
        self.n_real = int(n_candidates)
        s_pad = max(32, (self.n_real + 31) // 32 * 32)
        self.prob = IcrfProblem(s_pad, self.n_pc + (0 if use_mean_icrf else 1), self.datapoints,
                                1 if use_mean_icrf else 0, int(lower), int(upper), n_exp,
                                1 if self.std is not None else 0)
        self.n_pairs = n_exp * (n_exp - 1) // 2
        f64 = dict(dtype=torch.float64, device=dev)
        self.params = torch.zeros((s_pad, self.prob.n_params), **f64)
        self.curves = torch.empty((s_pad, self.datapoints), **f64)
        self.valid = torch.empty(s_pad, dtype=torch.int32, device=dev)
        self.tables = torch.empty(self.lib.cl_icrf_tables_bytes(C.byref(self.prob)), dtype=torch.uint8, device=dev)
        self.pair_acc = torch.empty((s_pad, self.n_pairs, 2), **f64)
        self.energy = torch.empty(s_pad, **f64)
        self.ws_bytes = self.lib.cl_icrf_energy_workspace_bytes(C.byref(self.prob), self.n_pixels)
        self.ws = torch.empty(max(self.ws_bytes, 16), dtype=torch.uint8, device=dev)
        # exchange buffer of the fused tail (generation counter + ticket; with peers: the slots the other
        # ranks push their pair sums into).  Single rank: a private zeroed buffer.
        self._own_exchange = torch.zeros(self.lib.cl_icrf_exchange_bytes(C.byref(self.prob), 1), dtype=torch.uint8,
                                         device=dev)
        self.peers = _lib.PeerGroup()
        self.peers.world, self.peers.rank = 1, 0
        self.peers.buffers[0] = self._own_exchange.data_ptr()
        self._peer_keepalive = None

    def attach_peers(self, exchange) -> None:
        """Use the peer-memory exchange of ``parallel.PeerExchange`` (one buffer per rank, mapped on this device):
        ``population()`` then sums the pair sums of all ranks inside its tail kernel."""
        self.peers = exchange.peer_group()
        self._peer_keepalive = exchange

    def set_params(self, params: Tensor) -> None:
        """params: (S, n_params) -- one row per candidate (device or host)."""
        p = torch.as_tensor(params, dtype=torch.float64)
        if p.shape != (self.n_real, self.prob.n_params):
            raise ValueError(f"params must be ({self.n_real}, {self.prob.n_params})")
        self.params[: self.n_real].copy_(p, non_blocking=True)

    @_plan_device
    def curves_and_tables(self) -> None:
        check(self.lib.cl_icrf_curves(C.byref(self.prob), _ptr(self.mean), _ptr(self.pca), _ptr(self.params),
                                      _ptr(self.curves), _ptr(self.valid), _ptr(self.tables), _stream()),
              "cl_icrf_curves")

    @_plan_device
    def partial(self) -> Tensor:
        name = "cl_icrf_energy_partial_u16" if self.wide else "cl_icrf_energy_partial"
        check(getattr(self.lib, name)(C.byref(self.prob), _ptr(self.tables), _ptr(self.dn), _ptr(self.std),
                                      self.exposures, self.n_pixels, _ptr(self.pair_acc), _ptr(self.ws),
                                      self.ws_bytes, _stream()), name)
        return self.pair_acc

    @_plan_device
    def finalize(self) -> Tensor:
        check(self.lib.cl_icrf_energy_finalize(C.byref(self.prob), _ptr(self.pair_acc), _ptr(self.valid),
                                               _ptr(self.energy), _stream()), "cl_icrf_energy_finalize")
        return self.energy[: self.n_real]

    @_plan_device
    def population(self, select=None) -> Tensor:
        """Partial kernel + fused tail (CTA reduction, exchange with the attached peers, finalize): the energies
        of the candidates whose curves / tables are current, over the pixels of ALL ranks.  ``select``: a
        ``_lib.DeSelectArgs`` -- the DE selection of the generation then runs in the same launch."""
        if self.n_pixels == 0:
            raise ValueError("population() needs at least one pixel on every rank")
        name = "cl_icrf_energy_population_u16" if self.wide else "cl_icrf_energy_population"
        check(getattr(self.lib, name)(C.byref(self.prob), _ptr(self.tables), _ptr(self.dn), _ptr(self.std),
                                      self.exposures, self.n_pixels, _ptr(self.valid), _ptr(self.pair_acc),
                                      _ptr(self.energy), _ptr(self.ws), self.ws_bytes, C.byref(self.peers),
                                      None if select is None else C.byref(select), _stream()), name)
        return self.energy[: self.n_real]

    def evaluate(self, params) -> Tensor:
        """Energies (S,) of a population (over the pixels of all attached ranks)."""
        self.set_params(params)
        self.curves_and_tables()
        return self.population()


class DeviceDE:
    """Differential evolution with the population on the device (``csrc/de.cu``): scipy's
    'currenttobest1bin' / dither / deferred-updating generation as two kernels around a caller-supplied
    population objective ``evaluate(params (S, P) device tensor) -> energies (S,) device tensor``.
    Nothing in ``step()`` synchronises with the host; ``poll()`` reads the 32-byte status block."""

    def __init__(self, evaluate, lower, upper, init_unit_population: Tensor, seed: int, dither=(0.0, 1.95),
                 recombination: float = 0.4, tol: float = 0.01, atol: float = 0.0):
        dev = _require_cuda(init_unit_population)
        self.device = dev
        self.lib = _lib.load()
        self.evaluate = evaluate
        self.pop = _f64c(init_unit_population).clone()
        self.S, self.P = (int(v) for v in self.pop.shape)
        f64 = dict(dtype=torch.float64, device=dev)
        self.lower = torch.as_tensor(np.asarray(lower, dtype=np.float64)).to(dev)
        self.upper = torch.as_tensor(np.asarray(upper, dtype=np.float64)).to(dev)
        self.trial = torch.empty_like(self.pop)
        self.params = torch.empty_like(self.pop)
        self.generation = torch.zeros(1, dtype=torch.int64, device=dev)
        self.status = torch.zeros(4, dtype=torch.int32, device=dev)
        self.best = torch.zeros(3, **f64)
        self.seed, self.dither, self.cr, self.tol, self.atol = int(seed), dither, float(recombination), float(tol), float(atol)
        # energies of the initial population (scipy: _calculate_population_energies + _promote_lowest_energy)
        self.energies = self.evaluate(self.scaled(self.pop)).clone()
        l = int(torch.argmin(self.energies))
        if l != 0:
            self.pop[[0, l]] = self.pop[[l, 0]]
            self.energies[[0, l]] = self.energies[[l, 0]]

    def scaled(self, unit: Tensor) -> Tensor:
        return 0.5 * (self.lower + self.upper) + (unit - 0.5) * torch.abs(self.upper - self.lower)

    @_plan_device
    def step(self) -> None:
        check(self.lib.cl_de_trial(_ptr(self.pop), self.S, self.P, float(self.dither[0]), float(self.dither[1]), self.cr,
                                   self.seed, _ptr(self.generation), _ptr(self.lower), _ptr(self.upper),
                                   _ptr(self.trial), _ptr(self.params), _stream()), "cl_de_trial")
        trial_energies = self.evaluate(self.params)
        check(self.lib.cl_de_select(_ptr(self.pop), _ptr(self.energies), _ptr(self.trial), _ptr(trial_energies),
                                    self.S, self.P, self.tol, self.atol, _ptr(self.generation), _ptr(self.status),
                                    _ptr(self.best), _stream()), "cl_de_select")

    # ---- fused generation on an IcrfEnergyPlan: 4 launches, capturable in a CUDA graph ----
    @classmethod
    def for_plan(cls, plan: "IcrfEnergyPlan", lower, upper, init_unit_population: Tensor, seed: int, **kw):
        """DE whose objective is ``plan`` (K4).  One generation = ``cl_de_trial_curves`` (trial vectors + candidate
        curves) and ``cl_icrf_energy_population`` (partial kernel + fused reduce / peer exchange / finalize /
        DE selection): three kernels, no NCCL launch, nothing on the host."""
        if plan.n_real != init_unit_population.shape[0] or plan.prob.n_params != init_unit_population.shape[1]:
            raise ValueError("the plan must be built for exactly this population")
        self = cls(lambda params: plan.evaluate(params), lower, upper, init_unit_population, seed, **kw)
        self.plan = plan
        self._select = None
        self._graph = None
        self._graph_steps = 0
        return self

    @_plan_device
    def step_fused(self) -> None:
        plan = self.plan
        check(self.lib.cl_de_trial_curves(C.byref(plan.prob), _ptr(self.pop), self.S, float(self.dither[0]),
                                          float(self.dither[1]), self.cr, self.seed, _ptr(self.generation),
                                          _ptr(self.lower), _ptr(self.upper), _ptr(self.trial), _ptr(plan.params),
                                          _ptr(plan.mean), _ptr(plan.pca), _ptr(plan.curves), _ptr(plan.valid),
                                          _ptr(plan.tables), _stream()), "cl_de_trial_curves")
        if self._select is None:
            sel = _lib.DeSelectArgs()
            sel.pop, sel.energies, sel.trial = _ptr(self.pop), _ptr(self.energies), _ptr(self.trial)
            sel.n_members, sel.n_params, sel.tol, sel.atol = self.S, self.P, self.tol, self.atol
            sel.generation, sel.status, sel.best = _ptr(self.generation), _ptr(self.status), _ptr(self.best)
            self._select = sel
        plan.population(self._select)            # ... -> finalize -> selection, in the tail kernel's last block

    def run_graph(self, generations: int, per_graph: int = 8) -> None:
        """Advance ``generations`` generations (a multiple of ``per_graph``) by replaying a CUDA graph of
        ``per_graph`` fused generations: every pointer and the generation counter live on the device, so the
        captured launches are valid for every replay."""
        if generations % per_graph:
            raise ValueError("generations must be a multiple of per_graph")
        if self._graph is None or self._graph_steps != per_graph:
            self.step_fused()                                # warm-up outside the capture (module load, attributes)
            generations -= 1
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for _ in range(per_graph):
                    self.step_fused()
            self._graph, self._graph_steps = g, per_graph
            for _ in range(generations % per_graph):
                self.step_fused()
            generations -= generations % per_graph
        for _ in range(generations // per_graph):
            self._graph.replay()

    def poll(self):
        """(converged, generations, best energy) -- one small device-to-host read."""
        st = self.status.cpu()
        return bool(st[0]), int(st[1]), float(self.best[0].cpu())

    @property
    def x(self) -> Tensor:
        return self.scaled(self.pop[0])


# ------------------------------------------------------------------------------------- linearity
@_on_device
def pair_statistics(x_val: Tensor, x_std: Optional[Tensor], y_val: Tensor, y_std: Optional[Tensor],
                    multiplier: float, lower: Optional[Sequence[Optional[float]]] = None,
                    upper: Optional[Sequence[Optional[float]]] = None) -> Tensor:
    """Fused thresholds -> scaled difference -> per-channel statistics over all leading axes of one
    exposure pair (measurand.py:375-428, 620-655, 318-350).  Returns a (2, 3, C) tensor:
    [absolute | relative] x [mean | std | error]."""
    _require_cuda(x_val, x_std, y_val, y_std)
    lib = _lib.load()
    if x_val.shape != y_val.shape:
        raise ValueError('Measurands are not broadcastable.')
    c = int(x_val.shape[-1])
    xv, xs, yv, ys = _f64c(x_val), _f64c(x_std), _f64c(y_val), _f64c(y_std)
    lo = hi = None
    if lower is not None or upper is not None:
        lower = [None] * c if lower is None else list(lower)
        upper = [None] * c if upper is None else list(upper)
        if len(lower) != c or len(upper) != c:
            raise ValueError("The length of 'lower' and 'upper' must match the size of the independent axis.")
        lo = (C.c_double * c)(*[-float("inf") if v is None else float(v) for v in lower])
        hi = (C.c_double * c)(*[float("inf") if v is None else float(v) for v in upper])
    stats = torch.empty((2, 3, c), dtype=torch.float64, device=x_val.device)
    ws_bytes = lib.cl_pair_statistics_workspace_bytes(c)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x_val.device)
    check(lib.cl_pair_statistics(_ptr(xv), _ptr(xs), _ptr(yv), _ptr(ys), float(multiplier), lo, hi, xv.numel(), c,
                                 _ptr(stats), _ptr(ws), ws_bytes, _stream()), "cl_pair_statistics")
    return stats


# ------------------------------------------------------------------------------------- Measurand operators
_BINARY_OPS = {"add": 0, "sub": 1, "mul": 2, "div": 3, "pow": 4}


def suffix_period(x_shape, y_shape) -> Optional[int]:
    """``y`` pairs with ``x`` element i <-> i % period when its shape is the same as ``x``'s, or equals ``x``'s trailing
    dimensions (after dropping leading 1s): a per-channel vector, a scalar.  Returns the period or None."""
    xs, ys = tuple(x_shape), tuple(y_shape)
    while ys and ys[0] == 1 and len(ys) > 1:
        ys = ys[1:]
    if ys == (1,) or ys == ():
        return 1
    if len(ys) <= len(xs) and xs[len(xs) - len(ys):] == ys:
        n = 1
        for d in ys:
            n *= int(d)
        return n
    return None


@_on_device
def measurand_binary(op: str, x_val: Tensor, x_std: Optional[Tensor], y_val: Tensor, y_std: Optional[Tensor]):
    """``x (op) y`` with first-order uncertainty propagation (measurand.py:106-241), one fused pass.  ``y`` must be
    the same shape as ``x`` or a suffix operand (see ``suffix_period``).  Returns (val, std or None)."""
    _require_cuda(x_val, x_std, y_val, y_std)
    lib = _lib.load()
    period = suffix_period(x_val.shape, y_val.shape)
    if period is None or x_val.numel() == 0:
        raise ValueError("measurand_binary needs y to be the same shape as x or a suffix of it")
    xv, xs, yv, ys = _f64c(x_val), _f64c(x_std), _f64c(y_val), _f64c(y_std)
    use_std = xs is not None or ys is not None
    out_v = torch.empty_like(xv)
    out_s = torch.empty_like(xv) if use_std else None
    check(lib.cl_measurand_binary(_BINARY_OPS[op], _ptr(xv), _ptr(xs), _ptr(yv), _ptr(ys), xv.numel(), int(period),
                                  _ptr(out_v), _ptr(out_s), _stream()), "cl_measurand_binary")
    return out_v, out_s


@_on_device
def measurand_log(val: Tensor, std: Optional[Tensor], base10: bool):
    """``log_e`` / ``log_10`` with the reference's literal uncertainty formulae (measurand.py:243-279)."""
    _require_cuda(val, std)
    lib = _lib.load()
    v, s = _f64c(val), _f64c(std)
    out_v = torch.empty_like(v)
    out_s = torch.empty_like(v) if s is not None else None
    check(lib.cl_measurand_log(1 if base10 else 0, _ptr(v), _ptr(s), v.numel(), _ptr(out_v), _ptr(out_s), _stream()),
          "cl_measurand_log")
    return out_v, out_s


@_on_device
def measurand_difference(x_val: Tensor, x_std: Optional[Tensor], y_val: Tensor, y_std: Optional[Tensor],
                         multiplier: float):
    """``compute_difference`` (measurand.py:620-655): returns (abs_val, abs_std, rel_val, rel_std), one pass."""
    _require_cuda(x_val, x_std, y_val, y_std)
    lib = _lib.load()
    if x_val.shape != y_val.shape:
        raise ValueError('Measurands are not broadcastable.')
    xv, xs, yv, ys = _f64c(x_val), _f64c(x_std), _f64c(y_val), _f64c(y_std)
    use_std = xs is not None or ys is not None
    av, rv = torch.empty_like(xv), torch.empty_like(xv)
    a_s = torch.empty_like(xv) if use_std else None
    r_s = torch.empty_like(xv) if use_std else None
    check(lib.cl_measurand_difference(_ptr(xv), _ptr(xs), _ptr(yv), _ptr(ys), float(multiplier), xv.numel(), _ptr(av),
                                      _ptr(a_s), _ptr(rv), _ptr(r_s), _stream()), "cl_measurand_difference")
    return av, a_s, rv, r_s


# ------------------------------------------------------------------------------------- noise profiles
@_on_device
def noise_profiles(frames: Tensor, mean_u8: Tensor, hist: Optional[Tensor] = None) -> Tensor:
    """Accumulate the joint (mean DN, frame DN) histogram per channel of ``frames`` (F, H, W, C) uint8 against the uint8
    mean frame (video_processing.py:92-104).  ``hist``: int64 (256, 256, C), created zeroed when not given."""
    _require_cuda(frames, mean_u8, hist)
    lib = _lib.load()
    if frames.dtype != torch.uint8 or mean_u8.dtype != torch.uint8 or frames.ndim < 2:
        raise TypeError("frames and the mean frame must be uint8")
    fr, mu = frames.contiguous(), mean_u8.contiguous()
    if tuple(fr.shape[1:]) != tuple(mu.shape):
        raise ValueError("the mean frame must have the shape of one frame")
    c = int(fr.shape[-1])
    if hist is None:
        hist = torch.zeros((256, 256, c), dtype=torch.int64, device=fr.device)
    elif hist.dtype != torch.int64 or tuple(hist.shape) != (256, 256, c) or not hist.is_contiguous():
        raise ValueError("hist must be a contiguous int64 (256, 256, C) tensor")
    check(lib.cl_noise_profiles(_ptr(fr), int(fr.shape[0]), mu.numel(), c, _ptr(mu), _ptr(hist), _stream()),
          "cl_noise_profiles")
    return hist


# ------------------------------------------------------------------------------------- histogram
@_on_device
def channel_histogram(val: Tensor, std: Optional[Tensor], channel: int, bins: int, included_range=None):
    """np.histogram of the finite values of one channel (measurand.py:430-469), weighted by 1/std when
    ``std`` is given.  Returns ``(hist, bin_edges)`` as NumPy arrays like np.histogram; only the ``bins``
    results (and, without a range, the two extrema) cross PCIe."""
    _require_cuda(val, std)
    lib = _lib.load()
    v = _f64c(val)
    s = _f64c(std)
    c_total = int(v.shape[-1])
    n_px = v.numel() // c_total
    if included_range is None:
        # np.histogram's _get_outer_edges over the samples that survive the masks
        col = v.reshape(-1, c_total)[:, channel]
        keep = torch.isfinite(col)
        if s is not None:
            keep &= s.reshape(-1, c_total)[:, channel] != 0
        kept = col[keep]
        if kept.numel() == 0:
            first, last = 0.0, 1.0
        else:
            first, last = float(kept.min()), float(kept.max())
    else:
        first, last = float(included_range[0]), float(included_range[1])
        if first > last:
            raise ValueError("max must be larger than min in range parameter.")
    if first == last:
        first, last = first - 0.5, last + 0.5
    edges_np = np.linspace(first, last, bins + 1, endpoint=True, dtype=np.float64)
    edges = torch.from_numpy(edges_np).to(v.device)
    hist = torch.empty(bins, dtype=torch.float64, device=v.device)
    check(lib.cl_channel_histogram(_ptr(v), _ptr(s), n_px, c_total, int(channel), int(bins), first, last, _ptr(edges),
                                   _ptr(hist), _stream()), "cl_channel_histogram")
    h = hist.cpu().numpy()
    return (h if s is not None else h.astype(np.intp)), edges_np


# ------------------------------------------------------------------------------------- egress
@_on_device
def quantize_8bit(val: Tensor, max_dn: float = 255.0, return_max: bool = False):
    """The array part of ImageSet.save_8bit (image_set.py:343-350): normalise by ``amax`` when it exceeds 1,
    scale by MAX_DN, round half-even, cast to uint8 -- on the device, so the result crosses PCIe as one
    byte per sample.  Returns the uint8 tensor (and the device scalar ``amax`` if asked)."""
    _require_cuda(val)
    if val.numel() == 0:
        raise ValueError("zero-size array to reduction operation maximum which has no identity")
    lib = _lib.load()
    v = _f64c(val)
    out = torch.empty(v.shape, dtype=torch.uint8, device=v.device)
    mx = torch.empty((), dtype=torch.float64, device=v.device)
    ws_bytes = lib.cl_quantize_8bit_workspace_bytes()
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=v.device)
    check(lib.cl_quantize_8bit(_ptr(v), v.numel(), float(max_dn), _ptr(out), _ptr(mx), _ptr(ws), ws_bytes,
                               _stream()), "cl_quantize_8bit")
    return (out, mx) if return_max else out


# ------------------------------------------------------------------------------------- custom ops
# The C-ABI layer as PyTorch custom ops (``torch.ops.camera_linearity.*``): functional, tensor-in / tensor-out
# wrappers over the functions above, one per entry point of include/camera_linearity.h that does data-path work.
# Optional per-exposure images travel as a list plus an index list (-1 = none): torch schemas have no
# Optional-in-list for custom ops.
def _pick(images: List[Tensor], index: Sequence[int], n: int) -> Optional[List[Optional[Tensor]]]:
    if not images:
        return None
    if len(index) != n:
        raise ValueError("index list must have one entry per exposure")
    return [None if int(i) < 0 else images[int(i)] for i in index]


@torch.library.custom_op("camera_linearity::linearize", mutates_args=(), device_types="cuda")
def _op_linearize(val: Tensor, std: Optional[Tensor], icrf: Tensor, icrf_diff: Optional[Tensor],
                  max_dn: float) -> List[Tensor]:
    v, s = linearize(val, std, icrf, icrf_diff, max_dn)
    return [v] if s is None else [v, s]


@torch.library.custom_op("camera_linearity::hdr_merge", mutates_args=(), device_types="cuda")
def _op_hdr_merge(dn: List[Tensor], std: List[Tensor], exposures: List[float], icrf: Tensor,
                  icrf_diff: Tensor, algo: int) -> List[Tensor]:
    v, s = hdr_merge(dn, std, exposures, icrf, icrf_diff, algo=algo)
    return [v, s]


@torch.library.custom_op("camera_linearity::hdr_merge_corrected", mutates_args=(), device_types="cuda")
def _op_hdr_merge_corrected(dn: List[Tensor], std: List[Tensor], std_index: List[int], std_lut: Optional[Tensor],
                            exposures: List[float], icrf: Tensor, icrf_diff: Tensor, darks: List[Tensor],
                            dark_index: List[int], dark_scales: List[float], dark_threshold: float,
                            median_kernel: int, flat: Optional[Tensor], flat_std: Optional[Tensor],
                            flat_means: Optional[Tensor], algo: int) -> List[Tensor]:
    """cl_hdr_merge with everything it takes: ``std[std_index[k]]`` is exposure k's uncertainty image (-1: sigma from
    ``std_lut``), ``darks[dark_index[k]]`` its dark frame (-1: none), ``dark_scales[k]`` the exposure scaling of that
    dark frame, the flat field with its ROI means (``flat_roi_means``)."""
    n = len(dn)
    v, s = hdr_merge(dn, _pick(std, std_index, n), exposures, icrf, icrf_diff, std_lut=std_lut,
                     darks=_pick(darks, dark_index, n), dark_scales=dark_scales if dark_scales else None,
                     dark_threshold=dark_threshold, median_kernel=median_kernel, flat=flat, flat_std=flat_std,
                     flat_means=flat_means, algo=algo)
    return [v, s]


@torch.library.custom_op("camera_linearity::flat_roi_means", mutates_args=(), device_types="cuda")
def _op_flat_roi_means(flat: Tensor, flat_std: Tensor, roi: List[int], max_dn: float) -> Tensor:
    return flat_roi_means(flat, flat_std, tuple(roi), max_dn)


@torch.library.custom_op("camera_linearity::welford_stack", mutates_args=(), device_types="cuda")
def _op_welford_stack(frames: Tensor, icrf: Optional[Tensor], max_dn: float) -> List[Tensor]:
    return list(welford_stack(frames, icrf, max_dn))


@torch.library.custom_op("camera_linearity::welford_update", mutates_args=("mean", "m2"), device_types="cuda")
def _op_welford_update(frames: Tensor, mean: Tensor, m2: Tensor, count0: int, icrf: Optional[Tensor],
                       max_dn: float) -> None:
    welford_update(frames, mean, m2, count0, icrf, max_dn)


@torch.library.custom_op("camera_linearity::welford_finalize", mutates_args=(), device_types="cuda")
def _op_welford_finalize(mean: Tensor, m2: Tensor, count: int, max_dn: float) -> List[Tensor]:
    sem, mean_u8 = welford_finalize(mean, m2, count, max_dn)
    return [sem, mean_u8]


@torch.library.custom_op("camera_linearity::welford_finalize_u16", mutates_args=(), device_types="cuda")
def _op_welford_finalize_u16(mean: Tensor, m2: Tensor, count: int, max_dn: float) -> List[Tensor]:
    """welford_finalize with the uint16 mean of 16-bit frames."""
    sem, mean_u16 = welford_finalize(mean, m2, count, max_dn, torch.uint16)
    return [sem, mean_u16]


@torch.library.custom_op("camera_linearity::gaussian_weight", mutates_args=(), device_types="cuda")
def _op_gaussian_weight(val: Tensor) -> List[Tensor]:
    return list(gaussian_weight(val))


def _icrf_problem(n_candidates: int, n_params: int, datapoints: int, use_mean: bool, lower: int, upper: int,
                  n_exposures: int, use_std: bool) -> IcrfProblem:
    if n_candidates % 32:
        raise ValueError("candidates must be padded to a multiple of 32 (one lane per candidate)")
    return IcrfProblem(int(n_candidates), int(n_params), int(datapoints), 1 if use_mean else 0, int(lower), int(upper),
                       int(n_exposures), 1 if use_std else 0)


@torch.library.custom_op("camera_linearity::icrf_energy_curves", mutates_args=(), device_types="cuda")
def _op_icrf_energy_curves(params: Tensor, mean_icrf: Optional[Tensor], pca: Tensor, lower: int, upper: int,
                           n_exposures: int, use_std: bool) -> List[Tensor]:
    """cl_icrf_curves: (S, n_params) candidates -> [curves (S, D) float64, valid (S,) int32, tables (uint8 scratch
    consumed by icrf_energy_partial)].  S must be a multiple of 32."""
    _require_cuda(params, mean_icrf, pca)
    lib = _lib.load()
    prm, pc = _f64c(params), _f64c(pca)
    s_, n_params = (int(v) for v in prm.shape)
    d_ = int(pc.shape[0])
    prob = _icrf_problem(s_, n_params, d_, mean_icrf is not None, lower, upper, n_exposures, use_std)
    curves = torch.empty((s_, d_), dtype=torch.float64, device=prm.device)
    valid = torch.empty(s_, dtype=torch.int32, device=prm.device)
    tables = torch.empty(lib.cl_icrf_tables_bytes(C.byref(prob)), dtype=torch.uint8, device=prm.device)
    mean = None if mean_icrf is None else _f64c(mean_icrf)
    check(lib.cl_icrf_curves(C.byref(prob), _ptr(mean), _ptr(pc), _ptr(prm), _ptr(curves), _ptr(valid), _ptr(tables),
                             _stream()), "cl_icrf_curves")
    return [curves, valid, tables]


@torch.library.custom_op("camera_linearity::icrf_energy_partial", mutates_args=(), device_types="cuda")
def _op_icrf_energy_partial(tables: Tensor, dn: Tensor, std: Optional[Tensor], exposures: List[float],
                            n_candidates: int, n_params: int, datapoints: int, use_mean: bool, lower: int,
                            upper: int) -> Tensor:
    """cl_icrf_energy_partial: per-(candidate, exposure pair) numerator / denominator sums over the given pixels,
    (S, pairs, 2) float64 -- what ranks all-reduce before icrf_energy_finalize.  A uint16 ``dn`` (16- / 12-bit
    cameras, datapoints <= 65536) goes to cl_icrf_energy_partial_u16."""
    _require_cuda(tables, dn, std)
    lib = _lib.load()
    if dn.dtype not in (torch.uint8, torch.uint16) or dn.ndim != 2:
        raise TypeError("dn must be a (pixels, N) uint8 or uint16 tensor")
    n_px, n_exp = (int(v) for v in dn.shape)
    if n_px and _max_dn(dn) >= datapoints:          # the kernel would read the curve's last row instead
        raise IndexError("digital numbers exceed the curve length")
    prob = _icrf_problem(n_candidates, n_params, datapoints, use_mean, lower, upper, n_exp, std is not None)
    sd = None if std is None else _f64c(std)
    acc = torch.empty((n_candidates, n_exp * (n_exp - 1) // 2, 2), dtype=torch.float64, device=dn.device)
    ws_bytes = lib.cl_icrf_energy_workspace_bytes(C.byref(prob), n_px)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dn.device)
    t = (C.c_double * n_exp)(*[float(x) for x in exposures])
    name = "cl_icrf_energy_partial_u16" if dn.dtype == torch.uint16 else "cl_icrf_energy_partial"
    check(getattr(lib, name)(C.byref(prob), _ptr(tables), _ptr(dn.contiguous()), _ptr(sd), t, n_px, _ptr(acc),
                             _ptr(ws), ws_bytes, _stream()), name)
    return acc


@torch.library.custom_op("camera_linearity::icrf_energy_finalize", mutates_args=(), device_types="cuda")
def _op_icrf_energy_finalize(pair_acc: Tensor, valid: Tensor, n_exposures: int) -> Tensor:
    """cl_icrf_energy_finalize: nanmean over the pairs of num / den, gated or NaN -> +inf."""
    _require_cuda(pair_acc, valid)
    lib = _lib.load()
    s_ = int(pair_acc.shape[0])
    prob = _icrf_problem(s_, 1, 2, True, 0, 1, n_exposures, False)
    energy = torch.empty(s_, dtype=torch.float64, device=pair_acc.device)
    check(lib.cl_icrf_energy_finalize(C.byref(prob), _ptr(_f64c(pair_acc)), _ptr(valid.contiguous()), _ptr(energy),
                                      _stream()), "cl_icrf_energy_finalize")
    return energy


@torch.library.custom_op("camera_linearity::pair_statistics", mutates_args=(), device_types="cuda")
def _op_pair_statistics(x_val: Tensor, x_std: Optional[Tensor], y_val: Tensor, y_std: Optional[Tensor],
                        multiplier: float, lower: List[float], upper: List[float]) -> Tensor:
    """cl_pair_statistics; empty ``lower`` / ``upper`` = no thresholds."""
    return pair_statistics(x_val, x_std, y_val, y_std, multiplier, list(lower) if lower else None,
                           list(upper) if upper else None)


@torch.library.custom_op("camera_linearity::quantize_8bit", mutates_args=(), device_types="cuda")
def _op_quantize_8bit(val: Tensor, max_dn: float) -> List[Tensor]:
    out, mx = quantize_8bit(val, max_dn, return_max=True)
    return [out, mx]


@torch.library.custom_op("camera_linearity::noise_profiles", mutates_args=(), device_types="cuda")
def _op_noise_profiles(frames: Tensor, mean_u8: Tensor) -> Tensor:
    return noise_profiles(frames, mean_u8)


@torch.library.custom_op("camera_linearity::measurand_binary", mutates_args=(), device_types="cuda")
def _op_measurand_binary(op: str, x_val: Tensor, x_std: Optional[Tensor], y_val: Tensor,
                         y_std: Optional[Tensor]) -> List[Tensor]:
    """op in add / sub / mul / div / pow; returns [val] or [val, std]."""
    v, s_ = measurand_binary(op, x_val, x_std, y_val, y_std)
    return [v] if s_ is None else [v, s_]
