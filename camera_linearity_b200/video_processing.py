"""Mean / standard-error frames of videos (reference: ``modules/video_processing.py:161-274``).

``welford_algorithm`` keeps the reference's signature.  Frames are decoded on the host (OpenCV)
straight into one of two pinned staging buffers; a full buffer is copied to the device on a copy
stream while the decoder fills the other one, and folded into the running float64 (mean, M2) state
with the exact sequential Welford recurrence (``ops.welford_update``, bit-identical to NumPy) --
decode, H2D and the update overlap (SURVEY.md 8f rank 2).  When a whole stack is already resident
on the device, ``welford_stack`` uses the integer fast path (K3).
Repair R9 (SURVEY.md 8.0): ``if ICRF is not None``; the float64 mean and SEM are returned next to
the reference's uint8 outputs.  16-bit (or 12-bit-in-uint16) frames give uint16 ``mean`` / ``std`` frames (the R9
extension of DESIGN.md section 3), written as 16-bit TIFFs by ``process_video`` / ``process_directory``.
"""
from __future__ import annotations

from pathlib import Path
from typing import List, Optional, Union

import numpy as np
import torch

from . import general_functions as gf
from . import ops
from .settings import GlobalSettings as gs

CHUNK_FRAMES = 32


def welford_stack(frames, ICRF=None):
    """frames: (F, H, W, C) uint8 or uint16 tensor/array already in memory.  Returns the same dict as
    ``welford_algorithm``; ``mean`` / ``std`` have the frames' dtype.  A uint16 stack of more than
    ``ops.WELFORD_U16_MAX_FRAMES`` frames is folded with the streaming form instead (same results)."""
    dev = gs.device()
    fr = torch.as_tensor(frames).to(dev)
    icrf = None if ICRF is None else torch.as_tensor(ICRF, dtype=torch.float64, device=dev)
    if fr.dtype == torch.uint16 and fr.shape[0] > ops.WELFORD_U16_MAX_FRAMES:
        mean = torch.zeros(tuple(fr.shape[1:]), dtype=torch.float64, device=dev)
        m2 = torch.zeros_like(mean)
        ops.welford_update(fr, mean, m2, 0, icrf, gs.MAX_DN)
        sem, mean_q = ops.welford_finalize(mean, m2, int(fr.shape[0]), gs.MAX_DN, fr.dtype)
    else:
        mean, sem, mean_q = ops.welford_stack(fr, icrf, gs.MAX_DN)
    std_q = torch.round(sem).nan_to_num(0.0).to(mean_q.dtype)        # video_processing.py:215 (D13)
    return {'mean': mean_q, 'std': std_q, 'mean_f64': mean, 'sem': sem, 'count': int(fr.shape[0])}


class _ChunkStager:
    """Two pinned host buffers of CHUNK_FRAMES frames feeding ``ops.welford_update``.

    push() copies a decoded frame into the buffer being filled; a full buffer is sent to the device on
    the copy stream and consumed on the current stream, both asynchronously, so the decoder keeps
    running.  A buffer is reused only after the update that read its device copy has finished
    (``free[i]`` event).  On the CPU device (host-logic tests) the same code runs without streams.
    The buffers have the first frame's dtype (uint8 or uint16); a frame of another dtype raises instead of being
    cast (NumPy would wrap uint16 samples modulo 256 into a uint8 buffer)."""

    def __init__(self, frame_shape, dtype, dev, icrf):
        self.dev, self.icrf = dev, icrf
        self.cuda = dev.type == "cuda"
        self.np_dtype = np.dtype(dtype)
        if self.np_dtype not in (np.uint8, np.uint16):
            raise TypeError(f"frames must be uint8 or uint16, got {self.np_dtype}")
        self.dtype = torch.uint8 if self.np_dtype == np.uint8 else torch.uint16
        shape = (CHUNK_FRAMES,) + tuple(frame_shape)
        self.host = [torch.empty(shape, dtype=self.dtype, pin_memory=self.cuda) for _ in range(2)]
        self.host_np = [h.numpy() for h in self.host]
        self.device = ([torch.empty(shape, dtype=self.dtype, device=dev) for _ in range(2)] if self.cuda
                       else self.host)
        self.copy_stream = torch.cuda.Stream(dev) if self.cuda else None
        self.free = [None, None]
        self.i = self.fill = self.count = 0
        self.mean = torch.zeros(tuple(frame_shape), dtype=torch.float64, device=dev)
        self.m2 = torch.zeros_like(self.mean)

    def push(self, frame):
        if self.fill == 0 and self.free[self.i] is not None:
            self.free[self.i].synchronize()                 # the previous user of this buffer pair is done
        frame = np.asarray(frame)
        if frame.dtype != self.np_dtype:
            raise TypeError(f"a {frame.dtype} frame in a video of {self.np_dtype} frames")
        self.host_np[self.i][self.fill] = frame
        self.fill += 1
        if self.fill == CHUNK_FRAMES:
            self._flush()

    def _flush(self):
        n, i = self.fill, self.i
        if n == 0:
            return
        chunk = self.device[i][:n]
        if self.cuda:
            main = torch.cuda.current_stream(self.dev)
            with torch.cuda.stream(self.copy_stream):
                chunk.copy_(self.host[i][:n], non_blocking=True)
                copied = torch.cuda.Event()
                copied.record(self.copy_stream)
            main.wait_event(copied)
        self.count = ops.welford_update(chunk, self.mean, self.m2, self.count, self.icrf, gs.MAX_DN)
        if self.cuda:
            self.free[i] = torch.cuda.Event()
            self.free[i].record(torch.cuda.current_stream(self.dev))
        self.i ^= 1
        self.fill = 0

    def finish(self):
        self._flush()
        return self.mean, self.m2, self.count


def welford_algorithm(file_paths: Union[Path, List[Path]], ICRF=None, use_std: Optional[bool] = False,
                      frame_source=None):
    """Welford mean / std frame over all frames of one or more videos (video_processing.py:161-219).

    Returns ``{'mean': uint8 mean frame, 'std': uint8 frame or None}`` exactly like the reference,
    plus ``'mean_f64'``, ``'sem'`` (float64, un-quantised; repair R9) and ``'count'``.  For uint16 frames
    ``mean`` / ``std`` are uint16 (the R9 extension).
    ``frame_source(path)`` may replace the OpenCV frame generator (used by the tests and bench).
    """
    if not isinstance(file_paths, list):
        file_paths = [file_paths]
    source = gf.video_frame_generator if frame_source is None else frame_source
    dev = gs.device()
    icrf = None if ICRF is None else torch.as_tensor(ICRF, dtype=torch.float64, device=dev)
    stager = None
    for file_path in file_paths:
        for frame in source(file_path):
            if frame is None:
                break
            if stager is None:
                first = np.asarray(frame)
                stager = _ChunkStager(first.shape, first.dtype, dev, icrf)
            stager.push(frame)
    if stager is None:
        raise ValueError("no frames decoded")
    mean, m2, count = stager.finish()
    sem, mean_q = ops.welford_finalize(mean, m2 if use_std else None, count, gs.MAX_DN, stager.dtype)
    std_q = None
    if use_std:
        std_q = torch.round(sem).nan_to_num(0.0).to(stager.dtype)   # :214-215 literal (all zeros, D13)
    return {'mean': mean_q, 'std': std_q, 'mean_f64': mean, 'sem': sem, 'count': count}


def compute_noise_profiles(video_files: List[Path], frame_source=None):
    """Noise profiles of a camera from videos of a static scene (video_processing.py:77-106): the joint histogram
    ``profiles[mean DN, frame DN, channel]`` over every frame, against the uint8 Welford mean frame.  Returns
    ``(profiles int64 (BITS, BITS, C) tensor, mean frame uint8 tensor)``.  Frames are decoded on the host into a pinned
    chunk buffer and binned on the device (``cl_noise_profiles``); 8-bit data (the reference indexes the profile
    with the frame bytes)."""
    if not isinstance(video_files, list):
        video_files = [video_files]
    source = gf.video_frame_generator if frame_source is None else frame_source
    mean_frame = welford_algorithm(video_files, None, False, frame_source=frame_source)['mean']       # :90
    if mean_frame.dtype != torch.uint8:
        raise TypeError("noise profiles are defined for 8-bit frames only; these frames are uint16")
    dev = mean_frame.device
    hist = None
    shape = (CHUNK_FRAMES,) + tuple(mean_frame.shape)
    host = torch.empty(shape, dtype=torch.uint8, pin_memory=dev.type == "cuda")
    host_np = host.numpy()
    fill = 0

    def flush(n):
        nonlocal hist
        if n:
            hist = ops.noise_profiles(host[:n].to(dev), mean_frame, hist)   # (synchronous copy: the buffer is reused)
    for video_file in video_files:                                                                  # :92-104
        for frame in source(video_file):
            if frame is None:
                break
            host_np[fill] = frame
            fill += 1
            if fill == CHUNK_FRAMES:
                flush(fill)
                fill = 0
    flush(fill)
    if hist is None:
        raise ValueError("no frames decoded")
    return hist, mean_frame


def process_video(video_path: Path, ICRF=None, use_std: Optional[bool] = True):
    """video_processing.py:222-236."""
    import cv2 as cv
    ret = welford_algorithm(video_path, ICRF, use_std)
    for key in ('mean', 'std'):
        if ret[key] is not None:
            save_path = str(video_path.parent.joinpath(video_path.name.replace('.avi', f'.{key}.tif')))
            cv.imwrite(save_path, ret[key].cpu().numpy())


def process_directory(dir_path: Path, ICRF=None, separately: Optional[bool] = True):
    """video_processing.py:239-274."""
    import cv2 as cv
    video_files = list(dir_path.glob("*.avi"))
    if not separately:
        ret = welford_algorithm(video_files, ICRF)
        for key in ('mean', 'std'):
            if ret[key] is not None:
                cv.imwrite(str(dir_path.joinpath(f'total_{key}.tif')), ret[key].cpu().numpy())
        return
    for path in video_files:
        ret = welford_algorithm(path, ICRF)
        for key in ('mean', 'std'):
            if ret[key] is not None:
                save_dir = path.parent.joinpath(key)
                save_dir.mkdir(exist_ok=True)
                name = path.name.replace('.avi', ' STD.tif' if key == 'std' else '.tif')
                cv.imwrite(str(save_dir.joinpath(name)), ret[key].cpu().numpy())
