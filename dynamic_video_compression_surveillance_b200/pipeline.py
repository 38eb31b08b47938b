"""Python host objects over the C ABI (include/dvc_b200.h).

``FramePipeline`` owns the per-stream state the reference keeps in local variables of
``filter_and_dilate_movements`` (prev_gray, accumulated_mask: frame_differencing.py:75-81) or of
``temporal_smoothing_flow`` (mask_queue: motion_compression_opt.py:61) and runs the loop body
(frame_differencing.py:85-133) for batches of frames on the GPU.  torch is used for device memory,
pinned host memory and streams only; every arithmetic step is a kernel behind the ABI.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import (DVC_DEGRADE_FD, DVC_DEGRADE_MCO, DVC_MODE_FD, DVC_MODE_FLOW, DVC_MODE_WINDOW, DVC_SHAPE_ELLIPSE,
                   DVC_SHAPE_RECT, DvcConfig, DvcCounters, check)

_MODES = {"fd": DVC_MODE_FD, "window": DVC_MODE_WINDOW, "flow": DVC_MODE_FLOW}
CALL_SITE_FARNEBACK = (0.3, 2, 9, 2, 5, 1.1, 0)      # motion_compression_opt.py:72-81
_SHAPES = {"rect": DVC_SHAPE_RECT, "ellipse": DVC_SHAPE_ELLIPSE}
_MORPH_OPS = {"erode": 0, "dilate": 1, "open": 2, "close": 3}


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("dynamic_video_compression_surveillance_b200 needs a CUDA device; there is no CPU fallback")


def _stream_ptr(stream) -> int:
    if stream is None:
        stream = torch.cuda.current_stream()
    return int(stream.cuda_stream)


def _dev_u8(t: torch.Tensor, name: str) -> torch.Tensor:
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.uint8 and t.is_contiguous()):
        raise TypeError(f"{name} must be a contiguous uint8 CUDA tensor")
    return t


def pinned_empty(shape) -> torch.Tensor:
    """Pinned host buffer (what cudaMemcpyAsync needs to overlap); ``.numpy()`` views it."""
    return torch.empty(tuple(shape), dtype=torch.uint8, pin_memory=True)


class FramePipeline:
    """Per-stream state + the loop body.  Keyword names and defaults are the reference's
    (frame_differencing.py:21-30; motion_compression_opt.py:29-31).

    ``n_streams=S > 1`` makes the object a lock-step group of S independent camera streams (the reference processes its
    files one after another, windows.py:142-160; BASELINE config 4) whose kernels share every launch: all frame / output
    arrays gain a leading stream axis ([S, T, H, W, 3]), ``begin_stream`` takes [S, H, W] planes, and every call
    advances each stream by T frames.  Results per stream equal those of S separate pipelines.

    ``mode="flow"`` runs temporal_smoothing_flow with compress_with_motion's arithmetic (motion_compression_opt.py:65-101,
    152-183; BASELINE config 5): ``mask`` receives the rectangle mask (the mask.mp4 frame), ``compressed`` the degraded frame,
    and there is no overlay (the reference's overlay.mp4 is the unmodified frame).  ``flow_threshold`` and ``farneback``
    (pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags) are the call's Farneback arguments; block_size
    defaults to 8 and kernel_size to 0 in this mode (other values raise the library's error)."""

    def __init__(self, width: int, height: int, mode: str = "fd", *, block_size: int | None = None,
                 motion_threshold: float = 0.5, min_area: float = 500, kernel_size: int | None = None,
                 release_factor: float = 0.5, quantization_level: float = 100, window_size: int = 30,
                 alpha_fraction: float = 0.2, morph_kernel: int = 2, morph_shape: str = "ellipse", max_batch: int = 16,
                 device: int | None = None, src_size: tuple | None = None, n_streams: int = 1, flow_threshold: float = 0.5,
                 farneback: tuple = CALL_SITE_FARNEBACK):
        _require_cuda()
        flow = mode == "flow"
        if block_size is None:
            block_size = 8 if flow else 4
        if kernel_size is None:
            kernel_size = 0 if flow else 7
        self._lib = _lib.load()
        self.width, self.height, self.mode = int(width), int(height), mode
        self.device = torch.cuda.current_device() if device is None else int(device)
        cfg = DvcConfig()
        self._lib.dvc_default_config(C.byref(cfg))
        cfg.width, cfg.height, cfg.mode = self.width, self.height, _MODES[mode]
        cfg.block_size, cfg.motion_threshold, cfg.min_area = int(block_size), float(motion_threshold), float(min_area)
        cfg.kernel_size, cfg.release_factor = int(kernel_size), float(release_factor)
        cfg.quantization_level = float(quantization_level)
        cfg.window_size, cfg.alpha_fraction = int(window_size), float(alpha_fraction)
        cfg.morph_kernel, cfg.morph_shape = int(morph_kernel), _SHAPES[morph_shape]
        cfg.max_batch, cfg.device = int(max_batch), self.device
        # frames given to process_host at another size (width, height): the library resizes them as cv2.resize does
        self.src_width, self.src_height = (int(src_size[0]), int(src_size[1])) if src_size else (self.width, self.height)
        if (self.src_width, self.src_height) != (self.width, self.height):
            cfg.src_width, cfg.src_height = self.src_width, self.src_height
        self.n_streams = max(1, int(n_streams))
        cfg.n_streams = self.n_streams
        self.cfg = cfg
        self.max_batch = int(max_batch)
        self._h = C.c_void_p()
        check(self._lib.dvc_create(C.byref(cfg), C.byref(self._h)))
        if flow:
            self.flow_threshold, self.farneback = float(flow_threshold), tuple(farneback)
            if (self.flow_threshold, self.farneback) != (0.5, CALL_SITE_FARNEBACK):
                self.set_flow_params(self.flow_threshold, self.farneback)

    def set_flow_params(self, flow_threshold: float = 0.5, farneback: tuple = CALL_SITE_FARNEBACK):
        """Flow mode: the threshold and the Farneback arguments (pyr_scale, levels, winsize, iterations, poly_n, poly_sigma,
        flags) of motion_compression_opt.py:72-83."""
        self._check(self._lib.dvc_set_flow_params(self._h, float(flow_threshold), *_flow_args(*farneback)))
        self.flow_threshold, self.farneback = float(flow_threshold), tuple(farneback)

    @property
    def flow_group(self) -> int:
        """Flow mode: Farneback pairs per launch group, the library's rule (DESIGN.md section 6c): every pair of a batch,
        n_streams * max_batch, as long as the group's scratch of 116 bytes per pixel and pair stays within 4 GiB."""
        per_pair = self.width * self.height * 116
        return max(1, min(self.n_streams * self.max_batch, (4 << 30) // per_pair, 4096))

    # -- lifecycle ----------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.dvc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc):
        check(rc, self._h)

    # -- state --------------------------------------------------------------------------------------
    def begin_stream(self, prev_gray: np.ndarray):
        """Seed prev_gray (frame_differencing.py:75-77 / motion_compression_opt.py:60) and clear the mask state."""
        g = np.ascontiguousarray(prev_gray, dtype=np.uint8)
        want = (self.height, self.width) if self.n_streams == 1 else (self.n_streams, self.height, self.width)
        if g.shape != want and g.shape != (1,) + want:
            raise ValueError(f"prev_gray must be {list(want)}")
        self._check(self._lib.dvc_begin_stream(self._h, g.ctypes.data))

    def begin_stream_frames(self, first_frames: np.ndarray):
        """Seed the stream(s) from the first decoded frame(s) [src_h, src_w, 3] ([S, ...] for a group): resize, BGR2GRAY and (fd
        mode) the (25, 25), sigma 30 blur run on the GPU (frame_differencing.py:74-77)."""
        f = np.ascontiguousarray(first_frames, dtype=np.uint8)
        want = (self.src_height, self.src_width, 3)
        want = want if self.n_streams == 1 else (self.n_streams,) + want
        if f.shape != want and f.shape != (1,) + want:
            raise ValueError(f"first_frames must be {list(want)}")
        self._check(self._lib.dvc_begin_stream_frames(self._h, f.ctypes.data))

    def get_state(self) -> bytes:
        n = self._lib.dvc_state_bytes(self._h)
        buf = np.empty(n, np.uint8)
        self._check(self._lib.dvc_get_state(self._h, buf.ctypes.data, n))
        return buf.tobytes()

    def set_state(self, blob: bytes):
        buf = np.frombuffer(blob, np.uint8)
        self._check(self._lib.dvc_set_state(self._h, buf.ctypes.data, buf.size))

    def counters(self) -> dict:
        c = DvcCounters()
        self._check(self._lib.dvc_get_counters(self._h, C.byref(c)))
        return {k: int(getattr(c, k)) for k, _ in DvcCounters._fields_}

    def profile(self, on: bool):
        """Record CUDA events around every kernel group of the loop (read with ``profile_read``)."""
        self._check(self._lib.dvc_profile_enable(self._h, int(bool(on))))

    def profile_read(self) -> dict:
        """{group: (milliseconds, launches)} since the last read; synchronises."""
        n = len(_lib.PROF_KERNELS)
        ms = (C.c_double * n)()
        ln = (C.c_int64 * n)()
        self._check(self._lib.dvc_profile_read(self._h, ms, ln, n))
        return {k: (float(ms[i]), int(ln[i])) for i, k in enumerate(_lib.PROF_KERNELS)}

    def launch_count(self) -> int:
        return int(self._lib.dvc_launch_count(self._h))

    def reset_counters(self):
        self._check(self._lib.dvc_reset_counters(self._h))

    # -- the loop body ------------------------------------------------------------------------------
    def process_device(self, frames: torch.Tensor, overlay: torch.Tensor | None = None,
                       compressed: torch.Tensor | None = None, mask: torch.Tensor | None = None, stream=None):
        """frames [T,H,W,3] uint8 on the GPU ([S,T,H,W,3] for a stream group), T <= max_batch.  Outputs are written
        into the given tensors (None = not produced).  Asynchronous on the current (or given) torch stream."""
        _dev_u8(frames, "frames")
        lead = () if self.n_streams == 1 else (self.n_streams,)
        T = frames.shape[len(lead)]
        if tuple(frames.shape) != lead + (T, self.height, self.width, 3):
            raise ValueError("frames must be [T, H, W, 3]" if not lead else f"frames must be [{self.n_streams}, T, H, W, 3]")
        for name, t, shp in (("overlay", overlay, frames.shape), ("compressed", compressed, frames.shape),
                             ("mask", mask, frames.shape[:-1])):
            if t is not None:
                _dev_u8(t, name)
                if tuple(t.shape) != tuple(shp):
                    raise ValueError(f"{name} has the wrong shape")
        ptr = lambda t: None if t is None else t.data_ptr()
        self._check(self._lib.dvc_process_batch(self._h, frames.data_ptr(), T, ptr(overlay), ptr(compressed), ptr(mask),
                                                _stream_ptr(stream)))

    def set_overlap(self, on: bool):
        """Pipeline consecutive process_device batches on two internal streams (mask kernels of batch c+1 overlap
        the degrade kernel of batch c).  Buffers must stay untouched until ``flush``."""
        self._check(self._lib.dvc_set_overlap(self._h, int(bool(on))))

    def flush(self, stream=None):
        """Make the current (or given) torch stream wait for every batch issued so far."""
        self._check(self._lib.dvc_flush(self._h, _stream_ptr(stream)))

    def process_host(self, frames, overlay=None, compressed=None, mask=None):
        """frames [N,H,W,3] uint8 HOST array (numpy or CPU torch tensor, pinned for full speed); outputs are host
        arrays of matching shape or None.  Upload, loop and download are pipelined in chunks of max_batch inside
        the library; returns when the outputs are complete."""
        def host_ptr(a, shape, name):
            if a is None:
                return None
            if isinstance(a, torch.Tensor):
                if a.is_cuda or a.dtype != torch.uint8 or not a.is_contiguous():
                    raise TypeError(f"{name} must be a contiguous uint8 CPU tensor")
                if tuple(a.shape) != tuple(shape):
                    raise ValueError(f"{name} has the wrong shape")
                return a.data_ptr()
            if not (isinstance(a, np.ndarray) and a.dtype == np.uint8 and a.flags.c_contiguous):
                raise TypeError(f"{name} must be a C-contiguous uint8 array")
            if tuple(a.shape) != tuple(shape):
                raise ValueError(f"{name} has the wrong shape")
            return a.ctypes.data
        lead = () if self.n_streams == 1 else (self.n_streams,)       # stream groups: [S, N, H, W, 3], stream-major
        n = int(frames.shape[len(lead)])
        fshape = lead + (n, self.height, self.width, 3)
        self._check(self._lib.dvc_process_host(self._h, host_ptr(frames, lead + (n, self.src_height, self.src_width, 3), "frames"), n,
                                               host_ptr(overlay, fshape, "overlay"),
                                               host_ptr(compressed, fshape, "compressed"),
                                               host_ptr(mask, fshape[:-1], "mask")))


# ---------------------------------------------------------------------------------------------------
# stage-level ops on CUDA tensors (one per cv2 call of the loop; used by parity tests and available to
# callers that want a single op)
# ---------------------------------------------------------------------------------------------------

def _lib_call(name, *args):
    _require_cuda()
    check(getattr(_lib.load(), name)(*args))


def bgr2gray(bgr: torch.Tensor) -> torch.Tensor:
    """cv2.cvtColor(BGR2GRAY) for [N,H,W,3] (frame_differencing.py:75,92)."""
    _dev_u8(bgr, "bgr")
    n, h, w, _ = bgr.shape
    out = torch.empty((n, h, w), dtype=torch.uint8, device=bgr.device)
    _lib_call("dvc_bgr2gray_u8", bgr.data_ptr(), out.data_ptr(), n, h, w, _stream_ptr(None))
    return out


def gray_absdiff_thresh(bgr: torch.Tensor, prev_gray: torch.Tensor, motion_threshold: float = 0.5, blur5: bool = True):
    """frame_differencing.py:92-97 for N consecutive frames -> (gray [N,H,W], mask [N,H,W])."""
    _dev_u8(bgr, "bgr"); _dev_u8(prev_gray, "prev_gray")
    n, h, w, _ = bgr.shape
    gray = torch.empty((n, h, w), dtype=torch.uint8, device=bgr.device)
    mask = torch.empty((n, h, w), dtype=torch.uint8, device=bgr.device)
    _lib_call("dvc_gray_absdiff_thresh_u8", bgr.data_ptr(), prev_gray.data_ptr(), gray.data_ptr(), mask.data_ptr(), n, h, w,
              float(motion_threshold), int(bool(blur5)), _stream_ptr(None))
    return gray, mask


def temporal_ring(masks: torch.Tensor, window_size: int = 30, alpha_fraction: float = 0.2) -> torch.Tensor:
    """motion_compression_opt.py:61,84-86 for N consecutive masks starting from an empty window."""
    _dev_u8(masks, "masks")
    n, h, w = masks.shape
    out = torch.empty_like(masks)
    _lib_call("dvc_temporal_ring_u8", masks.data_ptr(), out.data_ptr(), n, h, w, int(window_size), float(alpha_fraction),
              _stream_ptr(None))
    return out


def temporal_ema(acc: torch.Tensor, dilated: torch.Tensor, release_factor: float = 0.5) -> torch.Tensor:
    """frame_differencing.py:107 for N consecutive dilated masks; ``acc`` [H,W] is updated in place, the
    accumulator after every frame is returned [N,H,W]."""
    _dev_u8(acc, "acc"); _dev_u8(dilated, "dilated")
    n, h, w = dilated.shape
    out = torch.empty_like(dilated)
    _lib_call("dvc_temporal_ema_u8", acc.data_ptr(), dilated.data_ptr(), out.data_ptr(), n, h, w, float(release_factor),
              _stream_ptr(None))
    return out


def morph(masks: torch.Tensor, op: str, k: int, shape: str = "rect") -> torch.Tensor:
    """cv2.erode / dilate / morphologyEx(OPEN|CLOSE) on binary masks [N,H,W] (frame_differencing.py:106;
    motion_compression_opt.py:89-90)."""
    _dev_u8(masks, "masks")
    n, h, w = masks.shape
    out = torch.empty_like(masks)
    _lib_call("dvc_morph_u8", masks.data_ptr(), out.data_ptr(), n, h, w, _MORPH_OPS[op], _SHAPES[shape], int(k),
              _stream_ptr(None))
    return out


def contour_filter(masks: torch.Tensor, min_area: float = 500) -> torch.Tensor:
    """frame_differencing.py:100-104 on [N,H,W] masks."""
    _dev_u8(masks, "masks")
    n, h, w = masks.shape
    out = torch.empty_like(masks)
    _lib_call("dvc_contour_filter_u8", masks.data_ptr(), out.data_ptr(), n, h, w, float(min_area), _stream_ptr(None))
    return out


def resize_linear(images: torch.Tensor, dsize_wh) -> torch.Tensor:
    """cv2.resize(img, (w, h)) (INTER_LINEAR, uint8) on [N,H,W,3] or [N,H,W] images (frame_differencing.py:74,91)."""
    _dev_u8(images, "images")
    n, h, w = images.shape[:3]
    cn = 1 if images.dim() == 3 else int(images.shape[3])
    dw, dh = int(dsize_wh[0]), int(dsize_wh[1])
    out = torch.empty((n, dh, dw) if images.dim() == 3 else (n, dh, dw, cn), dtype=torch.uint8, device=images.device)
    _lib_call("dvc_resize_linear_u8", images.data_ptr(), out.data_ptr(), n, h, w, dh, dw, cn, _stream_ptr(None))
    return out


def mask_rectangles(masks: torch.Tensor) -> torch.Tensor:
    """motion_compression_opt.py:93-97 on [N,H,W] masks: every 8-connected component becomes its bounding
    rectangle, drawn the way cv2.rectangle((x, y), (x + w, y + h), 255, -1) draws it (both corners included)."""
    _dev_u8(masks, "masks")
    n, h, w = masks.shape
    out = torch.empty_like(masks)
    _lib_call("dvc_mask_rectangles_u8", masks.data_ptr(), out.data_ptr(), n, h, w, _stream_ptr(None))
    return out


def degrade_blend(bgr: torch.Tensor, mask: torch.Tensor, block_size: int = 4, quantization_level: float = 100,
                  flavour: str = "fd", want_overlay: bool = True, counters: torch.Tensor | None = None):
    """frame_differencing.py:110-111,115-130 (flavour 'fd') or motion_compression_opt.py:152-183 ('mco') on
    [N,H,W,3] frames and [N,H,W] uint8 masks -> (compressed, overlay or None)."""
    _dev_u8(bgr, "bgr"); _dev_u8(mask, "mask")
    n, h, w, _ = bgr.shape
    comp = torch.empty_like(bgr)
    ov = torch.empty_like(bgr) if want_overlay else None
    _lib_call("dvc_degrade_blend_u8", bgr.data_ptr(), mask.data_ptr(), comp.data_ptr(), None if ov is None else ov.data_ptr(),
              n, h, w, int(block_size), float(quantization_level), DVC_DEGRADE_FD if flavour == "fd" else DVC_DEGRADE_MCO,
              None if counters is None else counters.data_ptr(), _stream_ptr(None))
    return comp, ov


def dct_blocks(blocks: torch.Tensor, inverse: bool = False) -> torch.Tensor:
    """cv2.dct / cv2.idct (frame_differencing.py:122,124; motion_compression_opt.py:165,167) of a float32 CUDA stack
    [N, bh, bw] with bh, bw in 1..8, bit for bit."""
    if not (blocks.is_cuda and blocks.dtype == torch.float32 and blocks.dim() == 3 and blocks.is_contiguous()):
        raise ValueError("blocks: contiguous float32 CUDA tensor [N, bh, bw]")
    out = torch.empty_like(blocks)
    _lib_call("dvc_dct_blocks_f32", blocks.data_ptr(), out.data_ptr(), blocks.shape[0], blocks.shape[1], blocks.shape[2],
              1 if inverse else 0, _stream_ptr(None))
    return out


def gaussian_blur(planes: torch.Tensor, ksize: int, sigma: float) -> torch.Tensor:
    """cv2.GaussianBlur(img, (ksize, ksize), sigma) on uint8 planes [N,H,W] (frame_differencing.py:77,93)."""
    _dev_u8(planes, "planes")
    n, h, w = planes.shape
    out = torch.empty_like(planes)
    _lib_call("dvc_gaussian_blur_u8", planes.data_ptr(), out.data_ptr(), n, h, w, int(ksize), float(sigma), _stream_ptr(None))
    return out


def _flow_args(pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags):
    return (float(pyr_scale), int(levels), int(winsize), int(iterations), int(poly_n), float(poly_sigma), int(flags))


def farneback_flow(prev: torch.Tensor, next: torch.Tensor, pyr_scale: float = 0.3, levels: int = 2, winsize: int = 9,
                   iterations: int = 2, poly_n: int = 5, poly_sigma: float = 1.1, flags: int = 0) -> torch.Tensor:
    """cv2.calcOpticalFlowFarneback(prev, next, None, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags)
    (motion_compression_opt.py:72-81) for uint8 planes [H,W] or pairs [N,H,W] -> float32 flow [H,W,2] or [N,H,W,2].
    Defaults are the call site's.  poly_n other than 5 / 7 and flags other than 0 raise NotImplementedError."""
    _dev_u8(prev, "prev"); _dev_u8(next, "next")
    if prev.shape != next.shape or prev.dim() not in (2, 3):
        raise ValueError("prev and next must be [H, W] or [N, H, W] of the same shape")
    p, q = (prev[None], next[None]) if prev.dim() == 2 else (prev, next)
    n, h, w = p.shape
    out = torch.empty((n, h, w, 2), dtype=torch.float32, device=prev.device)
    _lib_call("dvc_farneback_flow_f32", p.data_ptr(), q.data_ptr(), out.data_ptr(), n, h, w,
              *_flow_args(pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags), _stream_ptr(None))
    return out[0] if prev.dim() == 2 else out


def flow_masks(grays: torch.Tensor, flow_threshold: float = 0.5, pyr_scale: float = 0.3, levels: int = 2, winsize: int = 9,
               iterations: int = 2, poly_n: int = 5, poly_sigma: float = 1.1, flags: int = 0) -> torch.Tensor:
    """The raw masks of temporal_smoothing_flow (motion_compression_opt.py:72-83) for a uint8 gray sequence [N+1,H,W]:
    [N,H,W], mask i = 255 where the float32 flow magnitude from frame i to frame i + 1 exceeds float32(flow_threshold)."""
    _dev_u8(grays, "grays")
    if grays.dim() != 3 or grays.shape[0] < 1:
        raise ValueError("grays must be [N+1, H, W] with N >= 0")
    n1, h, w = grays.shape
    out = torch.empty((n1 - 1, h, w), dtype=torch.uint8, device=grays.device)
    _lib_call("dvc_flow_masks_u8", grays.data_ptr(), out.data_ptr(), n1 - 1, h, w,
              *_flow_args(pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags), float(flow_threshold),
              _stream_ptr(None))
    return out
