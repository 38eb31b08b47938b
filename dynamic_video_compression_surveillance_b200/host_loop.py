"""Host side of the per-video pipelines: decode -> pinned chunk -> GPU loop -> encode, plus the reporting the
reference's GUI and performance_analysis.py depend on (file names, ``execution_times.txt`` layout, log lines).

Design (not the reference's): a decode thread fills pinned batch buffers from cv2.VideoCapture, the GPU loop runs
per batch through ``FramePipeline.process_host`` (upload / kernels / download double-buffered inside the library),
an encode thread feeds the two VideoWriters.  What stays on the host is what SURVEY.md section 8 leaves
there: codecs, the first frame's resize + heavy blur (frame_differencing.py:74,77; once per stream) and, unless the
caller asks for the GPU (``flow_masks_gpu``), Farneback flow (motion_compression_opt.py:72-82).
"""
from __future__ import annotations

import logging
import os
import time
from dataclasses import dataclass, field

import cv2
import numpy as np
import torch

from . import pipeline as P

FOURCC = "mp4v"                                              # frame_differencing.py:62, motion_compression_opt.py:49
FD_OVERLAY_NAME = "dilated_motion_mask_video.mp4"            # frame_differencing.py:52 (performance_analysis.py:146)
FD_COMPRESSED_NAME = "compressed_final_video.mp4"            # frame_differencing.py:53 (performance_analysis.py:147)
TIMES_NAME = "execution_times.txt"                           # parsed by performance_analysis.py:9-113


def video_stem(path: str) -> str:
    return os.path.splitext(os.path.basename(path))[0]


@dataclass
class StageTiming:
    title: str
    frames: int = 0
    total_s: float = 0.0
    avg_s: float = 0.0

    def lines(self):
        return [f"{self.title}:\n", f"  Frames processed: {self.frames}\n", f"  Total time: {self.total_s:.2f} seconds\n",
                f"  Average time per frame: {self.avg_s:.4f} seconds\n\n"]


def write_execution_times(path: str, stages: list[StageTiming], total_s: float) -> None:
    """The text layout performance_analysis.py parses (frame_differencing.py:152-157;
    motion_compression_opt.py:235-244)."""
    with open(path, "w") as f:
        for st in stages:
            f.writelines(st.lines())
        f.write(f"Total video processing time: {total_s:.2f} seconds\n")


@dataclass
class FdRun:
    frames: int = 0
    per_frame_s: list = field(default_factory=list)
    counters: dict = field(default_factory=dict)


def run_fd_stream(cap, first_frame, sinks, size_wh, params: dict, max_batch: int, device, progress_callback,
                  threaded: bool = True) -> FdRun:
    """The loop of frame_differencing.py:73-138 for one opened capture.  ``sinks`` = (overlay writer, compressed
    writer).  Raises on failure; the caller owns the reference's swallow-and-log policy.

    Three stages run concurrently over a small pool of pinned buffer sets: a decode thread (cap.read -> pinned input
    batch), this thread (GPU loop on the batch), an encode thread (the two VideoWriters).  cv2 releases the GIL in its
    codecs, so decode, GPU and encode overlap; output order and the 50-frame progress cadence are unchanged."""
    import queue
    import threading

    w, h = size_wh
    run = FdRun()
    n_sets = 3 if threaded else 1
    shape = (max_batch, h, w, 3)
    src_w, src_h = first_frame.shape[1], first_frame.shape[0]      # scale_factor != 1: frames are uploaded as decoded and
    in_shape = (max_batch, src_h, src_w, 3)                          # resized on the GPU (frame_differencing.py:91)
    sets = [dict(inp=P.pinned_empty(in_shape), ov=P.pinned_empty(shape), cp=P.pinned_empty(shape)) for _ in range(n_sets)]
    for st in sets:
        st["inp_v"], st["ov_v"], st["cp_v"] = st["inp"].numpy(), st["ov"].numpy(), st["cp"].numpy()
    free_q, ready_q = queue.Queue(), queue.Queue(maxsize=n_sets)
    enc_q = (queue.Queue(maxsize=n_sets), queue.Queue(maxsize=n_sets))     # one encode thread per VideoWriter
    lock = threading.Lock()
    for st in sets:
        free_q.put(st)
    errors = []
    stop = threading.Event()

    def fill(st) -> int:
        n = 0
        while n < max_batch:
            ok, frame = cap.read()
            if not ok:
                break
            st["inp_v"][n] = frame
            n += 1
        return n

    def drain(st, n, t0):
        for i in range(n):
            sinks[0].write(st["ov_v"][i])
            sinks[1].write(st["cp_v"][i])
            run.frames += 1
            if progress_callback is not None and run.frames % 50 == 0:      # frame_differencing.py:137-138
                progress_callback(run.frames)
        run.per_frame_s.extend([(time.time() - t0) / n] * n)

    def decoder():
        try:
            while not stop.is_set():
                st = free_q.get()
                if st is None:
                    break
                t0 = time.time()
                n = fill(st)
                ready_q.put((st, n, t0))
                if n < max_batch:
                    break
        except Exception as e:                                   # surfaced by the main thread
            errors.append(e)
            ready_q.put((None, 0, 0.0))

    def encoder(k):
        """Encode thread of sink k (0: overlay video, 1: compressed video).  The thread that finishes a buffer set
        last accounts the frames (count, per-frame time, progress callback) and hands the set back to the decoder."""
        try:
            while True:
                item = enc_q[k].get()
                if item is None:
                    break
                st, n, t0 = item
                view = st["ov_v"] if k == 0 else st["cp_v"]
                for i in range(n):
                    sinks[k].write(view[i])
                with lock:
                    st["pending"] -= 1
                    last = st["pending"] == 0
                if last:
                    for _ in range(n):
                        run.frames += 1
                        if progress_callback is not None and run.frames % 50 == 0:      # frame_differencing.py:137-138
                            progress_callback(run.frames)
                    run.per_frame_s.extend([(time.time() - t0) / n] * n)
                    free_q.put(st)
        except Exception as e:
            errors.append(e)
            stop.set()
            while enc_q[k].get() is not None:                    # keep the pipeline from blocking
                pass

    with P.FramePipeline(w, h, "fd", max_batch=max_batch, device=device, src_size=(src_w, src_h), **params) as pipe:
        pipe.begin_stream_frames(first_frame)     # resize + gray + (25, 25) sigma-30 blur on the GPU (frame_differencing.py:74-77)
        if not threaded:
            st = sets[0]
            while True:
                t0 = time.time()
                n = fill(st)
                if n == 0:
                    break
                pipe.process_host(st["inp"][:n], st["ov"][:n], st["cp"][:n])
                drain(st, n, t0)
        else:
            td = threading.Thread(target=decoder, daemon=True)
            tes = [threading.Thread(target=encoder, args=(k,), daemon=True) for k in (0, 1)]
            td.start()
            for t in tes:
                t.start()
            try:
                while True:
                    st, n, t0 = ready_q.get()
                    if st is None or n == 0 or errors:
                        break
                    pipe.process_host(st["inp"][:n], st["ov"][:n], st["cp"][:n])
                    st["pending"] = 2
                    for q in enc_q:
                        q.put((st, n, t0))
                    if n < max_batch:
                        break
            finally:
                stop.set()
                for q in enc_q:
                    q.put(None)
                free_q.put(None)
                for t in tes:
                    t.join()
                td.join(timeout=5)
            if errors:
                raise errors[0]
        run.counters = pipe.counters()
    return run


def smooth_masks_gpu(raw_masks: list, history: list, window_size: int, alpha_fraction: float, morph_kernel: int):
    """Window vote (motion_compression_opt.py:84-86) + close/open (:89-90) for a chunk of raw 0/255 masks.
    ``history`` = raw masks of the stream before this chunk (all of them while the stream is shorter than the
    window, else the last window_size-1), so the vote sees exactly the reference's deque."""
    stack = torch.from_numpy(np.stack(history + raw_masks)).cuda()
    voted = P.temporal_ring(stack, window_size, alpha_fraction)[len(history):].contiguous()
    closed = P.morph(voted, "close", morph_kernel, "ellipse")
    return P.morph(closed, "open", morph_kernel, "ellipse").cpu().numpy()


def smooth_rect_masks_gpu(raw_masks: list, history: list, window_size: int, alpha_fraction: float, morph_kernel: int):
    """smooth_masks_gpu followed by contours -> bounding rectangles (motion_compression_opt.py:93-97), all on the GPU:
    the chunk's mask.mp4 frames."""
    stack = torch.from_numpy(np.stack(history + raw_masks)).cuda()
    voted = P.temporal_ring(stack, window_size, alpha_fraction)[len(history):].contiguous()
    closed = P.morph(voted, "close", morph_kernel, "ellipse")
    return P.mask_rectangles(P.morph(closed, "open", morph_kernel, "ellipse")).cpu().numpy()


def first_gray_gpu(frame: np.ndarray) -> torch.Tensor:
    """cv2.cvtColor(frame, BGR2GRAY) of one host frame on the GPU (motion_compression_opt.py:60), left there."""
    return P.bgr2gray(torch.from_numpy(np.ascontiguousarray(frame))[None].cuda())[0]


def flow_masks_gpu(frames: list, prev_gray, flow_threshold: float = 0.5, farneback: tuple = (0.3, 2, 9, 2, 5, 1.1, 0)):
    """Raw flow masks of a chunk of BGR frames (motion_compression_opt.py:71-83) on the GPU: upload, BGR2GRAY, prepend
    the carried gray of the frame before the chunk, Farneback + magnitude + threshold.  ``prev_gray`` is that gray, a
    host array or a CUDA tensor [H,W]; ``farneback`` = (pyr_scale, levels, winsize, iterations, poly_n, poly_sigma,
    flags).  Returns (masks [N,H,W] uint8 host array, the last gray as a CUDA tensor to pass with the next chunk)."""
    prev = prev_gray if isinstance(prev_gray, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(prev_gray))
    prev = prev.cuda()
    if not frames:
        return np.empty((0,) + tuple(prev.shape), np.uint8), prev
    grays = P.bgr2gray(torch.from_numpy(np.stack(frames)).cuda())
    masks = P.flow_masks(torch.cat([prev[None], grays]), flow_threshold, *farneback)
    return masks.cpu().numpy(), grays[-1].clone()


def degrade_mco_gpu(frames: list, masks: list) -> np.ndarray:
    """compress_with_motion's arithmetic (motion_compression_opt.py:152-183) for a chunk."""
    comp, _ = P.degrade_blend(torch.from_numpy(np.stack(frames)).cuda(), torch.from_numpy(np.stack(masks)).cuda(),
                              8, 100, "mco", want_overlay=False)
    return comp.cpu().numpy()


def rectangles_from_mask(mask: np.ndarray) -> np.ndarray:
    """contours -> bounding rectangles (motion_compression_opt.py:93-97) on one host mask through the GPU stage op."""
    return P.mask_rectangles(torch.from_numpy(np.ascontiguousarray(mask))[None].cuda())[0].cpu().numpy()


def _rectangles_from_mask_cv2(mask: np.ndarray) -> np.ndarray:
    """The reference's own lines, kept for comparison in tools/ only."""
    out = np.zeros_like(mask)
    contours, _ = cv2.findContours(mask, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    for c in contours:
        x, y, w, h = cv2.boundingRect(c)
        cv2.rectangle(out, (x, y), (x + w, y + h), 255, -1)
    return out


def write_gpu_statistics(out_dir: str, counters: dict) -> str:
    """The in-loop statistics north_star asks for, next to execution_times.txt (an extra file: the reference's
    performance_analysis.py ignores it; its own compression percentage is derived from file sizes, perf:195-204).
    motion_pixel_percent = share of pixels painted in the overlay (acc > 127), static_block_percent = share of blocks degraded."""
    import json
    c = dict(counters)
    px, bl = max(1, int(c.get("pixels", 0))), max(1, int(c.get("blocks", 0)))
    c["motion_pixel_percent"] = 100.0 * int(c.get("motion_pixels", 0)) / px
    c["static_block_percent"] = 100.0 * int(c.get("static_blocks", 0)) / bl
    path = os.path.join(out_dir, "gpu_statistics.json")
    with open(path, "w") as f:
        json.dump(c, f, indent=1)
    return path


def attach_file_log(output_dir: str) -> str:
    """Add a processing.log FileHandler to the root logger unless one for that file is already attached
    (motion_compression_opt.py:8-27 behaviour)."""
    path = os.path.join(output_dir, "processing.log")
    root = logging.getLogger()
    if not any(isinstance(h, logging.FileHandler) and h.baseFilename == os.path.abspath(path) for h in root.handlers):
        fh = logging.FileHandler(path, mode="w")
        fh.setFormatter(logging.Formatter("%(asctime)s - %(levelname)s - %(message)s"))
        root.addHandler(fh)
    root.setLevel(logging.INFO)
    return path
