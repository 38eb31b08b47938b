"""Drop-in for the reference module of the same name: ``windows.py`` imports ``process_single_video_of`` from
here (windows.py:13,151).  Contracts follow motion_compression_opt.py:8-247.  GPU (C ABI): the K-frame window
vote (:84-86), close/open (:89-90), contours -> bounding rectangles (:93-97) and all of compress_with_motion's
arithmetic (:152-183).  Farneback flow + cartToPolar + threshold (:71-83) run on the host by default, as in the
reference; ``flow_device="gpu"`` moves gray conversion, flow and masks to the GPU (host_loop.flow_masks_gpu), which agrees
with cv2 about as closely as cv2's own dispatch paths agree with each other (DESIGN.md section 6).  Codecs stay on the host.
"""
import logging
import os
import sys
import time

import cv2
import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

from dynamic_video_compression_surveillance_b200 import host_loop as _hl  # noqa: E402

_CHUNK = 16
_FARNEBACK = (0.3, 2, 9, 2, 5, 1.1, 0)          # pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags (:72-81)


def setup_logging(output_dir):
    """motion_compression_opt.py:8-27: additive file handler, INFO level."""
    log_file = _hl.attach_file_log(output_dir)
    logging.getLogger().info(f"Logging configured. Log file saved in: {log_file}")


def _open_writer(path, fps, size, color=True):
    return cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*_hl.FOURCC), fps, size, isColor=color)


def temporal_smoothing_flow(video_path, output_dir, flow_threshold=0.5, alpha_fraction=0.2, window_size=30, morph_kernel=2,
                            save_name="overlay.mp4", mask_save_name="mask.mp4", flow_device="cpu"):
    """motion_compression_opt.py:29-109 -> (frames, total seconds, seconds per frame).  flow_device "cpu" (default):
    cv2 Farneback per frame on the host; "gpu": gray, flow and raw masks of each chunk on the GPU."""
    if flow_device not in ("cpu", "gpu"):
        raise ValueError(f"flow_device must be 'cpu' or 'gpu', not {flow_device!r}")
    t_start = time.time()
    cap = cv2.VideoCapture(video_path)
    if not cap.isOpened():
        logging.error(f"Error: Unable to open video file: {video_path}")
        return 0, 0, 0
    fps = cap.get(cv2.CAP_PROP_FPS)
    size = (int(cap.get(cv2.CAP_PROP_FRAME_WIDTH)), int(cap.get(cv2.CAP_PROP_FRAME_HEIGHT)))
    out_overlay = _open_writer(os.path.join(output_dir, save_name), fps, size)
    out_mask = _open_writer(os.path.join(output_dir, mask_save_name), fps, size, color=False)
    ok, frame = cap.read()
    if not ok:
        logging.error("Error: Unable to read the first frame.")
        cap.release()
        return 0, 0, 0

    on_gpu = flow_device == "gpu"
    prev_gray = _hl.first_gray_gpu(frame) if on_gpu else cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY)
    n_frames, history, exhausted = 0, [], False
    while not exhausted:
        frames, raws = [], []
        while len(frames) < _CHUNK:
            ok, frame = cap.read()
            if not ok:
                exhausted = True
                break
            if not on_gpu:
                gray = cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY)
                flow = cv2.calcOpticalFlowFarneback(prev_gray, gray, None, *_FARNEBACK)
                mag, _ = cv2.cartToPolar(flow[..., 0], flow[..., 1])
                raws.append((mag > flow_threshold).astype(np.uint8) * 255)
                prev_gray = gray
            frames.append(frame)
        if not frames:
            break
        if on_gpu:
            masks, prev_gray = _hl.flow_masks_gpu(frames, prev_gray, flow_threshold, _FARNEBACK)
            raws = list(masks)
        rects = _hl.smooth_rect_masks_gpu(raws, history, window_size, alpha_fraction, morph_kernel)
        seen = history + raws
        # while the stream is shorter than the window keep all of it (the vote's L = len(deque) must match);
        # afterwards the last window_size-1 raw masks are enough
        history = seen if n_frames + len(raws) < window_size else (seen[-(window_size - 1):] if window_size > 1 else [])
        for frame, mask in zip(frames, rects):
            n_frames += 1
            out_overlay.write(frame)
            out_mask.write(mask)
    cap.release()
    out_overlay.release()
    out_mask.release()
    total = time.time() - t_start
    avg = total / n_frames if n_frames > 0 else 0
    logging.info(f"Temporal smoothing flow completed for '{os.path.basename(video_path)}' in {total:.2f} seconds. Frames processed: {n_frames}")
    return n_frames, total, avg


def compress_with_motion(input_video, mask_video, output_dir):
    """motion_compression_opt.py:111-193 -> (frames, total seconds, seconds per frame)."""
    t_start = time.time()
    logging.info(f"Starting motion-based compression for: {os.path.basename(input_video)}")
    cap_in, cap_mask = cv2.VideoCapture(input_video), cv2.VideoCapture(mask_video)
    if not cap_in.isOpened():
        logging.error(f"Error: Unable to open input video: {input_video}")
        return 0, 0, 0
    if not cap_mask.isOpened():
        logging.error(f"Error: Unable to open mask video: {mask_video}")
        return 0, 0, 0
    fps = cap_in.get(cv2.CAP_PROP_FPS)
    size = (int(cap_in.get(cv2.CAP_PROP_FRAME_WIDTH)), int(cap_in.get(cv2.CAP_PROP_FRAME_HEIGHT)))
    out = _open_writer(os.path.join(output_dir, "compressed.mp4"), fps, size)

    n_frames, exhausted = 0, False
    while not exhausted:
        frames, masks = [], []
        while len(frames) < _CHUNK:
            ok_f, f = cap_in.read()
            ok_m, m = cap_mask.read()
            if not (ok_f and ok_m):
                exhausted = True
                break
            frames.append(f)
            masks.append(cv2.cvtColor(m, cv2.COLOR_BGR2GRAY) if m.ndim == 3 else m)      # :148-149
        if frames:
            for processed in _hl.degrade_mco_gpu(frames, masks):
                n_frames += 1
                out.write(processed)
    cap_in.release()
    cap_mask.release()
    out.release()
    total = time.time() - t_start
    avg = total / n_frames if n_frames > 0 else 0
    logging.info(f"Motion-based compression completed for '{os.path.basename(input_video)}' in {total:.2f} seconds. Frames processed: {n_frames}")
    return n_frames, total, avg


def process_single_video_of(video_path, output_dir, flow_device="cpu"):
    """motion_compression_opt.py:195-247: motion detection, then compression, then execution_times.txt.  flow_device: see
    temporal_smoothing_flow."""
    name = _hl.video_stem(video_path)
    out_dir = os.path.join(output_dir, name)
    os.makedirs(out_dir, exist_ok=True)
    setup_logging(out_dir)
    logging.info(f"=== Processing for video '{name}' started ===")

    logging.info("Step 1/2: Starting motion detection...")
    md = _hl.StageTiming("Motion Detection", *temporal_smoothing_flow(
        video_path, out_dir, flow_threshold=0.5, alpha_fraction=0.2, window_size=30, morph_kernel=2,
        save_name="overlay.mp4", mask_save_name="mask.mp4", flow_device=flow_device))
    logging.info(f"Step 1/2: Motion detection completed (elapsed: {md.total_s:.2f} s, avg per frame: {md.avg_s:.4f} s).")

    logging.info("Step 2/2: Starting compression...")
    cp = _hl.StageTiming("Compression", *compress_with_motion(os.path.join(out_dir, "overlay.mp4"),
                                                              os.path.join(out_dir, "mask.mp4"), out_dir))
    logging.info(f"Step 2/2: Compression completed (elapsed: {cp.total_s:.2f} s, avg per frame: {cp.avg_s:.4f} s).")

    times_path = os.path.join(out_dir, _hl.TIMES_NAME)
    _hl.write_execution_times(times_path, [md, cp], md.total_s + cp.total_s)
    logging.info(f"Execution times logged in: {times_path}")
    logging.info(f"=== Processing of '{name}' completed successfully. ===")
