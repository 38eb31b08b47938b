"""The flow loop restated on arrays, for the flow-loop tests: temporal_smoothing_flow (motion_compression_opt.py:65-101)
with the masks kept as arrays and compress_with_motion's arithmetic (:152-183) on each frame, BASELINE config 5.

Same cv2 calls in the same order as the reference, with ``oracle.flow_ops.flow_masks`` (cv2's scalar path, bit for bit) in
place of cv2's Farneback + cartToPolar + threshold and ``oracle.stage_ops.degrade_mco`` for the compressed frames."""
from collections import deque

import cv2
import numpy as np

from oracle import flow_ops
from oracle import stage_ops as so
from oracle.loops import morph_kernel_ellipse


def flow_loop(frames, flow_threshold=0.5, farneback=(0.3, 2, 9, 2, 5, 1.1, 0), window_size=30, alpha_fraction=0.2,
              morph_kernel=2, morph_shape="ellipse", quantization_level=100, prev_gray=None, history=None, degrade=True):
    """``farneback`` = (pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags).  ``frames[0]`` seeds prev_gray
    unless state is given; ``history`` is the raw-mask deque of an earlier chunk.  Returns dict of per-frame lists raw, voted,
    morphed, mask (the mask.mp4 frame), compressed (+ final state)."""
    frames = list(frames)
    if prev_gray is None:
        prev_gray = cv2.cvtColor(frames[0], cv2.COLOR_BGR2GRAY)
        frames = frames[1:]
    q = deque(history or [], maxlen=window_size)
    mk = (morph_kernel_ellipse(morph_kernel) if morph_shape == "ellipse"
          else np.ones((morph_kernel, morph_kernel), np.uint8)) if morph_kernel > 0 else None
    grays = [cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in frames]
    seq = [prev_gray] + grays
    raws = []
    for i in range(0, len(grays), 8):          # pairs in chunks: the model holds every pair's double box sums in memory
        raws.extend(flow_ops.flow_masks(np.stack(seq[i:i + 9]), flow_threshold, *farneback))
    out = dict(raw=[], voted=[], morphed=[], mask=[], compressed=[])
    for frame, raw in zip(frames, raws):
        q.append(raw)
        cumulative = np.sum(np.array(q), axis=0)
        voted = (cumulative >= (alpha_fraction * len(q) * 255)).astype(np.uint8) * 255
        m = voted
        if mk is not None:
            m = cv2.morphologyEx(m, cv2.MORPH_CLOSE, mk)
            m = cv2.morphologyEx(m, cv2.MORPH_OPEN, mk)
        rect = np.zeros_like(m)
        contours, _ = cv2.findContours(m, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
        for c in contours:
            x, y, w, h = cv2.boundingRect(c)
            cv2.rectangle(rect, (x, y), (x + w, y + h), 255, -1)
        out["raw"].append(raw)
        out["voted"].append(voted)
        out["morphed"].append(m)
        out["mask"].append(rect)
        if degrade:
            out["compressed"].append(so.degrade_mco(frame, rect, quantization_level))
    out["state_prev_gray"] = seq[-1]
    out["state_history"] = list(q)
    return out
