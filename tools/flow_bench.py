"""Throughput of the GPU Farneback flow at the drop-in's call site (motion_compression_opt.py:72-81) against cv2 on the host.

    python tools/flow_bench.py [--height 1080 --width 1920 --pool 64 --reps 5 --cv2-pairs 4 --out result.json]

Frames are synthetic (the make_of clip recipe) and stay resident on the GPU: a pool of --pool frames (64 x 1080p = 133 MB,
more than the 126 MB L2) is processed as pool-1 pairs per call.  Times are CUDA events around whole calls, after one
warm-up call.  Both entry points are measured:
  pairs     dvc_farneback_flow_f32 on pool-1 independent (prev, next) pairs: two pyramids per pair, flow written
  sequence  dvc_flow_masks_u8 on the pool as one sequence: one pyramid per frame, masks written
Bytes per full-resolution pixel are counted from the shapes (compulsory traffic of each kernel, every level, one pass over
its inputs and outputs; gathers and halo reads that hit in cache are not counted).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PARAMS = (0.3, 2, 9, 2, 5, 1.1, 0)


def level_sizes(h, w, pyr_scale, levels):
    k, s = 0, 1.0
    while k < levels:
        s *= pyr_scale
        if w * s < 32 or h * s < 32:
            break
        k += 1
    out = []
    for lv in range(k + 1):
        s = 1.0
        for _ in range(lv):
            s *= pyr_scale
        out.append((int(np.rint(h * s)), int(np.rint(w * s))))
    return out


def bytes_per_pixel(h, w, params, sequence):
    """Compulsory bytes per full-resolution pixel of one pair, per kernel."""
    pyr_scale, levels, winsize, iterations = params[:4]
    lv = level_sizes(h, w, pyr_scale, levels)
    frac = [a * b / (h * w) for a, b in lv]
    frames = 1 if sequence else 2                   # pyramids built per pair
    out = {
        "k_flow_level": frames * sum(f * 4 for f in frac) + frames * 1,          # float level image out, uint8 frame in
        "k_flow_poly": frames * sum(f * (4 + 20) for f in frac),                  # level image in, 5 coefficients out
        "k_flow_matrices": sum(f * (20 + 20 + 20) for f in frac) + sum(f * 8 for f in frac[:-1]),   # R0, R1, M (+ coarse flow)
        "k_flow_vsum": iterations * sum(f * (20 + 40) for f in frac),            # M in, double column sums out
        # column sums in; non-final iterations also read R0, R1 and write M; final: flow (8 B) or mask (1 B)
        "k_flow_solve": sum(f * (iterations * 40 + (iterations - 1) * 60) for f in frac)
                        + sum(f * 8 for f in frac[1:]) + (1 if sequence else 8),
    }
    out["total"] = sum(out.values())
    return out


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:                               # the measurement itself does not depend on it
        return f"unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--pool", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cv2-pairs", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import cv2
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("flow_bench needs a CUDA device")
    from dynamic_video_compression_surveillance_b200 import build, pipeline as P
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    build.build()

    h, w, n = a.height, a.width, a.pool
    clip = make_clip((h, w), n, seed=7)
    yy, xx = np.mgrid[0:h, 0:w]
    clip.background = np.stack([(xx * 255 // w), (yy * 255 // h), ((xx + yy) * 255 // (w + h))], -1).astype(np.uint8)
    grays_host = [cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in clip.frames()]
    grays = torch.from_numpy(np.stack(grays_host)).cuda()
    prev, nxt = grays[:-1].contiguous(), grays[1:].contiguous()

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return ms

    pairs = n - 1
    ms_pairs = timed(lambda: P.farneback_flow(prev, nxt, *PARAMS))
    ms_seq = timed(lambda: P.flow_masks(grays, 0.5, *PARAMS))

    t_cv2 = []
    for i in range(min(a.cv2_pairs, pairs)):
        t0 = time.perf_counter()
        f = cv2.calcOpticalFlowFarneback(grays_host[i], grays_host[i + 1], None, *PARAMS)
        mag, _ = cv2.cartToPolar(f[..., 0], f[..., 1])
        _ = (mag > 0.5)
        t_cv2.append(time.perf_counter() - t0)

    med = lambda v: float(np.median(v))
    res = {
        "gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0),
        "shape": [h, w], "params": list(PARAMS), "pool_frames": n, "pairs_per_call": pairs, "reps": a.reps,
        "levels_used": len(level_sizes(h, w, PARAMS[0], PARAMS[1])) - 1,
        "pairs_entry": {"ms_per_call": ms_pairs, "ms_per_pair": med(ms_pairs) / pairs, "pairs_per_s": pairs / med(ms_pairs) * 1e3,
                        "bytes_per_pixel": bytes_per_pixel(h, w, PARAMS, False)},
        "sequence_entry": {"ms_per_call": ms_seq, "ms_per_pair": med(ms_seq) / pairs, "pairs_per_s": pairs / med(ms_seq) * 1e3,
                           "bytes_per_pixel": bytes_per_pixel(h, w, PARAMS, True)},
        "cv2_cpu": {"version": cv2.__version__, "threads": cv2.getNumThreads(), "cpu_count": os.cpu_count(),
                    "ms_per_pair": [1e3 * t for t in t_cv2], "pairs_per_s": 1.0 / med(t_cv2) if t_cv2 else None},
    }
    for k in ("pairs_entry", "sequence_entry"):
        e = res[k]
        e["achieved_GB_per_s"] = e["bytes_per_pixel"]["total"] * h * w / (e["ms_per_pair"] * 1e-3) / 1e9
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
