"""Time the window loop's mask clean-up chain (close + open with a k x k element, motion_compression_opt.py:89-90) per frame,
for elements up to and beyond 33 x 33 (k_morph_chain below, the k_mlarge_* kernels above).

The chain runs inside the loop (FramePipeline "window", kernel_size 0) on resident synthetic frames; its time is the handle's
CUDA-event time of the morphology group (profile_read()["morph"]) over the timed batches; a batch's bit-planes (32 x 1080p:
8 MB) stay in L2.  Every size first checks a sample against cv2: one blob and one noise mask (the frame's width, at most 540
rows) through the stage op's close then open.  Writes one JSON document (--out) with the GPU's name and power limit.

    python tools/morph_large_bench.py --out profiles/r3_morph_large_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dynamic_video_compression_surveillance_b200 import pipeline as P  # noqa: E402
from dynamic_video_compression_surveillance_b200.synth import make_clip  # noqa: E402

SIZES = {"1080p": (1080, 1920), "4k": (2160, 3840)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def check_sample(shape, kind, k, seed):
    r = np.random.default_rng(seed)
    h, w = shape
    blob = np.zeros(shape, np.uint8)
    for _ in range(20):
        cv2.circle(blob, (int(r.integers(0, w)), int(r.integers(0, h))), int(r.integers(2, max(3, h // 6))), 255, -1)
    masks = np.stack([blob, (r.random(shape) < 0.3).astype(np.uint8) * 255])
    el = np.ones((k, k), np.uint8) if kind == "rect" else cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k))
    got = P.morph(P.morph(torch.from_numpy(masks).cuda(), "close", k, kind), "open", k, kind).cpu().numpy()
    for i in range(2):
        want = cv2.morphologyEx(cv2.morphologyEx(masks[i], cv2.MORPH_CLOSE, el), cv2.MORPH_OPEN, el)
        if not np.array_equal(got[i], want):
            raise SystemExit(f"{kind} {k} on {shape}: {int((got[i] != want).sum())} pixels differ from cv2")


def time_chain(frames, seed_gray, kind, k, batch, warmup, steps):
    n, h, w = frames.shape[:3]
    pipe = P.FramePipeline(w, h, "window", window_size=5, morph_kernel=k, morph_shape=kind, kernel_size=0, max_batch=batch)
    pipe.begin_stream(seed_gray)
    ov, cp = torch.empty_like(frames[:batch]), torch.empty_like(frames[:batch])
    done = 0
    for i in range(warmup + steps):
        if i == warmup:
            torch.cuda.synchronize()
            pipe.profile_read()
            pipe.profile(True)
        s = (i * batch) % (n - batch + 1)
        pipe.process_device(frames[s:s + batch], ov, cp)
        done += batch if i >= warmup else 0
    pipe.flush()
    ms, launches = pipe.profile_read()["morph"]
    pipe.close()
    return {"ms_per_frame": ms / done, "frames": done, "launches_per_batch": launches / steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1080p,4k")
    ap.add_argument("--ks", default="33,35,65,129,255")
    ap.add_argument("--kinds", default="rect,ellipse")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("morph_large_bench: needs a CUDA device")
    doc = {"gpu": gpu_info(), "what": "close + open per frame inside the window loop (CUDA events around the morphology group)",
           "batch": a.batch, "steps": a.steps, "results": []}
    for size in a.sizes.split(","):
        h, w = SIZES[size]
        clip = make_clip((h, w), a.batch + 8, seed=5)
        frames = torch.from_numpy(clip.frames()).cuda()
        seed_gray = cv2.cvtColor(frames[0].cpu().numpy(), cv2.COLOR_BGR2GRAY)
        body = frames[1:]
        for kind in a.kinds.split(","):
            for k in map(int, a.ks.split(",")):
                check_sample((min(h, 540), w), kind, k, k)
                r = dict(size=size, kind=kind, k=k, path="k_morph_chain" if k <= 33 else "k_mlarge",
                         **time_chain(body, seed_gray, kind, k, a.batch, a.warmup, a.steps))
                doc["results"].append(r)
                print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
