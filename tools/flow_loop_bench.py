"""Throughput of the flow loop (DVC_MODE_FLOW: BASELINE config 5 run as one loop) against today's stage-call chain.

    python tools/flow_loop_bench.py [--height 1080 --width 1920 --frames 32 --max-batch 16 --streams 1 8 --reps 3 --out r.json]

Each of S streams is a synthetic clip (the make_of recipe, one seed per stream) of --frames + 1 frames, resident on the GPU.
One run processes every frame of every stream, with the rectangle masks and the compressed frames as outputs:
  loop    one FramePipeline(w, h, "flow", n_streams=S, max_batch=B): begin_stream_frames (not timed), then the frames in batches
          of B per stream, overlap on, flushed
  stages  per stream, the chain host_loop assembled before the loop existed: bgr2gray -> flow_masks -> temporal_ring ->
          morph close -> morph open -> mask_rectangles -> degrade_blend(..., "mco")
The two are timed alternately (CUDA events around whole runs, after one warm-up run of each) and their outputs must be equal.
A separate run with dvc_profile_* on gives per-group times: flow (gray, pyramids, flow, written into the mask ring), vote +
morphology + rectangles, degrade, mask unpacking.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

FARNEBACK = (0.3, 2, 9, 2, 5, 1.1, 0)                       # motion_compression_opt.py:72-81
LOOP = dict(window_size=30, alpha_fraction=0.2, morph_kernel=2)      # the call site's values (:29-30)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--max-batch", type=int, default=16)
    ap.add_argument("--streams", type=int, nargs="+", default=[1, 8])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("flow_loop_bench needs a CUDA device")
    from flow_bench import gpu_info
    from dynamic_video_compression_surveillance_b200 import build, pipeline as P
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    build.build()

    h, w, n, B = a.height, a.width, a.frames, a.max_batch

    def clip(seed):
        c = make_clip((h, w), n + 1, seed=seed)
        yy, xx = np.mgrid[0:h, 0:w]
        c.background = np.stack([(xx * 255 // w), (yy * 255 // h), ((xx + yy) * 255 // (w + h))], -1).astype(np.uint8)
        return np.stack(list(c.frames()))

    def events(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    results = []
    for S in a.streams:
        host = np.stack([clip(100 + s) for s in range(S)])                  # [S, n + 1, h, w, 3]
        frames = torch.from_numpy(host).cuda()
        body = frames[:, 1:].contiguous()                                    # [S, n, h, w, 3]
        out = {k: (torch.empty(body.shape[:-1], dtype=torch.uint8, device="cuda"), torch.empty_like(body))
               for k in ("loop", "stages")}
        batch_in = [body[:, t:t + B].contiguous() for t in range(0, n, B)]
        batch_out = [(torch.empty(x.shape[:-1], dtype=torch.uint8, device="cuda"), torch.empty_like(x)) for x in batch_in]
        pipe = P.FramePipeline(w, h, "flow", max_batch=B, n_streams=S, **LOOP)
        pipe.set_overlap(True)
        first = host[:, 0] if S > 1 else host[0, 0]

        def loop_run():
            for x, (m, c) in zip(batch_in, batch_out):
                pipe.process_device(x if S > 1 else x[0], compressed=c if S > 1 else c[0], mask=m if S > 1 else m[0])
            pipe.flush()

        def loop_collect():
            m, c = out["loop"]
            for i, (bm, bc) in enumerate(batch_out):
                m[:, i * B:i * B + bm.shape[1]].copy_(bm)
                c[:, i * B:i * B + bc.shape[1]].copy_(bc)

        def stages_run():
            m, c = out["stages"]
            for s in range(S):
                grays = P.bgr2gray(frames[s])
                raw = P.flow_masks(grays, 0.5, *FARNEBACK)
                voted = P.temporal_ring(raw, LOOP["window_size"], LOOP["alpha_fraction"])
                closed = P.morph(voted, "close", LOOP["morph_kernel"], "ellipse")
                rect = P.mask_rectangles(P.morph(closed, "open", LOOP["morph_kernel"], "ellipse"))
                comp, _ = P.degrade_blend(body[s], rect, 8, 100, "mco", want_overlay=False)
                m[s].copy_(rect)
                c[s].copy_(comp)

        def loop_timed():
            pipe.begin_stream_frames(first)
            torch.cuda.synchronize()
            return events(loop_run)

        loop_timed(), events(stages_run)                                      # warm-up
        ms = {"loop": [], "stages": []}
        for _ in range(a.reps):
            ms["loop"].append(loop_timed())
            ms["stages"].append(events(stages_run))
        loop_collect()
        torch.cuda.synchronize()
        for k, name in ((0, "mask"), (1, "compressed")):
            if not torch.equal(out["loop"][k], out["stages"][k]):
                raise SystemExit(f"S={S}: loop and stage chain differ in {name}")
        motion = float((out["loop"][0] != 0).float().mean())

        pipe.begin_stream_frames(first)
        pipe.profile(True)
        loop_run()
        prof = pipe.profile_read()
        pipe.profile(False)
        pipe.close()

        fr = S * n
        med = lambda v: float(np.median(v))
        per = lambda keys: sum(prof[k][0] for k in keys) / fr
        results.append({
            "streams": S, "frames_per_stream": n, "max_batch": B, "flow_group_pairs": pipe.flow_group,
            "loop": {"ms_per_run": ms["loop"], "frames_per_s": fr / med(ms["loop"]) * 1e3},
            "stages": {"ms_per_run": ms["stages"], "frames_per_s": fr / med(ms["stages"]) * 1e3},
            "loop_over_stages": med(ms["stages"]) / med(ms["loop"]),
            "profiled_ms_per_frame": {"flow": per(["front"]), "vote_morph_rectangles": per(["vote", "morph", "ccl"]),
                                      "degrade": per(["degrade"]), "mask_unpack": per(["misc"])},
            "profiled_launches": {k: v[1] for k, v in prof.items() if v[1]},
            "outputs_equal": True, "mask_motion_fraction": motion,
        })
        del frames, body, out, batch_in, batch_out
        torch.cuda.empty_cache()

    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "shape": [h, w], "farneback": list(FARNEBACK),
           "flow_threshold": 0.5, "loop": LOOP, "reps": a.reps, "results": results}
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
