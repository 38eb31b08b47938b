#!/usr/bin/env python
"""Benchmark of the per-frame hot loop (BASELINE.json metric: 1080p frames/s, HBM roofline fraction).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1).  --dump-outputs writes a seeded sample of the overlay and compressed frames of the
last timed step (rank 0's streams for N > 1) to DIR as float32 .npy files (dump_outputs).

* N = 1: `value` is BASELINE configs[1] -- one 1080p stream, 1800 frames per step, K=5 window vote -- with the clip and
  the output buffers resident in HBM (11.2 GB in, 22.4 GB out per step, far larger than L2); `e2e` is the same loop
  through the host-buffer C-ABI call (dvc_process_host) with pinned host frames, H2D and D2H inside the timed region.
  The line also carries `modes.fd` (the frame_differencing.py loop proper: blur5 + contour filter + EMA), `streams64`
  (BASELINE configs[3] on this one GPU, resident and end to end) and the CPU baselines.
* N > 1: `value` is BASELINE configs[3] -- 64 concurrent 1080p camera streams (seeds 0..63) sharded 64/N per rank
  (sharding.shard_streams), each rank one lock-step stream group (dvc_config.n_streams), strong scaling: a step advances
  every stream by the same 224 frames whatever N is.  `e2e` is the same workload through dvc_process_host.  No collective
  on the per-frame path; one all-reduce of the statistics counters at the end.  `weak_single_stream` repeats the N = 1
  workload on every rank for comparison with round 1's curve.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree it runs from untouched (it may be read-only)

import numpy as np  # noqa: E402

METRIC = "1080p_frames_per_second"
UNIT = "frames/s"
LOOP = dict(window_size=5, alpha_fraction=0.2, morph_kernel=2, morph_shape="ellipse", kernel_size=7, block_size=4,
            motion_threshold=0.5, quantization_level=100)
# bytes per pixel per frame (DESIGN.md section 4)
K4_ALG_BYTES_PER_PX = 3 + 3 + 3 + 1.0 / 8          # read BGR, write compressed + overlay, read the mask bit-plane
SURVEY_LOOP_BYTES_PER_PX = 28                      # SURVEY.md section 8(d) accounting of the north_star loop (uint8 masks)
ACTUAL_LOOP_BYTES_PER_PX = 3 + 1.0 / 8 + K4_ALG_BYTES_PER_PX + 4 * (1.0 / 8)   # this design: K1 + mask planes + K4


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--frames", type=int, default=1800)
    p.add_argument("--resolution", default="1080p")
    p.add_argument("--max-batch", type=int, default=int(os.environ.get("DVC_BENCH_BATCH", "225")))
    p.add_argument("--e2e-frames", type=int, default=256)
    p.add_argument("--mode", default="window", choices=["window", "fd"])
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-overlap", action="store_true", help="strict per-batch stream order instead of the two-stream pipeline")
    # overrides of the loop parameters for the other BASELINE configs (e.g. config 3: --resolution 4k --frames 900
    # --kernel-size 15 --morph-kernel 15 --morph-shape rect); the default line is config 2
    p.add_argument("--kernel-size", type=int, default=None)
    p.add_argument("--morph-kernel", type=int, default=None)
    p.add_argument("--morph-shape", default=None, choices=["ellipse", "rect"])
    p.add_argument("--window-size", type=int, default=None)
    p.add_argument("--streams", type=int, default=64, help="camera streams of the sharded workload (BASELINE configs[3])")
    p.add_argument("--stream-batch", type=int, default=28, help="frames per stream per launch in the 64-stream workload")
    p.add_argument("--stream-batches-per-step", type=int, default=8)
    p.add_argument("--stream-e2e-frames", type=int, default=12, help="frames per stream per host call in the 64-stream e2e run")
    p.add_argument("--no-streams", action="store_true", help="N = 1: skip the 64-stream section")
    p.add_argument("--no-fd", action="store_true", help="N = 1: skip the fd-mode section")
    p.add_argument("--cpu-config1", action="store_true", help="also time BASELINE configs[0] (480p, 300 frames) on the host (~3-5 min)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write a seeded sample of what the last timed step computed (overlay and "
                        "compressed frames) to DIR/<name>.npy as float32, for comparing two builds output for output")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        p.error("--dump-outputs applies to --impl b200")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def mark(self):
        """Start of the timed region: samples before this wall-clock instant are ignored."""
        import datetime
        self.t_mark = datetime.datetime.now()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        self.power_max = None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                import datetime
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f")
                if getattr(self, "t_mark", None) and ts < self.t_mark:
                    continue
                sm.append(float(f[1])); mx.append(float(f[2]))
                self.power_max = max(self.power_max or 0.0, float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "sm_mhz_min": min(sm) if sm else None,
                "power_w_max": self.power_max}


# ---------------------------------------------------------------------------------------------------
# synthetic clip
# ---------------------------------------------------------------------------------------------------
def device_clip(clip, n_frames, device):
    """Render the synthetic clip directly into HBM (same bytes as clip.frames(): static background +
    rectangles pasted in order)."""
    import torch
    bg = torch.from_numpy(clip.background).to(device)
    out = torch.empty((n_frames,) + tuple(bg.shape), dtype=torch.uint8, device=device)
    out[:] = bg
    for t in range(n_frames):
        for (x, y, w, h), rect in zip(clip.rect_positions(t), clip.rects):
            out[t, y:y + h, x:x + w] = torch.tensor(rect[5], dtype=torch.uint8, device=device)
    return out


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the same loop (literal Python block loop, as the reference runs it)
# ---------------------------------------------------------------------------------------------------
def _cpu_loop(frames, mode, state, degrade):
    """One call of the oracle loop on `frames` (frame 0 seeds prev_gray when state is None).  degrade: True = the
    reference's literal Python block loop, "colour_only" = the cv2 calls without the block loop, False = masks only."""
    from oracle import loops
    if mode == "window":
        kw = dict(LOOP); kw["literal_blocks"] = True
        st = {} if state is None else dict(prev_gray=state["prev_gray"], history=state["history"])
        r = loops.window_loop(frames, degrade=degrade, **kw, **st)
        return r, dict(prev_gray=r["state_prev_gray"], history=r["state_history"])
    kw = dict(block_size=LOOP["block_size"], kernel_size=LOOP["kernel_size"], literal_blocks=True)
    st = {} if state is None else dict(prev_gray=state["prev_gray"], acc=state["acc"])
    r = loops.fd_loop(frames, degrade=degrade, **kw, **st)
    return r, dict(prev_gray=r["state_prev_gray"], acc=r["state_acc"])


def cpu_warm_state(clip, mode, n_warm=12):
    """Loop state after frames 1..n_warm (past the EMA / window warm-up, so blocks are static as in steady state);
    computed with the vectorised oracle path, which the tests pin to the literal one."""
    from oracle import loops
    frames = [clip[t % len(clip)] for t in range(n_warm + 1)]
    if mode == "window":
        kw = dict(LOOP); kw["literal_blocks"] = False
        r = loops.window_loop(frames, degrade=False, **kw)
        return dict(prev_gray=r["state_prev_gray"], history=r["state_history"]), n_warm + 1
    r = loops.fd_loop(frames, block_size=LOOP["block_size"], kernel_size=LOOP["kernel_size"], degrade=False)
    return dict(prev_gray=r["state_prev_gray"], acc=r["state_acc"]), n_warm + 1


def cpu_time_frames(clip, mode, state, t_next, n, degrade=True):
    """Time n consecutive frames starting at clip[t_next] from `state`; returns (seconds, new state, next t)."""
    frames = [clip[t % len(clip)] for t in range(t_next, t_next + n)]
    t0 = time.perf_counter()
    _, state = _cpu_loop(frames, mode, state, degrade)
    return time.perf_counter() - t0, state, t_next + n


def cpu_baselines(clip, mode, literal_frames=8):
    """BASELINE.md section 3: the reference loop (literal block loop) past its warm-up with the default thread count and
    with cv2.setNumThreads(1), and the cv2-only stage baseline (same calls, no Python block loop)."""
    import cv2
    default_threads = cv2.getNumThreads()
    state, t = cpu_warm_state(clip, mode)
    dt, state, t = cpu_time_frames(clip, mode, state, t, literal_frames)
    fps = literal_frames / dt
    ds, state, t = cpu_time_frames(clip, mode, state, t, 100, degrade="colour_only")
    cv2.setNumThreads(1)
    try:
        d1, state, t = cpu_time_frames(clip, mode, state, t, 3)
        ds1, state, t = cpu_time_frames(clip, mode, state, t, 40, degrade="colour_only")
    finally:
        cv2.setNumThreads(default_threads)
    return {"value": fps, "unit": UNIT, "cores": default_threads, "kind": "port",
            "sample": f"frames 13..{12 + literal_frames} of the same clip ({dt:.1f} s), after 12 warm-up frames; oracle/loops.py "
                      f"with the reference's literal Python block loop (frame_differencing.py:117-127); cv2 {cv2.__version__} "
                      f"threads={default_threads}, os.cpu_count()={os.cpu_count()}, IPP={cv2.ipp.useIPP()}",
            "single_thread_fps": 3 / d1, "single_thread_sample": "3 frames with cv2.setNumThreads(1)",
            "stages_only_fps": 100 / ds, "stages_only_single_thread_fps": 40 / ds1,
            "stages_only_sample": "100 (default threads) / 40 (1 thread) frames of the cv2 calls of the loop without the Python "
                                  "block loop: gray, absdiff, threshold, vote, close/open, dilate, overlay paint, BGR<->YCrCb"}


def cpu_config1():
    """BASELINE configs[0]: frame_differencing.py defaults on the synthetic 640x480 300-frame clip, all 299 frames."""
    import cv2
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    clip = make_clip("480p", 300, seed=0)
    frames = [clip[t] for t in range(300)]
    t0 = time.perf_counter()
    _cpu_loop(frames, "fd", None, True)
    dt = time.perf_counter() - t0
    return {"frames": 299, "seconds": dt, "s_per_frame": dt / 299, "fps": 299 / dt, "threads": cv2.getNumThreads(),
            "workload": "BASELINE configs[0]: 640x480, 300 frames, frame_differencing.py defaults, literal block loop"}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the loop on this box's host cores.  The reference is
    pure Python + cv2 and cannot travel as a compiled artefact, so this runs the oracle port (same cv2 calls, same
    Python block loop: oracle/loops.py), one frame of the same 1080p workload per step, after the loop's warm-up."""
    if rank != 0:
        return
    import cv2
    from dynamic_video_compression_surveillance_b200.synth import make_clip, RESOLUTIONS
    h, w = RESOLUTIONS[args.resolution]
    clip = make_clip(args.resolution, args.frames, seed=0)
    state, t = cpu_warm_state(clip, args.mode)
    for _ in range(max(0, args.warmup)):
        _, state, t = cpu_time_frames(clip, args.mode, state, t, 1)
    total = 0.0
    for _ in range(args.steps):
        dt, state, t = cpu_time_frames(clip, args.mode, state, t, 1)
        total += dt
    fps = args.steps / total
    threads = cv2.getNumThreads()
    cfg = (workload_config(args, h, w) if world == 1 else streams_config(args, h, w, world))
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
            "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": cfg | {"sample": "1 frame of stream 0 per step, after 12 warm-up frames"},
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"{args.steps} consecutive 1080p frames, one per step; oracle/loops.py literal block loop; "
                                       f"cv2 {cv2.__version__} threads={threads}, os.cpu_count()={os.cpu_count()}"},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def loop_name(mode):
    return {"window": f"north_star loop: gray/absdiff/threshold -> K={LOOP['window_size']} window vote -> {LOOP['morph_shape']}-"
                      f"{LOOP['morph_kernel']} close/open -> {LOOP['kernel_size']}x{LOOP['kernel_size']} dilate -> "
                      "overlay + 4x4 block-DCT degrade",
            "fd": "frame_differencing.py loop: gray/blur5/absdiff/threshold -> contour filter -> 7x7 dilate -> EMA -> overlay + "
                  "4x4 block-DCT degrade"}[mode]


def workload_config(args, h, w):
    cfg_name = "BASELINE configs[1]" if (args.resolution, args.frames) == ("1080p", 1800) else "BASELINE-style config"
    return {"workload": f"{cfg_name}: single {args.resolution} ({w}x{h}) synthetic stream per GPU, {args.frames} frames, "
                        f"{loop_name(args.mode)}", "mode": args.mode, "frames_per_step": args.frames, "max_batch": args.max_batch,
            "two_stream_overlap": not args.no_overlap,
            "pipeline": ("strict stream order" if args.no_overlap else
                         "batches pipelined over the handle's streams: mask kernels of batch n + 1 beside the degrade kernel of batch n"
                         + ("; fd mode: the front kernel on a third stream, one more batch ahead" if args.mode == "fd" else "")),
            "l2_policy": f"inputs (clip {args.frames * h * w * 3 / 1e9:.1f} GB) and outputs ({2 * args.frames * h * w * 3 / 1e9:.1f} GB) per step "
                         "are far larger than the 126 MB L2"}


def streams_config(args, h, w, world):
    per = args.stream_batch * args.stream_batches_per_step
    return {"workload": f"BASELINE configs[3]: {args.streams} concurrent {args.resolution} ({w}x{h}) synthetic camera streams (seeds 0.."
                        f"{args.streams - 1}) sharded {args.streams}/{world} per GPU, one lock-step stream group per rank, "
                        f"{loop_name('window')}", "mode": "window", "streams": args.streams, "streams_per_gpu": args.streams // world,
            "frames_per_step": args.streams * per, "frames_per_stream_per_step": per, "frames_per_stream_per_launch": args.stream_batch,
            "two_stream_overlap": not args.no_overlap,
            "l2_policy": f"every launch reads {args.streams // world * args.stream_batch * h * w * 3 / 1e9:.2f} GB of frames and writes twice "
                         "that, larger than the 126 MB L2; stream state (gray planes, mask rings) is per stream"}


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
class Ctx:
    """Per-rank plumbing: device, barrier over ranks, max-over-ranks reduction."""

    def __init__(self, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.rank, self.world, self.local_rank = torch, dist, rank, world, local_rank
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        if world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, x: float) -> list:
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [x]
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(o.item()) for o in out]


def timed_steps(ctx, pipe, one_pass, steps, warmup, sampler=None):
    """W untimed passes, then exactly `steps` passes between CUDA events, barrier + synchronize on both sides; returns
    (milliseconds, max over ranks; kernels this rank launched inside the timed region)."""
    torch = ctx.torch
    for _ in range(max(3, warmup)):
        one_pass()
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    launches0 = pipe.launch_count()
    if sampler is not None:
        sampler.mark()
    e0.record()
    for _ in range(steps):
        one_pass()
    e1.record()
    ctx.barrier()
    return ctx.max_over_ranks(e0.elapsed_time(e1)), pipe.launch_count() - launches0


DUMP_SAMPLES = 1 << 22          # elements kept per output array: 16 MB as float32


def dump_outputs(out_dir, arrays):
    """Write each device array of `arrays` to out_dir/<name>.npy as a float32 vector: the elements of the flattened array at
    the sorted positions np.random.default_rng(0).integers(0, size, DUMP_SAMPLES), or all of them when the array is no larger.
    The positions depend only on the array's size, so two builds run with the same arguments dump comparable samples."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        flat = t.reshape(-1)
        if flat.numel() > DUMP_SAMPLES:
            pos = np.sort(np.random.default_rng(0).integers(0, flat.numel(), DUMP_SAMPLES))
            flat = flat[torch.from_numpy(pos).to(flat.device)]
        np.save(os.path.join(out_dir, name + ".npy"), flat.cpu().numpy().astype(np.float32))


def profile_pass(ctx, pipe, one_pass, steps):
    """Second timed region, same steps, strict stream order (kernels serialised) with CUDA events around every kernel group on
    its launch stream: per-kernel times for the roofline are not inflated by concurrently running kernels."""
    torch = ctx.torch
    pipe.set_overlap(False)
    one_pass()
    ctx.barrier()
    pipe.profile(True)
    pipe.profile_read()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(steps):
        one_pass()
    p1.record()
    ctx.barrier()
    ms_serial = p0.elapsed_time(p1)
    prof = pipe.profile_read()
    pipe.profile(False)
    return ms_serial, prof


def k4_roofline(prof, ms_serial, frames_per_step, steps, px, loop_fps_per_gpu, dev, torch):
    peak, peak_src = peaks()
    k4_ms, k4_launches = prof["degrade"]
    frames_per_launch = frames_per_step * steps / max(1, k4_launches)
    k4_bytes = K4_ALG_BYTES_PER_PX * px * frames_per_launch
    k4_gbs = k4_bytes / (k4_ms / max(1, k4_launches) * 1e-3) / 1e9 if k4_ms > 0 else 0.0
    kernel_ms = {k: v[0] for k, v in prof.items() if v[1]}
    roofline = {"bound": "hbm", "kernel": "k_degrade4s (K4, persistent TMA ring: overlay + YCrCb + 4x4 DCT degrade + statistics)",
                "achieved": k4_gbs, "peak": peak, "unit": "GB/s", "frac": k4_gbs / peak, "peak_source": peak_src,
                "traffic": None, "alg_bytes_per_px": K4_ALG_BYTES_PER_PX, "frames_per_launch": frames_per_launch,
                "avg_launch_ms": k4_ms / max(1, k4_launches), "kernel_share_of_step": k4_ms / ms_serial if ms_serial else None,
                "timed_region": "second pass of the same K steps in strict stream order (no two-stream overlap) with CUDA events "
                                "around each kernel group on its launch stream",
                "serialised_fps_per_gpu": frames_per_step * steps / (ms_serial / 1e3),
                "kernel_ms_in_timed_region": kernel_ms,
                "loop": {"fps_per_gpu": loop_fps_per_gpu,
                         "survey_accounting": {"bytes_per_px": SURVEY_LOOP_BYTES_PER_PX,
                                               "frac": loop_fps_per_gpu * px * SURVEY_LOOP_BYTES_PER_PX / 1e9 / peak},
                         "this_design": {"bytes_per_px": ACTUAL_LOOP_BYTES_PER_PX,
                                         "frac": loop_fps_per_gpu * px * ACTUAL_LOOP_BYTES_PER_PX / 1e9 / peak}}}
    # K4 writes twice what it reads, and HBM absorbs writes more slowly than a read/write mix: report the kernel's write rate
    # next to a write-only (fill) rate measured here, as context for `frac` (which stays against the copy peak)
    try:
        fill_buf = torch.empty(1 << 31, dtype=torch.uint8, device=dev)
        best = None
        for _ in range(6):
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(); fill_buf.zero_(); f1.record(); torch.cuda.synchronize()
            t_ms = f0.elapsed_time(f1)
            best = t_ms if best is None else min(best, t_ms)
        fill_gbs = fill_buf.numel() / (best * 1e-3) / 1e9
        del fill_buf
        k4_write_gbs = 6.0 * px * frames_per_launch / (k4_ms / max(1, k4_launches) * 1e-3) / 1e9 if k4_ms > 0 else 0.0
        roofline["write_path"] = {"written_bytes_per_px": 6.0, "achieved_write": k4_write_gbs, "fill_peak_measured_here": fill_gbs,
                                  "unit": "GB/s", "frac_of_fill_peak": k4_write_gbs / fill_gbs if fill_gbs else None}
    except Exception:
        pass
    traffic_file = os.path.join(ROOT, "profiles", "k4_dram_bytes_per_launch.json")
    if os.path.exists(traffic_file):
        try:
            tf = json.load(open(traffic_file))
            roofline["traffic"] = tf["dram_bytes_per_frame"] * frames_per_launch
            roofline["traffic_source"] = tf.get("source")
        except Exception:
            pass
    return roofline


def measure_single_stream(ctx, args, mode, steps, sampler=None, want_e2e=True, dump_dir=None):
    """One 1080p stream per rank (BASELINE configs[1] at N = 1): resident loop, profile pass, end-to-end pass.  dump_dir: where
    to dump the last timed step's overlay and compressed frames (dump_outputs)."""
    import torch
    from dynamic_video_compression_surveillance_b200 import pipeline as P
    from dynamic_video_compression_surveillance_b200.synth import make_clip, RESOLUTIONS
    h, w = RESOLUTIONS[args.resolution]
    n, B, dev = args.frames, args.max_batch, ctx.dev
    clip = make_clip(args.resolution, n + 1, seed=ctx.rank)            # stream id = rank (SURVEY.md section 8d)
    frames = device_clip(clip, n + 1, dev)
    ov = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
    cp = torch.empty_like(ov)
    kw = dict(LOOP)
    if mode == "fd":
        for k in ("window_size", "alpha_fraction", "morph_kernel", "morph_shape"):
            kw.pop(k)
    pipe = P.FramePipeline(w, h, mode, max_batch=B, device=ctx.local_rank, **kw)
    if mode == "window":
        seed_gray = P.bgr2gray(frames[:1])[0].cpu().numpy()
    else:
        import cv2
        seed_gray = cv2.GaussianBlur(P.bgr2gray(frames[:1])[0].cpu().numpy(), (25, 25), 30)   # stays on the host (fd:77)
    pipe.begin_stream(seed_gray)
    pipe.set_overlap(not args.no_overlap)
    body = frames[1:]

    def one_pass():
        for i in range(0, n, B):
            pipe.process_device(body[i:i + B], ov[i:i + B], cp[i:i + B])
        pipe.flush()          # the current stream re-joins the library's internal streams

    ms, launches = timed_steps(ctx, pipe, one_pass, steps, args.warmup, sampler)
    if dump_dir is not None:
        dump_outputs(dump_dir, {"overlay": ov, "compressed": cp})
    value = steps * n * ctx.world / (ms / 1e3)
    ms_serial, prof = profile_pass(ctx, pipe, one_pass, steps)
    res = {"value": value, "ms": ms, "launches": launches, "ms_serial": ms_serial, "prof": prof, "frames_per_step": n,
           "counters": pipe.counters(), "clip": clip, "hw": (h, w)}
    if want_e2e:
        ne = min(args.e2e_frames, n)
        px = h * w
        hin = P.pinned_empty((ne, h, w, 3)); hov = P.pinned_empty((ne, h, w, 3)); hcp = P.pinned_empty((ne, h, w, 3))
        hin.copy_(body[:ne].cpu())
        for _ in range(3):
            pipe.process_host(hin, hov, hcp)
        ctx.barrier()
        t0 = time.perf_counter()
        reps = max(1, steps)
        for _ in range(reps):
            pipe.process_host(hin, hov, hcp)          # returns when the outputs are in host memory
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        per_gpu = ctx.gather(reps * ne / dt)
        res["e2e"] = {"value": reps * ne * ctx.world / ctx.max_over_ranks(dt), "unit": UNIT, "h2d_bytes_per_step": ne * px * 3,
                      "d2h_bytes_per_step": 2 * ne * px * 3, "frames_per_step": ne, "per_gpu": per_gpu,
                      "note": "dvc_process_host: pinned host frames in, overlay + compressed frames out, 8-frame chunks "
                              "double-buffered on copy/compute streams; wall clock around the blocking call"}
        del hin, hov, hcp
    pipe.close()
    del frames, ov, cp
    torch.cuda.empty_cache()
    return res


def measure_streams(ctx, args, steps, sampler=None, want_e2e=True, dump_dir=None):
    """BASELINE configs[3]: args.streams camera streams sharded over the ranks, one lock-step stream group per rank.  dump_dir:
    where to dump the last timed step's overlay and compressed frames of this rank's streams (dump_outputs)."""
    import torch
    from dynamic_video_compression_surveillance_b200 import pipeline as P, sharding
    from dynamic_video_compression_surveillance_b200.synth import make_clip, RESOLUTIONS
    h, w = RESOLUTIONS[args.resolution]
    px = h * w
    dev = ctx.dev
    ids = sharding.shard_streams(args.streams, ctx.world, ctx.rank)
    S, F, nb = len(ids), args.stream_batch, args.stream_batches_per_step
    clips = [make_clip(args.resolution, F + 1, seed=i) for i in ids]                 # seed = stream id (SURVEY.md section 8d)
    frames = torch.stack([device_clip(c, F + 1, dev) for c in clips])                 # [S][F + 1]
    seeds = P.bgr2gray(frames[:, 0].contiguous()).cpu().numpy()                         # [S][H][W]
    body = frames[:, 1:].contiguous()                                                   # [S][F]
    del frames
    ov = torch.empty_like(body)
    cp = torch.empty_like(body)
    pipe = P.FramePipeline(w, h, "window", max_batch=F, device=ctx.local_rank, n_streams=S, **LOOP)
    pipe.begin_stream(seeds)
    pipe.set_overlap(not args.no_overlap)

    def one_pass():
        # a step advances every stream by nb x F frames; the F resident frames of a stream are cycled (its state carries on)
        for _ in range(nb):
            pipe.process_device(body, ov, cp)
        pipe.flush()

    ms, launches = timed_steps(ctx, pipe, one_pass, steps, args.warmup, sampler)
    if dump_dir is not None:
        dump_outputs(dump_dir, {"overlay": ov, "compressed": cp})
    frames_per_step_rank = S * F * nb
    value = steps * args.streams * F * nb / (ms / 1e3)
    ms_serial, prof = profile_pass(ctx, pipe, one_pass, steps)
    res = {"value": value, "ms": ms, "launches": launches, "ms_serial": ms_serial, "prof": prof,
           "frames_per_step": frames_per_step_rank, "counters": pipe.counters(), "streams_per_gpu": S, "hw": (h, w)}
    if want_e2e:
        ne = args.stream_e2e_frames

        def e2e_pass(group, n_local, src):
            """Blocking dvc_process_host calls on a group of n_local streams; returns this rank's seconds for `reps` calls."""
            if n_local == 0:
                ctx.barrier()
                return 0.0, 1
            hin = P.pinned_empty((n_local, ne, h, w, 3)); hov = P.pinned_empty((n_local, ne, h, w, 3)); hcp = P.pinned_empty((n_local, ne, h, w, 3))
            for s_ in range(n_local):
                hin[s_].copy_(src[s_ % src.shape[0], :ne].cpu())
            hi, ho, hc = (hin, hov, hcp) if n_local > 1 else (hin[0], hov[0], hcp[0])
            for _ in range(2):
                group.process_host(hi, ho, hc)
            ctx.barrier()
            t0 = time.perf_counter()
            reps = max(2, min(steps, 6))
            for _ in range(reps):
                group.process_host(hi, ho, hc)
            torch.cuda.synchronize()
            return time.perf_counter() - t0, reps

        dt, reps = e2e_pass(pipe, S, body)
        per_gpu = ctx.gather(reps * S * ne / dt)
        e2e_equal = {"value": reps * args.streams * ne / ctx.max_over_ranks(dt), "unit": UNIT,
                     "h2d_bytes_per_step": S * ne * px * 3, "d2h_bytes_per_step": 2 * S * ne * px * 3,
                     "frames_per_step": S * ne, "per_gpu": per_gpu, "streams_per_gpu": [S] * ctx.world,
                     "note": f"dvc_process_host on the stream group: {S} streams x {ne} pinned host frames per call, chunks of one "
                             "frame per stream double-buffered on copy/compute streams; wall clock around the blocking call"}
        res["e2e"] = e2e_equal
        if ctx.world > 1:
            # End to end a rank is as fast as its share of the host's IO fabric (profiles/r2_scale8_pcie_probe.txt: four GPUs
            # of the box sit behind an uplink with 1.5x the bandwidth of the other four), so the streams are re-dealt in
            # proportion to the per-GPU rates just measured and the same workload is timed again.
            counts = [len(x) for x in sharding.shard_streams_weighted(args.streams, per_gpu)]
            Sw = counts[ctx.rank]
            grp = P.FramePipeline(w, h, "window", max_batch=F, device=ctx.local_rank, n_streams=max(1, Sw), **LOOP)
            grp.begin_stream(np.ascontiguousarray(seeds[np.arange(max(1, Sw)) % S]) if Sw != 1 else seeds[0])
            dtw, repsw = e2e_pass(grp, Sw, body)
            grp.close()
            per_gpu_w = ctx.gather(repsw * Sw * ne / dtw if Sw else 0.0)
            res["e2e"] = {"value": repsw * args.streams * ne / ctx.max_over_ranks(dtw), "unit": UNIT,
                          "h2d_bytes_per_step": Sw * ne * px * 3, "d2h_bytes_per_step": 2 * Sw * ne * px * 3,
                          "frames_per_step": Sw * ne, "per_gpu": per_gpu_w, "streams_per_gpu": counts,
                          "sharding": "streams dealt in proportion to each GPU's measured end-to-end rate (sharding.shard_streams_weighted)",
                          "equal_shards": e2e_equal, "note": e2e_equal["note"]}
    pipe.close()
    del body, ov, cp
    torch.cuda.empty_cache()
    return res


def measure_mco(ctx, args, steps):
    """BASELINE configs[4]: rectangle masks (what temporal_smoothing_flow hands over, motion_compression_opt.py:93-97) fed to the
    shared degrade kernel in MCO flavour (8x8, three quantised planes, re-gray: :152-183) on resident 1080p frames."""
    import torch
    from dynamic_video_compression_surveillance_b200 import pipeline as P
    from dynamic_video_compression_surveillance_b200.synth import make_clip, RESOLUTIONS
    h, w = RESOLUTIONS[args.resolution]
    n = 64
    clip = make_clip(args.resolution, n, seed=5)
    frames = device_clip(clip, n, ctx.dev)
    masks = torch.zeros((n, h, w), dtype=torch.uint8, device=ctx.dev)
    for t in range(n):
        for (x, y, rw, rh) in clip.rect_positions(t):
            masks[t, max(0, y - 8):y + rh + 9, max(0, x - 8):x + rw + 9] = 255
    for _ in range(3):
        P.degrade_blend(frames, masks, 8, 100, "mco", False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        P.degrade_blend(frames, masks, 8, 100, "mco", False)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    del frames, masks
    torch.cuda.empty_cache()
    peak, _ = peaks()
    fps = steps * n / (ms / 1e3)
    return {"workload": f"BASELINE configs[4]: {args.resolution} frames + rectangle masks -> degrade kernel, MCO flavour (8x8 blocks, Y/Cr/Cb "
                        "quantised, re-gray), 64 resident frames per call incl. mask packing", "value": fps, "unit": UNIT,
            "us_per_frame": 1e3 * ms / (steps * n), "alg_bytes_per_px": 7.0,
            "frac_of_hbm_peak": fps * h * w * 7.0 / 1e9 / peak}


def run_b200(args, rank, world, local_rank):
    import torch
    from dynamic_video_compression_surveillance_b200.synth import RESOLUTIONS
    ctx = Ctx(rank, world, local_rank)
    h, w = RESOLUTIONS[args.resolution]
    px = h * w
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                      # started early: nvidia-smi's own start-up must not fall into the timed region
    extra = {}
    dump_dir = args.dump_outputs if rank == 0 else None
    if world == 1:
        main = measure_single_stream(ctx, args, args.mode, args.steps, sampler, want_e2e=not args.no_e2e, dump_dir=dump_dir)
        clocks = sampler.stop()
        cfg, scaling = workload_config(args, h, w), "weak"
        if not args.no_fd and args.mode == "window":
            fd_steps = max(3, args.steps // 2)            # (a quarter of the steps gave the three-stream pipeline's ramp too much weight)
            fd = measure_single_stream(ctx, args, "fd", fd_steps, want_e2e=False)
            peak, _ = peaks()
            kms = {k: v[0] for k, v in fd["prof"].items() if v[1]}
            top = max(kms, key=kms.get)
            alg = {"degrade": K4_ALG_BYTES_PER_PX, "front": 4.0, "ccl": 2.0 / 8, "diff": 2 + 1.0 / 8, "ema": 3.0 / 8, "morph": 2.0 / 8}
            extra["modes"] = {"fd": {
                "workload": f"single {args.resolution} stream, {args.frames} frames per step, {loop_name('fd')}",
                "value": fd["value"], "unit": UNIT, "ms_per_step": fd["ms"] / fd_steps, "steps": fd_steps,
                "serialised_fps": fd["frames_per_step"] * fd_steps / (fd["ms_serial"] / 1e3),
                "kernel_ms_in_timed_region": kms, "dominant_kernel": top,
                "dominant_kernel_us_per_frame": 1e3 * kms[top] / (fd["frames_per_step"] * fd_steps),
                "dominant_kernel_frac_of_hbm_peak": alg.get(top, 0) * px * fd["frames_per_step"] * fd_steps / (kms[top] * 1e-3) / 1e9 / peak,
                "alg_bytes_per_px": alg}}
        if not args.no_fd and args.mode == "window":
            extra.setdefault("modes", {})["mco_degrade"] = measure_mco(ctx, args, max(3, args.steps // 2))
        if not args.no_streams and args.mode == "window" and args.resolution == "1080p":
            st = measure_streams(ctx, args, max(3, args.steps // 2), want_e2e=not args.no_e2e)
            extra["streams64"] = {"workload": streams_config(args, h, w, 1)["workload"], "value": st["value"], "unit": UNIT,
                                  "ms_per_step": st["ms"] / max(3, args.steps // 2), "frames_per_step": st["frames_per_step"],
                                  "e2e": st.get("e2e"), "vs_single_stream": st["value"] / main["value"]}
    else:
        main = measure_streams(ctx, args, args.steps, sampler, want_e2e=not args.no_e2e, dump_dir=dump_dir)
        clocks = sampler.stop() if rank == 0 else None
        cfg, scaling = streams_config(args, h, w, world), "strong"
        weak = measure_single_stream(ctx, args, "window", max(3, args.steps // 2), want_e2e=False)
        extra["weak_single_stream"] = {"workload": workload_config(args, h, w)["workload"], "value": weak["value"], "unit": UNIT,
                                       "scaling": "weak"}
    roofline = k4_roofline(main["prof"], main["ms_serial"], main["frames_per_step"], args.steps, px, main["value"] / world,
                           ctx.dev, torch)
    cnt = torch.tensor([v for v in main["counters"].values()], dtype=torch.int64, device=ctx.dev)
    if world > 1:
        ctx.dist.all_reduce(cnt, op=ctx.dist.ReduceOp.SUM)              # the only collective: final statistics
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baselines(main["clip"], args.mode)
        if args.cpu_config1:
            cpu_baseline["config1_480p"] = cpu_config1()
    if rank == 0:
        line = {"metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": main["ms"] / args.steps, "higher_is_better": True,
                "scaling": scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg, "clocks": clocks,
                "e2e": main.get("e2e"), "gpu_launches": main["launches"], "roofline": roofline, "cpu_baseline": cpu_baseline,
                "statistics": dict(zip(main["counters"].keys(), [int(v) for v in cnt.tolist()]))}
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        ctx.dist.destroy_process_group()


def main():
    args = parse_args()
    for key, val in (("kernel_size", args.kernel_size), ("morph_kernel", args.morph_kernel), ("morph_shape", args.morph_shape),
                     ("window_size", args.window_size)):
        if val is not None:
            LOOP[key] = val
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
