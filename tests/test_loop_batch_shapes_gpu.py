"""Both loops at the benchmark's batch shapes against the oracle loops (oracle/loops.py), every output frame.

The benchmark runs 225-frame batches at 1080p with the two-stream overlap on and no mask output, and a 64-stream group with
28 frames per stream per launch.  Those shapes reach code that small test batches never do: the fused front + vote kernel's
later 64-frame segments (which rebuild their window history from the frames), long fd front-end segments, the calls without
a mask output, and stream offsets beyond 4 GiB.  Here every mask and overlay must equal the oracle, every compressed frame
must equal pipeline.degrade_blend on the oracle's masks (the degrade kernel itself is held to the oracle in
tests/test_gpu_parity.py), frames at segment and batch boundaries must also equal so.degrade_fd, and the counters must equal
the statistics of the oracle's masks.  A failure names the case, the stream, the frame (counted from the first frame the
stream processed) and the output, with the number of differing pixels.

Fusion work on the window loop has to pass this file."""
import numpy as np
import pytest
import torch

from oracle import loops, stage_ops as so
from tests.test_gpu_parity import _check_degraded, _exact

pytestmark = pytest.mark.gpu

# bench.py's loop parameters (its LOOP), restated
LOOP = dict(window_size=5, alpha_fraction=0.2, morph_kernel=2, morph_shape="ellipse", kernel_size=7, block_size=4,
            motion_threshold=0.5, quantization_level=100)
FD = {k: v for k, v in LOOP.items() if k not in ("window_size", "alpha_fraction", "morph_kernel", "morph_shape")}
BS, Q = LOOP["block_size"], LOOP["quantization_level"]


@pytest.fixture(scope="module")
def P():
    from dynamic_video_compression_surveillance_b200 import pipeline
    return pipeline


def _clip(shape, n, seed, **kw):
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    return make_clip(shape, n, seed=seed, **kw)


def _device_frames(clip, out, start=0):
    """Render clip frames start .. start + len(out) - 1 straight into the device tensor `out` (the bytes of clip.frames():
    background, then the rectangles in order; clips without temporal noise)."""
    assert not clip.temporal_noise
    bg = torch.from_numpy(clip.background).to(out.device)
    for i in range(out.shape[0]):
        out[i] = bg
        for (x, y, w, h), rect in zip(clip.rect_positions(start + i), clip.rects):
            out[i, y:y + h, x:x + w] = torch.tensor(rect[5], dtype=torch.uint8, device=out.device)
    return out


def _assert_equal(got, want, where, what, t0=0):
    """got / want: [n, H, W] or [n, H, W, 3] uint8 arrays (torch, on any device, or numpy) holding frames t0 .. t0 + n - 1."""
    got, want = torch.as_tensor(got), torch.as_tensor(want)
    assert got.shape == want.shape, (where, what, tuple(got.shape), tuple(want.shape))
    want = want.to(got.device)
    if torch.equal(got, want):
        return
    d = got != want
    if d.dim() == 4:
        d = d.any(-1)
    per = d.reshape(d.shape[0], -1).sum(1).cpu().numpy()
    bad = np.nonzero(per)[0]
    f = int(bad[0])
    yx = tuple(int(v) for v in torch.nonzero(d[f])[0])
    raise AssertionError(f"{where}: {what} differs on {len(bad)} of {len(per)} frames; frame {t0 + f}: {int(per[f])} pixels "
                         f"differ, first at (y, x) {yx}: got {got[f][yx].tolist()}, want {want[f][yx].tolist()}")


class _WindowOracle:
    """loops.window_loop fed chunk by chunk, prev_gray and the raw-mask history carried between chunks."""

    def __init__(self, seed_gray, kw):
        self.pg, self.hist, self.kw = seed_gray, [], kw

    def __call__(self, frames):
        r = loops.window_loop(list(frames), prev_gray=self.pg, history=self.hist, degrade=False, **self.kw)
        self.pg, self.hist = r["state_prev_gray"], r["state_history"]
        return np.stack(r["mask"]), r


class _FdOracle:
    """loops.fd_loop fed chunk by chunk, prev_gray and the accumulator carried between chunks."""

    def __init__(self, seed_gray, kw):
        self.pg, self.acc, self.kw = seed_gray, None, kw

    def __call__(self, frames):
        r = loops.fd_loop(list(frames), prev_gray=self.pg, acc=self.acc, degrade=False, **self.kw)
        self.pg, self.acc = r["state_prev_gray"], r["state_acc"]
        return np.stack(r["acc"]), r


def _check_stream(P, where, frames, ov, cp, mk, oracle, samples=(), chunk=32, seen=None):
    """One stream's outputs (device tensors [N, ...]; mk may be None) against the oracle fed the same device frames in chunks:
    masks and overlays equal, compressed frames equal degrade_blend(frames, oracle masks), and at `samples` so.degrade_fd.
    `seen(result)` gets every chunk's oracle result.  Returns the counters the oracle masks imply."""
    exact = _exact(BS)
    n = frames.shape[0]
    motion = static = 0
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        fr = frames[a:b].cpu().numpy()
        ref, res = oracle(fr)
        if seen is not None:
            seen(res)
        if mk is not None:
            _assert_equal(mk[a:b], ref, where, "mask", a)
        got_ov = ov[a:b].cpu().numpy()
        for i in range(b - a):
            _assert_equal(got_ov[i:i + 1], so.overlay_paint(fr[i], ref[i])[None], where, "overlay", a + i)
        want, _ = P.degrade_blend(frames[a:b], torch.from_numpy(ref).to(frames.device), BS, Q, "fd", False)
        _assert_equal(cp[a:b], want, where, "compressed frame vs degrade_blend on the oracle masks", a)
        for t in samples:
            if a <= t < b:
                got, f, m = cp[t].cpu().numpy(), fr[t - a], ref[t - a]
                want = so.degrade_fd(f, m, BS, Q)
                if exact:
                    _assert_equal(got[None], want[None], where, "compressed frame vs so.degrade_fd", t)
                else:
                    try:
                        _check_degraded(got, want, f, m, BS, Q, False)
                    except AssertionError as e:
                        raise AssertionError(f"{where}: compressed frame vs so.degrade_fd, frame {t}: {e}") from e
        motion += int((ref > 127).sum())
        static += sum(int(so.block_all_zero(m, BS).sum()) for m in ref)
    return {"motion_pixels": motion, "static_blocks": static}


def _assert_counters(where, got, n, h, w, parts):
    want = {"frames": n, "pixels": n * h * w, "motion_pixels": sum(p["motion_pixels"] for p in parts),
            "blocks": n * (-(-h // BS)) * (-(-w // BS)), "static_blocks": sum(p["static_blocks"] for p in parts)}
    assert got == want, f"{where}: counters {got}, the oracle masks give {want}"


def _run(P, mode, kw, body, seed, batches, *, max_batch, want_mask=True, handoff_before=None, n_streams=1):
    """Feed `body` ([N, H, W, 3], or [S, N, H, W, 3] for a stream group) to a fresh handle in batches of the given lengths,
    two-stream overlap on, as bench.py calls it.  handoff_before=i: the state moves to a new handle before batch i.  Returns
    overlay, compressed, mask (None without mask output) and the counters summed over the handles."""
    group = n_streams > 1
    h, w = body.shape[-3:-1]

    def handle():
        p = P.FramePipeline(w, h, mode, max_batch=max_batch, n_streams=n_streams, **kw)
        p.set_overlap(True)
        return p

    pipe = handle()
    pipe.begin_stream(seed)
    ov, cp = torch.empty_like(body), torch.empty_like(body)
    mk = torch.empty(body.shape[:-1], dtype=torch.uint8, device=body.device) if want_mask else None
    counters, staged, t = {}, [], 0

    def add(c):
        for k, v in c.items():
            counters[k] = counters.get(k, 0) + v

    for i, T in enumerate(batches):
        if i == handoff_before:
            blob = pipe.get_state()
            add(pipe.counters())
            pipe.close()
            pipe = handle()
            pipe.set_state(blob)
        sl = slice(t, t + T)
        if group:                       # a group's batch is [S, T]: contiguous copies, written back after the flush
            fin = body[:, sl].contiguous()
            o, c = torch.empty_like(fin), torch.empty_like(fin)
            m = torch.empty(fin.shape[:-1], dtype=torch.uint8, device=fin.device) if want_mask else None
            staged.append((sl, fin, o, c, m))
            pipe.process_device(fin, o, c, m)
        else:
            pipe.process_device(body[sl], ov[sl], cp[sl], None if mk is None else mk[sl])
        t += T
    assert t == body.shape[-4]
    pipe.flush()
    torch.cuda.synchronize()
    add(pipe.counters())
    pipe.close()
    for sl, _, o, c, m in staged:
        ov[:, sl], cp[:, sl] = o, c
        if m is not None:
            mk[:, sl] = m
    return ov, cp, mk, counters


# ---------------------------------------------------------------------------------------------------------------------------
# 1, 2: the benchmark's single-stream lines (window, fd): 1080p, max_batch 225, overlap on, no mask output
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["window", "fd"])
def test_benchmark_line_1080p(P, mode):
    """Rank 0's clip, batches of 225 and 70 frames.  Window loop: the second batch wraps the 231-slot ring, its first segment
    reads history from the ring and its second rebuilds it from the frames.  fd loop: 8 front-end segments of 29 frames (the
    last 22), and the second batch starts from the accumulator the first left.  Then the benchmark's call without a mask
    output on a fresh handle, and the host-buffer call on the first 64 frames, must give the same outputs."""
    h, w, n = 1080, 1920, 295
    kw = LOOP if mode == "window" else FD
    case = f"1080p {mode} line"
    frames = _device_frames(_clip("1080p", n + 1, 0), torch.empty((n + 1, h, w, 3), dtype=torch.uint8, device="cuda"))
    first = frames[0].cpu().numpy()
    body = frames[1:]
    seed = so.bgr2gray(first) if mode == "window" else loops.first_frame_gray_fd(first)
    oracle = _WindowOracle(seed, kw) if mode == "window" else _FdOracle(seed, kw)
    ov, cp, mk, cnt = _run(P, mode, kw, body, seed, (225, 70), max_batch=225)
    exp = _check_stream(P, case, body, ov, cp, mk, oracle, samples=(0, 63, 64, 65, 128, 224, 225, n - 1))
    _assert_counters(case, cnt, n, h, w, [exp])
    del mk

    ov2, cp2, _, cnt2 = _run(P, mode, kw, body, seed, (225, 70), max_batch=225, want_mask=False)
    _assert_equal(ov2, ov, f"{case} without mask output", "overlay")
    _assert_equal(cp2, cp, f"{case} without mask output", "compressed frame")
    assert cnt2 == cnt, f"{case} without mask output: counters {cnt2}, with mask output {cnt}"
    del ov2, cp2

    pipe = P.FramePipeline(w, h, mode, max_batch=225, **kw)
    pipe.begin_stream(seed)
    hin = P.pinned_empty((64, h, w, 3))
    hin.copy_(body[:64].cpu())
    hov, hcp = P.pinned_empty((64, h, w, 3)), P.pinned_empty((64, h, w, 3))
    pipe.process_host(hin, hov, hcp)
    pipe.close()
    _assert_equal(hov, ov[:64], f"{case} host-buffer call", "overlay")
    _assert_equal(hcp, cp[:64], f"{case} host-buffer call", "compressed frame")


# ---------------------------------------------------------------------------------------------------------------------------
# 3: the fused front + vote kernel's segments, swept over window sizes
# ---------------------------------------------------------------------------------------------------------------------------
VOTE_CASES = [  # (name, width, window_size, alpha_fraction, morph_kernel, kernel_size)
    ("fused K=1", 256, 1, 0.4, 0, 0), ("fused K=2", 256, 2, 0.4, 0, 0), ("fused K=5", 256, 5, 0.4, 0, 0),
    ("fused K=8", 256, 8, 0.4, 0, 0),
    ("separate K=9", 256, 9, 0.4, 0, 0),              # K > 8: k_gray_diff_thresh + k_window_vote
    ("separate W=248 K=5", 248, 5, 0.4, 0, 0),        # W % 16 != 0: the same two kernels
    ("fused K=5 with morphology", 256, 5, 0.6, 2, 3),
]


@pytest.mark.parametrize("name,w,K,alpha,morph,dil", VOTE_CASES, ids=[c[0] for c in VOTE_CASES])
def test_vote_segments_against_oracle(P, name, w, K, alpha, morph, dil):
    """max_batch 225, batches 225, 65, 1, 130 and 64: the fused kernel cuts them into 64-frame segments (64/64/64/33, 64/1, 1,
    64/64/2, 64), so segments start inside batches, after a one-frame batch and right after a state hand-off to a new handle
    (before the third batch).  Temporal noise at threshold 1 makes about a quarter of the raw pixels fire independently
    from frame to frame, so the vote depends on every frame of the window: a segment that rebuilds its history from the
    wrong frames changes the masks."""
    h, n = 144, 485
    batches = (225, 65, 1, 130, 64)
    clip = _clip((h, w), n + 1, 11, temporal_noise=True).frames()
    kw = dict(LOOP, window_size=K, alpha_fraction=alpha, morph_kernel=morph, kernel_size=dil, motion_threshold=1.0)
    case = f"vote segments, {name}"
    seed = so.bgr2gray(clip[0])
    body = torch.from_numpy(clip[1:]).cuda()
    ov, cp, mk, cnt = _run(P, "window", kw, body, seed, batches, max_batch=225, handoff_before=2)
    dens = np.zeros(4)

    def seen(r):
        dens[:] += (np.mean(np.stack(r["raw"]) > 0), np.mean(np.stack(r["voted"]) > 0), np.mean(np.stack(r["mask"]) > 0), 1)

    samples = (0, 63, 64, 65, 127, 128, 192, 224, 225, 289, 290, 291, 355, 419, 420, 421, n - 1)
    exp = _check_stream(P, case, body, ov, cp, mk, _WindowOracle(seed, kw), samples=samples, chunk=97, seen=seen)
    _assert_counters(case, cnt, n, h, w, [exp])
    raw, voted, mask = dens[:3] / dens[3]
    assert 0.2 <= raw <= 0.8 and 0.05 <= voted <= 0.95 and 0.05 <= mask <= 0.95, \
        f"{case}: the case has gone trivial: raw density {raw:.3f}, voted {voted:.3f}, final mask {mask:.3f}"


# ---------------------------------------------------------------------------------------------------------------------------
# 4: an fd stream group whose batches need two contour-filter launches and the filter's global node arrays
# ---------------------------------------------------------------------------------------------------------------------------
def test_fd_stream_group_dense_masks(P):
    """480 x 640, two streams, max_batch 150: a full batch is 300 frames, the contour filter's scratch holds 256, so the batch
    takes two filter launches.  Temporal noise at threshold 0.5 gives raw masks with more row runs than the filter keeps in
    shared memory (8192 per frame).  Batches of 150 and 37; every frame of both streams against the oracle."""
    h, w, n, S = 480, 640, 187, 2
    clips = [_clip((h, w), n + 1, 60 + s, temporal_noise=True).frames() for s in range(S)]
    seeds = np.stack([loops.first_frame_gray_fd(c[0]) for c in clips])
    body = torch.from_numpy(np.stack([c[1:] for c in clips])).cuda()
    del clips
    ov, cp, mk, cnt = _run(P, "fd", FD, body, seeds, (150, 37), max_batch=150, n_streams=S)
    parts, runs, dens = [], [], []

    def seen(r):
        for raw in r["raw"]:
            on = raw > 0
            runs.append(int(on[:, 0].sum() + (on[:, 1:] & ~on[:, :-1]).sum()))
            dens.append(float(on.mean()))

    for s in range(S):
        parts.append(_check_stream(P, f"fd group 480p stream {s}", body[s], ov[s], cp[s], mk[s], _FdOracle(seeds[s], FD),
                                   samples=(0, 127, 128, 149, 150, n - 1), seen=seen))
    _assert_counters("fd group 480p", cnt, S * n, h, w, parts)
    assert np.median(runs) > 8192 and 0.2 <= np.mean(dens) <= 0.8, \
        f"fd group 480p: raw masks not dense enough: median row runs {np.median(runs)}, density {np.mean(dens):.3f}"


# ---------------------------------------------------------------------------------------------------------------------------
# 5: the 64-stream workload's launch: 11 GB of frames, stream offsets beyond 4 GiB
# ---------------------------------------------------------------------------------------------------------------------------
def test_64_stream_group_1080p(P):
    """bench.py's 64-stream section on one GPU: one lock-step group of 64 1080p streams (seeds 0..63), 28 frames per stream
    per launch, the same 28 frames sent twice as the benchmark cycles them.  Each stream must equal a solo handle fed the
    same sequence: masks of both launches, overlay and compressed frames of the last.  Streams 0 and 63 also against the
    oracle.  About 45 GB of device memory."""
    h, w, S, F = 1080, 1920, 64, 28
    body = torch.empty((S, F, h, w, 3), dtype=torch.uint8, device="cuda")
    first = torch.empty((1, h, w, 3), dtype=torch.uint8, device="cuda")
    seeds = np.empty((S, h, w), np.uint8)
    for s in range(S):
        clip = _clip("1080p", F + 1, s)
        _device_frames(clip, body[s], start=1)
        seeds[s] = so.bgr2gray(_device_frames(clip, first)[0].cpu().numpy())
    grp = P.FramePipeline(w, h, "window", max_batch=F, n_streams=S, **LOOP)
    grp.begin_stream(seeds)
    grp.set_overlap(True)
    ov, cp = torch.empty_like(body), torch.empty_like(body)
    masks = [torch.empty((S, F, h, w), dtype=torch.uint8, device="cuda") for _ in range(2)]
    for m in masks:
        grp.process_device(body, ov, cp, m)
    grp.flush()
    torch.cuda.synchronize()
    cnt = grp.counters()
    grp.close()
    solo_cnt = {}
    for s in range(S):
        where = f"64-stream group stream {s}"
        pipe = P.FramePipeline(w, h, "window", max_batch=F, **LOOP)
        pipe.begin_stream(seeds[s])
        o, c = torch.empty_like(body[s]), torch.empty_like(body[s])
        ms = torch.empty((2, F, h, w), dtype=torch.uint8, device="cuda")
        for launch in range(2):
            pipe.process_device(body[s], o, c, ms[launch])
        torch.cuda.synchronize()
        for k, v in pipe.counters().items():
            solo_cnt[k] = solo_cnt.get(k, 0) + v
        pipe.close()
        for launch in range(2):
            _assert_equal(masks[launch][s], ms[launch], where, f"mask (launch {launch + 1}) vs solo handle", launch * F)
        _assert_equal(ov[s], o, where, "overlay (launch 2) vs solo handle", F)
        _assert_equal(cp[s], c, where, "compressed frame (launch 2) vs solo handle", F)
        if s in (0, S - 1):
            fr = body[s].cpu().numpy()
            oracle = _WindowOracle(seeds[s], LOOP)
            for launch in range(2):
                ref, _ = oracle(fr)
                _assert_equal(masks[launch][s], ref, where, f"mask (launch {launch + 1}) vs oracle", launch * F)
    assert cnt == solo_cnt, f"64-stream group: counters {cnt}, the solo handles together {solo_cnt}"
    del body, ov, cp, masks
    torch.cuda.empty_cache()
