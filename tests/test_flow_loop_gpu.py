"""The flow loop (DVC_MODE_FLOW, FramePipeline(w, h, "flow")) against tests/flow_loop_ref.py::flow_loop: every output frame,
mask bytes and compressed bytes, and the counters against what degrade_blend(..., "mco", counters=...) accumulates for the same
frames and the reference masks.  Failures name the case, the stream, the frame and the output."""
import functools
import os
import sys

import cv2
import numpy as np
import pytest
import torch

from dynamic_video_compression_surveillance_b200.synth import make_clip

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALL_SITE = (0.3, 2, 9, 2, 5, 1.1, 0)          # motion_compression_opt.py:72-81


def _P():
    from dynamic_video_compression_surveillance_b200 import pipeline
    return pipeline


@functools.lru_cache(maxsize=None)
def _clip(h, w, n, seed):
    """Smooth background and moving objects, as oracle/make_golden.py::make_of builds the fixtures' clips: [n, h, w, 3]."""
    clip = make_clip((h, w), n, seed=seed)
    yy, xx = np.mgrid[0:h, 0:w]
    clip.background = np.stack([(xx * 255 // w), (yy * 255 // h), ((xx + yy) * 255 // (w + h))], -1).astype(np.uint8)
    return np.stack(list(clip.frames()))


@functools.lru_cache(maxsize=None)
def _oracle(clip_key, params):
    """flow_loop on frames 1.. of the clip, seeded with frame 0: (masks, compressed) arrays [n - 1, ...]."""
    from tests.flow_loop_ref import flow_loop
    out = flow_loop(list(_clip(*clip_key)), **dict(params))
    return np.stack(out["mask"]), np.stack(out["compressed"])


def _loop_kw(params):
    kw = dict(params)
    return dict(window_size=kw.get("window_size", 30), alpha_fraction=kw.get("alpha_fraction", 0.2),
                morph_kernel=kw.get("morph_kernel", 2), morph_shape=kw.get("morph_shape", "ellipse"))


def _pipe(w, h, params, max_batch, **extra):
    kw = dict(params)
    return _P().FramePipeline(w, h, "flow", max_batch=max_batch, flow_threshold=kw.get("flow_threshold", 0.5),
                              farneback=kw.get("farneback", CALL_SITE), **_loop_kw(params), **extra)


def _run(pipe, frames, batches, masks=True, compressed=True):
    """frames [n, h, w, 3] on the GPU, in consecutive batches of the given sizes -> host (masks, compressed) (None when off)."""
    n = frames.shape[0]
    m = torch.zeros(frames.shape[:-1], dtype=torch.uint8, device="cuda") if masks else None
    c = torch.zeros_like(frames) if compressed else None
    t, i = 0, 0
    while t < n:
        b = min(batches[i % len(batches)], n - t)
        pipe.process_device(frames[t:t + b], compressed=None if c is None else c[t:t + b], mask=None if m is None else m[t:t + b])
        t, i = t + b, i + 1
    pipe.flush()
    torch.cuda.synchronize()
    return (None if m is None else m.cpu().numpy()), (None if c is None else c.cpu().numpy())


def _same(case, got, want, what, stream=0, first_frame=1):
    assert got.shape == want.shape, f"{case}: {what} shape {got.shape} != {want.shape}"
    for t in range(want.shape[0]):
        if not np.array_equal(got[t], want[t]):
            raise AssertionError(f"{case}: stream {stream}, frame {t + first_frame}, {what}: "
                                 f"{int((got[t] != want[t]).sum())} bytes differ")


def _expected_counters(frames, masks):
    ctr = torch.zeros(5, dtype=torch.int64, device="cuda")
    _P().degrade_blend(frames.contiguous(), torch.from_numpy(masks).cuda(), 8, 100, "mco", want_overlay=False, counters=ctr)
    torch.cuda.synchronize()
    return dict(zip(("frames", "pixels", "motion_pixels", "blocks", "static_blocks"), (int(v) for v in ctr.cpu())))


def _check(case, clip_key, params, batches, max_batch):
    h, w = clip_key[0], clip_key[1]
    clip = _clip(*clip_key)
    want_m, want_c = _oracle(clip_key, params)
    frames = torch.from_numpy(clip[1:]).cuda()
    with _pipe(w, h, params, max_batch) as pipe:
        pipe.begin_stream_frames(clip[0])
        got_m, got_c = _run(pipe, frames, batches)
        counters = pipe.counters()
    _same(case, got_m, want_m, "mask")
    _same(case, got_c, want_c, "compressed")
    assert counters == _expected_counters(frames, want_m), f"{case}: counters {counters}"
    assert want_m.any() and not want_m.all(), f"{case}: degenerate masks"
    return want_m


# 1. shapes and parameters
CASES = {
    "240x352_K30_ellipse2": ((240, 352, 25, 41), (), [8]),
    "97x131_K5_rect3": ((97, 131, 25, 43), (("window_size", 5), ("alpha_fraction", 0.5), ("morph_kernel", 3),
                                            ("morph_shape", "rect"), ("flow_threshold", 0.3)), [6]),
    "240x352_K1_nomorph": ((240, 352, 13, 45), (("window_size", 1), ("morph_kernel", 0)), [5]),
    "1080p_K5": ((1080, 1920, 21, 44), (("window_size", 5),), [20]),
}


@pytest.mark.parametrize("case", list(CASES))
def test_flow_loop_matches_oracle(case):
    clip_key, params, batches = CASES[case]
    _check(case, clip_key, params, batches, max(batches))


def test_flow_loop_threshold_equal_to_a_magnitude():
    """A threshold equal to a magnitude the flow produces: that pixel is not motion (mag > thr, compared as float32)."""
    from oracle import flow_ops
    clip_key = (240, 352, 9, 46)
    g = np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in _clip(*clip_key)[:2]])
    mag = flow_ops.magnitude(flow_ops.farneback(g[0], g[1], *CALL_SITE))
    thr = float(np.sort(mag.ravel())[int(mag.size * 0.97)])
    assert (mag == np.float32(thr)).any()
    _check("threshold_equal", clip_key, (("flow_threshold", thr), ("window_size", 3)), [4], 4)


def test_flow_loop_farneback_parameters():
    """A non-default Farneback tuple through dvc_set_flow_params (a pyramid of another size) against the oracle with the same."""
    fb = (0.5, 3, 7, 3, 7, 1.5, 0)
    clip_key = (240, 352, 11, 47)
    params = (("farneback", fb), ("window_size", 4))
    clip = _clip(*clip_key)
    want_m, want_c = _oracle(clip_key, params)
    with _pipe(352, 240, (("window_size", 4),), 5) as pipe:
        pipe.set_flow_params(0.5, fb)
        pipe.begin_stream_frames(clip[0])
        got_m, got_c = _run(pipe, torch.from_numpy(clip[1:]).cuda(), [5])
    _same("farneback_params", got_m, want_m, "mask")
    _same("farneback_params", got_c, want_c, "compressed")


# 2. batching and state
BATCH_CLIP = (97, 131, 41, 48)
BATCH_PARAMS = (("window_size", 5), ("morph_kernel", 2))


@pytest.mark.parametrize("batches", [[40], [1], [7], [16], [3, 1, 7]], ids=lambda b: "b" + "_".join(map(str, b)))
def test_flow_loop_batches(batches):
    """One batch against batches of 1, 7 and 16 (ring of max_batch + K + 1 slots: every split wraps it, and a first batch
    shorter than K grows the vote's L)."""
    _check(f"batches {batches}", BATCH_CLIP, BATCH_PARAMS, batches, max(batches))


def test_flow_loop_state_hand_off_and_begin_variants():
    clip = _clip(*BATCH_CLIP)
    want_m, want_c = _oracle(BATCH_CLIP, BATCH_PARAMS)
    frames = torch.from_numpy(clip[1:]).cuda()
    h, w = BATCH_CLIP[:2]
    with _pipe(w, h, BATCH_PARAMS, 8) as a, _pipe(w, h, BATCH_PARAMS, 8) as b:
        a.begin_stream(cv2.cvtColor(clip[0], cv2.COLOR_BGR2GRAY))          # begin_stream with the gray plane
        m1, c1 = _run(a, frames[:13], [8])
        b.set_state(a.get_state())                                         # mid-stream into a second handle
        m2, c2 = _run(b, frames[13:], [8])
    _same("state hand-off", np.concatenate([m1, m2]), want_m, "mask")
    _same("state hand-off", np.concatenate([c1, c2]), want_c, "compressed")


# 3. stream groups
def test_flow_loop_stream_group_equals_solo_handles():
    """S = 4 streams of different clips at 1080p, S * T > the group's G: the pairs of one batch span several flow launch
    groups and cross stream boundaries inside a group.  Every stream equals a solo handle byte for byte."""
    S, T, h, w = 4, 6, 1080, 1920
    clips = [_clip(h, w, T + 1, 60 + s) for s in range(S)]
    params = (("window_size", 3),)
    frames = torch.from_numpy(np.stack([c[1:] for c in clips])).cuda()
    with _pipe(w, h, params, T, n_streams=S) as grp:
        G = grp.flow_group
        assert S * T > G > T, G
        grp.begin_stream_frames(np.stack([c[0] for c in clips]))
        grp.profile(True)
        m = torch.zeros(frames.shape[:-1], dtype=torch.uint8, device="cuda")
        c = torch.zeros_like(frames)
        grp.process_device(frames, compressed=c, mask=m)
        prof = grp.profile_read()
        gm, gc = m.cpu().numpy(), c.cpu().numpy()
    # launches of the flow: per stream gray + (level image + fit) per level, per group (matrices + 3 per iteration) per level
    L = 2
    groups = -(-S * T // G)
    assert prof["front"][1] == S * (1 + 2 * (L + 1)) + groups * (L + 1) * (1 + 3 * 2), (prof["front"], G)
    for s in range(S):
        with _pipe(w, h, params, T) as solo:
            solo.begin_stream_frames(clips[s][0])
            sm, sc = _run(solo, frames[s].contiguous(), [T])
        _same("stream group", gm[s], sm, "mask", stream=s)
        _same("stream group", gc[s], sc, "compressed", stream=s)
        assert sm.any(), f"stream {s}: no motion"


# 4. call variants
def test_flow_loop_call_variants():
    clip = _clip(*BATCH_CLIP)
    want_m, want_c = _oracle(BATCH_CLIP, BATCH_PARAMS)
    frames = torch.from_numpy(clip[1:]).cuda()
    h, w = BATCH_CLIP[:2]

    def fresh(**kw):
        p = _pipe(w, h, BATCH_PARAMS, 8, **kw)
        p.begin_stream_frames(clip[0])
        return p

    with fresh() as p:
        p.set_overlap(True)
        m, c = _run(p, frames, [8])
    _same("overlap on", m, want_m, "mask")
    _same("overlap on", c, want_c, "compressed")
    with fresh() as p:
        m, _ = _run(p, frames, [8], compressed=False)
    _same("compressed=None", m, want_m, "mask")
    with fresh() as p:
        _, c = _run(p, frames, [8], masks=False)
    _same("mask=None", c, want_c, "compressed")
    with fresh() as p:
        hm, hc = np.zeros(want_m.shape, np.uint8), np.zeros(want_c.shape, np.uint8)
        p.process_host(np.ascontiguousarray(clip[1:]), compressed=hc, mask=hm)
        counters = p.counters()
    _same("process_host", hm, want_m, "mask")
    _same("process_host", hc, want_c, "compressed")
    assert counters == _expected_counters(frames, want_m)


# 5. argument codes
def test_flow_loop_argument_codes():
    from dynamic_video_compression_surveillance_b200._lib import DVC_ERR_INVALID, DVC_ERR_UNSUPPORTED, DvcError
    P = _P()

    def code(fn):
        with pytest.raises(DvcError) as e:
            fn()
        return e.value.code

    assert code(lambda: P.FramePipeline(64, 48, "flow", block_size=4)) == DVC_ERR_UNSUPPORTED
    assert code(lambda: P.FramePipeline(64, 48, "flow", kernel_size=7)) == DVC_ERR_INVALID
    assert code(lambda: P.FramePipeline(64, 48, "flow", src_size=(128, 96))) == DVC_ERR_UNSUPPORTED
    assert code(lambda: P.FramePipeline(64, 48, "flow", farneback=(0.3, 2, 9, 2, 5, 1.1, 256))) == DVC_ERR_UNSUPPORTED
    assert code(lambda: P.FramePipeline(64, 48, "flow", farneback=(0.3, 2, 9, 2, 3, 1.1, 0))) == DVC_ERR_UNSUPPORTED
    assert code(lambda: P.FramePipeline(64, 48, "flow", farneback=(1.5, 2, 9, 2, 5, 1.1, 0))) == DVC_ERR_INVALID
    with P.FramePipeline(64, 48, "flow", max_batch=2) as p:
        f = torch.zeros((2, 48, 64, 3), dtype=torch.uint8, device="cuda")
        assert code(lambda: p.process_device(f, overlay=torch.zeros_like(f))) == DVC_ERR_INVALID
        assert code(lambda: p.process_host(f.cpu().numpy(), overlay=np.zeros((2, 48, 64, 3), np.uint8))) == DVC_ERR_INVALID
        assert code(lambda: p.set_flow_params(0.5, (0.3, 2, 9, 2, 5, 1.1, 256))) == DVC_ERR_UNSUPPORTED
        p.process_device(f, mask=torch.zeros(f.shape[:-1], dtype=torch.uint8, device="cuda"))     # still usable
    with P.FramePipeline(64, 48, "window", kernel_size=0, max_batch=2) as p:
        assert code(lambda: p.set_flow_params(0.5, CALL_SITE)) == DVC_ERR_INVALID


# 6. the drop-in
def test_dropin_gpu_masks_equal_flow_loop(tmp_path, monkeypatch):
    """The mask.mp4 frames temporal_smoothing_flow(flow_device="gpu") hands its writer equal flow_loop's masks on the decoded
    frames; the overlay.mp4 frames are the decoded frames."""
    from tests.flow_loop_ref import flow_loop
    sys.path.insert(0, os.path.join(ROOT, "dynamic_video_compression_surveillance_b200", "dropin"))
    sys.modules.pop("motion_compression_opt", None)
    import motion_compression_opt as mco
    h, w, n = 96, 128, 37                      # more than two 16-frame chunks
    src = str(tmp_path / "cam.mp4")
    wr = cv2.VideoWriter(src, cv2.VideoWriter_fourcc(*"mp4v"), 30, (w, h))
    for f in _clip(h, w, n, 5):
        wr.write(f)
    wr.release()
    cap, dec = cv2.VideoCapture(src), []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        dec.append(f)
    cap.release()
    written = {}
    orig = mco._open_writer

    class Recorder:
        def __init__(self, inner, sink):
            self.inner, self.sink = inner, sink

        def write(self, frame):
            self.sink.append(np.array(frame))
            self.inner.write(frame)

        def release(self):
            self.inner.release()

    monkeypatch.setattr(mco, "_open_writer", lambda path, fps, size, color=True:
                        Recorder(orig(path, fps, size, color), written.setdefault(os.path.basename(path), [])))
    nf, _, _ = mco.temporal_smoothing_flow(src, str(tmp_path), flow_device="gpu")
    want = flow_loop(dec, degrade=False)["mask"]
    assert nf == len(dec) - 1 == len(written["mask.mp4"]) == len(written["overlay.mp4"])
    for t, (a, b) in enumerate(zip(written["mask.mp4"], want)):
        assert np.array_equal(a, b), f"drop-in: frame {t + 1}, mask.mp4: {int((a != b).sum())} bytes differ"
    for t, (a, b) in enumerate(zip(written["overlay.mp4"], dec[1:])):
        assert np.array_equal(a, b), f"drop-in: frame {t + 1}, overlay.mp4"
    assert any(m.any() for m in want)
