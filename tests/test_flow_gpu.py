"""Farneback optical flow on the GPU (dvc_farneback_flow_f32 / dvc_flow_masks_u8) against cv2.calcOpticalFlowFarneback run
live on the host.

cv2 does not reproduce its own flow across dispatch paths, so parity is relative.  Per case:
  D_cv2 = the 99.9th percentile of |flow difference| between the default cv2 and its scalar path (setUseOptimized(False)),
  D_gpu = the same percentile between the GPU and the default cv2.
Required: D_gpu <= max(4 D_cv2, 1e-4), and raw-mask (|flow| > thr) pixels that differ from the default cv2 at most
max(4 x the scalar path's own flips, 1e-4 x pixels)."""
import os
import sys

import cv2
import numpy as np
import pytest
import torch

from dynamic_video_compression_surveillance_b200.synth import make_clip
from tests.golden_util import OF_FIXTURES, load_of

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALL_SITE = (0.3, 2, 9, 2, 5, 1.1, 0)          # motion_compression_opt.py:72-81


def _P():
    from dynamic_video_compression_surveillance_b200 import pipeline
    return pipeline


def _grays(h, w, n, seed):
    """Frames as oracle/make_golden.py::make_of builds them (smooth background, moving objects), as gray planes.  Sizes
    below 64 are crops of a 64 x 64 clip."""
    if h < 64 or w < 64:
        return [np.ascontiguousarray(g[:h, :w]) for g in _grays(max(h, 64), max(w, 64), n, seed)]
    clip = make_clip((h, w), n, seed=seed)
    yy, xx = np.mgrid[0:h, 0:w]
    clip.background = np.stack([(xx * 255 // w), (yy * 255 // h), ((xx + yy) * 255 // (w + h))], -1).astype(np.uint8)
    return [cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in clip.frames()]


def _cv2_flows(grays, params, optimized):
    cv2.setUseOptimized(optimized)
    try:
        return np.stack([cv2.calcOpticalFlowFarneback(a, b, None, *params) for a, b in zip(grays[:-1], grays[1:])])
    finally:
        cv2.setUseOptimized(True)


def _mask(flow, thr):
    mag, _ = cv2.cartToPolar(np.ascontiguousarray(flow[..., 0]), np.ascontiguousarray(flow[..., 1]))
    return mag > thr


def _masks(flows, thr):
    return np.stack([_mask(f, thr) for f in flows])


def _p999(a, b):
    return float(np.percentile(np.sqrt(((a.astype(np.float64) - b) ** 2).sum(-1)), 99.9))


def _gpu_flows(grays, params):
    g = torch.from_numpy(np.stack(grays)).cuda()
    return _P().farneback_flow(g[:-1].contiguous(), g[1:].contiguous(), *params).cpu().numpy()


def _check_parity(grays, params, thr=0.5):
    ref, scalar = _cv2_flows(grays, params, True), _cv2_flows(grays, params, False)
    gpu = _gpu_flows(grays, params)
    d_cv2, d_gpu = _p999(ref, scalar), _p999(gpu, ref)
    px = ref.shape[0] * ref.shape[1] * ref.shape[2]
    flips_cv2 = int((_masks(ref, thr) != _masks(scalar, thr)).sum())
    flips_gpu = int((_masks(ref, thr) != _masks(gpu, thr)).sum())
    msg = f"params {params}: D_gpu {d_gpu:.3g} D_cv2 {d_cv2:.3g}, mask flips gpu {flips_gpu} cv2 {flips_cv2} of {px}"
    print(msg)
    assert d_gpu <= max(4 * d_cv2, 1e-4), msg
    assert flips_gpu <= max(4 * flips_cv2, 1e-4 * px), msg
    return gpu


# 1. stage isolation: each row switches one more stage on
STAGES = [
    (0.5, 0, 1, 1, 5, 1.1, 0),       # polynomial expansion, matrices, solve (winsize 1)
    (0.5, 0, 5, 1, 5, 1.1, 0),       # box blur
    (0.5, 0, 9, 1, 5, 1.1, 0),
    (0.5, 0, 15, 1, 5, 1.1, 0),
    (0.5, 0, 9, 2, 5, 1.1, 0),       # matrices recomputed from the flow
    (0.5, 0, 9, 3, 5, 1.1, 0),
    (0.3, 1, 9, 2, 5, 1.1, 0),       # pyramid levels and flow upsampling
    (0.3, 2, 9, 2, 5, 1.1, 0),
    (0.3, 3, 9, 2, 5, 1.1, 0),
    (0.5, 1, 9, 2, 5, 1.1, 0),
    (0.5, 2, 9, 2, 5, 1.1, 0),
    (0.5, 3, 9, 2, 5, 1.1, 0),
    (0.5, 0, 9, 2, 7, 1.5, 0),       # poly_n 7
    (0.5, 2, 10, 2, 7, 1.5, 0),      # even winsize: box 2 * (winsize // 2) + 1, scaled by 1 / winsize^2
]


@pytest.mark.parametrize("params", STAGES, ids=[",".join(map(str, p[:6])) for p in STAGES])
def test_flow_stages_match_cv2(params):
    _check_parity(_grays(240, 352, 3, 41), params)


# 2. shapes: odd sizes, sizes that cut the level count below `levels`, 1080p
@pytest.mark.parametrize("hw", [(17, 23), (40, 56), (121, 163), (1, 37), (33, 1)])
def test_flow_shapes_match_cv2(hw):
    _check_parity(_grays(hw[0], hw[1], 3, 43), CALL_SITE)


def test_flow_1080p_matches_cv2():
    _check_parity(_grays(1080, 1920, 2, 44), CALL_SITE)


# 3. against the unmodified reference's recorded raw masks
@pytest.mark.parametrize("name", OF_FIXTURES)
def test_flow_masks_match_reference_fixture(name):
    from dynamic_video_compression_surveillance_b200 import host_loop
    masks, kw, (h, w, n) = load_of(name)
    seed = int(np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))["recipe"][3])
    grays = _grays(h, w, n, seed)
    thr = kw["flow_threshold"]
    got = _P().flow_masks(torch.from_numpy(np.stack(grays)).cuda(), thr, *CALL_SITE).cpu().numpy()
    raw = masks["raw"] != 0
    scalar = _masks(_cv2_flows(grays, CALL_SITE, False), np.float32(thr))
    flips_cv2, flips_gpu = int((scalar != raw).sum()), int(((got != 0) != raw).sum())
    print(f"{name}: raw-mask flips gpu {flips_gpu}, cv2 scalar path {flips_cv2}, of {raw.size}")
    assert flips_gpu <= max(4 * flips_cv2, 1e-4 * raw.size)
    rect = host_loop.smooth_rect_masks_gpu(list(got), [], kw["window_size"], kw["alpha_fraction"], kw["morph_kernel"])
    rect_diff = int(((rect != 0) != (masks["rect"] != 0)).sum())
    print(f"{name}: rectangle-mask pixels differing from the reference: {rect_diff} of {raw.size}")
    assert rect_diff <= _rect_bound(raw.size)


def _rect_bound(pixels):
    """Rectangle masks grow a raw-mask flip into a rectangle edge: allow 1e-3 of the pixels."""
    return 1e-3 * pixels


def test_flow_threshold_is_compared_as_float32():
    """0.3 is not a float32: numpy compares mag (float32) with float32(0.3), which is slightly above 0.3."""
    grays = _grays(80, 112, 3, 42)
    gpu = _gpu_flows(grays, CALL_SITE)
    mag, _ = cv2.cartToPolar(np.ascontiguousarray(gpu[..., 0]), np.ascontiguousarray(gpu[..., 1]))
    got = _P().flow_masks(torch.from_numpy(np.stack(grays)).cuda(), 0.3, *CALL_SITE).cpu().numpy()
    assert np.array_equal(got != 0, mag > 0.3)
    assert np.array_equal(got != 0, mag > np.float32(0.3))


# 4. exact self-consistency
def test_flow_masks_equal_flow_then_magnitude():
    grays = _grays(121, 163, 7, 45)
    g = torch.from_numpy(np.stack(grays)).cuda()
    for params, thr in ((CALL_SITE, 0.5), ((0.5, 3, 15, 3, 7, 1.5, 0), 0.3)):
        flow = _P().farneback_flow(g[:-1].contiguous(), g[1:].contiguous(), *params).cpu().numpy()
        mag = np.sqrt(flow[..., 0] * flow[..., 0] + flow[..., 1] * flow[..., 1])       # float32, no contraction
        got = _P().flow_masks(g, thr, *params).cpu().numpy()
        assert np.array_equal(got, (mag > np.float32(thr)).astype(np.uint8) * 255)


def test_flow_chunked_with_carried_gray_equals_one_call():
    from dynamic_video_compression_surveillance_b200 import host_loop
    h, w, n = 96, 128, 23
    clip = make_clip((h, w), n, seed=46)
    frames = list(clip.frames())
    first = host_loop.first_gray_gpu(frames[0])
    whole, last = host_loop.flow_masks_gpu(frames[1:], first)
    parts, carry = [], first
    for i in range(1, n, 5):
        m, carry = host_loop.flow_masks_gpu(frames[i:i + 5], carry)
        parts.append(m)
    assert np.array_equal(np.concatenate(parts), whole)
    assert torch.equal(carry, last)
    assert np.array_equal(last.cpu().numpy(), cv2.cvtColor(frames[-1], cv2.COLOR_BGR2GRAY))
    # host-array carry works the same
    m0, _ = host_loop.flow_masks_gpu(frames[1:6], cv2.cvtColor(frames[0], cv2.COLOR_BGR2GRAY))
    assert np.array_equal(m0, parts[0])


def test_flow_is_deterministic():
    grays = _grays(240, 352, 4, 47)
    a, b = _gpu_flows(grays, CALL_SITE), _gpu_flows(grays, CALL_SITE)
    assert a.tobytes() == b.tobytes()
    g = torch.from_numpy(np.stack(grays)).cuda()
    assert torch.equal(_P().flow_masks(g, 0.5), _P().flow_masks(g, 0.5))


def test_flow_pairs_are_independent_of_batching():
    grays = _grays(64, 80, 6, 48)
    whole = _gpu_flows(grays, CALL_SITE)
    single = np.stack([_gpu_flows(grays[i:i + 2], CALL_SITE)[0] for i in range(len(grays) - 1)])
    assert whole.tobytes() == single.tobytes()


# 5. argument checks
def test_flow_argument_checks():
    from dynamic_video_compression_surveillance_b200._lib import DvcError
    P = _P()
    g = torch.zeros((2, 48, 64), dtype=torch.uint8, device="cuda")
    a, b = g[:1], g[1:]
    for kw in (dict(flags=cv2.OPTFLOW_FARNEBACK_GAUSSIAN), dict(flags=cv2.OPTFLOW_USE_INITIAL_FLOW), dict(poly_n=3), dict(poly_n=6)):
        with pytest.raises(NotImplementedError):
            P.farneback_flow(a, b, **kw)
        with pytest.raises(NotImplementedError):
            P.flow_masks(g, 0.5, **kw)
    for kw in (dict(pyr_scale=0.0), dict(pyr_scale=1.0), dict(pyr_scale=1.5), dict(levels=-1), dict(winsize=0), dict(iterations=0)):
        with pytest.raises(DvcError) as e:
            P.farneback_flow(a, b, **kw)
        assert not isinstance(e.value, NotImplementedError)
        with pytest.raises(DvcError):
            P.flow_masks(g, 0.5, **kw)
    assert P.flow_masks(g[:1], 0.5).shape == (0, 48, 64)


# 6. the drop-in's flow_device switch
class _Recorder:
    def __init__(self, inner, sink):
        self.inner, self.sink = inner, sink

    def write(self, frame):
        self.sink.append(np.array(frame))
        self.inner.write(frame)

    def release(self):
        self.inner.release()


def _run_of(mco, monkeypatch, src, out_dir, **kw):
    written = {}
    orig = mco._open_writer

    def rec(path, fps, size, color=True):
        return _Recorder(orig(path, fps, size, color), written.setdefault(os.path.basename(path), []))
    monkeypatch.setattr(mco, "_open_writer", rec)
    mco.process_single_video_of(src, out_dir, **kw)
    monkeypatch.setattr(mco, "_open_writer", orig)
    return written


def test_dropin_of_flow_device_gpu(tmp_path, monkeypatch):
    import logging
    import re
    sys.path.insert(0, os.path.join(ROOT, "dynamic_video_compression_surveillance_b200", "dropin"))
    sys.modules.pop("motion_compression_opt", None)
    import motion_compression_opt as mco
    try:
        h, w, n = 96, 128, 40
        clip = make_clip((h, w), n, seed=5)
        yy, xx = np.mgrid[0:h, 0:w]
        clip.background = np.stack([(xx * 255 // w), (yy * 255 // h), ((xx + yy) * 255 // (w + h))], -1).astype(np.uint8)
        src = str(tmp_path / "cam1.mp4")
        wr = cv2.VideoWriter(src, cv2.VideoWriter_fourcc(*"mp4v"), 30, (w, h))
        for f in clip.frames():
            wr.write(f)
        wr.release()
        cpu = _run_of(mco, monkeypatch, src, str(tmp_path / "cpu"))
        gpu = _run_of(mco, monkeypatch, src, str(tmp_path / "gpu"), flow_device="gpu")
        for out in ("cpu", "gpu"):
            vdir = os.path.join(str(tmp_path / out), "cam1")
            for name in ("overlay.mp4", "mask.mp4", "compressed.mp4", "execution_times.txt", "processing.log"):
                assert os.path.exists(os.path.join(vdir, name)), (out, name)
            txt = open(os.path.join(vdir, "execution_times.txt")).read()
            assert txt.startswith("Motion Detection:\n  Frames processed: %d\n" % (n - 1))
            assert "\nCompression:\n  Frames processed: %d\n" % (n - 1) in txt
            lines = txt.splitlines()
            assert re.fullmatch(r"  Total time: [\d\.]+ seconds", lines[2]) and lines[-1].startswith("Total video processing time: ")
        assert len(gpu["mask.mp4"]) == len(cpu["mask.mp4"]) == n - 1
        assert all(np.array_equal(a, b) for a, b in zip(gpu["overlay.mp4"], cpu["overlay.mp4"]))
        mg, mc = np.stack(gpu["mask.mp4"]), np.stack(cpu["mask.mp4"])
        diff = int(((mg != 0) != (mc != 0)).sum())
        print(f"drop-in mask.mp4 pixels differing between flow_device gpu and cpu: {diff} of {mc.size}")
        assert diff <= _rect_bound(mc.size)
        # the default run is today's host-flow run: its masks are cv2's on the decoded frames
        cap, dec = cv2.VideoCapture(src), []
        while True:
            ok, f = cap.read()
            if not ok:
                break
            dec.append(cv2.cvtColor(f, cv2.COLOR_BGR2GRAY))
        cap.release()
        from dynamic_video_compression_surveillance_b200 import host_loop
        raws = list((_masks(_cv2_flows(dec, CALL_SITE, True), 0.5)).astype(np.uint8) * 255)
        ref = host_loop.smooth_rect_masks_gpu(raws, [], 30, 0.2, 2)
        assert np.array_equal(mc, ref)
        with pytest.raises(ValueError):
            mco.temporal_smoothing_flow(src, str(tmp_path), flow_device="tpu")
    finally:
        root = logging.getLogger()
        for hd in list(root.handlers):
            if isinstance(hd, logging.FileHandler):
                root.removeHandler(hd)
                hd.close()
        sys.modules.pop("motion_compression_opt", None)
        sys.path.remove(os.path.join(ROOT, "dynamic_video_compression_surveillance_b200", "dropin"))
