"""Structuring elements larger than 33 x 33 (the k_mlarge_* path) against cv2 and the oracle loops, every byte.

Binary morphology is exact, so cv2 on the host is the answer at any size: the stage op must equal cv2.erode / cv2.dilate /
cv2.morphologyEx, and the three loops with a large dilate or close/open must equal oracle/loops.py (fd, window) and
tests/flow_loop_ref.py::flow_loop (flow) on every output frame.  Elements larger than the image are covered: only offsets
inside the image count, as in cv2 with its default borders."""
import os

import cv2
import numpy as np
import pytest
import torch

from oracle import loops, stage_ops as so
from tests.test_loop_batch_shapes_gpu import FD, LOOP, _assert_counters, _assert_equal, _check_stream, _clip, _FdOracle, \
    _run, _WindowOracle

pytestmark = pytest.mark.gpu

RECT_K = [34, 35, 63, 64, 65, 128, 129, 255, 256, 1001]
ELLIPSE_K = [34, 35, 40, 64, 65, 101, 255]
SHAPES = [(1080, 1920), (97, 131), (1, 1), (5, 4000), (4000, 37)]


@pytest.fixture(scope="module")
def P():
    from dynamic_video_compression_surveillance_b200 import pipeline
    return pipeline


def _element(kind, k):
    return np.ones((k, k), np.uint8) if kind == "rect" else cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k))


def _masks(shape, seed):
    """A blob mask (filled rectangles and ellipses of sizes up to a quarter of the frame) and dense noise (density 0.5)."""
    r = np.random.default_rng(seed)
    h, w = shape
    blob = np.zeros(shape, np.uint8)
    for _ in range(12):
        cx, cy = int(r.integers(0, w)), int(r.integers(0, h))
        ax, ay = int(r.integers(1, max(2, w // 4))), int(r.integers(1, max(2, h // 4)))
        if r.random() < 0.5:
            cv2.rectangle(blob, (cx - ax, cy - ay), (cx + ax, cy + ay), 255, -1)
        else:
            cv2.ellipse(blob, (cx, cy), (ax, ay), 0, 0, 360, 255, -1)
    noise = (r.random(shape) < 0.5).astype(np.uint8) * 255
    return np.stack([blob, noise])


OPS = (("dilate", lambda m, e: cv2.dilate(m, e)), ("erode", lambda m, e: cv2.erode(m, e)),
       ("close", lambda m, e: cv2.morphologyEx(m, cv2.MORPH_CLOSE, e)), ("open", lambda m, e: cv2.morphologyEx(m, cv2.MORPH_OPEN, e)))


def _check_stage(P, masks, kind, k):
    el = _element(kind, k)
    d = torch.from_numpy(masks).cuda()
    for op, fn in OPS:
        got = P.morph(d, op, k, kind).cpu().numpy()
        for i in range(masks.shape[0]):
            want = fn(masks[i], el)
            assert np.array_equal(got[i], want), \
                f"{kind} {k} {op} on {masks.shape[1:]}, mask {i}: {int((got[i] != want).sum())} pixels differ"


# ---------------------------------------------------------------------------------------------------------------------------
# 1: the stage op against cv2
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("kind,k", [("rect", k) for k in RECT_K] + [("ellipse", k) for k in ELLIPSE_K])
def test_stage_op_against_cv2(P, shape, kind, k):
    _check_stage(P, _masks(shape, k), kind, k)


@pytest.mark.parametrize("kind,k", [("rect", 65), ("ellipse", 64)])
def test_stage_op_7680_wide(P, kind, k):
    """A 7680-wide frame: 240 words a row, the widest the bit-plane kernels take."""
    _check_stage(P, _masks((64, 7680), 3), kind, k)


@pytest.mark.parametrize("kind", ["rect", "ellipse"])
def test_element_larger_than_the_image(P, kind):
    """1001 on 97 x 131 and 255 on 5 x 4000 (above), and the largest k: every output pixel sees the whole image, so dilate is
    'any pixel set' and erode 'every pixel set'."""
    _check_stage(P, _masks((97, 131), 1), kind, 1001)
    _check_stage(P, _masks((5, 4000), 2), kind, 255)
    m = np.zeros((3, 5, 7), np.uint8)
    m[1, 2, 3] = 255
    m[2] = 255
    d = torch.from_numpy(m).cuda()
    for op, want in (("dilate", [0, 255, 255]), ("erode", [0, 0, 255])):
        got = P.morph(d, op, 32767, kind).cpu().numpy()
        for i in range(3):
            assert (got[i] == want[i]).all(), (kind, op, i)


def test_mixed_chains(P):
    """Ellipse 2 close / open (the merged 2 x 2 pass) then a rect 45 dilate, and a large element between small ones, as
    consecutive stage calls against cv2; then window-loop chains, where small and large primitives share one handle's chain:
    small runs before a large dilate, a small dilate after large close / open, and merged small rectangles before a large one."""
    masks = _masks((300, 410), 7)
    d = torch.from_numpy(masks).cuda()
    e2, e3, r45, r70, r5 = (_element(*a) for a in (("ellipse", 2), ("ellipse", 3), ("rect", 45), ("rect", 70), ("rect", 5)))
    got = P.morph(P.morph(P.morph(d, "close", 2, "ellipse"), "open", 2, "ellipse"), "dilate", 45, "rect").cpu().numpy()
    got2 = P.morph(P.morph(P.morph(d, "close", 3, "ellipse"), "dilate", 70, "rect"), "open", 5, "rect").cpu().numpy()
    for i in range(2):
        want = cv2.dilate(cv2.morphologyEx(cv2.morphologyEx(masks[i], cv2.MORPH_CLOSE, e2), cv2.MORPH_OPEN, e2), r45)
        assert np.array_equal(got[i], want), ("ellipse 2 close, open, rect 45 dilate", i)
        want = cv2.morphologyEx(cv2.dilate(cv2.morphologyEx(masks[i], cv2.MORPH_CLOSE, e3), r70), cv2.MORPH_OPEN, r5)
        assert np.array_equal(got2[i], want), ("ellipse 3 close, rect 70 dilate, rect 5 open", i)
    h, w, n = 120, 200, 24
    clip = _clip((h, w), n + 1, 21).frames()
    seed, body = so.bgr2gray(clip[0]), torch.from_numpy(clip[1:]).cuda()
    for name, kw in (("ellipse 2 + rect 45", dict(LOOP, morph_kernel=2, kernel_size=45)),
                     ("rect 3 + rect 35 + rect 5", dict(LOOP, morph_shape="rect", morph_kernel=3, kernel_size=35)),
                     ("ellipse 41 + rect 3", dict(LOOP, morph_kernel=41, kernel_size=3))):
        ov, cp, mk, cnt = _run(P, "window", kw, body, seed, (10, 14), max_batch=16)
        exp = _check_stream(P, f"window {name}", body, ov, cp, mk, _WindowOracle(seed, kw))
        _assert_counters(f"window {name}", cnt, n, h, w, [exp])


# ---------------------------------------------------------------------------------------------------------------------------
# 2: the loops against the oracle, every output frame
# ---------------------------------------------------------------------------------------------------------------------------
LOOP_SHAPE, LOOP_N = (180, 320), 40


def _loop_case(P, mode, kw, seed_clip, batches, max_batch, handoff_before=None):
    h, w = LOOP_SHAPE
    clip = _clip(LOOP_SHAPE, LOOP_N + 1, seed_clip).frames()
    body = torch.from_numpy(clip[1:]).cuda()
    seed = so.bgr2gray(clip[0]) if mode == "window" else loops.first_frame_gray_fd(clip[0])
    oracle = _WindowOracle(seed, kw) if mode == "window" else _FdOracle(seed, kw)
    case = f"{mode} {kw}"
    ov, cp, mk, cnt = _run(P, mode, kw, body, seed, batches, max_batch=max_batch, handoff_before=handoff_before)
    masks = []
    exp = _check_stream(P, case, body, ov, cp, mk, oracle, samples=(0, LOOP_N - 1),
                        seen=lambda r: masks.extend(r["acc"] if mode == "fd" else r["mask"]))
    _assert_counters(case, cnt, LOOP_N, h, w, [exp])
    m = np.stack(masks)
    assert m.any() and not m.all(), f"{case}: degenerate masks"


@pytest.mark.parametrize("k", [35, 63])
def test_fd_loop_large_dilate(P, k):
    _loop_case(P, "fd", dict(FD, kernel_size=k), 31, (16, 16, 8), 16)


def test_window_loop_large_close_open_and_dilate(P):
    _loop_case(P, "window", dict(LOOP, morph_kernel=40, morph_shape="ellipse", kernel_size=45), 32, (16, 16, 8), 16)


@pytest.mark.parametrize("mode", ["fd", "window"])
def test_loop_batch_split_with_state_hand_off(P, mode):
    """Batches of 7, 13, 20 with the state moving to a new handle before the second."""
    kw = dict(FD, kernel_size=41) if mode == "fd" else dict(LOOP, morph_kernel=37, morph_shape="rect", kernel_size=0)
    _loop_case(P, mode, kw, 33, (7, 13, 20), 20, handoff_before=1)


def test_stream_group_equals_solo_handles(P):
    """A 4-stream window group with a large close/open and dilate: every stream equals a solo handle byte for byte."""
    S, T, (h, w) = 4, 12, LOOP_SHAPE
    kw = dict(LOOP, morph_kernel=36, morph_shape="ellipse", kernel_size=50)
    clips = [_clip(LOOP_SHAPE, 2 * T + 1, 40 + s).frames() for s in range(S)]
    seeds = np.stack([so.bgr2gray(c[0]) for c in clips])
    body = torch.from_numpy(np.stack([c[1:] for c in clips])).cuda()
    ov, cp, mk, cnt = _run(P, "window", kw, body, seeds, (T, T), max_batch=T, n_streams=S)
    for s in range(S):
        o, c, m, _ = _run(P, "window", kw, body[s].contiguous(), seeds[s], (T, T), max_batch=T)
        _assert_equal(mk[s], m, f"stream group, stream {s}", "mask vs solo handle")
        _assert_equal(ov[s], o, f"stream group, stream {s}", "overlay vs solo handle")
        _assert_equal(cp[s], c, f"stream group, stream {s}", "compressed frame vs solo handle")
    ref, _ = _WindowOracle(seeds[0], kw)(body[0].cpu().numpy())
    _assert_equal(mk[0], ref, "stream group, stream 0", "mask vs oracle")


def test_flow_loop_large_close_open():
    from tests.test_flow_loop_gpu import _check
    _check("flow ellipse 35", (240, 352, 25, 41), (("window_size", 5), ("morph_kernel", 35)), [8, 5], 8)
    _check("flow rect 34", (240, 352, 25, 41), (("window_size", 5), ("morph_kernel", 34), ("morph_shape", "rect")), [24], 24)


# ---------------------------------------------------------------------------------------------------------------------------
# 3: the drop-in and the argument codes
# ---------------------------------------------------------------------------------------------------------------------------
def test_dropin_fd_kernel_size_41(tmp_path, monkeypatch):
    """process_single_video_fd(..., kernel_size=41) writes both videos; the frames it hands the writers equal the oracle on
    the decoded frames (overlay) and the degrade of the oracle's accumulator (compressed)."""
    from tests.test_dropin_gpu import DROPIN, _read_all, _smooth_clip, _write_clip
    from dynamic_video_compression_surveillance_b200 import pipeline as P
    monkeypatch.syspath_prepend(DROPIN)
    import sys
    sys.modules.pop("frame_differencing", None)
    import frame_differencing as fd
    h, w, n = 96, 128, 30
    src = str(tmp_path / "cam41.mp4")
    _write_clip(src, _smooth_clip(h, w, n, 11))
    dec = _read_all(src)
    written = {}
    real = cv2.VideoWriter

    class Recorder:
        def __init__(self, path, *a):
            self.inner, self.sink = real(path, *a), written.setdefault(os.path.basename(path), [])

        def write(self, frame):
            self.sink.append(np.array(frame))
            self.inner.write(frame)

        def release(self):
            self.inner.release()

    monkeypatch.setattr(fd.cv2, "VideoWriter", Recorder)
    fd.process_single_video_fd(src, str(tmp_path / "out"), kernel_size=41)
    monkeypatch.setattr(fd.cv2, "VideoWriter", real)
    sys.modules.pop("frame_differencing", None)
    vdir = tmp_path / "out" / "cam41"
    ov_name, cp_name = "dilated_motion_mask_video.mp4", "compressed_final_video.mp4"
    for name in (ov_name, cp_name):
        assert len(_read_all(str(vdir / name))) == n - 1, name
    ref = loops.fd_loop(dec, kernel_size=41, degrade=False)
    assert len(written[ov_name]) == len(written[cp_name]) == n - 1
    frames = torch.from_numpy(np.stack(dec[1:])).cuda()
    want_cp, _ = P.degrade_blend(frames, torch.from_numpy(np.stack(ref["acc"])).cuda(), 4, 100, "fd", False)
    want_cp = want_cp.cpu().numpy()
    for t in range(n - 1):
        assert np.array_equal(written[ov_name][t], ref["overlay"][t]), f"drop-in frame {t + 1}: overlay"
        assert np.array_equal(written[cp_name][t], want_cp[t]), f"drop-in frame {t + 1}: compressed"
    assert any((a > 127).any() for a in ref["acc"])


def test_argument_codes(P):
    from dynamic_video_compression_surveillance_b200._lib import DVC_ERR_UNSUPPORTED, DvcError

    def code(fn):
        with pytest.raises(DvcError) as e:
            fn()
        return e.value.code

    m = torch.zeros((1, 8, 8), dtype=torch.uint8, device="cuda")
    for kind in ("rect", "ellipse"):
        assert code(lambda: P.morph(m, "dilate", 32768, kind)) == DVC_ERR_UNSUPPORTED
        assert code(lambda: P.morph(m, "dilate", 0, kind)) == DVC_ERR_UNSUPPORTED
    assert code(lambda: P.FramePipeline(64, 48, "fd", kernel_size=32768)) == DVC_ERR_UNSUPPORTED
    assert code(lambda: P.FramePipeline(64, 48, "window", morph_kernel=32768)) == DVC_ERR_UNSUPPORTED
    assert code(lambda: P.FramePipeline(64, 48, "flow", morph_kernel=32768)) == DVC_ERR_UNSUPPORTED
    assert code(lambda: P.morph(torch.zeros((1, 4, 8200), dtype=torch.uint8, device="cuda"), "dilate", 40)) == DVC_ERR_UNSUPPORTED
