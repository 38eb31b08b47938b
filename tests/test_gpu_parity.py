"""GPU parity: every kernel behind the C ABI against the CPU oracle (run on the B200 box, `-m gpu`).

Bar (BASELINE.json north_star): masks bit-exact; frames bit-exact where the reference uses integer OpenCV
ops; DCT-degraded blocks bit-exact when this host's cv2 follows the recovered float32 sequences (4x4, 8x8 and every
clipped shape: oracle/stage_ops.py closed forms, checked per shape on this host), otherwise within 1 quantised-channel
level away from exact quantiser ties, with tie-block count, flipped-block count and PSNR reported.
"""
import os

import cv2
import numpy as np
import pytest
import torch

from oracle import loops, stage_ops as so
from tests.golden_util import FD_CLIPPED_FIXTURE, FD_FIXTURES, GOLDEN, OF_FIXTURES, load_fd, load_of, sha, unpack

pytestmark = pytest.mark.gpu

SHAPES = [(1, 1), (1, 7), (5, 1), (2, 2), (3, 5), (17, 33), (48, 64), (101, 67), (96, 256), (130, 400)]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


@pytest.fixture(scope="module")
def P():
    from dynamic_video_compression_surveillance_b200 import pipeline
    return pipeline


def rng(seed):
    return np.random.default_rng(seed)


@pytest.mark.parametrize("shape", SHAPES)
def test_bgr2gray(P, shape):
    img = rng(1).integers(0, 256, (3,) + shape + (3,), dtype=np.uint8)
    got = host(P.bgr2gray(dev(img)))
    for i in range(3):
        assert np.array_equal(got[i], so.bgr2gray(img[i]))


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("blur5", [False, True])
def test_gray_absdiff_thresh(P, shape, blur5):
    r = rng(2)
    n = 11
    base = r.integers(0, 256, shape + (3,), dtype=np.uint8)
    frames = np.stack([base.copy() for _ in range(n)])
    for t in range(n):                                   # sparse changes so masks are not trivially full
        m = r.random(shape) < 0.2
        frames[t][m] = r.integers(0, 256, (int(m.sum()), 3), dtype=np.uint8)
    prev = r.integers(0, 256, shape, dtype=np.uint8)
    for thr in (0.5, 3.0):
        gray, mask = P.gray_absdiff_thresh(dev(frames), dev(prev), thr, blur5)
        gray, mask = host(gray), host(mask)
        p = prev
        for t in range(n):
            g = so.bgr2gray(frames[t])
            if blur5:
                g = so.gaussian_blur5(g)
            assert np.array_equal(gray[t], g), (t, "gray")
            assert np.array_equal(mask[t], so.threshold_binary(so.absdiff(p, g), thr)), (t, "mask")
            p = g


@pytest.mark.parametrize("shape", [(1, 1), (3, 5), (17, 33), (48, 70), (101, 130), (64, 300)])
@pytest.mark.parametrize("kind,k", [("rect", 1), ("rect", 2), ("rect", 3), ("rect", 5), ("rect", 7), ("rect", 9), ("rect", 10), ("rect", 11),
                                    ("rect", 13), ("rect", 15), ("rect", 33), ("ellipse", 2), ("ellipse", 3), ("ellipse", 5), ("ellipse", 9)])
def test_morphology(P, shape, kind, k):
    r = rng(5)
    kernel = so.structuring_rect(k) if kind == "rect" else so.structuring_ellipse(k)
    masks = np.stack([(r.random(shape) < d).astype(np.uint8) * 255 for d in (0.02, 0.5, 0.97, 0.0, 1.0)])
    d = dev(masks)
    for op, fn in (("dilate", so.dilate), ("erode", so.erode), ("close", so.morph_close), ("open", so.morph_open)):
        got = host(P.morph(d, op, k, kind))
        for i in range(len(masks)):
            assert np.array_equal(got[i], fn(masks[i], kernel)), (op, i)


def test_morphology_tall_image_bands(P):
    r = rng(6)
    masks = np.stack([(r.random((1200, 96)) < d).astype(np.uint8) * 255 for d in (0.01, 0.6)])
    for kind, k in (("rect", 15), ("ellipse", 7)):
        kernel = so.structuring_rect(k) if kind == "rect" else so.structuring_ellipse(k)
        got = host(P.morph(dev(masks), "close", k, kind))
        for i in range(2):
            assert np.array_equal(got[i], cv2.morphologyEx(masks[i], cv2.MORPH_CLOSE, kernel))


@pytest.mark.parametrize("alpha,K", [(0.2, 30), (0.2, 5), (0.5, 4), (0.34, 7), (1.0, 3), (0.0, 3), (0.2, 1), (0.9, 31), (0.3, 32), (0.55, 60),
                                     (1.0, 127), (0.01, 100)])
def test_temporal_ring(P, alpha, K):
    r = rng(7)
    n, shape = (70 if K <= 31 else 170), (37, 83)
    masks = np.stack([(r.random(shape) < 0.3).astype(np.uint8) * 255 for _ in range(n)])
    got = host(P.temporal_ring(dev(masks), K, alpha))
    for t in range(n):
        ref = so.window_vote(list(masks[max(0, t - K + 1):t + 1]), alpha)
        assert np.array_equal(got[t], ref), t


@pytest.mark.parametrize("rf", [0.5, 0.3, 0.1, 0.7, 0.9, 1 / 3])
def test_temporal_ema(P, rf):
    r = rng(8)
    n, shape = 40, (33, 70)
    dil = np.stack([(r.random(shape) < 0.4).astype(np.uint8) * 255 for _ in range(n)])
    acc0 = r.integers(0, 256, shape, dtype=np.uint8)
    acc = dev(acc0.copy())
    got = host(P.temporal_ema(acc, dev(dil), rf))
    a = acc0
    for t in range(n):
        a = cv2.addWeighted(a, rf, dil[t], 1 - rf, 0)
        assert np.array_equal(got[t], a), t
    assert np.array_equal(host(acc), a)


def test_temporal_ema_all_accumulator_values(P):
    a0 = np.tile(np.arange(256, dtype=np.uint8), (2, 1))           # [2,256]: row 0 sees dil=0, row 1 dil=255
    dil = np.stack([np.stack([np.zeros(256, np.uint8), np.full(256, 255, np.uint8)])])
    for rf in (0.5, 0.3, 0.05, 0.95, 0.7):
        acc = dev(a0.copy())
        got = host(P.temporal_ema(acc, dev(dil), rf))[0]
        assert np.array_equal(got, cv2.addWeighted(a0, rf, dil[0], 1 - rf, 0)), rf


@pytest.mark.parametrize("ksize,sigma", [(25, 30.0), (5, 0), (3, 0), (7, 2.3), (11, 3.0), (31, 10.0), (33, 12.0), (1, 0)])
def test_gaussian_blur(P, ksize, sigma):
    """cv2.GaussianBlur on uint8 (frame_differencing.py:77: the first frame's (25, 25), sigma 30; :93): fixed point, exact."""
    r = rng(ksize)
    for shape in [(96, 128), (70, 91), (64, 14), (270, 480)]:
        img = r.integers(0, 256, (2,) + shape, dtype=np.uint8)
        got = host(P.gaussian_blur(dev(img), ksize, sigma))
        for i in range(2):
            assert np.array_equal(got[i], cv2.GaussianBlur(img[i], (ksize, ksize), sigma)), (ksize, sigma, shape)


@pytest.mark.parametrize("mode", ["fd", "window"])
@pytest.mark.parametrize("scale", [1.0, 0.5])
def test_begin_stream_frames_does_the_first_frame_work_on_the_gpu(P, mode, scale):
    """dvc_begin_stream_frames: resize + BGR2GRAY + (fd) GaussianBlur((25, 25), 30) of the first frame on the GPU
    (frame_differencing.py:74-77) must seed exactly the state the host-side cv2 calls seed."""
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    sh, sw, n = 128, 192, 10
    frames = make_clip((sh, sw), n, seed=77).frames()
    w, h = int(sw * scale), int(sh * scale)
    kw = dict(min_area=40) if mode == "fd" else dict(window_size=3, alpha_fraction=0.4)
    first = frames[0] if scale == 1.0 else cv2.resize(frames[0], (w, h))
    seed = loops.first_frame_gray_fd(first) if mode == "fd" else so.bgr2gray(first)
    outs = []
    for use_frames in (False, True):
        pipe = P.FramePipeline(w, h, mode, max_batch=4, src_size=(sw, sh) if scale != 1.0 else None, **kw)
        if use_frames:
            pipe.begin_stream_frames(frames[0])
        else:
            pipe.begin_stream(seed)
        ov = np.empty((n - 1, h, w, 3), np.uint8); cp = np.empty_like(ov); mk = np.empty((n - 1, h, w), np.uint8)
        pipe.process_host(np.ascontiguousarray(frames[1:]), ov, cp, mk)
        pipe.close()
        outs.append((ov, cp, mk))
    for a, b in zip(outs[0], outs[1]):
        assert np.array_equal(a, b)
    assert outs[0][2].any()


def _blob_mask(r, shape, n):
    m = np.zeros(shape, np.uint8)
    h, w = shape
    for _ in range(n):
        kind = r.integers(0, 3)
        cx, cy = int(r.integers(0, w)), int(r.integers(0, h))
        if kind == 0:
            cv2.circle(m, (cx, cy), int(r.integers(1, 25)), 255, int(r.choice([-1, 1, 2, 3])))
        elif kind == 1:
            cv2.rectangle(m, (cx, cy), (cx + int(r.integers(1, 40)), cy + int(r.integers(1, 40))), 255, int(r.choice([-1, 1, 2])))
        else:
            cv2.line(m, (cx, cy), (int(r.integers(0, w)), int(r.integers(0, h))), 255, int(r.integers(1, 4)))
    noise = r.random(shape) < 0.02
    m[noise] = 255 - m[noise]
    return m


@pytest.mark.parametrize("shape", [(96, 128), (61, 83), (120, 160), (32, 200), (7, 5), (1, 40)])
def test_contour_filter(P, shape):
    r = rng(9)
    masks = [_blob_mask(r, shape, int(r.integers(1, 12))) for _ in range(10)]
    masks += [(r.random(shape) < d).astype(np.uint8) * 255 for d in (0.3, 0.5, 0.6, 0.8, 0.0, 1.0)]
    masks = np.stack(masks)
    for min_area in (0, 5, 20, 100, 500):
        got = host(P.contour_filter(dev(masks), min_area))
        for i in range(len(masks)):
            assert np.array_equal(got[i], so.contour_filter_cv2(masks[i], min_area)), (i, min_area)


@pytest.mark.parametrize("shape", [(96, 128), (61, 83), (120, 160), (32, 200), (7, 5), (1, 40), (270, 480)])
def test_mask_rectangles(P, shape):
    r = rng(19)
    masks = [_blob_mask(r, shape, int(r.integers(1, 12))) for _ in range(8)]
    masks += [(r.random(shape) < d).astype(np.uint8) * 255 for d in (0.002, 0.03, 0.3, 0.6, 0.0, 1.0)]
    masks = np.stack(masks)
    got = host(P.mask_rectangles(dev(masks)))
    for i in range(len(masks)):
        assert np.array_equal(got[i], so.mask_rectangles_cv2(masks[i])), i


def test_mask_rectangles_1080p(P):
    r = rng(20)
    m = np.zeros((2, 1080, 1920), np.uint8)
    for k in range(2):
        for _ in range(40):
            cx, cy = int(r.integers(0, 1920)), int(r.integers(0, 1080))
            cv2.ellipse(m[k], (cx, cy), (int(r.integers(3, 120)), int(r.integers(3, 80))), float(r.integers(0, 180)), 0, 360, 255,
                        int(r.choice([-1, 2, 5])))
        noise = r.random(m[k].shape) < 0.0005
        m[k][noise] = 255
    got = host(P.mask_rectangles(dev(m)))
    for k in range(2):
        assert np.array_equal(got[k], so.mask_rectangles_cv2(m[k]))


@pytest.mark.parametrize("shape", [(48, 64), (120, 160), (37, 53), (270, 480), (1080, 1920)])
def test_resize_linear(P, shape):
    r = rng(56)
    h, w = shape
    img = r.integers(0, 256, (2, h, w, 3), dtype=np.uint8)
    for sf in ((0.5, 1.5, 0.3) if h >= 1080 else (0.5, 0.75, 0.3, 0.9, 0.25, 0.6, 0.99, 0.123, 1.0, 1.1, 1.5, 2.0)):
        dw, dh = int(w * sf), int(h * sf)
        if dw < 1 or dh < 1:
            continue
        got = host(P.resize_linear(dev(img), (dw, dh)))
        for i in range(2):
            assert np.array_equal(got[i], cv2.resize(img[i], (dw, dh))), (shape, sf, i)
    g = np.ascontiguousarray(img[..., 1])
    got = host(P.resize_linear(dev(g), (w // 2, h // 2)))
    assert np.array_equal(got[0], cv2.resize(g[0], (w // 2, h // 2)))


def test_bgr2gray_all_colours(P):
    """Every one of the 2^24 BGR triples through the IDP.2A gray conversion (K1 / blur kernels share it)."""
    v = np.arange(1 << 24, dtype=np.uint32)
    img = np.stack([v & 0xff, (v >> 8) & 0xff, v >> 16], axis=-1).astype(np.uint8).reshape(1, 4096, 4096, 3)
    got = host(P.bgr2gray(dev(img)))[0]
    assert np.array_equal(got, so.bgr2gray(img[0]))


def test_mask_rectangles_max_runs_per_word(P):
    """Isolated pixels on a 2-pixel grid: 16 runs in every word (all overflow slots of the run graph in use), one component
    per pixel; and a one-pixel checkerboard, which is a single 8-connected component."""
    grid = np.zeros((64, 160), np.uint8)
    grid[::2, ::2] = 255
    chk = ((np.add.outer(np.arange(48), np.arange(100)) & 1) * 255).astype(np.uint8)
    for m in (grid, np.ascontiguousarray(grid[:, 1:]), chk):
        got = host(P.mask_rectangles(dev(m[None])))[0]
        assert np.array_equal(got, so.mask_rectangles_cv2(m))
        assert np.array_equal(host(P.contour_filter(dev(m[None]), 0))[0], so.contour_filter_cv2(m, 0))


def test_contour_filter_1080p_blobs(P):
    r = rng(10)
    m = np.zeros((1080, 1920), np.uint8)
    for _ in range(60):
        cx, cy = int(r.integers(0, 1920)), int(r.integers(0, 1080))
        cv2.ellipse(m, (cx, cy), (int(r.integers(3, 120)), int(r.integers(3, 80))), float(r.integers(0, 180)), 0, 360, 255,
                    int(r.choice([-1, 2, 5])))
    noise = r.random(m.shape) < 0.01
    m[noise] = 255 - m[noise]
    got = host(P.contour_filter(dev(m[None]), 500))[0]
    assert np.array_equal(got, so.contour_filter_cv2(m, 500))


def _serpentine(h, w, r, gaps=1):
    """Walls on every other row with one opening at alternating ends: the background is one long corridor, so the flood of
    the contour filter's phase A has to travel every row (many sweep iterations), plus a little noise."""
    m = np.zeros((h, w), np.uint8)
    for y in range(1, h, 2):
        m[y, :] = 255
        m[y, (w - 1) if (y // 2) % 2 else 0] = 0
    noise = r.random((h, w)) < 0.01
    m[noise] = 255 - m[noise]
    return m


@pytest.mark.parametrize("shape", [(40, 2100), (23, 4200), (9, 1999), (300, 700), (200, 300), (1, 1), (2, 130), (17, 64), (33, 65), (3000, 70)])
def test_contour_filter_sweep_cases(P, shape):
    """Shapes and masks aimed at the one-launch sweep kernel (k_ccl_sweep.cuh): rows of two and four 64-bit words per lane,
    fewer rows than warps, runs and holes across word boundaries, long flood paths, more row runs than fit in shared
    memory (dense noise: global node arrays), and more frames than one launch takes."""
    r = rng(31)
    h, w = shape
    masks = [_blob_mask(r, shape, int(r.integers(3, 30))) for _ in range(3)]
    masks += [(r.random(shape) < d).astype(np.uint8) * 255 for d in (0.45, 0.7)]
    masks.append(_serpentine(h, w, r))
    ring = np.zeros(shape, np.uint8)                      # nested frames: holes inside holes, edges on word boundaries
    for k in range(0, min(h, w) // 2, 3):
        ring[k:h - k, k:w - k] = 255 if (k // 3) % 2 == 0 else 0
    masks.append(ring)
    bars = np.zeros(shape, np.uint8)                      # runs that start / end exactly at 64-pixel boundaries
    bars[::3, 64 * (w // 128):] = 255
    bars[1::3, :64 * (w // 128 + 1)] = 255
    masks.append(bars)
    masks = np.stack(masks)
    for min_area in (0, 3, 50):
        got = host(P.contour_filter(dev(masks), min_area))
        for i in range(len(masks)):
            assert np.array_equal(got[i], so.contour_filter_cv2(masks[i], min_area)), (shape, i, min_area)


def test_contour_filter_many_frames(P):
    r = rng(32)
    masks = np.stack([_blob_mask(r, (50, 90), int(r.integers(1, 9))) for _ in range(75)])
    got = host(P.contour_filter(dev(masks), 4))
    for i in range(len(masks)):
        assert np.array_equal(got[i], so.contour_filter_cv2(masks[i], 4)), i


def test_contour_filter_1080p_frames_and_noise(P):
    """The bench's kind of mask (outlines of rectangles: big holes) and dense noise at full size."""
    r = rng(33)
    a = np.zeros((1080, 1920), np.uint8)
    for (x, y, ww, hh) in ((100, 50, 240, 135), (300, 120, 256, 143), (1500, 800, 272, 151), (900, 400, 288, 159), (0, 900, 200, 180)):
        a[y:y + hh, x:x + ww] = 255
        a[y + 6:y + hh - 6, x + 8:x + ww - 8] = 0
    b = (r.random((1080, 1920)) < 0.5).astype(np.uint8) * 255
    c = _serpentine(1080, 1920, r)
    for m, min_area in ((a, 500), (b, 2), (c, 500)):
        got = host(P.contour_filter(dev(m[None]), min_area))[0]
        assert np.array_equal(got, so.contour_filter_cv2(m, min_area))


def _exact(bs, h=None, w=None):
    """Does this host's cv2 follow the recovered float32 sequences for every block shape a (h, w) frame cut into
    bs x bs blocks produces?  (True on the AVX-512 IPP build of the image; when False the tests fall back to the
    tie-classified tolerance bar and print the report.)"""
    ok = so.cv2_dct4_matches_closed_form() if bs == 4 else so.cv2_dct_matches_closed_form(bs, bs)
    if h is not None:
        rh, rw = h % bs, w % bs
        for sh in {(rh, bs), (bs, rw), (rh, rw)}:
            if sh[0] and sh[1] and sh != (bs, bs) and (h >= sh[0]) and (w >= sh[1]):
                ok = ok and so.cv2_dct_matches_closed_form(min(sh[0], h), min(sh[1], w))
    return ok


def _degrade_report(got, ref, planes, static, bs, q, max_off_tie, label=""):
    """Tolerance bar for hosts whose cv2 does not follow the closed forms: integer pixels exact, static blocks within
    `max_off_tie` away from blocks holding an exact quantiser tie in any quantised plane; prints tie-block count,
    flipped-block count and PSNR (SURVEY.md section 8d)."""
    h, w = static.shape[0] * bs, static.shape[1] * bs
    got, ref = got[:h, :w], ref[:h, :w]
    st_px = np.repeat(np.repeat(static, bs, 0), bs, 1)
    assert np.array_equal(got[~st_px], ref[~st_px])
    tie = np.zeros_like(static)
    for pl in planes:
        tie |= so.tie_blocks(pl[:h, :w], static, bs, q)
    tie_px = np.repeat(np.repeat(tie, bs, 0), bs, 1)
    d = np.abs(got.astype(int) - ref.astype(int))
    d = d.max(axis=2) if d.ndim == 3 else d
    flipped = (d.reshape(static.shape[0], bs, static.shape[1], bs).max(axis=(1, 3)) > max_off_tie) & static
    mse = np.mean((got.astype(float) - ref.astype(float)) ** 2)
    psnr = float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)
    print(f"[degrade report{label}] static blocks {int(static.sum())}, tie blocks {int(tie.sum())}, "
          f"flipped blocks {int(flipped.sum())}, max off-tie diff {int(d[st_px & ~tie_px].max(initial=0))}, PSNR {psnr:.2f} dB")
    assert d[st_px & ~tie_px].max(initial=0) <= max_off_tie
    assert not (flipped & ~tie).any()
    assert psnr > 40


def _check_degraded(got, ref, frame, acc, bs, q, exact):
    """Integer pixels must match; DCT blocks exactly (exact=True) or within 1 LSB away from ties."""
    if exact:
        assert np.array_equal(got, ref)
        return
    h, w = (acc.shape[0] // bs) * bs, (acc.shape[1] // bs) * bs
    static = so.block_all_zero(acc[:h, :w], bs)
    _degrade_report(got, ref, [so.bgr2ycrcb(frame)[..., 0]], static, bs, q, 1)


def _check_degraded_mco(got, ref, frame, mask, q=100):
    """MCO flavour (three quantised planes, then YCrCb -> BGR -> gray): exact when cv2 follows the 8x8 closed form, else
    within 2 grey levels (one level in each quantised plane) away from tie blocks, reported."""
    if so.cv2_dct_matches_closed_form(8, 8):
        assert np.array_equal(got, ref)
        return
    static = so.block_all_zero(mask, 8, full_blocks_only=True)[:mask.shape[0] // 8, :mask.shape[1] // 8]
    ycc = so.bgr2ycrcb(frame)
    _degrade_report(got, ref, [ycc[..., c] for c in range(3)], static, 8, q, 2, " mco")


@pytest.mark.parametrize("bh", range(1, 9))
@pytest.mark.parametrize("bw", range(1, 9))
def test_dct_blocks_match_cv2(P, bh, bw):
    """The float32 transform pair itself (dvc_dct_blocks_f32) against cv2.dct / cv2.idct on random blocks of every shape
    a clipped block can take: pixel-like integers, generic floats and quantised coefficients; equality of every bit."""
    if (bh, bw) == (1, 1):
        pytest.skip("1 x 1 is the identity")
    if not so.cv2_dct_matches_closed_form(bh, bw):
        pytest.skip("host cv2 does not follow the recovered float32 sequence for this shape")
    r = rng(100 * bh + bw)
    n = 3000
    xi = r.integers(-128, 128, (n, bh, bw)).astype(np.float32)
    xg = (r.standard_normal((n, bh, bw)) * 70).astype(np.float32)
    for x in (xi, xg):
        f = np.stack([cv2.dct(b) for b in x])
        assert np.array_equal(host(P.dct_blocks(dev(x))), f), ("forward", bh, bw)
        for q in (100.0, 7.5):
            qd = (np.round(f / np.float32(q)) * np.float32(q)).astype(np.float32)
            assert np.array_equal(host(P.dct_blocks(dev(qd), inverse=True)), np.stack([cv2.idct(b) for b in qd])), ("inverse", bh, bw, q)


@pytest.mark.parametrize("q", [100.0, 33.3, 8, 1, 0.3, 0.05])
@pytest.mark.parametrize("flavour", ["fd", "mco"])
def test_degrade_8x8_exact_on_many_dense_blocks(P, q, flavour):
    """block_size 8 (frame_differencing.py:203 / motion_compression_opt.py:156-183), 4 800 random blocks per level, all static:
    exact equality with the reference arithmetic, small q keeping every coefficient alive."""
    if not so.cv2_dct_matches_closed_form(8, 8):
        pytest.skip("host cv2 does not follow the recovered float32 8x8 sequence; covered by the tolerance bar")
    r = rng(6)
    t, h, w = 2, 240, 640
    frames = r.integers(0, 256, (t, h, w, 3), dtype=np.uint8)
    frames[1] = (frames[1] // 8) * 8
    acc = np.zeros((t, h, w), np.uint8)
    comp = host(P.degrade_blend(dev(frames), dev(acc), 8, q, flavour, False)[0])
    for i in range(t):
        ref = so.degrade_fd(frames[i], acc[i], 8, q) if flavour == "fd" else so.degrade_mco(frames[i], acc[i], q)
        bad = (comp[i] != ref).any(axis=2).reshape(h // 8, 8, w // 8, 8).any(axis=(1, 3)).sum()
        assert bad == 0, (q, flavour, i, int(bad))


@pytest.mark.parametrize("shape,bs", [((48, 64), 4), ((96, 128), 4), ((44, 60), 4), ((48, 64), 8), ((40, 72), 8)])
def test_degrade_fd(P, shape, bs):
    r = rng(11)
    exact = _exact(bs)
    frames = r.integers(0, 256, (3,) + shape + (3,), dtype=np.uint8)
    frames[1] = (frames[1] // 16) * 16                                    # flatter content: DC-dominated blocks
    frames[2, :, :, :] = np.linspace(0, 255, shape[1], dtype=np.uint8)[None, :, None]
    acc = np.zeros((3,) + shape, np.uint8)
    acc[:, 10:30, 20:40] = r.integers(0, 256, (3, 20, 20), dtype=np.uint8)
    acc[1, 5, 7] = 1
    cnt = torch.zeros(5, dtype=torch.int64, device="cuda")
    comp, ov = P.degrade_blend(dev(frames), dev(acc), bs, 100, "fd", True, cnt)
    comp, ov = host(comp), host(ov)
    n_static = 0
    for i in range(3):
        assert np.array_equal(ov[i], so.overlay_paint(frames[i], acc[i]))
        _check_degraded(comp[i], so.degrade_fd(frames[i], acc[i], bs, 100), frames[i], acc[i], bs, 100, exact)
        n_static += int(so.block_all_zero(acc[i], bs).sum())
    c = host(cnt)
    assert c[0] == 3 and c[1] == 3 * shape[0] * shape[1]
    assert c[2] == int((acc > 127).sum())
    assert c[3] == 3 * (shape[0] // bs) * (shape[1] // bs) and c[4] == n_static


@pytest.mark.parametrize("q", [100, 100.0, 33.3, 8, 7.5, 1, 250, 0.25, 0.3, 7.3, 0.05, 1000.5, 0.005, 2e6])
def test_degrade_fd_quantiser_ties_and_levels(P, q):
    """Blocks built to sit exactly on quantiser ties (d/q = n + 1/2) and a sweep of quantisation levels,
    including levels outside [0.01, 1e6], which the packed kernels leave to the general one."""
    if not so.cv2_dct4_matches_closed_form():
        pytest.skip("host cv2 does not follow the recovered float32 DCT sequence; covered by tolerance tests")
    r = rng(21)
    h, w = 64, 96                                       # W % 16 == 0
    frames = np.empty((4, h, w, 3), np.uint8)
    # grey frames: Y == value.  4x4 blocks whose DC = sum(Y-128)/4 is an exact multiple of q/2 when q = 100
    base = r.integers(100, 160, (h // 4, w // 4), dtype=np.int64)
    img = np.repeat(np.repeat(base, 4, 0), 4, 1)
    pat = np.zeros((4, 4), np.int64); pat[:2] = 1          # 8 pixels +1 -> sum shifts by 8
    img = img + np.tile(pat, (h // 4, w // 4))
    frames[0] = np.clip(img, 0, 255).astype(np.uint8)[..., None]
    frames[1] = r.integers(0, 256, (h, w, 1), dtype=np.uint8)
    frames[2] = r.integers(0, 256, (h, w, 3), dtype=np.uint8)
    frames[3] = (r.integers(0, 4, (h, w, 3)) * 85).astype(np.uint8)
    acc = np.zeros((4, h, w), np.uint8)
    comp, _ = P.degrade_blend(dev(frames), dev(acc), 4, q, "fd", False)
    comp = host(comp)
    for i in range(4):
        assert np.array_equal(comp[i], so.degrade_fd(frames[i], acc[i], 4, q)), (q, i)


@pytest.mark.parametrize("shape", [(48, 72), (8, 8), (4, 24), (100, 104), (8, 2064), (12, 2056), (8, 4112), (4, 16), (260, 16)])
def test_degrade_fd_widths_multiple_of_8(P, shape):
    # (8, 2064): row split into uneven parts; (12, 2056): W > 2048 and W % 16 != 0 (falls back to the non-ring kernel);
    # (260, 16): many block rows per tile, last tile of a frame shorter
    r = rng(22)
    exact = so.cv2_dct4_matches_closed_form()
    frames = r.integers(0, 256, (2,) + shape + (3,), dtype=np.uint8)
    acc = (r.random((2,) + shape) < 0.01).astype(np.uint8) * r.integers(1, 256, (2,) + shape, dtype=np.uint8)
    comp, ov = P.degrade_blend(dev(frames), dev(acc), 4, 100, "fd", True)
    comp, ov = host(comp), host(ov)
    for i in range(2):
        assert np.array_equal(ov[i], so.overlay_paint(frames[i], acc[i]))
        _check_degraded(comp[i], so.degrade_fd(frames[i], acc[i], 4, 100), frames[i], acc[i], 4, 100, exact)


@pytest.mark.parametrize("offset", [1, 8, 16])
@pytest.mark.parametrize("shape,bs", [((48, 64), 4), ((12, 2056), 4), ((48, 64), 8), ((12, 2056), 8)])
def test_degrade_fd_any_frame_alignment(P, shape, bs, offset):
    """Frames at byte offsets 1, 8 and 16 inside a larger allocation: kernels that need 8- or 16-byte aligned addresses
    (8-byte vector access, the ring's bulk copies) give way to ones that do not, with the outputs and counters of the
    aligned call."""
    r = rng(24)
    h, w = shape
    frames = r.integers(0, 256, (2, h, w, 3), dtype=np.uint8)
    acc = (r.random((2, h, w)) < 0.01).astype(np.uint8) * r.integers(1, 256, (2, h, w), dtype=np.uint8)
    buf = torch.empty(frames.size + 16, dtype=torch.uint8, device="cuda")
    shifted = buf[offset:offset + frames.size].view(frames.shape)
    shifted.copy_(dev(frames))
    assert shifted.data_ptr() % 16 == offset % 16
    outs = []
    for bgr in (dev(frames), shifted):
        cnt = torch.zeros(5, dtype=torch.int64, device="cuda")
        comp, ov = P.degrade_blend(bgr, dev(acc), bs, 100, "fd", True, cnt)
        outs.append((host(comp), host(ov), host(cnt)))
    for aligned, unaligned in zip(*outs):
        assert np.array_equal(aligned, unaligned)
    comp, ov, c = outs[1]
    exact = _exact(bs, h, w)
    hf, wf = (h // bs) * bs, (w // bs) * bs
    for i in range(2):
        ref = so.degrade_fd(frames[i], acc[i], bs, 100)
        assert np.array_equal(ov[i], so.overlay_paint(frames[i], acc[i]))
        if exact:
            assert np.array_equal(comp[i], ref)
        else:
            _check_degraded(comp[i][:hf, :wf], ref[:hf, :wf], frames[i][:hf, :wf], acc[i][:hf, :wf], bs, 100, False)
    assert c[2] == int((acc > 127).sum())
    assert c[4] == sum(int(so.block_all_zero(acc[i], bs).sum()) for i in range(2))


def test_degrade_fd_ring_wraps_many_tiles_per_cta(P):
    """The persistent K4 walks ~20 tiles per CTA here (24 frames x 120 block rows over 148 CTAs), so every stage of its
    shared-memory ring is reused several times with both barrier parities; moving rectangles put motion in many tiles."""
    r = rng(23)
    n, h, w = 24, 480, 640
    exact = so.cv2_dct4_matches_closed_form()
    frames = r.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    acc = np.zeros((n, h, w), np.uint8)
    for i in range(n):
        for k in range(3):
            y, x = int(r.integers(0, h - 60)), int(r.integers(0, w - 90))
            acc[i, y:y + int(r.integers(5, 60)), x:x + int(r.integers(5, 90))] = int(r.integers(1, 256))
    cnt = torch.zeros(5, dtype=torch.int64, device="cuda")
    comp, ov = P.degrade_blend(dev(frames), dev(acc), 4, 100, "fd", True, counters=cnt)
    comp, ov = host(comp), host(ov)
    for i in range(n):
        assert np.array_equal(ov[i], so.overlay_paint(frames[i], acc[i])), i
        _check_degraded(comp[i], so.degrade_fd(frames[i], acc[i], 4, 100), frames[i], acc[i], 4, 100, exact)
    c = cnt.cpu().numpy()
    assert c[2] == int((acc > 127).sum())
    nz_blocks = (acc.reshape(n, h // 4, 4, w // 4, 4) != 0).any(axis=(2, 4))
    assert c[4] == int((~nz_blocks).sum())


@pytest.mark.parametrize("q", [0.011, 0.05, 0.3, 33.3, 100.0])
def test_degrade_fd_exact_on_many_dense_blocks(P, q):
    """19 200 random blocks per level, exact equality: small q keeps every coefficient alive, which is where a one-bit
    difference in the arithmetic (e.g. a compiler-contracted multiply-add) shows up as a flipped truncation."""
    if not so.cv2_dct4_matches_closed_form():
        pytest.skip("host cv2 does not follow the recovered float32 DCT sequence; covered by tolerance tests")
    r = rng(5)
    t, h, w = 2, 240, 640
    frames = r.integers(0, 256, (t, h, w, 3), dtype=np.uint8)
    acc = np.zeros((t, h, w), np.uint8)
    comp = host(P.degrade_blend(dev(frames), dev(acc), 4, q, "fd", False)[0])
    for i in range(t):
        ref = so.degrade_fd(frames[i], acc[i], 4, q)
        bad = (comp[i] != ref).any(axis=2).reshape(h // 4, 4, w // 4, 4).any(axis=(1, 3)).sum()
        assert bad == 0, (q, i, int(bad))


def test_degrade_mco(P):
    r = rng(12)
    shape = (64, 96)
    frames = r.integers(0, 256, (2,) + shape + (3,), dtype=np.uint8)
    masks = np.zeros((2,) + shape, np.uint8)
    masks[0, 8:40, 16:50] = 255
    masks[1, 3, 90] = 3
    comp, _ = P.degrade_blend(dev(frames), dev(masks), 8, 100, "mco", False)
    comp = host(comp)
    for i in range(2):
        _check_degraded_mco(comp[i], so.degrade_mco(frames[i], masks[i]), frames[i], masks[i])


@pytest.mark.parametrize("shape,bs", [((30, 50), 4), ((480, 854), 4), ((37, 41), 4), ((6, 2), 4), ((3, 3), 4), ((90, 122), 8),
                                      ((1082, 1920), 4), ((20, 36), 8), ((35, 47), 4), ((41, 67), 8), ((43, 69), 8), ((45, 71), 8),
                                      ((46, 70), 8), ((540, 960), 8), ((7, 5), 8)])
def test_degrade_fd_clipped_edge_blocks(P, shape, bs):
    """Frame sizes that are not multiples of the block size: the reference slices the last blocks shorter
    (frame_differencing.py:117-121) and cv2.dct takes them rows-then-columns through its 1-D routine of each length
    (1..8, all restated exactly in csrc/k_dct8.cuh).  Everything is exact when cv2 follows the closed forms."""
    r = rng(33)
    h, w = shape
    exact = _exact(bs, h, w)
    n = 2
    frames = r.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    frames[1] = (frames[1] // 32) * 32
    acc = (r.random((n, h, w)) < 0.004).astype(np.uint8) * r.integers(1, 256, (n, h, w), dtype=np.uint8)
    cnt = torch.zeros(5, dtype=torch.int64, device="cuda")
    comp, ov = P.degrade_blend(dev(frames), dev(acc), bs, 100, "fd", True, counters=cnt)
    comp, ov = host(comp), host(ov)
    hf, wf = (h // bs) * bs, (w // bs) * bs
    n_static = 0
    for i in range(n):
        ref = so.degrade_fd(frames[i], acc[i], bs, 100)
        assert np.array_equal(ov[i], so.overlay_paint(frames[i], acc[i]))
        if hf and wf:
            _check_degraded(comp[i][:hf, :wf], ref[:hf, :wf], frames[i][:hf, :wf], acc[i][:hf, :wf], bs, 100, exact)
        edge = np.ones((h, w), bool)
        edge[:hf, :wf] = False
        static = so.block_all_zero(acc[i], bs)
        n_static += int(static.sum())
        st_px = np.repeat(np.repeat(static, bs, 0), bs, 1)[:h, :w]
        assert np.array_equal(comp[i][edge & ~st_px], ref[edge & ~st_px])          # colour round trip: integer, exact
        d = np.abs(comp[i].astype(int) - ref.astype(int)).max(axis=2)[edge & st_px]
        if d.size:
            if exact:
                assert d.max() == 0, (shape, i, int(d.max()), int((d > 0).sum()))
            else:
                assert np.mean(d <= 1) >= 0.9, (shape, i, float(np.mean(d <= 1)))
    c = cnt.cpu().numpy()
    assert c[2] == int((acc > 127).sum())
    assert c[3] == n * (-(-h // bs)) * (-(-w // bs)) and c[4] == n_static


def test_degrade_mco_partial_blocks_only_get_the_colour_round_trip(P):
    r = rng(34)
    h, w = 70, 100                                      # 8 full block rows + 6 rows, 12 full block columns + 4 columns
    frames = r.integers(0, 256, (2, h, w, 3), dtype=np.uint8)
    masks = np.zeros((2, h, w), np.uint8)
    masks[0, 10:30, 20:60] = 255
    comp = host(P.degrade_blend(dev(frames), dev(masks), 8, 100, "mco", False)[0])
    for i in range(2):
        ref = so.degrade_mco(frames[i], masks[i])
        assert np.array_equal(comp[i][64:, :], ref[64:, :]) and np.array_equal(comp[i][:, 96:], ref[:, 96:])
        _check_degraded_mco(comp[i][:64, :96], ref[:64, :96], frames[i][:64, :96], masks[i][:64, :96])


@pytest.mark.parametrize("mode", ["window", "fd"])
def test_loops_on_frame_sizes_not_multiple_of_block(P, mode):
    """854 x 480-like geometry (W % 4 == 2): every kernel of both loops on a size with clipped edge blocks."""
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n = 62, 110, 16
    frames = make_clip((h, w), n, seed=12).frames()
    exact = _exact(4, h, w)
    if mode == "window":
        kw = dict(window_size=5, alpha_fraction=0.2, morph_kernel=2, kernel_size=7)
        ref = loops.window_loop(list(frames), **kw)
        seed, mref = so.bgr2gray(frames[0]), np.stack(ref["mask"])
    else:
        kw = dict(min_area=50)
        ref = loops.fd_loop(list(frames), **kw)
        seed, mref = loops.first_frame_gray_fd(frames[0]), np.stack(ref["acc"])
    pipe = P.FramePipeline(w, h, mode, max_batch=8, **kw)
    pipe.begin_stream(seed)
    ov = np.empty((n - 1, h, w, 3), np.uint8); cp = np.empty_like(ov); mk = np.empty((n - 1, h, w), np.uint8)
    pipe.process_host(np.ascontiguousarray(frames[1:]), ov, cp, mk)
    c = pipe.counters()
    pipe.close()
    assert np.array_equal(mk, mref)
    assert np.array_equal(ov, np.stack(ref["overlay"]))
    rc = np.stack(ref["compressed"])
    hf, wf = (h // 4) * 4, (w // 4) * 4
    d = np.abs(cp.astype(int) - rc.astype(int))
    if exact:
        assert d.max() == 0
    else:
        assert np.mean(d[:, hf:, :] <= 1) > 0.9 and np.mean(d[:, :, wf:] <= 1) > 0.9
    assert c["blocks"] == (n - 1) * (-(-h // 4)) * (-(-w // 4))


def test_fd_loop_against_reference_fixture_with_clipped_blocks(P):
    """126 x 218 frames through the UNMODIFIED reference (tests/golden/fd_clipped_126x218.npz): masks and overlays are
    exact; so are the compressed frames, clipped 4x2 / 2x4 / 2x2 edge blocks included."""
    z, frames, kw, (h, w, n) = load_fd(FD_CLIPPED_FIXTURE)
    exact = _exact(4, h, w)
    pipe = P.FramePipeline(w, h, "fd", max_batch=8, **kw)
    pipe.begin_stream(loops.first_frame_gray_fd(frames[0]))
    ov = np.empty((n - 1, h, w, 3), np.uint8); cp = np.empty_like(ov); mk = np.empty((n - 1, h, w), np.uint8)
    pipe.process_host(np.ascontiguousarray(frames[1:]), ov, cp, mk)
    pipe.close()
    assert np.array_equal(mk, z["acc"])
    assert [sha(x) for x in ov] == list(z["overlay_sha"])
    hf, wf = (h // 4) * 4, (w // 4) * 4
    tail = z["compressed_tail"]
    d = np.abs(cp[-2:].astype(int) - tail.astype(int))
    if exact:
        assert d.max() == 0
    else:
        assert np.mean(d[:, :hf, :wf] > 1) < 1e-3
        assert np.mean(d[:, hf:, :] <= 1) > 0.9 and np.mean(d[:, :, wf:] <= 1) > 0.9
    assert (z["acc"][-1][hf:, :] == 0).any() or (z["acc"][-1][:, wf:] == 0).any()      # the fixture does have static edge pixels


def test_unsupported_is_loud(P):
    from dynamic_video_compression_surveillance_b200._lib import DvcUnsupported
    frames = torch.zeros((1, 32, 48, 3), dtype=torch.uint8, device="cuda")
    with pytest.raises(DvcUnsupported):
        P.degrade_blend(frames, torch.zeros((1, 32, 48), dtype=torch.uint8, device="cuda"), 16, 100, "fd")
    with pytest.raises(NotImplementedError):
        P.FramePipeline(64, 64, "fd", block_size=16)
    with pytest.raises(NotImplementedError):
        P.FramePipeline(64, 64, "window", window_size=200)


@pytest.mark.parametrize("bs", [1, 2, 3, 5, 6, 7])
def test_degrade_fd_other_block_sizes(P, bs):
    """The reference takes any block_size (frame_differencing.py:22,117-127); sizes 1..8 other than 4 and 8 run every block
    through the general exact path (1-D routines of k_dct8.cuh), clipped edge blocks included."""
    r = rng(40 + bs)
    h, w = 45, 70
    exact = all(so.cv2_dct_matches_closed_form(a, b) for a in {bs, h % bs or bs} for b in {bs, w % bs or bs} if (a, b) != (1, 1))
    frames = r.integers(0, 256, (2, h, w, 3), dtype=np.uint8)
    frames[1] = (frames[1] // 16) * 16
    acc = (r.random((2, h, w)) < 0.003).astype(np.uint8) * 200
    cnt = torch.zeros(5, dtype=torch.int64, device="cuda")
    comp, ov = P.degrade_blend(dev(frames), dev(acc), bs, 100, "fd", True, cnt)
    comp, ov = host(comp), host(ov)
    for i in range(2):
        assert np.array_equal(ov[i], so.overlay_paint(frames[i], acc[i]))
        ref = so.degrade_fd(frames[i], acc[i], bs, 100)
        if exact:
            assert np.array_equal(comp[i], ref), (bs, i, int((comp[i] != ref).sum()))
        else:
            assert np.mean(np.abs(comp[i].astype(int) - ref.astype(int)) <= 1) > 0.99
    c = host(cnt)
    assert c[3] == 2 * (-(-h // bs)) * (-(-w // bs)) and c[4] == sum(int(so.block_all_zero(acc[i], bs).sum()) for i in range(2))


# ---------------------------------------------------------------------------------------------------
# whole loop
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", FD_FIXTURES)
@pytest.mark.parametrize("max_batch", [4, 16])
def test_fd_loop_against_reference_fixture(P, name, max_batch):
    """The fd-exact loop against outputs of the UNMODIFIED reference (tests/golden/*.npz)."""
    z, frames, kw, (h, w, n) = load_fd(name)
    bs = kw.get("block_size", 4)
    exact = _exact(bs, h, w)
    pipe = P.FramePipeline(w, h, "fd", max_batch=max_batch, **kw)
    pipe.begin_stream(loops.first_frame_gray_fd(frames[0]))
    ov = np.empty((n - 1, h, w, 3), np.uint8)
    cp = np.empty_like(ov)
    acc = np.empty((n - 1, h, w), np.uint8)
    pipe.process_host(np.ascontiguousarray(frames[1:]), ov, cp, acc)
    assert np.array_equal(acc, z["acc"])
    assert [sha(x) for x in ov] == list(z["overlay_sha"])
    if exact:
        assert [sha(x) for x in cp] == list(z["compressed_sha"])
    assert np.array_equal(ov[-2:], z["overlay_tail"])
    for i in (-2, -1):
        _check_degraded(cp[i], z["compressed_tail"][i], frames[n + i], z["acc"][i], bs, kw.get("quantization_level", 100), exact)
    c = pipe.counters()
    assert c["frames"] == n - 1 and c["motion_pixels"] == int((z["acc"] > 127).sum())
    pipe.close()


@pytest.mark.parametrize("cfg", [dict(window_size=5, alpha_fraction=0.2, morph_kernel=2, kernel_size=7),
                                 dict(window_size=30, alpha_fraction=0.2, morph_kernel=2, kernel_size=0),
                                 dict(window_size=4, alpha_fraction=0.5, morph_kernel=3, morph_shape="rect", kernel_size=15),
                                 dict(window_size=7, alpha_fraction=0.34, morph_kernel=0, kernel_size=3)])
@pytest.mark.parametrize("noise", [False, True])
def test_window_loop_against_oracle(P, cfg, noise):
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n = 120, 176, 45
    frames = make_clip((h, w), n, seed=5, temporal_noise=noise).frames()
    thr = 6.0 if noise else 0.5
    ref = loops.window_loop(list(frames), motion_threshold=thr, **cfg)
    pipe = P.FramePipeline(w, h, "window", motion_threshold=thr, max_batch=8, **cfg)
    pipe.begin_stream(so.bgr2gray(frames[0]))
    d_frames = dev(frames[1:])
    ov = torch.empty_like(d_frames); cp = torch.empty_like(d_frames)
    mk = torch.empty(d_frames.shape[:3], dtype=torch.uint8, device="cuda")
    for i in range(0, n - 1, 8):
        pipe.process_device(d_frames[i:i + 8], ov[i:i + 8], cp[i:i + 8], mk[i:i + 8])
    torch.cuda.synchronize()
    ov, cp, mk = host(ov), host(cp), host(mk)
    exact = so.cv2_dct4_matches_closed_form()
    for t in range(n - 1):
        assert np.array_equal(mk[t], ref["mask"][t]), t
        assert np.array_equal(ov[t], ref["overlay"][t]), t
        _check_degraded(cp[t], ref["compressed"][t], frames[t + 1], ref["mask"][t], 4, 100, exact)
    pipe.close()


def test_window_front_end_gray_variants_measure_build():
    """The -DDVC_MEASURE flavour keeps three gray conversions in K1 for A/B runs (DVC_GRAY_IMPL: 0 PRMT + IMAD, 1 IDP.4A,
    2 IDP.2A = the product's): masks must not change.  Runs tools/gray_variants_check.py against libdvc_b200_measure.so
    when a tool has built it; the product library has no such switch (tests/test_abi_cpu.py)."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib = os.path.join(root, "dynamic_video_compression_surveillance_b200", "libdvc_b200_measure.so")
    if not os.path.exists(lib) or os.path.getmtime(lib) < os.path.getmtime(lib.replace("_measure.so", ".so")):
        pytest.skip("measure flavour not built or older than the product library (python -m dynamic_video_compression_surveillance_b200.build --measure)")
    for flag in ("0", "1", "2"):
        env = dict(os.environ, DVC_LIB_FLAVOUR="measure", DVC_GRAY_IMPL=flag)
        r = subprocess.run([sys.executable, os.path.join(root, "tools", "gray_variants_check.py")], capture_output=True, text=True,
                           timeout=300, cwd=root, env=env)
        assert r.returncode == 0 and "masks equal" in r.stdout, (flag, r.stdout[-500:], r.stderr[-1500:])


def test_two_stream_overlap_matches_strict_order(P):
    """dvc_set_overlap: mask kernels of batch c+1 overlap the degrade kernel of batch c (fd mode: the front kernel on a third stream,
    one more batch ahead); results must not change."""
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n = 120, 176, 70
    frames = make_clip((h, w), n, seed=9).frames()
    for mode, kw, seed in (("window", dict(window_size=5, alpha_fraction=0.2, morph_kernel=2, kernel_size=7), so.bgr2gray(frames[0])),
                           ("fd", {}, loops.first_frame_gray_fd(frames[0]))):
        res = []
        for overlap in (False, True):
            pipe = P.FramePipeline(w, h, mode, max_batch=4, **kw)
            pipe.begin_stream(seed)
            pipe.set_overlap(overlap)
            d = dev(frames[1:])
            ov = torch.empty_like(d); cp = torch.empty_like(d)
            mk = torch.empty(d.shape[:3], dtype=torch.uint8, device="cuda")
            for i in range(0, n - 1, 4):
                pipe.process_device(d[i:i + 4], ov[i:i + 4], cp[i:i + 4], mk[i:i + 4])
            pipe.flush()
            torch.cuda.synchronize()
            res.append((host(ov), host(cp), host(mk), pipe.counters()))
            pipe.close()
        for a, b in zip(res[0][:3], res[1][:3]):
            assert np.array_equal(a, b), mode
        assert res[0][3] == res[1][3]
        ref = loops.window_loop(list(frames), **kw) if mode == "window" else loops.fd_loop(list(frames))
        assert np.array_equal(res[1][2], np.stack(ref["mask" if mode == "window" else "acc"])), mode


def test_handles_on_two_devices_in_one_process(P):
    """One process driving several GPUs (the sharding module uses one process per GPU, the C ABI does not require it):
    kernel attributes and constant tables are set up per device."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n = 96, 128, 20
    frames = make_clip((h, w), n, seed=4).frames()
    kw = dict(window_size=5, alpha_fraction=0.2, morph_kernel=2, kernel_size=7)
    ref = loops.window_loop(list(frames), **kw)
    ref8 = loops.fd_loop(list(frames), block_size=8, degrade=False)
    for device in (1, 0):
        pipe = P.FramePipeline(w, h, "window", max_batch=8, device=device, **kw)
        pipe.begin_stream(so.bgr2gray(frames[0]))
        ov = np.empty((n - 1, h, w, 3), np.uint8); cp = np.empty_like(ov); mk = np.empty((n - 1, h, w), np.uint8)
        pipe.process_host(np.ascontiguousarray(frames[1:]), ov, cp, mk)
        pipe.close()
        assert np.array_equal(mk, np.stack(ref["mask"])), device
        assert np.array_equal(ov, np.stack(ref["overlay"])), device
        pipe = P.FramePipeline(w, h, "fd", max_batch=8, device=device, block_size=8)      # the 8x8 kernel's constant table
        pipe.begin_stream(loops.first_frame_gray_fd(frames[0]))
        pipe.process_host(np.ascontiguousarray(frames[1:]), ov, cp, mk)
        pipe.close()
        assert np.array_equal(mk, np.stack(ref8["acc"])), device
    torch.cuda.set_device(0)


def test_handles_driven_from_several_host_threads(P):
    """Four host threads, each with its own handle (the GUI runs the entry points from worker threads, windows.py:94-101):
    creation, one-time kernel set-up and the loops race each other; every stream must still equal the oracle."""
    import threading
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n = 64, 96, 24
    kw = dict(window_size=5, alpha_fraction=0.2, morph_kernel=2, kernel_size=7)
    clips = [make_clip((h, w), n, seed=40 + i).frames() for i in range(4)]
    refs = [loops.window_loop(list(c), **kw) if i % 2 == 0 else loops.fd_loop(list(c)) for i, c in enumerate(clips)]
    results, errors = [None] * 4, []

    def work(i):
        try:
            mode = "window" if i % 2 == 0 else "fd"
            pipe = P.FramePipeline(w, h, mode, max_batch=8, **(kw if mode == "window" else {}))
            pipe.begin_stream(so.bgr2gray(clips[i][0]) if mode == "window" else loops.first_frame_gray_fd(clips[i][0]))
            ov = np.empty((n - 1, h, w, 3), np.uint8); cp = np.empty_like(ov); mk = np.empty((n - 1, h, w), np.uint8)
            for a in range(0, n - 1, 8):
                b = min(n - 1, a + 8)
                pipe.process_host(np.ascontiguousarray(clips[i][1 + a:1 + b]), ov[a:b], cp[a:b], mk[a:b])
            pipe.close()
            results[i] = (ov, cp, mk)
        except Exception as e:          # surfaced below
            errors.append(e)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    exact = so.cv2_dct4_matches_closed_form()
    for i in range(4):
        ov, cp, mk = results[i]
        assert np.array_equal(mk, np.stack(refs[i]["mask" if i % 2 == 0 else "acc"])), i
        assert np.array_equal(ov, np.stack(refs[i]["overlay"])), i
        if exact:
            assert np.array_equal(cp, np.stack(refs[i]["compressed"])), i


def test_state_handoff_between_handles(P):
    """Frame-chunk sharding (SURVEY.md section 8e): a second handle continues a stream from a state blob."""
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n = 96, 128, 31
    frames = make_clip((h, w), n, seed=8).frames()
    for mode, kw in (("fd", {}), ("window", dict(window_size=5))):
        seed = loops.first_frame_gray_fd(frames[0]) if mode == "fd" else so.bgr2gray(frames[0])
        whole = P.FramePipeline(w, h, mode, max_batch=8, **kw)
        whole.begin_stream(seed)
        cp_ref = np.empty((n - 1, h, w, 3), np.uint8); mk_ref = np.empty((n - 1, h, w), np.uint8)
        whole.process_host(np.ascontiguousarray(frames[1:]), None, cp_ref, mk_ref)
        a = P.FramePipeline(w, h, mode, max_batch=8, **kw)
        b = P.FramePipeline(w, h, mode, max_batch=8, **kw)
        a.begin_stream(seed)
        cp = np.empty_like(cp_ref); mk = np.empty_like(mk_ref)
        cut = 13
        a.process_host(np.ascontiguousarray(frames[1:1 + cut]), None, cp[:cut], mk[:cut])
        b.set_state(a.get_state())
        b.process_host(np.ascontiguousarray(frames[1 + cut:]), None, cp[cut:], mk[cut:])
        assert np.array_equal(mk, mk_ref), mode
        assert np.array_equal(cp, cp_ref), mode
        for p in (whole, a, b):
            p.close()


def test_full_size_properties_1080p(P):
    """At BASELINE's 1080p size the oracle is too slow for every frame: check size-independent properties and
    spot-check two frames against the oracle."""
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n = 1080, 1920, 17
    frames = make_clip("1080p", n, seed=0).frames()
    cfg = dict(window_size=5, alpha_fraction=0.2, morph_kernel=2, kernel_size=7)
    pipe = P.FramePipeline(w, h, "window", max_batch=16, **cfg)
    pipe.begin_stream(so.bgr2gray(frames[0]))
    d = dev(frames[1:])
    ov = torch.empty_like(d); cp = torch.empty_like(d)
    mk = torch.empty(d.shape[:3], dtype=torch.uint8, device="cuda")
    pipe.process_device(d, ov, cp, mk)
    torch.cuda.synchronize()
    ov, cp, mk = host(ov), host(cp), host(mk)
    assert set(np.unique(mk)) <= {0, 255}
    moving = mk > 127
    # overlay is the frame except where the mask says motion, where it is pure red
    assert np.array_equal(ov[~moving], frames[1:][~moving])
    assert (ov[moving] == np.array([0, 0, 255], np.uint8)).all()
    # static blocks come out grey (B == G == R); the counters agree with the mask
    static_px = np.repeat(np.repeat(~(mk.reshape(n - 1, h // 4, 4, w // 4, 4) != 0).any(axis=(2, 4)), 4, 1), 4, 2)
    assert (cp[static_px][:, 0] == cp[static_px][:, 1]).all() and (cp[static_px][:, 1] == cp[static_px][:, 2]).all()
    c = pipe.counters()
    assert c["motion_pixels"] == int(moving.sum()) and c["static_blocks"] == int(static_px.sum()) // 16
    ref = loops.window_loop(list(frames[:8]), **cfg)
    exact = so.cv2_dct4_matches_closed_form()
    for t in (2, 6):
        assert np.array_equal(mk[t], ref["mask"][t])
        _check_degraded(cp[t], ref["compressed"][t], frames[t + 1], ref["mask"][t], 4, 100, exact)
    pipe.close()


# ---------------------------------------------------------------------------------------------------
# the other BASELINE.json configurations as parity cases
# ---------------------------------------------------------------------------------------------------
def test_config3_4k_large_morphology(P):
    """configs[2]: 4K stream, 15x15 morphology (close + open + dilate all 15x15 rect), K=5 window."""
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n = 2160, 3840, 7
    frames = make_clip("4k", n, seed=2).frames()
    cfg = dict(window_size=5, alpha_fraction=0.2, morph_kernel=15, morph_shape="rect", kernel_size=15)
    ref = loops.window_loop(list(frames), degrade=False, **cfg)
    pipe = P.FramePipeline(w, h, "window", max_batch=8, **cfg)
    pipe.begin_stream(so.bgr2gray(frames[0]))
    d = dev(frames[1:])
    ov = torch.empty_like(d); cp = torch.empty_like(d)
    mk = torch.empty(d.shape[:3], dtype=torch.uint8, device="cuda")
    pipe.process_device(d, ov, cp, mk)
    torch.cuda.synchronize()
    mk, ov, cp = host(mk), host(ov), host(cp)
    for t in range(n - 1):
        assert np.array_equal(mk[t], ref["mask"][t]), t
        assert np.array_equal(ov[t], ref["overlay"][t]), t
    exact = so.cv2_dct4_matches_closed_form()
    t = n - 2
    _check_degraded(cp[t], so.degrade_fd(frames[t + 1], ref["mask"][t], 4, 100), frames[t + 1], ref["mask"][t], 4, 100, exact)
    pipe.close()


def test_config4_concurrent_streams_are_independent(P):
    """configs[3]: many camera streams on one GPU, batches interleaved: every stream must equal its solo run."""
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n, S = 96, 160, 25, 6
    clips = [make_clip((h, w), n, seed=s).frames() for s in range(S)]
    cfg = dict(window_size=5, alpha_fraction=0.2, morph_kernel=2, kernel_size=7)
    solo = []
    for s in range(S):
        ref = loops.window_loop(list(clips[s]), **cfg)
        solo.append((np.stack(ref["mask"]), np.stack(ref["compressed"])))
    pipes = [P.FramePipeline(w, h, "window", max_batch=8, **cfg) for _ in range(S)]
    outs = []
    for s in range(S):
        pipes[s].begin_stream(so.bgr2gray(clips[s][0]))
        d = dev(clips[s][1:])
        outs.append((d, torch.empty_like(d), torch.empty(d.shape[:3], dtype=torch.uint8, device="cuda")))
    streams = [torch.cuda.Stream() for _ in range(S)]
    for i in range(0, n - 1, 8):                       # interleave the streams batch by batch
        for s in range(S):
            d, cp, mk = outs[s]
            with torch.cuda.stream(streams[s]):
                pipes[s].process_device(d[i:i + 8], None, cp[i:i + 8], mk[i:i + 8])
    torch.cuda.synchronize()
    exact = so.cv2_dct4_matches_closed_form()
    for s in range(S):
        assert np.array_equal(host(outs[s][2]), solo[s][0]), s
        if exact:
            assert np.array_equal(host(outs[s][1]), solo[s][1]), s
        pipes[s].close()


@pytest.mark.parametrize("mode", ["window", "fd"])
@pytest.mark.parametrize("shape", [(96, 128), (62, 110)])
def test_stream_group_equals_separate_pipelines(P, mode, shape):
    """dvc_config.n_streams: S camera streams advanced in lock step by shared launches (BASELINE config 4) must give, per
    stream, exactly what S separate handles give: masks, overlays, compressed frames, counters, over several batches of
    uneven length, through the device-pointer call and the host-buffer call, and across a state hand-off."""
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w = shape
    S, n = 3, 23
    kw = dict(window_size=4, alpha_fraction=0.3, morph_kernel=2, kernel_size=5) if mode == "window" else dict(min_area=40, kernel_size=5)
    clips = [make_clip((h, w), n, seed=50 + s, temporal_noise=(s == 1)).frames() for s in range(S)]
    seed_of = (lambda f: so.bgr2gray(f)) if mode == "window" else loops.first_frame_gray_fd
    solo_ov, solo_cp, solo_mk, solo_cnt = [], [], [], {}
    for s in range(S):
        pipe = P.FramePipeline(w, h, mode, max_batch=8, **kw)
        pipe.begin_stream(seed_of(clips[s][0]))
        ov = np.empty((n - 1, h, w, 3), np.uint8); cp = np.empty_like(ov); mk = np.empty((n - 1, h, w), np.uint8)
        pipe.process_host(np.ascontiguousarray(clips[s][1:]), ov, cp, mk)
        for k, v in pipe.counters().items():
            solo_cnt[k] = solo_cnt.get(k, 0) + v
        pipe.close()
        solo_ov.append(ov); solo_cp.append(cp); solo_mk.append(mk)
    solo_ov, solo_cp, solo_mk = np.stack(solo_ov), np.stack(solo_cp), np.stack(solo_mk)
    body = np.ascontiguousarray(np.stack([c[1:] for c in clips]))                 # [S, n-1, H, W, 3]
    seeds = np.stack([seed_of(c[0]) for c in clips])
    # (a) host-buffer call, whole clip
    grp = P.FramePipeline(w, h, mode, max_batch=8, n_streams=S, **kw)
    grp.begin_stream(seeds)
    ov = np.empty_like(body); cp = np.empty_like(body); mk = np.empty(body.shape[:-1], np.uint8)
    grp.process_host(body, ov, cp, mk)
    assert np.array_equal(mk, solo_mk) and np.array_equal(ov, solo_ov) and np.array_equal(cp, solo_cp)
    assert grp.counters() == solo_cnt
    # (b) device-pointer call in uneven batches, with a state hand-off to a fresh group in the middle
    grp.begin_stream(seeds)
    dbody = dev(body)
    dov = torch.empty_like(dbody); dcp = torch.empty_like(dbody); dmk = torch.empty(dbody.shape[:-1], dtype=torch.uint8, device="cuda")
    t = 0
    for T in (8, 3, 1, 8, 2):
        if t == 11:
            blob = grp.get_state()
            grp.close()
            grp = P.FramePipeline(w, h, mode, max_batch=8, n_streams=S, **kw)
            grp.set_state(blob)
        sl = slice(t, t + T)
        fin = dbody[:, sl].contiguous()
        o, c = torch.empty_like(fin), torch.empty_like(fin)
        m = torch.empty((S, T, h, w), dtype=torch.uint8, device="cuda")
        grp.process_device(fin, o, c, m)
        dov[:, sl], dcp[:, sl], dmk[:, sl] = o, c, m
        t += T
    torch.cuda.synchronize()
    grp.close()
    assert t == n - 1
    assert np.array_equal(host(dmk), solo_mk) and np.array_equal(host(dov), solo_ov) and np.array_equal(host(dcp), solo_cp)


@pytest.mark.parametrize("mode,shape,S", [("window", (96, 128), 1), ("window", (62, 110), 2), ("fd", (96, 128), 1), ("fd", (61, 83), 2)])
def test_no_writes_outside_the_output_buffers(P, mode, shape, S):
    """compute-sanitizer is closed on this pool (profiles/r2_sanitizer_unavailable.txt), so out-of-bounds global writes are hunted
    with canaries: every output of the loop is a view inside one allocation, separated by 64 KB bands of 0xA5 that must survive."""
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w = shape
    n, G = 11, 65536
    kw = dict(window_size=4, alpha_fraction=0.3, morph_kernel=2, kernel_size=7) if mode == "window" else dict(min_area=30)
    clips = [make_clip((h, w), n, seed=80 + s).frames() for s in range(S)]
    seeds = np.stack([(so.bgr2gray(c[0]) if mode == "window" else loops.first_frame_gray_fd(c[0])) for c in clips])
    body = np.ascontiguousarray(np.stack([c[1:] for c in clips]))
    T = n - 1
    fb, pb = S * T * h * w * 3, S * T * h * w
    arena = torch.full((4 * G + 2 * fb + pb,), 0xA5, dtype=torch.uint8, device="cuda")
    o_ov, o_cp, o_mk = G, 2 * G + fb, 3 * G + 2 * fb
    lead = (S,) if S > 1 else ()
    ov = arena[o_ov:o_ov + fb].view(lead + (T, h, w, 3)); cp = arena[o_cp:o_cp + fb].view(lead + (T, h, w, 3))
    mk = arena[o_mk:o_mk + pb].view(lead + (T, h, w))
    pipe = P.FramePipeline(w, h, mode, max_batch=T, n_streams=S, **kw)
    pipe.begin_stream(seeds if S > 1 else seeds[0])
    for overlap in (False, True):
        pipe.set_overlap(overlap)
        pipe.process_device(dev(body if S > 1 else body[0]), ov, cp, mk)
        pipe.flush()
        torch.cuda.synchronize()
    pipe.close()
    a = arena.cpu().numpy()
    for lo, hi in ((0, o_ov), (o_ov + fb, o_cp), (o_cp + fb, o_mk), (o_mk + pb, a.size)):
        assert (a[lo:hi] == 0xA5).all(), (mode, shape, S, lo, hi)
    assert (a[o_mk:o_mk + pb] != 0xA5).any()


def test_config5_farneback_masks_to_mco_degrade_1080p(P):
    """configs[4]: masks from the reference's Farneback + window vote + rectangles arithmetic
    (motion_compression_opt.py:72-97, on the CPU) fed to the shared degrade kernel in MCO flavour at 1080p."""
    from collections import deque
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    h, w, n = 1080, 1920, 4
    clip = make_clip("1080p", n, seed=1)
    yy, xx = np.mgrid[0:h, 0:w]
    clip.background = np.stack([(xx * 255 // w), (yy * 255 // h), ((xx + yy) * 255 // (w + h))], -1).astype(np.uint8)
    frames = clip.frames()
    prev = cv2.cvtColor(frames[0], cv2.COLOR_BGR2GRAY)
    q = deque(maxlen=30)
    kernel = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (2, 2))
    masks = []
    for f in frames[1:]:
        gray = cv2.cvtColor(f, cv2.COLOR_BGR2GRAY)
        flow = cv2.calcOpticalFlowFarneback(prev, gray, None, 0.3, 2, 9, 2, 5, 1.1, 0)
        mag, _ = cv2.cartToPolar(flow[..., 0], flow[..., 1])
        q.append((mag > 0.5).astype(np.uint8) * 255)
        sm = (np.sum(np.array(q), axis=0) >= 0.2 * len(q) * 255).astype(np.uint8) * 255
        sm = cv2.morphologyEx(cv2.morphologyEx(sm, cv2.MORPH_CLOSE, kernel), cv2.MORPH_OPEN, kernel)
        rect = np.zeros((h, w), np.uint8)
        for c in cv2.findContours(sm, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)[0]:
            x, y, ww, hh = cv2.boundingRect(c)
            cv2.rectangle(rect, (x, y), (x + ww, y + hh), 255, -1)
        masks.append(rect)
        prev = gray
    masks = np.stack(masks)
    comp, _ = P.degrade_blend(dev(frames[1:]), dev(masks), 8, 100, "mco", False)
    comp = host(comp)
    for i in (0, n - 2):
        _check_degraded_mco(comp[i], so.degrade_mco(frames[i + 1], masks[i]), frames[i + 1], masks[i])


@pytest.mark.parametrize("name", OF_FIXTURES)
def test_of_mask_chain_against_unmodified_reference_fixture(P, name):
    """k_window_vote, k_morph_chain and the rectangle kernels against masks tapped from the UNMODIFIED
    temporal_smoothing_flow (motion_compression_opt.py:83-97; Farneback stays on the CPU and is part of the fixture):
    stage by stage, and through the drop-in's chunked host helper with carried history."""
    from dynamic_video_compression_surveillance_b200 import host_loop
    m, kw, (h, w, n) = load_of(name)
    K, alpha, mk = kw["window_size"], kw["alpha_fraction"], kw["morph_kernel"]
    voted = P.temporal_ring(dev(m["raw"]), K, alpha)
    assert np.array_equal(host(voted), m["voted"])
    morphed = P.morph(P.morph(dev(m["voted"]), "close", mk, "ellipse"), "open", mk, "ellipse")
    assert np.array_equal(host(morphed), m["morphed"])
    assert np.array_equal(host(P.mask_rectangles(dev(m["morphed"]))), m["rect"])
    # the drop-in feeds chunks of raw masks with the deque's history carried on the host
    got, hist = [], []
    for c0 in range(0, n - 1, 7):
        chunk = [x for x in m["raw"][c0:c0 + 7]]
        got.append(host_loop.smooth_rect_masks_gpu(chunk, hist, K, alpha, mk))
        hist = (hist + chunk)[-(K - 1):] if K > 1 else []
    assert np.array_equal(np.concatenate(got), m["rect"])


def test_config1_480p_300_frames_against_unmodified_reference(P):
    """BASELINE configs[0]: frame_differencing.py with all defaults on the synthetic 640x480 300-frame clip.  The fixture
    holds the SHA-256 of every accumulated mask, overlay frame and compressed frame the UNMODIFIED reference produced
    (oracle/make_golden.py::make_config1, ~3 CPU minutes); the GPU loop must reproduce all 299 of each."""
    z = np.load(os.path.join(GOLDEN, "fd_config1_480x640x300.npz"))
    h, w, n, seed, noise = (int(v) for v in z["recipe"])
    from dynamic_video_compression_surveillance_b200.synth import make_clip
    frames = make_clip((h, w), n, seed=seed, temporal_noise=bool(noise)).frames()
    pipe = P.FramePipeline(w, h, "fd", max_batch=32)
    pipe.begin_stream(loops.first_frame_gray_fd(frames[0]))
    ov = np.empty((n - 1, h, w, 3), np.uint8); cp = np.empty_like(ov); acc = np.empty((n - 1, h, w), np.uint8)
    pipe.process_host(np.ascontiguousarray(frames[1:]), ov, cp, acc)
    pipe.close()
    assert [sha(x) for x in acc] == list(z["acc_sha"])
    assert [sha(x) for x in ov] == list(z["overlay_sha"])
    if _exact(4):
        assert [sha(x) for x in cp] == list(z["compressed_sha"])
    assert int((acc[-1] == 0).sum()) == int(z["static_px_last"])


def test_random_loop_configurations_against_oracle():
    """tools/loop_fuzz.py: random sizes, batch sizes and parameters of both loop flavours (window sizes 1..31, alpha 0..1,
    rect / ellipse elements, even kernel sizes, thresholds up to 200, release factors 0.05..0.9, several quantisation levels),
    state carried over several host calls; masks, overlays and compressed frames must equal the oracle loops."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "loop_fuzz.py"), "14", "11"], capture_output=True, text=True,
                       timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip().splitlines()[-1].startswith("all cases equal"), r.stdout[-3000:]
