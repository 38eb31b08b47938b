"""oracle/flow_ops.py (the exact-order numpy model of cv2.calcOpticalFlowFarneback) against cv2 itself, without a GPU.

The model follows cv2's scalar path, so every comparison runs cv2 under setUseOptimized(False) and requires equal bytes.
(cv2's default path dispatches to SIMD code with fused multiply-adds in the blur and resize once pyramid levels are used,
and that is a different function; tests/test_flow_gpu.py bounds the GPU's distance to it.)  With these equal,
tests/test_flow_exact_gpu.py can compare the CUDA kernels with the model pixel for pixel."""
import cv2
import numpy as np
import pytest

from oracle import flow_ops as fo
from tests.test_flow_gpu import CALL_SITE, STAGES, _grays


def _scalar(fn):
    cv2.setUseOptimized(False)
    try:
        return fn()
    finally:
        cv2.setUseOptimized(True)


def _cv2_flows(grays, params):
    return _scalar(lambda: np.stack([cv2.calcOpticalFlowFarneback(a, b, None, *params) for a, b in zip(grays[:-1], grays[1:])]))


def _model_flows(grays, params):
    g = np.stack(grays)
    return fo.farneback(g[:-1], g[1:], *params)


def _assert_bytes(got, want, what):
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, got.dtype, want.shape, want.dtype)
    if got.tobytes() == want.tobytes():
        return
    diff = got.view(f"u{got.itemsize}") != want.view(f"u{want.itemsize}")
    first = tuple(int(i) for i in np.argwhere(diff)[0])
    d = np.abs(got.astype(np.float64) - want.astype(np.float64))
    raise AssertionError(f"{what}: {int(diff.sum())} values differ, first at {first}: model {got[first]!r} cv2 {want[first]!r}, "
                         f"max |diff| {np.nanmax(d):.3g}")


# ---- constants --------------------------------------------------------------------------------------------------------
def _level_sigmas():
    out = set()
    for ps in np.round(np.arange(0.1, 0.901, 0.05), 2):
        for lv in range(6):
            s = 1.0
            for _ in range(lv):
                s *= float(ps)
            sigma = (1.0 / s - 1) * 0.5
            ks = max(fo.cv_round(sigma * 5) | 1, 3)
            if ks <= 255:                       # the GPU path's limit per level
                out.add((ks, sigma))
    return sorted(out)


def test_gauss_taps_equal_cv2_for_every_pyramid_level():
    """Every (ksize <= 255, sigma) a pyramid with pyr_scale 0.1..0.9 and levels 0..5 asks for, plus the fixed sigma <= 0
    kernels."""
    cases = _level_sigmas() + [(n, 0.0) for n in (1, 3, 5, 7, 9)] + [(n, -1.0) for n in (11, 15)]
    assert len(cases) > 60
    for ks, sigma in cases:
        _assert_bytes(fo.gauss_taps(ks, sigma), cv2.getGaussianKernel(ks, sigma, cv2.CV_32F).ravel(), f"taps ks={ks} sigma={sigma}")


@pytest.mark.parametrize("n,sigma", [(5, 1.1), (7, 1.5), (5, 0.0), (7, 0.0), (5, 1.5), (7, 1.1)])
def test_gram_inverse_equals_cv2_cholesky(n, sigma):
    """FarnebackPrepareGaussian inverts the Gram matrix with DECOMP_CHOLESKY; Gauss-Jordan differs in the last bits."""
    G = np.array(fo.gram_matrix(n, sigma)[3])
    ok, ref = cv2.invert(G, flags=cv2.DECOMP_CHOLESKY)
    assert ok
    _assert_bytes(np.array(fo.cholesky_inverse(G)), ref, f"inverse Gram poly_n={n} sigma={sigma}")


# ---- level images -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw", [(240, 352), (121, 163), (80, 66), (64, 65), (37, 53), (33, 33), (5, 9), (1, 40)])
@pytest.mark.parametrize("pyr_scale", [0.3, 0.5])
def test_level_images_equal_cv2_blur_then_resize(hw, pyr_scale):
    """(80, 66) at 0.5 is an exact 2x reduction with a width of 33: cv2's INTER_AREA fast path sums its last column in
    another order."""
    H, W = hw
    rng = np.random.default_rng(H * 1000 + W)
    frame = rng.integers(0, 256, (H, W), dtype=np.uint8)
    for lv in range(4):
        s = 1.0
        for _ in range(lv):
            s *= pyr_scale
        sigma = (1.0 / s - 1) * 0.5
        ks = max(fo.cv_round(sigma * 5) | 1, 3)
        w, h = fo.cv_round(W * s), fo.cv_round(H * s)
        if w < 1 or h < 1:
            continue

        def ref():
            b = cv2.GaussianBlur(frame.astype(np.float32), (ks, ks), sigma, sigma)
            return cv2.resize(b, (w, h), interpolation=cv2.INTER_LINEAR)
        _assert_bytes(fo.level_image(frame[None], w, h, ks, sigma)[0], _scalar(ref), f"level {lv} of {hw} at {pyr_scale}")


def test_level_geometry_stops_below_32():
    assert [p[:2] for p in fo.pyramid(240, 352, 0.3, 5)] == [(352, 240), (106, 72)]                  # 240 * 0.09 < 32
    assert len(fo.pyramid(64, 65, 0.5, 3)) == 2 and fo.pyramid(64, 65, 0.5, 3)[1][:2] == (32, 32)      # 32.5 rounds to 32
    assert len(fo.pyramid(63, 200, 0.5, 3)) == 1                                                        # one side keeps a level
    assert [p[:2] for p in fo.pyramid(1080, 1920, 0.3, 2)] == [(1920, 1080), (576, 324), (173, 97)]


# ---- whole flow -------------------------------------------------------------------------------------------------------
LEVELS0 = [p for p in STAGES if p[1] == 0] + [(0.5, 0, 15, 3, 7, 1.5, 0), (0.5, 0, 10, 2, 7, 0.0, 0)]


@pytest.mark.parametrize("params", LEVELS0, ids=[",".join(map(str, p[:6])) for p in LEVELS0])
def test_flow_without_levels_equals_cv2(params):
    grays = _grays(240, 352, 3, 41)
    _assert_bytes(_model_flows(grays, params), _cv2_flows(grays, params), f"{params}")


BORDER_SHAPES = [(1, 37), (33, 1), (7, 9), (9, 64), (10, 10), (11, 64), (2, 5), (64, 2), (5, 64), (6, 40)]


@pytest.mark.parametrize("hw", BORDER_SHAPES)
def test_flow_small_sides_equal_cv2(hw):
    """Sides below 10 (both ends of the border taper on one axis), winsize above the side, winsize 1."""
    grays = _grays(hw[0], hw[1], 3, 43)
    for params in ((0.5, 0, 9, 2, 5, 1.1, 0), (0.5, 0, 15, 2, 7, 1.5, 0), (0.5, 0, 1, 2, 5, 1.1, 0), CALL_SITE):
        _assert_bytes(_model_flows(grays, params), _cv2_flows(grays, params), f"{hw} {params}")


WITH_LEVELS = [p for p in STAGES if p[1] > 0] + [(0.5, lv, 10, 2, 7, 1.5, 0) for lv in (1, 2, 3)] + [(0.4, 2, 9, 2, 5, 1.1, 0)]


@pytest.mark.parametrize("params", WITH_LEVELS, ids=[",".join(map(str, p[:6])) for p in WITH_LEVELS])
def test_flow_with_levels_equals_cv2_scalar_path(params):
    """Every stage, the pyramid included, follows the scalar path exactly, so no stage needs a bound."""
    grays = _grays(240, 352, 3, 41)
    _assert_bytes(_model_flows(grays, params), _cv2_flows(grays, params), f"{params}")


@pytest.mark.parametrize("hw,params", [((120, 106), (0.3, 2, 9, 2, 5, 1.1, 0)), ((120, 107), (0.3, 2, 9, 2, 5, 1.1, 0)),
                                       ((120, 110), (0.3, 1, 9, 2, 5, 1.1, 0)), ((80, 64), (0.5, 2, 9, 2, 5, 1.1, 0)),
                                       ((80, 65), (0.5, 2, 9, 2, 5, 1.1, 0)), ((80, 66), (0.5, 2, 9, 2, 5, 1.1, 0)),
                                       ((128, 96), (0.5, 3, 9, 2, 5, 1.1, 0)), ((63, 200), (0.5, 2, 9, 2, 5, 1.1, 0)),
                                       ((64, 200), (0.5, 2, 9, 2, 5, 1.1, 0))])
def test_flow_at_pyramid_boundaries_equals_cv2(hw, params):
    grays = _grays(hw[0], hw[1], 3, 49)
    _assert_bytes(_model_flows(grays, params), _cv2_flows(grays, params), f"{hw} {params}")


def test_flow_flat_frames_equal_cv2():
    """Flat regions and exact zeros: the sign of zero flow follows cv2 (its x * a + 0 scaling of the coarse flow)."""
    g = np.zeros((3, 80, 96), np.uint8)
    g[1, 20:40, 30:50] = 200
    g[2, 22:42, 33:53] = 200
    g[:, 60:, :] = np.arange(96, dtype=np.uint8)[None, None, :]
    for params in (CALL_SITE, (0.5, 1, 5, 3, 7, 1.5, 0)):
        _assert_bytes(_model_flows(list(g), params), _cv2_flows(list(g), params), f"flat {params}")


def test_flow_1080p_call_site_equals_cv2():
    grays = _grays(1080, 1920, 2, 44)
    _assert_bytes(_model_flows(grays, CALL_SITE), _cv2_flows(grays, CALL_SITE), "1080p")


def test_flow_masks_equal_cv2_magnitude():
    """flow_masks shares the pyramids of a sequence and thresholds cv2.cartToPolar's float32 magnitude (scalar path: the
    default one may fuse x * x + y * y)."""
    grays = _grays(121, 163, 5, 45)
    ref = _cv2_flows(grays, CALL_SITE)
    mag = _scalar(lambda: np.stack([cv2.cartToPolar(np.ascontiguousarray(f[..., 0]), np.ascontiguousarray(f[..., 1]))[0]
                                    for f in ref]))
    _assert_bytes(fo.magnitude(ref), mag, "magnitude")
    thr = float(np.sort(mag.ravel())[mag.size // 2])                # a magnitude that occurs: the strict > at equality
    want = (mag > np.float32(thr)).astype(np.uint8) * 255
    _assert_bytes(fo.flow_masks(np.stack(grays), thr, *CALL_SITE), want, "masks")
