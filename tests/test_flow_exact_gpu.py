"""Farneback flow on the GPU (pipeline.farneback_flow / pipeline.flow_masks) against oracle/flow_ops.py, every pixel.

The model reproduces cv2's scalar path bit for bit (tests/test_flow_oracle_cpu.py), and the kernels write every float
operation in the same order, so each case requires equal bytes over all pixels of all pairs.  A one-ulp change anywhere in
the kernels fails here; tests/test_flow_gpu.py keeps the separate, relative check against cv2's default path."""
import numpy as np
import pytest
import torch

from oracle import flow_ops as fo
from tests.test_flow_gpu import CALL_SITE, STAGES, _grays

pytestmark = pytest.mark.gpu


def _P():
    from dynamic_video_compression_surveillance_b200 import pipeline
    return pipeline


def _assert_bytes(got, want, what):
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, got.dtype, want.shape, want.dtype)
    if got.tobytes() == want.tobytes():
        return
    diff = got.view(f"u{got.itemsize}") != want.view(f"u{want.itemsize}")
    first = tuple(int(i) for i in np.argwhere(diff)[0])
    d = np.abs(got.astype(np.float64) - want.astype(np.float64))
    raise AssertionError(f"{what}: {int(diff.sum())} values differ; first (pair, y, x[, c]) {first}: gpu {got[first]!r} model "
                         f"{want[first]!r}; max |diff| {np.nanmax(d):.3g}")


def _gpu_flow(g, params):
    t = torch.from_numpy(g).cuda()
    return _P().farneback_flow(t[:-1].contiguous(), t[1:].contiguous(), *params).cpu().numpy()


def _gpu_masks(g, thr, params):
    return _P().flow_masks(torch.from_numpy(g).cuda(), thr, *params).cpu().numpy()


def _mask_of(flow, thr):
    return (fo.magnitude(flow) > np.float32(thr)).astype(np.uint8) * 255


def _check(g, params, thr=0.5, what=""):
    """Both entry points against the model: the flow of every pair, and the mask sequence."""
    want = fo.farneback(g[:-1], g[1:], *params)
    _assert_bytes(_gpu_flow(g, params), want, f"flow {what} {params}")
    _assert_bytes(_gpu_masks(g, thr, params), _mask_of(want, thr), f"masks {what} {params} thr {thr}")
    return want


# ---- parameters ---------------------------------------------------------------------------------------------------------
PARAMS = STAGES + [(0.5, lv, 10, 2, 7, 1.5, 0) for lv in (0, 1, 2, 3)] + [(0.4, 2, 9, 2, 5, 1.1, 0), (0.5, 1, 9, 2, 5, 0.0, 0)]


@pytest.mark.parametrize("params", PARAMS, ids=[",".join(map(str, p[:6])) for p in PARAMS])
def test_flow_exact_parameters(params):
    _check(np.stack(_grays(240, 352, 3, 41)), params)


# ---- borders ------------------------------------------------------------------------------------------------------------
SIDES = [1, 2, 5, 9, 10, 11]


@pytest.mark.parametrize("hw", [(s, 64) for s in SIDES] + [(64, s) for s in SIDES] + [(7, 9), (10, 10)])
def test_flow_exact_small_sides(hw):
    """Sides below 10 apply both ends of the border taper on one axis; sides 1 and 2 reflect and clamp every tap."""
    g = np.stack(_grays(hw[0], hw[1], 3, 43))
    for params in ((0.5, 0, 9, 2, 5, 1.1, 0), (0.5, 0, 5, 3, 7, 1.5, 0), CALL_SITE):
        _check(g, params, what=str(hw))


def test_flow_exact_winsize_larger_than_image_and_winsize_1():
    g = np.stack(_grays(6, 40, 3, 50))
    for params in ((0.5, 0, 15, 2, 5, 1.1, 0), (0.5, 0, 41, 2, 7, 1.5, 0), (0.5, 0, 1, 3, 5, 1.1, 0)):
        _check(g, params, what="6x40")
    _check(np.stack(_grays(48, 64, 3, 51)), (0.5, 1, 1, 2, 5, 1.1, 0), what="48x64")


# ---- pyramid boundaries -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw,params", [((120, 106), (0.3, 1, 9, 2, 5, 1.1, 0)), ((120, 107), (0.3, 2, 9, 2, 5, 1.1, 0)),
                                       ((120, 110), (0.3, 2, 9, 2, 5, 1.1, 0)),
                                       ((80, 64), (0.5, 2, 9, 2, 5, 1.1, 0)), ((80, 65), (0.5, 2, 9, 2, 5, 1.1, 0)),
                                       ((80, 66), (0.5, 2, 9, 2, 5, 1.1, 0)), ((128, 96), (0.5, 3, 9, 2, 5, 1.1, 0)),
                                       ((136, 100), (0.5, 2, 9, 2, 5, 1.1, 0)), ((63, 200), (0.5, 2, 9, 2, 5, 1.1, 0)),
                                       ((64, 200), (0.5, 2, 9, 2, 5, 1.1, 0)), ((200, 63), (0.5, 2, 9, 2, 5, 1.1, 0))])
def test_flow_exact_pyramid_boundaries(hw, params):
    """W * s around 32 (a level is gained or lost), exact 2x reductions (cv2 runs INTER_AREA there; widths 33 and 50 leave
    columns to its scalar loop), and shapes where only one axis would keep a level."""
    _check(np.stack(_grays(hw[0], hw[1], 3, 49)), params, what=str(hw))


# ---- launch groups ------------------------------------------------------------------------------------------------------
def test_flow_exact_two_groups_of_tiny_pairs():
    """4 100 pairs of 33 x 33: groups of 4 096 and 4, so the second group and the mask sequence's slot-0 carry run."""
    g = np.stack(_grays(33, 33, 4101, 52))
    _check(g, CALL_SITE, what="4100 x 33x33")


def test_flow_exact_1080p_four_pairs():
    """1080p: three pairs per group, so four pairs make a full group and a partial one."""
    _check(np.stack(_grays(1080, 1920, 5, 53)), CALL_SITE, what="1080p x 4")


def test_flow_4k_one_pair_per_group():
    """2160 x 3840: one pair per group, so the carry into slot 0 runs twice.  Against single-pair calls of the same kernels
    (each pair is then alone in its group) plus the float32 magnitude, as exact bytes."""
    g = np.stack(_grays(2160, 3840, 4, 54))
    flow = _gpu_flow(g, CALL_SITE)
    single = np.stack([_gpu_flow(g[i:i + 2], CALL_SITE)[0] for i in range(3)])
    _assert_bytes(flow, single, "4K flow, 3 pairs vs one at a time")
    _assert_bytes(_gpu_masks(g, 0.5, CALL_SITE), _mask_of(single, 0.5), "4K masks")


# ---- threshold, 1080p, placement ----------------------------------------------------------------------------------------
def test_flow_exact_threshold_tie():
    """thr equal to a float32 magnitude in the flow: the strict > leaves those pixels out."""
    g = np.stack(_grays(121, 163, 4, 55))
    want = fo.farneback(g[:-1], g[1:], *CALL_SITE)
    mag = fo.magnitude(want)
    thr = float(np.sort(mag[mag > 0].ravel())[mag[mag > 0].size // 2])
    assert np.float32(thr) == thr and (mag == np.float32(thr)).any()
    got = _gpu_masks(g, thr, CALL_SITE)
    _assert_bytes(got, _mask_of(want, thr), f"masks at tie thr {thr}")
    assert not got[mag == np.float32(thr)].any()


def test_flow_exact_1080p_call_site():
    _check(np.stack(_grays(1080, 1920, 3, 44)), CALL_SITE, what="1080p")


def test_flow_exact_unaligned_inputs():
    """Frames inside a larger uint8 buffer at byte offsets 1 and 3."""
    g = np.stack(_grays(72, 100, 4, 56))
    n = g.size
    buf = torch.zeros(2 * n + 16, dtype=torch.uint8, device="cuda")
    buf[1:1 + n] = torch.from_numpy(g.ravel()).cuda()
    buf[n + 3:2 * n + 3] = torch.from_numpy(g.ravel()).cuda()
    a = buf[1:1 + n].view(g.shape)
    b = buf[n + 3:2 * n + 3].view(g.shape)
    assert a.storage_offset() == 1 and b.storage_offset() == n + 3
    want = fo.farneback(g[:-1], g[1:], *CALL_SITE)
    f = _P().farneback_flow(a[:-1], b[1:], *CALL_SITE).cpu().numpy()
    _assert_bytes(f, want, "flow from offsets 1 and 3")
    _assert_bytes(_P().flow_masks(b, 0.5, *CALL_SITE).cpu().numpy(), _mask_of(want, 0.5), "masks from offset 3")
