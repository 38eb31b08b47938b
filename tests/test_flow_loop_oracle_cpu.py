"""tests/flow_loop_ref.py::flow_loop against the masks the unmodified temporal_smoothing_flow produced (tests/golden/of_*.npz): the
rectangle mask (the mask.mp4 frame) of every frame."""
import os

import cv2
import numpy as np
import pytest

from dynamic_video_compression_surveillance_b200.synth import make_clip
from tests.flow_loop_ref import flow_loop
from tests.golden_util import GOLDEN, OF_FIXTURES, load_of


def _clip(h, w, n, seed):
    """The clip oracle/make_golden.py::make_of feeds the reference: smooth background, moving objects."""
    clip = make_clip((h, w), n, seed=seed)
    yy, xx = np.mgrid[0:h, 0:w]
    clip.background = np.stack([(xx * 255 // w), (yy * 255 // h), ((xx + yy) * 255 // (w + h))], -1).astype(np.uint8)
    return list(clip.frames())


@pytest.mark.parametrize("name", OF_FIXTURES)
def test_flow_loop_reproduces_reference_rectangles(name):
    masks, kw, (h, w, n) = load_of(name)
    seed = int(np.load(os.path.join(GOLDEN, name + ".npz"))["recipe"][3])
    out = flow_loop(_clip(h, w, n, seed), degrade=False, **kw)
    assert len(out["mask"]) == n - 1
    # The raw and voted masks differ from the fixture in a few pixels where cv2's default dispatch differs from its scalar
    # path, which flow_ops restates (DESIGN.md section 6c); the rectangles absorb them.
    for t, (a, b) in enumerate(zip(out["mask"], masks["rect"])):
        assert np.array_equal(a, b), f"{name}: rectangle mask of frame {t + 1}: {int((a != b).sum())} pixels differ"


def test_flow_loop_chunks_carry_state():
    """Chunks that hand prev_gray and the raw-mask history on give the outputs of one call, compressed frames included."""
    frames = _clip(64, 96, 12, 7)
    kw = dict(window_size=4, alpha_fraction=0.5, morph_kernel=3, morph_shape="rect", flow_threshold=0.3)
    one = flow_loop(frames, **kw)
    a = flow_loop(frames[:6], **kw)
    b = flow_loop(frames[6:], prev_gray=a["state_prev_gray"], history=a["state_history"], **kw)
    for key in ("raw", "mask", "compressed"):
        got = a[key] + b[key]
        assert len(got) == len(one[key]) == 11
        for t, (x, y) in enumerate(zip(got, one[key])):
            assert np.array_equal(x, y), f"{key} of frame {t + 1}"
    assert np.array_equal(b["state_prev_gray"], cv2.cvtColor(frames[-1], cv2.COLOR_BGR2GRAY))
