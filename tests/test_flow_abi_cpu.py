"""Argument rules of the Farneback entry points.  They are checked before any CUDA call, so they hold without a GPU."""
import pytest


@pytest.fixture(scope="module")
def lib():
    from dynamic_video_compression_surveillance_b200 import build, _lib
    build.build()
    return _lib.load()


OK = dict(n=1, H=48, W=64, pyr_scale=0.3, levels=2, winsize=9, iterations=2, poly_n=5, poly_sigma=1.1, flags=0)


def _flow(lib, **kw):
    a = dict(OK, **kw)
    return lib.dvc_farneback_flow_f32(None, None, None, a["n"], a["H"], a["W"], a["pyr_scale"], a["levels"], a["winsize"],
                                      a["iterations"], a["poly_n"], a["poly_sigma"], a["flags"], None)


def _masks(lib, **kw):
    a = dict(OK, **kw)
    return lib.dvc_flow_masks_u8(None, None, a["n"], a["H"], a["W"], a["pyr_scale"], a["levels"], a["winsize"], a["iterations"],
                                 a["poly_n"], a["poly_sigma"], a["flags"], 0.5, None)


@pytest.mark.parametrize("call", [_flow, _masks])
def test_flow_argument_codes(lib, call):
    from dynamic_video_compression_surveillance_b200._lib import DVC_ERR_INVALID, DVC_ERR_UNSUPPORTED
    assert call(lib) == DVC_ERR_INVALID                                   # valid parameters, null pointers
    assert b"null pointer" in lib.dvc_last_error(None)
    assert call(lib, n=0) == 0                                            # nothing to do
    for kw in (dict(pyr_scale=0.0), dict(pyr_scale=1.0), dict(pyr_scale=-0.5), dict(pyr_scale=float("nan")), dict(levels=-1),
               dict(winsize=0), dict(iterations=0), dict(n=-1), dict(H=0), dict(W=0), dict(poly_sigma=-1.0)):
        assert call(lib, **kw) == DVC_ERR_INVALID, kw
    for kw in (dict(poly_n=3), dict(poly_n=6), dict(flags=4), dict(flags=256), dict(H=40000)):
        assert call(lib, **kw) == DVC_ERR_UNSUPPORTED, kw
    assert call(lib, flags=256) == DVC_ERR_UNSUPPORTED and b"not implemented" in lib.dvc_last_error(None)
