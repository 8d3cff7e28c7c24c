"""The left-right check without a GPU: its definition (oracle.lr_check) on an analytic scene and on the edge cases of
the rounding rule, StereoMatcher's validation of `lr_check` / `return_valid`, and the graph cache key."""
import numpy as np
import pytest
import torch

from decnet_b200.predictor import StereoMatcher, cache_key
from oracle.lr_check import lr_check

NAN, INF = np.float32(np.nan), np.float32(np.inf)


def _padded(crop, H, W, mirror=False, fill=np.nan):
    """crop [B,h,w] -> [B,H,W] padded on the top / left (demo.py); mirror: the crop is stored mirrored, as the reverse run
    of a pair returns the right view's disparity."""
    B, h, w = crop.shape
    out = np.full((B, H, W), fill, dtype=np.float32)
    out[:, H - h:, W - w:] = crop[:, :, ::-1] if mirror else crop
    return out


def test_analytic_scene():
    """Background at d = 8, a block at d = 20 over columns [40, 60) of the left view, hence [20, 40) of the right one."""
    h, w = 5, 80
    dl = np.full((1, h, w), 8, dtype=np.float32)
    dl[:, :, 40:60] = 20
    dr = np.full((1, h, w), 8, dtype=np.float32)
    dr[:, :, 20:40] = 20
    for tol in (0.0, 1.0, 3.0):
        f, u16, valid = lr_check(_padded(dl, 27, 81), _padded(dr, 27, 81, mirror=True), h, w, tol)
        want = np.ones(w, dtype=bool)
        want[0:8] = False                                                  # the match falls left of the right image
        want[28:40] = False                                                # background occluded by the block
        assert valid.shape == (1, h, w) and valid.dtype == bool
        assert (valid == want).all()
        assert (f[~valid] == 0).all() and (u16[~valid] == 0).all()
        assert np.array_equal(f[valid], dl[valid])
        assert np.array_equal(u16[valid], (dl[valid] * 256).astype(np.uint16))
        assert f.dtype == np.float32 and u16.dtype == np.uint16


def _one_row(dl_row, dr_row, tol):
    dl = np.asarray(dl_row, dtype=np.float32)[None, None]
    dr = np.asarray(dr_row, dtype=np.float32)[None, None]
    return lr_check(_padded(dl, 3, dl.shape[2] + 2), _padded(dr, 3, dl.shape[2] + 2, mirror=True), 1, dl.shape[2], tol)


def test_half_pixel_ties_round_up():
    # x = 3, dl = 1.5: t + 0.5 = 2.0 exactly -> u = 2; dl = 2.5: 1.0 -> u = 1.  Only the column rounding up to matches.
    dr = [9, 9, 1.5, 9, 9, 9]
    f, _, v = _one_row([0, 0, 0, 1.5, 0, 0], dr, 0.0)
    assert v[0, 0, 3]
    f, _, v = _one_row([0, 0, 0, 2.5, 0, 0], [9, 2.5, 9, 9, 9, 9], 0.0)
    assert v[0, 0, 3] and f[0, 0, 3] == np.float32(2.5)
    f, _, v = _one_row([0, 0, 0, 2.5, 0, 0], [9, 9, 2.5, 9, 9, 9], 0.0)
    assert not v[0, 0, 3]                                                  # 1.0 -> u = 1, not 2
    # the image edges: x = 0, dl = 0.5 -> u = floor(0.0) = 0 (inside); dl = 0.5000001 -> u = -1 (outside)
    _, _, v = _one_row([0.5, 0, 0], [0.5, 0, 0], 0.0)
    assert v[0, 0, 0]
    _, _, v = _one_row([np.nextafter(np.float32(0.5), np.float32(1)), 0, 0], [0.5, 0, 0], 1.0)
    assert not v[0, 0, 0]
    # x = w - 1, dl = -0.5 -> u = w (outside); a negative dl that rounds to w - 1 is inside
    _, _, v = _one_row([0, 0, -0.5], [0, 0, -0.5], 0.0)
    assert not v[0, 0, 2]
    _, _, v = _one_row([0, 0, -0.4], [0, 0, -0.4], 0.0)
    assert v[0, 0, 2]


def test_non_finite_values():
    f, u16, v = _one_row([NAN, INF, -INF, 0, 0, 0], [0, 0, 0, 0, 0, 0], 1e30)
    assert not v[0, 0, :3].any() and (f[0, 0, :3] == 0).all() and (u16[0, 0, :3] == 0).all()
    assert v[0, 0, 3:].all()
    f, u16, v = _one_row([0, 0, 0, 0], [NAN, INF, -INF, 0], 1e30)
    assert v[0, 0].tolist() == [False, False, False, True]
    assert (f[0, 0] == 0).all() and (u16[0, 0] == 0).all()


def test_tolerance_is_inclusive():
    d = np.float32(2.0)
    for tol, ok in ((0.0, False), (0.25, True), (0.2499, False)):
        _, _, v = _one_row([0, 0, 0, d, 0], [0, d + np.float32(0.25), 0, 0, 0], tol)
        assert bool(v[0, 0, 3]) == ok, tol
    _, _, v = _one_row([0, 0, 0, d, 0], [0, d, 0, 0, 0], 0.0)
    assert v[0, 0, 3]


def test_u16_clamps_like_disp_to_u16():
    """Valid disparities above 255.99 clamp to 65535 as demo.py's format does (u = x - dl must stay inside the row)."""
    w = 400
    dl = np.zeros((1, 1, w), dtype=np.float32)
    dl[0, 0, 399] = 300.5
    dr = np.zeros((1, 1, w), dtype=np.float32)
    dr[0, 0, 99] = 300.5
    _, u16, v = lr_check(_padded(dl, 1, w), _padded(dr, 1, w, mirror=True), 1, w, 0.0)
    assert v[0, 0, 399] and u16[0, 0, 399] == 65535


def _no_cuda(monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("validation touched CUDA")
    for name in ("current_stream", "synchronize", "current_device", "is_available", "Stream", "device"):
        monkeypatch.setattr(torch.cuda, name, no_cuda)


BAD = [-1, -0.5, float("nan"), float("inf"), True, False, "1", [1.0]]


@pytest.mark.parametrize("bad", BAD)
def test_bad_tolerance_in_constructor(bad, monkeypatch):
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError, match="tolerance"):
        StereoMatcher(lr_check=bad)


def _bare_matcher(lr=None):
    """A matcher object with only the host-side state its argument checks read (no device, no weights)."""
    m = StereoMatcher.__new__(StereoMatcher)
    m.max_disp, m.lr_check = 216, lr
    return m


@pytest.mark.parametrize("bad", BAD)
def test_bad_tolerance_per_call(bad, monkeypatch):
    _no_cuda(monkeypatch)
    m = _bare_matcher()
    l = r = np.zeros((5, 7, 3), dtype=np.uint8)
    with pytest.raises(ValueError, match="tolerance"):
        m(l, r, lr_check=bad)
    with pytest.raises(ValueError, match="tolerance"):
        m.stream([(l, r)], lr_check=bad)
    with pytest.raises(ValueError, match="tolerance"):
        _bare_matcher(1.0)(l, r, lr_check=bad)


def test_return_valid_needs_a_check(monkeypatch):
    _no_cuda(monkeypatch)
    l = r = np.zeros((5, 7, 3), dtype=np.uint8)
    with pytest.raises(ValueError, match="return_valid"):
        _bare_matcher()(l, r, return_valid=True)
    with pytest.raises(ValueError, match="return_valid"):
        _bare_matcher().stream([(l, r)], return_valid=True)
    with pytest.raises(ValueError, match="return_valid"):
        _bare_matcher()([l], [r], return_valid=True)


def test_good_tolerances_are_floats():
    from decnet_b200.ops import lr_tolerance
    for good, want in ((0, 0.0), (1, 1.0), (2.5, 2.5), (np.float32(0.5), 0.5), (np.int64(3), 3.0)):
        got = lr_tolerance(good)
        assert type(got) is float and got == want


def test_cache_key_lr_flag():
    plain = cache_key(8, 540, 960, 216, "learned", "fp32")
    assert plain == (8, 540, 960, 216, "learned", "fp32")
    assert cache_key(8, 540, 960, 216, "learned", "fp32", False) == plain
    lr = cache_key(8, 540, 960, 216, "learned", "fp32", True)
    assert lr != plain and lr[:6] == plain
