"""Search range [min_disp, max_disp) without a GPU: oracle.disp_range's shift on hand-worked cases, the range arithmetic
of StereoMatcher against it, the graph cache key, and the validation of min_disp / max_disp before any device work."""
import numpy as np
import pytest
import torch

from decnet_b200.predictor import StereoMatcher, cache_key, disparity_range, round_max_disp
from oracle import disp_range as odr
from oracle.disp_range import shift_cols_u8


def _ramp(*shape):
    return (np.arange(int(np.prod(shape))) % 251 + 1).astype(np.uint8).reshape(shape)


# ------------------------------------------------------------------------------------------------------------- shift
def test_shift_zero_is_the_identity():
    img = _ramp(4, 5, 3)
    assert np.array_equal(shift_cols_u8(img, 0), img)


def test_shift_by_one_both_ways():
    img = _ramp(2, 4, 3)
    right = shift_cols_u8(img, 1)                                          # out[:, x] = img[:, x - 1]
    assert np.array_equal(right[:, 0], np.zeros((2, 3), np.uint8))
    assert np.array_equal(right[:, 1:], img[:, :3])
    left = shift_cols_u8(img, -1)                                          # out[:, x] = img[:, x + 1]
    assert np.array_equal(left[:, :3], img[:, 1:])
    assert np.array_equal(left[:, 3], np.zeros((2, 3), np.uint8))


def test_hand_worked_row():
    img = np.array([[[10, 11, 12], [20, 21, 22], [30, 31, 32]]], dtype=np.uint8)          # one row, w = 3
    assert shift_cols_u8(img, 2).tolist() == [[[0, 0, 0], [0, 0, 0], [10, 11, 12]]]
    assert shift_cols_u8(img, -2).tolist() == [[[30, 31, 32], [0, 0, 0], [0, 0, 0]]]


@pytest.mark.parametrize("k", [5, 6, 100, 2**24, -5, -6, -100, -2**24])
def test_shift_by_the_width_or_more_is_black(k):
    img = _ramp(3, 5, 3)
    out = shift_cols_u8(img, k)
    assert out.shape == img.shape and out.dtype == np.uint8 and not out.any()


def test_batched_equals_per_image():
    imgs = _ramp(3, 4, 7, 3)
    for k in (-8, -3, 0, 2, 6, 7):
        out = shift_cols_u8(imgs, k)
        assert out.shape == imgs.shape
        for b in range(3):
            assert np.array_equal(out[b], shift_cols_u8(imgs[b], k))


def test_shift_rejects_non_images():
    with pytest.raises(ValueError):
        shift_cols_u8(np.zeros((4, 5, 3), np.float32), 1)
    with pytest.raises(ValueError):
        shift_cols_u8(np.zeros((4, 5), np.uint8), 1)


# ------------------------------------------------------------------------------------------------------------- range
def test_zero_start_reproduces_round_max_disp():
    for end in (1, 26, 27, 28, 100, 192, 216, 768, 783, 2**24):
        assert disparity_range(0, end) == (0, round_max_disp(end)) == odr.disparity_range(0, end)


def test_ranges_against_the_oracle():
    g = np.random.default_rng(3)
    cases = [(243, 768), (27, 243), (-40, 50), (-300, -1), (-2**24, 2**24), (2**24 - 1, 2**24), (-5, -4)]
    cases += [tuple(sorted(int(v) for v in g.integers(-2000, 2000, 2))) for _ in range(200)]
    for lo, hi in cases:
        if hi == lo:
            continue
        got = disparity_range(lo, hi)
        assert got == odr.disparity_range(lo, hi)
        assert type(got[0]) is int and type(got[1]) is int
        assert got[0] == lo and got[1] % 27 == 0 and hi - lo <= got[1] < hi - lo + 27
    assert disparity_range(243, 768) == (243, 540)
    assert disparity_range(np.int64(-40), np.int32(50)) == (-40, 108)


BAD_RANGES = [(0, 0), (5, 5), (10, 3), (-1, -1), (0, -27), (True, 100), (0, True), (False, 27), (np.bool_(True), 50),
              (0.0, 100), (0, 100.0), (1.5, 100), ("0", 100), (0, "100"), (None, 100), (0, None),
              (-2**24 - 1, 0), (0, 2**24 + 1), (2**30, 2**31)]


@pytest.mark.parametrize("lo, hi", BAD_RANGES)
def test_bad_ranges(lo, hi):
    with pytest.raises(ValueError):
        disparity_range(lo, hi)
    with pytest.raises(ValueError):
        odr.disparity_range(lo, hi)


# ------------------------------------------------------------------------------------------------------------- cache key
def test_cache_key():
    plain = cache_key(8, 540, 960, 216, "learned", "fp32")
    assert cache_key(8, 540, 960, 216, "learned", "fp32", False, 0) == plain == (8, 540, 960, 216, "learned", "fp32")
    assert cache_key(8, 540, 960, 216, "learned", "fp32", True, 0) == plain + ("lr",)
    shifted = [cache_key(8, 540, 960, 216, "learned", "fp32", lr, k) for lr in (False, True) for k in (27, -27, 1, 243)]
    others = [cache_key(B, h, w, D, masks, prec, lr) for B in (4, 8) for h in (540, 541) for w in (960, 961)
              for D in (216, 243) for masks in ("learned", "image") for prec in ("fp32", "tf32") for lr in (False, True)]
    assert len(set(shifted)) == len(shifted)
    assert not set(shifted) & set(others)
    for key in shifted:
        assert key[:6] == plain
        lr = key[-1] == "lr"
        assert len(key) == 7 + lr                                           # one element for the shift, "lr" stays last
    assert cache_key(8, 540, 960, 216, "learned", "fp32", True, 27)[-1] == "lr"
    assert cache_key(8, 540, 960, 216, "learned", "fp32", False, 27)[-1] != "lr"


# ------------------------------------------------------------------------------------------------------------- validation
def _no_cuda(monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("validation touched CUDA")
    for name in ("current_stream", "synchronize", "current_device", "is_available", "Stream", "device"):
        monkeypatch.setattr(torch.cuda, name, no_cuda)


def _bare_matcher(min_disp=0, max_disp=216):
    """A matcher object with only the host-side state its argument checks read (no device, no weights)."""
    m = StereoMatcher.__new__(StereoMatcher)
    m.min_disp, m.max_disp, m.lr_check, m.fill, m.speckle_size, m.speckle_range = min_disp, max_disp, None, "none", 0, 1.0
    return m


def test_resolution():
    """None is the matcher's end; a call that gives one end takes the other from the matcher."""
    assert _bare_matcher()._range() == (0, 216)
    assert _bare_matcher(27, 243)._range() == (27, 216)
    assert _bare_matcher(27, 243)._range(0) == (0, 243)
    assert _bare_matcher(27, 243)._range(None, 100) == (27, 81)
    assert _bare_matcher(27, 243)._range(-40, 68) == (-40, 108)
    assert _bare_matcher(0, 108)._range(None, 192) == (0, 216)


@pytest.mark.parametrize("lo, hi", BAD_RANGES)
def test_bad_ranges_raise_before_device_work(lo, hi, monkeypatch):
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError):
        StereoMatcher(min_disp=lo, max_disp=hi)
    if lo is None or hi is None:                                           # a call's None is the matcher's end
        return
    m = _bare_matcher()
    l = r = np.zeros((5, 7, 3), dtype=np.uint8)
    with pytest.raises(ValueError):
        m(l, r, min_disp=lo, max_disp=hi)
    with pytest.raises(ValueError):
        m([l], [r], min_disp=lo, max_disp=hi)
    with pytest.raises(ValueError):
        m.stream([(l, r)], min_disp=lo, max_disp=hi)                       # at the call, not at the first item


def test_one_end_against_the_matchers_other_end(monkeypatch):
    _no_cuda(monkeypatch)
    l = r = np.zeros((5, 7, 3), dtype=np.uint8)
    m = _bare_matcher(27, 243)
    for kw in ({"min_disp": 243}, {"min_disp": 300}, {"max_disp": 27}, {"max_disp": 0}, {"min_disp": True},
               {"max_disp": 2**24 + 1}):
        with pytest.raises(ValueError, match="disp"):
            m(l, r, **kw)
        with pytest.raises(ValueError, match="disp"):
            m.stream(iter([(l, r)]), **kw)
    with pytest.raises(ValueError, match="larger than min_disp"):
        StereoMatcher(min_disp=216)                                       # the default max_disp is 192


def test_constructor_settings(monkeypatch):
    """What the constructor stores, read from a matcher whose construction stops at the device (no CUDA here)."""
    import decnet_b200.predictor as P
    seen = {}

    class Stop(Exception):
        pass

    def fake_model(**kw):
        seen.update(kw)
        raise Stop

    monkeypatch.setattr(P, "DecompMatching", fake_model)
    for lo, hi, want_max, want_width in ((0, 100, 108, 108), (0, 192, 216, 216), (243, 768, 783, 540), (-40, 50, 68, 108),
                                         (27, 243, 243, 216)):
        m = StereoMatcher.__new__(StereoMatcher)
        with pytest.raises(Stop):
            m.__init__(min_disp=lo, max_disp=hi)
        assert (m.min_disp, m.max_disp, seen["max_disp"]) == (lo, want_max, want_width)
