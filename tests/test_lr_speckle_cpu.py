"""Speckle filter without a GPU: its definition (oracle.lr_speckle) against OpenCV's cv2.filterSpeckles and on hand-worked
cases, its composition with both fills, and the validation of speckle_size / speckle_range by ops.lr_check and
StereoMatcher before any device work."""
import numpy as np
import pytest
import torch

from decnet_b200 import ops
from decnet_b200.predictor import StereoMatcher
from oracle.lr_fill import fill_background
from oracle.lr_guided import fill_guided
from oracle.lr_speckle import filter_speckles

F32 = np.float32


def _bits(a):
    return np.asarray(a, dtype=F32).view(np.int32)


def test_equals_cv2_filter_speckles():
    """On int16-representable maps (valid pixels nonzero multiples of 1/16, invalid ones 0) the oracle is
    cv2.filterSpeckles(16 * disp, 0, max_size, 16 * max_diff), image by image."""
    cv2 = pytest.importorskip("cv2")
    g = np.random.default_rng(0)
    for trial in range(120):
        B, h, w = int(g.integers(1, 4)), int(g.integers(1, 40)), int(g.integers(1, 40))
        q = (g.integers(1, 6, (B, h, w)) * 16 + g.integers(-3, 4, (B, h, w))).astype(np.int16)
        q[g.random((B, h, w)) < g.random() * 0.6] = 0
        max_size, qdiff = int(g.integers(0, 30)), int(g.integers(0, 40))
        disp, valid = q.astype(F32) / F32(16), q != 0
        got, keep = filter_speckles(disp, valid, max_size, qdiff / 16.0)
        for b in range(B):
            want = q[b].copy()
            cv2.filterSpeckles(want, 0, max_size, qdiff)
            assert np.array_equal((got[b] * 16).astype(np.int16), want), (trial, b)
            assert np.array_equal(keep[b], want != 0), (trial, b)


def _one(rows):
    """A [1,h,w] map from a list of rows, None marking an invalid pixel."""
    a = np.array([[np.nan if x is None else x for x in r] for r in rows], dtype=F32)[None]
    valid = ~np.isnan(a)
    return np.where(valid, a, F32(0)).astype(F32), valid


def test_region_of_max_size_goes_and_one_larger_stays():
    disp, valid = _one([[5, 5, None, 9],
                        [5, 5, None, None],
                        [None, None, None, 9]])
    out, keep = filter_speckles(disp, valid, 3, 0.0)
    assert keep[0, :2, :2].all() and (out[0, :2, :2] == 5).all()          # the 2x2 region (4 > 3) stays
    assert not keep[0, :, 3].any() and (out[0, :, 3] == 0).all()          # the single 9s go
    out, keep = filter_speckles(disp, valid, 4, 0.0)
    assert not keep.any() and (out == 0).all() and not np.signbit(out).any()


def test_difference_equal_to_the_range_connects():
    disp, valid = _one([[1.0, 1.5, 2.0, 2.75]])
    _, keep = filter_speckles(disp, valid, 3, 0.5)                        # 1 - 1.5 - 2 is one region of 3; 2.75 alone
    assert keep.tolist() == [[[False, False, False, False]]]
    _, keep = filter_speckles(disp, valid, 2, 0.5)
    assert keep.tolist() == [[[True, True, True, False]]]
    _, keep = filter_speckles(disp, valid, 2, 0.4999)
    assert not keep.any()
    _, keep = filter_speckles(disp, valid, 3, 0.75)                       # now all four join
    assert keep.all()


def test_range_zero_joins_equal_values_and_signed_zeros():
    disp, valid = _one([[0.0, -0.0, 0.0], [7.0, 7.0, 7.5]])
    out, keep = filter_speckles(disp, valid, 2, 0.0)
    assert keep[0, 0].all() and not keep[0, 1].any()
    assert np.array_equal(_bits(out[0, 0]), _bits([0.0, -0.0, 0.0]))      # kept pixels keep their bits


def test_overflow_to_inf_does_not_connect():
    big = F32(3e38)
    disp, valid = _one([[big, -big]])
    _, keep = filter_speckles(disp, valid, 1, float(np.finfo(F32).max))
    assert not keep.any()                                                  # 3e38 - (-3e38) = inf > FLT_MAX
    _, keep = filter_speckles(disp, valid, 1, 0.0)
    assert not keep.any()


def test_diagonal_pixels_do_not_connect():
    disp, valid = _one([[4, None, 4],
                        [None, 4, None],
                        [4, None, 4]])
    out, keep = filter_speckles(disp, valid, 1, 10.0)
    assert not keep.any()                                                  # five regions of one pixel each
    disp[0, 0, 1], valid[0, 0, 1] = 4, True
    _, keep = filter_speckles(disp, valid, 1, 10.0)
    assert keep[0, 0].all() and keep[0, 1, 1] and keep.sum() == 4          # the top row and the centre: one region of 4


def test_regions_never_join_across_images():
    disp = np.full((3, 2, 2), 6, dtype=F32)
    valid = np.zeros((3, 2, 2), dtype=bool)
    valid[0, 1, :] = valid[1, 0, :] = True                                 # image 0's last row touches image 1's first
    valid[2] = True
    _, keep = filter_speckles(disp, valid, 2, 1.0)
    assert not keep[0].any() and not keep[1].any() and keep[2].all()


def test_max_size_zero_is_the_identity():
    g = np.random.default_rng(1)
    disp = g.normal(30, 20, (2, 9, 13)).astype(F32)
    valid = g.random((2, 9, 13)) < 0.5
    out, keep = filter_speckles(disp, valid, 0, 0.0)
    assert np.array_equal(_bits(out), _bits(disp)) and np.array_equal(keep, valid)


def test_random_maps_properties():
    g = np.random.default_rng(2)
    for _ in range(20):
        B, h, w = 2, int(g.integers(1, 30)), int(g.integers(1, 30))
        disp = np.round(g.normal(20, 3, (B, h, w)) * 4).astype(F32) / 4
        valid = g.random((B, h, w)) < 0.7
        disp = np.where(valid, disp, F32(0)).astype(F32)
        out, keep = filter_speckles(disp, valid, int(g.integers(1, 8)), 0.5)
        assert out.dtype == np.float32 and keep.dtype == bool
        assert not (keep & ~valid).any()
        assert np.array_equal(_bits(out[keep]), _bits(disp[keep])) and (out[~keep] == 0).all()


def test_composition_with_both_fills():
    """A one-pixel island inside an occluded strip: the background fill spreads its wrong value over the strip's rows; with
    the speckle filter first, the strip takes the background's value again, and the island is no longer valid."""
    h, w = 4, 30
    disp = np.full((1, h, w), 8, dtype=F32)
    valid = np.ones((1, h, w), dtype=bool)
    valid[:, :, 10:20] = False                                             # the occluded strip
    disp[:, :, 20:] = 20                                                   # the foreground object right of it
    disp[:, 2, 14], valid[:, 2, 14] = 3, True                              # a coincidental pass, far too near
    disp = np.where(valid, disp, F32(0)).astype(F32)
    raw, _ = fill_background(disp, valid)
    assert (raw[0, 2, 10:20] == 3).all()
    d2, v2 = filter_speckles(disp, valid, 1, 1.0)
    assert not v2[0, 2, 14] and v2.sum() == valid.sum() - 1
    clean, _ = fill_background(d2, v2)
    assert (clean[0, :, 10:20] == 8).all()
    guide = np.full((1, h, w, 3), 40, dtype=np.uint8)
    guide[:, :, 20:] = 200
    g_raw, _ = fill_guided(disp, valid, guide)
    g_clean, _ = fill_guided(d2, v2, guide)
    assert (g_clean[0, :, 10:20] == 8).all() and not (g_raw[0, :, 10:20] == 8).all()


def test_oracle_argument_checks():
    d = np.zeros((1, 3, 4), dtype=F32)
    v = np.zeros((1, 3, 4), dtype=bool)
    for bad in ((-1, 1.0), (1, -0.5), (1, float("nan")), (1, float("inf")), (1, 1e39)):
        with pytest.raises(ValueError):
            filter_speckles(d, v, *bad)
    with pytest.raises(ValueError, match="must both be"):
        filter_speckles(d[0], v[0], 1, 1.0)


# ------------------------------------------------------------------------------------------------------- validation
def _no_cuda(monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("validation touched CUDA")
    for name in ("current_stream", "synchronize", "current_device", "is_available", "Stream", "device"):
        monkeypatch.setattr(torch.cuda, name, no_cuda)


def _bare_matcher(lr=None, fill="none", size=0, rng=1.0):
    """A matcher object with only the host-side state its argument checks read (no device, no weights)."""
    m = StereoMatcher.__new__(StereoMatcher)
    m.max_disp, m.lr_check, m.fill, m.speckle_size, m.speckle_range = 216, lr, fill, size, rng
    return m


BAD_SIZES = [True, False, np.bool_(True), -1, 1.5, 2.0, "10", None, [3]]
BAD_RANGES = [True, np.bool_(False), -0.5, float("nan"), float("inf"), -float("inf"), 1e39, "1", None]


def test_good_settings():
    assert ops.lr_speckle(0, 1) == (0, 1.0)
    for size, rng in ((100, 1.0), (np.int64(7), np.float32(0.5)), (2**40, 0), (1, 3.4e38)):
        got = ops.lr_speckle(size, rng)
        assert type(got[0]) is int and type(got[1]) is float and got == (int(size), float(rng))


@pytest.mark.parametrize("bad", BAD_SIZES)
def test_bad_size(bad, monkeypatch):
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError, match="speckle_size"):
        ops.lr_speckle(bad, 1.0)
    with pytest.raises(ValueError, match="speckle_size"):
        ops.lr_check(torch.zeros((2, 3, 3)), 3, 3, 1.0, speckle_size=bad)
    if bad is not None:
        with pytest.raises(ValueError, match="speckle_size"):
            StereoMatcher(lr_check=1.0, speckle_size=bad)
        m = _bare_matcher(1.0)
        l = r = np.zeros((5, 7, 3), dtype=np.uint8)
        with pytest.raises(ValueError, match="speckle_size"):
            m(l, r, speckle_size=bad)
        with pytest.raises(ValueError, match="speckle_size"):
            m([l], [r], speckle_size=bad)
        with pytest.raises(ValueError, match="speckle_size"):
            m.stream([(l, r)], speckle_size=bad)


@pytest.mark.parametrize("bad", BAD_RANGES)
def test_bad_range(bad, monkeypatch):
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError, match="speckle_range"):
        ops.lr_speckle(5, bad)
    with pytest.raises(ValueError, match="speckle_range"):
        ops.lr_check(torch.zeros((2, 3, 3)), 3, 3, 1.0, speckle_size=5, speckle_range=bad)
    with pytest.raises(ValueError, match="speckle_range"):
        ops.lr_check(torch.zeros((2, 3, 3)), 3, 3, 1.0, speckle_range=bad)             # checked even when off
    if bad is not None:
        with pytest.raises(ValueError, match="speckle_range"):
            StereoMatcher(lr_check=1.0, speckle_size=5, speckle_range=bad)
        m = _bare_matcher(1.0, size=5)
        l = r = np.zeros((5, 7, 3), dtype=np.uint8)
        with pytest.raises(ValueError, match="speckle_range"):
            m(l, r, speckle_range=bad)
        with pytest.raises(ValueError, match="speckle_range"):
            m([l], [r], speckle_range=bad)
        with pytest.raises(ValueError, match="speckle_range"):
            m.stream([(l, r)], speckle_range=bad)


def test_speckle_needs_a_check(monkeypatch):
    _no_cuda(monkeypatch)
    l = r = np.zeros((5, 7, 3), dtype=np.uint8)
    with pytest.raises(ValueError, match="speckle_size needs a left-right check"):
        _bare_matcher()(l, r, speckle_size=10)
    with pytest.raises(ValueError, match="speckle_size needs a left-right check"):
        _bare_matcher(size=10)(l, r)
    with pytest.raises(ValueError, match="speckle_size needs a left-right check"):
        _bare_matcher(size=10).stream([(l, r)])
    with pytest.raises(ValueError, match="speckle_size needs a left-right check"):
        _bare_matcher()([l], [r], speckle_size=3)


def test_resolution():
    """None is the matcher's setting; an explicit value overrides it, 0 turns the filter off."""
    assert _bare_matcher(1.0)._speckle(1.0) == (0, 1.0)
    assert _bare_matcher(1.0, size=50, rng=2.0)._speckle(1.0) == (50, 2.0)
    assert _bare_matcher(1.0, size=50, rng=2.0)._speckle(1.0, 0) == (0, 2.0)
    assert _bare_matcher(1.0, size=50, rng=2.0)._speckle(1.0, None, 0.25) == (50, 0.25)
    assert _bare_matcher(None)._speckle(3.0, 8, 1) == (8, 1.0)
    assert _bare_matcher(None, size=50)._speckle(None, 0) == (0, 1.0)        # off without a check is fine


def test_constructor_keeps_the_settings_and_validates_before_device_work(monkeypatch):
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError, match="speckle_size"):
        StereoMatcher(speckle_size=-3)
    with pytest.raises(ValueError, match="speckle_range"):
        StereoMatcher(speckle_range=float("nan"))
