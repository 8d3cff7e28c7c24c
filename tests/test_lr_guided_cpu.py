"""Guided hole filling without a GPU: its definition (oracle.lr_guided) on the analytic occlusion scene of the left-right
check, the properties the smoother's normalised interpolation must have, its line solver against a dense float64 solve,
and the validation of fill="guided" and its guide by ops.lr_check and StereoMatcher."""
import math

import numpy as np
import pytest
import torch

from decnet_b200 import ops
from decnet_b200.predictor import StereoMatcher
from oracle.lr_check import lr_check
from oracle.lr_fill import fill_background
from oracle.lr_guided import fill_guided, schedule, solve_line, weight_table

F32 = np.float32


def _padded(crop, H, W, mirror=False):
    B, h, w = crop.shape
    out = np.full((B, H, W), np.nan, dtype=np.float32)
    out[:, H - h:, W - w:] = crop[:, :, ::-1] if mirror else crop
    return out


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.int32)


def _scene():
    """test_lr_fill_cpu's scene: background at d = 8, a block at d = 20 over columns [40, 60), checked with tol 1; the guide
    is grey 60 with the block 255 brighter in every channel, so the weights across its outline are exactly 0."""
    h, w = 5, 80
    dl = np.full((1, h, w), 8, dtype=np.float32)
    dl[:, :, 40:60] = 20
    dr = np.full((1, h, w), 8, dtype=np.float32)
    dr[:, :, 20:40] = 20
    f, _, valid = lr_check(_padded(dl, 27, 81), _padded(dr, 27, 81, mirror=True), h, w, 1.0)
    guide = np.zeros((1, h, w, 3), dtype=np.uint8)
    guide[:, :, 40:60] = 255
    return dl, f, valid, guide


def test_analytic_scene():
    dl, f, valid, guide = _scene()
    assert weight_table(2.6)[765] == 0
    filled, u16 = fill_guided(f, valid, guide)
    assert filled.dtype == np.float32 and u16.dtype == np.uint16 and filled.shape == f.shape
    assert not valid[:, :, 28:40].any() and not valid[:, :, 0:8].any()
    assert (filled[:, :, 28:40] == 8).all() and (filled[:, :, 0:8] == 8).all()   # the background's value, not the block's
    assert not (filled[~valid] == 20).any()
    assert np.array_equal(_bits(filled[valid]), _bits(dl[valid]))
    assert np.array_equal(filled, dl)
    assert np.array_equal(u16, (filled * 256).astype(np.uint16))


def test_constant_power_of_two_map_fills_exactly():
    """num and den go through the same operations, and scaling by a power of two commutes with each rounding."""
    g = np.random.default_rng(1)
    h, w = 23, 37
    yy, xx = np.mgrid[0:h, 0:w]
    grey = (2 * xx + yy + g.integers(0, 4, (h, w))).astype(np.uint8)
    guide = np.stack([grey, grey // 2, 255 - grey], -1)[None]
    valid = g.random((1, h, w)) < 0.4
    valid[:, 5:15, 10:25] = False
    for value in (F32(4), F32(0.5), F32(-16)):
        disp = np.where(valid, value, F32(0)).astype(np.float32)
        filled, _ = fill_guided(disp, valid, guide)
        assert (filled == value).all()


def test_filled_values_within_the_valid_range_and_valid_bits_kept():
    g = np.random.default_rng(2)
    B, h, w = 2, 19, 41
    guide = (g.integers(0, 30, (B, h, w, 3)) + 100).astype(np.uint8)
    guide[1, :, 20:] += 100                                                # a strong vertical edge in image 1
    disp = g.uniform(-5, 90, (B, h, w)).astype(np.float32)
    valid = g.random((B, h, w)) < 0.3
    disp = np.where(valid, disp, F32(0)).astype(np.float32)
    filled, u16 = fill_guided(disp, valid, guide)
    assert np.array_equal(_bits(filled[valid]), _bits(disp[valid]))
    for b in range(B):
        lo, hi = disp[b][valid[b]].min(), disp[b][valid[b]].max()
        inv = filled[b][~valid[b]]
        assert (inv >= lo - 4 * np.spacing(abs(lo))).all() and (inv <= hi + 4 * np.spacing(abs(hi))).all()
    assert np.array_equal(u16, np.clip(filled * 256, 0, 65535).astype(np.uint16))


def test_image_without_a_valid_pixel_stays_zero():
    g = np.random.default_rng(3)
    disp = np.zeros((2, 6, 9), dtype=np.float32)
    valid = np.zeros((2, 6, 9), dtype=bool)
    disp[1, 2, 3], valid[1, 2, 3] = 6.5, True
    guide = g.integers(0, 256, (2, 6, 9, 3)).astype(np.uint8)
    filled, u16 = fill_guided(disp, valid, guide)
    assert (filled[0] == 0).all() and not np.signbit(filled[0]).any() and (u16[0] == 0).all()
    assert (filled[1] != 0).all()


def test_isolated_hole_cut_off_by_strong_edges_takes_the_background_value():
    h, w = 7, 9
    guide = np.zeros((1, h, w, 3), dtype=np.uint8)
    guide[0, 3, 4] = 255                                                   # k = 765 to every neighbour: weight exactly 0
    disp = np.full((1, h, w), 10, dtype=np.float32)
    disp[0, :, 5:] = 3
    valid = np.ones((1, h, w), dtype=bool)
    valid[0, 3, 4] = False
    disp[0, 3, 4] = 0
    filled, _ = fill_guided(disp, valid, guide)
    background, _ = fill_background(disp, valid)
    assert filled[0, 3, 4] == background[0, 3, 4] == 3                    # den is exactly 0 there
    mask = np.ones((1, h, w), dtype=bool)
    mask[0, 3, 4] = False
    assert np.array_equal(filled[mask], disp[mask])


def test_lambda_zero_is_the_background_fill():
    g = np.random.default_rng(4)
    B, h, w = 2, 11, 17
    disp = g.normal(30, 20, (B, h, w)).astype(np.float32)
    valid = g.random((B, h, w)) < 0.3
    valid[0, 4] = False
    disp = np.where(valid, disp, F32(0)).astype(np.float32)
    guide = g.integers(0, 256, (B, h, w, 3)).astype(np.uint8)
    filled, u16 = fill_guided(disp, valid, guide, lam=0.0)
    want, want_u16 = fill_background(disp, valid)
    assert np.array_equal(_bits(filled), _bits(want)) and np.array_equal(u16, want_u16)


def test_solver_agrees_with_a_dense_float64_solve():
    g = np.random.default_rng(5)
    for n in (1, 2, 3, 50, 200):
        a = (g.random(n - 1) * 100).astype(np.float32)
        a[g.random(n - 1) < 0.2] = 0
        f = g.uniform(-3, 10, n).astype(np.float32)
        A = np.diag(1 + np.r_[0, a] + np.r_[a, 0]).astype(np.float64) - np.diag(a, 1) - np.diag(a, -1)
        want = np.linalg.solve(A, f.astype(np.float64))
        (got,) = solve_line(a[None], [f[None]])
        assert got.dtype == np.float32
        np.testing.assert_allclose(got[0], want, rtol=2e-5, atol=1e-5 * np.abs(want).max())
    a = g.random((3, 4, 9)).astype(np.float32)                            # lines along the last axis of any batch shape
    rhs = [g.random((3, 4, 10)).astype(np.float32) for _ in range(2)]
    out = solve_line(a, rhs)
    for i in range(3):
        for j in range(4):
            for k in range(2):
                (one,) = solve_line(a[i, j][None], [rhs[k][i, j][None]])
                assert np.array_equal(out[k][i, j], one[0])


def test_schedule_and_weight_table():
    lam = 8000.0
    got = schedule(lam)
    assert [type(x) for x in got] == [np.float32] * 3
    assert got == [F32(lam * 1.5 * 16 / 63), F32(lam * 1.5 * 4 / 63), F32(lam * 1.5 / 63)]
    assert math.isclose(sum(float(x) for x in got), lam / 2, rel_tol=1e-6)   # 1.5 (16 + 4 + 1) / 63 = 1/2
    assert schedule(0.0) == [0, 0, 0]
    t = weight_table(2.6)
    assert t.dtype == np.float32 and t.shape == (766,) and t[0] == 1
    assert all(t[k] == F32(math.exp(-k / 2.6)) for k in range(766))
    nz = int((t > 0).sum())                                                # a subnormal tail, then underflow to 0
    assert (np.diff(t) <= 0).all() and 0 < t[nz - 1] < np.finfo(np.float32).tiny and (t[nz:] == 0).all()
    assert weight_table(1.0)[3] == F32(math.exp(-3.0))


def test_rgb_and_bgr_guides_agree():
    g = np.random.default_rng(6)
    disp = g.uniform(0, 50, (1, 9, 13)).astype(np.float32)
    valid = g.random((1, 9, 13)) < 0.3
    guide = g.integers(0, 256, (1, 9, 13, 3)).astype(np.uint8)
    a, _ = fill_guided(disp, valid, guide)
    b, _ = fill_guided(disp, valid, np.ascontiguousarray(guide[..., ::-1]))
    assert np.array_equal(_bits(a), _bits(b))


@pytest.mark.parametrize("h, w", [(1, 1), (1, 40), (40, 1)])
def test_single_row_and_column_images(h, w):
    g = np.random.default_rng(h * 100 + w)
    disp = np.full((1, h, w), 2, dtype=np.float32)
    valid = np.zeros((1, h, w), dtype=bool)
    valid.flat[::7] = True
    guide = np.full((1, h, w, 3), 50, dtype=np.uint8) + g.integers(0, 3, (1, h, w, 3)).astype(np.uint8)
    filled, u16 = fill_guided(np.where(valid, disp, F32(0)), valid, guide)
    assert filled.shape == (1, h, w) and (filled == 2).all() and (u16 == 512).all()
    (line,) = solve_line(np.zeros((1, max(h, w) - 1), np.float32), [np.arange(max(h, w), dtype=np.float32)[None]])
    assert np.array_equal(line[0], np.arange(max(h, w), dtype=np.float32))


def test_oracle_argument_shapes():
    d = np.zeros((1, 3, 4), dtype=np.float32)
    v = np.zeros((1, 3, 4), dtype=bool)
    with pytest.raises(ValueError, match="guide"):
        fill_guided(d, v, np.zeros((1, 3, 4, 3), dtype=np.float32))
    with pytest.raises(ValueError, match="guide"):
        fill_guided(d, v, np.zeros((1, 4, 3, 3), dtype=np.uint8))


# ------------------------------------------------------------------------------------------------------- validation
def _no_cuda(monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("validation touched CUDA")
    for name in ("current_stream", "synchronize", "current_device", "is_available", "Stream", "device"):
        monkeypatch.setattr(torch.cuda, name, no_cuda)


def _bare_matcher(lr=None, fill="none"):
    """A matcher object with only the host-side state its argument checks read (no device, no weights)."""
    m = StereoMatcher.__new__(StereoMatcher)
    m.max_disp, m.lr_check, m.fill = 216, lr, fill
    return m


def test_guided_is_a_fill():
    assert "guided" in ops.LR_FILLS and ops.lr_fill("guided") == "guided"


def test_ops_guide_is_required_for_guided_and_only_for_it(monkeypatch):
    _no_cuda(monkeypatch)
    pred = torch.zeros((2, 3, 3))
    guide = torch.zeros((1, 3, 3, 3), dtype=torch.uint8)
    with pytest.raises(ValueError, match="guide is required"):
        ops.lr_check(pred, 3, 3, 1.0, fill="guided")
    for fill in ("none", "background"):
        with pytest.raises(ValueError, match="guide is required"):
            ops.lr_check(pred, 3, 3, 1.0, fill=fill, guide=guide)
    with pytest.raises(ValueError, match="fill"):
        ops.lr_check(pred, 3, 3, 1.0, fill="Guided", guide=guide)


def test_guided_needs_a_check(monkeypatch):
    _no_cuda(monkeypatch)
    l = r = np.zeros((5, 7, 3), dtype=np.uint8)
    with pytest.raises(ValueError, match="fill needs a left-right check"):
        _bare_matcher()(l, r, fill="guided")
    with pytest.raises(ValueError, match="fill needs a left-right check"):
        _bare_matcher(fill="guided")(l, r)
    with pytest.raises(ValueError, match="fill needs a left-right check"):
        _bare_matcher(fill="guided").stream([(l, r)])
    with pytest.raises(ValueError, match="fill needs a left-right check"):
        _bare_matcher(fill="guided")([l], [r])


def test_guided_resolution():
    assert _bare_matcher(1.0)._lr(None, False, "guided") == (1.0, "guided")
    assert _bare_matcher(1.0, "guided")._lr(None, False, None) == (1.0, "guided")
    assert _bare_matcher(1.0, "guided")._lr(None, True, "background") == (1.0, "background")
    assert _bare_matcher(None, "guided")._lr(2.0, False, None) == (2.0, "guided")
    assert _bare_matcher(None, "guided")._lr(None, False, "none") == (None, "none")


def test_guided_in_constructor_validates_before_device_work(monkeypatch):
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError, match="fill"):
        StereoMatcher(lr_check=1.0, fill="guide")
