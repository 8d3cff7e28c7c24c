"""Background hole filling without a GPU: its definition (oracle.lr_fill) on the analytic occlusion scene of the left-right
check and on the edge cases of the row and column phases, and the validation of `fill` by ops.lr_check and StereoMatcher."""
import numpy as np
import pytest
import torch

from decnet_b200 import ops
from decnet_b200.predictor import StereoMatcher
from oracle.lr_check import lr_check
from oracle.lr_fill import fill_background

F32 = np.float32


def _padded(crop, H, W, mirror=False):
    B, h, w = crop.shape
    out = np.full((B, H, W), np.nan, dtype=np.float32)
    out[:, H - h:, W - w:] = crop[:, :, ::-1] if mirror else crop
    return out


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.int32)


def _fill(rows, valid=None):
    """fill_background of one image given as rows; valid defaults to the finite entries (NaN marks a hole)."""
    d = np.asarray(rows, dtype=np.float32)[None]
    v = np.isfinite(d) if valid is None else np.asarray(valid, dtype=bool)[None]
    f, u = fill_background(np.where(v, d, F32(0)), v)
    return f[0], u[0]


def test_analytic_scene():
    """Background at d = 8, a block at d = 20 over columns [40, 60): the check rejects [0, 8) (matches left of the right
    image) and [28, 40) (background occluded by the block); both fill with the background's 8."""
    h, w = 5, 80
    dl = np.full((1, h, w), 8, dtype=np.float32)
    dl[:, :, 40:60] = 20
    dr = np.full((1, h, w), 8, dtype=np.float32)
    dr[:, :, 20:40] = 20
    f, _, valid = lr_check(_padded(dl, 27, 81), _padded(dr, 27, 81, mirror=True), h, w, 1.0)
    filled, u16 = fill_background(f, valid)
    assert filled.dtype == np.float32 and u16.dtype == np.uint16 and filled.shape == (1, h, w)
    assert (filled[:, :, 28:40] == 8).all()                               # the occluded band takes the surface behind
    assert (filled[:, :, 0:8] == 8).all()                                 # the leading band extrapolates from the right
    assert np.array_equal(_bits(filled[valid]), _bits(dl[valid]))        # measured pixels unchanged
    assert np.array_equal(filled, dl)                                     # here the truth: the scene is a step of two planes
    assert np.array_equal(u16, (filled * 256).astype(np.uint16))


def test_single_valid_columns():
    nan = np.nan
    f, _ = _fill([[4.5, nan, nan, nan]])                                  # only column 0: a trailing run
    assert (f == F32(4.5)).all()
    f, _ = _fill([[nan, nan, nan, 2.25]])                                 # only column w - 1: a leading run
    assert (f == F32(2.25)).all()
    f, _ = _fill([[nan, nan, nan], [nan, 7.0, nan], [nan, nan, nan]])     # one valid pixel in the image
    assert (f == F32(7.0)).all()
    f, _ = _fill([[3.0]])
    assert f.tolist() == [[3.0]]


def test_row_rule_takes_the_smaller_neighbour():
    nan = np.nan
    f, _ = _fill([[9.0, nan, nan, 2.0, nan, 5.0, 6.0, nan]])
    assert f[0].tolist() == [9.0, 2.0, 2.0, 2.0, 2.0, 5.0, 6.0, 6.0]
    f, _ = _fill([[1.0, nan, 4.0]])
    assert f[0].tolist() == [1.0, 1.0, 4.0]


def test_empty_rows_top_interior_bottom():
    nan = np.nan
    rows = [[nan, nan, nan, nan],                                         # top: copies the first non-empty row
            [5.0, nan, 1.0, nan],                                         # row phase: 5 1 1 1
            [nan, nan, nan, nan],                                         # interior: per column min(above, below), strict
            [nan, nan, nan, nan],
            [2.0, 8.0, nan, 0.5],                                         # row phase: 2 8 0.5 0.5
            [nan, nan, nan, nan]]                                         # bottom: copies the last non-empty row
    f, u = _fill(rows)
    assert f[1].tolist() == [5.0, 1.0, 1.0, 1.0] and f[4].tolist() == [2.0, 8.0, 0.5, 0.5]
    assert f[0].tolist() == f[1].tolist()
    assert f[2].tolist() == f[3].tolist() == [2.0, 1.0, 0.5, 0.5]
    assert f[5].tolist() == f[4].tolist()
    assert np.array_equal(u, (f * 256).astype(np.uint16))


def test_empty_image_stays_zero_beside_a_valid_one():
    d = np.zeros((2, 3, 4), dtype=np.float32)
    v = np.zeros((2, 3, 4), dtype=bool)
    d[1, 1, 2], v[1, 1, 2] = 6.5, True
    f, u = fill_background(d, v)
    assert (f[0] == 0).all() and (u[0] == 0).all() and not np.signbit(f[0]).any()
    assert (f[1] == F32(6.5)).all() and (u[1] == 6.5 * 256).all()


def test_signed_zero_ties_keep_left_and_upper_bits():
    nz, pz = F32(-0.0), F32(0.0)
    v = [[True, False, True]]
    f, _ = _fill([[pz, 0, nz]], v)
    assert _bits(f[0]).tolist() == _bits([pz, pz, nz]).tolist()            # equal values: L's bits
    f, _ = _fill([[nz, 0, pz]], v)
    assert _bits(f[0]).tolist() == _bits([nz, nz, pz]).tolist()
    f, _ = _fill([[0, nz, 0]], [[False, True, False]])                     # runs copy the bits too
    assert _bits(f[0]).tolist() == _bits([nz, nz, nz]).tolist()
    f, _ = _fill([[pz], [0], [nz]], [[True], [False], [True]])             # column phase: A's bits on a tie
    assert _bits(f[:, 0]).tolist() == _bits([pz, pz, nz]).tolist()
    f, _ = _fill([[nz], [0], [pz]], [[True], [False], [True]])
    assert _bits(f[:, 0]).tolist() == _bits([nz, nz, pz]).tolist()
    f, _ = _fill([[2.0, 0, 2.0]], v)
    assert f[0].tolist() == [2.0, 2.0, 2.0]


def test_negative_and_large_values():
    nan = np.nan
    f, u = _fill([[-3.5, nan, 1.0, nan, 300.5, nan], [nan] * 6])
    assert f[0].tolist() == [-3.5, -3.5, 1.0, 1.0, 300.5, 300.5]
    assert f[1].tolist() == f[0].tolist()
    assert u[0].tolist() == [0, 0, 256, 256, 65535, 65535]               # disp_to_u16: negatives 0, > 255.99 clamps
    f, u = _fill([[nan, 256.0, nan, -0.25]])
    assert f[0].tolist() == [256.0, 256.0, -0.25, -0.25] and u[0].tolist() == [65535, 65535, 0, 0]


def test_every_output_is_a_copy_of_a_valid_value():
    g = np.random.default_rng(3)
    d = (g.normal(30, 40, (3, 17, 23))).astype(np.float32)
    v = g.random((3, 17, 23)) < 0.2
    v[1, 3:9] = False
    v[2] = False
    f, u = fill_background(np.where(v, d, F32(0)), v)
    for b in range(2):
        assert np.isin(f[b], d[b][v[b]]).all()
    assert np.array_equal(f[v], d[v]) and (f[2] == 0).all()
    assert np.array_equal(u, np.clip(f * 256, 0, 65535).astype(np.uint16))


def _no_cuda(monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("validation touched CUDA")
    for name in ("current_stream", "synchronize", "current_device", "is_available", "Stream", "device"):
        monkeypatch.setattr(torch.cuda, name, no_cuda)


BAD = ["foreground", "Background", "", None, 1, True, ["background"], b"background"]


def _bare_matcher(lr=None, fill="none"):
    """A matcher object with only the host-side state its argument checks read (no device, no weights)."""
    m = StereoMatcher.__new__(StereoMatcher)
    m.max_disp, m.lr_check, m.fill = 216, lr, fill
    return m


@pytest.mark.parametrize("bad", BAD)
def test_bad_fill_in_constructor(bad, monkeypatch):
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError, match="fill"):
        StereoMatcher(lr_check=1.0, fill=bad)


@pytest.mark.parametrize("bad", [b for b in BAD if b is not None])
def test_bad_fill_per_call(bad, monkeypatch):
    _no_cuda(monkeypatch)
    m = _bare_matcher(1.0)
    l = r = np.zeros((5, 7, 3), dtype=np.uint8)
    with pytest.raises(ValueError, match="fill"):
        m(l, r, fill=bad)
    with pytest.raises(ValueError, match="fill"):
        m([l], [r], fill=bad)
    with pytest.raises(ValueError, match="fill"):
        m.stream([(l, r)], fill=bad)
    with pytest.raises(ValueError, match="fill"):
        ops.lr_check(torch.zeros((2, 3, 3)), 3, 3, 1.0, fill=bad)


def test_fill_needs_a_check(monkeypatch):
    _no_cuda(monkeypatch)
    l = r = np.zeros((5, 7, 3), dtype=np.uint8)
    with pytest.raises(ValueError, match="fill needs a left-right check"):
        _bare_matcher()(l, r, fill="background")
    with pytest.raises(ValueError, match="fill needs a left-right check"):
        _bare_matcher(fill="background")(l, r)
    with pytest.raises(ValueError, match="fill needs a left-right check"):
        _bare_matcher(fill="background").stream([(l, r)])
    with pytest.raises(ValueError, match="fill needs a left-right check"):
        _bare_matcher(fill="background")([l], [r], return_valid=False)


def test_fill_resolution():
    """None is the matcher's setting; an explicit value overrides it in either direction."""
    assert _bare_matcher(1.0)._lr(None, False, None) == (1.0, "none")
    assert _bare_matcher(1.0)._lr(None, True, "background") == (1.0, "background")
    assert _bare_matcher(1.0, "background")._lr(None, False, None) == (1.0, "background")
    assert _bare_matcher(1.0, "background")._lr(2.0, False, "none") == (2.0, "none")
    assert _bare_matcher(None, "background")._lr(0.5, False, None) == (0.5, "background")
    assert _bare_matcher(None, "background")._lr(None, False, "none") == (None, "none")
