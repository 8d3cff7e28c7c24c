"""GPU: background hole filling of the left-right check.  ops.lr_check(..., fill="background") against oracle.lr_check followed
by oracle.lr_fill, bit for bit, on both paths of the row kernel (rows that fit its shared-memory chunk and wider ones); and
StereoMatcher(fill=...) against its definition: the filled result is oracle.lr_fill of the same call without fill."""
import numpy as np
import pytest
import torch

from decnet_b200 import StereoMatcher, _lib, ops
from oracle.lr_check import lr_check as oracle_lr_check
from oracle.lr_fill import fill_background

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
CHUNK = 4096                                                               # columns of one chunk of lr_check_fill_rows_kernel
SUBSETS = [(f, u, v) for f in (False, True) for u in (False, True) for v in (False, True) if f or u or v]


def _images(B, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8),
            torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8))


def _maps(B, H, W, ow, seed):
    """Padded forward / reverse predictions as test_lr_check_gpu's: NaN, +-inf, negative and > 256 values, half-pixel ties,
    and a reverse map that agrees with the forward one within 0..4 px at most matched columns of the crop."""
    g = np.random.default_rng(seed)
    fwd = (g.integers(-8, 90, (B, H, W)) + g.choice([0.0, 0.5, 0.25, 0.75], (B, H, W))).astype(np.float32)
    fwd[g.random((B, H, W)) < 0.02] = 300.5
    for v in (np.nan, np.inf, -np.inf):
        fwd[g.random((B, H, W)) < 0.01] = v
    rev = g.normal(40, 30, (B, H, W)).astype(np.float32)
    x = np.arange(W, dtype=np.float32) - np.float32(W - ow)              # column within the crop
    with np.errstate(invalid="ignore"):
        u = np.floor((x - fwd) + np.float32(0.5))
        hit = np.isfinite(u) & (u >= 0) & (u < ow) & (x >= 0) & (g.random((B, H, W)) < 0.7)
    b, y, xx = np.nonzero(hit)
    off = g.choice(np.array([0, 0.5, 1, 1.5, 3, 4], dtype=np.float32), b.size)
    rev[b, y, W - 1 - u[b, y, xx].astype(np.int64)] = fwd[b, y, xx] + off
    for v in (np.nan, np.inf):
        rev[g.random((B, H, W)) < 0.01] = v
    return fwd, rev


def _holes(fwd, oh, ow, seed):
    """Rows without a valid pixel (a NaN forward row fails the check): the top, an interior pair and the bottom row of
    image 0, every row of the last image when there are three or more, and on rows wider than a chunk, valid pixels only in
    the last, only in the first, or only in a middle stretch of columns (the look-ahead and the carries across chunks)."""
    B, H, W = fwd.shape
    crop = fwd[:, H - oh:, W - ow:]
    g = np.random.default_rng(seed)
    rows = sorted({0, oh // 2, min(oh // 2 + 1, oh - 1), oh - 1}) if oh > 2 else [0]
    crop[0, rows] = np.nan
    if B >= 3:
        crop[B - 1] = np.nan
    if ow > CHUNK and oh >= 4 and B >= 2:
        crop[1, 0, :ow - 40] = np.nan
        crop[1, 1, 40:] = np.nan
        crop[1, 2, :CHUNK + 100] = np.nan
        crop[1, 2, CHUNK + 300:] = np.nan
        crop[1, 3, g.random(ow) < 0.995] = np.nan
    return fwd


def _check(fwd, rev, oh, ow, tol):
    pred = torch.from_numpy(np.concatenate([fwd, rev])).to(DEV)
    f, _, v = oracle_lr_check(fwd, rev, oh, ow, tol)
    wf, wu = fill_background(f, v)
    for fo, uo, vo in SUBSETS:
        got = list(ops.lr_check(pred, oh, ow, tol, float_out=fo, u16_out=uo, valid_out=vo, fill="background"))
        assert len(got) == fo + uo + vo
        if fo:
            t = got.pop(0)
            assert t.dtype == torch.float32 and t.shape == wf.shape
            assert np.array_equal(t.cpu().numpy().view(np.int32), wf.view(np.int32)), (fo, uo, vo)
        if uo:
            t = got.pop(0)
            assert t.dtype == torch.uint16 and np.array_equal(t.cpu().numpy(), wu), (fo, uo, vo)
        if vo:
            t = got.pop(0)
            assert t.dtype == torch.bool and np.array_equal(t.cpu().numpy(), v), (fo, uo, vo)
    return wf, v


@pytest.mark.parametrize("tol", [0.0, 3.0])
@pytest.mark.parametrize("B, H, W, oh, ow", [
    (2, 6, 1, 5, 1), (3, 9, 31, 9, 31), (2, 9, 40, 7, 32), (3, 8, 33, 6, 33),
    (3, 10, 2920, 9, 2916),                                                # Middlebury's padded width, one chunk
    (2, 5, CHUNK + 27, 4, CHUNK + 1),                                      # one column more than a chunk
    (3, 7, 3 * CHUNK + 500, 6, 3 * CHUNK + 450),                           # four chunks, runs that cross them
])
def test_lr_check_fill_equals_oracle(tol, B, H, W, oh, ow):
    seed = B * 1000 + W + oh
    fwd, rev = _maps(B, H, W, ow, seed)
    if ow == 1:                                                            # few random values match inside one column
        fwd[:, H - oh + 1::2, W - 1] = 0.25
        rev[:, H - oh + 1::2, W - 1] = 0.25
    fwd = _holes(fwd, oh, ow, seed)
    wf, v = _check(fwd, rev, oh, ow, tol)
    assert v.any() and not v.all()
    if oh > 2:
        assert not v[0, 0].any() and not v[0, -1].any()                    # empty rows filled from their neighbours
        assert v[0].any() and np.isin(wf[0, 0], wf[0][v[0]]).all()
    if B >= 3:
        assert not v[-1].any() and (wf[-1] == 0).all()                     # an image without a valid pixel stays 0


def test_single_valid_pixel_and_edge_columns():
    """Images whose only valid pixels are one pixel, column 0 only, or column w - 1 only (every other crop pixel NaN)."""
    B, H, W, oh, ow = 3, 6, 60, 5, 50
    fwd, rev = _maps(B, H, W, ow, 5)
    crop = fwd[:, H - oh:, W - ow:]
    keep = np.zeros((B, oh, ow), dtype=bool)
    keep[0, 2, 25] = True
    keep[1, :, 0] = True
    keep[2, :, ow - 1] = True
    crop[~keep] = np.nan
    crop[0, 2, 25], crop[1, :, 0], crop[2, :, ow - 1] = 3.0, -0.5, 30.0   # u = x - dl inside the row
    for b, y, x in zip(*np.nonzero(keep)):
        rev[b, H - oh + y, W - 1 - int(np.floor(x - crop[b, y, x] + np.float32(0.5)))] = crop[b, y, x]
    wf, v = _check(fwd, rev, oh, ow, 0.0)
    assert v[0].sum() == 1 and (wf[0] == 3.0).all()
    assert v[1, :, 0].all() and (wf[1] == -0.5).all() and v[2, :, ow - 1].all() and (wf[2] == 30.0).all()


def test_signed_zero_ties():
    """Equal neighbours +0.0 / -0.0: the left one's bits (row phase) and the upper one's (column phase)."""
    B, H, W, oh, ow = 1, 3, 3, 3, 3
    fwd = np.full((B, H, W), np.nan, dtype=np.float32)
    fwd[0, 0, 0], fwd[0, 0, 2] = 0.0, -0.0
    fwd[0, 2, 0], fwd[0, 2, 2] = -0.0, 0.0
    rev = np.zeros((B, H, W), dtype=np.float32)
    wf, v = _check(fwd, rev, oh, ow, 0.0)
    assert v[0, 0].tolist() == [True, False, True] and not v[0, 1].any()
    assert np.signbit(wf[0]).tolist() == [[False, False, True], [False, False, True], [True, True, False]]


def test_fill_none_is_the_plain_check():
    B, H, W, oh, ow = 2, 27, 81, 20, 70
    fwd, rev = _maps(B, H, W, ow, 9)
    pred = torch.from_numpy(np.concatenate([fwd, rev])).to(DEV)
    for fo, uo, vo in SUBSETS:
        a = ops.lr_check(pred, oh, ow, 1.0, float_out=fo, u16_out=uo, valid_out=vo, fill="none")
        b = ops.lr_check(pred, oh, ow, 1.0, float_out=fo, u16_out=uo, valid_out=vo)
        assert len(a) == len(b) and all(torch.equal(x, y) for x, y in zip(a, b))
    f = torch.empty((B, oh, ow), device=DEV)
    ops._call("decnet_lr_check", pred, pred.data_ptr(), B, H, W, oh, ow, 1.0, f.data_ptr(), None, None)
    assert torch.equal(ops.lr_check(pred, oh, ow, 1.0, fill="none")[0], f)


def test_fill_entry_arguments():
    pred = torch.zeros((2, 27, 27), device=DEV)
    f = torch.empty((1, 27, 27), device=DEV)
    flags = torch.empty((1, 27), dtype=torch.uint8, device=DEV)
    with pytest.raises(_lib.DecnetError, match="float rows or row flags"):
        ops._call("decnet_lr_check_fill", pred, pred.data_ptr(), 1, 27, 27, 27, 27, 1.0, None, None, None, flags.data_ptr())
    with pytest.raises(_lib.DecnetError, match="float rows or row flags"):
        ops._call("decnet_lr_check_fill", pred, pred.data_ptr(), 1, 27, 27, 27, 27, 1.0, f.data_ptr(), None, None, None)
    with pytest.raises(_lib.DecnetError, match="crop"):
        ops._call("decnet_lr_check_fill", pred, pred.data_ptr(), 1, 27, 27, 28, 27, 1.0, f.data_ptr(), None, None,
                  flags.data_ptr())
    with pytest.raises(_lib.DecnetError, match="tolerance"):
        ops._call("decnet_lr_check_fill", pred, pred.data_ptr(), 1, 27, 27, 27, 27, -1.0, f.data_ptr(), None, None,
                  flags.data_ptr())
    with pytest.raises(ValueError, match="fill"):
        ops.lr_check(pred, 27, 27, 1.0, fill="nearest")


_MATCHERS = {}


def _matcher(masks="learned", skip=4, lr=1.0, fill="none"):
    key = (masks, skip, lr, fill)
    if key not in _MATCHERS:
        _MATCHERS[key] = StereoMatcher(masks=masks, skip_stage_id=skip, lr_check=lr, fill=fill)
    return _MATCHERS[key]


@pytest.mark.parametrize("masks", ["learned", "image"])
@pytest.mark.parametrize("skip", [4, 3])
def test_matcher_equals_definition(masks, skip):
    m = _matcher(masks, skip)
    B, h, w = 2, 130, 260
    l, r = _images(B, h, w, 11)
    disp, valid = m(l, r, return_valid=True)
    filled, fvalid = m(l, r, return_valid=True, fill="background")
    wf, wu = fill_background(disp.cpu().numpy(), valid.cpu().numpy())
    assert torch.equal(fvalid, valid) and not bool(valid.all())
    assert np.array_equal(filled.cpu().numpy().view(np.int32), wf.view(np.int32))
    assert np.array_equal(m(l, r, output="u16", fill="background").cpu().numpy(), wu)
    assert torch.equal(m(l, r, fill="none"), disp)                         # an explicit "none" is today's result
    dense = _matcher(masks, skip, fill="background")
    assert torch.equal(dense(l, r), filled) and torch.equal(dense(l, r, fill="none"), disp)


def test_fill_and_tolerance_changes_do_not_recapture():
    m = StereoMatcher(lr_check=0.5)
    l, r = _images(1, 60, 90, 3)
    d0, v0 = m(l, r, return_valid=True)
    assert m.captures == 1
    f0 = m(l, r, fill="background")
    f1, v1 = m(l, r, lr_check=3.0, fill="background", return_valid=True)
    assert torch.equal(m(l, r, fill="none"), d0)
    assert m.captures == 1 and list(m._graphs) == [(1, 60, 90, 216, "learned", "fp32", "lr")]
    assert torch.equal(f0[v0], d0[v0]) and torch.equal(f1[v1], m(l, r, lr_check=3.0)[v1])
    assert m.captures == 1


def test_host_kinds_and_stream():
    m = _matcher(fill="background")
    l, r = _images(2, 60, 90, 7)
    want_d, want_v = m(l, r, return_valid=True)
    assert not bool(want_v.all()) and torch.equal(want_d, m(l, r, fill="background"))
    d, v = m(l.cpu().numpy(), r.cpu().numpy(), return_valid=True)
    assert isinstance(d, np.ndarray) and d.dtype == np.float32 and v.dtype == np.bool_
    assert np.array_equal(d, want_d.cpu().numpy()) and np.array_equal(v, want_v.cpu().numpy())
    d, v = m(l[0].cpu(), r[0].cpu(), output="u16", return_valid=True)
    assert not d.is_cuda and d.dtype == torch.uint16 and d.shape == (60, 90) and torch.equal(v, want_v[0].cpu())
    listed = m([l[0].cpu().numpy(), l[1].cpu().numpy()], [r[0].cpu().numpy(), r[1].cpu().numpy()], return_valid=True)
    for i, (ld, lv) in enumerate(listed):
        assert np.array_equal(ld, want_d[i].cpu().numpy()) and np.array_equal(lv, want_v[i].cpu().numpy())
    sizes = [(60, 90), (60, 90), (54, 81), (60, 90)]
    items = [tuple(t.cpu().numpy() for t in _images(2, hh, ww, 30 + i)) for i, (hh, ww) in enumerate(sizes)]
    want = [m(a, b, output="u16", return_valid=True) for a, b in items]
    got = list(m.stream(items, output="u16", return_valid=True))
    assert len(got) == len(want)
    for (gd, gv), (wd, wv) in zip(got, want):
        assert isinstance(gd, np.ndarray) and np.array_equal(gd, wd) and np.array_equal(gv, wv)
    cpu_items = [tuple(torch.from_numpy(t) for t in it) for it in items]
    for a, (x, y) in zip(m.stream(cpu_items, lr_check=2.0), cpu_items):
        assert not a.is_cuda and torch.equal(a, m(x, y, lr_check=2.0))
    cuda_items = [tuple(t.to(DEV) for t in it) for it in cpu_items]
    plain = _matcher()
    for a, (x, y) in zip(plain.stream(cuda_items, fill="background"), cuda_items):
        assert a.is_cuda and torch.equal(a, plain(x, y, fill="background")) and torch.equal(a, m(x, y))


def test_filled_call_runs_only_our_kernels_after_the_replay():
    m = _matcher(fill="background")
    l, r = _images(1, 60, 90, 8)
    m(l, r)
    (st,) = m._graphs[(1, 60, 90, 216, "learned", "fp32", "lr")]
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof, torch.no_grad():
        m(l, r, output="u16")                                              # graph replay + check and fill
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert any("lr_check_fill_rows_kernel" in n for n in names)
    assert any("lr_fill_empty_rows_kernel" in n for n in names)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof, torch.no_grad():
        m._result(st, 60, 90, "u16", 1.0, True, "background")             # what runs between the replay and the result
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any("lr_check_fill_rows_kernel" in n for n in kernels)
    bad = [n for n in kernels if "at::native" in n]
    assert not bad, bad
