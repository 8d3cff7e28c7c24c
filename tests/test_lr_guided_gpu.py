"""GPU: guided hole filling of the left-right check.  ops.lr_check(..., fill="guided") against oracle.lr_check followed by
oracle.lr_guided.fill_guided, bit for bit, on rows and columns shorter and longer than the kernels' tiles; the weight table
entry by entry; the C entry's argument rules; and StereoMatcher(fill="guided") against its definition: the filled result
is fill_guided of the same call's (disparity, valid), guided by the call's own left images."""
import numpy as np
import pytest
import torch

from decnet_b200 import StereoMatcher, _lib, ops
from oracle.lr_check import lr_check as oracle_lr_check
from oracle.lr_guided import fill_guided, weight_table

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
TILE = 32                                                                  # columns of one tile of guided_rows_kernel
SUBSETS = [(f, u, v) for f in (False, True) for u in (False, True) for v in (False, True) if f or u or v]


def _images(B, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8),
            torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8))


def _maps(B, H, W, ow, seed):
    """Padded forward / reverse predictions as test_lr_fill_gpu's: NaN, +-inf, negative and > 256 values, half-pixel ties,
    and a reverse map that agrees with the forward one within 0..4 px at most matched columns of the crop."""
    g = np.random.default_rng(seed)
    fwd = (g.integers(-8, 90, (B, H, W)) + g.choice([0.0, 0.5, 0.25, 0.75], (B, H, W))).astype(np.float32)
    fwd[g.random((B, H, W)) < 0.02] = 300.5
    for v in (np.nan, np.inf, -np.inf):
        fwd[g.random((B, H, W)) < 0.01] = v
    rev = g.normal(40, 30, (B, H, W)).astype(np.float32)
    x = np.arange(W, dtype=np.float32) - np.float32(W - ow)
    with np.errstate(invalid="ignore"):
        u = np.floor((x - fwd) + np.float32(0.5))
        hit = np.isfinite(u) & (u >= 0) & (u < ow) & (x >= 0) & (g.random((B, H, W)) < 0.7)
    b, y, xx = np.nonzero(hit)
    off = g.choice(np.array([0, 0.5, 1, 1.5, 3, 4], dtype=np.float32), b.size)
    rev[b, y, W - 1 - u[b, y, xx].astype(np.int64)] = fwd[b, y, xx] + off
    for v in (np.nan, np.inf):
        rev[g.random((B, H, W)) < 0.01] = v
    return fwd, rev


def _guide(B, h, w, kind, seed):
    """"random": uniform noise (strong edges everywhere: den often 0 or subnormal, so the background fallback runs);
    "pieces": piecewise-constant blocks of a few colours with strong edges between them and mild noise inside."""
    g = np.random.default_rng(seed)
    if kind == "random":
        return g.integers(0, 256, (B, h, w, 3)).astype(np.uint8)
    cells = g.integers(0, 256, (B, h // 7 + 1, w // 11 + 1, 3))
    out = cells[:, np.arange(h) // 7][:, :, np.arange(w) // 11] + g.integers(0, 3, (B, h, w, 3))
    return np.clip(out, 0, 255).astype(np.uint8)


def _guided(pred, guide, oh, ow, tol, lam=ops.GUIDED_LAMBDA, sigma=ops.GUIDED_SIGMA):
    """The C entry with explicit lambda and sigma -> (float, uint16, valid) tensors."""
    B = pred.shape[0] // 2
    f = torch.empty((B, oh, ow), device=DEV)
    u = torch.empty((B, oh, ow), dtype=torch.uint16, device=DEV)
    v = torch.empty((B, oh, ow), dtype=torch.bool, device=DEV)
    flags = torch.empty((B, oh), dtype=torch.uint8, device=DEV)
    scratch = torch.empty(int(_lib.lib().decnet_lr_guided_fill_scratch_floats(B, oh, ow)), device=DEV)
    ops._call("decnet_lr_check_guided_fill", pred, pred.data_ptr(), guide.data_ptr(), B, *pred.shape[1:], oh, ow, tol, lam,
              sigma, f.data_ptr(), u.data_ptr(), v.data_ptr(), flags.data_ptr(), scratch.data_ptr())
    return f, u, v


def _check(fwd, rev, guide, oh, ow, tol):
    pred = torch.from_numpy(np.concatenate([fwd, rev])).to(DEV)
    g = torch.from_numpy(guide).to(DEV)
    f, _, v = oracle_lr_check(fwd, rev, oh, ow, tol)
    wf, wu = fill_guided(f, v, guide)
    for fo, uo, vo in SUBSETS:
        got = list(ops.lr_check(pred, oh, ow, tol, float_out=fo, u16_out=uo, valid_out=vo, fill="guided", guide=g))
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


@pytest.mark.parametrize("kind", ["random", "pieces"])
@pytest.mark.parametrize("tol", [0.0, 3.0])
@pytest.mark.parametrize("B, H, W, oh, ow", [
    (1, 1, 1, 1, 1), (2, 30, 1, 27, 1), (2, 1, 60, 1, 55), (3, 9, 31, 9, 31),
    (2, 12, 2920, 9, 2916),                                                # Middlebury's width: 92 row tiles
    (2, 4, 5 * TILE + 45, 3, 5 * TILE + 7),                                # a row of six tiles, the last one partial
    (2, 350, 5, 333, 3),                                                   # a column of 333: 42 register groups
])
def test_guided_fill_equals_oracle(kind, tol, B, H, W, oh, ow):
    seed = B * 1000 + W + oh + (kind == "pieces")
    fwd, rev = _maps(B, H, W, ow, seed)
    if ow == 1:                                                            # few random values match inside one column
        fwd[:, H - oh + 1::2, W - 1] = 0.25
        rev[:, H - oh + 1::2, W - 1] = 0.25
    if B >= 3:
        fwd[B - 1] = np.nan                                                # an image without a valid pixel stays 0
    wf, v = _check(fwd, rev, _guide(B, oh, ow, kind, seed), oh, ow, tol)
    if oh * ow > 1:
        assert v.any() and not v.all()
    if B >= 3:
        assert not v[-1].any() and (wf[-1] == 0).all()


def test_non_default_lambda_and_sigma():
    B, H, W, oh, ow = 2, 40, 70, 37, 64
    fwd, rev = _maps(B, H, W, ow, 21)
    pred = torch.from_numpy(np.concatenate([fwd, rev])).to(DEV)
    f0, _, v0 = oracle_lr_check(fwd, rev, oh, ow, 1.0)
    for kind, lam, sigma in (("pieces", 0.0, 2.6), ("pieces", 123.456, 7.3), ("random", 1e5, 40.0), ("pieces", 8000.0, 0.7)):
        guide = _guide(B, oh, ow, kind, 22)
        f, u, v = _guided(pred, torch.from_numpy(guide).to(DEV), oh, ow, 1.0, lam, sigma)
        wf, wu = fill_guided(f0, v0, guide, lam=lam, sigma=sigma)
        assert np.array_equal(f.cpu().numpy().view(np.int32), wf.view(np.int32)), (lam, sigma)
        assert np.array_equal(u.cpu().numpy(), wu) and np.array_equal(v.cpu().numpy(), v0)


def test_weight_table_every_entry():
    """The device table against the oracle's, all 766 entries; and through the edge weights: row k of a 766 x 2 guide has
    colour distance k between its two pixels, so the scratch's wh plane (after the table) holds w(k) at (k, 0)."""
    ks = np.arange(766)
    guide = np.zeros((1, 766, 2, 3), dtype=np.uint8)
    guide[0, :, 1] = np.stack([np.minimum(ks, 255), np.clip(ks - 255, 0, 255), np.clip(ks - 510, 0, 255)], -1)
    g = torch.from_numpy(guide).to(DEV)
    B, oh, ow = 1, 766, 2
    pred = torch.zeros((2, oh, ow), device=DEV)
    f = torch.empty((B, oh, ow), device=DEV)
    v = torch.empty((B, oh, ow), dtype=torch.bool, device=DEV)
    flags = torch.empty((B, oh), dtype=torch.uint8, device=DEV)
    scratch = torch.empty(int(_lib.lib().decnet_lr_guided_fill_scratch_floats(B, oh, ow)), device=DEV)
    for sigma in (ops.GUIDED_SIGMA, 1.0, 11.0, 100.0):
        ops._call("decnet_lr_check_guided_fill", pred, pred.data_ptr(), g.data_ptr(), B, oh, ow, oh, ow, 0.0, 1.0, sigma,
                  f.data_ptr(), None, v.data_ptr(), flags.data_ptr(), scratch.data_ptr())
        torch.cuda.synchronize()
        want = weight_table(sigma)
        table = scratch[:766].cpu().numpy()
        assert np.array_equal(table.view(np.int32), want.view(np.int32)), (sigma, np.nonzero(table != want))
        wh = scratch[768:768 + oh * ow].cpu().numpy().reshape(oh, ow)
        assert np.array_equal(wh[:, 0].view(np.int32), want.view(np.int32)) and (wh[:, 1] == 0).all()


def test_guided_entry_arguments():
    pred = torch.zeros((2, 27, 27), device=DEV)
    g = torch.zeros((1, 27, 27, 3), dtype=torch.uint8, device=DEV)
    f = torch.empty((1, 27, 27), device=DEV)
    v = torch.empty((1, 27, 27), dtype=torch.bool, device=DEV)
    flags = torch.empty((1, 27), dtype=torch.uint8, device=DEV)
    scratch = torch.empty(int(_lib.lib().decnet_lr_guided_fill_scratch_floats(1, 27, 27)), device=DEV)
    assert _lib.lib().decnet_lr_guided_fill_scratch_floats(2, 3, 5) == 768 + 5 * 30

    def call(**kw):
        a = dict(guide=g.data_ptr(), oh=27, tol=1.0, lam=8000.0, sigma=2.6, f=f.data_ptr(), v=v.data_ptr(),
                 flags=flags.data_ptr(), scratch=scratch.data_ptr())
        a.update(kw)
        ops._call("decnet_lr_check_guided_fill", pred, pred.data_ptr(), a["guide"], 1, 27, 27, a["oh"], 27, a["tol"], a["lam"],
                  a["sigma"], a["f"], None, a["v"], a["flags"], a["scratch"])

    call()
    for name in ("guide", "f", "v", "flags", "scratch"):
        with pytest.raises(_lib.DecnetError, match="null prediction, guide, float rows, mask, row flags or scratch"):
            call(**{name: None})
    with pytest.raises(_lib.DecnetError, match="crop"):
        call(oh=28)
    with pytest.raises(_lib.DecnetError, match="tolerance"):
        call(tol=-1.0)
    for lam in (-1.0, float("inf"), float("nan")):
        with pytest.raises(_lib.DecnetError, match="lambda must be finite and >= 0"):
            call(lam=lam)
    for sigma in (0.0, -2.0, float("inf"), float("nan")):
        with pytest.raises(_lib.DecnetError, match="sigma_color must be finite and > 0"):
            call(sigma=sigma)
    with pytest.raises(ValueError, match="guide must be a contiguous CUDA uint8"):
        ops.lr_check(pred, 27, 27, 1.0, fill="guided", guide=g[:, :, :26])
    with pytest.raises(ValueError, match="guide must be a contiguous CUDA uint8"):
        ops.lr_check(pred, 27, 27, 1.0, fill="guided", guide=g.cpu())
    with pytest.raises(ValueError, match="guide must be a contiguous CUDA uint8"):
        ops.lr_check(pred, 27, 27, 1.0, fill="guided", guide=g.float())
    with pytest.raises(ValueError, match="guide must be a contiguous CUDA uint8"):
        ops.lr_check(pred, 27, 27, 1.0, fill="guided", guide=g.transpose(1, 2))
    with pytest.raises(ValueError, match="guide is required"):
        ops.lr_check(pred, 27, 27, 1.0, fill="background", guide=g)


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
    captures = m.captures
    filled, fvalid = m(l, r, return_valid=True, fill="guided")
    wf, wu = fill_guided(disp.cpu().numpy(), valid.cpu().numpy(), l.cpu().numpy())
    assert torch.equal(fvalid, valid) and not bool(valid.all())
    assert np.array_equal(filled.cpu().numpy().view(np.int32), wf.view(np.int32))
    assert np.array_equal(m(l, r, output="u16", fill="guided").cpu().numpy(), wu)
    assert m.captures == captures and list(m._graphs) == [(B, h, w, 216, masks, "fp32", "lr")]
    dense = _matcher(masks, skip, fill="guided")
    assert torch.equal(dense(l, r), filled) and torch.equal(dense(l, r, fill="none"), disp)


def test_host_kinds_lists_and_stream():
    m = _matcher(fill="guided")
    l, r = _images(2, 60, 90, 7)
    want_d, want_v = m(l, r, return_valid=True)
    assert not bool(want_v.all()) and torch.equal(want_d, m(l, r, fill="guided"))
    d, v = m(l.cpu().numpy(), r.cpu().numpy(), return_valid=True)
    assert isinstance(d, np.ndarray) and d.dtype == np.float32 and v.dtype == np.bool_
    assert np.array_equal(d, want_d.cpu().numpy()) and np.array_equal(v, want_v.cpu().numpy())
    d, v = m(l[0].cpu(), r[0].cpu(), output="u16", return_valid=True)
    assert not d.is_cuda and d.dtype == torch.uint16 and d.shape == (60, 90) and torch.equal(v, want_v[0].cpu())
    listed = m([l[0].cpu().numpy(), l[1].cpu().numpy()], [r[0].cpu().numpy(), r[1].cpu().numpy()], return_valid=True)
    for i, (ld, lv) in enumerate(listed):
        assert np.array_equal(ld, want_d[i].cpu().numpy()) and np.array_equal(lv, want_v[i].cpu().numpy())
    # five items of one shape, then another: both buffer sets are reused while the next upload is in flight, and each
    # fill must read its own left images, not the next upload's
    sizes = [(60, 90)] * 5 + [(54, 81), (54, 81), (54, 81)]
    items = [tuple(t.cpu().numpy() for t in _images(2, hh, ww, 30 + i)) for i, (hh, ww) in enumerate(sizes)]
    want = [m(a, b, output="u16", return_valid=True) for a, b in items]
    got = list(m.stream(items, output="u16", return_valid=True))
    assert len(got) == len(want)
    for (gd, gv), (wd, wv) in zip(got, want):
        assert isinstance(gd, np.ndarray) and np.array_equal(gd, wd) and np.array_equal(gv, wv)
    cuda_items = [tuple(torch.from_numpy(t).to(DEV) for t in it) for it in items]
    plain = _matcher()
    for a, (x, y) in zip(plain.stream(cuda_items, fill="guided"), cuda_items):
        assert a.is_cuda and torch.equal(a, plain(x, y, fill="guided")) and torch.equal(a, m(x, y))


def test_guided_call_runs_only_our_kernels_after_the_replay():
    m = _matcher(fill="guided")
    l, r = _images(1, 60, 90, 8)
    m(l, r)
    (st,) = m._graphs[(1, 60, 90, 216, "learned", "fp32", "lr")]
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof, torch.no_grad():
        m._result(st, 60, 90, "u16", 1.0, True, "guided")                  # what runs between the replay and the result
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    for k in ("lr_check_fill_rows_kernel", "guided_table_kernel", "guided_prep_kernel", "guided_rows_kernel",
              "guided_cols_kernel", "guided_compose_kernel"):
        assert any(k in n for n in kernels), (k, kernels)
    bad = [n for n in kernels if "at::native" in n]
    assert not bad, bad
