"""GPU: the speckle filter of the left-right check.  ops.lr_check(..., speckle_size, speckle_range, fill=...) against
oracle.lr_check, then oracle.lr_speckle.filter_speckles, then the fill's oracle, bit for bit, for every output subset and
all three fills, on shapes around the labeller's 32 x 32 tiles and structures that cross every tile; the C entry's off
switch and argument rules; and StereoMatcher's speckle filter against its definition: the filter and the fill applied to
the same call's (disparity, valid) without one."""
import numpy as np
import pytest
import torch

from decnet_b200 import StereoMatcher, _lib, ops
from oracle.codec import disp_to_u16
from oracle.lr_check import lr_check as oracle_lr_check
from oracle.lr_fill import fill_background
from oracle.lr_guided import fill_guided
from oracle.lr_speckle import filter_speckles

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
TILE = 32                                                                  # the labeller's tiles are TILE x TILE pixels
FILLS = ("none", "background", "guided")
SUBSETS = [(f, u, v) for f in (False, True) for u in (False, True) for v in (False, True) if f or u or v]
PASS_ALL = 3e38                                                            # with a zero reverse map: see _feed


def _images(B, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8),
            torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8))


def _maps(B, H, W, ow, seed):
    """Padded forward / reverse predictions as test_lr_guided_gpu's: NaN, +-inf, negative and > 256 values, half-pixel ties,
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


def _feed(crop, H, W):
    """Padded (fwd, rev) that make the check return `crop` [B,h,w] as it is, NaN marking an invalid pixel: with tol 3e38
    and a zero reverse map, a forward value in (-0.5, 0.5] matches its own column, so it passes at every column."""
    B, h, w = crop.shape
    fwd = np.full((B, H, W), np.nan, dtype=np.float32)
    fwd[:, H - h:, W - w:] = crop
    return fwd, np.zeros((B, H, W), dtype=np.float32)


def _guide(B, h, w, seed):
    """Piecewise-constant blocks of a few colours with strong edges between them and mild noise inside."""
    g = np.random.default_rng(seed)
    cells = g.integers(0, 256, (B, h // 7 + 1, w // 11 + 1, 3))
    out = cells[:, np.arange(h) // 7][:, :, np.arange(w) // 11] + g.integers(0, 3, (B, h, w, 3))
    return np.clip(out, 0, 255).astype(np.uint8)


def _same(got, want, what):
    if want.dtype == np.float32:
        assert got.dtype == torch.float32 and np.array_equal(got.cpu().numpy().view(np.int32), want.view(np.int32)), what
    else:
        assert np.array_equal(got.cpu().numpy(), want), what


def _check(fwd, rev, oh, ow, tol, size, rng, seed=0):
    """Every fill and output subset of ops.lr_check with the filter against the oracle composition; -> the oracle's mask."""
    B = fwd.shape[0]
    pred = torch.from_numpy(np.concatenate([fwd, rev])).to(DEV)
    guide = _guide(B, oh, ow, seed)
    f, _, v = oracle_lr_check(fwd, rev, oh, ow, tol)
    d2, v2 = filter_speckles(f, v, size, rng)
    wants = {"none": (d2, disp_to_u16(d2, oh, ow)), "background": fill_background(d2, v2),
             "guided": fill_guided(d2, v2, guide)}
    for fill in FILLS:
        wf, wu = wants[fill]
        g = torch.from_numpy(guide).to(DEV) if fill == "guided" else None
        for fo, uo, vo in SUBSETS:
            got = list(ops.lr_check(pred, oh, ow, tol, float_out=fo, u16_out=uo, valid_out=vo, fill=fill, guide=g,
                                    speckle_size=size, speckle_range=rng))
            assert len(got) == fo + uo + vo
            what = (fill, fo, uo, vo, size, rng)
            if fo:
                _same(got.pop(0), wf, what)
            if uo:
                _same(got.pop(0), wu, what)
            if vo:
                t = got.pop(0)
                assert t.dtype == torch.bool and np.array_equal(t.cpu().numpy(), v2), what
    return v, v2


SHAPES = [
    (1, 1, 1, 1, 1), (2, 1, 70, 1, 65), (2, 70, 1, 65, 1),                 # one pixel, a single row, a single column
    (3, 45, 77, 40, 70),                                                   # not tile multiples, B >= 3
    (2, 70, 2920, 66, 2916),                                               # Middlebury's width
    (1, 5, 4200, 4, 4150),                                                 # rows wider than the fill's 4096-column chunk
]


@pytest.mark.parametrize("B, H, W, oh, ow", SHAPES)
def test_random_predictions(B, H, W, oh, ow):
    """The check of _maps' predictions: mostly one- and few-pixel regions, so most pixels the check passes go."""
    fwd, rev = _maps(B, H, W, ow, B * 100 + W + oh)
    v, v2 = _check(fwd, rev, oh, ow, 3.0, 4, 1.0, seed=W)
    if oh * ow > 100:
        assert v.any() and v2.sum() < v.sum()


@pytest.mark.parametrize("B, H, W, oh, ow", SHAPES)
def test_random_fed_maps(B, H, W, oh, ow):
    """Fed maps of k/64 levels, 80 % valid: regions of every size."""
    g = np.random.default_rng(oh * 7 + ow)
    crop = (np.clip(np.round(np.cumsum(g.normal(0, 1.5, (B, oh, ow)), axis=2) % 48) - 16, -31, 32) / 64).astype(np.float32)
    crop[g.random((B, oh, ow)) < 0.2] = np.nan
    fwd, rev = _feed(crop, H, W)
    for size, rng in ((3, 1 / 64), (25, 0.0)):
        v, v2 = _check(fwd, rev, oh, ow, PASS_ALL, size, rng, seed=ow)
        assert np.array_equal(v, ~np.isnan(crop))


def _serpentine(h, w):
    """One-pixel-wide path: every even row, joined by the last or the first column of the odd row between them."""
    m = np.zeros((h, w), dtype=bool)
    m[::2] = True
    m[1::4, -1] = True
    m[3::4, 0] = True
    return m


def _spiral(h, w):
    """One-pixel-wide square spiral inwards from the top-left corner, one-pixel gaps between its turns: segments of
    w-1 right, h-1 down, w-1 left, h-3 up, w-3 right, h-5 down, ..."""
    m = np.zeros((h, w), dtype=bool)
    y = x = 0
    m[0, 0] = True
    lens = [w - 1, h - 1, w - 1] + [n for k in range(1, max(h, w)) for n in (h - 1 - 2 * k, w - 1 - 2 * k)]
    for i, n in enumerate(lens):
        if n <= 0:
            break
        dy, dx = ((0, 1), (1, 0), (0, -1), (-1, 0))[i % 4]
        for _ in range(n):
            y, x = y + dy, x + dx
            m[y, x] = True
    return m


@pytest.mark.parametrize("kind", ["serpentine", "spiral"])
@pytest.mark.parametrize("B, H, W, oh, ow", [(2, 100, 140, 97, 131), (1, 70, 2920, 64, 2916)])
def test_paths_spanning_every_tile(kind, B, H, W, oh, ow):
    """A constant one-pixel-wide path through every tile is one region of n pixels: kept at max_size n - 1, gone at n."""
    m = (_serpentine if kind == "serpentine" else _spiral)(oh, ow)
    n = int(m.sum())
    crop = np.where(m, np.float32(0.25), np.float32(np.nan))[None].repeat(B, 0)
    fwd, rev = _feed(crop, H, W)
    _, v2 = _check(fwd, rev, oh, ow, PASS_ALL, n - 1, 0.0)
    assert np.array_equal(v2, crop == 0.25)
    _, v2 = _check(fwd, rev, oh, ow, PASS_ALL, n, 0.0)
    assert not v2.any()


def test_checkerboard_all_single_pixels():
    B, H, W, oh, ow = 2, 70, 100, 66, 99
    y, x = np.mgrid[0:oh, 0:ow]
    crop = np.where((x + y) % 2 == 0, np.float32(0.5), np.float32(np.nan))[None].repeat(B, 0)
    fwd, rev = _feed(crop, H, W)
    _, v2 = _check(fwd, rev, oh, ow, PASS_ALL, 1, 1.0)
    assert not v2.any()


def test_regions_of_max_size_and_one_more_across_tile_corners():
    B, H, W, oh, ow, size = 2, 100, 100, 96, 96, 4
    crop = np.full((B, oh, ow), np.nan, dtype=np.float32)
    crop[:, 31:33, 31:33] = 0.125                                          # 4 pixels, one in each of four tiles: goes
    crop[:, 63:65, 63:65] = -0.25                                          # 5 pixels around another corner: stays
    crop[:, 62, 63] = -0.25
    crop[:, 31, 63:65] = 0.5                                               # 4 pixels across a vertical border, then
    crop[:, 32, 63:65] = 0.5
    crop[:, 63:65, 31] = 0.0                                               # 3 + 2 across a horizontal border: stays
    crop[:, 63:66, 32] = 0.0
    fwd, rev = _feed(crop, H, W)
    _, v2 = _check(fwd, rev, oh, ow, PASS_ALL, size, 0.0)
    assert not v2[:, 31:33, 31:33].any() and v2[:, 63:65, 63:65].all() and not v2[:, 31:33, 63:65].any()
    assert v2[:, 63:66, 32].all() and int(v2.sum()) == B * 10


@pytest.mark.parametrize("B, H, W, oh, ow", [(3, 45, 77, 40, 70), (1, 300, 400, 290, 390)])
def test_all_valid_constant_map(B, H, W, oh, ow):
    crop = np.full((B, oh, ow), 0.375, dtype=np.float32)
    fwd, rev = _feed(crop, H, W)
    _, v2 = _check(fwd, rev, oh, ow, PASS_ALL, oh * ow - 1, 0.0)
    assert v2.all()
    _, v2 = _check(fwd, rev, oh, ow, PASS_ALL, oh * ow, 0.0)
    assert not v2.any()


def test_ramps_whose_step_equals_the_range():
    B, H, W, oh, ow = 2, 80, 100, 75, 97
    y, x = np.mgrid[0:oh, 0:ow]
    crop = (((x // 3 + y // 5) % 60) - 29).astype(np.float32) / 64        # steps of 1/64, a jump of 59/64 at the wrap
    crop = crop[None].repeat(B, 0)
    crop[1, ::9] = np.nan
    fwd, rev = _feed(crop, H, W)
    for rng, size in ((1 / 64, 200), (0.99 / 64, 14), (0.0, 15)):
        _check(fwd, rev, oh, ow, PASS_ALL, size, rng)


def test_piecewise_planar_scene():
    """Mostly valid, a few image-sized regions (the count's contention case), with scattered islands."""
    B, H, W, oh, ow = 2, 280, 400, 270, 390
    y, x = np.mgrid[0:oh, 0:ow]
    crop = np.where(x < 150, np.round((x * 0.001 + y * 0.002) * 64) / 64 - 0.4,
                    np.round((0.3 - x * 0.0005) * 64) / 64).astype(np.float32)[None].repeat(B, 0)
    g = np.random.default_rng(3)
    crop[g.random(crop.shape) < 0.03] = np.nan
    isl = g.random(crop.shape) < 0.01
    crop[isl] = 0.5
    fwd, rev = _feed(crop, H, W)
    v, v2 = _check(fwd, rev, oh, ow, PASS_ALL, 50, 1 / 64)
    assert v2.sum() > 0.9 * v.sum() and v2.sum() < v.sum()


# ------------------------------------------------------------------------------------------------------------ C entry
def _entry(pred, oh, ow, tol, size, rng, fill, guide=None, u16=True, valid=True):
    B = pred.shape[0] // 2
    f = torch.empty((B, oh, ow), device=DEV)
    u = torch.empty((B, oh, ow), dtype=torch.uint16, device=DEV) if u16 else None
    v = torch.empty((B, oh, ow), dtype=torch.bool, device=DEV) if valid else None
    flags = torch.empty((B, oh), dtype=torch.uint8, device=DEV)
    scratch = torch.empty(int(_lib.lib().decnet_lr_speckle_scratch_bytes(B, oh, ow, fill)), dtype=torch.uint8, device=DEV)
    ops._call("decnet_lr_check_speckle", pred, pred.data_ptr(), guide.data_ptr() if guide is not None else None, B,
              *pred.shape[1:], oh, ow, tol, size, rng, fill, ops.GUIDED_LAMBDA, ops.GUIDED_SIGMA, f.data_ptr(),
              u.data_ptr() if u is not None else None, v.data_ptr() if v is not None else None, flags.data_ptr(),
              scratch.data_ptr())
    return f, u, v


def test_size_zero_is_the_entries_without_the_filter():
    B, H, W, oh, ow = 2, 40, 70, 37, 64
    fwd, rev = _maps(B, H, W, ow, 5)
    pred = torch.from_numpy(np.concatenate([fwd, rev])).to(DEV)
    guide = torch.from_numpy(_guide(B, oh, ow, 5)).to(DEV)
    for fill in FILLS:
        g = guide if fill == "guided" else None
        want = ops.lr_check(pred, oh, ow, 1.0, True, True, True, fill=fill, guide=g)
        got = _entry(pred, oh, ow, 1.0, 0, 1.0, FILLS.index(fill), g)
        for a, b in zip(got, want):
            assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                               b.view(torch.int32) if b.dtype == torch.float32 else b), fill


def test_entry_arguments():
    lib = _lib.lib()
    n = 2 * 3 * 5
    assert lib.decnet_lr_speckle_scratch_bytes(2, 3, 5, 0) == lib.decnet_lr_speckle_scratch_bytes(2, 3, 5, 1) == 368
    assert lib.decnet_lr_speckle_scratch_bytes(2, 3, 5, 2) == 368 + 4 * (768 + 5 * n)
    pred = torch.zeros((2, 27, 27), device=DEV)
    g = torch.zeros((1, 27, 27, 3), dtype=torch.uint8, device=DEV)
    _entry(pred, 27, 27, 1.0, 5, 1.0, 0)
    with pytest.raises(_lib.DecnetError, match="fill must be 0"):
        _entry(pred, 27, 27, 1.0, 5, 1.0, 3)
    with pytest.raises(_lib.DecnetError, match="guide is required"):
        _entry(pred, 27, 27, 1.0, 5, 1.0, 2)
    with pytest.raises(_lib.DecnetError, match="guide is required"):
        _entry(pred, 27, 27, 1.0, 5, 1.0, 1, g)
    with pytest.raises(_lib.DecnetError, match="speckle size"):
        _entry(pred, 27, 27, 1.0, -1, 1.0, 0)
    for bad in (-1.0, float("inf"), float("nan")):
        with pytest.raises(_lib.DecnetError, match="speckle range"):
            _entry(pred, 27, 27, 1.0, 5, bad, 1)
    with pytest.raises(_lib.DecnetError, match="crop"):
        _entry(pred, 28, 27, 1.0, 5, 1.0, 0)
    with pytest.raises(_lib.DecnetError, match="tolerance"):
        _entry(pred, 27, 27, -1.0, 5, 1.0, 0)
    with pytest.raises(_lib.DecnetError, match="guided fill needs the mask"):
        _entry(pred, 27, 27, 1.0, 5, 1.0, 2, g, valid=False)
    big = torch.zeros((2, 1, 1), device=DEV)                               # B * ori_h * ori_w >= 2^31: checked before use
    with pytest.raises(_lib.DecnetError, match="int32 labels"):
        ops._call("decnet_lr_check_speckle", big, big.data_ptr(), None, 65536, 32768, 1, 32768, 1, 1.0, 5, 1.0, 0, 8000.0,
                  2.6, None, None, big.data_ptr(), None, big.data_ptr())


# ------------------------------------------------------------------------------------------------------------ matcher
_MATCHERS = {}


def _matcher(masks="learned", skip=4, lr=1.0, fill="none", size=0, rng=1.0):
    key = (masks, skip, lr, fill, size, rng)
    if key not in _MATCHERS:
        _MATCHERS[key] = StereoMatcher(masks=masks, skip_stage_id=skip, lr_check=lr, fill=fill, speckle_size=size,
                                       speckle_range=rng)
    return _MATCHERS[key]


@pytest.mark.parametrize("masks", ["learned", "image"])
@pytest.mark.parametrize("skip", [4, 3])
def test_matcher_equals_definition(masks, skip):
    m = _matcher(masks, skip)
    B, h, w = 2, 130, 260
    l, r = _images(B, h, w, 11)
    disp, valid = m(l, r, return_valid=True)
    keys, captures = list(m._graphs), m.captures
    d2, v2 = filter_speckles(disp.cpu().numpy(), valid.cpu().numpy(), 20, 1.0)
    assert v2.sum() < valid.sum().item()
    wants = {"none": (d2, disp_to_u16(d2, h, w)), "background": fill_background(d2, v2),
             "guided": fill_guided(d2, v2, l.cpu().numpy())}
    for fill, (wf, wu) in wants.items():
        got, gv = m(l, r, return_valid=True, fill=fill, speckle_size=20, speckle_range=1.0)
        _same(got, wf, fill)
        assert np.array_equal(gv.cpu().numpy(), v2)
        _same(m(l, r, output="u16", fill=fill, speckle_size=20), wu, fill)
    assert m.captures == captures and list(m._graphs) == keys == [(B, h, w, 216, masks, "fp32", "lr")]
    dense = _matcher(masks, skip, fill="background", size=20)
    assert torch.equal(dense(l, r), m(l, r, fill="background", speckle_size=20))
    assert torch.equal(dense(l, r, speckle_size=0, fill="none"), disp)


def test_host_kinds_lists_and_stream():
    m = _matcher(fill="background", size=12, rng=2.0)
    l, r = _images(2, 60, 90, 7)
    want_d, want_v = m(l, r, return_valid=True)
    d, v = m(l.cpu().numpy(), r.cpu().numpy(), return_valid=True)
    assert isinstance(d, np.ndarray) and np.array_equal(d, want_d.cpu().numpy()) and np.array_equal(v, want_v.cpu().numpy())
    d, v = m(l[0].cpu(), r[0].cpu(), output="u16", return_valid=True)
    assert not d.is_cuda and d.dtype == torch.uint16 and d.shape == (60, 90) and torch.equal(v, want_v[0].cpu())
    listed = m([l[0].cpu().numpy(), l[1].cpu().numpy()], [r[0].cpu().numpy(), r[1].cpu().numpy()], return_valid=True)
    for i, (ld, lv) in enumerate(listed):
        assert np.array_equal(ld, want_d[i].cpu().numpy()) and np.array_equal(lv, want_v[i].cpu().numpy())
    sizes = [(60, 90)] * 5 + [(54, 81), (54, 81), (54, 81)]
    items = [tuple(t.cpu().numpy() for t in _images(2, hh, ww, 30 + i)) for i, (hh, ww) in enumerate(sizes)]
    for fill in FILLS:
        want = [m(a, b, output="u16", return_valid=True, fill=fill) for a, b in items]
        got = list(m.stream(items, output="u16", return_valid=True, fill=fill))
        assert len(got) == len(want)
        for (gd, gv), (wd, wv) in zip(got, want):
            assert isinstance(gd, np.ndarray) and np.array_equal(gd, wd) and np.array_equal(gv, wv)
    cuda_items = [tuple(torch.from_numpy(t).to(DEV) for t in it) for it in items]
    plain = _matcher()
    for a, (x, y) in zip(plain.stream(cuda_items, fill="background", speckle_size=12, speckle_range=2.0), cuda_items):
        assert a.is_cuda and torch.equal(a, plain(x, y, fill="background", speckle_size=12, speckle_range=2.0))
        assert torch.equal(a, m(x, y))


def test_speckle_call_runs_only_our_kernels_after_the_replay():
    m = _matcher(fill="guided", size=10)
    l, r = _images(1, 60, 90, 8)
    m(l, r)
    (st,) = m._graphs[(1, 60, 90, 216, "learned", "fp32", "lr")]
    torch.cuda.synchronize()
    for fill, names in (("none", ("speckle_apply_kernel",)),
                        ("guided", ("lr_check_fill_rows_kernel", "lr_fill_empty_rows_kernel", "guided_rows_kernel"))):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof, torch.no_grad():
            m._result(st, 60, 90, "u16", 1.0, True, fill, (10, 1.0))         # what runs between the replay and the result
            torch.cuda.synchronize()
        kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        for k in ("speckle_tile_kernel", "speckle_merge_kernel", "speckle_count_kernel") + names:
            assert any(k in n for n in kernels), (k, kernels)
        bad = [n for n in kernels if "at::native" in n]
        assert not bad, bad
