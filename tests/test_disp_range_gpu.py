"""GPU: the search range [min_disp, max_disp).  The shifted prepare against the plain prepare of oracle.disp_range's shifted
image, disp_add against ATen's add, and StereoMatcher(min_disp=...) against its definition: the plain matcher on
(L, shift(R, k)) at the range's width, plus k; with the left-right check, ops.lr_check of both directions built that way.
Bit for bit throughout."""
import numpy as np
import pytest
import torch

from decnet_b200 import StereoMatcher, ops
from oracle.disp_range import shift_cols_u8

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
D = 108                                                                    # the width every matcher test searches


def _images(B, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8),
            torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8))


def _shift(img, k):
    return torch.from_numpy(shift_cols_u8(img.cpu().numpy(), k)).to(DEV)


def _flip(t):
    return torch.flip(t, [-2]).contiguous()


# ------------------------------------------------------------------------------------------------------ shifted prepare
@pytest.mark.parametrize("B, h, w", [(3, 31, 47), (1, 1, 1), (2, 28, 55), (4, 5, 30)])
@pytest.mark.parametrize("outputs", [(True, False), (False, True), (True, True)])
def test_shifted_prepare_equals_prepare_of_shifted_image(B, h, w, outputs):
    img, _ = _images(B, h, w, B * h + w)
    want01, want_norm = outputs
    for k in sorted({0, 1, -1, 26, 27, w - 1, w, w + 5, -w - 5}):
        got = ops.image_prepare_u8(img, want01=want01, want_norm=want_norm, col_shift=k)
        want = ops.image_prepare_u8(_shift(img, k), want01=want01, want_norm=want_norm)
        for g, t in zip(got, want):
            assert (g is None) == (t is None)
            if g is not None:
                assert torch.equal(g, t), (k, B, h, w)


def test_shifted_prepare_arguments():
    img, _ = _images(1, 4, 5, 1)
    for bad in (1.0, True, "1", None):
        with pytest.raises(ValueError, match="col_shift"):
            ops.image_prepare_u8(img, col_shift=bad)
    for k in (np.int64(3), 2**40, -2**40):                                 # any integer: beyond +-w all black
        got = ops.image_prepare_u8(img, col_shift=k)
        want = ops.image_prepare_u8(_shift(img, int(k)))
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


# ------------------------------------------------------------------------------------------------------------ disp_add
def _specials(n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(n, device=DEV, generator=g) * 300
    special = torch.tensor([float("nan"), float("inf"), -float("inf"), -0.0, 0.0, 3.4e38, -3.4e38, 1e-45, -27.0],
                           device=DEV)
    idx = torch.randint(0, n, (max(1, n // 5),), device=DEV, generator=g)
    x[idx] = special[torch.randint(0, len(special), idx.shape, device=DEV, generator=g)]
    return x


def _same_bits(a, b):
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a.view(torch.int32)[~na], b.view(torch.int32)[~nb])


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 1023, 4099, 3 * 65 * 259])
@pytest.mark.parametrize("start", [0, 1, 2, 3])
def test_disp_add_equals_aten(n, start):
    buf = _specials(n + start + 3, n + start)
    before = buf.clone()
    view = buf[start:start + n]                                            # contiguous, off the 16-byte alignment for start > 0
    for k in (27, -40, 0, 243, 0.5, 2**24):
        want = view + torch.tensor(k, dtype=torch.float32, device=DEV)
        assert ops.disp_add(view, k) is view
        assert _same_bits(view, want), (n, start, k)
        view.copy_(before[start:start + n])
    assert _same_bits(buf[:start], before[:start]) and _same_bits(buf[start + n:], before[start + n:])


def test_disp_add_shapes_and_arguments():
    x = _specials(2 * 31 * 47, 5).view(2, 31, 47)
    want = x + 27
    assert _same_bits(ops.disp_add(x, 27), want)
    assert ops.disp_add(torch.empty(0, device=DEV), 27).numel() == 0
    for bad in (True, float("nan"), 1e39, 0.1, "1"):
        with pytest.raises(ValueError, match="offset"):
            ops.disp_add(x, bad)
    with pytest.raises(TypeError):
        ops.disp_add(x.double(), 1)
    with pytest.raises(ValueError):
        ops.disp_add(x[:, :, ::2], 1)


# ------------------------------------------------------------------------------------------------------------ matcher
_MATCHERS = {}


def _matcher(masks="learned", skip=4, lr=None):
    if (masks, skip, lr) not in _MATCHERS:
        _MATCHERS[(masks, skip, lr)] = StereoMatcher(masks=masks, skip_stage_id=skip, lr_check=lr, max_graphs=8)
    return _MATCHERS[(masks, skip, lr)]


@pytest.mark.parametrize("masks", ["learned", "image"])
@pytest.mark.parametrize("skip", [4, 3])
def test_matcher_equals_definition(masks, skip):
    m = _matcher(masks, skip)
    B, h, w = 2, 50, 130
    l, r = _images(B, h, w, 11)
    for k in (27, 100, -40):
        plain = m(l, _shift(r, k), max_disp=D)
        want = plain + torch.tensor(k, dtype=torch.float32, device=DEV)
        got = m(l, r, min_disp=k, max_disp=k + D)
        assert torch.equal(got, want), k
        assert (B, h, w, D, masks, "fp32", ("min_disp", k)) in m._graphs
        u16 = m(l, r, output="u16", min_disp=k, max_disp=k + D)
        assert np.array_equal(u16.cpu().numpy(), ops.disp_to_u16(want.contiguous(), h, w).cpu().numpy())


@pytest.mark.parametrize("fill", ["none", "background", "guided"])
@pytest.mark.parametrize("speckle", [0, 20])
def test_lr_check_equals_definition(fill, speckle):
    m, m_lr = _matcher(), _matcher(lr=1.0)
    B, h, w = 2, 50, 130
    l, r = _images(B, h, w, 12)
    for k in (27, -40):
        off = torch.tensor(k, dtype=torch.float32, device=DEV)
        fwd = m(l, _shift(r, k), max_disp=D) + off
        rev = m(_flip(r), _shift(_flip(l), k), max_disp=D) + off                # the reverse run, not yet mirrored back
        pred = torch.cat([fwd, rev]).contiguous()
        want_f, want_u, want_v = ops.lr_check(pred, h, w, 1.0, float_out=True, u16_out=True, valid_out=True, fill=fill,
                                              guide=l if fill == "guided" else None, speckle_size=speckle)
        kw = dict(min_disp=k, max_disp=k + D, fill=fill, speckle_size=speckle)
        got_f, got_v = m_lr(l, r, return_valid=True, **kw)
        assert torch.equal(got_f, want_f) and torch.equal(got_v, want_v), k
        got_u = m_lr(l, r, output="u16", **kw)
        assert np.array_equal(got_u.cpu().numpy(), want_u.cpu().numpy())


def _entries(fn):
    """The C entries fn() calls through ops._call, in order.  (A spy rather than torch.profiler: every profiler session
    tears CUPTI down at its end, and the next one can miss its first kernels, which the profiler tests of the left-right
    check rely on seeing.)"""
    called, real = [], ops._call

    def spy(name, *args):
        called.append(name)
        return real(name, *args)
    with pytest.MonkeyPatch.context() as mp, torch.no_grad():
        mp.setattr(ops, "_call", spy)
        fn()
        torch.cuda.synchronize()
    return called


def test_zero_start_is_todays_graph():
    m = StereoMatcher()
    l, r = _images(1, 60, 90, 3)
    a = m(l, r)
    assert m.captures == 1
    b = m(l, r, min_disp=0)
    c = m(l, r, min_disp=0, max_disp=216)
    assert m.captures == 1 and torch.equal(a, b) and torch.equal(a, c)
    assert list(m._graphs) == [(1, 60, 90, 216, "learned", "fp32")]
    (st,) = m._graphs[(1, 60, 90, 216, "learned", "fp32")]
    called = _entries(lambda: m._step(st))                                # what the graph holds, launched eagerly
    assert called.count("decnet_image_prepare_u8") == 2
    assert "decnet_disp_add" not in called and "decnet_image_prepare_u8_shift" not in called


def test_new_start_captures_once_then_replays():
    m = StereoMatcher(max_graphs=8)
    l, r = _images(1, 60, 90, 4)
    first = m(l, r, min_disp=27, max_disp=243)
    assert m.captures == 1
    assert torch.equal(m(l, r, min_disp=27, max_disp=243), first) and m.captures == 1
    key = (1, 60, 90, 216, "learned", "fp32", ("min_disp", 27))
    assert list(m._graphs) == [key]
    (st,) = m._graphs[key]
    called = _entries(lambda: m._step(st))
    assert called.count("decnet_image_prepare_u8") == called.count("decnet_image_prepare_u8_shift") == 1
    assert called.count("decnet_disp_add") == 1 and called[-1] == "decnet_disp_add"      # the step's last launch
    other = StereoMatcher(min_disp=27, max_disp=243)
    assert (other.min_disp, other.max_disp) == (27, 243)
    assert torch.equal(other(l, r), first)


def test_host_kinds_lists_and_stream():
    m = _matcher(lr=1.0)
    kw = dict(min_disp=-40, max_disp=-40 + D)
    l, r = _images(2, 60, 90, 7)
    want_d, want_v = m(l, r, return_valid=True, **kw)
    d, v = m(l.cpu().numpy(), r.cpu().numpy(), return_valid=True, **kw)
    assert isinstance(d, np.ndarray) and np.array_equal(d, want_d.cpu().numpy()) and np.array_equal(v, want_v.cpu().numpy())
    d = m(l[0].cpu(), r[0].cpu(), **kw)
    assert not d.is_cuda and torch.equal(d, want_d[0].cpu())
    listed = m([l[0].cpu().numpy(), l[1].cpu().numpy()], [r[0].cpu().numpy(), r[1].cpu().numpy()], **kw)
    for i, ld in enumerate(listed):
        assert np.array_equal(ld, want_d[i].cpu().numpy())
    sizes = [(60, 90), (60, 90), (54, 81), (60, 90)]
    items = [tuple(t.cpu().numpy() for t in _images(2, hh, ww, 30 + i)) for i, (hh, ww) in enumerate(sizes)]
    want = [m(a, b, output="u16", **kw) for a, b in items]
    got = list(m.stream(items, output="u16", **kw))
    assert len(got) == len(want)
    for g, w_ in zip(got, want):
        assert isinstance(g, np.ndarray) and np.array_equal(g, w_)
    cuda_items = [tuple(torch.from_numpy(t).to(DEV) for t in it) for it in items]
    for a, b in zip(m.stream(cuda_items, lr_check=None, **kw), [m(x, y, **kw) for x, y in cuda_items]):
        assert a.is_cuda and torch.equal(a, b)
