"""GPU: the left-right check's kernels against torch.flip and oracle.lr_check, and StereoMatcher(lr_check=...)
against its definition: the plain matcher on (L, R) and on (mirror(R), mirror(L)), compared by the oracle.  Bit for bit,
which also shows that a pair's result does not depend on the other pairs of its batch (the LR graph runs at 2B)."""
import numpy as np
import pytest
import torch

from decnet_b200 import StereoMatcher, ops
from oracle.lr_check import lr_check as oracle_lr_check

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)


def _images(B, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8),
            torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8))


def _flip(t):
    return torch.flip(t, [-2 if t.dim() == 4 else -1])


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("h, w", [(1, 1), (3, 5), (7, 13), (6, 16), (5, 20), (2, 48), (130, 260)])
def test_mirror_swap_equals_flip(B, h, w):
    l, r = _images(B, h, w, h * 1000 + w)
    both_l, both_r = torch.empty((2 * B, h, w, 3), dtype=torch.uint8, device=DEV), torch.empty((2 * B, h, w, 3),
                                                                                                  dtype=torch.uint8, device=DEV)
    both_l[:B], both_r[:B] = l, r
    ops.mirror_swap_u8(both_l[:B], both_r[:B], both_l[B:], both_r[B:])    # into the second half, as the matcher does
    assert torch.equal(both_l[B:], _flip(r)) and torch.equal(both_r[B:], _flip(l))
    assert torch.equal(both_l[:B], l) and torch.equal(both_r[:B], r)


@pytest.mark.parametrize("offset", [1, 4])
def test_mirror_swap_unaligned(offset):
    """Views that start off a 16-byte boundary take the word or byte path."""
    B, h, w = 2, 9, 32
    n = B * h * w * 3
    l, r = _images(B, h, w, offset)
    buf = torch.zeros(4 * n + 64, dtype=torch.uint8, device=DEV)
    views = [buf[offset + k * (n + offset):offset + k * (n + offset) + n].view(B, h, w, 3) for k in range(4)]
    views[0].copy_(l)
    views[1].copy_(r)
    ops.mirror_swap_u8(views[0], views[1], views[2], views[3])
    assert torch.equal(views[2], _flip(r)) and torch.equal(views[3], _flip(l))


def _maps(B, H, W, ow, seed):
    """Padded forward / reverse predictions with NaN, +-inf, negative and > 256 values, a quarter of them half-pixel ties
    (x - (k + 0.5) + 0.5 is integral), and a reverse map that agrees with the forward one within 0..4 px at most matched
    columns of the crop (else few pixels would be valid)."""
    g = np.random.default_rng(seed)
    fwd = (g.integers(-8, 90, (B, H, W)) + g.choice([0.0, 0.5, 0.25, 0.75], (B, H, W))).astype(np.float32)
    fwd[g.random((B, H, W)) < 0.02] = 300.5
    for v in (np.nan, np.inf, -np.inf):
        fwd[g.random((B, H, W)) < 0.01] = v
    rev = g.normal(40, 30, (B, H, W)).astype(np.float32)
    x = np.arange(W, dtype=np.float32) - np.float32(W - ow)              # column within the crop
    with np.errstate(invalid="ignore"):
        u = np.floor((x - fwd) + np.float32(0.5))
    for b in range(B):
        for y in range(H):
            for xx in range(W - ow, W):
                uu = u[b, y, xx]
                if np.isfinite(uu) and 0 <= uu < ow and g.random() < 0.7:
                    rev[b, y, W - 1 - int(uu)] = fwd[b, y, xx] + np.float32(g.choice([0, 0.5, 1, 1.5, 3, 4]))
    for v in (np.nan, np.inf):
        rev[g.random((B, H, W)) < 0.01] = v
    return fwd, rev


@pytest.mark.parametrize("tol", [0.0, 1.0, 3.0])
@pytest.mark.parametrize("B, H, W, oh, ow", [(1, 27, 54, 27, 54), (2, 27, 81, 20, 70), (3, 54, 108, 49, 101)])
def test_lr_check_equals_oracle(tol, B, H, W, oh, ow):
    fwd, rev = _maps(B, H, W, ow, B * 100 + H + W)
    pred = torch.from_numpy(np.concatenate([fwd, rev])).to(DEV)
    f, u16, valid = ops.lr_check(pred, oh, ow, tol, float_out=True, u16_out=True, valid_out=True)
    wf, wu, wv = oracle_lr_check(fwd, rev, oh, ow, tol)
    assert valid.dtype == torch.bool and u16.dtype == torch.uint16 and f.shape == (B, oh, ow)
    assert np.array_equal(valid.cpu().numpy(), wv)
    assert np.array_equal(f.cpu().numpy().view(np.int32), wf.view(np.int32))                 # bits, including -0.0
    assert np.array_equal(u16.cpu().numpy(), wu)
    assert wv.any() and not wv.all()
    (only_u16,) = ops.lr_check(pred, oh, ow, tol, float_out=False, u16_out=True)
    (only_valid,) = ops.lr_check(pred, oh, ow, tol, float_out=False, valid_out=True)
    assert torch.equal(only_u16, u16) and torch.equal(only_valid, valid)


def test_lr_check_arguments():
    pred = torch.zeros((4, 27, 27), device=DEV)
    with pytest.raises(ValueError, match="2B"):
        ops.lr_check(pred[:3].contiguous(), 27, 27, 1.0)
    with pytest.raises(ValueError, match="crop"):
        ops.lr_check(pred, 28, 27, 1.0)
    with pytest.raises(ValueError, match="at least one"):
        ops.lr_check(pred, 27, 27, 1.0, float_out=False)
    with pytest.raises(ValueError, match="tolerance"):
        ops.lr_check(pred, 27, 27, float("nan"))
    with pytest.raises(ValueError, match="contiguous"):
        ops.lr_check(pred.transpose(1, 2), 27, 27, 1.0)
    with pytest.raises(ValueError, match="uint8"):
        ops.mirror_swap_u8(*[torch.zeros((1, 2, 2, 3), device=DEV)] * 4)
    u8 = torch.zeros((1, 2, 2, 3), dtype=torch.uint8, device=DEV)
    with pytest.raises(ValueError, match="does not match"):
        ops.mirror_swap_u8(u8, u8, u8, torch.zeros((1, 2, 3, 3), dtype=torch.uint8, device=DEV))


_MATCHERS = {}


def _matcher(masks="learned", skip=4, lr=None):
    if (masks, skip, lr) not in _MATCHERS:
        _MATCHERS[(masks, skip, lr)] = StereoMatcher(masks=masks, skip_stage_id=skip, lr_check=lr)
    return _MATCHERS[(masks, skip, lr)]


@pytest.mark.parametrize("masks", ["learned", "image"])
@pytest.mark.parametrize("skip", [4, 3])
def test_matcher_equals_definition(masks, skip):
    m, m_lr = _matcher(masks, skip), _matcher(masks, skip, 1.0)
    B, h, w = 2, 130, 260
    l, r = _images(B, h, w, 11)
    fwd = m(l, r)
    rev_raw = m(_flip(r).contiguous(), _flip(l).contiguous())              # the reverse run, not yet mirrored back
    disp, valid = m_lr(l, r, return_valid=True)
    # batch invariance: both halves of the 2B graph equal the B-sized runs of the plain matcher
    (st,) = m_lr._graphs[(B, h, w, 216, masks, "fp32", "lr")]
    H, W = st.pred.shape[-2:]
    assert torch.equal(st.pred[:B, H - h:, W - w:], fwd)
    assert torch.equal(st.pred[B:, H - h:, W - w:], rev_raw)
    wf, wu, wv = oracle_lr_check(fwd.cpu().numpy(), rev_raw.cpu().numpy(), h, w, 1.0)
    assert np.array_equal(valid.cpu().numpy(), wv)
    assert torch.equal(disp, torch.where(valid, fwd, torch.zeros_like(fwd)))
    u16 = m_lr(l, r, output="u16")
    plain_u16 = ops.disp_to_u16(fwd.contiguous(), h, w).cpu().numpy()     # (uint16 tensors have few ATen ops: compare in numpy)
    assert np.array_equal(u16.cpu().numpy(), np.where(wv, plain_u16, np.uint16(0)))
    assert np.array_equal(u16.cpu().numpy(), wu)


def test_tolerance_change_does_not_recapture():
    m = StereoMatcher(lr_check=0.5)
    l, r = _images(1, 60, 90, 3)
    d0, v0 = m(l, r, return_valid=True)
    assert m.captures == 1
    d1, v1 = m(l, r, lr_check=3.0, return_valid=True)
    d2, v2 = m(l, r, lr_check=0, return_valid=True)
    assert m.captures == 1
    assert bool((v1 >= v0).all()) and bool((v0 >= v2).all())              # a wider tolerance keeps every pixel it kept
    assert torch.equal(d1, torch.where(v1, d1, torch.zeros_like(d1))) and torch.equal(d1[v0], d0[v0])
    again = m(l, r, lr_check=None)                                         # None: the matcher's own tolerance
    assert torch.equal(again, d0)


def test_plain_and_lr_graphs_side_by_side():
    m = StereoMatcher()
    l, r = _images(1, 60, 90, 4)
    plain = m(l, r)
    assert m.captures == 1
    disp, valid = m(l, r, lr_check=1.0, return_valid=True)
    assert m.captures == 2 and len(m._graphs) == 2
    assert set(m._graphs) == {(1, 60, 90, 216, "learned", "fp32"), (1, 60, 90, 216, "learned", "fp32", "lr")}
    assert torch.equal(m(l, r), plain) and torch.equal(m(l, r, lr_check=1.0), disp) and m.captures == 2
    assert torch.equal(disp, torch.where(valid, plain, torch.zeros_like(plain)))


def _reference_layout(fe_sd, hot_sd, prefix="module."):
    sd = {f"{prefix}feature_extractor.{k}": v for k, v in fe_sd.items()}
    sd.update({prefix + k: v for k, v in hot_sd.items()})
    return sd


def test_weight_changes_recapture_the_lr_graph():
    from decnet_b200.params import make_featext_state, make_hotpath_state
    m = StereoMatcher(lr_check=1.0)
    l, r = _images(1, 60, 90, 5)
    before = m(l, r)
    other = _reference_layout(make_featext_state(5), make_hotpath_state(5))
    m.load_state_dict(other)
    after = m(l, r)
    assert not torch.equal(after, before)
    assert torch.equal(after, StereoMatcher(other, lr_check=1.0)(l, r))
    with torch.no_grad():
        m.model.refinement[2].conv[0].conv.weight.mul_(1.5)
    edited = m(l, r)
    assert not torch.equal(edited, after)
    assert torch.equal(edited, StereoMatcher(_reference_layout(m.fe.state_dict(), m.model.state_dict()), lr_check=1.0)(l, r))


def test_host_kinds_and_stream():
    m = _matcher(lr=1.0)
    l, r = _images(2, 60, 90, 7)
    want_d, want_v = m(l, r, return_valid=True)
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
    cuda_items = [tuple(torch.from_numpy(t).to(DEV) for t in it) for it in items]
    for a, b in zip(m.stream(cuda_items, lr_check=2.0), [m(x, y, lr_check=2.0) for x, y in cuda_items]):
        assert a.is_cuda and torch.equal(a, b)


def test_no_aten_flip_or_index_in_the_step():
    m = _matcher(lr=1.0)
    l, r = _images(1, 60, 90, 8)
    m(l, r)
    (st,) = m._graphs[(1, 60, 90, 216, "learned", "fp32", "lr")]
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof, torch.no_grad():
        m(l, r, output="u16")                                              # graph replay + lr_check
        m._step(st)                                                        # what the graph holds, launched eagerly
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert any("mirror_swap_u8_kernel" in n for n in names)
    assert any("lr_check_kernel" in n for n in names)
    bad = [n for n in names if "at::native" in n and any(k in n.lower() for k in ("flip", "index", "gather"))]
    assert not bad, bad
