"""GPU: the skip-stage bicubic kernel against ATen's, and StereoMatcher (images -> disparity through one CUDA graph per
shape) against the eager composition it replaces: image_prepare_u8 -> feature extractor -> DecompMatching -> crop."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from decnet_b200 import StereoMatcher, ops
from decnet_b200.model import DecompMatching

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)


def _values(shape, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(shape, device=DEV, generator=g) * 1e3
    x.view(-1)[::7] = 0.0
    x.view(-1)[1::11] = -x.view(-1)[1::11].abs()
    return x


def _aten(x, H, W):
    return F.interpolate((x * 3).unsqueeze(1), (H, W), mode="bicubic").squeeze(1)


@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 3, 4), (3, 7, 5), (2, 20, 36), (1, 225, 324)])
def test_bicubic_x3_equals_aten(shape):
    x = _values(shape, sum(shape))
    H, W = 3 * shape[1], 3 * shape[2]
    assert torch.equal(ops.bicubic_skip(x, H, W), _aten(x, H, W))


@pytest.mark.parametrize("src, dst", [((2, 7, 5), (10, 13)), ((1, 20, 36), (9, 11)), ((2, 4, 6), (4, 6))])
def test_bicubic_any_size_equals_aten(src, dst):
    x = _values(src, 5)
    assert torch.equal(ops.bicubic_skip(x, *dst), _aten(x, *dst))


def test_bicubic_band_slice_equals_aten():
    """bands.py: a row band (with halo) of the 1/3 map, up-sampled to 3x its own rows and the full width."""
    full = _values((2, 75, 108), 9)
    band = full[:, 17:42]
    assert torch.equal(ops.bicubic_skip(band.contiguous(), 75, 324), _aten(band, 75, 324))


def _features(B, H, W, seed=17):
    from decnet_b200.params import make_features
    return make_features(B, H, W, seed=seed, device=DEV)


def test_no_aten_bicubic_left():
    from decnet_b200.params import make_hotpath_state
    model = DecompMatching(max_disp=216, skip_stage_id=3)
    model.load_state_dict(make_hotpath_state(17))
    model = model.to(DEV)
    left, right = _features(1, 108, 162)
    model(left, right)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        model(left, right)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert any("bicubic_up3_kernel" in n for n in names)
    assert not any("upsample_bicubic" in n for n in names), [n for n in names if "bicubic" in n]


def _images(B, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8),
            torch.randint(0, 256, (B, h, w, 3), device=DEV, generator=g, dtype=torch.uint8))


def _eager(m, l, r, model=None):
    """The composition StereoMatcher replaces, launched op by op: padded prediction cropped to the input size."""
    model = model or m.model
    l01, lnorm = ops.image_prepare_u8(l)
    r01, rnorm = ops.image_prepare_u8(r)
    fl, fr = m.fe(lnorm), m.fe(rnorm)
    if m.masks == "learned":
        pred = model(fl, fr)[0]
    else:
        lm = ops.detail_detection(l01, 3, m.detail_thold)[::-1]
        rm = ops.detail_detection(r01, 3, m.detail_thold)[::-1]
        pred = model(fl, fr, lm, rm)[0]
    h, w = l.shape[1:3]
    return pred[:, pred.shape[1] - h:, pred.shape[2] - w:]


_MATCHERS = {}


def _matcher(masks="learned", skip=4):
    if (masks, skip) not in _MATCHERS:
        _MATCHERS[(masks, skip)] = StereoMatcher(masks=masks, skip_stage_id=skip)
    return _MATCHERS[(masks, skip)]


@pytest.mark.parametrize("masks", ["learned", "image"])
@pytest.mark.parametrize("skip", [4, 3])
def test_matcher_equals_eager_composition(masks, skip):
    m = _matcher(masks, skip)
    l, r = _images(2, 130, 260, 1)
    want = _eager(m, l, r)
    got = m(l, r)
    assert got.shape == (2, 130, 260) and got.dtype == torch.float32
    assert torch.equal(got, want), float((got - want).abs().max())
    assert torch.equal(m(l, r), want)                                     # replay of the captured graph
    u16 = m(l, r, output="u16")
    assert u16.dtype == torch.uint16
    assert torch.equal(u16, ops.disp_to_u16(want.contiguous(), 130, 260))


def test_cache_capture_and_eviction():
    m = StereoMatcher(max_graphs=2)
    a, b, c = _images(1, 60, 90, 2), _images(1, 54, 81, 3), _images(1, 40, 70, 4)
    first = m(*a)
    assert m.captures == 1
    assert torch.equal(m(*a), first) and m.captures == 1                  # same shape: replay only
    m(*b)
    assert m.captures == 2 and len(m._graphs) == 2
    m(*a)                                                                 # a is now the most recently used
    m(*c)                                                                 # evicts b
    assert m.captures == 3 and len(m._graphs) == 2
    assert (1, 54, 81, 216, "learned", "fp32") not in m._graphs
    m(*b)                                                                 # evicts a; b re-captured
    assert m.captures == 4
    assert torch.equal(m(*a), first) and m.captures == 5                  # a re-captured: same result
    m.clear()
    assert len(m._graphs) == 0


def _reference_layout(fe_sd, hot_sd, prefix="module."):
    sd = {f"{prefix}feature_extractor.{k}": v for k, v in fe_sd.items()}
    sd.update({prefix + k: v for k, v in hot_sd.items()})
    return sd


def test_weight_changes_are_never_served_stale():
    from decnet_b200.params import make_featext_state, make_hotpath_state
    m = StereoMatcher()
    l, r = _images(1, 60, 90, 5)
    before = m(l, r)
    other = _reference_layout(make_featext_state(5), make_hotpath_state(5))
    m.load_state_dict(other)
    after = m(l, r)
    assert not torch.equal(after, before)
    assert torch.equal(after, StereoMatcher(other)(l, r))
    with torch.no_grad():
        m.model.refinement[2].conv[0].conv.weight.mul_(1.5)
    edited = m(l, r)
    fresh = StereoMatcher(_reference_layout(m.fe.state_dict(), m.model.state_dict()))
    assert not torch.equal(edited, after)
    assert torch.equal(edited, fresh(l, r))


def test_per_call_max_disp():
    m = _matcher()
    l, r = _images(1, 60, 90, 6)
    model = DecompMatching(max_disp=216)
    model.load_state_dict(m.model.state_dict())
    model = model.to(DEV)
    m2 = StereoMatcher(max_disp=100)                                      # 108 by default
    assert m2.max_disp == 108
    got = m2(l, r, max_disp=192)                                          # runs as 216
    assert (1, 60, 90, 216, "learned", "fp32") in m2._graphs
    assert torch.equal(got, _eager(m, l, r, model))


def test_input_and_output_kinds():
    m = _matcher()
    l, r = _images(1, 60, 90, 7)
    want = m(l[0], r[0])
    assert want.is_cuda and want.shape == (60, 90)
    got = m(l[0].cpu().numpy(), r[0].cpu().numpy())
    assert isinstance(got, np.ndarray) and got.dtype == np.float32
    assert np.array_equal(got, want.cpu().numpy())
    cpu = m(l.cpu(), r.cpu(), output="u16")
    assert isinstance(cpu, torch.Tensor) and not cpu.is_cuda and cpu.shape == (1, 60, 90)
    keep = want.clone()
    l2, r2 = _images(1, 60, 90, 8)
    m(l2[0], r2[0])
    assert torch.equal(want, keep)                                        # an earlier result is not the static buffer
    tiny = m(*(t[:, :5, :7] .contiguous() for t in (l, r)))               # the smallest sizes pad to one 27 x 27 image
    assert tiny.shape == (1, 5, 7) and torch.isfinite(tiny).all()
    sizes = [(60, 90), (54, 81), (60, 90), (40, 70)]
    pairs = [tuple(t[0].cpu().numpy() for t in _images(1, h, w, 20 + i)) for i, (h, w) in enumerate(sizes)]
    listed = m([p[0] for p in pairs], [p[1] for p in pairs])
    for (pl, pr), got in zip(pairs, listed):
        assert np.array_equal(got, m(pl, pr))


def test_stream_in_order():
    m = _matcher()
    sizes = [(60, 90), (60, 90), (54, 81), (54, 81), (60, 90)]
    items = [tuple(t.cpu().numpy() for t in _images(2, h, w, 30 + i)) for i, (h, w) in enumerate(sizes)]
    want = [m(l, r, output="u16") for l, r in items]
    got = list(m.stream(items, output="u16"))
    assert len(got) == 5
    for a, b in zip(got, want):
        assert isinstance(a, np.ndarray) and np.array_equal(a, b)
    cuda_items = [tuple(torch.from_numpy(t).to(DEV) for t in it) for it in items]
    for a, b in zip(m.stream(cuda_items), [m(l, r) for l, r in cuda_items]):
        assert a.is_cuda and torch.equal(a, b)


def test_reference_checkpoint_layout():
    from decnet_b200.params import make_featext_state, make_hotpath_state
    sd = _reference_layout(make_featext_state(3), make_hotpath_state(3))
    m = StereoMatcher(sd)
    l, r = _images(1, 60, 90, 9)
    assert torch.isfinite(m(l, r)).all()
    with pytest.raises(ValueError, match="unexpected"):
        m.load_state_dict(dict(sd, **{"module.soft_attention.0.conv.7.conv.weight": torch.zeros(1)}))
    missing = dict(sd)
    del missing["module.soft_attention.0.conv.0.conv.weight"]
    with pytest.raises(ValueError, match=r"missing.*soft_attention\.0\.conv\.0\.conv\.weight"):
        m.load_state_dict(missing)
