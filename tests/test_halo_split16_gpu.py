"""split16 storage of the channels-last conv stacks: the writers (pack kernels, layout bridge, halo-conv epilogue) against a
Python restatement of the encoder bit for bit, and the split16-input halo conv (split = 3) against fp64."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def split16_ref(x, cp):
    """fp32 [..., cp] -> fp16 [..., 2*cp]: per 32-channel chunk of cl channels [fp16(2^11 * (x - h)) x cl | h x cl] with
    h = fp16(x), both rounded to nearest and saturating to +-65504 (common.cuh: split16_store)."""
    h = x.clamp(-65504.0, 65504.0).half()
    lo = ((x - h.float()) * 2048.0).clamp(-65504.0, 65504.0).half()
    out = torch.empty(x.shape[:-1] + (2 * cp,), dtype=torch.float16, device=x.device)
    for c0 in range(0, cp, 32):
        cl = min(32, cp - c0)
        out[..., 2 * c0:2 * c0 + cl] = lo[..., c0:c0 + cl]
        out[..., 2 * c0 + cl:2 * c0 + 2 * cl] = h[..., c0:c0 + cl]
    return out


def split16_decode(s, cp):
    """The value a split16 tensor stands for, h + 2^-11 * lo, as fp32 [..., cp]."""
    out = torch.empty(s.shape[:-1] + (cp,), dtype=torch.float32, device=s.device)
    for c0 in range(0, cp, 32):
        cl = min(32, cp - c0)
        out[..., c0:c0 + cl] = s[..., 2 * c0 + cl:2 * c0 + 2 * cl].float() + s[..., 2 * c0:2 * c0 + cl].float() / 2048.0
    return out


def _bits_equal(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a.view(torch.int16), b.view(torch.int16))


def _cp16(c):
    return (c + 15) // 16 * 16


@pytest.mark.parametrize("chans,cp", [((72, 72, 1), 160), ((145,), 160), ((40,), 48), ((390,), 400)])
def test_nchw_cat_to_nhwc_pad_split16_matches_the_encoder(chans, cp):
    """Tiled bridge (cp <= 383) and the element-per-thread one (cp = 400); border pixels and padding channels included."""
    from decnet_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    B, H, W = 2, 23, 45
    srcs = [torch.randn(B, c, H, W, device="cuda", generator=g) * 10 ** (i - 1) for i, c in enumerate(chans)]
    if chans[-1] == 1:
        srcs[-1] = srcs[-1][:, 0].contiguous() * 100.0          # single-channel source as [B,H,W]: a disparity map
    want = split16_ref(ops.nchw_cat_to_nhwc_pad(srcs, cp, round_tf32=False), cp)
    got = ops.nchw_cat_to_nhwc_pad(srcs, cp, split16=True)
    assert got.shape == (B, H + 2, W + 2, 2 * cp)
    assert _bits_equal(got, want)


@pytest.mark.parametrize("C,pad", [(8, True), (24, True), (72, True), (8, False)])
def test_dynup_pack_and_set_disp_split16_match_the_encoder(C, pad):
    from decnet_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(4)
    B, h, w = 2, 13, 37
    cp = _cp16(9 * C + 1)
    Lf = torch.randn(B, C, 3 * h, 3 * w, device="cuda", generator=g)
    disp = torch.rand(B, h, w, device="cuda", generator=g) * 200.0
    want = split16_ref(ops.dynup_pack_nhwc(disp, Lf, cp, round_tf32=False, pad=pad), cp)
    got = ops.dynup_pack_nhwc(disp, Lf, cp, pad=pad, split16=True)
    assert _bits_equal(got, want)
    # features ahead (disp = None, channel 0 zero), the disparity channel later
    pre = ops.dynup_pack_nhwc(None, Lf, cp, pad=pad, split16=True)
    assert _bits_equal(pre, split16_ref(ops.dynup_pack_nhwc(None, Lf, cp, round_tf32=False, pad=pad), cp))
    assert _bits_equal(ops.dynup_set_disp_nhwc(pre, disp, pad=pad), want)


def _layer(B, H, W, Cin, Cout, xs=1.0, ws=1.0, seed=22):
    from decnet_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, Cin, H, W, device="cuda", generator=g) * xs
    w = torch.randn(Cout, Cin, 3, 3, device="cuda", generator=g) * (2.0 / (9 * Cin)) ** 0.5 * ws
    b = torch.randn(Cout, device="cuda", generator=g) * 0.1 * xs * ws
    cp = _cp16(Cin)
    wp, bp, np_ = ops.pack_conv2d_tf32_weights(w, b, cp, split=True, split16_in=True)
    assert wp.shape == (9, np_, cp) and bp.numel() == np_ + 4
    return x, w, b, ops.nchw_cat_to_nhwc_pad([x], cp, split16=True), wp, bp, np_


@pytest.mark.parametrize("B,H,W,Cin,Cout", [(2, 180, 324, 73, 81), (2, 180, 324, 81, 81), (1, 60, 108, 145, 72),
                                            (1, 21, 47, 72, 36)])
@pytest.mark.parametrize("relu", [True, False])
def test_split16_input_conv_is_fp32_class(B, H, W, Cin, Cout, relu):
    from decnet_b200 import ops
    x, w, b, xs16, wp, bp, np_ = _layer(B, H, W, Cin, Cout)
    want = F.conv2d(x.double(), w.double(), b.double(), padding=1)
    want = (F.relu(want) if relu else want).float()
    got = ops.conv2d_tf32_nhwc_halo(xs16, wp, bp, relu, split=True)
    assert got.dtype == torch.float32 and got.shape == (B, H + 2, W + 2, np_)
    assert float(got[:, 0].abs().max()) == 0 and float(got[:, -1].abs().max()) == 0
    assert float(got[:, :, 0].abs().max()) == 0 and float(got[:, :, -1].abs().max()) == 0
    err = (got[:, 1:-1, 1:-1, :Cout].permute(0, 3, 1, 2) - want).abs().max().item()
    assert err <= 1e-5 * want.abs().max().item(), (err, want.abs().max().item())
    if np_ > Cout:
        assert got[..., Cout:].abs().max().item() == 0


@pytest.mark.parametrize("xs,ws", [(1.0, 1.0), (300.0, 1e-3), (1e-3, 30.0), (3e3, 1e-4)])
def test_split16_input_conv_across_operand_ranges(xs, ws):
    from decnet_b200 import ops
    x, w, b, xs16, wp, bp, np_ = _layer(2, 40, 52, 81, 81, xs, ws, seed=91)
    want = F.conv2d(x.double(), w.double(), b.double(), padding=1).float()
    got = ops.conv2d_tf32_nhwc_halo(xs16, wp, bp, False, split=True)
    err = (got[:, 1:-1, 1:-1, :81].permute(0, 3, 1, 2) - want).abs().max().item()
    assert err <= 1e-5 * want.abs().max().item(), (xs, ws, err, want.abs().max().item())


@pytest.mark.parametrize("B,H,W,Cin,Cout,relu", [(2, 60, 108, 81, 81, True), (1, 60, 108, 72, 72, False), (1, 33, 29, 145, 72, True)])
def test_split16_output_is_the_encoder_of_the_fp32_output(B, H, W, Cin, Cout, relu):
    """The epilogue's split16 store (np = 96: whole chunks; np = 80: a 16-channel last chunk) against the encoder applied to
    the same layer's fp32 output; the value it stands for is that output to 2^-22."""
    from decnet_b200 import ops
    _, _, _, xs16, wp, bp, np_ = _layer(B, H, W, Cin, Cout)
    f32 = ops.conv2d_tf32_nhwc_halo(xs16, wp, bp, relu, split=True)
    s16 = ops.conv2d_tf32_nhwc_halo(xs16, wp, bp, relu, split=True, split16_out=True)
    assert s16.dtype == torch.float16 and s16.shape == (B, H + 2, W + 2, 2 * np_)
    assert _bits_equal(s16, split16_ref(f32, np_))
    scale = float(f32.abs().max())
    assert float((split16_decode(s16, np_) - f32).abs().max()) <= 2 ** -21 * scale


def test_split16_beyond_the_fp16_range_stays_finite():
    """|x| > 65504: both halves saturate (the stored value is wrong, but finite), and so is everything computed from it."""
    from decnet_b200 import ops
    x, w, b, _, wp, bp, np_ = _layer(1, 20, 30, 81, 81)
    big = x * 1e6
    cp = _cp16(81)
    s = ops.nchw_cat_to_nhwc_pad([big], cp, split16=True)
    assert bool(torch.isfinite(s.float()).all())
    assert _bits_equal(s, split16_ref(ops.nchw_cat_to_nhwc_pad([big], cp, round_tf32=False), cp))
    out = ops.conv2d_tf32_nhwc_halo(s, wp, bp, True, split=True, split16_out=True)
    assert bool(torch.isfinite(out.float()).all())
    assert bool(torch.isfinite(ops.conv2d_tf32_nhwc_halo(out, wp, bp, False, split=True)).all())


def test_split16_argument_errors():
    from decnet_b200 import _lib, ops
    x, w, b, xs16, wp, bp, np_ = _layer(1, 8, 9, 40, 16)
    with pytest.raises(ValueError):
        ops.conv2d_tf32_nhwc_halo(xs16, wp, bp, True)                             # split16 input needs the split modes
    wp18, bp18, _ = ops.pack_conv2d_tf32_weights(w, b, 48, split=True)
    with pytest.raises(ValueError):
        ops.conv2d_tf32_nhwc_halo(xs16, wp18, bp18, True, split=True)             # the 18-tap pack reads fp32 input
    with pytest.raises(_lib.DecnetError):
        ops.nchw_cat_to_nhwc_pad([x], 40, split16=True)                           # cp % 16 != 0
