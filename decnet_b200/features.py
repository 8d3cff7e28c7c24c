"""SURVEY.md section 8f rank 2: the step BEFORE the hot path -- `FeatExtNetChannelPlus`
(modules/submodule.py:245-343), the U-shaped extractor that turns an image into the
{stage0..stage3} feature pyramid the decomposed-matching path consumes.

Same class name, constructor arguments, sub-module names and state_dict keys as the reference
(`feature_extractor.conv0.0.conv.weight`, `...deconv2.deconv.bn.running_var`, ...), inference
only (BN folded).  The layers are the units of model.py, so each one runs on the kernel that
fits it:
  * 3x3 stride-1 convs up to 24 channels (full and 1/3 resolution: where the pixels are):
    `conv2d_tcgen05_kernel` (TF32 tensor cores, NCHW); the `cat(x_up, x_pre)` in front of each
    Deconv2dBlock conv is read as two sources, never materialised;
  * ConvTranspose 3x3 stride 3 to 8 / 24 channels: `deconv3x3s3_kernel`;
  * 1x1 convs at full and 1/3 resolution: `conv2d_small_kernel` / the centre tap of `conv2d_tcgen05_kernel`;
  * the first stride-3 conv (8 -> 24 at full resolution): `conv3x3s3_nchw_kernel` (direct fp32);
  * everything at 1/9 and 1/27 resolution (6 480 and 720 pixels per SceneFlow image, about 7 GFLOP per image: the other two
    stride-3 convs, the 72 / 216-channel 3x3 layers, the ASPP with its dilated convs, the 1x1 fusions, the 216 -> 72
    transposed conv) runs channels-last on `conv2d_nhwc_halo_kernel`: 3x3 stride-1 layers of the 1/9 level in its conv mode
    on zero-bordered tensors, all the rest in its GEMM mode -- behind `im2col3x3` for strided / dilated / 1/27-level 3x3
    windows, with concatenations written as channel slices of one buffer and the transposed conv as a GEMM + pixel shuffle.
  No layer runs on a library: the units have no library branch (a layer no kernel covers raises DecnetError).
The module refuses CPU tensors like the rest of the package; `oracle/features.py` is the CPU
restatement used by the tests.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .model import Conv2dUnit, Deconv2dUnit, _Cached, _split, set_precision


class Deconv2dBlock(nn.Module):
    """Drop-in for modules/submodule.py:162-177: deconv(x) -> cat(x_up, x_pre) -> 2 convs."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1):
        super().__init__()
        self.deconv = Deconv2dUnit(in_channels, out_channels, kernel_size, stride, bn=True)
        self.conv = nn.Sequential(Conv2dUnit(out_channels * 2, out_channels, 3, 1, padding=1),
                                  Conv2dUnit(out_channels, out_channels, 3, 1, padding=1))

    def forward(self, x_pre, x):
        x_up = self.deconv(x)
        y = self.conv[0].forward_cat([x_up, x_pre])
        return self.conv[1](y), x_up


class ASPP(nn.Module):
    """Drop-in for modules/submodule.py:222-241 (no image-pool branch in the shipped version)."""

    def __init__(self, in_ch, out_ch, rates):
        super().__init__()
        self.stages = nn.Module()
        self.stages.add_module("c0", Conv2dUnit(in_ch, out_ch, 1, stride=1, padding=0, dilation=1))
        for i, rate in enumerate(rates):
            self.stages.add_module(f"c{i + 1}", Conv2dUnit(in_ch, out_ch, 3, stride=1, padding=rate, dilation=rate))

    def forward(self, x):
        return torch.cat([stage(x) for stage in self.stages.children()], dim=1)


def _w2d(unit):
    """Folded 3x3 / 1x1 conv weights as GEMM rows [Cout, taps*Cin] with column tap*Cin + c (im2col3x3's order)."""
    w, b = unit.folded()
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous(), b


class FeatExtNetChannelPlus(_Cached, nn.Module):
    """Drop-in for modules/submodule.py:245-343 with num_stage = 4, down_scale = 3 (the shipped config)."""

    precision = "fp32"

    def __init__(self, base_channels, num_stage=4, down_scale=3, precision="fp32"):
        super().__init__()
        assert num_stage == 4 and down_scale == 3, "the shipped configuration (demo.sh:1) is 4 stages, x3"
        c, s = base_channels, down_scale
        self.base_channels, self.num_stage, self.down_scale = c, num_stage, s
        self.conv0 = nn.Sequential(Conv2dUnit(3, c, 3, 1, padding=1), Conv2dUnit(c, c, 3, 1, padding=1))
        self.addition_trans0 = Conv2dUnit(c, c, 1, stride=1, padding=0)
        self.conv1 = nn.Sequential(Conv2dUnit(c, c * s, 3, stride=s, padding=1),
                                   Conv2dUnit(c * s, c * s, 3, 1, padding=1), Conv2dUnit(c * s, c * s, 3, 1, padding=1))
        self.addition_trans1 = Conv2dUnit(c * s, c * s, 1, stride=1, padding=0)
        self.deconv1 = Deconv2dBlock(c * s, c, kernel_size=3, stride=3)
        self.conv2 = nn.Sequential(Conv2dUnit(c * s, c * s ** 2, 3, stride=3, padding=1),
                                   Conv2dUnit(c * s ** 2, c * s ** 2, 3, 1, padding=1),
                                   Conv2dUnit(c * s ** 2, c * s ** 2, 3, 1, padding=1))
        self.addition_trans2 = Conv2dUnit(c * s ** 2, c * s ** 2, 1, stride=1, padding=0)
        self.deconv2 = Deconv2dBlock(c * s ** 2, c * s, kernel_size=3, stride=3)
        self.conv3_1 = Conv2dUnit(c * s ** 2, c * s ** 3, 3, stride=3, padding=1)
        self.conv3_2 = nn.Sequential(Conv2dUnit(c * s ** 3, c * s ** 3, 3, 1, padding=1),
                                     Conv2dUnit(c * s ** 3, c * s ** 3, 3, 1, padding=1))
        self.addition_ctx_collection = nn.Sequential(ASPP(c * s ** 3, c * s ** 3, [4, 8, 12]),
                                                     Conv2dUnit(4 * c * s ** 3, c * s ** 3, 1, stride=1, padding=0))
        self.addition_fusion = Conv2dUnit(2 * c * s ** 3, c * s ** 3, 1, stride=1, padding=0)
        self.deconv3 = Deconv2dBlock(c * s ** 3, c * s ** 2, kernel_size=3, stride=3)
        self.out_channels = [c * s ** 3, c * s ** 2, c * s, c]
        set_precision(self, precision)
        self.precision = precision
        self.eval()

    # ------------------------------------------------------------------------------------------------------------
    # packed weights of the coarse half (1/9 and 1/27 resolution), in this module's precision
    # ------------------------------------------------------------------------------------------------------------
    NSLICE = 108                                                 # output channels per GEMM launch of the 216-channel layers

    def _coarse_pack(self):
        self._check_inference()
        split = _split(self)

        def gemm(unit, cp, slices=None):
            w2, b = _w2d(unit)
            n = w2.shape[0]
            sl = slices or [(0, n)]
            return [ops.pack_gemm_weights(w2, b, cp, split, a, e) + (a, unit.relu) for a, e in sl]

        def halo(unit, cp):
            w, b = unit.folded()
            return ops.pack_conv2d_tf32_weights(w, b, cp, split=split) + (unit.relu,)

        def build():
            c1, c2, c3 = self.out_channels[2], self.out_channels[1], self.out_channels[0]        # 24, 72, 216
            ns = self.NSLICE
            sl3 = [(a, min(a + ns, c3)) for a in range(0, c3, ns)]
            ld3 = (c3 + 15) // 16 * 16 + 8 if c3 % ns else c3 + 8                               # 224: rows of the 1/27-level tensors
            ld3 = (c3 + 15) // 16 * 16
            P = {"ld3": ld3, "c": (c1, c2, c3)}
            k2 = (9 * c1 + 7) // 8 * 8
            np2 = (c2 + 15) // 16 * 16                                                          # 80
            P["conv2_0"] = gemm(self.conv2[0], k2)
            P["conv2_1"], P["conv2_2"] = halo(self.conv2[1], np2), halo(self.conv2[2], np2)
            P["trans2"] = gemm(self.addition_trans2, np2)
            k3 = (9 * c2 + 7) // 8 * 8
            P["conv3_1"] = gemm(self.conv3_1, k3, sl3)
            k33 = 9 * ld3                                                                       # im2col of a 224-wide tensor
            for name, unit in (("conv3_2_0", self.conv3_2[0]), ("conv3_2_1", self.conv3_2[1]),
                               ("aspp1", self.addition_ctx_collection[0].stages.c1), ("aspp2", self.addition_ctx_collection[0].stages.c2),
                               ("aspp3", self.addition_ctx_collection[0].stages.c3)):
                # the im2col rows hold ld3 columns per tap (the c3 real channels + zero padding): spread the weights likewise
                w, b = unit.folded()
                w2 = torch.zeros((w.shape[0], 9, ld3), dtype=torch.float32, device=w.device)
                w2[:, :, :c3] = w.permute(0, 2, 3, 1).reshape(w.shape[0], 9, c3)
                w2 = w2.reshape(w.shape[0], k33)
                P[name] = [ops.pack_gemm_weights(w2, b, k33, split, a, e) + (a, unit.relu) for a, e in sl3]
            P["aspp0"] = gemm(self.addition_ctx_collection[0].stages.c0, ld3, sl3)

            def wide_1x1(unit, blocks, ld_in):
                # input = `blocks` tensors of c3 channels each, stored at column offsets j*c3 of rows of ld_in floats
                w2, b = _w2d(unit)
                wz = torch.zeros((w2.shape[0], ld_in), dtype=torch.float32, device=w2.device)
                wz[:, :blocks * c3] = w2
                return [ops.pack_gemm_weights(wz, b, ld_in, split, a, e) + (a, unit.relu) for a, e in sl3]
            P["ld_ctx"] = (4 * c3 + 15) // 16 * 16 + 8                                           # 872... rows of the ASPP concat
            P["ld_cat"] = (2 * c3 + 15) // 16 * 16 + 8
            P["ctx_1x1"] = wide_1x1(self.addition_ctx_collection[1], 4, P["ld_ctx"])
            P["fusion"] = wide_1x1(self.addition_fusion, 2, P["ld_cat"])
            # ConvTranspose2d(c3 -> c2, k 3, s 3) + BN + ReLU as a GEMM to 9*c2 columns (tap-major) + pixel shuffle
            w, b = self.deconv3.deconv.folded()                                                 # [c3, c2, 3, 3], [c2]
            wd = w.permute(2, 3, 1, 0).reshape(9 * c2, c3).contiguous()                          # row (ky*3+kx)*c2 + co
            bd = b.repeat(9)
            sld = [(a, min(a + ns, 9 * c2)) for a in range(0, 9 * c2, ns)]
            P["deconv3"] = [ops.pack_gemm_weights(wd, bd, ld3, split, a, e) + (a, True) for a, e in sld]
            P["ld_up"] = 9 * c2 + 16
            ldc = (2 * c2 + 7) // 8 * 8 + 8                                                      # 152: cat(x_up, x_pre) + slice padding
            P["ld_dcat"] = ldc
            P["dconv0"] = halo_cat = None
            w, b = self.deconv3.conv[0].folded()                                                # [c2, 2*c2, 3, 3] on cat(x_up, x_pre)
            P["dconv0"] = ops.pack_conv2d_tf32_weights(w, b, ldc, split=split) + (True,)
            P["dconv1"] = halo(self.deconv3.conv[1], np2)
            w, b = self.conv1[0].folded()                                                       # first stride-3 conv: direct kernel
            P["conv1_0"] = (w.float().permute(1, 2, 3, 0).reshape(w.shape[1], 9, w.shape[0]).contiguous(), b.float().contiguous())
            return P
        return self._cached(("coarse", split), build)

    def _gemm(self, x, packs, out, split, col0=0, **kw):
        if not split:
            x = ops.rna_tf32(x)          # plain-TF32 mode: operands rounded to nearest (the MMA itself would truncate)
        for wp, bp, np_, a, relu in packs:
            ops.gemm_tc(x, wp, bp, out, relu, split=split, col=col0 + a, **kw)
        return out

    @staticmethod
    def _halo(x, pack, split):
        wp, bp, _, relu = pack
        return ops.conv2d_tf32_nhwc_halo(x if split else ops.rna_tf32(x), wp, bp, relu, split=split)

    @torch.no_grad()
    def forward(self, x):
        if not x.is_cuda:
            raise RuntimeError("decnet_b200 has no CPU path: FeatExtNetChannelPlus needs a CUDA tensor "
                               "(oracle/features.py is the CPU restatement for tests)")
        x = x.contiguous().float()
        B, _, H, W = x.shape
        if H % 27 or W % 27:
            raise ValueError(f"pad the image to multiples of 27 first (demo.py:75-81), got {H}x{W}")
        split = _split(self)
        pk = self._coarse_pack()
        c1, c2, c3 = pk["c"]
        ld3 = pk["ld3"]
        z = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=x.device)
        # ---- full and 1/3 resolution: NCHW, thin tensor-core kernel
        conv0 = self.conv0(x)                                   # [B,  c, H,    W   ]
        t = torch.empty((B, c1, H // 3, W // 3), dtype=torch.float32, device=x.device)
        ops._call("decnet_conv3x3s3_nchw", conv0, conv0.data_ptr(), pk["conv1_0"][0].data_ptr(), pk["conv1_0"][1].data_ptr(),
                  t.data_ptr(), B, conv0.shape[1], H, W, c1, 1)
        conv1 = self.conv1[2](self.conv1[1](t))                 # [B, 3c, H/3,  W/3 ]
        # ---- 1/9 resolution: zero-bordered channels-last [B, h2+2, w2+2, 80]
        h2, w2, h3, w3 = H // 9, W // 9, H // 27, W // 27
        np2 = pk["conv2_1"][2]
        a, _, _ = ops.im2col3x3(conv1, "nchw", c1, stride=3)
        t2 = self._gemm(a, pk["conv2_0"], z(B, h2 + 2, w2 + 2, np2), split, dst_hw=(h2, w2))
        for key in ("conv2_1", "conv2_2"):
            t2 = self._halo(t2, pk[key], split)
        conv2 = t2                                              # [B, h2+2, w2+2, 80] (72 channels + zero padding)
        # ---- 1/27 resolution: flat channels-last rows of ld3 = 224 floats (216 channels + zero padding)
        a, _, _ = ops.im2col3x3(conv2, "nhwc_pad", c2, stride=3)
        x31 = self._gemm(a, pk["conv3_1"], z(B, h3, w3, ld3), split)
        cat2 = z(B, h3, w3, pk["ld_cat"])                       # cat(conv3_2, ctx)
        a, _, _ = ops.im2col3x3(x31, "nhwc", ld3, kp=9 * ld3)
        y = self._gemm(a, pk["conv3_2_0"], z(B, h3, w3, ld3), split)
        a, _, _ = ops.im2col3x3(y, "nhwc", ld3, kp=9 * ld3)
        self._gemm(a, pk["conv3_2_1"], cat2, split)
        ctx = z(B, h3, w3, pk["ld_ctx"])                        # ASPP: cat(1x1, d4, d8, d12)
        self._gemm(x31, pk["aspp0"], ctx, split)
        for j, (key, rate) in enumerate((("aspp1", 4), ("aspp2", 8), ("aspp3", 12))):
            a, _, _ = ops.im2col3x3(x31, "nhwc", ld3, dilation=rate, kp=9 * ld3)
            self._gemm(a, pk[key], ctx, split, col0=(j + 1) * c3)
        self._gemm(ctx, pk["ctx_1x1"], cat2, split, col0=c3)
        conv3 = self._gemm(cat2, pk["fusion"], z(B, h3, w3, ld3), split)
        out = {"stage0": ops.nhwc_to_nchw(conv3, B, c3, h3, w3)}
        # ---- deconv3 block back at 1/9: GEMM-form transposed conv + shuffle into cat(x_up, x_pre), then two 3x3 convs
        up = self._gemm(conv3, pk["deconv3"], z(B * h3 * w3, pk["ld_up"]), split)
        dcat = z(B, h2 + 2, w2 + 2, pk["ld_dcat"])
        ops.deconv3x3s3_shuffle(up, dcat, B, h3, w3, c2, col=0)
        self._gemm(conv2, pk["trans2"], dcat, split, col0=c2, border=(B, h2, w2))
        r = self._halo(self._halo(dcat, pk["dconv0"], split), pk["dconv1"], split)
        res = ops.nhwc_to_nchw(r, B, c2, h2, w2, pad=True)
        out["stage1"] = res
        # ---- 1/3 and full resolution: NCHW again
        res, _ = self.deconv2(self.addition_trans1(conv1), res)
        out["stage2"] = res
        res, _ = self.deconv1(self.addition_trans0(conv0), res)
        out["stage3"] = res
        return out


def extract_pair(fe, left, right, prepare=None, prepare_right=None):
    """Features of both views, the right view on a forked second stream (the two extractions are independent;
    demo.py:166-167 runs them back to back inside the model).  `prepare` is applied to each input first
    (e.g. the uint8 -> padded / normalised image kernel), `prepare_right`, when given, to the right one instead (e.g. the
    shifted prepare of a search range not starting at 0), on the forked stream too.  Returns (left_feats, right_feats),
    joined on the current stream; capturable in a CUDA graph (two branches)."""
    main = torch.cuda.current_stream(left.device)
    side = getattr(fe, "_side", None)
    if side is None or side.device != left.device:
        side = fe._side = torch.cuda.Stream(left.device)
    prepare_right = prepare_right or prepare
    side.wait_stream(main)                               # fork
    with torch.cuda.stream(side):
        fr = fe(prepare_right(right) if prepare_right is not None else right)
    fl = fe(prepare(left) if prepare is not None else left)
    # join; the right view's tensors live in the side stream's pool and are reused only behind the next fork
    main.wait_stream(side)
    return fl, fr
