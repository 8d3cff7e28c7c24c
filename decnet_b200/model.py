"""Host-side mirror of the reference's hot-path modules, backed by libdecnet_b200.so.

Same class names, constructor arguments, forward signatures and state_dict keys as
modules/submodule.py (GetCostVolume :428, CostRegNetNoDown :608, disparity_regression :766,
GenerateSparseMask :347, DynamicUpsampling :566, SoftAttention :593, Refinement :666) so that a
reference checkpoint loads unchanged and the reference's stage loop can call them.  Every layer of
the hot path runs on a hand-written sm_100a kernel behind the C ABI (include/decnet_b200.h):
cost volume, 3-D aggregation (bf16 tcgen05 implicit GEMM), soft-argmin, the 2-D conv stacks of
a5 / a8 / a13 / a14 (tcgen05 implicit GEMMs on NCHW or zero-bordered channels-last fp32; the few
1..4-channel layers on a direct fp32 kernel), mask threshold, dynamic-upsampling pack + glue,
SpaMat / SpaVar, soft-attention pack, sigmoid + blend, disparity warp.  There is ONE route: no library
(cuDNN) branch, no global switch, no CPU path; a layer no kernel supports raises.

`precision` (per unit; `DecompMatching(precision=...)` sets it on every unit) is an arithmetic mode of
the SAME tensor-core kernels, not a backend:
  "fp32"  (default) error-compensated 3xTF32: operands split into TF32 hi + lo parts, three MMAs per tap
          into the fp32 accumulator -> fp32-class results (~2^-22 per product).  The parity gates against
          the reference's fp32 execution (<= 1e-3, masks bit-exact) run on this mode, and so does bench.py.
  "tf32"  plain TF32 operands, one MMA per tap: the precision class the reference itself gets from
          cuDNN on a GPU (torch.backends.cudnn.allow_tf32 defaults to True); faster, gated against
          cuDNN-TF32's own deviation from fp32.

Inference only (eval-mode BN folded into the weights; a unit in training mode raises).  CUDA tensors only.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops
from .modules import SpaMat, SpaVar

BN_EPS = 1e-5
PRECISIONS = ("fp32", "tf32")


def _sig_of(*mods):
    """Identity of everything a folded / packed weight cache was built from: (storage pointer, in-place version) of
    every parameter and buffer of the given modules.  load_state_dict (copy_ bumps the version), .to() / .cuda()
    (new storage) and in-place edits all change it, whichever parent module they were called on."""
    sig = []
    for m in mods:
        for t in list(m.parameters()) + list(m.buffers()):
            sig.append((t.data_ptr(), t._version))
    return tuple(sig)


class _Cached:
    """Weight caches keyed on _sig_of(self): rebuilt whenever a parameter or BN statistic changed."""

    def _cached(self, key, build):
        store = self.__dict__.setdefault("_wcache", {})
        sig = _sig_of(self)
        ent = store.get(key)
        if ent is None or ent[0] != sig:
            ent = (sig, build())
            store[key] = ent
        return ent[1]

    def _check_inference(self):
        if self.training:
            raise RuntimeError(f"{type(self).__name__}: decnet_b200 units are inference-only (eval-mode BatchNorm is folded "
                               "into the conv weights and no gradient reaches them); call .eval() first")


def _split(unit) -> int:
    """0 for the plain-TF32 mode, else the form of the fp32-class operand split (ops.SPLIT_KIND: 2 = TF32 hi*hi + fp16
    correction MMA, 1 = three TF32 MMAs).  The value is part of every packed-weight cache key, so packs made under one kind are
    never handed to the other."""
    if unit.precision not in PRECISIONS:
        raise ValueError(f"precision must be one of {PRECISIONS}, got {unit.precision!r}")
    return ops.SPLIT_KIND if unit.precision == "fp32" else 0


# --------------------------------------------------------------------------------------
# units with the reference's parameter names (conv.weight / conv.bias / bn.*)
# --------------------------------------------------------------------------------------
class Conv2dUnit(_Cached, nn.Module):
    """Conv2d [+ BN(eval)] [+ ReLU]; keys as modules/submodule.py:15-49."""

    precision = "fp32"

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, dilation=1, relu=True, bn=True,
                 padding=0):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size, stride=stride, dilation=dilation,
                              padding=padding, bias=not bn)
        self.bn = nn.BatchNorm2d(out_channels) if bn else None
        self.relu = relu

    def folded(self):
        self._check_inference()

        def build():
            w = self.conv.weight.detach()
            b = self.conv.bias.detach() if self.conv.bias is not None else torch.zeros(w.shape[0], device=w.device)
            if self.bn is not None:
                scale = self.bn.weight.detach() / torch.sqrt(self.bn.running_var + BN_EPS)
                w = w * scale.view(-1, 1, 1, 1)
                b = (b - self.bn.running_mean) * scale + self.bn.bias.detach()
            return (w.contiguous(), b.contiguous())
        return self._cached("folded", build)

    def _same_pad_3x3(self):
        c = self.conv
        d = c.dilation[0]
        return (c.kernel_size == (3, 3) and c.stride == (1, 1) and c.dilation == (d, d) and c.padding == (d, d)
                and c.groups == 1)

    def native(self):
        """Packed weights for the direct fp32 kernel when this layer is one of its shapes (else None)."""
        c = self.conv
        k, d = c.kernel_size[0], c.dilation[0]
        ok = (c.kernel_size[0] == c.kernel_size[1] and c.stride == (1, 1) and c.dilation[0] == c.dilation[1]
              and c.padding == (d * (k // 2), d * (k // 2)) and c.groups == 1
              and ops.conv2d_small_supported(c.in_channels, c.out_channels, k))
        if not ok:
            return None

        def build():
            w, b = self.folded()
            return (ops.pack_conv2d_weights(w), b.float().contiguous())
        return self._cached("native", build)

    def tensor_core(self, x):
        """Packed weights for the NCHW tcgen05 kernel when this layer / input is one of its shapes, else None.
        Thin layers (Cin < 8 with one output, or wide dilations on 4 channels) stay on the direct fp32
        kernel, which is faster there (scripts/exp_conv2d_tc.py)."""
        c = self.conv
        d = c.dilation[0]
        cin, cout = c.in_channels, c.out_channels
        split = _split(self)
        one = c.kernel_size == (1, 1) and c.stride == (1, 1) and c.padding == (0, 0) and c.groups == 1 and cin >= 8
        ok = ((one or (self._same_pad_3x3() and ((d <= 4 and (cin >= 8 or cout >= 3)) or (d <= 8 and cin >= 8))))
              and ops.conv2d_tf32_supported(cin, cout, x.shape[2], x.shape[3], 1 if one else d, split))
        if not ok:
            return None

        def build():
            w, b = self.folded()
            if one:                                  # a 1x1 conv is the centre tap of a 3x3 one
                w3 = torch.zeros((cout, cin, 3, 3), dtype=w.dtype, device=w.device)
                w3[:, :, 1, 1] = w[:, :, 0, 0]
                w = w3
            return ops.pack_conv2d_tf32_nchw_weights(w, b, split=split)
        return self._cached(("tc", split), build)

    def forward_cat(self, srcs, w_valid=None):
        """forward(torch.cat(srcs, 1)) with single-channel maps given as [B,H,W]; the concatenation is never
        materialised (the kernel reads each source through its own tensor map).
        w_valid: the tensors are right-padded to a 16-byte row pitch (see pad_pitch); columns >= w_valid of the
        result are zeros."""
        x0 = srcs[0]
        if w_valid is None and x0.shape[-1] % 4:
            # a width that is not a multiple of 4 (16-byte row pitch for TMA): run on right-padded copies and crop
            padded = [pad_pitch(t) for t in srcs]
            return unpad_pitch(self.forward_cat([t for t, _ in padded], w_valid=padded[0][1]), padded[0][1])
        chans = tuple(1 if t.dim() == 3 else t.shape[1] for t in srcs)
        c = self.conv
        d = c.dilation[0]
        split = _split(self)
        ok = (len(srcs) <= 3 and self._same_pad_3x3() and sum(chans) == c.in_channels
              and ops.conv2d_tf32_supported(ops.padded_cat_channels(chans), c.out_channels, x0.shape[-2], x0.shape[-1], d, split))
        if not ok:
            return self.forward(torch.cat([t.unsqueeze(1) if t.dim() == 3 else t for t in srcs], 1), w_valid=w_valid)
        wp, bp = self._cached(("tc_cat", split, chans),
                              lambda: ops.pack_conv2d_tf32_nchw_weights(*self.folded(), chans, split=split))
        return ops.conv2d_tf32_nchw_cat([t.contiguous() for t in srcs], wp, bp, c.out_channels, d, self.relu,
                                        w_valid or 0, split=split)

    def forward(self, x, addend=None, w_valid=None):
        if not (x.is_cuda and x.dtype == torch.float32):
            raise _lib.DecnetError("decnet_b200 units take float32 CUDA tensors (there is no CPU path)")
        c = self.conv
        if w_valid is None and addend is None and x.shape[-1] % 4 and self.native() is None:
            xp, wv = pad_pitch(x)                      # see forward_cat: pitch-padded copy, cropped result
            return unpad_pitch(self.forward(xp, w_valid=wv), wv)
        nat_first = c.kernel_size == (1, 1) and self.native() is not None      # tiny 1x1 layers: the direct kernel
        tc = self.tensor_core(x) if ((addend is None or c.out_channels == 1) and not nat_first) else None
        if tc is not None:
            return ops.conv2d_tf32_nchw_cat([x.contiguous()], tc[0], tc[1], c.out_channels, c.dilation[0], self.relu,
                                            w_valid or 0, split=_split(self),
                                            addend=None if addend is None else addend.contiguous())
        if w_valid:
            out = self.forward(x, addend)
            out[..., w_valid:] = 0                       # keep the pitch padding at zero behind a non-tensor-core layer
            return out
        nat = self.native()
        if nat is not None:
            return ops.conv2d_small(x.contiguous(), nat[0], nat[1], c.out_channels, c.kernel_size[0], c.dilation[0],
                                    self.relu, addend)
        raise _lib.DecnetError(f"Conv2dUnit {c.in_channels}->{c.out_channels} k{c.kernel_size} s{c.stride} d{c.dilation} on "
                               f"{tuple(x.shape)}: no decnet_b200 kernel covers this layer (and there is no library fallback)")


class Deconv2dUnit(_Cached, nn.Module):
    """ConvTranspose2d [+ BN(eval)] + ReLU; keys as modules/submodule.py:52-87 (bn=False: bias, as in
    GenerateSparseMask.deconv.0; bn=True: no bias, as in Deconv2dBlock.deconv of the feature extractor).
    Kernel 3, stride 3 (the only shape the model uses): deconv3x3s3_kernel, exact fp32."""

    precision = "fp32"

    def __init__(self, in_channels, out_channels, kernel_size, stride, bn=False):
        super().__init__()
        self.conv = nn.ConvTranspose2d(in_channels, out_channels, kernel_size, stride=stride, bias=not bn)
        self.bn = nn.BatchNorm2d(out_channels) if bn else None

    def folded(self):
        self._check_inference()

        def build():
            w = self.conv.weight.detach()                       # [Cin, Cout, k, k]
            b = self.conv.bias.detach() if self.conv.bias is not None else torch.zeros(w.shape[1], device=w.device)
            if self.bn is not None:
                scale = self.bn.weight.detach() / torch.sqrt(self.bn.running_var + BN_EPS)
                w = w * scale.view(1, -1, 1, 1)
                b = (b - self.bn.running_mean) * scale + self.bn.bias.detach()
            return (w.contiguous(), b.contiguous())
        return self._cached("folded", build)

    def forward(self, x):
        if not (x.is_cuda and x.dtype == torch.float32):
            raise _lib.DecnetError("decnet_b200 units take float32 CUDA tensors (there is no CPU path)")
        c = self.conv
        w, b = self.folded()
        if c.kernel_size == (3, 3) and c.stride == (3, 3) and c.padding == (0, 0) and ops.deconv3x3s3_supported(c.out_channels):
            return ops.deconv3x3s3(x.contiguous(), w, b, True)
        raise _lib.DecnetError(f"Deconv2dUnit {c.in_channels}->{c.out_channels} k{c.kernel_size} s{c.stride}: no decnet_b200 kernel "
                               f"covers this layer (and there is no library fallback)")


class Conv3dUnit(nn.Module):
    """Conv3d 3^3 pad 1 (no bias) + BN3d(eval) [+ ReLU]; keys as modules/submodule.py:90-123."""

    def __init__(self, in_channels, out_channels, relu=True):
        super().__init__()
        self.conv = nn.Conv3d(in_channels, out_channels, 3, padding=1, bias=False)
        self.bn = nn.BatchNorm3d(out_channels)
        self.relu = relu

    def scale_bias(self):
        scale = self.bn.weight.detach() / torch.sqrt(self.bn.running_var + BN_EPS)
        return scale, self.bn.bias.detach() - self.bn.running_mean * scale


def pad_pitch(t):
    """(tensor right-padded with zero columns to a width that is a multiple of 4, original width or None).
    The tensor-core Conv2d reads images through TMA, which needs 16-byte row strides: a KITTI-sized level
    (W = 1269, 423, 141) runs its conv stacks on such padded copies and crops the result (unpad_pitch)."""
    W = t.shape[-1]
    if W % 4 == 0:
        return t, None
    return F.pad(t, (0, 4 - W % 4)), W


def unpad_pitch(t, w_valid):
    return t if w_valid is None else t[..., :w_valid].contiguous()


# --------------------------------------------------------------------------------------
# a1/a2: cost volume
# --------------------------------------------------------------------------------------
class GetCostVolume(nn.Module):
    """Drop-in for modules/submodule.py:428-562, restricted to what the shipped model uses:
    warp_ope="homgrp", cost_func="cor", stage-0 candidates 0..D-1 (get_disp_samples :376-390).
    forward(left, right, disp_samples=[B,D,H,W] | max_disp=D) -> [B,C,D,H,W] fp32."""

    def __init__(self, warp_ope="homgrp", cost_func="cor"):
        super().__init__()
        if warp_ope != "homgrp" or cost_func != "cor":
            raise NotImplementedError("decnet_b200 implements the shipped configuration only: homgrp + cor")
        self.warp_ope, self.cost_func = warp_ope, cost_func

    def forward(self, left_feature_map, right_feature_map, **kargs):
        if kargs.get("disp_samples") is not None:
            D = int(kargs["disp_samples"].shape[1])
        else:
            D = int(kargs["max_disp"])
        return ops.cost_volume(left_feature_map.contiguous(), right_feature_map.contiguous(), D)


def get_disp_samples(max_dis, feature_map, stage_id=0, **_unused):
    """Stage-0 branch of modules/submodule.py:376-390 (the only one the model executes)."""
    B, _, H, W = feature_map.shape
    return torch.arange(int(max_dis), dtype=feature_map.dtype, device=feature_map.device) \
        .view(1, -1, 1, 1).expand(B, -1, H, W)


def disparity_regression(cost_vol, disp_samples=None):
    """Drop-in for modules/submodule.py:766-777 with integer candidates 0..D-1."""
    return ops.softargmin(cost_vol.contiguous())


# --------------------------------------------------------------------------------------
# a3: 3-D aggregation
# --------------------------------------------------------------------------------------
class CostRegNetNoDown(_Cached, nn.Module):
    """Drop-in for modules/submodule.py:608-662 (cost_func 'cor').  forward([B,C,D,H,W]) -> [B,D,H,W] on the
    hand-written bf16 implicit-GEMM kernel (decnet_conv3d_bf16: tcgen05, fp32 accumulation in TMEM); the north star's
    tolerance for this stage is 0.05 px EPE on the regressed disparity."""

    def __init__(self, in_channels, base_channels=None, cost_func="cor", down_scale=3):
        super().__init__()
        if cost_func != "cor":
            raise NotImplementedError("cost_func 'cor' only")
        c = in_channels
        self.conv0 = nn.Sequential(Conv3dUnit(c, c), Conv3dUnit(c, c))
        self.conv1 = nn.Sequential(Conv3dUnit(c, c), Conv3dUnit(c, c), Conv3dUnit(c, c))
        self.conv2 = nn.Sequential(Conv3dUnit(c, c), Conv3dUnit(c, c), Conv3dUnit(c, 1, relu=False))

    def units(self):
        return [*self.conv0, *self.conv1, *self.conv2]

    def forward(self, x):
        self._check_inference()
        from . import conv3d
        return conv3d.cost_regularizer_forward(self, x)


# --------------------------------------------------------------------------------------
# a5: learned lost-detail detector
# --------------------------------------------------------------------------------------
class GenerateSparseMask(_Cached, nn.Module):
    """Drop-in for modules/submodule.py:347-372."""

    def __init__(self, in_channels, down_scale=3):
        super().__init__()
        self.deconv = nn.Sequential(Deconv2dUnit(in_channels * down_scale, 8, 3, 3),
                                    Conv2dUnit(8, 3, 3, padding=1, relu=False))
        self.conv_sub = nn.Sequential(Conv2dUnit(in_channels, 8, 3, padding=1, relu=True, bn=False),
                                      Conv2dUnit(8, 3, 3, padding=1, relu=False))
        self.conv = nn.Sequential(Conv2dUnit(3, 3, 3, padding=1, relu=False),
                                  Conv2dUnit(3, 1, 1, padding=0, relu=False))

    def forward(self, cur_fea, pre_fea):
        cur_fea, wv = pad_pitch(cur_fea)
        pre = self.deconv[1](pad_pitch(self.deconv[0](pre_fea))[0], w_valid=wv)
        cur = self.conv_sub[1](self.conv_sub[0](cur_fea, w_valid=wv), w_valid=wv)
        res = (cur - pre) ** 2
        logit = self.conv[1](self.conv[0](res, w_valid=wv), w_valid=wv)
        return unpad_pitch(logit, wv).squeeze(1), unpad_pitch(cur, wv), unpad_pitch(pre, wv)

    def masks_pair(self, cur_l, pre_l, cur_r, pre_r, thold):
        """Left and right masks `sigmoid(forward(.)) > thold` with the tail fused: one kernel for both
        squared differences, and one for 1x1 conv + BN + sigmoid + threshold of both views (the comparison
        runs on the logit against the exact float where torch.sigmoid crosses `thold`)."""
        # widths that are not a multiple of 4 (KITTI) run on right-padded copies, the padding kept at zero (pad_pitch)
        cur_l, wv = pad_pitch(cur_l)
        cur_r, _ = pad_pitch(cur_r)
        pl = self.deconv[1](pad_pitch(self.deconv[0](pre_l))[0], w_valid=wv)
        pr = self.deconv[1](pad_pitch(self.deconv[0](pre_r))[0], w_valid=wv)
        cl = self.conv_sub[1](self.conv_sub[0](cur_l, w_valid=wv), w_valid=wv)
        cr = self.conv_sub[1](self.conv_sub[0](cur_r, w_valid=wv), w_valid=wv)
        rl, rr = ops.sqdiff_pair(cl, pl, cr, pr)
        xl, xr = self.conv[0](rl, w_valid=wv), self.conv[0](rr, w_valid=wv)

        def build():
            w, b = self.conv[1].folded()                    # [1,3,1,1], [1]
            return ([float(v) for v in w.flatten().cpu()], float(b.cpu()))
        w3, b1 = self._cached("head", build)
        ml, mr = ops.detail_head(xl.contiguous(), xr.contiguous(), w3, b1, ops.sigmoid_logit_threshold(thold, xl.device))
        return unpad_pitch(ml, wv), unpad_pitch(mr, wv)


# --------------------------------------------------------------------------------------
# a8: dynamic up-sampling
# --------------------------------------------------------------------------------------
class DynamicUpsampling(_Cached, nn.Module):
    """Drop-in for modules/submodule.py:566-589: channels-last pack kernel -> 3 tcgen05 convs on zero-bordered
    channels-last fp32 (conv2d_nhwc_halo_kernel) -> softmax / gather / pixel-shuffle glue kernel."""

    precision = "fp32"

    def __init__(self, in_channels, down_scale=3):
        super().__init__()
        assert down_scale == 3, "the reference hard-codes x3 (SURVEY.md D1)"
        n = down_scale ** 2 * 9
        self.weight_learning = nn.Sequential(Conv2dUnit(in_channels * 9 + 1, n, 3, padding=1),
                                             Conv2dUnit(n, n, 3, padding=1),
                                             Conv2dUnit(n, n, 3, padding=1, relu=False))

    def _pack(self):
        """(cp0, [(w_packed, bias, relu)] of the three convs) for the channels-last kernel, in this unit's precision."""
        self._check_inference()
        split = _split(self)

        def build():
            units = list(self.weight_learning)
            cin0 = units[0].conv.in_channels
            cp = (cin0 + 7) // 8 * 8
            packed = []
            for u in units:
                w, b = u.folded()
                wp, bp, np_ = ops.pack_conv2d_tf32_weights(w, b, cp, split=split)
                packed.append((wp, bp, u.relu))
                cp = np_
            return ((cin0 + 7) // 8 * 8, packed)
        return self._cached(("pack", split), build)

    def prepack(self, left_fea):
        """The feature channels of the conv input (everything but the disparity channel).  Independent of the
        disparity: the stage loop runs it ahead, on its second stream."""
        cp0, _ = self._pack()
        return ops.dynup_pack_nhwc(None, left_fea.contiguous(), cp0, round_tf32=not _split(self), pad=True)

    def forward(self, disp_map, left_fea, packed=None):
        disp_map = disp_map.contiguous()
        split = _split(self)
        cp0, packed_w = self._pack()
        # the tensors carry a one-pixel zero border, so one TMA fill per row tap serves the three column taps
        if packed is not None:
            x = ops.dynup_set_disp_nhwc(packed, disp_map, round_tf32=not split, pad=True)   # features packed ahead (prepack)
        else:
            x = ops.dynup_pack_nhwc(disp_map, left_fea.contiguous(), cp0, round_tf32=not split, pad=True)
        for i, (wp, bp, relu) in enumerate(packed_w):
            x = ops.conv2d_tf32_nhwc_halo(x, wp, bp, relu, round_out=(not split) and i + 1 < len(packed_w), split=split)
        return ops.dynup_glue_nhwc(x, disp_map, pad=True)


# --------------------------------------------------------------------------------------
# a13: soft attention (+ blend)
# --------------------------------------------------------------------------------------
class SoftAttention(nn.Module):
    """Drop-in for modules/submodule.py:593-604.  forward(x=[B,C+4,H,W]) -> sigmoid mask like the
    reference; `logits_cat()` + ops.blend() is the fused route the pipeline uses."""

    def __init__(self, in_channels, base_channels):
        super().__init__()
        self.conv = nn.Sequential(Conv2dUnit(in_channels, base_channels, 3, padding=1),
                                  Conv2dUnit(base_channels, base_channels, 3, padding=1),
                                  Conv2dUnit(base_channels, 1, 3, padding=1, relu=False))

    def logits(self, x):
        x, wv = pad_pitch(x)
        for u in self.conv:
            x = u(x, w_valid=wv)
        return unpad_pitch(x, wv)

    def logits_cat(self, left_fea, aux):
        """logits(cat(left_fea, aux)) with aux = [dense, sparse, left_mask, -var] as one [B,4,H,W] tensor."""
        left_fea, wv = pad_pitch(left_fea)
        aux, _ = pad_pitch(aux)
        x = self.conv[0].forward_cat([left_fea, aux], w_valid=wv)
        return unpad_pitch(self.conv[2](self.conv[1](x, w_valid=wv), w_valid=wv), wv)

    def forward(self, x):
        return torch.sigmoid(self.logits(x))


# --------------------------------------------------------------------------------------
# a14: refinement
# --------------------------------------------------------------------------------------
_REFINE_DIL = {0: (1,) * 6, 1: (1,) * 6, 2: (2, 1, 4, 1, 6, 1), 3: (3, 1, 6, 1, 9, 1)}


class Refinement(_Cached, nn.Module):
    """Drop-in for modules/submodule.py:666-762: warp kernel -> 7 convs (first one reading (left, warped, disp) as
    three sources) -> add."""

    precision = "fp32"

    def __init__(self, in_channels, base_channels=None, stage_id=-1, down_scale=3):
        super().__init__()
        c = in_channels
        dil = _REFINE_DIL[stage_id]
        chain = [(2 * c + 1, c), (c, c), (c, c), (c, c // 2), (c // 2, c // 2), (c // 2, c // 2)]
        layers = [Conv2dUnit(ci, co, 3, padding=d, dilation=d) for (ci, co), d in zip(chain, dil)]
        layers.append(Conv2dUnit(c // 2, 1, 3, padding=1, relu=False, bn=False))
        self.conv = nn.Sequential(*layers)

    def _wide_pack(self, n_wide):
        """Weights of the first `n_wide` layers for the zero-bordered channels-last kernel, in this unit's precision."""
        self._check_inference()
        split = _split(self)

        def build():
            units = list(self.conv)
            cp = (units[0].conv.in_channels + 7) // 8 * 8
            packed = []
            for u in units[:n_wide]:
                w, b = u.folded()
                wp, bp, np_ = ops.pack_conv2d_tf32_weights(w, b, cp, split=split)
                packed.append((wp, bp, u.relu))
                cp = np_
            return ((units[0].conv.in_channels + 7) // 8 * 8, packed)
        return self._cached(("wide", split, n_wide), build)

    def _is_wide(self):
        units = list(self.conv)
        return units[0].conv.out_channels >= 48 and all(u.conv.dilation == (1, 1) for u in units[:4])

    def _wide_head(self, srcs):
        """Wide level (1/9: 145 -> 72 -> 72 -> 72 -> 36 channels): GEMM-sized layers, too wide for the resident-weight NCHW
        kernel -> zero-bordered channels-last kernel between two layout bridges; returns the NCHW input of layer 4."""
        split = _split(self)
        cp0, packed = self._wide_pack(4)
        x = ops.nchw_cat_to_nhwc_pad(srcs, cp0, round_tf32=not split)
        for i, (wp, bp, relu) in enumerate(packed):
            x = ops.conv2d_tf32_nhwc_halo(x, wp, bp, relu, round_out=(not split) and i + 1 < len(packed), split=split)
        return ops.nhwc_pad_to_nchw(x, self.conv[3].conv.out_channels)

    def _tail(self, x, disp_map, start, wv, want_residual=True):
        for unit in list(self.conv)[start:-1]:
            x = unit(x, w_valid=wv)
        if want_residual:
            residual = unpad_pitch(self.conv[-1](x, w_valid=wv), wv).squeeze(1)
            return disp_map + residual, residual
        # inference: `disp + residual` (submodule.py:761) in the last conv's epilogue, the residual itself is not materialised
        add = disp_map if wv is None else pad_pitch(disp_map)[0]
        return unpad_pitch(self.conv[-1](x, addend=add, w_valid=wv), wv).squeeze(1), None

    def forward_packed(self, packed, disp_map, want_residual=True):
        """The conv stack on an already packed input cat(left, warped right, disp) [B,2C+1,H,W] (row-band mode: the
        warp needs global row coordinates, decnet_refine_pack_rows) -> (disp + residual, residual)."""
        disp_map = disp_map.contiguous()
        if self._is_wide():
            x, wv = pad_pitch(self._wide_head([packed.contiguous()]))
            return self._tail(x, disp_map, 4, wv, want_residual)
        x, wv = pad_pitch(packed.contiguous())
        return self._tail(x, disp_map, 0, wv, want_residual)

    def forward(self, left_fea, right_fea, disp_map, want_residual=True):
        """-> (disp + residual, residual) like the reference (submodule.py:747-762); want_residual=False (the model's inference
        path) adds the disparity in the last conv's epilogue and returns (disp + residual, None)."""
        disp_map = disp_map.contiguous()
        units = list(self.conv)
        c0 = units[0].conv
        C = left_fea.shape[1]
        split = _split(self)
        if self._is_wide():
            warped = ops.warp_bilinear(right_fea.contiguous(), disp_map)
            x, wv = pad_pitch(self._wide_head([left_fea.contiguous(), warped, disp_map]))
            return self._tail(x, disp_map, 4, wv, want_residual)
        Wp = (left_fea.shape[3] + 3) // 4 * 4
        if ops.conv2d_tf32_supported(ops.padded_cat_channels((C, C, 1)), c0.out_channels, left_fea.shape[2], Wp,
                                     c0.dilation[0], split):
            # first conv reads (left, warped right, disparity) as three sources: only the warp is materialised
            warped = ops.warp_bilinear(right_fea.contiguous(), disp_map)
            lp, wv = pad_pitch(left_fea.contiguous())
            x = units[0].forward_cat([lp, pad_pitch(warped)[0], pad_pitch(disp_map)[0]], w_valid=wv)
            return self._tail(x, disp_map, 1, wv, want_residual)
        return self.forward_packed(ops.refine_pack(left_fea.contiguous(), right_fea.contiguous(), disp_map), disp_map, want_residual)


# --------------------------------------------------------------------------------------
# a16: the stage loop
# --------------------------------------------------------------------------------------
class DecompMatching(nn.Module):
    """The decomposed-matching hot path: body of SparseDenseNetRefinementMask.forward after feature
    extraction (modules/SparseDenseNetRefinementMask.py:118-212), same hyper-parameters and the
    same sub-module names, so `load_state_dict(reference_state, strict=False)` picks up every
    hot-path weight (feature_extractor.* is ignored: out of scope).

    forward(left_feats, right_feats, left_mask_list=None, right_mask_list=None, is_check=False)
      left_feats/right_feats: {"stage0".."stage3"} NCHW fp32 CUDA tensors (C = 216,72,24,8)
      returns [pred] like the reference's inference path, or (pred, taps) with is_check.
    precision: "fp32" (3xTF32 tensor-core convs, fp32-class: the parity-gated default) or "tf32" (see module docstring).
    """

    def __init__(self, max_disp=216, base_channels=8, num_stage=4, down_scale=3, skip_stage_id=4,
                 use_detail=True, thold=0.9, channels=None, precision="fp32"):
        super().__init__()
        assert down_scale == 3 and num_stage == 4, "shipped configuration (demo.sh:1)"
        assert max_disp % (down_scale ** (num_stage - 1)) == 0, "max_disp must be a multiple of 27"
        self.max_disp, self.num_stage, self.down_scale = max_disp, num_stage, down_scale
        self.skip_stage_id, self.use_detail, self.thold = skip_stage_id, use_detail, thold
        ch = list(channels) if channels is not None else [27 * base_channels, 9 * base_channels,
                                                          3 * base_channels, base_channels]
        self.channels = ch
        self.get_cost_volume = GetCostVolume("homgrp", "cor")
        self.sparse_matching = nn.ModuleList([SpaMat() for _ in range(num_stage - 1)])
        self.sparse_var = nn.ModuleList([SpaVar() for _ in range(num_stage - 1)])
        self.cost_regularizer = CostRegNetNoDown(ch[0], ch[0] * 2, "cor", down_scale)
        self.detail_detection = nn.ModuleList([GenerateSparseMask(ch[i + 1], down_scale) for i in range(num_stage - 1)])
        self.dynamic_upsampling = nn.ModuleList([DynamicUpsampling(ch[i + 1], down_scale) for i in range(num_stage - 1)])
        self.soft_attention = nn.ModuleList([SoftAttention(ch[i + 1] + 4, base_channels) for i in range(num_stage - 1)])
        self.refinement = nn.ModuleList([Refinement(ch[i + 1], base_channels // (2 ** i), stage_id=i + 1,
                                                    down_scale=down_scale) for i in range(num_stage - 1)])
        self.set_precision(precision)
        self.eval()

    def set_precision(self, precision):
        """Arithmetic mode of every 2-D conv unit: "fp32" (3xTF32) or "tf32".  Returns self."""
        set_precision(self, precision)
        self.precision = precision
        return self

    def load_state_dict(self, state_dict, strict=False, **kw):
        sd = {k[7:] if k.startswith("module.") else k: v for k, v in state_dict.items()}   # demo.py:124-135
        sd = {k: v for k, v in sd.items() if not k.startswith("feature_extractor")}
        return super().load_state_dict(sd, strict=strict, **kw)

    # Masks (a5/a6) and the sparse ops (a9/a10) of every level depend on the features only, not on the disparity
    # coming up from the coarser level: they run on a second stream, forked at the start of forward() and joined
    # where the soft attention first needs them, so that they fill the SMs the main chain leaves idle (the last,
    # partial round of tiles of the persistent conv kernels, launch gaps).  Captured in a CUDA graph this becomes two
    # parallel branches.  `overlap = False` restores the single-stream order.
    overlap = True

    def _side_stream(self, main):
        """One side stream per (device, caller's stream): two callers on different streams never share it."""
        pool = self.__dict__.setdefault("_sides", {})
        key = (main.device, main.cuda_stream)
        if key not in pool:
            pool[key] = torch.cuda.Stream(main.device)
        return pool[key]

    @torch.no_grad()
    def forward(self, left_feats, right_feats, left_mask_list=None, right_mask_list=None, is_check=False,
                coarse_pred=None):
        """coarse_pred (test hook): a [B,H/27,W/27] disparity that replaces the result of the coarse dense stage, so the
        fp32-class stages can be checked against the reference without the bf16 aggregation's 0.05 px tolerance."""
        taps = {k: [] for k in ("pred", "dense", "sparse", "var", "soft_mask", "fusion", "residual",
                                "left_mask", "right_mask", "left_detail", "right_detail")} if is_check else None
        pred = None
        branch = events = packs = pack_events = side = main = None
        if self.overlap and not is_check:
            dev = left_feats["stage0"].device
            main = torch.cuda.current_stream(dev)
            side = self._side_stream(main)
            side.wait_stream(main)                       # fork: the features are ready on the main stream
            with torch.cuda.stream(side):
                branch, events, packs, pack_events = [], [], [], []
                # first what the main chain needs first: the feature channels of the first level's up-sampling input (the
                # other levels' packs follow the sparse launch below)
                packs, pack_events = [None] * (self.num_stage - 1), [None] * (self.num_stage - 1)

                def prepack(s):
                    if s < self.skip_stage_id:
                        pk = self.dynamic_upsampling[s - 1].prepack(left_feats[f"stage{s}"])
                        pk.record_stream(main)           # allocated in the side stream's pool, consumed on the main stream
                        ev = torch.cuda.Event()
                        ev.record(side)
                        packs[s - 1], pack_events[s - 1] = pk, ev
                prepack(1)
                # masks of every level first, then SpaMat + SpaVar of all levels in ONE launch (finest level's rows first: the
                # few rows of the coarse levels fill the machine behind them instead of being one-wave launches of their own)
                pre = (left_feats["stage0"].contiguous(), right_feats["stage0"].contiguous())
                lv = []
                for s in range(1, self.num_stage):
                    if s >= self.skip_stage_id:
                        continue
                    l = s - 1
                    Lf, Rf = left_feats[f"stage{s}"].contiguous(), right_feats[f"stage{s}"].contiguous()
                    D = self.max_disp // (self.down_scale ** (self.num_stage - s - 1))
                    if self.use_detail:
                        lm, rm = self.detail_detection[l].masks_pair(Lf, pre[0], Rf, pre[1], self.thold)
                        pre = (Lf, Rf)
                    else:
                        lm, rm = left_mask_list[l].contiguous(), right_mask_list[l].contiguous()
                    lv.append((Lf, Rf, lm, rm, D))
                outs = ops.spamat_spavar_forward_levels(lv[::-1])[::-1] if lv else []
                ev = torch.cuda.Event()
                ev.record(side)
                for s in range(1, self.num_stage):
                    if s >= self.skip_stage_id:
                        branch.append(None); events.append(None)
                        continue
                    (_, _, lm, rm, _), (sparse, var, _, _) = lv[s - 1], outs[s - 1]
                    for t in (lm, rm, sparse, var):
                        t.record_stream(main)
                    branch.append((lm, rm, sparse, var))
                    events.append(ev)
                for s in range(2, self.num_stage):
                    prepack(s)
        pre_l = pre_r = None
        for s in range(self.num_stage):
            Lf = left_feats[f"stage{s}"].contiguous()
            Rf = right_feats[f"stage{s}"].contiguous()
            D = self.max_disp // (self.down_scale ** (self.num_stage - s - 1))
            if s == 0:
                if coarse_pred is not None:
                    pred = coarse_pred.contiguous()
                else:
                    pred, cost = self.dense_stage(Lf, Rf, D)
                    if is_check:
                        taps["cost"] = cost
                pre_l, pre_r = Lf, Rf
            elif s >= self.skip_stage_id:
                # SparseDenseNetRefinementMask.py:143-144 (Middlebury's finest level): bicubic x3 of pred*3
                pred = ops.bicubic_skip(pred, Lf.shape[-2], Lf.shape[-1])
            else:
                l = s - 1
                if branch is not None:
                    if pack_events[l] is not None:
                        main.wait_event(pack_events[l])
                    dense = self.dynamic_upsampling[l](pred, Lf, packed=packs[l])
                    main.wait_event(events[l])                                     # join for this level
                    lm, rm, sparse, var = branch[l]
                else:
                    if self.use_detail:
                        lm, rm = self.detail_detection[l].masks_pair(Lf, pre_l, Rf, pre_r, self.thold)
                        if is_check:
                            ld, _, _ = self.detail_detection[l](Lf, pre_l)
                            rd, _, _ = self.detail_detection[l](Rf, pre_r)
                            taps["left_detail"].append(torch.sigmoid(ld).contiguous())
                            taps["right_detail"].append(torch.sigmoid(rd).contiguous())
                        pre_l, pre_r = Lf, Rf
                    else:
                        lm, rm = left_mask_list[l].contiguous(), right_mask_list[l].contiguous()
                    dense = self.dynamic_upsampling[l](pred, Lf)
                    sparse, var, _, _ = ops.spamat_spavar_forward(Lf, Rf, lm, rm, D)     # SpaMat + SpaVar, one pass
                aux = ops.attn_pack(None, dense, sparse, lm, var)                  # [dense, sparse, mask, -var]
                logit = self.soft_attention[l].logits_cat(Lf, aux).squeeze(1).contiguous()
                soft, fused = ops.blend(logit, dense, sparse, want_mask=is_check)
                pred, residual = self.refinement[l](Lf, Rf, fused, want_residual=is_check)
                if is_check:
                    for k, v in (("dense", dense), ("sparse", sparse), ("var", var), ("soft_mask", soft),
                                 ("fusion", fused), ("residual", residual), ("left_mask", lm), ("right_mask", rm)):
                        taps[k].append(v)
            if is_check:
                taps["pred"].append(pred)
        if side is not None:
            main.wait_stream(side)                       # join (a captured graph needs every forked stream back)
        return (pred, taps) if is_check else [pred]

    def dense_stage(self, Lf, Rf, D):
        """a1-a4: cost volume -> 3-D aggregation -> soft-argmin.  Returns (pred [B,H,W], cost [B,D,H,W])."""
        from . import conv3d
        self.cost_regularizer._check_inference()
        return conv3d.dense_pred(self.cost_regularizer, Lf, Rf, D)


def set_precision(module, precision):
    """Sets the conv arithmetic mode ("fp32" = 3xTF32, "tf32") on every decnet_b200 unit below `module` -- also for a
    reference model whose sub-modules were swapped for ours (INTEGRATION.md section 2)."""
    if precision not in PRECISIONS:
        raise ValueError(f"precision must be one of {PRECISIONS}, got {precision!r}")
    for m in module.modules():
        if isinstance(m, (Conv2dUnit, Deconv2dUnit, DynamicUpsampling, Refinement)):
            m.precision = precision
    return module
