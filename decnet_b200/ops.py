"""Torch-facing wrappers over the C ABI: validate tensors, pass raw device pointers and
the current CUDA stream.  PyTorch is plumbing here (memory + streams), not the product.
"""
from __future__ import annotations

import ctypes
import math
import numbers
import os

import numpy as np
import torch

from . import _lib


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _call(name, t, *args):
    """Call C entry `name` with args and the current stream, on t's device; raise DecnetError on a failed status."""
    with torch.cuda.device_of(t):
        st = getattr(_lib.lib(), name)(*args, _stream(t))
    _lib.check(st, name)


def _chk(name: str, t: torch.Tensor, ref: torch.Tensor | None = None, shape=None, split16_ok=False) -> None:
    """split16_ok: fp16 is accepted too, as the split16 storage of a channels-last tensor (see conv2d_tf32_nhwc_halo)."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise _lib.DecnetError(f"{name} must be a CUDA tensor (decnet_b200 has no CPU path)")
    if t.dtype != torch.float32 and not (split16_ok and t.dtype == torch.float16):
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    if ref is not None and t.device != ref.device:
        raise ValueError(f"{name} is on {t.device}, expected {ref.device}")
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {tuple(shape)}")


def _feat_args(ref_feas, tar_feas, ref_mask, tar_mask):
    _chk("ref_feas", ref_feas)
    if ref_feas.dim() != 4:
        raise ValueError("ref_feas must be [B,C,H,W]")
    B, Cc, H, W = ref_feas.shape
    _chk("tar_feas", tar_feas, ref_feas, (B, Cc, H, W))
    _chk("ref_mask", ref_mask, ref_feas, (B, H, W))
    _chk("tar_mask", tar_mask, ref_feas, (B, H, W))
    return B, Cc, H, W


def spamat_forward(ref_feas, tar_feas, ref_mask, tar_mask, max_disp, output=None, sum_sim=None, max_cost=None):
    """SpaMat forward -> (output, sum_similarities, max_cost), each [B,H,W]."""
    B, Cc, H, W = _feat_args(ref_feas, tar_feas, ref_mask, tar_mask)
    output = torch.empty_like(ref_mask) if output is None else output
    sum_sim = torch.empty_like(ref_mask) if sum_sim is None else sum_sim
    max_cost = torch.empty_like(ref_mask) if max_cost is None else max_cost
    for n, t in (("output", output), ("sum_similarities", sum_sim), ("max_cost", max_cost)):
        _chk(n, t, ref_feas, (B, H, W))
    _call("decnet_spamat_fwd", ref_feas,
          ref_feas.data_ptr(), tar_feas.data_ptr(), ref_mask.data_ptr(), tar_mask.data_ptr(),
          output.data_ptr(), sum_sim.data_ptr(), max_cost.data_ptr(),
          B, Cc, H, W, int(max_disp))
    return output, sum_sim, max_cost


def spavar_forward(ref_feas, tar_feas, ref_mask, tar_mask, disparity, max_disp,
                   output=None, sum_sim=None, max_cost=None):
    """SpaVar forward -> (variance, sum_similarities, max_cost)."""
    B, Cc, H, W = _feat_args(ref_feas, tar_feas, ref_mask, tar_mask)
    _chk("disparity", disparity, ref_feas, (B, H, W))
    output = torch.empty_like(ref_mask) if output is None else output
    sum_sim = torch.empty_like(ref_mask) if sum_sim is None else sum_sim
    max_cost = torch.empty_like(ref_mask) if max_cost is None else max_cost
    for n, t in (("output", output), ("sum_similarities", sum_sim), ("max_cost", max_cost)):
        _chk(n, t, ref_feas, (B, H, W))
    _call("decnet_spavar_fwd", ref_feas,
          ref_feas.data_ptr(), tar_feas.data_ptr(), ref_mask.data_ptr(), tar_mask.data_ptr(),
          disparity.data_ptr(), output.data_ptr(), sum_sim.data_ptr(), max_cost.data_ptr(),
          B, Cc, H, W, int(max_disp))
    return output, sum_sim, max_cost


def spamat_spavar_forward(ref_feas, tar_feas, ref_mask, tar_mask, max_disp):
    """Fused SpaMat + SpaVar(disparity = SpaMat output) -> (disp, var, sum_sim, max_cost)."""
    B, Cc, H, W = _feat_args(ref_feas, tar_feas, ref_mask, tar_mask)
    outs = [torch.empty_like(ref_mask) for _ in range(4)]
    _call("decnet_spamat_spavar_fwd", ref_feas,
          ref_feas.data_ptr(), tar_feas.data_ptr(), ref_mask.data_ptr(), tar_mask.data_ptr(),
          outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(), outs[3].data_ptr(),
          B, Cc, H, W, int(max_disp))
    return tuple(outs)


def spamat_spavar_forward_levels(levels):
    """Fused SpaMat + SpaVar of several pyramid levels in ONE launch.  levels: [(ref_feas, tar_feas, ref_mask, tar_mask,
    max_disp), ...] (finest level first for the best schedule) -> [(disp, var, sum_sim, max_cost), ...] in the same order."""
    n = len(levels)
    if not 1 <= n <= 4:
        raise ValueError("1..4 levels")
    outs, dims = [], []
    for (Lf, Rf, ml, mr, D) in levels:
        dims.append(_feat_args(Lf, Rf, ml, mr) + (int(D),))
        if Lf.device != levels[0][0].device:
            raise ValueError("all levels must live on one device")
        outs.append(tuple(torch.empty_like(ml) for _ in range(4)))
    vp = ctypes.c_void_p * n
    ia = ctypes.c_int * n
    _call("decnet_spamat_spavar_fwd_levels", levels[0][0], n,
          *[vp(*[lv[k].data_ptr() for lv in levels]) for k in range(4)],
          *[vp(*[o[k].data_ptr() for o in outs]) for k in range(4)],
          *[ia(*[d[k] for d in dims]) for k in range(5)])
    return outs


def spamat_backward(ref_feas, tar_feas, ref_mask, tar_mask, output, sum_sim, max_cost, grad_output,
                    max_disp, grad_ref=None, grad_tar=None):
    B, Cc, H, W = _feat_args(ref_feas, tar_feas, ref_mask, tar_mask)
    for n, t in (("output", output), ("sum_similarities", sum_sim), ("max_cost", max_cost),
                 ("grad_output", grad_output)):
        _chk(n, t, ref_feas, (B, H, W))
    grad_ref = torch.zeros_like(ref_feas) if grad_ref is None else grad_ref
    grad_tar = torch.zeros_like(tar_feas) if grad_tar is None else grad_tar
    _chk("grad_ref_feas", grad_ref, ref_feas, (B, Cc, H, W))
    _chk("grad_tar_feas", grad_tar, ref_feas, (B, Cc, H, W))
    _call("decnet_spamat_bwd", ref_feas,
          ref_feas.data_ptr(), tar_feas.data_ptr(), ref_mask.data_ptr(), tar_mask.data_ptr(),
          output.data_ptr(), sum_sim.data_ptr(), max_cost.data_ptr(), grad_output.data_ptr(),
          grad_ref.data_ptr(), grad_tar.data_ptr(), B, Cc, H, W, int(max_disp))
    return grad_ref, grad_tar


def spavar_backward(ref_feas, tar_feas, ref_mask, tar_mask, disparity, output, sum_sim, max_cost,
                    grad_output, max_disp, grad_ref=None, grad_tar=None, grad_disp=None):
    B, Cc, H, W = _feat_args(ref_feas, tar_feas, ref_mask, tar_mask)
    for n, t in (("disparity", disparity), ("output", output), ("sum_similarities", sum_sim),
                 ("max_cost", max_cost), ("grad_output", grad_output)):
        _chk(n, t, ref_feas, (B, H, W))
    grad_ref = torch.zeros_like(ref_feas) if grad_ref is None else grad_ref
    grad_tar = torch.zeros_like(tar_feas) if grad_tar is None else grad_tar
    grad_disp = torch.zeros_like(disparity) if grad_disp is None else grad_disp
    _chk("grad_ref_feas", grad_ref, ref_feas, (B, Cc, H, W))
    _chk("grad_tar_feas", grad_tar, ref_feas, (B, Cc, H, W))
    _chk("grad_disparity", grad_disp, ref_feas, (B, H, W))
    _call("decnet_spavar_bwd", ref_feas,
          ref_feas.data_ptr(), tar_feas.data_ptr(), ref_mask.data_ptr(), tar_mask.data_ptr(),
          disparity.data_ptr(), output.data_ptr(), sum_sim.data_ptr(), max_cost.data_ptr(),
          grad_output.data_ptr(), grad_ref.data_ptr(), grad_tar.data_ptr(), grad_disp.data_ptr(),
          B, Cc, H, W, int(max_disp))
    return grad_ref, grad_tar, grad_disp


def candidate_signature(ref_mask, tar_mask, max_disp):
    """(count int32 [B,H,W], hash int64 [B,H,W]) of every pixel's candidate set."""
    _chk("ref_mask", ref_mask)
    _chk("tar_mask", tar_mask, ref_mask, ref_mask.shape)
    B, H, W = ref_mask.shape
    count = torch.empty((B, H, W), dtype=torch.int32, device=ref_mask.device)
    hsh = torch.empty((B, H, W), dtype=torch.int64, device=ref_mask.device)
    _call("decnet_candidate_signature", ref_mask,
          ref_mask.data_ptr(), tar_mask.data_ptr(), count.data_ptr(), hsh.data_ptr(), B, H, W, int(max_disp))
    return count, hsh


# --------------------------------------------------------------------------------------
# dense stage + glue (SURVEY.md section 8 rows a2, a4, a6, a8, a13, a14)
# --------------------------------------------------------------------------------------
def cost_volume(left_fea, right_fea, D):
    """fp32 NCDHW cost volume [B,C,D,H,W] (reference layout)."""
    _chk("left_fea", left_fea)
    B, Cc, H, W = left_fea.shape
    _chk("right_fea", right_fea, left_fea, (B, Cc, H, W))
    vol = torch.empty((B, Cc, int(D), H, W), dtype=torch.float32, device=left_fea.device)
    _call("decnet_costvol_fwd", left_fea, left_fea.data_ptr(), right_fea.data_ptr(), vol.data_ptr(), B, Cc, H, W, int(D))
    return vol


def cost_volume_bf16_ndhwc(left_fea, right_fea, D, Cpad):
    """bf16 channels-last cost volume [B,D,H,W,Cpad] (input of the tcgen05 conv)."""
    _chk("left_fea", left_fea)
    B, Cc, H, W = left_fea.shape
    _chk("right_fea", right_fea, left_fea, (B, Cc, H, W))
    vol = torch.empty((B, int(D), H, W, int(Cpad)), dtype=torch.bfloat16, device=left_fea.device)
    _call("decnet_costvol_bf16_ndhwc", left_fea, left_fea.data_ptr(), right_fea.data_ptr(), vol.data_ptr(),
          B, Cc, int(Cpad), H, W, int(D))
    return vol


def softargmin(cost):
    _chk("cost", cost)
    B, D, H, W = cost.shape
    pred = torch.empty((B, H, W), dtype=torch.float32, device=cost.device)
    _call("decnet_softargmin", cost, cost.data_ptr(), pred.data_ptr(), B, D, H, W)
    return pred


def mask_threshold(prob_l, prob_r, thold, with_counts=False):
    _chk("prob_l", prob_l)
    _chk("prob_r", prob_r, prob_l, prob_l.shape)
    B, H, W = prob_l.shape
    ml, mr = torch.empty_like(prob_l), torch.empty_like(prob_r)
    cl = cr = None
    if with_counts:
        cl = torch.empty(B * H, dtype=torch.int32, device=prob_l.device)
        cr = torch.empty(B * H, dtype=torch.int32, device=prob_l.device)
    _call("decnet_mask_threshold", prob_l, prob_l.data_ptr(), prob_r.data_ptr(), float(thold), ml.data_ptr(),
          mr.data_ptr(), cl.data_ptr() if with_counts else None, cr.data_ptr() if with_counts else None, B, H, W)
    return (ml, mr, cl, cr) if with_counts else (ml, mr)


def sqdiff_pair(a0, b0, a1, b1):
    """((a0 - b0)**2, (a1 - b1)**2) in one launch (GenerateSparseMask, both views)."""
    _chk("a0", a0)
    for n, t in (("b0", b0), ("a1", a1), ("b1", b1)):
        _chk(n, t, a0, a0.shape)
    o0, o1 = torch.empty_like(a0), torch.empty_like(a1)
    _call("decnet_sqdiff_pair", a0, a0.data_ptr(), b0.data_ptr(), o0.data_ptr(), a1.data_ptr(), b1.data_ptr(), o1.data_ptr(),
          a0.numel())
    return o0, o1


_LOGIT_THOLD = {}


def sigmoid_logit_threshold(thold, device):
    """Smallest float32 x with torch.sigmoid(x) > thold on `device` (bisection over floats; sigmoid is monotone),
    so that `x >= result` reproduces `torch.sigmoid(x) > thold` bit for bit."""
    key = (float(thold), str(device))
    if key not in _LOGIT_THOLD:
        t = float(thold)
        lo = torch.tensor(-120.0, device=device)       # sigmoid(lo) == 0 <= t
        hi = torch.tensor(120.0, device=device)        # sigmoid(hi) == 1 >  t   (t < 1)
        if not (0.0 <= t < 1.0):
            raise ValueError("thold must be in [0, 1)")
        for _ in range(80):
            mid = ((lo.double() + hi.double()) * 0.5).float()
            if bool(mid == lo) or bool(mid == hi):
                break
            if bool(torch.sigmoid(mid) > t):
                hi = mid
            else:
                lo = mid
        _LOGIT_THOLD[key] = float(hi)
    return _LOGIT_THOLD[key]


def detail_head(x_l, x_r, w3, bias, logit_thold):
    """masks (left, right) from the 3-channel maps in front of GenerateSparseMask's last 1x1 conv."""
    _chk("x_l", x_l)
    B, c, H, W = x_l.shape
    if c != 3:
        raise ValueError("detail_head expects 3 channels")
    _chk("x_r", x_r, x_l, (B, 3, H, W))
    ml = torch.empty((B, H, W), dtype=torch.float32, device=x_l.device)
    mr = torch.empty_like(ml)
    _call("decnet_detail_head", x_l, x_l.data_ptr(), x_r.data_ptr(), (ctypes.c_float * 3)(*[float(v) for v in w3]),
          float(bias), float(logit_thold), ml.data_ptr(), mr.data_ptr(), B, H, W)
    return ml, mr


IMAGENET_MEAN, IMAGENET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)       # demo.py:85-86


def image_prepare_u8(img_u8, multiple=27, want01=True, want_norm=True, mean=IMAGENET_MEAN, std=IMAGENET_STD, col_shift=0):
    """uint8 RGB [B,h,w,3] (CUDA) -> (img01, img_norm) fp32 [B,3,H,W], top/left zero-padded to multiples of
    `multiple` like demo.py:75-81; img01 = v/255, img_norm = (v/255 - mean)/std (demo.py:82-88).  col_shift (an int)
    first shifts the image right by that many columns, black where the source column lies outside the image
    (oracle/disp_range.py's shift_cols_u8): the right view of a search range starting at min_disp = col_shift."""
    if not (isinstance(img_u8, torch.Tensor) and img_u8.is_cuda and img_u8.dtype == torch.uint8 and img_u8.is_contiguous()
            and img_u8.dim() == 4 and img_u8.shape[3] == 3):
        raise ValueError("img_u8 must be a contiguous CUDA uint8 tensor [B,h,w,3]")
    if isinstance(col_shift, (bool, np.bool_)) or not isinstance(col_shift, numbers.Integral):
        raise ValueError(f"col_shift must be an integer number of columns, got {col_shift!r}")
    B, h, w, _ = img_u8.shape
    H, W = -(-h // multiple) * multiple, -(-w // multiple) * multiple
    o01 = torch.empty((B, 3, H, W), dtype=torch.float32, device=img_u8.device) if want01 else None
    onm = torch.empty((B, 3, H, W), dtype=torch.float32, device=img_u8.device) if want_norm else None
    args = (img_u8.data_ptr(), o01.data_ptr() if want01 else None, onm.data_ptr() if want_norm else None,
            (ctypes.c_float * 3)(*mean), (ctypes.c_float * 3)(*std), B, h, w, H, W)
    if col_shift == 0:
        _call("decnet_image_prepare_u8", img_u8, *args)
    else:                                                                  # beyond +-w every column is black alike
        _call("decnet_image_prepare_u8_shift", img_u8, *args, max(-w, min(w, int(col_shift))))
    return o01, onm


def disp_to_u16(pred, ori_h, ori_w):
    """[B,H,W] fp32 disparity -> [B,ori_h,ori_w] uint16 (x256, clamped, cropped bottom/right) as demo.py:191-197."""
    _chk("pred", pred)
    B, H, W = pred.shape
    out = torch.empty((B, int(ori_h), int(ori_w)), dtype=torch.uint16, device=pred.device)
    _call("decnet_disp_to_u16", pred, pred.data_ptr(), out.data_ptr(), B, H, W, int(ori_h), int(ori_w))
    return out


def disp_add(pred, offset):
    """pred += offset in place, in fp32 rounded to nearest (pred + torch.float32(offset) bit for bit); pred a contiguous
    CUDA fp32 tensor of any shape, offset a real number (not a bool) that float32 represents exactly.  Returns pred."""
    _chk("pred", pred)
    if (isinstance(offset, (bool, np.bool_)) or not isinstance(offset, numbers.Real)
            or float(np.float32(offset)) != float(offset)):
        raise ValueError(f"offset must be a number that float32 represents exactly, got {offset!r}")
    if pred.numel():
        _call("decnet_disp_add", pred, pred.data_ptr(), float(offset), pred.numel())
    return pred


def mirror_swap_u8(left, right, out_left, out_right):
    """out_left = left view of the reverse direction = mirror(right), out_right = mirror(left) (mirror flips columns), all
    contiguous CUDA uint8 [B,h,w,3]; writes into the given tensors (views of a larger buffer are fine) and returns them."""
    shape = tuple(left.shape) if isinstance(left, torch.Tensor) else None
    for name, t in (("left", left), ("right", right), ("out_left", out_left), ("out_right", out_right)):
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.uint8 and t.is_contiguous() and t.dim() == 4
                and t.shape[3] == 3):
            raise ValueError(f"{name} must be a contiguous CUDA uint8 tensor [B,h,w,3]")
        if tuple(t.shape) != shape or t.device != left.device:
            raise ValueError(f"{name} {tuple(t.shape)} on {t.device} does not match left {shape} on {left.device}")
    B, h, w, _ = shape
    _call("decnet_mirror_swap_u8", left, left.data_ptr(), right.data_ptr(), out_left.data_ptr(), out_right.data_ptr(), B, h, w)
    return out_left, out_right


def lr_tolerance(tol):
    """A left-right check tolerance in pixels as a float: a finite real number >= 0 that is not a bool, else ValueError."""
    if isinstance(tol, (bool, np.bool_)) or not isinstance(tol, numbers.Real) or not math.isfinite(tol) or tol < 0:
        raise ValueError(f"the left-right check tolerance must be a finite number of pixels >= 0, got {tol!r}")
    return float(tol)


LR_FILLS = ("none", "background", "guided")
GUIDED_LAMBDA = 8000.0         # fill="guided": smoothness weight lambda of the fast global smoother (OpenCV's default)
GUIDED_SIGMA = 2.6             # and its colour scale on the L1 colour distance (OpenCV's 1.5 on the Euclidean one, x sqrt(3))


def lr_fill(fill):
    """A hole-filling rule of the left-right check: one of LR_FILLS, else ValueError."""
    if not isinstance(fill, str) or fill not in LR_FILLS:
        raise ValueError(f"fill must be one of {LR_FILLS}, got {fill!r}")
    return fill


def lr_speckle(size, rng):
    """Speckle filter settings of the left-right check -> (size, range): size an int >= 0 (not a bool; 0: off), range a
    number of disparity pixels that is finite as a float32 and >= 0 (not a bool), else ValueError."""
    if isinstance(size, (bool, np.bool_)) or not isinstance(size, numbers.Integral) or size < 0:
        raise ValueError(f"speckle_size must be an integer number of pixels >= 0 (0: off), got {size!r}")
    if (isinstance(rng, (bool, np.bool_)) or not isinstance(rng, numbers.Real) or not math.isfinite(rng) or rng < 0
            or abs(float(rng)) > float(np.finfo(np.float32).max)):
        raise ValueError(f"speckle_range must be a finite number of disparity pixels >= 0, got {rng!r}")
    return int(size), float(rng)


def lr_check(pred, ori_h, ori_w, tol, float_out=True, u16_out=False, valid_out=False, fill="none", guide=None,
             speckle_size=0, speckle_range=1.0):
    """Left-right consistency check (oracle/lr_check.py).  pred fp32 [2B,H,W]: the forward padded predictions, then
    those of the mirrored, swapped pairs.  Returns a tuple of the requested [B,ori_h,ori_w] outputs, in this order:
    float (the forward disparity where valid, else 0), uint16 (disp_to_u16's value where valid, else 0), bool valid.
    fill="background" fills the invalid pixels from their valid neighbours instead of 0 (oracle/lr_fill.py: the smaller
    value of the nearest valid pixels left and right in the row, then rows without one from the rows above and below);
    fill="guided" spreads the valid disparities along the left images `guide` (contiguous CUDA uint8 [B,ori_h,ori_w,3],
    required for it and rejected otherwise), stopping at colour edges (oracle/lr_guided.py, GUIDED_LAMBDA and
    GUIDED_SIGMA), with the background value where no valid pixel reaches; valid stays the check's mask, False on every
    filled pixel.  speckle_size > 0 removes speckles before the fill (oracle/lr_speckle.py): valid 4-neighbours whose
    disparities differ by at most speckle_range join a region, and every region of at most speckle_size pixels becomes
    invalid (0, or filled); valid is then the check's mask minus the speckles.  speckle_size = 0 runs no filter."""
    fill = lr_fill(fill)
    speckle_size, speckle_range = lr_speckle(speckle_size, speckle_range)
    if (guide is not None) != (fill == "guided"):
        raise ValueError(f"guide is required for fill=\"guided\" and only for it (fill={fill!r}, guide "
                         f"{'given' if guide is not None else 'missing'})")
    _chk("pred", pred)
    if pred.dim() != 3 or pred.shape[0] % 2 or pred.shape[0] == 0:
        raise ValueError(f"pred must be [2B,H,W] (forward then reverse), got {tuple(pred.shape)}")
    B2, H, W = pred.shape
    if not (0 < int(ori_h) <= H and 0 < int(ori_w) <= W):
        raise ValueError(f"crop {ori_h}x{ori_w} outside the {H}x{W} map")
    tol = lr_tolerance(tol)
    if not (float_out or u16_out or valid_out):
        raise ValueError("request at least one output")
    shape, dev = (B2 // 2, int(ori_h), int(ori_w)), pred.device
    if guide is not None and not (isinstance(guide, torch.Tensor) and guide.is_cuda and guide.dtype == torch.uint8
                                  and guide.is_contiguous() and tuple(guide.shape) == shape + (3,) and guide.device == dev):
        raise ValueError(f"guide must be a contiguous CUDA uint8 tensor {list(shape) + [3]} on {dev}, got "
                         + (f"{guide.dtype} {tuple(guide.shape)} on {guide.device}" if isinstance(guide, torch.Tensor)
                            else type(guide).__name__))
    f = torch.empty(shape, dtype=torch.float32, device=dev) if float_out or fill != "none" else None
    u = torch.empty(shape, dtype=torch.uint16, device=dev) if u16_out else None
    v = torch.empty(shape, dtype=torch.bool, device=dev) if valid_out or fill == "guided" else None
    args = (B2 // 2, H, W, int(ori_h), int(ori_w), float(tol))
    outs = tuple(t.data_ptr() if t is not None else None for t in (f, u, v))
    if speckle_size:
        kind = LR_FILLS.index(fill)
        flags = torch.empty(shape[:2], dtype=torch.uint8, device=dev) if fill != "none" else None
        scratch = torch.empty(int(_lib.lib().decnet_lr_speckle_scratch_bytes(*shape, kind)), dtype=torch.uint8, device=dev)
        size = min(speckle_size, 2**31 - 1)                                # a region has fewer pixels: the same filter
        _call("decnet_lr_check_speckle", pred, pred.data_ptr(), guide.data_ptr() if guide is not None else None, *args,
              size, speckle_range, kind, GUIDED_LAMBDA, GUIDED_SIGMA, *outs, flags.data_ptr() if flags is not None else None,
              scratch.data_ptr())
    elif fill == "none":
        _call("decnet_lr_check", pred, pred.data_ptr(), *args, *outs)
    else:                                                                  # the float rows are the fill's scratch too
        flags = torch.empty(shape[:2], dtype=torch.uint8, device=dev)
        if fill == "background":
            _call("decnet_lr_check_fill", pred, pred.data_ptr(), *args, *outs, flags.data_ptr())
        else:
            scratch = torch.empty(int(_lib.lib().decnet_lr_guided_fill_scratch_floats(*shape)), dtype=torch.float32,
                                  device=dev)
            _call("decnet_lr_check_guided_fill", pred, pred.data_ptr(), guide.data_ptr(), *args, GUIDED_LAMBDA,
                  GUIDED_SIGMA, *outs, flags.data_ptr(), scratch.data_ptr())
    return tuple(t for t, want in ((f, float_out), (u, u16_out), (v, valid_out)) if want)


def epe_3px(pred, gt, max_disp):
    """(epe, 3-px error %) of modules/loss.py:427-437 as device tensors."""
    _chk("pred", pred)
    _chk("gt", gt, pred, pred.shape)
    sums = torch.empty(3, dtype=torch.float64, device=pred.device)
    _call("decnet_epe_3px", pred, pred.data_ptr(), gt.data_ptr(), float(max_disp), sums.data_ptr(), pred.numel())
    return (sums[0] / sums[2]).float(), (100.0 - 100.0 * sums[1] / sums[2]).float()


def detail_detection(img, iters=3, thold=0.3):
    """Image-space lost-detail masks (reference: utils.detailDetection, demo.py:161-162) for images already padded
    to a multiple of 3**iters: img [B,3,H,W] in [0,1] -> [mask_full, mask_1/3, ...] fp32 {0,1} [B,H/3^i,W/3^i]."""
    _chk("img", img)
    B, c, H, W = img.shape
    if c != 3 or H % 3 ** iters or W % 3 ** iters:
        raise ValueError(f"img must be [B,3,H,W] with H, W multiples of {3 ** iters}, got {tuple(img.shape)}")
    scratch = torch.empty(int(_lib.lib().decnet_detail_level_scratch_floats(B, H, W)), dtype=torch.float32, device=img.device)
    masks, data = [], img
    for _ in range(iters):
        h, w = data.shape[2], data.shape[3]
        down = torch.empty((B, 3, h // 3, w // 3), dtype=torch.float32, device=img.device)
        mask = torch.empty((B, h, w), dtype=torch.float32, device=img.device)
        _call("decnet_detail_level", data, data.data_ptr(), down.data_ptr(), mask.data_ptr(), scratch.data_ptr(),
              float(thold), B, h, w)
        masks.append(mask)
        data = down
    return masks


def bicubic_skip(pred, out_h, out_w):
    """Skip-stage up-sampling (SparseDenseNetRefinementMask.py:143-144): pred [B,h,w] -> [B,out_h,out_w] equal, bit for bit,
    to F.interpolate((pred*3).unsqueeze(1), (out_h, out_w), mode="bicubic").squeeze(1) on CUDA."""
    _chk("pred", pred)
    if pred.dim() != 3:
        raise ValueError(f"pred must be [B,h,w], got {tuple(pred.shape)}")
    B, h, w = pred.shape
    out = torch.empty((B, int(out_h), int(out_w)), dtype=torch.float32, device=pred.device)
    _call("decnet_bicubic_up3", pred, pred.data_ptr(), out.data_ptr(), B, h, w, int(out_h), int(out_w))
    return out


def dynup_pack(disp, left_fea):
    _chk("disp", disp)
    B, h, w = disp.shape
    _chk("left_fea", left_fea, disp)
    Cc = left_fea.shape[1]
    if tuple(left_fea.shape) != (B, Cc, 3 * h, 3 * w):
        raise ValueError(f"left_fea {tuple(left_fea.shape)} is not 3x the disparity map {tuple(disp.shape)}")
    out = torch.empty((B, 9 * Cc + 1, h, w), dtype=torch.float32, device=disp.device)
    _call("decnet_dynup_pack", disp, disp.data_ptr(), left_fea.data_ptr(), out.data_ptr(), B, Cc, h, w)
    return out


def dynup_glue(logits, disp):
    _chk("disp", disp)
    B, h, w = disp.shape
    _chk("logits", logits, disp, (B, 81, h, w))
    out = torch.empty((B, 3 * h, 3 * w), dtype=torch.float32, device=disp.device)
    _call("decnet_dynup_glue", disp, logits.data_ptr(), disp.data_ptr(), out.data_ptr(), B, h, w)
    return out


def attn_pack(left_fea, dense, sparse, left_mask, var):
    """cat(left_fea, dense, sparse, left_mask, -var) -> [B,C+4,H,W]; left_fea=None packs the four maps only."""
    _chk("dense", dense)
    B, H, W = dense.shape
    Cc = 0
    if left_fea is not None:
        _chk("left_fea", left_fea, dense)
        Cc = left_fea.shape[1]
        if tuple(left_fea.shape) != (B, Cc, H, W):
            raise ValueError(f"left_fea {tuple(left_fea.shape)} does not match dense {tuple(dense.shape)}")
    for n, t in (("sparse", sparse), ("left_mask", left_mask), ("var", var)):
        _chk(n, t, dense, (B, H, W))
    out = torch.empty((B, Cc + 4, H, W), dtype=torch.float32, device=dense.device)
    _call("decnet_attn_pack", dense, left_fea.data_ptr() if left_fea is not None else None, dense.data_ptr(),
          sparse.data_ptr(), left_mask.data_ptr(), var.data_ptr(), out.data_ptr(), B, Cc, H, W)
    return out


def blend(logit, dense, sparse, want_mask=True):
    _chk("logit", logit)
    B, H, W = logit.shape
    _chk("dense", dense, logit, (B, H, W))
    _chk("sparse", sparse, logit, (B, H, W))
    fused = torch.empty_like(dense)
    soft = torch.empty_like(dense) if want_mask else None
    _call("decnet_blend", logit, logit.data_ptr(), dense.data_ptr(), sparse.data_ptr(),
          soft.data_ptr() if want_mask else None, fused.data_ptr(), B, H, W)
    return soft, fused


def warp_bilinear(right_fea, disp):
    _chk("right_fea", right_fea)
    B, Cc, H, W = right_fea.shape
    _chk("disp", disp, right_fea, (B, H, W))
    out = torch.empty_like(right_fea)
    _call("decnet_warp_bilinear", right_fea, right_fea.data_ptr(), disp.data_ptr(), out.data_ptr(), B, Cc, H, W)
    return out


def refine_pack(left_fea, right_fea, disp):
    _chk("left_fea", left_fea)
    B, Cc, H, W = left_fea.shape
    _chk("right_fea", right_fea, left_fea, (B, Cc, H, W))
    _chk("disp", disp, left_fea, (B, H, W))
    out = torch.empty((B, 2 * Cc + 1, H, W), dtype=torch.float32, device=left_fea.device)
    _call("decnet_refine_pack", left_fea, left_fea.data_ptr(), right_fea.data_ptr(), disp.data_ptr(), out.data_ptr(),
          B, Cc, H, W)
    return out


def haar_detail_masks(x, levels):
    """Haar lost-detail masks (row a7): x [B,1,H,W] -> ([mask_level1, ...] each [B,1,H/2^k,W/2^k], LL)."""
    _chk("x", x)
    if x.dim() != 4 or x.shape[1] != 1:
        raise ValueError("x must be [B,1,H,W]")
    th = (ctypes.c_float * 10)(*[float(np.float32(t)) for t in (np.arange(0, 1, 0.1) + 0.1)])
    masks, cur = [], x
    for _ in range(int(levels)):
        B, _, H, W = cur.shape
        h, w = H // 2, W // 2
        ll = torch.empty((B, 1, h, w), dtype=torch.float32, device=x.device)
        det = torch.empty_like(ll)
        mask = torch.empty_like(ll)
        ws = torch.empty(B * 12, dtype=torch.int32, device=x.device)
        _call("decnet_haar_level", cur, cur.data_ptr(), ll.data_ptr(), det.data_ptr(), mask.data_ptr(), ws.data_ptr(), th,
              B, H, W)
        masks.append(mask)
        cur = ll
    return masks, cur


# --------------------------------------------------------------------------------------
# tiny-channel 2-D convolutions (section 8f rank 1)
# --------------------------------------------------------------------------------------
def conv2d_small_supported(cin, cout, ksize):
    return bool(_lib.lib().decnet_conv2d_small_supported(int(cin), int(cout), int(ksize)))


def pack_conv2d_weights(w):
    """[Cout,Cin,k,k] -> [Cin][k*k][CoutP] fp32 (CoutP = Cout rounded up to 4)."""
    cout, cin, k, _ = w.shape
    coutp = (cout + 3) // 4 * 4
    out = torch.zeros((cin, k * k, coutp), dtype=torch.float32, device=w.device)
    out[:, :, :cout] = w.float().permute(1, 2, 3, 0).reshape(cin, k * k, cout)
    return out.contiguous()


def conv2d_small(x, w_packed, bias, cout, ksize, dilation=1, relu=False, addend=None):
    _chk("x", x)
    B, cin, H, W = x.shape
    out = torch.empty((B, cout, H, W), dtype=torch.float32, device=x.device)
    if addend is not None:
        _chk("addend", addend, x, (B, H, W))
    _call("decnet_conv2d_small", x, x.data_ptr(), w_packed.data_ptr(), bias.data_ptr(),
          addend.data_ptr() if addend is not None else None, out.data_ptr(), B, cin, H, W, int(cout), int(ksize),
          int(dilation), 1 if relu else 0)
    return out


def deconv3x3s3_supported(cout):
    return int(cout) in (8, 24)


def deconv3x3s3(x, w, bias, relu=True):
    _chk("x", x)
    B, cin, h, wd = x.shape
    cout = w.shape[1]
    out = torch.empty((B, cout, 3 * h, 3 * wd), dtype=torch.float32, device=x.device)
    _call("decnet_deconv3x3s3", x, x.data_ptr(), w.data_ptr(), bias.data_ptr(), out.data_ptr(), B, cin, h, wd, cout,
          1 if relu else 0)
    return out


# --------------------------------------------------------------------------------------
# GEMM-sized 3x3 Conv2d on tensor cores (TF32 tcgen05 implicit GEMM, channels-last)
# --------------------------------------------------------------------------------------
def rna_tf32(t):
    """Round an fp32 tensor to TF32 (nearest, ties away: cvt.rna) -- the MMA itself would truncate the low 13 mantissa bits."""
    return ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def split_tf32(t):
    """(hi, lo) with hi = rna_tf32(t), lo = rna_tf32(t - hi): the operand split of the 3xTF32 ("fp32-class") conv mode
    (t - hi is exact in fp32; hi*hi' + hi*lo' + lo*hi' reproduces the fp32 product to ~2^-22 relative)."""
    hi = rna_tf32(t)
    return hi, rna_tf32(t - hi)


# How the channels-last tensor-core kernel (conv2d_nhwc_tcgen05.cu) builds an fp32-class product, the `split` argument of
# its entry points: 1 = 3xTF32 (hi*hi + lo*hi + hi*lo, all kind::tf32), 2 = hi*hi in TF32 + both correction terms as ONE
# K-concatenated fp16 MMA ([lo16(x) | fp16(x)] * [hi16(w) ; lo16(w)]): a third fewer operand bytes through shared memory.
# The TF32 hi / lo parts have 11 significant bits, so fp16 holds them exactly once a per-layer power of two brings the weights
# into its exponent range; DECNET_SPLIT_KIND=1 selects the all-TF32 form (A/B measurements).
SPLIT_KIND = int(os.environ.get("DECNET_SPLIT_KIND", "2"))
if SPLIT_KIND not in (1, 2):
    raise ValueError("DECNET_SPLIT_KIND must be 1 or 2")


def _split_arg(split):
    return SPLIT_KIND if split else 0


def _fp16_split(hi, lo):
    """(sw, fp16(hi * 2^sw), fp16(lo * 2^(11+sw))): the weight halves of split kind 2's fp16 correction MMA.  sw is a 0-dim
    int32 tensor on hi's device (no host sync: packing may run under stream capture) with max|hi| * 2^sw just below 2^13,
    which brings the weights into fp16's exponent range with room on both sides."""
    m = hi.abs().max()
    e = torch.frexp(torch.where(torch.isfinite(m) & (m > 0), m, torch.ones_like(m)))[1]
    sw = (13 - e).clamp(-40, 40).to(torch.int32)
    wh = torch.ldexp(hi, sw).clamp(-65504.0, 65504.0).to(torch.float16)
    wl = torch.ldexp(lo, sw + 11).clamp(-65504.0, 65504.0).to(torch.float16)
    return sw, wh, wl


def _pack_split_weights(out, bias_np, split16_in=False):
    """out fp32 [T][NP][cp] -> ([2T][NP][cp] for the split modes of the channels-last kernel, bias [NP + 4]).
    Taps 0..T-1: the TF32 hi parts.  Taps T..2T-1, SPLIT_KIND 1: the TF32 lo parts; SPLIT_KIND 2: per 32-channel chunk of cl
    channels the 4*cl bytes [fp16(hi * 2^sw) x cl | fp16(lo * 2^(11+sw)) x cl] -- the B operand of the fp16 correction MMA,
    whose A operand is [fp16(2^11 * lo(x)) | fp16(x)]; both products carry the factor 2^(11+sw), and bias[NP] = 2^-(11+sw) is
    what the epilogue multiplies the correction accumulator with.  sw puts the largest weight just below 2^13.
    split16_in (activations stored as split16, kernel split = 3): only those fp16 taps, [T][NP][cp]; the kernel also multiplies
    their hi16 half with h = fp16(x), and bias[NP + 1] = 2^-sw scales that product back."""
    hi, lo = split_tf32(out)
    b = torch.zeros(bias_np.numel() + 4, dtype=torch.float32, device=out.device)
    b[:bias_np.numel()] = bias_np
    if SPLIT_KIND == 1 and not split16_in:
        b[bias_np.numel()] = 1.0
        return torch.cat((hi, lo), 0).contiguous(), b
    T, np_, cp = out.shape
    sw, wh, wl = _fp16_split(hi, lo)
    b2 = torch.zeros((T, np_, 2 * cp), dtype=torch.float16, device=out.device)
    for c0 in range(0, cp, 32):
        cl = min(32, cp - c0)
        b2[:, :, 2 * c0:2 * c0 + cl] = wh[:, :, c0:c0 + cl]
        b2[:, :, 2 * c0 + cl:2 * c0 + 2 * cl] = wl[:, :, c0:c0 + cl]
    b[bias_np.numel()] = torch.ldexp(torch.ones((), device=out.device), -(sw + 11))
    if split16_in:
        b[bias_np.numel() + 1] = torch.ldexp(torch.ones((), device=out.device), -sw)
        return b2.view(torch.float32).contiguous(), b
    return torch.cat((hi, b2.view(torch.float32)), 0).contiguous(), b


def pack_conv2d_tf32_weights(w, bias, cp, split=False, split16_in=False):
    """[Cout,Cin,3,3] (+ bias [Cout]) -> ([9][NP][cp] fp32, bias [NP]); NP = Cout rounded up to 16.
    split: [18][NP][cp] -- taps 0-8 the TF32 hi parts, 9-17 the correction operand (_pack_split_weights), bias [NP + 4].
    split16_in (with split): [9][NP][cp], the fp16 taps alone, for a layer whose input is stored as split16."""
    if split16_in and not split:
        raise ValueError("split16_in needs split=True")
    cout, cin = w.shape[:2]
    np_ = (cout + 15) // 16 * 16
    out = torch.zeros((9, np_, cp), dtype=torch.float32, device=w.device)
    out[:, :cout, :cin] = w.float().permute(2, 3, 0, 1).reshape(9, cout, cin)
    b = torch.zeros(np_, dtype=torch.float32, device=w.device)
    b[:cout] = bias.float()
    if split:
        out, b = _pack_split_weights(out, b, split16_in)
        return out, b, np_
    return rna_tf32(out).contiguous(), b.contiguous(), np_


def conv2d_tf32_nhwc(x_nhwc, w_packed, bias, relu, round_out=False):
    """x fp32 [B,H,W,cp] channels-last -> fp32 [B,H,W,NP] (round_out: outputs rounded to TF32 for a following tf32 conv)."""
    _chk("x_nhwc", x_nhwc)
    B, H, W, cp = x_nhwc.shape
    np_ = w_packed.shape[1]
    out = torch.empty((B, H, W, np_), dtype=torch.float32, device=x_nhwc.device)
    _call("decnet_conv2d_tf32_nhwc", x_nhwc, x_nhwc.data_ptr(), w_packed.data_ptr(), bias.data_ptr(), out.data_ptr(),
          B, H, W, cp, np_, 1 if relu else 0, 1 if round_out else 0)
    return out


# --------------------------------------------------------------------------------------
# small 3x3 Conv2d on NCHW fp32 tensors, TF32 tensor cores with pixels as the MN-major M dimension
# --------------------------------------------------------------------------------------
def conv2d_tf32_supported(cin, cout, H, W, dilation=1, split=False):
    return bool(_lib.lib().decnet_conv2d_tc_supported(int(cin), int(cout), int(H), int(W), int(dilation), _split_arg(split)))


def padded_cat_channels(src_channels):
    return sum((c + 7) // 8 * 8 for c in src_channels)


def _pad_cat_weights(w, src_channels, rows):
    """[Cout,Cin,3,3] -> fp32 [rows >= Cout, padded_cat_channels(src_channels), 3, 3], zero-filled: the input is a
    concatenation of tensors with these channel counts (sum = Cin), each padded to whole 8-channel chunks."""
    cout, cin = w.shape[:2]
    assert sum(src_channels) == cin, (src_channels, cin)
    wp = torch.zeros((rows, padded_cat_channels(src_channels), 3, 3), dtype=torch.float32, device=w.device)
    for j, c in enumerate(src_channels):
        o, i = padded_cat_channels(src_channels[:j]), sum(src_channels[:j])
        wp[:cout, o:o + c] = w[:, i:i + c].float()
    return wp


def pack_conv2d_tf32_nchw_weights(w, bias, src_channels=None, split=False):
    """[Cout,Cin,3,3] (+ bias [Cout]) -> (rows of 32 floats as include/decnet_b200.h describes, bias [CP]).
    src_channels: the input is a concatenation of tensors with these channel counts (sum = Cin), each
    padded to whole 8-channel chunks for decnet_conv2d_tc_nchw_cat.
    split: the hi rows followed by the lo rows (3xTF32 mode)."""
    cout = w.shape[0]
    wf = _pad_cat_weights(w, src_channels, cout) if src_channels is not None and len(src_channels) > 1 else w.float()
    cin = wf.shape[1]
    nck, cp = (cin + 7) // 8, (4 if cout <= 4 else (cout + 7) // 8 * 8)
    natoms = (3 * cp + 31) // 32
    # B[kh][ci][col = kw*CP + co]
    bm = torch.zeros((3, nck * 8, natoms * 32), dtype=torch.float32, device=w.device)
    for kw in range(3):
        bm[:, :cin, kw * cp: kw * cp + cout] = wf[:, :, :, kw].permute(2, 1, 0)       # [kh][ci][co]
    # -> [kh][chunk][atom][k][n]
    out = bm.view(3, nck, 8, natoms, 32).permute(0, 1, 3, 2, 4).contiguous()
    b = torch.zeros(cp + (4 if split else 0), dtype=torch.float32, device=w.device)
    b[:cout] = bias.float()
    if not split:
        out = rna_tf32(out)                                                            # cvt.rna to TF32
    elif SPLIT_KIND == 1:
        out = torch.cat(split_tf32(out), 0)
        b[cp] = 1.0
    else:
        out, b[cp] = _pack_nchw_split16(out)
    assert out.numel() == _lib.lib().decnet_conv2d_tc_packed_floats(int(cin), int(cout), _split_arg(split))
    return out.contiguous(), b.contiguous()


def _pack_nchw_split16(blocks):
    """blocks fp32 [kh][chunk][atom][8 k][32 n] -> (hi rows then fp16 correction rows, 2^-(11+sw)): split kind 2 of the thin
    NCHW kernel.  All three products of a pixel carry the factor S = 2^(11+sw): the TF32 hi rows hold hi(w) * S, and each 1 KB
    block of the second half is the MN-major SWIZZLE_64B fp16 operand [K atom 0: fp16(hi(w) * 2^sw) | K atom 1: fp16(lo(w) * S)],
    8 k x 32 n halves each, that meets [fp16(2^11 * lo(x)) | fp16(x)].  The rows are loaded by the same TMA map as the fp32
    rows (SWIZZLE_128B_ATOM_32B: 32-byte unit ^= bits 7-8 of the address), so the 16-byte units of a block are stored
    pre-permuted: unit g of the global block holds logical unit s64(s128a32(g)), s64 = 16-byte unit ^= bits 7-8."""
    hi, lo = split_tf32(blocks)
    sw, wh, wl = _fp16_split(hi, lo)
    kh, nck, natoms = blocks.shape[:3]
    logical = torch.stack((wh, wl), 3).contiguous()                                    # [kh][chunk][atom][2][8 k][32 n] halves
    units = logical.view(kh, nck, natoms, 64, 8)                                       # 64 sixteen-byte units per 1 KB block
    g = torch.arange(64, device=blocks.device)
    s1 = g ^ (((g >> 3) & 3) << 1)                                                     # s128a32: unit bits 1-2 ^= bits 3-4
    perm = s1 ^ ((s1 >> 3) & 3)                                                        # s64: unit bits 0-1 ^= bits 3-4
    packed = units[:, :, :, perm, :].contiguous().view(torch.float32).view(kh, nck, natoms, 8, 32)
    return torch.cat((torch.ldexp(hi, sw + 11), packed), 0), torch.ldexp(torch.ones((), device=blocks.device), -(sw + 11))


def conv2d_tf32_nchw(x, w_packed, bias_padded, cout, dilation=1, relu=False):
    _chk("x", x)
    B, cin, H, W = x.shape
    out = torch.empty((B, int(cout), H, W), dtype=torch.float32, device=x.device)
    _call("decnet_conv2d_tf32_nchw", x, x.data_ptr(), w_packed.data_ptr(), bias_padded.data_ptr(), out.data_ptr(),
          B, cin, int(cout), H, W, int(dilation), 1 if relu else 0)
    return out


def _cat_srcs(srcs):
    """The inputs of a convolution over torch.cat(srcs, 1): each [B,Ci,H,W] or [B,H,W] (one channel), on srcs[0]'s device
    -> (srcs[0], B, H, W, device pointer array, channel count array, n) as the *_cat entry points take them."""
    x0 = srcs[0]
    _chk("srcs[0]", x0)
    B, H, W = x0.shape[0], x0.shape[-2], x0.shape[-1]
    chans = []
    for i, t in enumerate(srcs):
        _chk(f"srcs[{i}]", t, x0)
        if (t.shape[0], t.shape[-2], t.shape[-1]) != (B, H, W):
            raise ValueError(f"srcs[{i}] {tuple(t.shape)} does not match srcs[0] {tuple(x0.shape)}")
        chans.append(1 if t.dim() == 3 else int(t.shape[1]))
    n = len(srcs)
    return x0, B, H, W, (ctypes.c_void_p * n)(*[t.data_ptr() for t in srcs]), (ctypes.c_int * n)(*chans), n


def conv2d_tf32_nchw_cat(srcs, w_packed, bias_padded, cout, dilation=1, relu=False, w_valid=0, split=False, addend=None):
    """Conv over torch.cat(srcs, 1) without building it; srcs: 1..3 tensors [B,Ci,H,W] or [B,H,W] (one channel).
    split: fp32-class operand split (w_packed from pack_conv2d_tf32_nchw_weights(split=True)).
    addend [B,H,W] (cout == 1): added after the activation in the epilogue."""
    x0, B, H, W, ptrs, cs, n = _cat_srcs(srcs)
    out = torch.empty((B, int(cout), H, W), dtype=torch.float32, device=x0.device)
    if addend is not None:
        _chk("addend", addend, x0, (B, H, W))
        if int(cout) != 1:
            raise ValueError("addend only for single-channel outputs")
    _call("decnet_conv2d_tc_nchw_cat_add", x0, ptrs, cs, n, w_packed.data_ptr(), bias_padded.data_ptr(),
          addend.data_ptr() if addend is not None else None, out.data_ptr(), B, int(cout), H, W, int(dilation),
          1 if relu else 0, int(w_valid), _split_arg(split))
    return out


def conv2d_tf32_rows_supported(cin_padded, cout, H, W, dilation=1):
    return bool(_lib.lib().decnet_conv2d_tf32_rows_supported(int(cin_padded), int(cout), int(H), int(W), int(dilation)))


def pack_conv2d_tf32_rows_weights(w, bias, src_channels=None):
    """[Cout<=8,Cin,3,3] (+ bias) -> (compact [3 kh][3 kw][nck][8 co][8 ci] fp32 TF32-rounded, bias [8]) for
    decnet_conv2d_tf32_rows_nchw_cat; every source of a concatenated input is padded to whole 8-channel chunks."""
    cout, cin = w.shape[:2]
    assert cout <= 8
    wf = _pad_cat_weights(w, tuple(src_channels) if src_channels else (cin,), 8)
    nck = wf.shape[1] // 8
    out = rna_tf32(wf.view(8, nck, 8, 3, 3).permute(3, 4, 1, 0, 2))             # [kh][kw][ck][co][ci]
    b = torch.zeros(8, dtype=torch.float32, device=w.device)
    b[:cout] = bias.float()
    return out.contiguous(), b.contiguous()


def conv2d_tf32_rows_nchw_cat(srcs, w_compact, bias8, cout, dilation=1, relu=False):
    x0, B, H, W, ptrs, cs, n = _cat_srcs(srcs)
    out = torch.empty((B, int(cout), H, W), dtype=torch.float32, device=x0.device)
    _call("decnet_conv2d_tf32_rows_nchw_cat", x0, ptrs, cs, n, w_compact.data_ptr(), bias8.data_ptr(), out.data_ptr(),
          B, int(cout), H, W, int(dilation), 1 if relu else 0)
    return out


def _nhwc_format(round_tf32, split16):
    """The storage-format argument of the channels-last writers: 0 fp32, 1 fp32 rounded to TF32, 2 split16."""
    return 2 if split16 else (1 if round_tf32 else 0)


def _nhwc_empty(B, h, w, cp, split16, device):
    """[B,h,w,cp] fp32, or its split16 form: the same bytes as fp16 [B,h,w,2*cp] (the dtype tells the formats apart)."""
    if split16:
        return torch.empty((B, h, w, 2 * cp), dtype=torch.float16, device=device)
    return torch.empty((B, h, w, cp), dtype=torch.float32, device=device)


def conv2d_tf32_nhwc_halo(x_pad, w_packed, bias, relu, round_out=False, split=False, split16_out=False):
    """x fp32 [B,h+2,w+2,cp] channels-last with a zero border -> fp32 [B,h+2,w+2,NP] (border zeros).
    split: 3xTF32 -- x unrounded fp32, w_packed [18][NP][cp] from pack_conv2d_tf32_weights(split=True).
    x fp16 [B,h+2,w+2,2*cp] is split16 storage (common.cuh: split16_store; needs split, w_packed [9][NP][cp] from
    split16_in=True, cp % 16 == 0).  split16_out: the output stored as split16 too, fp16 [B,h+2,w+2,2*NP]."""
    _chk("x_pad", x_pad, split16_ok=True)
    B, hp, wp, cp = x_pad.shape
    np_ = w_packed.shape[1]
    split16_in = x_pad.dtype == torch.float16
    if split16_in:
        cp //= 2
        if not split:
            raise ValueError("split16 input needs split=True")
    if w_packed.shape[0] != (18 if split and not split16_in else 9) or w_packed.shape[2] != cp:
        raise ValueError(f"w_packed {tuple(w_packed.shape)} does not match cp={cp}, split={split}, split16 input={split16_in}")
    out = _nhwc_empty(B, hp, wp, np_, split16_out, x_pad.device)
    _call("decnet_conv2d_tc_nhwc_halo", x_pad, x_pad.data_ptr(), w_packed.data_ptr(), bias.data_ptr(), out.data_ptr(),
          B, hp - 2, wp - 2, cp, np_, 1 if relu else 0, _nhwc_format(round_out, split16_out),
          3 if split16_in else _split_arg(split))
    return out


def nchw_cat_to_nhwc_pad(srcs, cp, round_tf32=True, split16=False):
    """cat(srcs, 1) (NCHW, single-channel maps as [B,H,W]) -> zero-bordered channels-last [B,H+2,W+2,cp]
    (round_tf32: values rounded to TF32 for the halo kernel's plain-TF32 mode; its 3xTF32 mode takes them unrounded;
    split16: stored as split16, fp16 [B,H+2,W+2,2*cp], for its split16-input mode)."""
    x0, B, H, W, ptrs, cs, n = _cat_srcs(srcs)
    out = _nhwc_empty(B, H + 2, W + 2, int(cp), split16, x0.device)
    _call("decnet_nchw_cat_to_nhwc_pad", x0, ptrs, cs, n, out.data_ptr(), B, H, W, int(cp), _nhwc_format(round_tf32, split16))
    return out


def nhwc_pad_to_nchw(x_pad, channels):
    _chk("x_pad", x_pad)
    B, hp, wp, np_ = x_pad.shape
    out = torch.empty((B, int(channels), hp - 2, wp - 2), dtype=torch.float32, device=x_pad.device)
    _call("decnet_nhwc_pad_to_nchw", x_pad, x_pad.data_ptr(), out.data_ptr(), B, int(channels), np_, hp - 2, wp - 2)
    return out


def dynup_pack_nhwc(disp, left_fea, cp, round_tf32=True, pad=False, split16=False):
    """pad=True: [B,h+2,w+2,cp] with a zero border (the layout conv2d_tf32_nhwc_halo chains on).
    disp=None: only the feature channels (channel 0 zero) -- dynup_set_disp_nhwc() completes it later.
    split16: stored as split16, fp16 [B,h(+2),w(+2),2*cp]."""
    _chk("left_fea", left_fea)
    B, Cc, H3, W3 = left_fea.shape
    if H3 % 3 or W3 % 3:
        raise ValueError(f"left_fea {tuple(left_fea.shape)} is not 3x a coarse grid")
    h, w = H3 // 3, W3 // 3
    if disp is not None:
        _chk("disp", disp, left_fea)
        if tuple(disp.shape) != (B, h, w):
            raise ValueError(f"left_fea {tuple(left_fea.shape)} is not 3x the disparity map {tuple(disp.shape)}")
    k = 2 if pad else 0
    out = _nhwc_empty(B, h + k, w + k, int(cp), split16, left_fea.device)
    _call("decnet_dynup_pack_nhwc", left_fea, disp.data_ptr() if disp is not None else None, left_fea.data_ptr(),
          out.data_ptr(), B, Cc, h, w, int(cp), _nhwc_format(round_tf32, split16), 1 if pad else 0)
    return out


def dynup_set_disp_nhwc(packed, disp, round_tf32=True, pad=False):
    """Writes channel 0 (the disparity) of a tensor packed with disp=None, in place, in the tensor's format (fp16: split16,
    round_tf32 ignored); returns it."""
    _chk("disp", disp)
    B, h, w = disp.shape
    _chk("packed", packed, disp, split16_ok=True)
    k = 2 if pad else 0
    if tuple(packed.shape[:3]) != (B, h + k, w + k):
        raise ValueError(f"packed {tuple(packed.shape)} does not match disp {tuple(disp.shape)} (pad={pad})")
    split16 = packed.dtype == torch.float16
    _call("decnet_dynup_set_disp_nhwc", disp, disp.data_ptr(), packed.data_ptr(), B, h, w,
          packed.shape[-1] // (2 if split16 else 1), _nhwc_format(round_tf32, split16), 1 if pad else 0)
    return packed


def dynup_glue_nhwc(logits_nhwc, disp, pad=False):
    _chk("disp", disp)
    B, h, w = disp.shape
    _chk("logits", logits_nhwc, disp)
    k = 2 if pad else 0
    if tuple(logits_nhwc.shape[:3]) != (B, h + k, w + k):
        raise ValueError(f"logits {tuple(logits_nhwc.shape)} do not match disp {tuple(disp.shape)} (pad={pad})")
    NP = logits_nhwc.shape[-1]
    out = torch.empty((B, 3 * h, 3 * w), dtype=torch.float32, device=disp.device)
    _call("decnet_dynup_glue_nhwc", disp, logits_nhwc.data_ptr(), disp.data_ptr(), out.data_ptr(), B, h, w, NP,
          1 if pad else 0)
    return out


# --------------------------------------------------------------------------------------
# feature extractor on the tensor-core GEMM (SURVEY.md section 8f rank 2): GEMM mode of the halo kernel + data movement
# --------------------------------------------------------------------------------------
def pack_gemm_weights(w2d, bias, cp, split=False, n0=0, n1=None):
    """[N, K] (+ bias [N]) rows n0..n1 -> ([1 or 2][NP][cp] fp32, bias [NP]), NP = (n1 - n0) rounded up to 16, K zero-padded to
    cp; split: the TF32 hi parts then the lo parts (3xTF32)."""
    n1 = w2d.shape[0] if n1 is None else n1
    n, k = n1 - n0, w2d.shape[1]
    np_ = (n + 15) // 16 * 16
    out = torch.zeros((1, np_, cp), dtype=torch.float32, device=w2d.device)
    out[0, :n, :k] = w2d[n0:n1].float()
    b = torch.zeros(np_, dtype=torch.float32, device=w2d.device)
    b[:n] = bias[n0:n1].float()
    if split:
        out, b = _pack_split_weights(out, b)
        return out, b, np_
    return rna_tf32(out).contiguous(), b.contiguous(), np_


def gemm_tc(x, w_packed, bias, out, relu, split=False, col=0, border=None, dst_hw=None):
    """out[:, col:col+NP] = act(x @ w^T + bias) on the tensor cores.  x [..., cp] rows (all leading dims flattened), out rows of
    out.shape[-1] floats.  border=(B,h,w): x and out are zero-bordered [B,h+2,w+2,.] tensors, border rows stay zero;
    dst_hw=(h,w): x is a flat [B*h*w, cp] grid, out a zero-bordered [B,h+2,w+2,.] tensor (interior written)."""
    _chk("x", x)
    _chk("out", out, x)
    cp, ldc, np_ = x.shape[-1], out.shape[-1], w_packed.shape[1]
    P = x.numel() // cp
    if w_packed.shape[0] != (2 if split else 1) or w_packed.shape[2] != cp:
        raise ValueError(f"w_packed {tuple(w_packed.shape)} does not match cp={cp}, split={split}")
    if col % 4 or col + np_ > ldc:
        raise ValueError(f"column slice [{col}, {col + np_}) does not fit rows of {ldc}")
    bB, bh, bw = border if border is not None else (0, 0, 0)
    dh, dw = dst_hw if dst_hw is not None else (0, 0)
    rows_out = out.numel() // ldc
    want = P if dst_hw is None else (P // (dh * dw)) * (dh + 2) * (dw + 2)
    if rows_out != want:
        raise ValueError(f"out has {rows_out} rows, expected {want}")
    _call("decnet_gemm_tc_nhwc", x, x.data_ptr(), w_packed.data_ptr(), bias.data_ptr(), out.data_ptr() + 4 * col, P, cp, np_, ldc,
          1 if relu else 0, _split_arg(split), bB, bh, bw, dh, dw)
    return out


def conv2d_nhwc_halo_into(x_pad, w_packed, bias, out_pad, relu, split=False, col=0):
    """3x3 conv on the zero-bordered layout writing channels [col, col+NP) of the wider bordered tensor out_pad."""
    _chk("x_pad", x_pad)
    _chk("out_pad", out_pad, x_pad)
    B, hp, wp, cp = x_pad.shape
    np_, ldc = w_packed.shape[1], out_pad.shape[-1]
    if tuple(out_pad.shape[:3]) != (B, hp, wp) or col % 4 or col + np_ > ldc:
        raise ValueError(f"out_pad {tuple(out_pad.shape)} / col {col} do not fit x_pad {tuple(x_pad.shape)}, NP {np_}")
    _call("decnet_conv2d_tc_nhwc_halo_ldc", x_pad, x_pad.data_ptr(), w_packed.data_ptr(), bias.data_ptr(),
          out_pad.data_ptr() + 4 * col, B, hp - 2, wp - 2, cp, np_, ldc, 1 if relu else 0, _split_arg(split))
    return out_pad


def im2col3x3(src, layout, C, stride=1, dilation=1, kp=None):
    """3x3 windows (zero padding = dilation) as GEMM rows [B*Ho*Wo, kp], column tap*C + c.
    layout: "nchw" [B,C,H,W]; "nhwc" flat [B,H,W,ld]; "nhwc_pad" zero-bordered [B,H+2,W+2,ld] (its interior is the grid)."""
    _chk("src", src)
    if layout == "nchw":
        B, _, H, W = src.shape
        sb, sc, sy, sx, off = src.shape[1] * H * W, H * W, W, 1, 0
    elif layout == "nhwc":
        B, H, W, ld = src.shape
        sb, sc, sy, sx, off = H * W * ld, 1, W * ld, ld, 0
    elif layout == "nhwc_pad":
        B, hp, wp, ld = src.shape
        H, W = hp - 2, wp - 2
        sb, sc, sy, sx, off = hp * wp * ld, 1, wp * ld, ld, (wp + 1) * ld
    else:
        raise ValueError(layout)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1                # k 3, pad = dilation = 1 for the strided convs
    kp = (9 * C + 7) // 8 * 8 if kp is None else kp
    out = torch.empty((B * Ho * Wo, kp), dtype=torch.float32, device=src.device)
    _call("decnet_im2col3x3", src, src.data_ptr() + 4 * off, out.data_ptr(), B, int(C), H, W, sb, sc, sy, sx, int(stride),
          int(dilation), Ho, Wo, kp)
    return out, Ho, Wo


def deconv3x3s3_shuffle(x, out_pad, B, h, w, cout, col=0):
    """GEMM-form ConvTranspose2d(k3, s3) result [B*h*w, ld] (column tap*cout + co) -> interior of out_pad [B,3h+2,3w+2,ldc]."""
    _chk("x", x)
    _chk("out_pad", out_pad, x, (B, 3 * h + 2, 3 * w + 2, out_pad.shape[-1]))
    _call("decnet_deconv3x3s3_shuffle", x, x.data_ptr(), out_pad.data_ptr(), B, h, w, int(cout), x.shape[-1], out_pad.shape[-1], int(col))
    return out_pad


def nhwc_to_nchw(x, B, C, h, w, pad=False):
    """Channels-last rows of x.shape[-1] floats (pad: zero-bordered [B,h+2,w+2,ld]) -> NCHW [B,C,h,w]."""
    _chk("x", x)
    out = torch.empty((B, int(C), h, w), dtype=torch.float32, device=x.device)
    _call("decnet_nhwc_to_nchw", x, x.data_ptr(), out.data_ptr(), B, int(C), x.shape[-1], h, w, 1 if pad else 0)
    return out


def conv3x3s3_nchw(x, w, bias, relu=True):
    """Conv2d(3x3, stride 3, pad 1) + bias [+ ReLU] on NCHW, direct fp32 (w [24,Cin,3,3], BN folded)."""
    _chk("x", x)
    B, cin, H, W = x.shape
    cout = w.shape[0]
    wpk = w.float().permute(1, 2, 3, 0).reshape(cin, 9, cout).contiguous()
    out = torch.empty((B, cout, (H - 1) // 3 + 1, (W - 1) // 3 + 1), dtype=torch.float32, device=x.device)
    _call("decnet_conv3x3s3_nchw", x, x.data_ptr(), wpk.data_ptr(), bias.float().contiguous().data_ptr(), out.data_ptr(), B, cin, H, W,
          cout, 1 if relu else 0)
    return out
