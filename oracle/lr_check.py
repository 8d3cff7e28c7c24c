"""oracle/lr_check.py -- TEST INFRASTRUCTURE ONLY.  numpy float32 definition of StereoMatcher's left-right consistency check,
which has no counterpart in the reference; decnet_lr_check (decnet_b200/csrc/codec.cu) is held to it bit for bit.

  lr_check        forward vs. mirrored reverse prediction: u = floor((x - dl) + 0.5), valid = isfinite(dl) & (0 <= u < w)
                  & (|dl - dr[u]| <= tol); outputs dl / demo.py's uint16 value where valid, 0 elsewhere, and the mask
"""
import numpy as np

from .codec import disp_to_u16


def lr_check(fwd_padded, rev_padded, ori_h, ori_w, tol):
    """Left-right consistency check of the padded [B,H,W] forward prediction against the padded prediction of the mirrored,
    swapped pairs (left view mirror(R), right view mirror(L)), both cropped like demo.py (the last ori_h rows / ori_w
    columns); the reverse crop is mirrored back.  In float32 throughout, pixel (b, y, x) with dl = forward, dr = reverse:
        u = floor((x - dl) + 0.5);  valid = isfinite(dl) & (0 <= u < ori_w) & (|dl - dr[b, y, int(u)]| <= tol)
    -> (float: dl where valid else 0, uint16: disp_to_u16's value where valid else 0, valid: bool), each [B,ori_h,ori_w]."""
    dl = np.asarray(fwd_padded, dtype=np.float32)[:, -ori_h:, -ori_w:]
    dr = np.asarray(rev_padded, dtype=np.float32)[:, -ori_h:, -ori_w:][:, :, ::-1]
    x = np.arange(ori_w, dtype=np.float32)[None, None, :]
    with np.errstate(invalid="ignore", over="ignore"):
        u = np.floor((x - dl) + np.float32(0.5))
        inside = np.isfinite(dl) & (u >= 0) & (u < ori_w)
        ui = np.where(inside, u, 0).astype(np.int64)
        back = np.take_along_axis(dr, ui, axis=2)
        valid = inside & (np.abs(dl - back) <= np.float32(tol))
    f = np.where(valid, dl, np.float32(0)).astype(np.float32)
    return f, disp_to_u16(f, ori_h, ori_w), valid
