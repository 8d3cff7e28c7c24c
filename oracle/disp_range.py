"""oracle/disp_range.py -- TEST INFRASTRUCTURE ONLY.  numpy definition of StereoMatcher's search range [min_disp, max_disp),
which has no counterpart in the reference; decnet_image_prepare_u8_shift and StereoMatcher(min_disp=...) are held to it.

For a pair (L, R) and k = min_disp the matcher runs the unchanged model, at max_disp = the range's width D, on
(L, shift_cols_u8(R, k)), and adds k to its padded prediction in float32 (one rounded add).  With the left-right check
the reverse direction is (mirror(R), shift_cols_u8(mirror(L), k)), plus k as well; the check, the fills and the speckle
filter then run unchanged on those predictions, the guided fill along the unshifted left image.

  shift_cols_u8     image column x takes the input's column x - k; columns whose source lies outside [0, w) are black (0)
  disparity_range   (min_disp, D): D = max_disp - min_disp rounded up to a multiple of 27 (demo.py:172-173)
"""
import numpy as np

MULTIPLE = 27
LIMIT = 2 ** 24                # beyond it an integer offset is no longer exact in float32


def shift_cols_u8(img, k):
    """uint8 [..., h, w, 3] -> the same shape with out[..., :, x, :] = img[..., :, x - k, :] where 0 <= x - k < w, else 0."""
    img = np.asarray(img)
    if img.dtype != np.uint8 or img.ndim < 3 or img.shape[-1] != 3:
        raise ValueError(f"img must be uint8 [..., h, w, 3], got {img.dtype} {img.shape}")
    k = int(k)
    w = img.shape[-2]
    out = np.zeros_like(img)
    if 0 <= k < w:
        out[..., k:, :] = img[..., :w - k, :]
    elif -w < k < 0:
        out[..., :w + k, :] = img[..., -k:, :]
    return out


def disparity_range(min_disp, max_disp):
    """The searched range of StereoMatcher(min_disp=min_disp, max_disp=max_disp) as (min_disp, D): it covers
    [min_disp, min_disp + D) with D the width max_disp - min_disp rounded up to a multiple of 27.  Both ends must be
    integers (not bools) in [-2**24, 2**24] with max_disp > min_disp, else ValueError."""
    for name, v in (("min_disp", min_disp), ("max_disp", max_disp)):
        if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer)):
            raise ValueError(f"{name} must be an integer, got {v!r}")
        if not -LIMIT <= v <= LIMIT:
            raise ValueError(f"{name} must lie in [-2**24, 2**24], got {v!r}")
    if max_disp <= min_disp:
        raise ValueError(f"max_disp must be larger than min_disp, got [{min_disp}, {max_disp})")
    width = int(max_disp) - int(min_disp)
    return int(min_disp), (width + MULTIPLE - 1) // MULTIPLE * MULTIPLE
