"""Generate tests/golden/detail_masks.npz from the UNMODIFIED reference function utils.utils.detailDetection
(build container only; needs cv2).  Inputs are regenerated from the seed by make_detail_image().

    python tests/golden/make_golden_detail.py
"""
import sys
import types
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

SEED, H, W = 41, 108, 162


def make_detail_image(seed=SEED, H=H, W=W):
    """Piecewise-smooth synthetic image in [0,1], float64 like `padding(img) / 255` in demo.py:158."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    img = np.zeros((H, W, 3))
    for c in range(3):
        img[..., c] = 0.5 + 0.25 * np.sin(xx / (7.0 + c)) * np.cos(yy / (5.0 + 2 * c))
    for _ in range(12):                      # rectangles: sharp edges = "lost details"
        y0, x0 = rng.integers(0, H - 10), rng.integers(0, W - 10)
        h, w = rng.integers(4, 30), rng.integers(4, 40)
        img[y0:y0 + h, x0:x0 + w] = rng.random(3)
    img += 0.02 * rng.standard_normal(img.shape)
    return np.clip(np.round(img * 255), 0, 255) / 255


if __name__ == "__main__":
    for m in ("matplotlib", "matplotlib.pyplot", "visdom"):
        sys.modules.setdefault(m, types.ModuleType(m))
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    from oracle import ref_loader
    sys.path.insert(0, str(ref_loader.REF))         # the original project's tree (oracle/ref_loader.py)
    from utils.utils import detailDetection          # the reference function itself (utils/utils.py:483-534)
    out = {"meta": np.array([SEED, H, W], dtype=np.int64)}
    for b, seed in enumerate((SEED, SEED + 1)):
        masks = detailDetection(make_detail_image(seed), scale=3, downsampling_iteration=3, name="g", thold=0.3)
        for i, m in enumerate(masks):
            out[f"mask{b}_{i}"] = np.packbits(m)
            out[f"shape{b}_{i}"] = np.array(m.shape, dtype=np.int64)
        print(seed, [round(float(m.mean()), 4) for m in masks])
    path = Path(__file__).resolve().parent / "detail_masks.npz"
    np.savez_compressed(path, **out)
    print("->", path, path.stat().st_size, "bytes")
