"""oracle/ref_loader.py -- TEST INFRASTRUCTURE.  Imports the UNMODIFIED reference package from the original DecNet
project's source tree (source(): $DECNET_REFERENCE, else BASELINE.json's reference_path) or from baseline/_ref (the
git-ignored copy __graft_entry__.build() stages from that tree so that it travels with the repository tree to a GPU
machine): stubs the missing matplotlib / visdom modules (utils/utils.py:8, eval.py:10) and registers
`modules.Sparse{Matching,Var}.build.lib` with an extension object of the caller's choice
(the CPU oracle by default) so `from ..build.lib import SpaMat` resolves
(modules/SparseMatching/functions/SpaMat.py:4).
"""
from __future__ import annotations

import json
import os
import sys
import types
from pathlib import Path

_ROOT = Path(__file__).resolve().parents[1]
STAGED = _ROOT / "baseline" / "_ref"


def _is_tree(p: Path) -> bool:
    try:
        return (p / "modules" / "submodule.py").exists()
    except OSError:                         # a location this user may not read (another user's home) counts as absent
        return False


def source() -> Path | None:
    """The original project's source tree, when this machine has one: $DECNET_REFERENCE, else BASELINE.json's
    reference_path."""
    cands = [Path(os.environ["DECNET_REFERENCE"])] if os.environ.get("DECNET_REFERENCE") else []
    try:
        cands.append(Path(json.loads((_ROOT / "BASELINE.json").read_text())["reference_path"]))
    except (OSError, KeyError, ValueError):
        pass
    return next((p for p in cands if _is_tree(p)), None)


REF = source() or STAGED


class _OracleSpaMatExt:
    """CPU stand-in with the pybind module's surface (SM_cuda.cpp:7-35)."""

    @staticmethod
    def sparse_matching_cuda_forward(L, R, ml, mr, out, ssim, mx, D):
        from . import sparse as osp
        o, s, m = osp.spamat_forward(L, R, ml, mr, D)
        out.copy_(o); ssim.copy_(s); mx.copy_(m)
        return 1

    @staticmethod
    def sparse_matching_cuda_backward(L, R, ml, mr, out, ssim, mx, g, dL, dR, D):
        from . import sparse as osp
        a, b = osp.spamat_backward(L, R, ml, mr, out, ssim, mx, g, D)
        dL.copy_(a); dR.copy_(b)
        return 1


class _OracleSpaVarExt:
    @staticmethod
    def sparse_var_cuda_forward(L, R, ml, mr, disp, out, ssim, mx, D):
        from . import sparse as osp
        o, s, m = osp.spavar_forward(L, R, ml, mr, disp, D)
        out.copy_(o); ssim.copy_(s); mx.copy_(m)
        return 1

    @staticmethod
    def sparse_var_cuda_backward(L, R, ml, mr, disp, out, ssim, mx, g, dL, dR, dd, D):
        from . import sparse as osp
        a, b, c = osp.spavar_backward(L, R, ml, mr, disp, out, ssim, mx, g, D)
        dL.copy_(a); dR.copy_(b); dd.copy_(c)
        return 1


def available() -> bool:
    return _is_tree(REF)


def install(spamat_ext=None, spavar_ext=None):
    """Make `import modules` (the reference package) work; returns the imported package."""
    if not available():
        raise RuntimeError("the original DecNet source tree was found neither at $DECNET_REFERENCE / BASELINE.json's "
                           "reference_path nor staged at baseline/_ref (run __graft_entry__.build() where it is present)")
    for m in ("matplotlib", "matplotlib.pyplot", "visdom"):
        if m not in sys.modules:
            sys.modules[m] = types.ModuleType(m)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    for pkg, name, ext in (("SparseMatching", "SpaMat", spamat_ext or _OracleSpaMatExt()),
                           ("SparseVar", "SpaVar", spavar_ext or _OracleSpaVarExt())):
        b = types.ModuleType(f"modules.{pkg}.build")
        l = types.ModuleType(f"modules.{pkg}.build.lib")
        setattr(l, name, ext)
        b.lib = l
        sys.modules[f"modules.{pkg}.build"] = b
        sys.modules[f"modules.{pkg}.build.lib"] = l
    if str(REF) not in sys.path:
        sys.path.insert(0, str(REF))
    import modules  # noqa: F401  (the reference package)
    return modules


def build_reference_model(max_disp=216, use_detail=True, thold=0.9, skip_stage_id=4, verbose=False):
    """The shipped configuration (demo.sh:1): 4 stages, down_scale 3, base_channels 8, cost 'cor'."""
    import contextlib
    import io
    mods = install()
    from modules.sync_batchnorm import convert_model
    ctx = contextlib.nullcontext() if verbose else contextlib.redirect_stdout(io.StringIO())
    with ctx:
        model = mods.get_model(name="SparseDenseNetRefinementMask", max_disp=max_disp, base_channels=8,
                               cost_func="cor", num_stage=4, down_scale=3, step=[1, 1, 1, 1],
                               samp_num=[8, 8, 8, 8], sample_spa_size_list=[-1, 3, 3, 3],
                               down_func_name="bilinear", weights=[1, 1, 1, 1], grad_method="detach",
                               if_overmask=False, skip_stage_id=skip_stage_id, use_detail=use_detail,
                               thold=thold)
        model = convert_model(model)
    return model.eval()
