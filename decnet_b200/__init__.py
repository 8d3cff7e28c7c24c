"""decnet_b200 -- Blackwell-native (sm_100a) implementation of DecNet's decomposed-matching
hot path behind the reference's module API.  See DESIGN.md / INTEGRATION.md."""
from . import _lib  # noqa: F401  (does not load the .so until first use)
from .modules import SpaMat, SpaMatFunction, SpaVar, SpaVarFunction
from .predictor import StereoMatcher

__all__ = ["SpaMat", "SpaMatFunction", "SpaVar", "SpaVarFunction", "StereoMatcher"]
__version__ = "0.1.0"
