"""StereoMatcher's host-side logic without a GPU: input validation, max_disp rounding, the checkpoint split and its
strictness, the graph cache key."""
import numpy as np
import pytest
import torch

from decnet_b200.predictor import cache_key, check_pair, round_max_disp, split_state_dict


def _u8(*shape):
    return np.zeros(shape, dtype=np.uint8)


def test_valid_inputs():
    assert check_pair(_u8(5, 7, 3), _u8(5, 7, 3)) == ("numpy", False, 1, 5, 7)
    t = torch.zeros((2, 9, 4, 3), dtype=torch.uint8)
    assert check_pair(t, t.clone()) == ("cpu", True, 2, 9, 4)


@pytest.mark.parametrize("left, right, what", [
    (_u8(5, 7, 3).astype(np.float32), _u8(5, 7, 3).astype(np.float32), "uint8"),
    (_u8(5, 7, 4), _u8(5, 7, 4), "RGB"),
    (_u8(5, 7), _u8(5, 7), "RGB"),
    (_u8(5, 7, 3), _u8(5, 8, 3), "differ"),
    (_u8(5, 7, 3), torch.zeros((5, 7, 3), dtype=torch.uint8), "same kind"),
    (_u8(0, 7, 3), _u8(0, 7, 3), "at least 1x1"),
    (_u8(0, 5, 7, 3), _u8(0, 5, 7, 3), "at least one pair"),
    ([[1, 2, 3]], [[1, 2, 3]], "numpy arrays or torch tensors"),
    (torch.zeros((5, 7, 3), dtype=torch.int16), torch.zeros((5, 7, 3), dtype=torch.int16), "uint8"),
])
def test_bad_inputs_raise_before_device_work(left, right, what, monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("validation touched CUDA")
    monkeypatch.setattr(torch.cuda, "current_stream", no_cuda)
    monkeypatch.setattr(torch.cuda, "synchronize", no_cuda)
    with pytest.raises(ValueError, match=what):
        check_pair(left, right)


def test_max_disp_rounding():
    assert round_max_disp(192) == 216
    assert round_max_disp(216) == 216
    assert round_max_disp(768) == 783
    assert round_max_disp(1) == 27
    for bad in (0, -27, 1.5, True, "192"):
        with pytest.raises(ValueError):
            round_max_disp(bad)


@pytest.fixture(scope="module")
def modules():
    from decnet_b200.features import FeatExtNetChannelPlus
    from decnet_b200.model import DecompMatching
    return FeatExtNetChannelPlus(8), DecompMatching()


def _reference_layout(prefix):
    from decnet_b200.params import make_featext_state, make_hotpath_state
    sd = {f"{prefix}feature_extractor.{k}": v for k, v in make_featext_state(3).items()}
    sd.update({prefix + k: v for k, v in make_hotpath_state(3).items()})
    return sd


@pytest.mark.parametrize("prefix", ["", "module."])
def test_checkpoint_split(modules, prefix):
    fe, model = modules
    fe_sd, hot_sd = split_state_dict(_reference_layout(prefix), fe.state_dict().keys(), model.state_dict().keys())
    assert set(fe_sd) == set(fe.state_dict()) and set(hot_sd) == set(model.state_dict())
    fe.load_state_dict(fe_sd, strict=True)
    model.load_state_dict(hot_sd, strict=True)
    assert torch.equal(fe.conv0[0].conv.weight, _reference_layout("")["feature_extractor.conv0.0.conv.weight"])


def test_checkpoint_strict(modules):
    fe, model = modules
    keys = fe.state_dict().keys(), model.state_dict().keys()
    sd = _reference_layout("module.")
    extra = dict(sd, **{"module.refinement.0.conv.9.conv.weight": torch.zeros(1)})
    with pytest.raises(ValueError, match=r"refinement\.0\.conv\.9\.conv\.weight"):
        split_state_dict(extra, *keys)
    missing = dict(sd)
    del missing["module.feature_extractor.deconv3.conv.1.bn.running_var"]
    with pytest.raises(ValueError, match=r"feature_extractor\.deconv3\.conv\.1\.bn\.running_var"):
        split_state_dict(missing, *keys)
    missing = dict(sd)
    del missing["module.cost_regularizer.conv0.0.conv.weight"]
    with pytest.raises(ValueError, match=r"cost_regularizer\.conv0\.0\.conv\.weight"):
        split_state_dict(missing, *keys)


def test_cache_key():
    k = cache_key(8, 540, 960, 216, "learned", "fp32")
    assert k == (8, 540, 960, 216, "learned", "fp32")
    others = [cache_key(4, 540, 960, 216, "learned", "fp32"), cache_key(8, 541, 960, 216, "learned", "fp32"),
              cache_key(8, 540, 961, 216, "learned", "fp32"), cache_key(8, 540, 960, 243, "learned", "fp32"),
              cache_key(8, 540, 960, 216, "image", "fp32"), cache_key(8, 540, 960, 216, "learned", "tf32")]
    assert len({k, *others}) == 7
