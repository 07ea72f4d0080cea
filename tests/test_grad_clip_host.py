"""CPU: the argument checks of the gradient-clipping entry points (rejected before any device work), FusedAdamW's
max_grad_norm validation and checkpoint handling, and the TrainConfig combinations fused clipping allows or refuses."""
import copy
import ctypes
import math

import pytest
import torch
import torch.nn as nn

from sow_b200 import _lib
from sow_b200._lib import SOWB_BF16, SOWB_F16, SOWB_F32, SowB200Error

SOWB_EINVAL = -1
TABLE, PARTIALS, SCALAR = ctypes.c_void_p(0x1000), ctypes.c_void_p(0x2000), ctypes.c_void_p(0x3000)


def _partials(chunks=TABLE, n_chunks=1, dtype=SOWB_BF16, grad_scale=None, partials=PARTIALS):
    return _lib.load().sow_grad_norm_partials(chunks, n_chunks, dtype, grad_scale, partials, None)


def _finalize(partials=PARTIALS, n_partials=4, max_norm=1.0, total_norm=SCALAR, clip_coef=SCALAR):
    return _lib.load().sow_grad_norm_finalize(partials, n_partials, max_norm, total_norm, clip_coef, None)


def _clip(n_chunks=1, dtype=SOWB_BF16, state_dtype=SOWB_F32, bc1=0.1, bc2=0.001, step_dev=None, found_inf=None,
          clip_coef=SCALAR):
    return _lib.load().sow_adam_multi_clip(TABLE, n_chunks, 8, 1e-3, 0.9, 0.999, 1e-8, 0.0, bc1, bc2, step_dev, None,
                                           found_inf, clip_coef, 1, dtype, state_dtype, None)


@pytest.mark.parametrize("fn,kw", [
    (_partials, dict(dtype=7)),                           # unknown dtype
    (_partials, dict(n_chunks=-1)),
    (_partials, dict(chunks=None)),                       # null chunk table with rows
    (_partials, dict(partials=None)),
    (_partials, dict(n_chunks=0, partials=None)),
    (_finalize, dict(n_partials=0)),
    (_finalize, dict(n_partials=-3)),
    (_finalize, dict(partials=None)),
    (_finalize, dict(total_norm=None)),
    (_finalize, dict(clip_coef=None)),
    (_finalize, dict(max_norm=0.0)),
    (_finalize, dict(max_norm=-1.0)),
    (_finalize, dict(max_norm=math.inf)),
    (_finalize, dict(max_norm=math.nan)),
    (_clip, dict(clip_coef=None)),                        # the coefficient is required
    (_clip, dict(n_chunks=-1)),
    (_clip, dict(dtype=7)),
    (_clip, dict(state_dtype=7)),
    (_clip, dict(dtype=SOWB_F32, state_dtype=SOWB_BF16)),  # the combinations sow_adam_multi_amp rejects
    (_clip, dict(dtype=SOWB_F32, state_dtype=SOWB_F16)),
    (_clip, dict(dtype=SOWB_BF16, state_dtype=SOWB_F16)),
    (_clip, dict(found_inf=ctypes.c_void_p(0x4000))),      # found_inf without the device step counter
    (_clip, dict(bc1=0.0)),
    (_clip, dict(bc2=-1.0)),
], ids=lambda v: getattr(v, "__name__", None) or ",".join(f"{k}={v[k]}" for k in v))
def test_clip_entry_points_reject_bad_arguments_without_a_device(fn, kw):
    assert fn(**kw) == SOWB_EINVAL
    name = {_partials: "sow_grad_norm_partials", _finalize: "sow_grad_norm_finalize", _clip: "sow_adam_multi_clip"}[fn]
    assert _lib.load().sow_last_error().decode().startswith(name)


def test_empty_partials_call_is_a_no_op():
    assert _partials(chunks=None, n_chunks=0) == 0


def test_max_grad_norm_validation():
    from sow_b200.optim import FusedAdamW
    p = nn.Parameter(torch.zeros(4))
    for ok in (None, 1.0, 1e-8, 3, 1e30):
        opt = FusedAdamW([p], max_grad_norm=ok)
        assert opt.param_groups[0]["max_grad_norm"] == ok
    FusedAdamW([{"params": [p], "max_grad_norm": 0.5}])
    for bad in (0.0, -1.0, math.inf, -math.inf, math.nan, True, "1.0", torch.tensor(1.0)):
        with pytest.raises(SowB200Error, match="max_grad_norm"):
            FusedAdamW([p], max_grad_norm=bad)
    opt = FusedAdamW([p])
    with pytest.raises(SowB200Error, match="max_grad_norm"):
        opt.add_param_group({"params": [nn.Parameter(torch.zeros(2))], "max_grad_norm": -2.0})
    assert opt.grad_norm(0) is None                        # no clipped step yet


def _two_group_optimizer():
    from sow_b200.optim import FusedAdamW
    a, b = nn.Parameter(torch.zeros(5, 3)), nn.Parameter(torch.zeros(7))
    return [a, b], FusedAdamW([{"params": [a], "max_grad_norm": 0.25}, {"params": [b]}], lr=1e-3)


def test_state_dict_round_trip_keeps_max_grad_norm():
    _, opt = _two_group_optimizer()
    sd = copy.deepcopy(opt.state_dict())
    assert sd["param_groups"][0]["max_grad_norm"] == 0.25 and sd["param_groups"][1]["max_grad_norm"] is None
    _, fresh = _two_group_optimizer()
    fresh.param_groups[0]["max_grad_norm"] = 9.0
    fresh.load_state_dict(sd)
    assert fresh.param_groups[0]["max_grad_norm"] == 0.25 and fresh.param_groups[1]["max_grad_norm"] is None


def test_checkpoint_without_the_key_loads_unclipped():
    """A state_dict written before max_grad_norm existed has no such key: the loaded groups read as unclipped."""
    from sow_b200.optim import _check_max_grad_norm
    _, opt = _two_group_optimizer()
    sd = copy.deepcopy(opt.state_dict())
    for g in sd["param_groups"]:
        del g["max_grad_norm"]
    _, fresh = _two_group_optimizer()
    fresh.load_state_dict(sd)
    for g in fresh.param_groups:
        assert _check_max_grad_norm(g.get("max_grad_norm")) is None


def test_fused_grad_clipping_needs_the_fused_optimizer():
    from sow_b200.trainer import SoWTrainer, TrainConfig
    cfg = TrainConfig(model="no_such_model", fused_optimizer=False, fused_grad_clipping=True, grad_clipping=1.0)
    with pytest.raises(ValueError, match="fused_grad_clipping"):
        SoWTrainer(cfg, torch.device("cpu"))


def test_loss_scaling_with_fused_grad_clipping_passes_the_configuration_checks():
    """The checks run at the top of SoWTrainer.__init__; with fused clipping, loss scaling + clipping gets past them and
    fails only when the (non-existent) model is built.  Without the flag the combination is still refused."""
    from sow_b200.trainer import SoWTrainer, TrainConfig
    kw = dict(model="no_such_model", dtype=torch.float16, loss_scaling=True, grad_clipping=1.0)
    with pytest.raises(KeyError, match="no_such_model"):
        SoWTrainer(TrainConfig(fused_grad_clipping=True, **kw), torch.device("cpu"))
    with pytest.raises(ValueError, match="loss_scaling"):
        SoWTrainer(TrainConfig(**kw), torch.device("cpu"))
