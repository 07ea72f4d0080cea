"""CPU: the argument checks of sow_adam_multi_amp (rejected before any device work), FusedAdamW's state_dtype validation and
its load_state_dict dtype policy, and the TrainConfig combinations loss scaling refuses."""
import copy
import ctypes

import pytest
import torch
import torch.nn as nn

from sow_b200 import _lib
from sow_b200._lib import SOWB_BF16, SOWB_F16, SOWB_F32, SowB200Error

SOWB_EINVAL = -1


def _amp(dtype=SOWB_BF16, state_dtype=SOWB_F32, bc1=0.1, bc2=0.001, step_dev=None, grad_scale=None, found_inf=None):
    """One call with a dummy (never dereferenced) chunk table: every rejected combination must return before any device
    work, so no GPU is needed."""
    lib = _lib.load()
    return lib.sow_adam_multi_amp(ctypes.c_void_p(0x1000), 1, 8, 1e-3, 0.9, 0.999, 1e-8, 0.0, bc1, bc2, step_dev,
                                  grad_scale, found_inf, 1, dtype, state_dtype, None)


@pytest.mark.parametrize("kw", [
    dict(dtype=7),                                        # unknown parameter dtype
    dict(state_dtype=7),                                  # unknown state dtype
    dict(dtype=SOWB_F32, state_dtype=SOWB_BF16),          # 16-bit state for fp32 parameters
    dict(dtype=SOWB_F32, state_dtype=SOWB_F16),
    dict(dtype=SOWB_BF16, state_dtype=SOWB_F16),          # neither the parameter dtype nor fp32
    dict(found_inf=ctypes.c_void_p(0x2000)),              # found_inf without the device step counter
    dict(bc1=0.0),                                        # host bias corrections must be positive
    dict(bc2=-1.0),
])
def test_adam_multi_amp_rejects_bad_arguments_without_a_device(kw):
    assert _amp(**kw) == SOWB_EINVAL
    assert _lib.load().sow_last_error().decode().startswith("sow_adam_multi_amp")


def test_state_dtype_validation():
    from sow_b200.optim import FusedAdamW

    def P(dt):
        return nn.Parameter(torch.zeros(4, dtype=dt))

    for pdt in (torch.float16, torch.bfloat16):
        FusedAdamW([P(pdt)], state_dtype=torch.float32)
        FusedAdamW([P(pdt)], state_dtype=pdt)
        FusedAdamW([{"params": [P(pdt)], "state_dtype": torch.float32}])
    FusedAdamW([P(torch.float32)], state_dtype=torch.float32)
    bad = [(torch.float32, torch.bfloat16), (torch.float32, torch.float16), (torch.bfloat16, torch.float16),
           (torch.float16, torch.bfloat16), (torch.float16, torch.float64), (torch.bfloat16, "float32")]
    for pdt, sdt in bad:
        with pytest.raises(SowB200Error, match="state_dtype"):
            FusedAdamW([P(pdt)], state_dtype=sdt)
    opt = FusedAdamW([P(torch.float16)])
    with pytest.raises(SowB200Error, match="state_dtype"):
        opt.add_param_group({"params": [P(torch.float32)], "state_dtype": torch.float16})


def test_load_state_dict_keeps_fp32_moments_of_state_dtype_groups():
    """torch's policy casts floating-point state to the parameter dtype; groups with state_dtype keep it, bit for bit."""
    from sow_b200.optim import FusedAdamW
    gen = torch.Generator().manual_seed(0)

    def make():
        a, b = nn.Parameter(torch.zeros(5, 3, dtype=torch.float16)), nn.Parameter(torch.zeros(7, dtype=torch.float16))
        return [a, b], FusedAdamW([{"params": [a], "state_dtype": torch.float32}, {"params": [b]}])

    (a, b), opt = make()
    for p in (a, b):
        opt.state[p] = {"step": torch.tensor(3.0), "exp_avg": torch.randn(p.shape, generator=gen) * 1e-6,
                        "exp_avg_sq": torch.rand(p.shape, generator=gen) * 1e-9}
    sd = copy.deepcopy(opt.state_dict())
    assert sd["param_groups"][0]["state_dtype"] == torch.float32 and sd["param_groups"][1]["state_dtype"] is None
    (a2, b2), fresh = make()
    fresh.load_state_dict(sd)
    for k in ("exp_avg", "exp_avg_sq"):
        got = fresh.state[a2][k]
        assert got.dtype == torch.float32
        assert torch.equal(got.view(torch.int32), opt.state[a][k].view(torch.int32))
        assert fresh.state[b2][k].dtype == torch.float16                      # torch's policy for the other group
    assert float(fresh.state[a2]["step"]) == 3.0


@pytest.mark.parametrize("kw", [dict(fused_optimizer=False), dict(grad_clipping=1.0), dict(dtype=torch.bfloat16)])
def test_loss_scaling_rejects_unsupported_combinations(kw):
    """Raised at the top of SoWTrainer.__init__, before any model is built (the model name does not even exist)."""
    from sow_b200.trainer import SoWTrainer, TrainConfig
    cfg = TrainConfig(model="no_such_model", loss_scaling=True, **{"dtype": torch.float16, **kw})
    with pytest.raises(ValueError, match="loss_scaling"):
        SoWTrainer(cfg, torch.device("cpu"))
