"""CPU: host-side logic of the tn_gradient mirror -- model surgery, state-dict wire format, legacy call forms,
compat TT algebra -- without any device compute."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err
from oracle import sow_oracle as O


class MLP(nn.Module):
    def __init__(self):
        super().__init__()
        self.fc1 = nn.Linear(24, 40, bias=True)
        self.fc2 = nn.Linear(40, 16, bias=False)
        self.head = nn.Linear(16, 4)

    def forward(self, x):
        return self.head(self.fc2(torch.tanh(self.fc1(x))))


def test_prepare_sow_replaces_targets_and_keeps_wire_format(golden_loop):
    from tn_gradient.layer.sow import SoWLinear
    from tn_gradient.prepare import SoWConfig, prepare_sow
    torch.manual_seed(0)
    model = MLP()
    w1 = model.fc1.weight.detach().clone()
    bias1 = model.fc1.bias
    cfg = SoWConfig(target_modules=["fc1", "fc2"], rank=4, scale=0.5, device="cpu", init_method="normal", decompose="keep")
    out = prepare_sow(model, cfg)
    assert out is model
    assert isinstance(model.fc1, SoWLinear) and isinstance(model.fc2, SoWLinear) and isinstance(model.head, nn.Linear)
    assert model.fc1.bias is bias1                                    # original Parameter reused (prepare.py:155-156)
    assert model.fc1.virtual_rank == 24 and model.fc2.virtual_rank == 16
    assert model.fc1.scale == 0.5 and model.fc1.rank == 4 and model.fc1.n_iter == 1
    assert torch.equal(model.fc1.acc_downweight, w1.T)                # (in, out) layout, prepare.py:150
    assert not model.fc1.acc_downweight.requires_grad and model.fc1.acc_upweight.numel() == 0
    assert model.fc1.downscale_weights[0].shape == (24, 4) and model.fc1.upscale_weights[0].shape == (4, 40)
    keys = sorted(k for k in model.state_dict().keys() if not k.startswith("head"))
    assert keys == sorted(golden_loop["loop/keep/state_dict_keys"].tolist())


def test_prepare_sow_pretraining_mode_has_empty_accumulation():
    from tn_gradient.prepare import SoWConfig, prepare_sow
    model = prepare_sow(MLP(), SoWConfig(target_modules=["fc1"], rank=2, init_method="normal", decompose=None))
    assert model.fc1.acc_downweight.numel() == 0 and model.fc1.acc_upweight.numel() == 0
    assert isinstance(model.fc2, nn.Linear)


def test_legacy_run_glue_call_form():
    """scripts/run_glue.py:54,564,574: SoWArgs + prepare_sow(model, target_modules, decompose=, args=)."""
    from tn_gradient.layer.sow import SoWArgs, SoWLinear
    from tn_gradient.prepare import prepare_sow
    args = SoWArgs(rank=3, n_iter=1, device="cpu", dtype=None, scale=0.25, init_method="normal")
    model = prepare_sow(MLP(), ["fc2"], decompose="keep", args=args)
    assert isinstance(model.fc2, SoWLinear) and model.fc2.rank == 3 and model.fc2.scale == 0.25


def test_dotted_target_names_match_by_suffix():
    from tn_gradient.layer.sow import SoWLinear
    from tn_gradient.prepare import SoWConfig, prepare_sow

    class Block(nn.Module):
        def __init__(self):
            super().__init__()
            self.attention = nn.ModuleDict({"output": nn.ModuleDict({"dense": nn.Linear(8, 8)})})
            self.output = nn.ModuleDict({"dense": nn.Linear(8, 8)})

    m = nn.ModuleDict({"layer0": Block()})
    prepare_sow(m, SoWConfig(target_modules=["attention.output.dense"], rank=2, init_method="normal", decompose="keep"))
    assert isinstance(m["layer0"].attention["output"]["dense"], SoWLinear)
    assert isinstance(m["layer0"].output["dense"], nn.Linear)


def test_forward_on_cpu_raises_instead_of_falling_back():
    from sow_b200 import SowB200Error
    from tn_gradient.layer.sow import SoWLinear
    layer = SoWLinear(16, 24, rank=4, init_method="normal")
    with pytest.raises(SowB200Error, match="no CPU fallback"):
        layer(torch.randn(2, 16))
    with pytest.raises(SowB200Error):
        layer.accumulate()


def test_sow_parameter_from_weights_keeps_identity():
    from tn_gradient.layer.sow import SoWParameter
    p = SoWParameter(6, 3, n_iter=2)
    ids = [id(x) for x in p]
    new = [torch.ones(6, 3), torch.zeros(6, 3)]
    p.from_weights(new)
    assert [id(x) for x in p] == ids
    assert torch.equal(p[0].data, new[0]) and torch.equal(p[1].data, new[1])
    assert "2 x (6, 3)" in p.extra_repr()


def test_load_sow_grows_empty_accumulation(tmp_path):
    from safetensors.torch import save_file
    from tn_gradient.prepare import SoWConfig, load_sow, prepare_sow
    torch.manual_seed(1)
    src = prepare_sow(MLP(), SoWConfig(target_modules=["fc1", "fc2"], rank=2, init_method="normal", decompose="keep"))
    path = str(tmp_path / "model.safetensors")
    save_file({k: v.contiguous() for k, v in src.state_dict().items() if v.numel()}, path)
    dst = prepare_sow(MLP(), SoWConfig(target_modules=["fc1", "fc2"], rank=2, init_method="normal", decompose=None))
    assert dst.fc1.acc_downweight.numel() == 0
    load_sow(dst, path)
    assert torch.equal(dst.fc1.acc_downweight, src.fc1.acc_downweight)
    assert not dst.fc1.acc_downweight.requires_grad
    assert torch.equal(dst.fc2.downscale_weights[0], src.fc2.downscale_weights[0])


def test_utils_match_reference_conventions():
    from tn_gradient.utils import closest_factorization, pad_matrix, unpad_matrix
    assert closest_factorization(81, 4) == ([3, 3, 3, 3], 81)
    m = torch.arange(6.0).reshape(2, 3)
    p = pad_matrix(m.to(torch.bfloat16), (4, 4))
    assert p.dtype == torch.float32 and p.shape == (4, 4) and float(p[3, 3]) == 0.0     # utils.py:82: default dtype
    assert torch.equal(unpad_matrix(p, (2, 3)), m)


def test_tt_compat_algebra_matches_reference(golden_tt):
    """+, *, scalar *, add_, round, norm on CPU cores (plain PyTorch compat path) vs the reference's outputs;
    reconstruction of the resulting cores is done by the oracle (TensorTrain.reconstruct itself is CUDA-only)."""
    from tn_gradient.tt import TensorTrain
    g = golden_tt
    cores = [torch.from_numpy(g[f"tt/arange/core{i}"]) for i in range(3)]
    tt = TensorTrain.from_cores(cores)
    assert tt.ranks == [1, 4, 4, 1] and tt.order == 3

    def rec(t):
        return O.tt_reconstruct([c.numpy() for c in t.cores])

    s = tt + tt
    assert s.ranks == list(g["tt/arange/add_ranks"])
    assert rel_err(rec(s), g["tt/arange/add_rec"]) < 1e-6
    p = tt * tt
    assert p.ranks == list(g["tt/arange/mul_ranks"])
    assert rel_err(rec(p), g["tt/arange/mul_rec"]) < 1e-6
    assert rel_err(rec((tt * tt).round([1, 4, 4, 1])), g["tt/arange/mul_round_rec"]) < 1e-5
    assert rel_err(rec(2.5 * tt), g["tt/arange/scaled_rec"]) < 1e-6
    assert rel_err(rec(tt.add_(-3)), g["tt/arange/addc_rec"]) < 1e-6
    assert abs(tt.norm() - float(g["tt/arange/norm"])) <= 2.0
    d = tt - tt
    assert float(np.abs(rec(d)).max()) < 1e-3


def test_colorized_str_runs():
    from tn_gradient.utils import __colorized_str__
    s = __colorized_str__(MLP())
    assert "fc1" in s and "trainable" in s


@pytest.mark.parametrize("rank,n_iter,fits", [(128, 4, False), (384, 1, False), (320, 1, True), (128, 2, True)])
def test_shared_input_group_runs_members_alone_above_the_group_rank_limit(rank, n_iter, fits):
    """One group call takes a concatenated padded rank of at most ops.MAX_GROUP_RANK = 1024; a wider q/k/v group must run
    its members one by one instead of failing."""
    from sow_b200 import ops
    from sow_b200.layer import SharedInputGroup, SoWLinear
    ms = [SoWLinear(64, 64, rank=rank, n_iter=n_iter, init_method="normal") for _ in range(3)]
    grp = SharedInputGroup(ms)
    assert ops.MAX_GROUP_RANK == 1024
    assert grp.usable() == fits
    assert grp.usable_traced() == (fits and n_iter == 1)
