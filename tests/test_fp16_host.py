"""CPU: the float16 dtype code of the C ABI and its Python mapping; the tensor-train wrappers keep bf16 / fp32 only."""
import os
import re

import pytest
import torch

from conftest import ROOT
from sow_b200 import _lib, ops
from sow_b200._lib import SowB200Error


def test_fp16_dtype_code_matches_the_header():
    with open(os.path.join(ROOT, "include", "sow_b200.h")) as f:
        header = f.read()
    m = re.search(r"#define SOWB_F16 (\d+)", header)
    assert m and int(m.group(1)) == 2 == _lib.SOWB_F16
    assert ops._dtype_code(torch.float16) == 2
    assert ops._dtype_code(torch.bfloat16) == _lib.SOWB_BF16 and ops._dtype_code(torch.float32) == _lib.SOWB_F32


def test_tensor_train_wrappers_reject_fp16():
    assert ops._tt_dtype_code(torch.bfloat16) == _lib.SOWB_BF16
    assert ops._tt_dtype_code(torch.float32) == _lib.SOWB_F32
    with pytest.raises(SowB200Error):
        ops._tt_dtype_code(torch.float16)
