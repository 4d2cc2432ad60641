"""CPU test: oracle/torch_chain.py reproduces the reference's torch path bit-for-bit and with the same number of
materialising ATen kernels, so that timing it on the GPU is a fair stand-in for the reference.  What the unmodified
reference's dequant.py::dequantize gives on the same seeded blocks is stored in tests/golden/torch_chain_reference.json
(tests/golden/make_golden.py)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch
import gguf
from torch.utils._python_dispatch import TorchDispatchMode

import oracle
from oracle import torch_chain

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "torch_chain_reference.json")
Q = gguf.GGMLQuantizationType
QTYPES = [Q.Q8_0, Q.Q4_0, Q.Q4_K, Q.Q5_K, Q.Q6_K, Q.BF16]
MATH_DTYPES = [None, torch.float32, torch.bfloat16]


class Count(TorchDispatchMode):
    VIEWS = ("view", "reshape", "split", "unsqueeze", "expand", "_unsafe_view", "alias", "detach", "select", "slice", "squeeze",
             "permute", "transpose", "t.default", "split_with_sizes", "_reshape_alias", "lift_fresh")

    def __init__(self):
        super().__init__()
        self.n = 0

    def __torch_dispatch__(self, func, types, args=(), kwargs=None):
        name = str(func)
        if not any(v in name for v in self.VIEWS):
            self.n += 1
        return func(*args, **(kwargs or {}))


def case_id(qt, md):
    return f"{qt.name}-{'default' if md is None else str(md).replace('torch.', '')}"


def inputs(qt):
    bs, ts = gguf.GGML_QUANT_SIZES[qt]
    return torch.from_numpy(oracle.random_blocks(int(qt), 96, seed=1)).reshape(-1), (96 * bs,)


def output_bits(t):
    """The elements of a dequantised tensor as unsigned integers of their width (bit patterns)."""
    b = t.contiguous().view(torch.uint8).numpy()
    return b.view({2: np.uint16, 4: np.uint32}[t.element_size()])


@pytest.mark.parametrize("qt", QTYPES, ids=lambda q: q.name)
@pytest.mark.parametrize("md", MATH_DTYPES)
def test_chain_equals_reference(qt, md):
    want = json.load(open(GOLDEN))[case_id(qt, md)]
    raw, shape = inputs(qt)
    with Count() as c_mine:
        b = torch_chain.dequantize(raw, qt, shape, dtype=md)
    assert str(b.dtype) == want["dtype"] and list(b.shape) == want["shape"]
    bits = output_bits(b)
    idx = np.array(want["sample_index"])
    assert bits[idx].tolist() == want["sample_bits"]
    assert hashlib.sha256(bits.tobytes()).hexdigest() == want["sha256"]
    assert c_mine.n == want["aten_kernels"], (c_mine.n, want["aten_kernels"])
