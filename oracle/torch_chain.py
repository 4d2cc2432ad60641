"""The reference's torch-GPU execution path, restated for A/B timing -- TEST / BENCH INFRASTRUCTURE ONLY.

The "reference torch-GPU path" that BASELINE.json asks the fused kernels to beat is re-expressed here, so that
the project can time it without the reference installed, as the same chain of unfused ATen ops the reference
issues per Linear call (dequant.py:30-44 -> dequantize_blocks_* -> `.to(dtype)` -> F.linear, ops.py:242-244),
including its per-call creation of the small shift tensors on the device.  tests/test_torch_chain.py pins this
file against outputs of the unmodified reference stored under tests/golden/ (bit-equal outputs AND the same
number of materialising ATen kernels).  Nothing in the product package imports it.

Types covered: the ones the BASELINE configs use on the GPU A/B (Q4_K, Q5_K, Q6_K, Q8_0, Q4_0, BF16).
"""
from __future__ import annotations

import torch

QK = 256


def _fields(blocks, *sizes):
    rest = blocks.shape[1] - sum(sizes)
    return torch.split(blocks, list(sizes) + [rest], dim=1)


def _shifts(vals, device, shape):
    # the reference builds these from Python lists on every call (dequant.py:121, 148-150, 171-172, 189)
    return torch.tensor(vals, device=device, dtype=torch.uint8).reshape(shape)


def _six_bit_pairs(sbytes):
    """dequant.py:129-139: 12 bytes -> eight 6-bit scales and eight 6-bit mins."""
    n = sbytes.shape[0]
    s = sbytes.view(torch.uint8).reshape((n, 3, 4))
    lo, mid, hi = torch.split(s, 1, dim=-2)
    sc = torch.cat([lo & 0x3F, (hi & 0x0F) | ((lo >> 2) & 0x30)], dim=-1)
    mn = torch.cat([mid & 0x3F, (hi >> 4) | ((mid >> 2) & 0x30)], dim=-1)
    return sc.reshape((n, 8)), mn.reshape((n, 8))


def chain_q8_0(blocks, dtype=None):      # dequant.py:65-69
    d, x = _fields(blocks, 2)
    return d.view(torch.float16).to(dtype) * x.view(torch.int8)


def chain_q4_0(blocks, dtype=None):      # dequant.py:115-123
    n = blocks.shape[0]
    d, qs = _fields(blocks, 2)
    d = d.view(torch.float16).to(dtype)
    q = qs.reshape((n, -1, 1, 16)) >> _shifts([0, 4], d.device, (1, 1, 2, 1))
    q = (q & 0x0F).reshape((n, -1)).to(torch.int8) - 8
    return d * q


def chain_q4_k(blocks, dtype=None):      # dequant.py:180-195
    n = blocks.shape[0]
    d, dmin, sbytes, qs = _fields(blocks, 2, 2, 12)
    d = d.view(torch.float16).to(dtype)
    dmin = dmin.view(torch.float16).to(dtype)
    sc, mn = _six_bit_pairs(sbytes)
    dl = (d * sc).reshape((n, -1, 1))
    ml = (dmin * mn).reshape((n, -1, 1))
    q = qs.reshape((n, -1, 1, 32)) >> _shifts([0, 4], d.device, (1, 1, 2, 1))
    q = (q & 0x0F).reshape((n, -1, 32))
    return (dl * q - ml).reshape((n, QK))


def chain_q5_k(blocks, dtype=None):      # dequant.py:159-178
    n = blocks.shape[0]
    d, dmin, sbytes, qh, qs = _fields(blocks, 2, 2, 12, QK // 8)
    d = d.view(torch.float16).to(dtype)
    dmin = dmin.view(torch.float16).to(dtype)
    sc, mn = _six_bit_pairs(sbytes)
    dl = (d * sc).reshape((n, -1, 1))
    ml = (dmin * mn).reshape((n, -1, 1))
    lo = qs.reshape((n, -1, 1, 32)) >> _shifts([0, 4], d.device, (1, 1, 2, 1))
    hi = qh.reshape((n, -1, 1, 32)) >> _shifts(list(range(8)), d.device, (1, 1, 8, 1))
    lo = (lo & 0x0F).reshape((n, -1, 32))
    hi = (hi & 0x01).reshape((n, -1, 32))
    q = lo | (hi << 4)
    return (dl * q - ml).reshape((n, QK))


def chain_q6_k(blocks, dtype=None):      # dequant.py:141-157
    n = blocks.shape[0]
    ql, qh, sc, d = _fields(blocks, QK // 2, QK // 4, QK // 16)
    sc = sc.view(torch.int8).to(dtype)
    d = d.view(torch.float16).to(dtype)
    dl = (d * sc).reshape((n, QK // 16, 1))
    lo = ql.reshape((n, -1, 1, 64)) >> _shifts([0, 4], d.device, (1, 1, 2, 1))
    lo = (lo & 0x0F).reshape((n, -1, 32))
    hi = qh.reshape((n, -1, 1, 32)) >> _shifts([0, 2, 4, 6], d.device, (1, 1, 4, 1))
    hi = (hi & 0x03).reshape((n, -1, 32))
    q = (lo | (hi << 4)).to(torch.int8) - 32
    q = q.reshape((n, QK // 16, -1))
    return (dl * q).reshape((n, QK))


def chain_bf16(blocks, dtype=None):      # dequant.py:61-62
    return (blocks.view(torch.int16).to(torch.int32) << 16).view(torch.float32)


_CHAINS = {8: (chain_q8_0, 32, 34), 2: (chain_q4_0, 32, 18), 12: (chain_q4_k, 256, 144), 13: (chain_q5_k, 256, 176),
           14: (chain_q6_k, 256, 210), 30: (chain_bf16, 1, 2)}


def dequantize(data, qtype, oshape, dtype=None):
    """dequant.py:30-44."""
    fn, _bs, ts = _CHAINS[int(qtype)]
    rows = data.reshape((-1, data.shape[-1])).view(torch.uint8)
    n_blocks = rows.numel() // ts
    return fn(rows.reshape((n_blocks, ts)), dtype).reshape(oshape)


def dequantize_tensor(data, qtype, oshape, dtype=None, dequant_dtype=None):
    """dequant.py:15-28 for a quantised tensor."""
    math = dtype if dequant_dtype == "target" else dequant_dtype
    return dequantize(data, qtype, oshape, dtype=math).to(dtype)


def linear(x, data, qtype, oshape, bias=None, dequant_dtype=None):
    """ops.py:242-244 + 193-211: dequant chain -> cast to x.dtype -> F.linear (cuBLAS)."""
    b = None if bias is None else bias.to(x.dtype)
    w = dequantize_tensor(data, qtype, oshape, x.dtype, dequant_dtype)
    return torch.nn.functional.linear(x, w, b)
