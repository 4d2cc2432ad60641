"""Drop-in for the reference's dequant.py: same public names, B200 kernels underneath.

Reference surface mirrored (file:line in city96/ComfyUI-GGUF):
    is_torch_compatible / is_quantized       dequant.py:9-13
    dequantize_tensor(tensor, dtype, dequant_dtype)   dequant.py:15-28
    dequantize(data, qtype, oshape, dtype)   dequant.py:30-44
    dequantize_functions                     dequant.py:287-301 (keys = supported types)

Every dequantisation is ONE launch of csrc/dequant.cu through the C ABI.  The result is
bit-identical to the reference for each (math dtype, output dtype) pair because the kernel
reproduces the reference's per-op rounding (see csrc/common.cuh).  There is no numpy / CPU
fallback (dequant.py:24-28 is intentionally not reproduced): unsupported types raise.
"""
from __future__ import annotations

import gguf
import torch

from . import _lib

TORCH_COMPATIBLE_QTYPES = (None, gguf.GGMLQuantizationType.F32, gguf.GGMLQuantizationType.F16)

_DT_CODE = {torch.float16: _lib.F16, torch.bfloat16: _lib.BF16, torch.float32: _lib.F32}
_Q = gguf.GGMLQuantizationType
SUPPORTED_QTYPES = (_Q.BF16, _Q.Q8_0, _Q.Q5_1, _Q.Q5_0, _Q.Q4_1, _Q.Q4_0, _Q.Q6_K, _Q.Q5_K, _Q.Q4_K, _Q.Q3_K, _Q.Q2_K,
                    _Q.IQ4_NL, _Q.IQ4_XS)


def is_torch_compatible(tensor):
    return tensor is None or getattr(tensor, "tensor_type", None) in TORCH_COMPATIBLE_QTYPES


def is_quantized(tensor):
    return not is_torch_compatible(tensor)


def dtype_code(dtype) -> int:
    try:
        return _DT_CODE[dtype]
    except KeyError:
        raise TypeError(f"ggufb200: unsupported dtype {dtype!r} (float16 / bfloat16 / float32 only)") from None


def math_code(dequant_dtype, target_dtype) -> int:
    """dequant.py:22 semantics: None -> fp16 math, "target" -> the requested dtype, else the explicit dtype."""
    if dequant_dtype is None:
        return _lib.F16
    if isinstance(dequant_dtype, str):
        if dequant_dtype != "target":
            raise ValueError(f"bad dequant_dtype {dequant_dtype!r}")
        return _lib.F16 if target_dtype is None else dtype_code(target_dtype)
    return dtype_code(dequant_dtype)


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _require_cuda(what: str):
    if not torch.cuda.is_available():
        raise _lib.GGUFB200Error(f"{what}: no CUDA device is visible and this package has no CPU fallback")


def _as_bytes(data: torch.Tensor) -> torch.Tensor:
    """Plain contiguous uint8 view of the packed payload (drops any tensor subclass)."""
    raw = data.as_subclass(torch.Tensor) if type(data) is not torch.Tensor else data
    if raw.dtype != torch.uint8:
        raw = raw.contiguous().view(torch.uint8)
    return raw.contiguous()


# The packed bytes handed to dequantize() are produced by loads, host-to-device copies or ordinary torch kernels, none of which
# signals programmatic launch completion before its last write -- so they are complete before our kernel starts and the
# GGUFB200_DEQUANT_SRC_STABLE promise (include/ggufb200.h) holds by construction.  Set to False to launch without it.
SRC_STABLE = True


def dequantize(data, qtype, oshape, dtype=None, out_dtype=None, src_stable=None):
    """dequant.py:30-44.  `dtype` is the MATH dtype (None = fp16); the result is in `out_dtype`
    (default: the math dtype, as in the reference where the block functions return it).
    BF16 always yields fp32 in the reference (dequant.py:61-62) unless out_dtype says otherwise."""
    qtype = gguf.GGMLQuantizationType(qtype)
    if qtype not in dequantize_functions:
        raise NotImplementedError(f"ggufb200: no kernel for qtype {getattr(qtype, 'name', qtype)!r} (and no CPU fallback)")
    block_size, type_size = gguf.GGML_QUANT_SIZES[qtype]
    math = _lib.F16 if dtype is None else dtype_code(dtype)
    if SRC_STABLE if src_stable is None else src_stable:
        math |= _lib.DEQUANT_SRC_STABLE
    if out_dtype is None:
        out_dtype = torch.float32 if qtype == _Q.BF16 else (torch.float16 if dtype is None else dtype)
    raw = _as_bytes(data)
    src_device = raw.device
    if raw.device.type != "cuda":
        _require_cuda("dequantize")
        raw = raw.to("cuda", non_blocking=False)
    n_bytes = raw.numel()
    if n_bytes % type_size != 0:
        raise ValueError(f"packed size {n_bytes} is not a multiple of the {qtype.name} block size {type_size}")
    n_blocks = n_bytes // type_size
    out = torch.empty(n_blocks * block_size, dtype=out_dtype, device=raw.device)
    with torch.cuda.device(raw.device):
        rc = _lib.lib().ggufb200_dequant(int(qtype), raw.data_ptr(), n_blocks, out.data_ptr(), dtype_code(out_dtype), math,
                                         _stream_ptr(raw.device))
    _lib.check(rc, f"ggufb200_dequant({qtype.name})")
    out = out.reshape(oshape)
    if src_device.type != "cuda":
        out = out.to(src_device)
    return out


def dequantize_tensor(tensor, dtype=None, dequant_dtype=None):
    """dequant.py:15-28 with the final `.to(dtype)` folded into the kernel."""
    qtype = getattr(tensor, "tensor_type", None)
    oshape = getattr(tensor, "tensor_shape", tensor.shape)
    if qtype in TORCH_COMPATIBLE_QTYPES:
        return tensor.to(dtype)
    if qtype not in dequantize_functions:
        raise NotImplementedError(
            f"ggufb200: qtype {getattr(qtype, 'name', repr(qtype))} is not supported; the reference's numpy fallback "
            "(dequant.py:24-28) is deliberately not provided")
    math_dt = dtype if dequant_dtype == "target" else dequant_dtype
    if dtype is None:
        out_dtype = None
    else:
        out_dtype = dtype
    return dequantize(tensor.data, qtype, oshape, dtype=math_dt, out_dtype=out_dtype)


def unpack_int(data, qtype):
    """Integer unpack (q, sc, mn) of every element -- the bit-exact integer contract, for tests."""
    qtype = gguf.GGMLQuantizationType(qtype)
    block_size, type_size = gguf.GGML_QUANT_SIZES[qtype]
    raw = _as_bytes(data)
    if raw.device.type != "cuda":
        _require_cuda("unpack_int")
        raw = raw.to("cuda")
    n_blocks = raw.numel() // type_size
    outs = [torch.empty(n_blocks * block_size, dtype=torch.int16, device=raw.device) for _ in range(3)]
    with torch.cuda.device(raw.device):
        rc = _lib.lib().ggufb200_unpack_int(int(qtype), raw.data_ptr(), n_blocks, outs[0].data_ptr(), outs[1].data_ptr(),
                                            outs[2].data_ptr(), _stream_ptr(raw.device))
    _lib.check(rc, f"ggufb200_unpack_int({qtype.name})")
    return tuple(outs)


def dequantize_rows(tensor, rows, dtype=None, dequant_dtype=None):
    """out[i] = dequant(W[rows[i]]): the gather the Embedding path needs, without touching other rows."""
    qtype = tensor.tensor_type
    shape = tuple(tensor.tensor_shape)
    n_table, K = shape[0], shape[-1]
    raw = _as_bytes(tensor.data)
    if raw.device.type != "cuda":
        _require_cuda("dequantize_rows")
        raw = raw.to("cuda")
    rows = rows.to(device=raw.device, dtype=torch.int64).contiguous()
    out_dtype = torch.float16 if dtype is None else dtype
    if qtype == _Q.BF16 and dtype is None:
        out_dtype = torch.float32
    math_dt = dtype if dequant_dtype == "target" else dequant_dtype
    out = torch.empty(rows.numel(), K, dtype=out_dtype, device=raw.device)
    with torch.cuda.device(raw.device):
        rc = _lib.lib().ggufb200_dequant_rows(int(qtype), raw.data_ptr(), n_table, K, rows.data_ptr(), rows.numel(), out.data_ptr(),
                                              dtype_code(out_dtype), math_code(math_dt, dtype), _stream_ptr(raw.device))
    _lib.check(rc, f"ggufb200_dequant_rows({qtype.name})")
    return out.reshape(*rows.shape, K)


def _make_entry(qtype):
    def run(blocks, block_size, type_size, dtype=None):
        n_blocks = blocks.numel() // type_size
        return dequantize(blocks, qtype, (n_blocks, block_size), dtype=dtype)
    run.__name__ = f"dequantize_blocks_{qtype.name}"
    return run


# same keys as the reference's table (dequant.py:287-301); values keep the (blocks, block_size, type_size, dtype) signature
dequantize_functions = {q: _make_entry(q) for q in SUPPORTED_QTYPES}
