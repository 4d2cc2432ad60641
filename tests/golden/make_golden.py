#!/usr/bin/env python
"""Generate the committed golden vectors from the UNMODIFIED reference.

Needs a checkout of the original ComfyUI-GGUF (city96/ComfyUI-GGUF, commit
795e45156ece) and runs on the CPU:

    python tests/golden/make_golden.py REFERENCE_DIR [dequant|linear|torch_chain|surface ...]

(default: all four groups; a group rewrites only its own files)

What is produced (all under tests/golden/):
  dequant_<QTYPE>.npz   seeded packed blocks + the reference's own outputs of
                        `dequant.py::dequantize(...).to(out)` for five
                        (math dtype, out dtype) combinations, as raw bit patterns
  linear_<QTYPE>_<act>.npz   x / packed W / F32 bias and the output of the
                        reference `ops.py::GGMLOps.Linear.forward` (run on CPU
                        through tests/fake_comfy)
  torch_chain_reference.json   per (qtype, math dtype) of tests/test_torch_chain.py:
                        dtype, SHA-256 of the bytes and a seeded sample of the
                        bit patterns of `dequant.py::dequantize`, and the number
                        of materialising ATen kernels it issues
  reference_surface.json   public function / class names of dequant.py and ops.py

The reference is imported by path and never copied: dequant.py via importlib,
ops.py through a throw-away package directory of symlinks in $TMPDIR.
"""
import ast
import hashlib
import importlib
import importlib.util
import json
import os
import sys
import tempfile

import numpy as np
import torch
import gguf

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = None      # the original checkout, from the command line
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "fake_comfy"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle  # noqa: E402  (only for the seeded block generator)

T = gguf.GGMLQuantizationType
QTYPES = [T.Q4_0, T.Q4_1, T.Q5_0, T.Q5_1, T.Q8_0, T.Q2_K, T.Q3_K, T.Q4_K, T.Q5_K, T.Q6_K, T.IQ4_NL, T.IQ4_XS, T.BF16]
TORCH_DT = {0: torch.float16, 1: torch.bfloat16, 2: torch.float32}
# (math dtype, out dtype): default fp16 math -> fp16 / bf16 / fp32, "target" bf16, explicit fp32
COMBOS = [(0, 0), (0, 1), (0, 2), (1, 1), (2, 2), (2, 0)]


def load_ref_dequant():
    spec = importlib.util.spec_from_file_location("ref_dequant", os.path.join(REF, "dequant.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_ref_ops():
    tmp = tempfile.mkdtemp(prefix="refpkg_")
    pkg = os.path.join(tmp, "refgguf")
    os.mkdir(pkg)
    open(os.path.join(pkg, "__init__.py"), "w").close()
    for f in ("dequant.py", "ops.py"):
        os.symlink(os.path.join(REF, f), os.path.join(pkg, f))
    sys.path.insert(0, tmp)
    return importlib.import_module("refgguf.ops")


def bits(t: torch.Tensor) -> np.ndarray:
    t = t.contiguous()
    if t.dtype == torch.float32:
        return t.numpy().view(np.uint32).copy()
    return t.view(torch.int16).numpy().view(np.uint16).copy()


def edge_blocks(qtype, raw):
    """Overwrite a few leading blocks with corner cases: all-zero / all-one payloads, zero and large scales."""
    bs, ts = gguf.GGML_QUANT_SIZES[qtype]
    if qtype == T.BF16:
        return raw
    offs = oracle._F16_FIELDS[int(qtype)]

    def set_f16(b, vals):
        for off, v in zip(offs, vals):
            raw[b, off:off + 2] = np.array([v], dtype=np.float16).view(np.uint8)

    raw[0, :] = 0
    set_f16(0, [1.0, 1.0])
    raw[1, :] = 0xFF
    set_f16(1, [0.5, -0.25])
    raw[2, :] = 0xAA
    set_f16(2, [0.0, 0.0])
    raw[3, :] = 0x55
    set_f16(3, [-2.0, 6.1e-5])      # smallest normal fp16 as the second field
    raw[4, :] = 0x0F
    set_f16(4, [5.96e-8, 1e-3])     # subnormal scale
    set_f16(5, [48.0, -3.0])        # big-ish scale on random payload (products stay finite in fp16)
    return raw


def make_dequant(ref):
    for qt in QTYPES:
        bs, ts = gguf.GGML_QUANT_SIZES[qt]
        n_blocks = 40 if bs == 256 else (136 if bs == 32 else 4099)
        raw = oracle.random_blocks(int(qt), n_blocks, seed=1000 + int(qt))
        raw = edge_blocks(qt, raw)
        tt = torch.from_numpy(raw.reshape(-1).copy())
        out = {"packed": raw.reshape(-1), "qtype": np.int32(int(qt)), "n_blocks": np.int64(n_blocks)}
        for math, od in COMBOS:
            md = None if math == 0 else TORCH_DT[math]
            with torch.no_grad():
                r = ref.dequantize(tt, qt, (n_blocks * bs,), dtype=md).to(TORCH_DT[od])
            out[f"out_m{math}_o{od}"] = bits(r)
        np.savez_compressed(os.path.join(HERE, f"dequant_{qt.name}.npz"), **out)
        print("wrote dequant", qt.name, n_blocks, "blocks")


def make_linear(refops):
    GGMLTensor, GGMLOps = refops.GGMLTensor, refops.GGMLOps
    cases = [(T.Q4_K, 512, 96), (T.Q8_0, 512, 96), (T.Q5_K, 512, 80), (T.Q6_K, 256, 72), (T.Q4_0, 320, 64), (T.BF16, 192, 40)]
    M = 24
    for qt, K, N in cases:
        bs, ts = gguf.GGML_QUANT_SIZES[qt]
        raw = oracle.random_blocks(int(qt), N * K // bs, seed=2000 + int(qt), scale=0.02).reshape(N, K // bs * ts)
        rng = np.random.default_rng(3000 + int(qt))
        bias = rng.normal(0, 0.02, size=N).astype(np.float32)
        x32 = rng.normal(0, 1, size=(M, K)).astype(np.float32)
        for act, name in ((torch.bfloat16, "bf16"), (torch.float16, "f16"), (torch.float32, "f32")):
            lin = GGMLOps.Linear(K, N)
            sd = {
                "weight": GGMLTensor(torch.from_numpy(raw.copy()), tensor_type=qt, tensor_shape=torch.Size((N, K))),
                "bias": GGMLTensor(torch.from_numpy(bias.copy()), tensor_type=T.F32, tensor_shape=torch.Size((N,))),
            }
            lin.load_state_dict(sd)
            x = torch.from_numpy(x32).to(act)
            with torch.no_grad():
                y = lin(x)
            assert type(y) is torch.Tensor and y.dtype == act and tuple(y.shape) == (M, N)
            np.savez_compressed(
                os.path.join(HERE, f"linear_{qt.name}_{name}.npz"),
                packed=raw.reshape(-1), qtype=np.int32(int(qt)), N=np.int64(N), K=np.int64(K), M=np.int64(M),
                bias=bias, x=bits(x), y=bits(y))
        print("wrote linear", qt.name)


def make_torch_chain(ref):
    """What tests/test_torch_chain.py compares oracle/torch_chain.py with: the full output is pinned by its SHA-256, a
    seeded sample of 64 bit patterns makes a mismatch readable."""
    from test_torch_chain import MATH_DTYPES, QTYPES as CHAIN_QTYPES, Count, case_id, inputs, output_bits
    out = {}
    for qt, md in ((qt, md) for md in MATH_DTYPES for qt in CHAIN_QTYPES):
        raw, shape = inputs(qt)
        with Count() as c:
            a = ref.dequantize(raw, qt, shape, dtype=md)
        b = output_bits(a)
        idx = np.sort(np.random.default_rng(0).choice(b.size, size=min(64, b.size), replace=False))
        out[case_id(qt, md)] = {"dtype": str(a.dtype), "shape": list(a.shape), "aten_kernels": c.n,
                                "sha256": hashlib.sha256(b.tobytes()).hexdigest(),
                                "sample_index": idx.tolist(), "sample_bits": b[idx].tolist()}
    with open(os.path.join(HERE, "torch_chain_reference.json"), "w") as f:       # one case per line
        f.write("{\n" + ",\n".join(f" {json.dumps(k)}: {json.dumps(v)}" for k, v in out.items()) + "\n}\n")
    print("wrote torch_chain_reference.json", len(out), "cases")


def make_surface():
    """Public top-level function / class names of the original dequant.py and ops.py (tests/test_host.py)."""
    def public(path):
        tree = ast.parse(open(path).read())
        return sorted(n.name for n in tree.body if isinstance(n, (ast.FunctionDef, ast.ClassDef)) and not n.name.startswith("_"))
    with open(os.path.join(HERE, "reference_surface.json"), "w") as f:
        json.dump({name: public(os.path.join(REF, name)) for name in ("dequant.py", "ops.py")}, f, indent=1)
        f.write("\n")
    print("wrote reference_surface.json")


if __name__ == "__main__":
    if len(sys.argv) < 2 or not os.path.isfile(os.path.join(sys.argv[1], "dequant.py")):
        sys.exit(__doc__)
    REF = os.path.abspath(sys.argv[1])
    groups = sys.argv[2:] or ["dequant", "linear", "torch_chain", "surface"]
    torch.manual_seed(0)
    if "dequant" in groups:
        make_dequant(load_ref_dequant())
    if "linear" in groups:
        make_linear(load_ref_ops())
    if "torch_chain" in groups:
        make_torch_chain(load_ref_dequant())
    if "surface" in groups:
        make_surface()
    print("total bytes:", sum(os.path.getsize(os.path.join(HERE, f)) for f in os.listdir(HERE) if f.endswith((".npz", ".json"))))
