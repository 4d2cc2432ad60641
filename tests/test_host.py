"""CPU tests of the host-side mirror of the reference interface (GGMLTensor / GGMLLayer / GGMLOps / loader)."""
import json
import os

import numpy as np
import pytest
import torch
import gguf

import oracle
from util import Q


def _q8_tensor(pkg, N=16, K=64, seed=0):
    raw = oracle.random_blocks(int(Q.Q8_0), N * K // 32, seed=seed).reshape(N, K // 32 * 34)
    return pkg.ops.GGMLTensor(torch.from_numpy(raw), tensor_type=Q.Q8_0, tensor_shape=torch.Size((N, K))), raw


def test_ggmltensor_shape_vs_size_and_identity(pkg):
    t, raw = _q8_tensor(pkg, 512 // 32, 1024)
    assert tuple(t.shape) == (16, 1024)              # logical shape (ops.py:87-91)
    assert tuple(t.size()) == (16, 1024 // 32 * 34)  # byte shape
    assert t.clone() is t and t.detach() is t        # ops.py:64-68
    p = torch.nn.Parameter(t, requires_grad=False)
    assert p is t or p.data_ptr() == t.data_ptr()
    assert getattr(p, "tensor_type", None) == Q.Q8_0
    u = t.to(torch.device("cpu"))
    assert u.tensor_type == Q.Q8_0 and tuple(u.tensor_shape) == (16, 1024) and u.patches == []
    t.patches = [("x", "k")]
    v = t.to(torch.device("cpu"))
    assert v.patches == [("x", "k")]                 # carried over by .to() (ops.py:57-62)
    e = t.new_empty((3, 5))
    assert isinstance(e, pkg.ops.GGMLTensor) and tuple(e.shape) == (3, 5) and e.tensor_type == Q.Q8_0
    assert t.copy_(torch.zeros(7)) is None           # shape mismatch is swallowed with a warning (ops.py:70-75)


def test_is_quantized_predicates(pkg):
    t, _ = _q8_tensor(pkg)
    f16 = pkg.ops.GGMLTensor(torch.zeros(4, dtype=torch.float16), tensor_type=Q.F16, tensor_shape=torch.Size((4,)))
    bf = pkg.ops.GGMLTensor(torch.zeros(8, dtype=torch.uint8), tensor_type=Q.BF16, tensor_shape=torch.Size((4,)))
    d = pkg.dequant
    assert d.is_quantized(t) and d.is_quantized(bf)          # BF16 counts as quantised (dequant.py:7)
    assert not d.is_quantized(f16) and not d.is_quantized(None) and not d.is_quantized(torch.zeros(2))
    assert d.is_torch_compatible(f16) and d.is_torch_compatible(None)


def test_math_code_semantics(pkg):
    d, L = pkg.dequant, pkg.lib
    assert d.math_code(None, torch.bfloat16) == L.F16               # default: fp16 math
    assert d.math_code("target", torch.bfloat16) == L.BF16
    assert d.math_code("target", torch.float32) == L.F32
    assert d.math_code(torch.float32, torch.bfloat16) == L.F32
    with pytest.raises(TypeError):
        d.dtype_code(torch.float64)


def test_no_cpu_fallback(pkg):
    """Without a GPU the product refuses to dequantise instead of computing on the host."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    t, _ = _q8_tensor(pkg)
    with pytest.raises(pkg.lib.GGUFB200Error):
        pkg.dequant.dequantize_tensor(t, torch.float16)
    unsupported = pkg.ops.GGMLTensor(torch.zeros(64, dtype=torch.uint8), tensor_type=Q.IQ2_XXS, tensor_shape=torch.Size((64,)))
    with pytest.raises(NotImplementedError):
        pkg.dequant.dequantize_tensor(unsupported, torch.float16)
    # torch-compatible tensors never touch the library
    f32 = pkg.ops.GGMLTensor(torch.ones(4), tensor_type=Q.F32, tensor_shape=torch.Size((4,)))
    assert pkg.dequant.dequantize_tensor(f32, torch.float16).dtype == torch.float16


def test_linear_state_dict_hooks(pkg):
    ops = pkg.ops.GGMLOps
    lin = ops.Linear(64, 16)
    assert lin.weight is None and lin.bias is None          # allocates nothing (ops.py:232-240)
    w, _ = _q8_tensor(pkg, 16, 64)
    w.is_largest_weight = True
    b = pkg.ops.GGMLTensor(torch.zeros(16), tensor_type=Q.F32, tensor_shape=torch.Size((16,)))
    missing, unexpected = lin.load_state_dict({"weight": w, "bias": b}, strict=False)
    assert not missing and not unexpected
    assert lin.weight is w or lin.weight.data_ptr() == w.data_ptr()
    assert lin.largest_layer is True and lin.is_ggml_quantized()
    sd = lin.state_dict()
    assert sd["weight"].device.type == "meta" and sd["bias"].device.type == "meta"
    assert sd["temp.weight"].shape == (16, 64) and sd["temp.weight"].dtype == torch.float16   # ops.py:155-160

    lin2 = ops.Linear(64, 16)
    res = lin2.load_state_dict({}, strict=False)
    assert "weight" in res.missing_keys and tuple(lin2.weight.shape) == (64, 16)              # ops.py:131-134


def test_unquantised_linear_runs_on_cpu(pkg):
    """F16/F32 weights are 'torch compatible': the layer takes the host's manual-cast path, no kernel involved."""
    lin = pkg.ops.GGMLOps.Linear(8, 4)
    w = pkg.ops.GGMLTensor(torch.randn(4, 8), tensor_type=Q.F32, tensor_shape=torch.Size((4, 8)))
    b = pkg.ops.GGMLTensor(torch.randn(4), tensor_type=Q.F32, tensor_shape=torch.Size((4,)))
    lin.load_state_dict({"weight": w, "bias": b})
    x = torch.randn(3, 8)
    y = lin(x)
    assert type(y) is torch.Tensor
    torch.testing.assert_close(y, torch.nn.functional.linear(x, w.as_subclass(torch.Tensor), b.as_subclass(torch.Tensor)))


def test_class_level_dequant_dtype_knob(pkg):
    """nodes.py:152-164 sets dequant_dtype/patch_dtype on the CLASS GGMLOps.Linear."""
    ops = pkg.ops.GGMLOps()
    try:
        ops.Linear.dequant_dtype = torch.float32
        assert pkg.ops.GGMLOps.Linear(4, 4).dequant_dtype is torch.float32
        assert pkg.ops.GGMLOps.Conv2d.dequant_dtype is None
    finally:
        ops.Linear.dequant_dtype = None


def test_move_patch_to_device(pkg):
    item = [(torch.ones(2), ("lora", (torch.ones(2, 1), torch.ones(1, 2), None)), 1.0)]
    out = pkg.ops.move_patch_to_device(item, torch.device("cpu"))
    assert isinstance(out, list) and isinstance(out[0], tuple) and out[0][2] == 1.0


def _write_gguf(path, arch="flux"):
    w = gguf.GGUFWriter(path, arch)
    rng = np.random.default_rng(0)
    wq8 = rng.normal(0, 0.02, size=(32, 64)).astype(np.float32)
    w.add_tensor("model.diffusion_model.a.weight", gguf.quants.quantize(wq8, Q.Q8_0), raw_dtype=Q.Q8_0)
    w.add_tensor("model.diffusion_model.b.weight", gguf.quants.quantize(wq8, Q.Q4_0), raw_dtype=Q.Q4_0)
    k = oracle.random_blocks(int(Q.Q4_K), 8 * 2, seed=1).reshape(8, 2 * 144)
    w.add_tensor("model.diffusion_model.c.weight", k, raw_dtype=Q.Q4_K)
    w.add_tensor("model.diffusion_model.a.bias", np.arange(32, dtype=np.float32))
    w.add_tensor("model.diffusion_model.h.weight", rng.normal(size=(4, 6)).astype(np.float16))
    bf = (rng.normal(size=16).astype(np.float32).view(np.uint32) >> 16).astype(np.uint16)
    w.add_tensor("model.diffusion_model.n.scale", bf.view(np.uint8), raw_dtype=Q.BF16)
    w.add_tensor("other.ignored", np.zeros(4, dtype=np.float32))
    w.write_header_to_file(); w.write_kv_data_to_file(); w.write_tensors_to_file(); w.close()
    return wq8, k, bf


def test_gguf_sd_loader_round_trip(pkg, tmp_path):
    path = str(tmp_path / "m.gguf")
    wq8, k, bf = _write_gguf(path)
    sd, arch = pkg.loader.gguf_sd_loader(path, return_arch=True)
    assert arch == "flux"
    assert set(sd) == {"a.weight", "b.weight", "c.weight", "a.bias", "h.weight", "n.scale"}   # prefix stripped, others dropped
    a = sd["a.weight"]
    assert isinstance(a, pkg.ops.GGMLTensor) and a.tensor_type == Q.Q8_0
    assert tuple(a.shape) == (32, 64) and tuple(a.size()) == (32, 64 // 32 * 34) and a.dtype == torch.uint8
    assert tuple(sd["c.weight"].shape) == (8, 512)
    assert np.array_equal(sd["c.weight"].as_subclass(torch.Tensor).numpy(), k)
    assert sd["a.bias"].dtype == torch.float32 and tuple(sd["a.bias"].shape) == (32,)
    assert sd["h.weight"].dtype == torch.float16 and tuple(sd["h.weight"].size()) == (4, 6)
    n = sd["n.scale"]                                          # 1-D BF16 is widened to fp32 at load (loader.py:122-124)
    assert n.dtype == torch.float32 and np.array_equal(n.numpy().view(np.uint32) >> 16, bf.astype(np.uint32))
    marked = [key for key, v in sd.items() if getattr(v, "is_largest_weight", False)]
    assert marked == ["c.weight"]                              # largest quantised payload (loader.py:133-137)
    # the packed bytes dequantise (oracle) to the quantiser's own reconstruction
    want = gguf.quants.dequantize(gguf.quants.quantize(wq8, Q.Q8_0), Q.Q8_0)
    got = oracle.dequant(a.as_subclass(torch.Tensor).numpy(), int(Q.Q8_0), oracle.DT_F32, oracle.DT_F32).reshape(32, 64)
    assert np.array_equal(got, want)


def test_loader_rejects_wrong_architectures(pkg, tmp_path):
    path = str(tmp_path / "t.gguf")
    _write_gguf(path, arch="llama")
    with pytest.raises(ValueError):
        pkg.loader.gguf_sd_loader(path)                        # image loader, text arch (loader.py:90-91)
    sd = pkg.loader.gguf_sd_loader(path, is_text_model=True)
    assert "a.weight" in sd
    path2 = str(tmp_path / "u.gguf")
    _write_gguf(path2, arch="flux")
    with pytest.raises(ValueError):
        pkg.loader.gguf_sd_loader(path2, is_text_model=True)   # loader.py:87-89


def test_t5_key_remap(pkg):
    sd = {"enc.blk.3.attn_q.weight": 1, "enc.blk.0.attn_rel_b.weight": 2, "token_embd.weight": 3, "enc.output_norm.weight": 4,
          "enc.blk.1.ffn_gate.weight": 5}
    out = pkg.loader.sd_map_replace(sd, pkg.loader.T5_SD_MAP)
    assert out == {"encoder.block.3.layer.0.SelfAttention.q.weight": 1,
                   "encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight": 2,
                   "shared.weight": 3, "encoder.final_layer_norm.weight": 4,
                   "encoder.block.1.layer.1.DenseReluDense.wi_0.weight": 5}


def test_surface_matches_reference(pkg, golden_dir):
    """Same public names as the reference modules for the hot-path surface (SURVEY.md 8b).  The reference's public names
    are stored in tests/golden/reference_surface.json (tests/golden/make_golden.py)."""
    surface = json.load(open(os.path.join(golden_dir, "reference_surface.json")))
    ref_dq = set(surface["dequant.py"])
    for name in ("is_torch_compatible", "is_quantized", "dequantize_tensor", "dequantize"):
        assert name in ref_dq and hasattr(pkg.dequant, name)
    ref_ops = set(surface["ops.py"])
    for name in ("GGMLTensor", "GGMLLayer", "GGMLOps", "move_patch_to_device"):
        assert name in ref_ops and hasattr(pkg.ops, name)
    for cls in ("Linear", "Conv2d", "Embedding", "LayerNorm", "GroupNorm"):
        assert hasattr(pkg.ops.GGMLOps, cls)
    for m in ("is_ggml_quantized", "ggml_load_from_state_dict", "ggml_save_to_state_dict", "get_weight", "cast_bias_weight",
              "forward_comfy_cast_weights", "forward_ggml_cast_weights"):
        assert hasattr(pkg.ops.GGMLLayer, m)
    assert pkg.ops.GGMLLayer.comfy_cast_weights is True and pkg.ops.GGMLLayer.dequant_dtype is None


def test_lora_side_terms_recognises_only_plain_lora(pkg):
    """Host logic of the LoRA side-GEMM route (SURVEY 8f rank 1): only (strength, ("lora", (up, down, alpha, None, None,
    None)), 1.0, None, None) entries qualify; everything else must fall back to calculate_weight."""
    f = pkg.ops.lora_side_terms
    up, down = torch.ones(8, 2), torch.ones(2, 16)
    terms = f([(0.5, ("lora", (up, down, 4.0, None, None, None)), 1.0, None, None), (1.0, ("lora", (up, down, None)), 1.0)])
    assert [t[0] for t in terms] == [0.5 * 4.0 / 2, 1.0] and terms[0][1] is up and terms[0][2] is down
    assert f([]) == []
    assert f([(0.5, ("diff", (up,)), 1.0, None, None)]) is None
    assert f([(0.5, up, 1.0, None, None)]) is None                                        # bare tensor = diff
    assert f([(0.5, ("lora", (up, down, 4.0, None, None, None)), 0.7, None, None)]) is None      # strength_model
    assert f([(0.5, ("lora", (up, down, 4.0, None, None, None)), 1.0, (0, 0, 4), None)]) is None  # offset
    assert f([(0.5, ("lora", (up, down, 4.0, None, None, None)), 1.0, None, lambda w: w)]) is None
    assert f([(0.5, ("lora", (up, down, 4.0, torch.ones(2, 2), None, None)), 1.0, None, None)]) is None   # LoCon mid
    assert f([(0.5, ("lora", (up, down, 4.0, None, torch.ones(8), None)), 1.0, None, None)]) is None     # DoRA
    assert f([(0.5, ("lora", (up, torch.ones(3, 16), 4.0, None, None, None)), 1.0, None, None)]) is None   # rank mismatch

    class LoRAAdapter:                      # newer ComfyUI wraps the same tuple in an adapter object
        def __init__(self, weights):
            self.weights = weights
    assert f([(1.0, LoRAAdapter((up, down, 2.0, None, None, None)), 1.0, None, None)])[0][0] == 1.0
