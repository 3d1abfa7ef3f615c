"""Tensor-core GEMM and fused transposed GEMM for 1x16 weights with in_group_size 16 (the 1-bit PV-tuned checkpoints).

Batches above the GEMV threshold run ONE fused dequant + tcgen05 launch (a 16-wide group is one 32-byte codebook entry),
and the backward w.r.t. the input is the fused transposed kernel: W is never written to HBM.  Layouts the kernels do not
cover (code rows that are not a 16-byte multiple) keep the GEMV passes.
"""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch
from helpers import TOL_BF16, TOL_FP16_TIGHT, TOL_NORTH_STAR, c_oracle_check, gpu_case, make_module, oracle_output, to_torch

from oracle import aqlm_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
LLAMA3_8B = [(4096, 4096), (4096, 14336), (14336, 4096)]


def _launches():
    from aqlm_b200 import _cabi

    return _cabi.launch_count()


def _transposed_ref(t, go):
    """(grad_out * scales) @ W_unscaled from the C oracle's dequantized (scaled) rows, fp32."""
    from oracle import c_oracle

    f32 = lambda a: a.float().cpu().numpy()  # noqa: E731
    W = c_oracle.dequantize_weight(t["codes"].cpu().numpy(), f32(t["codebooks"]), f32(t["scales"]))
    return f32(go) @ W


# ---- forward ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(512, 200), (1152, 456)])
@pytest.mark.parametrize("batch", [7, 16, 64, 100, 256, 300])
def test_g16_gemm_vs_oracle_small(shape, batch):
    from aqlm_b200.inference_kernels import cuda_kernel

    fin, fout = shape
    case = O.make_case(12000 + fin + batch, fin, fout, 1, 16, 16, batch, bias=(batch % 2 == 0))
    t = to_torch(case, DEV)
    cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], t["bias"])  # workspace sized outside the count
    before = _launches()
    y = cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], t["bias"])
    assert _launches() == before + 1, "one tensor-core launch, not one GEMV pass per 8 rows"
    assert O.relative_error(y.float().cpu().numpy(), oracle_output(case)) < TOL_FP16_TIGHT


@pytest.mark.parametrize("batch", [16, 64, 256])
@pytest.mark.parametrize("shape", LLAMA3_8B)
def test_g16_gemm_full_size(shape, batch):
    from aqlm_b200.inference_kernels import cuda_kernel

    fin, fout = shape
    t = gpu_case(fin, fout, 1, 16, batch, seed=fin + fout + batch + 16, g=16)
    y = cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], None)
    rel = c_oracle_check(t, y)
    assert rel < TOL_FP16_TIGHT, rel
    y2 = cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], None)
    assert torch.equal(y, y2)  # fixed-order split-K reduction
    yv = cuda_kernel.matmat(t["x"][:4], t["codes"], t["codebooks"], t["scales"], None).float()
    assert ((yv - y[:4].float()).abs().mean() / yv.abs().mean()).item() < 1e-3


def test_g16_gemm_bf16():
    from aqlm_b200.inference_kernels import cuda_kernel

    t = gpu_case(4096, 14336, 1, 16, 256, dtype=torch.bfloat16, seed=1616, g=16)
    y = cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], None)
    assert c_oracle_check(t, y) < TOL_BF16


def test_g16_gemm_without_workspace():
    """The C-ABI entry point without a workspace (no split-K)."""
    from aqlm_b200 import _cabi
    from aqlm_b200.inference_kernels import cuda_kernel

    case = O.make_case(12100, 1024, 256, 1, 16, 16, 32, True)
    t = to_torch(case, DEV)
    w = cuda_kernel.make_weight(t["codes"], t["codebooks"], t["scales"].reshape(-1), t["bias"])
    y = torch.empty((32, 256), dtype=torch.float16, device=DEV)
    before = _launches()
    _cabi.check(_cabi.lib().aqlm_b200_matmat_dequant(ctypes.byref(w), t["x"].data_ptr(), y.data_ptr(), 32,
                                                     torch.cuda.current_stream().cuda_stream))
    assert _launches() == before + 1
    assert O.relative_error(y.float().cpu().numpy(), oracle_output(case)) < TOL_FP16_TIGHT


def test_g16_gemm_row_stride_not_tma_compatible_falls_back():
    """in_features = 192: code rows of 24 bytes cannot be a TMA row stride; the GEMV passes still answer."""
    from aqlm_b200.inference_kernels import cuda_kernel

    case = O.make_case(12200, 192, 72, 1, 16, 16, 9, True)
    t = to_torch(case, DEV)
    y = cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], t["bias"]).float().cpu().numpy()
    assert O.relative_error(y, oracle_output(case)) < TOL_FP16_TIGHT


def test_g16_gemm_matches_gemv_passes():
    """The tensor-core path against the GEMV passes it replaces (AQLM_B200_DISABLE_TCGEN05=1) at 4096 -> 14336, bs 64."""
    from aqlm_b200 import _cabi
    from aqlm_b200.inference_kernels import cuda_kernel

    t = gpu_case(4096, 14336, 1, 16, 64, seed=12300, g=16)
    y = cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], None).float()
    saved = os.environ.get("AQLM_B200_DISABLE_TCGEN05")
    try:
        os.environ["AQLM_B200_DISABLE_TCGEN05"] = "1"
        _cabi.reload_tunables()
        before = _launches()
        yp = cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], None).float()
        assert _launches() == before + 8  # 64 rows in passes of 8
    finally:
        if saved is None:
            os.environ.pop("AQLM_B200_DISABLE_TCGEN05", None)
        else:
            os.environ["AQLM_B200_DISABLE_TCGEN05"] = saved
        _cabi.reload_tunables()
    assert ((y - yp).abs().mean() / yp.abs().mean()).item() < TOL_FP16_TIGHT


# ---- backward w.r.t. the input ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(512, 200), (1152, 456)])
@pytest.mark.parametrize("batch", [1, 7, 64, 256, 300])
def test_g16_transposed_vs_oracle_small(shape, batch):
    from aqlm_b200 import _cabi
    from aqlm_b200.inference_kernels import cuda_kernel

    fin, fout = shape
    t = gpu_case(fin, fout, 1, 16, 1, seed=12400 + fin + batch, g=16)
    go = torch.randn((batch, fout), dtype=torch.float16, device=DEV)
    ref = _transposed_ref(t, go)
    # the C-ABI entry point itself (no workspace): fused kernel, not ERR_UNSUPPORTED
    w = cuda_kernel.make_weight(t["codes"], t["codebooks"], t["scales"].reshape(-1), None)
    gx = torch.empty((batch, fin), dtype=torch.float16, device=DEV)
    before = _launches()
    rc = _cabi.lib().aqlm_b200_matmat_dequant_transposed(ctypes.byref(w), go.data_ptr(), gx.data_ptr(), batch, None, 0,
                                                         torch.cuda.current_stream().cuda_stream)
    assert rc == _cabi.OK, _cabi.lib().aqlm_b200_last_error()
    assert _launches() == before + 1
    assert O.relative_error(gx.float().cpu().numpy(), ref) < TOL_NORTH_STAR
    # the op (split-K with the persistent workspace)
    before = _launches()
    gx2 = cuda_kernel.matmat_dequant_transposed(go, t["codes"], t["codebooks"], t["scales"], None)
    assert _launches() == before + 1, "the backward must be ONE fused kernel (no dequant + library GEMM)"
    assert O.relative_error(gx2.float().cpu().numpy(), ref) < TOL_NORTH_STAR


@pytest.mark.parametrize("shape,dtype", [((4096, 14336), torch.float16), ((14336, 4096), torch.float16),
                                         ((4096, 4096), torch.bfloat16)])
def test_g16_transposed_full_size(shape, dtype):
    from aqlm_b200.inference_kernels import cuda_kernel

    fin, fout = shape
    t = gpu_case(fin, fout, 1, 16, 1, dtype=dtype, seed=12500 + fin, g=16)
    go = torch.randn((256, fout), dtype=dtype, device=DEV)
    gx = cuda_kernel.matmat_dequant_transposed(go, t["codes"], t["codebooks"], t["scales"], None)
    rel = O.relative_error(gx.float().cpu().numpy(), _transposed_ref(t, go))
    assert rel < (TOL_NORTH_STAR if dtype == torch.float16 else TOL_BF16), rel
    gx2 = cuda_kernel.matmat_dequant_transposed(go, t["codes"], t["codebooks"], t["scales"], None)
    assert torch.equal(gx, gx2)


def test_g16_module_autograd_never_materialises_w():
    """QuantizedLinear(in_group_size=16) on 32 rows: one launch forward, one launch backward, and the backward allocates
    less than W would take."""
    fin, fout = 4096, 4096
    case = O.make_case(12600, fin, fout, 1, 16, 16, 32, False)
    layer, t = make_module(case, DEV)
    assert layer.in_group_size == 16
    x = t["x"].clone().requires_grad_(True)
    go = torch.randn((32, fout), dtype=torch.float16, device=DEV)
    torch.autograd.grad(layer(x), x, go)  # binds the ops and sizes the workspaces of both directions
    before = _launches()
    y = layer(x)
    assert _launches() == before + 1
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    before = _launches()
    (gx,) = torch.autograd.grad(y, x, go)
    torch.cuda.synchronize()
    assert _launches() == before + 1
    assert torch.cuda.max_memory_allocated() - base < fout * fin * 2
    W = O.dequantize_weight(O.unpack_int_data(case["codes"], 16), case["codebooks"], case["scales"])
    assert O.relative_error(gx.float().cpu().numpy(), go.float().cpu().numpy() @ W) < TOL_NORTH_STAR


def test_g16_gemm_cuda_graph():
    """Capture the split-K g16 GEMM (workspace baked into the graph), replay it, compare with eager."""
    from aqlm_b200.inference_kernels import cuda_kernel

    t = gpu_case(4096, 4096, 1, 16, 64, seed=12700, g=16)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], None)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        yg = cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], None)
    t["x"].mul_(0.5)
    g.replay()
    torch.cuda.synchronize()
    ye = cuda_kernel.matmat_dequant(t["x"], t["codes"], t["codebooks"], t["scales"], None)
    assert torch.equal(yg, ye)
    assert c_oracle_check(t, yg) < TOL_FP16_TIGHT


# ---- end to end: a 1-bit style checkpoint (1x16, in_group_size 16) through from_pretrained -----------------------------
@pytest.fixture
def aqlm_alias(monkeypatch):
    pytest.importorskip("transformers")
    import aqlm_b200

    saved = {k: v for k, v in sys.modules.items() if k == "aqlm" or k.startswith("aqlm.")}
    aqlm_b200.install_as_aqlm()
    import transformers.quantizers.quantizer_aqlm as QA

    monkeypatch.setattr(QA, "is_accelerate_available", lambda: True)
    yield aqlm_b200
    for k in [k for k in sys.modules if k == "aqlm" or k.startswith("aqlm.")]:
        del sys.modules[k]
    sys.modules.update(saved)


def _write_g16_checkpoint(path, seed=0, hidden=128, inter=256, layers=2, heads=4, kv_heads=2, vocab=96):
    """A synthetic Llama checkpoint with 1x16 / in_group_size 16 linears; returns (config, dense dequantized state dict)."""
    from transformers import LlamaConfig, LlamaForCausalLM

    from aqlm_b200 import hf

    cfg = LlamaConfig(hidden_size=hidden, intermediate_size=inter, num_hidden_layers=layers, num_attention_heads=heads,
                      num_key_value_heads=kv_heads, vocab_size=vocab, max_position_embeddings=64, tie_word_embeddings=False)
    torch.manual_seed(seed)
    dense = LlamaForCausalLM(cfg).half()
    rng = np.random.default_rng(seed)
    ckpt, dense_sd, not_quantized = {}, {}, ["lm_head.weight", "lm_head"]
    for name, p in dense.state_dict().items():
        if name.endswith("_proj.weight"):
            out_f, in_f = p.shape
            codes = rng.integers(0, 2**16, size=(out_f, in_f // 16, 1))
            cb = (rng.standard_normal((1, 2**16, 1, 16)) * 0.08).astype(np.float16)
            sc = (0.75 + 0.5 * rng.random((out_f, 1, 1, 1))).astype(np.float16)
            ckpt.update(hf.quantized_state_entries(name[: -len(".weight")], torch.from_numpy(codes), torch.from_numpy(cb),
                                                   torch.from_numpy(sc), 16))
            dense_sd[name] = torch.from_numpy(O.dequantize_weight(codes, cb.astype(np.float32), sc.astype(np.float32))).half()
        else:
            ckpt[name] = dense_sd[name] = p.half()
            not_quantized.append(name)
    hf.save_quantized_checkpoint(path, cfg.to_dict(), ckpt,
                                 hf.quantization_config_dict(1, 16, in_group_size=16,
                                                             linear_weights_not_to_quantize=not_quantized))
    return cfg, dense_sd


def test_g16_checkpoint_prefill_logits_match_dense_model(tmp_path, aqlm_alias):
    from transformers import AutoModelForCausalLM, LlamaForCausalLM

    cfg, dense_sd = _write_g16_checkpoint(str(tmp_path / "m"), seed=16)
    model = AutoModelForCausalLM.from_pretrained(str(tmp_path / "m"), dtype=torch.float16).to(DEV).eval()
    mods = [m for n, m in model.named_modules() if n.endswith("_proj")]
    assert mods and all(type(m) is aqlm_alias.QuantizedLinear and m.in_group_size == 16 for m in mods)
    dense = LlamaForCausalLM(cfg).half()
    dense.load_state_dict(dense_sd)
    dense = dense.to(DEV).eval()
    ids = torch.randint(0, cfg.vocab_size, (1, 20), device=DEV)
    with torch.no_grad():
        before = _launches()
        lq = model(ids).logits.float()  # 20 rows per linear: tensor-core op
        assert _launches() - before == len(mods)  # one launch per linear
        ld = dense(ids).logits.float()
    rel = ((lq - ld).abs().mean() / ld.abs().mean()).item()
    assert rel < 5e-3, rel
