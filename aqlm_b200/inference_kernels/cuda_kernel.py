"""CUDA ops of the `aqlm` surface, backed by the aqlm_b200 C-ABI (reference inference_kernels/cuda_kernel.py).

Mirrors what the reference registers (cuda_kernel.py:13-132): torch.library ops
`aqlm::code{1x16,2x8,1x8}_matmat[_dequant[_transposed]]` with schema
`(Tensor input, Tensor codes, Tensor codebooks, Tensor scales, Tensor? bias) -> Tensor` plus fake/meta shapes so
`torch.compile` / CUDA-graph capture work, and a `CUDA_KERNEL` namespace exposing the functions the reference's
pybind module exports (cuda_kernel.cpp:686-699; used by benchmark/matmul_benchmark.py:103).  Differences:
no JIT build at import (the .so is prebuilt in-tree for sm_100a), `aqlm::generic_matmat[_dequant]` covers every
other KxN scheme (the reference sends those to Triton, kernel_selector.py:91-94), and CPU tensors are an error.
"""
from __future__ import annotations

import ctypes
import os
from types import SimpleNamespace
from typing import Optional

import torch

from .. import _cabi

CUDA_FOLDER = os.path.dirname(os.path.abspath(_cabi.LIB_PATH))

_DTYPES = {torch.float16: _cabi.F16, torch.bfloat16: _cabi.BF16}


def _dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        # same exception type and message as check_use_bfloat16 (reference cuda_kernel.cpp:9-25)
        raise NotImplementedError(
            f"AQLM CUDA kernels only support float16 and bfloat16. Got {t.dtype}. "
            "Please specify the correct `torch_dtype` when loading the model.") from None


def _require_cuda(*tensors: Optional[torch.Tensor]) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise NotImplementedError(
                "aqlm_b200 implements the CUDA (sm_100a) hot path only; got a tensor on "
                f"{t.device}. There is no CPU fallback in this package.")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise ValueError(f"all tensors must be on the same device, got {dev} and {t.device}")
    return dev


def make_weight(codes: torch.Tensor, codebooks: torch.Tensor, scales: Optional[torch.Tensor],
                bias: Optional[torch.Tensor]) -> "_cabi.Weight":
    """Describe one quantized matrix for the C-ABI.  Tensors must stay alive while the struct is used."""
    num_codebooks, codebook_size, out_group_size, in_group_size = codebooks.shape
    if codes.dim() == 2:  # the reference squeezes the codebook axis for 1x16 (cuda_kernel.cpp:167)
        codes = codes.unsqueeze(-1)
    out_groups, in_groups, k = codes.shape
    if k != num_codebooks:
        raise ValueError(f"codes have {k} codebooks, codebooks tensor has {num_codebooks}")
    nbits = int(codebook_size).bit_length() - 1
    if codes.dtype not in (torch.int8, torch.int16) or codes.element_size() != (1 if nbits <= 8 else 2):
        raise ValueError(f"codes dtype {codes.dtype} does not match {nbits}-bit codebooks")
    for name, t in (("codes", codes), ("codebooks", codebooks), ("scales", scales), ("bias", bias)):
        if t is not None and not t.is_contiguous():
            raise ValueError(f"{name} must be contiguous")
    w = _cabi.Weight()
    w.codes = codes.data_ptr()
    w.codebooks = codebooks.data_ptr()
    w.scales = scales.data_ptr() if scales is not None else None
    w.bias = bias.data_ptr() if bias is not None else None
    w.in_features = in_groups * in_group_size
    w.out_features = out_groups * out_group_size
    w.num_codebooks = num_codebooks
    w.nbits_per_codebook = nbits
    w.in_group_size = in_group_size
    w.out_group_size = out_group_size
    w.dtype = _dtype_code(codebooks)
    return w


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class _on_device:
    """Cheap device guard: only switches when the tensors live on a non-current device."""

    def __init__(self, device: torch.device):
        self.ctx = None
        if device.index is not None and device.index != torch.cuda.current_device():
            self.ctx = torch.cuda.device(device)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)


_WORKSPACES: dict = {}   # (device index, stream handle) -> workspace of eager launches on that stream
_GRAPH_WS: dict = {}     # device index -> workspace baked into CUDA graphs captured on that device
_RETIRED: list = []      # outgrown buffers are NEVER freed: a captured graph may still hold their address
_WS_MIN_BYTES = 4 << 20


def _grow(table: dict, key, device: torch.device, nbytes: int) -> torch.Tensor:
    ws = table.get(key)
    if ws is None or ws.numel() < nbytes:
        if ws is not None:
            _RETIRED.append(ws)
        ws = torch.zeros(max(nbytes, _WS_MIN_BYTES), dtype=torch.uint8, device=device)
        table[key] = ws
    return ws


def _workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    """Persistent zero-initialised workspace (ticket counters + fp32 partials) of the split-K GEMM and the LUT GEMV.

    * Eager launches: one buffer per (device, stream), so kernels on different streams never share tickets/partials.
    * Launches recorded into a CUDA graph: ONE dedicated buffer per device, never shared with eager launches (a replay
      on a side stream cannot race with default-stream kernels).  It is sized during the eager warm-up calls (every
      eager request also grows it), so the usual warm-up-then-capture recipe allocates nothing inside the capture; if
      it must grow inside a capture, the new block comes from that graph's pool and is kept alive here.
    * Buffers that are outgrown are retired, not freed: graph-baked pointers stay valid and the kernels' "counters are
      left at zero" invariant holds for every buffer.
    Graphs that contain workspace-using aqlm_b200 ops must not be replayed concurrently with each other on one device.
    """
    if torch.cuda.is_current_stream_capturing():
        return _grow(_GRAPH_WS, device.index, device, nbytes)
    _grow(_GRAPH_WS, device.index, device, nbytes)
    return _grow(_WORKSPACES, (device.index, _stream_ptr(device)), device, nbytes)


def _prepare(input, codes, codebooks, scales, bias):
    device = _require_cuda(input, codes, codebooks, scales, bias)
    _dtype_code(input)
    if input.dtype != codebooks.dtype:
        raise ValueError(f"input dtype {input.dtype} != codebooks dtype {codebooks.dtype}")
    w = make_weight(codes, codebooks, scales.reshape(-1) if scales is not None else None, bias)
    if input.shape[-1] != w.in_features:
        raise ValueError(f"input has {input.shape[-1]} features, weight expects {w.in_features}")
    flat_input = input.reshape(-1, input.shape[-1])
    if not flat_input.is_contiguous():
        flat_input = flat_input.contiguous()
    return device, w, flat_input


def _call_matmat_ws(device, w, flat_input, flat_output, flags: int) -> None:
    batch = flat_input.shape[0]
    with _on_device(device):
        L = _cabi.lib()
        need = L.aqlm_b200_matmat_workspace_bytes(ctypes.byref(w), batch) if batch > 0 else 0
        ws = _workspace(device, need) if need else None
        _cabi.check(L.aqlm_b200_matmat_ws(ctypes.byref(w), flat_input.data_ptr(), flat_output.data_ptr(), batch, flags,
                                          ws.data_ptr() if ws is not None else None,
                                          ws.numel() if ws is not None else 0, _stream_ptr(device)))


def matmat(input, codes, codebooks, scales, bias=None) -> torch.Tensor:
    """Fused gather + additive dequant + GEMV (+scale+bias), any scheme; for small batch (reference `*_matmat`).
    Batch-1 calls on 256-entry codebooks run the dot-product-LUT kernel."""
    device, w, flat_input = _prepare(input, codes, codebooks, scales, bias)
    flat_output = torch.empty((flat_input.shape[0], w.out_features), dtype=input.dtype, device=device)
    _call_matmat_ws(device, w, flat_input, flat_output, 0)
    return flat_output.reshape(input.shape[:-1] + (w.out_features,))


def matmat_dequant(input, codes, codebooks, scales, bias=None) -> torch.Tensor:
    """Fused dequant + tcgen05 tensor-core GEMM (+scale+bias); for large batch (reference `*_matmat_dequant`)."""
    device, w, flat_input = _prepare(input, codes, codebooks, scales, bias)
    batch = flat_input.shape[0]
    flat_output = torch.empty((batch, w.out_features), dtype=input.dtype, device=device)
    with _on_device(device):
        L = _cabi.lib()
        need = L.aqlm_b200_matmat_dequant_workspace_bytes(ctypes.byref(w), batch) if batch > 0 else 0
        ws = _workspace(device, need) if need else None
        _cabi.check(L.aqlm_b200_matmat_dequant_ws(ctypes.byref(w), flat_input.data_ptr(), flat_output.data_ptr(), batch,
                                                  ws.data_ptr() if ws is not None else None,
                                                  ws.numel() if ws is not None else 0, _stream_ptr(device)))
    return flat_output.reshape(input.shape[:-1] + (w.out_features,))


def matmat_grouped(input, codes, codebooks_stacked, scales, bias, seg_rows, partial: bool = False) -> torch.Tensor:
    """ONE launch for several 1x16 linears sharing `input`: `codes` [sum(seg_rows), in/8, 1] (row-concatenated),
    `codebooks_stacked` [n_seg, 1, 65536, 1, 8], `scales`/`bias` concatenated.  Returns [..., sum(seg_rows)] in the input
    dtype, or UNSCALED fp32 partials when `partial` (sharded path)."""
    device = _require_cuda(input, codes, codebooks_stacked, scales, bias)
    _dtype_code(input)
    n_seg = codebooks_stacked.shape[0]
    if n_seg != len(seg_rows) or not codebooks_stacked.is_contiguous():
        raise ValueError("codebooks_stacked must be a contiguous [n_seg, ...] stack matching seg_rows")
    w = make_weight(codes, codebooks_stacked[0], None if partial else scales.reshape(-1), None if partial else bias)
    if input.shape[-1] != w.in_features:
        raise ValueError(f"input has {input.shape[-1]} features, weight expects {w.in_features}")
    flat_input = input.reshape(-1, input.shape[-1])
    if not flat_input.is_contiguous():
        flat_input = flat_input.contiguous()
    batch = flat_input.shape[0]
    out = torch.empty((batch, w.out_features), dtype=torch.float32 if partial else input.dtype, device=device)
    seg = (ctypes.c_int64 * n_seg)(*[int(r) for r in seg_rows])
    with _on_device(device):
        _cabi.check(_cabi.lib().aqlm_b200_matmat_grouped(ctypes.byref(w), seg, n_seg, flat_input.data_ptr(), out.data_ptr(),
                                                         batch, _cabi.FLAG_PARTIAL_F32 if partial else 0,
                                                         _stream_ptr(device)))
    return out.reshape(input.shape[:-1] + (w.out_features,))


def matmat_partial(input, codes, codebooks) -> torch.Tensor:
    """UNSCALED fp32 partial products [batch, out] of an in_features shard (to be all-reduced)."""
    device = _require_cuda(input, codes, codebooks)
    w = make_weight(codes, codebooks, None, None)
    flat_input = input.reshape(-1, input.shape[-1]).contiguous()
    out = torch.empty((flat_input.shape[0], w.out_features), dtype=torch.float32, device=device)
    _call_matmat_ws(device, w, flat_input, out, _cabi.FLAG_PARTIAL_F32)
    return out


def scale_bias(partial: torch.Tensor, scales: torch.Tensor, bias: Optional[torch.Tensor], dtype: torch.dtype):
    """Epilogue after the all-reduce: (partial * scales + bias) rounded once to `dtype`."""
    device = _require_cuda(partial, scales, bias)
    partial = partial.contiguous()
    batch, out_features = partial.shape
    out = torch.empty((batch, out_features), dtype=dtype, device=device)
    code = _DTYPES[dtype]
    with _on_device(device):
        _cabi.check(_cabi.lib().aqlm_b200_scale_bias(partial.data_ptr(), scales.reshape(-1).data_ptr(),
                                                     bias.data_ptr() if bias is not None else None, out.data_ptr(),
                                                     batch, out_features, code, _stream_ptr(device)))
    return out


def dequant(codes, codebooks, scales=None) -> torch.Tensor:
    """W [out, in] (x scales if given): the reference's code*_dequant (cuda_kernel.cpp:184-227)."""
    device = _require_cuda(codes, codebooks, scales)
    scales_flat = scales.reshape(-1).contiguous() if scales is not None else None
    w = make_weight(codes, codebooks, scales_flat, None)
    weight = torch.empty((w.out_features, w.in_features), dtype=codebooks.dtype, device=device)
    with _on_device(device):
        _cabi.check(_cabi.lib().aqlm_b200_dequant(ctypes.byref(w), weight.data_ptr(), 1 if scales is not None else 0,
                                                  _stream_ptr(device)))
    return weight


def matmat_dequant_transposed(input, codes, codebooks, scales, bias=None) -> torch.Tensor:
    """Backward w.r.t. the input: grad_in = (grad_out * scales) @ W_unscaled (reference cuda_kernel.cpp:303-354).

    ONE fused kernel (csrc/gemm_tcgen05_t.cuh): W^T tiles are dequantized on chip into an MN-major tcgen05 operand, the
    per-row scale is folded into the tile, grad_out tiles arrive by TMA; W is never materialised and no library GEMM is
    called.  The reference's 2x8/1x8 variants forget the scaled input (cuda_kernel.cpp:497,518,662,683); not reproduced.
    `bias` is the forward bias [out]; it has no place in grad_input (the reference passes it to F::linear,
    cuda_kernel.cpp:348-353, which only type-checks when in == out) and is ignored.
    The fused kernel covers in_group_size 8 and 1x16 with in_group_size 16 (in_features % 128 == 0).  Layouts it does
    not cover (odd codebook counts, in_group_size 16 with several codebooks or 8-bit codes, ragged code rows) fall back
    to our dequant kernel + a dense matmul, as the reference does for every scheme.
    """
    device = _require_cuda(input, codes, codebooks, scales)
    _dtype_code(input)
    if input.dtype != codebooks.dtype:
        raise ValueError(f"grad_output dtype {input.dtype} != codebooks dtype {codebooks.dtype}")
    w = make_weight(codes, codebooks, scales.reshape(-1), None)
    if input.shape[-1] != w.out_features:
        raise ValueError(f"grad_output has {input.shape[-1]} features, weight has {w.out_features} output rows")
    flat = input.reshape(-1, input.shape[-1])
    if not flat.is_contiguous():
        flat = flat.contiguous()
    batch = flat.shape[0]
    out = torch.empty((batch, w.in_features), dtype=input.dtype, device=device)
    if batch == 0:
        return out.reshape(input.shape[:-1] + (w.in_features,))
    with _on_device(device):
        L = _cabi.lib()
        need = L.aqlm_b200_matmat_dequant_transposed_workspace_bytes(ctypes.byref(w), batch)
        ws = _workspace(device, need) if need else None
        rc = L.aqlm_b200_matmat_dequant_transposed(ctypes.byref(w), flat.data_ptr(), out.data_ptr(), batch,
                                                   ws.data_ptr() if ws is not None else None,
                                                   ws.numel() if ws is not None else 0, _stream_ptr(device))
    if rc == _cabi.ERR_UNSUPPORTED:
        weight = dequant(codes, codebooks, None)  # unscaled [out, in]
        out = (flat * scales.reshape(1, -1)) @ weight
    else:
        _cabi.check(rc)
    return out.reshape(input.shape[:-1] + (w.in_features,))


# ---- torch.library registration (reference cuda_kernel.py:13-132) ---------------------------------------
_SCHEMA = "(Tensor input, Tensor codes, Tensor codebooks, Tensor scales, Tensor? bias) -> Tensor"
_LIB = torch.library.Library("aqlm", "FRAGMENT")


def _fake_forward(input, codes, codebooks, scales, bias=None):
    return torch.empty(input.shape[:-1] + (codes.shape[0],), device=input.device, dtype=input.dtype)


def _fake_transposed(input, codes, codebooks, scales, bias=None):
    return torch.empty(input.shape[:-1] + (codes.shape[1] * codebooks.shape[3],), device=input.device,
                       dtype=input.dtype)


def _cpu_refusal(*args, **kwargs):
    raise NotImplementedError("aqlm_b200 ops run on CUDA (sm_100a) only; there is no CPU fallback in this package")


def _register(name: str, fn, fake) -> None:
    qual = f"aqlm::{name}"
    _LIB.define(f"{name}{_SCHEMA}")
    _LIB.impl(name, fn, "CUDA")
    _LIB.impl(name, _cpu_refusal, "CPU")
    torch.library.register_fake(qual, fake, lib=_LIB)


OP_NAMES = []
for _scheme in ("code1x16", "code2x8", "code1x8", "generic"):
    _register(f"{_scheme}_matmat", matmat, _fake_forward)
    _register(f"{_scheme}_matmat_dequant", matmat_dequant, _fake_forward)
    _register(f"{_scheme}_matmat_dequant_transposed", matmat_dequant_transposed, _fake_transposed)
    OP_NAMES += [f"{_scheme}_matmat", f"{_scheme}_matmat_dequant", f"{_scheme}_matmat_dequant_transposed"]

# The functions the reference's pybind module exports (cuda_kernel.cpp:686-699).
CUDA_KERNEL = SimpleNamespace(
    code1x16_matmat=matmat, code2x8_matmat=matmat, code1x8_matmat=matmat,
    code1x16_matmat_dequant=matmat_dequant, code2x8_matmat_dequant=matmat_dequant,
    code1x8_matmat_dequant=matmat_dequant,
    code1x16_matmat_dequant_transposed=matmat_dequant_transposed,
    code2x8_matmat_dequant_transposed=matmat_dequant_transposed,
    code1x8_matmat_dequant_transposed=matmat_dequant_transposed,
    code1x16_dequant=dequant, code2x8_dequant=dequant, code1x8_dequant=dequant,
)
