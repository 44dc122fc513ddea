"""Torch-tensor front end of the C ABI: argument checking, output allocation, stream hand-off.

PyTorch is used here only for device memory and streams.  Every function requires CUDA tensors and launches
on ``torch.cuda.current_stream()``; nothing falls back to ATen math.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from . import _lib

F32, BF16, F16, E4M3 = 0, 1, 2, 3
E4M3_MAX = 448.0
ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2
LN_IDENTITY, LN_WINDOW, LN_MERGE2X2 = 0, 1, 2
GEMM_TC, GEMM_SIMT = 0, 1

_DT = {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16}

# Count of kernel launches issued through this module (bench.py reports it as `gpu_launches`).
launch_count = 0


def _code(dtype: torch.dtype) -> int:
    try:
        return _DT[dtype]
    except KeyError:
        raise TypeError(f"cs_vit kernels take float32, bfloat16 or float16 tensors, got {dtype}") from None


def _dev(*tensors: Optional[torch.Tensor]) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("cs_vit kernels run on CUDA tensors only (there is no CPU fallback)")


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


_profile = None  # {"name": entry point, "events": [(start, stop, flops, bytes, gemm kernel id)]} while bench.py instruments a kernel


def begin_profile(name: str) -> None:
    """Bracket every launch of C-ABI entry ``name`` with CUDA events on the launch stream (bench.py roofline)."""
    global _profile
    _profile = {"name": name, "events": []}


def end_profile() -> dict:
    global _profile
    prof, _profile = _profile, None
    torch.cuda.synchronize()
    ev = prof["events"]
    out = {"launches": len(ev), "ms": sum(e[0].elapsed_time(e[1]) for e in ev),
           "flops": float(sum(e[2] for e in ev)), "bytes": float(sum(e[3] for e in ev))}
    for kind in sorted({e[4] for e in ev if e[4]}):      # csvit_linear: the same split per kernel the C side chose
        sel = [e for e in ev if e[4] == kind]
        out[f"kind{kind}"] = {"launches": len(sel), "ms": sum(e[0].elapsed_time(e[1]) for e in sel), "flops": float(sum(e[2] for e in sel))}
    return out


def _call(name: str, *args, flops: float = 0.0, nbytes: float = 0.0) -> None:
    global launch_count
    launch_count += 1
    if _profile is not None and _profile["name"] == name:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(getattr(_lib.load(), name)(*args))
        e1.record()
        kind = _lib.load().csvit_last_gemm_kernel() if name == "csvit_linear" else 0
        _profile["events"].append((e0, e1, flops, nbytes, kind))
        return
    _lib.check(getattr(_lib.load(), name)(*args))


def _rows2d(t: torch.Tensor) -> Tuple[int, int, int]:
    """(rows, cols, row pitch in elements) of a 2-D tensor whose last dim is contiguous."""
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError(f"expected a 2-D tensor with contiguous rows, got shape {tuple(t.shape)} strides {t.stride()}")
    return t.shape[0], t.shape[1], t.stride(0)


# ---------------------------------------------------------------------------------------------- integer maps
def window_index_map(H: int, W: int, ws: int, shift: int, device="cuda") -> torch.Tensor:
    out = torch.empty(H * W, dtype=torch.int32, device=device)
    _call("csvit_window_index_map", H, W, ws, shift, out.data_ptr(), _stream())
    return out


def shift_mask(H: int, W: int, ws: int, shift: int, device="cuda") -> torch.Tensor:
    nW, L = (H // ws) * (W // ws), ws * ws
    out = torch.empty(nW, L, L, dtype=torch.float32, device=device)
    _call("csvit_shift_mask", H, W, ws, shift, out.data_ptr(), _stream())
    return out


def rel_pos_index(ws: int, device="cuda") -> torch.Tensor:
    out = torch.empty(ws * ws, ws * ws, dtype=torch.int32, device=device)
    _call("csvit_rel_pos_index", ws, out.data_ptr(), _stream())
    return out


def merge_index_map(H: int, W: int, device="cuda") -> torch.Tensor:
    out = torch.empty((H // 2) * (W // 2), 4, dtype=torch.int32, device=device)
    _call("csvit_merge_index_map", H, W, out.data_ptr(), _stream())
    return out


def expand_rel_bias(table: torch.Tensor, ws: int) -> torch.Tensor:
    _dev(table)
    table = table.contiguous().float()
    heads = table.shape[1]
    out = torch.empty(heads, ws * ws, ws * ws, dtype=torch.float32, device=table.device)
    _call("csvit_expand_rel_bias", table.data_ptr(), out.data_ptr(), heads, ws, _stream())
    return out


# ---------------------------------------------------------------------------------------------- row kernels
def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, *, out_dtype=torch.float32,
              mode: int = LN_IDENTITY, grid: Tuple[int, int] = (0, 0), ws: int = 0, shift: int = 0,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x: fp32 ``[rows_in, C]`` (tokens of all images, row-major).  Returns ``[rows_out, C or 4C]``."""
    _dev(x, gamma, beta, out)
    if x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("layernorm input must be contiguous float32")
    rows_in, C = x.shape
    H, W = grid
    if mode == LN_MERGE2X2:
        rows, width = rows_in // 4, 4 * C
    else:
        rows, width = rows_in, C
    if gamma.numel() != width or beta.numel() != width:
        raise ValueError(f"layernorm affine width {gamma.numel()} != {width}")
    if out is None:
        out = torch.empty(rows, width, dtype=out_dtype, device=x.device)
    _call("csvit_layernorm", x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), float(eps), out.data_ptr(), _code(out.dtype),
          out.stride(0), rows, C, mode, H, W, ws, shift, _stream(),
          nbytes=float(rows * width * (4 + out.element_size())))
    return out


def affine_rows(x: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, *, out_dtype=torch.float32) -> torch.Tensor:
    _dev(x, scale, shift)
    if x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("affine_rows input must be contiguous float32")
    C = x.shape[-1]
    out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    _call("csvit_affine_rows", x.data_ptr(), scale.data_ptr(), shift.data_ptr(), out.data_ptr(), _code(out_dtype),
          x.numel() // C, C, _stream())
    return out


_MEAN = (ctypes.c_float * 3)(0.485, 0.456, 0.406)  # ref:cs_vit/net/ti_poser.py:240-242
_STD = (ctypes.c_float * 3)(0.229, 0.224, 0.225)


def patch_im2col(img: torch.Tensor, *, out_dtype=torch.bfloat16, normalize: bool = True) -> torch.Tensor:
    """img fp32 ``[B,3,S,S]`` in [0,1] -> ``[B*(S/4)^2, 48]`` normalised 4x4 patches."""
    _dev(img)
    if img.dtype != torch.float32 or not img.is_contiguous() or img.dim() != 4 or img.shape[1] != 3:
        raise ValueError("patch_im2col takes contiguous float32 [B,3,S,S]")
    B, _, S, S2 = img.shape
    if S != S2:
        raise ValueError("square images only")
    out = torch.empty(B * (S // 4) ** 2, 48, dtype=out_dtype, device=img.device)
    mean = _MEAN if normalize else (ctypes.c_float * 3)(0, 0, 0)
    std = _STD if normalize else (ctypes.c_float * 3)(1, 1, 1)
    _call("csvit_patch_im2col", img.data_ptr(), out.data_ptr(), _code(out_dtype), B, S, mean, std, _stream())
    return out


# ---------------------------------------------------------------------------------------------- GEMM engine
def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *, act: int = ACT_NONE,
           resid: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None,
           scatter: Optional[Tuple[int, int, int, int]] = None, impl: int = GEMM_TC) -> torch.Tensor:
    """``out[orow] = act(a @ w.T + bias) + resid[orow]``; see ``csvit_linear`` in include/csvit.h."""
    _dev(a, w, bias, resid, out)
    M, K, lda = _rows2d(a)
    N, K2, ldw = _rows2d(w)
    if K != K2 or a.dtype != w.dtype:
        raise ValueError(f"linear: A {tuple(a.shape)}/{a.dtype} vs W {tuple(w.shape)}/{w.dtype}")
    if out is None:
        out = torch.empty(M, N, dtype=out_dtype or a.dtype, device=a.device)
    _, No, ldo = _rows2d(out)
    if No != N:
        raise ValueError("linear: output width mismatch")
    ldr = 0
    if resid is not None:
        if resid.dtype != torch.float32:
            raise ValueError("linear: residual must be float32")
        ldr = _rows2d(resid)[2]
    if bias is not None and (bias.dtype != torch.float32 or bias.numel() != N):
        raise ValueError("linear: bias must be float32 [N]")
    sH, sW, sws, ssh = scatter if scatter is not None else (0, 0, 0, 0)
    _call("csvit_linear", a.data_ptr(), lda, w.data_ptr(), ldw, _code(a.dtype), M, N, K, _p(bias), act, _p(resid), ldr,
          out.data_ptr(), ldo, _code(out.dtype), sH, sW, sws, ssh, impl, _stream(), flops=2.0 * M * N * K)
    return out


def _fp8_operand(name: str, t: torch.Tensor, scale: torch.Tensor, what: str) -> Tuple[int, int, int]:
    rows, K, ld = _rows2d(t)
    if t.dtype != torch.float8_e4m3fn:
        raise ValueError(f"{name}: {what} must be float8_e4m3fn, got {t.dtype}")
    if scale.dtype != torch.float32 or scale.numel() != rows or not scale.is_contiguous():
        raise ValueError(f"{name}: {what} scale must be contiguous float32 [{rows}]")
    if K % 16 != 0 or ld % 16 != 0:
        raise ValueError(f"{name}: {what} width {K} and pitch {ld} must be multiples of 16")
    return rows, K, ld


def linear_fp8(a8: torch.Tensor, row_scale: torch.Tensor, w8: torch.Tensor, col_scale: torch.Tensor, bias: Optional[torch.Tensor] = None,
               act: int = ACT_NONE, out_dtype: torch.dtype = torch.float16) -> torch.Tensor:
    """``out = act(row_scale[:, None] * col_scale[None, :] * (a8 @ w8.T) + bias)`` on E4M3 operands (``csvit_linear_fp8``): ``a8 [M, K]``
    with per-row scales (``layernorm_post(..., copy_dtype=torch.float8_e4m3fn)``), ``w8 [N, K]`` with per-channel scales
    (:func:`quantize_weight_fp8`); fp32 accumulation; ``out_dtype`` fp32, bf16 or fp16."""
    _dev(a8, row_scale, w8, col_scale, bias)
    M, K, lda = _fp8_operand("linear_fp8", a8, row_scale, "a8")
    N, K2, ldw = _fp8_operand("linear_fp8", w8, col_scale, "w8")
    if K != K2 or N % 32 != 0:
        raise ValueError(f"linear_fp8: A {tuple(a8.shape)} vs W {tuple(w8.shape)} (N must be a multiple of 32)")
    if bias is not None and (bias.dtype != torch.float32 or bias.numel() != N or not bias.is_contiguous()):
        raise ValueError("linear_fp8: bias must be contiguous float32 [N]")
    out = torch.empty(M, N, dtype=out_dtype, device=a8.device)
    _call("csvit_linear_fp8", a8.data_ptr(), lda, row_scale.data_ptr(), w8.data_ptr(), ldw, col_scale.data_ptr(), M, N, K, _p(bias), act,
          out.data_ptr(), N, _code(out_dtype), _stream(), flops=2.0 * M * N * K)
    return out


def swinv2_qkv_fp8(a8: torch.Tensor, row_scale: torch.Tensor, w8: torch.Tensor, col_scale: torch.Tensor, bias: Optional[torch.Tensor],
                   qscale_log2: torch.Tensor, out_dtype: torch.dtype = torch.float16) -> torch.Tensor:
    """:func:`swinv2_qkv` on E4M3 operands (``csvit_swinv2_qkv_fp8``): the accumulator is dequantised by ``row_scale [M]`` and
    ``col_scale [3C]`` before the bias and the cosine normalisation; 16-bit ``qkv [M, 3C]``."""
    _dev(a8, row_scale, w8, col_scale, bias, qscale_log2)
    M, K, lda = _fp8_operand("swinv2_qkv_fp8", a8, row_scale, "a8")
    N, K2, ldw = _fp8_operand("swinv2_qkv_fp8", w8, col_scale, "w8")
    C = N // 3
    if K2 != K or N != 3 * C or C % 32 != 0 or out_dtype not in (torch.float16, torch.bfloat16):
        raise ValueError("swinv2_qkv_fp8: a8 [M, K] and w8 [3C, K] (C a multiple of 32), 16-bit out_dtype")
    if qscale_log2.dtype != torch.float32 or qscale_log2.numel() != C // 32 or not qscale_log2.is_contiguous():
        raise ValueError("swinv2_qkv_fp8: qscale_log2 must be contiguous float32 [C / 32]")
    if bias is not None and (bias.dtype != torch.float32 or bias.numel() != N or not bias.is_contiguous()):
        raise ValueError("swinv2_qkv_fp8: bias must be contiguous float32 [3C]")
    out = torch.empty(M, N, dtype=out_dtype, device=a8.device)
    _call("csvit_swinv2_qkv_fp8", a8.data_ptr(), lda, row_scale.data_ptr(), w8.data_ptr(), ldw, col_scale.data_ptr(), M, C, K, _p(bias),
          qscale_log2.data_ptr(), out.data_ptr(), N, _code(out_dtype), _stream(), flops=2.0 * M * N * K,
          nbytes=float(a8.numel() + w8.numel() + 2 * out.numel()))
    return out


def quantize_weight_fp8(w: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per-output-channel E4M3 form of a Linear weight ``[N, K]`` (a one-time pack, like the 16-bit weight copies):
    ``wscale[n] = amax |w[n, :]| / 448``, ``w8 = e4m3(w / wscale)``; an all-zero row gets scale 0 and a zero row."""
    w = w.detach().float()
    amax = w.abs().amax(dim=1)
    scale = amax / torch.full_like(amax, E4M3_MAX)      # correctly rounded (a Python-scalar divisor becomes a reciprocal multiply)
    q = torch.where(amax[:, None] > 0, w / torch.where(scale > 0, scale, torch.ones_like(scale))[:, None], torch.zeros_like(w))
    return q.clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).contiguous(), scale.contiguous()


MLP_FUSED_WIDTHS = (128, 256)


def mlp_fused(xn: torch.Tensor, w1: torch.Tensor, b1: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """In place ``x += GELU(xn @ w1.T + b1) @ w2.T + b2`` without materialising the hidden tensor (``csvit_mlp_fused``)."""
    _dev(xn, w1, b1, w2, b2, x)
    M, C, ldxn = _rows2d(xn)
    if w1.shape != (4 * C, C) or w2.shape != (C, 4 * C) or x.shape != (M, C) or x.dtype != torch.float32:
        raise ValueError("mlp_fused: shape mismatch")
    if not (xn.dtype == w1.dtype == w2.dtype) or xn.dtype not in (torch.bfloat16, torch.float16):
        raise ValueError("mlp_fused: xn / w1 / w2 must share a 16-bit dtype")
    _call("csvit_mlp_fused", xn.data_ptr(), ldxn, w1.data_ptr(), w1.stride(0), b1.data_ptr(), w2.data_ptr(), w2.stride(0),
          b2.data_ptr(), x.data_ptr(), x.stride(0), _code(xn.dtype), M, C, _stream(), flops=16.0 * M * C * C)
    return x


# ---------------------------------------------------------------------------------------------- attention
ATTN_FUSED_WIDTHS = (128, 256)
_LOG2E = 1.4426950408889634


def pack_attn_fused(wq: torch.Tensor, wk: torch.Tensor, wv: torch.Tensor, bq: torch.Tensor, bk: torch.Tensor, bv: torch.Tensor,
                    table: torch.Tensor, rel_index: torch.Tensor, dtype: torch.dtype, gamma: torch.Tensor, beta: torch.Tensor):
    """Operands of ``csvit_swin_attn_fused`` from the HF parameters (one-time packing, layouts in include/csvit.h):
    per-head q|k|v weight rows ``[3C, C]`` (16 bit) with layernorm_before's ``gamma`` folded into the columns, the matching fp32
    bias (``b + W beta``, q part pre-scaled by log2(e)/sqrt(32)), and the fp16 relative-position-bias rows ``[heads*49, 56]``
    (query-slot-major, log2 domain)."""
    C = wq.shape[0]
    heads = C // 32
    g64, be64 = gamma.detach().double(), beta.detach().double()
    fold_w = lambda w_: (w_.detach().double() * g64[None, :]).float()
    fold_b = lambda w_, b_: (b_.detach().double() + w_.detach().double() @ be64).float()
    w = torch.stack([fold_w(wq).view(heads, 32, C), fold_w(wk).view(heads, 32, C), fold_w(wv).view(heads, 32, C)], 1)
    qs = _LOG2E / 32.0 ** 0.5
    b = torch.stack([fold_b(wq, bq).view(heads, 32) * qs, fold_b(wk, bk).view(heads, 32), fold_b(wv, bv).view(heads, 32)], 1)
    return w.reshape(3 * C, C).to(dtype).contiguous(), b.reshape(3 * C).contiguous(), pack_rel_bias_log2(table, rel_index)


def pack_rel_bias_log2(table: torch.Tensor, rel_index: torch.Tensor) -> torch.Tensor:
    """fp16 ``[heads*49, 56]`` relative-position-bias rows of the tcgen05 attention kernels: row ``49h + i`` holds
    ``log2(e) * table[rel_index[i, j], h]`` for key slots ``j < 49`` and zeros beyond (HF:swin/modeling_swin.py:437-444)."""
    heads = table.shape[1]
    L = rel_index.shape[0]
    if L != 49:
        raise ValueError("pack_rel_bias_log2: 7x7 windows only")
    bias = table.detach().float()[rel_index.reshape(-1).long()].view(L, L, heads).permute(2, 0, 1)      # [h, i, j]
    op = torch.zeros(heads, L, 56, dtype=torch.float32, device=table.device)
    op[:, :, :L] = bias * _LOG2E                                                                        # [h, query slot, key slot]
    return op.to(torch.float16).reshape(heads * L, 56).contiguous()


def pack_qkv_prescaled(wq, wk, wv, bq, bk, bv, dtype: torch.dtype):
    """Stacked ``[3C, C]`` Q/K/V weight (16 bit) and fp32 bias with ``log2(e)/sqrt(32)`` folded into the q rows, so that the
    logits of ``swin_attn_core(..., q_prescaled=True)`` come out of the MMA in the softmax's log2 domain."""
    qs = _LOG2E / 32.0 ** 0.5
    w = torch.cat([wq.detach().float() * qs, wk.detach().float(), wv.detach().float()], 0)
    b = torch.cat([bq.detach().float() * qs, bk.detach().float(), bv.detach().float()], 0)
    return w.to(dtype).contiguous(), b.contiguous()


def swin_attn_core(qkv: torch.Tensor, bias_log2: torch.Tensor, B: int, H: int, W: int, heads: int, ws: int, shift: int,
                   token_order: bool = False, q_prescaled: bool = False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Window-attention core on tcgen05 (``csvit_swin_attn_core``): window-ordered 16-bit qkv ``[B*H*W, 3C]`` -> context
    ``[B*H*W, C]`` in window order, or in token order (window_reverse + un-shift folded into the store)."""
    _dev(qkv, bias_log2, out)
    rows, C3, ld = _rows2d(qkv)
    C = C3 // 3
    if qkv.dtype not in (torch.bfloat16, torch.float16) or rows != B * H * W or C != heads * 32 or ws != 7:
        raise ValueError(f"swin_attn_core: needs 16-bit qkv [B*H*W, 3C] with head_dim 32 and 7x7 windows (rows={rows} C={C} heads={heads} ws={ws})")
    if bias_log2.dtype != torch.float16 or tuple(bias_log2.shape) != (heads * 49, 56) or not bias_log2.is_contiguous():
        raise ValueError("swin_attn_core: bias_log2 must be contiguous float16 [heads*49, 56] (pack_rel_bias_log2)")
    if out is None:
        out = torch.empty(rows, C, dtype=qkv.dtype, device=qkv.device)
    L = ws * ws
    _call("csvit_swin_attn_core", qkv.data_ptr(), ld, bias_log2.data_ptr(), out.data_ptr(), _code(qkv.dtype), B, H, W, C, heads, ws,
          shift, 1 if token_order else 0, 1 if q_prescaled else 0, _stream(),
          flops=float(rows) * 4.0 * L * C, nbytes=float(rows) * C * 8.0)
    return out


def swin_attn_fused(x: torch.Tensor, eps: float, wqkv_h: torch.Tensor, bqkv_h: torch.Tensor,
                    bias_op: torch.Tensor, B: int, H: int, W: int, heads: int, ws: int, shift: int,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """LayerNorm + shift/partition + Q/K/V + window attention + reverse/un-shift in one tcgen05 kernel (``csvit_swin_attn_fused``):
    x fp32 ``[B*H*W, C]`` -> token-ordered 16-bit context ``[B*H*W, C]`` (the output projection follows on plain rows)."""
    _dev(x, wqkv_h, bqkv_h, bias_op, out)
    if x.dtype != torch.float32 or not x.is_contiguous() or x.dim() != 2:
        raise ValueError("swin_attn_fused input must be contiguous float32 [B*H*W, C]")
    rows, C = x.shape
    if rows != B * H * W or C != heads * 32 or C not in ATTN_FUSED_WIDTHS:
        raise ValueError(f"swin_attn_fused: rows={rows} C={C} heads={heads} not supported (C in {ATTN_FUSED_WIDTHS}, head_dim 32)")
    if wqkv_h.dtype not in (torch.bfloat16, torch.float16) or tuple(wqkv_h.shape) != (3 * C, C) or not wqkv_h.is_contiguous():
        raise ValueError("swin_attn_fused: wqkv_h must be contiguous 16-bit [3C, C]")
    if bqkv_h.dtype != torch.float32 or bqkv_h.numel() != 3 * C or bias_op.dtype != torch.float16 or tuple(bias_op.shape) != (heads * 49, 56) or not bias_op.is_contiguous():
        raise ValueError("swin_attn_fused: bqkv_h must be float32 [3C] and bias_op contiguous float16 [heads*49, 56]")
    if out is None:
        out = torch.empty(rows, C, dtype=wqkv_h.dtype, device=x.device)
    L = ws * ws
    _call("csvit_swin_attn_fused", x.data_ptr(), float(eps), wqkv_h.data_ptr(), bqkv_h.data_ptr(),
          bias_op.data_ptr(), out.data_ptr(), _code(wqkv_h.dtype), B, H, W, C, heads, ws, shift, _stream(),
          flops=float(rows) * (6.0 * C * C + 4.0 * L * C), nbytes=float(rows) * C * 6.0)
    return out


def window_attention(qkv: torch.Tensor, bias_exp: Optional[torch.Tensor], B: int, H: int, W: int, heads: int, ws: int,
                     shift: int, bias_log2: Optional[torch.Tensor] = None, token_order: bool = False) -> torch.Tensor:
    """Window attention on window-ordered qkv ``[B*H*W, 3C]``: fp32 qkv runs the exact kernel of the validation mode with the
    ``expand_rel_bias`` table ``[h,L,L]``; 16-bit qkv runs the tcgen05 core (``swin_attn_core``) with the ``pack_rel_bias_log2`` table."""
    if qkv.dtype != torch.float32:
        if bias_log2 is None:
            raise ValueError("window_attention: 16-bit qkv needs bias_log2 (ops.pack_rel_bias_log2)")
        return swin_attn_core(qkv, bias_log2, B, H, W, heads, ws, shift, token_order=token_order)
    if token_order:
        raise ValueError("window_attention: token-ordered output is built for the 16-bit kernels only")
    _dev(qkv, bias_exp)
    rows, C3, ld = _rows2d(qkv)
    C = C3 // 3
    if ld != C3 or rows != B * H * W:
        raise ValueError("window_attention: qkv must be dense [B*H*W, 3C]")
    out = torch.empty(rows, C, dtype=qkv.dtype, device=qkv.device)
    _call("csvit_window_attention", qkv.data_ptr(), _p(bias_exp), out.data_ptr(), _code(qkv.dtype), B, H, W, C,
          heads, ws, shift, _stream(), nbytes=float(qkv.numel() + out.numel()) * qkv.element_size())
    return out


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, n_seq: int, Lq: int, S: int, heads: int,
              scale: float, key_start: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q ``[n_seq*Lq, D]`` (may be a column slice), k/v ``[n_seq*S, D]``; exact fp32 softmax attention.

    ``key_start`` (contiguous CUDA int32 ``[n_seq]``, values in ``[0, S-1]``, never read by the host): sequence s attends to its
    last ``S - key_start[s]`` keys only (``csvit_attention_ragged``), bit-identical to a call on those keys alone."""
    _dev(q, k, v, key_start)
    rq, D, ldq = _rows2d(q)
    rk, _, ldk = _rows2d(k)
    _, _, ldv = _rows2d(v)
    if rq != n_seq * Lq or rk != n_seq * S or D != heads * 32:
        raise ValueError("attention: shape mismatch (head_dim must be 32)")
    out = torch.empty(rq, D, dtype=q.dtype, device=q.device)
    if key_start is None:
        _call("csvit_attention", q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), _code(q.dtype), ldq, ldk, ldv, D,
              n_seq, Lq, S, heads, float(scale), _stream())
        return out
    if key_start.dtype != torch.int32 or tuple(key_start.shape) != (n_seq,) or not key_start.is_contiguous():
        raise ValueError(f"attention: key_start must be a contiguous int32 tensor of shape [{n_seq}], got {key_start.dtype} "
                         f"{tuple(key_start.shape)}")
    _call("csvit_attention_ragged", q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), _code(q.dtype), ldq, ldk, ldv, D,
          n_seq, Lq, S, heads, float(scale), key_start.data_ptr(), _stream())
    return out


def stream_update(tok: torch.Tensor, ids: torch.Tensor, reset: Optional[torch.Tensor], tokens: torch.Tensor, hist: torch.Tensor,
                  head: torch.Tensor, timestamp: Optional[torch.Tensor] = None, stamps: Optional[torch.Tensor] = None):
    """Per-step state update of a streaming session (``csvit_stream_update``) for the nb rows of a step, row r being stream
    ``ids[r]`` (int32 ``[nb]``, distinct, -1 = padding row).  ``tok`` fp32 ``[nb, 3, D]``: the rows' new spatial tokens; ``reset``
    bool ``[nb]`` or None; the state ``tokens`` fp32 ``[num_streams, W, 3, D]`` (a ring per stream), ``hist`` / ``head`` int32
    ``[num_streams]`` and, for the realtime model, ``timestamp`` fp32 ``[nb]`` with ``stamps`` fp32 ``[num_streams, W]``.

    Returns ``(window [nb, W, 3, D], win_stamps [nb, W] or None, key_start int32 [nb])``: each row's history right-aligned, zeros
    outside it (the newest timestamp in ``win_stamps``), and ``W - hist``.  ``window[:, :, q]`` is contiguous (the storage is
    ``[3, nb, W, D]``), so the per-encoder operands need no copy.  Only the streams in ``ids`` are read or written."""
    _dev(tok, ids, reset, tokens, hist, head, timestamp, stamps)
    nb = tok.shape[0]
    if tokens.dim() != 4 or tokens.shape[2] != 3:
        raise ValueError(f"stream_update: tokens must be [num_streams, W, 3, D], got {tuple(tokens.shape)}")
    B, W, _, D = tokens.shape
    f32 = lambda t, shape: t.dtype == torch.float32 and tuple(t.shape) == shape and t.is_contiguous()   # noqa: E731
    i32 = lambda t, shape: t.dtype == torch.int32 and tuple(t.shape) == shape and t.is_contiguous()     # noqa: E731
    if not (f32(tok, (nb, 3, D)) and f32(tokens, (B, W, 3, D)) and D % 4 == 0):
        raise ValueError(f"stream_update: tok and tokens must be contiguous float32 [nb, 3, D] and [num_streams, W, 3, D] with D % 4 == 0, "
                         f"got {tok.dtype} {tuple(tok.shape)} and {tokens.dtype} {tuple(tokens.shape)}")
    if not (i32(ids, (nb,)) and i32(hist, (B,)) and i32(head, (B,))):
        raise ValueError(f"stream_update: ids must be contiguous int32 [{nb}] and hist / head contiguous int32 [{B}]")
    if reset is not None and not (reset.dtype == torch.bool and tuple(reset.shape) == (nb,) and reset.is_contiguous()):
        raise ValueError(f"stream_update: reset must be a contiguous bool tensor of shape [{nb}]")
    if (timestamp is None) != (stamps is None) or (stamps is not None and not (f32(timestamp, (nb,)) and f32(stamps, (B, W)))):
        raise ValueError(f"stream_update: timestamp and stamps go together, contiguous float32 [{nb}] and [{B}, {W}]")
    window = torch.empty(3, nb, W, D, dtype=torch.float32, device=tok.device)
    win_stamps = None if stamps is None else torch.empty(nb, W, dtype=torch.float32, device=tok.device)
    key_start = torch.empty(nb, dtype=torch.int32, device=tok.device)
    if nb > 0:
        _call("csvit_stream_update", tok.data_ptr(), _p(timestamp), ids.data_ptr(), _p(reset), nb, tokens.data_ptr(), _p(stamps),
              hist.data_ptr(), head.data_ptr(), B, W, D, window.data_ptr(), _p(win_stamps), key_start.data_ptr(), _stream(),
              nbytes=4.0 * nb * (2 * W + 1) * 3 * D)
    return window.permute(1, 2, 0, 3), win_stamps, key_start


# ---------------------------------------------------------------------------------------------- SwinV2
COPY_NONE, COPY_IDENTITY, COPY_WINDOW, COPY_MERGE2X2 = 0, 1, 2, 3


def swinv2_window_attention(qkv: torch.Tensor, bias_tab: torch.Tensor, logit_scale: torch.Tensor, B: int, H: int, W: int, heads: int,
                            ws: int, shift: int, mask_repeat: int = 2, token_order: bool = False) -> torch.Tensor:
    """Scaled-cosine window attention (``csvit_swinv2_window_attention``): qkv window-ordered ``[B*H*W, 3C]``, ``bias_tab`` fp32
    ``[heads, (2ws-1)^2]``, ``logit_scale`` fp32 ``[heads]`` (already clamped and exponentiated)."""
    _dev(qkv, bias_tab, logit_scale)
    rows, C3, ld = _rows2d(qkv)
    C = C3 // 3
    if ld != C3 or rows != B * H * W:
        raise ValueError("swinv2_window_attention: qkv must be dense [B*H*W, 3C]")
    if bias_tab.dtype != torch.float32 or tuple(bias_tab.shape) != (heads, (2 * ws - 1) ** 2) or not bias_tab.is_contiguous():
        raise ValueError(f"swinv2_window_attention: bias table must be contiguous float32 [{heads}, {(2 * ws - 1) ** 2}]")
    if logit_scale.dtype != torch.float32 or logit_scale.numel() != heads or not logit_scale.is_contiguous():
        raise ValueError("swinv2_window_attention: logit_scale must be contiguous float32 [heads]")
    out = torch.empty(rows, C, dtype=qkv.dtype, device=qkv.device)
    L = ws * ws
    _call("csvit_swinv2_window_attention", qkv.data_ptr(), bias_tab.data_ptr(), logit_scale.data_ptr(), out.data_ptr(),
          _code(qkv.dtype), B, H, W, C, heads, ws, shift, mask_repeat, 1 if token_order else 0, _stream(),
          flops=4.0 * rows * L * C, nbytes=float(qkv.numel() + out.numel()) * qkv.element_size())
    return out


def swinv2_qkv(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], qscale_log2: torch.Tensor) -> torch.Tensor:
    """SwinV2 Q/K/V projection with both ``F.normalize`` and the logit scale folded into the epilogue (``csvit_swinv2_qkv``):
    ``a [M, K]`` and ``w [3C, K]`` 16 bit, ``qscale_log2`` fp32 ``[heads]`` = log2(e) * exp(min(logit_scale, ln 100))."""
    _dev(a, w, qscale_log2)
    M, K, lda = _rows2d(a)
    N, K2, ldw = _rows2d(w)
    C = N // 3
    if K2 != K or N != 3 * C or a.dtype != w.dtype or a.dtype not in (torch.float16, torch.bfloat16):
        raise ValueError("swinv2_qkv: a [M, K] and w [3C, K] must share one 16-bit dtype")
    if qscale_log2.dtype != torch.float32 or qscale_log2.numel() != C // 32 or not qscale_log2.is_contiguous():
        raise ValueError("swinv2_qkv: qscale_log2 must be contiguous float32 [C / 32]")
    if bias is not None and (bias.dtype != torch.float32 or bias.numel() != N or not bias.is_contiguous()):
        raise ValueError("swinv2_qkv: bias must be contiguous float32 [3C]")
    out = torch.empty(M, N, dtype=a.dtype, device=a.device)
    _call("csvit_swinv2_qkv", a.data_ptr(), lda, w.data_ptr(), ldw, _code(a.dtype), M, C, K, bias.data_ptr() if bias is not None else None,
          qscale_log2.data_ptr(), out.data_ptr(), N, _stream(), flops=2.0 * M * N * K,
          nbytes=float(a.numel() + w.numel() + out.numel()) * a.element_size())
    return out


def swinv2_qkv_train(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], qscale_log2: torch.Tensor
                     ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Training form of :func:`swinv2_qkv` (``csvit_swinv2_qkv_train``) -> (the same 16-bit ``qkv [M, 3C]``, fp32 ``rnorm [M, 2C / 32]``):
    ``rnorm`` holds 1 / max(|x|, 1e-12) of every q head, then every k head, of the pre-normalisation rows (:func:`swinv2_cosnorm_bwd`)."""
    _dev(a, w, bias, qscale_log2)
    M, K, lda = _rows2d(a)
    N, K2, ldw = _rows2d(w)
    C = N // 3
    if K2 != K or N != 3 * C or C % 32 != 0 or a.dtype != w.dtype or a.dtype not in (torch.float16, torch.bfloat16):
        raise ValueError("swinv2_qkv_train: a [M, K] and w [3C, K] (C a multiple of 32) must share one 16-bit dtype")
    if qscale_log2.dtype != torch.float32 or qscale_log2.numel() != C // 32 or not qscale_log2.is_contiguous():
        raise ValueError("swinv2_qkv_train: qscale_log2 must be contiguous float32 [C / 32]")
    if bias is not None and (bias.dtype != torch.float32 or bias.numel() != N or not bias.is_contiguous()):
        raise ValueError("swinv2_qkv_train: bias must be contiguous float32 [3C]")
    out = torch.empty(M, N, dtype=a.dtype, device=a.device)
    rnorm = torch.empty(M, 2 * C // 32, dtype=torch.float32, device=a.device)
    _call("csvit_swinv2_qkv_train", a.data_ptr(), lda, w.data_ptr(), ldw, _code(a.dtype), M, C, K, _p(bias), qscale_log2.data_ptr(),
          out.data_ptr(), N, rnorm.data_ptr(), _stream(), flops=2.0 * M * N * K,
          nbytes=float(a.numel() + w.numel() + out.numel()) * a.element_size() + 4.0 * rnorm.numel())
    return out, rnorm


def swinv2_cosnorm_bwd(qkv: torch.Tensor, rnorm: torch.Tensor, qscale_log2: torch.Tensor, dq2: torch.Tensor, dk: torch.Tensor,
                       dv: torch.Tensor, *, dqscale: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Backward of the cosine normalisation of :func:`swinv2_qkv_train` (``csvit_swinv2_cosnorm_bwd``) -> (16-bit ``dqkv [rows, 3C]`` =
    dq | dk | dv, the operand of the Q/K/V backward GEMMs; fp32 ``dqscale [C / 32]``, the gradient of ``qscale_log2``).  ``qkv`` /
    ``rnorm``: the forward's outputs; ``dq2, dk, dv``: dense 16-bit ``[rows, C]`` gradients of q2 / k_hat / v.  ``dqscale`` (optional) is a
    zeroed fp32 ``[C / 32]`` accumulator to add into."""
    _dev(qkv, rnorm, qscale_log2, dq2, dk, dv, dqscale)
    rows, C3 = qkv.shape
    C = C3 // 3
    dt = qkv.dtype
    if dt not in (torch.float16, torch.bfloat16) or C3 != 3 * C or C % 32 != 0 or C > 2048 or not qkv.is_contiguous():
        raise ValueError("swinv2_cosnorm_bwd: qkv must be contiguous 16-bit [rows, 3C] with C a multiple of 32, <= 2048")
    for name, t in (("dq2", dq2), ("dk", dk), ("dv", dv)):
        if t.dtype != dt or tuple(t.shape) != (rows, C) or not t.is_contiguous():
            raise ValueError(f"swinv2_cosnorm_bwd: {name} must be contiguous {dt} [{rows}, {C}]")
    if rnorm.dtype != torch.float32 or tuple(rnorm.shape) != (rows, C // 16) or not rnorm.is_contiguous():
        raise ValueError(f"swinv2_cosnorm_bwd: rnorm must be contiguous float32 [{rows}, {C // 16}]")
    if qscale_log2.dtype != torch.float32 or qscale_log2.numel() != C // 32 or not qscale_log2.is_contiguous():
        raise ValueError("swinv2_cosnorm_bwd: qscale_log2 must be contiguous float32 [C / 32]")
    if dqscale is None:
        dqscale = torch.zeros(C // 32, dtype=torch.float32, device=qkv.device)
    elif dqscale.dtype != torch.float32 or dqscale.numel() != C // 32 or not dqscale.is_contiguous():
        raise ValueError("swinv2_cosnorm_bwd: dqscale must be contiguous float32 [C / 32]")
    dqkv = torch.empty_like(qkv)
    _call("csvit_swinv2_cosnorm_bwd", qkv.data_ptr(), rnorm.data_ptr(), qscale_log2.data_ptr(), dq2.data_ptr(), dk.data_ptr(), dv.data_ptr(),
          dqkv.data_ptr(), dqscale.data_ptr(), _code(dt), rows, C, _stream(),
          nbytes=float(rows) * C * 8.0 * qkv.element_size() + 4.0 * rnorm.numel())
    return dqkv, dqscale


def swinv2_bias_log2(bias_tab: torch.Tensor) -> torch.Tensor:
    """``[heads, 31 * 31]`` table of window 16 (16 sigmoid(cpb_mlp)) -> the padded log2-domain ``[heads, 31, 48]`` table of
    ``csvit_swinv2_attn_tc``."""
    heads = bias_tab.shape[0]
    out = torch.zeros(heads, 31, 48, dtype=torch.float32, device=bias_tab.device)
    out[:, :, :31] = bias_tab.float().view(heads, 31, 31) * 1.4426950408889634
    return out.contiguous()


def swinv2_attn_tc(qkv: torch.Tensor, bias_log2: torch.Tensor, B: int, H: int, W: int, heads: int, shift: int, mask_repeat: int = 2,
                   token_order: bool = False) -> torch.Tensor:
    """tcgen05 cosine window attention for 16 x 16 windows (``csvit_swinv2_attn_tc``) on the output of :func:`swinv2_qkv`."""
    _dev(qkv, bias_log2)
    rows, C3, ld = _rows2d(qkv)
    C = C3 // 3
    if rows != B * H * W or qkv.dtype not in (torch.float16, torch.bfloat16):
        raise ValueError("swinv2_attn_tc: qkv must be 16-bit [B*H*W, 3C]")
    if bias_log2.dtype != torch.float32 or tuple(bias_log2.shape) != (heads, 31, 48) or not bias_log2.is_contiguous():
        raise ValueError(f"swinv2_attn_tc: bias table must be contiguous float32 [{heads}, 31, 48]")
    out = torch.empty(rows, C, dtype=qkv.dtype, device=qkv.device)
    _call("csvit_swinv2_attn_tc", qkv.data_ptr(), ld, bias_log2.data_ptr(), out.data_ptr(), _code(qkv.dtype), B, H, W, C, heads, shift,
          mask_repeat, 1 if token_order else 0, _stream(), flops=4.0 * rows * 256 * C,
          nbytes=float(qkv.numel() + out.numel()) * qkv.element_size())
    return out


def swinv2_attn_tc_train(qkv: torch.Tensor, bias_log2: torch.Tensor, B: int, H: int, W: int, heads: int, shift: int,
                         mask_repeat: int = 2) -> Tuple[torch.Tensor, torch.Tensor]:
    """Training forward of :func:`swinv2_attn_tc` (``csvit_swinv2_attn_tc_train``): ``qkv`` = q2 | k_hat | v 16-bit ``[B*H*W, 3C]`` in window
    order -> (window-ordered ``ctx [B*H*W, C]``, fp32 ``lse2 [B*nW, heads, 256]``), the row statistics of :func:`swinv2_attn_tc_bwd`."""
    _dev(qkv, bias_log2)
    rows, C3, ld = _rows2d(qkv)
    C = C3 // 3
    if rows != B * H * W or C3 != 3 * C or C != 32 * heads or qkv.dtype not in (torch.float16, torch.bfloat16):
        raise ValueError("swinv2_attn_tc_train: qkv must be 16-bit [B*H*W, 3C] with C = 32 heads")
    if bias_log2.dtype != torch.float32 or tuple(bias_log2.shape) != (heads, 31, 48) or not bias_log2.is_contiguous():
        raise ValueError(f"swinv2_attn_tc_train: bias table must be contiguous float32 [{heads}, 31, 48]")
    out = torch.empty(rows, C, dtype=qkv.dtype, device=qkv.device)
    lse2 = torch.empty(rows // 256, heads, 256, dtype=torch.float32, device=qkv.device)
    _call("csvit_swinv2_attn_tc_train", qkv.data_ptr(), ld, bias_log2.data_ptr(), out.data_ptr(), lse2.data_ptr(), _code(qkv.dtype), B, H,
          W, C, heads, shift, mask_repeat, _stream(), flops=4.0 * rows * 256 * C,
          nbytes=float(qkv.numel() + out.numel()) * qkv.element_size() + 4.0 * lse2.numel())
    return out, lse2


def swinv2_attn_tc_bwd(qkv: torch.Tensor, ctx: torch.Tensor, lse2: torch.Tensor, dctx: torch.Tensor, bias_log2: torch.Tensor, B: int, H: int,
                       W: int, heads: int, shift: int, mask_repeat: int = 2, *, out: Optional[Tuple[torch.Tensor, ...]] = None
                       ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """Backward of :func:`swinv2_attn_tc_train` on tcgen05 (``csvit_swinv2_attn_tc_bwd``) -> (dq2, dk_hat, dv) 16-bit ``[B*H*W, C]`` and
    fp32 ``dbias_log2 [heads, 31, 48]``.  ``ctx`` / ``dctx``: the forward's output and its gradient, dense 16-bit ``[B*H*W, C]``.
    ``out`` (optional): caller-provided ``(dq, dk, dv)`` tensors with contiguous ``[B*H*W, C]`` rows."""
    _dev(qkv, ctx, lse2, dctx, bias_log2)
    rows, C3, ld = _rows2d(qkv)
    C = C3 // 3
    dt = qkv.dtype
    if rows != B * H * W or C3 != 3 * C or C != 32 * heads or dt not in (torch.float16, torch.bfloat16):
        raise ValueError("swinv2_attn_tc_bwd: qkv must be 16-bit [B*H*W, 3C] with C = 32 heads")
    for name, t in (("ctx", ctx), ("dctx", dctx)):
        if t.dtype != dt or tuple(t.shape) != (rows, C) or not t.is_contiguous():
            raise ValueError(f"swinv2_attn_tc_bwd: {name} must be contiguous {dt} [{rows}, {C}]")
    if lse2.dtype != torch.float32 or tuple(lse2.shape) != (rows // 256, heads, 256) or not lse2.is_contiguous():
        raise ValueError(f"swinv2_attn_tc_bwd: lse2 must be contiguous float32 [{rows // 256}, {heads}, 256]")
    if bias_log2.dtype != torch.float32 or tuple(bias_log2.shape) != (heads, 31, 48) or not bias_log2.is_contiguous():
        raise ValueError(f"swinv2_attn_tc_bwd: bias table must be contiguous float32 [{heads}, 31, 48]")
    if out is None:
        out = tuple(torch.empty(rows, C, dtype=dt, device=qkv.device) for _ in range(3))
    for t in out:
        if t.dtype != dt or t.shape[-1] != C or t.numel() != rows * C or not t.is_contiguous():
            raise ValueError(f"swinv2_attn_tc_bwd: gradient outputs must be contiguous {dt} [{rows}, {C}]")
    dq, dk, dv = out
    dbias = torch.empty(heads, 31, 48, dtype=torch.float32, device=qkv.device)
    _call("csvit_swinv2_attn_tc_bwd", qkv.data_ptr(), ld, ctx.data_ptr(), dctx.data_ptr(), lse2.data_ptr(), bias_log2.data_ptr(),
          dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), dbias.data_ptr(), _code(dt), B, H, W, C, heads, shift, mask_repeat, _stream(),
          flops=10.0 * rows * 256 * C, nbytes=float(qkv.numel() + 6 * ctx.numel()) * qkv.element_size() + 4.0 * lse2.numel())
    return dq, dk, dv, dbias


def swinv2_bias8_log2(bias_tab: torch.Tensor) -> torch.Tensor:
    """``[heads, 15 * 15]`` table of window 8 (16 sigmoid(cpb_mlp)) -> the padded log2-domain ``[heads, 15, 24]`` table of the 8 x 8 kernels.
    The row pitch of 24 floats makes the kernels' shared-memory bias loads and gradient reductions conflict-free: the 32 lanes of a warp are
    4 window rows x 8 columns of queries, and rows 24 floats apart start on banks 0, 24, 16 and 8."""
    heads = bias_tab.shape[0]
    out = torch.zeros(heads, 15, 24, dtype=torch.float32, device=bias_tab.device)
    out[:, :, :15] = bias_tab.float().view(heads, 15, 15) * 1.4426950408889634
    return out.contiguous()


def _attn8_check(name: str, qkv: torch.Tensor, bias_log2: torch.Tensor, B: int, H: int, W: int, heads: int) -> Tuple[int, int, int]:
    rows, C3, ld = _rows2d(qkv)
    C = C3 // 3
    if rows != B * H * W or C3 != 3 * C or C != 32 * heads or qkv.dtype not in (torch.float16, torch.bfloat16):
        raise ValueError(f"{name}: qkv must be 16-bit [B*H*W, 3C] with C = 32 heads")
    if bias_log2.dtype != torch.float32 or tuple(bias_log2.shape) != (heads, 15, 24) or not bias_log2.is_contiguous():
        raise ValueError(f"{name}: bias table must be contiguous float32 [{heads}, 15, 24]")
    return rows, C, ld


def swinv2_attn8_tc(qkv: torch.Tensor, bias_log2: torch.Tensor, B: int, H: int, W: int, heads: int, shift: int, mask_repeat: int = 2,
                    token_order: bool = False) -> torch.Tensor:
    """tcgen05 cosine window attention for 8 x 8 windows (``csvit_swinv2_attn8_tc``) on the output of :func:`swinv2_qkv`; ``bias_log2``
    from :func:`swinv2_bias8_log2`."""
    _dev(qkv, bias_log2)
    rows, C, ld = _attn8_check("swinv2_attn8_tc", qkv, bias_log2, B, H, W, heads)
    out = torch.empty(rows, C, dtype=qkv.dtype, device=qkv.device)
    _call("csvit_swinv2_attn8_tc", qkv.data_ptr(), ld, bias_log2.data_ptr(), out.data_ptr(), _code(qkv.dtype), B, H, W, C, heads, shift,
          mask_repeat, 1 if token_order else 0, _stream(), flops=4.0 * rows * 64 * C,
          nbytes=float(qkv.numel() + out.numel()) * qkv.element_size())
    return out


def swinv2_attn8_tc_train(qkv: torch.Tensor, bias_log2: torch.Tensor, B: int, H: int, W: int, heads: int, shift: int,
                          mask_repeat: int = 2) -> Tuple[torch.Tensor, torch.Tensor]:
    """Training forward of :func:`swinv2_attn8_tc` (``csvit_swinv2_attn8_tc_train``) -> (window-ordered ``ctx [B*H*W, C]``, fp32
    ``lse2 [B*nW, heads, 64]``), the row statistics of :func:`swinv2_attn8_tc_bwd`."""
    _dev(qkv, bias_log2)
    rows, C, ld = _attn8_check("swinv2_attn8_tc_train", qkv, bias_log2, B, H, W, heads)
    out = torch.empty(rows, C, dtype=qkv.dtype, device=qkv.device)
    lse2 = torch.empty(rows // 64, heads, 64, dtype=torch.float32, device=qkv.device)
    _call("csvit_swinv2_attn8_tc_train", qkv.data_ptr(), ld, bias_log2.data_ptr(), out.data_ptr(), lse2.data_ptr(), _code(qkv.dtype), B,
          H, W, C, heads, shift, mask_repeat, _stream(), flops=4.0 * rows * 64 * C,
          nbytes=float(qkv.numel() + out.numel()) * qkv.element_size() + 4.0 * lse2.numel())
    return out, lse2


def swinv2_attn8_tc_bwd(qkv: torch.Tensor, ctx: torch.Tensor, lse2: torch.Tensor, dctx: torch.Tensor, bias_log2: torch.Tensor, B: int,
                        H: int, W: int, heads: int, shift: int, mask_repeat: int = 2, *, out: Optional[Tuple[torch.Tensor, ...]] = None
                        ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """Backward of :func:`swinv2_attn8_tc_train` on tcgen05 (``csvit_swinv2_attn8_tc_bwd``) -> (dq2, dk_hat, dv) 16-bit ``[B*H*W, C]`` and
    fp32 ``dbias_log2 [heads, 15, 24]``.  Arguments as :func:`swinv2_attn_tc_bwd`."""
    _dev(qkv, ctx, lse2, dctx, bias_log2)
    rows, C, ld = _attn8_check("swinv2_attn8_tc_bwd", qkv, bias_log2, B, H, W, heads)
    dt = qkv.dtype
    for name, t in (("ctx", ctx), ("dctx", dctx)):
        if t.dtype != dt or tuple(t.shape) != (rows, C) or not t.is_contiguous():
            raise ValueError(f"swinv2_attn8_tc_bwd: {name} must be contiguous {dt} [{rows}, {C}]")
    if lse2.dtype != torch.float32 or tuple(lse2.shape) != (rows // 64, heads, 64) or not lse2.is_contiguous():
        raise ValueError(f"swinv2_attn8_tc_bwd: lse2 must be contiguous float32 [{rows // 64}, {heads}, 64]")
    if out is None:
        out = tuple(torch.empty(rows, C, dtype=dt, device=qkv.device) for _ in range(3))
    for t in out:
        if t.dtype != dt or t.shape[-1] != C or t.numel() != rows * C or not t.is_contiguous():
            raise ValueError(f"swinv2_attn8_tc_bwd: gradient outputs must be contiguous {dt} [{rows}, {C}]")
    dq, dk, dv = out
    dbias = torch.empty(heads, 15, 24, dtype=torch.float32, device=qkv.device)
    _call("csvit_swinv2_attn8_tc_bwd", qkv.data_ptr(), ld, ctx.data_ptr(), dctx.data_ptr(), lse2.data_ptr(), bias_log2.data_ptr(),
          dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), dbias.data_ptr(), _code(dt), B, H, W, C, heads, shift, mask_repeat, _stream(),
          flops=10.0 * rows * 64 * C, nbytes=float(qkv.numel() + 6 * ctx.numel()) * qkv.element_size() + 4.0 * lse2.numel())
    return dq, dk, dv, dbias


def layernorm_post(y: torch.Tensor, resid: Optional[torch.Tensor], gamma: torch.Tensor, beta: torch.Tensor, eps: float, *,
                   out: Optional[torch.Tensor] = None, copy_mode: int = COPY_NONE, copy_dtype: torch.dtype = torch.bfloat16,
                   geom: Tuple[int, int, int, int] = (0, 0, 0, 0)) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """``out = (resid) + LayerNorm(y)`` in fp32 and, in the same pass, the copy of ``out`` laid out for the next GEMM
    (``csvit_layernorm_post``).  ``geom`` = (H, W, ws, shift) of the copy's window order / merge grid.  Returns (out, copy).
    ``copy_dtype=torch.float8_e4m3fn`` (identity / window copies, ``csvit_layernorm_post_fp8``): the copy is the E4M3 operand of an FP8
    GEMM and comes with its per-row scales, ``(out, (copy, row_scale))``: ``row_scale = amax / 448`` per copy row and
    ``copy = e4m3(out * (448 / amax))`` (0 and a zero row where amax = 0)."""
    _dev(y, resid, gamma, beta, out)
    rows, C, ldy = _rows2d(y)
    if y.dtype != torch.float32:
        raise ValueError("layernorm_post input must be float32")
    if resid is not None and (resid.dtype != torch.float32 or tuple(resid.shape) != (rows, C) or not resid.is_contiguous()):
        raise ValueError("layernorm_post: residual must be contiguous float32 [rows, C]")
    if gamma.numel() != C or beta.numel() != C:
        raise ValueError(f"layernorm_post affine width {gamma.numel()} != {C}")
    if out is None:
        out = torch.empty(rows, C, dtype=torch.float32, device=y.device)
    elif out.dtype != torch.float32 or tuple(out.shape) != (rows, C) or not out.is_contiguous():
        raise ValueError("layernorm_post: out must be contiguous float32 [rows, C]")
    H, W, ws, shift = geom
    if copy_dtype == torch.float8_e4m3fn:
        if copy_mode not in (COPY_IDENTITY, COPY_WINDOW) or C % 16 != 0:
            raise ValueError("layernorm_post: E4M3 copies are identity or window ordered, with C a multiple of 16")
        copy = torch.empty(rows, C, dtype=copy_dtype, device=y.device)
        row_scale = torch.empty(rows, dtype=torch.float32, device=y.device)
        _call("csvit_layernorm_post_fp8", y.data_ptr(), ldy, _p(resid), gamma.data_ptr(), beta.data_ptr(), float(eps), out.data_ptr(),
              copy.data_ptr(), row_scale.data_ptr(), C, copy_mode, rows, C, H, W, ws, shift, _stream(),
              nbytes=float(rows * C * (9 + (4 if resid is not None else 0)) + 4 * rows))
        return out, (copy, row_scale)
    copy = None
    if copy_mode == COPY_MERGE2X2:
        copy = torch.empty(rows // 4, 4 * C, dtype=copy_dtype, device=y.device)
    elif copy_mode != COPY_NONE:
        copy = torch.empty(rows, C, dtype=copy_dtype, device=y.device)
    _call("csvit_layernorm_post", y.data_ptr(), ldy, _p(resid), gamma.data_ptr(), beta.data_ptr(), float(eps), out.data_ptr(), _p(copy),
          _code(copy_dtype), 0 if copy is None else copy.stride(0), copy_mode, rows, C, H, W, ws, shift, _stream(),
          nbytes=float(rows * C * (8 + (4 if resid is not None else 0) + (0 if copy is None else copy.element_size()))))
    return out, copy


# ---------------------------------------------------------------------------------------------- training step (backward)
CR_SUM, CR_CENTERED, CR_DOT = 0, 1, 2
EW_GELU_FWD, EW_GELU_BWD, EW_RELU_BWD = 0, 1, 2


def gemm_ex(a: torch.Tensor, a_mn: bool, b: torch.Tensor, b_mn: bool, *, out: Optional[torch.Tensor] = None,
            out_dtype: Optional[torch.dtype] = None, accumulate: bool = False, impl: int = GEMM_TC, split_k: int = 0) -> torch.Tensor:
    """``out[M,N] (+)= sum_k A(m,k) B(n,k)``; ``a_mn`` / ``b_mn`` say the operand is stored ``[K, M|N]`` (see ``csvit_gemm_ex``)."""
    _dev(a, b, out)
    if a.dtype == torch.float32 and impl == GEMM_TC:   # kind::tf32 is K-major only: transpose the (small) fp32 operands
        if a_mn:
            a, a_mn = transpose(a), False
        if b_mn:
            b, b_mn = transpose(b), False
    r0, c0, lda = _rows2d(a)
    r1, c1, ldb = _rows2d(b)
    M, K = (c0, r0) if a_mn else (r0, c0)
    N, K2 = (c1, r1) if b_mn else (r1, c1)
    if K != K2 or a.dtype != b.dtype:
        raise ValueError(f"gemm_ex: A {tuple(a.shape)}/{a.dtype} (mn={a_mn}) vs B {tuple(b.shape)}/{b.dtype} (mn={b_mn})")
    if out is None:
        if accumulate:
            raise ValueError("gemm_ex: accumulate needs an output tensor")
        out = torch.empty(M, N, dtype=out_dtype or a.dtype, device=a.device)
    Mo, No, ldo = _rows2d(out)
    if (Mo, No) != (M, N):
        raise ValueError("gemm_ex: output shape mismatch")
    _call("csvit_gemm_ex", a.data_ptr(), lda, int(a_mn), b.data_ptr(), ldb, int(b_mn), _code(a.dtype), M, N, K, out.data_ptr(), ldo,
          _code(out.dtype), int(accumulate), impl, split_k, _stream(), flops=2.0 * M * N * K)
    return out


def transpose(x: torch.Tensor) -> torch.Tensor:
    """fp32 ``[R, C]`` -> contiguous ``[C, R]`` (row pitch padded to a 16-byte multiple for TMA)."""
    _dev(x)
    R, C, ld = _rows2d(x)
    if x.dtype != torch.float32:
        raise TypeError("transpose: float32 only")
    parent = torch.empty(C, -(-R // 4) * 4, dtype=torch.float32, device=x.device)
    _call("csvit_transpose_f32", x.data_ptr(), ld, parent.data_ptr(), parent.stride(0), R, C, _stream())
    return parent[:, :R]


def col_reduce(a: torch.Tensor, mode: int = CR_SUM, *, b: Optional[torch.Tensor] = None, center: Optional[torch.Tensor] = None,
               window: Optional[Tuple[int, int, int, int]] = None, copy_dtype: Optional[torch.dtype] = None, sums: bool = True,
               s1: Optional[torch.Tensor] = None):
    """Column sums of ``a [rows, C]`` (+ second moment / dot, see ``csvit_col_reduce``) and, with ``copy_dtype``, a converted
    (optionally window-gathered) copy of the rows.  Returns ``(s1, s2, copy)`` with ``None`` for the parts not requested."""
    _dev(a, b, center)
    rows, C, lda = _rows2d(a)
    if s1 is None:          # a caller-provided s1 must already be zeroed (slices of one zero-filled workspace save launches)
        s1 = torch.zeros(C, dtype=torch.float32, device=a.device) if sums else None
    s2 = torch.zeros(C, dtype=torch.float32, device=a.device) if sums and mode != CR_SUM else None
    copy = torch.empty(rows, C, dtype=copy_dtype, device=a.device) if copy_dtype is not None else None
    ldb = 0
    if b is not None:
        if b.dtype != torch.float32 or b.shape != a.shape:
            raise ValueError("col_reduce: second operand must be float32 with the same shape")
        ldb = _rows2d(b)[2]
    H, W, ws, shift = window if window is not None else (0, 0, 0, 0)
    _call("csvit_col_reduce", a.data_ptr(), _code(a.dtype), lda, _p(b), ldb, _p(center), mode, rows, C,
          LN_WINDOW if window is not None else LN_IDENTITY, H, W, ws, shift, _p(copy), _code(copy_dtype or torch.float32),
          C, _p(s1), _p(s2), _stream())
    return s1, s2, copy


def row_scale_add(x: Optional[torch.Tensor], y: torch.Tensor, s: torch.Tensor, group_rows: int) -> torch.Tensor:
    """``x + s[row // group_rows] * y`` (``x`` may be None) on dense fp32 ``[rows, C]`` tensors (``csvit_row_scale_add``)."""
    _dev(x, y, s)
    rows, C = y.shape
    if y.dtype != torch.float32 or not y.is_contiguous() or (x is not None and (x.dtype != torch.float32 or x.shape != y.shape or not x.is_contiguous())):
        raise ValueError("row_scale_add: dense float32 operands of one shape")
    if s.dtype != torch.float32 or not s.is_contiguous() or s.numel() * group_rows != rows:
        raise ValueError("row_scale_add: s must be contiguous float32 with rows / group_rows entries")
    out = torch.empty_like(y)
    _call("csvit_row_scale_add", _p(x), y.data_ptr(), s.data_ptr(), out.data_ptr(), rows, C, group_rows, _stream())
    return out


def eltwise(op: int, a: torch.Tensor, b: Optional[torch.Tensor] = None) -> torch.Tensor:
    _dev(a, b)
    if not a.is_contiguous() or (b is not None and (not b.is_contiguous() or b.dtype != a.dtype or b.shape != a.shape)):
        raise ValueError("eltwise: operands must be contiguous with the same shape and dtype")
    out = torch.empty_like(a)
    _call("csvit_eltwise", op, a.data_ptr(), _p(b), out.data_ptr(), _code(a.dtype), a.numel(), _stream())
    return out


def affine2_rows(dy: torch.Tensor, x: torch.Tensor, a: torch.Tensor, b: torch.Tensor, c0: torch.Tensor,
                 resid: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``a[c]*dy + b[c]*x + c0[c] (+ resid)`` on dense fp32 ``[rows, C]`` tensors (BatchNorm1d backward)."""
    _dev(dy, x, a, b, c0, resid)
    for t in (dy, x, resid):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or t.shape != dy.shape):
            raise ValueError("affine2_rows: dense float32 operands of one shape")
    rows, C = dy.shape
    out = torch.empty_like(dy)
    _call("csvit_affine2_rows", dy.data_ptr(), x.data_ptr(), a.data_ptr(), b.data_ptr(), c0.data_ptr(), _p(resid), out.data_ptr(),
          rows, C, _stream())
    return out


def layernorm_bwd(x: torch.Tensor, dy: torch.Tensor, gamma: torch.Tensor, eps: float, *, mode: int = LN_IDENTITY,
                  grid: Tuple[int, int] = (0, 0), ws: int = 0, shift: int = 0, dres: Optional[torch.Tensor] = None,
                  dgamma: Optional[torch.Tensor] = None, dbeta: Optional[torch.Tensor] = None):
    """Backward of ``layernorm``: returns ``(dx [rows_in, C] fp32 = dres + dLN, dgamma, dbeta)``."""
    _dev(x, dy, gamma, dres)
    if x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("layernorm_bwd: x must be contiguous float32")
    rows_in, C = x.shape
    rows, width, ldy = _rows2d(dy)
    if (mode == LN_MERGE2X2 and (rows != rows_in // 4 or width != 4 * C)) or (mode != LN_MERGE2X2 and (rows != rows_in or width != C)):
        raise ValueError("layernorm_bwd: dy shape does not match the forward output")
    if dres is not None and (dres.dtype != torch.float32 or dres.shape != x.shape or not dres.is_contiguous()):
        raise ValueError("layernorm_bwd: dres must be contiguous float32 of x's shape")
    dx = torch.empty_like(x)
    if (dgamma is None) != (dbeta is None):
        raise ValueError("layernorm_bwd: pass both dgamma and dbeta accumulators or neither")
    if dgamma is None:      # caller-provided accumulators must already be zeroed
        dgamma = torch.zeros(width, dtype=torch.float32, device=x.device)
        dbeta = torch.zeros(width, dtype=torch.float32, device=x.device)
    H, W = grid
    _call("csvit_layernorm_bwd", x.data_ptr(), dy.data_ptr(), _code(dy.dtype), ldy, gamma.data_ptr(), float(eps), rows, C, mode, H, W,
          ws, shift, _p(dres), dx.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), _stream())
    return dx, dgamma, dbeta


def attention_bwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, dout: torch.Tensor, n_seq: int, Lq: int, S: int, heads: int,
                  scale: float, *, bias: Optional[torch.Tensor] = None, mask: Optional[Tuple[int, int, int, int]] = None,
                  dq: Optional[torch.Tensor] = None, dk: Optional[torch.Tensor] = None, dv: Optional[torch.Tensor] = None,
                  dbias: Optional[torch.Tensor] = None):
    """Backward of ``attention`` / ``window_attention``.  q/k/v/dout (and dq/dk/dv when given) may be column slices.
    Returns ``(dq, dk, dv, dbias or None)``."""
    _dev(q, k, v, dout, bias, dq, dk, dv)
    rq, D, ldq = _rows2d(q)
    rk, _, ldk = _rows2d(k)
    ldv, ldo = _rows2d(v)[2], _rows2d(dout)[2]
    if rq != n_seq * Lq or rk != n_seq * S or D != heads * 32 or dout.shape != q.shape:
        raise ValueError("attention_bwd: shape mismatch (head_dim must be 32)")
    dq = torch.empty(rq, D, dtype=q.dtype, device=q.device) if dq is None else dq
    dk = torch.empty(rk, D, dtype=q.dtype, device=q.device) if dk is None else dk
    dv = torch.empty(rk, D, dtype=q.dtype, device=q.device) if dv is None else dv
    if dbias is None and bias is not None:   # a caller-provided dbias must already be zeroed
        dbias = torch.zeros(heads, Lq, S, dtype=torch.float32, device=q.device)
    mH, mW, mws, msh = mask if mask is not None else (0, 0, 0, 0)
    _call("csvit_attention_bwd", q.data_ptr(), k.data_ptr(), v.data_ptr(), dout.data_ptr(), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(),
          _code(q.dtype), ldq, ldk, ldv, ldo, dq.stride(0), dk.stride(0), dv.stride(0), n_seq, Lq, S, heads, float(scale),
          _p(bias), _p(dbias), mH, mW, mws, msh, _stream())
    return dq, dk, dv, dbias


# ---------------------------------------------------------------------------------------------- host-side maps
def host_maps(H: int, W: int, ws: int, shift: int):
    """CPU evaluation of the kernels' closed-form integer maps (same inline functions, compiled for the host).
    Returns ``(window_index_map [H*W] int32, shift_mask [nW,L,L] fp32)`` as CPU tensors; needs no GPU."""
    nW, L = (H // ws) * (W // ws), ws * ws
    idx = torch.empty(H * W, dtype=torch.int32)
    mask = torch.empty(nW, L, L, dtype=torch.float32)
    lib = _lib.load()
    _lib.check(lib.csvit_host_window_index_map(H, W, ws, shift, idx.data_ptr()))
    _lib.check(lib.csvit_host_shift_mask(H, W, ws, shift, mask.data_ptr()))
    return idx, mask


def host_rel_pos_index(ws: int) -> torch.Tensor:
    out = torch.empty(ws * ws, ws * ws, dtype=torch.int32)
    _lib.check(_lib.load().csvit_host_rel_pos_index(ws, out.data_ptr()))
    return out


def host_merge_index_map(H: int, W: int) -> torch.Tensor:
    out = torch.empty((H // 2) * (W // 2), 4, dtype=torch.int32)
    _lib.check(_lib.load().csvit_host_merge_index_map(H, W, out.data_ptr()))
    return out


def set_gemm_tuning(cluster: int = 0, tma_store: int = -1, max_ctas: int = 0, pair: int = -1) -> None:
    """Ablation knobs of the GEMM engine (see ``csvit_set_gemm_tuning``); defaults restore automatic choices."""
    _lib.check(_lib.load().csvit_set_gemm_tuning(cluster, tma_store, max_ctas, pair))


# ---------------------------------------------------------------------------------------------- fp32 tail
def rot6d_to_axis_angle(d6: torch.Tensor) -> torch.Tensor:
    """``[..., 6]`` 6D rotations -> ``[..., 3]`` axis-angle (``csvit_rot6d_to_axis_angle``): ``matrix_to_axis_angle(
    rotation_6d_to_matrix(d6))`` of cs_vit.utils.geometry in one kernel."""
    _dev(d6)
    if d6.dtype != torch.float32 or d6.shape[-1] != 6:
        raise ValueError("rot6d_to_axis_angle: float32 [..., 6]")
    d6 = d6.contiguous()
    out = torch.empty(d6.shape[:-1] + (3,), dtype=torch.float32, device=d6.device)
    _call("csvit_rot6d_to_axis_angle", d6.data_ptr(), out.data_ptr(), d6.numel() // 6, _stream())
    return out


def mano_fk(pose: torch.Tensor, betas: torch.Tensor, root_norm: torch.Tensor, layer: dict, j_out: torch.Tensor, edges, rodrigues_mode: int = 0):
    """``Poser._pose_fk`` in one kernel (``csvit_mano_fk``).  ``pose [n,48]``, ``betas [n,10]``, ``root_norm [n,3]``;
    ``layer``: contiguous fp32 device buffers ``v_template, shapedirs, j_regressor, lbs_weights`` (+ optional ``posedirs``,
    ``pose_mean``) and the python list ``parents``; ``j_out [21,778]``; ``edges``: 20 joint pairs.
    Returns ``(joint_cam [n,21,3], verts_cam [n,778,3], root_transl [n,3])`` in millimetres."""
    import ctypes
    need = [pose, betas, root_norm, layer["v_template"], layer["shapedirs"], layer["j_regressor"], layer["lbs_weights"], j_out]
    _dev(*need, layer.get("posedirs"), layer.get("pose_mean"))
    for t in need + [t for t in (layer.get("posedirs"), layer.get("pose_mean")) if t is not None]:
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError("mano_fk: contiguous float32 operands only")
    n = pose.shape[0]
    if tuple(pose.shape) != (n, 48) or tuple(betas.shape) != (n, 10) or tuple(root_norm.shape) != (n, 3) or tuple(j_out.shape) != (21, 778) or \
            tuple(layer["v_template"].shape) != (778, 3) or tuple(layer["shapedirs"].shape) != (778, 3, 10) or \
            tuple(layer["j_regressor"].shape) != (16, 778) or tuple(layer["lbs_weights"].shape) != (778, 16) or len(edges) != 20:
        raise ValueError("mano_fk: shape mismatch (MANO: 778 vertices, 16 joints, 10 betas; 21 output joints, 20 bones)")
    parents = (ctypes.c_int * 16)(*[int(x) for x in layer["parents"]])
    e40 = (ctypes.c_int * 40)(*[int(x) for ab in edges for x in ab])
    joint_cam = torch.empty(n, 21, 3, dtype=torch.float32, device=pose.device)
    verts_cam = torch.empty(n, 778, 3, dtype=torch.float32, device=pose.device)
    root = torch.empty(n, 3, dtype=torch.float32, device=pose.device)
    _call("csvit_mano_fk", pose.data_ptr(), betas.data_ptr(), root_norm.data_ptr(), layer["v_template"].data_ptr(), layer["shapedirs"].data_ptr(),
          _p(layer.get("posedirs")), _p(layer.get("pose_mean")), layer["j_regressor"].data_ptr(), layer["lbs_weights"].data_ptr(), j_out.data_ptr(),
          parents, e40, int(rodrigues_mode), joint_cam.data_ptr(), verts_cam.data_ptr(), root.data_ptr(), n, _stream())
    return joint_cam, verts_cam, root


# ---------------------------------------------------------------------------------------------- input pipeline
def crop_resize(frames: torch.Tensor, boxes: torch.Tensor, size: int = 224, expansion_ratio: float = 0.0):
    """On-device hand crops (``csvit_crop_resize``): ``frames`` fp32 ``[N,3,H,W]`` in [0,1] or uint8 ``[N,H,W,3]``; ``boxes`` fp32
    ``[N,4]`` xyxy.  ``expansion_ratio > 0``: the boxes are tight boxes, made square and expanded as
    ref:cs_vit/utils/img.py:358-370; returns ``(patches [N,3,size,size] fp32, square_boxes [N,4])`` - the ``img_tensor`` /
    ``square_bboxes`` arguments of ``Poser.predict_batch`` (add the frame dimension with ``[:, None]``)."""
    _dev(frames, boxes)
    u8 = frames.dtype == torch.uint8
    if u8:
        if frames.dim() != 4 or frames.shape[-1] != 3:
            raise ValueError("crop_resize: uint8 frames must be [N,H,W,3]")
        N, H, W = frames.shape[:3]
    elif frames.dtype == torch.float32:
        if frames.dim() != 4 or frames.shape[1] != 3:
            raise ValueError("crop_resize: float frames must be [N,3,H,W]")
        N, _, H, W = frames.shape
    else:
        raise TypeError(f"crop_resize: frames must be float32 or uint8, got {frames.dtype}")
    if not frames.is_contiguous() or boxes.dtype != torch.float32 or tuple(boxes.shape) != (N, 4) or not boxes.is_contiguous():
        raise ValueError("crop_resize: frames must be contiguous and boxes contiguous float32 [N,4]")
    out = torch.empty(N, 3, size, size, dtype=torch.float32, device=frames.device)
    square = torch.empty(N, 4, dtype=torch.float32, device=frames.device)
    _call("csvit_crop_resize", frames.data_ptr(), 1 if u8 else 0, N, H, W, boxes.data_ptr(), float(expansion_ratio), square.data_ptr(),
          out.data_ptr(), size, _stream(), nbytes=float(out.numel()) * 4.0)
    return out, square


# ---------------------------------------------------------------------------------------------- multi-GPU
ALLREDUCE_FLAG_BYTES = 4096


def allreduce_f32(buf_ptrs, flag_ptrs, multicast_ptr: int, numel: int, rank: int, world: int, scale: float, ctas: int = 0) -> None:
    """In-place SUM * scale of one fp32 bucket held in symmetric memory by every rank (``csvit_allreduce_f32``), on the current
    stream.  ``buf_ptrs`` / ``flag_ptrs``: the bucket's / the flag region's device address on every rank (ints, rank order);
    ``multicast_ptr``: the bucket's NVSwitch multicast address or 0.  Collective: every rank calls it with the same arguments."""
    import ctypes
    if len(buf_ptrs) != world or len(flag_ptrs) != world:
        raise ValueError("allreduce_f32: need one buffer and one flag pointer per rank")
    bufs = (ctypes.c_void_p * world)(*[int(x) for x in buf_ptrs])
    flags = (ctypes.c_void_p * world)(*[int(x) for x in flag_ptrs])
    _call("csvit_allreduce_f32", bufs, flags, int(multicast_ptr) or None, int(numel), rank, world, float(scale), int(ctas), _stream(),
          nbytes=float(numel) * 4.0)
