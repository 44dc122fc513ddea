"""Attention building blocks of the CS-ViT head on the sm_100a kernels.

Same class names, constructor arguments and parameter names as ref:cs_vit/net/transformer_module.py
(``MHA`` :235-282, ``FeedForwardNetwork`` :285-297, ``EncoderBlock`` :300-319, ``DecoderBlock`` :322-353,
``CrossAttnDecoder`` :356-378, ``PositionalEncoding`` :16-81), so ``state_dict``s are interchangeable.  The
forwards are re-derived for the kernel library:

* Linear layers run on the tcgen05 GEMM engine with fp32 operands read as TF32 (the head's logits are
  multiplied by sqrt(head_dim) - quirk Q1 - which makes bf16 operands unusable, SURVEY.md §7 "Numerics");
  ``precision="fp32"`` switches to the exact-fp32 SIMT GEMM.
* Q/K/V share one GEMM when query and context coincide, K/V share one otherwise.
* The softmax core is the exact-fp32 short-sequence kernel (``csvit_attention``).
* Eval-mode ``BatchNorm1d`` over channels is a per-channel affine map (``csvit_affine_rows``); the two
  transposes of the reference disappear.
* Residual adds are GEMM epilogues.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn

from .. import autograd as ag
from .. import ops
from ._pack import PackCache, fold_batchnorm


class _KernelModule(nn.Module):
    """Common plumbing: precision switch, packed-parameter cache, CUDA-only guard."""

    precision: str = "bf16"

    def __init__(self):
        super().__init__()
        self._pack = PackCache()

    @property
    def _impl(self) -> int:
        return ops.GEMM_SIMT if self.precision == "fp32" else ops.GEMM_TC

    def _bn(self, name: str, bn: nn.BatchNorm1d):
        return self._pack.get(name, [bn.weight, bn.bias, bn.running_mean, bn.running_var], lambda: fold_batchnorm(bn))

    def _norm(self, name: str, bn: nn.BatchNorm1d, x2d: torch.Tensor, grad: bool) -> torch.Tensor:
        """BatchNorm1d over channels of ``[rows, C]``: batch statistics in train mode, folded running statistics in eval
        mode; differentiable when ``grad`` (ref:cs_vit/net/transformer_module.py:306-307,312,316)."""
        if grad or bn.training:
            return ag.batchnorm(x2d, bn)
        return ops.affine_rows(x2d, *self._bn(name, bn))

    def _grad(self, *tensors: Optional[torch.Tensor]) -> bool:
        """True when this call must be differentiable: autograd is on and an input or a parameter of the module wants a gradient."""
        if not torch.is_grad_enabled():
            return False
        return any(t is not None and t.requires_grad for t in tensors) or any(p.requires_grad for p in self.parameters())

    @staticmethod
    def _check(x: torch.Tensor) -> None:
        if not x.is_cuda:
            raise RuntimeError("cs_vit.net runs on CUDA tensors only (there is no CPU fallback)")


def _flat(x: torch.Tensor) -> torch.Tensor:
    return x.reshape(-1, x.shape[-1]).float().contiguous()


class PositionalEncoding(_KernelModule):
    def __init__(self, d_model: int, max_len: int = 512, mode: str = "absolute"):
        super().__init__()
        self.mode, self.d_model = mode, d_model
        if mode == "absolute":
            self.pe = nn.Embedding(max_len, d_model)
            self.register_buffer("positions", torch.arange(max_len))
        elif mode == "trope":
            if d_model % 2 != 0:
                raise ValueError(f"d_model must be even for RoPE, but got {d_model}")
            self.register_buffer("inv_freq", 1.0 / (10000 ** (torch.arange(0, d_model, 2).float() / d_model)))
        else:
            raise ValueError(f"Unsupported position mode: {mode}")

    def forward(self, x: torch.Tensor, t: Optional[torch.Tensor] = None, positions: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``positions`` (absolute mode, inference only; int64 ``[B, T]``): the embedding row each token gets instead of its index."""
        if self.mode == "absolute":
            if positions is not None:
                return x + self.pe.weight[positions]
            return x + self.pe.weight[: x.size(1)][None]
        if t is None:
            raise ValueError("t must be provided for 'trope' mode")
        # rotate input pairs (2i, 2i+1) by (t_last - t) * inv_freq_i   (quirk Q6)
        ang = (t[:, -1:] - t).float()[..., None] * self.inv_freq[None, None]
        c, s = torch.cos(ang), torch.sin(ang)
        a, b = x.reshape(*x.shape[:-1], -1, 2).unbind(-1)
        return torch.stack([a * c - b * s, a * s + b * c], dim=-1).flatten(-2)


class MHA(_KernelModule):
    def __init__(self, embed_dim: int, num_heads: int):
        super().__init__()
        assert embed_dim % num_heads == 0, "embed_dim must be divisible by num_heads"
        self.embed_dim, self.num_heads = embed_dim, num_heads
        self.head_dim = embed_dim // num_heads
        if self.head_dim != 32:
            raise NotImplementedError("the attention kernels require head_dim == 32")
        self.inv_sqrt_head_dim = 1 / (self.head_dim ** 0.5)
        self.query = nn.Linear(embed_dim, embed_dim)
        self.key = nn.Linear(embed_dim, embed_dim)
        self.value = nn.Linear(embed_dim, embed_dim)
        self.output = nn.Linear(embed_dim, embed_dim)

    def _stack(self, name: str, mods):
        ws = [m.weight for m in mods]
        bs = [m.bias for m in mods]
        w = self._pack.get(name + "w", ws, lambda: torch.cat([t.detach().float() for t in ws], 0).contiguous())
        b = self._pack.get(name + "b", bs, lambda: torch.cat([t.detach().float() for t in bs], 0).contiguous())
        return w, b

    def attend(self, x2d: torch.Tensor, ctx2d: Optional[torch.Tensor], n: int, L: int, S: int, resid: Optional[torch.Tensor],
               key_start: Optional[torch.Tensor] = None):
        """x2d [n*L, D]; ctx2d [n*S, D] or None for self-attention.  Returns resid + MHA(x, ctx) as [n*L, D].
        ``key_start`` (int32 [n], inference only): sequence i attends to its keys ``key_start[i]:S`` only (``ops.attention``)."""
        D, h = self.embed_dim, self.num_heads
        scale = 1.0 / self.inv_sqrt_head_dim      # logits are DIVIDED by 1/sqrt(d)  (ref :273, quirk Q1)
        if self._grad(x2d, ctx2d, resid):
            if key_start is not None:
                raise ValueError("MHA: key_start is an inference-only option (the differentiable path attends to every key)")
            return self._attend_grad(x2d, ctx2d, n, L, S, resid, scale)
        if ctx2d is None:
            w, b = self._stack("qkv", [self.query, self.key, self.value])
            qkv = ops.linear(x2d, w, b, impl=self._impl)
            q, k, v = qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:]
        else:
            wq, bq = self._stack("q", [self.query])
            wkv, bkv = self._stack("kv", [self.key, self.value])
            q = ops.linear(x2d, wq, bq, impl=self._impl)
            kv = ops.linear(ctx2d, wkv, bkv, impl=self._impl)
            k, v = kv[:, :D], kv[:, D:]
        ctx = ops.attention(q, k, v, n, L, S, h, scale, key_start=key_start)
        wo, bo = self._stack("o", [self.output])
        return ops.linear(ctx, wo, bo, resid=resid, impl=self._impl)

    def _attend_grad(self, x2d, ctx2d, n, L, S, resid, scale):
        """Same computation through the differentiable ops (cs_vit/autograd.py); Q/K/V stay separate parameters, so
        the stacked weight is a differentiable ``cat``."""
        D, h = self.embed_dim, self.num_heads
        q_, k_, v_ = self.query, self.key, self.value
        if ctx2d is None:
            qkv = ag.linear(x2d, torch.cat([q_.weight, k_.weight, v_.weight], 0), torch.cat([q_.bias, k_.bias, v_.bias], 0), impl=self._impl)
            c = ag.attention_packed(qkv, D, n, L, h, scale)
        else:
            q = ag.linear(x2d, q_.weight, q_.bias, impl=self._impl)
            kv = ag.linear(ctx2d, torch.cat([k_.weight, v_.weight], 0), torch.cat([k_.bias, v_.bias], 0), impl=self._impl)
            c = ag.attention_cross(q, kv, D, n, L, S, h, scale)
        return ag.linear(c, self.output.weight, self.output.bias, resid=resid, impl=self._impl)

    def forward(self, x: torch.Tensor, ctx: torch.Tensor) -> torch.Tensor:
        self._check(x)
        n, L, D = x.shape
        same = ctx is x
        out = self.attend(_flat(x), None if same else _flat(ctx), n, L, ctx.shape[1], None)
        return out.view(n, L, D)


class FeedForwardNetwork(_KernelModule):
    def __init__(self, dim: int):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(dim, 4 * dim), nn.GELU(), nn.Linear(4 * dim, dim))

    def run(self, y2d: torch.Tensor, resid: Optional[torch.Tensor]) -> torch.Tensor:
        f1, f2 = self.net[0], self.net[2]
        if self._grad(y2d, resid):
            hid = ag.gelu(ag.linear(y2d, f1.weight, f1.bias, impl=self._impl))
            return ag.linear(hid, f2.weight, f2.bias, resid=resid, impl=self._impl)
        hid = ops.linear(y2d, f1.weight.detach().float(), f1.bias.detach().float(), act=ops.ACT_GELU, impl=self._impl)
        return ops.linear(hid, f2.weight.detach().float(), f2.bias.detach().float(), resid=resid, impl=self._impl)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        self._check(x)
        return self.run(_flat(x), None).view(x.shape)


class EncoderBlock(_KernelModule):
    def __init__(self, dim: int, num_heads: int):
        super().__init__()
        self.attn = MHA(dim, num_heads)
        self.ffn = FeedForwardNetwork(dim)
        self.norm1 = nn.BatchNorm1d(dim)
        self.norm2 = nn.BatchNorm1d(dim)

    def forward(self, x: torch.Tensor, key_start: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``key_start`` (int32 [n], inference only): sequence i attends to its tokens ``key_start[i]:L`` only."""
        self._check(x)
        n, L, D = x.shape
        x2 = _flat(x)
        g = self._grad(x)
        y = self._norm("n1", self.norm1, x2, g)
        x2 = self.attn.attend(y, None, n, L, L, x2, key_start=key_start)
        y = self._norm("n2", self.norm2, x2, g)
        return self.ffn.run(y, x2).view(n, L, D)

    def forward_queries(self, x: torch.Tensor, nq: int) -> torch.Tensor:
        """First ``nq`` tokens of ``forward(x)`` without computing the rest (inference only).

        The "encoder" spatial head returns ``layers[-1](z)[:, :3]`` (ref:cs_vit/net/ti_poser.py:94-97): with a single executed
        layer the other 49 output rows are dead.  Keys / values still need every token, but the query projection, the attention
        rows, the output projection, BatchNorm 2 and the FFN only run for the kept rows (eval-mode BatchNorm is row-wise, so
        the kept rows are bit-identical to the full computation): 0.28 instead of 1.32 GFLOP per image at D = 1024."""
        self._check(x)
        n, L, D = x.shape
        if self._grad(x) or self.norm1.training or self.norm2.training:
            return self.forward(x)[:, :nq]        # batch statistics couple the rows: no pruning in the training path
        mha = self.attn
        xq = x[:, :nq].reshape(n * nq, D).float().contiguous()
        y = ops.affine_rows(_flat(x), *self._bn("n1", self.norm1))
        yq = y.view(n, L, D)[:, :nq].reshape(n * nq, D).contiguous()
        wq, bq = mha._stack("q", [mha.query])
        wkv, bkv = mha._stack("kv", [mha.key, mha.value])
        q = ops.linear(yq, wq, bq, impl=self._impl)
        kv = ops.linear(y, wkv, bkv, impl=self._impl)
        c = ops.attention(q, kv[:, :D], kv[:, D:], n, nq, L, mha.num_heads, 1.0 / mha.inv_sqrt_head_dim)
        wo, bo = mha._stack("o", [mha.output])
        x2 = ops.linear(c, wo, bo, resid=xq, impl=self._impl)
        y2 = ops.affine_rows(x2, *self._bn("n2", self.norm2))
        return self.ffn.run(y2, x2).view(n, nq, D)


class DecoderBlock(_KernelModule):
    def __init__(self, dim: int, num_heads: int):
        super().__init__()
        self.self_atten = MHA(dim, num_heads)
        self.cross_atten = MHA(dim, num_heads)
        self.ffn = FeedForwardNetwork(dim)
        self.norm1 = nn.BatchNorm1d(dim)
        self.norm2 = nn.BatchNorm1d(dim)
        self.norm3 = nn.BatchNorm1d(dim)

    def forward(self, x: torch.Tensor, ref: torch.Tensor) -> torch.Tensor:
        self._check(x)
        n, L, D = x.shape
        x2, r2 = _flat(x), _flat(ref)
        g = self._grad(x, ref)
        y = self._norm("n1", self.norm1, x2, g)
        x2 = self.self_atten.attend(y, None, n, L, L, x2)
        y = self._norm("n2", self.norm2, x2, g)
        x2 = self.cross_atten.attend(y, r2, n, L, ref.shape[1], x2)     # ``ref`` is not normalised (ref :345-346)
        y = self._norm("n3", self.norm3, x2, g)
        return self.ffn.run(y, x2).view(n, L, D)


class CrossAttnDecoder(_KernelModule):
    def __init__(self, dim: int, num_heads: int):
        super().__init__()
        self.cross_atten = MHA(dim, num_heads)
        self.ffn = FeedForwardNetwork(dim)
        self.norm1 = nn.BatchNorm1d(dim)
        self.norm2 = nn.BatchNorm1d(dim)

    def forward(self, x: torch.Tensor, ref: torch.Tensor, key_start: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``key_start`` (int32 [n], inference only): sequence i cross-attends to ``ref[i, key_start[i]:]`` only."""
        self._check(x)
        n, L, D = x.shape
        x2, r2 = _flat(x), _flat(ref)
        g = self._grad(x, ref)
        y = self._norm("n1", self.norm1, x2, g)
        x2 = self.cross_atten.attend(y, r2, n, L, ref.shape[1], x2, key_start=key_start)
        y = self._norm("n2", self.norm2, x2, g)
        return self.ffn.run(y, x2).view(n, L, D)


def set_precision(module: nn.Module, precision: str) -> None:
    # "fp8" (swinv2 backbones, inference): the head's kernels run exactly as in "fp16" (they only tell "fp32" apart)
    if precision not in ("bf16", "fp16", "fp32", "fp8"):
        raise ValueError(f"precision must be 'bf16', 'fp16', 'fp32' or 'fp8', got {precision!r}")
    for m in module.modules():
        if isinstance(m, _KernelModule) or hasattr(m, "precision"):
            m.precision = precision
