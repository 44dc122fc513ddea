"""Backward passes of the hot path on the sm_100a kernels (BASELINE configs[3]: the finetune step).

The reference trains through torch autograd over its eager ops (``loss.backward()`` at ref:scripts/finetune.py:224, through
HF:swin/modeling_swin.py:591-653 and ref:cs_vit/net/transformer_module.py:250-378).  Here every differentiable stage of
the kernel path is a ``torch.autograd.Function`` whose backward is written against the C ABI: autograd only routes
gradients between stages and into ``param.grad`` (where DDP's bucket hooks pick them up); no ATen math runs inside.

* ``SwinBlockFn`` / ``PatchMergeFn`` / ``PatchEmbedFn`` / ``LayerNormFn`` - the backbone, one Function per block so that
  the residual-gradient adds are fused into the LayerNorm-backward kernel and the fp32 gradient stream is converted to a
  16-bit tensor-core operand in the same pass that reduces the bias gradient (``csvit_col_reduce``).
* ``linear`` / ``batchnorm`` / ``attention`` / ``gelu`` - op-level Functions for the small fp32 (TF32) head.

Backward GEMMs (``csvit_gemm_ex``): dgrad ``dX = dY W`` reads W as an MN-major operand, wgrad ``dW = dY^T X`` reads both
operands MN-major with split-K over the tokens - no transposed copies in the 16-bit path.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import ops


def _c(g: torch.Tensor) -> torch.Tensor:
    return g if g.is_contiguous() else g.contiguous()


# =============================================================================================== backbone
class SwinBlockFn(Function):
    """One SwinLayer (HF:swin/modeling_swin.py:591-653) on the fp32 residual stream ``x [B*H*W, C]``.

    forward(x, ln1w, ln1b, wq, bq, wk, bk, wv, bv, table, wo, bo, ln2w, ln2b, w1, b1, w2, b2, pk, meta)
      ``pk``: packed operands {wqkv, bqkv, wo, w1, w2 (act dtype), bias (plain [h,L,L]), bias_log2 or None}
      ``meta``: (B, H, W, heads, ws, shift, eps, act dtype, impl)
    """

    @staticmethod
    def forward(ctx, x, ln1w, ln1b, wq, bq, wk, bk, wv, bv, table, wo, bo, ln2w, ln2b, w1, b1, w2, b2, pk, meta):
        B, H, W, heads, ws, shift, eps, act, impl = meta
        keep_scale = pk.get("keep_scale")      # [B] fp32 stochastic-depth scale of this block's attention branch, or None
        xn1 = ops.layernorm(x, ln1w, ln1b, eps, out_dtype=act, mode=ops.LN_WINDOW, grid=(H, W), ws=ws, shift=shift)
        qkv = ops.linear(xn1, pk["wqkv"], pk["bqkv"], out_dtype=act, impl=impl)
        att = ops.window_attention(qkv, pk["bias"], B, H, W, heads, ws, shift, bias_log2=pk["bias_log2"])
        if keep_scale is None:
            x1 = ops.linear(att, pk["wo"], bo, resid=x, out_dtype=torch.float32, scatter=(H, W, ws, shift), impl=impl)
        else:   # hidden = shortcut + drop_path(attention_output): whole samples dropped, the kept ones scaled by 1 / keep (HF:646)
            y = ops.linear(att, pk["wo"], bo, out_dtype=torch.float32, scatter=(H, W, ws, shift), impl=impl)
            x1 = ops.row_scale_add(x, y, keep_scale, H * W)
            del y
        ctx.keep_scale = keep_scale
        xn2 = ops.layernorm(x1, ln2w, ln2b, eps, out_dtype=act)
        h = ops.linear(xn2, pk["w1"], b1, out_dtype=act, impl=impl)
        a = ops.eltwise(ops.EW_GELU_FWD, h)
        x2 = ops.linear(a, pk["w2"], b2, resid=x1, out_dtype=torch.float32, impl=impl)
        ctx.save_for_backward(x, xn1, qkv, att, x1, xn2, h, a, ln1w, ln2w)
        ctx.pk, ctx.meta = pk, meta
        return x2

    @staticmethod
    @once_differentiable
    def backward(ctx, g2):
        x, xn1, qkv, att, x1, xn2, h, a, ln1w, ln2w = ctx.saved_tensors
        pk = ctx.pk
        B, H, W, heads, ws, shift, eps, act, impl = ctx.meta
        C = x.shape[1]
        f32 = torch.float32
        g2 = _c(g2)
        L = ws * ws
        nW = (H // ws) * (W // ws)
        # every small fp32 accumulator of this block (bias / LayerNorm / bias-table gradients) is a slice of ONE zero-filled
        # workspace: one fill kernel instead of twelve
        sizes = [C, 4 * C, C, C, C, 3 * C, C, C, heads * L * L, pk["table_rows"] * heads]
        wsp = torch.zeros(sum(sizes), dtype=f32, device=x.device)
        zb2, zb1, zl2w, zl2b, zbo, zbqkv, zl1w, zl1b, zdbias, zdtable = torch.split(wsp, sizes)
        # MLP half:  x2 = x1 + fc2(gelu(fc1(LN2(x1))))
        db2, _, g2c = ops.col_reduce(g2, copy_dtype=act, s1=zb2)
        dw2 = ops.gemm_ex(g2c, True, a, True, out_dtype=f32, impl=impl)
        da = ops.gemm_ex(g2c, False, pk["w2"], True, out_dtype=act, impl=impl)
        dh = ops.eltwise(ops.EW_GELU_BWD, da, h)
        del da
        db1, _, _ = ops.col_reduce(dh, s1=zb1)
        dw1 = ops.gemm_ex(dh, True, xn2, True, out_dtype=f32, impl=impl)
        dxn2 = ops.gemm_ex(dh, False, pk["w1"], True, out_dtype=act, impl=impl)
        del dh
        g1, dln2w, dln2b = ops.layernorm_bwd(x1, dxn2, ln2w, eps, dres=g2, dgamma=zl2w, dbeta=zl2b)
        # attention half:  x1[token(r)] = x[token(r)] + proj(attn(qkv(LN1(x)[token(r)])))   (r = window-ordered row)
        g1b = g1 if ctx.keep_scale is None else ops.row_scale_add(None, g1, ctx.keep_scale, H * W)      # the branch's share of dL/dx1
        dbo, _, g1w = ops.col_reduce(g1b, window=(H, W, ws, shift), copy_dtype=act, s1=zbo)
        del g1b
        dwo = ops.gemm_ex(g1w, True, att, True, out_dtype=f32, impl=impl)
        datt = ops.gemm_ex(g1w, False, pk["wo"], True, out_dtype=act, impl=impl)
        dqkv = torch.empty_like(qkv)
        _, _, _, dbias = ops.attention_bwd(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], datt, B * nW, L, L, heads, 1.0 / math.sqrt(32.0),
                                           bias=pk["bias"], mask=(H, W, ws, shift), dq=dqkv[:, :C], dk=dqkv[:, C:2 * C],
                                           dv=dqkv[:, 2 * C:], dbias=zdbias.view(heads, L, L))
        # bias[h,i,j] = table[index[i,j], h]  (HF:428-434): scatter-add of a [h,49,49] tensor into [169,h]
        dtable = zdtable.view(pk["table_rows"], heads)
        dtable.index_add_(0, pk["rel_index"], dbias.reshape(heads, L * L).t())
        dbqkv, _, _ = ops.col_reduce(dqkv, s1=zbqkv)
        dwqkv = ops.gemm_ex(dqkv, True, xn1, True, out_dtype=f32, impl=impl)
        dxn1 = ops.gemm_ex(dqkv, False, pk["wqkv"], True, out_dtype=act, impl=impl)
        g0, dln1w, dln1b = ops.layernorm_bwd(x, dxn1, ln1w, eps, mode=ops.LN_WINDOW, grid=(H, W), ws=ws, shift=shift, dres=g1,
                                               dgamma=zl1w, dbeta=zl1b)
        return (g0, dln1w, dln1b, dwqkv[:C], dbqkv[:C], dwqkv[C:2 * C], dbqkv[C:2 * C], dwqkv[2 * C:], dbqkv[2 * C:], dtable,
                dwo, dbo, dln2w, dln2b, dw1, db1, dw2, db2, None, None)


class PatchMergeFn(Function):
    """SwinPatchMerging (HF:326-349): 2x2 concat -> LayerNorm(4C) -> Linear(4C, 2C, bias=False)."""

    @staticmethod
    def forward(ctx, x, nw, nb, rw, rw_packed, meta):
        H, W, eps, act, impl = meta
        xm = ops.layernorm(x, nw, nb, eps, out_dtype=act, mode=ops.LN_MERGE2X2, grid=(H, W))
        y = ops.linear(xm, rw_packed, None, out_dtype=torch.float32, impl=impl)
        ctx.save_for_backward(x, xm, nw, rw_packed)
        ctx.meta = meta
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, xm, nw, rwp = ctx.saved_tensors
        H, W, eps, act, impl = ctx.meta
        _, _, gyc = ops.col_reduce(_c(gy), copy_dtype=act, sums=False)
        drw = ops.gemm_ex(gyc, True, xm, True, out_dtype=torch.float32, impl=impl)
        dxm = ops.gemm_ex(gyc, False, rwp, True, out_dtype=act, impl=impl)
        dx, dnw, dnb = ops.layernorm_bwd(x, dxm, nw, eps, mode=ops.LN_MERGE2X2, grid=(H, W))
        return dx, dnw, dnb, drw, None, None


class PatchEmbedFn(Function):
    """Normalize + Conv2d(3, C0, 4, stride 4) as im2col GEMM + LayerNorm (HF:227-252, 286-295; ref:ti_poser.py:239-243,425)."""

    @staticmethod
    def forward(ctx, images, pw, pb, lnw, lnb, pw_packed, meta):
        normalize, eps, act, impl = meta
        cols = ops.patch_im2col(images, out_dtype=act, normalize=normalize)
        y = ops.linear(cols, pw_packed, pb, out_dtype=torch.float32, impl=impl)
        x = ops.layernorm(y, lnw, lnb, eps)
        ctx.save_for_backward(cols, y, lnw)
        ctx.meta, ctx.wshape = meta, pw.shape
        return x

    @staticmethod
    @once_differentiable
    def backward(ctx, gx):
        cols, y, lnw = ctx.saved_tensors
        _, eps, act, impl = ctx.meta
        dy, dlnw, dlnb = ops.layernorm_bwd(y, _c(gx), lnw, eps)
        dpb, _, dyc = ops.col_reduce(dy, copy_dtype=act)
        dpw = ops.gemm_ex(dyc, True, cols, True, out_dtype=torch.float32, impl=impl)
        return None, dpw.view(ctx.wshape), dpb, dlnw, dlnb, None, None


class LayerNormFn(Function):
    """Plain fp32 LayerNorm over rows (the backbone's final norm, HF:882)."""

    @staticmethod
    def forward(ctx, x, w, b, eps):
        ctx.save_for_backward(x, w)
        ctx.eps = eps
        return ops.layernorm(x, w, b, eps)

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        dx, dw, db = ops.layernorm_bwd(x, _c(gy), w, ctx.eps)
        return dx, dw, db, None


# =============================================================================================== head (fp32 / TF32)
class _LinearFn(Function):
    @staticmethod
    def forward(ctx, a, w, b, resid, act, impl):
        y = ops.linear(a, w, b, act=act, resid=resid, impl=impl)
        ctx.save_for_backward(a, w, y if act == ops.ACT_RELU else None)
        ctx.act, ctx.impl, ctx.has_b, ctx.has_r = act, impl, b is not None, resid is not None
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        a, w, y = ctx.saved_tensors
        g = _c(g)
        gr = g if ctx.has_r else None
        if ctx.act == ops.ACT_RELU:
            g = ops.eltwise(ops.EW_RELU_BWD, g, y)
        da = ops.gemm_ex(g, False, w, True, impl=ctx.impl) if ctx.needs_input_grad[0] else None
        dw = ops.gemm_ex(g, True, a, True, impl=ctx.impl) if ctx.needs_input_grad[1] else None
        db = ops.col_reduce(g)[0] if ctx.has_b and ctx.needs_input_grad[2] else None
        return da, dw, db, gr, None, None


def linear(a: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], *, act: int = ops.ACT_NONE, resid: Optional[torch.Tensor] = None,
           impl: int = ops.GEMM_TC) -> torch.Tensor:
    """fp32 ``act(a @ w.T + b) + resid`` with a kernel backward (ACT_NONE / ACT_RELU only; GELU goes through ``gelu``)."""
    if act == ops.ACT_GELU:
        raise ValueError("autograd.linear: use linear(...) followed by gelu(...) so the pre-activation is kept")
    return _LinearFn.apply(a, w, b, resid, act, impl)


class _Linear16Fn(Function):
    """``a @ w.T + b`` on 16-bit tensor-core operands with fp32 accumulation, output and gradients (the operand policy of SwinBlockFn for
    code that is not written as one Function per block): the 16-bit copies of the activation and the weight are what is saved, and the
    backward GEMMs read them and the 16-bit copy of the incoming gradient AS STORED (MN-major operands of ``csvit_gemm_ex``) - no fp32
    transposes, twice the MMA rate of the TF32 path that ``linear`` takes on fp32 tensors."""

    @staticmethod
    def forward(ctx, a, w, b, act_dtype, out16):
        a16 = a if a.dtype == act_dtype else a.to(act_dtype)
        w16 = w.detach().to(act_dtype)
        y = ops.linear(a16, w16, b, out_dtype=act_dtype if out16 else torch.float32)
        ctx.save_for_backward(a16, w16)
        ctx.has_b, ctx.act_dtype = b is not None, act_dtype
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        a16, w16 = ctx.saved_tensors
        g = _c(g)
        want_db = ctx.has_b and ctx.needs_input_grad[2]
        db = None
        if g.dtype == torch.float32:      # one pass over the fp32 gradient: its 16-bit operand copy and the bias gradient
            if want_db:
                db, _, g16 = ops.col_reduce(g, copy_dtype=ctx.act_dtype)
            else:
                g16 = g.to(ctx.act_dtype)
        else:
            g16 = g
            if want_db:
                db = ops.col_reduce(g)[0]
        da = ops.gemm_ex(g16, False, w16, True, out_dtype=torch.float32) if ctx.needs_input_grad[0] else None
        dw = ops.gemm_ex(g16, True, a16, True, out_dtype=torch.float32) if ctx.needs_input_grad[1] else None
        return da, dw, db, None, None


def linear16(a: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], act_dtype: torch.dtype, out16: bool = False) -> torch.Tensor:
    """``a @ w.T + b`` computed on ``act_dtype`` (fp16 / bf16) tensor-core operands with a kernel backward on the same operands; fp32 result
    (``out16``: 16-bit, for tensors that only feed another 16-bit operand - the MLP's hidden activations, the attention's values)."""
    return _Linear16Fn.apply(a, w, b, act_dtype, out16)


class _CosNormFn(Function):
    """``x / max(|x|, 1e-12) * scale`` over the last axis of ``x [rows, heads, d]`` (F.normalize and the logit scale of SwinV2's cosine
    attention, V2:450-455; ``scale [heads]`` or None), emitted in ``out_dtype``; contiguous row-major operands (the Linear's own layout).  One hand-written backward instead of autograd's chain
    through norm / clamp / div / mul:  dx = (g' - x_hat (x_hat . g')) / |x|  with  g' = g * scale,  dscale = sum(g * x_hat)."""

    @staticmethod
    def forward(ctx, x, scale, out_dtype):
        nrm = torch.linalg.vector_norm(x, dim=-1, keepdim=True).clamp_min_(1e-12)
        xh = x / nrm
        ctx.save_for_backward(xh, nrm, scale)
        y = xh if scale is None else xh * scale.view(1, -1, 1)
        return y.to(out_dtype)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        xh, nrm, scale = ctx.saved_tensors
        g = g.float().contiguous()
        dscale = None
        if scale is not None:
            if ctx.needs_input_grad[1]:
                dscale = (g * xh).sum(dim=(0, 2)).view_as(scale)
            g = g * scale.view(1, -1, 1)
        dx = (g - xh * (xh * g).sum(dim=-1, keepdim=True)) / nrm
        return dx, dscale, None


def cosnorm(x: torch.Tensor, scale: Optional[torch.Tensor], out_dtype: torch.dtype) -> torch.Tensor:
    return _CosNormFn.apply(x, scale, out_dtype)


class _Swinv2CosineAttnFn(Function):
    """SwinV2 scaled-cosine window attention core for 16 x 16 windows, log2 domain (V2:421-487), on the library's tcgen05 kernels:
    forward ``csvit_swinv2_attn_tc_train`` (window-ordered context + the rows' lse2), backward ``csvit_swinv2_attn_tc_bwd``.
    ``q2 = q_hat * logit_scale * log2 e``, ``k = k_hat`` and ``v`` are 16-bit ``[rows, C]`` in window order; ``bias_log2`` is the fp32
    ``[heads, 31, 48]`` table of :func:`ops.swinv2_bias_log2` (log2 e * 16 sigmoid(cpb)).  The gradients of the logit scale and of the
    CPB-MLP reach their parameters through the differentiable construction of ``q2`` and ``bias_log2``."""

    @staticmethod
    def forward(ctx, q2, k, v, bias_log2, B, H, W, heads, shift, mask_repeat):
        qkv = torch.cat([q2, k, v], dim=1)
        bl2 = bias_log2.detach().contiguous()
        out, lse2 = ops.swinv2_attn_tc_train(qkv, bl2, B, H, W, heads, shift, mask_repeat)
        ctx.save_for_backward(qkv, out, lse2, bl2)
        ctx.geom = (B, H, W, heads, shift, mask_repeat)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        qkv, out, lse2, bl2 = ctx.saved_tensors
        dq, dk, dv, dbias = ops.swinv2_attn_tc_bwd(qkv, out, lse2, _c(g.to(out.dtype)), bl2, *ctx.geom)
        return dq, dk, dv, dbias, None, None, None, None, None, None


def swinv2_cosine_attention(q2: torch.Tensor, k: torch.Tensor, v: torch.Tensor, bias_log2: torch.Tensor, B: int, H: int, W: int, heads: int,
                            shift: int, mask_repeat: int = 2) -> torch.Tensor:
    """Differentiable SwinV2 cosine-attention core of 16 x 16 windows -> 16-bit window-ordered ``ctx [rows, C]`` (see
    :class:`_Swinv2CosineAttnFn`); gradients ``dq2, dk, dv`` (16 bit) and ``dbias_log2`` (fp32)."""
    return _Swinv2CosineAttnFn.apply(q2, k, v, bias_log2, B, H, W, heads, shift, mask_repeat)


class _PermuteRowsFn(Function):
    """``x[:, idx]`` for a PERMUTATION ``idx`` of the token axis (roll + window_partition, or their inverse): the backward is the gather by the
    inverse permutation, not autograd's scatter-add."""

    @staticmethod
    def forward(ctx, x, idx, inv):
        ctx.save_for_backward(idx, inv)
        return x.index_select(1, idx)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        idx, inv = ctx.saved_tensors
        return g.index_select(1, inv), None, None


def permute_rows(x: torch.Tensor, idx: torch.Tensor, inv: torch.Tensor) -> torch.Tensor:
    return _PermuteRowsFn.apply(x, idx, inv)


class _GeluFn(Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return ops.eltwise(ops.EW_GELU_FWD, x)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return ops.eltwise(ops.EW_GELU_BWD, _c(g), x)


def gelu(x: torch.Tensor) -> torch.Tensor:
    return _GeluFn.apply(x)


class _BatchNormFn(Function):
    """BatchNorm1d over channels of ``x [rows, C]`` (the reference normalises ``[n, C, L]`` over (n, L), ref:transformer_module.py:312).
    ``mean`` / ``rstd`` are the statistics in use: the batch's in train mode, the running ones in eval mode."""

    @staticmethod
    def forward(ctx, x, w, b, mean, rstd, batch_stats):
        scale = (w * rstd).contiguous()
        shift = (b - mean * scale).contiguous()
        ctx.save_for_backward(x, mean, rstd, scale)
        ctx.batch_stats = batch_stats
        return ops.affine_rows(x, scale, shift)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, mean, rstd, scale = ctx.saved_tensors
        g = _c(g)
        rows = x.shape[0]
        sdy, sdyx, _ = ops.col_reduce(g, ops.CR_DOT, b=x)
        dgamma = rstd * (sdyx - mean * sdy)          # sum dy * xhat
        if ctx.batch_stats:
            m2 = dgamma / rows
            bx = (-scale * m2 * rstd).contiguous()
            c0 = (-scale * sdy / rows - bx * mean).contiguous()
        else:
            bx = torch.zeros_like(scale)
            c0 = bx
        dx = ops.affine2_rows(g, x, scale, bx, c0)
        return dx, dgamma, sdy, None, None, None


def batchnorm(x: torch.Tensor, bn: torch.nn.BatchNorm1d) -> torch.Tensor:
    """Train mode: batch statistics (biased variance for the normalisation, unbiased for the running update, momentum as in
    ``nn.BatchNorm1d``).  Eval mode: running statistics.  Either way one affine kernel, differentiable."""
    rows, C = x.shape
    if bn.training:
        with torch.no_grad():
            s1, _, _ = ops.col_reduce(x)
            mean = (s1 / rows).contiguous()
            _, d2, _ = ops.col_reduce(x, ops.CR_CENTERED, center=mean)
            var = d2 / rows
            rstd = torch.rsqrt(var + bn.eps)
            if bn.track_running_stats and bn.running_mean is not None:
                mom = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked.item() + 1)
                bn.running_mean.mul_(1 - mom).add_(mean, alpha=mom)
                bn.running_var.mul_(1 - mom).add_(d2 / max(rows - 1, 1), alpha=mom)
                bn.num_batches_tracked.add_(1)
        return _BatchNormFn.apply(x, bn.weight, bn.bias, mean, rstd, True)
    mean = bn.running_mean.detach().float()
    rstd = torch.rsqrt(bn.running_var.detach().float() + bn.eps)
    return _BatchNormFn.apply(x, bn.weight, bn.bias, mean, rstd, False)


class _CrossAttentionFn(Function):
    """Dense MHA core, queries ``q [n*L, D]`` against the packed ``kv [n*S, 2D]`` (K | V column blocks)."""

    @staticmethod
    def forward(ctx, q, kv, D, n, L, S, heads, scale):
        out = ops.attention(q, kv[:, :D], kv[:, D:], n, L, S, heads, scale)
        ctx.save_for_backward(q, kv)
        ctx.cfg = (D, n, L, S, heads, scale)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        q, kv = ctx.saved_tensors
        D, n, L, S, heads, scale = ctx.cfg
        dq, dkv = torch.empty_like(q), torch.empty_like(kv)
        ops.attention_bwd(q, kv[:, :D], kv[:, D:], _c(g), n, L, S, heads, scale, dq=dq, dk=dkv[:, :D], dv=dkv[:, D:])
        return dq, dkv, None, None, None, None, None, None


def attention_packed(qkv: torch.Tensor, D: int, n: int, L: int, heads: int, scale: float) -> torch.Tensor:
    """Self-attention on the packed ``[n*L, 3D]`` projection (Q | K | V column blocks)."""
    return _SelfAttentionFn.apply(qkv, D, n, L, heads, scale)


def attention_cross(q: torch.Tensor, kv: torch.Tensor, D: int, n: int, L: int, S: int, heads: int, scale: float) -> torch.Tensor:
    return _CrossAttentionFn.apply(q, kv, D, n, L, S, heads, scale)


class _SelfAttentionFn(Function):
    @staticmethod
    def forward(ctx, qkv, D, n, L, heads, scale):
        out = ops.attention(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], n, L, L, heads, scale)
        ctx.save_for_backward(qkv)
        ctx.cfg = (D, n, L, heads, scale)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (qkv,) = ctx.saved_tensors
        D, n, L, heads, scale = ctx.cfg
        dqkv = torch.empty_like(qkv)
        ops.attention_bwd(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], _c(g), n, L, L, heads, scale,
                          dq=dqkv[:, :D], dk=dqkv[:, D:2 * D], dv=dqkv[:, 2 * D:])
        return dqkv, None, None, None, None, None
