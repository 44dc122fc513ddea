"""Swin-v1 backbone on the sm_100a kernels - replaces ``transformers.AutoModel.from_pretrained(dir)``.

The reference delegates its backbone to HuggingFace (ref:cs_vit/net/ti_poser.py:246) and consumes exactly
``.config.hidden_size``, ``.config.num_heads``, ``.parameters()``, ``.train()/.eval()`` and
``__call__(pixel_values).last_hidden_state`` (ref:cs_vit/net/ti_poser.py:247-253, 426).  This module offers that
seam with the same parameter names and shapes as ``SwinModel`` (HF:swin/modeling_swin.py), so HF checkpoints
and the reference's ``ckpt["merged"]`` (keys ``backbone.*``) load unchanged, but the forward never touches
ATen math: per block it issues

    LN+shift+partition gather -> QKV GEMM -> window attention -> out-proj GEMM with un-shift scatter + residual
    LN -> fc1 GEMM with GELU epilogue -> fc2 GEMM with residual epilogue

on ``libcsvit_sm100.so``.  The residual stream, LayerNorm statistics, softmax and GELU stay fp32.  ``precision``
picks the tensor-core operand format: ``"bf16"`` (8-bit mantissa) or ``"fp16"`` (11-bit mantissa, identical MMA
rate; features land ~8x closer to the fp32 reference, which the sharp-softmax head needs, DESIGN.md "Numerics"),
or ``"fp32"`` = exact fp32 FMA everywhere (validation mode for the 1e-4 bar).
"""
from __future__ import annotations

import json
import os
from types import SimpleNamespace
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from .. import ops
from ._pack import PackCache


PRECISIONS = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}


class SwinConfigLite(SimpleNamespace):
    """The subset of ``SwinConfig`` the hot path reads (HF:swin/configuration_swin.py)."""

    @classmethod
    def from_dict(cls, d: Dict) -> "SwinConfigLite":
        model_type = d.get("model_type", "swin")
        if model_type != "swin":
            raise NotImplementedError(
                f"backbone model_type '{model_type}' is not built: only Swin v1 (window 7) has sm_100a kernels "
                f"(SwinV2 is the next row of SURVEY.md §8f); there is no fallback path")
        embed_dim = d.get("embed_dim", 96)
        depths = list(d.get("depths", [2, 2, 6, 2]))
        cfg = cls(
            model_type=model_type,
            image_size=d.get("image_size", 224),
            patch_size=d.get("patch_size", 4),
            num_channels=d.get("num_channels", 3),
            embed_dim=embed_dim,
            depths=depths,
            num_heads=list(d.get("num_heads", [3, 6, 12, 24])),
            window_size=d.get("window_size", 7),
            mlp_ratio=d.get("mlp_ratio", 4.0),
            qkv_bias=d.get("qkv_bias", True),
            layer_norm_eps=d.get("layer_norm_eps", 1e-5),
            use_absolute_embeddings=d.get("use_absolute_embeddings", False),
            hidden_act=d.get("hidden_act", "gelu"),
            drop_path_rate=d.get("drop_path_rate", 0.1),
            hidden_size=int(embed_dim * 2 ** (len(depths) - 1)),
        )
        if cfg.patch_size != 4 or cfg.num_channels != 3 or cfg.mlp_ratio != 4.0 or not cfg.qkv_bias:
            raise NotImplementedError("only patch 4 / RGB / mlp_ratio 4 / qkv_bias Swin configurations are built")
        if cfg.use_absolute_embeddings or cfg.hidden_act != "gelu":
            raise NotImplementedError("absolute position embeddings / non-GELU activations are not built")
        if any(cfg.embed_dim * 2 ** s != 32 * h for s, h in enumerate(cfg.num_heads)):
            raise NotImplementedError("the attention kernels require head_dim == 32 at every stage")
        return cfg


def _holder(**children) -> nn.Module:
    m = nn.Module()
    for k, v in children.items():
        setattr(m, k, v)
    return m


class _SelfAttnParams(nn.Module):
    def __init__(self, dim: int, heads: int, ws: int):
        super().__init__()
        self.query = nn.Linear(dim, dim)
        self.key = nn.Linear(dim, dim)
        self.value = nn.Linear(dim, dim)
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * ws - 1) ** 2, heads))
        ys, xs = torch.meshgrid(torch.arange(ws), torch.arange(ws), indexing="ij")
        dy = ys.reshape(-1, 1) - ys.reshape(1, -1) + ws - 1
        dx = xs.reshape(-1, 1) - xs.reshape(1, -1) + ws - 1
        self.register_buffer("relative_position_index", (dy * (2 * ws - 1) + dx).to(torch.int64))


class _BlockParams(nn.Module):
    """Parameter holder with ``SwinLayer``'s names (HF:swin/modeling_swin.py:534-546)."""

    def __init__(self, dim: int, heads: int, ws: int, eps: float):
        super().__init__()
        self.layernorm_before = nn.LayerNorm(dim, eps=eps)
        self.attention = _holder(self=_SelfAttnParams(dim, heads, ws), output=_holder(dense=nn.Linear(dim, dim)))
        self.layernorm_after = nn.LayerNorm(dim, eps=eps)
        self.intermediate = _holder(dense=nn.Linear(dim, 4 * dim))
        self.output = _holder(dense=nn.Linear(4 * dim, dim))


class SwinBackboneB200(nn.Module):
    def __init__(self, config: SwinConfigLite, precision: str = "bf16"):
        super().__init__()
        self.config = config
        self.precision = precision
        self.fuse_attn = True  # csvit_swin_attn_fused for C in {128, 256}: LN + QKV + window attention in one tcgen05 kernel
        self.fuse_attn_widths = ops.ATTN_FUSED_WIDTHS   # (ablation: restrict the fused kernel to a subset of its widths)
        self._drop_path_rand: List[torch.Tensor] = []   # test hook: the [B] uniform draws of the next stochastic-depth calls, in call order
        self.fuse_mlp = True   # csvit_mlp_fused for C in {128, 256}: hidden activations never leave the SM
        # Inference runs the batch through the whole backbone in chunks of this many images (0 = all at once).  Images are
        # independent, so the result is bit-identical; what changes is locality: a chunk's inter-kernel tensors (tens of MB)
        # stay resident in the 126 MB L2 between the kernel that writes them and the one that reads them, instead of making
        # a round trip through HBM as the 100-800 MB tensors of a 256-image batch do (profiles/r1_micro_batch_sweep.txt).
        self.micro_batch = 0
        c0, eps, ws = config.embed_dim, config.layer_norm_eps, config.window_size
        self.embeddings = _holder(
            patch_embeddings=_holder(projection=nn.Conv2d(3, c0, kernel_size=4, stride=4)),
            norm=nn.LayerNorm(c0, eps=eps))
        stages: List[nn.Module] = []
        for s, (depth, heads) in enumerate(zip(config.depths, config.num_heads)):
            dim = c0 * 2 ** s
            stage = nn.Module()
            stage.blocks = nn.ModuleList([_BlockParams(dim, heads, ws, eps) for _ in range(depth)])
            if s < len(config.depths) - 1:
                stage.downsample = _holder(reduction=nn.Linear(4 * dim, 2 * dim, bias=False), norm=nn.LayerNorm(4 * dim, eps=eps))
            stages.append(stage)
        self.encoder = _holder(layers=nn.ModuleList(stages))
        self.layernorm = nn.LayerNorm(config.hidden_size, eps=eps)
        self._pack = PackCache()

    # ------------------------------------------------------------------------------------------ construction
    @classmethod
    def from_pretrained(cls, path: str, precision: str = "bf16") -> "SwinBackboneB200":
        """Load an HF-format directory (``config.json`` + ``model.safetensors`` / ``pytorch_model.bin``)."""
        with open(os.path.join(path, "config.json")) as f:
            cfg = SwinConfigLite.from_dict(json.load(f))
        model = cls(cfg, precision)
        st = os.path.join(path, "model.safetensors")
        if os.path.exists(st):
            from safetensors.torch import load_file
            sd = load_file(st)
        else:
            sd = torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu")
        sd = {(k[len("swin."):] if k.startswith("swin.") else k): v for k, v in sd.items()}
        missing, unexpected = model.load_state_dict(sd, strict=False)
        missing = [k for k in missing if not k.endswith("relative_position_index")]
        unexpected = [k for k in unexpected if not k.startswith("pooler")]
        if missing or unexpected:
            raise RuntimeError(f"backbone checkpoint mismatch: missing {missing[:5]} unexpected {unexpected[:5]}")
        model.eval()
        return model

    # ------------------------------------------------------------------------------------------ packing
    @property
    def _fp32(self) -> bool:
        if self.precision == "fp8":
            raise ValueError("precision='fp8' is built for the swinv2 backbone only: the Swin v1 stage 0-1 fused kernels have no fp8 form")
        if self.precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(PRECISIONS)}, got {self.precision!r}")
        return self.precision == "fp32"

    @property
    def _act_dtype(self) -> torch.dtype:
        _ = self._fp32
        return PRECISIONS[self.precision]

    def _w(self, key: str, tensors, build):
        return self._pack.get(f"{self.precision}/{key}", tensors, build)

    def _weight(self, key: str, lin_weight: torch.Tensor) -> torch.Tensor:
        dt = self._act_dtype
        return self._w(key, [lin_weight], lambda: lin_weight.detach().reshape(lin_weight.shape[0], -1).to(dt).contiguous())

    def _f32(self, key: str, t: torch.Tensor) -> torch.Tensor:
        return self._w(key, [t], lambda: t.detach().float().contiguous())

    # ------------------------------------------------------------------------------------------ forward
    def _block(self, x: torch.Tensor, blk: _BlockParams, key: str, B: int, H: int, W: int, heads: int, shift: int) -> None:
        """One SwinLayer, in place on the fp32 residual stream x [B*H*W, C]   (HF:swin/modeling_swin.py:591-653)."""
        cfg = self.config
        ws = cfg.window_size
        if min(H, W) <= ws:  # HF:548-554
            ws, shift = min(H, W), 0
        C = x.shape[1]
        act = self._act_dtype
        impl = ops.GEMM_SIMT if self._fp32 else ops.GEMM_TC
        sa = blk.attention.self
        qkv_src = [sa.query.weight, sa.key.weight, sa.value.weight]
        bqkv_src = [sa.query.bias, sa.key.bias, sa.value.bias]
        eps = cfg.layer_norm_eps
        ln1 = blk.layernorm_before
        proj = blk.attention.output.dense
        wproj, bproj = self._weight(key + "wproj", proj.weight), self._f32(key + "bproj", proj.bias)
        if self._fp32:
            # validation mode: exact fp32 kernels (SIMT GEMMs, fp32 attention), window-ordered context scattered by the out-proj
            wqkv = self._w(key + "wqkv", qkv_src, lambda: torch.cat([w.detach() for w in qkv_src], 0).to(act).contiguous())
            bqkv = self._w(key + "bqkv", bqkv_src, lambda: torch.cat([b.detach() for b in bqkv_src], 0).float().contiguous())
            bias = self._w(key + "relbias", [sa.relative_position_bias_table],
                           lambda: ops.expand_rel_bias(sa.relative_position_bias_table.detach(), ws))
            xn = ops.layernorm(x, self._f32(key + "ln1w", ln1.weight), self._f32(key + "ln1b", ln1.bias), eps, out_dtype=act,
                               mode=ops.LN_WINDOW, grid=(H, W), ws=ws, shift=shift)
            qkv = ops.linear(xn, wqkv, bqkv, out_dtype=act, impl=impl)
            ctx = ops.window_attention(qkv, bias, B, H, W, heads, ws, shift)
            ops.linear(ctx, wproj, bproj, resid=x, out=x, scatter=(H, W, ws, shift), impl=impl)
        else:
            if ws != 7 or C != 32 * heads:
                raise NotImplementedError(f"the tcgen05 window-attention kernels are built for 7x7 windows and head_dim 32 "
                                          f"(got window {ws}, C={C}, heads={heads}); use precision='fp32'")
            if self.fuse_attn and C in self.fuse_attn_widths:
                # narrow stages: layernorm_before + shift/partition + Q/K/V + window attention + reverse/un-shift in ONE tcgen05
                # kernel (csrc/attn_fused.cu); xn, qkv, logits and probabilities stay on the SM.  Out-proj on plain rows.
                src = qkv_src + bqkv_src + [sa.relative_position_bias_table, ln1.weight, ln1.bias]
                wqkv_h, bqkv_h, bias_op = self._w(key + "attn_fused", src, lambda: ops.pack_attn_fused(
                    sa.query.weight, sa.key.weight, sa.value.weight, sa.query.bias, sa.key.bias, sa.value.bias,
                    sa.relative_position_bias_table, sa.relative_position_index, act, ln1.weight, ln1.bias))
                ctx = ops.swin_attn_fused(x, eps, wqkv_h, bqkv_h, bias_op, B, H, W, heads, ws, shift)
                ops.linear(ctx, wproj, bproj, resid=x, out=x, impl=impl)
            else:
                # LayerNorm (window-ordered 16-bit rows) -> Q/K/V GEMM (log2(e)/sqrt(32) folded into the q rows) -> tcgen05 attention
                # core on TMA-loaded operand tiles (csrc/attn_core.cu), token-ordered context -> out-proj on plain rows with the
                # TMA residual epilogue (narrow rows: the scatter epilogue of the out-proj is faster than its TMA form)
                wqs, bqs = self._w(key + "wqkv_qs", qkv_src + bqkv_src, lambda: ops.pack_qkv_prescaled(
                    sa.query.weight, sa.key.weight, sa.value.weight, sa.query.bias, sa.key.bias, sa.value.bias, act))
                bias_l2 = self._w(key + "relbias_l2", [sa.relative_position_bias_table],
                                  lambda: ops.pack_rel_bias_log2(sa.relative_position_bias_table, sa.relative_position_index))
                xn = ops.layernorm(x, self._f32(key + "ln1w", ln1.weight), self._f32(key + "ln1b", ln1.bias), eps, out_dtype=act,
                                   mode=ops.LN_WINDOW, grid=(H, W), ws=ws, shift=shift)
                qkv = ops.linear(xn, wqs, bqs, out_dtype=act, impl=impl)
                tok = C >= 256
                ctx = ops.swin_attn_core(qkv, bias_l2, B, H, W, heads, ws, shift, token_order=tok, q_prescaled=True)
                ops.linear(ctx, wproj, bproj, resid=x, out=x, impl=impl, **({} if tok else {"scatter": (H, W, ws, shift)}))
        # layernorm_after + intermediate (GELU) + output + residual   (HF:510-531, 648-650)
        ln2 = blk.layernorm_after
        fc1, fc2 = blk.intermediate.dense, blk.output.dense
        xn = ops.layernorm(x, self._f32(key + "ln2w", ln2.weight), self._f32(key + "ln2b", ln2.bias), eps, out_dtype=act)
        if self.fuse_mlp and not self._fp32 and C in ops.MLP_FUSED_WIDTHS:
            # narrow stages: fc1 + GELU + fc2 + residual in one kernel, the [M, 4C] hidden tensor stays on chip
            ops.mlp_fused(xn, self._weight(key + "w1", fc1.weight), self._f32(key + "b1", fc1.bias),
                          self._weight(key + "w2", fc2.weight), self._f32(key + "b2", fc2.bias), x)
            return
        hid = ops.linear(xn, self._weight(key + "w1", fc1.weight), self._f32(key + "b1", fc1.bias), act=ops.ACT_GELU,
                         out_dtype=act, impl=impl)
        ops.linear(hid, self._weight(key + "w2", fc2.weight), self._f32(key + "b2", fc2.bias), resid=x, out=x, impl=impl)

    def forward_features(self, images: torch.Tensor, normalize: bool, return_stages: bool = False):
        """images fp32 ``[n,3,S,S]``; ``normalize`` folds the ImageNet mean/std of
        ref:cs_vit/net/ti_poser.py:239-243 into the patch unfold.  Returns fp32 ``[n, (S/32)^2, hidden]``.

        With autograd enabled and trainable parameters the differentiable path runs (one ``autograd.Function`` per block,
        activations kept for the backward kernels); otherwise the in-place inference path."""
        cfg = self.config
        if not images.is_cuda:
            raise RuntimeError("SwinBackboneB200 runs on CUDA tensors only (there is no CPU fallback)")
        n, _, S, S2 = images.shape
        if S != S2 or S % (32 * cfg.window_size) != 0:
            raise ValueError(f"image side {S} must be a multiple of {32 * cfg.window_size} (no padding path, SURVEY.md §8b)")
        wants_grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if not return_stages and (wants_grad or (self.training and cfg.drop_path_rate > 0)):
            # (return_stages is a diagnostic of the inference path; a train-mode forward with stochastic depth takes this path
            # under no_grad too - HF drops paths whenever module.training is set)
            return self._forward_train(images, normalize)
        with torch.no_grad():
            return self._forward_infer(images, normalize, return_stages)

    # ------------------------------------------------------------------------------------------ training path
    def _block_pack(self, blk: _BlockParams, key: str, ws: int) -> Dict:
        act = self._act_dtype
        sa = blk.attention.self
        qkv_src = [sa.query.weight, sa.key.weight, sa.value.weight]
        bqkv_src = [sa.query.bias, sa.key.bias, sa.value.bias]
        tab = sa.relative_position_bias_table
        return {
            "wqkv": self._w(key + "wqkv", qkv_src, lambda: torch.cat([w.detach() for w in qkv_src], 0).to(act).contiguous()),
            "bqkv": self._w(key + "bqkv", bqkv_src, lambda: torch.cat([b.detach() for b in bqkv_src], 0).float().contiguous()),
            "bias": self._w(key + "relbias", [tab], lambda: ops.expand_rel_bias(tab.detach(), ws)),
            "bias_log2": None if self._fp32 else self._w(key + "relbias_l2", [tab], lambda: ops.pack_rel_bias_log2(tab, sa.relative_position_index)),
            "wo": self._weight(key + "wproj", blk.attention.output.dense.weight),
            "w1": self._weight(key + "w1", blk.intermediate.dense.weight),
            "w2": self._weight(key + "w2", blk.output.dense.weight),
            "rel_index": self._w(key + "relidx", [sa.relative_position_index], lambda: sa.relative_position_index.reshape(-1).long()),
            "table_rows": tab.shape[0],
        }

    def _forward_train(self, images: torch.Tensor, normalize: bool) -> torch.Tensor:
        """Differentiable forward: same kernels, out-of-place residual stream, activations saved per block
        (cs_vit/autograd.py holds the backward of every stage)."""
        from .. import autograd as ag
        cfg = self.config
        n, _, S, _ = images.shape
        act = self._act_dtype
        impl = ops.GEMM_SIMT if self._fp32 else ops.GEMM_TC
        eps = cfg.layer_norm_eps
        H = W = S // 4
        pe = self.embeddings.patch_embeddings.projection
        x = ag.PatchEmbedFn.apply(images.float().contiguous(), pe.weight, pe.bias, self.embeddings.norm.weight, self.embeddings.norm.bias,
                                  self._weight("pe_w", pe.weight), (normalize, eps, act, impl))
        # stochastic depth (HF:353-377, 543, 646, 716): block k of the whole encoder drops its attention branch per sample with
        # probability linspace(0, drop_path_rate, sum(depths))[k] in train mode
        total_blocks = sum(cfg.depths)
        rates = torch.linspace(0, cfg.drop_path_rate, total_blocks).tolist() if self.training and cfg.drop_path_rate > 0 else [0.0] * total_blocks
        k = -1
        for s, stage in enumerate(self.encoder.layers):
            heads = cfg.num_heads[s]
            for i, blk in enumerate(stage.blocks):
                k += 1
                ws, shift = cfg.window_size, (0 if i % 2 == 0 else cfg.window_size // 2)
                if min(H, W) <= ws:  # HF:548-554
                    ws, shift = min(H, W), 0
                sa = blk.attention.self
                pk = dict(self._block_pack(blk, f"s{s}b{i}/", ws))
                if rates[k] > 0.0:
                    keep = 1.0 - rates[k]
                    # the uniform draw HF makes per call (torch.rand((B,1,1))); tests pin it to the reference's draws
                    u = self._drop_path_rand.pop(0).to(x.device, torch.float32) if self._drop_path_rand else torch.rand(n, device=x.device)
                    pk["keep_scale"] = (torch.floor(keep + u) / keep).contiguous()
                x = ag.SwinBlockFn.apply(
                    x, blk.layernorm_before.weight, blk.layernorm_before.bias, sa.query.weight, sa.query.bias, sa.key.weight,
                    sa.key.bias, sa.value.weight, sa.value.bias, sa.relative_position_bias_table, blk.attention.output.dense.weight,
                    blk.attention.output.dense.bias, blk.layernorm_after.weight, blk.layernorm_after.bias, blk.intermediate.dense.weight,
                    blk.intermediate.dense.bias, blk.output.dense.weight, blk.output.dense.bias, pk,
                    (n, H, W, heads, ws, shift, eps, act, impl))
            if hasattr(stage, "downsample"):
                ds = stage.downsample
                x = ag.PatchMergeFn.apply(x, ds.norm.weight, ds.norm.bias, ds.reduction.weight,
                                          self._weight(f"s{s}/dsr", ds.reduction.weight), (H, W, eps, act, impl))
                H, W = H // 2, W // 2
        out = ag.LayerNormFn.apply(x, self.layernorm.weight, self.layernorm.bias, eps)
        return out.view(n, H * W, cfg.hidden_size)

    def _forward_infer(self, images: torch.Tensor, normalize: bool, return_stages: bool = False, out: Optional[torch.Tensor] = None):
        cfg = self.config
        n, _, S, _ = images.shape
        mb = self.micro_batch
        if mb and n > mb and not return_stages:
            images = images.float().contiguous()
            full = torch.empty(n, (S // 32) ** 2, cfg.hidden_size, dtype=torch.float32, device=images.device)
            for lo in range(0, n, mb):
                self._forward_infer(images[lo:lo + mb], normalize, out=full[lo:lo + mb])
            return full
        act = self._act_dtype
        impl = ops.GEMM_SIMT if self._fp32 else ops.GEMM_TC
        eps = cfg.layer_norm_eps
        H = W = S // 4
        cols = ops.patch_im2col(images.float().contiguous(), out_dtype=act, normalize=normalize)
        pe = self.embeddings.patch_embeddings.projection
        y = ops.linear(cols, self._weight("pe_w", pe.weight), self._f32("pe_b", pe.bias), out_dtype=torch.float32, impl=impl)
        x = ops.layernorm(y, self._f32("pe_lnw", self.embeddings.norm.weight), self._f32("pe_lnb", self.embeddings.norm.bias), eps)
        stages = []
        for s, stage in enumerate(self.encoder.layers):
            heads = cfg.num_heads[s]
            for i, blk in enumerate(stage.blocks):
                self._block(x, blk, f"s{s}b{i}/", n, H, W, heads, 0 if i % 2 == 0 else cfg.window_size // 2)
            if return_stages:
                stages.append(x.view(n, H * W, -1).clone())
            if hasattr(stage, "downsample"):
                ds = stage.downsample
                xm = ops.layernorm(x, self._f32(f"s{s}/dsw", ds.norm.weight), self._f32(f"s{s}/dsb", ds.norm.bias), eps,
                                   out_dtype=act, mode=ops.LN_MERGE2X2, grid=(H, W))
                x = ops.linear(xm, self._weight(f"s{s}/dsr", ds.reduction.weight), None, out_dtype=torch.float32, impl=impl)
                H, W = H // 2, W // 2
        out = ops.layernorm(x, self._f32("final_w", self.layernorm.weight), self._f32("final_b", self.layernorm.bias), eps,
                            out=None if out is None else out.view(n * H * W, cfg.hidden_size))
        out = out.view(n, H * W, cfg.hidden_size)
        return (out, stages) if return_stages else out

    def forward(self, pixel_values: torch.Tensor, **_unused) -> SimpleNamespace:
        """HF seam: ``pixel_values`` are already normalised   (ref:cs_vit/net/ti_poser.py:425-426)."""
        return SimpleNamespace(last_hidden_state=self.forward_features(pixel_values, normalize=False), pooler_output=None)
