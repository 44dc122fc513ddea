"""SwinV2 backbone on the sm_100a kernels (SURVEY.md §8f row 1).

Every shipped CS-ViT configuration points ``backbone`` at a ``swinv2-*-patch4-window16-256`` HuggingFace directory
(SURVEY.md §0.2); the reference loads it with ``AutoModel.from_pretrained`` (ref:cs_vit/net/ti_poser.py:246) and reads
``last_hidden_state`` (ref:cs_vit/net/ti_poser.py:426).  This module is that seam for ``model_type == "swinv2"``, with
``Swinv2Model``'s parameter names and shapes (V2: = transformers/models/swinv2/modeling_swinv2.py), so HF checkpoints and
the reference's ``ckpt["merged"]`` (keys ``backbone.*``) load unchanged.  The inference path below is the tuned one; the
differentiable path of the finetune step (``_forward_train``) is functional: kernel GEMMs / LayerNorm / GELU with kernel
backwards, the cosine-attention core in torch.

Per block (res-post-norm, V2:662-715) the forward issues, on ``libcsvit_sm100.so``:

    xw (16-bit copy of x in this block's shifted-window order, written by the PREVIOUS LayerNorm kernel)
      -> QKV GEMM (no key bias) -> cosine window attention (csvit_swinv2_window_attention)
      (its store un-partitions / un-shifts: token-ordered context) -> out-proj GEMM, fp32, plain rows (TMA-store epilogue)
      -> csvit_layernorm_post: x += LN(y), and the 16-bit token-order copy of x for fc1
      -> fc1 GEMM + GELU -> fc2 GEMM (fp32)
      -> csvit_layernorm_post: x += LN(z), and the 16-bit copy of x in the NEXT block's window order (or the 2x2-merged
         [N/4, 4C] operand of patch merging)

so roll / window_partition / window_reverse / the merge concat never run as copies, as in the v1 path.
"""
from __future__ import annotations

import json
import math
import os
from types import SimpleNamespace
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from .. import ops
from ._pack import PackCache
from .swin_b200 import PRECISIONS, _holder


_LOG2E = 1.4426950408889634


class Swinv2ConfigLite(SimpleNamespace):
    """The subset of ``Swinv2Config`` the hot path reads (HF:swinv2/configuration_swinv2.py)."""

    @classmethod
    def from_dict(cls, d: Dict) -> "Swinv2ConfigLite":
        if d.get("model_type") != "swinv2":
            raise ValueError(f"not a swinv2 configuration: model_type={d.get('model_type')!r}")
        embed_dim = d.get("embed_dim", 96)
        depths = list(d.get("depths", [2, 2, 6, 2]))
        cfg = cls(
            model_type="swinv2",
            image_size=d.get("image_size", 256),
            patch_size=d.get("patch_size", 4),
            num_channels=d.get("num_channels", 3),
            embed_dim=embed_dim,
            depths=depths,
            num_heads=list(d.get("num_heads", [3, 6, 12, 24])),
            window_size=d.get("window_size", 16),
            pretrained_window_sizes=list(d.get("pretrained_window_sizes") or [0] * len(depths)),
            mlp_ratio=d.get("mlp_ratio", 4.0),
            qkv_bias=d.get("qkv_bias", True),
            layer_norm_eps=d.get("layer_norm_eps", 1e-5),
            use_absolute_embeddings=d.get("use_absolute_embeddings", False),
            hidden_act=d.get("hidden_act", "gelu"),
            drop_path_rate=d.get("drop_path_rate", 0.1),
            hidden_size=int(embed_dim * 2 ** (len(depths) - 1)),
        )
        if cfg.patch_size != 4 or cfg.num_channels != 3 or cfg.mlp_ratio != 4.0 or not cfg.qkv_bias:
            raise NotImplementedError("only patch 4 / RGB / mlp_ratio 4 / qkv_bias SwinV2 configurations are built")
        if cfg.use_absolute_embeddings or cfg.hidden_act != "gelu":
            raise NotImplementedError("absolute position embeddings / non-GELU activations are not built")
        if any(cfg.embed_dim * 2 ** s != 32 * h for s, h in enumerate(cfg.num_heads)):
            raise NotImplementedError("the attention kernels require head_dim == 32 at every stage")
        return cfg

    def stage_geometry(self, s: int) -> Tuple[int, int, int]:
        """(token-grid side, window side, shift of odd blocks) of stage ``s``   (V2:622-625, 735)."""
        res = self.image_size // self.patch_size // 2 ** s
        ws = min(res, self.window_size)
        shift = 0 if res <= ws else self.window_size // 2
        return res, ws, shift


class _SelfAttnParamsV2(nn.Module):
    def __init__(self, dim: int, heads: int):
        super().__init__()
        self.logit_scale = nn.Parameter(torch.log(10 * torch.ones((heads, 1, 1))))
        self.continuous_position_bias_mlp = nn.Sequential(nn.Linear(2, 512, bias=True), nn.ReLU(inplace=True),
                                                          nn.Linear(512, heads, bias=False))
        self.query = nn.Linear(dim, dim)
        self.key = nn.Linear(dim, dim, bias=False)
        self.value = nn.Linear(dim, dim)


class _BlockParamsV2(nn.Module):
    """Parameter holder with ``Swinv2Layer``'s names (V2:596-620)."""

    def __init__(self, dim: int, heads: int, eps: float):
        super().__init__()
        self.attention = _holder(self=_SelfAttnParamsV2(dim, heads), output=_holder(dense=nn.Linear(dim, dim)))
        self.layernorm_before = nn.LayerNorm(dim, eps=eps)
        self.intermediate = _holder(dense=nn.Linear(dim, 4 * dim))
        self.output = _holder(dense=nn.Linear(4 * dim, dim))
        self.layernorm_after = nn.LayerNorm(dim, eps=eps)


def relative_coords_table(ws: int, pretrained_ws: int = 0) -> torch.Tensor:
    """[(2ws-1)^2, 2] log-spaced relative coordinates, row (dy + ws - 1) * (2ws - 1) + (dx + ws - 1)   (V2:489-510)."""
    r = torch.arange(-(ws - 1), ws, dtype=torch.float32)
    t = torch.stack(torch.meshgrid([r, r], indexing="ij"), dim=-1)
    if pretrained_ws > 0:
        t = t / (pretrained_ws - 1)
    elif ws > 1:
        t = t / (ws - 1)
    t = t * 8
    t = torch.sign(t) * torch.log2(torch.abs(t) + 1.0) / math.log2(8)
    return t.reshape(-1, 2)


def _attn_tables_log2(sa: _SelfAttnParamsV2, coords: torch.Tensor, ws: int, heads: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """The tcgen05 attention cores' per-head inputs, built differentiably from the parameters (V2:450-460, log2 domain):
    ``qs [heads]`` = log2 e * exp(min(logit_scale, ln 100)) and the contiguous padded ``bl2`` = log2 e * 16 sigmoid(cpb_mlp(coords)),
    ``[heads, 31, 48]`` for 16 x 16 windows or ``[heads, 15, 24]`` for 8 x 8 (``coords``: ``relative_coords_table(ws, ...)``)."""
    P = 2 * ws - 1
    qs = torch.clamp(sa.logit_scale, max=math.log(1.0 / 0.01)).exp().reshape(heads) * _LOG2E
    table = sa.continuous_position_bias_mlp(coords)                                                          # [P * P, heads]
    bl2 = torch.nn.functional.pad((16.0 * _LOG2E) * torch.sigmoid(table).t().reshape(heads, P, P), (0, (48 if ws == 16 else 24) - P))
    return qs, bl2.contiguous()


class Swinv2BackboneB200(nn.Module):
    def __init__(self, config: Swinv2ConfigLite, precision: str = "bf16"):
        super().__init__()
        self.config = config
        self.precision = precision
        # 16-bit inference on 16 x 16 windows: the tcgen05 attention kernel (CSVIT_V2_ATTN=mma selects round 1's mma.sync kernel: ablation)
        self._v2_tcgen05 = os.environ.get("CSVIT_V2_ATTN", "tcgen05") != "mma"
        # differentiable path, 16-bit modes, cosine-attention core: torch SDPA (memory-efficient backend) by default;
        # CSVIT_V2_TRAIN_ATTN=tcgen05 runs 16 x 16 windows on the library's tcgen05 forward / backward pair, math: materialised scores
        train_attn = os.environ.get("CSVIT_V2_TRAIN_ATTN", "sdpa")
        self._v2_train_sdpa = train_attn != "math"
        self._v2_train_tc = train_attn == "tcgen05"
        # 8 x 8 windows (the last stage at 256^2; every stage of the window-8 checkpoints), 16-bit modes, opt-in and independent of the
        # switches above: CSVIT_V2_ATTN8=tcgen05 for inference (default mma: round 1's mma.sync kernel), CSVIT_V2_TRAIN_ATTN8=tcgen05 for the
        # differentiable path (default sdpa: the core of CSVIT_V2_TRAIN_ATTN's SDPA / math choice)
        self._v2_tcgen05_8 = os.environ.get("CSVIT_V2_ATTN8", "mma") == "tcgen05"
        self._v2_train_tc8 = os.environ.get("CSVIT_V2_TRAIN_ATTN8", "sdpa") == "tcgen05"
        # CSVIT_V2_TRAIN_BLOCK=fused (opt-in): in the 16-bit modes with 16-bit Linears, every block with 16 x 16 or 8 x 8 windows runs as ONE
        # autograd Function (autograd.Swinv2BlockFn, on those windows' tcgen05 cores) instead of the op-level chain below
        self._v2_train_block = os.environ.get("CSVIT_V2_TRAIN_BLOCK", "off") == "fused"
        c0, eps = config.embed_dim, config.layer_norm_eps
        self.embeddings = _holder(
            patch_embeddings=_holder(projection=nn.Conv2d(3, c0, kernel_size=4, stride=4)),
            norm=nn.LayerNorm(c0, eps=eps))
        stages: List[nn.Module] = []
        for s, (depth, heads) in enumerate(zip(config.depths, config.num_heads)):
            dim = c0 * 2 ** s
            stage = nn.Module()
            stage.blocks = nn.ModuleList([_BlockParamsV2(dim, heads, eps) for _ in range(depth)])
            if s < len(config.depths) - 1:
                stage.downsample = _holder(reduction=nn.Linear(4 * dim, 2 * dim, bias=False), norm=nn.LayerNorm(2 * dim, eps=eps))
            stages.append(stage)
        self.encoder = _holder(layers=nn.ModuleList(stages))
        self.layernorm = nn.LayerNorm(config.hidden_size, eps=eps)
        self._pack = PackCache()
        self._drop_path_rand: List[torch.Tensor] = []   # test hook: the [B] uniform draws of the next stochastic-depth calls, in call order

    # ------------------------------------------------------------------------------------------ construction
    @classmethod
    def from_pretrained(cls, path: str, precision: str = "bf16") -> "Swinv2BackboneB200":
        """Load an HF-format directory (``config.json`` + ``model.safetensors`` / ``pytorch_model.bin``)."""
        with open(os.path.join(path, "config.json")) as f:
            cfg = Swinv2ConfigLite.from_dict(json.load(f))
        model = cls(cfg, precision)
        st = os.path.join(path, "model.safetensors")
        if os.path.exists(st):
            from safetensors.torch import load_file
            sd = load_file(st)
        else:
            sd = torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu")
        sd = {(k[len("swinv2."):] if k.startswith("swinv2.") else k): v for k, v in sd.items()}
        missing, unexpected = model.load_state_dict(sd, strict=False)
        # old checkpoints carry the (recomputable) coordinate table / index buffers; pooler / classifier heads are not used
        unexpected = [k for k in unexpected if not (k.startswith("pooler") or k.startswith("classifier")
                                                    or k.endswith("relative_coords_table") or k.endswith("relative_position_index"))]
        if missing or unexpected:
            raise RuntimeError(f"backbone checkpoint mismatch: missing {missing[:5]} unexpected {unexpected[:5]}")
        model.eval()
        return model

    # ------------------------------------------------------------------------------------------ packing
    @property
    def _fp32(self) -> bool:
        if self.precision not in PRECISIONS and self.precision != "fp8":
            raise ValueError(f"precision must be one of {sorted(PRECISIONS) + ['fp8']}, got {self.precision!r}")
        return self.precision == "fp32"

    @property
    def _fp8(self) -> bool:
        """Inference mode "fp8": the Q/K/V and fc1 GEMMs on E4M3 operands (per-token scales from the LayerNorm kernel that writes
        their operand, per-channel weight scales); every other op, and every activation, as in "fp16"."""
        return self.precision == "fp8"

    @property
    def _act_dtype(self) -> torch.dtype:
        _ = self._fp32
        return torch.float16 if self._fp8 else PRECISIONS[self.precision]

    def _weight_fp8(self, key: str, tensors, build) -> Tuple[torch.Tensor, torch.Tensor]:
        """(E4M3 weight, fp32 per-channel scale) of a Linear, packed once per parameter version."""
        return self._w(key, tensors, lambda: ops.quantize_weight_fp8(build()))

    def _w(self, key: str, tensors, build):
        return self._pack.get(f"{self.precision}/{key}", tensors, build)

    def _weight(self, key: str, lin_weight: torch.Tensor) -> torch.Tensor:
        dt = self._act_dtype
        return self._w(key, [lin_weight], lambda: lin_weight.detach().reshape(lin_weight.shape[0], -1).to(dt).contiguous())

    def _f32(self, key: str, t: torch.Tensor) -> torch.Tensor:
        return self._w(key, [t], lambda: t.detach().float().contiguous())

    def _attn_tables(self, sa: _SelfAttnParamsV2, key: str, ws: int, pretrained_ws: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """([heads, (2ws-1)^2] bias table = 16 sigmoid(cpb_mlp(coords)), [heads] exp(min(logit_scale, ln 100))): functions of the
        parameters only (V2:455-472), so they are evaluated once per parameter version (a pack step like ``fold_batchnorm``, not
        part of the per-image path): the CPB-MLP is a 2 -> 512 -> heads net on (2ws-1)^2 <= 961 points."""
        mlp = sa.continuous_position_bias_mlp
        src = [mlp[0].weight, mlp[0].bias, mlp[2].weight]

        def build_bias():
            dev = mlp[0].weight.device
            t = relative_coords_table(ws, pretrained_ws).to(dev)
            w0 = mlp[0].weight.detach().float()
            hid = torch.relu(t[:, :1] * w0[:, 0] + t[:, 1:] * w0[:, 1] + mlp[0].bias.detach().float())
            tab = hid @ mlp[2].weight.detach().float().t()
            return (16.0 * torch.sigmoid(tab)).t().contiguous()

        bias = self._pack.get(f"fp32/{key}cpb{ws}", src, build_bias)
        scale = self._pack.get(f"fp32/{key}lscale", [sa.logit_scale],
                               lambda: torch.clamp(sa.logit_scale.detach().float().reshape(-1), max=math.log(1.0 / 0.01)).exp().contiguous())
        return bias, scale

    # ------------------------------------------------------------------------------------------ forward
    def _copy_spec(self, s: int, i: int) -> Tuple[int, Tuple[int, int, int, int]]:
        """Where the LayerNorm kernel that FINISHES block (s, i) must put the 16-bit copy of x: the next block's window order,
        the patch-merging concat, or nowhere (last block of the network)."""
        cfg = self.config
        res, ws, shift = cfg.stage_geometry(s)
        if i + 1 < cfg.depths[s]:
            return ops.COPY_WINDOW, (res, res, ws, shift if (i + 1) % 2 == 1 else 0)
        if s + 1 < len(cfg.depths):
            return ops.COPY_MERGE2X2, (res, res, 1, 0)
        return ops.COPY_NONE, (res, res, 1, 0)

    def forward_features(self, images: torch.Tensor, normalize: bool, return_stages: bool = False):
        """images fp32 ``[n,3,S,S]``; ``normalize`` folds the ImageNet mean/std of ref:cs_vit/net/ti_poser.py:239-243 into the
        patch unfold.  Returns fp32 ``[n, (S/32)^2, hidden]``."""
        cfg = self.config
        if not images.is_cuda:
            raise RuntimeError("Swinv2BackboneB200 runs on CUDA tensors only (there is no CPU fallback)")
        n, _, S, S2 = images.shape
        if S != S2 or S != cfg.image_size:
            # HF fixes each layer's window / shift from config.image_size (V2:603-606); other input sizes would need its
            # padding path, which is not built
            raise ValueError(f"image side {S}x{S2} must equal the backbone's image_size {cfg.image_size}")
        for s in range(len(cfg.depths)):
            res, ws, _ = cfg.stage_geometry(s)
            if res % ws != 0 or res % 2 != 0 and s + 1 < len(cfg.depths):
                raise ValueError(f"stage {s}: {res}x{res} tokens not divisible by window {ws} (no padding path)")
        wants_grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if not return_stages and (wants_grad or (self.training and cfg.drop_path_rate > 0)):
            return self._forward_train(images, normalize)
        with torch.no_grad():
            return self._forward_infer(images, normalize, return_stages)

    # ------------------------------------------------------------------------------------------ training path
    def _forward_train(self, images: torch.Tensor, normalize: bool) -> torch.Tensor:
        """Differentiable forward of the finetune step (ref:scripts/finetune.py:211-227 with a swinv2 backbone, which is what every
        shipped configuration uses).  Every Linear, LayerNorm and GELU runs on this library's kernels with kernel backwards
        (cs_vit/autograd.py; 16-bit modes: ``linear16`` - 16-bit tensor-core operands saved and read as stored by the backward GEMMs, fp32
        accumulation / residual stream / gradients; validation mode: exact fp32); the window gather / scatter are permutation Functions
        and stochastic depth a torch elementwise op.  The scaled-cosine attention core (V2:421-487): q / k normalisation + logit scale
        by ``autograd.cosnorm``, then - in the 16-bit modes - ONE library fused attention call per block (torch
        ``scaled_dot_product_attention``, memory-efficient backend) with continuous position bias + 2 x shift mask as its additive term,
        so the [windows, heads, 256, 256] scores are never materialised; the validation mode keeps plain differentiable torch code.
        With ``CSVIT_V2_TRAIN_ATTN=tcgen05``, blocks with 16 x 16 windows in the 16-bit modes run the library's own tcgen05 pair instead
        (``autograd.swinv2_cosine_attention``:
        csvit_swinv2_attn_tc_train / csvit_swinv2_attn_tc_bwd) on the window-ordered [rows, C] operands - no transposing reshapes and no
        [heads, L, L] bias expansion: the bias enters as the log2-domain [heads, 31, 48] table built differentiably from 16 sigmoid(CPB-MLP),
        and its gradient comes back as that table's gradient.  With ``CSVIT_V2_TRAIN_ATTN8=tcgen05``, 8 x 8 windows run the 8 x 8 pair the same
        way (``autograd.swinv2_cosine_attention8``, table [heads, 15, 24]); otherwise they keep SDPA.  With ``CSVIT_V2_TRAIN_BLOCK=fused``
        (16-bit modes and Linears), every block with 16 x 16 or 8 x 8 windows is instead ONE ``autograd.Swinv2BlockFn`` on those tcgen05 cores:
        no permutation Functions, the cosine normalisation in the Q/K/V GEMM epilogue (csvit_swinv2_qkv_train) and its backward in one row
        kernel (csvit_swinv2_cosnorm_bwd).  Matches HF's autograd on the gradient golden (tests/test_swinv2_gpu.py)."""
        from .. import autograd as ag
        if self._fp8:
            raise ValueError("precision='fp8' is inference only: the differentiable path and the finetune step run in bf16, fp16 or fp32")
        cfg = self.config
        n, _, S, _ = images.shape
        impl = ops.GEMM_SIMT if self._fp32 else ops.GEMM_TC
        eps = cfg.layer_norm_eps
        dev = images.device
        cols = ops.patch_im2col(images.float().contiguous(), out_dtype=torch.float32, normalize=normalize)
        pe = self.embeddings.patch_embeddings.projection
        tf32_linear = os.environ.get("CSVIT_V2_TRAIN_LINEAR", "16") == "tf32"
        if self._fp32 or tf32_linear:
            lin = lambda a_, w_, b_, out16=False: ag.linear(a_, w_, b_, impl=impl)    # noqa: E731  (exact fp32 / TF32 on fp32 tensors)
        else:
            lin = lambda a_, w_, b_, out16=False: ag.linear16(a_, w_, b_, self._act_dtype, out16)      # noqa: E731  (16-bit operands)
        x = ag.linear(cols, pe.weight.reshape(pe.weight.shape[0], -1), pe.bias, impl=impl)
        x = ag.LayerNormFn.apply(x, self.embeddings.norm.weight, self.embeddings.norm.bias, eps)
        total_blocks = sum(cfg.depths)
        rates = torch.linspace(0, cfg.drop_path_rate, total_blocks).tolist() if self.training and cfg.drop_path_rate > 0 else [0.0] * total_blocks
        k = -1

        def drop_scale(rate: float) -> Optional[torch.Tensor]:     # [n] per-sample stochastic-depth scale of one branch, one draw
            if rate <= 0.0:
                return None
            keep = 1.0 - rate
            u = self._drop_path_rand.pop(0).to(dev, torch.float32) if self._drop_path_rand else torch.rand(n, device=dev)
            return torch.floor(keep + u) / keep

        def drop_path(branch: torch.Tensor, rate: float, tokens: int) -> torch.Tensor:      # V2: both residual branches (V2:706, 710)
            scale = drop_scale(rate)
            if scale is None:
                return branch
            return (branch.view(n, tokens, -1) * scale[:, None, None]).view(-1, branch.shape[-1])

        for s, stage in enumerate(self.encoder.layers):
            heads = cfg.num_heads[s]
            H, ws, stage_shift = cfg.stage_geometry(s)
            N, L, nW = H * H, ws * ws, (H // ws) ** 2
            C = x.shape[1]
            rel_index = self._w(f"relidx{ws}", [], lambda: ops.rel_pos_index(ws, device=dev).long().reshape(-1))
            coords = self._w(f"coords{ws}_{cfg.pretrained_window_sizes[s]}", [], lambda: relative_coords_table(ws, cfg.pretrained_window_sizes[s]).to(dev))
            for i, blk in enumerate(stage.blocks):
                k += 1
                shift = stage_shift if i % 2 == 1 else 0
                idx = self._w(f"widx{H}_{ws}_{shift}", [], lambda: ops.window_index_map(H, H, ws, shift, device=dev).long())
                inv = self._w(f"winv{H}_{ws}_{shift}", [], lambda: torch.argsort(ops.window_index_map(H, H, ws, shift, device=dev).long()))
                sa = blk.attention.self
                if self._v2_train_block and ws in (8, 16) and not self._fp32 and not tf32_linear:
                    # the whole block as one Function; both stochastic-depth draws are taken here, in the op-level path's order
                    # (attention branch, then MLP branch)
                    qs, bl2 = _attn_tables_log2(sa, coords, ws, heads)
                    s_a = drop_scale(rates[k])
                    s_m = drop_scale(rates[k])
                    x = ag.swinv2_block(x, blk, qs, bl2, s_a, s_m, n, H, ws, shift, heads, eps, self._act_dtype)
                    continue
                xw = ag.permute_rows(x.view(n, N, C), idx, inv).reshape(n * N, C)   # roll(-s) + window_partition as one gather
                q = lin(xw, sa.query.weight, sa.query.bias)
                kk = lin(xw, sa.key.weight, None)
                v = lin(xw, sa.value.weight, sa.value.bias, out16=True)
                if ws == 16 and self._v2_train_tc and not self._fp32:
                    # 16 x 16 windows, 16-bit modes: the tcgen05 core in the log2 domain; q2 = q_hat * logit_scale * log2 e, k_hat and v go in
                    # as the window-ordered [rows, C] rows of the Linears, ctx comes out in the same order for the out-projection
                    act = self._act_dtype
                    d = C // heads
                    qs, bl2 = _attn_tables_log2(sa, coords, ws, heads)
                    q2 = ag.cosnorm(q.view(n * N, heads, d), qs, act).view(n * N, C)
                    kn = ag.cosnorm(kk.view(n * N, heads, d), None, act).view(n * N, C)
                    ctx = ag.swinv2_cosine_attention(q2, kn, v, bl2, n, H, H, heads, shift)
                elif ws == 8 and self._v2_train_tc8 and not self._fp32:
                    # 8 x 8 windows: the same construction on the 8 x 8 pair, bias table [heads, 15, 24]
                    act = self._act_dtype
                    d = C // heads
                    qs, bl2 = _attn_tables_log2(sa, coords, ws, heads)
                    q2 = ag.cosnorm(q.view(n * N, heads, d), qs, act).view(n * N, C)
                    kn = ag.cosnorm(kk.view(n * N, heads, d), None, act).view(n * N, C)
                    ctx = ag.swinv2_cosine_attention8(q2, kn, v, bl2, n, H, H, heads, shift)
                else:
                    lscale = torch.clamp(sa.logit_scale, max=math.log(1.0 / 0.01)).exp()                             # V2:450-453
                    qh, kh, vh = (t.view(n * nW, L, heads, C // heads).transpose(1, 2) for t in (q, kk, v))
                    table = sa.continuous_position_bias_mlp(coords)                                                      # [(2ws-1)^2, heads]
                    bias = 16.0 * torch.sigmoid(table[rel_index].view(L, L, heads).permute(2, 0, 1))                     # V2:455-460
                    mask = self._w(f"mask{H}_{ws}_{shift}", [], lambda: ops.shift_mask(H, H, ws, shift, device=dev)) if shift > 0 else None
                    if self._v2_train_sdpa and not self._fp32:
                        # 16-bit modes: the core as ONE fused library attention (torch SDPA, memory-efficient backend) instead of materialised
                        # [windows, heads, L, L] fp32 scores forward and backward.  q is normalised and scaled, k normalised, in fp32 before the
                        # 16-bit cast; (window, head) is folded into SDPA's head dimension so that the additive term bias (+ 2 * shift mask,
                        # HF adds the mask twice: V2:462-468) broadcasts over the images and receives its gradient.
                        act = self._act_dtype
                        d = C // heads
                        # F.normalize + logit scale (V2:450-455) on the Linear's own [rows, heads, d] layout, straight to 16 bit
                        qn = ag.cosnorm(q.view(n * N, heads, d), lscale.reshape(heads), act).view(n * nW, L, heads, d).transpose(1, 2)
                        kn = ag.cosnorm(kk.view(n * N, heads, d), None, act).view(n * nW, L, heads, d).transpose(1, 2)
                        from torch.nn.attention import SDPBackend, sdpa_kernel
                        with sdpa_kernel([SDPBackend.EFFICIENT_ATTENTION, SDPBackend.MATH]):     # (the automatic choice takes the math path here)
                            if mask is None:
                                # no shift mask: one bias [1, heads, L, L] for every window - windows fold into the batch and q / k / v go in as the
                                # strided [n * nW, heads, L, d] views of the Linear outputs (no transposing copies)
                                add = bias[None].to(act).contiguous()          # (a permuted-stride bias sends SDPA down its math path)
                                ctx = torch.nn.functional.scaled_dot_product_attention(qn, kn, vh, attn_mask=add, scale=1.0)
                            else:
                                add = (bias[None] + 2.0 * mask[:, None]).reshape(1, nW * heads, L, L).to(act).contiguous()
                                q4, k4, v4 = (t.reshape(n, nW * heads, L, d) for t in (qn, kn, vh))
                                ctx = torch.nn.functional.scaled_dot_product_attention(q4, k4, v4, attn_mask=add, scale=1.0)
                        ctx = ctx.reshape(n * nW, heads, L, d).transpose(1, 2).reshape(n * N, C)        # stays 16 bit: the out-proj's operand
                    else:
                        scores = torch.nn.functional.normalize(qh, dim=-1) @ torch.nn.functional.normalize(kh, dim=-1).transpose(-1, -2)
                        scores = scores * lscale + bias[None]
                        if mask is not None:
                            scores = (scores.view(n, nW, heads, L, L) + 2.0 * mask[None, :, None]).view(n * nW, heads, L, L)
                        ctx = (scores.softmax(dim=-1) @ vh.float()).transpose(1, 2).reshape(n * N, C)
                proj = blk.attention.output.dense
                ya = lin(ctx.contiguous(), proj.weight, proj.bias)
                ya = ag.permute_rows(ya.view(n, N, C), inv, idx).reshape(n * N, C)  # window_reverse + roll(+s)
                ya = ag.LayerNormFn.apply(ya.contiguous(), blk.layernorm_before.weight, blk.layernorm_before.bias, eps)
                x = x + drop_path(ya, rates[k], N)                                                                   # res-post-norm, V2:705-706
                fc1, fc2 = blk.intermediate.dense, blk.output.dense
                hid = ag.gelu(lin(x, fc1.weight, fc1.bias, out16=True))
                z = lin(hid, fc2.weight, fc2.bias)
                z = ag.LayerNormFn.apply(z, blk.layernorm_after.weight, blk.layernorm_after.bias, eps)
                x = x + drop_path(z, rates[k], N)                                                                    # V2:708-710
            if hasattr(stage, "downsample"):
                ds = stage.downsample
                g4 = x.view(n, H, H, C)
                cat = torch.cat([g4[:, 0::2, 0::2], g4[:, 1::2, 0::2], g4[:, 0::2, 1::2], g4[:, 1::2, 1::2]], dim=-1).reshape(-1, 4 * C)
                x = lin(cat.contiguous(), ds.reduction.weight, None)                                # V2: reduction, then norm
                x = ag.LayerNormFn.apply(x, ds.norm.weight, ds.norm.bias, eps)
        Hl = cfg.stage_geometry(len(cfg.depths) - 1)[0]
        out = ag.LayerNormFn.apply(x, self.layernorm.weight, self.layernorm.bias, eps)
        return out.view(n, Hl * Hl, cfg.hidden_size)

    def _forward_infer(self, images: torch.Tensor, normalize: bool, return_stages: bool):
        cfg = self.config
        n, _, S, _ = images.shape
        act = self._act_dtype
        impl = ops.GEMM_SIMT if self._fp32 else ops.GEMM_TC
        eps = cfg.layer_norm_eps
        dev = images.device
        fp8 = self._fp8
        qdt = torch.float8_e4m3fn if fp8 else act      # the Q/K/V and fc1 operand copies: (E4M3, row scale) pairs in fp8 mode
        cols = ops.patch_im2col(images.float().contiguous(), out_dtype=act, normalize=normalize)
        pe = self.embeddings.patch_embeddings.projection
        y = ops.linear(cols, self._weight("pe_w", pe.weight), self._f32("pe_b", pe.bias), out_dtype=torch.float32, impl=impl)
        res0, ws0, _ = cfg.stage_geometry(0)
        # x = LN(patch embedding), plus its copy in block (0, 0)'s window order
        x, xw = ops.layernorm_post(y, None, self._f32("pe_lnw", self.embeddings.norm.weight), self._f32("pe_lnb", self.embeddings.norm.bias),
                                   eps, out=y, copy_mode=ops.COPY_WINDOW, copy_dtype=qdt, geom=(res0, res0, ws0, 0))
        stages = []
        for s, stage in enumerate(self.encoder.layers):
            heads = cfg.num_heads[s]
            H, ws, stage_shift = cfg.stage_geometry(s)
            C = x.shape[1]
            for i, blk in enumerate(stage.blocks):
                key = f"s{s}b{i}/"
                shift = stage_shift if i % 2 == 1 else 0
                sa = blk.attention.self
                qkv_src = [sa.query.weight, sa.key.weight, sa.value.weight]
                if fp8:
                    wqkv8, sqkv = self._weight_fp8(key + "wqkv8", qkv_src, lambda: torch.cat([w.detach() for w in qkv_src], 0))
                    qkv_proj = lambda b_, qs_: ops.swinv2_qkv_fp8(xw[0], xw[1], wqkv8, sqkv, b_, qs_, out_dtype=act)   # noqa: E731
                else:
                    wqkv = self._w(key + "wqkv", qkv_src, lambda: torch.cat([w.detach() for w in qkv_src], 0).to(act).contiguous())
                    qkv_proj = lambda b_, qs_: ops.swinv2_qkv(xw, wqkv, b_, qs_)                                            # noqa: E731
                bqkv_src = [sa.query.bias, sa.value.bias]
                bqkv = self._w(key + "bqkv", bqkv_src, lambda: torch.cat(
                    [sa.query.bias.detach().float(), torch.zeros_like(sa.query.bias, dtype=torch.float32), sa.value.bias.detach().float()], 0).contiguous())
                bias_tab, lscale = self._attn_tables(sa, key, ws, cfg.pretrained_window_sizes[s])
                # the attention kernels un-partition / un-shift on their store: the out-proj runs on plain token rows
                if ws == 16 and not self._fp32 and self._v2_tcgen05:
                    # 256-token windows, 16-bit operands: both F.normalize and the logit scale in the Q/K/V GEMM epilogue, attention
                    # on tcgen05 with the probabilities kept in TMEM (csvit_swinv2_qkv + csvit_swinv2_attn_tc)
                    qs = self._pack.get(f"fp32/{key}qscale2", [sa.logit_scale], lambda: (lscale * 1.4426950408889634).contiguous())
                    bl2 = self._pack.get(f"fp32/{key}cpb{ws}log2", [bias_tab], lambda: ops.swinv2_bias_log2(bias_tab))
                    qkv = qkv_proj(bqkv, qs)
                    ctx = ops.swinv2_attn_tc(qkv, bl2, n, H, H, heads, shift, token_order=True)
                elif ws == 8 and not self._fp32 and self._v2_tcgen05_8:
                    # 64-token windows on the tcgen05 8 x 8 kernel (CSVIT_V2_ATTN8=tcgen05)
                    qs = self._pack.get(f"fp32/{key}qscale2", [sa.logit_scale], lambda: (lscale * 1.4426950408889634).contiguous())
                    bl2 = self._pack.get(f"fp32/{key}cpb{ws}log2", [bias_tab], lambda: ops.swinv2_bias8_log2(bias_tab))
                    qkv = qkv_proj(bqkv, qs)
                    ctx = ops.swinv2_attn8_tc(qkv, bl2, n, H, H, heads, shift, token_order=True)
                elif fp8:
                    qkv = ops.linear_fp8(xw[0], xw[1], wqkv8, sqkv, bqkv, out_dtype=act)
                    ctx = ops.swinv2_window_attention(qkv, bias_tab, lscale, n, H, H, heads, ws, shift, token_order=True)
                else:
                    qkv = ops.linear(xw, wqkv, bqkv, out_dtype=act, impl=impl)
                    ctx = ops.swinv2_window_attention(qkv, bias_tab, lscale, n, H, H, heads, ws, shift, token_order=True)
                proj = blk.attention.output.dense
                ya = ops.linear(ctx, self._weight(key + "wproj", proj.weight), self._f32(key + "bproj", proj.bias), out_dtype=torch.float32,
                                impl=impl)
                ln1, ln2 = blk.layernorm_before, blk.layernorm_after
                _, x16 = ops.layernorm_post(ya, x, self._f32(key + "ln1w", ln1.weight), self._f32(key + "ln1b", ln1.bias), eps, out=x,
                                            copy_mode=ops.COPY_IDENTITY, copy_dtype=qdt)
                fc1, fc2 = blk.intermediate.dense, blk.output.dense
                if fp8:
                    w18, s1 = self._weight_fp8(key + "w18", [fc1.weight], lambda: fc1.weight.detach())
                    hid = ops.linear_fp8(x16[0], x16[1], w18, s1, self._f32(key + "b1", fc1.bias), act=ops.ACT_GELU, out_dtype=act)
                else:
                    hid = ops.linear(x16, self._weight(key + "w1", fc1.weight), self._f32(key + "b1", fc1.bias), act=ops.ACT_GELU,
                                     out_dtype=act, impl=impl)
                z = ops.linear(hid, self._weight(key + "w2", fc2.weight), self._f32(key + "b2", fc2.bias), out_dtype=torch.float32, impl=impl)
                mode, geom = self._copy_spec(s, i)
                _, xw = ops.layernorm_post(z, x, self._f32(key + "ln2w", ln2.weight), self._f32(key + "ln2b", ln2.bias), eps, out=x,
                                           copy_mode=mode, copy_dtype=qdt if mode == ops.COPY_WINDOW else act, geom=geom)
            if return_stages:
                stages.append(x.view(n, H * H, C).clone())
            if hasattr(stage, "downsample"):
                ds = stage.downsample
                red = ops.linear(xw, self._weight(f"s{s}/dsr", ds.reduction.weight), None, out_dtype=torch.float32, impl=impl)
                Hn, wsn, _ = cfg.stage_geometry(s + 1)
                x, xw = ops.layernorm_post(red, None, self._f32(f"s{s}/dsw", ds.norm.weight), self._f32(f"s{s}/dsb", ds.norm.bias), eps,
                                           out=red, copy_mode=ops.COPY_WINDOW, copy_dtype=qdt, geom=(Hn, Hn, wsn, 0))
        Hl = cfg.stage_geometry(len(cfg.depths) - 1)[0]
        out = ops.layernorm(x, self._f32("final_w", self.layernorm.weight), self._f32("final_b", self.layernorm.bias), eps)
        out = out.view(n, Hl * Hl, cfg.hidden_size)
        return (out, stages) if return_stages else out

    def forward(self, pixel_values: torch.Tensor, **_unused) -> SimpleNamespace:
        """HF seam: ``pixel_values`` are already normalised   (ref:cs_vit/net/ti_poser.py:425-426)."""
        return SimpleNamespace(last_hidden_state=self.forward_features(pixel_values, normalize=False), pooler_output=None)


def load_backbone(path: str, precision: str = "bf16") -> nn.Module:
    """``AutoModel.from_pretrained(path)`` of the reference (ref:cs_vit/net/ti_poser.py:246): picks the kernel backbone from the
    directory's ``config.json``; unknown model types fail loudly (there is no fallback to HF modules)."""
    from .swin_b200 import SwinBackboneB200
    with open(os.path.join(path, "config.json")) as f:
        model_type = json.load(f).get("model_type", "swin")
    if model_type == "swin":
        return SwinBackboneB200.from_pretrained(path, precision=precision)
    if model_type == "swinv2":
        return Swinv2BackboneB200.from_pretrained(path, precision=precision)
    raise NotImplementedError(f"backbone model_type '{model_type}' has no sm_100a kernels (built: swin, swinv2)")
