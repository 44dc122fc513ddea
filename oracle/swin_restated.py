"""Restatement of the HuggingFace Swin-v1 forward (the reference's backbone), CPU fp32 by default.  TEST INFRASTRUCTURE.

Follows ``transformers/models/swin/modeling_swin.py`` (abbreviated HF:) as executed through
``AutoModel.from_pretrained(dir)(pixel_values).last_hidden_state`` (ref:cs_vit/net/ti_poser.py:246,426).
It is deliberately written with the *tensor shuffles* the original uses (roll / view / permute, slice-assigned
region image for the mask) rather than the closed-form index maps of the CUDA kernels, so that the two
derivations check each other.  Everything is a pure function of a ``state_dict`` in the HF key schema, evaluated in
that state dict's dtype and on its device (the index and mask tensors built here follow it).
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


# ------------------------------------------------------------------------------------------------ integer logic
def window_partition(x: Tensor, ws: int) -> Tensor:
    """[B,H,W,C] -> [B*nW, ws, ws, C]   (HF:141-150)."""
    B, H, W, C = x.shape
    x = x.reshape(B, H // ws, ws, W // ws, ws, C)
    return x.permute(0, 1, 3, 2, 4, 5).reshape(-1, ws, ws, C)


def window_reverse(win: Tensor, ws: int, H: int, W: int) -> Tensor:
    """[B*nW, ws, ws, C] -> [B,H,W,C]   (HF:153-160)."""
    C = win.shape[-1]
    x = win.reshape(-1, H // ws, W // ws, ws, ws, C)
    return x.permute(0, 1, 3, 2, 4, 5).reshape(-1, H, W, C)


def relative_position_index(ws: int) -> Tensor:
    """[ws*ws, ws*ws] int64   (HF:461-473)."""
    ys, xs = torch.meshgrid(torch.arange(ws), torch.arange(ws), indexing="ij")
    coords = torch.stack([ys.reshape(-1), xs.reshape(-1)])          # [2, L]
    rel = (coords[:, :, None] - coords[:, None, :]).permute(1, 2, 0).contiguous()  # [L, L, 2]
    rel[..., 0] += ws - 1
    rel[..., 1] += ws - 1
    rel[..., 0] *= 2 * ws - 1
    return rel.sum(-1)


def shift_attention_mask(H: int, W: int, ws: int, shift: int) -> Tensor:
    """[nW, L, L] in {0, -100}   (HF:556-582).  ``shift`` must be > 0."""
    img = torch.zeros(1, H, W, 1)
    spans = (slice(0, -ws), slice(-ws, -shift), slice(-shift, None))
    region = 0
    for hs in spans:
        for wsl in spans:
            img[:, hs, wsl, :] = region
            region += 1
    flat = window_partition(img, ws).reshape(-1, ws * ws)
    diff = flat[:, None, :] - flat[:, :, None]
    return torch.where(diff != 0, torch.tensor(-100.0), torch.tensor(0.0))


def window_gather_index(H: int, W: int, ws: int, shift: int) -> Tensor:
    """Flat token id read by (window, slot) after roll(-shift) + window_partition: [nW*L] int64."""
    ids = torch.arange(H * W).reshape(1, H, W, 1)
    if shift > 0:
        ids = torch.roll(ids, shifts=(-shift, -shift), dims=(1, 2))   # HF:615-616
    return window_partition(ids, ws).reshape(-1)


def merge_gather_index(H: int, W: int) -> Tensor:
    """Source tokens of every merged token in HF's concat order: [(H/2)*(W/2), 4] int64   (HF:338-345)."""
    ids = torch.arange(H * W).reshape(H, W)
    parts = [ids[0::2, 0::2], ids[1::2, 0::2], ids[0::2, 1::2], ids[1::2, 1::2]]
    return torch.stack([p.reshape(-1) for p in parts], dim=-1)


# ------------------------------------------------------------------------------------------------ float path
def _ln(x: Tensor, sd: Dict[str, Tensor], prefix: str, eps: float) -> Tensor:
    return F.layer_norm(x, (x.shape[-1],), sd[prefix + ".weight"], sd[prefix + ".bias"], eps)


def _lin(x: Tensor, sd: Dict[str, Tensor], prefix: str) -> Tensor:
    return F.linear(x, sd[prefix + ".weight"], sd.get(prefix + ".bias"))


def window_self_attention(xw: Tensor, sd: Dict[str, Tensor], p: str, heads: int, ws: int, mask) -> Tensor:
    """xw [nWB, L, C] -> [nWB, L, C]: SwinSelfAttention + SwinSelfOutput   (HF:410-459, 476-486)."""
    nWB, L, C = xw.shape
    d = C // heads

    def split(t):
        return t.reshape(nWB, L, heads, d).transpose(1, 2)

    q = split(_lin(xw, sd, p + ".self.query"))
    k = split(_lin(xw, sd, p + ".self.key"))
    v = split(_lin(xw, sd, p + ".self.value"))
    scores = (q @ k.transpose(-1, -2)) / math.sqrt(d)                                   # HF:424-426
    table = sd[p + ".self.relative_position_bias_table"]
    index = sd.get(p + ".self.relative_position_index", relative_position_index(ws))
    bias = table[index.reshape(-1).to(table.device)].reshape(L, L, heads).permute(2, 0, 1)  # HF:428-434
    scores = scores + bias[None]
    if mask is not None:                                                                # HF:436-443
        nW = mask.shape[0]
        mask = mask.to(scores)
        scores = (scores.reshape(nWB // nW, nW, heads, L, L) + mask[None, :, None]).reshape(nWB, heads, L, L)
    probs = scores.softmax(-1)                                                          # HF:446
    ctx = (probs @ v).transpose(1, 2).reshape(nWB, L, C)                                # HF:452-455
    return _lin(ctx, sd, p + ".output.dense")                                           # HF:479-483


def drop_path(x: Tensor, drop_prob: float, u: Tensor) -> Tensor:
    """Stochastic depth per sample with the uniform draw ``u [B]`` made explicit   (HF:353-366: ``floor(keep + rand)``, kept
    samples divided by ``keep``)."""
    keep = 1.0 - drop_prob
    mask = torch.floor(keep + u.to(x.dtype)).reshape((x.shape[0],) + (1,) * (x.dim() - 1))
    return x.div(keep) * mask


def swin_layer(x: Tensor, sd: Dict[str, Tensor], p: str, H: int, W: int, heads: int, ws: int, shift: int, eps: float,
               drop_prob: float = 0.0, drop_u=None) -> Tensor:
    """One SwinLayer on x [B, H*W, C]   (HF:591-653).  H, W must be multiples of ws (no padding path).  ``drop_prob > 0`` with the
    draw ``drop_u [B]``: train-mode stochastic depth of the attention branch (HF:543, 646)."""
    B, N, C = x.shape
    if min(H, W) <= ws:                                   # HF:548-554 set_shift_and_window_size
        shift, ws = 0, min(H, W)
    shortcut = x
    h = _ln(x, sd, p + ".layernorm_before", eps).reshape(B, H, W, C)
    if shift > 0:
        h = torch.roll(h, shifts=(-shift, -shift), dims=(1, 2))
    windows = window_partition(h, ws).reshape(-1, ws * ws, C)
    mask = shift_attention_mask(H, W, ws, shift) if shift > 0 else None
    a = window_self_attention(windows, sd, p + ".attention", heads, ws, mask)
    h = window_reverse(a.reshape(-1, ws, ws, C), ws, H, W)
    if shift > 0:
        h = torch.roll(h, shifts=(shift, shift), dims=(1, 2))
    branch = h.reshape(B, N, C)
    if drop_prob > 0.0:
        branch = drop_path(branch, drop_prob, drop_u)
    x = shortcut + branch                                                                # HF:646
    y = _ln(x, sd, p + ".layernorm_after", eps)
    y = F.gelu(_lin(y, sd, p + ".intermediate.dense"))                                   # exact erf, HF:510-519
    return x + _lin(y, sd, p + ".output.dense")                                          # HF:650


def patch_merging(x: Tensor, sd: Dict[str, Tensor], p: str, H: int, W: int, eps: float) -> Tensor:
    """[B, H*W, C] -> [B, H*W/4, 2C]   (HF:326-349)."""
    B, N, C = x.shape
    g = x.reshape(B, H, W, C)
    cat = torch.cat([g[:, 0::2, 0::2], g[:, 1::2, 0::2], g[:, 0::2, 1::2], g[:, 1::2, 1::2]], dim=-1).reshape(B, -1, 4 * C)
    return F.linear(_ln(cat, sd, p + ".norm", eps), sd[p + ".reduction.weight"])


def patch_embed(pixels: Tensor, sd: Dict[str, Tensor], eps: float) -> Tensor:
    """[B,3,S,S] (already normalised) -> [B, (S/4)^2, C0]   (HF:286-295, 227-252)."""
    y = F.conv2d(pixels, sd["embeddings.patch_embeddings.projection.weight"],
                 sd["embeddings.patch_embeddings.projection.bias"], stride=4)
    y = y.flatten(2).transpose(1, 2)
    return _ln(y, sd, "embeddings.norm", eps)


def swin_forward(pixels: Tensor, sd: Dict[str, Tensor], depths: Sequence[int], heads: Sequence[int], ws: int = 7,
                 eps: float = 1e-5, return_stages: bool = False, drop_path_rate: float = 0.0, drop_draws=None):
    """``SwinModel.forward(...).last_hidden_state``   (HF:847-899, 734-794, 683-708).  ``drop_path_rate > 0`` = train mode with
    stochastic depth: block k uses ``linspace(0, rate, sum(depths))[k]`` (HF:716) and the next row of ``drop_draws [n, B]``."""
    rates = torch.linspace(0, drop_path_rate, sum(depths)).tolist()
    draws = list(drop_draws) if drop_draws is not None else []
    k = -1
    S = pixels.shape[-1]
    H = W = S // 4
    x = patch_embed(pixels, sd, eps)
    stage_out: List[Tensor] = []
    for s, (depth, h) in enumerate(zip(depths, heads)):
        for i in range(depth):
            shift = 0 if i % 2 == 0 else ws // 2                                        # HF:672-680
            k += 1
            p_drop = rates[k] if drop_path_rate > 0.0 else 0.0
            x = swin_layer(x, sd, f"encoder.layers.{s}.blocks.{i}", H, W, h, ws, shift, eps, p_drop,
                           draws.pop(0) if p_drop > 0.0 else None)
        stage_out.append(x)
        if s < len(depths) - 1:
            x = patch_merging(x, sd, f"encoder.layers.{s}.downsample", H, W, eps)
            H, W = H // 2, W // 2
    out = _ln(x, sd, "layernorm", eps)                                                   # HF:882-883
    return (out, stage_out) if return_stages else out
