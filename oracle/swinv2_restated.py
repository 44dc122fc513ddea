"""Restatement of the HuggingFace SwinV2 forward (the backbone of every shipped CS-ViT config).  TEST INFRASTRUCTURE.

Follows ``transformers/models/swinv2/modeling_swinv2.py`` (abbreviated V2:) as executed through
``AutoModel.from_pretrained(dir)(pixel_values).last_hidden_state`` (ref:cs_vit/net/ti_poser.py:246,426; the shipped
configs name ``swinv2-*-patch4-window16-256`` directories, SURVEY.md §0.2).  Written with the tensor shuffles of the
original (roll / view / permute, slice-assigned region image) rather than the closed-form maps of the CUDA kernels, so
the two derivations check each other.  Pure functions of a ``state_dict`` in the HF key schema, evaluated in its dtype
and on its device: CPU fp32 for the goldens and the benchmark's CPU baseline, fp64 on the GPU for the batch-256 SwinV2-B
reference (tests/test_swinv2b_batch256_gpu.py).  Pinned against the live ``Swinv2Model`` by ``oracle/make_swinv2_goldens.py``.
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence, Tuple

import torch
import torch.nn.functional as F

from .swin_restated import (_lin, _ln, patch_embed, relative_position_index, shift_attention_mask, window_partition,
                            window_reverse)

Tensor = torch.Tensor


def window_and_shift(res: int, window: int, shift: int) -> Tuple[int, int]:
    """``Swinv2Layer._compute_window_shift`` for square maps   (V2:622-625)."""
    ws = min(res, window)
    return ws, (0 if res <= ws else shift)


def relative_coords_table(ws: int, pretrained_ws: int = 0) -> Tensor:
    """[(2ws-1)^2, 2] log-spaced relative coordinates   (V2:489-510)."""
    r = torch.arange(-(ws - 1), ws, dtype=torch.int64).float()
    table = torch.stack(torch.meshgrid([r, r], indexing="ij")).permute(1, 2, 0).contiguous().unsqueeze(0)
    if pretrained_ws > 0:
        table = table / (pretrained_ws - 1)
    elif ws > 1:
        table = table / (ws - 1)
    table = table * 8
    table = torch.sign(table) * torch.log2(torch.abs(table) + 1.0) / math.log2(8)
    return table.reshape(-1, 2)


def continuous_position_bias(sd: Dict[str, Tensor], p: str, ws: int, heads: int, pretrained_ws: int = 0) -> Tensor:
    """16 sigmoid(cpb_mlp(coords))[rel index] -> [heads, L, L]   (V2:460-472)."""
    w0 = sd[p + ".continuous_position_bias_mlp.0.weight"]
    t = relative_coords_table(ws, pretrained_ws).to(w0)                                  # the state dict's dtype and device
    hid = F.relu(F.linear(t, w0, sd[p + ".continuous_position_bias_mlp.0.bias"]))
    table = F.linear(hid, sd[p + ".continuous_position_bias_mlp.2.weight"])              # [(2ws-1)^2, heads]
    L = ws * ws
    bias = table[relative_position_index(ws).reshape(-1).to(table.device)].reshape(L, L, heads).permute(2, 0, 1)
    return 16 * torch.sigmoid(bias)


def cosine_window_attention(xw: Tensor, sd: Dict[str, Tensor], p: str, heads: int, ws: int, mask, pretrained_ws: int = 0) -> Tensor:
    """xw [nWB, L, C] -> [nWB, L, C]: Swinv2SelfAttention + Swinv2SelfOutput   (V2:421-487, 528-538)."""
    nWB, L, C = xw.shape
    d = C // heads

    def split(t):
        return t.reshape(nWB, L, heads, d).transpose(1, 2)

    q = split(_lin(xw, sd, p + ".self.query"))
    k = split(F.linear(xw, sd[p + ".self.key.weight"]))                                  # no key bias (V2:414)
    v = split(_lin(xw, sd, p + ".self.value"))
    scores = F.normalize(q, dim=-1) @ F.normalize(k, dim=-1).transpose(-2, -1)           # V2:452-454
    scale = torch.clamp(sd[p + ".self.logit_scale"], max=math.log(1.0 / 0.01)).exp()     # V2:455
    scores = scores * scale
    scores = scores + continuous_position_bias(sd, p + ".self", ws, heads, pretrained_ws)[None]
    if mask is not None:                                                                 # V2:466-474: the mask is added twice
        nW = mask.shape[0]
        mask = mask.to(scores)
        scores = scores.reshape(nWB // nW, nW, heads, L, L) + mask[None, :, None]
        scores = scores + mask[None, :, None]
        scores = scores.reshape(nWB, heads, L, L)
    probs = scores.softmax(-1)
    ctx = (probs @ v).transpose(1, 2).reshape(nWB, L, C)
    return _lin(ctx, sd, p + ".output.dense")


def swinv2_layer(x: Tensor, sd: Dict[str, Tensor], p: str, H: int, W: int, heads: int, window: int, shift: int, eps: float,
                 pretrained_ws: int = 0) -> Tensor:
    """One Swinv2Layer on x [B, H*W, C] (res-post-norm)   (V2:662-715).  H, W multiples of the window (no padding path)."""
    B, N, C = x.shape
    ws, shift = window_and_shift(min(H, W), window, shift)
    shortcut = x
    h = x.reshape(B, H, W, C)
    if shift > 0:
        h = torch.roll(h, shifts=(-shift, -shift), dims=(1, 2))
    windows = window_partition(h, ws).reshape(-1, ws * ws, C)
    mask = shift_attention_mask(H, W, ws, shift) if shift > 0 else None
    a = cosine_window_attention(windows, sd, p + ".attention", heads, ws, mask, pretrained_ws)
    h = window_reverse(a.reshape(-1, ws, ws, C), ws, H, W)
    if shift > 0:
        h = torch.roll(h, shifts=(shift, shift), dims=(1, 2))
    x = shortcut + _ln(h.reshape(B, N, C), sd, p + ".layernorm_before", eps)             # V2:707-708
    y = F.gelu(_lin(x, sd, p + ".intermediate.dense"))
    y = _lin(y, sd, p + ".output.dense")
    return x + _ln(y, sd, p + ".layernorm_after", eps)                                   # V2:710-712


def patch_merging_v2(x: Tensor, sd: Dict[str, Tensor], p: str, H: int, W: int, eps: float) -> Tensor:
    """[B, H*W, C] -> [B, H*W/4, 2C]: concat -> reduction -> norm   (V2:365-388)."""
    B, N, C = x.shape
    g = x.reshape(B, H, W, C)
    cat = torch.cat([g[:, 0::2, 0::2], g[:, 1::2, 0::2], g[:, 0::2, 1::2], g[:, 1::2, 1::2]], dim=-1).reshape(B, -1, 4 * C)
    return _ln(F.linear(cat, sd[p + ".reduction.weight"]), sd, p + ".norm", eps)


def swinv2_forward(pixels: Tensor, sd: Dict[str, Tensor], depths: Sequence[int], heads: Sequence[int], window: int = 16,
                   eps: float = 1e-5, pretrained_window_sizes: Sequence[int] = (0, 0, 0, 0), return_stages: bool = False):
    """``Swinv2Model.forward(...).last_hidden_state``   (V2:933-1001, 804-872, 747-775)."""
    S = pixels.shape[-1]
    H = W = S // 4
    x = patch_embed(pixels, sd, eps)                                                     # same as v1 (V2:265-291, 325-334)
    stage_out: List[Tensor] = []
    for s, (depth, h) in enumerate(zip(depths, heads)):
        for i in range(depth):
            shift = 0 if i % 2 == 0 else window // 2                                     # V2:735
            x = swinv2_layer(x, sd, f"encoder.layers.{s}.blocks.{i}", H, W, h, window, shift, eps, pretrained_window_sizes[s])
        stage_out.append(x)
        if s < len(depths) - 1:
            x = patch_merging_v2(x, sd, f"encoder.layers.{s}.downsample", H, W, eps)
            H, W = H // 2, W // 2
    out = _ln(x, sd, "layernorm", eps)
    return (out, stage_out) if return_stages else out
