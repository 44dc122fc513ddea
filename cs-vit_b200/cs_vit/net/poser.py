"""``Poser`` - the CS-ViT hand-pose regressor on the sm_100a kernels (drop-in for ref:cs_vit/net/ti_poser.py).

Public surface kept from the reference (SURVEY.md §8b): constructor arguments and defaults
(ref:cs_vit/net/ti_poser.py:192-210), ``Poser.TrainingPhase``, ``.phase()``, ``.predict_batch()`` with the same
input/output tensors (:641-722), ``.forward(batch)`` with the same return structure (:815-855), and the
``state_dict`` key schema.  What changed is everything underneath: the backbone is ``SwinBackboneB200`` instead
of HF ``AutoModel``, the head runs on the GEMM / attention / affine kernels of ``libcsvit_sm100.so``, image
normalisation is folded into the patch unfold, and for the "encoder" spatial head only the layer whose
output is used is executed (the reference runs six and discards five, quirk Q2).

The tiny fp32 tail (6D -> axis-angle, MANO forward kinematics, loss) stays in PyTorch on the GPU, as
SURVEY.md §2.3 K18-K20 prescribes.
"""
from __future__ import annotations

import os

import math
import os.path as osp
from enum import Enum
from itertools import chain
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn as nn

from .. import autograd as ag
from .. import ops
from ..constants import TARGET_JOINTS_CONNECTION
from ..utils.geometry import axis_angle_to_matrix, matrix_to_axis_angle, rotation_6d_to_matrix
from ..utils.joint import mean_connection_length
from .blocks import (CrossAttnDecoder, DecoderBlock, EncoderBlock, PositionalEncoding, _KernelModule, _flat,
                     set_precision)
from .swin_b200 import SwinBackboneB200  # noqa: F401  (re-exported)
from .swinv2_b200 import load_backbone


def derivative(x: torch.Tensor, dim: int) -> torch.Tensor:
    """Central finite difference along ``dim`` (length shrinks by 2)   (ref:cs_vit/net/ti_poser.py:31-51)."""
    assert dim < x.ndim and x.size(dim) >= 3
    n = x.size(dim)
    return (x.narrow(dim, 2, n - 2) - x.narrow(dim, 0, n - 2)) / 2.0


class SpatialEncoder(_KernelModule):
    def __init__(self, embed_dim: int, num_heads: int, num_layer: int, layer_type: str = "decoder"):
        super().__init__()
        self.embed_dim, self.num_heads, self.num_layer, self.layer_type = embed_dim, num_heads, num_layer, layer_type
        self.pe_spatial = PositionalEncoding(embed_dim, mode="absolute")
        if layer_type == "decoder":
            self.layers = nn.ModuleList([DecoderBlock(embed_dim, num_heads) for _ in range(num_layer)])
        elif layer_type == "encoder":
            self.layers = nn.ModuleList([EncoderBlock(embed_dim, num_heads) for _ in range(num_layer)])
        else:
            raise NotImplementedError(f"unknown layer type: {layer_type}")

    def forward(self, x: torch.Tensor, ctx: torch.Tensor) -> torch.Tensor:
        """x ``(B,Q,D)`` queries, ctx ``(B,L,D)`` patches -> ``(B,Q,D)``   (ref:cs_vit/net/ti_poser.py:80-97)."""
        if self.layer_type == "decoder":
            x = self.pe_spatial(x)
            for layer in self.layers:
                x = layer(x, ctx)
            return x
        # "encoder": the reference feeds the SAME embedded input to every layer and returns the last layer's
        # output (ref :94-97, typo ``x_embeb``), so only layers[-1] contributes to the result.
        z = self.pe_spatial(torch.cat([x, ctx], dim=1))
        return self.layers[-1].forward_queries(z, x.shape[1])


class TemporalEncoder(_KernelModule):
    def __init__(self, embed_dim: int, num_heads: int, num_layer: int, target: str = "realtime",
                 trope_scalar: float = 20.0, do_zero_init: bool = True):
        assert target in ["realtime", "full"]
        super().__init__()
        self.embed_dim, self.num_heads, self.num_layer = embed_dim, num_heads, num_layer
        self.target, self.trope_scalar = target, trope_scalar
        block = EncoderBlock if target == "full" else CrossAttnDecoder
        self.pe_temporal = PositionalEncoding(embed_dim, mode="absolute" if target == "full" else "trope")
        self.layers = nn.ModuleList([block(embed_dim, num_heads) for _ in range(num_layer)])
        self.zero_conv = nn.Linear(embed_dim, embed_dim, bias=False)
        if do_zero_init:
            nn.init.zeros_(self.zero_conv.weight)

    def forward(self, x: torch.Tensor, timestamp: Optional[torch.Tensor] = None,
                key_start: Optional[torch.Tensor] = None) -> torch.Tensor:
        """x ``(B,T,D)``, timestamp ``(B,T)`` ms   (ref:cs_vit/net/ti_poser.py:140-158).

        ``key_start`` (inference only; int32 ``[B]``): clip b attends to its frames ``key_start[b]:T`` only, which gives bit for bit
        the result of a call on that shorter clip: on every slot for the "full" target, whose frame j takes the absolute position
        ``max(j - key_start[b], 0)``; on the newest slot for the realtime target, whose trope angles are relative to that frame."""
        assert (self.target == "realtime" and timestamp is not None) or self.target == "full"
        if self.target == "realtime":
            seq = self.pe_temporal(x, timestamp / self.trope_scalar)
            u = seq[:, -1:]
            for layer in self.layers:
                u = layer(u, seq, key_start=key_start)
        else:
            positions = None
            if key_start is not None:
                slots = torch.arange(x.shape[1], device=x.device)
                positions = torch.clamp(slots[None] - key_start[:, None].long(), min=0)
            u = self.pe_temporal(x, positions=positions)
            for layer in self.layers:
                u = layer(u, key_start=key_start)
        if self._grad(u):
            out = ag.linear(_flat(u), self.zero_conv.weight, None, impl=self._impl)
        else:
            out = ops.linear(_flat(u), self.zero_conv.weight.detach().float(), None, impl=self._impl)
        return out.view(u.shape)


class PerspectiveEncoder(_KernelModule):
    def __init__(self, patch_res: int, persp_dim: int, embed_dim: int):
        super().__init__()
        self.layer = nn.Sequential()
        self.proj = nn.Linear(patch_res * persp_dim, embed_dim)
        for _ in range(3):
            self.layer.extend([nn.BatchNorm1d(embed_dim, affine=True), nn.Linear(embed_dim, embed_dim, bias=True), nn.ReLU()])
        self.layer.append(nn.Linear(embed_dim, embed_dim))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """``(n, patch_res*persp_dim)`` -> ``(n, D)``   (ref:cs_vit/net/ti_poser.py:161-182)."""
        self._check(x)
        last = self.layer[9]
        if self._grad(x):    # differentiable ops (train-mode BatchNorm uses batch statistics)
            y = ag.linear(_flat(x), self.proj.weight, self.proj.bias, impl=self._impl)
            for k in range(3):
                bn, lin = self.layer[3 * k], self.layer[3 * k + 1]
                y = ag.linear(self._norm(f"bn{k}", bn, y, True), lin.weight, lin.bias, act=ops.ACT_RELU, impl=self._impl)
            return ag.linear(y, last.weight, last.bias, impl=self._impl)
        y = ops.linear(_flat(x), self.proj.weight.detach().float(), self.proj.bias.detach().float(), impl=self._impl)
        for k in range(3):
            bn, lin = self.layer[3 * k], self.layer[3 * k + 1]
            y = self._norm(f"bn{k}", bn, y, False)
            y = ops.linear(y, lin.weight.detach().float(), lin.bias.detach().float(), act=ops.ACT_RELU, impl=self._impl)
        return ops.linear(y, last.weight.detach().float(), last.bias.detach().float(), impl=self._impl)


def _load_mano(smplx_path: str, mano_layer: Optional[nn.Module]) -> nn.Module:
    if mano_layer is not None:
        return mano_layer
    if os.environ.get("CSVIT_MANO") == "synthetic":
        # explicit opt-in for boxes without the licensed MANO files (throughput / parity runs of the unmodified reference scripts,
        # whose Poser(...) call has no mano_layer argument): the seeded stand-in used by the tests and the bench
        import warnings
        from ..utils.mano_standin import SyntheticMANO
        warnings.warn("CSVIT_MANO=synthetic: using the seeded MANO stand-in, predicted meshes are NOT anatomical")
        return SyntheticMANO()
    try:
        import smplx  # noqa: F401  (ref:cs_vit/net/ti_poser.py:12,268)
    except ImportError as e:
        raise ImportError(
            "the MANO layer needs the `smplx` package and the licensed MANO files; neither ships with this "
            "repo.  Pass mano_layer=cs_vit.utils.mano_standin.SyntheticMANO() for parity / throughput work.") from e
    return smplx.create(smplx_path, "mano", is_rhand=True, use_pca=False)


class Poser(nn.Module):

    class TrainingPhase(Enum):
        SPATIAL = "spatial"
        TEMPORAL = "temporal"
        INFERENCE = "inference"

    def __init__(
        self,
        backbone: str,
        num_pose_query: int = 16,
        num_spatial_layer: int = 6,
        spatial_layer_type: str = "decoder",
        num_temporal_layer: int = 2,
        temporal_init_method: str = "zero",
        expansion_ratio: float = 1.25,
        temporal_supervision: str = "full",
        trope_scalar: float = 20.0,
        num_latent_layer: Optional[int] = None,
        persp_embed_method: str = "dense",
        persp_decorate: str = "query",
        smplx_path: str = osp.join(osp.dirname(__file__), "../../model/smplx_models"),
        image_size: int = 256,
        global_positioning: str = "direct",
        # --- additions of this implementation (keyword-only in practice) ---
        mano_layer: Optional[nn.Module] = None,
        precision: str = "bf16",
    ):
        super().__init__()
        assert (num_latent_layer is not None and persp_decorate == "patch") or (num_latent_layer is None)
        assert spatial_layer_type in ["decoder", "encoder"]
        assert temporal_supervision in ["full", "realtime"]
        assert persp_embed_method in ["dense", "sparse"]
        assert persp_decorate in ["query", "patch"]
        assert global_positioning in ["direct", "orientation"]

        self.backbone_ckpt_dir = backbone
        self.num_pose_query = num_pose_query
        self.num_spatial_layer = num_spatial_layer
        self.spatial_layer_type = spatial_layer_type
        self.num_temporal_layer = num_temporal_layer
        self.temporal_init_method = temporal_init_method
        self.expansion_ratio = expansion_ratio
        self.temporal_supervision = temporal_supervision
        self.trope_scalar = trope_scalar
        self.num_latent_layer = num_latent_layer
        self.persp_embed_method = persp_embed_method
        self.persp_decorate = persp_decorate
        self.smplx_path = smplx_path
        self.image_size = image_size
        self.global_positioning = global_positioning
        self.training_phase = Poser.TrainingPhase.INFERENCE

        self.backbone = load_backbone(backbone, precision=precision)   # swin (v1) or swinv2, by config.json
        self.hidden_dim = self.backbone.config.hidden_size
        heads = self.backbone.config.num_heads
        self.num_heads = heads[-1] if isinstance(heads, list) else heads
        self.num_p = self.image_size // 32
        if num_latent_layer is not None:     # training-only consistency branch of the "ti" configurations (ref :255-265)
            from .latent_transformers import ScaleRotComplexEmbedTransformationGroup
            self.latent_trans = ScaleRotComplexEmbedTransformationGroup(
                num_layers=num_latent_layer, embed_dim=self.hidden_dim, num_heads=self.num_heads, num_p=self.num_p, num_q=self.num_p)
        else:
            self.latent_trans = None
        self._latent_override = None         # tests: (scale_coef [B], angle_rad [B]) instead of the random draw

        self.rmano_layer = _load_mano(smplx_path, mano_layer)
        self.rmano_layer.requires_grad_(False)
        self.rmano_layer.eval()

        reg_file = osp.join(osp.dirname(__file__), "sh_joint_regressor.npy")
        if osp.exists(reg_file):
            jreg = torch.from_numpy(np.load(reg_file)).float()
        else:
            # The real [21,778] regressor is a data file of the reference repository and is also stored in
            # every checkpoint (persistent buffer), which overrides this seeded stand-in on load.
            from ..utils.mano_standin import synthetic_joint_regressor
            jreg = synthetic_joint_regressor()
        self.register_buffer("J_regressor_mano", jreg, persistent=True)

        D = self.hidden_dim
        self.query_token = nn.Parameter(torch.randn(3, D) * (1 / D ** 0.5))
        self.perspective_mlp = PerspectiveEncoder(16 ** 2 if persp_embed_method == "dense" else 4, 2, D)
        self.spatial_encoder = SpatialEncoder(D, self.num_heads, num_spatial_layer, spatial_layer_type)

        def temporal():
            return TemporalEncoder(D, self.num_heads, num_temporal_layer, target=temporal_supervision,
                                   trope_scalar=trope_scalar, do_zero_init=(temporal_init_method == "zero"))

        self.pose_temporal_encoder = temporal()
        self.shape_temporal_encoder = temporal()
        self.root_temporal_encoder = temporal()
        self.pose_decoder = nn.Sequential(nn.Linear(D, num_pose_query * 6))
        self.shape_decoder = nn.Sequential(nn.Linear(D, 10))
        self.root_decoder = nn.Sequential(nn.Linear(D, 3))

        self.set_precision(precision)
        self.phase(Poser.TrainingPhase.INFERENCE)

    # ------------------------------------------------------------------------------------------ modes
    def set_precision(self, precision: str) -> None:
        """"bf16" / "fp16": that operand format in the backbone's tensor-core GEMMs + TF32 head (production).
        "fp32": exact fp32 everywhere (validation).  "fp8" (swinv2 backbones, inference only): the backbone's Q/K/V and fc1 GEMMs on
        E4M3 operands with per-token and per-channel scales, everything else as in "fp16"."""
        if precision == "fp8" and getattr(self.backbone.config, "model_type", None) != "swinv2":
            raise ValueError("precision='fp8' is built for the swinv2 backbone only: the Swin v1 stage 0-1 fused kernels have no fp8 form")
        set_precision(self, precision)
        self.backbone.precision = precision
        self.precision = precision

    def phase(self, phase) -> None:
        """Same train/eval and requires_grad toggles as ref:cs_vit/net/ti_poser.py:339-397."""
        self.training_phase = phase
        spatial = [self.backbone, self.perspective_mlp, self.spatial_encoder, self.pose_decoder, self.shape_decoder, self.root_decoder]
        temporal = [self.pose_temporal_encoder, self.shape_temporal_encoder, self.root_temporal_encoder]
        if phase == Poser.TrainingPhase.INFERENCE:
            self.eval()
            for p in self.parameters():
                p.requires_grad_(False)
            return
        train_set, frozen_set = (spatial, temporal) if phase == Poser.TrainingPhase.SPATIAL else (temporal, spatial)
        for m in train_set:
            m.train()
        for m in frozen_set:
            m.eval()
        self.query_token.requires_grad_(phase == Poser.TrainingPhase.SPATIAL)
        for p in chain(*(m.parameters() for m in train_set)):
            p.requires_grad_(True)
        for p in chain(*(m.parameters() for m in frozen_set)):
            p.requires_grad_(False)

    # ------------------------------------------------------------------------------------------ forward pieces
    def _linear_head(self, seq: nn.Sequential, x: torch.Tensor) -> torch.Tensor:
        lin = seq[0]
        if torch.is_grad_enabled() and (x.requires_grad or lin.weight.requires_grad):
            # the three output heads (96 / 10 / 3 columns) stay PyTorch in the training step (SURVEY.md §2.3 K18)
            return torch.nn.functional.linear(x, lin.weight, lin.bias)
        impl = ops.GEMM_SIMT if self.precision == "fp32" else ops.GEMM_TC
        y = ops.linear(_flat(x), lin.weight.detach().float(), lin.bias.detach().float(), impl=impl)
        return y.view(*x.shape[:-1], -1)

    def _frame_context(self, flat: torch.Tensor, persp_flat: torch.Tensor):
        """Per-frame inputs of the spatial encoder: ``flat`` ``[N,3,H,W]``, ``persp_flat`` ``[N, p]`` -> queries ``[N,3,D]``,
        patches ``[N,L,D]``.  Every op here works frame by frame (eval-mode BatchNorm is a row-wise affine map)."""
        N = flat.shape[0]
        patches = self.backbone.forward_features(flat, normalize=True)                 # [N, L, D] fp32
        persp_bias = self.perspective_mlp(persp_flat)                                   # [N, D]
        queries = self.query_token[None].expand(N, -1, -1)
        if self.persp_decorate == "query":
            queries = queries + persp_bias[:, None, :]
        else:
            patches = patches + persp_bias[:, None, :]
        return queries, patches

    def _frame_tokens(self, flat: torch.Tensor, persp_flat: torch.Tensor) -> torch.Tensor:
        """The per-frame part of the model: backbone, perspective bias and spatial encoder -> tokens ``[N,3,D]`` fp32."""
        queries, patches = self._frame_context(flat, persp_flat)
        return self.spatial_encoder(queries.contiguous(), patches)

    def _temporal_decode(self, tokens: torch.Tensor, timestamp: Optional[torch.Tensor], key_start: Optional[torch.Tensor] = None,
                         slot: Optional[int] = None):
        """The cross-frame part: tokens ``[B,T,3,D]`` -> pose_aa ``[B,T',16,3]``, shape ``[B,T',10]``, root ``[B,T',3]``.
        ``key_start`` (inference only): clip b uses its frames ``key_start[b]:T`` only.  ``slot`` (full model, inference only):
        decode frame ``slot`` of every clip alone (T' = 1); the output heads and the forward kinematics run on that frame only."""
        if self.training_phase in (Poser.TrainingPhase.INFERENCE, Poser.TrainingPhase.TEMPORAL):
            encoders = (self.pose_temporal_encoder, self.shape_temporal_encoder, self.root_temporal_encoder)
            streams = []
            for qi, enc in enumerate(encoders):
                x = tokens[:, :, qi].contiguous()
                if self.temporal_supervision == "realtime":
                    streams.append(x[:, -1:] + enc(x, timestamp, key_start=key_start))
                else:
                    y = x + enc(x, key_start=key_start)
                    streams.append(y if slot is None else y[:, slot:slot + 1])
            pose_tok, shape_tok, root_tok = streams
        else:
            pose_tok, shape_tok, root_tok = tokens[:, :, 0], tokens[:, :, 1], tokens[:, :, 2]
        pose_6d = self._linear_head(self.pose_decoder, pose_tok)
        pose_6d = pose_6d.reshape(*pose_6d.shape[:2], self.num_pose_query, 6)
        if torch.is_grad_enabled() and pose_6d.requires_grad:
            pose_aa = matrix_to_axis_angle(rotation_6d_to_matrix(pose_6d))        # differentiable torch form (training step)
        else:
            pose_aa = ops.rot6d_to_axis_angle(pose_6d)                             # one kernel (csrc/tail.cu)
        shape = self._linear_head(self.shape_decoder, shape_tok)
        root = self._linear_head(self.root_decoder, root_tok)
        return pose_aa, shape, root

    def _decode_pose(self, imgs: torch.Tensor, timestamp: torch.Tensor, persp_vec: torch.Tensor):
        """imgs ``[N,T,3,H,W]`` in [0,1] -> pose_aa ``[N,T',16,3]``, shape ``[N,T',10]``, root ``[N,T',3]``
        (ref:cs_vit/net/ti_poser.py:404-559; T' = 1 in realtime temporal mode, quirk Q7)."""
        B, T = imgs.shape[:2]
        flat = imgs.reshape(B * T, *imgs.shape[2:])
        queries, patches = self._frame_context(flat, persp_vec.reshape(B * T, -1))
        # Latent consistency branch (ref :442-457): a second copy of the patches, scaled / rotated in latent space, goes through
        # the same spatial encoder; the batch doubles (n = 2) and the copy's predictions are rotated back below.
        n = 1
        if self.latent_trans is not None:
            if self._latent_override is not None:
                scale_coef, angle_rad = (t.to(patches.device, patches.dtype) for t in self._latent_override)
            else:
                scale_coef = torch.randn(B, device=patches.device, dtype=patches.dtype).clamp(-0.3, 0.3) + 1.0
                angle_rad = torch.rand(B, device=patches.device, dtype=patches.dtype) * 2 * math.pi
            patches = torch.cat([patches, self.latent_trans.do_sr(patches, scale_coef, angle_rad)], dim=0)
            queries = torch.cat([queries, queries], dim=0)
            timestamp = torch.cat([timestamp, timestamp], dim=0)
            n = 2
        tokens = self.spatial_encoder(queries.contiguous(), patches)                    # [n BT, 3, D]
        pose_aa, shape, root = self._temporal_decode(tokens.reshape(n * B, T, 3, -1), timestamp)
        if self.latent_trans is not None:      # rotate the transformed copy's predictions back (ref :537-557)
            Tp = pose_aa.shape[1]
            sin, cos = torch.sin(-angle_rad), torch.cos(-angle_rad)
            zero, one = torch.zeros_like(sin), torch.ones_like(sin)
            rot_z = torch.stack([cos, -sin, zero, sin, cos, zero, zero, zero, one], dim=-1).view(B, 1, 3, 3).expand(B, Tp, 3, 3)
            pose_back = matrix_to_axis_angle(rot_z[:, :, None] @ axis_angle_to_matrix(pose_aa[B:]))
            pose_aa = torch.cat([pose_aa[:B], pose_back], dim=0)
            root_back = torch.einsum("btk,btkc->btc", root[B:], rot_z.transpose(-1, -2)) / scale_coef[:, None, None]
            root = torch.cat([root[:B], root_back], dim=0)
        return pose_aa, shape, root

    def _pose_fk(self, pose_aa: torch.Tensor, shape: torch.Tensor, root_transl_norm: torch.Tensor):
        """MANO forward kinematics, joint regression, de-normalisation to mm   (ref:cs_vit/net/ti_poser.py:561-607)."""
        B, T = pose_aa.shape[:2]
        flat_pose = pose_aa.reshape(B * T, -1)
        fused = self._mano_fused_operands()
        if fused is not None and not (torch.is_grad_enabled() and (pose_aa.requires_grad or shape.requires_grad or root_transl_norm.requires_grad)):
            # inference: skinning, joint regression, bone length and de-normalisation in ONE kernel (csrc/tail.cu) instead of ~120
            # elementwise / small-GEMM launches
            layer, mode = fused
            joint_cam, verts_cam, root_transl = ops.mano_fk(
                flat_pose.contiguous().float(), shape.reshape(B * T, -1).contiguous().float(), root_transl_norm.reshape(B * T, 3).contiguous().float(),
                layer, self._w_jreg(), TARGET_JOINTS_CONNECTION, rodrigues_mode=mode)
            return joint_cam.view(B, T, -1, 3), verts_cam.view(B, T, -1, 3), root_transl.view(B, T, 3)
        mano = self.rmano_layer(betas=shape.reshape(B * T, -1), global_orient=flat_pose[:, :3], hand_pose=flat_pose[:, 3:],
                                transl=torch.zeros(B * T, 3, device=pose_aa.device))
        verts = mano.vertices
        joints = torch.einsum("nvd,jv->njd", verts, self.J_regressor_mano)
        mean_len = 1e3 * mean_connection_length(joints, TARGET_JOINTS_CONNECTION).reshape(B, T, 1)
        root_transl = root_transl_norm * mean_len
        verts_cam = ((verts - joints[:, :1]) * 1e3).reshape(B, T, -1, 3) + root_transl[:, :, None]
        joint_cam = ((joints - joints[:, :1]) * 1e3).reshape(B, T, -1, 3) + root_transl[:, :, None]
        return joint_cam, verts_cam, root_transl

    def _w_jreg(self) -> torch.Tensor:
        j = self.J_regressor_mano
        return j if (j.dtype == torch.float32 and j.is_contiguous()) else j.float().contiguous()

    def _mano_fused_operands(self):
        """Buffers of the MANO layer for ``ops.mano_fk`` and its Rodrigues form, or None when the layer is not one this kernel
        restates.  The seeded stand-in is verified against its own torch forward on the GPU (tests/test_tail_gpu.py).  A real
        ``smplx`` MANO layer (use_pca=False) is standard LBS as well and is accepted only when ``self.fused_mano_smplx`` is set:
        its path (posedirs, hand-pose mean, smplx's Rodrigues epsilon) follows the published ``smplx.lbs`` but cannot be pinned
        here - smplx and the licensed MANO files are not in this image."""
        layer = self.rmano_layer
        from ..utils.mano_standin import SyntheticMANO
        if isinstance(layer, SyntheticMANO):
            mode, names = 0, {}
        elif getattr(self, "fused_mano_smplx", False) and all(hasattr(layer, a) for a in ("v_template", "shapedirs", "posedirs", "J_regressor", "lbs_weights", "parents")):
            mode, names = 1, {"posedirs": layer.posedirs}
            if not getattr(layer, "flat_hand_mean", True) and hasattr(layer, "hand_mean"):
                names["pose_mean"] = layer.hand_mean
        else:
            return None
        key = (id(layer), str(layer.v_template.device))
        if getattr(self, "_mano_pack_key", None) != key:
            f32 = lambda t: t.detach().float().contiguous()        # noqa: E731
            parents = [int(x) for x in (layer.parents.tolist() if torch.is_tensor(layer.parents) else layer.parents)]
            self._mano_pack = {"v_template": f32(layer.v_template), "shapedirs": f32(layer.shapedirs), "j_regressor": f32(layer.J_regressor),
                               "lbs_weights": f32(layer.lbs_weights), "parents": [-1] + parents[1:], **{k: f32(v) for k, v in names.items()}}
            self._mano_pack_key = key
        return self._mano_pack, mode

    def _sample_persp_dir_vec(self, num_sample: int, bbox: torch.Tensor, focal: torch.Tensor, princpt: torch.Tensor):
        """Unit-ray (x, y) components on a grid over the box, ``[B,T,p,p,2]``   (ref:cs_vit/net/ti_poser.py:609-639)."""
        g = torch.linspace(0.5 / num_sample, 1 - 0.5 / num_sample, num_sample, device=bbox.device)
        xs = bbox[..., 0:1] + (bbox[..., 2:3] - bbox[..., 0:1]) * g
        ys = bbox[..., 1:2] + (bbox[..., 3:4] - bbox[..., 1:2]) * g
        grid = torch.stack([xs[..., :, None].expand(-1, -1, -1, num_sample), ys[..., None, :].expand(-1, -1, num_sample, -1)], dim=-1)
        d = (grid - princpt[:, :, None, None, :]) / focal[:, :, None, None, :]
        d = torch.cat([d, torch.ones_like(d[..., :1])], dim=-1)
        return (d / torch.norm(d, dim=-1, keepdim=True))[..., :2]

    # ------------------------------------------------------------------------------------------ public API
    def predict_batch(self, img_tensor: torch.Tensor, square_bboxes: torch.Tensor, timestamp: torch.Tensor,
                      focal: torch.Tensor, princpt: torch.Tensor) -> Dict[str, torch.Tensor]:
        """Same contract as ref:cs_vit/net/ti_poser.py:641-722: ``img_tensor (B,T,3,S,S)`` in [0,1],
        ``square_bboxes (B,T,4)`` xyxy, ``timestamp (B,T)`` ms, ``focal/princpt (B,T,2)``."""
        if not img_tensor.is_cuda:
            raise RuntimeError("Poser.predict_batch runs on CUDA tensors only (there is no CPU fallback)")
        self._check_positioning()
        directions = self._persp_directions(square_bboxes, focal, princpt)
        pose_aa, shape, root_transl_norm = self._decode_pose(img_tensor, timestamp, directions)
        joint_cam, verts_cam, root_transl = self._pose_fk(pose_aa, shape, root_transl_norm)
        return {"joint_cam": joint_cam, "verts_cam": verts_cam, "pose_aa": pose_aa, "shape": shape,
                "root_transl_norm": root_transl_norm, "root_transl": root_transl}

    def _check_positioning(self) -> None:
        if self.global_positioning == "orientation":
            # Upstream this mode passes the [B,T,3] axis-angle (not the rotated matrix) to
            # matrix_to_axis_angle (ref:cs_vit/net/ti_poser.py:709), which raises on shape for T != 3.
            raise NotImplementedError("global_positioning='orientation' is broken in the reference (ti_poser.py:709)")

    def _persp_directions(self, square_bboxes: torch.Tensor, focal: torch.Tensor, princpt: torch.Tensor) -> torch.Tensor:
        """Perspective-encoder input per frame: ``[B,T,16,16,2]`` ("dense") or ``[B,T,2,2,2]`` ("sparse") from ``(B,T,·)`` boxes
        and intrinsics."""
        if self.persp_embed_method == "dense":
            directions = self._sample_persp_dir_vec(16, square_bboxes, focal, princpt)
        else:
            u0 = (square_bboxes[..., 0] - princpt[..., 0]) / focal[..., 0]
            u1 = (square_bboxes[..., 2] - princpt[..., 0]) / focal[..., 0]
            v0 = (square_bboxes[..., 1] - princpt[..., 1]) / focal[..., 1]
            v1 = (square_bboxes[..., 3] - princpt[..., 1]) / focal[..., 1]
            top = torch.stack([torch.stack([u0, v0], -1), torch.stack([u1, v0], -1)], dim=2)
            bot = torch.stack([torch.stack([u0, v1], -1), torch.stack([u1, v1], -1)], dim=2)
            directions = torch.stack([top, bot], dim=2)      # [B,T,2,2,2]
        return directions

    def _criterion(self, predict, batch, host_logs: bool = True):
        """ref:cs_vit/net/ti_poser.py:724-778.  ``host_logs=False`` returns the five components as one device tensor instead of
        Python floats: no device->host sync, so the step can be captured in a CUDA graph (``cs_vit.train.GraphedFinetuneStep``)."""
        T = predict["joint_cam"].shape[1]
        # slices, not index lists: an index list becomes a host tensor + H2D copy, which cannot be captured in a CUDA graph
        idx = slice(None) if self.temporal_supervision != "realtime" else slice(-1, None)   # last frame of prediction AND labels
        pj, gj, valid = predict["joint_cam"][:, idx], batch["joint_cam"][:, idx], batch["joint_valid"][:, idx]
        loss_cam = torch.mean((pj - gj).norm(dim=-1) * valid)
        loss_rel = torch.mean(((pj - pj[:, :, :1]) - (gj - gj[:, :, :1])).norm(dim=-1) * valid)
        loss_shape = (predict["shape"][:, idx] - batch["mano_shape"][:, idx]).abs().mean()
        zero = torch.zeros_like(loss_shape)
        loss_vel, loss_accel, loss_temporal = zero, zero, zero
        if self.training_phase == Poser.TrainingPhase.TEMPORAL and self.temporal_supervision == "full":
            vp, vg = derivative(predict["joint_cam"], 1), derivative(batch["joint_cam"], 1)
            ap, ag = derivative(vp, 1), derivative(vg, 1)
            loss_vel = (vp - vg).norm(dim=-1).mean()
            loss_accel = (ap - ag).norm(dim=-1).mean()
            loss_temporal = 1e-2 * (loss_vel + loss_accel)
        # one device->host transfer for all five scalars instead of five .item() syncs
        parts = torch.stack([loss_cam, loss_rel, loss_shape, loss_vel, loss_accel])
        if not host_logs:
            return loss_cam + loss_rel + loss_shape + loss_temporal, parts.detach()
        logs = dict(zip(("cam", "rel", "shape", "loss_vel", "loss_accel"), parts.tolist()))
        return loss_cam + loss_rel + loss_shape + loss_temporal, logs

    def loss_tensors(self, batch):
        """``predict_batch`` + ``_criterion`` without any host synchronisation: ``(loss, parts[5], predict)``, all on the device."""
        predict = self.predict_batch(img_tensor=batch["patches"], square_bboxes=batch["square_bboxes"],
                                     timestamp=batch["timestamp"], focal=batch["focal"], princpt=batch["princpt"])
        if self.latent_trans is None:
            loss, parts = self._criterion(predict, batch, host_logs=False)
            return loss, parts, predict
        b = batch["patches"].shape[0]
        loss_o, parts = self._criterion({k: v[:b] for k, v in predict.items()}, batch, host_logs=False)
        loss_t, _ = self._criterion({k: v[b:] for k, v in predict.items()}, batch, host_logs=False)
        return loss_o + 1e-2 * loss_t, parts, predict

    def _vis(self, predict, batch):
        """Reprojection overlay for TensorBoard (ref:cs_vit/net/ti_poser.py:780-813).  Host-side cv2 drawing is
        outside the hot path (SURVEY.md §2.1 'Image utils'); returns None when the frames are not on disk."""
        try:
            from ..utils.img import reprojection_overlay
            return reprojection_overlay(predict, batch, TARGET_JOINTS_CONNECTION)
        except Exception:  # missing files / cv2: visualisation must never break a training step
            return None

    def forward(self, batch):
        """Training-step forward with the reference's return structure (ref:cs_vit/net/ti_poser.py:815-855)."""
        batch_size = batch["patches"].shape[0]
        predict = self.predict_batch(img_tensor=batch["patches"], square_bboxes=batch["square_bboxes"],
                                     timestamp=batch["timestamp"], focal=batch["focal"], princpt=batch["princpt"])
        predict_origin = {k: v[:batch_size].clone() for k, v in predict.items()}
        loss_origin, origin_dict = self._criterion(predict_origin, batch)
        loss, trans_val, trans_dict = loss_origin, 0.0, {}
        if self.latent_trans is not None:     # consistency loss on the latent-transformed copy (ref :835-837)
            predict_trans = {k: v[batch_size:].clone() for k, v in predict.items()}
            loss_trans, trans_dict = self._criterion(predict_trans, batch)
            loss = loss_origin + 1e-2 * loss_trans
            trans_val = loss_trans.item()
        return {
            "loss": loss,
            "logs": {
                "scalar": {"total": loss.item(), "origin": {"origin": loss_origin.item(), **origin_dict},
                           "trans": {"trans": trans_val, **trans_dict}},
                "image": {"img_reproj": self._vis(predict_origin, batch)},
            },
        }
