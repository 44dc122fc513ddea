"""Tests of the SwinV2 per-block training path (CSVIT_V2_TRAIN_BLOCK=fused, cs_vit.autograd.Swinv2BlockFn) and its two kernels:
csvit_swinv2_qkv_train (the Q/K/V GEMM with the cosine normalisation's row scales as a second output) and csvit_swinv2_cosnorm_bwd (the
normalisation's backward), the block path against the op-level path with both tcgen05 cores (each measured against the fp32 mode of the
same weights), HF's gradient golden, stochastic depth with recorded draws, the graphed finetune step, and the switch."""
import json
import math
import os

import pytest
import torch

from test_swinv2_attn_bwd_gpu import LOG2E, _golden_errors
from test_swinv2_gpu import _backbone, rel, v2_case

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from cs_vit import ops as o
    return o


# ---------------------------------------------------------------------------------------------------- kernels


@gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("rows,C", [(4100, 128), (1000, 256), (33000, 256), (777, 512), (300, 1024)])
def test_qkv_train_matches_inference_gemm(ops, rows, C, dtype):
    """The 16-bit output is swinv2_qkv's bit for bit (rows not a multiple of the 128-row tile; 33000 x 768 takes the CTA-pair kernel), and
    rnorm is 1 / |x| of every q and k head of x = a @ w.T + b, evaluated in fp64 from the same 16-bit operands, within 1e-4 relative."""
    g = torch.Generator(device="cuda").manual_seed(rows + C)
    heads = C // 32
    a = torch.randn(rows, C, device="cuda", generator=g).to(dtype)
    w = (torch.randn(3 * C, C, device="cuda", generator=g) / math.sqrt(C)).to(dtype)
    b = 0.5 * torch.randn(3 * C, device="cuda", generator=g)
    qs = LOG2E * (1.0 + 9.0 * torch.rand(heads, device="cuda", generator=g))
    want = ops.swinv2_qkv(a, w, b, qs)
    got, rnorm = ops.swinv2_qkv_train(a, w, b, qs)
    assert torch.equal(got, want)
    x = (a.double() @ w.double().t() + b.double())[:, :2 * C].reshape(rows, 2 * heads, 32)
    ref = 1.0 / x.norm(dim=-1).clamp_min(1e-12)
    assert rnorm.shape == (rows, 2 * heads)
    assert ((rnorm.double() - ref).abs() / ref).max().item() <= 1e-4


def _cosnorm_case(rows, heads, dtype, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    C = 32 * heads
    xq = torch.randn(rows, heads, 32, device="cuda", generator=g) * (0.2 + 3 * torch.rand(rows, heads, 1, device="cuda", generator=g))
    xk = torch.randn(rows, heads, 32, device="cuda", generator=g) * (0.2 + 3 * torch.rand(rows, heads, 1, device="cuda", generator=g))
    s = LOG2E * (math.log(10.0) + 0.8 * torch.randn(heads, device="cuda", generator=g)).clamp(max=math.log(100.0)).exp()
    nq, nk = xq.norm(dim=-1).clamp_min(1e-12), xk.norm(dim=-1).clamp_min(1e-12)
    q2 = (xq / nq[..., None] * s.view(1, heads, 1)).reshape(rows, C).to(dtype)
    kh = (xk / nk[..., None]).reshape(rows, C).to(dtype)
    v = torch.randn(rows, C, device="cuda", generator=g).to(dtype)
    qkv = torch.cat([q2, kh, v], 1).contiguous()
    rnorm = torch.cat([1.0 / nq, 1.0 / nk], 1).contiguous()
    dq2, dk, dv = (torch.randn(rows, C, device="cuda", generator=g).to(dtype) for _ in range(3))
    return xq, xk, s, qkv, rnorm, dq2, dk, dv


@gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("rows,heads", [(8192, 4), (3001, 3), (2048, 8), (999, 16), (512, 32)])
def test_cosnorm_bwd_matches_fp32_autograd(ops, rows, heads, dtype):
    """Against fp32 autograd of normalize(x) * s on the unrounded x: dq / dk within 2x the error of that reference rounded to the same 16-bit
    format, dv copied exactly, and dqscale within 1e-4 of its definition (sum of q_hat . dq2, q_hat = q2 / s) in fp64 on the stored
    operands and within 1.5x the error that definition makes against the autograd gradient of s."""
    xq, xk, s, qkv, rnorm, dq2, dk, dv = _cosnorm_case(rows, heads, dtype, rows + heads)
    C = 32 * heads
    dqkv, dqs = ops.swinv2_cosnorm_bwd(qkv, rnorm, s.contiguous(), dq2, dk, dv)
    xq_, xk_, s_ = xq.clone().requires_grad_(True), xk.clone().requires_grad_(True), s.clone().requires_grad_(True)
    yq = torch.nn.functional.normalize(xq_, dim=-1) * s_.view(1, heads, 1)
    yk = torch.nn.functional.normalize(xk_, dim=-1)
    torch.autograd.backward([yq, yk], [dq2.float().view(rows, heads, 32), dk.float().view(rows, heads, 32)])
    ref_q, ref_k = xq_.grad.reshape(rows, C), xk_.grad.reshape(rows, C)
    for got, ref in ((dqkv[:, :C], ref_q), (dqkv[:, C:2 * C], ref_k)):
        e, e16 = rel(got, ref), rel(ref.to(dtype), ref)
        assert e <= 2 * e16, (e, e16)
    assert torch.equal(dqkv[:, 2 * C:], dv)
    qhat = qkv[:, :C].double().view(rows, heads, 32) / s.double().view(1, heads, 1)
    want = (qhat * dq2.double().view(rows, heads, 32)).sum(dim=(0, 2))
    assert ((dqs.double() - want).abs() / want.abs().clamp_min(1e-30)).max().item() <= 1e-4
    assert rel(dqs, s_.grad) <= 1.5 * rel(want, s_.grad.double()) + 1e-6


@gpu
def test_cosnorm_bwd_accumulates_and_rejects_bad_operands(ops):
    xq, xk, s, qkv, rnorm, dq2, dk, dv = _cosnorm_case(640, 4, torch.float16, 3)
    _, once = ops.swinv2_cosnorm_bwd(qkv, rnorm, s.contiguous(), dq2, dk, dv)
    acc = once.clone()
    ops.swinv2_cosnorm_bwd(qkv, rnorm, s.contiguous(), dq2, dk, dv, dqscale=acc)
    assert torch.allclose(acc, 2 * once, rtol=1e-5, atol=0)
    with pytest.raises(ValueError):
        ops.swinv2_cosnorm_bwd(qkv, rnorm[:, :4].contiguous(), s.contiguous(), dq2, dk, dv)
    with pytest.raises(ValueError):
        ops.swinv2_cosnorm_bwd(qkv, rnorm, s.contiguous(), dq2, dk.to(torch.bfloat16), dv)


# ---------------------------------------------------------------------------------------------------- backbone


def _grads(tmp, precision, window, block, px, drop_rand=None):
    """Features and gradients of a random swinv2_xs at 256^2 (window 16: stages 0-2 on 16 x 16 windows, stage 3 on 8 x 8; window 8: every
    stage on 8 x 8), with both tcgen05 training cores on (CSVIT_V2_TRAIN_ATTN=CSVIT_V2_TRAIN_ATTN8=tcgen05) and the block path on or off."""
    from cs_vit.net.swinv2_b200 import load_backbone
    from cs_vit.synthetic import make_random_backbone_dir
    d = make_random_backbone_dir(os.path.join(tmp, f"v2xs_w{window}"), "swinv2_xs", seed=0, image_size=256, window_size=window)
    model = load_backbone(d, precision=precision).cuda()
    model._v2_train_tc = model._v2_train_tc8 = True
    model._v2_train_block = block
    model.train()
    if drop_rand is None:
        model.config.drop_path_rate = 0.0
    else:
        model.config.drop_path_rate = 0.1
        model._drop_path_rand = [u.clone() for u in drop_rand]
    for p_ in model.parameters():
        p_.requires_grad_(True)
    feats = model.forward_features(px, normalize=False)
    if drop_rand is not None:
        assert not model._drop_path_rand          # every recorded draw was consumed
    R = torch.randn(feats.shape, generator=torch.Generator().manual_seed(5)).cuda()
    (feats * R).sum().backward()
    torch.cuda.synchronize()
    return feats.detach(), {n: p.grad.detach().double() for n, p in model.named_parameters()}


def _compare(tmp, precision, window, drop_rand=None):
    px = torch.randn(2, 3, 256, 256, generator=torch.Generator().manual_seed(12)).cuda()
    f32, g32 = _grads(tmp, "fp32", window, False, px, drop_rand)
    f_op, g_op = _grads(tmp, precision, window, False, px, drop_rand)
    f_bl, g_bl = _grads(tmp, precision, window, True, px, drop_rand)

    def total(g):
        return math.sqrt(sum(float((g[n] - g32[n]).norm()) ** 2 for n in g32) / sum(float(g32[n].norm()) ** 2 for n in g32))
    e_op, e_bl = total(g_op), total(g_bl)
    print(f"w{window} {precision}{' drop-path' if drop_rand else ''}: features block {rel(f_bl, f32):.3e} op-level {rel(f_op, f32):.3e}; "
          f"gradients block {e_bl:.3e} op-level {e_op:.3e}")
    assert rel(f_bl, f32) <= 1.5 * rel(f_op, f32) + 1e-4
    assert e_bl <= 1.5 * e_op, (e_bl, e_op)


@gpu
@pytest.mark.parametrize("window", [16, 8])
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_block_path_against_op_level_path(precision, window, tmp_path):
    """Shifted and unshifted blocks of both window sizes: the block path's features and global gradient error against the fp32 mode are
    within 1.5x of the op-level path's (both tcgen05 cores on)."""
    _compare(str(tmp_path), precision, window)


@gpu
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_block_path_stochastic_depth(precision, tmp_path):
    """drop_path_rate 0.1 with recorded draws (some samples dropped on either branch): the block path consumes the draws in the op-level
    path's order and stays within the bounds of test_block_path_against_op_level_path."""
    g = torch.Generator().manual_seed(7)
    draws = []
    for i in range(2 * 7):                        # swinv2_xs: 8 blocks of two branches; block 0 has rate 0 and draws nothing
        u = torch.rand(2, generator=g) * 0.8 + 0.2
        if i % 3 == 1:
            u[i % 2] = 0.0                        # floor(keep + 0) = 0: that sample's branch is dropped
        draws.append(u)
    _compare(str(tmp_path), precision, 16, drop_rand=draws)


def _golden_grads(precision, tmp_path, block):
    from test_swinv2_oracle import V2_GRAD_CASES
    sd, px, gold, case = v2_case(sorted(V2_GRAD_CASES)[0])
    model = _backbone(case, precision, str(tmp_path))
    model.config.drop_path_rate = 0.0
    model._v2_train_tc = model._v2_train_tc8 = True
    model._v2_train_block = block
    model.train()
    for p_ in model.parameters():
        p_.requires_grad_(True)
    feats = model.forward_features(px.cuda(), normalize=False)
    R = torch.randn(feats.shape, generator=torch.Generator().manual_seed(case["projection_seed"])).cuda()
    (feats * R).sum().backward()
    torch.cuda.synchronize()
    return feats.detach(), {n: p.grad for n, p in model.named_parameters()}, gold


@gpu
def test_w16_golden_with_block_path(tmp_path):
    """The gradient golden train_swinv2_xs_w16_linear with the block path (fp16): features at the existing 3e-3 bar, and the error over all
    parameters at most 1.5x that of the op-level path with both tcgen05 cores.  Prints the last stage's query.bias errors of both paths."""
    feats, g_bl, gold = _golden_grads("fp16", tmp_path, True)
    _, g_op, _ = _golden_grads("fp16", tmp_path, False)
    assert rel(feats.cpu(), torch.from_numpy(gold["features"])) < 3e-3
    for n, g in g_bl.items():
        assert g is not None and torch.isfinite(g).all(), n
    e_bl, per_bl = _golden_errors(g_bl, gold)
    e_op, per_op = _golden_errors(g_op, gold)
    qb = [n for n in per_bl if n.startswith("encoder.layers.3.") and n.endswith("query.bias")]
    print(f"fp16: total error block {e_bl:.3e} op-level {e_op:.3e}; last-stage query.bias "
          + ", ".join(f"{n}: block {per_bl[n]:.3e} op-level {per_op[n]:.3e}" for n in qb))
    assert e_bl <= 1.5 * e_op, (e_bl, e_op)


@gpu
def test_graphed_finetune_step_with_block_path(tmp_path):
    """The finetune step on a swinv2_xs Poser (fp16, window 16, block path on) captured as one CUDA graph: it replays, the loss is finite and
    falls, and equals the eager step's loss trajectory within 1e-3 relative (the bar of the window-8 graphed-step test)."""
    from cs_vit.net import Poser
    from cs_vit.synthetic import make_inputs, make_random_backbone_dir, randomize_head_
    from cs_vit.train import GradReducer, GraphedFinetuneStep, finetune_step
    from cs_vit.utils.mano_standin import SyntheticMANO
    d = make_random_backbone_dir(str(tmp_path / "v2xs"), "swinv2_xs", seed=0, image_size=256, window_size=16)
    with open(os.path.join(d, "config.json")) as f:
        cfg = json.load(f)
    cfg["drop_path_rate"] = 0.0
    with open(os.path.join(d, "config.json"), "w") as f:
        json.dump(cfg, f)
    traj = {}
    for mode in ("eager", "graph"):
        torch.manual_seed(0)
        model = Poser(d, image_size=256, mano_layer=SyntheticMANO(), spatial_layer_type="encoder", persp_decorate="patch", precision="fp16")
        randomize_head_(model, seed=1)
        model.phase(Poser.TrainingPhase.SPATIAL)
        model = model.cuda()
        model.backbone._v2_train_block = True          # CSVIT_V2_TRAIN_BLOCK=fused
        batch = {k: v.cuda() for k, v in make_inputs(4, 1, 256, seed=3, labels=True).items()}
        params = [p for p in model.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=2e-5, fused=True, capturable=(mode == "graph"))
        reducer = GradReducer(params)
        if mode == "eager":
            traj[mode] = [finetune_step(model, batch, opt, reducer).item() for _ in range(6)]
        else:
            step = GraphedFinetuneStep(model, batch, opt, reducer, warmup=3)
            traj[mode] = [step(batch).item() for _ in range(3)]
    assert all(math.isfinite(v) for v in traj["graph"]) and traj["graph"][-1] < traj["eager"][0], traj
    for a, b in zip(traj["graph"], traj["eager"][3:]):
        assert abs(a - b) <= 1e-3 * abs(b), traj


# ---------------------------------------------------------------------------------------------------- the switch


def _tiny_config(window):
    from cs_vit.net.swinv2_b200 import Swinv2ConfigLite
    return Swinv2ConfigLite.from_dict({"model_type": "swinv2", "embed_dim": 32, "depths": [2, 2], "num_heads": [1, 2], "window_size": window,
                                       "image_size": 64})


def test_block_switch_read_at_construction(monkeypatch):
    """CSVIT_V2_TRAIN_BLOCK is read when the backbone is built, is off by default, and leaves the attention switches alone."""
    from cs_vit.net.swinv2_b200 import Swinv2BackboneB200
    monkeypatch.delenv("CSVIT_V2_TRAIN_BLOCK", raising=False)
    m = Swinv2BackboneB200(_tiny_config(8))
    assert not m._v2_train_block
    monkeypatch.setenv("CSVIT_V2_TRAIN_BLOCK", "fused")
    m2 = Swinv2BackboneB200(_tiny_config(8))
    monkeypatch.delenv("CSVIT_V2_TRAIN_BLOCK")
    assert m2._v2_train_block and not m2._v2_train_tc and not m2._v2_train_tc8 and not m._v2_train_block


@gpu
@pytest.mark.parametrize("precision,window,blocks", [("fp16", 8, 4), ("bf16", 8, 4), ("fp32", 8, 0), ("fp16", 4, 0)])
def test_block_switch_selects_blocks(monkeypatch, precision, window, blocks):
    """With the switch on, 16-bit blocks with 8 x 8 windows run as Swinv2BlockFn; the fp32 mode and windows without a tcgen05 core (4 x 4)
    take the op-level path."""
    from cs_vit import autograd as ag
    from cs_vit.net.swinv2_b200 import Swinv2BackboneB200
    monkeypatch.setenv("CSVIT_V2_TRAIN_BLOCK", "fused")
    calls = []
    real = ag.swinv2_block
    monkeypatch.setattr(ag, "swinv2_block", lambda *a, **k: calls.append(1) or real(*a, **k))
    torch.manual_seed(0)
    m = Swinv2BackboneB200(_tiny_config(window), precision=precision).cuda()
    m.config.drop_path_rate = 0.0
    m.train()
    feats = m.forward_features(torch.randn(2, 3, 64, 64).cuda(), normalize=False)
    feats.square().sum().backward()
    torch.cuda.synchronize()
    assert len(calls) == blocks
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.parameters())
