"""GPU tests of the differentiable SwinV2 cosine-attention core on tcgen05 (csvit_swinv2_attn_tc_train / csvit_swinv2_attn_tc_bwd,
cs_vit.autograd.swinv2_cosine_attention): the kernels against fp32 autograd of the natural-domain formula (bounded by the error torch
SDPA - the other training core - makes on the same rounded inputs), reproducibility and contracts, the backbone's gradients against
HF's golden and against the SDPA core, and the graphed finetune step on a SwinV2 backbone."""
import json
import math
import os

import numpy as np
import pytest
import torch

from test_swinv2_gpu import _backbone, rel

pytestmark = pytest.mark.gpu

LOG2E = 1.4426950408889634
LN2 = math.log(2.0)
# absolute ceilings on the relative error norm against fp32, whatever SDPA achieves (on a B200 the fp16 kernel errors of the cases below
# are 3-5e-4, SDPA's 1.5-1.8e-3)
CEIL = {torch.float16: 5e-3, torch.bfloat16: 3e-2}


@pytest.fixture(scope="module")
def ops():
    from cs_vit import ops as o
    return o


def _rel_index48(device):
    """[256 * 256] index of (dy + 15) * 48 + dx + 15 for query i, key j of a 16 x 16 window (the padded bias-table layout)."""
    i = torch.arange(256, device=device)
    dy = (i[:, None] >> 4) - (i[None, :] >> 4)
    dx = (i[:, None] & 15) - (i[None, :] & 15)
    return ((dy + 15) * 48 + dx + 15).reshape(-1)


def _inputs(B, H, heads, dtype, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    C, rows = 32 * heads, B * H * H
    scale = (math.log(10.0) + 0.8 * torch.randn(heads, device="cuda", generator=g)).clamp(max=math.log(100.0)).exp()
    qh = torch.nn.functional.normalize(torch.randn(rows, heads, 32, device="cuda", generator=g), dim=-1)
    kh = torch.nn.functional.normalize(torch.randn(rows, heads, 32, device="cuda", generator=g), dim=-1)
    q2 = (qh * (scale * LOG2E).view(1, heads, 1)).reshape(rows, C).to(dtype)
    k = kh.reshape(rows, C).to(dtype)
    v = torch.randn(rows, C, device="cuda", generator=g).to(dtype)
    tab = 16 * torch.sigmoid(2 * torch.randn(heads, 961, device="cuda", generator=g))          # like 16 sigmoid(cpb_mlp), in (0, 16)
    from cs_vit import ops
    bl2 = ops.swinv2_bias_log2(tab)
    dout = torch.randn(rows, C, device="cuda", generator=g).to(dtype)
    return q2, k, v, bl2, dout


def _reference(q2, k, v, bl2, dout, B, H, heads, shift, mask_repeat):
    """fp32 autograd of softmax(q_hat k_hat^T s + 16 sigmoid(cpb) + mask_repeat * mask) v, written in the natural domain on the
    log2-domain inputs (q2 ln 2 = q_hat s, bias_log2 ln 2 = 16 sigmoid(cpb))."""
    from cs_vit import ops
    L, C = 256, 32 * heads
    nW = (H // 16) ** 2
    qf, kf, vf = (t.float().view(B * nW, L, heads, 32).transpose(1, 2).requires_grad_(True) for t in (q2, k, v))
    bf = bl2.clone().requires_grad_(True)
    s = LN2 * (qf @ kf.transpose(-1, -2) + bf.view(heads, -1)[:, _rel_index48(q2.device)].view(1, heads, L, L))
    if shift:
        m = ops.shift_mask(H, H, 16, shift)
        s = (s.view(B, nW, heads, L, L) + mask_repeat * m[None, :, None]).view(B * nW, heads, L, L)
    p = s.softmax(-1)
    lse2 = torch.logsumexp(s, -1) / LN2
    o = p @ vf
    o.backward(dout.float().view(B * nW, L, heads, 32).transpose(1, 2))
    back = lambda t: t.transpose(1, 2).reshape(B * H * H, C)      # noqa: E731
    return back(o.detach()), lse2.detach(), back(qf.grad), back(kf.grad), back(vf.grad), bf.grad


def _sdpa(q2, k, v, bl2, dout, B, H, heads, shift, mask_repeat):
    """The SDPA core of the training path on the same 16-bit inputs: (ctx, dq2, dk, dv, dbias_log2)."""
    from cs_vit import ops
    from torch.nn.attention import SDPBackend, sdpa_kernel
    L, C, dt = 256, 32 * heads, q2.dtype
    nW = (H // 16) ** 2
    qf, kf, vf = (t.detach().view(B * nW, L, heads, 32).transpose(1, 2).requires_grad_(True) for t in (q2, k, v))
    bf = bl2.clone().requires_grad_(True)
    add = LN2 * bf.view(heads, -1)[:, _rel_index48(q2.device)].view(1, heads, L, L)
    if shift:
        add = (add + mask_repeat * ops.shift_mask(H, H, 16, shift)[:, None]).reshape(1, nW * heads, L, L)
        q4, k4, v4 = (t.reshape(B, nW * heads, L, 32) for t in (qf, kf, vf))
    else:
        q4, k4, v4 = qf, kf, vf
    with sdpa_kernel([SDPBackend.EFFICIENT_ATTENTION]):
        o = torch.nn.functional.scaled_dot_product_attention(q4, k4, v4, attn_mask=add.to(dt).contiguous(), scale=LN2)
    o = o.reshape(B * nW, heads, L, 32)
    o.backward(dout.view(B * nW, L, heads, 32).transpose(1, 2))
    back = lambda t: t.transpose(1, 2).reshape(B * H * H, C)      # noqa: E731
    return back(o.detach()), back(qf.grad), back(kf.grad), back(vf.grad), bf.grad


def _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift, mask_repeat=2, out=None):
    qkv = torch.cat([q2, k, v], 1)
    ctx, lse2 = ops.swinv2_attn_tc_train(qkv, bl2, B, H, H, heads, shift, mask_repeat)
    grads = ops.swinv2_attn_tc_bwd(qkv, ctx, lse2, dout, bl2, B, H, H, heads, shift, mask_repeat, out=out)
    return (ctx, lse2) + tuple(grads)


CASES = [(32, 4, 0, 2), (32, 4, 8, 2), (64, 1, 8, 1), (16, 16, 0, 3), (16, 3, 0, 2), (48, 2, 8, 1), (32, 8, 8, 5), (32, 8, 8, 13),
         (64, 4, 0, 8), (64, 4, 8, 8), (32, 8, 0, 8), (32, 8, 8, 8), (16, 16, 0, 8)]      # + the SwinV2-B stage 0-2 shapes at batch 8


@pytest.mark.parametrize("H,heads,shift,B", CASES)
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_kernels_match_fp32_autograd(ops, H, heads, shift, B, dtype):
    q2, k, v, bl2, dout = _inputs(B, H, heads, dtype, seed=11 * H + heads + shift + B)
    ref = _reference(q2, k, v, bl2, dout, B, H, heads, shift, 2)
    got = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift)
    sd = _sdpa(q2, k, v, bl2, dout, B, H, heads, shift, 2)
    names = ("ctx", "dq2", "dk", "dv", "dbias")
    errs = {n: rel(g, r) for n, g, r in zip(names, (got[0],) + got[2:], (ref[0],) + ref[2:])}
    sdpa = {n: rel(s, r) for n, s, r in zip(names, sd, (ref[0],) + ref[2:])}
    for n in names:
        assert errs[n] <= 1.5 * sdpa[n] and errs[n] < CEIL[dtype], (n, errs, sdpa)
    assert (got[1] - ref[1].view_as(got[1])).abs().max().item() < 2e-2       # lse2 (log2 units): the rounded-probability sums
    assert torch.equal(got[5][:, :, 31:], torch.zeros_like(got[5][:, :, 31:]))


@pytest.mark.parametrize("heads,shift", [(3, 8), (1, 0)])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_backward_reproducible_and_contracts(ops, heads, shift, dtype):
    B, H = 3, 32
    rows, C = B * H * H, 32 * heads
    q2, k, v, bl2, dout = _inputs(B, H, heads, dtype, seed=5 + heads)
    a = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift)
    b = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift)
    for x, y in zip(a[:5], b[:5]):
        assert torch.equal(x, y)                                               # ctx, lse2, dq, dk, dv: bit-identical
    assert (a[5] - b[5]).abs().max().item() <= 1e-6 * max(1.0, a[5].abs().max().item())
    # guard-banded outputs: nothing written outside [rows, C]
    guard = 4096
    bufs = [torch.full((rows * C + 2 * guard,), 7.0, dtype=dtype, device="cuda") for _ in range(3)]
    views = tuple(t[guard:guard + rows * C].view(rows, C) for t in bufs)
    c = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift, out=views)
    for t, x, y in zip(bufs, c[2:5], a[2:5]):
        assert torch.equal(x, y)
        assert (t[:guard] == 7).all() and (t[-guard:] == 7).all()
    if shift:
        z = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift, mask_repeat=0)
        ref0 = _reference(q2, k, v, bl2, dout, B, H, heads, shift, 0)
        assert rel(z[2], ref0[2]) < CEIL[dtype] and rel(a[2], ref0[2]) > CEIL[dtype]
        assert rel(z[5], a[5]) > 1e-2


def _golden_grads(precision, tmp_path, train_attn):
    from test_swinv2_oracle import V2_GRAD_CASES, v2_case
    name = sorted(V2_GRAD_CASES)[0]
    sd, px, gold, case = v2_case(name)
    model = _backbone(case, precision, str(tmp_path))
    model.config.drop_path_rate = 0.0
    model._v2_train_tc = train_attn == "tcgen05"          # what CSVIT_V2_TRAIN_ATTN selects
    model.train()
    for p_ in model.parameters():
        p_.requires_grad_(True)
    feats = model.forward_features(px.cuda(), normalize=False)
    R = torch.randn(feats.shape, generator=torch.Generator().manual_seed(case["projection_seed"])).cuda()
    (feats * R).sum().backward()
    torch.cuda.synchronize()
    return feats.detach(), {n: p.grad for n, p in model.named_parameters()}, gold


def _golden_errors(grads, gold):
    """(relative error norm over every golden gradient, {name: relative error} of the parameters above 1e-4 of the gradient norm)."""
    names = [str(n) for n in gold["param_names"]]
    gnorm = float(np.sqrt((gold["grad_norm"] ** 2).sum()))
    num = den = 0.0
    per = {}
    for i, n in enumerate(names):
        if "grad/" + n in gold:
            ref = torch.from_numpy(gold["grad/" + n]).double()
            num += float((grads[n].cpu().double() - ref).norm()) ** 2
            den += float(ref.norm()) ** 2
            if gold["grad_norm"][i] > 1e-4 * gnorm:
                per[n] = rel(grads[n].cpu(), ref)
    return math.sqrt(num / den), per


@pytest.mark.parametrize("precision,tol", [("fp16", 3e-3), ("bf16", 3e-2)])
def test_backbone_gradients_with_tcgen05_core_match_hf_golden(precision, tol, tmp_path):
    """The gradient golden of the existing fp16 test (train_swinv2_xs_w16_linear) forced through the tcgen05 core, at the same bars: features,
    every gradient norm and projection, and the worst per-parameter error of the stages that run the core (16 x 16 windows, stages 0-2).
    The last stage (8 x 8 windows) keeps SDPA; its smallest gradients (e.g. query.bias, 2e-4 of the gradient norm) are sums that cancel
    to a few parts in a thousand and move by a factor two with the forward's last-bit differences upstream, so they are held to the
    norm / projection bars only.  bf16: tol 3e-2 (8-bit mantissa; measured on a B200: features 6e-3, worst stage 0-2 parameter 0.18)."""
    from oracle.make_train_goldens import projections
    feats, grads, gold = _golden_grads(precision, tmp_path, "tcgen05")
    assert rel(feats.cpu(), torch.from_numpy(gold["features"])) < tol
    names = [str(n) for n in gold["param_names"]]
    gnorm = float(np.sqrt((gold["grad_norm"] ** 2).sum()))
    for i, n in enumerate(names):
        g = grads[n]
        assert g is not None and torch.isfinite(g).all(), n
        assert abs(g.double().norm().item() - gold["grad_norm"][i]) < 10 * tol * gold["grad_norm"][i] + 1e-5 * gnorm, n
        assert np.allclose(projections(g.cpu(), n), gold["grad_proj"][i], rtol=0, atol=10 * tol * gold["grad_norm"][i] * 4 + 1e-5 * gnorm), n
    _, per = _golden_errors(grads, gold)
    worst = max(e for n, e in per.items() if not n.startswith("encoder.layers.3."))
    assert worst < 10 * tol, worst


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_tcgen05_core_gradients_match_sdpa_core(precision, tmp_path):
    """Same model, same inputs, both training cores.  Over all parameters the tcgen05 core's gradients are at most 1.5x as far from HF's
    fp32 golden as the SDPA core's (the rule of test_kernels_match_fp32_autograd, applied to the whole model), and every parameter holding
    at least 1 % of the gradient norm agrees between the cores within 2x the kernel ceiling (the difference of two errors)."""
    _, g_tc, gold = _golden_grads(precision, tmp_path, "tcgen05")
    _, g_sd, _ = _golden_grads(precision, tmp_path, "sdpa")
    e_tc, _ = _golden_errors(g_tc, gold)
    e_sd, _ = _golden_errors(g_sd, gold)
    assert e_tc <= 1.5 * e_sd, (e_tc, e_sd)
    total = math.sqrt(sum(float(g.double().norm()) ** 2 for g in g_sd.values()))
    bar = 2 * CEIL[torch.float16 if precision == "fp16" else torch.bfloat16]
    for n, g in g_sd.items():
        if g.norm() > 1e-2 * total:
            assert rel(g_tc[n], g) < bar, (n, rel(g_tc[n], g))


def test_graphed_finetune_step_on_swinv2_backbone(tmp_path):
    """The finetune step on a swinv2_xs Poser (fp16, 16 x 16 windows: the tcgen05 core) captured as one CUDA graph: it replays, the loss
    is finite and falls, and equals the eager step's loss trajectory within 1e-3 relative."""
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
        model.backbone._v2_train_tc = True          # CSVIT_V2_TRAIN_ATTN=tcgen05
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
