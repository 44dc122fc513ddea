"""GPU tests of the SwinV2 8 x 8-window cosine attention on tcgen05 (csvit_swinv2_attn8_tc / _train / _bwd,
cs_vit.autograd.swinv2_cosine_attention8): the kernels against fp32 autograd (bounded by 1.5x the error torch SDPA makes on the same
rounded inputs), reproducibility, mask, store-order and guard-band contracts, and the backbone switches CSVIT_V2_ATTN8 /
CSVIT_V2_TRAIN_ATTN8 against HF's goldens, the fp32 mode and the SDPA core."""
import json
import math
import os

import pytest
import torch

from test_swinv2_attn_bwd_gpu import CEIL, LN2, LOG2E, _golden_errors
from test_swinv2_gpu import V2_CASES, _backbone, rel, v2_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from cs_vit import ops as o
    return o


def _rel_index24(device):
    """[64 * 64] index of (dy + 7) * 24 + dx + 7 for query i, key j of an 8 x 8 window (the padded bias-table layout)."""
    i = torch.arange(64, device=device)
    dy = (i[:, None] >> 3) - (i[None, :] >> 3)
    dx = (i[:, None] & 7) - (i[None, :] & 7)
    return ((dy + 7) * 24 + dx + 7).reshape(-1)


def _inputs(B, H, heads, dtype, seed):
    from cs_vit import ops
    g = torch.Generator(device="cuda").manual_seed(seed)
    C, rows = 32 * heads, B * H * H
    scale = (math.log(10.0) + 0.8 * torch.randn(heads, device="cuda", generator=g)).clamp(max=math.log(100.0)).exp()
    qh = torch.nn.functional.normalize(torch.randn(rows, heads, 32, device="cuda", generator=g), dim=-1)
    kh = torch.nn.functional.normalize(torch.randn(rows, heads, 32, device="cuda", generator=g), dim=-1)
    q2 = (qh * (scale * LOG2E).view(1, heads, 1)).reshape(rows, C).to(dtype)
    k = kh.reshape(rows, C).to(dtype)
    v = torch.randn(rows, C, device="cuda", generator=g).to(dtype)
    tab = 16 * torch.sigmoid(2 * torch.randn(heads, 225, device="cuda", generator=g))
    bl2 = ops.swinv2_bias8_log2(tab)
    dout = torch.randn(rows, C, device="cuda", generator=g).to(dtype)
    return q2, k, v, bl2, dout


def _reference(q2, k, v, bl2, dout, B, H, heads, shift, mask_repeat):
    """fp32 autograd on materialised scores, natural domain: (ctx, lse2, dq2, dk, dv, dbias_log2)."""
    from cs_vit import ops
    L, C = 64, 32 * heads
    nW = (H // 8) ** 2
    qf, kf, vf = (t.float().view(B * nW, L, heads, 32).transpose(1, 2).requires_grad_(True) for t in (q2, k, v))
    bf = bl2.clone().requires_grad_(True)
    s = LN2 * (qf @ kf.transpose(-1, -2) + bf.view(heads, -1)[:, _rel_index24(q2.device)].view(1, heads, L, L))
    if shift:
        m = ops.shift_mask(H, H, 8, shift)
        s = (s.view(B, nW, heads, L, L) + mask_repeat * m[None, :, None]).view(B * nW, heads, L, L)
    p = s.softmax(-1)
    lse2 = torch.logsumexp(s, -1) / LN2
    o = p @ vf
    o.backward(dout.float().view(B * nW, L, heads, 32).transpose(1, 2))
    back = lambda t: t.transpose(1, 2).reshape(B * H * H, C)      # noqa: E731
    return back(o.detach()), lse2.detach(), back(qf.grad), back(kf.grad), back(vf.grad), bf.grad


def _sdpa(q2, k, v, bl2, dout, B, H, heads, shift, mask_repeat):
    """Torch SDPA (memory-efficient backend) on the same 16-bit inputs: (ctx, dq2, dk, dv, dbias_log2)."""
    from cs_vit import ops
    from torch.nn.attention import SDPBackend, sdpa_kernel
    L, C, dt = 64, 32 * heads, q2.dtype
    nW = (H // 8) ** 2
    qf, kf, vf = (t.detach().view(B * nW, L, heads, 32).transpose(1, 2).requires_grad_(True) for t in (q2, k, v))
    bf = bl2.clone().requires_grad_(True)
    add = LN2 * bf.view(heads, -1)[:, _rel_index24(q2.device)].view(1, heads, L, L)
    if shift:
        add = (add + mask_repeat * ops.shift_mask(H, H, 8, shift)[:, None]).reshape(1, nW * heads, L, L)
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
    ctx, lse2 = ops.swinv2_attn8_tc_train(qkv, bl2, B, H, H, heads, shift, mask_repeat)
    grads = ops.swinv2_attn8_tc_bwd(qkv, ctx, lse2, dout, bl2, B, H, H, heads, shift, mask_repeat, out=out)
    return (ctx, lse2) + tuple(grads)


# (H, heads, shift, B): B * nW odd and even, heads 1 / 3 / 4 / 32, shift 0 / 4, H 8 / 16 / 64 (and 24: 9 windows per image);
# (8, 32, 0, 32) is SwinV2-B's stage 3 at batch 32
CASES = [(8, 1, 0, 1), (8, 4, 4, 3), (8, 32, 0, 32), (8, 32, 0, 5), (16, 3, 0, 2), (16, 4, 4, 1), (16, 1, 4, 3), (16, 32, 4, 1),
         (24, 4, 4, 1), (64, 1, 4, 1), (64, 3, 4, 2), (64, 4, 0, 2), (32, 4, 4, 2)]


@pytest.mark.parametrize("H,heads,shift,B", CASES)
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_attn8_kernels_match_fp32_autograd(ops, H, heads, shift, B, dtype):
    q2, k, v, bl2, dout = _inputs(B, H, heads, dtype, seed=13 * H + heads + shift + B)
    ref = _reference(q2, k, v, bl2, dout, B, H, heads, shift, 2)
    got = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift)
    sd = _sdpa(q2, k, v, bl2, dout, B, H, heads, shift, 2)
    names = ("ctx", "dq2", "dk", "dv", "dbias")
    errs = {n: rel(g, r) for n, g, r in zip(names, (got[0],) + got[2:], (ref[0],) + ref[2:])}
    sdpa = {n: rel(s, r) for n, s, r in zip(names, sd, (ref[0],) + ref[2:])}
    print(f"H{H} heads{heads} shift{shift} B{B} {dtype}: kernel {errs} sdpa {sdpa}")
    for n in names:
        assert errs[n] <= 1.5 * sdpa[n] and errs[n] < CEIL[dtype], (n, errs, sdpa)
    assert (got[1] - ref[1].view_as(got[1])).abs().max().item() < 2e-2       # lse2 (log2 units): the rounded-probability sums
    assert torch.equal(got[5][:, :, 15:], torch.zeros_like(got[5][:, :, 15:]))
    # the inference kernel computes the training forward's context
    qkv = torch.cat([q2, k, v], 1)
    assert torch.equal(ops.swinv2_attn8_tc(qkv, bl2, B, H, H, heads, shift), got[0])


@pytest.mark.parametrize("H,heads,shift,B", [(24, 3, 4, 1), (8, 1, 0, 3)])      # odd window counts: a half-filled last tile
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_attn8_reproducible_and_contracts(ops, H, heads, shift, B, dtype):
    rows, C = B * H * H, 32 * heads
    q2, k, v, bl2, dout = _inputs(B, H, heads, dtype, seed=5 + heads)
    a = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift)
    b = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift)
    for x, y in zip(a[:5], b[:5]):
        assert torch.equal(x, y)                                               # ctx, lse2, dq, dk, dv: bit-identical
    assert (a[5] - b[5]).abs().max().item() <= 1e-6 * max(1.0, a[5].abs().max().item())
    # guard-banded outputs: nothing written past the last row of the odd window count (or before the first)
    guard = 4096
    bufs = [torch.full((rows * C + 2 * guard,), 7.0, dtype=dtype, device="cuda") for _ in range(3)]
    views = tuple(t[guard:guard + rows * C].view(rows, C) for t in bufs)
    c = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift, out=views)
    for t, x, y in zip(bufs, c[2:5], a[2:5]):
        assert torch.equal(x, y)
        assert (t[:guard] == 7).all() and (t[-guard:] == 7).all()
    # the forward's operand, lse2 and context buffers: a half-filled tile reads zeros past the end and writes nothing there
    qkv_g = torch.full((rows + 64, 3 * C), 7.0, dtype=dtype, device="cuda")
    qkv_g[:rows] = torch.cat([q2, k, v], 1)
    ctx_g = ops.swinv2_attn8_tc(qkv_g[:rows], bl2, B, H, H, heads, shift)
    assert torch.equal(ctx_g, a[0])
    # token order: the window-ordered output scattered by window_index_map
    tok = ops.swinv2_attn8_tc(torch.cat([q2, k, v], 1), bl2, B, H, H, heads, shift, token_order=True)
    idx = ops.window_index_map(H, H, 8, shift, device="cuda").long()
    want = torch.empty_like(a[0]).view(B, H * H, C)
    want[:, idx] = a[0].view(B, H * H, C)
    assert torch.equal(tok, want.view(rows, C))


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_attn8_mask_repeat_contract(ops, dtype):
    """mask_repeat = 0 drops the shift mask: it matches the unmasked reference and differs from the masked one when shift = 4."""
    B, H, heads, shift = 2, 16, 3, 4
    q2, k, v, bl2, dout = _inputs(B, H, heads, dtype, seed=77)
    a = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift)
    z = _kernels(ops, q2, k, v, bl2, dout, B, H, heads, shift, mask_repeat=0)
    ref0 = _reference(q2, k, v, bl2, dout, B, H, heads, shift, 0)
    assert rel(z[0], ref0[0]) < CEIL[dtype] and rel(a[0], ref0[0]) > CEIL[dtype]
    assert rel(z[2], ref0[2]) < CEIL[dtype] and rel(a[2], ref0[2]) > CEIL[dtype]
    assert rel(z[5], a[5]) > 1e-2


def test_attn8_rejects_bad_geometry(ops):
    q2, k, v, bl2, _ = _inputs(1, 16, 2, torch.float16, seed=1)
    qkv = torch.cat([q2, k, v], 1)
    with pytest.raises(RuntimeError, match="shift 0 or 4"):
        ops.swinv2_attn8_tc(qkv, bl2, 1, 16, 16, 2, 8)
    with pytest.raises(RuntimeError, match="windows of 8"):
        ops.swinv2_attn8_tc(qkv[: 12 * 12], bl2, 1, 12, 12, 2, 0)


# ---------------------------------------------------------------------------------------------------- backbone


def _golden_grads(precision, tmp_path, tc):
    """Features and gradients of the w16 gradient golden with both tcgen05 cores (CSVIT_V2_TRAIN_ATTN=CSVIT_V2_TRAIN_ATTN8=tcgen05) or
    neither (SDPA)."""
    from test_swinv2_oracle import V2_GRAD_CASES
    sd, px, gold, case = v2_case(sorted(V2_GRAD_CASES)[0])
    model = _backbone(case, precision, str(tmp_path))
    model.config.drop_path_rate = 0.0
    model._v2_train_tc = model._v2_train_tc8 = tc
    model.train()
    for p_ in model.parameters():
        p_.requires_grad_(True)
    feats = model.forward_features(px.cuda(), normalize=False)
    R = torch.randn(feats.shape, generator=torch.Generator().manual_seed(case["projection_seed"])).cuda()
    (feats * R).sum().backward()
    torch.cuda.synchronize()
    return feats.detach(), {n: p.grad for n, p in model.named_parameters()}, gold


def test_w16_golden_with_both_tcgen05_cores(tmp_path):
    """The gradient golden train_swinv2_xs_w16_linear with the 16 x 16 and the 8 x 8 tcgen05 cores on (stage 3 runs the new core): features,
    every gradient norm and projection at the existing fp16 / bf16 bars; over all parameters the error is at most 1.5x that of the SDPA
    cores.  Prints the last stage's query.bias error (the parameter that kept the 16 x 16 core opt-in)."""
    from oracle.make_train_goldens import projections
    import numpy as np
    for precision, tol in (("fp16", 3e-3), ("bf16", 3e-2)):
        feats, g_tc, gold = _golden_grads(precision, tmp_path, True)
        _, g_sd, _ = _golden_grads(precision, tmp_path, False)
        assert rel(feats.cpu(), torch.from_numpy(gold["features"])) < tol
        names = [str(n) for n in gold["param_names"]]
        gnorm = float(np.sqrt((gold["grad_norm"] ** 2).sum()))
        for i, n in enumerate(names):
            g = g_tc[n]
            assert g is not None and torch.isfinite(g).all(), n
            assert abs(g.double().norm().item() - gold["grad_norm"][i]) < 10 * tol * gold["grad_norm"][i] + 1e-5 * gnorm, n
            assert np.allclose(projections(g.cpu(), n), gold["grad_proj"][i], rtol=0, atol=10 * tol * gold["grad_norm"][i] * 4 + 1e-5 * gnorm), n
        e_tc, per_tc = _golden_errors(g_tc, gold)
        e_sd, per_sd = _golden_errors(g_sd, gold)
        qb = [n for n in per_tc if n.startswith("encoder.layers.3.") and n.endswith("query.bias")]
        print(f"{precision}: total error tcgen05 {e_tc:.3e} sdpa {e_sd:.3e}; last-stage query.bias "
              + ", ".join(f"{n}: tcgen05 {per_tc[n]:.3e} sdpa {per_sd[n]:.3e}" for n in qb)
              + f"; worst parameter tcgen05 {max(per_tc.values()):.3e} sdpa {max(per_sd.values()):.3e}")
        assert e_tc <= 1.5 * e_sd, (precision, e_tc, e_sd)


def _w8_grads(tmp, precision, attn8, px):
    from cs_vit.synthetic import make_random_backbone_dir
    from cs_vit.net.swinv2_b200 import load_backbone
    d = make_random_backbone_dir(os.path.join(tmp, "v2xs_w8"), "swinv2_xs", seed=0, image_size=256, window_size=8)
    model = load_backbone(d, precision=precision).cuda()
    model.config.drop_path_rate = 0.0
    model._v2_train_tc8 = attn8 == "tcgen05"          # what CSVIT_V2_TRAIN_ATTN8 selects
    model.train()
    for p_ in model.parameters():
        p_.requires_grad_(True)
    feats = model.forward_features(px, normalize=False)
    R = torch.randn(feats.shape, generator=torch.Generator().manual_seed(5)).cuda()
    (feats * R).sum().backward()
    torch.cuda.synchronize()
    return feats.detach(), {n: p.grad.detach().double() for n, p in model.named_parameters()}


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_window8_backbone_gradients(precision, tmp_path):
    """A window-8 swinv2_xs at 256^2 (shift 4 at stages 0-2, every stage on 8 x 8 windows): the tcgen05 core's gradients are at most 1.5x
    as far from the fp32 mode's gradients of the same weights as the SDPA core's (the fp32 mode is pinned to HF by the goldens)."""
    px = torch.randn(2, 3, 256, 256, generator=torch.Generator().manual_seed(12)).cuda()
    f32, g32 = _w8_grads(str(tmp_path), "fp32", "sdpa", px)
    f_tc, g_tc = _w8_grads(str(tmp_path), precision, "tcgen05", px)
    f_sd, g_sd = _w8_grads(str(tmp_path), precision, "sdpa", px)

    def total(g):
        return math.sqrt(sum(float((g[n] - g32[n]).norm()) ** 2 for n in g32) / sum(float(g32[n].norm()) ** 2 for n in g32))
    e_tc, e_sd = total(g_tc), total(g_sd)
    print(f"{precision}: features tcgen05 {rel(f_tc, f32):.3e} sdpa {rel(f_sd, f32):.3e}; gradients tcgen05 {e_tc:.3e} sdpa {e_sd:.3e}")
    assert rel(f_tc, f32) <= 1.5 * rel(f_sd, f32) + 1e-4
    assert e_tc <= 1.5 * e_sd, (e_tc, e_sd)


@pytest.mark.parametrize("name", sorted(V2_CASES))
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_inference_with_tcgen05_attn8_matches_hf_goldens(name, precision, tmp_path):
    """CSVIT_V2_ATTN8=tcgen05: the 8 x 8 windows (every stage of swinv2_xs_w8, the last stage of the w16 cases) on the new kernel, at the
    bars of the existing golden test."""
    sd, px, gold, case = v2_case(name)
    model = _backbone(case, precision, str(tmp_path))
    model._v2_tcgen05_8 = True
    with torch.no_grad():
        out, stages = model.forward_features(px.cuda(), normalize=False, return_stages=True)
    tol = {"fp16": 2e-3, "bf16": 1e-2}[precision]
    err = rel(out.cpu(), torch.from_numpy(gold["last_hidden_state"]))
    serr = [rel(t[:, ::case["stage_token_stride"]].cpu(), torch.from_numpy(gold[f"stage{s}"])) for s, t in enumerate(stages)]
    print(f"{name} {precision}: last {err:.2e} stages {['%.1e' % e for e in serr]}")
    assert err < tol and max(serr) < tol


def test_graphed_finetune_step_on_window8_backbone(tmp_path):
    """The finetune step on a window-8 swinv2_xs Poser (fp16, CSVIT_V2_TRAIN_ATTN8=tcgen05) captured as one CUDA graph: it replays, the
    loss is finite and falls, and equals the eager step's loss trajectory within 1e-3 relative."""
    from cs_vit.net import Poser
    from cs_vit.synthetic import make_inputs, make_random_backbone_dir, randomize_head_
    from cs_vit.train import GradReducer, GraphedFinetuneStep, finetune_step
    from cs_vit.utils.mano_standin import SyntheticMANO
    d = make_random_backbone_dir(str(tmp_path / "v2xs8"), "swinv2_xs", seed=0, image_size=256, window_size=8)
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
        model.backbone._v2_train_tc8 = True          # CSVIT_V2_TRAIN_ATTN8=tcgen05
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


def test_switches_read_at_construction(monkeypatch):
    """CSVIT_V2_ATTN8 / CSVIT_V2_TRAIN_ATTN8 are read when the backbone is built, default off, and leave CSVIT_V2_TRAIN_ATTN's switch alone."""
    from cs_vit.net.swinv2_b200 import Swinv2BackboneB200, Swinv2ConfigLite
    cfg = Swinv2ConfigLite.from_dict({"model_type": "swinv2", "embed_dim": 32, "depths": [1, 1], "num_heads": [1, 2], "window_size": 8,
                                      "image_size": 64})
    m = Swinv2BackboneB200(cfg)
    assert not m._v2_tcgen05_8 and not m._v2_train_tc8 and not m._v2_train_tc
    monkeypatch.setenv("CSVIT_V2_ATTN8", "tcgen05")
    monkeypatch.setenv("CSVIT_V2_TRAIN_ATTN8", "tcgen05")
    m = Swinv2BackboneB200(cfg)
    assert m._v2_tcgen05_8 and m._v2_train_tc8 and not m._v2_train_tc
