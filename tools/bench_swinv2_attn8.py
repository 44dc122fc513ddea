"""GPU microbench of the SwinV2 8 x 8-window cosine attention, fp16, batch 32 (B): the four stages of a window-8 SwinV2-B at 256^2 (64^2 / 4
heads, 32^2 / 8, 16^2 / 16 with shift 4, and 8^2 / 32 heads with shift 0 - the last one is also stage 3 of every window-16 SwinV2-B).
On the same inputs it times with CUDA events
  tcgen05:  csvit_swinv2_attn8_tc (inference, token order), csvit_swinv2_attn8_tc_train (forward) and csvit_swinv2_attn8_tc_bwd
  mma:      csvit_swinv2_window_attention with ws = 8 (round 1's mma.sync kernel, the inference default)
  sdpa:     the core _forward_train issues by default - bias gather 16 sigmoid(table[rel_index]) (+ 2 x shift mask), torch SDPA
            (memory-efficient backend) forward, and its backward including the bias-gather backward
and reports ns per (window, head).  Then (unless STEP=0) it times a graphed finetune step of a window-8 SwinV2-B Poser (fp16, batch B),
alternating CSVIT_V2_TRAIN_ATTN8 = sdpa / tcgen05 twice.  Writes profiles/r4_swinv2_attn8_microbench.json (or $OUT) with the GPU name
and power limit read in the same run."""
import json
import math
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs-vit_b200"))
import torch  # noqa: E402
from torch.nn.attention import SDPBackend, sdpa_kernel  # noqa: E402

from cs_vit import ops  # noqa: E402

B = int(os.environ.get("B", "32"))
ITERS = int(os.environ.get("ITERS", "50"))
LOG2E, LN2 = 1.4426950408889634, math.log(2.0)
SHAPES = [(64, 4, 4), (32, 8, 4), (16, 16, 4), (8, 32, 0)]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:      # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def events(fn, iters=ITERS):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernels():
    dt, L = torch.float16, 64
    rows_out = []
    for H, heads, shift in SHAPES:
        g = torch.Generator(device="cuda").manual_seed(H + heads + shift)
        C, rows = 32 * heads, B * H * H
        nW = (H // 8) ** 2
        windows = B * nW
        scale = torch.full((heads,), 10.0, device="cuda")
        qh = torch.nn.functional.normalize(torch.randn(rows, heads, 32, device="cuda", generator=g), dim=-1)
        kh = torch.nn.functional.normalize(torch.randn(rows, heads, 32, device="cuda", generator=g), dim=-1)
        q2 = (qh * (scale * LOG2E).view(1, heads, 1)).reshape(rows, C).to(dt)
        k = kh.reshape(rows, C).to(dt)
        v = torch.randn(rows, C, device="cuda", generator=g).to(dt)
        dout = torch.randn(rows, C, device="cuda", generator=g).to(dt)
        table = 2 * torch.randn(225, heads, device="cuda", generator=g)
        tab16 = (16 * torch.sigmoid(table)).t().contiguous()
        bl2 = ops.swinv2_bias8_log2(tab16)
        rel_index = ops.rel_pos_index(8).long().reshape(-1)
        mask = ops.shift_mask(H, H, 8, shift) if shift else None
        qkv = torch.cat([q2, k, v], 1)
        raw = torch.cat([qh.reshape(rows, C).to(dt), k, v], 1)          # the mma.sync kernel normalises q and k itself
        holder = {}

        def tc_inf():
            holder["inf"] = ops.swinv2_attn8_tc(qkv, bl2, B, H, H, heads, shift, token_order=True)

        def tc_fwd():
            holder["ctx"], holder["lse2"] = ops.swinv2_attn8_tc_train(qkv, bl2, B, H, H, heads, shift)

        def tc_bwd():
            holder["g"] = ops.swinv2_attn8_tc_bwd(qkv, holder["ctx"], holder["lse2"], dout, bl2, B, H, H, heads, shift)

        def mma():
            holder["mma"] = ops.swinv2_window_attention(raw, tab16, scale, B, H, H, heads, 8, shift, token_order=True)

        tc_fwd()
        t_inf, t_f, t_b, t_mma = events(tc_inf), events(tc_fwd), events(tc_bwd), events(mma)
        qn = (q2.float() * LN2).to(dt)
        tabp = table.clone().requires_grad_(True)

        def sdpa_fwd():
            qv, kv, vv = (t.detach().view(windows, L, heads, 32).transpose(1, 2).requires_grad_(True) for t in (qn, k, v))
            bias = 16.0 * torch.sigmoid(tabp[rel_index].view(L, L, heads).permute(2, 0, 1))
            with sdpa_kernel([SDPBackend.EFFICIENT_ATTENTION, SDPBackend.MATH]):
                if mask is None:
                    o = torch.nn.functional.scaled_dot_product_attention(qv, kv, vv, attn_mask=bias[None].to(dt).contiguous(), scale=1.0)
                else:
                    add = (bias[None] + 2.0 * mask[:, None]).reshape(1, nW * heads, L, L).to(dt).contiguous()
                    q4, k4, v4 = (t.reshape(B, nW * heads, L, 32) for t in (qv, kv, vv))
                    o = torch.nn.functional.scaled_dot_product_attention(q4, k4, v4, attn_mask=add, scale=1.0)
            holder["sd"] = o

        gout = dout.view(windows, L, heads, 32).transpose(1, 2)

        def sdpa_bwd():
            tabp.grad = None
            holder["sd"].reshape(windows, heads, L, 32).backward(gout, retain_graph=True)

        sdpa_fwd()
        t_sf, t_sb = events(sdpa_fwd), events(sdpa_bwd)
        items = windows * heads
        ns = lambda ms: round(ms * 1e6 / items, 2)      # noqa: E731
        row = {"H": H, "heads": heads, "shift": shift, "windows_x_heads": items,
               "ns_per_window_head": {"tcgen05_infer": ns(t_inf), "tcgen05_fwd_train": ns(t_f), "tcgen05_bwd": ns(t_b), "mma_sync_infer": ns(t_mma),
                                      "sdpa_fwd": ns(t_sf), "sdpa_bwd_incl_bias_gather": ns(t_sb)},
               "max_abs_diff_infer_tcgen05_vs_mma": (holder["inf"].float() - holder["mma"].float()).abs().max().item()}
        rows_out.append(row)
        print(json.dumps(row), flush=True)
        holder.clear()
        torch.cuda.empty_cache()
    return rows_out


def finetune_ab(steps=20):
    from cs_vit.net import Poser
    from cs_vit.synthetic import make_inputs, make_random_backbone_dir, randomize_head_
    from cs_vit.train import GradReducer, GraphedFinetuneStep
    from cs_vit.utils.mano_standin import SyntheticMANO
    d = make_random_backbone_dir(os.path.join(tempfile.mkdtemp(prefix="csvit_attn8_"), "swinv2_b_w8"), "swinv2_b", seed=0, image_size=256,
                                 window_size=8)
    batch = {k: v.cuda() for k, v in make_inputs(B, 1, 256, seed=100, labels=True).items()}
    out = []
    for arm in ("sdpa", "tcgen05", "sdpa", "tcgen05"):
        torch.manual_seed(0)
        model = Poser(d, image_size=256, mano_layer=SyntheticMANO(), spatial_layer_type="encoder", persp_decorate="patch", precision="fp16")
        randomize_head_(model)
        model.phase(Poser.TrainingPhase.SPATIAL)
        model = model.cuda()
        model.backbone._v2_train_tc8 = arm == "tcgen05"       # what CSVIT_V2_TRAIN_ATTN8 selects
        params = [p for p in model.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-5, fused=True, capturable=True)
        step = GraphedFinetuneStep(model, batch, opt, GradReducer(params), warmup=3)
        ms = events(lambda: step(batch), iters=steps)
        r = {"arm": f"CSVIT_V2_TRAIN_ATTN8={arm}", "step_ms": round(ms, 3), "images_per_s": round(B * 1e3 / ms, 1),
             "loss": step(batch).item()}
        print(json.dumps(r), flush=True)
        out.append(r)
        del step, opt, model
        torch.cuda.empty_cache()
    return out


def main():
    out = {"gpu": gpu_info(), "batch": B, "dtype": "fp16", "iters": ITERS, "shapes": kernels()}
    if os.environ.get("STEP", "1") != "0":
        out["finetune_window8_swinv2_b_graphed"] = finetune_ab()
    path = os.environ.get("OUT", os.path.join(ROOT, "profiles", "r4_swinv2_attn8_microbench.json"))
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
