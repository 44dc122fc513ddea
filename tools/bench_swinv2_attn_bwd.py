"""GPU microbench: the SwinV2-B cosine-attention core of the finetune step at batch 32 (16 x 16 windows: stage 0 64^2 / 4 heads, stage 1
32^2 / 8 heads, both shifts, stage 2 16^2 / 16 heads), fp16.  On the same inputs it times with CUDA events
  tcgen05: csvit_swinv2_attn_tc_train (forward) and csvit_swinv2_attn_tc_bwd (backward)
  sdpa:    the core _forward_train issues with CSVIT_V2_TRAIN_ATTN=sdpa - bias gather 16 sigmoid(table[rel_index]) (+ 2 x shift mask), torch
           SDPA (memory-efficient backend) forward, and its backward including the bias-gather backward (IndexBackward)
and reports microseconds per launch, ns per (window, head) and each path's relative error norm against fp32 autograd (ctx, dq, dk, dv,
dbias).  Writes profiles/r3_swinv2_attn_bwd_microbench.json (or $OUT) with the GPU name and power limit read in the same run."""
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs-vit_b200"))
import torch  # noqa: E402
from torch.nn.attention import SDPBackend, sdpa_kernel  # noqa: E402

from cs_vit import ops  # noqa: E402

B = int(os.environ.get("B", "32"))
ITERS = int(os.environ.get("ITERS", "20"))
LOG2E, LN2 = 1.4426950408889634, math.log(2.0)
SHAPES = [(64, 4, 0), (64, 4, 8), (32, 8, 0), (32, 8, 8), (16, 16, 0)]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:      # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def events(fn):
    """(mean ms of fn over ITERS after 3 warm-up calls)."""
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(ITERS):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / ITERS


def rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-30)).item()


def main():
    dt = torch.float16
    out = {"gpu": gpu_info(), "batch": B, "dtype": "fp16", "iters": ITERS, "shapes": []}
    for H, heads, shift in SHAPES:
        g = torch.Generator(device="cuda").manual_seed(H + heads + shift)
        C, rows, L = 32 * heads, B * H * H, 256
        nW = (H // 16) ** 2
        windows = B * nW
        scale = torch.full((heads,), 10.0, device="cuda")
        qh = torch.nn.functional.normalize(torch.randn(rows, heads, 32, device="cuda", generator=g), dim=-1)
        kh = torch.nn.functional.normalize(torch.randn(rows, heads, 32, device="cuda", generator=g), dim=-1)
        q2 = (qh * (scale * LOG2E).view(1, heads, 1)).reshape(rows, C).to(dt)
        k = kh.reshape(rows, C).to(dt)
        v = torch.randn(rows, C, device="cuda", generator=g).to(dt)
        dout = torch.randn(rows, C, device="cuda", generator=g).to(dt)
        table = 2 * torch.randn(961, heads, device="cuda", generator=g)              # CPB-MLP output [31 * 31, heads]
        tab16 = 16 * torch.sigmoid(table)
        bl2 = ops.swinv2_bias_log2(tab16.t().contiguous())
        rel_index = ops.rel_pos_index(16).long().reshape(-1)
        mask = ops.shift_mask(H, H, 16, shift) if shift else None

        # ---- tcgen05 pair
        qkv = torch.cat([q2, k, v], 1)
        holder = {}

        def tc_fwd():
            holder["ctx"], holder["lse2"] = ops.swinv2_attn_tc_train(qkv, bl2, B, H, H, heads, shift)

        def tc_bwd():
            holder["g"] = ops.swinv2_attn_tc_bwd(qkv, holder["ctx"], holder["lse2"], dout, bl2, B, H, H, heads, shift)

        tc_fwd()
        t_tc_f = events(tc_fwd)
        t_tc_b = events(tc_bwd)

        # ---- SDPA core as _forward_train issues it (q / k / v the strided [windows, heads, L, d] views of [rows, heads, d])
        # natural-domain q = q2 ln 2 rounded to 16 bit, as cosnorm would emit q_hat * scale
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
            holder["sd"] = (o.reshape(windows, heads, L, 32), qv, kv, vv)

        gout = dout.view(windows, L, heads, 32).transpose(1, 2)

        def sdpa_bwd():
            o = holder["sd"][0]
            tabp.grad = None
            o.backward(gout, retain_graph=True)

        sdpa_fwd()
        t_sd_f = events(sdpa_fwd)
        t_sd_b = events(sdpa_bwd)

        # ---- errors against fp32 autograd of the natural-domain formula on the same rounded inputs
        qf, kf, vf = (t.float().view(windows, L, heads, 32).transpose(1, 2).requires_grad_(True) for t in (qn, k, v))
        tf = table.clone().requires_grad_(True)
        s = qf @ kf.transpose(-1, -2) + 16.0 * torch.sigmoid(tf[rel_index].view(L, L, heads).permute(2, 0, 1))[None]
        if mask is not None:
            s = (s.view(B, nW, heads, L, L) + 2.0 * mask[None, :, None]).view(windows, heads, L, L)
        of = s.softmax(-1) @ vf
        of.backward(gout.float())
        back = lambda t: t.transpose(1, 2).reshape(rows, C)      # noqa: E731
        ref = {"ctx": back(of.detach()), "dq": back(qf.grad), "dk": back(kf.grad), "dv": back(vf.grad)}
        # d loss / d (16 sigmoid(table)) of the fp32 reference in the table layout [heads, 31, 31] (tf.grad carries the sigmoid's derivative)
        sig = torch.sigmoid(table)
        dbias_ref = (tf.grad / (16.0 * sig * (1 - sig))).t().reshape(heads, 31, 31)      # d loss / d (16 sigmoid(table))
        del of, s, qf, kf, vf
        dq, dk, dv, dbl2 = holder["g"]
        err_tc = {"ctx": rel(holder["ctx"], ref["ctx"]), "dq": rel(dq * LOG2E, ref["dq"]), "dk": rel(dk, ref["dk"]), "dv": rel(dv, ref["dv"]),
                  "dbias": rel(dbl2[:, :, :31] * LOG2E, dbias_ref)}
        sdpa_fwd()
        sdpa_bwd()
        o, qv, kv, vv = holder["sd"]
        sig_g = tabp.grad / (16.0 * sig * (1 - sig))
        err_sd = {"ctx": rel(back(o.detach()), ref["ctx"]), "dq": rel(back(qv.grad), ref["dq"]), "dk": rel(back(kv.grad), ref["dk"]),
                  "dv": rel(back(vv.grad), ref["dv"]), "dbias": rel(sig_g.t().reshape(heads, 31, 31), dbias_ref)}
        items = windows * heads
        row = {"H": H, "heads": heads, "shift": shift, "windows_x_heads": items,
               "tcgen05": {"fwd_us": t_tc_f * 1e3, "bwd_us": t_tc_b * 1e3, "fwd_ns_per_item": t_tc_f * 1e6 / items,
                           "bwd_ns_per_item": t_tc_b * 1e6 / items, "err_vs_fp32": err_tc},
               "sdpa": {"fwd_us": t_sd_f * 1e3, "bwd_us": t_sd_b * 1e3, "fwd_ns_per_item": t_sd_f * 1e6 / items,
                        "bwd_ns_per_item": t_sd_b * 1e6 / items, "err_vs_fp32": err_sd}}
        out["shapes"].append(row)
        print(json.dumps(row), flush=True)
        holder.clear()
        torch.cuda.empty_cache()
    path = os.environ.get("OUT", os.path.join(ROOT, "profiles", "r3_swinv2_attn_bwd_microbench.json"))
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
