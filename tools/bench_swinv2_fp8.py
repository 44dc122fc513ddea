"""FP8 inference mode of the SwinV2 backbone against fp16, on one GPU.

    python tools/bench_swinv2_fp8.py [--out FILE] [--steps K] [--reps R]

The model is the one of tools/bench_stream.py (SwinV2-B at 256², realtime temporal Poser, "encoder" head, ``randomize_head_``).
In one run it records:

  predict_batch   graphed ``predict_batch`` (``cs_vit.graph.GraphedPredict``) of one frame per image at batch 256 and 32, the fp16 and
                  fp8 graphs alternated R times; CUDA-event time per call and images/s.
  gemms           every stage's Q/K/V projection (the cosine-normalising epilogue at stages 0-2, the plain one at stage 3, as the model
                  runs them) and fc1 + GELU at batch 256 and 32: fp16 operands against E4M3 operands, CUDA events over K calls after a
                  warm-up, achieved TFLOP/s = 2 M N K / time.
  stream          graphed ``RealtimeStream.step`` at 256 streams, window 8, fp16 and fp8 alternated R times.
  accuracy        the backbone errors of tests/test_fp8_gpu.py::test_fp8_backbone_accuracy: fp8 and fp16 modes against the fp32 mode,
                  and the fp32 emulation of the fp8 mode against exact fp32.

The GPU's name, power limit and maximum SM clock are read in the same run; the SM clock is sampled while each timed loop runs.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs-vit_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch  # noqa: E402

from bench_stream import KEYS, build_model, smi, timed  # noqa: E402

STAGE_C = (128, 256, 512, 1024)
TOKENS = (4096, 1024, 256, 64)


def bench_gemms(B: int, steps: int):
    from cs_vit import ops
    from test_fp8_gpu import quant_rows
    rows = []
    g = torch.Generator(device="cuda").manual_seed(0)
    for s, C in enumerate(STAGE_C):
        M = B * TOKENS[s]
        x = torch.randn(M, C, device="cuda", generator=g)
        x16 = x.half()
        a8, rs = quant_rows(x)
        qs = torch.full((C // 32,), 14.4, device="cuda")
        for kind, N in (("qkv", 3 * C), ("fc1", 4 * C)):
            w = 0.05 * torch.randn(N, C, device="cuda", generator=g)
            w16 = w.half()
            w8, cs = ops.quantize_weight_fp8(w)
            b = torch.zeros(N, device="cuda")
            if kind == "qkv" and s < 3:
                f16 = lambda: ops.swinv2_qkv(x16, w16, b, qs)                                   # noqa: E731
                f8 = lambda: ops.swinv2_qkv_fp8(a8, rs, w8, cs, b, qs)                          # noqa: E731
            elif kind == "qkv":
                f16 = lambda: ops.linear(x16, w16, b, out_dtype=torch.float16)                  # noqa: E731
                f8 = lambda: ops.linear_fp8(a8, rs, w8, cs, b, out_dtype=torch.float16)        # noqa: E731
            else:
                f16 = lambda: ops.linear(x16, w16, b, act=ops.ACT_GELU, out_dtype=torch.float16)       # noqa: E731
                f8 = lambda: ops.linear_fp8(a8, rs, w8, cs, b, act=ops.ACT_GELU, out_dtype=torch.float16)      # noqa: E731
            row = {"stage": s, "kind": kind, "M": M, "N": N, "K": C}
            for name, f in (("fp16", f16), ("fp8", f8)):
                for _ in range(3):
                    f()
                ms, sample = timed(f, steps)
                row[name] = {"us": round(1e3 * ms, 2), "tflops": round(2.0 * M * N * C / (ms * 1e-3) / 1e12, 1), "sm_clock_and_power_during": sample}
            row["fp8_speedup"] = round(row["fp16"]["us"] / row["fp8"]["us"], 3)
            rows.append(row)
            del w, w16, w8
        del x, x16, a8
    torch.cuda.empty_cache()
    return rows


def bench_predict(model, B: int, steps: int, reps: int):
    from cs_vit.graph import GraphedPredict
    from cs_vit.synthetic import make_inputs
    inp = {k: v.cuda() for k, v in make_inputs(B, 1, 256, seed=5).items()}
    graphs = {}
    for p in ("fp16", "fp8"):
        model.set_precision(p)
        graphs[p] = GraphedPredict(model, inp)
    runs = {p: [] for p in graphs}
    for _ in range(reps):
        for p, gp in graphs.items():
            ms, sample = timed(lambda: gp(*(inp[k] for k in KEYS)), steps)
            runs[p].append({"ms_per_call": round(ms, 3), "images_per_s": round(B / (ms / 1e3), 1), "sm_clock_and_power_during": sample})
    a, b = graphs["fp16"].static_out["joint_cam"].double(), graphs["fp8"].static_out["joint_cam"].double()
    out = {"batch": B, "runs": runs, "best_ms": {p: min(r["ms_per_call"] for r in v) for p, v in runs.items()},
           "joint_cam_rel_diff_fp8_vs_fp16": ((a - b).norm() / a.norm()).item()}
    out["fp8_speedup"] = round(out["best_ms"]["fp16"] / out["best_ms"]["fp8"], 3)
    del graphs
    torch.cuda.empty_cache()
    return out


def bench_stream(model, streams: int, steps: int, reps: int):
    from cs_vit.stream import RealtimeStream
    from cs_vit.synthetic import make_inputs
    inp = make_inputs(streams, 1, 256, seed=9)
    frame = {k: inp[k][:, 0].contiguous().cuda() for k in KEYS if k != "timestamp"}
    clock = {"t": 0}
    sessions = {}
    for p in ("fp16", "fp8"):
        model.set_precision(p)
        sessions[p] = RealtimeStream(model, streams, 8)

    def step(sess):
        clock["t"] += 1
        ts = torch.full((streams,), 33.333 * clock["t"], device="cuda")
        return sess.step(frame["patches"], frame["square_bboxes"], ts, frame["focal"], frame["princpt"])

    for p, sess in sessions.items():
        model.set_precision(p)
        for _ in range(10):
            step(sess)
    runs = {p: [] for p in sessions}
    for _ in range(reps):
        for p, sess in sessions.items():
            ms, sample = timed(lambda: step(sess), steps)
            runs[p].append({"ms_per_step": round(ms, 3), "predictions_per_s": round(streams / (ms / 1e3), 1), "sm_clock_and_power_during": sample})
    out = {"streams": streams, "window": 8, "runs": runs, "best_ms": {p: min(r["ms_per_step"] for r in v) for p, v in runs.items()}}
    out["fp8_speedup"] = round(out["best_ms"]["fp16"] / out["best_ms"]["fp8"], 3)
    del sessions
    torch.cuda.empty_cache()
    return out


def accuracy(tmp: str):
    from cs_vit.net.swinv2_b200 import load_backbone
    from cs_vit.synthetic import SWINV2_VARIANTS, make_random_backbone_dir
    from oracle import swinv2_restated as v2
    from test_fp8_gpu import _emulated_forward, rel
    from test_swinv2_oracle import v2_case
    res = []
    for name, attn8 in (("swinv2_t_w16", False), ("swinv2_xs_w8", False), ("swinv2_xs_w8", True)):
        sd, px, _, case = v2_case(name)
        _, depths, heads = SWINV2_VARIANTS[case["variant"]]
        d = make_random_backbone_dir(os.path.join(tmp, name), case["variant"], seed=case["weight_seed"], image_size=case["image_size"],
                                     window_size=case["window"])
        model = load_backbone(d, precision="fp32").cuda()
        model._v2_tcgen05_8 = attn8
        out = {}
        with torch.no_grad():
            for p in ("fp32", "fp16", "fp8"):
                model.precision = p
                out[p] = model.forward_features(px.cuda(), normalize=False).cpu()
            emu = _emulated_forward(sd, px, depths, heads, case["window"])
            exact = v2.swinv2_forward(px, sd, depths, heads, window=case["window"])
        res.append({"case": name, "attn8_tcgen05": attn8, "fp8_vs_fp32_mode": rel(out["fp8"], out["fp32"]),
                    "fp16_vs_fp32_mode": rel(out["fp16"], out["fp32"]), "fp8_emulation_vs_fp32": rel(emu, exact)})
    return res


def main():
    import tempfile
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_swinv2_fp8.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_swinv2_fp8 measures on a CUDA device; none is visible")
    res = {"gpu": smi("name,power.limit,clocks.max.sm"), "torch": torch.__version__}
    res["accuracy"] = accuracy(tempfile.mkdtemp(prefix="csvit_fp8_acc_"))
    res["gemms"] = {f"batch{B}": bench_gemms(B, 4 * a.steps) for B in (256, 32)}
    model = build_model("swinv2_b", 256, "realtime")
    res["predict_batch"] = [bench_predict(model, B, a.steps, a.reps) for B in (256, 32)]
    res["stream"] = bench_stream(model, 256, a.steps, a.reps)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "accuracy": res["accuracy"],
                      "gemm_speedups": {k: [(r["stage"], r["kind"], r["fp16"]["us"], r["fp8"]["us"], r["fp8"]["tflops"]) for r in v]
                                        for k, v in res["gemms"].items()},
                      "predict_batch": [(r["batch"], r["best_ms"], r["fp8_speedup"], r["joint_cam_rel_diff_fp8_vs_fp16"]) for r in res["predict_batch"]],
                      "stream": (res["stream"]["best_ms"], res["stream"]["fp8_speedup"])}))


if __name__ == "__main__":
    main()
