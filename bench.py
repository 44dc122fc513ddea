#!/usr/bin/env python
"""Headline benchmark: images/sec of the Swin-B spatial model forward (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision fp16|bf16] [--dump-outputs DIR]

One "step" = one ``Poser.predict_batch`` over a batch of 256 synthetic 224x224 crops per GPU (Swin-B backbone,
"encoder" spatial head, perspective embedding added to the patches - the ``spatial_dexycb_swinb_spenc_addpat``
configuration), random-init weights, eval mode.  Data-parallel: every rank owns its own batch, no data-path
collective (SURVEY.md §8e), so scaling is weak and ``value`` = all ranks' images / max-over-ranks device time.

Keys beyond the base contract:
  roofline      the GEMM engine (tcgen05 kernel) timed live with CUDA events on the launch stream in a second,
                instrumented pass of the same K steps: algorithmic FLOPs (2MNK summed over the launches) /
                summed launch time, against MEASURED_PEAKS.json's sustained bf16 figure.
  e2e           same metric through the public API with HOST (pinned) inputs: per step an H2D copy of that
                step's batch and a D2H read of the predicted joints, double-buffered on a copy stream.
  cpu_baseline  the oracle port (HF SwinModel + restated head, all six head layers executed like the
                reference) on the host cores, on a bounded sample, rank 0 at N=1 only.
  roofline_attention / roofline_attention_fused
                the two tcgen05 window-attention kernels (attn_core.cu: 20 launches/step, attn_fused.cu: 4), timed the same
                way, against the measured HBM copy bandwidth (they are HBM-bound: 8C resp. 6C algorithmic bytes per token).
  bf16          the same timed loop with bf16 instead of fp16 tensor-core operands (identical MMA rate).  The headline
                ``dtype`` is fp16: it is the 16-bit format whose joints / vertices meet the 1e-2 parity bar on this
                configuration (bf16 operand ROUNDING ALONE puts them at 1.2e-2 / 1.5e-2, DESIGN.md "Numerics").
  check         joints of the timed graph-replay path vs an eager run of the same batch (must be identical) and finite.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "cs-vit_b200"))

import torch  # noqa: E402

BATCH = 256
FLOP_PER_IMAGE = 31.15e9     # executed algorithmic FLOPs: 30.860 backbone + 0.281 head layer (K/V for 52 tokens, the rest for the 3 kept
                             # query rows; BASELINE.md §3 counts the full layer: 32.19) + 0.010
METRIC = "images/sec Swin-B spatial fwd @224^2 bs256"
# SwinV2 w16 @256 (SURVEY.md §8f-1, the shipped configuration family): 24 N C^2 + 4 L N C per block (L = 256 / 64-token windows)
# + merges + embed = 43.57 (B) / 13.20 (T) GFLOP per image; "encoder" head layer on 3 + 64 tokens.
V2_FLOP_PER_IMAGE = {"swinv2_b": 43.57e9 + 0.34e9, "swinv2_t": 13.20e9 + 0.19e9}


def image_side(variant: str) -> int:
    return 256 if variant.startswith("swinv2") else 224


def variant_table(variant: str):
    from cs_vit.synthetic import SWIN_VARIANTS, SWINV2_VARIANTS
    return SWINV2_VARIANTS[variant] if variant in SWINV2_VARIANTS else SWIN_VARIANTS[variant]


def metric_name(variant: str) -> str:
    return METRIC if variant == "swin_b" else f"images/sec {variant} spatial fwd @{image_side(variant)}^2"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--precision", choices=["bf16", "fp16"], default="fp16")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--variant", default="swin_b")
    ap.add_argument("--workload", choices=["spatial", "temporal", "finetune"], default="spatial",
                    help="spatial = BASELINE configs[1] (headline); temporal = configs[2]: 8-frame clips, realtime cross-frame attention; "
                         "finetune = configs[3]: forward + backward + AdamW step, batch 32/GPU, gradient allreduce over NCCL")
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--cpu-sample", type=int, default=16, help="images per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip roofline / e2e / fp16 passes (debug)")
    ap.add_argument("--latent-layers", type=int, default=0, help="finetune workload: num_latent_layer of the 'ti' configurations "
                    "(spatial_dexycb_swinb_spenc_addpat_ti ships 3); 0 = no latent consistency branch")
    ap.add_argument("--micro-batch", type=int, default=-1, help="images per backbone pass (L2-resident chunks); -1 = library default, 0 = whole batch")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels one by one instead of replaying a CUDA graph")
    ap.add_argument("--comm", choices=["auto", "symm", "nccl"], default="auto", help="finetune gradient transport: this library's "
                    "allreduce kernel over symmetric memory (symm; auto picks it under NCCL groups) or NCCL all_reduce")
    ap.add_argument("--no-finetune-record", action="store_true", help="spatial workload: skip the compact finetune sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (rank 0; "
                    "float32 / float64, at most 64 MB in all) so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    return a


DUMP_BYTES = 64_000_000


def dump_outputs(path: str, arrays) -> None:
    """``path/<name>.npy`` for every tensor of ``arrays``, as float32 (float64 stays float64).  A tensor larger than its even
    share of DUMP_BYTES is written as every k-th of its flattened elements (k fixed by the size): the same positions in every run."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    share = (DUMP_BYTES - 4096) // len(arrays)      # 4096: room for the .npy headers
    for name, t in arrays.items():
        t = t.detach()
        t = t.double() if t.dtype == torch.float64 else t.float()
        keep = share // t.element_size()
        if t.numel() > keep:
            t = t.reshape(-1)[::-(-t.numel() // keep)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_rate(variant: str, sample: int, steps: int, warmup: int):
    """Reference algorithm on the host cores: HF ``SwinModel`` (the third-party code the reference's backbone
    call executes) + the restated CS-ViT head from oracle/, fp32, inference mode, all available threads."""
    sys.path.insert(0, ROOT)
    from cs_vit.net import Poser
    from cs_vit.synthetic import SWIN_VARIANTS, make_inputs, make_random_backbone_dir, randomize_head_
    from cs_vit.utils.mano_standin import SyntheticMANO
    from oracle import head_restated as head

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    tmp = tempfile.mkdtemp(prefix="csvit_bench_cpu_")
    S = image_side(variant)
    bdir = make_random_backbone_dir(os.path.join(tmp, variant), variant, seed=0, image_size=S)
    torch.manual_seed(0)
    model = Poser(bdir, image_size=S, mano_layer=SyntheticMANO(), spatial_layer_type="encoder", persp_decorate="patch")
    randomize_head_(model)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    _, depths, heads = variant_table(variant)
    opt = head.HeadOptions(num_heads=heads[-1], depths=depths, swin_heads=heads, spatial_layer_type="encoder",
                           persp_decorate="patch", phase="spatial")
    features_fn, kind_note = None, "oracle restatement of HF Swin"
    if variant.startswith("swinv2"):
        from oracle import swinv2_restated as v2r
        bsd = {k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")}
        _mean = torch.tensor(head.IMAGENET_MEAN)[None, :, None, None]
        _std = torch.tensor(head.IMAGENET_STD)[None, :, None, None]
        features_fn = lambda x: v2r.swinv2_forward((x - _mean) / _std, bsd, depths, heads, window=16)  # noqa: E731
        kind_note = "oracle restatement of HF Swinv2"
    try:
        import transformers
        hf = transformers.AutoModel.from_pretrained(bdir).eval()
        mean = torch.tensor(head.IMAGENET_MEAN)[None, :, None, None]
        std = torch.tensor(head.IMAGENET_STD)[None, :, None, None]
        features_fn = lambda x: hf((x - mean) / std).last_hidden_state  # noqa: E731
        kind_note = f"HF transformers {transformers.__version__} {type(hf).__name__}"
    except Exception:
        pass
    inputs = make_inputs(sample, 1, S, seed=0)
    mano = SyntheticMANO()
    times = []
    with torch.inference_mode():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            head.predict_batch(inputs, sd, opt, mano, features_fn=features_fn, execute_all=True)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    ms = 1e3 * statistics.median(times)
    return sample / (ms / 1e3), ms, threads, f"{sample} images/step, fp32, {kind_note} + restated head (6 layers executed), torch {torch.__version__}"


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warm, steps = a.warmup, a.steps
    rate, ms, threads, note = cpu_reference_rate(a.variant, a.cpu_sample, steps, warm)
    print(json.dumps({
        "impl": "reference", "metric": metric_name(a.variant), "value": round(rate, 3), "unit": "images/s", "n_gpus": a.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": round(ms, 2), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": f"{a.variant} spatial model (encoder head, addpat) forward, CPU sample of {a.cpu_sample} images"},
        "cpu_baseline": {"value": round(rate, 3), "unit": "images/s", "cores": threads, "kind": "port", "sample": note},
        "e2e": {"value": round(rate, 3), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        sm, mx, reasons = [], 0.0, set()
        for t, line in self.rows:
            if t0 <= t <= t1:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[0])); mx = max(mx, float(f[1]))
                except (ValueError, IndexError):
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}

    def stop(self):
        if self.proc:
            self.proc.terminate()


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p["bf16_tflops_sustained"], p["hbm_gbs"], "measured"
    except Exception:
        return 1400.0, 6650.0, "fallback"


def kernel_traffic(a, key, field="traffic_bytes_per_launch"):
    """DRAM bytes per launch of a kernel group ("gemm", "attn_core", "attn_fused") from the committed ncu capture of this exact workload
    (profiles/r2_dram_traffic.json, tools/dram_traffic.py); None for any other workload / variant / batch.  field="tensor_pipe_pct":
    ncu's sm__pipe_tensor_cycles_active of one launch of that kernel (profiles/r2_ncu_attention_key_metrics.txt) - a committed
    capture, not a number measured by this run (ncu cannot run inside a timed region)."""
    if a.variant != "swin_b" or a.workload != "spatial" or a.batch != BATCH:
        return None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_dram_traffic.json")) as f:
            return json.load(f)[key].get(field)
    except Exception:
        return None


def run_ours(a):
    import torch.distributed as dist
    from cs_vit import ops
    from cs_vit.net import Poser
    from cs_vit.synthetic import make_inputs, make_random_backbone_dir, randomize_head_
    from cs_vit.utils.mano_standin import SyntheticMANO

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl ours) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    tmp = tempfile.mkdtemp(prefix=f"csvit_bench_{rank}_")
    S = image_side(a.variant)
    bdir = make_random_backbone_dir(os.path.join(tmp, a.variant), a.variant, seed=0, image_size=S)
    torch.manual_seed(0)
    temporal = a.workload == "temporal"
    T = a.frames if temporal else 1
    clips = a.batch // T                      # same number of images per GPU in both workloads
    model = Poser(bdir, image_size=S, mano_layer=SyntheticMANO(), spatial_layer_type="encoder", persp_decorate="patch",
                  precision=a.precision, temporal_supervision="realtime" if temporal else "full",
                  temporal_init_method="random" if temporal else "zero")
    randomize_head_(model)
    model.phase(Poser.TrainingPhase.INFERENCE if temporal else Poser.TrainingPhase.SPATIAL)
    model.eval()
    model = model.to(dev)
    if a.micro_batch >= 0:
        model.backbone.micro_batch = a.micro_batch

    host = make_inputs(clips, T, S, seed=100 + rank)
    flop_per_image = V2_FLOP_PER_IMAGE.get(a.variant, FLOP_PER_IMAGE)
    keys = ("patches", "square_bboxes", "timestamp", "focal", "princpt")
    pinned = {k: host[k].pin_memory() for k in keys}
    resident = {k: pinned[k].to(dev) for k in keys}

    from cs_vit.graph import GraphedPredict

    def eager_step(inp):
        with torch.no_grad():
            return model.predict_batch(inp["patches"], inp["square_bboxes"], inp["timestamp"], inp["focal"], inp["princpt"])

    graphs = {}

    def step(inp, slot=0):
        """One predict_batch; replays a captured CUDA graph (one per input-buffer slot and precision)."""
        if a.no_graph:
            return eager_step(inp)
        key = (model.precision, slot)
        if key not in graphs:
            graphs[key] = GraphedPredict(model, inp)
        return graphs[key](inp["patches"], inp["square_bboxes"], inp["timestamp"], inp["focal"], inp["princpt"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n0 = ops.launch_count
    eager_step(resident)
    launches_per_step = ops.launch_count - n0

    def timed_loop(steps, fn=None):
        """K steps on device-resident inputs, CUDA events, max over ranks.  Returns (ms_total, launches, last step's outputs)."""
        fn = fn or step
        barrier()
        n0 = ops.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = fn(resident)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return ms.item(), max(ops.launch_count - n0, launches_per_step * steps), res

    if not a.no_graph:      # the capture (and its own warm-up runs) stays out of the timed window, also with --warmup 0
        graphs[(model.precision, 0)] = GraphedPredict(model, resident)
    for _ in range(a.warmup):
        step(resident)
    sampler = ClockSampler(local) if rank == 0 else None
    t0 = time.perf_counter()
    ms_total, launches, last = timed_loop(a.steps)
    t1 = time.perf_counter()
    clocks = sampler.window(t0, t1) if sampler else None
    if a.dump_outputs and rank == 0:      # now: the graph's output buffers are overwritten by the passes below
        dump_outputs(a.dump_outputs, last)
    del last
    value = world * a.batch * a.steps / (ms_total / 1e3)
    peak_tf, peak_gbs, peak_kind = peaks()

    out = {
        "metric": metric_name(a.variant), "value": round(value, 1), "unit": "images/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": round(ms_total / a.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": a.precision, "data": "synthetic",
        "config": {"workload": (f"{a.variant} temporal model (realtime cross-frame attention), {clips} clips x {T} frames/GPU, {S}x{S}"
                                if temporal else
                                f"{a.variant} spatial model (encoder head, addpat, dense persp) predict_batch, batch {a.batch}/GPU, {S}x{S}, T=1"),
                   "global_batch": a.batch * world, "parallelism": f"dp{world}",
                   "l2_policy": "per-step inputs (154 MB) and activations (>1 GB) exceed the 126 MB L2; no explicit flush",
                   "operands": f"{a.precision} tensor-core operands, fp32 accumulate/residual/LN/softmax, TF32 head",
                   "launch": "eager" if a.no_graph else "CUDA graph replay of the step"},
        "gpu_launches": launches,
        "model_flops_frac_of_peak": round(value / world * flop_per_image / (peak_tf * 1e12), 4),
        "clocks": clocks,
    }

    if not a.no_extras:
        # ---- roofline of the dominant kernel (GEMM engine), instrumented pass over the same K steps ----------
        ops.begin_profile("csvit_linear")
        timed_loop(a.steps, eager_step)      # per-launch events need individual launches (no graph replay)
        prof = ops.end_profile()
        if prof["launches"]:
            def tc_block(pr, kernel, traffic, tpipe=None):
                ach = pr["flops"] / (pr["ms"] / 1e3) / 1e12
                return {"bound": "tensor", "kernel": kernel, "achieved": round(ach, 1), "peak": peak_tf, "unit": "TFLOP/s",
                        "frac": round(ach / peak_tf, 4), "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peak_kind})",
                        "traffic": traffic, "tensor_pipe_pct_ncu": tpipe, "launches_per_step": pr["launches"] // a.steps,
                        "share_of_step": round(pr["ms"] / a.steps / (ms_total / a.steps), 3),
                        "avg_launch_us": round(1e3 * pr["ms"] / pr["launches"], 2)}
            pair = prof.get("kind1")
            if pair and pair["launches"]:
                # the dominant kernel: gemm_pair_kernel (CTA pairs, cta_group::2) - the launches csvit_linear routed to it
                out["roofline"] = tc_block(pair, "gemm_pair_kernel (tcgen05.mma.cta_group::2, 256x256 tiles): the large Linears of the backbone", kernel_traffic(a, "gemm_pair"),
                                           kernel_traffic(a, "gemm_pair", "tensor_pipe_pct"))
                out["roofline_all_linear"] = tc_block(prof, "csvit_linear, every launch: gemm_pair_kernel + gemm_tc_kernel (small / odd shapes, memory-bound "
                                                            "stage-0 shapes, the TF32 head)", kernel_traffic(a, "gemm"))
            else:
                out["roofline"] = tc_block(prof, "csvit_linear: gemm_tc_kernel / gemm_pair_kernel", kernel_traffic(a, "gemm"))
        # ---- the tcgen05 window-attention kernels (HBM-bound), same instrumented pass -------------------------------
        for key, entry, kern, bpt, tkey in (
                ("roofline_attention", "csvit_swin_attn_core", "swin_attn_core_kernel: q/k/v tiles by TMA, QK^T and PV on tcgen05/TMEM (stages 2-3)", "8C", "attn_core"),
                ("roofline_attention_fused", "csvit_swin_attn_fused", "swin_attn_fused_kernel: LN + QKV + attention in one tcgen05 kernel (stages 0-1)", "6C", "attn_fused")):
            ops.begin_profile(entry)
            timed_loop(a.steps, eager_step)
            prof = ops.end_profile()
            if prof["launches"]:
                gbs = prof["bytes"] / (prof["ms"] / 1e3) / 1e9
                out[key] = {"bound": "hbm", "kernel": kern, "achieved": round(gbs, 1), "peak": peak_gbs, "unit": "GB/s",
                            "frac": round(gbs / peak_gbs, 4), "algorithmic_bytes_per_token": bpt, "traffic": kernel_traffic(a, tkey),
                            "tensor_pipe_pct_ncu": kernel_traffic(a, tkey, "tensor_pipe_pct"),
                            "tflops": round(prof["flops"] / (prof["ms"] / 1e3) / 1e12, 1),
                            "launches_per_step": prof["launches"] // a.steps,
                            "share_of_step": round(prof["ms"] / a.steps / (ms_total / a.steps), 3),
                            "avg_launch_us": round(1e3 * prof["ms"] / prof["launches"], 2)}
        # ---- the timed path's result against an eager run of the same batch --------------------------------------
        g_out = step(resident)["joint_cam"].clone()
        e_out = eager_step(resident)["joint_cam"]
        torch.cuda.synchronize()
        out["check"] = {"joint_cam_finite": bool(torch.isfinite(g_out).all().item()),
                        "graph_vs_eager_max_abs_diff": float((g_out - e_out).abs().max().item())}
        # ---- end-to-end: host inputs, H2D + D2H inside the timed region, double-buffered ------------------------
        copy_stream = torch.cuda.Stream(device=dev)
        bufs = [{k: torch.empty_like(resident[k]) for k in keys} for _ in range(2)]
        host_out = torch.empty(clips, 1, 21, 3).pin_memory()
        h2d = sum(pinned[k].numel() * pinned[k].element_size() for k in keys)

        def e2e_loop(steps):
            barrier()
            main = torch.cuda.current_stream()
            ready = [torch.cuda.Event(), torch.cuda.Event()]
            freed = [torch.cuda.Event(), torch.cuda.Event()]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()

            def upload(i):
                with torch.cuda.stream(copy_stream):
                    if i >= 2:
                        copy_stream.wait_event(freed[i % 2])
                    for k in keys:
                        bufs[i % 2][k].copy_(pinned[k], non_blocking=True)
                    ready[i % 2].record(copy_stream)

            copy_stream.wait_event(e0)
            upload(0)
            for i in range(steps):
                if i + 1 < steps:
                    upload(i + 1)
                main.wait_event(ready[i % 2])
                res = step(bufs[i % 2], slot=1 + i % 2)
                host_out.copy_(res["joint_cam"], non_blocking=True)
                freed[i % 2].record(main)
            e1.record()
            torch.cuda.synchronize()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return ms.item()

        e2e_loop(2)
        ms_e2e = e2e_loop(a.steps)
        out["e2e"] = {"value": round(world * a.batch * a.steps / (ms_e2e / 1e3), 1), "unit": "images/s",
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": host_out.numel() * 4,
                      "note": "predict_batch on pinned host tensors; H2D on a copy stream overlapped with the previous step's compute; "
                              "D2H returns joint_cam only (what scripts/eval.py consumes) - the other five result tensors stay on the device"}
        # ---- the other 16-bit operand format ---------------------------------------------------------------
        other = "fp16" if a.precision == "bf16" else "bf16"
        model.set_precision(other)
        for _ in range(2):
            step(resident)
        ms_o, _, _ = timed_loop(a.steps)
        out[other] = {"value": round(world * a.batch * a.steps / (ms_o / 1e3), 1), "unit": "images/s",
                      "ms_per_step": round(ms_o / a.steps, 3)}
        model.set_precision(a.precision)

    if sampler:
        sampler.stop()
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        rate, ms, threads, note = cpu_reference_rate(a.variant, a.cpu_sample, 2, 1)
        out["cpu_baseline"] = {"value": round(rate, 3), "unit": "images/s", "cores": threads, "kind": "port", "sample": note}
    if not a.no_extras and not a.no_finetune_record and not temporal and a.variant == "swin_b":
        # ---- configs[3] beside the headline, so that the driver's 1/2/4/8-GPU scaling record carries it: the graphed finetune
        # step at batch 32/GPU with the gradient allreduce (the one collective on this target's data path)
        del model, graphs, resident, pinned
        torch.cuda.empty_cache()
        fa = argparse.Namespace(**vars(a))
        fa.batch = 32
        ft = finetune_measure(fa, world, rank, local, dev, steps=min(a.steps, 10), warmup=2, comm=a.comm, split=False)
        out["finetune"] = {k: ft[k] for k in ("metric", "value", "unit", "ms_per_step", "n_gpus", "steps", "skipped_steps",
                                              "ms_per_step_without_allreduce", "allreduce_ms_exposed") if k in ft}
        out["finetune"]["allreduce"] = ft["config"]["allreduce"]
        out["finetune"]["launch"] = ft["config"]["launch"]
    if rank == 0:
        print(json.dumps(out), flush=True)
    hard_exit_if_distributed(world)


def finetune_measure(a, world, rank, local, dev, steps, warmup, comm="auto", split=True, dump=None):
    """BASELINE configs[3]: Swin-B spatial finetune step (ref:scripts/finetune.py:211-227), per-GPU batch 32 (the reference's
    value, SURVEY.md §6), data-parallel: the gradient buckets are reduced by cs_vit/train.py::GradReducer (this library's
    allreduce kernel over symmetric memory, or NCCL with --comm nccl) overlapped with backward.  Returns the result dict;
    ``dump``: directory for dump_outputs() of the last timed step."""
    import torch.distributed as dist
    from cs_vit import ops
    from cs_vit.net import Poser
    from cs_vit.synthetic import make_inputs, make_random_backbone_dir, randomize_head_
    from cs_vit.train import GradReducer, GraphedFinetuneStep, broadcast_parameters, finetune_step, scaled_lr
    from cs_vit.utils.mano_standin import SyntheticMANO

    B = a.batch if a.batch != BATCH else 32
    tmp = tempfile.mkdtemp(prefix=f"csvit_bench_ft_{rank}_")
    S = image_side(a.variant)
    bdir = make_random_backbone_dir(os.path.join(tmp, a.variant), a.variant, seed=0, image_size=S)
    torch.manual_seed(0)
    model = Poser(bdir, image_size=S, mano_layer=SyntheticMANO(), spatial_layer_type="encoder", persp_decorate="patch",
                  precision=a.precision, num_latent_layer=a.latent_layers or None)
    randomize_head_(model)
    model.phase(Poser.TrainingPhase.SPATIAL)          # train mode: batch-statistics BatchNorm, trainable spatial modules
    model = model.to(dev)
    broadcast_parameters(model)
    trainable = [p for p in model.parameters() if p.requires_grad]
    reducer = GradReducer(trainable, comm=comm)
    graphed = not a.no_graph
    opt = torch.optim.AdamW(trainable, lr=scaled_lr(1e-5, world, B), fused=True, capturable=graphed)
    batch = {k: v.to(dev) for k, v in make_inputs(B, 1, S, seed=100 + rank, labels=True).items()}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    losses = []
    gstep = None
    if graphed:      # the whole step (forward, loss, backward, reduction, clip, AdamW) replayed as one CUDA graph
        gstep = GraphedFinetuneStep(model, batch, opt, reducer, warmup=max(warmup, 2))
        run_step = lambda: gstep(batch).clone()      # noqa: E731
    else:
        run_step = lambda: finetune_step(model, batch, opt, reducer)      # noqa: E731
        for _ in range(max(warmup, 2)):              # step 1 also learns the bucket order
            losses.append(run_step().item())
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    n0 = ops.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        last = run_step()
        losses.append(last)
    e1.record()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    if dump and rank == 0:      # the step returns the loss; its product is the updated parameters
        dump_outputs(dump, {"loss": last, "trainable_params": torch.cat([p.detach().reshape(-1) for p in trainable])})
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches = ops.launch_count - n0
    if gstep is not None:
        launches = gstep.launches_per_step * steps       # graph replays: the captured C-ABI launches of one step, per replay
    nparams = sum(p.numel() for p in trainable)
    value = world * B * steps / (ms.item() / 1e3)
    peak_tf, _, _ = peaks()
    res = {
        "metric": ("images/sec Swin-B" if a.variant == "swin_b" else f"images/sec {a.variant}") + f" spatial finetune step (fwd+bwd+AdamW) bs{B}/GPU",
        "value": round(value, 1), "unit": "images/s",
        "n_gpus": world, "steps": steps, "warmup": max(warmup, 2), "ms_per_step": round(ms.item() / steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": a.precision, "data": "synthetic",
        "config": {"launch": "one CUDA graph per step (cs_vit.train.GraphedFinetuneStep)" if graphed else "eager",
                   "workload": f"{a.variant} spatial model finetune step (Poser.forward loss, backward, grad clip 5.0, fused AdamW), "
                               f"batch {B}/GPU, {S}x{S}, train-mode BatchNorm"
                               + (f", latent consistency branch with {a.latent_layers} layers ('ti' configuration)" if a.latent_layers else ""),
                   "global_batch": B * world, "parallelism": f"dp{world}",
                   "allreduce": f"{nparams * 4 / 1e6:.1f} MB fp32 gradients in {len(reducer.bucket_summary())} flat buckets, reduced from "
                                f"grad-ready hooks on a side stream; transport: {reducer.transport}",
                   "operands": f"{a.precision} tensor-core operands forward and backward, fp32 accumulate / gradients / optimizer"},
        "gpu_launches": launches,
        "model_flops_frac_of_peak": round(3 * value / world * FLOP_PER_IMAGE / (peak_tf * 1e12), 4),
        "skipped_steps": gstep.skipped_steps if gstep is not None else None,
        "losses": [round(float(x), 3) for x in losses],
        "clocks": sampler.window(t0, t1) if sampler else None,
    }
    if sampler:
        sampler.stop()
    if world > 1 and graphed:
        # exposed communication = this step minus the same graphed step with the reduction switched off (local gradients only)
        reducer.remove()
        local_red = GradReducer(trainable, comm="nccl")
        local_red.world = 1
        lstep = GraphedFinetuneStep(model, batch, opt, local_red, warmup=2)
        barrier()
        e0.record()
        for _ in range(steps):
            lstep(batch)
        e1.record()
        torch.cuda.synchronize()
        ms_l = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms_l, op=dist.ReduceOp.MAX)
        res["ms_per_step_without_allreduce"] = round(ms_l.item() / steps, 3)
        res["allreduce_ms_exposed"] = round((ms.item() - ms_l.item()) / steps, 3)
        del lstep
    elif split:
        # forward / backward split of one more (eager) step (events, not part of the timed region)
        from cs_vit.train import invalidate_packs
        invalidate_packs(model)
        reducer.zero_grad()
        model.loss_tensors(batch)[0].backward()      # untimed: re-packs the weights for the eager path
        reducer.finish()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        reducer.zero_grad()
        ev[0].record()
        eager_loss, _, _ = model.loss_tensors(batch)
        ev[1].record()
        eager_loss.backward()
        reducer.finish()
        ev[2].record()
        torch.cuda.synchronize()
        res["eager_forward_ms"] = round(ev[0].elapsed_time(ev[1]), 3)
        res["eager_backward_ms"] = round(ev[1].elapsed_time(ev[2]), 3)
    del gstep, run_step
    return res


def hard_exit_if_distributed(world):
    """A replayable graph that holds captured communication work must be gone before the communicator is torn down (otherwise
    destroy_process_group can wait forever); after the final barrier a hard exit is the robust teardown."""
    import torch.distributed as dist
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


def run_finetune(a):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl ours) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    res = finetune_measure(a, world, rank, local, dev, a.steps, a.warmup, comm=a.comm, dump=a.dump_outputs)
    if rank == 0:
        print(json.dumps(res), flush=True)
    hard_exit_if_distributed(world)


def main():
    a = parse()
    if a.impl == "reference":
        run_reference_arm(a)
    elif a.workload == "finetune":
        run_finetune(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
