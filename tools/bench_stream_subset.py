"""Streaming sessions that step a subset of their streams (``step(..., streams=ids)``): cost against the number of frames, an
unsynchronised-camera trace, and the state-update kernel.

    python tools/bench_stream_subset.py [--out FILE] [--steps K] [--reps R] [--cases swinv2_b:256,swin_b:224] [--trace-ticks N]

The model is the temporal model of ``tools/bench_stream.py``: "encoder" spatial head, perspective embedding added to the patches,
random temporal init, ``randomize_head_``, fp16 backbone operands, window 8, graphed sessions; the realtime model and the full
model at lag 0.  For each backbone (SwinV2-B at 256², Swin-B at 224²) and model:

  1. step time against n   A session of capacity 1024 and max_batch 256 steps the same n of its streams every step, for n in
                           {1, 8, 32, 64, 128, 256}; a lockstep session of ``bucket(n)`` streams steps all of them, its first n
                           rows carrying the same frames.  The two arms alternate R times (CUDA events over K steps).  The largest
                           output difference between their n rows is reported (the contract makes it 0).
  2. arrival trace         300 cameras at 30 fps with random phase and 5 % of the frames dropped, served at 120 Hz ticks: each tick
                           steps the streams whose frame arrived since the last tick.  Baseline: graphed ``predict_batch`` (one
                           ``GraphedPredict`` per bucket) on each arriving stream's last 8 frames.  Ticks run back to back (GPU
                           throughput, not paced in real time); the first ticks fill every stream's window untimed, the next ones
                           compare the two arms' outputs, then the arms alternate R times over the same timed ticks.
  3. state-update kernel   ``ops.stream_update`` at capacity 1024, nb = 256 distinct streams with saturated histories, D = 1024
                           (SwinV2-B / Swin-B width), once per launch with L2 flushed by a 256 MB write before it; bytes moved
                           over the CUDA-event time.

The GPU's name, power limit and maximum SM clock are read in the same run, and the SM clock and power draw are sampled while each
timed loop is on the GPU.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs-vit_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

from bench_stream import KEYS, OUT_KEYS, WINDOW, build_model, smi, timed  # noqa: E402

CAPACITY, MAX_BATCH = 1024, 256
HBM_TBPS = 7.7


def _session(model, supervision: str, num_streams: int, max_batch: int):
    from cs_vit.stream import FullTemporalStream, RealtimeStream
    if supervision == "realtime":
        return RealtimeStream(model, num_streams, WINDOW, max_batch=max_batch)
    return FullTemporalStream(model, num_streams, WINDOW, lag=0, max_batch=max_batch)


def _maxdiff(a: dict, b: dict, rows: int) -> float:
    return max((a[k][:rows].double() - b[k][:rows].double()).abs().max().item() for k in OUT_KEYS)


def step_time_vs_n(model, supervision: str, side: int, ns, steps: int, reps: int):
    from cs_vit.synthetic import make_inputs
    from cs_vit.stream import bucket
    F = 4
    inp = make_inputs(MAX_BATCH, F, side, seed=100)
    frames = {k: inp[k].cuda() for k in KEYS if k != "timestamp"}
    g = torch.Generator().manual_seed(0)
    sub = _session(model, supervision, CAPACITY, MAX_BATCH)
    out = []
    for n in ns:
        nb = bucket(n, MAX_BATCH)
        ids = torch.randperm(CAPACITY, generator=g)[:n]                # the same n streams every step
        lock = _session(model, supervision, nb, nb)
        clock = {"sub": 0, "lock": 0}

        def frame(t: int, rows: int):
            f = {k: v[:rows, t % F] for k, v in frames.items()}
            f["timestamp"] = torch.full((rows,), 33.333 * t, device="cuda")
            return [f[k] for k in KEYS]

        def step_sub():
            clock["sub"] += 1
            return sub.step(*frame(clock["sub"], n), streams=ids)

        def step_lock():
            clock["lock"] += 1
            f = frame(clock["lock"], nb)
            if nb > n:                                  # rows n.. carry row 0's frame, as the subset session's padding rows do
                f = [torch.cat([x[:n], x[:1].expand((nb - n,) + x.shape[1:])]) for x in f]
            return lock.step(*f)

        # the subset arm's streams start where the previous n left them: reset them on their first step here
        sub.step(*frame(0, n), reset=torch.ones(n, dtype=torch.bool, device="cuda"), streams=ids)
        lock.step(*[torch.cat([x[:n], x[:1].expand((nb - n,) + x.shape[1:])]) if nb > n else x for x in frame(0, nb)],
                  reset=torch.ones(nb, dtype=torch.bool, device="cuda"))
        for _ in range(WINDOW + 2):
            step_sub()
            step_lock()
        diff = 0.0
        for _ in range(3):
            a = {k: v.clone() for k, v in step_sub().items()}
            diff = max(diff, _maxdiff(a, step_lock(), n))
        runs = {"subset": [], "lockstep": []}
        for _ in range(reps):
            for arm, fn in (("subset", step_sub), ("lockstep", step_lock)):
                ms, sample = timed(fn, steps)
                runs[arm].append({"ms_per_step": round(ms, 3), "sm_clock_and_power_during": sample})
        best = {arm: min(r["ms_per_step"] for r in v) for arm, v in runs.items()}
        row = {"n": n, "bucket": nb, "subset_capacity_1024": runs["subset"], "lockstep_num_streams_bucket": runs["lockstep"],
               "best_ms_subset": best["subset"], "best_ms_lockstep": best["lockstep"],
               "subset_over_lockstep": round(best["subset"] / best["lockstep"], 4), "max_abs_diff_between_arms": diff}
        print(json.dumps(row), flush=True)
        out.append(row)
        del lock
        torch.cuda.empty_cache()
    del sub
    torch.cuda.empty_cache()
    return out


def make_trace(cameras: int, ticks: int, seed: int):
    """Per tick: the cameras whose frame arrived in (t - 1/120 s, t], with each camera's received-frame index and timestamp (ms).
    30 fps per camera with a random phase, 5 % of the frames dropped."""
    g = torch.Generator().manual_seed(seed)
    phase = torch.rand(cameras, generator=g) / 30.0
    received = [0] * cameras
    per_tick = []
    frame_no = [0] * cameras
    for k in range(ticks):
        t0, t1 = k / 120.0, (k + 1) / 120.0
        arrivals = []
        for c in range(cameras):
            while phase[c].item() + frame_no[c] / 30.0 < t1:
                t_frame = phase[c].item() + frame_no[c] / 30.0
                frame_no[c] += 1
                if t_frame < t0 or torch.rand(1, generator=g).item() < 0.05:
                    continue
                arrivals.append((c, received[c], 1000.0 * t_frame))
                received[c] += 1
        order = torch.randperm(len(arrivals), generator=g).tolist()         # arrival order within a tick is arbitrary
        per_tick.append([arrivals[i] for i in order])
    return per_tick


def arrival_trace(model, supervision: str, side: int, ticks: int, steps_warm: int, steps_check: int, reps: int):
    from cs_vit.graph import GraphedPredict
    from cs_vit.stream import bucket
    from cs_vit.synthetic import make_inputs
    cameras, F = 300, 12
    trace = make_trace(cameras, ticks, seed=1)
    inp = make_inputs(cameras, F, side, seed=101)
    video = {k: inp[k].flatten(0, 1).cuda() for k in KEYS if k != "timestamp"}         # camera c, frame j -> row c * F + j % F
    stamps = {}                                                                         # (camera, received index) -> ms
    for arr in trace:
        for c, j, ms in arr:
            stamps[(c, j)] = ms
    timed_ticks = ticks - steps_warm - steps_check
    assert timed_ticks > 0
    first_timed = steps_warm + steps_check
    for arr in trace[steps_warm:]:
        assert all(j >= WINDOW - 1 for _, j, _ in arr), "every camera must have a full window once the warm-up ticks are over"
    hist_buckets = {}
    for arr in trace[first_timed:]:
        b = bucket(len(arr), MAX_BATCH)
        hist_buckets[b] = hist_buckets.get(b, 0) + 1
    # device-side per-tick operands, built before any timing
    ops_tick = []
    for arr in trace:
        n = len(arr)
        nb = bucket(n, MAX_BATCH) if n else 0
        cams = [c for c, _, _ in arr]
        rows = torch.tensor([c * F + j % F for c, j, _ in arr], dtype=torch.long)
        clip = torch.tensor([[c * F + (j - WINDOW + 1 + i) % F for i in range(WINDOW)] for c, j, _ in arr], dtype=torch.long).reshape(-1, WINDOW)
        clip_ts = torch.tensor([[stamps.get((c, j - WINDOW + 1 + i), 0.0) for i in range(WINDOW)] for c, j, _ in arr]).reshape(-1, WINDOW)
        if nb > n:                                   # padding rows of the sliding arm: copies of row 0
            clip = torch.cat([clip, clip[:1].expand(nb - n, WINDOW)])
            clip_ts = torch.cat([clip_ts, clip_ts[:1].expand(nb - n, WINDOW)])
        ops_tick.append({"ids": torch.tensor(cams, dtype=torch.long), "n": n, "nb": nb, "rows": rows.cuda(),
                         "ts": torch.tensor([ms for _, _, ms in arr], dtype=torch.float32).cuda(), "clip": clip.cuda(), "clip_ts": clip_ts.cuda()})
    session = _session(model, supervision, CAPACITY, MAX_BATCH)
    sliding = {}

    def step_session(op):
        if op["n"] == 0:
            return session.step(*[video[k][:0] if k != "timestamp" else op["ts"] for k in KEYS], streams=[])
        f = {k: video[k].index_select(0, op["rows"]) for k in video}
        f["timestamp"] = op["ts"]
        return session.step(*[f[k] for k in KEYS], streams=op["ids"])

    def step_sliding(op):
        if op["n"] == 0:
            return None
        nb = op["nb"]
        if nb not in sliding:
            ex = {k: video[k].index_select(0, op["clip"].flatten()).unflatten(0, (nb, WINDOW)) for k in video}
            ex["timestamp"] = op["clip_ts"]
            sliding[nb] = GraphedPredict(model, ex)
        gp = sliding[nb]
        for k in video:
            torch.index_select(video[k], 0, op["clip"].flatten(), out=gp.static_in[k].view(nb * WINDOW, *video[k].shape[1:]))
        gp.static_in["timestamp"].copy_(op["clip_ts"])
        return gp(*(gp.static_in[k] for k in KEYS))

    # capture every bucket of the trace in both arms before timing: the session on streams the trace never uses
    spare = torch.arange(cameras, CAPACITY)
    for nb in sorted({op["nb"] for op in ops_tick if op["nb"]}):
        f = {k: video[k][:1].expand((nb,) + video[k].shape[1:]).contiguous() for k in video}
        f["timestamp"] = torch.zeros(nb, device="cuda")
        session.step(*[f[k] for k in KEYS], streams=spare[:nb])
        step_sliding(next(op for op in ops_tick if op["nb"] == nb))
    for op in ops_tick[:steps_warm]:
        step_session(op)
    diff, compared = 0.0, 0
    frame_sel = slice(None) if supervision == "realtime" else slice(WINDOW - 1, WINDOW)
    for op in ops_tick[steps_warm:first_timed]:
        a = {k: v.clone() for k, v in step_session(op).items()}
        b = step_sliding(op)
        if b is not None:
            diff = max(diff, max((a[k].double() - b[k][:op["n"], frame_sel].double()).abs().max().item() for k in OUT_KEYS))
            compared += op["n"]
    timed_ops = ops_tick[first_timed:]
    preds = sum(op["n"] for op in timed_ops)
    runs = {"session": [], "sliding_predict_batch": []}
    for _ in range(reps):
        for arm, fn in (("session", step_session), ("sliding_predict_batch", step_sliding)):
            it = iter(timed_ops)
            ms, sample = timed(lambda: fn(next(it)), len(timed_ops))
            runs[arm].append({"ms_per_tick": round(ms, 3), "predictions_per_s": round(preds / (ms * len(timed_ops) / 1e3), 1),
                              "sm_clock_and_power_during": sample})
    best = {arm: max(v, key=lambda x: x["predictions_per_s"]) for arm, v in runs.items()}
    res = {"cameras": cameras, "fps": 30, "drop": 0.05, "tick_hz": 120, "timed_ticks": len(timed_ops),
           "frames_per_tick_mean": round(preds / len(timed_ops), 2), "bucket_histogram": dict(sorted(hist_buckets.items())),
           "runs": runs, "best": {arm: {k: v[k] for k in ("ms_per_tick", "predictions_per_s")} for arm, v in best.items()},
           "speedup": round(best["session"]["predictions_per_s"] / best["sliding_predict_batch"]["predictions_per_s"], 2),
           "compared_predictions": compared, "max_abs_diff_between_arms": diff}
    print(json.dumps({k: v for k, v in res.items() if k != "runs"}), flush=True)
    del sliding, session
    torch.cuda.empty_cache()
    return res


def update_kernel(D: int = 1024, nb: int = 256, launches: int = 50):
    from cs_vit import ops
    g = torch.Generator().manual_seed(2)
    tokens = torch.randn(CAPACITY, WINDOW, 3, D, device="cuda")
    stamps = torch.randn(CAPACITY, WINDOW, device="cuda")
    hist = torch.full((CAPACITY,), WINDOW, dtype=torch.int32, device="cuda")
    head = torch.randint(0, WINDOW, (CAPACITY,), generator=g).to(torch.int32).cuda()
    tok = torch.randn(nb, 3, D, device="cuda")
    ts = torch.randn(nb, device="cuda")
    ids = [torch.randperm(CAPACITY, generator=g)[:nb].to(torch.int32).cuda() for _ in range(launches)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = {}
    for name, st, t in (("realtime", stamps, ts), ("full", None, None)):
        for i in range(3):
            ops.stream_update(tok, ids[i], None, tokens, hist, head, t, st)
        ms = []
        for i in range(launches):
            flush.fill_(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.stream_update(tok, ids[i], None, tokens, hist, head, t, st)
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        ms.sort()
        med = ms[len(ms) // 2]
        # saturated histories: read the new tokens and W - 1 stored slots, write the window and one state slot (+ the stamps)
        nbytes = 4.0 * nb * 3 * D * (1 + (WINDOW - 1) + WINDOW + 1) + 4.0 * nb * 3 + (4.0 * nb * (1 + WINDOW - 1 + WINDOW + 1) if st is not None else 0)
        res[name] = {"nb": nb, "capacity": CAPACITY, "window": WINDOW, "D": D, "bytes": nbytes, "median_us": round(1e3 * med, 2),
                     "min_us": round(1e3 * ms[0], 2), "GB_per_s": round(nbytes / (med * 1e-3) / 1e9, 1),
                     "share_of_7.7_TB_per_s": round(nbytes / (med * 1e-3) / (HBM_TBPS * 1e12), 3), "l2": "flushed before each launch"}
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_stream_subset.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--cases", default="swinv2_b:256,swin_b:224")
    ap.add_argument("--ns", default="1,8,32,64,128,256")
    ap.add_argument("--trace-ticks", type=int, default=200, help="120 Hz ticks: 60 fill the windows, 20 are compared, the rest timed")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("tools/bench_stream_subset.py needs a CUDA device: there is no CPU fallback")
    result = {"gpu": {"device": torch.cuda.get_device_name(0), "name_power_limit_max_sm_clock": smi("name,power.limit,clocks.max.sm")},
              "steps_per_timed_loop": a.steps, "alternations": a.reps, "window": WINDOW, "precision": "fp16",
              "capacity": CAPACITY, "max_batch": MAX_BATCH, "cases": []}
    result["state_update_kernel"] = update_kernel()
    ns = [int(x) for x in a.ns.split(",")]
    for c in a.cases.split(","):
        variant, side = c.split(":")
        for supervision in ("realtime", "full"):
            model = build_model(variant, int(side), supervision)
            case = {"variant": variant, "image_side": int(side), "supervision": supervision}
            if supervision == "full":
                case["lag"] = 0
            print(json.dumps(case), flush=True)
            case["step_time_vs_n"] = step_time_vs_n(model, supervision, int(side), ns, a.steps, a.reps)
            case["arrival_trace"] = arrival_trace(model, supervision, int(side), a.trace_ticks, 60, 20, a.reps)
            result["cases"].append(case)
            del model
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"out": a.out, "gpu": result["gpu"]}))


if __name__ == "__main__":
    main()
