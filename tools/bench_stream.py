"""Streaming inference of the temporal Poser: the session's ``step`` against ``predict_batch`` on sliding windows.

    python tools/bench_stream.py [--supervision realtime|full] [--lag L,...] [--out FILE] [--steps K] [--reps R]

The model is the temporal model of ``bench.py --workload temporal``: "encoder" spatial head, perspective embedding added to the
patches, random temporal init, ``randomize_head_``, fp16 backbone operands, window 8; ``--supervision`` picks the realtime
model (default) or the full one.  For Swin-B at 224² and SwinV2-B at 256², each with 32 and 256 streams, two arms are timed
with CUDA events, alternated R times in one run:

  (a) sliding   graphed ``predict_batch`` (``cs_vit.graph.GraphedPredict``) on each stream's last 8 frames: what a user of the
                temporal model does without a session.  Each step gathers the window from a device-resident video into the
                graph's static input buffer and replays the graph; 8 backbone passes per prediction.  The full model's
                prediction is its frame ``-1 - lag``.
  (b) stream    graphed ``RealtimeStream.step`` (realtime) or ``FullTemporalStream.step`` with ``lag`` (full) on each stream's
                newest frame; 1 backbone pass per prediction.

Both arms make one prediction per stream per step.  The full model is measured once per lag in ``--lag`` (default 0 and 4;
the realtime model has lag 0 only).  After the timed loops both arms run on the same frames for a few more steps and every
output key is compared (largest absolute difference; the session's contract is 0).  The GPU's name, power limit and
maximum SM clock are read in the same run, and the SM clock and power draw are sampled while each timed loop is on the GPU.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs-vit_b200"))
import torch  # noqa: E402

WINDOW = 8
KEYS = ("patches", "square_bboxes", "timestamp", "focal", "princpt")
OUT_KEYS = ("joint_cam", "verts_cam", "pose_aa", "shape", "root_transl_norm", "root_transl")


def smi(query: str) -> str:
    try:
        return subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={query}", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip()
    except Exception as e:      # noqa: BLE001
        return f"nvidia-smi unavailable: {e}"


def build_model(variant: str, side: int, supervision: str):
    from cs_vit.net import Poser
    from cs_vit.synthetic import make_random_backbone_dir, randomize_head_
    from cs_vit.utils.mano_standin import SyntheticMANO
    d = make_random_backbone_dir(os.path.join(tempfile.mkdtemp(prefix="csvit_stream_"), variant), variant, seed=0, image_size=side)
    torch.manual_seed(0)
    model = Poser(d, image_size=side, mano_layer=SyntheticMANO(), spatial_layer_type="encoder", persp_decorate="patch",
                  precision="fp16", temporal_supervision=supervision, temporal_init_method="random")
    randomize_head_(model)
    model.phase(Poser.TrainingPhase.INFERENCE)
    return model.cuda()


class Video:
    """F distinct device-resident frames per stream, played in a loop, and per-stream 30 fps timestamps for ``n_steps`` steps."""

    def __init__(self, streams: int, side: int, frames: int, n_steps: int):
        from cs_vit.synthetic import make_inputs
        inp = make_inputs(streams, frames, side, seed=100)
        self.F = frames
        self.frames = {k: inp[k].cuda() for k in ("patches", "square_bboxes", "focal", "princpt")}
        off = 1000.0 * torch.arange(streams, dtype=torch.float32)[:, None]
        self.stamps = (off + 33.333 * torch.arange(n_steps, dtype=torch.float32)[None]).cuda()
        self.idx = {}

    def clip(self, t: int, out: dict) -> None:
        """Frames t-7..t of every stream into the [B, 8, ...] buffers ``out`` (one gather per input)."""
        key = t % self.F
        if key not in self.idx:
            self.idx[key] = torch.tensor([(t - WINDOW + 1 + i) % self.F for i in range(WINDOW)], device="cuda")
        for k, v in self.frames.items():
            torch.index_select(v, 1, self.idx[key], out=out[k])
        out["timestamp"].copy_(self.stamps[:, t - WINDOW + 1:t + 1])

    def frame(self, t: int) -> dict:
        f = {k: v[:, t % self.F] for k, v in self.frames.items()}
        f["timestamp"] = self.stamps[:, t]
        return f


def timed(fn, steps: int):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    sample = smi("clocks.sm,power.draw")      # read while the enqueued steps run
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, sample


def run_case(variant: str, side: int, streams: int, steps: int, reps: int, supervision: str = "realtime", lag: int = 0):
    from cs_vit.graph import GraphedPredict
    from cs_vit.stream import FullTemporalStream, RealtimeStream
    model = build_model(variant, side, supervision)
    n_steps = WINDOW + 8 + (reps + 1) * steps + 16
    video = Video(streams, side, frames=12, n_steps=n_steps)
    clip = {k: torch.empty(streams, WINDOW, *v.shape[2:], dtype=v.dtype, device="cuda") for k, v in video.frames.items()}
    clip["timestamp"] = torch.empty(streams, WINDOW, device="cuda")
    video.clip(WINDOW - 1, clip)
    sliding = GraphedPredict(model, clip)
    for k in KEYS:                     # the gather writes straight into the graph's input buffers
        clip[k] = sliding.static_in[k]
    if supervision == "realtime":
        session = RealtimeStream(model, streams, WINDOW)
    else:
        session = FullTemporalStream(model, streams, WINDOW, lag=lag)
    # the sliding arm's output frame that the session's step returns (the realtime model outputs the newest frame only)
    frame_a = slice(None) if supervision == "realtime" else slice(WINDOW - 1 - lag, WINDOW - lag)
    clock = {"a": WINDOW - 1, "b": 0}

    def step_a():
        video.clip(clock["a"], clip)
        clock["a"] += 1
        return sliding(*(clip[k] for k in KEYS))

    def step_b():
        f = video.frame(clock["b"])
        clock["b"] += 1
        return session.step(*(f[k] for k in KEYS))

    for _ in range(WINDOW + 2):        # capture + fill every stream's window; a few sliding steps to warm up
        step_b()
    for _ in range(3):
        step_a()
    res = {"a": [], "b": []}
    for _ in range(reps):
        for arm, fn in (("a", step_a), ("b", step_b)):
            ms, sample = timed(fn, steps)
            res[arm].append({"ms_per_step": round(ms, 3), "predictions_per_s": round(streams / (ms / 1e3), 1),
                             "sm_clock_and_power_during": sample})
    # the same frames through both arms: stream b's newest frame is frame clock_b - 1; run the sliding arm on that window
    maxdiff = {k: 0.0 for k in OUT_KEYS}
    for _ in range(3):
        ob = {k: v.clone() for k, v in step_b().items()}
        clock["a"] = clock["b"] - 1
        oa = step_a()
        for k in OUT_KEYS:
            maxdiff[k] = max(maxdiff[k], (oa[k][:, frame_a].double() - ob[k].double()).abs().max().item())
    torch.cuda.synchronize()
    best = {arm: max(r, key=lambda x: x["predictions_per_s"]) for arm, r in res.items()}
    out = {"variant": variant, "image_side": side, "streams": streams, "window": WINDOW, "precision": "fp16"}
    if supervision != "realtime":
        out.update(supervision=supervision, lag=lag)
    out.update({"sliding_predict_batch": {"runs": res["a"], "best_predictions_per_s": best["a"]["predictions_per_s"],
                                          "best_ms_per_step": best["a"]["ms_per_step"], "backbone_images_per_step": streams * WINDOW},
                f"{supervision}_stream": {"runs": res["b"], "best_predictions_per_s": best["b"]["predictions_per_s"],
                                          "best_ms_per_step": best["b"]["ms_per_step"], "backbone_images_per_step": streams},
                "speedup": round(best["b"]["predictions_per_s"] / best["a"]["predictions_per_s"], 2),
                "max_abs_diff_between_arms": maxdiff})
    del sliding, session, model, video, clip
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--supervision", choices=("realtime", "full"), default="realtime")
    ap.add_argument("--lag", default=None, help="comma-separated output lags of the full model (default 0,4; realtime: 0 only)")
    ap.add_argument("--out", default=None, help="default profiles/r6_stream_realtime.json or profiles/r7_stream_full.json")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--cases", default="swin_b:224:32,swin_b:224:256,swinv2_b:256:32,swinv2_b:256:256")
    a = ap.parse_args()
    lags = [int(x) for x in (a.lag or ("0" if a.supervision == "realtime" else "0,4")).split(",")]
    if a.supervision == "realtime" and lags != [0]:
        ap.error("the realtime model predicts the newest frame: --lag 0 only")
    if not all(0 <= lag < WINDOW for lag in lags):
        ap.error(f"--lag values must be in [0, {WINDOW - 1}]")
    out_file = a.out or os.path.join(ROOT, "profiles", "r6_stream_realtime.json" if a.supervision == "realtime" else "r7_stream_full.json")
    if not torch.cuda.is_available():
        raise RuntimeError("tools/bench_stream.py needs a CUDA device: there is no CPU fallback")
    result = {"gpu": {"device": torch.cuda.get_device_name(0), "name_power_limit_max_sm_clock": smi("name,power.limit,clocks.max.sm")},
              "steps_per_timed_loop": a.steps, "alternations": a.reps, "cases": []}
    if a.supervision != "realtime":
        result["supervision"] = a.supervision
    for c in a.cases.split(","):
        variant, side, streams = c.split(":")
        for lag in lags:
            r = run_case(variant, int(side), int(streams), a.steps, a.reps, a.supervision, lag)
            print(json.dumps(r), flush=True)
            result["cases"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(out_file)), exist_ok=True)
    with open(out_file, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"out": out_file, "gpu": result["gpu"]}))


if __name__ == "__main__":
    main()
