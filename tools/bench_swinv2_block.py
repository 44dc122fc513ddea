"""GPU A/B of the SwinV2 per-block training path (CSVIT_V2_TRAIN_BLOCK=fused, autograd.Swinv2BlockFn) against the op-level path, both with
the tcgen05 attention cores on (CSVIT_V2_TRAIN_ATTN=CSVIT_V2_TRAIN_ATTN8=tcgen05).

    python tools/bench_swinv2_block.py            graphed SwinV2-B finetune step (fp16, batch B = 32, 256^2) for the window-16 and the
                                                  window-8 checkpoint, arms op-level / block alternated twice, plus CUDA-event times and
                                                  achieved HBM bandwidth of csvit_swinv2_cosnorm_bwd at the SwinV2-B stage shapes;
                                                  JSON with the GPU name and power limit read in the same run -> $OUT
                                                  (default profiles/r5_swinv2_block_ab.json)
    python tools/bench_swinv2_block.py profile    torch.profiler table of one eager window-16 step with the block path -> $OUT
                                                  (default profiles/r5_swinv2_block_profile.txt)
"""
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs-vit_b200"))
import torch  # noqa: E402

from cs_vit import ops  # noqa: E402

B = int(os.environ.get("B", "32"))
STEPS = int(os.environ.get("STEPS", "20"))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:      # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def events(fn, iters):
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


def _poser(d, block):
    from cs_vit.net import Poser
    from cs_vit.synthetic import randomize_head_
    from cs_vit.utils.mano_standin import SyntheticMANO
    torch.manual_seed(0)
    model = Poser(d, image_size=256, mano_layer=SyntheticMANO(), spatial_layer_type="encoder", persp_decorate="patch", precision="fp16")
    randomize_head_(model)
    model.phase(Poser.TrainingPhase.SPATIAL)
    model = model.cuda()
    bb = model.backbone
    bb._v2_train_tc = bb._v2_train_tc8 = True          # CSVIT_V2_TRAIN_ATTN=CSVIT_V2_TRAIN_ATTN8=tcgen05
    bb._v2_train_block = block                          # CSVIT_V2_TRAIN_BLOCK=fused
    return model


def _checkpoint(window):
    from cs_vit.synthetic import make_random_backbone_dir
    return make_random_backbone_dir(os.path.join(tempfile.mkdtemp(prefix="csvit_block_"), f"swinv2_b_w{window}"), "swinv2_b", seed=0,
                                    image_size=256, window_size=window)


def finetune_ab(window):
    from cs_vit.synthetic import make_inputs
    from cs_vit.train import GradReducer, GraphedFinetuneStep
    d = _checkpoint(window)
    batch = {k: v.cuda() for k, v in make_inputs(B, 1, 256, seed=100, labels=True).items()}
    out = []
    for arm in ("op-level", "block", "op-level", "block"):
        model = _poser(d, arm == "block")
        params = [p for p in model.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-5, fused=True, capturable=True)
        step = GraphedFinetuneStep(model, batch, opt, GradReducer(params), warmup=3)
        ms = events(lambda: step(batch), STEPS)
        r = {"window": window, "arm": arm, "step_ms": round(ms, 3), "images_per_s": round(B * 1e3 / ms, 1), "loss": step(batch).item()}
        print(json.dumps(r), flush=True)
        out.append(r)
        del step, opt, model
        torch.cuda.empty_cache()
    return out


def cosnorm_bwd_kernel():
    """csvit_swinv2_cosnorm_bwd at the four SwinV2-B stages (window-16 checkpoint, batch B): 16 * C bytes a row plus rnorm.  The timed calls
    rotate over enough input sets (>= 512 MB together, more than four times the 126 MB L2) that every call reads its operands from HBM."""
    out = []
    for H, C in ((64, 128), (32, 256), (16, 512), (8, 1024)):
        rows, heads = B * H * H, C // 32
        g = torch.Generator(device="cuda").manual_seed(C)
        sets = []
        for _ in range(max(2, -(-(512 << 20) // (rows * C * 16)))):
            qkv = torch.randn(rows, 3 * C, device="cuda", generator=g).half()
            grads = [torch.randn(rows, C, device="cuda", generator=g).half() for _ in range(3)]
            sets.append((qkv, torch.rand(rows, 2 * heads, device="cuda", generator=g) + 0.5, grads))
        qs = torch.full((heads,), 14.4, device="cuda")
        it = [0]

        def call():
            qkv, rn, (dq2, dk, dv) = sets[it[0] % len(sets)]
            it[0] += 1
            ops.swinv2_cosnorm_bwd(qkv, rn, qs, dq2, dk, dv)
        ms = events(call, 50)
        nbytes = rows * C * 16 + rows * 2 * heads * 4
        r = {"H": H, "C": C, "rows": rows, "us": round(ms * 1e3, 2), "bytes": nbytes, "TB_per_s": round(nbytes / ms / 1e9, 2)}
        print(json.dumps(r), flush=True)
        out.append(r)
        del sets
        torch.cuda.empty_cache()
    return out


def profile():
    from torch.profiler import ProfilerActivity, profile as tprofile
    from cs_vit.synthetic import make_inputs
    model = _poser(_checkpoint(16), True)
    batch = {k: v.cuda() for k, v in make_inputs(B, 1, 256, seed=1, labels=True).items()}

    def step():
        model.zero_grad(set_to_none=True)
        model(batch)["loss"].backward()
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        step()
        torch.cuda.synchronize()
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=32, max_name_column_width=70)
    info = gpu_info()
    text = (f"# one eager SwinV2-B (window 16) finetune step, batch {B}, 256^2, fp16, CSVIT_V2_TRAIN_BLOCK=fused with both tcgen05 cores\n"
            f"# {info['device']}; nvidia-smi name, power limit, max SM clock: {info['nvidia_smi']}\n{table}\n")
    path = os.environ.get("OUT", os.path.join(ROOT, "profiles", "r5_swinv2_block_profile.txt"))
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        f.write(text)
    print(text)


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "profile":
        profile()
        return
    out = {"gpu": gpu_info(), "batch": B, "dtype": "fp16", "image": 256, "steps": STEPS, "cosnorm_bwd": cosnorm_bwd_kernel(),
           "finetune_swinv2_b_graphed": finetune_ab(16) + finetune_ab(8)}
    path = os.environ.get("OUT", os.path.join(ROOT, "profiles", "r5_swinv2_block_ab.json"))
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
