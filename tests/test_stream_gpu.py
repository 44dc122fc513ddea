"""Streaming inference for the realtime temporal Poser (``cs_vit.stream.RealtimeStream``) and the ragged head attention under it.

* Kernel: ``ops.attention(..., key_start=)`` (``csvit_attention_ragged``) against ``ops.attention`` on each sequence's valid keys alone,
  bit for bit, in fp32 / bf16 / fp16.
* Session: every step of a 4-stream, window-4 session, graphed and eager, against ``predict_batch`` on the one clip of each stream's
  frames since its last reset (at most ``window`` of them), bit for bit in every precision and for every output key.
* Errors: the constructor's ``ValueError`` cases, on the CPU.
"""
import os
import tempfile

import pytest
import torch

from helpers import OUT_KEYS

_TMP = tempfile.mkdtemp(prefix="csvit_stream_tests_")
_DIRS = {}


def _backbone(variant: str, side: int) -> str:
    from cs_vit.synthetic import make_random_backbone_dir
    if variant not in _DIRS:
        v2 = variant.startswith("swinv2")
        _DIRS[variant] = make_random_backbone_dir(os.path.join(_TMP, variant), variant, seed=0, image_size=side,
                                                  window_size=16 if v2 else 0)
    return _DIRS[variant]


def _realtime_poser(variant: str, side: int, layer_type: str, precision: str, **kw):
    from cs_vit.net import Poser
    from cs_vit.synthetic import randomize_head_
    from cs_vit.utils.mano_standin import SyntheticMANO
    torch.manual_seed(0)
    args = dict(image_size=side, mano_layer=SyntheticMANO(), spatial_layer_type=layer_type,
                persp_decorate="patch" if layer_type == "encoder" else "query", precision=precision,
                temporal_supervision="realtime", temporal_init_method="random")
    args.update(kw)
    model = Poser(_backbone(variant, side), **args)
    randomize_head_(model)
    model.phase(Poser.TrainingPhase.INFERENCE)
    return model


# ---------------------------------------------------------------------------------------------------- kernel
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("S", [1, 8, 67, 128])
@pytest.mark.parametrize("Lq", [1, 3])
def test_ragged_attention_matches_shorter_calls(dtype, S, Lq):
    from cs_vit import ops
    heads, D, n = 2, 64, 7
    g = torch.Generator().manual_seed(1000 * S + Lq)
    q = (0.3 * torch.randn(n * Lq, 3 * D, generator=g)).to(dtype).cuda()[:, D:2 * D]      # column slice, pitch 3D
    kv = (0.3 * torch.randn(n * S, 2 * D, generator=g)).to(dtype).cuda()
    k, v = kv[:, :D], kv[:, D:]
    ks = torch.randint(0, S, (n,), generator=g)
    ks[0], ks[1] = 0, S - 1
    key_start = ks.to(torch.int32).cuda()
    scale = 32 ** 0.5                         # the head's logit multiplier (quirk Q1)
    got = ops.attention(q, k, v, n, Lq, S, heads, scale, key_start=key_start)
    for s in range(n):
        r0, r1 = s * S + int(ks[s]), (s + 1) * S
        want = ops.attention(q[s * Lq:(s + 1) * Lq], k[r0:r1], v[r0:r1], 1, Lq, r1 - r0, heads, scale)
        assert torch.equal(got[s * Lq:(s + 1) * Lq], want), f"sequence {s} (key_start {int(ks[s])}) differs from the shorter call"
    zero = ops.attention(q, k, v, n, Lq, S, heads, scale, key_start=torch.zeros(n, dtype=torch.int32, device="cuda"))
    assert torch.equal(zero, ops.attention(q, k, v, n, Lq, S, heads, scale))
    assert torch.isfinite(got.float()).all()


@pytest.mark.gpu
def test_ragged_attention_rejects_bad_key_start():
    from cs_vit import ops
    q = torch.zeros(4, 32, device="cuda")
    kv = torch.zeros(4 * 5, 32, device="cuda")
    for bad in (torch.zeros(4, dtype=torch.int64, device="cuda"), torch.zeros(3, dtype=torch.int32, device="cuda"),
                torch.zeros(8, dtype=torch.int32, device="cuda")[::2]):
        with pytest.raises(ValueError, match="key_start"):
            ops.attention(q, kv, kv, 4, 1, 5, 1, 1.0, key_start=bad)


# ---------------------------------------------------------------------------------------------------- session
STREAMS, WINDOW, STEPS = 4, 4, 10
# step -> streams reset at that step: stream 0 never (it slides a full window from step 4 on), stream 2 on every step
RESETS = {s: {2} | ({1} if s in (3, 7) else set()) | ({3} if s == 5 else set()) for s in range(STEPS)}

SESSION_CASES = [(v, side, layer, prec) for v, side in (("swin_xs", 224), ("swinv2_xs", 256))
                 for layer in ("encoder", "decoder") for prec in ("fp16", "bf16", "fp32")]
SESSION_CASES.append(("swin_t", 224, "encoder", "fp16"))


def _stream_inputs(side: int, seed: int):
    """[STREAMS, STEPS, ...] frames; per-stream timestamps with different offsets and jittered 30 fps spacing."""
    from cs_vit.synthetic import make_inputs
    inp = make_inputs(STREAMS, STEPS, side, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    dt = 33.333 + 4.0 * torch.rand(STREAMS, STEPS, generator=g)
    inp["timestamp"] = 1000.0 * torch.arange(STREAMS, dtype=torch.float32)[:, None] + torch.cumsum(dt, dim=1)
    return {k: v.cuda() for k, v in inp.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("variant,side,layer_type,precision", SESSION_CASES)
def test_stream_matches_predict_batch(variant, side, layer_type, precision):
    from cs_vit.stream import RealtimeStream
    model = _realtime_poser(variant, side, layer_type, precision).cuda()
    inp = _stream_inputs(side, seed=7)
    sessions = {"graphed": RealtimeStream(model, STREAMS, WINDOW), "eager": RealtimeStream(model, STREAMS, WINDOW, graph=False)}
    start = [0] * STREAMS                     # first frame of each stream's history
    for t in range(STEPS):
        for b in RESETS[t]:
            start[b] = t
        reset = torch.tensor([b in RESETS[t] for b in range(STREAMS)], device="cuda")
        frame = {k: inp[k][:, t].contiguous() for k in ("patches", "square_bboxes", "timestamp", "focal", "princpt")}
        got = {name: {k: v.clone() for k, v in s.step(frame["patches"], frame["square_bboxes"], frame["timestamp"], frame["focal"],
                                                      frame["princpt"], reset=reset).items()}
               for name, s in sessions.items()}
        for b in range(STREAMS):
            f0 = max(start[b], t - WINDOW + 1)
            with torch.no_grad():
                want = model.predict_batch(*(inp[k][b:b + 1, f0:t + 1] for k in ("patches", "square_bboxes", "timestamp", "focal", "princpt")))
            for name, out in got.items():
                for k in OUT_KEYS:
                    assert out[k].shape[1] == 1 and want[k].shape[1] == 1
                    a, w = out[k][b:b + 1], want[k]
                    assert torch.equal(a, w), (f"{name} step {t} stream {b} ({t + 1 - f0} frames) {k}: "
                                               f"max |diff| {(a.double() - w.double()).abs().max().item():.3e}")
        for s in sessions.values():
            assert s.hist.tolist() == [min(t + 1 - start[b], WINDOW) for b in range(STREAMS)]


@pytest.mark.gpu
def test_stream_temporal_path_is_not_trivial():
    """With temporal_init_method="random" the temporal encoders change the prediction, so the session tests above exercise them."""
    model = _realtime_poser("swin_xs", 224, "encoder", "fp32").cuda()
    inp = _stream_inputs(224, seed=3)
    with torch.no_grad():
        full = model.predict_batch(*(inp[k][:1, :WINDOW] for k in ("patches", "square_bboxes", "timestamp", "focal", "princpt")))
        last = model.predict_batch(*(inp[k][:1, WINDOW - 1:WINDOW] for k in ("patches", "square_bboxes", "timestamp", "focal", "princpt")))
    assert not torch.equal(full["joint_cam"], last["joint_cam"])


# ---------------------------------------------------------------------------------------------------- errors (CPU)
def test_stream_rejects_unsupported_models():
    from cs_vit.net import Poser
    from cs_vit.stream import RealtimeStream
    model = _realtime_poser("swin_xs", 224, "encoder", "fp32")
    with pytest.raises(ValueError, match="window"):
        RealtimeStream(model, 2, 129)
    with pytest.raises(ValueError, match="window"):
        RealtimeStream(model, 2, 0)
    model.train()
    with pytest.raises(ValueError, match="eval mode"):
        RealtimeStream(model, 2, 8)
    model.phase(Poser.TrainingPhase.TEMPORAL)
    model.eval()
    with pytest.raises(ValueError, match="INFERENCE"):
        RealtimeStream(model, 2, 8)
    full = _realtime_poser("swin_xs", 224, "encoder", "fp32", temporal_supervision="full")
    with pytest.raises(ValueError, match="realtime"):
        RealtimeStream(full, 2, 8)
