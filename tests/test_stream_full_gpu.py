"""Streaming inference for the full temporal Poser (``cs_vit.stream.FullTemporalStream``) and the ragged self-attention under it.

* Module: a "full" ``TemporalEncoder`` with ``key_start`` against calls on each clip's valid frames alone, bit for bit on every
  valid slot, in fp32 / bf16 / fp16.
* Session: every step of a 4-stream, window-4 session, graphed and eager, lag 0 and lag 2, against ``predict_batch`` on the one
  clip of each stream's frames since its last reset (at most ``window`` of them) at frame ``-1 - lag``, bit for bit in every
  precision and for every output key; ``valid`` against h > lag.
* Non-triviality: the temporal encoders and the look-ahead change the prediction.
* Errors: the constructor's ``ValueError`` cases, on the CPU; the differentiable ``EncoderBlock`` path refuses ``key_start``.
"""
import pytest
import torch

from helpers import OUT_KEYS
from test_stream_gpu import RESETS, STEPS, STREAMS, WINDOW, _backbone, _realtime_poser, _stream_inputs

LAGS = (0, 2)


def _full_poser(variant: str, side: int, layer_type: str, precision: str):
    from cs_vit.net import Poser
    from cs_vit.synthetic import randomize_head_
    from cs_vit.utils.mano_standin import SyntheticMANO
    torch.manual_seed(0)
    model = Poser(_backbone(variant, side), image_size=side, mano_layer=SyntheticMANO(), spatial_layer_type=layer_type,
                  persp_decorate="patch" if layer_type == "encoder" else "query", precision=precision,
                  temporal_supervision="full", temporal_init_method="random")
    randomize_head_(model)
    model.phase(Poser.TrainingPhase.INFERENCE)
    return model


def _clip(inp, b: int, f0: int, t: int):
    return [inp[k][b:b + 1, f0:t + 1] for k in ("patches", "square_bboxes", "timestamp", "focal", "princpt")]


def _frame(inp, t: int):
    return [inp[k][:, t].contiguous() for k in ("patches", "square_bboxes", "timestamp", "focal", "princpt")]


# ---------------------------------------------------------------------------------------------------- module
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("T", [1, 4, 8])
@pytest.mark.parametrize("layers", [1, 3])
def test_full_temporal_encoder_key_start_matches_shorter_clips(precision, T, layers):
    from cs_vit.net.blocks import set_precision
    from cs_vit.net.poser import TemporalEncoder
    from cs_vit.synthetic import randomize_head_
    torch.manual_seed(100 * T + layers)
    D, heads, B = 128, 4, 6
    enc = TemporalEncoder(D, heads, layers, target="full", do_zero_init=False)
    randomize_head_(enc, seed=T)
    set_precision(enc, precision)
    enc = enc.cuda().eval()
    g = torch.Generator().manual_seed(T)
    x = torch.randn(B, T, D, generator=g).cuda()
    ks = torch.randint(0, T, (B,), generator=g)
    ks[0], ks[1] = 0, T - 1
    with torch.no_grad():
        got = enc(x, key_start=ks.to(torch.int32).cuda())
        assert torch.equal(enc(x, key_start=torch.zeros(B, dtype=torch.int32, device="cuda")), enc(x))
        for b in range(B):
            k0 = int(ks[b])
            want = enc(x[b:b + 1, k0:].contiguous())
            assert torch.equal(got[b:b + 1, k0:], want), f"clip {b} (key_start {k0}) differs from the call on its {T - k0} frames"
    assert torch.isfinite(got).all()


# ---------------------------------------------------------------------------------------------------- session
SESSION_CASES = [(v, side, layer, prec) for v, side in (("swin_xs", 224), ("swinv2_xs", 256))
                 for layer in ("encoder", "decoder") for prec in ("fp16", "bf16", "fp32")]
SESSION_CASES.append(("swin_t", 224, "encoder", "fp16"))


@pytest.mark.gpu
@pytest.mark.parametrize("variant,side,layer_type,precision", SESSION_CASES)
def test_full_stream_matches_predict_batch(variant, side, layer_type, precision):
    from cs_vit.stream import FullTemporalStream
    model = _full_poser(variant, side, layer_type, precision).cuda()
    inp = _stream_inputs(side, seed=11)
    sessions = {(name, lag): FullTemporalStream(model, STREAMS, WINDOW, lag=lag, graph=(name == "graphed"))
                for name in ("graphed", "eager") for lag in LAGS}
    start = [0] * STREAMS                     # first frame of each stream's history
    for t in range(STEPS):
        for b in RESETS[t]:
            start[b] = t
        reset = torch.tensor([b in RESETS[t] for b in range(STREAMS)], device="cuda")
        got = {key: {k: v.clone() for k, v in s.step(*_frame(inp, t), reset=reset).items()} for key, s in sessions.items()}
        for b in range(STREAMS):
            f0 = max(start[b], t - WINDOW + 1)
            h = t + 1 - f0
            with torch.no_grad():
                want = model.predict_batch(*_clip(inp, b, f0, t))
            for (name, lag), out in got.items():
                assert out["valid"].dtype == torch.bool and out["valid"].shape == (STREAMS,)
                assert bool(out["valid"][b]) == (h > lag), f"{name} lag {lag} step {t} stream {b}: valid with {h} frames"
                for k in OUT_KEYS:
                    a = out[k][b:b + 1]
                    assert a.shape[1] == 1
                    if h <= lag:
                        assert torch.isfinite(a).all(), f"{name} lag {lag} step {t} stream {b} {k}: invalid row not finite"
                        continue
                    w = want[k][:, h - 1 - lag:h - lag]
                    assert torch.equal(a, w), (f"{name} lag {lag} step {t} stream {b} ({h} frames) {k}: "
                                               f"max |diff| {(a.double() - w.double()).abs().max().item():.3e}")
        for s in sessions.values():
            assert s.hist.tolist() == [min(t + 1 - start[b], WINDOW) for b in range(STREAMS)]


@pytest.mark.gpu
def test_full_stream_temporal_path_is_not_trivial():
    """With temporal_init_method="random" the temporal encoders and the look-ahead change the prediction, so the session tests
    above exercise them."""
    from cs_vit.stream import FullTemporalStream
    model = _full_poser("swin_xs", 224, "encoder", "fp32").cuda()
    inp = _stream_inputs(224, seed=3)
    with torch.no_grad():
        clip = model.predict_batch(*_clip(inp, 0, 0, WINDOW - 1))
        alone = model.predict_batch(*_clip(inp, 0, WINDOW - 1, WINDOW - 1))
    assert not torch.equal(clip["joint_cam"][:, -1:], alone["joint_cam"])
    lag0 = FullTemporalStream(model, STREAMS, WINDOW, lag=0)
    lag2 = FullTemporalStream(model, STREAMS, WINDOW, lag=2)
    seen = []
    for t in range(WINDOW):
        o0 = lag0.step(*_frame(inp, t))["joint_cam"].clone()
        o2 = lag2.step(*_frame(inp, t))["joint_cam"].clone()
        seen.append(o0)
    assert not torch.equal(o2, o0)
    assert not torch.equal(o2, seen[WINDOW - 3]), "lag 2 must see the two frames after the one it decodes"


# ---------------------------------------------------------------------------------------------------- errors
@pytest.mark.gpu
def test_differentiable_encoder_block_refuses_key_start():
    from cs_vit.net.blocks import EncoderBlock
    block = EncoderBlock(64, 2).cuda()
    x = torch.randn(3, 4, 64, device="cuda", requires_grad=True)
    with pytest.raises(ValueError, match="key_start"):
        block(x, key_start=torch.zeros(3, dtype=torch.int32, device="cuda"))


def test_encoder_block_attention_refuses_key_start_with_grad():
    """The check sits in ``MHA.attend`` ahead of any kernel, so it holds on the CPU too."""
    from cs_vit.net.blocks import EncoderBlock
    block = EncoderBlock(64, 2)
    x2 = torch.randn(12, 64, requires_grad=True)
    with pytest.raises(ValueError, match="key_start"):
        block.attn.attend(x2, None, 3, 4, 4, x2, key_start=torch.zeros(3, dtype=torch.int32))


def test_full_stream_rejects_bad_arguments():
    from cs_vit.net import Poser
    from cs_vit.stream import FullTemporalStream
    model = _full_poser("swin_xs", 224, "encoder", "fp32")
    for window in (0, 129):
        with pytest.raises(ValueError, match="window"):
            FullTemporalStream(model, 2, window)
    for lag in (-1, 8):
        with pytest.raises(ValueError, match="lag"):
            FullTemporalStream(model, 2, 8, lag=lag)
    with pytest.raises(ValueError, match="num_streams"):
        FullTemporalStream(model, 0, 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        FullTemporalStream(model, 2, 8, lag=7)
    model.train()
    with pytest.raises(ValueError, match="eval mode"):
        FullTemporalStream(model, 2, 8)
    model.phase(Poser.TrainingPhase.TEMPORAL)
    model.eval()
    with pytest.raises(ValueError, match="INFERENCE"):
        FullTemporalStream(model, 2, 8)
    with pytest.raises(ValueError, match="full"):
        FullTemporalStream(_realtime_poser("swin_xs", 224, "encoder", "fp32"), 2, 8)
