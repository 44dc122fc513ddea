"""Streaming sessions that step any subset of their streams (``step(..., streams=ids)``) and the state-update kernel under them.

* Kernel: ``ops.stream_update`` (``csvit_stream_update``) against a torch restatement of the lockstep sessions' shift of the
  right-aligned window (``cat`` + ``where``) applied to the selected streams, bit for bit, for W in {1, 4, 128} and D in {768, 1024}:
  resets, saturated histories, padding rows anywhere in the batch, and every stream outside the step unchanged.
* Sessions: capacity 6, window 4, max_batch 4 (buckets 1 / 2 / 4, n = 3 padded to 4) over 14 ticks of a fixed arrival pattern,
  ``RealtimeStream`` and ``FullTemporalStream`` at lag 0 and 2, graphed and eager, in every precision: every returned row against
  ``predict_batch`` on that stream's own clip, and the history length of every stream.
* A bucket of 64 rows for 33 frames; ``streams=list(range(B))`` against the lockstep call; device memory over 50 ticks once every
  bucket is captured; the ``ValueError`` cases, on the CPU and through ``step``.
"""
import pytest
import torch

from helpers import OUT_KEYS
from test_stream_full_gpu import _full_poser
from test_stream_gpu import _realtime_poser

KEYS = ("patches", "square_bboxes", "timestamp", "focal", "princpt")


# ---------------------------------------------------------------------------------------------------- kernel
def _restated_push(ref, tok, ts, ids, reset, W):
    """The lockstep sessions' ``_push`` and stamps update on the rows whose id is >= 0, with padding rows (id -1) set to zeros and
    key_start W - 1.  ``ref``: right-aligned tokens [B, W, 3, D], stamps [B, W] (or None), hist [B]; updated in place."""
    nb = ids.numel()
    sel = ids >= 0
    rows = ids[sel].long()
    hist = torch.where(reset[sel], torch.zeros_like(ref["hist"][rows]), ref["hist"][rows])
    hist = torch.clamp(hist + 1, max=W)
    key_start = W - hist
    valid = torch.arange(W, device=tok.device)[None] >= key_start[:, None]
    tokens = torch.cat([ref["tokens"][rows, 1:], tok[sel][:, None]], dim=1)
    tokens = torch.where(valid[:, :, None, None], tokens, torch.zeros((), device=tok.device))
    ref["tokens"][rows] = tokens
    ref["hist"][rows] = hist
    want = {"window": torch.zeros(nb, *tokens.shape[1:], device=tok.device), "key_start": torch.full_like(ids, W - 1)}
    want["window"][sel] = tokens
    want["key_start"][sel] = key_start
    if ts is not None:
        t = ts[sel]
        stamps = torch.where(valid, torch.cat([ref["stamps"][rows, 1:], t[:, None]], dim=1), t[:, None])
        ref["stamps"][rows] = stamps
        want["stamps"] = torch.zeros(nb, W, device=tok.device)
        want["stamps"][sel] = stamps
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("W", [1, 4, 128])
@pytest.mark.parametrize("D", [768, 1024])
@pytest.mark.parametrize("realtime", [True, False])
def test_stream_update_matches_restated_push(W, D, realtime):
    from cs_vit import ops
    B, nb = 10, 8
    ticks = W + 6                                  # stream 0 arrives every tick, so its history saturates
    g = torch.Generator().manual_seed(1000 * W + D + realtime)
    dev = "cuda"
    state = {"tokens": torch.zeros(B, W, 3, D, device=dev), "hist": torch.zeros(B, dtype=torch.int32, device=dev),
             "head": torch.zeros(B, dtype=torch.int32, device=dev), "stamps": torch.zeros(B, W, device=dev) if realtime else None}
    ref = {"tokens": torch.zeros(B, W, 3, D, device=dev), "hist": torch.zeros(B, dtype=torch.int32, device=dev),
           "stamps": torch.zeros(B, W, device=dev) if realtime else None}
    saturated = False
    for t in range(ticks):
        n = 0 if t == 2 else int(torch.randint(1, nb + 1, (1,), generator=g))
        others = (torch.randperm(B - 1, generator=g)[:n - 1] + 1).tolist() if n else []
        rows = torch.tensor(([0] if n else []) + others + [-1] * (nb - n), dtype=torch.int32)
        ids = rows[torch.randperm(nb, generator=g)].to(dev)           # padding rows anywhere in the batch
        reset = (torch.rand(nb, generator=g) < 0.2).to(dev)
        reset[ids == 0] = t == W + 2                                    # stream 0 saturates, then resets once
        tok = torch.randn(nb, 3, D, generator=g).to(dev)
        ts = (33.3 * t + torch.rand(nb, generator=g)).to(dev) if realtime else None
        before = {k: v.clone() for k, v in state.items() if v is not None}
        window, stamps, key_start = ops.stream_update(tok, ids, reset, state["tokens"], state["hist"], state["head"], ts, state["stamps"])
        want = _restated_push(ref, tok, ts, ids, reset, W)
        assert window.shape == (nb, W, 3, D) and all(window[:, :, q].is_contiguous() for q in range(3))
        assert torch.equal(window, want["window"]), f"tick {t}: window differs"
        assert torch.equal(key_start, want["key_start"]), f"tick {t}: key_start {key_start.tolist()} != {want['key_start'].tolist()}"
        if realtime:
            assert torch.equal(stamps, want["stamps"]), f"tick {t}: stamps differ"
        else:
            assert stamps is None
        assert torch.equal(state["hist"], ref["hist"]), f"tick {t}: hist {state['hist'].tolist()} != {ref['hist'].tolist()}"
        untouched = torch.tensor([b not in ids.tolist() for b in range(B)], device=dev)
        for k, v in before.items():
            assert torch.equal(state[k][untouched], v[untouched]), f"tick {t}: state {k} of a stream outside the step changed"
        saturated |= int(state["hist"][0]) == W
    assert saturated


@pytest.mark.gpu
def test_stream_update_rejects_bad_operands():
    from cs_vit import ops
    B, W, D, nb = 3, 2, 64, 2
    tokens, hist, head = torch.zeros(B, W, 3, D, device="cuda"), *(torch.zeros(B, dtype=torch.int32, device="cuda") for _ in range(2))
    tok, ids = torch.zeros(nb, 3, D, device="cuda"), torch.zeros(nb, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="ids"):
        ops.stream_update(tok, ids.long(), None, tokens, hist, head)
    with pytest.raises(ValueError, match="tok"):
        ops.stream_update(tok.half(), ids, None, tokens, hist, head)
    with pytest.raises(ValueError, match="reset"):
        ops.stream_update(tok, ids, torch.zeros(nb + 1, dtype=torch.bool, device="cuda"), tokens, hist, head)
    with pytest.raises(ValueError, match="timestamp"):
        ops.stream_update(tok, ids, None, tokens, hist, head, torch.zeros(nb, device="cuda"), None)


# ---------------------------------------------------------------------------------------------------- sessions
CAPACITY, WIN, MAXB = 6, 4, 4
# tick -> stream ids in row order.  Stream 0 arrives at every tick but the empty one (its history saturates); stream 5 is idle
# from tick 1 to tick 8, more than the window; tick 3 has one stream; ticks 2, 7, 10 have three (bucket 4 with a padding row).
ARRIVALS = [[0, 1, 2, 5], [3, 0], [0, 4, 1], [0], [], [2, 0, 3, 4], [0, 1], [4, 0, 3], [0, 2, 1, 3], [5, 0], [0, 3, 2],
            [1, 0, 4, 5], [0, 2], [3, 5, 0, 1]]
RESETS = {5: {2}, 7: {4}, 10: {0}, 12: {2}}      # resets mid-history, one of the every-tick stream
TICKS = len(ARRIVALS)

SUBSET_CASES = [(v, side, prec) for v, side in (("swin_xs", 224), ("swinv2_xs", 256)) for prec in ("fp16", "bf16", "fp32")]
SUBSET_CASES.append(("swinv2_xs", 256, "fp8"))


def _inputs(streams: int, ticks: int, side: int, seed: int):
    """[streams, ticks, ...] frames: stream b's frame at tick t; per-stream timestamps, 30 fps with jitter, advancing on every
    tick whether or not the stream delivers its frame."""
    from cs_vit.synthetic import make_inputs
    inp = make_inputs(streams, ticks, side, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    dt = 33.333 + 4.0 * torch.rand(streams, ticks, generator=g)
    inp["timestamp"] = 1000.0 * torch.arange(streams, dtype=torch.float32)[:, None] + torch.cumsum(dt, dim=1)
    return {k: v.cuda() for k, v in inp.items()}


def _model(supervision: str, variant: str, side: int, precision: str):
    if supervision == "realtime":
        return _realtime_poser(variant, side, "encoder", precision).cuda()
    return _full_poser(variant, side, "encoder", precision).cuda()


def _sessions(model, supervision: str, num_streams: int, max_batch: int, graphed=(True, False)):
    from cs_vit.stream import FullTemporalStream, RealtimeStream
    if supervision == "realtime":
        return {(g, 0): RealtimeStream(model, num_streams, WIN, graph=g, max_batch=max_batch) for g in graphed}
    return {(g, lag): FullTemporalStream(model, num_streams, WIN, lag=lag, graph=g, max_batch=max_batch) for g in graphed for lag in (0, 2)}


def _check_outputs(model, inp, ids, t, frames, got, supervision):
    """Every returned row of stream b against predict_batch on b's frames since its last reset (at most WIN of them)."""
    for i, b in enumerate(ids):
        clip = frames[b][-WIN:]
        h = len(clip)
        with torch.no_grad():
            want = model.predict_batch(*(inp[k][b:b + 1, clip] for k in KEYS))
        for (graphed, lag), out in got.items():
            name = f"{'graphed' if graphed else 'eager'} lag {lag} tick {t} stream {b} ({h} frames)"
            if supervision == "full":
                assert bool(out["valid"][i]) == (h > lag), f"{name}: valid"
            for k in OUT_KEYS:
                a = out[k][i:i + 1]
                if supervision == "full" and h <= lag:
                    assert torch.isfinite(a).all(), f"{name} {k}: invalid row not finite"
                    continue
                w = want[k] if supervision == "realtime" else want[k][:, h - 1 - lag:h - lag]
                assert torch.equal(a, w), f"{name} {k}: max |diff| {(a.double() - w.double()).abs().max().item():.3e}"


def _tick(inp, ids, t, resets):
    frame = [inp[k][ids, t] for k in KEYS]
    reset = torch.tensor([b in resets for b in ids], dtype=torch.bool, device="cuda")
    return frame, reset


@pytest.mark.gpu
@pytest.mark.parametrize("supervision", ["realtime", "full"])
@pytest.mark.parametrize("variant,side,precision", SUBSET_CASES)
def test_subset_sessions_match_predict_batch(supervision, variant, side, precision):
    model = _model(supervision, variant, side, precision)
    inp = _inputs(CAPACITY, TICKS, side, seed=17)
    sessions = _sessions(model, supervision, CAPACITY, MAXB)
    frames = [[] for _ in range(CAPACITY)]          # ticks of each stream's frames since its last reset
    for t, ids in enumerate(ARRIVALS):
        resets = RESETS.get(t, set())
        for b in ids:
            if b in resets:
                frames[b] = []
            frames[b].append(t)
        frame, reset = _tick(inp, ids, t, resets)
        got = {key: {k: v.clone() for k, v in s.step(*frame, reset=reset, streams=ids).items()} for key, s in sessions.items()}
        for out in got.values():
            assert all(v.shape[0] == len(ids) for v in out.values())
        _check_outputs(model, inp, ids, t, frames, got, supervision)
        for s in sessions.values():
            assert s.hist.tolist() == [min(len(f), WIN) for f in frames], f"tick {t}: hist"
    for (graphed, _), s in sessions.items():
        assert sorted(s.graphs) == ([1, 2, 4] if graphed else [])


@pytest.mark.gpu
def test_subset_session_large_bucket():
    """33 frames run in the 64-row graph: every row still equals the single-clip predict_batch."""
    from cs_vit.stream import bucket
    model = _model("realtime", "swinv2_xs", 256, "fp16")
    inp = _inputs(64, 2, 256, seed=23)
    (s,) = _sessions(model, "realtime", 64, 64, graphed=(True,)).values()
    frames = [[] for _ in range(64)]
    for t, ids in enumerate([list(range(0, 64, 2)) + [63], list(range(63, 30, -1))]):
        assert len(ids) == 33 and bucket(len(ids), 64) == 64
        resets = {40} if t == 1 else set()
        for b in ids:
            frames[b] = [t] if b in resets else frames[b] + [t]
        frame, reset = _tick(inp, ids, t, resets)
        got = {(True, 0): {k: v.clone() for k, v in s.step(*frame, reset=reset, streams=ids).items()}}
        _check_outputs(model, inp, ids, t, frames, got, "realtime")
    assert sorted(s.graphs) == [64]
    assert s.hist.tolist() == [min(len(f), WIN) for f in frames]


@pytest.mark.gpu
@pytest.mark.parametrize("supervision", ["realtime", "full"])
def test_all_streams_in_order_equals_lockstep_step(supervision):
    model = _model(supervision, "swin_xs", 224, "fp16")
    B = 4
    inp = _inputs(B, 7, 224, seed=29)
    sub = _sessions(model, supervision, B, B, graphed=(True,))
    lock = _sessions(model, supervision, B, B, graphed=(True,))
    for t in range(7):
        reset = torch.tensor([t == 3 and b == 1 for b in range(B)], device="cuda")
        frame = [inp[k][:, t].contiguous() for k in KEYS]
        for key in lock:
            a = lock[key].step(*frame, reset=reset)
            b = sub[key].step(*frame, reset=reset, streams=list(range(B)))
            for k in a:
                assert torch.equal(a[k], b[k]), f"tick {t} {key} {k}"
            assert torch.equal(lock[key].hist, sub[key].hist)


@pytest.mark.gpu
@pytest.mark.parametrize("supervision", ["realtime", "full"])
def test_subset_session_memory_is_flat(supervision):
    """Once every bucket has its graph, steps allocate no device memory."""
    model = _model(supervision, "swinv2_xs", 256, "fp16")
    ticks = 54
    inp = _inputs(CAPACITY, ticks, 256, seed=31)
    g = torch.Generator().manual_seed(5)
    pattern = [[0], [1, 2], [3, 4, 5], [0, 1, 2, 3]]                      # buckets 1, 2, 4 (n = 3 padded)
    pattern += [torch.randperm(CAPACITY, generator=g)[:int(torch.randint(0, MAXB + 1, (1,), generator=g))].tolist() for _ in range(50)]
    steps = [_tick(inp, ids, t, {ids[0]} if ids and t % 7 == 3 else set()) + (ids,) for t, ids in enumerate(pattern)]
    sessions = _sessions(model, supervision, CAPACITY, MAXB, graphed=(True,)).values()
    for frame, reset, ids in steps[:4]:
        for s in sessions:
            s.step(*frame, reset=reset, streams=ids)
    assert all(sorted(s.graphs) == [1, 2, 4] for s in sessions)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    for frame, reset, ids in steps[4:]:
        for s in sessions:
            assert s.step(*frame, reset=reset, streams=ids)["joint_cam"].shape[0] == len(ids)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == before


@pytest.mark.gpu
def test_step_rejects_bad_streams():
    model = _model("realtime", "swin_xs", 224, "fp32")
    inp = _inputs(CAPACITY, 1, 224, seed=37)
    (s,) = _sessions(model, "realtime", CAPACITY, MAXB, graphed=(True,)).values()
    frame, _ = _tick(inp, [0, 1], 0, set())
    for bad in ([0, 0], [0, CAPACITY], [-1, 2]):
        with pytest.raises(ValueError, match="stream ids"):
            s.step(*frame, streams=bad)
    with pytest.raises(ValueError, match="max_batch"):
        s.step(*_tick(inp, [0, 1, 2, 3, 4], 0, set())[0], streams=[0, 1, 2, 3, 4])
    with pytest.raises(ValueError, match="one row per stream id"):
        s.step(*frame, streams=[0, 1, 2])
    with pytest.raises(ValueError, match="reset"):
        s.step(*frame, reset=torch.zeros(3, dtype=torch.bool, device="cuda"), streams=[0, 1])
    out = s.step(*_tick(inp, [], 0, set())[0], streams=[])
    assert all(v.shape[0] == 0 for v in out.values()) and not s.graphs
    assert s.hist.tolist() == [0] * CAPACITY


# ---------------------------------------------------------------------------------------------------- errors and buckets (CPU)
def test_buckets():
    from cs_vit.stream import bucket
    assert sorted({bucket(n, 256) for n in range(1, 257)}) == [1, 2, 4, 8, 16, 32, 64, 96, 128, 160, 192, 224, 256]
    assert all(n <= bucket(n, 256) <= n + 31 for n in range(33, 257))
    assert [bucket(n, 4) for n in (1, 2, 3, 4)] == [1, 2, 4, 4]
    assert [bucket(n, 100) for n in (33, 65, 97, 100)] == [64, 96, 100, 100]


def test_stream_ids_and_rows_are_checked():
    from cs_vit.stream import _check_rows, _stream_ids
    assert _stream_ids(None, 3, 3).tolist() == [0, 1, 2]
    assert _stream_ids([2, 0], 3, 2).tolist() == [2, 0]
    assert _stream_ids(torch.tensor([1], dtype=torch.int32), 3, 2).tolist() == [1]
    assert _stream_ids([], 3, 2).numel() == 0
    for bad in ([1, 1], [0, 3], [-1], torch.tensor([0.0]), [0.5], torch.tensor([[0]])):
        with pytest.raises(ValueError, match="stream"):
            _stream_ids(bad, 3, 3)
    with pytest.raises(ValueError, match="max_batch"):
        _stream_ids([0, 1, 2], 3, 2)
    with pytest.raises(ValueError, match="max_batch"):
        _stream_ids(None, 3, 2)

    def rows(n, ts=None):
        return {"patches": torch.zeros(n, 3, 8, 8), "square_bboxes": torch.zeros(n, 4), "timestamp": torch.zeros(n) if ts is None else ts,
                "focal": torch.zeros(n, 2), "princpt": torch.zeros(n, 2)}
    _check_rows(2, rows(2), torch.zeros(2, dtype=torch.bool))
    _check_rows(0, rows(0), None)
    for bad in (rows(3), {**rows(2), "focal": torch.zeros(1, 2)}, rows(2, ts=torch.zeros(2, 1)), {**rows(2), "patches": torch.zeros(2, 3)}):
        with pytest.raises(ValueError, match="one row per stream id"):
            _check_rows(2, bad, None)
    for bad in (torch.zeros(2), torch.zeros(3, dtype=torch.bool)):
        with pytest.raises(ValueError, match="reset"):
            _check_rows(2, rows(2), bad)


def test_sessions_reject_bad_max_batch():
    from cs_vit.stream import FullTemporalStream, RealtimeStream
    rt = _realtime_poser("swin_xs", 224, "encoder", "fp32")
    full = _full_poser("swin_xs", 224, "encoder", "fp32")
    for bad in (0, 5):
        with pytest.raises(ValueError, match="max_batch"):
            RealtimeStream(rt, 4, 4, max_batch=bad)
        with pytest.raises(ValueError, match="max_batch"):
            FullTemporalStream(full, 4, 4, max_batch=bad)
