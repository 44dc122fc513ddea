"""Streaming inference for the temporal ``Poser``: one backbone pass per new frame.

Run on a live video with ``predict_batch``, consecutive clips share T-1 frames and every call repeats the backbone, perspective
MLP and spatial encoder on all of them.  Everything before the temporal encoders works frame by frame, and the temporal
encoders only need the per-frame ``[3, D]`` spatial tokens of the last T frames (plus their timestamps for the realtime
model).  The sessions here keep those tokens on the device, so a step runs the per-frame part on the B new frames only and
the temporal part on the cached window.

* ``RealtimeStream``: ``temporal_supervision="realtime"``, which predicts the newest frame of a clip.
* ``FullTemporalStream``: ``temporal_supervision="full"`` (the default), which predicts every frame of a clip from the
  whole clip.  The session decodes one frame per stream, ``lag`` frames behind the newest, so that frame sees ``lag`` frames
  of look-ahead at ``lag`` frames of latency.

Streams start and reset independently.  A stream that has seen h < window frames since its last reset attends to its
h newest slots only (``key_start = window - h`` in the head's attention kernel, ``csvit_attention_ragged``), so its
output equals ``predict_batch`` on its h-frame clip, bit for bit.

Streams also arrive independently: ``step(..., streams=ids)`` takes frames for any subset of the ``num_streams`` streams, at most
``max_batch`` of them, and runs the per-frame part on those frames only.  A stream that is not in ``ids`` is not touched; its
history is made of the frames it received.  A step on n frames runs the graph of the smallest bucket that holds n (1, 2, 4, 8,
16, 32, then multiples of 32, capped at ``max_batch``); its padding rows carry stream id -1 and change no state.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Union

import torch

from . import ops
from .graph import KEYS

_MAX_WINDOW = 128          # key limit of the head's attention kernel (csrc/attention_simt.cu)


def _check_session(name: str, supervision: str, model, num_streams: int, window: int, max_batch: Optional[int]) -> None:
    from .net.poser import Poser
    if model.training_phase != Poser.TrainingPhase.INFERENCE:
        raise ValueError(f"{name} needs a model in the INFERENCE phase, got {model.training_phase}")
    if model.training:
        raise ValueError(f"{name} needs a model in eval mode (call model.eval())")
    if model.temporal_supervision != supervision:
        raise ValueError(f"{name} needs temporal_supervision={supervision!r}, got {model.temporal_supervision!r}")
    if not 1 <= window <= _MAX_WINDOW:
        raise ValueError(f"window must be in [1, {_MAX_WINDOW}] (the head attention kernel's key limit), got {window}")
    if num_streams < 1:
        raise ValueError(f"num_streams must be >= 1, got {num_streams}")
    if max_batch is not None and not 1 <= max_batch <= num_streams:
        raise ValueError(f"max_batch must be in [1, num_streams] = [1, {num_streams}], got {max_batch}")


def bucket(n: int, max_batch: int) -> int:
    """Rows of the graph that runs a step on n frames: the next of 1, 2, 4, 8, 16, 32, 64, 96, ... (powers of two up to 32,
    then multiples of 32), capped at ``max_batch``.  Above 32 frames a step pads at most 31 rows."""
    b = 1 << max(n - 1, 0).bit_length() if n <= 32 else 32 * -(-n // 32)
    return min(b, max_batch)


def _stream_ids(streams: Union[None, Sequence[int], torch.Tensor], num_streams: int, max_batch: int) -> torch.Tensor:
    """The int64 CPU tensor of a step's stream ids; ``None`` is every stream in order.  Raises ``ValueError`` for ids that are
    not distinct integers in [0, num_streams) or more than ``max_batch`` of them."""
    if streams is None:
        ids = torch.arange(num_streams)
    elif torch.is_tensor(streams):
        if streams.device.type != "cpu" or streams.dim() != 1 or streams.dtype.is_floating_point or streams.dtype == torch.bool \
                or streams.is_complex():
            raise ValueError(f"streams must be a list or a 1-D CPU integer tensor, got {streams.dtype} {tuple(streams.shape)} "
                             f"on {streams.device}")
        ids = streams.long()
    else:
        ids = list(streams)
        if not all(isinstance(i, int) or (torch.is_tensor(i) and i.dim() == 0 and not i.dtype.is_floating_point) for i in ids):
            raise ValueError("streams must be a list of integer stream indices")
        ids = torch.tensor([int(i) for i in ids], dtype=torch.int64)
    n = ids.numel()
    if n > max_batch:
        raise ValueError(f"{n} frames in one step, max_batch is {max_batch}")
    if n and (int(ids.min()) < 0 or int(ids.max()) >= num_streams):
        raise ValueError(f"stream ids must be in [0, {num_streams}), got {ids.tolist()}")
    if torch.unique(ids).numel() != n:
        raise ValueError(f"stream ids must be distinct (one frame per stream and step), got {ids.tolist()}")
    return ids


def _check_rows(n: int, inputs: Dict[str, torch.Tensor], reset: Optional[torch.Tensor]) -> None:
    """Every input has one row per stream id: ``patches [n,3,S,S]``, ``timestamp [n]``, ``reset`` bool ``[n]`` or None."""
    rows = {k: tuple(v.shape) for k, v in inputs.items()}
    if inputs["patches"].dim() != 4 or tuple(inputs["timestamp"].shape) != (n,) or any(s[:1] != (n,) for s in rows.values()):
        raise ValueError(f"step takes one row per stream id ({n} ids): patches [{n},3,S,S], square_bboxes [{n},4], timestamp [{n}], "
                         f"focal / princpt [{n},2], got {rows}")
    if reset is not None and (reset.dtype != torch.bool or tuple(reset.shape) != (n,)):
        raise ValueError(f"reset must be a bool tensor of shape [{n}]")


class _TokenWindow:
    """What both sessions share: the per-stream spatial tokens (a ring of ``window`` slots per stream, ``[num_streams, window, 3,
    D]`` fp32), history lengths and ring heads ``[num_streams]`` int32 on the device, the per-frame part of a step, the state update
    (``ops.stream_update``), stream-id handling and the per-bucket CUDA graphs.  Subclasses implement ``_advance``."""

    def __init__(self, model, num_streams: int, window: int, graph: bool, max_batch: Optional[int]):
        model._check_positioning()
        dev = model.query_token.device
        if dev.type != "cuda":
            raise RuntimeError(f"{type(self).__name__} runs on CUDA only (there is no CPU fallback): move the model to the GPU first")
        self.model, self.num_streams, self.window = model, num_streams, window
        self.max_batch = num_streams if max_batch is None else max_batch
        self.use_graph = graph
        B, W, M = num_streams, window, self.max_batch
        self.tokens = torch.zeros(B, W, 3, model.hidden_dim, device=dev)
        self.stamps = None
        self.hist = torch.zeros(B, dtype=torch.int32, device=dev)
        self.head = torch.zeros(B, dtype=torch.int32, device=dev)
        # stream ids of a step's rows (-1 = padding), staged through two pinned buffers: the host refills one only after the
        # copy that last read it has run
        self._ids = torch.full((M,), -1, dtype=torch.int32, device=dev)
        self._ids_host = [torch.empty(M, dtype=torch.int32, pin_memory=True) for _ in range(2)]
        self._ids_copied = [None, None]
        self._ticks = 0
        self.graphs: Dict[int, torch.cuda.CUDAGraph] = {}
        self._pool = None
        self.static_in = None       # max_batch-row input buffers; bucket nb's graph reads their first nb rows
        self.static_out = None      # max_batch-row output buffers; bucket nb's graph writes their first nb rows

    def recapture(self) -> None:
        """Drop every captured graph; the next ``step`` of each bucket captures a new one (needed after the weights change)."""
        self.graphs = {}
        self._pool = None

    def _push(self, patches, square_bboxes, timestamp, focal, princpt, reset, ids):
        """Runs the per-frame part on the new frames and moves them into their streams' history.  Returns the temporal operands
        of ``ops.stream_update``: ``window [nb, W, 3, D]``, ``stamps [nb, W]`` (realtime) or None, ``key_start`` int32 ``[nb]``."""
        m = self.model
        directions = m._persp_directions(square_bboxes[:, None], focal[:, None], princpt[:, None])
        tok = m._frame_tokens(patches.contiguous(), directions.reshape(patches.shape[0], -1))  # [nb, 3, D]
        ts = None if self.stamps is None else timestamp.to(torch.float32).contiguous()
        return ops.stream_update(tok.contiguous(), ids, reset, self.tokens, self.hist, self.head, ts, self.stamps)

    def _predictions(self, pose_aa, shape, root_transl_norm) -> Dict[str, torch.Tensor]:
        joint_cam, verts_cam, root_transl = self.model._pose_fk(pose_aa, shape, root_transl_norm)
        return {"joint_cam": joint_cam, "verts_cam": verts_cam, "pose_aa": pose_aa, "shape": shape,
                "root_transl_norm": root_transl_norm, "root_transl": root_transl}

    def _empty(self) -> Dict[str, torch.Tensor]:
        """The outputs of a step on no frames."""
        m, dev = self.model, self.tokens.device
        J, V = m.J_regressor_mano.shape
        shapes = {"joint_cam": (J, 3), "verts_cam": (V, 3), "pose_aa": (m.num_pose_query, 3), "shape": (10,),
                  "root_transl_norm": (3,), "root_transl": (3,)}
        return {k: torch.empty(0, 1, *s, device=dev) for k, s in shapes.items()}

    def _advance(self, patches, square_bboxes, timestamp, focal, princpt, reset, ids) -> Dict[str, torch.Tensor]:
        raise NotImplementedError

    def _stage_ids(self, ids: torch.Tensor, nb: int) -> None:
        """``self._ids[:nb]`` = ids padded with -1, by one host-to-device copy from a pinned buffer (no device sync)."""
        k = self._ticks % 2
        self._ticks += 1
        if self._ids_copied[k] is not None:
            self._ids_copied[k].synchronize()
        host = self._ids_host[k]
        host[:ids.numel()].copy_(ids)
        host[ids.numel():nb].fill_(-1)
        self._ids[:nb].copy_(host[:nb], non_blocking=True)
        self._ids_copied[k] = torch.cuda.Event()
        self._ids_copied[k].record()

    def _run_static(self, nb: int):
        i = self.static_in
        return self._advance(*(i[k][:nb] for k in KEYS), i["reset"][:nb], self._ids[:nb])

    def _capture(self, nb: int) -> None:
        self._ids[:nb].fill_(-1)               # the warm-up steps run on padding rows only: they leave the state untouched
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(2):                # populates the packed-weight caches for this batch size
                warm = self._run_static(nb)
        torch.cuda.current_stream().wait_stream(side)
        if self.static_out is None:
            self.static_out = {k: torch.empty((self.max_batch,) + v.shape[1:], dtype=v.dtype, device=v.device) for k, v in warm.items()}
        del warm
        torch.cuda.synchronize()
        if self._pool is None:
            self._pool = torch.cuda.graph_pool_handle()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, pool=self._pool), torch.no_grad():
            for k, v in self._run_static(nb).items():
                self.static_out[k][:nb].copy_(v)
        self.graphs[nb] = graph

    def step(self, patches: torch.Tensor, square_bboxes: torch.Tensor, timestamp: torch.Tensor, focal: torch.Tensor,
             princpt: torch.Tensor, reset: Optional[torch.Tensor] = None,
             streams: Union[None, Sequence[int], torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        ids = _stream_ids(streams, self.num_streams, self.max_batch)
        n = ids.numel()
        inputs = dict(zip(KEYS, (patches, square_bboxes, timestamp, focal, princpt)))
        _check_rows(n, inputs, reset)
        if not patches.is_cuda:
            raise RuntimeError(f"{type(self).__name__}.step runs on CUDA tensors only (there is no CPU fallback)")
        if n == 0:
            return self._empty()
        if not self.use_graph:
            self._stage_ids(ids, n)
            with torch.no_grad():
                return self._advance(*inputs.values(), None if reset is None else reset.contiguous(), self._ids[:n])
        nb = bucket(n, self.max_batch)
        if self.static_in is None:
            self.static_in = {k: torch.empty((self.max_batch,) + v.shape[1:], dtype=v.dtype, device=patches.device)
                              for k, v in inputs.items()}
            self.static_in["reset"] = torch.zeros(self.max_batch, dtype=torch.bool, device=patches.device)
        static = self.static_in
        for k, v in inputs.items():
            if v.data_ptr() != static[k].data_ptr():
                static[k][:n].copy_(v, non_blocking=True)
            if nb > n:                        # padding rows: copies of a real row, so every op sees ordinary values
                static[k][n:nb].copy_(static[k][:1].expand((nb - n,) + static[k].shape[1:]))
        if reset is None:
            static["reset"][:n].zero_()
        elif reset.data_ptr() != static["reset"].data_ptr():
            static["reset"][:n].copy_(reset, non_blocking=True)
        if nb not in self.graphs:
            self._capture(nb)
        self._stage_ids(ids, nb)
        self.graphs[nb].replay()
        return {k: v[:n] for k, v in self.static_out.items()}

class RealtimeStream(_TokenWindow):
    """Per-stream history of a realtime ``Poser`` for ``num_streams`` streams and a window of ``window`` frames.

    ``step(patches [n,3,S,S], square_bboxes [n,4], timestamp [n], focal [n,2], princpt [n,2], reset=None, streams=None)`` adds
    one frame to each of the n streams ``streams`` (distinct indices in [0, num_streams), a list or a CPU integer tensor, at most
    ``max_batch`` of them; None = every stream in order) and returns ``predict_batch``'s dict with T' = 1: row i is the
    prediction for the newest frame of stream ``streams[i]``.  ``reset`` (bool ``[n]``) drops a stream's history before this
    frame is added.  A stream that is not in ``streams`` is not touched: its tokens, timestamps and history length stay as they
    are.  Contract: after a reset (or the start) stream b has received frames f_1..f_t, in any pattern of steps; ``step``'s
    output for f_t is bit-identical to ``model.predict_batch`` on the one clip f_max(1, t-window+1)..f_t of that stream.  The
    model sees the gaps between a stream's frames through their timestamps.

    Device state, updated with no host synchronisation by one kernel per step (``ops.stream_update``): tokens ``[num_streams,
    window, 3, D]`` fp32 and timestamps ``[num_streams, window]``, a ring per stream, the history length ``hist`` and the ring
    head ``[num_streams]`` int32.

    With ``graph=True`` each step replays a CUDA graph of its bucket (``bucket(n, max_batch)`` rows), captured the first time the
    bucket is used (two warm-up steps on padding rows first, which change no state).  The graphs share one memory pool, and
    their inputs and outputs are the leading rows of ``max_batch``-row buffers.  The returned tensors are views of those
    buffers: clone them if they must outlive the next step.  The graphs hold the packed weights of their capture: after
    changing the weights call ``recapture()``.  ``step`` with no streams returns empty outputs and launches nothing.
    """

    def __init__(self, model, num_streams: int, window: int, graph: bool = True, max_batch: Optional[int] = None):
        _check_session("RealtimeStream", "realtime", model, num_streams, window, max_batch)
        super().__init__(model, num_streams, window, graph, max_batch)
        self.stamps = torch.zeros(num_streams, window, device=self.tokens.device)

    def _advance(self, patches, square_bboxes, timestamp, focal, princpt, reset, ids) -> Dict[str, torch.Tensor]:
        window, stamps, key_start = self._push(patches, square_bboxes, timestamp, focal, princpt, reset, ids)
        return self._predictions(*self.model._temporal_decode(window, stamps, key_start))


class FullTemporalStream(_TokenWindow):
    """Per-stream history of a full temporal ``Poser`` (``temporal_supervision="full"``) for ``num_streams`` streams, a window
    of ``window`` frames and a fixed output lag of ``lag`` frames.

    ``step(patches [n,3,S,S], square_bboxes [n,4], timestamp [n], focal [n,2], princpt [n,2], reset=None, streams=None)`` adds
    one frame to each of the n streams ``streams`` (as in ``RealtimeStream``) and returns ``predict_batch``'s dict with T' = 1,
    plus ``"valid"`` (bool ``[n]``), row i for stream ``streams[i]``.  ``reset`` (bool ``[n]``) drops a stream's history before
    this frame is added.  Timestamps are accepted and unused: the full model's positional encoding is absolute.  Contract: after
    a reset (or the start) stream b has received frames f_1..f_t, in any pattern of steps; let h = min(t, window).  Its
    ``valid`` is true iff h > lag, and then every output of stream b is bit-identical to ``model.predict_batch`` on the clip
    f_(t-h+1)..f_t of that stream, taken at frame index ``-1 - lag``: the prediction for f_(t-lag), which sees ``lag`` later
    frames.  Outputs of invalid streams are finite and carry no meaning.

    Device state: tokens ``[num_streams, window, 3, D]`` fp32 (a ring per stream), ``hist`` and the ring head ``[num_streams]``
    int32.  In the gathered window slot j of a stream takes the absolute position ``max(j - (window - h), 0)``, so its frames
    take the positions they have in its h-frame clip.  The decoded slot is ``window - 1 - lag`` for every stream; the output
    heads and the forward kinematics run on that slot alone.

    CUDA graphs, buckets and ``recapture()`` work as in ``RealtimeStream``.
    """

    def __init__(self, model, num_streams: int, window: int, lag: int = 0, graph: bool = True, max_batch: Optional[int] = None):
        _check_session("FullTemporalStream", "full", model, num_streams, window, max_batch)
        if not 0 <= lag <= window - 1:
            raise ValueError(f"lag must be in [0, window - 1] = [0, {window - 1}], got {lag}")
        super().__init__(model, num_streams, window, graph, max_batch)
        self.lag = lag

    def _empty(self) -> Dict[str, torch.Tensor]:
        out = super()._empty()
        out["valid"] = torch.empty(0, dtype=torch.bool, device=self.tokens.device)
        return out

    def _advance(self, patches, square_bboxes, timestamp, focal, princpt, reset, ids) -> Dict[str, torch.Tensor]:
        window, _, key_start = self._push(patches, square_bboxes, timestamp, focal, princpt, reset, ids)
        out = self._predictions(*self.model._temporal_decode(window, None, key_start, slot=self.window - 1 - self.lag))
        out["valid"] = key_start < self.window - self.lag          # h = window - key_start > lag
        return out
