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
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from .graph import KEYS

_MAX_WINDOW = 128          # key limit of the head's attention kernel (csrc/attention_simt.cu)


def _check_session(name: str, supervision: str, model, num_streams: int, window: int) -> None:
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


class _TokenWindow:
    """What both sessions share: the right-aligned per-stream spatial tokens ``[B, window, 3, D]`` fp32 and history lengths
    ``[B]`` int32 on the device, the per-frame part of a step, reset handling and the CUDA-graph capture.  Slots outside a
    stream's history hold zeros; the attention kernel never reads them as keys.  Subclasses implement ``_advance``."""

    def __init__(self, model, num_streams: int, window: int, graph: bool):
        model._check_positioning()
        dev = model.query_token.device
        if dev.type != "cuda":
            raise RuntimeError(f"{type(self).__name__} runs on CUDA only (there is no CPU fallback): move the model to the GPU first")
        self.model, self.num_streams, self.window = model, num_streams, window
        self.use_graph = graph
        B, W = num_streams, window
        self.tokens = torch.zeros(B, W, 3, model.hidden_dim, device=dev)
        self.hist = torch.zeros(B, dtype=torch.int32, device=dev)
        self._slot = torch.arange(W, dtype=torch.int32, device=dev)
        self.graph = None

    def recapture(self) -> None:
        """Drop the captured graph; the next ``step`` captures a new one (needed after the weights change)."""
        self.graph = None

    def _state(self):
        """The device tensors a step updates (saved and restored around the capture's warm-up steps)."""
        return [self.tokens, self.hist]

    def _push(self, patches, square_bboxes, focal, princpt, reset):
        """Runs the per-frame part on the new frames and shifts them into the window.  Returns ``key_start`` int32 ``[B]`` and
        the mask of each stream's history slots ``[B, window]``."""
        m, W = self.model, self.window
        directions = m._persp_directions(square_bboxes[:, None], focal[:, None], princpt[:, None])
        tok = m._frame_tokens(patches.contiguous(), directions.reshape(patches.shape[0], -1))  # [B, 3, D]
        hist = self.hist if reset is None else torch.where(reset, torch.zeros_like(self.hist), self.hist)
        hist = torch.clamp(hist + 1, max=W)
        key_start = W - hist
        valid = self._slot[None] >= key_start[:, None]                                          # [B, W]
        tokens = torch.cat([self.tokens[:, 1:], tok[:, None]], dim=1)
        self.tokens.copy_(torch.where(valid[:, :, None, None], tokens, torch.zeros((), device=tokens.device)))
        self.hist.copy_(hist)
        return key_start, valid

    def _predictions(self, pose_aa, shape, root_transl_norm) -> Dict[str, torch.Tensor]:
        joint_cam, verts_cam, root_transl = self.model._pose_fk(pose_aa, shape, root_transl_norm)
        return {"joint_cam": joint_cam, "verts_cam": verts_cam, "pose_aa": pose_aa, "shape": shape,
                "root_transl_norm": root_transl_norm, "root_transl": root_transl}

    def _advance(self, patches, square_bboxes, timestamp, focal, princpt, reset) -> Dict[str, torch.Tensor]:
        raise NotImplementedError

    def _capture(self, inputs) -> None:
        self.static_in = {k: v.clone(memory_format=torch.contiguous_format) for k, v in inputs.items()}
        state = [t.clone() for t in self._state()]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(2):                # populates the packed-weight caches and the allocator pool
                self._run_static()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph), torch.no_grad():
            self.static_out = self._run_static()
        for dst, src in zip(self._state(), state):     # undo the warm-up steps
            dst.copy_(src)
        self.graph = graph

    def _run_static(self):
        i = self.static_in
        return self._advance(*(i[k] for k in KEYS), i["reset"])

    def step(self, patches: torch.Tensor, square_bboxes: torch.Tensor, timestamp: torch.Tensor, focal: torch.Tensor,
             princpt: torch.Tensor, reset: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        B = self.num_streams
        if patches.dim() != 4 or patches.shape[0] != B or tuple(timestamp.shape) != (B,):
            raise ValueError(f"step takes one frame per stream: patches [{B},3,S,S] and timestamp [{B}], got "
                             f"{tuple(patches.shape)} and {tuple(timestamp.shape)}")
        if not patches.is_cuda:
            raise RuntimeError(f"{type(self).__name__}.step runs on CUDA tensors only (there is no CPU fallback)")
        if reset is not None and (reset.dtype != torch.bool or tuple(reset.shape) != (B,)):
            raise ValueError(f"reset must be a bool tensor of shape [{B}]")
        if not self.use_graph:
            with torch.no_grad():
                return self._advance(patches, square_bboxes, timestamp, focal, princpt, reset)
        if reset is None:
            reset = torch.zeros(B, dtype=torch.bool, device=patches.device)
        inputs = dict(zip(KEYS + ("reset",), (patches, square_bboxes, timestamp, focal, princpt, reset)))
        if self.graph is None:
            self._capture(inputs)
        for k, v in inputs.items():
            if v.data_ptr() != self.static_in[k].data_ptr():
                self.static_in[k].copy_(v, non_blocking=True)
        self.graph.replay()
        return self.static_out


class RealtimeStream(_TokenWindow):
    """Per-stream history of a realtime ``Poser`` for ``num_streams`` streams and a window of ``window`` frames.

    ``step(patches [B,3,S,S], square_bboxes [B,4], timestamp [B], focal [B,2], princpt [B,2], reset=None)`` adds one frame per
    stream and returns ``predict_batch``'s dict with T' = 1: the prediction for each stream's newest frame.  ``reset`` (bool
    ``[B]``) drops a stream's history before this frame is added.  Contract: after a reset (or the start) stream b has
    received frames f_1..f_t; ``step``'s output for f_t is bit-identical to ``model.predict_batch`` on the one clip
    f_max(1, t-window+1)..f_t of that stream.

    Device state, updated with no host synchronisation: tokens ``[B, window, 3, D]`` fp32 and timestamps ``[B, window]``,
    right-aligned with the newest frame in the last slot, and the history length ``[B]`` int32.  Slots outside a stream's
    history hold zeros and the newest timestamp; the attention kernel never reads them.

    With ``graph=True`` the first ``step`` captures the whole step as one CUDA graph (as ``cs_vit.graph.GraphedPredict``
    does: static input buffers, two warm-up steps whose effect on the history is undone) and every step replays it.  The
    returned tensors are views of static buffers: clone them if they must outlive the next step.  The graph holds the
    packed weights of the capture: after changing the weights call ``recapture()``.
    """

    def __init__(self, model, num_streams: int, window: int, graph: bool = True):
        _check_session("RealtimeStream", "realtime", model, num_streams, window)
        super().__init__(model, num_streams, window, graph)
        self.stamps = torch.zeros(num_streams, window, device=self.tokens.device)

    def _state(self):
        return super()._state() + [self.stamps]

    def _advance(self, patches, square_bboxes, timestamp, focal, princpt, reset) -> Dict[str, torch.Tensor]:
        key_start, valid = self._push(patches, square_bboxes, focal, princpt, reset)
        ts = timestamp.to(self.stamps.dtype)
        stamps = torch.cat([self.stamps[:, 1:], ts[:, None]], dim=1)
        self.stamps.copy_(torch.where(valid, stamps, ts[:, None]))
        return self._predictions(*self.model._temporal_decode(self.tokens, self.stamps, key_start))


class FullTemporalStream(_TokenWindow):
    """Per-stream history of a full temporal ``Poser`` (``temporal_supervision="full"``) for ``num_streams`` streams, a window
    of ``window`` frames and a fixed output lag of ``lag`` frames.

    ``step(patches [B,3,S,S], square_bboxes [B,4], timestamp [B], focal [B,2], princpt [B,2], reset=None)`` adds one frame per
    stream and returns ``predict_batch``'s dict with T' = 1, plus ``"valid"`` (bool ``[B]``).  ``reset`` (bool ``[B]``) drops a
    stream's history before this frame is added.  Timestamps are accepted and unused: the full model's positional encoding is
    absolute.  Contract: after a reset (or the start) stream b has received frames f_1..f_t; let h = min(t, window).
    ``valid[b]`` is true iff h > lag, and then every output of stream b is bit-identical to ``model.predict_batch`` on the clip
    f_(t-h+1)..f_t of that stream, taken at frame index ``-1 - lag``: the prediction for f_(t-lag), which sees ``lag`` later
    frames.  Outputs of invalid streams are finite and carry no meaning.

    Device state, updated with no host synchronisation: tokens ``[B, window, 3, D]`` fp32, right-aligned with the newest frame
    in the last slot, and the history length ``[B]`` int32.  Slot j of stream b takes the absolute position
    ``max(j - (window - h), 0)``, so a stream's frames take the positions they have in its h-frame clip.  The decoded slot is
    ``window - 1 - lag`` for every stream; the output heads and the forward kinematics run on that slot alone.

    CUDA graphs and ``recapture()`` work as in ``RealtimeStream``.
    """

    def __init__(self, model, num_streams: int, window: int, lag: int = 0, graph: bool = True):
        _check_session("FullTemporalStream", "full", model, num_streams, window)
        if not 0 <= lag <= window - 1:
            raise ValueError(f"lag must be in [0, window - 1] = [0, {window - 1}], got {lag}")
        super().__init__(model, num_streams, window, graph)
        self.lag = lag

    def _advance(self, patches, square_bboxes, timestamp, focal, princpt, reset) -> Dict[str, torch.Tensor]:
        key_start, _ = self._push(patches, square_bboxes, focal, princpt, reset)
        out = self._predictions(*self.model._temporal_decode(self.tokens, None, key_start, slot=self.window - 1 - self.lag))
        out["valid"] = self.hist > self.lag
        return out
