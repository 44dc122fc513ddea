"""Finetune-step host logic: the training loop body of ref:scripts/finetune.py:193-289 and its data-parallel gradient
reduction (DDP's bucketed allreduce, ref:scripts/finetune.py:133-135; SURVEY.md §2.2 C2).

``GradReducer`` is the NVLink-era replacement for ``DistributedDataParallel(find_unused_parameters=True)`` on this path:

* gradients are gathered into a few large flat fp32 buckets (default 64 MB: on NVSwitch the allreduce cost is launch
  latency + bytes / 900 GB/s, not per-link hops, so few large buckets beat DDP's 25 MB default) with one multi-tensor copy
  per bucket, and the optimizer reads them back as views - no per-parameter accumulate or unflatten kernels;
* a bucket's reduction is launched from the post-accumulate-grad hook of its last parameter, i.e. overlapped with the rest of
  the backward pass (buckets are ordered by reverse gradient-ready order, learned on step 1).  On the B200 box the buckets live
  in SYMMETRIC memory and the reduction is this library's own kernel (``csvit_allreduce_f32``, csrc/allreduce.cu: NVSwitch
  multicast ``multimem.ld_reduce`` / ``multimem.st`` when mapped, two-shot P2P loads / stores otherwise) on a high-priority side
  stream - small CTAs that co-reside with the persistent backward GEMMs, where NCCL's channels queue behind them; any other
  backend (gloo in the CPU tests) uses its ``all_reduce``;
* parameters that never receive a gradient (the five discarded "encoder" head layers, quirk Q2; frozen phases) are left
  out of the buckets instead of being searched for on every step (what ``find_unused_parameters=True`` does in the reference);
* ``finish()`` waits for the handles and scales by 1 / world once per bucket.

Works with any ``torch.distributed`` backend: NCCL on the B200 box, gloo in the CPU tests (tests/test_distributed.py).
"""
from __future__ import annotations

import math
import os
from typing import Dict, Iterable, List, Optional

import torch
import torch.distributed as dist


def scaled_lr(base_lr: float, world_size: int, batch_size: int, base_batch: int = 44) -> float:
    """Square-root learning-rate scaling of ref:scripts/finetune.py:138-139."""
    return math.sqrt(world_size * batch_size / base_batch) * base_lr


class GradReducer:
    def __init__(self, params: Iterable[torch.nn.Parameter], bucket_bytes: int = 64 << 20, group=None, comm: str = "auto"):
        """``comm``: ``"symm"`` = this library's allreduce kernel over symmetric (NVLink peer / NVSwitch multicast) memory,
        ``"nccl"`` = ``dist.all_reduce`` of the process group's backend, ``"auto"`` = symm for CUDA parameters under an NCCL
        group when the symmetric-memory rendezvous succeeds, else the backend's all_reduce (gloo in the CPU tests)."""
        self.params: List[torch.nn.Parameter] = [p for p in params if p.requires_grad]
        self.bucket_bytes = bucket_bytes
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        if comm not in ("auto", "symm", "nccl"):
            raise ValueError(f"comm must be auto / symm / nccl, got {comm!r}")
        self.comm = comm
        self.comm_ctas = int(os.environ.get("CSVIT_AR_CTAS", "0"))      # grid of the allreduce kernel (0 = library default), same on all ranks
        self.poison: Optional[torch.Tensor] = None   # device scalar (0 or NaN) folded into the first bucket flushed this step
        self._symm = None                     # {"buf", "handle", "ptrs", "mc", "flag_off"} once the symmetric buffer exists
        self._comm_stream = None
        self._events: List = []
        self._order: List[int] = []           # parameter indices in gradient-ready order (learned on the first step)
        self._buckets: Optional[List[dict]] = None
        self._bucket_of: Dict[int, int] = {}
        self._handles: List = []
        self._unbucketed: List[int] = []
        self._hooks = [p.register_post_accumulate_grad_hook(self._make_hook(i)) for i, p in enumerate(self.params)]

    # ------------------------------------------------------------------------------------------ hooks
    def _make_hook(self, i: int):
        def hook(param):
            if self._buckets is None:
                self._order.append(i)
                return
            b = self._bucket_of.get(i)
            if b is None:
                return                      # did not get a gradient on the first step: not bucketed (reduced in finish())
            bucket = self._buckets[b]
            bucket["pending"] -= 1
            if bucket["pending"] == 0:
                self._flush(bucket)
        return hook

    def _flush(self, bucket: dict) -> None:
        """All gradients of the bucket are ready: gather them into the flat buffer with ONE multi-tensor copy (instead of one
        accumulate kernel per parameter) and start the bucket's allreduce."""
        have = [(v, self.params[i].grad) for v, i in zip(bucket["views"], bucket["idxs"]) if self.params[i].grad is not None]
        if len(have) < len(bucket["idxs"]):
            bucket["flat"].zero_()
        if have:
            torch._foreach_copy_([v for v, _ in have], [g for _, g in have])
        bucket["flushed"] = True
        if self.poison is not None:          # a non-finite local loss must reach every rank: NaN in one element of one bucket
            bucket["flat"][:1].add_(self.poison)
            self.poison = None
        if self.world > 1:
            if self._symm is not None:
                # own kernel over peer memory on a high-priority side stream: forked here (the bucket is complete), joined in finish()
                from . import ops
                ready = torch.cuda.Event()
                ready.record()
                with torch.cuda.stream(self._comm_stream):
                    self._comm_stream.wait_event(ready)
                    sy = self._symm
                    off = bucket["offset"] * 4
                    ops.allreduce_f32([q + off for q in sy["ptrs"]], [q + sy["flag_off"] for q in sy["ptrs"]],
                                      sy["mc"] + off if sy["mc"] else 0, bucket["padded"], sy["rank"], self.world, 1.0 / self.world,
                                      ctas=self.comm_ctas)
                    done = torch.cuda.Event()
                    done.record()
                self._events.append(done)
            else:
                self._handles.append(dist.all_reduce(bucket["flat"], op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def _build(self) -> None:
        """After the first backward: bucket the parameters that received gradients, in gradient-ready order.  Every rank must
        issue the same collectives on the same buffers, so membership is the UNION over ranks (a parameter that got a gradient
        anywhere is bucketed everywhere) and the order is rank 0's."""
        order = list(self._order)
        if self.world > 1:
            dev = self.params[0].device if self.params else torch.device("cpu")
            present = torch.zeros(len(self.params), dtype=torch.int32, device=dev)
            if order:
                present[torch.tensor(order, device=dev)] = 1
            dist.all_reduce(present, op=dist.ReduceOp.MAX, group=self.group)
            seen = set(order)
            order += [i for i in torch.nonzero(present).flatten().tolist() if i not in seen]
            ranked = torch.tensor(order + [-1] * (len(self.params) - len(order)), dtype=torch.int64, device=dev)
            dist.broadcast(ranked, src=dist.get_global_rank(self.group, 0) if self.group is not None else 0, group=self.group)
            order = [i for i in ranked.tolist() if i >= 0]
        buckets, cur, cur_bytes = [], [], 0
        for i in order:
            p = self.params[i]
            nbytes = p.numel() * 4
            if cur and (cur_bytes + nbytes > self.bucket_bytes or p.device != self.params[cur[0]].device):
                buckets.append(cur)
                cur, cur_bytes = [], 0
            cur.append(i)
            cur_bytes += nbytes
        if cur:
            buckets.append(cur)
        self._buckets = []
        sizes = [sum(self.params[i].numel() for i in idxs) for idxs in buckets]
        padded = [(n + 3) // 4 * 4 for n in sizes]
        offsets = [sum(padded[:b]) for b in range(len(padded))]
        self._try_symmetric(sum(padded), buckets)
        for b, idxs in enumerate(buckets):
            dev = self.params[idxs[0]].device
            if self._symm is not None:
                flat = self._symm["buf"][offsets[b]:offsets[b] + sizes[b]]
            else:
                flat = self._alloc_flat(sizes[b], dev)
            views, off = [], 0
            for i in idxs:
                p = self.params[i]
                views.append(flat[off:off + p.numel()].view_as(p))
                off += p.numel()
                self._bucket_of[i] = b
            self._buckets.append({"flat": flat, "idxs": idxs, "views": views, "pending": len(idxs), "flushed": False,
                                  "offset": offsets[b], "padded": padded[b]})
        self._unbucketed = [i for i in range(len(self.params)) if i not in self._bucket_of]

    def _alloc_flat(self, numel: int, device) -> torch.Tensor:
        return torch.zeros(numel, dtype=torch.float32, device=device)

    def _try_symmetric(self, total: int, buckets: List[List[int]]) -> None:
        """One symmetric allocation for all buckets (16-byte aligned starts) + the barrier flags, mapped into every peer."""
        if self.world == 1 or self.comm == "nccl" or not buckets:
            return
        devs = {self.params[i].device for idxs in buckets for i in idxs}
        backend = dist.get_backend(self.group)
        if len(devs) != 1 or next(iter(devs)).type != "cuda" or "nccl" not in str(backend) or self.world > 8:
            if self.comm == "symm":
                raise RuntimeError(f"comm='symm' needs CUDA parameters on one device under an NCCL group of <= 8 ranks (backend {backend})")
            return
        dev = next(iter(devs))
        try:
            import torch.distributed._symmetric_memory as symm
            from .ops import ALLREDUCE_FLAG_BYTES
            group = self.group if self.group is not None else dist.group.WORLD
            buf = symm.empty(total + ALLREDUCE_FLAG_BYTES // 4, dtype=torch.float32, device=dev)
            buf.zero_()
            handle = symm.rendezvous(buf, group)
            ptrs = [int(q) for q in handle.buffer_ptrs]
            mc = int(getattr(handle, "multicast_ptr", 0) or 0)
            torch.cuda.synchronize(dev)
            dist.barrier(group=self.group)            # every rank's flags are zero before the first kernel touches them
            self._symm = {"buf": buf, "handle": handle, "ptrs": ptrs, "mc": mc, "flag_off": total * 4, "rank": dist.get_rank(self.group)}
            self._comm_stream = torch.cuda.Stream(device=dev, priority=-1)
        except Exception as e:      # no P2P mapping between these GPUs (or symmetric memory not built in): the backend's allreduce
            if self.comm == "symm":
                raise
            import warnings
            warnings.warn(f"GradReducer: symmetric-memory allreduce unavailable ({type(e).__name__}: {e}); using {backend} all_reduce")
            self._symm = None

    # ------------------------------------------------------------------------------------------ per-step API
    def zero_grad(self) -> None:
        """Gradients start every step as ``None``: autograd then hands each parameter a fresh tensor (no read-modify-write), which the
        bucket's flush copies into the flat buffer.  (Use this instead of ``optimizer.zero_grad``.)"""
        for p in self.params:
            p.grad = None
        for bucket in self._buckets or []:
            bucket["pending"] = len(bucket["idxs"])
            bucket["flushed"] = False

    def finish(self) -> None:
        """Call after ``loss.backward()``: completes the reduction and leaves the averaged gradients in ``param.grad`` (as views of
        the flat buckets)."""
        if self._buckets is None:
            self._build()
        for bucket in self._buckets:          # first step, or a bucket whose parameters did not all fire this step
            if not bucket["flushed"]:
                self._flush(bucket)
        for h in self._handles:
            h.wait()
        self._handles = []
        for done in self._events:              # join the side stream's allreduce kernels (they also applied the 1 / world)
            torch.cuda.current_stream().wait_event(done)
        self._events = []
        for bucket in self._buckets:
            if self.world > 1 and self._symm is None:
                bucket["flat"].mul_(1.0 / self.world)
            for v, i in zip(bucket["views"], bucket["idxs"]):
                # world > 1: every rank takes the averaged gradient, also a rank whose own gradient was None this step (its share
                # of the sum was zero) - otherwise the replicas drift apart (DDP find_unused_parameters semantics)
                if self.world > 1 or self.params[i].grad is not None:
                    self.params[i].grad = v
        capturing = torch.cuda.is_available() and torch.cuda.is_current_stream_capturing()
        if self.world > 1 and self._unbucketed and not capturing:      # (a captured step is static: what had no gradient never gets one)
            # a gradient that appears after step 1 (phase change): the set of parameters to reduce must be agreed on, so that
            # every rank issues the same collectives - one MAX-allreduced presence mask, then zeros stand in for absent gradients
            dev = self.params[self._unbucketed[0]].device
            present = torch.tensor([1 if self.params[i].grad is not None else 0 for i in self._unbucketed], dtype=torch.int32, device=dev)
            dist.all_reduce(present, op=dist.ReduceOp.MAX, group=self.group)
            for flag, i in zip(present.tolist(), self._unbucketed):
                if flag:
                    p = self.params[i]
                    if p.grad is None:
                        p.grad = torch.zeros_like(p, dtype=torch.float32)
                    dist.all_reduce(p.grad, op=dist.ReduceOp.SUM, group=self.group)
                    p.grad.mul_(1.0 / self.world)

    def bucket_summary(self) -> List[int]:
        return [b["flat"].numel() * 4 for b in (self._buckets or [])]

    @property
    def transport(self) -> str:
        """What moves the gradients: this library's kernel over NVSwitch multicast / NVLink P2P, or the backend's all_reduce."""
        if self.world == 1:
            return "none (single rank)"
        if self._symm is not None:
            return "csvit_allreduce_f32 over " + ("NVSwitch multicast (multimem.ld_reduce / multimem.st)" if self._symm["mc"] else "NVLink P2P loads / stores (two-shot)")
        return f"{dist.get_backend(self.group)} all_reduce"

    def remove(self) -> None:
        for h in self._hooks:
            h.remove()
        self._hooks = []


def broadcast_parameters(module: torch.nn.Module, src: int = 0, group=None) -> None:
    """DDP-constructor semantics (SURVEY.md §2.2 C1): every rank starts from rank ``src``'s parameters and buffers."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    with torch.no_grad():
        for t in list(module.parameters()) + list(module.buffers()):
            dist.broadcast(t, src=src, group=group)


def _all_ranks_finite(loss: torch.Tensor, group=None) -> bool:
    """True when the loss is finite on EVERY rank (one 4-byte MIN allreduce), so that all ranks skip a batch together."""
    ok = torch.isfinite(loss.detach()).to(torch.int32).reshape(1)
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
    return bool(ok.item())


skipped_steps = 0      # batches finetune_step() skipped because of a non-finite loss (ref:scripts/finetune.py:219-222 prints and continues)


def finetune_step(model: torch.nn.Module, batch: dict, optimizer: torch.optim.Optimizer, reducer: Optional[GradReducer] = None,
                  max_norm: float = 5.0) -> torch.Tensor:
    """One iteration of ref:scripts/finetune.py:211-227: forward (``Poser.forward`` -> loss), the reference's NaN guard (:219-222:
    a non-finite loss skips the batch BEFORE backward - here on every rank together, otherwise the gradient allreduce would
    deadlock or poison the healthy replicas), backward, gradient averaging across ranks, ``clip_grad_norm_(5.0)``, optimizer
    step (skipped too if the clipped norm is not finite).  Returns the detached loss."""
    global skipped_steps
    if getattr(model, "precision", None) == "fp8":
        raise ValueError("precision='fp8' is inference only: run the finetune step in bf16, fp16 or fp32")
    if reducer is not None:
        reducer.zero_grad()
    else:
        optimizer.zero_grad(set_to_none=True)
    out = model(batch)
    loss = out["loss"]
    if not _all_ranks_finite(loss, reducer.group if reducer is not None else None):
        skipped_steps += 1
        return loss.detach()
    loss.backward()
    if reducer is not None:
        reducer.finish()
    total = torch.nn.utils.clip_grad_norm_([p for p in model.parameters() if p.grad is not None], max_norm)
    if not bool(torch.isfinite(total).item()):      # (identical on every rank: computed from the averaged gradients)
        skipped_steps += 1
        return loss.detach()
    optimizer.step()
    return loss.detach()


def invalidate_packs(model: torch.nn.Module) -> None:
    """Drop every module's packed (16-bit / stacked) parameter copies.  Needed before EAGER use of a model whose optimizer steps
    ran inside a replayed CUDA graph: replays do not bump ``Tensor._version``, which is what ``PackCache`` watches."""
    for m in model.modules():
        pack = getattr(m, "_pack", None)
        if pack is not None:
            pack.clear()


class GraphedFinetuneStep:
    """The finetune step (zero grads, forward, loss, backward, gradient reduction, clip, optimizer) as ONE CUDA graph.

    At the reference's batch size (32 per GPU) the eager step is bound by the ~2300 host launches it issues (37 ms for 26 ms of
    GPU work on B200).  Everything in the step is stream-ordered device work with static shapes - the kernels of this library,
    torch's fp32 tail, ``clip_grad_norm_`` and a ``capturable`` fused AdamW - so after a few eager warm-up steps (which also
    build the reducer's buckets and the optimizer state) the whole step is captured once and replayed.  Inputs are copied
    into static buffers; the loss and its components are read from static output tensors (no ``.item()`` inside the step:
    ``Poser.loss_tensors``).  The optimizer must have been created with ``fused=True, capturable=True``.  A non-finite loss or
    gradient norm suppresses that step's update on the device (``found_inf``); ``skipped_steps`` counts them.  Call ``invalidate_packs(model)``
    before using the model eagerly again (evaluation between epochs).
    """

    def __init__(self, model: torch.nn.Module, batch: dict, optimizer: torch.optim.Optimizer, reducer: Optional[GradReducer] = None,
                 max_norm: float = 5.0, warmup: int = 3):
        if getattr(model, "precision", None) == "fp8":
            raise ValueError("precision='fp8' is inference only: run the finetune step in bf16, fp16 or fp32")
        self.model, self.optimizer, self.reducer, self.max_norm = model, optimizer, reducer, max_norm
        self.static = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in batch.items()}
        self.params = [p for p in model.parameters() if p.requires_grad]
        if reducer is None:
            self.reducer = GradReducer(self.params)      # also world size 1: keeps .grad in stable flat buffers for the graph
        dev = self.params[0].device
        self.found_inf = torch.zeros((), dtype=torch.float32, device=dev)      # 0-d, like GradScaler's (the fused kernel broadcasts it)
        self.skipped = torch.zeros((), dtype=torch.float32, device=dev)
        if not getattr(optimizer, "_step_supports_amp_scaling", False):
            raise ValueError("GraphedFinetuneStep needs a fused optimizer that honours `found_inf` (torch.optim.AdamW(fused=True, capturable=True))")
        optimizer.grad_scale, optimizer.found_inf = None, self.found_inf
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 2)):
                self._step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        from . import ops
        n0 = ops.launch_count
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, self.parts = self._step()
        self.launches_per_step = ops.launch_count - n0      # C-ABI kernel launches one replay stands for

    def _step(self):
        self.reducer.zero_grad()
        loss, parts, _ = self.model.loss_tensors(self.static)
        # Device-side guard (no host check is possible inside a graph), GradScaler's mechanism: the fused AdamW kernel is a no-op -
        # parameters, both moments and the step count untouched - when ``found_inf`` is non-zero.  The flag must be the same on
        # every rank: a non-finite local loss poisons one element of the first gradient bucket with NaN, the allreduce carries it
        # to every rank, and the norm of the AVERAGED gradients (identical everywhere) is what is tested - no extra collective.
        zero = torch.zeros((), dtype=torch.float32, device=loss.device)
        self.reducer.poison = torch.where(torch.isfinite(loss.detach()), zero, zero + float("nan")).reshape(1)
        loss.backward()
        self.reducer.finish()
        total = torch.nn.utils.clip_grad_norm_([p for p in self.params if p.grad is not None], self.max_norm)
        bad = (~torch.isfinite(total)).to(torch.float32).reshape(())
        self.found_inf.copy_(bad)
        self.skipped.add_(bad)
        self.optimizer.step()
        return loss.detach(), parts

    @property
    def skipped_steps(self) -> int:
        """Steps whose update was suppressed because the loss or the gradient norm was not finite (host sync)."""
        return int(self.skipped.item())

    def __call__(self, batch: dict) -> torch.Tensor:
        for k, v in batch.items():
            if torch.is_tensor(v) and v.data_ptr() != self.static[k].data_ptr():
                self.static[k].copy_(v, non_blocking=True)
        self.graph.replay()
        return self.loss
