"""PCGrad weight method on the B200 path — the surface train.py / engine.py use
(`WeightMethods('pcgrad', n_tasks=3, device=...)`, module/weight_methods.py:409-468, 727-761).

The per-task backward passes still go through torch.autograd.grad (one per task over the shared parameters, like
the reference :432-433).  The reference's fourth pass over the task-specific parameters (:443) is not run: those
gradients are folded from the per-task passes (ops.fold_task_grads).  The projection runs in
Gram space on the device: one pass for the T(T+1)/2 dots, a one-thread solve that replays the
reference's shuffle/dot/project loop, one combine pass.  The host never reads a dot product back, so the
`if g_i_g_j < 0` host sync of the reference (:455) is gone.  Python's global `random` is consumed exactly
like the reference (one in-place `random.shuffle` of the task list per outer task, SURVEY Q6).
"""
from __future__ import annotations

import random
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _ext
from . import distributed as mdist
from ._ext import call, fptr, ptr, stream
from .ops import deferred_wgrad_finish, fold_task_grads, wgrad_only_for


def draw_visit_orders(n_tasks: int, rng=None) -> List[List[int]]:
    """The task visit orders of _project_conflicting: the list is shuffled IN PLACE once per outer task, so
    permutations compound.  Consumes the RNG exactly like `random.shuffle(grads)` on a list of n_tasks."""
    shuffle = (rng or random).shuffle
    idx = list(range(n_tasks))
    orders = []
    for _ in range(n_tasks):
        shuffle(idx)
        orders.append(list(idx))
    return orders


_chunk_cache: Dict[Tuple[int, ...], Tuple[torch.Tensor, int]] = {}


def _chunk_table(numels: Sequence[int], device) -> Tuple[torch.Tensor, int]:
    key = (tuple(numels), str(device))
    ent = _chunk_cache.get(key)
    if ent is None:
        ck = _ext.load().mtd_pcgrad_chunk_elems()
        rows = [[s, off] for s, n in enumerate(numels) for off in range(0, n, ck)]
        ent = (_ext.device_table(rows, torch.int32, device), len(rows))
        _chunk_cache[key] = ent
    return ent


def _float_bits(x: float) -> int:
    return int(torch.tensor(x, dtype=torch.float32).view(torch.int32).item())


def pcgrad_merge(task_grads: Sequence[Sequence[Optional[torch.Tensor]]], orders, mean: bool,
                 seg_scales: Optional[Sequence[float]] = None, return_debug: bool = False):
    """merged_p = scale_p * sum_k coef_k * g_k[p] for every parameter p.

    task_grads[k][p] is task k's gradient for parameter p (None = the task has no gradient there).
    Returns the list of merged gradients (views into one flat buffer, parameter order preserved).
    """
    T = len(task_grads)
    P = len(task_grads[0])
    ref = next(g for tg in task_grads for g in tg if g is not None)
    device = ref.device
    shapes, numels = [], []
    for p in range(P):
        g = next((task_grads[k][p] for k in range(T) if task_grads[k][p] is not None), None)
        if g is None:
            raise _ext.MtdError("pcgrad_merge: parameter without any gradient needs an explicit shape")
        shapes.append(g.shape)
        numels.append(g.numel())
    flat = torch.empty(sum(numels), dtype=torch.float32, device=device)
    rows, off = [], 0
    keep = []
    for p in range(P):
        row = []
        for k in range(4):
            g = task_grads[k][p] if k < T else None
            if g is not None:
                g = g.contiguous()
                keep.append(g)
                row.append(fptr(g))
            else:
                row.append(0)
        scale = 1.0 if seg_scales is None else seg_scales[p]
        row += [flat.data_ptr() + 4 * off, numels[p], _float_bits(scale), 0]
        rows.append(row)
        off += numels[p]
    seg = _ext.device_table(rows, torch.int64, device)
    chunks, n_chunks = _chunk_table(numels, device)
    # `orders` is either a host list (copied through pinned staging) or an int32 device tensor [T*T] the caller
    # keeps refreshed (CUDA-graph replays)
    ords = orders if isinstance(orders, torch.Tensor) else _ext.device_table(orders, torch.int32, device)
    gram_ws = torch.empty(16, dtype=torch.float64, device=device)
    coef = torch.empty(4, dtype=torch.float32, device=device)
    cmat = torch.empty(T * T, dtype=torch.float32, device=device) if return_debug else None
    gram = torch.empty(T * T, dtype=torch.float64, device=device) if return_debug else None
    call("mtd_pcgrad_project", ptr(seg), ptr(chunks), n_chunks, T, ptr(ords), 1 if mean else 0, ptr(gram_ws), fptr(coef),
         fptr(cmat), ptr(gram), stream())
    merged, off = [], 0
    for p in range(P):
        merged.append(flat[off:off + numels[p]].view(shapes[p]))
        off += numels[p]
    if return_debug:
        return merged, {"coef": coef[:T], "C": cmat.view(T, T), "gram": gram.view(T, T), "flat": flat}
    return merged


def _cuda_gram(shards):
    """<shard_a, shard_b> for a <= b on the device (fp64), for distributed.pcgrad_sharded."""
    T, dev = len(shards), shards[0].device
    row = [fptr(s) for s in shards] + [0] * (4 - T) + [0, shards[0].numel(), _float_bits(1.0), 0]
    seg = _ext.device_table([row], torch.int64, dev)
    chunks, n_chunks = _chunk_table([shards[0].numel()], dev)
    gram = torch.empty(16, dtype=torch.float64, device=dev)
    call("mtd_pcgrad_gram", ptr(seg), ptr(chunks), n_chunks, T, ptr(gram), stream())
    return gram


def _cuda_solve_combine(shards, gram, orders, mean, scale):
    T, dev = len(shards), shards[0].device
    out = torch.empty_like(shards[0])
    row = [fptr(s) for s in shards] + [0] * (4 - T) + [fptr(out), out.numel(), _float_bits(scale), 0]
    seg = _ext.device_table([row], torch.int64, dev)
    chunks, n_chunks = _chunk_table([out.numel()], dev)
    ords = orders if isinstance(orders, torch.Tensor) else _ext.device_table(orders, torch.int32, dev)
    coef = torch.empty(4, dtype=torch.float32, device=dev)
    call("mtd_pcgrad_solve_combine", ptr(seg), ptr(chunks), n_chunks, T, ptr(ords), 1 if mean else 0, ptr(gram), fptr(coef),
         None, None, stream())
    return out


class WeightMethod:
    def __init__(self, n_tasks: int, device: torch.device):
        super().__init__()
        self.n_tasks = n_tasks
        self.device = device

    def get_weighted_loss(self, losses, **kwargs):
        raise NotImplementedError

    def backward(self, losses, shared_parameters=None, task_specific_parameters=None, last_shared_parameters=None,
                 representation=None, **kwargs):
        loss, extra_outputs = self.get_weighted_loss(
            losses=losses, shared_parameters=shared_parameters, task_specific_parameters=task_specific_parameters,
            last_shared_parameters=last_shared_parameters, representation=representation, **kwargs)
        loss.backward()
        return loss, extra_outputs

    def __call__(self, losses, **kwargs):
        return self.backward(losses, **kwargs)

    def parameters(self) -> List[torch.Tensor]:
        """return learnable parameters"""
        return []


class PCGrad(WeightMethod):
    """module/weight_methods.py:409-468.

    One backward pass per task (torch.autograd.grad over the shared parameters) gives the per-task shared gradients,
    projected in Gram space on the device.  The same passes fold the gradient of losses.sum() for the task-specific
    parameters (ops.fold_task_grads: their weight gradient is linear in each layer's dz, which every pass computes
    anyway), so the reference's fourth backward pass (:443) is not run; its result is the same up to fp32 summation
    order.  A task-specific parameter that no task loss reaches raises, like the reference's autograd.grad."""

    def __init__(self, n_tasks: int, device: torch.device, reduction="sum"):
        super().__init__(n_tasks, device=device)
        assert reduction in ["mean", "sum"]
        self.reduction = reduction

    def get_weighted_loss(self, losses, shared_parameters=None, task_specific_parameters=None, **kwargs):
        raise NotImplementedError

    def _set_pc_grads(self, losses, shared_parameters, task_specific_parameters=None):
        if isinstance(shared_parameters, torch.Tensor):
            shared_parameters = [shared_parameters]
        shared_parameters = list(shared_parameters)
        if task_specific_parameters is not None:
            if isinstance(task_specific_parameters, torch.Tensor):
                task_specific_parameters = [task_specific_parameters]
            task_specific_parameters = list(task_specific_parameters)
        if mdist.active():
            return self._set_pc_grads_distributed(losses, shared_parameters, task_specific_parameters)
        # shared part (:431-439): one backward pass per task, weight-gradient GEMMs only for the shared set; the task
        # specific part (:442-447, the gradient of losses.sum()) is folded from the same passes
        shared_grads = []
        with wgrad_only_for(shared_parameters), fold_task_grads(task_specific_parameters or []) as fold:
            for k, l in enumerate(losses):
                fold.last_pass = k + 1 == len(losses)
                with deferred_wgrad_finish():        # one batched finishing pass per task backward
                    shared_grads.append(torch.autograd.grad(l, shared_parameters, retain_graph=not fold.last_pass))
        merged = self._project_conflicting(shared_grads)
        for p, g in zip(shared_parameters, merged):
            p.grad = g
        if task_specific_parameters is not None:
            for p, g in zip(task_specific_parameters, fold.grads):
                p.grad = g

    def _set_pc_grads_distributed(self, losses, shared_parameters, task_specific_parameters):
        """Same gradients as the single-process path on the concatenated batch (SURVEY §8e), with the collectives
        overlapped: the reduce-scatter of each task's shared gradients proceeds on the communication stream while the
        next backward pass computes (distributed.py).  The all-reduce of the folded task-specific gradients follows the
        last pass and overlaps the sharded projection."""
        pipe = mdist.ShardedPCGrad()
        with wgrad_only_for(shared_parameters), fold_task_grads(task_specific_parameters or []) as fold:
            for k, l in enumerate(losses):
                fold.last_pass = k + 1 == len(losses)
                with deferred_wgrad_finish():
                    g = torch.autograd.grad(l, shared_parameters, retain_graph=not fold.last_pass)
                pipe.submit(g)
        ts_pending = mdist.allreduce_mean_list_async(fold.grads) if task_specific_parameters is not None else None
        orders = self.refresh_orders(shared_parameters[0].device)
        merged = pipe.finish(orders, self.reduction == "mean", _cuda_gram, _cuda_solve_combine)
        for p, g in zip(shared_parameters, merged):
            p.grad = g
        if ts_pending is not None:
            for p, g in zip(task_specific_parameters, ts_pending.wait()):
                p.grad = g

    def refresh_orders(self, device):
        """Draw this step's task visit orders from Python's `random` (exactly like the reference) into a persistent
        pinned buffer and enqueue its copy to a persistent device buffer.  A captured CUDA graph contains that copy
        node, so the graph runner only calls `draw_orders_host()` before each replay."""
        T = self.n_tasks
        if getattr(self, "_orders_host", None) is None or self._orders_dev.device != torch.device(device):
            self._orders_host = torch.zeros(T * T, dtype=torch.int32).pin_memory()
            self._orders_dev = torch.zeros(T * T, dtype=torch.int32, device=device)
        self.draw_orders_host()
        self._orders_dev.copy_(self._orders_host, non_blocking=True)
        return self._orders_dev

    def draw_orders_host(self):
        orders = draw_visit_orders(self.n_tasks)        # every rank draws the same orders (same `random` seed)
        self._orders_host.copy_(torch.tensor(orders, dtype=torch.int32).reshape(-1))
        return orders

    def _project_conflicting(self, grads: List[Tuple[torch.Tensor]]):
        assert len(grads) == self.n_tasks
        orders = self.refresh_orders(grads[0][0].device)
        if mdist.active():
            return mdist.pcgrad_sharded(grads, orders, self.reduction == "mean", _cuda_gram, _cuda_solve_combine)
        return pcgrad_merge(grads, orders, mean=(self.reduction == "mean"))

    def backward(self, losses, parameters=None, shared_parameters=None, task_specific_parameters=None, **kwargs):
        self._set_pc_grads(losses, shared_parameters, task_specific_parameters)
        return None, {}  # NOTE: to align with all other weight methods


class WeightMethods:
    """module/weight_methods.py:727-747.  Only `pcgrad` — the method the MTD-GAN recipe uses (README.md:82) —
    exists on the B200 path; the other ten reference methods are out of scope (SURVEY §2 #3b)."""

    def __init__(self, method: str, n_tasks: int, device: torch.device, **kwargs):
        assert method in list(METHODS.keys()), f"unknown method {method}."
        self.method = METHODS[method](n_tasks=n_tasks, device=device, **kwargs)

    def get_weighted_loss(self, losses, **kwargs):
        return self.method.get_weighted_loss(losses, **kwargs)

    def backward(self, losses, **kwargs):
        return self.method.backward(losses, **kwargs)

    def __ceil__(self, losses, **kwargs):
        return self.backward(losses, **kwargs)

    def parameters(self):
        return self.method.parameters()


METHODS = dict(pcgrad=PCGrad)
