"""Autograd-connected host wrappers over the C-ABI kernels.  All activations are NHWC fp32 CUDA
tensors of shape (B, H, W, C); every op is a torch.autograd.Function whose forward AND backward are
calls into libmtdgan_sm100a.so — PyTorch supplies memory, streams and the autograd tape only.
"""
from __future__ import annotations

import os
import weakref
from dataclasses import dataclass


import torch
from torch.autograd import Function

from . import _ext
from ._ext import call, fptr, ptr, stream

ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
LEAK = 0.2


def _empty(shape, like):
    return torch.empty(shape, dtype=torch.float32, device=like.device)


# ------------------------------------------------------------------------------------------------
# packed-weight cache: reference-layout Parameters stay the masters (state_dict / optimizer
# compatible); K-major packed copies are rebuilt when the parameter's version counter or storage moves.
# ------------------------------------------------------------------------------------------------
_pack_cache: dict = {}        # id(weight object) -> {(kind, transposed, stride): (tag, packed)}


def clear_pack_cache():
    """Invalidate every packed copy (used before CUDA-graph capture so the packing kernels are captured too).  The
    registry of (weight, kind, cfg) stays, so `repack_stale()` can rebuild everything in a few batched launches.

    Packed copies are keyed on the parameter's version counter and storage pointer.  Writes through `p.data`
    (`p.data.normal_()`, weight clipping, EMA swaps) do NOT move the version counter: call this function (exported as
    `mtdgan_b200.invalidate_weight_caches()`) after such a write, or write under `torch.no_grad()` on `p` itself.
    Construction-time `.data` init (the reference's `__init_weights`) and `load_state_dict` need nothing: the first
    runs before any pack exists, the second bumps the version."""
    for slot in _pack_cache.values():
        for key, ent in list(slot.items()):
            slot[key] = (None,) + tuple(ent[1:])


def _cache_slot(weight) -> dict:
    k = id(weight)
    slot = _pack_cache.get(k)
    if slot is None:
        slot = {}
        _pack_cache[k] = slot
        weakref.finalize(weight, _pack_cache.pop, k, None)     # entry dies with the tensor object
    return slot


def _pack_into(w: torch.Tensor, kind: str, cfg: "ConvCfg", out: torch.Tensor):
    if "_tf32" in kind:
        # tensor-core packs: tile-major (blocked) layout with the TF32 rounding ([hi | lo] split for 3xTF32) fused in
        mode = 3 if kind.endswith("_tf32x3") else 1
        if kind.startswith("fwd"):
            call("mtd_conv_pack_fwd_blocked", fptr(w), cfg.transposed, cfg.cout, cfg.cin, cfg.kh, cfg.kw, mode, fptr(out),
                 stream())
        else:
            call("mtd_conv_pack_dgrad_blocked", fptr(w), cfg.transposed, cfg.cout, cfg.cin, cfg.kh, cfg.kw, cfg.stride, mode,
                 fptr(out), stream())
    elif kind.startswith("fwd"):
        call("mtd_conv_pack_fwd", fptr(w), cfg.transposed, cfg.cout, cfg.cin, cfg.kh, cfg.kw, fptr(out), stream())
    else:
        call("mtd_conv_pack_dgrad", fptr(w), cfg.transposed, cfg.cout, cfg.cin, cfg.kh, cfg.kw, cfg.stride, fptr(out),
             stream())


def _packed(weight: torch.Tensor, kind: str, cfg: "ConvCfg") -> torch.Tensor:
    """K-major packed copy of a reference-layout weight.  Cached per weight OBJECT (weakly: entries die
    with the parameter, so a recycled allocation can never alias a stale entry) and invalidated by the
    tensor's version counter / storage pointer.  Cache entry: (tag, packed, weakref(weight), kind, cfg)."""
    slot = _cache_slot(weight)
    key = (kind, cfg.transposed, cfg.stride)
    tag = (weight._version, weight.data_ptr())
    ent = slot.get(key)
    if ent is not None and ent[0] == tag:
        return ent[1]
    w = weight.detach()
    n = w.numel() * (2 if kind.endswith("_tf32x3") else 1)
    # A stale entry is re-packed IN PLACE: a captured CUDA graph holds the buffer's address (its convolutions read it,
    # its batched re-pack writes it), so the buffer must live exactly as long as the weight does
    out = ent[1] if (ent is not None and ent[1] is not None and ent[1].numel() == n and ent[1].device == w.device) else _empty((n,), w)
    _pack_into(w, kind, cfg, out)
    slot[key] = (tag, out, weakref.ref(weight), kind, cfg)
    return out


def repack_stale(params=None) -> int:
    """Rebuild, in a few BATCHED launches (24 packs per kernel), every registered packed copy whose weight has changed
    since it was packed (optimizer step, load_state_dict, cache invalidation).  `params` restricts it to those
    parameters.  Layers pack lazily on first use anyway; calling this once after each optimizer step replaces ~230
    per-layer pack launches per train step by ~10.  Returns the number of packs rebuilt."""
    want = None if params is None else {id(p) for p in params}
    todo = []
    for wid, slot in _pack_cache.items():
        if want is not None and wid not in want:
            continue
        for key, ent in slot.items():
            if len(ent) < 5:
                continue
            weight = ent[2]()
            if weight is None or not weight.is_cuda:
                continue
            tag = (weight._version, weight.data_ptr())
            if ent[0] != tag:
                todo.append((slot, key, ent, weight, tag))
    if not todo:
        return 0
    call("mtd_conv_pack_batch_begin")
    try:
        for slot, key, ent, weight, tag in todo:
            kind, cfg = ent[3], ent[4]
            w = weight.detach()
            n = w.numel() * (2 if kind.endswith("_tf32x3") else 1)
            out = ent[1] if (ent[1] is not None and ent[1].numel() == n and ent[1].device == w.device) else _empty((n,), w)
            _pack_into(w, kind, cfg, out)
            slot[key] = (tag, out, ent[2], kind, cfg)
    finally:
        call("mtd_conv_pack_batch_end", stream())
    return len(todo)


# Weight-gradient request filter.  torch.autograd.grad(l, inputs=...) prunes built-in ops' unused
# outputs, but a Python Function only sees the static `needs_input_grad`; the PCGrad driver
# (weight_methods.py) names the parameters it is asking for so the other layers skip their wgrad GEMMs.
_wgrad_filter = None          # None = compute for every weight that requires grad


class wgrad_only_for:
    def __init__(self, params):
        self.ptrs = None if params is None else {p.data_ptr() for p in params}

    def __enter__(self):
        global _wgrad_filter
        self.prev, _wgrad_filter = _wgrad_filter, self.ptrs
        return self

    def __exit__(self, *exc):
        global _wgrad_filter
        _wgrad_filter = self.prev
        return False


def _wgrad_wanted(weight) -> bool:
    return _wgrad_filter is None or weight.data_ptr() in _wgrad_filter


# Deferred weight-gradient finishing.  Inside `deferred_wgrad_finish()` (the PCGrad driver wraps each of its
# torch.autograd.grad calls in one) a layer only queues its packed gradient.  The FIRST forward instance of a weight
# to run its backward returns the (still unfilled) dw tensor, later instances of the same weight return None, and
# when the context exits one batched dot + one batched unpack launch finish every layer AND sum the instances —
# replacing ~500 per-layer launches and autograd's ~600 gradient-accumulation adds per train step.  The dw tensors
# are only consumed after autograd.grad returns, so filling them late is safe; under plain `.backward()`
# (AccumulateGrad may clone or accumulate immediately) finishing stays immediate.
_finish_queue = None          # None, or {weight data_ptr: (dw, [instance tuples])}
_fin_chunk_cache: dict = {}


# Weight-gradient GEMMs are off the critical path of a backward pass (nothing consumes them before the batched
# finishing at the end of the autograd.grad call), so inside a deferred-finishing context they can be issued on a side
# stream and overlap the act_bwd -> dgrad chain of the following layers (MTDGAN_WGRAD_STREAM=0 disables it; in a captured
# step the side stream becomes a parallel branch of the graph; measured 43.1 -> 42.5 ms per step).  Their operands are kept alive until the join.
_WGRAD_SIDE = os.environ.get("MTDGAN_WGRAD_STREAM", "1") == "1"
_side_streams: dict = {}
_side_keepalive: list = []
_side_used = False


def _on_side_stream(fn, *keep):
    """Run fn() on the side stream after everything queued so far on the current stream."""
    global _side_used
    main = torch.cuda.current_stream()
    key = (main.device.index, main.cuda_stream)
    side = _side_streams.get(key)
    if side is None:
        side = _side_streams[key] = torch.cuda.Stream(device=main.device)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        fn()
    _side_keepalive.extend(keep)
    _side_used = True


def _join_side_stream():
    global _side_used
    if _side_used:
        main = torch.cuda.current_stream()
        side = _side_streams.get((main.device.index, main.cuda_stream))
        if side is not None:
            main.wait_stream(side)
        _side_used = False


class deferred_wgrad_finish:
    def __enter__(self):
        global _finish_queue, _bias_slab, _zw_slab
        self.prev, _finish_queue = _finish_queue, {}
        self.prev_slab, _bias_slab = _bias_slab, None
        self.prev_zw, _zw_slab = _zw_slab, None
        return self

    def __exit__(self, *exc):
        global _finish_queue, _bias_slab, _zw_slab
        q, _finish_queue = _finish_queue, self.prev
        zw_keepalive = _zw_slab               # the finishing kernels read the <G, W~> accumulators through raw pointers
        _bias_slab = self.prev_slab
        _zw_slab = self.prev_zw
        _join_side_stream()
        if q and exc[0] is None:
            _flush_finish(q)
        del zw_keepalive
        _side_keepalive.clear()
        return False


# Bias gradients are column sums accumulated with atomics, i.e. they need zeroed memory.  Inside a deferred-finishing
# context (one per PCGrad autograd.grad call, ~250 layers) they are carved from ONE zeroed slab instead of one memset
# node per layer.
_BIAS_SLAB_FLOATS = 1 << 18
_bias_slab = None             # [tensor, next free offset] of the active context


_zw_slab = None               # [float64 tensor, next free offset]: <G, W~> accumulators of the active context


def _zw_alloc(n: int, like):
    """n zeroed doubles for mtd_act_bwd_sn (only inside a deferred-finishing context)."""
    global _zw_slab
    if _zw_slab is None:
        _zw_slab = [torch.zeros(8192, dtype=torch.float64, device=like.device), 0]
    t, off = _zw_slab
    if off + n > t.numel():
        return None                          # slab exhausted: the caller falls back to the dot pass
    _zw_slab[1] = off + n
    return t[off:off + n]


def _dbias_alloc(n: int, like):
    """-> (dbias tensor, 1 if it is known to be all zero else 0)"""
    global _bias_slab
    if _finish_queue is not None:
        if _bias_slab is None:
            _bias_slab = [torch.zeros(_BIAS_SLAB_FLOATS, dtype=torch.float32, device=like.device), 0]
        t, off = _bias_slab
        step = (n + 63) // 64 * 64                      # keep every slice 256-byte aligned
        if off + step <= t.numel():
            _bias_slab[1] = off + step
            return t[off:off + n], 1
    return _empty((n,), like), 0


def _flush_finish(groups):
    first = next(iter(groups.values()))
    dev = first[0].device
    rows, dot_numels, head_numels, heads, rowdims = [], [], [], [], []
    for dw, insts in groups.values():
        base = len(rows)
        heads.append(base)
        head_numels.append(dw.numel())
        for k, (gp, w, u, v, inv, cfg, zwp, flags) in enumerate(insts):
            T = cfg.kh * cfg.kw
            sN, sC, flip = (T, cfg.cout * T, 1) if cfg.transposed else (cfg.cin * T, T, 0)
            sn = inv is not None
            rows.append([gp.data_ptr() if gp is not None else 0, dw.data_ptr(), w.data_ptr() if sn else 0,
                         u.data_ptr() if sn else 0, v.data_ptr() if sn else 0, inv.data_ptr() if sn else 0, cfg.cout, T, cfg.cin,
                         sN, sC, flip | flags,
                         cfg.cin * T, base + k, base + k + 1 if k + 1 < len(insts) else -1, zwp])
            dot_numels.append(gp.numel() if (sn and not zwp and gp is not None) else 0)
            rowdims.append((T, cfg.cin))
    key = (tuple(dot_numels), tuple(heads), tuple(rowdims), str(dev))
    ent = _fin_chunk_cache.get(key)
    if ent is None:
        ck = [_ext.load().mtd_wgrad_finish_chunk_elems(t, c) for t, c in rowdims]     # whole packed rows per chunk
        dchunks = [[s_, off] for s_, n in enumerate(dot_numels) for off in range(0, n, ck[s_])]
        hchunks = [[h, off] for h, n in zip(heads, head_numels) for off in range(0, n, ck[h])]
        ent = (_ext.device_table(dchunks, torch.int32, dev) if dchunks else None, len(dchunks),
               _ext.device_table(hchunks, torch.int32, dev), len(hchunks))
        _fin_chunk_cache[key] = ent
    seg = _ext.device_table(rows, torch.int64, dev)
    dots = torch.empty(len(rows), dtype=torch.float64, device=dev)
    call("mtd_wgrad_finish_batched", ptr(seg), len(rows), ptr(ent[0]), ent[1], ptr(ent[2]), ent[3], ptr(dots), stream())


# Task-gradient fold.  PCGrad needs, besides the per-task gradients of the shared parameters, the gradient of the SUM of
# the task losses for the task-specific parameters.  Each task-specific layer lies on the path from some task loss to
# the shared encoder, so the per-task backward passes already compute its dz (the gradient at its pre-activation) for
# their task; its weight gradient (x (x) dz), bias gradient (sum dz) and spectral-norm correction (linear in G) are
# linear in dz, and the activation masks are the same in every pass.  Inside `fold_task_grads(params)` a layer whose
# weight is in `params` folds each pass's dz into one accumulator per forward instance (mtd_act_bwd_acc, in place of
# its plain activation backward) and issues nothing for its weight; one weight-gradient GEMM per instance and one
# batched finishing pass then give the same gradients as a separate backward pass of the summed loss, without it.
_fold = None                  # the active fold_task_grads, or None


class _FoldRec:
    """One forward instance (autograd node) of a folded layer."""

    def __init__(self, node, weight, x1, x2, dz_like, bias_grad, inv_sigma, u, v, zw, cfg, shapes):
        self.node = node                    # keeps id(node), the record's key, from being reused
        self.weight, self.x1, self.x2 = weight, x1, x2
        self.acc = _empty(dz_like.shape, dz_like)
        self.bias_grad, self.inv_sigma, self.u, self.v, self.zw = bias_grad, inv_sigma, u, v, zw
        self.cfg, self.shapes = cfg, shapes
        self.gp = None                      # packed weight gradient, once its GEMM is issued


class fold_task_grads:
    """Folds the task-specific gradients of several backward passes over one graph (see above).  Set `last_pass`
    before the final pass: each instance's weight-gradient GEMM is then issued as soon as that pass has folded it, and
    runs on the side stream alongside the rest of the pass.  After the context exits, `grads` holds the gradient of
    every parameter in `params`, in order."""

    def __init__(self, params):
        self.params = list(params)
        self.ptrs = {p.data_ptr() for p in self.params}
        self.records = {}                   # id(autograd node) -> _FoldRec
        self.bias_grads = {}                # bias data_ptr -> accumulated gradient (zeroed slab slice)
        self.last_pass = False
        self.grads = None
        self._fslab = self._dslab = None

    def __enter__(self):
        global _fold
        self.prev, _fold = _fold, self
        return self

    def __exit__(self, *exc):
        global _fold
        _fold = self.prev
        if exc[0] is None:
            self.grads = self._finish()
        self.records = {}
        return False

    def wants(self, weight) -> bool:
        return weight.data_ptr() in self.ptrs

    def _zeros(self, n, dtype, like):
        """n zeroed entries carved from one slab per fold (one memset instead of one per accumulator)."""
        f = dtype == torch.float32
        slab = self._fslab if f else self._dslab
        if slab is None:
            slab = [torch.zeros(1 << 16 if f else 1024, dtype=dtype, device=like.device), 0]
            if f:
                self._fslab = slab
            else:
                self._dslab = slab
        step = (n + 63) // 64 * 64                     # 256-byte aligned slices
        if slab[1] + step > slab[0].numel():
            return torch.zeros(n, dtype=dtype, device=like.device)
        t = slab[0][slab[1]:slab[1] + n]
        slab[1] += step
        return t

    def act_bwd(self, node, g1, pre_out, weight, bias, want_bias, inv_sigma, u, v, x1, x2, cfg: "ConvCfg", shapes, has_add):
        """Activation backward of a folded layer: returns this pass's (unscaled) dz and folds it into the instance's
        accumulators."""
        sn = inv_sigma is not None
        G = inv_sigma.numel() if sn else 1
        rec = self.records.get(id(node))
        first = rec is None
        if first:
            if sn and (has_add or cfg.post_act != ACT_NONE or cfg.pre_act not in (ACT_NONE, ACT_LEAKY) or G > 4):
                raise _ext.MtdError(f"task-gradient fold: no kernel for a spectrally-normalised layer with {cfg}")
            bias_grad = None
            if want_bias:
                bias_grad = self.bias_grads.get(bias.data_ptr())
                if bias_grad is None:
                    bias_grad = self.bias_grads[bias.data_ptr()] = self._zeros(cfg.cout, torch.float32, g1)
            zw = self._zeros(G, torch.float64, g1) if sn else None
            rec = self.records[id(node)] = _FoldRec(node, weight, x1, x2, g1, bias_grad, inv_sigma, u, v, zw, cfg, shapes)
        act = cfg.pre_act
        dz = _empty(g1.shape, g1) if act != ACT_NONE else g1
        y_in = pre_out if (act != ACT_NONE or sn) else None
        call("mtd_act_bwd_acc", fptr(g1), fptr(y_in), fptr(dz) if act != ACT_NONE else None, fptr(rec.acc), 1 if first else 0,
             fptr(rec.bias_grad), fptr(bias) if sn else None, ptr(rec.zw), fptr(inv_sigma), G, g1.numel() // cfg.cout,
             cfg.cout, act, cfg.slope, stream())
        if self.last_pass:
            self._issue_wgrad(rec)
        return dz

    def _issue_wgrad(self, rec):
        """One weight-gradient GEMM over the whole accumulated batch (pre-scaled by 1/sigma of each call)."""
        if rec.gp is not None:
            return
        B, H, W, C1, C2 = rec.shapes
        rec.gp = gp = _empty((rec.weight.numel(),), rec.acc)
        launch = lambda: _conv_wgrad_launch(rec.x1, rec.x2, rec.acc, gp, B, H, W, C1, C2, rec.cfg)
        if _WGRAD_SIDE and _finish_queue is not None and not torch.is_anomaly_enabled():
            _on_side_stream(launch, rec.x1, rec.x2, rec.acc, gp)       # joined when the deferred-finishing pass exits
        else:
            launch()

    def _finish(self):
        groups = {}
        for rec in self.records.values():
            self._issue_wgrad(rec)
            w = rec.weight.detach()
            if rec.inv_sigma is not None:
                u, v, G = rec.u, rec.v, rec.inv_sigma.numel()
                insts = [(rec.gp if g == 0 else None, w, u[g] if u.dim() == 2 else u, v[g] if v.dim() == 2 else v,
                          rec.inv_sigma[g:g + 1], rec.cfg, rec.zw.data_ptr() + 8 * g, 2 if g == 0 else 4) for g in range(G)]
            else:
                insts = [(rec.gp, w, None, None, None, rec.cfg, 0, 0)]
            grp = groups.get(w.data_ptr())
            if grp is None:
                groups[w.data_ptr()] = (torch.empty_like(w), insts)
            else:
                grp[1].extend(insts)            # instances of one weight are summed by the batched finishing pass
        _join_side_stream()
        if groups:
            _flush_finish(groups)
        out = []
        for p in self.params:
            g = groups.get(p.data_ptr())
            g = g[0] if g is not None else self.bias_grads.get(p.data_ptr())
            if g is None:
                raise _ext.MtdError(f"task-gradient fold: parameter of shape {tuple(p.shape)} was reached by no backward "
                                    "pass (it is not used in the graph of the losses)")
            out.append(g)
        return out


@dataclass(frozen=True)
class ConvCfg:
    cin: int                 # total input channels (C1 + C2)
    cout: int
    kh: int = 3
    kw: int = 3
    stride: int = 1
    pad: int = 1
    transposed: int = 0      # weight stored in ConvTranspose2d layout (Cin, Cout, kh, kw)
    pre_act: int = ACT_NONE
    post_act: int = ACT_NONE
    slope: float = LEAK
    fuse_add1_is_input: bool = False   # add1 is x1 itself (block residual): its gradient is fused into dgrad
    freeze: bool = False               # treat weight / bias as constants (no wgrad, no dbias)


_USE_TC = os.environ.get("MTDGAN_CONV", "auto")      # "simt" forces the exact-fp32 kernel everywhere
tc_launches = 0                                       # tcgen05 conv launches so far (tests / bench evidence)


_TC_PASSES = 1 if os.environ.get("MTDGAN_TF32", "x3") == "x1" else 3
_WGRAD_PASSES = 3 if os.environ.get("MTDGAN_WGRAD_TF32", "x1") == "x3" else 1


_TC_VERSION = 1


def set_tc_version(version: int) -> int:
    """Forward/dgrad tensor-core kernel generation (1: A through shared memory, 2: A through TMEM, multi-tile)."""
    global _TC_VERSION
    prev = _ext.load().mtd_tc_set_version(int(version))
    _TC_VERSION = int(version)
    return prev


def _tc_version() -> int:
    return _TC_VERSION


def set_wgrad_passes(passes: int):
    global _WGRAD_PASSES
    assert passes in (1, 3)
    _WGRAD_PASSES = passes


def set_conv_mode(mode: str, passes: int | None = None):
    """"auto": tcgen05 kernels where they apply, exact fp32 SIMT elsewhere; "simt": exact fp32 only.
    passes: 3 = error-compensated 3xTF32 (fp32-grade, default), 1 = plain TF32 (<= 2e-3)."""
    global _USE_TC, _TC_PASSES
    assert mode in ("auto", "simt")
    _USE_TC = mode
    if passes is not None:
        assert passes in (1, 3)
        _TC_PASSES = passes


def _tc_kind(base: str) -> str:
    return base + ("_tf32x3" if _TC_PASSES == 3 else "_tf32")


def _tc_ok(B, H, W, C1, C2, N, kh, kw, stride, pad) -> bool:
    """Kernel selection: the tcgen05 TF32 kernel takes stride-1 layers with C % 32 == 0, N % 32 == 0 and
    >= 2048 output pixels; skinny-M / thin / strided layers stay on the exact-fp32 SIMT kernel."""
    return _USE_TC != "simt" and _ext.load().mtd_conv_fwd_tc_supported(B, H, W, C1, C2, N, kh, kw, stride, pad) == 1


# Scratch for the stream-K wave of the tensor-core kernels (include/mtdgan_b200.h): one per (device, stream),
# contents undefined between calls.  32 MB cover every layer of the model at any batch size (the stream-K wave holds
# fewer tiles than there are SMs).
_TC_WS_FLOATS = 8 << 20
_tc_ws_cache: dict = {}


def _tc_workspace(device) -> torch.Tensor:
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    ws = _tc_ws_cache.get(key)
    if ws is None:
        ws = torch.empty(_TC_WS_FLOATS, dtype=torch.float32, device=device)
        _tc_ws_cache[key] = ws
    return ws


def _scale_group(scale, B: int) -> int:
    """Samples per 1/sigma entry: `scale` holds one entry per independent reference call batched together."""
    if scale is None or scale.numel() == 1:
        return 0
    g = scale.numel()
    assert B % g == 0, (B, g)
    return B // g


def _conv_forward_launch(x1, x2, weight, bias, scale, y, aux, add1, add2, cfg: ConvCfg):
    B, H, W, C1 = x1.shape
    C2 = 0 if x2 is None else x2.shape[3]
    tc = _tc_ok(B, H, W, C1, C2, cfg.cout, cfg.kh, cfg.kw, cfg.stride, cfg.pad)
    if tc:
        wp = _packed(weight, _tc_kind("fwd"), cfg)
    else:
        wp = _packed(weight, "fwd", cfg) if cfg.kh * cfg.kw > 1 or cfg.transposed else weight.detach()
    args = (fptr(x1), fptr(x2), fptr(wp), fptr(bias), fptr(scale), _scale_group(scale, B), fptr(y), fptr(aux), fptr(add1),
            fptr(add2), B, H, W, C1,
            C2, cfg.cout, cfg.kh, cfg.kw, cfg.stride, cfg.pad, cfg.pre_act, cfg.post_act, cfg.slope)
    if tc:
        global tc_launches
        tc_launches += 1
        ws = _tc_workspace(y.device)
        call("mtd_conv_fwd_tc", *args, _TC_PASSES, fptr(ws), ws.numel(), stream())
    else:
        call("mtd_conv_fwd", *args, stream())


def _conv_wgrad_launch(x1, x2, dz, gp, B, H, W, C1, C2, cfg: ConvCfg):
    """gp[N][T][C1+C2] (packed, forward orientation) = sum over pixels of dz (x) x."""
    st = stream()
    if _USE_TC != "simt" and _ext.load().mtd_conv_wgrad_tc_supported(B, H, W, C1, C2, cfg.cout, cfg.kh, cfg.kw, cfg.stride,
                                                                      cfg.pad) == 1:
        global tc_launches
        tc_launches += 1
        # plain TF32 for the weight gradient: it is a leaf reduction over >= 20 pixels (errors do not compound through
        # layers like forward / dgrad do), measured <= 1e-3 vs fp64 — inside the north_star's 2e-3 tensor-core bound
        call("mtd_conv_wgrad_tc", fptr(x1), fptr(x2), fptr(dz), fptr(gp), B, H, W, C1, C2, cfg.cout, cfg.kh, cfg.kw, cfg.stride,
             cfg.pad, _WGRAD_PASSES, st)
    else:
        call("mtd_conv_wgrad", fptr(x1), fptr(x2), fptr(dz), fptr(gp), B, H, W, C1, C2, cfg.cout, cfg.kh, cfg.kw, cfg.stride,
             cfg.pad, st)


def _conv_dgrad_launch(dz, weight, dx, scale, add1, B, H, W, cin_sub, cin_off, cfg: ConvCfg):
    """dx (B,H,W,cin_sub) = scale * dgrad(dz) (+ add1) for input channels [cin_off, cin_off + cin_sub)."""
    T = cfg.kh * cfg.kw
    st = stream()
    if cfg.stride == 1:
        tc = _tc_ok(B, H, W, cfg.cout, 0, cin_sub, cfg.kh, cfg.kw, 1, cfg.pad)
    else:   # 4x4 stride-2: four parity classes of 2x2-tap stride-1 convs over dz (B,H/2,W/2,Cout)
        tc = (cfg.stride == 2 and cfg.kh == 4 and cfg.kw == 4 and cfg.pad == 1 and cin_off == 0 and cin_sub == cfg.cin
              and H % 2 == 0 and W % 2 == 0 and _tc_ok(B, H // 2, W // 2, cfg.cout, 0, cin_sub, 1, 1, 1, 0))
    if tc:
        global tc_launches
        tc_launches += 1
        wpd = _packed(weight, _tc_kind("dgrad"), cfg)
        ws = _tc_workspace(dx.device)
        call("mtd_conv_dgrad_tc", fptr(dz), wpd.data_ptr() + 4 * cin_off * T * cfg.cout, fptr(dx), fptr(scale),
             _scale_group(scale, B), fptr(add1), None,
             None, 0, cfg.slope, B, H, W, cin_sub, cfg.cout, cfg.kh, cfg.kw, cfg.stride, cfg.pad, _TC_PASSES, cfg.cin,
             None, 0, fptr(ws), ws.numel(), st)
    else:
        wpd = _packed(weight, "dgrad", cfg)
        call("mtd_conv_dgrad", fptr(dz), wpd.data_ptr() + 4 * cin_off * T * cfg.cout, fptr(dx), fptr(scale),
             _scale_group(scale, B), fptr(add1), None,
             None, 0, cfg.slope, B, H, W, cin_sub, cfg.cout, cfg.kh, cfg.kw, cfg.stride, cfg.pad, st)


def _conv_dgrad_launch_cat(dz, weight, dx1, dx2, scale, B, H, W, C1, C2, cfg: ConvCfg) -> bool:
    """Both halves of a torch.cat layer's data gradient from ONE tensor-core launch (dz streamed once).  Returns False
    when the shape is not eligible (the caller then issues one launch per source)."""
    if (cfg.stride != 1 or C1 % 32 or C2 % 32 or _tc_version() != 1
            or not _tc_ok(B, H, W, cfg.cout, 0, C1 + C2, cfg.kh, cfg.kw, 1, cfg.pad)):
        return False
    global tc_launches
    tc_launches += 1
    wpd = _packed(weight, _tc_kind("dgrad"), cfg)
    ws = _tc_workspace(dx1.device)
    call("mtd_conv_dgrad_tc", fptr(dz), fptr(wpd), fptr(dx1), fptr(scale), _scale_group(scale, B), None, None, None, 0, cfg.slope,
         B, H, W, C1 + C2, cfg.cout, cfg.kh, cfg.kw, 1, cfg.pad, _TC_PASSES, cfg.cin, fptr(dx2), C1, fptr(ws), ws.numel(), stream())
    return True


class ConvFn(Function):
    """y = post_act( pre_act( scale * conv(cat[x1, x2], W) + b ) + add1 + add2 ).

    `weight` is the reference-layout parameter (Conv2d / ConvTranspose2d / Linear).  For spectrally
    normalised layers `inv_sigma` (G,), `u` (G, rows), `v` (G, cols) are the power-iteration results of the G
    independent reference calls batched in x1 (G = 1: one call; G = 2: e.g. D(real) and D(fake) as one batch, each
    half scaled by its own 1/sigma) and the backward applies dW_orig = sum_g (G_g - <G_g,W~_g> u_g v_g^T)/sigma_g.
    """

    @staticmethod
    def forward(ctx, x1, x2, weight, bias, inv_sigma, u, v, add1, add2, cfg: ConvCfg):
        B, H, W, C1 = x1.shape
        C2 = 0 if x2 is None else x2.shape[3]
        assert C1 + C2 == cfg.cin, (C1, C2, cfg)
        Ho = (H + 2 * cfg.pad - cfg.kh) // cfg.stride + 1
        Wo = (W + 2 * cfg.pad - cfg.kw) // cfg.stride + 1
        y = _empty((B, Ho, Wo, cfg.cout), x1)
        has_add = add1 is not None or add2 is not None
        need_graph = any(ctx.needs_input_grad)
        aux = _empty(y.shape, x1) if (need_graph and cfg.pre_act != ACT_NONE and has_add) else None
        _conv_forward_launch(x1, x2, weight, bias, inv_sigma, y, aux, add1, add2, cfg)
        ctx.cfg = cfg
        ctx.has_add = has_add
        ctx.weight_obj = weight          # identity key of the packed-weight cache
        ctx.shapes = (B, H, W, C1, C2)
        ctx.save_for_backward(x1, x2, weight, inv_sigma, u, v, y, aux, bias)
        return y

    @staticmethod
    def backward(ctx, dy):
        cfg: ConvCfg = ctx.cfg
        x1, x2, weight, inv_sigma, u, v, y, aux, bias = ctx.saved_tensors
        weight = ctx.weight_obj
        B, H, W, C1, C2 = ctx.shapes
        need = list(ctx.needs_input_grad)
        if cfg.freeze:
            need[2] = need[3] = False
        dy = dy.contiguous()
        M = dy.numel() // cfg.cout
        st = stream()
        # 1) through post_act, then the adds, then pre_act
        g1 = dy
        if cfg.post_act != ACT_NONE:
            g1 = _empty(dy.shape, dy)
            call("mtd_act_bwd", fptr(dy), fptr(y), fptr(g1), None, 0, M, cfg.cout, cfg.post_act, cfg.slope, st)
        d_add = g1 if ctx.has_add else None
        folded = _fold is not None and need[2] and _fold.wants(weight)
        if folded:         # weight and bias gradients are folded across the passes (fold_task_grads), none is issued here
            dz = _fold.act_bwd(ctx, g1, aux if aux is not None else y, weight, bias, need[3], inv_sigma, u, v, x1, x2, cfg,
                               ctx.shapes, ctx.has_add)
            need[2] = need[3] = False
        dbias, dbz = _dbias_alloc(cfg.cout, dy) if need[3] else (None, 0)
        want_w = need[2] and _wgrad_wanted(weight)
        G = 1 if inv_sigma is None else inv_sigma.numel()
        # spectrally-normalised layer inside a deferred-finishing pass: the correction coefficient <G_g, W~_g> of every
        # batched call g comes out of the activation-backward pass itself (mtd_act_bwd_sn) -- no dot pass later
        zw = None
        # Deferred finishing hands autograd a dw tensor that is only filled when the context exits.  That is sound while
        # nothing inspects gradients mid-pass; anomaly mode (NaN checks on every backward output) finishes immediately.
        deferred = _finish_queue is not None and not torch.is_anomaly_enabled()
        if (want_w and inv_sigma is not None and deferred and cfg.post_act == ACT_NONE and not ctx.has_add
                and cfg.pre_act in (ACT_NONE, ACT_LEAKY) and cfg.cout % 4 == 0 and G <= 4):
            zw = _zw_alloc(G, dy)
        if folded:
            pass
        elif zw is not None:
            if dbias is not None and not dbz:
                dbias.zero_()
            # dz is written pre-scaled by 1/sigma of its call: dgrad then needs no scale, and ONE weight-gradient GEMM over
            # the whole batch yields sum_g G_g / sigma_g (the per-call corrections are separate rank-1 terms)
            dz = _empty(dy.shape, dy)
            call("mtd_act_bwd_sn", fptr(g1), fptr(y), fptr(dz), fptr(dbias), fptr(bias), zw.data_ptr(), fptr(inv_sigma), G, M,
                 cfg.cout, cfg.pre_act, cfg.slope, st)
        elif cfg.pre_act != ACT_NONE:
            pre_out = aux if aux is not None else y
            dz = _empty(dy.shape, dy)
            call("mtd_act_bwd", fptr(g1), fptr(pre_out), fptr(dz), fptr(dbias), dbz, M, cfg.cout, cfg.pre_act, cfg.slope, st)
        else:
            dz = g1
            if dbias is not None:
                call("mtd_act_bwd", fptr(g1), None, None, fptr(dbias), dbz, M, cfg.cout, ACT_NONE, cfg.slope, st)
        # 2) weight gradient (packed), then to reference layout (+ spectral-norm correction).  Issued BEFORE the data
        #    gradient: on the side stream it then runs concurrently with this layer's dgrad and the layers after it
        dw = None
        if want_w:
            Bg = B // G
            insts = []          # (gp, w, u, v, 1/sigma, cfg, pointer to <G,W~> or 0, flag bits: 2 gp pre-scaled, 4 no gp)
            if zw is not None:
                gp = _empty((weight.numel(),), dy)
                if _WGRAD_SIDE:
                    _on_side_stream(lambda: _conv_wgrad_launch(x1, x2, dz, gp, B, H, W, C1, C2, cfg), x1, x2, dz, gp)
                else:
                    _conv_wgrad_launch(x1, x2, dz, gp, B, H, W, C1, C2, cfg)      # sum_g G_g / sigma_g in one GEMM
                for g in range(G):
                    insts.append((gp if g == 0 else None, weight.detach(), u[g] if u.dim() == 2 else u, v[g] if v.dim() == 2 else v,
                                  inv_sigma[g:g + 1], cfg, zw.data_ptr() + 8 * g, 2 if g == 0 else 4))
            else:
                for g in range(G):          # one packed weight gradient per batched reference call (own u, v, sigma)
                    gp = _empty((weight.numel(),), dy)
                    if G == 1:
                        if _WGRAD_SIDE and deferred:
                            _on_side_stream(lambda gp=gp: _conv_wgrad_launch(x1, x2, dz, gp, B, H, W, C1, C2, cfg), x1, x2, dz, gp)
                        else:
                            _conv_wgrad_launch(x1, x2, dz, gp, B, H, W, C1, C2, cfg)
                        insts.append((gp, weight.detach(), None if u is None else u.reshape(-1),
                                      None if v is None else v.reshape(-1), inv_sigma, cfg, 0, 0))
                    else:
                        sl = slice(g * Bg, (g + 1) * Bg)
                        _conv_wgrad_launch(x1[sl], None if x2 is None else x2[sl], dz[sl], gp, Bg, H, W, C1, C2, cfg)
                        insts.append((gp, weight.detach(), u[g], v[g], inv_sigma[g:g + 1], cfg, 0, 0))
            if deferred:
                grp = _finish_queue.get(weight.data_ptr())
                if grp is None:
                    dw = torch.empty_like(weight)
                    _finish_queue[weight.data_ptr()] = (dw, insts)
                else:
                    grp[1].extend(insts)           # summed into the first instance's dw by the batched unpack
            else:
                for k, (gp, wd, ug, vg, inv_g, _, _zw, _fl) in enumerate(insts):
                    part = torch.empty_like(weight)
                    scratch = torch.empty(4, dtype=torch.float32, device=dy.device) if inv_g is not None else None
                    call("mtd_conv_wgrad_finish", fptr(gp), fptr(part), cfg.transposed, cfg.cout, cfg.cin, cfg.kh, cfg.kw,
                         fptr(wd) if inv_g is not None else None, fptr(ug), fptr(vg), fptr(inv_g), ptr(scratch), st)
                    dw = part if k == 0 else dw + part
        # 3) data gradients
        dx1 = dx2 = None
        dscale = None if zw is not None else inv_sigma       # zw path: dz already carries 1/sigma
        both = False
        if C2 and need[0] and need[1] and not cfg.fuse_add1_is_input:
            dx1, dx2 = _empty((B, H, W, C1), dy), _empty((B, H, W, C2), dy)
            both = _conv_dgrad_launch_cat(dz, weight, dx1, dx2, dscale, B, H, W, C1, C2, cfg)
        if need[0] and not both:
            dx1 = _empty((B, H, W, C1), dy)
            fuse = g1 if cfg.fuse_add1_is_input else None
            _conv_dgrad_launch(dz, weight, dx1, dscale, fuse, B, H, W, C1, 0, cfg)
        if C2 and need[1] and not both:
            dx2 = _empty((B, H, W, C2), dy)
            _conv_dgrad_launch(dz, weight, dx2, dscale, None, B, H, W, C2, C1, cfg)
        d_add1 = d_add if (need[7] and not cfg.fuse_add1_is_input) else None
        d_add2 = d_add if need[8] else None
        return dx1, dx2, dw, dbias, None, None, None, d_add1, d_add2, None


def conv(x1, weight, bias, cfg: ConvCfg, x2=None, inv_sigma=None, u=None, v=None, add1=None, add2=None):
    return ConvFn.apply(x1, x2, weight, bias, inv_sigma, u, v, add1, add2, cfg)


# ------------------------------------------------------------------------------------------------
# Res-FFT-Conv block: out = x + relu(img_conv(x)) + irfft2(relu(fft_conv(cat[Re,Im] rfft2(x))))
# ------------------------------------------------------------------------------------------------
_IMG_CFG = {}


def _img_cfg(c):
    if c not in _IMG_CFG:
        _IMG_CFG[c] = ConvCfg(cin=c, cout=c, kh=3, kw=3, stride=1, pad=1, pre_act=ACT_RELU)
    return _IMG_CFG[c]


class FFTConvBlockFn(Function):
    """One fused FFT_ConvBlock (arch/Ours/networks.py:21-36) on an NHWC tensor."""

    @staticmethod
    def forward(ctx, x, img_w, img_b, fft_w, fft_b):
        B, H, W, C = x.shape
        st = stream()
        cfg = _img_cfg(C)
        need_graph = any(ctx.needs_input_grad)
        if _ext.load().mtd_fft_supported(H, W, C) != 1:
            raise _ext.MtdError(f"FFT_ConvBlock on the B200 path supports 32 channels and 1 <= H, W <= 512; got "
                                f"C={C}, H={H}, W={W}")
        spec = _empty((_ext.load().mtd_fft_spec_elems(B, H, W, C),), x)
        call("mtd_fft_rows_fwd", fptr(x), fptr(spec), B, H, W, C, st)
        spec2 = _empty(spec.shape, x) if need_graph else spec          # in place when nothing is saved
        call("mtd_fft_cols_mix", fptr(spec), fptr(spec2), fptr(fft_w.detach()), fptr(fft_b.detach()), B, H, W, C, st)
        img = _empty(x.shape, x)
        out = _empty(x.shape, x)
        if need_graph:
            _conv_forward_launch(x, None, img_w, img_b.detach(), None, img, None, None, None, cfg)
            call("mtd_fft_rows_inv", fptr(spec2), fptr(x), fptr(img), fptr(out), B, H, W, C, st)
        else:
            # inference: the identity branch rides in the conv epilogue (img = relu(conv(x)) + x), so the inverse row pass
            # reads ONE residual operand instead of two (33.5 MB less HBM traffic per block at 512 x 512)
            _conv_forward_launch(x, None, img_w, img_b.detach(), None, img, None, x, None, cfg)
            call("mtd_fft_rows_inv", fptr(spec2), fptr(img), None, fptr(out), B, H, W, C, st)
        if need_graph:
            ctx.img_w_obj = img_w
            ctx.save_for_backward(x, img_w, fft_w, fft_b, spec, img)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, img_w, fft_w, fft_b, spec, img = ctx.saved_tensors
        img_w = ctx.img_w_obj
        B, H, W, C = x.shape
        if H not in (64, 128, 256) or W not in (64, 128, 256, 512):
            raise _ext.MtdError(f"FFT_ConvBlock backward is built for H in (64, 128, 256) and W in (64, 128, 256, 512) "
                                f"(training patches are 64 x 64); got H={H}, W={W}")
        st = stream()
        cfg = _img_cfg(C)
        need = ctx.needs_input_grad
        dout = dout.contiguous()
        lib = _ext.load()
        # frequency branch
        gspec = _empty(spec.shape, x)
        call("mtd_fft_rows_fwd", fptr(dout), fptr(gspec), B, H, W, C, st)
        part = _empty((lib.mtd_fft_bwd_part_elems(B, W),), x)
        dfw = torch.empty_like(fft_w)
        dfb = torch.empty_like(fft_b)
        call("mtd_fft_cols_mix_bwd", fptr(spec), fptr(gspec), fptr(gspec), fptr(fft_w.detach()), fptr(fft_b.detach()),
             fptr(part), fptr(dfw), fptr(dfb), B, H, W, C, st)
        # image branch
        M = B * H * W
        dz = _empty(x.shape, x)
        dib = _empty((C,), x)
        call("mtd_act_bwd", fptr(dout), fptr(img), fptr(dz), fptr(dib), 0, M, C, ACT_RELU, LEAK, st)
        dx = None
        if need[0]:
            dxc = _empty(x.shape, x)      # dgrad(dz) + dout   (residual path fused)
            _conv_dgrad_launch(dz, img_w, dxc, None, dout, B, H, W, C, 0, cfg)
            dx = _empty(x.shape, x)       # + frequency-branch gradient, fused into the inverse row pass
            call("mtd_fft_rows_inv", fptr(gspec), fptr(dxc), None, fptr(dx), B, H, W, C, st)
        diw = None
        if need[1] and _wgrad_wanted(img_w):
            gp = _empty((img_w.numel(),), x)
            _conv_wgrad_launch(x, None, dz, gp, B, H, W, C, 0, cfg)
            diw = torch.empty_like(img_w)
            call("mtd_conv_wgrad_finish", fptr(gp), fptr(diw), 0, C, C, 3, 3, None, None, None, None, None, st)
        return dx, diw, dib, dfw, dfb


def fft_conv_block(x, img_w, img_b, fft_w, fft_b):
    return FFTConvBlockFn.apply(x, img_w, img_b, fft_w, fft_b)


# ------------------------------------------------------------------------------------------------
# resampling / elementwise
# ------------------------------------------------------------------------------------------------
class Upsample2xFn(Function):
    @staticmethod
    def forward(ctx, x):
        B, H, W, C = x.shape
        out = _empty((B, 2 * H, 2 * W, C), x)
        call("mtd_upsample2x_fwd", fptr(x), fptr(out), B, H, W, C, stream())
        ctx.dims = (B, H, W, C)
        return out

    @staticmethod
    def backward(ctx, dout):
        B, H, W, C = ctx.dims
        dout = dout.contiguous()
        din = _empty((B, H, W, C), dout)
        call("mtd_upsample2x_bwd", fptr(dout), fptr(din), B, H, W, C, stream())
        return din


class PixelShuffle2Fn(Function):
    @staticmethod
    def forward(ctx, x):
        B, H, W, C4 = x.shape
        C = C4 // 4
        out = _empty((B, 2 * H, 2 * W, C), x)
        call("mtd_pixel_shuffle2", fptr(x), fptr(out), B, H, W, C, 0, stream())
        ctx.dims = (B, H, W, C)
        return out

    @staticmethod
    def backward(ctx, dout):
        B, H, W, C = ctx.dims
        dout = dout.contiguous()
        din = _empty((B, H, W, 4 * C), dout)
        call("mtd_pixel_shuffle2", fptr(dout), fptr(din), B, H, W, C, 1, stream())
        return din


class Clip01Fn(Function):
    @staticmethod
    def forward(ctx, x):
        x = x.contiguous()
        y = torch.empty_like(x)
        call("mtd_clip01_fwd", fptr(x), fptr(y), x.numel(), stream())
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dy = dy.contiguous()
        dx = torch.empty_like(x)
        call("mtd_clip01_bwd", fptr(x), fptr(dy), fptr(dx), x.numel(), stream())
        return dx


class MulConstFn(Function):
    """x * m with m a constant (dropout keep-mask already scaled by 1/(1-p))."""

    @staticmethod
    def forward(ctx, x, m):
        x = x.contiguous()
        out = torch.empty_like(x)
        call("mtd_mul", fptr(x), fptr(m), fptr(out), x.numel(), stream())
        ctx.save_for_backward(m)
        return out

    @staticmethod
    def backward(ctx, dout):
        (m,) = ctx.saved_tensors
        dout = dout.contiguous()
        dx = torch.empty_like(dout)
        call("mtd_mul", fptr(dout), fptr(m), fptr(dx), dout.numel(), stream())
        return dx, None


class LayoutFn(Function):
    """NCHW <-> NHWC (only where a multi-channel drop-in module is called stand-alone)."""

    @staticmethod
    def forward(ctx, x, to_nhwc: bool):
        x = x.contiguous()
        if to_nhwc:
            B, C, H, W = x.shape
            out = _empty((B, H, W, C), x)
        else:
            B, H, W, C = x.shape
            out = _empty((B, C, H, W), x)
        call("mtd_layout_transpose", fptr(x), fptr(out), B, C, H * W, 1 if to_nhwc else 0, stream())
        ctx.to_nhwc = to_nhwc
        return out

    @staticmethod
    def backward(ctx, dout):
        return LayoutFn.apply(dout, not ctx.to_nhwc), None


def to_nhwc(x):
    """(B,C,H,W) -> (B,H,W,C); free (a view) when C == 1."""
    if x.shape[1] == 1:
        return x.reshape(x.shape[0], x.shape[2], x.shape[3], 1)
    return LayoutFn.apply(x, True)


def to_nchw(x):
    if x.shape[3] == 1:
        return x.reshape(x.shape[0], 1, x.shape[1], x.shape[2])
    return LayoutFn.apply(x, False)


def check_input(x: torch.Tensor, what: str):
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise _ext.MtdError(f"{what}: expected a CUDA tensor — the B200 hot path has no CPU fallback")
    if x.dtype != torch.float32:
        raise _ext.MtdError(f"{what}: expected float32, got {x.dtype}")
    _ext.load()
    return x.contiguous()
