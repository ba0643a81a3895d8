#!/usr/bin/env python
"""MTD-GAN hot-path benchmark (contract: `python bench.py --gpus N --steps K --warmup W [--impl reference]`).

Own arm (default): the full MTD-GAN train step — G forward, 4 D forwards, RC/NDS losses, PCGrad (3+1 backward
passes), AdamW on D, G forward + D forward, backward, AdamW on G (the reference's engine.py:40-55) — on
20 synthetic 64x64 patches per GPU (BASELINE.json configs[2]; configs[3] at N > 1), every kernel of which is
launched from libmtdgan_sm100a.so.  Also reports generator inference on 1x512x512 slices (configs[1]).
Reference arm (`--impl reference`): the CPU oracle port of the same step on the box's host cores (the Python
reference cannot travel to the GPU box; SURVEY §8c).

One JSON line on stdout (rank 0).  `--dump-outputs DIR` also writes what the last timed train step computed (losses,
loss terms, the weights it leaves) as DIR/<name>.npy.  Every timed step starts from the same seeded state on the same
inputs, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line.  Libraries print there too (NCCL's version banner at NCCL_DEBUG=VERSION or
# WARN), so file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor.
_JSON_FD = None


def claim_stdout():
    """Called by main() only (importing this module, e.g. from the cpu_baseline child process, must not touch fd 1)."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    if _JSON_FD is None:
        print(json.dumps(line), flush=True)
    else:
        os.write(_JSON_FD, (json.dumps(line) + "\n").encode())


import numpy as np  # noqa: E402
import torch  # noqa: E402

PATCH, BATCH = 64, 20
F_ALG_TRAIN = 99.3e9          # useful conv+linear FLOP per patch per train step (SURVEY §8d)
B_ALG_INFER = 3.22e9          # algorithmic HBM bytes per 512^2 slice (SURVEY §8d)
N_SHARED = 28_609_920


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ----------------------------------------------------------------------------------------------------
# own arm
# ----------------------------------------------------------------------------------------------------
def flops_of(name, a):
    """Algorithmic FLOPs (2*MAC) of one conv entry-point call from its argument list."""
    if name in ("mtd_conv_fwd", "mtd_conv_fwd_tc"):
        B, H, W, C1, C2, N, kh, kw, s, p = a[10:20]
        Ho, Wo = (H + 2 * p - kh) // s + 1, (W + 2 * p - kw) // s + 1
        return 2.0 * B * Ho * Wo * N * (C1 + C2) * kh * kw
    if name in ("mtd_conv_dgrad", "mtd_conv_dgrad_tc"):
        B, H, W, Cin, Cout, kh, kw, s, p = a[10:19]
        Ho, Wo = (H + 2 * p - kh) // s + 1, (W + 2 * p - kw) // s + 1
        return 2.0 * B * Ho * Wo * Cout * Cin * kh * kw
    if name in ("mtd_conv_wgrad", "mtd_conv_wgrad_tc"):
        B, H, W, C1, C2, N, kh, kw, s, p = a[4:14]
        Ho, Wo = (H + 2 * p - kh) // s + 1, (W + 2 * p - kw) // s + 1
        return 2.0 * B * Ho * Wo * N * (C1 + C2) * kh * kw
    return 0.0


GROUPS = {"conv": ("mtd_conv_fwd", "mtd_conv_fwd_tc", "mtd_conv_dgrad", "mtd_conv_dgrad_tc", "mtd_conv_wgrad", "mtd_conv_wgrad_tc"),
          "conv_aux": ("mtd_conv_pack_fwd", "mtd_conv_pack_dgrad", "mtd_conv_pack_fwd_blocked", "mtd_conv_pack_dgrad_blocked", "mtd_conv_wgrad_finish", "mtd_act_bwd", "mtd_split_tf32",
                       "mtd_round_tf32"),
          "fft": ("mtd_fft_rows_fwd", "mtd_fft_cols_mix", "mtd_fft_rows_inv", "mtd_fft_cols_mix_bwd"),
          "spectral_norm": ("mtd_sn_power_iter",), "pcgrad": ("mtd_pcgrad_project",), "adamw": ("mtd_adamw_step",)}


DUMP_D_SAMPLE = 1 << 20      # discriminator parameters --dump-outputs writes: a fixed, seeded sample of the 68.4 M


def step_outputs(out, model):
    """What a train step hands its caller, as float32 host arrays: the losses and loss terms it returns and the weights
    it leaves behind (every generator parameter, DUMP_D_SAMPLE discriminator parameters at seeded positions)."""
    d_losses, d_det, g_loss, g_det = out
    arrays = {"d_losses": d_losses, "g_loss": g_loss}
    arrays.update({k.replace("/", "_"): v for k, v in {**d_det, **g_det}.items()})       # 'D/real_enc' -> D_real_enc
    arrays["generator_params"] = torch.cat([p.detach().flatten() for p in model.Generator.parameters()])
    d_flat = torch.cat([p.detach().flatten() for p in model.Discriminator.parameters()])
    idx = torch.randint(0, d_flat.numel(), (DUMP_D_SAMPLE,), generator=torch.Generator().manual_seed(0))
    arrays["discriminator_params_sample"] = d_flat[idx.to(d_flat.device)]
    return {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_own(args):
    import mtdgan_b200
    from mtdgan_b200 import _ext
    from mtdgan_b200.data import synthetic_pair
    from mtdgan_b200.optim import FusedAdamW
    from mtdgan_b200 import distributed as mdist
    from arch.Ours.networks import MTD_GAN_Method
    from module.weight_methods import WeightMethods

    rank, world, local = dist_env()
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    mtdgan_b200.require_cuda_extension()
    if world > 1:
        mdist.init()
    torch.manual_seed(2024)
    random.seed(2024)
    model = MTD_GAN_Method().to(dev).train()
    D, G = model.Discriminator, model.Generator
    opt_D = FusedAdamW([{"params": list(D.parameters())}, {"params": [], "lr": 0.025}], lr=1e-4, weight_decay=5e-4)
    opt_G = FusedAdamW(G.parameters(), lr=1e-4, weight_decay=5e-4)
    wm = WeightMethods("pcgrad", n_tasks=3, device=dev)
    shared, ts, last = list(D.shared_parameters()), list(D.task_specific_parameters()), list(D.last_shared_parameters())
    xh, yh = synthetic_pair(BATCH, PATCH, seed=1234, rank=rank, pin=True)
    xd, yd = xh.to(dev), yh.to(dev)

    from mtdgan_b200.graphs import GraphedTrainStep
    gparams = list(G.parameters())
    runner = GraphedTrainStep(model, opt_D, opt_G, wm,
                              post_g_backward=(lambda: mdist.allreduce_mean_grads(gparams)) if world > 1 else None)
    # Every timed step starts from this state (weights, spectral-norm vectors, optimizer moments, RNGs), restored outside
    # the timed window.  The fp32 atomics of some kernels differ in the last bits from run to run, and the GAN's
    # trajectory grows such differences to O(1) within a few dozen steps: a fixed start keeps each step's outputs
    # reproducible, and the work a step does does not depend on the values.
    init_state = runner._snapshot()

    def eager_step(x, y):
        dl, _, gl, _ = runner.eager_step(x, y)
        return dl, gl

    use_graph = not args.no_graph
    eager_step(xd, yd)                                  # first step: lazy one-time work (per-layer packing, table builds)
    l0 = _ext.kernel_launch_count()
    eager_step(xd, yd)
    launches = _ext.kernel_launch_count() - l0          # kernels of this library per steady-state step (replays run the same)
    if use_graph:
        # At N > 1 the step contains NCCL collectives (reduce-scatter / all-reduce / all-gather of the PCGrad path, the
        # generator-gradient all-reduce); NCCL kernels are capturable, every rank captures and replays the same graph.
        # MTD_BENCH_NCCL_GRAPH=0 falls back to eager launches at N > 1.
        if world > 1 and os.environ.get("MTD_BENCH_NCCL_GRAPH", "1") == "0":
            use_graph = False
        else:
            runner.capture(xd, yd, warmup=2)

    last = [None]             # what the latest step returned (graph output buffers: valid until the next replay)

    def step(x, y):
        last[0] = runner(x, y)
        dl, _, gl, _ = last[0]
        return dl, gl

    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)      # > 126 MB L2

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(n, e2e):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        sink = torch.empty(4, dtype=torch.float32).pin_memory()
        for s, e in ev:
            runner._restore(init_state)
            flush.zero_()
            s.record()
            if e2e:
                x, y = xh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True)
                dl, gl = step(x, y)
                sink[:3].copy_(dl.detach(), non_blocking=True)
                sink[3:].copy_(gl.detach().reshape(1), non_blocking=True)
            else:
                step(xd, yd)
            e.record()
        torch.cuda.synchronize()
        return [s.elapsed_time(e) for s, e in ev]

    for _ in range(max(args.warmup, 3)):
        step(xd, yd)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(args.steps, e2e=False)
    barrier()
    ms_e2e = timed(args.steps, e2e=True)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, step_outputs(last[0], model))
    t_dev, t_e2e = sum(ms), sum(ms_e2e)
    if world > 1:
        t = torch.tensor([t_dev, t_e2e], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        t_dev, t_e2e = float(t[0]), float(t[1])

    # ---- per-kernel-class times: one extra (untimed) step with CUDA events around every C-ABI call
    breakdown, roof = None, None
    torch.cuda.synchronize()
    if rank == 0:
        # The eager step is enqueued from Python at ~10 us per call -- slower than the GPU executes it, so an event pair
        # around a call would also time the host gap in front of it.  A 0.3 s device-side spin gives the host a head
        # start: the whole step is queued behind it and then runs back to back, and the events time kernels only.
        torch.cuda._sleep(int(0.3 * 1.9e9))
        _ext.start_profile()
    eager_step(xd, yd)                      # every rank runs it (the step contains collectives at N > 1)
    rec = _ext.stop_profile() if rank == 0 else None
    barrier()
    if rank == 0:
        total_ms = sum(r[2] for r in rec)
        if os.environ.get("MTD_BENCH_DUMP"):       # per-call records (entry point, integer args, ms) for offline analysis
            with open(os.environ["MTD_BENCH_DUMP"], "w") as fh:
                for name, a, t in rec:
                    fh.write(json.dumps([name, [v for v in a if isinstance(v, int) and abs(v) < 1 << 31], round(t, 5)]) + "\n")
        by = {}
        for name, a, t in rec:
            d = by.setdefault(name, {"ms": 0.0, "calls": 0, "flop": 0.0})
            d["ms"] += t; d["calls"] += 1; d["flop"] += flops_of(name, a)
        breakdown = {g: {"ms": round(sum(by[n]["ms"] for n in names if n in by), 3),
                         "calls": sum(by[n]["calls"] for n in names if n in by)} for g, names in GROUPS.items()}
        known = {n for names in GROUPS.values() for n in names}
        breakdown["other"] = {"ms": round(sum(v["ms"] for k, v in by.items() if k not in known), 3),
                              "calls": sum(v["calls"] for k, v in by.items() if k not in known)}
        breakdown["sum_ms"] = round(total_ms, 3)
        pk = peaks()
        conv_ms = sum(by[n]["ms"] for n in GROUPS["conv"] if n in by)
        conv_flop = sum(by[n]["flop"] for n in GROUPS["conv"] if n in by)
        conv_calls = sum(by[n]["calls"] for n in GROUPS["conv"] if n in by)
        timing = "CUDA events around every call of one eager step (includes host launch gaps)"
        if use_graph and getattr(runner, "trace", None):
            # Kernel-only times: re-issue each stateless kernel family of the CAPTURED step (same calls, same buffers,
            # same order) as its own CUDA graph and time its replay with events -- no host gaps, no event overhead.
            fam_ms = {}
            for gname in ("conv", "conv_aux", "fft"):
                fg, ncalls = runner.family_graph(set(GROUPS[gname]))
                fg.replay()
                torch.cuda.synchronize()
                evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
                for s_, e_ in evs:
                    flush.zero_()
                    s_.record(); fg.replay(); e_.record()
                torch.cuda.synchronize()
                fam_ms[gname] = (statistics.mean(s_.elapsed_time(e_) for s_, e_ in evs), ncalls)
                breakdown[gname] = {"ms": round(fam_ms[gname][0], 3), "calls": ncalls,
                                    "eager_event_ms": breakdown[gname]["ms"]}
                del fg
            if os.environ.get("MTD_BENCH_PER_ENTRY"):      # kernel-only time of every stateless entry point (analysis aid)
                per = {}
                safe = set(GROUPS["conv"]) | set(GROUPS["conv_aux"]) | set(GROUPS["fft"]) | {
                    "mtd_upsample2x_fwd", "mtd_upsample2x_bwd", "mtd_pixel_shuffle2", "mtd_clip01_fwd", "mtd_clip01_bwd",
                    "mtd_mul", "mtd_add3", "mtd_layout_transpose"}
                for nm in sorted({n for n, _ in runner.trace} & safe):
                    fg, ncalls = runner.family_graph({nm})
                    fg.replay(); torch.cuda.synchronize()
                    s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s_.record()
                    for _ in range(3):
                        fg.replay()
                    e_.record(); torch.cuda.synchronize()
                    per[nm] = {"ms": round(s_.elapsed_time(e_) / 3, 3), "calls": ncalls}
                    del fg
                breakdown["per_entry"] = per
            conv_ms, conv_calls = fam_ms["conv"]
            total_ms = t_dev / args.steps
            breakdown["timing"] = ("conv / conv_aux / fft: replay of that family's calls of the captured step as its own CUDA "
                                   "graph (kernel-only); other rows: events around the calls of one eager step")
            timing = "replay of the captured step's conv-family calls as one CUDA graph, CUDA events, mean of 5"
        # achieved = ALGORITHMIC FLOP (SURVEY §8d: F_alg = 99.3 GF per patch per step, useful conv + linear work) over the
        # conv family's kernel-only time; the FLOP the launches actually execute (redundant decoder traversals of the
        # fourth backward pass, the generator forward that is NOT re-run, ...) are reported beside it
        ach_exec = conv_flop / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
        ach = F_ALG_TRAIN * BATCH / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
        by_kind = {}
        for name, a, t in rec:
            fl = flops_of(name, a)
            if fl:
                kind = "wgrad" if "wgrad" in name else "dgrad" if "dgrad" in name else "fwd"
                by_kind[kind] = by_kind.get(kind, 0.0) + fl
        roof = {"kernel": "implicit-GEMM conv family (fwd + dgrad + wgrad)", "bound": "tensor", "achieved": round(ach, 3),
                "peak": pk["tflops_sustained"], "unit": "TFLOP/s", "frac": round(ach / pk["tflops_sustained"], 5),
                "flop_basis": "algorithmic: F_alg 99.3 GF/patch x 20 patches per launch-set (SURVEY 8d)",
                "executed_tflops": round(ach_exec, 3), "frac_executed": round(ach_exec / pk["tflops_sustained"], 5),
                "executed_gflop_per_patch": {k: round(v / BATCH / 1e9, 2) for k, v in sorted(by_kind.items())},
                "algorithmic_gflop_per_patch": F_ALG_TRAIN / 1e9,
                # DRAM bytes of ONE representative launch of the dominant kernel from an `ncu --set full` capture
                # (profiles/r01_ncu_full_conv_tc_v1_v3.txt): conv_tc_kernel<128,3>, B=20 32x32 256->128 3x3 --
                # 23.37 MB read + 2.6 KB written vs 23.3 MB compulsory (input + hi|lo weights; the output stays in L2)
                "traffic": 23375104, "traffic_source": "ncu dram__bytes_read+write of one conv_tc_kernel<128,3> launch "
                "(B=20 32x32 256->128 3x3; algorithmic input+weight bytes 23.3 MB, output L2-resident), not the family average",
                "peak_source": pk["source"] + ", sustained bf16 dense (kernel timed inside a long step)",
                # fp32-grade results need 3 TF32 MMAs per product and TF32 runs at half the bf16 rate: the same peak
                # expressed in useful fp32-equivalent FLOP/s is peak / 6
                "peak_3xtf32_equiv": round(pk["tflops_sustained"] / 6, 1), "frac_of_3xtf32_peak": round(ach / (pk["tflops_sustained"] / 6), 4),
                "timing": timing,
                "algorithmic_flop_per_launch": round(F_ALG_TRAIN * BATCH / max(conv_calls, 1)), "launches_per_step": conv_calls,
                "avg_launch_ms": round(conv_ms / max(conv_calls, 1), 5), "share_of_step": round(conv_ms / total_ms, 4),
                "pcgrad": {"bound": "hbm", "achieved": round(7 * N_SHARED * 4 / (by["mtd_pcgrad_project"]["ms"] * 1e-3) / 1e9, 1),
                           "peak": pk["hbm_gbs"], "unit": "GB/s",
                           "frac": round(7 * N_SHARED * 4 / (by["mtd_pcgrad_project"]["ms"] * 1e-3) / 1e9 / pk["hbm_gbs"], 4)}
                if "mtd_pcgrad_project" in by else None}

    # ---- generator inference (configs[1]: one 1x512x512 slice; configs[4]: 64 slices per GPU, slices sharded by rank,
    #      no collective).  The forward is replayed as a CUDA graph per micro-batch (mtdgan_b200.inference).
    infer = run_inference(args, model, dev, rank, world, flush)

    gpu_eager = None
    if rank == 0 and world == 1 and not args.no_gpu_eager:
        try:
            gpu_eager = run_gpu_eager_baseline(dev, xd, yd)
        except Exception as ex:       # a baseline leg must never take the measurement down with it
            gpu_eager = {"failed": f"{type(ex).__name__}: {ex}"}
    if rank == 0 and roof is not None and world == 1:
        try:
            roof["tf32_peak"] = measure_tf32_peak(dev)
        except Exception as ex:
            roof["tf32_peak"] = {"failed": f"{type(ex).__name__}: {ex}"}

    if rank != 0:
        return None
    patches = BATCH * world
    line = {
        "metric": "train patches/s (64x64, bs20/GPU)", "value": round(patches * args.steps / (t_dev * 1e-3), 3), "unit": "patches/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(t_dev / args.steps, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "MTD_GAN_Method full train step (G + MTL-D + RC/NDS + PCGrad + AdamW), 20 synthetic 1x64x64 patches/GPU "
                               "(BASELINE configs[2]/[3])", "global_batch": patches, "patch": PATCH,
                   "parallelism": f"dp{world}", "l2": "256 MiB buffer written between timed steps (L2 flush)",
                   "weights": "random init, seed 2024", "optimizer": "fused AdamW lr 1e-4 wd 5e-4",
                   "timed_step_state": "every timed step starts from the seeded initial weights, optimizer state and RNGs "
                                       "(restored outside the timed window)",
                   "execution": "whole step replayed as one CUDA graph" if use_graph else "eager launches",
                   "conv_precision": "tcgen05 3xTF32 (fp32-grade) + exact fp32 SIMT for thin/strided layers"},
        "e2e": {"value": round(patches * args.steps / (t_e2e * 1e-3), 3), "unit": "patches/s",
                "h2d_bytes_per_step": 2 * BATCH * PATCH * PATCH * 4, "d2h_bytes_per_step": 16},
        "gpu_launches": int(launches) * args.steps, "gpu_launches_per_step": int(launches),
        "useful_tflops": round(F_ALG_TRAIN * patches * args.steps / (t_dev * 1e-3) / 1e12, 3),
        "roofline": roof, "kernel_breakdown_ms": breakdown, "inference": infer, "gpu_eager_baseline": gpu_eager, "clocks": clocks,
    }
    return line


# Bytes of DRAM traffic per 512x512 slice measured by `ncu --set full` over one batch-1 generator forward (sum of
# dram__bytes_read.sum + dram__bytes_write.sum over its 105 kernels; profiles/r02_ncu_infer512_launches.csv): 5.51 GB vs
# 3.22 GB algorithmic -- the half spectrum makes two HBM round trips per block (rows -> columns -> rows) that B_alg
# assumes stay on chip.
INFER_TRAFFIC_BYTES = 5513783296


def run_inference(args, model, dev, rank, world, flush):
    from mtdgan_b200.data import synthetic_pair
    from mtdgan_b200.inference import GraphedGenerator, shard_slices
    from mtdgan_b200 import _ext
    G = model.Generator
    model.eval()
    pk = peaks()
    n_inf = max(10, min(30, args.steps))

    def ev_pairs(n):
        return [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]

    with torch.no_grad():
        # -- configs[1]: batch 1
        xs_h = synthetic_pair(1, 512, seed=4321, rank=rank, pin=True)[0]
        xs = xs_h.to(dev)
        g1 = GraphedGenerator(G, 512, 512, micro_batch=1).capture()
        for _ in range(3):
            g1(xs)
        torch.cuda.synchronize()
        ev = ev_pairs(n_inf)
        for s, e in ev:
            flush.zero_()
            s.record(); g1(xs); e.record()
        torch.cuda.synchronize()
        inf_ms = [s.elapsed_time(e) for s, e in ev]
        out_h = torch.empty(1, 1, 512, 512).pin_memory()
        ev2 = ev_pairs(n_inf)
        for s, e in ev2:
            flush.zero_()
            s.record(); out_h.copy_(g1(xs_h.to(dev, non_blocking=True)), non_blocking=True); e.record()
        torch.cuda.synchronize()
        inf_e2e = [s.elapsed_time(e) for s, e in ev2]
        # eager (ungraphed) for comparison + per-entry-point kernel times of one forward
        ev3 = ev_pairs(5)
        for s, e in ev3:
            s.record(); G(xs); e.record()
        torch.cuda.synchronize()
        eager_ms = statistics.mean(s.elapsed_time(e) for s, e in ev3)
        per_entry = None
        if rank == 0:
            torch.cuda._sleep(int(0.05 * 1.9e9))
            _ext.start_profile()
            G(xs)
            rec = _ext.stop_profile()
            per_entry = {}
            for name, a, t in rec:
                d = per_entry.setdefault(name, {"ms": 0.0, "calls": 0})
                d["ms"] = round(d["ms"] + t, 4); d["calls"] += 1
        del g1

        # -- configs[4]: 64 slices per GPU; choose the micro-batch by a short sweep (1 / 2 / 4), keep the best
        per_gpu = args.infer_batch
        xb_h = synthetic_pair(per_gpu, 512, seed=777, rank=rank, pin=True)[0]
        ob_h = torch.empty(per_gpu, 1, 512, 512).pin_memory()
        xb = xb_h.to(dev)
        ob = torch.empty_like(xb)
        best = None
        for mb in (1, 2, 4):
            gb = GraphedGenerator(G, 512, 512, micro_batch=mb).capture()
            gb(xb[:2 * mb], ob[:2 * mb])
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); gb(xb[:8], ob[:8]); e.record()
            torch.cuda.synchronize()
            t = s.elapsed_time(e) / 8
            if best is None or t < best[1]:
                best = (mb, t)
            del gb
        gb = GraphedGenerator(G, 512, 512, micro_batch=best[0]).capture()
        gb(xb, ob)
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        reps = 3
        evb = ev_pairs(reps)
        for s, e in evb:
            flush.zero_()
            s.record(); gb(xb, ob); e.record()
        torch.cuda.synchronize()
        tb = sum(s.elapsed_time(e) for s, e in evb)
        evc = ev_pairs(reps)
        for s, e in evc:
            flush.zero_()
            s.record()
            gb(xb_h.to(dev, non_blocking=True), ob)
            ob_h.copy_(ob, non_blocking=True)
            e.record()
        torch.cuda.synchronize()
        tc = sum(s.elapsed_time(e) for s, e in evc)
        if world > 1:
            t = torch.tensor([tb, tc], device=dev, dtype=torch.float64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            tb, tc = float(t[0]), float(t[1])
        del gb
    lo, hi = shard_slices(per_gpu * world, world, rank)
    assert hi - lo == per_gpu
    if rank != 0:
        return None
    sl = 1e3 / statistics.mean(inf_ms)
    slb = per_gpu * world * reps / (tb * 1e-3)
    return {"metric": "512x512 denoised slices/s (generator inference)",
            "batch1": {"config": "BASELINE configs[1]: 1x1x512x512, one CUDA-graph replay per slice", "value": round(sl, 3),
                       "ms_per_slice": round(statistics.mean(inf_ms), 4), "e2e_value": round(1e3 / statistics.mean(inf_e2e), 3),
                       "eager_ms_per_slice": round(eager_ms, 4),
                       "roofline": {"bound": "hbm", "achieved": round(B_ALG_INFER * sl / 1e9, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
                                    "frac": round(B_ALG_INFER * sl / 1e9 / pk["hbm_gbs"], 4), "traffic": INFER_TRAFFIC_BYTES,
                                    "algorithmic_bytes_per_slice": B_ALG_INFER},
                       "kernel_ms_per_entry": per_entry},
            "batched": {"config": f"BASELINE configs[4]: {per_gpu} slices per GPU x {world} GPU(s), slices sharded by rank, no "
                                  f"collective; micro-batch {best[0]} per graph replay", "value": round(slb, 3),
                        "slices": per_gpu * world, "ms_per_slice_per_gpu": round(tb / reps / per_gpu, 4),
                        "e2e_value": round(per_gpu * world * reps / (tc * 1e-3), 3),
                        "h2d_bytes_per_batch": per_gpu * 512 * 512 * 4, "d2h_bytes_per_batch": per_gpu * 512 * 512 * 4,
                        "roofline": {"bound": "hbm", "achieved": round(B_ALG_INFER * slb / world / 1e9, 1), "peak": pk["hbm_gbs"],
                                     "unit": "GB/s", "frac": round(B_ALG_INFER * slb / world / 1e9 / pk["hbm_gbs"], 4)},
                        "timing": "CUDA events around the whole batch, max over ranks, 256 MiB L2 flush between batches"},
            "value": round(slb, 3), "scaling": "weak (independent slices; no collective)"}


def run_gpu_eager_baseline(dev, xd, yd):
    """The GPU bar (SURVEY §8d Config 3): the reference's algorithm as plain torch ops (the oracle restatement; cuDNN /
    cuFFT / ATen kernels, torch-eager) on the SAME B200, same weights and inputs, timed with CUDA events.  Never the
    product path -- a reported baseline like cpu_baseline."""
    from oracle.train_step import OracleTrainer
    sd = {k: v.to(dev) for k, v in oracle_state().items()}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark,
             torch.backends.cudnn.deterministic)
    out = {"what": "oracle restatement of engine.py:40-55 in torch-eager on cuda (cuDNN/cuFFT/ATen), B=20 64x64, "
                   "3 warm-up + 8 timed steps, CUDA events", "torch": torch.__version__,
           "cudnn": torch.backends.cudnn.version()}
    modes = {"fp32_reference_flags": dict(tf32=False, bench=False, det=True),       # train.py:75-76 + TF32 off (fp32 parity)
             "tf32_reference_flags": dict(tf32=True, bench=False, det=True),        # train.py:75-76, torch's default conv TF32
             "tf32_cudnn_benchmark": dict(tf32=True, bench=True, det=False)}        # fastest stock configuration
    try:
        for name, m in modes.items():
            torch.backends.cudnn.allow_tf32 = m["tf32"]
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.benchmark = m["bench"]
            torch.backends.cudnn.deterministic = m["det"]
            random.seed(2024)
            tr = OracleTrainer(sd)
            for _ in range(3):
                tr.step(xd, yd)
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(8)]
            for s, e in ev:
                s.record(); tr.step(xd, yd); e.record()
            torch.cuda.synchronize()
            ms = statistics.median(s.elapsed_time(e) for s, e in ev)
            out[name] = {"ms_per_step": round(ms, 3), "patches_per_s": round(BATCH / ms * 1e3, 2)}
            del tr
        # generator inference, batch 1, 512x512 (configs[1]) in the same three modes' fastest and fp32
        from oracle import mtdgan_oracle as O
        from mtdgan_b200.data import synthetic_pair
        xs = synthetic_pair(1, 512, seed=4321)[0].to(dev)
        gsd = {k[len("Generator."):]: v for k, v in sd.items() if k.startswith("Generator.")}
        for name, tf32 in (("infer512_fp32", False), ("infer512_tf32", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cudnn.benchmark = True
            torch.backends.cudnn.deterministic = False
            with torch.no_grad():
                for _ in range(3):
                    O.generator_forward(gsd, xs)
                torch.cuda.synchronize()
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
                for s, e in ev:
                    s.record(); O.generator_forward(gsd, xs); e.record()
                torch.cuda.synchronize()
            ms = statistics.median(s.elapsed_time(e) for s, e in ev)
            out[name] = {"ms_per_slice": round(ms, 3), "slices_per_s": round(1e3 / ms, 2)}
    finally:
        (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark,
         torch.backends.cudnn.deterministic) = saved
    return out


def measure_tf32_peak(dev):
    """Dense TF32 matmul peak measured the way MEASURED_PEAKS.json measured bf16: torch.matmul 8192^3 with
    allow_tf32, best of 10 (burst) and back to back for ~2 s (sustained)."""
    saved = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); a @ b; e.record()
            torch.cuda.synchronize()
            best = min(best, s.elapsed_time(e))
        reps = max(10, int(2000.0 / best))
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            a @ b
        e.record()
        torch.cuda.synchronize()
        sus = s.elapsed_time(e) / reps
        fl = 2.0 * n ** 3
        return {"tf32_tflops": round(fl / best / 1e9, 1), "tf32_tflops_sustained": round(fl / sus / 1e9, 1),
                "how": "torch.matmul fp32 8192^3, torch.backends.cuda.matmul.allow_tf32=True: best of 10 / back to back ~2 s"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = saved


# ----------------------------------------------------------------------------------------------------
# CPU legs (oracle port)
# ----------------------------------------------------------------------------------------------------
def oracle_state():
    """Reference-identical initial weights (the drop-in modules reproduce the reference's init RNG order)."""
    from arch.Ours.networks import MTD_GAN_Method
    torch.manual_seed(2024)
    random.seed(2024)
    m = MTD_GAN_Method()
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def cpu_train_steps(batch, steps, warmup):
    from oracle.train_step import OracleTrainer
    from oracle.mtdgan_oracle import synthetic_pair
    torch.set_num_threads(os.cpu_count())
    tr = OracleTrainer(oracle_state())
    x, y = synthetic_pair(batch, PATCH, seed=1234)
    for _ in range(warmup):
        tr.step(x, y)
    t0 = time.perf_counter()
    for _ in range(steps):
        tr.step(x, y)
    return (time.perf_counter() - t0) / max(steps, 1)


def run_cpu_baseline():
    """Bounded sample (~10-30 s of CPU work) of the SAME workload as the GPU arm and the reference arm: 1 warm-up + 3
    timed train steps on 20 synthetic 64x64 patches (BASELINE configs[2])."""
    code = (f"import bench, json; t = bench.cpu_train_steps({BATCH}, 3, 1); "
            "print(json.dumps({'s_per_step': t}))")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    t = json.loads(r.stdout.strip().splitlines()[-1])["s_per_step"]
    return {"value": round(BATCH / t, 4), "unit": "patches/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"oracle port (torch-CPU, all host threads) of the full train step on {BATCH} synthetic 64x64 patches "
                      "(BASELINE configs[2], the GPU arm's batch): 1 warm-up + 3 timed steps", "s_per_step": round(t, 3)}


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return None
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    from oracle.train_step import OracleTrainer
    from oracle.mtdgan_oracle import synthetic_pair
    torch.set_num_threads(os.cpu_count())
    tr = OracleTrainer(oracle_state())
    # The batch is ALWAYS the GPU arm's (20 patches), so the two arms compare equal configurations; --steps sets the
    # number of timed steps (patches/s is a rate, so fewer steps suit a slow host).  At least one untimed step runs first.
    batch = BATCH
    x, y = synthetic_pair(batch, PATCH, seed=1234)
    for _ in range(max(1, args.warmup)):
        tr.step(x, y)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tr.step(x, y)
    dt = time.perf_counter() - t0
    v = round(batch * args.steps / dt, 4)
    return {"impl": "reference", "metric": "train patches/s (64x64, bs20/GPU)", "value": v, "unit": "patches/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "MTD_GAN_Method full train step (G + MTL-D + RC/NDS + PCGrad + AdamW), 20 synthetic 1x64x64 "
                                   "patches (BASELINE configs[2]): CPU oracle port of the reference (torch-CPU, all host threads)",
                       "global_batch": batch, "patch": PATCH, "parallelism": "cpu"},
            "cpu_baseline": {"value": v, "unit": "patches/s", "cores": os.cpu_count(), "kind": "port",
                             "sample": f"{args.steps} timed steps of {batch} synthetic 64x64 patches each"},
            "e2e": {"value": v, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of the captured CUDA graph")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the torch-eager-on-GPU baseline leg")
    ap.add_argument("--infer-batch", type=int, default=64, help="512x512 slices per GPU of the batched inference leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed train step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    claim_stdout()
    if args.impl == "reference":
        line = run_reference(args)
        if line is not None:
            emit(line)
        return
    line = run_own(args)
    rank, world, _ = dist_env()
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = run_cpu_baseline()
            except Exception as ex:      # the baseline leg must never take the measurement down with it
                line["cpu_baseline"] = {"value": None, "unit": "patches/s", "cores": os.cpu_count(), "kind": "port",
                                        "sample": f"failed: {type(ex).__name__}: {ex}"}
        emit(line)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
