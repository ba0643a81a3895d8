#!/usr/bin/env python
"""Device time of every tensor-core weight-gradient call (mtd_conv_wgrad_tc) of one B = 20 train step, at its own shape.

Each call is captured as a CUDA graph and replayed `--reps` times; the L2 is overwritten (256 MB memset) before every
replay, and only the replay lies between the CUDA events.  For each shape the table gives the median us, the plan the
host picked (kernel, Cout tile BN, split over pixels, pipeline stages), the L2 -> SM bytes the kernel's own model
predicts, the compulsory bytes (x + dz read, dW written once) and executed TFLOP/s.  The card's name, power limit and
SM clock are read in the same process.

    python tools/bench_wgrad.py [--reps 20] [--bn 64] [--ksplit 4] [--json out.json]

--bn / --ksplit force the Cout tile / the split (MTD_WG_BN / MTD_WG_KSPLIT) for a sweep."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# (B, H, W, C1, C2, N, k, stride, pad, calls per step): every mtd_conv_wgrad_tc shape of the B = 20 train step, from a
# per-call dump of bench.py (MTD_BENCH_DUMP): the generator's 32-channel layers (B = 20) and the discriminator's
# encoder, task decoders and torch.cat skips (B = 40: real and fake patches in one grouped pass).  (H, W) = input dims.
LAYERS = [
    (20, 64, 64, 32, 0, 32, 3, 1, 1, 41),
    (40, 64, 64, 64, 0, 64, 3, 1, 1, 6),
    (40, 64, 64, 64, 0, 64, 4, 2, 1, 6),
    (40, 32, 32, 64, 0, 256, 1, 1, 0, 1),
    (40, 32, 32, 64, 0, 64, 3, 1, 1, 3),
    (40, 32, 32, 64, 0, 128, 3, 1, 1, 6),
    (40, 32, 32, 128, 128, 64, 3, 1, 1, 3),
    (40, 32, 32, 128, 0, 128, 3, 1, 1, 6),
    (40, 32, 32, 128, 0, 128, 4, 2, 1, 6),
    (40, 16, 16, 128, 0, 512, 1, 1, 0, 1),
    (40, 16, 16, 128, 0, 128, 3, 1, 1, 3),
    (40, 16, 16, 128, 0, 256, 3, 1, 1, 6),
    (40, 16, 16, 256, 256, 128, 3, 1, 1, 3),
    (40, 16, 16, 256, 0, 256, 3, 1, 1, 6),
    (40, 16, 16, 256, 0, 256, 4, 2, 1, 6),
    (40, 8, 8, 256, 0, 1024, 1, 1, 0, 1),
    (40, 8, 8, 256, 0, 256, 3, 1, 1, 3),
    (40, 8, 8, 256, 0, 512, 3, 1, 1, 6),
    (40, 8, 8, 512, 512, 256, 3, 1, 1, 3),
    (40, 8, 8, 512, 0, 512, 3, 1, 1, 6),
    (40, 8, 8, 512, 0, 512, 4, 2, 1, 6),
    (40, 4, 4, 512, 0, 2048, 1, 1, 0, 1),
    (40, 4, 4, 512, 0, 512, 3, 1, 1, 15),
    (40, 4, 4, 512, 512, 512, 3, 1, 1, 3),
    (40, 4, 4, 512, 0, 512, 4, 2, 1, 6),
    (40, 2, 2, 512, 0, 2048, 1, 1, 0, 1),
    (40, 2, 2, 512, 0, 512, 3, 1, 1, 15),
    (40, 2, 2, 512, 512, 512, 3, 1, 1, 3),
    (40, 2, 2, 512, 0, 512, 4, 2, 1, 6),
    (40, 1, 1, 512, 0, 512, 1, 1, 0, 12),
    (40, 1, 1, 512, 0, 2048, 1, 1, 0, 1),
]

KIND = {1: "halo", 0: "taps"}
HALO_BOX = 8 * 10 * 128          # one dx-shifted halo box: 10 rows x 8 pixels x 32 channels x 4 B
BLK = 64 * 128                   # one 32-channel block of a 64-pixel k-step


def out_dims(H, W, k, s, p):
    return (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1


def model_bytes(layer, plan):
    """L2 -> SM bytes of one call under the kernel's own model (every k-step lands its full stage, plain TF32)."""
    B, H, W, C1, C2, N, k, s, p, _ = layer
    kind, bn = plan[0], plan[1]
    Ho, Wo = out_dims(H, W, k, s, p)
    kchunks = (C1 + C2) // 32
    n_nt = N // bn
    if kind == 1:
        ptiles = B * (Ho // 8) * (Wo // 8)
        return ptiles * kchunks * n_nt * (3 * HALO_BOX + bn // 32 * BLK)
    tw = min(Wo, 64)
    th = min(64 // tw, Ho)
    tb = 64 // (tw * th)
    ptiles = (Wo // tw) * (Ho // th) * ((B + tb - 1) // tb)
    units = k * k * kchunks
    per_nt = sum(min(4, units - 4 * m) + bn // 32 for m in range((units + 3) // 4))
    return ptiles * per_nt * BLK * n_nt


def compulsory_bytes(layer):
    B, H, W, C1, C2, N, k, s, p, _ = layer
    Ho, Wo = out_dims(H, W, k, s, p)
    return 4 * (B * H * W * (C1 + C2) + B * Ho * Wo * N + N * k * k * (C1 + C2))


def flop(layer):
    B, H, W, C1, C2, N, k, s, p, _ = layer
    Ho, Wo = out_dims(H, W, k, s, p)
    return 2.0 * B * Ho * Wo * N * (C1 + C2) * k * k


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return [v.strip() for v in q.split(",")]
    except Exception as e:           # the table is still worth having; say why the card line is missing
        return [f"unknown ({e})"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--passes", type=int, default=1, choices=[1, 3])
    ap.add_argument("--bn", type=int, default=0)
    ap.add_argument("--ksplit", type=int, default=0)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if args.bn:
        os.environ["MTD_WG_BN"] = str(args.bn)
    if args.ksplit:
        os.environ["MTD_WG_KSPLIT"] = str(args.ksplit)
    import ctypes
    import torch
    from mtdgan_b200 import _ext
    lib = _ext.load()
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(0)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    print("card:", ", ".join(card()), flush=True)
    print(f"{'layer (B,H,W,C1,C2,N,k,s,p)':36s} {'kernel':>6s} {'BN':>4s} {'ks':>4s} {'kper':>5s} {'CTAs':>5s} {'stg':>4s} "
          f"{'us':>8s} {'model MB':>9s} {'compul MB':>9s} {'TFLOP/s':>8s}")
    rows, tot_us = [], 0.0
    for layer in LAYERS:
        B, H, W, C1, C2, N, k, s, p, calls = layer
        plan = (ctypes.c_int * 5)()
        if hasattr(lib, "mtd_conv_wgrad_tc_plan"):
            if lib.mtd_conv_wgrad_tc_plan(B, H, W, C1, C2, N, k, k, s, p, args.passes, ctypes.addressof(plan)) != 0:
                print(f"{str(layer[:9]):36s} not accepted at this BN / split", flush=True)
                continue
        else:                              # a build from before the plan query: tap-streaming kernel, widest Cout tile
            plan[0], plan[1], plan[3] = 0, 128 if N >= 128 else 64 if N >= 64 else 32, -1
        Ho, Wo = out_dims(H, W, k, s, p)
        x1 = torch.randn(B, H, W, C1, device=dev, generator=gen)
        x2 = torch.randn(B, H, W, C2, device=dev, generator=gen) if C2 else None
        dz = torch.randn(B, Ho, Wo, N, device=dev, generator=gen)
        gp = torch.empty(N, k * k, C1 + C2, device=dev)
        st = torch.cuda.Stream()

        def launch():
            rc = lib.mtd_conv_wgrad_tc(x1.data_ptr(), None if x2 is None else x2.data_ptr(), dz.data_ptr(), gp.data_ptr(),
                                       B, H, W, C1, C2, N, k, k, s, p, args.passes,
                                       ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
            return rc

        with torch.cuda.stream(st):
            rc = launch()                  # warm-up: module load, tensor maps, function attributes
        torch.cuda.synchronize()
        if rc != 0:
            print(f"{str(layer[:9]):36s} not accepted (status {rc})", flush=True)
            continue
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            launch()
        g.replay()
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        us = statistics.median(ts)
        # stages the launcher picks (same rule as launch_wg / launch_wg_halo)
        if plan[0] == 1:
            sb = 3 * HALO_BOX + plan[1] // 32 * BLK
            stages = min(8, 210 * 1024 // sb)
        else:
            sb = (2 if args.passes == 3 else 1) * (4 + plan[1] // 32) * (32 if args.passes == 3 else 64) * 128
            stages = min(8, 200 * 1024 // sb)
        stages = min(stages, max(2, plan[3])) if plan[3] >= 0 else -1      # -1: not known for an older build
        mb = model_bytes(layer, plan) / 1e6 if args.passes == 1 else float("nan")
        cb = compulsory_bytes(layer) / 1e6
        tf = flop(layer) / us / 1e6
        tot_us += us * calls
        row = {"layer": list(layer[:9]), "calls": calls, "kernel": KIND[plan[0]], "bn": plan[1], "ksplit": plan[2],
               "kper": plan[3], "ctas": plan[4], "stages": stages, "us": round(us, 2), "us_min": round(min(ts), 2),
               "model_mb": round(mb, 1), "compulsory_mb": round(cb, 1), "tflops": round(tf, 1)}
        rows.append(row)
        print(f"{str(tuple(layer[:9])):36s} {row['kernel']:>6s} {plan[1]:4d} {plan[2]:4d} {plan[3]:5d} {plan[4]:5d} {stages:4d} "
              f"{us:8.1f} {mb:9.1f} {cb:9.1f} {tf:8.1f}", flush=True)
        del g
    print(f"sum over the step's calls (us x calls per step): {tot_us:.1f} us", flush=True)
    if args.json:
        with open(args.json, "w") as fh:
            json.dump({"card": card(), "passes": args.passes, "bn": args.bn, "ksplit": args.ksplit, "rows": rows,
                       "sum_us": round(tot_us, 1)}, fh, indent=1)


if __name__ == "__main__":
    main()
