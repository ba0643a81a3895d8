"""Generator inference rate at several slice sizes: GraphedGenerator (one CUDA-graph replay per micro-batch) at 512 x 512,
the non-power-of-two sizes the Bluestein FFTs open up, and a non-square slice.

    python tools/bench_slice_sizes.py [--out FILE] [--slices 16] [--reps 5]
    python tools/bench_slice_sizes.py --profile [--out FILE]

The timing run reports slices/s and ms per megapixel per (size, micro-batch), with the card name and power limit read in
the same process.  --profile is a separate run (tracing slows the host): torch.profiler over one eager forward per size
at micro-batch 1, kernel time split into the FFT family (kernels named fft_*) and the convolutions (conv_*).
Inputs: --slices seeded slices per size, held on the device (at 512 x 512 and micro-batch 8 one layer's activations are
268 MB, well past the 126 MB L2)."""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

SIZES = [(512, 512), (500, 500), (509, 509), (384, 512), (300, 300)]
MICRO_BATCHES = [1, 8]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def model():
    from arch.Ours.networks import MTD_GAN_Method
    torch.manual_seed(2024)
    random.seed(2024)
    return MTD_GAN_Method().to("cuda").eval().Generator


def slices(n, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    y = torch.clamp(1.6 * torch.rand(n, 1, H, W, generator=g) - 0.3, 0, 1)
    return torch.clamp(y + 0.1 * torch.randn(n, 1, H, W, generator=g), 0, 1).to("cuda")


def timing(G, n, reps):
    from mtdgan_b200.inference import GraphedGenerator
    rows = []
    with torch.no_grad():
        for H, W in SIZES:
            x = slices(n, H, W, seed=H * 1000 + W)
            out = torch.empty_like(x)
            for mb in MICRO_BATCHES:
                runner = GraphedGenerator(G, H, W, micro_batch=mb).capture()
                runner(x, out)
                torch.cuda.synchronize()
                ms = []
                for _ in range(reps):
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record()
                    runner(x, out)
                    e.record()
                    torch.cuda.synchronize()
                    ms.append(s.elapsed_time(e) / n)
                del runner
                t = statistics.median(ms)
                rows.append({"H": H, "W": W, "micro_batch": mb, "slices": n, "reps": reps, "ms_per_slice": round(t, 4),
                             "ms_per_slice_min_max": [round(min(ms), 4), round(max(ms), 4)],
                             "slices_per_s": round(1e3 / t, 2), "ms_per_megapixel": round(t / (H * W / 1e6), 4)})
                print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
    return rows


def profile(G):
    from torch.profiler import ProfilerActivity, profile as tprofile
    rows = []
    with torch.no_grad():
        for H, W in SIZES:
            x = slices(1, H, W, seed=H * 1000 + W)
            G(x)
            torch.cuda.synchronize()
            with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
                G(x)
                torch.cuda.synchronize()
            fam = {"fft": 0.0, "conv": 0.0, "other": 0.0}
            kernels = {}
            for ev in prof.key_averages():
                us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                if us <= 0:
                    continue
                name = ev.key
                f = "fft" if "fft_" in name else "conv" if "conv" in name else "other"
                fam[f] += us / 1e3
                kernels[name[:120]] = round(us / 1e3, 4)
            rows.append({"H": H, "W": W, "ms_by_family": {k: round(v, 4) for k, v in fam.items()},
                         "fft_share": round(fam["fft"] / max(1e-9, sum(fam.values())), 4), "kernels_ms": kernels})
            print(json.dumps({k: v for k, v in rows[-1].items() if k != "kernels_ms"}), file=sys.stderr, flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="write the JSON result here as well as to stdout")
    ap.add_argument("--slices", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_slice_sizes: needs a CUDA device")
    G = model()
    res = {"card": card()}
    if args.profile:
        res["profile_eager_forward_batch1"] = profile(G)
    else:
        res["graphed_inference"] = timing(G, args.slices, args.reps)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
