"""Eager vs graphed discriminator step (IRFDDiscriminatorStep, use_cuda_graph False / True) on the GPU.

    python scripts/bench_d_step_graph.py [--pairs 32] [--min-seconds 1.0] [--rounds 3] [--json OUT]

Two identical 256^2 models (same seed, spectral-norm power iterations converged), one per step flavour: the two steps
are timed alternately, --rounds times each, with CUDA events over at least --min-seconds of back-to-back steps.  Kernel
launches per step are counted for both in a separate profiled step (torch.profiler, CUDA activity: every kernel,
including the ATen ones; a graph replay reports the kernels of its nodes), beside the launches through the project's
C ABI (ops.launch_count).  The card name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed(fn, min_seconds):
    """Mean ms per call of fn() over >= min_seconds of back-to-back calls."""
    reps, total = 0, 0.0
    while total < min_seconds * 1e3:
        n = max(1, reps or 4)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
        reps += n
    return total / reps


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:  # the number still stands, without the power limit beside it
        q = f"unknown ({exc})"
    return name, q


def kernels_per_step(fn):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    from speak_hack_b200 import ops

    torch.cuda.synchronize()
    before = ops.launch_count
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    native = ops.launch_count - before
    names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
    copies = sum(1 for n in names if n.startswith(("Memcpy", "Memset")))
    return {"kernels": len(names) - copies, "memcpy_memset": copies, "abi_launches": native}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=32)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_d_step_graph: needs a CUDA device")
    import speak_hack_b200 as P
    from speak_hack_b200.trainer import IRFDDiscriminatorStep

    dev = torch.device("cuda:0")
    name, power = card()
    g = torch.Generator().manual_seed(7)
    xs, xt = [(torch.rand(args.pairs, 3, 256, 256, generator=g) * 2 - 1).to(dev) for _ in range(2)]
    steps = {}
    for graph in (False, True):
        torch.manual_seed(0)
        net = P.IRFD().to(dev).train()
        with torch.no_grad():
            for _ in range(6):
                net.D(xs)
        ds = IRFDDiscriminatorStep(net, use_cuda_graph=graph)
        steps["graph" if graph else "eager"] = (ds, (lambda d: lambda: d.step(xs, xt))(ds))
    for _, fn in steps.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    out = {"card": name, "power_limit,max_sm_clock": power, "pairs": args.pairs, "res": 256,
           "graph_capture_abi_launches": steps["graph"][0].graph_launches}
    for k, (_, fn) in steps.items():
        out[f"{k}_launches_per_step"] = kernels_per_step(fn)
    ms = {k: [] for k in steps}
    for _ in range(args.rounds):
        for k, (_, fn) in steps.items():
            ms[k].append(timed(fn, args.min_seconds))
    for k, v in ms.items():
        out[f"{k}_ms_per_step"] = v
        out[f"{k}_pairs_per_sec"] = args.pairs / (min(v) * 1e-3)
    out["speedup_graph_over_eager"] = min(ms["eager"]) / min(ms["graph"])
    out["captures"] = steps["graph"][0].captures
    print(json.dumps(out), flush=True)
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
