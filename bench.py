#!/usr/bin/env python
"""bench.py — IRFD train-step throughput on B200 (BASELINE.json metric: IRFD train samples/sec @256^2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--batch B] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A step = one generator training step of the reference (train.py:186-210 restricted to the differentiable losses,
SURVEY §8(d) config 3): zero_grad -> IRFD.forward (train mode, inputs require grad so the encoders are differentiated)
-> MSE(x_s,x̂_s)+MSE(x_t,x̂_t)+MSE(fi_s,fi_t) -> backward -> Adam(lr 2e-4) on Gd.  `--batch` pairs per GPU (default
32: BASELINE config 3 at N=1, weak scaling to config 4's global 256 at N=8).  Synthetic U(-1,1) 256x256 pairs,
random-init weights (seed 0).  Prints ONE JSON line on rank 0.

--impl reference: the CPU restatement of the reference (oracle/irfd_oracle.py, "port": the reference itself is Python
and does not travel to the GPU box) running the same step on the host cores, on a bounded sample.

--dump-outputs DIR (native arm, rank 0): after the timed steps, what the last timed step computed is written as
DIR/<name>.npy, so that two builds run with the same arguments (same seeded inputs and weights) can be compared output
for output.  train: the step's loss, Gd's parameters after the Adam update and its gradients, every encoder stage's
gradients and the encoders' BatchNorm running statistics; gen_infer / infer512: the generated images; d_step: the loss,
its three terms, D's parameters after the update and its gradients.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_TRAIN_PER_PAIR = 529.4e9   # algorithmic, fwd + 2x bwd, recompute not counted (BASELINE.md §2)
METRIC = "irfd_train_pairs_per_sec_256"
UNIT = "pairs/s"

# Every BASELINE.json config that runs on a GPU.  The default invocation is `train` (config 3; config 4 = the same
# step at N>1, `--global-batch 256` gives the 2x128 / 4x64 / 8x32 shards it names).
CONFIGS = {
    "train": {"metric": METRIC, "unit": UNIT, "flops_per_unit": FLOPS_TRAIN_PER_PAIR, "batch": 32},
    # config 2: StyleGenerator inference alone, eval, features |N(0,1)|*0.5 (SURVEY §8(d)); 56.195 GF per image
    "gen_infer": {"metric": "gd_infer_images_per_sec_256", "unit": "images/s", "flops_per_unit": 56.195e9, "batch": 32},
    # config 5: IRFD inference at 512^2 with SynthesisNetwork(resolution=512), 8 pairs per GPU, replicas only
    "infer512": {"metric": "irfd_infer_pairs_per_sec_512", "unit": "pairs/s", "flops_per_unit": 397.7e9, "batch": 8},
    # SURVEY §8(f) N1: the discriminator step (train.py:157-183).  Per pair: D forward on 4 images (119.2 GF) + their
    # backward (238.4) + R1 on 2 images (forward, image-gradient chain, second-order forward chain, wgrads: 238.4) +
    # one IRFD forward under no_grad (176.45) = 772.5 GF (D forward 29.8 GF / image, SURVEY §8(f))
    "d_step": {"metric": "irfd_d_step_pairs_per_sec_256", "unit": "pairs/s", "flops_per_unit": 772.5e9, "batch": 32},
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="train", choices=sorted(CONFIGS), help="BASELINE.json workload (default: "
                    "config 3, the G train step)")
    ap.add_argument("--batch", type=int, default=0, help="units (pairs / images) per GPU; 0 = the config's own")
    ap.add_argument("--global-batch", type=int, default=0, help="total pairs over all GPUs (config 4: 256)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="the step's launch sequence launched kernel by kernel "
                    "instead of as one CUDA graph (profiling: ncu lists the same kernels the graph replays)")
    ap.add_argument("--cpu-sample", type=int, default=8, help="pairs per CPU-baseline step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write what the last timed step computed as "
                    "DIR/<name>.npy (float32 / float64, a fixed seeded sample of large arrays, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the native arm's outputs (--impl native)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.global_batch:
        if args.global_batch % world:
            ap.error(f"--global-batch {args.global_batch} does not split over {world} ranks")
        args.batch = args.global_batch // world
    if not args.batch:
        args.batch = CONFIGS[args.config]["batch"]
    return args


DUMP_MAX_ELEMENTS = 1 << 21   # per array; a larger one is written as a sample of about this many elements
DUMP_MAX_BYTES = 64 << 20
DUMP_SEED = 20240229


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each tensor as out_dir/<name>.npy: float64 stays float64, every other dtype becomes float32.  A tensor of
    more than DUMP_MAX_ELEMENTS elements is flattened and sampled at sorted indices drawn from DUMP_SEED, so runs with
    the same arguments sample the same positions."""
    import numpy as np
    import torch

    out = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMENTS:
            g = torch.Generator().manual_seed(DUMP_SEED)
            idx = torch.randint(0, t.numel(), (DUMP_MAX_ELEMENTS,), generator=g).unique()
            t = t.reshape(-1)[idx.to(t.device)]
        out[name] = (t if t.dtype == torch.float64 else t.float()).cpu().numpy()
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.lines:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle port)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_train_steps(pairs: int, steps: int, warmup: int, budget_s: float):
    """Reference G step on the host cores with the oracle modules.  Returns (pairs/s, steps done, threads, seconds)."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import irfd_oracle as O

    threads = os.cpu_count() or 1
    try:
        threads = len(os.sched_getaffinity(0))
    except Exception:
        pass
    torch.set_num_threads(threads)
    torch.manual_seed(O.WEIGHT_SEED)
    net = O.IRFDRef(use_checkpoint=True).train()
    opt = torch.optim.Adam(net.Gd.parameters(), lr=2e-4)
    x_s, x_t = O.synthetic_pair(pairs)

    def step():
        opt.zero_grad(set_to_none=True)
        for p in net.parameters():
            p.grad = None
        xs, xt = x_s.clone().requires_grad_(True), x_t.clone().requires_grad_(True)
        out = net(xs, xt)
        l_id, l_rec = O.irfd_losses(xs, xt, out)
        (l_id + l_rec).backward()
        opt.step()
        return float((l_id + l_rec).detach())

    torch.manual_seed(O.FORWARD_SEED)
    t_start = time.time()
    for _ in range(warmup):
        step()
        if time.time() - t_start > budget_s / 3:
            break
    done, t0 = 0, time.time()
    for _ in range(steps):
        step()
        done += 1
        if time.time() - t_start > budget_s:
            break
    dt = time.time() - t0
    return pairs * done / dt, done, threads, dt


def _host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_infer_steps(config: str, units: int, steps: int, warmup: int, budget_s: float):
    """Oracle port of the inference configs on the host cores (eval mode, no_grad).  gen_infer: one StyleGenerator
    call on `units` feature rows; infer512: IRFD.forward on `units` 512^2 pairs with SynthesisNetwork(resolution=512).
    Returns (units/s, steps done, threads, seconds)."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import irfd_oracle as O

    threads = _host_threads()
    torch.set_num_threads(threads)
    torch.manual_seed(O.WEIGHT_SEED)
    if config == "gen_infer":
        net = O.StyleGeneratorRef(input_dim=6144).eval()
        feat = torch.randn(units, 6144, generator=torch.Generator().manual_seed(O.DATA_SEED)).abs() * 0.5

        def step():
            with torch.no_grad():
                return net(feat)
    else:
        net = O.IRFDRef()
        net.Gd = O.StyleGeneratorRef(input_dim=6144, resolution=512)
        net = net.eval()
        x_s, x_t = O.synthetic_pair(units, res=512)

        def step():
            with torch.no_grad():
                return net(x_s, x_t)

    t_start = time.time()
    for _ in range(warmup):
        step()
        if time.time() - t_start > budget_s / 3:
            break
    done, t0 = 0, time.time()
    for _ in range(steps):
        step()
        done += 1
        if time.time() - t_start > budget_s:
            break
    dt = time.time() - t0
    return units * done / dt, done, threads, dt


CPU_SAMPLE_DESC = {
    "train": "G train step(s) of {u} pair(s) @256^2 (oracle port with reentrant checkpoints, fp32, torch CPU)",
    "gen_infer": "StyleGenerator eval forward(s) on {u} feature rows -> 256^2 images (oracle port, fp32, torch CPU)",
    "infer512": "IRFD eval forward(s) on {u} pair(s) @512^2, SynthesisNetwork(512) (oracle port, fp32, torch CPU)",
    "d_step": "D train step(s) on {u} pair(s) @256^2 (oracle port: 4 D calls + IRFD forward + 2 R1 double backwards + Adam, "
              "fp32, torch CPU)",
}
CPU_UNITS = {"train": 8, "gen_infer": 8, "infer512": 1, "d_step": 1}   # bounded sample of the GPU arm's batch, per CPU step


def cpu_d_steps(pairs: int, steps: int, warmup: int, budget_s: float):
    """Reference D step (train.py:157-183, 246-255) on the host cores with the oracle modules."""
    import torch
    import torch.nn.functional as F

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import irfd_oracle as O

    threads = _host_threads()
    torch.set_num_threads(threads)
    torch.manual_seed(O.WEIGHT_SEED)
    net = O.IRFDRef().train()
    opt = torch.optim.Adam(net.D.parameters(), lr=5e-5)
    x_s, x_t = O.synthetic_pair(pairs)

    def noisy(x):
        return x + torch.randn_like(x) * 0.1

    def bce(logits, label):
        return F.binary_cross_entropy_with_logits(logits, torch.full_like(logits, label))

    def r1(x):
        x = x.clone().requires_grad_(True)
        g = torch.autograd.grad(outputs=net.D(x).sum(), inputs=x, create_graph=True)[0]
        return g.pow(2).reshape(g.shape[0], -1).sum(1).mean()

    def step():
        opt.zero_grad(set_to_none=True)
        loss = (bce(net.D(noisy(x_s)), 0.9) + bce(net.D(noisy(x_t)), 0.9)) / 2
        with torch.no_grad():
            out = net(x_s, x_t)
        loss = loss + (bce(net.D(noisy(out[0])), 0.1) + bce(net.D(noisy(out[1])), 0.1)) / 2
        loss = loss + (r1(x_s) + r1(x_t)) / 2
        loss.backward()
        opt.step()

    t_start = time.time()
    for _ in range(warmup):
        step()
        if time.time() - t_start > budget_s / 3:
            break
    done, t0 = 0, time.time()
    for _ in range(steps):
        step()
        done += 1
        if time.time() - t_start > budget_s:
            break
    dt = time.time() - t0
    return pairs * done / dt, done, threads, dt


def cpu_arm(config: str, units: int, steps: int, warmup: int, budget_s: float):
    if config == "train":
        return cpu_train_steps(units, steps, warmup, budget_s)
    if config == "d_step":
        return cpu_d_steps(units, steps, warmup, budget_s)
    return cpu_infer_steps(config, units, steps, warmup, budget_s)


def run_reference(args):
    """The reference's own CPU path (oracle port: the reference is Python and does not travel to the GPU box), all
    host threads, same --steps / --warmup as the native arm, each step a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    units = CPU_UNITS[args.config]
    # no time budget: every one of the --steps steps is timed
    val, done, threads, dt = cpu_arm(args.config, units, args.steps, args.warmup, budget_s=float("inf"))
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": val, "unit": cfg["unit"], "n_gpus": args.gpus,
        "steps": done, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(done, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_DESC[args.config] + " — on host CPU, oracle port of the reference",
                   "units_per_step": units, "pairs_per_step": units if args.config != "gen_infer" else None},
        "cpu_baseline": {"value": val, "unit": cfg["unit"], "cores": threads, "kind": "port",
                         "sample": f"{done} " + CPU_SAMPLE_DESC[args.config].format(u=units) + f", {dt:.1f} s"},
        "e2e": {"value": val, "unit": cfg["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


WORKLOAD_DESC = {
    "train": "IRFD G train step (3xResNet-50 enc x2 images + S<->T swap + StyleGAN-v1 gen x2 + 3xMSE + backward incl. "
             "encoders + Adam on Gd) @256^2, BASELINE config 3",
    "gen_infer": "StyleGenerator inference alone (mapping + synthesis: 12 conv3x3 with noise/lrelu/style epilogues, "
                 "bilinear x2, to_rgb) @256^2, eval, BASELINE config 2",
    "infer512": "IRFD inference (6 encoder passes on 512^2 images + swap + 2 generator calls with "
                "SynthesisNetwork(resolution=512)), eval, BASELINE config 5",
    "d_step": "IRFD discriminator step (4 x D forward/backward on instance-noised real and reconstructed images, IRFD "
              "forward under no_grad, R1 penalty x2 with its second-order chain, Adam on D) @256^2, train.py:157-183 "
              "(SURVEY §8(f) N1)",
}


# ----------------------------------------------------------------------------------------------------------------------
# native arm
# ----------------------------------------------------------------------------------------------------------------------
def _teardown(trainer, dist, world):
    """Multi-rank exit: a captured CUDA graph that contains NCCL kernels keeps the communicator busy and
    destroy_process_group() blocks on it, so release the graph, rendezvous once more and leave without destroying."""
    if world <= 1:
        return
    import torch

    if trainer is not None:
        trainer.graph = None
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


def build_roofline(fam, rsteps):
    """Roofline object of the dominant tensor-core family from per-launch CUDA-event records (ops.gemm_timing_end())."""
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained")
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    if not peak_tf:
        peak_tf, peak_src = 1400.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)"
    hbm = {k: v for k, v in fam.items() if k.endswith("HBM)")}      # memory-bound families: "flops" holds bytes
    fam = {k: v for k, v in fam.items() if k not in hbm}
    top = max(fam.values(), key=lambda f: f["ms"]) if fam else None
    roofline = None
    peak_bw = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None
    try:  # per-launch DRAM bytes of the dominant family from the committed ncu capture (scripts/ncu_traffic.sh)
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
            traffic = json.load(fh)
    except Exception:
        pass

    def fam_entry(v):
        # per-launch roofline: each launch is bounded by max(flops / tensor peak, algorithmic bytes / HBM peak)
        bound_ms = sum(max(f / (peak_tf * 1e12), b / (peak_bw * 1e9)) * 1e3 for _, f, b in v["records"])
        hbm_bound = sum(1 for _, f, b in v["records"] if b / (peak_bw * 1e9) > f / (peak_tf * 1e12))
        return {"ms_per_step": v["ms"] / rsteps, "tflops": v["flops"] / (v["ms"] * 1e-3) / 1e12,
                "launches_per_step": v["launches"] / rsteps, "gflop_per_step": v["flops"] / rsteps / 1e9,
                "algorithmic_gbytes_per_step": v["bytes"] / rsteps / 1e9,
                "per_launch_bound_ms_per_step": bound_ms / rsteps, "frac_of_per_launch_bound": bound_ms / v["ms"],
                "hbm_bound_launches_per_step": hbm_bound / rsteps}

    if top:
        ach = top["flops"] / (top["ms"] * 1e-3) / 1e12
        tr = (traffic or {}).get(top["name"])
        roofline = {"bound": "tensor", "kernel": top["name"], "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": ach / peak_tf, "traffic": tr["dram_bytes_per_launch"] if tr else None,
                    "algorithmic_bytes_per_launch": top["bytes"] / max(top["launches"], 1),
                    "peak_source": peak_src,
                    "launches_per_step": top["launches"] / rsteps, "ms_per_step": top["ms"] / rsteps,
                    "families": {k: fam_entry(v) for k, v in fam.items()},
                    "hbm_families": {k: {"ms_per_step": v["ms"] / rsteps, "gbytes_per_step": v["flops"] / rsteps / 1e9,
                                         "achieved_gbs": v["flops"] / (v["ms"] * 1e-3) / 1e9,
                                         "frac_of_measured_hbm": v["flops"] / (v["ms"] * 1e-3) / 1e9 / peak_bw}
                                     for k, v in hbm.items()},
                    "ncu": "profiles/r2_final_launches_summary.md (launch list with DRAM bytes), profiles/r2b_ncu_full_summary.md + r2_ncu_full_summary.md "
                           "(--set full of the top kernels), profiles/r2_conv_shapes.md (per-shape roofline), "
                           "profiles/r2_graph_timeline.md"}

    return roofline


def run_native(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl native needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import speak_hack_b200 as P
    from speak_hack_b200 import ops
    from speak_hack_b200.trainer import IRFDTrainer

    B = args.batch
    torch.manual_seed(0)                        # identical weights on every rank
    model = P.IRFD().to(dev).train()
    trainer = IRFDTrainer(model, lr=2e-4, use_cuda_graph=not args.no_graph)
    if args.no_graph:
        trainer.train_step = trainer.train_step_static_eager
    g = torch.Generator().manual_seed(7 + rank)  # each rank its own shard of the global batch
    host_s = (torch.rand(B, 3, 256, 256, generator=g) * 2 - 1).pin_memory()
    host_t = (torch.rand(B, 3, 256, 256, generator=g) * 2 - 1).pin_memory()
    x_s, x_t = host_s.to(dev), host_t.to(dev)
    torch.manual_seed(11)                       # same CPU draws (swap, style mixing) on every rank

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        trainer.train_step(x_s, x_t)
    barrier()

    # ---- timed region 1: inputs resident in HBM ("value")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    ops.launch_count = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    for _ in range(args.steps):
        trainer.train_step(x_s, x_t)
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms_value = max_over_ranks(e0.elapsed_time(e1))
    launches = ops.launch_count
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None

    # ---- timed region 2: end to end (pinned host inputs -> H2D every step, loss read back every step)
    barrier()
    copy_stream = torch.cuda.Stream(dev)
    main_stream = torch.cuda.current_stream(dev)

    stage = [(torch.empty_like(x_s), torch.empty_like(x_t)) for _ in range(2)]   # double-buffered device staging
    consumed = [None, None]                                                       # main-stream event: buffer read

    def h2d(slot):
        """One step's inputs, pinned host -> device staging buffer `slot`, on the copy stream."""
        with torch.cuda.stream(copy_stream):
            if consumed[slot] is not None:
                copy_stream.wait_event(consumed[slot])
            stage[slot][0].copy_(host_s, non_blocking=True)
            stage[slot][1].copy_(host_t, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return ev

    e0.record()
    last = None
    ready = h2d(0)
    for i in range(args.steps):
        slot = i & 1
        main_stream.wait_event(ready)
        loss = trainer.train_step(*stage[slot])  # graph mode: D2D into the static inputs + one graph replay
        consumed[slot] = torch.cuda.Event()
        consumed[slot].record(main_stream)
        if i + 1 < args.steps:
            ready = h2d(slot ^ 1)               # the next step's H2D overlaps this step's compute
        last = float(loss.item())               # D2H of the step's result
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs and rank == 0:   # before the passes below move the parameters again
        from speak_hack_b200.trainer import STAGES

        arrays = {"loss": loss, "gd_params": trainer.flat, "gd_grads": trainer.gflat}
        arrays.update({f"encoder_grads_stage{k}": trainer.stage_flats[k] for k in STAGES})
        arrays["encoder_bn_buffers"] = torch.cat([b.reshape(-1).float() for e in trainer.encoders
                                                  for b in e.buffers() if b.is_floating_point()])
        dump_outputs(args.dump_outputs, arrays)

    # ---- N > 1: on-hardware check of the exchange (reference semantics: DDP averages the per-rank gradients,
    # train.py:399-401).  One step through the captured graph WITH its NCCL buckets, then — from the same parameters,
    # BN buffers, CPU draws and device RNG seed — one step through a second graph captured WITHOUT communication; the
    # per-rank gradients of the second are all-gathered and their mean compared with the first's buffers.
    dp_check = None
    if world > 1 and trainer.use_cuda_graph:
        snap = trainer.snapshot()

        def seeded_step():
            torch.manual_seed(1234)
            torch.cuda.manual_seed(4321)
            trainer.train_step(x_s, x_t)
            torch.cuda.synchronize()
            return [g.clone() for g in trainer.gradient_buffers()]

        averaged = seeded_step()
        trainer.restore(snap)
        trainer.buckets.enabled = False          # changes the graph key: the step is recaptured without collectives
        local = seeded_step()
        trainer.buckets.enabled = True
        trainer.restore(snap)
        worst = 0.0
        for a, l in zip(averaged, local):
            parts = [torch.empty_like(l) for _ in range(world)]
            dist.all_gather(parts, l)
            mean = torch.stack([p.double() for p in parts]).mean(0)
            worst = max(worst, float((a.double() - mean).norm() / mean.norm().clamp_min(1e-300)))
        t = torch.tensor([worst], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dp_check = {"max_rel_l2_vs_mean_of_rank_gradients": float(t.item()), "buffers": len(averaged),
                    "elements": int(sum(a.numel() for a in averaged))}

    # ---- roofline pass: per-launch CUDA events around every tensor-core GEMM launch (same stream), few steps
    # (the whole step runs on one stream, so an event pair times exactly the launch between its two records)
    ops.use_side_stream = False                  # weight gradients on the main stream: every launch timed alone
    ops.gemm_timing_begin()
    rsteps = min(args.steps, 3)
    for _ in range(rsteps):
        # the captured step's own launch sequence, kernel by kernel (events cannot be recorded inside a graph replay)
        trainer.train_step_static_eager(x_s, x_t)
    torch.cuda.synchronize()
    fam = ops.gemm_timing_end()
    if rank != 0:
        _teardown(trainer, dist, world)
        return

    roofline = build_roofline(fam, rsteps)

    n_pairs = B * world * args.steps
    value = n_pairs / (ms_value * 1e-3)
    e2e_val = n_pairs / (ms_e2e * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_value / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD_DESC["train"], "pairs_per_step": B * world,
                   "pairs_per_gpu": B, "global_batch_pairs": B * world, "parallelism": f"dp{world}",
                   "launch_mode": "one CUDA graph per step" if trainer.use_cuda_graph else "eager",
                   "l2_policy": "inputs+activations (>10 GB/step) far exceed the 126 MB L2; no explicit flush",
                   "algorithmic_tflop_per_step_per_gpu": FLOPS_TRAIN_PER_PAIR * B / 1e12},
        "model_tflops_per_gpu": FLOPS_TRAIN_PER_PAIR * B / (ms_value / args.steps * 1e-3) / 1e12,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": 2 * host_s.numel() * 4,
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps, "last_loss": last},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
    }
    if dp_check is not None:
        line["dp_check"] = dp_check
    if world == 1 and not args.no_cpu_baseline:
        try:
            val, done, threads, dt = cpu_train_steps(args.cpu_sample, 3, 1, budget_s=90.0)
            line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"{done} " + CPU_SAMPLE_DESC["train"].format(u=args.cpu_sample)
                                              + f", {dt:.1f} s after 1 warm-up step"}
        except Exception as exc:  # the baseline is informative; never lose the GPU line over it
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": f"failed: {exc}"}
    print(json.dumps(line), flush=True)
    _teardown(trainer, dist, world)


def run_native_infer(args):
    """BASELINE configs 2 (gen_infer) and 5 (infer512): eval-mode, no_grad forward captured in one CUDA graph
    (speak_hack_b200/inference.py).  N>1 = N independent replicas ("replicas only": inference has no collective); the
    barrier + max-over-ranks timing of the contract still applies."""
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl native needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import speak_hack_b200 as P
    from speak_hack_b200 import ops
    from speak_hack_b200.inference import GraphedCall, IRFDInference

    cfg = CONFIGS[args.config]
    B = args.batch
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(7 + rank)
    differentiable = args.config == "d_step"
    if args.config == "d_step":
        from speak_hack_b200.trainer import IRFDDiscriminatorStep

        model = P.IRFD().to(dev).train()
        dstep = IRFDDiscriminatorStep(model)
        host_in = [(torch.rand(B, 3, 256, 256, generator=g) * 2 - 1).pin_memory() for _ in range(2)]
        dev_in = [t.to(dev) for t in host_in]
        with torch.no_grad():  # let the spectral-norm power iterations converge (fresh u/v give weights ~1e3 too large)
            for _ in range(6):
                model.D(dev_in[0])
        eager = lambda: dstep.step(*dev_in)                                # noqa: E731
        runner = lambda a, b: dstep.step(a, b)                            # noqa: E731  (eager launches: no graph)
        pick = lambda out: [out.reshape(1)]                                # noqa: E731
        names = ["loss"]
    elif args.config == "gen_infer":
        model = P.StyleGenerator(input_dim=6144).to(dev).eval()
        host_in = [(torch.randn(B, 6144, generator=g).abs() * 0.5).pin_memory()]
        dev_in = [t.to(dev) for t in host_in]
        eager = lambda: model(*dev_in)                                     # noqa: E731
        runner = GraphedCall(lambda f: model(f), dev_in) if not args.no_graph else None
        pick = lambda out: [out]                                           # noqa: E731
        names = ["images"]
    else:
        model = P.IRFD()
        model.Gd.synthesis = P.SynthesisNetwork(resolution=512)            # BASELINE config 5 / SURVEY Q9
        model = model.to(dev)
        host_in = [(torch.rand(B, 3, 512, 512, generator=g) * 2 - 1).pin_memory() for _ in range(2)]
        dev_in = [t.to(dev) for t in host_in]
        # fresh BatchNorm running statistics make eval-mode activations reach 1e18 (SURVEY Q6): give the buffers two
        # train-mode forwards first so the timed inference runs on representative magnitudes
        model.train()
        with torch.no_grad():
            for _ in range(2):
                model(*dev_in)
        model.eval()
        eager = lambda: model(*dev_in)                                     # noqa: E731
        runner = IRFDInference(model, *dev_in) if not args.no_graph else None
        pick = lambda out: [out[0], out[1]]                                # noqa: E731
        names = ["x_s_recon", "x_t_recon"]
    torch.manual_seed(11)

    def step(inputs):
        if differentiable:
            return runner(*inputs)
        with torch.no_grad():
            return runner(*inputs) if runner is not None else model(*inputs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        out = step(dev_in)
    barrier()
    finite = bool(all(torch.isfinite(o).all() for o in pick(out)))

    # ---- timed region 1: inputs resident in HBM
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    ops.launch_count = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    for _ in range(args.steps):
        step(dev_in)
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms_value = max_over_ranks(e0.elapsed_time(e1))
    launches = ops.launch_count
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None

    # ---- timed region 2: end to end.  Every step: pinned host inputs -> device (copy stream, double-buffered), one
    # forward, the generated images -> pinned host (D2H stream, double-buffered).  The host waits for step i-1's images
    # while step i computes, and for the last step's images before the clock stops.
    barrier()
    main_stream = torch.cuda.current_stream(dev)
    h2d_stream, d2h_stream = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    stage_in = [[torch.empty_like(t) for t in dev_in] for _ in range(2)]
    outs0 = pick(out)
    stage_out = [[torch.empty_like(o) for o in outs0] for _ in range(2)]
    host_out = [[torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs0] for _ in range(2)]
    consumed, fetched = [None, None], [None, None]

    def h2d(slot):
        with torch.cuda.stream(h2d_stream):
            if consumed[slot] is not None:
                h2d_stream.wait_event(consumed[slot])
            for d, h in zip(stage_in[slot], host_in):
                d.copy_(h, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(h2d_stream)
        return ev

    e0.record()
    ready = h2d(0)
    for i in range(args.steps):
        slot = i & 1
        main_stream.wait_event(ready)
        if fetched[slot] is not None:
            main_stream.wait_event(fetched[slot])       # stage_out[slot] has been read by its D2H copy
        o = pick(step(stage_in[slot]))
        for d, src in zip(stage_out[slot], o):
            d.copy_(src, non_blocking=True)             # the graph's static outputs are overwritten by the next replay
        done = torch.cuda.Event()
        done.record(main_stream)
        consumed[slot] = done
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(done)
            for h, d in zip(host_out[slot], stage_out[slot]):
                h.copy_(d, non_blocking=True)
            fetched[slot] = torch.cuda.Event()
            fetched[slot].record(d2h_stream)
        if i + 1 < args.steps:
            ready = h2d(slot ^ 1)
        if i >= 1:
            fetched[slot ^ 1].synchronize()             # the previous step's images are on the host
    d2h_stream.synchronize()
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    checksum = float(host_out[(args.steps - 1) & 1][0].double().abs().mean())
    if args.dump_outputs and rank == 0:
        arrays = dict(zip(names, host_out[(args.steps - 1) & 1]))
        if args.config == "d_step":
            arrays.update(zip(("loss_real", "loss_fake", "r1"), dstep.last))
            arrays.update(d_params=dstep.flat, d_grads=dstep.gflat)
        dump_outputs(args.dump_outputs, arrays)

    # ---- roofline pass: eager launches, per-launch CUDA events around every tensor-core GEMM (one stream)
    ops.use_side_stream = False
    ops.gemm_timing_begin()
    rsteps = min(args.steps, 3)
    with torch.set_grad_enabled(differentiable):
        for _ in range(rsteps):
            eager()
    torch.cuda.synchronize()
    fam = ops.gemm_timing_end()
    if rank != 0:
        _teardown(None, dist, world)
        return
    roofline = build_roofline(fam, rsteps)

    units = B * world * args.steps
    ms_step = ms_value / args.steps
    line = {
        "metric": cfg["metric"], "value": units / (ms_value * 1e-3), "unit": cfg["unit"], "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD_DESC[args.config], "units_per_gpu": B, "units_per_step": B * world,
                   "parallelism": f"replicas x{world} (no collective)" if world > 1 else "single GPU",
                   "launch_mode": ("eager launches" if differentiable or runner is None else "one CUDA graph per forward"),
                   "l2_policy": "activations of one forward (>1 GB) exceed the 126 MB L2; no explicit flush",
                   "algorithmic_tflop_per_step_per_gpu": cfg["flops_per_unit"] * B / 1e12,
                   "outputs_finite": finite},
        "model_tflops_per_gpu": cfg["flops_per_unit"] * B / (ms_step * 1e-3) / 1e12,
        "e2e": {"value": units / (ms_e2e * 1e-3), "unit": cfg["unit"],
                "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in host_in),
                "d2h_bytes_per_step": sum(o.numel() * o.element_size() for o in outs0),
                "ms_per_step": ms_e2e / args.steps, "output_abs_mean": checksum},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
    }
    if world == 1 and not args.no_cpu_baseline:
        try:
            u = CPU_UNITS[args.config]
            val, done, threads, dt = cpu_arm(args.config, u, 2 if args.config == "d_step" else 3, 1, budget_s=90.0)
            line["cpu_baseline"] = {"value": val, "unit": cfg["unit"], "cores": threads, "kind": "port",
                                    "sample": f"{done} " + CPU_SAMPLE_DESC[args.config].format(u=u)
                                              + f", {dt:.1f} s after 1 warm-up step"}
        except Exception as exc:
            line["cpu_baseline"] = {"value": None, "unit": cfg["unit"], "cores": None, "kind": "port",
                                    "sample": f"failed: {exc}"}
    print(json.dumps(line), flush=True)
    _teardown(None, dist, world)


def main():
    args = parse_args()
    wd = float(os.environ.get("IRFD_BENCH_WATCHDOG_S", "0") or 0)
    if wd > 0:  # debugging aid: dump every thread's stack and exit if the run has not finished after `wd` seconds
        import faulthandler

        faulthandler.dump_traceback_later(wd, exit=True)
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "train":
        run_native(args)
    else:
        run_native_infer(args)


if __name__ == "__main__":
    main()
