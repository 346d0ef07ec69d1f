"""Eval-mode IRFD inference at several image sizes: one JSON line per size.

For `--pairs` source/target pairs at each size it times, from CUDA events around CUDA-graph replays (warm-up first, then
at least `--seconds` of replays):
  * the three encoders' eval pass as IRFD.forward runs it (the lockstep EncoderGroup pass when its tiles allow, else the
    per-encoder passes): ms per call and pairs/s;
  * a full IRFDInference call (encoders, device-side swap, generator): ms per call and pairs/s;
and reports the tile fill sum(valid pixels) / (128 * tiles) of each 3x3 stage's conv launch, from the geometry query,
plus the GPU name and power limit read in the same run (nvidia-smi, read-only).

    python scripts/bench_any_size.py [--pairs 64] [--sizes 224,256,320,384,250] [--seconds 1.0]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as e:  # noqa: BLE001 - report what could not be read, keep measuring
        return f"unavailable ({e})", None


def time_call(fn, seconds):
    """ms per call of fn() (a graph replay) from CUDA events: 3 warm-up calls, a short probe, then >= `seconds`."""
    import torch

    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        fn()
    e1.record()
    e1.synchronize()
    probe = e0.elapsed_time(e1) / 5
    iters = max(10, int(seconds * 1000 / max(probe, 1e-3)) + 1)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters, iters


def tile_fill(n_images, h, w, wgroups):
    from speak_hack_b200 import ops

    fills = []
    for hs, ws in ops.resnet_stage_hw(h, w)[1:]:  # the stride-1 3x3 convs of layer1..4
        g = ops.conv_geometry(n_images, hs, ws, 3, wgroups)
        tiles = g[4] * g[5] * g[6]
        fills.append({"hw": [hs, ws], "boxed": bool(g[0]), "box": [g[1], g[2], g[3]], "tiles": tiles,
                      "fill": round(n_images * hs * ws / (128.0 * tiles), 4)})
    return fills


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--sizes", default="224,256,320,384,250")
    ap.add_argument("--seconds", type=float, default=1.0)
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_any_size.py needs a CUDA device (no CPU fallback)")
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import irfd_oracle as O
    import speak_hack_b200 as P
    from speak_hack_b200.inference import GraphedCall, IRFDInference

    dev = torch.device("cuda:0")
    name, power = gpu_info()
    B = args.pairs
    torch.manual_seed(O.WEIGHT_SEED)
    model = P.IRFD().to(dev).train()
    # fresh BatchNorm running statistics blow eval-mode activations up: two train-mode forwards at 256^2 first
    x_s, x_t = O.synthetic_pair(B)
    with torch.no_grad():
        for _ in range(2):
            model(x_s.to(dev), x_t.to(dev))
    model.eval()
    for s in [int(v) for v in args.sizes.split(",")]:
        x_s, x_t = O.synthetic_pair(B, res=s)
        xs, xt = x_s.to(dev), x_t.to(dev)
        lockstep = model.encoder_group.can_run(torch.cat([xs, xt]), 2)
        enc = GraphedCall(lambda a, b: model._encode_all(a, b), [xs, xt])
        enc_ms, enc_iters = time_call(lambda: enc(xs, xt), args.seconds)
        del enc
        full = IRFDInference(model, xs, xt)
        full_ms, full_iters = time_call(lambda: full(xs, xt), args.seconds)
        del full
        torch.cuda.empty_cache()
        line = {
            "size": [s, s], "pairs": B,
            "encoder_path": "lockstep" if lockstep else "per-encoder",
            "encoders_ms": round(enc_ms, 4), "encoders_pairs_per_s": round(B * 1000.0 / enc_ms, 1),
            "encoders_replays": enc_iters,
            "irfd_inference_ms": round(full_ms, 4), "irfd_inference_pairs_per_s": round(B * 1000.0 / full_ms, 1),
            "irfd_inference_replays": full_iters,
            "conv3x3_tile_fill": tile_fill(3 * 2 * B, s, s, 3) if lockstep else tile_fill(B, s, s, 1),
            "gpu": name, "power_limit": power,
        }
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
