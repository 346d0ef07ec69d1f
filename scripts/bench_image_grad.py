"""Cost of the encoders' image gradient (the stem's data gradient) on the GPU.

    python scripts/bench_image_grad.py [--pairs 32] [--res 256] [--min-seconds 1.0] [--json OUT]

Kernels, at the lockstep shape (E = 3 encoders, 2 x pairs images of res^2, P = 2 * pairs * (res/2)^2 pixels per
encoder): the dcol GEMM (dz0 [E*P, 64] bf16 @ W -> dcol [E*P, 192] bf16) and col2im_stem (dcol -> dx [2*pairs, 3, res,
res] fp32), each timed alone with CUDA events over at least --min-seconds of back-to-back launches, each against its
byte bound at the HBM bandwidth measured in the same run (a device-to-device copy of 4 GiB).  The working sets
(0.4-1.6 GB) are larger than the 126 MB L2.

End to end: the backward time of mse(Ei(Gd(f)), t) with Ei a lone train-mode encoder over 2 x pairs generated images,
against the same call with Gd's output detached (no image gradient, no generator backward), and the image gradient
alone: Ei on a non-leaf image against the same image as a leaf.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def timed(fn, min_seconds):
    """Mean ms per call of fn() over >= min_seconds of back-to-back calls (after a warm-up call)."""
    fn()
    torch.cuda.synchronize()
    reps, total = 0, 0.0
    while total < min_seconds * 1e3:
        n = max(1, reps or 10)
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=32)
    ap.add_argument("--res", type=int, default=256)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_image_grad: needs a CUDA device")
    import speak_hack_b200 as P
    from speak_hack_b200 import ops

    dev = torch.device("cuda:0")
    name, power = card()
    E, n, res = 3, 2 * args.pairs, args.res
    P_ = n * (res // 2) ** 2
    res_out = {"card": name, "power_limit,max_sm_clock": power, "pairs": args.pairs, "res": res, "E": E,
               "pixels_per_encoder": P_}

    big = torch.empty(1 << 30, dtype=torch.float32, device=dev)
    dst = torch.empty_like(big)
    ms = timed(lambda: dst.copy_(big), args.min_seconds)
    hbm = 2 * big.numel() * 4 / (ms * 1e-3)
    del big, dst
    res_out["hbm_copy_GBps"] = hbm / 1e9

    g = torch.Generator().manual_seed(0)
    ws = [(torch.randn(64, 3, 7, 7, generator=g) * 0.05).to(dev) for _ in range(E)]
    wk = ops.pack_conv_weights_stacked(ws, ops.PACK_FLAT_T, 192)
    dz0 = torch.randn(E * P_, 64, generator=g).to(dev, torch.bfloat16)
    dcol = ops.conv_gemm_grouped(dz0.view(1, 1, -1, 64), wk, 1, wgroups=E)
    gemm_ms = timed(lambda: ops.conv_gemm_grouped(dz0.view(1, 1, -1, 64), wk, 1, wgroups=E), args.min_seconds)
    c2i_ms = timed(lambda: ops.col2im_stem(dcol.view(-1, 192), E, n, res, res), args.min_seconds)
    gemm_bytes = E * P_ * (64 + 192) * 2 + wk.numel() * 2
    # col2im reads the 147 used columns of every dcol row (the zero padding from 147 on is never loaded)
    c2i_bytes = E * P_ * 147 * 2 + n * 3 * res * res * 4
    for key, t, b, flops in (("dcol_gemm", gemm_ms, gemm_bytes, 2.0 * E * P_ * 64 * 192),
                             ("col2im_stem", c2i_ms, c2i_bytes, 0.0)):
        bound = b / hbm * 1e3
        res_out[key] = {"ms": t, "bytes": b, "byte_bound_ms": bound, "share_of_byte_bound": bound / t,
                        "TFLOPs": flops / (t * 1e-3) / 1e12}
    del dz0, dcol

    # end to end: Ei(Gd(f)) with and without the image gradient
    torch.manual_seed(0)
    gd = P.StyleGenerator(input_dim=6144).to(dev).train()
    enc = P.ResNet50Encoder().to(dev).train()
    feat = torch.randn(n, 6144, device=dev) * 0.5
    tgt = torch.randn(n, 2048, 1, 1, device=dev)

    def bwd_ms(make_img, reps=10):
        times = []
        for i in range(reps + 2):
            img = make_img()
            loss = P.mse_loss(enc(img), tgt)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss.backward()
            e1.record()
            e1.synchronize()
            if i >= 2:
                times.append(e0.elapsed_time(e1))
            gd.zero_grad(set_to_none=True)
            enc.zero_grad(set_to_none=True)
        return sorted(times)[len(times) // 2]

    x_leaf = (torch.rand(n, 3, res, res, device=dev) * 2 - 1).requires_grad_(True)
    runs = {k: [] for k in ("chain", "chain_detached", "enc_non_leaf", "enc_leaf")}
    for _ in range(2):   # alternate the variants
        runs["chain"].append(bwd_ms(lambda: gd(feat)))
        runs["chain_detached"].append(bwd_ms(lambda: gd(feat).detach()))
        runs["enc_non_leaf"].append(bwd_ms(lambda: x_leaf * 1))
        runs["enc_leaf"].append(bwd_ms(lambda: x_leaf))
    med = {k: sorted(v)[len(v) // 2] for k, v in runs.items()}
    res_out["backward_ms_median"] = med
    res_out["extra_backward_ms_chain_vs_detached"] = med["chain"] - med["chain_detached"]
    res_out["extra_backward_ms_image_grad_only"] = med["enc_non_leaf"] - med["enc_leaf"]
    res_out["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    print(json.dumps(res_out, indent=1))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res_out, f, indent=1)


if __name__ == "__main__":
    main()
