"""-m gpu: every tcgen05 GEMM kernel instance (conv_gemm_kernel per-tap / boxed, conv_halo_kernel, wgrad_gemm_kernel,
wgrad_halo_kernel and the split-K reduce kernels) element by element against a float64 reference of the same operation,
at shapes where every CTA serves several tiles.

Reference: float64 from the bf16 operands exactly as the kernel reads them.  A product of two bf16 values is exact in
float64, so the reference is the exact result up to float64 rounding (~2^-53 relative).  Next to it the same pass computes
S = sum |x| * |w| (the accumulation condition number): an fp32 accumulation of the same products is off by at most a
multiple of 2^-24 * S whatever the order.

Criterion, per output element (never a whole-tensor norm, which lets k wrong elements of N through at sqrt(k / N)):
    |got - ref| <= EPS_OUT * |ref| + EPS_ACC * S_epi + EPS_F32 * T
  EPS_OUT = 2^-8 : the unit roundoff of bf16 (8-bit significand): one round-to-nearest errs by at most u / (1 + u)
                   relative, so one rounding uses up to 99.6 % of this term; the fp32 error of the value being rounded
                   is paid for by the EPS_ACC term (S >= |acc|).
  EPS_ACC = 2^-16: fp32 accumulation error relative to S.  The worst case for K = 4608 terms is K * 2^-24 = 2^-11.8, but
                   a tensor-core sum of K products errs like sqrt(K) * 2^-24 (0.3 % of the worst case at K = 576), so
                   2^-16 keeps a factor > 30 over what an order-independent fp32 sum does.
  S_epi           : S passed through the epilogue: times |scale| (AFFINE), |sp1| (STYLE y); res and bias add exactly;
                   ReLU / leaky ReLU are 1-Lipschitz.
  EPS_F32 = 2^-20, T = sum of |terms| of the fp32 epilogue expression (acc*scale, shift, res, nw*noise, ...): each fp32
                   operation there rounds at 2^-24 relative to its operands, which matters only where they cancel.
Statistics partials (STATS, BNBWD, BNBWD_RES) are compared row by row with their own 128-pixel tile: a 128-term fp32
sum in any order is within 128 * 2^-24 * sum |terms| of the exact sum (terms are products of bf16 values, exact in fp32).

A failure names the instance (irfd_conv_gemm_plan / irfd_conv_wgrad_plan), the tile, the CTA that served it and the
worst element.  CASES / WGRAD_CASES are the coverage tables; tests/test_gemm_plan_cpu.py checks, without a GPU, that
they reach every kernel instance with >= 3 tiles per CTA.
"""
from __future__ import annotations

import math
import os
import zlib
from contextlib import contextmanager
from dataclasses import dataclass
from typing import Tuple

import pytest
import torch

pytestmark = pytest.mark.gpu

PLAIN, STATS, STYLE, AFFINE, BNBWD, BNBWD_RES = 0, 1, 2, 3, 4, 5
MODE_NAMES = ("PLAIN", "STATS", "STYLE", "AFFINE", "BNBWD", "BNBWD_RES")

EPS_OUT = 2.0 ** -8
EPS_ACC = 2.0 ** -16
EPS_F32 = 2.0 ** -20
EPS_SUM = 128 * 2.0 ** -24  # one 128-row tile partial, fp32, any order
U32 = 2.0 ** -24
EPS_WG = 2.0 ** -17  # weight gradients: see test_wgrad_fp64


# ----------------------------------------------------------------------------------------------------------------------
# coverage tables
# ----------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class ConvCase:
    name: str
    mode: int
    n: int
    h: int
    w: int
    cin: int
    cout: int
    k: int
    block_n: int = 0
    env: Tuple[Tuple[str, str], ...] = ()
    wgroups: int = 1
    a_shared: bool = False  # x is one group's [rows, cin] matrix read by every group (the stem)
    relu: int = 0           # AFFINE: 0 none, 1 ReLU, 2 leaky ReLU(0.2)
    res: bool = False       # AFFINE residual
    bias: bool = False      # PLAIN bias
    stat_groups: int = 0    # BNBWD modes: statistic groups of z (0: 2 per weight group)
    sampled: bool = False   # production size: compare sampled tiles, all partial rows

    def plan_args(self):
        """(n, h, w, cin, cout, ksize, mode, wgroups, a_shared, force_block_n) as the ops wrapper passes them."""
        n, h, w = self.n, self.h, self.w
        if self.a_shared:  # ops passes the stacked output rows
            n, h, w = 1, 1, self.w * self.wgroups
        return (n, h, w, self.cin, self.cout, self.k, self.mode, self.wgroups, self.a_shared, self.block_n)


@dataclass(frozen=True)
class WgradCase:
    name: str
    n: int  # TOTAL images (all groups); a 2-D row matrix is n = 1, h = 1, w = rows
    h: int
    w: int
    cin: int
    cout: int
    k: int
    groups: int = 1
    x_shared: bool = False
    reduce_cin: int = 0
    reduce_taps: int = 0
    beta: bool = False  # accumulate into a non-zero dw (beta = 1)
    env: Tuple[Tuple[str, str], ...] = ()
    sampled: bool = False  # production size: compare 16 output channels (every input channel and tap of each)

    def plan_args(self):
        n, h, w = self.n, self.h, self.w
        if self.x_shared:
            n, h, w = 1, 1, self.w * self.groups
        return (n, h, w, self.cin, self.cout, self.k, self.groups, self.x_shared, self.reduce_cin, self.reduce_taps)


# Every GEMM launch shape of one B = 32 train step (3 encoders x 64 images at 256^2, 64 generator codes) and one d_step,
# as test_production_launches_are_listed records them.  Conv: (n, h, w, cin, cout, ksize, mode, wgroups, a_shared,
# force_block_n); wgrad: (n, h, w, cin, cout, ksize, groups, x_shared, reduce_cin, reduce_taps).
PROD_CONV_LAUNCHES = [
    (1,1,512,512,4608,1,0,1,0,0), (1,1,512,4608,512,1,0,1,0,0), (1,1,512,4608,512,1,3,1,0,0),
    (1,1,2048,512,4608,1,0,1,0,0), (1,1,2048,4608,512,1,0,1,0,0), (1,1,2048,4608,512,1,3,1,0,0),
    (1,1,8192,512,4608,1,0,1,0,0), (1,1,8192,4608,512,1,0,1,0,0), (1,1,8192,4608,512,1,3,1,0,0),
    (1,1,12288,512,4608,1,0,3,0,0), (1,1,12288,4608,512,1,1,3,0,0), (1,1,32768,512,2304,1,0,1,0,0),
    (1,1,32768,2304,512,1,0,1,0,0), (1,1,32768,2304,512,1,3,1,0,0), (1,1,49152,256,2304,1,0,3,0,0),
    (1,1,49152,2304,256,1,1,3,0,0), (1,1,131072,256,1152,1,0,1,0,0), (1,1,131072,1152,256,1,0,1,0,0),
    (1,1,131072,1152,256,1,3,1,0,0), (1,1,196608,128,1152,1,0,3,0,0), (1,1,196608,1152,128,1,1,3,0,0),
    (1,1,524288,128,576,1,0,1,0,0), (1,1,524288,576,128,1,0,1,0,0), (1,1,524288,576,128,1,3,1,0,0),
    (1,1,3145728,192,64,1,1,3,1,0), (32,4,4,512,512,3,0,1,0,0), (32,4,4,512,512,3,3,1,0,0),
    (32,8,8,512,512,3,0,1,0,0), (32,8,8,512,512,3,2,1,0,0), (32,8,8,512,512,3,3,1,0,0),
    (32,16,16,512,512,3,0,1,0,0), (32,16,16,512,512,3,2,1,0,0), (32,16,16,512,512,3,3,1,0,0),
    (32,32,32,512,512,3,0,1,0,0), (32,32,32,512,512,3,2,1,0,0), (32,32,32,512,512,3,3,1,0,0),
    (32,64,64,256,256,3,0,1,0,0), (32,64,64,256,256,3,2,1,0,0), (32,64,64,256,256,3,3,1,0,0),
    (32,64,64,512,256,3,2,1,0,0), (32,128,128,128,128,3,0,1,0,0), (32,128,128,128,128,3,2,1,0,0),
    (32,128,128,128,128,3,3,1,0,0), (32,128,128,256,128,3,2,1,0,0), (32,256,256,64,64,3,0,1,0,0),
    (32,256,256,64,64,3,2,1,0,0), (32,256,256,64,64,3,3,1,0,0), (32,256,256,128,64,3,2,1,0,0),
    (64,8,8,512,512,3,0,1,0,0), (64,8,8,512,512,3,2,1,0,0), (64,16,16,512,512,3,0,1,0,0),
    (64,16,16,512,512,3,2,1,0,0), (64,32,32,512,512,3,0,1,0,0), (64,32,32,512,512,3,2,1,0,0),
    (64,64,64,256,256,3,0,1,0,0), (64,64,64,256,256,3,2,1,0,0), (64,64,64,256,512,3,0,1,0,0),
    (64,64,64,512,256,3,2,1,0,0), (64,128,128,128,128,3,0,1,0,0), (64,128,128,128,128,3,2,1,0,0),
    (64,128,128,128,256,3,0,1,0,0), (64,128,128,256,128,3,2,1,0,0), (64,256,256,64,64,3,0,1,0,0),
    (64,256,256,64,64,3,2,1,0,0), (64,256,256,64,128,3,0,1,0,0), (64,256,256,128,64,3,2,1,0,0),
    (192,8,8,512,512,3,1,3,0,0), (192,8,8,512,512,3,4,3,0,0), (192,8,8,512,2048,1,0,3,0,0),
    (192,8,8,512,2048,1,1,3,0,0), (192,8,8,1024,2048,1,1,3,0,0), (192,8,8,2048,512,1,1,3,0,0),
    (192,8,8,2048,512,1,4,3,0,0), (192,8,8,2048,1024,1,0,3,0,0), (192,16,16,256,256,3,1,3,0,0),
    (192,16,16,256,256,3,4,3,0,0), (192,16,16,256,1024,1,0,3,0,0), (192,16,16,256,1024,1,1,3,0,0),
    (192,16,16,512,1024,1,0,3,0,0), (192,16,16,512,1024,1,1,3,0,0), (192,16,16,1024,256,1,1,3,0,0),
    (192,16,16,1024,256,1,4,3,0,0), (192,16,16,1024,512,1,0,3,0,0), (192,16,16,1024,512,1,1,3,0,0),
    (192,32,32,128,128,3,1,3,0,0), (192,32,32,128,128,3,4,3,0,0), (192,32,32,128,512,1,0,3,0,0),
    (192,32,32,128,512,1,1,3,0,0), (192,32,32,256,512,1,0,3,0,0), (192,32,32,256,512,1,1,3,0,0),
    (192,32,32,512,128,1,1,3,0,0), (192,32,32,512,128,1,4,3,0,0), (192,32,32,512,256,1,0,3,0,0),
    (192,32,32,512,256,1,1,3,0,0), (192,64,64,64,64,1,0,3,0,0), (192,64,64,64,64,1,1,3,0,0),
    (192,64,64,64,64,3,1,3,0,0), (192,64,64,64,64,3,4,3,0,0), (192,64,64,64,256,1,0,3,0,0),
    (192,64,64,64,256,1,1,3,0,0), (192,64,64,128,256,1,0,3,0,0), (192,64,64,256,64,1,0,3,0,0),
    (192,64,64,256,64,1,1,3,0,0), (192,64,64,256,64,1,4,3,0,0), (192,64,64,256,128,1,1,3,0,0),
]
PROD_WGRAD_LAUNCHES = [
    (1,1,512,4608,512,1,1,0,512,9), (1,1,2048,4608,512,1,1,0,512,9), (1,1,8192,4608,512,1,1,0,512,9),
    (1,1,12288,4608,512,1,3,0,512,9), (1,1,32768,2304,512,1,1,0,256,9), (1,1,49152,2304,256,1,3,0,256,9),
    (1,1,131072,1152,256,1,1,0,128,9), (1,1,196608,1152,128,1,3,0,128,9), (1,1,524288,576,128,1,1,0,64,9),
    (1,1,3145728,192,64,1,3,1,147,1), (32,4,4,512,512,3,1,0,0,0), (32,8,8,512,512,3,1,0,0,0),
    (32,16,16,512,512,3,1,0,0,0), (32,32,32,512,512,3,1,0,0,0), (32,64,64,256,256,3,1,0,0,0),
    (32,128,128,128,128,3,1,0,0,0), (32,256,256,64,64,3,1,0,0,0), (64,8,8,512,512,3,1,0,0,0),
    (64,16,16,512,512,3,1,0,0,0), (64,32,32,512,512,3,1,0,0,0), (64,64,64,256,256,3,1,0,0,0),
    (64,64,64,512,256,3,1,0,0,0), (64,128,128,128,128,3,1,0,0,0), (64,128,128,256,128,3,1,0,0,0),
    (64,256,256,64,64,3,1,0,0,0), (64,256,256,128,64,3,1,0,0,0), (192,8,8,512,512,3,3,0,0,0),
    (192,8,8,512,2048,1,3,0,0,0), (192,8,8,1024,2048,1,3,0,0,0), (192,8,8,2048,512,1,3,0,0,0),
    (192,16,16,256,256,3,3,0,0,0), (192,16,16,256,1024,1,3,0,0,0), (192,16,16,512,1024,1,3,0,0,0),
    (192,16,16,1024,256,1,3,0,0,0), (192,16,16,1024,512,1,3,0,0,0), (192,32,32,128,128,3,3,0,0,0),
    (192,32,32,128,512,1,3,0,0,0), (192,32,32,256,512,1,3,0,0,0), (192,32,32,512,128,1,3,0,0,0),
    (192,32,32,512,256,1,3,0,0,0), (192,64,64,64,64,1,3,0,0,0), (192,64,64,64,64,3,3,0,0,0),
    (192,64,64,64,256,1,3,0,0,0), (192,64,64,256,64,1,3,0,0,0), (192,64,64,256,128,1,3,0,0,0),
]


CLUSTER = (("IRFD_GEMM_CLUSTER", "1"),)
MMA2 = (("IRFD_GEMM_2SM", "1"),)
LOCKSTEP = (("IRFD_WARP_EPI", "0"),)
NO_HALO = (("IRFD_CONV_HALO", "0"),)


def _per_tap_cases():
    """conv_gemm_kernel (linear geometry): every mode x BLOCK_N x CTA pairing x epilogue.  Tile counts x n tiles land
    in (3, 4) x 148 whatever the pairing (a pair serves 2 m tiles per unit on 74 slots): every CTA serves 3 or 4 units
    and the last round is ragged.  Shapes alternate between 3x3 at 32^2 (8 tiles per image) and 1x1, one and three
    weight groups, so that every instance runs a multi-tap K loop or a grouped weight matrix somewhere."""
    cases = []
    i = 0
    for mode in (PLAIN, STATS, STYLE, AFFINE, BNBWD, BNBWD_RES):
        for bn in (64, 128, 256):
            pairings = [()]
            if bn >= 128:
                pairings.append(CLUSTER)
                if mode in (PLAIN, STATS, BNBWD):
                    pairings.append(MMA2)
            for pair in pairings:
                epis = [()] if mode == STYLE or pair == MMA2 else [(), LOCKSTEP]
                for epi in epis:
                    i += 1
                    wide = i % 2 == 0 and mode != BNBWD_RES          # cout = 2 * BLOCK_N: two n tiles
                    cout = bn * (2 if wide else 1)
                    three = i % 3 != 0 and mode != STYLE               # 3x3 at 32^2, else 1x1 rows
                    groups = 3 if (i % 4 in (1, 2) and mode != STYLE) else 1
                    if three:
                        n, h, w, k = (30 if wide else 63), 32, 32, 3
                    else:
                        n, h, w, k = (120 if wide else 252), 16, 16, 1
                    cin = 128 if i % 5 == 0 else 64
                    relu, res = (i % 3, i % 2 == 1) if mode == AFFINE else (0, False)
                    tag = f"{MODE_NAMES[mode]}-bn{bn}" + ("-cl" if pair == CLUSTER else "-2sm" if pair == MMA2 else "")
                    tag += "-lockstep" if epi else ""
                    cases.append(ConvCase(tag, mode, n, h, w, cin, cout, k, block_n=bn, env=pair + epi,
                                          wgroups=groups, relu=relu, res=res,
                                          bias=mode == PLAIN and i % 2 == 1 and groups == 1))
    return cases


def _prod_conv(name, launch, relu=0):
    """A sampled case at a recorded launch shape (plan arguments as in PROD_CONV_LAUNCHES)."""
    n, h, w, cin, cout, k, mode, wgroups, a_shared, block_n = launch
    if a_shared:
        w //= wgroups
    return ConvCase(name, mode, n, h, w, cin, cout, k, block_n=block_n, wgroups=wgroups, a_shared=bool(a_shared),
                    relu=relu, stat_groups=2 * wgroups if mode in (BNBWD, BNBWD_RES) else 0, sampled=True)


CASES = _per_tap_cases() + [
    # an even number of rounds: 592 tiles = exactly 4 per CTA
    ConvCase("PLAIN-bn64-even-rounds", PLAIN, 1, 1, 592 * 128, 64, 64, 1, block_n=64),
    ConvCase("STATS-bn64-even-rounds-lockstep", STATS, 74, 32, 32, 64, 64, 3, block_n=64, env=LOCKSTEP),
    # ragged M (pointwise, m_total % 128 != 0: lockstep epilogue, the last tile half out of bounds)
    ConvCase("PLAIN-bn64-ragged-m", PLAIN, 1, 1, 500 * 128 - 37, 64, 64, 1, block_n=64, bias=True),
    ConvCase("STATS-bn256-ragged-m", STATS, 1, 1, 500 * 128 - 100, 64, 256, 1, block_n=256),
    ConvCase("AFFINE-bn128-ragged-m", AFFINE, 1, 1, 250 * 128 - 5, 64, 256, 1, block_n=128, relu=1, res=True),
    # the stem: one group's im2col rows read by the three weight groups
    ConvCase("STATS-bn64-a-shared", STATS, 1, 1, 168 * 128, 192, 64, 1, block_n=64, wgroups=3, a_shared=True),
    ConvCase("AFFINE-bn64-a-shared", AFFINE, 1, 1, 168 * 128, 192, 64, 1, block_n=64, wgroups=3, a_shared=True,
             relu=1),
    ConvCase("PLAIN-bn128-a-shared-cl", PLAIN, 1, 1, 168 * 128, 192, 128, 1, block_n=128, wgroups=3,
             a_shared=True, env=CLUSTER),
    # conv_halo_kernel: 3x3, W % 128 == 0, Cout = BLOCK_N 64 / 128; 448 / 450 tiles of 256 pixels
    ConvCase("halo-PLAIN-bn64-w256", PLAIN, 7, 64, 256, 64, 64, 3),
    ConvCase("halo-PLAIN-bn128-w128", PLAIN, 9, 100, 128, 64, 128, 3, bias=True),
    ConvCase("halo-STATS-bn64-w128", STATS, 9, 100, 128, 128, 64, 3),
    ConvCase("halo-STATS-bn128-w256", STATS, 7, 64, 256, 64, 128, 3),
    ConvCase("halo-STYLE-bn64-w256", STYLE, 7, 64, 256, 64, 64, 3),
    ConvCase("halo-STYLE-bn128-w128", STYLE, 9, 100, 128, 64, 128, 3),
    ConvCase("halo-AFFINE-bn64-relu0", AFFINE, 7, 64, 256, 64, 64, 3, relu=0, res=False),
    ConvCase("halo-AFFINE-bn64-relu0-res", AFFINE, 9, 100, 128, 64, 64, 3, relu=0, res=True),
    ConvCase("halo-AFFINE-bn64-relu1-res", AFFINE, 7, 64, 256, 64, 64, 3, relu=1, res=True),
    ConvCase("halo-AFFINE-bn64-lrelu", AFFINE, 7, 64, 256, 64, 64, 3, relu=2),
    ConvCase("halo-AFFINE-bn128-lrelu-res", AFFINE, 7, 64, 256, 64, 128, 3, relu=2, res=True),
    ConvCase("halo-AFFINE-bn128-relu1", AFFINE, 9, 100, 128, 64, 128, 3, relu=1),
    # boxed conv_gemm_kernel: 56^2 (2-row boxes), 28^2 (4-row boxes), 250^2 (128-column segments, ragged)
    ConvCase("boxed-PLAIN-bn64-56", PLAIN, 18, 56, 56, 64, 64, 3, block_n=64),
    ConvCase("boxed-AFFINE-bn64-250", AFFINE, 1, 250, 250, 64, 64, 3, block_n=64, relu=2, res=True),
    ConvCase("boxed-PLAIN-bn128-250", PLAIN, 1, 250, 250, 64, 128, 3, block_n=128),
    ConvCase("boxed-AFFINE-bn128-28", AFFINE, 72, 28, 28, 64, 128, 3, block_n=128, relu=1, res=True, wgroups=3),
    ConvCase("boxed-PLAIN-bn256-28", PLAIN, 72, 28, 28, 64, 256, 3, block_n=256),
    ConvCase("boxed-AFFINE-bn256-56", AFFINE, 18, 56, 56, 128, 256, 3, block_n=256, relu=0, res=True),
    # one production launch shape (PROD_CONV_LAUNCHES) per instance the B = 32 train step and d_step launch, the
    # cheapest of each, plus the encoder's 3x3 @64 layers: sampled tiles, every partial row
    *[_prod_conv(name, launch, **kw) for name, launch, kw in (
        ("prod-gen-dgrad-64@256", (32, 256, 256, 64, 64, 3, 0, 1, 0, 0), {}),
        ("prod-gen-dgrad-128@128", (32, 128, 128, 128, 128, 3, 0, 1, 0, 0), {}),
        ("prod-gen-fprop-64@256", (32, 256, 256, 64, 64, 3, 2, 1, 0, 0), {}),
        ("prod-gen-fprop-128@128", (32, 128, 128, 128, 128, 3, 2, 1, 0, 0), {}),
        ("prod-disc-conv1-64@256", (32, 256, 256, 64, 64, 3, 3, 1, 0, 0), {"relu": 2}),
        ("prod-disc-conv1-128@128", (32, 128, 128, 128, 128, 3, 3, 1, 0, 0), {"relu": 2}),
        ("prod-rows-4608-512", (1, 1, 512, 4608, 512, 1, 0, 1, 0, 0), {}),
        ("prod-rows-512-4608", (1, 1, 512, 512, 4608, 1, 0, 1, 0, 0), {}),
        ("prod-rows-512-4608-2048", (1, 1, 2048, 512, 4608, 1, 0, 1, 0, 0), {}),
        ("prod-enc-fprop-64-64-1x1@64", (192, 64, 64, 64, 64, 1, 1, 3, 0, 0), {}),
        ("prod-enc-fprop-64-64-3x3@64", (192, 64, 64, 64, 64, 3, 1, 3, 0, 0), {}),
        ("prod-enc-fprop-512-128-1x1@32", (192, 32, 32, 512, 128, 1, 1, 3, 0, 0), {}),
        ("prod-enc-fprop-512-2048-1x1@8", (192, 8, 8, 512, 2048, 1, 1, 3, 0, 0), {}),
        ("prod-gen-fprop-512@8", (32, 8, 8, 512, 512, 3, 2, 1, 0, 0), {}),
        ("prod-gen-fprop-512@8x64", (64, 8, 8, 512, 512, 3, 2, 1, 0, 0), {}),
        ("prod-gen-fprop-512@16", (64, 16, 16, 512, 512, 3, 2, 1, 0, 0), {}),
        ("prod-disc-im2col-512", (1, 1, 512, 4608, 512, 1, 3, 1, 0, 0), {"relu": 2}),
        ("prod-disc-im2col-8192", (1, 1, 8192, 4608, 512, 1, 3, 1, 0, 0), {"relu": 2}),
        ("prod-disc-im2col-32768", (1, 1, 32768, 2304, 512, 1, 3, 1, 0, 0), {"relu": 2}),
        ("prod-enc-dgrad-64-256-1x1@64", (192, 64, 64, 256, 64, 1, 4, 3, 0, 0), {}),
        ("prod-enc-dgrad-64-64-3x3@64", (192, 64, 64, 64, 64, 3, 4, 3, 0, 0), {}),
        ("prod-enc-dgrad-128-512-1x1@32", (192, 32, 32, 512, 128, 1, 4, 3, 0, 0), {}),
        ("prod-enc-dgrad-512-2048-1x1@8", (192, 8, 8, 2048, 512, 1, 4, 3, 0, 0), {}),
    )],
]

def _prod_wgrad(name, launch):
    n, h, w, cin, cout, k, groups, x_shared, reduce_cin, reduce_taps = launch
    if x_shared:
        w //= groups
    return WgradCase(name, n, h, w, cin, cout, k, groups=groups, x_shared=bool(x_shared), reduce_cin=reduce_cin,
                     reduce_taps=reduce_taps, sampled=True)


WGRAD_CASES = [
    # per-tap wgrad_gemm_kernel, BLOCK_N = the widest of 256 / 128 / 64 dividing Cout
    WgradCase("tap-bn64-reduce1", 4, 16, 16, 64, 64, 3),
    WgradCase("tap-bn64-reduce8-ragged", 1, 1, 30000, 64, 64, 1),
    WgradCase("tap-bn64-reduce8-ragged-beta", 1, 1, 300000, 64, 64, 1, beta=True),
    WgradCase("tap-bn128-reduce4", 12, 32, 32, 64, 128, 3),
    WgradCase("tap-bn256-reduce4-groups3", 12, 32, 32, 64, 256, 3, groups=3),
    WgradCase("tap-bn256-transpose9", 8, 16, 16, 512, 512, 3),
    WgradCase("tap-bn256-transpose9-beta", 8, 16, 16, 512, 512, 3, beta=True),
    WgradCase("tap-bn256-transpose1", 8, 16, 16, 512, 512, 1),
    WgradCase("tap-bn256-reduce4-rows", 1, 1, 8192, 512, 512, 1),
    WgradCase("tap-halo-off", 4, 32, 128, 64, 64, 3, env=(("IRFD_WGRAD_HALO", "0"),)),
    # im2col operands: 3x3 stride 2 (k = tap * C + c, reduce_cin = C, reduce_taps = 9), the stem (K_total 192 holds
    # 147 real rows: not tileable, so it takes the non-transposing reduce)
    WgradCase("tap-im2col-3x3s2-groups3", 1, 1, 3 * 2048, 9 * 256, 256, 1, groups=3, reduce_cin=256, reduce_taps=9),
    WgradCase("tap-stem-x-shared", 1, 1, 16384, 192, 64, 1, groups=3, x_shared=True, reduce_cin=147, reduce_taps=1),
    # wgrad_halo_kernel (default selection: Cout <= 128, W >= 64; IRFD_WGRAD_HALO=2: every eligible shape)
    WgradCase("halo-w128", 4, 32, 128, 64, 64, 3),
    WgradCase("halo-w64-groups3-ragged", 9, 50, 64, 64, 128, 3, groups=3),
    WgradCase("halo-w256-beta", 2, 8, 256, 128, 64, 3, beta=True),
    WgradCase("halo-forced-transpose9", 4, 16, 32, 512, 256, 3, env=(("IRFD_WGRAD_HALO", "2"),)),
    WgradCase("halo-forced-reduce4", 4, 16, 32, 64, 256, 3, env=(("IRFD_WGRAD_HALO", "2"),)),
    # one production launch shape (PROD_WGRAD_LAUNCHES) per (GEMM, reduce) pair the train step and d_step launch
    *[_prod_wgrad(name, launch) for name, launch in (
        ("prod-halo-reduce4", (64, 128, 128, 256, 128, 3, 1, 0, 0, 0)),
        ("prod-halo-reduce8-enc-3x3@64", (192, 64, 64, 64, 64, 3, 3, 0, 0, 0)),
        ("prod-tap64-reduce4", (192, 64, 64, 256, 64, 1, 3, 0, 0, 0)),
        ("prod-tap64-reduce8", (192, 64, 64, 64, 64, 1, 3, 0, 0, 0)),
        ("prod-tap64-stem", (1, 1, 3145728, 192, 64, 1, 3, 1, 147, 1)),
        ("prod-tap128-reduce1-im2col", (1, 1, 196608, 1152, 128, 1, 3, 0, 128, 9)),
        ("prod-tap128-reduce4", (192, 32, 32, 512, 128, 1, 3, 0, 0, 0)),
        ("prod-tap128-reduce8-im2col", (1, 1, 524288, 576, 128, 1, 1, 0, 64, 9)),
        ("prod-tap256-reduce4", (192, 32, 32, 128, 512, 1, 3, 0, 0, 0)),
        ("prod-tap256-reduce8", (192, 64, 64, 64, 256, 1, 3, 0, 0, 0)),
        ("prod-tap256-transpose1", (192, 8, 8, 512, 2048, 1, 3, 0, 0, 0)),
        ("prod-tap256-transpose9-im2col", (1, 1, 512, 4608, 512, 1, 1, 0, 512, 9)),
    )],
]


# ----------------------------------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------------------------------
@contextmanager
def _env(pairs):
    old = {k: os.environ.get(k) for k, _ in pairs}
    os.environ.update(dict(pairs))
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def _seed(case):
    """A seed of the case's own: outputs come from the caching allocator, so a tile a kernel failed to store could
    otherwise still hold the equal result of an earlier case with the same shape."""
    return zlib.crc32(case.name.encode())


def _bf16(shape, g, dev, scale=1.0):
    return (torch.randn(shape, generator=g) * scale).to(dev).to(torch.bfloat16)


def _instance(plan):
    if plan["halo"]:
        return f"conv_halo_kernel<{plan['block_n']}>"
    return (f"conv_gemm_kernel<{plan['block_n']}, CL={2 if plan['cluster'] > 1 else 1}, MMA2={int(plan['cluster'] == 3)}"
            f", BOX={plan['boxed']}> warp_epi={plan['warp_epi']}")


class TileMap:
    """Pixel <-> tile <-> CTA of one conv launch, from the plan query and the geometry query."""

    def __init__(self, c: ConvCase, plan, dev):
        from speak_hack_b200 import ops

        self.plan = plan
        self.pair = 2 if plan["cluster"] > 1 else 1
        self.slots = plan["grid"] // self.pair
        n, h, w = c.plan_args()[:3]
        self.m = n * h * w
        pix = torch.arange(self.m, device=dev)
        if plan["halo"]:  # 256-pixel tiles: two rows x 128 columns, (image, row pair, column segment)
            img, rem = pix // (h * w), pix % (h * w)
            self.tile = (img * (h // 2) + (rem // w) // 2) * (w // 128) + (rem % w) // 128
            self.tiles = self.m // 256
        elif plan["boxed"]:
            geo = ops.conv_geometry(n, h, w, c.k, c.wgroups)
            _, tw, th, tn, tiles_w, tiles_h, _ = geo
            img, rem = pix // (h * w), pix % (h * w)
            self.tile = ((img // tn) * tiles_h + (rem // w) // th) * tiles_w + (rem % w) // tw
            self.tiles = plan["m_tiles"]
        else:
            self.tile = pix // 128
            self.tiles = plan["m_tiles"]

    def unit(self, tile, n_tile):
        return (tile // self.pair) * self.plan["n_tiles"] + n_tile

    def cta(self, tile, n_tile):
        u = self.unit(tile, n_tile)
        return (u % self.slots) * self.pair + tile % self.pair, u // self.slots

    def sampled_tiles(self, seed=0):
        """Tiles of CTAs 0, 1 and grid-1 in every round, the first and last two tiles, the tiles holding the first and
        last rows / columns of a few images (taken from the pixel map), 16 random ones: all n tiles of each."""
        nt = self.plan["n_tiles"]
        units = torch.arange(self.plan["units"])
        slot = units % self.slots
        pick = units[(slot == 0) | (slot == min(1, self.slots - 1)) | (slot == self.slots - 1)]
        tiles = set()
        for u in pick.tolist():
            t0 = (u // nt) * self.pair
            tiles.update(range(t0, t0 + self.pair))
        tiles.update([0, 1, self.tiles - 2, self.tiles - 1])
        g = _gen(seed)
        tiles.update(torch.randint(0, self.tiles, (16,), generator=g).tolist())
        return sorted(t for t in tiles if 0 <= t < self.tiles)


def _edge_pixels(n, h, w, dev, images=(0, 1)):
    out = []
    for i in images:
        if i >= n:
            continue
        base = i * h * w
        rows = torch.tensor([0, h - 1], device=dev)
        cols = torch.arange(w, device=dev)
        out.append(base + (rows[:, None] * w + cols[None, :]).reshape(-1))
        r = torch.arange(h, device=dev)
        out.append(base + (r[:, None] * w + torch.tensor([0, w - 1], device=dev)[None, :]).reshape(-1))
    return torch.cat(out) if out else torch.empty(0, dtype=torch.long, device=dev)


def conv_ref(x, wk, k, wgroups, a_shared, pix, shape, chunk=1 << 26):
    """float64 (acc, S) at output pixels `pix` ([P] flat NHWC indices) of the stride-1 same-padding conv of the bf16
    operands; weight group of a pixel = pix // (pixels per group); a_shared: x holds one group's rows."""
    n, h, w = shape
    cin = x.shape[-1]
    cout = wk.shape[0] // wgroups
    m = n * h * w
    m_g = m // wgroups
    xf = x.reshape(-1, cin)
    acc = torch.empty(pix.numel(), cout, dtype=torch.float64, device=x.device)
    s = torch.empty_like(acc)
    step = max(1, chunk // (k * k * cin))
    taps = [(dh, dw) for dh in range(-(k // 2), k // 2 + 1) for dw in range(-(k // 2), k // 2 + 1)]
    for g in range(wgroups):
        wg = wk[g * cout:(g + 1) * cout].double()
        sel = ((pix // m_g) == g).nonzero().squeeze(1)
        for c0 in range(0, sel.numel(), step):
            idx = sel[c0:c0 + step]
            p = pix[idx]
            if a_shared:
                patch = xf[p % m_g].double()
            elif k == 1:
                patch = xf[p].double()
            else:
                img, rem = p // (h * w), p % (h * w)
                hh, ww = rem // w, rem % w
                cols = []
                for dh, dw in taps:
                    y2, x2 = hh + dh, ww + dw
                    ok = (y2 >= 0) & (y2 < h) & (x2 >= 0) & (x2 < w)
                    q = (img * h + y2.clamp(0, h - 1)) * w + x2.clamp(0, w - 1)
                    cols.append(xf[q].double() * ok[:, None])
                patch = torch.cat(cols, 1)
            acc[idx] = patch @ wg.t()
            s[idx] = patch.abs() @ wg.abs().t()
    return acc, s


def _check(name, got, ref, bound, where):
    """Element-wise: raise with the worst element (relative to its bound) located by `where(flat_index)`."""
    err = (got.double() - ref).abs()
    ratio = err / bound.clamp_min(1e-300)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    if not worst <= 1.0:  # also catches NaN
        i = int(torch.nan_to_num(ratio, nan=math.inf).argmax())
        bad = int((ratio > 1).sum()) + int(ratio.isnan().sum())
        pytest.fail(f"{name}: {bad} elements out of bound; worst at {where(i)}: got {float(got.reshape(-1)[i]):.6g} "
                    f"ref {float(ref.reshape(-1)[i]):.6g} bound {float(bound.reshape(-1)[i]):.3g} "
                    f"(|err|/bound {worst:.3g})")
    return worst


def _note(family, ratio):
    print(f"[fp64] |err|/bound {ratio:.3e}  {family}")  # the margin each check leaves (run with -s)


# ----------------------------------------------------------------------------------------------------------------------
# conv GEMMs
# ----------------------------------------------------------------------------------------------------------------------
def _operands(c: ConvCase, dev, seed):
    g = _gen(seed)
    ktot = c.k * c.k * c.cin
    if c.a_shared:
        x = _bf16((c.w, c.cin), g, dev)
    else:
        x = _bf16((c.n, c.h, c.w, c.cin), g, dev)
    wk = _bf16((c.wgroups * c.cout, ktot), g, dev, scale=1.0 / math.sqrt(ktot))
    return g, x, wk


def _run_conv(c: ConvCase, dev):
    """Launch the case; returns (outputs dict, extra operands dict)."""
    from speak_hack_b200 import ops

    g, x, wk = _operands(c, dev, _seed(c))
    n, h, w = c.plan_args()[:3]
    m = n * h * w
    extra = {}
    out = {}
    if c.mode == PLAIN and (c.wgroups > 1):
        assert not c.bias, "the grouped entry point takes no bias"
        out["y"] = ops.conv_gemm_grouped(x, wk, c.k, ops.EPI_PLAIN, wgroups=c.wgroups, a_shared=c.a_shared,
                                         force_block_n=c.block_n).reshape(m, c.cout)
    elif c.mode == PLAIN:
        if c.bias:
            extra["bias"] = torch.randn(c.cout, generator=g).to(dev)
        out["y"] = ops.conv_gemm(x, wk, c.k, ops.EPI_PLAIN, bias=extra.get("bias"),
                                 force_block_n=c.block_n).reshape(m, c.cout)
    elif c.mode == STATS:
        y, ssum, ssq = ops.conv_gemm_grouped(x, wk, c.k, ops.EPI_STATS, wgroups=c.wgroups, a_shared=c.a_shared,
                                             force_block_n=c.block_n)
        out.update(y=y.reshape(m, c.cout), ssum=ssum, ssq=ssq)
    elif c.mode == STYLE:
        extra["bias"] = torch.randn(c.cout, generator=g).to(dev)
        extra["nw"] = torch.randn(c.cout, generator=g).to(dev)
        extra["noise"] = torch.randn(m, generator=g).to(dev)
        extra["sp1"] = (torch.randn(c.n, c.cout, generator=g) + 1).to(dev)
        extra["s1"] = torch.randn(c.n, c.cout, generator=g).to(dev)
        a, y = ops.conv_gemm(x, wk, c.k, ops.EPI_STYLE, bias=extra["bias"], nw=extra["nw"], noise=extra["noise"],
                             sp1=extra["sp1"], s1=extra["s1"], force_block_n=c.block_n)
        out.update(a=a.reshape(m, c.cout), y=y.reshape(m, c.cout))
    elif c.mode == AFFINE:
        extra["scale"] = (torch.rand(c.wgroups, c.cout, generator=g) + 0.5).to(dev)
        extra["shift"] = torch.randn(c.wgroups, c.cout, generator=g).to(dev)
        res = _bf16((m, c.cout), g, dev) if c.res else None
        extra["res"] = res
        out["y"] = ops.conv_gemm_affine_grouped(x, wk, c.k, extra["scale"], extra["shift"], res=res, relu=c.relu,
                                                wgroups=c.wgroups, a_shared=c.a_shared,
                                                force_block_n=c.block_n).reshape(m, c.cout)
    else:
        sg = c.stat_groups or 2 * c.wgroups
        z = _bf16((c.n, c.h, c.w, c.cout), g, dev)
        extra["mean"] = (torch.randn(sg, c.cout, generator=g) * 0.3).to(dev)
        extra["rstd"] = (torch.rand(sg, c.cout, generator=g) + 0.5).to(dev)
        extra["z"] = z.reshape(m, c.cout)
        extra["sg"] = sg
        if c.mode == BNBWD:
            extra["gamma"] = [torch.randn(c.cout, generator=g).to(dev) for _ in range(c.wgroups)]
            extra["beta"] = [torch.randn(c.cout, generator=g).to(dev) for _ in range(c.wgroups)]
            y, part = ops.conv_gemm_bnbwd_grouped(x, wk, c.k, z, extra["mean"], extra["rstd"], extra["gamma"],
                                                  extra["beta"], sg, force_block_n=c.block_n)
        else:
            g2 = _bf16((c.n, c.h, c.w, c.cout), g, dev)
            bits = torch.randint(0, 256, (m * c.cout // 8,), generator=g, dtype=torch.uint8).to(dev)
            extra["g2"] = g2.reshape(m, c.cout)
            extra["bits"] = bits
            y, part = ops.conv_gemm_bnbwd_res_grouped(x, wk, c.k, z, extra["mean"], extra["rstd"], g2, bits, sg,
                                                      wgroups=c.wgroups, force_block_n=c.block_n)
            # the epilogue adds g2 to the bf16-ROUNDED dgrad (the staged tile): the same launch in PLAIN mode gives
            # that operand bit for bit (same MMA sequence; bit identity of the instances is test_gpu_conv_gemm's)
            with _env(NO_HALO):
                extra["dgrad_bf16"] = ops.conv_gemm_grouped(x, wk, c.k, ops.EPI_PLAIN, wgroups=c.wgroups,
                                                            force_block_n=c.block_n).reshape(m, c.cout)
        out.update(y=y.reshape(m, c.cout), part=part)
    return x, wk, out, extra


def _xhat(extra, rows, m, c):
    sg = extra["sg"]
    grp = rows // (m // sg)
    return (extra["z"][rows].double() - extra["mean"].double()[grp]) * extra["rstd"].double()[grp]


def _conv_expect(c: ConvCase, x, wk, out, extra, rows, m):
    """float64 expected values and bounds of every output at `rows` ([P] flat pixels): dict name -> (got, ref, bound)."""
    n, h, w = c.plan_args()[:3]
    acc, s = conv_ref(x, wk, c.k, c.wgroups, c.a_shared, rows, (n, h, w))
    cout = c.cout
    grp = rows // (m // c.wgroups)
    res = {}
    if c.mode in (PLAIN, STATS):
        ref = acc + (extra["bias"].double()[None, :] if "bias" in extra else 0.0)
        res["y"] = (out["y"][rows], ref, EPS_OUT * ref.abs() + EPS_ACC * s + EPS_F32 * ref.abs())
    elif c.mode == STYLE:
        img = rows // (h * w)
        nz = extra["nw"].double()[None, :] * extra["noise"].double()[rows, None]
        z = acc + extra["bias"].double()[None, :] + nz
        a = torch.where(z > 0, z, 0.2 * z)
        t = EPS_F32 * (acc.abs() + extra["bias"].double().abs()[None, :] + nz.abs())
        res["a"] = (out["a"][rows], a, EPS_OUT * a.abs() + EPS_ACC * s + t)
        sp1 = extra["sp1"].double()[img]
        s1 = extra["s1"].double()[img]
        y = a * sp1 + s1
        res["y"] = (out["y"][rows], y, EPS_OUT * y.abs() + sp1.abs() * (EPS_ACC * s + t) + EPS_F32 * s1.abs())
    elif c.mode == AFFINE:
        sc = extra["scale"].double()[grp]
        sh = extra["shift"].double()[grp]
        r = extra["res"][rows].double() if extra["res"] is not None else 0.0
        pre = acc * sc + sh + r
        ref = pre if c.relu == 0 else (pre.clamp_min(0) if c.relu == 1 else torch.where(pre > 0, pre, 0.2 * pre))
        t = EPS_F32 * ((acc * sc).abs() + sh.abs() + (r.abs() if torch.is_tensor(r) else 0.0))
        res["y"] = (out["y"][rows], ref, EPS_OUT * ref.abs() + EPS_ACC * sc.abs() * s + t)
    elif c.mode == BNBWD:
        xh = _xhat(extra, rows, m, c)
        gam = torch.stack(extra["gamma"]).double()[grp]
        bet = torch.stack(extra["beta"]).double()[grp]
        pre = gam * xh + bet
        got = out["y"][rows]
        # where gamma*xhat + beta is within fp32 rounding of 0 the kernel's fp32 mask may go either way
        amb = pre.abs() <= 2.0 ** -20 * ((gam * xh).abs() + bet.abs())
        keep = torch.where(amb, got != 0, pre > 0)
        ref = acc * keep
        res["y"] = (got, ref, EPS_OUT * ref.abs() + EPS_ACC * s * keep)
    else:
        byte = extra["bits"].reshape(m, cout // 8)[rows].long()
        bit = ((byte[:, :, None] >> torch.arange(8, device=byte.device)) & 1).reshape(-1, cout).double()
        g2 = extra["g2"][rows].double()
        ref = (acc + g2) * bit
        # two roundings: the dgrad to bf16 (staged), then dgrad + g2 to bf16
        res["y"] = (out["y"][rows], ref, EPS_OUT * (ref.abs() + acc.abs() * bit) + EPS_ACC * s * bit)
        # the staged dgrad itself: exactly what the launch in PLAIN mode stores
        res["dgrad_bf16"] = (extra["dgrad_bf16"][rows], acc, EPS_OUT * acc.abs() + EPS_ACC * s)
    return res


def _check_partials(c: ConvCase, out, extra, m, tmap, name):
    """Every statistics partial row against the fp64 sums over its own 128-pixel tile."""
    cout = c.cout
    tiles = (m + 127) // 128
    pad = tiles * 128 - m
    y = out["y"].double()
    if c.mode == STATS:
        terms = [y, y * y]
        got = [out["ssum"], out["ssq"]]
    else:
        if c.mode == BNBWD:
            f = y  # the masked gradient as stored
        else:  # the fp32 sum of the staged bf16 dgrad and g2, masked (before its own rounding to bf16)
            byte = extra["bits"].reshape(m, cout // 8).long()
            bit = ((byte[:, :, None] >> torch.arange(8, device=byte.device)) & 1).reshape(m, cout).double()
            f = (extra["dgrad_bf16"].double() + extra["g2"].double()).float().double() * bit
        xh = _xhat(extra, torch.arange(m, device=y.device), m, c)
        terms = [f, f * xh]
        got = [out["part"][:, 0], out["part"][:, 1]]
    for which, (t, gp) in enumerate(zip(terms, got)):
        t = torch.cat([t, t.new_zeros(pad, cout)]).reshape(tiles, 128, cout)
        ref = t.sum(1)
        # BNBWD: xhat is fp32 in the kernel (2^-23 relative)
        bound = (EPS_SUM + 4 * U32) * t.abs().sum(1) + 1e-30
        assert gp.shape == (tiles, cout), (gp.shape, tiles)

        def where(i, which=which):
            tile, ch = divmod(i, cout)
            cta, rnd = tmap.cta(tile, ch // tmap.plan["block_n"]) if not tmap.plan["halo"] else (None, None)
            return f"partial {which} tile {tile} channel {ch} (CTA {cta}, round {rnd})"

        _note(f"partials {MODE_NAMES[c.mode]}", _check(f"{name} partial[{which}]", gp.double(), ref, bound, where))


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_conv_gemm_fp64(cuda_device, case):
    from speak_hack_b200 import ops

    c = case
    dev = cuda_device
    with _env(c.env):
        plan = ops.conv_plan(*c.plan_args())
        assert plan is not None, c
        x, wk, out, extra = _run_conv(c, dev)
    torch.cuda.synchronize()
    inst = f"{c.name}: {MODE_NAMES[c.mode]} {_instance(plan)}"
    tmap = TileMap(c, plan, dev)
    n, h, w = c.plan_args()[:3]
    m = n * h * w
    if c.sampled:
        tiles = torch.tensor(tmap.sampled_tiles(), device=dev)
        rows = torch.isin(tmap.tile, tiles).nonzero().squeeze(1)
        if not c.a_shared:
            rows = torch.unique(torch.cat([rows, _edge_pixels(n, h, w, dev, images=(0, n // 2, n - 1))]))
    else:
        rows = torch.arange(m, device=dev)
    chunk = max(1, (1 << 22) // c.cout)
    family = ("halo " if plan["halo"] else "boxed " if plan["boxed"] else "per-tap ") + MODE_NAMES[c.mode]
    for r0 in range(0, rows.numel(), chunk):
        r = rows[r0:r0 + chunk]
        for name, (got, ref, bound) in _conv_expect(c, x, wk, out, extra, r, m).items():
            def where(i, r=r, name=name):
                p, ch = divmod(i, c.cout)
                pix = int(r[p])
                tile = int(tmap.tile[pix])
                cta, rnd = tmap.cta(tile, ch // plan["block_n"])
                return (f"{inst}, output {name} pixel {pix} channel {ch}, tile {tile} n tile {ch // plan['block_n']}"
                        f" (CTA {cta}, round {rnd})")

            _note(family, _check(f"{inst} [{name}]", got, ref, bound, where))
    if c.mode in (STATS, BNBWD, BNBWD_RES):
        _check_partials(c, out, extra, m, tmap, inst)


# ----------------------------------------------------------------------------------------------------------------------
# weight gradients
# ----------------------------------------------------------------------------------------------------------------------
def wgrad_ref(x, dy, c: WgradCase, outs):
    """float64 (dW, S) per group at output channels `outs`, [len(outs)][rc * taps] as the kernel stores OIHW."""
    cout, cin, k = c.cout, c.cin, c.k
    rows = dy.numel() // cout
    m_g = rows // c.groups
    dyf = dy.reshape(rows, cout)[:, outs]
    cout = len(outs)
    xf = x.reshape(-1, cin)
    refs = []
    for g in range(c.groups):
        dg = dyf[g * m_g:(g + 1) * m_g].double()
        if c.x_shared or k == 1:
            xg = (xf if c.x_shared else xf[g * m_g:(g + 1) * m_g]).double()
            gk, sk = dg.t() @ xg, dg.abs().t() @ xg.abs()  # [cout][K]
            rc = c.reduce_cin or cin
            rt = c.reduce_taps or 1
            refs.append((gk[:, :rc * rt].reshape(cout, rt, rc).permute(0, 2, 1).reshape(cout, -1),
                         sk[:, :rc * rt].reshape(cout, rt, rc).permute(0, 2, 1).reshape(cout, -1)))
            continue
        ng = c.n // c.groups
        xg = x[g * ng:(g + 1) * ng].double()
        xp = torch.nn.functional.pad(xg, (0, 0, 1, 1, 1, 1))
        gs, ss = [], []
        for tap in range(9):
            dh, dw = tap // 3, tap % 3
            xs = xp[:, dh:dh + c.h, dw:dw + c.w, :].reshape(-1, cin)
            gs.append(dg.t() @ xs)
            ss.append(dg.abs().t() @ xs.abs())
        refs.append((torch.stack(gs, 2).reshape(cout, -1), torch.stack(ss, 2).reshape(cout, -1)))
    return refs


@pytest.mark.parametrize("case", WGRAD_CASES, ids=[c.name for c in WGRAD_CASES])
def test_wgrad_fp64(cuda_device, case):
    from speak_hack_b200 import ops

    c = case
    dev = cuda_device
    g = _gen(_seed(c))
    rows = c.n * c.h * c.w
    if c.x_shared:
        x = _bf16((c.w, c.cin), g, dev)
        dy = _bf16((c.w * c.groups, c.cout), g, dev)
    elif c.k == 1 and c.n == 1:
        x = _bf16((rows, c.cin), g, dev)
        dy = _bf16((rows, c.cout), g, dev)
    else:
        x = _bf16((c.n, c.h, c.w, c.cin), g, dev)
        dy = _bf16((c.n, c.h, c.w, c.cout), g, dev)
    rc = c.reduce_cin or c.cin
    taps = (c.reduce_taps or 1) if c.reduce_cin else c.k * c.k
    shape = (c.cout, rc, taps)
    init = [torch.randn(shape, generator=g).to(dev) if c.beta else None for _ in range(c.groups)]
    with _env(c.env):
        plan = ops.wgrad_plan(*c.plan_args())
        assert plan is not None, c
        if c.groups == 1 and not c.x_shared:
            x4 = x if x.dim() == 4 else x.view(1, 1, rows, c.cin)
            dy4 = dy if dy.dim() == 4 else dy.view(1, 1, rows, c.cout)
            dws = [ops.conv_wgrad(x4, dy4, c.k, dw=init[0].clone() if c.beta else None, beta=1.0 if c.beta else 0.0,
                                  reduce_cin=c.reduce_cin, reduce_taps=c.reduce_taps, out_shape=shape)]
        else:
            assert not c.beta, "the grouped entry point overwrites"
            dws = [torch.empty(shape, dtype=torch.float32, device=dev) for _ in range(c.groups)]
            ops.conv_wgrad_grouped(x, dy, c.k, dws, x_shared=c.x_shared, reduce_cin=c.reduce_cin,
                                   reduce_taps=c.reduce_taps)
    torch.cuda.synchronize()
    inst = (f"{c.name}: {'wgrad_halo_kernel' if plan['halo'] else 'wgrad_gemm_kernel<%d>' % plan['block_n']} + "
            f"{ops.WGRAD_REDUCE_KERNELS[plan['reduce']]}, {plan['splits']} splits of {plan['kb_per_split']} k blocks "
            f"({plan['num_kb']} per group)")
    # fp32: each split sums kb_per_split * (64 or 128) pixels in TMEM, the reduce adds the splits.  With terms of random
    # sign the partial sums grow like sqrt(k) and the rounding errors add like a random walk: the error of the whole sum
    # is about 2^-24 * S whatever the pixel count or split count (S = sum |x| * |dy|).  EPS_WG = 2^-17 = 128 * 2^-24:
    # the worst element of every case stays below 16 * 2^-24 * S, and a misplaced or dropped 16-pixel block (2^-15 to 2^-14
    # of S at the production sizes) is outside the bound.
    outs = torch.arange(c.cout, device=dev)
    if c.sampled:
        outs = torch.unique(torch.cat([torch.tensor([0, 1, c.cout - 1]), torch.randint(0, c.cout, (13,), generator=g)]))
        outs = outs.to(dev)
    for gi, ((ref, s), dw) in enumerate(zip(wgrad_ref(x, dy, c, outs), dws)):
        got = dw.reshape(c.cout, -1)[outs]
        if c.beta:
            ref = ref + init[gi].double().reshape(c.cout, -1)[outs]
        bound = EPS_WG * s + 2 * U32 * ref.abs() + 1e-30

        def where(i, gi=gi):
            o, r = divmod(i, rc * taps)
            ch, tap = divmod(r, taps)
            return f"{inst}, group {gi} dW[{int(outs[o])}][{ch}][tap {tap}]"

        _note(("halo" if plan["halo"] else "per-tap") + " wgrad",
              _check(inst, got, ref, bound, where))


# ----------------------------------------------------------------------------------------------------------------------
# split bf16 (the generator's <= 32^2 layers)
# ----------------------------------------------------------------------------------------------------------------------
def _half_ulp_ok(y, lo):
    """|lo| <= ulp(y) / 2, exactly (ulp of a bf16 value: 2^(exponent - 7); half an ulp is a power of two)."""
    yf = y.float()
    e = torch.frexp(yf.abs().clamp_min(2.0 ** -126))[1]  # |y| in [2^(e-1), 2^e)
    half_ulp = torch.ldexp(torch.ones_like(yf), (e - 1 - 7 - 1).to(torch.int32))
    return bool((lo.float().abs() <= half_ulp).all())


@pytest.mark.parametrize("n,h,w,cin,cout,bn", [(63, 32, 32, 64, 64, 64), (30, 16, 16, 128, 256, 128),
                                              (64, 8, 8, 512, 512, 0)])
def test_conv_gemm_style_split_fp64(cuda_device, n, h, w, cin, cout, bn):
    from speak_hack_b200 import ops

    c = ConvCase("style-split", STYLE, n, h, w, cin, cout, 3, block_n=bn)
    dev = cuda_device
    x, wk, out, extra = _run_conv(c, dev)
    a2, y2, lo = ops.conv_gemm(x, wk, 3, ops.EPI_STYLE, bias=extra["bias"], nw=extra["nw"], noise=extra["noise"],
                               sp1=extra["sp1"], s1=extra["s1"], force_block_n=bn, split_y=True)
    torch.cuda.synchronize()
    m = n * h * w
    assert torch.equal(a2.reshape(m, cout), out["a"]) and torch.equal(y2.reshape(m, cout), out["y"])
    lo = lo.reshape(m, cout)
    assert _half_ulp_ok(out["y"], lo)
    rows = torch.arange(m, device=dev)
    exp = _conv_expect(c, x, wk, out, extra, rows, m)
    _, yref, _ = exp["y"]
    got = out["y"].double() + lo.double()
    # y + y_lo carries ~16 significant bits: 2^-15 relative, plus the accumulation term the y bound carries
    sp1 = extra["sp1"].double()[rows // (h * w)]
    acc, s = conv_ref(x, wk, 3, 1, False, rows, (n, h, w))
    bound = 2.0 ** -15 * yref.abs() + sp1.abs() * EPS_ACC * s + EPS_F32 * (yref.abs() + acc.abs() * sp1.abs() + 1)
    _note("style split", _check("conv_gemm_style_split y + y_lo", got, yref, bound, lambda i: divmod(i, cout)))


@pytest.mark.parametrize("b,h,w,c", [(64, 4, 4, 512), (64, 8, 8, 512), (7, 32, 32, 64)])
def test_upsample2x_split_fp64(cuda_device, b, h, w, c):
    import ctypes

    from speak_hack_b200 import _lib, ops

    dev = cuda_device
    g = _gen(31)
    y = torch.randn(b, h, w, c, generator=g).to(dev)
    hi = y.to(torch.bfloat16)
    lo = (y - hi.float()).to(torch.bfloat16)
    out = ops.upsample2x_fwd(hi, lo)
    out_plain = ops.upsample2x_fwd(hi)
    plain = torch.empty_like(out_plain)
    rc = _lib.load().irfd_upsample2x_fwd(ctypes.c_void_p(hi.data_ptr()), ctypes.c_void_p(plain.data_ptr()), b, h, w, c,
                                         ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "irfd_upsample2x_fwd")
    torch.cuda.synchronize()
    assert torch.equal(out_plain, plain)  # in_lo = NULL is the plain upsample, bit for bit
    src = (hi.double() + lo.double()).permute(0, 3, 1, 2)
    ref = torch.nn.functional.interpolate(src, scale_factor=2, mode="bilinear", align_corners=False)
    ref = ref.permute(0, 2, 3, 1)
    # one bf16 rounding of the result (2^-9) with fp32 arithmetic on weights that sum to 1
    bound = EPS_OUT * ref.abs() + EPS_F32 * src.abs().amax() + 1e-30
    _note("upsample split", _check("upsample2x_split_fwd", out, ref, bound, lambda i: i))


@pytest.mark.parametrize("b,c", [(64, 512), (3, 64)])
def test_const_input_split_fp64(cuda_device, b, c):
    from speak_hack_b200 import ops

    dev = cuda_device
    g = _gen(41)
    cst = torch.randn(1, c, 4, 4, generator=g).to(dev)
    bias = torch.randn(c, generator=g).to(dev)
    nw = torch.randn(c, generator=g).to(dev)
    noise = torch.randn(b, 16, generator=g).to(dev)
    sp1 = (torch.randn(b, c, generator=g) + 1).to(dev)
    s1 = torch.randn(b, c, generator=g).to(dev)
    a0, y0, y0_lo = ops.const_input_fwd(cst, bias, nw, noise, sp1, s1, split_y=True)
    a1, y1 = ops.const_input_fwd(cst, bias, nw, noise, sp1, s1)
    torch.cuda.synchronize()
    assert torch.equal(a0, a1) and torch.equal(y0, y1)
    assert _half_ulp_ok(y0, y0_lo)
    # a0 = const + bias + nw * noise (no activation on this stage), y0 = a0 * sp1 + s1
    a = (cst.double().reshape(1, c, 16).permute(0, 2, 1) + bias.double() + nw.double() * noise.double()[:, :, None])
    y = a * sp1.double()[:, None, :] + s1.double()[:, None, :]
    t = EPS_F32 * (a.abs() + (nw.double() * noise.double()[:, :, None]).abs() + bias.double().abs() + 1)
    _check("const_input a0", a0.reshape(b, 16, c), a, EPS_OUT * a.abs() + t, lambda i: i)
    bound = 2.0 ** -15 * y.abs() + t * (sp1.double().abs()[:, None, :] + 1)
    _note("const split", _check("const_input y0 + y0_lo", y0.reshape(b, 16, c).double() + y0_lo.reshape(b, 16, c).double(),
                                y, bound, lambda i: i))


# ----------------------------------------------------------------------------------------------------------------------
# production launches
# ----------------------------------------------------------------------------------------------------------------------
# C entry point -> how to read (plan arguments, extras) from its positional arguments
_CONV_ARGS = {  # name: (mode index or fixed mode, wgroups, a_shared, force_block_n)
    "irfd_conv_gemm": (("arg", 10), None, None, 18),
    "irfd_conv_gemm_style_split": (("fixed", STYLE), None, None, 16),
    "irfd_conv_gemm_grouped": (("arg", 9), 12, 13, 14),
    "irfd_conv_gemm_affine": (("fixed", AFFINE), None, None, 13),
    "irfd_conv_gemm_affine_grouped": (("fixed", AFFINE), 13, 14, 15),
    "irfd_conv_gemm_bnbwd_grouped": (("fixed", BNBWD), 16, None, 17),
    "irfd_conv_gemm_bnbwd_res_grouped": (("fixed", BNBWD_RES), 16, None, 17),
}


def record_launches(fn):
    """Runs fn() and returns the conv GEMM launches (plan arguments (n, h, w, cin, cout, ksize, mode, wgroups,
    a_shared, force_block_n)) and weight-gradient launches (n, h, w, cin, cout, ksize, groups, x_shared, reduce_cin,
    reduce_taps) it made, as sets of tuples."""
    from speak_hack_b200 import ops

    conv, wgrad = set(), set()
    orig = ops._call

    def call(name, *a, **kw):
        if name in _CONV_ARGS:
            (how, mi), wg, sh, fb = _CONV_ARGS[name]
            mode = a[mi] if how == "arg" else mi
            conv.add((a[1], a[2], a[3], a[4], a[6], a[7], mode, a[wg] if wg else 1, int(bool(a[sh])) if sh else 0,
                      a[fb]))
        elif name == "irfd_conv_wgrad":
            wgrad.add((a[2], a[3], a[4], a[5], a[6], a[7], 1, 0, a[10], a[11]))
        elif name == "irfd_conv_wgrad_grouped":
            wgrad.add((a[2], a[3], a[4], a[5], a[6], a[7], a[12], a[13], a[10], a[11]))
        return orig(name, *a, **kw)

    ops._call = call
    try:
        fn()
        torch.cuda.synchronize()
    finally:
        ops._call = orig
    return conv, wgrad


def _train_and_d_step(dev, pairs=32):
    """One eager G train step and one D step of the benchmark's workloads (pairs x 2 images at 256^2)."""
    import speak_hack_b200 as P
    from speak_hack_b200.trainer import IRFDDiscriminatorStep, IRFDTrainer

    g = torch.Generator().manual_seed(7)
    x_s = (torch.rand(pairs, 3, 256, 256, generator=g) * 2 - 1).to(dev)
    x_t = (torch.rand(pairs, 3, 256, 256, generator=g) * 2 - 1).to(dev)
    torch.manual_seed(0)
    model = P.IRFD().to(dev).train()
    trainer = IRFDTrainer(model, lr=2e-4, use_cuda_graph=False)
    trainer.train_step_static_eager(x_s, x_t)
    IRFDDiscriminatorStep(model).step(x_s, x_t)


def test_production_launches_are_listed(cuda_device):
    """PROD_CONV_LAUNCHES / PROD_WGRAD_LAUNCHES (from which tests/test_gemm_plan_cpu.py derives the instances the
    sampled production cases must reach) list every GEMM launch shape of the B = 32 train step and of d_step."""
    conv, wgrad = record_launches(lambda: _train_and_d_step(cuda_device))
    assert conv and wgrad
    assert not conv - set(PROD_CONV_LAUNCHES), \
        f"conv launches missing from PROD_CONV_LAUNCHES: {sorted(conv - set(PROD_CONV_LAUNCHES))}"
    assert not wgrad - set(PROD_WGRAD_LAUNCHES), \
        f"wgrad launches missing from PROD_WGRAD_LAUNCHES: {sorted(wgrad - set(PROD_WGRAD_LAUNCHES))}"

