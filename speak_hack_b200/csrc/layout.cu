// Data-movement kernels around the GEMMs: weight packing, explicit im2col for the few strided convs of ResNet-50
// (7x7/2 stem, 3x3/2, 1x1/2 — torchvision/models/resnet.py:197, 133-137, 241), their adjoints, and max/avg pooling.
// All activations NHWC bf16, 16-byte vector accesses, one 8-channel vector per thread.
#include "host_util.h"
#include "rowvec.cuh"

namespace irfd {

// ---------------------------------------------------------------------------------------------------------------
// Weight packing (fp32 OIHW parameter -> bf16 GEMM operand).  dst is always [rows][K] row-major.
//   mode 0 FPROP: dst[o][tap*I + i]            = w[o][i][tap]
//   mode 1 DGRAD: dst[i][(T-1-tap)*O + o]      = w[o][i][tap]      (spatially flipped, in/out swapped)
//   mode 2 DCOL : dst[tap*I + i][o]            = w[o][i][tap]      (for dcol = dz @ W)
//   mode 3 FLAT : dst[o][k], k < kpad          = w[o][k] (k < I*T) else 0   (stem: K = c*49 + kh*7 + kw, padded)
//   mode 4 FLAT_T: dst[k][o], k < kpad         = w[o][k] (k < I*T) else 0   (stem data gradient: dcol = dz @ W)
// ---------------------------------------------------------------------------------------------------------------
__global__ void pack_weight_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ dst, int O, int I, int T,
                                   int mode, int kpad) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (mode == 3) {
    if (idx >= (size_t)O * kpad) return;
    const int o = idx / kpad, k = idx % kpad;
    dst[idx] = __float2bfloat16(k < I * T ? w[(size_t)o * I * T + k] : 0.f);
    return;
  }
  if (mode == 4) {
    if (idx >= (size_t)O * kpad) return;
    const int k = idx / O, o = idx % O;
    dst[idx] = __float2bfloat16(k < I * T ? w[(size_t)o * I * T + k] : 0.f);
    return;
  }
  if (idx >= (size_t)O * I * T) return;
  const int tap = idx % T;
  const int i = (idx / T) % I;
  const int o = idx / ((size_t)T * I);
  const __nv_bfloat16 v = __float2bfloat16(w[idx]);
  size_t d;
  if (mode == 0) d = ((size_t)o * T + tap) * I + i;
  else if (mode == 1) d = ((size_t)i * T + (T - 1 - tap)) * O + o;
  else d = ((size_t)tap * I + i) * O + o;
  dst[d] = v;
}

// ---------------------------------------------------------------------------------------------------------------
// Stem im2col: x NCHW fp32 [N,3,H,W] -> col [N*Ho*Wo][kpad] bf16, 7x7 stride 2 pad 3, k = c*49 + kh*7 + kw
// ---------------------------------------------------------------------------------------------------------------
// One block per (image, output row): the 3 x 7 input rows it needs are staged once in shared memory (zero padded by
// 3 columns on both sides and for out-of-range rows), then every thread assembles 8-element column vectors from
// shared memory.  (The first version gathered each element straight from global memory: 0.45 ms, L1-wavefront-bound;
// the second decoded k = (c*7 + kh)*7 + kw with two integer divisions per ELEMENT: 0.25 ms, issue-bound.)  A thread
// now owns one 8-element vector position v of the kpad-wide row for every eighth output pixel: its eight shared-memory
// offsets are computed once, the loop over pixels is eight loads and one 16-byte store.
constexpr int kStemPixPar = 8;  // output pixels in flight per block pass
__global__ void __launch_bounds__(256)
im2col_stem_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ col, int N, int H, int W, int kpad) {
  extern __shared__ float srow[];  // [3][7][W + 6]
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2, P = W + 6;
  const int n = blockIdx.x / Ho, oh = blockIdx.x - n * Ho;
  // stage: one warp per (channel, kernel row) input row, 16-byte loads when W % 4 == 0 (scalar otherwise), all of a warp's loads
  // independent (the per-element version walked 29 dependent iterations with two divisions each)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int cr = warp; cr < 21; cr += nwarps) {  // cr = c * 7 + kh
    const int c = cr / 7, kh = cr - c * 7;
    const int ih = oh * 2 + kh - 3;
    float* dst = srow + cr * P;
    if (lane < 3) {
      dst[lane] = 0.f;
      dst[P - 3 + lane] = 0.f;
    }
    if (ih >= 0 && ih < H && (W & 3) == 0) {
      const float4* src = reinterpret_cast<const float4*>(x + (((size_t)n * 3 + c) * H + ih) * W);
      for (int j = lane; j < W / 4; j += 32) {
        const float4 q = __ldg(src + j);
        dst[3 + 4 * j] = q.x;
        dst[4 + 4 * j] = q.y;
        dst[5 + 4 * j] = q.z;
        dst[6 + 4 * j] = q.w;
      }
    } else if (ih >= 0 && ih < H) {  // W % 4 != 0: rows are not 16-byte aligned, scalar loads
      const float* src = x + (((size_t)n * 3 + c) * H + ih) * W;
      for (int j = lane; j < W; j += 32) dst[3 + j] = __ldg(src + j);
    } else {
      for (int j = lane; j < W; j += 32) dst[3 + j] = 0.f;
    }
  }
  __syncthreads();
  const int vec_per_row = kpad / 8;            // blockDim.x == kStemPixPar * vec_per_row (host)
  const int v = threadIdx.x % vec_per_row;
  int off[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    const int k = v * 8 + t;                   // k = (c * 7 + kh) * 7 + kw
    off[t] = k < 147 ? (k / 7) * P + (k % 7) : -1;
  }
  const size_t pix0 = ((size_t)n * Ho + oh) * Wo;
  for (int ow = threadIdx.x / vec_per_row; ow < Wo; ow += kStemPixPar) {
    float f[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) f[t] = off[t] >= 0 ? srow[off[t] + 2 * ow] : 0.f;
    store8(col + (pix0 + ow) * kpad + v * 8, f);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Stem data gradient, the adjoint of im2col_stem summed over `nsets` column matrices (the encoders that read the same
// image):  dx[n][c][y][x] = sum_e sum_kh sum_kw dcol[e][(n*Ho + oh)*Wo + ow][(c*7 + kh)*7 + kw]  over the taps with
// y = 2*oh + kh - 3 and x = 2*ow + kw - 3 inside the stem output (Ho = ceil(H/2)).  A gather in a fixed order (per set
// the taps in kh, kw order, then the sets in order): no atomics, deterministic.
// ---------------------------------------------------------------------------------------------------------------
// A block owns a 32 x 32 tile of output pixels of one image; its taps come from a 19 x 19 window of dcol pixels
// (oh in [y0/2 - 1, y0/2 + 17]).  Per (set, channel) the window is staged in shared memory: channel c's 49 taps are the
// seven 16-byte vectors from element 8*floor(49c/8) of the row (column padding from 147 on is never read), and the
// staged pixel stride is odd in 4-byte words so the 16 distinct pixels a warp reads per tap sit in distinct banks.
// The next stage's loads are issued before the current stage is summed (ten 16-byte loads in flight per thread).
// Neighbouring tiles share the 3-pixel halo of their windows; it is read from L2, HBM sees each dcol byte about once.
constexpr int kC2iTile = 32;                   // output tile edge (even: the window starts at y0/2 - 1)
constexpr int kC2iWin = kC2iTile / 2 + 3;      // dcol pixels per window edge
constexpr int kC2iVec = 7;                     // 16-byte vectors per (pixel, channel)
constexpr int kC2iStride = kC2iVec * 4 + 1;    // staged words per pixel
constexpr int kC2iThreads = 256;
constexpr int kC2iPix = kC2iTile * kC2iTile / kC2iThreads;  // output pixels per thread
constexpr int kC2iStage = kC2iWin * kC2iWin * kC2iVec;      // 16-byte vectors per stage
constexpr int kC2iLoads = (kC2iStage + kC2iThreads - 1) / kC2iThreads;

__device__ __forceinline__ void c2i_load(uint4 (&q)[kC2iLoads], const __nv_bfloat16* __restrict__ src, int c, int oh0,
                                         int ow0, int Ho, int Wo, int ld) {
  const int v0 = c * 49 / 8;
#pragma unroll
  for (int j = 0; j < kC2iLoads; ++j) {
    const int i = threadIdx.x + j * kC2iThreads;
    const int p = i / kC2iVec, v = i - p * kC2iVec;
    const int oh = oh0 + p / kC2iWin, ow = ow0 + p % kC2iWin;
    q[j] = make_uint4(0, 0, 0, 0);  // outside the stem output: the tap falls on padding, contributes 0
    if (i < kC2iStage && (unsigned)oh < (unsigned)Ho && (unsigned)ow < (unsigned)Wo)
      q[j] = ldg16(src + ((size_t)oh * Wo + ow) * ld + (v0 + v) * 8);
  }
}

__device__ __forceinline__ void c2i_store(const uint4 (&q)[kC2iLoads], uint32_t* stage) {
#pragma unroll
  for (int j = 0; j < kC2iLoads; ++j) {
    const int i = threadIdx.x + j * kC2iThreads;
    if (i >= kC2iStage) break;
    const int p = i / kC2iVec, v = i - p * kC2iVec;
    uint32_t* d = stage + p * kC2iStride + v * 4;
    d[0] = q[j].x;
    d[1] = q[j].y;
    d[2] = q[j].z;
    d[3] = q[j].w;
  }
}

__global__ void __launch_bounds__(kC2iThreads, 2)
col2im_stem_kernel(const __nv_bfloat16* __restrict__ dcol, float* __restrict__ dx, int N, int H, int W, int ld,
                   int nsets) {
  __shared__ uint32_t stage[kC2iWin * kC2iWin * kC2iStride];
  const __nv_bfloat16* sb = reinterpret_cast<const __nv_bfloat16*>(stage);
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
  const int n = blockIdx.z, y0 = blockIdx.y * kC2iTile, x0 = blockIdx.x * kC2iTile;
  const int oh0 = y0 / 2 - 1, ow0 = x0 / 2 - 1;
  const size_t set_stride = (size_t)N * Ho * Wo * ld;
  const __nv_bfloat16* img = dcol + (size_t)n * Ho * Wo * ld;
  float acc[3][kC2iPix];
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int r = 0; r < kC2iPix; ++r) acc[c][r] = 0.f;
  uint4 q[kC2iLoads];
  c2i_load(q, img, 0, oh0, ow0, Ho, Wo, ld);
  for (int e = 0; e < nsets; ++e) {
#pragma unroll 1
    for (int c = 0; c < 3; ++c) {
      __syncthreads();  // the previous stage is consumed
      c2i_store(q, stage);
      __syncthreads();
      const int en = c == 2 ? e + 1 : e;
      if (en < nsets) c2i_load(q, img + en * set_stride, c == 2 ? 0 : c + 1, oh0, ow0, Ho, Wo, ld);
      const int off = c * 49 - (c * 49 / 8) * 8;  // tap 0's element in the staged vectors
#pragma unroll
      for (int r = 0; r < kC2iPix; ++r) {
        const int t = threadIdx.x + r * kC2iThreads, ty = t / kC2iTile, tx = t % kC2iTile;
        // (y + 3 - kh) even; y0 is even, so the first tap has the parity of ty + 1.  Window row of (oh): oh - oh0.
        float a = 0.f;
        for (int kh = (ty + 1) & 1; kh < 7; kh += 2) {
          const int py = (ty + 3 - kh) / 2 + 1;
          for (int kw = (tx + 1) & 1; kw < 7; kw += 2) {
            const int px = (tx + 3 - kw) / 2 + 1;
            a += __bfloat162float(sb[(py * kC2iWin + px) * 2 * kC2iStride + off + kh * 7 + kw]);
          }
        }
        // registers, not a runtime-indexed (local-memory) array
        acc[0][r] += c == 0 ? a : 0.f;
        acc[1][r] += c == 1 ? a : 0.f;
        acc[2][r] += c == 2 ? a : 0.f;
      }
    }
  }
#pragma unroll
  for (int r = 0; r < kC2iPix; ++r) {
    const int t = threadIdx.x + r * kC2iThreads, y = y0 + t / kC2iTile, x = x0 + t % kC2iTile;
    if (y >= H || x >= W) continue;
#pragma unroll
    for (int c = 0; c < 3; ++c) dx[(((size_t)n * 3 + c) * H + y) * W + x] = acc[c][r];
  }
}

// 3x3 stride-2 pad-1 im2col on NHWC bf16: col[pix][tap*C + c]
__global__ void im2col_3x3s2_kernel(const __nv_bfloat16* __restrict__ a, __nv_bfloat16* __restrict__ col, int N, int H,
                                    int W, int C) {
  const unsigned Ho = (H + 1) / 2, Wo = (W + 1) / 2, vc = C / 8;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;  // host checks total < 2^32
  const size_t total = (size_t)N * Ho * Wo * 9 * vc;
  if (idx >= total) return;
  const int v = idx % vc;
  const int tap = (idx / vc) % 9;
  const unsigned pix = idx / (vc * 9u);
  const int ow = pix % Wo, oh = (pix / Wo) % Ho, n = pix / ((unsigned)Wo * Ho);
  const int ih = oh * 2 + tap / 3 - 1, iw = ow * 2 + tap % 3 - 1;
  uint4 val = make_uint4(0, 0, 0, 0);
  if (ih >= 0 && ih < H && iw >= 0 && iw < W)
    val = *reinterpret_cast<const uint4*>(a + (((size_t)n * H + ih) * W + iw) * C + v * 8);
  *reinterpret_cast<uint4*>(col + ((size_t)pix * 9 + tap) * C + v * 8) = val;
}

// adjoint: dx[n,h,w,c] = sum over (oh,ow,tap) hitting (h,w) of dcol[(oh,ow)][tap*C + c]
__global__ void col2im_3x3s2_kernel(const __nv_bfloat16* __restrict__ dcol, __nv_bfloat16* __restrict__ dx, int N,
                                    int H, int W, int C) {
  const unsigned Ho = H / 2, Wo = W / 2, vc = C / 8;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;  // host checks total < 2^32
  const size_t total = (size_t)N * H * W * vc;
  if (idx >= total) return;
  const int v = idx % vc;
  const unsigned pix = idx / vc;
  const int w = pix % W, h = (pix / W) % H, n = pix / ((unsigned)W * H);
  float acc[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) acc[t] = 0.f;
  // h = 2*oh + kh - 1
  for (int kh = 0; kh < 3; ++kh) {
    const int th = h - kh + 1;
    if (th < 0 || (th & 1)) continue;
    const int oh = th >> 1;
    if (oh >= Ho) continue;
    for (int kw = 0; kw < 3; ++kw) {
      const int tw = w - kw + 1;
      if (tw < 0 || (tw & 1)) continue;
      const int ow = tw >> 1;
      if (ow >= Wo) continue;
      float f[8];
      load8(dcol + ((((size_t)n * Ho + oh) * Wo + ow) * 9 + kh * 3 + kw) * C + v * 8, f);
#pragma unroll
      for (int t = 0; t < 8; ++t) acc[t] += f[t];
    }
  }
  store8(dx + (size_t)pix * C + v * 8, acc);
}

// 1x1 stride-2 gather: out[n,oh,ow,:] = a[n,2oh,2ow,:]
__global__ void subsample2_kernel(const __nv_bfloat16* __restrict__ a, __nv_bfloat16* __restrict__ out, int N, int H,
                                  int W, int C) {
  const unsigned Ho = (H + 1) / 2, Wo = (W + 1) / 2, vc = C / 8;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;  // host checks total < 2^32
  if (idx >= (size_t)N * Ho * Wo * vc) return;
  const int v = idx % vc;
  const unsigned pix = idx / vc;
  const int ow = pix % Wo, oh = (pix / Wo) % Ho, n = pix / ((unsigned)Wo * Ho);
  *reinterpret_cast<uint4*>(out + (size_t)pix * C + v * 8) =
      *reinterpret_cast<const uint4*>(a + (((size_t)n * H + 2 * oh) * W + 2 * ow) * C + v * 8);
}

// out[n,h,w,:] = a[n,h,w,:] (or 0 if a == null) + (h,w even ? b[n,h/2,w/2,:] : 0)     (adjoint of subsample2, fused add)
__global__ void scatter_add_s2_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ b,
                                      __nv_bfloat16* __restrict__ out, int N, int H, int W, int C) {
  const unsigned vc = C / 8;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;  // host checks total < 2^32
  if (idx >= (size_t)N * H * W * vc) return;
  const int v = idx % vc;
  const unsigned pix = idx / vc;
  const int w = pix % W, h = (pix / W) % H, n = pix / ((unsigned)W * H);
  float f[8];
  if (a != nullptr) load8(a + (size_t)pix * C + v * 8, f);
  else {
#pragma unroll
    for (int t = 0; t < 8; ++t) f[t] = 0.f;
  }
  if (!(h & 1) && !(w & 1)) {
    float g[8];
    load8(b + (((size_t)n * (H / 2) + h / 2) * (W / 2) + w / 2) * C + v * 8, g);
#pragma unroll
    for (int t = 0; t < 8; ++t) f[t] += g[t];
  }
  store8(out + (size_t)pix * C + v * 8, f);
}

// ---------------------------------------------------------------------------------------------------------------
// MaxPool2d(3, stride 2, pad 1) forward (+ argmax tap, first maximum in scan order like ATen) and backward (gather).
// ---------------------------------------------------------------------------------------------------------------
__global__ void maxpool_fwd_kernel(const __nv_bfloat16* __restrict__ a, __nv_bfloat16* __restrict__ out,
                                   uint8_t* __restrict__ arg, int N, int H, int W, int C) {
  const unsigned Ho = (H + 1) / 2, Wo = (W + 1) / 2, vc = C / 8;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;  // host checks total < 2^32
  if (idx >= (size_t)N * Ho * Wo * vc) return;
  const int v = idx % vc;
  const unsigned pix = idx / vc;
  const int ow = pix % Wo, oh = (pix / Wo) % Ho, n = pix / ((unsigned)Wo * Ho);
  float best[8];
  int bi[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    best[t] = -INFINITY;
    bi[t] = 0;
  }
  for (int tap = 0; tap < 9; ++tap) {
    const int ih = oh * 2 + tap / 3 - 1, iw = ow * 2 + tap % 3 - 1;
    if (ih < 0 || ih >= H || iw < 0 || iw >= W) continue;
    float f[8];
    load8(a + (((size_t)n * H + ih) * W + iw) * C + v * 8, f);
#pragma unroll
    for (int t = 0; t < 8; ++t)
      if (f[t] > best[t]) {
        best[t] = f[t];
        bi[t] = tap;
      }
  }
  store8(out + (size_t)pix * C + v * 8, best);
  uint2 packed;
  packed.x = bi[0] | (bi[1] << 8) | (bi[2] << 16) | (bi[3] << 24);
  packed.y = bi[4] | (bi[5] << 8) | (bi[6] << 16) | (bi[7] << 24);
  *reinterpret_cast<uint2*>(arg + (size_t)pix * C + v * 8) = packed;
}

// A thread owns a 2 x 2 quad of input pixels (rows 2i, 2i+1; columns 2j, 2j+1) for 8 channels.  With stride 2,
// kernel 3, pad 1 the quad only lies in the pooling windows (i..i+1) x (j..j+1): an even row 2i belongs to window row i
// through tap kh = 1, the odd row 2i+1 to window rows i+1 (kh = 0) and i (kh = 2).  The four windows' gradient and
// argmax vectors are loaded ONCE and serve the nine (pixel, window) pairs; per pixel the candidates are added in
// ascending tap order, the order of a 3 x 3 walk.  (Round-2 history: the 3 x 3 walk with parity tests was issue-bound
// at 1.3 TB/s; one pixel per thread with its <= 2 x 2 candidate windows re-read every window 2.25 times: 1.8 TB/s.)
// grid = (N * H/2 row pairs, segments of (W/2) * C/8 quads).
__global__ void __launch_bounds__(256)
maxpool_bwd_kernel(const __nv_bfloat16* __restrict__ dout, const __nv_bfloat16* __restrict__ dout2,
                   const uint8_t* __restrict__ arg, __nv_bfloat16* __restrict__ dx, int N, int H, int W, int C) {
  const unsigned Ho = H / 2, Wo = W / 2, vc = C >> 3;
  const unsigned q = blockIdx.y * blockDim.x + threadIdx.x;
  if (q >= Wo * vc) return;
  const int j = q / vc, v = q - j * vc;
  const int n = blockIdx.x / Ho, i = blockIdx.x - n * Ho;
  float g[2][2][8];
  uint2 am[2][2];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      am[a][b] = make_uint2(0xffffffffu, 0xffffffffu);  // no tap matches 0xff: windows outside the image contribute 0
#pragma unroll
      for (int t = 0; t < 8; ++t) g[a][b][t] = 0.f;
      if ((unsigned)(i + a) < Ho && (unsigned)(j + b) < Wo) {
        const size_t op = (((size_t)n * Ho + i + a) * Wo + j + b) * C + v * 8;
        am[a][b] = __ldg(reinterpret_cast<const uint2*>(arg + op));
        unpack8(ldg16(dout + op), g[a][b]);
        if (dout2 != nullptr) {
          float g2[8];
          unpack8(ldg16(dout2 + op), g2);
#pragma unroll
          for (int t = 0; t < 8; ++t) g[a][b][t] += g2[t];
        }
      }
    }
#pragma unroll
  for (int pa = 0; pa < 2; ++pa)
#pragma unroll
    for (int pb = 0; pb < 2; ++pb) {
      float acc[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) acc[t] = 0.f;
      // row candidates of input row 2i + pa in ascending tap order: (window a, tap kh)
#pragma unroll
      for (int ra = 0; ra < 2; ++ra) {
        const int a = pa ? 1 - ra : 0;          // odd row: window i+1 (kh 0) first, then window i (kh 2)
        const int kh = pa ? (ra ? 2 : 0) : 1;
        if (!pa && ra) continue;                // an even row has one candidate
#pragma unroll
        for (int rb = 0; rb < 2; ++rb) {
          const int b = pb ? 1 - rb : 0;
          const int kw = pb ? (rb ? 2 : 0) : 1;
          if (!pb && rb) continue;
          const unsigned tap = kh * 3 + kw;
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            const unsigned m = ((t < 4 ? am[a][b].x : am[a][b].y) >> ((t & 3) * 8)) & 0xffu;
            if (m == tap) acc[t] += g[a][b][t];
          }
        }
      }
      store8(dx + (((size_t)n * H + 2 * i + pa) * W + 2 * j + pb) * C + v * 8, acc);
    }
}

// AdaptiveAvgPool2d(1): [N, HW, C] bf16 -> [N, C] fp32 ; backward broadcasts dfeat/HW
__global__ void __launch_bounds__(kRvThreads)
avgpool_fwd_kernel(const __nv_bfloat16* __restrict__ a, float* __restrict__ out, int HW, int C) {
  extern __shared__ float red_smem[];
  RowVec rv(C);
  float acc[1][8];
#pragma unroll
  for (int t = 0; t < 8; ++t) acc[0][t] = 0.f;
  if (rv.active) {
    for (int r = rv.row_lane; r < HW; r += rv.rows_par) {
      float f[8];
      load8(a + ((size_t)blockIdx.x * HW + r) * C + rv.cv * 8, f);
#pragma unroll
      for (int t = 0; t < 8; ++t) acc[0][t] += f[t];
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) acc[0][t] *= 1.f / HW;
  }
  block_reduce_rows<1>(rv, C, acc, red_smem, out + (size_t)blockIdx.x * C, 0);
}

__global__ void avgpool_bwd_kernel(const float* __restrict__ dfeat, __nv_bfloat16* __restrict__ g, int N, int HW,
                                   int C) {
  const unsigned vc = C / 8;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;  // host checks total < 2^32
  if (idx >= (size_t)N * HW * vc) return;
  const int v = idx % vc;
  const unsigned pix = idx / vc;
  const unsigned n = pix / (unsigned)HW;
  float f[8];
  loadf8(dfeat + (size_t)n * C + v * 8, f);
#pragma unroll
  for (int t = 0; t < 8; ++t) f[t] *= 1.f / HW;
  store8(g + (size_t)pix * C + v * 8, f);
}

// ---------------------------------------------------------------------------------------------------------------
// NCHW fp32 <-> NHWC bf16 (the reference's module interfaces are NCHW fp32; the kernels work on NHWC bf16).  Used by
// the standalone forwards of the per-layer modules (SynthesisBlock, ApplyNoise, ApplyStyle); the fused paths never
// materialise NCHW activations.  32 x 32 (channel x pixel) tiles through shared memory: coalesced on both sides.
// c_pad >= c: channels [c, c_pad) of the NHWC tensor are written as zero (64-channel GEMM tiles) / ignored.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
nchw_to_nhwc_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, int C, int HW, int c_pad) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, p = p0 + tx;
    tile[i][tx] = (c < C && p < HW) ? in[((size_t)b * C + c) * HW + p] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int p = p0 + i, c = c0 + tx;
    if (p < HW && c < c_pad) out[((size_t)b * HW + p) * c_pad + c] = __float2bfloat16(tile[tx][i]);
  }
}

__global__ void __launch_bounds__(256)
nhwc_to_nchw_kernel(const __nv_bfloat16* __restrict__ in, float* __restrict__ out, int C, int HW, int c_pad) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const int p = p0 + i, c = c0 + tx;
    tile[i][tx] = (p < HW && c < c_pad) ? __bfloat162float(in[((size_t)b * HW + p) * c_pad + c]) : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, p = p0 + tx;
    if (c < C && p < HW) out[((size_t)b * C + c) * HW + p] = tile[tx][i];
  }
}

}  // namespace irfd

using namespace irfd;

#define GRID1D(total) (unsigned)(((total) + 255) / 256), 256, 0, stream
#define CHECK_TOTAL32(total) IRFD_CHECK_ARG((total) > 0 && (total) < ((size_t)1 << 32) - 256, "tensor too large for 32-bit indexing")
#define BF(p) reinterpret_cast<__nv_bfloat16*>(p)
#define CBF(p) reinterpret_cast<const __nv_bfloat16*>(p)

extern "C" int irfd_pack_conv_weight(const float* w, void* dst, int o, int i, int taps, int mode, int kpad,
                                     cudaStream_t stream) {
  IRFD_CHECK_ARG(w && dst && o > 0 && i > 0 && taps > 0 && mode >= 0 && mode <= 4, "pack_conv_weight: bad argument");
  IRFD_CHECK_ARG(mode != 4 || kpad >= i * taps, "pack_conv_weight: FLAT_T needs kpad >= %d (got %d)", i * taps, kpad);
  const size_t total = mode >= 3 ? (size_t)o * kpad : (size_t)o * i * taps;
  pack_weight_kernel<<<GRID1D(total)>>>(w, BF(dst), o, i, taps, mode, kpad);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_im2col_stem(const float* x, void* col, int n, int h, int w, int kpad, cudaStream_t stream) {
  IRFD_CHECK_ARG(x && col && kpad >= 152 && kpad % 8 == 0 && h > 0 && w > 0, "im2col_stem: bad argument");
  const size_t smem = (size_t)21 * (w + 6) * sizeof(float);
  IRFD_CHECK_ARG(n > 0 && smem <= 48 * 1024, "im2col_stem: image too wide for the row stage (W <= 579, got %d)", w);
  IRFD_CHECK_ARG(kStemPixPar * (kpad / 8) <= 256 && (kpad / 8) % 4 == 0, "im2col_stem: kpad a multiple of 32 and <= 256");
  im2col_stem_kernel<<<(unsigned)(n * ((h + 1) / 2)), kStemPixPar * (kpad / 8), smem, stream>>>(x, BF(col), n, h, w,
                                                                                              kpad);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_col2im_stem(const void* dcol, float* dx, int n, int h, int w, int kpad, int nsets,
                                cudaStream_t stream) {
  IRFD_CHECK_ARG(dcol && dx && ((uintptr_t)dcol & 15) == 0, "col2im_stem: null or unaligned pointer");
  IRFD_CHECK_ARG(nsets >= 1 && nsets <= 4, "col2im_stem: 1..4 column sets (got %d)", nsets);
  IRFD_CHECK_ARG(kpad >= 152 && kpad % 8 == 0, "col2im_stem: kpad a multiple of 8 and >= 152 (got %d)", kpad);
  IRFD_CHECK_ARG(n > 0 && n <= 65535 && h > 0 && w > 0 && h <= 65535 * kC2iTile && w <= 65535 * kC2iTile,
                 "col2im_stem: bad shape n=%d h=%d w=%d", n, h, w);
  col2im_stem_kernel<<<dim3((unsigned)((w + kC2iTile - 1) / kC2iTile), (unsigned)((h + kC2iTile - 1) / kC2iTile),
                            (unsigned)n), kC2iThreads, 0, stream>>>(CBF(dcol), dx, n, h, w, kpad, nsets);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_im2col_3x3s2(const void* a, void* col, int n, int h, int w, int c, cudaStream_t stream) {
  IRFD_CHECK_ARG(a && col && c % 8 == 0 && h > 0 && w > 0, "im2col_3x3s2: bad argument");
  const size_t total = (size_t)n * ((h + 1) / 2) * ((w + 1) / 2) * 9 * (c / 8);
  CHECK_TOTAL32(total);
  im2col_3x3s2_kernel<<<GRID1D(total)>>>(CBF(a), BF(col), n, h, w, c);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_col2im_3x3s2(const void* dcol, void* dx, int n, int h, int w, int c, cudaStream_t stream) {
  IRFD_CHECK_ARG(dcol && dx && c % 8 == 0 && h % 2 == 0 && w % 2 == 0, "col2im_3x3s2: bad argument");
  const size_t total = (size_t)n * h * w * (c / 8);
  CHECK_TOTAL32(total);
  col2im_3x3s2_kernel<<<GRID1D(total)>>>(CBF(dcol), BF(dx), n, h, w, c);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_subsample2(const void* a, void* out, int n, int h, int w, int c, cudaStream_t stream) {
  IRFD_CHECK_ARG(a && out && c % 8 == 0 && h > 0 && w > 0, "subsample2: bad argument");
  const size_t total = (size_t)n * ((h + 1) / 2) * ((w + 1) / 2) * (c / 8);
  CHECK_TOTAL32(total);
  subsample2_kernel<<<GRID1D(total)>>>(CBF(a), BF(out), n, h, w, c);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_scatter_add_s2(const void* a, const void* b, void* out, int n, int h, int w, int c,
                                   cudaStream_t stream) {
  IRFD_CHECK_ARG(b && out && c % 8 == 0 && h % 2 == 0 && w % 2 == 0, "scatter_add_s2: bad argument");
  const size_t total = (size_t)n * h * w * (c / 8);
  CHECK_TOTAL32(total);
  scatter_add_s2_kernel<<<GRID1D(total)>>>(CBF(a), CBF(b), BF(out), n, h, w, c);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_maxpool_fwd(const void* a, void* out, void* argmax, int n, int h, int w, int c,
                                cudaStream_t stream) {
  IRFD_CHECK_ARG(a && out && argmax && c % 8 == 0 && h > 0 && w > 0, "maxpool_fwd: bad argument");
  const size_t total = (size_t)n * ((h + 1) / 2) * ((w + 1) / 2) * (c / 8);
  CHECK_TOTAL32(total);
  maxpool_fwd_kernel<<<GRID1D(total)>>>(CBF(a), BF(out), reinterpret_cast<uint8_t*>(argmax), n, h, w, c);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_maxpool_bwd(const void* dout, const void* dout2, const void* argmax, void* dx, int n, int h, int w,
                                int c, cudaStream_t stream) {
  IRFD_CHECK_ARG(dout && dx && argmax && c % 8 == 0 && h % 2 == 0 && w % 2 == 0, "maxpool_bwd: bad argument");
  IRFD_CHECK_ARG((long long)w * c < (1ll << 24) && (long long)n * h < (1ll << 31), "maxpool_bwd: bad shape");
  maxpool_bwd_kernel<<<dim3((unsigned)(n * (h / 2)), (unsigned)(((w / 2) * (c / 8) + 255) / 256)), 256, 0, stream>>>(
      CBF(dout), CBF(dout2), reinterpret_cast<const uint8_t*>(argmax), BF(dx), n, h, w, c);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_avgpool_fwd(const void* a, float* out, int n, int hw, int c, cudaStream_t stream) {
  IRFD_CHECK_ARG(a && out && c % 8 == 0 && c <= 2048 && hw > 0, "avgpool_fwd: bad argument");
  avgpool_fwd_kernel<<<n, kRvThreads, 2048 * sizeof(float), stream>>>(CBF(a), out, hw, c);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_avgpool_bwd(const float* dfeat, void* g, int n, int hw, int c, cudaStream_t stream) {
  IRFD_CHECK_ARG(dfeat && g && c % 8 == 0 && hw > 0, "avgpool_bwd: bad argument");
  const size_t total = (size_t)n * hw * (c / 8);
  CHECK_TOTAL32(total);
  avgpool_bwd_kernel<<<GRID1D(total)>>>(dfeat, BF(g), n, hw, c);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_nchw_to_nhwc_bf16(const float* in, void* out, int b, int c, int hw, int c_pad, cudaStream_t stream) {
  IRFD_CHECK_ARG(in && out && b > 0 && c > 0 && hw > 0 && c_pad >= c, "nchw_to_nhwc_bf16: bad argument");
  nchw_to_nhwc_kernel<<<dim3((hw + 31) / 32, (c_pad + 31) / 32, b), 256, 0, stream>>>(
      in, reinterpret_cast<__nv_bfloat16*>(out), c, hw, c_pad);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_nhwc_bf16_to_nchw(const void* in, float* out, int b, int c, int hw, int c_pad, cudaStream_t stream) {
  IRFD_CHECK_ARG(in && out && b > 0 && c > 0 && hw > 0 && c_pad >= c, "nhwc_bf16_to_nchw: bad argument");
  nhwc_to_nchw_kernel<<<dim3((hw + 31) / 32, (c_pad + 31) / 32, b), 256, 0, stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(in), out, c, hw, c_pad);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}
