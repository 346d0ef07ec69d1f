// Weight-gradient GEMM for stride-1 "same" convolutions (ksize 1 or 3) on tcgen05 tensor cores.
//
//   dWt[k, n] = sum_pixels  X[pixel + shift(tap), c] * dY[pixel, n]        k = tap*Cin + c,  n = out channel
//
// The reduction runs over PIXELS, which is the strided dimension of NHWC, so both operands are fed to the tensor core
// MN-major (tcgen05 transposes in the datapath; no transposed copies are ever materialised):
//   A tile (M = 128 = two 64-channel atoms of (tap, c-chunk))  <- two 4-D TMA boxes [64 pixels x 64 ch] of X, shifted
//   B tile (N = BLOCK_N out channels = BLOCK_N/64 atoms)        <- 2-D TMA boxes [64 pixels x 64 ch] of dY
// Split-K over pixel ranges: each CTA owns (k-pair, n-tile, pixel-range) and writes an fp32 partial
// [split][Ktot][Cout]; the wgrad_reduce kernels sum the splits in a fixed order (deterministic) into OIHW fp32.
// wgrad_halo_kernel (further down) is the 3x3 variant that keeps all nine taps of a Cin chunk in TMEM and streams X
// once per chunk instead of once per (tap, chunk) pair.
#include <stdlib.h>

#include "host_util.h"
#include "ptx.cuh"

namespace irfd {

struct WgradArgs {
  int M_total, N_total, K_total;
  int num_pairs, num_n_tiles, splits;
  int num_kb, kb_per_split;
  int taps, kw, pad, cin_chunks, num_atoms;
  int H, W;
  float* partial;  // [groups][splits][K_total][N_total]
  // Weight groups (the same layer of the three IRFD encoders in ONE launch): the pixel range is stacked group-major,
  // group g owns k-blocks [g * num_kb, (g + 1) * num_kb) and its own partial block; x_shared: every group reads the
  // SAME x rows (the stem's shared im2col matrix), only dY is stacked.
  int groups, x_shared;
};

constexpr int kMaxWgGroups = 4;
struct WgDst {
  float* p[kMaxWgGroups];
};

constexpr int kWgThreads = 192;  // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue
constexpr int kWgWaves = 1;      // split-K target: CTAs per SM over the launch (1 measured faster than 2: fewer partials)
constexpr int kWgMinKb = 16;    // shorter splits only multiply prologues and fp32 partial traffic

template <int BLOCK_N>
struct WgCfg {
  static constexpr int A_BYTES = 2 * 8192;
  static constexpr int B_BYTES = (BLOCK_N / 64) * 8192;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  // at most 196 KB per CTA: the weight gradients run on the side stream beside the row-streaming BatchNorm / style
  // kernels and their finalize launches, which need the rest of the SM's shared memory to become co-resident
  static constexpr int RAW_STAGES = (200704 - 1024 - 1024) / STAGE_BYTES;
  static constexpr int STAGES = RAW_STAGES > 8 ? 8 : RAW_STAGES;
  static constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + 1024;
  static constexpr uint32_t TMEM_COLS = BLOCK_N <= 64 ? 64 : (BLOCK_N <= 128 ? 128 : 256);
};

template <int BLOCK_N>
__global__ void __launch_bounds__(kWgThreads, 1)
wgrad_gemm_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_dy,
                  const WgradArgs p) {
  using Cfg = WgCfg<BLOCK_N>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* done_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(done_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // work item: (group, k-pair, n tile, split)
  int item = blockIdx.x;
  const int split = item % p.splits;
  item /= p.splits;
  const int n_tile = item % p.num_n_tiles;
  item /= p.num_n_tiles;
  const int pair = item % p.num_pairs;
  const int grp = item / p.num_pairs;
  int kb_begin = split * p.kb_per_split;
  int kb_end = kb_begin + p.kb_per_split;
  if (kb_end > p.num_kb) kb_end = p.num_kb;
  const int my_kb = kb_end > kb_begin ? kb_end - kb_begin : 0;
  const int kb_off = grp * p.num_kb;             // dY (and x unless shared) are stacked group-major
  const int kb_off_x = p.x_shared ? 0 : kb_off;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(done_bar, 1);
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc<Cfg::TMEM_COLS>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // TMA producer: whole warp converged, one elected lane issues
    if (lane == 0) {
      tma_prefetch_desc(&map_x);
      tma_prefetch_desc(&map_dy);
    }
    __syncwarp();
    int atom[2];
    atom[0] = pair * 2;
    atom[1] = pair * 2 + 1 < p.num_atoms ? pair * 2 + 1 : p.num_atoms - 1;  // odd tail: duplicate, discarded later
    int dh[2], dw[2], c0[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int tap = atom[i] / p.cin_chunks;
      c0[i] = (atom[i] - tap * p.cin_chunks) * 64;
      dh[i] = tap / p.kw - p.pad;
      dw[i] = tap % p.kw - p.pad;
    }
    int stage = 0;
    uint32_t phase = 0;
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      const int p0 = (kb + kb_off) * 64;
      const int px = (kb + kb_off_x) * 64;
      const int w0 = px % p.W;
      const int h0 = (px / p.W) % p.H;
      const int n0 = px / (p.W * p.H);
      mbar_wait(&empty_bar[stage], phase ^ 1);
      uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
      uint8_t* sb = sa + Cfg::A_BYTES;
      if (elect_one_sync()) {
        mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
        tma_load_4d(sa, &map_x, &full_bar[stage], c0[0], w0 + dw[0], h0 + dh[0], n0);
        tma_load_4d(sa + 8192, &map_x, &full_bar[stage], c0[1], w0 + dw[1], h0 + dh[1], n0);
#pragma unroll
        for (int j = 0; j < BLOCK_N / 64; ++j)
          tma_load_2d(sb + j * 8192, &map_dy, &full_bar[stage], n_tile * BLOCK_N + j * 64, p0);
      }
      __syncwarp();
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp == 1) {
    // MMA issuer: whole warp converged, one elected lane issues (keeps descriptors in uniform registers)
    constexpr uint32_t idesc = make_idesc_bf16(128, BLOCK_N, 1, 1);  // both operands MN-major
    int stage = 0;
    uint32_t phase = 0;
    for (int i = 0; i < my_kb; ++i) {
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
      const uint64_t adesc0 = make_smem_desc_sw128(a_addr, 8192, 1024);
      const uint64_t bdesc0 = make_smem_desc_sw128(a_addr + Cfg::A_BYTES, 8192, 1024);
      if (elect_one_sync()) {
#pragma unroll
        for (int k = 0; k < 4; ++k)  // 16 pixels (= 16 rows of 128 B = 2048 B = 128 address units) per MMA
          umma_bf16(tmem_base, adesc0 + 128 * k, bdesc0 + 128 * k, idesc, (i | k) != 0 ? 1u : 0u);
        umma_commit(&empty_bar[stage]);
      }
      __syncwarp();
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1;
      }
    }
    if (elect_one_sync()) umma_commit(done_bar);
    __syncwarp();
  } else {
    // epilogue: 4 warps, thread <-> TMEM lane <-> k row
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const int atom_i = r >> 6;
    const bool valid = (pair * 2 + atom_i) < p.num_atoms;
    const size_t krow = (size_t)pair * 128 + r;
    float* dst = p.partial + (((size_t)grp * p.splits + split) * p.K_total + krow) * p.N_total + (size_t)n_tile * BLOCK_N;
    if (my_kb > 0) {
      mbar_wait(done_bar, 0);
      tc_fence_after();
    }
#pragma unroll 1
    for (int chunk = 0; chunk < BLOCK_N / 32; ++chunk) {
      uint32_t v[32];
      if (my_kb > 0) {
        tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + chunk * 32, v);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int t = 0; t < 32; ++t) v[t] = 0u;
      }
      if (valid) {
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          float4 o = make_float4(__uint_as_float(v[4 * t]), __uint_as_float(v[4 * t + 1]),
                                 __uint_as_float(v[4 * t + 2]), __uint_as_float(v[4 * t + 3]));
          *reinterpret_cast<float4*>(dst + chunk * 32 + 4 * t) = o;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
}

// dW[o][c][tap] (OIHW, fp32) = beta * dW + sum_s partial[s][tap*Cin + c][o]
// Block = (256 / LANES) consecutive outputs (coalesced partial reads) x LANES split lanes: every thread sums the
// splits s = lane, lane + LANES, ... with four loads in flight, the partial sums are combined in a fixed order
// (bit-deterministic).  The first version walked all splits (up to 148) serially in one thread per output: ~20 us of
// pure load latency per launch on the 1x1 layers.
template <int LANES>  // split lanes per output: 256 threads = (256 / LANES) consecutive outputs x LANES
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ partial, WgDst dws, int splits, int K_total, int N_total, int cin,
                    int taps, float beta) {
  constexpr int OUTS = 256 / LANES;
  float* __restrict__ dw = dws.p[blockIdx.y];  // weight group = blockIdx.y
  partial += (size_t)blockIdx.y * splits * K_total * N_total;
  __shared__ float part[LANES][OUTS + 1];
  const int o = threadIdx.x % OUTS, w = threadIdx.x / OUTS;
  const size_t idx = (size_t)blockIdx.x * OUTS + o;  // over [K_total][N_total], n fastest
  const size_t stride = (size_t)K_total * N_total;
  const bool in_range = idx < stride;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (in_range) {
    const float* p = partial + idx;
    int s = w;
    for (; s + 3 * LANES < splits; s += 4 * LANES) {
      a0 += __ldg(p + (size_t)s * stride);
      a1 += __ldg(p + (size_t)(s + LANES) * stride);
      a2 += __ldg(p + (size_t)(s + 2 * LANES) * stride);
      a3 += __ldg(p + (size_t)(s + 3 * LANES) * stride);
    }
    for (; s < splits; s += LANES) a0 += __ldg(p + (size_t)s * stride);
  }
  float acc = (a0 + a1) + (a2 + a3);
  if (LANES > 1) {
    part[w][o] = acc;
    __syncthreads();
    if (w != 0) return;
    acc = 0.f;
#pragma unroll
    for (int i = 0; i < LANES; ++i) acc += part[i][o];
  }
  if (!in_range) return;
  const int n = (int)(idx % N_total);
  const int k = (int)(idx / N_total);
  if (k >= cin * taps) return;  // zero-padded K tail (stem)
  const int tap = k / cin, c = k - tap * cin;
  float* d = dw + ((size_t)n * cin + c) * taps + tap;
  *d = (beta != 0.f) ? beta * (*d) + acc : acc;
}

// Few splits but large outputs (the 512x512x9 layers: 2.4 M elements): the partials are [k = tap*Cin + c][n] with n
// fastest while OIHW wants (c, tap) fastest, so a one-thread-per-output kernel writes 4 bytes at an 18 KB stride.  Here
// a block owns 32 n x 32 c x all taps: coalesced 128-byte reads along n (summing the splits in order), a shared-memory
// tile transposed on the fly, then each n row is written as 32*taps contiguous floats.
template <int TAPS>
__global__ void __launch_bounds__(256)
wgrad_reduce_transpose_kernel(const float* __restrict__ partial, WgDst dws, int splits, int K_total, int N_total,
                              int cin, float beta) {
  constexpr int ROW = 32 * TAPS;
  float* __restrict__ dw = dws.p[blockIdx.z];  // weight group = blockIdx.z
  partial += (size_t)blockIdx.z * splits * K_total * N_total;
  __shared__ float tile[32][ROW + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // tx -> n within the tile, ty -> (tap, c) lane
  const int n0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const size_t stride = (size_t)K_total * N_total;
  for (int i0 = ty; i0 < ROW; i0 += 32) {  // i = tap * 32 + c_local; four partial rows (x splits) in flight per thread
    const float* p[4];
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + 8 * u, tap = i >> 5, cl = i & 31;
      p[u] = partial + ((size_t)tap * cin + c0 + cl) * N_total + n0 + tx;
    }
    for (int sidx = 0; sidx < splits; ++sidx) {
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[u] += __ldg(p[u] + (size_t)sidx * stride);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + 8 * u;
      tile[tx][(i & 31) * TAPS + (i >> 5)] = acc[u];
    }
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {  // one n row per warp iteration: 32 * TAPS contiguous floats of OIHW
    float* d = dw + ((size_t)(n0 + r) * cin + c0) * TAPS;
    for (int j = tx; j < ROW; j += 32) d[j] = (beta != 0.f) ? beta * d[j] + tile[r][j] : tile[r][j];
  }
}

// The split-K reduce kernel launch_wgrad_reduce runs (irfd_conv_wgrad_plan reports it): few splits, one thread per
// output; many splits (1x1 layers, halo kernel: up to 148), 8 lanes share the walk.
enum { kWgRedTranspose9 = 0, kWgRedTranspose1 = 1, kWgRed1 = 2, kWgRed4 = 3, kWgRed8 = 4 };

static int wgrad_reduce_kind(int splits, int K_total, int N_total, int cin, int taps) {
  const size_t total = (size_t)K_total * N_total;
  // the transposing kernel needs whole 32 x 32 tiles and the plain k = tap*cin + c layout (no padded K tail)
  const bool tileable = cin % 32 == 0 && N_total % 32 == 0 && K_total == cin * taps && (taps == 9 || taps == 1);
  if (splits <= 6 && tileable && total >= (size_t)1 << 18) return taps == 9 ? kWgRedTranspose9 : kWgRedTranspose1;
  if (splits <= 6) return kWgRed1;
  return splits <= 24 ? kWgRed4 : kWgRed8;
}

static void launch_wgrad_reduce(const float* partial, const WgDst& dws, int groups, int splits, int K_total, int N_total,
                                int cin, int taps, float beta, cudaStream_t stream) {
  const size_t total = (size_t)K_total * N_total;
  switch (wgrad_reduce_kind(splits, K_total, N_total, cin, taps)) {
    case kWgRedTranspose9:
      wgrad_reduce_transpose_kernel<9><<<dim3(N_total / 32, cin / 32, groups), 256, 0, stream>>>(
          partial, dws, splits, K_total, N_total, cin, beta);
      break;
    case kWgRedTranspose1:
      wgrad_reduce_transpose_kernel<1><<<dim3(N_total / 32, cin / 32, groups), 256, 0, stream>>>(
          partial, dws, splits, K_total, N_total, cin, beta);
      break;
    case kWgRed1:
      wgrad_reduce_kernel<1><<<dim3((unsigned)((total + 255) / 256), groups), 256, 0, stream>>>(
          partial, dws, splits, K_total, N_total, cin, taps, beta);
      break;
    case kWgRed4:
      wgrad_reduce_kernel<4><<<dim3((unsigned)((total + 63) / 64), groups), 256, 0, stream>>>(
          partial, dws, splits, K_total, N_total, cin, taps, beta);
      break;
    default:
      wgrad_reduce_kernel<8><<<dim3((unsigned)((total + 31) / 32), groups), 256, 0, stream>>>(
          partial, dws, splits, K_total, N_total, cin, taps, beta);
  }
}

// ------------------------------------------------------------------------------------------------
// Halo-reuse weight gradient for 3x3 convs (any W that is a multiple of 16).
//
// The per-tap kernel above streams, for every (tap, Cin-chunk) pair, ALL pixels of X again (9x the activation traffic
// through L2 -> SM; measured fabric-bound at ~9 TB/s on the generator's 256^2 layers).  Here a CTA owns one 64-channel
// Cin chunk x one 64-wide Cout tile x a pixel range and keeps all nine taps' accumulators in TMEM (five M=128 MMAs of
// tap pairs = 320 columns): per 128-pixel K block ONE TMA box brings the [TH+2][TW+2] halo of X, and the A operand of
// tap (dy, dx) for the 16 pixels starting at (row r, column s) is that buffer at line (r + dy) * (TW + 2) + s + dx —
// only the MN-major descriptor start moves; the second 64-row atom of each M=128 MMA is the next tap, reached through
// the descriptor's leading-dimension byte offset (128 B for a dx step, (TW + 2 - 2) lines for the dy wrap).
// ------------------------------------------------------------------------------------------------
struct WgHaloArgs {
  int N_total, K_total, cin;
  int chunks, num_n_tiles, splits;
  int num_kb, kb_per_split;  // K blocks of 128 pixels
  int H, W, TH, TW, P;       // image size, pixel block (TH rows x TW columns), halo pitch in lines (TW + 2)
  int hblocks, wsegs;        // H / TH, W / TW
  int spr_shift;             // log2(16-pixel segments per block row)
  int a_tx_bytes;            // (TH + 2) * (TW + 2) * 128
  float* partial;            // [groups][splits][K_total][N_total]
  int groups;                // weight groups stacked along the images (see WgradArgs); num_kb is PER GROUP
};

constexpr int kWhA = 50176;   // halo stage (<= 3 x 130 lines), 1024-aligned
constexpr int kWhB = 16384;   // 128 pixels x 64 output channels
constexpr int kWhStages = 3;
constexpr int kWhSmem = 1024 + kWhStages * (kWhA + kWhB) + 1024;

__global__ void __launch_bounds__(kWgThreads, 1)
wgrad_halo_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_dy,
                  const WgHaloArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kWhStages * (kWhA + kWhB));
  uint64_t* empty_bar = full_bar + kWhStages;
  uint64_t* done_bar = empty_bar + kWhStages;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(done_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  int item = blockIdx.x;
  const int split = item % p.splits;
  item /= p.splits;
  const int n_tile = item % p.num_n_tiles;
  item /= p.num_n_tiles;
  const int chunk = item % p.chunks;
  const int grp = item / p.chunks;
  const int kb_begin = split * p.kb_per_split;
  int kb_end = kb_begin + p.kb_per_split;
  if (kb_end > p.num_kb) kb_end = p.num_kb;
  const int my_kb = kb_end > kb_begin ? kb_end - kb_begin : 0;
  const int kb_off = grp * p.num_kb;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kWhStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(done_bar, 1);
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc<512>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // TMA producer: whole warp converged, one elected lane issues
    if (lane == 0) {
      tma_prefetch_desc(&map_x);
      tma_prefetch_desc(&map_dy);
    }
    __syncwarp();
    int stage = 0;
    uint32_t phase = 0;
    for (int kbl = kb_begin; kbl < kb_end; ++kbl) {
      const int kb = kbl + kb_off;
      const int wseg = kb % p.wsegs;
      const int t = kb / p.wsegs;
      const int hb = t % p.hblocks;
      const int n0 = t / p.hblocks;
      const int h0 = hb * p.TH, w0 = wseg * p.TW;
      const int m0 = (n0 * p.H + h0) * p.W + w0;
      mbar_wait(&empty_bar[stage], phase ^ 1);
      uint8_t* sa = smem + stage * (kWhA + kWhB);
      if (elect_one_sync()) {
        mbar_expect_tx(&full_bar[stage], p.a_tx_bytes + kWhB);
        tma_load_4d(sa, &map_x, &full_bar[stage], chunk * 64, w0 - 1, h0 - 1, n0);
        tma_load_2d(sa + kWhA, &map_dy, &full_bar[stage], n_tile * 64, m0);
      }
      __syncwarp();
      if (++stage == kWhStages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp == 1) {
    // MMA issuer: whole warp converged, one elected lane issues
    constexpr uint32_t idesc = make_idesc_bf16(128, 64, 1, 1);  // both operands MN-major
    // tap pairs (0,1) (2,3) (4,5) (6,7) (8,x): first tap's line offset dy * P + dx, second atom `lbo` lines further
    const uint32_t P = (uint32_t)p.P;
    const uint32_t off[5] = {0u, 2u, P + 1u, 2u * P, 2u * P + 2u};
    const uint32_t lbo[5] = {1u, P - 2u, 1u, 1u, 1u};  // pair 4's second atom is a throw-away duplicate shift
    const uint32_t spr_mask = (1u << p.spr_shift) - 1u;
    int stage = 0;
    uint32_t phase = 0;
    for (int i = 0; i < my_kb; ++i) {
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      const uint32_t a_addr = smem_u32(smem + stage * (kWhA + kWhB));
      const uint64_t bdesc0 = make_smem_desc_sw128(a_addr + kWhA, 8192, 1024);
      uint64_t adesc[5];
#pragma unroll
      for (int q = 0; q < 5; ++q) adesc[q] = make_smem_desc_sw128(a_addr + off[q] * 128u, lbo[q] * 128u, 1024);
      if (elect_one_sync()) {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {  // 16 pixels per MMA
          const uint32_t r = (uint32_t)ks >> p.spr_shift, sg = (uint32_t)ks & spr_mask;
          const uint64_t a_step = (uint64_t)((r * P + sg * 16u) * 8u);  // lines -> 16-byte address units
#pragma unroll
          for (int q = 0; q < 5; ++q)
            umma_bf16(tmem_base + q * 64, adesc[q] + a_step, bdesc0 + 128 * ks, idesc, (i | ks) != 0 ? 1u : 0u);
        }
        umma_commit(&empty_bar[stage]);
      }
      __syncwarp();
      if (++stage == kWhStages) {
        stage = 0;
        phase ^= 1;
      }
    }
    if (elect_one_sync()) umma_commit(done_bar);
    __syncwarp();
  } else {
    // epilogue: 4 warps; TMEM lane = (tap parity within the pair) * 64 + input channel
    const int q4 = warp & 3;
    const int ci = (q4 & 1) * 32 + lane;
    if (my_kb > 0) {
      mbar_wait(done_bar, 0);
      tc_fence_after();
    }
#pragma unroll 1
    for (int pr = 0; pr < 5; ++pr) {
      const int tap = 2 * pr + (q4 >> 1);
      const size_t krow = (size_t)tap * p.cin + (size_t)chunk * 64 + ci;
      float* dst = p.partial + (((size_t)grp * p.splits + split) * p.K_total + krow) * p.N_total + (size_t)n_tile * 64;
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
        uint32_t v[32];
        if (my_kb > 0) {
          tmem_ld32(tmem_base + (uint32_t(q4 * 32) << 16) + pr * 64 + half * 32, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int t = 0; t < 32; ++t) v[t] = 0u;
        }
        if (tap < 9) {
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            float4 o = make_float4(__uint_as_float(v[4 * t]), __uint_as_float(v[4 * t + 1]),
                                   __uint_as_float(v[4 * t + 2]), __uint_as_float(v[4 * t + 3]));
            *reinterpret_cast<float4*>(dst + half * 32 + 4 * t) = o;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem_base);
}

// Geometry of the halo wgrad for a [n, h, w] image batch; false when the shape is not eligible.
// Split count for `groups` weight groups sharing one launch: the CTAs of all groups must fit ONE wave when possible;
// otherwise pick the count whose (waves x k-blocks per split) is smallest (a few CTAs spilling into a second wave
// double the kernel time), smaller counts winning ties (fewer fp32 partials).
static int grouped_splits(int base_per_group, int groups, int num_kb, int max_splits) {
  const int sms = num_sms();
  if (max_splits < 1) max_splits = 1;
  int fit = sms / (base_per_group * groups);
  if (fit >= 1) return fit < max_splits ? fit : max_splits;
  int best = 1;
  long long best_cost = -1;
  for (int s = 1; s <= max_splits && s <= 8; ++s) {
    const long long ctas = (long long)base_per_group * groups * s;
    const long long waves = (ctas + sms - 1) / sms;
    const long long cost = waves * ((num_kb + s - 1) / s) * 16 + s;  // + s: partial traffic breaks ties
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = s;
    }
  }
  return best;
}

// n = images PER GROUP
static bool wgrad_halo_plan(int n, int h, int w, int cin, int cout, int ksize, WgHaloArgs* a, int groups = 1) {
  const char* e = getenv("IRFD_WGRAD_HALO");
  if (e && atoi(e) == 0) return false;
  if (ksize != 3 || w < 16 || w % 16 != 0 || cin % 64 != 0 || cout % 64 != 0) return false;
  // Measured on B200 (scripts/exp_wgrad_halo.py): 2.6x faster on the 256^2 layers with Cout 64, 1.4x at 128^2 / Cout
  // 128 and on the encoder's 64^2 stage; with Cout >= 256 or narrow images the per-tap kernel's 256-wide tile wins.
  // IRFD_WGRAD_HALO=2 forces the halo kernel on every eligible shape (tests).
  if (!(e && atoi(e) == 2) && (cout > 128 || w < 64)) return false;
  int TW, TH;
  if (w >= 128) {
    if (w % 128 != 0) return false;
    TW = 128;
    TH = 1;
  } else {
    if (128 % w != 0 || h % (128 / w) != 0) return false;
    TW = w;
    TH = 128 / w;
  }
  a->N_total = cout;
  a->K_total = 9 * cin;
  a->cin = cin;
  a->chunks = cin / 64;
  a->num_n_tiles = cout / 64;
  a->H = h; a->W = w; a->TH = TH; a->TW = TW; a->P = TW + 2;
  a->hblocks = h / TH;
  a->wsegs = w / TW;
  a->num_kb = n * a->hblocks * a->wsegs;
  int spr = TW / 16, sh = 0;
  while ((1 << sh) < spr) ++sh;
  a->spr_shift = sh;
  a->a_tx_bytes = (TH + 2) * (TW + 2) * 128;
  a->groups = groups;
  const int base = a->chunks * a->num_n_tiles;
  int splits;
  if (groups == 1) {
    splits = num_sms() / base;  // one CTA per SM is resident: the launch must fit one wave
    if (splits > a->num_kb) splits = a->num_kb;
    if (splits < 1) splits = 1;
  } else {
    splits = grouped_splits(base, groups, a->num_kb, a->num_kb);
  }
  a->kb_per_split = (a->num_kb + splits - 1) / splits;
  a->splits = (a->num_kb + a->kb_per_split - 1) / a->kb_per_split;
  return true;
}

template <int BLOCK_N>
static int launch_wgrad(const CUtensorMap& mx, const CUtensorMap& mdy, const WgradArgs& a, int grid, cudaStream_t stream) {
  using Cfg = WgCfg<BLOCK_N>;
  static bool configured = false;
  auto kern = wgrad_gemm_kernel<BLOCK_N>;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_last_error("cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return IRFD_ERR_CUDA;
    }
    configured = true;
  }
  kern<<<grid, kWgThreads, Cfg::SMEM_BYTES, stream>>>(mx, mdy, a);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

// n = images PER GROUP
static void wgrad_plan(int n, int h, int w, int cin, int cout, int ksize, WgradArgs* a, int* block_n, int groups = 1) {
  const long long m_total = (long long)n * h * w;
  a->groups = groups;
  a->x_shared = 0;
  a->M_total = (int)m_total;
  a->N_total = cout;
  a->taps = ksize * ksize;
  a->kw = ksize;
  a->pad = ksize / 2;
  a->cin_chunks = cin / 64;
  a->K_total = a->taps * cin;
  a->num_atoms = a->taps * a->cin_chunks;
  a->num_pairs = (a->num_atoms + 1) / 2;
  *block_n = cout % 256 == 0 ? 256 : (cout % 128 == 0 ? 128 : 64);
  a->num_n_tiles = cout / *block_n;
  a->num_kb = (int)((m_total + 63) / 64);
  // One CTA per SM is resident (200 KB of pipeline stages), so the launch must fit ONE wave: rounding the split count
  // up left a second wave of a handful of CTAs (e.g. 153 = 148 + 5) that doubled the kernel time.
  const int base = a->num_pairs * a->num_n_tiles;
  const int max_splits = (a->num_kb + kWgMinKb - 1) / kWgMinKb;  // at least kWgMinKb k-blocks (64 pixels each) per split
  int splits;
  if (groups == 1) {
    splits = (kWgWaves * num_sms()) / base;
    if (splits > max_splits) splits = max_splits;
    if (splits < 1) splits = 1;
  } else {
    splits = grouped_splits(base, groups, a->num_kb, max_splits);
  }
  a->kb_per_split = (a->num_kb + splits - 1) / splits;
  a->splits = (a->num_kb + a->kb_per_split - 1) / a->kb_per_split;
}

}  // namespace irfd

using namespace irfd;

static long long wgrad_ws_bytes(int n_g, int h, int w, int cin, int cout, int ksize, int groups) {
  WgHaloArgs ha;
  if (wgrad_halo_plan(n_g, h, w, cin, cout, ksize, &ha, groups))
    return (long long)groups * ha.splits * ha.K_total * ha.N_total * 4;
  WgradArgs a;
  int bn;
  wgrad_plan(n_g, h, w, cin, cout, ksize, &a, &bn, groups);
  return (long long)groups * a.splits * a.K_total * a.N_total * 4;
}

extern "C" long long irfd_wgrad_workspace_bytes(int n, int h, int w, int cin, int cout, int ksize) {
  return wgrad_ws_bytes(n, h, w, cin, cout, ksize, 1);
}

// n = TOTAL images (all groups); with x_shared, n/h/w describe dY's stacked rows and x holds one group's rows
extern "C" long long irfd_wgrad_workspace_bytes_grouped(int n, int h, int w, int cin, int cout, int ksize, int groups) {
  if (groups < 1 || groups > kMaxWgGroups) return -1;
  if (n % groups == 0) return wgrad_ws_bytes(n / groups, h, w, cin, cout, ksize, groups);
  return wgrad_ws_bytes(1, 1, (int)(((long long)n * h * w) / groups), cin, cout, ksize, groups);  // 2-D row matrices
}

// Which kernels a weight-gradient call launches (halo or per-tap GEMM, then one split-K reduce): the one place the
// selection lives (conv_wgrad_impl launches what it says; irfd_conv_wgrad_plan exports it).  n, h, w: ONE group.
struct WgradSel {
  bool halo;
  WgHaloArgs ha;  // halo
  WgradArgs a;    // per-tap
  int block_n, splits, kb_per_split, num_kb, grid;
  int red_cin, red_taps, reduce_kind;
};

static int wgrad_select(int n, int h, int w, int cin, int cout, int ksize, int groups, int x_shared, int reduce_cin,
                        int reduce_taps, WgradSel* s) {
  IRFD_CHECK_ARG(ksize == 1 || ksize == 3, "conv_wgrad: ksize must be 1 or 3");
  IRFD_CHECK_ARG(cin % 64 == 0 && cout % 64 == 0, "conv_wgrad: channels must be multiples of 64");
  IRFD_CHECK_ARG(!x_shared || ksize == 1, "conv_wgrad: a shared x operand needs ksize 1");
  const long long m_group = (long long)n * h * w;
  IRFD_CHECK_ARG(groups == 1 || m_group % 128 == 0, "conv_wgrad: grouped launches need 128-pixel multiples per group");
  s->halo = !x_shared && wgrad_halo_plan(n, h, w, cin, cout, ksize, &s->ha, groups);
  int K_total, N_total, taps;
  if (s->halo) {
    s->block_n = 64;
    s->splits = s->ha.splits;
    s->kb_per_split = s->ha.kb_per_split;
    s->num_kb = s->ha.num_kb;
    s->grid = groups * s->ha.chunks * s->ha.num_n_tiles * s->ha.splits;
    K_total = s->ha.K_total;
    N_total = s->ha.N_total;
    taps = 9;
  } else {
    wgrad_plan(n, h, w, cin, cout, ksize, &s->a, &s->block_n, groups);
    s->a.x_shared = x_shared;
    s->splits = s->a.splits;
    s->kb_per_split = s->a.kb_per_split;
    s->num_kb = s->a.num_kb;
    s->grid = groups * s->a.num_pairs * s->a.num_n_tiles * s->a.splits;
    K_total = s->a.K_total;
    N_total = s->a.N_total;
    taps = s->a.taps;
  }
  s->red_cin = reduce_cin > 0 ? reduce_cin : cin;
  s->red_taps = reduce_cin > 0 ? reduce_taps : taps;
  s->reduce_kind = wgrad_reduce_kind(s->splits, K_total, N_total, s->red_cin, s->red_taps);
  return IRFD_OK;
}

static int conv_wgrad_impl(const void* x, const void* dy, int n, int h, int w, int cin, int cout, int ksize,
                           const WgDst& dws, int groups, int x_shared, float beta, int reduce_cin, int reduce_taps,
                           void* workspace, long long workspace_bytes, cudaStream_t stream) {
  // n, h, w: geometry of ONE group
  IRFD_CHECK_ARG(x && dy && workspace, "conv_wgrad: null pointer");
  WgradSel sel;
  {
    const int rc = wgrad_select(n, h, w, cin, cout, ksize, groups, x_shared, reduce_cin, reduce_taps, &sel);
    if (rc != IRFD_OK) return rc;
  }
  const long long m_group = (long long)n * h * w;
  if (sel.halo) {
    WgHaloArgs& ha = sel.ha;
    IRFD_CHECK_ARG(workspace_bytes >= (long long)groups * ha.splits * ha.K_total * ha.N_total * 4,
                   "conv_wgrad: workspace too small");
    ha.partial = reinterpret_cast<float*>(workspace);
    CUtensorMap mx, mdy;
    {
      const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)w, (uint64_t)h, (uint64_t)n * groups};
      const uint64_t str[3] = {(uint64_t)cin * 2, (uint64_t)w * cin * 2, (uint64_t)h * w * cin * 2};
      const uint32_t box[4] = {64, (uint32_t)(ha.TW + 2), (uint32_t)(ha.TH + 2), 1};
      int rc = make_tmap_bf16(&mx, x, 4, dims, str, box, true);
      if (rc) return rc;
    }
    {
      const uint64_t dims[2] = {(uint64_t)cout, (uint64_t)(m_group * groups)};
      const uint64_t str[1] = {(uint64_t)cout * 2};
      const uint32_t box[2] = {64, 128};
      int rc = make_tmap_bf16(&mdy, dy, 2, dims, str, box, true);
      if (rc) return rc;
    }
    static bool configured = false;
    if (!configured) {
      cudaError_t e = cudaFuncSetAttribute(wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWhSmem);
      if (e != cudaSuccess) {
        set_last_error("cudaFuncSetAttribute(wgrad halo smem=%d): %s", kWhSmem, cudaGetErrorString(e));
        return IRFD_ERR_CUDA;
      }
      configured = true;
    }
    wgrad_halo_kernel<<<sel.grid, kWgThreads, kWhSmem, stream>>>(mx, mdy, ha);
    IRFD_CHECK_LAUNCH();
    launch_wgrad_reduce(ha.partial, dws, groups, ha.splits, ha.K_total, ha.N_total, sel.red_cin, sel.red_taps, beta,
                        stream);
    IRFD_CHECK_LAUNCH();
    return IRFD_OK;
  }
  WgradArgs& a = sel.a;
  const int block_n = sel.block_n;
  IRFD_CHECK_ARG(workspace_bytes >= (long long)groups * a.splits * a.K_total * a.N_total * 4,
                 "conv_wgrad: workspace too small");
  a.partial = reinterpret_cast<float*>(workspace);

  const int xg = x_shared ? 1 : groups;  // groups stacked in x
  int H = h, W = w, NB = n * xg;
  if (ksize == 1) {
    H = 1; W = (int)(m_group * xg); NB = 1;
  }
  int tw, th, tn;
  if (W >= 64) {
    IRFD_CHECK_ARG(ksize == 1 || W % 64 == 0, "conv_wgrad: W=%d must be a multiple of 64", W);
    tw = 64; th = 1; tn = 1;
  } else {
    IRFD_CHECK_ARG(64 % W == 0, "conv_wgrad: W=%d must divide 64", W);
    tw = W;
    const int rows = 64 / W;
    if (H >= rows) {
      IRFD_CHECK_ARG(H % rows == 0, "conv_wgrad: H=%d must be a multiple of %d", H, rows);
      th = rows; tn = 1;
    } else {
      IRFD_CHECK_ARG(rows % H == 0, "conv_wgrad: H=%d must divide %d", H, rows);
      th = H; tn = rows / H;
    }
  }
  a.H = H; a.W = W;

  CUtensorMap mx, mdy;
  {
    const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)W, (uint64_t)H, (uint64_t)NB};
    const uint64_t str[3] = {(uint64_t)cin * 2, (uint64_t)W * cin * 2, (uint64_t)H * W * cin * 2};
    const uint32_t box[4] = {64, (uint32_t)tw, (uint32_t)th, (uint32_t)tn};
    int rc = make_tmap_bf16(&mx, x, 4, dims, str, box, true);
    if (rc) return rc;
  }
  {
    const uint64_t dims[2] = {(uint64_t)cout, (uint64_t)(m_group * groups)};
    const uint64_t str[1] = {(uint64_t)cout * 2};
    const uint32_t box[2] = {64, 64};
    int rc = make_tmap_bf16(&mdy, dy, 2, dims, str, box, true);
    if (rc) return rc;
  }
  int rc;
  switch (block_n) {
    case 64: rc = launch_wgrad<64>(mx, mdy, a, sel.grid, stream); break;
    case 128: rc = launch_wgrad<128>(mx, mdy, a, sel.grid, stream); break;
    default: rc = launch_wgrad<256>(mx, mdy, a, sel.grid, stream); break;
  }
  if (rc) return rc;
  launch_wgrad_reduce(a.partial, dws, groups, a.splits, a.K_total, a.N_total, sel.red_cin, sel.red_taps, beta, stream);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_conv_wgrad(const void* x, const void* dy, int n, int h, int w, int cin, int cout, int ksize,
                               float* dw, float beta, int reduce_cin, int reduce_taps, void* workspace,
                               long long workspace_bytes, cudaStream_t stream) {
  IRFD_CHECK_ARG(dw != nullptr, "conv_wgrad: null pointer");
  WgDst dws;
  for (int i = 0; i < kMaxWgGroups; ++i) dws.p[i] = i == 0 ? dw : nullptr;
  return conv_wgrad_impl(x, dy, n, h, w, cin, cout, ksize, dws, 1, 0, beta, reduce_cin, reduce_taps, workspace,
                         workspace_bytes, stream);
}

// `groups` weight gradients in one launch pair: x [n, h, w, cin] and dy [n, h, w, cout] stack the groups' images
// group-major (n = TOTAL images, n % groups == 0; 2-D row matrices pass n = 1, h = 1, w = total rows); dw is a HOST
// array of `groups` device pointers (one OIHW fp32 gradient each).  x_shared != 0 (ksize 1): x holds ONE group's rows,
// read by every group (the stem's im2col matrix); n/h/w then describe dy.
// n, h, w of a grouped call (TOTAL images, or a 2-D row matrix [1, 1, rows]) -> the geometry of one group
static int wgrad_group_shape(int n, int h, int w, int groups, int* ng, int* hg, int* wg) {
  *ng = n; *hg = h; *wg = w;
  if (n % groups == 0) {
    *ng = n / groups;
  } else {  // 2-D row matrix [1, 1, rows, K]
    IRFD_CHECK_ARG(n == 1 && h == 1 && w % groups == 0, "conv_wgrad_grouped: rows do not split into groups");
    *wg = w / groups;
  }
  return IRFD_OK;
}

extern "C" int irfd_conv_wgrad_grouped(const void* x, const void* dy, int n, int h, int w, int cin, int cout, int ksize,
                                       float* const* dw, float beta, int reduce_cin, int reduce_taps, int groups,
                                       int x_shared, void* workspace, long long workspace_bytes, cudaStream_t stream) {
  IRFD_CHECK_ARG(dw != nullptr && groups >= 1 && groups <= kMaxWgGroups, "conv_wgrad_grouped: 1..4 groups");
  WgDst dws;
  for (int i = 0; i < kMaxWgGroups; ++i) dws.p[i] = i < groups ? dw[i] : nullptr;
  for (int i = 0; i < groups; ++i) IRFD_CHECK_ARG(dws.p[i] != nullptr, "conv_wgrad_grouped: null gradient pointer");
  int ng, hg, wg;
  const int rc = wgrad_group_shape(n, h, w, groups, &ng, &hg, &wg);
  if (rc != IRFD_OK) return rc;
  return conv_wgrad_impl(x, dy, ng, hg, wg, cin, cout, ksize, dws, groups, x_shared, beta, reduce_cin, reduce_taps,
                         workspace, workspace_bytes, stream);
}

// Host-only query of the kernels irfd_conv_wgrad_grouped launches for these arguments (groups = 1: irfd_conv_wgrad).
extern "C" int irfd_conv_wgrad_plan(int n, int h, int w, int cin, int cout, int ksize, int groups, int x_shared,
                                    int reduce_cin, int reduce_taps, int* out_host) {
  IRFD_CHECK_ARG(out_host != nullptr, "conv_wgrad_plan: null output");
  IRFD_CHECK_ARG(groups >= 1 && groups <= kMaxWgGroups, "conv_wgrad_plan: 1..4 groups");
  int ng, hg, wg;
  int rc = wgrad_group_shape(n, h, w, groups, &ng, &hg, &wg);
  if (rc != IRFD_OK) return rc;
  WgradSel sel;
  rc = wgrad_select(ng, hg, wg, cin, cout, ksize, groups, x_shared, reduce_cin, reduce_taps, &sel);
  if (rc != IRFD_OK) return rc;
  const int v[7] = {sel.halo ? 1 : 0, sel.block_n, sel.splits, sel.kb_per_split, sel.num_kb, sel.grid, sel.reduce_kind};
  for (int i = 0; i < 7; ++i) out_host[i] = v[i];
  return IRFD_OK;
}
