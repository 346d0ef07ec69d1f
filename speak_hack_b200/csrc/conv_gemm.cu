// Implicit-GEMM convolution (fprop and dgrad) on tcgen05 tensor cores.
//
//   Y[m, n] = sum_{tap, c} X[pixel(m) + shift(tap), c] * Wk[n, tap, c]        m = linear NHWC pixel, n = out channel
//
// * Operands are bf16, accumulation is fp32 in TMEM (double-buffered: 2 x BLOCK_N columns).
// * A tiles (128 pixels x 64 channels) arrive by 4-D TMA boxes over the NHWC tensor; the conv halo/padding is the
//   TMA out-of-bounds zero fill, so there is no im2col buffer and no boundary code.
// * B tiles (BLOCK_N out-channels x 64 k) arrive by 2-D TMA boxes over the packed [Cout][tap][Cin] weight.
// * Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer, warps 2..9 = epilogue
//   (TMEM -> registers -> fused math -> swizzled smem staging -> TMA store).  Producer and issuer run their loops
//   warp-converged and put only the TMA / MMA / commit instruction under elect.sync (see ptx.cuh: elect_one_sync).
// * Persistent: grid = #SMs, each CTA walks tiles  tile = blockIdx.x + i * gridDim.x  (n-tile fastest, so the CTAs
//   running concurrently share A tiles in L2).
// * conv_halo_kernel (further down) is the variant for 3x3 convs on rows of >= 128 pixels: one halo tile per
//   64-channel chunk serves all nine taps.
// * Shapes whose 128 consecutive pixels are not one TMA box (3x3 at 56^2, 28^2, 14^2, 7^2, odd sizes) run the
//   box-tiled instances (conv_gemm_kernel<..., BOX = true>, PLAIN / AFFINE): a tile is a box of <= 128 pixels.
//
// Epilogue modes
//   PLAIN : y = acc (+ bias[n])                                       -> bf16           (dgrad, 1x1, generic)
//   STATS : y = acc -> bf16, plus per-tile per-channel sum / sum-of-squares of the stored values (train-mode BN)
//   AFFINE: y = act( acc*scale[n] + shift[n] [+ res[m,n]] ) -> bf16, act = none / ReLU / leaky ReLU(0.2)
//           (inference: eval-mode BatchNorm, ReLU and the residual add of a Bottleneck folded into the conv,
//           torchvision/models/resnet.py:143-164; discriminator: conv + bias + leaky_relu, styleganv1.py:662-694)
//   STYLE : z = acc + bias[n] + nw[n]*noise[m];  a = lrelu_0.2(z);  y = a*sp1[b,n] + s1[b,n]
//           -> a (bf16, kept for backward) and y (bf16, next layer's input)
//           reference: styleganv1.py:625-628 / 630-633 (conv -> ApplyNoise -> leaky_relu -> ApplyStyle)
#include <stdlib.h>

#include "host_util.h"
#include "ptx.cuh"

namespace irfd {

enum { EPI_PLAIN = 0, EPI_STATS = 1, EPI_STYLE = 2, EPI_AFFINE = 3, EPI_BNBWD = 4, EPI_BNBWD_RES = 5 };

struct ConvGemmArgs {
  int M_total, N_total;
  int num_m_tiles, num_n_tiles;
  int taps, kw, pad, cin_chunks;
  int H, W, HW, B;
  const float* bias;
  const float* nw;
  const float* noise;
  const float* sp1;
  const float* s1;
  float* stat_sum;
  float* stat_sq;
  const __nv_bfloat16* res;  // AFFINE: optional residual [M_total][N_total]
  __nv_bfloat16* y_lo;       // STYLE: optional second half of a split-bf16 y (y ~= y + y_lo), direct 16-byte stores
  // Weight groups (the three ResNet-50 encoders run as ONE launch per layer, model.py:84-90): the pixel tiles are
  // stacked group-major, m tile t belongs to group t / wg_tiles and multiplies rows [grp * N_total, ...) of the
  // stacked weight matrix; per-channel epilogue vectors (AFFINE scale/shift, PLAIN bias) are [groups][N_total].
  // a_mod_tiles > 0: every group reads the SAME A operand (the stem's shared im2col matrix): A tile = t % a_mod_tiles.
  int wg_tiles;
  int a_mod_tiles;
  int relu;                  // AFFINE: 0 = none, 1 = ReLU, 2 = leaky ReLU (slope 0.2)
  // BNBWD: this GEMM is the data gradient of a conv whose INPUT was relu(BN(z)) (torchvision resnet.py:146-152).  Its
  // epilogue applies the ReLU mask (recomputed from z) to the activation gradient it produces and sums, per channel
  // and 128-pixel tile, g and g * xhat — the reduce pass of that BatchNorm's backward, which then needs no launch and
  // no second read of the gradient.  stat_sum receives the partials as [m tile][2][N_total].
  // BNBWD_RES: the same for the BatchNorm that closes a Bottleneck (out = relu(bn3(z) + identity), resnet.py:154-161),
  // whose output gradient is this GEMM's result (the next block's conv1 data gradient) PLUS that block's shortcut
  // gradient bn_g2; the ReLU mask comes from the bit plane irfd_bn_apply_sets wrote (bn_bits, [M_total][N_total/8]).
  const __nv_bfloat16* bn_z;  // [M_total][N_total]
  const __nv_bfloat16* bn_g2;
  const uint8_t* bn_bits;
  const float* bn_mean;       // [statistic groups][N_total]
  const float* bn_rstd;
  const float* bn_gamma[4];   // per weight group
  const float* bn_beta[4];
  int sg_tiles;               // m tiles per statistic group
  int warp_epi;               // non-STYLE modes of conv_gemm_kernel: per-warp epilogue (epilogue_tile_warp)
  // Box-tiled geometry (conv_gemm_kernel<..., BOX = true>): m tile t is the TMA box of box_tw x box_th x box_tn output
  // pixels at column tile t % box_tiles_w, row tile (t / box_tiles_w) % box_tiles_h, image tile t / (tiles_w * tiles_h)
  // (see irfd_conv_gemm_geometry).  Unused by the linear geometry.
  int box_tw, box_th, box_tn, box_tiles_w, box_tiles_h;
};

constexpr int kNumThreads = 320;      // 10 warps
constexpr int kEpiThreads = 256;      // warps 2..9
constexpr int kMiscBytes = 12 * 1024; // vectors / reduction scratch / barriers
constexpr int kStgBytes = 16384;      // one 128 x 64 bf16 staging tile
constexpr int kSmemLimit = 232448;    // 227 KB

template <int BLOCK_N, int MODE>
struct GemmCfg {
  static constexpr int A_BYTES = 128 * 128;
  static constexpr int B_BYTES = BLOCK_N * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int NUM_OUT = (MODE == EPI_STYLE) ? 2 : 1;
  static constexpr int STG_TOTAL = 4 * kStgBytes;  // STYLE: 2 outputs x 2 tiles; other modes: 8 warps x 2 slabs of 4 KB
  static constexpr int RAW_STAGES = (kSmemLimit - 1024 - STG_TOTAL - kMiscBytes) / STAGE_BYTES;
  static constexpr int STAGES = RAW_STAGES > 8 ? 8 : RAW_STAGES;
  static constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + STG_TOTAL + kMiscBytes;
  static constexpr uint32_t TMEM_COLS = (2 * BLOCK_N <= 128) ? 128 : (2 * BLOCK_N <= 256 ? 256 : 512);
};

// Box-tiled geometry: first output pixel (column, row, image) of m tile `m_tile`.
__device__ __forceinline__ void box_origin(const ConvGemmArgs& p, int m_tile, int& w0, int& h0, int& n0) {
  const int t = m_tile / p.box_tiles_w;
  w0 = (m_tile - t * p.box_tiles_w) * p.box_tw;
  h0 = (t % p.box_tiles_h) * p.box_th;
  n0 = (t / p.box_tiles_h) * p.box_tn;
}

// Box-tiled geometry: flat NHWC pixel of row r of the tile whose origin is (w0, h0, n0), or -1 when the row lies past
// the box (r >= tw * th * tn: stale A rows) or outside the tensor (a partial last tile, which the TMA store clips).
__device__ __forceinline__ int box_pixel(const ConvGemmArgs& p, int w0, int h0, int n0, int r) {
  const int wi = r % p.box_tw;
  const int t = r / p.box_tw;
  const int hi = t % p.box_th;
  const int ni = t / p.box_th;
  const int w = w0 + wi, h = h0 + hi, n = n0 + ni;
  if (ni >= p.box_tn || w >= p.W || h >= p.H || n >= p.B) return -1;
  return (n * p.H + h) * p.W + w;
}

// ------------------------------------------------------------------------------------------------
// Epilogue of ONE 128-row accumulator (TMEM columns [acc_col, acc_col + BLOCK_N)) whose first output row is the flat
// pixel m0: TMEM -> registers -> fused math -> swizzled smem staging -> TMA store (+ STATS partials).
// Called by the 8 epilogue warps (threads 64..319).  NBUF = staging buffers per output (1 or 2).
// `release_bar`: arrived on (one lane per warp) as soon as the accumulator has been drained into registers.
// BOX (PLAIN / AFFINE only): m0 = m tile * 128 of the box-tiled geometry; the first tw*th*tn staging rows are the box in
// TMA order and go out as ONE 4-D store box (map_out is the 4-D [N][H][W][Cout] map), which clips rows outside the
// tensor; the residual is read at each row's own pixel.
// ------------------------------------------------------------------------------------------------
template <int BLOCK_N, int MODE, int NBUF, bool BOX = false>
__device__ __forceinline__ void epilogue_acc(const ConvGemmArgs& p, const CUtensorMap* map_out,
                                             const CUtensorMap* map_out2, uint32_t tmem_base, uint32_t acc_col,
                                             int m0, int n_tile, uint64_t* release_bar, uint8_t* stg_base, float* vec,
                                             uint32_t& chunk_counter) {
  static_assert(!BOX || MODE == EPI_PLAIN || MODE == EPI_AFFINE, "the box-tiled geometry serves PLAIN / AFFINE only");
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int e = warp - 2;
  const int q = warp & 3;       // TMEM lane quarter this warp may touch
  const int half = e >> 2;      // which 32-column half of each 64-column chunk
  const int etid = threadIdx.x - 64;
  const int r = q * 32 + lane;  // tile row == TMEM lane
  float* vb = vec;              // [256] bias
  float* vnw = vec + 256;       // [256] noise weight
  float* vsp1 = vec + 512;      // [2][256]
  float* vs1 = vec + 1024;      // [2][256]
  const int m_tile = m0 >> 7;
  const int ng0 = n_tile * BLOCK_N;
  const int pg0 = (m_tile / p.wg_tiles) * p.N_total + ng0;  // first channel of this tile in the per-group vectors
  float noise_r = 0.f;
  int img_local = 0;
  int bw0 = 0, bh0 = 0, bn0 = 0, box_row = -1;  // BOX: tile origin and this thread's output pixel
  if constexpr (BOX) {
    box_origin(p, m_tile, bw0, bh0, bn0);
    box_row = box_pixel(p, bw0, bh0, bn0, r);
  }
  if constexpr (MODE == EPI_STYLE) {
    const int nimg = p.HW < 128 ? 128 / p.HW : 1;
    const int b0 = m0 / p.HW;
    // (the last barrier of the previous accumulator's chunk loop already separates its vector reads from these writes)
    for (int i = etid; i < BLOCK_N; i += kEpiThreads) {
      vb[i] = p.bias[ng0 + i];
      vnw[i] = p.nw[ng0 + i];
    }
    for (int i = etid; i < nimg * BLOCK_N; i += kEpiThreads) {
      const int img = i / BLOCK_N, c = i - img * BLOCK_N;
      int bb = b0 + img;
      if (bb >= p.B) bb = p.B - 1;
      vsp1[img * 256 + c] = p.sp1[(size_t)bb * p.N_total + ng0 + c];
      vs1[img * 256 + c] = p.s1[(size_t)bb * p.N_total + ng0 + c];
    }
    named_bar_sync(1, kEpiThreads);
    if (m0 + r < p.M_total) noise_r = p.noise[m0 + r];
    img_local = p.HW < 128 ? r / p.HW : 0;
  } else if constexpr (MODE == EPI_PLAIN) {
    if (p.bias != nullptr) {
      for (int i = etid; i < BLOCK_N; i += kEpiThreads) vb[i] = p.bias[pg0 + i];
      named_bar_sync(1, kEpiThreads);
    }
  } else if constexpr (MODE == EPI_AFFINE) {
    for (int i = etid; i < BLOCK_N; i += kEpiThreads) {
      vb[i] = p.bias[pg0 + i];   // shift
      vnw[i] = p.nw[pg0 + i];    // scale
    }
    named_bar_sync(1, kEpiThreads);
  }
#pragma unroll 1
  for (int chunk = 0; chunk < BLOCK_N / 64; ++chunk, ++chunk_counter) {
    uint32_t v[32];
    uint32_t zw[16];  // BNBWD: this thread's 16 rows x 2 channels of z for the column phase, in flight during the drain
    uint32_t gw[16];  // BNBWD_RES: the shortcut gradient, same cells
    uint8_t bw[16];   // BNBWD_RES: the mask byte of the 8 channels around this thread's pair
    if constexpr (MODE == EPI_BNBWD || MODE == EPI_BNBWD_RES) {
      const size_t cell0 = (size_t)(m0 + (etid >> 5) * 16) * p.N_total + ng0 + chunk * 64 + 2 * (etid & 31);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        zw[i] = __ldg(reinterpret_cast<const uint32_t*>(p.bn_z + cell0 + (size_t)i * p.N_total));
        if constexpr (MODE == EPI_BNBWD_RES) {
          gw[i] = __ldg(reinterpret_cast<const uint32_t*>(p.bn_g2 + cell0 + (size_t)i * p.N_total));
          bw[i] = __ldg(p.bn_bits + ((cell0 + (size_t)i * p.N_total) >> 3));
        }
      }
    }
    const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + acc_col + chunk * 64 + half * 32;
    tmem_ld32(taddr, v);
    tmem_ld_wait();
    if (chunk == BLOCK_N / 64 - 1 && release_bar != nullptr) {
      // accumulator fully drained into registers: hand the TMEM buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(release_bar);
    }
    const int buf = (NBUF == 2) ? (chunk_counter & 1) : 0;
    uint8_t* stg0 = stg_base + buf * kStgBytes;
    uint8_t* stg1 = stg_base + (NBUF + buf) * kStgBytes;
    // staging buffer `buf` was last used NBUF chunks ago: make sure its TMA store has drained it
    if (warp == 2) {  // store leader: the elected lane of warp 2 (elect.sync is deterministic for a full mask)
      __syncwarp();
      if (elect_one_sync()) tma_store_wait_read<NBUF - 1>();
    }
    named_bar_sync(1, kEpiThreads);
    const int cbase = chunk * 64 + half * 32;  // column within the BLOCK_N tile
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      float o[8], o2[8];
      float rres[8];
      if constexpr (MODE == EPI_AFFINE) {
        if (p.res != nullptr && (BOX ? box_row >= 0 : m0 + r < p.M_total)) {
          const uint4 u = *reinterpret_cast<const uint4*>(p.res + (size_t)(BOX ? box_row : m0 + r) * p.N_total + ng0 +
                                                          cbase + jj * 8);
          const float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
          rres[0] = a0.x; rres[1] = a0.y; rres[2] = a1.x; rres[3] = a1.y;
          rres[4] = a2.x; rres[5] = a2.y; rres[6] = a3.x; rres[7] = a3.y;
        } else {
#pragma unroll
          for (int t = 0; t < 8; ++t) rres[t] = 0.f;
        }
      }
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int c = cbase + jj * 8 + t;
        float acc = __uint_as_float(v[jj * 8 + t]);
        if constexpr (MODE == EPI_STYLE) {
          float z = acc + vb[c] + vnw[c] * noise_r;
          float a = z > 0.f ? z : 0.2f * z;
          o[t] = a;
          o2[t] = a * vsp1[img_local * 256 + c] + vs1[img_local * 256 + c];
        } else if constexpr (MODE == EPI_PLAIN) {
          o[t] = (p.bias != nullptr) ? acc + vb[c] : acc;
        } else if constexpr (MODE == EPI_AFFINE) {
          const float y = acc * vnw[c] + vb[c] + rres[t];
          o[t] = p.relu == 1 ? fmaxf(y, 0.f) : (p.relu == 2 ? (y > 0.f ? y : 0.2f * y) : y);
        } else {
          o[t] = acc;
        }
      }
      const int j = half * 4 + jj;  // 16-byte chunk index inside the 128-byte staging row
      const int phys = j ^ (r & 7);
      uint4 pk;
      pk.x = pack_bf16x2(o[0], o[1]);
      pk.y = pack_bf16x2(o[2], o[3]);
      pk.z = pack_bf16x2(o[4], o[5]);
      pk.w = pack_bf16x2(o[6], o[7]);
      *reinterpret_cast<uint4*>(stg0 + r * 128 + phys * 16) = pk;
      if constexpr (MODE == EPI_STYLE) {
        uint4 pk2;
        pk2.x = pack_bf16x2(o2[0], o2[1]);
        pk2.y = pack_bf16x2(o2[2], o2[3]);
        pk2.z = pack_bf16x2(o2[4], o2[5]);
        pk2.w = pack_bf16x2(o2[6], o2[7]);
        *reinterpret_cast<uint4*>(stg1 + r * 128 + phys * 16) = pk2;
        if (p.y_lo != nullptr && m0 + r < p.M_total) {
          // the rounding residual of y, itself rounded to bf16: the bilinear upsample that consumes y reads
          // y + y_lo (~16 mantissa bits), so the next conv's operand is rounded ONCE like the fp32 reference's
          // would be.  Only requested for the small layers (<= 32^2), where the extra bytes are free.
          const float2 h0 = unpack_bf16x2(pk2.x), h1 = unpack_bf16x2(pk2.y), h2 = unpack_bf16x2(pk2.z),
                       h3 = unpack_bf16x2(pk2.w);
          uint4 lo;
          lo.x = pack_bf16x2(o2[0] - h0.x, o2[1] - h0.y);
          lo.y = pack_bf16x2(o2[2] - h1.x, o2[3] - h1.y);
          lo.z = pack_bf16x2(o2[4] - h2.x, o2[5] - h2.y);
          lo.w = pack_bf16x2(o2[6] - h3.x, o2[7] - h3.y);
          *reinterpret_cast<uint4*>(p.y_lo + (size_t)(m0 + r) * p.N_total + ng0 + cbase + jj * 8) = lo;
        }
      }
    }
    fence_proxy_async_smem();
    named_bar_sync(1, kEpiThreads);
    if constexpr (MODE == EPI_BNBWD || MODE == EPI_BNBWD_RES) {
      // column phase on the staged chunk: thread = (channel pair, 16-row group); mask the gradient in place, sum
      // g and g * xhat over the rows (same expressions as bn_bwd_reduce_kernel)
      const int pr = etid & 31;
      const int g = etid >> 5;
      const int cc = ng0 + chunk * 64 + 2 * pr;
      const size_t so = (size_t)(m_tile / p.sg_tiles) * p.N_total + cc;
      const float2 mm = __ldg(reinterpret_cast<const float2*>(p.bn_mean + so));
      const float2 rs = __ldg(reinterpret_cast<const float2*>(p.bn_rstd + so));
      float2 ga = make_float2(0.f, 0.f), be = make_float2(0.f, 0.f);
      if constexpr (MODE == EPI_BNBWD) {
        const int grp = m_tile / p.wg_tiles;
        const float* gam =
            grp == 0 ? p.bn_gamma[0] : (grp == 1 ? p.bn_gamma[1] : (grp == 2 ? p.bn_gamma[2] : p.bn_gamma[3]));
        const float* bet = grp == 0 ? p.bn_beta[0] : (grp == 1 ? p.bn_beta[1] : (grp == 2 ? p.bn_beta[2] : p.bn_beta[3]));
        ga = __ldg(reinterpret_cast<const float2*>(gam + cc));
        be = __ldg(reinterpret_cast<const float2*>(bet + cc));
      }
      const int bit0 = (2 * pr) & 7;
      float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int row = g * 16 + i;
        const int phys = (pr >> 2) ^ (row & 7);
        uint32_t* cell = reinterpret_cast<uint32_t*>(stg0 + row * 128 + phys * 16 + (pr & 3) * 4);
        float2 f = unpack_bf16x2(*cell);
        const float2 z = unpack_bf16x2(zw[i]);
        const float x0 = (z.x - mm.x) * rs.x, x1 = (z.y - mm.y) * rs.y;
        if constexpr (MODE == EPI_BNBWD) {
          f.x = (ga.x * x0 + be.x) > 0.f ? f.x : 0.f;
          f.y = (ga.y * x1 + be.y) > 0.f ? f.y : 0.f;
        } else {
          const float2 h = unpack_bf16x2(gw[i]);
          f.x = ((bw[i] >> bit0) & 1) ? f.x + h.x : 0.f;
          f.y = ((bw[i] >> (bit0 + 1)) & 1) ? f.y + h.y : 0.f;
        }
        *cell = pack_bf16x2(f.x, f.y);
        s0 += f.x;
        q0 += f.x * x0;
        s1 += f.y;
        q1 += f.y * x1;
      }
      float* red = vec;  // [8][64][2]
      red[(g * 64 + 2 * pr) * 2 + 0] = s0;
      red[(g * 64 + 2 * pr) * 2 + 1] = q0;
      red[(g * 64 + 2 * pr + 1) * 2 + 0] = s1;
      red[(g * 64 + 2 * pr + 1) * 2 + 1] = q1;
      fence_proxy_async_smem();
      named_bar_sync(1, kEpiThreads);
      if (warp == 2) {
        __syncwarp();
        if (elect_one_sync()) {
          tma_store_2d(map_out, stg0, ng0 + chunk * 64, m0);
          tma_store_commit();
        }
      }
      if (etid < 128) {
        const int ch = etid & 63, which = etid >> 6;
        float acc = 0.f;
#pragma unroll
        for (int gg = 0; gg < 8; ++gg) acc += red[(gg * 64 + ch) * 2 + which];
        p.stat_sum[((size_t)m_tile * 2 + which) * p.N_total + ng0 + chunk * 64 + ch] = acc;
      }
      continue;
    }
    if (warp == 2) {
      __syncwarp();
      if (elect_one_sync()) {
        if constexpr (BOX) tma_store_4d(map_out, stg0, ng0 + chunk * 64, bw0, bh0, bn0);
        else tma_store_2d(map_out, stg0, ng0 + chunk * 64, m0);
        if constexpr (MODE == EPI_STYLE) tma_store_2d(map_out2, stg1, ng0 + chunk * 64, m0);
        tma_store_commit();
      }
    }
    if constexpr (MODE == EPI_STATS) {
      // per-channel sum / sum of squares over the 128 rows of this staged chunk (values as stored, bf16)
      const int pr = etid & 31;  // channel pair
      const int g = etid >> 5;   // 16-row group
      float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int row = g * 16 + i;
        const int phys = (pr >> 2) ^ (row & 7);
        const uint32_t w = *reinterpret_cast<const uint32_t*>(stg0 + row * 128 + phys * 16 + (pr & 3) * 4);
        const float2 f = unpack_bf16x2(w);
        s0 += f.x;
        q0 += f.x * f.x;
        s1 += f.y;
        q1 += f.y * f.y;
      }
      float* red = vec;  // [8][64][2]
      red[(g * 64 + 2 * pr) * 2 + 0] = s0;
      red[(g * 64 + 2 * pr) * 2 + 1] = q0;
      red[(g * 64 + 2 * pr + 1) * 2 + 0] = s1;
      red[(g * 64 + 2 * pr + 1) * 2 + 1] = q1;
      named_bar_sync(1, kEpiThreads);
      if (etid < 128) {
        const int ch = etid & 63, which = etid >> 6;
        float acc = 0.f;
#pragma unroll
        for (int gg = 0; gg < 8; ++gg) acc += red[(gg * 64 + ch) * 2 + which];
        float* dst = which ? p.stat_sq : p.stat_sum;
        dst[(size_t)m_tile * p.N_total + ng0 + chunk * 64 + ch] = acc;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Per-warp epilogue (conv_gemm_kernel, every mode but STYLE).  The pointwise layers of the encoders have one to eight
// k-blocks per tile: their time is the epilogue, and in epilogue_acc all eight warps walk the 64-column chunks in
// lockstep through two 256-thread barriers per chunk (drain -> barrier -> stage -> barrier -> one 16 KB TMA store).
// Here the warps are decoupled: warp (q, h) owns rows 32q..32q+31 of every chunk whose running index has parity h,
// drains all 64 columns of it, stages them in its OWN 4 KB slab (two per warp) and issues its own [32 x 64] TMA store:
// only __syncwarp on the plain path.  The statistics modes add one 128-thread barrier per chunk (the four quarter
// warps of a chunk combine their column sums in rank order: deterministic).
// ------------------------------------------------------------------------------------------------
constexpr int kSlabBytes = 4096;

template <int BLOCK_N, int MODE>
__device__ __forceinline__ void epilogue_tile_warp(const ConvGemmArgs& p, const CUtensorMap* map_slab, uint32_t tmem_base,
                                                   uint32_t acc_col, int m0, int n_tile, uint64_t* release_bar,
                                                   uint8_t* stg_base, float* vec, uint32_t& chunk_counter,
                                                   uint32_t& my_slabs, bool release_at_leader = false) {
  static_assert(MODE != EPI_STYLE, "STYLE keeps the two-output epilogue");
  // 2-SM MMA: the accumulators of both CTAs are written by the leader's MMA warp, which waits on ITS barrier
  auto release = [&]() {
    if (release_at_leader) mbar_arrive_cluster(release_bar, 0);
    else mbar_arrive(release_bar);
  };
  constexpr int CHUNKS = BLOCK_N / 64;
  constexpr bool kSums = MODE == EPI_STATS || MODE == EPI_BNBWD || MODE == EPI_BNBWD_RES;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int e = warp - 2;
  const int q = warp & 3;   // TMEM lane quarter this warp may touch
  const int h = e >> 2;     // chunk parity this warp serves
  const int m_tile = m0 >> 7;
  const int ng0 = n_tile * BLOCK_N;
  const int pg0 = (m_tile / p.wg_tiles) * p.N_total + ng0;
  const int row = m0 + q * 32 + lane;  // this thread's output row
  uint8_t* slabs = stg_base + e * 2 * kSlabBytes;
  float* wvec = vec + e * 128;         // per-warp [2][64]: AFFINE scale | shift, PLAIN bias (statistics modes: `vec` = red)
  // the chunks of this tile this warp serves: first, first + 2, ...
  const int first = (h - (int)chunk_counter) & 1;
  const int last_mine = first < CHUNKS ? first + 2 * ((CHUNKS - 1 - first) / 2) : -1;
  if (last_mine < 0) {  // nothing to drain from this accumulator
    __syncwarp();
    if (lane == 0) release();
  }
#pragma unroll 1
  for (int chunk = first; chunk < CHUNKS; chunk += 2) {
    const int cg0 = ng0 + chunk * 64;  // first channel of the chunk
    uint32_t zw[32], gw[32];
    uint8_t bw[32];
    if constexpr (MODE == EPI_BNBWD || MODE == EPI_BNBWD_RES) {
      // column phase operands (lane = channel pair, 32 rows of this warp), in flight during the drain
      const size_t cell0 = (size_t)(m0 + q * 32) * p.N_total + cg0 + 2 * lane;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        zw[i] = __ldg(reinterpret_cast<const uint32_t*>(p.bn_z + cell0 + (size_t)i * p.N_total));
        if constexpr (MODE == EPI_BNBWD_RES) {
          gw[i] = __ldg(reinterpret_cast<const uint32_t*>(p.bn_g2 + cell0 + (size_t)i * p.N_total));
          bw[i] = __ldg(p.bn_bits + ((cell0 + (size_t)i * p.N_total) >> 3));
        }
      }
    }
    if constexpr (MODE == EPI_AFFINE || MODE == EPI_PLAIN) {
      if (MODE == EPI_AFFINE || p.bias != nullptr) {
        __syncwarp();  // previous chunk's reads of wvec
        wvec[lane] = MODE == EPI_AFFINE ? p.nw[pg0 + chunk * 64 + lane] : 0.f;            // scale
        wvec[lane + 32] = MODE == EPI_AFFINE ? p.nw[pg0 + chunk * 64 + 32 + lane] : 0.f;
        wvec[64 + lane] = p.bias[pg0 + chunk * 64 + lane];                                 // shift / bias
        wvec[96 + lane] = p.bias[pg0 + chunk * 64 + 32 + lane];
        __syncwarp();
      }
    }
    uint32_t va[32], vb[32];
    const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + acc_col + chunk * 64;
    tmem_ld32(taddr, va);
    tmem_ld32(taddr + 32, vb);
    tmem_ld_wait();
    if (chunk == last_mine) {  // this warp is done with the accumulator
      tc_fence_before();
      __syncwarp();
      if (lane == 0) release();
    }
    uint8_t* slab = slabs + (my_slabs & 1) * kSlabBytes;
    if (lane == 0) tma_store_wait_read<1>();  // the store issued from this slab two chunks ago has read it
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 8; ++j) {  // 16-byte pieces of this thread's 128-byte staging row
      float o[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int c = j * 8 + t;
        const float acc = __uint_as_float(c < 32 ? va[c & 31] : vb[c & 31]);
        if constexpr (MODE == EPI_AFFINE) o[t] = acc * wvec[c] + wvec[64 + c];
        else if constexpr (MODE == EPI_PLAIN) o[t] = p.bias != nullptr ? acc + wvec[64 + c] : acc;
        else o[t] = acc;
      }
      if constexpr (MODE == EPI_AFFINE) {
        if (p.res != nullptr && row < p.M_total) {
          const uint4 u = *reinterpret_cast<const uint4*>(p.res + (size_t)row * p.N_total + cg0 + j * 8);
          const float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
          o[0] += a0.x; o[1] += a0.y; o[2] += a1.x; o[3] += a1.y;
          o[4] += a2.x; o[5] += a2.y; o[6] += a3.x; o[7] += a3.y;
        }
#pragma unroll
        for (int t = 0; t < 8; ++t)
          o[t] = p.relu == 1 ? fmaxf(o[t], 0.f) : (p.relu == 2 ? (o[t] > 0.f ? o[t] : 0.2f * o[t]) : o[t]);
      }
      uint4 pk;
      pk.x = pack_bf16x2(o[0], o[1]);
      pk.y = pack_bf16x2(o[2], o[3]);
      pk.z = pack_bf16x2(o[4], o[5]);
      pk.w = pack_bf16x2(o[6], o[7]);
      *reinterpret_cast<uint4*>(slab + lane * 128 + ((j ^ (lane & 7)) << 4)) = pk;
    }
    if constexpr (kSums) {
      __syncwarp();
      // column phase: lane = channel pair (2 * lane, 2 * lane + 1) over the warp's 32 rows, straight from the slab
      float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
      if constexpr (MODE == EPI_STATS) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const uint32_t w = *reinterpret_cast<const uint32_t*>(slab + i * 128 + (((lane >> 2) ^ (i & 7)) << 4) + (lane & 3) * 4);
          const float2 f = unpack_bf16x2(w);
          s0 += f.x;
          q0 += f.x * f.x;
          s1 += f.y;
          q1 += f.y * f.y;
        }
      } else {
        const int cc = cg0 + 2 * lane;
        const size_t so = (size_t)(m_tile / p.sg_tiles) * p.N_total + cc;
        const float2 mm = __ldg(reinterpret_cast<const float2*>(p.bn_mean + so));
        const float2 rs = __ldg(reinterpret_cast<const float2*>(p.bn_rstd + so));
        float2 ga = make_float2(0.f, 0.f), be = make_float2(0.f, 0.f);
        if constexpr (MODE == EPI_BNBWD) {
          const int grp = m_tile / p.wg_tiles;
          const float* gam =
              grp == 0 ? p.bn_gamma[0] : (grp == 1 ? p.bn_gamma[1] : (grp == 2 ? p.bn_gamma[2] : p.bn_gamma[3]));
          const float* bet = grp == 0 ? p.bn_beta[0] : (grp == 1 ? p.bn_beta[1] : (grp == 2 ? p.bn_beta[2] : p.bn_beta[3]));
          ga = __ldg(reinterpret_cast<const float2*>(gam + cc));
          be = __ldg(reinterpret_cast<const float2*>(bet + cc));
        }
        const int bit0 = (2 * lane) & 7;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          uint32_t* cell = reinterpret_cast<uint32_t*>(slab + i * 128 + (((lane >> 2) ^ (i & 7)) << 4) + (lane & 3) * 4);
          float2 f = unpack_bf16x2(*cell);
          const float2 z = unpack_bf16x2(zw[i]);
          const float x0 = (z.x - mm.x) * rs.x, x1 = (z.y - mm.y) * rs.y;
          if constexpr (MODE == EPI_BNBWD) {
            f.x = (ga.x * x0 + be.x) > 0.f ? f.x : 0.f;
            f.y = (ga.y * x1 + be.y) > 0.f ? f.y : 0.f;
          } else {
            const float2 g2 = unpack_bf16x2(gw[i]);
            f.x = ((bw[i] >> bit0) & 1) ? f.x + g2.x : 0.f;
            f.y = ((bw[i] >> (bit0 + 1)) & 1) ? f.y + g2.y : 0.f;
          }
          *cell = pack_bf16x2(f.x, f.y);
          s0 += f.x;
          q0 += f.x * x0;
          s1 += f.y;
          q1 += f.y * x1;
        }
      }
      // red[slab parity][h][q][64 channels][2]: the four quarter warps of this chunk, combined by quarter 0
      float* red = vec + ((((my_slabs & 1) * 2 + h) * 4 + q) * 64) * 2;
      *reinterpret_cast<float4*>(red + 4 * lane) = make_float4(s0, q0, s1, q1);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      tma_store_2d(map_slab, slab, cg0, m0 + q * 32);
      tma_store_commit();
    }
    if constexpr (kSums) {
      named_bar_sync(1 + h, 128);
      if (q == 0) {
        const float* r0 = vec + ((((my_slabs & 1) * 2 + h) * 4) * 64) * 2 + 4 * lane;
        float4 t = *reinterpret_cast<const float4*>(r0);
#pragma unroll
        for (int k = 1; k < 4; ++k) {
          const float4 u = *reinterpret_cast<const float4*>(r0 + k * 128);
          t.x += u.x;
          t.y += u.y;
          t.z += u.z;
          t.w += u.w;
        }
        if constexpr (MODE == EPI_STATS) {
          const size_t d = (size_t)m_tile * p.N_total + cg0 + 2 * lane;
          *reinterpret_cast<float2*>(p.stat_sum + d) = make_float2(t.x, t.z);
          *reinterpret_cast<float2*>(p.stat_sq + d) = make_float2(t.y, t.w);
        } else {
          const size_t d = (size_t)m_tile * 2 * p.N_total + cg0 + 2 * lane;
          *reinterpret_cast<float2*>(p.stat_sum + d) = make_float2(t.x, t.z);
          *reinterpret_cast<float2*>(p.stat_sum + d + p.N_total) = make_float2(t.y, t.w);
        }
      }
    }
    ++my_slabs;
  }
  chunk_counter += CHUNKS;
}

// CL = CTAs per cluster (1 or 2).  With CL = 2 the pair works on two vertically adjacent pixel tiles of the same n tile
// and weight group: the [BLOCK_N x 64] weight tile of every k-block is the same for both, so each CTA fetches HALF of it
// and multicasts that half into both CTAs' stages.  For BLOCK_N = 256 the weight tile is two thirds of what an SM pulls
// from L2 per k-block (32 KB against 16 KB of pixels); the pair cuts the L2's output by a third (optional: measured
// neutral, see cluster_mode()).  A stage may be refilled only when BOTH CTAs' MMAs have read it: the MMA warp commits to
// the empty barrier of both CTAs (count CL).
//
// MMA2 (with CL = 2): the pair executes 2-SM MMAs (tcgen05 cta_group::2, M = 256): each CTA loads ONLY its half of the
// weight tile (its SM ingests A 16 KB + B 16 KB per k-block instead of 16 + 32), the leader's MMA warp issues for both,
// commits go to both CTAs' barriers, both CTAs' epilogue warps release the accumulator at the leader.
//
// BOX: the box-tiled geometry for 3x3 layers whose 128 consecutive pixels are not one TMA box (W neither dividing 128 nor
// a multiple of it, or H not fitting whole boxes: 56^2, 28^2, 14^2, 7^2, odd sizes).  An m tile is a box of
// P = tw*th*tn <= 128 pixels (see irfd_conv_gemm_geometry); every tap loads that box shifted by the tap offset, the
// out-of-bounds zero fill is the padding as before.  A rows P..127 keep stale shared memory: MMA rows are independent,
// so they only reach accumulator rows that are never stored.  M stays 128.  Single CTA, lockstep epilogue.
template <int BLOCK_N, int MODE, int CL = 1, bool MMA2 = false, bool BOX = false>
__global__ void __launch_bounds__(kNumThreads, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const __grid_constant__ CUtensorMap map_out, const __grid_constant__ CUtensorMap map_out2,
                 const ConvGemmArgs p) {
  using Cfg = GemmCfg<BLOCK_N, MODE>;
  constexpr int STAGES = Cfg::STAGES;
  static_assert(STAGES >= 2, "pipeline too shallow");
  static_assert(!MMA2 || (CL == 2 && MODE != EPI_STYLE), "the 2-SM MMA needs a CTA pair and the per-warp epilogue");
  static_assert(!BOX || (CL == 1 && (MODE == EPI_PLAIN || MODE == EPI_AFFINE)), "box tiles: one CTA, PLAIN / AFFINE");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stg_base = smem + STAGES * Cfg::STAGE_BYTES;
  uint8_t* misc = stg_base + Cfg::STG_TOTAL;
  float* vec = reinterpret_cast<float*>(misc);                       // 6 * 256 floats (STYLE) / red scratch (STATS)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(misc + 8192);     // [STAGES]
  uint64_t* empty_bar = full_bar + STAGES;                           // [STAGES]
  uint64_t* tmem_full = empty_bar + STAGES;                          // [2]
  uint64_t* tmem_empty = tmem_full + 2;                              // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // work unit = CL consecutive m tiles x one n tile; unit u -> (u / num_n_tiles, u % num_n_tiles); this CTA takes m tile
  // CL * (u / num_n_tiles) + its rank in the cluster
  const int crank = CL > 1 ? (int)cluster_ctarank() : 0;
  const int unit0 = blockIdx.x / CL, unit_step = gridDim.x / CL;
  const int total_units = (p.num_m_tiles / CL) * p.num_n_tiles;
  const int num_kb = p.taps * p.cin_chunks;
  constexpr uint16_t kClusterMask = (1u << CL) - 1;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], MMA2 ? 1 : CL);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], MMA2 ? 16 : 8);
    }
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 0) {
    if (MMA2) tmem_alloc_2sm<Cfg::TMEM_COLS>(tmem_ptr);
    else tmem_alloc<Cfg::TMEM_COLS>(tmem_ptr);
  }
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();  // the peer's barriers are initialised before anything is multicast at them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (whole warp converged, one lane issues)
    {
      if (lane == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
      }
      __syncwarp();
      // bytes one stage's A box brings (the full box, out-of-bounds fill included)
      const uint32_t a_bytes = BOX ? (uint32_t)(p.box_tw * p.box_th * p.box_tn) * 128u : (uint32_t)Cfg::A_BYTES;
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = unit0; unit < total_units; unit += unit_step) {
        const int m_tile = (unit / p.num_n_tiles) * CL + crank;
        const int n_tile = unit % p.num_n_tiles;
        int w0, h0, n0;
        if constexpr (BOX) {
          box_origin(p, m_tile, w0, h0, n0);
        } else {
          const int m0 = (p.a_mod_tiles > 0 ? m_tile % p.a_mod_tiles : m_tile) * 128;
          w0 = m0 % p.W;
          h0 = (m0 / p.W) % p.H;
          n0 = m0 / (p.W * p.H);
        }
        const int b_row = (m_tile / p.wg_tiles) * p.N_total + n_tile * BLOCK_N;
        for (int tap = 0; tap < p.taps; ++tap) {
          const int dh = tap / p.kw - p.pad;
          const int dw = tap % p.kw - p.pad;
          for (int ch = 0; ch < p.cin_chunks; ++ch) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
            if (MMA2) {
              if (elect_one_sync()) {  // both CTAs' bytes are counted on the leader's barrier
                if (crank == 0) mbar_expect_tx(&full_bar[stage], 2 * (Cfg::A_BYTES + Cfg::B_BYTES / 2));
                tma_load_4d_2sm(sa, &map_a, &full_bar[stage], ch * 64, w0 + dw, h0 + dh, n0);
                tma_load_2d_2sm(sa + Cfg::A_BYTES, &map_b, &full_bar[stage], (tap * p.cin_chunks + ch) * 64,
                                b_row + crank * (BLOCK_N / 2));
              }
            } else if (elect_one_sync()) {
              mbar_expect_tx(&full_bar[stage], a_bytes + Cfg::B_BYTES);
              tma_load_4d(sa, &map_a, &full_bar[stage], ch * 64, w0 + dw, h0 + dh, n0);
              if (CL == 1)
                tma_load_2d(sa + Cfg::A_BYTES, &map_b, &full_bar[stage], (tap * p.cin_chunks + ch) * 64, b_row);
              else  // this CTA's share of the weight tile, into both CTAs' stage
                tma_load_2d_mc(sa + Cfg::A_BYTES + crank * (Cfg::B_BYTES / CL), &map_b, &full_bar[stage],
                               (tap * p.cin_chunks + ch) * 64, b_row + crank * (BLOCK_N / CL), kClusterMask);
            }
            __syncwarp();
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (whole warp converged, one lane issues)
    if (!MMA2 || crank == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(MMA2 ? 256 : 128, BLOCK_N, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      for (int unit = unit0; unit < total_units; unit += unit_step, ++iter) {
        const int as = iter & 1;
        const uint32_t aphase = (iter >> 1) & 1;
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BLOCK_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint64_t adesc0 = make_smem_desc_sw128(a_addr, 0, 1024);
          const uint64_t bdesc0 = make_smem_desc_sw128(a_addr + Cfg::A_BYTES, 0, 1024);
          if (elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < 4; ++k)  // +32 bytes per K=16 step: +2 in the descriptor's 16-byte address field
              if (MMA2) umma_bf16_2sm(d_tmem, adesc0 + 2 * k, bdesc0 + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
              else umma_bf16(d_tmem, adesc0 + 2 * k, bdesc0 + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            if (MMA2) umma_commit_2sm_mc(&empty_bar[stage], kClusterMask);
            else if (CL == 1) umma_commit(&empty_bar[stage]);
            else umma_commit_mc(&empty_bar[stage], kClusterMask);
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (elect_one_sync()) {
          if (MMA2) umma_commit_2sm_mc(&tmem_full[as], kClusterMask);
          else umma_commit(&tmem_full[as]);
        }
        __syncwarp();
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (8 warps)
    int iter = 0;
    uint32_t chunk_counter = 0, my_slabs = 0;
    for (int unit = unit0; unit < total_units; unit += unit_step, ++iter) {
      const int as = iter & 1;
      const uint32_t aphase = (iter >> 1) & 1;
      const int m_tile = (unit / p.num_n_tiles) * CL + crank;
      const int n_tile = unit % p.num_n_tiles;
      mbar_wait(&tmem_full[as], aphase);
      tc_fence_after();
      if constexpr (MODE != EPI_STYLE && !BOX) {
        if (p.warp_epi) {
          epilogue_tile_warp<BLOCK_N, MODE>(p, &map_out2, tmem_base, as * BLOCK_N, m_tile * 128, n_tile, &tmem_empty[as],
                                            stg_base, vec, chunk_counter, my_slabs, MMA2);
          continue;
        }
      }
      epilogue_acc<BLOCK_N, MODE, 2, BOX>(p, &map_out, &map_out2, tmem_base, as * BLOCK_N, m_tile * 128, n_tile,
                                          &tmem_empty[as], stg_base, vec, chunk_counter);
    }
    // the staging buffers only have to outlive the TMA engine's READS; global visibility comes with grid completion
    if (MODE != EPI_STYLE && !BOX && p.warp_epi) {
      if (lane == 0) tma_store_wait_read<0>();
    } else if (warp == 2) {
      __syncwarp();
      if (elect_one_sync()) tma_store_wait_read<0>();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();  // the peer may still multicast into this CTA's stages / commit to its barriers
  if (warp == 0) {
    if (MMA2) tmem_dealloc_2sm<Cfg::TMEM_COLS>(tmem_base);
    else tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}


// ------------------------------------------------------------------------------------------------
// Halo-reuse variant for 3x3 convs on wide images (W % 128 == 0, H even) with BLOCK_N <= 128 — the generator's
// 128^2 / 256^2 layers, which the per-tap kernel above runs L2->SM fabric-bound (every tap re-fetches its A tile:
// 9 x 16 KB per 128 pixels and 64 input channels).
//
// Tile = 256 output pixels = two image rows x 128 columns -> two accumulators.  Per 64-channel chunk ONE 4-D TMA box
// brings the [4 rows][130 columns][64 ch] halo (65 KB) that serves all nine taps of both rows: the A operand of tap
// (dy, dx) for output row j is the same smem buffer at line offset (j + dy) * 130 + dx, i.e. only the descriptor start
// address moves (128-byte lines; the 128-byte swizzle is a function of the absolute smem address, so a shifted start
// stays consistent with what TMA wrote; measured: filling the descriptor's base-offset field instead gives garbage).  Each [BLOCK_N x 64] weight tile feeds both accumulators.
// L2->SM bytes per 128 pixels x 64 channels: 33 KB (A) + 36 KB (B, N = 64) instead of 144 KB + 72 KB.
//
// Warp roles: warp 0 = halo (A) producer, warp 1 = MMA issuer, warps 2..9 = epilogue, warp 10 = weight (B) producer.
// ------------------------------------------------------------------------------------------------
constexpr int kHaloThreads = 352;
constexpr int kHaloCols = 130;
constexpr int kHaloRows = 4;

template <int BLOCK_N, int MODE>
struct HaloCfg {
  static_assert(BLOCK_N == 64 || BLOCK_N == 128, "two double-buffered accumulators need 4 x BLOCK_N <= 512 TMEM columns");
  static constexpr int A_BYTES = kHaloRows * kHaloCols * 128;  // 66,560 = 65 x 1024
  static constexpr int A_STAGES = 2;
  static constexpr int B_BYTES = BLOCK_N * 128;
  static constexpr int NUM_OUT = (MODE == EPI_STYLE) ? 2 : 1;
  static constexpr int NBUF = (NUM_OUT == 2) ? 1 : 2;  // staging buffers per output
  static constexpr int STG_TOTAL = NUM_OUT * NBUF * kStgBytes;
  static constexpr int RAW_B = (kSmemLimit - 1024 - A_STAGES * A_BYTES - STG_TOTAL - kMiscBytes) / B_BYTES;
  static constexpr int B_STAGES = RAW_B > 8 ? 8 : RAW_B;
  static constexpr int SMEM_BYTES = 1024 + A_STAGES * A_BYTES + B_STAGES * B_BYTES + STG_TOTAL + kMiscBytes;
  static constexpr uint32_t TMEM_COLS = 4 * BLOCK_N <= 256 ? 256 : 512;
  static_assert(A_BYTES % 1024 == 0 && B_STAGES >= 2, "halo stage must keep 1024-byte alignment");
};

struct HaloArgs {
  int wsegs, hpairs;  // W / 128, H / 2
  int total_tiles;    // 256-pixel tiles x n tiles
};

template <int BLOCK_N, int MODE>
__global__ void __launch_bounds__(kHaloThreads, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const __grid_constant__ CUtensorMap map_out, const __grid_constant__ CUtensorMap map_out2,
                 const ConvGemmArgs p, const HaloArgs hp) {
  using Cfg = HaloCfg<BLOCK_N, MODE>;
  constexpr int BST = Cfg::B_STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_b = smem + Cfg::A_STAGES * Cfg::A_BYTES;
  uint8_t* stg_base = smem_b + BST * Cfg::B_BYTES;
  uint8_t* misc = stg_base + Cfg::STG_TOTAL;
  float* vec = reinterpret_cast<float*>(misc);
  uint64_t* full_a = reinterpret_cast<uint64_t*>(misc + 8192);  // [2]
  uint64_t* empty_a = full_a + 2;                               // [2]
  uint64_t* full_b = empty_a + 2;                               // [BST]
  uint64_t* empty_b = full_b + BST;                             // [BST]
  uint64_t* tmem_full = empty_b + BST;                          // [2]
  uint64_t* tmem_empty = tmem_full + 2;                         // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int chunks = p.cin_chunks;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&full_a[i], 1);
      mbar_init(&empty_a[i], 1);
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 8);
    }
    for (int i = 0; i < BST; ++i) {
      mbar_init(&full_b[i], 1);
      mbar_init(&empty_b[i], 1);
    }
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc<Cfg::TMEM_COLS>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // tile -> (n tile, image, row pair, column segment); n tile fastest like the per-tap kernel
  auto decode = [&](int tile, int& n_tile, int& n0, int& h0, int& w0) {
    const int m2 = tile / p.num_n_tiles;
    n_tile = tile - m2 * p.num_n_tiles;
    const int wseg = m2 % hp.wsegs;
    const int t = m2 / hp.wsegs;
    const int hpair = t % hp.hpairs;
    n0 = t / hp.hpairs;
    h0 = hpair * 2;
    w0 = wseg * 128;
  };

  if (warp == 0) {
    // ------------------------------------------------------------------ halo (A) producer
    {
      if (lane == 0) tma_prefetch_desc(&map_a);
      __syncwarp();
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < hp.total_tiles; tile += gridDim.x) {
        int n_tile, n0, h0, w0;
        decode(tile, n_tile, n0, h0, w0);
        for (int ch = 0; ch < chunks; ++ch) {
          mbar_wait(&empty_a[stage], phase ^ 1);
          if (elect_one_sync()) {
            mbar_expect_tx(&full_a[stage], Cfg::A_BYTES);
            tma_load_4d(smem + stage * Cfg::A_BYTES, &map_a, &full_a[stage], ch * 64, w0 - 1, h0 - 1, n0);
          }
          __syncwarp();
          if (++stage == Cfg::A_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 10) {
    // ------------------------------------------------------------------ weight (B) producer
    {
      if (lane == 0) tma_prefetch_desc(&map_b);
      __syncwarp();
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < hp.total_tiles; tile += gridDim.x) {
        const int n_tile = tile % p.num_n_tiles;
        for (int ch = 0; ch < chunks; ++ch) {
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(&empty_b[stage], phase ^ 1);
            if (elect_one_sync()) {
              mbar_expect_tx(&full_b[stage], Cfg::B_BYTES);
              tma_load_2d(smem_b + stage * Cfg::B_BYTES, &map_b, &full_b[stage], (tap * chunks + ch) * 64,
                          n_tile * BLOCK_N);
            }
            __syncwarp();
            if (++stage == BST) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (whole warp converged, one lane issues)
    {
      constexpr uint32_t idesc = make_idesc_bf16(128, BLOCK_N, 0, 0);
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      int iter = 0;
      for (int tile = blockIdx.x; tile < hp.total_tiles; tile += gridDim.x, ++iter) {
        const int as = iter & 1;
        const uint32_t aphase = (iter >> 1) & 1;
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * 2 * BLOCK_N;
        for (int ch = 0; ch < chunks; ++ch) {
          mbar_wait(&full_a[sa], pa);
          // descriptor of the halo's first line; a tap / K step only adds to its 16-byte-granular address field
          const uint64_t adesc0 = make_smem_desc_sw128(smem_u32(smem + sa * Cfg::A_BYTES), 0, 1024);
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            constexpr int kLine = 128 / 16;  // one halo line (pixel) in descriptor address units
            const int dy = tap / 3, dx = tap % 3;
            mbar_wait(&full_b[sb], pb);
            tc_fence_after();
            const uint64_t bdesc0 = make_smem_desc_sw128(smem_u32(smem_b + sb * Cfg::B_BYTES), 0, 1024);
            if (elect_one_sync()) {
#pragma unroll
              for (int j = 0; j < 2; ++j) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_bf16(d_tmem + j * BLOCK_N, adesc0 + ((j + dy) * kHaloCols + dx) * kLine + 2 * k, bdesc0 + 2 * k,
                            idesc, (tap | k) != 0 ? 1u : (ch != 0 ? 1u : 0u));
              }
              umma_commit(&empty_b[sb]);
            }
            __syncwarp();
            if (++sb == BST) {
              sb = 0;
              pb ^= 1;
            }
          }
          if (elect_one_sync()) umma_commit(&empty_a[sa]);
          __syncwarp();
          if (++sa == Cfg::A_STAGES) {
            sa = 0;
            pa ^= 1;
          }
        }
        if (elect_one_sync()) umma_commit(&tmem_full[as]);
        __syncwarp();
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (8 warps): two accumulators per tile
    int iter = 0;
    uint32_t chunk_counter = 0;
    for (int tile = blockIdx.x; tile < hp.total_tiles; tile += gridDim.x, ++iter) {
      const int as = iter & 1;
      const uint32_t aphase = (iter >> 1) & 1;
      int n_tile, n0, h0, w0;
      decode(tile, n_tile, n0, h0, w0);
      const int m0 = (n0 * p.H + h0) * p.W + w0;
      mbar_wait(&tmem_full[as], aphase);
      tc_fence_after();
      epilogue_acc<BLOCK_N, MODE, Cfg::NBUF>(p, &map_out, &map_out2, tmem_base, as * 2 * BLOCK_N, m0, n_tile, nullptr,
                                             stg_base, vec, chunk_counter);
      epilogue_acc<BLOCK_N, MODE, Cfg::NBUF>(p, &map_out, &map_out2, tmem_base, as * 2 * BLOCK_N + BLOCK_N, m0 + p.W,
                                             n_tile, &tmem_empty[as], stg_base, vec, chunk_counter);
    }
    // the staging buffers only have to outlive the TMA engine's READS; global visibility comes with grid completion
    if (warp == 2) {
      __syncwarp();
      if (elect_one_sync()) tma_store_wait_read<0>();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------------
template <int BLOCK_N, int MODE, int CL = 1, bool MMA2 = false, bool BOX = false>
static int launch_conv_gemm(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mo, const CUtensorMap& mo2,
                            const ConvGemmArgs& a, int grid, cudaStream_t stream) {
  using Cfg = GemmCfg<BLOCK_N, MODE>;
  static bool configured = false;
  auto kern = conv_gemm_kernel<BLOCK_N, MODE, CL, MMA2, BOX>;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_last_error("cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return IRFD_ERR_CUDA;
    }
    configured = true;
  }
  if (CL == 1) {
    kern<<<grid, kNumThreads, Cfg::SMEM_BYTES, stream>>>(ma, mb, mo, mo2, a);
  } else {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kNumThreads);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kern, ma, mb, mo, mo2, a);
  }
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

template <int MODE>
static int dispatch_block_n(int block_n, const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mo,
                            const CUtensorMap& mo2, const ConvGemmArgs& a, int grid, int cluster, cudaStream_t stream) {
  if constexpr (MODE == EPI_PLAIN || MODE == EPI_STATS || MODE == EPI_BNBWD) {
    if (cluster == 3) {  // CTA pairs with 2-SM MMAs
      if (block_n == 128) return launch_conv_gemm<128, MODE, 2, true>(ma, mb, mo, mo2, a, grid, stream);
      if (block_n == 256) return launch_conv_gemm<256, MODE, 2, true>(ma, mb, mo, mo2, a, grid, stream);
    }
  }
  if (cluster >= 2) {
    if (block_n == 128) return launch_conv_gemm<128, MODE, 2>(ma, mb, mo, mo2, a, grid, stream);
    if (block_n == 256) return launch_conv_gemm<256, MODE, 2>(ma, mb, mo, mo2, a, grid, stream);
  }
  switch (block_n) {
    case 64: return launch_conv_gemm<64, MODE>(ma, mb, mo, mo2, a, grid, stream);
    case 128: return launch_conv_gemm<128, MODE>(ma, mb, mo, mo2, a, grid, stream);
    case 256: return launch_conv_gemm<256, MODE>(ma, mb, mo, mo2, a, grid, stream);
  }
  set_last_error("bad BLOCK_N %d", block_n);
  return IRFD_ERR_INVALID_ARGUMENT;
}

template <int MODE>
static int dispatch_box(int block_n, const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mo,
                        const ConvGemmArgs& a, int grid, cudaStream_t stream) {
  switch (block_n) {
    case 64: return launch_conv_gemm<64, MODE, 1, false, true>(ma, mb, mo, mo, a, grid, stream);
    case 128: return launch_conv_gemm<128, MODE, 1, false, true>(ma, mb, mo, mo, a, grid, stream);
    case 256: return launch_conv_gemm<256, MODE, 1, false, true>(ma, mb, mo, mo, a, grid, stream);
  }
  set_last_error("bad BLOCK_N %d", block_n);
  return IRFD_ERR_INVALID_ARGUMENT;
}


template <int BLOCK_N, int MODE>
static int launch_conv_halo(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mo, const CUtensorMap& mo2,
                            const ConvGemmArgs& a, const HaloArgs& h, int grid, cudaStream_t stream) {
  using Cfg = HaloCfg<BLOCK_N, MODE>;
  static bool configured = false;
  auto kern = conv_halo_kernel<BLOCK_N, MODE>;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_last_error("cudaFuncSetAttribute(halo smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return IRFD_ERR_CUDA;
    }
    configured = true;
  }
  kern<<<grid, kHaloThreads, Cfg::SMEM_BYTES, stream>>>(ma, mb, mo, mo2, a, h);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

template <int MODE>
static int dispatch_halo(int block_n, const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mo,
                         const CUtensorMap& mo2, const ConvGemmArgs& a, const HaloArgs& h, int grid,
                         cudaStream_t stream) {
  if (block_n == 64) return launch_conv_halo<64, MODE>(ma, mb, mo, mo2, a, h, grid, stream);
  return launch_conv_halo<128, MODE>(ma, mb, mo, mo2, a, h, grid, stream);
}

// IRFD_GEMM_CLUSTER: 1 = CTA pairs with multicast weight tiles where the layer allows it, 0 (default) = never.
// Measured (round 2, every GEMM shape of the train step, L2 flushed): 12.76 ms/step without, 12.83 ms with — on the
// large-K layers the L2 -> SM stream is at 62 % of its peak and the tensor pipe busy 83 % of the cycles (ncu), so the
// weight-tile traffic is not what bounds them.  Kept as a tested option.
static int cluster_mode() {
  const char* e = getenv("IRFD_GEMM_CLUSTER");
  return e ? atoi(e) : 0;
}
// IRFD_GEMM_2SM: 1 = CTA pairs with 2-SM MMAs (cta_group::2) for the plain / statistics / BN-backward epilogues; 0
// (default).  Measured (every GEMM shape of the train step): 12.65 ms/step without, 13.49 ms with — bit-identical results,
// no shape more than 4 % faster, the HBM-bound pointwise layers 20-45 % slower (the pair runs in lockstep).
static int mma2_mode() {
  const char* e = getenv("IRFD_GEMM_2SM");
  return e ? atoi(e) : 0;
}

// IRFD_WARP_EPI: 1 (default) = per-warp epilogue in conv_gemm_kernel (all modes but STYLE), 0 = the lockstep one.
static int warp_epi_mode() {
  const char* e = getenv("IRFD_WARP_EPI");
  return e ? atoi(e) : 1;
}

// IRFD_CONV_HALO: 0 = never, 1 (default) = wide 3x3 layers with Cout 64/128, read at every call (tests flip it).
static int halo_mode() {
  const char* e = getenv("IRFD_CONV_HALO");
  return e ? atoi(e) : 1;
}

}  // namespace irfd

using namespace irfd;

extern "C" int irfd_conv_gemm_m_tiles(int n, int h, int w) {
  long long m = (long long)n * h * w;
  return (int)((m + 127) / 128);
}

// Pixel-tile geometry of a conv_gemm launch: the one place the shape rule lives (irfd_conv_gemm_geometry exports it).
// (H, W, NB) is the 4-D view the A operand's tensor map spans; a pointwise conv is one long row of pixels.
//   linear: 128 consecutive NHWC pixels form one (tw, th, tn) TMA box (W divides 128 or is a multiple of 128 for 3x3
//           convs, whole rows / whole images per tile); m tile t = pixels [128 t, 128 t + 128), a ragged last tile.
//   boxed : every shape the linear geometry rejects (conv_gemm_kernel<..., BOX = true>): a tile is a box of
//           P = tw*th*tn <= 128 pixels.  W < 128: tw = W, th = min(H, 128 / W), and if th == H, tn = 128 / (H*W)
//           images (at most NB; with weight groups the largest divisor of the per-group image count, so that every
//           tile belongs to one group).  W > 128: tw = 128, th = tn = 1, ceil(W / 128) column tiles per row.  Tiles are
//           ordered image-major, then rows, then columns.
struct TileGeom {
  int boxed, tw, th, tn, tiles_w, tiles_h, tiles_n;
  int H, W, NB;
};

static int tile_geometry(int n, int h, int w, int ksize, int wgroups, int a_shared, TileGeom* g) {
  IRFD_CHECK_ARG(ksize == 1 || ksize == 3, "conv_gemm: ksize must be 1 or 3 (got %d)", ksize);
  IRFD_CHECK_ARG(wgroups >= 1, "conv_gemm: bad weight group count %d", wgroups);
  const long long m_total_ll = (long long)n * h * w;
  IRFD_CHECK_ARG(n > 0 && h > 0 && w > 0 && m_total_ll < (1ll << 31) - 256, "conv_gemm: bad pixel count");
  const int m_total = (int)m_total_ll;
  int H = h, W = w, NB = n;
  if (ksize == 1) {  // pointwise conv == plain GEMM over a single long row of pixels
    H = 1;
    W = a_shared ? m_total / wgroups : m_total;  // a shared A operand only has one group's rows
    NB = 1;
  }
  g->H = H;
  g->W = W;
  g->NB = NB;
  // linear geometry
  bool linear = wgroups == 1 || m_total_ll % (128ll * wgroups) == 0;
  if (W >= 128) {
    linear = linear && (ksize == 1 || W % 128 == 0);
    g->tw = 128; g->th = 1; g->tn = 1;
  } else {
    const int rows = 128 / W;
    linear = linear && 128 % W == 0 && (H >= rows ? H % rows == 0 : rows % H == 0);
    g->tw = W;
    g->th = H >= rows ? rows : H;
    g->tn = H >= rows ? 1 : rows / H;
  }
  if (linear) {
    g->boxed = 0;
    if (W >= 128) {
      g->tiles_w = (W + 127) / 128;  // pointwise: a ragged last tile
      g->tiles_h = H;
      g->tiles_n = NB;
    } else {
      g->tiles_w = 1;
      g->tiles_h = H / g->th;
      g->tiles_n = (NB + g->tn - 1) / g->tn;
    }
    return IRFD_OK;
  }
  // box-tiled geometry
  IRFD_CHECK_ARG(NB % wgroups == 0,
                 "conv_gemm: %d weight groups need whole tiles per group (n=%d h=%d w=%d ksize=%d)", wgroups, n, h, w,
                 ksize);
  g->boxed = 1;
  if (W > 128) {
    g->tw = 128; g->th = 1; g->tn = 1;
  } else {
    g->tw = W;
    g->th = H < 128 / W ? H : 128 / W;
    int tn = 1;
    if (g->th == H) {
      tn = 128 / (H * W);
      if (tn > NB) tn = NB;
      if (wgroups > 1)
        while ((NB / wgroups) % tn) --tn;
    }
    g->tn = tn;
  }
  g->tiles_w = (W + g->tw - 1) / g->tw;
  g->tiles_h = (H + g->th - 1) / g->th;
  g->tiles_n = (NB + g->tn - 1) / g->tn;
  return IRFD_OK;
}

extern "C" int irfd_conv_gemm_geometry(int n, int h, int w, int ksize, int wgroups, int* out_host) {
  IRFD_CHECK_ARG(out_host != nullptr, "conv_gemm_geometry: null output");
  TileGeom g;
  const int rc = tile_geometry(n, h, w, ksize, wgroups, 0, &g);
  if (rc != IRFD_OK) return rc;
  const int v[7] = {g.boxed, g.tw, g.th, g.tn, g.tiles_w, g.tiles_h, g.tiles_n};
  for (int i = 0; i < 7; ++i) out_host[i] = v[i];
  return IRFD_OK;
}

struct BnBwdFold {  // EPI_BNBWD / EPI_BNBWD_RES operands (see ConvGemmArgs)
  const void* z;
  const float *mean, *rstd;
  const float* const* gamma;  // BNBWD
  const float* const* beta;
  const void* g2;             // BNBWD_RES
  const void* bits;
  int stat_groups;
};

// Which kernel instance a conv_gemm call launches and how its work spreads over the persistent CTAs: the one place the
// selection lives (conv_gemm_impl launches what it says; irfd_conv_gemm_plan exports it).  Reads the IRFD_* variables
// at call time and makes no CUDA call beyond num_sms().
struct ConvPlan {
  TileGeom geo;
  int use_halo, block_n, cluster, warp_epi;
  int num_m_tiles, num_n_tiles;
  int units;  // work units the CTAs walk (unit u: CTA slot u % slots, slots = grid / pair size, pair size 2 when
              // cluster > 1): halo tiles of 256 pixels x n tiles, or pair-size groups of 128-pixel m tiles x n tiles
  int grid;   // CTAs launched
};

static int conv_gemm_plan(int n, int h, int w, int cin, int cout, int ksize, int mode, int wgroups, int a_shared,
                          int force_block_n, ConvPlan* pl) {
  IRFD_CHECK_ARG(ksize == 1 || ksize == 3, "conv_gemm: ksize must be 1 or 3 (got %d)", ksize);
  IRFD_CHECK_ARG(cin % 64 == 0 && cin > 0, "conv_gemm: Cin must be a multiple of 64 (got %d)", cin);
  IRFD_CHECK_ARG(cout % 64 == 0 && cout > 0, "conv_gemm: Cout must be a multiple of 64 (got %d)", cout);
  IRFD_CHECK_ARG(mode >= 0 && mode <= 5, "conv_gemm: bad mode %d", mode);
  const long long m_total_ll = (long long)n * h * w;
  IRFD_CHECK_ARG(m_total_ll > 0 && m_total_ll < (1ll << 31) - 256, "conv_gemm: bad pixel count");
  const int m_total = (int)m_total_ll;
  IRFD_CHECK_ARG(wgroups >= 1, "conv_gemm: bad weight group count %d", wgroups);
  IRFD_CHECK_ARG(wgroups == 1 || (mode != EPI_STYLE), "conv_gemm: weight groups are not available in STYLE mode");
  IRFD_CHECK_ARG(!a_shared || (ksize == 1 && wgroups > 1), "conv_gemm: a shared A operand needs ksize 1 and groups > 1");

  TileGeom& geo = pl->geo;
  {
    const int rc = tile_geometry(n, h, w, ksize, wgroups, a_shared, &geo);
    if (rc != IRFD_OK) return rc;
  }
  const bool boxed = geo.boxed != 0;
  IRFD_CHECK_ARG(!boxed || mode == EPI_PLAIN || mode == EPI_AFFINE,
                 "conv_gemm: n=%d h=%d w=%d (ksize %d) needs box tiles, which serve the plain and affine epilogues only "
                 "(mode %d)", n, h, w, ksize, mode);
  const int H = geo.H, W = geo.W;
  const int num_m_tiles = boxed ? geo.tiles_w * geo.tiles_h * geo.tiles_n : (m_total + 127) / 128;
  const int wg_tiles = wgroups > 1 ? num_m_tiles / wgroups : 0x7fffffff;
  const int a_mod_tiles = a_shared ? num_m_tiles / wgroups : 0;
  pl->num_m_tiles = num_m_tiles;
  pl->warp_epi = (mode != EPI_STYLE && !boxed && m_total % 128 == 0 && warp_epi_mode() != 0) ? 1 : 0;

  int block_n = force_block_n;
  if (block_n == 0) {
    block_n = 64;
    const int cands[3] = {256, 128, 64};
    for (int i = 0; i < 3; ++i) {
      if (cout % cands[i] == 0 && (long long)num_m_tiles * (cout / cands[i]) >= num_sms()) {
        block_n = cands[i];
        break;
      }
    }
    // small-M layers: 128-wide tiles on >= 2/3 of the SMs beat 64-wide tiles on all of them (measured,
    // scripts/exp_blockn.py: 512->512 3x3 @8^2 x64 images 41 -> 29 us, 2048->512 1x1 23.5 -> 18.4 us)
    if (block_n == 64 && cout % 128 == 0 && (long long)num_m_tiles * (cout / 128) * 3 >= 2ll * num_sms()) block_n = 128;
  }
  IRFD_CHECK_ARG((block_n == 64 || block_n == 128 || block_n == 256) && cout % block_n == 0,
                 "conv_gemm: BLOCK_N %d incompatible with Cout %d", block_n, cout);
  // halo-reuse kernel: 3x3, rows of >= 128 pixels, Cout of one 64/128-wide tile (the fabric-bound generator layers)
  const int hmode = halo_mode();
  const bool use_halo = hmode != 0 && !boxed && mode != EPI_BNBWD && mode != EPI_BNBWD_RES && wgroups == 1 && ksize == 3 && W % 128 == 0 && H % 2 == 0 &&
                        (cout == 64 || cout == 128) &&
                        (force_block_n == 0 || force_block_n == cout);
  if (use_halo) block_n = cout;
  pl->use_halo = use_halo ? 1 : 0;
  pl->block_n = block_n;
  pl->num_n_tiles = cout / block_n;
  // CTA pairs (multicast weight tiles): two consecutive m tiles must belong to the same weight group / A matrix
  int cluster = 1;
  if (!use_halo && !boxed && (cluster_mode() != 0 || mma2_mode() != 0) && block_n >= 128 && num_m_tiles % 2 == 0 &&
      (wgroups == 1 || wg_tiles % 2 == 0) && (a_mod_tiles == 0 || a_mod_tiles % 2 == 0))
    cluster = (mma2_mode() != 0 && pl->warp_epi && (mode == EPI_PLAIN || mode == EPI_STATS || mode == EPI_BNBWD)) ? 3 : 2;
  pl->cluster = cluster;
  if (use_halo) {  // one CTA per SM, each walking 256-pixel tiles (two image rows x 128 columns)
    pl->units = geo.NB * (H / 2) * (W / 128) * pl->num_n_tiles;
    pl->grid = pl->units < num_sms() ? pl->units : num_sms();
  } else {
    const int cl = cluster > 1 ? 2 : 1;
    pl->units = (num_m_tiles / cl) * pl->num_n_tiles;
    const int slots = num_sms() / cl;
    pl->grid = (pl->units < slots ? pl->units : slots) * cl;
  }
  return IRFD_OK;
}

extern "C" int irfd_conv_gemm_plan(int n, int h, int w, int cin, int cout, int ksize, int mode, int wgroups,
                                   int a_shared, int force_block_n, int* out_host) {
  IRFD_CHECK_ARG(out_host != nullptr, "conv_gemm_plan: null output");
  ConvPlan pl;
  const int rc = conv_gemm_plan(n, h, w, cin, cout, ksize, mode, wgroups, a_shared, force_block_n, &pl);
  if (rc != IRFD_OK) return rc;
  const int v[9] = {pl.use_halo, pl.geo.boxed, pl.block_n, pl.cluster, pl.warp_epi,
                    pl.num_m_tiles, pl.num_n_tiles, pl.units, pl.grid};
  for (int i = 0; i < 9; ++i) out_host[i] = v[i];
  return IRFD_OK;
}

static int conv_gemm_impl(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize, void* out,
                          void* out2, void* out_lo, int mode, const float* bias, const float* nw, const float* noise,
                          const float* sp1, const float* s1, float* stat_sum, float* stat_sq, const void* res, int relu,
                          int force_block_n, cudaStream_t stream, int wgroups = 1, int a_shared = 0,
                          const BnBwdFold* fold = nullptr) {
  IRFD_CHECK_ARG(x && wk && out, "conv_gemm: null pointer");
  ConvPlan pl;
  {
    const int rc = conv_gemm_plan(n, h, w, cin, cout, ksize, mode, wgroups, a_shared, force_block_n, &pl);
    if (rc != IRFD_OK) return rc;
  }
  const TileGeom& geo = pl.geo;
  const bool boxed = geo.boxed != 0;
  const int m_total = n * h * w;
  const int H = geo.H, W = geo.W, NB = geo.NB;
  const int tw = geo.tw, th = geo.th, tn = geo.tn;
  const bool use_halo = pl.use_halo != 0;
  const int block_n = pl.block_n, cluster = pl.cluster;

  ConvGemmArgs a;
  a.M_total = m_total;
  a.N_total = cout;
  a.num_m_tiles = pl.num_m_tiles;
  a.num_n_tiles = pl.num_n_tiles;
  a.box_tw = tw;
  a.box_th = th;
  a.box_tn = tn;
  a.box_tiles_w = geo.tiles_w;
  a.box_tiles_h = geo.tiles_h;
  a.taps = ksize * ksize;
  a.kw = ksize;
  a.pad = ksize / 2;
  a.cin_chunks = cin / 64;
  a.H = H; a.W = W; a.HW = h * w; a.B = n;
  a.bias = bias; a.nw = nw; a.noise = noise; a.sp1 = sp1; a.s1 = s1;
  a.stat_sum = stat_sum; a.stat_sq = stat_sq;
  a.res = reinterpret_cast<const __nv_bfloat16*>(res);
  a.y_lo = reinterpret_cast<__nv_bfloat16*>(out_lo);
  a.wg_tiles = wgroups > 1 ? a.num_m_tiles / wgroups : 0x7fffffff;
  a.a_mod_tiles = a_shared ? a.num_m_tiles / wgroups : 0;
  a.relu = relu;
  if (mode == EPI_AFFINE) IRFD_CHECK_ARG(bias && nw, "conv_gemm: AFFINE mode needs scale and shift");
  if (mode == EPI_STYLE) {
    IRFD_CHECK_ARG(bias && nw && noise && sp1 && s1 && out2, "conv_gemm: STYLE mode needs bias/nw/noise/sp1/s1/out2");
    IRFD_CHECK_ARG(h * w >= 64, "conv_gemm: STYLE mode needs >= 64 pixels per image");
  }
  if (mode == EPI_STATS) IRFD_CHECK_ARG(stat_sum && stat_sq, "conv_gemm: STATS mode needs stat buffers");
  a.warp_epi = pl.warp_epi;
  a.bn_z = nullptr;
  a.bn_mean = a.bn_rstd = nullptr;
  for (int i = 0; i < 4; ++i) a.bn_gamma[i] = a.bn_beta[i] = nullptr;
  a.sg_tiles = 0x7fffffff;
  a.bn_g2 = nullptr;
  a.bn_bits = nullptr;
  if (mode == EPI_BNBWD || mode == EPI_BNBWD_RES) {
    IRFD_CHECK_ARG(fold && fold->z && fold->mean && fold->rstd && stat_sum,
                   "conv_gemm: BNBWD modes need z, mean, rstd and the partial buffer");
    if (mode == EPI_BNBWD) IRFD_CHECK_ARG(fold->gamma && fold->beta, "conv_gemm: BNBWD mode needs gamma and beta");
    if (mode == EPI_BNBWD_RES)
      IRFD_CHECK_ARG(fold->g2 && fold->bits && cout % 8 == 0, "conv_gemm: BNBWD_RES mode needs g2 and the mask plane");
    IRFD_CHECK_ARG(wgroups <= 4 && m_total % 128 == 0 && fold->stat_groups >= wgroups &&
                       fold->stat_groups % wgroups == 0 && a.num_m_tiles % fold->stat_groups == 0,
                   "conv_gemm: BNBWD needs whole 128-pixel tiles per statistic group (%d tiles, %d groups, %d sets)",
                   a.num_m_tiles, fold->stat_groups, wgroups);
    a.bn_z = reinterpret_cast<const __nv_bfloat16*>(fold->z);
    a.bn_mean = fold->mean;
    a.bn_rstd = fold->rstd;
    for (int i = 0; i < wgroups && mode == EPI_BNBWD; ++i) {
      IRFD_CHECK_ARG(fold->gamma[i] && fold->beta[i], "conv_gemm: BNBWD gamma/beta pointer %d is null", i);
      a.bn_gamma[i] = fold->gamma[i];
      a.bn_beta[i] = fold->beta[i];
    }
    a.bn_g2 = reinterpret_cast<const __nv_bfloat16*>(fold->g2);
    a.bn_bits = reinterpret_cast<const uint8_t*>(fold->bits);
    a.sg_tiles = a.num_m_tiles / fold->stat_groups;
  }

  CUtensorMap ma, mb, mo, mo2;
  {
    const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)W, (uint64_t)H, (uint64_t)NB};
    const uint64_t str[3] = {(uint64_t)cin * 2, (uint64_t)W * cin * 2, (uint64_t)H * W * cin * 2};
    uint32_t box[4] = {64, (uint32_t)tw, (uint32_t)th, (uint32_t)tn};
    if (use_halo) {
      box[1] = kHaloCols;
      box[2] = kHaloRows;
      box[3] = 1;
    }
    int rc = make_tmap_bf16(&ma, x, 4, dims, str, box, true);
    if (rc) return rc;
  }
  {
    const uint64_t ktot = (uint64_t)a.taps * cin;
    const uint64_t dims[2] = {ktot, (uint64_t)cout * wgroups};
    const uint64_t str[1] = {ktot * 2};
    const uint32_t box[2] = {64, (uint32_t)(block_n / (cluster > 1 ? 2 : 1))};  // a CTA pair loads half a weight tile each
    int rc = make_tmap_bf16(&mb, wk, 2, dims, str, box, true);
    if (rc) return rc;
  }
  if (boxed) {  // the epilogue stores each tile as one 4-D box over [NB][H][W][cout]; TMA clips what lies outside
    const uint64_t dims[4] = {(uint64_t)cout, (uint64_t)W, (uint64_t)H, (uint64_t)NB};
    const uint64_t str[3] = {(uint64_t)cout * 2, (uint64_t)W * cout * 2, (uint64_t)H * W * cout * 2};
    const uint32_t box[4] = {64, (uint32_t)tw, (uint32_t)th, (uint32_t)tn};
    const int rc = make_tmap_bf16(&mo, out, 4, dims, str, box, true);
    if (rc) return rc;
    if (mode == EPI_PLAIN) return dispatch_box<EPI_PLAIN>(block_n, ma, mb, mo, a, pl.grid, stream);
    return dispatch_box<EPI_AFFINE>(block_n, ma, mb, mo, a, pl.grid, stream);
  }
  {
    const uint64_t dims[2] = {(uint64_t)cout, (uint64_t)m_total};
    const uint64_t str[1] = {(uint64_t)cout * 2};
    const uint32_t box[2] = {64, 128};
    int rc = make_tmap_bf16(&mo, out, 2, dims, str, box, true);
    if (rc) return rc;
    if (mode == EPI_STYLE) {
      rc = make_tmap_bf16(&mo2, out2 ? out2 : out, 2, dims, str, box, true);
    } else {  // the per-warp epilogue stores [32 pixels x 64 channels] slabs
      const uint32_t slab_box[2] = {64, 32};
      rc = make_tmap_bf16(&mo2, out, 2, dims, str, slab_box, true);
    }
    if (rc) return rc;
  }
  if (use_halo) {
    HaloArgs hargs;
    hargs.wsegs = W / 128;
    hargs.hpairs = H / 2;
    hargs.total_tiles = pl.units;
    switch (mode) {
      case EPI_PLAIN: return dispatch_halo<EPI_PLAIN>(block_n, ma, mb, mo, mo2, a, hargs, pl.grid, stream);
      case EPI_STATS: return dispatch_halo<EPI_STATS>(block_n, ma, mb, mo, mo2, a, hargs, pl.grid, stream);
      case EPI_STYLE: return dispatch_halo<EPI_STYLE>(block_n, ma, mb, mo, mo2, a, hargs, pl.grid, stream);
      case EPI_AFFINE: return dispatch_halo<EPI_AFFINE>(block_n, ma, mb, mo, mo2, a, hargs, pl.grid, stream);
    }
    return IRFD_ERR_INVALID_ARGUMENT;
  }
  switch (mode) {
    case EPI_PLAIN: return dispatch_block_n<EPI_PLAIN>(block_n, ma, mb, mo, mo2, a, pl.grid, cluster, stream);
    case EPI_STATS: return dispatch_block_n<EPI_STATS>(block_n, ma, mb, mo, mo2, a, pl.grid, cluster, stream);
    case EPI_STYLE: return dispatch_block_n<EPI_STYLE>(block_n, ma, mb, mo, mo2, a, pl.grid, cluster, stream);
    case EPI_AFFINE: return dispatch_block_n<EPI_AFFINE>(block_n, ma, mb, mo, mo2, a, pl.grid, cluster, stream);
    case EPI_BNBWD: return dispatch_block_n<EPI_BNBWD>(block_n, ma, mb, mo, mo2, a, pl.grid, cluster, stream);
    case EPI_BNBWD_RES: return dispatch_block_n<EPI_BNBWD_RES>(block_n, ma, mb, mo, mo2, a, pl.grid, cluster, stream);
  }
  return IRFD_ERR_INVALID_ARGUMENT;
}

extern "C" int irfd_conv_gemm(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize,
                              void* out, void* out2, int mode, const float* bias, const float* nw, const float* noise,
                              const float* sp1, const float* s1, float* stat_sum, float* stat_sq, int force_block_n,
                              cudaStream_t stream) {
  IRFD_CHECK_ARG(mode >= 0 && mode <= 2, "conv_gemm: bad mode %d", mode);
  return conv_gemm_impl(x, n, h, w, cin, wk, cout, ksize, out, out2, nullptr, mode, bias, nw, noise, sp1, s1, stat_sum,
                        stat_sq, nullptr, 0, force_block_n, stream);
}

extern "C" int irfd_conv_gemm_style_split(const void* x, int n, int h, int w, int cin, const void* wk, int cout,
                                          int ksize, void* out_a, void* out_y, void* out_y_lo, const float* bias,
                                          const float* nw, const float* noise, const float* sp1, const float* s1,
                                          int force_block_n, cudaStream_t stream) {
  IRFD_CHECK_ARG(out_y_lo != nullptr, "conv_gemm_style_split: out_y_lo is required");
  return conv_gemm_impl(x, n, h, w, cin, wk, cout, ksize, out_a, out_y, out_y_lo, EPI_STYLE, bias, nw, noise, sp1, s1,
                        nullptr, nullptr, nullptr, 0, force_block_n, stream);
}

// Grouped variants: `wgroups` weight sets stacked along the rows of wk ([wgroups * cout][k*k*cin]), the n images split
// evenly group-major; a_shared != 0: x holds ONE group's pixels ([n / wgroups] images), read by every group.
extern "C" int irfd_conv_gemm_grouped(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize,
                                      void* out, int mode, float* stat_sum, float* stat_sq, int wgroups, int a_shared,
                                      int force_block_n, cudaStream_t stream) {
  IRFD_CHECK_ARG(mode == EPI_PLAIN || mode == EPI_STATS, "conv_gemm_grouped: mode must be 0 (plain) or 1 (stats)");
  return conv_gemm_impl(x, n, h, w, cin, wk, cout, ksize, out, nullptr, nullptr, mode, nullptr, nullptr, nullptr,
                        nullptr, nullptr, stat_sum, stat_sq, nullptr, 0, force_block_n, stream, wgroups, a_shared);
}

// Data gradient of a conv whose input was relu(BN(z)), with that BatchNorm's backward reduce pass folded into the
// epilogue: out = dgrad * (gamma*xhat + beta > 0) (bf16), partial[m tile][2][cout] = per-tile sums of g and g*xhat.
// Finish with irfd_bn_backward_finish_sets.  stat_groups = TOTAL statistic groups of z (a multiple of wgroups).
extern "C" int irfd_conv_gemm_bnbwd_grouped(const void* x, int n, int h, int w, int cin, const void* wk, int cout,
                                            int ksize, void* out, const void* bn_z, const float* bn_mean,
                                            const float* bn_rstd, const float* const* bn_gamma,
                                            const float* const* bn_beta, float* partial, int stat_groups, int wgroups,
                                            int force_block_n, cudaStream_t stream) {
  IRFD_CHECK_ARG(wgroups >= 1 && wgroups <= 4, "conv_gemm_bnbwd: 1..4 weight groups");
  const BnBwdFold fold{bn_z, bn_mean, bn_rstd, bn_gamma, bn_beta, nullptr, nullptr, stat_groups};
  return conv_gemm_impl(x, n, h, w, cin, wk, cout, ksize, out, nullptr, nullptr, EPI_BNBWD, nullptr, nullptr, nullptr,
                        nullptr, nullptr, partial, nullptr, nullptr, 0, force_block_n, stream, wgroups, 0, &fold);
}

// The same for the BatchNorm that closes a Bottleneck: out = (dgrad + g2) * mask, mask from the bit plane of
// irfd_bn_apply_sets ([pixels][cout/8]); out is the masked gradient both bn3's backward and the shortcut consume.
extern "C" int irfd_conv_gemm_bnbwd_res_grouped(const void* x, int n, int h, int w, int cin, const void* wk, int cout,
                                                int ksize, void* out, const void* bn_z, const float* bn_mean,
                                                const float* bn_rstd, const void* g2, const void* mask_bits,
                                                float* partial, int stat_groups, int wgroups, int force_block_n,
                                                cudaStream_t stream) {
  IRFD_CHECK_ARG(wgroups >= 1 && wgroups <= 4, "conv_gemm_bnbwd_res: 1..4 weight groups");
  const BnBwdFold fold{bn_z, bn_mean, bn_rstd, nullptr, nullptr, g2, mask_bits, stat_groups};
  return conv_gemm_impl(x, n, h, w, cin, wk, cout, ksize, out, nullptr, nullptr, EPI_BNBWD_RES, nullptr, nullptr,
                        nullptr, nullptr, nullptr, partial, nullptr, nullptr, 0, force_block_n, stream, wgroups, 0,
                        &fold);
}

extern "C" int irfd_conv_gemm_affine_grouped(const void* x, int n, int h, int w, int cin, const void* wk, int cout,
                                             int ksize, void* out, const float* scale, const float* shift,
                                             const void* res, int relu, int wgroups, int a_shared, int force_block_n,
                                             cudaStream_t stream) {
  return conv_gemm_impl(x, n, h, w, cin, wk, cout, ksize, out, nullptr, nullptr, EPI_AFFINE, shift, scale, nullptr,
                        nullptr, nullptr, nullptr, nullptr, res, relu, force_block_n, stream, wgroups, a_shared);
}

extern "C" int irfd_conv_gemm_affine(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize,
                                     void* out, const float* scale, const float* shift, const void* res, int relu,
                                     int force_block_n, cudaStream_t stream) {
  return conv_gemm_impl(x, n, h, w, cin, wk, cout, ksize, out, nullptr, nullptr, EPI_AFFINE, shift, scale, nullptr, nullptr,
                        nullptr, nullptr, nullptr, res, relu, force_block_n, stream);
}
