// Spectral normalisation of the discriminator's weights (torch.nn.utils.spectral_norm with n_power_iterations = 1,
// eps = 1e-12, styleganv1.py:643-654) for every layer of one D call in a fixed number of launches.
//   W is weight_orig viewed as [rows, cols] (conv: [Cout, Cin*k*k], dense: [out, in]); u [rows], v [cols].
//   forward, train  : t = W^T u                                   (sn_wtu_kernel, column tiles)
//                     v = t / max(|t|, eps);  wv = W v              (sn_wv_kernel, one warp per row)
//                     u = wv / max(|wv|, eps);  sigma = u . wv;  W_sn = W / sigma   (sn_scale_kernel)
//   forward, eval   : wv = W v;  sigma = u . wv;  W_sn = W / sigma  (stored u and v, no update)
//   backward        : dW = (G - <G, W_sn> u v^T) / sigma            (u, v constants, as in torch)
// Every reduction runs in a fixed order without atomics: each block writes its partial, and every consumer of a
// per-layer total re-sums the same partials in the same order, so the results are bit-reproducible.
#include "host_util.h"

namespace irfd {

constexpr int kSnMaxLayers = 32;
constexpr int kSnThreads = 256;
constexpr int kSnColTile = 32;                       // columns per sn_wtu block (8 row lanes x 32 columns)
constexpr int kSnRowsPerBlk = kSnThreads / 32;       // rows per sn_wv block (one warp per row)
constexpr int kSnElemChunk = kSnThreads * 32;        // weight elements per sn_scale / backward block

struct SnLayer {
  const float* w;      // forward: W (weight_orig);  backward: G (gradient w.r.t. W_sn)
  const float* w2;     // backward: W_sn
  float* u;            // forward: the module buffer;  backward: the saved u
  float* v;
  float* out;          // forward: W_sn;  backward: dW
  float* u_save;       // forward only, optional: copies of the u / v this call used (what the backward needs)
  float* v_save;
  int rows, cols;
  int blk_col, blk_row, blk_elem;  // first block of this layer in each kernel's grid
  int t_off, wv_off;               // offsets into the t [sum cols] and wv [sum rows] workspaces
};

struct SnTable {
  SnLayer l[kSnMaxLayers];
  int n;
  float eps;
};

__device__ __forceinline__ int sn_find(const SnTable& T, int b, int which) {
  int i = 0;
  for (int j = 1; j < T.n; ++j) {
    const int first = which == 0 ? T.l[j].blk_col : (which == 1 ? T.l[j].blk_row : T.l[j].blk_elem);
    if (b >= first) i = j;
  }
  return i;
}

__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// sum of p[0 .. n) by one block in a fixed order; the result is returned to every thread
__device__ float block_sum(const float* __restrict__ p, int n, float* red) {
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += p[i];
  s = warp_sum(s);
  __syncthreads();  // red may still be read by a previous call
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int w = 0; w < kSnThreads / 32; ++w) t += red[w];
  return t;
}

// t = W^T u for a 32-column tile; partial |t|^2 per block
__global__ void __launch_bounds__(kSnThreads) sn_wtu_kernel(SnTable T, float* __restrict__ t, float* __restrict__ pt2) {
  __shared__ float red[kSnRowsPerBlk][kSnColTile];
  const int li = sn_find(T, blockIdx.x, 0);
  const SnLayer& L = T.l[li];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = (blockIdx.x - L.blk_col) * kSnColTile + tx;
  float acc = 0.f;
  if (col < L.cols) {
    const float* wp = L.w + col;
#pragma unroll 4
    for (int r = ty; r < L.rows; r += kSnRowsPerBlk) acc += __ldg(wp + (size_t)r * L.cols) * __ldg(L.u + r);
  }
  red[ty][tx] = acc;
  __syncthreads();
  if (ty == 0) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kSnRowsPerBlk; ++k) s += red[k][tx];
    if (col < L.cols) t[L.t_off + col] = s;
    const float sq = warp_sum(col < L.cols ? s * s : 0.f);
    if (tx == 0) pt2[blockIdx.x] = sq;
  }
}

// wv = W v for 8 rows (train: v = t / max(|t|, eps), written back by the layer's first block); partial |wv|^2
__global__ void __launch_bounds__(kSnThreads) sn_wv_kernel(SnTable T, int train, const float* __restrict__ t,
                                                            const float* __restrict__ pt2, float* __restrict__ wv,
                                                            float* __restrict__ pwv2) {
  __shared__ float red[kSnThreads / 32];
  const int li = sn_find(T, blockIdx.x, 1);
  const SnLayer& L = T.l[li];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float inv_nt = 0.f;
  if (train) {
    const int ncb = (L.cols + kSnColTile - 1) / kSnColTile;
    inv_nt = __fdiv_rn(1.f, fmaxf(__fsqrt_rn(block_sum(pt2 + L.blk_col, ncb, red)), T.eps));
  }
  const float* tv = train ? t + L.t_off : L.v;
  const int local = blockIdx.x - L.blk_row;
  if (train && local == 0) {
    for (int k = threadIdx.x; k < L.cols; k += blockDim.x) {
      const float vk = tv[k] * inv_nt;
      L.v[k] = vk;
      if (L.v_save) L.v_save[k] = vk;
    }
  } else if (!train && local == 0 && L.v_save) {
    for (int k = threadIdx.x; k < L.cols; k += blockDim.x) L.v_save[k] = L.v[k];
  }
  const int r = local * kSnRowsPerBlk + warp;
  float s = 0.f;
  if (r < L.rows) {
    const float* wp = L.w + (size_t)r * L.cols;
    if (train) {
#pragma unroll 4
      for (int k = lane; k < L.cols; k += 32) s += __ldg(wp + k) * (tv[k] * inv_nt);
    } else {
#pragma unroll 4
      for (int k = lane; k < L.cols; k += 32) s += __ldg(wp + k) * tv[k];
    }
    s = warp_sum(s);
    if (lane == 0) wv[L.wv_off + r] = s;
  }
  __syncthreads();
  if (lane == 0) red[warp] = r < L.rows ? s * s : 0.f;
  __syncthreads();
  if (threadIdx.x == 0) {
    float q = 0.f;
#pragma unroll
    for (int w = 0; w < kSnThreads / 32; ++w) q += red[w];
    pwv2[blockIdx.x] = q;
  }
}

// sigma (and, in train mode, the new u); W_sn = W / sigma for one chunk of the layer
__global__ void __launch_bounds__(kSnThreads) sn_scale_kernel(SnTable T, int train, const float* __restrict__ wv,
                                                               const float* __restrict__ pwv2, float* __restrict__ sigma) {
  __shared__ float red[kSnThreads / 32];
  const int li = sn_find(T, blockIdx.x, 2);
  const SnLayer& L = T.l[li];
  const float* wvl = wv + L.wv_off;
  float nrm = 1.f;
  if (train) {
    const int nrb = (L.rows + kSnRowsPerBlk - 1) / kSnRowsPerBlk;
    nrm = fmaxf(__fsqrt_rn(block_sum(pwv2 + L.blk_row, nrb, red)), T.eps);
  }
  float s = 0.f;
  for (int r = threadIdx.x; r < L.rows; r += blockDim.x) {
    const float ur = train ? __fdiv_rn(wvl[r], nrm) : L.u[r];
    s += ur * wvl[r];
  }
  s = warp_sum(s);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  float sg = 0.f;
#pragma unroll
  for (int w = 0; w < kSnThreads / 32; ++w) sg += red[w];
  const int local = blockIdx.x - L.blk_elem;
  if (local == 0) {
    if (threadIdx.x == 0) sigma[li] = sg;
    for (int r = threadIdx.x; r < L.rows; r += blockDim.x) {
      const float ur = train ? __fdiv_rn(wvl[r], nrm) : L.u[r];
      if (train) L.u[r] = ur;
      if (L.u_save) L.u_save[r] = ur;
    }
  }
  const size_t n = (size_t)L.rows * L.cols;
  const size_t e0 = (size_t)local * kSnElemChunk;
  const size_t e1 = e0 + kSnElemChunk < n ? e0 + kSnElemChunk : n;
  for (size_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) L.out[e] = __fdiv_rn(__ldg(L.w + e), sg);
}

// backward pass 1: partial <G, W_sn> per chunk
__global__ void __launch_bounds__(kSnThreads) sn_bwd_dot_kernel(SnTable T, float* __restrict__ pdot) {
  __shared__ float red[kSnThreads / 32];
  const int li = sn_find(T, blockIdx.x, 2);
  const SnLayer& L = T.l[li];
  const size_t n = (size_t)L.rows * L.cols;
  const size_t e0 = (size_t)(blockIdx.x - L.blk_elem) * kSnElemChunk;
  const size_t e1 = e0 + kSnElemChunk < n ? e0 + kSnElemChunk : n;
  float s = 0.f;
  for (size_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) s += __ldg(L.w + e) * __ldg(L.w2 + e);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float q = 0.f;
#pragma unroll
    for (int w = 0; w < kSnThreads / 32; ++w) q += red[w];
    pdot[blockIdx.x] = q;
  }
}

// backward pass 2: dW = (G - <G, W_sn> u v^T) / sigma
__global__ void __launch_bounds__(kSnThreads) sn_bwd_apply_kernel(SnTable T, const float* __restrict__ pdot,
                                                                   const float* __restrict__ sigma) {
  __shared__ float red[kSnThreads / 32];
  const int li = sn_find(T, blockIdx.x, 2);
  const SnLayer& L = T.l[li];
  const size_t n = (size_t)L.rows * L.cols;
  const int nb = (int)((n + kSnElemChunk - 1) / kSnElemChunk);
  const float c = block_sum(pdot + L.blk_elem, nb, red);
  const float sg = sigma[li];
  const size_t e0 = (size_t)(blockIdx.x - L.blk_elem) * kSnElemChunk;
  const size_t e1 = e0 + kSnElemChunk < n ? e0 + kSnElemChunk : n;
  for (size_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
    const int r = (int)(e / L.cols), k = (int)(e - (size_t)r * L.cols);
    L.out[e] = __fdiv_rn(__ldg(L.w + e) - c * L.u[r] * L.v[k], sg);
  }
}

// Fills the per-layer geometry of T (block ranges, workspace offsets); returns the workspace floats needed.
static long long sn_plan(SnTable& T, const int* rows, const int* cols, int n, int* nblk_col, int* nblk_row,
                         int* nblk_elem) {
  int bc = 0, br = 0, be = 0, toff = 0, wvoff = 0;
  for (int i = 0; i < n; ++i) {
    SnLayer& L = T.l[i];
    L.rows = rows[i];
    L.cols = cols[i];
    L.blk_col = bc;
    L.blk_row = br;
    L.blk_elem = be;
    L.t_off = toff;
    L.wv_off = wvoff;
    bc += (cols[i] + kSnColTile - 1) / kSnColTile;
    br += (rows[i] + kSnRowsPerBlk - 1) / kSnRowsPerBlk;
    be += (int)(((long long)rows[i] * cols[i] + kSnElemChunk - 1) / kSnElemChunk);
    toff += cols[i];
    wvoff += rows[i];
  }
  T.n = n;
  *nblk_col = bc;
  *nblk_row = br;
  *nblk_elem = be;
  const long long fwd = (long long)toff + bc + wvoff + br;
  return fwd > be ? fwd : be;
}

static int sn_check_shapes(const int* rows, const int* cols, int n, const char* what) {
  IRFD_CHECK_ARG(rows && cols, "%s: null rows/cols array", what);
  IRFD_CHECK_ARG(n >= 1 && n <= kSnMaxLayers, "%s: 1..%d layers per call", what, kSnMaxLayers);
  long long tot_rows = 0, tot_cols = 0;
  for (int i = 0; i < n; ++i) {
    IRFD_CHECK_ARG(rows[i] > 0 && cols[i] > 0, "%s: layer %d has an empty [%d, %d] matrix", what, i, rows[i], cols[i]);
    IRFD_CHECK_ARG((long long)rows[i] * cols[i] < (1LL << 31), "%s: layer %d has more than 2^31 elements", what, i);
    tot_rows += rows[i];
    tot_cols += cols[i];
  }
  IRFD_CHECK_ARG(tot_rows < (1LL << 31) && tot_cols < (1LL << 31), "%s: too many rows/columns in one call", what);
  return IRFD_OK;
}

}  // namespace irfd

using namespace irfd;

extern "C" long long irfd_spectral_norm_workspace_bytes(const int* rows_host, const int* cols_host, int nlayers) {
  if (sn_check_shapes(rows_host, cols_host, nlayers, "spectral_norm_workspace_bytes") != IRFD_OK) return -1;
  SnTable T;
  int bc, br, be;
  return 4 * sn_plan(T, rows_host, cols_host, nlayers, &bc, &br, &be);
}

extern "C" int irfd_spectral_norm_fwd(const float* const* w, float* const* u, float* const* v, float* const* w_sn,
                                      float* u_save, float* v_save, float* sigma, const int* rows_host,
                                      const int* cols_host, int nlayers, int power_iteration, float eps,
                                      void* workspace, long long workspace_bytes, cudaStream_t stream) {
  const int rc = sn_check_shapes(rows_host, cols_host, nlayers, "spectral_norm_fwd");
  if (rc != IRFD_OK) return rc;
  IRFD_CHECK_ARG(w && u && v && w_sn && sigma && workspace, "spectral_norm_fwd: null pointer");
  IRFD_CHECK_ARG(eps > 0.f, "spectral_norm_fwd: eps must be positive");
  SnTable T;
  int bc, br, be;
  const long long need = 4 * sn_plan(T, rows_host, cols_host, nlayers, &bc, &br, &be);
  IRFD_CHECK_ARG(workspace_bytes >= need, "spectral_norm_fwd: workspace too small (%lld < %lld bytes)",
                 workspace_bytes, need);
  long long uo = 0, vo = 0;
  for (int i = 0; i < nlayers; ++i) {
    IRFD_CHECK_ARG(w[i] && u[i] && v[i] && w_sn[i], "spectral_norm_fwd: null pointer in layer %d", i);
    SnLayer& L = T.l[i];
    L.w = w[i];
    L.w2 = nullptr;
    L.u = u[i];
    L.v = v[i];
    L.out = w_sn[i];
    L.u_save = u_save ? u_save + uo : nullptr;
    L.v_save = v_save ? v_save + vo : nullptr;
    uo += L.rows;
    vo += L.cols;
  }
  T.eps = eps;
  float* ws = reinterpret_cast<float*>(workspace);
  float* t = ws;
  float* pt2 = t + vo;
  float* wv = pt2 + bc;
  float* pwv2 = wv + uo;
  if (power_iteration) {
    sn_wtu_kernel<<<bc, kSnThreads, 0, stream>>>(T, t, pt2);
    IRFD_CHECK_LAUNCH();
  }
  sn_wv_kernel<<<br, kSnThreads, 0, stream>>>(T, power_iteration ? 1 : 0, t, pt2, wv, pwv2);
  IRFD_CHECK_LAUNCH();
  sn_scale_kernel<<<be, kSnThreads, 0, stream>>>(T, power_iteration ? 1 : 0, wv, pwv2, sigma);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}

extern "C" int irfd_spectral_norm_bwd(const float* const* g, const float* const* w_sn, const float* u, const float* v,
                                      const float* sigma, float* const* dw, const int* rows_host, const int* cols_host,
                                      int nlayers, void* workspace, long long workspace_bytes, cudaStream_t stream) {
  const int rc = sn_check_shapes(rows_host, cols_host, nlayers, "spectral_norm_bwd");
  if (rc != IRFD_OK) return rc;
  IRFD_CHECK_ARG(g && w_sn && u && v && sigma && dw && workspace, "spectral_norm_bwd: null pointer");
  SnTable T;
  int bc, br, be;
  const long long need = 4 * sn_plan(T, rows_host, cols_host, nlayers, &bc, &br, &be);
  IRFD_CHECK_ARG(workspace_bytes >= need, "spectral_norm_bwd: workspace too small (%lld < %lld bytes)",
                 workspace_bytes, need);
  long long uo = 0, vo = 0;
  for (int i = 0; i < nlayers; ++i) {
    IRFD_CHECK_ARG(g[i] && w_sn[i] && dw[i], "spectral_norm_bwd: null pointer in layer %d", i);
    SnLayer& L = T.l[i];
    L.w = g[i];
    L.w2 = w_sn[i];
    L.u = const_cast<float*>(u) + uo;
    L.v = const_cast<float*>(v) + vo;
    L.out = dw[i];
    L.u_save = L.v_save = nullptr;
    uo += L.rows;
    vo += L.cols;
  }
  T.eps = 0.f;
  float* pdot = reinterpret_cast<float*>(workspace);
  sn_bwd_dot_kernel<<<be, kSnThreads, 0, stream>>>(T, pdot);
  IRFD_CHECK_LAUNCH();
  sn_bwd_apply_kernel<<<be, kSnThreads, 0, stream>>>(T, pdot, sigma);
  IRFD_CHECK_LAUNCH();
  return IRFD_OK;
}
