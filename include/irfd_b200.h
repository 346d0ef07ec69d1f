/* irfd_b200.h — C ABI of libirfd_b200.so: the sm_100a kernels behind the IRFD hot path.
 *
 * The reference (johndpope/SPEAK-hack) has no FFI layer: its hot path is Python `nn.Module` code calling ATen.
 * Each entry point below therefore names the reference call site(s) whose arithmetic it replaces.  The Python host
 * (speak_hack_b200/*.py) keeps the reference's module surface (IRFD, StyleGenerator, ... — model.py:28-126,
 * styleganv1.py:448-635) and calls these functions through ctypes with raw device pointers and the current stream.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - activations are NHWC bf16 ("pixels x channels"); parameters/gradients handed back to PyTorch are fp32 in the
 *     reference's own layouts (OIHW conv weights, [out,in] linear weights);
 *   - functions enqueue work on `stream` and return immediately; they never allocate, never synchronise and keep no
 *     global state beyond immutable lazily-created function attributes;
 *   - return value: IRFD_OK (0) or a negative error code; `irfd_last_error()` gives the message (thread-local).
 *   - there is no CPU fallback: on a machine without an sm_100 GPU every launch returns IRFD_ERR_CUDA.
 */
#ifndef IRFD_B200_H_
#define IRFD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IRFD_ABI_VERSION 1

#define IRFD_OK 0
#define IRFD_ERR_INVALID_ARGUMENT (-1)
#define IRFD_ERR_CUDA (-2)

/* Opaque CUDA stream handle (cudaStream_t). */
typedef struct CUstream_st* irfd_stream_t;

int irfd_abi_version(void);
const char* irfd_last_error(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution, stride 1, "same" padding, ksize in {1, 3}  (tcgen05 + TMEM + TMA).
 * Replaces: nn.Conv2d 3x3 of SynthesisBlock (styleganv1.py:615-616, 625, 630) with its ApplyNoise / leaky_relu /
 *           ApplyStyle tail (styleganv1.py:453-456, 463-468, 626-633) fused as the epilogue (mode 2);
 *           the stride-1 convs of torchvision Bottleneck (torchvision/models/resnet.py:143-155) with the batch
 *           statistics of the following BatchNorm2d gathered in the epilogue (mode 1);
 *           every dgrad of those convs (mode 0, weights pre-flipped by irfd_pack_conv_weight).
 *   x      [n,h,w,cin]  bf16 NHWC        wk  [cout][ksize*ksize][cin] bf16 (tap-major K)
 *   out    [n,h,w,cout] bf16             out2 same shape (mode 2 only: out = a = lrelu(z), out2 = styled y)
 *   mode 0: out = acc (+ bias[cout] if bias != NULL)
 *   mode 1: out = acc; stat_sum/stat_sq [m_tiles][cout] fp32 per-128-pixel-tile partial sums (of the stored bf16)
 *   mode 2: z = acc + bias[c] + nw[c]*noise[pixel]; a = lrelu(z, 0.2); y = a*sp1[b,c] + s1[b,c]
 *           noise [n*h*w] fp32, sp1/s1 [n][cout] fp32 (sp1 = style0 + 1)
 *   force_block_n: 0 = heuristic, else 64/128/256.
 * Shape rules: cin % 64 == 0, cout % 64 == 0.  Two pixel-tile geometries (irfd_conv_gemm_geometry says which one a
 * shape gets):
 *   linear: 128 consecutive NHWC pixels are one tile — every pointwise conv of >= 128 pixels (ragged last tile), and
 *           3x3 convs whose w divides 128 or is a multiple of 128 with 128 pixels forming whole rows / whole images.
 *           Every mode.  With wgroups > 1 each group must cover a whole number of 128-pixel tiles.
 *   boxed : every other shape (any n, h, w >= 1): a tile is a box of tw x th x tn <= 128 output pixels (w < 128:
 *           tw = w, th = min(h, 128 / w), whole images per box when th == h; w > 128: 128-pixel row segments).
 *           Modes 0 (plain) and 3 (affine) only — the eval-mode encoders' modes; the others return
 *           IRFD_ERR_INVALID_ARGUMENT.  With wgroups > 1 the image count must split evenly into the groups (3x3 only).
 */
int irfd_conv_gemm_m_tiles(int n, int h, int w);
/* Host-only tile-geometry query (no CUDA call): out_host[7] = {boxed (0 linear / 1 boxed), tw, th, tn, tiles_w,
 * tiles_h, tiles_n}; the launch has tiles_w * tiles_h * tiles_n pixel tiles (== irfd_conv_gemm_m_tiles when linear).
 * Boxed tiles are ordered image-major, then rows, then columns.  Returns IRFD_ERR_INVALID_ARGUMENT for shapes neither
 * geometry serves. */
int irfd_conv_gemm_geometry(int n, int h, int w, int ksize, int wgroups, int* out_host);
int irfd_conv_gemm(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize, void* out,
                   void* out2, int mode, const float* bias, const float* nw, const float* noise, const float* sp1,
                   const float* s1, float* stat_sum, float* stat_sq, int force_block_n, irfd_stream_t stream);

/* STYLE mode with a split-bf16 y: additionally writes out_y_lo = bf16(y - bf16(y)) so that the bilinear upsample that
 * consumes y (irfd_upsample2x_split_fwd) sees ~16 mantissa bits and the next conv's operand is rounded once, like the
 * fp32 reference's would be (styleganv1.py:623-635).  Used for the <= 32^2 layers, where the extra bytes are free. */
int irfd_conv_gemm_style_split(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize,
                               void* out_a, void* out_y, void* out_y_lo, const float* bias, const float* nw,
                               const float* noise, const float* sp1, const float* s1, int force_block_n,
                               irfd_stream_t stream);

/* Grouped launches: the three ResNet-50 encoders of IRFD (model.py:33-35, 84-90) run the same layer shapes on the same
 * images with different weights, so one launch per layer serves all three.  wk stacks `wgroups` weight sets along its
 * rows ([wgroups*cout][k*k*cin]); the n images are split evenly, group-major ([wgroups][n/wgroups] images); each
 * group must cover whole tiles (see the shape rules above).  a_shared != 0 (ksize 1 only): x holds one group's rows and is
 * read by every group (the stem's im2col matrix).  mode 0 (plain) or 1 (stats; partials stay [m_tiles][cout]).
 * The affine variant takes scale/shift as [wgroups][cout]. */
int irfd_conv_gemm_grouped(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize, void* out,
                           int mode, float* stat_sum, float* stat_sq, int wgroups, int a_shared, int force_block_n,
                           irfd_stream_t stream);
int irfd_conv_gemm_affine_grouped(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize,
                                  void* out, const float* scale, const float* shift, const void* res, int relu,
                                  int wgroups, int a_shared, int force_block_n, irfd_stream_t stream);

/* Affine variant (mode 3): y = act(acc*scale[c] + shift[c] [+ res[pixel,c]]) -> bf16; relu: 0 none, 1 ReLU,
 * 2 leaky ReLU(0.2) (the discriminator's conv + bias + leaky_relu, styleganv1.py:662-669,689-694, with scale = 1).  Folds an eval-mode
 * BatchNorm2d (scale/shift from irfd_bn_eval_affine), the ReLU and the Bottleneck residual add into the conv
 * (torchvision/models/resnet.py:143-164 in eval mode); res is NHWC bf16 of the output shape or NULL. */
int irfd_conv_gemm_affine(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize, void* out,
                          const float* scale, const float* shift, const void* res, int relu, int force_block_n,
                          irfd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Weight gradient of the same convolutions (tcgen05, both operands MN-major, deterministic split-K over pixels).
 * Replaces: autograd's convolution_backward(weight) for styleganv1.py:615-616 and torchvision resnet.py:133-141.
 *   x  [n,h,w,cin] bf16 (the conv input)   dy [n,h,w,cout] bf16 (gradient w.r.t. the raw conv output)
 *   dw [cout][cin][ksize][ksize] fp32 (OIHW, the reference parameter layout):  dw = beta*dw + grad
 *   workspace: >= irfd_wgrad_workspace_bytes(...) bytes of device scratch (fp32 split-K partials).
 *   reduce_cin/reduce_taps (0 = cin/ksize^2): how the GEMM's K index maps onto dw: k -> (tap = k / reduce_cin,
 *   c = k % reduce_cin), dw[o][c][tap], k >= reduce_cin*reduce_taps dropped.  Lets an explicit-im2col matrix (ksize 1,
 *   cin = taps*C) produce OIHW gradients for the strided convs (3x3/2: reduce_cin=C, reduce_taps=9; stem: 147, 1).
 */
long long irfd_wgrad_workspace_bytes(int n, int h, int w, int cin, int cout, int ksize);
int irfd_conv_wgrad(const void* x, const void* dy, int n, int h, int w, int cin, int cout, int ksize, float* dw,
                    float beta, int reduce_cin, int reduce_taps, void* workspace, long long workspace_bytes,
                    irfd_stream_t stream);
/* `groups` weight gradients (the same layer of the three IRFD encoders) in one launch pair: x / dy stack the groups'
 * images group-major (n = TOTAL images; 2-D row matrices pass n = 1, h = 1, w = total rows), dw is a HOST array of
 * `groups` device pointers.  x_shared != 0 (ksize 1): x holds ONE group's rows read by every group (the stem's im2col
 * matrix).  Fewer split-K partials than `groups` separate launches (the CTAs of all groups share the one wave). */
long long irfd_wgrad_workspace_bytes_grouped(int n, int h, int w, int cin, int cout, int ksize, int groups);
int irfd_conv_wgrad_grouped(const void* x, const void* dy, int n, int h, int w, int cin, int cout, int ksize,
                            float* const* dw, float beta, int reduce_cin, int reduce_taps, int groups, int x_shared,
                            void* workspace, long long workspace_bytes, irfd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * BatchNorm2d around the encoder convs (torch.nn.BatchNorm2d in torchvision Bottleneck, resnet.py:143-164).
 *   irfd_bn_finalize : per-tile partial sums (conv epilogue, mode 1) -> mean/rstd [c]; momentum update of the running
 *                      buffers applied `running_updates` times (the reference's reentrant checkpoint re-runs the
 *                      forward, model.py:84-90, SURVEY Q3); running_mean may be NULL.
 *   irfd_bn_eval_rstd: eval mode, rstd = 1/sqrt(running_var + eps).
 *   irfd_bn_apply    : out = [relu]( gamma*(z-mean)*rstd + beta  [+ res]  [or + BN2(res) when mean2 != NULL] )
 *   irfd_bn_backward : g = (g1 [+ g2]) * (act > 0 if act != NULL);  dz = gamma*rstd*(g - mean(g) - xhat*mean(g*xhat));
 *                      (batch_stats = 0, eval mode: dz = gamma*rstd*g);
 *                      dgamma/dbeta = grad_beta*old + new;  g_out (optional) receives the masked g (identity shortcut).
 * All activations [rows, c] bf16 (NHWC flattened), c % 8 == 0, c <= 2048.
 * groups >= 1: statistic groups stacked along the row axis (e.g. the source and the target half of a paired encoder
 * pass, which the reference normalises in two separate BatchNorm2d calls): tiles/count are per group, rows is the
 * total, mean/rstd are [groups][c], gamma/beta/dgamma/dbeta are shared, running buffers are updated group by group.
 */
int irfd_bn_finalize(const float* psum, const float* psq, int tiles, int c, long long count, float eps, float momentum,
                     float* mean, float* rstd, float* running_mean, float* running_var, int running_updates,
                     int groups, irfd_stream_t stream);
int irfd_bn_eval_rstd(const float* running_var, float eps, float* rstd, int c, irfd_stream_t stream);
int irfd_bn_eval_affine(const float* running_mean, const float* running_var, const float* gamma, const float* beta,
                        float eps, float* scale, float* shift, int c, irfd_stream_t stream);
/* second momentum update from saved batch mean/rstd (what the reference's checkpoint recompute does, SURVEY Q3) */
int irfd_bn_running_update(const float* mean, const float* rstd, float eps, long long count, float momentum,
                           float* running_mean, float* running_var, int c, irfd_stream_t stream);
int irfd_bn_apply(const void* z, const float* mean, const float* rstd, const float* gamma, const float* beta,
                  const void* res, const float* mean2, const float* rstd2, const float* gamma2, const float* beta2,
                  void* out, long long rows, int c, int relu, int groups, irfd_stream_t stream);
long long irfd_bn_bwd_workspace_bytes(long long rows, int c, int groups);
int irfd_bn_backward(const void* g1, const void* g2, const void* act, const void* z, const float* mean,
                     const float* rstd, const float* gamma, const float* beta, void* dz, void* g_out, float* dgamma,
                     float* dbeta, float grad_beta, int batch_stats, long long rows, int c, int groups, void* workspace,
                     long long workspace_bytes, irfd_stream_t stream);
/* mask: act != NULL -> (act > 0);  act == NULL and beta != NULL -> recomputed as gamma*xhat + beta > 0 (a BN+ReLU
 * without residual, saves reading the activation);  both NULL -> g already masked. */

/* Parameter SETS: the same BatchNorm layer of the three IRFD encoders (model.py:33-35: Ei, Ee, Ep are three
 * independent ResNet-50s fed the same images) normalised by ONE launch sequence.  The statistic groups are stacked
 * set-major along the row axis ([nsets][groups per set] x rows-per-group); batch statistics (mean/rstd, and the
 * workspace c1/c2) are per group, gamma/beta/running buffers/dgamma/dbeta per set, passed as HOST arrays of `nsets`
 * device pointers (read at call time).  irfd_bn_finalize_sets takes groups PER SET, the other two the TOTAL group count. */
int irfd_bn_eval_affine_sets(const float* const* running_mean, const float* const* running_var,
                             const float* const* gamma, const float* const* beta, float eps, float* scale, float* shift,
                             int c, int nsets, irfd_stream_t stream); /* scale/shift: [nsets][c] */
int irfd_bn_finalize_sets(const float* psum, const float* psq, int tiles, int c, long long count, float eps,
                          float momentum, float* mean, float* rstd, float* const* running_mean,
                          float* const* running_var, int running_updates, int groups, int nsets,
                          irfd_stream_t stream);
int irfd_bn_apply_sets(const void* z, const float* mean, const float* rstd, const float* const* gamma,
                       const float* const* beta, const void* res, const float* mean2, const float* rstd2,
                       const float* const* gamma2, const float* const* beta2, void* out, void* mask_bits,
                       long long rows, int c, int relu, int groups, int nsets, irfd_stream_t stream);
/* mask_bits (optional, relu only): [rows][c/8] bytes, bit t of byte j = out[row][8j+t] > 0.  irfd_bn_backward_sets takes
 * it in place of the post-ReLU tensor when act_is_bits != 0 (a sixteenth of the bytes on the widest activations).
 * With g_out != NULL the reduce pass stores the masked gradient and the apply pass reads only g_out and z. */
int irfd_bn_backward_sets(const void* g1, const void* g2, const void* act, int act_is_bits, const void* z,
                          const float* mean, const float* rstd, const float* const* gamma, const float* const* beta,
                          void* dz, void* g_out, float* const* dgamma, float* const* dbeta, float grad_beta,
                          int batch_stats, long long rows, int c, int groups, int nsets, void* workspace,
                          long long workspace_bytes, irfd_stream_t stream);

/* BatchNorm backward with the reduce pass folded into the dgrad GEMM that produces the activation gradient
 * (torchvision resnet.py:146-152: conv -> bn -> relu -> conv; the second conv's data gradient is the first BN's input):
 *   irfd_conv_gemm_bnbwd_grouped : out = dgrad(x, wk) * relu-mask(z) (bf16); partial[m tile][2][cout] = per 128-pixel
 *                                  tile sums of g and g*xhat.  stat_groups = statistic groups of z (multiple of wgroups).
 *   irfd_bn_backward_finish_sets : dgamma/dbeta from the partials, dz from the masked g and z.  tiles = partial rows per
 *                                  statistic group; workspace >= 2*groups*c floats. */
int irfd_conv_gemm_bnbwd_grouped(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize,
                                 void* out, const void* bn_z, const float* bn_mean, const float* bn_rstd,
                                 const float* const* bn_gamma, const float* const* bn_beta, float* partial,
                                 int stat_groups, int wgroups, int force_block_n, irfd_stream_t stream);
/* the BatchNorm that closes a Bottleneck: out = (dgrad + g2) * mask(mask_bits); see irfd_bn_apply_sets */
int irfd_conv_gemm_bnbwd_res_grouped(const void* x, int n, int h, int w, int cin, const void* wk, int cout, int ksize,
                                     void* out, const void* bn_z, const float* bn_mean, const float* bn_rstd,
                                     const void* g2, const void* mask_bits, float* partial, int stat_groups,
                                     int wgroups, int force_block_n, irfd_stream_t stream);
int irfd_bn_backward_finish_sets(const void* g, const void* z, const float* mean, const float* rstd,
                                 const float* const* gamma, void* dz, float* const* dgamma, float* const* dbeta,
                                 float grad_beta, int batch_stats, long long rows, int c, int groups, int nsets,
                                 const float* partial, int tiles, void* workspace, long long workspace_bytes,
                                 irfd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Layout / gather kernels for the strided ResNet convs and pooling (torchvision resnet.py:197-205, 133-137, 241).
 *   irfd_pack_conv_weight: fp32 OIHW -> bf16 GEMM operand. mode 0 fprop [o][tap][i]; 1 dgrad [i][flip(tap)][o];
 *                          2 dcol [(tap,i)][o]; 3 flat [o][kpad] (stem, k = c*49+kh*7+kw, zero padded).
 *   irfd_im2col_stem     : x NCHW fp32 [n,3,h,w] -> col [n*ho*wo][kpad] bf16 (7x7, stride 2, pad 3), w <= 579.
 *   irfd_im2col_3x3s2 / irfd_col2im_3x3s2: 3x3 stride-2 pad-1 gather [pix][tap*c + ch] and its adjoint.
 *   The forward gathers (stem, 3x3/2, 1x1/2, max pool) take any h, w and produce ceil(h/2) x ceil(w/2) outputs
 *   (torchvision's sizes); the adjoints (col2im, scatter_add, maxpool_bwd) need even h, w.
 *   irfd_subsample2 / irfd_scatter_add_s2: 1x1 stride-2 gather; adjoint fused with an add (a may be NULL).
 *   irfd_maxpool_fwd/bwd : MaxPool2d(3,2,1) with uint8 argmax taps (first maximum, like ATen).
 *   irfd_avgpool_fwd/bwd : AdaptiveAvgPool2d(1): [n,hw,c] bf16 <-> [n,c] fp32.
 */
int irfd_pack_conv_weight(const float* w, void* dst, int o, int i, int taps, int mode, int kpad, irfd_stream_t stream);
int irfd_im2col_stem(const float* x, void* col, int n, int h, int w, int kpad, irfd_stream_t stream);
int irfd_im2col_3x3s2(const void* a, void* col, int n, int h, int w, int c, irfd_stream_t stream);
int irfd_col2im_3x3s2(const void* dcol, void* dx, int n, int h, int w, int c, irfd_stream_t stream);
int irfd_subsample2(const void* a, void* out, int n, int h, int w, int c, irfd_stream_t stream);
int irfd_scatter_add_s2(const void* a, const void* b, void* out, int n, int h, int w, int c, irfd_stream_t stream);
int irfd_maxpool_fwd(const void* a, void* out, void* argmax, int n, int h, int w, int c, irfd_stream_t stream);
int irfd_maxpool_bwd(const void* dout, const void* dout2, const void* argmax, void* dx, int n, int h, int w, int c,
                     irfd_stream_t stream); /* dout2 (optional) is added to dout before routing */
int irfd_avgpool_fwd(const void* a, float* out, int n, int hw, int c, irfd_stream_t stream);
int irfd_avgpool_bwd(const float* dfeat, void* g, int n, int hw, int c, irfd_stream_t stream);
/* NCHW fp32 [b,c,hw] <-> NHWC bf16 [b,hw,c_pad] (c_pad >= c; padded channels are zero): the standalone forwards of the
 * reference's per-layer modules (styleganv1.py:612-635 SynthesisBlock) enter and leave the NHWC kernels through these. */
int irfd_nchw_to_nhwc_bf16(const float* in, void* out, int b, int c, int hw, int c_pad, irfd_stream_t stream);
int irfd_nhwc_bf16_to_nchw(const void* in, float* out, int b, int c, int hw, int c_pad, irfd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Synthesis-network pieces that are not conv epilogues (styleganv1.py:593-635).
 *   irfd_const_input_fwd/bwd: const[1,c,4,4] + bias -> ApplyNoise -> ApplyStyle (styleganv1.py:596-599).
 *   irfd_upsample2x_fwd/bwd : nn.Upsample(scale 2, bilinear, align_corners=False) (styleganv1.py:621,624) + adjoint.
 *   irfd_style_bwd          : backward of the fused epilogue of irfd_conv_gemm mode 2: dz (bf16) plus the reductions
 *                             ds1/dsp1 [b,c], dbias/dnw [c].
 *   irfd_to_rgb_fwd/bwd     : 1x1 conv c->3 + bias, NCHW fp32 image out (styleganv1.py:588,607).
 */
int irfd_const_input_fwd(const float* cst, const float* bias, const float* nw, const float* noise, const float* sp1,
                         const float* s1, void* a0, void* y0, int b, int c, irfd_stream_t stream);
int irfd_const_input_bwd(const void* dy, const void* a0, const float* noise, const float* sp1, float* dsp1, float* ds1,
                         float* dconst, float* dbias, float* dnw, int b, int c, irfd_stream_t stream);
int irfd_upsample2x_fwd(const void* in, void* out, int b, int h, int w, int c, irfd_stream_t stream);
/* split-bf16 variants: the input of the upsample is in + in_lo (in_lo / y0_lo may be NULL = plain variant) */
int irfd_upsample2x_split_fwd(const void* in, const void* in_lo, void* out, int b, int h, int w, int c,
                              irfd_stream_t stream);
int irfd_const_input_split_fwd(const float* cst, const float* bias, const float* nw, const float* noise,
                               const float* sp1, const float* s1, void* a0, void* y0, void* y0_lo, int b, int c,
                               irfd_stream_t stream);
int irfd_upsample2x_bwd(const void* dout, void* din, int b, int h, int w, int c, irfd_stream_t stream);
/* standalone ApplyNoise (styleganv1.py:453-456) and ApplyStyle (:463-468) on NCHW fp32: out = x + w[c]*noise[b,hw];
 * out = x*(style[b,c]+1) + style[b,C+c] */
int irfd_apply_noise_nchw(const float* x, const float* w, const float* noise, float* out, int b, int c, int hw,
                          irfd_stream_t stream);
int irfd_apply_style_nchw(const float* x, const float* style, float* out, int b, int c, int hw, irfd_stream_t stream);
long long irfd_style_bwd_workspace_bytes(int b, int hw, int c);
int irfd_style_bwd(const void* dy, const void* a, const float* noise, const float* sp1, void* dz, float* ds1,
                   float* dsp1, float* dbias, float* dnw, int b, int hw, int c, void* workspace,
                   long long workspace_bytes, irfd_stream_t stream);
int irfd_to_rgb_fwd(const void* y, const float* w, const float* bias, float* out, int b, int hw, int c,
                    irfd_stream_t stream);
long long irfd_to_rgb_bwd_workspace_bytes(int b, int hw, int c);
int irfd_to_rgb_bwd(const float* drgb, const void* y, const float* w, void* dy, float* dw, float* dbias, int b, int hw,
                    int c, void* workspace, long long workspace_bytes, irfd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * fp32 dense layers: `FC` = F.linear(x, W*w_lrmul, b*b_lrmul) + leaky_relu(0.2) (styleganv1.py:471-495) and the
 * emotion head Linear(2048,8)+softmax (model.py:41,121-122).  Batch <= 64 rows.
 *   irfd_linear_bwd: dz is the gradient w.r.t. the pre-activation (see irfd_lrelu_bwd);
 *                    dx = dx_beta*dx + wmul*dz@W (skipped if dx NULL); dw = dw_beta*dw + wmul*dz^T@x; db likewise*bmul.
 */
int irfd_linear_fwd(const float* x, const float* w, const float* bias, float* y, int b, int n, int k, float wmul,
                    float bmul, int lrelu, irfd_stream_t stream);
int irfd_lrelu_bwd(const float* dy, const float* y, float* dz, long long n, irfd_stream_t stream);
int irfd_linear_bwd(const float* dz, const float* x, const float* w, float* dx, float dx_beta, float* dw, float* db,
                    float dw_beta, int b, int n, int k, float wmul, float bmul, irfd_stream_t stream);
int irfd_softmax_rows(const float* x, float* y, int b, int n, irfd_stream_t stream);
int irfd_scale_copy(const float* src, float* dst, float scale, long long n, irfd_stream_t stream);
int irfd_split_style(const float* style, float* sp1, float* s1, int b, int c, irfd_stream_t stream);
int irfd_merge_style_grad(const float* dsp1, const float* ds1, float* dstyle, int b, int c, irfd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Device-side routing (lets a whole training step be one static CUDA graph).  The random decisions are still drawn
 * from the CPU generator in the reference's order and uploaded as ctrl (int32): ctrl[0] = swap_type (model.py:98),
 * ctrl[1+g] = first style-mixed row of generator call g, or L when that call does not mix (styleganv1.py:548-552).
 *   irfd_style_rows_fwd: rows_t[l][b][k] = l >= ctrl[ctrl_idx] ? w2[b][k] : coef(l) * w[b][k], coef = psi for l < cutoff
 *                        (styleganv1.py:536-553: truncation applies to w only, mixed rows are w2's untruncated rows);  _bwd: dw = sum_l coef(l)*drows_t[l] (all rows, as in the reference,
 *                        whose no_grad overwrite keeps routing the mixed rows' gradient into the mapping output).
 *   irfd_swap_cat_fwd  : S<->T swap of code type ctrl[0] + concat [identity|emotion|pose] -> [b, 3c] (model.py:97-108),
 *                        pure copies (bit-exact);  _bwd scatters the two gradients back to the six codes.
 */
int irfd_style_rows_fwd(const float* w, const float* w2, const int* ctrl, int ctrl_idx, float psi, int cutoff,
                        float* rows_t, int l, int b, int k, irfd_stream_t stream);
/* two generator calls stacked along the batch: rows [0, b_first) use ctrl[ctrl_idx], rows [b_first, b) ctrl[ctrl_idx+1] */
int irfd_style_rows_pair_fwd(const float* w, const float* w2, const int* ctrl, int ctrl_idx, float psi, int cutoff,
                             float* rows_t, int l, int b, int k, int b_first, irfd_stream_t stream);
int irfd_style_rows_bwd(const float* drows_t, float psi, int cutoff, float* dw, int l, int b, int k,
                        irfd_stream_t stream);
int irfd_swap_cat_fwd(const float* fi_s, const float* fe_s, const float* fp_s, const float* fi_t, const float* fe_t,
                      const float* fp_t, const int* ctrl, float* gen_s, float* gen_t, int b, int c,
                      irfd_stream_t stream);
int irfd_swap_cat_bwd(const float* dgen_s, const float* dgen_t, const int* ctrl, float* dfi_s, float* dfe_s,
                      float* dfp_s, float* dfi_t, float* dfe_t, float* dfp_t, int b, int c, irfd_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Losses and optimiser: nn.MSELoss means (model.py:356-372), clip_grad_norm_ + Adam (train.py:205-210, 346).
 *   irfd_mse_fwd : out[0] = out_beta*out[0] + mean((a-b)^2)   (double accumulation, fixed order)
 *   irfd_mse_bwd : da = gscale[0]*2(a-b)/n, db = -da (either may be NULL)
 *   irfd_sumsq   : out[0] = out_beta*out[0] + sum(g^2)
 *   irfd_adam_step: torch.optim.Adam update on a flat buffer; if total_sumsq != NULL the gradient is first scaled by
 *                  min(1, max_norm/(sqrt(total_sumsq[0])+1e-6)).
 */
long long irfd_reduce_workspace_bytes(void);
int irfd_mse_fwd(const float* a, const float* b, long long n, float* out, float out_beta, void* workspace,
                 long long workspace_bytes, irfd_stream_t stream);
int irfd_mse_bwd(const float* a, const float* b, long long n, const float* gscale, float* da, float* db,
                 irfd_stream_t stream);
int irfd_sumsq(const float* g, long long n, float* out, float out_beta, void* workspace, long long workspace_bytes,
               irfd_stream_t stream);
int irfd_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                   float eps, int step, int* step_dev, const float* total_sumsq, float max_norm, irfd_stream_t stream);
/* step_dev (optional, device int32): when given it is incremented on the device and used instead of `step`, so a
 * captured CUDA graph replays with the right bias correction. */

/* ------------------------------------------------------------------------------------------------------------------
 * Discriminator pieces that are not conv epilogues (styleganv1.py:637-695).
 *   irfd_from_rgb_fwd   : spectral-norm 1x1 conv 3 -> c on the NCHW fp32 image + bias + leaky_relu(0.2) -> NHWC bf16
 *                         (styleganv1.py:643,662); w is [c][3] fp32 (already divided by sigma); bias may be NULL and
 *                         lrelu = 0 gives the plain linear map (used by the R1 second-order chain).
 *   irfd_bias_lrelu_bwd : backward of y = leaky_relu(conv + bias): dz = g * (y > 0 ? 1 : 0.2) (bf16), dbias = sum dz.
 * ------------------------------------------------------------------------------------------------------------------ */
int irfd_from_rgb_fwd(const float* x, const float* w, const float* bias, void* out, int b, int hw, int c, int lrelu,
                      irfd_stream_t stream);
long long irfd_bias_lrelu_bwd_workspace_bytes(long long rows, int c);
int irfd_bias_lrelu_bwd(const void* g, const void* y, void* dz, float* dbias, long long rows, int c, void* workspace,
                        long long workspace_bytes, irfd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* IRFD_B200_H_ */
