/* p2pvg_b200 — C ABI of the sm_100a kernels behind the p2pvg training hot path.
 *
 * The reference (yccyenchicheng/p2pvg) has no FFI of its own: its boundary for this path is the Python
 * module API (models/p2p_model.py, models/lstm.py, models/dcgan_64.py, models/dcgan_128.py,
 * misc/criterion.py).  The drop-in Python modules in p2pvg_b200/ keep that API and call the entry
 * points below through ctypes.  Each entry point cites the reference lines whose arithmetic it
 * replaces.  Conventions:
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless stated otherwise;
 *   - the caller (PyTorch) owns every buffer; the library allocates nothing persistent;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return 0 on success, a negative P2PVG_ERR_* code otherwise; p2pvg_last_error() gives the text
 *     (thread-local).  There is no CPU fallback: unsupported shapes are errors.
 *   - dtype: 0 = fp32, 1 = bf16 ("act dtype" of the conv stacks); statistics/LSTM/optimizer are fp32.
 *   - activations are NHWC, flattened to [rows, C]; a "group" is one encoder/decoder call of the
 *     reference (BatchNorm statistics are per group, SURVEY.md §3.3).
 */
#ifndef P2PVG_B200_H
#define P2PVG_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
struct p2pvg_conv_fusion;

#define P2PVG_OK 0
#define P2PVG_ERR_BAD_ARG -1
#define P2PVG_ERR_UNSUPPORTED -2
#define P2PVG_ERR_CUDA -3
#define P2PVG_ERR_WORKSPACE -4

#define P2PVG_F32 0
#define P2PVG_BF16 1

#define P2PVG_ACT_NONE 0
#define P2PVG_ACT_LRELU 1 /* LeakyReLU(0.2): models/dcgan_64.py:10,22 */
#define P2PVG_ACT_TANH 2  /* models/dcgan_64.py:45, models/lstm.py:18 */
#define P2PVG_ACT_RELU 4   /* models/h36m_mlp.py:33-41 */
#define P2PVG_ACT_SIGMOID 3 /* models/dcgan_64.py:77 (stand-alone decoder forward; act_fwd only) */

int p2pvg_version(void);
const char* p2pvg_last_error(void);
/* 1 when the tcgen05/TMA GEMM can be used on this process' device (driver entry points resolved). */
int p2pvg_has_tcgen05(void);
/* 0 = pick automatically (tcgen05 for bf16 operands), 1 = force the CUDA-core GEMM, 2 = force tcgen05 */
int p2pvg_set_gemm_impl(int impl);
/* p2pvg_gemm `flags` (per call; there is no process-global precision state):
 *   P2PVG_GEMM_TF32          fp32 operands MAY run on tcgen05 kind::tf32 (LSTM GEMMs of the bf16 training mode).  The
 *                            tensor-core kernel needs both operands K-major, K >= 32, 16-byte aligned bases and row
 *                            pitches (TMA); any other fp32 GEMM of such a call runs on the exact CUDA-core kernel --
 *                            a documented, precision-INCREASING dispatch between two kernels of this library (never a
 *                            CPU or vendor-library fallback).
 *   P2PVG_GEMM_TF32_REQUIRE  with P2PVG_GEMM_TF32: return P2PVG_ERR_UNSUPPORTED instead of dispatching to the
 *                            CUDA-core kernel when the operands are not TMA-compatible. */
#define P2PVG_GEMM_TF32 1
#define P2PVG_GEMM_TF32_REQUIRE 2

/* C[M,N] = (accumulate ? C : 0) + opA(A)*opB(B) + bias[n] + addend[m,n]
 *   a_mn=0: A[m*lda+k] (K-major), a_mn=1: A[k*lda+m];  b_mn=0: B[n*ldb+k], b_mn=1: B[k*ldb+n].
 * Replaces the library GEMMs behind nn.Conv2d / nn.ConvTranspose2d (models/dcgan_64.py:8,20,43,64,76 after
 * lowering), nn.Linear and nn.LSTMCell (models/lstm.py:13-17,54-57) and their autograd backward.
 * bf16 operands run on tcgen05 tensor cores (fp32 accumulation in TMEM); fp32 operands on CUDA cores (exact) unless
 * `flags` allows TF32 (see above).  Documented dispatch between two kernels of this library: bf16 operands whose base
 * address or row pitch is not 16-byte aligned (not expressible as a TMA tensor map) run on the CUDA-core kernel with the
 * same arithmetic contract; p2pvg_set_gemm_impl(2) turns that case into P2PVG_ERR_UNSUPPORTED.
 * workspace: split-K partials for the tensor-core path (may be NULL when ws_bytes == 0). */
int p2pvg_gemm(const void* A, int in_dtype, int a_mn, int64_t lda, const void* B, int b_mn, int64_t ldb, void* C, int c_dtype,
               int64_t ldc, int M, int N, int K, int accumulate, const float* bias, const void* addend, int64_t ldd,
               void* workspace, size_t ws_bytes, int flags, void* stream);

/* Implicit-GEMM 4x4 / stride-2 / pad-1 convolution family on NHWC bf16 tensors (TMA 4-D pixel-box loads feeding tcgen05;
 * no im2col / col2im buffers).  H, W = size of the SMALL map (the big map is 2H x 2W).
 *   kind 0: c_small[N,H,W,Cn] = conv_s2(a_big[N,2H,2W,Ck]) . b[Cn,(kh,kw,Ck)] + bias       nn.Conv2d(.,.,4,2,1) forward
 *           (models/dcgan_64.py:8) and the data-gradient of nn.ConvTranspose2d(.,.,4,2,1) (models/dcgan_64.py:20)
 *   kind 1: c[Cm,(kh,kw,Cn)] = sum_pix a_small[pix,Cm]^T . gather_s2(b_big[N,2H,2W,Cn])    the weight gradients of both (fp32)
 *   kind 2: c_big[N,2H,2W,Cn] = convT_s2(a_small[N,H,W,Ck]) . b[Ck,(kh,kw,Cn)] + bias + addend[src]   ConvTranspose2d forward
 *           and the Conv2d data-gradient; `addend` (fp32, big-map layout) is the skip half of torch.cat([d, skip], 1)
 *           (models/dcgan_64.py:84-87) computed once per distinct source call; image n adds addend image
 *           grp_src[n / imgs_per_group] * imgs_per_group + n % imgs_per_group.
 * 3x3 / stride-1 / pad-1 variants for the vgg_64 layers (models/vgg_64.py:8-13), both maps H x W:
 *   kind 3: c[N,H,W,Cn] = conv3x3(a[N,H,W,Ck]) . b[Cn,(kh,kw,Ck)] + bias + addend[src]       forward; `addend` (fp32 [.,H,W,Cn])
 *           is the skip half of torch.cat([up(d), skip], 1) (models/vgg_64.py:97-104), indexed like kind 2
 *   kind 4: c[Cm,(kh,kw,Cn)] = sum_pix a[pix,Cm]^T . gather_3x3(b[N,H,W,Cn])                  weight gradient (fp32)
 *   kind 5: kind 3 with mirrored tap offsets, b = [Cin,(kh,kw,Cout)]                          data gradient
 * Returns P2PVG_ERR_UNSUPPORTED for shapes outside the pixel-box tiling (channels not a multiple of 64, ...). */
int p2pvg_conv_gemm(int kind, const void* a, const void* b, int64_t ldb, void* c, int c_dtype, int64_t ldc, int N, int H, int W, int Ck,
                    int Cn, int Cm, const float* bias, const void* addend, const int* grp_src, int imgs_per_group, int accumulate,
                    void* workspace, size_t ws_bytes, const struct p2pvg_conv_fusion* fusion, void* stream);

/* Optional epilogue fusions of p2pvg_conv_gemm (kinds 0, 2, 3, 5; `fusion` may be NULL, every member may be NULL).
 * nn.BatchNorm2d in training mode sits between every pair of convolutions (models/dcgan_64.py:9,21, models/vgg_64.py:9): its
 * batch statistics need the whole convolution output, so the producing GEMM emits them from its accumulator registers
 * instead of a separate pass over the stored tensor.
 *   fwd_stat_partial  out, float2 [pixel tile of 128 output rows x phase (kind 2: 4 output parities, else 1)][Cn]:
 *                     (sum y, sum y^2) of the tile's rows, y as stored (bf16-rounded for a bf16 output).  The tile of GEMM
 *                     row block mt and phase ph is row mt*phases + ph; reduce per group with p2pvg_bn_fwd_finalize_tiles
 *                     (rows of one BatchNorm group must be a multiple of 128).
 *   bwd_*             reserved for the BatchNorm-backward reduction of a data-gradient GEMM (sum dz, sum dz*xhat).
 *   addend_dtype      the skip-half addend may be stored in bf16 (it is the output of another p2pvg_conv_gemm call). */
typedef struct p2pvg_conv_fusion {
  void* fwd_stat_partial;
  const void* bwd_raw;
  const float* bwd_mean;
  const float* bwd_invstd;
  const float* bwd_scale;
  const float* bwd_shift;
  void* bwd_stat_partial;
  int64_t rows_per_group;
  int addend_dtype; /* dtype of `addend`: P2PVG_F32 (default, also without a fusion struct) or P2PVG_BF16 (half the epilogue read traffic) */
} p2pvg_conv_fusion_t;

/* vgg_64 data movement (models/vgg_64.py), NHWC, dtype f32 | bf16.
 *   im2col3  : col[(n,y,x), tap*C + c] = x[n, y + sgn*(kh-1), x + sgn*(kw-1), c], row pitch ld >= 9C (pad columns zeroed);
 *              explicit lowering of nn.Conv2d(.,.,3,1,1) (models/vgg_64.py:9) for the fp32 path and the 3-channel ends
 *   col2im3  : y[(n,y,x), c] = bias[c] + sum_tap col[(n, y-(kh-1), x-(kw-1)), tap*C + c]   nn.ConvTranspose2d(64,nc,3,1,1)
 *              (models/vgg_64.py:88) after the [pix,64] x [64,9*nc] GEMM
 *   maxpool2 : nn.MaxPool2d(2,2) (models/vgg_64.py:47) forward / backward (first maximum in row-major order takes the gradient)
 *   upsample2: nn.UpsamplingNearest2d(scale_factor=2) (models/vgg_64.py:91) forward / backward
 *   gather_add: dst[g] += src_f32[grp_src[g]] over chunks of n elements (skip-half addend, explicit path). */
int p2pvg_im2col3(const void* x, void* col, int dtype, int N, int H, int W, int C, int ld, int sgn, void* stream);
int p2pvg_col2im3(const void* col, void* y, int dtype, int N, int H, int W, int C, int ld, const float* bias, void* stream);
int p2pvg_maxpool2_fwd(const void* x, void* y, int dtype, int N, int H, int W, int C, void* stream);
int p2pvg_maxpool2_bwd(const void* x, const void* dy, void* dx, int dtype, int N, int H, int W, int C, void* stream);
int p2pvg_upsample2_fwd(const void* x, void* y, int dtype, int N, int H, int W, int C, void* stream);
int p2pvg_upsample2_bwd(const void* dy, void* dx, int dtype, int N, int H, int W, int C, void* stream);
int p2pvg_gather_add(void* dst, int dtype, const float* src, const int* grp_src, int G, int64_t n, void* stream);

/* 4x4 / stride 2 / pad 1 lowering (nn.Conv2d(nin,nout,4,2,1), models/dcgan_64.py:8; and the data-gradient of
 * nn.ConvTranspose2d(nin,nout,4,2,1), models/dcgan_64.py:20): x [N,H,W,C] -> col [N*H/2*W/2, 16*C], K order (kh,kw,c). */
int p2pvg_im2col_k4s2p1(const void* x, void* col, int dtype, int N, int H, int W, int C, void* stream);
/* Inverse gather (ConvTranspose2d forward after the GEMM, Conv2d data-gradient): y [N,2Hi,2Wi,C] from
 * col [N*Hi*Wi,16*C]; optional second operand col2 holds the skip-connection half of torch.cat([d, skip], 1)
 * (models/dcgan_64.py:84-87) computed once per distinct source call: image n reads col2 image
 * grp_src[n / imgs_per_group]*imgs_per_group + n % imgs_per_group. */
int p2pvg_col2im_k4s2p1(const void* col, const void* col2, const int* grp_src, int imgs_per_group, void* y, int dtype, int N,
                        int Hi, int Wi, int C, const float* bias, int accumulate, void* stream);
/* dst (contiguous, dims[4]) = src gathered with per-destination-dimension strides (weight packing, NCHW->NHWC, casts). */
int p2pvg_permute4(const void* src, int src_dtype, void* dst, int dst_dtype, const int* dims /*host*/,
                   const int64_t* src_strides /*host*/, int accumulate, void* stream);
/* Frames x [N, C, H*W] fp32 (the layout the data loaders hand to P2PModel.forward, models/p2p_model.py:185-197) -> channels-last
 * [N, H*W, C], written once in fp32 (dst_f32: the MSE target, may be NULL) and once in the activation dtype (dst_act: input
 * of the first convolution, may be NULL) from a single read.  C in {2,3,4}, H*W % 4 == 0; one-channel frames need no
 * conversion (NCHW == NHWC). */
int p2pvg_nchw_to_nhwc_dual(const float* src, float* dst_f32, void* dst_act, int act_dtype, int64_t N, int hw, int C, void* stream);
int p2pvg_add_indexed(void* dst, const void* src, int dtype, const int* dst_idx, int F, int64_t n, void* stream);
int p2pvg_group_sum(const void* in, void* out, int dtype, const int* grp_src, int G, int F, int64_t n, void* stream);
/* dst[a][q][p] = src[a][p][q] for a < A (tiled, coalesced both ways): nn.Conv2d / nn.ConvTranspose2d weights
 * [A][B][kh*kw] -> the GEMM layout [A][(kh,kw)][B] (models/dcgan_64.py:8,20) and the weight gradients back. */
int p2pvg_transpose_batched(const void* src, int src_dtype, void* dst, int dst_dtype, int A, int P, int Q, void* stream);
/* dst[g*R, g*C] = blockdiag(src[R, C], ..., src[R, C]): lets the 1/3-channel ends of the conv stacks (K = 16*nc or N = 16*nc,
 * models/dcgan_64.py:34,76) run as [M/g, g*C] GEMMs whose TMA boxes are never out of bounds. */
int p2pvg_blockdiag(const void* src, int src_dtype, void* dst, int dst_dtype, int R, int C, int g, void* stream);

/* nn.BatchNorm2d in training mode (models/dcgan_64.py:9,21,44,65), statistics per group. */
size_t p2pvg_bn_workspace_bytes(int G, int C);
int p2pvg_bn_fwd_stats(const void* x, int dtype, int G, int64_t R, int C, const float* gamma, const float* beta, float eps,
                       void* ws, size_t ws_bytes, float* mean, float* invstd, float* var_unbiased, float* scale, float* shift,
                       void* stream);
int p2pvg_bn_act(const void* x, void* y, int dtype, const float* scale, const float* shift, int G, int64_t R, int C, int act,
                 void* stream);
/* y may be NULL for LeakyReLU: the activation derivative is then recomputed from sign(x*scale+shift) (saves one read of y). */
int p2pvg_bn_bwd(const void* dy, const void* x, const void* y, int dtype, const float* mean, const float* invstd,
                 const float* gamma, int G, int64_t R, int C, int act, void* ws, size_t ws_bytes, void* dx, float* sum_dz,
                 float* sum_dzx, const float* scale, const float* shift, void* stream);
/* The same two BatchNorm reductions when their per-tile column sums were produced by a GEMM epilogue (p2pvg_conv_fusion):
 * partial is float2 [G * parts_per_group][ldp]; channel c of group g sums the group's partial rows over the `fold` column
 * groups f*C + c (a GEMM row may hold several pixels / filter taps of one channel).  R = elements per (group, channel).
 * fp64 combine in a fixed order (deterministic).  Replaces the statistics pass of nn.BatchNorm2d (models/dcgan_64.py:9). */
int p2pvg_bn_fwd_finalize_tiles(const void* partial, int parts_per_group, int ldp, int fold, int G, int64_t R, int C,
                                const float* gamma, const float* beta, float eps, float* mean, float* invstd, float* var_unbiased,
                                float* scale, float* shift, void* stream);
int p2pvg_bn_bwd_finalize_tiles(const void* partial, int parts_per_group, int ldp, int fold, int G, int C, float* sum_dz,
                                float* sum_dzx, void* stream);
/* apply pass of the BatchNorm + activation backward alone (the per-channel sums sum_dz / sum_dzx are given) */
int p2pvg_bn_bwd_apply(const void* dy, const void* x, const void* y, int dtype, const float* mean, const float* invstd,
                       const float* gamma, int G, int64_t R, int C, int act, void* dx, const float* sum_dz, const float* sum_dzx,
                       const float* scale, const float* shift, void* stream);
/* eval-mode BatchNorm (running statistics; generate.py / p2p_generate): scale = gamma/sqrt(rvar+eps), shift = beta-rmean*scale */
int p2pvg_bn_eval_coeffs(const float* gamma, const float* beta, const float* rmean, const float* rvar, float eps, int C,
                         float* scale, float* shift, void* stream);
int p2pvg_bn_param_grad(const float* sum_dz, const float* sum_dzx, int G, int C, float* dgamma, float* dbeta, void* stream);
/* running_mean / running_var EMA applied call by call in the reference's call order (SURVEY.md A.3 item 7). */
int p2pvg_bn_ema(float* rmean, float* rvar, const float* mean, const float* var_unbiased, const int* order, int ncalls, int C,
                 float momentum, void* stream);

/* nn.LSTMCell pointwise part (models/lstm.py:41,89): gates [B,4R] in: pre-activations (i,f,g,o), out: activations. */
int p2pvg_lstm_pointwise_fwd(float* gates, const float* c_prev, float* c_out, float* h_out, int B, int R, void* stream);
int p2pvg_lstm_pointwise_bwd(const float* dh, const float* dc_next, const float* gates, const float* c_prev, const float* c,
                             float* dgates, float* dc_prev, int B, int R, void* stream);
/* Whole-sequence recurrence of one nn.LSTMCell layer in ONE persistent launch (the W_hh slice of a CTA stays on chip for all
 * timesteps).  tf32 = 1 dispatches by hidden size: R in {64,128,256}: thread-block clusters of 8 CTAs, hardware cluster barrier per
 * timestep; R = 512: clusters of 16 CTAs (non-portable size), slabs of 16 / 32 / 48 batch rows per cluster chosen so that the
 * resident clusters cover the batch in one wave, backward reduction scattered through distributed shared memory, the part of the
 * weight slice that does not fit the registers in shared memory (16-row slabs) or tensor memory (larger slabs).  tf32 = 0, or
 * tf32 = 1 with R not in {64,128,256,512}: cooperative grid with a grid barrier per timestep, exact fp32 FFMA products.
 *   forward : gates_s = pre_s + b_hh + h_{s-1}.W_hh^T -> (i,f,g,o) -> c_s, h_s       pre [S,B,4R] = x-part incl. b_ih
 *             gates [S,B,4R] out (activations), hs / cs [S+1,B,R] with slot 0 = initial state (zeros, models/lstm.py:21-27)
 *   backward: dh_s = dhtop_s + dG_{s+1}.W_hh, cell backward -> dG [S,B,4R] (gradient w.r.t. the gate pre-activations)
 * `counter` is a zero-initialised uint32 in device memory (the grid barrier of the cooperative variant); R %% 64 == 0, R <= 256, or
 * R = 512 (tf32 = 1: any batch; tf32 = 0: as long as the cooperative grid fits).  Unsupported shapes return P2PVG_ERR_UNSUPPORTED.
 * tf32 = 1: the recurrent products on the tensor cores (mma.sync m16n8k8 tf32, fp32 accumulation). */
int p2pvg_lstm_scan_fwd(const float* pre, const float* whh, const float* bhh, float* gates, float* hs, float* cs, int S, int B, int R,
                        int tf32, unsigned* counter, void* stream);
int p2pvg_lstm_scan_bwd(const float* dhtop, const float* whh, const float* gates, const float* cs, float* dG, int S, int B, int R,
                        int tf32, unsigned* counter, void* stream);
/* diagnostics: cudaOccupancyMaxActiveClusters of the hidden-size-512 scans (clusters of 16 CTAs): which = 0 / 1 / 3 forward with
 * 16- / 32- / 48-row slabs, 2 / 4 / 5 backward with 16- / 32- / 48-row slabs; -1 on error */
int p2pvg_lstm_cluster512_max_clusters(int which);
/* the same for the hidden-size-256 scans (clusters of 8 CTAs): which = 0 / 1 forward with 16- / 32-row slabs, 2 / 3 backward */
int p2pvg_lstm_cluster_max_clusters(int which);
/* gaussian_lstm.reparameterize (models/lstm.py:76-81) for posterior and prior + KLCriterion.forward
 * (misc/criterion.py:10-15) summed over all elements (division by opt.batch_size happens in finalize_losses). */
int p2pvg_reparam_kl_fwd(const float* mu, const float* lv, const float* mu_p, const float* lv_p, const float* eps,
                         const float* eps_p, float* z, float* z_p, int n, float* kl_sum, void* stream);
int p2pvg_reparam_kl_bwd(const float* mu, const float* lv, const float* mu_p, const float* lv_p, const float* eps,
                         const float* eps_p, const float* dz, const float* dz_p, float kl_coef, float* dmu, float* dlv,
                         float* dmu_p, float* dlv_p, int n, void* stream);
/* torch.cat([h, global_z | z, time_until_cp, delta_time], 1) (models/p2p_model.py:241-242,247,252) for all steps. */
int p2pvg_build_concat(float* dst, const float* A, const int* ia, int ga, const float* Bm, const int* ib, int gb,
                       const float* tuc, const float* dt, int S, int B, int ld /* row pitch >= ga+gb+2, zero padded */, void* stream);
int p2pvg_gather_add_cols(float* dst, const float* src, const int* idx, int S, int T, int B, int g, int W, int col0, int init,
                          void* stream);
/* align_loss += MSE(h[0], h_pred) with h[0] = batch row 0 broadcast (models/p2p_model.py:224-225), value + gradients. */
int p2pvg_align(const float* H, const int* in_idx, const float* h_pred, int P, int B, int g, float coef, float* loss_partial,
                float* d_hpred, float* dH, void* stream);
/* out[c] (+)= sum_r x[r*ld + c] — bias gradients. */
int p2pvg_colsum(const void* x, int dtype, int64_t rows, int cols, int64_t ld, float* out, int accumulate, void* ws /* >= 1024*cols floats */,
                 size_t ws_bytes, void* stream);
int p2pvg_act_fwd(float* x, int64_t n, int act, void* stream);
int p2pvg_act_bwd(const float* dy, const float* y, float* dx, int64_t n, int act, void* stream);

/* nn.Sigmoid (models/dcgan_64.py:77) + nn.MSELoss (models/p2p_model.py:254,256): per-group sum of squared error
 * partials [G, p2pvg_mse_chunks()] and d(loss)/d(raw) = coef[g]*2*(s-x)*s*(1-s). */
int p2pvg_mse_chunks(void);
int p2pvg_sigmoid_mse(const void* raw, int dtype, const float* x, const int* tgt, const float* coef, int G, int64_t E,
                      void* pred, void* d_raw, float* partial, void* stream);
/* The last decoder layer of the dcgan stacks (C = 1 or 3 image channels) fused with its loss: ConvTranspose2d(2*64, C, 4, 2, 1) +
 * nn.Sigmoid (models/dcgan_64.py:75-79, models/dcgan_128.py:82-84) + nn.MSELoss against frame tgt[g] (models/p2p_model.py:254,256).
 * col [G*B*Hi*Wi, 16*C] / col2 [nsrc*B*Hi*Wi, 16*C]: the 16 tap products (x C channels) of every input pixel of the decoder half /
 * of the shared skip half (group g uses skip source grp_src[g]), as produced by p2pvg_gemm.  Writes d(loss)/d(raw)
 * [G, B*2Hi*2Wi*C] (NHWC) and the squared-error partials [G, p2pvg_mse_chunks()]; the raw output is never materialised. */
int p2pvg_convt_c1_loss(const void* col, const void* col2, int dtype, const int* grp_src, const float* bias, const float* x, const int* tgt,
                        const float* coef, int G, int B, int Hi, int Wi, int C, void* d_raw, float* partial, void* stream);
/* h36m pose backbone (models/h36m_mlp.py): nn.LayerNorm of residual_linear (:43,46) forward / backward (fp32, row-wise; dx may alias
 * dy; dgamma == NULL skips the parameter gradients) and the plain nn.MSELoss on [B,17,3] poses (models/p2p_model.py:254,256) with
 * the same partial-sum layout as p2pvg_sigmoid_mse. */
int p2pvg_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* rstd, int64_t rows, int C,
                        float eps, void* stream);
int p2pvg_layernorm_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma, float* dx,
                        float* dgamma, float* dbeta, int64_t rows, int C, void* ws, size_t ws_bytes, void* stream);
int p2pvg_mse_plain(const float* pred, const float* x, const int* tgt, const float* coef, int G, int64_t E, float* d_pred, float* partial,
                    void* stream);
/* the four scalars returned by P2PModel.forward (models/p2p_model.py:271): out[0..3] = mse,kld,cpc,align (/seq_len). */
int p2pvg_finalize_losses(const float* mse_partial, int n_recon, int has_cpc, double E, const float* kl_sum, float batch_size,
                          const float* align_partial, int n_align, float seq_len, float* out, void* stream);
/* Early read-back of the step's scalars (models/p2p_model.py:271 returns them as host numbers: `mse.data.cpu().numpy()`): the
 * kernel stores src[0..n) and then *seq into page-locked, device-mapped host memory host_mapped[0..n] (n floats + one int);
 * the host polls host_mapped[n] for the sequence number it wrote to *seq before launching.  The values are final once the
 * forward pass is done, so the caller gets them while the backward passes and the optimiser of the same step still run;
 * everything else stays stream-ordered.  n <= 64. */
int p2pvg_publish_scalars(const float* src, int n, float* host_mapped, const int* seq, void* stream);
/* optim.Adam.step of PyTorch 1.0 (README.md:62; models/p2p_model.py:273-280) on a flat parameter arena. */
int p2pvg_adam_legacy(float* p, const float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2,
                      double eps, const int* step_ptr, void* stream);
int p2pvg_scale(float* x, int64_t n, float a, void* stream);

#ifdef __cplusplus
}
#endif
#endif
