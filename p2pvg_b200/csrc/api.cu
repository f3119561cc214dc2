// extern "C" surface of libp2pvg_b200.so (declared in include/p2pvg_b200.h): argument checking,
// thread-local error state, GEMM dispatch (tcgen05 vs CUDA-core).
#include <stdarg.h>
#include <string.h>

#include "../../include/p2pvg_b200.h"

#include "common.cuh"

static thread_local char g_err[512] = "";

void p2pvg_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int p2pvg_check_launch(const char* what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    p2pvg_set_error("%s: %s", what, cudaGetErrorString(e));
    (void)cudaGetLastError();
    return P2PVG_ERR_CUDA;
  }
  return P2PVG_OK;
}

// ---- implemented in the other translation units ----
int p2pvg_gemm_simt(const void*, int, int, long long, const void*, int, long long, void*, int, long long, int, int, int, int,
                    const float*, const void*, long long, void*, size_t, cudaStream_t);
int p2pvg_gemm_tf32(const void*, long long, const void*, long long, void*, int, long long, int, int, int, int, const float*,
                    const void*, long long, cudaStream_t);
int p2pvg_gemm_tc(const void*, int, long long, const void*, int, long long, void*, int, long long, int, int, int, int, const float*,
                  const void*, long long, void*, size_t, cudaStream_t);
int p2pvg_gemm_tc_available();
int p2pvg_layernorm_fwd_impl(const float*, const float*, const float*, float*, float*, float*, long long, int, float, cudaStream_t);
int p2pvg_layernorm_bwd_impl(const float*, const float*, const float*, const float*, const float*, float*, float*, float*, long long, int,
                             void*, size_t, cudaStream_t);
int p2pvg_mse_plain_impl(const float*, const float*, const int*, const float*, int, long long, float*, float*, int, cudaStream_t);
int p2pvg_conv_gemm_impl(int, const void*, const void*, long long, void*, int, long long, int, int, int, int, int, int, const float*,
                         const float*, const int*, int, int, void*, size_t, void*, int, cudaStream_t);
int p2pvg_bn_fwd_finalize_tiles_impl(const void*, int, int, int, int, long long, int, const float*, const float*, float, float*, float*, float*,
                                     float*, float*, cudaStream_t);
int p2pvg_bn_bwd_finalize_tiles_impl(const void*, int, int, int, int, int, float*, float*, cudaStream_t);
int p2pvg_bn_bwd_apply_impl(const void*, const void*, const void*, int, const float*, const float*, const float*, int, long long, int, int,
                            void*, const float*, const float*, const float*, const float*, cudaStream_t);
int p2pvg_im2col_k4s2p1_impl(const void*, void*, int, int, int, int, int, cudaStream_t);
int p2pvg_im2col3_impl(const void*, void*, int, int, int, int, int, int, int, cudaStream_t);
int p2pvg_col2im3_impl(const void*, void*, int, int, int, int, int, int, const float*, cudaStream_t);
int p2pvg_maxpool2_fwd_impl(const void*, void*, int, int, int, int, int, cudaStream_t);
int p2pvg_maxpool2_bwd_impl(const void*, const void*, void*, int, int, int, int, int, cudaStream_t);
int p2pvg_upsample2_fwd_impl(const void*, void*, int, int, int, int, int, cudaStream_t);
int p2pvg_upsample2_bwd_impl(const void*, void*, int, int, int, int, int, cudaStream_t);
int p2pvg_gather_add_impl(void*, int, const float*, const int*, int, long long, cudaStream_t);
int p2pvg_col2im_k4s2p1_impl(const void*, const void*, const int*, int, void*, int, int, int, int, int, const float*, int, cudaStream_t);
int p2pvg_permute4_impl(const void*, int, void*, int, const int*, const long long*, int, cudaStream_t);
int p2pvg_nchw_to_nhwc_dual_impl(const float*, float*, void*, int, long long, int, int, cudaStream_t);
int p2pvg_add_indexed_impl(void*, const void*, int, const int*, int, long long, cudaStream_t);
int p2pvg_group_sum_impl(const void*, void*, int, const int*, int, int, long long, cudaStream_t);
int p2pvg_blockdiag_impl(const void*, int, void*, int, int, int, int, cudaStream_t);
int p2pvg_transpose_batched_impl(const void*, int, void*, int, int, int, int, cudaStream_t);
size_t p2pvg_bn_workspace_bytes_impl(int, int);
int p2pvg_bn_fwd_stats_impl(const void*, int, int, long long, int, const float*, const float*, float, void*, size_t, float*, float*,
                            float*, float*, float*, cudaStream_t);
int p2pvg_bn_act_impl(const void*, void*, int, const float*, const float*, int, long long, int, int, cudaStream_t);
int p2pvg_bn_bwd_impl(const void*, const void*, const void*, int, const float*, const float*, const float*, int, long long, int, int,
                      void*, size_t, void*, float*, float*, const float*, const float*, cudaStream_t);
int p2pvg_bn_param_grad_impl(const float*, const float*, int, int, float*, float*, cudaStream_t);
int p2pvg_bn_ema_impl(float*, float*, const float*, const float*, const int*, int, int, float, cudaStream_t);
int p2pvg_bn_eval_coeffs_impl(const float*, const float*, const float*, const float*, float, int, float*, float*, cudaStream_t);
int p2pvg_lstm_pointwise_fwd_impl(float*, const float*, float*, float*, int, int, cudaStream_t);
int p2pvg_lstm_pointwise_bwd_impl(const float*, const float*, const float*, const float*, const float*, float*, float*, int, int,
                                  cudaStream_t);
int p2pvg_lstm_scan_fwd_impl(const float*, const float*, const float*, float*, float*, float*, int, int, int, int, unsigned*, cudaStream_t);
bool p2pvg_lstm_cluster_supported(int);
int p2pvg_lstm_cluster_fwd_impl(const float*, const float*, const float*, float*, float*, float*, int, int, int, cudaStream_t);
int p2pvg_lstm_cluster_bwd_impl(const float*, const float*, const float*, const float*, float*, int, int, int, cudaStream_t);
int p2pvg_lstm_scan_bwd_impl(const float*, const float*, const float*, const float*, float*, int, int, int, int, unsigned*, cudaStream_t);
int p2pvg_lstm_cluster512_fwd_impl(const float*, const float*, const float*, float*, float*, float*, int, int, cudaStream_t);
int p2pvg_lstm_cluster512_bwd_impl(const float*, const float*, const float*, const float*, float*, int, int, cudaStream_t);
int p2pvg_lstm_cluster512_max_clusters_impl(int);
int p2pvg_lstm_cluster_max_clusters_impl(int);
int p2pvg_reparam_kl_fwd_impl(const float*, const float*, const float*, const float*, const float*, const float*, float*, float*, int,
                              float*, cudaStream_t);
int p2pvg_reparam_kl_bwd_impl(const float*, const float*, const float*, const float*, const float*, const float*, const float*,
                              const float*, float, float*, float*, float*, float*, int, cudaStream_t);
int p2pvg_build_concat_impl(float*, const float*, const int*, int, const float*, const int*, int, const float*, const float*, int, int,
                            int, cudaStream_t);
int p2pvg_gather_add_cols_impl(float*, const float*, const int*, int, int, int, int, int, int, int, cudaStream_t);
int p2pvg_align_impl(const float*, const int*, const float*, int, int, int, float, float*, float*, float*, cudaStream_t);
int p2pvg_colsum_impl(const void*, int, long long, int, long long, float*, int, void*, size_t, cudaStream_t);
int p2pvg_act_fwd_impl(float*, long long, int, cudaStream_t);
int p2pvg_act_bwd_impl(const float*, const float*, float*, long long, int, cudaStream_t);
int p2pvg_mse_chunks_impl();
int p2pvg_sigmoid_mse_impl(const void*, int, const float*, const int*, const float*, int, long long, void*, void*, float*, cudaStream_t);
int p2pvg_finalize_losses_impl(const float*, int, int, double, const float*, float, const float*, int, float, float*, cudaStream_t);
int p2pvg_publish_scalars_impl(const float*, int, float*, const int*, cudaStream_t);
int p2pvg_convt_c1_loss_impl(const void*, const void*, int, const int*, const float*, const float*, const int*, const float*, int, int, int, int,
                             int, void*, float*, cudaStream_t);
int p2pvg_adam_legacy_impl(float*, const float*, float*, float*, long long, double, double, double, double, const int*, cudaStream_t);
int p2pvg_scale_impl(float*, long long, float, cudaStream_t);

static int g_gemm_impl = 0;  // 0 auto, 1 simt, 2 tcgen05
int p2pvg_gemm_impl_forced() { return g_gemm_impl; }

#define ST ((cudaStream_t)stream)

extern "C" {

int p2pvg_version(void) { return 100; }
const char* p2pvg_last_error(void) { return g_err; }
int p2pvg_has_tcgen05(void) { return p2pvg_gemm_tc_available(); }
int p2pvg_set_gemm_impl(int impl) {
  if (impl < 0 || impl > 2) return P2PVG_ERR_BAD_ARG;
  g_gemm_impl = impl;
  return P2PVG_OK;
}

int p2pvg_gemm(const void* A, int in_dtype, int a_mn, int64_t lda, const void* B, int b_mn, int64_t ldb, void* C, int c_dtype,
               int64_t ldc, int M, int N, int K, int accumulate, const float* bias, const void* addend, int64_t ldd,
               void* workspace, size_t ws_bytes, int flags, void* stream) {
  P2PVG_REQUIRE(A && B && C, P2PVG_ERR_BAD_ARG, "gemm: null operand");
  P2PVG_REQUIRE(M >= 0 && N >= 0 && K >= 0, P2PVG_ERR_BAD_ARG, "gemm: negative size");
  bool want_tc = (in_dtype == P2PVG_BF16) && g_gemm_impl != 1;
  // fp32 operands (LSTM / parity mode) always run on the CUDA cores; "forced tcgen05" only makes the bf16 path
  // refuse to fall back when an operand is not TMA-compatible.
  if (want_tc)
    return p2pvg_gemm_tc(A, a_mn, lda, B, b_mn, ldb, C, c_dtype, ldc, M, N, K, accumulate, bias, addend, ldd, workspace, ws_bytes, ST);
  if (in_dtype == P2PVG_F32 && (flags & P2PVG_GEMM_TF32) && g_gemm_impl != 1) {
    // documented dispatch (include/p2pvg_b200.h): TF32 tensor cores for K-major TMA-compatible operands, the exact
    // CUDA-core kernel otherwise -- unless the caller asked for an error instead
    int rc = P2PVG_ERR_UNSUPPORTED;
    if (!a_mn && !b_mn && K >= 32) rc = p2pvg_gemm_tf32(A, lda, B, ldb, C, c_dtype, ldc, M, N, K, accumulate, bias, addend, ldd, ST);
    if (rc != P2PVG_ERR_UNSUPPORTED) return rc;
    if (flags & P2PVG_GEMM_TF32_REQUIRE) {
      p2pvg_set_error("gemm: fp32 operands not eligible for the TF32 tensor-core kernel (need K-major, K >= 32, 16-byte aligned bases / pitches): M=%d N=%d K=%d a_mn=%d b_mn=%d",
                      M, N, K, a_mn, b_mn);
      return P2PVG_ERR_UNSUPPORTED;
    }
  }
  return p2pvg_gemm_simt(A, in_dtype, a_mn, lda, B, b_mn, ldb, C, c_dtype, ldc, M, N, K, accumulate, bias, addend, ldd, workspace,
                         ws_bytes, ST);
}

int p2pvg_conv_gemm(int kind, const void* a, const void* b, int64_t ldb, void* c, int c_dtype, int64_t ldc, int N, int H, int W, int Ck,
                    int Cn, int Cm, const float* bias, const void* addend, const int* grp_src, int imgs_per_group, int accumulate,
                    void* workspace, size_t ws_bytes, const p2pvg_conv_fusion_t* fusion, void* stream) {
  P2PVG_REQUIRE(a && b && c, P2PVG_ERR_BAD_ARG, "conv_gemm: null operand");
  void* fwd_stat = fusion ? fusion->fwd_stat_partial : nullptr;
  P2PVG_REQUIRE(!fusion || fusion->bwd_stat_partial == nullptr, P2PVG_ERR_UNSUPPORTED, "conv_gemm: backward BatchNorm fusion is reserved");
  P2PVG_REQUIRE(!(fwd_stat && accumulate), P2PVG_ERR_BAD_ARG, "conv_gemm: statistics of an accumulating GEMM are not defined");
  const int add_dt = fusion ? fusion->addend_dtype : P2PVG_F32;
  P2PVG_REQUIRE(add_dt == P2PVG_F32 || add_dt == P2PVG_BF16, P2PVG_ERR_BAD_ARG, "conv_gemm: bad addend dtype %d", add_dt);
  return p2pvg_conv_gemm_impl(kind, a, b, ldb, c, c_dtype, ldc, N, H, W, Ck, Cn, Cm, bias, reinterpret_cast<const float*>(addend), grp_src,
                              imgs_per_group, accumulate, workspace, ws_bytes, fwd_stat, add_dt, ST);
}

int p2pvg_im2col_k4s2p1(const void* x, void* col, int dtype, int N, int H, int W, int C, void* stream) {
  return p2pvg_im2col_k4s2p1_impl(x, col, dtype, N, H, W, C, ST);
}
int p2pvg_col2im_k4s2p1(const void* col, const void* col2, const int* grp_src, int imgs_per_group, void* y, int dtype, int N,
                        int Hi, int Wi, int C, const float* bias, int accumulate, void* stream) {
  return p2pvg_col2im_k4s2p1_impl(col, col2, grp_src, imgs_per_group, y, dtype, N, Hi, Wi, C, bias, accumulate, ST);
}
int p2pvg_permute4(const void* src, int src_dtype, void* dst, int dst_dtype, const int* dims, const int64_t* src_strides,
                   int accumulate, void* stream) {
  return p2pvg_permute4_impl(src, src_dtype, dst, dst_dtype, dims, (const long long*)src_strides, accumulate, ST);
}
int p2pvg_nchw_to_nhwc_dual(const float* src, float* dst_f32, void* dst_act, int act_dtype, int64_t N, int hw, int C, void* stream) {
  return p2pvg_nchw_to_nhwc_dual_impl(src, dst_f32, dst_act, act_dtype, (long long)N, hw, C, ST);
}
int p2pvg_add_indexed(void* dst, const void* src, int dtype, const int* dst_idx, int F, int64_t n, void* stream) {
  return p2pvg_add_indexed_impl(dst, src, dtype, dst_idx, F, n, ST);
}
int p2pvg_im2col3(const void* x, void* col, int dtype, int N, int H, int W, int C, int ld, int sgn, void* stream) {
  return p2pvg_im2col3_impl(x, col, dtype, N, H, W, C, ld, sgn, ST);
}
int p2pvg_col2im3(const void* col, void* y, int dtype, int N, int H, int W, int C, int ld, const float* bias, void* stream) {
  return p2pvg_col2im3_impl(col, y, dtype, N, H, W, C, ld, bias, ST);
}
int p2pvg_maxpool2_fwd(const void* x, void* y, int dtype, int N, int H, int W, int C, void* stream) {
  return p2pvg_maxpool2_fwd_impl(x, y, dtype, N, H, W, C, ST);
}
int p2pvg_maxpool2_bwd(const void* x, const void* dy, void* dx, int dtype, int N, int H, int W, int C, void* stream) {
  return p2pvg_maxpool2_bwd_impl(x, dy, dx, dtype, N, H, W, C, ST);
}
int p2pvg_upsample2_fwd(const void* x, void* y, int dtype, int N, int H, int W, int C, void* stream) {
  return p2pvg_upsample2_fwd_impl(x, y, dtype, N, H, W, C, ST);
}
int p2pvg_upsample2_bwd(const void* dy, void* dx, int dtype, int N, int H, int W, int C, void* stream) {
  return p2pvg_upsample2_bwd_impl(dy, dx, dtype, N, H, W, C, ST);
}
int p2pvg_gather_add(void* dst, int dtype, const float* src, const int* grp_src, int G, int64_t n, void* stream) {
  return p2pvg_gather_add_impl(dst, dtype, src, grp_src, G, n, ST);
}
int p2pvg_transpose_batched(const void* src, int src_dtype, void* dst, int dst_dtype, int A, int P, int Q, void* stream) {
  return p2pvg_transpose_batched_impl(src, src_dtype, dst, dst_dtype, A, P, Q, ST);
}
int p2pvg_blockdiag(const void* src, int src_dtype, void* dst, int dst_dtype, int R, int C, int g, void* stream) {
  return p2pvg_blockdiag_impl(src, src_dtype, dst, dst_dtype, R, C, g, ST);
}
int p2pvg_group_sum(const void* in, void* out, int dtype, const int* grp_src, int G, int F, int64_t n, void* stream) {
  return p2pvg_group_sum_impl(in, out, dtype, grp_src, G, F, n, ST);
}
size_t p2pvg_bn_workspace_bytes(int G, int C) { return p2pvg_bn_workspace_bytes_impl(G, C); }
int p2pvg_bn_fwd_stats(const void* x, int dtype, int G, int64_t R, int C, const float* gamma, const float* beta, float eps,
                       void* ws, size_t ws_bytes, float* mean, float* invstd, float* var_unbiased, float* scale, float* shift,
                       void* stream) {
  return p2pvg_bn_fwd_stats_impl(x, dtype, G, R, C, gamma, beta, eps, ws, ws_bytes, mean, invstd, var_unbiased, scale, shift, ST);
}
int p2pvg_bn_act(const void* x, void* y, int dtype, const float* scale, const float* shift, int G, int64_t R, int C, int act,
                 void* stream) {
  return p2pvg_bn_act_impl(x, y, dtype, scale, shift, G, R, C, act, ST);
}
int p2pvg_bn_bwd(const void* dy, const void* x, const void* y, int dtype, const float* mean, const float* invstd,
                 const float* gamma, int G, int64_t R, int C, int act, void* ws, size_t ws_bytes, void* dx, float* sum_dz,
                 float* sum_dzx, const float* scale, const float* shift, void* stream) {
  return p2pvg_bn_bwd_impl(dy, x, y, dtype, mean, invstd, gamma, G, R, C, act, ws, ws_bytes, dx, sum_dz, sum_dzx, scale, shift, ST);
}
int p2pvg_bn_fwd_finalize_tiles(const void* partial, int parts_per_group, int ldp, int fold, int G, int64_t R, int C,
                                const float* gamma, const float* beta, float eps, float* mean, float* invstd, float* var_unbiased,
                                float* scale, float* shift, void* stream) {
  return p2pvg_bn_fwd_finalize_tiles_impl(partial, parts_per_group, ldp, fold, G, R, C, gamma, beta, eps, mean, invstd, var_unbiased, scale,
                                          shift, ST);
}
int p2pvg_bn_bwd_finalize_tiles(const void* partial, int parts_per_group, int ldp, int fold, int G, int C, float* sum_dz,
                                float* sum_dzx, void* stream) {
  return p2pvg_bn_bwd_finalize_tiles_impl(partial, parts_per_group, ldp, fold, G, C, sum_dz, sum_dzx, ST);
}
int p2pvg_bn_bwd_apply(const void* dy, const void* x, const void* y, int dtype, const float* mean, const float* invstd,
                       const float* gamma, int G, int64_t R, int C, int act, void* dx, const float* sum_dz, const float* sum_dzx,
                       const float* scale, const float* shift, void* stream) {
  return p2pvg_bn_bwd_apply_impl(dy, x, y, dtype, mean, invstd, gamma, G, R, C, act, dx, sum_dz, sum_dzx, scale, shift, ST);
}
int p2pvg_bn_param_grad(const float* sum_dz, const float* sum_dzx, int G, int C, float* dgamma, float* dbeta, void* stream) {
  return p2pvg_bn_param_grad_impl(sum_dz, sum_dzx, G, C, dgamma, dbeta, ST);
}
int p2pvg_bn_eval_coeffs(const float* gamma, const float* beta, const float* rmean, const float* rvar, float eps, int C,
                         float* scale, float* shift, void* stream) {
  return p2pvg_bn_eval_coeffs_impl(gamma, beta, rmean, rvar, eps, C, scale, shift, ST);
}
int p2pvg_bn_ema(float* rmean, float* rvar, const float* mean, const float* var_unbiased, const int* order, int ncalls, int C,
                 float momentum, void* stream) {
  return p2pvg_bn_ema_impl(rmean, rvar, mean, var_unbiased, order, ncalls, C, momentum, ST);
}
int p2pvg_lstm_pointwise_fwd(float* gates, const float* c_prev, float* c_out, float* h_out, int B, int R, void* stream) {
  return p2pvg_lstm_pointwise_fwd_impl(gates, c_prev, c_out, h_out, B, R, ST);
}
int p2pvg_lstm_pointwise_bwd(const float* dh, const float* dc_next, const float* gates, const float* c_prev, const float* c,
                             float* dgates, float* dc_prev, int B, int R, void* stream) {
  return p2pvg_lstm_pointwise_bwd_impl(dh, dc_next, gates, c_prev, c, dgates, dc_prev, B, R, ST);
}
// tensor-core mode: thread-block-cluster scans, lstm_cluster.cu for R in {64,128,256} and lstm_cluster512.cu (clusters of 16
// CTAs) for R = 512 (BASELINE config 5); the cooperative-grid scans serve the exact-fp32 mode and every other R
int p2pvg_lstm_scan_fwd(const float* pre, const float* whh, const float* bhh, float* gates, float* hs, float* cs, int S, int B, int R,
                        int tf32, unsigned* counter, void* stream) {
  if (tf32 && R == 512) return p2pvg_lstm_cluster512_fwd_impl(pre, whh, bhh, gates, hs, cs, S, B, ST);
  if (tf32 && p2pvg_lstm_cluster_supported(R)) return p2pvg_lstm_cluster_fwd_impl(pre, whh, bhh, gates, hs, cs, S, B, R, ST);
  return p2pvg_lstm_scan_fwd_impl(pre, whh, bhh, gates, hs, cs, S, B, R, tf32, counter, ST);
}
int p2pvg_lstm_scan_bwd(const float* dhtop, const float* whh, const float* gates, const float* cs, float* dG, int S, int B, int R,
                        int tf32, unsigned* counter, void* stream) {
  if (tf32 && R == 512) return p2pvg_lstm_cluster512_bwd_impl(dhtop, whh, gates, cs, dG, S, B, ST);
  if (tf32 && p2pvg_lstm_cluster_supported(R)) return p2pvg_lstm_cluster_bwd_impl(dhtop, whh, gates, cs, dG, S, B, R, ST);
  return p2pvg_lstm_scan_bwd_impl(dhtop, whh, gates, cs, dG, S, B, R, tf32, counter, ST);
}
int p2pvg_lstm_cluster512_max_clusters(int which) { return p2pvg_lstm_cluster512_max_clusters_impl(which); }
int p2pvg_lstm_cluster_max_clusters(int which) { return p2pvg_lstm_cluster_max_clusters_impl(which); }
int p2pvg_reparam_kl_fwd(const float* mu, const float* lv, const float* mu_p, const float* lv_p, const float* eps,
                         const float* eps_p, float* z, float* z_p, int n, float* kl_sum, void* stream) {
  return p2pvg_reparam_kl_fwd_impl(mu, lv, mu_p, lv_p, eps, eps_p, z, z_p, n, kl_sum, ST);
}
int p2pvg_reparam_kl_bwd(const float* mu, const float* lv, const float* mu_p, const float* lv_p, const float* eps,
                         const float* eps_p, const float* dz, const float* dz_p, float kl_coef, float* dmu, float* dlv,
                         float* dmu_p, float* dlv_p, int n, void* stream) {
  return p2pvg_reparam_kl_bwd_impl(mu, lv, mu_p, lv_p, eps, eps_p, dz, dz_p, kl_coef, dmu, dlv, dmu_p, dlv_p, n, ST);
}
int p2pvg_build_concat(float* dst, const float* A, const int* ia, int ga, const float* Bm, const int* ib, int gb,
                       const float* tuc, const float* dt, int S, int B, int ld, void* stream) {
  return p2pvg_build_concat_impl(dst, A, ia, ga, Bm, ib, gb, tuc, dt, S, B, ld, ST);
}
int p2pvg_gather_add_cols(float* dst, const float* src, const int* idx, int S, int T, int B, int g, int W, int col0, int init,
                          void* stream) {
  return p2pvg_gather_add_cols_impl(dst, src, idx, S, T, B, g, W, col0, init, ST);
}
int p2pvg_align(const float* H, const int* in_idx, const float* h_pred, int P, int B, int g, float coef, float* loss_partial,
                float* d_hpred, float* dH, void* stream) {
  return p2pvg_align_impl(H, in_idx, h_pred, P, B, g, coef, loss_partial, d_hpred, dH, ST);
}
int p2pvg_colsum(const void* x, int dtype, int64_t rows, int cols, int64_t ld, float* out, int accumulate, void* ws, size_t ws_bytes,
                 void* stream) {
  return p2pvg_colsum_impl(x, dtype, rows, cols, ld, out, accumulate, ws, ws_bytes, ST);
}
int p2pvg_act_fwd(float* x, int64_t n, int act, void* stream) { return p2pvg_act_fwd_impl(x, n, act, ST); }
int p2pvg_act_bwd(const float* dy, const float* y, float* dx, int64_t n, int act, void* stream) {
  return p2pvg_act_bwd_impl(dy, y, dx, n, act, ST);
}
int p2pvg_mse_chunks(void) { return p2pvg_mse_chunks_impl(); }
int p2pvg_convt_c1_loss(const void* col, const void* col2, int dtype, const int* grp_src, const float* bias, const float* x, const int* tgt,
                        const float* coef, int G, int B, int Hi, int Wi, int C, void* d_raw, float* partial, void* stream) {
  P2PVG_REQUIRE(col && col2 && grp_src && x && tgt && coef && d_raw && partial, P2PVG_ERR_BAD_ARG, "convt_c1_loss: null argument");
  return p2pvg_convt_c1_loss_impl(col, col2, dtype, grp_src, bias, x, tgt, coef, G, B, Hi, Wi, C, d_raw, partial, ST);
}
int p2pvg_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* rstd, int64_t rows, int C,
                        float eps, void* stream) {
  return p2pvg_layernorm_fwd_impl(x, gamma, beta, y, mean, rstd, rows, C, eps, ST);
}
int p2pvg_layernorm_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma, float* dx,
                        float* dgamma, float* dbeta, int64_t rows, int C, void* ws, size_t ws_bytes, void* stream) {
  return p2pvg_layernorm_bwd_impl(dy, x, mean, rstd, gamma, dx, dgamma, dbeta, rows, C, ws, ws_bytes, ST);
}
int p2pvg_mse_plain(const float* pred, const float* x, const int* tgt, const float* coef, int G, int64_t E, float* d_pred, float* partial,
                    void* stream) {
  return p2pvg_mse_plain_impl(pred, x, tgt, coef, G, E, d_pred, partial, p2pvg_mse_chunks_impl(), ST);
}
int p2pvg_sigmoid_mse(const void* raw, int dtype, const float* x, const int* tgt, const float* coef, int G, int64_t E,
                      void* pred, void* d_raw, float* partial, void* stream) {
  return p2pvg_sigmoid_mse_impl(raw, dtype, x, tgt, coef, G, E, pred, d_raw, partial, ST);
}
int p2pvg_finalize_losses(const float* mse_partial, int n_recon, int has_cpc, double E, const float* kl_sum, float batch_size,
                          const float* align_partial, int n_align, float seq_len, float* out, void* stream) {
  return p2pvg_finalize_losses_impl(mse_partial, n_recon, has_cpc, E, kl_sum, batch_size, align_partial, n_align, seq_len, out, ST);
}
int p2pvg_publish_scalars(const float* src, int n, float* host_mapped, const int* seq, void* stream) {
  return p2pvg_publish_scalars_impl(src, n, host_mapped, seq, ST);
}
int p2pvg_adam_legacy(float* p, const float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2,
                      double eps, const int* step_ptr, void* stream) {
  return p2pvg_adam_legacy_impl(p, g, m, v, n, lr, beta1, beta2, eps, step_ptr, ST);
}
int p2pvg_scale(float* x, int64_t n, float a, void* stream) { return p2pvg_scale_impl(x, n, a, ST); }

}  // extern "C"
