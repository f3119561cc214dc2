"""ctypes binding of libp2pvg_b200.so (C ABI declared in include/p2pvg_b200.h).

``CudaKernels`` is the kernel backend the engine talks to.  There is no CPU / PyTorch fallback: if the
shared library is missing the import of the product path fails loudly.
"""
from __future__ import annotations

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libp2pvg_b200.so")

F32, BF16 = 0, 1
ACT_NONE, ACT_LRELU, ACT_TANH, ACT_SIGMOID, ACT_RELU = 0, 1, 2, 3, 4

_lib = None


class KernelError(RuntimeError):
    pass


def load_library():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(p2pvg_b200 has no CPU fallback)")
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.p2pvg_last_error.restype = ctypes.c_char_p
        _lib.p2pvg_bn_workspace_bytes.restype = ctypes.c_size_t
    return _lib


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError(f"unsupported dtype {t.dtype}")


_vp = ctypes.c_void_p
_i = ctypes.c_int
_i64 = ctypes.c_int64
_f = ctypes.c_float
_d = ctypes.c_double
_sz = ctypes.c_size_t


def _p(t):
    if t is None:
        return _vp(0)
    return _vp(t.data_ptr())


class ConvFusion(ctypes.Structure):
    """p2pvg_conv_fusion_t (include/p2pvg_b200.h)."""
    _fields_ = [("fwd_stat_partial", ctypes.c_void_p), ("bwd_raw", ctypes.c_void_p), ("bwd_mean", ctypes.c_void_p),
                ("bwd_invstd", ctypes.c_void_p), ("bwd_scale", ctypes.c_void_p), ("bwd_shift", ctypes.c_void_p),
                ("bwd_stat_partial", ctypes.c_void_p), ("rows_per_group", ctypes.c_int64), ("addend_dtype", ctypes.c_int)]


class _Workspaces:
    """Scratch buffers of one device, shared by every CudaKernels view of it.  ``gen`` counts re-allocations: a captured
    CUDA graph that used a workspace is stale once it moved (TrainEngine.graph_generation)."""

    def __init__(self):
        self.gemm, self.bn, self.gen = {}, {}, 0


_BACKENDS = {}


def kernels_for(device):
    """The one kernel backend of a device (workspaces are allocated once per device, not per caller)."""
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("p2pvg_b200 has no CPU path: CUDA tensors / modules only")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _BACKENDS:
        _BACKENDS[idx] = CudaKernels(torch.device("cuda", idx))
    return _BACKENDS[idx]


class CudaKernels:
    """Launches the sm_100a kernels on the current torch CUDA stream of its device."""

    name = "cuda"

    def __init__(self, device=None):
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise RuntimeError("p2pvg_b200 needs a CUDA device (no CPU fallback)")
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._ws = _Workspaces()
        self.lane = 0   # workspace set in use: the engine switches to lane 1 for work enqueued on its side stream
        self.launches = 0
        self.gemm_flags = 0   # P2PVG_GEMM_* flags passed with every p2pvg_gemm call of this view

    def with_mode(self, tf32: bool):
        """A view of this backend (same library, same workspaces) whose fp32-operand GEMMs may (tf32=True) or may not run
        at TF32 precision.  The precision policy travels with every call; nothing is process-global."""
        import copy
        v = copy.copy(self)
        v.gemm_flags = 1 if tf32 else 0
        v.launches = 0
        return v

    @property
    def ws_gen(self):
        return self._ws.gen

    # -- helpers ---------------------------------------------------------------------------
    def _stream(self):
        return _vp(torch.cuda.current_stream(self.device).cuda_stream)

    def _ck(self, rc):
        self.launches += 1
        if rc != 0:
            raise KernelError(f"p2pvg_b200 error {rc}: {self.lib.p2pvg_last_error().decode()}")

    def gemm_workspace(self):
        ws = self._ws.gemm.get(self.lane)
        if ws is None:
            ws = self._ws.gemm[self.lane] = torch.empty(256 << 20, dtype=torch.uint8, device=self.device)
            self._ws.gen += 1
        return ws

    def bn_workspace(self, G, C):
        need = self.lib.p2pvg_bn_workspace_bytes(_i(G), _i(C))
        ws = self._ws.bn.get(self.lane)
        if ws is None or ws.numel() < need:
            ws = self._ws.bn[self.lane] = torch.empty(max(need, 16 << 20), dtype=torch.uint8, device=self.device)
            self._ws.gen += 1
        return ws

    def set_gemm_impl(self, impl: str):
        self._ck(self.lib.p2pvg_set_gemm_impl(_i({"auto": 0, "simt": 1, "tc": 2}[impl])))
        self.launches -= 1

    def set_fp32_gemm_mode(self, mode: int):
        """0: fp32 GEMMs exact on the CUDA cores; 1: K-major fp32 GEMMs on the tensor cores at TF32 precision
        (this view only; passed per call as P2PVG_GEMM_TF32)."""
        self.gemm_flags = 1 if mode else 0

    def has_tcgen05(self) -> bool:
        return bool(self.lib.p2pvg_has_tcgen05())

    # -- GEMM ------------------------------------------------------------------------------
    def gemm(self, A, B, C, M, N, K, a_mn=False, b_mn=False, lda=None, ldb=None, ldc=None, accumulate=False, bias=None,
             addend=None, ldd=None):
        lda = lda if lda is not None else (M if a_mn else K)
        ldb = ldb if ldb is not None else (N if b_mn else K)
        ldc = ldc if ldc is not None else N
        ldd = ldd if ldd is not None else N
        assert A.dtype == B.dtype
        ws = self.gemm_workspace()
        self._ck(self.lib.p2pvg_gemm(_p(A), _i(_dt(A)), _i(int(a_mn)), _i64(lda), _p(B), _i(int(b_mn)), _i64(ldb), _p(C),
                                     _i(_dt(C)), _i64(ldc), _i(M), _i(N), _i(K), _i(int(accumulate)), _p(bias), _p(addend),
                                     _i64(ldd), _p(ws), _sz(ws.numel() if ws is not None else 0), _i(self.gemm_flags), self._stream()))

    # -- implicit-GEMM convolutions ---------------------------------------------------------
    def conv_gemm(self, kind, a, b, c, N, H, W, Ck, Cn, Cm=0, ldb=None, ldc=None, bias=None, addend=None, grp_src=None,
                  imgs_per_group=0, accumulate=False, stat_partial=None):
        """kind 0..5 of p2pvg_conv_gemm (see include/p2pvg_b200.h).  H, W: small-map size.  stat_partial: fp32 buffer of
        [tiles * phases, Cn, 2] receiving the BatchNorm forward statistics of the output (epilogue fusion)."""
        taps = 9 if kind >= 3 else 16
        if ldb is None:
            ldb = taps * Ck if kind in (0, 3, 5) else taps * Cn
        if ldc is None:
            ldc = taps * Cn if kind in (1, 4) else Cn
        ws = self.gemm_workspace()
        fusion = None
        if stat_partial is not None or (addend is not None and addend.dtype == torch.bfloat16):
            fusion = ctypes.byref(ConvFusion(fwd_stat_partial=stat_partial.data_ptr() if stat_partial is not None else None,
                                             addend_dtype=_dt(addend) if addend is not None else F32))
        self._ck(self.lib.p2pvg_conv_gemm(_i(kind), _p(a), _p(b), _i64(ldb), _p(c), _i(_dt(c)), _i64(ldc), _i(N), _i(H), _i(W), _i(Ck),
                                          _i(Cn), _i(Cm), _p(bias), _p(addend), _p(grp_src), _i(imgs_per_group), _i(int(accumulate)),
                                          _p(ws), _sz(ws.numel()), fusion, self._stream()))

    # -- conv lowering ---------------------------------------------------------------------
    def im2col(self, x, col, N, H, W, C):
        self._ck(self.lib.p2pvg_im2col_k4s2p1(_p(x), _p(col), _i(_dt(x)), _i(N), _i(H), _i(W), _i(C), self._stream()))

    def col2im(self, col, y, N, Hi, Wi, C, bias=None, col2=None, grp_src=None, imgs_per_group=0, accumulate=False):
        self._ck(self.lib.p2pvg_col2im_k4s2p1(_p(col), _p(col2), _p(grp_src), _i(imgs_per_group), _p(y), _i(_dt(col)), _i(N),
                                              _i(Hi), _i(Wi), _i(C), _p(bias), _i(int(accumulate)), self._stream()))

    def im2col3(self, x, col, N, H, W, C, ld, sgn=1):
        self._ck(self.lib.p2pvg_im2col3(_p(x), _p(col), _i(_dt(x)), _i(N), _i(H), _i(W), _i(C), _i(ld), _i(sgn), self._stream()))

    def col2im3(self, col, y, N, H, W, C, ld, bias=None):
        self._ck(self.lib.p2pvg_col2im3(_p(col), _p(y), _i(_dt(col)), _i(N), _i(H), _i(W), _i(C), _i(ld), _p(bias), self._stream()))

    def maxpool2_fwd(self, x, y, N, H, W, C):
        self._ck(self.lib.p2pvg_maxpool2_fwd(_p(x), _p(y), _i(_dt(x)), _i(N), _i(H), _i(W), _i(C), self._stream()))

    def maxpool2_bwd(self, x, dy, dx, N, H, W, C):
        self._ck(self.lib.p2pvg_maxpool2_bwd(_p(x), _p(dy), _p(dx), _i(_dt(x)), _i(N), _i(H), _i(W), _i(C), self._stream()))

    def upsample2_fwd(self, x, y, N, H, W, C):
        self._ck(self.lib.p2pvg_upsample2_fwd(_p(x), _p(y), _i(_dt(x)), _i(N), _i(H), _i(W), _i(C), self._stream()))

    def upsample2_bwd(self, dy, dx, N, H, W, C):
        self._ck(self.lib.p2pvg_upsample2_bwd(_p(dy), _p(dx), _i(_dt(dy)), _i(N), _i(H), _i(W), _i(C), self._stream()))

    def gather_add(self, dst, src, grp_src, G, n):
        self._ck(self.lib.p2pvg_gather_add(_p(dst), _i(_dt(dst)), _p(src), _p(grp_src), _i(G), _i64(n), self._stream()))

    def permute4(self, src, dst, dims, strides, accumulate=False):
        d = (_i * 4)(*dims)
        s = (_i64 * 4)(*strides)
        self._ck(self.lib.p2pvg_permute4(_p(src), _i(_dt(src)), _p(dst), _i(_dt(dst)), d, s, _i(int(accumulate)), self._stream()))

    def nchw_to_nhwc_dual(self, src, dst_f32, dst_act, N, hw, C):
        """frames [N,C,hw] fp32 -> [N,hw,C] in fp32 and/or the activation dtype from one read"""
        self._ck(self.lib.p2pvg_nchw_to_nhwc_dual(_p(src), _p(dst_f32) if dst_f32 is not None else None,
                                                  _p(dst_act) if dst_act is not None else None,
                                                  _i(_dt(dst_act) if dst_act is not None else 0), _i64(N), _i(hw), _i(C), self._stream()))

    def add_indexed(self, dst, src, dst_idx, F, n):
        self._ck(self.lib.p2pvg_add_indexed(_p(dst), _p(src), _i(_dt(dst)), _p(dst_idx), _i(F), _i64(n), self._stream()))

    def transpose_batched(self, src, dst, A, P, Q):
        """dst[a][q][p] = src[a][p][q]"""
        self._ck(self.lib.p2pvg_transpose_batched(_p(src), _i(_dt(src)), _p(dst), _i(_dt(dst)), _i(A), _i(P), _i(Q), self._stream()))

    def blockdiag(self, src, dst, R, C, g):
        self._ck(self.lib.p2pvg_blockdiag(_p(src), _i(_dt(src)), _p(dst), _i(_dt(dst)), _i(R), _i(C), _i(g), self._stream()))

    def group_sum(self, inp, out, grp_src, G, F, n):
        self._ck(self.lib.p2pvg_group_sum(_p(inp), _p(out), _i(_dt(inp)), _p(grp_src), _i(G), _i(F), _i64(n), self._stream()))

    # -- batch norm ------------------------------------------------------------------------
    def bn_fwd_stats(self, x, G, R, C, gamma, beta, mean, invstd, var_unb, scale, shift, eps=1e-5):
        ws = self.bn_workspace(G, C)
        self._ck(self.lib.p2pvg_bn_fwd_stats(_p(x), _i(_dt(x)), _i(G), _i64(R), _i(C), _p(gamma), _p(beta), _f(eps), _p(ws),
                                             _sz(ws.numel()), _p(mean), _p(invstd), _p(var_unb), _p(scale), _p(shift),
                                             self._stream()))

    def bn_fwd_finalize_tiles(self, partial, parts_per_group, ldp, fold, G, R, C, gamma, beta, mean, invstd, var_unb, scale, shift, eps=1e-5):
        self._ck(self.lib.p2pvg_bn_fwd_finalize_tiles(_p(partial), _i(parts_per_group), _i(ldp), _i(fold), _i(G), _i64(R), _i(C), _p(gamma),
                                                      _p(beta), _f(eps), _p(mean), _p(invstd), _p(var_unb), _p(scale), _p(shift),
                                                      self._stream()))

    def bn_bwd_finalize_tiles(self, partial, parts_per_group, ldp, fold, G, C, sum_dz, sum_dzx):
        self._ck(self.lib.p2pvg_bn_bwd_finalize_tiles(_p(partial), _i(parts_per_group), _i(ldp), _i(fold), _i(G), _i(C), _p(sum_dz),
                                                      _p(sum_dzx), self._stream()))

    def bn_bwd_apply(self, dy, x, y, mean, invstd, gamma, G, R, C, act, dx, sum_dz, sum_dzx, scale=None, shift=None):
        self._ck(self.lib.p2pvg_bn_bwd_apply(_p(dy), _p(x), _p(y), _i(_dt(x)), _p(mean), _p(invstd), _p(gamma), _i(G), _i64(R), _i(C),
                                             _i(act), _p(dx), _p(sum_dz), _p(sum_dzx), _p(scale), _p(shift), self._stream()))

    def bn_act(self, x, y, scale, shift, G, R, C, act):
        self._ck(self.lib.p2pvg_bn_act(_p(x), _p(y), _i(_dt(x)), _p(scale), _p(shift), _i(G), _i64(R), _i(C), _i(act), self._stream()))

    def bn_bwd(self, dy, x, y, mean, invstd, gamma, G, R, C, act, dx, sum_dz, sum_dzx, scale=None, shift=None):
        """y=None (LeakyReLU only): derivative recomputed from sign(x*scale+shift)."""
        ws = self.bn_workspace(G, C)
        self._ck(self.lib.p2pvg_bn_bwd(_p(dy), _p(x), _p(y), _i(_dt(x)), _p(mean), _p(invstd), _p(gamma), _i(G), _i64(R), _i(C),
                                       _i(act), _p(ws), _sz(ws.numel()), _p(dx), _p(sum_dz), _p(sum_dzx), _p(scale), _p(shift),
                                       self._stream()))

    def bn_param_grad(self, sum_dz, sum_dzx, G, C, dgamma, dbeta):
        self._ck(self.lib.p2pvg_bn_param_grad(_p(sum_dz), _p(sum_dzx), _i(G), _i(C), _p(dgamma), _p(dbeta), self._stream()))

    def bn_eval_coeffs(self, gamma, beta, rmean, rvar, C, scale, shift, eps=1e-5):
        self._ck(self.lib.p2pvg_bn_eval_coeffs(_p(gamma), _p(beta), _p(rmean), _p(rvar), _f(eps), _i(C), _p(scale), _p(shift),
                                               self._stream()))

    def bn_ema(self, rmean, rvar, mean, var_unb, order, ncalls, C, momentum=0.1):
        self._ck(self.lib.p2pvg_bn_ema(_p(rmean), _p(rvar), _p(mean), _p(var_unb), _p(order), _i(ncalls), _i(C), _f(momentum),
                                       self._stream()))

    # -- recurrent phase -------------------------------------------------------------------
    def lstm_pointwise_fwd(self, gates, c_prev, c_out, h_out, B, R):
        self._ck(self.lib.p2pvg_lstm_pointwise_fwd(_p(gates), _p(c_prev), _p(c_out), _p(h_out), _i(B), _i(R), self._stream()))

    def lstm_pointwise_bwd(self, dh, dc_next, gates, c_prev, c, dgates, dc_prev, B, R):
        self._ck(self.lib.p2pvg_lstm_pointwise_bwd(_p(dh), _p(dc_next), _p(gates), _p(c_prev), _p(c), _p(dgates), _p(dc_prev), _i(B),
                                                   _i(R), self._stream()))

    def lstm_scan_fwd(self, pre, whh, bhh, gates, hs, cs, S, B, R, counter, tf32=False):
        self._ck(self.lib.p2pvg_lstm_scan_fwd(_p(pre), _p(whh), _p(bhh), _p(gates), _p(hs), _p(cs), _i(S), _i(B), _i(R), _i(int(tf32)),
                                              _p(counter), self._stream()))

    def lstm_scan_bwd(self, dhtop, whh, gates, cs, dG, S, B, R, counter, tf32=False):
        self._ck(self.lib.p2pvg_lstm_scan_bwd(_p(dhtop), _p(whh), _p(gates), _p(cs), _p(dG), _i(S), _i(B), _i(R), _i(int(tf32)),
                                              _p(counter), self._stream()))

    def reparam_kl_fwd(self, mu, lv, mu_p, lv_p, eps, eps_p, z, z_p, n, kl_sum):
        self._ck(self.lib.p2pvg_reparam_kl_fwd(_p(mu), _p(lv), _p(mu_p), _p(lv_p), _p(eps), _p(eps_p), _p(z), _p(z_p), _i(n),
                                               _p(kl_sum), self._stream()))

    def reparam_kl_bwd(self, mu, lv, mu_p, lv_p, eps, eps_p, dz, dz_p, kl_coef, dmu, dlv, dmu_p, dlv_p, n):
        self._ck(self.lib.p2pvg_reparam_kl_bwd(_p(mu), _p(lv), _p(mu_p), _p(lv_p), _p(eps), _p(eps_p), _p(dz), _p(dz_p),
                                               _f(kl_coef), _p(dmu), _p(dlv), _p(dmu_p), _p(dlv_p), _i(n), self._stream()))

    def build_concat(self, dst, A, ia, ga, Bm, ib, gb, tuc, dt, S, B, ld=None):
        self._ck(self.lib.p2pvg_build_concat(_p(dst), _p(A), _p(ia), _i(ga), _p(Bm), _p(ib), _i(gb), _p(tuc), _p(dt), _i(S), _i(B),
                                             _i(ld if ld is not None else ga + gb + 2), self._stream()))

    def gather_add_cols(self, dst, src, idx, S, T, B, g, W, col0, init=False):
        self._ck(self.lib.p2pvg_gather_add_cols(_p(dst), _p(src), _p(idx), _i(S), _i(T), _i(B), _i(g), _i(W), _i(col0),
                                                _i(int(init)), self._stream()))

    def align(self, H, in_idx, h_pred, P, B, g, coef, loss_partial, d_hpred, dH):
        self._ck(self.lib.p2pvg_align(_p(H), _p(in_idx), _p(h_pred), _i(P), _i(B), _i(g), _f(coef), _p(loss_partial), _p(d_hpred),
                                      _p(dH), self._stream()))

    def colsum(self, x, rows, cols, ld, out, accumulate=False):
        ws = self.bn_workspace(1, 1)
        self._ck(self.lib.p2pvg_colsum(_p(x), _i(_dt(x)), _i64(rows), _i(cols), _i64(ld), _p(out), _i(int(accumulate)), _p(ws),
                                       _sz(ws.numel()), self._stream()))

    def act_fwd(self, x, n, act):
        self._ck(self.lib.p2pvg_act_fwd(_p(x), _i64(n), _i(act), self._stream()))

    def act_bwd(self, dy, y, dx, n, act):
        self._ck(self.lib.p2pvg_act_bwd(_p(dy), _p(y), _p(dx), _i64(n), _i(act), self._stream()))

    # -- losses / optimiser ----------------------------------------------------------------
    def mse_chunks(self):
        return int(self.lib.p2pvg_mse_chunks())

    def sigmoid_mse(self, raw, x, tgt, coef, G, E, pred, d_raw, partial):
        self._ck(self.lib.p2pvg_sigmoid_mse(_p(raw), _i(_dt(raw)), _p(x), _p(tgt), _p(coef), _i(G), _i64(E), _p(pred), _p(d_raw),
                                            _p(partial), self._stream()))

    def convt_c1_loss(self, col, col2, grp_src, bias, x, tgt, coef, G, B, Hi, Wi, d_raw, partial, C=1):
        self._ck(self.lib.p2pvg_convt_c1_loss(_p(col), _p(col2), _i(_dt(col)), _p(grp_src), _p(bias), _p(x), _p(tgt), _p(coef), _i(G), _i(B),
                                              _i(Hi), _i(Wi), _i(C), _p(d_raw), _p(partial), self._stream()))

    def layernorm_fwd(self, x, gamma, beta, y, mean, rstd, rows, C, eps=1e-5):
        self._ck(self.lib.p2pvg_layernorm_fwd(_p(x), _p(gamma), _p(beta), _p(y), _p(mean), _p(rstd), _i64(rows), _i(C), _f(eps), self._stream()))

    def layernorm_bwd(self, dy, x, mean, rstd, gamma, dx, dgamma, dbeta, rows, C):
        ws = self.bn_workspace(1, 1)
        self._ck(self.lib.p2pvg_layernorm_bwd(_p(dy), _p(x), _p(mean), _p(rstd), _p(gamma), _p(dx), _p(dgamma), _p(dbeta), _i64(rows), _i(C),
                                              _p(ws), _sz(ws.numel()), self._stream()))

    def mse_plain(self, pred, x, tgt, coef, G, E, d_pred, partial):
        self._ck(self.lib.p2pvg_mse_plain(_p(pred), _p(x), _p(tgt), _p(coef), _i(G), _i64(E), _p(d_pred), _p(partial), self._stream()))

    def publish_scalars(self, src, n, host_pinned, seq):
        """src[0..n) + *seq -> page-locked host memory (zero-copy store from the device)"""
        self._ck(self.lib.p2pvg_publish_scalars(_p(src), _i(n), _vp(host_pinned.data_ptr()), _p(seq), self._stream()))

    def finalize_losses(self, mse_partial, n_recon, has_cpc, E, kl_sum, batch_size, align_partial, n_align, seq_len, out):
        self._ck(self.lib.p2pvg_finalize_losses(_p(mse_partial), _i(n_recon), _i(int(has_cpc)), _d(float(E)), _p(kl_sum),
                                                _f(batch_size), _p(align_partial), _i(n_align), _f(seq_len), _p(out),
                                                self._stream()))

    def adam(self, p, g, m, v, n, lr, beta1, beta2, eps, step_t):
        self._ck(self.lib.p2pvg_adam_legacy(_p(p), _p(g), _p(m), _p(v), _i64(n), _d(lr), _d(beta1), _d(beta2), _d(eps),
                                            _p(step_t), self._stream()))

    def scale(self, x, n, a):
        self._ck(self.lib.p2pvg_scale(_p(x), _i64(n), _f(a), self._stream()))
