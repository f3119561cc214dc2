"""Every CUDA kernel of libp2pvg_b200.so (called through the C ABI) against the torch emulation of the
same entry point (tests/emu_backend.py), fp32 and bf16, including ragged / tail shapes."""
import pytest
import torch

pytestmark = pytest.mark.gpu

ACT_NONE, ACT_LRELU, ACT_TANH = 0, 1, 2


@pytest.fixture(scope="module")
def KS():
    from p2pvg_b200._lib import CudaKernels
    from tests.emu_backend import EmuKernels
    return CudaKernels("cuda"), EmuKernels("cuda")


def rnd(*shape, dtype=torch.float32, scale=1.0, seed=None):
    if seed is not None:
        torch.manual_seed(seed)
    return (torch.randn(*shape, device="cuda") * scale).to(dtype)


def close(a, b, dtype=torch.float32, rtol=None, atol=None, what=""):
    if rtol is None:
        rtol, atol = (1e-4, 1e-5) if dtype == torch.float32 else (1.6e-2, 1e-2)
    a, b = a.float(), b.float()
    err = (a - b).abs()
    tol = atol + rtol * b.abs()
    bad = (err > tol).sum().item()
    assert bad == 0, f"{what}: {bad}/{a.numel()} mismatches, max err {err.max().item():.3e}"


DT = [torch.float32, torch.bfloat16]


@pytest.mark.parametrize("impl", ["simt"])
@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("a_mn,b_mn", [(False, False), (False, True), (True, True), (True, False)])
@pytest.mark.parametrize("M,N,K", [(70, 50, 33), (256, 128, 64), (5, 10, 258), (130, 1024, 17)])
def test_gemm_simt(KS, impl, dtype, a_mn, b_mn, M, N, K):
    Kc, Ke = KS
    Kc.set_gemm_impl(impl)
    try:
        A = rnd(K, M, dtype=dtype, seed=1) if a_mn else rnd(M, K, dtype=dtype, seed=1)
        B = rnd(K, N, dtype=dtype) if b_mn else rnd(N, K, dtype=dtype)
        bias = rnd(N)
        add = rnd(M, N, dtype=dtype)
        for cdt in ([dtype] if dtype == torch.float32 else [torch.float32, torch.bfloat16]):
            add_c = add.to(cdt)
            C1 = rnd(M, N, dtype=cdt)
            C2 = C1.clone()
            for acc in (False, True):
                Kc.gemm(A, B, C1, M, N, K, a_mn=a_mn, b_mn=b_mn, accumulate=acc, bias=bias, addend=add_c)
                Ke.gemm(A, B, C2, M, N, K, a_mn=a_mn, b_mn=b_mn, accumulate=acc, bias=bias, addend=add_c)
                close(C1, C2, cdt, rtol=1e-4 if cdt == torch.float32 else 1.6e-2, atol=1e-3 if dtype == torch.float32 else 5e-2,
                      what=f"gemm acc={acc}")
    finally:
        Kc.set_gemm_impl("auto")


TC_SHAPES = [
    # M, N, K, a_mn, b_mn
    (128, 128, 64, False, False), (256, 128, 256, False, False), (300, 200, 136, False, False),
    (128, 64, 64, False, False), (70, 16, 128, False, False), (1000, 48, 72, False, False),
    (256, 128, 128, False, True), (192, 4096, 128, False, True), (130, 16, 128, False, True),
    (128, 128, 128, True, True), (64, 1024, 4096, True, True), (512, 136, 1000, True, True), (128, 16, 3000, True, True),
    (256, 128, 64, True, False), (104, 72, 200, True, False),
    (128, 128, 16, False, False), (2048, 64, 16, False, False), (64, 1024, 100000, True, True),
]


@pytest.mark.parametrize("M,N,K,a_mn,b_mn", TC_SHAPES)
def test_gemm_tcgen05(KS, M, N, K, a_mn, b_mn):
    Kc, Ke = KS
    assert Kc.has_tcgen05(), "driver entry point cuTensorMapEncodeTiled not available"
    Kc.set_gemm_impl("tc")
    try:
        dt = torch.bfloat16
        A = rnd(K, M, dtype=dt, seed=21) if a_mn else rnd(M, K, dtype=dt, seed=21)
        B = rnd(K, N, dtype=dt) if b_mn else rnd(N, K, dtype=dt)
        bias = rnd(N)
        for cdt in (torch.float32, torch.bfloat16):
            add = rnd(M, N, dtype=cdt)
            C1 = rnd(M, N, dtype=cdt)
            C2 = C1.clone()
            Kc.gemm(A, B, C1, M, N, K, a_mn=a_mn, b_mn=b_mn)
            Ke.gemm(A, B, C2, M, N, K, a_mn=a_mn, b_mn=b_mn)
            tol = dict(rtol=2e-3, atol=2e-3 * K ** 0.5) if cdt == torch.float32 else dict(rtol=1.6e-2, atol=1e-2 * K ** 0.5)
            close(C1, C2, cdt, what="plain", **tol)
            Kc.gemm(A, B, C1, M, N, K, a_mn=a_mn, b_mn=b_mn, accumulate=True, bias=bias, addend=add)
            Ke.gemm(A, B, C2, M, N, K, a_mn=a_mn, b_mn=b_mn, accumulate=True, bias=bias, addend=add)
            close(C1, C2, cdt, what="acc+bias+addend", **tol)
    finally:
        Kc.set_gemm_impl("auto")


def test_gemm_tcgen05_strided_views(KS):
    """Sub-matrix operands (leading dimension > extent), as the engine uses for packed weight halves."""
    Kc, Ke = KS
    Kc.set_gemm_impl("tc")
    try:
        big = rnd(512, 256, dtype=torch.bfloat16, seed=22)
        A = big[:, 64:]          # [512, 192] with lda = 256  (offset 128 B: 16-byte aligned)
        Bm = rnd(96, 192, dtype=torch.bfloat16)
        C1 = torch.zeros(512, 96, device="cuda")
        C2 = torch.zeros_like(C1)
        Kc.gemm(A, Bm, C1, 512, 96, 192, lda=256)
        Ke.gemm(A, Bm, C2, 512, 96, 192, lda=256)
        close(C1, C2, rtol=2e-3, atol=3e-2)
    finally:
        Kc.set_gemm_impl("auto")


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("N,H,C", [(3, 8, 64), (2, 16, 1), (2, 8, 3), (1, 64, 4)])
def test_im2col_col2im(KS, dtype, N, H, C):
    Kc, Ke = KS
    x = rnd(N, H, H, C, dtype=dtype, seed=2)
    Ho = H // 2
    c1 = torch.empty(N * Ho * Ho * 16 * C, device="cuda", dtype=dtype)
    c2 = torch.empty_like(c1)
    Kc.im2col(x, c1, N, H, H, C)
    Ke.im2col(x, c2, N, H, H, C)
    assert torch.equal(c1, c2)
    # col2im with a shared second operand and bias
    col = rnd(N * Ho * Ho, 16 * C, dtype=dtype)
    G, ipg = N, 1
    colS = rnd(2 * ipg * Ho * Ho, 16 * C, dtype=dtype)
    src = torch.tensor([i % 2 for i in range(G)], dtype=torch.int32, device="cuda")
    bias = rnd(C)
    for acc in (False, True):
        y1 = rnd(N, H, H, C, dtype=dtype, seed=3)
        y2 = y1.clone()
        Kc.col2im(col, y1, N, Ho, Ho, C, bias=bias, col2=colS, grp_src=src, imgs_per_group=ipg, accumulate=acc)
        Ke.col2im(col, y2, N, Ho, Ho, C, bias=bias, col2=colS, grp_src=src, imgs_per_group=ipg, accumulate=acc)
        close(y1, y2, dtype, what="col2im")
    y1 = torch.empty(N, H, H, C, device="cuda", dtype=dtype)
    y2 = torch.empty_like(y1)
    Kc.col2im(col, y1, N, Ho, Ho, C)
    Ke.col2im(col, y2, N, Ho, Ho, C)
    close(y1, y2, dtype, what="col2im plain")


def test_col2im_is_adjoint_of_im2col(KS):
    Kc, _ = KS
    N, H, C = 2, 8, 8
    x = rnd(N, H, H, C, seed=4)
    col = torch.empty(N * 16 * 16 * C, device="cuda")
    Kc.im2col(x, col, N, H, H, C)
    w = rnd(col.numel())
    y = torch.empty(N, H, H, C, device="cuda")
    Kc.col2im(w, y, N, H // 2, H // 2, C)
    assert abs((col * w).sum().item() - (x * y).sum().item()) < 1e-2


@pytest.mark.parametrize("sd,dd", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16), (torch.bfloat16, torch.float32)])
def test_permute4(KS, sd, dd):
    Kc, Ke = KS
    w = rnd(6, 5, 4, 4, dtype=sd, seed=5)
    d1 = torch.zeros(6 * 16 * 5, device="cuda", dtype=dd)
    d2 = d1.clone()
    for acc in (False, True):
        Kc.permute4(w, d1, (6, 4, 4, 5), (5 * 16, 4, 1, 16), accumulate=acc)
        Ke.permute4(w, d2, (6, 4, 4, 5), (5 * 16, 4, 1, 16), accumulate=acc)
        close(d1, d2, dd, what="permute4")
    assert torch.equal(d2.float().reshape(6, 4, 4, 5)[:, 1, 2, 3], (2 * w.float()[:, 3, 1, 2]).to(dd).float())


@pytest.mark.parametrize("sd,dd", [(torch.float32, torch.bfloat16), (torch.bfloat16, torch.float32), (torch.float32, torch.float32),
                                   (torch.bfloat16, torch.bfloat16)])
@pytest.mark.parametrize("n", [4 * 1000 + 0, 4 * 1000 + 3, 1 << 20])
def test_permute4_flat_cast(KS, sd, dd, n):
    """contiguous copy / cast (the bf16 operand copies of the LSTM weight-gradient GEMMs): 16-byte-vector path when the length
    is a multiple of 4, generic path otherwise; both are exact round-to-nearest casts"""
    Kc, _ = KS
    src = rnd(n, dtype=sd, seed=9)
    dst = torch.zeros(n + 8, device="cuda", dtype=dd)
    Kc.permute4(src, dst, (n, 1, 1, 1), (1, 0, 0, 0))
    assert torch.equal(dst[:n], src.to(dd)) and not dst[n:].any()
    dst.zero_()
    Kc.permute4(src, dst, (1, n, 1, 1), (0, 1, 0, 0))
    assert torch.equal(dst[:n], src.to(dd)) and not dst[n:].any()
    if n % 8 == 0:   # contiguous source described with several dims (one-channel frames: NCHW == NHWC)
        dst.zero_()
        Kc.permute4(src, dst, (n // 8, 8, 1, 1), (8, 1, 8, 0))
        assert torch.equal(dst[:n], src.to(dd)) and not dst[n:].any()
        dst.zero_()
        Kc.permute4(src, dst, (n // 8, 2, 4, 1), (8, 1, 2, 0))   # a real permutation of the same data: generic path
        assert torch.equal(dst[:n], src.view(n // 8, 4, 2).transpose(1, 2).reshape(-1).to(dd))


@pytest.mark.parametrize("C", [2, 3, 4])
@pytest.mark.parametrize("adt", [torch.bfloat16, torch.float32, None])
def test_nchw_to_nhwc_dual(KS, C, adt):
    """frames NCHW -> channels-last in fp32 and the activation dtype from one read: a pure data movement, bit exact against
    torch.permute (+ round-to-nearest bf16 cast)"""
    Kc, _ = KS
    N, H = 37, 12
    x = rnd(N, C, H, H, seed=40 + C)
    d32 = torch.zeros(N * H * H * C, device="cuda")
    da = torch.zeros(N * H * H * C, device="cuda", dtype=adt) if adt is not None else None
    Kc.nchw_to_nhwc_dual(x, d32, da, N, H * H, C)
    want = x.permute(0, 2, 3, 1).contiguous().view(-1)
    assert torch.equal(d32, want)
    if da is not None:
        assert torch.equal(da, want.to(adt))
        d32b = torch.zeros_like(d32)
        Kc.nchw_to_nhwc_dual(x, None, da.zero_(), N, H * H, C)      # activation copy only
        assert torch.equal(da, want.to(adt)) and not d32b.any()
    with pytest.raises(RuntimeError):
        Kc.nchw_to_nhwc_dual(x, d32, da, N, H * H - 2, C)           # H*W % 4 != 0 is an error, not a fallback


@pytest.mark.parametrize("dtype", DT)
def test_add_indexed_group_sum(KS, dtype):
    Kc, Ke = KS
    n = 64
    dst = rnd(5, n, dtype=dtype, seed=6)
    d2 = dst.clone()
    src = rnd(2, n, dtype=dtype)
    idx = torch.tensor([3, 1], dtype=torch.int32, device="cuda")
    Kc.add_indexed(dst, src, idx, 2, n)
    Ke.add_indexed(d2, src, idx, 2, n)
    close(dst, d2, dtype)
    inp = rnd(6, n, dtype=dtype)
    gs = torch.tensor([0, 2, 0, 1, 2, 2], dtype=torch.int32, device="cuda")
    o1 = torch.empty(3, n, device="cuda", dtype=dtype)
    o2 = torch.empty_like(o1)
    Kc.group_sum(inp, o1, gs, 6, 3, n)
    Ke.group_sum(inp, o2, gs, 6, 3, n)
    close(o1, o2, dtype)


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("G,R,C,act", [(3, 50, 64, ACT_LRELU), (4, 3, 128, ACT_TANH), (2, 1000, 512, ACT_LRELU), (5, 37, 256, ACT_LRELU)])
def test_batchnorm(KS, dtype, G, R, C, act):
    Kc, Ke = KS
    x = rnd(G, R, C, dtype=dtype, seed=7) * 2 + 0.5
    gamma, beta = rnd(C) * 0.1 + 1, rnd(C) * 0.1
    outs = []
    for K in (Kc, Ke):
        st = [torch.zeros(G * C, device="cuda") for _ in range(5)]
        K.bn_fwd_stats(x, G, R, C, gamma, beta, *st)
        y = torch.empty_like(x)
        K.bn_act(x, y, st[3], st[4], G, R, C, act)
        outs.append((st, y))
    for a, b in zip(outs[0][0], outs[1][0]):
        close(a, b, rtol=2e-4, atol=1e-5, what="bn stats")
    close(outs[0][1], outs[1][1], dtype, what="bn act")
    st, y = outs[1]
    dy = rnd(G, R, C, dtype=dtype)
    res = []
    for K in (Kc, Ke):
        dx = torch.empty_like(x)
        s0, s1 = torch.zeros(G * C, device="cuda"), torch.zeros(G * C, device="cuda")
        K.bn_bwd(dy, x, y, st[0], st[1], gamma, G, R, C, act, dx, s0, s1)
        dg, db = torch.zeros(C, device="cuda"), torch.zeros(C, device="cuda")
        K.bn_param_grad(s0, s1, G, C, dg, db)
        res.append((dx, s0, s1, dg, db))
    close(res[0][0], res[1][0], dtype, what="bn dx")
    for i in range(1, 5):
        close(res[0][i], res[1][i], rtol=1e-3, atol=1e-3 * max(1.0, R ** 0.5), what=f"bn sums {i}")
    # EMA in call order
    order = torch.tensor([G - 1, 0, 1, 0], dtype=torch.int32, device="cuda")
    r = []
    for K in (Kc, Ke):
        rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
        K.bn_ema(rm, rv, st[0], st[2], order, 4, C)
        r.append((rm, rv))
    close(r[0][0], r[1][0], rtol=1e-6, atol=1e-7)
    close(r[0][1], r[1][1], rtol=1e-6, atol=1e-7)


def test_batchnorm_matches_torch(KS):
    Kc, _ = KS
    G, B, H, C = 3, 4, 8, 64
    x = rnd(G, B * H * H, C, seed=8) * 3 + 1
    gamma, beta = rnd(C) + 1, rnd(C)
    st = [torch.zeros(G * C, device="cuda") for _ in range(5)]
    Kc.bn_fwd_stats(x, G, B * H * H, C, gamma, beta, *st)
    y = torch.empty_like(x)
    Kc.bn_act(x, y, st[3], st[4], G, B * H * H, C, ACT_NONE)
    for g in range(G):
        xn = x[g].reshape(B, H, H, C).permute(0, 3, 1, 2)
        ref = torch.nn.functional.batch_norm(xn, None, None, gamma, beta, True, 0.1, 1e-5)
        close(y[g].reshape(B, H, H, C).permute(0, 3, 1, 2), ref, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_bn_bwd_without_activation_tensor(KS, dtype):
    K, _ = KS
    torch.manual_seed(2)
    G, R, C = 3, 200, 64
    x = (torch.randn(G, R, C, device="cuda") * 2 + 0.3).to(dtype)
    gamma, beta = torch.randn(C, device="cuda") * 0.1 + 1, torch.randn(C, device="cuda") * 0.1
    st = [torch.zeros(G * C, device="cuda") for _ in range(5)]
    K.bn_fwd_stats(x, G, R, C, gamma, beta, *st)
    y = torch.empty_like(x)
    K.bn_act(x, y, st[3], st[4], G, R, C, 1)
    dy = torch.randn(G, R, C, device="cuda").to(dtype)
    outs = []
    for use_y in (True, False):
        dx = torch.empty_like(x)
        s0, s1 = torch.zeros(G * C, device="cuda"), torch.zeros(G * C, device="cuda")
        if use_y:
            K.bn_bwd(dy, x, y, st[0], st[1], gamma, G, R, C, 1, dx, s0, s1)
        else:
            K.bn_bwd(dy, x, None, st[0], st[1], gamma, G, R, C, 1, dx, s0, s1, scale=st[3], shift=st[4])
        outs.append((dx, s0, s1))
    for a, b in zip(*outs):
        assert torch.equal(a, b) or (a.float() - b.float()).abs().max().item() <= 1e-6


def test_lstm_pointwise_and_reparam(KS):
    Kc, Ke = KS
    B, R = 7, 256
    res = []
    for K in (Kc, Ke):
        gates = rnd(B, 4 * R, seed=9)
        cp = rnd(B, R)
        c, h = torch.empty(B, R, device="cuda"), torch.empty(B, R, device="cuda")
        K.lstm_pointwise_fwd(gates, cp, c, h, B, R)
        dh, dcn = rnd(B, R), rnd(B, R)
        dg, dcp = torch.empty(B, 4 * R, device="cuda"), torch.empty(B, R, device="cuda")
        K.lstm_pointwise_bwd(dh, dcn, gates, cp, c, dg, dcp, B, R)
        dg2, dcp2 = torch.empty_like(dg), torch.empty_like(dcp)
        K.lstm_pointwise_bwd(dh, None, gates, cp, c, dg2, dcp2, B, R)
        res.append((gates, c, h, dg, dcp, dg2, dcp2))
    for a, b in zip(*res):
        close(a, b, rtol=2e-5, atol=2e-6)
    n = 5 * 3 * 10
    res = []
    for K in (Kc, Ke):
        torch.manual_seed(10)
        mu, lv, mup, lvp, e, ep, dz, dzp = (rnd(n) * 0.5 for _ in range(8))
        z, zp, kl = torch.empty(n, device="cuda"), torch.empty(n, device="cuda"), torch.zeros(4, device="cuda")
        K.reparam_kl_fwd(mu, lv, mup, lvp, e, ep, z, zp, n, kl)
        outs = [torch.empty(n, device="cuda") for _ in range(4)]
        K.reparam_kl_bwd(mu, lv, mup, lvp, e, ep, dz, None, 0.3, *outs, n)
        outs2 = [torch.empty(n, device="cuda") for _ in range(4)]
        K.reparam_kl_bwd(mu, lv, mup, lvp, e, ep, None, dzp, 1.0, *outs2, n)
        res.append([z, zp, kl[:1]] + outs + outs2)
    for a, b in zip(*res):
        close(a, b, rtol=2e-5, atol=2e-6)


def test_concat_gather_align_colsum_act(KS):
    Kc, Ke = KS
    T, B, g, z, S = 6, 3, 128, 10, 4
    H = rnd(T, B, g, seed=11)
    Z = rnd(S, B, z)
    ia = torch.tensor([0, 2, 3, 4], dtype=torch.int32, device="cuda")
    ib = torch.tensor([0, 1, 2, 3], dtype=torch.int32, device="cuda")
    tuc, dt = rnd(S), rnd(S)
    W = g + z + 2
    res = []
    for K in (Kc, Ke):
        dst = torch.empty(S, B, W, device="cuda")
        K.build_concat(dst, H, ia, g, Z, ib, z, tuc, dt, S, B)
        dH = torch.zeros(T, B, g, device="cuda")
        K.gather_add_cols(dH, dst, ia, S, T, B, g, W, 0, init=True)
        K.gather_add_cols(dH, dst, torch.full((S,), T - 1, dtype=torch.int32, device="cuda"), S, T, B, g, W, 0)
        hp = rnd(S, B, g, seed=12)
        lp = torch.zeros(S, device="cuda")
        dhp = torch.ones(S, B, g, device="cuda")
        K.align(H, ia, hp, S - 1, B, g, 0.5, lp, dhp, dH)
        cs = torch.zeros(W, device="cuda")
        K.colsum(dst, S * B, W, W, cs)
        K.colsum(dst, S * B, W, W, cs, accumulate=True)
        a = dst.clone()
        K.act_fwd(a, a.numel(), ACT_TANH)
        da = torch.empty_like(a)
        K.act_bwd(dst, a, da, a.numel(), ACT_TANH)
        res.append((dst, dH, lp, dhp, cs, a, da))
    for i, (a, b) in enumerate(zip(*res)):
        close(a, b, rtol=2e-5, atol=2e-5, what=f"item {i}")


@pytest.mark.parametrize("dtype", DT)
def test_sigmoid_mse_finalize_adam(KS, dtype):
    Kc, Ke = KS
    G, E, T = 3, 2 * 64 * 64, 5
    raw = rnd(G, E, dtype=dtype, seed=13)
    x = torch.rand(T, E, device="cuda")
    tgt = torch.tensor([1, 2, 4], dtype=torch.int32, device="cuda")
    coef = torch.tensor([1.0 / E, 1.0 / E, 100.0 / E], device="cuda")
    res = []
    for K in (Kc, Ke):
        pred, draw = torch.empty_like(raw), torch.empty_like(raw)
        part = torch.zeros(G * 32, device="cuda")
        K.sigmoid_mse(raw, x, tgt, coef, G, E, pred, draw, part)
        kl = torch.tensor([3.0, 0, 0, 0], device="cuda")
        al = torch.tensor([0.1, 0.2], device="cuda")
        out = torch.zeros(4, device="cuda")
        K.finalize_losses(part, G - 1, True, E, kl, 4.0, al, 2, float(T), out)
        res.append((pred, draw, part.reshape(G, 32).sum(1), out))
    close(res[0][0], res[1][0], dtype)
    close(res[0][1], res[1][1], dtype, rtol=2e-2, atol=1e-6)
    close(res[0][2], res[1][2], rtol=1e-4, atol=1e-3)
    close(res[0][3], res[1][3], rtol=1e-4, atol=1e-6)
    n = 1000
    res = []
    for K in (Kc, Ke):
        torch.manual_seed(14)
        p, g, m, v = rnd(n), rnd(n) * 1e-3, rnd(n) * 1e-4, rnd(n).abs() * 1e-6
        step = torch.tensor([3], dtype=torch.int32, device="cuda")
        K.adam(p, g, m, v, n, 1e-3, 0.9, 0.999, 1e-8, step)
        res.append((p, m, v))
    for a, b in zip(*res):
        close(a, b, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("Hi", [8, 6, 32])
def test_convt_c1_loss_equals_col2im_plus_sigmoid_mse(C, Hi):
    """Fused last decoder layer (tap gather + bias + sigmoid + MSE + d raw) against the two-kernel path it replaces.
    Several image sizes (the gather handles the borders per pixel)."""
    from p2pvg_b200._lib import CudaKernels
    K = CudaKernels("cuda")
    torch.manual_seed(0)
    G, B, nsrc, T = 5, 3, 2, 7
    N = G * B
    col = (torch.randn(N * Hi * Hi, 16 * C, device="cuda") * 0.5).bfloat16()
    col2 = (torch.randn(nsrc * B * Hi * Hi, 16 * C, device="cuda") * 0.5).bfloat16()
    src = torch.tensor([0, 1, 1, 0, 1], dtype=torch.int32, device="cuda")
    tgt = torch.tensor([1, 2, 3, 4, 6], dtype=torch.int32, device="cuda")
    bias = torch.tensor([0.3, -0.2, 0.1][:C], device="cuda")
    E = B * 4 * Hi * Hi * C
    x = torch.rand(T, E, device="cuda")
    coef = torch.rand(G, device="cuda") + 0.5
    raw = torch.empty(N * 4 * Hi * Hi * C, device="cuda", dtype=torch.bfloat16)
    K.col2im(col, raw, N, Hi, Hi, C, bias=bias, col2=col2, grp_src=src, imgs_per_group=B)
    d_ref = torch.empty_like(raw)
    p_ref = torch.zeros(G * K.mse_chunks(), device="cuda")
    K.sigmoid_mse(raw, x, tgt, coef, G, E, None, d_ref, p_ref)
    d_got = torch.empty_like(raw)
    p_got = torch.zeros(G * K.mse_chunks(), device="cuda")
    K.convt_c1_loss(col, col2, src, bias, x, tgt, coef, G, B, Hi, Hi, d_got, p_got, C=C)
    # the two-kernel path rounds the pre-sigmoid value to bf16 once more than the fused one
    assert torch.allclose(p_got.reshape(G, -1).sum(1), p_ref.reshape(G, -1).sum(1), rtol=5e-3)
    assert (d_got.float() - d_ref.float()).abs().max().item() <= 2e-2 * d_ref.float().abs().max().item()
    # exact check against torch on the same bf16 operands: col is [pixel][tap][channel]
    c = col.float().reshape(G, B, Hi, Hi, 4, 4, C)
    c2 = col2.float().reshape(nsrc, B, Hi, Hi, 4, 4, C)[src.long()]
    tot = (c + c2).permute(0, 1, 6, 4, 5, 2, 3).reshape(N, C * 16, Hi * Hi)   # fold wants [N, C*kh*kw, L]
    want = torch.nn.functional.fold(tot, (2 * Hi, 2 * Hi), kernel_size=4, stride=2, padding=1)   # [N, C, 2Hi, 2Hi]
    want = (want + bias.view(1, C, 1, 1)).permute(0, 2, 3, 1).reshape(G, E)                      # NHWC per group
    s = torch.sigmoid(want)
    diff = s - x[tgt.long()]
    assert torch.allclose(p_got.reshape(G, -1).sum(1), (diff * diff).sum(1), rtol=1e-4)
    dref = coef[:, None] * 2 * diff * s * (1 - s)
    assert (d_got.float().reshape(G, E) - dref).abs().max().item() <= 1e-2 * dref.abs().max().item()
