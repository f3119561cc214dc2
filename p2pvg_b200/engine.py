"""Host-side schedule of one p2pvg training step on the sm_100a kernels.

Restructures ``P2PModel.forward`` (reference models/p2p_model.py:185-271) into time-batched phases
(SURVEY.md §3.3) without changing its results:

  Phase E  every frame is encoded once, BatchNorm statistics grouped per frame (= per reference call);
  Phase R  posterior / prior / frame-predictor LSTMs: input-side GEMMs batched over time, the recurrent
           part scanned step by step; reparameterisation, KL and the alignment loss fused;
  Phase D  all S recon decodes + the CPC decode in one batch, BatchNorm grouped per call, the skip half of
           every ``torch.cat([d, skip])`` ConvTranspose computed once per distinct skip frame;
  backward D -> R -> E, Adam on (predictor, posterior, encoder, decoder), then the CPC chain through the
  *updated* decoder / predictor weights into the prior (the reference's two-phase update on its pinned
  PyTorch 1.0, "Mode A" of SURVEY.md §8c), Adam on the prior.

The engine only sequences kernels of a backend object (p2pvg_b200._lib.CudaKernels); all arithmetic on
device data happens inside those kernels.
"""
from __future__ import annotations

import math
import os
import time
from collections import OrderedDict

import numpy as np
import torch

ACT_NONE, ACT_LRELU, ACT_TANH = 0, 1, 2
BN_MOMENTUM = 0.1
# BatchNorm statistics come out of a GEMM epilogue only where the tile's MMA time hides the extra epilogue work: reduction
# length x tile width of the GEMM must reach this many MACs per output row (measured: low-K tiles are epilogue-bound and get
# slower, DESIGN.md)
BN_FUSE_MIN = 2048 * 128


def skip_schedule(seq_len, probs, skip_prob, n_past):
    """Executed timesteps and their (time_until_cp, delta_time) counters — integer / exact-rational logic
    of models/p2p_model.py:209-229, computed on the host in Python doubles exactly like the reference."""
    cp_ix = seq_len - 1
    prev_i, skip_count, out = 0, 0, []
    max_skip = seq_len * skip_prob
    for i in range(1, seq_len):
        if probs[i - 1] <= skip_prob and i >= n_past and skip_count < max_skip and i != 1 and i != cp_ix:
            skip_count += 1
            continue
        out.append((i, (cp_ix - i + 1) / cp_ix, (i - prev_i) / cp_ix))
        prev_i = i
    return out


class StepPlan:
    """Index tables of one step (which frame feeds which call), built on the host."""

    def __init__(self, T, probs, opt):
        sched = skip_schedule(T, probs, opt["skip_prob"], opt["n_past"])
        self.T, self.S = T, len(sched)
        S = self.S
        self.in_frame = [i - 1 for i, _, _ in sched]
        self.tgt_frame = [i for i, _, _ in sched]
        self.tuc = [t for _, t, _ in sched]
        self.dt = [d for _, _, d in sched]
        src, cur = [], None
        for i, _, _ in sched:  # models/p2p_model.py:235-238
            if opt["last_frame_skip"] or i <= opt["n_past"]:
                cur = i - 1
            if cur is None:
                raise ValueError("n_past must be >= 1 (the reference has no skip tensor otherwise)")
            src.append(cur)
        self.skip_src = src + [src[-1]]  # the CPC decode reuses the last skip
        self.nskip = max(self.skip_src) + 1
        self.has_cpc = S > 0 and sched[-1][0] == T - 1
        # encoder call order of the reference: x_cp, then (x[i-1], x[i]) per executed step
        self.enc_order = [T - 1] + [f for s in range(S) for f in (self.in_frame[s], self.tgt_frame[s])]
        ints = OrderedDict(
            in_idx=self.in_frame + [self.in_frame[-1]],
            tgt_idx=self.tgt_frame + [T - 1],          # last entry: CPC target x_cp
            glob_idx=[T - 1] * (S + 1),
            z_idx=list(range(S + 1)),
            skip_src=self.skip_src,
            enc_order=self.enc_order,
            dec_order=list(range(S + 1)),
            skip_dst=list(range(self.nskip)),
        )
        self.int_layout, off, flat = {}, 0, []
        for k, v in ints.items():
            self.int_layout[k] = (off, len(v))
            flat += v
            off += len(v)
        self.int_host = torch.tensor(flat, dtype=torch.int32)
        self.f_host = torch.tensor([self.tuc + [self.tuc[-1]], self.dt + [self.dt[-1]]], dtype=torch.float64).float()
        self.key = (T, S, self.nskip, self.has_cpc)


class ParamArena:
    """Flat fp32 storage of one module's parameters (+ grads + Adam moments) with named views, so the optimiser is one
    kernel per module.  The arenas of all modules are carved out of ONE allocation per kind (`pool`), laid out in the order
    the gradients become final, so the data-parallel exchange is one all-reduce per contiguous bucket."""

    def __init__(self, named_tensors, device, pool=None):
        self.names, self.shapes, self.offsets = [], {}, {}
        off = 0
        for k, v in named_tensors.items():
            self.names.append(k)
            self.shapes[k] = tuple(v.shape)
            self.offsets[k] = off
            off += (v.numel() + 3) // 4 * 4  # keep every view 16-byte aligned
        self.numel = off
        if pool is None:
            self.flat, self.grad, self.m, self.v = (torch.zeros(off, dtype=torch.float32, device=device) for _ in range(4))
            self.base = 0
        else:
            self.base = pool["used"]
            pool["used"] += (off + 63) // 64 * 64
            self.flat, self.grad, self.m, self.v = (pool[nm][self.base:self.base + off] for nm in ("flat", "grad", "m", "v"))
        self.step_t = torch.zeros(1, dtype=torch.int32, device=device)
        self.p, self.g = {}, {}
        for k, v in named_tensors.items():
            o, n = self.offsets[k], v.numel()
            self.p[k] = self.flat[o:o + n].view(self.shapes[k])
            self.g[k] = self.grad[o:o + n].view(self.shapes[k])
            self.p[k].copy_(v.detach().to(device=device, dtype=torch.float32))

    @staticmethod
    def padded(named_tensors):
        n = sum((v.numel() + 3) // 4 * 4 for v in named_tensors.values())
        return (n + 63) // 64 * 64

    def moment_views(self, k):
        o, n = self.offsets[k], int(np.prod(self.shapes[k])) if self.shapes[k] else 1
        return self.m[o:o + n].view(self.shapes[k]), self.v[o:o + n].view(self.shapes[k])


# arena order = order in which the gradients of Mode A become final: backward #1 finishes decoder, frame predictor and
# posterior first (one exchange bucket), then the encoder, then backward #2 the prior
ARENA_ORDER = ("decoder", "frame_predictor", "posterior", "encoder", "prior")


def is_param_key(key):
    return not (key.endswith("running_mean") or key.endswith("running_var") or key.endswith("num_batches_tracked"))


class TrainEngine:
    def __init__(self, state, cfg, opt, kernels, act_dtype=torch.float32, mode="A"):
        """state: module -> {state_dict key: tensor} (reference key names, SURVEY.md A.1)."""
        # bf16 mode: the fp32 LSTM GEMMs run on the tensor cores at TF32 precision; fp32 mode stays exact.  The policy is
        # a property of this engine's view of the backend and travels with every GEMM call.
        tc_lstm = (act_dtype == torch.bfloat16) and hasattr(kernels, "with_mode")
        self.K = kernels.with_mode(tc_lstm) if hasattr(kernels, "with_mode") else kernels
        self.dev = kernels.device
        self.cfg, self.opt = dict(cfg), dict(opt)
        self.adt = act_dtype
        self.mode = mode
        self.g, self.z, self.R = cfg["g_dim"], cfg["z_dim"], cfg["rnn_size"]
        self.backbone = cfg.get("backbone", "dcgan")
        if self.backbone in ("dcgan", "vgg"):
            self.nc, self.W0 = cfg["channels"], cfg["image_width"]
            if self.backbone == "vgg" and self.W0 not in (64, 128):
                self.W0 = cfg.get("vgg_width", 64)  # fixtures name the backbone in image_width
            self.chans = [64, 128, 256, 512] if self.W0 == 64 else [64, 128, 256, 512, 512]
            if self.W0 not in (64, 128):
                raise ValueError("dcgan backbones exist for 64 and 128 pixel frames")
            self.n = len(self.chans)
            self.frame_elems = self.nc * self.W0 * self.W0
        else:
            self.frame_elems = 51  # h36m pose: 17 joints x 3
        self.arena, self.buffers = {}, {}
        params = {m: OrderedDict((k, v) for k, v in state[m].items() if is_param_key(k)) for m in ARENA_ORDER}
        total = sum(ParamArena.padded(params[m]) for m in ARENA_ORDER)
        self.pool = dict(used=0, **{nm: torch.zeros(total, dtype=torch.float32, device=self.dev) for nm in ("flat", "grad", "m", "v")})
        for m in ARENA_ORDER:
            self.arena[m] = ParamArena(params[m], self.dev, pool=self.pool)
            self.buffers[m] = {k: v.detach().clone().to(self.dev) for k, v in state[m].items() if not is_param_key(k)}
        self._bufs = {}
        self._buf_gen = 0
        self._plans, self._uploaded = {}, None
        self._packed = {}
        self._graphs = {}
        self.dist = None  # (torch.distributed, group, world_size) when batch-sharded over several GPUs
        self.tc_lstm = tc_lstm
        # one persistent launch per LSTM layer and direction instead of two launches per timestep, for the hidden sizes the scan
        # kernels cover (R = 512: clusters of 16 CTAs, tensor-core mode only -- the exact-fp32 cooperative grid cannot keep a 4 MB
        # W_hh resident)
        self.fused_scan = hasattr(kernels, "lstm_scan_fwd") and self.R % 64 == 0 and (self.R <= 256 or (self.R == 512 and tc_lstm))
        # bf16 mode: 4x4/s2 (transposed) convolutions with >= 64 channels on both sides run as implicit GEMMs (4-D TMA
        # pixel-box gathers), without im2col / col2im buffers.  P2PVG_IMPLICIT=0 keeps the explicit lowering, the independent
        # second lowering that the bf16 tests compare against.
        self.implicit = (act_dtype == torch.bfloat16) and hasattr(kernels, "conv_gemm") and os.environ.get("P2PVG_IMPLICIT", "1") != "0"
        # 1/3-channel ends (K = 16 nc or N = 16 nc < 64): four pixel rows are multiplied as one row against a block-diagonal
        # copy of the weight, so that no TMA box is out of bounds (measured 3x faster than the partially-OOB boxes)
        self.bd = (act_dtype == torch.bfloat16) and hasattr(kernels, "blockdiag")
        # the skip-half addend of the implicit (transposed) convolutions is stored in the activation dtype: it is read once per
        # decode call by the main GEMM's epilogue (fp32 doubled that traffic and its L2 footprint)
        self.addend_dtype = act_dtype
        # 1- and 3-channel bf16 stacks: tap gather + sigmoid + MSE of the last decoder layer as one kernel (no raw-output tensor)
        self.fuse_last = hasattr(kernels, "convt_c1_loss") and act_dtype == torch.bfloat16
        # BatchNorm forward statistics come out of the producing implicit GEMM's epilogue (per-tile column sums) instead of a
        # separate pass over the stored tensor, where the tile shape allows it and it pays (stat_buf)
        self.fuse_stats = self.implicit
        # independent chains of small kernels (the prior LSTM, the LSTM weight gradients, backward #2) run on side streams
        # inside the captured graph.  bf16 mode only: the exact-fp32 mode scans on cooperative grids, which must not share the
        # GPU with a second grid-barrier kernel (bf16 with a hidden size the cluster scans do not cover, e.g. 192, also scans
        # on cooperative grids and still runs the prior and posterior scans side by side).
        self.concurrent = getattr(kernels, "name", "") == "cuda" and act_dtype == torch.bfloat16
        self.streams, self._dirty, self._serial = {}, set(), False
        # early read-back of the four scalars (P2PModel.forward): zero-copy store into page-locked host memory right after the
        # loss finalisation, polled by the host while the rest of the step is still running
        self.early_loss = getattr(kernels, "name", "") == "cuda" and hasattr(kernels, "publish_scalars") \
            and os.environ.get("P2PVG_EARLY_LOSS", "1") != "0"
        self._pub_seq = 0
        if self.early_loss:
            self._pub_host = torch.zeros(8, dtype=torch.float32).pin_memory()
            self._pub_np = self._pub_host.numpy()
            self._pub_seq_np = self._pub_np.view(np.int32)
            self._pub_seq_dev = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.last_plan = None
        self.phase_events = None

    # ------------------------------------------------------------------ side streams ("lanes")
    # lane 0 = the caller's stream.  lane 1: the prior LSTM while the posterior runs on lane 0 (independent recurrences until
    # z); lane 2: LSTM weight gradients (never on the critical path); lane 3: backward #2 (CPC chain + prior BPTT, independent
    # of the encoder backward).  Every lane has its own workspaces (K.lane).  All of it is captured into the one CUDA graph.
    LANE_PRIOR, LANE_WGRAD, LANE_BWD2 = 1, 2, 3

    def fork(self, lane=2):
        """Context manager: kernels enqueued inside run on side stream `lane`, after everything enqueued on the current
        stream so far.  Forks are only taken from lane 0 (no nesting) and never while phases are being timed."""
        import contextlib
        if not self.concurrent or self.phase_events is not None or self._serial or self.K.lane != 0:
            return contextlib.nullcontext()
        st = self.streams.get(lane)
        if st is None:
            st = self.streams[lane] = torch.cuda.Stream(device=self.dev)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))
        st.wait_event(ev)
        self._dirty.add(lane)
        eng = self

        @contextlib.contextmanager
        def ctx():
            eng.K.lane = lane
            try:
                with torch.cuda.stream(st):
                    yield
            finally:
                eng.K.lane = 0
        return ctx()

    def join(self, *lanes):
        """The current stream waits for everything enqueued on the given side lanes (default: all)."""
        for lane in (lanes or tuple(self._dirty)):
            if lane in self._dirty:
                ev = torch.cuda.Event()
                ev.record(self.streams[lane])
                torch.cuda.current_stream(self.dev).wait_event(ev)
                if self.K.lane == 0:   # a side lane that joins another one does not relieve lane 0 of its own join
                    self._dirty.discard(lane)

    def lbuf(self, name, numel, dtype=None):
        """Scratch buffer private to the lane that is enqueueing (concurrent lanes must not share scratch)."""
        return self.buf(f"{name}@{self.K.lane}" if self.K.lane else name, numel, dtype)

    # ------------------------------------------------------------------ memory
    def buf(self, name, numel, dtype=None):
        dtype = dtype or self.adt
        t = self._bufs.get(name)
        if t is None or t.numel() < numel or t.dtype != dtype:
            if t is not None:
                # a captured CUDA graph holds the raw address of every buffer it touched: once one of them is
                # re-allocated (a longer sequence, more executed steps) every graph captured so far is stale
                self._buf_gen += 1
            t = torch.zeros(int(numel), dtype=dtype, device=self.dev)
            self._bufs[name] = t
        return t

    def graph_generation(self):
        """Changes whenever a buffer a captured graph may have baked in was re-allocated (engine pool or the
        kernel backend's workspaces)."""
        return (self._buf_gen, getattr(self.K, "ws_gen", 0))

    def fbuf(self, name, numel):
        return self.buf(name, numel, torch.float32)

    # ------------------------------------------------------------------ weights
    def enc_names(self, l):
        if l < self.n:
            return f"c{l + 1}.main.0", f"c{l + 1}.main.1"
        return f"c{self.n + 1}.0", f"c{self.n + 1}.1"

    def dec_names(self, k):
        """k = -1: upc1;  k in [0, n-1]: the stride-2 stages (the last one has no BatchNorm)."""
        if k < 0:
            return "upc1.0", "upc1.1"
        if k < self.n - 1:
            return f"upc{k + 2}.main.0", f"upc{k + 2}.main.1"
        return f"upc{self.n + 1}.0", None

    def pack_weights(self, which=("encoder", "decoder")):
        """fp32 master weights -> GEMM-layout copies in the activation dtype.
        Conv   W[Cout,Cin,4,4]  -> Wp[Cout,(kh,kw,ci)];   ConvT  W[Cin,Cout,4,4] -> Wp[Cin,(kh,kw,co)]."""
        K = self.K
        if "encoder" in which:
            P = self.arena["encoder"].p
            for l in range(self.n + 1):
                w = P[self.enc_names(l)[0] + ".weight"]
                co, ci = w.shape[0], w.shape[1]
                wp = self.buf(f"wp_enc{l}", co * 16 * ci)
                K.transpose_batched(w, wp, co, ci, 16)   # [co][ci][tap] -> [co][tap][ci]
                self._packed[f"enc{l}"] = wp
                if self.bd and l == 0 and (16 * ci) % 64 != 0:
                    bd = self.buf("wbd_enc0", 4 * co * 64 * ci)
                    K.blockdiag(wp, bd, co, 16 * ci, 4)
                    b4 = self.fbuf("bias4_enc0", 4 * co)
                    K.permute4(P[self.enc_names(l)[0] + ".bias"], b4, (4, co, 1, 1), (0, 1, 0, 0))
                    self._packed["enc0.bd"], self._packed["enc0.bias4"] = bd, b4
        if "decoder" in which:
            P = self.arena["decoder"].p
            for k in range(-1, self.n):
                cn = self.dec_names(k)[0]
                w = P[cn + ".weight"]
                ci, co = w.shape[0], w.shape[1]
                wp = self.buf(f"wp_dec{k}", ci * 16 * co)
                K.transpose_batched(w, wp, ci, co, 16)   # [ci][co][tap] -> [ci][tap][co]
                self._packed[f"dec{k}"] = wp
                if self.bd and k == self.n - 1 and (16 * co) % 64 != 0:
                    cd = ci // 2
                    for half, off in (("D", 0), ("S", cd * 16 * co)):
                        bd = self.buf(f"wbd_dec_last{half}", 4 * cd * 64 * co)
                        K.blockdiag(wp[off:], bd, cd, 16 * co, 4)
                        self._packed[f"dec_last.bd{half}"] = bd
                if k == -1:  # bias of the 1x1 -> 4x4 ConvTranspose, repeated over the 16 taps
                    b16 = self.fbuf("bias16_upc1", 16 * co)
                    K.permute4(P[cn + ".bias"], b16, (16, co, 1, 1), (0, 1, 0, 0))
                    self._packed["dec-1.bias16"] = b16

    def pack_lstm_weights(self):
        """Tensor-core (TF32) mode only: K-major fp32 copies of the LSTM weights for the GEMMs whose natural
        operand layout is MN-major (data gradients), and a zero-padded embed weight so that the row pitch of
        the 258 / 140-wide inputs is TMA-compatible."""
        if not self.tc_lstm:
            return
        K = self.K
        for m in ("frame_predictor", "posterior", "prior"):
            P = self.arena[m].p
            R = self.R
            w = P["embed.weight"]
            in_dim = w.shape[1]
            in_p = (in_dim + 7) // 8 * 8
            # re-pitch [R,in_dim] -> [R,in_p]: columns >= in_dim pick up the first elements of the next row
            # (finite weights); they only ever multiply the zero padding columns of the input, so the product is exact
            wp = self.fbuf(f"{m}_embed_pad", R * in_p)
            K.permute4(w, wp, (R, in_p, 1, 1), (in_dim, 1, 0, 0))
            self._packed[f"{m}.embed_pad"] = wp
            for name, shape in [("embed.weight", (R, in_dim))] + [(f"lstm.{l}.weight_{k}", (4 * R, R)) for l in range(self.lstm_layers(m)) for k in ("ih", "hh")] + \
                    ([("output.0.weight", (self.g, R))] if m == "frame_predictor" else []):
                o, i = shape
                wt = self.fbuf(f"{m}_{name}_T", o * i)
                K.transpose_batched(P[name], wt, 1, o, i)   # [o][i] -> [i][o]
                self._packed[f"{m}.{name}.T"] = wt

    def lin_dinput(self, m, name, dY, out, rows, out_dim, in_dim, **kw):
        """out[rows,in_dim] (+)= dY[rows,out_dim] . W[out_dim,in_dim]"""
        if self.tc_lstm:
            self.K.gemm(dY, self._packed[f"{m}.{name}.T"], out, rows, in_dim, out_dim, **kw)
        else:
            self.K.gemm(dY, self.arena[m].p[name], out, rows, in_dim, out_dim, b_mn=True, **kw)

    def lin_wgrad(self, dY, X, gW, rows, out_dim, in_dim, ldx=None, reuse_dy=False):
        """gW[out_dim,in_dim] = dY[rows,out_dim]^T . X[rows,in_dim(+pad)]  (reduction over rows).  reuse_dy: the previous
        lin_wgrad call on this lane had the same dY (W_hh then W_ih of one LSTM layer): its bf16 copy is still in place."""
        K = self.K
        ldx = ldx or in_dim
        if self.tc_lstm and out_dim % 8 == 0 and ldx % 8 == 0:
            a = self.lbuf("wg_castA", rows * out_dim, torch.bfloat16)
            b = self.lbuf("wg_castB", rows * ldx, torch.bfloat16)
            if not reuse_dy:
                K.permute4(dY, a, (rows * out_dim, 1, 1, 1), (1, 0, 0, 0))
            K.permute4(X, b, (rows * ldx, 1, 1, 1), (1, 0, 0, 0))
            K.gemm(a, b, gW, out_dim, in_dim, rows, a_mn=True, b_mn=True, lda=out_dim, ldb=ldx)
        else:
            K.gemm(dY, X, gW, out_dim, in_dim, rows, a_mn=True, b_mn=True, lda=out_dim, ldb=ldx)

    # ------------------------------------------------------------------ plan upload
    def upload_plan(self, plan):
        ints = self.buf("plan_int", 16 * 1024, torch.int32)
        fl = self.fbuf("plan_f", 4096)
        n = plan.int_host.numel()
        ints[:n].copy_(plan.int_host, non_blocking=True)
        S1 = plan.S + 1
        fl[:2 * S1].copy_(plan.f_host.reshape(-1), non_blocking=True)
        self.ix = {k: ints[o:o + ln] for k, (o, ln) in plan.int_layout.items()}
        self.tuc, self.dt = fl[:S1], fl[S1:2 * S1]
        E = self.frame_elems
        coef = [1.0 / (self.B * E)] * plan.S + [self.opt["weight_cpc"] / (self.B * E)]
        cf = self.fbuf("plan_coef", 256)
        cf[:S1].copy_(torch.tensor(coef, dtype=torch.float64).float(), non_blocking=True)
        self.coef = cf[:S1]

    # ------------------------------------------------------------------ phases
    def step(self, x, probs=None, eps=None, return_device=False, use_graph=False):
        """x: [T,B,C,H,W] fp32 on the device.  probs: host numpy uniform draws (None -> np.random.uniform,
        like models/p2p_model.py:215).  eps: [S,2,B,z] N(0,1) (None -> torch.randn on the device)."""
        T, B = int(x.shape[0]), int(x.shape[1])
        opt = self.opt
        if probs is None:
            probs = np.random.uniform(0, 1, T - 1)
        # the index tables only depend on WHICH timesteps execute: plans are cached per pattern, and a pattern that is already
        # on the device (always the case with skip_prob = 0) is not uploaded again
        sched = skip_schedule(T, probs, opt["skip_prob"], opt["n_past"])
        pkey = (T, tuple(i for i, _, _ in sched), bool(opt["last_frame_skip"]), int(opt["n_past"]))
        plan = self._plans.get(pkey)
        if plan is None:
            if len(self._plans) > 4096:
                self._plans.clear()
            plan = self._plans[pkey] = StepPlan(T, probs, opt)
        self.last_plan = plan
        self.T, self.B, self.S = T, B, plan.S
        if eps is None:
            eps = torch.randn(plan.S, 2, B, self.z, device=self.dev, dtype=torch.float32)
        ukey = (pkey, B, float(opt["weight_cpc"]), self.graph_generation())
        if ukey != self._uploaded:
            self.upload_plan(plan)
            self._uploaded = ukey
        if self.early_loss:
            self._pub_seq = (self._pub_seq + 1) & 0x3FFFFFFF
            self._pub_seq_dev.fill_(self._pub_seq)
        if use_graph:
            out = self._step_graphed(x, eps, plan)
        else:
            self.eps = eps.contiguous()
            out = self._run(x, plan)
        return out if return_device else out.cpu().numpy()

    def read_losses(self, out):
        """The four scalars of the step just enqueued, as a host numpy array.  With the early read-back the call returns as soon
        as the forward half of the step has produced them (the backward passes / optimiser keep running; all later work is
        stream-ordered behind them); otherwise it is a blocking device-to-host copy of `out`."""
        if not self.early_loss:
            return out.cpu().numpy()
        seq, flag, t0, spins = self._pub_seq, self._pub_seq_np, time.perf_counter(), 0
        stream = torch.cuda.current_stream(self.dev)
        while flag[4] != seq:
            spins += 1
            if spins & 0x3FF == 0 and time.perf_counter() - t0 > 2e-3:
                # not there after 2 ms of spinning: make sure the stream is still alive (a failed kernel must raise, not hang)
                if stream.query():
                    if flag[4] == seq:
                        break
                    torch.cuda.synchronize(self.dev)   # surfaces a sticky CUDA error if there is one
                    if flag[4] != seq:
                        return out.cpu().numpy()        # the step ran without the publish kernel (foreign replay): plain read-back
                    break
                if time.perf_counter() - t0 > 300.0:
                    raise RuntimeError("p2pvg_b200: loss read-back timed out")
                time.sleep(0)
        return self._pub_np[:4].copy()

    def _step_graphed(self, x, eps, plan):
        """CUDA-graph replay of the whole step.  The first call with a new (T,B,S,...) signature runs eagerly
        (allocating every buffer), the second captures, later ones only replay; index tables, counters and
        inputs live in static device buffers that are refreshed before each replay."""
        # host scalars that the kernels receive by value are part of the signature: a replay would silently keep
        # the values seen at capture time (lr, loss weights, configured batch size, Adam beta1)
        opt = self.opt
        key = plan.key + (self.B, tuple(x.shape[2:]), float(opt["lr"]), float(opt["beta1"]), float(opt["beta"]),
                          float(opt["weight_align"]), float(opt["weight_cpc"]), int(opt["batch_size"]), self.mode,
                          self.dist[2] if self.dist is not None else 1)
        xs = self.fbuf("x_static", x.numel()).view(-1)[:x.numel()].view(x.shape)
        es = self.fbuf("eps_static", eps.numel()).view(-1)[:eps.numel()].view(eps.shape)
        xs.copy_(x, non_blocking=True)
        # the caller's batch tensor is not read again by this step: an input pipeline that attached a callback
        # (p2pvg_b200.data.DevicePrefetcher) may refill its slot from here on instead of after the whole step
        consumed = getattr(x, "_p2pvg_on_consumed", None)
        if consumed is not None:
            ev = torch.cuda.Event()
            ev.record()
            consumed(ev)
        es.copy_(eps, non_blocking=True)
        self.eps = es
        st = self._graphs.get(key)
        if st is not None and st != "warm" and st[2] != self.graph_generation():
            st = None   # some buffer moved since this graph was captured
        if st is None:
            # eager run: allocates / grows every buffer this signature needs
            gen0 = self.graph_generation()
            out = self._run(xs, plan)
            if self.graph_generation() != gen0:
                self._graphs.clear()   # older graphs point into freed buffers
            self._graphs[key] = "warm"
            return out
        if st == "warm":
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            n0 = self.K.launches
            gen0 = self.graph_generation()
            with torch.cuda.graph(g):
                self._run(xs, plan)
            if self.graph_generation() != gen0:
                raise RuntimeError("a buffer was re-allocated during CUDA-graph capture (the warm-up run must size every buffer)")
            self._graphs[key] = st = (g, self.K.launches - n0, gen0)
        st[0].replay()
        self.K.launches += st[1]
        return self._bufs["loss_out"][:4]

    def _mark(self, name):
        """Phase timing for profiling (eager mode only): tools/profile_step.py --phases."""
        if self.phase_events is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.phase_events.append((name, e))

    def _run(self, x, plan):
        self._run_inner(x, plan)
        self._mark("end")
        return self._bufs["loss_out"][:4]

    def _run_inner(self, x, plan):
        self._mark("start")
        for name, fn, lane in self.phases(x, plan):
            if lane:
                with self.fork(lane):
                    fn()
            else:
                fn()
            self._mark(name)
        self.join()

    def phases(self, x, plan):
        """The step as an ordered list of (name, thunk, lane).  _run executes them in order -- a phase with lane != 0 is
        enqueued on that side stream and runs concurrently with the phases after it until they join; time_phases()
        captures each one alone into its own CUDA graph (bench.py: per-phase times, LSTM-phase roofline).

        Mode A (the reference's two-phase update, SURVEY.md §0.5): backward #2 (CPC chain + prior BPTT) reads the UPDATED
        decoder / frame-predictor weights and nothing of the encoder's, so those three modules are stepped as soon as
        their gradients exist and backward #2 runs beside the encoder backward."""
        def adam_of(mods, repack=False):
            def f():
                self.join()
                self.adam(mods)
                if repack:   # backward #2 runs through the UPDATED decoder / predictor weights
                    self.pack_weights(("decoder",))
                    self.pack_lstm_weights()
            return f

        ph = [("pack", lambda: (self.pack_weights(), self.pack_lstm_weights()), 0),
              ("encode_fwd", lambda: self.encode(x, plan), 0),
              ("lstm_fwd", lambda: self.recurrent_fwd(plan), 0),
              ("decode_fwd", lambda: (self.decode(plan), self.losses_fwd(plan)), 0),
              ("decoder_bwd", lambda: self.backward_decoder(plan), 0),
              ("lstm_bwd", lambda: self.backward_recurrent(plan), 0)]
        if self.mode == "A" and self.dist is not None and self.concurrent and not self._serial:
            # data parallel: the exchange of the first bucket (decoder + predictor + posterior), their Adam step, the re-pack
            # and backward #2 form ONE chain on the side lane -- the all-reduce overlaps the encoder backward
            a3 = adam_of(("frame_predictor", "posterior", "decoder"), repack=True)
            ph += [("allreduce+adam3+repack+prior_bwd", lambda: (a3(), self.backward_prior(plan)), self.LANE_BWD2),
                   ("encoder_bwd", lambda: self.encoder_backward(plan), 0),
                   ("adam_enc+prior", adam_of(("encoder", "prior")), 0)]
        elif self.mode == "A":
            ph += [("adam3+repack", adam_of(("frame_predictor", "posterior", "decoder"), repack=True), 0),
                   ("prior_bwd", lambda: self.backward_prior(plan), self.LANE_BWD2),
                   ("encoder_bwd", lambda: self.encoder_backward(plan), 0),
                   ("adam_enc+prior", adam_of(("encoder", "prior")), 0)]
        else:
            ph += [("prior_bwd", lambda: self.backward_prior(plan), self.LANE_BWD2),
                   ("encoder_bwd", lambda: self.encoder_backward(plan), 0),
                   ("adam5", adam_of(("frame_predictor", "posterior", "encoder", "decoder", "prior")), 0)]
        return ph

    def time_phases(self, x, reps=5):
        """Device time (ms) of every phase of a step on batch `x`, each phase captured ALONE (no concurrent lanes) into its
        own CUDA graph and replayed `reps` times between CUDA events.  Leaves the optimiser / BatchNorm state advanced:
        measurement only.  No collectives (single-rank measurement)."""
        plan = self.last_plan
        saved, self.dist = self.dist, None
        out = {}
        try:
            self._run(x, plan)   # eager: every buffer exists, activations of this batch are in place
            torch.cuda.synchronize(self.dev)
            self._serial = True
            for name, fn, _ in self.phases(x, plan):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    fn()
                g.replay()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    g.replay()
                e1.record()
                torch.cuda.synchronize(self.dev)
                out[name] = e0.elapsed_time(e1) / reps
                del g
        finally:
            self._serial = False
            self.dist = saved
            self._graphs.clear()
        return out

    def frames_nhwc(self, x):
        """Frames NCHW fp32 -> NHWC: self.x_nhwc (fp32, the MSE target) and the returned activation-dtype copy (input of the
        first convolution); multi-channel inputs are converted by one kernel that reads the frames once."""
        K, T, B, nc, W0 = self.K, self.T, self.B, self.nc, self.W0
        N = T * B
        hw = W0 * W0
        xs = x.contiguous()
        if nc == 1 and xs.dtype == torch.float32:
            self.x_nhwc = xs.view(-1)  # one channel: NCHW == NHWC, the MSE target is the input itself
            dual = False
        else:
            self.x_nhwc = self.fbuf("x_nhwc", N * hw * nc)
            dual = xs.dtype == torch.float32 and nc in (2, 3, 4) and hw % 4 == 0 and xs.is_cuda
            if not dual:
                K.permute4(xs, self.x_nhwc, (N, hw, nc, 1), (nc * hw, 1, hw, 0))
        if self.adt == torch.float32:
            a = self.x_nhwc
            if dual:
                K.nchw_to_nhwc_dual(xs, self.x_nhwc, None, N, hw, nc)
        else:
            a = self.buf("x_act", N * hw * nc)
            if dual:  # one read of the frames, both copies
                K.nchw_to_nhwc_dual(xs, self.x_nhwc, a, N, hw, nc)
            else:
                K.permute4(xs, a, (N, hw, nc, 1), (nc * hw, 1, hw, 0))
        return a

    # -- Phase E ----------------------------------------------------------------------------
    def encode(self, x, plan):
        K, T, B, n, nc, W0 = self.K, self.T, self.B, self.n, self.nc, self.W0
        P = self.arena["encoder"].p
        N = T * B
        a = self.frames_nhwc(x)
        self.enc_in = a
        self.enc = []
        H = W0
        for l in range(n):
            cin = nc if l == 0 else self.chans[l - 1]
            cout = self.chans[l]
            Ho = H // 2
            M = N * Ho * Ho
            raw = self.buf(f"enc_raw{l}", M * cout)
            y = self.buf(f"enc_y{l}", M * cout)
            cn, bn = self.enc_names(l)
            imp = self.implicit and cin % 64 == 0 and cout % 64 == 0
            col = None
            sp = None
            if imp:
                sp = self.stat_buf(f"enc{l}", M, 1, cout, B * Ho * Ho, kred=16 * cin)
                K.conv_gemm(0, a, self._packed[f"enc{l}"], raw, N, Ho, Ho, cin, cout, bias=P[cn + ".bias"],
                            stat_partial=sp["buf"] if sp else None)
            else:
                col = self.buf(f"enc_col{l}", M * 16 * cin)
                K.im2col(a, col, N, H, H, cin)
                if l == 0 and "enc0.bd" in self._packed:
                    K.gemm(col, self._packed["enc0.bd"], raw, M // 4, 4 * cout, 64 * cin, bias=self._packed["enc0.bias4"])
                else:
                    K.gemm(col, self._packed[f"enc{l}"], raw, M, cout, 16 * cin, bias=P[cn + ".bias"])
            st = self.bn_forward("enc", l, raw, y, T, B * Ho * Ho, cout, P[bn + ".weight"], P[bn + ".bias"], ACT_LRELU, tiles=sp)
            self.enc.append(dict(col=col, raw=raw, y=y, st=st, cin=cin, cout=cout, Hin=H, Hout=Ho, M=M, imp=imp, inp=a))
            a, H = y, Ho
        # final 4x4 valid conv == GEMM over the flattened 4x4xC map
        ctop = self.chans[-1]
        cn, bn = self.enc_names(n)
        raw = self.buf("enc_rawf", N * self.g)
        y = self.buf("enc_yf", N * self.g)
        K.gemm(a, self._packed[f"enc{n}"], raw, N, self.g, 16 * ctop, bias=P[cn + ".bias"])
        st = self.bn_forward("enc", n, raw, y, T, B, self.g, P[bn + ".weight"], P[bn + ".bias"], ACT_TANH)
        self.enc_final = dict(inp=a, raw=raw, y=y, st=st)
        if self.adt == torch.float32:
            self.Hlat = y
        else:
            self.Hlat = self.fbuf("Hlat", N * self.g)
            K.permute4(y, self.Hlat, (N * self.g, 1, 1, 1), (1, 0, 0, 0))
        # running statistics: one EMA update per reference call, in call order
        ncalls = len(plan.enc_order)
        Bf = self.buffers["encoder"]
        for l in range(n + 1):
            st = self.enc[l]["st"] if l < n else self.enc_final["st"]
            bn = self.enc_names(l)[1]
            K.bn_ema(Bf[bn + ".running_mean"], Bf[bn + ".running_var"], st["mean"], st["varu"], self.ix["enc_order"], ncalls,
                     st["C"], BN_MOMENTUM)
            Bf[bn + ".num_batches_tracked"] += ncalls

    def stat_buf(self, tag, rows, phases, C, rows_per_group, kred=1 << 30):
        """Workspace for the per-tile BatchNorm statistics of a GEMM epilogue, or None when the fusion does not apply
        (a 128-row tile must not straddle two BatchNorm groups) or does not pay (kred = reduction length of one tile: short
        reductions leave the epilogue no MMA time to hide behind).  rows: GEMM rows (per phase)."""
        bn_tile = 256 if C % 256 == 0 else 128 if C > 64 else 64
        if not self.fuse_stats or rows_per_group % 128 != 0 or rows % 128 != 0 or kred * bn_tile < BN_FUSE_MIN:
            return None
        buf = self.fbuf(f"bnpart_{tag}", (rows // 128) * phases * C * 2)
        return dict(buf=buf, parts_per_group=(rows_per_group // 128) * phases, ldp=C, fold=1)

    def bn_forward(self, tag, idx, raw, y, G, R, C, gamma, beta, act, tiles=None):
        """Batch statistics per group + normalise + activation.  tiles: statistics partials already produced by the
        epilogue of the GEMM that wrote `raw` (stat_buf) -- then only the tiny finalize kernel runs instead of a pass over raw."""
        K = self.K
        names = ("mean", "invstd", "varu", "scale", "shift", "sdz", "sdzx")
        st = {nm: self.fbuf(f"{tag}_bn{idx}_{nm}", G * C) for nm in names}
        st.update(G=G, R=R, C=C, act=act, gamma=gamma)
        if tiles is not None:
            K.bn_fwd_finalize_tiles(tiles["buf"], tiles["parts_per_group"], tiles["ldp"], tiles["fold"], G, R, C, gamma, beta,
                                    st["mean"], st["invstd"], st["varu"], st["scale"], st["shift"])
        else:
            K.bn_fwd_stats(raw, G, R, C, gamma, beta, st["mean"], st["invstd"], st["varu"], st["scale"], st["shift"])
        K.bn_act(raw, y, st["scale"], st["shift"], G, R, C, act)
        return st

    # -- Phase R ----------------------------------------------------------------------------
    def in_pitch(self, in_dim):
        """Row pitch of the LSTM input matrices: padded to a multiple of 8 floats in tensor-core mode."""
        return (in_dim + 7) // 8 * 8 if self.tc_lstm else in_dim

    def lstm_layers(self, m):
        return len({k.split(".")[1] for k in self.arena[m].p if k.startswith("lstm.")})

    def lstm_forward(self, m, X, steps, in_dim):
        """embed -> n x LSTMCell over `steps` timesteps.  X: [steps*B, in_dim].  Returns the top layer's
        hidden states [steps*B, R] (a view of the saved state)."""
        K, B, R = self.K, self.B, self.R
        P = self.arena[m].p
        L = self.lstm_layers(m)
        rows = steps * B
        E = self.fbuf(f"{m}_E", rows * R)
        ldx = self.in_pitch(in_dim)
        if self.tc_lstm:
            K.gemm(X, self._packed[f"{m}.embed_pad"], E, rows, R, ldx, bias=P["embed.bias"])
        else:
            K.gemm(X, P["embed.weight"], E, rows, R, in_dim, bias=P["embed.bias"])
        sv = dict(X=X, E=E, steps=steps, in_dim=in_dim, ldx=ldx, layers=[])
        inp = E
        for l in range(L):
            Pre = self.fbuf(f"{m}_pre{l}", rows * 4 * R)
            gates = self.fbuf(f"{m}_gates{l}", rows * 4 * R)
            hs = self.fbuf(f"{m}_h{l}", (steps + 1) * B * R)
            cs = self.fbuf(f"{m}_c{l}", (steps + 1) * B * R)
            hs[:B * R].zero_()
            cs[:B * R].zero_()
            K.gemm(inp, P[f"lstm.{l}.weight_ih"], Pre, rows, 4 * R, R, bias=P[f"lstm.{l}.bias_ih"])
            whh, bhh = P[f"lstm.{l}.weight_hh"], P[f"lstm.{l}.bias_hh"]
            if self.fused_scan:
                ctr = self.lbuf("scan_counter", 4, torch.int32)
                ctr.zero_()
                K.lstm_scan_fwd(Pre, whh, bhh, gates, hs, cs, steps, B, R, ctr, tf32=self.tc_lstm)
            for s in range(0 if not self.fused_scan else steps, steps):
                gs = gates[s * B * 4 * R:(s + 1) * B * 4 * R]
                K.gemm(hs[s * B * R:(s + 1) * B * R], whh, gs, B, 4 * R, R, bias=bhh, addend=Pre[s * B * 4 * R:(s + 1) * B * 4 * R])
                K.lstm_pointwise_fwd(gs, cs[s * B * R:(s + 1) * B * R], cs[(s + 1) * B * R:(s + 2) * B * R],
                                     hs[(s + 1) * B * R:(s + 2) * B * R], B, R)
            sv["layers"].append(dict(gates=gates, hs=hs, cs=cs, inp=inp))
            inp = hs[B * R:(steps + 1) * B * R]
        sv["top"] = inp
        return sv

    def recurrent_fwd(self, plan):
        K, B, S, g, z, R = self.K, self.B, self.S, self.g, self.z, self.R
        H = self.Hlat
        ix = self.ix
        win = 2 * g + 2
        lw = self.in_pitch(win)
        Xpost = self.fbuf("Xpost", S * B * lw)
        Xprior = self.fbuf("Xprior", S * B * lw)
        K.build_concat(Xpost, H, ix["tgt_idx"], g, H, ix["glob_idx"], g, self.tuc, self.dt, S, B, ld=lw)
        K.build_concat(Xprior, H, ix["in_idx"], g, H, ix["glob_idx"], g, self.tuc, self.dt, S, B, ld=lw)
        self.sv = {}
        heads = {}

        def gaussian(m, X):
            sv = self.lstm_forward(m, X, S, win)
            P = self.arena[m].p
            mu = self.fbuf(f"{m}_mu", S * B * z)
            lv = self.fbuf(f"{m}_lv", S * B * z)
            K.gemm(sv["top"], P["mu_net.weight"], mu, S * B, z, R, bias=P["mu_net.bias"])
            K.gemm(sv["top"], P["logvar_net.weight"], lv, S * B, z, R, bias=P["logvar_net.bias"])
            heads[m] = (mu, lv)
            self.sv[m] = sv

        # posterior and prior are independent recurrences until z (models/p2p_model.py:244-245): two lanes
        with self.fork(self.LANE_PRIOR):
            gaussian("prior", Xprior)
        gaussian("posterior", Xpost)
        self.join(self.LANE_PRIOR)
        self.mu, self.lv = heads["posterior"]
        self.mu_p, self.lv_p = heads["prior"]
        n = S * B * z
        self.eps_post = self.fbuf("eps_post", n)
        self.eps_prior = self.fbuf("eps_prior", n)
        K.permute4(self.eps, self.eps_post, (S, B * z, 1, 1), (2 * B * z, 1, 0, 0))
        K.permute4(self.eps[:, 1], self.eps_prior, (S, B * z, 1, 1), (2 * B * z, 1, 0, 0))
        self.Zall = self.fbuf("Zall", (S + 1) * B * z)  # rows 0..S-1 posterior z, row S = prior z of the last step
        self.Zp = self.fbuf("Zp", n)
        self.kl_sum = self.fbuf("kl_sum", 4)
        K.reparam_kl_fwd(self.mu, self.lv, self.mu_p, self.lv_p, self.eps_post, self.eps_prior, self.Zall, self.Zp, n, self.kl_sum)
        K.permute4(self.Zp[(S - 1) * B * z:], self.Zall[S * B * z:], (B * z, 1, 1, 1), (1, 0, 0, 0))
        # frame predictor over S recon steps + the CPC step (models/p2p_model.py:247,252)
        wp = g + z + 2
        Xpred = self.fbuf("Xpred", (S + 1) * B * self.in_pitch(wp))
        K.build_concat(Xpred, H, ix["in_idx"], g, self.Zall, ix["z_idx"], z, self.tuc, self.dt, S + 1, B, ld=self.in_pitch(wp))
        sv = self.lstm_forward("frame_predictor", Xpred, S + 1, wp)
        self.sv["frame_predictor"] = sv
        P = self.arena["frame_predictor"].p
        self.h_pred = self.fbuf("h_pred", (S + 1) * B * g)
        K.gemm(sv["top"], P["output.0.weight"], self.h_pred, (S + 1) * B, g, R, bias=P["output.0.bias"])
        K.act_fwd(self.h_pred, (S + 1) * B * g, ACT_TANH)

    # -- Phase D ----------------------------------------------------------------------------
    def decode(self, plan):
        K, B, S, n, g = self.K, self.B, self.S, self.n, self.g
        G = S + 1
        P = self.arena["decoder"].p
        N = G * B
        if self.adt == torch.float32:
            hp = self.h_pred
        else:
            hp = self.buf("hp_act", N * g)
            K.permute4(self.h_pred, hp, (N * g, 1, 1, 1), (1, 0, 0, 0))
        ctop = self.chans[-1]
        cn, bn = self.dec_names(-1)
        raw = self.buf("dec_raw_1", N * 16 * ctop)
        d = self.buf("dec_d_1", N * 16 * ctop)
        K.gemm(hp, self._packed["dec-1"], raw, N, 16 * ctop, g, b_mn=True, bias=self._packed["dec-1.bias16"])
        st = self.bn_forward("dec", -1, raw, d, G, B * 16, ctop, P[bn + ".weight"], P[bn + ".bias"], ACT_LRELU)
        self.dec_first = dict(inp=hp, raw=raw, d=d, st=st)
        self.dec = []
        Hi = 4
        nskip = plan.nskip
        for k in range(n):
            cd = self.chans[n - 1 - k]
            cout = self.chans[n - 2 - k] if k < n - 1 else self.nc
            skip = self.enc[n - 1 - k]["y"]  # frames are a prefix -> the first nskip frames
            Md, Ms = N * Hi * Hi, nskip * B * Hi * Hi
            wp = self._packed[f"dec{k}"]
            wD, wS = wp[:cd * 16 * cout], wp[cd * 16 * cout:]
            cn, bn = self.dec_names(k)
            Mo = N * 4 * Hi * Hi
            raw = self.buf(f"dec_raw{k}", Mo * cout)
            imp = self.implicit and cd % 64 == 0 and cout % 64 == 0
            sp = rec_fused = None
            if imp:
                # skip half once per distinct source frame (fp32, bias folded in), added in the epilogue of the main GEMM
                addS = self.buf(f"dec_addS{k}", nskip * B * 4 * Hi * Hi * cout, self.addend_dtype)
                K.conv_gemm(2, skip, wS, addS, nskip * B, Hi, Hi, cd, cout, bias=P[cn + ".bias"])
                sp = self.stat_buf(f"dec{k}", Md, 4, cout, B * Hi * Hi, kred=4 * cd) if k < n - 1 else None
                K.conv_gemm(2, d, wD, raw, N, Hi, Hi, cd, cout, addend=addS, grp_src=self.ix["skip_src"], imgs_per_group=B,
                            stat_partial=sp["buf"] if sp else None)
            else:
                colD = self.buf("dec_colD", Md * 16 * cout)
                colS = self.buf("dec_colS", Ms * 16 * cout)
                if k == n - 1 and "dec_last.bdD" in self._packed:
                    K.gemm(d, self._packed["dec_last.bdD"], colD, Md // 4, 64 * cout, 4 * cd, b_mn=True)
                    K.gemm(skip, self._packed["dec_last.bdS"], colS, Ms // 4, 64 * cout, 4 * cd, b_mn=True)
                else:
                    K.gemm(d, wD, colD, Md, 16 * cout, cd, b_mn=True)
                    K.gemm(skip, wS, colS, Ms, 16 * cout, cd, b_mn=True)
                if k == n - 1 and cout in (1, 3) and self.fuse_last:
                    # last layer of a 1- / 3-channel stack: the tap gather, sigmoid and loss run as ONE kernel in losses_fwd
                    rec_fused = (colD, colS, Hi, P[cn + ".bias"])
                else:
                    K.col2im(colD, raw, N, Hi, Hi, cout, bias=P[cn + ".bias"], col2=colS, grp_src=self.ix["skip_src"], imgs_per_group=B)
            rec = dict(inp=d, skip=skip, raw=raw, cd=cd, cout=cout, Hi=Hi, Md=Md, Ms=Ms, imp=imp, fused_loss=rec_fused)
            if k < n - 1:
                dn = self.buf(f"dec_d{k}", Mo * cout)
                rec["st"] = self.bn_forward("dec", k, raw, dn, G, B * 4 * Hi * Hi, cout, P[bn + ".weight"], P[bn + ".bias"], ACT_LRELU, tiles=sp)
                rec["d"] = dn
                d = dn
            self.dec.append(rec)
            Hi *= 2
        Bf = self.buffers["decoder"]
        for k in range(-1, n - 1):
            st = self.dec_first["st"] if k < 0 else self.dec[k]["st"]
            bn = self.dec_names(k)[1]
            K.bn_ema(Bf[bn + ".running_mean"], Bf[bn + ".running_var"], st["mean"], st["varu"], self.ix["dec_order"], G, st["C"], BN_MOMENTUM)
            Bf[bn + ".num_batches_tracked"] += G

    def losses_fwd(self, plan):
        K, B, S = self.K, self.B, self.S
        G = S + 1
        E = B * self.nc * self.W0 * self.W0
        raw = self.dec[-1]["raw"]
        self.d_rawout = self.buf("dec_d_rawout", G * E)
        self.mse_partial = self.fbuf("mse_partial", G * K.mse_chunks())
        fl = self.dec[-1].get("fused_loss")
        if fl is not None:
            colD, colS, Hi, bias = fl
            K.convt_c1_loss(colD, colS, self.ix["skip_src"], bias, self.x_nhwc, self.ix["tgt_idx"], self.coef, G, B, Hi, Hi,
                            self.d_rawout, self.mse_partial, C=self.nc)
        else:
            K.sigmoid_mse(raw, self.x_nhwc, self.ix["tgt_idx"], self.coef, G, E, None, self.d_rawout, self.mse_partial)
        self.align_partial = self.fbuf("align_partial", max(S, 1))
        self.d_hpred = self.fbuf("d_hpred", G * B * self.g)
        self.dH = self.fbuf("dH", self.T * B * self.g)

    # -- backward ---------------------------------------------------------------------------
    def decoder_backward(self, g0, g1, want_wgrad, want_skip):
        """Backward of the decoder calls [g0, g1).  Seeds: d_rawout.  Produces d_hpred[g0:g1] (fp32) and,
        if requested, weight gradients (into the decoder grad arena) and the skip gradients."""
        K, B, n, g = self.K, self.B, self.n, self.g
        Gn = g1 - g0
        N = Gn * B
        A = self.arena["decoder"]
        nskip = self.last_plan.nskip
        E = self.nc * self.W0 * self.W0
        dy = self.d_rawout[g0 * B * E:g1 * B * E]
        for k in range(n - 1, -1, -1):
            rec = self.dec[k]
            cd, cout, Hi = rec["cd"], rec["cout"], rec["Hi"]
            Md, Ms = N * Hi * Hi, nskip * B * Hi * Hi
            cn, bn = self.dec_names(k)
            Ho = 2 * Hi
            rows_o = N * Ho * Ho
            if k < n - 1:  # BatchNorm + LeakyReLU backward of this stage's output
                st = rec["st"]
                sl = slice(g0 * B * Ho * Ho * cout, g1 * B * Ho * Ho * cout)
                c0, c1 = g0 * st["C"], g1 * st["C"]
                self.bn_backward(dy, rec["raw"][sl], rec["d"][sl], st, c0, c1, Gn, B * Ho * Ho, cout, ACT_LRELU)
                if want_wgrad:
                    K.bn_param_grad(st["sdz"][c0:c1], st["sdzx"][c0:c1], Gn, cout, A.g[bn + ".weight"], A.g[bn + ".bias"])
                    A.g[cn + ".bias"].zero_()  # bias feeding a training-mode BatchNorm: gradient is exactly zero
            elif want_wgrad:
                K.colsum(dy, rows_o, cout, cout, A.g[cn + ".bias"])
            wp = self._packed[f"dec{k}"]
            wD, wS = wp[:cd * 16 * cout], wp[cd * 16 * cout:]
            x_in = rec["inp"][g0 * B * Hi * Hi * cd:g1 * B * Hi * Hi * cd]
            dd = self.buf(f"dec_gd{k}", Md * cd)
            if want_wgrad:
                gw = self.fbuf(f"gwp_dec{k}", 2 * cd * 16 * cout)
            if rec["imp"]:
                # data gradient = stride-2 conv of dy; weight gradients gather dy by filter tap; the skip half works
                # on dy summed over the calls that share a skip frame (conv is linear) -- no col buffers at all
                if want_wgrad:
                    K.conv_gemm(1, x_in, dy, gw[:cd * 16 * cout], N, Hi, Hi, 0, cout, Cm=cd)
                if want_skip:
                    dyS = self.buf(f"scratch_dyS{k}", nskip * B * Ho * Ho * cout)
                    K.group_sum(dy, dyS, self.ix["skip_src"][g0:g1], Gn, nskip, B * Ho * Ho * cout)
                    dsk = self.buf(f"dskip{k}", Ms * cd)
                    K.conv_gemm(0, dyS, wS, dsk, nskip * B, Hi, Hi, cout, cd)
                    rec["dskip"] = dsk
                    if want_wgrad:
                        K.conv_gemm(1, rec["skip"], dyS, gw[cd * 16 * cout:], nskip * B, Hi, Hi, 0, cout, Cm=cd)
                if want_wgrad:
                    K.transpose_batched(gw, A.g[cn + ".weight"], 2 * cd, 16, cout)   # [2cd][tap][co] -> [2cd][co][tap]
                K.conv_gemm(0, dy, wD, dd, N, Hi, Hi, cout, cd)
            else:
                dcol = self.buf("scratch_dcol", Md * 16 * cout)
                K.im2col(dy, dcol, N, Ho, Ho, cout)
                bdl = k == n - 1 and "dec_last.bdD" in self._packed
                if bdl:
                    K.gemm(dcol, self._packed["dec_last.bdD"], dd, Md // 4, 4 * cd, 64 * cout)
                else:
                    K.gemm(dcol, wD, dd, Md, cd, 16 * cout)
                if want_wgrad:
                    K.gemm(x_in, dcol, gw[:cd * 16 * cout], cd, 16 * cout, Md, a_mn=True, b_mn=True, lda=cd, ldb=16 * cout)
                if want_skip:
                    dcolS = self.buf("scratch_dcolS", Ms * 16 * cout)
                    K.group_sum(dcol, dcolS, self.ix["skip_src"][g0:g1], Gn, nskip, B * Hi * Hi * 16 * cout)
                    dsk = self.buf(f"dskip{k}", Ms * cd)
                    if bdl:
                        K.gemm(dcolS, self._packed["dec_last.bdS"], dsk, Ms // 4, 4 * cd, 64 * cout)
                    else:
                        K.gemm(dcolS, wS, dsk, Ms, cd, 16 * cout)
                    rec["dskip"] = dsk
                    if want_wgrad:
                        K.gemm(rec["skip"], dcolS, gw[cd * 16 * cout:], cd, 16 * cout, Ms, a_mn=True, b_mn=True, lda=cd, ldb=16 * cout)
                if want_wgrad:
                    K.transpose_batched(gw, A.g[cn + ".weight"], 2 * cd, 16, cout)   # [2cd][tap][co] -> [2cd][co][tap]
            dy = dd
        # upc1: BatchNorm + LeakyReLU, then the g -> 4x4xCtop GEMM
        ctop = self.chans[-1]
        cn, bn = self.dec_names(-1)
        st = self.dec_first["st"]
        sl = slice(g0 * B * 16 * ctop, g1 * B * 16 * ctop)
        c0, c1 = g0 * ctop, g1 * ctop
        self.bn_backward(dy, self.dec_first["raw"][sl], self.dec_first["d"][sl], st, c0, c1, Gn, B * 16, ctop, ACT_LRELU)
        hp = self.dec_first["inp"][g0 * B * g:g1 * B * g]
        if want_wgrad:
            K.bn_param_grad(st["sdz"][c0:c1], st["sdzx"][c0:c1], Gn, ctop, A.g[bn + ".weight"], A.g[bn + ".bias"])
            A.g[cn + ".bias"].zero_()
            gw = self.fbuf("gwp_dec-1", g * 16 * ctop)
            K.gemm(hp, dy, gw, g, 16 * ctop, N, a_mn=True, b_mn=True, lda=g, ldb=16 * ctop)
            K.transpose_batched(gw, A.g[cn + ".weight"], g, 16, ctop)
        dhp = self.d_hpred[g0 * B * g:g1 * B * g]
        if self.adt == torch.float32:
            K.gemm(dy, self._packed["dec-1"], dhp, N, g, 16 * ctop)
        else:
            tmp = self.buf("dhp_act", N * g)
            K.gemm(dy, self._packed["dec-1"], tmp, N, g, 16 * ctop)
            K.permute4(tmp, dhp, (N * g, 1, 1, 1), (1, 0, 0, 0))

    def bn_backward(self, dy, raw, y, st, c0, c1, G, R, C, act):
        """BatchNorm + activation backward in place (dy -> d raw).  On the CUDA backend the LeakyReLU derivative is
        recomputed from sign(raw*scale+shift), so the activation tensor is not read again."""
        K = self.K
        if getattr(K, "name", "") == "cuda" and act == ACT_LRELU:
            K.bn_bwd(dy, raw, None, st["mean"][c0:c1], st["invstd"][c0:c1], st["gamma"], G, R, C, act, dy, st["sdz"][c0:c1],
                     st["sdzx"][c0:c1], scale=st["scale"][c0:c1], shift=st["shift"][c0:c1])
        else:
            K.bn_bwd(dy, raw, y, st["mean"][c0:c1], st["invstd"][c0:c1], st["gamma"], G, R, C, act, dy, st["sdz"][c0:c1],
                     st["sdzx"][c0:c1])

    def lstm_backward(self, m, dtop, steps, want_wgrad, want_dx, dx_out=None):
        """Reverse-time scan.  dtop: [steps*B, R] gradient w.r.t. the top layer's hidden outputs (it is
        overwritten).  Returns dX [steps*B, in_dim] if want_dx."""
        K, B, R = self.K, self.B, self.R
        sv = self.sv[m]
        A = self.arena[m]
        P = A.p
        L = len(sv["layers"])
        rows = steps * B
        dH = dtop
        for l in range(L - 1, -1, -1):
            lay = sv["layers"][l]
            dG = self.fbuf(f"{m}_dG{l}", rows * 4 * R)
            dcA = self.fbuf(f"{m}_dcA", B * R)
            dcB = self.fbuf(f"{m}_dcB", B * R)
            dht = self.fbuf(f"{m}_dht", B * R)
            whh = P[f"lstm.{l}.weight_hh"]
            dc_next = None
            if self.fused_scan:
                ctr = self.lbuf("scan_counter", 4, torch.int32)
                ctr.zero_()
                K.lstm_scan_bwd(dH, whh, lay["gates"], lay["cs"], dG, steps, B, R, ctr, tf32=self.tc_lstm)
            for s in (range(steps - 1, -1, -1) if not self.fused_scan else ()):
                dh_s = dH[s * B * R:(s + 1) * B * R]
                if s < steps - 1:
                    # dh_total = dH[s] + dG[s+1] . W_hh
                    self.lin_dinput(m, f"lstm.{l}.weight_hh", dG[(s + 1) * B * 4 * R:(s + 2) * B * 4 * R], dht, B, 4 * R, R, addend=dh_s)
                    dh_s = dht
                dc_prev = dcA if (s % 2 == 0) else dcB
                K.lstm_pointwise_bwd(dh_s, dc_next, lay["gates"][s * B * 4 * R:(s + 1) * B * 4 * R],
                                     lay["cs"][s * B * R:(s + 1) * B * R], lay["cs"][(s + 1) * B * R:(s + 2) * B * R],
                                     dG[s * B * 4 * R:(s + 1) * B * 4 * R], dc_prev, B, R)
                dc_next = dc_prev
            if want_wgrad:
                with self.fork(self.LANE_WGRAD):   # off the critical path: nothing below reads a weight gradient
                    self.lin_wgrad(dG, lay["hs"], A.g[f"lstm.{l}.weight_hh"], rows, 4 * R, R)
                    self.lin_wgrad(dG, lay["inp"], A.g[f"lstm.{l}.weight_ih"], rows, 4 * R, R, reuse_dy=True)
                    K.colsum(dG, rows, 4 * R, 4 * R, A.g[f"lstm.{l}.bias_ih"])
                    K.colsum(dG, rows, 4 * R, 4 * R, A.g[f"lstm.{l}.bias_hh"])
            dIn = self.fbuf(f"{m}_dIn{l}", rows * R)
            self.lin_dinput(m, f"lstm.{l}.weight_ih", dG, dIn, rows, 4 * R, R)
            dH = dIn
        dE = dH
        in_dim = sv["in_dim"]
        if want_wgrad:
            with self.fork(self.LANE_WGRAD):
                self.lin_wgrad(dE, sv["X"], A.g["embed.weight"], rows, R, in_dim, ldx=sv["ldx"])
                K.colsum(dE, rows, R, R, A.g["embed.bias"])
        if want_dx:
            dX = dx_out if dx_out is not None else self.fbuf(f"{m}_dX", rows * in_dim)
            self.lin_dinput(m, "embed.weight", dE, dX, rows, R, in_dim)
            return dX
        return None

    def gaussian_heads_backward(self, m, dmu, dlv, steps, want_wgrad):
        K, B, R, z = self.K, self.B, self.R, self.z
        A = self.arena[m]
        rows = steps * B
        top = self.sv[m]["top"]
        dtop = self.fbuf(f"{m}_dtop", rows * R)
        K.gemm(dmu, A.p["mu_net.weight"], dtop, rows, R, z, b_mn=True)
        K.gemm(dlv, A.p["logvar_net.weight"], dtop, rows, R, z, b_mn=True, accumulate=True)
        if want_wgrad:
            K.gemm(dmu, top, A.g["mu_net.weight"], z, R, rows, a_mn=True, b_mn=True, lda=z, ldb=R)
            K.gemm(dlv, top, A.g["logvar_net.weight"], z, R, rows, a_mn=True, b_mn=True, lda=z, ldb=R)
            K.colsum(dmu, rows, z, z, A.g["mu_net.bias"])
            K.colsum(dlv, rows, z, z, A.g["logvar_net.bias"])
        return dtop

    def backward_decoder(self, plan):
        """loss = mse + beta*kld + weight_align*align  (models/p2p_model.py:261-262): decoder part + the loss scalars."""
        K, B, S, g, z, R, T = self.K, self.B, self.S, self.g, self.z, self.R, self.T
        opt = self.opt
        self.d_hpred[:(S + 1) * B * g].zero_()
        self.dH[:T * B * g].zero_()
        self.decoder_backward(0, S, want_wgrad=True, want_skip=True)
        # alignment loss (value + gradients into d_hpred / dH)
        K.align(self.Hlat, self.ix["in_idx"], self.h_pred, S - 1, B, g, float(opt["weight_align"]), self.align_partial,
                self.d_hpred, self.dH)
        # the four scalars
        self.loss_out = self.fbuf("loss_out", 4)
        E = B * self.frame_elems
        K.finalize_losses(self.mse_partial, S, plan.has_cpc, E, self.kl_sum, float(opt["batch_size"]), self.align_partial,
                          max(S - 1, 0), float(T), self.loss_out)
        if self.early_loss:
            K.publish_scalars(self.loss_out, 4, self._pub_host, self._pub_seq_dev)

    def backward_recurrent(self, plan):
        """Backward #1 through the three LSTMs: d h_pred -> frame predictor -> (z) -> posterior / prior -> dH."""
        K, B, S, g, z, R, T = self.K, self.B, self.S, self.g, self.z, self.R, self.T
        opt = self.opt
        # frame predictor (recon steps only; the CPC step has no cotangent in this pass)
        A = self.arena["frame_predictor"]
        rows = S * B
        dpre = self.fbuf("pred_dpre", (S + 1) * B * g)
        K.act_bwd(self.d_hpred, self.h_pred, dpre, rows * g, ACT_TANH)
        top = self.sv["frame_predictor"]["top"]
        self.lin_wgrad(dpre, top, A.g["output.0.weight"], rows, g, R)
        K.colsum(dpre, rows, g, g, A.g["output.0.bias"])
        dtop = self.fbuf("pred_dtop", (S + 1) * B * R)
        self.lin_dinput("frame_predictor", "output.0.weight", dpre, dtop, rows, g, R)
        wp = g + z + 2
        dXpred = self.lstm_backward("frame_predictor", dtop, S, want_wgrad=True, want_dx=True)
        # posterior / prior seeds: d z_post from the predictor input, beta * dKL
        dz = self.fbuf("dz_post", S * B * z)
        K.permute4(dXpred[g:], dz, (S * B, z, 1, 1), (wp, 1, 0, 0))
        n = S * B * z
        dmu, dlv, dmu_p, dlv_p = (self.fbuf(nm, n) for nm in ("dmu", "dlv", "dmu_p", "dlv_p"))
        K.reparam_kl_bwd(self.mu, self.lv, self.mu_p, self.lv_p, self.eps_post, self.eps_prior, dz, None,
                         float(opt["beta"]) / float(opt["batch_size"]), dmu, dlv, dmu_p, dlv_p, n)
        win = 2 * g + 2
        with self.fork(self.LANE_PRIOR):
            dtop_p = self.gaussian_heads_backward("prior", dmu_p, dlv_p, S, want_wgrad=False)
            dXprior = self.lstm_backward("prior", dtop_p, S, want_wgrad=False, want_dx=True)
        dtop = self.gaussian_heads_backward("posterior", dmu, dlv, S, want_wgrad=True)
        dXpost = self.lstm_backward("posterior", dtop, S, want_wgrad=True, want_dx=True)
        self.join(self.LANE_PRIOR)
        # latent gradients -> dH[T,B,g]
        ix = self.ix
        K.gather_add_cols(self.dH, dXpost, ix["tgt_idx"], S, T, B, g, win, 0)
        K.gather_add_cols(self.dH, dXpost, ix["glob_idx"], S, T, B, g, win, g)
        K.gather_add_cols(self.dH, dXprior, ix["in_idx"], S, T, B, g, win, 0)
        K.gather_add_cols(self.dH, dXprior, ix["glob_idx"], S, T, B, g, win, g)
        K.gather_add_cols(self.dH, dXpred, ix["in_idx"], S, T, B, g, wp, 0)

    def encoder_backward(self, plan):
        K, T, B, n, g = self.K, self.T, self.B, self.n, self.g
        A = self.arena["encoder"]
        N = T * B
        nskip = plan.nskip
        # lane 0 waits for the LSTM weight gradients (a no-op in single-GPU mode A, whose Adam step has joined every lane)
        self.join(self.LANE_WGRAD)
        if self.adt == torch.float32:
            dy = self.dH
        else:
            dy = self.buf("dH_act", N * g)
            K.permute4(self.dH, dy, (N * g, 1, 1, 1), (1, 0, 0, 0))
        cn, bn = self.enc_names(n)
        fin = self.enc_final
        st = fin["st"]
        K.bn_bwd(dy, fin["raw"], fin["y"], st["mean"], st["invstd"], st["gamma"], T, B, g, ACT_TANH, dy, st["sdz"], st["sdzx"])
        K.bn_param_grad(st["sdz"], st["sdzx"], T, g, A.g[bn + ".weight"], A.g[bn + ".bias"])
        A.g[cn + ".bias"].zero_()
        ctop = self.chans[-1]
        gw = self.fbuf(f"gwp_enc{n}", g * 16 * ctop)
        K.gemm(dy, fin["inp"], gw, g, 16 * ctop, N, a_mn=True, b_mn=True, lda=g, ldb=16 * ctop)
        K.transpose_batched(gw, A.g[cn + ".weight"], g, 16, ctop)
        gy = self.buf(f"enc_gy{n - 1}", N * 16 * ctop)
        K.gemm(dy, self._packed[f"enc{n}"], gy, N, 16 * ctop, g, b_mn=True)
        for l in range(n - 1, -1, -1):
            rec = self.enc[l]
            cin, cout, M, Ho = rec["cin"], rec["cout"], rec["M"], rec["Hout"]
            # skip-connection gradient from the decoder stage that consumed this layer's output
            k = n - 1 - l
            dsk = self.dec[k].get("dskip")
            if dsk is not None:
                K.add_indexed(gy, dsk, self.ix["skip_dst"], nskip, B * Ho * Ho * cout)
            cn, bn = self.enc_names(l)
            st = rec["st"]
            self.bn_backward(gy, rec["raw"], rec["y"], st, 0, T * cout, T, B * Ho * Ho, cout, ACT_LRELU)
            K.bn_param_grad(st["sdz"], st["sdzx"], T, cout, A.g[bn + ".weight"], A.g[bn + ".bias"])
            A.g[cn + ".bias"].zero_()
            gw = self.fbuf(f"gwp_enc{l}", cout * 16 * cin)
            if rec["imp"]:
                K.conv_gemm(1, gy, rec["inp"], gw, N, Ho, Ho, 0, cin, Cm=cout)
            else:
                K.gemm(gy, rec["col"], gw, cout, 16 * cin, M, a_mn=True, b_mn=True, lda=cout, ldb=16 * cin)
            K.transpose_batched(gw, A.g[cn + ".weight"], cout, 16, cin)   # [co][tap][ci] -> [co][ci][tap]
            if l > 0:
                gprev = self.buf(f"enc_gy{l - 1}", N * rec["Hin"] * rec["Hin"] * cin)
                if rec["imp"]:
                    K.conv_gemm(2, gy, self._packed[f"enc{l}"], gprev, N, Ho, Ho, cout, cin)
                else:
                    dcol = self.buf("scratch_dcol", M * 16 * cin)
                    K.gemm(gy, self._packed[f"enc{l}"], dcol, M, 16 * cin, cout, b_mn=True)
                    K.col2im(dcol, gprev, N, Ho, Ho, cin)
                gy = gprev

    def backward_prior(self, plan):
        """prior_loss = kld + weight_cpc*cpc (models/p2p_model.py:266-268): CPC chain through decoder and
        frame predictor (their *current* weights), then BPTT through the prior with weight gradients."""
        K, B, S, g, z, R = self.K, self.B, self.S, self.g, self.z, self.R
        opt = self.opt
        n = S * B * z
        dzp = self.fbuf("dz_prior", n)
        dzp[:n].zero_()
        if plan.has_cpc:
            self.decoder_backward(S, S + 1, want_wgrad=False, want_skip=False)
            A = self.arena["frame_predictor"]
            sv = self.sv["frame_predictor"]
            dpre = self.fbuf("cpc_dpre", B * g)
            K.act_bwd(self.d_hpred[S * B * g:], self.h_pred[S * B * g:], dpre, B * g, ACT_TANH)
            dh = self.fbuf("cpc_dh", B * R)
            self.lin_dinput("frame_predictor", "output.0.weight", dpre, dh, B, g, R)
            L = len(sv["layers"])
            dG = self.fbuf("cpc_dG", B * 4 * R)
            dcp = self.fbuf("cpc_dc", B * R)
            for l in range(L - 1, -1, -1):
                lay = sv["layers"][l]
                K.lstm_pointwise_bwd(dh, None, lay["gates"][S * B * 4 * R:(S + 1) * B * 4 * R], lay["cs"][S * B * R:(S + 1) * B * R],
                                     lay["cs"][(S + 1) * B * R:(S + 2) * B * R], dG, dcp, B, R)
                dh2 = self.fbuf(f"cpc_dh{l}", B * R)
                self.lin_dinput("frame_predictor", f"lstm.{l}.weight_ih", dG, dh2, B, 4 * R, R)
                dh = dh2
            wp = g + z + 2
            dX = self.fbuf("cpc_dX", B * wp)
            self.lin_dinput("frame_predictor", "embed.weight", dh, dX, B, R, wp)
            K.permute4(dX[g:], dzp[(S - 1) * B * z:], (B, z, 1, 1), (wp, 1, 0, 0))
        dmu, dlv, dmu_p, dlv_p = (self.fbuf(nm, n) for nm in ("dmu", "dlv", "dmu_p", "dlv_p"))
        K.reparam_kl_bwd(self.mu, self.lv, self.mu_p, self.lv_p, self.eps_post, self.eps_prior, None, dzp,
                         1.0 / float(opt["batch_size"]), dmu, dlv, dmu_p, dlv_p, n)
        dtop = self.gaussian_heads_backward("prior", dmu_p, dlv_p, S, want_wgrad=True)
        self.lstm_backward("prior", dtop, S, want_wgrad=True, want_dx=False)

    # -- optimiser --------------------------------------------------------------------------
    def grad_bucket(self, modules):
        """The contiguous slice of the pooled gradient arena that holds `modules` (they must be neighbours in ARENA_ORDER)."""
        idx = sorted(ARENA_ORDER.index(m) for m in modules)
        assert idx == list(range(idx[0], idx[-1] + 1)), f"{modules} are not contiguous in the arena"
        first, last = self.arena[ARENA_ORDER[idx[0]]], self.arena[ARENA_ORDER[idx[-1]]]
        return self.pool["grad"][first.base:last.base + last.numel]

    def allreduce(self, modules):
        """Data parallel: replicas hold batch shards; average the gradients of `modules` over NVLink -- ONE ncclAllReduce
        (AVG, no separate scaling pass) per contiguous bucket of the pooled arena."""
        dist, group, world = self.dist
        mods = sorted(modules, key=ARENA_ORDER.index)
        runs, cur = [], [mods[0]]
        for m in mods[1:]:
            if ARENA_ORDER.index(m) == ARENA_ORDER.index(cur[-1]) + 1:
                cur.append(m)
            else:
                runs.append(cur)
                cur = [m]
        runs.append(cur)
        for run in runs:
            buf = self.grad_bucket(run)
            if buf.is_cuda:
                dist.all_reduce(buf, op=dist.ReduceOp.AVG, group=group)
            else:   # gloo (CPU tests) has no AVG
                dist.all_reduce(buf, group=group)
                self.K.scale(buf, buf.numel(), 1.0 / world)

    def adam(self, modules):
        opt = self.opt
        self.join()   # weight gradients / side chains produced on other lanes
        if self.dist is not None:
            self.allreduce(modules)
        for m in modules:
            A = self.arena[m]
            A.step_t += 1
            self.K.adam(A.flat, A.grad, A.m, A.v, A.numel, float(opt["lr"]), float(opt["beta1"]), 0.999, 1e-8, A.step_t)

    # -- export -----------------------------------------------------------------------------
    def state_dict(self, m):
        out = OrderedDict()
        for k in self.arena[m].names:
            out[k] = self.arena[m].p[k]
        out.update(self.buffers[m])
        return out
