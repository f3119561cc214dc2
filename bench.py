#!/usr/bin/env python
"""Benchmark of the p2pvg training hot path (BASELINE.json): frames/s of one P2PModel.forward train step
(forward + both backwards + five Adam updates) on synthetic batches of the BASELINE configurations.

    python bench.py [--config C2|C3|C4|C5] [--gpus N] [--steps K] [--warmup W] [--skip-prob P] [--strong] [--impl reference]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One JSON line on stdout (rank 0).  --dump-outputs DIR (rank 0) writes what the last of the K timed steps handed its caller
as DIR/<name>.npy, float32: the four losses, every module's updated parameters and their gradients, and the BatchNorm
running statistics (see dump_outputs).  The inputs (weights, batch, noise, skip draws) are seeded, so two builds run
with the same arguments can be compared output for output.
  value       device-timed throughput (CUDA events, max over ranks) of K graph-replayed steps, batch resident in HBM
  e2e         the same through the public drop-in API (p2pvg_b200.data.DevicePrefetcher feeding
              models.p2p_model.P2PModel.__call__): every step's batch is copied from pinned host memory inside the timed
              region and the four loss scalars are read back every step
  roofline    dominant kernel family.  C2/C3/C4: all bf16 tcgen05 launches of a step (useful FLOPs / CUDA-event time of
              those launches, instrumented eager pass) against the measured bf16 peak.  C5: the LSTM phases against HBM.
  roofline_lstm  the recurrent phases (forward scan + BPTT of the three LSTMs incl. reparameterisation / KL): SURVEY §8(d)
              model bytes S*3*Q_fwd over the phase time (each phase captured into its own CUDA graph and replayed between
              CUDA events), against the measured HBM copy bandwidth
  phases_ms   the same per-phase device times for the whole step
  cpu_baseline / --impl reference: the CPU oracle (port of the reference path) on the host cores, bounded sample
  library_baseline (C2, one GPU): the reference's step as stock torch-CUDA ops + autograd (cuDNN / cuBLAS, TF32 allowed) on
              the same GPU and workload -- what "PyTorch on a B200" does without this library
Configs (BASELINE.json `configs`; SURVEY.md §8d): C2 mnist dcgan_64 T=30 B=256/GPU (the config the metric is quoted on; default);
C3 weizmann-shaped vgg_64 C=3 T=30 B=128/GPU; C4 bair-shaped dcgan_128 C=3 T=30 global B=512 (64/GPU at 8 GPUs);
C5 human36m h36m_mlp T=60 rnn_size 512 global B=2048 (256/GPU at 8 GPUs).  C4/C5 keep the per-GPU share of the 8-GPU
configuration at every N (weak scaling) unless --strong, which fixes the global batch and divides it by N.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/sec (train step, device-timed) MovingMNIST 64x64 seq30"

CONFIGS = {
    "C2": dict(desc="mnist dcgan_64 seq_len 30 batch 256 per GPU (BASELINE configs[1])", backbone="dcgan_64", dataset="mnist", channels=1,
               width=64, T=30, rnn=256, per_gpu=256, global_batch=None, ref_batch=16, f_enc=205.5e6, f_dec=408.9e6),
    "C3": dict(desc="weizmann-shaped vgg_64 (3-ch 64x64) seq_len 30 batch 128 per GPU (BASELINE configs[2])", backbone="vgg_64",
               dataset="weizmann", channels=3, width=64, T=30, rnn=256, per_gpu=128, global_batch=None, ref_batch=4, f_enc=2281.2e6,
               f_dec=3489.1e6),
    "C4": dict(desc="bair-shaped dcgan_128 (3-ch 128x128) seq_len 30 global batch 512 over 8 GPUs = 64 per GPU (BASELINE configs[3])",
               backbone="dcgan_128", dataset="bair", channels=3, width=128, T=30, rnn=256, per_gpu=64, global_batch=512, ref_batch=4,
               f_enc=966.8e6, f_dec=1931.5e6),
    "C5": dict(desc="human36m h36m_mlp seq_len 60 rnn_size 512 global batch 2048 over 8 GPUs = 256 per GPU (BASELINE configs[4])",
               backbone="h36m_mlp", dataset="h36m", channels=1, width=None, T=60, rnn=512, per_gpu=256, global_batch=2048, ref_batch=256,
               f_enc=0.129e6, f_dec=0.297e6),
}
G_DIM, Z_DIM = 128, 10


def rnn_model(R, g=G_DIM, z=Z_DIM):
    """SURVEY.md §8(d): forward FLOPs per sample per executed step and parameter count of the three LSTMs."""
    f_post = 2 * (2 * g + 2) * R + 16 * R * R + 4 * R * z
    f_pred = 2 * (g + z + 2) * R + 32 * R * R + 2 * R * g
    p_gauss = (2 * g + 2) * R + R + (8 * R * R + 8 * R) + 2 * (R * z + z)
    p_pred = (g + z + 2) * R + R + 2 * (8 * R * R + 8 * R) + R * g + g
    return 2 * f_post + f_pred, 2 * p_gauss + p_pred


def algorithmic_flops(c, T, B):
    """W = 3T F_enc + (3T-2) F_dec + 3(T-1) F_rnn per sequence (SURVEY.md §8d; skip_prob = 0)."""
    f_rnn, _ = rnn_model(c["rnn"])
    return B * (3 * T * c["f_enc"] + (3 * T - 2) * c["f_dec"] + 3 * (T - 1) * f_rnn)


def lstm_model_bytes(c, S, B):
    """(steps) * 3 * Q_fwd, Q_fwd = 4 [P_rnn + B ((2g+2) 2 + (g+z+2) + 16R + 16R + 8z + g + 1)]  (SURVEY.md §8d)."""
    R, g, z = c["rnn"], G_DIM, Z_DIM
    _, p_rnn = rnn_model(R)
    q = 4 * (p_rnn + B * ((2 * g + 2) * 2 + (g + z + 2) + 16 * R + 16 * R + 8 * z + g + 1))
    return S * 3 * q, q


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"], which="measured (MEASURED_PEAKS.json: sustained bf16, copy HBM)")
    return dict(tflops=1590.0, hbm=6650.0, which="fallback (B200_PROFILING.md)")


class ClockSampler:
    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [c.strip() for c in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except Exception:
                continue
            for nm, v in zip(names, f[2:]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


DUMP_LIMIT = 64_000_000   # bytes --dump-outputs may write in all
DUMP_WHOLE = 4096         # arrays up to this many elements are always written whole


def step_outputs(eng, losses):
    """What one train step hands its caller (P2PModel exposes the parameters and their .grad as views of the engine's
    arenas): the losses, per module every updated parameter and its gradient, and the BatchNorm running statistics."""
    arrays = {"losses": losses}
    for m, A in eng.arena.items():
        for k in A.names:
            arrays[f"{m}.{k}"] = A.p[k]
            arrays[f"{m}.{k}.grad"] = A.g[k]
        arrays.update({f"{m}.{k}": v for k, v in eng.buffers[m].items() if v.is_floating_point()})
    return {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy (float32), DUMP_LIMIT bytes at most.  If the arrays are larger than that
    together, each one of more than DUMP_WHOLE elements is replaced by the same fraction of its flattened elements, in
    index order, at indices drawn from a fixed seed: every run and every build samples the same positions."""
    os.makedirs(out_dir, exist_ok=True)
    header = 128   # bytes of a .npy header for these shapes
    room = (DUMP_LIMIT - len(arrays) * (header + 4 * (DUMP_WHOLE + 1))) // 4
    frac = min(1.0, room / sum(a.size for a in arrays.values()))
    written = 0
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        keep = min(a.size, max(DUMP_WHOLE, int(a.size * frac)))
        if keep < a.size:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        path = os.path.join(out_dir, f"{name}.npy")
        np.save(path, a)
        written += os.path.getsize(path)
    assert written <= DUMP_LIMIT, written
    log(f"wrote {len(arrays)} arrays ({written / 1e6:.1f} MB, {100 * frac:.0f}% of the elements of the large ones) to {out_dir}")


def oracle_cfg(c):
    cfg = dict(g_dim=G_DIM, z_dim=Z_DIM, rnn_size=c["rnn"], predictor_rnn_layers=2, posterior_rnn_layers=1, prior_rnn_layers=1)
    if c["backbone"] == "h36m_mlp":
        cfg.update(backbone="mlp")
        width = "mlp"
    elif c["backbone"] == "vgg_64":
        cfg.update(backbone="vgg", channels=c["channels"], image_width=64)
        width = "vgg"
    else:
        cfg.update(channels=c["channels"], image_width=c["width"])
        width = c["width"]
    return cfg, width


def synth_batch(c, T, B, gen, device=None):
    if c["backbone"] == "h36m_mlp":   # loader standardises poses to std 3 (data/human36m/human36m.py:23,262)
        return 3 * torch.randn(T, B, 17, 3, generator=gen)
    return torch.rand(T, B, c["channels"], c["width"], c["width"], generator=gen)


def cpu_reference_steps(c, T, B, steps, warmup, threads, skip_prob):
    """Times the CPU oracle (port of reference models/p2p_model.py:185-271, Mode A) on a [T,B] batch."""
    from oracle import p2p_oracle as O
    from p2pvg_b200.engine import StepPlan
    torch.set_num_threads(threads)
    cfg, width = oracle_cfg(c)
    state = O.build_state(cfg, seed=1)
    adam = {m: O.new_adam_state(state[m]) for m in O.MODULES}
    opt = O.default_opt(batch_size=B, skip_prob=skip_prob)
    gen = torch.Generator().manual_seed(1234)
    times = []
    for it in range(warmup + steps):
        x = synth_batch(c, T, B, gen)
        probs = np.random.RandomState(it).uniform(0, 1, T - 1)
        eps = O.draw_eps(StepPlan(T, probs, opt).S, B, Z_DIM, seed=it)
        t0 = time.perf_counter()
        O.train_step(state, adam, x, opt, width, eps, probs, mode="A")
        dt = time.perf_counter() - t0
        log(f'cpu reference step {it} ({threads} threads): {dt:.2f} s')
        if it >= warmup:
            times.append(dt)
    return times


def cpu_baseline(c, T, skip_prob, steps, warmup):
    """Oracle port on the host cores.  The reference path is ~93k small ATen ops per step (SURVEY.md §3.2); beyond a few
    dozen threads the per-op fork/join cost dominates: on the 2xx-core GPU hosts an all-core run did not finish ONE
    T=30,B=16 step in 9 minutes (gpurun_out/r2a, round 2), 32 threads take 3.3 s.  Default = min(cores, 32);
    P2PVG_CPU_THREADS=a,b,... times each listed thread count and reports the best."""
    B = c["ref_batch"]
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    env = os.environ.get("P2PVG_CPU_THREADS")
    counts = [int(v) for v in env.split(",")] if env else [min(ncpu, 32)]
    runs = {}
    for th in counts:
        t = cpu_reference_steps(c, T, B, steps, warmup, th, skip_prob)
        runs[th] = T * B * len(t) / sum(t)
    best = max(runs, key=runs.get)
    sample = f"{steps} steps of T={T},B={B} of the oracle port (oracle/p2p_oracle.py, Mode A, torch CPU fp32); host has {ncpu} cores; " + \
             ", ".join(f"{th} threads: {v:.1f} frames/s" for th, v in runs.items()) + \
             "; more threads are slower on this path (per-op fork/join), see bench.py:cpu_baseline"
    return dict(value=runs[best], unit="frames/s", cores=best, kind="port", sample=sample), runs


def config_dict(c, name, T, B, world, skip_prob, graph, strong):
    return dict(workload=f"{name}: {c['desc']}", global_batch=B * world, seq_len=T, skip_prob=skip_prob, parallelism=f"dp{world}",
                cuda_graph=bool(graph), l2="per-step working set (GBs of activations) far exceeds the 126 MB L2; no flush needed",
                update_mode="A (reference two-phase update)", scaling_mode="strong" if strong else "weak")


def run_reference(args, c):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    T = args.seq or c["T"]
    world = args.gpus
    B = per_gpu_batch(args, c, world)
    base, runs = cpu_baseline(c, T, args.skip_prob, max(1, args.steps), max(0, min(args.warmup, 1)))
    val = base["value"]
    line = dict(metric=METRIC, value=val, unit="frames/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * T * c["ref_batch"] / val, higher_is_better=True, scaling="strong" if args.strong else "weak",
                vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=config_dict(c, args.config, T, B, world, args.skip_prob, not args.no_graph, args.strong),
                cpu_baseline=base, e2e=dict(value=val, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


def per_gpu_batch(args, c, world):
    if args.batch:
        return args.batch
    if args.strong:
        gb = c["global_batch"] or c["per_gpu"]
        return max(1, gb // world)
    return c["per_gpu"]


def library_baseline(c, T, B, dev, steps=3):
    """The reference's step as stock torch-CUDA ops + autograd on this GPU (oracle restatement run on the device; cuDNN /
    cuBLAS with TF32 allowed = the fastest stock configuration measured, profiles/torch_cuda_baseline_r01.txt)."""
    from oracle import p2p_oracle as O
    cfg, width = oracle_cfg(c)
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.benchmark = True
    try:
        state = {m: {k: v.to(dev) for k, v in sd.items()} for m, sd in O.build_state(cfg, seed=1).items()}
        adam = {m: O.new_adam_state(state[m]) for m in O.MODULES}
        opt = O.default_opt(batch_size=B)
        x = synth_batch(c, T, B, torch.Generator().manual_seed(1)).to(dev)
        probs = np.random.RandomState(0).uniform(0, 1, T - 1)
        eps = O.draw_eps(T - 1, B, Z_DIM, seed=3).to(dev)
        times = []
        for it in range(steps + 2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            O.train_step(state, adam, x, opt, width, eps, probs, mode="A")
            e1.record()
            torch.cuda.synchronize()
            if it >= 2:
                times.append(e0.elapsed_time(e1))
        ms = float(np.median(times))
        del state, adam, x
        torch.cuda.empty_cache()
        return dict(value=T * B / ms * 1e3, unit="frames/s", ms_per_step=ms, precision="tf32 (allow_tf32, cudnn.benchmark)",
                    what="reference train step as stock torch-CUDA ops + autograd (cuDNN/cuBLAS) on the same GPU, same T and B")
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = prev


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--batch", type=int, default=0, help="sequences per GPU (default: the config's)")
    ap.add_argument("--seq", type=int, default=0)
    ap.add_argument("--skip-prob", type=float, default=0.0, help="0.5 = the README's MNIST value (random frame skipping, np.random.seed(0))")
    ap.add_argument("--strong", action="store_true", help="fixed global batch divided by the number of GPUs")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-library", action="store_true")
    ap.add_argument("--skip-phases", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    c = CONFIGS[args.config]
    if args.impl == "reference":
        return run_reference(args, c)

    import importlib
    from p2pvg_b200.models.p2p_model import P2PModel
    from p2pvg_b200.data import DevicePrefetcher, bind_host_to_gpu

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # pinned staging memory is first-touched by this process: keep it on the GPU's NUMA node (H2D at full PCIe rate)
    all_cpus = bind_host_to_gpu(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    T = args.seq or c["T"]
    B = per_gpu_batch(args, c, world)
    os.environ["P2PVG_PRECISION"] = args.precision
    # multi-GPU: the NCCL all-reduces are captured into the step graph as well (P2PVG_DP_GRAPH=0 disables)
    dp_graph = os.environ.get("P2PVG_DP_GRAPH", "1") != "0"
    os.environ["P2PVG_GRAPH"] = "0" if (args.no_graph or (world > 1 and not dp_graph)) else "1"
    torch.manual_seed(1)
    np.random.seed(0)
    backbone = importlib.import_module(f"p2pvg_b200.models.{c['backbone']}")
    opt = types.SimpleNamespace(dataset=c["dataset"], backbone_net=backbone, lr=1e-3, beta1=0.9, beta=1e-4, weight_cpc=100.0,
                                weight_align=0.5, skip_prob=args.skip_prob, n_past=1, last_frame_skip=False, batch_size=B)
    model = P2PModel(B, c["channels"], G_DIM, Z_DIM, c["rnn"], 1, 1, 2, opt=opt).cuda()
    model.train()
    gen = torch.Generator().manual_seed(1234 + rank)
    x_host = synth_batch(c, T, B, gen).pin_memory()
    x_dev = x_host.to(dev)
    eng = model.engine(c["width"] or 0)
    if world > 1:
        eng.dist = (dist, None, world)
    K = eng.K
    use_graph = model.use_graph
    pose = c["backbone"] == "h36m_mlp"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    log(f'{args.config}: model built (T={T}, B={B}/GPU, world {world}); warm-up')
    # ---- device-timed, batch resident in HBM --------------------------------------------------------
    nwarm = max(args.warmup, 3)
    for _ in range(nwarm):
        eng.step(x_dev, use_graph=use_graph, return_device=True)
    if args.skip_prob > 0 and use_graph:
        # random frame skipping: every (T, executed steps) signature has its own CUDA graph -- warm up until a run of
        # steps needed no new capture, so that the timed region only replays
        quiet = 0
        while quiet < 12 and nwarm < 150:
            n_before = sum(1 for v in eng._graphs.values() if v != "warm")
            warm_before = sum(1 for v in eng._graphs.values() if v == "warm")
            eng.step(x_dev, use_graph=use_graph, return_device=True)
            nwarm += 1
            same = (sum(1 for v in eng._graphs.values() if v != "warm") == n_before and
                    sum(1 for v in eng._graphs.values() if v == "warm") == warm_before == 0)
            quiet = quiet + 1 if same else 0
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    n0 = K.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    tw0 = time.time()
    e0.record()
    executed = 0
    for _ in range(args.steps):
        out = eng.step(x_dev, use_graph=use_graph, return_device=True)
        executed += eng.last_plan.S
    e1.record()
    barrier()
    tw1 = time.time()
    if args.dump_outputs and rank == 0:   # now: every later step trains the same model on and reuses the loss buffer
        dump_outputs(args.dump_outputs, step_outputs(eng, out))
    launches = K.launches - n0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = ms.item() / args.steps
    log(f'timed region done: {ms_step:.2f} ms/step')
    clocks = sampler.stop(tw0, tw1) if rank == 0 else None
    value = T * B * world / (ms_step * 1e-3)

    # ---- end to end through the public API ----------------------------------------------------------
    def host_batches(n):
        for _ in range(n):
            yield x_host

    def call(xb):
        return model((None, xb, None), 0, T - 1) if pose else model(xb, 0, T - 1)

    # ONE input pipeline for warm-up and timed steps, so that the timed region sees its steady state (no stream / slot set-up, no
    # un-overlapped first copy): 3 warm-up steps, then exactly K steps, each of which issues the host->device copy of a following
    # batch (one batch more than consumed is supplied, so the last timed step does too -> K copies of h2d_bytes_per_step inside
    # the region).  One train step per batch, nothing else reads it -> the slot may be refilled as soon as the step has copied it
    # away; with several GPUs the refill is left where it was (after the step = during the next forward), away from the
    # all-reduce phases.
    e2e_warm = 3
    pf = DevicePrefetcher(host_batches(e2e_warm + args.steps + 1), dev, early_release=(world == 1),
                          copy_streams=int(os.environ.get("P2PVG_BENCH_COPY_STREAMS", "1")))
    feed = iter(pf)
    for _ in range(e2e_warm):
        call(next(feed))
        pf.release()
    barrier()
    e0.record()
    for _ in range(args.steps):
        losses = call(next(feed))
        pf.release()
    e1.record()
    barrier()
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_val = T * B * world / (ms2.item() / args.steps * 1e-3)
    log(f'e2e done: {ms2.item() / args.steps:.2f} ms/step')
    # the same loop WITHOUT the host->device copy (batch already resident): separates the per-step host / synchronisation
    # latency (the reference API returns host scalars every step, so the GPU idles while Python prepares the next step)
    # from the cost of the H2D copy itself
    e0.record()
    for _ in range(args.steps):
        call(x_dev)
    e1.record()
    barrier()
    ms3 = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms3, op=dist.ReduceOp.MAX)
    # host cost of enqueueing one step (no synchronisation inside the loop): what the GPU waits for after every
    # synchronous loss read-back
    torch.cuda.synchronize(dev)
    th0 = time.perf_counter()
    for _ in range(args.steps):
        eng.step(x_dev, use_graph=use_graph, return_device=True)
    host_enqueue_ms = (time.perf_counter() - th0) / args.steps * 1e3
    torch.cuda.synchronize(dev)
    barrier()
    # raw host->device rate of this box for the step's input (GPU otherwise idle), one copy at a time and split over
    # several streams: an exposed H2D copy means the box sustains less than bytes_per_step / ms_per_step
    def h2d_rate(nstreams, reps=3):
        streams = [torch.cuda.Stream(dev) for _ in range(nstreams)]
        dst = torch.empty_like(x_dev)
        hs, ds = x_host.view(-1).chunk(nstreams), dst.view(-1).chunk(nstreams)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(reps):
            for st, h, d in zip(streams, hs, ds):
                with torch.cuda.stream(st):
                    d.copy_(h, non_blocking=True)
        torch.cuda.synchronize(dev)
        return reps * x_host.numel() * x_host.element_size() / (time.perf_counter() - t0) / 1e9
    h2d_rates = {f"{n}_streams": round(h2d_rate(n), 2) for n in (1, 2, 4)}
    barrier()
    e2e_detail = dict(ms_per_step=ms2.item() / args.steps, ms_per_step_batch_resident=ms3.item() / args.steps,
                      host_enqueue_ms_per_step=host_enqueue_ms, h2d_gbps_gpu_idle=h2d_rates,
                      h2d_gbps_needed=x_host.numel() * x_host.element_size() / (ms_step * 1e-3) / 1e9,
                      loss_readback=("early: four scalars + sequence number stored to page-locked host memory right after the loss "
                                     "finalisation and polled by P2PModel.forward; the backward passes / optimiser of step i overlap the "
                                     "host work of step i+1" if eng.early_loss else "blocking device-to-host copy after the whole step"),
                      note="ms_per_step_batch_resident - device-timed ms_per_step = per-step host + sync latency; "
                           "ms_per_step - ms_per_step_batch_resident = exposed part of the H2D copy")

    pk = peaks()
    roof = roof_lstm = phases = None
    if rank == 0:
        np.random.seed(0)
        saved_dist, eng.dist = eng.dist, None   # everything below is a rank-0-only measurement: no collectives
        try:
            eng.step(x_dev, use_graph=False, return_device=True)   # plan of the measured pattern for the instrumented passes
        finally:
            eng.dist = saved_dist
        S_meas = eng.last_plan.S
    # ---- roofline of the tensor-core kernels: instrumented eager pass ------------------------------
    if rank == 0 and args.precision == "bf16" and not pose:
        rec = []
        orig = K.gemm

        def timed_gemm(A, Bm, C, M, N, Kd, **kw):
            if A.dtype == torch.bfloat16:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                orig(A, Bm, C, M, N, Kd, **kw)
                b.record()
                # block-diagonal weights (thin first / last layers): 3/4 of the executed MACs multiply structural zeros
                useful = 0.25 if Bm.data_ptr() in {t.data_ptr() for k_, t in eng._packed.items() if ".bd" in k_} else 1.0
                rec.append((a, b, useful * 2.0 * M * N * Kd, (M, N, Kd, bool(kw.get("a_mn")), bool(kw.get("b_mn")), str(C.dtype))))
            else:
                orig(A, Bm, C, M, N, Kd, **kw)

        orig_conv = K.conv_gemm

        def timed_conv(kind, a_, b_, c_, N_, H_, W_, Ck, Cn, Cm=0, **kw):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            orig_conv(kind, a_, b_, c_, N_, H_, W_, Ck, Cn, Cm=Cm, **kw)
            b.record()
            taps = 9 if kind >= 3 else 16
            pix = float(N_) * H_ * W_   # small-map pixels; every kind does `taps` worth of MACs per (pixel, Ck|Cm, Cn)
            fl_ = 2.0 * pix * taps * (Cm if kind in (1, 4) else Ck) * Cn
            rec.append((a, b, fl_, (f"conv_gemm kind{kind}", N_, H_, W_, Ck, Cn, Cm)))

        K.gemm = timed_gemm
        K.conv_gemm = timed_conv
        saved_dist, eng.dist = eng.dist, None  # rank-0-only pass: no collectives
        eng._serial = True                     # one stream: a GEMM must not share the GPU with a side lane while it is timed
        try:
            np.random.seed(0)
            eng.step(x_dev, use_graph=False, return_device=True)
            torch.cuda.synchronize()
        finally:
            eng._serial = False
            eng.dist = saved_dist
            del K.gemm, K.conv_gemm   # instance attributes shadowing the methods
        tms = sum(r[0].elapsed_time(r[1]) for r in rec)
        fl = sum(r[2] for r in rec)
        if os.environ.get("P2PVG_DUMP_GEMMS"):
            rows = [dict(shape=r[3], ms=r[0].elapsed_time(r[1]), tflops=r[2] / (r[0].elapsed_time(r[1]) * 1e-3) / 1e12) for r in rec]
            json.dump(rows, open(os.environ["P2PVG_DUMP_GEMMS"], "w"))
        ach = fl / (tms * 1e-3) / 1e12
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic_r02.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get(args.config)
        w_alg = algorithmic_flops(c, T, B)
        roof = dict(bound="tensor",
                    kernel="conv_gemm_kernel + gemm_tc_kernel: all bf16 tcgen05 launches of the step (persistent, TMA 2-D/4-D staged, "
                           "tcgen05.mma kind::f16, double-buffered TMEM accumulators)",
                    achieved=ach, peak=pk["tflops"], unit="TFLOP/s", frac=ach / pk["tflops"], traffic=traffic, peak_source=pk["which"],
                    launches_per_step=len(rec), gemm_ms_per_step=tms,
                    executed_gemm_tflop_per_step=fl / 1e12,   # useful MACs only (zeros of block-diagonal weights excluded)
                    step_executed_frac=(fl / (ms_step * 1e-3)) / 1e12 / pk["tflops"],
                    survey_W_tflop_per_step=w_alg / 1e12,
                    note="step_executed_frac = executed tcgen05 FLOPs over the WHOLE step time; survey_W (SURVEY §8d) counts the "
                         "skip half of every decoder layer once per decode although the engine computes it once per distinct skip "
                         "frame, so W is not used as a numerator")
    # ---- per-phase device times and the LSTM HBM roofline ------------------------------------------
    if rank == 0 and not args.skip_phases:
        phases = eng.time_phases(x_dev)
        tp = os.path.join(ROOT, "profiles", "traffic_r02.json")
        lstm_traffic = json.load(open(tp)).get("C5") if (pose and os.path.exists(tp)) else None
        t_lstm = phases["lstm_fwd"] + phases["lstm_bwd"] + phases["prior_bwd"]
        model_bytes, q_fwd = lstm_model_bytes(c, S_meas, B)
        ach = model_bytes / (t_lstm * 1e-3) / 1e9
        roof_lstm = dict(bound="hbm", kernel="recurrent phases: lstm_cl_{fwd,bwd} cluster scans + input / head GEMMs + reparam_kl + concat "
                                             "(posterior, prior, frame predictor; forward, BPTT #1, prior BPTT #2 incl. the CPC chain)",
                         achieved=ach, peak=pk["hbm"], unit="GB/s", frac=ach / pk["hbm"], traffic=lstm_traffic, peak_source=pk["which"],
                         model_bytes_per_step=model_bytes, q_fwd_bytes=q_fwd, executed_timesteps=S_meas, phase_ms=t_lstm,
                         note="model bytes S*3*Q_fwd of SURVEY §8(d); the cluster scans keep W_hh in registers and move fewer HBM bytes "
                              "than the model, so this is a time-to-model ratio, not measured DRAM traffic")
        if pose:
            roof = roof_lstm
    # ---- library baseline: stock torch-CUDA on the same GPU ----------------------------------------
    lib = None
    if rank == 0 and world == 1 and args.config == "C2" and not args.skip_library and args.skip_prob == 0:
        try:
            lib = library_baseline(c, T, B, dev)
            log(f'library baseline: {lib["ms_per_step"]:.1f} ms/step')
        except Exception as e:   # e.g. out of memory next to a large configuration: report, never fail the bench
            lib = dict(unavailable=repr(e)[:200])
    # ---- CPU baseline (oracle port) on the host cores: bounded sample -------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:   # reported at N = 1 only (the contract): bounded sample on the host cores
        if all_cpus:
            os.sched_setaffinity(0, all_cpus)
        cpu, _ = cpu_baseline(c, T, args.skip_prob, 2, 1)
        log(f'cpu baseline done: {cpu}')

    if rank == 0:
        line = dict(metric=METRIC, value=value, unit="frames/s", n_gpus=world, steps=args.steps, warmup=nwarm,
                    ms_per_step=ms_step, higher_is_better=True, scaling="strong" if args.strong else "weak", vs_baseline=None,
                    dtype=("bf16" if args.precision == "bf16" else "f32"), data="synthetic",
                    config=config_dict(c, args.config, T, B, world, args.skip_prob, use_graph, args.strong),
                    roofline=roof, roofline_lstm=roof_lstm, phases_ms=phases, cpu_baseline=cpu, library_baseline=lib,
                    e2e=dict(value=e2e_val, unit="frames/s", h2d_bytes_per_step=int(x_host.numel() * 4), d2h_bytes_per_step=20 if eng.early_loss else 16,
                             detail=e2e_detail),
                    gpu_launches=int(launches), executed_timesteps_per_step=executed / args.steps, clocks=clocks,
                    losses=[float(v) for v in losses])
        print(json.dumps(line), flush=True)
    if world > 1:
        # tear-down must never hang the launcher: drop the CUDA graphs that hold captured NCCL kernels, give
        # destroy_process_group a bounded time, then leave without running interpreter-exit hooks
        import gc
        barrier()
        torch.cuda.synchronize()
        eng._graphs.clear()
        gc.collect()
        sys.stdout.flush()
        sys.stderr.flush()
        t = threading.Thread(target=dist.destroy_process_group, daemon=True)
        t.start()
        t.join(15)
        os._exit(0)


if __name__ == "__main__":
    main()
