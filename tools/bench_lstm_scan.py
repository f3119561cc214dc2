#!/usr/bin/env python
"""CUDA-event timing of the persistent LSTM scan kernels: tf32 = 1 runs the thread-block-cluster scans for R in {64,128,256,512},
tf32 = 0 (or any other R) the cooperative-grid scans."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from p2pvg_b200._lib import CudaKernels  # noqa: E402

K = CudaKernels("cuda")
print("cluster-16 scans: cudaOccupancyMaxActiveClusters fwd(16 rows) / fwd(32 rows) / bwd =",
      [K.lib.p2pvg_lstm_cluster512_max_clusters(i) for i in range(3)])
print("cluster-8 scans (R=256): max active clusters fwd MT1 / fwd MT2 / bwd MT1 / bwd MT2 =",
      [K.lib.p2pvg_lstm_cluster_max_clusters(i) for i in range(4)])
S, R = 30, int(os.environ.get("R", "256"))
for B in (16, 64, 128, 256):
    dev = "cuda"
    pre = torch.randn(S, B, 4 * R, device=dev) * 0.5
    whh = torch.randn(4 * R, R, device=dev) / R ** 0.5
    bhh = torch.randn(4 * R, device=dev) * 0.1
    gates = torch.empty(S, B, 4 * R, device=dev)
    hs = torch.zeros(S + 1, B, R, device=dev)
    cs = torch.zeros(S + 1, B, R, device=dev)
    dG = torch.empty(S, B, 4 * R, device=dev)
    dh = torch.randn(S, B, R, device=dev)
    ctr = torch.zeros(4, dtype=torch.int32, device=dev)
    for tf32 in (True, False):
        if not tf32 and R == 512 and B > 128:
            continue   # exact-fp32 R=512 above 128 rows runs as per-step kernels in the engine (the cooperative grid does not fit)
        res = []
        for which in ("fwd", "bwd"):
            ts = []
            for rep in range(6):
                ctr.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                if which == "fwd":
                    K.lstm_scan_fwd(pre, whh, bhh, gates, hs, cs, S, B, R, ctr, tf32=tf32)
                else:
                    K.lstm_scan_bwd(dh, whh, gates, cs, dG, S, B, R, ctr, tf32=tf32)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            res.append(min(ts[2:]))
        print(f"R={R} B={B:4d} tf32={int(tf32)}: fwd {res[0] * 1e3 / S:6.2f} us/step  bwd {res[1] * 1e3 / S:6.2f} us/step")
