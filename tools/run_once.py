#!/usr/bin/env python3
"""Dev tool (GPU box): one forward of B streams x T samples (for ncu captures).
   usage: run_once.py B T [mode] [s] [ks] [diffdel]    ((s, ks): a kernel selector of ntm_set_tuning, include/ntm_b200.h)"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import ntm_b200
from ntm_b200 import lib, signals

B, T = int(sys.argv[1]), int(sys.argv[2])
mode = sys.argv[3] if len(sys.argv) > 3 else "fp32"
s = int(sys.argv[4]) if len(sys.argv) > 4 else 0
ks = int(sys.argv[5]) if len(sys.argv) > 5 else 0
diffdel = len(sys.argv) > 6
dev = torch.device("cuda:0")
tag = "cfg3" if diffdel else "cfg2"
z = np.load(os.path.join(ROOT, f"tests/golden/ckpt_{tag}.npz"))
sd = {k: torch.from_numpy(z[k]) for k in z.files if k not in ("model_type", "weights_dir")}
lib.load().ntm_set_tuning(s, ks)
with torch.inference_mode():
    x = signals.stream_batch_device(B, T, dev, dur=10.0).reshape(B, 1, T)
    if diffdel:
        m = ntm_b200.DiffDelRNN(1, 64, 1, False, max_delay=signals.DELAY_MAX).to(dev)
        m.load_state_dict(sd)
        m.mode = mode
        d = signals.delay_trajectory_device(B, T, dev).reshape(B, 1, T)
        y, _ = m.predict(x, d)
    else:
        m = ntm_b200.RNN(1, 64, 1, False).to(dev)
        m.load_state_dict(sd)
        m.mode = mode
        y = m.predict(x)
    torch.cuda.synchronize()
    print("checksum", float(y.double().sum()))
