#!/usr/bin/env python3
"""Dev tool (GPU box): time the fp32 kernel for every (streams_per_cta, ksplit) at a few batch sizes."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np
import torch
import ntm_b200
from ntm_b200 import lib, signals

dev = torch.device("cuda:0")
z = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "tests/golden/ckpt_cfg2.npz"))
sd = {k: torch.from_numpy(z[k]) for k in z.files if k not in ("model_type", "weights_dir")}
m = ntm_b200.RNN(1, 64, 1, False).to(dev)
m.load_state_dict(sd)
mode = sys.argv[1] if len(sys.argv) > 1 else "fp32"
m.mode = mode
L = lib.load()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
print(f"mode={mode}")
with torch.inference_mode():
    for B, T in ((1, 48000), (8, 48000), (148, 24000), (1024, 24000), (4096, 12000), (16384, 6000)):
        x = signals.stream_batch_device(B, T, dev, dur=10.0).reshape(B, 1, T)
        for ks in (4, 2):
            for s in (1, 2, 4, 8):
                if B / s > 20000 or (B == 1 and s > 1) or (ks == 2 and s > 2):
                    continue
                L.ntm_set_tuning(s, ks)
                m.initialize_hidden()
                m(x[:, :, :512])
                torch.cuda.synchronize()
                best = 1e9
                for _ in range(2):
                    m.initialize_hidden()
                    e0.record(); m(x); e1.record(); torch.cuda.synchronize()
                    best = min(best, e0.elapsed_time(e1))
                print(f"B={B:6d} T={T:6d} ks={ks} s={s:2d}: {best:9.3f} ms  {B*T/best/1e3:10.3f} Msamples/s  "
                      f"{best*1e6/T:8.1f} ns/step", flush=True)
L.ntm_set_tuning(0, 0)
