#!/usr/bin/env python3
"""Dev tool (GPU box): the stream-major tcgen05 kernel per operand format, job-queue and static schedule, at throughput widths.
usage: tcs_speed.py [B T]..."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import ntm_b200
from ntm_b200 import lib, signals
from conftest import load_ckpt

dev = "cuda:0"
L = lib.load()
sms = L.ntm_query(lib.Q_SM_COUNT)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
args = [int(v) for v in sys.argv[1:]]
widths = list(zip(args[::2], args[1::2])) or [(sms * 256, 3000), (65536, 3000), (sms * 128, 3000)]
with torch.inference_mode():
    m = ntm_b200.RNN(1, 64, 1, False).to(dev)
    m.load_state_dict(load_ckpt("cfg2"))
    m.mode = "fp32"
    m.initialize_hidden(); m.warm_start()
    hw = m.hidden.clone()
    for B, T in widths:
        x = signals.stream_batch_device(B, T, dev, dur=10.0).reshape(B, 1, T)
        ref = None
        for mode in ("f16", "f16x3", "tf32", "bf16"):
            m.mode = mode
            tiles = 2 if B >= 190 * sms else 1
            for sched in ("dynamic", "static"):
                L.ntm_set_tuning(tiles + (4 if sched == "static" else 0), 4)
                m.hidden = hw.expand(1, B, 64).contiguous(); m(x[:, :, :300])
                best = 1e9
                for _ in range(3):
                    m.hidden = hw.expand(1, B, 64).contiguous()
                    e0.record(); y = m(x); e1.record(); torch.cuda.synchronize()
                    best = min(best, e0.elapsed_time(e1))
                if ref is None:
                    L.ntm_set_tuning(8, 3)
                    m.mode = "f16x3"
                    m.hidden = hw.expand(1, 512, 64).contiguous()
                    ref = m(x[:512])
                    m.mode = mode
                err = float((y[:512] - ref).abs().max())
                esr = float(((y[:512] - ref) ** 2).sum() / (ref ** 2).sum())
                print(f"B={B} T={T} {mode:6s} {sched:7s} tiles={tiles}: {best:8.3f} ms {B*T/best/1e6:7.3f} Gs/s "
                      f"{best*1e-3*1.965e9*sms/(B*T):6.2f} clk/stream-step/SM | vs strict mma.sync (512 streams): max-abs {err:.2e} ESR {esr:.2e}",
                      flush=True)
L.ntm_set_tuning(0, 0)
