#!/usr/bin/env python3
"""Dev tool (GPU box): BASELINE cfg 3 (DiffDelGRU, 256 streams x 30 s, predict() semantics) per arithmetic mode.

    python tools/experiments/cfg3_time.py [--modes f16,fp32] [--max-delay N]

Prints the time per step and a hash of the four results (y, pre_d, final state, delay history), so that two builds can
be compared output for output on the same seeded inputs."""
import argparse
import hashlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import ntm_b200
from ntm_b200 import signals
from conftest import load_ckpt

ap = argparse.ArgumentParser()
ap.add_argument("--modes", default="f16,fp32")
ap.add_argument("--max-delay", type=int, default=signals.DELAY_MAX)
args = ap.parse_args()

dev = "cuda:0"
B, T = 256, 30 * 48000
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
print(f"# {torch.cuda.get_device_name(0)}, max_delay {args.max_delay}", flush=True)
with torch.inference_mode():
    md = ntm_b200.DiffDelRNN(1, 64, 1, False, max_delay=args.max_delay).to(dev)
    md.load_state_dict(load_ckpt("cfg3"))
    md.diffdel.check_delay = False
    x = signals.stream_batch_device(B, T, dev, dur=30.0).reshape(B, 1, T)
    d = signals.delay_trajectory_device(B, T, dev).reshape(B, 1, T)
    for mode in args.modes.split(","):
        md.mode = mode
        md.predict(x[:, :, :4800], d[:, :, :4800])
        torch.cuda.synchronize()
        e0.record(); y, p = md.predict(x, d); e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        h = hashlib.sha256()
        for t in (y, p, md.hidden, md.diffdel.buffer):
            h.update(t.contiguous().cpu().numpy().tobytes())
        print(f"cfg3 {mode} max_delay {args.max_delay}: {ms:.1f} ms, {B*T/ms/1e6:.3f} Gsamples/s, {ms*1e6/T:.1f} ns/step, "
              f"results {h.hexdigest()[:16]}", flush=True)
