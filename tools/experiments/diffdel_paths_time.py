#!/usr/bin/env python3
"""Dev tool (GPU box): DiffDelRNN launches whose pre_d history does not fit the on-chip ring of the mma.sync kernels, so that
the GRU writes pre_d and the stand-alone delay line (csrc/delay.cu) runs behind it (cfg 3 weights, skip off):

  256 x 30 s, D = 10001     f16 (lean 4-stream mma.sync kernel) and fp32 (CUDA-core kernel), DiffDelRNN.forward
  2048 x 10 s, D = 2001     f16, the 8-stream mma.sync form (automatic choice at 2048 streams), DiffDelRNN.forward
  batch 1, D = 2001         DelayBlockStream.process on 64-sample device blocks + stream synchronisation, delay check on / off

Batched forms: CUDA events around each forward call from the same warm state, median over --reps calls after one untimed
call.  Block stream: host clock around each block, median and p99 over --blocks blocks after --warmup blocks.

--hashes prints a digest of y, pre_d, the final state and the rolled history for fp32, f16, f16x3 and tf32 at D = 366, 2001
and 10001, batched (a predict() call, then a warm-up call and a normal call) and through DelayBlockStream, so that two builds
can be compared output for output on the same seeded inputs."""
import argparse
import hashlib
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch

import ntm_b200
from conftest import load_ckpt
from ntm_b200 import signals

DEV = "cuda:0"
FS = 48000
BLK = 64


def model(mode, max_delay):
    m = ntm_b200.DiffDelRNN(1, 64, 1, False, max_delay=max_delay).to(DEV)
    m.load_state_dict(load_ckpt("cfg3"))
    m.mode = mode
    return m


def inputs(B, T, D, seed=0):
    x = signals.stream_batch_device(B, T, DEV, dur=T / FS).reshape(B, 1, T)
    g = torch.Generator(device=DEV).manual_seed(seed)
    ph = torch.rand((B, 1, 1), device=DEV, generator=g) * 6.0
    t = torch.arange(T, device=DEV, dtype=torch.float32).reshape(1, 1, T)
    d = (0.5 * (D - 1) * (1.0 + 0.9 * torch.sin(t / 700.0 + ph))).contiguous()   # 0.05 .. 0.95 of max_delay
    return x, d


def digest(*ts):
    h = hashlib.sha256()
    for t in ts:
        h.update(t.detach().float().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def batched(mode, B, sec, D, reps):
    m = model(mode, D - 1)
    T = int(sec * FS)
    x, d = inputs(B, T, D)
    with torch.inference_mode():
        m.initialize_hidden(1, D - 1)
        m.warm_start()
        h0 = m.hidden.expand(1, B, 64).contiguous()
        hist0 = m.diffdel.buffer.expand(B, 1, -1).contiguous()
        m.diffdel.check_delay = False          # time the recurrent launch(es), not the assert's synchronisation
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ms = []
        for k in range(reps + 1):
            m.hidden, m.diffdel.buffer = h0, hist0
            torch.cuda.synchronize()
            ev[0].record()
            y, pre = m(x, d)
            ev[1].record()
            torch.cuda.synchronize()
            if k:
                ms.append(ev[0].elapsed_time(ev[1]))
        kernel = ntm_b200.lib.query(ntm_b200.lib.Q_LAST_KERNEL)
        med = sorted(ms)[len(ms) // 2]
        print(f"{B:5d} x {sec:g} s  D = {D:5d}  {mode:5s}  kernel {kernel}  median {med:9.2f} ms  "
              f"{B * T / med * 1e3:10.4g} samples/s  {digest(y, pre, m.hidden, m.diffdel.buffer)}", flush=True)


def block_stream(mode, D, blocks, warmup):
    m = model(mode, D - 1)
    n = blocks + warmup
    x, d = inputs(1, n * BLK, D, seed=1)
    sync = torch.cuda.current_stream(DEV).synchronize
    with torch.inference_mode():
        for check in (True, False):
            m.initialize_hidden(1, D - 1)
            m.warm_start()
            m.diffdel.check_delay = check
            bs = m.block_stream(1, BLK)
            lat, ys, ps = [], [], []
            for k in range(n):
                xb, db = x[:, :, k * BLK:(k + 1) * BLK], d[:, :, k * BLK:(k + 1) * BLK]
                t0 = time.perf_counter()
                y, pre = bs.process(xb, db)
                sync()
                dt = time.perf_counter() - t0
                ys.append(y.clone())
                ps.append(pre.clone())
                if k >= warmup:
                    lat.append(dt)
            h, hist = bs.close()
            lat.sort()
            print(f"    1 x {BLK}-sample blocks  D = {D:5d}  {mode:5s}  DelayBlockStream, check {'on ' if check else 'off'}  "
                  f"median {lat[len(lat) // 2] * 1e6:7.1f} us  p99 {lat[int(len(lat) * 0.99)] * 1e6:7.1f} us  "
                  f"{digest(torch.cat(ys, 2), torch.cat(ps, 2), h, hist)}", flush=True)


def hashes():
    for D in (366, 2001, 10001):
        for mode in ("fp32", "f16", "f16x3", "tf32"):
            m = model(mode, D - 1)
            B, T = 16, 2 * FS
            x, d = inputs(B, T, D, seed=D)
            with torch.inference_mode():
                y, pre = m.predict(x, d)
                out = [y, pre, m.hidden, m.diffdel.buffer]
                y, pre = m(x[:, :, :4096], d[:, :, :4096], warmup=True)
                out += [y, pre, m.hidden, m.diffdel.buffer]
                y, pre = m(x[:, :, 4096:9000], d[:, :, 4096:9000])
                out += [y, pre, m.hidden, m.diffdel.buffer]
                bs = m.block_stream(B, BLK)
                for k in range(40):
                    y, pre = bs.process(x[:, :, k * BLK:(k + 1) * BLK].contiguous(), d[:, :, k * BLK:(k + 1) * BLK].contiguous())
                    out += [y.clone(), pre.clone()]
                out += list(bs.close())
                print(f"hash D = {D:5d}  {mode:5s}  {digest(*out)}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--blocks", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--hashes", action="store_true")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else 'unknown'}")
    if args.hashes:
        hashes()
        return
    batched("f16", 256, 30, 10001, args.reps)
    batched("fp32", 256, 30, 10001, args.reps)
    batched("f16", 2048, 10, 2001, args.reps)
    block_stream("f16", 2001, args.blocks, args.warmup)


if __name__ == "__main__":
    main()
