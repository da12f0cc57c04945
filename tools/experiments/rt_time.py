#!/usr/bin/env python3
"""Dev tool (GPU box): per-block latency of real-time block mode, batch 1, 64-sample blocks, f16.

  GRU server     RealtimeStream.process / step() of the plain RNN (cfg 1 weights)

and for DiffDelRNN (cfg 3 weights) with history lengths D = 366 (cfg 3, max_delay 365) and D = 10001 (the reference's
default max_delay 10000):

  server         RealtimeDelayStream.process: host blocks x, d in, host y, pre_d out (one resident kernel)
  server step()  the same through the fixed x_in / d_in blocks
  block stream   DelayBlockStream.process on device blocks + stream synchronisation (delay check on: one more sync)
  forward        DiffDelRNN.forward per device block + stream synchronisation (allocation, checks, delay-assert sync)

Host clock around each call (every form ends in a synchronisation or a host handshake); median and p99 over --blocks blocks
after --warmup blocks.  Each process() form's output over the timed signal is checked against one long forward call."""
import argparse
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
T = 64


def stats(lat):
    lat = sorted(lat)
    return f"median {lat[len(lat) // 2] * 1e6:7.1f} us  p99 {lat[int(len(lat) * 0.99)] * 1e6:7.1f} us"


def timed(fn, blocks, warmup):
    out, lat = [], []
    for k, blk in enumerate(blocks):
        t0 = time.perf_counter()
        r = fn(*blk)
        dt = time.perf_counter() - t0
        out.append(tuple(v.clone() for v in r))
        if k >= warmup:
            lat.append(dt)
    return out, lat


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=300)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else 'unknown'}")
    n = args.blocks + args.warmup
    x = torch.from_numpy(signals.stream_batch(1, n * T)).contiguous()
    with torch.inference_mode():
        g = ntm_b200.RNN(1, 64, 1, False).to(DEV)
        g.load_state_dict(load_ckpt("cfg1"))
        g.mode = "f16"
        g.initialize_hidden()
        g.warm_start()
        h0 = g.hidden.clone()
        yref = g(x.to(DEV).reshape(1, 1, -1)).cpu().reshape(1, -1)
        g.hidden = h0
        torch.cuda.synchronize()
        rt = g.realtime_stream(1, T)
        try:
            out, lat = timed(lambda xb: (rt.process(xb),), [(x[:, k * T:(k + 1) * T].contiguous(),) for k in range(n)],
                             args.warmup)
            same = torch.equal(torch.cat([o[0] for o in out], 1), yref)
            print(f"GRU server, process()                    {stats(lat)}  {'bit-identical' if same else 'MISMATCH'}")
            lat = []
            for k in range(args.blocks):
                t0 = time.perf_counter()
                rt.step()
                lat.append(time.perf_counter() - t0)
            print(f"GRU server, step()                       {stats(lat)}")
        finally:
            rt.close()

        for max_d in (365, 10000):
            D = max_d + 1
            m = ntm_b200.DiffDelRNN(1, 64, 1, False, max_delay=max_d).to(DEV)
            m.load_state_dict(load_ckpt("cfg3"))
            m.mode = "f16"
            m.initialize_hidden(1, max_d)
            m.warm_start()
            h0, hist0 = m.hidden.clone(), m.diffdel.buffer.clone()
            d = torch.from_numpy(signals.delay_trajectory(1, n * T) * ((D - 0.5) / 292.0)).float().contiguous()
            yref, pref = m(x.to(DEV).reshape(1, 1, -1), d.to(DEV).reshape(1, 1, -1))
            yref, pref = yref.cpu().reshape(1, -1), pref.cpu().reshape(1, -1)
            hb = [(x[:, k * T:(k + 1) * T].contiguous(), d[:, k * T:(k + 1) * T].contiguous()) for k in range(n)]
            db = [(a.to(DEV).reshape(1, 1, T), b.to(DEV).reshape(1, 1, T)) for a, b in hb]
            sync = torch.cuda.current_stream(DEV).synchronize

            def same(out):
                y = torch.cat([o[0].cpu().reshape(1, -1) for o in out], 1)
                p = torch.cat([o[1].cpu().reshape(1, -1) for o in out], 1)
                return "bit-identical" if torch.equal(y, yref) and torch.equal(p, pref) else "MISMATCH"

            print(f"D = {D}")
            m.hidden, m.diffdel.buffer = h0.clone(), hist0.clone()
            st = m.realtime_stream(1, T)
            try:
                out, lat = timed(st.process, hb, args.warmup)
                print(f"  DiffDel server, process()              {stats(lat)}  {same(out)}")
                lat = []
                for k in range(args.blocks):
                    t0 = time.perf_counter()
                    st.step()
                    lat.append(time.perf_counter() - t0)
                print(f"  DiffDel server, step()                 {stats(lat)}")
            finally:
                st.close()
            for check in (True, False):
                m.diffdel.check_delay = check
                m.hidden, m.diffdel.buffer = h0.clone(), hist0.clone()
                bs = m.block_stream(1, T)

                def blk(a, b):
                    r = bs.process(a, b)
                    sync()
                    return r
                out, lat = timed(blk, db, args.warmup)
                bs.close()
                print(f"  DelayBlockStream, delay check {'on ' if check else 'off'}     {stats(lat)}  {same(out)}")
            m.diffdel.check_delay = True
            m.hidden, m.diffdel.buffer = h0.clone(), hist0.clone()

            def fwd(a, b):
                r = m(a, b)
                sync()
                return r
            out, lat = timed(fwd, db, args.warmup)
            print(f"  DiffDelRNN.forward per block           {stats(lat)}  {same(out)}")


if __name__ == "__main__":
    main()
