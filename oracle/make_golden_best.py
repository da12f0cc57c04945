#!/usr/bin/env python3
"""Golden vectors for ALL shipped `_BEST` checkpoints (12: 6 GRU, 6 DiffDelGRU), from the REAL reference.

Run in the build container only (imports /root/reference/code/model.py):
    python oracle/make_golden_best.py
Writes tests/golden/golden_best12.npz: per checkpoint i the state_dict tensors (`w{i}_<key>`), the class name and folder,
the warm-start state after `warm_start()` (input independent: a 64-float known answer per checkpoint), and for two
signals inside every checkpoint's stable regime the reference `predict` output in float32 (B = 1), the float64 ground
truth's distance (the reference's own fp32-vs-fp64 floor, a scalar per case).  DiffDelGRU: `y` and `pre_d`, the delay
trajectory being signals.delay_trajectory (max_delay = signals.DELAY_MAX, as code/test-model.py:223 would derive it).
Asserts on the way that oracle/ref_torch.py is bit-identical to the reference classes and that oracle/ntm_oracle.c agrees
to float32 round-off for every checkpoint, i.e. pins the oracle on all shipped weights.
"""
import glob
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
sys.path.insert(0, ROOT)
for name in ("soundfile", "librosa", "librosa.filters"):
    m = types.ModuleType(name)
    if name == "librosa.filters":
        m.mel = None
    sys.modules.setdefault(name, m)
sys.path.insert(0, os.path.join(REF, "code"))
import model as refmodel  # noqa: E402

import ntm_b200  # noqa: E402,F401
from ntm_b200 import signals  # noqa: E402
from oracle import c_oracle, ref_torch, save_golden  # noqa: E402

torch.set_num_threads(1)
SIGS = ("sweepnoise_lo", "sine")
T = 4096


def main():
    dirs = sorted(os.path.basename(p) for p in glob.glob(os.path.join(REF, "weights", "*_BEST")))
    assert len(dirs) == 12, dirs
    out = {"n": len(dirs), "signals": np.array(SIGS), "T": T, "max_delay": signals.DELAY_MAX}
    for i, dirname in enumerate(dirs):
        kind = "DiffDelGRU" if dirname.startswith("DiffDelGRU") else "GRU"
        sd = torch.load(os.path.join(REF, "weights", dirname, "best.pth"), map_location="cpu", weights_only=True)
        out[f"kind{i}"], out[f"dir{i}"] = kind, dirname
        for k, v in sd.items():
            out[f"w{i}_{k}"] = v.numpy()
        w = c_oracle.GruWeights.from_state_dict(sd)
        net, net64 = ref_torch.RefNet(sd), ref_torch.RefNet(sd, torch.float64)
        with torch.inference_mode():
            if kind == "GRU":
                m = refmodel.RNN(1, 64, 1, False)
                m.load_state_dict(sd, strict=True)
                m.initialize_hidden(); m.warm_start()
            else:
                m = refmodel.DiffDelRNN(1, 64, 1, False, max_delay=signals.DELAY_MAX)
                m.load_state_dict(sd, strict=True)
                m.initialize_hidden(1, signals.DELAY_MAX); m.warm_start()
                out[f"hist_warm{i}"] = m.diffdel.buffer.numpy().reshape(-1).copy()
            out[f"h_warm{i}"] = m.hidden.numpy().reshape(-1).copy()
            for j, sig in enumerate(SIGS):
                x = signals.signal(sig, T, seed=100 + j)
                xt = torch.from_numpy(x).reshape(1, 1, -1)
                if kind == "GRU":
                    y = m.predict(xt).numpy().reshape(-1)
                    yp, _ = net.predict(xt)
                    assert np.array_equal(y, yp.numpy().reshape(-1)), "ref_torch != reference"
                    y64 = net64.predict(xt)[0].numpy().reshape(-1)
                    yc, _ = c_oracle.rnn_predict(w, x.reshape(1, -1))
                else:
                    d = signals.delay_trajectory(1, T, first_stream=j)[0]
                    dtt = torch.from_numpy(d).reshape(1, 1, -1)
                    y, pre = m.predict(xt, dtt)
                    y, pre = y.numpy().reshape(-1), pre.numpy().reshape(-1)
                    yp, prep, _, _ = ref_torch.diffdel_predict(net, xt, dtt, signals.DELAY_MAX)
                    assert np.array_equal(y, yp.numpy().reshape(-1)) and np.array_equal(pre, prep.numpy().reshape(-1))
                    y64 = net64.predict(xt)[0].numpy().reshape(-1)             # ground truth of pre_d
                    yc, prec, _, _ = c_oracle.diffdel_predict(w, x.reshape(1, -1), d.reshape(1, -1), signals.DELAY_MAX)
                    out[f"pre{i}_{sig}"] = pre
                    out[f"d_{sig}"] = d
                floor = float(np.max(np.abs((pre if kind != "GRU" else y) - y64)))
                cerr = float(np.max(np.abs(yc.reshape(-1) - y)))
                print(f"{i:2d} {kind:10s} {sig:14s} floor={floor:.2e} C-f32 vs ref={cerr:.2e}  {dirname}")
                # a checkpoint whose own fp32-vs-fp64 floor is large on a signal is chaotic there: any summation order drifts
                assert cerr < max(5e-6, 4.0 * floor), (cerr, floor)
                out[f"x_{sig}"] = x
                out[f"y{i}_{sig}"] = y
                out[f"floor{i}_{sig}"] = floor
    p = os.path.join(ROOT, "tests", "golden", "golden_best12.npz")
    print("written", save_golden(p, **out))


if __name__ == "__main__":
    main()
