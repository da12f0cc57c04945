#!/usr/bin/env python3
"""Generate tests/golden/*.npz from the REAL reference (imports /root/reference/code/model.py).

Run in the build container only (the GPU box has no /root/reference):
    python oracle/make_golden.py
What it writes (all float32 unless noted):
  tests/golden/ckpt_cfg{1,2,3}.npz    the three BASELINE.json checkpoints' state_dict tensors (data, not code)
  tests/golden/golden_cfg{1,2,3}.npz  per checkpoint: warm-start hidden state, and for each named signal the
                                      input, the reference RNN/DiffDelRNN.predict output (B=1, fp32), the
                                      float64 ground truth and the reference's own fp32-vs-fp64 floor
  tests/golden/golden_long_cfg1.npz   cfg 1 at full size (10 s @ 48 kHz): decimated output + statistics
  tests/golden/golden_delay.npz       TimeVaryingDelayLine cases (edge delays, T<D, warmup)
It also asserts that oracle/ref_torch.py is bit-identical to the imported reference classes and that
oracle/ntm_oracle.c agrees with them to float32 round-off, i.e. it pins the oracle.
"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
sys.path.insert(0, ROOT)

for name in ("soundfile", "librosa", "librosa.filters"):     # absent here; only plotting/IO helpers use them
    m = types.ModuleType(name)
    if name == "librosa.filters":
        m.mel = None
    sys.modules.setdefault(name, m)
sys.path.insert(0, os.path.join(REF, "code"))
import model as refmodel  # noqa: E402  (the reference)

import ntm_b200  # noqa: E402,F401
from ntm_b200 import signals  # noqa: E402
from oracle import c_oracle, ref_torch, save_golden  # noqa: E402

torch.set_num_threads(1)
GOLD = os.path.join(ROOT, "tests", "golden")
os.makedirs(GOLD, exist_ok=True)

CKPTS = {
    "cfg1": ("GRU", "GRU-HS[64]-L[ESR]-DS[ReelToReel_Dataset_MiniPulse100_CHOWTAPE]_BEST"),
    "cfg2": ("GRU", "GRU-HS[64]-L[DCPreESR]-DS[ReelToReel_Dataset_MiniPulse100_AKAI_IPS[7.5]_MAXELL]_BEST"),
    "cfg3": ("DiffDelGRU", "DiffDelGRU-HS[64]-L[DCPreESR]-DS[ReelToReel_Dataset_MiniPulse100_CHOWTAPE_WOWFLUTTER]_BEST"),
}
SIGNALS = ("sweepnoise", "sweepnoise_lo", "noise", "pulse", "sine", "sine1k", "silence")
T_SHORT = 8192


def load_sd(dirname):
    return torch.load(os.path.join(REF, "weights", dirname, "best.pth"), map_location="cpu", weights_only=True)


def main():
    for tag, (kind, dirname) in CKPTS.items():
        sd = load_sd(dirname)
        np.savez_compressed(os.path.join(GOLD, f"ckpt_{tag}.npz"), model_type=kind, weights_dir=dirname,
                            **{k: v.numpy() for k, v in sd.items()})
        w = c_oracle.GruWeights.from_state_dict(sd)
        net = ref_torch.RefNet(sd)
        net64 = ref_torch.RefNet(sd, torch.float64)
        out = {}
        if kind == "GRU":
            m = refmodel.RNN(1, 64, 1, False)
            m.load_state_dict(sd)
            m.eval()
            with torch.inference_mode():
                m.initialize_hidden()
                m.warm_start()
                out["h_warm"] = m.hidden.numpy().reshape(-1).copy()
                for i, sig in enumerate(SIGNALS):
                    x = signals.signal(sig, T_SHORT, seed=i)
                    xt = torch.from_numpy(x).reshape(1, 1, -1)
                    y = m.predict(xt).numpy().reshape(-1)
                    y_port, _ = net.predict(xt)
                    assert np.array_equal(y, y_port.numpy().reshape(-1)), "ref_torch != reference"
                    y64, _ = net64.predict(xt)
                    y64 = y64.numpy().reshape(-1)
                    yc, _ = c_oracle.rnn_predict(w, x.reshape(1, -1))
                    yc64, _ = c_oracle.rnn_predict(w, x.reshape(1, -1), f64=True)
                    floor = float(np.max(np.abs(y - y64)))
                    print(f"{tag} {sig:14s} floor(ref f32 vs f64)={floor:.2e}  C-f32 vs ref={np.max(np.abs(yc - y)):.2e}"
                          f"  C-f64 vs torch-f64={np.max(np.abs(yc64 - y64)):.2e}")
                    assert np.max(np.abs(yc64 - y64)) < 1e-9
                    out[f"x_{sig}"] = x
                    out[f"y_{sig}"] = y
                    out[f"y64_{sig}"] = y64
                    out[f"floor_{sig}"] = floor
                if tag == "cfg1":
                    # same checkpoint with skip=True (code/model.py:83-84)
                    ms = refmodel.RNN(1, 64, 1, True)
                    ms.load_state_dict(sd)
                    x = out["x_noise"]
                    out["y_skip_noise"] = ms.predict(torch.from_numpy(x).reshape(1, 1, -1)).numpy().reshape(-1)
        else:
            max_delay = signals.DELAY_MAX
            m = refmodel.DiffDelRNN(1, 64, 1, False, max_delay=max_delay)
            m.load_state_dict(sd)
            m.eval()
            with torch.inference_mode():
                m.initialize_hidden(1, max_delay)
                m.warm_start()
                out["h_warm"] = m.hidden.numpy().reshape(-1).copy()
                out["hist_warm"] = m.diffdel.buffer.numpy().reshape(-1).copy()
                out["max_delay"] = max_delay
                for i, sig in enumerate(SIGNALS):
                    x = signals.signal(sig, T_SHORT, seed=i)
                    d = signals.delay_trajectory(1, T_SHORT, first_stream=i)[0]
                    xt = torch.from_numpy(x).reshape(1, 1, -1)
                    dtt = torch.from_numpy(d).reshape(1, 1, -1)
                    y, pre = m.predict(xt, dtt)
                    y, pre = y.numpy().reshape(-1), pre.numpy().reshape(-1)
                    yp, prep, _, bufp = ref_torch.diffdel_predict(net, xt, dtt, max_delay)
                    assert np.array_equal(y, yp.numpy().reshape(-1)) and np.array_equal(pre, prep.numpy().reshape(-1))
                    assert np.array_equal(m.diffdel.buffer.numpy(), bufp.numpy())
                    yc, prec, _, histc = c_oracle.diffdel_predict(w, x.reshape(1, -1), d.reshape(1, -1), max_delay)
                    # delay stage alone is bit-exact given the same pre_d
                    yd, _ = c_oracle.delay_forward(pre.reshape(1, -1), d.reshape(1, -1),
                                                   out["hist_warm"].reshape(1, -1))
                    assert np.array_equal(yd.reshape(-1), y), "C delay line not bit-exact vs reference"
                    pre64, _ = net64.predict(xt)
                    floor = float(np.max(np.abs(pre - pre64.numpy().reshape(-1))))
                    print(f"{tag} {sig:14s} floor={floor:.2e} C-f32 vs ref: pre_d {np.max(np.abs(prec - pre)):.2e}"
                          f" y {np.max(np.abs(yc - y)):.2e}")
                    out[f"x_{sig}"] = x
                    out[f"d_{sig}"] = d
                    out[f"y_{sig}"] = y
                    out[f"pre_{sig}"] = pre
                    out[f"pre64_{sig}"] = pre64.numpy().reshape(-1)
                    out[f"floor_{sig}"] = floor
                    out[f"hist_{sig}"] = m.diffdel.buffer.numpy().reshape(-1).copy()
        save_golden(os.path.join(GOLD, f"golden_{tag}.npz"), **out)

    # ---- cfg 1 at full size: B=1, T=480000 (10 s @ 48 kHz), reference RNN.predict ----
    sd = load_sd(CKPTS["cfg1"][1])
    m = refmodel.RNN(1, 64, 1, False)
    m.load_state_dict(sd)
    T = 480000
    x = signals.signal("sweepnoise", T, seed=0)
    with torch.inference_mode():
        y = m.predict(torch.from_numpy(x).reshape(1, 1, -1)).numpy().reshape(-1)
        y64, _ = ref_torch.RefNet(sd, torch.float64).predict(torch.from_numpy(x).reshape(1, 1, -1))
    y64 = y64.numpy().reshape(-1)
    step = 97
    print(f"cfg1 long floor={np.max(np.abs(y - y64)):.2e}")
    np.savez_compressed(os.path.join(GOLD, "golden_long_cfg1.npz"), T=T, step=step, x_dec=x[::step], y_dec=y[::step],
                        y64_dec=y64[::step], y_head=y[:64], y_tail=y[-64:], y_sum=float(np.sum(y, dtype=np.float64)),
                        y_rms=float(np.sqrt(np.mean(y.astype(np.float64) ** 2))),
                        x_sum=float(np.sum(x, dtype=np.float64)), floor=float(np.max(np.abs(y - y64))),
                        esr_vs_f64=c_oracle.esr(y, y64.astype(np.float32)))

    # ---- delay line cases straight from the reference class ----
    rng = np.random.default_rng(5)
    cases = {}
    for name, (B, T, D, dkind) in {
        "frac": (3, 700, 37, "frac"), "integer": (2, 300, 16, "int"), "short_T": (2, 9, 40, "frac"),
        "edge": (1, 64, 8, "edge"), "negfrac": (1, 64, 8, "neg"),
    }.items():
        x = rng.standard_normal((B, 1, T)).astype(np.float32)
        if dkind == "frac":
            d = (rng.random((B, 1, T)) * D).astype(np.float32)
        elif dkind == "int":
            d = rng.integers(0, D + 1, (B, 1, T)).astype(np.float32)
        elif dkind == "edge":
            d = np.tile(np.array([0.0, D, D - 0.5, 0.5, 1.0, D - 1e-3, 1e-3, D / 2], np.float32), T // 8).reshape(B, 1, T)
        else:
            d = (-rng.random((B, 1, T))).astype(np.float32) * 0.999
        dl = refmodel.TimeVaryingDelayLine(max_delay=D)
        dl.buffer = torch.from_numpy(rng.standard_normal((B, 1, D)).astype(np.float32))
        hist0 = dl.buffer.numpy().copy()
        with torch.inference_mode():
            y1 = dl(torch.from_numpy(x), torch.from_numpy(d)).numpy()
            hist1 = dl.buffer.numpy().copy()
            y2 = dl(torch.from_numpy(x), torch.from_numpy(d), warmup=True).numpy()
            hist2 = dl.buffer.numpy().copy()
        for form in (False, True):
            yc, hc = c_oracle.delay_forward(x[:, 0], d[:, 0], hist0[:, 0], window=form)
            assert np.array_equal(yc, y1[:, 0]) and np.array_equal(hc, hist1[:, 0]), (name, form)
        yr, hr = ref_torch.delay_forward(torch.from_numpy(x), torch.from_numpy(d), torch.from_numpy(hist0))
        assert np.array_equal(yr.numpy(), y1) and np.array_equal(hr.numpy(), hist1)
        cases.update({f"{name}_x": x, f"{name}_d": d, f"{name}_hist0": hist0, f"{name}_y": y1, f"{name}_hist1": hist1,
                      f"{name}_ywarm": y2, f"{name}_hist2": hist2})
        print(f"delay case {name}: C oracle bit-exact")
    np.savez_compressed(os.path.join(GOLD, "golden_delay.npz"), **cases)
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    main()
