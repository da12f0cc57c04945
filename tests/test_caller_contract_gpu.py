"""SURVEY.md section 8 row a12: the drop-in classes driven the way the reference's caller code/test-model.py drives them.

The calls of its construction block (:192-247: the hidden size parsed from the checkpoint's directory name, the model built
with the script's INPUT_SIZE / OUTPUT_SIZE / SKIP, load_state_dict of best.pth, .to(device); a DiffDelGRU or an
ADD_DELAY delay line sized `int(1.25 * max_delay_s * fs)` from the dataset's delay analyser), its prediction branch
(:479-484, `model.predict(input[, d_traj])` inside torch.inference_mode()) and `apply_delay` (:259-290) -- restated here,
the import swap of INTEGRATION.md.  Golden values: what the reference's own RNN / DiffDelRNN.predict return on the same
inputs (tests/golden/golden_cfg{1,3}.npz, oracle/make_golden.py); the delay read is checked bit-exactly against the oracle.
Outputs must agree to the fp32-class tolerance (max-abs <= 1e-5).
"""
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLD, load_ckpt, load_golden
import ntm_b200
from ntm_b200 import signals
from oracle import c_oracle

pytestmark = pytest.mark.gpu
FS = 44100          # the reference's dataset rate (code/test-model.py:76)
TOL = 1e-5
DEV = torch.device("cuda")


def _build(tag, max_delay_s=0.0):
    """The construction block for one checkpoint (stored in tests/golden with its directory name)."""
    name = str(np.load(os.path.join(GOLD, f"ckpt_{tag}.npz"))["weights_dir"])
    hs = int(re.search(r"-HS\[(\d+)\]-", name).group(1))
    if name.split("-")[0] == "GRU":
        model = ntm_b200.RNN(input_size=1, hidden_size=hs, output_size=1, skip=False)
    else:
        model = ntm_b200.DiffDelRNN(input_size=1, hidden_size=hs, output_size=1, skip=False,
                                    max_delay=int(1.25 * max_delay_s * FS))
    model.load_state_dict(load_ckpt(tag))
    return model.to(DEV)


@pytest.mark.parametrize("mode", ["fp32", "f16x3"])
def test_gru_through_the_reference_caller_block(mode):
    g = load_golden("golden_cfg1")
    model = _build("cfg1")
    assert isinstance(model, ntm_b200.RNN) and model.hidden_size == 64
    model.mode = mode
    x = torch.from_numpy(g["x_sweepnoise_lo"]).reshape(1, 1, -1)
    with torch.inference_mode():                                            # how code/test-model.py:296 calls it
        output = model.predict(x.to(DEV))
    err = float(np.abs(output.cpu().numpy().reshape(-1) - g["y_sweepnoise_lo"]).max())
    assert err <= TOL, err


@pytest.mark.parametrize("mode", ["fp32", "f16x3"])
def test_diffdel_through_the_reference_caller_block(mode):
    """The caller sizes the delay line from the trajectory (not the checkpoint's 365 samples): same output."""
    g = load_golden("golden_cfg3")
    d = g["d_sweepnoise_lo"]
    max_delay_s = float(d.max()) / FS
    model = _build("cfg3", max_delay_s)
    assert isinstance(model, ntm_b200.DiffDelRNN) and model.max_delay == int(1.25 * max_delay_s * FS)
    assert model.max_delay != int(g["max_delay"])
    model.mode = mode
    x = torch.from_numpy(g["x_sweepnoise_lo"]).reshape(1, 1, -1)
    d_traj = torch.from_numpy(d).reshape(1, 1, -1)
    with torch.inference_mode():
        output, output_pre_d = model.predict(x.to(DEV), d_traj.to(DEV))
    assert float(np.abs(output_pre_d.cpu().numpy().reshape(-1) - g["pre_sweepnoise_lo"]).max()) <= TOL
    assert float(np.abs(output.cpu().numpy().reshape(-1) - g["y_sweepnoise_lo"]).max()) <= TOL


def test_apply_delay_block_with_the_drop_in_delay_line():
    """`apply_delay` (code/test-model.py:259-290, the ADD_DELAY scheme): 4096-sample segments with the history carried by the
    delay line object, `delay.init_buffer(output.shape[0])` with ONE argument (the reference's own class rejects that call:
    its init_buffer takes (N, max_d), code/model.py:326 -- SURVEY 8f rank 1).  Checked bit-exactly against the oracle's
    delay line."""
    B, T = 3, 10000
    d_n = signals.delay_trajectory(B, T)
    max_delay_s = float(d_n.max()) / FS
    delay = ntm_b200.TimeVaryingDelayLine(max_delay=int(1.25 * max_delay_s * FS))
    assert delay.max_delay == int(1.25 * max_delay_s * FS)
    out = torch.from_numpy(signals.stream_batch(B, T)).reshape(B, 1, T).to(DEV)
    d = torch.from_numpy(d_n).reshape(B, 1, T).to(DEV)
    with torch.inference_mode():
        delay.init_buffer(out.shape[0])
        y = torch.cat([delay(out[:, :, s:s + 4096], d[:, :, s:s + 4096]) for s in range(0, T, 4096)], -1)
    yo, _ = c_oracle.delay_forward(out.cpu().numpy()[:, 0], d_n, np.zeros((B, delay.max_delay), np.float32))
    assert np.array_equal(y.cpu().numpy()[:, 0], yo)
