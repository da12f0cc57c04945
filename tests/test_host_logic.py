"""Host-side mirror of the reference interface (code/model.py): constructor arguments, attributes, state_dict
compatibility and the quirks of SURVEY.md section 9.3 that do not need a GPU."""
import copy
import os

import numpy as np
import pytest
import torch

from conftest import load_ckpt, load_golden
import ntm_b200
from ntm_b200 import DiffDelRNN, RNN, TimeVaryingDelayLine, signals


def test_rnn_ctor_and_state_dict_keys():
    m = RNN(input_size=1, hidden_size=64, output_size=1, skip=False)
    assert (m.input_size, m.hidden_size, m.output_size, m.skip, m.hidden) == (1, 64, 1, False, None)
    assert list(m.state_dict().keys()) == ["GRU.weight_ih_l0", "GRU.weight_hh_l0", "GRU.bias_ih_l0",
                                           "GRU.bias_hh_l0", "output.weight", "output.bias"]
    m.load_state_dict(load_ckpt("cfg1"), strict=True)
    m.load_state_dict(load_ckpt("cfg2"), strict=True)
    assert RNN().hidden_size == 8                      # reference default (code/model.py:22)


def test_diffdel_ctor_and_state_dict_keys():
    m = DiffDelRNN(input_size=1, hidden_size=64, output_size=1, skip=False, max_delay=364)
    assert "output.bias" not in m.state_dict() and not any("buffer" in k for k in m.state_dict())
    m.load_state_dict(load_ckpt("cfg3"), strict=True)
    # fresh model: batch-2 history of length max_delay+1 (SURVEY 9.3#2, code/model.py:370,375)
    assert tuple(m.diffdel.buffer.shape) == (2, 1, 365) and m.diffdel.max_delay == 365
    m.initialize_hidden(5, 100)
    assert tuple(m.diffdel.buffer.shape) == (5, 1, 101) and m.hidden is None
    with pytest.raises(RuntimeError):
        m.load_state_dict(load_ckpt("cfg1"), strict=True)      # GRU checkpoint has a head bias


def test_delay_line_attrs():
    d = TimeVaryingDelayLine(max_delay=40, channels=1)
    assert d.max_delay == 40 and tuple(d.buffer.shape) == (2, 1, 40) and len(d.state_dict()) == 0
    d.init_buffer(3, 17)
    assert d.max_delay == 17 and tuple(d.buffer.shape) == (3, 1, 17) and float(d.buffer.abs().sum()) == 0.0
    d.init_buffer(4)                                   # apply_delay's one-argument call (code/test-model.py:268)
    assert tuple(d.buffer.shape) == (4, 1, 17)
    d.detach_buffer()


def test_module_copies_and_moves():
    m = RNN(1, 64, 1, False)
    m2 = copy.deepcopy(m)
    assert m2._engine is not m._engine and m2._engine.handle is None
    m.double().float().eval()


def test_all_shipped_checkpoints_load_strict():
    """Every checkpoint whose state_dict the repository stores as the reference shipped it: the twelve `_BEST` runs
    (golden set golden_best12, oracle/make_golden_best.py), keys and shapes exactly as in best.pth; the class and the
    hidden size come from the directory name, like code/test-model.py's construction block."""
    import re
    g = load_golden("golden_best12")
    kinds = set()
    for i in range(int(g["n"])):
        name, pre = str(g[f"dir{i}"]), f"w{i}_"
        sd = {k[len(pre):]: torch.from_numpy(g[k]) for k in g.files if k.startswith(pre)}
        hs = int(re.search(r"-HS\[(\d+)\]-", name).group(1))
        cls = RNN if name.split("-")[0] == "GRU" else DiffDelRNN
        cls(1, hs, 1, False).load_state_dict(sd, strict=True)
        kinds.add(cls)
    assert int(g["n"]) == 12 and kinds == {RNN, DiffDelRNN}


def test_signals_are_seeded():
    a = signals.stream_batch(8, 4096)
    b = signals.stream_batch(8, 4096)
    assert np.array_equal(a, b) and a.dtype == np.float32
    assert np.array_equal(signals.stream_batch(4, 4096, first_stream=4), a[4:])
    assert np.abs(a).max() <= 0.75
    d = signals.delay_trajectory(2, 48000)
    assert d.max() <= 292.0 + 1e-3 and d.min() >= 188.0 - 1e-3 and signals.DELAY_MAX == 365


def test_hidden_state_padding_helpers():
    """Hidden sizes below 64 run zero-padded in the 64-unit kernels: `self.hidden` keeps the reference's (1, B, H) shape, the engine sees
    (1, B, 64) with zeros behind (model.py: _to_engine / _from_engine); the goldens of tests/test_hidden_sizes.py load strictly."""
    for H in (1, 8, 16, 32, 63, 64):
        m = RNN(1, H, 1, False)
        h = torch.arange(3 * H, dtype=torch.float32).reshape(1, 3, H)
        e = m._to_engine(h)
        assert tuple(e.shape) == (1, 3, 64) and torch.equal(e[..., :H], h) and float(e[..., H:].abs().sum()) == 0.0
        back = m._from_engine(e)
        assert tuple(back.shape) == (1, 3, H) and torch.equal(back, h) and back.is_contiguous()
        assert m._to_engine(None) is None and m._from_engine(None) is None
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_hs.npz"))
    for i in range(int(g["n"])):
        pre = f"w{i}_"
        sd = {k[len(pre):]: torch.from_numpy(g[k]) for k in g.files if k.startswith(pre)}
        H = int(g[f"H{i}"])
        m = RNN(1, H, 1, bool(g[f"skip{i}"])) if str(g[f"kind{i}"]) == "GRU" else DiffDelRNN(1, H, 1, False, max_delay=int(g["max_delay"]))
        m.load_state_dict(sd, strict=True)
        assert m.GRU.weight_hh_l0.shape == (3 * H, H)
