"""Real-time block mode with the resident server kernel (ntm_rt_*, BASELINE cfg 5): host blocks in, host blocks out, state
carried on chip.  Bar: bit-identical to one long forward call of the same streams (SURVEY.md section 9.3 #1: the
reference's block-wise and one-shot results are identical), final state handed back, idle timeout and argument errors."""
import time

import numpy as np
import pytest
import torch

from conftest import load_ckpt
from ntm_b200 import RNN, lib, signals

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def make(mode="f16", skip=False):
    m = RNN(input_size=1, hidden_size=64, output_size=1, skip=skip).to(DEV)
    m.load_state_dict(load_ckpt("cfg1"))
    m.mode = mode
    return m


@pytest.mark.parametrize("B,T,nblk,mode,skip", [(1, 64, 150, "f16", False), (3, 100, 20, "f16", True),
                                                 (4, 256, 8, "bf16", False), (1, 1, 100, "f16", False),
                                                 (2, 33, 30, "tf32", False)])
def test_realtime_stream_equals_one_call(B, T, nblk, mode, skip):
    m = make(mode, skip)
    xh = torch.from_numpy(signals.stream_batch(B, T * nblk)).contiguous()
    with torch.inference_mode():
        m.initialize_hidden()
        m.warm_start()
        hw = m.hidden.expand(1, B, 64).contiguous()
        m.hidden = hw.clone()
        yref = m(xh.to(DEV).reshape(B, 1, -1)).cpu().reshape(B, -1)
        href = m.hidden.cpu()
        torch.cuda.synchronize()
        m.hidden = hw.clone()
        n0 = lib.query(lib.Q_KERNEL_LAUNCHES)
        rt = m.realtime_stream(B, T)
        out = [rt.process(xh[:, k * T:(k + 1) * T].contiguous()).clone() for k in range(nblk)]
        h = rt.close().cpu()
        assert lib.query(lib.Q_KERNEL_LAUNCHES) == n0 + 1            # ONE launch for the whole stream
    assert torch.equal(torch.cat(out, 1), yref)
    assert torch.equal(h, href)


def test_realtime_stream_numpy_blocks_and_shapes():
    m = make()
    with torch.inference_mode():
        m.initialize_hidden()
        rt = m.realtime_stream(2, 16)
        y = rt.process(np.zeros((2, 1, 16), np.float32))
        assert tuple(y.shape) == (2, 1, 16) and bool(torch.isfinite(y).all())
        with pytest.raises(RuntimeError, match="HOST block"):
            rt.process(np.zeros((2, 15), np.float32))
        with pytest.raises(RuntimeError, match="HOST block"):
            rt.process(torch.zeros(2, 16, device=DEV))
        rt.close()
        with pytest.raises(RuntimeError, match="closed"):
            rt.process(np.zeros((2, 16), np.float32))
        with pytest.raises(RuntimeError, match="closed"):
            rt.step()


def test_realtime_stream_limits_and_idle_timeout():
    m = make()
    with torch.inference_mode():
        m.initialize_hidden()
        with pytest.raises(RuntimeError, match="invalid"):
            m.realtime_stream(5, 64)
        with pytest.raises(RuntimeError, match="invalid"):
            m.realtime_stream(1, 257)
        m.mode = "fp32"
        with pytest.raises(RuntimeError, match="unsupported"):
            m.realtime_stream(1, 64)
        m.mode = "f16"
        rt = m.realtime_stream(1, 64, idle_timeout_ms=200)
        rt.process(torch.zeros(1, 64))
        time.sleep(0.8)                                   # the server leaves by itself ...
        with pytest.raises(RuntimeError, match="closed"):
            rt.process(torch.zeros(1, 64))                # ... and the next block reports it instead of hanging
        rt.close()
        torch.cuda.synchronize()
