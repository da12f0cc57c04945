"""Real-time block mode of the full tape model (DiffDelRNN: GRU + head + wow/flutter delay line): the resident server
(ntm_rt_diffdel_*, RealtimeDelayStream) and the device-side DelayBlockStream.  Bar: bit-identical to one long
DiffDelRNN.forward over the concatenated signal from the same state and delay history -- y, pre_d, the final state and
the rolled history -- plus the delay assert, argument limits and the idle timeout.  Every stream is closed in a
`finally`, so no resident kernel outlives its test.  The last two tests cover both kinds of stream: the RNN's and the
DiffDelRNN's share their C-side core and their Python classes."""
import ctypes
import time

import numpy as np
import pytest
import torch

from conftest import load_ckpt
from ntm_b200 import RNN, DiffDelRNN, lib, signals

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TC_MODES = ["f16", "bf16", "tf32", "f16x3"]
# largest history length D the server's on-chip ring takes, by streams (include/ntm_b200.h)
D_LIMIT = {1: 32639, 2: 16255, 3: 8063, 4: 8063}


def warmed(B, max_d, mode="f16", skip=False):
    """cfg 3 model after initialize_hidden(1, max_d) + warm_start(), its state and history broadcast to B streams
    (predict() semantics); the history length is D = max_d + 1."""
    m = DiffDelRNN(input_size=1, hidden_size=64, output_size=1, skip=skip, max_delay=max_d).to(DEV)
    m.load_state_dict(load_ckpt("cfg3"))
    m.mode = mode
    m.initialize_hidden(1, max_d)
    m.warm_start()
    return m, m.hidden.expand(1, B, 64).contiguous(), m.diffdel.buffer.expand(B, 1, -1).contiguous()


def signals_for(B, N, D):
    """Host (B, N) input and a wow/flutter trajectory scaled so that its largest delay comes close to D."""
    x = torch.from_numpy(signals.stream_batch(B, N))
    d = torch.from_numpy(signals.delay_trajectory(B, N) * np.float32((D - 0.5) / 292.0))
    return x.contiguous(), d.contiguous()


def one_call(m, h, hist, x, d):
    """Reference: one DiffDelRNN.forward over the whole signal -> host y, pre_d, state, history."""
    B = x.shape[0]
    m.hidden, m.diffdel.buffer = h.clone(), hist.clone()
    y, pre = m(x.to(DEV).reshape(B, 1, -1), d.to(DEV).reshape(B, 1, -1))
    return y.cpu().reshape(B, -1), pre.cpu().reshape(B, -1), m.hidden.cpu(), m.diffdel.buffer.cpu()


def run_server(m, h, hist, x, d, T):
    B, N = x.shape
    m.hidden, m.diffdel.buffer = h.clone(), hist.clone()
    n0 = lib.query(lib.Q_KERNEL_LAUNCHES)
    rt = m.realtime_stream(B, T)
    try:
        ys, ps = [], []
        for k in range(N // T):
            y, p = rt.process(x[:, k * T:(k + 1) * T].contiguous(), d[:, k * T:(k + 1) * T].contiguous())
            ys.append(y.clone())
            ps.append(p.clone())
    finally:
        h_out, hist_out = rt.close()
    assert lib.query(lib.Q_KERNEL_LAUNCHES) == n0 + 1            # ONE launch for the whole stream
    return torch.cat(ys, 1), torch.cat(ps, 1), h_out.cpu(), hist_out.cpu()


def assert_same(got, ref):
    for g, r, name in zip(got, ref, ("y", "pre_d", "hidden", "delay history")):
        assert g.shape == r.shape and torch.equal(g, r), name


@pytest.mark.parametrize("skip", [False, True])
@pytest.mark.parametrize("mode", TC_MODES)
@pytest.mark.parametrize("T", [1, 33, 64, 256])
@pytest.mark.parametrize("B", [1, 3, 4])
def test_realtime_delay_stream_equals_one_call(B, T, mode, skip):
    max_d = signals.DELAY_MAX
    N = T * max(3, 1100 // T)
    with torch.inference_mode():
        m, h, hist = warmed(B, max_d, mode, skip)
        x, d = signals_for(B, N, max_d + 1)
        ref = one_call(m, h, hist, x, d)
        got = run_server(m, h, hist, x, d, T)
    assert_same(got, ref)


@pytest.mark.parametrize("B,T,max_d,nblk", [
    (1, 64, 20, 20),                   # D < block_len
    (3, 256, 16, 6),
    (2, 64, 3000, 10),                 # D > total length: the history is still mostly the one carried in
    (1, 64, D_LIMIT[1] - 1, 600),      # D at the on-chip limit; the stream outruns the ring several times
    (2, 128, D_LIMIT[2] - 1, 140),
    (4, 256, D_LIMIT[4] - 1, 40),
])
def test_realtime_delay_stream_history_lengths(B, T, max_d, nblk):
    with torch.inference_mode():
        m, h, hist = warmed(B, max_d)
        hist = hist + torch.from_numpy(signals.stream_batch(B, max_d + 1)).to(DEV).reshape(B, 1, -1)   # a history to read
        x, d = signals_for(B, T * nblk, max_d + 1)
        ref = one_call(m, h, hist, x, d)
        got = run_server(m, h, hist, x, d, T)
    assert_same(got, ref)


@pytest.mark.parametrize("mode", ["fp32", "f16", "f16x3"])
@pytest.mark.parametrize("B,T", [(1, 64), (3, 100)])
def test_delay_block_stream_equals_one_call(B, T, mode):
    N = T * 12
    with torch.inference_mode():
        m, h, hist = warmed(B, signals.DELAY_MAX, mode)
        x, d = signals_for(B, N, signals.DELAY_MAX + 1)
        ref = one_call(m, h, hist, x, d)
        m.hidden, m.diffdel.buffer = h.clone(), hist.clone()
        bs = m.block_stream(B, T)
        xd, dd = x.to(DEV).reshape(B, 1, -1), d.to(DEV).reshape(B, 1, -1)
        out, out_pre = torch.empty((B, 1, T), device=DEV), torch.empty((B, 1, T), device=DEV)
        ys, ps = [], []
        for k in range(N // T):
            sl = slice(k * T, (k + 1) * T)
            y, p = bs.process(xd[:, :, sl], dd[:, :, sl], *((out, out_pre) if k % 2 else ()))
            assert (y is out) == bool(k % 2)
            ys.append(y.clone())
            ps.append(p.clone())
        h_out, hist_out = bs.close()
        assert m.hidden is h_out and m.diffdel.buffer is hist_out
        got = (torch.cat(ys, 2).cpu().reshape(B, -1), torch.cat(ps, 2).cpu().reshape(B, -1), h_out.cpu(), hist_out.cpu())
    assert_same(got, ref)


@pytest.mark.parametrize("kind", ["server", "block"])
def test_refused_delay_block_changes_nothing(kind):
    B, T, max_d = 2, 64, signals.DELAY_MAX
    with torch.inference_mode():
        m, h, hist = warmed(B, max_d)
        x, d = signals_for(B, T * 6, max_d + 1)
        ref = one_call(m, h, hist, x, d)
        bad_far, bad_nan = d[:, :T].clone(), d[:, :T].clone()
        bad_far[1, 17] = max_d + 1.5                   # d > D
        bad_nan[0, 3] = float("nan")
        m.hidden, m.diffdel.buffer = h.clone(), hist.clone()
        ys, ps = [], []
        if kind == "server":
            st = m.realtime_stream(B, T)
            try:
                for k in range(6):
                    if k in (2, 4):
                        with pytest.raises(AssertionError, match="delay"):
                            st.process(x[:, :T].clone(), bad_far if k == 2 else bad_nan)
                    y, p = st.process(x[:, k * T:(k + 1) * T].contiguous(), d[:, k * T:(k + 1) * T].contiguous())
                    ys.append(y.clone())
                    ps.append(p.clone())
            finally:
                h_out, hist_out = st.close()
            got = (torch.cat(ys, 1), torch.cat(ps, 1), h_out.cpu(), hist_out.cpu())
        else:
            bs = m.block_stream(B, T)
            for k in range(6):
                if k in (2, 4):
                    bad = (bad_far if k == 2 else bad_nan).to(DEV).reshape(B, 1, T)
                    with pytest.raises(AssertionError, match="delay"):
                        bs.process(torch.zeros((B, 1, T), device=DEV), bad)
                y, p = bs.process(x[:, k * T:(k + 1) * T].to(DEV).reshape(B, 1, T), d[:, k * T:(k + 1) * T].to(DEV).reshape(B, 1, T))
                ys.append(y.clone())
                ps.append(p.clone())
            h_out, hist_out = bs.close()
            got = (torch.cat(ys, 2).cpu().reshape(B, -1), torch.cat(ps, 2).cpu().reshape(B, -1), h_out.cpu(), hist_out.cpu())
    assert_same(got, ref)


def test_realtime_delay_stream_check_off_passes_the_block():
    """check_delay = False: the block is handed over as is (the reference without its assert)."""
    with torch.inference_mode():
        m, _, _ = warmed(1, 40)
        m.diffdel.check_delay = False
        st = m.realtime_stream(1, 16)
        try:
            y, p = st.process(torch.zeros(1, 16), torch.full((1, 16), 100.0))
            assert bool(torch.isfinite(y).all()) and bool(torch.isfinite(p).all())
        finally:
            st.close()


def test_realtime_delay_stream_limits_and_idle_timeout():
    with torch.inference_mode():
        m, _, _ = warmed(1, signals.DELAY_MAX)
        for B, T in ((5, 64), (1, 257)):
            m.initialize_hidden(B, signals.DELAY_MAX)
            with pytest.raises(RuntimeError, match="invalid"):
                m.realtime_stream(B, T)
        for B in (1, 2, 4):
            m.initialize_hidden(B, D_LIMIT[B])                   # D = limit + 1
            with pytest.raises(RuntimeError, match="unsupported"):
                m.realtime_stream(B, 64)
        m.initialize_hidden(1, signals.DELAY_MAX)
        m.mode = "fp32"
        with pytest.raises(RuntimeError, match="unsupported"):
            m.realtime_stream(1, 64)
        m.mode = "f16"
        st = m.realtime_stream(1, 64)
        try:
            y, _ = st.process(np.zeros((1, 1, 64), np.float32), np.zeros((1, 1, 64), np.float32))
            assert tuple(y.shape) == (1, 1, 64)
            with pytest.raises(RuntimeError, match="HOST blocks"):
                st.process(torch.zeros(1, 64), torch.zeros(1, 63))
        finally:
            st.close()
        with pytest.raises(RuntimeError, match="closed"):
            st.process(torch.zeros(1, 64), torch.zeros(1, 64))
        with pytest.raises(RuntimeError, match="closed"):
            st.step()
        st = m.realtime_stream(1, 64, idle_timeout_ms=200)
        try:
            st.process(torch.zeros(1, 64), torch.zeros(1, 64))
            time.sleep(0.8)                                      # the server leaves by itself ...
            with pytest.raises(RuntimeError, match="closed"):
                st.process(torch.zeros(1, 64), torch.zeros(1, 64))   # ... and the next block reports it instead of hanging
        finally:
            st.close()
        torch.cuda.synchronize()


def test_cross_kind_calls_are_refused():
    """ntm_rt_process / ntm_rt_close on a DiffDelRNN stream and ntm_rt_diffdel_process / _close on an RNN stream return
    NTM_EINVAL and leave both streams open: they then process and close exactly as if the calls had not been made."""
    B, T, nblk = 2, 64, 4
    L = lib.load()

    def ptr(t):
        return ctypes.c_void_p(t.data_ptr())
    with torch.inference_mode():
        m, h, hist = warmed(B, signals.DELAY_MAX)
        x, d = signals_for(B, T * nblk, signals.DELAY_MAX + 1)
        ref = one_call(m, h, hist, x, d)
        g = RNN(input_size=1, hidden_size=64, output_size=1).to(DEV)
        g.load_state_dict(load_ckpt("cfg1"))
        g.mode = "f16"
        g.hidden = h.clone()
        gref = (g(x.to(DEV).reshape(B, 1, -1)).cpu().reshape(B, -1), g.hidden.cpu())
        g.hidden, m.hidden, m.diffdel.buffer = h.clone(), h.clone(), hist.clone()
        torch.cuda.synchronize()
        rt, rtd = g.realtime_stream(B, T), m.realtime_stream(B, T)
        try:
            blk, out = torch.zeros(B, T), torch.empty(B, T)
            assert L.ntm_rt_process(rtd._rt, ptr(blk), ptr(out)) == -1
            assert L.ntm_rt_close(rtd._rt, None) == -1
            assert L.ntm_rt_diffdel_process(rt._rt, ptr(blk), ptr(blk), ptr(out), None) == -1
            assert L.ntm_rt_diffdel_close(rt._rt, None, None) == -1
            ys, yds, pds = [], [], []
            for k in range(nblk):
                xb, db = x[:, k * T:(k + 1) * T].contiguous(), d[:, k * T:(k + 1) * T].contiguous()
                ys.append(rt.process(xb).clone())
                y, p = rtd.process(xb, db)
                yds.append(y.clone())
                pds.append(p.clone())
        finally:
            h_g = rt.close().cpu()
            h_m, hist_m = rtd.close()
    assert torch.equal(torch.cat(ys, 1), gref[0]) and torch.equal(h_g, gref[1])
    assert_same((torch.cat(yds, 1), torch.cat(pds, 1), h_m.cpu(), hist_m.cpu()), ref)


@pytest.mark.parametrize("kind", ["rnn", "diffdel"])
def test_block_stream_refuses_bad_blocks_and_outputs(kind):
    """A caller's output that is too short, has the wrong shape, lives on the host or has another dtype, and an input
    block with two channels, raise before anything is written: the outputs keep their contents, and the stream continues
    exactly like one that never saw the bad calls."""
    B, T = 2, 64
    with torch.inference_mode():
        if kind == "rnn":
            m = RNN(input_size=1, hidden_size=64, output_size=1).to(DEV)
            m.load_state_dict(load_ckpt("cfg1"))
            m.mode = "f16"
            m.initialize_hidden()
        else:
            m, _, _ = warmed(B, signals.DELAY_MAX)
            m.initialize_hidden(B, signals.DELAY_MAX)
        x = torch.from_numpy(signals.stream_batch(B, 2 * T)).to(DEV).reshape(B, 1, -1)
        d = torch.full_like(x, 3.5)

        def blocks(k):
            sl = slice(k * T, (k + 1) * T)
            return (x[:, :, sl],) if kind == "rnn" else (x[:, :, sl], d[:, :, sl])
        good, bad = m.block_stream(B, T), m.block_stream(B, T)
        outs = [torch.full((B, 1, T // 2), 7.0, device=DEV),                  # shorter than the block
                torch.full((B, 2, T), 7.0, device=DEV),                       # two channels
                torch.full((B + 1, 1, T), 7.0, device=DEV),                   # one stream too many
                torch.full((B, 1, T), 7.0),                                   # host
                torch.full((B, 1, T), 7.0, device=DEV, dtype=torch.float64)]
        for o in outs:
            before = o.clone()
            with pytest.raises(RuntimeError, match="^out: "):
                bad.process(*blocks(0), o)
            if kind == "diffdel":
                with pytest.raises(RuntimeError, match="^out_pre_d: "):
                    bad.process(*blocks(0), None, o)
            torch.cuda.synchronize()
            assert torch.equal(o, before)
        with pytest.raises(RuntimeError, match="^x: "):
            bad.process(torch.zeros((B, 2, T), device=DEV), *blocks(0)[1:])
        for k in range(2):
            want, got = good.process(*blocks(k)), bad.process(*blocks(k))
            if kind == "rnn":
                want, got = (want,), (got,)
            for w, g in zip(want, got):
                assert torch.equal(w, g)
