"""Tensor-core modes (warp-level mma.sync kernel csrc/gru_mma.cu, stream-major tcgen05 kernel csrc/gru_tcs.cu) through the C ABI.

Tolerance (BASELINE.json north_star): tf32/bf16-class MMA modes -- ESR of the output against the reference's fp32
output <= 1e-4 on numerically stable inputs.  "f16" rounds the operands to an 11-bit significand exactly like tf32 and
is held to the same bound; "bf16" (8-bit significand) is the opt-in low-accuracy mode and is only required to stay
finite and roughly right (SURVEY.md H2 measured ESR 1e-3..1e-2 for it).
Where a checkpoint amplifies round-off on a signal (reference fp32-vs-fp64 floor >= 5e-6: the cfg-1 pulse train) or the
target is (near) silence -- ESR of a ~1e-3 DC level -- the bound is on max-abs instead.
"""
import numpy as np
import pytest
import torch

from conftest import SIGNALS, load_ckpt, load_golden
from ntm_b200 import DiffDelRNN, RNN, lib, signals
from oracle import c_oracle, ref_torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ESR_TOL = 1e-4
TC_MODES = ("f16", "tf32")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def make_rnn(tag, mode, skip=False):
    m = RNN(input_size=1, hidden_size=64, output_size=1, skip=skip).to(DEV)
    m.load_state_dict(load_ckpt(tag))
    m.mode = mode
    return m


@pytest.fixture(autouse=True)
def _auto_tuning():
    lib.load().ntm_set_tuning(0, 0)
    yield
    lib.load().ntm_set_tuning(0, 0)


def test_mode_mask():
    mask = lib.query(lib.Q_MODE_MASK)
    for m in ("fp32", "tf32", "bf16", "f16", "f16x3"):
        assert mask >> lib.MODES[m] & 1
    assert lib.MODES["strict"] == lib.MODES["tf32x3"] == lib.MODES["f16x3"]
    m = make_rnn("cfg1", "f16")
    with pytest.raises(RuntimeError, match="unsupported"):
        x = torch.zeros(1, 1, 8, device=DEV)
        lib.check(lib.load().ntm_gru_forward(m._handle(torch.device(DEV)), 17, x.data_ptr(), 8, x.data_ptr(), 8, None,
                                             torch.zeros(64, device=DEV).data_ptr(), 1, 8, 0, None))


# kernel selectors (ntm_set_tuning): (n, 3) mma.sync kernel with n = 4, 8 streams per CTA, (4, 6) its lean 4-stream form
# (gru_mma4.cu: what cfg 2 / 3 / 5 run; f16 / bf16 / strict -- tf32 falls through to the general kernel), (tiles, 4) stream-major
# tcgen05 kernel
KERNELS = [(8, 3), (4, 3), (4, 6), (1, 4), (2, 4)]


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("mode", TC_MODES)
@pytest.mark.parametrize("tag", ["cfg1", "cfg2"])
def test_tc_predict_esr_vs_golden(tag, mode, kernel):
    lib.load().ntm_set_tuning(*kernel)
    m = make_rnn(tag, mode)
    g = load_golden(f"golden_{tag}")
    with torch.inference_mode():
        for sig in SIGNALS:
            y = m.predict(dev(g[f"x_{sig}"]).reshape(1, 1, -1)).cpu().numpy().reshape(-1)
            ref = g[f"y_{sig}"]
            stable = float(g[f"floor_{sig}"]) < 5e-6 and sig != "silence"
            if stable:
                assert c_oracle.esr(y, ref) <= ESR_TOL, (tag, mode, sig, c_oracle.esr(y, ref))
                assert np.max(np.abs(y - ref)) <= 5e-3, (tag, mode, sig)
            else:
                # the checkpoint amplifies round-off on this signal: the reference's own fp32-vs-fp64 distance (`floor`) is what
                # an operand unit round-off of 2^-24 grows to, so 11-bit operands (2^-11: 2^13 times coarser) may grow to
                # half of 2^13 floors (achieved: <= 1560 floors, profiles/r02_parity.json)
                bound = min(5e-2, 4096.0 * float(g[f"floor_{sig}"]))
                assert np.all(np.isfinite(y)) and np.max(np.abs(y - ref)) <= bound, (tag, mode, sig, np.max(np.abs(y - ref)), bound)


def test_bf16_is_finite_and_close():
    m = make_rnn("cfg2", "bf16")
    g = load_golden("golden_cfg2")
    with torch.inference_mode():
        y = m.predict(dev(g["x_sweepnoise_lo"]).reshape(1, 1, -1)).cpu().numpy().reshape(-1)
    assert np.all(np.isfinite(y)) and c_oracle.esr(y, g["y_sweepnoise_lo"]) <= 1e-2     # (achieved 4e-3: 8-bit significand)


@pytest.mark.parametrize("mode", TC_MODES)
def test_tc_batch_vs_oracle_and_kernel_selectors(mode):
    """64 mixed streams x 0.25 s against the torch restatement of the reference; every (streams per group,
    groups per CTA) variant of the kernel and a ragged batch give the same answer per stream."""
    m = make_rnn("cfg2", mode)
    B, T = 77, 12000
    xh = signals.stream_batch(B, T, dur=10.0)
    x = dev(xh).reshape(B, 1, T)
    yr, _ = ref_torch.RefNet(load_ckpt("cfg2")).predict(torch.from_numpy(xh).reshape(B, 1, T))
    with torch.inference_mode():
        y0 = m.predict(x)
        per_stream = ((y0.cpu() - yr) ** 2).sum(2) / ((yr ** 2).sum(2) + 1e-5)
        assert float(per_stream.max()) <= ESR_TOL
        assert abs(c_oracle.esr(y0.cpu().numpy(), yr.numpy())) <= ESR_TOL
        # g = 3: warp-level mma.sync kernel with n streams per CTA; g = 4: stream-major tcgen05 kernel, n tiles per CTA
        fam = {}
        for n, g in ((8, 3), (4, 3), (4, 6), (1, 4), (2, 4)):
            lib.load().ntm_set_tuning(n, g)
            y = m.predict(x)
            per_stream = ((y.cpu() - yr) ** 2).sum(2) / ((yr ** 2).sum(2) + 1e-5)
            assert float(per_stream.max()) <= ESR_TOL, (n, g)
            # same kernel family and form: same arithmetic (the 4-streams-per-CTA forms use their own reciprocals; the lean
            # kernel (4, 6) is the (4, 3) form bit for bit)
            first = fam.setdefault((3 if g == 6 else g, n == 4), y)
            assert float((y - first).abs().max()) <= 1e-6, (n, g)      # same kernel family: same arithmetic
            for b in (0, 31, 76):
                assert float((m.predict(x[b:b + 1]) - y[b:b + 1]).abs().max()) <= 1e-6


@pytest.mark.parametrize("kernel", [(0, 0)] + KERNELS)
@pytest.mark.parametrize("mode", TC_MODES + ("f16x3",))
def test_tc_segmentation_state_and_skip(mode, kernel):
    lib.load().ntm_set_tuning(*kernel)
    m = make_rnn("cfg1", mode)
    B, T = 5, 3000
    x = dev(signals.stream_batch(B, T)).reshape(B, 1, T)
    with torch.inference_mode():
        y_all = m.predict(x)
        h_all = m.hidden.clone()
        m.predict(x[:, :, :0])
        parts, s = [], 0
        for n in (64, 1, 31, 32, 33, 2000, 839):
            parts.append(m(x[:, :, s:s + n]))
            s += n
        assert s == T
        assert torch.equal(torch.cat(parts, 2), y_all) and torch.equal(m.hidden, h_all)
        ms = make_rnn("cfg1", mode, skip=True)
        assert torch.allclose(ms.predict(x), y_all + x, atol=1e-7, rtol=0)
        view = x[:, :, 7:1507]                               # unaligned, strided rows
        assert torch.equal(m.predict(view), m.predict(view.contiguous()))


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("mode", TC_MODES)
def test_tc_diffdel(mode, kernel):
    lib.load().ntm_set_tuning(*kernel)
    g = load_golden("golden_cfg3")
    D = int(g["max_delay"])
    m = DiffDelRNN(input_size=1, hidden_size=64, output_size=1, skip=False, max_delay=D).to(DEV)
    m.load_state_dict(load_ckpt("cfg3"))
    m.mode = mode
    with torch.inference_mode():
        for sig in ("sweepnoise", "noise", "sine"):
            x, d = dev(g[f"x_{sig}"]).reshape(1, 1, -1), dev(g[f"d_{sig}"]).reshape(1, 1, -1)
            y, pre = m.predict(x, d)
            y, pre = y.cpu().numpy().reshape(-1), pre.cpu().numpy().reshape(-1)
            assert c_oracle.esr(pre, g[f"pre_{sig}"]) <= ESR_TOL, (sig, c_oracle.esr(pre, g[f"pre_{sig}"]))
            assert c_oracle.esr(y, g[f"y_{sig}"]) <= ESR_TOL, (sig, c_oracle.esr(y, g[f"y_{sig}"]))
            # the fused delay read is bit-exact given the engine's own pre_d and warm history
            m.initialize_hidden(1, m.max_delay)
            m.warm_start()
            hist_w = m.diffdel.buffer.cpu().numpy().reshape(1, -1)
            yo, _ = c_oracle.delay_forward(pre.reshape(1, -1), g[f"d_{sig}"].reshape(1, -1), hist_w)
            assert np.array_equal(yo.reshape(-1), y), sig
        # batch + ragged segments with carried state and history
        B, T = 19, 4000
        x = dev(signals.stream_batch(B, T)).reshape(B, 1, T)
        d = dev(signals.delay_trajectory(B, T)).reshape(B, 1, T)
        y_all, p_all = m.predict(x, d)
        hist_all = m.diffdel.buffer.clone()
        m.predict(x[:, :, :0], d[:, :, :0])
        ys, ps, s = [], [], 0
        for n in (2048, 100, 1, 365, 1486):
            yy, pp = m(x[:, :, s:s + n], d[:, :, s:s + n])
            ys.append(yy)
            ps.append(pp)
            s += n
        assert s == T
        assert torch.equal(torch.cat(ps, 2), p_all) and torch.equal(torch.cat(ys, 2), y_all)
        assert torch.equal(m.diffdel.buffer, hist_all)


def test_tc_cfg2_width_and_host_pipeline():
    """1024 streams (cfg 2 width): sampled streams against the host oracle, split-batch checksum, host pipeline."""
    m = make_rnn("cfg2", "f16")
    B, T = 1024, 6000
    x = signals.stream_batch_device(B, T, DEV, dur=10.0).reshape(B, 1, T)
    with torch.inference_mode():
        y = m.predict(x)
        halves = torch.cat([m.predict(x[:512]), m.predict(x[512:])], 0)
        assert float((halves - y).abs().max()) <= 1e-6
        pick = [0, 1, 2, 3, 509, 1022, 1023]
        yr, _ = ref_torch.RefNet(load_ckpt("cfg2")).predict(x[pick].cpu())
        per_stream = ((y[pick].cpu() - yr) ** 2).sum(2) / ((yr ** 2).sum(2) + 1e-5)
        assert float(per_stream.max()) <= ESR_TOL
        xh = x[:16].cpu().pin_memory()
        assert torch.equal(m.predict_host(xh, chunk=2048), m.predict(x[:16]).cpu())


def test_stream_major_kernel_large_batch():
    """The stream-major tcgen05 kernel (csrc/gru_tcs.cu) at the width where the dispatcher picks it: several ragged
    128-stream tiles per CTA, sampled streams against the host oracle, agreement with the mma.sync kernel, tile
    independence (a stream's result does not depend on which tile or CTA it lands in), bf16 operands finite."""
    m = make_rnn("cfg2", "f16")
    sms = lib.query(lib.Q_SM_COUNT)
    B, T = 110 * sms + 37, 1500                    # automatic dispatch: >= 110 streams per SM
    x = signals.stream_batch_device(B, T, DEV, dur=10.0).reshape(B, 1, T)
    with torch.inference_mode():
        m.initialize_hidden()
        m.warm_start()                                # batch-1 warm state (mma.sync kernel), broadcast below
        hw = m.hidden.clone()

        def run(xb):
            m.hidden = hw.expand(1, xb.shape[0], 64).contiguous()
            return m(xb), m.hidden.clone()

        y, h = run(x)
        assert lib.query(lib.Q_LAST_KERNEL) == 3
        pick = [0, 1, 127, 128, 255, 256, 4097, B - 38, B - 1]
        yr, _ = ref_torch.RefNet(load_ckpt("cfg2")).predict(x[pick].cpu())
        per_stream = ((y[pick].cpu() - yr) ** 2).sum(2) / ((yr ** 2).sum(2) + 1e-5)
        assert float(per_stream.max()) <= ESR_TOL
        lib.load().ntm_set_tuning(8, 3)
        ym, _ = run(x[:2048])
        assert lib.query(lib.Q_LAST_KERNEL) == 1
        per_stream = ((y[:2048] - ym) ** 2).sum(2) / ((ym ** 2).sum(2) + 1e-5)
        assert float(per_stream.max()) <= ESR_TOL
        for tiles in (1, 2):                      # same arithmetic whatever the tiling / batch offset
            lib.load().ntm_set_tuning(tiles, 4)
            sub, hs = run(x[300:300 + 777])
            assert lib.query(lib.Q_LAST_KERNEL) == 3
            assert torch.equal(sub, y[300:300 + 777])
            assert torch.equal(hs[0], h[0, 300:300 + 777])
        lib.load().ntm_set_tuning(0, 0)
        m.mode = "bf16"
        yb, _ = run(x)
        assert lib.query(lib.Q_LAST_KERNEL) == 3 and bool(torch.isfinite(yb).all())
        assert float(((yb - y) ** 2).sum() / (y ** 2).sum()) <= 5e-2


def test_stream_major_dynamic_schedule_equals_static_schedule():
    """More tile groups than SMs with a partial last wave: the kernel pulls (group, time chunk) jobs from a queue and a
    group's state migrates between SMs through h_out.  Results and final state must equal the static schedule's bit
    for bit (tuning (tiles + 4, 4) forces the static schedule), for one and two tiles per CTA."""
    m = make_rnn("cfg2", "f16")
    sms = lib.query(lib.Q_SM_COUNT)
    with torch.inference_mode():
        m.initialize_hidden()
        m.warm_start()
        hw = m.hidden.clone()
        for tiles, B, T in ((2, sms * 256 + 300, 700), (1, sms * 128 + 1000, 900)):
            x = signals.stream_batch_device(B, T, DEV, dur=10.0).reshape(B, 1, T)
            outs = []
            for sel in (tiles, tiles + 4):                        # dynamic schedule, static schedule
                lib.load().ntm_set_tuning(sel, 4)
                m.hidden = hw.expand(1, B, 64).contiguous()
                outs.append((m(x), m.hidden.clone()))
                assert lib.query(lib.Q_LAST_KERNEL) == 3
            assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
            assert bool(torch.isfinite(outs[0][0]).all())
            del x, outs


def test_removed_kernel_selectors_are_rejected():
    """A tuning pair outside the table of include/ntm_b200.h fails the launch with "invalid argument" instead of running some
    other configuration; the pairs of the table still run the kernel they name."""
    L = lib.load()
    B, T = 8, 256
    x = torch.from_numpy(signals.stream_batch(B, T)).to(DEV).reshape(B, 1, T)
    cases = [("f16", (16, 3)),                          # 16 streams per CTA
             ("f16", (1 + 4 * (3 + 1), 4)),             # tcgen05 kernel variant 3
             ("fp32", (4, 0x104)),                      # MUFU activations of the fp32 kernel
             ("f16", (4, 2)), ("fp32", (8, 3)), ("fp32", (4, 2)), ("f16", (3, 4))]
    with torch.inference_mode():
        for mode, sel in cases:
            m = make_rnn("cfg2", mode)
            L.ntm_set_tuning(*sel)
            with pytest.raises(RuntimeError, match="invalid argument"):
                m.predict(x)
        kept = [("f16", (0, 0), 4), ("f16", (4, 3), 1), ("f16", (8, 3), 1), ("f16", (4, 6), 4), ("tf32", (4, 6), 1),
                ("f16", (1, 4), 3), ("f16", (2, 4), 3), ("f16", (5, 4), 3), ("f16", (6, 4), 3),
                ("fp32", (0, 0), 0), ("fp32", (8, 4), 0), ("fp32", (2, 2), 0), ("fp32", (0, 4), 0)]
        for mode, sel, kernel in kept:
            m = make_rnn("cfg2", mode)
            L.ntm_set_tuning(*sel)
            m.predict(x)
            assert lib.query(lib.Q_LAST_KERNEL) == kernel, (mode, sel)


def test_full_size_cfg2_properties():
    """BASELINE config 2 at FULL size (1024 streams x 60 s = 2.95e9 samples, tensor-core mode, the bench workload) through
    size-independent properties: causality / segmentation (the first second of the full run equals a one-second run, bit
    for bit), stream independence (sampled streams re-run alone give the same samples), two sampled streams against the
    host oracle over the first two seconds, everything finite, and the state equals the state of a chunked run."""
    m = make_rnn("cfg2", "f16")
    B, T, FS = 1024, 60 * 48000, 48000
    x = signals.stream_batch_device(B, T, DEV, dur=60.0).reshape(B, 1, T)
    with torch.inference_mode():
        y = m.predict(x)
        h_full = m.hidden.clone()
        assert lib.query(lib.Q_LAST_KERNEL) == 4       # cfg 2's width: the lean 4-stream mma.sync form
        assert bool(torch.isfinite(y[:, :, ::97]).all()) and bool(torch.isfinite(y[:, :, -4096:]).all())
        y1 = m.predict(x[:, :, :FS])
        assert torch.equal(y1, y[:, :, :FS])
        # chunked continuation reproduces the tail and the final state
        m.predict(x[:, :, :T - 3 * FS])
        tail = m(x[:, :, T - 3 * FS:])
        assert torch.equal(tail, y[:, :, T - 3 * FS:]) and torch.equal(m.hidden, h_full)
        pick = [0, 517, 1023]
        for b in pick:                                   # a stream alone (same 4-per-CTA form) == the stream in the batch
            assert torch.equal(m.predict(x[b:b + 1, :, :2 * FS]), y[b:b + 1, :, :2 * FS])
        yr, _ = ref_torch.RefNet(load_ckpt("cfg2")).predict(x[pick, :, :2 * FS].cpu())
        per_stream = ((y[pick, :, :2 * FS].cpu() - yr) ** 2).sum(2) / ((yr ** 2).sum(2) + 1e-5)
        assert float(per_stream.max()) <= ESR_TOL


@pytest.mark.parametrize("max_delay", [100, 364, 1000, 2000, 6000])
@pytest.mark.parametrize("mode,tuning,kernel", [("f16", (0, 0), 4), ("f16x3", (0, 0), 4), ("f16", (4, 3), 1),
                                                ("f16", (8, 3), 1), ("tf32", (0, 0), 1), ("fp32", (0, 0), 0)])
def test_tc_diffdel_delay_read_paths_bit_exact(mode, tuning, kernel, max_delay):
    """The fused delay read of the mma.sync kernels keeps the last D + 129 samples of pre_d per stream (D = max_delay + 1)
    in shared memory when they fit (D <= 1919 at four streams per CTA, D <= 895 at eight: max_delay = 1000 takes the ring
    in one and L2 in the other) and reads its taps back through L2 otherwise, as the fp32 kernel always does.  Every
    kernel and path must reproduce the oracle's delay line bit for bit on the engine's own pre_d and warm history, across
    segment boundaries; a warm-up segment returns pre_d itself and still rolls the history."""
    lib.load().ntm_set_tuning(*tuning)
    m = DiffDelRNN(input_size=1, hidden_size=64, output_size=1, skip=False, max_delay=max_delay).to(DEV)
    m.load_state_dict(load_ckpt("cfg3"))
    m.mode = mode
    B, T = 6, 9000
    rng = np.random.default_rng(max_delay)
    x = dev(signals.stream_batch(B, T)).reshape(B, 1, T)
    dn = (0.5 * max_delay * (1.0 + 0.9 * np.sin(np.arange(T)[None, :] / 700.0 + rng.uniform(0, 6, (B, 1))))).astype(np.float32)
    dn[:, ::50] = np.floor(dn[:, ::50])                   # integer delays too
    dn[0, :10] = 0.0
    d = dev(dn).reshape(B, 1, T)
    with torch.inference_mode():
        m.initialize_hidden(1, m.max_delay)                 # the reference's warm start is batch 1 (SURVEY 9.3 #3)
        m.warm_start()
        hist_w = m.diffdel.buffer.cpu().numpy().reshape(1, -1)
        m.hidden = m.hidden.expand(1, B, 64).contiguous()
        m.diffdel.buffer = m.diffdel.buffer.expand(B, 1, -1).contiguous()
        ys, ps, s = [], [], 0
        warm = slice(4032, 4532)                            # the warm-up segment
        for n in (31, 4000, 1, 500, 4468):
            yy, pp = m(x[:, :, s:s + n], d[:, :, s:s + n], warmup=s == warm.start)
            assert lib.query(lib.Q_LAST_KERNEL) == kernel
            ys.append(yy)
            ps.append(pp)
            s += n
        assert s == T
        y, pre = torch.cat(ys, 2).cpu().numpy().reshape(B, T), torch.cat(ps, 2).cpu().numpy().reshape(B, T)
        assert np.array_equal(y[:, warm], pre[:, warm])
        # the oracle runs over all of pre_d: the segments after the warm-up one read the history it rolled
        yo, ho = c_oracle.delay_forward(pre, dn, np.repeat(hist_w, B, 0))
        yo[:, warm] = pre[:, warm]
        assert np.array_equal(yo, y)
        assert np.array_equal(ho.reshape(B, -1), m.diffdel.buffer.cpu().numpy().reshape(B, -1))
        assert np.all(np.isfinite(y))
