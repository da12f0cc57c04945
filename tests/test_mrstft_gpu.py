"""On-device multi-resolution STFT loss (csrc/stft.cu, MultiResolutionSTFTLoss) against the float64 restatement of auraloss
in oracle/ref_mrstft.py.  Bound: |L - L64| <= max(2e-5 |L64|, 2 |L32 - L64|), L32 = the torch.stft restatement in
float32 (the engine computes in fp32 with double sums; a silent target or a 1e-3 signal puts the fp32 restatement itself
further from float64 than 2e-5)."""
import numpy as np
import pytest
import torch

from conftest import load_ckpt, load_golden
from ntm_b200 import MultiResolutionSTFTLoss, RNN, driver, lib, signals
from oracle import ref_mrstft

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NON_DEFAULT = dict(fft_sizes=(256, 4096), hop_sizes=(64, 1024), win_lengths=(256, 3000), w_sc=0.0, w_lin_mag=1.0)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(DEV)


def within_bound(got, o, t, **kw):
    l64 = ref_mrstft.mrstft_numpy(o, t, **kw)
    l32 = float(ref_mrstft.mrstft_torch(torch.from_numpy(np.float32(o)), torch.from_numpy(np.float32(t)), **kw))
    return abs(got - l64) <= max(2e-5 * abs(l64), 2 * abs(l32 - l64)), (got, l64, l32)


def cases():
    rng = np.random.default_rng(5)
    g = load_golden("golden_cfg2")
    y = g["y_sweepnoise"].astype(np.float32)
    out = {"gru_vs_perturbed": (y[None, None], (y + 0.01 * rng.standard_normal(y.shape))[None, None])}
    t = (0.2 * rng.standard_normal((1, 1, 20000))).astype(np.float32)
    out["dc_offset"] = (t + 0.05, t)
    t5 = (0.2 * rng.standard_normal((5, 1, 9000))).astype(np.float32)
    out["batch5"] = (t5 + (0.02 * rng.standard_normal(t5.shape)) * np.arange(1, 6)[:, None, None], t5)
    t = (0.2 * rng.standard_normal((2, 1, 1025))).astype(np.float32)
    out["T1025"] = (t + 0.02 * rng.standard_normal(t.shape), t)
    t = (0.2 * rng.standard_normal((2, 1, 48001))).astype(np.float32)            # 48001 = 1 mod 120, 240, 50
    out["T_off_hop"] = (t + 0.02 * rng.standard_normal(t.shape), t)
    out["silent_target"] = ((0.1 * rng.standard_normal((1, 1, 10000))), np.zeros((1, 1, 10000)))
    t = (1e-3 * rng.standard_normal((2, 1, 12000))).astype(np.float32)
    out["amplitude_1e-3"] = (t + 1e-4 * rng.standard_normal(t.shape), t)
    return {k: (np.float32(o), np.float32(t)) for k, (o, t) in out.items()}


CASES = cases()


@pytest.mark.parametrize("case", sorted(CASES))
def test_mrstft_vs_float64_oracle(case):
    o, t = CASES[case]
    n0 = lib.query(lib.Q_KERNEL_LAUNCHES)
    got = float(MultiResolutionSTFTLoss()(dev(o), dev(t)))
    assert lib.query(lib.Q_KERNEL_LAUNCHES) == n0 + 3                     # one launch per resolution
    ok, info = within_bound(got, o, t)
    assert ok, (case, info)


@pytest.mark.parametrize("case", ("batch5", "T_off_hop", "amplitude_1e-3"))
def test_mrstft_non_default_resolutions(case):
    o, t = CASES[case]
    n0 = lib.query(lib.Q_KERNEL_LAUNCHES)
    got = float(MultiResolutionSTFTLoss(**NON_DEFAULT)(dev(o), dev(t)))
    assert lib.query(lib.Q_KERNEL_LAUNCHES) == n0 + 2
    ok, info = within_bound(got, o, t, **NON_DEFAULT)
    assert ok, (case, info)


def test_batch_sc_is_one_ratio_and_per_example_follows_row_windows():
    o, t = CASES["batch5"]
    L = MultiResolutionSTFTLoss()
    whole = float(L(dev(o), dev(t)))
    per = L.per_example(dev(o), dev(t)).cpu().numpy()
    rows = [ref_mrstft.mrstft_numpy(o[i:i + 1], t[i:i + 1]) for i in range(5)]
    assert np.allclose(per, rows, rtol=2e-5)
    assert abs(whole - float(np.mean(per))) > 1e-3 * whole               # batch-norm SC != mean of per-row losses
    # ragged windows on a sliced [:, :, cut:] view: row b over [first[b], first[b] + count[b]) of the view
    B, T, cut = 6, 12000, 700
    rng = np.random.default_rng(9)
    tt = (0.2 * rng.standard_normal((B, 1, T))).astype(np.float32)
    oo = (tt + 0.03 * rng.standard_normal(tt.shape)).astype(np.float32)
    od, td = dev(oo)[:, :, cut:], dev(tt)[:, :, cut:]
    first = [0, 5, 1000, 3001, 200, 10000]
    count = [T - cut, 4001, 1025, 99999, 1024, 500]                      # row 3 is clipped, rows 4 and 5 are too short
    got = L.per_example(od, td, first, count).cpu().numpy()
    for b in range(B):
        n = min(count[b], T - cut - first[b])
        if n <= 1024:
            assert np.isnan(got[b]), (b, got[b])
            continue
        ref = float(L(od[b:b + 1, :, first[b]:first[b] + n], td[b:b + 1, :, first[b]:first[b] + n]))
        assert abs(got[b] - ref) <= 1e-6 * abs(ref), (b, got[b], ref)


def test_identical_signals_give_exactly_zero():
    t = 0.3 * torch.randn(4, 1, 30000, device=DEV)
    assert float(MultiResolutionSTFTLoss()(t, t)) == 0.0
    assert float(MultiResolutionSTFTLoss(**NON_DEFAULT)(t, t)) == 0.0
    assert torch.all(MultiResolutionSTFTLoss().per_example(t, t) == 0.0)


def test_full_width_1024_streams_x_480000():
    """The size auraloss cannot hold (its 512/50 spectrogram alone would be ~80 GB here): one call, sampled rows checked."""
    B, T = 1024, 480000
    g = torch.Generator(device=DEV).manual_seed(3)
    t = 0.2 * torch.randn(B, 1, T, device=DEV, generator=g)
    o = t + 0.02 * torch.randn(B, 1, T, device=DEV, generator=g)
    L = MultiResolutionSTFTLoss()
    per = L.per_example(o, t).cpu().numpy()
    whole = float(L(o, t))
    assert np.all(np.isfinite(per)) and np.isfinite(whole)
    for b in (0, 1, 137, 400, 511, 777, 1000, 1023):
        ok, info = within_bound(float(per[b]), o[b:b + 1].cpu().numpy(), t[b:b + 1].cpu().numpy())
        assert ok, (b, info)


def test_argument_errors():
    t = torch.zeros(2, 1, 4000, device=DEV)
    with pytest.raises(RuntimeError, match="no CPU path"):
        MultiResolutionSTFTLoss()(t.cpu(), t.cpu())
    with pytest.raises(RuntimeError, match="differ"):
        MultiResolutionSTFTLoss()(t, t[:, :, :3000])
    with pytest.raises(RuntimeError, match="reflect padding"):
        MultiResolutionSTFTLoss()(t[:, :, :1024], t[:, :, :1024])
    with pytest.raises(NotImplementedError):
        MultiResolutionSTFTLoss(fft_sizes=(1000,), hop_sizes=(100,), win_lengths=(600,))
    with pytest.raises(ValueError):
        MultiResolutionSTFTLoss(fft_sizes=(512,), hop_sizes=(50,), win_lengths=(600,))
    for kw in ({"w_phs": 1.0}, {"scale": "mel"}, {"n_bins": 64}, {"perceptual_weighting": True},
               {"scale_invariance": True}, {"window": "hamming_window"}, {"output": "full"}):
        with pytest.raises(NotImplementedError):
            MultiResolutionSTFTLoss(**kw)
    with pytest.raises(RuntimeError, match="power"):                     # the op checks what the class checks
        lib.ops().mrstft_sums_rows(t, t, None, None, [1000], [100], [600])


def test_batched_evaluator_mrstft(tmp_path):
    m = RNN(1, 64, 1, False).to(DEV)
    m.load_state_dict(load_ckpt("cfg2"))
    m.mode = "f16"
    rng = np.random.default_rng(4)
    lens = [5000, 7321, 2049, 9000, 1500]
    x = signals.stream_batch(len(lens), max(lens), dur=1.0)
    examples = []
    for i, n in enumerate(lens):
        pi, pt = str(tmp_path / f"in_{i}.wav"), str(tmp_path / f"tg_{i}.wav")
        driver.write_wav(pi, x[i, :n], 44100)
        driver.write_wav(pt, 0.9 * x[i, :n] + 0.01 * rng.standard_normal(n).astype(np.float32), 44100)
        examples.append({"input_file": pi, "target_file": pt})
    res = driver.BatchedEvaluator(m, max_streams=3, mrstft=True).run(examples, init_len=1024)
    L = MultiResolutionSTFTLoss()
    with torch.inference_mode():
        for ex, r in zip(examples, res):
            a, _ = driver.read_wav(ex["input_file"])
            t, _ = driver.read_wav(ex["target_file"])
            y = m.predict(torch.from_numpy(a[0]).to(DEV).reshape(1, 1, -1))
            if a.shape[1] - 1024 <= 1024:                                # the cut window is shorter than torch.stft accepts
                assert np.isnan(r["MR-STFT"])
                continue
            ref = float(L(y[:, :, 1024:], torch.from_numpy(t[0]).to(DEV).reshape(1, 1, -1)[:, :, 1024:]))
            assert r["MR-STFT"] == pytest.approx(ref, rel=1e-6)
    assert "MR-STFT" in driver.mean_losses(res[:4])
    plain = driver.BatchedEvaluator(m, max_streams=3).run(examples[:2], init_len=1024)
    assert all("MR-STFT" not in r for r in plain)
    assert "MR-STFT" not in driver.mean_losses(plain)
