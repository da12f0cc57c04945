"""Batched evaluation driver (neural-tape-modeling_b200/driver.py): .wav I/O on the CPU, batched prediction + losses on
the GPU equal to the reference-style one-file-at-a-time loop."""
import os
import struct
import wave

import numpy as np
import pytest
import torch

from conftest import load_ckpt
from ntm_b200 import DCPreESR, ESRLoss, RNN, driver, signals


def test_wav_roundtrip_float32_stereo_and_segments(tmp_path):
    rng = np.random.default_rng(0)
    a = rng.standard_normal((2, 1000)).astype(np.float32) * 3.0          # float files are NOT clipped / normalised
    p = str(tmp_path / "a.wav")
    driver.write_wav(p, a, 44100)
    info = driver.wav_info(p)
    assert (info["fs"], info["channels"], info["frames"], info["format"], info["bits"]) == (44100, 2, 1000, 3, 32)
    b, fs = driver.read_wav(p)
    assert fs == 44100 and np.array_equal(a, b)
    seg, _ = driver.read_wav(p, frame_offset=100, num_frames=250)
    assert np.array_equal(seg, a[:, 100:350])
    tail, _ = driver.read_wav(p, frame_offset=990, num_frames=500)
    assert np.array_equal(tail, a[:, 990:])
    driver.write_wav(p, a[0], 48000)                                      # mono from a 1-D array
    m, fs = driver.read_wav(p)
    assert fs == 48000 and m.shape == (1, 1000) and np.array_equal(m[0], a[0])


def test_wav_reads_pcm_files(tmp_path):
    p16 = str(tmp_path / "p16.wav")
    v = (np.arange(-5, 5) * 3000).astype("<i2")
    with wave.open(p16, "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(8000); w.writeframes(v.tobytes())
    a, fs = driver.read_wav(p16)
    assert fs == 8000 and np.allclose(a[0], v.astype(np.float32) / 32768.0)
    p24 = str(tmp_path / "p24.wav")
    vals = np.array([0, 1, -1, 8388607, -8388608, 123456, -654321], dtype=np.int32)
    raw = b"".join(struct.pack("<i", int(x))[:3] for x in vals)
    with wave.open(p24, "wb") as w:
        w.setnchannels(1); w.setsampwidth(3); w.setframerate(8000); w.writeframes(raw)
    a, _ = driver.read_wav(p24)
    assert np.allclose(a[0], vals.astype(np.float64) / 8388608.0)
    bad = str(tmp_path / "bad.wav")
    open(bad, "wb").write(b"RIFFxxxxWAVX")
    with pytest.raises(ValueError):
        driver.wav_info(bad)


@pytest.mark.gpu
def test_batched_evaluator_equals_one_file_at_a_time(tmp_path):
    dev = "cuda:0"
    m = RNN(1, 64, 1, False).to(dev)
    m.load_state_dict(load_ckpt("cfg2"))
    m.mode = "f16"
    rng = np.random.default_rng(1)
    lens = [5000, 7321, 2048, 9000, 1500, 6000, 4097]
    x = signals.stream_batch(len(lens), max(lens), dur=1.0)
    examples = []
    for i, n in enumerate(lens):
        xin = np.stack([x[i, :n], (np.arange(n) % 441 == 0).astype(np.float32)])       # audio + pulse track
        tgt = np.stack([0.9 * x[i, :n] + 0.01 * rng.standard_normal(n).astype(np.float32), xin[1]])
        pi, pt = str(tmp_path / f"in_{i}.wav"), str(tmp_path / f"tg_{i}.wav")
        driver.write_wav(pi, xin, 44100)
        driver.write_wav(pt, tgt, 44100)
        examples.append({"input_file": pi, "target_file": pt})
    examples.append({"input_file": examples[3]["input_file"], "target_file": examples[3]["target_file"],
                     "offset": 1000, "length": 3000})                                   # a dataset-style segment
    out_dir = str(tmp_path / "pred")
    res = driver.BatchedEvaluator(m, max_streams=3).run(examples, out_dir=out_dir, init_len=1024)
    assert len(res) == len(examples)
    with torch.inference_mode():
        for ex, r in zip(examples, res):
            a, fs = driver.read_wav(ex["input_file"], ex.get("offset", 0), ex.get("length", -1))
            t, _ = driver.read_wav(ex["target_file"], ex.get("offset", 0), ex.get("length", -1))
            xi = torch.from_numpy(a[0]).to(dev).reshape(1, 1, -1)
            y1 = m.predict(xi)                                                           # the reference's per-file call
            yw, fs2 = driver.read_wav(r["output_file"])
            assert fs2 == fs == 44100 and r["frames"] == a.shape[1]
            assert np.array_equal(yw[0], y1.cpu().numpy().reshape(-1))                   # batch == one file at a time
            td = torch.from_numpy(t[0]).to(dev).reshape(1, 1, -1)
            # (the loss sums are accumulated with atomics: equal up to the order of double additions)
            assert r["ESR"] == pytest.approx(float(ESRLoss()(y1[:, :, 1024:], td[:, :, 1024:])), rel=1e-6)
            assert r["DCPreESR"] == pytest.approx(float(DCPreESR()(y1[:, :, 1024:], td[:, :, 1024:])), rel=1e-6)
            assert np.isfinite(r["ESR"]) and r["ESR"] > 0.0 and np.isfinite(r["DCPreESR"])
    assert res[-1]["input_name"].endswith("_[1000:4000].wav")


def test_read_trajectory_dict_and_plain_files(tmp_path):
    t = np.linspace(0.004, 0.006, 1000)
    pd_, pp = str(tmp_path / "trajectory_1_.npy"), str(tmp_path / "plain.npy")
    np.save(pd_, {"delay_trajectory": t, "input_peaks": np.arange(3), "output_peaks": np.arange(3)})   # the dataset's format
    np.save(pp, t.astype(np.float32))
    assert np.array_equal(driver.read_trajectory(pd_), t)
    assert np.array_equal(driver.read_trajectory(pd_, 100, 250), t[100:350])
    assert np.allclose(driver.read_trajectory(pp, 990, 500), t[990:], rtol=1e-6)
    res = [{"ESR": 1.0, "DCPreESR": 4.0}, {"ESR": 3.0, "DCPreESR": 0.0}]
    assert driver.mean_losses(res) == {"ESR": 2.0, "DCPreESR": 2.0}
    assert driver.mean_losses([{"frames": 3}]) == {}


def _delay_examples(tmp_path, lens, fs=44100, seed=2):
    rng = np.random.default_rng(seed)
    x = signals.stream_batch(len(lens), max(lens), dur=1.0)
    d = signals.delay_trajectory(len(lens), max(lens)) / fs                 # the dataset stores SECONDS
    examples = []
    for i, n in enumerate(lens):
        pi, pt, pj = (str(tmp_path / f"input_{i}_.wav"), str(tmp_path / f"target_{i}_.wav"),
                      str(tmp_path / f"trajectory_{i}_.npy"))
        driver.write_wav(pi, np.stack([x[i, :n], (np.arange(n) % 441 == 0).astype(np.float32)]), fs)
        driver.write_wav(pt, 0.8 * x[i, :n] + 0.01 * rng.standard_normal(n).astype(np.float32), fs)
        np.save(pj, {"delay_trajectory": d[i, :n].astype(np.float64)})
        examples.append({"input_file": pi, "target_file": pt, "trajectory_file": pj})
    examples.append(dict(examples[1], offset=500, length=2500))             # a dataset-style segment of file 1
    return examples


def _traj_samples(ex, dev):
    a, fs = driver.read_wav(ex["input_file"], ex.get("offset", 0), ex.get("length", -1))
    t = driver.read_trajectory(ex["trajectory_file"], ex.get("offset", 0), ex.get("length", -1))
    return a, fs, (torch.from_numpy(t.astype(np.float32)) * float(fs)).to(dev).reshape(1, 1, -1)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "f16"])
def test_batched_evaluator_diffdel_equals_one_file_at_a_time(tmp_path, mode):
    from ntm_b200 import DiffDelRNN
    dev = "cuda:0"
    m = DiffDelRNN(1, 64, 1, False, max_delay=signals.DELAY_MAX).to(dev)
    m.load_state_dict(load_ckpt("cfg3"))
    m.mode = mode
    examples = _delay_examples(tmp_path, [5000, 7321, 2048, 6000, 4097])
    res = driver.BatchedEvaluator(m, max_streams=4).run(examples, out_dir=str(tmp_path / "pred"), init_len=512,
                                                        write_pre_d=True)
    with torch.inference_mode():
        for ex, r in zip(examples, res):
            a, fs, d = _traj_samples(ex, dev)
            t, _ = driver.read_wav(ex["target_file"], ex.get("offset", 0), ex.get("length", -1))
            y1, p1 = m.predict(torch.from_numpy(a[0]).to(dev).reshape(1, 1, -1), d)     # the reference's per-file call
            assert np.array_equal(driver.read_wav(r["output_file"])[0][0], y1.cpu().numpy().reshape(-1))
            assert np.array_equal(driver.read_wav(r["pre_d_file"])[0][0], p1.cpu().numpy().reshape(-1))
            td = torch.from_numpy(t[0]).to(dev).reshape(1, 1, -1)
            assert r["ESR"] == pytest.approx(float(ESRLoss()(y1[:, :, 512:], td[:, :, 512:])), rel=1e-6)
            assert r["DCPreESR"] == pytest.approx(float(DCPreESR()(y1[:, :, 512:], td[:, :, 512:])), rel=1e-6)
    means = driver.mean_losses(res)
    assert means["ESR"] == pytest.approx(np.mean([r["ESR"] for r in res]))


@pytest.mark.gpu
def test_batched_evaluator_add_delay_equals_reference_style_chunk_loop(tmp_path):
    """GRU + stand-alone delay line (ADD_DELAY): one batched call == per file, 4096-sample chunks with a carried buffer
    (apply_delay, code/test-model.py:259-290)."""
    from ntm_b200 import TimeVaryingDelayLine
    dev = "cuda:0"
    m = RNN(1, 64, 1, False).to(dev)
    m.load_state_dict(load_ckpt("cfg2"))
    examples = _delay_examples(tmp_path, [9000, 4096, 12345, 100])
    delay = TimeVaryingDelayLine(max_delay=signals.DELAY_MAX)
    res = driver.BatchedEvaluator(m, max_streams=3, delay=delay).run(examples, out_dir=str(tmp_path / "pred"),
                                                                     init_len=64)
    ref_delay = TimeVaryingDelayLine(max_delay=signals.DELAY_MAX)
    with torch.inference_mode():
        for ex, r in zip(examples, res):
            a, fs, d = _traj_samples(ex, dev)
            y = m.predict(torch.from_numpy(a[0]).to(dev).reshape(1, 1, -1))
            ref_delay.init_buffer(1)
            out = torch.cat([ref_delay(y[:, :, s:s + 4096], d[:, :, s:s + 4096]) for s in range(0, y.shape[-1], 4096)], -1)
            assert np.array_equal(driver.read_wav(r["output_file"])[0][0], out.cpu().numpy().reshape(-1))
            t, _ = driver.read_wav(ex["target_file"], ex.get("offset", 0), ex.get("length", -1))
            td = torch.from_numpy(t[0]).to(dev).reshape(1, 1, -1)
            assert r["ESR"] == pytest.approx(float(ESRLoss()(out[:, :, 64:], td[:, :, 64:])), rel=1e-6)
    with pytest.raises(ValueError):
        driver.BatchedEvaluator(__import__("ntm_b200").DiffDelRNN(1, 64, 1, False, max_delay=8), delay=delay)


def test_evaluator_trajectory_sources_and_errors(tmp_path):
    """Host logic of the delay modes (no GPU): seconds -> samples like `meta['delay_trajectory'].float() * fs`
    (code/test-model.py:349-351), file slicing by offset / length, and the error paths."""
    t = np.linspace(0.004, 0.006, 1000)
    tr = driver.BatchedEvaluator._trajectory
    got = tr({"delay_trajectory": t}, 600, 44100)
    assert got.dtype == torch.float32 and got.shape == (600,)
    assert torch.equal(got, torch.from_numpy(t[:600].astype(np.float32)) * 44100.0)
    p = str(tmp_path / "trajectory_3_.npy")
    np.save(p, {"delay_trajectory": t})
    seg = tr({"trajectory_file": p, "offset": 100, "length": 250}, 250, 48000)
    assert torch.equal(seg, torch.from_numpy(t[100:350].astype(np.float32)) * 48000.0)
    with pytest.raises(KeyError):
        tr({"input_file": "x.wav"}, 10, 44100)
    with pytest.raises(ValueError):
        tr({"delay_trajectory": t[:5]}, 10, 44100)
    from ntm_b200 import DiffDelRNN, TimeVaryingDelayLine
    with pytest.raises(ValueError):                       # ADD_DELAY is a plain-GRU mode (code/test-model.py:354)
        driver.BatchedEvaluator(DiffDelRNN(1, 64, 1, False, max_delay=8), delay=TimeVaryingDelayLine(max_delay=8))


# ---- the native RIFF/WAVE reader against reference-held audio (SURVEY 8f rank 4; VERDICT r01 #10) -------------------------
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _reference_layout_wavs(dirname, n=24):
    """n seeded files in the two layouts of the reference's results/**.wav (tests/golden/ref_*_head.wav keep the originals'
    headers): int16 PCM, here with an odd-sized LIST chunk and its pad byte before the data, and float32 with fact + PEAK
    chunks; mono and stereo, 44.1 / 48 kHz, lengths from 6000 frames up."""
    rng = np.random.default_rng(11)
    paths = []
    for i in range(n):
        ch, fs, frames, pcm = 1 + i % 2, (44100, 48000)[i // 2 % 2], 6000 + 397 * i, i % 4 < 2
        if pcm:
            data = (rng.standard_normal((frames, ch)) * 6000).clip(-32768, 32767).astype("<i2").tobytes()
            fmt = struct.pack("<HHIIHH", 1, ch, fs, fs * ch * 2, ch * 2, 16)
            extra = [(b"LIST", b"INFOISFT\x05\x00\x00\x00ntm\x00\x00")]                     # 17 bytes: padded to 18
        else:
            data = (rng.standard_normal((frames, ch)) * 0.3).astype("<f4").tobytes()
            fmt = struct.pack("<HHIIHH", 3, ch, fs, fs * ch * 4, ch * 4, 32)
            extra = [(b"fact", struct.pack("<I", frames)), (b"PEAK", struct.pack("<II", 1, 0) + b"\x00" * 8 * ch)]
        body = b"WAVE"
        for cid, payload in [(b"fmt ", fmt)] + extra + [(b"data", data)]:
            body += struct.pack("<4sI", cid, len(payload)) + payload + b"\x00" * (len(payload) & 1)
        paths.append(os.path.join(dirname, f"gen_{i:02d}.wav"))
        with open(paths[-1], "wb") as f:
            f.write(b"RIFF" + struct.pack("<I", len(body)) + body)
    return paths


def _scipy_float(path):
    import warnings
    import scipy.io.wavfile as wavfile
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fs, a = wavfile.read(path)
    a = a.reshape(len(a), -1).T
    if a.dtype == np.int16:
        a = a.astype(np.float32) / 32768.0
    return fs, np.ascontiguousarray(a.astype(np.float32))


def test_read_wav_equals_scipy_on_every_reference_held_wav(tmp_path):
    """The reference-held excerpts of tests/golden and seeded files in the same two layouts (the reference's results/**
    holds int16 and float32 files with extra RIFF chunks), whole-file and segment reads (`frame_offset` / `num_frames`
    of code/dataset.py:362-365), against scipy.io.wavfile."""
    files = [os.path.join(GOLD, n) for n in ("ref_int16_head.wav", "ref_float32_head.wav")]
    files += _reference_layout_wavs(str(tmp_path))
    kinds = set()
    for i, path in enumerate(files):
        fs, want = _scipy_float(path)
        info = driver.wav_info(path)
        kinds.add((info["format"], info["bits"]))
        assert (info["fs"], info["channels"], info["frames"]) == (fs, want.shape[0], want.shape[1]), path
        got, fs2 = driver.read_wav(path)
        assert fs2 == fs and np.array_equal(got, want), path
        off, n = 1000 + 37 * i, 4096
        seg, _ = driver.read_wav(path, off, n)
        assert np.array_equal(seg, want[:, off:off + n]), path
        tail, _ = driver.read_wav(path, want.shape[1] - 100, 4096)          # clipped at the end of the file
        assert np.array_equal(tail, want[:, -100:]), path
    assert kinds == {(1, 16), (3, 32)}


@pytest.mark.parametrize("name", ["ref_int16_head.wav", "ref_float32_head.wav"])
def test_read_wav_on_committed_reference_excerpts(name):
    """The first 2048 frames of one int16 and one float32 reference-held file (tests/golden/, cut by
    oracle/make_golden_wav.py with the original headers and extra chunks kept): runs wherever the repository is."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name)
    fs, want = _scipy_float(path)
    got, fs2 = driver.read_wav(path)
    assert fs2 == fs == 44100 and got.shape == (1, 2048) and np.array_equal(got, want)
    seg, _ = driver.read_wav(path, 100, 50)
    assert np.array_equal(seg, want[:, 100:150])
