"""Batched evaluation driver: many (file, segment) examples per launch instead of `DataLoader(batch_size=1)`.

Replaces the per-file loop of the reference's evaluation flow (code/test-model.py:332-353 prediction, :367-388 cut +
losses, :882-893 .wav output) and the segment reads of code/dataset.py:348-379 (`torchaudio.load(file, num_frames=length,
frame_offset=offset, normalize=False)`): examples are packed into one zero-padded (B, 1, T_max) batch -- the model is
causal, so trailing padding never changes a real sample --, predicted with predict() semantics per stream (zero state,
1024-sample warm start), cut by INIT_LEN, scored on the device (ESR / DCPreESR, optionally MR-STFT) and optionally
written back as float32 .wav files.  The on-disk format is the reference's: float32 (or PCM) RIFF/WAVE, channel 0 = audio,
channel 1 (if any) = the 100 Hz pulse track (SURVEY.md section 8f rank 4).  No soundfile / torchaudio needed.

All three prediction modes of the reference's loss loop (code/test-model.py:346-368) are covered: plain GRU, DiffDelGRU
with the example's delay trajectory (`meta['delay_trajectory'] * fs`, :349-352), and GRU followed by the stand-alone delay
line (`ADD_DELAY`, `apply_delay`, :259-290,354-360).  Trajectories come from the dataset's `trajectory_*.npy` files (a
pickled dict with key 'delay_trajectory' in seconds, code/utilities/utilities.py:273-284) or from an array in the example.
"""
import os
import struct

import numpy as np
import torch

from .losses import DCPreESR, ESRLoss, MultiResolutionSTFTLoss

_PCM, _FLOAT, _EXTENSIBLE = 1, 3, 0xFFFE


def wav_info(path):
    """Parse the RIFF header: {'fs', 'channels', 'frames', 'format' (1 PCM / 3 float), 'bits', 'data_offset'}."""
    with open(path, "rb") as f:
        riff, _, wave = struct.unpack("<4sI4s", f.read(12))
        if riff != b"RIFF" or wave != b"WAVE":
            raise ValueError(f"{path}: not a RIFF/WAVE file")
        fmt = None
        while True:
            hdr = f.read(8)
            if len(hdr) < 8:
                raise ValueError(f"{path}: no data chunk")
            cid, size = struct.unpack("<4sI", hdr)
            if cid == b"fmt ":
                raw = f.read(size)
                tag, ch, fs, _, align, bits = struct.unpack("<HHIIHH", raw[:16])
                if tag == _EXTENSIBLE and size >= 26:
                    tag = struct.unpack("<H", raw[24:26])[0]
                fmt = (tag, ch, fs, align, bits)
                if size & 1:
                    f.read(1)
            elif cid == b"data":
                if fmt is None:
                    raise ValueError(f"{path}: data chunk before fmt chunk")
                tag, ch, fs, align, bits = fmt
                if tag not in (_PCM, _FLOAT) or (tag == _FLOAT and bits not in (32, 64)) or \
                        (tag == _PCM and bits not in (8, 16, 24, 32)):
                    raise ValueError(f"{path}: unsupported sample format (tag {tag}, {bits} bits)")
                remaining = os.path.getsize(path) - f.tell()
                size = min(size, remaining) if size not in (0, 0xFFFFFFFF) else remaining
                return {"fs": fs, "channels": ch, "frames": size // align, "format": tag, "bits": bits,
                        "data_offset": f.tell()}
            else:
                f.seek(size + (size & 1), os.SEEK_CUR)


def read_wav(path, frame_offset=0, num_frames=-1):
    """-> (float32 array (channels, frames), fs).  Float files are returned as stored (the reference reads with
    normalize=False, code/dataset.py:362-365); PCM files are scaled to [-1, 1)."""
    info = wav_info(path)
    ch, bits, tag = info["channels"], info["bits"], info["format"]
    first = max(0, min(int(frame_offset), info["frames"]))
    n = info["frames"] - first if num_frames is None or num_frames < 0 else max(0, min(int(num_frames), info["frames"] - first))
    bps = bits // 8
    with open(path, "rb") as f:
        f.seek(info["data_offset"] + first * ch * bps)
        raw = f.read(n * ch * bps)
    if tag == _FLOAT:
        a = np.frombuffer(raw, dtype="<f4" if bits == 32 else "<f8").astype(np.float32, copy=False)
    elif bits == 8:
        a = (np.frombuffer(raw, dtype=np.uint8).astype(np.float32) - 128.0) / 128.0
    elif bits == 16:
        a = np.frombuffer(raw, dtype="<i2").astype(np.float32) / 32768.0
    elif bits == 32:
        a = (np.frombuffer(raw, dtype="<i4").astype(np.float64) / 2147483648.0).astype(np.float32)
    else:                                                   # 24-bit PCM: sign-extend three little-endian bytes
        b = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 3).astype(np.int32)
        v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
        a = ((v ^ 0x800000) - 0x800000).astype(np.float32) / 8388608.0
    return np.ascontiguousarray(a.reshape(-1, ch).T), info["fs"]


def write_wav(path, data, fs):
    """float32 IEEE .wav; data: (frames,) or (channels, frames)."""
    a = np.asarray(data, dtype=np.float32)
    a = a.reshape(1, -1) if a.ndim == 1 else a
    ch, frames = a.shape
    payload = np.ascontiguousarray(a.T).astype("<f4").tobytes()
    with open(path, "wb") as f:
        f.write(struct.pack("<4sI4s", b"RIFF", 4 + 8 + 16 + 8 + 4 + 8 + len(payload), b"WAVE"))
        f.write(struct.pack("<4sIHHIIHH", b"fmt ", 16, _FLOAT, ch, int(fs), int(fs) * ch * 4, ch * 4, 32))
        f.write(struct.pack("<4sII", b"fact", 4, frames))
        f.write(struct.pack("<4sI", b"data", len(payload)))
        f.write(payload)


def read_trajectory(path, offset=0, length=-1):
    """Delay trajectory in SECONDS for frames [offset, offset+length) of a file: `trajectory_*.npy` holds a pickled dict
    {'delay_trajectory', 'input_peaks', 'output_peaks', ...} (code/utilities/utilities.py:273-284); a plain array file is
    accepted too.  The slice is the reference's `T_delay[offset:end]` (code/dataset.py:383)."""
    a = np.load(path, allow_pickle=True)
    if a.dtype == object and a.ndim == 0:
        a = a.item()["delay_trajectory"]
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    end = len(a) if length is None or length < 0 else int(offset) + int(length)
    return a[int(offset):end]


def mean_losses(results, keys=("ESR", "DCPreESR", "MR-STFT")):
    """Dataset mean of the per-example losses = the reference's `results_dict[key] / num_batches` with batch size 1
    (code/test-model.py:385-397)."""
    return {k: float(np.mean([r[k] for r in results])) for k in keys if results and all(k in r for r in results)}


class BatchedEvaluator:
    """Predict (and score) many examples per launch.

    examples: dicts with 'input_file' and optionally 'target_file', 'offset' (frames, default 0), 'length' (frames,
    default: to the end of the file) -- the fields of `AudioDataset.examples` (code/dataset.py:348-379) -- and, for the
    delay modes, 'delay_trajectory' (array, SECONDS, one value per frame of the segment) or 'trajectory_file'
    (`trajectory_*.npy`, sliced with the example's offset / length).
    `model` is an ntm_b200.RNN or DiffDelRNN on a CUDA device; `delay` is an optional stand-alone
    ntm_b200.TimeVaryingDelayLine applied after a plain RNN (the reference's ADD_DELAY); `max_streams` examples are
    packed per launch.  `mrstft=True` adds the reference's third loss, auraloss `MultiResolutionSTFTLoss()`
    (code/test-model.py:253), as r['MR-STFT'], over the same window and in the same per-group pass."""

    def __init__(self, model, max_streams=1024, delay=None, mrstft=False):
        from .model import DiffDelRNN
        self.model, self.max_streams, self.delay = model, int(max_streams), delay
        self.diffdel = isinstance(model, DiffDelRNN)
        if self.diffdel and delay is not None:
            raise ValueError("ADD_DELAY applies to the plain GRU only (code/test-model.py:354)")
        self.losses = {"ESR": ESRLoss(), "DCPreESR": DCPreESR(dc_pre=True)}
        if mrstft:
            self.losses["MR-STFT"] = MultiResolutionSTFTLoss()

    @staticmethod
    def _load(ex, key):
        a, fs = read_wav(ex[key], ex.get("offset", 0), ex.get("length", -1))
        return a[0], fs                                       # channel 0 = audio (channel 1 = pulse track)

    @staticmethod
    def _trajectory(ex, n, fs):
        """The example's delay trajectory in SAMPLES (`meta['delay_trajectory'].float() * fs`, code/test-model.py:349-351,
        356-358): float32 first, then scaled, like the reference."""
        if "delay_trajectory" in ex:
            t = np.asarray(ex["delay_trajectory"], dtype=np.float64).reshape(-1)
        elif "trajectory_file" in ex:
            t = read_trajectory(ex["trajectory_file"], ex.get("offset", 0), ex.get("length", -1))
        else:
            raise KeyError("a delay mode needs 'delay_trajectory' or 'trajectory_file' in every example")
        if len(t) < n:
            raise ValueError(f"delay trajectory has {len(t)} values for a segment of {n} frames")
        return torch.from_numpy(t[:n].astype(np.float32)) * float(fs)

    def _apply_delay(self, d, y):
        """`apply_delay` (code/test-model.py:259-290): fresh zero history for every stream, then the delay line over the
        whole signal (the reference walks 4096-sample chunks with a carried buffer; the kernel carries the same history
        inside one call, so the result is identical)."""
        self.delay.init_buffer(y.shape[0])
        return self.delay(y, d)

    def run(self, examples, out_dir=None, init_len=0, write_pre_d=False):
        """-> one dict per example: {'input_name', 'frames', 'fs', ['ESR', 'DCPreESR', ['MR-STFT',]] ['output_file']}; losses are
        computed after cutting the first `init_len` samples (INIT_LEN, code/test-model.py:323-325,367-370)."""
        dev = self.model._device()
        need_d = self.diffdel or self.delay is not None
        results = []
        with torch.inference_mode():
            for b0 in range(0, len(examples), self.max_streams):
                group = examples[b0:b0 + self.max_streams]
                loaded = [self._load(ex, "input_file") for ex in group]
                lens = [len(a) for a, _ in loaded]
                B, Tmax = len(group), max(max(lens), 1)
                xh = torch.zeros((B, 1, Tmax), dtype=torch.float32, pin_memory=True)
                for i, (a, _) in enumerate(loaded):
                    xh[i, 0, :lens[i]] = torch.from_numpy(a)
                x = xh.to(dev, non_blocking=True)
                pre = None
                if need_d:                                   # zero delay over the padding: reads only what exists
                    dh = torch.zeros((B, 1, Tmax), dtype=torch.float32, pin_memory=True)
                    for i, ex in enumerate(group):
                        dh[i, 0, :lens[i]] = self._trajectory(ex, lens[i], loaded[i][1])
                    d = dh.to(dev, non_blocking=True)
                if self.diffdel:
                    y, pre = self.model.predict(x, d)
                else:
                    y = self.model.predict(x)
                    if self.delay is not None:
                        y = self._apply_delay(d, y)
                yh = y.cpu() if out_dir is not None else None
                ph = pre.cpu() if out_dir is not None and write_pre_d and pre is not None else None
                # targets of the whole group, padded like the inputs; every example is scored over its own window
                # [init_len, min(len(target), len(input))) in ONE launch per loss (ESRLoss.per_example)
                scored = [i for i, ex in enumerate(group) if "target_file" in ex]
                group_losses = {}
                if scored:
                    th = torch.zeros((B, 1, Tmax), dtype=torch.float32, pin_memory=True)
                    counts = torch.zeros(B, dtype=torch.int64)
                    for i in scored:
                        t, _ = self._load(group[i], "target_file")
                        n = min(len(t), lens[i])
                        th[i, 0, :n] = torch.from_numpy(np.array(t[:n]))
                        counts[i] = max(n - init_len, 0)
                    td = th.to(dev, non_blocking=True)
                    first = torch.full((B,), int(init_len), dtype=torch.int64)
                    for key, fn in self.losses.items():
                        group_losses[key] = fn.per_example(y, td, first, counts).cpu()
                for i, ex in enumerate(group):
                    name = os.path.basename(ex["input_file"])
                    off = ex.get("offset", 0)
                    stem, ext = os.path.splitext(name)
                    res = {"input_name": f"{stem}_[{off}:{off + lens[i]}]{ext}", "frames": lens[i], "fs": loaded[i][1]}
                    if "target_file" in ex:
                        for key in self.losses:
                            res[key] = float(group_losses[key][i])
                    if out_dir is not None:
                        os.makedirs(out_dir, exist_ok=True)
                        res["output_file"] = os.path.join(out_dir, f"{stem}_[{off}:{off + lens[i]}]_pred.wav")
                        write_wav(res["output_file"], yh[i, 0, :lens[i]].numpy(), loaded[i][1])
                        if ph is not None:
                            res["pre_d_file"] = os.path.join(out_dir, f"{stem}_[{off}:{off + lens[i]}]_pred_pre_d.wav")
                            write_wav(res["pre_d_file"], ph[i, 0, :lens[i]].numpy(), loaded[i][1])
                    results.append(res)
        return results
