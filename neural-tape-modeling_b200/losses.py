"""Evaluation losses of the reference's test flow, computed on the device by the engine (csrc/esr.cu, csrc/stft.cu).

Drop-in for the three loss objects `code/test-model.py:250-254` builds:
    'ESR':      ESRLoss()                 code/Automated_GuitarAmpModelling/CoreAudioML/training.py:5-16
    'DCPreESR': DCPreESR(dc_pre=True)     code/GreyBoxDRC/loss_funcs.py:32-52 (DC_PreEmph :6-30 + ESR)
    'MR-STFT':  MultiResolutionSTFTLoss() auraloss/freq.py (defaults; restated in oracle/ref_mrstft.py)
Same call: `loss_fcn(output, target)` with (B, 1, T) tensors -> 0-dim float32 tensor (no host synchronisation).
No CPU path: non-CUDA tensors raise.
"""
import torch

from . import lib


def _row_windows(B, T, dev, first, count):
    """first / count as contiguous int64 tensors on dev (or None), and the clipped window length of every row."""
    if first is not None:
        first = torch.as_tensor(first, dtype=torch.int64).to(dev).contiguous()
    if count is not None:
        count = torch.as_tensor(count, dtype=torch.int64).to(dev).contiguous()
    f0 = torch.zeros(B, dtype=torch.int64, device=dev) if first is None else first.clamp(0, T)
    n = (T - f0) if count is None else torch.minimum(count.clamp(min=0), T - f0)
    return first, count, n


class ESRLoss(torch.nn.Module):
    """Error-to-signal ratio; `dc_pre=True` applies the reference's 2000-tap DC pre-emphasis filter to both signals."""

    def __init__(self, dc_pre=False):
        super().__init__()
        self.epsilon = 0.00001
        self.dc_pre = bool(dc_pre)

    @staticmethod
    def _rows(t, name):
        if t.dim() == 3:
            if t.shape[1] != 1:
                raise RuntimeError(f"ntm_b200: {name} must be (B, 1, T), got {tuple(t.shape)}")
            t = t[:, 0, :]
        elif t.dim() != 2:
            raise RuntimeError(f"ntm_b200: {name} must be (B, 1, T) or (B, T), got {tuple(t.shape)}")
        if t.dtype != torch.float32:
            t = t.float()
        if t.shape[1] > 0 and t.stride(1) != 1:
            t = t.contiguous()
        return t

    def forward(self, output, target):
        if not output.is_cuda or not target.is_cuda:
            raise RuntimeError("ntm_b200: the engine has no CPU path; move output/target to a CUDA device")
        if output.shape != target.shape:
            raise RuntimeError(f"ntm_b200: output {tuple(output.shape)} and target {tuple(target.shape)} differ")
        o, t = self._rows(output, "output"), self._rows(target, "target")
        if t.device != o.device:
            raise RuntimeError("ntm_b200: output and target live on different devices")
        B, T = o.shape
        sums = lib.ops().esr_sums(o, t, self.dc_pre)
        n = max(B * T, 1)
        return ((sums[0] / n) / (sums[1] / n + self.epsilon)).float()

    def per_example(self, output, target, first=None, count=None):
        """One loss per row of a (ragged) batch in ONE launch: row b is scored over its own window of samples
        [first[b], first[b] + count[b]) -- what the reference computes with batch size 1, file by file, after cutting
        INIT_LEN (code/test-model.py:367-370,385-397).  first / count: int64 tensors of B values or None (0 / T).
        -> float32 tensor of B losses (no host synchronisation)."""
        if not output.is_cuda or not target.is_cuda:
            raise RuntimeError("ntm_b200: the engine has no CPU path; move output/target to a CUDA device")
        if output.shape != target.shape:
            raise RuntimeError(f"ntm_b200: output {tuple(output.shape)} and target {tuple(target.shape)} differ")
        o, t = self._rows(output, "output"), self._rows(target, "target")
        B, T = o.shape
        first, count, n = _row_windows(B, T, o.device, first, count)
        sums = lib.ops().esr_sums_rows(o, t, first, count, self.dc_pre)
        n = n.clamp(min=1).to(torch.float64)
        return ((sums[:, 0] / n) / (sums[:, 1] / n + self.epsilon)).float()


class DCPreESR(ESRLoss):
    """`from GreyBoxDRC.loss_funcs import ESRLoss as DCPreESR` (code/test-model.py:28): dc_pre defaults to True."""

    def __init__(self, dc_pre=True):
        super().__init__(dc_pre=dc_pre)


class MultiResolutionSTFTLoss(torch.nn.Module):
    """auraloss `MultiResolutionSTFTLoss` (auraloss/freq.py) with its constructor keywords and defaults: the mean over the
    resolutions of w_sc SC + w_log_mag LogMag + w_lin_mag LinMag on the clamped STFT magnitudes (Hann window, center=True,
    reflect padding).  Same call: `loss_fcn(output, target)` with (B, 1, T) tensors -> 0-dim float32 tensor (no host
    synchronisation).  One fused pass per resolution (csrc/stft.cu); the spectrograms are never materialised.
    FFT sizes: powers of two from 256 to 4096.  Phase, mel / chroma scaling, perceptual weighting, scale invariance and
    other windows raise NotImplementedError."""

    def __init__(self, fft_sizes=(1024, 2048, 512), hop_sizes=(120, 240, 50), win_lengths=(600, 1200, 240),
                 window="hann_window", w_sc=1.0, w_log_mag=1.0, w_lin_mag=0.0, w_phs=0.0, sample_rate=None, scale=None,
                 n_bins=None, perceptual_weighting=False, scale_invariance=False, eps=1e-8, output="loss",
                 reduction="mean", mag_distance="L1", device=None):
        super().__init__()
        self.fft_sizes, self.hop_sizes, self.win_lengths = [int(v) for v in fft_sizes], [int(v) for v in hop_sizes], \
            [int(v) for v in win_lengths]
        if not (len(self.fft_sizes) == len(self.hop_sizes) == len(self.win_lengths)) or not self.fft_sizes:
            raise ValueError("fft_sizes, hop_sizes and win_lengths must have the same non-zero length")
        unsupported = {"w_phs": (w_phs, 0.0), "scale": (scale, None), "n_bins": (n_bins, None),
                       "perceptual_weighting": (perceptual_weighting, False),
                       "scale_invariance": (scale_invariance, False), "window": (window, "hann_window"),
                       "output": (output, "loss"), "eps": (eps, 1e-8), "reduction": (reduction, "mean"),
                       "mag_distance": (mag_distance, "L1")}
        for name, (value, default) in unsupported.items():
            if value != default:
                raise NotImplementedError(f"ntm_b200: MultiResolutionSTFTLoss({name}={value!r}) is not implemented "
                                          f"(only {name}={default!r})")
        for n, hop, win in zip(self.fft_sizes, self.hop_sizes, self.win_lengths):
            if n < 256 or n > 4096 or n & (n - 1):
                raise NotImplementedError(f"ntm_b200: fft sizes must be powers of two from 256 to 4096, got {n}")
            if not 1 <= win <= n or hop < 1:
                raise ValueError(f"ntm_b200: need 1 <= win_length <= fft_size and hop_size >= 1, got {(n, hop, win)}")
        self.w_sc, self.w_log_mag, self.w_lin_mag = float(w_sc), float(w_log_mag), float(w_lin_mag)
        self.sample_rate = sample_rate

    def _sums(self, output, target, first, count):
        if not output.is_cuda or not target.is_cuda:
            raise RuntimeError("ntm_b200: the engine has no CPU path; move output/target to a CUDA device")
        if output.shape != target.shape:
            raise RuntimeError(f"ntm_b200: output {tuple(output.shape)} and target {tuple(target.shape)} differ")
        o, t = ESRLoss._rows(output, "output"), ESRLoss._rows(target, "target")
        if t.device != o.device:
            raise RuntimeError("ntm_b200: output and target live on different devices")
        B, T = o.shape
        first, count, n = _row_windows(B, T, o.device, first, count)
        sums = lib.ops().mrstft_sums_rows(o, t, first, count, self.fft_sizes, self.hop_sizes, self.win_lengths)
        return sums, n

    def _combine(self, sc, log_mag, lin_mag):
        """Mean over the resolutions (last axis) of the weighted terms; a term of weight 0 is not evaluated (auraloss)."""
        loss = torch.zeros_like(sc)
        if self.w_sc:
            loss = loss + self.w_sc * sc
        if self.w_log_mag:
            loss = loss + self.w_log_mag * log_mag
        if self.w_lin_mag:
            loss = loss + self.w_lin_mag * lin_mag
        return loss.mean(dim=-1)

    def _bins(self, n):
        """Magnitude elements per row and resolution: F (N/2 + 1), F = 1 + n // hop.  n: (B,) int64 -> (B, n_res) double."""
        hop = torch.tensor(self.hop_sizes, dtype=torch.int64, device=n.device)
        half = torch.tensor([v // 2 + 1 for v in self.fft_sizes], dtype=torch.int64, device=n.device)
        return ((1 + n[:, None] // hop) * half).to(torch.float64)

    def forward(self, output, target):
        T = output.shape[-1]
        for n in self.fft_sizes:
            if T <= n // 2:
                raise RuntimeError(f"ntm_b200: reflect padding by {n // 2} needs more than {n // 2} samples, got {T}")
        sums, n = self._sums(output, target, None, None)
        s = sums.sum(dim=0)                                          # (n_res, 4): SC is one ratio over the whole batch
        elems = self._bins(n).sum(dim=0)
        return self._combine(s[:, 0].sqrt() / s[:, 1].sqrt(), s[:, 2] / elems, s[:, 3] / elems).float()

    def per_example(self, output, target, first=None, count=None):
        """One loss per row of a (ragged) batch, row b over its own window [first[b], first[b] + count[b]) as
        ESRLoss.per_example (the INIT_LEN cut of code/test-model.py:367-370; the reflection is relative to the window).
        A row whose window has no more than fft_size / 2 samples gets NaN.  -> float32 tensor of B losses."""
        sums, n = self._sums(output, target, first, count)
        elems = self._bins(n)
        return self._combine(sums[..., 0].sqrt() / sums[..., 1].sqrt(), sums[..., 2] / elems, sums[..., 3] / elems).float()
