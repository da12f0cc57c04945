"""Restatements of auraloss `MultiResolutionSTFTLoss` with its defaults (auraloss/freq.py: STFTLoss, SpectralConvergenceLoss,
STFTMagnitudeLoss), the third loss of the reference's evaluation loop (code/test-model.py:253).  auraloss itself is not a
dependency; these restate its source line by line and are what the engine's csrc/stft.cu is tested against.

    mrstft_torch  (a) the auraloss lines with torch.stft, in the dtype and on the device of the inputs
    mrstft_numpy  (b) explicit float64 numpy: reflect index map, zero-padded periodic Hann window, np.fft.rfft

Both take (B, 1, T) or (B, T) arrays and return the whole-batch loss: per resolution
    SC      = ||Y - X||_F / ||Y||_F over the whole batch (one ratio, not a mean of per-row ratios)
    LogMag  = mean |ln X - ln Y|
    LinMag  = mean |X - Y|
with X, Y = sqrt(max(|STFT|^2, 1e-8)) of output / target, and the loss is the mean over the resolutions of
w_sc SC + w_log_mag LogMag + w_lin_mag LinMag (a term with weight 0 is not evaluated, as in auraloss).
"""
import numpy as np

FFT_SIZES = (1024, 2048, 512)
HOP_SIZES = (120, 240, 50)
WIN_LENGTHS = (600, 1200, 240)
EPS = 1e-8


def _combine(terms, w_sc, w_log_mag, w_lin_mag):
    total = 0.0
    for sc, logm, linm in terms:
        loss = 0.0
        if w_sc:
            loss = loss + w_sc * sc
        if w_log_mag:
            loss = loss + w_log_mag * logm
        if w_lin_mag:
            loss = loss + w_lin_mag * linm
        total = total + loss
    return total / len(terms)


def mrstft_torch(output, target, fft_sizes=FFT_SIZES, hop_sizes=HOP_SIZES, win_lengths=WIN_LENGTHS, w_sc=1.0,
                 w_log_mag=1.0, w_lin_mag=0.0):
    """(a): torch.stft (center=True, reflect padding) on whatever dtype / device the tensors have -> 0-dim tensor."""
    import torch
    x, y = output.reshape(output.shape[0], -1), target.reshape(target.shape[0], -1)
    terms = []
    for n_fft, hop, win in zip(fft_sizes, hop_sizes, win_lengths):
        window = torch.hann_window(win, dtype=x.dtype, device=x.device)

        def mag(s):
            z = torch.stft(s, n_fft, hop, win, window, return_complex=True)
            return torch.sqrt(torch.clamp(z.real ** 2 + z.imag ** 2, min=EPS))

        xm, ym = mag(x), mag(y)
        terms.append((torch.linalg.norm(ym - xm) / torch.linalg.norm(ym),
                      torch.mean(torch.abs(torch.log(xm) - torch.log(ym))),
                      torch.mean(torch.abs(xm - ym))))
    return _combine(terms, w_sc, w_log_mag, w_lin_mag)


def reflect_index(T, n_fft, hop):
    """(frames, n_fft) indices into a row of T samples: frame f starts at f * hop - n_fft // 2, reflected at both ends."""
    if T <= n_fft // 2:
        raise ValueError(f"reflect padding by {n_fft // 2} needs more than {n_fft // 2} samples, got {T}")
    frames = 1 + T // hop
    i = np.arange(frames)[:, None] * hop - n_fft // 2 + np.arange(n_fft)[None, :]
    i = np.where(i < 0, -i, i)
    return np.where(i >= T, 2 * (T - 1) - i, i)


def padded_hann(n_fft, win):
    """Periodic Hann window of length win centred in n_fft points (zeros elsewhere), float64."""
    w = np.zeros(n_fft)
    off = (n_fft - win) // 2
    w[off:off + win] = 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(win) / win)
    return w


def stft_mag_numpy(x, n_fft, hop, win):
    """(B, frames, n_fft // 2 + 1) clamped magnitudes of the rows of x, float64."""
    x = np.asarray(x, dtype=np.float64).reshape(np.shape(x)[0], -1)
    frames = x[:, reflect_index(x.shape[1], n_fft, hop)] * padded_hann(n_fft, win)
    z = np.fft.rfft(frames, axis=-1)
    return np.sqrt(np.maximum(z.real ** 2 + z.imag ** 2, EPS))


def mrstft_numpy(output, target, fft_sizes=FFT_SIZES, hop_sizes=HOP_SIZES, win_lengths=WIN_LENGTHS, w_sc=1.0,
                 w_log_mag=1.0, w_lin_mag=0.0):
    """(b): explicit float64 restatement -> float."""
    terms = []
    for n_fft, hop, win in zip(fft_sizes, hop_sizes, win_lengths):
        xm, ym = stft_mag_numpy(output, n_fft, hop, win), stft_mag_numpy(target, n_fft, hop, win)
        terms.append((np.linalg.norm(ym - xm) / np.linalg.norm(ym), np.mean(np.abs(np.log(xm) - np.log(ym))),
                      np.mean(np.abs(xm - ym))))
    return float(_combine(terms, w_sc, w_log_mag, w_lin_mag))
