"""The two restatements of auraloss `MultiResolutionSTFTLoss` in oracle/ref_mrstft.py agree: (a) torch.stft in float64
and (b) the explicit float64 numpy form (reflect index map, padded Hann window, rfft), at odd and minimal lengths, at the
default and at non-default resolutions.  CPU only."""
import numpy as np
import pytest
import torch

from oracle import ref_mrstft

NON_DEFAULT = dict(fft_sizes=(256, 4096), hop_sizes=(64, 1024), win_lengths=(256, 3000), w_sc=0.0, w_lin_mag=1.0)


def pair(B, T, seed):
    rng = np.random.default_rng(seed)
    t = 0.2 * rng.standard_normal((B, 1, T))
    return t + 0.02 * rng.standard_normal((B, 1, T)), t


@pytest.mark.parametrize("T, kw", ((1025, {}), (4801, {}), (2049, NON_DEFAULT), (4801, NON_DEFAULT)),
                         ids=("defaults-1025", "defaults-4801", "non_default-2049", "non_default-4801"))
def test_torch_stft_restatement_equals_numpy_restatement(T, kw):
    o, t = pair(2, T, T)
    a = float(ref_mrstft.mrstft_torch(torch.from_numpy(o), torch.from_numpy(t), **kw))
    b = ref_mrstft.mrstft_numpy(o, t, **kw)
    assert abs(a - b) <= 1e-12 * abs(b), (a, b)


def test_minimal_length_and_batch_norm_sc():
    """T = N/2 + 1 for N = 2048 is the shortest row torch.stft accepts; the batch SC is one ratio over all rows."""
    o, t = pair(3, 1025, 7)
    o[1] *= 3.0
    b = ref_mrstft.mrstft_numpy(o, t)
    assert abs(float(ref_mrstft.mrstft_torch(torch.from_numpy(o), torch.from_numpy(t))) - b) <= 1e-12 * b
    rows = np.mean([ref_mrstft.mrstft_numpy(o[i:i + 1], t[i:i + 1]) for i in range(3)])
    assert abs(rows - b) > 1e-3 * b


def test_reflect_padding_needs_more_than_half_an_fft():
    o, t = pair(1, 1024, 1)
    with pytest.raises(RuntimeError):
        ref_mrstft.mrstft_torch(torch.from_numpy(o), torch.from_numpy(t))
    with pytest.raises(ValueError):
        ref_mrstft.mrstft_numpy(o, t)
