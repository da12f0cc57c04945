#!/usr/bin/env python3
"""Dev tool (GPU box): the on-device multi-resolution STFT loss (csrc/stft.cu) against the fp32 torch.stft restatement of
auraloss MultiResolutionSTFTLoss (oracle/ref_mrstft.py, chunked over rows so that its spectrograms fit in memory), both
timed with CUDA events after warm-up on the same GPU, plus the agreement check of tests/test_mrstft_gpu.py against the same
restatement in float64: |L - L64| <= max(2e-5 |L64|, 2 |L32 - L64|).

Floors from shapes (per sample of the two signals, default resolutions): FFT work 2 x sum 5 N log2 N / hop flops against
the fp32 CUDA-core rate (SMs x 128 lanes x 2 flops x max SM clock), and 8 bytes of HBM traffic against 7.7 TB/s."""
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch

import ntm_b200
from oracle import ref_mrstft

DEV = "cuda:0"
RES = list(zip(ref_mrstft.FFT_SIZES, ref_mrstft.HOP_SIZES, ref_mrstft.WIN_LENGTHS))
HBM_BPS = 7.7e12


def restatement(o, t, dtype, rows_per_chunk):
    """auraloss lines with torch.stft, whole-batch semantics, accumulated over row chunks."""
    terms = []
    for n_fft, hop, win in RES:
        window = torch.hann_window(win, dtype=dtype, device=o.device)
        s = torch.zeros(4, dtype=torch.float64, device=o.device)
        elems = 0
        for b0 in range(0, o.shape[0], rows_per_chunk):
            def mag(x):
                z = torch.stft(x[b0:b0 + rows_per_chunk, 0].to(dtype), n_fft, hop, win, window, return_complex=True)
                return torch.sqrt(torch.clamp(z.real ** 2 + z.imag ** 2, min=ref_mrstft.EPS))
            xm, ym = mag(o), mag(t)
            s += torch.stack([((ym - xm) ** 2).sum(), (ym ** 2).sum(), (torch.log(xm) - torch.log(ym)).abs().sum(),
                              (xm - ym).abs().sum()]).double()
            elems += xm.numel()
            del xm, ym
        terms.append(s[0].sqrt() / s[1].sqrt() + s[2] / elems)
    return sum(terms) / len(terms)


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    best, v = 1e30, None
    for _ in range(reps):
        e0.record()
        v = fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / 1e3)
    return best, float(v)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    clock_mhz = float(q.split(",")[2].split()[0])
    fma_peak = sms * 128 * 2 * clock_mhz * 1e6
    flops_per_sample = 2 * sum(5 * n * math.log2(n) / hop for n, hop, _ in RES)
    print(f"card: {q}  ({sms} SMs)")
    print(f"floors per sample (two signals): {flops_per_sample:.0f} nominal FFT flop -> fp32 CUDA-core peak "
          f"{fma_peak / 1e12:.1f} TFLOP/s; 8 B HBM -> {HBM_BPS / 1e12:.1f} TB/s")
    L = ntm_b200.MultiResolutionSTFTLoss()
    ok_all = True
    for B, secs in ((256, 30), (1024, 10)):
        T = 48000 * secs
        g = torch.Generator(device=DEV).manual_seed(B)
        t = 0.2 * torch.randn(B, 1, T, device=DEV, generator=g)
        o = t + 0.02 * torch.randn(B, 1, T, device=DEV, generator=g)
        chunk = 16
        te, le = timed(lambda: L(o, t), 5)
        tr, l32 = timed(lambda: restatement(o, t, torch.float32, chunk), 2)
        l64 = float(restatement(o, t, torch.float64, chunk // 2))
        ok = abs(le - l64) <= max(2e-5 * abs(l64), 2 * abs(l32 - l64))
        ok_all &= ok
        n = B * T
        fl, by = flops_per_sample * n / te, 8 * n / te
        f_fma, f_hbm = fl / fma_peak, by / HBM_BPS
        print(f"B={B:5d} x {secs} s (T={T}): engine {te * 1e3:9.2f} ms = {n / te / 1e9:6.2f} Gsamples/s | "
              f"torch.stft fp32 restatement ({chunk}-row chunks) {tr * 1e3:9.2f} ms = {n / tr / 1e9:6.3f} Gsamples/s | "
              f"engine {tr / te:5.1f}x faster")
        print(f"    achieved {fl / 1e12:6.2f} TFLOP/s nominal = {100 * f_fma:5.1f} % of the FMA floor, {by / 1e9:7.1f} GB/s = "
              f"{100 * f_hbm:4.1f} % of the HBM floor -> the {'FMA' if f_fma >= f_hbm else 'HBM'} floor is the nearer bound")
        print(f"    loss engine {le:.9f}  fp32 restatement {l32:.9f}  float64 restatement {l64:.9f}  "
              f"|L-L64|/L64 {abs(le - l64) / abs(l64):.2e}  bound {'ok' if ok else 'FAILED'}", flush=True)
        del t, o
        torch.cuda.empty_cache()
    print("agreement check:", "passed" if ok_all else "FAILED")
    return 0 if ok_all else 1


if __name__ == "__main__":
    sys.exit(main())
