// Stand-alone time-varying fractional delay line (HBM-bound elementwise gather).
// Replaces TimeVaryingDelayLine.forward, code/model.py:269-320, as used on its own by apply_delay
// (code/test-model.py:259-290).  The reference materialises three (B,1,T,D+1) temporaries; here every
// output sample reads two past samples (history or this call's input) -- 12 algorithmic bytes per sample.
#include "ntm_common.cuh"

namespace ntm {

namespace {

// VEC: rows of d and y are 16-byte aligned (base and leading dimension): a thread owns DELAY_SPT consecutive samples,
// loads their delays with 16-byte loads, issues its tap gathers as independent instructions, and stores 16 bytes at a time.
// History of this kernel (1024 x 1 440 000 samples, D = 365; the copy peak of this GPU is 6.54 TB/s, a plain two-reads-one-write
// elementwise pass -- torch.add -- reaches 6.97; profiles/r02f_delay_line.txt):
//   one sample per thread                         2.44 TB/s   d -> index -> x -> y is a dependent chain with 4 bytes in flight per thread
//   8 samples per thread, 16 independent gathers  4.63-4.72   (lane-strided samples: 2.57; shared-memory staging of d and the reachable
//                                                             x window with double-buffered cp.async: 4.66, 3.9 at D = 2000 -- dropped)
//   + second tap reused from the neighbour sample 5.20        9 gathers per thread instead of 16: the gathers cost L1 passes
//   + 32 groups per thread, next delays prefetched 6.38       few long-lived CTAs instead of one CTA per 2048 samples
constexpr int DELAY_SPT = 8;
// Few, long-lived CTAs: a thread walks over up to DELAY_ITER groups of its row (a grid stride apart) and loads the delays of its next
// group before it gathers the taps of the current one -- one exposed HBM round trip per group instead of two dependent ones, and
// no CTA launch per 2048 samples.  Measured at 1024 x 1 440 000, D = 365 (profiles/r02f_delay_line.txt): 4.63 TB/s with one group
// per thread, 5.20 with the tap reuse below, 5.85 / 6.07 / 6.18 / 6.36 at 4 / 8 / 16 / 32 groups per thread.  Small problems keep one
// group per thread (the launcher never drops below DELAY_MIN_CTAS_PER_SM CTAs per SM).
constexpr int DELAY_ITER = 32;
constexpr int DELAY_MIN_CTAS_PER_SM = 12;

template <bool VEC>
__global__ void __launch_bounds__(256, 3) delay_kernel(const float* __restrict__ x, long long ldx,
                                                    const float* __restrict__ d, long long ldd,
                                                    float* __restrict__ y, long long ldy,
                                                    const float* __restrict__ hist_in, long long B, long long T,
                                                    int D, int warmup)
{
    const long long b = blockIdx.y;
    const float* xr = x + b * ldx;
    const float* hr = hist_in + b * (long long)D;
    const float* dr = d + b * ldd;
    float* yr = y + b * ldy;
    auto past = [&](long long i) { return i >= 0 ? __ldg(xr + i) : __ldg(hr + D + i); };
    {
        // VEC: this row's d (x in warm-up mode) and y share their position inside a 16-byte line (the launcher checked it); the
        // first `head` samples up to the line boundary and the last (T - head) % DELAY_SPT go through the scalar tail below
        const int head = VEC ? (int)((4 - ((reinterpret_cast<uintptr_t>(warmup ? xr : dr) >> 2) & 3)) & 3) : 0;
        const int groups = T > head ? (int)((T - head) / DELAY_SPT) : 0;       // (the launcher keeps T below 2^34)
        const float4* __restrict__ src4 = reinterpret_cast<const float4*>((warmup ? xr : dr) + head);   // (VEC only)
        const int stride = (int)(gridDim.x * blockDim.x);
        int gq = (int)(blockIdx.x * blockDim.x + threadIdx.x);
        static_assert(DELAY_SPT == 8, "two float4 of delays per group");
        float4 dn0 = make_float4(0.0f, 0.0f, 0.0f, 0.0f), dn1 = dn0;
        if (VEC && gq < groups) {
            dn0 = __ldg(src4 + 2ll * gq);
            dn1 = __ldg(src4 + 2ll * gq + 1);
        }
        for (; gq < groups; gq += stride) {
            const long long t = head + (long long)gq * DELAY_SPT;
            float dv[DELAY_SPT], v[DELAY_SPT];
            if (VEC) {
                dv[0] = dn0.x; dv[1] = dn0.y; dv[2] = dn0.z; dv[3] = dn0.w; dv[4] = dn1.x; dv[5] = dn1.y; dv[6] = dn1.z; dv[7] = dn1.w;
                if (gq < groups - stride) {
                    dn0 = __ldg(src4 + 2ll * (gq + stride));
                    dn1 = __ldg(src4 + 2ll * (gq + stride) + 1);
                }
            } else {                                              // rows not 16-byte aligned: same grouping, 4-byte accesses
#pragma unroll
                for (int j = 0; j < DELAY_SPT; ++j) dv[j] = __ldg((warmup ? xr : dr) + t + j);
            }
            if (!warmup) {
                // the arithmetic of delay_read (ntm_common.cuh) in three passes: tap weights and addresses, loads, sums.
                // A tap outside j in [0, D] gets weight 0 and a harmless address (adding an exact zero = skipping the tap).
                float w[DELAY_SPT][2], p[DELAY_SPT][2];
                int off[DELAY_SPT][2];                            // tap address relative to x[t] (32-bit: fewer registers, more
                                                                  // resident threads = more bytes in flight)
#pragma unroll
                for (int j = 0; j < DELAY_SPT; ++j) {
                    const float fl = floorf(dv[j]);
#pragma unroll
                    for (int tap = 0; tap < 2; ++tap) {
                        const float jf = fl + (float)tap;
                        const bool ok = jf >= 0.0f && jf <= (float)D;
                        w[j][tap] = ok ? fmaxf(__fsub_rn(1.0f, fabsf(__fsub_rn(jf, dv[j]))), 0.0f) : 0.0f;
                        off[j][tap] = ok ? j - (int)jf : j;
                    }
                }
                const float* xt = xr + t;
                if (t > (long long)D) {                           // no tap of this group can reach the carried history
#pragma unroll
                    for (int j = 0; j < DELAY_SPT; ++j) p[j][0] = __ldg(xt + off[j][0]);
                    // the second tap of sample j is the first tap of sample j - 1 whenever both delays have the same integer
                    // part (x[t + j - fl - 1] either way): the load is predicated off then -- 9 gathers per thread instead of
                    // 16 on a smooth trajectory, same values
                    p[0][1] = __ldg(xt + off[0][1]);
#pragma unroll
                    for (int j = 1; j < DELAY_SPT; ++j)
                        p[j][1] = off[j][1] == off[j - 1][0] ? p[j - 1][0] : __ldg(xt + off[j][1]);
                } else {
                    const float* ht = hr + D + t;
#pragma unroll
                    for (int j = 0; j < DELAY_SPT; ++j) {
                        p[j][0] = __ldg((t + off[j][0] >= 0 ? xt : ht) + off[j][0]);
                        p[j][1] = __ldg((t + off[j][1] >= 0 ? xt : ht) + off[j][1]);
                    }
                }
#pragma unroll
                for (int j = 0; j < DELAY_SPT; ++j)
                    v[j] = __fadd_rn(__fadd_rn(0.0f, __fmul_rn(w[j][1], p[j][1])), __fmul_rn(w[j][0], p[j][0]));
            } else {
#pragma unroll
                for (int j = 0; j < DELAY_SPT; ++j) v[j] = dv[j];
            }
            if (VEC) {
#pragma unroll
                for (int q = 0; q < DELAY_SPT / 4; ++q)
                    reinterpret_cast<float4*>(yr + t)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < DELAY_SPT; ++j) yr[t + j] = v[j];
            }
        }
        // the samples in front of the first group and the ragged tail, by the first block
        if (blockIdx.x == 0) {
            const long long t = (int)threadIdx.x < head ? (long long)threadIdx.x : (long long)groups * DELAY_SPT + threadIdx.x;
            if (t < T) yr[t] = warmup ? xr[t] : delay_read(dr[t], t, D, past);
        }
    }
}

// new history = last D samples of (history || x), any T (code/model.py:314-315)
__global__ void __launch_bounds__(256) roll_history_kernel(const float* __restrict__ x, long long ldx,
                                                           const float* __restrict__ hist_in,
                                                           float* __restrict__ hist_out, long long T, int D)
{
    const long long b = blockIdx.y;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < D;
         i += (long long)gridDim.x * blockDim.x) {
        const long long src = T - D + i;
        hist_out[b * D + i] = src >= 0 ? x[b * ldx + src] : hist_in[b * D + D + src];
    }
}

__global__ void __launch_bounds__(256) delay_check_kernel(const float* __restrict__ d, long long ldd, long long T,
                                                          float Dmax, int* flag)
{
    const long long b = blockIdx.y;
    bool bad = false;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < T;
         t += (long long)gridDim.x * blockDim.x)
        bad |= !(d[b * ldd + t] <= Dmax);      // (NaN trips the check like the reference's assert, code/model.py:283)
    if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(flag, 1);
}

int sm_count()          // of the current device
{
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
        return 148;
    return n;
}

unsigned grid_x(long long n)
{
    long long g = (n + 255) / 256;
    if (g > 2048) g = 2048;
    if (g < 1) g = 1;
    return (unsigned)g;
}

}  // namespace

cudaError_t launch_delay(const float* x, long long ldx, const float* d, long long ldd, float* y, long long ldy,
                         const float* hist_in, float* hist_out, long long B, long long T, long long D, int warmup,
                         cudaStream_t st)
{
    if (B <= 0) return cudaSuccess;
    if (T >= (1ll << 33)) return cudaErrorInvalidValue;      // 32-bit group indices inside the kernel (2^33 samples = 2 days of audio per row)
    for (long long b0 = 0; b0 < B; b0 += 65535) {       // gridDim.y limit
        const long long nb = (B - b0) < 65535 ? (B - b0) : 65535;
        if (T > 0) {
            // warm-up copies x -> y: then x takes d's place in the alignment test
            const float* src = warmup ? x : d;
            const long long lds = warmup ? ldx : ldd;
            // 16-byte accesses need every row's src and y at the same position inside a 16-byte line (any position: the
            // kernel peels up to three samples in front)
            const bool vec = ((((unsigned long long)(src + b0 * lds)) ^ ((unsigned long long)(y + b0 * ldy))) & 15ull) == 0 &&
                             (nb == 1 || ((lds - ldy) & 3) == 0);
            // x-blocks per row: DELAY_ITER groups per thread, but at least DELAY_MIN_CTAS_PER_SM CTAs per SM over all rows and at
            // most one thread per group
            const long long per_row = (T / DELAY_SPT + 255) / 256;
            long long want = (per_row + DELAY_ITER - 1) / DELAY_ITER;
            const long long floor_ctas = ((long long)sm_count() * DELAY_MIN_CTAS_PER_SM + nb - 1) / nb;
            if (want < floor_ctas) want = floor_ctas;
            if (want > per_row) want = per_row;
            if (want < 1) want = 1;
            const dim3 grid(grid_x(want * 256), (unsigned)nb);
            if (vec)
                delay_kernel<true><<<grid, 256, 0, st>>>(x + b0 * ldx, ldx, d + b0 * ldd, ldd, y + b0 * ldy, ldy,
                                                         hist_in + b0 * D, nb, T, (int)D, warmup);
            else
                delay_kernel<false><<<grid, 256, 0, st>>>(x + b0 * ldx, ldx, d + b0 * ldd, ldd, y + b0 * ldy, ldy,
                                                          hist_in + b0 * D, nb, T, (int)D, warmup);
            ++g_launches;
        }
        if (D > 0) {
            roll_history_kernel<<<dim3(grid_x(D), (unsigned)nb), 256, 0, st>>>(x + b0 * ldx, ldx, hist_in + b0 * D,
                                                                                hist_out + b0 * D, T, (int)D);
            ++g_launches;
        }
    }
    return cudaGetLastError();
}

cudaError_t launch_delay_check(const float* d, long long ldd, long long B, long long T, long long D, int* flag_dev,
                               cudaStream_t st)
{
    if (B <= 0 || T <= 0) return cudaSuccess;
    for (long long b0 = 0; b0 < B; b0 += 65535) {
        const long long nb = (B - b0) < 65535 ? (B - b0) : 65535;
        delay_check_kernel<<<dim3(grid_x(T), (unsigned)nb), 256, 0, st>>>(d + b0 * ldd, ldd, T, (float)D, flag_dev);
        ++g_launches;
    }
    return cudaGetLastError();
}

}  // namespace ntm
