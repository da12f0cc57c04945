// Multi-resolution STFT loss on the device: per-row sums of auraloss `MultiResolutionSTFTLoss` (auraloss/freq.py, the third
// loss of the reference's evaluation loop, code/test-model.py:253) for (B, 1, T) output / target pairs.
//
// Per resolution (N, hop, win), for the row window of n samples: torch.stft(x, N, hop, win, hann_window(win)) with
// center=True -- F = 1 + n / hop frames, frame f starting at f hop - N/2, reflected at both ends of the window, the periodic
// Hann window of length win at offset (N - win) / 2 of the frame -- and the clamped magnitudes |X| = sqrt(max(re^2 + im^2,
// 1e-8)) of the N/2 + 1 one-sided bins.  The kernel returns four double sums per (row, resolution):
//     s0 = sum (|Y| - |X|)^2    s1 = sum |Y|^2    s2 = sum |ln|X| - ln|Y||    s3 = sum ||X| - |Y||
// from which the caller forms SC = sqrt(s0) / sqrt(s1), LogMag = s2 / (F (N/2 + 1)) and LinMag = s3 / (F (N/2 + 1)).
//
// One fused pass per resolution; the spectrogram never leaves the SM.  A CTA of 256 threads owns work items of (row, block of
// consecutive frames) and transforms PASS_POINTS complex points per signal at a time (2048 / (N/2) frames).  Each signal's
// frame goes through the usual real FFT: the N/2-point complex FFT of z[m] = x[2m] + i x[2m+1] and the split
// X[k] = (Z[k] + conj Z[N/2-k]) / 2 + W_N^k (Z[k] - conj Z[N/2-k]) / 2i.  Output and target run through the same code, so
// loss(t, t) is exactly 0.  (Packing the two signals into one complex FFT would halve the transforms but give X and Y from
// different formulas.)  The complex FFT is a Stockham autosort of radix-8 stages and one radix-2/4 stage, in place in
// shared memory: every thread loads its butterflies' points into registers, the CTA synchronises, then every thread stores.
// The first stage reads the row straight from global memory (reflection and window applied on load; the frames of a block
// overlap win / hop times, so the re-reads hit L1).  Twiddles and the window come from per-CTA shared-memory tables built
// in double (sincospi), i.e. accurate to fp32 rounding.  Partial sums are fp32 within a pass and double across passes; one
// double atomicAdd per item and sum.
#include <math.h>

#include "ntm_common.cuh"

namespace ntm {

namespace {

// 256 threads, 2 CTAs per SM (__launch_bounds__): 128 registers and no spills; a bound of 3 CTAs (80 registers) spills at N >= 1024
constexpr int STFT_THREADS = 256;
constexpr int PASS_POINTS = 2048;                          // complex points per signal and pass
constexpr int BUF_POINTS = 2 * PASS_POINTS;                // both signals
constexpr int STFT_MAX_PASSES = 8;                         // passes per work item, at most

// shared-memory index of complex point i: one float2 of padding per 16 breaks the power-of-two strides of the Stockham stores
__device__ __forceinline__ int padi(int i) { return i + (i >> 4); }
constexpr int BUF_FLOAT2 = BUF_POINTS + BUF_POINTS / 16;

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b)
{
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float2 mul_mi(float2 a) { return make_float2(a.y, -a.x); }   // -i a

// forward DFTs (exp(-2 pi i q r / R)) of R points in registers, natural order in and out
__device__ __forceinline__ void dft(float2 (&v)[2])
{
    const float2 a = v[0];
    v[0] = cadd(a, v[1]);
    v[1] = csub(a, v[1]);
}
__device__ __forceinline__ void dft4(float2& a0, float2& a1, float2& a2, float2& a3)
{
    const float2 s02 = cadd(a0, a2), d02 = csub(a0, a2), s13 = cadd(a1, a3), d13 = mul_mi(csub(a1, a3));
    a0 = cadd(s02, s13);
    a2 = csub(s02, s13);
    a1 = cadd(d02, d13);
    a3 = csub(d02, d13);
}
__device__ __forceinline__ void dft(float2 (&v)[4]) { dft4(v[0], v[1], v[2], v[3]); }
__device__ __forceinline__ void dft(float2 (&v)[8])
{
    float2 e0 = v[0], e1 = v[2], e2 = v[4], e3 = v[6], o0 = v[1], o1 = v[3], o2 = v[5], o3 = v[7];
    dft4(e0, e1, e2, e3);
    dft4(o0, o1, o2, o3);
    constexpr float H = 0.70710678118654752f;               // W_8 = (H, -H)
    o1 = make_float2(H * (o1.x + o1.y), H * (o1.y - o1.x));
    o2 = mul_mi(o2);
    o3 = make_float2(-H * (o3.x - o3.y), -H * (o3.x + o3.y));
    v[0] = cadd(e0, o0); v[4] = csub(e0, o0);
    v[1] = cadd(e1, o1); v[5] = csub(e1, o1);
    v[2] = cadd(e2, o2); v[6] = csub(e2, o2);
    v[3] = cadd(e3, o3); v[7] = csub(e3, o3);
}

// W_N^e for 0 <= e < N from the table of W_N^m, m < N/2 (W_N^(m + N/2) = -W_N^m)
template <int M>
__device__ __forceinline__ float2 twiddle(const float2* tw, int e)
{
    const float2 w = tw[e & (M - 1)];
    return e < M ? w : make_float2(-w.x, -w.y);
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    return v;
}

// Row context of one work item: the rows of both signals at the window start, the window length and the first frame.
struct ItemCtx {
    const float* x[2];     // output, target
    long long n;           // samples in the row window
    long long frames;      // F = 1 + n / hop
    long long f0;          // first frame of this pass
};

// Sample i (0 <= i < N) of the frame whose window starts at row sample ws (= frame start + (N - win) / 2), windowed; 0
// outside the window.  edge: the window reaches past an end of the row window and the index is reflected.
__device__ __forceinline__ float frame_sample(const float* x, long long n, long long ws, int wi, int win, bool edge,
                                              const float* hann)
{
    if (wi < 0 || wi >= win) return 0.0f;
    long long p = ws + wi;
    if (edge) {
        p = p < 0 ? -p : p;
        p = p >= n ? 2 * (n - 1) - p : p;                  // n > N/2: one reflection suffices
    }
    return hann[wi] * __ldg(x + p);
}

// One Stockham stage of radix R after NS points (the product of the earlier radices); FIRST: the input comes from the rows.
template <int N, int R, int NS, bool FIRST>
__device__ __forceinline__ void fft_stage(float2* buf, const float2* tw, const ItemCtx& c, int hop, int win, const float* hann)
{
    constexpr int M = N / 2, FP = PASS_POINTS / M, QS = M / R;         // frames per pass, butterflies per frame
    constexpr int PER_THREAD = BUF_POINTS / R / STFT_THREADS;
    float2 v[PER_THREAD][R];
    int base[PER_THREAD], j[PER_THREAD];
#pragma unroll
    for (int u = 0; u < PER_THREAD; ++u) {
        const int g = threadIdx.x + u * STFT_THREADS;
        const int s = g / (FP * QS), f = (g / QS) % FP;
        j[u] = g % QS;
        base[u] = s * PASS_POINTS + f * M;
        if (FIRST) {
            const int off = (N - win) / 2;
            const long long ws = (c.f0 + f) * hop - N / 2 + off;
            const bool live = c.f0 + f < c.frames, edge = ws < 0 || ws + win > c.n;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int wi = 2 * (j[u] + r * QS) - off;
                v[u][r] = live ? make_float2(frame_sample(c.x[s], c.n, ws, wi, win, edge, hann),
                                             frame_sample(c.x[s], c.n, ws, wi + 1, win, edge, hann))
                               : make_float2(0.0f, 0.0f);
            }
        } else {
#pragma unroll
            for (int r = 0; r < R; ++r) v[u][r] = buf[padi(base[u] + j[u] + r * QS)];
        }
    }
    if (!FIRST) __syncthreads();                            // every point of the stage is in registers: store in place
#pragma unroll
    for (int u = 0; u < PER_THREAD; ++u) {
        const int k = j[u] & (NS - 1);
        if (NS > 1) {
            const int e = k * (2 * M / (NS * R));           // in units of W_N
#pragma unroll
            for (int r = 1; r < R; ++r) v[u][r] = cmul(v[u][r], twiddle<M>(tw, e * r));
        }
        dft(v[u]);
        const int d = base[u] + (j[u] - k) * R + k;
#pragma unroll
        for (int r = 0; r < R; ++r) buf[padi(d + r * NS)] = v[u][r];
    }
    __syncthreads();
}

template <int N, int NS = 1>
__device__ __forceinline__ void fft_stages(float2* buf, const float2* tw, const ItemCtx& c, int hop, int win, const float* hann)
{
    constexpr int M = N / 2, R = M / NS >= 8 ? 8 : M / NS;
    fft_stage<N, R, NS, NS == 1>(buf, tw, c, hop, win, hann);
    if constexpr (NS * R < M) fft_stages<N, NS * R>(buf, tw, c, hop, win, hann);
}

// |X[k]|^2 from Z[k] = a, Z[N/2 - k] = b and W_N^k = w (the real-FFT split)
__device__ __forceinline__ float split_power(float2 a, float2 b, float2 w)
{
    const float2 ze = make_float2(0.5f * (a.x + b.x), 0.5f * (a.y - b.y));
    const float2 zo = make_float2(0.5f * (a.y + b.y), -0.5f * (a.x - b.x));
    const float2 x = cadd(ze, cmul(w, zo));
    return fmaf(x.x, x.x, x.y * x.y);
}

struct Partial {
    float sq, ref, lg, ab;
    __device__ __forceinline__ void add(float px, float py)
    {
        px = fmaxf(px, 1e-8f);
        py = fmaxf(py, 1e-8f);
        const float d = sqrtf(py) - sqrtf(px);             // two square roots: p_X + p_Y - 2 sqrt(p_X p_Y) cancels
        sq = fmaf(d, d, sq);
        ref += py;
        lg += fabsf(logf(px / py));                         // = 2 |ln|X| - ln|Y||
        ab += fabsf(d);
    }
};

template <int N>
__global__ void __launch_bounds__(STFT_THREADS, 2) stft_loss_kernel(const float* __restrict__ out, long long ldo,
                                                                 const float* __restrict__ tgt, long long ldt, long long B,
                                                                 long long T, const long long* __restrict__ first,
                                                                 const long long* __restrict__ count, int hop, int win,
                                                                 int passes, long long items_per_row, int res, int n_res,
                                                                 double* __restrict__ sums)
{
    constexpr int M = N / 2, FP = PASS_POINTS / M;
    extern __shared__ __align__(16) unsigned char smem[];
    float2* buf = reinterpret_cast<float2*>(smem);
    float2* tw = buf + BUF_FLOAT2;
    float* hann = reinterpret_cast<float*>(tw + M);
    __shared__ double red[STFT_THREADS / 32][4];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int m = tid; m < M; m += STFT_THREADS) {
        double s, c;
        sincospi(-2.0 * m / N, &s, &c);
        tw[m] = make_float2((float)c, (float)s);
    }
    for (int i = tid; i < win; i += STFT_THREADS) {
        const double s = sinpi((double)i / win);            // periodic Hann: 0.5 - 0.5 cos(2 pi i / win) = sin^2(pi i / win)
        hann[i] = (float)(s * s);
    }
    __syncthreads();

    for (long long item = blockIdx.x; item < B * items_per_row; item += gridDim.x) {
        const long long b = item / items_per_row, blk = item % items_per_row;
        // row window [first[b], first[b] + count[b]), clipped to the row (as esr.cu); reflection is relative to it
        long long w0 = first ? first[b] : 0;
        w0 = w0 < 0 ? 0 : (w0 > T ? T : w0);
        long long n = T - w0;
        if (count) { const long long cn = count[b]; n = cn < 0 ? 0 : (cn < n ? cn : n); }
        double* row_sums = sums + (b * n_res + res) * 4;
        if (n <= N / 2) {                                   // torch.stft raises here; the host cannot see device counts
            if (blk == 0 && tid < 4) atomicAdd(row_sums + tid, __longlong_as_double(0x7ff8000000000000ll));
            continue;
        }
        ItemCtx c;
        c.x[0] = out + b * ldo + w0;
        c.x[1] = tgt + b * ldt + w0;
        c.n = n;
        c.frames = 1 + n / hop;
        const long long fb = blk * (long long)(FP * passes);
        if (fb >= c.frames) continue;
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        for (int p = 0; p < passes; ++p) {
            c.f0 = fb + (long long)p * FP;
            if (c.f0 >= c.frames) break;                    // (CTA-uniform)
            fft_stages<N>(buf, tw, c, hop, win, hann);
            Partial q{0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
            for (int u = 0; u < PASS_POINTS / STFT_THREADS; ++u) {
                const int e = tid + u * STFT_THREADS, f = e / M, k = e % M;
                if (c.f0 + f >= c.frames) continue;
                const int i0 = f * M + k, i1 = f * M + ((M - k) & (M - 1));
                const float2 ax = buf[padi(i0)], bx = buf[padi(i1)];
                const float2 ay = buf[padi(PASS_POINTS + i0)], by = buf[padi(PASS_POINTS + i1)];
                const float2 w = tw[k];
                q.add(split_power(ax, bx, w), split_power(ay, by, w));
                if (k == 0) {                               // bin N/2 = Re Z[0] - Im Z[0]
                    const float nx = ax.x - ax.y, ny = ay.x - ay.y;
                    q.add(nx * nx, ny * ny);
                }
            }
            acc[0] += (double)q.sq;
            acc[1] += (double)q.ref;
            acc[2] += 0.5 * (double)q.lg;
            acc[3] += (double)q.ab;
            __syncthreads();                                // the next pass overwrites buf
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const double v = warp_sum(acc[i]);
            if (lane == 0) red[warp][i] = v;
        }
        __syncthreads();
        if (tid < 4) {
            double v = 0.0;
#pragma unroll
            for (int w = 0; w < STFT_THREADS / 32; ++w) v += red[w][tid];
            atomicAdd(row_sums + tid, v);
        }
    }
}

template <int N>
cudaError_t launch_one(const float* out, long long ldo, const float* tgt, long long ldt, long long B, long long T,
                       const long long* first, const long long* count, int hop, int win, int res, int n_res, double* sums,
                       int sm_count, cudaStream_t st)
{
    constexpr int M = N / 2, FP = PASS_POINTS / M;
    const size_t smem = sizeof(float2) * (BUF_FLOAT2 + M) + sizeof(float) * N;      // window table sized for win = N
    static OncePerDevice configured;
    cudaError_t e = configured.run([&] {
        return cudaFuncSetAttribute(stft_loss_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    });
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, stft_loss_kernel<N>, STFT_THREADS, smem);
    if (e != cudaSuccess) return e;
    const long long resident = (long long)sm_count * (per_sm > 0 ? per_sm : 1);
    // fewer passes per item only when the rows are too few to fill the GPU; more passes amortise the table set-up
    const long long frames = 1 + T / hop;
    int passes = STFT_MAX_PASSES;
    auto items = [&] { return (frames + (long long)FP * passes - 1) / ((long long)FP * passes); };
    while (passes > 1 && B * items() < 2 * resident) passes >>= 1;
    const long long per_row = items();
    const long long grid = B * per_row < resident ? B * per_row : resident;
    stft_loss_kernel<N><<<(unsigned)grid, STFT_THREADS, smem, st>>>(out, ldo, tgt, ldt, B, T, first, count, hop, win, passes,
                                                                     per_row, res, n_res, sums);
    ++g_launches;
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_stft_loss(const float* out, long long ldo, const float* tgt, long long ldt, long long B, long long T,
                             const long long* first, const long long* count, int n_res, const int* fft_sizes,
                             const int* hop_sizes, const int* win_lengths, double* sums, int sm_count, cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * 4 * (size_t)B * (size_t)n_res, st);
    if (e != cudaSuccess || B <= 0 || T <= 0) return e;
    for (int r = 0; r < n_res && e == cudaSuccess; ++r) {
        const int hop = hop_sizes[r], win = win_lengths[r];
        switch (fft_sizes[r]) {
            case 256: e = launch_one<256>(out, ldo, tgt, ldt, B, T, first, count, hop, win, r, n_res, sums, sm_count, st); break;
            case 512: e = launch_one<512>(out, ldo, tgt, ldt, B, T, first, count, hop, win, r, n_res, sums, sm_count, st); break;
            case 1024: e = launch_one<1024>(out, ldo, tgt, ldt, B, T, first, count, hop, win, r, n_res, sums, sm_count, st); break;
            case 2048: e = launch_one<2048>(out, ldo, tgt, ldt, B, T, first, count, hop, win, r, n_res, sums, sm_count, st); break;
            case 4096: e = launch_one<4096>(out, ldo, tgt, ldt, B, T, first, count, hop, win, r, n_res, sums, sm_count, st); break;
            default: return cudaErrorInvalidValue;
        }
    }
    return e;
}

}  // namespace ntm
