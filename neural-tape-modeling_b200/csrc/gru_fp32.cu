// Exact-fp32 persistent GRU kernel (CUDA cores) -- the parity anchor and the batch-1 real-time path.
//
// Replaces the per-timestep loop behind `self.GRU(x, self.hidden)` + `self.output(x)` of
// RNN.forward / DiffDelRNN.forward (code/model.py:81-82, :412-413; gate equations torch rnn.py:1221-1224).
// For DiffDelRNN it writes pre_d and the stand-alone delay line (delay.cu) runs behind it (capi.cu run_gru).
//
// Layout: one CTA owns S streams for ALL T timesteps (no per-step launch, no HBM round trip of the state).
//   - W_hh (192x64) lives in REGISTERS: thread (j, q) of 64*KS threads holds the three gate rows of hidden
//     unit j restricted to the k-slice q (3 * 64/KS floats), for the whole kernel.
//   - the hidden states of a chunk of CH steps are kept in a shared-memory ring (slot t = state before step t).
//     Every step each thread reads its k-slice of the current slot with broadcast LDS.128, does 3*64/KS FMAs
//     per stream, and the KS partial sums are combined with a transposing butterfly, so the KS lanes of a
//     hidden unit end up owning different streams and no activation is computed twice.  The only things on
//     the recurrence's critical path are: LDS -> FMA chain -> shuffles -> gates -> STS -> one barrier.
//   - the 64-wide output head is NOT in the step loop: at the end of a chunk it is evaluated for all CH steps
//     at once from the state ring (a [CH*S x 64] . [64] product), then flushed with coalesced stores.  x is staged
//     per chunk with cp.async (double-buffered).
#include "ntm_common.cuh"

namespace ntm {

namespace {

// Activations: libm-grade expf / tanhf (<= 2 ulp) and IEEE division.
__device__ __forceinline__ float sigmoid_f(float a) { return 1.0f / (1.0f + expf(-a)); }

template <int KS, int SP>
struct Transpose;   // combine the KS partial sums; lane q ends up owning streams i*KS + q

template <int SP>
struct Transpose<1, SP> {
    static __device__ __forceinline__ void run(const float (&acc)[SP], float (&own)[SP], int) {
#pragma unroll
        for (int i = 0; i < SP; ++i) own[i] = acc[i];
    }
};
template <int SP>
struct Transpose<2, SP> {
    static __device__ __forceinline__ void run(const float (&acc)[SP], float (&own)[SP / 2], int q) {
        const bool hi = q & 1;
#pragma unroll
        for (int i = 0; i < SP / 2; ++i) {
            const float keep = hi ? acc[2 * i + 1] : acc[2 * i];
            const float send = hi ? acc[2 * i] : acc[2 * i + 1];
            own[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
        }
    }
};
template <int SP>
struct Transpose<4, SP> {
    static __device__ __forceinline__ void run(const float (&acc)[SP], float (&own)[SP / 4], int q) {
        const bool b0 = q & 1, b1 = q & 2;
        float t1[SP / 2];
#pragma unroll
        for (int p = 0; p < SP / 2; ++p) {
            const float keep = b0 ? acc[2 * p + 1] : acc[2 * p];
            const float send = b0 ? acc[2 * p] : acc[2 * p + 1];
            t1[p] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
        }
#pragma unroll
        for (int i = 0; i < SP / 4; ++i) {
            const float keep = b1 ? t1[2 * i + 1] : t1[2 * i];
            const float send = b1 ? t1[2 * i] : t1[2 * i + 1];
            own[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
        }
    }
};

template <int KS, int S>
struct Cfg {
    static constexpr int NT = 64 * KS;             // threads
    static constexpr int NW = NT / 32;             // warps
    static constexpr int KK = 64 / KS;             // k values per thread
    static constexpr int HS = 64 + 32 / KS;        // smem row stride of one stream's state (conflict-free STS)
    static constexpr int SO = (S + KS - 1) / KS;   // streams owned per lane after the transpose
    static constexpr int SP = SO * KS;             // S padded to a multiple of KS
    static constexpr int CH = S >= 8 ? 32 : 64;    // steps per chunk (state ring depth)
    static constexpr int RING = (CH + 1) * S * HS; // floats
    static constexpr int SMEM_FLOATS = RING + 2 * S * CH + S * CH + 64;
    static constexpr int SMEM_BYTES = SMEM_FLOATS * 4;
};

template <int KS, int S>
__global__ void __launch_bounds__(64 * KS, 2) gru_fp32_kernel(const GruArgs a)
{
    using C = Cfg<KS, S>;
    constexpr int NT = C::NT, NW = C::NW, KK = C::KK, HS = C::HS, SO = C::SO, SP = C::SP, CH = C::CH;

    extern __shared__ __align__(16) float smem[];
    float* const hring = smem;                     // [CH+1][S][HS]
    float* const xs = hring + C::RING;             // [2][S][CH]
    float* const ys = xs + 2 * S * CH;             // [S][CH]
    float* const wos = ys + S * CH;                // [64]

    const int tid = threadIdx.x;
    const int j = tid / KS;              // hidden unit
    const int q = tid % KS;              // k-slice, later: owned-stream residue
    const int lane = tid & 31, warp = tid >> 5;
    const long long b0 = (long long)blockIdx.x * S;
    const int ns = (int)((a.B - b0) < (long long)S ? (a.B - b0) : (long long)S);

    // ---- parameters -> registers -------------------------------------------------------------
    const float* __restrict__ blob = a.blob;
    float w[3][KK];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int i = 0; i < KK / 4; ++i) {
            const float4 v = *reinterpret_cast<const float4*>(blob + BlobLayout::W_HH + (g * 64 + j) * 64 +
                                                              4 * (q + KS * i));
            w[g][4 * i + 0] = v.x; w[g][4 * i + 1] = v.y; w[g][4 * i + 2] = v.z; w[g][4 * i + 3] = v.w;
        }
    const float wir = blob[BlobLayout::W_IH + j], wiz = blob[BlobLayout::W_IH + 64 + j],
                win = blob[BlobLayout::W_IH + 128 + j];
    const float br = blob[BlobLayout::B_IH + j] + blob[BlobLayout::B_HH + j];
    const float bz = blob[BlobLayout::B_IH + 64 + j] + blob[BlobLayout::B_HH + 64 + j];
    const float bin = blob[BlobLayout::B_IH + 128 + j], bhn = blob[BlobLayout::B_HH + 128 + j];
    const float bo = blob[BlobLayout::B_OUT];
    if (tid < 64) wos[tid] = blob[BlobLayout::W_OUT + tid];

    // ---- initial state -> ring slot 0 ------------------------------------------------------------
    for (int idx = tid; idx < S * 64; idx += NT) {
        const int s = idx >> 6, k = idx & 63;
        hring[s * HS + k] = (s < ns && a.h_in) ? a.h_in[(b0 + s) * 64 + k] : 0.0f;
    }
    auto load_x = [&](int buf, long long t0) {
        const int n = (int)((a.T - t0) < (long long)CH ? (a.T - t0) : (long long)CH);
        for (int idx = tid; idx < S * CH; idx += NT) {
            const int s = idx / CH, tt = idx % CH;
            float* dst = xs + (buf * S + s) * CH + tt;
            if (s < ns && tt < n) cp_async4(dst, a.x + (b0 + s) * a.ldx + t0 + tt);
            else *dst = 0.0f;
        }
        cp_async_commit();
    };
    load_x(0, 0);
    __syncthreads();
    float hown[SO];
#pragma unroll
    for (int i = 0; i < SO; ++i) {
        const int s = i * KS + q;
        hown[i] = (s < S) ? hring[s * HS + j] : 0.0f;
    }

    const long long nchunks = (a.T + CH - 1) / CH;
    for (long long c = 0; c < nchunks; ++c) {
        const long long t0 = c * CH;
        const int n = (int)((a.T - t0) < (long long)CH ? (a.T - t0) : (long long)CH);
        const int xb = (int)(c & 1);
        const float* xcur = xs + xb * S * CH;
        cp_async_wait_all();
        __syncthreads();                       // xs[xb] landed; ring slot 0, ys and xs[xb^1] are free again
        if (c + 1 < nchunks) load_x(xb ^ 1, t0 + CH);

        for (int tt = 0; tt < n; ++tt) {
            const float* hcur = hring + tt * (S * HS);       // state before this step
            float* hnext = hring + (tt + 1) * (S * HS);
            // ---- partial mat-vec: 3 gate rows x k-slice, all S streams --------------------------
            float acc[3][SP];
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
                for (int s = 0; s < SP; ++s) acc[g][s] = 0.0f;
#pragma unroll
            for (int s = 0; s < S; ++s) {
#pragma unroll
                for (int i = 0; i < KK / 4; ++i) {
                    const float4 hv = *reinterpret_cast<const float4*>(hcur + s * HS + 4 * (q + KS * i));
#pragma unroll
                    for (int g = 0; g < 3; ++g) {
                        float v = acc[g][s];
                        v = fmaf(w[g][4 * i + 0], hv.x, v);
                        v = fmaf(w[g][4 * i + 1], hv.y, v);
                        v = fmaf(w[g][4 * i + 2], hv.z, v);
                        v = fmaf(w[g][4 * i + 3], hv.w, v);
                        acc[g][s] = v;
                    }
                }
            }
            float own[3][SO];
            Transpose<KS, SP>::run(acc[0], own[0], q);
            Transpose<KS, SP>::run(acc[1], own[1], q);
            Transpose<KS, SP>::run(acc[2], own[2], q);

            // ---- gates + state blend for the owned (j, stream) pairs --------------------------------
#pragma unroll
            for (int i = 0; i < SO; ++i) {
                const int s = i * KS + q;
                const bool live = s < S;             // padded lanes compute garbage in lock-step, store nothing
                const float xv = xcur[(live ? s : 0) * CH + tt];
                const float r = sigmoid_f(fmaf(wir, xv, br) + own[0][i]);
                const float z = sigmoid_f(fmaf(wiz, xv, bz) + own[1][i]);
                const float nn = tanhf(fmaf(r, own[2][i] + bhn, fmaf(win, xv, bin)));
                const float hn = fmaf(hown[i] - nn, z, nn);      // (h - n) * z + n
                hown[i] = hn;
                if (live) hnext[s * HS + j] = hn;
            }
            __syncthreads();                   // new state published
        }

        // ---- output head for the whole chunk: y[s][tt] = w_out . h(slot tt+1) + b (+ x) -----------------
        // half a warp reads one 64-float state row (conflict-free LDS.128), 16-lane shuffle reduction.
        {
            const int half = lane >> 4, l16 = lane & 15;
            const float4 wv = *reinterpret_cast<const float4*>(wos + 4 * l16);
            for (int row = warp * 2 + half; row < S * CH; row += NW * 2) {
                const int s = row / CH, tt = row % CH;
                const float4 hv = *reinterpret_cast<const float4*>(hring + (tt + 1) * (S * HS) + s * HS + 4 * l16);
                float p = fmaf(wv.x, hv.x, fmaf(wv.y, hv.y, fmaf(wv.z, hv.z, wv.w * hv.w)));
#pragma unroll
                for (int off = 8; off >= 1; off >>= 1) p += __shfl_xor_sync(0xffffffffu, p, off);
                if (l16 == 0 && tt < n) ys[s * CH + tt] = p + bo + (a.skip ? xcur[s * CH + tt] : 0.0f);
            }
        }
        __syncthreads();                       // ys complete; all reads of the ring done
        // carry: slot n becomes slot 0 of the next chunk
        if (n != 0) {
            for (int idx = tid; idx < S * 64; idx += NT) {
                const int s = idx >> 6, k = idx & 63;
                hring[s * HS + k] = hring[n * (S * HS) + s * HS + k];
            }
        }
        for (int idx = tid; idx < S * CH; idx += NT) {
            const int s = idx / CH, tt = idx % CH;
            if (s < ns && tt < n) a.y[(b0 + s) * a.ldy + t0 + tt] = ys[s * CH + tt];
        }
    }

    // ---- final state ------------------------------------------------------------------------------
#pragma unroll
    for (int i = 0; i < SO; ++i) {
        const int s = i * KS + q;
        if (s < ns) a.h_out[(b0 + s) * 64 + j] = hown[i];
    }
}

template <int KS, int S>
cudaError_t launch_one(const GruArgs& a, cudaStream_t st)
{
    using C = Cfg<KS, S>;
    static OncePerDevice once;
    cudaError_t e = once.run([] {
        return cudaFuncSetAttribute(gru_fp32_kernel<KS, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    });
    if (e != cudaSuccess) return e;
    const long long grid = (a.B + S - 1) / S;
    gru_fp32_kernel<KS, S><<<(unsigned)grid, C::NT, C::SMEM_BYTES, st>>>(a);
    ++g_launches;
    return cudaGetLastError();
}

}  // namespace

// streams: streams per CTA (1, 2, 4 or 8); ksplit: k-slices per hidden unit (2 with <= 2 streams per CTA, or 4)
cudaError_t launch_gru_fp32(const GruArgs& a, int streams, int ksplit, cudaStream_t st)
{
    if (a.B <= 0 || a.T <= 0) return cudaSuccess;
    if (a.d) return cudaErrorInvalidValue;          // plain GRU only
    if (ksplit == 2) {
        switch (streams) {
            case 1: return launch_one<2, 1>(a, st);
            case 2: return launch_one<2, 2>(a, st);
        }
    } else if (ksplit == 4) {
        switch (streams) {
            case 1: return launch_one<4, 1>(a, st);
            case 2: return launch_one<4, 2>(a, st);
            case 4: return launch_one<4, 4>(a, st);
            case 8: return launch_one<4, 8>(a, st);
        }
    }
    return cudaErrorInvalidValue;
}

}  // namespace ntm
