// Shared declarations of the engine's translation units (internal; the public ABI is include/ntm_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

namespace ntm {

constexpr int H64 = 64;      // hidden size all shipped checkpoints use (SURVEY.md section 2.1 #16)
constexpr int G192 = 192;    // 3 gates x 64, row order r,z,n (torch rnn.py:1221-1224)

// Device parameter blob (floats), written once by ntm_gru_prepare.
struct BlobLayout {
    static constexpr int W_HH = 0;                    // 192 x 64, PyTorch layout
    static constexpr int W_IH = W_HH + G192 * H64;    // 192
    static constexpr int B_IH = W_IH + G192;          // 192
    static constexpr int B_HH = B_IH + G192;          // 192
    static constexpr int W_OUT = B_HH + G192;         // 64
    static constexpr int B_OUT = W_OUT + H64;         // 1 (0 when the head has no bias)
    static constexpr int FP32_END = B_OUT + 4;
    // B-operand images of the stream-major tcgen05 kernel (gru_tcs.cu, pack_tc_images): row n = gate * 64 + unit (192
    // rows), k contiguous, rows pre-scaled by -log2 e (r, z) / 2 log2 e (n); one image per operand format:
    //   f16, bf16   80 k of 2 bytes: W_hh row | the K augmentation carrying W_i x + b (see gru_tcs.cu)
    //   f16x3       192 k of 2 bytes (strict): G W_hi | G W_hi / 2^8 | (G W)_lo, G = TcsConsts::gain
    //   tf32        64 k of 4 bytes
    static constexpr int IMG_F16 = FP32_END;
    static constexpr int IMG_BF16 = IMG_F16 + 192 * 80 / 2;
    static constexpr int IMG_F16X3 = IMG_BF16 + 192 * 80 / 2;
    static constexpr int IMG_TF32 = IMG_F16X3 + 192 * 192 / 2;
    static constexpr int TOTAL = IMG_TF32 + 192 * 64;
    __host__ __device__ static constexpr int tc_image(int fmt)
    {
        return fmt == 1 ? IMG_BF16 : fmt == 2 ? IMG_TF32 : fmt == 3 ? IMG_F16X3 : IMG_F16;
    }
};
static_assert(BlobLayout::FP32_END % 4 == 0, "tensor-core images must stay 16-byte aligned");

// Mailbox of a real-time stream (ntm_rt_*, ntm_rt_diffdel_*): page-locked, mapped host memory shared by the host thread and
// the resident server kernel (gru_mma.cu, RT form).  The host writes a block into x (DiffDelRNN: and its delay trajectory
// into d), then bumps seq_in; the kernel writes y (DiffDelRNN: and the head output before the delay into pre), then sets
// seq_out = seq_in.  seq_in == RT_STOP ends the kernel.  An RNN stream leaves d and pre unused.
constexpr int RT_MAXBLK = 256;          // samples per block, at most
constexpr int RT_MAXSTREAMS = 4;
constexpr unsigned RT_STOP = 0xffffffffu;
struct RtMailbox {
    volatile unsigned seq_in;
    unsigned pad0[31];
    float x[RT_MAXSTREAMS][RT_MAXBLK];
    float d[RT_MAXSTREAMS][RT_MAXBLK];
    volatile unsigned seq_out;
    unsigned pad1[31];
    float y[RT_MAXSTREAMS][RT_MAXBLK];
    float pre[RT_MAXSTREAMS][RT_MAXBLK];
};

// Arguments of one recurrent launch; d == nullptr selects the plain RNN.forward path.
struct GruArgs {
    const float* blob;
    const float* x;
    float* y;
    const float* h_in;      // B x 64 or nullptr (zero state)
    float* h_out;           // B x 64 (may alias h_in)
    const float* d;         // delay trajectory (samples) or nullptr
    float* pre;             // GRU head output before the delay (DiffDelRNN only)
    const float* hist_in;   // B x D
    float* hist_out;        // B x D
    long long B, T, ldx, ldy, ldd, ldp;
    int D;
    int warmup;
    int skip;
    int ring_len;                   // DiffDelRNN, mma.sync kernels: samples of pre_d kept per stream in shared memory
                                    // (delay_ring_len; capi.cu chooses it)
    int sm_count;                   // SMs of the handle's device (host-side dispatch only)
    RtMailbox* rt;                  // real-time server forms only (x, y and, DiffDelRNN, d, pre point into it)
    unsigned long long rt_idle_ns;  // the server leaves after this long without a block
};

// Warp-uniform per-unit constants of the stream-major tcgen05 kernel (gru_tcs.cu); passed as a kernel parameter so
// that they are constant-bank operands.  Scaled like the gate rows they belong to (-log2 e for r, z; 2 log2 e for n).
struct TcsConsts {
    float cn_w[64];   // W_in
    float cn_b[64];   // b_in
    float wo[64];     // output head
    // operand formats without the K augmentation (strict f16x3, tf32): input projection and biases are added in fp32
    float cr_w[64], cr_b[64];   // W_ir, b_ir + b_hr
    float cz_w[64], cz_b[64];   // W_iz, b_iz + b_hz
    float ch_b[64];             // b_hn
    float bo;
    float gain_inv;             // strict form: the weight image is scaled by the power of two `gain` (f16 range), 1 / gain
};

// per-TU launchers -------------------------------------------------------------------------------
// The launchers run exactly the configuration they are given (capi.cu resolve_launch chooses it).  Only the mma.sync
// launchers have a DiffDelRNN form (a.d != nullptr, with a.ring_len set); the others run the plain GRU.
cudaError_t launch_gru_fp32(const GruArgs& a, int streams, int ksplit, cudaStream_t st);
cudaError_t launch_gru_tcs(const GruArgs& a, const TcsConsts& kc, int fmt, int sm_count, int tiles, bool static_schedule,
                           cudaStream_t st);
void fill_tcs_consts(const float* blob_host, TcsConsts* kc);
cudaError_t launch_gru_mma(const GruArgs& a, int fmt, int streams, bool defer_head, cudaStream_t st);
cudaError_t launch_gru_mma4(const GruArgs& a, int fmt, cudaStream_t st);   // GRU and DiffDelGRU, f16 / bf16 / strict f16x3, four
                                                                             // streams per CTA, 4x unrolled
// Resident real-time server, <= 4 streams; a.d != nullptr selects its DiffDelRNN form.
cudaError_t launch_gru_mma_rt(const GruArgs& a, int fmt, cudaStream_t st);
void pack_tc_images(float* blob_host);   // host: fills BlobLayout::IMG_* from the fp32 part of the blob
cudaError_t launch_delay(const float* x, long long ldx, const float* d, long long ldd, float* y, long long ldy,
                         const float* hist_in, float* hist_out, long long B, long long T, long long D, int warmup,
                         cudaStream_t st);
cudaError_t launch_delay_check(const float* d, long long ldd, long long B, long long T, long long D, int* flag_dev,
                               cudaStream_t st);

// 16-bit host transport: n elements (a multiple of 8), 16-byte aligned buffers
cudaError_t launch_half_to_float(const void* src, float* dst, long long n, int sm_count, cudaStream_t st);
cudaError_t launch_float_to_half(const float* src, void* dst, long long n, int sm_count, cudaStream_t st);

// per_row == 0: sums[2] over all B x T samples; per_row != 0: sums[B][2], row b over samples [first[b], first[b] + count[b])
// (first / count: device arrays or nullptr = 0 / T)
cudaError_t launch_esr(const float* out, long long ldo, const float* tgt, long long ldt, long long B, long long T,
                       int dc_pre, double* sums, int sm_count, cudaStream_t st, const long long* first = nullptr,
                       const long long* count = nullptr, int per_row = 0);

// Multi-resolution STFT loss (stft.cu): sums[B][n_res][4], one memset and one launch per resolution; row b over samples
// [first[b], first[b] + count[b]) as launch_esr.  fft_sizes / hop_sizes / win_lengths: HOST arrays, validated by the caller.
cudaError_t launch_stft_loss(const float* out, long long ldo, const float* tgt, long long ldt, long long B, long long T,
                             const long long* first, const long long* count, int n_res, const int* fft_sizes,
                             const int* hop_sizes, const int* win_lengths, double* sums, int sm_count, cudaStream_t st);

extern std::atomic<unsigned long long> g_launches;   // engine kernels launched by this process (ntm_query)

// One-time per-device kernel configuration (cudaFuncSetAttribute) without mutable statics that race when several host
// threads drive several devices: a bit per device, set after the first successful configuration (idempotent if two
// threads race to it).
struct OncePerDevice {
    std::atomic<unsigned long long> done{0};
    template <class F>
    cudaError_t run(F configure)
    {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        if (dev < 64 && ((done.load(std::memory_order_acquire) >> dev) & 1ull)) return cudaSuccess;
        e = configure();
        if (e == cudaSuccess && dev < 64) done.fetch_or(1ull << dev, std::memory_order_release);
        return e;
    }
};

// ------------------------------------------------------------------------------------------------
// Fractional delay read shared by the fused and the stand-alone kernels.
// Reference: TimeVaryingDelayLine.forward, code/model.py:294-311 -- weights relu(1 - |j - d|) over the taps
// j = 0..D; only j = floor(d) and floor(d)+1 can be non-zero.  Weights and products are rounded exactly as
// the reference rounds them (float sub/abs/sub, float mul, one float add) so the result is bit-identical.
template <class LoadPast>
__device__ __forceinline__ float delay_read(float dt, long long t, int D, LoadPast past)
{
    const float fl = floorf(dt);
    float acc = 0.0f;
#pragma unroll
    for (int tap = 1; tap >= 0; --tap) {
        const float jf = fl + (float)tap;
        if (jf >= 0.0f && jf <= (float)D) {
            const float w = fmaxf(__fsub_rn(1.0f, fabsf(__fsub_rn(jf, dt))), 0.0f);
            acc = __fadd_rn(acc, __fmul_rn(w, past(t - (long long)jf)));
        }
    }
    return acc;
}

// On-chip pre_d ring of the fused DiffDelRNN form of the mma.sync kernels (gru_mma.cu, gru_mma4.cu): the last ring_len samples
// of pre_d per stream stay in shared memory, the carried history at positions -D .. -1, so that the delay taps of a chunk
// never leave the chip.  ring_len is the smallest power of two (>= 64) that is >= D + MMA_CH + 1.  A batched launch gets
// DELAY_RING_BUDGET bytes per CTA, so that four CTAs still share an SM: D <= 1919 at four streams per CTA, D <= 895 at eight.
// Every other DiffDelRNN launch runs the plain GRU into pre_d and the stand-alone delay line (delay.cu) behind it (capi.cu
// run_gru).  The real-time DiffDelRNN server is one CTA on an SM of its own and keeps its ring across blocks in up to
// RT_RING_BUDGET bytes: ring_len 32768 (D <= 32639) for one stream, 16384 (D <= 16255) for two, 8192 (D <= 8063) for three
// or four.  Its total shared memory stays under the 227 KB a CTA may opt into.
constexpr int MMA_CH = 128;   // steps per staged chunk of the mma.sync kernels
constexpr int DELAY_RING_BUDGET = 48 * 1024;
constexpr int RT_RING_BUDGET = 128 * 1024;
// ring_len for history length D and `streams` streams per CTA, or 0 if the ring does not fit `budget` bytes
inline int delay_ring_len(long long D, long long streams, long long budget)
{
    long long rl = 64;
    while (rl < D + MMA_CH + 1) rl *= 2;
    return rl * streams * 4 <= budget ? (int)rl : 0;
}

// DiffDelRNN ring helpers of the mma.sync kernels, for a CTA of NT threads that owns the ns streams from b0 on.  hist_in and
// hist_out hold each stream's last D samples of pre_d, oldest first.  ptxas reschedules the kernels' step loops when the
// shape of this code changes, so compare their SASS after editing it.  The ring delay read stays in each kernel: every
// shared form of it tried did that.

// Carried history -> positions -D .. -1 of the pre_d ring.
template <int NT>
__device__ __forceinline__ void delay_ring_prefill(const GruArgs& a, long long b0, int ns, int tid, float* ring)
{
    const int rmask = a.ring_len - 1;
    for (long long idx = tid; idx < (long long)ns * a.D; idx += NT) {
        const int s = (int)(idx / a.D);
        const int i = (int)(idx % a.D);
        ring[s * a.ring_len + ((i - a.D) & rmask)] = a.hist_in[(b0 + s) * (long long)a.D + i];
    }
}

// Rolled delay history (code/model.py:314-315): hist_out = ring positions end - D .. end - 1, once the CTA has written
// pre_d up to position end - 1 (end: a.T for a batched launch, the samples since open for the server).  They are still in
// the ring because ring_len >= D + MMA_CH + 1.
template <int NT>
__device__ __forceinline__ void delay_ring_roll(const GruArgs& a, long long b0, int ns, int tid, const float* ring,
                                                long long end)
{
    const int rmask = a.ring_len - 1;
    for (long long idx = tid; idx < (long long)ns * a.D; idx += NT) {
        const int s = (int)(idx / a.D), i = (int)(idx % a.D);
        a.hist_out[(b0 + s) * (long long)a.D + i] = ring[s * a.ring_len + ((int)(end - a.D + i) & rmask)];
    }
}

__device__ __forceinline__ float ex2_approx(float x)
{
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x)
{
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- packed fp32 arithmetic (sm_100: add / mul / fma .f32x2 = FADD2 / FMUL2 / FFMA2): one issue slot for two lanes' worth of
// fp32 work on a register pair -- for kernels bound by issue slots rather than by the FMA pipe
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk(float lo, float hi)
{
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c)
{
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b)
{
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b)
{
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src)
{
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sa), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

}  // namespace ntm
