// extern "C" launch layer: the drop-in boundary declared in include/ntm_b200.h.
// No torch types, no exceptions, no hidden allocation on the device-pointer entry points.
#include <atomic>
#include <mutex>
#include <new>
#include <string.h>
#include <time.h>

#include "../../include/ntm_b200.h"
#include "ntm_common.cuh"

namespace ntm {
std::atomic<unsigned long long> g_launches{0};
}

namespace {

constexpr unsigned HANDLE_MAGIC = 0x4e544d42u;   // "NTMB"
thread_local int t_last_cuda = 0;
// Kernel-selection knob (tests, benchmarks; the pairs are tabled in include/ntm_b200.h): a process-wide default
// (ntm_set_tuning) that a handle may override (ntm_handle_set_tuning).  Packed into one atomic word so that concurrent
// launches from several threads read a consistent pair; nothing on the launch path writes shared state except the two
// counters below.
struct Tuning {
    int s = 0, ks = 0;
};
std::atomic<unsigned long long> g_tuning{0};
unsigned long long pack_tuning(int s, int ks) { return ((unsigned long long)(unsigned)s << 32) | (unsigned)ks; }
Tuning unpack_tuning(unsigned long long v) { return Tuning{(int)(v >> 32), (int)(v & 0xffffffffull)}; }
// NTM_Q_LAST_KERNEL (also kept per handle)
std::atomic<int> g_last_kernel{-1};

struct HostPipe {            // staging of the *_host entry points
    cudaStream_t s_in = nullptr, s_run = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {}, ev_run[2] = {}, ev_out[2] = {};
    float* buf = nullptr;    // one slab: x[2], d[2], y[2], pre[2], h, hist[2]
    size_t cap = 0;
    bool ready = false;
};

struct Handle {
    unsigned magic;
    int device;
    int sm_count;
    int has_bias;
    float* blob;
    ntm::TcsConsts tcs;      // host copy of the stream-major kernel's constant-bank parameters
    HostPipe pipe;
    std::atomic<int> refs{1};                        // ntm_gru_prepare's reference + one per ntm_retain / open real-time stream
    std::atomic<unsigned long long> tuning{~0ull};   // ~0: follow the process-wide default
    std::atomic<int> last_kernel{-1};
};

int cuda_fail(cudaError_t e)
{
    t_last_cuda = (int)e;
    return NTM_ECUDA;
}
#define CU(call)                                   \
    do {                                           \
        cudaError_t e_ = (call);                   \
        if (e_ != cudaSuccess) return cuda_fail(e_); \
    } while (0)

constexpr int MAX_DEVICES = 64;
struct CheckCtx {            // ntm_delay_check: persistent result flag of one device
    std::mutex mu;
    int* dev_flag = nullptr;
    int* host_flag = nullptr;
};
CheckCtx g_check[MAX_DEVICES];

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

Handle* as_handle(void* p)
{
    Handle* h = static_cast<Handle*>(p);
    return (h && h->magic == HANDLE_MAGIC) ? h : nullptr;
}

constexpr int MODE_MASK = (1 << NTM_MODE_FP32) | (1 << NTM_MODE_TF32) | (1 << NTM_MODE_BF16) | (1 << NTM_MODE_F16) |
                          (1 << NTM_MODE_F16X3);
// operand format selector of the tensor-core launchers (tc_prims.cuh FMT_*)
int mode_fmt(int mode) { return mode == NTM_MODE_TF32 ? 2 : mode == NTM_MODE_BF16 ? 1 : mode == NTM_MODE_F16X3 ? 3 : 0; }
bool mode_supported(int mode) { return mode >= 0 && mode < 31 && ((MODE_MASK >> mode) & 1); }

// Recurrent kernels, by their NTM_Q_LAST_KERNEL id
enum Kernel { K_FP32 = 0, K_MMA = 1, K_TCS = 3, K_MMA4 = 4 };

// One launch's kernel and configuration, fully resolved: the launchers decide nothing.
struct LaunchCfg {
    int kernel = -1;
    int fp32_streams = 0, fp32_ksplit = 0;   // K_FP32: streams per CTA (1, 2, 4, 8), k-slices per hidden unit (2, 4)
    int mma_streams = 0;                     // K_MMA: streams per CTA (4, 8)
    bool defer_head = false;                 // K_MMA, 4 streams per CTA: the deferred-head form
    int tcs_tiles = 0;                       // K_TCS: 128-stream tiles per CTA (1, 2)
    bool static_schedule = false;            // K_TCS: one CTA per tile group, no job queue
    int ring_len = 0;                        // DiffDelRNN, K_MMA / K_MMA4: the fused form's pre_d ring (GruArgs::ring_len);
                                             // 0: the GRU into pre_d, then the stand-alone delay line
};

constexpr long long TCS_MIN_STREAMS_PER_SM = 110;     // crossover mma.sync -> stream-major tcgen05 kernel (DESIGN.md 3.3)

// Every kernel-selection rule of the engine: (mode, batch, SMs, DiffDelRNN launch with history length D and warm-up flag,
// tuning pair) -> configuration, or NTM_EINVAL for a tuning pair that has no meaning in this mode (the table in
// include/ntm_b200.h).
int resolve_launch(int mode, long long B, int sm_count, bool delay, long long D, int warmup, Tuning tune, LaunchCfg* out)
{
    LaunchCfg c;
    const int s = tune.s, ks = tune.ks;
    const bool automatic = s == 0 && ks == 0;
    if (mode == NTM_MODE_FP32) {
        // (streams per CTA, k-split), 0 = automatic; the 2-way k-split exists for one and two streams per CTA
        if ((s != 0 && s != 1 && s != 2 && s != 4 && s != 8) || (ks != 0 && ks != 2 && ks != 4)) return NTM_EINVAL;
        if (ks == 2 && s != 1 && s != 2) return NTM_EINVAL;
        c.kernel = K_FP32;
        c.fp32_streams = s;
        if (s == 0) {
            // fill the SMs first (two CTAs per SM), then grow the streams per CTA
            const long long per_cta = (B + 2ll * sm_count - 1) / (2ll * sm_count);
            c.fp32_streams = 1;
            while (c.fp32_streams < 8 && c.fp32_streams < per_cta) c.fp32_streams <<= 1;
        }
        // measured on B200 (tools/experiments/sweep_fp32.py): the 2-way k-split wins while a CTA owns <= 2 streams
        c.fp32_ksplit = ks != 0 ? ks : c.fp32_streams <= 2 ? 2 : 4;
        *out = c;
        return NTM_OK;
    }
    const bool strict = mode == NTM_MODE_F16X3;
    // four streams per CTA, 16-bit operands or the strict mode (cfg 2's width and below, GRU and DiffDelGRU): the lean form of
    // gru_mma4.cu (same results, bit for bit: 194.5 vs 215 ns/step at 1024 streams, 162 vs 168 at batch 1).  The strict form
    // only while every CTA has an SM of its own: with two CTAs per SM the general kernel's 4-stream form is faster, 361.7 vs
    // 366.8 ns/step at 1024 streams.  f16 / bf16 up to THREE such CTAs per SM: 5.19 vs 5.03e9 samples/s at 1480 streams, 6.23 vs
    // 6.04 at 1776 against the 8-stream form; beyond 12 streams per SM the 8-stream form wins: 6.96 vs 5.08 at 2048.
    const bool lean_ok = mode != NTM_MODE_TF32;
    const bool lean_auto = strict ? B <= 4ll * sm_count : B <= 12ll * sm_count;
    if (automatic) {
        // latency regime (few streams per SM): warp-level mma.sync kernels; throughput regime (>= one 128-stream tile per
        // SM): stream-major tcgen05 kernel (every operand format)
        if (B >= (long long)sm_count * TCS_MIN_STREAMS_PER_SM) {
            c.kernel = K_TCS;
            // one tile per SM (time-multiplexed by the job queue) beats two resident tiles until ~190 streams per SM (measured)
            c.tcs_tiles = B >= 190ll * sm_count ? 2 : 1;
        } else {
            c.kernel = lean_ok && lean_auto ? K_MMA4 : K_MMA;
        }
    } else if (ks == 3 && (s == 4 || s == 8)) {                 // general mma.sync kernel, s streams per CTA
        c.kernel = K_MMA;
        c.mma_streams = s;
    } else if (ks == 6 && s == 4) {                             // lean 4-stream kernel (tf32 has none: general kernel)
        c.kernel = lean_ok ? K_MMA4 : K_MMA;
    } else if (ks == 4 && (s == 1 || s == 2 || s == 5 || s == 6)) {   // tcgen05, 1 or 2 tiles per CTA (+ 4: static schedule)
        c.kernel = K_TCS;
        c.tcs_tiles = s & 3;
        c.static_schedule = s > 4;
    } else {
        return NTM_EINVAL;
    }
    if (c.kernel == K_MMA) {
        // automatic: 4 streams per CTA (shorter dependent step) up to two such CTAs per SM -- measured 216 vs 243 ns/step at
        // 1024 streams, 172 vs 238 at <= 592 (profiles/r02_mma_variants.txt); the strict form too since its 4-stream layout
        // carries the state residual in the otherwise dead columns (two MMAs per product instead of three): 363 vs 394
        // ns/step at 1024 streams, 264 vs 388 at batch 1 (profiles/r02_strict_paircol.txt)
        if (c.mma_streams == 0) c.mma_streams = B <= 8ll * sm_count ? 4 : 8;
        // the deferred head wins while every 4-stream CTA has an SM of its own (B <= 4 streams per SM; rounded modes)
        c.defer_head = c.mma_streams == 4 && !strict && (B + 3) / 4 <= sm_count;
    }
    // DiffDelRNN: the mma.sync kernels read the delay taps from an on-chip ring of pre_d at the chunk flush where the ring
    // fits (ntm_common.cuh delay_ring_len).  Every other launch -- a longer history, a warm-up call, the fp32 and tcgen05
    // kernels -- runs the delay line as a second, HBM-bound pass over pre_d (delay.cu: 12 bytes per sample, near the copy
    // peak).  Reading the taps back through L2 inside the recurrent kernel instead stalls the whole persistent CTA at every
    // chunk flush (256 x 30 s at D = 10001, f16: 239 vs 283 ms), and the tcgen05 kernel's job queue may still be producing,
    // on another SM, the samples a tap reaches back to.
    if (delay && !warmup && (c.kernel == K_MMA || c.kernel == K_MMA4))
        c.ring_len = ntm::delay_ring_len(D, c.kernel == K_MMA ? c.mma_streams : 4, ntm::DELAY_RING_BUDGET);
    *out = c;
    return NTM_OK;
}

// One recurrent launch (a.d != nullptr: DiffDelRNN).  A DiffDelRNN configuration without a ring runs in two passes on `st`:
// the recurrent kernel as a plain GRU with its head output into pre_d, then the delay line and the history roll over it.
int run_gru(Handle* hd, int mode, const ntm::GruArgs& a0, cudaStream_t st)
{
    if (!mode_supported(mode)) return NTM_EUNSUPPORTED;
    unsigned long long tv = hd->tuning.load(std::memory_order_relaxed);
    if (tv == ~0ull) tv = g_tuning.load(std::memory_order_relaxed);
    LaunchCfg c;
    const int rc = resolve_launch(mode, a0.B, hd->sm_count, a0.d != nullptr, a0.D, a0.warmup, unpack_tuning(tv), &c);
    if (rc != NTM_OK) return rc;
    const int fmt = mode_fmt(mode);
    const bool two_pass = a0.d != nullptr && c.ring_len == 0;
    ntm::GruArgs a = a0;
    a.ring_len = c.ring_len;
    if (two_pass) {
        a.y = a0.pre; a.ldy = a0.ldp;
        a.d = nullptr; a.pre = nullptr;
    }
    switch (c.kernel) {
        case K_FP32: CU(ntm::launch_gru_fp32(a, c.fp32_streams, c.fp32_ksplit, st)); break;
        case K_MMA: CU(ntm::launch_gru_mma(a, fmt, c.mma_streams, c.defer_head, st)); break;
        case K_MMA4: CU(ntm::launch_gru_mma4(a, fmt, st)); break;
        default: CU(ntm::launch_gru_tcs(a, hd->tcs, fmt, hd->sm_count, c.tcs_tiles, c.static_schedule, st)); break;
    }
    hd->last_kernel.store(c.kernel, std::memory_order_relaxed);
    g_last_kernel.store(c.kernel, std::memory_order_relaxed);
    if (two_pass)         // warm-up: y = pre_d, history still rolled
        CU(ntm::launch_delay(a0.pre, a0.ldp, a0.d, a0.ldd, a0.y, a0.ldy, a0.hist_in, a0.hist_out, a0.B, a0.T, a0.D,
                             a0.warmup, st));
    return NTM_OK;
}

int pipe_init(Handle* hd, size_t floats)
{
    HostPipe& p = hd->pipe;
    if (!p.ready) {
        CU(cudaStreamCreateWithFlags(&p.s_in, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&p.s_run, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&p.s_out, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CU(cudaEventCreateWithFlags(&p.ev_in[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&p.ev_run[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&p.ev_out[i], cudaEventDisableTiming));
        }
        p.ready = true;
    }
    if (p.cap < floats) {
        if (p.buf) CU(cudaFree(p.buf));
        p.buf = nullptr;
        p.cap = 0;
        cudaError_t e = cudaMalloc(&p.buf, floats * sizeof(float));
        if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); return NTM_ENOMEM; }
        CU(e);
        p.cap = floats;
    }
    return NTM_OK;
}

// Shared body of the two *_host entry points (d_host == nullptr: plain GRU).
// half_io (plain GRU only): x_host / y_host hold IEEE binary16 samples; they cross the host link as such and are widened /
// narrowed on the device (csrc/convert.cu) around the same fp32 kernels.
int predict_host(Handle* hd, int mode, const float* x_host, const float* d_host, float* y_host, float* pre_host,
                 float* h_host, float* hist_host, int64_t B, int64_t T, int64_t D, int skip, int64_t chunk_T,
                 bool half_io = false)
{
    if (!x_host || !y_host || !h_host || B < 0 || T < 0) return NTM_EINVAL;
    const bool delay = d_host != nullptr;
    if (delay && (!pre_host || !hist_host || D < 0)) return NTM_EINVAL;
    if (delay && half_io) return NTM_EUNSUPPORTED;
    if (!mode_supported(mode)) return NTM_EUNSUPPORTED;
    if (B == 0) return NTM_OK;
    DeviceGuard g(hd->device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);

    int64_t C = chunk_T > 0 ? chunk_T : (int64_t)((64ll << 20) / (4 * B));   // ~64 MiB per staged array
    if (C < 2048) C = 2048;
    C = (C + 63) & ~63ll;                                                     // keep rows 256-byte aligned
    if (C > T) C = (T + 63) & ~63ll;
    if (C == 0) C = 64;
    const size_t slab = (size_t)B * (size_t)C;
    const size_t narr = delay ? 8 : half_io ? 6 : 4;      // half_io: two more slabs hold the four binary16 staging arrays
    const size_t hfl = (size_t)B * 64, histfl = delay ? (size_t)B * (size_t)D : 0;
    int rc = pipe_init(hd, narr * slab + hfl + 2 * histfl + 64);
    if (rc != NTM_OK) return rc;
    HostPipe& p = hd->pipe;
    float* dx[2] = {p.buf, p.buf + slab};
    float* dy[2] = {p.buf + 2 * slab, p.buf + 3 * slab};
    float* dd[2] = {nullptr, nullptr};
    float* dp[2] = {nullptr, nullptr};
    if (delay) {
        dd[0] = p.buf + 4 * slab; dd[1] = p.buf + 5 * slab;
        dp[0] = p.buf + 6 * slab; dp[1] = p.buf + 7 * slab;
    }
    // binary16 staging (slab elements = half a float slab each): in[2], out[2]
    uint16_t* hx[2] = {nullptr, nullptr};
    uint16_t* hy[2] = {nullptr, nullptr};
    if (half_io) {
        uint16_t* hb = reinterpret_cast<uint16_t*>(p.buf + 4 * slab);
        hx[0] = hb; hx[1] = hb + slab; hy[0] = hb + 2 * slab; hy[1] = hb + 3 * slab;
    }
    const uint16_t* x16 = reinterpret_cast<const uint16_t*>(x_host);
    uint16_t* y16 = reinterpret_cast<uint16_t*>(y_host);
    float* dh = p.buf + narr * slab;
    float* dhist[2] = {dh + hfl, dh + hfl + histfl};

    CU(cudaMemcpyAsync(dh, h_host, hfl * sizeof(float), cudaMemcpyHostToDevice, p.s_run));
    if (delay && histfl)
        CU(cudaMemcpyAsync(dhist[0], hist_host, histfl * sizeof(float), cudaMemcpyHostToDevice, p.s_run));

    const int64_t nchunks = (T + C - 1) / C;
    int hcur = 0;
    for (int64_t c = 0; c < nchunks; ++c) {
        const int64_t t0 = c * C, n = (T - t0) < C ? (T - t0) : C;
        const int k = (int)(c & 1);
        // host -> device (stream s_in); the staging slot is free once the kernel of chunk c-2 finished
        if (c >= 2) CU(cudaStreamWaitEvent(p.s_in, p.ev_run[k], 0));
        if (half_io)
            CU(cudaMemcpy2DAsync(hx[k], C * 2, x16 + t0, T * 2, n * 2, B, cudaMemcpyHostToDevice, p.s_in));
        else
            CU(cudaMemcpy2DAsync(dx[k], C * sizeof(float), x_host + t0, T * sizeof(float), n * sizeof(float), B,
                                 cudaMemcpyHostToDevice, p.s_in));
        if (delay)
            CU(cudaMemcpy2DAsync(dd[k], C * sizeof(float), d_host + t0, T * sizeof(float), n * sizeof(float), B,
                                 cudaMemcpyHostToDevice, p.s_in));
        CU(cudaEventRecord(p.ev_in[k], p.s_in));
        // recurrent kernel (stream s_run); its output slot is free once chunk c-2 was copied out
        CU(cudaStreamWaitEvent(p.s_run, p.ev_in[k], 0));
        if (c >= 2) CU(cudaStreamWaitEvent(p.s_run, p.ev_out[k], 0));
        ntm::GruArgs a{};
        a.blob = hd->blob; a.sm_count = hd->sm_count; a.x = dx[k]; a.y = dy[k]; a.h_in = dh; a.h_out = dh;
        a.B = B; a.T = n; a.ldx = C; a.ldy = C; a.skip = skip;
        if (delay) {
            a.d = dd[k]; a.ldd = C; a.pre = dp[k]; a.ldp = C; a.D = (int)D;
            a.hist_in = dhist[hcur]; a.hist_out = dhist[hcur ^ 1];
            hcur ^= 1;
        }
        if (half_io) CU(ntm::launch_half_to_float(hx[k], dx[k], (long long)slab, hd->sm_count, p.s_run));
        rc = run_gru(hd, mode, a, p.s_run);
        if (rc != NTM_OK) return rc;
        if (half_io) CU(ntm::launch_float_to_half(dy[k], hy[k], (long long)slab, hd->sm_count, p.s_run));
        CU(cudaEventRecord(p.ev_run[k], p.s_run));
        // device -> host (stream s_out)
        CU(cudaStreamWaitEvent(p.s_out, p.ev_run[k], 0));
        if (half_io)
            CU(cudaMemcpy2DAsync(y16 + t0, T * 2, hy[k], C * 2, n * 2, B, cudaMemcpyDeviceToHost, p.s_out));
        else
            CU(cudaMemcpy2DAsync(y_host + t0, T * sizeof(float), dy[k], C * sizeof(float), n * sizeof(float), B,
                                 cudaMemcpyDeviceToHost, p.s_out));
        if (delay)
            CU(cudaMemcpy2DAsync(pre_host + t0, T * sizeof(float), dp[k], C * sizeof(float), n * sizeof(float), B,
                                 cudaMemcpyDeviceToHost, p.s_out));
        CU(cudaEventRecord(p.ev_out[k], p.s_out));
    }
    CU(cudaMemcpyAsync(h_host, dh, hfl * sizeof(float), cudaMemcpyDeviceToHost, p.s_run));
    if (delay && histfl)
        CU(cudaMemcpyAsync(hist_host, dhist[hcur], histfl * sizeof(float), cudaMemcpyDeviceToHost, p.s_run));
    CU(cudaStreamSynchronize(p.s_in));
    CU(cudaStreamSynchronize(p.s_run));
    CU(cudaStreamSynchronize(p.s_out));
    return NTM_OK;
}

}  // namespace

extern "C" {

int ntm_query(int what)
{
    switch (what) {
        case NTM_Q_VERSION: return NTM_API_VERSION;
        case NTM_Q_DEVICE_COUNT: {
            int n = 0;
            if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
            return n;
        }
        case NTM_Q_SM_COUNT: {
            int dev = 0, n = 0;
            if (cudaGetDevice(&dev) != cudaSuccess ||
                cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
                cudaGetLastError();
                return 0;
            }
            return n;
        }
        case NTM_Q_MODE_MASK: return MODE_MASK;
        case NTM_Q_KERNEL_LAUNCHES: return (int)(ntm::g_launches.load() & 0x7fffffffull);
        case NTM_Q_LAST_KERNEL: return g_last_kernel.load();
        default: return NTM_EINVAL;
    }
}

const char* ntm_strerror(int code)
{
    switch (code) {
        case NTM_OK: return "ok";
        case NTM_EINVAL: return "invalid argument";
        case NTM_EUNSUPPORTED: return "unsupported hidden size or arithmetic mode";
        case NTM_ENOMEM: return "out of device memory";
        case NTM_ECUDA: return cudaGetErrorString((cudaError_t)t_last_cuda);
        case NTM_EDELAY: return "delay exceeds max_delay (history length)";
        case NTM_ENODEVICE: return "no usable CUDA device (sm_100 required)";
        case NTM_ECLOSED: return "real-time stream is closed (stopped or idle timeout)";
        default: return "unknown error";
    }
}

int ntm_last_cuda_error(void) { return t_last_cuda; }

int ntm_set_tuning(int streams_per_cta, int ksplit)
{
    if (streams_per_cta < 0 || ksplit < 0) return NTM_EINVAL;
    g_tuning.store(pack_tuning(streams_per_cta, ksplit), std::memory_order_relaxed);
    return NTM_OK;
}

int ntm_handle_set_tuning(void* handle, int streams_per_cta, int ksplit)
{
    Handle* hd = as_handle(handle);
    if (!hd || streams_per_cta < -1 || ksplit < 0) return NTM_EINVAL;
    hd->tuning.store(streams_per_cta < 0 ? ~0ull : pack_tuning(streams_per_cta, ksplit), std::memory_order_relaxed);
    return NTM_OK;
}

int ntm_handle_last_kernel(void* handle)
{
    Handle* hd = as_handle(handle);
    return hd ? hd->last_kernel.load(std::memory_order_relaxed) : NTM_EINVAL;
}

int ntm_gru_prepare(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, const float* w_out,
                    const float* b_out, int H, int device, void** handle)
{
    if (!handle) return NTM_EINVAL;
    *handle = nullptr;
    if (!w_ih || !w_hh || !b_ih || !b_hh || !w_out) return NTM_EINVAL;
    if (H < 1 || H > ntm::H64) return NTM_EUNSUPPORTED;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return NTM_ENODEVICE; }
    if (device < 0 || device >= ndev) return NTM_EINVAL;
    int major = 0;
    CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) return NTM_ENODEVICE;          // the library carries sm_100a code only
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);

    using L = ntm::BlobLayout;
    float* host = new (std::nothrow) float[L::TOTAL];
    if (!host) return NTM_ENOMEM;
    memset(host, 0, sizeof(float) * L::TOTAL);
    // PyTorch layout, gate-major (r, z, n), H units per gate.  H < 64: the model is embedded in the 64-unit engine -- unit u of
    // gate g goes to row 64 g + u, the other rows and columns stay zero.  A padded unit has r = z = 1/2, n = tanh(0) = 0 and
    // therefore keeps the state 0 it starts from; its column of W_hh and its head weight are zero, so no real unit or output
    // sample depends on it: the H-unit GRU of code/model.py:44-45, term for term.
    for (int g3 = 0; g3 < 3; ++g3) {
        for (int u = 0; u < H; ++u) {
            const int src = g3 * H + u, dst = g3 * ntm::H64 + u;
            memcpy(host + L::W_HH + (size_t)dst * ntm::H64, w_hh + (size_t)src * H, sizeof(float) * H);
            host[L::W_IH + dst] = w_ih[src];
            host[L::B_IH + dst] = b_ih[src];
            host[L::B_HH + dst] = b_hh[src];
        }
    }
    memcpy(host + L::W_OUT, w_out, sizeof(float) * H);
    host[L::B_OUT] = b_out ? b_out[0] : 0.0f;
    ntm::pack_tc_images(host);
    ntm::TcsConsts tcs;
    ntm::fill_tcs_consts(host, &tcs);

    Handle* hd = new (std::nothrow) Handle();
    if (!hd) { delete[] host; return NTM_ENOMEM; }
    hd->magic = HANDLE_MAGIC;
    hd->device = device;
    hd->has_bias = b_out != nullptr;
    hd->tcs = tcs;
    hd->blob = nullptr;
    cudaError_t e = cudaDeviceGetAttribute(&hd->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc(&hd->blob, sizeof(float) * L::TOTAL);
    if (e == cudaSuccess) e = cudaMemcpy(hd->blob, host, sizeof(float) * L::TOTAL, cudaMemcpyHostToDevice);
    delete[] host;
    if (e != cudaSuccess) {
        if (hd->blob) cudaFree(hd->blob);
        delete hd;
        return cuda_fail(e);
    }
    *handle = hd;
    return NTM_OK;
}

int ntm_retain(void* handle)
{
    Handle* hd = as_handle(handle);
    if (!hd) return NTM_EINVAL;
    hd->refs.fetch_add(1, std::memory_order_relaxed);
    return NTM_OK;
}

void ntm_destroy(void* handle) { ntm_release(handle); }

void ntm_release(void* handle)
{
    Handle* hd = as_handle(handle);
    if (!hd) return;
    if (hd->refs.fetch_sub(1, std::memory_order_acq_rel) > 1) return;      // an open real-time stream / a retained user
    DeviceGuard g(hd->device);
    HostPipe& p = hd->pipe;
    if (p.ready) {
        cudaStreamDestroy(p.s_in); cudaStreamDestroy(p.s_run); cudaStreamDestroy(p.s_out);
        for (int i = 0; i < 2; ++i) {
            cudaEventDestroy(p.ev_in[i]); cudaEventDestroy(p.ev_run[i]); cudaEventDestroy(p.ev_out[i]);
        }
    }
    if (p.buf) cudaFree(p.buf);
    if (hd->blob) cudaFree(hd->blob);
    hd->magic = 0;
    delete hd;
}

static int copy_state(const float* h_in, float* h_out, int64_t B, cudaStream_t st)
{
    if (h_in == h_out) return NTM_OK;
    if (h_in) CU(cudaMemcpyAsync(h_out, h_in, sizeof(float) * (size_t)B * 64, cudaMemcpyDeviceToDevice, st));
    else CU(cudaMemsetAsync(h_out, 0, sizeof(float) * (size_t)B * 64, st));
    return NTM_OK;
}

int ntm_gru_forward(void* handle, int mode, const float* x, int64_t ldx, float* y, int64_t ldy, const float* h_in,
                    float* h_out, int64_t B, int64_t T, int skip, void* stream)
{
    Handle* hd = as_handle(handle);
    if (!hd || B < 0 || T < 0) return NTM_EINVAL;
    if (B == 0) return NTM_OK;
    if (!h_out) return NTM_EINVAL;
    DeviceGuard g(hd->device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);
    if (T == 0) return copy_state(h_in, h_out, B, (cudaStream_t)stream);
    if (!x || !y || ldx < T || ldy < T) return NTM_EINVAL;
    ntm::GruArgs a{};
    a.blob = hd->blob; a.sm_count = hd->sm_count; a.x = x; a.y = y; a.h_in = h_in; a.h_out = h_out;
    a.B = B; a.T = T; a.ldx = ldx; a.ldy = ldy; a.skip = skip;
    return run_gru(hd, mode, a, (cudaStream_t)stream);
}

int ntm_diffdel_forward(void* handle, int mode, const float* x, int64_t ldx, const float* d, int64_t ldd, float* y,
                        int64_t ldy, float* pre_d, int64_t ldp, const float* h_in, float* h_out, const float* hist_in,
                        float* hist_out, int64_t B, int64_t T, int64_t D, int warmup, int skip, void* stream)
{
    Handle* hd = as_handle(handle);
    if (!hd || B < 0 || T < 0 || D < 0 || D > 0x7fffffff) return NTM_EINVAL;
    if (B == 0) return NTM_OK;
    if (!h_out || (D > 0 && (!hist_in || !hist_out || hist_in == hist_out))) return NTM_EINVAL;
    DeviceGuard g(hd->device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);
    if (T == 0) {                                   // nothing to compute: state and history are unchanged
        if (D > 0)
            CU(cudaMemcpyAsync(hist_out, hist_in, sizeof(float) * (size_t)B * (size_t)D, cudaMemcpyDeviceToDevice,
                               (cudaStream_t)stream));
        return copy_state(h_in, h_out, B, (cudaStream_t)stream);
    }
    if (!x || !d || !y || !pre_d || ldx < T || ldd < T || ldy < T || ldp < T || y == pre_d) return NTM_EINVAL;
    ntm::GruArgs a{};
    a.blob = hd->blob; a.sm_count = hd->sm_count; a.x = x; a.y = y; a.h_in = h_in; a.h_out = h_out; a.d = d; a.pre = pre_d;
    a.hist_in = hist_in; a.hist_out = hist_out;
    a.B = B; a.T = T; a.ldx = ldx; a.ldy = ldy; a.ldd = ldd; a.ldp = ldp;
    a.D = (int)D; a.warmup = warmup; a.skip = skip;
    return run_gru(hd, mode, a, (cudaStream_t)stream);
}

int ntm_delay_forward(const float* x, int64_t ldx, const float* d, int64_t ldd, float* y, int64_t ldy,
                      const float* hist_in, float* hist_out, int64_t B, int64_t T, int64_t D, int warmup, int device,
                      void* stream)
{
    if (B < 0 || T < 0 || D < 0 || D > 0x7fffffff) return NTM_EINVAL;
    if (B == 0) return NTM_OK;
    if (D > 0 && (!hist_in || !hist_out || hist_in == hist_out)) return NTM_EINVAL;
    if (T > 0 && (!x || !y || x == y || (!warmup && !d) || ldx < T || ldy < T || (d && ldd < T))) return NTM_EINVAL;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);
    CU(ntm::launch_delay(x, ldx, d, ldd, y, ldy, hist_in, hist_out, B, T, D, warmup, (cudaStream_t)stream));
    return NTM_OK;
}

int ntm_delay_check(const float* d, int64_t ldd, int64_t B, int64_t T, int64_t D, int device, void* stream)
{
    if (B < 0 || T < 0 || D < 0) return NTM_EINVAL;
    if (B == 0 || T == 0) return NTM_OK;
    if (!d || ldd < T || device < 0 || device >= MAX_DEVICES) return NTM_EINVAL;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);
    // one persistent flag pair per device (device int + page-locked host int), created on first use: no allocation, no
    // cudaFree (a device-wide synchronisation) on the call path; the mutex serialises concurrent checks on one device
    // (the call synchronises its stream anyway)
    CheckCtx& c = g_check[device];
    std::lock_guard<std::mutex> lock(c.mu);
    if (!c.dev_flag) {
        CU(cudaMalloc(&c.dev_flag, sizeof(int)));
        cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&c.host_flag), sizeof(int), cudaHostAllocDefault);
        if (e != cudaSuccess) { cudaFree(c.dev_flag); c.dev_flag = nullptr; return cuda_fail(e); }
    }
    *c.host_flag = 0;
    CU(cudaMemsetAsync(c.dev_flag, 0, sizeof(int), (cudaStream_t)stream));
    CU(ntm::launch_delay_check(d, ldd, B, T, D, c.dev_flag, (cudaStream_t)stream));
    CU(cudaMemcpyAsync(c.host_flag, c.dev_flag, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return *c.host_flag ? NTM_EDELAY : NTM_OK;
}

// ---- real-time streams: a resident server kernel fed through a mapped host mailbox --------------------------------
}  // extern "C"

namespace {

constexpr unsigned RT_MAGIC = 0x4e545254u;   // "NTRT"
struct RtStream {
    unsigned magic;
    Handle* hd;
    int B, T;
    bool delay;               // DiffDelRNN stream (ntm_rt_diffdel_*)
    bool check;               // DiffDelRNN: refuse blocks with d > D or NaN (NTM_EDELAY)
    int64_t D;
    ntm::RtMailbox* mb;       // page-locked, mapped
    float* h_dev;             // B x 64 state, read at open, written when the server leaves
    float* hist_dev;          // DiffDelRNN: B x D delay history, read at open, written when the server leaves
    cudaStream_t st;
    unsigned seq;
    bool dead;                // the server left (stop, idle timeout or error)
};
// The stream behind p if it is one of the given kind (an RNN stream for ntm_rt_*, a DiffDelRNN stream for ntm_rt_diffdel_*).
RtStream* as_rt(void* p, bool delay)
{
    RtStream* r = static_cast<RtStream*>(p);
    return (r && r->magic == RT_MAGIC && r->delay == delay) ? r : nullptr;
}
double now_s()
{
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}
void rt_free(RtStream* r)
{
    if (r->st) cudaStreamDestroy(r->st);
    if (r->h_dev) cudaFree(r->h_dev);
    if (r->hist_dev) cudaFree(r->hist_dev);
    if (r->mb) cudaFreeHost(r->mb);
    Handle* hd = r->hd;
    r->magic = 0;
    delete r;
    ntm_release(hd);
}

// Publish block `++r->seq` (its data is already in the mailbox) and wait until the server has answered it.
int rt_handshake(RtStream* r)
{
    __atomic_thread_fence(__ATOMIC_SEQ_CST);            // the block is in memory before its sequence number
    ntm::RtMailbox* mb = r->mb;
    const unsigned seq = ++r->seq;
    mb->seq_in = seq;
    const double t0 = now_s();
    unsigned spins = 0;
    while (mb->seq_out != seq) {
        if ((++spins & 0xfff) == 0 && now_s() - t0 > 0.05) {
            // slow path: has the server left (idle timeout, error)?
            const cudaError_t q = cudaStreamQuery(r->st);
            if (q != cudaErrorNotReady) {
                r->dead = true;
                return q == cudaSuccess ? NTM_ECLOSED : cuda_fail(q);
            }
            if (now_s() - t0 > 10.0) { r->dead = true; return NTM_ECLOSED; }
        }
    }
    __atomic_thread_fence(__ATOMIC_SEQ_CST);
    return NTM_OK;
}

// Both kinds of stream: validation, allocation, state and history upload, launch.  An RNN stream has delay == false, D == 0.
int rt_open(void* handle, int mode, const float* h_host, const float* hist_host, int64_t B, int64_t block_len, int64_t D,
            int skip, bool delay, bool check, int idle_timeout_ms, void** rt)
{
    if (!rt) return NTM_EINVAL;
    *rt = nullptr;
    Handle* hd = as_handle(handle);
    if (!hd || B < 1 || B > ntm::RT_MAXSTREAMS || block_len < 1 || block_len > ntm::RT_MAXBLK || D < 0 ||
        idle_timeout_ms < 1)
        return NTM_EINVAL;
    if (!mode_supported(mode) || mode == NTM_MODE_FP32) return NTM_EUNSUPPORTED;     // the server is the mma.sync kernel
    const int ring_len = delay && D <= 0x7fffffff ? ntm::delay_ring_len(D, B, ntm::RT_RING_BUDGET) : 0;
    if (delay && ring_len == 0) return NTM_EUNSUPPORTED;              // the ring must fit on chip
    DeviceGuard g(hd->device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);
    RtStream* r = new (std::nothrow) RtStream();       // value-initialised: null pointers, seq 0, not dead
    if (!r) return NTM_ENOMEM;
    hd->refs.fetch_add(1, std::memory_order_relaxed);        // the resident kernel reads the handle's blob until close
    r->magic = RT_MAGIC; r->hd = hd; r->B = (int)B; r->T = (int)block_len; r->delay = delay; r->check = check; r->D = D;
    const size_t hbytes = sizeof(float) * 64 * (size_t)B, histbytes = sizeof(float) * (size_t)B * (size_t)D;
    cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&r->mb), sizeof(ntm::RtMailbox), cudaHostAllocMapped);
    if (e == cudaSuccess) {
        memset(r->mb, 0, sizeof(ntm::RtMailbox));
        e = cudaMalloc(&r->h_dev, hbytes);
    }
    if (e == cudaSuccess && D > 0) e = cudaMalloc(&r->hist_dev, histbytes);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&r->st, cudaStreamNonBlocking);
    if (e == cudaSuccess)
        e = h_host ? cudaMemcpyAsync(r->h_dev, h_host, hbytes, cudaMemcpyHostToDevice, r->st)
                   : cudaMemsetAsync(r->h_dev, 0, hbytes, r->st);
    if (e == cudaSuccess && D > 0)
        e = hist_host ? cudaMemcpyAsync(r->hist_dev, hist_host, histbytes, cudaMemcpyHostToDevice, r->st)
                      : cudaMemsetAsync(r->hist_dev, 0, histbytes, r->st);
    ntm::RtMailbox* mb_dev = nullptr;
    if (e == cudaSuccess) e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&mb_dev), r->mb, 0);
    if (e == cudaSuccess) {
        ntm::GruArgs a{};
        a.blob = hd->blob; a.sm_count = hd->sm_count; a.h_in = r->h_dev; a.h_out = r->h_dev;
        a.B = B; a.T = block_len; a.skip = skip;
        a.x = &mb_dev->x[0][0]; a.y = &mb_dev->y[0][0];
        a.ldx = a.ldd = a.ldy = a.ldp = ntm::RT_MAXBLK;
        if (delay) {
            // the server rolls the history in place: it reads hist_in into its ring at start and writes hist_out when it leaves
            a.d = &mb_dev->d[0][0]; a.pre = &mb_dev->pre[0][0]; a.D = (int)D; a.ring_len = ring_len;
            a.hist_in = r->hist_dev; a.hist_out = r->hist_dev;
        }
        a.rt = mb_dev; a.rt_idle_ns = (unsigned long long)idle_timeout_ms * 1000000ull;
        e = ntm::launch_gru_mma_rt(a, mode_fmt(mode), r->st);
    }
    if (e != cudaSuccess) { rt_free(r); return cuda_fail(e); }
    *rt = r;
    return NTM_OK;
}

// One block: rows into the mailbox, handshake, rows out.  d_host: DiffDelRNN only; pre_d_host: nullptr = not returned.
int rt_process(RtStream* r, const float* x_host, const float* d_host, float* y_host, float* pre_d_host)
{
    if (r->dead) return NTM_ECLOSED;
    const size_t T = (size_t)r->T;
    if (r->check) {                 // before the block is handed over: a refused block changes neither state nor history
        const float lim = (float)r->D;
        for (size_t i = 0; i < (size_t)r->B * T; ++i)
            if (!(d_host[i] <= lim)) return NTM_EDELAY;
    }
    ntm::RtMailbox* mb = r->mb;
    for (int s = 0; s < r->B; ++s) {
        memcpy(&mb->x[s][0], x_host + s * T, sizeof(float) * T);
        if (d_host) memcpy(&mb->d[s][0], d_host + s * T, sizeof(float) * T);
    }
    const int rc = rt_handshake(r);
    if (rc != NTM_OK) return rc;
    for (int s = 0; s < r->B; ++s) {
        memcpy(y_host + s * T, &mb->y[s][0], sizeof(float) * T);
        if (pre_d_host) memcpy(pre_d_host + s * T, &mb->pre[s][0], sizeof(float) * T);
    }
    return NTM_OK;
}

// Stop the server, read back the final state and history it writes on its way out (nullptr: skip), free the stream.
int rt_close(RtStream* r, float* h_host_out, float* hist_host_out)
{
    DeviceGuard g(r->hd->device);
    r->mb->seq_in = ntm::RT_STOP;
    cudaError_t e = cudaStreamSynchronize(r->st);
    if (e == cudaSuccess && h_host_out)
        e = cudaMemcpy(h_host_out, r->h_dev, sizeof(float) * 64 * (size_t)r->B, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && hist_host_out && r->D > 0)
        e = cudaMemcpy(hist_host_out, r->hist_dev, sizeof(float) * (size_t)r->B * (size_t)r->D, cudaMemcpyDeviceToHost);
    rt_free(r);
    return e == cudaSuccess ? NTM_OK : cuda_fail(e);
}

}  // namespace

extern "C" {

int ntm_rt_open(void* handle, int mode, const float* h_host, int64_t B, int64_t block_len, int skip, int idle_timeout_ms,
                void** rt)
{
    return rt_open(handle, mode, h_host, nullptr, B, block_len, 0, skip, false, false, idle_timeout_ms, rt);
}

int ntm_rt_process(void* rt, const float* x_host, float* y_host)
{
    RtStream* r = as_rt(rt, false);
    if (!r || !x_host || !y_host) return NTM_EINVAL;
    return rt_process(r, x_host, nullptr, y_host, nullptr);
}

int ntm_rt_close(void* rt, float* h_host_out)
{
    RtStream* r = as_rt(rt, false);
    return r ? rt_close(r, h_host_out, nullptr) : NTM_EINVAL;
}

int ntm_rt_diffdel_open(void* handle, int mode, const float* h_host, const float* hist_host, int64_t B, int64_t block_len,
                        int64_t D, int skip, int check_delay, int idle_timeout_ms, void** rt)
{
    return rt_open(handle, mode, h_host, hist_host, B, block_len, D, skip, true, check_delay != 0, idle_timeout_ms, rt);
}

int ntm_rt_diffdel_process(void* rt, const float* x_host, const float* d_host, float* y_host, float* pre_d_host)
{
    RtStream* r = as_rt(rt, true);
    if (!r || !x_host || !d_host || !y_host) return NTM_EINVAL;
    return rt_process(r, x_host, d_host, y_host, pre_d_host);
}

int ntm_rt_diffdel_close(void* rt, float* h_host_out, float* hist_host_out)
{
    RtStream* r = as_rt(rt, true);
    return r ? rt_close(r, h_host_out, hist_host_out) : NTM_EINVAL;
}

int ntm_esr_sums(const float* out, int64_t ldo, const float* target, int64_t ldt, int64_t B, int64_t T, int dc_pre,
                 double* sums, int device, void* stream)
{
    if (B < 0 || T < 0 || !sums) return NTM_EINVAL;
    if (B > 0 && T > 0 && (!out || !target || ldo < T || ldt < T)) return NTM_EINVAL;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    CU(ntm::launch_esr(out, ldo, target, ldt, B, T, dc_pre, sums, sms, (cudaStream_t)stream));
    return NTM_OK;
}

int ntm_esr_sums_rows(const float* out, int64_t ldo, const float* target, int64_t ldt, int64_t B, int64_t T,
                      const int64_t* first, const int64_t* count, int dc_pre, double* sums, int device, void* stream)
{
    if (B < 0 || T < 0 || (B > 0 && !sums)) return NTM_EINVAL;
    if (B > 0 && T > 0 && (!out || !target || ldo < T || ldt < T)) return NTM_EINVAL;
    if (B == 0) return NTM_OK;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    CU(ntm::launch_esr(out, ldo, target, ldt, B, T, dc_pre, sums, sms, (cudaStream_t)stream,
                       reinterpret_cast<const long long*>(first), reinterpret_cast<const long long*>(count), 1));
    return NTM_OK;
}

int ntm_mrstft_sums_rows(const float* out, int64_t ldo, const float* target, int64_t ldt, int64_t B, int64_t T,
                         const int64_t* first, const int64_t* count, int n_res, const int* fft_sizes,
                         const int* hop_sizes, const int* win_lengths, double* sums, int device, void* stream)
{
    if (B < 0 || T < 0 || n_res < 1 || !fft_sizes || !hop_sizes || !win_lengths || (B > 0 && !sums)) return NTM_EINVAL;
    if (B > 0 && T > 0 && (!out || !target || ldo < T || ldt < T)) return NTM_EINVAL;
    for (int r = 0; r < n_res; ++r) {
        const int n = fft_sizes[r];
        if (n < 256 || n > 4096 || (n & (n - 1)) || hop_sizes[r] < 1 || win_lengths[r] < 1 || win_lengths[r] > n)
            return NTM_EINVAL;
    }
    if (B == 0) return NTM_OK;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice);
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    CU(ntm::launch_stft_loss(out, ldo, target, ldt, B, T, reinterpret_cast<const long long*>(first),
                             reinterpret_cast<const long long*>(count), n_res, fft_sizes, hop_sizes, win_lengths, sums, sms,
                             (cudaStream_t)stream));
    return NTM_OK;
}

int ntm_gru_predict_host(void* handle, int mode, const float* x_host, float* y_host, float* h_host, int64_t B,
                         int64_t T, int skip, int64_t chunk_T)
{
    Handle* hd = as_handle(handle);
    if (!hd) return NTM_EINVAL;
    return predict_host(hd, mode, x_host, nullptr, y_host, nullptr, h_host, nullptr, B, T, 0, skip, chunk_T);
}

int ntm_gru_predict_host_f16(void* handle, int mode, const void* x_host_f16, void* y_host_f16, float* h_host, int64_t B,
                             int64_t T, int skip, int64_t chunk_T)
{
    Handle* hd = as_handle(handle);
    if (!hd) return NTM_EINVAL;
    return predict_host(hd, mode, static_cast<const float*>(x_host_f16), nullptr, static_cast<float*>(y_host_f16), nullptr,
                        h_host, nullptr, B, T, 0, skip, chunk_T, true);
}

int ntm_diffdel_predict_host(void* handle, int mode, const float* x_host, const float* d_host, float* y_host,
                             float* pre_d_host, float* h_host, float* hist_host, int64_t B, int64_t T, int64_t D,
                             int skip, int64_t chunk_T)
{
    Handle* hd = as_handle(handle);
    if (!hd || !d_host) return NTM_EINVAL;
    return predict_host(hd, mode, x_host, d_host, y_host, pre_d_host, h_host, hist_host, B, T, D, skip, chunk_T);
}

}  // extern "C"
