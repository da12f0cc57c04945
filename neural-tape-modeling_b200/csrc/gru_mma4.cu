// Lean form of the warp-level mma.sync GRU kernel for the widths BASELINE cfg 2, 3 and 5 run at: GRU and DiffDelGRU, f16 / bf16
// operands or the strict f16x3 mode, FOUR streams per CTA, up to two CTAs per SM (up to 8 streams per SM).
//
// Arithmetic, fragment layout and results are those of gru_mma.cu's 4-stream form, bit for bit (`self.GRU(x, self.hidden)` +
// `self.output(x)` of RNN.forward / DiffDelRNN.forward, code/model.py:81-82, :412-413, the delay read of :422; torch
// rnn.py:1221-1224): warp w owns hidden units [16w, 16w+16) as the
// three m16 tiles r, z, n; W_hh fragments in registers; the streams sit in the even columns of the n8 tile; r and n MMAs
// interleaved, z behind; own reciprocals; late blend; head as a fourth tile with K split over the warps.
//
// What differs is everything around the arithmetic.  With two CTAs per SM the step loop is limited by how many instructions and
// shared-memory accesses the two warps of a sub-partition push through it, not by a pipe (profiles/r02d_mma_lone_vs_paired.txt:
// one more LDS per step costs 8 %, ten more instructions 19 %), so the loop is unrolled four steps deep and everything that
// can be amortised over the four is:
//   * x is staged per stream with time contiguous ([stream][CH + 8]) and read as ONE LDS.128 per four steps (was one LDS per step
//     plus its address arithmetic); staging itself moves 16 bytes per cp.async where the rows allow it.  The 8 floats of row
//     padding matter: with rows exactly CH = 128 floats apart the four streams' float4s sit in the same banks and the LDS.128 is
//     served in four passes -- 204.4 ns/step at 1024 streams against 194.5 with any padding that spreads them (4 .. 24 floats
//     measured alike), 164.4 -> 161.7 at batch 1, cfg 3 173.2 -> 171.3 (profiles/r02f_lean_chunk_pad_sweep.txt);
//   * the head partial sums of four steps leave as ONE STS.128 per warp lane (was an STS.64 + three address instructions per
//     step), which also keeps the head accumulators away from their HMMA (the "deferred head" effect without its burst);
//   * the two state tiles alternate at compile time (no tile address arithmetic, no toggle), the loop counter and its compare
//     are paid once per four steps.
// tf32, the real-time server and every other width stay in gru_mma.cu.
#include <type_traits>

#include "gates.cuh"
#include "mma_frag.cuh"
#include "tc_prims.cuh"

namespace ntm {

using namespace tc;
using namespace mmaf;

namespace {

constexpr float LOG2E_F4 = 1.4426950408889634f;
constexpr int MMA4_CH = 128;         // steps per staged chunk
constexpr int MMA4_XPAD = 8;         // padding of a staged x row in floats
constexpr int MMA4_YPAD = 4;         // padding of a head-partial row in floats, >= 4

template <int FMT>
struct Mma4Cfg {
    using F = Frag<FMT, false>;
    static constexpr int SC = 4;                     // streams per CTA (columns 0, 2, 4, 6 of the n8 tile)
    static constexpr int CH = MMA4_CH;               // steps per staged chunk
    static constexpr int XLD = CH + MMA4_XPAD;       // staged x row of one stream
    static constexpr int YLD = CH + MMA4_YPAD;       // head partials of one (warp, stream): position p holds sample p - 1
    static constexpr int TILE_BYTES = 8 * F::ROW_BYTES;
    static constexpr int OFF_HB = 0;                                         // [2][8][ROW_BYTES]
    static constexpr int OFF_XS = (2 * TILE_BYTES + 127) / 128 * 128;        // [2][SC][CH] floats
    static constexpr int OFF_YP = OFF_XS + 2 * SC * XLD * 4;                 // [4 warps][SC][YLD] floats
    static constexpr int OFF_DS = OFF_YP + 4 * SC * YLD * 4;                 // [2][SC][CH] delay trajectory (DiffDelRNN)
    static constexpr int SMEM_BYTES = OFF_DS + 2 * SC * CH * 4;              // + the pre_d ring [SC][ring_len], sized at launch
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src)
{
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem_src) : "memory");
}

// (The head's fragment words are selected from the eight in registers: loading them again with an LDS.64, which helps the
// general kernel's deferred-head form, measured slower here at every width: 167.3 vs 162.0 ns/step at batch 1.)
// STRICT: the fp32-grade f16x3 mode in its pair-column layout (gru_mma.cu, PAIRCOL): a stream's even column carries h_hi, the odd
// column next to it the scaled residual h_lo'; W_hi [h_hi | h_lo'] and W_lo' h_hi -- two MMAs per product --, Newton-refined
// reciprocals (gates_strict).
template <int FMT, bool STRICT>
__global__ void __launch_bounds__(128, 2) gru_mma4_kernel(const GruArgs a)
{
    static_assert(FMT == FMT_F16 || (FMT == FMT_BF16 && !STRICT), "16-bit operand formats; the strict form is f16");
    constexpr int NP = STRICT ? 2 : 1;
    using C = Mma4Cfg<FMT>;
    using F = Frag<FMT, false>;
    constexpr int SC = C::SC, CH = C::CH, NK = F::NK, YLD = C::YLD, XLD = C::XLD;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* const hb = smem + C::OFF_HB;
    float* const xs = reinterpret_cast<float*>(smem + C::OFF_XS);
    float* const yp = reinterpret_cast<float*>(smem + C::OFF_YP);
    float* const ds = reinterpret_cast<float*>(smem + C::OFF_DS);
    float* const ring = reinterpret_cast<float*>(smem + C::SMEM_BYTES);      // [SC][a.ring_len] when a.ring_len > 0

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int gid = lane >> 2, tig = lane & 3;        // tig = this thread's stream
    const int u0 = 16 * warp + 2 * gid, u1 = u0 + 1;
    const long long b0 = (long long)blockIdx.x * SC;
    const int ns = (int)((a.B - b0) < (long long)SC ? (a.B - b0) : (long long)SC);
    const float* __restrict__ blob = a.blob;

    // ---- W_hh fragments -> registers (layout and K permutation of gru_mma.cu) ---------------------------------------------
    uint32_t areg[NP][3][NK][4];
    {
        const float sc[3] = {-LOG2E_F4, -LOG2E_F4, 2.0f * LOG2E_F4};
#pragma unroll
        for (int tile = 0; tile < 3; ++tile) {
            const float* lo = blob + BlobLayout::W_HH + (tile * 64 + u0) * 64;      // rows 0-7: unit u0, rows 8-15: unit u1
            const float* hi = lo + 64;
#pragma unroll
            for (int ks = 0; ks < NK; ++ks) {
                const int k = tig * 16 + 4 * ks;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float* row = (i & 1) ? hi : lo;
                    const float w0 = sc[tile] * row[k + 2 * (i >> 1)], w1 = sc[tile] * row[k + 2 * (i >> 1) + 1];
                    areg[0][tile][ks][i] = pack2<FMT>(w0, w1);
                    if (STRICT) {
                        const float2 wh = __half22float2(__floats2half2_rn(w0, w1));
                        areg[NP - 1][tile][ks][i] = pack2<FMT>((w0 - wh.x) * SPLIT_SCALE, (w1 - wh.y) * SPLIT_SCALE);
                    }
                }
            }
        }
    }
    const UnitConst uc[2] = {load_unit_const(blob, u0), load_unit_const(blob, u1)};
    const float bo = blob[BlobLayout::B_OUT];
    uint32_t ahead[4];                                // head tile: row 0 = w_out rounded, row 8 = the rounding residual
    {
        float w[4], hi[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            w[i] = gid == 0 ? blob[BlobLayout::W_OUT + tig * 16 + 4 * warp + i] : 0.0f;
            hi[i] = FMT == FMT_BF16 ? __bfloat162float(__float2bfloat16_rn(w[i])) : __half2float(__float2half_rn(w[i]));
        }
        const float rs = STRICT ? SPLIT_SCALE : 1.0f;      // (strict: row 8 = w_lo', scaled like the state residual)
        ahead[0] = pack2<FMT>(hi[0], hi[1]); ahead[1] = pack2<FMT>((w[0] - hi[0]) * rs, (w[1] - hi[1]) * rs);
        ahead[2] = pack2<FMT>(hi[2], hi[3]); ahead[3] = pack2<FMT>((w[2] - hi[2]) * rs, (w[3] - hi[3]) * rs);
    }

    // x staging: [buf][stream][CH], time contiguous.  16-byte copies when every row chunk is 16-byte aligned.
    const bool vec = ((reinterpret_cast<uintptr_t>(a.x) | (uintptr_t)(a.ldx * 4)) & 15) == 0;
    auto load_x = [&](int buf, long long t0) {
        const int n = (int)((a.T - t0) < (long long)CH ? (a.T - t0) : (long long)CH);
        float* dstb = xs + buf * SC * XLD;
        if (vec && n == CH) {
            for (int idx = tid; idx < SC * CH / 4; idx += 128) {
                const int s = idx / (CH / 4), q = idx % (CH / 4);
                if (s < ns) cp_async16(dstb + s * XLD + 4 * q, a.x + (b0 + s) * a.ldx + t0 + 4 * q);
                else *reinterpret_cast<float4*>(dstb + s * XLD + 4 * q) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            }
        } else {
            for (int idx = tid; idx < SC * CH; idx += 128) {
                const int s = idx / CH, tt = idx % CH;
                if (s < ns && tt < n) cp_async4(dstb + s * XLD + tt, a.x + (b0 + s) * a.ldx + t0 + tt);
                else dstb[s * XLD + tt] = 0.0f;
            }
        }
        cp_async_commit();
    };

    // DiffDelRNN (code/model.py:393-424): the head output is pre_d, y is the fractional-delay read of it (delay_read,
    // ntm_common.cuh: bit-exact against the reference given the same pre_d), fused at the chunk flush.  The taps come from an
    // on-chip ring of the last ring_len >= D + CH samples of pre_d per stream (carried history included) when it fits, from the
    // chunk just written through L2 otherwise; the delay trajectory is staged like x.
    const bool delay = a.d != nullptr;
    float* __restrict__ head_out = delay ? a.pre : a.y;
    const long long ldo = delay ? a.ldp : a.ldy;
    const int rmask = a.ring_len - 1;
    const bool use_ring = delay && !a.warmup && a.ring_len > 0;
    auto load_d = [&](int buf, long long t0) {
        const int n = (int)((a.T - t0) < (long long)CH ? (a.T - t0) : (long long)CH);
        float* dstb = ds + buf * SC * CH;
        for (int idx = tid; idx < SC * CH; idx += 128) {
            const int s = idx / CH, tt = idx % CH;
            if (s < ns && tt < n) cp_async4(dstb + idx, a.d + (b0 + s) * a.ldd + t0 + tt);
        }
        cp_async_commit();
    };
    if (use_ring) {                                          // carried history -> ring positions -D .. -1
        for (long long idx = tid; idx < (long long)ns * a.D; idx += 128) {
            const int s = (int)(idx / a.D);
            const int i = (int)(idx % a.D);
            ring[s * a.ring_len + ((i - a.D) & rmask)] = a.hist_in[(b0 + s) * (long long)a.D + i];
        }
    }

    // ---- initial state: fp32 in registers, rounded copy into state tile 0; the odd (dead) columns of both tiles stay zero ----
    float hst[2] = {0.0f, 0.0f};
    if (tig < ns && a.h_in) { hst[0] = a.h_in[(b0 + tig) * 64 + u0]; hst[1] = a.h_in[(b0 + tig) * 64 + u1]; }
    auto state_words = [&](float v0, float v1, uint32_t& whi, uint32_t& wlo) {
        whi = pack2<FMT>(v0, v1);
        wlo = 0u;
        if (STRICT) {
            const float2 hf = __half22float2(__floats2half2_rn(v0, v1));
            wlo = pack2<FMT>((v0 - hf.x) * SPLIT_SCALE, (v1 - hf.y) * SPLIT_SCALE);
        }
    };
    {
        uint32_t whi, wlo;
        state_words(hst[0], hst[1], whi, wlo);
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
            for (int e = 0; e < 2; ++e)
                *reinterpret_cast<uint32_t*>(hb + t * C::TILE_BYTES + (2 * tig + e) * F::ROW_BYTES + u0 * 2) = t ? 0u : (e ? wlo : whi);
    }

    // per-thread addresses: B fragments of tile t, state word of tile t, x row, head-partial row
    const uint8_t* const frag[2] = {hb + gid * F::ROW_BYTES + tig * 32, hb + C::TILE_BYTES + gid * F::ROW_BYTES + tig * 32};
    uint8_t* const word[2] = {hb + 2 * tig * F::ROW_BYTES + u0 * 2, hb + C::TILE_BYTES + 2 * tig * F::ROW_BYTES + u0 * 2};
    float* const yrow = yp + (warp * SC + tig) * YLD;          // written by the lanes gid == 0

    // One GRU step: MMAs on state tile P, gates, new state into tile P ^ 1.  Returns this warp's head partial of the sample
    // BEFORE this step (the head tile is contracted with the state the step reads).
    auto step = [&](auto PT, float xx) -> float {
        constexpr int P = decltype(PT)::value;
        uint32_t b[8];
        {
            const uint4 v0 = *reinterpret_cast<const uint4*>(frag[P]);
            const uint4 v1 = *reinterpret_cast<const uint4*>(frag[P] + 16);
            b[0] = v0.x; b[1] = v0.y; b[2] = v0.z; b[3] = v0.w; b[4] = v1.x; b[5] = v1.y; b[6] = v1.z; b[7] = v1.w;
        }
        float acc[3][4], accl[STRICT ? 3 : 1][4], ch[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            acc[0][i] = acc[1][i] = acc[2][i] = ch[i] = 0.0f;
            if (STRICT) accl[0][i] = accl[STRICT ? 1 : 0][i] = accl[STRICT ? 2 : 0][i] = 0.0f;
        }
        auto tile_mma = [&](int tile, int ks) {
            mma_sync<FMT>(acc[tile], areg[0][tile][ks], b[2 * ks], b[2 * ks + 1]);
            if (STRICT) mma_sync<FMT>(accl[STRICT ? tile : 0], areg[NP - 1][tile][ks], b[2 * ks], b[2 * ks + 1]);
        };
        // critical path first: r -> n -> h' is the step's dependent chain; r and n alternate, z follows
#pragma unroll
        for (int ks = 0; ks < NK; ++ks) {
            tile_mma(0, ks);
            tile_mma(2, ks);
        }
#pragma unroll
        for (int ks = 0; ks < NK; ++ks) tile_mma(1, ks);
        {
            const uint32_t h0 = (warp & 2) ? ((warp & 1) ? b[6] : b[4]) : ((warp & 1) ? b[2] : b[0]);
            const uint32_t h1 = (warp & 2) ? ((warp & 1) ? b[7] : b[5]) : ((warp & 1) ? b[3] : b[1]);
            mma_sync<FMT>(ch, ahead, h0, h1);
        }
        if (STRICT) {                          // W h = W_hi h_hi + 2^-11 (W_hi h_lo' [odd column] + W_lo' h_hi)
#pragma unroll
            for (int tile = 0; tile < 3; ++tile)
#pragma unroll
                for (int i = 0; i < 4; i += 2)
                    acc[tile][i] = fmaf(SPLIT_INV, acc[tile][i + 1] + accl[STRICT ? tile : 0][i], acc[tile][i]);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            if (STRICT) {
                const float pr = acc[0][2 * u] + fmaf(uc[u].cr_w, xx, uc[u].cr_b);
                const float pz = acc[1][2 * u] + fmaf(uc[u].cz_w, xx, uc[u].cz_b);
                hst[u] = gates_strict(pr, pz, acc[2][2 * u] + uc[u].ch_b, fmaf(uc[u].cn_w, xx, uc[u].cn_b), hst[u]);
            } else {
                float z, dn;
                gates_rz_dn_fast_r(uc[u], acc[0][2 * u], acc[1][2 * u], acc[2][2 * u], xx, z, dn);
                hst[u] = gates_blend1_late(z, dn, hst[u]);
            }
        }
        {
            uint32_t whi, wlo;
            state_words(hst[0], hst[1], whi, wlo);
            *reinterpret_cast<uint32_t*>(word[P ^ 1]) = whi;
            if (STRICT) *reinterpret_cast<uint32_t*>(word[P ^ 1] + F::ROW_BYTES) = wlo;
        }
        __syncthreads();                       // next state tile published; all reads of the old one are done
        return STRICT ? fmaf(SPLIT_INV, ch[1] + ch[2], ch[0]) : ch[0] + ch[2];
    };
    using T0 = std::integral_constant<int, 0>;
    using T1 = std::integral_constant<int, 1>;

    const long long nchunks = (a.T + CH - 1) / CH;
    int cur = 0;                               // tile holding the current state at a chunk boundary (0 unless a chunk was odd)
    load_x(0, 0);
    if (use_ring) load_d(0, 0);
    for (long long c = 0; c < nchunks; ++c) {
        const long long t0 = c * CH;
        const int n = (int)((a.T - t0) < (long long)CH ? (a.T - t0) : (long long)CH);
        const int xb = (int)(c & 1);
        const float* xcur = xs + xb * SC * XLD;
        cp_async_wait_all();
        __syncthreads();                       // xs[xb] landed; state tile `cur` complete; previous flush done
        if (c + 1 < nchunks) {
            load_x(xb ^ 1, t0 + CH);
            if (use_ring) load_d(xb ^ 1, t0 + CH);
        }

        const float* xrow = xcur + tig * XLD;
        int tt = 0;
        if (cur == 0) {
            for (; tt + 4 <= n; tt += 4) {
                const float4 x4 = *reinterpret_cast<const float4*>(xrow + tt);
                float4 y4;
                y4.x = step(T0{}, x4.x);
                y4.y = step(T1{}, x4.y);
                y4.z = step(T0{}, x4.z);
                y4.w = step(T1{}, x4.w);
                if (gid == 0) *reinterpret_cast<float4*>(yrow + tt) = y4;       // positions tt .. tt+3 = samples tt-1 .. tt+2
            }
        }
        for (; tt < n; ++tt) {                 // tail of the last chunk (or a chunk entered on tile 1)
            const float y1 = cur == 0 ? step(T0{}, xrow[tt]) : step(T1{}, xrow[tt]);
            if (gid == 0) yrow[tt] = y1;
            cur ^= 1;
        }
        {                                      // head of the chunk's last step: one more MMA on the final state tile
            const uint8_t* src = (cur == 0 ? frag[0] : frag[1]) + (warp >> 1) * 16;
            const uint4 v = *reinterpret_cast<const uint4*>(src);
            float ch[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            mma_sync<FMT>(ch, ahead, (warp & 1) ? v.z : v.x, (warp & 1) ? v.w : v.y);
            if (gid == 0) yrow[n] = STRICT ? fmaf(SPLIT_INV, ch[1] + ch[2], ch[0]) : ch[0] + ch[2];
        }
        __syncthreads();
        // ---- flush the chunk: head output = sum of the four warps' partials + bias (+ x) ------------------------------
        for (int idx = tid; idx < SC * CH; idx += 128) {
            const int s = idx / CH, t = idx % CH;
            if (s < ns && t < n) {
                float v = yp[s * YLD + t + 1] + yp[(SC + s) * YLD + t + 1] + yp[(2 * SC + s) * YLD + t + 1] +
                          yp[(3 * SC + s) * YLD + t + 1] + bo;
                if (a.skip) v += xcur[s * XLD + t];
                head_out[(b0 + s) * ldo + t0 + t] = v;
                if (delay && a.warmup) a.y[(b0 + s) * a.ldy + t0 + t] = v;
                if (use_ring) ring[s * a.ring_len + ((int)(t0 + t) & rmask)] = v;
            }
        }
        if (use_ring) {
            __syncthreads();
            const float* dcur = ds + xb * SC * CH;
            for (int idx = tid; idx < SC * CH; idx += 128) {
                const int s = idx / CH, t = idx % CH;
                if (s < ns && t < n) {
                    const long long tg = t0 + t;
                    const float* rrow = ring + s * a.ring_len;
                    a.y[(b0 + s) * a.ldy + tg] = delay_read(dcur[idx], tg, a.D, [&](long long i) { return rrow[(int)i & rmask]; });
                }
            }
        } else if (delay && !a.warmup) {
            __syncthreads();                   // this chunk's pre_d is visible CTA-wide (L2 reads below)
            for (int idx = tid; idx < SC * CH; idx += 128) {
                const int s = idx / CH, t = idx % CH;
                if (s < ns && t < n) {
                    const long long tg = t0 + t;
                    const float* prow = a.pre + (b0 + s) * a.ldp;
                    const float* hrow = a.hist_in + (b0 + s) * (long long)a.D;
                    a.y[(b0 + s) * a.ldy + tg] = delay_read(a.d[(b0 + s) * a.ldd + tg], tg, a.D,
                                                            [&](long long i) { return i >= 0 ? __ldcg(prow + i) : hrow[a.D + i]; });
                }
            }
        }
    }
    if (tig < ns) { a.h_out[(b0 + tig) * 64 + u0] = hst[0]; a.h_out[(b0 + tig) * 64 + u1] = hst[1]; }
    if (delay) {                               // rolled delay history (code/model.py:314-315)
        __syncthreads();
        for (long long idx = tid; idx < (long long)ns * a.D; idx += 128) {
            const int s = (int)(idx / a.D);
            const long long i = idx % a.D;
            const long long src = a.T - a.D + i;
            a.hist_out[(b0 + s) * (long long)a.D + i] =
                src >= 0 ? __ldcg(a.pre + (b0 + s) * a.ldp + src) : a.hist_in[(b0 + s) * (long long)a.D + a.D + src];
        }
    }
}

template <int FMT, bool STRICT = false>
cudaError_t launch_mma4_one(const GruArgs& a, cudaStream_t st)
{
    using C = Mma4Cfg<FMT>;
    static OncePerDevice once;
    cudaError_t e = once.run([] {
        return cudaFuncSetAttribute(gru_mma4_kernel<FMT, STRICT>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES + 48 * 1024);
    });
    if (e != cudaSuccess) return e;
    // DiffDelRNN: keep the last D + CH samples of pre_d per stream on chip if they fit (<= 48 KB of ring per CTA); longer
    // histories read their taps back through L2
    GruArgs b = a;
    b.ring_len = 0;
    int smem_bytes = C::SMEM_BYTES;
    if (a.d != nullptr && !a.warmup) {
        long long rl = 64;
        while (rl < (long long)a.D + C::CH + 1) rl *= 2;
        if (rl * C::SC * 4 <= 48 * 1024) {
            b.ring_len = (int)rl;
            smem_bytes += (int)(rl * C::SC * 4);
        }
    }
    gru_mma4_kernel<FMT, STRICT><<<(unsigned)((a.B + C::SC - 1) / C::SC), 128, smem_bytes, st>>>(b);
    ++g_launches;
    return cudaGetLastError();
}

}  // namespace

// GRU and DiffDelGRU batches, f16 / bf16 operands or the strict f16x3 mode, four streams per CTA.
cudaError_t launch_gru_mma4(const GruArgs& a, int fmt, cudaStream_t st)
{
    if (a.B <= 0 || a.T <= 0) return cudaSuccess;
    if (fmt != FMT_F16 && fmt != FMT_BF16 && fmt != FMT_F16X3) return cudaErrorInvalidValue;
    if (fmt == FMT_F16X3) return launch_mma4_one<FMT_F16, true>(a, st);
    return fmt == FMT_BF16 ? launch_mma4_one<FMT_BF16>(a, st) : launch_mma4_one<FMT_F16>(a, st);
}

}  // namespace ntm
