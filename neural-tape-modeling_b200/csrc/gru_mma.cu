// Warp-level tensor-core persistent GRU kernel (mma.sync, accumulators in registers) -- the LATENCY regime of the
// batched path: a few streams per SM (BASELINE cfg 2: 1024 streams over 148 SMs, cfg 3: 256 streams).
//
// Why not tcgen05 here: measured on B200 (profiles/r01_tc_probe.txt) a tcgen05.mma costs >= ~40 clk of tensor pipe
// however small N is, and the issue -> commit -> mbarrier -> tcgen05.ld hand-off adds ~220 clk, so one GRU step
// through TMEM cannot go below ~700 clk before the gates are even touched; a dependent chain of four
// mma.sync.m16n8k16 takes ~80 clk with the accumulators already in the registers that evaluate the gates.
// The tcgen05 kernel (gru_tc.cu) takes over once an SM owns enough streams to be throughput-bound.
//
// Replaces the same reference arithmetic as the other kernels: `self.GRU(x, self.hidden)` + `self.output(x)` of
// RNN.forward / DiffDelRNN.forward (code/model.py:81-82, :412-413; torch rnn.py:1221-1224) and the delay read
// of code/model.py:422.
//
// One CTA = 4 warps owns 8 streams (one n8 tile) for all T steps.  Warp w owns hidden units [16w, 16w+16): three m16 tiles
//   tile A rows 0-7: r of units 16w+0..7, rows 8-15: z of the same units      -> c0,c1 = r   c2,c3 = z   (unit u0)
//   tile B the same for units 16w+8..15                                          -> c0,c1 = r   c2,c3 = z   (unit u1)
//   tile C rows 0-7: n of units 16w+0..7, rows 8-15: n of units 16w+8..15        -> c0,c1 = n(u0) c2,c3 = n(u1)
// so thread (gid = lane/4, tig = lane%4) ends up with r, z, n of units u0 = 16w+gid, u1 = u0+8 for streams 2tig,
// 2tig+1 of every n8 tile: no cross-thread exchange between the MMA and the gates.  W_hh fragments stay in registers
// for the whole kernel (pre-scaled by -log2 e / 2 log2 e, rounded once to the operand format).  The rounded state
// lives in a double-buffered shared-memory tile laid out so that each thread fetches all its B fragments of a step
// with two (f16/bf16) or four (tf32) LDS.128; the fp32 state never leaves registers.  One __syncthreads per step.
#include "gates.cuh"
#include "mma_frag.cuh"
#include "tc_prims.cuh"

namespace ntm {

using namespace tc;
using namespace mmaf;

namespace {

constexpr float LOG2E_F = 1.4426950408889634f;

template <int FMT, bool SPLIT = false>
struct MmaCfg {
    static constexpr int S = 8;                      // columns of the state tile (streams per CTA of the 8-stream form)
    static constexpr int CH = MMA_CH;                // steps per staged chunk (measured at 1024 streams: 32 -> 232.7 ns/step, 64 -> 238, 128 -> 221.7, 256 -> 220.1)
    static constexpr int YP_LD = S + 2;              // even: float2 stores of the head partials
    static constexpr int HB_BYTES = S * Frag<FMT, SPLIT>::ROW_BYTES;
    static constexpr int OFF_HB = 0;                               // [2][S][ROW_BYTES]
    static constexpr int OFF_XS = (2 * HB_BYTES + 127) / 128 * 128;   // [2][CH][S] floats
    static constexpr int OFF_YP = OFF_XS + 2 * CH * S * 4;         // [4 warps][CH][YP_LD] floats
    static constexpr int OFF_DS = (OFF_YP + 4 * CH * YP_LD * 4 + 15) / 16 * 16;   // [2][CH][S] delay trajectory (DiffDelRNN)
    static constexpr int SMEM_BYTES = OFF_DS + 2 * CH * S * 4;                    // + the pre_d ring, sized at launch
};

// HALF: the CTA owns 4 streams, placed in the EVEN columns of its n8 tile (stream s <-> column 2s), and
// skips the gate math, state stores and outputs of the odd columns: half the MUFU / FMA work per step for the same
// MMAs -- the shorter dependent step wins whenever there are CTAs to spare (B <= 4 streams per SM: cfg 3, cfg 5).
// RT (HALF only): resident real-time server -- the CTA stays on its SM, keeps weights, state and staging on chip and
// processes one block of a.T samples per mailbox hand-shake (a.rt, mapped host memory; a.x / a.y point into it), so a block
// costs two PCIe round trips instead of a kernel launch, a prologue and a stream synchronisation.
// DEFER (HALF only): the output head's accumulators are consumed one iteration later (see the head block); wins when a
// warp has its SM sub-partition to itself (one CTA per SM: cfg 3, cfg 5, the real-time server), loses otherwise.
// RTD (RT only): the DiffDelRNN server -- each block also brings its delay trajectory (a.d) and returns pre_d (a.pre) next
// to y, through the same mailbox.  The pre_d ring persists across blocks on the time axis of a 64-bit sample counter since open (the
// carried history at -D .. -1), so every block's y is the one long fused call's, bit for bit; the rolled history is read
// back from the ring when the server leaves.
template <int FMT, bool HALF, bool RT = false, bool DEFER = RT, bool SPLIT = false, bool RTD = false>
// (HALF is only dispatched up to two CTAs per SM: the full register file removes its spills, 197 vs 204 ns/step; the
// strict form keeps two sets of weight fragments in registers)
__global__ void __launch_bounds__(128, (FMT == FMT_TF32 || HALF || SPLIT) ? 2 : 4) gru_mma_kernel(const GruArgs a)
{
    static_assert(!RT || HALF, "the real-time server uses the 4-streams-per-CTA form");
    static_assert(!RTD || RT, "the DiffDelRNN server is a form of the real-time server");
    static_assert(!SPLIT || (FMT == FMT_F16 && !DEFER), "the strict form: f16 pairs, immediate head");
    constexpr int NP = SPLIT ? 2 : 1;                // operand parts (hi, lo')
    constexpr int SL = SPLIT ? 1 : 0;                // accumulators per tile: W_hi h_hi | (strict) W_hi h_lo' , W_lo' h_hi
    // PAIRCOL: strict form with four streams per CTA.  The odd column next to a stream's even column, dead in the rounded
    // modes, carries the stream's scaled residual h_lo': ONE MMA with W_hi then yields W_hi h_hi (even column) and W_hi h_lo'
    // (odd column) and a second one with W_lo' yields W_lo' h_hi -- two MMAs per product instead of three, one set of B
    // fragments, one head MMA (row 0 = w_hi, row 8 = w_lo': c0 + 2^-11 (c1 + c2)).  25 HMMAs per warp and step instead of 38.
    constexpr bool PAIRCOL = SPLIT && HALF;
    constexpr int NPB = PAIRCOL ? 1 : NP;            // parts of the state tile a thread loads B fragments from
    constexpr int SC = HALF ? 4 : 8;                 // streams per CTA
    constexpr int CS = HALF ? 2 : 1;                 // column stride of a stream
    constexpr int NE = HALF ? 1 : 2;                 // live columns per thread and n8 tile
    using C = MmaCfg<FMT, SPLIT>;
    using F = Frag<FMT, SPLIT>;
    constexpr int S = C::S, CH = C::CH, NK = F::NK, BW = F::BW;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* const hb = smem + C::OFF_HB;
    float* const xs = reinterpret_cast<float*>(smem + C::OFF_XS);
    float* const yp = reinterpret_cast<float*>(smem + C::OFF_YP);
    float* const ds = reinterpret_cast<float*>(smem + C::OFF_DS);
    float* const ring = reinterpret_cast<float*>(smem + C::SMEM_BYTES);      // [SC][a.ring_len] when a.ring_len > 0

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int gid = lane >> 2, tig = lane & 3;
    const int u0 = 16 * warp + 2 * gid, u1 = u0 + 1;      // adjacent units: their rounded states share a store
    const long long b0 = (long long)blockIdx.x * SC;
    const int ns = (int)((a.B - b0) < (long long)SC ? (a.B - b0) : (long long)SC);
    const float* __restrict__ blob = a.blob;

    // ---- W_hh fragments -> registers -------------------------------------------------------------------------
    // MMA k index (ks, kk) <-> actual hidden index is a free bijection as long as A and B agree: it is chosen so that
    // a thread's B fragments of a whole step are plain vector loads from the state tile
    //   f16/bf16: thread tig consumes elements tig*16 + 4ks + {0,1 | 2,3} in k-step ks
    //   tf32:     thread tig consumes elements (ks/2)*16 + tig*4 + 2(ks%2) + {0 | 1}
    uint32_t areg[NP][3][NK][4];
    {
        const float sc_rz = -LOG2E_F, sc_n = 2.0f * LOG2E_F;
        const float* wr0 = blob + BlobLayout::W_HH + (0 * 64 + u0) * 64;
        const float* wz0 = blob + BlobLayout::W_HH + (1 * 64 + u0) * 64;
        const float* wn0 = blob + BlobLayout::W_HH + (2 * 64 + u0) * 64;
        const float* wr1 = wr0 + 64;
        const float* wz1 = wz0 + 64;
        const float* wn1 = wn0 + 64;
        const float* lo[3] = {wr0, wz0, wn0};      // tile 0: r, tile 1: z, tile 2: n; rows 0-7 unit u0, rows 8-15 unit u1
        const float* hi[3] = {wr1, wz1, wn1};
        const float slo[3] = {sc_rz, sc_rz, sc_n}, shi[3] = {sc_rz, sc_rz, sc_n};
#pragma unroll
        for (int tile = 0; tile < 3; ++tile)
#pragma unroll
            for (int ks = 0; ks < NK; ++ks) {
                if (FMT == FMT_TF32) {
                    const int k = (ks >> 1) * 16 + tig * 4 + 2 * (ks & 1);
                    areg[0][tile][ks][0] = to_tf32(slo[tile] * lo[tile][k]);
                    areg[0][tile][ks][1] = to_tf32(shi[tile] * hi[tile][k]);
                    areg[0][tile][ks][2] = to_tf32(slo[tile] * lo[tile][k + 1]);
                    areg[0][tile][ks][3] = to_tf32(shi[tile] * hi[tile][k + 1]);
                } else {
                    const int k = tig * 16 + 4 * ks;
                    // fragment register i: a0 (row gid, k..k+1) a1 (row gid+8, k..k+1) a2 (row gid, k+2..k+3) a3 (row gid+8, ..)
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float* row = (i & 1) ? hi[tile] : lo[tile];
                        const float sc = (i & 1) ? shi[tile] : slo[tile];
                        const float w0 = sc * row[k + 2 * (i >> 1)], w1 = sc * row[k + 2 * (i >> 1) + 1];
                        areg[0][tile][ks][i] = pack2<FMT>(w0, w1);
                        if (SPLIT) {
                            const float2 wh = __half22float2(__floats2half2_rn(w0, w1));
                            areg[NP - 1][tile][ks][i] = pack2<FMT>((w0 - wh.x) * SPLIT_SCALE, (w1 - wh.y) * SPLIT_SCALE);
                        }
                    }
                }
            }
    }
    // per-unit constants (index 0: u0, 1: u1), scaled like the weights
    const UnitConst uc[2] = {load_unit_const(blob, u0), load_unit_const(blob, u1)};
    const float bo = blob[BlobLayout::B_OUT];
    // Output head on the tensor core: an extra m16 tile whose row 0 is w_out rounded to the operand format and whose
    // row 8 is the rounding residual (so w_out enters with ~2x the operand precision); the other rows are zero.  It is
    // contracted with the SAME B fragments, i.e. with the rounded state of the previous step, K split over the four
    // warps (warp w takes k-steps w*NK/4 ..), and lands in c0..c3 of the lanes gid == 0: y(2tig) = c0 + c2, y(2tig+1) =
    // c1 + c3.  The four warps' partial sums are added at the chunk flush.
    // Strict form: row 0 = w_hi and row 8 = w_lo' are contracted with the hi part of the state, a second fragment (row 0 =
    // 0, row 8 = w_hi) with its lo' part INTO THE SAME accumulators: c0, c1 = w_hi h_hi and c2, c3 = w_lo' h_hi + w_hi h_lo',
    // y = c0 + 2^-11 c2.
    constexpr int HK = NK / 4;
    uint32_t ahead[HK][4];
    uint32_t ahead2[SPLIT ? 2 : 1] = {};             // a1, a3 of the second fragment (a0 = a2 = 0)
#pragma unroll
    for (int q = 0; q < HK; ++q) {
        const int ks = warp * HK + q;
        float w[4], hi[4], lo[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int k = FMT == FMT_TF32 ? (ks >> 1) * 16 + tig * 4 + 2 * (ks & 1) + (i & 1) : tig * 16 + 4 * ks + i;
            w[i] = (gid == 0 && (FMT != FMT_TF32 || i < 2)) ? blob[BlobLayout::W_OUT + k] : 0.0f;
            if (FMT == FMT_TF32) hi[i] = __uint_as_float(to_tf32(w[i]));
            else if (FMT == FMT_BF16) hi[i] = __bfloat162float(__float2bfloat16_rn(w[i]));
            else hi[i] = __half2float(__float2half_rn(w[i]));
            lo[i] = SPLIT ? (w[i] - hi[i]) * SPLIT_SCALE : w[i] - hi[i];
        }
        if (FMT == FMT_TF32) {      // a0 (row 0, k) a1 (row 8, k) a2 (row 0, k+1) a3 (row 8, k+1)
            ahead[q][0] = to_tf32(hi[0]); ahead[q][1] = to_tf32(lo[0]); ahead[q][2] = to_tf32(hi[1]); ahead[q][3] = to_tf32(lo[1]);
        } else {                    // a0 (row 0, k..k+1) a1 (row 8, k..k+1) a2 (row 0, k+2..k+3) a3 (row 8, k+2..k+3)
            ahead[q][0] = pack2<FMT>(hi[0], hi[1]); ahead[q][1] = pack2<FMT>(lo[0], lo[1]);
            ahead[q][2] = pack2<FMT>(hi[2], hi[3]); ahead[q][3] = pack2<FMT>(lo[2], lo[3]);
            if (SPLIT) { ahead2[0] = ahead[q][0]; ahead2[SPLIT ? 1 : 0] = ahead[q][2]; }
        }
    }
    // this warp's k-steps of the B fragments (warp-uniform selects; a dynamic index would spill the array)
    auto head_mma = [&](const uint32_t (&bp)[NPB][BW], float (&c)[4]) {
        c[0] = c[1] = c[2] = c[3] = 0.0f;
#pragma unroll
        for (int q = 0; q < HK; ++q) {
#pragma unroll
            for (int part = 0; part < NPB; ++part) {
                const uint32_t (&b)[BW] = bp[part];
                uint32_t b0, b1;
                if (HK == 1) {
                    b0 = (warp & 2) ? ((warp & 1) ? b[6] : b[4]) : ((warp & 1) ? b[2] : b[0]);
                    b1 = (warp & 2) ? ((warp & 1) ? b[7] : b[5]) : ((warp & 1) ? b[3] : b[1]);
                } else {
                    b0 = (warp & 2) ? ((warp & 1) ? b[12 + 2 * q] : b[8 + 2 * q]) : ((warp & 1) ? b[4 + 2 * q] : b[2 * q]);
                    b1 = (warp & 2) ? ((warp & 1) ? b[13 + 2 * q] : b[9 + 2 * q]) : ((warp & 1) ? b[5 + 2 * q] : b[1 + 2 * q]);
                }
                if (part == 0) {
                    mma_sync<FMT>(c, ahead[q], b0, b1);
                } else {
                    const uint32_t a2[4] = {0u, ahead2[0], 0u, ahead2[NP - 1]};
                    mma_sync<FMT>(c, a2, b0, b1);
                }
            }
        }
    };
    // The same for the step loop.  Deferred-head forms (a warp alone on its SM sub-partition), f16 / bf16, rounded modes: this
    // warp's two words of the fragment are loaded again with one LDS.64 at a per-warp address instead of being selected from the
    // eight in registers (four SEL per step): 171.6 -> 168.1 ns/step at batch 1, cfg 3 181.7 -> 178.6.  With two CTAs per SM the
    // same change costs 8 % (215.7 -> 232.2 ns/step: one more shared-memory access per step in front of an HMMA), so the
    // immediate-head form keeps the selects (profiles/r02_mma_variants.txt).
    auto head_mma_step = [&](const uint8_t* tile, const uint32_t (&bp)[NPB][BW], float (&c)[4]) {
        if (DEFER && HK == 1 && NPB == 1 && !SPLIT) {
            const uint2 w2 = *reinterpret_cast<const uint2*>(tile + gid * F::ROW_BYTES + tig * 32 + warp * 8);
            c[0] = c[1] = c[2] = c[3] = 0.0f;
            mma_sync<FMT>(c, ahead[0], w2.x, w2.y);
        } else {
            head_mma(bp, c);
        }
    };
    // the two columns of a head tile -> the samples of streams 2tig, 2tig + 1
    auto head_value = [&](const float (&c)[4]) {
        if (PAIRCOL) return make_float2(fmaf(SPLIT_INV, c[1] + c[2], c[0]), 0.0f);
        return SPLIT ? make_float2(fmaf(SPLIT_INV, c[2], c[0]), fmaf(SPLIT_INV, c[3], c[1])) : make_float2(c[0] + c[2], c[1] + c[3]);
    };
    auto load_bfrag = [&](const uint8_t* tile, uint32_t (&bp)[NPB][BW]) {
        // f16/bf16: the thread's 16 elements are contiguous (2 vectors); tf32: vector q holds elements
        // q*16 + tig*4 .. +3 (4 vectors, a quarter-warp reads 64 contiguous bytes); strict form: the lo' part of the row
        // follows the hi part
#pragma unroll
        for (int part = 0; part < NPB; ++part) {
            const uint8_t* src = tile + gid * F::ROW_BYTES + part * F::PART_BYTES + (FMT == FMT_TF32 ? tig * 16 : tig * 32);
#pragma unroll
            for (int q = 0; q < BW / 4; ++q) {
                const uint4 v = *reinterpret_cast<const uint4*>(src + q * (FMT == FMT_TF32 ? 64 : 16));
                bp[part][4 * q] = v.x; bp[part][4 * q + 1] = v.y; bp[part][4 * q + 2] = v.z; bp[part][4 * q + 3] = v.w;
            }
        }
    };

    // rounded state of units (u0, u0 + 1) of the stream in column `col` of a state tile
    auto put_state = [&](uint8_t* tile, int col, float v0, float v1) {
        if (PAIRCOL) {                                 // hi pair -> the stream's own column, scaled residual pair -> the next one
            const __half2 hi = __floats2half2_rn(v0, v1);
            const float2 hf = __half22float2(hi);
            const __half2 lo = __floats2half2_rn((v0 - hf.x) * SPLIT_SCALE, (v1 - hf.y) * SPLIT_SCALE);
            *reinterpret_cast<uint32_t*>(tile + col * F::ROW_BYTES + u0 * 2) = *reinterpret_cast<const uint32_t*>(&hi);
            *reinterpret_cast<uint32_t*>(tile + (col + 1) * F::ROW_BYTES + u0 * 2) = *reinterpret_cast<const uint32_t*>(&lo);
        } else {
            store_state2<FMT, SPLIT>(tile + col * F::ROW_BYTES, u0, v0, v1);
        }
    };

    __shared__ __align__(16) float rt_xblk[RT ? RT_MAXSTREAMS * RT_MAXBLK : 4];   // server form: one block of x ...
    __shared__ __align__(16) float rt_yblk[RT ? RT_MAXSTREAMS * RT_MAXBLK : 4];   // ... and of y, staged on chip
    // DiffDelRNN server: the block's d and pre_d stage in the trajectory staging `ds`, which this form does not use otherwise
    static_assert(2 * RT_MAXSTREAMS * RT_MAXBLK <= 2 * CH * S, "the server's d and pre_d blocks fit in ds");
    float* const rt_dblk = ds;
    float* const rt_pblk = ds + RT_MAXSTREAMS * RT_MAXBLK;
    // DiffDelRNN (code/model.py:393-424): the head output is pre_d, y is the fractional-delay read of it (delay_read), fused
    // at the chunk flush with its taps from the on-chip pre_d ring (ntm_common.cuh; capi.cu runs this form only where the
    // ring fits); the delay trajectory is staged like x
    const bool delay = RTD || a.d != nullptr;
    float* __restrict__ head_out = delay ? a.pre : a.y;
    const long long ldo = delay ? a.ldp : a.ldy;

    auto load_x = [&](int buf, long long t0) {
        const int n = (int)((a.T - t0) < (long long)CH ? (a.T - t0) : (long long)CH);
        float* dstb = xs + buf * CH * S;
        for (int idx = tid; idx < CH * S; idx += 128) {
            const int col = idx % S, tt = idx / S, s = col / CS;
            if (col % CS == 0 && s < ns && tt < n) {
                // (server form: the whole block was fetched into shared memory in one PCIe round trip)
                if (RT) dstb[tt * S + col] = rt_xblk[s * RT_MAXBLK + t0 + tt];
                else cp_async4(dstb + tt * S + col, a.x + (b0 + s) * a.ldx + t0 + tt);
            } else {
                dstb[tt * S + col] = 0.0f;
            }
        }
        cp_async_commit();
    };

    const int rmask = a.ring_len - 1;
    auto load_d = [&](int buf, long long t0) {               // the chunk's delay trajectory, staged like x
        const int n = (int)((a.T - t0) < (long long)CH ? (a.T - t0) : (long long)CH);
        float* dstb = ds + buf * CH * S;
        for (int idx = tid; idx < CH * SC; idx += 128) {
            const int s = idx % SC, tt = idx / SC;
            if (s < ns && tt < n) cp_async4(dstb + tt * S + s, a.d + (b0 + s) * a.ldd + t0 + tt);
        }
        cp_async_commit();
    };
    if (delay) delay_ring_prefill<128>(a, b0, ns, tid, ring);

    // ---- initial state: fp32 in registers (hst[unit][stream]), rounded copy into state tile 0 ---------------------
    float hst[2][2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int col = 2 * tig + e, s = col / CS;
        const bool live = col % CS == 0 && s < ns;
#pragma unroll
        for (int u = 0; u < 2; ++u) hst[u][e] = (live && a.h_in) ? a.h_in[(b0 + s) * 64 + u0 + u] : 0.0f;
        if (!PAIRCOL || e == 0) {
            put_state(hb, col, hst[0][e], hst[1][e]);
            put_state(hb + C::HB_BYTES, col, 0.0f, 0.0f);                                    // dead columns stay finite
        }
    }
    const long long nchunks = (a.T + CH - 1) / CH;
    int cur = 0;
    unsigned rt_seen = 0;
    long long rt_pos = 0;                      // DiffDelRNN server: samples since open, the ring's time axis
    __shared__ unsigned rt_flag;
    do {
    if (RT) {
        // wait for the host to publish the next block (one uncached read of mapped host memory per poll)
        if (tid == 0) {
            unsigned long long t_wait;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_wait));
            unsigned sq;
            while ((sq = a.rt->seq_in) == rt_seen) {
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (now - t_wait > a.rt_idle_ns) { sq = RT_STOP; break; }
            }
            rt_flag = sq;
        }
        __syncthreads();
        if (rt_flag == RT_STOP) break;
        rt_seen = rt_flag;
        // fetch the block: every thread keeps up to 8 uncached loads of mapped host memory in flight (one round trip;
        // DiffDelRNN: x and d, 16 loads in the same round trip)
        const int total = ns * (int)a.T;
        float v[8], w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int idx = tid + 128 * i;
            v[i] = idx < total ? __ldcv(a.x + (idx / (int)a.T) * a.ldx + idx % (int)a.T) : 0.0f;
            if (RTD) w[i] = idx < total ? __ldcv(a.d + (idx / (int)a.T) * a.ldd + idx % (int)a.T) : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int idx = tid + 128 * i;
            if (idx < total) {
                rt_xblk[(idx / (int)a.T) * RT_MAXBLK + idx % (int)a.T] = v[i];
                if (RTD) rt_dblk[(idx / (int)a.T) * RT_MAXBLK + idx % (int)a.T] = w[i];
            }
        }
        __syncthreads();
    }
    load_x(0, 0);
    if (delay && !RTD) load_d(0, 0);
    for (long long c = 0; c < nchunks; ++c) {
        const long long t0 = c * CH;
        const int n = (int)((a.T - t0) < (long long)CH ? (a.T - t0) : (long long)CH);
        const int xb = (int)(c & 1);
        const float* xcur = xs + xb * CH * S;
        cp_async_wait_all();
        __syncthreads();                       // xs[xb] landed; state tile `cur` complete; previous flush done
        if (c + 1 < nchunks) {
            load_x(xb ^ 1, t0 + CH);
            if (delay && !RTD) load_d(xb ^ 1, t0 + CH);
        }

        float hpend[4];
        for (int tt = 0; tt < n; ++tt) {
            const uint8_t* hcur = hb + cur * C::HB_BYTES;
            uint8_t* hnext = hb + (cur ^ 1) * C::HB_BYTES;
            float acc[3][4];
            float accs[3][SPLIT ? 2 : 1][4];      // strict form: W_hi h_lo' and W_lo' h_hi (scaled by 2^11)
            uint32_t breg[NPB][BW];
            load_bfrag(hcur, breg);
#pragma unroll
            for (int tile = 0; tile < 3; ++tile) {
                acc[tile][0] = acc[tile][1] = acc[tile][2] = acc[tile][3] = 0.0f;
                if (SPLIT)
#pragma unroll
                    for (int i = 0; i < 4; ++i) accs[tile][0][i] = accs[tile][SL][i] = 0.0f;
            }
            if (!HALF) {
                // throughput form: input projection and biases enter through the accumulators (fewer FP32 instructions
                // after the MMAs: 976 vs 1027 ns/step at 8192 streams; the 4-stream latency form measured slower with it)
                const float2 xi = *reinterpret_cast<const float2*>(xcur + tt * S + 2 * tig);
#pragma unroll
                for (int u = 0; u < 2; ++u)
#pragma unroll
                    for (int e = 0; e < NE; ++e) {
                        acc[0][2 * u + e] = fmaf(uc[u].cr_w, e ? xi.y : xi.x, uc[u].cr_b);
                        acc[1][2 * u + e] = fmaf(uc[u].cz_w, e ? xi.y : xi.x, uc[u].cz_b);
                        acc[2][2 * u + e] = uc[u].ch_b;
                    }
            }
            // critical path first: r -> n -> h' is the dependent chain of the step, z only enters the final blend.  The r and
            // n tiles alternate (two dependent accumulator chains keep the pipe busy), the z tile follows and overlaps r's
            // gate math.  (Measured 233.7 vs 239.1 ns/step at 1024 streams against the ks-outer order over tiles that mixed
            // r and z rows; splitting z into two half-K chains gained nothing; bit-identical results.)
            // Strict form: three independent accumulator chains per tile (hi.hi, hi.lo', lo'.hi), issued r, n, then z; the
            // scaled chains are folded into the main accumulator once all MMAs are in flight.
            auto tile_mmas = [&](int tile, int ks) {
                mma_sync<FMT>(acc[tile], areg[0][tile][ks], breg[0][2 * ks], breg[0][2 * ks + 1]);
                if (SPLIT) {
                    if (!PAIRCOL)
                        mma_sync<FMT>(accs[tile][0], areg[0][tile][ks], breg[NPB - 1][2 * ks], breg[NPB - 1][2 * ks + 1]);
                    mma_sync<FMT>(accs[tile][SL], areg[NP - 1][tile][ks], breg[0][2 * ks], breg[0][2 * ks + 1]);
                }
            };
            {
#pragma unroll
            for (int ks = 0; ks < NK; ++ks)
#pragma unroll
                for (int tile = 0; tile < 3; tile += 2) tile_mmas(tile, ks);
#pragma unroll
            for (int ks = 0; ks < NK; ++ks) tile_mmas(1, ks);
            }

            // ---- head of the PREVIOUS step from the same B fragments (see `ahead`) -------------------------------
            // DEFER: its accumulators are only consumed at the top of the NEXT iteration (hpend).  With the add + store in
            // this iteration ptxas places them three instructions behind the head HMMA, in the middle of the r / n chains,
            // and the in-order warp stalls there for the HMMA latency on every step: 189.9 -> 176.7 ns/step with one warp
            // per SM sub-partition.  With two or more warps per sub-partition that stall is hidden by the other warps and
            // the compact 12-HMMA burst of the deferred form collides on the tensor pipe instead (221 -> 232 ns/step at
            // 1024 streams, 948 -> 1000 at 8192), so the immediate form stays there.
            if (DEFER) {
                if (tt > 1 && gid == 0)
                    *reinterpret_cast<float2*>(yp + (warp * CH + tt - 2) * C::YP_LD + 2 * tig) = head_value(hpend);
                head_mma_step(hcur, breg, hpend);
            } else {
                float ch[4];
                head_mma_step(hcur, breg, ch);
                if (tt > 0 && gid == 0)
                    *reinterpret_cast<float2*>(yp + (warp * CH + tt - 1) * C::YP_LD + 2 * tig) = head_value(ch);
            }
            // ---- gates, state blend, rounded state for the next step, head partials ------------------------------
            const float2 xv = *reinterpret_cast<const float2*>(xcur + tt * S + 2 * tig);
            float z[2][2], dn[2][2], hn[2][2];
            if (SPLIT) {                       // fold the scaled chains: W h = hi.hi + 2^-11 (hi.lo' + lo'.hi)
#pragma unroll
                for (int tile = 0; tile < 3; ++tile)
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (PAIRCOL) {             // W_hi h_lo' sits in the odd column of the main accumulator
                            if ((i & 1) == 0)
                                acc[tile][i] = fmaf(SPLIT_INV, acc[tile][i + 1] + accs[tile][SL][i], acc[tile][i]);
                        } else if (!HALF || (i & 1) == 0) {
                            acc[tile][i] = fmaf(SPLIT_INV, accs[tile][0][i] + accs[tile][SL][i], acc[tile][i]);
                        }
            }
            if (SPLIT) {                       // strict activations (gates.cuh), nothing shared between pairs
#pragma unroll
                for (int u = 0; u < 2; ++u)
#pragma unroll
                    for (int e = 0; e < NE; ++e) {
                        const float xx = e ? xv.y : xv.x;
                        float pr = acc[0][2 * u + e], pz = acc[1][2 * u + e], ahn = acc[2][2 * u + e];
                        if (HALF) {            // (non-HALF: the accumulators already hold W_i x + b for r, z and b_hn for n)
                            pr += fmaf(uc[u].cr_w, xx, uc[u].cr_b);
                            pz += fmaf(uc[u].cz_w, xx, uc[u].cz_b);
                            ahn += uc[u].ch_b;
                        }
                        hn[u][e] = gates_strict(pr, pz, ahn, fmaf(uc[u].cn_w, xx, uc[u].cn_b), hst[u][e]);
                    }
            }
#pragma unroll
            for (int u = 0; u < 2; ++u)
#pragma unroll
                for (int e = 0; e < (SPLIT ? 0 : NE); ++e) {
                    // r has its own reciprocal at every width: sharing 1/(d_r d_z) (4.5 instead of 5.5 MUFU per pair)
                    // measured slower even in the throughput regime (1052 vs 1030 ns/step at 8192 streams)
                    const float xx = e ? xv.y : xv.x;
                    if (HALF) {
                        gates_rz_dn_fast_r(uc[u], acc[0][2 * u + e], acc[1][2 * u + e], acc[2][2 * u + e], xx,
                                           z[u][e], dn[u][e]);
                    } else {                   // accumulators already hold W_i x + b (r, z) and b_hn (n)
                        const float r = rcp_approx(1.0f + ex2_approx(acc[0][2 * u + e]));
                        dn[u][e] = 1.0f + ex2_approx(fminf(fmaf(r, acc[2][2 * u + e], fmaf(uc[u].cn_w, xx, uc[u].cn_b)), EX2_CLAMP));
                        z[u][e] = rcp_approx(1.0f + ex2_approx(acc[1][2 * u + e]));
                    }
                }
#pragma unroll
            for (int e = 0; e < (SPLIT ? 0 : NE); ++e) {
                if (HALF) {                    // own n-gate reciprocals, shorter dependent chain (sharing them between the two
                                               // units measured 227.3 vs 221.5 ns/step even with two CTAs per SM)
                    // `_late`: everything that does not depend on the n gate's reciprocal is evaluated in front of it, one
                    // FMA behind the step's last MUFU instead of three (221.7 -> 215.6 ns/step at 1024 streams, 176.9 ->
                    // 171.6 at batch 1, profiles/r02_mma_variants.txt)
                    hn[0][e] = gates_blend1_late(z[0][e], dn[0][e], hst[0][e]);
                    hn[1][e] = gates_blend1_late(z[1][e], dn[1][e], hst[1][e]);
                } else {                       // the two hidden units of one stream share the n-gate reciprocal
                    gates_blend2(z[0][e], dn[0][e], hst[0][e], z[1][e], dn[1][e], hst[1][e], hn[0][e], hn[1][e]);
                }
            }
#pragma unroll
            for (int e = 0; e < NE; ++e) {
                hst[0][e] = hn[0][e];
                hst[1][e] = hn[1][e];
                put_state(hnext, 2 * tig + e, hn[0][e], hn[1][e]);
            }
            cur ^= 1;
            __syncthreads();                   // next state tile published; all reads of the old one are done
        }

        if (n > 0) {                           // head of the chunk's last step: one more MMA on the final state tile
            if (DEFER && n > 1 && gid == 0)    // (the pending head of the step before it)
                *reinterpret_cast<float2*>(yp + (warp * CH + n - 2) * C::YP_LD + 2 * tig) = head_value(hpend);
            uint32_t bfin[NPB][BW];
            float ch[4];
            load_bfrag(hb + cur * C::HB_BYTES, bfin);
            head_mma(bfin, ch);
            if (gid == 0)
                *reinterpret_cast<float2*>(yp + (warp * CH + n - 1) * C::YP_LD + 2 * tig) = head_value(ch);
            __syncthreads();
        }
        // ---- flush the chunk: y = sum of the four warps' partials + bias (+ x) ------------------------------------
        for (int idx = tid; idx < SC * CH; idx += 128) {
            const int s = idx / CH, tt = idx % CH, col = s * CS;
            if (s < ns && tt < n) {
                float v = yp[tt * C::YP_LD + col] + yp[(CH + tt) * C::YP_LD + col] + yp[(2 * CH + tt) * C::YP_LD + col] +
                          yp[(3 * CH + tt) * C::YP_LD + col] + bo;
                if (a.skip) v += xcur[tt * S + col];
                if (RTD) {
                    rt_pblk[s * RT_MAXBLK + t0 + tt] = v;
                    ring[s * a.ring_len + ((int)(rt_pos + t0 + tt) & rmask)] = v;
                    continue;
                }
                if (RT) rt_yblk[s * RT_MAXBLK + t0 + tt] = v;
                else head_out[(b0 + s) * ldo + t0 + tt] = v;
                if (delay) ring[s * a.ring_len + ((int)(t0 + tt) & rmask)] = v;
            }
        }
        if (RTD) {
            // the same delay read on the server's time axis; the block's y stages next to x
            __syncthreads();
            for (int idx = tid; idx < SC * CH; idx += 128) {
                const int s = idx / CH, tt = idx % CH;
                if (s < ns && tt < n) {
                    const float* rrow = ring + s * a.ring_len;
                    rt_yblk[s * RT_MAXBLK + t0 + tt] = delay_read(rt_dblk[s * RT_MAXBLK + t0 + tt], rt_pos + t0 + tt, a.D,
                                                                  [&](long long i) { return rrow[(int)i & rmask]; });
                }
            }
        } else if (delay) {
            // delay taps from the on-chip ring (the last ring_len >= D + CH samples of pre_d, history included) and the
            // staged trajectory: no L2 round trip of the samples this CTA has just produced
            __syncthreads();
            const float* dcur = ds + xb * CH * S;
            for (int idx = tid; idx < SC * CH; idx += 128) {
                const int s = idx / CH, tt = idx % CH;
                if (s < ns && tt < n) {
                    const long long tg = t0 + tt;
                    const float* rrow = ring + s * a.ring_len;
                    a.y[(b0 + s) * a.ldy + tg] =
                        delay_read(dcur[tt * S + s], tg, a.D, [&](long long i) { return rrow[(int)i & rmask]; });
                }
            }
        }
    }

    if (RT) {
        __syncthreads();
        // the block's output goes out in full 128-byte lines (a warp writes 32 consecutive samples of one stream)
        for (int idx = tid; idx < ns * RT_MAXBLK; idx += 128) {
            const int sidx = idx / RT_MAXBLK, t = idx % RT_MAXBLK;
            if (t < (int)a.T) {
                a.y[sidx * a.ldy + t] = rt_yblk[sidx * RT_MAXBLK + t];
                if (RTD) a.pre[sidx * a.ldp + t] = rt_pblk[sidx * RT_MAXBLK + t];
            }
        }
        __threadfence_system();                // this block's y (and pre_d) is visible to the host ...
        __syncthreads();
        if (tid == 0) a.rt->seq_out = rt_seen; // ... before its sequence number is
        if (RTD) rt_pos += a.T;
    }
    } while (RT);

    // ---- final state; rolled delay history --------------------------------------------------------------------------
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            const int s = (2 * tig + e) / CS;
            if (s < ns) a.h_out[(b0 + s) * 64 + u0 + u] = hst[u][e];
        }
    if (delay) {                               // rolled history from the ring (the server's time axis: samples since open)
        __syncthreads();
        delay_ring_roll<128>(a, b0, ns, tid, ring, RTD ? rt_pos : a.T);
    }
}

template <int FMT, bool HALF, bool DEFER = false, bool SPLIT = false>
cudaError_t launch_mma_one(const GruArgs& a, cudaStream_t st)
{
    using C = MmaCfg<FMT, SPLIT>;
    static OncePerDevice once;
    cudaError_t e = once.run([] {
        return cudaFuncSetAttribute(gru_mma_kernel<FMT, HALF, false, DEFER, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    C::SMEM_BYTES + DELAY_RING_BUDGET);
    });
    if (e != cudaSuccess) return e;
    constexpr int SC = HALF ? 4 : C::S;
    const long long grid = (a.B + SC - 1) / SC;
    const int smem_bytes = C::SMEM_BYTES + (a.d ? a.ring_len * SC * 4 : 0);
    gru_mma_kernel<FMT, HALF, false, DEFER, SPLIT><<<(unsigned)grid, 128, smem_bytes, st>>>(a);
    ++g_launches;
    return cudaGetLastError();
}

template <int FMT, bool SPLIT, bool RTD>
cudaError_t launch_mma_rt_fmt(const GruArgs& a, cudaStream_t st)
{
    using C = MmaCfg<FMT, SPLIT>;
    const int ring_bytes = RTD ? (int)(a.B * a.ring_len * 4) : 0;
    cudaError_t e = cudaFuncSetAttribute(gru_mma_kernel<FMT, true, true, !SPLIT, SPLIT, RTD>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         C::SMEM_BYTES + (RTD ? RT_RING_BUDGET : 0));
    if (e != cudaSuccess) return e;
    gru_mma_kernel<FMT, true, true, !SPLIT, SPLIT, RTD><<<1, 128, C::SMEM_BYTES + ring_bytes, st>>>(a);
    ++g_launches;
    return cudaGetLastError();
}

template <bool RTD>
cudaError_t launch_mma_rt(const GruArgs& a, int fmt, cudaStream_t st)
{
    switch (fmt) {
        case FMT_F16X3: return launch_mma_rt_fmt<FMT_F16, true, RTD>(a, st);
        case FMT_TF32: return launch_mma_rt_fmt<FMT_TF32, false, RTD>(a, st);
        case FMT_BF16: return launch_mma_rt_fmt<FMT_BF16, false, RTD>(a, st);
        default: return launch_mma_rt_fmt<FMT_F16, false, RTD>(a, st);
    }
}

template <int FMT>
cudaError_t launch_mma_fmt(const GruArgs& a, int streams, bool defer_head, cudaStream_t st)
{
    if (streams == 8) return launch_mma_one<FMT, false>(a, st);
    return defer_head ? launch_mma_one<FMT, true, true>(a, st) : launch_mma_one<FMT, true>(a, st);
}

}  // namespace

// fmt: FMT_F16 / FMT_BF16 / FMT_TF32 / FMT_F16X3 (strict: f16 hi/lo pairs, three MMAs per product).  streams: streams per CTA,
// 4 (HALF) or 8.  defer_head: the deferred-head form of the 4-stream kernel (rounded modes only; see DEFER).  DiffDelRNN
// (a.d != nullptr): a.ring_len from delay_ring_len at `streams` streams per CTA and DELAY_RING_BUDGET.
cudaError_t launch_gru_mma(const GruArgs& a, int fmt, int streams, bool defer_head, cudaStream_t st)
{
    if (a.B <= 0 || a.T <= 0) return cudaSuccess;
    if (streams != 4 && streams != 8) return cudaErrorInvalidValue;
    if (a.d && a.ring_len <= a.D + MMA_CH) return cudaErrorInvalidValue;
    switch (fmt) {
        case FMT_F16X3:
            return streams == 4 ? launch_mma_one<FMT_F16, true, false, true>(a, st)
                                : launch_mma_one<FMT_F16, false, false, true>(a, st);
        case FMT_TF32: return launch_mma_fmt<FMT_TF32>(a, streams, defer_head, st);
        case FMT_BF16: return launch_mma_fmt<FMT_BF16>(a, streams, defer_head, st);
        default: return launch_mma_fmt<FMT_F16>(a, streams, defer_head, st);
    }
}

// The resident real-time server (one CTA, <= 4 streams, blocks of a.T <= RT_MAXBLK samples; see RtMailbox).  a.x and a.y
// point into a.rt; a.d != nullptr selects the DiffDelRNN server, whose a.d and a.pre point into a.rt too (hist_in /
// hist_out: B x D, may alias; a.ring_len from delay_ring_len at B streams and RT_RING_BUDGET).
cudaError_t launch_gru_mma_rt(const GruArgs& a, int fmt, cudaStream_t st)
{
    if (a.B <= 0 || a.B > RT_MAXSTREAMS || a.T <= 0 || a.T > RT_MAXBLK || !a.rt) return cudaErrorInvalidValue;
    if (!a.d) return launch_mma_rt<false>(a, fmt, st);
    if (!a.pre || a.D < 0 || (a.D > 0 && (!a.hist_in || !a.hist_out)) || a.ring_len <= a.D + MMA_CH)
        return cudaErrorInvalidValue;
    return launch_mma_rt<true>(a, fmt, st);
}

}  // namespace ntm
