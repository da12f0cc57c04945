// Fragment helpers shared by the warp-level mma.sync kernels (gru_mma.cu, gru_mma4.cu): operand formats, the MMA itself,
// the rounded-state tile.  Internal to the engine.
#pragma once
#include <cuda_fp16.h>

#include "tc_prims.cuh"

namespace ntm {
namespace mmaf {

using namespace tc;

// SPLIT (f16 only): the strict, fp32-grade mode.  Every operand is carried as two f16 numbers, v = hi + lo' / 2^11 with
// hi = f16(v) and lo' = f16((v - hi) * 2^11) (the power-of-two scaling keeps lo' a NORMAL f16 number down to |v| ~ 2^-25,
// so the pair holds 22 significand bits like 3xTF32 does, at half the MMA count), and the contraction is evaluated as
//     W h  ~=  W_hi h_hi  +  2^-11 (W_hi h_lo' + W_lo' h_hi)            (the dropped W_lo h_lo term is ~2^-22 relative)
// with fp32 accumulation: three MMAs where the rounded-operand modes issue one.
template <int FMT, bool SPLIT = false>
struct Frag {
    static constexpr int ELT = FMT == FMT_TF32 ? 4 : 2;
    static constexpr int NK = FMT == FMT_TF32 ? 8 : 4;            // MMAs along K = 64
    static constexpr int NP = SPLIT ? 2 : 1;                      // operand parts (hi, lo')
    static constexpr int PART_BYTES = 64 * ELT;                   // one part of a stream's state row
    static constexpr int ROW_BYTES = NP * PART_BYTES + 16;        // padded row of the state tile (conflict-free stores)
    static constexpr int BW = 16 * ELT / 4;                       // 32-bit words of B fragments per thread, n-tile and part
};
constexpr float SPLIT_SCALE = 2048.0f, SPLIT_INV = 1.0f / 2048.0f;

template <int FMT>
__device__ __forceinline__ void mma_sync(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    if (FMT == FMT_TF32)
        asm volatile(
            "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
            : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
            : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    else if (FMT == FMT_BF16)
        asm volatile(
            "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
            : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
            : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    else
        asm volatile(
            "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
            : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
            : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int FMT>
__device__ __forceinline__ uint32_t pack2(float lo, float hi)
{
    if (FMT == FMT_BF16) return pack_bf16(lo, hi);
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&h);
}

// rounded states of the adjacent units (unit, unit + 1) of one stream; unit is even
template <int FMT, bool SPLIT = false>
__device__ __forceinline__ void store_state2(uint8_t* row, int unit, float v0, float v1)
{
    if (FMT == FMT_TF32) {
        *reinterpret_cast<uint2*>(row + unit * 4) = make_uint2(to_tf32(v0), to_tf32(v1));
    } else if (SPLIT) {       // hi part, then the scaled residual 128 bytes further (Frag::PART_BYTES)
        const __half2 hi = __floats2half2_rn(v0, v1);
        const float2 hf = __half22float2(hi);
        const __half2 lo = __floats2half2_rn((v0 - hf.x) * SPLIT_SCALE, (v1 - hf.y) * SPLIT_SCALE);
        *reinterpret_cast<uint32_t*>(row + unit * 2) = *reinterpret_cast<const uint32_t*>(&hi);
        *reinterpret_cast<uint32_t*>(row + 128 + unit * 2) = *reinterpret_cast<const uint32_t*>(&lo);
    } else {
        *reinterpret_cast<uint32_t*>(row + unit * 2) = pack2<FMT>(v0, v1);
    }
}

}  // namespace mmaf
}  // namespace ntm
