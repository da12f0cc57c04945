// GRU gate arithmetic shared by the tensor-core kernels (fp32, MUFU ex2/rcp).
//
// Follows torch rnn.py:1221-1224 as used by code/model.py:81, :412:
//     r = sigmoid(W_ir x + b_ir + W_hr h + b_hr)      z = sigmoid(W_iz x + b_iz + W_hz h + b_hz)
//     n = tanh(W_in x + b_in + r * (W_hn h + b_hn))   h' = (1 - z) * n + z * h
// with every pre-activation pre-scaled on the way in (weights and constants by -log2 e for r, z and by 2 log2 e for n):
//     sigmoid(a) = 1 / (1 + 2^(-a log2 e))            tanh(a) = 1 - 2 / (1 + 2^(2 a log2 e))
// MUFU is the scarce pipe (16 lanes/clk/SM): the 8-stream form shares 1/(d_n0 d_n1) between the n gates of two units of one
// stream (gates_blend2).  Arguments of ex2 are clamped to 60 so that a product of two denominators stays below 2^121.
#pragma once
#include "ntm_common.cuh"

namespace ntm {

struct UnitConst {
    float cr_w, cr_b, cz_w, cz_b, cn_w, cn_b, ch_b;
};

__device__ __forceinline__ UnitConst load_unit_const(const float* __restrict__ blob, int j)
{
    constexpr float L = 1.4426950408889634f;
    UnitConst c;
    c.cr_w = -L * blob[BlobLayout::W_IH + j];
    c.cr_b = -L * (blob[BlobLayout::B_IH + j] + blob[BlobLayout::B_HH + j]);
    c.cz_w = -L * blob[BlobLayout::W_IH + 64 + j];
    c.cz_b = -L * (blob[BlobLayout::B_IH + 64 + j] + blob[BlobLayout::B_HH + 64 + j]);
    c.cn_w = 2.0f * L * blob[BlobLayout::W_IH + 128 + j];
    c.cn_b = 2.0f * L * blob[BlobLayout::B_IH + 128 + j];
    c.ch_b = 2.0f * L * blob[BlobLayout::B_HH + 128 + j];
    return c;
}

constexpr float EX2_CLAMP = 60.0f;

// Latency-regime form: r has its own reciprocal (r -> n -> h' is the step's critical path; sharing 1/(d_r d_z) makes r
// wait for z's ex2 and two more multiplies), z's ex2 / rcp fill the MUFU pipe's idle slots.  5.5 MUFU per pair.
__device__ __forceinline__ void gates_rz_dn_fast_r(const UnitConst& c, float ar, float az, float an, float x, float& z, float& dn)
{
    // (no clamp on the n gate's 2^s: its denominator gets its OWN reciprocal in this form, and 2^s = inf gives 1 / dn = 0, n = 1 --
    // the limit; the clamp only matters where denominators are multiplied.  Two FMNMX less per step; measured neutral.)
    const float r = rcp_approx(1.0f + ex2_approx(ar + fmaf(c.cr_w, x, c.cr_b)));
    dn = 1.0f + ex2_approx(fmaf(r, an + c.ch_b, fmaf(c.cn_w, x, c.cn_b)));
    z = rcp_approx(1.0f + ex2_approx(az + fmaf(c.cz_w, x, c.cz_b)));
}

// new states of two pairs (their n-gate denominators share one reciprocal).  Only pair up the SAME stream (two hidden
// units): a reciprocal shared between two streams would make a stream's rounding depend on its neighbour.
__device__ __forceinline__ void gates_blend2(float z0, float dn0, float h0, float z1, float dn1, float h1, float& hn0, float& hn1)
{
    const float qinv = rcp_approx(dn0 * dn1);
    const float n0 = fmaf(-2.0f, dn1 * qinv, 1.0f);
    const float n1 = fmaf(-2.0f, dn0 * qinv, 1.0f);
    hn0 = fmaf(z0, h0 - n0, n0);
    hn1 = fmaf(z1, h1 - n1, n1);
}

// The single-pair blend with everything that does not depend on the n gate's reciprocal moved in front of it:
//     h' = (1 - z) (1 - 2 q) + z h = [z h + 1 - z] + [-2 (1 - z)] q,   q = 1 / dn
// -- ONE dependent FMA behind the last MUFU of the step instead of three.
__device__ __forceinline__ float gates_blend1_late(float z, float dn, float h)
{
    const float a = fmaf(z, h - 1.0f, 1.0f), b = fmaf(2.0f, z, -2.0f);
    return fmaf(b, rcp_approx(dn), a);
}

// ---- strict (fp32-grade) activations ---------------------------------------------------------------------------------
// MUFU ex2.approx / rcp.approx are accurate to ~2 ulp, but their error is SYSTEMATIC: a constant relative bias of 1 ulp in
// the gate values moves the output of the cfg-2 checkpoint by 1.7e-5 (numpy emulation), a random +-2 ulp only by 2e-6 --
// the recurrence integrates a bias.  The strict mode therefore refines every reciprocal with one Newton step (error <= 1 ulp,
// unbiased); 2^x stays on MUFU.
__device__ __forceinline__ float rcp_strict(float d)
{
    const float r = rcp_approx(d);
    return fmaf(r, fmaf(-d, r, 1.0f), r);
}
// One (unit, stream) pair in the strict mode: own reciprocals everywhere (nothing shared, no products of denominators).
// pr, pz: complete scaled pre-activations of r and z; ahn = W_hn h + b_hn, gin = W_in x + b_in (scaled); returns the new state.
__device__ __forceinline__ float gates_strict(float pr, float pz, float ahn, float gin, float h)
{
    const float r = rcp_strict(1.0f + ex2_approx(fminf(pr, EX2_CLAMP)));
    const float dn = 1.0f + ex2_approx(fminf(fmaf(r, ahn, gin), EX2_CLAMP));
    const float z = rcp_strict(1.0f + ex2_approx(fminf(pz, EX2_CLAMP)));
    const float n = fmaf(-2.0f, rcp_strict(dn), 1.0f);
    return fmaf(z, h - n, n);
}

}  // namespace ntm
