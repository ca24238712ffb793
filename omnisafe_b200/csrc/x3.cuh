// Split-bf16 ("bf16x3") tensor-core arithmetic: the parity-grade mode of the MLP tiles.
//
// Every fp32 operand x is stored as three bf16 tiles x0 + x1 + x2 == x (exactly: x0 = rn_bf16(x),
// x1 = rn_bf16(x - x0), x2 = x - x0 - x1 which has <= 8 significant bits).  A product A * B is issued as the
// six kind::f16 MMAs  sum_{i+j<=2} A_i B_j  (the dropped terms are <= 2^-26 relative) with fp32 accumulation
// in TMEM, small terms first.  Every bf16 x bf16 product is exact in fp32, so the result carries fp32-level
// accuracy -- unlike kind::tf32 (10-bit mantissa), this mode meets the reference's fp32 Linear layers
// (omnisafe/utils/model.py:L105-111) at the tolerance of the exact-FMA path.
//
// Unlike tf32, 16-bit operands have an MN-major view under the ordinary 128-byte swizzle, so ONE stored
// activation tile [sample][feature] serves the forward GEMM (K-major, contraction over features) and the
// weight-gradient GEMM (MN-major, contraction over samples): no transposed copies, no role-swapped MMAs.
//
// Tile formats (base 1024-byte aligned):
//   SW128: [R][64] bf16, row pitch 128 B, 16-byte chunk index XOR (row & 7)            (layout type 2)
//   SW32 : [R][16] bf16, row pitch  32 B, 16-byte chunk index XOR ((row >> 2) & 1)     (layout type 6)
// An x3 tile is three such sub-tiles back to back (hi, mid, lo), `split` bytes apart.
#pragma once
#include "umma.cuh"

namespace osb {
namespace x3 {

using namespace umma;

// ---- descriptors ------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t desc_make(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}
// SW128 tile: 8-row groups 1024 B apart, both as K-major (rows = M/N index) and MN-major (rows = K index,
// one 64-element atom along M/N, so the leading offset is never used).
constexpr int LBO_DEFAULT = 16;
__device__ __forceinline__ uint64_t desc128(uint32_t saddr) { return desc_make(saddr, LBO_DEFAULT, 1024, 2); }
// SW32 tile: 8-row groups 256 B apart.
__device__ __forceinline__ uint64_t desc32(uint32_t saddr) { return desc_make(saddr, LBO_DEFAULT, 256, 6); }
// descriptor + byte offset (start-address field only; all tiles live below 256 KB of shared memory)
__device__ __forceinline__ uint64_t desc_add(uint64_t d, uint32_t bytes) { return d + (uint64_t)(bytes >> 4); }

// kind::f16 instruction descriptor, bf16 x bf16 -> fp32
__device__ __forceinline__ constexpr uint32_t idesc_bf16(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// D (+)= A * B over `nk` k-steps of 16, with the six split products (small terms first).
//   a0 / b0: descriptors of the hi sub-tiles at k-step 0; asplit / bsplit: bytes between sub-tiles;
//   akstep / bkstep: bytes per k-step (K-major: 32; MN-major: 16 rows * pitch).
//   bsplit == 0 marks an exactly representable B (e.g. the ones tile): only the three A terms are issued.
__device__ __forceinline__ void gemm_x3(uint32_t tmem_d, uint64_t a0, uint32_t asplit, uint32_t akstep,
                                        uint64_t b0, uint32_t bsplit, uint32_t bkstep, uint32_t idesc, int nk,
                                        bool accumulate) {
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll 1
    for (int ks = 0; ks < nk; ++ks) {
        const uint64_t a = desc_add(a0, (uint32_t)ks * akstep), b = desc_add(b0, (uint32_t)ks * bkstep);
        const uint64_t a1 = desc_add(a, asplit), a2 = desc_add(a, 2 * asplit);
        if (bsplit == 0) {
            mma_bf16(tmem_d, a2, b, idesc, acc);
            mma_bf16(tmem_d, a1, b, idesc, 1u);
            mma_bf16(tmem_d, a, b, idesc, 1u);
        } else {
            const uint64_t b1 = desc_add(b, bsplit), b2 = desc_add(b, 2 * bsplit);
            mma_bf16(tmem_d, a2, b, idesc, acc);
            mma_bf16(tmem_d, a, b2, idesc, 1u);
            mma_bf16(tmem_d, a1, b1, idesc, 1u);
            mma_bf16(tmem_d, a1, b, idesc, 1u);
            mma_bf16(tmem_d, a, b1, idesc, 1u);
            mma_bf16(tmem_d, a, b, idesc, 1u);
        }
        acc = 1u;
    }
}


// Warp-uniform variant for a dedicated MMA-issue warp: all 32 lanes run the descriptor arithmetic (uniform
// datapath), only the elected lane executes the MMAs.  (Issued from divergent code, every tcgen05.mma is
// wrapped by the compiler in a uniformisation loop that costs more than the MMA itself.)
__device__ __forceinline__ void gemm_x3_warp(bool leader, uint32_t tmem_d, uint64_t a0, uint32_t asplit, uint32_t akstep,
                                             uint64_t b0, uint32_t bsplit, uint32_t bkstep, uint32_t idesc, int nk,
                                             bool accumulate) {
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll 1
    for (int ks = 0; ks < nk; ++ks) {
        const uint64_t a = desc_add(a0, (uint32_t)ks * akstep), b = desc_add(b0, (uint32_t)ks * bkstep);
        const uint64_t a1 = desc_add(a, asplit), a2 = desc_add(a, 2 * asplit);
        const uint64_t b1 = desc_add(b, bsplit), b2 = desc_add(b, 2 * bsplit);
        if (bsplit == 0) {
            if (leader) {
                mma_bf16(tmem_d, a2, b, idesc, acc);
                mma_bf16(tmem_d, a1, b, idesc, 1u);
                mma_bf16(tmem_d, a, b, idesc, 1u);
            }
        } else {
            if (leader) {
                mma_bf16(tmem_d, a2, b, idesc, acc);
                mma_bf16(tmem_d, a, b2, idesc, 1u);
                mma_bf16(tmem_d, a1, b1, idesc, 1u);
                mma_bf16(tmem_d, a1, b, idesc, 1u);
                mma_bf16(tmem_d, a, b1, idesc, 1u);
                mma_bf16(tmem_d, a, b, idesc, 1u);
            }
        }
        __syncwarp();
        acc = 1u;
    }
}

// ---- fp32 <-> three bf16 ----------------------------------------------------------------------------
// pack two floats into one bf16x2 word (lo half = a, hi half = b), round to nearest even
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}
__device__ __forceinline__ float bf16lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }
// (a, b) -> words w0, w1, w2 with a == lo(w0) + lo(w1) + lo(w2), b == hi(w0) + hi(w1) + hi(w2)
__device__ __forceinline__ void split2(float a, float b, uint32_t& w0, uint32_t& w1, uint32_t& w2) {
    w0 = pack_bf16x2(a, b);
    const float ra = a - bf16lo(w0), rb = b - bf16hi(w0);
    w1 = pack_bf16x2(ra, rb);
    w2 = pack_bf16x2(ra - bf16lo(w1), rb - bf16hi(w1));
}

// byte offset of element (r, c) of a SW128 / SW32 sub-tile
__device__ __forceinline__ uint32_t off128(int r, int c) {
    return (uint32_t)(r * 128 + ((((c >> 3) ^ (r & 7)) << 4) | ((c & 7) << 1)));
}
__device__ __forceinline__ uint32_t off32(int r, int c) {
    return (uint32_t)(r * 32 + ((((c >> 3) ^ ((r >> 2) & 1)) << 4) | ((c & 7) << 1)));
}
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void lds128(uint32_t a, uint32_t& x, uint32_t& y, uint32_t& z, uint32_t& w) {
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(x), "=r"(y), "=r"(z), "=r"(w) : "r"(a));
}
__device__ __forceinline__ void sts16(uint32_t a, uint16_t v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"(v) : "memory");
}

// store 16 consecutive columns [c0, c0 + 16) (c0 % 16 == 0) of row r of a SW128 x3 tile
__device__ __forceinline__ void store16_x3(uint32_t base, uint32_t split, int r, int c0, const float (&v)[16]) {
    uint32_t w0[8], w1[8], w2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) split2(v[2 * i], v[2 * i + 1], w0[i], w1[i], w2[i]);
    const uint32_t row = base + (uint32_t)(r * 128);
    const int ch = c0 >> 3;
    const uint32_t o0 = row + (uint32_t)(((ch) ^ (r & 7)) << 4), o1 = row + (uint32_t)(((ch + 1) ^ (r & 7)) << 4);
    sts128(o0, w0[0], w0[1], w0[2], w0[3]); sts128(o1, w0[4], w0[5], w0[6], w0[7]);
    sts128(o0 + split, w1[0], w1[1], w1[2], w1[3]); sts128(o1 + split, w1[4], w1[5], w1[6], w1[7]);
    sts128(o0 + 2 * split, w2[0], w2[1], w2[2], w2[3]); sts128(o1 + 2 * split, w2[4], w2[5], w2[6], w2[7]);
}
// load them back as fp32 (exact reconstruction)
__device__ __forceinline__ void load16_x3(uint32_t base, uint32_t split, int r, int c0, float (&v)[16]) {
    const uint32_t row = base + (uint32_t)(r * 128);
    const int ch = c0 >> 3;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const uint32_t o = row + (uint32_t)(((ch + half) ^ (r & 7)) << 4);
        uint32_t a[4], b[4], c[4];
        lds128(o, a[0], a[1], a[2], a[3]);
        lds128(o + split, b[0], b[1], b[2], b[3]);
        lds128(o + 2 * split, c[0], c[1], c[2], c[3]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            v[8 * half + 2 * i] = (bf16lo(a[i]) + bf16lo(b[i])) + bf16lo(c[i]);
            v[8 * half + 2 * i + 1] = (bf16hi(a[i]) + bf16hi(b[i])) + bf16hi(c[i]);
        }
    }
}
// store the 16 columns of row r of a SW32 x3 tile ([R][16])
__device__ __forceinline__ void store16_x3_sw32(uint32_t base, uint32_t split, int r, const float (&v)[16]) {
    uint32_t w0[8], w1[8], w2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) split2(v[2 * i], v[2 * i + 1], w0[i], w1[i], w2[i]);
    const uint32_t row = base + (uint32_t)(r * 32);
    const int x = (r >> 2) & 1;
    const uint32_t o0 = row + (uint32_t)(x << 4), o1 = row + (uint32_t)((x ^ 1) << 4);
    sts128(o0, w0[0], w0[1], w0[2], w0[3]); sts128(o1, w0[4], w0[5], w0[6], w0[7]);
    sts128(o0 + split, w1[0], w1[1], w1[2], w1[3]); sts128(o1 + split, w1[4], w1[5], w1[6], w1[7]);
    sts128(o0 + 2 * split, w2[0], w2[1], w2[2], w2[3]); sts128(o1 + 2 * split, w2[4], w2[5], w2[6], w2[7]);
}

// single element stores (weight staging)
__device__ __forceinline__ void store1_x3(uint32_t base, uint32_t split, uint32_t off, float x) {
    uint32_t w0, w1, w2;
    split2(x, 0.f, w0, w1, w2);
    sts16(base + off, (uint16_t)w0); sts16(base + split + off, (uint16_t)w1); sts16(base + 2 * split + off, (uint16_t)w2);
}

// ---- mbarrier / issue helpers on 32-bit shared addresses ----------------------------------------------
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void mma_commit_a(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t p;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(p));
    return p != 0;
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// M = 64 accumulator (row 16 q + l in lane l < 16 of lane quarter q): thread t < 16 receives row t, columns
// [c, c + 8); thread t >= 16 row t - 16, columns [c + 8, c + 16) -- all 32 threads carry data.
__device__ __forceinline__ void tmem_ld8_m64(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.16x32bx2.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8], 8;\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// 8 consecutive columns [c0, c0 + 8) (c0 % 8 == 0) of row r of a SW128 x3 tile
__device__ __forceinline__ void store8_x3(uint32_t base, uint32_t split, int r, int c0, const float (&v)[8]) {
    uint32_t w0[4], w1[4], w2[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) split2(v[2 * i], v[2 * i + 1], w0[i], w1[i], w2[i]);
    const uint32_t o = base + (uint32_t)(r * 128 + (((c0 >> 3) ^ (r & 7)) << 4));
    sts128(o, w0[0], w0[1], w0[2], w0[3]);
    sts128(o + split, w1[0], w1[1], w1[2], w1[3]);
    sts128(o + 2 * split, w2[0], w2[1], w2[2], w2[3]);
}
__device__ __forceinline__ void load8_x3(uint32_t base, uint32_t split, int r, int c0, float (&v)[8]) {
    const uint32_t o = base + (uint32_t)(r * 128 + (((c0 >> 3) ^ (r & 7)) << 4));
    uint32_t a[4], b[4], c[4];
    lds128(o, a[0], a[1], a[2], a[3]);
    lds128(o + split, b[0], b[1], b[2], b[3]);
    lds128(o + 2 * split, c[0], c[1], c[2], c[3]);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[2 * i] = (bf16lo(a[i]) + bf16lo(b[i])) + bf16lo(c[i]);
        v[2 * i + 1] = (bf16hi(a[i]) + bf16hi(b[i])) + bf16hi(c[i]);
    }
}


// tanh with fp32-level accuracy (the MUFU tanh.approx has 2^-11 relative error):
//   |x| <  1: x + x^3 p(x^2), p = degree-6 minimax fit (relative error of the result 5e-9 before rounding);
//   otherwise 1 - 2 / (exp(2|x|) + 1) with ex2.approx / rcp.approx.  Max relative error 1.2e-7 (2 ulp).
__device__ __forceinline__ float tanh_acc(float x) {
    const float ax = fabsf(x);
    const float x2 = x * x;
    float p = fmaf(x2, -3.497081634e-04f, 2.272918122e-03f);
    p = fmaf(p, x2, -7.910109125e-03f);
    p = fmaf(p, x2, 2.146438509e-02f);
    p = fmaf(p, x2, -5.387288332e-02f);
    p = fmaf(p, x2, 1.333224624e-01f);
    p = fmaf(p, x2, -3.333328962e-01f);
    const float small = fmaf(p * x2, x, x);
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(ax * 2.8853900817779268f));   // exp(2|x|)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    const float big = copysignf(fmaf(-2.0f, r, 1.0f), x);
    return ax < 1.0f ? small : big;
}

}  // namespace x3
}  // namespace osb
