// Tensor-core (tcgen05, kind::tf32, TMEM accumulators) variant of the fused minibatch
// forward + loss + backward kernel -- the "fast" arithmetic mode of csrc/update.cu (which stays as
// the exact-fp32 parity path).  Same interface, same per-CTA partial-gradient outputs.
//
// All GEMM operands are fp32 tiles in shared memory in the K-major 128B-swizzled canonical layout
// (csrc/umma.cuh).  TF32 has no usable MN-major view of such a tile, so every activation that is
// needed with the sample index as the contraction dimension (weight gradients) is produced a second
// time in transposed form by a role-swapped MMA (D^T = W * X^T) instead of a transposed copy:
//
//   per 128-sample tile and network (O <= 64):
//     MMA1  Z1    [s][n] = X  * W1^T      -> H1    = tanh(.+b1)            (A operand of layer 2)
//     MMA2  Z1^T  [n][s] = W1 * X^T       -> H1^T                          (B operand of dW2)
//     MMA3  Z2    [s][n] = H1 * W2^T      -> H2
//     MMA4  OUT   [s][o] = H2 * W3^T      -> per-sample loss, dOUT
//     MMA5  dZ2   [s][k] = dOUT * W3      -> * (1 - H2^2)                  (B operand of dZ1^T)
//     MMA6  dZ2^T [k][s] = W3^T * dOUT^T  -> * (1 - H2^2)                  (A operand of dW2)
//     MMA7  dW2   [j][k] += dZ2^T * H1    (TMEM accumulator kept across tiles)
//     MMA8  dZ1^T [k][s] = W2^T * dZ2^T   -> * (1 - H1^2)                  (A operand of dW1)
//     MMA9  dW1   [j][o] += dZ1^T * X     (TMEM accumulator kept across tiles)
//   dW3, the bias gradients and d log_std stay on the CUDA cores (tiny).
#include "common.cuh"
#include "mlp.cuh"
#include "umma.cuh"

namespace osb {

using namespace umma;

constexpr int TT = 128;                 // samples per tile
constexpr uint32_t BUF = TT * 64 * 4;   // 32 KB activation buffer ([128][64] or [64][128] fp32)

enum TcLoss { TC_PPO_CLIP = 0, TC_RATIO = 1, TC_FOCOPS = 2, TC_COST = 3, TC_FVP = 4, TC_P3O = 5 };   // TC_FVP: dOUT supplied (Fisher-vector product)

struct TcBatch {
    const float* obs; const float* act; const float* logp; const float* adv_r; const float* adv_c;
    const float* tv_r; const float* tv_c; const float* moments; const int* perm;
    long long total; unsigned perm_seed; long long mb_start; int mb_count;
    int identity_stride;     // > 0: row = (mb_start + local) * identity_stride (full-batch passes, fvp_sample_freq)
};
struct TcArgs {
    TcBatch b;
    int kind; float clip, entropy_coef;
    const float* lagrange;
    const float* theta;
    float* gpart;
    float* stats_part;
    const int* stop_flag;
    int O, A, P, net_mask;
    const float* fvp_dmu;    // TC_FVP: tangent of mu per row [total][A] (fvp_tangent_tc_kernel)
    const float* fvp_vec;    // TC_FVP: direction v (log_std block of F v)
    float fvp_scale;         // TC_FVP: 1 / (rows * A)
    const float* mu_old;     // TC_FOCOPS: old-policy mean per row, log_std of the old policy,
    const float* logstd_old;
    float focops_lam, focops_eta;
    const float* focops_mask_mean;   // device scalar mean_i 1{KL_i <= eta} of this minibatch (pass 2) or null (pass 1)
    int forward_only;        // pass 1 of FOCOPS: statistics only, no backward
};

__device__ __forceinline__ unsigned long long tc_feistel(unsigned long long k, unsigned long long n, unsigned seed) {
    int bits = 2;
    while ((1ull << bits) < n) bits += 2;
    const int half = bits >> 1;
    const unsigned mask = (1u << half) - 1u;
    unsigned long long x = k;
    do {
        unsigned l = (unsigned)(x >> half) & mask, r = (unsigned)x & mask;
#pragma unroll
        for (int round = 0; round < 4; ++round) {
            const unsigned f = mix32(r ^ (seed + 0x9E3779B9u * (unsigned)(round + 1))) & mask;
            const unsigned nl = r;
            r = l ^ f;
            l = nl;
        }
        x = ((unsigned long long)l << half) | r;
    } while (x >= n);
    return x;
}

// TMEM column map
constexpr uint32_t C_Z = 0, C_ZT = 64, C_ZT2 = 192, C_OUT = 320, C_DW2 = 336, C_DW1 = 400, C_DW3 = 464, TMEM_COLS = 512;
constexpr int NTC = 512;   // 16 warps: lane quarter q = warp % 4, column group h = warp / 4 (0..3)

// 16-column variants of the row accessors (c0 % 16 == 0)
__device__ __forceinline__ void store_row16(uint32_t base, int r, int c0, int R, const float (&v)[16]) {
    const uint32_t row = base + (uint32_t)((c0 >> 5) * R * 128 + r * 128);
    const int ch0 = (c0 & 31) >> 2;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(row + (uint32_t)(((ch0 + i) ^ (r & 7)) << 4)),
                     "f"(tf32r(v[4 * i])), "f"(tf32r(v[4 * i + 1])), "f"(tf32r(v[4 * i + 2])), "f"(tf32r(v[4 * i + 3]))
                     : "memory");
}
__device__ __forceinline__ void load_row16(uint32_t base, int r, int c0, int R, float (&v)[16]) {
    const uint32_t row = base + (uint32_t)((c0 >> 5) * R * 128 + r * 128);
    const int ch0 = (c0 & 31) >> 2;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                     : "=f"(v[4 * i]), "=f"(v[4 * i + 1]), "=f"(v[4 * i + 2]), "=f"(v[4 * i + 3])
                     : "r"(row + (uint32_t)(((ch0 + i) ^ (r & 7)) << 4)));
}

// CHUNKED = obs dim > 64: layer 1 runs as a K loop over 64-column chunks of X / W1 (forward: Z1 and Z1^T
// accumulate over chunks; backward: one dW1 chunk per MMA, flushed from TMEM into this CTA's partial gradient).
// EXT = the two-pass / supplied-dOUT loss kinds (FOCOPS, P3O, FVP); the plain instantiation (PPO-clip, ratio,
// cost surrogate: the headline path) carries none of their registers or branches.
template <bool CHUNKED, bool EXT>
__global__ void __launch_bounds__(NTC, 1) minibatch_grad_tc_kernel(TcArgs p) {
    if (p.stop_flag && *p.stop_flag) return;
    // one network selected: grid.y == 1 and all of grid.x (up to one CTA per SM) works on that network
    const int net = (gridDim.y == 1) ? (__ffs(p.net_mask) - 1) : (int)blockIdx.y;
    if (!((p.net_mask >> net) & 1)) return;

    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;   // tiles need 1024 B alignment
    const uint32_t B0 = smem_u32(smem_raw) + pad;   // X -> H2 -> dZ1^T
    const uint32_t B1 = B0 + BUF;                   // X^T
    const uint32_t B2 = B1 + BUF;                   // H1 -> dZ2
    const uint32_t B3 = B2 + BUF;                   // H1^T
    const uint32_t B4 = B3 + BUF;                   // dOUT (first 16 KB) -> dZ2^T
    const uint32_t sW1 = B4 + BUF;                  // [64][64]
    const uint32_t sW2 = sW1 + 16384;               // [64][64]
    const uint32_t sW2T = sW2 + 16384;              // [64][64]
    const uint32_t sW3 = sW2T + 16384;              // [16][64]   (2 atoms x 16 rows)
    const uint32_t sW3T = sW3 + 4096;               // [64][32]   (cols >= out zero)
    float* sB1 = reinterpret_cast<float*>(smem_raw + pad + 5 * BUF + 3 * 16384 + 4096 + 8192);
    float* sB2 = sB1 + 64;
    float* sB3 = sB2 + 64;            // [16]
    float* sLs = sB3 + 16;            // logstd[16], sigma[16], dlogstd acc[16]
    float* sStat = sLs + 48;          // [8]
    float* sRed = sStat + 8;          // [4 * 8 + 4 * 16 + 4 * 16]
    float* sB3acc = sRed + 160;       // [16]
    float* sOld = sB3acc + 16;        // old policy: log_std[16], 1 / sigma_old^2 [16]
    long long* sRowBuf = reinterpret_cast<long long*>(sOld + 32);   // [2][128] rows of this / the next tile
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;           // h in [0, 4)
    const int O = p.O, A = p.A;
    const NetLayout L = net_layout(net, O, A);
    const int noff = net_offset(net, O, A);
    const float* theta = p.theta + noff;
    float* gout = p.gpart + (size_t)blockIdx.x * p.P + noff;
    const int ntiles = (p.b.mb_count + TT - 1) / TT;
    const float inv_b = 1.0f / (float)p.b.mb_count;

    // ---- weights -> swizzled K-major tiles (loads batched so they are all in flight together) ----
    {
        float w1v[8], w2v[8], w3v[2];
        const int k = tid & 63;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = (tid >> 6) + 8 * j;
            w1v[j] = (!CHUNKED && k < O) ? __ldg(theta + L.off_w1 + n * O + k) : 0.f;
            w2v[j] = __ldg(theta + L.off_w2 + n * 64 + k);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int o = (tid >> 6) + 8 * j;
            w3v[j] = (o < L.out) ? __ldg(theta + L.off_w3 + o * 64 + k) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = (tid >> 6) + 8 * j;
            sts(tile_addr(sW1, n, k, 64), tf32r(w1v[j]));
            const float w2 = tf32r(w2v[j]);
            sts(tile_addr(sW2, n, k, 64), w2);
            sts(tile_addr(sW2T, k, n, 64), w2);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int o = (tid >> 6) + 8 * j;
            const float w = tf32r(w3v[j]);
            sts(tile_addr(sW3, o, k, 16), w);
            sts(tile_addr(sW3T, k, o, 64), w);
        }
    }
    for (int i = tid; i < 64 * 16; i += NTC) sts(tile_addr(sW3T, i >> 4, 16 + (i & 15), 64), 0.f);
    if (tid < 64) { sB1[tid] = __ldg(theta + L.off_b1 + tid); sB2[tid] = __ldg(theta + L.off_b2 + tid); }
    if (tid < 16) {
        sB3[tid] = (tid < L.out) ? __ldg(theta + L.off_b3 + tid) : 0.f;
        const float ls = (net == 0 && tid < A) ? __ldg(theta + L.off_logstd + tid) : 0.f;
        sLs[tid] = ls; sLs[16 + tid] = expf(ls); sLs[32 + tid] = 0.f;
        const float lso = (net == 0 && tid < A && p.logstd_old) ? __ldg(p.logstd_old + tid) : 0.f;
        sOld[tid] = lso; sOld[16 + tid] = expf(-2.f * lso);
    }
    if (tid < 8) sStat[tid] = 0.f;
    if (tid < 16) sB3acc[tid] = 0.f;
    if (tid == 0) { mbar_init(&bar, 1); mbar_init_fence(); }
    if (warp == 0) tmem_alloc(&tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    uint32_t phase = 0;

    const float lam = (p.lagrange != nullptr) ? __ldg(p.lagrange) : 0.f;
    float m_r = 0.f, s_r = 1.f, m_c = 0.f;
    if (p.b.moments) { m_r = __ldg(p.b.moments + 0); s_r = __ldg(p.b.moments + 1); m_c = __ldg(p.b.moments + 2); }
    const bool is_fvp = EXT && p.kind == TC_FVP, is_focops = EXT && p.kind == TC_FOCOPS, is_p3o = EXT && p.kind == TC_P3O;
    float ab1 = 0.f, ab2 = 0.f;
    bool first_tile = true;
    const int s_row = 32 * q + lane;       // sample row of this thread in [s][.] accumulators
    const int t_row = 16 * q + lane;       // row (valid for lane < 16) in [64][.] accumulators
    const int c16 = 16 * h;                // 16-column group of the plain epilogues
    const int c32 = 32 * h;                // 32-column group of the transposed epilogues

    const bool vec = (O & 3) == 0;            // rows 16 B aligned: 128-bit gathers, prefetched one tile ahead
    auto tile_rows = [&](int tile, long long* dst) {
        if (tid < TT) {
            const int local = tile * TT + tid;
            long long row = -1;
            if (local < p.b.mb_count) {
                const long long k = p.b.mb_start + local;
                if (p.b.identity_stride > 0) row = k * p.b.identity_stride;
                else row = p.b.perm ? (long long)p.b.perm[k] : (long long)tc_feistel((unsigned long long)k, (unsigned long long)p.b.total, p.b.perm_seed);
            }
            dst[tid] = row;
        }
    };
    float4 xpre[4];
    auto prefetch_x = [&](const long long* rows) {
        const int k4 = (tid & 15) << 2;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const long long row = rows[(tid >> 4) + 32 * j];
            xpre[j] = (row >= 0 && k4 < O) ? __ldg(reinterpret_cast<const float4*>(p.b.obs + row * O + k4))
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    // CHUNKED: one 64-column chunk of this thread's X elements in flight (global -> registers -> tile)
    const int nchunks = (O + 63) >> 6;
    float xr[16];
    auto load_chunk = [&](const long long* rows, int c) {
        if (vec) {
            const int col = c * 64 + ((tid & 15) << 2);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const long long row = rows[(tid >> 4) + 32 * j];
                const float4 v = (row >= 0 && col < O) ? __ldg(reinterpret_cast<const float4*>(p.b.obs + row * O + col))
                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                xr[4 * j] = v.x; xr[4 * j + 1] = v.y; xr[4 * j + 2] = v.z; xr[4 * j + 3] = v.w;
            }
        } else {
            const int col = c * 64 + (tid & 63);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const long long row = rows[(tid >> 6) + 8 * j];
                xr[j] = (row >= 0 && col < O) ? __ldg(p.b.obs + row * O + col) : 0.f;
            }
        }
    };
    auto store_chunk = [&](uint32_t dst, bool transposed) {     // dst: [128 s][64 k] K-major, or its transpose [64 k][128 s]
        if (vec) {
            const int k4 = (tid & 15) << 2;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int m = (tid >> 4) + 32 * j;
                const float a = tf32r(xr[4 * j]), b = tf32r(xr[4 * j + 1]), c = tf32r(xr[4 * j + 2]), d = tf32r(xr[4 * j + 3]);
                if (!transposed) {
                    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tile_addr(dst, m, k4, TT)), "f"(a), "f"(b),
                                 "f"(c), "f"(d)
                                 : "memory");
                } else {
                    sts(tile_addr(dst, k4 + 0, m, 64), a); sts(tile_addr(dst, k4 + 1, m, 64), b);
                    sts(tile_addr(dst, k4 + 2, m, 64), c); sts(tile_addr(dst, k4 + 3, m, 64), d);
                }
            }
        } else {
            const int k = tid & 63;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int m = (tid >> 6) + 8 * j;
                const float v = tf32r(xr[j]);
                if (!transposed) sts(tile_addr(dst, m, k, TT), v);
                else sts(tile_addr(dst, k, m, 64), v);
            }
        }
    };
    auto load_w1_chunk = [&](int c) {                            // W1[:, 64c : 64c+64] -> sW1 (zero padded)
        const int k = tid & 63, col = c * 64 + k;
        float w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = (col < O) ? __ldg(theta + L.off_w1 + ((tid >> 6) + 8 * j) * O + col) : 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) sts(tile_addr(sW1, (tid >> 6) + 8 * j, k, 64), tf32r(w[j]));
    };
    int rpar = 0;
    tile_rows(blockIdx.x, sRowBuf);
    __syncthreads();
    if (CHUNKED) load_chunk(sRowBuf, 0);
    else if (vec) prefetch_x(sRowBuf);

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // ---- P0: X and X^T tiles (data of this tile was prefetched into registers) ---------------
        long long* sRow = sRowBuf + rpar * TT;
        long long* sRowNext = sRowBuf + (rpar ^ 1) * TT;
        const bool has_next = tile + (int)gridDim.x < ntiles;
        if (has_next) tile_rows(tile + gridDim.x, sRowNext);     // visible after the next barrier
        if (CHUNKED) {
            // X is staged chunk by chunk inside P1 (and again, transposed, inside P6)
        } else if (vec) {
            const int k4 = (tid & 15) << 2;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int m = (tid >> 4) + 32 * j;
                const float4 v = make_float4(tf32r(xpre[j].x), tf32r(xpre[j].y), tf32r(xpre[j].z), tf32r(xpre[j].w));
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tile_addr(B0, m, k4, TT)), "f"(v.x),
                             "f"(v.y), "f"(v.z), "f"(v.w)
                             : "memory");
                sts(tile_addr(B1, k4 + 0, m, 64), v.x);
                sts(tile_addr(B1, k4 + 1, m, 64), v.y);
                sts(tile_addr(B1, k4 + 2, m, 64), v.z);
                sts(tile_addr(B1, k4 + 3, m, 64), v.w);
            }
        } else {
            const int k = tid & 63;
            float xv[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const long long row = sRow[(tid >> 6) + 8 * j];
                xv[j] = (row >= 0 && k < O) ? __ldg(p.b.obs + row * O + k) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int m = (tid >> 6) + 8 * j;
                const float v = tf32r(xv[j]);
                sts(tile_addr(B0, m, k, TT), v);
                sts(tile_addr(B1, k, m, 64), v);
            }
        }
        fence_async_smem();
        __syncthreads();
        // ---- P1: Z1 and Z1^T ---------------------------------------------------------------------
        if (CHUNKED) {
            for (int c = 0; c < nchunks; ++c) {
                load_w1_chunk(c);                     // the previous chunk's MMAs completed: B0 / sW1 are free
                store_chunk(B0, false);
                fence_async_smem();
                __syncthreads();
                if (c + 1 < nchunks) load_chunk(sRow, c + 1);      // next chunk's rows fly during the MMAs
                if (tid == 0) {
                    tc_fence_after();
                    tc_gemm(tmem + C_Z, B0, TT, sW1, 64, 128, 64, 64, c > 0);
                    tc_gemm(tmem + C_ZT, sW1, 64, B0, TT, 64, 128, 64, c > 0);
                    mma_commit(&bar);
                }
                mbar_wait(&bar, phase); phase ^= 1;
                tc_fence_after();
            }
        } else {
            if (tid == 0) {
                tc_fence_after();
                tc_gemm(tmem + C_Z, B0, TT, sW1, 64, 128, 64, 64, false);
                tc_gemm(tmem + C_ZT, sW1, 64, B0, TT, 64, 128, 64, false);
                mma_commit(&bar);
            }
            mbar_wait(&bar, phase); phase ^= 1;
            tc_fence_after();
        }
        {   // plain epilogue only: H1 is all that layer 2 needs
            float v[16];
            tmem_ld16(tmem + lane_base + C_Z + c16, v);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = tanh_fast(v[i] + sB1[c16 + i]);
            store_row16(B2, s_row, c16, TT, v);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        // ---- P2: Z2 (-> C_Z) and Z2^T (-> C_ZT2); the H1^T epilogue runs while these MMAs execute ----
        if (tid == 0) {
            tc_fence_after();
            tc_gemm(tmem + C_Z, B2, TT, sW2, 64, 128, 64, 64, false);
            tc_gemm(tmem + C_ZT2, sW2, 64, B2, TT, 64, 128, 64, false);
            mma_commit(&bar);
        }
        {   // deferred: H1^T = tanh(Z1^T + b1) -> B3 (B operand of dW2, needed only in P5)
            float w[32];
            tmem_ld32(tmem + lane_base + C_ZT + c32, w);
            if (lane < 16) {
                const float bb = sB1[t_row];
#pragma unroll
                for (int i = 0; i < 32; ++i) w[i] = tanh_fast(w[i] + bb);
                store_row32(B3, t_row, c32, 64, w);
            }
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        {
            float v[16];
            tmem_ld16(tmem + lane_base + C_Z + c16, v);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = tanh_fast(v[i] + sB2[c16 + i]);
            store_row16(B0, s_row, c16, TT, v);                  // H2 (X is dead)
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        // ---- P3: OUT -> loss -> dOUT (B4, cols 0..31) --------------------------------------------
        if (tid == 0) {
            tc_fence_after();
            tc_gemm(tmem + C_OUT, B0, TT, sW3, 16, 128, 16, 64, false);
            mma_commit(&bar);
        }
        {   // deferred: H2^T = tanh(Z2^T + b2) -> B2 (H1 is dead: MMA3 / MMA3T completed)
            float w[32];
            tmem_ld32(tmem + lane_base + C_ZT2 + c32, w);
            if (lane < 16) {
                const float bb = sB2[t_row];
#pragma unroll
                for (int i = 0; i < 32; ++i) w[i] = tanh_fast(w[i] + bb);
                store_row32(B2, t_row, c32, 64, w);
            }
        }
        // per-sample scalars: issue the global loads before blocking on the MMA
        float pf_act[16], pf_mu[16], pf_logp = 0.f, pf_advr = 0.f, pf_advc = 0.f, pf_tv = 0.f;
        const long long prow = (h == 0) ? sRow[s_row] : -1;
        {
#pragma unroll
            for (int a = 0; a < 16; ++a) { pf_act[a] = 0.f; pf_mu[a] = 0.f; }
            if (prow >= 0) {
                if (net == 0) {
                    const float* src = is_fvp ? p.fvp_dmu : p.b.act;
#pragma unroll
                    for (int a = 0; a < 16; ++a)
                        if (a < A) pf_act[a] = __ldg(src + prow * A + a);
                    if (is_focops) {
#pragma unroll
                        for (int a = 0; a < 16; ++a)
                            if (a < A) pf_mu[a] = __ldg(p.mu_old + prow * A + a);
                    }
                    if (!is_fvp) {
                        pf_logp = __ldg(p.b.logp + prow);
                        pf_advr = __ldg(p.b.adv_r + prow);
                        pf_advc = __ldg(p.b.adv_c + prow);
                    }
                } else {
                    pf_tv = __ldg((net == 1 ? p.b.tv_r : p.b.tv_c) + prow);
                }
            }
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        if (h == 0) {
            float st[5] = {0.f, 0.f, 0.f, 0.f, 0.f};   // loss, ratio, kl, count, focops mask
            float dls[16];
#pragma unroll
            for (int a = 0; a < 16; ++a) dls[a] = 0.f;
            float o16[16], d32[32];
            tmem_ld16(tmem + lane_base + C_OUT, o16);
#pragma unroll
            for (int i = 0; i < 32; ++i) d32[i] = 0.f;
            if (prow >= 0) {
                if (net != 0) {
                    const float d = o16[0] + sB3[0] - pf_tv;
                    st[0] = d * d; st[3] = 1.f;
                    d32[0] = 2.f * d * inv_b;
                } else if (is_fvp) {
                    // dOUT = diag(sigma^-2) J v / (rows * A): the backward below then yields J^T of it
#pragma unroll
                    for (int a = 0; a < 16; ++a)
                        if (a < A) {
                            const float sd = sLs[16 + a];
                            d32[a] = pf_act[a] / (sd * sd) * p.fvp_scale;
                        }
                    st[3] = 1.f;
                } else {
                    float logp_new = 0.f, diff[16];
#pragma unroll
                    for (int a = 0; a < 16; ++a) {
                        diff[a] = 0.f;
                        if (a < A) {
                            const float sd = sLs[16 + a];
                            const float d = pf_act[a] - (o16[a] + sB3[a]);
                            diff[a] = d;
                            logp_new += -(d * d) / (2.f * sd * sd) - sLs[a] - 0.9189385332046727f;
                        }
                    }
                    const float ratio = expf(logp_new - pf_logp);
                    const float adv_r = (pf_advr - m_r) / s_r;
                    const float adv_c = pf_advc - m_c;
                    const float adv = (adv_r - lam * adv_c) / (1.f + lam);
                    float dlogp, loss, dmask = 0.f;
                    if (is_focops) {
                        // first_order/focops.py:L62-108 incl. the reference's [b,1] x [b] broadcast:
                        //   loss = mean_i(mask_i kl_i) - mean_i(mask_i) * mean_j(ratio_j adv_j) / lam
                        float kl = 0.f;
#pragma unroll
                        for (int a = 0; a < 16; ++a)
                            if (a < A) {
                                const float sn = sLs[16 + a];
                                const float dm = (o16[a] + sB3[a]) - pf_mu[a];
                                kl += (sOld[a] - sLs[a]) + (sn * sn + dm * dm) * 0.5f * sOld[16 + a] - 0.5f;
                            }
                        dmask = (kl <= p.focops_eta) ? 1.f : 0.f;
                        const float mbar = p.focops_mask_mean ? __ldg(p.focops_mask_mean) : dmask;
                        loss = kl * dmask - mbar * ratio * adv / p.focops_lam;
                        dlogp = -mbar * adv * ratio / p.focops_lam * inv_b;
                        st[2] = kl; st[4] = dmask;
                    } else if (p.kind == TC_PPO_CLIP || is_p3o) {
                        const float rc = fminf(fmaxf(ratio, 1.f - p.clip), 1.f + p.clip);
                        const float s1 = ratio * adv, s2 = rc * adv;
                        loss = -fminf(s1, s2);
                        dlogp = (s1 <= s2) ? -adv * ratio * inv_b : 0.f;
                        if (is_p3o) {   // + kappa * relu(mean(ratio adv_c) + Jc - limit), gate from pass 1
                            const bool pass2 = p.focops_mask_mean != nullptr;
                            const float gate = pass2 ? __ldg(p.focops_mask_mean) : 0.f;
                            dlogp += gate * adv_c * ratio * inv_b;
                            st[2] = pass2 ? gate * (ratio * adv_c + p.focops_eta) : ratio * adv_c;   // Loss/Loss_pi_cost
                        }
                    } else if (p.kind == TC_RATIO) {
                        loss = -ratio * adv; dlogp = -adv * ratio * inv_b;
                    } else {
                        loss = ratio * adv_c; dlogp = adv_c * ratio * inv_b;
                    }
                    st[0] = loss; st[1] = ratio; st[3] = 1.f;
#pragma unroll
                    for (int a = 0; a < 16; ++a)
                        if (a < A) {
                            const float sd = sLs[16 + a];
                            const float iv = 1.f / (sd * sd);
                            d32[a] = dlogp * diff[a] * iv;
                            dls[a] = dlogp * (diff[a] * diff[a] * iv - 1.f);
                            if (is_focops) {
                                const float dm = (o16[a] + sB3[a]) - pf_mu[a];
                                d32[a] += dmask * inv_b * dm * sOld[16 + a];
                                dls[a] += dmask * inv_b * (sd * sd * sOld[16 + a] - 1.f);
                            }
                        }
                }
            }
            store_row32(B4, s_row, 0, TT, d32);
#pragma unroll
            for (int o = 0; o < 16; ++o) sts(tile_addr(B4 + 16384u, o, s_row, 16), tf32r(d32[o]));   // dOUT^T [o][s]
            // deterministic reductions over the 128 sample threads (warps with h == 0)
#pragma unroll
            for (int i = 0; i < 5; ++i) st[i] = warp_sum(st[i]);
            if (net == 0) {
#pragma unroll
                for (int a = 0; a < 16; ++a) dls[a] = warp_sum(dls[a]);
            }
            float db[16];   // db3[o] = sum_s dOUT[s][o]
#pragma unroll
            for (int a = 0; a < 16; ++a) db[a] = (a < L.out) ? warp_sum(d32[a]) : 0.f;
            if (lane == 0) {
#pragma unroll
                for (int i = 0; i < 5; ++i) sRed[q * 8 + i] = st[i];
#pragma unroll
                for (int a = 0; a < 16; ++a) { sRed[32 + q * 16 + a] = dls[a]; sRed[96 + q * 16 + a] = db[a]; }
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid < 5) sStat[tid] += sRed[tid] + sRed[8 + tid] + sRed[16 + tid] + sRed[24 + tid];
        if (net == 0 && tid >= 32 && tid < 48) {
            const int a = tid - 32;
            sLs[32 + a] += sRed[32 + a] + sRed[48 + a] + sRed[64 + a] + sRed[80 + a];
        }
        if (tid >= 64 && tid < 64 + L.out) {
            const int a = tid - 64;
            sB3acc[a] += sRed[96 + a] + sRed[112 + a] + sRed[128 + a] + sRed[144 + a];
        }
        if (EXT && p.forward_only) {   // FOCOPS / P3O pass 1: statistics only
            if (CHUNKED) { if (has_next) load_chunk(sRowNext, 0); }
            else if (vec && has_next) prefetch_x(sRowNext);
            first_tile = false;
            rpar ^= 1;
            __syncthreads();
            continue;
        }
        // ---- P4: dZ2, dZ2^T and dW3^T += H2^T dOUT ------------------------------------------------
        if (tid == 0) {
            tc_fence_after();
            tc_gemm(tmem + C_Z, B4, TT, sW3T, 64, 128, 64, 16, false);
            tc_gemm(tmem + C_ZT, sW3T, 64, B4, TT, 64, 128, 16, false);
            tc_gemm(tmem + C_DW3, B2, 64, B4 + 16384u, 16, 64, 16, 128, !first_tile);
            mma_commit(&bar);
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        {
            float w[32], hh[32];
            tmem_ld32(tmem + lane_base + C_ZT + c32, w);
            if (lane < 16) {
                load_row32(B2, t_row, c32, 64, hh);              // H2^T
#pragma unroll
                for (int i = 0; i < 32; ++i) w[i] *= (1.f - hh[i] * hh[i]);
                store_row32(B4, t_row, c32, 64, w);              // dZ2^T [k][s]
            }
        }
        __syncthreads();           // every read of H2^T (B2) is done before dZ2 overwrites it
        {
            float v[16], hh[16];
            tmem_ld16(tmem + lane_base + C_Z + c16, v);
            load_row16(B0, s_row, c16, TT, hh);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] *= (1.f - hh[i] * hh[i]);
            store_row16(B2, s_row, c16, TT, v);                  // dZ2 [s][k]
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        // ---- P5: dW2 += dZ2^T H1 ; dZ1^T = W2^T dZ2^T --------------------------------------------
        if (CHUNKED) load_chunk(sRow, 0);             // chunk 0 of THIS tile again: P6 needs X^T chunk by chunk
        else if (vec && has_next) prefetch_x(sRowNext);    // global loads of the next tile fly during P5 / P6
        if (tid == 0) {
            tc_fence_after();
            tc_gemm(tmem + C_DW2, B4, 64, B3, 64, 64, 64, 128, !first_tile);
            tc_gemm(tmem + C_ZT, sW2T, 64, B2, TT, 64, 128, 64, false);
            mma_commit(&bar);
        }
        if (tid < 64) {   // db2[j] = sum_s dZ2^T[j][s]
            float c = 0.f, v[32];
#pragma unroll 1
            for (int a4 = 0; a4 < 4; ++a4) {
                load_row32(B4, tid, 32 * a4, 64, v);
#pragma unroll
                for (int i = 0; i < 32; ++i) c += v[i];
            }
            ab2 += c;
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        {
            float w[32], hh[32];
            tmem_ld32(tmem + lane_base + C_ZT + c32, w);
            if (lane < 16) {
                load_row32(B3, t_row, c32, 64, hh);
#pragma unroll
                for (int i = 0; i < 32; ++i) w[i] *= (1.f - hh[i] * hh[i]);
                store_row32(B0, t_row, c32, 64, w);              // dZ1^T [k][s] (H2 is dead)
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        // ---- P6: dW1 += dZ1^T X --------------------------------------------------------------------
        if (CHUNKED) {
            for (int c = 0; c < nchunks; ++c) {
                store_chunk(B1, true);               // X^T chunk [64 k][128 s]
                fence_async_smem();
                tc_fence_before();                   // (c > 0) every read of the previous chunk's accumulator is done
                __syncthreads();
                if (c + 1 < nchunks) load_chunk(sRow, c + 1);
                if (tid == 0) {
                    tc_fence_after();
                    tc_gemm(tmem + C_DW1, B0, 64, B1, 64, 64, 64, 128, false);
                    mma_commit(&bar);
                }
                if (c == 0 && tid < 64) {   // db1[j] = sum_s dZ1^T[j][s]
                    float cs = 0.f, v[32];
#pragma unroll 1
                    for (int a4 = 0; a4 < 4; ++a4) {
                        load_row32(B0, tid, 32 * a4, 64, v);
#pragma unroll
                        for (int i = 0; i < 32; ++i) cs += v[i];
                    }
                    ab1 += cs;
                }
                mbar_wait(&bar, phase); phase ^= 1;
                tc_fence_after();
                {   // flush this chunk of dW1 into the CTA's partial gradient (each element owned by one thread)
                    float v[16];
                    tmem_ld16(tmem + lane_base + C_DW1 + c16, v);
                    if (lane < 16) {
                        float* qrow = gout + L.off_w1 + t_row * O + c * 64 + c16;
                        const int nvalid = O - (c * 64 + c16);          // columns of this 16-group inside [0, O)
                        if (!first_tile) {                              // all loads first (independent), then the stores
                            float old[16];
#pragma unroll
                            for (int i = 0; i < 16; ++i) old[i] = (i < nvalid) ? __ldcg(qrow + i) : 0.f;
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] += old[i];
                        }
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            if (i < nvalid) __stcg(qrow + i, v[i]);
                    }
                }
            }
            if (has_next) load_chunk(sRowNext, 0);
        } else {
        if (tid == 0) {
            tc_fence_after();
            tc_gemm(tmem + C_DW1, B0, 64, B1, 64, 64, 64, 128, !first_tile);
            mma_commit(&bar);
        }
        if (tid < 64) {   // db1[j] = sum_s dZ1^T[j][s]
            float c = 0.f, v[32];
#pragma unroll 1
            for (int a4 = 0; a4 < 4; ++a4) {
                load_row32(B0, tid, 32 * a4, 64, v);
#pragma unroll
                for (int i = 0; i < 32; ++i) c += v[i];
            }
            ab1 += c;
        }
        mbar_wait(&bar, phase); phase ^= 1;      // B0 / B1 are rewritten by the next tile's gather
        tc_fence_after();
        }
        first_tile = false;
        rpar ^= 1;
        __syncthreads();
    }

    // ---- write this CTA's partial gradient segment (staged through smem so that stores coalesce) ----
    if (EXT && p.forward_only) {
        if (tid < 8) p.stats_part[((size_t)blockIdx.x * 3 + net) * 8 + tid] = sStat[tid];
    } else {
        float v[16];
        float* stage = reinterpret_cast<float*>(smem_raw + pad);            // B0 region: [2][64][65]
        tmem_ld16(tmem + lane_base + C_DW2 + c16, v);
        if (lane < 16)
#pragma unroll
            for (int i = 0; i < 16; ++i) stage[t_row * 65 + c16 + i] = v[i];
        if (!CHUNKED) {
            tmem_ld16(tmem + lane_base + C_DW1 + c16, v);
            if (lane < 16)
#pragma unroll
                for (int i = 0; i < 16; ++i) stage[64 * 65 + t_row * 65 + c16 + i] = v[i];
        }
        if (h == 0) {   // dW3^T [k][o] accumulator (M = 64 layout)
            tmem_ld16(tmem + lane_base + C_DW3, v);
            if (lane < 16)
#pragma unroll
                for (int o = 0; o < 16; ++o) stage[2 * 64 * 65 + o * 65 + t_row] = v[o];
        }
        __syncthreads();
        for (int i = tid; i < 64 * 64; i += NTC) gout[L.off_w2 + i] = stage[(i >> 6) * 65 + (i & 63)];
        if (!CHUNKED)
            for (int i = tid; i < 64 * O; i += NTC) gout[L.off_w1 + i] = stage[64 * 65 + (i / O) * 65 + (i % O)];
        for (int i = tid; i < L.out * 64; i += NTC) gout[L.off_w3 + i] = stage[2 * 64 * 65 + (i >> 6) * 65 + (i & 63)];
        if (tid < 64) { gout[L.off_b1 + tid] = ab1; gout[L.off_b2 + tid] = ab2; }
        if (tid < L.out) gout[L.off_b3 + tid] = sB3acc[tid];
        if (net == 0 && tid < A) {
            float g = sLs[32 + tid];
            if (blockIdx.x == 0 && (p.kind == TC_PPO_CLIP || is_p3o || is_focops)) g -= p.entropy_coef / (float)A;
            // log_std block of the Fisher matrix: (2/A) v, counted once (natural_pg.py:L74-119, analytic form)
            if (is_fvp) g = (blockIdx.x == 0) ? 2.f / (float)A * __ldg(p.fvp_vec + L.off_logstd + tid) : 0.f;
            gout[L.off_logstd + tid] = g;
        }
        if (tid < 8) p.stats_part[((size_t)blockIdx.x * 3 + net) * 8 + tid] = sStat[tid];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------
// Forward-mode tangent pass of the Fisher-vector product (NaturalPG._fvp, base/natural_pg.py:L74-119):
//   dmu[row][a] = J_mu(row) v      for the rows 0, stride, 2*stride, ...
// The weight tile of every layer is stored with the direction's block stacked under it
// ([W ; V], 128 rows), so ONE N = 128 MMA yields the pre-activation and the first tangent term:
//     [Z1 | X V1^T]            = X   [W1;V1]^T
//     [Z2 | H1 V2^T + dH1 W2^T] = H1 [W2;V2]^T  (+)  dH1 W2^T   (accumulated into the right half)
//     dmu                       = H2 V3^T + dH2 W3^T + vb3
// The backward half (J^T diag(sigma^-2) dmu) is minibatch_grad_tc_kernel with kind TC_FVP.
struct FvpTanArgs {
    const float* obs; long long total; int stride;
    const float* theta; const float* vec; float* dmu; int O, A;
};
constexpr uint32_t F_Z1 = 0, F_Z2 = 128, F_DMU = 256;

template <bool CHUNKED>     // obs dim > 64: K loop over 64-column chunks of X / [W1;V1]
__global__ void __launch_bounds__(NTC, 1) fvp_tangent_tc_kernel(FvpTanArgs p) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
    const uint32_t B0 = smem_u32(smem_raw) + pad;   // X -> H2
    const uint32_t B1 = B0 + BUF;                   // H1 -> dH2
    const uint32_t B2 = B1 + BUF;                   // dH1
    const uint32_t sWV1 = B2 + BUF;                 // [128][64]: rows 0..63 W1, 64..127 V1
    const uint32_t sWV2 = sWV1 + 32768;             // [128][64]: W2 ; V2
    const uint32_t sWV3 = sWV2 + 32768;             // [32][64]:  rows 0..15 W3, 16..31 V3
    float* sB1 = reinterpret_cast<float*>(smem_raw + pad + 3 * BUF + 2 * 32768 + 8192);
    float* sB2 = sB1 + 64;
    float* sVB1 = sB2 + 64;
    float* sVB2 = sVB1 + 64;
    float* sVB3 = sVB2 + 64;           // [16]
    long long* sRowBuf = reinterpret_cast<long long*>(sVB3 + 16);   // [2][128]
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int O = p.O, A = p.A;
    const NetLayout L = actor_layout(O, A);
    const long long nrows = (p.total + p.stride - 1) / p.stride;
    const int ntiles = (int)((nrows + TT - 1) / TT);

    {   // stacked weight tiles (loads batched so they are all in flight together)
        float w1v[8], v1v[8], w2v[8], v2v[8], w3v[2], v3v[2];
        const int k = tid & 63;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = (tid >> 6) + 8 * j;
            w1v[j] = (!CHUNKED && k < O) ? __ldg(p.theta + L.off_w1 + n * O + k) : 0.f;
            v1v[j] = (!CHUNKED && k < O) ? __ldg(p.vec + L.off_w1 + n * O + k) : 0.f;
            w2v[j] = __ldg(p.theta + L.off_w2 + n * 64 + k);
            v2v[j] = __ldg(p.vec + L.off_w2 + n * 64 + k);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int o = (tid >> 6) + 8 * j;
            w3v[j] = (o < A) ? __ldg(p.theta + L.off_w3 + o * 64 + k) : 0.f;
            v3v[j] = (o < A) ? __ldg(p.vec + L.off_w3 + o * 64 + k) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = (tid >> 6) + 8 * j;
            sts(tile_addr(sWV1, n, k, 128), tf32r(w1v[j]));
            sts(tile_addr(sWV1, 64 + n, k, 128), tf32r(v1v[j]));
            sts(tile_addr(sWV2, n, k, 128), tf32r(w2v[j]));
            sts(tile_addr(sWV2, 64 + n, k, 128), tf32r(v2v[j]));
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int o = (tid >> 6) + 8 * j;
            sts(tile_addr(sWV3, o, k, 32), tf32r(w3v[j]));
            sts(tile_addr(sWV3, 16 + o, k, 32), tf32r(v3v[j]));
        }
    }
    if (tid < 64) {
        sB1[tid] = __ldg(p.theta + L.off_b1 + tid); sB2[tid] = __ldg(p.theta + L.off_b2 + tid);
        sVB1[tid] = __ldg(p.vec + L.off_b1 + tid); sVB2[tid] = __ldg(p.vec + L.off_b2 + tid);
    }
    if (tid < 16) sVB3[tid] = (tid < A) ? __ldg(p.vec + L.off_b3 + tid) : 0.f;
    if (tid == 0) { mbar_init(&bar, 1); mbar_init_fence(); }
    if (warp == 0) tmem_alloc(&tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    uint32_t phase = 0;
    const int s_row = 32 * q + lane, c16 = 16 * h;

    const bool vec4 = (O & 3) == 0;
    auto tile_rows = [&](int tile, long long* dst) {
        if (tid < TT) {
            const long long k = (long long)tile * TT + tid;
            dst[tid] = (k < nrows) ? k * p.stride : -1;
        }
    };
    float4 xpre[4];
    auto prefetch_x = [&](const long long* rows) {
        const int k4 = (tid & 15) << 2;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const long long row = rows[(tid >> 4) + 32 * j];
            xpre[j] = (row >= 0 && k4 < O) ? __ldg(reinterpret_cast<const float4*>(p.obs + row * O + k4))
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    const int nchunks = (O + 63) >> 6;
    float xr[16];
    auto load_chunk = [&](const long long* rows, int c) {
        if (vec4) {
            const int col = c * 64 + ((tid & 15) << 2);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const long long row = rows[(tid >> 4) + 32 * j];
                const float4 v = (row >= 0 && col < O) ? __ldg(reinterpret_cast<const float4*>(p.obs + row * O + col))
                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                xr[4 * j] = v.x; xr[4 * j + 1] = v.y; xr[4 * j + 2] = v.z; xr[4 * j + 3] = v.w;
            }
        } else {
            const int col = c * 64 + (tid & 63);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const long long row = rows[(tid >> 6) + 8 * j];
                xr[j] = (row >= 0 && col < O) ? __ldg(p.obs + row * O + col) : 0.f;
            }
        }
    };
    auto store_chunk = [&]() {
        if (vec4) {
            const int k4 = (tid & 15) << 2;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tile_addr(B0, (tid >> 4) + 32 * j, k4, TT)),
                             "f"(tf32r(xr[4 * j])), "f"(tf32r(xr[4 * j + 1])), "f"(tf32r(xr[4 * j + 2])), "f"(tf32r(xr[4 * j + 3]))
                             : "memory");
        } else {
            const int k = tid & 63;
#pragma unroll
            for (int j = 0; j < 16; ++j) sts(tile_addr(B0, (tid >> 6) + 8 * j, k, TT), tf32r(xr[j]));
        }
    };
    auto load_wv1_chunk = [&](int c) {                 // [W1 ; V1][:, 64c : 64c+64] -> sWV1 (zero padded)
        const int k = tid & 63, col = c * 64 + k;
        float w[8], v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = (tid >> 6) + 8 * j;
            w[j] = (col < O) ? __ldg(p.theta + L.off_w1 + n * O + col) : 0.f;
            v[j] = (col < O) ? __ldg(p.vec + L.off_w1 + n * O + col) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = (tid >> 6) + 8 * j;
            sts(tile_addr(sWV1, n, k, 128), tf32r(w[j]));
            sts(tile_addr(sWV1, 64 + n, k, 128), tf32r(v[j]));
        }
    };
    int rpar = 0;
    tile_rows(blockIdx.x, sRowBuf);
    __syncthreads();
    if (CHUNKED) load_chunk(sRowBuf, 0);
    else if (vec4) prefetch_x(sRowBuf);

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        long long* sRow = sRowBuf + rpar * TT;
        long long* sRowNext = sRowBuf + (rpar ^ 1) * TT;
        const bool has_next = tile + (int)gridDim.x < ntiles;
        if (has_next) tile_rows(tile + gridDim.x, sRowNext);
        if (CHUNKED) {
            // staged chunk by chunk below
        } else if (vec4) {
            const int k4 = (tid & 15) << 2;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int m = (tid >> 4) + 32 * j;
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tile_addr(B0, m, k4, TT)),
                             "f"(tf32r(xpre[j].x)), "f"(tf32r(xpre[j].y)), "f"(tf32r(xpre[j].z)), "f"(tf32r(xpre[j].w))
                             : "memory");
            }
        } else {
            const int k = tid & 63;
            float xv[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const long long row = sRow[(tid >> 6) + 8 * j];
                xv[j] = (row >= 0 && k < O) ? __ldg(p.obs + row * O + k) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) sts(tile_addr(B0, (tid >> 6) + 8 * j, k, TT), tf32r(xv[j]));
        }
        fence_async_smem();
        __syncthreads();
        // ---- layer 1: [Z1 | X V1^T] ----------------------------------------------------------------
        if (CHUNKED) {
            for (int c = 0; c < nchunks; ++c) {
                load_wv1_chunk(c);
                store_chunk();
                fence_async_smem();
                __syncthreads();
                if (c + 1 < nchunks) load_chunk(sRow, c + 1);
                else if (has_next) load_chunk(sRowNext, 0);
                if (tid == 0) {
                    tc_fence_after();
                    tc_gemm(tmem + F_Z1, B0, TT, sWV1, 128, 128, 128, 64, c > 0);
                    mma_commit(&bar);
                }
                mbar_wait(&bar, phase); phase ^= 1;
                tc_fence_after();
            }
        } else {
            if (vec4 && has_next) prefetch_x(sRowNext);      // next tile's rows fly during the three layers
            if (tid == 0) {
                tc_fence_after();
                tc_gemm(tmem + F_Z1, B0, TT, sWV1, 128, 128, 128, 64, false);
                mma_commit(&bar);
            }
            mbar_wait(&bar, phase); phase ^= 1;
            tc_fence_after();
        }
        {
            float z[16], dz[16];
            tmem_ld16(tmem + lane_base + F_Z1 + c16, z);
            tmem_ld16(tmem + lane_base + F_Z1 + 64 + c16, dz);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float hh = tanh_fast(z[i] + sB1[c16 + i]);
                dz[i] = (1.f - hh * hh) * (dz[i] + sVB1[c16 + i]);
                z[i] = hh;
            }
            store_row16(B1, s_row, c16, TT, z);      // H1
            store_row16(B2, s_row, c16, TT, dz);     // dH1
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        // ---- layer 2: [Z2 | H1 V2^T + dH1 W2^T] ------------------------------------------------------
        if (tid == 0) {
            tc_fence_after();
            tc_gemm(tmem + F_Z2, B1, TT, sWV2, 128, 128, 128, 64, false);
            tc_gemm(tmem + F_Z2 + 64, B2, TT, sWV2, 128, 128, 64, 64, true);
            mma_commit(&bar);
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        {
            float z[16], dz[16];
            tmem_ld16(tmem + lane_base + F_Z2 + c16, z);
            tmem_ld16(tmem + lane_base + F_Z2 + 64 + c16, dz);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float hh = tanh_fast(z[i] + sB2[c16 + i]);
                dz[i] = (1.f - hh * hh) * (dz[i] + sVB2[c16 + i]);
                z[i] = hh;
            }
            store_row16(B0, s_row, c16, TT, z);      // H2  (X is dead)
            store_row16(B1, s_row, c16, TT, dz);     // dH2 (H1 is dead: layer-2 MMAs completed)
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        // ---- output tangent: dmu = H2 V3^T + dH2 W3^T + vb3 -------------------------------------------
        if (tid == 0) {
            tc_fence_after();
            tc_gemm(tmem + F_DMU, B0, TT, sWV3 + 2048u, 32, 128, 16, 64, false);
            tc_gemm(tmem + F_DMU, B1, TT, sWV3, 32, 128, 16, 64, true);
            mma_commit(&bar);
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        if (h == 0) {
            float o16[16];
            tmem_ld16(tmem + lane_base + F_DMU, o16);
            const long long row = sRow[s_row];
            if (row >= 0) {
#pragma unroll
                for (int a = 0; a < 16; ++a)
                    if (a < A) p.dmu[row * A + a] = o16[a] + sVB3[a];
            }
        }
        tc_fence_before();
        rpar ^= 1;
        __syncthreads();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, TMEM_COLS);
}

}  // namespace osb

using namespace osb;

static size_t tc_smem_bytes() {
    return 1024 + 5 * (size_t)BUF + 3 * 16384 + 4096 + 8192 + (64 + 64 + 16 + 48 + 8 + 160 + 16 + 32) * 4 + 2 * 128 * 8 + 64;
}
static size_t fvp_tan_smem_bytes() {
    return 1024 + 3 * (size_t)BUF + 2 * 32768 + 8192 + (4 * 64 + 16) * 4 + 2 * 128 * 8 + 64;
}

static int launch_grad_tc(const TcArgs& p, int nblocks, cudaStream_t stream) {
    const size_t smem = tc_smem_bytes();
    static bool attr = false;
    if (!attr) {
        OSB_CUDA(cudaFuncSetAttribute(minibatch_grad_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        OSB_CUDA(cudaFuncSetAttribute(minibatch_grad_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        OSB_CUDA(cudaFuncSetAttribute(minibatch_grad_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        OSB_CUDA(cudaFuncSetAttribute(minibatch_grad_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = true;
    }
    const bool single = (p.net_mask & (p.net_mask - 1)) == 0;     // one network: it gets every CTA
    dim3 grid(nblocks, single ? 1 : 3);
    const bool ext = p.kind == TC_FOCOPS || p.kind == TC_FVP || p.kind == TC_P3O;
    if (p.O > 64) {
        if (ext) minibatch_grad_tc_kernel<true, true><<<grid, NTC, smem, stream>>>(p);
        else minibatch_grad_tc_kernel<true, false><<<grid, NTC, smem, stream>>>(p);
    } else {
        if (ext) minibatch_grad_tc_kernel<false, true><<<grid, NTC, smem, stream>>>(p);
        else minibatch_grad_tc_kernel<false, false><<<grid, NTC, smem, stream>>>(p);
    }
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

extern "C" {

// CTAs along x of the tensor-core kernel: three networks share the 148 SMs (49 each); a single
// network (full-batch actor passes of the natural-gradient family) spreads over all of them.
int osb_tc_grid_blocks(long long rows, int net_mask) {
    const long long tiles = (rows + TT - 1) / TT;
    const int cap = ((net_mask & (net_mask - 1)) == 0) ? 148 : 49;
    return (int)(tiles < cap ? tiles : cap);
}

// FOCOPS pass 1 -> mean_i mask_i of the minibatch (stats slot 4 / slot 3 of the actor), fixed order.
//   P3O:    out = kappa if mean_i(ratio_i adv_c_i) + (Jc - limit) > 0 else 0   (slot 2 / slot 3)
__global__ void tc_mask_mean_kernel(const float* __restrict__ stats_part, int nblocks, float* __restrict__ out,
                                    const int* __restrict__ stop_flag, int kind, float kappa, float jc_minus_limit) {
    if (threadIdx.x != 0 || (stop_flag && *stop_flag)) return;
    const int slot = (kind == TC_P3O) ? 2 : 4;
    float m = 0.f, n = 0.f;
    for (int b = 0; b < nblocks; ++b) { m += stats_part[((size_t)b * 3) * 8 + slot]; n += stats_part[((size_t)b * 3) * 8 + 3]; }
    const float mean = n > 0.f ? m / n : 0.f;
    out[0] = (kind == TC_P3O) ? ((mean + jc_minus_limit > 0.f) ? kappa : 0.f) : mean;
}

// Tensor-core (TF32 tcgen05) variant of osb_minibatch_grad: same arguments, O <= 64, A <= 16.
// gpart holds osb_tc_grid_blocks(mb_count, net_mask) rows of P floats.
int osb_minibatch_grad_tc(const float* theta, int O, int A, const float* obs, const float* act,
                          const float* logp, const float* adv_r, const float* adv_c,
                          const float* tv_r, const float* tv_c, const float* mu_old,
                          const float* moments, const int* perm, long long total, unsigned perm_seed,
                          long long mb_start, int mb_count, int loss_kind, float clip,
                          float entropy_coef, float focops_lam, float focops_eta,
                          const float* lagrange, const float* logstd_old, int net_mask, float* gpart,
                          float* stats_part, const int* stop_flag, void* stream) {
    static float* d_mask_mean = nullptr;   // FOCOPS scratch scalar
    OSB_CHECK_ARG(theta && obs && act && logp && adv_r && adv_c && tv_r && tv_c && moments, "null input");
    OSB_CHECK_ARG(O > 0 && O <= 512 && A > 0 && A <= 16 && mb_count > 0 && total > 0, "tensor-core path needs O <= 512, A <= 16");
    OSB_CHECK_ARG(mb_start >= 0 && mb_start + mb_count <= total, "minibatch window out of range");
    OSB_CHECK_ARG((loss_kind >= 0 && loss_kind <= 3) || loss_kind == TC_P3O, "loss kind");
    OSB_CHECK_ARG(loss_kind != TC_FOCOPS || (mu_old && logstd_old), "FOCOPS needs mu_old/logstd_old");
    OSB_CHECK_ARG(net_mask > 0 && net_mask < 8, "net_mask");
    TcArgs p;
    p.b = TcBatch{obs, act, logp, adv_r, adv_c, tv_r, tv_c, moments, perm, total, perm_seed, mb_start, mb_count, 0};
    p.kind = loss_kind; p.clip = clip; p.entropy_coef = entropy_coef; p.lagrange = lagrange;
    p.theta = theta; p.gpart = gpart; p.stats_part = stats_part; p.stop_flag = stop_flag;
    p.O = O; p.A = A; p.P = actor_layout(O, A).size + 2 * critic_layout(O, A).size; p.net_mask = net_mask;
    p.fvp_dmu = nullptr; p.fvp_vec = nullptr; p.fvp_scale = 0.f;
    p.mu_old = mu_old; p.logstd_old = logstd_old; p.focops_lam = focops_lam; p.focops_eta = focops_eta;
    p.focops_mask_mean = nullptr; p.forward_only = 0;
    const int nb = osb_tc_grid_blocks(mb_count, net_mask);
    if ((loss_kind == TC_FOCOPS || loss_kind == TC_P3O) && (net_mask & 1)) {
        // pass 1: actor forward only -> mean mask of the minibatch (the reference's [b,1] x [b] broadcast)
        if (!d_mask_mean) OSB_CUDA(cudaMalloc(&d_mask_mean, sizeof(float)));
        TcArgs q = p;
        q.forward_only = 1; q.net_mask = 1;
        const int nb1 = osb_tc_grid_blocks(mb_count, 1);
        int rc = launch_grad_tc(q, nb1, (cudaStream_t)stream);
        if (rc) return rc;
        tc_mask_mean_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(stats_part, nb1, d_mask_mean, stop_flag, loss_kind,
                                                                focops_lam, focops_eta);
        OSB_LAUNCH_CHECK();
        p.focops_mask_mean = d_mask_mean;
    }
    return launch_grad_tc(p, nb, (cudaStream_t)stream);
}

// Tensor-core Fisher-vector product partials (O <= 64): tangent forward (dmu scratch [total][A]) then
// the actor backward of minibatch_grad_tc_kernel.  gpart: osb_tc_grid_blocks(rows, 1) rows of
// P_actor floats; stats_scratch: that many * 24 floats.  Reduce with osb_reduce_partials.
int osb_fvp_partials_tc(const float* theta_actor, const float* vec, int O, int A, const float* obs,
                        long long total, int stride, float* dmu, float* gpart, float* stats_scratch,
                        void* stream) {
    OSB_CHECK_ARG(theta_actor && vec && obs && dmu && gpart && stats_scratch && total > 0 && stride > 0, "bad argument");
    OSB_CHECK_ARG(O > 0 && O <= 512 && A > 0 && A <= 16, "tensor-core path needs O <= 512, A <= 16");
    const long long nrows = (total + stride - 1) / stride;
    OSB_CHECK_ARG(nrows < (1ll << 31), "too many rows");
    const int nb = osb_tc_grid_blocks(nrows, 1);
    cudaStream_t s = (cudaStream_t)stream;
    {
        FvpTanArgs t{obs, total, stride, theta_actor, vec, dmu, O, A};
        const size_t smem = fvp_tan_smem_bytes();
        static bool attr = false;
        if (!attr) {
            OSB_CUDA(cudaFuncSetAttribute(fvp_tangent_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            OSB_CUDA(cudaFuncSetAttribute(fvp_tangent_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr = true;
        }
        if (O > 64) fvp_tangent_tc_kernel<true><<<nb, NTC, smem, s>>>(t);
        else fvp_tangent_tc_kernel<false><<<nb, NTC, smem, s>>>(t);
        OSB_LAUNCH_CHECK();
    }
    TcArgs p;
    p.b = TcBatch{obs, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, total, 0u, 0, (int)nrows, stride};
    p.kind = TC_FVP; p.clip = 0.f; p.entropy_coef = 0.f; p.lagrange = nullptr;
    p.theta = theta_actor; p.gpart = gpart; p.stats_part = stats_scratch; p.stop_flag = nullptr;
    p.O = O; p.A = A; p.P = actor_layout(O, A).size; p.net_mask = 1;
    p.fvp_dmu = dmu; p.fvp_vec = vec; p.fvp_scale = 1.0f / ((float)nrows * (float)A);
    p.mu_old = nullptr; p.logstd_old = nullptr; p.focops_lam = 1.f; p.focops_eta = 0.f;
    p.focops_mask_mean = nullptr; p.forward_only = 0;
    return launch_grad_tc(p, nb, s);
}

}  // extern "C"
