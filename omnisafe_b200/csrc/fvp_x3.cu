// Split-bf16 (parity-grade tensor-core) Fisher-vector product, forward half: the tangent of the policy mean along a
// parameter direction v, for every sample of the batch.
//
//   NaturalPG._fvp (algorithms/on_policy/base/natural_pg.py:L74-119):  F v = grad( (grad KL)^T v ), which for the
//   Gaussian actor at theta = theta_old is  [ (2 / A) v_logsigma ;  (1 / (B A)) sum_s J(s)^T diag(sigma^-2) J(s) v_mu ]
//   (SURVEY §8a row 13).  This kernel computes d mu(s) = J(s) v_mu by forward-mode differentiation of the MLP:
//       T1 = X V1^T + bv1,              dH1 = (1 - H1^2) T1
//       T2 = dH1 W2^T + H1 V2^T + bv2,  dH2 = (1 - H2^2) T2
//       dmu = dH2 W3^T + H2 V3^T + bv3
//   next to the ordinary forward (Z1 = X W1^T + b1, H1 = tanh Z1, ...), every GEMM as six kind::f16 MMAs over the three
//   bf16 pieces of its fp32 operands (csrc/x3.cuh) with fp32 accumulation in TMEM.  The backward half J^T diag(sigma^-2)
//   dmu / (B A) is minibatch_grad_x3_kernel with the supplied-dOUT loss kind (csrc/update_x3.cu).
//
// One CTA per SM, tiles of 128 samples: two activation buffers (value and tangent; X / H1 / H2 overwrite each other in
// place, as do dH1 / dH2), the weights W1 V1 W2 V2 W3 V3 resident as bf16x3 tiles (204 KB of shared memory in all).
#include "common.cuh"
#include "mlp.cuh"
#include "x3.cuh"

namespace osb {

using namespace x3;

constexpr int FT = 128;
constexpr int FNT = 256;                                             // 8 warps: lane quarter q = warp % 4, column half h = warp / 4
constexpr uint32_t F_SUB = FT * 128, F_ACT = 3 * F_SUB;              // [128][64] bf16 x3
constexpr uint32_t F_WSUB = 64 * 128, F_W = 3 * F_WSUB, F_W3SUB = 16 * 128, F_W3 = 3 * F_W3SUB;
constexpr uint32_t FO_A0 = 0, FO_A1 = F_ACT, FO_W1 = 2 * F_ACT, FO_V1 = FO_W1 + F_W, FO_W2 = FO_V1 + F_W, FO_V2 = FO_W2 + F_W,
                   FO_W3 = FO_V2 + F_W, FO_V3 = FO_W3 + F_W3, FO_MISC = FO_V3 + F_W3;
// misc floats: b1[64] bv1[64] b2[64] bv2[64] bv3[16]; long long rows[128]; barrier; tmem slot
constexpr uint32_t FO_ROWS = FO_MISC + (4 * 64 + 16) * 4, FO_BAR = FO_ROWS + FT * 8, FO_SLOT = FO_BAR + 8, F_SMEM = FO_SLOT + 8;

struct FvpX3Args {
    const float* obs; long long total; int stride;
    const float* theta; const float* vec; float* dmu;
    int O, A;
};

// [rows][64] (rows = 64 or 16, zero padded) fp32 matrix with row pitch `ld` -> bf16x3 SW128 tile
__device__ __forceinline__ void stage_matrix_x3(uint32_t dst, uint32_t sub, const float* __restrict__ src, int rows_valid,
                                                int rows, int ld, int cols_valid, int tid) {
    for (int i = tid; i < rows * 32; i += FNT) {
        const int n = i >> 5, k = (i & 31) << 1;
        const float a = (n < rows_valid && k < cols_valid) ? __ldg(src + n * ld + k) : 0.f;
        const float b = (n < rows_valid && k + 1 < cols_valid) ? __ldg(src + n * ld + k + 1) : 0.f;
        uint32_t w0, w1, w2;
        split2(a, b, w0, w1, w2);
        const uint32_t off = off128(n, k);
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(dst + off), "r"(w0) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(dst + sub + off), "r"(w1) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(dst + 2 * sub + off), "r"(w2) : "memory");
    }
}

__global__ void __launch_bounds__(FNT, 1) fvp_tangent_x3_kernel(FvpX3Args p) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
    const uint32_t sbase = smem_u32(smem_raw) + pad;
    uint8_t* gbase = smem_raw + pad;
    float* sB1 = reinterpret_cast<float*>(gbase + FO_MISC);
    float* sBv1 = sB1 + 64;
    float* sB2 = sBv1 + 64;
    float* sBv2 = sB2 + 64;
    float* sBv3 = sBv2 + 64;       // [16]
    long long* sRow = reinterpret_cast<long long*>(gbase + FO_ROWS);
    const uint32_t bar = sbase + FO_BAR;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gbase + FO_SLOT);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int O = p.O, A = p.A;
    const NetLayout L = actor_layout(O, A);
    // ---- weights and direction -> bf16x3 tiles ---------------------------------------------------------------------
    stage_matrix_x3(sbase + FO_W1, F_WSUB, p.theta + L.off_w1, 64, 64, O, O, tid);
    stage_matrix_x3(sbase + FO_V1, F_WSUB, p.vec + L.off_w1, 64, 64, O, O, tid);
    stage_matrix_x3(sbase + FO_W2, F_WSUB, p.theta + L.off_w2, 64, 64, 64, 64, tid);
    stage_matrix_x3(sbase + FO_V2, F_WSUB, p.vec + L.off_w2, 64, 64, 64, 64, tid);
    stage_matrix_x3(sbase + FO_W3, F_W3SUB, p.theta + L.off_w3, A, 16, 64, 64, tid);
    stage_matrix_x3(sbase + FO_V3, F_W3SUB, p.vec + L.off_w3, A, 16, 64, 64, tid);
    if (tid < 64) {
        sB1[tid] = __ldg(p.theta + L.off_b1 + tid); sBv1[tid] = __ldg(p.vec + L.off_b1 + tid);
        sB2[tid] = __ldg(p.theta + L.off_b2 + tid); sBv2[tid] = __ldg(p.vec + L.off_b2 + tid);
    }
    if (tid < 16) sBv3[tid] = (tid < A) ? __ldg(p.vec + L.off_b3 + tid) : 0.f;
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(1u) : "memory");
        mbar_init_fence();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 256);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    constexpr uint32_t C_Z = 0, C_T = 64, C_OUT = 128;
    uint32_t phase = 0;
    const bool leader = (warp == 0) && elect_one_sync();
    const uint64_t dA0 = desc128(sbase + FO_A0), dA1 = desc128(sbase + FO_A1);
    const uint64_t dW1 = desc128(sbase + FO_W1), dV1 = desc128(sbase + FO_V1), dW2 = desc128(sbase + FO_W2), dV2 = desc128(sbase + FO_V2);
    const uint64_t dW3 = desc128(sbase + FO_W3), dV3 = desc128(sbase + FO_V3);
    const uint32_t id_fwd = idesc_bf16(128, 64, 0, 0), id_out = idesc_bf16(128, 16, 0, 0);

    const long long nrows = (p.total + p.stride - 1) / p.stride;
    const long long ntiles = (nrows + FT - 1) / FT;
    const int xm = tid >> 1, xh = (tid & 1) << 5;          // X gather: row, 32-column half
    const bool vec4 = (O & 3) == 0;
    const int s_row = 32 * q + lane;

    // the rows of a tile are gathered into registers one tile ahead (under the layer-2 / layer-3 phases of the previous tile)
    float xpre[32];
    long long row_pre = -1;
    auto gather = [&](long long tile) {
        const long long k = tile * FT + xm;
        row_pre = (tile < ntiles && k < nrows) ? k * p.stride : -1;
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
            const int c0 = xh + 8 * c8;
            if (vec4) {
#pragma unroll
                for (int v4 = 0; v4 < 2; ++v4) {
                    const int c = c0 + 4 * v4;
                    const float4 x = (row_pre >= 0 && c < O) ? __ldg(reinterpret_cast<const float4*>(p.obs + row_pre * O + c))
                                                             : make_float4(0.f, 0.f, 0.f, 0.f);
                    xpre[8 * c8 + 4 * v4] = x.x; xpre[8 * c8 + 4 * v4 + 1] = x.y; xpre[8 * c8 + 4 * v4 + 2] = x.z; xpre[8 * c8 + 4 * v4 + 3] = x.w;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) xpre[8 * c8 + i] = (row_pre >= 0 && c0 + i < O) ? __ldg(p.obs + row_pre * O + c0 + i) : 0.f;
            }
        }
    };
    gather(blockIdx.x);
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        {   // X tile (the previous tile's MMAs have completed: both buffers are free)
            if ((tid & 1) == 0) sRow[xm] = row_pre;
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = xpre[8 * c8 + i];
                store8_x3(sbase + FO_A0, F_SUB, xm, xh + 8 * c8, v);
            }
        }
        fence_async_smem();
        __syncthreads();
        // ---- layer 1: Z1 = X W1^T, T1 = X V1^T ------------------------------------------------------------------------
        if (warp == 0) {
            tc_fence_after();
            gemm_x3_warp(leader, tmem + C_Z, dA0, F_SUB, 32u, dW1, F_WSUB, 32u, id_fwd, 4, false);
            gemm_x3_warp(leader, tmem + C_T, dA0, F_SUB, 32u, dV1, F_WSUB, 32u, id_fwd, 4, false);
            if (leader) mma_commit_a(bar);
            __syncwarp();
        }
        mbar_wait_a(bar, phase); phase ^= 1;
        tc_fence_after();
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {                    // H1 over X, dH1 into the tangent buffer
            const int c0 = 32 * h + 8 * c8;
            float z[8], t[8];
            tmem_ld8(tmem + lane_base + C_Z + (uint32_t)c0, z);
            tmem_ld8(tmem + lane_base + C_T + (uint32_t)c0, t);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float hh = tanh_acc(z[i] + sB1[c0 + i]);
                z[i] = hh;
                t[i] = (1.f - hh * hh) * (t[i] + sBv1[c0 + i]);
            }
            store8_x3(sbase + FO_A0, F_SUB, s_row, c0, z);
            store8_x3(sbase + FO_A1, F_SUB, s_row, c0, t);
        }
        fence_async_smem(); tc_fence_before();
        __syncthreads();
        // ---- layer 2: Z2 = H1 W2^T, T2 = dH1 W2^T + H1 V2^T -------------------------------------------------------------
        if (warp == 0) {
            tc_fence_after();
            gemm_x3_warp(leader, tmem + C_Z, dA0, F_SUB, 32u, dW2, F_WSUB, 32u, id_fwd, 4, false);
            gemm_x3_warp(leader, tmem + C_T, dA1, F_SUB, 32u, dW2, F_WSUB, 32u, id_fwd, 4, false);
            gemm_x3_warp(leader, tmem + C_T, dA0, F_SUB, 32u, dV2, F_WSUB, 32u, id_fwd, 4, true);
            if (leader) mma_commit_a(bar);
            __syncwarp();
        }
        gather(tile + gridDim.x);                            // next tile's rows fly under layers 2 and 3
        mbar_wait_a(bar, phase); phase ^= 1;
        tc_fence_after();
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {                    // H2 over H1, dH2 over dH1
            const int c0 = 32 * h + 8 * c8;
            float z[8], t[8];
            tmem_ld8(tmem + lane_base + C_Z + (uint32_t)c0, z);
            tmem_ld8(tmem + lane_base + C_T + (uint32_t)c0, t);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float hh = tanh_acc(z[i] + sB2[c0 + i]);
                z[i] = hh;
                t[i] = (1.f - hh * hh) * (t[i] + sBv2[c0 + i]);
            }
            store8_x3(sbase + FO_A0, F_SUB, s_row, c0, z);
            store8_x3(sbase + FO_A1, F_SUB, s_row, c0, t);
        }
        fence_async_smem(); tc_fence_before();
        __syncthreads();
        // ---- layer 3: dmu = dH2 W3^T + H2 V3^T + bv3 ---------------------------------------------------------------------
        if (warp == 0) {
            tc_fence_after();
            gemm_x3_warp(leader, tmem + C_OUT, dA1, F_SUB, 32u, dW3, F_W3SUB, 32u, id_out, 4, false);
            gemm_x3_warp(leader, tmem + C_OUT, dA0, F_SUB, 32u, dV3, F_W3SUB, 32u, id_out, 4, true);
            if (leader) mma_commit_a(bar);
            __syncwarp();
        }
        const long long row = (h == 0) ? sRow[s_row] : -1;
        mbar_wait_a(bar, phase); phase ^= 1;
        tc_fence_after();
        if (h == 0) {
            float o16[16];
            tmem_ld16(tmem + lane_base + C_OUT, o16);
            if (row >= 0)
                for (int a = 0; a < A; ++a) p.dmu[row * A + a] = o16[a] + sBv3[a];
        }
        tc_fence_before();
        __syncthreads();          // the layer-3 MMAs (readers of both buffers) completed; every thread is done with sRow
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

}  // namespace osb

using namespace osb;

extern "C" {

int osb_x3_fvp_backward(const float* theta_actor, const float* vec, int O, int A, const float* obs, long long total, int stride,
                        const float* dmu, float* gpart, float* stats_scratch, void* stream);

// Split-bf16 Fisher-vector product partials (O <= 64): tangent forward (dmu scratch [total][A]) then the actor backward
// of minibatch_grad_x3_kernel with dOUT = dmu / sigma^2 / (rows * A).  gpart: osb_tc_grid_blocks(rows, 1) rows of
// P_actor floats; stats_scratch: that many * 24 floats.  Reduce with osb_reduce_partials.  NaturalPG._fvp,
// natural_pg.py:L74-119.
int osb_fvp_partials_x3(const float* theta_actor, const float* vec, int O, int A, const float* obs, long long total,
                        int stride, float* dmu, float* gpart, float* stats_scratch, void* stream) {
    OSB_CHECK_ARG(theta_actor && vec && obs && dmu && gpart && stats_scratch && total > 0 && stride > 0, "bad argument");
    OSB_CHECK_ARG(O > 0 && O <= 64 && A > 0 && A <= 16, "bf16x3 path needs O <= 64, A <= 16");
    const long long nrows = (total + stride - 1) / stride;
    OSB_CHECK_ARG(nrows < (1ll << 31), "too many rows");
    FvpX3Args t{obs, total, stride, theta_actor, vec, dmu, O, A};
    const size_t smem = 1024 + F_SMEM;
    static bool attr = false;
    if (!attr) {
        OSB_CUDA(cudaFuncSetAttribute(fvp_tangent_x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = true;
    }
    const long long tiles = (nrows + FT - 1) / FT;
    static int n_sm = 0;
    if (!n_sm) { int dev = 0; OSB_CUDA(cudaGetDevice(&dev)); OSB_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev)); }
    const int blocks = (int)(tiles < n_sm ? tiles : n_sm);
    fvp_tangent_x3_kernel<<<blocks, FNT, smem, (cudaStream_t)stream>>>(t);
    OSB_LAUNCH_CHECK();
    return osb_x3_fvp_backward(theta_actor, vec, O, A, obs, total, stride, dmu, gpart, stats_scratch, stream);
}

}  // extern "C"
