// Tensor-core (tcgen05, TF32) full-batch actor forward: the fast variant of actor_eval_kernel
// (csrc/update.cu).  Stores mu(theta) per row (old-policy snapshot) or reduces
// sum KL(old||new), sum ratio*adv, sum ratio*adv_c, sum ratio, count, sum ratio*adv_r in fp64.
// Two CTAs per SM (~100 KB smem, 128 TMEM columns each) so one CTA's epilogue overlaps the other's MMA.
#include "common.cuh"
#include "mlp.cuh"
#include "umma.cuh"

namespace osb {

using namespace umma;

constexpr int ET = 128;
constexpr uint32_t EBUF = ET * 64 * 4;

struct EvalTcArgs {
    const float* obs; const float* act; const float* logp; const float* adv_r; const float* adv_c;
    const float* mu_old; const float* logstd_old; const float* moments; const float* lagrange;
    const float* theta; float* mu_store; double* part;
    long long total; int stride, O, A;
};

__global__ void __launch_bounds__(NTHREADS, 2) actor_eval_tc_kernel(EvalTcArgs p) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
    const uint32_t B0 = smem_u32(smem_raw) + pad;   // X -> H2
    const uint32_t B2 = B0 + EBUF;                  // H1
    const uint32_t sW1 = B2 + EBUF, sW2 = sW1 + 16384, sW3 = sW2 + 16384;
    float* sB1 = reinterpret_cast<float*>(smem_raw + pad + 2 * EBUF + 2 * 16384 + 4096);
    float* sB2 = sB1 + 64;
    float* sB3 = sB2 + 64;      // [16]
    float* sLs = sB3 + 16;      // logstd_new[16], sigma_new[16], logstd_old[16], sigma_old[16]
    double* sRedD = reinterpret_cast<double*>(sLs + 64);       // [4][8]
    long long* sRow = reinterpret_cast<long long*>(sRedD + 32);  // [128]
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int O = p.O, A = p.A;
    const NetLayout L = actor_layout(O, A);
    const float* theta = p.theta;
    {
        float w1v[16], w2v[16], w3v[4];
        const int k = tid & 63;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int n = (tid >> 6) + 4 * j;
            w1v[j] = (k < O && O <= 64) ? __ldg(theta + L.off_w1 + n * O + k) : 0.f;
            w2v[j] = __ldg(theta + L.off_w2 + n * 64 + k);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int o = (tid >> 6) + 4 * j;
            w3v[j] = (o < A) ? __ldg(theta + L.off_w3 + o * 64 + k) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int n = (tid >> 6) + 4 * j;
            sts(tile_addr(sW1, n, k, 64), tf32r(w1v[j]));
            sts(tile_addr(sW2, n, k, 64), tf32r(w2v[j]));
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) sts(tile_addr(sW3, (tid >> 6) + 4 * j, k, 16), tf32r(w3v[j]));
    }
    if (tid < 64) { sB1[tid] = __ldg(theta + L.off_b1 + tid); sB2[tid] = __ldg(theta + L.off_b2 + tid); }
    if (tid < 16) {
        sB3[tid] = (tid < A) ? __ldg(theta + L.off_b3 + tid) : 0.f;
        const float ls = (tid < A) ? __ldg(theta + L.off_logstd + tid) : 0.f;
        const float lo = (tid < A && p.logstd_old) ? __ldg(p.logstd_old + tid) : 0.f;
        sLs[tid] = ls; sLs[16 + tid] = expf(ls); sLs[32 + tid] = lo; sLs[48 + tid] = expf(lo);
    }
    if (tid == 0) { mbar_init(&bar, 1); mbar_init_fence(); }
    if (warp == 0) tmem_alloc(&tmem_slot, 128);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    constexpr uint32_t C_Z = 0, C_OUT = 64;
    uint32_t phase = 0;

    const int nchunks = (O + 63) >> 6;
    const long long nrows = (p.total + p.stride - 1) / p.stride;
    const long long ntiles = (nrows + ET - 1) / ET;
    const float lam = p.lagrange ? __ldg(p.lagrange) : 0.f;
    float m_r = 0.f, s_r = 1.f, m_c = 0.f;
    if (p.moments) { m_r = __ldg(p.moments); s_r = __ldg(p.moments + 1); m_c = __ldg(p.moments + 2); }
    double acc[6] = {0, 0, 0, 0, 0, 0};

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        if (tid < ET) {
            const long long k = tile * ET + tid;
            sRow[tid] = (k < nrows) ? k * p.stride : -1;
        }
        __syncthreads();
        for (int c = 0; c < nchunks; ++c) {     // layer 1 as a K loop over 64-column chunks of X / W1 (one chunk if O <= 64)
            const int k = tid & 63, col = c * 64 + k;
            if (nchunks > 1) {
                float w1c[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) w1c[j] = (col < O) ? __ldg(theta + L.off_w1 + ((tid >> 6) + 4 * j) * O + col) : 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) sts(tile_addr(sW1, (tid >> 6) + 4 * j, k, 64), tf32r(w1c[j]));
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                float xv[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const long long row = sRow[(tid >> 6) + 4 * (16 * half + j)];
                    xv[j] = (row >= 0 && col < O) ? __ldg(p.obs + row * O + col) : 0.f;
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) sts(tile_addr(B0, (tid >> 6) + 4 * (16 * half + j), k, ET), tf32r(xv[j]));
            }
            fence_async_smem();
            __syncthreads();
            if (tid == 0) { tc_fence_after(); tc_gemm(tmem + C_Z, B0, ET, sW1, 64, 128, 64, 64, c > 0); mma_commit(&bar); }
            mbar_wait(&bar, phase); phase ^= 1;
            tc_fence_after();
        }
        {
            float v[32];
            tmem_ld32(tmem + lane_base + C_Z + 32 * h, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = tanh_fast(v[i] + sB1[32 * h + i]);
            store_row32(B2, 32 * q + lane, 32 * h, ET, v);
        }
        fence_async_smem(); tc_fence_before();
        __syncthreads();
        if (tid == 0) { tc_fence_after(); tc_gemm(tmem + C_Z, B2, ET, sW2, 64, 128, 64, 64, false); mma_commit(&bar); }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        {
            float v[32];
            tmem_ld32(tmem + lane_base + C_Z + 32 * h, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = tanh_fast(v[i] + sB2[32 * h + i]);
            store_row32(B0, 32 * q + lane, 32 * h, ET, v);
        }
        fence_async_smem(); tc_fence_before();
        __syncthreads();
        if (tid == 0) { tc_fence_after(); tc_gemm(tmem + C_OUT, B0, ET, sW3, 16, 128, 16, 64, false); mma_commit(&bar); }
        // prefetch per-sample scalars while the MMA runs
        const long long row = (h == 0) ? sRow[32 * q + lane] : -1;
        float pa[16], pm[16], plogp = 0.f, padvr = 0.f, padvc = 0.f;
#pragma unroll
        for (int a = 0; a < 16; ++a) { pa[a] = 0.f; pm[a] = 0.f; }
        if (row >= 0 && !p.mu_store) {
#pragma unroll
            for (int a = 0; a < 16; ++a)
                if (a < A) { pa[a] = __ldg(p.act + row * A + a); pm[a] = __ldg(p.mu_old + row * A + a); }
            plogp = __ldg(p.logp + row); padvr = __ldg(p.adv_r + row); padvc = __ldg(p.adv_c + row);
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        if (h == 0) {
            float o16[16];
            tmem_ld16(tmem + lane_base + C_OUT, o16);
            if (row >= 0) {
                if (p.mu_store) {
                    for (int a = 0; a < A; ++a) p.mu_store[row * A + a] = o16[a] + sB3[a];
                } else {
                    float logp_new = 0.f, kl = 0.f;
#pragma unroll
                    for (int a = 0; a < 16; ++a)
                        if (a < A) {
                            const float mu = o16[a] + sB3[a], sd = sLs[16 + a], so = sLs[48 + a];
                            const float d = pa[a] - mu;
                            logp_new += -(d * d) / (2.f * sd * sd) - sLs[a] - 0.9189385332046727f;
                            const float vr = (so / sd) * (so / sd);
                            const float t1 = (pm[a] - mu) / sd;
                            kl += 0.5f * (vr + t1 * t1 - 1.f - logf(vr));
                        }
                    const float ratio = expf(logp_new - plogp);
                    const float adv_r = (padvr - m_r) / s_r, adv_c = padvc - m_c;
                    const float adv = (adv_r - lam * adv_c) / (1.f + lam);
                    acc[0] += (double)kl; acc[1] += (double)(ratio * adv); acc[2] += (double)(ratio * adv_c);
                    acc[3] += (double)ratio; acc[4] += 1.0; acc[5] += (double)(ratio * adv_r);
                }
            }
        }
        tc_fence_before();
        __syncthreads();
    }
    if (!p.mu_store) {
#pragma unroll
        for (int i = 0; i < 6; ++i) acc[i] = warp_sum(acc[i]);
        if (h == 0 && lane == 0)
            for (int i = 0; i < 6; ++i) sRedD[q * 8 + i] = acc[i];
        __syncthreads();
        if (tid < 6) p.part[(size_t)blockIdx.x * 8 + tid] = sRedD[tid] + sRedD[8 + tid] + sRedD[16 + tid] + sRedD[24 + tid];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

}  // namespace osb

using namespace osb;

extern "C" {

__global__ void eval_tc_reduce_kernel(const double* __restrict__ part, int nblocks, double* __restrict__ out) {
    // 32 groups x 8 statistics: group g sums CTAs g, g+32, ... ; the 32 group sums fold in a fixed order
    __shared__ double sh[32][8];
    const int q = threadIdx.x & 7, g = threadIdx.x >> 3;
    double s = 0.0;
    for (int b = g; b < nblocks; b += 32) s += part[(size_t)b * 8 + q];
    sh[g][q] = s;
    __syncthreads();
    if (threadIdx.x < 8) {
        double t = 0.0;
        for (int i = 0; i < 32; ++i) t += sh[i][threadIdx.x];
        out[threadIdx.x] = (threadIdx.x < 6) ? t : 0.0;
    }
}

// Tensor-core variant of osb_actor_eval (O <= 512; layer 1 K-chunked above 64); same arguments and outputs.
int osb_actor_eval_tc(const float* theta_actor, int O, int A, const float* obs, const float* act,
                      const float* logp, const float* adv_r, const float* adv_c, const float* mu_old,
                      const float* logstd_old, const float* moments, const float* lagrange,
                      long long total, int stride, float* mu_store, double* workspace, double* out,
                      void* stream) {
    OSB_CHECK_ARG(theta_actor && obs && total > 0 && stride > 0 && O > 0 && O <= 512 && A > 0 && A <= 16, "bad argument (O <= 512)");
    OSB_CHECK_ARG(mu_store || (act && logp && adv_r && adv_c && mu_old && logstd_old && workspace && out), "null input");
    EvalTcArgs p{obs, act, logp, adv_r, adv_c, mu_old, logstd_old, moments, lagrange, theta_actor, mu_store, workspace, total, stride, O, A};
    const size_t smem = 1024 + 2 * (size_t)EBUF + 2 * 16384 + 4096 + (64 + 64 + 16 + 64) * 4 + 32 * 8 + 128 * 8 + 64;
    static bool attr = false;
    if (!attr) {
        OSB_CUDA(cudaFuncSetAttribute(actor_eval_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = true;
    }
    const long long nrows = (total + stride - 1) / stride;
    const long long tiles = (nrows + ET - 1) / ET;
    const int blocks = (int)(tiles < 296 ? tiles : 296);
    cudaStream_t s = (cudaStream_t)stream;
    actor_eval_tc_kernel<<<blocks, NTHREADS, smem, s>>>(p);
    OSB_LAUNCH_CHECK();
    if (!mu_store) {
        eval_tc_reduce_kernel<<<1, 256, 0, s>>>(workspace, blocks, out);
        OSB_LAUNCH_CHECK();
    }
    return OSB_OK;
}

}  // extern "C"
