// Fused rollout step: HBM-resident synthetic Box envs + ObsNormalize + ActionScale + actor /
// reward-critic / cost-critic forwards + Gaussian sample / log-prob + slab append + episode stats.
//
// One launch per environment step replaces, per step, the reference's
//   ConstraintActorCritic.step        models/actor_critic/constraint_actor_critic.py:L84-109
//   ActionScale.step / ObsNormalize.step   envs/wrapper.py:L510-514, L231-241
//   Normalizer.normalize/_push        common/normalizer.py:L88-139
//   VectorOnPolicyBuffer.store        common/buffer/vector_onpolicy_buffer.py:L96-99
//   the per-env done loop             adapter/onpolicy_adapter.py:L114-136 (+ _log_value L155-157)
//
// Grid = (ceil(N/32) env tiles) x (3 networks).  Actor CTAs sample the action, run the env
// transition, append the step to the time-major slabs and feed the running-normaliser sums; critic
// CTAs write V_r / V_c and the bootstrap values of paths cut in the previous step.  The grid-wide
// ObsNormalize reduction is done with order-independent fixed-point atomics and finalised by the
// last actor CTA of the launch; the next launch (= kernel boundary = grid sync) consumes it.
#include "common.cuh"
#include <stdlib.h>
#include "mlp.cuh"
#include "umma.cuh"
#include "x3.cuh"

namespace osb {

constexpr int RT = 32;                       // envs per tile
constexpr double FIX_SCALE = 68719476736.0;  // 2^36 fixed point for the normaliser sums

struct EnvSpec {
    int O, A;
    int max_episode_steps;
    uint32_t seed;
    uint32_t term_threshold;  // terminate iff hash < threshold (0 = never)
    uint32_t env_id_offset;   // global env id of local env 0 (rank * N)
    float cost_threshold;
    int obs_normalize;
};

struct EnvState {
    float* s_raw;        // [2][N][O] raw observation of the current state (by step parity:
                         //   launch t reads buffer t&1 and writes buffer (t+1)&1)
    float* final_raw;    // [2][N][O] raw final observation of envs that finished (by step parity)
    int* ep_step;        // [N]
    uint32_t* episode;   // [N]
    uint32_t* gstep;     // [N] total env steps taken (termination hash counter)
    float* ep_ret;       // [N] running episode return / cost / length (adapter bookkeeping)
    float* ep_cost;      // [N]
    int* ep_len;         // [N]
    const float* bias;   // [O]
};

// Saute / Simmer safety state (adapter/saute_adapter.py:L135-217, simmer_adapter.py:L97-131): the networks see
// [normalised obs | z]; z starts an epoch at `init`, z <- (z - cost / budget) / gamma after every step, the stored reward
// becomes `unsafe_reward` once z <= 0, z returns to 1 when the episode ends (final observations carry z = 1).
struct SauteSpec {
    float* safety;       // [2][N] by step parity (like s_raw), or null: plain OnPolicyAdapter
    float budget;        // per-step safety budget (saute_adapter.py:L62-68)
    float gamma;         // saute_gamma
    float unsafe_reward;
    float init;          // z at the epoch's reset: 1 (Saute) or the relative budget (Simmer)
};

// EarlyTerminatedAdapter.step (adapter/early_terminated_adapter.py:L56-98), per env: the accumulated cost (never cleared
// by ordinary episode ends) exceeding cost_limit terminates the episode: reward 0, terminated = 1, the env is reset and
// the accumulator cleared.
struct EarlySpec {
    float* cost_acc;     // [N] or null
    float cost_limit;
};

struct NormState {
    float* mean;    // [O] running mean            (Normalizer._mean)
    float* sumsq;   // [O] running sum of squares  (Normalizer._sumsq)
    float* std;     // [O] max(sqrt(sumsq/(count-1)), 1e-2)
    float* mean1;   // [O] stats after pushing only the final-observation rows
    float* std1;    // [O]
    long long* count;          // [2]: [0] running count, [1] count used for mean1/std1
    long long* acc_all;        // [2][O] fixed-point sum x, sum x^2 over all next-obs rows
    long long* acc_fin;        // [2][O] same over final-observation rows
    int* fin_count;            // [1]
    int* had_fin;              // [1] previous launch pushed final rows
    unsigned int* ticket;      // [1]
};

struct Slabs {
    float* obs;      // [T][N][O] normalised observation fed to the networks
    float* act;      // [T][N][A]
    float* logp;     // [T][N]
    float* rew;      // [T][N]
    float* cost;     // [T][N]
    float* val_r;    // [T][N]
    float* val_c;    // [T][N]
    float* boot_r;   // [T][N] bootstrap values at truncated / epoch-end path ends
    float* boot_c;   // [T][N]
    uint8_t* flags;  // [T][N]
    float* epfin;    // [3][T][N] (EpRet, EpCost, EpLen) written where an episode finished
};

// ---------------------------------------------------------------------------------------------
// env arithmetic (bit-identical to oracle/synthetic_env.py)
__device__ __forceinline__ float env_reset_value(const EnvSpec& e, uint32_t gid, uint32_t episode,
                                                 int j) {
    return u32_to_unit(hash4(e.seed, gid, episode, (uint32_t)j));
}
__device__ __forceinline__ float env_next_value(float s, float a, float b) {
    float v = __fadd_rn(__fadd_rn(__fmul_rn(0.95f, s), __fmul_rn(0.1f, a)), b);
    return fminf(fmaxf(v, -10.f), 10.f);
}

// Chan / Golub / LeVeque batched update as Normalizer._push writes it (normalizer.py:L102-120),
// fp32 state, batch moments derived from the fixed-point sums.
__device__ void norm_push(float& mean, float& sumsq, long long count_old, long long n,
                          long long sx_fix, long long sxx_fix) {
    const double sx = (double)sx_fix / FIX_SCALE, sxx = (double)sxx_fix / FIX_SCALE;
    const double mraw = sx / (double)n;
    double m2 = sxx - (double)n * mraw * mraw;
    if (m2 < 0.0) m2 = 0.0;
    const float mean_raw = (float)mraw, sumq_raw = (float)m2;
    const long long count = count_old + n;
    const float delta = __fadd_rn(mean_raw, -mean);
    mean = __fadd_rn(mean, __fdiv_rn(__fmul_rn(delta, (float)n), (float)count));
    const float d2 = __fmul_rn(delta, delta);
    const float corr = __fdiv_rn(__fmul_rn(__fmul_rn(d2, (float)count_old), (float)n), (float)count);
    sumsq = __fadd_rn(sumsq, __fadd_rn(sumq_raw, corr));
}
__device__ __forceinline__ float norm_std(float sumsq, long long count) {
    const float var = __fdiv_rn(sumsq, (float)(count - 1));
    return fmaxf(sqrtf(var), 1e-2f);
}

// Executed by the last-arriving actor CTA: fold the launch's sums into the running statistics.
__device__ void norm_finalize(const NormState& ns, int O, long long n_all) {
    __threadfence();
    const int nfin = *((volatile int*)ns.fin_count);
    long long count = __ldcg(ns.count);          // (.cg: in the persistent kernel another SM may have written these last step)
    for (int j = threadIdx.x; j < O; j += blockDim.x) {
        float mean = __ldcg(ns.mean + j), sumsq = __ldcg(ns.sumsq + j);
        long long c = count;
        if (nfin > 0) {
            norm_push(mean, sumsq, c, nfin, __ldcg(ns.acc_fin + j), __ldcg(ns.acc_fin + O + j));
            c += nfin;
            ns.mean1[j] = mean;
            ns.std1[j] = norm_std(sumsq, c);
        }
        norm_push(mean, sumsq, c, n_all, __ldcg(ns.acc_all + j), __ldcg(ns.acc_all + O + j));
        c += n_all;
        ns.mean[j] = mean;
        ns.sumsq[j] = sumsq;
        ns.std[j] = norm_std(sumsq, c);
        ns.acc_all[j] = 0; ns.acc_all[O + j] = 0;
        ns.acc_fin[j] = 0; ns.acc_fin[O + j] = 0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        ns.count[1] = count + nfin;
        ns.count[0] = count + nfin + n_all;
        *ns.had_fin = nfin > 0 ? 1 : 0;
        *ns.fin_count = 0;
        *ns.ticket = 0u;
    }
}

// x * 2^36 rounded to the nearest integer.  The scaling by a power of two is exact in fp32 as well (|x| <= 10 by the env
// spec), so one fp32 -> int64 conversion gives the same integer as the fp64 product did.
__device__ __forceinline__ long long to_fix(float x) { return __float2ll_rn(x * 68719476736.0f); }

// ---------------------------------------------------------------------------------------------
// reset of all envs (OnPolicyAdapter.rollout resets every epoch: onpolicy_adapter.py:L80) and the
// normaliser push of the reset observations (ObsNormalize.reset, wrapper.py:L243-261).
__global__ void __launch_bounds__(NTHREADS) env_reset_kernel(EnvSpec es, EnvState st, NormState ns, SauteSpec sa,
                                                             int N) {
    __shared__ float sNew[RT][KC + 1];
    __shared__ int s_last;
    const int env0 = blockIdx.x * RT;
    const int O = es.O;
    const int e = threadIdx.x >> 3, q = threadIdx.x & 7;
    const int env = env0 + e;
    const bool ok = env < N;
    uint32_t epi = 0;
    if (ok) epi = st.episode[env] + 1u;
    for (int c0 = 0; c0 < O; c0 += KC) {
        for (int j = c0 + q; j < min(O, c0 + KC); j += 8) {
            float v = 0.f;
            if (ok) {
                v = env_reset_value(es, es.env_id_offset + env, epi, j);
                st.s_raw[(size_t)env * O + j] = v;  // buffer 0: step 0 reads parity 0
            }
            sNew[e][j - c0] = v;
        }
        __syncthreads();
        if (es.obs_normalize) {
            const int j = c0 + threadIdx.x;
            if (threadIdx.x < KC && j < O) {
                long long sx = 0, sxx = 0;
                for (int r = 0; r < RT; ++r)
                    if (env0 + r < N) {
                        const float v = sNew[r][threadIdx.x];
                        sx += to_fix(v);
                        sxx += to_fix(__fmul_rn(v, v));
                    }
                atomicAdd((unsigned long long*)(ns.acc_all + j), (unsigned long long)sx);
                atomicAdd((unsigned long long*)(ns.acc_all + O + j), (unsigned long long)sxx);
            }
        }
        __syncthreads();
    }
    if (ok && q == 0) {
        st.episode[env] = epi;
        st.ep_step[env] = 0;
        st.ep_ret[env] = 0.f;
        st.ep_cost[env] = 0.f;
        st.ep_len[env] = 0;
        if (sa.safety) sa.safety[env] = sa.init;   // buffer 0: step 0 reads parity 0
    }
    if (es.obs_normalize) {
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_last = (atomicAdd(ns.ticket, 1u) == gridDim.x - 1) ? 1 : 0;
        __syncthreads();
        if (s_last) norm_finalize(ns, O, (long long)N);
    }
}

// Philox4x32-10 (fast-mode noise); counter = (env gid, global step, lane block, 0).
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
}
__device__ float philox_normal(uint32_t seed, uint32_t gid, uint32_t step, int a) {
    uint32_t c[4] = {gid, step, (uint32_t)(a >> 2), 0x0B200u};
    uint32_t k0 = seed, k1 = 0xCAFEF00Du;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c, k0, k1);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    const int pair = (a & 3) >> 1;
    const float u0 = ((float)(c[2 * pair] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u1 = ((float)(c[2 * pair + 1] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float r = sqrtf(-2.0f * logf(u0));
    float sn, cs;
    sincosf(6.283185307179586f * u1, &sn, &cs);
    return (a & 1) ? r * sn : r * cs;
}

// both normals of action pair pr (actions 2 pr, 2 pr + 1): same values as philox_normal(seed, gid, step, 2 pr [+ 1])
__device__ void philox_normal2(uint32_t seed, uint32_t gid, uint32_t step, int pr, float& n0, float& n1) {
    uint32_t c[4] = {gid, step, (uint32_t)(pr >> 1), 0x0B200u};
    uint32_t k0 = seed, k1 = 0xCAFEF00Du;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c, k0, k1);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    const int pair = pr & 1;
    const float u0 = ((float)(c[2 * pair] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u1 = ((float)(c[2 * pair + 1] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float r = sqrtf(-2.0f * logf(u0));
    float sn, cs;
    sincosf(6.283185307179586f * u1, &sn, &cs);
    n0 = r * cs; n1 = r * sn;
}

struct StepArgs {
    EnvSpec es;
    EnvState st;
    NormState ns;
    Slabs sl;
    SauteSpec sa;
    EarlySpec et;
    const float* theta;   // flat [actor | critic_r | critic_c]
    const float* eps;     // [N][A] noise of this step (parity mode) or null (Philox fast mode)
    uint32_t noise_seed;
    uint32_t global_step; // epoch * T + t, Philox counter
    int t, T, N;
    int is_tail;          // t == T: critics only (epoch-end bootstrap)
    int precision;        // 0 = fp32 FMA tiles of 32 envs, 1 = tcgen05 TF32 tiles of 128 envs, 2 = split-bf16 tcgen05 tiles (O <= 64)
    unsigned int* bar_ctr;    // persistent epoch kernel: grid-barrier arrival counter and release flag (zero at launch)
    unsigned int* bar_flag;
    long long* dbg;           // optional clock64 stamps (persistent kernel), normally null
};

// normalise (or copy) a tile of raw observations into sX (chunk kc), zero padded.
// z = per-env safety state (Saute) appended as column O of the network input (rows are On = O + 1 wide then), or null;
// z_one: the final observations of finished episodes carry z = 1 (the state was reset before the augmentation).
__device__ __forceinline__ void load_obs_tile(const float* __restrict__ raw, int env0, int N, int O,
                                              int kc, const float* sMean, const float* sStd,
                                              bool normalize, float* sX, float* obs_out,
                                              const float* z = nullptr, bool z_one = false) {
    const int c0 = kc * KC;
    const int On = O + (z ? 1 : 0);
    for (int i = threadIdx.x; i < RT * KC; i += NTHREADS) {
        const int e = i / KC, k = i % KC;
        const int env = env0 + e, j = c0 + k;
        float v = 0.f;
        if (env < N && j < O) {
            v = raw[(size_t)env * O + j];
            if (normalize) {
                v = __fdiv_rn(__fadd_rn(v, -sMean[j]), sStd[j]);
                v = fminf(fmaxf(v, -5.f), 5.f);
            }
            if (obs_out) obs_out[(size_t)env * On + j] = v;
        } else if (env < N && j == O && z) {
            v = z_one ? 1.f : __ldcg(z + env);
            if (obs_out) obs_out[(size_t)env * On + j] = v;
        }
        sX[e * LD + k] = v;
    }
}

// cost of this step (indicator on the next value of state dim 0) from the current raw state and the sampled action
__device__ __forceinline__ float env_step_cost(const EnvSpec& es, float s0, float act0, float bias0) {
    float a = __fadd_rn(__fadd_rn(act0, 1.f), -1.f);
    a = fminf(fmaxf(a, -1.f), 1.f);
    return (env_next_value(s0, a, bias0) > es.cost_threshold) ? 1.f : 0.f;
}

// SauteAdapter.step (saute_adapter.py:L172-217) for one env: z <- (z - cost / budget) / gamma, reward override once
// z <= 0, z <- 1 when the episode ends.  Returns the reward to store (episode returns keep the original one).
__device__ __forceinline__ float saute_step(const SauteSpec& sa, int t, int N, int env, float rew, float cost, bool fin) {
    if (!sa.safety) return rew;
    float z = __ldcg(sa.safety + (size_t)(t & 1) * N + env);
    z = __fdiv_rn(__fadd_rn(z, -__fdiv_rn(cost, sa.budget)), sa.gamma);
    const float out = (z > 0.f) ? rew : sa.unsafe_reward;
    sa.safety[(size_t)((t + 1) & 1) * N + env] = fin ? 1.f : z;
    return out;
}

__global__ void __launch_bounds__(NTHREADS) rollout_step_kernel(StepArgs p) {
    extern __shared__ __align__(16) float smem[];
    NetSmem W;
    float* base = carve_net_smem<false>(smem, W);
    float* sX = base;  base += RT * LD;
    float* sH1 = base; base += RT * LD;
    float* sH2 = base; base += RT * LD;
    float* sO = base;  base += RT * LDO;
    float* sMean = base; base += p.es.O;
    float* sStd = base;  base += p.es.O;
    float* sAct = base;  base += RT * OUTP;
    float* sNew = base;  base += RT * (KC + 1);
    float* sFin = base;  base += RT * (KC + 1);
    float* sRew = base;  base += RT;
    float* sCost = base; base += RT;
    int* sFlag = reinterpret_cast<int*>(base); base += RT;
    __shared__ int s_last, s_anyfin;

    const int net = p.is_tail ? (int)blockIdx.y + 1 : (int)blockIdx.y;
    const int env0 = blockIdx.x * RT;
    const int O = p.es.O, A = p.es.A, N = p.N, T = p.T, t = p.t;
    const int On = O + (p.sa.safety ? 1 : 0);            // network input width (Saute: [obs | z])
    const float* z_cur = p.sa.safety ? p.sa.safety + (size_t)(t & 1) * N : nullptr;
    const int nchunks = (On + KC - 1) / KC;
    const NetLayout L = net_layout(net, On, A);
    const float* theta = p.theta + net_offset(net, On, A);
    const bool normalize = p.es.obs_normalize && p.ns.count[0] > 1;
    const float* s_cur = p.st.s_raw + (size_t)(t & 1) * N * O;
    float* s_nxt = p.st.s_raw + (size_t)((t + 1) & 1) * N * O;

    load_net_rest<false>(theta, L, W);
    load_w1_chunk(theta, L, 0, W);
    auto load_chunk_cur = [&](int kc) {
        load_w1_chunk(theta, L, kc, W);
        for (int j = threadIdx.x; j < O; j += NTHREADS) { sMean[j] = p.ns.mean[j]; sStd[j] = p.ns.std[j]; }
        load_obs_tile(s_cur, env0, N, O, kc, sMean, sStd, normalize, sX, nullptr, z_cur);
    };

    // ---- bootstrap values of paths that ended in the previous step (critic CTAs only) --------
    if (net != 0 && t > 0) {
        if (threadIdx.x == 0) s_anyfin = 0;
        __syncthreads();
        if (threadIdx.x < RT && env0 + threadIdx.x < N) {
            const unsigned f = p.sl.flags[(size_t)(t - 1) * N + env0 + threadIdx.x];
            if ((f & OSB_FLAG_TRUNCATED) && !(f & OSB_FLAG_TERMINATED)) s_anyfin = 1;
        }
        __syncthreads();
        if (s_anyfin) {
            const bool norm1 = p.es.obs_normalize && p.ns.count[1] > 1;
            const float* fin = p.st.final_raw + (size_t)((t - 1) & 1) * N * O;
            auto load_chunk_fin = [&](int kc) {
                load_w1_chunk(theta, L, kc, W);
                for (int j = threadIdx.x; j < O; j += NTHREADS) { sMean[j] = p.ns.mean1[j]; sStd[j] = p.ns.std1[j]; }
                load_obs_tile(fin, env0, N, O, kc, sMean, sStd, norm1, sX, nullptr, z_cur, true);
            };
            for (int j = threadIdx.x; j < O; j += NTHREADS) { sMean[j] = p.ns.mean1[j]; sStd[j] = p.ns.std1[j]; }
            __syncthreads();
            load_obs_tile(fin, env0, N, O, 0, sMean, sStd, norm1, sX, nullptr, z_cur, true);
            __syncthreads();
            mlp_hidden<RT>(sX, sH1, sH2, W, nchunks, load_chunk_fin);
            mlp_out<RT>(sH2, sO, W, 1);
            if (threadIdx.x < RT && env0 + threadIdx.x < N) {
                const size_t idx = (size_t)(t - 1) * N + env0 + threadIdx.x;
                const unsigned f = p.sl.flags[idx];
                if ((f & OSB_FLAG_TRUNCATED) && !(f & OSB_FLAG_TERMINATED))
                    (net == 1 ? p.sl.boot_r : p.sl.boot_c)[idx] = sO[threadIdx.x * LDO];
            }
            __syncthreads();
            if (nchunks > 1) { load_w1_chunk(theta, L, 0, W); }
        }
    }

    // ---- forward on the current observation ------------------------------------------------
    for (int j = threadIdx.x; j < O; j += NTHREADS) { sMean[j] = p.ns.mean[j]; sStd[j] = p.ns.std[j]; }
    __syncthreads();
    if (net == 0 && nchunks > 1) {
        // write the whole normalised observation row once (chunks > 0 are not revisited below)
        for (int kc = 1; kc < nchunks; ++kc)
            load_obs_tile(s_cur, env0, N, O, kc, sMean, sStd, normalize, sX,
                          p.sl.obs + (size_t)t * N * On, z_cur);
        __syncthreads();
    }
    load_obs_tile(s_cur, env0, N, O, 0, sMean, sStd, normalize, sX,
                  (net == 0) ? p.sl.obs + (size_t)t * N * On : nullptr, z_cur);
    __syncthreads();
    mlp_hidden<RT>(sX, sH1, sH2, W, nchunks, load_chunk_cur);
    mlp_out<RT>(sH2, sO, W, L.out);

    if (net != 0) {
        if (threadIdx.x < RT && env0 + threadIdx.x < N) {
            const float v = sO[threadIdx.x * LDO];
            if (!p.is_tail) {
                (net == 1 ? p.sl.val_r : p.sl.val_c)[(size_t)t * N + env0 + threadIdx.x] = v;
            } else {
                // epoch end: bootstrap with V(next obs) unless the path already ended at T-1
                const size_t idx = (size_t)(T - 1) * N + env0 + threadIdx.x;
                if (p.sl.flags[idx] == 0) (net == 1 ? p.sl.boot_r : p.sl.boot_c)[idx] = v;
            }
        }
    }

    // ---- actor CTA: sample, log-prob ---------------------------------------------------------
    if (net == 0) {
        // thread -> (env e = tid / 8, lane q = tid % 8); action components a = q, q + 8
        const int e = threadIdx.x >> 3, q = threadIdx.x & 7;
        const int env = env0 + e;
        const bool ok = env < N;
        float lp = 0.f;
        for (int a = q; a < A; a += 8) {
            const float mu = sO[e * LDO + a];
            const float sd = expf(__ldg(theta + L.off_logstd + a));
            float eps = 0.f;
            if (ok)
                eps = p.eps ? p.eps[(size_t)env * A + a]
                            : philox_normal(p.noise_seed, p.es.env_id_offset + env, p.global_step, a);
            const float act = __fadd_rn(mu, __fmul_rn(sd, eps));   // Normal.rsample: loc + eps*scale
            // Normal.log_prob: -((x-loc)^2)/(2 var) - log(scale) - log(sqrt(2 pi))
            const float d = __fadd_rn(act, -mu);
            const float var = __fmul_rn(sd, sd);
            float term = __fdiv_rn(-__fmul_rn(d, d), __fmul_rn(2.f, var));
            term = __fadd_rn(__fadd_rn(term, -logf(sd)), -0.9189385332046727f);
            lp += term;
            sAct[e * OUTP + a] = act;
            if (ok) p.sl.act[((size_t)t * N + env) * A + a] = act;
        }
        lp += __shfl_xor_sync(0xffffffffu, lp, 1);
        lp += __shfl_xor_sync(0xffffffffu, lp, 2);
        lp += __shfl_xor_sync(0xffffffffu, lp, 4);
        if (ok && q == 0) p.sl.logp[(size_t)t * N + env] = lp;
    }
    __syncthreads();

    // ---- env transition ----------------------------------------------------------------------
    if (net == 0) {
        const int e = threadIdx.x >> 3, q = threadIdx.x & 7;
        const int env = env0 + e;
        const bool ok = env < N;
        const uint32_t gid = p.es.env_id_offset + env;
        int ep_step = 0; uint32_t epi = 0, gstep = 0;
        if (ok) { ep_step = p.st.ep_step[env]; epi = p.st.episode[env]; gstep = p.st.gstep[env]; }
        const bool trunc = ok && (ep_step + 1 >= p.es.max_episode_steps);
        const bool term = ok && p.es.term_threshold != 0u &&
                          hash4(p.es.seed ^ 0xA5A5A5A5u, gid, gstep, 0xFFFFu) < p.es.term_threshold;
        const bool fin_env = term || trunc;               // the env's own episode end
        bool early = false;                               // EarlyTerminated: accumulated cost over the limit
        float acc_cost = 0.f;
        if (ok && p.et.cost_acc) {
            acc_cost = __fadd_rn(p.et.cost_acc[env], env_step_cost(p.es, s_cur[(size_t)env * O], sAct[e * OUTP], __ldg(p.st.bias)));
            early = acc_cost > p.et.cost_limit;
        }
        const bool fin = fin_env || early;
        const uint32_t epi_inc = (fin_env && early) ? 2u : 1u;   // the env's auto-reset and then the adapter's reset
        float part = 0.f, s0n = 0.f;
        float* finrow = p.st.final_raw + ((size_t)(t & 1) * N + (ok ? env : 0)) * O;
        for (int c0 = 0; c0 < O; c0 += KC) {
            for (int j = c0 + q; j < min(O, c0 + KC); j += 8) {
                float nv = 0.f, fv = 0.f;
                if (ok) {
                    // ActionScale (wrapper.py:L510-512) from [-1,1] onto the env's [-1,1] box
                    float a = sAct[e * OUTP + (j % A)];
                    a = __fadd_rn(__fadd_rn(a, 1.f), -1.f);
                    a = fminf(fmaxf(a, -1.f), 1.f);
                    const float s = s_cur[(size_t)env * O + j];
                    const float sn = env_next_value(s, a, __ldg(p.st.bias + j));
                    part = __fadd_rn(part, __fmul_rn(sn, sn));
                    if (j == 0) s0n = sn;
                    fv = sn;
                    nv = fin ? env_reset_value(p.es, gid, epi + epi_inc, j) : sn;
                    s_nxt[(size_t)env * O + j] = nv;
                    if (fin) finrow[j] = sn;
                }
                sNew[e * (KC + 1) + (j - c0)] = nv;
                sFin[e * (KC + 1) + (j - c0)] = fin ? fv : 0.f;
            }
            if (c0 == 0 && q == 0) sFlag[e] = fin ? 1 : 0;
            __syncthreads();
            if (p.es.obs_normalize) {
                const int j = c0 + threadIdx.x;
                if (threadIdx.x < KC && j < O) {
                    long long sx = 0, sxx = 0, fx = 0, fxx = 0;
                    for (int r = 0; r < RT; ++r)
                        if (env0 + r < N) {
                            const float v = sNew[r * (KC + 1) + threadIdx.x];
                            sx += to_fix(v); sxx += to_fix(__fmul_rn(v, v));
                            if (sFlag[r]) {
                                const float w = sFin[r * (KC + 1) + threadIdx.x];
                                fx += to_fix(w); fxx += to_fix(__fmul_rn(w, w));
                            }
                        }
                    atomicAdd((unsigned long long*)(p.ns.acc_all + j), (unsigned long long)sx);
                    atomicAdd((unsigned long long*)(p.ns.acc_all + O + j), (unsigned long long)sxx);
                    if (fx != 0 || fxx != 0) {
                        atomicAdd((unsigned long long*)(p.ns.acc_fin + j), (unsigned long long)fx);
                        atomicAdd((unsigned long long*)(p.ns.acc_fin + O + j), (unsigned long long)fxx);
                    }
                }
            }
            __syncthreads();
        }
        // reward = 1 - mean_j s'_j^2 with the fixed summation tree shared with the oracle
        part = __fadd_rn(part, __shfl_xor_sync(0xffffffffu, part, 1));
        part = __fadd_rn(part, __shfl_xor_sync(0xffffffffu, part, 2));
        part = __fadd_rn(part, __shfl_xor_sync(0xffffffffu, part, 4));
        if (ok && q == 0) {
            const float rew = early ? 0.f : __fadd_rn(1.f, -__fdiv_rn(part, (float)O));
            const float cst = (s0n > p.es.cost_threshold) ? 1.f : 0.f;
            const size_t idx = (size_t)t * N + env;
            p.sl.rew[idx] = saute_step(p.sa, t, N, env, rew, cst, fin);
            p.sl.cost[idx] = cst;
            p.sl.flags[idx] = (uint8_t)(((term || early) ? OSB_FLAG_TERMINATED : 0u) | (trunc ? OSB_FLAG_TRUNCATED : 0u));
            if (p.et.cost_acc) p.et.cost_acc[env] = early ? 0.f : acc_cost;
            // adapter bookkeeping: _log_value, _log_metrics, _reset_log (onpolicy_adapter.py:L138-175)
            const float er = __fadd_rn(p.st.ep_ret[env], rew);
            const float ec = __fadd_rn(p.st.ep_cost[env], cst);
            const int el = p.st.ep_len[env] + 1;
            if (fin) {
                const size_t TN = (size_t)T * N;
                p.sl.epfin[idx] = er;
                p.sl.epfin[TN + idx] = ec;
                p.sl.epfin[2 * TN + idx] = (float)el;
                p.st.ep_ret[env] = 0.f; p.st.ep_cost[env] = 0.f; p.st.ep_len[env] = 0;
                p.st.episode[env] = epi + epi_inc;
                p.st.ep_step[env] = 0;
            } else {
                p.st.ep_ret[env] = er; p.st.ep_cost[env] = ec; p.st.ep_len[env] = el;
                p.st.ep_step[env] = ep_step + 1;
            }
            p.st.gstep[env] = gstep + 1u;
        }
        if (p.es.obs_normalize && threadIdx.x == 0) {
            int nf = 0;
            for (int r = 0; r < RT; ++r) nf += (env0 + r < N) ? sFlag[r] : 0;
            if (nf) atomicAdd(p.ns.fin_count, nf);
        }
    }
    // every CTA (actor and critic) has now consumed the normaliser state of this step; the last
    // one to arrive folds the step's sums into it for the next launch.
    if (p.es.obs_normalize && !p.is_tail) {
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0)
            s_last = (atomicAdd(p.ns.ticket, 1u) == gridDim.x * gridDim.y - 1) ? 1 : 0;
        __syncthreads();
        if (s_last) norm_finalize(p.ns, O, (long long)N);
    }
}

// ---------------------------------------------------------------------------------------------
// Tensor-core variant of the step kernel (train_cfgs.matmul_precision = tf32, O <= 64): tiles of 128
// envs, the three layer GEMMs of a network as tcgen05.mma kind::tf32 with TMEM accumulators, operands
// staged as 128B-swizzled K-major smem tiles.  Everything around the GEMMs (ObsNormalize, sampling,
// env transition, slab append, normaliser sums, ticket) is the arithmetic of rollout_step_kernel.
constexpr int RTC = 128;
constexpr int SNW = KC + 1;   // row stride of the next-state staging tiles

// X3 = false: kind::tf32 tiles (5e-3);  X3 = true: split-bf16 tiles (csrc/x3.cuh), fp32-level values / log-probs:
// one bf16x3 activation buffer (X, H1, H2 overwrite each other in place), accurate tanh, warp-uniform MMA issue.
constexpr uint32_t RX_SUB = RTC * 128, RX_WSUB = 64 * 128, RX_W3SUB = 16 * 128;
constexpr uint32_t RTC_FOFF_TF32 = 2 * RTC * 256 + 2 * 16384 + 4096, RTC_FOFF_X3 = 3 * RX_SUB + 6 * RX_WSUB + 3 * RX_W3SUB;

// PERSIST = true: ONE cooperative launch runs the whole epoch (steps 0 .. T, the last one being the critics' epoch-end
// bootstrap): the weight tiles, biases and the TMEM allocation stay resident, every step ends in a grid barrier whose
// last arriver folds the step's normaliser sums into the running statistics before it releases the others
// (adapter/onpolicy_adapter.py:L58-136 is the loop this replaces).  Data written by other CTAs in earlier steps
// (raw states, flags, normaliser statistics) is read with ld.global.cg.
template <bool X3, bool PERSIST>
__global__ void __launch_bounds__(NTHREADS, 1) rollout_step_tc_kernel(StepArgs p) {
    using namespace umma;
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
    const uint32_t B0 = smem_u32(smem_raw) + pad;       // X -> H2   (X3: X -> H1 -> H2, bf16x3)
    const uint32_t B2 = B0 + RTC * 256;                 // H1        (X3: unused)
    const uint32_t sW1 = X3 ? B0 + 3 * RX_SUB : B2 + RTC * 256;
    const uint32_t sW2 = sW1 + (X3 ? 3 * RX_WSUB : 16384u), sW3 = sW2 + (X3 ? 3 * RX_WSUB : 16384u);
    float* fbase = reinterpret_cast<float*>(smem_raw + pad + (X3 ? RTC_FOFF_X3 : RTC_FOFF_TF32));
    float* sB1 = fbase;            // [64]
    float* sB2 = sB1 + 64;         // [64]
    float* sB3 = sB2 + 64;         // [16]
    float* sMean = sB3 + 16;       // [64]
    float* sRstd = sMean + 64;     // [64]  1 / std
    float* sAct = sRstd + 64;      // [128][16]
    float* sRaw = sAct + RTC * OUTP;           // [128][65] raw current state of the tile (actor CTAs; kept by the obs staging)
    float* sSn = sRaw + RTC * SNW;             // [128][65] state after the transition, before any reset
    long long* sAcc = reinterpret_cast<long long*>(sSn + RTC * SNW);    // [4][4][64] partial fixed-point sums
    int* sFlag = reinterpret_cast<int*>(sAcc + 4 * 4 * 64);             // [128] bit 0 finished, bit 1 terminated, bit 2 truncated
    uint32_t* sEpi = reinterpret_cast<uint32_t*>(sFlag + RTC);          // [128] episode counter
    int* sStep = reinterpret_cast<int*>(sEpi + RTC);                    // [128] step inside the episode
    uint32_t* sGstep = reinterpret_cast<uint32_t*>(sStep + RTC);        // [128] total steps of the env (termination hash counter)
    float* sSd = reinterpret_cast<float*>(sGstep + RTC);                // [3][16] sigma, 2 sigma^2, log sigma per action
    float* sEarlyAcc = sSd + 48;                                        // [128] accumulated cost incl. this step (EarlyTerminated)
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    __shared__ int s_last, s_anyfin;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;
    const int net = PERSIST ? (int)blockIdx.y : (p.is_tail ? (int)blockIdx.y + 1 : (int)blockIdx.y);
    const int env0 = blockIdx.x * RTC;
    const int O = p.es.O, A = p.es.A, N = p.N, T = p.T;
    const int On = O + (p.sa.safety ? 1 : 0);            // network input width (Saute: [obs | z]), <= 64 here
    const NetLayout L = net_layout(net, On, A);
    const float* theta = p.theta + net_offset(net, On, A);
    const int e_env = tid >> 1, e_half = tid & 1;       // actor CTAs: 2 threads per env in the transition
    const int my_env = env0 + e_env;
    const bool my_ok = (net == 0) && my_env < N;

    if constexpr (X3) {   // weights -> bf16x3 tiles (all loads first)
        float a1[8], b1[8], a2[8], b2[8], a3[2], b3[2];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int i = tid + j * NTHREADS, n = i >> 5, k = (i & 31) << 1;
            a1[j] = (k < On) ? __ldg(theta + L.off_w1 + n * On + k) : 0.f;
            b1[j] = (k + 1 < On) ? __ldg(theta + L.off_w1 + n * On + k + 1) : 0.f;
            a2[j] = __ldg(theta + L.off_w2 + n * 64 + k); b2[j] = __ldg(theta + L.off_w2 + n * 64 + k + 1);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int i = tid + j * NTHREADS, o = i >> 5, k = (i & 31) << 1;
            a3[j] = (o < L.out) ? __ldg(theta + L.off_w3 + o * 64 + k) : 0.f;
            b3[j] = (o < L.out) ? __ldg(theta + L.off_w3 + o * 64 + k + 1) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int i = tid + j * NTHREADS, n = i >> 5, k = (i & 31) << 1;
            uint32_t w0, w1, w2;
            const uint32_t off = x3::off128(n, k);
            x3::split2(a1[j], b1[j], w0, w1, w2);
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sW1 + off), "r"(w0) : "memory");
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sW1 + RX_WSUB + off), "r"(w1) : "memory");
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sW1 + 2 * RX_WSUB + off), "r"(w2) : "memory");
            x3::split2(a2[j], b2[j], w0, w1, w2);
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sW2 + off), "r"(w0) : "memory");
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sW2 + RX_WSUB + off), "r"(w1) : "memory");
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sW2 + 2 * RX_WSUB + off), "r"(w2) : "memory");
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int i = tid + j * NTHREADS, o = i >> 5, k = (i & 31) << 1;
            uint32_t w0, w1, w2;
            const uint32_t off = x3::off128(o, k);
            x3::split2(a3[j], b3[j], w0, w1, w2);
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sW3 + off), "r"(w0) : "memory");
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sW3 + RX_W3SUB + off), "r"(w1) : "memory");
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sW3 + 2 * RX_W3SUB + off), "r"(w2) : "memory");
        }
    } else
    {   // weights (batched loads)
        float w1v[16], w2v[16], w3v[4];
        const int k = tid & 63;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int n = (tid >> 6) + 4 * j;
            w1v[j] = (k < On) ? __ldg(theta + L.off_w1 + n * On + k) : 0.f;
            w2v[j] = __ldg(theta + L.off_w2 + n * 64 + k);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int o = (tid >> 6) + 4 * j;
            w3v[j] = (o < L.out) ? __ldg(theta + L.off_w3 + o * 64 + k) : 0.f;
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
    if (tid < 16) sB3[tid] = (tid < L.out) ? __ldg(theta + L.off_b3 + tid) : 0.f;
    if (net == 0 && tid < 16) {          // Normal(mu, sigma): sigma = exp(log_std) is state independent
        const float sd = (tid < A) ? expf(__ldg(theta + L.off_logstd + tid)) : 1.f;
        sSd[tid] = sd; sSd[16 + tid] = __fmul_rn(2.f, __fmul_rn(sd, sd)); sSd[32 + tid] = logf(sd);
    }
    if (tid == 0) { mbar_init(&bar, 1); mbar_init_fence(); s_anyfin = 0; }
    if (warp == 0) tmem_alloc(&tmem_slot, 128);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    constexpr uint32_t C_Z = 0, C_OUT = 64;
    uint32_t phase = 0;

    // development aid (tools/rollout_stage_times.py): clock64 stamps of thread 0 of the first actor and reward-critic CTA
    const bool dbg_on = PERSIST && p.dbg != nullptr && blockIdx.x == 0 && blockIdx.y < 2 && tid == 0;
    int dbg_n = 0;
#define RSTAMP(id) do { if (dbg_on && dbg_n < 250) { long long* d_ = p.dbg + (blockIdx.y ? 512 : 0); d_[1 + 2 * dbg_n] = (id); d_[2 + 2 * dbg_n] = clock64(); ++dbg_n; d_[0] = dbg_n; } } while (0)
    const int t_first = PERSIST ? 0 : p.t, t_last = PERSIST ? T : p.t;
#pragma unroll 1
    for (int t = t_first; t <= t_last; ++t) {
    const bool is_tail = t == T;
    if (PERSIST && is_tail && net == 0) break;          // the tail step is the critics' (no barrier follows it)
    const float* eps_t = PERSIST ? (p.eps ? p.eps + (size_t)t * N * A : nullptr) : p.eps;
    const uint32_t gstep_t = PERSIST ? p.global_step + (uint32_t)t : p.global_step;
    const bool normalize = p.es.obs_normalize && __ldcg(p.ns.count) > 1;
    const float* s_cur = p.st.s_raw + (size_t)(t & 1) * N * O;
    float* s_nxt = p.st.s_raw + (size_t)((t + 1) & 1) * N * O;
    if (PERSIST) { if (tid == 0) s_anyfin = 0; __syncthreads(); }
    // which envs of this tile finish in this step (time limit / hash-driven termination): known before the forward
    if (net == 0 && tid < RTC) {
        const int env = env0 + tid;
        int fl = 0, ep_step = 0; uint32_t epi = 0, gstep = 0;
        if (env < N) {
            ep_step = p.st.ep_step[env]; epi = p.st.episode[env]; gstep = p.st.gstep[env];
            const bool trunc = ep_step + 1 >= p.es.max_episode_steps;
            const bool term = p.es.term_threshold != 0u &&
                              hash4(p.es.seed ^ 0xA5A5A5A5u, p.es.env_id_offset + env, gstep, 0xFFFFu) < p.es.term_threshold;
            fl = ((term || trunc) ? 1 : 0) | (term ? 2 : 0) | (trunc ? 4 : 0);
        }
        sFlag[tid] = fl; sEpi[tid] = epi; sStep[tid] = ep_step; sGstep[tid] = gstep;
    }
    RSTAMP(1);

    // does this critic tile need bootstrap values for paths cut in the previous step?
    if (net != 0 && t > 0 && tid < RTC && env0 + tid < N) {
        const unsigned f = __ldcg(p.sl.flags + (size_t)(t - 1) * N + env0 + tid);
        if ((f & OSB_FLAG_TRUNCATED) && !(f & OSB_FLAG_TERMINATED)) s_anyfin = 1;
    }
    __syncthreads();
    const int first_pass = (net != 0 && t > 0 && s_anyfin) ? 0 : 1;

    // pass 0: final observations of the previous step (critics, rare); pass 1: current observation
#pragma unroll 1
    for (int pass = first_pass; pass < 2; ++pass) {
        const float* raw = pass ? s_cur : p.st.final_raw + (size_t)((t - 1) & 1) * N * O;
        const float* gmean = pass ? p.ns.mean : p.ns.mean1;
        const float* gstd = pass ? p.ns.std : p.ns.std1;
        const bool norm_on = pass ? normalize : (p.es.obs_normalize && __ldcg(p.ns.count + 1) > 1);
        float* obs_out = (pass && net == 0) ? p.sl.obs + (size_t)t * N * On : nullptr;
        const bool own_state = PERSIST && pass && net == 0 && t > t_first;
        if (tid < 64) { sMean[tid] = (tid < O) ? __ldcg(gmean + tid) : 0.f; sRstd[tid] = (tid < O) ? __ldcg(gstd + tid) : 1.f; }
        __syncthreads();
        if ((O & 3) == 0 && On == O) {   // 128-bit row loads, all 8 in flight per thread
            const int kq = tid & 15, k4 = kq << 2;
            float4 xv[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int env = env0 + (tid >> 4) + 16 * j;
                if (own_state) {          // persistent kernel, actor CTA: the state this CTA wrote in the previous step is still in smem
                    const float* r = sRaw + ((tid >> 4) + 16 * j) * SNW + k4;
                    xv[j] = (env < N && k4 < O) ? make_float4(r[0], r[1], r[2], r[3]) : make_float4(0.f, 0.f, 0.f, 0.f);
                } else
                xv[j] = (env < N && k4 < O) ? __ldcg(reinterpret_cast<const float4*>(raw + (size_t)env * O + k4))
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            const float m0 = sMean[k4], m1 = sMean[k4 + 1], m2 = sMean[k4 + 2], m3 = sMean[k4 + 3];
            const float r0 = sRstd[k4], r1 = sRstd[k4 + 1], r2 = sRstd[k4 + 2], r3 = sRstd[k4 + 3];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int e = (tid >> 4) + 16 * j;
                const int env = env0 + e;
                float4 v = xv[j];
                if (pass && net == 0 && k4 < O) { float* r = sRaw + e * SNW + k4; r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w; }
                if (env < N && k4 < O) {
                    if (norm_on) {
                        v.x = fminf(fmaxf(__fdiv_rn(__fadd_rn(v.x, -m0), r0), -5.f), 5.f);
                        v.y = fminf(fmaxf(__fdiv_rn(__fadd_rn(v.y, -m1), r1), -5.f), 5.f);
                        v.z = fminf(fmaxf(__fdiv_rn(__fadd_rn(v.z, -m2), r2), -5.f), 5.f);
                        v.w = fminf(fmaxf(__fdiv_rn(__fadd_rn(v.w, -m3), r3), -5.f), 5.f);
                    }
                    if (obs_out) *reinterpret_cast<float4*>(obs_out + (size_t)env * O + k4) = v;
                }
                if constexpr (X3) {
                    uint32_t w0[2], w1[2], w2[2];
                    x3::split2(v.x, v.y, w0[0], w1[0], w2[0]);
                    x3::split2(v.z, v.w, w0[1], w1[1], w2[1]);
                    const uint32_t o = B0 + x3::off128(e, k4);
                    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(o), "r"(w0[0]), "r"(w0[1]) : "memory");
                    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(o + RX_SUB), "r"(w1[0]), "r"(w1[1]) : "memory");
                    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(o + 2 * RX_SUB), "r"(w2[0]), "r"(w2[1]) : "memory");
                } else {
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tile_addr(B0, e, k4, RTC)),
                             "f"(tf32r(v.x)), "f"(tf32r(v.y)), "f"(tf32r(v.z)), "f"(tf32r(v.w))
                             : "memory");
                }
            }
        } else {
            const int k = tid & 63;
            const float mk = sMean[k], sk = sRstd[k];
#pragma unroll 8
            for (int j = 0; j < 32; ++j) {
                const int e = (tid >> 6) + 4 * j;
                const int env = env0 + e;
                float v = 0.f;
                if (env < N && k < O) {
                    v = own_state ? sRaw[e * SNW + k] : __ldcg(raw + (size_t)env * O + k);
                    if (pass && net == 0) sRaw[e * SNW + k] = v;
                    if (norm_on) v = fminf(fmaxf(__fdiv_rn(__fadd_rn(v, -mk), sk), -5.f), 5.f);
                    if (obs_out) obs_out[(size_t)env * On + k] = v;
                }
                if constexpr (X3) x3::store1_x3(B0, RX_SUB, x3::off128(e, k), v);
                else sts(tile_addr(B0, e, k, RTC), tf32r(v));
            }
        }
        if (On != O) {          // Saute: column O of the tile = the safety state (1 on final observations)
            __syncthreads();    // the staging loop above zero-filled that column
            if (tid < RTC) {
                const int env = env0 + tid;
                float z = 0.f;
                if (env < N) {
                    z = pass ? __ldcg(p.sa.safety + (size_t)(t & 1) * N + env) : 1.f;
                    if (obs_out) obs_out[(size_t)env * On + O] = z;
                }
                if constexpr (X3) x3::store1_x3(B0, RX_SUB, x3::off128(tid, O), z);
                else sts(tile_addr(B0, tid, O, RTC), tf32r(z));
            }
        }
        fence_async_smem();
        __syncthreads();
        RSTAMP(2);
        if constexpr (X3) {
            // three layers on bf16x3 tiles, one activation buffer: every epilogue starts after its layer's MMAs completed
            const bool leader = (warp == 0) && x3::elect_one_sync();
            const uint64_t dAct = x3::desc128(B0), dW1 = x3::desc128(sW1), dW2 = x3::desc128(sW2), dW3 = x3::desc128(sW3);
            if (warp == 0) {
                tc_fence_after();
                x3::gemm_x3_warp(leader, tmem + C_Z, dAct, RX_SUB, 32u, dW1, RX_WSUB, 32u, x3::idesc_bf16(128, 64, 0, 0), 4, false);
                if (leader) mma_commit(&bar);
                __syncwarp();
            }
            mbar_wait(&bar, phase); phase ^= 1;
            RSTAMP(3);
            tc_fence_after();
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
                const int c0 = 32 * h + 8 * c8;
                float v[8];
                x3::tmem_ld8(tmem + lane_base + C_Z + (uint32_t)c0, v);
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = x3::tanh_acc(v[i] + sB1[c0 + i]);
                x3::store8_x3(B0, RX_SUB, 32 * q + lane, c0, v);
            }
            fence_async_smem(); tc_fence_before();
            __syncthreads();
            if (warp == 0) {
                tc_fence_after();
                x3::gemm_x3_warp(leader, tmem + C_Z, dAct, RX_SUB, 32u, dW2, RX_WSUB, 32u, x3::idesc_bf16(128, 64, 0, 0), 4, false);
                if (leader) mma_commit(&bar);
                __syncwarp();
            }
            mbar_wait(&bar, phase); phase ^= 1;
            RSTAMP(4);
            tc_fence_after();
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
                const int c0 = 32 * h + 8 * c8;
                float v[8];
                x3::tmem_ld8(tmem + lane_base + C_Z + (uint32_t)c0, v);
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = x3::tanh_acc(v[i] + sB2[c0 + i]);
                x3::store8_x3(B0, RX_SUB, 32 * q + lane, c0, v);
            }
            fence_async_smem(); tc_fence_before();
            __syncthreads();
            if (warp == 0) {
                tc_fence_after();
                x3::gemm_x3_warp(leader, tmem + C_OUT, dAct, RX_SUB, 32u, dW3, RX_W3SUB, 32u, x3::idesc_bf16(128, 16, 0, 0), 4, false);
                if (leader) mma_commit(&bar);
                __syncwarp();
            }
            mbar_wait(&bar, phase); phase ^= 1;
            RSTAMP(5);
            tc_fence_after();
        } else {
        if (tid == 0) { tc_fence_after(); tc_gemm(tmem + C_Z, B0, RTC, sW1, 64, 128, 64, 64, false); mma_commit(&bar); }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        {
            float v[32];
            tmem_ld32(tmem + lane_base + C_Z + 32 * h, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = tanh_fast(v[i] + sB1[32 * h + i]);
            store_row32(B2, 32 * q + lane, 32 * h, RTC, v);
        }
        fence_async_smem(); tc_fence_before();
        __syncthreads();
        if (tid == 0) { tc_fence_after(); tc_gemm(tmem + C_Z, B2, RTC, sW2, 64, 128, 64, 64, false); mma_commit(&bar); }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        {
            float v[32];
            tmem_ld32(tmem + lane_base + C_Z + 32 * h, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = tanh_fast(v[i] + sB2[32 * h + i]);
            store_row32(B0, 32 * q + lane, 32 * h, RTC, v);
        }
        fence_async_smem(); tc_fence_before();
        __syncthreads();
        if (tid == 0) { tc_fence_after(); tc_gemm(tmem + C_OUT, B0, RTC, sW3, 16, 128, 16, 64, false); mma_commit(&bar); }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        }
        if (h == 0) {
            float o16[16];
            tmem_ld16(tmem + lane_base + C_OUT, o16);
            const int e = 32 * q + lane;
            const int env = env0 + e;
            if (net != 0) {
                if (env < N) {
                    const float v = o16[0] + sB3[0];
                    if (pass == 0) {
                        const size_t idx = (size_t)(t - 1) * N + env;
                        const unsigned f = __ldcg(p.sl.flags + idx);
                        if ((f & OSB_FLAG_TRUNCATED) && !(f & OSB_FLAG_TERMINATED))
                            (net == 1 ? p.sl.boot_r : p.sl.boot_c)[idx] = v;
                    } else if (!is_tail) {
                        (net == 1 ? p.sl.val_r : p.sl.val_c)[(size_t)t * N + env] = v;
                    } else {
                        const size_t idx = (size_t)(T - 1) * N + env;
                        if (__ldcg(p.sl.flags + idx) == 0) (net == 1 ? p.sl.boot_r : p.sl.boot_c)[idx] = v;
                    }
                }
            } else {
#pragma unroll
                for (int a = 0; a < 16; ++a) sAct[e * OUTP + a] = o16[a] + sB3[a];   // mu
            }
        }
        tc_fence_before();
        __syncthreads();
    }

    RSTAMP(6);
    if (net == 0) {
        // ---- sample + log-prob.  A <= 8: thread -> (env e = 64 g + tid / 4, action pair pr = tid % 4): one Philox block
        //      yields both normals of the pair (Box-Muller cos / sin); the log-prob terms are summed in the tree
        //      ((t0+t1)+(t2+t3)) + ((t4+t5)+(t6+t7)) of rollout_step_kernel.  A > 8: one action per lane as there. -----------
        if (A <= 8) {
            const int pr = tid & 3, a0 = 2 * pr, a1 = a0 + 1;
#pragma unroll 1
            for (int g = 0; g < 2; ++g) {
                const int e = 64 * g + (tid >> 2);
                const int env = env0 + e;
                const bool ok = env < N;
                float n0 = 0.f, n1 = 0.f;
                if (ok && a0 < A) {
                    if (eps_t) { n0 = eps_t[(size_t)env * A + a0]; n1 = (a1 < A) ? eps_t[(size_t)env * A + a1] : 0.f; }
                    else philox_normal2(p.noise_seed, p.es.env_id_offset + env, gstep_t, pr, n0, n1);
                }
                float lp = 0.f;
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int a = a0 + u;
                    if (a < A) {
                        const float mu = sAct[e * OUTP + a];
                        const float sd = sSd[a];
                        const float act = __fadd_rn(mu, __fmul_rn(sd, u ? n1 : n0));      // Normal.rsample: loc + eps * scale
                        const float d = __fadd_rn(act, -mu);
                        float term = __fdiv_rn(-__fmul_rn(d, d), sSd[16 + a]);               // / (2 var)
                        term = __fadd_rn(__fadd_rn(term, -sSd[32 + a]), -0.9189385332046727f);
                        lp += term;
                        sAct[e * OUTP + a] = act;
                        if (ok) p.sl.act[((size_t)t * N + env) * A + a] = act;
                    }
                }
                lp += __shfl_xor_sync(0xffffffffu, lp, 1);
                lp += __shfl_xor_sync(0xffffffffu, lp, 2);
                if (ok && pr == 0) p.sl.logp[(size_t)t * N + env] = lp;
            }
        } else {
            const int qq = tid & 7;
#pragma unroll 1
            for (int g = 0; g < RTC / 32; ++g) {
                const int e = 32 * g + (tid >> 3);
                const int env = env0 + e;
                const bool ok = env < N;
                float lp = 0.f;
                for (int a = qq; a < A; a += 8) {
                    const float mu = sAct[e * OUTP + a];
                    const float sd = sSd[a];
                    float eps = 0.f;
                    if (ok)
                        eps = eps_t ? eps_t[(size_t)env * A + a]
                                    : philox_normal(p.noise_seed, p.es.env_id_offset + env, gstep_t, a);
                    const float act = __fadd_rn(mu, __fmul_rn(sd, eps));
                    const float d = __fadd_rn(act, -mu);
                    float term = __fdiv_rn(-__fmul_rn(d, d), sSd[16 + a]);
                    term = __fadd_rn(__fadd_rn(term, -sSd[32 + a]), -0.9189385332046727f);
                    lp += term;
                    sAct[e * OUTP + a] = act;
                    if (ok) p.sl.act[((size_t)t * N + env) * A + a] = act;
                }
                lp += __shfl_xor_sync(0xffffffffu, lp, 1);
                lp += __shfl_xor_sync(0xffffffffu, lp, 2);
                lp += __shfl_xor_sync(0xffffffffu, lp, 4);
                if (ok && qq == 0) p.sl.logp[(size_t)t * N + env] = lp;
            }
        }
        __syncthreads();
        if (p.et.cost_acc) {      // EarlyTerminated: the step's cost is known from state dim 0 -> finish flags before the transition
            if (tid < RTC && env0 + tid < N) {
                const int env = env0 + tid;
                const float acc = __fadd_rn(p.et.cost_acc[env], env_step_cost(p.es, sRaw[tid * SNW], sAct[tid * OUTP], __ldg(p.st.bias)));
                if (acc > p.et.cost_limit) sFlag[tid] |= ((sFlag[tid] & 1) ? 16 : 0) | 1 | 2 | 8;   // bit 3 early, bit 4 both ends at once
                sEarlyAcc[tid] = acc;
            }
            __syncthreads();
        }
        RSTAMP(7);
        // ---- env transition + normaliser sums, elementwise: thread -> (dim j = tid % 64, env quarter g = tid / 64).
        //      The raw state comes from shared memory (kept by the obs staging), the next state goes out in whole
        //      rows (coalesced), the fixed-point column sums accumulate in registers. ---------------------------------------
        {
            const int j = tid & 63, g = tid >> 6;
            long long sx = 0, sxx = 0, fx = 0, fxx = 0;
            if (j < O) {
                const int ja = j % A;
                const float bj = __ldg(p.st.bias + j);
#pragma unroll 4
                for (int e = 32 * g; e < 32 * g + 32; ++e) {
                    const int env = env0 + e;
                    if (env < N) {
                        // ActionScale (wrapper.py:L510-512) from [-1,1] onto the env's [-1,1] box
                        float a = sAct[e * OUTP + ja];
                        a = __fadd_rn(__fadd_rn(a, 1.f), -1.f);
                        a = fminf(fmaxf(a, -1.f), 1.f);
                        const float sn = env_next_value(sRaw[e * SNW + j], a, bj);
                        const int fl = sFlag[e];
                        float nv = sn;
                        if (fl & 1) {
                            nv = env_reset_value(p.es, p.es.env_id_offset + env, sEpi[e] + ((fl & 16) ? 2u : 1u), j);
                            p.st.final_raw[((size_t)(t & 1) * N + env) * O + j] = sn;
                            fx += to_fix(sn); fxx += to_fix(__fmul_rn(sn, sn));
                        }
                        s_nxt[(size_t)env * O + j] = nv;
                        if (PERSIST) sRaw[e * SNW + j] = nv;            // next step's obs staging of this CTA reads it back from here
                        sSn[e * SNW + j] = sn;
                        sx += to_fix(nv); sxx += to_fix(__fmul_rn(nv, nv));
                    }
                }
            }
            if (p.es.obs_normalize) {
                sAcc[(g * 4 + 0) * 64 + j] = sx; sAcc[(g * 4 + 1) * 64 + j] = sxx;
                sAcc[(g * 4 + 2) * 64 + j] = fx; sAcc[(g * 4 + 3) * 64 + j] = fxx;
            }
        }
        __syncthreads();
        RSTAMP(8);
        // ---- reward / cost / flags / episode bookkeeping: 2 threads per env.  Thread `e_half` owns the partial sums
        //      p_q, q = 4*e_half .. 4*e_half+3 (dims j = q mod 8): the summation tree is the one of the spec
        //      ((p0+p1)+(p2+p3)) + ((p4+p5)+(p6+p7)). ------------------------------------------------------------------
        {
            const int env = my_env;
            const bool ok = my_ok;
            float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
            for (int jb = 4 * e_half; jb < O; jb += 8) {
#pragma unroll
                for (int qi = 0; qi < 4; ++qi) {
                    const int j = jb + qi;
                    if (j < O) { const float sn = sSn[e_env * SNW + j]; part[qi] = __fadd_rn(part[qi], __fmul_rn(sn, sn)); }
                }
            }
            float tot = __fadd_rn(__fadd_rn(part[0], part[1]), __fadd_rn(part[2], part[3]));
            tot = __fadd_rn(tot, __shfl_xor_sync(0xffffffffu, tot, 1));
            if (ok && e_half == 0) {
                const int fl = sFlag[e_env];
                const bool fin = fl & 1, term = fl & 2, trunc = fl & 4;
                const uint32_t epi = sEpi[e_env];
                const bool early = fl & 8;
                const float rew = early ? 0.f : __fadd_rn(1.f, -__fdiv_rn(tot, (float)O));
                const float cst = (sSn[e_env * SNW] > p.es.cost_threshold) ? 1.f : 0.f;
                if (p.et.cost_acc) p.et.cost_acc[env] = early ? 0.f : sEarlyAcc[e_env];
                const size_t idx = (size_t)t * N + env;
                p.sl.rew[idx] = saute_step(p.sa, t, N, env, rew, cst, fin);
                p.sl.cost[idx] = cst;
                p.sl.flags[idx] = (uint8_t)((term ? OSB_FLAG_TERMINATED : 0u) | (trunc ? OSB_FLAG_TRUNCATED : 0u));
                const float erv = __fadd_rn(p.st.ep_ret[env], rew);
                const float ecv = __fadd_rn(p.st.ep_cost[env], cst);
                const int el = p.st.ep_len[env] + 1;
                if (fin) {
                    const size_t TN = (size_t)T * N;
                    p.sl.epfin[idx] = erv;
                    p.sl.epfin[TN + idx] = ecv;
                    p.sl.epfin[2 * TN + idx] = (float)el;
                    p.st.ep_ret[env] = 0.f; p.st.ep_cost[env] = 0.f; p.st.ep_len[env] = 0;
                    p.st.episode[env] = epi + ((fl & 16) ? 2u : 1u);
                    p.st.ep_step[env] = 0;
                } else {
                    p.st.ep_ret[env] = erv; p.st.ep_cost[env] = ecv; p.st.ep_len[env] = el;
                    p.st.ep_step[env] = sStep[e_env] + 1;
                }
                p.st.gstep[env] = sGstep[e_env] + 1u;
            }
        }
        if (p.es.obs_normalize) {
            if (tid < O) {
                long long a0 = 0, a1 = 0, a2 = 0, a3 = 0;
                for (int gg = 0; gg < 4; ++gg) {
                    a0 += sAcc[(gg * 4 + 0) * 64 + tid]; a1 += sAcc[(gg * 4 + 1) * 64 + tid];
                    a2 += sAcc[(gg * 4 + 2) * 64 + tid]; a3 += sAcc[(gg * 4 + 3) * 64 + tid];
                }
                atomicAdd((unsigned long long*)(p.ns.acc_all + tid), (unsigned long long)a0);
                atomicAdd((unsigned long long*)(p.ns.acc_all + O + tid), (unsigned long long)a1);
                if (a2 != 0 || a3 != 0) {
                    atomicAdd((unsigned long long*)(p.ns.acc_fin + tid), (unsigned long long)a2);
                    atomicAdd((unsigned long long*)(p.ns.acc_fin + O + tid), (unsigned long long)a3);
                }
            }
            if (tid == 64) {
                int nfin = 0;
                for (int r = 0; r < RTC; ++r) nfin += (env0 + r < N) ? (sFlag[r] & 1) : 0;
                if (nfin) atomicAdd(p.ns.fin_count, nfin);
            }
        }
    }
    RSTAMP(9);
    if (PERSIST) {
        if (!is_tail) {
            // grid barrier; the last CTA to arrive folds the step's sums into the running statistics, then releases
            __threadfence();
            __syncthreads();
            if (tid == 0) s_last = (atomicAdd(p.bar_ctr, 1u) == gridDim.x * gridDim.y * (unsigned)(t + 1) - 1u) ? 1 : 0;
            __syncthreads();
            if (s_last) {
                if (p.es.obs_normalize) norm_finalize(p.ns, O, (long long)N);
                __threadfence();
                __syncthreads();
                if (tid == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p.bar_flag), "r"((unsigned)(t + 1)) : "memory");
            } else if (tid == 0) {
                unsigned v;
                do { asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p.bar_flag) : "memory"); } while (v < (unsigned)(t + 1));
            }
            __syncthreads();
            RSTAMP(10);
        }
    } else if (p.es.obs_normalize && !is_tail) {
        __threadfence();
        __syncthreads();
        if (tid == 0) s_last = (atomicAdd(p.ns.ticket, 1u) == gridDim.x * gridDim.y - 1) ? 1 : 0;
        __syncthreads();
        if (s_last) norm_finalize(p.ns, O, (long long)N);
    }
    }   // step loop
#undef RSTAMP
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

static size_t rollout_tc_smem_bytes(bool x3) {
    return 1024 + (x3 ? RTC_FOFF_X3 : RTC_FOFF_TF32) +
           (64 + 64 + 16 + 64 + 64 + RTC * OUTP + 2 * RTC * SNW) * sizeof(float) + 4 * 4 * 64 * sizeof(long long) +
           5 * RTC * sizeof(int) + 48 * sizeof(float) + 64;
}

// Window of the last <= W finished episodes in (step, env) append order: Logger deque semantics
// (common/logger.py:L253-282 with window_lens; adapter/onpolicy_adapter.py:L159-175).
// ring[3][W] holds (EpRet, EpCost, EpLen); meta[0] = number of valid entries, meta[1] = head.
// Single CTA of 1024 threads: find the first row (from the end) after which >= W episodes finished,
// then append rows in order with a block-wide ordered compaction (exclusive scan of counts).
__global__ void __launch_bounds__(1024) episode_window_kernel(const uint8_t* __restrict__ flags,
                                                              const float* __restrict__ epfin,
                                                              int T, int N, int W,
                                                              float* __restrict__ ring,
                                                              int* __restrict__ meta) {
    __shared__ int s_cnt, s_total, s_warp[32], s_base;
    const size_t TN = (size_t)T * N;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int seg = (N + 1023) / 1024;          // contiguous envs per thread
    const int lo = min(N, tid * seg), hi = min(N, lo + seg);
    if (tid == 0) s_total = 0;
    int first_row = T;
    for (int t = T - 1; t >= 0; --t) {
        if (tid == 0) s_cnt = 0;
        __syncthreads();
        int cnt = 0;
        for (int i = lo; i < hi; ++i) cnt += flags[(size_t)t * N + i] != 0;
        if (cnt) atomicAdd(&s_cnt, cnt);
        __syncthreads();
        first_row = t;
        if (tid == 0) s_total += s_cnt;
        __syncthreads();
        if (s_total >= W) break;
    }
    __syncthreads();
    const int total_new = s_total;
    if (total_new == 0) return;
    const int head0 = meta[1], count0 = meta[0];
    const int skip = total_new > W ? total_new - W : 0;   // only the last W appended entries survive
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int t = first_row; t < T; ++t) {
        int cnt = 0;
        for (int i = lo; i < hi; ++i) cnt += flags[(size_t)t * N + i] != 0;
        // block exclusive scan of cnt
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_warp[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            int w = s_warp[lane], wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += v;
            }
            s_warp[lane] = wi - w;   // exclusive warp offsets
            if (lane == 31) s_cnt = wi;  // row total
        }
        __syncthreads();
        int seq = s_base + s_warp[wid] + incl - cnt;   // sequence index of my first entry
        for (int i = lo; i < hi; ++i) {
            const size_t idx = (size_t)t * N + i;
            if (flags[idx] != 0) {
                if (seq >= skip) {
                    const int pos = (head0 + (seq - skip)) % W;
                    ring[0 * W + pos] = epfin[idx];
                    ring[1 * W + pos] = epfin[TN + idx];
                    ring[2 * W + pos] = epfin[2 * TN + idx];
                }
                ++seq;
            }
        }
        __syncthreads();
        if (tid == 0) s_base += s_cnt;
        __syncthreads();
    }
    if (tid == 0) {
        const int kept = total_new - skip;
        meta[1] = (head0 + kept) % W;
        meta[0] = min(W, count0 + kept);
    }
}

// window_sums[4] = {sum EpRet, sum EpCost, sum EpLen, count} over the ring (fp64).
__global__ void window_sums_kernel(const float* __restrict__ ring, const int* __restrict__ meta,
                                   int W, double* __restrict__ window_sums) {
    if (threadIdx.x != 0) return;
    const int count = meta[0];
    double s[3] = {0, 0, 0};
    for (int q = 0; q < 3; ++q)
        for (int i = 0; i < count; ++i) s[q] += (double)ring[q * W + i];
    window_sums[0] = s[0]; window_sums[1] = s[1]; window_sums[2] = s[2];
    window_sums[3] = (double)count;
}

}  // namespace osb

using namespace osb;

static SauteSpec g_saute = {nullptr, 1.f, 1.f, 0.f, 1.f};
static EarlySpec g_early = {nullptr, 0.f};

static size_t rollout_smem_bytes(int O) {   // O = network input width
    size_t f = NETSMEM_FLOATS_FWD + 3 * RT * LD + RT * LDO + 2 * (size_t)O + RT * OUTP +
               2 * RT * (KC + 1) + 3 * RT;
    return f * sizeof(float);
}

extern "C" {

// Opaque-struct-free C ABI: the caller passes plain device pointers.
int osb_env_reset(int O, int A, int max_episode_steps, unsigned seed, unsigned term_threshold,
                  unsigned env_id_offset, float cost_threshold, int obs_normalize, int N,
                  float* s_raw, float* final_raw, int* ep_step, unsigned* episode, unsigned* gstep,
                  float* ep_ret, float* ep_cost, int* ep_len, const float* bias,
                  float* norm_mean, float* norm_sumsq, float* norm_std, float* norm_mean1,
                  float* norm_std1, long long* norm_count, long long* acc_all, long long* acc_fin,
                  int* fin_count, int* had_fin, unsigned* ticket, void* stream) {
    OSB_CHECK_ARG(O > 0 && A > 0 && A <= OUTP && N > 0, "bad dims (need 0 < A <= 16)");
    EnvSpec es{O, A, max_episode_steps, seed, term_threshold, env_id_offset, cost_threshold, obs_normalize};
    EnvState st{s_raw, final_raw, ep_step, episode, gstep, ep_ret, ep_cost, ep_len, bias};
    NormState ns{norm_mean, norm_sumsq, norm_std, norm_mean1, norm_std1, norm_count, acc_all,
                 acc_fin, fin_count, had_fin, ticket};
    env_reset_kernel<<<(N + RT - 1) / RT, NTHREADS, 0, (cudaStream_t)stream>>>(es, st, ns, g_saute, N);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

static long long* g_rollout_dbg = nullptr;

static int launch_step(StepArgs& p, cudaStream_t stream) {
    const int On = p.es.O + (p.sa.safety ? 1 : 0);
    if ((p.precision == 1 || p.precision == 2) && On <= 64) {
        const bool x3 = p.precision == 2;
        const size_t smem_tc = rollout_tc_smem_bytes(x3);
        static bool attr_tc = false;
        if (!attr_tc) {
            OSB_CUDA(cudaFuncSetAttribute(rollout_step_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rollout_tc_smem_bytes(false)));
            OSB_CUDA(cudaFuncSetAttribute(rollout_step_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rollout_tc_smem_bytes(true)));
            OSB_CUDA(cudaFuncSetAttribute(rollout_step_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rollout_tc_smem_bytes(false)));
            OSB_CUDA(cudaFuncSetAttribute(rollout_step_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rollout_tc_smem_bytes(true)));
            attr_tc = true;
        }
        dim3 grid_tc((p.N + RTC - 1) / RTC, p.is_tail ? 2 : 3);
        if (p.bar_ctr != nullptr) {
            // the whole epoch in one cooperative launch (every CTA resident: the step barrier is a software grid barrier)
            OSB_CUDA(cudaMemsetAsync(p.bar_ctr, 0, 2 * sizeof(unsigned int), stream));
            void* args[] = {&p};
            osb_count_launch();
            OSB_CUDA(cudaLaunchCooperativeKernel(x3 ? (void*)rollout_step_tc_kernel<true, true> : (void*)rollout_step_tc_kernel<false, true>,
                                                 dim3((p.N + RTC - 1) / RTC, 3), dim3(NTHREADS), args, smem_tc, stream));
            return OSB_OK;
        }
        if (x3) rollout_step_tc_kernel<true, false><<<grid_tc, NTHREADS, smem_tc, stream>>>(p);
        else rollout_step_tc_kernel<false, false><<<grid_tc, NTHREADS, smem_tc, stream>>>(p);
        OSB_LAUNCH_CHECK();
        return OSB_OK;
    }
    const size_t smem = rollout_smem_bytes(On);
    static size_t attr = 0;
    if (smem > attr) {
        OSB_CUDA(cudaFuncSetAttribute(rollout_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    dim3 grid((p.N + RT - 1) / RT, p.is_tail ? 2 : 3);
    rollout_step_kernel<<<grid, NTHREADS, smem, stream>>>(p);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

// Saute / Simmer mode of the following osb_env_reset / osb_rollout_* calls (process-wide until changed): safety = [2][N]
// device floats (the safety state z by step parity), or NULL for the plain OnPolicyAdapter semantics.  The networks then
// take O + 1 inputs ([normalised obs | z]) and the obs slab rows are O + 1 wide.  saute_adapter.py:L135-217.
int osb_rollout_set_saute(float* safety, float safety_budget, float saute_gamma, float unsafe_reward, float safety_init) {
    OSB_CHECK_ARG(safety == nullptr || (safety_budget > 0.f && saute_gamma > 0.f), "safety_budget and saute_gamma must be positive");
    g_saute = SauteSpec{safety, safety_budget, saute_gamma, unsafe_reward, safety_init};
    return OSB_OK;
}

// EarlyTerminated mode of the following osb_rollout_* calls (process-wide until changed): cost_acc = [N] device floats
// (per-env accumulated cost, persistent across episodes and epochs) or NULL.  early_terminated_adapter.py:L56-98.
int osb_rollout_set_early_termination(float* cost_acc, float cost_limit) {
    g_early = EarlySpec{cost_acc, cost_limit};
    return OSB_OK;
}

// development aid: clock64 stamps of the persistent rollout kernel go to buf (1024 long long), NULL turns it off
int osb_rollout_debug_buffer(long long* buf) { g_rollout_dbg = buf; return OSB_OK; }

int osb_rollout_step(int O, int A, int max_episode_steps, unsigned seed, unsigned term_threshold,
                     unsigned env_id_offset, float cost_threshold, int obs_normalize, int N, int T,
                     int t, float* s_raw, float* final_raw, int* ep_step, unsigned* episode,
                     unsigned* gstep, float* ep_ret, float* ep_cost, int* ep_len, const float* bias,
                     float* norm_mean, float* norm_sumsq, float* norm_std, float* norm_mean1,
                     float* norm_std1, long long* norm_count, long long* acc_all,
                     long long* acc_fin, int* fin_count, int* had_fin, unsigned* ticket,
                     float* obs, float* act, float* logp, float* rew, float* cost, float* val_r,
                     float* val_c, float* boot_r, float* boot_c, unsigned char* flags, float* epfin,
                     const float* theta, const float* eps, unsigned noise_seed,
                     unsigned global_step, int precision, void* stream) {
    OSB_CHECK_ARG(O > 0 && A > 0 && A <= OUTP && N > 0 && T > 0, "bad dims (need 0 < A <= 16)");
    OSB_CHECK_ARG(t >= 0 && t <= T, "step index out of range");
    StepArgs p;
    p.es = EnvSpec{O, A, max_episode_steps, seed, term_threshold, env_id_offset, cost_threshold, obs_normalize};
    p.st = EnvState{s_raw, final_raw, ep_step, episode, gstep, ep_ret, ep_cost, ep_len, bias};
    p.ns = NormState{norm_mean, norm_sumsq, norm_std, norm_mean1, norm_std1, norm_count, acc_all,
                     acc_fin, fin_count, had_fin, ticket};
    p.sl = Slabs{obs, act, logp, rew, cost, val_r, val_c, boot_r, boot_c, flags, epfin};
    p.sa = g_saute; p.et = g_early;
    p.theta = theta; p.eps = eps; p.noise_seed = noise_seed; p.global_step = global_step;
    p.t = t; p.T = T; p.N = N; p.is_tail = (t == T) ? 1 : 0; p.precision = precision;
    p.bar_ctr = nullptr; p.bar_flag = nullptr; p.dbg = nullptr;
    return launch_step(p, (cudaStream_t)stream);
}

int osb_rollout_epoch(int O, int A, int max_episode_steps, unsigned seed, unsigned term_threshold,
                      unsigned env_id_offset, float cost_threshold, int obs_normalize, int N, int T,
                      float* s_raw, float* final_raw, int* ep_step, unsigned* episode,
                      unsigned* gstep, float* ep_ret, float* ep_cost, int* ep_len, const float* bias,
                      float* norm_mean, float* norm_sumsq, float* norm_std, float* norm_mean1,
                      float* norm_std1, long long* norm_count, long long* acc_all,
                      long long* acc_fin, int* fin_count, int* had_fin, unsigned* ticket,
                      float* obs, float* act, float* logp, float* rew, float* cost, float* val_r,
                      float* val_c, float* boot_r, float* boot_c, unsigned char* flags, float* epfin,
                      const float* theta, const float* eps_all, unsigned noise_seed,
                      unsigned epoch_index, int W, float* ring, int* meta, double* window_sums,
                      int precision, void* stream) {
    OSB_CHECK_ARG(O > 0 && A > 0 && A <= OUTP && N > 0 && T > 0, "bad dims (need 0 < A <= 16)");
    cudaStream_t s = (cudaStream_t)stream;
    int rc = osb_env_reset(O, A, max_episode_steps, seed, term_threshold, env_id_offset,
                           cost_threshold, obs_normalize, N, s_raw, final_raw, ep_step, episode,
                           gstep, ep_ret, ep_cost, ep_len, bias, norm_mean, norm_sumsq, norm_std,
                           norm_mean1, norm_std1, norm_count, acc_all, acc_fin, fin_count, had_fin,
                           ticket, stream);
    if (rc) return rc;
    StepArgs p;
    p.es = EnvSpec{O, A, max_episode_steps, seed, term_threshold, env_id_offset, cost_threshold, obs_normalize};
    p.st = EnvState{s_raw, final_raw, ep_step, episode, gstep, ep_ret, ep_cost, ep_len, bias};
    p.ns = NormState{norm_mean, norm_sumsq, norm_std, norm_mean1, norm_std1, norm_count, acc_all,
                     acc_fin, fin_count, had_fin, ticket};
    p.sl = Slabs{obs, act, logp, rew, cost, val_r, val_c, boot_r, boot_c, flags, epfin};
    p.sa = g_saute; p.et = g_early;
    p.theta = theta; p.noise_seed = noise_seed; p.T = T; p.N = N; p.precision = precision;
    p.bar_ctr = nullptr; p.bar_flag = nullptr; p.dbg = g_rollout_dbg;
    // tensor-core modes with every CTA resident (grid = env tiles x 3 networks <= SMs): one persistent launch per epoch
    static const bool stepwise = getenv("OSB_ROLLOUT_STEPWISE") != nullptr;
    static int n_sm = 0;
    if (!n_sm) { int dev = 0; OSB_CUDA(cudaGetDevice(&dev)); OSB_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev)); }
    if (!stepwise && (precision == 1 || precision == 2) && O + (g_saute.safety ? 1 : 0) <= 64 && ((N + RTC - 1) / RTC) * 3 <= n_sm) {
        static unsigned int* d_bar = nullptr;
        if (!d_bar) OSB_CUDA(cudaMalloc(&d_bar, 64));
        p.bar_ctr = d_bar; p.bar_flag = d_bar + 1;
        p.t = 0; p.is_tail = 0; p.eps = eps_all; p.global_step = epoch_index * (unsigned)T;
        rc = launch_step(p, s);
        if (rc) return rc;
        return osb_episode_window(flags, epfin, T, N, W, ring, meta, window_sums, stream);
    }
    for (int t = 0; t <= T; ++t) {
        p.t = t; p.is_tail = (t == T) ? 1 : 0;
        p.eps = (eps_all && t < T) ? eps_all + (size_t)t * N * A : nullptr;
        p.global_step = epoch_index * (unsigned)T + (unsigned)t;
        rc = launch_step(p, s);
        if (rc) return rc;
    }
    return osb_episode_window(flags, epfin, T, N, W, ring, meta, window_sums, stream);
}

int osb_episode_window(const unsigned char* flags, const float* epfin, int T, int N, int W,
                       float* ring, int* meta, double* window_sums, void* stream) {
    OSB_CHECK_ARG(flags && epfin && ring && meta && window_sums && W > 0, "bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    episode_window_kernel<<<1, 1024, 0, s>>>(flags, epfin, T, N, W, ring, meta);
    OSB_LAUNCH_CHECK();
    window_sums_kernel<<<1, 32, 0, s>>>(ring, meta, W, window_sums);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

}  // extern "C"
