// Optimiser-side kernels: partial-gradient reduction, per-network grad-norm clipping, Adam,
// on-device Lagrange multiplier update, KL early-stop flag, and the block-parallel conjugate
// gradient vector algebra for CPO / TRPO-Lag.
//
// Replaces the reference's
//   clip_grad_norm_ + optimizer.step()   algorithms/on_policy/base/policy_gradient.py:L436-443,L476-483,L517-524
//   critic L2 regulariser                base/policy_gradient.py:L431-433
//   torch.optim.Adam (single-tensor)     (dependency; restated: lerp first moment, addcmul second)
//   Lagrange.update_lagrange_multiplier  common/lagrange.py:L114-136
//   KL early stop                        base/policy_gradient.py:L383-397
//   conjugate_gradients                  utils/math.py:L86-132
#include "common.cuh"
#include "mlp.cuh"
#include "optim.cuh"
#include <cooperative_groups.h>
#include <string.h>
#include <type_traits>

namespace osb {

constexpr int OT = 256;

struct ReduceArgs {
    const float* gpart;       // [nblocks][P]
    const float* stats_part;  // [nblocks][3][8]
    int nblocks, P, O, A;
    float* theta;
    float* grad;              // [P]
    float critic_norm_coef;   // 0 -> off
    int net_mask;
    float* sumsq_part;        // [3][NB]
    int* adam_step;           // [3]
    float* train_stats;       // [3][8] running sums over minibatch steps
    const int* stop_flag;
};

__global__ void __launch_bounds__(OT) grad_reduce_kernel(ReduceArgs p) {
    if (p.stop_flag && *p.stop_flag) return;
    const int net = blockIdx.y;
    if (!((p.net_mask >> net) & 1)) return;
    __shared__ float red[OT / 32], red2[OT / 32];
    const NetLayout L = net_layout(net, p.O, p.A);
    const int noff = net_offset(net, p.O, p.A);
    const int pl = blockIdx.x * OT + threadIdx.x;
    float g = 0.f;
    if (pl < L.size) {
        const int q = noff + pl;
        for (int b = 0; b < p.nblocks; ++b) g += p.gpart[(size_t)b * p.P + q];
        if (net != 0 && p.critic_norm_coef > 0.f) g += 2.f * p.critic_norm_coef * p.theta[q];
        p.grad[q] = g;
    }
    float th = 0.f;
    if (pl < L.size && net != 0) th = p.theta[noff + pl];
    float s = warp_sum(g * g), s2 = warp_sum(th * th);
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = s; red2[threadIdx.x >> 5] = s2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f, t2 = 0.f;
        for (int w = 0; w < OT / 32; ++w) { t += red[w]; t2 += red2[w]; }
        p.sumsq_part[net * gridDim.x + blockIdx.x] = t;
        p.sumsq_part[(3 + net) * gridDim.x + blockIdx.x] = t2;   // sum theta^2 (critic regulariser)
        if (blockIdx.x == 0) {
            p.adam_step[net] += 1;
            // per-minibatch means of the loss statistics; the regulariser is added in clip_adam
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int b = 0; b < p.nblocks; ++b)
                for (int i = 0; i < 4; ++i) acc[i] += p.stats_part[((size_t)b * 3 + net) * 8 + i];
            const float inv = acc[3] > 0.f ? 1.f / acc[3] : 0.f;
            float* ts = p.train_stats + net * 8;
            ts[0] += acc[0] * inv;   // mean loss of this minibatch
            ts[1] += acc[1] * inv;   // mean ratio
            ts[2] += acc[2] * inv;   // mean kl (FOCOPS)
            ts[3] += 1.f;            // number of minibatch steps
        }
    }
}

struct AdamArgs {
    float* grad;
    float* theta;
    float* m;
    float* v;
    const int* adam_step;      // [3]
    const float* sumsq_part;   // [3][NB]
    int NB, O, A;
    float max_grad_norm;       // <= 0 -> no clipping
    float lr[3];
    float grad_scale;          // 1 / world_size applied before Adam (avg_grads)
    float critic_norm_coef;
    float* train_stats;
    int do_clip, do_adam, net_mask;
    const int* stop_flag;
};

__global__ void __launch_bounds__(OT) clip_adam_kernel(AdamArgs p) {
    if (p.stop_flag && *p.stop_flag) return;
    const int net = blockIdx.y;
    if (!((p.net_mask >> net) & 1)) return;
    const NetLayout L = net_layout(net, p.O, p.A);
    const int pl = blockIdx.x * OT + threadIdx.x;
    if (p.do_clip && net != 0 && p.critic_norm_coef > 0.f && blockIdx.x == 0 && threadIdx.x == 0) {
        // logged critic loss = mse + coef * sum(theta^2) (policy_gradient.py:L429-433)
        float t2 = 0.f;
        for (int b = 0; b < p.NB; ++b) t2 += p.sumsq_part[(3 + net) * p.NB + b];
        p.train_stats[net * 8] += p.critic_norm_coef * t2;
    }
    if (pl >= L.size) return;
    const int q = net_offset(net, p.O, p.A) + pl;
    float g = p.grad[q];
    if (p.do_clip && p.max_grad_norm > 0.f) {
        float tot = 0.f;
        for (int b = 0; b < p.NB; ++b) tot += p.sumsq_part[net * p.NB + b];
        g *= clip_coef(p.max_grad_norm, tot);
        p.grad[q] = g;
    }
    if (!p.do_adam) return;
    g *= p.grad_scale;
    const AdamBias b = adam_bias(p.lr[net], p.adam_step[net]);
    float m = p.m[q], v = p.v[q];
    p.theta[q] = adam_update(g, p.theta[q], m, v, b);
    p.m[q] = m; p.v[q] = v;
}

// Multi-rank all-reduce of the fused kernel: a one-shot exchange over NVLink peer memory (cudaIpc-mapped buffers,
// NVSwitch gives every peer full bandwidth).  Each rank publishes its clipped flat gradient (99 KB) in its own exchange
// buffer, raises a step flag in every peer's memory, waits for the peers' flags, then sums the peers' buffers in rank
// order (deterministic, identical on every rank) straight into the Adam update -- the reference's order
// clip -> average -> step (policy_gradient.py:L437-443; distributed.py:L193-198 avg_grads).
struct P2PExchange {
    float* const* peer_buf;        // [world] exchange buffers, each [2][P] (double-buffered by step parity)
    unsigned int* const* peer_flag; // [world] flag arrays, each [2][world]
    int world, rank;
    unsigned int step_id;          // monotonically increasing, identical on all ranks
    int* error_flag;               // set when a peer does not show up (timeout) instead of hanging the GPU
};

// Partial reduction + critic L2 term + per-network clip (+ all-reduce) + Adam in ONE cooperative launch
// (grid.sync() between the norm reduction and the parameter update).
struct FusedOptArgs {
    ReduceArgs r;
    float* m;
    float* v;
    float max_grad_norm;
    float lr[3];
};
struct P2POptArgs : FusedOptArgs {
    P2PExchange x;
};
template <bool P2P> using OptArgs = std::conditional_t<P2P, P2POptArgs, FusedOptArgs>;

// Fixed-order sum of the per-CTA partial gradients of one parameter, 16 loads in flight at a time
// (the in-order issue would otherwise serialise one L2 round trip per small batch).
__device__ __forceinline__ float reduce_partials16(const float* __restrict__ gpart, int nblocks, int P, int q) {
    float g = 0.f;
    for (int b = 0; b < nblocks; b += 16) {
        float t[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) t[u] = (b + u < nblocks) ? __ldcg(gpart + (size_t)(b + u) * P + q) : 0.f;
        g += (((t[0] + t[1]) + (t[2] + t[3])) + ((t[4] + t[5]) + (t[6] + t[7]))) +
             (((t[8] + t[9]) + (t[10] + t[11])) + ((t[12] + t[13]) + (t[14] + t[15])));
    }
    return g;
}

// After the grid barrier: warp 0 of every CTA folds the per-CTA squared norms (lanes stride over CTAs, fixed
// butterfly) into the clip scale and the Adam step sizes; in CTA 0 warp 1 folds the loss statistics.
__device__ __forceinline__ void clip_scale_and_stats(const FusedOptArgs& p, int net, int step_t, float* s_scale,
                                                     AdamBias* s_bias) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int G = gridDim.x;
    if (warp == 0 || (warp == 1 && blockIdx.x == 0)) {
        float tot = 0.f, t2 = 0.f;
        for (int b = lane; b < G; b += 32) { tot += __ldcg(p.r.sumsq_part + net * G + b); t2 += __ldcg(p.r.sumsq_part + (3 + net) * G + b); }
        tot = warp_sum(tot); t2 = warp_sum(t2);
        if (warp == 0) {
            if (lane == 0) {
                *s_scale = clip_coef(p.max_grad_norm, tot);
                *s_bias = adam_bias(p.lr[net], step_t);
            }
        } else {
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int b = lane; b < p.r.nblocks; b += 32)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[i] += __ldcg(p.r.stats_part + ((size_t)b * 3 + net) * 8 + i);
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i] = warp_sum(acc[i]);
            if (lane == 0) {
                p.r.adam_step[net] = step_t;                   // every CTA read it before the grid barrier
                fold_train_stats(p.r.train_stats + net * 8, acc, net != 0, p.r.critic_norm_coef, &t2);
            }
        }
    }
}

__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// P2P = false: one rank.  P2P = true: several ranks, averaged through the P2PExchange between clip and Adam.
template <bool P2P>
__global__ void __launch_bounds__(OT) optim_fused_kernel(OptArgs<P2P> p) {
    namespace cg = cooperative_groups;
    if (p.r.stop_flag && *p.r.stop_flag) return;          // uniform across the grid and across ranks
    const int net = blockIdx.y;
    const bool active = ((p.r.net_mask >> net) & 1) != 0;
    __shared__ float red[OT / 32], red2[OT / 32];
    __shared__ float s_scale;
    __shared__ AdamBias s_bias;
    const NetLayout L = net_layout(net, p.r.O, p.r.A);
    const int noff = net_offset(net, p.r.O, p.r.A);
    const int pl = blockIdx.x * OT + threadIdx.x;
    const int q = noff + pl;
    float g = 0.f, th = 0.f;
    int step_t = 0;
    if (active) {
        step_t = p.r.adam_step[net] + 1;                   // read before the grid barrier, bumped after it
        if (pl < L.size) {
            g = reduce_partials16(p.r.gpart, p.r.nblocks, p.r.P, q);
            th = p.r.theta[q];
            if (net != 0 && p.r.critic_norm_coef > 0.f) g += 2.f * p.r.critic_norm_coef * th;
        }
        float s = warp_sum(g * g), s2 = warp_sum(net != 0 ? th * th : 0.f);
        if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = s; red2[threadIdx.x >> 5] = s2; }
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f, t2 = 0.f;
            for (int w = 0; w < OT / 32; ++w) { t += red[w]; t2 += red2[w]; }
            p.r.sumsq_part[net * gridDim.x + blockIdx.x] = t;
            p.r.sumsq_part[(3 + net) * gridDim.x + blockIdx.x] = t2;
        }
    }
    cg::this_grid().sync();
    if (active) clip_scale_and_stats(p, net, step_t, &s_scale, &s_bias);
    __syncthreads();
    bool exchange_ok = true;
    if constexpr (P2P) {
        // ---- publish the clipped gradient, exchange flags over NVLink ---------------------------------------
        const P2PExchange& x = p.x;
        const int par = (int)(x.step_id & 1u);
        float* mine = x.peer_buf[x.rank] + (size_t)par * p.r.P;
        if (pl < L.size) mine[q] = active ? g * s_scale : 0.f;
        __threadfence_system();
        cg::this_grid().sync();
        if (blockIdx.x == 0 && blockIdx.y == 0) {
            if ((int)threadIdx.x < x.world)       // tell every peer (and myself) that my buffer for this step is ready
                st_release_sys(x.peer_flag[threadIdx.x] + par * x.world + x.rank, x.step_id);
            if ((int)threadIdx.x < x.world) {     // wait until every peer's buffer for this step is ready
                const unsigned int* f = x.peer_flag[x.rank] + par * x.world + threadIdx.x;
                const long long t0 = clock64();
                while (ld_acquire_sys(f) != x.step_id) {
                    if (clock64() - t0 > 4000000000LL) { *x.error_flag = 1; break; }   // ~2 s: fail instead of hanging
                }
            }
        }
        cg::this_grid().sync();
        // a peer that never published (time-out above) leaves its buffer stale: skip the step instead of applying garbage --
        // the sticky error flag is raised by the host (distributed.p2p_check), the parameters stay those of the last good step
        exchange_ok = *((volatile int*)x.error_flag) == 0;
    }
    if (active && pl < L.size && exchange_ok) {
        if constexpr (P2P) {                     // sum the peers in rank order
            const int par = (int)(p.x.step_id & 1u);
            float sum = 0.f;
            for (int r = 0; r < p.x.world; ++r) {
                const float* pb = p.x.peer_buf[r] + (size_t)par * p.r.P;
                float v;
                asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(pb + q) : "memory");
                sum += v;
            }
            g = sum / (float)p.x.world;
        } else {
            g *= s_scale;
        }
        p.r.grad[q] = g;
        float m = p.m[q], v = p.v[q];
        p.r.theta[q] = adam_update(g, th, m, v, s_bias);
        p.m[q] = m; p.v[q] = v;
    }
}

// lambda <- clamp(Adam(lambda, grad = -(Jc - limit)), 0, upper).  state[4] = {lambda, m, v, t}.
// window_sums[4] = {sum EpRet, sum EpCost, sum EpLen, count} (already all-reduced).
__global__ void lagrange_update_kernel(const double* __restrict__ window_sums, float cost_limit,
                                       float lambda_lr, float upper_bound, float* __restrict__ state,
                                       int* __restrict__ nan_flag) {
    if (threadIdx.x != 0) return;
    const double cnt = window_sums[3];
    if (!(cnt > 0.0)) { *nan_flag = 1; return; }   // reference asserts `Jc` is not NaN (ppo_lag.py:L74)
    const double jc = window_sums[1] / cnt;
    const float g = (float)(-(jc - (double)cost_limit));
    float lam = state[0], m = state[1], v = state[2];
    const int t = (int)state[3] + 1;
    lam = adam_update(g, lam, m, v, adam_bias(lambda_lr, t));
    lam = fmaxf(lam, 0.f);
    if (upper_bound >= 0.f) lam = fminf(lam, upper_bound);
    state[0] = lam; state[1] = m; state[2] = v; state[3] = (float)t;
}

// PID-Lagrangian controller (common/pid_lagrange.py:L95-125), Python-float (fp64) arithmetic.
// pid_state: [0] integral term, [1] EMA of delta, [2] EMA of Jc, [3] cost penalty, [4] deque length,
// [5] deque head (oldest entry), [8 + i] ring buffer of the delayed cost EMAs (capacity d_delay <= 56).
// lagrange_state[0] <- (float) cost penalty = the multiplier the update kernels read.
__global__ void pid_lagrange_kernel(const double* __restrict__ window_sums, double kp, double ki, double kd,
                                    int d_delay, double a_p, double a_d, int sum_norm, int diff_norm,
                                    double penalty_max, double cost_limit, double* __restrict__ st,
                                    float* __restrict__ lagrange_state, int* __restrict__ nan_flag) {
    if (threadIdx.x != 0) return;
    const double cnt = window_sums[3];
    if (!(cnt > 0.0)) { *nan_flag = 1; return; }
    const double jc = window_sums[1] / cnt;
    // separately rounded fp64 operations (no FMA contraction): bit-identical to the Python floats
    const double delta = __dadd_rn(jc, -cost_limit);
    double pid_i = fmax(0.0, __dadd_rn(st[0], __dmul_rn(delta, ki)));
    if (diff_norm) pid_i = fmax(0.0, fmin(1.0, pid_i));
    double delta_p = __dmul_rn(st[1], a_p);
    delta_p = __dadd_rn(delta_p, __dmul_rn(__dadd_rn(1.0, -a_p), delta));
    double cost_d = __dmul_rn(st[2], a_d);
    cost_d = __dadd_rn(cost_d, __dmul_rn(__dadd_rn(1.0, -a_d), jc));
    int n = (int)st[4], head = (int)st[5];
    const double oldest = st[8 + head];
    const double pid_d = fmax(0.0, __dadd_rn(cost_d, -oldest));
    const double pid_o = __dadd_rn(__dadd_rn(__dmul_rn(kp, delta_p), pid_i), __dmul_rn(kd, pid_d));
    double pen = fmax(0.0, pid_o);
    if (diff_norm) pen = fmin(1.0, pen);
    if (!(diff_norm || sum_norm)) pen = fmin(pen, penalty_max);
    if (n < d_delay) { st[8 + (head + n) % d_delay] = cost_d; ++n; }
    else { st[8 + head] = cost_d; head = (head + 1) % d_delay; }
    st[0] = pid_i; st[1] = delta_p; st[2] = cost_d; st[3] = pen; st[4] = (double)n; st[5] = (double)head;
    lagrange_state[0] = (float)pen;
}

// KL early stop: eval_out[0] = sum KL (over samples and action dims), eval_out[4] = sample count.
// kl_state[4] = {last kl, iterations executed, stopped flag as float, 0}.  The reference compares the fp32 KL with a Python
// float (`kl.item() > target_kl`, policy_gradient.py:L395), so the test is done in double against the double target: a
// float target would round e.g. 0.1 up to 0.100000001 and miss a KL of exactly that float.
__global__ void kl_check_kernel(const double* __restrict__ eval_out, double target_kl, int early_stop,
                                int* __restrict__ stop_flag, float* __restrict__ kl_state) {
    if (threadIdx.x != 0) return;
    if (*stop_flag) return;
    const float kl = (float)(eval_out[0] / eval_out[4]);
    kl_state[0] = kl;
    kl_state[1] += 1.f;
    if (early_stop && (double)kl > target_kl) { *stop_flag = 1; kl_state[2] = 1.f; }
}

// out[q] = scale * sum_b gpart[b][q] + add_scale * add[q]
__global__ void __launch_bounds__(OT) reduce_partials_kernel(const float* __restrict__ gpart, int nblocks,
                                                             int stride, int n, float scale,
                                                             const float* __restrict__ add,
                                                             float add_scale, float* __restrict__ out) {
    const int q = blockIdx.x * OT + threadIdx.x;
    if (q >= n) return;
    float g = 0.f;
    for (int b = 0; b < nblocks; ++b) g += gpart[(size_t)b * stride + q];
    g *= scale;
    if (add) g += add_scale * add[q];
    out[q] = g;
}

// ---- conjugate gradient (utils/math.py:L86-132); single CTA of 1024 threads ---------------------
__device__ double block_dot(const float* a, const float* b, int n, double* sred) {
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s += (double)a[i] * (double)b[i];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = s;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sred[w];
    __syncthreads();
    return t;
}

// cg_scalars[4] = {rdotr, done flag, iterations run, 0}
__global__ void __launch_bounds__(1024) cg_init_kernel(const float* __restrict__ b, int n, float* x,
                                                       float* r, float* pv, float* cg_scalars) {
    __shared__ double sred[32];
    for (int i = threadIdx.x; i < n; i += blockDim.x) { x[i] = 0.f; r[i] = b[i]; pv[i] = b[i]; }
    __syncthreads();
    const double rr = block_dot(r, r, n, sred);
    if (threadIdx.x == 0) { cg_scalars[0] = (float)rr; cg_scalars[1] = 0.f; cg_scalars[2] = 0.f; cg_scalars[3] = 0.f; }
}

__global__ void __launch_bounds__(1024) cg_step_kernel(const float* __restrict__ z, int n, float* x,
                                                       float* r, float* pv, float* cg_scalars,
                                                       float residual_tol, float eps) {
    __shared__ double sred[32];
    if (cg_scalars[1] != 0.f) return;   // converged earlier (uniform)
    const float rdotr = cg_scalars[0];
    const float pz = (float)block_dot(pv, z, n, sred);
    const float alpha = rdotr / (pz + eps);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        x[i] += alpha * pv[i];
        r[i] -= alpha * z[i];
    }
    __syncthreads();
    const float new_rdotr = (float)block_dot(r, r, n, sred);
    const bool done = sqrtf(new_rdotr) < residual_tol;
    if (!done) {
        const float mu = new_rdotr / (rdotr + eps);
        for (int i = threadIdx.x; i < n; i += blockDim.x) pv[i] = r[i] + mu * pv[i];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        cg_scalars[2] += 1.f;
        if (done) cg_scalars[1] = 1.f; else cg_scalars[0] = new_rdotr;
    }
}

__global__ void __launch_bounds__(1024) dot_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                   int n, float* __restrict__ out) {
    __shared__ double sred[32];
    const double d = block_dot(a, b, n, sred);
    if (threadIdx.x == 0) out[0] = (float)d;
}

// out = y + alpha * x
__global__ void axpy_kernel(const float* __restrict__ x, const float* __restrict__ y, float alpha, int n,
                            float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = y[i] + alpha * x[i];
}

}  // namespace osb

using namespace osb;

// Arguments of the partial reduction, shared by grad_reduce_kernel and optim_fused_kernel
static ReduceArgs reduce_args(const float* gpart, const float* stats_part, int nblocks, int O, int A, const float* theta,
                              float* grad, float critic_norm_coef, int net_mask, float* sumsq_part, int* adam_step,
                              float* train_stats, const int* stop_flag) {
    return {gpart, stats_part, nblocks, actor_layout(O, A).size + 2 * critic_layout(O, A).size, O, A,
            const_cast<float*>(theta), grad, critic_norm_coef, net_mask, sumsq_part, adam_step, train_stats, stop_flag};
}

// osb_optim_fused (x == NULL) and osb_optim_fused_p2p (x = the peer-memory exchange between the ranks)
static int optim_fused(const float* gpart, const float* stats_part, int nblocks, int O, int A, float* theta, float* grad,
                       float* adam_m, float* adam_v, int* adam_step, float critic_norm_coef, float max_grad_norm,
                       float lr_actor, float lr_critic_r, float lr_critic_c, int net_mask, float* sumsq_part,
                       float* train_stats, const int* stop_flag, const P2PExchange* x, void* stream) {
    OSB_CHECK_ARG(gpart && stats_part && theta && grad && adam_m && adam_v && adam_step && sumsq_part && train_stats, "null pointer");
    OSB_CHECK_ARG(!x || (x->peer_buf && x->peer_flag && x->error_flag && x->world > 1 && x->world <= OT && x->rank >= 0 &&
                         x->rank < x->world), "bad p2p argument");
    P2POptArgs a = {{reduce_args(gpart, stats_part, nblocks, O, A, theta, grad, critic_norm_coef, net_mask, sumsq_part,
                                 adam_step, train_stats, stop_flag),
                     adam_m, adam_v, max_grad_norm, {lr_actor, lr_critic_r, lr_critic_c}},
                    x ? *x : P2PExchange{}};
    void* args[] = {x ? (void*)&a : (void*)static_cast<FusedOptArgs*>(&a)};   // one rank: the base part only
    osb_count_launch();
    OSB_CUDA(cudaLaunchCooperativeKernel(x ? (void*)optim_fused_kernel<true> : (void*)optim_fused_kernel<false>,
                                         dim3(osb_optim_blocks(O, A), 3), dim3(OT), args, 0, (cudaStream_t)stream));
    return OSB_OK;
}

extern "C" {

int osb_optim_blocks(int O, int A) {
    const int sa = actor_layout(O, A).size, sc = critic_layout(O, A).size;
    const int mx = sa > sc ? sa : sc;
    return (mx + OT - 1) / OT;
}

// grad <- sum of the CTA partials (+ 2*coef*theta for the critics); advances adam_step[net] and the
// running training statistics.  sumsq_part: 6 * osb_optim_blocks floats.
int osb_grad_reduce(const float* gpart, const float* stats_part, int nblocks, int O, int A,
                    const float* theta, float* grad, float critic_norm_coef, int net_mask,
                    float* sumsq_part, int* adam_step, float* train_stats, const int* stop_flag,
                    void* stream) {
    OSB_CHECK_ARG(gpart && stats_part && theta && grad && sumsq_part && adam_step && train_stats, "null pointer");
    const ReduceArgs p = reduce_args(gpart, stats_part, nblocks, O, A, theta, grad, critic_norm_coef, net_mask, sumsq_part,
                                     adam_step, train_stats, stop_flag);
    grad_reduce_kernel<<<dim3(osb_optim_blocks(O, A), 3), OT, 0, (cudaStream_t)stream>>>(p);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

// Per-network clip_grad_norm_ (do_clip) and/or Adam step (do_adam).  Multi-rank order of the
// reference: clip locally -> average across ranks (grad_scale = 1/world after the all-reduce SUM) ->
// optimizer step (policy_gradient.py:L437-443).
int osb_clip_adam(float* grad, float* theta, float* adam_m, float* adam_v, const int* adam_step,
                  const float* sumsq_part, int O, int A, float max_grad_norm, float lr_actor,
                  float lr_critic_r, float lr_critic_c, float grad_scale, float critic_norm_coef,
                  float* train_stats, int do_clip, int do_adam, int net_mask, const int* stop_flag,
                  void* stream) {
    OSB_CHECK_ARG(grad && theta && adam_m && adam_v && adam_step && sumsq_part && train_stats, "null pointer");
    AdamArgs p;
    p.critic_norm_coef = critic_norm_coef; p.train_stats = train_stats;
    p.grad = grad; p.theta = theta; p.m = adam_m; p.v = adam_v; p.adam_step = adam_step;
    p.sumsq_part = sumsq_part; p.NB = osb_optim_blocks(O, A); p.O = O; p.A = A;
    p.max_grad_norm = max_grad_norm; p.lr[0] = lr_actor; p.lr[1] = lr_critic_r; p.lr[2] = lr_critic_c;
    p.grad_scale = grad_scale; p.do_clip = do_clip; p.do_adam = do_adam; p.net_mask = net_mask;
    p.stop_flag = stop_flag;
    clip_adam_kernel<<<dim3(p.NB, 3), OT, 0, (cudaStream_t)stream>>>(p);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

// grad_reduce + clip + Adam fused in one cooperative launch (single-rank path).
int osb_optim_fused(const float* gpart, const float* stats_part, int nblocks, int O, int A,
                    float* theta, float* grad, float* adam_m, float* adam_v, int* adam_step,
                    float critic_norm_coef, float max_grad_norm, float lr_actor, float lr_critic_r,
                    float lr_critic_c, int net_mask, float* sumsq_part, float* train_stats,
                    const int* stop_flag, void* stream) {
    return optim_fused(gpart, stats_part, nblocks, O, A, theta, grad, adam_m, adam_v, adam_step, critic_norm_coef,
                       max_grad_norm, lr_actor, lr_critic_r, lr_critic_c, net_mask, sumsq_part, train_stats, stop_flag,
                       nullptr, stream);
}

// ---- NVLink peer-memory exchange buffers (cudaIpc) -----------------------------------------------------
int osb_p2p_alloc(long long bytes, void** ptr, unsigned char* handle64) {
    OSB_CHECK_ARG(bytes > 0 && ptr && handle64, "bad argument");
    void* d = nullptr;
    OSB_CUDA(cudaMalloc(&d, (size_t)bytes));
    OSB_CUDA(cudaMemset(d, 0, (size_t)bytes));
    cudaIpcMemHandle_t h;
    OSB_CUDA(cudaIpcGetMemHandle(&h, d));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle64, &h, 64);
    *ptr = d;
    return OSB_OK;
}

int osb_p2p_open(const unsigned char* handle64, void** ptr) {
    OSB_CHECK_ARG(handle64 && ptr, "bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void* d = nullptr;
    OSB_CUDA(cudaIpcOpenMemHandle(&d, h, cudaIpcMemLazyEnablePeerAccess));
    *ptr = d;
    return OSB_OK;
}

// grad_reduce + clip + one-shot NVLink all-reduce + Adam in one cooperative launch (multi-rank path).
// peer_buf / peer_flag: DEVICE arrays of `world` pointers (own entry = own allocation).
int osb_optim_fused_p2p(const float* gpart, const float* stats_part, int nblocks, int O, int A,
                        float* theta, float* grad, float* adam_m, float* adam_v, int* adam_step,
                        float critic_norm_coef, float max_grad_norm, float lr_actor,
                        float lr_critic_r, float lr_critic_c, int net_mask, float* sumsq_part,
                        float* train_stats, const int* stop_flag, void* peer_buf, void* peer_flag,
                        int world, int rank, unsigned step_id, int* error_flag, void* stream) {
    const P2PExchange x = {(float* const*)peer_buf, (unsigned int* const*)peer_flag, world, rank, step_id, error_flag};
    return optim_fused(gpart, stats_part, nblocks, O, A, theta, grad, adam_m, adam_v, adam_step, critic_norm_coef,
                       max_grad_norm, lr_actor, lr_critic_r, lr_critic_c, net_mask, sumsq_part, train_stats, stop_flag,
                       &x, stream);
}

int osb_lagrange_update(const double* window_sums, float cost_limit, float lambda_lr,
                        float upper_bound, float* state, int* nan_flag, void* stream) {
    OSB_CHECK_ARG(window_sums && state && nan_flag, "null pointer");
    lagrange_update_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(window_sums, cost_limit, lambda_lr, upper_bound, state, nan_flag);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

int osb_pid_lagrange_update(const double* window_sums, double pid_kp, double pid_ki, double pid_kd,
                            int pid_d_delay, double pid_delta_p_ema_alpha, double pid_delta_d_ema_alpha,
                            int sum_norm, int diff_norm, double penalty_max, double cost_limit,
                            double* pid_state, float* lagrange_state, int* nan_flag, void* stream) {
    OSB_CHECK_ARG(window_sums && pid_state && lagrange_state && nan_flag, "null pointer");
    OSB_CHECK_ARG(pid_d_delay >= 1 && pid_d_delay <= 56, "pid_d_delay must be in [1, 56]");
    pid_lagrange_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(window_sums, pid_kp, pid_ki, pid_kd, pid_d_delay,
                                                           pid_delta_p_ema_alpha, pid_delta_d_ema_alpha, sum_norm,
                                                           diff_norm, penalty_max, cost_limit, pid_state,
                                                           lagrange_state, nan_flag);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

int osb_kl_check(const double* eval_out, double target_kl, int early_stop, int* stop_flag,
                 float* kl_state, void* stream) {
    OSB_CHECK_ARG(eval_out && stop_flag && kl_state, "null pointer");
    kl_check_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(eval_out, target_kl, early_stop, stop_flag, kl_state);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

int osb_reduce_partials(const float* gpart, int nblocks, int stride, int n, float scale,
                        const float* add, float add_scale, float* out, void* stream) {
    OSB_CHECK_ARG(gpart && out && n > 0 && nblocks > 0 && stride >= n, "bad argument");
    reduce_partials_kernel<<<(n + OT - 1) / OT, OT, 0, (cudaStream_t)stream>>>(gpart, nblocks, stride, n, scale, add, add_scale, out);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

int osb_cg_init(const float* b, int n, float* x, float* r, float* p, float* cg_scalars, void* stream) {
    OSB_CHECK_ARG(b && x && r && p && cg_scalars && n > 0, "bad argument");
    cg_init_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(b, n, x, r, p, cg_scalars);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

int osb_cg_step(const float* z, int n, float* x, float* r, float* p, float* cg_scalars,
                float residual_tol, float eps, void* stream) {
    OSB_CHECK_ARG(z && x && r && p && cg_scalars && n > 0, "bad argument");
    cg_step_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(z, n, x, r, p, cg_scalars, residual_tol, eps);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

int osb_dot(const float* a, const float* b, int n, float* out, void* stream) {
    OSB_CHECK_ARG(a && b && out && n > 0, "bad argument");
    dot_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(a, b, n, out);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

int osb_axpy(const float* x, const float* y, float alpha, int n, float* out, void* stream) {
    OSB_CHECK_ARG(x && y && out && n > 0, "bad argument");
    axpy_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(x, y, alpha, n, out);
    OSB_LAUNCH_CHECK();
    return OSB_OK;
}

}  // extern "C"
