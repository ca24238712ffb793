// Host-side (C++) epoch drivers: the whole minibatch update loop of one epoch is issued from one
// C-ABI call so that no Python sits between the ~800 kernel launches, plus a thin dlopen binding of
// NCCL for the per-step flat gradient all-reduce (utils/distributed.py:L142-228 avg_grads/dist_avg).
#include "common.cuh"
#include "mlp.cuh"
#include <dlfcn.h>
#include <stdlib.h>
#include <string.h>

// ---- NCCL through dlopen (the library torch already loaded; no link-time dependency) ----------
namespace {
typedef struct { char internal[128]; } nccl_uid_t;
typedef int (*fn_get_uid)(nccl_uid_t*);
typedef int (*fn_init_rank)(void**, int, nccl_uid_t, int);
typedef int (*fn_allreduce)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*fn_destroy)(void*);
typedef const char* (*fn_errstr)(int);
struct NcclApi {
    void* handle = nullptr;
    fn_get_uid get_uid = nullptr;
    fn_init_rank init_rank = nullptr;
    fn_allreduce allreduce = nullptr;
    fn_destroy destroy = nullptr;
    fn_errstr errstr = nullptr;
} g_nccl;

int nccl_load(const char* libpath) {
    if (g_nccl.handle) return OSB_OK;
    void* h = dlopen(libpath, RTLD_NOW | RTLD_GLOBAL);
    if (!h) { osb_set_error(dlerror()); return OSB_ERR_UNSUPPORTED; }
    g_nccl.get_uid = (fn_get_uid)dlsym(h, "ncclGetUniqueId");
    g_nccl.init_rank = (fn_init_rank)dlsym(h, "ncclCommInitRank");
    g_nccl.allreduce = (fn_allreduce)dlsym(h, "ncclAllReduce");
    g_nccl.destroy = (fn_destroy)dlsym(h, "ncclCommDestroy");
    g_nccl.errstr = (fn_errstr)dlsym(h, "ncclGetErrorString");
    if (!g_nccl.get_uid || !g_nccl.init_rank || !g_nccl.allreduce || !g_nccl.destroy) {
        osb_set_error("libnccl is missing a required symbol");
        return OSB_ERR_UNSUPPORTED;
    }
    g_nccl.handle = h;
    return OSB_OK;
}
int nccl_check(int rc, const char* what) {
    if (rc == 0) return OSB_OK;
    char buf[256];
    snprintf(buf, sizeof(buf), "%s failed: %s", what, g_nccl.errstr ? g_nccl.errstr(rc) : "nccl error");
    osb_set_error(buf);
    return OSB_ERR_CUDA;
}
}  // namespace

extern "C" {

int osb_nccl_unique_id(const char* libpath, unsigned char* id128) {
    OSB_CHECK_ARG(libpath && id128, "null pointer");
    int rc = nccl_load(libpath);
    if (rc) return rc;
    nccl_uid_t uid;
    rc = nccl_check(g_nccl.get_uid(&uid), "ncclGetUniqueId");
    if (rc) return rc;
    memcpy(id128, uid.internal, 128);
    return OSB_OK;
}

int osb_nccl_init(const char* libpath, const unsigned char* id128, int nranks, int rank,
                  void** comm_out) {
    OSB_CHECK_ARG(libpath && id128 && comm_out && nranks > 0 && rank >= 0 && rank < nranks, "bad argument");
    int rc = nccl_load(libpath);
    if (rc) return rc;
    nccl_uid_t uid;
    memcpy(uid.internal, id128, 128);
    void* comm = nullptr;
    rc = nccl_check(g_nccl.init_rank(&comm, nranks, uid, rank), "ncclCommInitRank");
    if (rc) return rc;
    *comm_out = comm;
    return OSB_OK;
}

int osb_nccl_allreduce(void* comm, void* buf, long long count, int is_f64, void* stream) {
    OSB_CHECK_ARG(comm && buf && count > 0 && g_nccl.handle, "bad argument / nccl not initialised");
    return nccl_check(g_nccl.allreduce(buf, buf, (size_t)count, is_f64 ? 8 : 7, 0, comm, (cudaStream_t)stream),
                      "ncclAllReduce");
}

int osb_nccl_destroy(void* comm) {
    if (comm && g_nccl.handle) return nccl_check(g_nccl.destroy(comm), "ncclCommDestroy");
    return OSB_OK;
}

// ---- one epoch of PolicyGradient._update (policy_gradient.py:L345-405) -----------------------
// net_mask: bit0 actor, bit1 reward critic, bit2 cost critic (NaturalPG-style critic-only passes use
// 6).  perm = [update_iters][total] slab rows (parity mode: the reference DataLoader order) or NULL
// (in-kernel Feistel permutation keyed by perm_seed + iteration).  When the actor is trained the old
// policy is snapshotted first (mu_old, logstd_old) and after every pass the full-batch KL is
// evaluated; with kl_early_stop the device-side stop flag turns the remaining launches into no-ops.
// comm != NULL: world_size ranks; gradients are clipped locally, summed with one flat NCCL
// all-reduce per minibatch step and divided by world_size before Adam (policy_gradient.py:L437-443).
int osb_ppo_update_epoch(float* theta, float* grad, float* adam_m, float* adam_v, int* adam_step,
                         int O, int A, const float* obs, const float* act, const float* logp,
                         const float* adv_r, const float* adv_c, const float* tv_r,
                         const float* tv_c, float* mu_old, float* logstd_old, const float* moments,
                         const int* perm, long long total, unsigned perm_seed, int batch_size,
                         int update_iters, int loss_kind, float clip, float entropy_coef,
                         float focops_lam, float focops_eta, const float* lagrange, int net_mask,
                         float critic_norm_coef, float max_grad_norm, float lr_actor,
                         float lr_critic, double target_kl, int kl_early_stop, float* gpart,
                         float* stats_part, float* sumsq_part, float* train_stats, double* eval_ws,
                         double* eval_out, int* stop_flag, float* kl_state, int precision,
                         void* comm, int world_size, void* peer_buf, void* peer_flag, int rank,
                         int* p2p_error, void* stream) {
    OSB_CHECK_ARG(theta && grad && adam_m && adam_v && adam_step && obs && moments, "null pointer");
    OSB_CHECK_ARG(batch_size > 0 && update_iters >= 0 && total > 0 && world_size >= 1, "bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    const int P = osb::actor_layout(O, A).size + 2 * osb::critic_layout(O, A).size;
    OSB_CUDA(cudaMemsetAsync(stop_flag, 0, sizeof(int), s));
    OSB_CUDA(cudaMemsetAsync(kl_state, 0, 4 * sizeof(float), s));
    OSB_CUDA(cudaMemsetAsync(train_stats, 0, 3 * 8 * sizeof(float), s));
    int rc;
    // precision 1 = TF32 tcgen05 tiles (O <= 64, loss kinds 0/1/3); otherwise the fp32 FMA parity path
    // precision 2 = split-bf16 ("bf16x3") tcgen05 tiles: fp32-level results on the tensor cores (O <= 64,
    // loss kinds 0/1/3)
    const bool use_x3 = precision == 2 && O <= 64 && (loss_kind == 0 || loss_kind == 1 || loss_kind == 2 || loss_kind == 3 || loss_kind == 5);   // FOCOPS (2), P3O (5): stepwise launches
    const bool use_x3e = precision == 2 && O <= 64;
    const bool use_tc = precision == 1 && O <= 512;
    const bool train_actor = (net_mask & 1) != 0;
    if (train_actor) {
        OSB_CHECK_ARG(mu_old && logstd_old && eval_ws && eval_out, "actor update needs mu_old/logstd_old/eval buffers");
        rc = (use_x3e ? osb_actor_eval_x3 : use_tc ? osb_actor_eval_tc : osb_actor_eval)(theta, O, A, obs, nullptr, nullptr, nullptr, nullptr,
                                                          nullptr, nullptr, nullptr, nullptr, total, 1, mu_old,
                                                          nullptr, nullptr, stream);
        if (rc) return rc;
        OSB_CUDA(cudaMemcpyAsync(logstd_old, theta, A * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    const float gscale = 1.0f / (float)world_size;
    // bf16x3 + (one rank | NVLink peer exchange): the whole iteration is one persistent kernel with the optimiser inside
    const bool p2p_ok = world_size > 1 && peer_buf && peer_flag && p2p_error;
    const bool fuse_x3 = use_x3 && loss_kind != 2 && loss_kind != 5 && (world_size == 1 || p2p_ok) && !getenv("OSB_X3_NO_FUSE");
    for (int it = 0; it < update_iters; ++it) {
        const int* perm_it = perm ? perm + (size_t)it * total : nullptr;
        if (fuse_x3) {
            rc = osb_ppo_update_iter_x3(theta, grad, adam_m, adam_v, adam_step, O, A, obs, act, logp, adv_r, adv_c, tv_r,
                                        tv_c, moments, perm_it, total, perm_seed + 0x9E3779B9u * (unsigned)it, batch_size,
                                        loss_kind, clip, entropy_coef, lagrange, net_mask, critic_norm_coef, max_grad_norm,
                                        lr_actor, lr_critic, lr_critic, gpart, stats_part, train_stats, stop_flag,
                                        world_size > 1 ? peer_buf : nullptr, world_size > 1 ? peer_flag : nullptr, world_size,
                                        rank, p2p_error, stream);
            if (rc) return rc;
        }
        for (long long start = 0; start < total && !fuse_x3; start += batch_size) {
            const int count = (int)((total - start < batch_size) ? (total - start) : batch_size);
            rc = (use_x3 ? osb_minibatch_grad_x3 : use_tc ? osb_minibatch_grad_tc : osb_minibatch_grad)(
                theta, O, A, obs, act, logp, adv_r, adv_c, tv_r, tv_c, mu_old, moments, perm_it, total,
                perm_seed + 0x9E3779B9u * (unsigned)it, start, count, loss_kind, clip, entropy_coef,
                focops_lam, focops_eta, lagrange, logstd_old, net_mask, gpart, stats_part, stop_flag, stream);
            if (rc) return rc;
            const int nb = (use_tc || use_x3) ? osb_tc_grid_blocks(count, net_mask) : osb_update_grid_blocks(count);
            if (world_size > 1 && peer_buf && peer_flag && p2p_error) {
                // one cooperative kernel: reduce + clip + one-shot NVLink peer-memory all-reduce + Adam
                static unsigned p2p_step = 0;
                rc = osb_optim_fused_p2p(gpart, stats_part, nb, O, A, theta, grad,
                                         adam_m, adam_v, adam_step, critic_norm_coef, max_grad_norm, lr_actor,
                                         lr_critic, lr_critic, net_mask, sumsq_part, train_stats, stop_flag,
                                         peer_buf, peer_flag, world_size, rank, ++p2p_step, p2p_error, stream);
            } else if (!(comm && world_size > 1)) {
                rc = osb_optim_fused(gpart, stats_part, nb, O, A, theta, grad,
                                     adam_m, adam_v, adam_step, critic_norm_coef, max_grad_norm, lr_actor,
                                     lr_critic, lr_critic, net_mask, sumsq_part, train_stats, stop_flag, stream);
            } else {
                rc = osb_grad_reduce(gpart, stats_part, nb, O, A, theta, grad,
                                     critic_norm_coef, net_mask, sumsq_part, adam_step, train_stats,
                                     stop_flag, stream);
                if (rc) return rc;
                rc = osb_clip_adam(grad, theta, adam_m, adam_v, adam_step, sumsq_part, O, A,
                                   max_grad_norm, lr_actor, lr_critic, lr_critic, 1.f, critic_norm_coef, train_stats, 1, 0, net_mask,
                                   stop_flag, stream);
                if (rc) return rc;
                rc = osb_nccl_allreduce(comm, grad, P, 0, stream);
                if (rc) return rc;
                rc = osb_clip_adam(grad, theta, adam_m, adam_v, adam_step, sumsq_part, O, A,
                                   max_grad_norm, lr_actor, lr_critic, lr_critic, gscale, critic_norm_coef, train_stats, 0, 1, net_mask,
                                   stop_flag, stream);
            }
            if (rc) return rc;
        }
        if (train_actor) {
            rc = (use_x3e ? osb_actor_eval_x3 : use_tc ? osb_actor_eval_tc : osb_actor_eval)(theta, O, A, obs, act, logp, adv_r, adv_c, mu_old,
                                                              logstd_old, moments, lagrange, total, 1, nullptr,
                                                              eval_ws, eval_out, stream);
            if (rc) return rc;
            if (comm && world_size > 1) {
                rc = osb_nccl_allreduce(comm, eval_out, 8, 1, stream);
                if (rc) return rc;
            }
            rc = osb_kl_check(eval_out, target_kl, kl_early_stop, stop_flag, kl_state, stream);
            if (rc) return rc;
        }
    }
    return OSB_OK;
}

}  // extern "C"
