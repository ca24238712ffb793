// Arithmetic of one optimiser step -- clip_grad_norm_, torch.optim.Adam and the logged loss statistics -- shared by
// the split (grad_reduce + clip_adam), fused and persistent bf16x3 update paths and the Lagrange multiplier update.
// Each path keeps its own reduction order; only the per-value arithmetic lives here, so every path rounds alike.
#pragma once
#include "common.cuh"

namespace osb {

// torch.optim.Adam bias corrections of step t (betas 0.9 / 0.999), computed in fp64 like torch's Python floats
struct AdamBias {
    float step_size;   // lr / (1 - 0.9^t)
    float bc2_sqrt;    // sqrt(1 - 0.999^t)
};
__device__ __forceinline__ AdamBias adam_bias(float lr, int t) {
    const double bc1 = 1.0 - pow(0.9, (double)t), bc2 = 1.0 - pow(0.999, (double)t);
    return {(float)((double)lr / bc1), (float)sqrt(bc2)};
}

// One torch.optim.Adam step of one parameter (single-tensor path, eps 1e-8, no weight decay) in torch's rounding
// order: updates the moments m, v and returns the new parameter.
__device__ __forceinline__ float adam_update(float g, float th, float& m, float& v, AdamBias b) {
    m = __fadd_rn(m, __fmul_rn(0.1f, __fadd_rn(g, -m)));                       // exp_avg.lerp_(grad, 1 - beta1)
    v = __fadd_rn(__fmul_rn(v, 0.999f), __fmul_rn(__fmul_rn(0.001f, g), g));   // exp_avg_sq.mul_(beta2).addcmul_(g, g, 1 - beta2)
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(v), b.bc2_sqrt), 1e-8f);
    return __fadd_rn(th, __fmul_rn(-b.step_size, __fdiv_rn(m, denom)));
}

// clip_grad_norm_ scale of one network from its squared gradient norm; max_norm <= 0 turns clipping off
__device__ __forceinline__ float clip_coef(float max_norm, float sumsq) {
    return (max_norm > 0.f) ? fminf(max_norm / (sqrtf(sumsq) + 1e-6f), 1.0f) : 1.0f;
}

// Adds one minibatch to a network's running statistics ts[0..3] = {mean loss, mean ratio, mean kl, #minibatches}.
// acc = {sum loss, sum ratio, sum kl, sample count}.  A critic's logged loss also carries the regulariser
// coef * sum(theta^2) (policy_gradient.py:L429-433), added to the loss mean in the same accumulation; *sum_th2 is
// read only for a critic.
__device__ __forceinline__ void fold_train_stats(float* ts, const float* acc, bool critic, float coef, const float* sum_th2) {
    const float inv = acc[3] > 0.f ? 1.f / acc[3] : 0.f;
    ts[0] += acc[0] * inv + (critic ? coef * *sum_th2 : 0.f);
    ts[1] += acc[1] * inv;
    ts[2] += acc[2] * inv;
    ts[3] += 1.f;
}

}  // namespace osb
