"""Oracle: the optimiser step shared by every update path -- partial-gradient reduction, critic L2 term,
per-network clip_grad_norm_ and one torch-Adam step -- restated for the kernel tests.  TEST INFRASTRUCTURE ONLY.

Two references:
  adam_f32       torch.optim.Adam, single-tensor path (betas 0.9 / 0.999, eps 1e-8, no weight decay), in numpy
                 float32 with the kernels' operation order: every operation is rounded once, so given the same state and
                 gradient the first and second moments are reproduced bit for bit.
  grad_check     fp64 sum of the per-CTA partial gradients (+ 2 coef theta for the critics), the per-network norm and
                 clip coefficient min(max / (|g| + 1e-6), 1), and the bars a float32 kernel result is held to.
"""
from __future__ import annotations

import math

import numpy as np

F = np.float32
U = 2.0 ** -24          # unit roundoff of float32


def adam_f32(theta, m, v, g, t: int, lr: float):
    """One Adam step at step count t (>= 1, the count after this step) with learning rate lr (a float32 value):
        m' = m + 0.1f (g + (-m))                         exp_avg.lerp_(grad, 1 - beta1)
        v' = v 0.999f + (0.001f g) g                     exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
        denom = sqrt(v') / f32(sqrt(bc2)) + 1e-8f
        theta' = theta + (-f32(lr / bc1)) (m' / denom)
    bc1 = 1 - 0.9^t and bc2 = 1 - 0.999^t in fp64.  Returns float32 (theta', m', v')."""
    theta, m, v, g = (np.asarray(x, F) for x in (theta, m, v, g))
    bc1 = 1.0 - 0.9 ** t
    bc2 = 1.0 - 0.999 ** t
    step = F(float(F(lr)) / bc1)
    bc2_sqrt = F(math.sqrt(bc2))
    m1 = m + F(0.1) * (g + (-m))
    v1 = v * F(0.999) + (F(0.001) * g) * g
    denom = np.sqrt(v1) / bc2_sqrt + F(1e-8)
    th1 = theta + (-step) * (m1 / denom)
    return th1.astype(F), m1.astype(F), v1.astype(F)


def ulp_diff(a, b) -> np.ndarray:
    """Distance in float32 units in the last place (+0 and -0 are the same point)."""
    def key(x):
        i = np.asarray(x, F).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(key(a) - key(b))


def clip_coef64(norm: float, max_grad_norm: float) -> float:
    """clip_grad_norm_'s coefficient in fp64 (no clipping for max_grad_norm <= 0)."""
    return min(max_grad_norm / (norm + 1e-6), 1.0) if max_grad_norm > 0 else 1.0


def check_grad(got, g64, bound, max_grad_norm: float, what: str = '', l2_raw: float = 1e-6,
               l2_clip: float = 1e-5) -> float:
    """Stored (clipped) float32 gradient of ONE network against the fp64 reference g64.

    bound: elementwise summation bound of the unclipped gradient (n_terms * 2^-24 * sum of |terms|).
    - unclipped (coef64 == 1): |got - g64| <= bound elementwise and l2-relative <= l2_raw;
    - clipped: l2-relative <= l2_clip against coef64 * g64, and got / g64 is ONE scalar c for the whole network:
      |got - c g64| <= 2 c bound + 2^-23 |got| elementwise, where c is the least-squares ratio and |c / coef64 - 1| <= l2_clip.
    A norm within 1e-5 of max_grad_norm may go either way, but only as one coefficient over the network (the elementwise
    bar against the single c).  Returns c."""
    got = np.asarray(got, np.float64)
    g64 = np.asarray(g64, np.float64)
    norm = float(np.linalg.norm(g64))
    coef = clip_coef64(norm, max_grad_norm)
    near = max_grad_norm > 0 and abs(norm - max_grad_norm) <= 1e-5 * max_grad_norm
    if norm == 0.0:
        assert np.all(got == 0.0), f'{what}: zero gradient expected'
        return 1.0
    want = coef * g64
    rel = float(np.linalg.norm(got - want) / np.linalg.norm(want))
    c = float((got * g64).sum() / (g64 * g64).sum())
    if coef == 1.0 and not near:
        assert rel <= l2_raw, f'{what}: gradient l2-relative error {rel:.2e} > {l2_raw:.0e}'
        excess = np.abs(got - g64) - bound
        assert excess.max() <= 0.0, (f'{what}: {int((excess > 0).sum())} elements outside the summation bound, worst '
                                     f'|err| {np.abs(got - g64)[excess.argmax()]:.3e} > {bound[excess.argmax()]:.3e}')
    else:
        assert rel <= l2_clip, f'{what}: clipped gradient l2-relative error {rel:.2e} > {l2_clip:.0e} (coef64 {coef:.6f})'
        assert abs(c / coef - 1.0) <= l2_clip or (near and abs(c - 1.0) <= l2_clip), (what, c, coef)
        excess = np.abs(got - c * g64) - (2 * c * bound + 2 * U * np.abs(got))
        assert excess.max() <= 0.0, (f'{what}: the clipped gradient is not one coefficient times the gradient on '
                                     f'{int((excess > 0).sum())} elements (c = {c:.7f})')
    return c


def check_adam(pre, post, g, t: int, lr: float, what: str = '', theta_ulp: int = 1) -> None:
    """post = (theta', m', v') of a kernel against adam_f32(pre, g): moments bit for bit, theta' to theta_ulp ulp."""
    th1, m1, v1 = adam_f32(*pre, g, t, lr)
    for name, got, want, tol in (('m', post[1], m1, 0), ('v', post[2], v1, 0), ('theta', post[0], th1, theta_ulp)):
        d = ulp_diff(got, want)
        assert d.max() <= tol, (f'{what}: Adam {name} differs from the fp32 restatement by up to {int(d.max())} ulp on '
                                f'{int((d > tol).sum())} elements (step {t}, lr {lr})')
