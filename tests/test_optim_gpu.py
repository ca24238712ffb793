"""GPU: the optimiser step of every update path against a reference partial reduction + clip_grad_norm_ + torch-Adam
(oracle/optim.py), checked after EVERY step and re-based on the kernel's own state, so that an error cannot hide inside
a whole-epoch tolerance:

  A  osb_optim_fused (one rank) and osb_grad_reduce + osb_clip_adam (the multi-rank order clip -> average -> Adam) on
     synthetic partial gradients whose per-network norms are chosen to clip, not clip and clip by 0.1 %;
  B  the persistent bf16x3 iteration (osb_ppo_update_iter_x3), one minibatch per launch, on each of its optimiser
     branches: speculative Adam before the norm barrier, speculative with a redo after a clip, chunked;
  C  the persistent iteration with several minibatches per launch and clipping that toggles, against the stepwise loop;
  D  the Lagrange multiplier update and the KL early-stop check;
  E  the conjugate-gradient state kernels, dot / axpy and the partial reduction.

Bars: Adam moments bit for bit and parameters to 1 ulp against the fp32 restatement given the kernel's stored gradient;
the stored gradient within the fp32 summation bound of the fp64 sum of the partials (l2-relative 1e-6), 1e-5 once
clipped, and always one clip coefficient per network.
"""
import math

import numpy as np
import pytest
import torch

from oracle import actor_critic as oac
from oracle import learner as ol
from oracle.optim import F, U, adam_f32, check_adam, check_grad, clip_coef64, ulp_diff
from test_update_gpu import _rand_data, _rows, _setup

pytestmark = pytest.mark.gpu

NETS = ol.NETS
COEF = 1e-3                      # critic_norm_coef
LRS = (3e-4, 7e-4, 1.3e-3)       # actor, reward critic, cost critic: all different, so a swapped index fails
NEPI = 512                       # epilogue threads per CTA of the persistent kernel: slices up to this size are speculative


def _lib():
    from omnisafe_b200._lib import current_stream, lib, ptr
    return lib(), ptr, current_stream()


def _sections(O, A):
    lay = oac.layout(O, A)
    return [(lay[n]['start'], lay[n]['size']) for n in NETS]


def _same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.int32), np.asarray(b).view(np.int32))


def _ref_grad(sec, gp, theta_pre, coef):
    """fp64 reference of the reduction: per network (g64, elementwise bound, |g64|).  g64 = sum_b gpart_b (+ 2 coef theta
    for the critics, theta before the step).  Bound: a float32 sum of n terms, in any order, is within (n - 1) 2^-24 sum|terms|
    to first order; n = nblocks + 1 with the regulariser, and the +1 more covers the rounding of 2 coef theta."""
    nb = gp.shape[0]
    th = torch.as_tensor(np.asarray(theta_pre), device=gp.device).double()
    g = gp.double().sum(0)
    ab = gp.double().abs().sum(0)
    out = []
    for k, (s, n) in enumerate(sec):
        gk, ak = g[s:s + n], ab[s:s + n]
        if k and coef > 0:
            reg = 2.0 * float(F(coef)) * th[s:s + n]
            gk, ak = gk + reg, ak + reg.abs()
        g64 = gk.cpu().numpy()
        out.append((g64, ((nb + 1) * U * ak).cpu().numpy(), float(np.linalg.norm(g64))))
    return out


def _check_step(sec, pre, post, ref, mask, max_norm, lrs, what, grad_scale=1.0, stats=None, coef=COEF):
    """One optimiser step of every network: masked-out networks bit-identical; the others against the references."""
    for k, (s, n) in enumerate(sec):
        sl = slice(s, s + n)
        tag = f'{what} {NETS[k]}'
        if not (mask >> k) & 1:
            for key in ('theta', 'm', 'v', 'grad'):
                assert _same_bits(post[key][sl], pre[key][sl]), f'{tag}: masked-out network changed ({key})'
            assert post['step'][k] == pre['step'][k], f'{tag}: masked-out adam_step changed'
            if 'ts' in pre:
                assert _same_bits(post['ts'][8 * k:8 * k + 8], pre['ts'][8 * k:8 * k + 8]), f'{tag}: train_stats changed'
            continue
        t = int(pre['step'][k]) + 1
        assert post['step'][k] == t, f'{tag}: adam_step {post["step"][k]} != {t}'
        g64, bound, _ = ref[k]
        check_grad(post['grad'][sl], g64, bound, max_norm, tag)
        g = post['grad'][sl]
        if grad_scale != 1.0:
            g = (g * F(grad_scale)).astype(F)
        check_adam((pre['theta'][sl], pre['m'][sl], pre['v'][sl]), (post['theta'][sl], post['m'][sl], post['v'][sl]),
                   g, t, lrs[k], tag)
        if stats is not None:        # logger rows: per-minibatch means + coef * sum(theta^2) for the critics, step count
            acc = stats[:, k, :4].astype(np.float64).sum(0)
            want = np.array([acc[0] / acc[3], acc[1] / acc[3], acc[2] / acc[3], 1.0])
            if k and coef > 0:
                want[0] += float(F(coef)) * float((pre['theta'][sl].astype(np.float64) ** 2).sum())
            got = post['ts'][8 * k:8 * k + 4].astype(np.float64) - pre['ts'][8 * k:8 * k + 4]
            # float32 sums over the CTAs (any order) and of theta^2, the running sum itself rounded once more
            tol = (stats.shape[0] + 4) * U * np.abs(stats[:, k, :4]).sum(0) / acc[3] + 4 * U * np.abs(post['ts'][8 * k:8 * k + 4])
            if k and coef > 0:
                tol[0] += n * U * float(F(coef)) * float((pre['theta'][sl].astype(np.float64) ** 2).sum())
            tol += 1e-6 * np.abs(want) + 1e-12
            assert (np.abs(got - want) <= tol).all(), (tag, got, want)


# ================= A. stepwise optimiser kernels on synthetic partials ==================================================
class _Opt:
    """Device state of the stepwise optimiser kernels for one (O, A)."""

    def __init__(self, dev, O, A, seed):
        lib, _, _ = _lib()
        self.dev, self.O, self.A = dev, O, A
        self.sec = _sections(O, A)
        self.P = oac.layout(O, A)['total']
        f32 = dict(dtype=torch.float32, device=dev)
        self.theta = torch.as_tensor(oac.init_theta(O, A, seed=seed)).to(dev)
        self.grad = torch.zeros(self.P, **f32)
        self.m = torch.zeros(self.P, **f32)
        self.v = torch.zeros(self.P, **f32)
        self.step = torch.zeros(4, dtype=torch.int32, device=dev)
        self.NB = lib.osb_optim_blocks(O, A)
        self.sumsq = torch.zeros(6 * self.NB, **f32)
        self.ts = torch.zeros(24, **f32)
        self.stop = torch.zeros(1, dtype=torch.int32, device=dev)

    def snap(self):
        torch.cuda.synchronize()
        return {k: getattr(self, k).cpu().numpy().copy() for k in ('theta', 'grad', 'm', 'v', 'step', 'ts')}

    def partials(self, gen, nblocks, targets, coef=COEF):
        """Random per-CTA partials [nblocks][P], each network scaled so that |sum_b gpart_b + 2 coef theta| = targets[k]
        (0: an all-zero gradient); stats_part [nblocks][3][8] with positive sample counts in slot 3."""
        gp = torch.randn(nblocks, self.P, generator=gen, device=self.dev)
        th = self.theta.double()
        for k, (s, n) in enumerate(self.sec):
            if targets[k] == 0:
                gp[:, s:s + n] = 0.0
                continue
            G = gp[:, s:s + n].double().sum(0)
            r = 2.0 * float(F(coef)) * th[s:s + n] if (k and coef > 0) else torch.zeros_like(G)
            a, b, c = float(G @ G), float(G @ r), float(r @ r) - targets[k] ** 2
            gp[:, s:s + n] *= (-b + math.sqrt(b * b - a * c)) / a
        stats = torch.randn(nblocks, 3, 8, generator=gen, device=self.dev)
        stats[:, :, 3] = torch.floor(64 + 64 * torch.rand(nblocks, 3, generator=gen, device=self.dev))
        return gp.contiguous(), stats.contiguous()

    def fused(self, gp, stats, mask, max_norm, lrs=LRS, coef=COEF):
        lib, ptr, s = _lib()
        lib.osb_optim_fused(ptr(gp), ptr(stats), gp.shape[0], self.O, self.A, ptr(self.theta), ptr(self.grad),
                            ptr(self.m), ptr(self.v), ptr(self.step), coef, max_norm, *lrs, mask, ptr(self.sumsq),
                            ptr(self.ts), ptr(self.stop), s)

    def reduce(self, gp, stats, mask, coef=COEF):
        lib, ptr, s = _lib()
        lib.osb_grad_reduce(ptr(gp), ptr(stats), gp.shape[0], self.O, self.A, ptr(self.theta), ptr(self.grad), coef,
                            mask, ptr(self.sumsq), ptr(self.step), ptr(self.ts), ptr(self.stop), s)

    def clip_adam(self, mask, max_norm, do_clip, do_adam, grad_scale=1.0, lrs=LRS, coef=COEF):
        lib, ptr, s = _lib()
        lib.osb_clip_adam(ptr(self.grad), ptr(self.theta), ptr(self.m), ptr(self.v), ptr(self.step), ptr(self.sumsq),
                          self.O, self.A, max_norm, *lrs, grad_scale, coef, ptr(self.ts), do_clip, do_adam, mask,
                          ptr(self.stop), s)

    def split(self, gp, stats, mask, max_norm, lrs=LRS, coef=COEF):
        """One rank of the multi-rank order: reduce, clip, (all-reduce of one rank = identity), Adam."""
        self.reduce(gp, stats, mask, coef)
        self.clip_adam(mask, max_norm, 1, 0, lrs=lrs, coef=coef)
        self.clip_adam(mask, max_norm, 0, 1, lrs=lrs, coef=coef)

    def kernel_coef(self, k, max_norm):
        """clip_adam's coefficient from the slice norms it reads: fminf(max / (sqrtf(sum_b sumsq_b) + 1e-6f), 1)."""
        tot = F(0)
        for x in self.sumsq.cpu().numpy()[k * self.NB:(k + 1) * self.NB]:
            tot = F(tot + x)
        return F(min(F(F(max_norm) / F(np.sqrt(tot) + F(1e-6))), F(1))) if max_norm > 0 else F(1)


@pytest.mark.parametrize('nblocks', [1, 15, 16, 17, 49, 148])
@pytest.mark.parametrize('O,A', [(60, 8), (17, 6), (64, 16), (376, 8)])
def test_optim_fused_steps(cuda, O, A, nblocks):
    """20 steps of osb_optim_fused with fresh partials: the actor clips by 10x, the reward critic is at 0.1x of the
    threshold and the cost critic at 1.001x; three different learning rates.  (376, 8) is the largest actor on the
    fp32 path (the osb_optim_blocks grid); nblocks covers the 16-wide load groups of the partial reduction."""
    st = _Opt(cuda, O, A, seed=O + nblocks)
    gen = torch.Generator(device=cuda).manual_seed(1000 * O + nblocks)
    for step in range(20):
        gp, stats = st.partials(gen, nblocks, (10.0, 0.1, 1.001))
        pre = st.snap()
        ref = _ref_grad(st.sec, gp, pre['theta'], COEF)
        st.fused(gp, stats, 7, 1.0)
        _check_step(st.sec, pre, st.snap(), ref, 7, 1.0, LRS, f'step {step}', stats=stats.cpu().numpy())


@pytest.mark.parametrize('path', ['fused', 'split'])
def test_optim_large_step_count(cuda, path):
    """Bias correction at large t: a sequence starting from adam_step = 9999 with a non-zero Adam state."""
    st = _Opt(cuda, 60, 8, seed=3)
    gen = torch.Generator(device=cuda).manual_seed(11)
    st.step[:3] = 9999
    st.m.copy_(1e-2 * torch.randn(st.P, generator=gen, device=cuda))
    st.v.copy_(1e-4 * torch.rand(st.P, generator=gen, device=cuda))
    for step in range(5):
        gp, stats = st.partials(gen, 17, (3.0, 0.2, 1.5))
        pre = st.snap()
        ref = _ref_grad(st.sec, gp, pre['theta'], COEF)
        (st.fused if path == 'fused' else st.split)(gp, stats, 7, 1.0)
        _check_step(st.sec, pre, st.snap(), ref, 7, 1.0, LRS, f'{path} t={10000 + step}', stats=stats.cpu().numpy())


@pytest.mark.parametrize('path', ['fused', 'split'])
@pytest.mark.parametrize('mask', [7, 6, 1, 2, 4])
def test_optim_net_mask(cuda, mask, path):
    """Networks outside net_mask keep theta, m, v, grad, adam_step and their train_stats rows bit for bit."""
    st = _Opt(cuda, 60, 8, seed=mask)
    gen = torch.Generator(device=cuda).manual_seed(mask)
    st.grad.copy_(torch.randn(st.P, generator=gen, device=cuda))
    st.m.copy_(1e-2 * torch.randn(st.P, generator=gen, device=cuda))
    st.v.copy_(1e-4 * torch.rand(st.P, generator=gen, device=cuda))
    st.step[:3] = torch.tensor([5, 9, 13], dtype=torch.int32)
    st.ts.copy_(torch.randn(24, generator=gen, device=cuda))
    for step in range(3):
        gp, stats = st.partials(gen, 17, (10.0, 0.1, 1.001))
        pre = st.snap()
        ref = _ref_grad(st.sec, gp, pre['theta'], COEF)
        (st.fused if path == 'fused' else st.split)(gp, stats, mask, 1.0)
        _check_step(st.sec, pre, st.snap(), ref, mask, 1.0, LRS, f'{path} mask {mask} step {step}',
                    stats=stats.cpu().numpy())


def test_optim_stop_flag(cuda):
    """With the early-stop flag raised every optimiser entry point is a no-op, adam_step and train_stats included."""
    st = _Opt(cuda, 60, 8, seed=1)
    gen = torch.Generator(device=cuda).manual_seed(2)
    gp, stats = st.partials(gen, 17, (10.0, 0.1, 1.001))
    st.fused(gp, stats, 7, 1.0)                    # a non-trivial state first
    st.grad.copy_(torch.randn(st.P, generator=gen, device=cuda))
    st.stop.fill_(1)
    pre = st.snap()
    st.fused(gp, stats, 7, 1.0)
    st.reduce(gp, stats, 7)
    st.clip_adam(7, 1.0, 1, 1)
    post = st.snap()
    for key in pre:
        assert _same_bits(post[key], pre[key]), key


@pytest.mark.parametrize('path', ['fused', 'split'])
@pytest.mark.parametrize('max_norm', [0.0, -1.0])
def test_optim_no_clip_and_zero_gradient(cuda, max_norm, path):
    """max_grad_norm <= 0 never clips (gradients of norm 100 pass unscaled); a network whose gradient is all zero
    (reward critic, no L2 term) takes a zero step from a zero Adam state."""
    st = _Opt(cuda, 60, 8, seed=4)
    gen = torch.Generator(device=cuda).manual_seed(5)
    s, n = st.sec[1]
    for step in range(3):
        gp, stats = st.partials(gen, 17, (100.0, 0.0, 50.0), coef=0.0)
        pre = st.snap()
        ref = _ref_grad(st.sec, gp, pre['theta'], 0.0)
        (st.fused if path == 'fused' else st.split)(gp, stats, 7, max_norm, coef=0.0)
        post = st.snap()
        _check_step(st.sec, pre, post, ref, 7, max_norm, LRS, f'{path} max {max_norm} step {step}', coef=0.0,
                    stats=stats.cpu().numpy())
        assert _same_bits(post['theta'][s:s + n], pre['theta'][s:s + n]) and not post['m'][s:s + n].any()


@pytest.mark.parametrize('world', [1, 2, 4])
def test_clip_allreduce_adam_split_path(cuda, world):
    """The multi-rank order of the reference (policy_gradient.py:L437-443, restated by oracle.learner.update_ppo_multirank):
    every rank reduces and clips its own gradient (osb_grad_reduce + osb_clip_adam(do_clip=1, do_adam=0)), the clipped
    gradients are summed (the all-reduce, simulated here in rank order), then osb_clip_adam(do_clip=0, do_adam=1,
    grad_scale=1/world) takes one Adam step on the average.  With one rank this equals osb_optim_fused."""
    O, A, nblocks, max_norm = 60, 8, 17, 1.0
    st = _Opt(cuda, O, A, seed=world)
    twin = _Opt(cuda, O, A, seed=world)                # world == 1: the same steps through osb_optim_fused
    gen = torch.Generator(device=cuda).manual_seed(100 + world)
    targets = [(10.0, 0.1, 1.001), (0.5, 2.0, 0.9), (3.0, 0.99, 0.2), (0.7, 1.2, 4.0)]
    for step in range(5):
        parts = [st.partials(gen, nblocks, targets[r]) for r in range(world)]
        pre = st.snap()
        clipped, want = [], [np.zeros(n) for _, n in st.sec]
        for r, (gp, stats) in enumerate(parts):
            st.step.copy_(torch.as_tensor(pre['step']))      # every rank starts from the same counters
            st.ts.copy_(torch.as_tensor(pre['ts']))
            st.reduce(gp, stats, 7)
            raw = st.snap()['grad']
            st.clip_adam(7, max_norm, 1, 0)
            cl = st.snap()['grad']
            ref = _ref_grad(st.sec, gp, pre['theta'], COEF)
            for k, (s, n) in enumerate(st.sec):
                g64, bound, norm = ref[k]
                check_grad(raw[s:s + n], g64, bound, 0.0, f'rank {r} {NETS[k]} raw')
                c = st.kernel_coef(k, max_norm)           # one float coefficient per network, applied once per element
                assert _same_bits(cl[s:s + n], (raw[s:s + n] * c).astype(F)), (r, NETS[k])
                check_grad(cl[s:s + n], g64, bound, max_norm, f'rank {r} {NETS[k]} clipped')
                want[k] += clip_coef64(norm, max_norm) * g64
            clipped.append(st.grad.clone())
        total = clipped[0]
        for r in range(1, world):
            total = total + clipped[r]
        st.grad.copy_(total)
        st.clip_adam(7, max_norm, 0, 1, grad_scale=float(F(1.0 / world)))
        post = st.snap()
        for k, (s, n) in enumerate(st.sec):
            rel = np.linalg.norm(post['grad'][s:s + n] - want[k]) / np.linalg.norm(want[k])
            assert rel <= 1e-5, (NETS[k], rel)
            g = (post['grad'][s:s + n] * F(1.0 / world)).astype(F)
            t = int(pre['step'][k]) + 1
            assert post['step'][k] == t
            check_adam((pre['theta'][s:s + n], pre['m'][s:s + n], pre['v'][s:s + n]),
                       (post['theta'][s:s + n], post['m'][s:s + n], post['v'][s:s + n]), g, t, LRS[k], NETS[k])
        if world == 1:
            twin.fused(parts[0][0], parts[0][1], 7, max_norm)
            tw = twin.snap()
            assert (tw['step'] == post['step']).all()
            ref = _ref_grad(st.sec, parts[0][0], pre['theta'], COEF)
            for k, (s, n) in enumerate(st.sec):
                rel = np.linalg.norm(tw['grad'][s:s + n] - post['grad'][s:s + n]) / np.linalg.norm(post['grad'][s:s + n])
                assert rel <= 1e-5, (NETS[k], rel)
            for key in ('theta', 'm', 'v'):
                bad = ~np.isclose(tw[key], post[key], rtol=1e-5, atol=1e-9)
                assert bad.mean() <= 1e-3, (key, int(bad.sum()))


# ================= B. persistent bf16x3 iteration, one minibatch per launch ============================================
_X3_SHAPES = {16384: (256, 64), 8192: (128, 64), 4096: (64, 64), 2048: (32, 64), 512: (16, 32)}
# (id, O, A, rows per launch, net_mask, optimiser branch per network (s = speculative, c = chunked, - = masked out),
#  threshold: 'none' = max_grad_norm 40 (no network clips), 'split' = between the networks' norms on every launch,
#  'alt' = 40 and 'split' on alternate launches).  Consecutive cases change (O, A): the static weight image is re-zeroed.
X3_CASES = [
    ('bench', 60, 8, 16384, 7, 'sss', 'none'),
    ('o64_a16', 64, 16, 8192, 7, 'sss', 'alt'),
    ('redo', 60, 8, 16384, 7, 'sss', 'split'),
    ('critics', 17, 6, 4096, 6, '-ss', 'alt'),
    ('mixed', 60, 8, 2048, 7, 'css', 'alt'),
    ('a1', 33, 1, 4096, 7, 'sss', 'alt'),
    ('chunked', 60, 8, 512, 7, 'ccc', 'alt'),
    ('actor148', 60, 8, 16384, 1, 's--', 'split'),
]


def _split_threshold(norms):
    """A max_grad_norm that clips some of the given networks and not others, at least 2 % from every norm (all of them
    when the norms are too close to separate)."""
    x = np.sort(norms)
    if len(x) > 1 and (x[1:] / x[:-1]).max() > 1.05:
        j = int(np.argmax(x[1:] / x[:-1]))
        return float(math.sqrt(x[j] * x[j + 1]))
    return 0.5 * float(x[0])


@pytest.mark.timeout(300)
@pytest.mark.parametrize('name,O,A,rows,mask,branches,rule', X3_CASES, ids=[c[0] for c in X3_CASES])
def test_x3_persistent_step(cuda, name, O, A, rows, mask, branches, rule):
    """Per-step invariants of the in-kernel optimiser: the stored gradient against the fp64 sum of the stepwise bf16x3
    kernel's partials (same tiles, same grid, different summation order) on the pre-step parameters, theta / m / v
    against the fp32 Adam restatement applied to that gradient, adam_step, masked-out networks untouched."""
    lib, ptr, s = _lib()
    N, T = _X3_SHAPES[rows]
    rng = np.random.default_rng(rows + O)
    theta = oac.init_theta(O, A, seed=O)
    data = _rand_data(rng, N, T, O, A, theta)
    agent, buf, eng = _setup(cuda, data, N, T, O, A, theta)
    sec = _sections(O, A)
    P = oac.layout(O, A)['total']
    lag = torch.tensor([0.2, 0, 0, 0], dtype=torch.float32, device=cuda)
    G = lib.osb_tc_grid_blocks(rows, mask)
    got_branch = ''.join('-' if not (mask >> k) & 1 else ('s' if -(-n // G) <= NEPI else 'c') for k, (_, n) in enumerate(sec))
    assert got_branch == branches, f'{name}: grid {G} gives branches {got_branch}, the case is meant for {branches}'
    active = [k for k in range(3) if (mask >> k) & 1]
    mixed_launches = 0
    for launch in range(6):
        perm = torch.as_tensor(_rows(rng.permutation(rows), N, T)).to(cuda)
        # reference partials on the pre-step parameters
        lib.osb_minibatch_grad_x3(ptr(agent.theta), O, A, *eng._batch_ptrs(), ptr(eng.mu_old), ptr(buf.adv_moments),
                                  ptr(perm), rows, 0, 0, rows, 0, 0.2, 0.0, 1.0, 0.0, ptr(lag), ptr(eng.logstd_old), mask,
                                  ptr(eng.gpart), ptr(eng.stats_part), 0, s)
        gp = eng.gpart[:G * P].view(G, P).clone()
        stats = eng.stats_part[:G * 24].view(G, 3, 8).cpu().numpy()
        torch.cuda.synchronize()
        pre = {k: t.cpu().numpy().copy() for k, t in (('theta', agent.theta), ('grad', agent.grad), ('m', agent.adam_m),
                                                      ('v', agent.adam_v), ('step', agent.adam_step),
                                                      ('ts', eng.train_stats))}
        ref = _ref_grad(sec, gp, pre['theta'], COEF)
        norms = [ref[k][2] for k in active]
        use_split = rule == 'split' or (rule == 'alt' and launch % 2 == 1)
        max_norm = _split_threshold(norms) if use_split else 40.0
        clips = [clip_coef64(ref[k][2], max_norm) < 1.0 for k in range(3)]
        if rule == 'none':
            assert not any(clips[k] for k in active), f'{name}: norms {norms} reach max_grad_norm 40'
        mixed_launches += len({clips[k] for k in active}) > 1
        lib.osb_ppo_update_iter_x3(ptr(agent.theta), ptr(agent.grad), ptr(agent.adam_m), ptr(agent.adam_v),
                                   ptr(agent.adam_step), O, A, *eng._batch_ptrs(), ptr(buf.adv_moments), ptr(perm), rows, 0,
                                   rows, 0, 0.2, 0.0, ptr(lag), mask, COEF, max_norm, *LRS, ptr(eng.gpart),
                                   ptr(eng.stats_part), ptr(eng.train_stats), ptr(eng.stop_flag), 0, 0, 1, 0, 0, s)
        torch.cuda.synchronize()
        post = {k: t.cpu().numpy().copy() for k, t in (('theta', agent.theta), ('grad', agent.grad), ('m', agent.adam_m),
                                                       ('v', agent.adam_v), ('step', agent.adam_step),
                                                       ('ts', eng.train_stats))}
        taken = ' '.join(f'{NETS[k]}={"-" if k not in active else ("speculative" if branches[k] == "s" else "chunked") + ("+redo" if branches[k] == "s" and clips[k] else "+clip" if clips[k] else "")}'
                         for k in range(3))
        print(f'{name} launch {launch}: G={G} max_grad_norm={max_norm:.4g} norms={[f"{x:.4g}" for x in norms]} {taken}')
        _check_step(sec, pre, post, ref, mask, max_norm, LRS, f'{name} launch {launch}', stats=stats)
    if name == 'redo':
        assert mixed_launches == 6, f'{name}: every launch should clip some networks and not others'


# ================= C. persistent iteration, several minibatches per launch, toggling clip ==============================
@pytest.mark.timeout(300)
@pytest.mark.parametrize('O,A,N,T,batch', [(60, 8, 256, 250, 16384), (64, 16, 128, 192, 8192), (60, 8, 64, 100, 2048)],
                         ids=['60x8_b16384_short_last', '64x16_b8192', '60x8_b2048_mixed'])
def test_x3_persistent_toggling_clip_equals_stepwise(cuda, O, A, N, T, batch):
    """Several minibatches per launch (the weight image is rebuilt inside the kernel between steps) with max_grad_norm at
    the median of the per-step, per-network gradient norms, so that clipping toggles from step to step and networks
    take different branches in the same step; the launch-per-minibatch loop (osb_minibatch_grad_x3 + osb_optim_fused)
    is the reference, at the bar of test_x3_fused_iteration_equals_stepwise."""
    lib, ptr, s = _lib()
    rng = np.random.default_rng(N + T + O)
    theta = oac.init_theta(O, A, seed=7)
    data = _rand_data(rng, N, T, O, A, theta)
    B = N * T
    iters = 2
    perms = torch.as_tensor(np.stack([_rows(rng.permutation(B), N, T) for _ in range(iters)])).to(cuda)
    sec = _sections(O, A)
    P = oac.layout(O, A)['total']

    def run(max_norm, fused):
        agent, buf, eng = _setup(cuda, data, N, T, O, A, theta)
        lag = torch.tensor([0.2, 0, 0, 0], dtype=torch.float32, device=cuda)
        norms = []
        for it in range(iters):
            if fused:
                lib.osb_ppo_update_iter_x3(ptr(agent.theta), ptr(agent.grad), ptr(agent.adam_m), ptr(agent.adam_v),
                                           ptr(agent.adam_step), O, A, *eng._batch_ptrs(), ptr(buf.adv_moments),
                                           ptr(perms[it]), B, 0, batch, 0, 0.2, 0.0, ptr(lag), 7, COEF, max_norm, *LRS,
                                           ptr(eng.gpart), ptr(eng.stats_part), ptr(eng.train_stats), ptr(eng.stop_flag),
                                           0, 0, 1, 0, 0, s)
                continue
            for start in range(0, B, batch):
                count = min(batch, B - start)
                lib.osb_minibatch_grad_x3(ptr(agent.theta), O, A, *eng._batch_ptrs(), ptr(eng.mu_old),
                                          ptr(buf.adv_moments), ptr(perms[it]), B, 0, start, count, 0, 0.2, 0.0, 1.0, 0.0,
                                          ptr(lag), ptr(eng.logstd_old), 7, ptr(eng.gpart), ptr(eng.stats_part), 0, s)
                nb = lib.osb_tc_grid_blocks(count, 7)
                g = eng.gpart[:nb * P].view(nb, P).double().sum(0)
                th = agent.theta.double()
                norms.append([float((g[a:a + n] + (2.0 * float(F(COEF)) * th[a:a + n] if k else 0.0)).norm())
                              for k, (a, n) in enumerate(sec)])
                lib.osb_optim_fused(ptr(eng.gpart), ptr(eng.stats_part), nb, O, A, ptr(agent.theta), ptr(agent.grad),
                                    ptr(agent.adam_m), ptr(agent.adam_v), ptr(agent.adam_step), COEF, max_norm, *LRS, 7,
                                    ptr(eng.sumsq_part), ptr(eng.train_stats), 0, s)
        torch.cuda.synchronize()
        out = tuple(t.cpu().numpy().copy() for t in (agent.theta, agent.adam_m, agent.adam_v, agent.adam_step))
        return out, eng.train_stats.cpu().numpy().reshape(3, 8).copy(), np.array(norms)

    # the threshold: median of the dry run's norms of the network whose norm varies most from step to step (off the
    # median itself by 0.07 %, so that no norm of the real run lands on it)
    _, _, dry = run(1e9, False)
    k_sel = int(np.argmax(dry.max(0) / dry.min(0)))
    max_norm = float(np.median(dry[:, k_sel])) * 1.0007
    want, ts_want, norms = run(max_norm, False)
    clip = norms > max_norm
    print(f'max_grad_norm {max_norm:.4g} (median of {NETS[k_sel]}); clipping steps per network {clip.sum(0).tolist()} '
          f'of {len(clip)}')
    assert np.abs(norms / max_norm - 1.0).min() > 1e-5, 'a norm sits on the threshold: the branch would be a coin toss'
    assert any(clip[:, k].any() and not clip[:, k].all() for k in range(3)), 'clipping never toggles'
    assert any(clip[i].any() and not clip[i].all() for i in range(len(clip))), 'no step has networks on different branches'
    got, ts_got, _ = run(max_norm, True)
    assert (got[3] == want[3]).all() and got[3][0] == iters * -(-B // batch)
    for a, b, name in zip(want[:3], got[:3], ('theta', 'm', 'v')):
        # identical arithmetic, different summation order of the partial gradients -> a few ulp on the gradient
        bad = ~np.isclose(b, a, rtol=1e-4, atol=1e-7)
        assert bad.mean() < 2e-3, (name, bad.sum(), np.abs(a - b).max())
    np.testing.assert_allclose(ts_got[:, :4], ts_want[:, :4], rtol=1e-4, atol=1e-6)


# ================= D. Lagrange multiplier and KL early stop ============================================================
def _jc_sequence():
    k = np.arange(300)
    jc = 25.0 + 8.0 * np.sin(k / 7.0) + 0.37
    jc[110:200] = 12.5          # long stretch below the limit: lambda is pinned at 0
    jc[200:240] = 60.0          # far above: lambda climbs (to the upper bound when there is one)
    return jc


@pytest.mark.parametrize('upper', [None, 0.8])
def test_lagrange_update_sequence(cuda, upper):
    """300 steps of osb_lagrange_update: per step (re-based on the device state) lambda / m / v against the fp32 Adam
    restatement + clamp (m, v bit for bit, lambda to 1 ulp, t + 1); free-running against oracle.Lagrange (torch Adam on a
    Parameter, clamp_) within 1e-5 -- torch's CPU lerp may fuse a multiply-add, hence the looser free-running bar.  An
    empty window sets nan_flag and leaves the state, t included, untouched; the next window continues the sequence."""
    from omnisafe_b200.common.lagrange import Lagrange

    cost_limit, lam0, lr = 25.0, 0.001, 0.035
    lag = Lagrange(cost_limit, lam0, lr, lagrangian_upper_bound=upper, device=cuda)
    ref = ol.Lagrange(cost_limit, lam0, lr, upper_bound=upper)
    jcs = _jc_sequence()
    assert (np.diff(np.sign(jcs - cost_limit)) != 0).sum() >= 6
    ws = torch.zeros(4, dtype=torch.float64, device=cuda)
    pinned = at_upper = 0
    lam_max = 0.0
    for i, jc in enumerate(jcs):
        if i == 150:
            pre = lag.state.cpu().numpy().copy()
            ws.zero_()
            lag.update_lagrange_multiplier(ws)
            assert int(lag.nan_flag.item()) == 1 and _same_bits(lag.state.cpu().numpy(), pre)
            lag.nan_flag.zero_()
        cnt = float(7 + i % 5)
        ws.copy_(torch.tensor([1.0, jc * cnt, 3.0, cnt], dtype=torch.float64))
        jc_k = (jc * cnt) / cnt                               # the kernel's fp64 window mean
        pre = lag.state.cpu().numpy().copy()
        lag.update_lagrange_multiplier(ws)
        post = lag.state.cpu().numpy().copy()
        assert int(lag.nan_flag.item()) == 0
        t = int(pre[3]) + 1
        assert post[3] == t
        g = F(-(jc_k - float(F(cost_limit))))
        th1, m1, v1 = adam_f32(pre[0], pre[1], pre[2], g, t, lr)
        lam = np.maximum(th1, F(0))
        if upper is not None:
            lam = np.minimum(lam, F(upper))
        assert _same_bits(post[1], m1) and _same_bits(post[2], v1), (i, post, m1, v1)
        assert ulp_diff(post[0], lam) <= 1, (i, post[0], lam)
        want = ref.update(jc_k)
        assert abs(float(post[0]) - want) <= 1e-5, (i, float(post[0]), want)
        pinned += post[0] == 0.0
        at_upper += upper is not None and post[0] == F(upper)
        lam_max = max(lam_max, float(post[0]))
    assert pinned >= 30, pinned
    if upper is not None:
        assert at_upper >= 5, at_upper
    else:
        assert lam_max > 0.8, lam_max


def test_kl_check(cuda):
    """kl = eval_out[0] / eval_out[4]; the pass counter includes the stopping pass (Train/StopIter = i + 1); once
    stopped, later calls change nothing; early_stop = 0 never stops; and the comparison is the reference's
    `kl.item() > target_kl`: the fp32 KL against the Python float target."""
    lib, ptr, s = _lib()
    ev = torch.zeros(8, dtype=torch.float64, device=cuda)
    stop = torch.zeros(1, dtype=torch.int32, device=cuda)
    kls = torch.zeros(4, dtype=torch.float32, device=cuda)

    def call(kl_sum, n, target, early):
        ev[0], ev[4] = kl_sum, n
        lib.osb_kl_check(ptr(ev), target, early, ptr(stop), ptr(kls), s)
        torch.cuda.synchronize()
        return int(stop.item()), kls.cpu().numpy().copy()

    seq = [0.005, 0.019, 0.03, 0.001, 0.5]
    for early in (1, 0):
        stop.zero_()
        kls.zero_()
        stopped_at = None
        for i, kl in enumerate(seq):
            prev = kls.cpu().numpy().copy()
            st, k = call(kl * 4096.0, 4096.0, 0.02, early)
            if stopped_at is not None:
                assert st == 1 and _same_bits(k, prev), 'a stopped pass changed the KL state'
                continue
            assert k[0] == F(kl * 4096.0 / 4096.0) and k[1] == i + 1
            if early and kl > 0.02:
                stopped_at = i
                assert st == 1 and k[2] == 1.0
            else:
                assert st == 0 and k[2] == 0.0
        assert stopped_at == (2 if early else None)
    # one ulp either side of the target, for targets whose float rounding lies above (0.1, 0.3) or below (0.02, 1/3)
    for target in (0.02, 0.1, 0.3, 1.0 / 3.0, 0.01):
        kf = F(target)
        for kl in (np.nextafter(kf, F(0)), kf, np.nextafter(kf, F(1))):
            stop.zero_()
            kls.zero_()
            st, _ = call(float(kl), 1.0, target, 1)
            # 0.1 caught a float-versus-float comparison: f32(0.1) > 0.1, so a KL of exactly f32(0.1) stops the reference
            assert st == int(float(kl) > target), (target, float(kl))


# ================= E. conjugate gradients, dot / axpy, partial reduction ===============================================
def _spd(n, kappa, seed):
    """z = M p for M = H diag(lam) H, H = I - 2 u u^T (symmetric orthogonal): SPD, eigenvalues geometrically spaced in
    [1, kappa], so the condition number is exactly kappa; applied in O(n) in the dtype / device of p."""
    rng = np.random.default_rng(seed)
    u = rng.standard_normal(n)
    u /= np.linalg.norm(u)
    lam = np.geomspace(1.0, kappa, n) if n > 1 else np.array([math.sqrt(kappa)])
    rng.shuffle(lam)

    def op(p):
        uu = torch.as_tensor(u, dtype=p.dtype, device=p.device)
        ll = torch.as_tensor(lam, dtype=p.dtype, device=p.device)
        h = p - 2 * uu * torch.dot(uu, p)
        h = ll * h
        return h - 2 * uu * torch.dot(uu, h)
    return op


def _cg64(op, b, iters, tol, eps=1e-6):
    """oracle.learner.conjugate_gradients in fp64 (that function works in fp32), with the residual history."""
    b = torch.as_tensor(b, dtype=torch.float64)
    x = torch.zeros_like(b)
    r = b.clone()
    p = r.clone()
    rdotr = torch.dot(r, r)
    res = [math.sqrt(float(rdotr))]
    done = 0
    for k in range(iters):
        z = op(p)
        alpha = rdotr / (torch.dot(p, z) + eps)
        x = x + alpha * p
        r = r - alpha * z
        new_rdotr = torch.dot(r, r)
        res.append(math.sqrt(float(new_rdotr)))
        if math.sqrt(float(new_rdotr)) < tol:
            done = k + 1
            break
        p = r + new_rdotr / (rdotr + eps) * p
        rdotr = new_rdotr
    return x.numpy(), res, done


@pytest.mark.parametrize('kappa', [10.0, 1e4])
@pytest.mark.parametrize('n', [1, 1023, 1024, 1025, 8592, 28816])
def test_cg_vs_oracle(cuda, n, kappa):
    """osb_cg_init / osb_cg_step with z = M p computed by torch between steps, against oracle.learner.conjugate_gradients
    in fp32 and the same iteration in fp64: x, iteration count and converged flag; a residual_tol that is reached at step
    k < iters sets the flag at k and freezes x afterwards."""
    lib, ptr, s = _lib()
    op = _spd(n, kappa, seed=n)
    b = np.random.default_rng(n + 1).standard_normal(n).astype(F)
    iters = 10
    rel = lambda a, w: float(np.linalg.norm(a - w) / np.linalg.norm(w))   # noqa: E731

    def gpu(tol):
        bt = torch.as_tensor(b).to(cuda)
        x, r, p = (torch.zeros(n, device=cuda) for _ in range(3))
        sc = torch.zeros(4, device=cuda)
        lib.osb_cg_init(ptr(bt), n, ptr(x), ptr(r), ptr(p), ptr(sc), s)
        flags, xs = [], []
        for _ in range(iters):
            z = op(p).contiguous()
            lib.osb_cg_step(ptr(z), n, ptr(x), ptr(r), ptr(p), ptr(sc), tol, 1e-6, s)
            torch.cuda.synchronize()
            flags.append(float(sc[1]))
            xs.append(x.cpu().numpy().copy())
        return xs, flags, int(sc[2].item())

    # residual_tol 1e-10 is not reached in 10 steps: x and the count are compared, the flag stays down (for n = 1 the
    # float32 residual after the first step is rounding noise, so its flag is not compared)
    x64, res, done64 = _cg64(op, b, iters, 1e-10)
    x32 = ol.conjugate_gradients(op, b, iters).numpy()
    xs, flags, count = gpu(1e-10)
    err32 = rel(x32, x64)
    bar = max(1e-6, 4 * err32)     # fp64 dot products: at least as close to fp64 as the fp32 oracle
    print(f'n {n} kappa {kappa:g}: |x - x64| / |x64| = {rel(xs[-1], x64):.2e} (oracle fp32 {err32:.2e})')
    assert rel(xs[-1], x64) <= bar and rel(xs[-1], x32) <= bar + err32
    if n > 1:
        assert not done64 and count == iters and not any(flags)
    if kappa > 100:
        return      # the residual of the geometric spectrum does not fall below its first value within 10 steps
    # a tolerance reached at step k: below every earlier post-step residual by 1.5x or more (the kernel, like the
    # reference, only tests the residual after a step); the geometric mean of the two sides leaves 1.22x either way
    ks = [j for j in range(2, iters) if min(res[1:j]) / res[j] >= 1.5]
    k = ks[0] if ks else 1
    tol = math.sqrt(min(res[1:k]) * res[k]) if ks else 2.0 * res[1]
    x64, _, done64 = _cg64(op, b, iters, tol)
    calls = []
    x32 = ol.conjugate_gradients(lambda v: (calls.append(1), op(v))[1], b, iters, residual_tol=tol).numpy()
    xs, flags, count = gpu(tol)
    assert done64 == k and len(calls) - 1 == k, (k, done64, len(calls) - 1)
    assert count == k and flags == [0.0] * (k - 1) + [1.0] * (iters - k + 1), (k, count, flags)
    assert all(_same_bits(x, xs[k - 1]) for x in xs[k:]), 'x moved after convergence'
    err32 = rel(x32, x64)
    assert rel(xs[-1], x64) <= max(1e-6, 4 * err32)


@pytest.mark.parametrize('n', [1, 1023, 1024, 1025, 8592, 28816])
def test_dot_axpy(cuda, n):
    """osb_dot (fp64 accumulation, one rounding) to 1 ulp of the fp64 dot product; osb_axpy to 1 ulp of y + alpha x."""
    lib, ptr, s = _lib()
    rng = np.random.default_rng(n)
    a = (rng.standard_normal(n) * np.exp(rng.uniform(-3, 3, n))).astype(F)
    b = rng.standard_normal(n).astype(F)
    at, bt = torch.as_tensor(a).to(cuda), torch.as_tensor(b).to(cuda)
    out = torch.zeros(n + 4, device=cuda)
    lib.osb_dot(ptr(at), ptr(bt), n, ptr(out), s)
    want = float(np.dot(a.astype(np.float64), b.astype(np.float64)))
    got = float(out[0].item())
    assert ulp_diff(got, want) <= 1 or abs(got - want) <= n * 2.0 ** -50 * float(np.abs(a.astype(np.float64) * b).sum())
    alpha = float(F(-0.37))
    lib.osb_axpy(ptr(at), ptr(bt), alpha, n, ptr(out), s)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    assert ulp_diff(got[:n], (b.astype(np.float64) + alpha * a.astype(np.float64)).astype(F)).max() <= 1
    assert not got[n:].any(), 'axpy wrote past n'


@pytest.mark.parametrize('add', [False, True])
@pytest.mark.parametrize('nblocks', [1, 17, 148])
def test_reduce_partials(cuda, nblocks, add):
    """out = scale sum_b gpart[b][:n] + add_scale add (the damping term of the Fisher-vector product), rows of stride > n,
    against fp64 at the summation bound; nothing past n is written."""
    lib, ptr, s = _lib()
    n, stride = 8592, 8592 + 37
    gen = torch.Generator(device=cuda).manual_seed(nblocks)
    gp = torch.randn(nblocks, stride, generator=gen, device=cuda)
    vec = torch.randn(n, generator=gen, device=cuda)
    out = torch.full((n + 8,), 7.0, device=cuda)
    scale, add_scale = float(F(-1.0 / 3.0)), float(F(0.1))
    lib.osb_reduce_partials(ptr(gp), nblocks, stride, n, scale, ptr(vec) if add else 0, add_scale, ptr(out), s)
    torch.cuda.synchronize()
    g = gp[:, :n].double()
    want = scale * g.sum(0) + (add_scale * vec.double() if add else 0.0)
    bound = (nblocks + 2) * U * (abs(scale) * g.abs().sum(0) + (add_scale * vec.double().abs() if add else 0.0))
    got = out.cpu().numpy()
    err = np.abs(got[:n] - want.cpu().numpy())
    assert (err <= bound.cpu().numpy()).all(), float((err / bound.cpu().numpy()).max())
    assert (got[n:] == 7.0).all()
