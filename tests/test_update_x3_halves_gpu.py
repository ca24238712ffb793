"""The bf16x3 update kernel works on each 128-sample tile as two 64-sample halves (one per epilogue warp group, M = 64
GEMMs).  These cases exercise the shapes the split creates -- a last tile whose half b is empty or partial, grids with
CTAs that get no tile, A = 16 -- at the bars of tests/test_update_x3_gpu.py, and check that the persistent kernel is
bit-for-bit deterministic."""
import os

import numpy as np
import pytest
import torch

import test_update_x3_gpu as x3t
from oracle import actor_critic as oac
from test_update_gpu import _rand_data, _rows, _setup

pytestmark = pytest.mark.gpu


@pytest.mark.timeout(300)
@pytest.mark.parametrize('valid', [1, 63, 64, 65, 127])
@pytest.mark.parametrize('O,A,loss_kind', [(60, 8, 0), (64, 16, 1)])
def test_x3_grad_last_tile_rows(cuda, O, A, loss_kind, valid):
    """Minibatch of 3 full tiles + `valid` rows: half b of the last tile is empty (valid <= 64) or partial."""
    x3t.test_x3_grad_vs_autograd(cuda, O, A, 20, 30, loss_kind, 3 * 128 + valid)


def _epoch(cuda, data, N, T, O, A, theta, perms, batch, iters, fused):
    if fused:
        os.environ.pop('OSB_X3_NO_FUSE', None)
    else:
        os.environ['OSB_X3_NO_FUSE'] = '1'
    try:
        agent, buf, eng = _setup(cuda, data, N, T, O, A, theta)
        lag = torch.tensor([0.2, 0, 0, 0], dtype=torch.float32, device=cuda)
        eng.ppo_epoch(loss_kind=0, lagrange=lag, net_mask=7, batch_size=batch, update_iters=iters, clip=0.2,
                      critic_norm_coef=0.001, max_grad_norm=0.5, lr_actor=3e-4, lr_critic=3e-4,
                      target_kl=10.0, kl_early_stop=False, perm=perms, precision=2)
        torch.cuda.synchronize()
    finally:
        os.environ.pop('OSB_X3_NO_FUSE', None)
    return ((agent.theta.cpu().numpy(), agent.adam_m.cpu().numpy(), agent.adam_v.cpu().numpy(), agent.adam_step.cpu().numpy()),
            eng.train_stats.cpu().numpy().reshape(3, 8).copy())


# B % batch = the last minibatch: 1, 64 (one tile, half b empty), 81 (half b partial), 307 (3 tiles, 51 rows in the
# last), 123 (half b partial); the grid is sized for the first minibatch, so the short last one leaves CTAs without a tile
@pytest.mark.timeout(300)
@pytest.mark.parametrize('N,T,O,A,batch,iters', [
    (3, 171, 60, 8, 512, 2), (64, 17, 60, 8, 512, 2), (65, 17, 60, 8, 512, 2), (63, 13, 60, 8, 512, 2),
    (127, 5, 60, 8, 512, 1), (64, 17, 64, 16, 512, 2), (65, 17, 33, 16, 512, 2),
])
def test_x3_fused_halves_equal_stepwise(cuda, N, T, O, A, batch, iters):
    """Persistent kernel == launch-per-minibatch path (bars of test_x3_fused_iteration_equals_stepwise)."""
    rng = np.random.default_rng(N * T + A)
    theta = oac.init_theta(O, A, seed=2)
    data = _rand_data(rng, N, T, O, A, theta)
    B = N * T
    perms = torch.as_tensor(np.stack([_rows(rng.permutation(B), N, T) for _ in range(iters)])).to(cuda)
    (step, s0), (fused, s1) = (_epoch(cuda, data, N, T, O, A, theta, perms, batch, iters, f) for f in (False, True))
    assert (step[3] == fused[3]).all() and fused[3][0] == iters * -(-B // batch)
    assert not np.allclose(fused[0], theta)
    for a, b, name in zip(step[:3], fused[:3], ('theta', 'm', 'v')):
        bad = ~np.isclose(a, b, rtol=1e-4, atol=1e-7)
        assert bad.mean() < 2e-3, (name, bad.sum(), np.abs(a - b).max())
    np.testing.assert_allclose(s1[:, :4], s0[:, :4], rtol=1e-4, atol=1e-6)


@pytest.mark.timeout(300)
@pytest.mark.parametrize('A', [8, 16])
def test_x3_fused_deterministic(cuda, A):
    """Two identical runs of the persistent kernel give bit-identical parameters and Adam state."""
    N, T, O = 64, 40, 60
    rng = np.random.default_rng(11)
    theta = oac.init_theta(O, A, seed=3)
    data = _rand_data(rng, N, T, O, A, theta)
    perms = torch.as_tensor(np.stack([_rows(rng.permutation(N * T), N, T) for _ in range(2)])).to(cuda)
    runs = [_epoch(cuda, data, N, T, O, A, theta, perms, 1000, 2, True) for _ in range(2)]
    for a, b in zip(runs[0][0], runs[1][0]):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    assert np.array_equal(runs[0][1], runs[1][1])
