"""Multi-rank PARITY check (run under torchrun on >= 2 GPUs): each rank plays one rank of the unmodified reference's
`parallel = 2` run (tests/golden/update_ppolag_parallel2.npz: its own data and DataLoader orders, replicated parameters)
through every data-parallel path of the library --

  bf16x3 persistent kernel, clipped slices pushed over NVLink peer memory inside the kernel   (the bench path)
  bf16x3 per-minibatch kernels + reduce / clip / ncclAllReduce / Adam as separate launches      (OSB_X3_NO_FUSE, OSB_NO_P2P)
  fp32 tiles + optim_fused_kernel<true> (one-shot peer-memory all-reduce inside the optimiser kernel)
  fp32 tiles + NCCL

-- and must land on the reference's parameters (fp32 bar) with bit-identical parameters on all ranks.
Reference order: clip locally -> average -> Adam (policy_gradient.py:L437-443, distributed.py:L193-198)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np
import torch
import torch.distributed as dist

from omnisafe_b200.utils import distributed
from test_update_gpu import _rows, _setup

torch.cuda.set_device(int(os.environ['LOCAL_RANK']))
distributed.init_process_group('cuda')
rank, world = dist.get_rank(), dist.get_world_size()
assert world >= 2
dev = torch.device('cuda', int(os.environ['LOCAL_RANK']))
g = np.load(os.path.join(ROOT, 'tests', 'golden', 'update_ppolag_parallel2.npz'))
N, T, O, A = int(g['N']), int(g['T']), int(g['O']), int(g['A'])
r = rank % 2                                   # ranks >= 2 replay the two recorded shards again (the average is unchanged)
data = {k[len(f'r{r}_data_'):]: g[k] for k in g.files if k.startswith(f'r{r}_data_')}
perms = torch.as_tensor(np.stack([_rows(p_, N, T) for p_ in g[f'perms_r{r}'][::2]])).to(dev)
assert world % 2 == 0
from omnisafe_b200.common.lagrange import Lagrange

results = {}
for name, prec, env in (('bf16x3 persistent + NVLink push', 2, {}),
                        ('bf16x3 stepwise + NCCL', 2, {'OSB_X3_NO_FUSE': '1', 'OSB_NO_P2P': '1'}),
                        ('bf16x3 stepwise + p2p optimiser kernel', 2, {'OSB_X3_NO_FUSE': '1'}),
                        ('fp32 + p2p optimiser kernel', 0, {}),
                        ('fp32 + NCCL', 0, {'OSB_NO_P2P': '1'})):
    for k in ('OSB_X3_NO_FUSE', 'OSB_NO_P2P'):
        os.environ.pop(k, None)
    os.environ.update(env)
    agent, buf, eng = _setup(dev, data, N, T, O, A, g['theta0'])
    lag = Lagrange(float(g['cost_limit']), float(g['lam0']), float(g['lambda_lr']), device=dev)
    ws = torch.tensor([0.0, float(g['Jc']) * 10, 0.0, 10.0], dtype=torch.float64, device=dev)
    lag.update_lagrange_multiplier(ws)
    eng.ppo_epoch(loss_kind=0, lagrange=lag.state, net_mask=7, batch_size=int(g['batch_size']), update_iters=int(g['update_iters']),
                  clip=0.2, entropy_coef=0.0, critic_norm_coef=0.001, max_grad_norm=40.0, lr_actor=3e-4, lr_critic=3e-4,
                  target_kl=0.02, kl_early_stop=True, perm=perms, precision=prec)
    torch.cuda.synchronize()
    distributed.p2p_check()
    th = agent.theta.clone()
    ref = th.clone(); dist.broadcast(ref, 0)
    same = bool(torch.equal(ref, th))
    got, want = th.cpu().numpy(), g['theta1']
    bad = ~np.isclose(got, want, rtol=2e-4, atol=2e-6)
    kls = eng.kl_state.cpu().numpy()
    ok = bool(same and bad.mean() < 1e-3 and np.abs(got - want).max() < 2e-3 and int(kls[1]) == int(g['stop_iter'][-1])
              and abs(float(lag.lagrangian_multiplier) - float(g['lam1'])) < 1e-6)
    results[name] = ok
    if rank == 0:
        print(f'{name:42s}: identical across ranks {same}; vs reference parallel=2: {int(bad.sum())}/{bad.size} outside 2e-4, max abs '
              f'{np.abs(got - want).max():.2e}; kl {kls[0]:.6f} (ref {float(g["kl"][-1]):.6f}) iters {int(kls[1])}  -> {"OK" if ok else "FAIL"}', flush=True)
for k in ('OSB_X3_NO_FUSE', 'OSB_NO_P2P'):
    os.environ.pop(k, None)
dist.barrier()
allok = all(results.values())
if rank == 0:
    print('MULTI-RANK PARITY', 'OK' if allok else 'FAILED', flush=True)
dist.destroy_process_group()
sys.exit(0 if allok else 1)
