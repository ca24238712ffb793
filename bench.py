"""bench.py -- env-steps/sec over full on-policy SafeRL epochs (rollout + dual GAE + update).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--algo PPOLag|CPO|TRPOLag|FOCOPS] [--obs-dim D] [--precision bf16x3|tf32|fp32]
                    [--dump-outputs DIR]

A "step" is one epoch of a BASELINE.json workload: by default `configs[1]` = PPOLag on the synthetic Box env
(obs 60 / act 8), 4096 HBM-resident envs per GPU, T = 128 steps per env (524 288 samples per GPU), update_iters 8,
batch_size 16384 -- i.e. the reference's `Time/FPS = steps_per_epoch / epoch_time`
(omnisafe/algorithms/on_policy/base/policy_gradient.py:L280).  `--algo CPO` is `configs[2]`, `--algo TRPOLag|FOCOPS
--obs-dim 17|60|111|376` is the sweep of `configs[4]`.  Prints ONE JSON line.

  value   : device-timed (CUDA events, barrier + synchronize on both sides, max over ranks), everything resident in
            HBM, in-kernel Philox noise.  Arithmetic = `--precision`, default bf16x3: every layer GEMM runs on the
            tensor cores as six kind::f16 MMAs over the three bf16 pieces of its fp32 operands with fp32
            accumulation -- held by the tests to the bar of the exact-fp32 path (reference: fp32 Linear layers).
            The tf32 mode (5e-3) is reported as a labelled extra, never as the headline.
  e2e     : the same metric through the public `omnisafe_b200.Agent(...)` training loop with HOST buffers: every
            epoch the standard-normal action-noise stream is copied from pinned host memory (parity-mode input of
            the rollout) and the epoch's logged metrics are read back.
  --dump-outputs DIR : after the timed steps, what the last timed epoch handed its caller is written as DIR/<name>.npy
            (float32; float64 where the library keeps float64): the parameters after the update, the epoch's rollout and
            GAE slabs (a fixed, seeded sample of their (t, env) rows), the observation-normaliser statistics, the
            episode-window sums, the update statistics and the Lagrange state.  The workload is seeded, so the same
            arguments give the same inputs from run to run and two builds can be compared output for output.
  --impl reference : the CPU restatement of the reference path (oracle/, torch-CPU + numpy) timed on the host cores
            on the SAME workload size (4096 envs x T = 128 per step); /root/reference does not exist on the GPU box.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(algo='PPOLag', env='SyntheticBox-v0', obs_dim=60, act_dim=8, envs_per_gpu=4096,
                steps_per_env=128, batch_size=16384, update_iters=8, max_episode_steps=64)
ALGOS = ('PPOLag', 'CPO', 'TRPOLag', 'FOCOPS')
DTYPES = {'bf16x3': 'bf16x3 (fp32 operands as 3 bf16 pieces, 6 tcgen05 kind::f16 MMAs per product, fp32 accumulate: fp32-level '
                    'results; GAE fp64 carry)',
          'tf32': 'tf32 (fp32 storage/accumulate; GAE fp64 carry)',
          'fp32': 'f32 (FMA tiles; GAE fp64 carry)'}


# ------------------------------------------------------------------------------------------------
def _peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p['bf16_tflops'],
                'bf16_tflops_sustained': p.get('bf16_tflops_sustained', p['bf16_tflops']), 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index: int) -> None:
        self.rows, self._stop, self.gpu = [], threading.Event(), gpu_index
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self) -> None:
        while not self._stop.is_set():
            try:
                out = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                      '-i', str(self.gpu)], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(',')])
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join(timeout=3)

    def summary(self) -> dict:
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (('hw_slowdown', 4), ('hw_thermal_slowdown', 5), ('sw_thermal_slowdown', 6), ('sw_power_cap', 7)):
                if len(r) > col and r[col].lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
def _custom_cfgs(world: int, log_dir: str, epochs: int, obs_dim: int | None = None, precision: str | None = None) -> dict:
    w = WORKLOAD
    spe = world * w['envs_per_gpu'] * w['steps_per_env']
    cfg = {
        'seed': 0,
        'train_cfgs': {'device': 'cuda', 'vector_env_nums': w['envs_per_gpu'], 'parallel': world,
                       'total_steps': spe * epochs},
        'algo_cfgs': {'steps_per_epoch': spe, 'batch_size': w['batch_size'], 'update_iters': w['update_iters']},
        'logger_cfgs': {'log_dir': log_dir, 'use_tensorboard': False, 'save_model_freq': 10 ** 9},
        'env_cfgs': {'obs_dim': obs_dim or w['obs_dim'], 'act_dim': w['act_dim'], 'max_episode_steps': w['max_episode_steps']},
    }
    if precision:
        cfg['train_cfgs']['matmul_precision'] = precision
    return cfg


def _workload_name(algo: str, obs_dim: int) -> str:
    which = ('configs[1]' if (algo, obs_dim) == ('PPOLag', 60) else 'configs[2]' if (algo, obs_dim) == ('CPO', 60)
             else 'configs[4] obs-dim sweep' if algo in ('TRPOLag', 'FOCOPS') else 'variant')
    return (f'{algo} SyntheticBox-v0 obs{obs_dim}/act8, 4096 envs/GPU x T=128, batch 16384, update_iters 8 '
            f'(BASELINE.json {which})')


def _flops_per_sample(O: int, A: int) -> int:
    """fwd + bwd multiply-adds x2 of the three trunks (actor O-64-64-A, two critics O-64-64-1);
    backward = 2x forward except that no dX is formed for layer 1 (SURVEY §8a row 3)."""
    def net(out):
        fwd = 2 * (O * 64 + 64 * 64 + 64 * out)
        bwd = 2 * (O * 64 + 2 * 64 * 64 + 2 * 64 * out)
        return fwd + bwd
    return net(A) + 2 * net(1)


DUMP_ROWS = 16384          # (t, env) rows of each per-epoch slab written by --dump-outputs: 5 MB at obs_dim 60


def dump_outputs(algo, out_dir: str) -> None:
    """--dump-outputs: the outputs of the epoch algo.train_epoch() last ran, as DIR/<name>.npy."""
    d, env = algo._buf.data, algo._env
    T, N = d['reward'].shape
    rows = np.sort(np.random.default_rng(0).choice(T * N, size=min(DUMP_ROWS, T * N), replace=False))
    rows = torch.as_tensor(rows, device=d['reward'].device)
    out = {'theta': algo._actor_critic.theta, 'obs_norm_mean': env._obs_normalizer.mean,
           'obs_norm_std': env._obs_normalizer.std, 'window_sums': env.window_sums,
           'train_stats': algo._engine.train_stats, 'kl_state': algo._engine.kl_state, 'sample_rows': rows}
    lagrange = getattr(algo, '_lagrange', None)
    if lagrange is not None:
        out['lagrange_state'] = lagrange.state
    for name, v in d.items():
        if v is not None and tuple(v.shape[:2]) == (T, N):
            out['slab_' + name] = v.reshape(T * N, *v.shape[2:])[rows]
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        v = v.detach().cpu()
        np.save(os.path.join(out_dir, name + '.npy'), v.numpy().astype(np.float64 if v.dtype in (torch.float64, torch.int64) else np.float32))


def run_b200(args) -> dict:
    import torch.distributed as dist

    import omnisafe_b200
    from omnisafe_b200._lib import current_stream, lib, ptr
    from omnisafe_b200.utils import distributed

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N > 1)'
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')     # NCCL's version banner / warnings go to stderr: stdout carries ONE JSON line
        distributed.init_process_group('cuda')
    w = WORKLOAD
    T, N, O, A = w['steps_per_env'], w['envs_per_gpu'], args.obs_dim, w['act_dim']
    samples_global = world * N * T

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """K calls of fn bracketed by barrier + synchronize, device time (ms), max over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def make(precision):
        tmp = tempfile.mkdtemp(prefix='osb_bench_')
        agent = omnisafe_b200.Agent(args.algo, w['env'], custom_cfgs=_custom_cfgs(world, tmp, args.steps + args.warmup + 16, O, precision))
        return agent.agent

    algo = make(args.precision)
    warm = max(args.warmup, 3)

    # ---- device-resident number ("value") -------------------------------------------------------
    for _ in range(warm):
        algo.train_epoch()
    barrier()
    l0 = lib().osb_launch_count()
    with ClockSampler(local_rank) as clk:
        ms = timed(algo.train_epoch, args.steps)
    launches = int(lib().osb_launch_count() - l0)
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(algo, args.dump_outputs)
    ms_per_step = ms / args.steps
    value = samples_global / (ms_per_step * 1e-3)

    # ---- end to end through the public loop with host buffers ----------------------------------
    host_eps = torch.randn(T, N, A, dtype=torch.float32).pin_memory()
    dev_eps = torch.empty(T, N, A, dtype=torch.float32, device='cuda')
    d2h = {'bytes': 0}

    def e2e_epoch():
        dev_eps.copy_(host_eps, non_blocking=True)            # H2D of this epoch's noise stream
        row = algo.train_epoch(eps=dev_eps, log=True)          # logs => D2H read of the epoch metrics
        d2h['bytes'] = row['d2h_bytes']

    for _ in range(2):
        e2e_epoch()
    ms_e2e = timed(e2e_epoch, args.steps) / args.steps
    e2e = {'value': samples_global / (ms_e2e * 1e-3), 'unit': 'env-steps/s',
           'h2d_bytes_per_step': host_eps.numel() * 4, 'd2h_bytes_per_step': d2h['bytes'],
           'ms_per_step': ms_e2e}

    # ---- stage split + roofline of the dominant kernel, timed live with CUDA events -------------
    peaks = _peaks()
    eng, buf, ac = algo._engine, algo._buf, algo._actor_critic
    lag_state = getattr(getattr(algo, '_lagrange', None), 'state', None)
    if lag_state is None:
        lag_state = torch.zeros(4, dtype=torch.float32, device='cuda')
    d = buf.data
    total = T * N
    ms_roll = timed(lambda: algo._env.rollout(algo._steps_per_epoch, ac, buf, algo._logger), 5) / 5
    ms_gae = timed(buf.finish_paths, 50) / 50
    ms_upd = timed(algo._update, 5) / 5
    flop_per_sample = _flops_per_sample(O, A)
    n_mb = -(-total // w['batch_size'])
    x3_path = args.precision == 'bf16x3' and O <= 64
    if x3_path:
        # one launch of the persistent kernel = one update iteration = n_mb minibatch steps (forward + loss + backward + optimiser)
        def iter_launch():
            lib().osb_ppo_update_iter_x3(ptr(ac.theta), ptr(ac.grad), ptr(ac.adam_m), ptr(ac.adam_v), ptr(ac.adam_step), O, A,
                                         ptr(d['obs']), ptr(d['act']), ptr(d['logp']), ptr(d['adv_r']), ptr(d['adv_c']),
                                         ptr(d['target_value_r']), ptr(d['target_value_c']), ptr(buf.adv_moments), 0, total, 12345,
                                         w['batch_size'], 0, 0.2, 0.0, ptr(lag_state), 7, 0.001, 40.0, 0.0, 0.0, 0.0,
                                         ptr(eng.gpart), ptr(eng.stats_part), ptr(eng.train_stats), 0, 0, 0, 1, 0, 0, current_stream())
        ms_k = timed(iter_launch, 10) / 10          # learning rates 0: the parameters stay put
        kname, rows_per_launch = 'minibatch_grad_x3_kernel<fused> (persistent: 1 launch = 1 update iteration)', total
        # dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full (profiles/r02_ncu_update_x3.md)
        traffic = 218.8e6 if (O == 60 and A == 8 and total == 524288 and args.algo == 'PPOLag') else None
    else:
        fn = lib().osb_minibatch_grad_tc if args.precision == 'tf32' else lib().osb_minibatch_grad

        def iter_launch():
            fn(ptr(ac.theta), O, A, ptr(d['obs']), ptr(d['act']), ptr(d['logp']), ptr(d['adv_r']), ptr(d['adv_c']),
               ptr(d['target_value_r']), ptr(d['target_value_c']), ptr(eng.mu_old), ptr(buf.adv_moments), 0, total, 12345, 0,
               w['batch_size'], 0, 0.2, 0.0, 1.0, 0.0, ptr(lag_state), ptr(eng.logstd_old), 7, ptr(eng.gpart),
               ptr(eng.stats_part), 0, current_stream())
        ms_k = timed(iter_launch, 50) / 50
        kname = 'minibatch_grad_tc_kernel' if args.precision == 'tf32' else 'minibatch_grad_kernel'
        rows_per_launch = w['batch_size']
        traffic = 14.57e6 if (args.precision == 'tf32' and O == 60) else None     # ncu --set full, profiles/r01_ncu_minibatch_grad_tc.md
    # the GAE scan where HBM is its bound: a horizon whose 277 MB of algorithmic traffic do not fit L2 (the epoch's own
    # T = 128 launch moves 17 MB and is latency bound)
    from omnisafe_b200.common.buffer import VectorOnPolicyBuffer
    T_long = 2048
    lbuf = VectorOnPolicyBuffer(4, 2, T_long, 0.99, 0.95, 0.95, 'gae', 0.0, True, True, num_envs=N, device='cuda', keep_discounted_ret=False)
    for k_ in ('reward', 'cost', 'value_r', 'value_c', 'boot_r', 'boot_c'):
        lbuf.data[k_].normal_()
    lbuf.data['flags'][w['max_episode_steps'] - 1::w['max_episode_steps']] = 2          # the bench env's time-limit truncations
    for _ in range(3):
        lbuf.finish_paths()
    ms_gae_long = timed(lbuf.finish_paths, 20) / 20
    gae_long_gbs = 33.0 * T_long * N / (ms_gae_long * 1e-3) / 1e9
    del lbuf
    ach_tf = flop_per_sample * rows_per_launch / (ms_k * 1e-3) / 1e12
    row_bytes = 4.0 * (O + A + 5)
    gae_gbs = 33.0 * total / (ms_gae * 1e-3) / 1e9
    roofline = {
        'kernel': kname, 'bound': 'tensor', 'achieved': ach_tf, 'peak': peaks['bf16_tflops_sustained'], 'unit': 'TFLOP/s',
        'frac': ach_tf / peaks['bf16_tflops_sustained'], 'traffic': traffic,
        'algorithmic_flops_per_launch': float(flop_per_sample) * rows_per_launch,
        'algorithmic_bytes': row_bytes * rows_per_launch + 4.0 * eng.P * (rows_per_launch // w['batch_size']),   # sample rows read once + one gradient per minibatch step
        'peak_source': peaks['source'] + ' (cuBLAS bf16, sustained); fp32-equivalent FLOPs are counted once although the '
                       'bf16x3 mode executes 6 bf16 MMAs per product' if x3_path else peaks['source'] + ' (cuBLAS bf16, sustained)',
        'us_per_launch': ms_k * 1e3, 'us_per_minibatch_step': ms_k * 1e3 / (rows_per_launch // w['batch_size']),
        'mma_executed_tflops': ach_tf * 6.0 if x3_path else None,
        'ncu': ({'tensor_pipe_active_pct': 18.9, 'dram_bytes_per_launch': 218.8e6, 'source': 'profiles/r02_ncu_update_x3.md (ncu --set full, one launch)'}
                if (x3_path and O == 60 and args.algo == 'PPOLag') else None),
        'gae': {'kernel': 'gae_stream_kernel<TMA>', 'bound': 'hbm', 'achieved': gae_gbs, 'peak': peaks['hbm_gbs'],
                'unit': 'GB/s', 'frac': gae_gbs / peaks['hbm_gbs'], 'us_per_launch': ms_gae * 1e3, 'bytes_per_sample': 33,
                'note': 'T = 128: 17 MB, latency bound (one wave of 128 CTAs, one tile each)'},
        'gae_long_horizon': {'kernel': 'gae_stream_kernel<TMA>', 'bound': 'hbm', 'achieved': gae_long_gbs, 'peak': peaks['hbm_gbs'],
                             'unit': 'GB/s', 'frac': gae_long_gbs / peaks['hbm_gbs'], 'us_per_launch': ms_gae_long * 1e3,
                             'bytes_per_sample': 33, 'workload': f'T = {T_long} x {N} envs = {33 * T_long * N / 1e6:.0f} MB algorithmic (> L2), timed live with CUDA events'},
        'rollout_step': {'kernel': 'rollout_step_tc_kernel<bf16x3, persistent> (1 launch = 1 epoch)' if x3_path else ('rollout_step_tc_kernel<tf32, persistent> (1 launch = 1 epoch)' if args.precision == 'tf32' and O <= 64 else 'rollout_step_kernel'),
                         'bound': 'latency', 'us_per_step': ms_roll * 1e3 / (T + 1),
                         'achieved_tflops': (2 * (O * 64 + 64 * 64 + 64 * A) + 4 * (O * 64 + 64 * 64 + 64)) * N / (ms_roll * 1e-3 / (T + 1)) / 1e12,
                         'appended_bytes_per_step': row_bytes * N},
        'stage_ms': {'rollout': ms_roll, 'gae': ms_gae, 'update': ms_upd},
    }

    out = {
        'metric': f'env-steps/sec (rollout+GAE+update) {args.algo.replace("PPOLag", "PPO-Lag")}', 'value': value, 'unit': 'env-steps/s',
        'n_gpus': world, 'steps': args.steps, 'warmup': warm, 'ms_per_step': ms_per_step,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': DTYPES[args.precision] if (x3_path or args.precision != 'bf16x3') else DTYPES['fp32'] + ' [obs_dim > 64 is not on the bf16x3 path]',
        'data': 'synthetic',
        'config': {'workload': _workload_name(args.algo, O), 'algo': args.algo, 'obs_dim': O, 'envs_per_gpu': N, 'steps_per_env': T,
                   'global_samples_per_step': samples_global, 'parallelism': f'dp{world}', 'matmul_precision': args.precision,
                   'l2_policy': f'inputs larger than L2 (per-epoch slabs ~{(row_bytes + 48) * total / 1e6:.0f} MB > 126 MB)' if (row_bytes + 48) * total > 126e6
                   else 'per-epoch slabs fit L2; every epoch rewrites them (rollout) before the update reads them',
                   'noise': 'in-kernel Philox'},
        'e2e': e2e, 'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline,
    }
    if rank == 0 and world == 1 and not args.no_extras and args.precision == 'bf16x3':
        del algo
        alt = make('tf32')
        for _ in range(3):
            alt.train_epoch()
        ms_alt = timed(alt.train_epoch, max(3, args.steps // 2)) / max(3, args.steps // 2)
        out['extra'] = {'tf32': {'value': samples_global / (ms_alt * 1e-3), 'unit': 'env-steps/s', 'ms_per_step': ms_alt,
                                 'note': 'kind::tf32 tiles: 10-bit mantissa, certified only to 5e-3 -- NOT the headline'}}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out['cpu_baseline'] = cpu_baseline(args)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out if rank == 0 else {}


# ------------------------------------------------------------------------------------------------
def _oracle_epoch(state, n_envs: int, algo: str):
    """One epoch of the CPU restatement on n_envs envs (same T / update schedule)."""
    from oracle import gae as ogae
    from oracle import learner as ol
    from oracle import rollout as orollout

    w = WORKLOAD
    T, A = w['steps_per_env'], w['act_dim']
    eps = state['rng'].standard_normal((T, n_envs, A)).astype(np.float32)
    L = state['learner']
    theta = L.flat()
    window = state['window']
    sl = orollout.rollout_epoch(state['env'], state['norm'], theta, T, eps, window=window)
    out = ogae.dual_gae_slab(sl['rew'], sl['cost'], sl['val_r'], sl['val_c'], sl['flags'], sl['boot_r'], sl['boot_c'],
                             0.99, 0.95, 0.95)
    sr, sc = ogae.standardize(out['adv_r'], out['adv_c'])
    B = T * n_envs
    em = lambda x: np.ascontiguousarray(np.swapaxes(x, 0, 1)).reshape(B, *x.shape[2:])   # noqa: E731
    data = {'obs': em(sl['obs']), 'act': em(sl['act']), 'logp': em(sl['logp']), 'adv_r': em(sr), 'adv_c': em(sc),
            'target_value_r': em(out['tv_r']), 'target_value_c': em(out['tv_c'])}
    jc = float(np.mean([c for _, c, _ in window[-100:]]))
    bs = max(64, w['batch_size'] * n_envs // w['envs_per_gpu'])
    perms = [state['rng'].permutation(B) for _ in range(w['update_iters'])]
    if algo in ('PPOLag', 'FOCOPS'):
        lam = state['lagrange'].update(jc)
        L.update_ppo(data, perms, lam, batch_size=bs, focops={'lam': 1.5, 'eta': 0.02} if algo == 'FOCOPS' else None)
        return B
    # natural-gradient family: critics over the minibatches, then one full-batch actor step
    t = {k: torch.as_tensor(v) for k, v in data.items()}
    for perm in perms:
        perm = torch.as_tensor(np.asarray(perm, np.int64))
        for s in range(0, B, bs):
            idx = perm[s:s + bs]
            L.critic_step('reward_critic', t['obs'][idx], t['target_value_r'][idx], 0.001, 40.0)
            L.critic_step('cost_critic', t['obs'][idx], t['target_value_c'][idx], 0.001, 40.0)
    if algo == 'TRPOLag':
        lam = state['lagrange'].update(jc)
        adv = (t['adv_r'] - lam * t['adv_c']) / (1 + lam)
        ol.trpo_actor_step(L, t['obs'], t['act'], t['logp'], adv)
    else:  # CPO
        ol.cpo_actor_step(L, t['obs'], t['act'], t['logp'], t['adv_r'], t['adv_c'], jc - 25.0)
    return B


def _oracle_state(n_envs: int, obs_dim: int):
    from oracle import actor_critic as oac
    from oracle import learner as ol
    from oracle.normalizer import Normalizer
    from oracle.synthetic_env import SyntheticBoxEnv

    w = WORKLOAD
    return {'env': SyntheticBoxEnv(n_envs, obs_dim, w['act_dim'], max_episode_steps=w['max_episode_steps'], seed=0),
            'norm': Normalizer((obs_dim,)), 'learner': ol.Learner(oac.init_theta(obs_dim, w['act_dim'], 0), obs_dim, w['act_dim']),
            'lagrange': ol.Lagrange(25.0, 0.001, 0.035), 'rng': np.random.default_rng(0), 'window': []}


def _host_threads() -> int:
    """Threads for the CPU arm.  torch-CPU on these small layers collapses when oversubscribed
    (128 threads on the GPU box made one 64-env epoch take minutes), so the arm uses up to 16."""
    cores = os.cpu_count() or 1
    n = min(cores, 16)
    torch.set_num_threads(n)
    return n


REF_ENVS = WORKLOAD['envs_per_gpu']      # the reference arm runs the FULL per-GPU workload: same config as the GPU arm
REF_ENVS_SECOND_ORDER = 1024             # TRPOLag / CPO: 33 full-batch double-backward passes per epoch on the CPU -> a FIXED quarter


def _ref_envs(algo: str) -> int:
    return REF_ENVS if algo in ('PPOLag', 'FOCOPS') else min(REF_ENVS, REF_ENVS_SECOND_ORDER)


def cpu_baseline(args) -> dict:
    """The oracle port timed on the host cores: one full-size epoch (after a small warm-up epoch that pays for thread
    pool / allocator start-up)."""
    threads = _host_threads()
    _oracle_epoch(_oracle_state(128, args.obs_dim), 128, args.algo)
    n = _ref_envs(args.algo)
    st = _oracle_state(n, args.obs_dim)
    t0 = time.time(); B = _oracle_epoch(st, n, args.algo); dt = time.time() - t0
    return {'value': B / dt, 'unit': 'env-steps/s', 'cores': threads, 'kind': 'port',
            'sample': f'1 {args.algo} epoch (rollout+GAE+update, update_iters 8, batch 16384) on {n} envs x T=128 = {B} env-steps (fixed size; the GPU arm runs 4096), '
                      f'oracle/ torch-CPU+numpy restatement, {threads} torch threads of {os.cpu_count()} cores, {dt:.1f} s'}


def run_reference(args) -> dict:
    """--impl reference: the CPU restatement of the reference path on the host cores, every step one epoch of the
    same workload as the GPU arm (4096 envs x T = 128).  Under torchrun only rank 0 works."""
    if int(os.environ.get('RANK', '0')) != 0:
        return {}
    threads = _host_threads()
    steps, warm = args.steps, max(args.warmup, 1)
    n = _ref_envs(args.algo)
    _oracle_epoch(_oracle_state(128, args.obs_dim), 128, args.algo)        # thread pool / allocator start-up
    st = _oracle_state(n, args.obs_dim)
    for _ in range(min(warm, 2)):                     # epochs are seconds long: two warm-up epochs settle the caches
        _oracle_epoch(st, n, args.algo)
    t0 = time.time()
    done = 0
    for _ in range(steps):
        done += _oracle_epoch(st, n, args.algo)
    dt = time.time() - t0
    v = done / dt
    sample = (f'each step = 1 {args.algo} epoch (rollout+GAE+update, update_iters 8, batch 16384) on {n} envs x T=128 (fixed size; the GPU arm\'s per-GPU '
              f'workload is 4096 envs); oracle/ torch-CPU+numpy restatement of the reference path, {threads} torch threads of {os.cpu_count()} cores')
    return {'impl': 'reference', 'metric': f'env-steps/sec (rollout+GAE+update) {args.algo.replace("PPOLag", "PPO-Lag")}', 'value': v,
            'unit': 'env-steps/s', 'n_gpus': args.gpus, 'steps': steps, 'warmup': min(warm, 2),
            'ms_per_step': dt / steps * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': _workload_name(args.algo, args.obs_dim), 'algo': args.algo, 'obs_dim': args.obs_dim,
                       'envs_per_gpu': n, 'steps_per_env': WORKLOAD['steps_per_env'], 'sample_envs': n},
            'cpu_baseline': {'value': v, 'unit': 'env-steps/s', 'cores': threads, 'kind': 'port', 'sample': sample},
            'e2e': {'value': v, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--algo', default=WORKLOAD['algo'], choices=ALGOS)
    ap.add_argument('--obs-dim', type=int, default=WORKLOAD['obs_dim'])
    ap.add_argument('--precision', default='bf16x3', choices=['bf16x3', 'tf32', 'fp32'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the b200 path (--impl b200)')
    # stdout carries exactly ONE JSON line: whatever libraries print while the bench runs (e.g. NCCL's version banner, written
    # by C code straight to fd 1) is sent to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        out = run_reference(args) if args.impl == 'reference' else run_b200(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    if out:
        print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
