"""Record what the UNMODIFIED reference exposes to a drop-in replacement, as golden data:

    python tests/golden/make_golden_reference_api.py

* reference_configs.json   -- the `defaults` block of every upstream on-policy YAML that omnisafe_b200 ships, flattened
                              to dotted keys (tests/test_configs_ref_cpu.py);
* reference_evaluator.json -- what the reference Evaluator restores from a checkpoint written by omnisafe_b200: the
                              config entries it reads, the state-dict layout its actor and observation normaliser load
                              strictly, the normaliser statistics it ends up with and the deterministic action of the
                              loaded actor (tests/test_checkpoint_ref_cpu.py);
* reference_api.json       -- the algorithm registry, the on-policy namespace and the signatures that the import swap of
                              omnisafe_b200.integration relies on (tests/test_dropin_ref_cpu.py).

Like make_golden.py it needs the reference checkout (imported through oracle/ref_shim.py); the tests read only the
recorded files.
"""
from __future__ import annotations

import inspect
import json
import os
import sys
import tempfile

import torch
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden  # noqa: E402,F401  (installs the reference shim and registers RefSyntheticBox)

from oracle import ref_shim  # noqa: E402

MINE = os.path.join(make_golden.ROOT, 'omnisafe_b200', 'configs', 'on-policy')

# the config.json entries the reference Evaluator reads for an on-policy Box agent (omnisafe/evaluator.py:L113-303, L386-395)
EVALUATOR_CONFIG_KEYS = ('algo', 'env_id', 'env_cfgs', 'algo_cfgs.obs_normalize', 'model_cfgs.actor_type',
                         'model_cfgs.actor.hidden_sizes', 'model_cfgs.actor.activation',
                         'model_cfgs.weight_initialization_mode')


def flat(d, pre=''):
    out = {}
    for k, v in d.items():
        if isinstance(v, dict):
            out.update(flat(v, pre + k + '.'))
        else:
            out[pre + k] = v
    return out


def lookup(d, dotted):
    for k in dotted.split('.'):
        d = d[k]
    return d


def write_checkpoint(log_dir):
    """A PPOLag checkpoint written by omnisafe_b200 (CPU tensors, no kernel launch): obs 12 / act 3, the oracle's
    seed-3 parameters, a non-trivial observation normaliser.  Returns the run directory."""
    from omnisafe_b200.common.logger import Logger
    from omnisafe_b200.common.normalizer import Normalizer
    from omnisafe_b200.models import ConstraintActorCritic
    from omnisafe_b200.utils.config import get_default_kwargs_yaml
    from oracle import actor_critic as oac

    O, A = 12, 3
    cfgs = get_default_kwargs_yaml('PPOLag', 'SyntheticBox-v0', 'on-policy')
    cfgs.recurisve_update({'exp_name': 'PPOLag-{SyntheticBox-v0}', 'env_id': 'SyntheticBox-v0', 'algo': 'PPOLag',
                           'env_cfgs': {'obs_dim': O, 'act_dim': A, 'max_episode_steps': 8, 'term_prob': 0.0},
                           'logger_cfgs': {'log_dir': log_dir}, 'train_cfgs': {'epochs': 1}})
    ac = ConstraintActorCritic(O, A, cfgs.model_cfgs, epochs=1, device='cpu')
    ac.load_flat(oac.init_theta(O, A, seed=3))
    norm = Normalizer((O,), clip=5.0, device='cpu')
    norm.mean.copy_(torch.linspace(-0.2, 0.2, O)); norm.std.fill_(1.5); norm.sumsq.fill_(2.25 * 99); norm.count[0] = 100
    logger = Logger(log_dir, cfgs.exp_name, seed=0, config=cfgs)
    logger.setup_torch_saver({'pi': ac.actor_state_dict, 'obs_normalizer': norm})
    logger.torch_save()
    logger.close()
    return logger.log_dir


def gen_configs():
    ref = os.path.join(ref_shim.REFERENCE_ROOT, 'omnisafe', 'configs', 'on-policy')
    out = {}
    for name in sorted(f[:-5] for f in os.listdir(MINE) if f.endswith('.yaml')):
        with open(os.path.join(ref, name + '.yaml')) as fh:
            out[name] = flat(yaml.safe_load(fh)['defaults'])
    with open(os.path.join(HERE, 'reference_configs.json'), 'w') as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write('\n')


def gen_evaluator():
    from omnisafe.evaluator import Evaluator

    with tempfile.TemporaryDirectory() as tmp:
        run_dir = write_checkpoint(tmp)
        with open(os.path.join(run_dir, 'config.json')) as fh:
            cfg = json.load(fh)
        ev = Evaluator()
        ev.load_saved(save_dir=run_dir, model_name='epoch-0.pt')
    obs = torch.linspace(-1, 1, 12).reshape(1, 12)
    with torch.no_grad():
        act = ev._actor.predict(obs, deterministic=True)
    w = ev._env
    while not hasattr(w, '_obs_normalizer'):
        w = w._env
    nz = w._obs_normalizer
    out = {
        'config': {k: lookup(cfg, k) for k in EVALUATOR_CONFIG_KEYS},
        'pi_state_dict': {k: list(v.shape) for k, v in ev._actor.state_dict().items()},
        'obs_normalizer_state_dict': {k: list(v.shape) for k, v in nz.state_dict().items()},
        'obs_normalizer_mean': nz.mean.tolist(), 'obs_normalizer_std': nz.std.tolist(),
        'obs': obs.reshape(-1).tolist(), 'act': act.reshape(-1).tolist(),
    }
    with open(os.path.join(HERE, 'reference_evaluator.json'), 'w') as fh:
        json.dump(out, fh, indent=1)
        fh.write('\n')


def gen_api():
    import omnisafe.algorithms.on_policy as ref_on_policy
    from omnisafe.algorithms import registry
    from omnisafe.algorithms.base_algo import BaseAlgo
    from omnisafe.common.lagrange import Lagrange

    out = {
        'registry': sorted(registry.REGISTRY._module_dict),
        'on_policy_classes': sorted(n for n in dir(ref_on_policy) if isinstance(getattr(ref_on_policy, n), type)),
        'base_algo_init': list(inspect.signature(BaseAlgo.__init__).parameters),
        'lagrange_update_lagrange_multiplier': list(inspect.signature(Lagrange.update_lagrange_multiplier).parameters),
    }
    with open(os.path.join(HERE, 'reference_api.json'), 'w') as fh:
        json.dump(out, fh, indent=1)
        fh.write('\n')


if __name__ == '__main__':
    torch.set_num_threads(1)
    gen_configs()
    gen_evaluator()
    gen_api()
    print('reference API fixtures written to', HERE)
