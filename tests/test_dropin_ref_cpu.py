"""INTEGRATION.md §2 executed: the import swap of omnisafe_b200.integration applied to a stand-in of the upstream
`omnisafe` package that carries the upstream algorithm registry, on-policy namespace and signatures recorded from the
unmodified reference in tests/golden/reference_api.json (tests/golden/make_golden_reference_api.py).  The upstream
`omnisafe.Agent` looks the class up in that registry and calls it with (env_id, cfgs) built from the upstream YAML; the
same call on the swapped registry reaches the omnisafe_b200 class -- up to its device check (the path has no CPU
fallback)."""
import inspect
import json
import os
import sys
import types

import pytest


def _stand_in_reference(api, monkeypatch):
    """`omnisafe`, `omnisafe.algorithms[.registry|.on_policy]` and `omnisafe.envs.core` with the recorded upstream names."""
    class Registry:
        def __init__(self, names):
            self._module_dict = {n: type(n, (), {}) for n in names}

        def get(self, name):
            return self._module_dict[name]

    class EnvRegistry:
        def __init__(self):
            self.registered = []

        def register(self, cls):
            self.registered.append(cls)
            return cls

    mods = {n: types.ModuleType(n) for n in ('omnisafe', 'omnisafe.algorithms', 'omnisafe.algorithms.registry',
                                             'omnisafe.algorithms.on_policy', 'omnisafe.envs', 'omnisafe.envs.core')}
    mods['omnisafe.algorithms.registry'].REGISTRY = Registry(api['registry'])
    for name in api['on_policy_classes']:
        cls = mods['omnisafe.algorithms.registry'].REGISTRY.get(name)
        setattr(mods['omnisafe.algorithms.on_policy'], name, cls)
        setattr(mods['omnisafe.algorithms'], name, cls)
    core = mods['omnisafe.envs.core']
    core.CMDP = type('CMDP', (), {})
    core.ENV_REGISTRY = EnvRegistry()
    core.support_envs = lambda: [e for c in core.ENV_REGISTRY.registered for e in c._support_envs]
    for parent, child in (('omnisafe', 'algorithms'), ('omnisafe', 'envs'), ('omnisafe.algorithms', 'registry'),
                          ('omnisafe.algorithms', 'on_policy'), ('omnisafe.envs', 'core')):
        setattr(mods[parent], child, mods[f'{parent}.{child}'])
    for name, mod in mods.items():
        monkeypatch.setitem(sys.modules, name, mod)
    return mods


def test_reference_agent_constructs_the_accelerated_class(golden_dir, tmp_path, monkeypatch):
    import omnisafe_b200
    import omnisafe_b200.integration as integ
    from omnisafe_b200.algorithms import on_policy as mine
    from omnisafe_b200.utils.config import Config, recursive_check_config

    with open(os.path.join(golden_dir, 'reference_api.json')) as fh:
        api = json.load(fh)
    mods = _stand_in_reference(api, monkeypatch)
    ref_registry = mods['omnisafe.algorithms.registry'].REGISTRY

    upstream = ref_registry.get('PPOLag')
    swapped = integ.install(mods['omnisafe'])
    assert {'PPOLag', 'CPO', 'TRPOLag', 'FOCOPS', 'PPO', 'TRPO', 'PCPO', 'RCPO', 'PDO'} <= set(swapped)
    assert swapped == sorted(integ.accelerated_classes())                  # every accelerated class has an upstream name
    assert ref_registry.get('PPOLag') is mine.PPOLag and ref_registry.get('PPOLag') is not upstream
    for name in swapped:
        assert ref_registry.get(name) is getattr(mine, name), name
        assert getattr(mods['omnisafe.algorithms.on_policy'], name) is getattr(mine, name), name
        assert getattr(mods['omnisafe.algorithms'], name) is getattr(mine, name), name
    # the HBM-resident env id is known to the upstream env table, and is not steppable on the host
    (placeholder,) = mods['omnisafe.envs.core'].ENV_REGISTRY.registered
    assert placeholder._support_envs == ['SyntheticBox-v0']
    with pytest.raises(RuntimeError, match='stepped in-kernel'):
        placeholder('SyntheticBox-v0')
    # same constructor contract as BaseAlgo (algorithms/base_algo.py:L34-53): (env_id, cfgs)
    assert list(inspect.signature(mine.PPOLag.__init__).parameters) == api['base_algo_init']
    # the reference's Agent: upstream PPOLag.yaml + custom_cfgs, then registry.get(algo)(env_id, cfgs)
    custom = {'train_cfgs': {'vector_env_nums': 8, 'total_steps': 8 * 16 * 2},
              'algo_cfgs': {'steps_per_epoch': 8 * 16, 'batch_size': 32, 'update_iters': 2},
              'logger_cfgs': {'use_tensorboard': False, 'use_wandb': False, 'log_dir': str(tmp_path)}}
    with open(os.path.join(golden_dir, 'reference_configs.json')) as fh:
        upstream_yaml = {}
        for dotted, v in json.load(fh)['PPOLag'].items():
            *path, leaf = dotted.split('.')
            d = upstream_yaml
            for k in path:
                d = d.setdefault(k, {})
            d[leaf] = v
    recursive_check_config(custom, upstream_yaml)
    cfgs = Config.dict2config(upstream_yaml)
    cfgs.recurisve_update({**custom, 'exp_name': 'PPOLag-{SyntheticBox-v0}', 'env_id': 'SyntheticBox-v0', 'algo': 'PPOLag'})
    with pytest.raises(RuntimeError, match='omnisafe_b200 runs this path as sm_100a CUDA kernels only'):
        ref_registry.get('PPOLag')(env_id='SyntheticBox-v0', cfgs=cfgs)    # default device 'cpu' -> OUR class refuses
    # an unknown custom key is rejected before the class is reached
    with pytest.raises(KeyError):
        omnisafe_b200.Agent('PPOLag', 'SyntheticBox-v0', custom_cfgs={'algo_cfgs': {'no_such_key': 1}})
    # the accelerated Lagrange keeps the reference signature update_lagrange_multiplier(Jc: float)
    from omnisafe_b200.common.lagrange import Lagrange
    assert list(inspect.signature(Lagrange.update_lagrange_multiplier).parameters) == \
        api['lagrange_update_lagrange_multiplier']
