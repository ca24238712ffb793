"""CPU: every shipped YAML `defaults` block equals the upstream block of the same algorithm key for key (plus the
`matmul_precision` extension and the env_cfgs placeholder).  The upstream blocks are recorded from the unmodified
reference in tests/golden/reference_configs.json (tests/golden/make_golden_reference_api.py)."""
import json
import os

import yaml

MINE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'omnisafe_b200', 'configs', 'on-policy')


def _flat(d, pre=''):
    out = {}
    for k, v in d.items():
        if isinstance(v, dict):
            out.update(_flat(v, pre + k + '.'))
        else:
            out[pre + k] = v
    return out


def test_yaml_defaults_equal_upstream(golden_dir):
    from omnisafe_b200.algorithms import ALGORITHMS

    with open(os.path.join(golden_dir, 'reference_configs.json')) as fh:
        upstream = json.load(fh)
    names = sorted(f[:-5] for f in os.listdir(MINE) if f.endswith('.yaml'))
    assert set(names) == set(ALGORITHMS['on-policy'])          # one YAML per registered class
    assert set(names) == set(upstream)                          # and one recorded upstream block per YAML
    for name in names:
        ref = upstream[name]
        with open(os.path.join(MINE, name + '.yaml')) as fh:
            doc = yaml.safe_load(fh)
        mine = _flat(doc['defaults'])
        assert mine.pop('train_cfgs.matmul_precision') == 'fp32', name        # parity arithmetic by default
        assert mine == ref, (name, {k: (ref.get(k), mine.get(k)) for k in set(ref) | set(mine) if ref.get(k) != mine.get(k)})
        assert 'SyntheticBox-v0' in doc                                           # the B200 workload block
