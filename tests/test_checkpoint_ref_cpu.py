"""CPU: a checkpoint written by omnisafe_b200 (same classes, CPU tensors, no kernel launch) holds what the UNMODIFIED
reference Evaluator (`omnisafe/evaluator.py:L113-303`) loads.  tests/golden/reference_evaluator.json records, from the
reference Evaluator loading this very checkpoint (tests/golden/make_golden_reference_api.py), the config entries it
reads, the state-dict layout its actor and observation normaliser load strictly, the statistics it restored and the
deterministic action of the restored actor."""
import json
import os

import numpy as np
import torch


def _forward(sd, obs, activation):
    """The reference's Gaussian actor mean (Linear, act, Linear, act, Linear) straight from a checkpoint's state dict."""
    act = {'tanh': torch.tanh, 'relu': torch.relu}[activation]
    layers = sorted({int(k.split('.')[1]) for k in sd if k.startswith('mean.')})
    x = obs
    for j, i in enumerate(layers):
        x = x @ sd[f'mean.{i}.weight'].T + sd[f'mean.{i}.bias']
        if j < len(layers) - 1:
            x = act(x)
    return x


def test_reference_evaluator_loads_our_checkpoint(tmp_path, golden_dir):
    from omnisafe_b200.common.logger import Logger
    from omnisafe_b200.common.normalizer import Normalizer
    from omnisafe_b200.models import ConstraintActorCritic
    from omnisafe_b200.utils.config import get_default_kwargs_yaml
    from oracle import actor_critic as oac

    with open(os.path.join(golden_dir, 'reference_evaluator.json')) as fh:
        ref = json.load(fh)
    O, A = 12, 3
    cfgs = get_default_kwargs_yaml('PPOLag', 'SyntheticBox-v0', 'on-policy')
    cfgs.recurisve_update({'exp_name': 'PPOLag-{SyntheticBox-v0}', 'env_id': 'SyntheticBox-v0', 'algo': 'PPOLag',
                           'env_cfgs': {'obs_dim': O, 'act_dim': A, 'max_episode_steps': 8, 'term_prob': 0.0},
                           'logger_cfgs': {'log_dir': str(tmp_path)}, 'train_cfgs': {'epochs': 1}})
    ac = ConstraintActorCritic(O, A, cfgs.model_cfgs, epochs=1, device='cpu')
    theta = oac.init_theta(O, A, seed=3)
    ac.load_flat(theta)
    norm = Normalizer((O,), clip=5.0, device='cpu')
    norm.mean.copy_(torch.linspace(-0.2, 0.2, O)); norm.std.fill_(1.5); norm.sumsq.fill_(2.25 * 99); norm.count[0] = 100
    logger = Logger(str(tmp_path), cfgs.exp_name, seed=0, config=cfgs)
    logger.setup_torch_saver({'pi': ac.actor_state_dict, 'obs_normalizer': norm})
    logger.torch_save()
    logger.close()

    # the config entries the Evaluator reads hold what the reference read from the same run
    with open(os.path.join(logger.log_dir, 'config.json')) as fh:
        cfg = json.load(fh)
    for dotted, want in ref['config'].items():
        got = cfg
        for k in dotted.split('.'):
            got = got[k]
        assert got == want, dotted
    # the reference loads both state dicts strictly: same keys, same shapes
    ckpt = torch.load(os.path.join(logger.log_dir, 'torch_save', 'epoch-0.pt'), weights_only=False)
    for key, layout in (('pi', ref['pi_state_dict']), ('obs_normalizer', ref['obs_normalizer_state_dict'])):
        assert {k: list(v.shape) for k, v in ckpt[key].items()} == layout, key
    # the reference actor restored from OUR parameters: same deterministic action as the oracle forward
    obs = torch.tensor(ref['obs'], dtype=torch.float32).reshape(1, O)
    act_ref = np.asarray(ref['act'], np.float32).reshape(1, A)
    with torch.no_grad():
        np.testing.assert_allclose(_forward(ckpt['pi'], obs, cfg['model_cfgs']['actor']['activation']).numpy(), act_ref,
                                   rtol=1e-6, atol=1e-6)
    nets = oac.unflatten(torch.as_tensor(theta), O, A)
    np.testing.assert_allclose(act_ref, oac.mlp(nets['actor'], obs).numpy(), rtol=1e-6, atol=1e-6)
    # and the reference's wrapper stack normalised with OUR statistics
    np.testing.assert_allclose(ref['obs_normalizer_mean'], norm.mean.numpy())
    np.testing.assert_allclose(ref['obs_normalizer_std'], norm.std.numpy())
    np.testing.assert_allclose(ckpt['obs_normalizer']['_mean'].numpy(), norm.mean.numpy())
    np.testing.assert_allclose(ckpt['obs_normalizer']['_std'].numpy(), norm.std.numpy())
