"""Warm-up task construction (mirror of morl/warm_up.py:24-77): one randomly initialised policy per evenly spaced
scalarisation weight, with its PPO agent, a snapshot of the environment's running normalisation, and its evaluated
objectives. Policies are created on the device; environments come from the hooks of pgmorl_b200.mopg."""
from copy import deepcopy

import torch

from . import mopg
from .a2c_ppo_acktr import algo
from .a2c_ppo_acktr.model import Policy
from .sample import Sample
from .scalarization_methods import WeightedSumScalarization
from .utils import generate_weights_batch_dfs


def initialize_warm_up_batch(args, device):
    """-> (sample_batch, scalarization_batch), one entry per weight of the simplex grid
    [min_weight, max_weight] with step delta_weight (warm_up.py:26-27)."""
    if args.algo != 'ppo':
        raise NotImplementedError("only PPO is part of the PG-MORL path (warm_up.py:42-54)")
    device = torch.device(device)
    weights_batch = []
    generate_weights_batch_dfs(0, args.obj_num, args.min_weight, args.max_weight, args.delta_weight, [], weights_batch)
    probe = mopg._gym_make(args.env_name)                     # only read for the observation / action spaces
    sample_batch, scalarization_batch = [], []
    for weights in weights_batch:
        # same construction order as the reference: policy (consumes torch's global RNG for the orthogonal init),
        # agent, then a throw-away vectorised env whose initial running moments become the sample's env_params
        actor_critic = Policy(probe.observation_space.shape, probe.action_space,
                              base_kwargs={'layernorm': args.layernorm, 'hidden_size': getattr(args, 'hidden_size', 64)},
                              obj_num=args.obj_num, device=device)
        actor_critic.to(device).double()
        agent = algo.PPO(actor_critic, args.clip_param, args.ppo_epoch, args.num_mini_batch, args.value_loss_coef,
                         args.entropy_coef, lr=args.lr, eps=1e-5, max_grad_norm=args.max_grad_norm)
        envs = mopg._make_vec_envs(env_name=args.env_name, seed=args.seed, num_processes=args.num_processes,
                                   gamma=args.gamma, log_dir=None, device=device, allow_early_resets=False,
                                   obj_rms=args.obj_rms, ob_rms=args.ob_rms)
        env_params = {key: (deepcopy(getattr(envs, key)) if getattr(envs, key) is not None else None)
                      for key in ('ob_rms', 'ret_rms', 'obj_rms')}
        envs.close()
        sample = Sample(env_params, actor_critic, agent, optgraph_id=-1)
        sample.objs = mopg.evaluation(args, sample)
        sample_batch.append(sample)
        scalarization_batch.append(WeightedSumScalarization(num_objs=args.obj_num, weights=weights))
    probe.close()
    return sample_batch, scalarization_batch
