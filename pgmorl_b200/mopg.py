"""MOPG worker with the reference's contract (morl/mopg.py:25-182) and its population-batched form.

`MOPG_worker(args, task_id, task, device, iteration, num_updates, start_time, results_queue, done_event)`
keeps the signature and the queue protocol of the reference: every `update_iter` iterations (and at the end)
it puts {'task_id', 'offspring_batch': np.ndarray[object] of Sample, 'done'} on `results_queue`, then waits on
`done_event`. Inside, rollout inference, GAE/advantage and the PPO update run on the GPU (K1, K2, K3).

`mopg_population_update(args, task_batch, ...)` advances ALL tasks of this GPU's shard together: one K1 launch
per environment step for every task's observations, then one K2 and one K3 launch per iteration for the whole
population -- the form the bench measures. Environment stepping (MuJoCo) stays on the host and is out of scope;
environments are created through the hooks below (defaults: the reference's own factories when importable).
"""
import time
from collections import deque
from copy import deepcopy

import numpy as np
import torch

from . import kernels as K
from ._lib import PpoHyper
from .a2c_ppo_acktr import utils
from .a2c_ppo_acktr.storage import RolloutStorage
from .population_state import PopulationMOPG
from .sample import Sample

_HOOKS = {"make_vec_envs": None, "gym_make": None, "make_raw_vec_envs": None}


def set_env_hooks(make_vec_envs=None, gym_make=None, make_raw_vec_envs=None):
    """Install the environment factories (signature of a2c_ppo_acktr.envs.make_vec_envs / gym.make).
    `make_raw_vec_envs(**same kwargs)` returns vectorised environments WITHOUT the VecNormalize wrapper:
    `reset() -> raw obs [N,O]`, `step(actions) -> (raw obs [N,O] f64, raw scalar rewards [N], done [N], infos with the raw
    'obj' vector and optionally 'bad_transition')`. When it is installed, `mopg_population_update` keeps the running
    normalisation on the device (K6, vec_normalize.DeviceVecNormalize, SURVEY 8(f2)); pass `False` to uninstall."""
    if make_vec_envs is not None:
        _HOOKS["make_vec_envs"] = make_vec_envs
    if gym_make is not None:
        _HOOKS["gym_make"] = gym_make
    if make_raw_vec_envs is not None:
        _HOOKS["make_raw_vec_envs"] = make_raw_vec_envs or None


def _make_vec_envs(**kw):
    if _HOOKS["make_vec_envs"] is None:
        from a2c_ppo_acktr.envs import make_vec_envs as ref_factory      # the reference's factory, if installed
        _HOOKS["make_vec_envs"] = ref_factory
    return _HOOKS["make_vec_envs"](**kw)


def _gym_make(name):
    if _HOOKS["gym_make"] is None:
        import gym
        _HOOKS["gym_make"] = gym.make
    return _HOOKS["gym_make"](name)


def _step_noise(N, dims):
    """The action noise of one environment step, drawn from torch's global CPU generator as the reference's
    dist.sample() draws it: normal_(0,1) [N,A] for a Gaussian head, exponential_(1) [N,n] for a Categorical head
    (torch.multinomial's single-sample path), float64."""
    eps = torch.empty(N, dims.act, dtype=torch.float64)
    return eps.exponential_(1) if dims.categorical else eps.normal_(0, 1)


def _env_actions(act, dims):
    """Actions as the environments receive them: int64 category indices [.., 1] for a Categorical head (the reference's
    VecPyTorch.step_async squeezes a LongTensor), the float32 block otherwise."""
    return act.to(torch.int64) if dims.categorical else act


def evaluation(args, sample):
    """Average (optionally discounted) objective vector of `eval_num` deterministic episodes (mopg.py:25-46)."""
    eval_env = _gym_make(args.env_name)
    objs = np.zeros(args.obj_num)
    ob_rms = sample.env_params['ob_rms']
    policy = sample.actor_critic
    with torch.no_grad():
        for eval_id in range(args.eval_num):
            eval_env.seed(args.seed + eval_id)
            ob = eval_env.reset()
            done = False
            gamma = 1.0
            while not done:
                if args.ob_rms:
                    ob = np.clip((ob - ob_rms.mean) / np.sqrt(ob_rms.var + 1e-8), -10.0, 10.0)
                _, action, _, _ = policy.act(torch.Tensor(ob).unsqueeze(0), None, None, deterministic=True)
                ob, _, done, info = eval_env.step(action.cpu())
                objs += gamma * info['obj']
                if not args.raw:
                    gamma *= args.gamma
    eval_env.close()
    objs /= args.eval_num
    return objs


def evaluation_batch(args, samples):
    """`evaluation` of several samples at once (SURVEY section 8(f2)): the same episodes, seeds and per-sample arithmetic
    as mopg.py:25-46, with the evaluation environments of all samples stepped in lockstep so that every environment step
    costs ONE K1 launch (deterministic mode, one row per sample) and one read-back instead of one per sample.
    Samples whose episode has ended wait for the others; their rows are computed and ignored. Returns a list of
    objective vectors, identical to [evaluation(args, s) for s in samples]."""
    P = len(samples)
    if P == 0:
        return []
    policy0 = samples[0].actor_critic
    dims, device = policy0.dims, policy0.device
    flat = torch.stack([s.actor_critic.flat for s in samples]).contiguous()
    envs = [_gym_make(args.env_name) for _ in samples]
    objs = [np.zeros(args.obj_num) for _ in samples]
    host_obs = torch.zeros(P, 1, dims.obs, dtype=torch.float32).pin_memory()
    dev_obs = torch.empty(P, 1, dims.obs, dtype=torch.float32, device=device)
    out = None
    with torch.no_grad():
        for eval_id in range(args.eval_num):
            obs = []
            for env in envs:
                env.seed(args.seed + eval_id)
                obs.append(env.reset())
            running = list(range(P))
            gamma = [1.0] * P
            while running:
                for p in running:
                    ob = obs[p]
                    if args.ob_rms:
                        ob_rms = samples[p].env_params['ob_rms']
                        ob = np.clip((ob - ob_rms.mean) / np.sqrt(ob_rms.var + 1e-8), -10.0, 10.0)
                    host_obs[p, 0] = torch.Tensor(ob)
                dev_obs.copy_(host_obs, non_blocking=True)
                out = K.policy_forward(flat, dev_obs, dims, mode=K.ACT_DETERMINISTIC, out=out)
                action = _env_actions(out[1].cpu(), dims)
                still = []
                for p in running:
                    obs[p], _, done, info = envs[p].step(action[p])
                    objs[p] += gamma[p] * info['obj']
                    if not args.raw:
                        gamma[p] *= args.gamma
                    if not done:
                        still.append(p)
                running = still
    for env in envs:
        env.close()
    return [o / args.eval_num for o in objs]


def _restore_rms(envs, env_params):
    for key in ('ob_rms', 'ret_rms', 'obj_rms'):
        if env_params[key] is not None:
            setattr(envs.venv, key, deepcopy(env_params[key]))


def _snapshot_rms(envs):
    return {key: (deepcopy(getattr(envs, key)) if getattr(envs, key) is not None else None)
            for key in ('ob_rms', 'ret_rms', 'obj_rms')}


def MOPG_worker(args, task_id, task, device, iteration, num_updates, start_time, results_queue, done_event):
    """One task, reference contract (mopg.py:60-182)."""
    scalarization = task.scalarization
    env_params, actor_critic, agent = task.sample.env_params, task.sample.actor_critic, task.sample.agent
    envs = _make_vec_envs(env_name=args.env_name, seed=args.seed, num_processes=args.num_processes, gamma=args.gamma,
                          log_dir=None, device=device, allow_early_resets=False, obj_rms=args.obj_rms, ob_rms=args.ob_rms)
    _restore_rms(envs, env_params)
    rollouts = RolloutStorage(num_steps=args.num_steps, num_processes=args.num_processes,
                              obs_shape=envs.observation_space.shape, action_space=envs.action_space,
                              recurrent_hidden_state_size=actor_critic.recurrent_hidden_state_size,
                              obj_num=args.obj_num, device=actor_critic.flat.device)
    obs = envs.reset()
    rollouts.obs[0].copy_(torch.as_tensor(obs).to(rollouts.obs.device, torch.float32))
    episode_rewards = deque(maxlen=10)
    total_num_updates = int(args.num_env_steps) // args.num_steps // args.num_processes
    offspring_batch = []
    start_iter, final_iter = iteration, min(iteration + num_updates, total_num_updates)
    for j in range(start_iter, final_iter):
        torch.manual_seed(j)
        if args.use_linear_lr_decay:
            utils.update_linear_schedule(agent.optimizer, j * args.lr_decay_ratio, total_num_updates, args.lr)
        for step in range(args.num_steps):
            with torch.no_grad():
                value, action, action_log_prob, rhs = actor_critic.act(rollouts.obs[step], None, rollouts.masks[step])
            obs, _, done, infos = envs.step(action.cpu())
            obj_tensor = torch.zeros([args.num_processes, args.obj_num], dtype=torch.float64)
            for idx, info in enumerate(infos):
                obj_tensor[idx] = torch.from_numpy(np.asarray(info['obj'], dtype=np.float64))
                if 'episode' in info.keys():
                    episode_rewards.append(info['episode']['r'])
            masks = torch.FloatTensor([[0.0] if done_ else [1.0] for done_ in done])
            bad_masks = torch.FloatTensor([[0.0] if 'bad_transition' in info.keys() else [1.0] for info in infos])
            rollouts.insert(obs, rollouts.recurrent_hidden_states[step + 1], action, action_log_prob, value,
                            obj_tensor, masks, bad_masks)
        with torch.no_grad():
            next_value = actor_critic.get_value(rollouts.obs[-1], None, rollouts.masks[-1])
        rollouts.compute_returns(next_value, args.use_gae, args.gamma, args.gae_lambda, args.use_proper_time_limits)
        obj_rms_var = envs.obj_rms.var if envs.obj_rms is not None else None
        agent.update(rollouts, scalarization, obj_rms_var)
        rollouts.after_update()
        sample = Sample(_snapshot_rms(envs), deepcopy(actor_critic), deepcopy(agent))
        sample.objs = evaluation(args, sample)
        offspring_batch.append(sample)
        if args.rl_log_interval > 0 and (j + 1) % args.rl_log_interval == 0 and len(episode_rewards) > 1 and task_id == 0:
            total_num_steps = (j + 1) * args.num_processes * args.num_steps
            end = time.time()
            print("[RL] Updates {}, num timesteps {}, FPS {}, time {:.2f} seconds".format(
                j + 1, total_num_steps, int(total_num_steps / (end - start_time)), end - start_time))
        if (j + 1) % args.update_iter == 0 or j == final_iter - 1:
            results_queue.put({'task_id': task_id, 'offspring_batch': np.array(offspring_batch),
                               'done': j == final_iter - 1})
            offspring_batch = []
    envs.close()
    done_event.wait()


_POP_CACHE = {}


def _population(dims, P, args, hyper, dev, cluster, clipped_value_loss=True):
    """The device-resident population shard of this (shape, size, schedule, PPO options): rollout buffers, K3 workspace,
    pinned staging and the captured per-step graphs are allocated ONCE and reused by every generation (SURVEY 8(f1)).
    The return branch is args.use_gae / args.use_proper_time_limits (default: GAE with proper time limits, as the
    reference's run.py:56-70 sets them)."""
    from .rollout import StepPipe
    use_gae, use_ptl = bool(getattr(args, "use_gae", True)), bool(getattr(args, "use_proper_time_limits", True))
    key = (dims, P, args.num_steps, args.num_processes, args.ppo_epoch, args.num_mini_batch, args.gamma, args.gae_lambda,
           str(dev), cluster, use_gae, use_ptl, bool(clipped_value_loss))
    hit = _POP_CACHE.get(key)
    if hit is None:
        if len(_POP_CACHE) >= 4:                       # a run alternates between at most a few shard sizes
            _POP_CACHE.pop(next(iter(_POP_CACHE)))
        pop = PopulationMOPG(dims, P, args.num_steps, args.num_processes, ppo_epoch=args.ppo_epoch,
                             num_mini_batch=args.num_mini_batch, gamma=args.gamma, gae_lambda=args.gae_lambda,
                             hyper=hyper, device=dev, cluster=cluster, use_gae=use_gae, use_proper_time_limits=use_ptl,
                             clipped_value_loss=bool(clipped_value_loss))
        hit = _POP_CACHE[key] = {"pop": pop, "pipe": StepPipe(pop), "raw": None}
    hit["pop"].hyper = hyper
    return hit


def _snapshot_samples(task_batch, pop, lr, env_params_of):
    """One Sample per task from the device state (mopg.py:146-149): the policy / Adam tensors are clones of the shard's
    rows, everything else is copied from the task's sample."""
    out = []
    step = pop.adam_step.tolist()
    for p, task in enumerate(task_batch):
        ac, agent = deepcopy(task.sample.actor_critic), deepcopy(task.sample.agent)
        ac.flat = pop.params[p].clone()
        agent.optimizer.exp_avg, agent.optimizer.exp_avg_sq = pop.adam_m[p].clone(), pop.adam_v[p].clone()
        agent.optimizer.step_count = int(step[p])
        agent.optimizer.param_groups[0]['lr'] = lr
        out.append(Sample(env_params_of(p), ac, agent))
    return out


def _population_update_raw(args, task_batch, cache, device, start_iter, final_iter, total_num_updates, stats):
    """The rollout loop of `mopg_population_update` with the normalisation on the device: the host only steps the raw
    simulators; per environment step ONE graph replay (rollout.StepPipe) uploads their answer, K6 turns it into the
    normalised observation / reward / mask slots of the rollout buffers and K1 acts on the new observation."""
    from .rollout import StepPipe
    from .vec_normalize import DeviceVecNormalize
    pop = cache["pop"]
    P, T, N, M = len(task_batch), args.num_steps, args.num_processes, args.obj_num
    dims = pop.dims
    kw = dict(env_name=args.env_name, seed=args.seed, num_processes=N, gamma=args.gamma, log_dir=None, device=device,
              allow_early_resets=False, obj_rms=args.obj_rms, ob_rms=args.ob_rms)
    envs_all = [_HOOKS["make_raw_vec_envs"](**kw) for _ in task_batch]
    # a2c/envs.py:86-91: VecNormalize(ret=False) without a discount, else VecNormalize(gamma=...); ob / obj moments optional
    sig = (bool(args.ob_rms), args.gamma is not None, bool(args.obj_rms), args.gamma)
    if cache["raw"] is None or cache["raw"]["sig"] != sig:
        vn = DeviceVecNormalize(P, N, dims.obs, M, ob=args.ob_rms, ret=args.gamma is not None, obj_rms=args.obj_rms,
                                gamma=args.gamma if args.gamma is not None else 0.99, device=pop.device)
        cache["raw"] = {"sig": sig, "vn": vn, "pipe": StepPipe(pop, vn)}
    vn, pipe = cache["raw"]["vn"], cache["raw"]["pipe"]
    vn.reset_state()
    for p, task in enumerate(task_batch):
        vn.load_task(p, task.sample.env_params)
    vn.reset(np.stack([np.asarray(e.reset(), dtype=np.float64) for e in envs_all]), pop.obs[:, 0:N])
    offspring = [[] for _ in range(P)]
    raw_obs, raw_rew, raw_obj = pipe.h_raw_obs.numpy(), pipe.h_raw_rew.numpy(), pipe.h_raw_obj.numpy()
    done_h, bad_h = pipe.h_done.numpy(), pipe.h_bad.numpy()
    for j in range(start_iter, final_iter):
        torch.manual_seed(j)
        lr = args.lr - (args.lr * ((j * args.lr_decay_ratio) / float(total_num_updates))) if args.use_linear_lr_decay else args.lr
        pop.set_lr(lr)
        pop.masks[:, 0] = 1.0 if j == start_iter else pop.masks[:, T]
        pop.bad_masks[:, 0] = 1.0 if j == start_iter else pop.bad_masks[:, T]
        if j > start_iter:
            pop.obs[:, 0:N].copy_(pop.obs[:, T * N:])                                               # after_update (storage.py:71-75)
        for step in range(T + 1):
            # slot `step`: normalise the simulators' answer to the previous actions (none at step 0), then act on it
            eps_t = _step_noise(N, dims) if step < T else None
            act_host = pipe.step(step, eps_t, sample=step < T, normalise=step > 0)
            if step == T:
                break
            t0 = time.perf_counter()
            act_env = _env_actions(act_host, dims)
            for p, envs in enumerate(envs_all):
                ob, rew, done, infos = envs.step(act_env[p])
                raw_obs[p] = ob
                raw_rew[p] = np.asarray(rew, dtype=np.float64).reshape(N)
                done_h[p] = done
                for n, info in enumerate(infos):
                    raw_obj[p, n] = info['obj']
                    bad_h[p, n] = 0.0 if 'bad_transition' in info.keys() else 1.0
            stats["env_s"] += time.perf_counter() - t0
        vn.mark_stepped()
        if vn.has_obj:
            pop.obj_var.copy_(vn.obj_var.to(torch.float32))
        else:
            pop.obj_var.fill_(1.0 - 1e-8)
        pop.perm.copy_(torch.stack([torch.randperm(T * N) for _ in range(args.ppo_epoch)]).to(torch.int32)[None])
        pop.update_only()
        new = _snapshot_samples(task_batch, pop, lr, vn.snapshot)
        t0 = time.perf_counter()
        for p, objs in enumerate(evaluation_batch(args, new)):
            new[p].objs = objs
            offspring[p].append(new[p])
        stats["eval_s"] += time.perf_counter() - t0
    for envs in envs_all:
        envs.close()
    return offspring


def mopg_population_update(args, task_batch, device, iteration, num_updates, start_time=None, cluster=0, stats=None):
    """All tasks of this shard advance together; returns offspring[task_id] = list of Samples (one per iteration),
    the content the reference's workers put on the queue (morl/morl.py:93-99). `stats` (optional dict) receives the
    seconds spent inside the environments' step() calls (`env_s`) and in the evaluation episodes (`eval_s`)."""
    P = len(task_batch)
    stats = stats if stats is not None else {}
    stats.setdefault("env_s", 0.0); stats.setdefault("eval_s", 0.0)
    first = task_batch[0].sample.actor_critic
    dims, dev = first.dims, first.flat.device
    total_num_updates = int(args.num_env_steps) // args.num_steps // args.num_processes
    ag0 = task_batch[0].sample.agent
    g0 = ag0.optimizer.param_groups[0]
    hyper = PpoHyper(ag0.clip_param, ag0.value_loss_coef, ag0.entropy_coef, ag0.max_grad_norm, g0["betas"][0],
                     g0["betas"][1], g0["eps"])
    cache = _population(dims, P, args, hyper, dev, cluster, ag0.use_clipped_value_loss)
    pop, pipe = cache["pop"], cache["pipe"]
    envs_all = []
    raw_mode = _HOOKS["make_raw_vec_envs"] is not None
    for p, task in enumerate(task_batch):
        ac, opt = task.sample.actor_critic, task.sample.agent.optimizer
        pop.params[p].copy_(ac.flat); pop.adam_m[p].copy_(opt.exp_avg); pop.adam_v[p].copy_(opt.exp_avg_sq)
        pop.adam_step[p] = opt.step_count
        pop.weights[p].copy_(torch.as_tensor(np.asarray(task.scalarization.weights, dtype=np.float64), dtype=torch.float32))
        if raw_mode:
            continue
        envs = _make_vec_envs(env_name=args.env_name, seed=args.seed, num_processes=args.num_processes, gamma=args.gamma,
                              log_dir=None, device=device, allow_early_resets=False, obj_rms=args.obj_rms, ob_rms=args.ob_rms)
        _restore_rms(envs, task.sample.env_params)
        envs_all.append(envs)
    T, N, M = args.num_steps, args.num_processes, args.obj_num
    if raw_mode:
        return _population_update_raw(args, task_batch, cache, device, iteration, min(iteration + num_updates, total_num_updates),
                                      total_num_updates, stats)
    obs_h = pipe.h_obs.numpy()                                            # pinned [P,N,O]: this step's observations
    rew_h, mask_h, bad_h = (pop.staging()[k].numpy() for k in ("rewards", "masks", "bad_masks"))   # pinned, whole rollout
    for p, e in enumerate(envs_all):
        obs_h[p] = np.asarray(e.reset(), dtype=np.float32)
    offspring = [[] for _ in range(P)]
    start_iter, final_iter = iteration, min(iteration + num_updates, total_num_updates)
    for j in range(start_iter, final_iter):
        torch.manual_seed(j)              # every task of a generation sees the same streams (mopg.py:96)
        lr = args.lr - (args.lr * ((j * args.lr_decay_ratio) / float(total_num_updates))) if args.use_linear_lr_decay else args.lr
        pop.set_lr(lr)
        if j == start_iter:
            mask_h[:, 0] = 1.0; bad_h[:, 0] = 1.0
        else:                                                             # after_update (storage.py:71-75)
            mask_h[:, 0] = mask_h[:, T]; bad_h[:, 0] = bad_h[:, T]
        for step in range(T):
            act_host = pipe.step(step, _step_noise(N, dims))              # one graph replay: H2D, K1 into slot `step`, D2H
            act_env = _env_actions(act_host, dims)
            t0 = time.perf_counter()
            for p, envs in enumerate(envs_all):
                obs, _, done, infos = envs.step(act_env[p])
                obs_h[p] = np.asarray(obs, dtype=np.float32)
                for n, info in enumerate(infos):
                    rew_h[p, step, n] = info['obj']
                    mask_h[p, step + 1, n] = 0.0 if done[n] else 1.0
                    bad_h[p, step + 1, n] = 0.0 if 'bad_transition' in info.keys() else 1.0
            stats["env_s"] += time.perf_counter() - t0
        pipe.step(T, None, sample=False)                                  # value of the last obs (mopg.py:132-135)
        # reward vectors / masks were only collected on the host during the rollout: one upload each before K2
        for k in ("rewards", "masks", "bad_masks"):
            getattr(pop, k).copy_(pop.staging()[k], non_blocking=True)
        for p, envs in enumerate(envs_all):
            var = envs.obj_rms.var if envs.obj_rms is not None else np.ones(M) - 1e-8
            pop.obj_var[p].copy_(torch.as_tensor(np.asarray(var, dtype=np.float64) * np.ones(M), dtype=torch.float32))
        pop.perm.copy_(torch.stack([torch.randperm(T * N) for _ in range(args.ppo_epoch)]).to(torch.int32)[None])
        pop.update_only()                                                                           # K2 + K3
        new = _snapshot_samples(task_batch, pop, lr, lambda p: _snapshot_rms(envs_all[p]))
        t0 = time.perf_counter()
        for p, objs in enumerate(evaluation_batch(args, new)):
            new[p].objs = objs
            offspring[p].append(new[p])
        stats["eval_s"] += time.perf_counter() - t0
    for envs in envs_all:
        envs.close()
    return offspring
