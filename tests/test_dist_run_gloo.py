"""The SHARDED generation loop (pgmorl_b200.morl.run under torch.distributed, SURVEY 8(e)) on CPU with gloo, world size 2,
against the same loop in a single process.

The device stages are replaced by a deterministic stand-in for `mopg_population_update` (tasks are independent, exactly
like the real one), so what is tested is the host protocol of morl/morl.py:84-143 in its sharded form: task i trains on
rank i % W, ONE all-gather of packed records per generation, stubs for remote samples, redundant selection on identical
metadata, lossless migration of (policy, Adam state, running moments) for elites that change owner, and the split of the
final archive files between the ranks. Everything the run writes must be identical to the single-process run, byte for
byte for the text files and bit for bit for the saved policies / moments."""
import os
import pickle
import socket
from copy import deepcopy
from types import SimpleNamespace

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from pgmorl_b200 import morl
from pgmorl_b200.a2c_ppo_acktr import algo
from pgmorl_b200.a2c_ppo_acktr.model import Policy
from pgmorl_b200.sample import Sample
from pgmorl_b200.scalarization_methods import WeightedSumScalarization
from pgmorl_b200.utils import generate_weights_batch_dfs
from pgmorl_b200.vec_normalize import RunningMeanStd


class _Box:
    def __init__(self, n):
        self.shape = (n,)


_Box.__name__ = "Box"
O, A, M = 5, 2, 2


def _args(save_dir, method):
    T, N = 8, 2
    return SimpleNamespace(
        env_name="none", seed=0, obj_num=M, num_steps=T, num_processes=N, num_env_steps=8 * T * N, warmup_iter=2,
        update_iter=2, selection_method=method, min_weight=0.0, max_weight=1.0, delta_weight=0.2, save_dir=save_dir,
        layernorm=False, algo="ppo", clip_param=0.2, ppo_epoch=2, num_mini_batch=2, value_loss_coef=0.5, entropy_coef=0.0,
        lr=3e-4, max_grad_norm=0.5, gamma=0.995, obj_rms=True, ob_rms=True, eval_num=1, raw=True,
        use_linear_lr_decay=True, lr_decay_ratio=1.0, use_gae=True, gae_lambda=0.95, use_proper_time_limits=True,
        rl_log_interval=0, pbuffer_num=100, pbuffer_size=2, num_tasks=6, num_weight_candidates=7, sparsity=1.0)


def _objs(flat, weights, j):
    """Smooth positive objectives that depend on the policy AND the weight the task trained with."""
    s = flat.double()
    a, b = float(s[:20].abs().mean()), float(s[20:40].abs().mean())
    w = np.asarray(weights, dtype=np.float64)
    return np.array([5.0 + 0.3 * j + 3.0 * w[0] + a, 5.0 + 0.3 * j + 3.0 * w[1] + b])


def _fake_warm_up(args, device):
    weights_batch, samples, scals = [], [], []
    generate_weights_batch_dfs(0, args.obj_num, args.min_weight, args.max_weight, args.delta_weight, [], weights_batch)
    for weights in weights_batch:
        ac = Policy((O,), _Box(A), obj_num=M, device="cpu")
        agent = algo.PPO(ac, args.clip_param, args.ppo_epoch, args.num_mini_batch, args.value_loss_coef, args.entropy_coef,
                         lr=args.lr, eps=1e-5, max_grad_norm=args.max_grad_norm)
        env_params = {'ob_rms': RunningMeanStd(shape=(O,)), 'ret_rms': RunningMeanStd(), 'obj_rms': RunningMeanStd()}
        s = Sample(env_params, ac, agent, optgraph_id=-1)
        s.objs = _objs(ac.flat, weights, 0)
        samples.append(s)
        scals.append(WeightedSumScalarization(num_objs=M, weights=weights))
    return samples, scals


def _fake_mopg(args, task_batch, device, iteration, num_updates, start_time=None, cluster=0):
    total = int(args.num_env_steps) // args.num_steps // args.num_processes
    out = []
    for task in task_batch:
        w = np.asarray(task.scalarization.weights, dtype=np.float64)
        cur, produced = task.sample, []
        for j in range(iteration, min(iteration + num_updates, total)):
            s = Sample.copy_from(cur)
            g = torch.Generator().manual_seed(j)
            noise = torch.randn(s.actor_critic.flat.shape, generator=g)
            s.actor_critic.flat = (s.actor_critic.flat * 0.999 + 0.01 * float(w[0]) * noise).float()
            opt = s.agent.optimizer
            opt.exp_avg = opt.exp_avg * 0.9 + 0.1 * noise
            opt.exp_avg_sq = opt.exp_avg_sq * 0.999 + 0.001 * noise * noise
            opt.step_count += args.ppo_epoch * args.num_mini_batch
            opt.param_groups[0]['lr'] = args.lr * (1.0 - j / total)
            for key, k in (('ob_rms', O), ('ret_rms', 0), ('obj_rms', M)):
                r = s.env_params[key]
                shape = (k,) if k else ()
                r.mean = np.asarray(r.mean) * np.ones(shape) + 0.1 * float(w[1]) + 0.01 * j
                r.var = np.asarray(r.var) * np.ones(shape) * 1.01
                r.count = r.count + args.num_steps
            s.objs = _objs(s.actor_critic.flat, w, j + 1)
            produced.append(s)
            cur = s
        out.append(produced)
    return out


def _run(save_dir, method, patch=setattr):
    """`patch` installs the stand-ins; the test's own process passes monkeypatch.setattr so that the real device stages
    are back for the tests that run after it."""
    patch(morl, "initialize_warm_up_batch", _fake_warm_up)
    patch(morl, "mopg_population_update", _fake_mopg)
    if not torch.cuda.is_available():
        # no CPU fallback exists in the product: the archive's dominance filter is K5. On a machine without a GPU this
        # test (host protocol only) lets the ORACLE stand in for that one kernel.
        from oracle import selection_oracle as so
        from pgmorl_b200 import ep as ep_mod
        patch(ep_mod, "get_ep_indices", lambda objs: list(so.get_ep_indices(np.asarray(objs, dtype=np.float64))))
    return morl.run(_args(save_dir, method), device="cpu")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, save_dir, method):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ep, population, graph, timings = _run(save_dir, method)
        # every rank must hold the same metadata; exactly the owner holds the state
        meta = np.concatenate([np.asarray(ep.obj_batch).reshape(-1), [len(population.sample_batch), len(graph.objs)]])
        both = [torch.zeros(len(meta), dtype=torch.float64) for _ in range(world)]
        dist.all_gather(both, torch.from_numpy(meta))
        assert all(torch.equal(both[0], b) for b in both)
        for s in list(ep.sample_batch) + list(population.sample_batch):
            assert s.is_stub == (s.owner != rank)
        if rank == 0:
            with open(os.path.join(save_dir, "migrated.count"), "w") as fp:
                fp.write(str(sum(t["migrated"] for t in timings)))
    finally:
        dist.destroy_process_group()


def _tree(root):
    out = {}
    for d, _, files in os.walk(root):
        for f in files:
            out[os.path.relpath(os.path.join(d, f), root)] = os.path.join(d, f)
    return out


import pytest


@pytest.mark.parametrize("method", ["prediction-guided", "moead", "ra", "random"])
def test_sharded_run_equals_single_process_run(tmp_path, monkeypatch, method):
    if method == "prediction-guided":
        pytest.importorskip("torch")
        if not torch.cuda.is_available():
            pytest.skip("prediction-guided selection launches K4 / K5 (the sharded GPU test covers it)")
    one, two = str(tmp_path / "w1"), str(tmp_path / "w2")
    _run(one, method, monkeypatch.setattr)
    mp.spawn(_worker, args=(2, _free_port(), two, method), nprocs=2, join=True)
    migrated = int(open(os.path.join(two, "migrated.count")).read())
    os.remove(os.path.join(two, "migrated.count"))
    assert (migrated > 0) == (method in ("moead", "random", "prediction-guided")), migrated   # 'ra' keeps every task on its rank
    a, b = _tree(one), _tree(two)
    assert sorted(a) == sorted(b) and any(k.startswith("final/EP_policy_") for k in a)
    for k in sorted(a):
        if k.endswith(".txt"):
            assert open(a[k]).read() == open(b[k]).read(), k
        elif k.endswith(".pt"):
            x, y = torch.load(a[k]), torch.load(b[k])
            assert list(x) == list(y) and all(torch.equal(x[n], y[n]) for n in x), k
        elif k.endswith(".pkl"):
            x, y = pickle.load(open(a[k], "rb")), pickle.load(open(b[k], "rb"))
            for key in ('ob_rms', 'ret_rms', 'obj_rms'):
                assert np.array_equal(np.asarray(x[key].mean), np.asarray(y[key].mean)), (k, key)
                assert np.array_equal(np.asarray(x[key].var), np.asarray(y[key].var)), (k, key)
                assert float(x[key].count) == float(y[key].count), (k, key)


def test_sample_state_roundtrip_is_lossless():
    from pgmorl_b200 import dist as pd
    samples, _ = _fake_warm_up(_args("/tmp", "ra"), "cpu")
    s = _fake_mopg(_args("/tmp", "ra"), [SimpleNamespace(sample=samples[1], scalarization=SimpleNamespace(weights=[0.3, 0.7]))],
                   "cpu", 0, 2)[0][-1]
    s.env_params['obj_rms'] = RunningMeanStd()                  # still scalar-shaped: before its first update
    payload = pd.pack_sample_state(s)
    assert payload.dtype == torch.float64 and payload.numel() == pd.sample_state_len(s.actor_critic.dims)
    t = pd.unpack_sample_state(payload, samples[0], objs=deepcopy(s.objs), optgraph_id=7)
    assert torch.equal(t.actor_critic.flat, s.actor_critic.flat)
    assert torch.equal(t.agent.optimizer.exp_avg, s.agent.optimizer.exp_avg)
    assert torch.equal(t.agent.optimizer.exp_avg_sq, s.agent.optimizer.exp_avg_sq)
    assert t.agent.optimizer.step_count == s.agent.optimizer.step_count
    assert t.agent.optimizer.param_groups[0]['lr'] == s.agent.optimizer.param_groups[0]['lr']
    for key in ('ob_rms', 'ret_rms', 'obj_rms'):
        assert np.array_equal(np.asarray(t.env_params[key].mean), np.asarray(s.env_params[key].mean))
        assert np.shape(t.env_params[key].mean) == np.shape(s.env_params[key].mean)
        assert np.array_equal(np.asarray(t.env_params[key].var), np.asarray(s.env_params[key].var))
        assert t.env_params[key].count == s.env_params[key].count
    assert t.optgraph_id == 7 and np.array_equal(t.objs, s.objs)
