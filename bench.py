#!/usr/bin/env python
"""Benchmark of the PG-MORL hot path (BASELINE.json metric: MOPG env-steps/s; configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|...] [--dump-outputs DIR]

One "step" = one MOPG iteration of the population shard on one batch of synthetic trajectories: rollout inference
(K1) + vector GAE / advantage (K2) + PPO update of E epochs x B minibatches with Adam (K3). Every GEN_ITERS-th step
closes a GENERATION (morl/morl.py:62-177): the ranks all-gather the packed per-task records (task id, parent node,
weight, objective vector of every iteration), every rank updates opt-graph / Pareto archive / population and runs the
prediction-guided selection (K4 fits + K5 greedy scoring) redundantly on the gathered table, and the (policy, Adam,
moments) state of elites that change owner moves point to point -- INSIDE the timed region, at every N (N = 1: no
collective, same selection). Workload at N=1 = BASELINE.json configs[1]: HalfCheetah shape, 6 tasks x 4 envs x 2048
steps, 10 epochs x 32 minibatches. With N > 1 (torchrun, one rank per GPU) every rank owns its own tasks: 6 per GPU for
the weak configs, 64 / N for `--config humanoid64` (BASELINE.json configs[3], strong split).

Prints ONE JSON line (rank 0):
  value       device-timed throughput of the K timed steps (CUDA events on the launching stream, max over ranks), inputs
              resident in HBM, generation boundaries included; `mopg_only` = the same without the boundary steps' extra
  e2e         the same metric through the host-buffer API: every step does a BLOCKING H2D copy of THAT step's inputs from
              pinned memory, K1-K3, a D2H read of the losses and a host wait -- host wall clock, nothing overlapped
  generation  one whole generation (GEN_ITERS e2e steps + exchange + selection + migration) as one wall-clock unit
  api         one iteration through the drop-in `mopg_population_update` (per-step K1 / K6 over replay environments)
  roofline / cpu_baseline / selection / clocks as the task statement prescribes.
`--impl reference` times the reference's CPU path on the host cores: the UNMODIFIED reference where /root/reference is
importable (kind "reference"), else the oracle port with the reference's op sequence (kind "port"; the GPU box has no
/root/reference), process per task, one thread each, tasks = tasks/GPU x WORLD_SIZE, selection at the generation boundary
by the CPU oracle (scipy least_squares + python scoring).
"""
import argparse
import glob
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))      # synth_envs (synthetic selection states, replay environments)

CONFIGS = {
    # name: (env shape, tasks per GPU (weak) or in total (strong), T, N, E, B, gamma, scaling)
    "c2": ("halfcheetah", 6, 2048, 4, 10, 32, 0.995, "weak"),       # BASELINE.json configs[1]
    "walker64": ("walker2d", 64, 2048, 4, 10, 32, 0.995, "weak"),    # population sweep points (configs[4])
    "walker256": ("walker2d", 256, 2048, 4, 10, 32, 0.995, "weak"),
    "walker1024": ("walker2d", 1024, 2048, 4, 10, 32, 0.995, "weak"),
    "hopper3": ("hopper3", 15, 2048, 4, 10, 32, 0.995, "weak"),
    "humanoid8": ("humanoid", 8, 2048, 8, 10, 32, 0.99, "weak"),
    "humanoid16": ("humanoid", 16, 2048, 8, 10, 32, 0.99, "weak"),
    "humanoid32": ("humanoid", 32, 2048, 8, 10, 32, 0.99, "weak"),
    "humanoid64": ("humanoid", 64, 2048, 8, 10, 32, 0.99, "strong"),  # BASELINE.json configs[3]: 64 tasks over 2/4/8 GPUs
}
GEN_ITERS = 20           # update_iter of the reference's launch scripts (scripts/walker2d-v2.py:40)


def flops_per_env_step(d, E):
    """Algorithmic FLOPs (SURVEY.md section 8(d)): K1 forward once; K3 fwd + weight-grad + input-grad x E."""
    O, A, M, H = d.obs, d.act, d.obj, d.hidden
    actor, critic = O * H + H * H + H * A, O * H + H * H + H * M
    fwd = 2 * (actor + critic)
    per_epoch = fwd + fwd + 2 * (H * H + H * A) + 2 * (H * H + H * M)
    return fwd, per_epoch * E


def bytes_per_env_step(d, E):
    """Algorithmic HBM bytes: K1 128 B, K2 36 B, K3 per epoch one 29-float record + 4 B index (Walker dims)."""
    O, A, M = d.obs, d.act, d.obj
    k1 = 4 * (O + A + A + 1 + M)
    k2 = 4 * (M + M + 2 + M + 1)
    k3 = E * (4 * (O + A + 1 + 2 * M + 1) + 4)
    return k1, k2, k3


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        if self.index is None:          # ranks other than 0: one sampler per job (eight concurrent nvidia-smi pollers stall launches)
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.1] or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_inputs(d, P, T, N, E, seed, first_task=0):
    """Seeded synthetic trajectories / noise / permutations / weights / initial policies of tasks
    first_task .. first_task + P - 1 (identical bytes for the GPU path and the CPU arm)."""
    from pgmorl_b200 import synthetic
    traj = synthetic.make_trajectories(P, T, N, d, seed=seed)
    eps, perm = synthetic.host_rng_streams(0, T, N, d.act, E)
    w = synthetic.simplex_weights(d.obj, 0.2 if d.obj == 2 else 0.25)
    weights = np.stack([w[(first_task + p) % len(w)] for p in range(P)])
    obj_var = np.tile(np.array([1.3, 0.7, 0.9][:d.obj]), (P, 1))
    flats = [synthetic.init_policy_flat(d, seed=1000 + first_task + p).numpy() for p in range(P)]
    return traj, eps, perm, weights, obj_var, flats


# ------------------------------------------------------------------------------------------------------------------
# The generation boundary on synthetic objectives (environment evaluation is host work outside the scope): the REAL
# exchange / bookkeeping / selection / migration code of pgmorl_b200.morl + dist on a synthetic optimisation history.
# ------------------------------------------------------------------------------------------------------------------
class GenerationBoundary:
    def __init__(self, d, n_tasks, world, rank, pop=None, cpu=False, seed=3):
        import synth_envs
        from pgmorl_b200 import dist as pdist
        from pgmorl_b200.scalarization_methods import WeightedSumScalarization
        self.pd, self.d, self.M, self.W, self.rank, self.pop, self.cpu = pdist, d, d.obj, world, rank, pop, cpu
        self.n_tasks = n_tasks
        M = d.obj
        # steady-state sizes: the recorded 6-task history holds 48 population members (8 per task) and the 2-objective
        # performance buffers cap the population at 200 (100 x 2), the 3-objective ones at 420 (210 x 2)
        n_pop = min(8 * n_tasks, 200 if M == 2 else 420)
        self.args, self.graph, self.population, self.ep = synth_envs.make_selection_state(
            M, max(n_pop, n_tasks), 50, seed=seed, num_tasks=n_tasks)
        self.args.update_iter = GEN_ITERS
        for s in list(self.population.sample_batch) + list(self.ep.sample_batch):
            s.owner = (s.optgraph_id or 0) % world
        self.template = WeightedSumScalarization(num_objs=M, weights=np.ones(M) / M)
        grid = [w for w in __import__("pgmorl_b200.synthetic", fromlist=["x"]).simplex_weights(M, 0.2 if M == 2 else 0.25)]
        self.elites = list(self.population.sample_batch[:n_tasks])
        self.weights = [np.asarray(grid[i % len(grid)], dtype=np.float64) for i in range(n_tasks)]
        self.mine = pdist.shard_tasks(n_tasks, world, rank)
        self.gen = 0
        self.n_state = pdist.sample_state_len(d)
        self.picks = []
        self._next_objs = None
        if cpu:   # CPU arm: the archive's dominance filter and the selection come from the oracle (no GPU visible)
            from oracle import selection_oracle as so
            from pgmorl_b200 import ep as ep_mod
            ep_mod.get_ep_indices = lambda objs: list(so.get_ep_indices(np.asarray(objs, dtype=np.float64)))

    def _objs(self, task):
        """Synthetic objective vectors of the GEN_ITERS offspring of `task` this generation (seeded per task and
        generation: independent of how the tasks are sharded)."""
        import synth_envs
        rng = np.random.RandomState(100003 * (self.gen + 1) + task)
        o = np.array(self.elites[task].objs, dtype=np.float64)
        out = []
        for _ in range(GEN_ITERS):
            o = o + synth_envs._response(rng, o, self.weights[task]) / GEN_ITERS
            out.append(o.copy())
        return np.stack(out)

    def _select_cpu(self):
        """prediction_guided_selection with the CPU oracle: scipy least_squares for every fit, python greedy scoring."""
        from copy import deepcopy
        from oracle import selection_oracle as so
        pop, graph, args, M = self.population, self.graph, self.args, self.M
        view = so.GraphArrays(graph)
        cands = []
        for s in pop.sample_batch:
            tw = pop._test_weights(graph, s, args.num_weight_candidates) if M == 2 else None
            if M != 2:
                raise NotImplementedError("CPU boundary: 2-objective configs only")
            if len(tw) == 0:
                continue
            theta = [so.fit_scipy(x, y, w, ub).x for x, y, w, ub in so.fit_inputs(view, s.optgraph_id, M, False)]
            t = np.array(tw, dtype=np.float64)
            t = t / t.sum(axis=1, keepdims=True)
            pred = view.objs[s.optgraph_id][None, :] + np.stack([so.model(t[:, m], *theta[m]) for m in range(M)], axis=1)
            cands += [(s, w, p) for w, p in zip(tw, pred)]
        best = so.greedy_select_2d(np.asarray(self.ep.obj_batch), np.array([c[2] for c in cands]), args.sparsity,
                                   args.num_tasks)[0]
        elites, scals = [], []
        for b in best:
            if b < 0:
                break
            sc = deepcopy(self.template)
            sc.update_weights(cands[int(b)][1] / np.sum(cands[int(b)][1]))
            elites.append(cands[int(b)][0]); scals.append(sc)
        return elites, scals

    def prepare(self):
        """Stand-in for the evaluation episodes of the generation that is about to close (host work during the
        iterations, outside this path's scope): the synthetic objective vectors of this rank's tasks. Not timed."""
        self._next_objs = [self._objs(i) for i in self.mine]

    def run(self):
        """One generation boundary; returns the seconds spent in (exchange, bookkeeping, selection, migration)."""
        import synth_envs
        import torch
        pd, M, W, rank = self.pd, self.M, self.W, self.rank
        if self._next_objs is None:
            self.prepare()
        t0 = time.perf_counter()
        local = pd.pack_records(self.mine, [self.elites[i].optgraph_id for i in self.mine],
                                [self.weights[i] for i in self.mine], self._next_objs)
        self._next_objs = None
        table = pd.all_gather_records(local, self.n_tasks)
        t1 = time.perf_counter()
        all_samples, offspring = [], []
        for task, parent, w, objs in pd.unpack_records(table, M):
            prev = parent
            for it, o in enumerate(objs):
                s = synth_envs.ObjSample(o.copy())
                s.owner = pd.owner_of(task, W)
                all_samples.append(s)
                if (it + 1) % self.args.update_iter == 0:
                    prev = self.graph.insert(w.copy(), o.copy(), prev)
                    s.optgraph_id = prev
                    offspring.append(s)
        self.population.update(offspring)
        if not self.cpu:
            self.population.prefetch_fits(self.args, self.graph)      # the K4 chain runs under the archive update
        self.ep.update(all_samples)
        t2 = time.perf_counter()
        np.random.seed(1000 + self.gen)
        if self.cpu:
            elites, scals = self._select_cpu()
        else:
            elites, scals, _ = self.population.prediction_guided_selection(self.args, self.gen, self.ep, self.graph, self.template)
            torch.cuda.synchronize()
        t3 = time.perf_counter()
        while len(elites) < self.n_tasks:        # "Too few candidates": keep the loop full with the best remaining members
            elites.append(self.population.sample_batch[len(elites) % len(self.population.sample_batch)])
            scals.append(self.template)
        # migration of the elites whose state lives on another rank than their next task (task i trains on rank i % W);
        # the payload is the owner's device snapshot of that policy (real sizes: params + Adam moments + running moments)
        pop = self.pop
        plan = pd.plan_migration([e.owner for e in elites], W)
        if pop is not None and W > 1:
            def get_state(task):
                p = task % pop.P
                par, m, v, step = pop.snapshot_state(self.gen, p)
                out = torch.zeros(self.n_state, dtype=torch.float64, device=pop.device)
                n = self.d.n_par
                out[:n], out[n:2 * n], out[2 * n:3 * n] = par, m, v
                out[3 * n] = step
                return out

            def put_state(task, t):
                p, n = task // W, self.d.n_par
                pop.params[p].copy_(t[:n]); pop.adam_m[p].copy_(t[n:2 * n]); pop.adam_v[p].copy_(t[2 * n:3 * n])
            pd.migrate_states(plan, get_state, put_state, self.n_state, device=pop.device)
        if pop is not None:
            w32 = torch.as_tensor(np.stack([np.asarray(scals[i].weights, dtype=np.float64) for i in self.mine]), dtype=torch.float32)
            pop.weights.copy_(w32)
            torch.cuda.synchronize()
        t4 = time.perf_counter()
        self.elites = elites
        self.weights = [np.asarray(s.weights, dtype=np.float64) for s in scals]
        self.picks.append([(e.optgraph_id, tuple(np.round(w, 12))) for e, w in zip(elites, self.weights)])
        self.gen += 1
        return {"exchange_s": t1 - t0, "bookkeeping_s": t2 - t1, "selection_s": t3 - t2, "migration_s": t4 - t3,
                "migrated": len(plan), "n_pop": len(self.population.sample_batch), "archive": int(len(self.ep.obj_batch))}


# ------------------------------------------------------------------------------------------------------------------
# reference arm (CPU)
# ------------------------------------------------------------------------------------------------------------------
def reference_available():
    return os.path.isdir("/root/reference/morl") and os.path.isdir("/root/reference/externals/pytorch-a2c-ppo-acktr-gail")


def cpu_reference_leg(d, P_total, T, N, E, B, gamma, steps, warmup, boundary=True):
    """Reference CPU path on the host cores: process per task, one torch thread each (morl/morl.py:34,84-88), the
    unmodified reference's Policy / RolloutStorage / PPO.update where /root/reference is importable, else the oracle
    port (same op sequence). Returns a dict with env-steps/s, ms per step, processes, kind, per-step times."""
    kind = "reference" if reference_available() else "port"
    if kind == "reference":
        from oracle.ref_mopg_runner import timed_population_iteration
    else:
        from oracle.mopg_torch_port import timed_population_iteration
    cores = os.cpu_count() or 1
    procs = min(P_total, cores)
    traj, eps, perm, weights, obj_var, flats = synthetic_inputs(d, P_total, T, N, E, seed=1)
    trajs = [{k: v[p].numpy() for k, v in traj.items()} for p in range(P_total)]
    dims = (d.obs, d.act, d.obj)
    kw = dict(gamma=gamma, lam=0.95, ppo_epoch=E, num_mini_batch=B)
    for _ in range(warmup):
        timed_population_iteration(flats[:procs], dims, trajs[:procs], 0, 3e-4, weights, obj_var, procs, **kw)
    gb = GenerationBoundary(d, P_total, 1, 0, pop=None, cpu=True) if boundary and d.obj == 2 else None
    walls, bnd = [], []
    for i in range(steps):
        wall, per_task, _ = timed_population_iteration(flats, dims, trajs, i, 3e-4, weights, obj_var, procs, **kw)
        if gb is not None and (i + 1) % GEN_ITERS == 0:
            t0 = time.perf_counter()
            gb.run()
            bnd.append(time.perf_counter() - t0)
        walls.append(wall)
    total = float(np.sum(walls) + np.sum(bnd))
    return {"value": P_total * T * N * steps / total, "ms_per_step": 1e3 * total / steps, "procs": procs, "kind": kind,
            "mopg_only_ms_per_step": 1e3 * float(np.mean(walls)), "boundary_ms": [1e3 * b for b in bnd]}


def selection_leg(cpu=True):
    """Secondary BASELINE metric: prediction-guided selection ms/generation on the recorded synthetic histories
    (tests/golden/selection_{2d,3d}.npz, last generation): product path = K4 front-end kernels + K4 fits (+ the host's
    test-weight enumeration under them) + K5 greedy loop; CPU = oracle port (scipy least_squares + python scoring; 3-D scoring timed on ONE of the 15 rounds
    and scaled, stated in `cpu_sample`)."""
    import torch
    from helpers import rebuild_selection_state
    from synth_envs import make_selection_state
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    out = {}
    torch.set_default_dtype(torch.float64)
    try:
        for name, M in (("selection_2d.npz", 2), ("selection_3d.npz", 3)):
            z = np.load(os.path.join(ROOT, "tests", "golden", name))
            g = int(z["meta"][1]) - 1
            times = []
            for rep in range(4):
                args_s, graph, pop, ep = rebuild_selection_state(z, g, M)
                np.random.seed(1000 + g)
                template = WeightedSumScalarization(num_objs=M, weights=np.ones(M) / M)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                elites, scals, pred = pop.prediction_guided_selection(args_s, g, ep, graph, template)
                torch.cuda.synchronize()
                times.append(time.perf_counter() - t0)
            key = f"{M}d"
            out[key] = {"ms_per_generation": 1e3 * min(times[1:]), "n_pop": len(pop.sample_batch),
                        "candidates": len(pop.last_candidates), "fits": len(pop.last_fits["x"]),
                        "archive": int(len(ep.obj_batch)), "tasks": args_s.num_tasks}
            if cpu:
                from oracle import selection_oracle as so
                f = pop.last_fits
                t0 = time.perf_counter()
                for x, y, w, ub in zip(f["x"], f["y"], f["w"], f["ub"]):
                    so.fit_scipy(x, y, w, ub)
                t_fit = time.perf_counter() - t0
                cand = np.array([c["prediction"] for c in pop.last_candidates])
                t0 = time.perf_counter()
                if M == 2:
                    so.greedy_select_2d(z[f"g{g}_round0_vep"], cand, args_s.sparsity, args_s.num_tasks)
                    t_sel = time.perf_counter() - t0
                else:
                    so.greedy_select_3d(z[f"g{g}_round0_vep"], cand, args_s.sparsity, 1)
                    t_sel = (time.perf_counter() - t0) * args_s.num_tasks
                out[key]["cpu_ms_per_generation"] = 1e3 * (t_fit + t_sel)
                out[key]["cpu_sample"] = ("scipy least_squares on every fit + python scoring, 1 core"
                                          + ("" if M == 2 else "; scoring timed on 1 of 15 greedy rounds and scaled"))
        # full performance buffers (SURVEY.md section 8(d): n_pop 200 / 1 400 candidates / archive 300 and
        # n_pop 420 / 2 940 candidates / archive 500), built directly by tests/synth_envs.make_selection_state
        for M, n_pop, n_ep in ((2, 200, 300), (3, 420, 500)):
            times = []
            for rep in range(3):
                args_s, graph, pop, ep = make_selection_state(M, n_pop, n_ep, seed=3)
                np.random.seed(7)
                template = WeightedSumScalarization(num_objs=M, weights=np.ones(M) / M)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                pop.prediction_guided_selection(args_s, 0, ep, graph, template)
                torch.cuda.synchronize()
                times.append(time.perf_counter() - t0)
            key = f"{M}d_full"
            out[key] = {"ms_per_generation": 1e3 * min(times[1:]), "n_pop": n_pop, "candidates": len(pop.last_candidates),
                        "fits": len(pop.last_fits["x"]), "archive": n_ep, "tasks": args_s.num_tasks}
            if cpu:
                from oracle import selection_oracle as so
                f = pop.last_fits
                sub = range(0, len(f["x"]), 8)                       # every 8th fit, scaled
                t0 = time.perf_counter()
                for i in sub:
                    so.fit_scipy(f["x"][i], f["y"][i], f["w"][i], f["ub"][i])
                t_fit = (time.perf_counter() - t0) * len(f["x"]) / len(sub)
                cand = np.array([c["prediction"] for c in pop.last_candidates])
                csub = cand[:: max(1, len(cand) // 40)]              # ~40 candidates of one greedy round, scaled
                t0 = time.perf_counter()
                (so.greedy_select_2d if M == 2 else so.greedy_select_3d)(ep.obj_batch, csub, args_s.sparsity, 1)
                t_sel = (time.perf_counter() - t0) * len(cand) / len(csub) * args_s.num_tasks
                out[key]["cpu_ms_per_generation"] = 1e3 * (t_fit + t_sel)
                out[key]["cpu_sample"] = ("scipy least_squares on every 8th fit and python scoring of ~40 candidates of one "
                                          "greedy round, both scaled to the full counts, 1 core")
    finally:
        torch.set_default_dtype(torch.float32)
    return out


def api_leg(d, P, T, N, E, B, gamma, device, cluster):
    """One MOPG iteration through the DROP-IN call `mopg.mopg_population_update` (the per-step loop of
    morl/mopg.py:103-144: one K1 launch per environment step for all tasks, the K2 / K3 update, the Sample snapshots),
    over replay environments that hand back pre-generated observations (environment time ~ 0), in both modes:
    host-normalised observations (`make_vec_envs`) and raw simulator output normalised on the device by K6."""
    import torch
    from types import SimpleNamespace
    import synth_envs
    from pgmorl_b200 import mopg, synthetic
    from pgmorl_b200.a2c_ppo_acktr import algo
    from pgmorl_b200.a2c_ppo_acktr.model import Policy
    from pgmorl_b200.sample import Sample, Task
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    traj = synthetic.make_trajectories(P, T, N, d, seed=1)
    trajs = [{k: v[p].numpy() for k, v in traj.items()} for p in range(P)]
    args = SimpleNamespace(env_name="replay", seed=0, obj_num=d.obj, num_steps=T, num_processes=N,
                           num_env_steps=40 * T * N, ppo_epoch=E, num_mini_batch=B, gamma=gamma, gae_lambda=0.95, lr=3e-4,
                           use_linear_lr_decay=True, lr_decay_ratio=1.0, obj_rms=True, ob_rms=True, eval_num=1, raw=True,
                           update_iter=GEN_ITERS, rl_log_interval=0)
    order = iter(range(10 ** 9))
    mopg.set_env_hooks(make_vec_envs=lambda **kw: synth_envs.ReplayVecEnv(trajs[next(order) % P], d, [1.3, 0.7, 0.9][:d.obj]),
                       gym_make=lambda name: synth_envs.ToyEvalEnv(d, horizon=1), make_raw_vec_envs=False)
    w = synthetic.simplex_weights(d.obj, 0.2 if d.obj == 2 else 0.25)
    tasks = []
    for p in range(P):
        torch.manual_seed(1000 + p)
        ac = Policy((d.obs,), synth_envs._Box(d.act), obj_num=d.obj, device=device)
        agent = algo.PPO(ac, 0.2, E, B, 0.5, 0.0, lr=3e-4, eps=1e-5, max_grad_norm=0.5)
        env = synth_envs.ReplayVecEnv(trajs[p], d, [1.3, 0.7, 0.9][:d.obj])
        s = Sample({k: getattr(env, k) for k in ("ob_rms", "ret_rms", "obj_rms")}, ac, agent, objs=np.ones(d.obj), optgraph_id=0)
        tasks.append(Task(s, WeightedSumScalarization(num_objs=d.obj, weights=w[p % len(w)])))
    out = {}
    for mode in ("host_normalised", "device_normalised"):
        if mode == "device_normalised":       # raw simulator output, running normalisation on the device (K6)
            mopg.set_env_hooks(make_raw_vec_envs=lambda **kw: synth_envs.RawReplayVecEnv(trajs[next(order) % P], d))
        rows = []
        for it in range(3):
            stats = {}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mopg.mopg_population_update(args, tasks, device, it, 1, cluster=cluster, stats=stats)
            torch.cuda.synchronize()
            rows.append((time.perf_counter() - t0, stats["env_s"], stats["eval_s"]))
        wall, env_s, eval_s = min(rows[1:])
        ms = 1e3 * (wall - env_s - eval_s)
        out[mode] = {"ms_per_iteration": 1e3 * wall, "ms_in_env_step_calls": 1e3 * env_s, "ms_in_evaluation": 1e3 * eval_s,
                     "ms_excluding_env_and_evaluation": ms, "env_steps_per_s_excluding_env": P * T * N / (ms * 1e-3),
                     "us_per_env_time_step_excluding_env": 1e3 * ms / T}
    mopg.set_env_hooks(make_raw_vec_envs=False)
    out["note"] = ("wall clock of mopg_population_update(num_updates=1): per environment step ONE CUDA-graph replay (H2D of the "
                   "staged step, [K6,] K1 into the rollout slot, D2H of the actions) + stream synchronise for all tasks, then K2 / "
                   "K3, the Sample snapshots and one toy evaluation episode per task; the Python time inside the replay "
                   "environments' step() and the evaluation episodes is reported separately; best of 2 after 1 warm-up")
    return out


K3_SOURCES = {      # the files a kernel family is compiled from (pgmorl_b200/csrc/)
    "k3_ppo_fast_kernel": ("k3_fast.cuh", "k3_ppo.cu", "net.cuh", "common.cuh"),
    "k3_tc_kernel": ("k3_tc.cuh", "tc.cuh", "tc_pair.cuh", "k3_ppo.cu", "net.cuh", "common.cuh"),
    "k3_tcw_kernel": ("k3_tcw.cuh", "tc.cuh", "tc_pair.cuh", "k3_ppo.cu", "net.cuh", "common.cuh"),
}


def measure_ffma_peak(dev, sms):
    """FP32 FMA throughput of this GPU in TFLOP/s, measured live with the packed-FFMA2 burn kernel of the diagnostics
    library on 2 CTAs x 512 threads per SM (CUDA events, best of 5): (burst, sustained) = a 0.3 ms launch at the clock the
    part idles at, and a 4 ms launch during which a full-chip FMA load pulls the SM clock down. MEASURED_PEAKS.json carries
    only the HBM and tensor peaks."""
    import ctypes
    import torch
    from pgmorl_b200 import _lib
    ctas = 2 * sms
    out = torch.empty(ctas * 512, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    res = []
    for iters in (512, 8192):
        best = 0.0
        for rep in range(6):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check_diag(_lib.diag_lib().pgm_ffma2_burn(_lib.ptr(out), ctas, iters, st))
            e1.record()
            e1.synchronize()
            if rep:
                best = max(best, ctas * 512 * iters * 64 * 2 * 2 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        res.append(best)
        time.sleep(0.2)
    return tuple(res)


def k3_source_hash(kernel="k3_ppo_fast_kernel"):
    h = hashlib.sha256()
    for f in K3_SOURCES[kernel.split(":")[0]]:
        h.update(open(os.path.join(ROOT, "pgmorl_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/traffic.json, written by
    profiles/ncu_traffic.py next to the raw CSV it was read from). null when no capture exists for this kernel or when the
    K3 sources changed since the capture (stale)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except OSError:
        return None, None
    e = t.get(kernel)
    if not e:
        return None, None
    if e.get("source_sha") != k3_source_hash(kernel):
        return None, f"stale: {e.get('csv')} was captured at source hash {e.get('source_sha')}"
    return e["dram_bytes"], e.get("csv")


DUMP_BYTES = 60 << 20       # data of all dumped arrays together; with the .npy headers the directory stays under 64 MB


def dump_outputs(out_dir, arrays):
    """Write `arrays` (name -> numpy array) as out_dir/<name>.npy in float32 / float64. When they hold more than DUMP_BYTES,
    every array is cut to the same fraction of its elements: a flat sample at sorted indices drawn from a generator seeded
    by the array's name, so that two runs with the same arguments write the same sample."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: a if a.dtype in (np.float32, np.float64) else a.astype(np.float64) for k, a in arrays.items()}
    frac = min(1.0, DUMP_BYTES / sum(a.nbytes for a in arrays.values()))
    for name, a in arrays.items():
        if frac < 1.0:
            flat = a.reshape(-1)
            rng = np.random.default_rng(zlib.crc32(name.encode()))
            a = flat[np.sort(rng.choice(flat.size, int(flat.size * frac), replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--cluster", type=lambda s: int(s, 0), default=int(os.environ.get("PGM_PPO_CLUSTER", "0"), 0))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-selection", action="store_true")
    ap.add_argument("--no-api", action="store_true")
    ap.add_argument("--no-boundary", action="store_true", help="leave the generation boundary out of the timed loops")
    ap.add_argument("--quarter-sample", action="store_true",
                    help="reference arm: T/4 steps per iteration (same minibatch size) instead of the full-size iteration")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed for rank 0's tasks (updated policies and "
                         "Adam state, rollout values / actions / log-probs, returns, advantages, losses, task weights) as "
                         "DIR/<name>.npy, at most 64 MB in all (a fixed seeded sample of larger outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        # CPU-only arm: hide the GPUs before torch is imported (fork-based worker pools cannot follow the CUDA
        # autograd threads torch starts when a device is visible)
        os.environ["CUDA_VISIBLE_DEVICES"] = ""

    from pgmorl_b200.layout import ENV_SHAPES
    env, P_cfg, T, N, E, B, gamma, scaling = CONFIGS[args.config]
    d = ENV_SHAPES[env]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if scaling == "strong":
        assert P_cfg % world == 0, f"{args.config}: {P_cfg} tasks do not split over {world} ranks"
        P, n_tasks = P_cfg // world, P_cfg
    else:
        P, n_tasks = P_cfg, P_cfg * world
    # stdout carries exactly ONE JSON line: whatever native libraries write to file descriptor 1 (NCCL prints its version
    # banner / debug output there) is sent to stderr, and the JSON line goes to a private duplicate of the real stdout
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    S = T * N
    metric = "MOPG env-steps/sec (rollout infer + GAE + PPO update)"
    boundary_on = not args.no_boundary and d.obj == 2
    workload = {"workload": f"{env}-shape population MOPG update: {P} tasks/GPU x {N} envs x {T} steps, "
                            f"{E} PPO epochs x {B} minibatches, obs {d.obs} act {d.act} obj {d.obj}, 64-64 tanh MLP"
                            + (f"; every {GEN_ITERS}th step closes a generation (record all-gather + prediction-guided selection "
                               f"+ elite migration over all {n_tasks} tasks) inside the timed region" if boundary_on else ""),
                "tasks_per_gpu": P, "tasks_total": n_tasks, "envs": N, "steps": T, "ppo_epochs": E, "minibatches": B,
                "generation_iters": GEN_ITERS, "l2": "flushed between timed iterations (256 MiB write)"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        Ts, Bs = (max(T // 4, 1), max(B // 4, 1)) if args.quarter_sample else (T, B)
        r = cpu_reference_leg(d, n_tasks, Ts, N, E, Bs, gamma, args.steps, min(args.warmup, 1), boundary=boundary_on)
        sample = (f"each step = one MOPG iteration of ALL {n_tasks} tasks ({P} per GPU x {world} GPUs) on T={Ts} steps x {N} envs with "
                  f"{Bs} minibatches of {Ts * N // Bs} rows x {E} epochs, process per task, 1 torch thread each, {r['procs']} processes"
                  + (f"; CPU-oracle selection (scipy least_squares + python scoring) at every {GEN_ITERS}th step" if boundary_on else ""))
        workload_ref = dict(workload, steps=Ts, minibatches=Bs)
        line = {"impl": "reference", "metric": metric, "value": r["value"], "unit": "env-steps/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_ref,
                "mopg_only": {"ms_per_step": r["mopg_only_ms_per_step"],
                              "value": n_tasks * Ts * N / (r["mopg_only_ms_per_step"] * 1e-3)},
                "boundary_ms": r["boundary_ms"],
                "cpu_baseline": {"value": r["value"], "unit": "env-steps/s", "cores": r["procs"], "kind": r["kind"],
                                 "host_cores": os.cpu_count(), "sample": sample},
                "e2e": {"value": r["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
        return 0

    # ------------------------------------------------------------------ our arm (B200)
    import torch
    import torch.distributed as dist
    from pgmorl_b200.population_state import PopulationMOPG

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        from pgmorl_b200 import dist as pdist
        # every rank pair's NCCL channels are opened once at start-up, at the size of one migrated state, as morl.run does
        pdist.warm_up_p2p(dev, n_elems=pdist.sample_state_len(d))
    pop = PopulationMOPG(d, P, T, N, ppo_epoch=E, num_mini_batch=B, gamma=gamma, device=dev, cluster=args.cluster)
    pop.alloc_snapshots(GEN_ITERS)
    # rank r owns the global tasks {r, r + W, ...} (dist.shard_tasks); inputs seeded per rank
    traj, eps, perm, weights, obj_var, flats = synthetic_inputs(d, P, T, N, E, seed=1 + rank, first_task=rank * P)
    for p in range(P):
        pop.load_task(p, flats[p], weights=weights[p], obj_var=obj_var[p])
    pop.set_lr(3e-4)
    host = dict(obs=traj["obs"], rewards=traj["rewards"], masks=traj["masks"], bad_masks=traj["bad_masks"],
                eps=eps.to(torch.float32), perm=perm.to(torch.int32))
    pop.upload(**host)                      # also leaves the inputs in the pinned staging buffers
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    gb = GenerationBoundary(d, n_tasks, world, rank, pop=pop) if boundary_on else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)
    bnd_log = []

    def boundary(i):
        if gb is not None and (i + 1) % GEN_ITERS == 0:
            # the boundary consumes the finished generation (the objectives come from evaluating the final policies):
            # wait for the queued iterations first so that the host-side breakdown below is the boundary's own time
            torch.cuda.synchronize()
            bnd_log.append(gb.run())

    def prepare(i):
        if gb is not None and (i + 1) % GEN_ITERS == 0:
            gb.prepare()

    def run_device(steps):
        """-> (device ms per step incl. boundaries, device ms per step of the MOPG part alone)"""
        marks = []
        for i in range(steps):
            flush.fill_(i & 0xFF)                      # evict L2 between timed iterations (not timed)
            prepare(i)
            s, m, e = ev(), ev(), ev()
            s.record()
            pop.step()
            pop.snapshot(i)
            m.record()
            boundary(i)
            e.record()
            marks.append((s, m, e))
        torch.cuda.synchronize()
        return (sum(s.elapsed_time(e) for s, m, e in marks) / steps, sum(s.elapsed_time(m) for s, m, e in marks) / steps)

    def run_e2e(steps):
        """Host wall clock: blocking H2D of this step's inputs (pinned) -> K1-K3 -> D2H of the losses -> host wait, plus
        the generation boundary. -> (ms per step incl. boundaries, ms per step of the MOPG part alone)"""
        tot = mopg = 0.0
        for i in range(steps):
            flush.fill_(i & 0xFF)
            prepare(i)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pop.step_from_staged(snapshot_slot=i)
            t1 = time.perf_counter()
            boundary(i)
            t2 = time.perf_counter()
            tot += t2 - t0; mopg += t1 - t0
        return 1e3 * tot / steps, 1e3 * mopg / steps

    # stage breakdown (K1 / K2 / K3) with events around each launch, a few steps, outside the timed runs
    def stage_times(steps=10):
        from pgmorl_b200 import kernels as K
        acc = np.zeros(3)
        for i in range(steps):
            flush.fill_(i)
            e0, e1, e2, e3 = ev(), ev(), ev(), ev()
            e0.record()
            K.policy_forward(pop.params, pop.obs, d, eps=pop.eps, rows_a=S, out=(pop.value, pop.action, pop.logp))
            e1.record()
            K.gae_adv(pop.rewards, pop.value.view(P, T + 1, N, d.obj), pop.masks, pop.bad_masks, gamma, 0.95,
                      weights=pop.weights, obj_var=pop.obj_var, out=(pop.returns, pop.adv))
            e2.record()
            K.ppo_update(pop.params, pop.adam_m, pop.adam_v, pop.adam_step, pop.lr, pop.obs, pop.action, pop.logp,
                         pop.value, pop.returns.view(P, S, d.obj), pop.adv.view(P, S), pop.perm, B, d,
                         hyper=pop.hyper, workspace=pop.workspace, cluster=args.cluster, losses=pop.losses)
            e3.record()
            torch.cuda.synchronize()
            acc += (e0.elapsed_time(e1), e1.elapsed_time(e2), e2.elapsed_time(e3))
        return acc / steps

    run_device(max(args.warmup, 3))
    run_e2e(3)
    if gb is not None:
        gb.run(); gb.run()             # two untimed boundaries: K4 / K5 / NCCL warm-up (lazy module loading, communicator)
    bnd_log.clear()
    clocks = ClockSampler(local_rank if rank == 0 else None)     # rank 0 samples its GPU; started BEFORE the barrier so that
    clocks.start()                                                 # the fork of the sampler does not skew the ranks
    barrier()
    t0 = time.perf_counter()
    ms, ms_mopg = run_device(args.steps)
    n_bnd_device = len(bnd_log)
    barrier()
    ms_e2e, ms_e2e_mopg = run_e2e(args.steps)
    barrier()
    t1 = time.perf_counter()
    clk = clocks.stop(t0, t1)
    bnd_timed = list(bnd_log)
    if args.dump_outputs and rank == 0:
        # taken here: the generation and stage-time runs below move the population state on
        dump_outputs(args.dump_outputs, {k: getattr(pop, k).cpu().numpy() for k in (
            "params", "adam_m", "adam_v", "adam_step", "value", "action", "logp", "returns", "adv", "losses", "weights")})
    # one whole generation as a unit: GEN_ITERS e2e steps + the boundary, wall clock (skipped steps never happen: the
    # boundary fires on the last of the GEN_ITERS steps)
    gen = None
    if gb is not None:
        bnd_log.clear()
        gb.prepare()
        barrier()
        tg0 = time.perf_counter()
        for i in range(GEN_ITERS):
            pop.step_from_staged(snapshot_slot=i)
            boundary(i)
        barrier()
        gen_s = time.perf_counter() - tg0
        gen = {"wall_ms": 1e3 * gen_s, "iterations": GEN_ITERS, "boundary": bnd_log[-1] if bnd_log else None}
    stages = stage_times()
    if world > 1:
        t = torch.tensor([ms, ms_e2e, ms_mopg, ms_e2e_mopg, gen["wall_ms"] if gen else 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e, ms_mopg, ms_e2e_mopg, gw = t.tolist()
        if gen:
            gen["wall_ms"] = gw
    bnd_max = None
    if gb is not None and bnd_timed:          # slowest rank's time in each timed boundary (rank 0's breakdown is in per_boundary)
        tot = torch.tensor([sum(v for k, v in b.items() if k.endswith("_s")) for b in bnd_timed], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        bnd_max = [1e3 * x for x in tot.tolist()]
    picks_equal = None
    if gb is not None and world > 1:      # every rank must have picked the same (elite, weight) pairs in every generation
        hsh = int(hashlib.sha256(repr(gb.picks).encode()).hexdigest()[:15], 16)
        tt = torch.tensor([hsh], device=dev, dtype=torch.int64)
        lst = [torch.zeros_like(tt) for _ in range(world)]
        dist.all_gather(lst, tt)
        picks_equal = bool(all(int(x) == hsh for x in lst))
    finite = bool(torch.isfinite(pop.params).all() and torch.isfinite(pop.losses).all())
    ffma_measured = None
    if rank == 0:
        try:
            ffma_measured = measure_ffma_peak(dev, torch.cuda.get_device_properties(dev).multi_processor_count)
        except Exception:
            ffma_measured = None

    if rank == 0:
        env_steps = world * P * S
        fwd, upd = flops_per_env_step(d, E)
        k1b, k2b, k3b = bytes_per_env_step(d, E)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        sm_max = peaks.get("sm_max_mhz", 1965.0)
        ffma_nominal = 2 * 128 * 148 * sm_max * 1e6 / 1e12       # FP32 FFMA TFLOP/s at the max SM clock (128 lanes per SM)
        # denominator of the FP32 roofline: the nominal rate, which profiles/micro/ffma_rate.cu reproduces on this part
        # (127.7 FMA/clk/SM with FFMA2 = 74.3 TFLOP/s at 1 965 MHz). The live burn kernel of this run is reported next to it;
        # it reaches ~80 % of that (operand selection costs it register-bank conflicts) and is NOT used as the peak: a lower
        # denominator would only flatter the fraction.
        ffma_peak = max(ffma_nominal, ffma_measured[0]) if ffma_measured else ffma_nominal
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        k3_ms = float(stages[2])
        k3_tflops = P * S * upd / (k3_ms * 1e-3) / 1e12
        # which K3 kernel ran: the tensor-core path (tcgen05 on FP16 operand pairs) is chosen explicitly (cluster 32) or by
        # the library from 8 tasks on for the shapes it is built for; otherwise the FP32 FFMA cluster kernels
        wide = (d.obs, d.act, d.obj) == (376, 17, 2)          # Humanoid: the streamed tensor-core kernel (csrc/k3_tcw.cuh)
        cl = args.cluster & 0xFF
        tc = (cl in (32, 64) or (wide and cl in (0, 128)) or
              (cl == 0 and P >= 8 and (d.obs, d.act, d.obj) in ((17, 6, 2), (11, 3, 3))))
        kernel = "k3_tcw_kernel" if (tc and wide) else ("k3_tc_kernel" if tc else "k3_ppo_fast_kernel")
        traffic, traffic_src = measured_traffic(f"{kernel}:{args.config}")
        common = {"unit": "TFLOP/s", "achieved": k3_tflops, "traffic": traffic, "traffic_source": traffic_src,
                  "algorithmic_bytes_per_launch": P * S * k3b / E, "algorithmic_flops_per_launch": P * S * upd,
                  "launch_ms": k3_ms, "hbm_achieved_gbs": P * S * k3b / (k3_ms * 1e-3) / 1e9, "hbm_peak_gbs": hbm_peak,
                  "hbm_peak_source": "measured" if peaks else "fallback",
                  "fp32_ffma_peak_tflops": ffma_peak, "frac_of_fp32_ffma_peak": k3_tflops / ffma_peak}
        if tc:
            tpeak = peaks.get("bf16_tflops_sustained", 1400.0)    # FP16 and BF16 UMMA run at the same rate
            roofline = dict(common, kernel=kernel, bound="tensor", peak=tpeak, frac=k3_tflops / tpeak,
                            peak_source=("measured" if peaks else "fallback") + " dense 16-bit tensor peak (sustained)",
                            note="algorithmic FLOPs; the kernel executes 3 MMAs per product (FP16 operand pairs, FP32-level "
                                 "accuracy) on 128xNx16 tiles with N <= 64, which are shared-memory-operand bound (113 B/clk "
                                 "measured, profiles/tc_mma_bench.py), and its tanh epilogues are XU-pipe bound: see "
                                 "profiles/README_r01.md")
        else:
            roofline = dict(common, kernel=kernel, bound="fp32-ffma", peak=ffma_peak, frac=k3_tflops / ffma_peak,
                            peak_source=(f"2*128 lanes*148 SMs*{sm_max:.0f} MHz; profiles/micro/ffma_rate.cu measures 127.7 FMA/clk/SM with "
                                         "FFMA2 on this part (no FP32 peak in MEASURED_PEAKS.json); a live FFMA2 burn of this run is in "
                                         "fp32_ffma_measured_tflops"),
                            fp32_ffma_nominal_tflops=ffma_nominal,
                            fp32_ffma_measured_tflops=({"burst": ffma_measured[0], "sustained_4ms": ffma_measured[1]} if ffma_measured else None),
                            note="small populations are latency/occupancy bound: 6 chains of 320 dependent Adam steps")
        launches_per_step = pop.GPU_LAUNCHES_PER_STEP
        line = {
            "metric": metric, "value": env_steps / (ms * 1e-3), "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload,
            "clocks": clk,
            "mopg_only": {"value": env_steps / (ms_mopg * 1e-3), "ms_per_step": ms_mopg,
                          "note": "the same timed steps without the generation-boundary work (round-1 definition of value)"},
            "e2e": {"value": env_steps / (ms_e2e * 1e-3), "unit": "env-steps/s", "ms_per_step": ms_e2e,
                    "mopg_only_ms_per_step": ms_e2e_mopg, "timer": "host wall clock, blocking H2D -> K1-K3 -> D2H per step",
                    "h2d_bytes_per_step": pop.h2d_bytes, "d2h_bytes_per_step": pop.d2h_bytes},
            # K1, K2, pack, K3 per step in both timed loops; per generation boundary the archive filter (2), K4 (1), K5 init /
            # finish (2) and one scoring + one pick launch per selected task
            "gpu_launches": launches_per_step * args.steps * 2 + len(bnd_timed) * (5 + 2 * n_tasks),
            "roofline": roofline,
            "stages_ms": {"k1_forward": float(stages[0]), "k2_gae_adv": float(stages[1]), "k3_pack_ppo": k3_ms},
            "stage_hbm_gbs": {"k1_forward": P * (S + N) * k1b / (stages[0] * 1e-3) / 1e9,
                              "k2_gae_adv": P * S * k2b / (stages[1] * 1e-3) / 1e9},
            "ppo_cluster": args.cluster, "k3_path": "tensor-core" if tc else "fp32-ffma", "finite": finite,
        }
        if gen is not None:
            gen["env_steps_per_s"] = env_steps * GEN_ITERS / (gen["wall_ms"] * 1e-3)
            gen["unit"] = "env-steps/s over one generation (GEN_ITERS x [H2D + K1-K3 + D2H] + record exchange + selection + migration), wall clock"
            line["generation"] = gen
            line["boundaries_in_timed_region"] = {"device_loop": n_bnd_device, "e2e_loop": len(bnd_timed) - n_bnd_device,
                                                  "per_boundary": bnd_timed, "boundary_ms_max_over_ranks": bnd_max,
                                                  "picks_identical_on_all_ranks": picks_equal}
        if world == 1 and not args.no_selection:
            try:
                line["selection"] = selection_leg(cpu=not args.no_cpu_baseline)
            except Exception as ex:
                line["selection"] = {"error": repr(ex)[:200]}
        if world == 1 and not args.no_api and d.obj == 2:
            try:
                line["api"] = api_leg(d, P, T, N, E, B, gamma, dev, args.cluster)
                line["api"]["bulk_ms_per_iteration"] = ms_e2e_mopg
            except Exception as ex:
                line["api"] = {"error": repr(ex)[:300]}
        if world == 1 and not args.no_cpu_baseline:
            # fresh CPU-only process: fork-based worker pools cannot follow CUDA/autograd use in this one
            env_cpu = dict(os.environ, CUDA_VISIBLE_DEVICES="")
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2",
                                    "--warmup", "1", "--config", args.config, "--no-boundary"],
                                   capture_output=True, text=True, env=env_cpu, timeout=900)
                ref = json.loads(r.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = ref["cpu_baseline"]
                line["cpu_baseline"]["ms_per_step"] = ref["ms_per_step"]
                line["cpu_baseline"]["sample"] += "; 2 timed steps after 1 warm-up, no generation boundary in this sample"
            except Exception as ex:   # keep the GPU numbers even if the CPU leg fails
                line["cpu_baseline"] = {"error": repr(ex)[:200]}
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
