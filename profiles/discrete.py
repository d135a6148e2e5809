"""Time per MOPG iteration (K1 + K2 + K3) of a Categorical policy next to a Box policy of the same dims.

    python profiles/discrete.py [--out FILE]

Shape (O, A or n, M) = (2, 4, 2), Deep-Sea-Treasure-like, hidden width 64, at 6 and 64 tasks. Each iteration is the C2
schedule (T 2048 x 4 envs, 10 epochs x 32 minibatches of 256 rows) run by PopulationMOPG.step(): K1 over the whole
trajectory, K2, then K3 (pack + update) on the auto plan. Categorical heads run the generic cluster kernel; the Box
policy of these dims runs what the planner picks for it (the fast cluster kernel). Timed with CUDA events around each
iteration after overwriting a 256 MB buffer (L2 flushed); median of 5 after 2 warm-up iterations. The card's name and
power limit are printed with the numbers."""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pgmorl_b200 import synthetic  # noqa: E402
from pgmorl_b200.layout import DIST_CATEGORICAL, DIST_GAUSSIAN, NetDims  # noqa: E402
from pgmorl_b200.population_state import PopulationMOPG  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def time_iteration(P, dist, T=2048, N=4, E=10, B=32, reps=5, warm=2):
    d = NetDims(2, 4, 2, 64, dist)
    pop = PopulationMOPG(d, P, T, N, ppo_epoch=E, num_mini_batch=B)
    S = T * N
    g = torch.Generator(device="cpu").manual_seed(0)
    for p in range(P):
        pop.load_task(p, synthetic.init_policy_flat(d, seed=p), weights=np.full(d.obj, 1.0 / d.obj), obj_var=np.ones(d.obj))
    pop.set_lr(3e-4)
    traj = synthetic.make_trajectories(P, T, N, d, seed=1)
    pop.obs.copy_(traj["obs"].reshape(P, (T + 1) * N, d.obs))
    pop.rewards.copy_(traj["rewards"]); pop.masks.copy_(traj["masks"]); pop.bad_masks.copy_(traj["bad_masks"])
    eps = torch.empty(1, S, d.act, dtype=torch.float64)
    eps.exponential_(1, generator=g) if dist == DIST_CATEGORICAL else eps.normal_(0, 1, generator=g)
    pop.eps.copy_(eps)
    pop.perm.copy_(torch.stack([torch.randperm(S, generator=g) for _ in range(E)]).to(torch.int32)[None])
    flush = torch.empty(64 * 2 ** 20, dtype=torch.float32, device="cuda")      # 256 MB > 126 MB of L2
    times = []
    for i in range(warm + reps):
        flush.fill_(float(i))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pop.step()
        e1.record()
        torch.cuda.synchronize()
        if i >= warm:
            times.append(e0.elapsed_time(e1))
    assert torch.isfinite(pop.params).all() and torch.isfinite(pop.losses).all()
    return float(np.median(times)), float(np.min(times)), float(np.max(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = [f"card: {card()}  (name, power limit, max SM clock)",
             "(O, A|n, M) = (2, 4, 2), hidden 64, T 2048 x 4 envs, 10 epochs x 32 minibatches; ms per MOPG iteration "
             "(K1 + K2 + K3, L2 flushed), median [min, max] of 5 after 2 warm-up",
             f"{'tasks':>5s} {'head':12s} {'median':>9s} {'min':>9s} {'max':>9s}"]
    for P in (6, 64):
        for name, dist in (("Box", DIST_GAUSSIAN), ("Categorical", DIST_CATEGORICAL)):
            med, lo, hi = time_iteration(P, dist)
            lines.append(f"{P:5d} {name:12s} {med:9.3f} {lo:9.3f} {hi:9.3f}")
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
