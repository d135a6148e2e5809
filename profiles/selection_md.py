"""Prediction-guided selection at 4 objectives on the GPU, at a mid size (120 members, archive of 200) and at the size
of the 3-objective full-size problem (420 members, ~3 400 candidates, archive of 500), built by
tests/synth_envs.make_selection_state. Reports, best of 3 each:
  * the whole `prediction_guided_selection` call (host clock, device synchronise on both sides);
  * K5 alone (`kernels.select_greedy` on the call's own inputs) and per greedy round;
  * the literal restatement of the reference's scorer (tests/hv_ref.py: update_ep + hypervolume + sparsity) per
    candidate on one host core, on a few of the call's round-0 candidates -- what the reference pays per candidate
    per round, in a process per candidate.
Prints a report and writes it to the path given (default profiles/r05/selection_md.txt).

    python profiles/selection_md.py [out.txt]
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import hv_ref                                              # noqa: E402
import synth_envs                                          # noqa: E402
from oracle import selection_oracle as so                  # noqa: E402
from pgmorl_b200 import kernels as K                       # noqa: E402
from pgmorl_b200.scalarization_methods import WeightedSumScalarization   # noqa: E402

SIZES = [("mid", 120, 200), ("full", 420, 500)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi unavailable"


def selection_call(n_pop, n_ep):
    """One prediction_guided_selection on a fresh state; -> (seconds, K5 inputs)."""
    args, graph, pop, ep = synth_envs.make_selection_state(4, n_pop, n_ep)
    template = WeightedSumScalarization(num_objs=4, weights=np.ones(4) / 4)
    seen, real = [], K.select_greedy

    def spy(e, c, alpha, num_tasks):
        if num_tasks == args.num_tasks:
            seen.append((np.array(e), np.array(c), alpha, num_tasks))
        return real(e, c, alpha, num_tasks)
    K.select_greedy = spy
    try:
        np.random.seed(0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pop.prediction_guided_selection(args, 0, ep, graph, template)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        K.select_greedy = real
    return dt, seen[0]


def main(out_path):
    lines = [f"card: {card()}", "float64 K5, 4 objectives; best of 3; host clock with torch.cuda.synchronize() on both sides", ""]
    selection_call(40, 60)                                  # loads the module and warms every launch path
    for name, n_pop, n_ep in SIZES:
        calls = [selection_call(n_pop, n_ep) for _ in range(3)]
        ep, cand, alpha, num_tasks = calls[0][1]
        k5 = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            K.select_greedy(ep, cand, alpha, num_tasks)
            torch.cuda.synchronize()
            k5.append(time.perf_counter() - t0)
        rng = np.random.RandomState(0)
        ref = []
        for i in rng.choice(len(cand), 5, replace=False):
            t0 = time.process_time()
            front = so.update_ep(ep, cand[i])
            hv_ref.hv(front); so.sparsity_md(front)
            ref.append(time.process_time() - t0)
        lines += [f"[{name}] members {n_pop}, archive {len(ep)}, candidates {len(cand)}, rounds {num_tasks}",
                  f"  prediction_guided_selection: {min(c[0] for c in calls):.3f} s  (all: {', '.join(f'{c[0]:.3f}' for c in calls)})",
                  f"  K5 select_greedy: {min(k5):.3f} s, {1e3 * min(k5) / num_tasks:.1f} ms per greedy round",
                  f"  restatement, one host core: {np.median(ref):.3f} s per candidate (median of 5; range {min(ref):.3f}-{max(ref):.3f})",
                  f"  -> one round of the reference's scorer on one core: ~{np.median(ref) * len(cand):.0f} s", ""]
    report = "\n".join(lines)
    print(report)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(report + "\n")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r05", "selection_md.txt"))
