"""Full-size prediction-guided selection at 3 objectives with large archives: K5's shared-memory path against its
global-memory path (csrc/k5_select.cu, PGM_SEL_GLOBAL).

For archives of 500, 2 000, 5 000, 10 000 and 20 000 points, tests/synth_envs.make_selection_state(3, 420, n_ep) gives
the full-size problem (420 members, ~2 940 candidates, 15 tasks). One prediction_guided_selection call per size
records K5's inputs and is timed as a whole; then `kernels.select_greedy` runs on those inputs:
  * warm-up: one call of every path timed below;
  * REPS timed calls, host clock with a device synchronise on both sides; at 500 and 2 000 points (where both paths
    run) the default and the forced global path alternate, and their outputs are compared bit for bit.
The working set of the global path (per-CTA scratch + base data) is stated against the card's L2 size. The card's
name, power limit and max SM clock are read in the same run.

    python profiles/selection_large3d.py [--out DIR] [--reps N] [--sizes 500,2000,...]
Writes DIR/selection_large3d.json and DIR/selection_large3d.txt (default DIR: profiles/r08).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import synth_envs                                          # noqa: E402
from pgmorl_b200 import kernels as K                       # noqa: E402
from pgmorl_b200._lib import lib                           # noqa: E402
from pgmorl_b200.scalarization_methods import WeightedSumScalarization   # noqa: E402

N_POP = 420
SHARED_LIMIT = 2111          # archive + num_tasks + 1 of the shared-memory incremental scorer
CTAS = 296                   # S3G_CTAS in csrc/k5_select.cu


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi unavailable"


def selection_call(n_ep):
    """One prediction_guided_selection on a fresh state; -> (seconds, K5 inputs of the greedy call)."""
    args, graph, pop, ep = synth_envs.make_selection_state(3, N_POP, n_ep)
    template = WeightedSumScalarization(num_objs=3, weights=np.ones(3) / 3)
    seen, real = [], K.select_greedy

    def spy(e, c, alpha, num_tasks, **kw):
        if num_tasks == args.num_tasks:
            seen.append((np.array(e), np.array(c), alpha, num_tasks))
        return real(e, c, alpha, num_tasks, **kw)
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


def timed(inputs, force_global):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = K.select_greedy(*inputs, force_global=force_global)       # ends in device -> host copies
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sizes", default="500,2000,5000,10000,20000")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    os.makedirs(a.out, exist_ok=True)
    props = torch.cuda.get_device_properties(0)
    l2 = int(getattr(props, "L2_cache_size", 0))
    rep = {"card": card(), "device": props.name, "sms": props.multi_processor_count, "l2_bytes": l2,
           "n_pop": N_POP, "reps": a.reps, "sizes": []}
    lines = [f"card: {rep['card']}  ({props.name}, {props.multi_processor_count} SMs, L2 {l2 / 2**20:.0f} MiB)"]
    for n_ep in [int(s) for s in a.sizes.split(",")]:
        call_s, inputs = selection_call(n_ep)
        ep, cand, alpha, T = inputs
        E, C = len(ep), len(cand)
        nmax = E + T + 1
        both = nmax <= SHARED_LIMIT
        ws_default = int(lib().pgm_select_workspace_bytes_x(E, C, 3, T, 0))
        ws_global = int(lib().pgm_select_workspace_bytes_x(E, C, 3, T, 1))
        scratch = min(C, CTAS) * (97 * nmax + 16)
        paths = [False, True] if both else [False]
        ref = {}
        for g in paths:                                               # warm-up
            ref[g] = timed(inputs, g)[1]
        times = {g: [] for g in paths}
        for _ in range(a.reps):
            for g in paths:                                           # alternate the paths
                dt, out = timed(inputs, g)
                assert same(out, ref[g]), "a repeated call changed its output"
                times[g].append(dt)
        identical = same(ref[False], ref[True]) if both else None
        row = {"archive": E, "candidates": C, "tasks": T, "front_max": nmax,
               "default_path": "shared" if both else "global",
               "whole_call_s": call_s,
               "k5_default_s": times[False], "k5_global_s": times.get(True),
               "paths_bit_identical": identical,
               "workspace_default_bytes": ws_default, "workspace_global_bytes": ws_global,
               "global_scratch_bytes": scratch, "scratch_over_l2": scratch / l2 if l2 else None}
        rep["sizes"].append(row)
        line = (f"archive {E:6d}  candidates {C}  tasks {T}  default={row['default_path']:6s}  "
                f"whole call {call_s:.3f} s  K5 default min {min(times[False]):.3f} s")
        if both:
            line += f"  K5 global min {min(times[True]):.3f} s  bit-identical {identical}"
        line += f"  global scratch {scratch / 2**20:.0f} MiB ({row['scratch_over_l2']:.2f} x L2)"
        lines.append(line)
        print(line, flush=True)
    with open(os.path.join(a.out, "selection_large3d.json"), "w") as f:
        json.dump(rep, f, indent=1)
    with open(os.path.join(a.out, "selection_large3d.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
