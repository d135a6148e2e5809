"""K1 + K3 time per MOPG iteration at hidden widths 32 / 64 / 128 (profiles/r06/README.md).

    python profiles/hidden_width.py [--out FILE]

Workloads: C2 (6 tasks, T 2048 x 4 envs, 10 epochs x 32 minibatches of 256 rows, Walker2d dims) and the same iteration
for 64 Walker2d tasks. Per width and workload: K1 over the whole trajectory (value for (T+1) N rows, sampled actions for
T N), then K3 (pack + update) on the auto plan, timed with CUDA events over 5 iterations after 2 warm-up iterations. Width
64 runs the kernels the default policy runs (tensor-core K3 from 8 tasks on); 32 and 128 run the FFMA kernels. The card's
name and power limit are printed with the numbers."""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pgmorl_b200 import kernels as K, synthetic  # noqa: E402
from pgmorl_b200.layout import NetDims  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def time_iteration(P, H, T=2048, N=4, E=10, B=32, reps=5, warm=2):
    d = NetDims(17, 6, 2, H)
    dev = torch.device("cuda")
    S = T * N
    params = torch.stack([synthetic.init_policy_flat(d, seed=p) for p in range(P)]).float().to(dev)
    m, v = torch.zeros_like(params), torch.zeros_like(params)
    step = torch.zeros(P, dtype=torch.int32, device=dev)
    lr = torch.full((P,), 3e-4, dtype=torch.float64, device=dev)
    g = torch.Generator(device="cpu").manual_seed(0)
    obs = torch.randn(P, (T + 1) * N, d.obs, generator=g).to(dev)
    eps = torch.randn(1, S, d.act, generator=g).to(dev)
    ret = torch.randn(P, S, d.obj, generator=g).to(dev)
    adv = torch.randn(P, S, generator=g).to(dev)
    perm = torch.stack([torch.randperm(S, generator=g) for _ in range(E)]).to(torch.int32).to(dev)[None].contiguous()
    ws = K.ppo_workspace(P, S, d, dev)
    k1, k3 = [], []
    for i in range(warm + reps):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        value, action, logp = K.policy_forward(params, obs, d, eps=eps, rows_a=S)
        e1.record()
        K.ppo_update(params, m, v, step, lr, obs, action, logp, value, ret, adv, perm, B, d, workspace=ws)
        e2.record()
        torch.cuda.synchronize()
        if i >= warm:
            k1.append(e0.elapsed_time(e1)); k3.append(e1.elapsed_time(e2))
    assert torch.isfinite(params).all()
    return float(np.median(k1)), float(np.median(k3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = [f"card: {card()}  (name, power limit, max SM clock)",
             "median of 5 MOPG iterations after 2 warm-up; ms per iteration (K1 over T+1 steps, K3 = pack + E x B Adam steps)",
             f"{'workload':24s} {'H':>4s} {'K1 ms':>9s} {'K3 ms':>9s} {'K1+K3 ms':>9s}"]
    for name, P in (("C2 (6 tasks)", 6), ("64 Walker tasks", 64)):
        for H in (32, 64, 128):
            t1, t3 = time_iteration(P, H)
            lines.append(f"{name:24s} {H:4d} {t1:9.3f} {t3:9.3f} {t1 + t3:9.3f}")
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
