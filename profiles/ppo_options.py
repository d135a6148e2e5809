"""Cost of the non-default PPO options on the GPU: K2 per return branch of compute_returns, and K3 with the clipped
against the unclipped value loss, at the shapes of bench.py's configs. CUDA events around back-to-back launches on
device-resident inputs (the K2 inputs of 256 tasks are 80 MB, so the smaller populations run from L2 after the first
pass; stated in the output). Prints a report and writes it to the path given (default profiles/r04/ppo_options.txt).

    python profiles/ppo_options.py [out.txt]
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pgmorl_b200 import kernels as K, synthetic          # noqa: E402
from pgmorl_b200.layout import NetDims                    # noqa: E402

BRANCHES = [("A gae+ptl", True, True), ("B nstep+ptl", False, True), ("C gae", True, False), ("D nstep", False, False)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi unavailable"


def time_ms(fn, reps):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def k2_rows(P, T=2048, N=4, M=2, reps=200):
    g = torch.Generator(device="cuda").manual_seed(P)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    rew, val = r(P, T, N, M), r(P, T + 1, N, M)
    masks = (torch.rand(P, T + 1, N, device="cuda", generator=g) > 0.01).float()
    bad = (torch.rand(P, T + 1, N, device="cuda", generator=g) > 0.01).float()
    w, ov, boot = torch.full((P, M), 1.0 / M, device="cuda"), torch.ones(P, M, device="cuda"), r(P, N, M)
    out = (torch.empty_like(rew), torch.empty(P, T, N, device="cuda"))
    rows = []
    for name, gae, ptl in BRANCHES:
        f = lambda: K.returns_adv(rew, val, masks, bad, 0.995, 0.95, use_gae=gae, use_proper_time_limits=ptl, weights=w,
                                  obj_var=ov, boot=None if gae else boot, out=out)
        rows.append((name, 1e3 * time_ms(f, reps)))
    return rows


def k3_rows(d, P, T, N, E=10, B=32, reps=5):
    traj = synthetic.make_trajectories(P, T, N, d, seed=1)
    S = T * N
    params = torch.stack([synthetic.init_policy_flat(d, seed=100 + p) for p in range(P)]).float().cuda()
    obs = traj["obs"].float().cuda().reshape(P, (T + 1) * N, d.obs)
    eps, perm = synthetic.host_rng_streams(0, T, N, d.act, E)
    value, action, logp = K.policy_forward(params, obs, d, eps=eps.float().cuda().reshape(1, S, d.act), rows_a=S)
    ret, adv = K.gae_adv(traj["rewards"].float().cuda(), value.view(P, T + 1, N, d.obj), traj["masks"].float().cuda(),
                         traj["bad_masks"].float().cuda(), 0.995, 0.95, weights=torch.full((P, d.obj), 0.5, device="cuda"))
    perm = perm.to(torch.int32).cuda()[None].contiguous()
    lr = torch.full((P,), 3e-4, dtype=torch.float64, device="cuda")
    ws = K.ppo_workspace(P, S, d, "cuda")
    rows = []
    for clipped in (True, False):
        p0 = params.clone()
        m, v, st = torch.zeros_like(p0), torch.zeros_like(p0), torch.zeros(P, dtype=torch.int32, device="cuda")
        f = lambda: K.ppo_update(p0, m, v, st, lr, obs, action, logp, value, ret.view(P, S, d.obj), adv.view(P, S), perm,
                                 B, d, workspace=ws, clipped_value_loss=clipped)
        rows.append(("clipped" if clipped else "unclipped", time_ms(f, reps)))
    return rows


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r04", "ppo_options.txt")
    lines = [f"# card (name, power limit, max SM clock): {card()}",
             "# K2: us per launch (returns + scalarised normalised advantage), T = 2048, N = 4, M = 2, 200 back-to-back launches",
             "#     on resident inputs (P = 6 and 64 fit in L2; P = 256 is 80 MB of inputs)"]
    for P in (6, 64, 256):
        lines.append(f"K2 P={P:4d}  " + "  ".join(f"{n}: {us:8.2f} us" for n, us in k2_rows(P)))
    lines.append("# K3: ms per MOPG iteration (record pack + E x B = 10 x 32 Adam steps), auto plan, 5 back-to-back updates")
    for name, d, P, N in (("c2", NetDims(17, 6, 2), 6, 4), ("walker64", NetDims(17, 6, 2), 64, 4),
                          ("humanoid8", NetDims(376, 17, 2), 8, 8)):
        rows = k3_rows(d, P, 2048, N)
        ratio = rows[1][1] / rows[0][1]
        lines.append(f"K3 {name:10s} " + "  ".join(f"{n}: {ms:8.4f} ms" for n, ms in rows) + f"  unclipped/clipped {ratio:.4f}")
    text = "\n".join(lines) + "\n"
    print(text, end="")
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
