"""The sharded generation loop on real GPUs over NCCL (SURVEY 8(e), morl/morl.py:84-143): two ranks, one GPU each, run
`pgmorl_b200.morl.run` under torch.distributed.run on the replay environments of the whole-run golden. Asserted:
 (i)   the gathered metadata (archive, population, opt-graph) and the selected (elite, weight) pairs of every generation
       are bit-identical on both ranks and equal to the single-GPU run's;
 (ii)  every file the run writes equals the single-GPU run's byte for byte (text) / bit for bit (policies, moments) -- which
       includes the parameters, Adam state and running moments of elites that MIGRATED between the GPUs;
 (iii) the result still matches the unmodified reference's golden run within 1e-4.
Skipped below 2 visible GPUs."""
import os
import pickle
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _launch(nproc, save_dir, method):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(HERE, "dist_run_worker.py"), save_dir, method]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def _tree(root):
    out = {}
    for d, _, files in os.walk(root):
        for f in files:
            if not f.startswith("rank"):
                out[os.path.relpath(os.path.join(d, f), root)] = os.path.join(d, f)
    return out


@pytest.mark.parametrize("method", ["prediction-guided", "moead"])
def test_two_gpu_run_equals_single_gpu_run(tmp_path, method):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 visible GPUs")
    one, two = str(tmp_path / "w1"), str(tmp_path / "w2")
    os.makedirs(one), os.makedirs(two)
    _launch(1, one, method)
    _launch(2, two, method)
    ref = pickle.load(open(os.path.join(one, "rank0.pkl"), "rb"))
    ranks = [pickle.load(open(os.path.join(two, f"rank{r}.pkl"), "rb")) for r in range(2)]
    # (i) identical metadata and identical picks on every rank, equal to the single-GPU run
    for got in ranks:
        for key in ("ep_objs", "pop_objs", "graph_objs"):
            assert np.array_equal(got[key], ref[key]), key
        assert got["pop_nodes"] == ref["pop_nodes"] and got["graph_prev"] == ref["graph_prev"]
        assert len(got["timings"]) == len(ref["timings"]) == 3
        for tg, tr in zip(got["timings"], ref["timings"]):
            assert tg["elite_nodes"] == tr["elite_nodes"]
            assert all(np.array_equal(a, b) for a, b in zip(tg["weights"], tr["weights"]))
    assert sum(t["migrated"] for t in ranks[0]["timings"]) > 0, "no elite changed owner: migration not exercised"
    owned = sorted(ranks[0]["owned_ep"] + ranks[1]["owned_ep"])
    assert owned == list(range(len(ref["ep_objs"]))), "every archive member's state lives on exactly one rank"
    # (ii) every file identical
    a, b = _tree(one), _tree(two)
    assert sorted(a) == sorted(b)
    for k in sorted(a):
        if k.endswith(".txt"):
            assert open(a[k]).read() == open(b[k]).read(), k
        elif k.endswith(".pt"):
            x, y = torch.load(a[k]), torch.load(b[k])
            assert list(x) == list(y) and all(torch.equal(x[n], y[n]) for n in x), k
        elif k.endswith(".pkl"):
            x, y = pickle.load(open(a[k], "rb")), pickle.load(open(b[k], "rb"))
            for key in ('ob_rms', 'ret_rms', 'obj_rms'):
                if x[key] is None:
                    assert y[key] is None
                    continue
                assert np.array_equal(np.asarray(x[key].mean), np.asarray(y[key].mean)), (k, key)
                assert np.array_equal(np.asarray(x[key].var), np.asarray(y[key].var)), (k, key)
    # (iii) the reference's golden run
    gold = os.path.join(GOLDEN, "run_2d" if method == "prediction-guided" else "run_2d_" + method)
    got = np.loadtxt(os.path.join(two, "final", "objs.txt"), delimiter=",")
    want = np.loadtxt(os.path.join(gold, "final", "objs.txt"), delimiter=",")
    assert np.allclose(got, want, rtol=1e-4, atol=2e-6)
