"""tests/dist_run_worker.py with policies of hidden width HIDDEN (tests/test_gpu_hidden.py):

    python -m torch.distributed.run ... tests/dist_run_hidden_worker.py SAVE_DIR [selection_method] HIDDEN
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import dist_run_worker  # noqa: E402
import synth_envs  # noqa: E402

HIDDEN = int(sys.argv.pop())
_run_args_2d = synth_envs.run_args_2d


def _run_args(save_dir, **kw):
    args = _run_args_2d(save_dir, **kw)
    args.hidden_size = HIDDEN
    return args


synth_envs.run_args_2d = _run_args

if __name__ == "__main__":
    dist_run_worker.main()
