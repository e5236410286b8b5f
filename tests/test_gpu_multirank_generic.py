"""generic_batch_plot and stand-alone compute_global_extrema under torchrun: the ranks share the work on their own
GPUs and return what one process returns (``tests/multigpu_generic_worker.py``).  With fewer GPUs than ranks the
ranks share the GPUs and only the generic batch runs."""

import os
import subprocess
import sys

import pytest

from tests.test_gpu_api import _write_tree

pytestmark = pytest.mark.gpu


def test_generic_batch_and_standalone_extrema_across_ranks(tmp_path):
    n_ranks = int(os.environ.get("CSG_TEST_WORLD", "2"))  # 8: more ranks than some rounds have items (empty slices)
    _write_tree(tmp_path)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    # two items per rank and round: several rounds, the last one uneven
    env = dict(os.environ, CSG_GENERIC_GROUP="2")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n_ranks}", "--master-addr", "127.0.0.1",
           "--master-port", "29543", os.path.join(root, "tests", "multigpu_generic_worker.py"), str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root, env=env)
    if r.returncode != 0:  # the whole log in the test's temporary directory (the assertion shows its tails)
        (tmp_path / "multigpu_generic_worker_failure.log").write_text(r.stdout + "\n=====\n" + r.stderr)
    assert r.returncode == 0 and f"MULTIGPU_GENERIC_OK world={n_ranks} " in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
