"""The multi-rank generic batch on CPU: gloo ranks in child processes drive ``GroupedExecutor`` (with a comm)
under ``run_batch`` as ``generic_batch_plot`` does under ``torchrun``; see ``tests/generic_gloo_worker.py``."""

import json
import os
import socket
import subprocess
import sys

import pytest

from tests.generic_gloo_worker import SCENARIOS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return str(s.getsockname()[1])


def _run(world, work):
    port = _free_port()
    procs = [
        subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "generic_gloo_worker.py"), str(r), str(world), port, str(work)],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT)
        for r in range(world)
    ]
    outs = [p.communicate(timeout=240) for p in procs]
    for p, (out, err) in zip(procs, outs):
        assert p.returncode == 0, out[-2000:] + err[-4000:]
    runs: dict = {}
    for out, _err in outs:
        for line in out.splitlines():
            if line.startswith("RESULT "):
                rec = json.loads(line[len("RESULT "):])
                runs.setdefault(rec["scenario"], {})[rec["rank"]] = rec
    assert sorted(runs) == sorted(name for name, *_ in SCENARIOS)
    return runs


def _sorted_lists(state):
    return {k: sorted(v) if isinstance(v, list) else v for k, v in state.items()}


@pytest.mark.parametrize("world", [2, 3])
def test_ranks_share_the_items_of_a_generic_batch(tmp_path, world):
    runs = _run(world, tmp_path)
    for name, items, _group, done in SCENARIOS:
        ranks = runs[name]
        assert sorted(ranks) == list(range(world)), name
        pending = [x for x in items if x not in done]
        # every item is processed by exactly one rank
        processed = [x for rec in ranks.values() for g in rec["groups"] for x in g]
        assert sorted(processed) == sorted(pending), (name, processed)
        # every rank returns the same, complete result list
        first = ranks[0]["results"]
        assert sorted(x for x, _s in first) == sorted(pending), name
        assert all(rec["results"] == first for rec in ranks.values()), name
        # rank 0 alone writes the progress file, and it writes it at least once (at the end)
        assert ranks[0]["writes"] and all(not rec["writes"] for r, rec in ranks.items() if r != 0), name
        assert all(rec["final"] == ranks[0]["final"] for rec in ranks.values()), name
        status = dict(map(tuple, first))
        if name == "group_raises":
            failed = {x for rec in ranks.values() for g in rec["groups"] if "boom" in g for x in g}
            assert "boom" in failed
            assert {x for x, s in status.items() if s == "error"} == failed
            assert all(s == "ok" for x, s in status.items() if x not in failed)
            assert sorted(ranks[0]["final"]["errors"]) == sorted(repr(x) for x in failed)
            continue
        # the same statuses and the same final progress file as one process run from the same starting file
        single = ranks[0]["single"]
        assert single["results"] == first, name
        assert _sorted_lists(ranks[0]["final"]) == _sorted_lists(single["final"]), name
        assert status.get("empty", "no_data") == "no_data"
        if name == "resume":
            assert sorted(ranks[0]["final"]["completed_items"]) == sorted(repr(x) for x in items if x != "empty")
        # a round holds up to group_size items per rank, so no group is larger than group_size
        assert max((len(g) for rec in ranks.values() for g in rec["groups"]), default=0) <= _group
