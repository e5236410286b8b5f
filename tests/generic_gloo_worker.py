"""One gloo rank (CPU) of the multi-rank generic batch: ``GroupedExecutor`` with a comm under ``run_batch``, the
way ``generic_batch_plot`` drives them under ``torchrun``, with a fake group function in place of the GPU work.

Every scenario runs the same item list on every rank; the rank prints one ``RESULT <json>`` line per scenario
with what it returned, which groups it processed and which progress-file writes it made.  Rank 0 also runs each
scenario as one process (no comm) from the same starting progress file, for comparison.
usage: generic_gloo_worker.py RANK WORLD PORT WORKDIR
"""

import functools
import json
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# name, items, group size, items already completed in the starting progress file
SCENARIOS = [
    ("uneven", [f"i{k}" for k in range(11)] + ["empty"], 2, []),
    ("fewer_items_than_ranks", ["only"], 3, []),
    ("nothing_pending", ["a", "b"], 2, ["a", "b"]),
    ("group_raises", [f"i{k}" for k in range(5)] + ["boom"] + [f"j{k}" for k in range(4)], 2, []),
    ("resume", [f"i{k}" for k in range(13)] + ["empty"], 2, ["i1", "i4", "i5", "i12"]),
]


def main():
    rank, world, port, work = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=port, RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist

    from configurable_spectrograms_b200 import batch_runner
    from configurable_spectrograms_b200.batch_runner import run_batch
    from configurable_spectrograms_b200.comm import TorchComm
    from configurable_spectrograms_b200.generic_batch import GroupedExecutor

    dist.init_process_group("gloo", rank=rank, world_size=world)
    comm = TorchComm(dist, group=dist.new_group(backend="gloo"))
    writes = []

    def spy_open(path, mode="r", *args, **kwargs):
        if "w" in mode:
            writes.append(os.path.basename(path))
        return open(path, mode, *args, **kwargs)

    batch_runner.open = spy_open  # module global: shadows the builtin inside run_batch only

    def run(name, items, group_size, done, with_comm):
        groups = []

        def process(group):
            groups.append(list(group))
            if "boom" in group:
                raise RuntimeError("group machinery failed")
            return [(item, "no_data" if item == "empty" else "ok") for item in group]

        tag = f"{name}_{'ranks' if with_comm else 'single'}"
        path = os.path.join(work, f"{tag}.json")
        if done and (rank == 0 or not with_comm):
            with open(path + ".tmp", "w") as handle:
                json.dump({"completed_items": [repr(x) for x in done], "errors": [], "no_data": [], "last_index": len(done) - 1,
                           "schema_version": 1}, handle)
            shutil.move(path + ".tmp", path)
        if with_comm:
            dist.barrier()  # the starting file exists before any rank looks for it
        writes.clear()
        res = run_batch(items, None, functools.partial(GroupedExecutor, process, group_size, comm if with_comm else None),
                        progress_json_path=path, flush_batch_size=2, install_signal_handlers=False,
                        _comm=comm if with_comm else None)
        if with_comm:
            dist.barrier()  # rank 0's last write is on disk before anyone reads the final file
        with open(path) as handle:
            final = json.load(handle)
        return {"results": sorted(map(list, res)), "groups": groups, "writes": list(writes), "final": final}

    for name, items, group_size, done in SCENARIOS:
        out = {"scenario": name, "rank": rank, **run(name, items, group_size, done, True)}
        if rank == 0:
            out["single"] = run(name, items, group_size, done, False)
        print("RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
