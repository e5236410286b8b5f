"""torchrun worker for the multi-GPU generic batch and stand-alone extrema test.  Rank 0 first runs
``generic_batch_plot`` as one process (before the job's process group exists); then every rank runs it over the
same items under ``torchrun``, and the statuses, the progress JSON and the pixels of every ``generic.png`` must
match the single-process run.  Then stand-alone ``compute_global_extrema`` on the golden tree must return the
reference's dicts on every rank and read no cube once its cache is complete.
With fewer GPUs than ranks the ranks share the GPUs over a gloo process group and only the generic batch runs
(its exchanges are host objects; the extrema exchange needs one GPU per rank).
usage: multigpu_generic_worker.py WORKDIR (the golden tree written there by the parent test)
"""

import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ORDER = ("ees", "eeb", "ies", "ieb")


def _items_and_builder():
    import numpy as np

    from tests.helpers import dataset_from_arrays, load_npz

    tree = load_npz("extrema_tree.npz")
    orbits = sorted({int(k.split("_")[0]) for k in tree if k[0].isdigit()})
    items = [f"{o}_{kind}" for o in orbits for kind in ("f32", "f64")] + ["nodata", "raises"]

    def build(item):
        if item == "nodata":
            return []
        if item == "raises":
            raise RuntimeError("this item's builder fails")
        orbit, kind = item.split("_")
        out = []
        for inst in ORDER:
            if f"{orbit}_{inst}_data" not in tree:
                continue
            ds = dataset_from_arrays({v: tree[f"{orbit}_{inst}_{v}"] for v in ("time_unix", "data", "energy", "pitch_angle")})
            data = ds["data"].astype(np.float64) if kind == "f64" else ds["data"]
            out.append({"x": ds["times"], "y": ds["energy"], "data": data, "label": inst})
        return out

    return items, build


def _plot(items, build, tag):
    from configurable_spectrograms_b200.generic_batch import generic_batch_plot

    return generic_batch_plot(items, f"./generic_{tag}", build, y_scale="linear", z_scale="log", colormap="viridis",
                              max_workers=1, progress_json_path=f"./generic_{tag}.json", flush_batch_size=3,
                              install_signal_handlers=False)


def _sorted_lists(state):
    return {k: sorted(v) if isinstance(v, list) else v for k, v in state.items()}


def main():
    import numpy as np
    import torch

    os.chdir(sys.argv[1])
    local = int(os.environ["LOCAL_RANK"])
    shared = torch.cuda.device_count() < int(os.environ["WORLD_SIZE"])
    device = local % torch.cuda.device_count()
    torch.cuda.set_device(device)
    items, build = _items_and_builder()
    if local == 0:  # the single-process run, in the same job, before the process group exists
        single = _plot(items, build, "single")
        assert sorted(single) == sorted(
            [(x, "ok") for x in items if x not in ("nodata", "raises")] + [("nodata", "no_data"), ("raises", "error")]), single

    import torch.distributed as dist

    from configurable_spectrograms_b200 import _lib, cdf_utils, png
    from configurable_spectrograms_b200.fast.extrema import compute_global_extrema
    from tests.helpers import load_json

    if shared:
        dist.init_process_group("gloo")
    else:
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))
    rank, world = dist.get_rank(), dist.get_world_size()

    # ---- generic_batch_plot across the ranks
    res = _plot(items, build, "ranks")
    everyone = [None] * world
    dist.all_gather_object(everyone, sorted(res))
    assert all(r == everyone[0] for r in everyone), everyone
    # the groups of this rank ran on its own GPU: no context on another device was ever created
    assert set(_lib._default_ctx) == {device}, (rank, sorted(_lib._default_ctx))
    dist.barrier()
    if rank == 0:
        assert sorted(res) == sorted(single), (res, single)
        ranks_json, single_json = json.load(open("./generic_ranks.json")), json.load(open("./generic_single.json"))
        assert _sorted_lists(ranks_json) == _sorted_lists(single_json), (ranks_json, single_json)
        drawn = [x for x, status in single if status == "ok"]
        for item in drawn:
            a = png.decode_rgba(open(f"./generic_ranks/{item}/generic.png", "rb").read())
            b = png.decode_rgba(open(f"./generic_single/{item}/generic.png", "rb").read())
            assert np.array_equal(a, b), item
        assert not os.path.exists("./generic_ranks/nodata") and not os.path.exists("./generic_ranks/raises")

    if shared:
        dist.barrier()
        if rank == 0:
            print(f"MULTIGPU_GENERIC_OK world={world} shared_gpus={torch.cuda.device_count()}")
        dist.destroy_process_group()
        return

    # ---- stand-alone compute_global_extrema across the ranks
    gold = load_json("extrema_tree.json")
    for kwargs, path, key in ((dict(max_percentile=99.0), "./FAST_calculated_extrema.json", "batch_extrema"),
                              (dict(compute_mins=True), "./other.json", "pool95_mins")):
        zs = "log" if key == "batch_extrema" else "linear"
        got = compute_global_extrema("./FAST_data", "linear", zs, ORDER, extrema_json_path=path, **kwargs)
        assert got == gold[key], (rank, key, got, gold[key])
        dist.barrier()
        assert json.load(open(path)) == gold[key], (rank, key)
        # the cache is complete: a second call plans no scan and reads no cube
        real, reads = cdf_utils.load_fast_cdf_dataset, []
        cdf_utils.load_fast_cdf_dataset = lambda *a, **k: (reads.append(a), real(*a, **k))[1]
        try:
            again = compute_global_extrema("./FAST_data", "linear", zs, ORDER, extrema_json_path=path, **kwargs)
        finally:
            cdf_utils.load_fast_cdf_dataset = real
        assert again == gold[key] and reads == [], (rank, key, len(reads))
        dist.barrier()
    assert set(_lib._default_ctx) == {device}, (rank, sorted(_lib._default_ctx))
    dist.barrier()
    if rank == 0:
        print(f"MULTIGPU_GENERIC_OK world={world} shared_gpus=0")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
