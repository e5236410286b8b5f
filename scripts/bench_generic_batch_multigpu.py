#!/usr/bin/env python
"""generic_batch_plot on BASELINE config 5 items across the GPUs of one box: one process per GPU.

    torchrun --nproc-per-node N scripts/bench_generic_batch_multigpu.py --items-per-rank K   # weak scaling
    torchrun --nproc-per-node N scripts/bench_generic_batch_multigpu.py --items M            # strong scaling

Every item is a generic stress cube (100 000 time x 96 x 64, float32, 2.46 GB) that ``build_datasets_fn`` makes
from the item's seed, so each rank only ever holds the cubes of its own items.  One untimed call (one item per
rank) creates the contexts and pinned buffers; the timed call runs between two barriers and ends when every
rank's PNG files are written.  Rank 0 prints one JSON line: wall seconds, items/s, input GB/s (cube bytes over
wall time), the mean time ``build_datasets_fn`` took per item (host work inside the timed call), and the GPU's
name and power limit.
"""

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

T, P, E = 100_000, 96, 64
TILE = 1_000  # rows drawn from the item's seed; the cube repeats them


def make_builder(build_seconds: list):
    times = 946684800.0 + 0.02 * np.arange(T)
    energy = np.geomspace(4.0, 30000.0, E)[::-1].astype(np.float32)

    def build(item):
        t0 = time.perf_counter()
        rng = np.random.default_rng(1000 + item)
        tile = (rng.random((TILE, P, E), dtype=np.float32) * 1000.0).astype(np.float32)
        tile[rng.random((TILE, P, E)) < 0.005] = np.nan
        cube = np.empty((T, P, E), np.float32)
        cube.reshape(T // TILE, TILE, P, E)[:] = tile
        build_seconds.append(time.perf_counter() - t0)
        return [{"x": times, "y": energy, "data": cube, "label": f"cube {item}", "y_max": 4000}]

    return build


def gpu_identity(device: int) -> dict:
    import torch

    out = {"gpu": torch.cuda.get_device_name(device), "power_limit_w": "unknown"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", f"--id={device}"],
                           capture_output=True, text=True, timeout=30)
        if q.returncode == 0 and q.stdout.strip():
            out["power_limit_w"] = float(q.stdout.strip().splitlines()[0])
    except (OSError, ValueError, subprocess.SubprocessError):
        pass
    return out


def main():
    ap = argparse.ArgumentParser()
    mode = ap.add_mutually_exclusive_group(required=True)
    mode.add_argument("--items-per-rank", type=int, help="weak scaling: this many items per rank")
    mode.add_argument("--items", type=int, help="strong scaling: this many items in all")
    ap.add_argument("--group", type=int, default=2, help="items per rank and round (CSG_GENERIC_GROUP)")
    ap.add_argument("--workers", type=int, default=2, help="max_workers of generic_batch_plot")
    args = ap.parse_args()
    os.environ["CSG_GENERIC_GROUP"] = str(args.group)

    import torch
    import torch.distributed as dist

    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA GPU")
    torch.cuda.set_device(local)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank = dist.get_rank() if world > 1 else 0

    from configurable_spectrograms_b200.generic_batch import generic_batch_plot

    box = [tempfile.mkdtemp(prefix="generic_multigpu_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None) if rank == 0 else None]
    if world > 1:
        dist.broadcast_object_list(box, src=0)
    work = box[0]
    n_items = args.items if args.items is not None else args.items_per_rank * world
    build_seconds: list = []
    build = make_builder(build_seconds)

    def run(tag, items):
        return generic_batch_plot(items, os.path.join(work, tag), build, y_scale="linear", z_scale="log", colormap="viridis",
                                  max_workers=args.workers, progress_json_path=os.path.join(work, f"{tag}.json"),
                                  install_signal_handlers=False)

    try:
        run("warmup", list(range(10_000, 10_000 + world)))
        build_seconds.clear()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        res = run("timed", list(range(n_items)))
        if world > 1:
            dist.barrier()
        wall = time.perf_counter() - t0
        builds = [build_seconds]
        if world > 1:
            builds = [None] * world
            dist.all_gather_object(builds, build_seconds)
        if rank == 0:
            per_item = [s for part in builds for s in part]
            cube_bytes = 4 * T * P * E
            print(json.dumps({
                "workload": "config5 generic stress cubes (100000, 96, 64) float32, 2.46 GB each, built from a seed per item",
                "scaling": "strong" if args.items is not None else "weak", "world": world, "items": n_items,
                "items_per_rank": n_items / world, "group_per_rank": args.group, "max_workers": args.workers,
                "wall_s": round(wall, 3), "items_per_s": round(n_items / wall, 3),
                "input_gb_per_s": round(n_items * cube_bytes / wall / 1e9, 2),
                "build_s_per_item_mean": round(float(np.mean(per_item)), 3) if per_item else None,
                "statuses": sorted({status for _item, status in res}), "results": len(res),
                **gpu_identity(local),
            }), flush=True)
    finally:
        if world > 1:
            dist.barrier()
        if rank == 0:
            shutil.rmtree(work, ignore_errors=True)
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
