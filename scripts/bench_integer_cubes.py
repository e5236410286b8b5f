"""Integer count cubes read at their stored width: one GPU call, one JSON line on stdout.

(a) K1 device time (CUDA events over many launches on the launching stream) on a FAST-shaped shard of
    125 orbits x 4 instruments (T=800, P=64, E=96, 4 pitch-angle groups; larger than the 126 MB L2) for each
    integer dtype, alternated in the same call with the same counts as float32 and as float64 (the bytes the
    host-widening path moved).  Algorithmic bytes = cube bytes as stored + (G+1)*T*E float64 sums (float32
    sums for the float32 cube), reported against MEASURED_PEAKS.json hbm_gbs (when present) and the 7.49 TB/s
    read ceiling of DESIGN.md section 4.
(b) Wall clock of FAST_plot_spectrograms_directory on a tree of CDF_UINT2 files against the same counts as
    CDF_DOUBLE, alternated, and whether both runs wrote identical PNG files and extrema JSON.

usage: python scripts/bench_integer_cubes.py [--orbits 125] [--reps 20] [--rounds 5] [--tree-orbits 16] [--out DIR]
"""

from __future__ import annotations

import argparse
import contextlib
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from unittest import mock

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

READ_CEILING_GBS = 7490.0  # DESIGN.md section 4: pure-read stream ceiling with K1's addressing (scripts/read_bw.cu)
T, P, E, G = 800, 64, 96, 4


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def k1_timing(args):
    import torch

    from configurable_spectrograms_b200 import _lib
    from configurable_spectrograms_b200.engine import Batch, compute_dtype
    from configurable_spectrograms_b200.fast.pipeline import pitch_angle_bits
    from configurable_spectrograms_b200 import synth
    from configurable_spectrograms_b200.fast.constants import DEFAULT_PITCH_ANGLE_CATEGORIES

    ctx = _lib.Context(0)
    dev = torch.device("cuda", 0)
    n_files = 4 * args.orbits
    bits, keys = pitch_angle_bits(synth.pitch_angle_bins(), DEFAULT_PITCH_ANGLE_CATEGORIES)
    assert len(keys) == G
    gen = torch.Generator(device=dev).manual_seed(7)
    counts = torch.randint(0, 128, (n_files, T, P, E), generator=gen, device=dev, dtype=torch.int16)  # every dtype holds them
    # the counts are below 128: an unsigned cube has the bits of the signed one of its width and shares its memory
    kinds = {"int8": torch.int8, "uint8": "int8", "int16": torch.int16, "uint16": "int16", "int32": torch.int32,
             "uint32": "int32", "float32": torch.float32, "float64": torch.float64}
    batches, tensors, ref_sums = {}, {}, None
    for name, tdt in kinds.items():
        cube = tensors[tdt] if isinstance(tdt, str) else counts.to(tdt)
        tensors[name] = cube
        D = compute_dtype(np.dtype(name))
        b = Batch(ctx, D, n_groups=G)
        step = cube[0].numel() * cube.element_size()
        for i in range(n_files):
            b.add_file(None, bits, shape=(T, P, E), layout=_lib.LAYOUT_TPE, device_ptr=cube.data_ptr() + i * step, cube_dtype=np.dtype(name))
        b.collapse()
        kern = {key[:2] for key in b.d_files}
        assert kern == {(_lib.LAYOUT_TPE, _lib.K1_STREAM)}, (name, kern)
        got = np.concatenate([b.sums(i, g).astype(np.float64).ravel() for i in (0, n_files - 1) for g in range(G + 1)])
        if ref_sums is None:
            ref_sums = got
        assert np.array_equal(got, ref_sums), name  # every dtype collapses to the same sums
        batches[name] = b
    del counts
    torch.cuda.synchronize()
    times = {name: [] for name in kinds}
    for _ in range(args.rounds):
        for name, b in batches.items():
            b._launch_k1(b.d_files, b.d_runs, b.d_bits)  # warm
            ctx.timer_start(0)
            for _ in range(args.reps):
                b._launch_k1(b.d_files, b.d_runs, b.d_bits)
            ctx.timer_stop(0)
            times[name].append(ctx.timer_ms(0) / args.reps)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    out = {}
    for name, ms in times.items():
        es = np.dtype(name).itemsize
        sums_es = 4 if name == "float32" else 8
        nbytes = n_files * (T * P * E * es + (G + 1) * T * E * sums_es)
        med = float(np.median(ms))
        rate = nbytes / (med / 1e3) / 1e9
        out[name] = {"k1_ms_median": round(med, 4), "k1_ms_min": round(min(ms), 4), "k1_ms_max": round(max(ms), 4),
                     "algorithmic_bytes": int(nbytes), "achieved_gbs": round(rate, 1),
                     "of_read_ceiling": round(rate / READ_CEILING_GBS, 3),
                     "of_measured_peak": round(rate / float(peaks["hbm_gbs"]), 3) if "hbm_gbs" in peaks else None}
    ctx.sync()
    return {"files": n_files, "shape_tpe": [T, P, E], "groups": G, "reps_per_round": args.reps, "rounds": args.rounds,
            "measured_peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "not present",
            "read_ceiling_gbs": READ_CEILING_GBS, "by_dtype": out}


def _write_tree(root, n_orbits, dtype):
    """A synthetic FAST tree whose files are real CDF files with ``data`` of ``dtype`` (the same counts for
    every dtype: the synthetic Poisson counts with NaN set to 0)."""
    from configurable_spectrograms_b200 import synth
    from tests import cdf_writer as W

    manifest = synth.write_fast_directory(os.path.join(root, "FAST_data"), n_orbits, seed=5, dtype=np.float64,
                                          csv_path=os.path.join(root, "FAST_Cusp_Indices.csv"))
    stored = 0
    with mock.patch.dict(W.CDF_TYPES, {np.dtype(np.uint16): 12}):  # CDF_UINT2, which the test writer does not list
        for files in manifest["orbits"].values():
            for path in files.values():
                arrays = dict(np.load(path + ".npz"))
                os.remove(path + ".npz")
                arrays["data"] = np.nan_to_num(arrays["data"], nan=0.0).astype(dtype)
                stored += arrays["data"].nbytes
                W.write_fast_cdf(path, arrays)
    return stored


def _digest(base):
    h = {}
    for dirpath, _dirs, fs in os.walk(base):
        for fn in fs:
            p = os.path.join(dirpath, fn)
            h[os.path.relpath(p, base)] = hashlib.sha256(open(p, "rb").read()).hexdigest()
    return h


def directory_timing(args, work):
    from configurable_spectrograms_b200 import cdf_utils
    from configurable_spectrograms_b200.fast.batch_directory import FAST_plot_spectrograms_directory

    trees = {}
    for name, dt in (("uint16", np.uint16), ("float64", np.float64)):
        root = os.path.join(work, name)
        os.makedirs(root)
        trees[name] = (root, _write_tree(root, args.tree_orbits, dt))
    here = os.getcwd()
    wall = {name: [] for name in trees}
    digests = {}
    try:
        for rep in range(args.dir_reps + 1):  # rep 0 warms up
            for name, (root, _) in trees.items():
                os.chdir(root)
                cdf_utils.filtered_orbits_cache.clear()
                cdf_utils.orbit_column_cache.clear()
                out = f"./plots_{rep}/"
                t0 = time.perf_counter()
                res = FAST_plot_spectrograms_directory("./FAST_data", output_base=out, y_scale="linear", z_scale="log",
                                                       colormap="cividis", max_processing_percentile=99, max_workers=2,
                                                       progress_json_path=f"./progress_{rep}.json")
                dt = time.perf_counter() - t0
                if rep:
                    wall[name].append(dt)
                else:
                    digests[name] = (sorted((r["orbit"], r["status"]) for r in res), _digest(out),
                                     open("./FAST_calculated_extrema.json").read())
    finally:
        os.chdir(here)
    same = digests["uint16"] == digests["float64"]
    return {"orbits": args.tree_orbits, "instruments": 4, "reps": args.dir_reps,
            "cube_bytes_as_stored": {name: int(b) for name, (_, b) in trees.items()},
            "wall_s_median": {name: round(float(np.median(v)), 3) for name, v in wall.items()},
            "wall_s_all": {name: [round(x, 3) for x in v] for name, v in wall.items()},
            "identical_outputs": bool(same), "pngs": len(digests["float64"][1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--orbits", type=int, default=125)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--tree-orbits", type=int, default=16)
    ap.add_argument("--dir-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this directory")
    args = ap.parse_args()
    card = _card()
    result = {"bench": "integer_cubes", "card": card, "k1": k1_timing(args)}
    work = tempfile.mkdtemp(prefix="csg_int_tree_")
    try:
        with contextlib.redirect_stdout(sys.stderr):  # the driver's log lines; stdout carries the JSON line only
            result["directory"] = directory_timing(args, work)
    finally:
        shutil.rmtree(work, ignore_errors=True)
    line = json.dumps(result)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        open(os.path.join(args.out, "integer_cubes.json"), "w").write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
