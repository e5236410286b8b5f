#!/usr/bin/env python
"""K4 with panels on a log energy axis: the time of ``png.encode_figures_device`` on the same FAST figures
(bench.py's workload: 4800 x 2400 at 200 dpi, turbo, log z) drawn once with linear y and once with log y.

The rasters are computed once (K1-K3, bench.py's synthetic orbits); the two figure lists differ only in the
y scale.  Each call encodes every figure of one variant and ends with the read-back of the files, so the host
clock around it measures the whole stage; the variants alternate within the run (linear first on even
repeats, log first on odd ones) so both see the same machine.  A few figures of each variant are compared with
the host composer first.  Prints one JSON line: seconds per call, GPU name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--orbits", type=int, default=16, help="orbits whose figures (20 each) are encoded")
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--seed", type=int, default=4)
    args = ap.parse_args()

    import torch

    import bench
    from configurable_spectrograms_b200 import _lib, png
    from configurable_spectrograms_b200.fast.pipeline import BatchStep, ShardPlan
    from configurable_spectrograms_b200.fast.plotting import figure_from_spec

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    files, orbits, total = bench.orbit_layout(args.orbits, 0, args.seed)
    cubes = bench.generate_cubes(torch, files, total, dev)
    torch.cuda.synchronize()
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = _lib.Context(0, stream=stream.cuda_stream)
    shard = ShardPlan(ctx, "linear", "log", zoom_duration_minutes=6, instrument_order=bench.ORDER)
    for ob in orbits:
        dsets = {}
        for inst, fd in ob["files"].items():
            f = files[fd["index"]]
            dsets[inst] = {"times": fd["times"], "energy": fd["energy"], "pitch_angle": fd["pitch_angle"],
                           "shape": (f["T"], bench.P, bench.E), "device_ptr": cubes.data_ptr() + 4 * f["offset"]}
        shard.add_orbit(ob["orbit"], dsets, ob["lines"])
    sequence = [(ob["orbit"], {i: True for i in bench.ORDER}) for ob in orbits]
    step = BatchStep(shard, sequence, max_percentile=99.0, lut259=bench.turbo_like_lut(), want_index=False)
    step.run({})
    step.finish()
    norms = shard.batch.norms()
    specs = [sp for ob in orbits for wx in (False, True) for sp in shard.figures[slice(*step.figure_ranges[(ob["orbit"], wx)])]]

    def figures(y_scale, device=True, which=None):
        shard.y_scale = y_scale  # figure_from_spec reads the axis scale from the shard
        try:
            chosen = specs if which is None else [specs[k] for k in which]
            return [f for f in (figure_from_spec(shard, sp, "turbo", norms=norms, device_rasters=device)[0] for sp in chosen)
                    if f is not None]
        finally:
            shard.y_scale = "linear"

    variants = {"linear": figures("linear"), "log": figures("log")}
    d_rgba = shard.batch.d_rgba.ptr
    sample = list(range(0, len(specs), max(1, len(specs) // 4)))[:4]
    for name in variants:  # parity on a few figures, and the warm-up of every shape
        dev_figs, host_figs = figures(name, True, sample), figures(name, False, sample)
        for blob, fig in zip(png.encode_figures_device(ctx, d_rgba, dev_figs, dpi=200), host_figs):
            assert np.array_equal(png.decode_rgba(blob), fig.compose(200)), f"{name}: device PNG differs from the host composer"
        png.encode_figures_device(ctx, d_rgba, variants[name], dpi=200)
    times = {name: [] for name in variants}
    kernel = {name: [] for name in variants}
    sizes = {}
    for r in range(args.repeats):
        for name in (("linear", "log") if r % 2 == 0 else ("log", "linear")):
            phases: dict = {}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            blobs = png.encode_figures_device(ctx, d_rgba, variants[name], dpi=200, timings=phases)
            times[name].append(time.perf_counter() - t0)
            kernel[name].append(phases.get("encode_kernel_and_sizes", 0.0))
            sizes[name] = sum(len(b) for b in blobs)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    out = {"gpu": smi.stdout.strip(), "figures": {k: len(v) for k, v in variants.items()},
           "canvas": [int(round(variants["linear"][0].figsize[0] * 200)), int(round(variants["linear"][0].figsize[1] * 200))],
           "repeats": args.repeats}
    for name in variants:
        t = np.array(times[name])
        out[name] = {"call_s": [round(v, 5) for v in t], "median_s": float(np.median(t)), "min_s": float(t.min()),
                     "max_s": float(t.max()), "kernel_wait_median_s": float(np.median(kernel[name])),
                     "figures_per_s": len(variants[name]) / float(np.median(t)), "png_bytes": sizes[name]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
