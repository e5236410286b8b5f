#!/usr/bin/env python
"""bench.py -- orbits/sec of the FAST batch path (BASELINE.json metric) on N B200s.

One step = one pass of the hot path over this rank's shard of synthetic FAST orbits
(linear y / log z, turbo, max_processing_percentile=99, fresh extrema cache):

  K1  collapse every cube once (all pitch-angle groups + total + row flags)
  K2b pooled extrema: radix histograms, prefix scan, exact prefix percentiles (+ all-gather
      of bucket totals across ranks)
  K2a 1/99 percentiles + safe_vmin of every figure row
  K3  normalise + LUT rasterise every panel of every figure (pitch-angle grids given/raw for
      4 instruments + instrument grids given/raw, full + cusp-zoom columns)

``value``  : whole-job orbits/s, cubes resident in HBM, CUDA-event timed, max over ranks.
``e2e``    : same metric through the host-buffer path: H2D of the cubes from pinned memory,
             the same stages, D2H of every RGBA raster into pinned memory, inside the timed
             region.
Workload (weak scaling): 125 orbits per GPU = config 4 (1000 orbits) at 8 GPUs.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ORDER = ("ees", "eeb", "ies", "ieb")
NOMINAL_T = {"ees": 800, "ies": 800, "eeb": 903, "ieb": 903}
P, E = 64, 96
METRIC = "orbits/sec (whole box, device-timed)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--orbits-per-gpu", type=int, default=125)
    ap.add_argument("--total-orbits", type=int, default=0,
                    help="strong scaling: this many orbits in all, split over the GPUs (1000 = BASELINE config 4; fits one B200)")
    ap.add_argument("--cpu-sample-orbits", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-png", action="store_true")
    ap.add_argument("--png-orbits", type=int, default=8, help="orbits whose figures (20 each) go through the device PNG stage")
    ap.add_argument("--seed", type=int, default=4)
    ap.add_argument("--no-api-e2e", action="store_true", help="skip the public-API end-to-end leg (directory of .npz side-cars -> PNGs on disk)")
    ap.add_argument("--api-orbits", type=int, default=0, help="orbits of the api_e2e directory (default: --orbits-per-gpu)")
    ap.add_argument("--api-ref", action="store_true", help="also run the unmodified reference over the SAME api_e2e directory (minutes)")
    ap.add_argument("--no-verify", action="store_true", help="skip the parity leg (outside the timed region)")
    ap.add_argument("--verify-orbits", type=int, default=3, help="orbits of this shard whose every panel is compared with the oracle")
    ap.add_argument("--profile-region", default="steps", choices=("steps", "png"),
                    help="what sits between cudaProfilerStart/Stop for `ncu --profile-from-start off`: the timed steps or the PNG stage")
    ap.add_argument("--profile-host", default=None, help="write a cProfile of the timed step loop to this path")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


# ----------------------------------------------------------------------------------------
# synthetic workload (shapes of `FAST CDF variables.txt`; generated on the GPU with torch --
# plumbing only -- so a 10 GB shard does not take minutes of host RNG)
# ----------------------------------------------------------------------------------------
def orbit_layout(n_orbits, first_orbit, seed):
    """Host-side description of the shard: per file shape, times, cusp lines, intensity."""
    from configurable_spectrograms_b200 import synth

    rng = np.random.default_rng(seed + 7919 * first_orbit)
    energy = synth.energy_bins()
    pitch = synth.pitch_angle_bins()
    files, orbits = [], []
    offset = 0
    for k in range(n_orbits):
        g = first_orbit + k
        start = 946684800.0 + 7980.0 * g
        has_cusp = g % 3 == 0
        storm = g in (1, 2, 5)
        entry = {"orbit": 13000 + g, "files": {}, "lines": {}}
        for inst in ORDER:
            T = NOMINAL_T[inst]
            cadence = 2.5 if inst.endswith("s") else 0.6
            times = start + cadence * np.arange(T, dtype=np.float64)
            lines = []
            win = None
            if has_cusp:
                lo = int(T * 0.4) + int(rng.integers(0, 20))
                hi = lo + (47 if inst.endswith("s") else 259)
                win = (lo, hi)
                lines = [float(times[lo]), float(times[hi])]
            files.append({"inst": inst, "T": T, "offset": offset, "intensity": (8.0 if storm else 1.0) * (3.0 if inst[0] == "e" else 0.3), "win": win, "seed": seed * 100003 + g * 4 + ORDER.index(inst)})
            entry["files"][inst] = {"index": len(files) - 1, "times": times, "energy": energy, "pitch_angle": pitch}
            entry["lines"][inst] = lines
            offset += T * P * E
        orbits.append(entry)
    return files, orbits, offset


def generate_cubes(torch, files, total_elems, device):
    """Poisson counts with the structure of synth.make_cube, 1 % NaN; one flat float32 tensor."""
    cubes = torch.empty(total_elems, dtype=torch.float32, device=device)
    p = torch.arange(P, device=device, dtype=torch.float32)[None, :, None]
    e = torch.arange(E, device=device, dtype=torch.float32)[None, None, :]
    cutoff = 1e-4 + 1.0 / (1.0 + torch.exp(-(e - 0.30 * E) / 0.8))
    peak = torch.exp(-(((e - 0.55 * E) / (0.22 * E)) ** 2)) * (1.0 + 0.6 * torch.cos(2 * torch.pi * p / P))
    bump_e = torch.exp(-(((e - 0.7 * E) / (0.1 * E)) ** 2))
    gen = torch.Generator(device=device)
    for f in files:
        T = f["T"]
        gen.manual_seed(f["seed"])
        t = torch.arange(T, device=device, dtype=torch.float32)[:, None, None]
        lam = f["intensity"] * cutoff * (0.15 + peak * (1.0 + 0.5 * torch.sin(2 * torch.pi * t / T * 3.0)))
        if f["win"] is not None:
            bump = torch.zeros(T, 1, 1, device=device)
            bump[f["win"][0] : f["win"][1]] = 4.0
            lam = lam * (1.0 + bump * bump_e)
        cube = torch.poisson(lam, generator=gen)
        cube[torch.rand(cube.shape, device=device, generator=gen) < 0.01] = float("nan")
        cubes[f["offset"] : f["offset"] + T * P * E] = cube.reshape(-1)
    return cubes


def turbo_like_lut():
    """A deterministic 259 x 4 uint8 table (matplotlib's tables are not on the box; indices, not
    colours, are what parity grades)."""
    from configurable_spectrograms_b200.colormaps import get_lut

    return get_lut("turbo")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.window = [None, None]  # host perf_counter interval of the GPU work being measured

    def mark(self, which):
        self.window[which] = time.perf_counter()

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.perf_counter()] + [c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        t0, t1 = self.window
        rows = [r[1:] for r in self.rows if (t0 is None or r[0] >= t0) and (t1 is None or r[0] <= t1 + 0.15)]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = sorted({n for r in rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "window": "warm-up + timed steps + per-stage passes (GPU busy throughout)"}


# ----------------------------------------------------------------------------------------
# the reference arm / CPU baseline: the oracle port of the reference's numeric path
# ----------------------------------------------------------------------------------------
def cpu_sample_orbits(n, seed):
    from configurable_spectrograms_b200 import synth

    rng = np.random.default_rng(seed)
    out = []
    energy, pitch = synth.energy_bins(), synth.pitch_angle_bins()
    for k in range(n):
        dsets, lines = {}, {}
        for inst in ORDER:
            T = NOMINAL_T[inst]
            win = (int(T * 0.4), int(T * 0.4) + (47 if inst.endswith("s") else 259)) if k % 3 == 0 else None
            cube = synth.make_cube(rng, T, intensity=(8.0 if k == 1 else 1.0) * (3.0 if inst[0] == "e" else 0.3), cusp_window=win)
            times = synth.make_times(T, start=946684800.0 + 7980.0 * k, cadence=2.5 if inst.endswith("s") else 0.6)
            dsets[inst] = {"times": times, "data": cube, "energy": energy, "pitch_angle": pitch}
            lines[inst] = [float(times[win[0]]), float(times[win[1]])] if win else []
        out.append((13000 + k, dsets, lines))
    return out


def run_cpu_port(orbits, steps, warmup):
    from oracle import cpu_pipeline as CP

    cores = os.cpu_count() or 1
    times = []
    for i in range(warmup + steps):
        t, _state, _n = CP.run_step(orbits, "linear", "log", 99.0, workers=cores)
        if i >= warmup:
            times.append(t)
    return float(np.mean(times)), cores


def measured_read_stream_peak():
    """GB/s of a pure-read stream with K1's addressing, from the committed run of scripts/read_bw.cu."""
    import re

    try:
        text = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r1_read_bw.txt")).read()
    except OSError:
        return None
    m = re.search(r"^K1-like.*?([0-9]+\.[0-9]+) GB/s", text, re.M)
    return float(m.group(1)) if m else None


def scratch_dir(prefix):
    """A scratch directory on the fastest local filesystem (tmpfs when there is one)."""
    import tempfile

    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    return tempfile.mkdtemp(prefix=prefix, dir=base)


def workload_config(n_local, world):
    """The ``config`` both arms print (the reference arm times a bounded sample OF this workload)."""
    return {
        "workload": f"config4 shard: {n_local} orbits/GPU ({world * n_local} orbits total; 1000 at 8 GPUs), "
                    "4 instruments, FAST batch step linear y / log z, turbo, max_processing_percentile=99",
        "orbits_per_gpu": n_local, "bytes_per_orbit": int(sum(NOMINAL_T[i] for i in ORDER) * P * E * 4),
        "l2_policy": f"inputs larger than L2 ({n_local * sum(NOMINAL_T[i] for i in ORDER) * P * E * 4 / 1e9:.1f} GB of cubes streamed per step)",
    }


def run_reference_directory(n_orbits, seed, steps, warmup, render="display"):
    """The UNMODIFIED reference (``oracle/_ref``) over a synthetic directory of ``n_orbits`` orbits:
    ``FAST_plot_spectrograms_directory`` with a fork pool on every host core, fresh JSON state and
    output tree per step.  Returns (mean seconds per step, cores, pngs per step, png bytes per step)."""
    import shutil

    from oracle import ref_driver as RD

    work = scratch_dir("csg_ref_")
    try:
        RD.prepare_directory(work, n_orbits, seed=seed)
        cores = os.cpu_count() or 1
        times, last = [], None
        for i in range(warmup + steps):
            last = RD.run_directory(work, workers=cores, render=render)
            bad = [r for r in last["results"] if r.get("status") != "ok"]
            if bad:
                raise RuntimeError(f"reference run reported errors: {bad[:2]}")
            if i >= warmup:
                times.append(last["seconds"])
        return float(np.mean(times)), cores, last["pngs"], last["png_bytes"]
    finally:
        shutil.rmtree(work, ignore_errors=True)


def reference_arm(args):
    """``--impl reference``: the reference's own CPU implementation of the path on the host cores.
    ``oracle/_ref`` (the unmodified reference under the cdflib / matplotlib stand-ins of
    ``oracle/stubs.py``) when it travelled with the snapshot, else the numpy port of its numeric
    work (``oracle/cpu_pipeline.py``).  Each step = one whole batch step over a bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_driver as RD

    n = args.cpu_sample_orbits
    world = int(os.environ.get("WORLD_SIZE", "1"))
    extra = {}
    if RD.available():
        sec, cores, pngs, png_bytes = run_reference_directory(n, args.seed, args.steps, args.warmup)
        kind = "reference"
        sample = (f"{n} synthetic FAST orbits (4 instruments, nominal shapes) as .npz side-cars on tmpfs; the unmodified reference's "
                  f"FAST_plot_spectrograms_directory: serial extrema pre-pass + fork ProcessPoolExecutor({cores}), both submissions, "
                  f"{pngs} PNGs ({png_bytes / 1e6:.1f} MB) per step; cdflib -> .npz stub, matplotlib -> numpy norm+LUT, nearest "
                  "resample to figsize x dpi (4800 x 2400) + Pillow PNG (no text / Agg anti-aliasing: optimistic for the reference)")
        warm = args.warmup
        # the numeric-only port beside it (no file IO, no PNG): what round 1 reported
        psec, _ = run_cpu_port(cpu_sample_orbits(n, args.seed), 1, 0)
        extra["port_numeric_only"] = {"value": n / psec, "unit": "orbits/s", "kind": "port"}
    else:
        warm = min(args.warmup, 1)
        sec, cores = run_cpu_port(cpu_sample_orbits(n, args.seed), args.steps, warm)
        kind = "port"
        sample = f"{n} synthetic FAST orbits (4 instruments, nominal shapes), both submissions, numeric path only (no Agg/PNG): oracle/_ref did not travel"
    value = n / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "orbits/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.orbits_per_gpu, world),
        "cpu_baseline": {"value": value, "unit": "orbits/s", "cores": cores, "kind": kind, "sample": sample, "sample_orbits": n, **extra},
        "e2e": {"value": value, "unit": "orbits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ----------------------------------------------------------------------------------------
# parity leg (outside every timed region): the bench workload itself against numpy / the oracle
# ----------------------------------------------------------------------------------------
def _host_cube(cubes, f):
    n = f["T"] * P * E
    return cubes[f["offset"] : f["offset"] + n].cpu().numpy().reshape(f["T"], P, E)


def verify_shard(args, torch, cubes, files, orbits, shard, step, state, lut, rank, world):
    """``parity_checked``: (1) K1 sums of sampled files bit for bit against ``np.nansum``; (2) the global
    z_max / y_max of EVERY instrument against an independent oracle over the whole ascending orbit
    sequence -- per-file value histograms (the synthetic sums are integer counts), prefix by prefix,
    numpy's rank arithmetic restated in float32 (``oracle/restate.percentile_rank`` / ``lerp``) --
    itself pinned against brute-force ``np.nanpercentile(np.concatenate(blocks so far), p)`` on
    sampled prefixes (``CS/fast/extrema.py:270-300``); (3) every panel of every figure of both
    submissions of a few orbits -- resolved bounds and colormap index planes -- against the oracle
    port of the reference's figure builders (``oracle/cpu_pipeline.py`` + ``oracle/restate.py``)."""
    import math

    from configurable_spectrograms_b200.fast.pipeline import check_norm_status
    from oracle import cpu_pipeline as CP
    from oracle import restate as R

    t_start = time.perf_counter()
    out = {"ok": True, "failures": []}

    def fail(msg):
        out["ok"] = False
        if len(out["failures"]) < 8:
            out["failures"].append(msg)

    b = shard.batch
    energy = orbits[0]["files"][ORDER[0]]["energy"]
    # ---- (1) + per-file oracle inputs for (2)
    per_file = []  # (inst index, global orbit index, value histogram, per-energy positive counts)
    blocks = {i: [] for i in range(len(ORDER))}  # positives of this rank's first files (brute-force pin)
    n_sums_checked = 0
    first = rank * len(orbits)
    for k, ob in enumerate(orbits):
        for inst in ORDER:
            fd = ob["files"].get(inst)
            if fd is None:
                continue
            f = files[fd["index"]]
            cube = _host_cube(cubes, f)
            with np.errstate(invalid="ignore", over="ignore"):
                m = np.nansum(cube, axis=1)
            if k % 16 == 0:
                fid = shard.orbits[k]["files"][inst]
                got = b.sums(fid, 0)
                same = (got.view(np.uint32) == m.view(np.uint32)) | (np.isnan(got) & np.isnan(m))
                n_sums_checked += 1
                if not same.all():
                    fail(f"K1 total differs from np.nansum: orbit {ob['orbit']} {inst}")
            ok = np.isfinite(m) & (m > 0)
            pos = m[ok]
            if not (np.all(pos == np.floor(pos)) and (pos.size == 0 or pos.max() < 2**24)):
                fail("synthetic sums are not integer counts: the histogram oracle does not apply")
                return out
            per_file.append((ORDER.index(inst), first + k, np.bincount(pos.astype(np.int64)), ok.sum(axis=0).astype(np.int64)))
            if k < 8:
                blocks[ORDER.index(inst)].append(pos)
    out["k1_files_checked"] = n_sums_checked
    if world > 1:
        gathered = [None] * world
        torch.distributed.all_gather_object(gathered, per_file)
        per_file = [row for part in gathered for row in part]
    if rank == 0:
        e_sorted = np.sort(np.asarray(energy, dtype=np.float64))
        e_order = np.argsort(np.asarray(energy, dtype=np.float64), kind="stable")
        n_prefix, brute = 0, 0
        for ii, inst in enumerate(ORDER):
            rows = sorted((r for r in per_file if r[0] == ii), key=lambda r: r[1])
            width = max(len(r[2]) for r in rows)
            hist = np.zeros(width, dtype=np.int64)
            ecount = np.zeros(len(energy), dtype=np.int64)
            best_z, best_e = -np.inf, -np.inf
            per_prefix = []
            for _ii, _oi, h, ec in rows:
                hist[: len(h)] += h
                ecount += ec
                n = int(hist.sum())
                cand_z = 0.0
                if n:
                    lo, hi, g = R.percentile_rank(n, 99.0, np.float32)
                    cum = np.cumsum(hist)
                    a, c = np.searchsorted(cum, [lo, hi], side="right")
                    cand_z = float(R.lerp(np.float32(a), np.float32(c), g, np.float32))
                cand_e = 0.0
                if ecount.sum():
                    cum_e = np.cumsum(ecount[e_order])
                    idx = min(int(np.searchsorted(cum_e, 0.99 * cum_e[-1], side="right")), len(e_sorted) - 1)
                    # the reference keys only energies that have seen a count; zero-count keys do not move the sum
                    cand_e = float(e_sorted[idx])
                per_prefix.append(cand_z)
                best_z, best_e = max(best_z, cand_z), max(best_e, cand_e)
                n_prefix += 1
            stem = f"{inst}_linear_log"
            want_z, want_y = float(math.ceil(best_z)), int(min(4000, math.ceil(best_e)))
            if state.get(f"{stem}_z_max") != want_z:
                fail(f"{stem}_z_max: GPU {state.get(f'{stem}_z_max')} != oracle {want_z}")
            if state.get(f"{stem}_y_max") != want_y:
                fail(f"{stem}_y_max: GPU {state.get(f'{stem}_y_max')} != oracle {want_y}")
            # pin the histogram oracle itself: brute-force numpy on the first prefixes (the storm orbits live there)
            pool = []
            for k, blk in enumerate(blocks[ii]):
                pool.append(blk)
                want = float(np.nanpercentile(np.concatenate(pool), 99.0))
                brute += 1
                if per_prefix[k] != want:
                    fail(f"{inst} prefix {k}: histogram oracle {per_prefix[k]} != np.nanpercentile {want}")
        out.update(extrema_instruments=len(ORDER), extrema_prefixes_walked=n_prefix, extrema_prefixes_brute_force=brute,
                   extrema={k: v for k, v in state.items() if k.endswith(("_z_max", "_y_max"))})
    # ---- (3) panels of a few orbits of this rank: a cusp orbit, a storm orbit, a plain one
    b.rasterise(want_rgba=True, want_index=True)
    b.ctx.sync()
    norms = b.norms()
    picks = []
    for want in (lambda g: g % 3 == 0, lambda g: g in (1, 2, 5), lambda g: g % 3 != 0 and g not in (1, 2, 5)):
        picks += [k for k in range(len(orbits)) if want(first + k) and k not in picks][:1]
    picks = (picks + [k for k in range(len(orbits)) if k not in picks])[: max(1, args.verify_orbits)]
    old_native = CP.NATIVE_LOG
    CP.NATIVE_LOG = False  # the correctly rounded float32 log10 the parity tests grade against
    n_panels = n_figs = 0

    def compare(fig, expected, what):
        nonlocal n_panels
        exp = iter(expected)
        need = fig.zoom is not None and fig.zoom_needed
        for row in fig.rows:
            for pid in [row.full_panel] + ([row.zoom_panel] if need else []):
                e = next(exp, "missing")
                if isinstance(e, str):
                    return fail(f"{what}: the oracle draws fewer panels")
                if pid is None:
                    if e is not None:
                        fail(f"{what}: panel missing on the GPU side")
                    continue
                try:
                    check_norm_status(norms[pid], str(what))
                except ValueError:
                    if e is not None:
                        fail(f"{what}: norm rejected on the GPU side only")
                    continue
                if e is None:
                    fail(f"{what}: norm rejected by the oracle only")
                elif not np.array_equal(b.panel_index(pid), e[0]):
                    fail(f"{what} {row.label}: colormap index plane differs")
                n_panels += 1
        if next(exp, "end") != "end":
            fail(f"{what}: the oracle draws more panels")

    try:
        with np.errstate(all="ignore"):
            for k in sorted(picks):
                ob = orbits[k]
                dsets = {inst: {"times": fd["times"], "energy": fd["energy"], "pitch_angle": fd["pitch_angle"],
                                "data": _host_cube(cubes, files[fd["index"]])} for inst, fd in ob["files"].items()}
                lines = ob["lines"]
                for wx in (False, True):
                    figs = iter(shard.figures[slice(*step.figure_ranges[(ob["orbit"], wx)])])
                    extrema = state if wx else None
                    for inst in ORDER:
                        ov = R.extrema_overrides(extrema, inst, "linear", "log")
                        for variant, kw in (("given", dict(y_min=ov[0], y_max=ov[1], z_min=ov[2], z_max=ov[3])), ("raw", {})):
                            fig = next(figs)
                            compare(fig, CP.pitch_angle_grid(dsets[inst], lines.get(inst), "log", lut, minutes=6, **kw),
                                    (ob["orbit"], inst, variant, wx))
                            n_figs += 1
                    first_lines = next((lines.get(i) for i in ORDER if i in dsets), None)
                    for variant, ge in (("given", extrema), ("raw", None)):
                        fig = next(figs)
                        compare(fig, CP.instrument_grid(dsets, first_lines, "log", lut, ge, "linear", minutes=6),
                                (ob["orbit"], "grid", variant, wx))
                        n_figs += 1
    finally:
        CP.NATIVE_LOG = old_native
    out.update(panel_orbits=[orbits[k]["orbit"] for k in sorted(picks)], figures_checked=n_figs, panels_checked=n_panels,
               seconds=round(time.perf_counter() - t_start, 2))
    if world > 1:  # every rank checked its own panels: one verdict
        oks = [None] * world
        torch.distributed.all_gather_object(oks, (out["ok"], n_panels, out["failures"]))
        out["ok"] = all(o[0] for o in oks)
        out["panels_checked"] = sum(o[1] for o in oks)
        out["failures"] = [m for o in oks for m in o[2]][:8]
    return out


# ----------------------------------------------------------------------------------------
# api_e2e: the call a user makes -- FAST_plot_spectrograms_directory on a directory -> PNGs on disk
# ----------------------------------------------------------------------------------------
def write_api_directory(work, cubes, files, orbits, n_orbits):
    """The first ``n_orbits`` orbits of this rank's synthetic shard as a FAST tree: empty ``.cdf`` markers +
    ``.cdf.npz`` side-cars (what both arms read; CDF decoding itself is out of scope) + the cusp TSV."""
    from concurrent.futures import ThreadPoolExecutor
    from datetime import datetime, timezone

    from configurable_spectrograms_b200 import synth

    root = os.path.join(work, "FAST_data")
    rows = [synth.CUSP_CSV_COLUMNS]
    jobs = []
    for ob in orbits[:n_orbits]:
        start = float(ob["files"][ORDER[0]]["times"][0])
        dt = datetime.fromtimestamp(start, tz=timezone.utc)
        folder = os.path.join(root, f"{dt.year:04d}", f"{dt.month:02d}")
        os.makedirs(folder, exist_ok=True)
        cells = {}
        for inst in ORDER:
            fd = ob["files"][inst]
            f = files[fd["index"]]
            path = os.path.join(folder, synth.fast_filename(inst, start, ob["orbit"]))
            jobs.append((path, f, fd))
            cells[inst] = (os.path.basename(path),) + (tuple(str(v) for v in f["win"]) if f["win"] else ("", ""))
        rows.append("\t".join([str(ob["orbit"]), folder, f"fa_k0_orb_{ob['orbit']}_v01.cdf", "0", "0"]
                              + [x for inst in ("eeb", "ees", "ieb", "ies") for x in ("True",) + cells[inst]]))

    def write(job):
        path, f, fd = job
        open(path, "wb").close()
        np.savez(path + ".npz", time_unix=fd["times"], data=_host_cube(cubes, f),
                 energy=np.asarray(fd["energy"], np.float32)[None, None, :], pitch_angle=np.asarray(fd["pitch_angle"], np.float32)[None, :, None])

    with ThreadPoolExecutor(max_workers=8) as pool:
        list(pool.map(write, jobs))
    with open(os.path.join(work, "FAST_Cusp_Indices.csv"), "w") as fh:
        fh.write("\n".join(rows) + "\n")
    return len(jobs)


def api_e2e_leg(args, cubes, files, orbits, state, with_reference, dist=None, rank=0, world=1):
    """Wall clock of the public API on a fresh directory: discovery, streaming ingest through pinned
    slots, K1, the global-extrema pre-pass, planning, K2a, K3, K4 and the PNG files on disk.  With several
    ranks the directory is rank 0's shard and every rank takes its share of those orbits (the same directory,
    more GPUs: strong scaling of the call); the clock is the slowest rank's."""
    import shutil

    from configurable_spectrograms_b200 import cdf_utils, overlay
    from configurable_spectrograms_b200.fast.batch_directory import FAST_plot_spectrograms_directory

    n = min(args.api_orbits or args.orbits_per_gpu, len(orbits))
    cwd = os.getcwd()
    box = [None, 0, 0.0]
    if rank == 0:
        work = scratch_dir("csg_api_")
        t0 = time.perf_counter()
        box = [work, write_api_directory(work, cubes, files, orbits, n), time.perf_counter() - t0]
    if world > 1:
        dist.broadcast_object_list(box, src=0)
    work, n_files, t_write = box

    def clock():
        """seconds since the previous call, as the maximum over ranks (ranks leave a barrier together)"""
        if world > 1:
            dist.barrier()
        now = time.perf_counter()
        sec, clock.t = now - clock.t, now
        return sec

    clock.t = 0.0
    try:
        os.chdir(work)
        out = {}
        for label in ("cold", "warm", "warm2"):  # cold: first call of the process (plans, scratch, page cache); warm: steady state
            if rank == 0:
                for name in ("progress.json", "FAST_calculated_extrema.json"):
                    if os.path.exists(name):
                        os.remove(name)
                shutil.rmtree("FAST_plots", ignore_errors=True)
            cdf_utils.filtered_orbits_cache.clear()
            cdf_utils.orbit_column_cache.clear()
            # every run composes its text sprites anew: a directory of NEW orbits has its own times of day, titles
            # and colour-bar values, and a warm run over the same orbits would find them all in the atlas
            overlay.ATLAS.clear()
            phases: dict = {}
            prof = None
            if label == "warm2" and os.environ.get("CSG_API_PROFILE") and rank == 0:  # main-thread cProfile of one steady-state call
                import cProfile

                prof = cProfile.Profile()
                prof.enable()
            clock()
            res = FAST_plot_spectrograms_directory(
                "./FAST_data", output_base="./FAST_plots/", y_scale="linear", z_scale="log", zoom_duration_minutes=6, colormap="turbo",
                max_processing_percentile=99, max_workers=16, progress_json_path="./progress.json", verbose=False, _timings=phases,
            )
            sec = clock()
            if prof is not None:
                import pstats

                prof.disable()
                with open(os.environ["CSG_API_PROFILE"], "w") as fh:
                    pstats.Stats(prof, stream=fh).sort_stats("cumulative").print_stats(70)
                    pstats.Stats(prof, stream=fh).sort_stats("tottime").print_stats(40)
            if rank != 0:
                continue
            bad = [r for r in res if r.get("status") != "ok"]
            pngs = sum(len(fs) for _d, _s, fs in os.walk("./FAST_plots"))
            png_bytes = sum(os.path.getsize(os.path.join(d, f)) for d, _s, fs in os.walk("./FAST_plots") for f in fs)
            got = json.load(open("./FAST_calculated_extrema.json"))
            out[label] = {"seconds": sec, "orbits_per_s": n / sec, "pngs": pngs, "png_mb": png_bytes / 1e6, "errors": len(bad),
                          "results": len(res), "phases_s": {k: round(v, 4) for k, v in phases.items()}}
        if rank != 0:
            return None
        if out["warm2"]["seconds"] < out["warm"]["seconds"]:  # `warm` = the better of the two steady-state calls
            out["warm"], out["warm2"] = out["warm2"], out["warm"]
        # the same extrema as the device-resident arm computed for these orbits?  (only when the directory IS the shard)
        same = None
        if n == len(orbits) and world == 1:
            same = all(got.get(k) == v for k, v in state.items() if k.endswith(("_z_max", "_y_max")))
        line = {"value": out["warm"]["orbits_per_s"], "unit": "orbits/s", "orbits": n, "files": n_files, "n_gpus": world,
                "input_gb": sum(files[fd["index"]]["T"] for ob in orbits[:n] for fd in ob["files"].values()) * P * E * 4 / 1e9,
                "directory_write_s": round(t_write, 2), "cold": out["cold"], "warm": out["warm"], "warm_other": out["warm2"], "extrema_equal_device_arm": same,
                "what": "FAST_plot_spectrograms_directory(dir, max_processing_percentile=99, turbo) on .npz side-cars in tmpfs -> "
                        "PNG files at the reference's 200 dpi (panels resampled, axes / labels / colour bars drawn) on tmpfs; everything inside the clock"
                        + ("; ONE directory shared by all ranks (strong scaling), phases are rank 0's" if world > 1 else "")}
        if with_reference and world == 1:
            from oracle import ref_driver as RD

            if RD.available():
                r = RD.run_directory(work, workers=os.cpu_count() or 1, render="display")
                line["reference_same_directory"] = {"seconds": r["seconds"], "orbits_per_s": n / r["seconds"], "pngs": r["pngs"],
                                                    "png_mb": r["png_bytes"] / 1e6, "cores": r["workers"], "kind": "reference"}
        return line
    finally:
        os.chdir(cwd)
        if world > 1:
            dist.barrier()
        if rank == 0:
            shutil.rmtree(work, ignore_errors=True)


DUMP_RGBA_PIXELS = 2_000_000  # 32 MB as float32 RGBA: with the other arrays well inside 64 MB


def dump_outputs(out_dir, state, batch):
    """What one step hands its caller, as float arrays under ``out_dir``, so that two builds can be compared
    output for output on the same seeded workload:

    ``extrema.npy``          float64, the ``*_y_min / _y_max / _z_min / _z_max`` entries of the global extrema
                             in sorted key order (None -> NaN)
    ``panel_vmin_vmax.npy``  float64 (panels, 2), every panel's resolved norm bounds, by panel id
    ``rgba_sample.npy``      float32 (pixels, 4), the RGBA rasters at a fixed, seeded sample of
                             ``DUMP_RGBA_PIXELS`` pixel positions (all of them when there are fewer)"""
    os.makedirs(out_dir, exist_ok=True)
    keys = sorted(k for k in state if k.endswith(("_y_min", "_y_max", "_z_min", "_z_max")))
    extrema = np.array([np.nan if state[k] is None else float(state[k]) for k in keys], dtype=np.float64)
    norms = batch.norms()
    bounds = np.stack([norms["vmin"], norms["vmax"]], axis=1).astype(np.float64)
    rgba = batch.all_rgba().reshape(-1, 4)
    if len(rgba) > DUMP_RGBA_PIXELS:
        rgba = rgba[np.sort(np.random.default_rng(0).choice(len(rgba), DUMP_RGBA_PIXELS, replace=False))]
    for name, arr in (("extrema", extrema), ("panel_vmin_vmax", bounds), ("rgba_sample", rgba.astype(np.float32))):
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def bind_near_gpu(torch, local):
    """Multi-rank runs: keep this process (and so the first-touch placement of its pinned staging
    buffers) on the CPUs of the GPU's NUMA node, so every rank's H2D traffic stays on its own socket."""
    try:
        props = torch.cuda.get_device_properties(local)
        bdf = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        cpus = set()
        for part in open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip().split(","):
            if not part:
                continue
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except (OSError, AttributeError, ValueError):
        pass
    return None


# ----------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
        return
    import torch

    from configurable_spectrograms_b200 import _lib
    from configurable_spectrograms_b200.fast.extrema import extrema_enqueue, extrema_finish
    from configurable_spectrograms_b200.fast.pipeline import BatchStep, ShardPlan

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    comm = None
    numa_cpus = bind_near_gpu(torch, local) if world > 1 else None
    if world > 1:
        import torch.distributed as dist

        from configurable_spectrograms_b200.comm import TorchComm

        dist.init_process_group("nccl", device_id=dev)
        comm = TorchComm(dist, dev)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # nvidia-smi needs ~1 s before its first row: start it ahead of the GPU work
    strong = args.total_orbits > 0
    if strong and args.total_orbits % world:
        raise SystemExit(f"--total-orbits {args.total_orbits} does not divide over {world} GPUs")
    n_local = args.total_orbits // world if strong else args.orbits_per_gpu
    first = rank * n_local
    files, orbits, total_elems = orbit_layout(n_local, first, args.seed)
    cubes = generate_cubes(torch, files, total_elems, dev)
    torch.cuda.synchronize()
    # one explicit stream for everything: libcsgpu kernels, torch events and the NCCL exchanges
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    ctx = _lib.Context(local, stream=tstream.cuda_stream)
    lut = turbo_like_lut()

    # global ascending orbit sequence (every rank knows every orbit number; files all present)
    sequence = [(13000 + g, {i: True for i in ORDER}) for g in range(world * n_local)]

    def build_shard(base_ptr):
        shard = ShardPlan(ctx, "linear", "log", zoom_duration_minutes=6, instrument_order=ORDER)
        shard.first_orbit_index = first
        for ob in orbits:
            dsets = {}
            for inst, fd in ob["files"].items():
                f = files[fd["index"]]
                dsets[inst] = {"times": fd["times"], "energy": fd["energy"], "pitch_angle": fd["pitch_angle"],
                               "shape": (f["T"], P, E), "device_ptr": base_ptr + 4 * f["offset"]}
            shard.add_orbit(ob["orbit"], dsets, ob["lines"])
        return shard

    # ------------------------------------------------------------ device-resident arm
    shard = build_shard(cubes.data_ptr())
    step = BatchStep(shard, sequence, max_percentile=99.0, comm=comm, lut259=lut, want_index=False)
    t_plan = time.perf_counter()
    state0 = step.run({})  # plans the panels on the first pass
    step.finish()
    t_plan = time.perf_counter() - t_plan
    sampler.mark(0)
    for _ in range(args.warmup):
        step.run({})
    step.finish()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = ctx.launch_count()
    if args.profile_region == "steps":
        torch.cuda.profiler.start()  # cudaProfilerStart: `ncu --profile-from-start off` sees the timed steps only
    host_t0 = time.perf_counter()
    prof = None
    if args.profile_host:
        import cProfile

        prof = cProfile.Profile()
        prof.enable()
    ev0.record(tstream)
    for _ in range(args.steps):
        state = step.run({})
    ev1.record(tstream)
    if args.profile_region == "steps":
        torch.cuda.profiler.stop()
    if prof is not None:
        prof.disable()
        import io
        import pstats

        buf = io.StringIO()
        pstats.Stats(prof, stream=buf).sort_stats("cumulative").print_stats(45)
        open(f"{args.profile_host}.rank{rank}", "w").write(buf.getvalue())
    host_enqueue_ms = (time.perf_counter() - host_t0) * 1e3 / args.steps
    step.finish()
    barrier()
    if args.dump_outputs and rank == 0:  # before the per-stage passes below rewrite the rasters
        dump_outputs(args.dump_outputs, state, shard.batch)

    def exchange_of(sh):
        sel = getattr(sh, "_pool_selector_side", None) or getattr(sh, "_pool_selector", None)
        return getattr(sel, "_exchange", None) if sel is not None else None

    # the last two timed steps' exchanges as rank 0's GPU saw them (6 per step): [start, published, peers seen] in us
    trace_in_step = None
    if world > 1 and getattr(exchange_of(shard), "kind", "") == "peer":
        trace_in_step = exchange_of(shard).trace(12)
    launches = ctx.launch_count() - launches0
    ms_total = ev0.elapsed_time(ev1)
    assert state == state0, "extrema changed between steps"
    # per-kernel stage times: separate passes, CUDA events on the launching stream, `reps`
    # back-to-back launches per event pair so the launch latency is not billed to the kernel
    # (every stage streams far more than the 126 MB L2, so repeats do not hit cache)
    def timed(fn, n=3, reps=5):
        out = []
        for _ in range(n):
            ctx.timer_start(0)
            for _ in range(reps):
                fn()
            ctx.timer_stop(0)
            out.append(ctx.timer_ms(0) / reps)
        return float(np.mean(out))

    k1_ms = timed(shard.collapse)
    stats_ms = timed(shard.batch.run_stats)
    prep_ms = timed(shard.batch.prepare)
    raster_ms = timed(lambda: shard.batch.rasterise(want_rgba=True, want_index=False))

    pool = []
    for _ in range(5):  # device time of the K2b launches alone (host bookkeeping excluded)
        ctx.timer_start(0)
        pending = extrema_enqueue(shard, sequence, ORDER, "linear", "log", {}, max_percentile=99.0, comm=comm, per_step=False)
        ctx.timer_stop(0)
        extrema_finish(pending)
        pool.append(ctx.timer_ms(0))
    pool_ms = float(np.mean(pool))
    trace_alone = None
    if world > 1:
        sel_main = getattr(shard, "_pool_selector", None)
        ex_main = getattr(sel_main, "_exchange", None) if sel_main is not None else None
        if getattr(ex_main, "kind", "") == "peer":
            trace_alone = ex_main.trace(12)
    sampler.mark(1)
    clocks = sampler.stop() if rank == 0 else None

    # ------------------------------------------------- parity of this very workload (outside the metric)
    parity = None
    if not args.no_verify:
        parity = verify_shard(args, torch, cubes, files, orbits, shard, step, state, lut, rank, world)

    # ------------------------------------------------- K4 (outside the metric): figures -> PNG bytes
    png_stage = None
    if rank == 0 and not args.no_png:
        from configurable_spectrograms_b200 import png as PNG
        from configurable_spectrograms_b200.fast.plotting import figure_from_spec

        # (no collective here: the rasters of the last pass are still in HBM, the figures' zoom flags
        # were resolved by step.finish() above)
        norms = shard.batch.norms()
        n_fig_orbits = min(args.png_orbits, n_local)
        specs = [sp for ob in orbits[:n_fig_orbits] for wx in (False, True)
                 for sp in shard.figures[slice(*step.figure_ranges[(ob["orbit"], wx)])]]
        figs = [f for f in (figure_from_spec(shard, sp, "turbo", norms=norms, device_rasters=True)[0] for sp in specs) if f is not None]
        PNG.encode_figures_device(ctx, shard.batch.d_rgba.ptr, figs, dpi=200)  # warm-up: tables, sprites, device and pinned scratch
        phases: dict = {}
        if args.profile_region == "png":
            torch.cuda.profiler.start()
        t0 = time.perf_counter()
        blobs = PNG.encode_figures_device(ctx, shard.batch.d_rgba.ptr, figs, dpi=200, timings=phases)
        dev_s = time.perf_counter() - t0
        if args.profile_region == "png":
            torch.cuda.profiler.stop()

        def raw_size(f):  # filtered bytes of the figure at 200 dpi
            W, H = int(round(f.figsize[0] * 200)), int(round(f.figsize[1] * 200))
            return 4 * H * W + H

        raw_bytes = sum(raw_size(f) for f in figs)
        # the host encoder on the same mosaic (zlib level 6, one thread), a few figures
        sample = figs[:: max(1, len(figs) // 6)][:6]
        host_s, host_bytes = 0.0, 0
        for f, blob in zip(sample, [blobs[figs.index(f)] for f in sample]):
            img = PNG.decode_rgba(blob)
            t0 = time.perf_counter()
            host_bytes += len(PNG.encode_rgba(img))
            host_s += time.perf_counter() - t0
        png_stage = {"figures": len(figs), "raw_gb": raw_bytes / 1e9, "device_s": dev_s, "device_figures_per_s": len(figs) / dev_s,
                     "device_raw_gb_per_s": raw_bytes / 1e9 / dev_s, "device_ratio": raw_bytes / max(1, sum(len(b) for b in blobs)),
                     "phases_s": phases, "host_zlib6_s_per_figure_1thread": host_s / max(1, len(sample)),
                     "host_zlib6_ratio": sum(raw_size(f) for f in sample) / max(1, host_bytes),
                     "note": "figures at the reference's 200 dpi (4800 x 2400 for the two-column grids): resample + annotations composed "
                             "and DEFLATE-encoded on the GPU, D2H of the compressed bytes and PNG framing included; not part of `value`"}
    # the carrier of the extrema exchange and what its all-gathers waited for (rank skew + link latency)
    exchange, exchange_info = None, {"exchange": "none (1 rank)"}
    if world > 1:
        sel = getattr(shard, "_pool_selector_side", None) or getattr(shard, "_pool_selector", None)
        exchange = getattr(sel, "_exchange", None) if sel is not None else None
        kind = getattr(exchange, "kind", "unknown")
        exchange_info = {"exchange": "peer mailboxes over NVLink (csrc/peer.cu)" if kind == "peer" else "NCCL all_gather_into_tensor",
                         "exchanges_per_step": 6, "rendezvous": "torch.distributed NCCL (barriers, timing all-reduce only)"}
        if kind == "peer":
            exchange_info["wait_us"] = exchange.wait_stats(60)
            exchange_info["trace_us_last_two_timed_steps"] = trace_in_step
            exchange_info["trace_us_k2b_alone"] = trace_alone
    t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    total_orbits = world * n_local
    value = total_orbits / (ms_step / 1e3)

    cube_bytes = 4 * total_elems
    sums_bytes = sum(5 * f["T"] * E * 4 for f in files)  # algorithmic: (G+1)*T*E*s per file
    fallbacks = shard.batch.stats_fallbacks()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = (cube_bytes + sums_bytes) / (k1_ms / 1e3) / 1e9
    # DRAM bytes of one K1 launch from the committed `ncu --set full` capture of this same workload
    # (profiles/r2_k1_traffic.json -- the round-1 capture as a fallback -- written by scripts/ncu_summary.py --traffic)
    traffic = None
    for name in ("r2_k1_traffic.json", "r1_k1_traffic.json"):
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", name)))
            if tr.get("orbits_per_gpu") == n_local and tr.get("algorithmic_bytes") == int(cube_bytes + sums_bytes):
                traffic = int(tr["dram_bytes_read"] + tr["dram_bytes_write"])
                break
        except (OSError, ValueError, KeyError):
            pass
    # the whole step against the same roofline: SURVEY.md section 8(d)'s B_orbit, i.e. cube read +
    # (G+1) sums written + one pass over the total for the pooled extrema + per panel pixel
    # (stats read + raster read + RGBA write)
    s_el = 4
    step_bytes = cube_bytes + sums_bytes + sum(f["T"] * E * s_el for f in files) + shard.batch.n_pixels * (2 * s_el + 4)
    step_gbs = step_bytes / ((float(ms_total) / args.steps) / 1e3) / 1e9

    # ------------------------------------------------------------------- e2e arm
    e2e = None
    if not args.no_e2e:
        host = torch.empty(total_elems, dtype=torch.float32, pin_memory=True)
        host.copy_(cubes)
        torch.cuda.synchronize()
        n_px = shard.batch.n_pixels
        rgba_host = torch.empty(n_px, dtype=torch.int32, pin_memory=True)
        rgba_view = None

        def e2e_step():
            # H2D of this step's inputs (pinned -> HBM) on the context stream, then the step; the
            # rasters leave on the copy-out stream, so step k's read-back shares the (full duplex)
            # link with step k+1's upload.  side_join: the next K3 must not overwrite rasters that
            # are still being copied (enqueued after the upload, so the upload itself never waits).
            ctx._check(ctx.lib.csg_h2d(ctx.handle, cubes.data_ptr(), host.data_ptr(), cube_bytes))
            ctx.side_join()
            step.run({})
            ctx.d2h_side(rgba_host.data_ptr(), shard.batch.d_rgba.ptr, n_px * 4)
            step.finish()

        def e2e_drain():
            ctx.side_sync()

        e2e_step()
        e2e_drain()
        # stand-alone ceilings of the two copies the e2e step makes: the same pinned buffers, no kernels, every
        # rank at once (the ranks share the host's memory and PCIe fabric) -- e2e is bounded by max(H2D, D2H) of these
        def copy_rate(fn, nbytes, reps=3):
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            ctx.sync()
            ctx.side_sync()
            barrier()
            dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                torch.distributed.all_reduce(dt, op=torch.distributed.ReduceOp.MAX)
            return world * nbytes * reps / float(dt.item()) / 1e9

        h2d_gbs = copy_rate(lambda: ctx._check(ctx.lib.csg_h2d(ctx.handle, cubes.data_ptr(), host.data_ptr(), cube_bytes)), cube_bytes)
        d2h_gbs = copy_rate(lambda: ctx.d2h_side(rgba_host.data_ptr(), shard.batch.d_rgba.ptr, n_px * 4), n_px * 4)
        barrier()
        t0 = time.perf_counter()
        n_e2e = max(2, min(args.steps, 4))
        for _ in range(n_e2e):
            e2e_step()
        e2e_drain()  # the last step's rasters are in host memory before the clock stops
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(dt, op=torch.distributed.ReduceOp.MAX)
        e2e_value = total_orbits / (float(dt.item()) / n_e2e)
        ceiling = world * n_local / (cube_bytes / (h2d_gbs / world * 1e9))  # orbits/s if nothing but the upload took time
        e2e = {"value": e2e_value, "unit": "orbits/s",
               "h2d_bytes_per_step": int(cube_bytes), "d2h_bytes_per_step": int(n_px * 4), "steps": n_e2e,
               "h2d_ceiling_gbs": h2d_gbs, "d2h_ceiling_gbs": d2h_gbs, "h2d_achieved_gbs": e2e_value / total_orbits * world * cube_bytes / 1e9,
               "frac_of_h2d_ceiling": e2e_value / ceiling,
               "note": "ceilings: aggregate over all ranks of the same pinned copies alone (no kernels), all ranks copying at once"}

    # ------------------------------------------------ api_e2e: the public call, directory -> PNG files
    api = None
    if not args.no_api_e2e:  # (every rank takes part: the directory driver shards the orbits itself)
        api = api_e2e_leg(args, cubes, files, orbits, state, args.api_ref, torch.distributed if world > 1 else None, rank, world)

    # ----------------------------------------------------------- CPU baseline beside it
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import ref_driver as RD

        n = args.cpu_sample_orbits
        if RD.available():
            sec, cores, pngs, png_bytes = run_reference_directory(n, args.seed, 1, 0)
            cpu = {"value": n / sec, "unit": "orbits/s", "cores": cores, "kind": "reference", "sample_orbits": n,
                   "sample": f"{n} synthetic FAST orbits of the same workload through the unmodified reference's FAST_plot_spectrograms_directory "
                             f"(oracle/_ref under the cdflib/matplotlib stand-ins, fork pool on {cores} cores, {pngs} PNGs at figsize x dpi without text), {sec:.1f} s wall"}
        else:
            sec, cores = run_cpu_port(cpu_sample_orbits(n, args.seed), 1, 0)
            cpu = {"value": n / sec, "unit": "orbits/s", "cores": cores, "kind": "port", "sample_orbits": n,
                   "sample": f"{n} synthetic FAST orbits of the same workload, both submissions, numeric path only (no Agg/PNG), {sec:.1f} s wall"}

    if rank == 0:
        read_peak = measured_read_stream_peak()
        line = {
            "metric": METRIC, "value": value, "unit": "orbits/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(n_local, world),
            "collective": exchange_info,
            "plan": {"panels_per_gpu": shard.batch.n_panels, "regions_per_gpu": shard.batch.n_regions,
                     "pixels_per_gpu": shard.batch.n_pixels, "numa_bound_cpus": numa_cpus},
            "roofline": {"bound": "hbm", "kernel": "collapse_stream_kernel<float,4,384>", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "ms": k1_ms,
                         "algorithmic_bytes": int(cube_bytes + sums_bytes),
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
                         # the peak above is a COPY (read + write bytes); K1 is 93 % reads, and a pure-read stream with
                         # K1's addressing reaches more (scripts/read_bw.cu; the committed measurement is read from profiles/r1_read_bw.txt)
                         "read_stream_peak": read_peak, "frac_of_read_stream_peak": achieved / read_peak if read_peak else None},
            "step_roofline": {"algorithmic_bytes": int(step_bytes), "achieved": step_gbs, "peak": peak, "unit": "GB/s",
                              "frac": step_gbs / peak, "note": "this rank's whole step (K1+K2b+K2a+K3), SURVEY 8(d) B_orbit x orbits / step time"},
            "parity_checked": parity, "png_stage": png_stage, "e2e": e2e, "api_e2e": api, "gpu_launches": int(launches), "clocks": clocks, "cpu_baseline": cpu,
            "stage_ms": {"collapse": k1_ms, "pool_extrema": pool_ms, "region_stats": stats_ms, "panel_prepare": prep_ms,
                         "rasterise": raster_ms, "host_enqueue_per_step": host_enqueue_ms, "first_step_with_planning": t_plan * 1e3,
                         "percentile_regions_needing_radix_fallback": fallbacks},
        }
        emit(line)
    if world > 1:
        if exchange is not None and hasattr(exchange, "close"):
            exchange.close()  # collective: unmap the peers' mailboxes, barrier, free the own one
        torch.distributed.destroy_process_group()


_JSON_FD = None  # the real stdout while everything else is diverted to stderr (see the bottom of the file)


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, on the real stdout."""
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    fd = 1 if _JSON_FD is None else _JSON_FD
    while data:
        data = data[os.write(fd, data):]


if __name__ == "__main__":
    # stdout carries the JSON line and nothing else: what this process, its worker processes (the reference's
    # fork pool logs to stdout) or a library print meanwhile goes to stderr
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    main()
