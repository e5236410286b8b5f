"""Global per-instrument axis extrema (reference ``fast/extrema.py``).

Same call signature, JSON cache schema and control flow as the reference's
``compute_global_extrema`` -- including its quirks, which are results: the
linear/linear combo re-uses its own keys from the second orbit on (``:208-243``), the
``complete`` flag compares an orbit index with a file count (``:315-319``), log-scale
combos only transform cached linear/linear values (``:201-220``).

The arithmetic is different: the reference re-concatenates every positive sample seen so
far and calls ``np.nanpercentile`` after each (orbit, instrument) step (quadratic); here
all files are collapsed once on the GPU (K1) and the running maximum over every prefix
pool is selected exactly from scanned radix histograms (K2b, ``pool_select.py``).
"""

from __future__ import annotations

import copy
import json
import math
import os
from collections.abc import Iterable
from typing import Any

import numpy as np

from ..logging_utils import log_exception
from ..percentile_utils import round_extrema
from .constants import FAST_EXTREMA_JSON_PATH


def _extrema_overrides(global_extrema, inst, y_scale, z_scale):
    """Rounded ``(y_min, y_max, z_min, z_max)`` for one instrument (``:26-70``).

    >>> extrema = {"ees_linear_linear_y_max": 1234, "ees_linear_linear_z_min": 0.0123}
    >>> _extrema_overrides(extrema, "ees", "linear", "linear")
    (None, 1300.0, 0.012, None)
    >>> _extrema_overrides(None, "ees", "linear", "linear")
    (None, None, None, None)
    """
    if not isinstance(global_extrema, dict):
        return None, None, None, None
    stem = f"{inst}_{y_scale}_{z_scale}"
    out = []
    for axis, how in (("y_min", "down"), ("y_max", "up"), ("z_min", "down"), ("z_max", "up")):
        value = global_extrema.get(f"{stem}_{axis}")
        out.append(None if value is None else round_extrema(value, how))
    return tuple(out)


def _walk(sequence, instrument_order, y_scale, z_scale, state, totals, log_floor_cutoff, log_floor_value,
          on_scan, on_step_done=None):
    """The reference's orbit x instrument loop (``:183-331``) with the scan abstracted.

    ``sequence``: [(orbit, {inst: handle})] ascending.  ``on_scan(inst, orbit_index, handle)``
    is called where the reference loads a file and updates its pools, and must return
    ``(candidate_energy_max, candidate_intensity_max, intensity_min_store)``.
    """

    def safe_log(value):  # :151-161
        if value is None:
            return float(log_floor_value)
        try:
            value = float(value)
        except (TypeError, ValueError):
            return float(log_floor_value)
        if not np.isfinite(value) or value <= log_floor_cutoff:
            return float(log_floor_value)
        return float(np.log10(value))

    orbit_numbers = [o for o, _ in sequence]
    last_key = f"{y_scale}_{z_scale}_last_orbit"
    stored = state.get(last_key, -1)
    last_done = int(stored) if isinstance(stored, (int, float)) else -1
    y_log, z_log = y_scale == "log", z_scale == "log"
    if on_step_done is None and _walk_chains(sequence, instrument_order, y_scale, z_scale, state, totals, last_done, on_scan):
        return state
    # key strings of every instrument, built once (the loop below runs orbits x instruments times)
    keys = []
    for inst in instrument_order:
        stem, ll = f"{inst}_{y_scale}_{z_scale}", f"{inst}_linear_linear"
        keys.append((inst, f"{stem}_extrema_progress", f"{ll}_y_max", f"{ll}_z_max", f"{ll}_y_min", f"{ll}_z_min",
                     f"{stem}_y_max", f"{stem}_y_min", f"{stem}_z_max", f"{stem}_z_min"))
    other_last = [f"{other}_{y_scale}_{z_scale}_last_orbit" for other in instrument_order]
    max_orbit = max(orbit_numbers) if orbit_numbers else -1
    for orbit_index, (orbit, handles) in enumerate(sequence):
        if orbit <= last_done:
            continue
        for inst, progress_key, ll_y, ll_z, ll_ymin, ll_zmin, k_ymax, k_ymin, k_zmax, k_zmin in keys:
            entry = state.get(progress_key)
            if isinstance(entry, dict) and entry.get("complete"):
                continue
            have_y, have_z = ll_y in state, ll_z in state
            if have_y:
                state[k_ymax] = safe_log(state[ll_y]) if y_log else state[ll_y]
                state[k_ymin] = log_floor_value if y_log else state.get(ll_ymin, 0)
            if have_z:
                state[k_zmax] = safe_log(state[ll_z]) if z_log else state[ll_z]
                state[k_zmin] = log_floor_value if z_log else state.get(ll_zmin, 0)
            if have_y and have_z:
                state[progress_key] = {"processed_index": max(totals[inst] - 1, -1), "total": totals[inst], "complete": True}
                for other in other_last:
                    state.pop(other, None)
                state[last_key] = max_orbit
                if on_step_done:
                    on_step_done(reuse=True)
                continue
            cand_e, cand_z, z_min_store = on_scan(inst, orbit_index, handles.get(inst))
            prev_e, prev_z = state.get(k_ymax), state.get(k_zmax)
            merged_e = max(float(prev_e), cand_e) if isinstance(prev_e, (int, float)) else cand_e
            merged_z = max(float(prev_z), cand_z) if isinstance(prev_z, (int, float)) else cand_z
            state[k_ymin] = 0
            state[k_ymax] = int(min(4000, math.ceil(merged_e)))
            state[k_zmin] = z_min_store
            state[k_zmax] = float(math.ceil(merged_z))
            state[progress_key] = {
                "processed_index": orbit_index,
                "total": totals[inst],
                "complete": orbit_index + 1 >= totals[inst],
            }
            for other in other_last:
                state.pop(other, None)
            state[last_key] = orbit
            if on_step_done:
                on_step_done(reuse=False)
    return state


def chain_ranges(sequence, instrument_order, y_scale, z_scale, state, totals, last_done=None):
    """``(first, {inst: stop})`` -- the orbit-index range every instrument's chain of scan steps
    covers -- when the walk is nothing but independent max-merge chains (see
    :func:`_walk_chains`); ``None`` when some step re-uses, skips or completes differently."""
    if last_done is None:
        stored = state.get(f"{y_scale}_{z_scale}_last_orbit", -1)
        last_done = int(stored) if isinstance(stored, (int, float)) else -1
    if not sequence or not instrument_order or (y_scale == "linear" and z_scale == "linear"):
        return None
    for inst in instrument_order:
        entry = state.get(f"{inst}_{y_scale}_{z_scale}_extrema_progress")
        if isinstance(entry, dict) and entry.get("complete"):
            return None
        if f"{inst}_linear_linear_y_max" in state or f"{inst}_linear_linear_z_max" in state:
            return None
    first = next((k for k, (orbit, _h) in enumerate(sequence) if orbit > last_done), None)
    if first is None:
        return None
    last_index = len(sequence) - 1
    # every later orbit must pass the `orbit <= last_done` gate too (ascending sequences always do)
    if any(orbit <= last_done for orbit, _h in sequence[first:]):
        return None
    # the per-step loop runs first..stop: it breaks after the step that makes the instrument
    # "complete" (orbit_index + 1 >= total, :315-319), and always runs one step
    return first, {inst: min(last_index, max(first, totals[inst] - 1)) for inst in instrument_order}


def _walk_chains(sequence, instrument_order, y_scale, z_scale, state, totals, last_done, on_scan) -> bool:
    """The loop of :func:`_walk` when every (orbit, instrument) step is a plain scan step: nothing
    is re-used from the linear/linear keys, nothing is complete, nobody watches the intermediate
    states.  Then the instruments are independent max-merge chains and only their last writes
    survive, so each chain runs on local variables and ``state`` is written once -- the same
    arithmetic in the same order per instrument, without ~25 dict operations per step.
    Returns False (state untouched) when the preconditions do not hold."""
    ranges = chain_ranges(sequence, instrument_order, y_scale, z_scale, state, totals, last_done)
    if ranges is None:
        return False
    first, stops = ranges
    results = {}
    last_executed = first
    range_max = getattr(on_scan, "range_max", None)
    for inst in instrument_order:
        stem = f"{inst}_{y_scale}_{z_scale}"
        prev_e, prev_z = state.get(f"{stem}_y_max"), state.get(f"{stem}_z_max")
        # the per-step loop below runs first..stop: it breaks after the step that makes the
        # instrument "complete" (orbit_index + 1 >= total, :315-319), and always runs one step
        stop = stops[inst]
        folded = range_max(inst, first, stop) if range_max is not None else None
        if folded is not None:
            # ceil and min(4000, .) are monotone, so folding the max-merge over the steps equals
            # one merge with the largest candidate: min(4000, ceil(max(prev, c_first..c_stop)))
            cand_e, cand_z, z_min_store = folded
            merged_e = max(float(prev_e), cand_e) if isinstance(prev_e, (int, float)) else cand_e
            merged_z = max(float(prev_z), cand_z) if isinstance(prev_z, (int, float)) else cand_z
            prev_e = int(min(4000, math.ceil(merged_e)))
            prev_z = float(math.ceil(merged_z))
        else:
            z_min_store = 0
            for orbit_index in range(first, stop + 1):
                cand_e, cand_z, z_min_store = on_scan(inst, orbit_index, sequence[orbit_index][1].get(inst))
                merged_e = max(float(prev_e), cand_e) if isinstance(prev_e, (int, float)) else cand_e
                merged_z = max(float(prev_z), cand_z) if isinstance(prev_z, (int, float)) else cand_z
                prev_e = int(min(4000, math.ceil(merged_e)))
                prev_z = float(math.ceil(merged_z))
        results[inst] = (stem, prev_e, prev_z, z_min_store, stop)
        last_executed = max(last_executed, stop)
    # the writes of the last step of every chain
    for inst in instrument_order:
        stem, y_max, z_max, z_min_store, stop = results[inst]
        state[f"{stem}_y_min"] = 0
        state[f"{stem}_y_max"] = y_max
        state[f"{stem}_z_min"] = z_min_store
        state[f"{stem}_z_max"] = z_max
        state[f"{stem}_extrema_progress"] = {
            "processed_index": stop,
            "total": totals[inst],
            "complete": stop + 1 >= totals[inst],
        }
        state.pop(f"{inst}_{y_scale}_{z_scale}_last_orbit", None)
    state.pop(f"{y_scale}_{z_scale}_last_orbit", None)
    state[f"{y_scale}_{z_scale}_last_orbit"] = sequence[last_executed][0]
    return True


def plan_scanned_steps(sequence, instrument_order, y_scale, z_scale, state, log_floor_cutoff=0.1, log_floor_value=-1.0):
    """Dry run: which (instrument -> [orbit_index]) steps reach the scan with this cache state."""
    steps: dict[str, list[int]] = {i: [] for i in instrument_order}
    totals = {i: sum(1 for _, h in sequence if i in h) for i in instrument_order}

    def record(inst, orbit_index, handle):
        steps[inst].append(orbit_index)
        return 0.0, 0.0, 0

    _walk(sequence, instrument_order, y_scale, z_scale, copy.deepcopy(state), totals, log_floor_cutoff,
          log_floor_value, record)
    return steps, totals


def energy_candidates(energies: list[np.ndarray], counts, as_array: bool = False, shared_table=None):
    """Per-step 99 %-coverage energy (``:270-278``) from per-file per-energy positive counts.

    ``energies[k]`` / ``counts[k]`` belong to the k-th scanned file of one instrument.  The
    reference keeps a dict keyed by ``float(energy_value)`` holding only energies that have
    seen a positive count; zero-count keys do not move the cumulative sum, so searching the
    union of all keys finds the same energy.
    """
    n = len(energies)
    if n == 0:
        return np.zeros(0) if as_array else []
    shared = shared_table is not None or all(e is energies[0] for e in energies)
    if shared:  # the usual case: every file of the instrument carries the same energy table
        e0, keys, idx = shared_table if shared_table is not None else shared_energy_table(energies[0])
        c = np.asarray(counts, dtype=np.int64)[:, : len(e0)]
        if len(keys) == len(e0):
            per_file = np.empty((n, len(keys)), dtype=np.int64)
            per_file[:, idx] = c
        else:
            per_file = np.zeros((len(keys), n), dtype=np.int64)
            np.add.at(per_file, idx, c.T)
            per_file = per_file.T
    else:
        keys = np.unique(np.concatenate([np.asarray(e, dtype=np.float64) for e in energies]))
        per_file = np.zeros((n, len(keys)), dtype=np.int64)
        for k, (e, c) in enumerate(zip(energies, counts)):
            e = np.asarray(e, dtype=np.float64)
            np.add.at(per_file[k], np.searchsorted(keys, e), np.asarray(c[: len(e)], dtype=np.int64))
    running = np.cumsum(per_file, axis=0)  # counts per key after each step
    along = np.cumsum(running, axis=1)
    total = along[:, -1]
    target = 0.99 * total
    first = (along > target[:, None]).argmax(axis=1)
    out = np.where(total > 0, keys[first], 0.0)
    return out if as_array else out.tolist()


def shared_energy_table(energy):
    """(float64 energies, sorted unique keys, inverse index): the static part of :func:`energy_candidates`."""
    e0 = np.asarray(energy, dtype=np.float64)
    keys, idx = np.unique(e0, return_inverse=True)
    return e0, keys, idx


def _energy_plan(shard, comm, instrument_order, steps, owners, first):
    """Who holds the per-energy counts of every scanned step (static per plan; exchanged once)."""
    local = [(inst, oi + first, shard.file_meta[file]["energy"]) for inst, oi, file in owners]
    parts = comm.allgather_object(local) if comm.size > 1 else [local]
    n_max = max((len(p) for p in parts), default=0)
    max_E = max((len(e) for p in parts for _, _, e in p), default=1)  # same on every rank: shapes of the exchange
    where, energies = {}, {}
    for rk, part in enumerate(parts):
        for row, (inst, oi, energy) in enumerate(part):
            where[(inst, oi)] = rk * n_max + row
            energies[(inst, oi)] = energy
    plan = {}
    for inst in instrument_order:
        present = [oi for oi in steps[inst] if (inst, oi) in where]
        en = [energies[(inst, oi)] for oi in present]
        # after a pickle round trip equal tables are distinct objects: fold them back together
        uniq: list[np.ndarray] = []
        for k, e in enumerate(en):
            for u in uniq:
                if u is e or (u.shape == np.shape(e) and np.array_equal(u, e, equal_nan=True)):
                    en[k] = u
                    break
            else:
                uniq.append(e)
        # static index maps of the per-step candidate fill (extrema_finish): position of every
        # present step inside steps[inst]
        steps_arr = np.asarray(steps[inst], dtype=np.int64)
        pos = np.searchsorted(steps_arr, np.asarray(present, dtype=np.int64)) if present else np.zeros(0, np.int64)
        ascending = bool(np.all(np.diff(steps_arr) > 0)) if len(steps_arr) > 1 else True
        table = shared_energy_table(en[0]) if en and all(e is en[0] for e in en) else None
        plan[inst] = (present, np.asarray([where[(inst, oi)] for oi in present], dtype=np.int64), en, steps_arr, pos, ascending, table)
    return plan, n_max, max_E


def _device_y_tables(instrument_order, eplan, max_E):
    """Static energy tables for ``csg_pool_energy_candidates`` -- or None when some instrument's
    files do not share one table of distinct, NaN-free energies (the host path handles those)."""
    n_inst = len(instrument_order)
    order = np.zeros((n_inst, max_E), dtype=np.int32)
    keys = np.zeros((n_inst, max_E), dtype=np.float64)
    n_keys = np.zeros(n_inst, dtype=np.int32)
    covered = {}
    for ii, inst in enumerate(instrument_order):
        present, _rows, _en, steps_arr, pos, ascending, table = eplan[inst]
        if not ascending:
            return None
        cov = np.zeros(int(steps_arr.max()) + 1 if len(steps_arr) else 0, dtype=bool)
        if present:
            if table is None:
                return None
            e0, uniq, _idx = table
            if len(uniq) != len(e0) or len(e0) > max_E or np.isnan(e0).any():
                return None
            o = np.argsort(e0, kind="stable")
            order[ii, : len(e0)], keys[ii, : len(e0)], n_keys[ii] = o, e0[o], len(e0)
            idx = np.full(len(steps_arr), -1, dtype=np.int64)
            idx[pos] = 1
            cov[steps_arr] = np.maximum.accumulate(idx) >= 0
        covered[inst] = cov
    return {"order": order, "keys": keys, "n_keys": n_keys, "covered": covered}


def extrema_enqueue(shard, sequence, instrument_order, y_scale, z_scale, state, *, compute_mins=False,
                    max_percentile=95.0, log_floor_cutoff=0.1, log_floor_value=-1.0, comm=None, per_step=True,
                    overlap=False):
    """Enqueue the pooled-extrema selection (K2b) for an already collapsed :class:`pipeline.ShardPlan`.

    Everything runs asynchronously on the context's stream (``pool_select.DevicePoolSelector``);
    the returned token is redeemed by :func:`extrema_finish`, so the caller can enqueue more GPU
    work (K2a) in between and hide the host bookkeeping behind it.

    ``sequence[k] = (orbit, {inst: True})`` must list the GLOBAL ascending orbit sequence
    (all ranks); ``shard.orbits`` holds this rank's contiguous slice starting at
    ``shard.first_orbit_index``.

    ``per_step=False`` promises that :func:`extrema_finish` will not be asked for the state after
    every step (no ``on_step_done``): when the walk then reduces to independent max-merge chains
    (:func:`chain_ranges`) the y candidates are max-merged on the device too and the per-file
    counts never travel to the host.

    ``overlap=True``: the selection runs on the batch context's side context (its own high-priority
    stream, ordered after everything enqueued on the batch context so far), so kernels the caller
    enqueues on the batch context afterwards (K2a, K3 of the panels that need no extrema) run
    concurrently with the digit loop and its cross-GPU exchanges.
    """
    from ..pool_select import DevicePoolSelector, SingleRank

    comm = comm or SingleRank()
    instrument_order = tuple(instrument_order)
    first = getattr(shard, "first_orbit_index", 0)
    # which steps reach the scan depends only on the orbit sequence and the cache state: plan once
    cache = shard.__dict__.setdefault("_extrema_plan_cache", {})
    key = (id(sequence), len(sequence), instrument_order, y_scale, z_scale, json.dumps(state, sort_keys=True, default=str),
           log_floor_cutoff, log_floor_value, first, len(shard.orbits))
    hit = cache.get(key)
    if hit is None:
        steps, totals = plan_scanned_steps(sequence, instrument_order, y_scale, z_scale, state, log_floor_cutoff,
                                           log_floor_value)
        local_steps = {
            inst: [oi - first for oi in steps[inst] if first <= oi < first + len(shard.orbits)]
            for inst in instrument_order
        }
        items, inst_len, owners = shard.pool_items(local_steps)
        eplan, n_max, max_E = _energy_plan(shard, comm, instrument_order, steps, owners, first)
        max_E = (max_E + 3) & ~3  # count rows pack to 16 bytes (exchange payloads)
        ranges = chain_ranges(sequence, instrument_order, y_scale, z_scale, state, totals)
        ytab = _device_y_tables(instrument_order, eplan, max_E) if ranges is not None else None
        if ytab is not None:
            first_step, stops = ranges
            # positions of this rank that take part in each chain (global orbit index <= stop)
            ytab["limit"] = np.array(
                [sum(1 for i2, oi, _f in owners if i2 == inst and oi + first <= stops[inst]) for inst in instrument_order],
                dtype=np.int32)
            ytab["zero"] = {}
            for inst in instrument_order:
                cov = ytab["covered"][inst]
                seg = np.zeros(stops[inst] + 1 - first_step, dtype=bool)
                part = cov[first_step : stops[inst] + 1]
                seg[: len(part)] = part
                ytab["zero"][inst] = not bool(seg.all())  # some step of the chain sees the 0.0 candidate
        if len(cache) > 8:
            cache.clear()
        # the entry holds `sequence` itself, so its id() cannot be recycled while the entry lives
        hit = cache[key] = (sequence, steps, totals, items, inst_len, owners, eplan, n_max, max_E, ytab)
    _, steps, totals, items, inst_len, owners, eplan, n_max, max_E, ytab = hit
    ydev = ytab if not per_step else None
    requests = [{"inst": ii, "p": max_percentile, "mode": "running_max"} for ii in range(len(instrument_order))]
    if compute_mins:
        requests += [{"inst": ii, "p": 1, "mode": "last"} for ii in range(len(instrument_order))]
    attr = "_pool_selector_side" if overlap else "_pool_selector"
    selector = getattr(shard, attr, None)
    if selector is None:  # persistent scratch across steps
        selector = DevicePoolSelector(shard.batch, ctx=shard.batch.ctx.side_context() if overlap else None)
        setattr(shard, attr, selector)
    if overlap:
        selector.ctx.wait_for(shard.batch.ctx)  # the collapsed sums (K1) are complete before the histograms read them
    selector.enqueue(shard.batch.dtype, items, len(instrument_order), inst_len, max_E, requests, comm=comm,
                     count_rows=n_max, ydev=ydev)
    return {
        "shard": shard, "sequence": sequence, "instrument_order": instrument_order, "y_scale": y_scale, "z_scale": z_scale,
        "state": state, "compute_mins": compute_mins, "log_floor_cutoff": log_floor_cutoff,
        "log_floor_value": log_floor_value, "comm": comm, "steps": steps, "totals": totals, "first": first,
        "items": items, "inst_len": inst_len, "owners": owners, "requests": requests, "max_E": max_E, "selector": selector,
        "eplan": eplan, "n_max": n_max, "ydev": ydev,
    }


def extrema_finish(pending, on_step_done=None):
    """Wait for the selection's read-backs and run the reference's bookkeeping walk on the results."""
    from ..pool_select import GpuPoolBackend, prefix_percentiles

    shard, comm = pending["shard"], pending["comm"]
    instrument_order, steps = pending["instrument_order"], pending["steps"]
    requests, compute_mins = pending["requests"], pending["compute_mins"]
    selector = pending["selector"]
    if pending.get("ydev") is not None:
        return _finish_device_y(pending, on_step_done)
    # ---- y extrema: per-step energy candidates from every rank's per-file positive counts
    # (available after the first histogram pass; this overlaps the digit loop on the GPU)
    all_counts, npos = selector.result_counts()  # multi-rank: every rank's rows (device all-gather)
    n_seq = len(pending["sequence"])
    cand_e: dict[str, np.ndarray] = {}  # per orbit index: the candidate the reference's step would see
    for inst in instrument_order:
        present, rows, energies, steps_arr, pos, ascending, table = pending["eplan"][inst]
        dense = np.zeros(n_seq, dtype=np.float64)
        if present and ascending:
            ce = energy_candidates(energies, all_counts[rows], as_array=True, shared_table=table)
            # steps without a file repeat the previous candidate (0.0 before the first file)
            idx = np.full(len(steps_arr), -1, dtype=np.int64)
            idx[pos] = np.arange(len(present))
            filled = np.maximum.accumulate(idx)
            dense[steps_arr] = np.where(filled >= 0, ce[np.maximum(filled, 0)], 0.0)
        elif present:
            by_step = dict(zip(present, energy_candidates(energies, all_counts[rows])))
            running = 0.0
            for oi in steps[inst]:
                running = by_step.get(oi, running)
                dense[oi] = running
        cand_e[inst] = dense
    # ---- z extrema: the device selection
    values = selector.result_values()
    if values is None:
        # more distinct candidate buckets survived than the device table holds: same kernels,
        # digit loop driven from the host (arbitrary candidate counts)
        backend = getattr(shard, "_pool_backend", None)
        if backend is None:
            backend = shard._pool_backend = GpuPoolBackend(shard.batch)
        values, _, _ = prefix_percentiles(
            backend, shard.batch.dtype, pending["items"], len(instrument_order), pending["inst_len"], pending["max_E"],
            requests, comm=comm,
        )
    n_inst = len(instrument_order)
    per_inst = {}
    for ii, inst in enumerate(instrument_order):
        z = values[ii]
        z_min = 0
        if compute_mins:
            zm = values[n_inst + ii]
            z_min = float(zm) if zm is not None else 0
        per_inst[inst] = (cand_e[inst], float(z) if z is not None else 0.0, z_min)

    def scan(inst, orbit_index, handle):
        ce, z, z_min = per_inst[inst]
        return float(ce[orbit_index]), z, z_min

    def range_max(inst, first, stop):
        """Largest candidates over the steps first..stop (None: NaN candidates, walk step by step)."""
        ce, z, z_min = per_inst[inst]
        top = float(ce[first : stop + 1].max())
        if top != top or z != z:
            return None
        return top, z, z_min

    scan.range_max = range_max
    return _walk(pending["sequence"], instrument_order, pending["y_scale"], pending["z_scale"], pending["state"],
                 pending["totals"], pending["log_floor_cutoff"], pending["log_floor_value"], scan, on_step_done)


def _finish_device_y(pending, on_step_done):
    """:func:`extrema_finish` when both extrema were max-merged on the device: one read-back of
    ``n_requests + n_instruments`` numbers, then one merge per instrument."""
    if on_step_done is not None:
        raise ValueError("extrema_enqueue(per_step=False) cannot report the state after every step")
    from ..pool_select import GpuPoolBackend, prefix_percentiles

    shard, comm = pending["shard"], pending["comm"]
    instrument_order, requests = pending["instrument_order"], pending["requests"]
    selector, ydev = pending["selector"], pending["ydev"]
    values = selector.result_values()
    ycands = selector.result_y_candidates()
    if values is None:  # slot-table overflow: same kernels, digit loop driven from the host
        backend = getattr(shard, "_pool_backend", None)
        if backend is None:
            backend = shard._pool_backend = GpuPoolBackend(shard.batch)
        values, _, _ = prefix_percentiles(
            backend, shard.batch.dtype, pending["items"], len(instrument_order), pending["inst_len"], pending["max_E"],
            requests, comm=comm,
        )
    n_inst = len(instrument_order)
    per_inst = {}
    for ii, inst in enumerate(instrument_order):
        z = values[ii]
        z_min = 0
        if pending["compute_mins"]:
            zm = values[n_inst + ii]
            z_min = float(zm) if zm is not None else 0
        top = ycands[ii]
        if top is None:
            top = 0.0  # no file took part: every step of the chain saw the empty-pool candidate
        elif ydev["zero"][inst]:
            top = max(top, 0.0)
        per_inst[inst] = (top, float(z) if z is not None else 0.0, z_min)

    def scan(inst, orbit_index, handle):
        raise AssertionError("per-step scan requested from a device-merged selection")

    scan.range_max = lambda inst, first, stop: per_inst[inst]
    state = pending["state"]
    totals = pending["totals"]
    stored = state.get(f"{pending['y_scale']}_{pending['z_scale']}_last_orbit", -1)
    last_done = int(stored) if isinstance(stored, (int, float)) else -1
    if not _walk_chains(pending["sequence"], instrument_order, pending["y_scale"], pending["z_scale"], state, totals,
                        last_done, scan):
        raise AssertionError("chain preconditions changed between enqueue and finish")
    return state


def extrema_from_shard(shard, sequence, instrument_order, y_scale, z_scale, state, *, compute_mins=False,
                       max_percentile=95.0, log_floor_cutoff=0.1, log_floor_value=-1.0, comm=None,
                       on_step_done=None):
    """Update ``state`` from an already collapsed :class:`pipeline.ShardPlan` (enqueue + finish)."""
    pending = extrema_enqueue(shard, sequence, instrument_order, y_scale, z_scale, state, compute_mins=compute_mins,
                              max_percentile=max_percentile, log_floor_cutoff=log_floor_cutoff,
                              log_floor_value=log_floor_value, comm=comm, per_step=on_step_done is not None)
    return extrema_finish(pending, on_step_done)


def load_extrema_state(extrema_json_path: str = FAST_EXTREMA_JSON_PATH) -> dict[str, Any]:
    """The cached extrema JSON (``{}`` when absent or unreadable, reference ``:137-149``)."""
    if not os.path.exists(extrema_json_path):
        return {}
    try:
        with open(extrema_json_path) as handle:
            return json.load(handle)
    except (OSError, json.JSONDecodeError) as exc:
        log_exception(f"[EXTREMA] Failed to read existing extrema JSON '{extrema_json_path}' (starting fresh)", exc, level="message")
        return {}


def orbits_the_scan_needs(sequence, instrument_order, y_scale, z_scale, state, log_floor_cutoff=0.1, log_floor_value=-1.0):
    """``{orbit index: {instrument, ...}}`` -- the files whose cubes the pre-pass still has to read with this
    cache state (a finished or re-usable cache needs none: the walk then only copies / transforms keys)."""
    steps, _ = plan_scanned_steps(sequence, tuple(instrument_order), y_scale, z_scale, state, log_floor_cutoff, log_floor_value)
    needs: dict[int, set] = {}
    for inst, indices in steps.items():
        for oi in indices:
            needs.setdefault(oi, set()).add(inst)
    return needs


def compute_global_extrema(
    directory_path: str,
    y_scale: str,
    z_scale: str,
    instrument_order: Iterable[str],
    extrema_json_path: str = FAST_EXTREMA_JSON_PATH,
    compute_mins: bool = False,
    max_percentile: float = 95.0,
    log_floor_cutoff: float = 0.1,
    log_floor_value: float = -1.0,
    flush_batch_size: int = 10,
    _shard=None,
    _comm=None,
) -> dict[str, Any]:
    """Compute or resume the cached per-instrument extrema (reference ``:73-366``).

    ``_shard`` (internal) re-uses sums a batch driver already holds on the GPU; stand-alone, the files the
    scan needs stream through pinned slots chunk by chunk (``Batch.collapse_pending``), so neither host
    RAM nor HBM holds more than a few chunks of cubes.

    ``flush_batch_size`` is accepted for call compatibility: the reference rewrites the JSON every
    ``flush_batch_size`` steps of a pass that takes minutes to hours, so that an interrupted run can resume
    (``:333-344``); here the whole pass is a few kernel launches whose results -- the maxima over EVERY
    prefix pool -- arrive together, so there is no meaningful intermediate state to persist and the cache
    is written once, complete, when the pass is done.
    """
    from ..cdf_utils import load_fast_cdf_dataset
    from .orbit_discovery import discover_orbit_files

    instrument_order = tuple(instrument_order)
    state = load_extrema_state(extrema_json_path)

    orbit_files = discover_orbit_files(directory_path, instrument_order)
    orbits = sorted(orbit_files)
    sequence = [(o, {i: True for i in orbit_files[o]}) for o in orbits]
    last_key = f"{y_scale}_{z_scale}_last_orbit"

    def dump():
        if _comm is not None and getattr(_comm, "rank", 0) != 0:
            return  # every rank holds the same state; rank 0 owns the cache file
        payload = state
        if last_key in state:
            payload = {last_key: state[last_key], **{k: v for k, v in state.items() if k != last_key}}
        try:
            with open(extrema_json_path, "w") as handle:
                json.dump(payload, handle, indent=2)
        except OSError as exc:
            log_exception("[EXTREMA] flush failure", exc, level="message")

    shard = _shard
    touched = False
    if shard is None:
        needs = orbits_the_scan_needs(sequence, instrument_order, y_scale, z_scale, state, log_floor_cutoff, log_floor_value)
        if needs:
            from .. import _lib
            from .pipeline import ShardPlan, ingest_orbits

            shard = ShardPlan(_lib.default_context(), y_scale, z_scale, instrument_order=instrument_order)
            shard.first_orbit_index = 0

            def load_one(oi, alloc):
                datasets = {}
                for inst in needs.get(oi, ()):
                    path = orbit_files[orbits[oi]].get(inst)
                    if path is None:
                        continue
                    try:
                        datasets[inst] = load_fast_cdf_dataset(path, data_alloc=alloc)
                    except Exception as exc:
                        log_exception(f"[EXTREMA] Ingest failure inst={inst} orbit={orbits[oi]} file={path}", exc, level="message")
                return orbits[oi], datasets, None

            def refused(orbit, exc):
                log_exception(f"[EXTREMA] Ingest failure orbit={orbit}", exc, level="message")

            ingest_orbits(shard, range(len(orbits)), load_one, refused)
    if shard is None:
        # nothing reaches the scan (everything re-used or complete): only the bookkeeping runs
        totals = {i: sum(1 for _, h in sequence if i in h) for i in instrument_order}

        def unreachable(inst, orbit_index, handle):
            raise AssertionError("scan step without a planned shard")

        def step_done(reuse: bool):
            nonlocal touched
            touched = True

        _walk(sequence, instrument_order, y_scale, z_scale, state, totals, log_floor_cutoff, log_floor_value,
              unreachable, step_done)
    else:
        before = json.dumps(state, sort_keys=True, default=str)
        extrema_from_shard(
            shard, sequence, instrument_order, y_scale, z_scale, state, compute_mins=compute_mins,
            max_percentile=max_percentile, log_floor_cutoff=log_floor_cutoff, log_floor_value=log_floor_value,
            comm=_comm,
        )
        touched = json.dumps(state, sort_keys=True, default=str) != before
    if touched:
        dump()
    if last_key in state:
        return {last_key: state[last_key], **{k: v for k, v in state.items() if k != last_key}}
    return state
