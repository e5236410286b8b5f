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
from dataclasses import dataclass
from typing import Any, NamedTuple

import numpy as np

from ..comm import TorchComm, block_of, current_device, rank_world
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


def _last_done(state, y_scale, z_scale) -> int:
    """The last orbit the cached walk of this (y, z) combo finished (-1: none or unreadable)."""
    stored = state.get(f"{y_scale}_{z_scale}_last_orbit", -1)
    return int(stored) if isinstance(stored, (int, float)) else -1


def _merge(prev_e, prev_z, cand_e, cand_z):
    """One step's running-max merge as the reference stores it: ``(y_max, z_max)``, an int capped at
    4000 and a float (the JSON cache is compared and written as is, so the types are part of the result)."""
    merged_e = max(float(prev_e), cand_e) if isinstance(prev_e, (int, float)) else cand_e
    merged_z = max(float(prev_z), cand_z) if isinstance(prev_z, (int, float)) else cand_z
    return int(min(4000, math.ceil(merged_e))), float(math.ceil(merged_z))


def _walk(sequence, instrument_order, y_scale, z_scale, state, totals, log_floor_cutoff, log_floor_value,
          on_scan, on_step_done=None, *, range_max=None):
    """The reference's orbit x instrument loop (``:183-331``) with the scan abstracted.

    ``sequence``: [(orbit, {inst: handle})] ascending.  ``on_scan(inst, orbit_index, handle)``
    is called where the reference loads a file and updates its pools, and must return
    ``(candidate_energy_max, candidate_intensity_max, intensity_min_store)``.  ``range_max(inst, first,
    stop)``: the same for the largest candidates of steps first..stop (None: unknown), to fold a chain.
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
    last_done = _last_done(state, y_scale, z_scale)
    y_log, z_log = y_scale == "log", z_scale == "log"
    if on_step_done is None and _walk_chains(sequence, instrument_order, y_scale, z_scale, state, totals, last_done,
                                             on_scan, range_max):
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
            y_max, z_max = _merge(state.get(k_ymax), state.get(k_zmax), cand_e, cand_z)
            state[k_ymin] = 0
            state[k_ymax] = y_max
            state[k_zmin] = z_min_store
            state[k_zmax] = z_max
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
        last_done = _last_done(state, y_scale, z_scale)
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


def _walk_chains(sequence, instrument_order, y_scale, z_scale, state, totals, last_done, on_scan, range_max) -> bool:
    """The loop of :func:`_walk` when every (orbit, instrument) step is a plain scan step: nothing
    is re-used from the linear/linear keys, nothing is complete, nobody watches the intermediate
    states.  Then the instruments are independent max-merge chains and only their last writes
    survive, so each chain runs on local variables and ``state`` is written once -- the same
    arithmetic in the same order per instrument, without ~25 dict operations per step, or with
    ``range_max`` one merge per chain.  Returns False (state untouched) when the preconditions do not hold."""
    ranges = chain_ranges(sequence, instrument_order, y_scale, z_scale, state, totals, last_done)
    if ranges is None:
        return False
    first, stops = ranges
    results = {}
    last_executed = first
    for inst in instrument_order:
        stem = f"{inst}_{y_scale}_{z_scale}"
        prev_e, prev_z = state.get(f"{stem}_y_max"), state.get(f"{stem}_z_max")
        stop = stops[inst]
        folded = range_max(inst, first, stop) if range_max is not None else None
        if folded is not None:
            # ceil and min(4000, .) are monotone, so folding the max-merge over the steps equals
            # one merge with the largest candidate: min(4000, ceil(max(prev, c_first..c_stop)))
            cand_e, cand_z, z_min_store = folded
            prev_e, prev_z = _merge(prev_e, prev_z, cand_e, cand_z)
        else:
            z_min_store = 0
            for orbit_index in range(first, stop + 1):
                cand_e, cand_z, z_min_store = on_scan(inst, orbit_index, sequence[orbit_index][1].get(inst))
                prev_e, prev_z = _merge(prev_e, prev_z, cand_e, cand_z)
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


class _EnergyPlan(NamedTuple):
    """One instrument's part of :func:`_energy_plan`."""

    present: list  # scanned steps (orbit indices) whose file some rank holds
    rows: np.ndarray  # their rows in the gathered per-file count table
    energies: list  # their energy tables (equal tables folded into one object)
    steps: np.ndarray  # every scanned step of the instrument
    pos: np.ndarray  # position of every present step inside `steps`
    ascending: bool  # `steps` strictly ascending
    table: tuple | None  # shared_energy_table() when every present file shares one table


def _energy_plan(shard, comm, instrument_order, steps, owners, first):
    """Who holds the per-energy counts of every scanned step (static per plan; exchanged once):
    ``({inst: _EnergyPlan}, count rows per rank, max_E)``."""
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
        # static index maps of the per-step candidate fill (extrema_finish)
        steps_arr = np.asarray(steps[inst], dtype=np.int64)
        pos = np.searchsorted(steps_arr, np.asarray(present, dtype=np.int64)) if present else np.zeros(0, np.int64)
        ascending = bool(np.all(np.diff(steps_arr) > 0)) if len(steps_arr) > 1 else True
        table = shared_energy_table(en[0]) if en and all(e is en[0] for e in en) else None
        rows = np.asarray([where[(inst, oi)] for oi in present], dtype=np.int64)
        plan[inst] = _EnergyPlan(present, rows, en, steps_arr, pos, ascending, table)
    return plan, n_max, max_E


def _device_y_tables(instrument_order, eplan, max_E, ranges, owners, first):
    """Static energy tables for ``csg_pool_energy_candidates`` over the chains of
    :func:`chain_ranges` -- or None when there are no chains, or some instrument's files do not
    share one table of distinct, NaN-free energies (the host path handles those)."""
    if ranges is None:
        return None
    first_step, stops = ranges
    n_inst = len(instrument_order)
    order = np.zeros((n_inst, max_E), dtype=np.int32)
    keys = np.zeros((n_inst, max_E), dtype=np.float64)
    n_keys = np.zeros(n_inst, dtype=np.int32)
    zero = {}
    for ii, inst in enumerate(instrument_order):
        ep = eplan[inst]
        if not ep.ascending:
            return None
        cov = np.zeros(int(ep.steps.max()) + 1 if len(ep.steps) else 0, dtype=bool)
        if ep.present:
            if ep.table is None:
                return None
            e0, uniq, _idx = ep.table
            if len(uniq) != len(e0) or len(e0) > max_E or np.isnan(e0).any():
                return None
            o = np.argsort(e0, kind="stable")
            order[ii, : len(e0)], keys[ii, : len(e0)], n_keys[ii] = o, e0[o], len(e0)
            idx = np.full(len(ep.steps), -1, dtype=np.int64)
            idx[ep.pos] = 1
            cov[ep.steps] = np.maximum.accumulate(idx) >= 0
        # some step of the chain sees the 0.0 candidate (no file yet)
        part = cov[first_step : stops[inst] + 1]
        zero[inst] = not (len(part) == stops[inst] + 1 - first_step and bool(part.all()))
    # positions of this rank that take part in each chain (global orbit index <= stop)
    limit = np.array([sum(1 for i2, oi, _f in owners if i2 == inst and oi + first <= stops[inst]) for inst in instrument_order],
                     dtype=np.int32)
    return {"order": order, "keys": keys, "n_keys": n_keys, "limit": limit, "zero": zero}


class _ExtremaPlan(NamedTuple):
    """One entry of ``shard._extrema_plan_cache``: what depends only on the orbit sequence and the cache state."""

    sequence: list  # held so that its id(), part of the cache key, cannot be recycled while the entry lives
    totals: dict
    items: np.ndarray  # this rank's POOL_ITEM rows
    inst_len: np.ndarray
    eplan: dict  # {inst: _EnergyPlan}
    n_max: int  # count rows per rank in the gathered per-file count table
    max_E: int
    ytab: dict | None  # _device_y_tables()


@dataclass
class PendingExtrema:
    """The selection :func:`extrema_enqueue` left running, and what :func:`extrema_finish` needs to redeem it."""

    shard: Any
    selector: Any  # pool_select.DevicePoolSelector
    comm: Any
    sequence: list
    instrument_order: tuple
    y_scale: str
    z_scale: str
    state: dict
    totals: dict
    compute_mins: bool
    log_floor_cutoff: float
    log_floor_value: float
    requests: list
    items: np.ndarray  # items, inst_len, max_E: the host-driven fallback's input
    inst_len: np.ndarray
    max_E: int
    eplan: dict
    ydev: dict | None  # the y candidates were max-merged on the device with these tables


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
        ytab = _device_y_tables(instrument_order, eplan, max_E, ranges, owners, first)
        if len(cache) > 8:
            cache.clear()
        hit = cache[key] = _ExtremaPlan(sequence, totals, items, inst_len, eplan, n_max, max_E, ytab)
    ydev = hit.ytab if not per_step else None
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
    selector.enqueue(shard.batch.dtype, hit.items, len(instrument_order), hit.inst_len, hit.max_E, requests, comm=comm,
                     count_rows=hit.n_max, ydev=ydev)
    return PendingExtrema(
        shard=shard, selector=selector, comm=comm, sequence=sequence, instrument_order=instrument_order,
        y_scale=y_scale, z_scale=z_scale, state=state, totals=hit.totals, compute_mins=compute_mins,
        log_floor_cutoff=log_floor_cutoff, log_floor_value=log_floor_value, requests=requests, items=hit.items,
        inst_len=hit.inst_len, max_E=hit.max_E, eplan=hit.eplan, ydev=ydev,
    )


def extrema_finish(pending: PendingExtrema, on_step_done=None):
    """Wait for the selection's read-backs and run the reference's bookkeeping walk on the results.

    The y candidates are per step, from every rank's per-file counts -- or, when
    :func:`extrema_enqueue` max-merged them on the device, one per instrument."""
    device_y = pending.ydev is not None
    if device_y and on_step_done is not None:
        raise ValueError("extrema_enqueue(per_step=False) cannot report the state after every step")
    order = pending.instrument_order
    if not device_y:
        # the per-file counts are read back after the first histogram pass: the per-step candidates
        # are built while the digit loop runs on the GPU, before anything waits for the values
        all_counts, _npos = pending.selector.result_counts()  # multi-rank: every rank's rows (device all-gather)
        cand_e = {}  # {inst: [orbit index] -> the candidate the reference's step sees}
        for inst in order:
            ep = pending.eplan[inst]
            dense = np.zeros(len(pending.sequence), dtype=np.float64)
            if ep.present and ep.ascending:
                ce = energy_candidates(ep.energies, all_counts[ep.rows], as_array=True, shared_table=ep.table)
                # steps without a file repeat the previous candidate (0.0 before the first file)
                idx = np.full(len(ep.steps), -1, dtype=np.int64)
                idx[ep.pos] = np.arange(len(ep.present))
                filled = np.maximum.accumulate(idx)
                dense[ep.steps] = np.where(filled >= 0, ce[np.maximum(filled, 0)], 0.0)
            elif ep.present:
                by_step = dict(zip(ep.present, energy_candidates(ep.energies, all_counts[ep.rows])))
                running = 0.0
                for oi in ep.steps.tolist():
                    running = by_step.get(oi, running)
                    dense[oi] = running
            cand_e[inst] = dense
    values = _selected_values(pending)
    n_inst = len(order)
    z, z_min = {}, {}
    for ii, inst in enumerate(order):
        z[inst] = float(values[ii]) if values[ii] is not None else 0.0
        zm = values[n_inst + ii] if pending.compute_mins else None
        z_min[inst] = float(zm) if zm is not None else 0
    if device_y:
        top = {}
        for inst, y in zip(order, pending.selector.result_y_candidates()):
            if y is None:
                y = 0.0  # no file took part: every step of the chain saw the empty-pool candidate
            elif pending.ydev["zero"][inst]:
                y = max(y, 0.0)
            top[inst] = y

        def scan(inst, orbit_index, handle):
            raise AssertionError("per-step scan requested from a device-merged selection")

        def range_max(inst, first, stop):
            return top[inst], z[inst], z_min[inst]
    else:

        def scan(inst, orbit_index, handle):
            return float(cand_e[inst][orbit_index]), z[inst], z_min[inst]

        def range_max(inst, first, stop):
            """Largest candidates over the steps first..stop (None: NaN candidates, walk step by step)."""
            y = float(cand_e[inst][first : stop + 1].max())
            if y != y or z[inst] != z[inst]:
                return None
            return y, z[inst], z_min[inst]

    return _walk(pending.sequence, order, pending.y_scale, pending.z_scale, pending.state, pending.totals,
                 pending.log_floor_cutoff, pending.log_floor_value, scan, on_step_done, range_max=range_max)


def _selected_values(pending: PendingExtrema) -> list:
    """One value per request (None: empty pool): the device selection's, or -- when more candidate
    buckets survived than its slot table holds -- the same kernels with the digit loop driven from
    the host, on a backend kept as ``shard._pool_backend``."""
    from ..pool_select import GpuPoolBackend, prefix_percentiles

    values = pending.selector.result_values()
    if values is None:
        shard = pending.shard
        backend = getattr(shard, "_pool_backend", None)
        if backend is None:
            backend = shard._pool_backend = GpuPoolBackend(shard.batch)
        values, _, _ = prefix_percentiles(backend, shard.batch.dtype, pending.items, len(pending.instrument_order),
                                          pending.inst_len, pending.max_E, pending.requests, comm=pending.comm)
    return values


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

    Stand-alone under ``torchrun`` (``torch.distributed`` initialised, several ranks) the ranks share the
    scan like the directory driver's: each reads the files of its contiguous block of the ascending orbit
    sequence on its own GPU, and the pooled extrema are exchanged.  Rank 0 reads the cache and hands it to
    the others, every rank returns the same dict, and rank 0 alone writes the JSON.

    ``flush_batch_size`` is accepted for call compatibility: the reference rewrites the JSON every
    ``flush_batch_size`` steps of a pass that takes minutes to hours, so that an interrupted run can resume
    (``:333-344``); here the whole pass is a few kernel launches whose results -- the maxima over EVERY
    prefix pool -- arrive together, so there is no meaningful intermediate state to persist and the cache
    is written once, complete, when the pass is done.
    """
    from ..cdf_utils import load_fast_cdf_dataset
    from .orbit_discovery import discover_orbit_files

    instrument_order = tuple(instrument_order)
    comm, device = _comm, 0
    rank, world, dist = rank_world() if _shard is None and _comm is None else (0, 1, None)
    if world > 1:
        import torch

        device = current_device()
        comm = TorchComm(dist, torch.device("cuda", device))
        # every rank plans the same scan from rank 0's reading, and no rank reads the file rank 0 rewrites
        box = [load_extrema_state(extrema_json_path) if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        state = box[0]
    else:
        state = load_extrema_state(extrema_json_path)

    orbit_files = discover_orbit_files(directory_path, instrument_order)
    orbits = sorted(orbit_files)
    sequence = [(o, {i: True for i in orbit_files[o]}) for o in orbits]
    last_key = f"{y_scale}_{z_scale}_last_orbit"

    def dump():
        if comm is not None and getattr(comm, "rank", 0) != 0:
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

            lo, hi = block_of(len(orbits), rank, world)
            shard = ShardPlan(_lib.default_context(device), y_scale, z_scale, instrument_order=instrument_order)
            shard.first_orbit_index = lo

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

            ingest_orbits(shard, range(lo, hi), load_one, refused)
            if world > 1:
                shard.agree_dtype(dist, world)
                if lo >= hi:  # a rank past the last orbit still joins the exchange, with empty outputs of K1
                    shard.collapse_pending()
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
            comm=comm,
        )
        touched = json.dumps(state, sort_keys=True, default=str) != before
    if touched:
        dump()
    if last_key in state:
        return {last_key: state[last_key], **{k: v for k, v in state.items() if k != last_key}}
    return state
