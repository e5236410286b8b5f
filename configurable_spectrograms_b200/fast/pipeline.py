"""One GPU shard of the FAST batch path: cubes -> sums -> extrema -> panels -> rasters.

This is the B200 re-design of what the reference does per worker process
(``fast/process_orbit.py`` -> ``fast/plotting.py`` -> ``plotting.py``): instead of one
orbit per process and twelve ``np.nansum`` per figure, every cube of the shard is
reduced once (K1), every percentile the figure builders need is selected in one launch
(K2a), the pooled extrema come from the same collapsed matrices (K2b) and every panel
of every figure is rasterised in one launch (K3).  Host Python only plans descriptor
tables and composes figures.

The planner restates the reference's masks and bound selection verbatim (citations
inline) so that panels, bounds and figure/file naming are identical.
"""

from __future__ import annotations

import os
from dataclasses import dataclass, field

import numpy as np

from .. import _lib
from ..engine import WANT_GEOMETRY, WANT_PERCENTILES, WANT_REDUCTIONS, Batch, compute_dtype
from .constants import DEFAULT_INSTRUMENT_ORDER, DEFAULT_PITCH_ANGLE_CATEGORIES, PITCH_ANGLE_ROW_KEYS


def pitch_angle_bits(pitch_angle: np.ndarray, categories: dict, row_keys=PITCH_ANGLE_ROW_KEYS):
    """(uint8[P] membership bits, row keys present) -- ``fast/plotting.py:121-127``.

    Closed intervals, NaN bins match nothing; bit g belongs to the g-th present row key.
    """
    keys = [k for k in row_keys if k in categories]
    bits = np.zeros(len(pitch_angle), dtype=np.uint8)
    with np.errstate(invalid="ignore"):
        for g, key in enumerate(keys):
            member = np.zeros(len(pitch_angle), dtype=bool)
            for lo, hi in categories[key]:
                member |= (pitch_angle >= lo) & (pitch_angle <= hi)
            bits |= (member.astype(np.uint8) << g).astype(np.uint8)
    return bits, keys


def zoom_window(vertical_lines, zoom_duration_minutes):
    """(center, duration) of the zoom column -- ``plotting.py:586-596``; None without lines."""
    if not vertical_lines:
        return None
    if len(vertical_lines) == 1:
        return vertical_lines[0], zoom_duration_minutes * 60
    center = 0.5 * (vertical_lines[0] + vertical_lines[1])
    return center, max(zoom_duration_minutes * 60, abs(vertical_lines[1] - vertical_lines[0]) * 1.5)


@dataclass
class RowSpec:
    label: str
    file: int
    group: int
    full_panel: int | None
    zoom_panel: int | None
    times: np.ndarray
    energy: np.ndarray  # the y axis handed to make_spectrogram (unfiltered)
    vmin: float | None = None
    vmax: float | None = None


@dataclass
class FigureSpec:
    kind: str  # "pitch-angle" | "instrument-grid"
    orbit: int
    variant: str  # "given" | "raw"
    instrument: str | None
    title: str
    rows: list[RowSpec] = field(default_factory=list)
    vertical_lines: list[float] | None = None
    zoom: tuple[float, float] | None = None
    zoom_needed: bool = False  # filled per step from the K1 row flags (resolve_zoom_flags)
    zoom_windows: list[int] = field(default_factory=list)
    error: str | None = None


class ShardPlan:
    """Plans and runs the batch path for a list of orbits on one GPU."""

    def __init__(self, ctx, y_scale="linear", z_scale="linear", zoom_duration_minutes=6.25,
                 instrument_order=DEFAULT_INSTRUMENT_ORDER, pitch_angle_categories=None, dtype=None):
        """``dtype``: the cube dtype D every kernel computes in (numpy sums, ranks and normalises in the
        array's own dtype, so D is part of the result).  ``None`` = taken from the first cube added; a
        later cube of another float dtype is refused (:meth:`add_orbit`) -- never cast silently."""
        self.ctx = ctx
        self.y_scale, self.z_scale = y_scale, z_scale
        self.zoom_minutes = zoom_duration_minutes
        self.instrument_order = tuple(instrument_order)
        self.categories = pitch_angle_categories or DEFAULT_PITCH_ANGLE_CATEGORIES
        self.n_groups = len([k for k in PITCH_ANGLE_ROW_KEYS if k in self.categories])
        self._dtype = None if dtype is None else np.dtype(dtype)
        self._batch = None if dtype is None else Batch(ctx, dtype, n_groups=self.n_groups)
        self.orbits: list[dict] = []  # {"orbit", "files": {inst: file_id}, "lines": {inst: [..]}}
        self.file_meta: list[dict] = []
        self.figures: list[FigureSpec] = []
        self._panel_cache: dict = {}
        self._region_cache: dict = {}
        self._cols_cache: dict = {}
        self._full_stats: dict = {}  # (file, group) -> percentile region over the [0,4000] eV cells, every row
        self._window_cache: dict = {}
        self._full_region_of: dict = {}  # region id -> (file, group) for full panels over every time row

    @property
    def batch(self) -> Batch:
        if self._batch is None:  # nothing added yet: float32 (FAST counts are CDF_FLOAT) unless a dtype was given
            if self._dtype is None:
                self._dtype = np.dtype(np.float32)
            self._batch = Batch(self.ctx, self._dtype, n_groups=self.n_groups)
        return self._batch

    @staticmethod
    def compute_dtype(data_dtype) -> np.dtype:
        """The dtype numpy computes a cube of ``data_dtype`` in: float32 / float64 stay; everything else
        (integer counts) goes through float64, the dtype ``np.nanpercentile`` and matplotlib use for it."""
        return compute_dtype(data_dtype)

    # ------------------------------------------------------------- phase 1: files
    def add_orbit(self, orbit: int, datasets: dict, lines: dict | None = None):
        """``datasets``: {inst: load_fast_cdf_dataset(...) dict}; ``lines``: {inst: cusp timestamps}.

        Raises ``TypeError`` when a cube's float dtype differs from the shard's: the reference computes
        every file in its own dtype, and pools of mixed dtypes in float64 (``np.concatenate`` promotes,
        ``CS/fast/extrema.py:280``); one shard computes in one dtype, so the caller has to keep files
        of different dtypes in different shards rather than have them cast behind its back."""
        for inst, ds in datasets.items():
            if "device_ptr" in ds:
                continue
            want = self.compute_dtype(np.asarray(ds["data"]).dtype)
            if self._dtype is None:
                self._dtype = want
                self._batch = Batch(self.ctx, want, n_groups=self.n_groups)
            elif want != self._dtype:
                raise TypeError(f"orbit {orbit} {inst}: cube dtype {np.asarray(ds['data']).dtype} in a {self._dtype} shard "
                                "(mixed dtypes are not cast silently: use one shard per dtype)")
        entry = {"orbit": orbit, "files": {}, "lines": lines or {}}
        for inst, ds in datasets.items():
            energy = np.asarray(ds["energy"])
            pitch = np.asarray(ds["pitch_angle"])
            bits, keys = pitch_angle_bits(pitch, self.categories)
            if "device_ptr" in ds:  # cube already resident in HBM (T,P,E C-order unless "layout" says otherwise)
                fid = self.batch.add_file(None, bits, shape=ds["shape"], layout=ds.get("layout"), device_ptr=ds["device_ptr"])
            else:
                data = np.asarray(ds["data"])
                # integer counts only (see compute_dtype); 8/16/32-bit ones stay as stored (in their pinned
                # staging slot) -- K1 reads them and writes the exact float64 sums
                if data.dtype != self.batch.dtype and data.dtype not in _lib.INT_CUBE_CODES:
                    data = data.astype(self.batch.dtype)
                fid = self.batch.add_file(data, bits)
            self.file_meta.append({"times": np.asarray(ds["times"]), "energy": energy, "keys": keys, "inst": inst, "orbit": orbit})
            entry["files"][inst] = fid
        self.orbits.append(entry)

    def agree_dtype(self, dist, world: int):
        """Collective (every rank of a multi-rank scan, after its ingest): one pool, one key width, so every
        rank computes in the same dtype.  A rank that read no cube (more GPUs than orbits, or a block the scan
        does not need) adopts its peers'; ranks that read cubes of different float dtypes cannot share a pool
        (:meth:`add_orbit` refuses that within a shard for the same reason)."""
        mine = self._dtype.name if self.file_meta else None
        seen: list = [None] * world
        dist.all_gather_object(seen, mine)
        kinds = sorted({d for d in seen if d is not None})
        if len(kinds) > 1:
            raise TypeError(f"ranks read cubes of different dtypes ({', '.join(kinds)}): one run computes in one dtype")
        if kinds and self._dtype != np.dtype(kinds[0]):
            self._dtype = np.dtype(kinds[0])
            self._batch = None
            if self.orbits:  # orbits added without files: their (empty) K1 outputs again, in the new batch
                self.collapse_pending()

    def upload(self):
        self.batch.upload_cubes()

    def collapse(self):
        self.batch.collapse()

    def collapse_pending(self) -> int:
        """Streaming ingest (``engine.Batch.collapse_pending``): upload + K1 for the orbits added since
        the last call; their cubes are not kept, neither on the host nor in HBM."""
        return self.batch.collapse_pending()

    # ------------------------------------------------------------ phase 2: panels
    def _energy_cols(self, file: int, lo, hi):
        """Columns kept by ``(E >= lo) & (E <= hi)`` (builder order, no flip) and the same
        after make_spectrogram's descending flip (``plotting.py:192-202``)."""
        energy = self.file_meta[file]["energy"]
        key = (energy.ctypes.data, len(energy), float(lo), float(hi))
        hit = self._cols_cache.get(key)
        if hit is None:
            with np.errstate(invalid="ignore"):
                keep = np.flatnonzero((energy >= lo) & (energy <= hi)).astype(np.int32)
            flipped = keep
            if len(keep) and energy[keep[0]] > energy[keep[-1]]:
                flipped = keep[::-1].copy()
            hit = self._cols_cache[key] = (keep, flipped)
        return hit

    def _region(self, file, group, cols, rows_key, rows, want_pct):
        key = (file, group, cols.ctypes.data, len(cols), rows_key)
        rid = self._region_cache.get(key)
        if rid is None:
            if isinstance(rows, tuple):
                rid = self.batch.add_region(file, group, cols, t0=rows[0], nt=rows[1], want_pct=want_pct)
            else:
                rid = self.batch.add_region(file, group, cols, rows=rows, want_pct=want_pct)
            self._region_cache[key] = rid
        else:
            self.batch.require_stats(rid, want_pct)
        return rid

    def _panel(self, region, pct_region, z_min, z_max, stat_region=-1):
        key = (region, pct_region, z_min, z_max, stat_region)
        pid = self._panel_cache.get(key)
        if pid is None:
            pid = self.batch.add_panel(region, pct_region, self.z_scale == "log", z_min, z_max, stat_region)
            self._panel_cache[key] = pid
        return pid

    def _rows_full(self, file):
        """Row mask of the full panel: ``x >= x[0]`` and ``x <= x[-1]`` (``plotting.py:212-219``)."""
        t = self.file_meta[file]["times"]
        with np.errstate(invalid="ignore"):
            m = (t >= t[0]) & (t <= t[-1])
        if m.all():
            return "full", (0, len(t))
        return "full", np.flatnonzero(m)

    def _rows_zoom(self, file, zoom):
        t = self.file_meta[file]["times"]
        center, duration = zoom
        half = duration / 2
        with np.errstate(invalid="ignore"):
            m = (t >= center - half) & (t <= center + half)  # plotting.py:204-210
        return ("zoom", float(center), float(duration)), np.flatnonzero(m)

    def _zoom_window(self, file, group_bit, zoom) -> int:
        """Window id for ``np.any(~np.isnan(d[mask_zoom]))`` (``plotting.py:597-603``), answered on
        the device from the K1 row flags (``csg_window_any``)."""
        key = (file, group_bit, float(zoom[0]), float(zoom[1]))
        wid = self._window_cache.get(key)
        if wid is None:
            t = self.file_meta[file]["times"]
            center, duration = zoom
            with np.errstate(invalid="ignore"):
                m = (t >= center - duration / 2) & (t <= center + duration / 2)
            wid = self._window_cache[key] = self.batch.add_window(file, group_bit, np.flatnonzero(m))
        return wid

    def resolve_zoom_flags(self, window_any: np.ndarray):
        """Fill every figure's ``zoom_needed`` from the downloaded ``csg_window_any`` result."""
        if not hasattr(self, "_zoom_index") or self._zoom_index[0] != len(self.figures):
            ids, starts, figs = [], [], []
            for fig in self.figures:
                fig.zoom_needed = False
                if fig.zoom_windows:
                    starts.append(len(ids))
                    ids.extend(fig.zoom_windows)
                    figs.append(fig)
            self._zoom_index = (len(self.figures), np.asarray(ids, dtype=np.int64), np.asarray(starts, dtype=np.int64), figs)
        _, ids, starts, figs = self._zoom_index
        if len(figs) == 0:
            return
        hit = np.maximum.reduceat(window_any[ids], starts)
        for fig, h in zip(figs, hit.tolist()):
            fig.zoom_needed = bool(h)

    def _rows_for_dataset(self, fig, label, file, group, builder_cols, z_given, zoom):
        """One dataset dict of the figure builders + its make_spectrogram panels."""
        meta = self.file_meta[file]
        if len(builder_cols) == 0 or len(meta["times"]) == 0:
            return  # matrix_full_plot.size == 0 -> dataset skipped (fast/plotting.py:132-133,283-284)
        z_lo, z_hi = z_given
        pct = -1
        if z_lo is None or z_hi is None:
            # compute_percentile_bounds(matrix_full_plot, 1, 99, z_min, z_max) on the builder matrix
            pct = self._region(file, group, builder_cols, "full", (0, len(meta["times"])), WANT_PERCENTILES)
        # make_spectrogram always clips energy to [0, 4000] here: y_axis_min/max are not
        # forwarded by generic_plot_multirow_optional_zoom (plotting.py:618-636 vs :104-105)
        plain, cols = self._energy_cols(file, 0, 4000)
        if pct >= 0 and builder_cols is plain:
            self._full_stats[(file, group)] = pct  # same cell set as the full panel (stats are order-free)
        row = RowSpec(label=label, file=file, group=group, full_panel=None, zoom_panel=None,
                      times=meta["times"], energy=meta["energy"])
        if len(cols):
            rk, rows = self._rows_full(file)
            n_rows = rows[1] if isinstance(rows, tuple) else len(rows)
            if n_rows:
                shared = self._full_stats.get((file, group), -1) if isinstance(rows, tuple) else -1
                reg = self._region(file, group, cols, rk, rows, WANT_GEOMETRY if shared >= 0 else WANT_REDUCTIONS)
                if isinstance(rows, tuple):
                    self._full_region_of[reg] = (file, group)
                row.full_panel = self._panel(reg, pct, z_lo, z_hi, shared)
            if zoom is not None:
                rk, rows = self._rows_zoom(file, zoom)
                if len(rows):
                    reg = self._region(file, group, cols, rk, rows, WANT_REDUCTIONS)
                    row.zoom_panel = self._panel(reg, pct, z_lo, z_hi)
        row.vmin, row.vmax = z_lo, z_hi
        fig.rows.append(row)

    def plan_pitch_angle_grid(self, orbit_entry, inst, variant, y_min=None, y_max=None, z_min=None, z_max=None):
        """``FAST_plot_pitch_angle_grid`` (``fast/plotting.py:34-174``) for one file."""
        file = orbit_entry["files"][inst]
        meta = self.file_meta[file]
        lines = orbit_entry["lines"].get(inst) or None
        fig = FigureSpec("pitch-angle", orbit_entry["orbit"], variant, inst,
                         f"Orbit {orbit_entry['orbit']} - Pitch Angle {inst} ESA Spectrograms",
                         vertical_lines=lines)
        y_lo = 0 if y_min is None else y_min
        y_hi = 4000 if y_max is None else y_max
        builder_cols, _ = self._energy_cols(file, y_lo, y_hi)
        fig.zoom = zoom_window(lines, self.zoom_minutes)
        for g, key in enumerate(meta["keys"]):
            self._rows_for_dataset(fig, key.title(), file, g + 1, builder_cols, (z_min, z_max), fig.zoom)
        if fig.zoom is not None:
            fig.zoom_windows = [self._zoom_window(r.file, r.group, fig.zoom) for r in fig.rows]
        self.figures.append(fig)
        return fig

    def plan_instrument_grid(self, orbit_entry, variant, global_extrema=None, y_min=None, y_max=None, z_min=None, z_max=None):
        """``FAST_plot_instrument_grid`` (``fast/plotting.py:177-328``) for one orbit."""
        fig = FigureSpec("instrument-grid", orbit_entry["orbit"], variant, None,
                         f"Orbit {orbit_entry['orbit']} -  ESA Spectrograms")
        lines = None
        pending = []
        for inst in self.instrument_order:
            file = orbit_entry["files"].get(inst)
            if file is None:
                continue
            if lines is None and orbit_entry["lines"] is not None and inst in orbit_entry["lines"]:
                lines = orbit_entry["lines"][inst]  # first instrument decides, even when empty (:258-265)
            if isinstance(global_extrema, dict):
                kp = f"{inst}_{self.y_scale}_{self.z_scale}"
                y_lo = global_extrema.get(f"{kp}_y_min", 0 if y_min is None else y_min)
                y_hi = global_extrema.get(f"{kp}_y_max", 4000 if y_max is None else y_max)
                row_z = (global_extrema.get(f"{kp}_z_min"), global_extrema.get(f"{kp}_z_max"))
            else:
                y_lo = 0 if y_min is None else y_min
                y_hi = 4000 if y_max is None else y_max
                row_z = (None, None)
            pending.append((inst, file, y_lo, y_hi, row_z))
        fig.vertical_lines = lines if lines else None
        fig.zoom = zoom_window(lines, self.zoom_minutes) if lines else None
        for inst, file, y_lo, y_hi, row_z in pending:
            builder_cols, _ = self._energy_cols(file, y_lo, y_hi)
            # vmin/vmax = percentiles or the per-instrument extrema; a figure-level z_min/z_max
            # argument overrides them inside generic_plot_multirow_optional_zoom (plotting.py:632-633)
            z_lo = row_z[0] if z_min is None else z_min
            z_hi = row_z[1] if z_max is None else z_max
            self._rows_for_dataset(fig, inst.upper(), file, 0, builder_cols, (z_lo, z_hi), fig.zoom)
        if fig.zoom is not None:
            fig.zoom_windows = [self._zoom_window(r.file, 0, fig.zoom) for r in fig.rows]
        self.figures.append(fig)
        return fig

    def reset_plan(self):
        """Drop every planned figure / panel (files and their collapsed sums stay valid)."""
        self.batch.reset_tables()
        self.figures = []
        self._panel_cache, self._region_cache, self._full_stats, self._window_cache = {}, {}, {}, {}
        self._full_region_of = {}
        if hasattr(self, "_zoom_index"):
            del self._zoom_index

    # ------------------------------------------------------------------ execution
    def share_full_stats(self):
        """One pass per cell set: a full panel planned BEFORE the percentile region of the same cells existed
        (the "given" figures come first, ``fast/process_orbit.py:148-190``) asked for its own reductions; the
        percentile region over the [0, 4000] eV rows of the same (file, group) computes exactly those
        (safe_vmin, nanmin / nanmax are order-free), so such panels are pointed at it and regions nobody
        reads any more become geometry only -- K2a touches every cell set once instead of twice."""
        b = self.batch
        own = set()
        for (region, _pct, _lo, _hi, stat_region), pid in self._panel_cache.items():  # every panel of the plan
            if stat_region < 0:
                shared = self._full_stats.get(self._full_region_of.get(region))
                if shared is not None and shared != region:
                    b.set_stat_region(pid, shared)
                    continue
                own.add(region)
        for rid in self._full_region_of:
            if rid not in own:
                b.drop_reductions(rid)

    def upload_tables(self):
        self.share_full_stats()
        self.batch.upload_tables()

    def run_panels(self, lut259=None, want_index=True):
        """K2a, panel norms and K3 over the uploaded tables (``lut259=None``: the LUT already set)."""
        b = self.batch
        b.run_stats()
        b.prepare()
        if lut259 is not None:
            b.set_lut(lut259)
        b.rasterise(want_rgba=lut259 is not None or b.d_lut is not None, want_index=want_index)

    def run_once(self, lut259, want_index=True):
        """Compute every planned figure of a collapsed shard once: tables, zoom windows, :meth:`run_panels`,
        then the figures' ``zoom_needed`` flags (the rasters stay on the device)."""
        self.upload_tables()
        self.batch.run_windows()
        self.run_panels(lut259, want_index)
        self.resolve_zoom_flags(self.batch.window_any())

    def pool_items(self, steps_by_inst: dict[str, list[int]]):
        """POOL_ITEM table for the scanned (orbit index) steps of every instrument."""
        from .._lib import POOL_ITEM

        rows = []
        inst_len = np.zeros(len(self.instrument_order), dtype=np.int32)
        owners = []
        for ii, inst in enumerate(self.instrument_order):
            pos = 0
            for oi in steps_by_inst.get(inst, []):
                file = self.orbits[oi]["files"].get(inst)
                if file is None:
                    continue
                f = self.batch.files[file]
                rows.append((self.batch.mat_off(file, 0), f["T"], f["E"], ii, pos))
                owners.append((inst, oi, file))
                pos += 1
            inst_len[ii] = pos
        items = np.array(rows, dtype=POOL_ITEM) if rows else np.zeros(0, POOL_ITEM)
        return items, inst_len, owners


def chunk_orbits() -> int:
    """Orbits per streaming chunk (``CSG_CHUNK_ORBITS``, default 8; a malformed value means the default): a
    nominal 4-instrument orbit is 84 MB of cubes, so the default keeps one pinned slot / the device staging
    buffer near 0.7 GB."""
    try:
        return max(1, int(os.environ.get("CSG_CHUNK_ORBITS", "8")))
    except ValueError:
        return 8


def ingest_orbits(shard: ShardPlan, indices, load, refused, n_threads: int = 4):
    """Streaming ingest: add the orbits ``indices`` to ``shard`` and collapse them, :func:`chunk_orbits` at a time.

    ``load(index, alloc) -> (orbit, datasets, lines)`` runs on one of ``n_threads`` loader threads and decodes
    the orbit's cubes into ``alloc(shape, dtype)``: pinned memory of the chunk's staging slot.  Chunk k+1 is
    decoded while chunk k is uploaded and collapsed (``ShardPlan.collapse_pending``), so neither host RAM nor
    HBM holds more cubes than the three slots of the context's ring (``CSG_SLOT_BYTES`` each).  An orbit whose
    cubes ``add_orbit`` refuses (a float dtype other than the shard's) goes to ``refused(orbit, exc)`` and is
    added without files."""
    from concurrent.futures import ThreadPoolExecutor
    from functools import partial

    from ..logging_utils import log_exception

    indices = list(indices)
    if not indices:
        return
    chunk_n = chunk_orbits()
    chunks = [indices[a : a + chunk_n] for a in range(0, len(indices), chunk_n)]
    slot_bytes = int(os.environ.get("CSG_SLOT_BYTES", str(max(1 << 28, chunk_n * 100 * (1 << 20)))))
    ring = _lib.shared_ring(shard.ctx, n_slots=3, slot_bytes=slot_bytes)
    try:
        with ThreadPoolExecutor(max_workers=n_threads) as pool:
            def submit(chunk):
                slot = ring.acquire()
                return slot, [pool.submit(load, i, partial(ring.alloc, slot)) for i in chunk]

            in_flight = submit(chunks[0])
            for k in range(len(chunks)):
                slot, futures = in_flight
                loaded = [f.result() for f in futures]
                in_flight = submit(chunks[k + 1]) if k + 1 < len(chunks) else None
                for orbit, datasets, lines in loaded:
                    try:
                        shard.add_orbit(orbit, datasets, lines)
                    except TypeError as exc:
                        refused(orbit, exc)
                        shard.add_orbit(orbit, {}, {})
                shard.collapse_pending()
                ring.release(slot)
    finally:
        ring.drain()  # the ring belongs to the context and serves the next call too
    if ring.overflow_bytes:
        log_exception(f"[INGEST] {ring.overflow_bytes} bytes of cubes did not fit the pinned slots "
                      f"({slot_bytes} bytes each; CSG_SLOT_BYTES / CSG_CHUNK_ORBITS) and were uploaded from pageable memory",
                      level="message")


class BatchStep:
    """One batch step of the reference's directory driver for this rank's shard of orbits.

    ``fast/batch_directory.py:159-171`` runs the global-extrema pre-pass, then ``:237-243``
    submits every orbit twice (without and with the extrema) to ``FAST_process_single_orbit``,
    which draws {given, raw} pitch-angle grids per instrument and {given, raw} instrument grids
    (``fast/process_orbit.py:148-253``).  Here the whole shard goes through K1 -> K2b -> K2a ->
    K3 as a handful of launches.  The panel tables are planned once from metadata (times,
    energies, pitch angles, cusp rows); the z bounds that depend on this step's extrema live in
    the batch's slot table, so a step re-plans only if the extrema change the *geometry*
    (y bounds / missing keys).
    """

    def __init__(self, shard: ShardPlan, sequence, max_percentile=95.0, comm=None, lut259=None, want_index=False,
                 compute_mins=False, plot_orbits=None, submissions=(False, True)):
        """``plot_orbits``: orbit numbers to draw (default: every orbit of the shard; the extrema
        pre-pass always covers the whole sequence).  ``submissions``: which of the reference's two
        submissions per orbit to plan -- without / with the global extrema."""
        self.plot_orbits = None if plot_orbits is None else set(plot_orbits)
        self.submissions = tuple(submissions)
        self.shard = shard
        self.sequence = sequence
        self.max_percentile = max_percentile
        self.comm = comm
        self.want_index = want_index
        self.compute_mins = compute_mins
        self.lut = lut259
        self._sig = None
        self._slots: dict = {}
        self._win_pin = None
        self.state: dict | None = None

    # -- what of the extrema state shapes the plan (everything else flows through z slots)
    def _bounds(self, state):
        from .extrema import _extrema_overrides

        sh = self.shard
        out = {}
        for inst in dict.fromkeys(tuple(sh.instrument_order) + tuple(DEFAULT_INSTRUMENT_ORDER)):
            stem = f"{inst}_{sh.y_scale}_{sh.z_scale}"
            ov = _extrema_overrides(state, inst, sh.y_scale, sh.z_scale)
            raw = tuple(state.get(f"{stem}_{k}") for k in ("y_min", "y_max", "z_min", "z_max"))
            out[inst] = (ov, raw)
        return out

    @staticmethod
    def _signature(bounds):
        return tuple(
            (inst, ov[0], ov[1], ov[2] is None, ov[3] is None, raw[0], raw[1], raw[2] is None, raw[3] is None)
            for inst, (ov, raw) in bounds.items()
        )

    def _plan(self, state, bounds):
        sh, b = self.shard, self.shard.batch
        sh.reset_plan()
        self._slots = {}
        slotted = dict(state)
        given = {}
        for inst, (ov, raw) in bounds.items():
            stem = f"{inst}_{sh.y_scale}_{sh.z_scale}"
            zr = []
            for name, v in (("zr_min", ov[2]), ("zr_max", ov[3])):
                if v is None:
                    zr.append(None)
                else:
                    zr.append(b.zslot(v))
                    self._slots[(inst, name)] = zr[-1]
            given[inst] = (ov[0], ov[1], zr[0], zr[1])
            for name, key, v in (("z_min", f"{stem}_z_min", raw[2]), ("z_max", f"{stem}_z_max", raw[3])):
                if v is not None:
                    slotted[key] = self._slots[(inst, name)] = b.zslot(v)
        self.figure_ranges = {}  # (orbit, with_extrema) -> [first, last) in shard.figures
        for ob in sh.orbits:
            if self.plot_orbits is not None and ob["orbit"] not in self.plot_orbits:
                continue
            for with_extrema in self.submissions:  # batch_directory.py:237-243
                first = len(sh.figures)
                for inst in DEFAULT_INSTRUMENT_ORDER:  # process_orbit.py:124 walks the default order
                    if inst not in ob["files"]:
                        continue
                    if with_extrema:
                        sh.plan_pitch_angle_grid(ob, inst, "given", *given[inst])
                    else:
                        sh.plan_pitch_angle_grid(ob, inst, "given")
                    sh.plan_pitch_angle_grid(ob, inst, "raw")
                sh.plan_instrument_grid(ob, "given", global_extrema=slotted if with_extrema else None)
                sh.plan_instrument_grid(ob, "raw", global_extrema=None)
                self.figure_ranges[(ob["orbit"], with_extrema)] = (first, len(sh.figures))
        sh.upload_tables()
        if self.lut is not None:
            b.set_lut(self.lut)
        self._win_pin = b.ctx.pinned(max(b.n_windows, 1))

    def _update_slots(self, bounds):
        b = self.shard.batch
        for inst, (ov, raw) in bounds.items():
            for name, v in (("zr_min", ov[2]), ("zr_max", ov[3]), ("z_min", raw[2]), ("z_max", raw[3])):
                slot = self._slots.get((inst, name))
                if slot is not None:
                    b.set_zslot(slot.slot, v)

    def run(self, cache_state: dict | None = None, state: dict | None = None, collapse: bool = True) -> dict:
        """Enqueue one whole step; returns the extrema state (rasters stay on the device).

        ``state``: an already computed extrema dict (e.g. from ``compute_global_extrema`` with its
        JSON cache) -- the K2b pre-pass is skipped and only the figures run."""
        from .extrema import extrema_enqueue, extrema_finish

        sh, b = self.shard, self.shard.batch
        planned = self._sig is not None
        want_rgba = b.d_lut is not None
        early = False
        if collapse:
            sh.collapse()

        def independent_stages():
            # nothing here depends on this step's extrema: K2a for every region, and K3 for the
            # panels that read no z slot (the raw variants) -- the GPU stays busy while the host
            # turns the pooled results into bounds
            b.run_windows()
            b.run_stats()
            b.prepare(part=0)
            # with several ranks the digit loop and its peer exchanges are still running on the side stream
            # at this point, and K3's persistent blocks would fill every SM to the last register: leave room
            # (measured at 8 GPUs: the loop's next kernel waited 190-360 us for K3 to END)
            share = self.comm is not None and state is None and planned
            if share:
                b.ctx._check(b.ctx.lib.csg_rasterise_blocks_per_sm(b.ctx.handle, _k3_shared_blocks()))
            try:
                b.rasterise(want_rgba=want_rgba, want_index=self.want_index, part=0)
            finally:
                if share:
                    b.ctx._check(b.ctx.lib.csg_rasterise_blocks_per_sm(b.ctx.handle, 0))

        if state is None:
            pending = extrema_enqueue(sh, self.sequence, sh.instrument_order, sh.y_scale, sh.z_scale,
                                      dict(cache_state or {}), compute_mins=self.compute_mins,
                                      max_percentile=self.max_percentile, comm=self.comm, per_step=False,
                                      overlap=planned)
            if planned:
                independent_stages()
                early = True
            state = extrema_finish(pending)
        elif planned:
            independent_stages()
            early = True
        bounds = self._bounds(state)
        sig = self._signature(bounds)
        if sig != self._sig:
            self._plan(state, bounds)
            self._sig = sig
            b.run_windows()
            b.run_stats()
            early = False
        else:
            self._update_slots(bounds)
        want_rgba = b.d_lut is not None
        if early:
            b.prepare(part=1)
            b.rasterise(want_rgba=want_rgba, want_index=self.want_index, part=1)
        else:
            b.prepare()
            b.rasterise(want_rgba=want_rgba, want_index=self.want_index)
        if b.n_windows:
            b.ctx._check(b.ctx.lib.csg_d2h(b.ctx.handle, self._win_pin.ptr, b.d_window_any.ptr, b.n_windows))
        self.state = state
        return state

    def finish(self):
        """Wait for the step and fill the figures' ``zoom_needed`` flags."""
        b = self.shard.batch
        b.ctx.sync()
        if b.n_windows:
            self.shard.resolve_zoom_flags(self._win_pin.view(np.uint8, b.n_windows))
        return self.state


def _k3_shared_blocks() -> int:
    """K3 blocks per SM while the extrema chain runs beside it (``CSG_K3_SHARED_BLOCKS``, default 2; 0 = no cap)."""
    try:
        return max(0, int(os.environ.get("CSG_K3_SHARED_BLOCKS", "2")))
    except ValueError:
        return 2


def check_norm_status(norm_row, what: str | None = None):
    """Raise what matplotlib would raise at draw time for an invalid panel normalisation; ``what`` names
    the panel and adds its bounds to the message."""
    st = int(norm_row["status"])
    if st == _lib.NORM_VMIN_GT_VMAX:
        msg = "vmin must be less or equal to vmax"
    elif st == _lib.NORM_INVALID:
        msg = "Invalid vmin or vmax"
    else:
        return
    if what is not None:
        msg += f" ({what}: vmin={norm_row['vmin']}, vmax={norm_row['vmax']})"
    raise ValueError(msg)
