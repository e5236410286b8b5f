"""Batch driver: every orbit of a directory through the GPU path (reference ``fast/batch_directory.py``).

Same signature, progress-JSON schema, output tree and return value as the reference's
``FAST_plot_spectrograms_directory``.  What changes is the execution model: the reference fans
orbits out to a ``ProcessPoolExecutor`` (one orbit per task, ten figures each re-loading and
re-collapsing the files); here the orbits of this rank are ONE shard resident in HBM:

  K1  every cube collapsed once (all pitch-angle groups + total + zoom flags)
  K2b the global-extrema pre-pass from the same collapsed matrices (``compute_global_extrema``
      with its resumable JSON cache; NCCL exchange when several ranks share the directory)
  K2a 1st / 99th percentiles and safe_vmin of every panel of every figure, one launch
  K3  every panel rasterised, one launch

after which host threads compose the figures (labels, ticks, cusp markers) and DEFLATE the
PNGs.  ``max_workers`` sizes that thread pool.  Multi-GPU: launch one process per GPU with
``torchrun`` -- ranks take contiguous blocks of the ascending orbit sequence.
"""

from __future__ import annotations

import json
import os
import signal
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass
from typing import Any

from .. import _lib
from ..cdf_utils import get_cdf_file_type, get_timestamps_for_orbit, load_fast_cdf_dataset, load_filtered_orbits
from ..colormaps import get_lut
from ..comm import block_of, current_device, rank_world
from ..constants import DEFAULT_ZOOM_WINDOW_MINUTES
from ..figure import close_all_axes_and_clear
from ..logging_utils import configure_log_batch, flush_log_buffer, log_exception
from .constants import DEFAULT_INSTRUMENT_ORDER, FAST_CDF_DATA_FOLDER_PATH, FAST_OUTPUT_BASE, FAST_PLOTTING_PROGRESS_JSON
from .extrema import compute_global_extrema
from .orbit_discovery import _add_to_orbit_list, _classify_error_reason, _parse_year_month, discover_orbit_files
from .pipeline import BatchStep, ShardPlan, chunk_orbits, ingest_orbits
from .plotting import figure_from_spec
from .process_orbit import SAVE_DPI, figure_filename

_INSTRUMENT_KEYS = DEFAULT_INSTRUMENT_ORDER

__all__ = ["FAST_plot_spectrograms_directory"]


def FAST_plot_spectrograms_directory(
    directory_path: str = FAST_CDF_DATA_FOLDER_PATH,
    output_base: str = FAST_OUTPUT_BASE,
    y_scale: str = "linear",
    z_scale: str = "log",
    zoom_duration_minutes: float = DEFAULT_ZOOM_WINDOW_MINUTES,
    instrument_order: tuple[str, ...] = _INSTRUMENT_KEYS,
    verbose: bool = True,
    progress_json_path: str | None = FAST_PLOTTING_PROGRESS_JSON,
    ignore_progress_json: bool = False,
    use_tqdm: bool | None = None,
    colormap: str = "viridis",
    cusp_marker_style: str = "both",
    cusp_marker_kwargs: dict | None = None,
    max_workers: int = 4,
    orbit_timeout_seconds: int | float = 60,
    instrument_timeout_seconds: int | float = 30,
    retry_timeouts: bool = True,
    flush_batch_size: int = 10,
    log_flush_batch_size: int | None = None,
    max_processing_percentile: float | None = None,
    override_plots: bool = True,
    _timings: dict | None = None,
) -> list[dict[str, Any]]:
    """Plot every orbit under ``directory_path`` (reference ``:32-433``).

    Returns one result dict per submission (``{"orbit", "status", "errors"}``); like the
    reference every orbit is submitted twice when ``max_processing_percentile`` is given (once
    without, once with the global extrema, ``:237-243``).  Progress keys:
    ``{y}_{z}_last_orbit``, ``{y}_{z}_error_plotting``, ``orbit_{y}_{z}_timed_out`` and the
    per-reason error lists (``:277-321``).  Raises ``KeyboardInterrupt`` on SIGINT / SIGTERM.

    Timeouts keep the reference's soft, after-the-fact semantics (``process_orbit.py:203-211,276-283``): a
    chunk of orbits is planned, rasterised, encoded and written together, its wall time is shared evenly
    between its submissions, and a share above ``orbit_timeout_seconds`` marks them ``"timeout"``
    (``timeout_type: "orbit"``, listed under ``orbit_{y}_{z}_timed_out``).  With ``retry_timeouts`` every
    timed-out orbit is re-run once through ``FAST_process_single_orbit`` without global extrema
    (``instrument_timeout_seconds`` applies there) and cleared from the lists when it succeeds
    (``:422-431,455-514``); retries run on single-GPU calls only.

    Memory: cubes stream through three pinned host slots and one device staging buffer
    (``CSG_CHUNK_ORBITS`` orbits at a time, default 8); only the collapsed sums (6 MB per orbit) stay in
    HBM for the whole call.  ``_timings`` (internal, bench): seconds per phase.
    """
    interrupted = {"flag": False}

    def _signal_handler(signum, frame):
        interrupted["flag"] = True
        log_exception(f"[INTERRUPT] Signal {signum} received. Requesting shutdown...", level="message")
        raise KeyboardInterrupt

    previous = {}
    try:
        for sig in (signal.SIGINT, signal.SIGTERM):
            previous[sig] = signal.signal(sig, _signal_handler)
    except (ValueError, OSError) as exc:
        log_exception("[WARN] Could not register signal handlers", exc, level="message")

    import time as _time

    t_call = _time.perf_counter()
    try:
        return _run_directory(
            directory_path, output_base, y_scale, z_scale, zoom_duration_minutes, tuple(instrument_order), verbose,
            progress_json_path, ignore_progress_json, colormap, cusp_marker_style, cusp_marker_kwargs, max_workers,
            flush_batch_size, log_flush_batch_size, max_processing_percentile, override_plots,
            orbit_timeout_seconds, instrument_timeout_seconds, retry_timeouts, _timings,
        )
    finally:
        if _timings is not None:  # what is left once the phases are subtracted: releasing the shard's buffers
            _timings["release"] = _time.perf_counter() - t_call - sum(v for k, v in _timings.items() if "/" not in k)
        for sig, handler in previous.items():
            try:
                signal.signal(sig, handler)
            except (ValueError, OSError):
                pass


@dataclass
class _Chunk:
    """A chunk's K4 state between its encode and its progress records."""

    encode: Any  # the open png.DeferredEncode of its last group, None once read back (or with nothing to draw)
    writes: list  # futures of the framing + writing of its files
    paths: list
    planned: list  # (result, saves) per submission
    n_jobs: int
    seconds: float  # wall time so far

    def read_back(self) -> None:
        """Wait for the encode kernel and hand the last group to the writers."""
        if self.encode is not None:
            self.writes, self.encode = self.encode.complete(), None


class _OpenEncode:
    """Leaves no deferred K4 encode open when the chunk loop is left by an exception (an interrupt): the next
    call in this process finds the encoder context free."""

    def __init__(self, current):
        self._current = current

    def __enter__(self):
        return self

    def __exit__(self, kind, _value, _trace):
        chunk = self._current()
        if kind is not None and chunk is not None and chunk.encode is not None:
            try:
                chunk.encode.abandon()
            except Exception:
                pass
        return False


def _render_threads(n_threads: int) -> int:
    """Threads that plan the figures of a chunk (``CSG_RENDER_THREADS``, default 1).  The planning is
    interpreter-bound, so threads only take turns and pay for it: 0.72-0.78 s per 1250 figures with 16 or 4
    threads, 0.61-0.66 s with one.  More can help where ``os.path.exists`` / ``makedirs`` are slow (network
    file systems)."""
    try:
        return max(1, min(int(os.environ.get("CSG_RENDER_THREADS", "1")), max(1, n_threads)))
    except ValueError:
        return 1


def _run_directory(directory_path, output_base, y_scale, z_scale, zoom_duration_minutes, instrument_order, verbose,
                   progress_json_path, ignore_progress_json, colormap, cusp_marker_style, cusp_marker_kwargs, max_workers,
                   flush_batch_size, log_flush_batch_size, max_processing_percentile, override_plots,
                   orbit_timeout_seconds=60, instrument_timeout_seconds=30, retry_timeouts=True, timings=None):
    import time as _time

    from .extrema import load_extrema_state, orbits_the_scan_needs

    def tick(name, t0):
        if timings is not None:
            timings[name] = timings.get(name, 0.0) + _time.perf_counter() - t0
        return _time.perf_counter()

    t_phase = _time.perf_counter()
    rank, world, dist = rank_world()
    frame = load_filtered_orbits()
    configure_log_batch(log_flush_batch_size or flush_batch_size)

    orbit_to_instruments = discover_orbit_files(directory_path, instrument_order)
    sorted_orbits = sorted(orbit_to_instruments.items(), key=lambda kv: kv[0])
    total_orbits = len(sorted_orbits)

    # ---- resume state (reference :173-213)
    progress_key = f"{y_scale}_{z_scale}_last_orbit"
    error_key = f"{y_scale}_{z_scale}_error_plotting"
    timeout_key = f"orbit_{y_scale}_{z_scale}_timed_out"
    progress: dict[str, Any] = {}
    last_completed, error_orbits = None, set()
    if progress_json_path is not None and not ignore_progress_json:
        try:
            with open(progress_json_path) as f:
                progress = json.load(f)
            last_completed = progress.get(progress_key)
            error_orbits = set(progress.get(error_key, []))
        except (OSError, json.JSONDecodeError) as exc:
            log_exception(f"[ERROR] Failed to load progress JSON from {progress_json_path}. Starting fresh.", exc, level="error")
            progress = {}
    start_idx = 0
    if last_completed is not None:
        start_idx = next((i for i, (o, _) in enumerate(sorted_orbits) if o > last_completed), total_orbits)
        log_exception(f"[RESUME] Skipping {start_idx} orbits (up to orbit {last_completed}). "
                      f"{len(error_orbits)} error orbits will also be skipped.", level="message")
    else:
        log_exception("[RESUME] No previous progress found. Starting from the first orbit. "
                      f"{len(error_orbits)} error orbits will be skipped if present.", level="message")
    pending = [o for o, _ in sorted_orbits[start_idx:] if o not in error_orbits]
    pending_set = set(pending)
    flush_batch_size = max(1, flush_batch_size)
    n_threads = max(1, int(max_workers))

    # ---- this rank's contiguous block of the ascending orbit sequence
    lo, hi = block_of(total_orbits, rank, world)
    comm = None
    if world > 1:
        import torch

        from ..comm import TorchComm

        comm = TorchComm(dist, torch.device("cuda", torch.cuda.current_device()))
    need_extrema = max_processing_percentile is not None
    sequence = [(o, {i: True for i in files}) for o, files in sorted_orbits]
    mine = sorted_orbits[lo:hi]
    # which cubes this rank has to read: every pending orbit it draws, and -- for the extrema pre-pass -- the
    # (orbit, instrument) steps that still reach the scan given the cached extrema JSON (a finished cache needs none)
    scan_needs: dict[int, set] = {}
    if need_extrema:
        scan_needs = orbits_the_scan_needs(sequence, instrument_order, y_scale, z_scale, load_extrema_state())
    results: list[dict[str, Any]] = []
    ctx = _lib.default_context(current_device())
    shard = ShardPlan(ctx, y_scale, z_scale, zoom_duration_minutes, instrument_order=instrument_order)
    shard.first_orbit_index = lo
    load_errors: dict[int, list[str]] = {}

    # ---- phase A: streaming ingest (pipeline.ingest_orbits): loader threads decode the next chunk's files
    # into a pinned staging slot while the previous chunk is uploaded and collapsed; the sums and row flags of
    # every orbit stay in HBM
    def load_one(index, alloc):
        orbit, files = mine[index]
        wanted = set(scan_needs.get(lo + index, ()))
        if orbit in pending_set:
            wanted |= set(instrument_order)
        datasets, lines, errors = {}, {}, []
        for inst in DEFAULT_INSTRUMENT_ORDER:
            path = files.get(inst)
            if not path or inst not in instrument_order or inst not in wanted:
                continue
            try:
                detected = get_cdf_file_type(path)
                if detected is None or detected == "orb":
                    continue
                ds = load_fast_cdf_dataset(path, data_alloc=alloc)
                datasets[inst] = ds
                lines[inst] = get_timestamps_for_orbit(frame, orbit, detected, ds["times"])
            except Exception as exc:
                err = f"[FAIL] Plotting Orbit {orbit} pitch angle grid for {inst}"
                log_exception(err, exc, level="error")
                errors.append(err)
        if errors:
            load_errors[orbit] = errors
        return orbit, datasets, lines

    def refused(orbit, exc):  # a cube of another float dtype than the shard's: refused, not cast
        err = f"[FAIL] Orbit {orbit} processing"
        log_exception(err, exc, level="error")
        load_errors.setdefault(orbit, []).append(err)

    t_phase = tick("discover_and_resume", t_phase)
    ingest_orbits(shard, range(len(mine)), load_one, refused, n_threads=n_threads)
    if world > 1:
        shard.agree_dtype(dist, world)
    if not mine:  # such a rank still joins the extrema exchange, with empty outputs of K1
        shard.collapse_pending()
    # ranks that loaded only part of the sequence still index it globally
    if not need_extrema:
        shard.first_orbit_index = 0
    t_phase = tick("ingest_and_collapse", t_phase)

    # ---- phase B: global extrema pre-pass (reference :159-171), from the collapsed matrices already in HBM
    global_extrema = None
    if need_extrema:
        global_extrema = compute_global_extrema(
            directory_path, y_scale, z_scale, instrument_order, compute_mins=False,
            max_percentile=float(max_processing_percentile), log_floor_cutoff=0.1, log_floor_value=-1.0,
            flush_batch_size=flush_batch_size, _shard=shard, _comm=comm,
        )
    t_phase = tick("global_extrema", t_phase)

    # ---- phase C: the figures, chunk by chunk: K2a + K3 for the chunk's panels, the figures planned on host
    # threads from panel references, composed and PNG-encoded on the device (K4: no raster ever crosses PCIe
    # uncompressed), files written, progress recorded -- an interrupt loses at most the chunk in flight
    loaded_set = {orbit for orbit, _files in mine}
    my_pending = [o for o in pending if o in loaded_set]
    chunk_n = chunk_orbits()
    submissions = (False, True) if need_extrema else (False,)
    lut = get_lut(colormap)
    b = shard.batch
    pdisk = dict(progress)
    since_flush = 0

    def record(result, pdisk):
        orbit = result["orbit"]
        pdisk[progress_key] = orbit
        pdisk.setdefault(error_key, [])
        pdisk.setdefault(timeout_key, [])
        status = result.get("status")
        if status == "error":
            _add_to_orbit_list(pdisk, error_key, orbit)
            for msg in result.get("errors") or []:
                reason = _classify_error_reason(msg)
                inst = next((c for c in _INSTRUMENT_KEYS if c in msg.lower()), "unknown")
                _add_to_orbit_list(pdisk, f"{inst}_{y_scale}_{z_scale}_error-{reason}", orbit)
                _add_to_orbit_list(pdisk, f"{y_scale}_{z_scale}_error-{reason}", orbit)
        elif status == "timeout":  # reference :316-324
            if result.get("timeout_type") == "orbit":
                _add_to_orbit_list(pdisk, timeout_key, orbit)
            elif result.get("timeout_type") == "instrument":
                inst = result.get("timeout_instrument") or "unknown_instrument"
                _add_to_orbit_list(pdisk, f"{inst}_{y_scale}_{z_scale}_timed_out", orbit)

    from ..png import write_figures_device

    png_timings: dict | None = {} if timings is not None else None
    code_cache: dict = {}  # the DEFLATE code fitted to the first chunk's figures serves the whole run
    # K4 runs on a companion context (its own stream): chunk k's encode kernel works while the host plans chunk
    # k + 1 and its K2a / K3 run on the main stream -- into the OTHER of two raster buffers, the one chunk k - 1's
    # encode has long finished with.  A chunk passes through three states: `encoding` (kernel launched),
    # `writing` (compressed bytes read back, native threads framing and writing), settled (progress recorded).
    encoder_ctx = ctx.background_context()  # least urgent stream: K2a / K3 of the next chunk overtake the encoder
    raster_buffers: list = [None, None]
    encoding = writing = None
    n_chunk = 0

    def settle(chunk: _Chunk, since_flush):
        """The host half of a chunk ends here: its PNG files are on disk (the framing and writing ran on the
        encoder's finisher thread while the next chunk was ingested and planned), then the soft timeouts and
        the progress records -- in that order, so that progress never names an orbit whose files are missing."""
        t_wait = _time.perf_counter()
        for fut in chunk.writes:
            fut.result()
        seconds = chunk.seconds + _time.perf_counter() - t_wait
        for path in chunk.paths:
            log_exception(f"[SAVED] {path}", level="message")
        # soft timeouts, checked after the work like the reference's (process_orbit.py:203-211,276-283): a
        # chunk's wall time is shared evenly between its submissions
        share = seconds / max(1, chunk.n_jobs)
        for result, _s in chunk.planned:
            if share > orbit_timeout_seconds and result["status"] == "ok":
                log_exception(f"[TIMEOUT] Orbit {result['orbit']} exceeded {orbit_timeout_seconds:.0f}s total.", level="message")
                result["status"], result["timeout_type"] = "timeout", "orbit"
            results.append(result)
            if verbose:
                log_exception(f"[BATCH] Completed orbit {result['orbit']}: {result['status']}", level="message")
            if progress_json_path is not None and rank == 0:
                record(result, pdisk)
                since_flush += 1
                if since_flush >= flush_batch_size:
                    _write_json(progress_json_path, pdisk)
                    since_flush = 0
        return since_flush

    with ThreadPoolExecutor(max_workers=_render_threads(n_threads)) as pool, _OpenEncode(lambda: encoding):
        for a in range(0, len(my_pending), chunk_n):
            chunk = my_pending[a : a + chunk_n]
            t_chunk = _time.perf_counter()
            step = BatchStep(shard, sequence, comm=comm, lut259=lut, plot_orbits=chunk, submissions=submissions)
            b.d_rgba = raster_buffers[n_chunk & 1]  # not the buffer the previous chunk's encode kernel is reading
            step.run(state=global_extrema if global_extrema is not None else {}, collapse=False)
            t_phase = tick("plan_and_enqueue", t_phase)
            step.finish()
            raster_buffers[n_chunk & 1] = b.d_rgba
            n_chunk += 1
            norms = b.norms() if b.n_panels else None
            t_phase = tick("kernels_wait", t_phase)

            def render(job, step=step, norms=norms):
                """One submission of one orbit (= one FAST_process_single_orbit call of the reference)."""
                orbit, with_extrema = job
                result: dict[str, Any] = {"orbit": orbit, "status": "ok", "errors": []}
                saves: list[tuple[str, Any]] = []  # (path, figure): encoded and written after the planning pass
                for err in load_errors.get(orbit, []):
                    result["status"] = "error"
                    result["errors"].append(err)
                files = orbit_to_instruments[orbit]
                first_path = next((files[k] for k in DEFAULT_INSTRUMENT_ORDER if k in files), None)
                year, month = _parse_year_month(first_path) if first_path else ("unknown", "unknown")
                out_dir = os.path.join(output_base, str(year), str(month), str(orbit))
                os.makedirs(out_dir, exist_ok=True)
                first, last = step.figure_ranges.get((orbit, with_extrema), (0, 0))
                for spec in shard.figures[first:last]:
                    what = f"pitch angle grid for {spec.instrument}" if spec.kind == "pitch-angle" else "instrument grid"
                    try:
                        fig, _canvas = figure_from_spec(shard, spec, colormap, cusp_marker_style, cusp_marker_kwargs, norms=norms,
                                                        device_rasters=True)
                        if fig is None:
                            continue
                        path = os.path.join(out_dir, figure_filename(spec, y_scale, z_scale, colormap))
                        if not override_plots and os.path.exists(path):
                            log_exception(f"[SKIP] Plot already exists, skipping: {path}", level="message")
                            close_all_axes_and_clear(fig)
                        else:
                            saves.append((path, fig))
                    except Exception as exc:
                        err = f"[FAIL] Plotting Orbit {orbit} {what}"
                        log_exception(err, exc, level="error")
                        result["status"] = "error"
                        if err not in result["errors"]:
                            result["errors"].append(err)
                return result, saves

            jobs = [(o, flag) for o in chunk for flag in submissions]
            planned = list(pool.map(render, jobs))
            # the reference runs the submissions one after the other: a later one finds the earlier one's file
            # and skips it unless override_plots is set, in which case the later one wins
            by_path: dict[str, Any] = {}
            for _r, job_saves in planned:
                for path, fig in job_saves:
                    if path in by_path and not override_plots:
                        log_exception(f"[SKIP] Plot already exists, skipping: {path}", level="message")
                        close_all_axes_and_clear(fig)
                        continue
                    if path in by_path:
                        close_all_axes_and_clear(by_path[path])
                    by_path[path] = fig
            saves = list(by_path.items())
            t_phase = tick("figures_host", t_phase)
            if writing is not None:  # the chunk before last: its files were written while two chunks were planned
                since_flush = settle(writing, since_flush)
                writing = None
                t_phase = tick("png_wait_previous_chunk", t_phase)
            if encoding is not None:  # the last chunk: its kernel ran while this one was planned
                encoding.read_back()
                writing, encoding = encoding, None
                t_phase = tick("png_read_back", t_phase)
            handle = None  # nothing to draw: the chunk still takes its turn, so that progress is recorded in orbit order
            if saves:
                encoder_ctx.wait_for(ctx)  # (the rasters are complete: step.finish() above; ordering kept explicit)
                handle = write_figures_device(encoder_ctx, b.d_rgba.ptr, saves, max_workers=n_threads, dpi=SAVE_DPI,
                                              timings=png_timings, defer=True, code_cache=code_cache, max_segments=1_000_000)
                for _path, fig in saves:
                    close_all_axes_and_clear(fig)
            encoding = _Chunk(handle, [], [path for path, _f in saves], planned, len(jobs), _time.perf_counter() - t_chunk)
            t_phase = tick("png_encode", t_phase)
        for state in (writing, encoding):  # oldest first: progress is recorded in orbit order
            if state is not None:
                state.read_back()
                since_flush = settle(state, since_flush)
        t_phase = tick("png_wait_last_chunk", t_phase)

    if world > 1:  # every rank returns every result; rank 0 owns the progress file
        gathered: list = [None] * world
        dist.all_gather_object(gathered, results)
        results = [r for part in gathered for r in part]
        if rank == 0 and progress_json_path is not None:
            pdisk = dict(progress)
            for r in sorted(results, key=lambda r: r["orbit"]):
                record(r, pdisk)
    if progress_json_path is not None and rank == 0 and (results or os.path.exists(progress_json_path)):
        _write_json(progress_json_path, pdisk)
    flush_log_buffer(force=True)
    if retry_timeouts and world == 1:
        results = _retry_timed_out_orbits(results, orbit_to_instruments, frame, zoom_duration_minutes, y_scale, z_scale,
                                          instrument_order, colormap, output_base, orbit_timeout_seconds,
                                          instrument_timeout_seconds, override_plots, cusp_marker_style, cusp_marker_kwargs,
                                          progress_json_path)
    tick("finish", t_phase)
    if timings is not None:
        timings.update({f"png/{k}": v for k, v in (png_timings or {}).items()})
    return results


def _retry_timed_out_orbits(results, orbit_to_instruments, frame, zoom_duration_minutes, y_scale, z_scale, instrument_order,
                            colormap, output_base, orbit_timeout_seconds, instrument_timeout_seconds, override_plots,
                            cusp_marker_style, cusp_marker_kwargs, progress_json_path):
    """Every orbit whose status is ``'timeout'`` once more, one orbit at a time through
    ``FAST_process_single_orbit`` without global extrema -- the reference's retry pool (``:455-492``:
    ``orbit_args_fn(o, files, None)``).  Like there, the results collapse to one entry per orbit when
    anything was retried, and a successful retry clears the orbit from every ``*_timed_out`` list."""
    from .process_orbit import FAST_process_single_orbit

    timed_out = sorted({r["orbit"] for r in results if r.get("status") == "timeout"})
    if not timed_out:
        return results
    log_exception(f"[RETRY] Retrying {len(timed_out)} timed-out orbits once.", level="message")
    retried = []
    for orbit in timed_out:
        if orbit not in orbit_to_instruments:
            continue
        try:
            r = FAST_process_single_orbit(
                orbit, orbit_to_instruments[orbit], frame, zoom_duration_minutes, y_scale, z_scale, instrument_order, colormap,
                output_base, orbit_timeout_seconds=orbit_timeout_seconds, instrument_timeout_seconds=instrument_timeout_seconds,
                global_extrema=None, override_plots=override_plots, cusp_marker_style=cusp_marker_style,
                cusp_marker_kwargs=cusp_marker_kwargs,
            )
            log_exception(f"[RETRY] Completed orbit {orbit}: {r.get('status')}", level="message")
            if progress_json_path is not None and r.get("status") == "ok":
                _clear_timeout_flag(progress_json_path, orbit, y_scale, z_scale)
        except Exception as exc:
            log_exception(f"[RETRY] Orbit {orbit} retry failed", exc, level="error")
            r = {"orbit": orbit, "status": "error", "errors": [str(exc)]}
        retried.append(r)
    merged = {r["orbit"]: r for r in results}
    for r in retried:
        merged[r["orbit"]] = r
    return list(merged.values())


def _clear_timeout_flag(progress_json_path, orbit, y_scale, z_scale):
    """Remove ``orbit`` from every ``*_timed_out`` list of the progress JSON (reference ``:495-514``)."""
    try:
        with open(progress_json_path) as f:
            pdisk = json.load(f)
    except (OSError, json.JSONDecodeError) as exc:
        log_exception("[WARN] Could not read progress JSON for retry cleanup", exc, level="message")
        return
    changed = False
    for key in [k for k in pdisk if k.endswith(f"_{y_scale}_{z_scale}_timed_out")]:
        if isinstance(pdisk.get(key), list) and orbit in pdisk[key]:
            pdisk[key] = [x for x in pdisk[key] if x != orbit]
            changed = True
    if changed:
        _write_json(progress_json_path, pdisk)


def _write_json(path, data):
    try:
        with open(path, "w") as f:
            json.dump(data, f, indent=2)
    except OSError as exc:
        log_exception("[ERROR] Failed to write progress JSON", exc, level="error")
