"""Process and save every ESA figure of one orbit (reference ``fast/process_orbit.py``).

Same signature, file names and return dict as the reference's ``FAST_process_single_orbit``.
The reference renders ten figures through ten independent loads and collapses of the same
files; here the orbit's files are loaded and collapsed ONCE (K1, every pitch-angle group in one
pass), all panels of all ten figures go through one percentile launch and one raster launch,
and the figures are composed and PNG-encoded from the finished rasters.
"""

from __future__ import annotations

import gc
import os
import time as _time
from typing import Any

from .. import _lib
from ..cdf_utils import get_cdf_file_type, get_timestamps_for_orbit, load_fast_cdf_dataset
from ..colormaps import get_lut
from ..figure import close_all_axes_and_clear
from ..logging_utils import log_exception
from .constants import DEFAULT_INSTRUMENT_ORDER
from .extrema import _extrema_overrides
from .orbit_discovery import _parse_year_month
from .pipeline import FigureSpec, ShardPlan
from ..png import write_figures_device
from .plotting import figure_from_spec

__all__ = ["FAST_process_single_orbit", "figure_filename", "plan_orbit_figures", "SAVE_DPI"]

#: ``fig.savefig(out_path, dpi=200)`` (reference ``:110``): a 24 x 12 in grid becomes 4800 x 2400 pixels
SAVE_DPI = 200


def figure_filename(spec: FigureSpec, y_scale: str, z_scale: str, colormap: str) -> str:
    """The PNG name the reference gives this figure (``:165-168,186-189,231-234,252``)."""
    tail = "given_extrema" if spec.variant == "given" else "raw"
    if spec.kind == "pitch-angle":
        cusp_tag = "_cusp" if spec.vertical_lines else ""
        return f"{spec.orbit}{cusp_tag}_pitch-angle_ESA_{spec.instrument}_y-{y_scale}_z-{z_scale}_{tail}-{colormap}.png"
    return f"{spec.orbit}_instrument-grid_ESA_y-{y_scale}_z-{z_scale}_{tail}-{colormap}.png"


def plan_orbit_figures(shard: ShardPlan, orbit_entry: dict, global_extrema) -> list[FigureSpec]:
    """The figures of one ``FAST_process_single_orbit`` submission, in the reference's order:
    per instrument {given, raw} pitch-angle grids (``:124-190``), then {given, raw} instrument
    grids (``:212-253``)."""
    specs = []
    for inst in DEFAULT_INSTRUMENT_ORDER:
        if inst not in orbit_entry["files"]:
            continue
        ov = _extrema_overrides(global_extrema, inst, shard.y_scale, shard.z_scale)
        specs.append(shard.plan_pitch_angle_grid(orbit_entry, inst, "given", *ov))
        specs.append(shard.plan_pitch_angle_grid(orbit_entry, inst, "raw"))
    specs.append(shard.plan_instrument_grid(orbit_entry, "given", global_extrema=global_extrema))
    specs.append(shard.plan_instrument_grid(orbit_entry, "raw", global_extrema=None))
    return specs


def FAST_process_single_orbit(
    orbit_number: int,
    instrument_file_paths: dict[str, str],
    filtered_orbits_dataframe,
    zoom_duration_minutes: float,
    y_axis_scale: str,
    z_axis_scale: str,
    instrument_order: tuple[str, ...],
    colormap: str,
    output_base_directory: str,
    orbit_timeout_seconds: int | float = 60,
    instrument_timeout_seconds: int | float = 30,
    global_extrema: dict[str, int | float] | None = None,
    override_plots: bool = True,
    cusp_marker_style: str = "both",
    cusp_marker_kwargs: dict | None = None,
) -> dict[str, Any]:
    """Render and save all ESA spectrogram plots of one orbit.

    Returns ``{"orbit", "status" ('ok' | 'error' | 'timeout'), "errors"[, "timeout_type",
    "timeout_instrument"]}`` (reference ``:92,285-290``).  Timeouts are the reference's soft
    wall-clock checks (``:197-209,262-283``).
    """
    result: dict[str, Any] = {"orbit": orbit_number, "status": "ok", "errors": []}
    orbit_start = _time.time()
    timeout_type = timeout_instrument = None

    def save(fig, out_path, desc, ctx, d_rgba_ptr):
        """The panels are still in HBM: the figure is composed at ``SAVE_DPI`` and DEFLATE-encoded on the device."""
        if not override_plots and os.path.exists(out_path):
            log_exception(f"[SKIP] Plot already exists, skipping: {out_path}", level="message")
            close_all_axes_and_clear(fig)
            return
        try:
            log_exception(f"[DEBUG] Saving {desc} plot: y_axis_scale={y_axis_scale}, z_axis_scale={z_axis_scale}, "
                          f"filename={out_path}", level="message")
            write_figures_device(ctx, d_rgba_ptr, [(out_path, fig)], max_workers=1, dpi=SAVE_DPI)
            log_exception(f"[SAVED] {out_path}", level="message")
        except Exception as exc:
            log_exception(f"[FAIL] Saving figure {out_path}", exc, level="error")
            result["status"] = "error"
            result["errors"].append(str(exc))
        finally:
            close_all_axes_and_clear(fig)

    try:
        first_path = next((instrument_file_paths[k] for k in DEFAULT_INSTRUMENT_ORDER if k in instrument_file_paths), None)
        year, month = _parse_year_month(first_path) if first_path else ("unknown", "unknown")
        output_dir = os.path.join(output_base_directory, str(year), str(month), str(orbit_number))
        os.makedirs(output_dir, exist_ok=True)

        # ---- load every instrument once (the reference reloads each file five times or more)
        datasets, lines = {}, {}
        for inst in DEFAULT_INSTRUMENT_ORDER:
            path = instrument_file_paths.get(inst)
            if not path:
                continue
            try:
                detected = get_cdf_file_type(path)
                if detected is None or detected == "orb":
                    continue
                ds = load_fast_cdf_dataset(path)
                datasets[inst] = ds
                lines[inst] = get_timestamps_for_orbit(filtered_orbits_dataframe, orbit_number, detected, ds["times"])
            except Exception as exc:
                err = f"[FAIL] Plotting Orbit {orbit_number} pitch angle grid for {inst}"
                log_exception(err, exc, level="error")
                result["status"] = "error"
                result["errors"].append(err)
        if datasets:
            # the shard computes in the files' own dtype (numpy's results depend on it); files of different
            # float dtypes in one orbit are refused by add_orbit -> "[FAIL] Orbit ... processing" below
            shard = ShardPlan(_lib.default_context(), y_axis_scale, z_axis_scale, zoom_duration_minutes,
                              instrument_order=tuple(instrument_order))
            shard.add_orbit(orbit_number, datasets, lines)
            shard.upload()
            shard.collapse()
            specs = plan_orbit_figures(shard, shard.orbits[0], global_extrema)
            shard.run_once(get_lut(colormap), want_index=False)
            b = shard.batch
            norms = b.norms()
            group_start, group_key = _time.time(), None
            for spec in specs:
                key = spec.instrument if spec.kind == "pitch-angle" else "instrument_grid"
                if key != group_key:
                    group_start, group_key = _time.time(), key
                what = (f"pitch angle grid for {spec.instrument}" if spec.kind == "pitch-angle" else "instrument grid")
                try:
                    fig, _canvas = figure_from_spec(shard, spec, colormap, cusp_marker_style, cusp_marker_kwargs, norms=norms,
                                                    device_rasters=True)
                    if fig is not None:
                        desc = (f"pitch-angle {spec.instrument}" if spec.kind == "pitch-angle" else "instrument-grid")
                        desc += " (given extrema)" if spec.variant == "given" else " (raw extrema)"
                        save(fig, os.path.join(output_dir, figure_filename(spec, y_axis_scale, z_axis_scale, colormap)), desc,
                             b.ctx, b.d_rgba.ptr)
                except Exception as exc:
                    err = f"[FAIL] Plotting Orbit {orbit_number} {what}"
                    log_exception(err, exc, level="error")
                    result["status"] = "error"
                    if err not in result["errors"]:
                        result["errors"].append(err)
                if _time.time() - group_start > instrument_timeout_seconds and timeout_type is None:
                    timeout_type, timeout_instrument = "instrument", key
                    log_exception(f"[TIMEOUT] {key} in orbit {orbit_number} exceeded {instrument_timeout_seconds:.0f}s. "
                                  "Aborting.", level="message")
                    break
        if _time.time() - orbit_start > orbit_timeout_seconds and timeout_type is None:
            timeout_type = "orbit"
            log_exception(f"[TIMEOUT] Orbit {orbit_number} exceeded {orbit_timeout_seconds:.0f}s total.", level="message")
        if timeout_type is not None:
            result["status"] = "timeout"
            result["timeout_type"] = timeout_type
            if timeout_instrument:
                result["timeout_instrument"] = timeout_instrument
            return result
    except Exception as exc:
        err = f"[FAIL] Orbit {orbit_number} processing"
        log_exception(err, exc, level="error")
        result["status"] = "error"
        result["errors"].append(err)
    finally:
        gc.collect()
    return result
