"""Single-output FAST ESA spectrogram rendering (reference ``fast/plotting.py``).

``FAST_plot_pitch_angle_grid`` and ``FAST_plot_instrument_grid`` keep the reference's
signatures.  Each call plans its panels with :class:`pipeline.ShardPlan` (the verbatim
restatement of the reference's masks and bound selection) and runs them as ONE collapse of the
file(s) -- every pitch-angle group in a single pass over the cube instead of the reference's
four gathers + twelve ``np.nansum`` -- one percentile launch and one raster launch.  The batch
driver (``fast/batch_directory.py``) uses the same planner for a whole shard of orbits.
"""

from __future__ import annotations

from typing import Any

import numpy as np

from .. import _lib
from ..cdf_utils import get_cdf_file_type, get_timestamps_for_orbit, load_fast_cdf_dataset
from ..colormaps import get_lut
from ..figure import DeviceRaster, FigureCanvas, SpectrogramFigure
from ..logging_utils import log_exception
from ..plotting import _finish_multirow, date2num, draw_panel
from .constants import DEFAULT_INSTRUMENT_ORDER, DEFAULT_PITCH_ANGLE_CATEGORIES
from .pipeline import FigureSpec, ShardPlan, check_norm_status

__all__ = ["FAST_plot_pitch_angle_grid", "FAST_plot_instrument_grid", "figure_from_spec"]


def figure_from_spec(shard: ShardPlan, spec: FigureSpec, colormap="viridis", cusp_marker_style="both",
                     cusp_marker_kwargs=None, norms=None, device_rasters=False):
    """Compose the figure ``generic_plot_multirow_optional_zoom`` would return for one planned
    figure (reference ``plotting.py:583-698``) from the shard's finished rasters.

    ``norms``: the batch's downloaded normalisations (``Batch.norms``), fetched when omitted; the
    rasters are downloaded per panel.  ``device_rasters``: the panels stay in HBM
    (``figure.DeviceRaster`` references into the batch's RGBA buffer) and the figure is meant for
    ``png.encode_figures_device``.  Raises the ``ValueError`` matplotlib would raise at draw time
    for an invalid normalisation.
    """
    if not spec.rows:
        return None, None
    b = shard.batch
    if norms is None:
        norms = b.norms()
    n_cols = 2 if (spec.zoom is not None and spec.zoom_needed) else 1
    n_rows = len(spec.rows)
    fig = SpectrogramFigure(figsize=(12 * n_cols, 3 * n_rows))
    canvas = FigureCanvas(fig)
    axes = np.empty((n_rows, n_cols), dtype=object)
    for i in range(n_rows):
        for j in range(n_cols):
            axes[i, j] = fig.add_subplot(n_rows, n_cols, i * n_cols + j + 1)

    def raster(pid):
        if device_rasters:
            return DeviceRaster(b.panel_offset(pid), *b.panel_shape(pid)), None
        return b.panel_rgba(pid), (b.panel_index(pid) if b.d_index is not None else None)

    log_scale = shard.z_scale == "log"
    for i, row in enumerate(spec.rows):
        for j, pid in enumerate((row.full_panel, row.zoom_panel)[:n_cols]):
            if pid is None:
                continue  # make_spectrogram returned (None, None): the subplot stays empty
            nm = norms[pid]
            check_norm_status(nm, f"orbit {spec.orbit} {spec.kind} {row.label}")
            rgba, index = raster(pid)
            # the axes only need the ends of the panel's time and energy ranges (extent, limits, markers)
            region = b.panel_region(pid)
            t_first, t_last = b.region_time_ends(region)
            e_index = b.region_energy_index(region)
            y_kept = row.energy[e_index[[0, -1]]] if len(e_index) > 2 else row.energy[e_index]
            if len(e_index) > 2:
                y_kept = _Ends(y_kept, len(e_index))
            x_plot = (date2num(float(row.times[t_first])), date2num(float(row.times[t_last])))
            ax = axes[i, j]
            if j == 1:
                centre, duration = spec.zoom
                ax.set_xlim(date2num(centre - duration / 2), date2num(centre + duration / 2))
            else:
                ax.set_xlim(x_plot[0], x_plot[-1])
            draw_panel(ax, rgba, index, float(nm["vmin"]), float(nm["vmax"]), log_scale, x_plot, y_kept,
                       y_axis_scale_function=shard.y_scale, colormap=colormap, vertical_lines_unix=spec.vertical_lines,
                       cusp_marker_style=cusp_marker_style, cusp_marker_kwargs=cusp_marker_kwargs)
    datasets = [{"x": r.times, "label": r.label} for r in spec.rows]
    _finish_multirow(fig, axes, datasets, spec.vertical_lines, spec.title)
    return fig, canvas


class _Ends:
    """First and last value of a long axis array that report the original length (``draw_panel`` looks at
    ``[0]``, ``[-1]`` and ``len``): a batch of thousands of figures does not slice every axis in full."""

    __slots__ = ("first", "last", "n")

    def __init__(self, pair, n):
        self.first, self.last, self.n = pair[0], pair[-1], n

    def __len__(self):
        return self.n

    def __getitem__(self, k):
        if k == 0:
            return self.first
        if k == -1:
            return self.last
        raise IndexError("only the ends of the axis are kept")


def _run_single(shard: ShardPlan, spec: FigureSpec, colormap, cusp_marker_style, cusp_marker_kwargs):
    if not spec.rows:
        return None, None
    shard.run_once(get_lut(colormap), want_index=True)
    return figure_from_spec(shard, spec, colormap, cusp_marker_style, cusp_marker_kwargs)


def FAST_plot_pitch_angle_grid(
    cdf_file_path: str,
    filtered_orbits_df=None,
    orbit_number: int | None = None,
    zoom_duration_minutes: float = 6.25,
    scale_function_y: str = "linear",
    scale_function_z: str = "linear",
    pitch_angle_categories: dict[str, list[tuple[float, float]]] | None = None,
    show: bool = True,
    colormap: str = "viridis",
    y_min: float | None = None,
    y_max: float | None = None,
    z_min: float | None = None,
    z_max: float | None = None,
    cusp_marker_style: str = "both",
    cusp_marker_kwargs: dict | None = None,
) -> tuple[Any, Any]:
    """A grid of ESA spectrograms, one row per pitch-angle category, with a zoom column when the
    orbit has cusp boundary timestamps and the window holds data (reference ``:34-174``).
    Returns ``(fig, canvas)`` or ``(None, None)`` when no category yields a dataset."""
    if pitch_angle_categories is None:
        pitch_angle_categories = DEFAULT_PITCH_ANGLE_CATEGORIES
    instrument_type = get_cdf_file_type(cdf_file_path)
    dataset = load_fast_cdf_dataset(cdf_file_path)
    vertical_lines = None
    if filtered_orbits_df is not None and orbit_number is not None:
        vertical_lines = get_timestamps_for_orbit(filtered_orbits_df, orbit_number, instrument_type, dataset["times"])
        if not vertical_lines:
            log_exception(f"No vertical lines found for orbit {orbit_number} in {cdf_file_path}. Skipping.", level="message")
    key = instrument_type or "unknown"
    shard = ShardPlan(_lib.default_context(), scale_function_y, scale_function_z, zoom_duration_minutes,
                      instrument_order=(key,), pitch_angle_categories=pitch_angle_categories)
    shard.add_orbit(orbit_number, {key: dataset}, {key: vertical_lines})
    shard.upload()
    shard.collapse()
    spec = shard.plan_pitch_angle_grid(shard.orbits[0], key, "given", y_min, y_max, z_min, z_max)
    spec.title = f"Orbit {orbit_number} - Pitch Angle {instrument_type} ESA Spectrograms"
    if not spec.rows:
        log_exception(f"[WARNING] No pitch angle datasets to plot for {cdf_file_path}.", level="message")
        return None, None
    return _run_single(shard, spec, colormap, cusp_marker_style, cusp_marker_kwargs)


def FAST_plot_instrument_grid(
    cdf_file_paths: dict[str, str],
    filtered_orbits_df=None,
    orbit_number: int | None = None,
    zoom_duration_minutes: float = 6.25,
    scale_function_y: str = "linear",
    scale_function_z: str = "linear",
    instrument_order: tuple[str, ...] = DEFAULT_INSTRUMENT_ORDER,
    show: bool = True,
    colormap: str = "viridis",
    y_min: float | None = None,
    y_max: float | None = None,
    z_min: float | None = None,
    z_max: float | None = None,
    global_extrema: dict[str, int | float] | None = None,
    cusp_marker_style: str = "both",
    cusp_marker_kwargs: dict | None = None,
) -> tuple[Any, Any]:
    """One row per instrument of an orbit (reference ``:177-328``); per-row bounds from
    ``global_extrema`` (unrounded) or 1st / 99th percentiles; files that fail to load are logged
    and skipped.  Returns ``(fig, canvas)`` or ``(None, None)``."""
    datasets, lines = {}, {}
    first = True
    for inst in instrument_order:
        path = cdf_file_paths.get(inst)
        if not path:
            continue
        try:
            ds = load_fast_cdf_dataset(path)
            datasets[inst] = ds
            if first and filtered_orbits_df is not None and orbit_number is not None:
                # only the first loadable instrument is asked for cusp timestamps (reference :258-265)
                lines[inst] = get_timestamps_for_orbit(filtered_orbits_df, orbit_number, get_cdf_file_type(path), ds["times"])
                if not lines[inst]:
                    log_exception(f"No vertical lines found for orbit {orbit_number} in {path}. Skipping.", level="message")
            first = False
        except Exception as exc:
            log_exception(f"Failed to load CDF for {inst} at {path}. Skipping.", exc, level="error")
    if not datasets:
        return None, None
    shard = ShardPlan(_lib.default_context(), scale_function_y, scale_function_z, zoom_duration_minutes,
                      instrument_order=tuple(instrument_order))  # dtype from the files; mixed float dtypes raise
    shard.add_orbit(orbit_number, datasets, lines if lines else None)
    shard.upload()
    shard.collapse()
    spec = shard.plan_instrument_grid(shard.orbits[0], "given", global_extrema=global_extrema, y_min=y_min, y_max=y_max,
                                      z_min=z_min, z_max=z_max)
    return _run_single(shard, spec, colormap, cusp_marker_style, cusp_marker_kwargs)
