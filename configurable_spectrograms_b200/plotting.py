"""Generic spectrogram plotting on the GPU path (reference ``plotting.py``).

Same public functions and argument meaning as the reference: ``make_spectrogram``,
``generic_plot_spectrogram_set``, ``generic_plot_multirow_optional_zoom``,
``close_all_axes_and_clear``.  The numeric work of one ``make_spectrogram`` call --
``COLLAPSE_FUNCTION`` (``:188``), the energy / zoom / x-range masks (``:191-219``),
``compute_percentile_bounds`` (``:259``), ``safe_vmin`` (``:261-262``), the log / linear z
clamps (``:276-279,308-315``) and what ``imshow`` + the norm + the colormap would colour
(``:280-287,316-324``) -- runs in libcsgpu (K1, K2a, K3); the host keeps the axes metadata,
labels, ticks and cusp markers, recorded on raster axes (``figure.py``).

There is no CPU fallback: without libcsgpu / a CUDA device these functions raise ``CsgError``.
"""

from __future__ import annotations

from datetime import datetime, timezone

import math

import numpy as np

from . import _lib
from .colormaps import get_lut
from .constants import AXIS_LABEL_FONT_SIZE, PLOT_FIGURE_HEIGHT_INCHES, PLOT_FIGURE_WIDTH_INCHES, TICK_LABEL_FONT_SIZE
from .cusp_marking import draw_cusp_both_markers, draw_cusp_bracket_marker, draw_cusp_line_markers
from .engine import Batch, compute_dtype
from .fast.pipeline import check_norm_status, zoom_window
from .figure import FigureCanvas, SpectrogramFigure, close_all_axes_and_clear
from .logging_utils import log_message

__all__ = [
    "SpectrogramGroup",
    "make_spectrogram",
    "generic_plot_spectrogram_set",
    "generic_plot_multirow_optional_zoom",
    "close_all_axes_and_clear",
    "date2num",
    "num2date",
]

_CUSP_MARKER_DRAWERS = {
    "line": draw_cusp_line_markers,
    "bracket": draw_cusp_bracket_marker,
    "both": draw_cusp_both_markers,
}
#: colormaps whose high end is red: the cusp line switches to white on them (reference ``:45-50``)
_RED_HEAVY_COLORMAPS = {"turbo", "jet", "hot", "inferno", "magma", "plasma", "autumn", "gist_heat", "Reds", "YlOrRd", "OrRd"}


def date2num(unix_seconds):
    """matplotlib's ``date2num(datetime.fromtimestamp(t, tz=utc))``: days since 1970-01-01 UTC
    (the reference's x axis, ``:221-223``), vectorised.

    ``datetime.fromtimestamp`` rounds the fraction half-to-even to microseconds; matplotlib's
    ``_dt64_to_ordinalf`` then computes ``(whole_seconds + microseconds * 1000 / 1e9) / 86400``
    in float64.  Both steps are reproduced so the extents and marker positions match bit for bit.
    """
    if type(unix_seconds) in (float, int, np.float64):  # the per-panel limits and marker positions: plain float math
        frac, whole = math.modf(float(unix_seconds))
        micro = float(round(frac * 1e6))  # round(): half to even, like np.rint
        if micro == 0.0:
            micro = math.copysign(0.0, frac)  # (np.rint keeps the sign of a zero)
        if micro >= 1e6:
            whole, micro = whole + 1.0, micro - 1e6
        if micro < 0:  # negative timestamps: borrow a second, like divmod
            whole, micro = whole - 1.0, micro + 1e6
        return (whole + (micro * 1000.0) / 1.0e9) / 86400.0
    t = np.asarray(unix_seconds, dtype=np.float64)
    frac, whole = np.modf(t)
    micro = np.rint(frac * 1e6)
    carry = micro >= 1e6
    whole = np.where(carry, whole + 1.0, whole)
    micro = np.where(carry, micro - 1e6, micro)
    neg = micro < 0  # negative timestamps: borrow a second, like divmod
    whole = np.where(neg, whole - 1.0, whole)
    micro = np.where(neg, micro + 1e6, micro)
    days = (whole + (micro * 1000.0) / 1.0e9) / 86400.0
    return float(days) if days.ndim == 0 else days


def num2date(days, tz=timezone.utc):
    from datetime import timedelta

    return datetime(1970, 1, 1, tzinfo=timezone.utc) + timedelta(microseconds=round(float(days) * 86400e6))


def _colormap_name(colormap) -> str:
    return colormap if isinstance(colormap, str) else getattr(colormap, "name", "custom")


def _as_cube(data_array_3d, collapse_axis):
    cube = np.asarray(data_array_3d)
    if cube.ndim != 3:
        raise ValueError(f"make_spectrogram expects a 3-D array, got shape {cube.shape}")
    if collapse_axis != 1:
        cube = np.moveaxis(cube, collapse_axis, 1)
    if cube.dtype not in (np.float32, np.float64) and cube.dtype not in _lib.INT_CUBE_CODES:
        cube = cube.astype(np.float64)  # numpy sums and ranks integer input exactly; float64 keeps that
    return cube  # 8/16/32-bit integers stay as stored: K1 reads them and writes the exact float64 sums


def make_spectrogram(
    x_axis_values,
    y_axis_values,
    data_array_3d,
    x_axis_min=None,
    x_axis_max=None,
    x_axis_is_unix=True,
    x_axis_label=None,
    center_timestamp=None,
    window_duration_seconds=None,
    y_axis_scale_function=None,
    y_axis_label=None,
    y_axis_min=0,
    y_axis_max=4000,
    z_axis_scale_function=None,
    z_axis_min=None,
    z_axis_max=None,
    z_axis_label=None,
    collapse_axis=1,
    colormap="viridis",
    axis_object=None,
    instrument_label=None,
    vertical_lines_unix=None,
    cusp_marker_style="both",
    cusp_marker_kwargs=None,
    _context=None,
    _group=None,
):
    """Plot a spectrogram by collapsing a 3-D array along an axis (reference ``:92-389``).

    Returns ``(axis_object, x_axis_plot)`` or ``(None, None)`` when every energy bin / time step
    is filtered out.  ``axis_object`` is a :class:`figure.PanelAxes` holding the RGBA raster
    (``.images[-1].rgba``, row 0 = lowest energy), the LUT index plane (``.index``) and the
    resolved ``vmin`` / ``vmax``.
    """
    log_message(
        f"[DEBUG] make_spectrogram: y_axis_scale_function={y_axis_scale_function}, "
        f"z_axis_scale_function={z_axis_scale_function}, z_axis_min={z_axis_min}, "
        f"z_axis_max={z_axis_max}, colormap={colormap}"
    )
    x_axis = np.asarray(x_axis_values)
    y_axis = np.asarray(y_axis_values)
    cube = _as_cube(data_array_3d, collapse_axis)

    # energy mask (:191-198); the all-NaN-column mask is a no-op after nansum (all-NaN -> 0.0)
    with np.errstate(invalid="ignore"):
        keep = np.flatnonzero((y_axis >= y_axis_min) & (y_axis <= y_axis_max))
    if cube.shape[0] == 0 or len(keep) == 0:
        log_message("[WARNING] All energy bins were filtered out. No data to plot.")
        return None, None
    y_kept = y_axis[keep]
    if y_kept[0] > y_kept[-1]:  # descending energies: flip (:200-202)
        y_kept, keep = y_kept[::-1], keep[::-1]

    rows = np.arange(len(x_axis))
    if center_timestamp is not None and window_duration_seconds is not None:  # :204-210
        half = window_duration_seconds / 2
        with np.errstate(invalid="ignore"):
            rows = rows[(x_axis[rows] >= center_timestamp - half) & (x_axis[rows] <= center_timestamp + half)]
    if x_axis_min is not None or x_axis_max is not None:  # :212-219
        with np.errstate(invalid="ignore"):
            m = np.ones(len(rows), dtype=bool)
            if x_axis_min is not None:
                m &= x_axis[rows] >= x_axis_min
            if x_axis_max is not None:
                m &= x_axis[rows] <= x_axis_max
        rows = rows[m]
    x_sel = x_axis[rows]
    if x_axis_is_unix:
        x_axis_plot = date2num(x_sel) if len(x_sel) else np.zeros(0)
        x_label = x_axis_label if x_axis_label is not None else "Time (UTC)"
    else:
        x_axis_plot = x_sel
        x_label = x_axis_label if x_axis_label is not None else "X"

    if axis_object is None:
        fig = SpectrogramFigure(figsize=(PLOT_FIGURE_WIDTH_INCHES, PLOT_FIGURE_HEIGHT_INCHES))
        FigureCanvas(fig)
        axis_object = fig.add_subplot(1, 1, 1)
    else:
        fig = axis_object.figure

    if center_timestamp is not None and window_duration_seconds is not None:
        lo, hi = center_timestamp - window_duration_seconds / 2, center_timestamp + window_duration_seconds / 2
        if x_axis_is_unix:
            axis_object.set_xlim(date2num(lo), date2num(hi))
        else:
            axis_object.set_xlim(lo, hi)
    else:
        axis_object.set_xlim(x_axis_plot[0], x_axis_plot[-1])  # IndexError on an empty x, like the reference (:253)
    if len(rows) == 0:
        log_message("[WARNING] No data to plot after filtering. Skipping plot.")
        return None, None

    # ---- the numeric path on the GPU: K1 collapse, K2a bounds, K3 norm + colormap
    log_scale = z_axis_scale_function == "log"
    annotate = dict(x_label=x_label, x_axis_is_unix=x_axis_is_unix, y_axis_scale_function=y_axis_scale_function,
                    y_axis_label=y_axis_label, y_axis_min=y_axis_min, y_axis_max=y_axis_max, z_axis_label=z_axis_label,
                    colormap=colormap, instrument_label=instrument_label, vertical_lines_unix=vertical_lines_unix,
                    cusp_marker_style=cusp_marker_style, cusp_marker_kwargs=cusp_marker_kwargs)
    if _group is not None:  # planned now, computed with every other panel of the group, drawn by group.run()
        _group.plan(cube, keep, rows, log_scale, z_axis_min, z_axis_max, axis_object, x_axis_plot, y_kept, annotate)
        return axis_object, x_axis_plot
    ctx = _context or _lib.default_context()
    batch = Batch(ctx, compute_dtype(cube.dtype), n_groups=0)
    f = batch.add_file(cube)
    batch.upload_cubes()
    batch.collapse()
    region = batch.add_region(f, 0, keep, rows=rows, want_pct=z_axis_min is None or z_axis_max is None)
    panel = batch.add_panel(region, -1, log_scale, z_axis_min, z_axis_max)
    batch.upload_tables()
    batch.run_stats()
    batch.prepare()
    batch.set_lut(get_lut(colormap))
    batch.rasterise(want_rgba=True, want_index=True)
    z_lo, z_hi = _resolved_bounds(batch.norms()[panel], batch.stats()[region] if log_scale else None, log_scale)
    draw_panel(axis_object, batch.panel_rgba(panel), batch.panel_index(panel), z_lo, z_hi, log_scale, x_axis_plot, y_kept, **annotate)
    return axis_object, x_axis_plot


def _resolved_bounds(norm, stats, log_scale):
    """``(vmin, vmax)`` of a panel's resolved normalisation; raises what matplotlib raises when the figure is
    drawn with an invalid one, and logs the reference's warning for a log panel that holds non-positive cells
    (``:264-275``)."""
    check_norm_status(norm)
    z_lo, z_hi = float(norm["vmin"]), float(norm["vmax"])
    if log_scale and stats is not None:
        if stats["n_pos"] < stats["n_valid"] + stats["n_nan"] or not (np.isfinite(z_lo) and z_hi > z_lo > 0):
            log_message("[WARNING] Non-positive values found in matrix for log colorbar. "
                        "Masking to z_axis_min and enforcing log scale.")
    return z_lo, z_hi


class SpectrogramGroup:
    """Many ``make_spectrogram`` calls, one pass over the GPU.

    The reference draws every generic item in its own worker process (``generic_batch.py:90-118``); one call
    here costs a handful of kernel launches that leave a B200 idle.  A group collects the panels of many
    figures instead -- every cube is uploaded and collapsed as it is planned (streaming:
    ``Batch.collapse_pending``; the host array is not kept) -- then :meth:`run` selects every panel's
    percentiles in ONE K2a launch, rasterises them in ONE K3 launch and finishes the axes from device
    rasters, so the figures go to ``png.write_figures_device`` without a pixel crossing PCIe uncompressed.
    One batch per compute dtype (numpy computes each cube in its own dtype; integer cubes in float64)."""

    def __init__(self, colormap="viridis", context=None):
        self.ctx = context or _lib.default_context()
        self.colormap = colormap
        self.batches: dict = {}
        self.pending: list = []

    def plan(self, cube, keep, rows, log_scale, z_min, z_max, axis_object, x_axis_plot, y_kept, annotate):
        dtype = compute_dtype(cube.dtype)
        batch = self.batches.get(dtype)
        if batch is None:
            batch = self.batches[dtype] = Batch(self.ctx, dtype, n_groups=0)
        f = batch.add_file(cube)
        batch.collapse_pending()
        region = batch.add_region(f, 0, keep, rows=rows, want_pct=z_min is None or z_max is None)
        panel = batch.add_panel(region, -1, log_scale, z_min, z_max)
        self.pending.append((batch, region, panel, log_scale, axis_object, x_axis_plot, y_kept, annotate))

    def run(self) -> list:
        """Compute and draw everything planned so far.  Returns one entry per planned panel: ``None``, or the
        exception drawing it raised (an invalid normalisation) -- the caller decides which figure that fails."""
        from .figure import DeviceRaster

        lut = get_lut(self.colormap)
        for batch in self.batches.values():
            batch.upload_tables()
            batch.run_stats()
            batch.prepare()
            batch.set_lut(lut)
            batch.rasterise(want_rgba=True, want_index=False)
        tables = {id(b): (b.norms(), b.stats()) for b in self.batches.values()}
        outcome = []
        for batch, region, panel, log_scale, axis_object, x_axis_plot, y_kept, annotate in self.pending:
            norms, stats = tables[id(batch)]
            try:
                z_lo, z_hi = _resolved_bounds(norms[panel], stats[region] if log_scale else None, log_scale)
                ne, nt = batch.panel_shape(panel)
                draw_panel(axis_object, DeviceRaster(batch.panel_offset(panel), ne, nt), None, z_lo, z_hi, log_scale, x_axis_plot,
                           y_kept, **annotate)
                axis_object.images[-1].batch = batch  # which RGBA buffer the raster lives in
                outcome.append(None)
            except ValueError as exc:
                outcome.append(exc)
        self.pending = []
        return outcome

    def rgba_ptr(self, figure) -> int:
        """Device address of the RGBA buffer a figure's panels live in (one compute dtype per figure)."""
        owners = {id(ax.images[-1].batch): ax.images[-1].batch for ax in figure.axes if ax.images and hasattr(ax.images[-1], "batch")}
        if len(owners) != 1:
            raise ValueError("a figure drawn from a group must hold panels of one cube dtype")
        return next(iter(owners.values())).d_rgba.ptr


def _decade_ticks(z_lo, z_hi):
    """Colour-bar ticks of a log panel: the powers of ten inside [z_lo, z_hi] (reference ``:288-299``)."""
    z_lo, z_hi = float(z_lo), float(z_hi)
    if not (z_lo > 0 and z_hi > 0 and math.isfinite(z_lo) and math.isfinite(z_hi)):
        return None
    decades = range(int(math.floor(math.log10(z_lo))), int(math.ceil(math.log10(z_hi))) + 1)
    return [10**k for k in decades if z_lo <= 10**k <= z_hi]


def _energy_ticks(y_axis_min, y_axis_max):
    """The reference's y ticks for a linear energy axis (``:335-352``): a step of one power of ten read off
    the PRINTED form of ``y_axis_max`` (so 4000 and 4000.0 tick differently, as there), an upper tick of
    ``d`` or ``d + 0.5`` leading digits, ticks up to 10 % beyond it."""
    printed = str(y_axis_max)
    width, lead, nxt = len(printed), int(printed[0]), int(printed[1])
    if nxt >= 5:
        step, top = 10**width, lead * 10 ** (width - 1)
    else:
        step, top = 10 ** (width - 1), (lead + 0.5) * 10 ** (width - 1)
    return [v for v in range(y_axis_min, int(top) + 1, step) if v / top <= 1.1]


def draw_panel(axis_object, rgba, index, z_lo, z_hi, log_scale, x_axis_plot, y_kept, *, x_label="Time (UTC)",
               x_axis_is_unix=True, y_axis_scale_function=None, y_axis_label=None, y_axis_min=0, y_axis_max=4000,
               z_axis_label=None, colormap="viridis", instrument_label=None, vertical_lines_unix=None,
               cusp_marker_style="both", cusp_marker_kwargs=None):
    """What ``make_spectrogram`` puts on the axes once the raster exists (reference ``:280-387``): the image
    with its extent, a colour bar (decade ticks on a log panel), axis labels, energy ticks, the time format
    chosen by the displayed span, cusp markers inside the plotted range, the path's font sizes."""
    ax, fig = axis_object, axis_object.figure
    image = ax.imshow(rgba, aspect="auto", origin="lower", extent=(x_axis_plot[0], x_axis_plot[-1], y_kept[0], y_kept[-1]),
                      cmap=_colormap_name(colormap), norm="log" if log_scale else None, vmin=z_lo, vmax=z_hi, index=index)
    bar = fig.colorbar(image, ax=ax, label="Counts" if z_axis_label is None else z_axis_label,
                       ticks=_decade_ticks(z_lo, z_hi) if log_scale else None)
    ax.set_xlabel(x_label)
    ax.set_ylabel("Energy (eV)" if y_axis_label is None else y_axis_label)
    if instrument_label is not None:
        ax.set_title(instrument_label)
    if len(y_kept) >= 2:
        if y_axis_scale_function == "log":
            ax.set_yscale("log")
        else:
            ticks = _energy_ticks(y_axis_min, y_axis_max)
            if ticks:
                ax.set_yticks(ticks)
                ax.set_yticklabels([f"{int(v)}" for v in ticks])
    if x_axis_is_unix:  # seconds matter only on a window shorter than two minutes (:357-368)
        left, right = ax.get_xlim()
        # (num2date(right) - num2date(left)).total_seconds(): both ends rounded to microseconds, then subtracted
        span_us = round(float(right) * 86400e6) - round(float(left) * 86400e6)
        ax.xaxis.set_major_formatter("%H:%M:%S" if span_us / 1e6 < 120 else "%H:%M")
    if vertical_lines_unix is not None and len(vertical_lines_unix) > 0:
        positions = [date2num(float(v)) for v in vertical_lines_unix] if x_axis_is_unix else vertical_lines_unix
        inside = [v for v in positions if x_axis_plot[0] <= v <= x_axis_plot[-1]]
        options = dict(cusp_marker_kwargs or {})
        options.setdefault("line_color", "white" if colormap in _RED_HEAVY_COLORMAPS else "red")
        _CUSP_MARKER_DRAWERS.get(cusp_marker_style, draw_cusp_both_markers)(ax, inside, **options)
    for target, which, length in ((ax, "major", 8), (ax, "minor", 5), (bar.ax, "major", 6), (bar.ax, "minor", 3)):
        extra = {"axis": "both"} if target is ax else {}
        target.tick_params(which=which, labelsize=TICK_LABEL_FONT_SIZE, length=length, width=1, **extra)
    for label in (ax.xaxis.label, ax.yaxis.label):
        label.set_fontsize(AXIS_LABEL_FONT_SIZE)
    bar.ax.set_ylabel("Counts", fontsize=AXIS_LABEL_FONT_SIZE)
    return image


def generic_plot_spectrogram_set(
    datasets,
    collapse_axis=1,
    zoom_center=None,
    zoom_window_seconds=None,
    vertical_lines=None,
    x_is_unix=True,
    y_scale="linear",
    z_scale="linear",
    colormap="viridis",
    figure_title=None,
    show=False,
    y_min=None,
    y_max=None,
    z_min=None,
    z_max=None,
    cusp_marker_style="both",
    cusp_marker_kwargs=None,
    _group=None,
):
    """A vertical stack of generic spectrograms (reference ``:392-502``): one ``make_spectrogram``
    per dataset dict (required keys ``x, y, data``; optional ``label, y_label, z_label, x_label,
    y_min, y_max, z_min, z_max``).  Returns ``(fig, canvas)`` or ``(None, None)``."""
    if not datasets:
        return None, None
    fig = SpectrogramFigure(figsize=(10, 3 * len(datasets)))
    canvas = FigureCanvas(fig)
    for row_index, dataset in enumerate(datasets):
        axis_obj = fig.add_subplot(len(datasets), 1, row_index + 1)
        ds_y_min, ds_y_max = dataset.get("y_min", y_min), dataset.get("y_max", y_max)
        ds_z_min, ds_z_max = dataset.get("z_min", z_min), dataset.get("z_max", z_max)
        inferred_y_max = dataset["y"].max() if ds_y_max is None and dataset.get("y") is not None else ds_y_max
        make_spectrogram(
            x_axis_values=dataset["x"],
            y_axis_values=dataset["y"],
            data_array_3d=dataset["data"],
            collapse_axis=collapse_axis,
            center_timestamp=zoom_center,
            window_duration_seconds=zoom_window_seconds,
            x_axis_is_unix=x_is_unix,
            y_axis_scale_function=y_scale,
            z_axis_scale_function=z_scale,
            y_axis_min=ds_y_min if ds_y_min is not None else 0,
            y_axis_max=inferred_y_max if inferred_y_max is not None else 4000,
            z_axis_min=ds_z_min,
            z_axis_max=ds_z_max,
            colormap=colormap,
            y_axis_label=dataset.get("y_label", "Energy (eV)"),
            z_axis_label=dataset.get("z_label", "Counts"),
            x_axis_label="Time (UTC)" if x_is_unix else dataset.get("x_label"),
            vertical_lines_unix=vertical_lines,
            cusp_marker_style=cusp_marker_style,
            cusp_marker_kwargs=cusp_marker_kwargs,
            axis_object=axis_obj,
            _group=_group,
        )
        if dataset.get("label"):
            axis_obj.set_title(dataset["label"])
    if figure_title:
        fig.suptitle(figure_title)
    fig.tight_layout(rect=(0, 0, 1, 0.97))
    return fig, canvas


def generic_plot_multirow_optional_zoom(
    datasets,
    vertical_lines=None,
    zoom_duration_minutes=6.25,
    y_scale="linear",
    z_scale="linear",
    colormap="viridis",
    show=False,
    title=None,
    row_label_pad=50,
    row_label_rotation=90,
    y_min=None,
    y_max=None,
    z_min=None,
    z_max=None,
    cusp_marker_style="both",
    cusp_marker_kwargs=None,
):
    """Rows of spectrograms with an optional zoom column (reference ``:505-698``).

    Dataset keys read: ``x, y, data, vmin, vmax, label`` -- exactly the reference's set (its
    ``y_min / y_max / z_min / z_max`` dataset keys are ignored there too, so every panel is
    clipped to the default 0-4000 eV).
    """
    if not datasets:
        return None, None
    zoom_needed = False
    centre = duration = None
    zoom = zoom_window(vertical_lines, zoom_duration_minutes) if vertical_lines is not None and len(vertical_lines) > 0 else None
    if zoom is not None:
        centre, duration = zoom
        left, right = centre - duration / 2, centre + duration / 2
        for ds in datasets:
            t, d = np.asarray(ds["x"]), np.asarray(ds["data"])
            with np.errstate(invalid="ignore"):
                mask_zoom = (t >= left) & (t <= right)
            if np.any(~np.isnan(d[mask_zoom])):
                zoom_needed = True
                break
    n_rows, n_cols = len(datasets), 2 if zoom_needed else 1
    fig = SpectrogramFigure(figsize=(12 * n_cols, 3 * n_rows))
    canvas = FigureCanvas(fig)
    axes = np.empty((n_rows, n_cols), dtype=object)
    for i in range(n_rows):
        for j in range(n_cols):
            axes[i, j] = fig.add_subplot(n_rows, n_cols, i * n_cols + j + 1)
    for i, ds in enumerate(datasets):
        times, energy, data3d = ds["x"], ds["y"], ds["data"]
        vmin, vmax = ds.get("vmin"), ds.get("vmax")
        common = dict(
            x_axis_values=times, y_axis_values=energy, data_array_3d=data3d, collapse_axis=1, x_axis_is_unix=True,
            instrument_label=None, y_axis_scale_function=y_scale, z_axis_scale_function=z_scale,
            vertical_lines_unix=vertical_lines, cusp_marker_style=cusp_marker_style, cusp_marker_kwargs=cusp_marker_kwargs,
            z_axis_min=vmin if z_min is None else z_min, z_axis_max=vmax if z_max is None else z_max, colormap=colormap,
        )
        make_spectrogram(x_axis_min=times[0], x_axis_max=times[-1], axis_object=axes[i, 0], **common)
        if n_cols == 2:
            make_spectrogram(center_timestamp=centre, window_duration_seconds=duration, axis_object=axes[i, 1], **common)
    _finish_multirow(fig, axes, datasets, vertical_lines, title, row_label_pad, row_label_rotation)
    return fig, canvas


def _utc(seconds) -> str:
    return datetime.fromtimestamp(float(seconds), tz=timezone.utc).strftime("%Y-%m-%d %H:%M:%S")


def _finish_multirow(fig, axes, datasets, vertical_lines, title, row_label_pad=50, row_label_rotation=90):
    """What a multirow figure carries besides its panels (reference ``:659-693``): the dataset label as the
    y label of every row's first panel, "Full" / "Zoomed" column heads, the title, and two footers -- the
    time span of the first dataset and, in red, the marked (cusp) range."""
    for row, dataset in zip(axes, datasets):
        row[0].set_ylabel(dataset.get("label", ""), fontsize=AXIS_LABEL_FONT_SIZE, rotation=row_label_rotation,
                          labelpad=row_label_pad, va="center")
    for head, ax in zip(("Full", "Zoomed"), axes[0]):
        ax.set_title(head, fontsize=AXIS_LABEL_FONT_SIZE)
    if title:
        fig.suptitle(title, fontsize=AXIS_LABEL_FONT_SIZE + 2)
    footers = [(0.01, f"Data timespan: {_utc(datasets[0]['x'][0])} to {_utc(datasets[0]['x'][-1])} UTC", "black")]
    if vertical_lines is not None and len(vertical_lines) > 0:
        footers.append((0.045, f"Marked range: {_utc(min(vertical_lines))} to {_utc(max(vertical_lines))} UTC", "red"))
    fig.subplots_adjust(bottom=0.18)
    for height, text, colour in footers:
        fig.text(0.5, height, text, ha="center", va="bottom", fontsize=13, color=colour)
    fig.tight_layout(rect=(0, 0.08, 1, 0.95))
