"""K4's host tables: the canvas rows, tiles, content rows and row maps that ``png._device_tables`` builds for a list
of device-raster figures, and their split into groups under a segment budget (``png._groups``).  No GPU needed."""

import math

import numpy as np
import pytest

from configurable_spectrograms_b200 import png
from configurable_spectrograms_b200._lib import PNG_CANVAS, TILE_ROW_MAP
from configurable_spectrograms_b200.figure import DeviceRaster, SpectrogramFigure
from configurable_spectrograms_b200.plotting import draw_panel

DPI = 100


def _figure(scales, n_cols=2, ne=74, nt=300, width=12.0, host=False):
    """A grid of panels drawn by ``plotting.draw_panel`` from device rasters (or host arrays), one y scale each."""
    n_rows = -(-len(scales) // n_cols)
    fig = SpectrogramFigure(figsize=(width * n_cols, 3 * n_rows))
    for k, scale in enumerate(scales):
        ax = fig.add_subplot(n_rows, n_cols, k + 1)
        x = (10957.0, 10957.0 + nt * 2.5 / 86400.0)
        ax.set_xlim(*x)
        rgba = np.zeros((ne, nt, 4), np.uint8) if host else DeviceRaster(k * ne * nt, ne, nt)
        draw_panel(ax, rgba, None, 1.0, 100.0, True, x, np.array((4.0, 4000.0)), y_axis_scale_function=scale,
                   colormap="turbo", instrument_label=f"panel {k}")
    fig.suptitle(f"Orbit 13000 - {len(scales)} panels")
    return fig


def _figures():
    return [
        _figure(["log", "linear", "log", "linear"]),  # two log panels of one geometry: one map
        _figure(["linear"], n_cols=1, width=30.0),  # three segments per scanline
        _figure(["linear", "log", "linear", "log"]),  # the same map again, in another figure
        _figure(["log"], n_cols=1, ne=20, width=4.0),  # a map of its own
    ]


def test_device_tables_follow_each_figures_tiles():
    figs = _figures()
    t = png._device_tables(figs, DPI)
    assert t.canvases.dtype == PNG_CANVAS and len(t.canvases) == len(t.n_rows) == len(figs)
    tile_first = row_first = 0
    mapped_at: dict = {}  # row-map key -> offsets the tiles that show it point at
    for fig, c, n in zip(figs, t.canvases, t.n_rows):
        ft = fig.tiles(DPI)
        rows = ft.content_rows()
        r, g, b, a = ft.background
        assert (c["W"], c["H"], c["background"]) == (ft.W, ft.H, r | (g << 8) | (b << 16) | (a << 24))
        assert (c["tile_first"], c["tile_count"]) == (tile_first, len(ft.records))
        assert c["segs_per_row"] == math.ceil(ft.W / 1024)
        assert c["row_first"] == row_first and n == len(rows)
        assert np.array_equal(t.rows[row_first : row_first + n], rows)
        tiles, own = t.tiles[tile_first : tile_first + len(ft.records)], ft.table()
        mapped = (own["flags"] & TILE_ROW_MAP) != 0
        for name in own.dtype.names:  # everything but the row-map offsets is the figure's own table
            if name != "row_map":
                assert np.array_equal(tiles[name], own[name]), name
        assert np.array_equal(tiles["row_map"][~mapped], own["row_map"][~mapped])
        for k in np.flatnonzero(mapped):
            key, m = ft.map_of(int(k))
            off = int(tiles["row_map"][k])
            assert np.array_equal(t.row_maps[off : off + len(m)], m)
            mapped_at.setdefault(key, set()).add(off)
        tile_first += len(ft.records)
        row_first += n
    assert len(t.tiles) == tile_first and len(t.rows) == row_first
    # two distinct maps; every one stored once and every tile that shows it points at that copy
    distinct = {key: m for fig in figs for key, m in fig.tiles(DPI).row_maps}
    assert len(mapped_at) == len(distinct) == 2 and all(len(offs) == 1 for offs in mapped_at.values())
    assert len(t.row_maps) == sum(len(m) for m in distinct.values())


def test_groups_split_under_the_segment_budget():
    t = png._device_tables(_figures() * 2, DPI)
    segs = t.canvases["segs_per_row"].astype(np.int64) * t.n_rows
    for budget in (1, int(segs.min()), int(segs.max()), int(segs.max() + segs.min()), int(segs.sum()) - 1, 10**9):
        canvases = t.canvases.copy()
        groups = png._groups(canvases, t.n_rows, budget)
        assert groups[0].first == 0 and groups[-1].stop == len(segs)
        assert all(a.stop == b.first for a, b in zip(groups[:-1], groups[1:]))
        for g in groups:
            inner = segs[g.first : g.stop]
            assert g.stop > g.first and g.n_seg == inner.sum()
            assert np.array_equal(canvases["seg_first"][g.first : g.stop], np.cumsum(inner) - inner)  # restarts at 0
            assert g.n_seg <= budget or g.stop - g.first == 1
            if g.stop < len(segs):  # the next figure was refused because it would go over the budget
                assert g.n_seg + segs[g.stop] > budget
        for k in np.flatnonzero(segs > budget):  # a figure larger than the budget: a group of its own
            assert any((g.first, g.stop) == (k, k + 1) for g in groups), (budget, k)
    assert len(png._groups(t.canvases.copy(), t.n_rows, 1)) == len(segs)
    assert len(png._groups(t.canvases.copy(), t.n_rows, 10**9)) == 1
    empty = png._device_tables([], DPI)
    assert len(empty.canvases) == 0 and empty.row_maps is None and png._groups(empty.canvases, empty.n_rows, 10) == []


def test_host_raster_panels_are_refused():
    with pytest.raises(TypeError, match="needs panels drawn from device rasters"):
        png._device_tables([_figure(["log"], n_cols=1), _figure(["linear"], n_cols=1, host=True)], DPI)
