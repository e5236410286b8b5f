"""Panels on a log energy axis (``y_scale="log"``) on the device: K4 places the rows of a panel through the
host's row map in both its counting and its encoding pass, and every public entry point that takes
``y_scale="log"`` draws that axis -- the device PNGs equal the host composer pixel for pixel."""

import io
import json
import os

import numpy as np
import pytest

from tests.test_gpu_api import ORDER, _write_tree
from tests.test_log_energy_axis_cpu import _independent_map

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from configurable_spectrograms_b200 import _lib

    return _lib.Context(0)


def _download(ctx, d_rgba_ptr, raster):
    host = np.empty((raster.ne, raster.nt, 4), dtype=np.uint8)
    ctx._check(ctx.lib.csg_d2h(ctx.handle, host.ctypes.data, d_rgba_ptr + 4 * raster.offset, host.nbytes))
    ctx.sync()
    return host


def _twin_figures(flat, specs, grid):
    """The same figure twice (host arrays / device references), panels drawn by ``plotting.draw_panel`` with a
    y scale of their own; odd panels show their image inside wider time limits (a zoom-width image)."""
    from configurable_spectrograms_b200.figure import DeviceRaster, SpectrogramFigure
    from configurable_spectrograms_b200.plotting import draw_panel

    figs = []
    n_rows, n_cols = grid
    for device in (False, True):
        fig = SpectrogramFigure(figsize=(12 * n_cols, 3 * n_rows))
        for k, (cell, off, ne, nt, scale, y) in enumerate(specs):
            ax = fig.add_subplot(n_rows, n_cols, cell)
            x0 = 10957.0 + 0.01 * k
            x1 = x0 + nt * 2.5 / 86400.0
            ax.set_xlim(x0 - (0.001 if k % 2 else 0.0), x1 + (0.002 if k % 2 else 0.0))
            rgba = DeviceRaster(off, ne, nt) if device else flat[off : off + ne * nt].view(np.uint8).reshape(ne, nt, 4)
            draw_panel(ax, rgba, None, 1.0, 2400.0, k % 2 == 0, (x0, x1), np.array(y), y_axis_scale_function=scale,
                       colormap="turbo", instrument_label="Full" if k == 0 else None,
                       vertical_lines_unix=[(x0 + 0.3 * (x1 - x0)) * 86400.0] if k == 1 else None)
        fig.suptitle(f"Orbit 13000 - {len(specs)} panels, log and linear energy axes", fontsize=16)
        fig.tight_layout(rect=(0, 0.03, 1, 0.95))
        figs.append(fig)
    return figs


def _figures(ctx):
    rng = np.random.default_rng(21)
    palette = rng.integers(0, 256, 300, dtype=np.uint32) | np.uint32(0xFF000000)
    shapes = [(74, 800), (74, 181), (700, 90), (2, 300), (74, 903), (1, 40), (96, 2100)]
    offs, parts, pos = [], [], 0
    for i, (ne, nt) in enumerate(shapes):
        if i == 4:
            px = rng.integers(0, 2**32, ne * nt, dtype=np.uint64).astype(np.uint32)  # incompressible
        else:
            idx = np.clip((rng.normal(0, 1, (ne, nt)).cumsum(axis=1) * 3 + 150 + 2 * np.arange(ne)[:, None]).astype(int), 0, 299)
            px = palette[idx].reshape(-1)
        offs.append(pos)
        parts.append(px)
        pos += (ne * nt + 3) & ~3
        parts.append(np.zeros(((ne * nt + 3) & ~3) - ne * nt, np.uint32))
    flat = np.concatenate(parts)
    d_rgba = ctx.to_device(flat)
    fast, rev = (4.0, 4000.0), (4000.0, 4.0)
    layouts = [
        # (grid, [(cell, panel, y scale, extent ends)]): a FAST grid of log and linear rows, one with more rows
        # than pixels, a downward axis, the fallbacks (two rows / one row / a non-positive end) beside them
        ((4, 2), [(1, 0, "log", fast), (2, 1, "log", fast), (3, 2, "log", fast), (4, 1, "linear", fast),
                  (5, 0, "linear", fast), (6, 1, "log", rev), (7, 4, "log", fast), (8, 3, "log", (0.0, 4000.0))]),
        ((1, 1), [(1, 6, "log", (1e-2, 1e5))]),
        ((2, 1), [(1, 5, "log", fast), (2, 3, "log", (4.1, 4.9))]),
        ((1, 1), [(1, 0, "linear", fast)]),
    ]
    host_figs, dev_figs = [], []
    for grid, cells in layouts:
        specs = [(cell, offs[p], *shapes[p], scale, y) for cell, p, scale, y in cells]
        h, d = _twin_figures(flat, specs, grid)
        host_figs.append(h)
        dev_figs.append(d)
    return d_rgba, host_figs, dev_figs


def test_device_png_matches_host_compose_on_log_axes(ctx, tmp_path):
    from PIL import Image

    from configurable_spectrograms_b200 import png
    from configurable_spectrograms_b200._lib import TILE_ROW_MAP

    d_rgba, host_figs, dev_figs = _figures(ctx)
    t = host_figs[0].tiles(100)
    assert sum(bool(t.records[k][9] & TILE_ROW_MAP) for k in t.sources) == 5  # the log panels that have a warp to show
    for budget, dpi in ((160_000, 100), (700, 100), (160_000, 200), (900, 200), (160_000, 37), (300, 37)):
        blobs = png.encode_figures_device(ctx, d_rgba.ptr, dev_figs, max_segments=budget, dpi=dpi)
        assert len(blobs) == len(host_figs)
        for blob, fig in zip(blobs, host_figs):
            want = fig.compose(dpi)
            assert np.array_equal(png.decode_rgba(blob), want), (budget, dpi)
            assert np.array_equal(np.asarray(Image.open(io.BytesIO(blob)).convert("RGBA")), want), (budget, dpi)
    # deferred mode (the directory driver's), files through the native writer: everything deferred / only the last
    # of several groups
    paths = [str(tmp_path / f"f{k}.png") for k in range(len(dev_figs))]
    for budget in (160_000, 700):
        handle = png.encode_figures_device(ctx, d_rgba.ptr, dev_figs, dpi=100, max_segments=budget, paths=paths, wait=False,
                                           defer=True)
        for fut in handle.complete():
            fut.result()
        for path, fig in zip(paths, host_figs):
            assert np.array_equal(png.decode_rgba(open(path, "rb").read()), fig.compose(100)), budget
            os.remove(path)


def test_tile_with_row_map_flag_and_no_map_table_raises(ctx, tmp_path, monkeypatch):
    """A TILE_ROW_MAP tile with a NULL ``d_row_maps`` is reported by the kernel; no file is written, and the
    context encodes again afterwards."""
    from configurable_spectrograms_b200 import png

    d_rgba, host_figs, dev_figs = _figures(ctx)
    tables = png._device_tables

    def without_maps(figures, dpi):
        canvases, tiles, rows, row_maps, per_figure = tables(figures, dpi)
        assert row_maps is not None
        return canvases, tiles, rows, None, per_figure

    monkeypatch.setattr(png, "_device_tables", without_maps)
    path = str(tmp_path / "f.png")
    with pytest.raises(ValueError, match="row map"):
        png.write_figures_device(ctx, d_rgba.ptr, [(path, dev_figs[0])], dpi=100)
    assert not os.path.exists(path)
    with pytest.raises(ValueError, match=r"figure [012]: a tile reads a row map"):  # the figures with mapped tiles
        png.encode_figures_device(ctx, d_rgba.ptr, dev_figs, dpi=37)
    monkeypatch.setattr(png, "_device_tables", tables)
    blob = png.encode_figures_device(ctx, d_rgba.ptr, dev_figs[:1], dpi=100)[0]
    assert np.array_equal(png.decode_rgba(blob), host_figs[0].compose(100))


def _check_rows_against_cpu_map(t, img):
    """The log panels of composed / decoded image ``img`` show, canvas row by canvas row, the storage row the
    log transform gives (the independent CPU map), and that is not what a linear axis shows.  Pixels that a
    tile drawn on top of the panel covers (cusp lines and brackets) are left out."""
    from configurable_spectrograms_b200._lib import TILE_ROW_MAP
    from configurable_spectrograms_b200.figure import nearest_index

    n = 0
    for k in sorted(t.sources):
        off, ne, nt, x, y, w, h, _a, _b, flags, _m = t.records[k]
        if not flags & TILE_ROW_MAP:
            continue
        _ne, _h, y_lo, y_hi = t.map_of(k)[0]
        rows, near = _independent_map(ne, h, y_lo, y_hi)
        assert not near.any()
        assert not np.array_equal(rows, ne - 1 - nearest_index(h, ne))
        free = np.ones((h, w), dtype=bool)
        for r in t.records[:k]:  # the first tile covering a pixel wins
            free[max(r[4] - y, 0) : max(r[4] + r[6] - y, 0), max(r[3] - x, 0) : max(r[3] + r[5] - x, 0)] = False
        assert free.any(axis=1).all() and free.mean() > 0.5  # cusp lines cover whole columns of a narrow zoom panel
        want = t.sources[k][rows][:, nearest_index(w, nt)]
        assert np.array_equal(img[y : y + h, x : x + w][free], want[free])
        n += 1
    return n


def test_single_figure_entry_points_draw_a_log_axis():
    from configurable_spectrograms_b200.plotting import generic_plot_spectrogram_set, make_spectrogram

    rng = np.random.default_rng(8)
    times = 946684800.0 + 2.5 * np.arange(300)
    energy = np.geomspace(4.0, 30000.0, 48)[::-1].copy()
    cube = rng.poisson(3.0, (300, 5, 48)).astype(np.float32)
    ax, _x = make_spectrogram(times, energy, cube, y_axis_scale_function="log", y_axis_max=40000, z_axis_scale_function="log")
    assert ax.yscale == "log"
    fig = ax.figure
    assert _check_rows_against_cpu_map(fig.tiles(100), fig.compose(100)) == 1
    fig, _canvas = generic_plot_spectrogram_set(
        [{"x": times, "y": energy, "data": cube, "label": "a"}, {"x": times, "y": energy[:20], "data": cube[:, :, :20], "label": "b"}],
        y_scale="log", z_scale="log", show=False)
    for dpi in (100, 200):
        assert _check_rows_against_cpu_map(fig.tiles(dpi), fig.compose(dpi)) == 2


@pytest.mark.parametrize("z_scale", ["linear", "log"])
@pytest.mark.parametrize("percentile", [99, None])
def test_directory_driver_draws_log_energy_axes(tmp_path, monkeypatch, z_scale, percentile):
    """FAST_plot_spectrograms_directory with y_scale="log": its device-composed PNGs equal what the per-orbit
    worker writes when every figure is composed on the host (the oracle) from the same rasters; the panels of a
    decoded file follow the CPU row map."""
    from configurable_spectrograms_b200 import cdf_utils, png
    from configurable_spectrograms_b200.cdf_utils import load_filtered_orbits
    from configurable_spectrograms_b200.fast import process_orbit
    from configurable_spectrograms_b200.fast.batch_directory import FAST_plot_spectrograms_directory
    from configurable_spectrograms_b200.fast.orbit_discovery import discover_orbit_files
    from configurable_spectrograms_b200.figure import DeviceRaster

    _write_tree(tmp_path)
    monkeypatch.chdir(tmp_path)
    cdf_utils.filtered_orbits_cache.clear()
    cdf_utils.orbit_column_cache.clear()
    res = FAST_plot_spectrograms_directory("./FAST_data", output_base="./FAST_plots/", y_scale="log", z_scale=z_scale,
                                           colormap="cividis", max_processing_percentile=percentile, max_workers=2,
                                           progress_json_path="./progress.json")
    assert res and all(r["status"] == "ok" for r in res), res
    prog = json.load(open("./progress.json"))
    assert prog[f"log_{z_scale}_error_plotting"] == []
    extrema = json.load(open("./FAST_calculated_extrema.json")) if percentile is not None else None

    host_tiles = {}

    def host_writer(ctx, d_rgba_ptr, jobs, max_workers=1, dpi=None, **_kw):
        for path, fig in jobs:
            for ax in fig.axes:
                for img in ax.images:
                    if isinstance(img.rgba, DeviceRaster):
                        img.rgba = _download(ctx, d_rgba_ptr, img.rgba)
            fig.savefig(path, dpi=dpi)
            host_tiles[os.path.basename(path)] = fig.tiles(dpi)

    monkeypatch.setattr(process_orbit, "write_figures_device", host_writer)
    files = discover_orbit_files("./FAST_data", ORDER)
    checked = mapped = 0
    for orbit in (13000, 13002):
        r = process_orbit.FAST_process_single_orbit(orbit, files[orbit], load_filtered_orbits(), 6, "log", z_scale, ORDER,
                                                    "cividis", "./host_out/", global_extrema=extrema)
        assert r["status"] == "ok", r
        names = sorted(os.listdir(f"./host_out/2000/01/{orbit}"))
        assert names and all(f"_y-log_z-{z_scale}_" in n for n in names), names
        for name in names:
            dev = png.decode_rgba(open(f"./FAST_plots/2000/01/{orbit}/{name}", "rb").read())
            host = png.decode_rgba(open(f"./host_out/2000/01/{orbit}/{name}", "rb").read())
            assert np.array_equal(dev, host), name
            mapped += _check_rows_against_cpu_map(host_tiles[name], dev)
            checked += 1
    assert checked >= 4 and mapped >= checked
