"""Panels on a log energy axis (``y_scale="log"``), host side: the row map that places a panel's evenly spaced
rows through the log transform, the composer and content rows that use it, and the log axis' ticks."""

import math

import numpy as np
import pytest

from configurable_spectrograms_b200 import figure as F
from configurable_spectrograms_b200._lib import TILE_ROW_MAP
from configurable_spectrograms_b200.overlay import ATLAS
from configurable_spectrograms_b200.plotting import draw_panel

FAST_NE, FAST_LO, FAST_HI = 74, 4.0, 4000.0


def _independent_map(ne, h, y_lo, y_hi):
    """Row k covers the data interval [y_lo + k dy, y_lo + (k + 1) dy]; on screen it sits between the logs of
    its ends.  Every pixel centre is looked up among those edges.  Returns (map, number of centres within 1e-9
    of an edge, in axis fraction)."""
    dy = (y_hi - y_lo) / ne
    l0, l1 = math.log10(y_lo), math.log10(y_hi)
    edges = (np.log10(y_lo + np.arange(ne + 1) * dy) - l0) / (l1 - l0)  # increasing for either orientation
    centres = (h - np.arange(h) - 0.5) / h  # canvas row 0 is the top
    k = np.clip(np.searchsorted(edges, centres, side="right") - 1, 0, ne - 1)
    near = np.abs(centres[:, None] - edges[None, :]).min(axis=1) <= 1e-9
    return k, near


def _fast_box_heights():
    """Box heights of the panels of a FAST grid (4 rows, full + zoom columns, 24 x 12 in) at dpi 100 / 200 / 37."""
    out = {}
    for dpi in (100, 200, 37):
        fig = _grid(["log"] * 8, ne=FAST_NE, nt=30)
        t = fig.tiles(dpi)
        out[dpi] = sorted({r[6] for k, r in enumerate(t.records) if k in t.sources})
    return out


def _raster(ne, nt, seed=0):
    """Every row its own colour band, so that any misplaced row shows."""
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (ne, nt, 4), dtype=np.uint8)
    img[..., 0] = (np.arange(ne) * 7 % 256)[:, None]
    img[..., 3] = 255
    return img


def _grid(scales, ne=FAST_NE, nt=60, y=(FAST_LO, FAST_HI), n_cols=2, seed=0):
    """A FAST-shaped grid (panels drawn by ``plotting.draw_panel``) with the given y scale per panel."""
    n_rows = len(scales) // n_cols
    fig = F.SpectrogramFigure(figsize=(12 * n_cols, 3 * n_rows))
    for k, scale in enumerate(scales):
        ax = fig.add_subplot(n_rows, n_cols, k + 1)
        x = (10957.0, 10957.0 + nt * 2.5 / 86400.0)
        ax.set_xlim(*x)
        draw_panel(ax, _raster(ne, nt, seed + k), None, 1.0, 100.0, True, x, np.array(y), y_axis_scale_function=scale,
                   colormap="turbo", instrument_label=f"panel {k}")
    fig.suptitle("Orbit 13000 - log energy axis")
    return fig


def _panel_records(t):
    return [(k, t.records[k]) for k in sorted(t.sources)]


# ------------------------------------------------------------------------------------------ the row map
def test_row_map_matches_the_log_transform_on_fast_geometry():
    heights = _fast_box_heights()
    assert all(len(h) == 1 and h[0] > 8 for h in heights.values())
    for dpi, (h,) in heights.items():
        for lo, hi in ((FAST_LO, FAST_HI), (FAST_HI, FAST_LO)):
            want, near = _independent_map(FAST_NE, h, lo, hi)
            key, got = F.log_row_map(FAST_NE, h, lo, hi)
            assert key == (FAST_NE, h, lo, hi) and got.dtype == np.int32 and got.shape == (h,)
            assert near.sum() == 0, (dpi, lo, hi)
            assert np.array_equal(got, want), (dpi, lo, hi)
        # the warp the reference shows: the lowest row fills a large part of the panel, the upper half of the
        # rows shares a thin band at the top
        got = F.log_row_map(FAST_NE, h, FAST_LO, FAST_HI)[1]
        assert np.count_nonzero(got == 0) > 0.3 * h
        assert np.count_nonzero(got >= FAST_NE // 2) < 0.15 * h
        assert got[-1] == 0 and np.all(np.diff(got) <= 0)


@pytest.mark.parametrize("ne, h, lo, hi", [
    (400, 97, 4.0, 4000.0),      # more rows than pixels: some rows get no pixel
    (74, 1, 4.0, 4000.0),        # a box one pixel high
    (1, 50, 4.0, 4000.0),        # one row
    (1, 1, 10.0, 20.0),
    (30, 211, 4.1, 4.9),         # narrower than one decade
    (16, 333, 1e-3, 1e5),
])
def test_row_map_edge_cases(ne, h, lo, hi):
    want, near = _independent_map(ne, h, lo, hi)
    got = F.log_row_map(ne, h, lo, hi)[1]
    assert got.min() >= 0 and got.max() <= ne - 1
    same = got == want
    assert np.all(same | near), np.flatnonzero(~same & ~near)
    if ne > h:
        assert len(np.unique(got)) <= h < ne


def _mapped_tiles(fig, dpi):
    t = fig.tiles(dpi)
    return t, [(k, r) for k, r in _panel_records(t) if r[9] & TILE_ROW_MAP]


@pytest.mark.parametrize("extent", [(100.0, 100.0), (0.0, 4000.0), (-5.0, 4000.0), (4000.0, 0.0)])
def test_fallback_keeps_linear_rows(extent):
    """An empty or non-positive extent, or a single row, has no log warp to show: the rows stay evenly spaced,
    the image is what a linear axis with the same ticks shows."""
    for ne, y in ((12, extent), (1, (4.0, 4000.0))):
        fig = _grid(["log", "log"], ne=ne, y=y, n_cols=1)
        t, mapped = _mapped_tiles(fig, 100)
        assert mapped == [] and t.row_maps == []
        img = fig.compose(100)
        for k, rec in _panel_records(t):
            off, pne, nt, x, y0, w, h = rec[:7]
            src = t.sources[k]
            want = src[pne - 1 - F.nearest_index(h, pne)][:, F.nearest_index(w, nt)]
            assert np.array_equal(img[y0 : y0 + h, x : x + w], want)


# ------------------------------------------------------------------------------- compose and content rows
@pytest.mark.parametrize("dpi", [100, 200, 37])
def test_compose_warps_log_panels_and_content_rows_cover_every_change(dpi):
    fig = _grid(["log", "linear", "log", "log"], n_cols=2, seed=dpi)
    fig.axes[3].images[-1].extent = (*fig.axes[3].images[-1].extent[:2], 4000.0, 4.0)  # an axis running downwards
    t = fig.tiles(dpi)
    img = fig.compose(dpi)
    panels = _panel_records(t)
    assert [bool(r[9] & TILE_ROW_MAP) for _k, r in panels] == [True, False, True, True]
    for ax, (k, (off, ne, nt, x, y, w, h, _a, _b, flags, _m)) in zip(fig.axes, panels):
        src = t.sources[k]
        if flags & TILE_ROW_MAP:
            ex = ax.images[-1].extent
            rows = F.log_row_map(ne, h, float(ex[2]), float(ex[3]))[1]
            assert np.array_equal(t.map_of(k)[1], rows)
        else:
            rows = ne - 1 - F.nearest_index(h, ne)
        assert np.array_equal(img[y : y + h, x : x + w], src[rows][:, F.nearest_index(w, nt)]), k
    _check_content_rows(t, img)


def _check_content_rows(t, img):
    rows = t.content_rows()
    assert rows[0] == 0 and np.all(np.diff(rows) > 0) and rows[-1] < t.H
    listed = np.zeros(t.H, dtype=bool)
    listed[rows] = True
    changed = np.flatnonzero(np.any(img[1:] != img[:-1], axis=(1, 2))) + 1
    assert listed[changed].all(), changed[~listed[changed]]


@pytest.mark.parametrize("first", ["linear", "log"])
def test_content_rows_cache_tells_log_from_linear(first):
    """A log panel and a linear panel of the same geometry (same tiles, same ticks) change rows in different
    places: neither may be handed the other's content rows from the caches."""
    F._content_rows_cache.clear()
    F._change_rows_cache.clear()

    def build(scale):
        fig = F.SpectrogramFigure(figsize=(8, 3))
        ax = fig.add_subplot(1, 1, 1)
        ax.set_xlim(0.0, 1.0)
        ax.imshow(_raster(30, 40, 5), extent=(0.0, 1.0, 4.1, 4.9))  # no decade and no m * 10^k inside: no ticks
        ax.set_yticks([])
        ax.set_yscale(scale)
        return fig

    order = [first, "log" if first == "linear" else "linear"]
    tables = {}
    for scale in order:
        fig = build(scale)
        t = fig.tiles(100)
        tables[scale] = t.table()
        _check_content_rows(t, fig.compose(100))
    a, b = tables["linear"], tables["log"]
    for field in ("y", "h", "ne", "x", "w"):
        assert np.array_equal(a[field], b[field]), field  # the geometry the caches key on is the same
    assert (b["flags"] & TILE_ROW_MAP).any() and not (a["flags"] & TILE_ROW_MAP).any()


def test_table_places_maps_at_the_given_offsets():
    fig = _grid(["log", "log", "linear", "log"], n_cols=2)
    fig.axes[2].images[-1].extent = (*fig.axes[2].images[-1].extent[:2], 10.0, 1000.0)
    fig.axes[2].set_yscale("log")
    t = fig.tiles(100)
    assert len(t.row_maps) == 2  # the panels of one extent and height share a map
    own = t.table()
    mapped = np.flatnonzero(own["flags"] & TILE_ROW_MAP)
    concat = np.concatenate([m[1] for m in t.row_maps])
    for k in mapped:
        assert np.array_equal(concat[own["row_map"][k] : own["row_map"][k] + own["h"][k]], t.map_of(int(k))[1])
    placed = t.table([1000, 5])
    assert sorted(set(placed["row_map"][mapped].tolist())) == [5, 1000]
    assert np.array_equal(placed[own["flags"] & TILE_ROW_MAP == 0], own[own["flags"] & TILE_ROW_MAP == 0])


# ---------------------------------------------------------------------------------------------- ticks
def _tick_rows(t, x_right, length, line_w):
    """Canvas rows of the tick marks of `length` pixels that end at the box's left frame."""
    solid = ATLAS.solid((0, 0, 0, 255))[0]
    return sorted(r[4] for r in t.records if r[0] == solid and r[9] & 1 and r[3] == x_right - length and r[5] == length
                  and r[6] == line_w)


@pytest.mark.parametrize("dpi", [100, 200, 37])
def test_log_axis_ticks_sit_on_the_log_transform(dpi):
    pt = dpi / 72.0
    major, minor, line_w = max(2, round(8 * pt)), max(1, round(5 * pt)), max(1, round(0.8 * pt))
    fig = _grid(["log", "linear"], n_cols=1)
    t = fig.tiles(dpi)
    (k_log, rec_log), (k_lin, rec_lin) = _panel_records(t)
    for rec, scale in ((rec_log, "log"), (rec_lin, "linear")):
        bx, by, bh = rec[3], rec[4], rec[6]
        x_right = bx - line_w
        l0, l1 = math.log10(FAST_LO), math.log10(FAST_HI)

        def on_transform(rows, values):  # each mark's top row is its centre's position, rounded
            exact = sorted(by + bh - (math.log10(v) - l0) / (l1 - l0) * bh - line_w / 2 for v in values)
            return len(rows) == len(exact) and all(abs(r - e) <= 0.5 for r, e in zip(rows, exact))

        in_box = [r for r in _tick_rows(t, x_right, minor, line_w) if by - line_w <= r <= by + bh]
        if scale == "log":
            want_minor = [m * 10.0**e for e in range(0, 4) for m in range(2, 10) if FAST_LO <= m * 10.0**e <= FAST_HI]
            assert len(want_minor) == 25
            assert on_transform(in_box, want_minor), in_box
            majors = [r for r in _tick_rows(t, x_right, major, line_w) if by - line_w <= r <= by + bh]
            assert on_transform(majors, (10.0, 100.0, 1000.0)), majors
        else:
            assert in_box == []


def test_minor_tick_rule():
    assert F.log_minor_ticks(4.0, 40.0) == [4.0, 5.0, 6.0, 7.0, 8.0, 9.0, 20.0, 30.0, 40.0]
    assert F.log_minor_ticks(40.0, 4.0) == F.log_minor_ticks(4.0, 40.0)
    assert F.log_minor_ticks(4.1, 4.9) == []
    assert len(F.log_minor_ticks(1.0, 1e10)) == 80  # floor(10) - ceil(0) = 10 decades: still ticked
    assert F.log_minor_ticks(1.0, 1e11) == [] and F.log_minor_ticks(0.5, 1e10) != []  # 11 decades: none
    assert F.log_minor_ticks(0.0, 10.0) == [] and F.log_minor_ticks(5.0, 5.0) == []
