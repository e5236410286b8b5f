"""Figures at display resolution: the stand-in for the matplotlib objects the reference draws into.

The reference hands every panel to ``Axes.imshow(aspect="auto")`` and lets Agg resample it into the axes
box, draw ticks, labels, colour bars and markers, and composite the figure at ``figsize x dpi`` pixels
(``plotting.py:280-387,606-611``; 24 x 12 in at 200 dpi = 4800 x 2400 for the FAST grids,
``fast/process_orbit.py:110``).  Here a figure is a list of *tiles* (``csg_png_tile``): every panel is a
finished RGBA raster (K3) stretched nearest-neighbour over its image rectangle, every annotation a sprite
of ``overlay.ATLAS`` -- rendered text at its own size, or one pixel / one colour ramp stretched into a
line, a frame edge, a colour bar.  The same tile list is

* evaluated by :meth:`SpectrogramFigure.compose` in numpy (the oracle, and ``savefig`` for figures whose
  rasters are host arrays), and
* composed + DEFLATE-encoded on the device by ``png.encode_figures_device`` (``csrc/png.cu``) for figures
  whose panels stay in HBM (:class:`DeviceRaster`) -- pixel for pixel the same image.

The layout is this package's own (margins from the rendered label sizes, one colour bar per panel at a
twentieth of the box height, ticks on "nice" times of day); it follows the reference's figure sizes, fonts
and content, not matplotlib's ``tight_layout`` arithmetic.  The classes are duck-typed like their
matplotlib namesakes so the mirrored functions (``plotting.make_spectrogram`` ...) and ``cusp_marking``
read like the reference's.
"""

from __future__ import annotations

import itertools
import math
from datetime import datetime, timedelta, timezone

import numpy as np

from . import png
from ._lib import PNG_TILE, TILE_OVERLAY, TILE_ROW_MAP, TILE_TOP_ORIGIN
from .overlay import ATLAS

_COLORS = {
    "black": (0, 0, 0, 255),
    "red": (255, 0, 0, 255),
    "white": (255, 255, 255, 255),
    "blue": (0, 0, 255, 255),
    "green": (0, 128, 0, 255),
    "gray": (128, 128, 128, 255),
}
_BACKGROUND = (255, 255, 255, 255)
DEFAULT_DPI = 100


def _rgba(color) -> tuple[int, int, int, int]:
    if isinstance(color, str):
        return _COLORS.get(color, (0, 0, 0, 255))
    c = tuple(color)
    if all(0.0 <= float(v) <= 1.0 for v in c):
        c = tuple(int(round(float(v) * 255)) for v in c)
    return (int(c[0]), int(c[1]), int(c[2]), int(c[3]) if len(c) > 3 else 255)


def nearest_index(n_dst: int, n_src: int) -> np.ndarray:
    """Source index of every destination pixel, nearest neighbour on pixel centres:
    ``floor((d + 0.5) * n_src / n_dst)`` evaluated in float32 exactly like ``csrc/png.cu``."""
    scale = np.float32(n_src) / np.float32(n_dst)
    k = ((np.arange(n_dst, dtype=np.float32) + np.float32(0.5)) * scale).astype(np.int64)
    return np.minimum(k, n_src - 1)


_change_rows_cache: dict = {}
_content_rows_cache: dict = {}
_row_map_cache: dict = {}


def log_row_map(ne: int, h: int, y_lo: float, y_hi: float) -> tuple:
    """``(key, map)``: the storage row (0 = the extent's ``y_lo`` end) that every canvas row of a panel ``h``
    pixels high shows when its ``ne`` evenly spaced rows are drawn on a log axis from ``y_lo`` (bottom) to
    ``y_hi`` (top), the way Agg resamples ``imshow`` through ``set_yscale("log")``.  Canvas row ``d`` (0 = top)
    is sampled at its centre, ``f = (h - d - 0.5) / h`` of the way up, in float64.  Cached: the panels of a
    grid share one map, and ``key`` names it in the content-row caches."""
    key = (int(ne), int(h), float(y_lo), float(y_hi))
    hit = _row_map_cache.get(key)
    if hit is None:
        f = (h - np.arange(h, dtype=np.float64) - 0.5) / h
        l0, l1 = math.log10(y_lo), math.log10(y_hi)
        value = 10.0 ** (l0 + f * (l1 - l0))
        k = np.floor((value - y_lo) / (y_hi - y_lo) * ne)
        rows = np.clip(k, 0, ne - 1).astype(np.int32)
        rows.flags.writeable = False
        if len(_row_map_cache) > 4096:
            _row_map_cache.clear()
        hit = _row_map_cache[key] = (key, rows)
    return hit


def _change_rows(ne: int, h: int, row_map: tuple | None = None) -> np.ndarray:
    """Destination rows (0-based, inside a tile ``h`` pixels high) at which the source row changes: nearest
    neighbour, or the rows of ``row_map`` (a :func:`log_row_map`)."""
    key = (ne, h) if row_map is None else (ne, h, row_map[0])
    hit = _change_rows_cache.get(key)
    if hit is None:
        idx = nearest_index(h, ne) if row_map is None else row_map[1]
        hit = _change_rows_cache[key] = np.concatenate([[0], np.flatnonzero(np.diff(idx)) + 1]).astype(np.int32)
        if len(_change_rows_cache) > 4096:
            _change_rows_cache.clear()
    return hit


class _Label:
    def __init__(self):
        self.text, self.fontsize, self.rotation = "", None, None

    def set_fontsize(self, size):
        self.fontsize = size


class _AxisSide:
    def __init__(self):
        self.label = _Label()
        self.major_formatter = None

    def set_major_formatter(self, formatter):
        self.major_formatter = formatter


class DeviceRaster:
    """A panel that stays in HBM: where its RGBA raster lives in a batch's ``d_rgba`` buffer
    (pixel offset, energies, time steps).  Stands in for the host array in ``imshow``; figures made
    of such panels are composed and PNG-encoded on the device (``png.encode_figures_device``)."""

    __slots__ = ("offset", "ne", "nt")

    def __init__(self, offset: int, ne: int, nt: int):
        self.offset, self.ne, self.nt = int(offset), int(ne), int(nt)

    @property
    def shape(self):
        return (self.ne, self.nt, 4)

    @property
    def size(self):
        return self.ne * self.nt * 4


class RasterImage:
    """What ``imshow`` returned: one colour-mapped panel."""

    def __init__(self, rgba, index, extent, cmap, vmin, vmax, norm):
        self.rgba, self.index, self.extent = rgba, index, extent
        self.cmap, self.vmin, self.vmax, self.norm = cmap, vmin, vmax, norm


class Colorbar:
    """A colour bar beside its panel: ramp of the panel's colormap, ticks, label."""

    def __init__(self, image, label, ticks=None, fmt=None):
        self.image, self.label, self.ticks, self.format = image, label, ticks, fmt
        self.ax = PanelAxes(None)  # the tick_params / set_ylabel calls the reference makes on cbar.ax


class PanelAxes:
    """One subplot: a raster, its axes metadata and the marker primitives drawn on top."""

    def __init__(self, figure):
        self.figure = figure
        self.images: list[RasterImage] = []
        self.lines: list[dict] = []
        self.texts: list[dict] = []
        self.xaxis, self.yaxis = _AxisSide(), _AxisSide()
        self.title, self.title_fontsize = "", None
        self._xlim = (0.0, 1.0)
        self.yticks = None
        self.yticklabels = None
        self.yscale = "linear"
        self.tick_labelsize = None
        self.tick_length = None
        self.minor_tick_length = None
        self.colorbar: Colorbar | None = None
        self.row_label_pad = 0

    # -- the Axes calls the path makes (plotting.py:234-387, cusp_marking.py)
    def imshow(self, rgba, aspect="auto", origin="lower", extent=None, cmap=None, norm=None, vmin=None, vmax=None,
               index=None):
        """Store an already colour-mapped (E', T', 4) uint8 raster (row 0 = lowest energy)."""
        img = RasterImage(rgba if isinstance(rgba, DeviceRaster) else np.asarray(rgba), index, extent, cmap, vmin, vmax, norm)
        self.images.append(img)
        return img

    def set_xlim(self, left, right):
        self._xlim = (float(left), float(right))

    def get_xlim(self):
        return self._xlim

    def set_xlabel(self, text, **kw):
        self.xaxis.label.text = text
        if "fontsize" in kw:
            self.xaxis.label.fontsize = kw["fontsize"]

    def set_ylabel(self, text, **kw):
        self.yaxis.label.text = text
        if "fontsize" in kw:
            self.yaxis.label.fontsize = kw["fontsize"]
        if "labelpad" in kw:
            self.row_label_pad = kw["labelpad"]

    def set_title(self, text, **kw):
        self.title = text
        if "fontsize" in kw:
            self.title_fontsize = kw["fontsize"]

    def set_yticks(self, ticks):
        self.yticks = list(ticks)

    def set_yticklabels(self, labels):
        self.yticklabels = list(labels)

    def set_yscale(self, scale):
        self.yscale = scale

    def tick_params(self, **kw):
        if kw.get("which", "major") == "major":
            self.tick_labelsize = kw.get("labelsize", self.tick_labelsize)
            self.tick_length = kw.get("length", self.tick_length)
        elif kw["which"] == "minor":
            self.minor_tick_length = kw.get("length", self.minor_tick_length)

    def axvline(self, x, **kw):
        line = {"kind": "vline", "x": float(x), **kw}
        self.lines.append(line)
        return line

    def plot(self, xs, ys, **kw):
        line = {"kind": "polyline", "x": [float(v) for v in xs], "y": [float(v) for v in ys], **kw}
        self.lines.append(line)
        return (line,)

    def text(self, x, y, s, **kw):
        entry = {"x": float(x), "y": float(y), "text": s, **kw}
        self.texts.append(entry)
        return entry

    def get_xaxis_transform(self):
        return "xaxis"  # x in data units, y in axes fraction


class FigureCanvas:
    def __init__(self, figure):
        self.figure = figure
        figure.canvas = self


# --------------------------------------------------------------------------------------------
# tick choices
# --------------------------------------------------------------------------------------------
_TIME_STEPS = (1, 2, 5, 10, 15, 30, 60, 120, 300, 600, 900, 1800, 3600, 7200, 10800, 21600, 43200, 86400)


def time_ticks(left_days: float, right_days: float, max_ticks: int = 7):
    """Tick positions (days since 1970, the x unit of the path) on round times of day."""
    span = (right_days - left_days) * 86400.0
    if not (span > 0) or not math.isfinite(span):
        return []
    step = next((s for s in _TIME_STEPS if span / s <= max_ticks), 86400 * math.ceil(span / 86400 / max_ticks))
    first = math.ceil(left_days * 86400.0 / step - 1e-9) * step
    out, t = [], first
    while t <= right_days * 86400.0 + 1e-6 and len(out) < 64:
        out.append(t / 86400.0)
        t += step
    return out


def _format_time(days: float, fmt: str) -> str:
    return (datetime(1970, 1, 1, tzinfo=timezone.utc) + timedelta(seconds=round(days * 86400.0))).strftime(fmt)


def linear_ticks(lo: float, hi: float, max_ticks: int = 6):
    if not (math.isfinite(lo) and math.isfinite(hi)) or hi <= lo:
        return []
    raw = (hi - lo) / max_ticks
    mag = 10.0 ** math.floor(math.log10(raw))
    step = next(m * mag for m in (1, 2, 5, 10) if m * mag >= raw)
    first = math.ceil(lo / step - 1e-9) * step
    return [first + k * step for k in range(int((hi - first) / step + 1e-9) + 1)]


def log_minor_ticks(lo: float, hi: float) -> list[float]:
    """Unlabelled minor ticks of a log axis, ``LogLocator(subs="auto")``: ``m * 10**k`` (m = 2..9) inside
    ``[lo, hi]``, none when the axis covers more than 10 decades (matplotlib's ``numdec > 10``)."""
    lo, hi = min(lo, hi), max(lo, hi)
    if not (lo > 0 and math.isfinite(hi)) or lo == hi:
        return []
    if math.floor(math.log10(hi)) - math.ceil(math.log10(lo)) > 10:
        return []
    decades = range(math.floor(math.log10(lo)), math.floor(math.log10(hi)) + 1)
    return [m * 10.0**k for k in decades for m in range(2, 10) if lo <= m * 10.0**k <= hi]


def _format_number(v: float) -> str:
    if v == 0:
        return "0"
    if abs(v) >= 1e4 or abs(v) < 1e-2:
        mant, exp = f"{v:.1e}".split("e")
        mant = mant.rstrip("0").rstrip(".")
        return f"{mant}e{int(exp)}" if mant != "1" else f"1e{int(exp)}"
    return f"{v:g}"


_OVERLAY_FLAGS = TILE_OVERLAY | TILE_TOP_ORIGIN


class FigureTiles:
    """The tile list of one figure: what both composers consume."""

    __slots__ = ("W", "H", "records", "sources", "background", "row_maps")

    def __init__(self, W, H, background):
        self.W, self.H, self.background = int(W), int(H), background
        self.records: list[tuple] = []  # PNG_TILE fields, in drawing priority (the first tile covering a pixel wins)
        self.sources: dict = {}         # record index -> DeviceRaster | ndarray, for the panel rasters
        self.row_maps: list[tuple] = []  # the distinct log_row_map()s of the panels; a TILE_ROW_MAP record's
        # last field is its index here until table() turns it into an offset

    def sprite(self, ref, x, y, w=None, h=None):
        off, sh, sw = ref
        w, h = sw if w is None else w, sh if h is None else h
        if w <= 0 or h <= 0:
            return
        x = min(max(int(x), 0), max(self.W - w, 0))
        y = min(max(int(y), 0), max(self.H - h, 0))
        self.records.append((off, sh, sw, x, y, min(w, self.W - x), min(h, self.H - y), 0, 0, _OVERLAY_FLAGS, 0))

    def rect(self, color, x, y, w, h):
        """A filled rectangle (clipped to the canvas)."""
        x0, y0 = max(int(x), 0), max(int(y), 0)
        x1, y1 = min(int(x) + int(w), self.W), min(int(y) + int(h), self.H)
        if x1 > x0 and y1 > y0:
            self.records.append((ATLAS.solid(color)[0], 1, 1, x0, y0, x1 - x0, y1 - y0, 0, 0, _OVERLAY_FLAGS, 0))

    def raster(self, source, ne, nt, x, y, w, h, row_map=None):
        """A panel; ``row_map`` (a :func:`log_row_map` of height ``h``) places its rows instead of the nearest
        row and the origin="lower" flip."""
        if w <= 0 or h <= 0 or ne <= 0 or nt <= 0:
            return
        off = source.offset if isinstance(source, DeviceRaster) else 0
        flags = slot = 0
        if row_map is not None:
            keys = [m[0] for m in self.row_maps]
            if row_map[0] not in keys:
                self.row_maps.append(row_map)
                keys.append(row_map[0])
            flags, slot = TILE_ROW_MAP, keys.index(row_map[0])
        self.sources[len(self.records)] = source
        self.records.append((off, ne, nt, int(x), int(y), int(w), int(h), 0, 0, flags, slot))

    def map_of(self, k: int) -> tuple:
        """The row map of record ``k`` (a TILE_ROW_MAP tile)."""
        return self.row_maps[self.records[k][10]]

    def table(self, map_offsets=None) -> np.ndarray:
        """The records as ``PNG_TILE`` rows.  A TILE_ROW_MAP tile's ``row_map`` is the offset of its map in the
        concatenation of ``row_maps``, or ``map_offsets[i]`` for map ``i`` when the caller places them."""
        if not self.records:
            return np.zeros(0, dtype=PNG_TILE)
        # (a structured array straight from the tuples is built field by field per record: 3x slower)
        n_fields = len(PNG_TILE.names)
        flat = np.fromiter(itertools.chain.from_iterable(self.records), dtype=np.int64, count=len(self.records) * n_fields)
        flat = flat.reshape(len(self.records), n_fields)
        out = np.empty(len(flat), dtype=PNG_TILE)
        out["rgba_off"] = flat[:, 0]
        out.view(np.int32).reshape(len(flat), PNG_TILE.itemsize // 4)[:, 2:] = flat[:, 1:]
        if self.row_maps:
            if map_offsets is None:
                map_offsets = np.cumsum([0] + [len(m[1]) for m in self.row_maps[:-1]])
            mapped = (out["flags"] & TILE_ROW_MAP) != 0
            out["row_map"][mapped] = np.asarray(map_offsets, dtype=np.int64)[out["row_map"][mapped]]
        return out

    def content_rows(self, table: np.ndarray | None = None) -> np.ndarray:
        """Ascending scanlines whose content may differ from the line above: where a tile starts, ends or
        moves on to another source row (the device encodes these; the runs in between repeat)."""
        t = self.table() if table is None else table
        # rows depend on the vertical geometry only, which the figures of one kind share -- and on the row map
        # of every panel on a log axis (a linear panel of the same geometry changes rows elsewhere)
        mapped = np.flatnonzero(t["flags"] & TILE_ROW_MAP) if self.row_maps else np.zeros(0, np.int64)
        maps = tuple((int(k), self.map_of(int(k))[0]) for k in mapped)
        key = (self.H, t["y"].tobytes(), t["h"].tobytes(), t["ne"].tobytes(), maps) if len(t) else (self.H,)
        hit = _content_rows_cache.get(key)
        if hit is not None:
            return hit
        mark = np.zeros(self.H + 2, dtype=bool)
        mark[0] = True
        if len(t):
            y, h, ne = t["y"].astype(np.int64), t["h"].astype(np.int64), t["ne"].astype(np.int64)
            mark[np.minimum(y, self.H)] = True
            mark[np.minimum(y + h, self.H)] = True
            for k in mapped:
                rows = _change_rows(int(ne[k]), int(h[k]), self.map_of(int(k))) + int(y[k])
                mark[rows[rows <= self.H]] = True
            h = h.copy()
            h[mapped] = -1  # handled above
            one_to_one = (ne == h) & (h > 1)
            if one_to_one.any():  # sprites at their own size: every row is new (+1 / -1 over their spans)
                delta = np.zeros(self.H + 2, dtype=np.int32)
                np.add.at(delta, np.minimum(y[one_to_one], self.H), 1)
                np.add.at(delta, np.minimum(y[one_to_one] + h[one_to_one], self.H), -1)
                mark[:-1] |= np.cumsum(delta[:-1]) > 0
            for k in np.flatnonzero((ne != h) & (ne > 1) & (h > 0)):  # resampled rasters and ramps: a few per figure
                rows = _change_rows(int(ne[k]), int(h[k])) + int(y[k])
                mark[rows[rows <= self.H]] = True
        rows = np.flatnonzero(mark[: self.H]).astype(np.int32)
        if len(_content_rows_cache) > 256:
            _content_rows_cache.clear()
        _content_rows_cache[key] = rows
        return rows


_static_blocks: dict = {}
_tick_blocks: dict = {}  # time / colour-bar tick marks and labels, relative to their box: (tiles, extent)


def _extent(block) -> tuple[int, int, int, int]:
    """``(x min, y min, x max, y max)`` of a block of ``(off, ne, nt, x, y, w, h)`` tiles: when the shifted
    extent lies inside the canvas, none of the tiles needs clamping."""
    if not block:
        return (0, 0, 0, 0)
    return (min(t[3] for t in block), min(t[4] for t in block), max(t[3] + t[5] for t in block), max(t[4] + t[6] for t in block))


def _place(records, block, extent, ox, oy, W, H):
    """Append ``block`` shifted by (ox, oy); tiles are moved inside the canvas only when the block leaves it."""
    if extent[0] + ox >= 0 and extent[1] + oy >= 0 and extent[2] + ox <= W and extent[3] + oy <= H:
        records.extend([(o, a, b, x + ox, y + oy, w, h, 0, 0, _OVERLAY_FLAGS, 0) for o, a, b, x, y, w, h in block])
        return
    for o, a, b, x, y, w, h in block:
        x, y = min(max(x + ox, 0), max(W - w, 0)), min(max(y + oy, 0), max(H - h, 0))
        records.append((o, a, b, x, y, min(w, W - x), min(h, H - y), 0, 0, _OVERLAY_FLAGS, 0))
ATLAS.on_clear(lambda: (_static_blocks.clear(), _tick_blocks.clear()))  # both hold sprite offsets


def _static_block(ax: "PanelAxes", img: RasterImage, cw: int, ch: int, pt: float, pad: int, y_lo: float, y_hi: float, title_h: int = 0):
    """``(tiles, geometry)`` of a subplot's figure-independent part, relative to the cell's top-left corner:
    tiles as ``(rgba_off, ne, nt, x, y, w, h, flags)``; geometry = ``(box x, box y, box w, box h, tick label px,
    tick length, line width, colour-bar x, colour-bar width, colour-bar tick label px)`` or ``None`` when the
    cell leaves no room for a box.  The margins come from the rendered sizes of the labels; the room kept for
    the (per-figure) time and colour-bar tick labels is that of a five-digit label."""
    black = (0, 0, 0, 255)
    tick_px = max(6, int(round((ax.tick_labelsize or 10) * pt)))
    tick_len = max(2, int(round((ax.tick_length or 4) * pt)))
    minor_len = max(1, int(round((ax.minor_tick_length or 2) * pt)))
    line_w = max(1, int(round(0.8 * pt)))
    solid = ATLAS.solid(black)[0]
    tiles: list[tuple] = []

    def rect(x, y, w, h):
        if w > 0 and h > 0:
            tiles.append((solid, 1, 1, int(x), int(y), int(w), int(h), _OVERLAY_FLAGS))

    def sprite(ref, x, y, w=None, h=None):
        tiles.append((ref[0], ref[1], ref[2], max(int(x), 0), max(int(y), 0), ref[2] if w is None else int(w),
                      ref[1] if h is None else int(h), _OVERLAY_FLAGS))

    def label_px(label, default=10):
        return max(6, int(round((label.fontsize or default) * pt)))

    ylabel = ATLAS.text(ax.yaxis.label.text, label_px(ax.yaxis.label), rotate=True) if ax.yaxis.label.text else None
    xlabel = ATLAS.text(ax.xaxis.label.text, label_px(ax.xaxis.label)) if ax.xaxis.label.text else None
    log_y = ax.yscale == "log" and y_lo > 0 and y_hi > 0 and y_lo != y_hi
    if ax.yticks is not None:
        yt = [float(v) for v in ax.yticks]
        yl = list(ax.yticklabels) if ax.yticklabels is not None else [_format_number(v) for v in yt]
    elif log_y:
        yt = [10.0 ** k for k in range(math.ceil(math.log10(min(y_lo, y_hi)) - 1e-9), math.floor(math.log10(max(y_lo, y_hi)) + 1e-9) + 1)]
        yl = [_format_number(v) for v in yt]
    else:
        yt = linear_ticks(min(y_lo, y_hi), max(y_lo, y_hi))
        yl = [_format_number(v) for v in yt]
    y_refs = [ATLAS.text(str(s), tick_px) for s in yl]
    cb = ax.colorbar
    cb_px, cb_label, cb_room = tick_px, None, 0
    if cb is not None:
        cb_px = max(6, int(round((cb.ax.tick_labelsize or ax.tick_labelsize or 10) * pt)))
        cb_room = ATLAS.text("00000", cb_px)[2]
        text = cb.ax.yaxis.label.text or cb.label
        if text:
            cb_label = ATLAS.text(text, max(6, int(round((cb.ax.yaxis.label.fontsize or ax.yaxis.label.fontsize or 10) * pt))), rotate=True)
    # ---- margins -> the axes box
    m_left = pad + (ylabel[2] + pad if ylabel else 0) + max([r[2] for r in y_refs] or [0]) + pad + tick_len
    m_bottom = tick_len + pad + tick_px + pad + (xlabel[1] + pad if xlabel else 0) + pad
    m_top = pad + (title_h + pad if title_h else 0)  # the title itself changes with every orbit: drawn by the caller
    bh = ch - m_top - m_bottom
    bar_w = cb_gap = 0
    m_right = 2 * pad
    if cb is not None:
        bar_w, cb_gap = max(4, bh // 20), 3 * pad
        m_right = cb_gap + bar_w + tick_len + pad + cb_room + pad + (cb_label[2] + pad if cb_label else 0) + pad
    bx, by, bw = m_left, m_top, cw - m_left - m_right
    if bw < 8 or bh < 8:
        return [], None
    # ---- frame, energy ticks, labels
    rect(bx - line_w, by - line_w, bw + 2 * line_w, line_w)
    rect(bx - line_w, by + bh, bw + 2 * line_w, line_w)
    rect(bx - line_w, by, line_w, bh)
    rect(bx + bw, by, line_w, bh)
    for v, ref in zip(yt, y_refs):
        if log_y:
            f = (math.log10(v) - math.log10(y_lo)) / (math.log10(y_hi) - math.log10(y_lo)) if v > 0 else -1.0
        else:
            f = (v - y_lo) / (y_hi - y_lo) if y_hi != y_lo else 0.0
        py = by + bh - f * bh
        if by - 0.5 <= py <= by + bh + 0.5:
            rect(bx - line_w - tick_len, int(round(py - line_w / 2)), tick_len, line_w)
            sprite(ref, bx - line_w - tick_len - pad - ref[2], int(round(py - ref[1] / 2)))
    if log_y:
        for v in log_minor_ticks(y_lo, y_hi):
            py = by + bh - (math.log10(v) - math.log10(y_lo)) / (math.log10(y_hi) - math.log10(y_lo)) * bh
            rect(bx - line_w - minor_len, int(round(py - line_w / 2)), minor_len, line_w)
    if ylabel:
        sprite(ylabel, pad, int(by + bh / 2 - ylabel[1] / 2))
    if xlabel:
        sprite(xlabel, int(bx + bw / 2 - xlabel[2] / 2), by + bh + line_w + tick_len + pad + tick_px + pad)
    # ---- colour bar: frame, the colormap's ramp (highest value on top), label
    kx = bx + bw + cb_gap
    if cb is not None:
        from .colormaps import get_lut

        rect(kx - line_w, by - line_w, bar_w + 2 * line_w, line_w)
        rect(kx - line_w, by + bh, bar_w + 2 * line_w, line_w)
        rect(kx - line_w, by, line_w, bh)
        rect(kx + bar_w, by, line_w, bh)
        sprite(ATLAS.ramp(get_lut(img.cmap or "viridis")), kx, by, bar_w, bh)
        if cb_label:
            sprite(cb_label, kx + bar_w + line_w + tick_len + pad + cb_room + pad, int(by + bh / 2 - cb_label[1] / 2))
    return tiles, (bx, by, bw, bh, tick_px, tick_len, line_w, kx, bar_w, cb_px)


class SpectrogramFigure:
    """A grid of panels with the Figure calls the path makes (plotting.py:69-87,461-497,606-693)."""

    _next_number = 1

    def __init__(self, figsize=(10, 3)):
        self.figsize = tuple(figsize)
        self.axes: list[PanelAxes] = []
        self._grid: dict[int, tuple[int, int, int]] = {}
        self.colorbars: list[Colorbar] = []
        self.suptitle_text, self.suptitle_fontsize = None, None
        self.texts: list[dict] = []
        self.canvas = None
        self.rect = (0.0, 0.0, 1.0, 1.0)
        self.number = SpectrogramFigure._next_number
        SpectrogramFigure._next_number += 1

    def add_subplot(self, n_rows, n_cols, index):
        ax = PanelAxes(self)
        self.axes.append(ax)
        self._grid[id(ax)] = (int(n_rows), int(n_cols), int(index))
        return ax

    def colorbar(self, image, ax=None, label=None, ticks=None, format=None):
        cb = Colorbar(image, label, ticks, format)
        self.colorbars.append(cb)
        if ax is not None:
            ax.colorbar = cb
        return cb

    def suptitle(self, text, **kw):
        self.suptitle_text, self.suptitle_fontsize = text, kw.get("fontsize")

    def text(self, x, y, s, **kw):
        self.texts.append({"x": x, "y": y, "text": s, **kw})

    def tight_layout(self, rect=None, **kw):
        if rect is not None:
            self.rect = tuple(float(v) for v in rect)

    def subplots_adjust(self, **kw):
        pass  # superseded by tight_layout in every figure of the path

    def delaxes(self, ax):
        if ax in self.axes:
            self.axes.remove(ax)
            self._grid.pop(id(ax), None)

    def clf(self):
        self.axes, self._grid, self.colorbars, self.texts = [], {}, [], []

    # ------------------------------------------------------------------ layout
    def tiles(self, dpi: float | None = None) -> FigureTiles:
        """The figure as tiles on a ``figsize x dpi`` canvas."""
        dpi = float(dpi or DEFAULT_DPI)
        W, H = max(1, int(round(self.figsize[0] * dpi))), max(1, int(round(self.figsize[1] * dpi)))
        out = FigureTiles(W, H, _BACKGROUND)
        pt = dpi / 72.0  # pixels per point
        pad = max(2, int(round(3 * pt)))
        black = (0, 0, 0, 255)
        if not self.axes:
            return out
        n_rows = max(self._grid[id(a)][0] for a in self.axes)
        n_cols = max(self._grid[id(a)][1] for a in self.axes)
        left, bottom, right, top = self.rect
        area_x, area_w = left * W, (right - left) * W
        area_y, area_h = (1.0 - top) * H, (top - bottom) * H
        if self.suptitle_text:
            t_w, t_h, parts = ATLAS.text_parts(self.suptitle_text, int(round((self.suptitle_fontsize or 14) * pt)))
            x0, y0 = max(0, (W - t_w) // 2), max(pad, int(area_y) - t_h - pad) if top < 1.0 else pad
            for ref, dx, dy in parts:
                out.sprite(ref, x0 + dx, y0 + dy)
            if top >= 1.0:
                area_y += t_h + 2 * pad
                area_h -= t_h + 2 * pad
        for entry in self.texts:  # figure text: (x, y) in figure fractions, y from the bottom
            ref = ATLAS.text(entry["text"], int(round(entry.get("fontsize", 10) * pt)), _rgba(entry.get("color", "black")))
            x = entry["x"] * W - (ref[2] / 2 if entry.get("ha") == "center" else (ref[2] if entry.get("ha") == "right" else 0))
            y = (1.0 - entry["y"]) * H - (ref[1] if entry.get("va", "bottom") == "bottom" else (ref[1] / 2 if entry.get("va") == "center" else 0))
            out.sprite(ref, int(round(x)), int(round(y)))
        cell_w, cell_h = area_w / n_cols, area_h / n_rows
        for ax in self.axes:
            r, c, idx = self._grid[id(ax)]
            i, j = (idx - 1) // c, (idx - 1) % c
            self._axes_tiles(out, ax, area_x + j * cell_w, area_y + i * cell_h, cell_w, cell_h, pt, pad, black)
        return out

    def _axes_tiles(self, out: FigureTiles, ax: PanelAxes, cx, cy, cw, ch, pt, pad, black):
        """One subplot as tiles.  Everything that does not change from figure to figure of a batch -- the box
        geometry, frames, energy ticks and their labels, axis labels, the room for the title, the colour bar's frame, ramp
        and label -- is built once per distinct set of settings (``_static_block``) and only shifted to the
        cell; the cusp markers, the time ticks, the colour-bar ticks and the panel itself are per figure."""
        if not ax.images:
            return
        img = ax.images[-1]
        ne, nt = img.rgba.shape[:2]
        if ne * nt == 0:
            return
        cx, cy = int(round(cx)), int(round(cy))
        x_lo, x_hi = ax._xlim
        ex = img.extent if img.extent is not None else (x_lo, x_hi, 0.0, 1.0)
        y_lo, y_hi = float(ex[2]), float(ex[3])
        cb = ax.colorbar
        # (width, height, word sprites): a title changes with every orbit, its words and its height do not
        title = ATLAS.text_parts(ax.title, max(6, int(round((ax.title_fontsize or 12) * pt)))) if ax.title else None
        title_h = title[1] if title else 0
        key = (int(cw), int(ch), pt, pad, ax.tick_labelsize, ax.tick_length, ax.minor_tick_length, ax.yaxis.label.text, ax.yaxis.label.fontsize,
               ax.xaxis.label.text, ax.xaxis.label.fontsize, title_h,
               None if ax.yticks is None else tuple(ax.yticks), None if ax.yticklabels is None else tuple(ax.yticklabels),
               ax.yscale, y_lo, y_hi, cb is not None,
               None if cb is None else (cb.label, cb.ax.yaxis.label.text, cb.ax.yaxis.label.fontsize, cb.ax.tick_labelsize, img.cmap))
        hit = _static_blocks.get(key)
        if hit is None:
            hit = _static_blocks[key] = _static_block(ax, img, int(cw), int(ch), pt, pad, y_lo, y_hi, title_h)
            if len(_static_blocks) > 512:
                _static_blocks.clear()
        block, geo = hit
        if geo is None:
            return  # the cell is too small for a box
        bx, by, bw, bh, tick_px, tick_len, line_w, kx, bar_w, cb_px = geo
        bx, by, kx = bx + cx, by + cy, kx + cx
        span = x_hi - x_lo
        scale = bw / span if span != 0 else 0.0
        records = out.records

        # ---- markers first (the first tile covering a pixel wins): vertical lines, brackets, captions
        for ln in reversed(ax.lines):  # later artists are on top
            colour = _rgba(ln.get("color", "black"))
            lw = max(1, int(round(float(ln.get("linewidth", 1)) * pt)))
            if ln["kind"] == "vline":
                px = bx + (ln["x"] - x_lo) * scale
                if bx <= px <= bx + bw:
                    out.rect(colour, int(round(px - lw / 2)), by, lw, bh)
            else:  # polyline in (data x, axes-fraction y): horizontal / vertical strokes of a bracket
                pts = [(bx + (x - x_lo) * scale, by + (1.0 - y) * bh) for x, y in zip(ln["x"], ln["y"])]
                for (xa, ya), (xb, yb) in zip(pts[:-1], pts[1:]):
                    if abs(xa - xb) < 0.5:
                        out.rect(colour, int(round(xa - lw / 2)), int(round(min(ya, yb))), lw, int(round(abs(ya - yb))) + lw)
                    else:
                        out.rect(colour, int(round(min(xa, xb))), int(round(ya - lw / 2)), int(round(abs(xa - xb))) + lw, lw)
        for t in ax.texts:
            ref = ATLAS.text(t["text"], max(6, int(round((t.get("fontsize") or ax.tick_labelsize or 10) * pt))), _rgba(t.get("color", "black")))
            out.sprite(ref, int(round(bx + (t["x"] - x_lo) * scale - ref[2] / 2)), int(round(by + (1.0 - t["y"]) * bh)))
        # ---- the static block, shifted to this cell
        records.extend([(o, a, b, x + cx, y + cy, w, h, 0, 0, f, 0) for (o, a, b, x, y, w, h, f) in block])
        if title:
            x0 = max(0, int(bx + bw / 2 - title[0] / 2))
            for ref, dx, dy in title[2]:
                out.sprite(ref, x0 + dx, cy + pad + dy)
        # ---- time ticks and colour-bar ticks: positions relative to the box, shared by every panel that shows
        # the same time range / value range at the same size (the rows of a grid; the variants of a figure)
        fmt = ax.xaxis.major_formatter
        x_key = (x_lo, x_hi, fmt, tick_px, bw, line_w, tick_len, pad)
        x_hit = _tick_blocks.get(x_key)
        if x_hit is None:
            solid_black = ATLAS.solid(black)[0]
            if isinstance(fmt, str):  # a time axis (the formatter is the strftime pattern the reference picks)
                xt = time_ticks(x_lo, x_hi)
                xl = [_format_time(v, fmt) for v in xt]
            else:
                xt = linear_ticks(x_lo, x_hi)
                xl = [_format_number(v) for v in xt]
            x_block = []
            for v, label in zip(xt, xl):
                px = (v - x_lo) * scale
                if -0.5 <= px <= bw + 0.5:
                    ref = ATLAS.text(label, tick_px)
                    x_block.append((solid_black, 1, 1, int(round(px - line_w / 2)), line_w, line_w, tick_len))
                    x_block.append((ref[0], ref[1], ref[2], int(round(px - ref[2] / 2)), line_w + tick_len + pad, ref[2], ref[1]))
            if len(_tick_blocks) > 8192:
                _tick_blocks.clear()
            x_hit = _tick_blocks[x_key] = (x_block, _extent(x_block))
        W, H = out.W, out.H
        _place(records, x_hit[0], x_hit[1], bx, by + bh, W, H)  # below the box
        if cb is not None:
            v0, v1 = float(img.vmin), float(img.vmax)
            c_key = (v0, v1, img.norm, None if cb.ticks is None else tuple(cb.ticks), bh, cb_px, line_w, tick_len, pad, bar_w)
            c_hit = _tick_blocks.get(c_key)
            if c_hit is None:
                solid_black = ATLAS.solid(black)[0]
                log_z = img.norm == "log" and v0 > 0 and v1 > 0
                if cb.ticks is not None:
                    cb_ticks = [float(t) for t in cb.ticks]
                elif log_z:
                    cb_ticks = [10.0 ** k for k in range(math.ceil(math.log10(v0) - 1e-9), math.floor(math.log10(v1) + 1e-9) + 1)]
                else:
                    cb_ticks = linear_ticks(v0, v1, 5)
                l0, l1 = (math.log10(v0), math.log10(v1)) if log_z else (v0, v1)
                c_block = []
                for v in cb_ticks:
                    if l1 == l0 or (log_z and v <= 0):
                        continue
                    f = ((math.log10(v) if log_z else v) - l0) / (l1 - l0)
                    if -1e-9 <= f <= 1.0 + 1e-9:
                        py = bh - f * bh
                        ref = ATLAS.text(_format_number(v), cb_px)
                        c_block.append((solid_black, 1, 1, bar_w + line_w, int(round(py - line_w / 2)), tick_len, line_w))
                        c_block.append((ref[0], ref[1], ref[2], bar_w + line_w + tick_len + pad, int(round(py - ref[1] / 2)), ref[2], ref[1]))
                c_hit = _tick_blocks[c_key] = (c_block, _extent(c_block))
            _place(records, c_hit[0], c_hit[1], kx, by, W, H)  # beside the colour bar
        # ---- the panel itself: the image covers its extent inside the x limits (imshow aspect="auto")
        ix0 = int(round(min(max(bx + (float(ex[0]) - x_lo) * scale, bx), bx + bw)))
        ix1 = int(round(min(max(bx + (float(ex[1]) - x_lo) * scale, bx), bx + bw)))
        if ix1 - ix0 < 1:
            ix0, ix1 = bx, bx + bw
        # a log energy axis: the rows are placed through the log transform (imshow + set_yscale("log")); with
        # a non-positive or empty extent, or a single row, matplotlib has no warp to show and the rows stay linear
        row_map = None
        if ax.yscale == "log" and 0 < y_lo < math.inf and 0 < y_hi < math.inf and y_lo != y_hi and ne >= 2:
            row_map = log_row_map(ne, bh, y_lo, y_hi)
        out.raster(img.rgba, ne, nt, ix0, by, ix1 - ix0, bh, row_map)

    # --------------------------------------------------------------- composing
    def compose(self, dpi: float | None = None) -> np.ndarray:
        """The figure as one (H, W, 4) uint8 image: the numpy evaluation of :meth:`tiles` (the oracle of
        the device composer, ``csrc/png.cu``).  Needs host rasters."""
        t = self.tiles(dpi)
        canvas = np.empty((t.H, t.W, 4), dtype=np.uint8)
        canvas[:] = t.background
        atlas = ATLAS.pixels()
        for k in range(len(t.records) - 1, -1, -1):  # the first tile of the list ends up on top
            off, ne, nt, x, y, w, h, _vf, _vc, flags, _map = t.records[k]
            src = t.sources.get(k)
            if isinstance(src, DeviceRaster):
                raise TypeError("this panel lives on the device: encode the figure with png.encode_figures_device")
            source = atlas[off : off + ne * nt].view(np.uint8).reshape(ne, nt, 4) if flags & TILE_OVERLAY else src
            if flags & TILE_ROW_MAP:
                rows = t.map_of(k)[1]  # storage rows, lowest energy = 0, like the device reads them
            else:
                rows = nearest_index(h, ne)
                if not flags & TILE_TOP_ORIGIN:
                    rows = ne - 1 - rows  # rasters store the lowest energy first (imshow origin="lower")
            canvas[y : y + h, x : x + w] = source[rows][:, nearest_index(w, nt)]
        return canvas

    def savefig(self, path, dpi=None, compress_level: int = 6, **kw):
        png.write_rgba(path, self.compose(dpi), compress_level=compress_level)


def close_all_axes_and_clear(fig) -> None:
    """Release a figure's panels (reference ``plotting.py:69-89``)."""
    if fig is None:
        return
    try:
        for ax in list(getattr(fig, "axes", [])):
            fig.delaxes(ax)
        fig.clf()
    except Exception:
        pass
