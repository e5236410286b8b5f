"""CPU tests of the host-side API pieces that need no GPU: PNG round trip, raster figure
composition, cusp markers, batch_runner's resumable progress."""

import functools
import json
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest


def test_png_round_trip_through_written_files(tmp_path):
    from configurable_spectrograms_b200 import png

    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (37, 53, 4), dtype=np.uint8)
    data = png.encode_rgba(img)
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    assert np.array_equal(png.decode_rgba(data), img)
    for i in (0, 2):
        png.write_rgba(tmp_path / f"{i}.png", img[i:])
    assert np.array_equal(png.decode_rgba((tmp_path / "2.png").read_bytes()), img[2:])
    from PIL import Image  # an independent decoder agrees

    assert np.array_equal(np.asarray(Image.open(tmp_path / "0.png")), img)


def _raster_tiles(tiles):
    return [(tiles.records[k], src) for k, src in sorted(tiles.sources.items())]


def test_figure_compose_and_markers():
    from configurable_spectrograms_b200.cusp_marking import draw_cusp_both_markers, draw_cusp_bracket_marker
    from configurable_spectrograms_b200.figure import FigureCanvas, SpectrogramFigure, close_all_axes_and_clear

    fig = SpectrogramFigure(figsize=(24, 6))
    canvas = FigureCanvas(fig)
    assert canvas.figure is fig and fig.canvas is canvas
    axes = [fig.add_subplot(2, 2, k + 1) for k in range(4)]
    for k, ax in enumerate(axes[:3]):
        rgba = np.full((5, 20 + 10 * k, 4), 40 * (k + 1), dtype=np.uint8)
        rgba[0] = (255, 0, 255, 255)  # lowest energy row: must end up at the bottom of the image
        im = ax.imshow(rgba, extent=(0.0, 1.0, 4.0, 4000.0), vmin=1.0, vmax=10.0, cmap="viridis")
        ax.set_xlim(0.0, 1.0)
        ax.set_ylabel("Energy (eV)")
        fig.colorbar(im, ax=ax, label="Counts")
    artists = draw_cusp_both_markers(axes[0], [0.25, 0.75], line_color="white")
    assert len(artists) == 5  # two lines per position + the bracket
    assert draw_cusp_bracket_marker(axes[0], []) == []
    one = draw_cusp_bracket_marker(axes[1], [0.5], caption="cusp")
    assert len(one) == 2 and axes[1].texts[-1]["text"] == "cusp"
    fig.suptitle("a title")
    img = fig.compose(dpi=50)
    assert img.shape == (300, 1200, 4) and img.dtype == np.uint8
    tiles = fig.tiles(50)
    rasters = _raster_tiles(tiles)
    assert len(rasters) == 3  # the fourth subplot holds no image
    (_off, ne, nt, x, y, w, h, *_rest), _src = rasters[0]
    assert (ne, nt) == (5, 20) and w > 100 and h > 30  # stretched over the axes box (imshow aspect="auto")
    assert (img[y + h - 1, x + 1] == (255, 0, 255, 255)).all() and (img[y, x + 1] == (40, 40, 40, 40)).all()
    line_x = x + round(0.25 * w)
    near = img[y + h // 2, line_x - 3 : line_x + 4]
    assert (near == (255, 255, 255, 255)).all(axis=1).any()  # the white cusp line on top of the black one ...
    assert (near == (0, 0, 0, 255)).all(axis=1).any()  # ... whose wider stroke shows on both sides
    assert (img[y + h + 2 : y + h + 30, x - 2 : x + w + 2] != 255).any()  # the bracket below the axis
    assert (img[:12] != 255).any()  # the title
    close_all_axes_and_clear(fig)
    assert fig.axes == []


def test_run_batch_progress_and_resume(tmp_path):
    from configurable_spectrograms_b200.batch_runner import run_batch

    path = tmp_path / "progress.json"

    def worker(item):
        if item == "boom":
            raise RuntimeError("x")
        return item, ("no_data" if item == "empty" else "ok")

    factory = functools.partial(ThreadPoolExecutor, max_workers=2)
    res = run_batch(["a", "empty", "boom", "b"], worker, factory, progress_json_path=str(path), flush_batch_size=2,
                    install_signal_handlers=False)
    assert sorted(res) == [("a", "ok"), ("b", "ok"), ("boom", "error"), ("empty", "no_data")]
    state = json.load(open(path))
    assert sorted(state["completed_items"]) == ["'a'", "'b'"] and state["errors"] == ["'boom'"]
    assert state["no_data"] == ["'empty'"] and state["last_index"] == 3 and state["schema_version"] == 1
    res = run_batch(["a", "b", "c"], worker, factory, progress_json_path=str(path), install_signal_handlers=False)
    assert res == [("c", "ok")]
    res = run_batch(["a"], worker, factory, progress_json_path=str(path), ignore_progress_json=True, install_signal_handlers=False)
    assert res == [("a", "ok")]


def test_date2num_matches_datetime_path():
    from datetime import datetime, timezone

    from configurable_spectrograms_b200.plotting import date2num
    from oracle import stubs

    rng = np.random.default_rng(1)
    t = 946684800.0 + rng.random(2000) * 3e7
    t[:4] = [946684800.0, 946684800.5, 946684800.0000005, 946684800.9999995]
    ref = np.array([stubs.date2num(datetime.fromtimestamp(float(x), tz=timezone.utc)) for x in t])
    assert np.array_equal(date2num(t).view(np.uint64), ref.view(np.uint64))
    assert date2num(946684800.0) == ref[0]
    # the scalar path (plain float arithmetic: panel limits, marker positions) against the vectorised one,
    # bit for bit, negative timestamps and signed zeros included
    more = np.concatenate([t, rng.uniform(-1e6, 2e9, 5000), [0.0, -0.0, -0.5, -1e-7, 1e-7, 1.9999995, 0.9999995]])
    scalars = np.array([date2num(float(x)) for x in more])
    assert np.array_equal(scalars.view(np.uint64), date2num(more).view(np.uint64))


def test_png_up_filter_decode_and_adler_of_segments():
    """Host side of the device PNG stage: the decoder undoes filter 2 (Up), and the Adler-32 of a
    stream follows from per-segment partial sums (what csrc/png.cu emits per scanline segment)."""
    import struct
    import zlib

    from configurable_spectrograms_b200 import png

    rng = np.random.default_rng(4)
    segs = [rng.integers(0, 256, int(n), dtype=np.uint8) for n in (1, 4097, 4096, 13, 4097, 2)]
    sa = [int(s.astype(np.int64).sum()) % 65521 for s in segs]
    sb = [int(((len(s) - np.arange(len(s))) * s.astype(np.int64)).sum()) % 65521 for s in segs]
    assert png.adler32_of_segments(sa, sb, [len(s) for s in segs]) == zlib.adler32(np.concatenate(segs).tobytes())
    assert png.adler32_of_segments([], [], []) == zlib.adler32(b"")
    img = rng.integers(0, 256, (9, 6, 4), dtype=np.uint8)
    flat = img.reshape(9, 24)
    for kinds in ([2] * 9, [0, 2, 2, 0, 2, 0, 0, 2, 2]):
        raw = np.zeros((9, 25), np.uint8)
        for r, kind in enumerate(kinds):
            raw[r, 0] = kind
            raw[r, 1:] = flat[r] - (flat[r - 1] if (kind == 2 and r > 0) else 0)
        data = (png._SIGNATURE + png._chunk(b"IHDR", struct.pack(">IIBBBBB", 6, 9, 8, 6, 0, 0, 0))
                + png._chunk(b"IDAT", zlib.compress(raw.tobytes())) + png._chunk(b"IEND", b""))
        assert np.array_equal(png.decode_rgba(data), img)


def test_figure_layout_serves_host_and_device_rasters():
    from configurable_spectrograms_b200.figure import DeviceRaster, SpectrogramFigure, nearest_index

    rng = np.random.default_rng(2)
    shapes = [(74, 300), (74, 90), (30, 300)]
    figs = []
    for device in (False, True):
        fig = SpectrogramFigure(figsize=(12, 6))
        for cell, (ne, nt) in zip((1, 2, 3), shapes):
            ax = fig.add_subplot(2, 2, cell)
            ax.imshow(DeviceRaster(16 * cell, ne, nt) if device else rng.integers(0, 255, (ne, nt, 4), dtype=np.uint8),
                      extent=(0.0, float(nt), 0.0, 1.0))
            ax.set_xlim(0.0, float(nt))
            ax.axvline(12.0, color="red", linewidth=4)
        figs.append(fig)
    t0, t1 = figs[0].tiles(100), figs[1].tiles(100)
    assert (t0.W, t0.H) == (t1.W, t1.H) == (1200, 600) == figs[0].compose(100).shape[1::-1]
    assert [r[1:] for r in t0.records] == [r[1:] for r in t1.records]  # same geometry; only the raster offsets differ
    assert [rec[0] for rec, _s in _raster_tiles(t1)] == [16, 32, 48]
    with pytest.raises(TypeError):
        figs[1].compose()
    # nearest neighbour on pixel centres, float32 like the device: identity at 1:1, whole repeats at k:1
    assert np.array_equal(nearest_index(7, 7), np.arange(7)) and np.array_equal(nearest_index(12, 4), np.repeat(np.arange(4), 3))
    rows = t0.content_rows()
    assert rows[0] == 0 and np.all(np.diff(rows) > 0) and rows[-1] < t0.H


def test_png_assembly_and_native_writer_splice_repeated_lines():
    """``png.assemble_png``: content scanlines come as byte-aligned DEFLATE pieces (here from zlib, standing in
    for the device's segments), the runs of repeated lines in between are ``png.zero_run`` constants; the file
    decodes (own decoder and Pillow: Adler-32 and CRC verified) to the composed image."""
    import io
    import zlib

    from PIL import Image

    from configurable_spectrograms_b200 import png
    from configurable_spectrograms_b200.figure import SpectrogramFigure

    rng = np.random.default_rng(4)
    fig = SpectrogramFigure(figsize=(26, 4))
    for cell, nt in ((1, 300), (2, 41)):
        ax = fig.add_subplot(1, 2, cell)
        im = ax.imshow(rng.integers(0, 255, (9, nt, 4), dtype=np.uint8), extent=(0.0, 1.0, 4.0, 4000.0), cmap="turbo", vmin=1.0, vmax=9.0)
        ax.set_xlim(0.0, 1.0)
        ax.set_xlabel("Time (UTC)")
        fig.colorbar(im, ax=ax, label="Counts")
    tiles = fig.tiles(100)
    img, rows = fig.compose(100), tiles.content_rows()
    W, H = tiles.W, tiles.H
    assert W > 2048 and 0 < len(rows) < H  # three segments per scanline, and some lines repeat
    for r in range(1, H):  # every line that is not listed repeats the one above
        if r not in set(rows.tolist()):
            assert np.array_equal(img[r], img[r - 1]), r
    per_row = (W + 1023) // 1024
    segs, adler = [], []
    for r in rows:
        line = img[r].reshape(-1)
        for c in range(per_row):
            raw = (b"\x00" if c == 0 else b"") + line[4096 * c : 4096 * (c + 1)].tobytes()
            comp = zlib.compressobj(6, zlib.DEFLATED, -15)
            segs.append(comp.compress(raw) + comp.flush(zlib.Z_SYNC_FLUSH))
            b = np.frombuffer(raw, np.uint8).astype(np.int64)
            adler.append((int(b.sum() % 65521), int((b * (len(b) - np.arange(len(b)))).sum() % 65521)))
    packed = np.frombuffer(b"".join(segs), np.uint8)
    offsets = np.concatenate([[0], np.cumsum([len(x) for x in segs])])
    blob = b"".join(bytes(p) for p in png.assemble_png(W, H, rows, per_row, packed, offsets, 0, np.array(adler, dtype=np.uint32)))
    assert np.array_equal(png.decode_rgba(blob), img)
    assert np.array_equal(np.asarray(Image.open(io.BytesIO(blob)).convert("RGBA")), img)
    # ---- the native framer / writer (csg_png_write_files, a host-only entry point of the library): two files
    # from one packed buffer, the second canvas' segments and rows at an offset; plus a path that cannot be opened
    import tempfile

    from configurable_spectrograms_b200 import _lib

    lib = _lib.load_library()
    adler2 = np.concatenate([np.array(adler, dtype=np.uint32)] * 2)
    packed2 = np.concatenate([packed, packed])
    sizes = np.array([len(x) for x in segs] * 2)
    offsets2 = np.concatenate([[0], np.cumsum(sizes)])
    rows2 = np.concatenate([rows, rows]).astype(np.int32)
    canvases = np.zeros(2, dtype=_lib.PNG_CANVAS)
    canvases["W"], canvases["H"], canvases["segs_per_row"] = W, H, per_row
    canvases["seg_first"], canvases["row_first"] = (0, len(segs)), (0, len(rows))
    n_rows = [len(rows), len(rows)]
    with tempfile.TemporaryDirectory() as tmp:
        paths = [os.path.join(tmp, "a.png"), os.path.join(tmp, "b \u00e9.png")]
        png.write_files_native(lib, paths, canvases, n_rows, rows2, packed2, offsets2, adler2, n_threads=2)
        for path in paths:
            data = open(path, "rb").read()
            assert np.array_equal(png.decode_rgba(data), img)
            assert np.array_equal(np.asarray(Image.open(io.BytesIO(data)).convert("RGBA")), img)
        with pytest.raises(OSError, match="not written"):
            png.write_files_native(lib, [os.path.join(tmp, "missing_dir", "c.png"), paths[0]], canvases, n_rows, rows2, packed2,
                                   offsets2, adler2)
        assert np.array_equal(png.decode_rgba(open(paths[0], "rb").read()), img)  # the good file of a failing group is still written


def test_png_custom_huffman_tables_decode_with_zlib():
    """png.custom_tables: a dynamic-Huffman code fitted to symbol counts.  The device tokeniser's bit
    stream (header, filter literal, literals / matches, end of block, sync flush) is replayed on the
    host with these tables and must inflate to the original pixels -- with fitted counts and with
    none at all (every symbol the tokeniser can emit still has a code)."""
    import random
    import zlib

    from configurable_spectrograms_b200 import png

    random.seed(3)
    for trial in range(12):
        npx = random.randint(1, 300)
        palette = [0, 0xFF0000FF, 0xFF112233, 0x01020304]
        pix = [random.choice(palette + [random.getrandbits(32)]) for _ in range(npx)]
        seq, p, run, dist = [], 0, 0, 0
        while p < npx:  # csrc/png.cu's tokeniser at pixel granularity (one lane owning the whole line)
            x = pix[p]
            if run and x == pix[p - dist] and run < png.MATCH_PIXELS:
                run += 1
                p += 1
                continue
            if run:
                seq.append((run, dist))
                run = 0
            k = next((d for d in range(1, min(p, png.WINDOW_PIXELS) + 1) if pix[p - d] == x), 0)
            if k:
                run, dist = 1, k
            else:
                seq.append(x)
            p += 1
        if run:
            seq.append((run, dist))
        counts = np.zeros(316, np.int64)
        if trial % 2:
            for t in seq:
                if isinstance(t, tuple):
                    counts[257 + png._symbol_of(4 * t[0], png._LEN_BASE)] += 1
                    counts[286 + png._symbol_of(4 * t[1], png._DIST_BASE)] += 1
                else:
                    for shift in (0, 8, 16, 24):
                        counts[(t >> shift) & 255] += 1
        T = png.custom_tables(counts)
        assert int(max(T["lit_len"])) <= 9 and int(max(T["dist_len"])) <= 14 and int(max(T["len_len"])) <= 14
        acc = [0, 0]

        def put(value, bits):
            acc[0] |= int(value) << acc[1]
            acc[1] += int(bits)

        head = sum(int(T["header"][w]) << (32 * w) for w in range(40))
        put(head & ((1 << int(T["header_bits"])) - 1), T["header_bits"])
        put(T["lit_code"][0], T["lit_len"][0])  # the filter-type byte
        for t in seq:
            if isinstance(t, tuple):
                put(T["len_code"][t[0]], T["len_len"][t[0]])
                put(T["dist_code"][t[1]], T["dist_len"][t[1]])
            else:
                for shift in (0, 8, 16, 24):
                    b = (t >> shift) & 255
                    put(T["lit_code"][b], T["lit_len"][b])
        put(T["eob_code"], T["eob_len"])
        put(0, 3)
        stream = acc[0].to_bytes((acc[1] + 7) // 8, "little") + b"\x00\x00\xff\xff" + b"\x01\x00\x00\xff\xff"
        assert zlib.decompress(stream, -15) == b"\x00" + b"".join(int(x).to_bytes(4, "little") for x in pix)


def test_grouped_executor_serves_run_batch(tmp_path):
    """``generic_batch.GroupedExecutor`` under ``run_batch``: items are handed over in groups, every item
    still gets its own future / status / progress entry, a failing group fails its items only."""
    from configurable_spectrograms_b200.batch_runner import run_batch
    from configurable_spectrograms_b200.generic_batch import GroupedExecutor

    groups = []

    def process(items):
        groups.append(list(items))
        if "boom" in items:
            raise RuntimeError("group machinery failed")
        return [(item, "no_data" if item == "empty" else "ok") for item in items]

    items = [f"i{k}" for k in range(7)] + ["empty"]
    path = tmp_path / "progress.json"
    res = run_batch(items, None, functools.partial(GroupedExecutor, process, 3), progress_json_path=str(path),
                    install_signal_handlers=False)
    assert sorted(res) == sorted([(f"i{k}", "ok") for k in range(7)] + [("empty", "no_data")])
    assert [x for g in groups for x in g] == items and max(len(g) for g in groups) <= 3
    state = json.loads(path.read_text())
    assert sorted(state["completed_items"]) == sorted(repr(f"i{k}") for k in range(7)) and state["no_data"] == [repr("empty")]
    res = run_batch(["a", "boom", "b"], None, functools.partial(GroupedExecutor, process, 8), progress_json_path=None,
                    install_signal_handlers=False)
    assert sorted(res) == [("a", "error"), ("b", "error"), ("boom", "error")]


def test_text_sprites_are_composed_from_glyphs_and_survive_an_atlas_reset():
    """``overlay.SpriteAtlas.text``: strings are put together from per-character coverage masks (one Pillow
    render per character and size).  A figure composed before and after ``ATLAS.clear()`` (which also empties
    the layout caches that hold sprite offsets) is the same image; repeated strings share one sprite."""
    from configurable_spectrograms_b200.figure import SpectrogramFigure
    from configurable_spectrograms_b200.overlay import ATLAS, SpriteAtlas

    atlas = SpriteAtlas()
    a, b = atlas.text("12:34", 28), atlas.text("12:34", 28)
    assert a == b and atlas.text("12:35", 28) != a
    sprite = atlas.sprite(a)
    assert sprite.shape == (a[1], a[2], 4) and sprite[..., 3].min() == 255  # opaque on its background
    ink = sprite[..., 0] < 128
    assert ink.any() and not ink[0].any() and not ink[-1].any() and not ink[:, 0].any() and not ink[:, -1].any()  # 1 px margin
    two = atlas.sprite(atlas.text("Orbit 7\nees", 28))
    one = atlas.sprite(atlas.text("Orbit 7", 28))
    assert two.shape[0] > one.shape[0] and two.shape[1] == one.shape[1]  # centred under the wider line
    up = atlas.sprite(atlas.text("Counts", 28, rotate=True))
    flat = atlas.sprite(atlas.text("Counts", 28))
    assert np.array_equal(up, np.rot90(flat))
    red = atlas.sprite(atlas.text("9", 28, color=(255, 0, 0, 255)))
    assert (red[..., 0] == 255).all() and (red[..., 1] < 255).any()

    # a long string as one sprite per word (titles): put together, the words are the line
    line = "Orbit 13042 - EES pitch angle (0, 30) gyp"
    width, height, parts = atlas.text_parts(line, 33)
    canvas = np.full((height, width, 4), 255, dtype=np.uint8)
    for ref, dx, dy in parts:
        canvas[dy : dy + ref[1], dx : dx + ref[2]] = np.minimum(canvas[dy : dy + ref[1], dx : dx + ref[2]], atlas.sprite(ref))
    whole = atlas._blend((0, 0, 0, 255), (255, 255, 255, 255))[atlas._line(line, 33)]
    assert np.array_equal(canvas[: whole.shape[0], : whole.shape[1]], whole[:height, :width])
    assert len(parts) == len(line.split()) and atlas.text_parts("Orbit 99", 33)[2][0][0] == parts[0][0]  # "Orbit" is shared
    w2, h2, p2 = atlas.text_parts("ab\nabcdef", 33)
    assert h2 > height and p2[0][1] > 0 and p2[1][1] == 0 and p2[1][2] > p2[0][2]  # centred first line, second line below

    def build():
        rng = np.random.default_rng(2)
        fig = SpectrogramFigure(figsize=(12, 4))
        ax = fig.add_subplot(1, 1, 1)
        im = ax.imshow(rng.integers(0, 255, (24, 200, 4), dtype=np.uint8), extent=(10957.0, 10957.02, 4.0, 4000.0),
                       cmap="turbo", vmin=1.0, vmax=2400.0)
        ax.set_xlim(10957.0, 10957.02)
        ax.xaxis.set_major_formatter("%H:%M")
        ax.set_ylabel("Energy (eV)")
        ax.set_title("Orbit 13042 EES")
        fig.suptitle("Pitch angle grid\nOrbit 13042")
        fig.colorbar(im, ax=ax, label="Counts")
        return fig

    before = build().compose(100)
    ATLAS.clear()
    after = build().compose(100)
    assert np.array_equal(before, after)


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5, 6])
def test_content_rows_property_on_random_figures(seed):
    """K4's host half on random layouts (grid, size, dpi, panel shapes, log / linear colour bars, markers): a
    scanline that ``content_rows`` does not list is pixel-identical to the line above it in the composed
    image -- the property that lets the device encode the listed lines only -- and Adler-32 partial sums of
    arbitrary segmentations combine to zlib's checksum."""
    import zlib

    from configurable_spectrograms_b200 import png
    from configurable_spectrograms_b200.figure import SpectrogramFigure

    rng = np.random.default_rng(seed)
    n_rows, n_cols = int(rng.integers(1, 4)), int(rng.integers(1, 3))
    fig = SpectrogramFigure(figsize=(float(rng.uniform(4, 13)) * n_cols, float(rng.uniform(1.5, 3.5)) * n_rows))
    if seed % 2:
        fig.suptitle(f"Orbit {13000 + seed} - random layout\nline two")
    for cell in range(1, n_rows * n_cols + 1):
        if rng.random() < 0.15:
            continue  # an empty cell
        ne, nt = int(rng.integers(1, 90)), int(rng.integers(1, 700))
        ax = fig.add_subplot(n_rows, n_cols, cell)
        x0 = 10957.0 + float(rng.random())
        x1 = x0 + float(rng.uniform(1e-4, 0.03))
        log = bool(rng.random() < 0.5)
        im = ax.imshow(rng.integers(0, 255, (ne, nt, 4), dtype=np.uint8), extent=(x0, x1, 4.0, 4000.0), cmap="viridis",
                       norm="log" if log else None, vmin=1.0 if log else 0.0, vmax=float(rng.uniform(20, 5000)))
        ax.set_xlim(x0, x1)
        ax.xaxis.set_major_formatter("%H:%M:%S" if x1 - x0 < 120 / 86400 else "%H:%M")
        ax.set_ylabel("Energy (eV)")
        ax.set_title(f"panel {cell} of seed {seed}")
        if rng.random() < 0.7:
            fig.colorbar(im, ax=ax, label="Counts")
        if rng.random() < 0.6:
            ax.axvline(x0 + 0.4 * (x1 - x0), color="red", linewidth=float(rng.uniform(0.5, 4)))
    dpi = float(rng.choice([37, 72, 100, 150]))
    tiles = fig.tiles(dpi)
    img = fig.compose(dpi)
    assert img.shape == (tiles.H, tiles.W, 4)
    rows = tiles.content_rows()
    assert rows[0] == 0 and np.all(np.diff(rows) > 0) and rows[-1] < tiles.H
    listed = np.zeros(tiles.H, dtype=bool)
    listed[rows] = True
    for line in np.flatnonzero(~listed):
        assert np.array_equal(img[line], img[line - 1]), (seed, int(line))
    # Adler-32 from per-segment partial sums, any segmentation
    raw = rng.integers(0, 256, int(rng.integers(1, 40_000)), dtype=np.uint8)
    cuts = np.unique(np.concatenate([[0, len(raw)], rng.integers(0, len(raw) + 1, 12)]))
    sa, sb, ln = [], [], []
    for a, b in zip(cuts[:-1], cuts[1:]):
        seg = raw[a:b].astype(np.int64)
        sa.append(int(seg.sum() % 65521))
        sb.append(int((seg * (len(seg) - np.arange(len(seg)))).sum() % 65521))
        ln.append(len(seg))
    assert png.adler32_of_segments(np.array(sa), np.array(sb), np.array(ln)) == zlib.adler32(raw.tobytes())
