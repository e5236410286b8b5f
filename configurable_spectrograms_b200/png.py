"""PNG hand-off for the RGBA rasters (the on-disk product of the reference:
``fast/process_orbit.py:98-117``, ``generic_batch.py:108-113``).

Two encoders, one file format (8-bit RGBA, non-interlaced):

* :func:`encode_rgba` / :func:`write_rgba` -- filter 0 + zlib DEFLATE on the host, for figures whose
  rasters are host arrays (the single-figure entry points);
* :func:`encode_figures_device` / :func:`write_figures_device` -- figures whose panels are K3 rasters
  in HBM are composed, Up-filtered and DEFLATE-encoded on the GPU (``csrc/png.cu``); only the
  compressed bytes cross PCIe.  The host adds the zlib header / trailer and the PNG chunk framing.

Both decode to the same pixels (``tests/test_gpu_api.py``); the host composer is the oracle of the
device one.
"""

from __future__ import annotations

import os
import struct
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

_SIGNATURE = b"\x89PNG\r\n\x1a\n"


def _chunk(tag: bytes, payload: bytes) -> bytes:
    return struct.pack(">I", len(payload)) + tag + payload + struct.pack(">I", zlib.crc32(tag + payload) & 0xFFFFFFFF)


def encode_rgba(image: np.ndarray, compress_level: int = 6) -> bytes:
    """(H, W, 4) uint8 -> PNG bytes (8-bit RGBA, no interlace, filter type 0 on every row)."""
    img = np.ascontiguousarray(image, dtype=np.uint8)
    if img.ndim != 3 or img.shape[2] != 4:
        raise ValueError(f"expected an (H, W, 4) uint8 image, got {img.shape}")
    h, w, _ = img.shape
    raw = np.zeros((h, 1 + 4 * w), dtype=np.uint8)  # leading filter byte 0 per scanline
    raw[:, 1:] = img.reshape(h, 4 * w)
    ihdr = struct.pack(">IIBBBBB", w, h, 8, 6, 0, 0, 0)
    return _SIGNATURE + _chunk(b"IHDR", ihdr) + _chunk(b"IDAT", zlib.compress(raw.tobytes(), compress_level)) + _chunk(b"IEND", b"")


def write_rgba(path, image: np.ndarray, compress_level: int = 6) -> None:
    data = encode_rgba(image, compress_level)
    with open(path, "wb") as f:
        f.write(data)


def decode_rgba(data: bytes) -> np.ndarray:
    """Inverse of :func:`encode_rgba` (filter-0 RGBA only) -- used by the round-trip tests."""
    if data[:8] != _SIGNATURE:
        raise ValueError("not a PNG")
    pos, idat, shape = 8, b"", None
    while pos < len(data):
        (n,) = struct.unpack(">I", data[pos : pos + 4])
        tag, payload = data[pos + 4 : pos + 8], data[pos + 8 : pos + 8 + n]
        (crc,) = struct.unpack(">I", data[pos + 8 + n : pos + 12 + n])
        if zlib.crc32(tag + payload) & 0xFFFFFFFF != crc:
            raise ValueError("PNG chunk CRC mismatch")
        if tag == b"IHDR":
            w, h, depth, ctype = struct.unpack(">IIBB", payload[:10])
            if (depth, ctype) != (8, 6):
                raise ValueError("only 8-bit RGBA is supported")
            shape = (h, w)
        elif tag == b"IDAT":
            idat += payload
        pos += 12 + n
    h, w = shape
    raw = np.frombuffer(zlib.decompress(idat), dtype=np.uint8).reshape(h, 1 + 4 * w)
    kinds = set(np.unique(raw[:, 0]).tolist())
    if kinds <= {0}:
        return raw[:, 1:].reshape(h, w, 4).copy()
    if not kinds <= {0, 2}:
        raise ValueError(f"only filter types 0 (None) and 2 (Up) are supported, found {sorted(kinds)}")
    out = raw[:, 1:].copy()
    up = raw[:, 0] == 2
    if up.all():  # every line is a difference to the one above: a running sum modulo 256
        out = np.cumsum(out, axis=0, dtype=np.uint64).astype(np.uint8)
    else:
        for r in range(h):
            if up[r] and r > 0:
                out[r] += out[r - 1]
    return out.reshape(h, w, 4)


def write_many(jobs, compress_level: int = 6, max_workers: int = 8) -> None:
    """``jobs``: iterable of (path, image).  Encodes and writes on a thread pool."""
    jobs = list(jobs)
    if not jobs:
        return
    with ThreadPoolExecutor(max_workers=max(1, min(max_workers, len(jobs)))) as pool:
        list(pool.map(lambda j: write_rgba(j[0], j[1], compress_level), jobs))


# ----------------------------------------------------------------------------------------
# device encoder (csrc/png.cu)
# ----------------------------------------------------------------------------------------
_ADLER = 65521

# RFC 1951 3.2.5 / 3.2.7
_LEN_BASE = (3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258)
_LEN_EXTRA = (0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0)
_DIST_BASE = (1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
              6145, 8193, 12289, 16385, 24577)
_DIST_EXTRA = (0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13)
_CL_ORDER = (16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15)
MATCH_PIXELS, WINDOW_PIXELS = 64, 128  # longest match / farthest distance the device tokeniser emits, in pixels


def _limited_lengths(freq, maxlen: int) -> list[int]:
    """Huffman code lengths (<= maxlen) for the symbols with a non-zero count; at least two get a code."""
    import heapq

    n = len(freq)
    syms = [s for s in range(n) if freq[s] > 0] or [0]
    lens = [0] * n
    if len(syms) == 1:
        lens[syms[0]] = lens[1 if syms[0] == 0 else 0] = 1
        return lens
    weight = {s: max(int(freq[s]), 1) for s in syms}
    while True:
        heap = [(w, i, (s,)) for i, (s, w) in enumerate(weight.items())]
        heapq.heapify(heap)
        serial, depth = len(heap), dict.fromkeys(syms, 0)
        while len(heap) > 1:
            a, b = heapq.heappop(heap), heapq.heappop(heap)
            for s in a[2] + b[2]:
                depth[s] += 1
            serial += 1
            heapq.heappush(heap, (a[0] + b[0], serial, a[2] + b[2]))
        if max(depth.values()) <= maxlen:
            for s, d in depth.items():
                lens[s] = d
            return lens
        weight = {s: (w + 1) // 2 + 1 for s, w in weight.items()}  # flatten the distribution and retry


def _canonical_codes(lens) -> list[int]:
    top = max(lens) if lens else 0
    per_len = [0] * (top + 2)
    for length in lens:
        if length:
            per_len[length] += 1
    code, first = 0, [0] * (top + 2)
    for bits in range(1, top + 1):
        code = (code + per_len[bits - 1]) << 1
        first[bits] = code
    codes = [0] * len(lens)
    for s, length in enumerate(lens):
        if length:
            codes[s] = first[length]
            first[length] += 1
    return codes


def _reverse(value: int, bits: int) -> int:
    out = 0
    for i in range(bits):
        out |= ((value >> i) & 1) << (bits - 1 - i)
    return out


def _dynamic_header(ll_lens, d_lens) -> tuple[int, int]:
    """(bits, count) of a dynamic block's header after BFINAL/BTYPE: HLIT, HDIST, HCLEN, the code-length
    code and the run-length coded lengths of both alphabets (RFC 1951 3.2.7)."""
    hlit = max(257, max(i for i, l in enumerate(ll_lens) if l) + 1)
    hdist = max(1, max((i for i, l in enumerate(d_lens) if l), default=0) + 1)
    seq = list(ll_lens[:hlit]) + list(d_lens[:hdist])
    items, i = [], 0
    while i < len(seq):
        length, j = seq[i], i
        while j < len(seq) and seq[j] == length:
            j += 1
        run = j - i
        if length == 0:
            while run >= 11:
                r = min(run, 138)
                items.append((18, r - 11, 7))
                run -= r
            if run >= 3:
                items.append((17, run - 3, 3))
                run = 0
            items += [(0, 0, 0)] * run
        else:
            items.append((length, 0, 0))
            run -= 1
            while run >= 3:
                r = min(run, 6)
                items.append((16, r - 3, 2))
                run -= r
            items += [(length, 0, 0)] * run
        i = j
    cl_freq = [0] * 19
    for s, _x, _n in items:
        cl_freq[s] += 1
    cl_lens = _limited_lengths(cl_freq, 7)
    cl_codes = _canonical_codes(cl_lens)
    hclen = max(4, max(k for k in range(19) if cl_lens[_CL_ORDER[k]]) + 1)
    acc, n = 0, 0

    def put(value, bits):
        nonlocal acc, n
        acc |= value << n
        n += bits

    put(hlit - 257, 5), put(hdist - 1, 5), put(hclen - 4, 4)
    for k in range(hclen):
        put(cl_lens[_CL_ORDER[k]], 3)
    for s, x, nx in items:
        put(_reverse(cl_codes[s], cl_lens[s]), cl_lens[s])
        if nx:
            put(x, nx)
    return acc, n


def _symbol_of(value: int, base) -> int:
    c = len(base) - 1
    while base[c] > value:
        c -= 1
    return c


def custom_tables(counts) -> np.ndarray:
    """``csg_png_tables`` of a dynamic-Huffman code fitted to symbol counts (``csg_png_count``: 286
    literal / length counts, then 30 distance counts).  Every symbol the device tokeniser can emit gets
    a code whatever the counts say; literal / length codes use at most 9 bits, distance codes at most 7
    (the kernel's buffers are sized for that)."""
    from ._lib import PNG_TABLES

    counts = np.asarray(counts, dtype=np.int64)
    ll = counts[:286].copy()
    dd = counts[286:316].copy()
    ll[:257] += 1  # every literal byte and the end-of-block symbol may occur
    len_syms = [257 + _symbol_of(4 * n, _LEN_BASE) for n in range(1, MATCH_PIXELS + 1)]
    dist_syms = [_symbol_of(4 * k, _DIST_BASE) for k in range(1, WINDOW_PIXELS + 1)]
    for s in set(len_syms):
        ll[s] += 1
    for s in set(dist_syms):
        dd[s] += 1
    ll_lens, d_lens = _limited_lengths(ll.tolist(), 9), _limited_lengths(dd.tolist(), 7)
    ll_codes, d_codes = _canonical_codes(ll_lens), _canonical_codes(d_lens)
    t = np.zeros(1, dtype=PNG_TABLES)[0]
    for v in range(256):
        t["lit_code"][v], t["lit_len"][v] = _reverse(ll_codes[v], ll_lens[v]), ll_lens[v]
    for n in range(1, MATCH_PIXELS + 1):
        s = len_syms[n - 1]
        c = s - 257
        t["len_code"][n] = _reverse(ll_codes[s], ll_lens[s]) | ((4 * n - _LEN_BASE[c]) << ll_lens[s])
        t["len_len"][n], t["len_sym"][n] = ll_lens[s] + _LEN_EXTRA[c], s
    for k in range(1, WINDOW_PIXELS + 1):
        c = dist_syms[k - 1]
        t["dist_code"][k] = _reverse(d_codes[c], d_lens[c]) | ((4 * k - _DIST_BASE[c]) << d_lens[c])
        t["dist_len"][k], t["dist_sym"][k] = d_lens[c] + _DIST_EXTRA[c], c
    t["eob_code"], t["eob_len"] = _reverse(ll_codes[256], ll_lens[256]), ll_lens[256]
    head, nbits = _dynamic_header(ll_lens, d_lens)
    head = 0b100 | (head << 3)  # BFINAL = 0, BTYPE = 10 (dynamic Huffman), LSB first
    nbits += 3
    if nbits > 40 * 32:
        raise ValueError("dynamic block header does not fit the device table")
    t["header_bits"] = nbits
    for w in range((nbits + 31) // 32):
        t["header"][w] = (head >> (32 * w)) & 0xFFFFFFFF
    return t


def adler32_of_segments(sum_bytes: np.ndarray, weighted: np.ndarray, lengths: np.ndarray) -> int:
    """Adler-32 of the concatenation of segments from their partial sums: ``sum_bytes[k]`` = sum of
    the bytes of segment k, ``weighted[k]`` = sum of ``(n_k - t) * byte_t`` (both mod 65521),
    ``lengths[k]`` = n_k.  With A the running byte sum (+1) before a segment, the segment adds
    ``n_k * A + weighted[k]`` to B."""
    sa = np.asarray(sum_bytes, dtype=np.int64) % _ADLER
    sb = np.asarray(weighted, dtype=np.int64) % _ADLER
    n = np.asarray(lengths, dtype=np.int64)
    a_before = np.concatenate([[1], (1 + np.cumsum(sa)) % _ADLER])[:-1] if len(sa) else np.zeros(0, np.int64)
    a = int((1 + int(sa.sum())) % _ADLER)
    b = int((((n % _ADLER) * a_before) % _ADLER + sb).sum() % _ADLER)
    return (b << 16) | a


_zero_runs: dict = {}


def zero_run(width: int, n_lines: int) -> bytes:
    """``n_lines`` scanlines that repeat the line above -- filter type 2 ("Up") followed by ``4 * width``
    zero bytes each -- as a byte-aligned piece of a raw DEFLATE stream (ends with an empty stored block,
    like the device's segments, so pieces concatenate).  A constant per (width, run length): cached."""
    key = (width, n_lines)
    hit = _zero_runs.get(key)
    if hit is None:
        comp = zlib.compressobj(6, zlib.DEFLATED, -15)
        line = b"\x02" + bytes(4 * width)
        hit = comp.compress(line * n_lines) + comp.flush(zlib.Z_SYNC_FLUSH)
        if len(_zero_runs) > 4096:
            _zero_runs.clear()
        _zero_runs[key] = hit
    return hit


def assemble_png(W: int, H: int, rows, per_row: int, packed, offsets, s0: int, adler) -> list:
    """The PNG file of one canvas as a list of buffers (the compressed stream is not copied).

    ``rows``: the canvas' content scanlines (ascending); their segments -- ``per_row`` per scanline, numbered
    from ``s0`` -- are ``packed[offsets[s] : offsets[s + 1]]`` (byte-aligned DEFLATE pieces) with Adler-32
    partial sums ``adler[s] = (sum of bytes, sum of (n - t) * byte_t)`` of their filtered bytes.  The
    scanlines in between repeat the line above: :func:`zero_run` pieces."""
    n_rows_c = len(rows)
    s1 = s0 + per_row * n_rows_c
    # filtered bytes per device segment: 4 per pixel, plus the filter-type byte on a line's first segment
    chunk = np.arange(s1 - s0) % per_row
    npx = np.minimum(1024, W - 1024 * chunk)
    seg_len = 4 * npx + (chunk == 0)
    gap = np.diff(np.concatenate([rows, [H]])) - 1  # repeated lines after every content row
    line_bytes = 1 + 4 * W
    has_gap = np.flatnonzero(gap > 0)
    # Adler-32 pieces in stream order: per content row its segments, then (maybe) a run of Up lines whose
    # only non-zero bytes are the filter bytes (value 2) at the start of every line
    n_pieces = (s1 - s0) + len(has_gap)
    sa, sb, ln = np.zeros(n_pieces, np.int64), np.zeros(n_pieces, np.int64), np.zeros(n_pieces, np.int64)
    seg_pos = np.arange(s1 - s0) + np.searchsorted(has_gap, np.arange(s1 - s0) // per_row, side="left")
    sa[seg_pos], sb[seg_pos], ln[seg_pos] = adler[s0:s1, 0], adler[s0:s1, 1], seg_len
    if len(has_gap):
        g = gap[has_gap].astype(np.int64)
        run_pos = (has_gap + 1) * per_row + np.arange(len(has_gap))
        L = g * line_bytes
        sa[run_pos] = (2 * g) % _ADLER
        sb[run_pos] = (2 * (g * L - line_bytes * (g * (g - 1) // 2))) % _ADLER  # sum over lines k of (L - k * line_bytes) * 2
        ln[run_pos] = L
    check = adler32_of_segments(sa, sb, ln)
    pieces: list = []
    start = 0
    for r in has_gap.tolist():  # device bytes up to and including content row r, then the run after it
        end = (r + 1) * per_row
        pieces.append(memoryview(packed[offsets[s0 + start] : offsets[s0 + end]]))
        pieces.append(zero_run(W, int(gap[r])))
        start = end
    if start < s1 - s0:
        pieces.append(memoryview(packed[offsets[s0 + start] : offsets[s1]]))
    head, tail = b"\x78\x01", b"\x01\x00\x00\xff\xff" + struct.pack(">I", check)
    crc = zlib.crc32(head, zlib.crc32(b"IDAT"))
    size = len(head) + len(tail)
    for piece in pieces:
        crc = zlib.crc32(piece, crc)  # releases the GIL on large buffers
        size += len(piece)
    crc = zlib.crc32(tail, crc)
    ihdr = struct.pack(">IIBBBBB", W, H, 8, 6, 0, 0, 0)
    return [_SIGNATURE + _chunk(b"IHDR", ihdr) + struct.pack(">I", size) + b"IDAT" + head, *pieces,
            tail + struct.pack(">I", crc & 0xFFFFFFFF) + _chunk(b"IEND", b"")]


def zero_segment_table(widths) -> np.ndarray:
    """``csg_png_zero_segment`` entries for every segment length the canvases of these widths produce: the
    1024-pixel chunks and the last chunk of a scanline, with and without the leading filter byte (2 = Up)."""
    from ._lib import PNG_ZERO_SEGMENT

    lengths = set()
    for W in set(int(w) for w in widths):
        per_row = (W + 1023) // 1024
        for chunk in range(per_row):
            npx = min(1024, W - 1024 * chunk)
            lengths.add(4 * npx + (1 if chunk == 0 else 0))
    table = np.zeros(len(lengths), dtype=PNG_ZERO_SEGMENT)
    for entry, n_raw in zip(table, sorted(lengths)):
        comp = zlib.compressobj(9, zlib.DEFLATED, -15)
        raw = (b"\x02" if n_raw & 1 else b"") + bytes(n_raw - (n_raw & 1))
        piece = comp.compress(raw) + comp.flush(zlib.Z_SYNC_FLUSH)
        if len(piece) > 56:
            raise ValueError(f"zero segment of {n_raw} bytes compresses to {len(piece)} bytes (> 56)")
        entry["n_raw"], entry["len"] = n_raw, len(piece)
        entry["bytes"][: len(piece)] = np.frombuffer(piece, np.uint8)
    return table


def _device_tables(figures, dpi):
    """Tile / canvas / row tables of a list of figures.  Returns ``(canvases, tiles, rows, row_maps, per_figure)``
    with ``canvases`` a list of mutable rows of ``PNG_CANVAS`` (``seg_first`` is filled per group), ``tiles`` one
    ``PNG_TILE`` array, ``rows`` one int32 array of content rows, ``row_maps`` the int32 row maps of the panels
    on a log energy axis (each distinct map once; ``None`` when there are none) and ``per_figure`` =
    [(W, H, content rows)]."""
    from ._lib import PNG_TILE
    from .figure import DeviceRaster

    def pack(c):
        r, g, b, a = c
        return r | (g << 8) | (b << 16) | (a << 24)

    canvases, tile_parts, row_parts, per_figure = [], [], [], []
    map_at, map_parts = {}, []  # row-map key -> offset in the concatenated maps
    n_tiles = n_rows = n_map = 0
    for fig in figures:
        t = fig.tiles(dpi)
        for src in t.sources.values():
            if not isinstance(src, DeviceRaster):
                raise TypeError("encode_figures_device needs panels drawn from device rasters (figure.DeviceRaster)")
        for key, rows in t.row_maps:
            if key not in map_at:
                map_at[key] = n_map
                map_parts.append(rows)
                n_map += len(rows)
        table = t.table([map_at[key] for key, _rows in t.row_maps])
        rows = t.content_rows(table)
        canvases.append([t.W, t.H, n_tiles, len(table), pack(t.background), 0, (t.W + 1023) // 1024, n_rows])
        tile_parts.append(table)
        row_parts.append(rows)
        per_figure.append((t.W, t.H, rows))
        n_tiles += len(table)
        n_rows += len(rows)
    tiles = np.concatenate(tile_parts) if n_tiles else np.zeros(1, PNG_TILE)
    rows = np.concatenate(row_parts) if n_rows else np.zeros(1, np.int32)
    row_maps = np.concatenate(map_parts).astype(np.int32) if n_map else None
    return canvases, tiles, rows, row_maps, per_figure


def encode_figures_device(ctx, d_rgba_ptr: int, figures, dpi: float | None = None, max_segments: int = 400_000, consume=None,
                          timings: dict | None = None, wait: bool = True, code_cache: dict | None = None,
                          paths=None, write_threads: int = 16, defer: bool = False):
    """PNG bytes of every figure, composed and DEFLATE-encoded on the GPU.

    ``figures``: :class:`figure.SpectrogramFigure` objects whose panels were drawn from
    :class:`figure.DeviceRaster` references into the RGBA buffer at ``d_rgba_ptr`` (a batch's
    ``d_rgba``); annotations come from ``overlay.ATLAS``.  Same pixels as ``SpectrogramFigure.compose(dpi)``
    (the host oracle).  The device encodes the scanlines with new content; the runs of repeated lines in
    between (a resampled panel shows every raster row several times) are constants spliced in here
    (:func:`zero_run`).  Figures are processed in groups of at most ``max_segments`` scanline segments
    (scratch: 4.6 KB each).

    ``consume(first_figure_index, parts)``: instead of returning the files, hand every group's files
    -- each a list of buffers, some aliasing pinned scratch that is valid only during the call -- to the
    caller (``write_figures_device`` writes them straight to disk without assembling them in memory).
    ``timings`` (optional dict) accumulates host seconds per phase.  The DEFLATE code is a dynamic-Huffman
    code fitted to the symbol statistics of the first group of figures (one counting pass of the same
    tokeniser over every 4th scanline segment) and used for the whole call.  ``code_cache`` (a dict the
    caller keeps): the fitted code is stored there and reused by later calls instead of being fitted again
    (the chunks of one directory run look alike).

    ``paths`` (one per figure): frame and write the files natively (``csg_png_write_files``: CRC-32 +
    ``writev`` from the pinned buffer on ``write_threads`` native threads, no interpreter lock held) instead of
    building them here; nothing is returned or handed to ``consume`` then.

    ``defer=True`` (with ``wait=False``): the LAST group's encode kernel is only launched; the call returns a
    :class:`DeferredEncode` whose ``complete()`` reads the sizes back, compacts, copies out and hands the
    group to the finisher thread -- the caller does host work (plans the next chunk) while the kernel runs,
    and must call ``complete()`` before the next encode on this context.

    ``wait=False`` (needs ``consume`` or ``paths``): return as soon as the last group is read back, with the futures of
    the host work (framing + ``consume``) still running on the context's finisher thread; the caller
    collects them (``future.result()``) before it relies on the files.  The next call on the same context
    may start meanwhile -- the two pinned read-back buffers are fenced by those futures.
    """
    import time

    def tick(name, t0):
        if timings is not None:
            timings[name] = timings.get(name, 0.0) + time.perf_counter() - t0
        return time.perf_counter()

    from ._lib import PNG_CANVAS
    from .overlay import ATLAS

    lib = ctx.lib
    figures = list(figures)
    t0 = time.perf_counter()
    canvases, tiles, rows, row_maps, per_figure = _device_tables(figures, dpi)
    slot = int(lib.csg_png_slot_bytes())
    scratch = ctx.__dict__.setdefault("_png_scratch", {})
    if scratch.get("deferred") is not None:
        raise RuntimeError("a deferred encode is still open on this context: call its complete() first")
    if defer and wait:
        raise ValueError("defer=True needs wait=False")

    def dev(name, nbytes):
        buf = scratch.get(name)
        if buf is None or buf.nbytes < nbytes:
            buf = scratch[name] = ctx.alloc(int(nbytes * 1.2) + 256)
        return buf

    d_tiles, d_rows = ctx.to_device(tiles), ctx.to_device(rows)
    d_row_maps = ctx.to_device(row_maps) if row_maps is not None else None
    maps_ptr = d_row_maps.ptr if d_row_maps is not None else None
    zero_table = zero_segment_table([c[0] for c in canvases]) if canvases else np.zeros(0, dtype=np.uint8)
    d_zero = ctx.to_device(zero_table) if len(zero_table) else None
    zero_args = (d_zero.ptr if d_zero is not None else None, len(zero_table))
    d_overlay = ATLAS.device_ptr(ctx)
    d_error = dev("error", 4)
    d_error.zero()
    t0 = tick("tile_tables", t0)
    # Groups are pipelined: while a background thread frames (CRC-32) and hands over group g from one pinned
    # buffer, this thread already encodes, compacts and reads back group g + 1 into the other one.  The
    # thread and the fences of the two buffers belong to the context, so the pipeline runs across calls too.
    if not wait and consume is None and paths is None:
        raise ValueError("wait=False needs a consume callback or paths (the files are handed over, not returned)")
    if paths is not None and len(paths) != len(figures):
        raise ValueError(f"{len(paths)} paths for {len(figures)} figures")
    results: dict[int, list] = {}
    pipe = scratch.get("finisher")
    if pipe is None:
        pipe = scratch["finisher"] = {"pool": ThreadPoolExecutor(max_workers=1, thread_name_prefix="csg-png"),
                                      "framers": ThreadPoolExecutor(max_workers=16, thread_name_prefix="csg-crc"),
                                      "in_flight": [None, None], "groups": 0}
    finisher, framers, in_flight = pipe["pool"], pipe["framers"], pipe["in_flight"]  # in_flight: the future reading pinned buffer 0 / 1
    mine: list = []

    def launch(k, group, n_seg):
        """Tables of the group, the code of the call (first group), the encode kernel: nothing waits for the GPU
        except the one-time count pass."""
        t0 = time.perf_counter()
        table = np.array([tuple(c) for c in group], dtype=PNG_CANVAS)
        d_canvases = ctx.to_device(table)
        if k == 0:  # the code of this call
            if code_cache is not None and "tables" in code_cache:
                ctx._check(lib.csg_png_set_tables(ctx.handle, code_cache["tables"].ctypes.data))
            else:
                d_counts = dev("counts", 316 * 4)
                d_counts.zero()
                ctx._check(lib.csg_png_set_tables(ctx.handle, None))  # the count pass needs valid symbol tables
                ctx._check(lib.csg_png_count(ctx.handle, d_rgba_ptr, d_overlay, d_canvases.ptr, len(group), d_tiles.ptr, None,
                                             d_rows.ptr, n_seg, 4, d_counts.ptr, *zero_args, maps_ptr))
                tables = np.ascontiguousarray(custom_tables(d_counts.download(np.uint32, 316)))
                ctx._check(lib.csg_png_set_tables(ctx.handle, tables.ctypes.data))
                if code_cache is not None:
                    code_cache["tables"] = tables
            t0 = tick("code_tables", t0)
        d_slots, d_sizes, d_adler = dev("slots", n_seg * slot), dev("sizes", n_seg * 4), dev("adler", n_seg * 8)
        ctx._check(lib.csg_png_encode(ctx.handle, d_rgba_ptr, d_overlay, d_canvases.ptr, len(group), d_tiles.ptr, None,
                                      d_rows.ptr, n_seg, d_slots.ptr, d_sizes.ptr, d_adler.ptr, d_error.ptr, *zero_args, maps_ptr))
        tick("encode_launch", t0)
        return (k, group, n_seg, d_canvases, d_slots, d_sizes, d_adler)

    def complete(state):
        """Sizes back (waits for the kernel), compaction, read-back into a pinned buffer, hand-over."""
        k, group, n_seg, _d_canvases, d_slots, d_sizes, d_adler = state
        t0 = time.perf_counter()
        sizes = d_sizes.download(np.int32, n_seg, sync=False)
        bad = d_error.download(np.int32, 1, sync=False)
        adler = d_adler.download(np.uint32, 2 * n_seg).reshape(n_seg, 2)  # synchronises
        if bad[0] < 0:
            raise ValueError(f"figure {k - int(bad[0]) - 1}: a tile reads a row map, but no row-map table was given")
        if bad[0]:
            raise ValueError(f"figure {k + int(bad[0]) - 1}: more than {int(lib.csg_png_max_segment_tiles())} tiles meet in one "
                             "1024-pixel scanline segment")
        t0 = tick("encode_kernel_and_sizes", t0)
        offsets = np.zeros(n_seg + 1, dtype=np.int64)
        np.cumsum(sizes, out=offsets[1:])
        total = int(offsets[-1])
        d_off = dev("offsets", n_seg * 8)
        d_off.upload(offsets[:-1])
        d_packed = dev("packed", total)
        ctx._check(lib.csg_png_compact(ctx.handle, d_slots.ptr, d_sizes.ptr, d_off.ptr, n_seg, d_packed.ptr))
        parity = pipe["groups"] & 1
        if in_flight[parity] is not None:
            in_flight[parity].result()  # the group that last used this pinned buffer is on disk
            in_flight[parity] = None
            t0 = tick("wait_for_host", t0)
        name = f"pinned{parity}"
        pin = scratch.get(name)
        if pin is None or pin.nbytes < total:
            pin = scratch[name] = ctx.pinned(int(total * 1.2) + 4096)
        ctx._check(lib.csg_d2h(ctx.handle, pin.ptr, d_packed.ptr, total))
        ctx.sync()
        t0 = tick("compact_and_d2h", t0)

        def finish(first=k, group=group, jobs=per_figure[k : k + len(group)], packed=pin.array, offsets=offsets, adler=adler):
            t1 = time.perf_counter()
            if paths is not None:
                write_files_native(lib, paths[first : first + len(group)], group, jobs, rows, packed, offsets, adler, write_threads)
                tick("frame_and_write_native", t1)
                return
            parts = list(framers.map(lambda job: assemble_png(job[1][0], job[1][1], job[1][2], job[0][6], packed, offsets, job[0][5], adler),
                                     zip(group, jobs)))
            t1 = tick("framing_crc", t1)
            if consume is not None:
                consume(first, parts)  # the buffers alias pinned scratch that the group after next overwrites
            else:
                results[first] = [b"".join(p) for p in parts]
            tick("consume", t1)

        in_flight[parity] = finisher.submit(finish)
        mine.append(in_flight[parity])
        pipe["groups"] += 1

    def settle_failed():
        for fut in mine:  # leave no work of a failed call behind
            try:
                fut.result()
            except Exception:
                pass

    k = 0
    open_state = None
    try:
        while k < len(figures):
            # ---- the next group of figures that fits the segment budget
            group, n_seg = [], 0
            while k + len(group) < len(figures):
                c = canvases[k + len(group)]
                segs = c[6] * len(per_figure[k + len(group)][2])
                if group and n_seg + segs > max_segments:
                    break
                c[5] = n_seg
                group.append(c)
                n_seg += segs
            state = launch(k, group, n_seg)
            k += len(group)
            if defer and k >= len(figures):
                open_state = state
                break
            complete(state)
    except BaseException:
        settle_failed()
        raise
    if open_state is not None:
        keep_alive = {"tables": (d_tiles, d_rows, d_zero, d_row_maps)}  # device tables the open kernel reads

        def complete_open():
            try:
                complete(open_state)
            except BaseException:
                settle_failed()
                raise
            finally:
                scratch["deferred"] = None
                keep_alive.clear()
            return mine

        def abandon_open():
            try:
                ctx.sync()  # the kernel still reads the tables kept alive here
            finally:
                scratch["deferred"] = None
                keep_alive.clear()
                settle_failed()

        handle = DeferredEncode(complete_open, abandon_open)
        scratch["deferred"] = handle
        return handle
    if not wait:
        return mine
    t0 = time.perf_counter()
    for fut in mine:
        fut.result()
    tick("wait_for_host", t0)
    return [blob for first in sorted(results) for blob in results[first]]


class DeferredEncode:
    """The open end of ``encode_figures_device(..., defer=True)``: ``complete()`` finishes the last group and
    returns the futures of every group's host work (framing + writing)."""

    def __init__(self, complete, abandon=None):
        self._complete, self._abandon = complete, abandon
        self.futures: list | None = None

    def complete(self) -> list:
        if self._complete is not None:
            fn, self._complete, self._abandon = self._complete, None, None
            self.futures = fn()
        return self.futures or []

    def abandon(self) -> None:
        """Give the last group up (an interrupted run): wait for its kernel, release the context for the next
        encode; the groups already handed over finish as usual."""
        if self._abandon is not None:
            fn, self._complete, self._abandon = self._abandon, None, None
            fn()


def write_files_native(lib, paths, group, jobs, rows, packed, offsets, adler, n_threads: int = 16) -> None:
    """Frame and write one group's files through ``csg_png_write_files``.  ``group``: the canvases' table rows
    (``[W, H, tile_first, tile_count, background, seg_first, segs_per_row, row_first]``); ``jobs``:
    ``(W, H, content rows)`` per figure; ``rows``: every canvas' content rows, concatenated."""
    from ._lib import PNG_FILE, CsgError

    table = np.zeros(len(group), dtype=PNG_FILE)
    encoded = [os.fsencode(p) + b"\0" for p in paths]
    keep = [np.frombuffer(e, dtype=np.uint8) for e in encoded]
    for entry, c, job, name in zip(table, group, jobs, keep):
        entry["path"] = name.ctypes.data
        entry["row_first"], entry["seg_first"] = c[7], c[5]
        entry["width"], entry["height"], entry["n_rows"], entry["segs_per_row"] = c[0], c[1], len(job[2]), c[6]
    rows = np.ascontiguousarray(rows, dtype=np.int32)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    adler = np.ascontiguousarray(adler, dtype=np.uint32)
    status = lib.csg_png_write_files(table.ctypes.data, len(table), rows.ctypes.data, packed.ctypes.data, offsets.ctypes.data,
                                     adler.ctypes.data, int(n_threads))
    if status:
        bad = [(p, os.strerror(int(e["status"]))) for p, e in zip(paths, table) if e["status"]]
        if bad:
            raise OSError(f"{len(bad)} PNG file(s) not written, first: {bad[0][0]}: {bad[0][1]}")
        raise CsgError(f"csg_png_write_files failed with status {status}")


def write_figures_device(ctx, d_rgba_ptr: int, jobs, max_workers: int = 8, **kwargs):
    """``jobs``: iterable of (path, figure).  Device encode; every group's files are framed and written
    straight from the pinned read-back buffer by native threads (``csg_png_write_files``).  With
    ``wait=False`` the call returns the futures of the framing + writing still under way (see
    :func:`encode_figures_device`); the files are complete once every ``future.result()`` has returned."""
    jobs = list(jobs)
    if not jobs:
        return []
    out = encode_figures_device(ctx, d_rgba_ptr, [fig for _p, fig in jobs], paths=[str(p) for p, _f in jobs],
                                write_threads=max(1, int(max_workers)), **kwargs)
    return out if kwargs.get("wait") is False else []  # (futures, or a DeferredEncode with defer=True)
