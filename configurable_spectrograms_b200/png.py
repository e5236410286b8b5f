"""PNG hand-off for the RGBA rasters (the on-disk product of the reference:
``fast/process_orbit.py:98-117``, ``generic_batch.py:108-113``).

Two encoders, one file format (8-bit RGBA, non-interlaced):

* :func:`encode_rgba` / :func:`write_rgba` -- filter 0 + zlib DEFLATE on the host, for figures whose
  rasters are host arrays (the single-figure entry points);
* :func:`encode_figures_device` / :func:`write_figures_device` -- figures whose panels are K3 rasters
  in HBM are composed, Up-filtered and DEFLATE-encoded on the GPU (``csrc/png.cu``); only the
  compressed bytes cross PCIe.  The host adds the zlib header / trailer and the PNG chunk framing.  It
  returns the PNG bytes, writes the files and waits, or writes them deferred (``defer=True``: the last
  group's kernel still runs when the call returns).

Both decode to the same pixels (``tests/test_gpu_api.py``); the host composer is the oracle of the
device one.
"""

from __future__ import annotations

import os
import struct
import time
import zlib
from concurrent.futures import ThreadPoolExecutor
from typing import NamedTuple

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


class DeviceTables(NamedTuple):
    """What K4 reads of a list of figures (:func:`_device_tables`)."""

    canvases: np.ndarray  # PNG_CANVAS, one row per figure; seg_first counts from the figure's group (_groups)
    tiles: np.ndarray  # PNG_TILE, every figure's tiles in figure order
    rows: np.ndarray  # int32 content rows: figure k's are rows[row_first : row_first + n_rows[k]]
    n_rows: np.ndarray  # content rows per figure
    row_maps: np.ndarray | None  # int32 row maps of the panels on a log energy axis, each distinct map once


def _device_tables(figures, dpi) -> DeviceTables:
    """Tile / canvas / row tables of a list of figures (an empty tile or row table is one zero entry)."""
    from ._lib import PNG_CANVAS, PNG_TILE
    from .figure import DeviceRaster

    widths, heights, backgrounds, tile_parts, row_parts = [], [], [], [], []
    map_at, map_parts = {}, []  # row-map key -> offset in the concatenated maps
    n_map = 0
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
        r, g, b, a = t.background
        widths.append(t.W)
        heights.append(t.H)
        backgrounds.append(r | (g << 8) | (b << 16) | (a << 24))
        tile_parts.append(table)
        row_parts.append(t.content_rows(table))
    n_tiles = np.array([len(t) for t in tile_parts], dtype=np.int64)
    n_rows = np.array([len(r) for r in row_parts], dtype=np.int64)
    canvases = np.zeros(len(figures), dtype=PNG_CANVAS)
    canvases["W"], canvases["H"], canvases["background"] = widths, heights, backgrounds
    canvases["tile_first"], canvases["tile_count"] = np.cumsum(n_tiles) - n_tiles, n_tiles
    canvases["segs_per_row"] = (canvases["W"] + 1023) // 1024
    canvases["row_first"] = np.cumsum(n_rows) - n_rows
    tiles = np.concatenate(tile_parts) if n_tiles.sum() else np.zeros(1, PNG_TILE)
    rows = np.concatenate(row_parts) if n_rows.sum() else np.zeros(1, np.int32)
    row_maps = np.concatenate(map_parts).astype(np.int32) if n_map else None
    return DeviceTables(canvases, tiles, rows, n_rows, row_maps)


class _Group(NamedTuple):
    """Figures ``first .. stop - 1`` of a call: one encode kernel."""

    first: int
    stop: int
    n_seg: int  # their scanline segments


def _groups(canvases, n_rows, max_segments: int) -> list[_Group]:
    """Split the figures, in order, into groups of at most ``max_segments`` scanline segments and number every
    canvas' segments from its group's first (``seg_first``).  A group takes at least one figure, so a figure
    larger than the budget is a group of its own."""
    segs = (canvases["segs_per_row"].astype(np.int64) * n_rows).tolist()
    groups, seg_first = [], []
    first = n_seg = 0
    for k, s in enumerate(segs):
        if k > first and n_seg + s > max_segments:
            groups.append(_Group(first, k, n_seg))
            first, n_seg = k, 0
        seg_first.append(n_seg)
        n_seg += s
    if segs:
        groups.append(_Group(first, len(segs), n_seg))
    canvases["seg_first"] = seg_first
    return groups


def _tick(timings, name, t0):
    if timings is not None:
        timings[name] = timings.get(name, 0.0) + time.perf_counter() - t0
    return time.perf_counter()


class _Encoder:
    """K4's host state on one context, kept across calls: the grow-only device scratch, the two pinned read-back
    buffers with the futures of the host work that reads them, the finisher thread that frames and hands over the
    groups, its framer pool, and the open deferred encode.  Groups are pipelined: while the finisher frames
    (CRC-32) and hands over group g from one pinned buffer, the caller already encodes, compacts and reads back
    group g + 1 into the other one -- across calls too."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.scratch: dict = {}
        self.pinned: list = [None, None]
        self.in_flight: list = [None, None]  # the future of the host work reading pinned buffer 0 / 1
        self.groups = 0  # groups read back on this context: the parity of the next pinned buffer
        self.finisher = ThreadPoolExecutor(max_workers=1, thread_name_prefix="csg-png")
        self.framers = ThreadPoolExecutor(max_workers=16, thread_name_prefix="csg-crc")
        self.deferred: DeferredEncode | None = None

    @staticmethod
    def of(ctx) -> "_Encoder":
        enc = ctx.__dict__.get("_png_encoder")
        if enc is None:
            enc = ctx._png_encoder = _Encoder(ctx)
        return enc

    def dev(self, name: str, nbytes: int):
        buf = self.scratch.get(name)
        if buf is None or buf.nbytes < nbytes:
            buf = self.scratch[name] = self.ctx.alloc(int(nbytes * 1.2) + 256)
        return buf


class _Launched(NamedTuple):
    """A group whose encode kernel is enqueued.  It holds what the kernel reads: its canvas table, and through
    ``call`` the call's tiles, content rows, zero-segment table and row maps."""

    call: "_Call"
    group: _Group
    d_canvases: object
    d_slots: object
    d_sizes: object
    d_adler: object


class _Call:
    """One :func:`encode_figures_device` call: its device tables, the groups it launches and reads back, and the
    futures of their host work."""

    def __init__(self, enc: _Encoder, d_rgba_ptr: int, tables: DeviceTables, timings, code_cache, paths, write_threads):
        from .overlay import ATLAS

        ctx = enc.ctx
        self.enc, self.ctx, self.lib, self.tables = enc, ctx, ctx.lib, tables
        self.d_rgba_ptr, self.timings, self.code_cache = d_rgba_ptr, timings, code_cache
        self.paths, self.write_threads = paths, write_threads
        self.slot = int(self.lib.csg_png_slot_bytes())
        self.d_tiles, self.d_rows = ctx.to_device(tables.tiles), ctx.to_device(tables.rows)
        self.d_row_maps = ctx.to_device(tables.row_maps) if tables.row_maps is not None else None
        zero_table = zero_segment_table(tables.canvases["W"]) if len(tables.canvases) else np.zeros(0, dtype=np.uint8)
        self.d_zero = ctx.to_device(zero_table) if len(zero_table) else None
        self.zero_args = (self.d_zero.ptr if self.d_zero is not None else None, len(zero_table))
        self.maps_ptr = self.d_row_maps.ptr if self.d_row_maps is not None else None
        self.d_overlay = ATLAS.device_ptr(ctx)
        self.d_error = enc.dev("error", 4)
        self.d_error.zero()
        self.futures: list = []
        self.results: dict[int, list] = {}

    def tick(self, name, t0):
        return _tick(self.timings, name, t0)

    def launch(self, group: _Group) -> _Launched:
        """The group's canvas table, the code of the call (first group), the encode kernel: nothing waits for the
        GPU except the one-time count pass."""
        ctx, lib, enc, n_seg = self.ctx, self.lib, self.enc, group.n_seg
        t0 = time.perf_counter()
        d_canvases = ctx.to_device(self.tables.canvases[group.first : group.stop])
        n_canvases = group.stop - group.first
        if group.first == 0:  # the code of this call
            if self.code_cache is not None and "tables" in self.code_cache:
                ctx._check(lib.csg_png_set_tables(ctx.handle, self.code_cache["tables"].ctypes.data))
            else:
                d_counts = enc.dev("counts", 316 * 4)
                d_counts.zero()
                ctx._check(lib.csg_png_set_tables(ctx.handle, None))  # the count pass needs valid symbol tables
                ctx._check(lib.csg_png_count(ctx.handle, self.d_rgba_ptr, self.d_overlay, d_canvases.ptr, n_canvases,
                                             self.d_tiles.ptr, None, self.d_rows.ptr, n_seg, 4, d_counts.ptr,
                                             *self.zero_args, self.maps_ptr))
                tables = np.ascontiguousarray(custom_tables(d_counts.download(np.uint32, 316)))
                ctx._check(lib.csg_png_set_tables(ctx.handle, tables.ctypes.data))
                if self.code_cache is not None:
                    self.code_cache["tables"] = tables
            t0 = self.tick("code_tables", t0)
        d_slots, d_sizes, d_adler = enc.dev("slots", n_seg * self.slot), enc.dev("sizes", n_seg * 4), enc.dev("adler", n_seg * 8)
        ctx._check(lib.csg_png_encode(ctx.handle, self.d_rgba_ptr, self.d_overlay, d_canvases.ptr, n_canvases, self.d_tiles.ptr,
                                      None, self.d_rows.ptr, n_seg, d_slots.ptr, d_sizes.ptr, d_adler.ptr, self.d_error.ptr,
                                      *self.zero_args, self.maps_ptr))
        self.tick("encode_launch", t0)
        return _Launched(self, group, d_canvases, d_slots, d_sizes, d_adler)

    def complete(self, launched: _Launched) -> None:
        """Sizes back (waits for the kernel), compaction, read-back into a pinned buffer, hand-over to the finisher."""
        ctx, lib, enc = self.ctx, self.lib, self.enc
        group, n_seg = launched.group, launched.group.n_seg
        t0 = time.perf_counter()
        sizes = launched.d_sizes.download(np.int32, n_seg, sync=False)
        bad = self.d_error.download(np.int32, 1, sync=False)
        adler = launched.d_adler.download(np.uint32, 2 * n_seg).reshape(n_seg, 2)  # synchronises
        if bad[0] < 0:
            raise ValueError(f"figure {group.first - int(bad[0]) - 1}: a tile reads a row map, but no row-map table was given")
        if bad[0]:
            raise ValueError(f"figure {group.first + int(bad[0]) - 1}: more than {int(lib.csg_png_max_segment_tiles())} tiles "
                             "meet in one 1024-pixel scanline segment")
        t0 = self.tick("encode_kernel_and_sizes", t0)
        offsets = np.zeros(n_seg + 1, dtype=np.int64)
        np.cumsum(sizes, out=offsets[1:])
        total = int(offsets[-1])
        d_off = enc.dev("offsets", n_seg * 8)
        d_off.upload(offsets[:-1])
        d_packed = enc.dev("packed", total)
        ctx._check(lib.csg_png_compact(ctx.handle, launched.d_slots.ptr, launched.d_sizes.ptr, d_off.ptr, n_seg, d_packed.ptr))
        parity = enc.groups & 1
        if enc.in_flight[parity] is not None:
            enc.in_flight[parity].result()  # the group that last used this pinned buffer is handed over
            enc.in_flight[parity] = None
            t0 = self.tick("wait_for_host", t0)
        pin = enc.pinned[parity]
        if pin is None or pin.nbytes < total:
            pin = enc.pinned[parity] = ctx.pinned(int(total * 1.2) + 4096)
        ctx._check(lib.csg_d2h(ctx.handle, pin.ptr, d_packed.ptr, total))
        ctx.sync()
        self.tick("compact_and_d2h", t0)
        enc.in_flight[parity] = enc.finisher.submit(self._finish, group, pin.array, offsets, adler)
        self.futures.append(enc.in_flight[parity])
        enc.groups += 1

    def _finish(self, group: _Group, packed, offsets, adler) -> None:
        """The host work of a read-back group, on the finisher thread: its files framed and written natively, or
        framed into bytes."""
        t1 = time.perf_counter()
        canvases = self.tables.canvases[group.first : group.stop]
        n_rows = self.tables.n_rows[group.first : group.stop]
        if self.paths is not None:
            write_files_native(self.lib, self.paths[group.first : group.stop], canvases, n_rows, self.tables.rows, packed,
                               offsets, adler, self.write_threads)
            self.tick("frame_and_write_native", t1)
            return
        rows = self.tables.rows

        def frame(canvas, n):
            first = int(canvas["row_first"])
            return assemble_png(int(canvas["W"]), int(canvas["H"]), rows[first : first + int(n)], int(canvas["segs_per_row"]),
                                packed, offsets, int(canvas["seg_first"]), adler)

        parts = list(self.enc.framers.map(frame, canvases, n_rows))
        t1 = self.tick("framing_crc", t1)
        self.results[group.first] = [b"".join(p) for p in parts]
        self.tick("consume", t1)  # the join keeps this phase name, so bench lines stay comparable

    def settle(self) -> None:
        """Leave no host work of a failed or abandoned call behind."""
        for fut in self.futures:
            try:
                fut.result()
            except Exception:
                pass

    def wait(self) -> list:
        """Every group's host work done: the PNG files (an empty list when they were written)."""
        t0 = time.perf_counter()
        for fut in self.futures:
            fut.result()
        self.tick("wait_for_host", t0)
        return [blob for first in sorted(self.results) for blob in self.results[first]]


def encode_figures_device(ctx, d_rgba_ptr: int, figures, dpi: float | None = None, max_segments: int = 400_000,
                          timings: dict | None = None, code_cache: dict | None = None, paths=None, write_threads: int = 16,
                          defer: bool = False):
    """PNG bytes of every figure, composed and DEFLATE-encoded on the GPU.

    ``figures``: :class:`figure.SpectrogramFigure` objects whose panels were drawn from
    :class:`figure.DeviceRaster` references into the RGBA buffer at ``d_rgba_ptr`` (a batch's
    ``d_rgba``); annotations come from ``overlay.ATLAS``.  Same pixels as ``SpectrogramFigure.compose(dpi)``
    (the host oracle).  The device encodes the scanlines with new content; the runs of repeated lines in
    between (a resampled panel shows every raster row several times) are constants spliced in here
    (:func:`zero_run`).  Figures are processed in groups of at most ``max_segments`` scanline segments
    (scratch: 4.6 KB each).

    ``timings`` (optional dict) accumulates host seconds per phase.  The DEFLATE code is a dynamic-Huffman
    code fitted to the symbol statistics of the first group of figures (one counting pass of the same
    tokeniser over every 4th scanline segment) and used for the whole call.  ``code_cache`` (a dict the
    caller keeps): the fitted code is stored there and reused by later calls instead of being fitted again
    (the chunks of one directory run look alike).

    ``paths`` (one per figure): frame and write the files natively (``csg_png_write_files``: CRC-32 +
    ``writev`` from the pinned buffer on ``write_threads`` native threads, no interpreter lock held) instead of
    building them here; the call returns an empty list once they are written.

    ``defer=True`` (needs ``paths``): the LAST group's encode kernel is only launched; the call returns a
    :class:`DeferredEncode` whose ``complete()`` reads the sizes back, compacts, copies out and hands the
    group to the finisher thread -- the caller does host work (plans the next chunk) while the kernel runs,
    and must call ``complete()`` or ``abandon()`` before the next encode on this context.  The files are
    complete once every future ``complete()`` returns has its ``result()``.
    """
    figures = list(figures)
    t0 = time.perf_counter()
    tables = _device_tables(figures, dpi)
    enc = _Encoder.of(ctx)
    if enc.deferred is not None:
        raise RuntimeError("a deferred encode is still open on this context: call its complete() first")
    if defer and paths is None:
        raise ValueError("defer=True needs paths (the files are written, not returned)")
    if paths is not None and len(paths) != len(figures):
        raise ValueError(f"{len(paths)} paths for {len(figures)} figures")
    call = _Call(enc, d_rgba_ptr, tables, timings, code_cache, paths, write_threads)
    _tick(timings, "tile_tables", t0)
    groups = _groups(tables.canvases, tables.n_rows, max_segments)
    last = groups.pop() if defer and groups else None
    try:
        for group in groups:
            call.complete(call.launch(group))
        if last is not None:
            last = call.launch(last)
    except BaseException:
        call.settle()
        raise
    if not defer:
        return call.wait()
    handle = DeferredEncode(last)
    if last is not None:
        enc.deferred = handle
    return handle


class DeferredEncode:
    """The open end of ``encode_figures_device(..., defer=True)``: its last group, whose encode kernel may still
    run.  ``complete()`` finishes that group and returns the futures of every group's host work (framing +
    writing)."""

    def __init__(self, last: _Launched | None):
        self._last = last
        self.futures: list | None = None if last is not None else []

    def complete(self) -> list:
        last, self._last = self._last, None
        if last is not None:
            call = last.call
            try:
                call.complete(last)
            except BaseException:
                call.settle()
                raise
            finally:
                call.enc.deferred = None
            self.futures = call.futures
        return self.futures or []

    def abandon(self) -> None:
        """Give the last group up (an interrupted run): wait for its kernel, release the context for the next
        encode; the groups already handed over finish as usual."""
        last, self._last = self._last, None
        if last is not None:
            call = last.call
            try:
                call.ctx.sync()  # the kernel still reads the tables `last` holds
            finally:
                call.enc.deferred = None
                call.settle()


def write_files_native(lib, paths, canvases, n_rows, rows, packed, offsets, adler, n_threads: int = 16) -> None:
    """Frame and write one group's files through ``csg_png_write_files``.  ``canvases``: the figures' ``PNG_CANVAS``
    rows; ``n_rows``: their content rows each; ``rows``: every canvas' content rows, concatenated."""
    from ._lib import PNG_FILE, CsgError

    table = np.zeros(len(canvases), dtype=PNG_FILE)
    keep = [np.frombuffer(os.fsencode(p) + b"\0", dtype=np.uint8) for p in paths]
    table["path"] = [name.ctypes.data for name in keep]
    table["row_first"], table["seg_first"] = canvases["row_first"], canvases["seg_first"]
    table["width"], table["height"] = canvases["W"], canvases["H"]
    table["n_rows"], table["segs_per_row"] = n_rows, canvases["segs_per_row"]
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
    straight from the pinned read-back buffer by native threads (``csg_png_write_files``).  Returns ``[]`` once
    the files are written, or with ``defer=True`` the :class:`DeferredEncode` of the last group (see
    :func:`encode_figures_device`)."""
    jobs = list(jobs)
    if not jobs:
        return []
    return encode_figures_device(ctx, d_rgba_ptr, [fig for _p, fig in jobs], paths=[str(p) for p, _f in jobs],
                                 write_threads=max(1, int(max_workers)), **kwargs)
