"""Batched device engine over libcsgpu: cubes -> sums -> stats -> norms -> rasters.

A :class:`Batch` holds every counts cube of one dtype resident in HBM together with
the descriptor tables the kernels walk (files, regions, panels, index pool).  The
reference-shaped host functions (``plotting.make_spectrogram`` ...) build batches of
one file; the FAST batch driver builds one batch per GPU shard.

Data layout in HBM (DESIGN.md section 3):
  cubes   one allocation, each file 256-byte aligned, in its stored dtype (D, or an 8/16/32-bit
          integer type when D is float64)
  sums    per file [(G+1)][E][Tp] dtype D, energy-major (group 0 = every pitch bin; Tp = T
          rounded up to a multiple of 4) -- the orientation imshow draws (matrix_plot = collapsed.T)
  flags   per file [T] uint8 (bit g: a non-NaN cell exists in row t of group g)
  pool    int32 column / row index lists shared by regions
  rgba / index   per panel [E'][T'] uint32 / uint16, row 0 = lowest energy
"""

from __future__ import annotations

import ctypes as C
from collections import namedtuple

import numpy as np

from . import _lib
from ._lib import (
    FILE_DESC,
    FLAG_WINDOW,
    PANEL,
    PANEL_NORM,
    REGION,
    REGION_STATS,
    Context,
    CsgError,
    DevBuf,
    np_cube_code,
    np_dtype_code,
)


#: One row of the region, panel and zoom-window tables, with the fields of the ABI mirror dtypes in
#: their order: ``np.array(rows, dtype=REGION)`` is the table the kernels read.
RegionRow = namedtuple("RegionRow", REGION.names)
PanelRow = namedtuple("PanelRow", PANEL.names)
WindowRow = namedtuple("WindowRow", FLAG_WINDOW.names)

#: ``csg_region.want_pct``: what K2a computes for a region
WANT_REDUCTIONS, WANT_PERCENTILES, WANT_GEOMETRY = 0, 1, 2
# a region asked for more than once keeps the most it was asked for
_WANT_RANK = {WANT_GEOMETRY: 0, WANT_REDUCTIONS: 1, WANT_PERCENTILES: 2}


def _align(n: int, a: int = 256) -> int:
    return (n + a - 1) // a * a


def compute_dtype(cube_dtype) -> np.dtype:
    """The dtype numpy computes a cube of ``cube_dtype`` in: float32 / float64 stay; integer counts go through
    float64 (``np.nansum`` sums them exactly in int64 / uint64; ``np.nanpercentile`` and matplotlib work in float64)."""
    dt = np.dtype(cube_dtype)
    return dt if dt in (np.float32, np.float64) else np.dtype(np.float64)


def classify_cube(cube: np.ndarray):
    """(array to upload, layout, (T,P,E)) for a (time, pitch, energy) cube or view.

    ``load_fast_cdf_dataset`` hands out either a C-contiguous (T,P,E) array or the
    transposed *view* of a stored (T,E,P) array (reference ``cdf_utils.py:254-255``);
    numpy's ``nansum(axis=1)`` adds in a different order for the two, so the storage
    order is part of the input.
    """
    if cube.ndim != 3:
        raise ValueError(f"expected a 3-D (time, pitch, energy) cube, got shape {cube.shape}")
    T, P, E = cube.shape
    if cube.flags.c_contiguous:
        return cube, _lib.LAYOUT_TPE, (T, P, E)
    stored = cube.transpose(0, 2, 1)
    if stored.flags.c_contiguous:
        return stored, _lib.LAYOUT_TEP, (T, P, E)
    return np.ascontiguousarray(cube), _lib.LAYOUT_TPE, (T, P, E)


class ZSlot(float):
    """A z bound that lives in the batch's device table ``d_zvals`` instead of in the panel.

    Behaves like the float it currently holds; panels built from it reference ``slot``, so the
    bound can change every step (global extrema of this step) without re-planning the panels.
    Two slots never compare equal, even when they hold the same value right now.
    """

    __slots__ = ("slot",)

    def __new__(cls, value, slot: int):
        obj = super().__new__(cls, np.nan if value is None else value)
        obj.slot = int(slot)
        return obj

    def __eq__(self, other):
        return isinstance(other, ZSlot) and other.slot == self.slot

    def __ne__(self, other):
        return not self.__eq__(other)

    def __hash__(self):
        return hash(("ZSlot", self.slot))


class Batch:
    """Cubes of one compute dtype D on one GPU plus the tables of everything to compute from them.

    A float64 batch also takes 8/16/32-bit integer cubes (``_lib.INT_CUBE_CODES``): K1 reads them at their
    stored width and writes float64 sums, the same bits as the cube widened to float64."""

    def __init__(self, ctx: Context, dtype, n_groups: int = 0):
        if not 0 <= n_groups <= _lib.MAX_GROUPS:
            raise ValueError(f"n_groups must be 0..{_lib.MAX_GROUPS}")
        self.ctx = ctx
        self.dtype = np.dtype(dtype)
        self.code = np_dtype_code(dtype)
        self.G = int(n_groups)
        self.files: list[dict] = []
        self._regions: list[RegionRow] = []
        self._panels: list[PanelRow] = []
        self._pool: list[np.ndarray] = []
        self._pool_len = 0
        self._pool_cache: dict[bytes, int] = {}
        self._sums_elems = 0
        self._flags_bytes = 0
        self._bits: list[np.ndarray] = []
        self._bits_len = 0
        self._cube_bytes = 0
        self._pixels = 0
        # device state
        self.d_cubes: DevBuf | None = None
        self.d_sums: DevBuf | None = None
        self.d_flags: DevBuf | None = None
        self.d_bits: DevBuf | None = None
        self.d_runs: DevBuf | None = None
        self.d_files: dict[int, tuple[DevBuf, int, int, int]] = {}
        self.d_regions: DevBuf | None = None
        self.d_pool: DevBuf | None = None
        self.d_stats: DevBuf | None = None
        self.d_panels: DevBuf | None = None
        self.d_norms: DevBuf | None = None
        self.d_rgba: DevBuf | None = None
        self.d_index: DevBuf | None = None
        self.d_lut: DevBuf | None = None
        self.d_thr: DevBuf | None = None
        self.d_zvals: DevBuf | None = None
        self._windows: list[WindowRow] = []
        self.d_windows: DevBuf | None = None
        self.d_window_any: DevBuf | None = None
        self._zvals: list[float] = []
        self._zvals_dirty = False
        self._raster_blocks = 0
        self._tables_dirty = True
        self._runs_cache: dict[bytes, tuple] = {}
        self._table_bufs: dict[str, DevBuf] = {}
        self.d_stage: DevBuf | None = None  # collapse_pending(): the cubes of one call
        self._n_collapsed = 0
        self._sums_valid_bytes = 0
        self._flags_valid_bytes = 0

    # ------------------------------------------------------------------ files
    def add_file(self, cube: np.ndarray | None, pa_bits: np.ndarray | None = None, *, shape=None, layout=None, device_ptr=None,
                 cube_dtype=None) -> int:
        """Register one cube (host array, or a device pointer with ``shape``/``layout`` and ``cube_dtype``, by
        default the batch dtype)."""
        if cube is not None:
            if cube.dtype != self.dtype and not (self.dtype == np.float64 and cube.dtype in _lib.INT_CUBE_CODES):
                raise TypeError(f"cube dtype {cube.dtype} != batch dtype {self.dtype}")
            host, layout, (T, P, E) = classify_cube(cube)
            cube_dtype = cube.dtype
        else:
            host = None
            T, P, E = shape
            layout = _lib.LAYOUT_TPE if layout is None else layout
            cube_dtype = self.dtype if cube_dtype is None else np.dtype(cube_dtype)
            if cube_dtype != self.dtype and not (self.dtype == np.float64 and cube_dtype in _lib.INT_CUBE_CODES):
                raise TypeError(f"cube dtype {cube_dtype} != batch dtype {self.dtype}")
        if self.G > 0:
            if pa_bits is None or len(pa_bits) != P:
                raise ValueError("pa_bits (uint8[P]) is required when the batch has pitch-angle groups")
            bits = np.ascontiguousarray(pa_bits, dtype=np.uint8)
        else:
            bits = np.zeros(P, dtype=np.uint8)
        f = {
            "T": T,
            "P": P,
            "E": E,
            "layout": layout,
            "dtype": np.dtype(cube_dtype),
            "code": np_cube_code(cube_dtype),
            "host": host,
            "device_ptr": device_ptr,
            "cube_off": self._cube_bytes,
            "sums_off": self._sums_elems,
            "flags_off": self._flags_bytes,
            "bits_off": self._bits_len,
        }
        f["Tp"] = (T + 3) // 4 * 4
        self._cube_bytes += _align(T * P * E * f["dtype"].itemsize)
        self._sums_elems += _align((self.G + 1) * E * f["Tp"] * self.dtype.itemsize) // self.dtype.itemsize
        self._flags_bytes += _align(T, 4)
        self._bits.append(bits)
        self._bits_len += P
        self.files.append(f)
        self._tables_dirty = True
        return len(self.files) - 1

    @property
    def cube_bytes(self) -> int:
        return sum(f["T"] * f["P"] * f["E"] * f["dtype"].itemsize for f in self.files)

    def upload_cubes(self):
        """H2D of every host cube into one device allocation (async on the ctx stream)."""
        need = any(f["host"] is not None for f in self.files)
        if need and (self.d_cubes is None or self.d_cubes.nbytes < self._cube_bytes):
            self.d_cubes = self.ctx.alloc(self._cube_bytes)
        for f in self.files:
            if f["host"] is not None:
                self.d_cubes.upload(f["host"], f["cube_off"])
                f["device_ptr"] = self.d_cubes.ptr + f["cube_off"]
        self._tables_dirty = True

    def _table(self, name: str, arr: np.ndarray) -> DevBuf:
        """Upload a small table into a persistent, grow-only device buffer (stream-ordered re-use: the
        kernels still reading the previous contents precede this copy on the stream; no cudaFree /
        cudaMalloc -- both synchronise the device -- in a steady-state streaming loop)."""
        arr = np.ascontiguousarray(arr)
        buf = self._table_bufs.get(name)
        if buf is None or buf.nbytes < arr.nbytes:
            buf = self._table_bufs[name] = self.ctx.alloc(max(2 * arr.nbytes, 4096))
        buf.upload(arr)
        return buf

    def _file_tables(self, indices, ptr_of, tag="all"):
        """Descriptor tables for the files ``indices``: one per (storage layout, K1 kernel, E) and cube dtype -- a
        launch handles files of one kind; the key of an integer file's table ends with its cube dtype code.
        ``ptr_of(i)``: device address of file i's cube.  Returns ``({key: (table, n, blocks, max_P, max_E)}, d_runs,
        d_bits)``; the pitch-angle membership bytes
        are packed for these files only (``bits_off`` is local to the returned ``d_bits``)."""
        lib = self.ctx.lib
        indices = list(indices)
        groups: dict[tuple, list[int]] = {}
        for i in indices:
            f = self.files[i]
            if f["T"] <= 0:
                continue
            kern = lib.csg_collapse_kernel_for(f["T"], f["P"], f["E"], f["code"], f["layout"], ptr_of(i), self.G)
            # every file of a stream-kernel table shares one energy count (it fixes the block shape)
            key = (f["layout"], kern, f["E"] if kern == _lib.K1_STREAM else 0)
            groups.setdefault(key if f["code"] == self.code else key + (f["code"],), []).append(i)
        # runs of constant pitch-angle group membership (stream kernel), one entry per distinct table
        runs_tab: list[np.ndarray] = []
        runs_len = 0
        runs_of: dict[bytes, tuple[int, int, int]] = {}
        for (layout, kern, *_), idx in groups.items():
            if kern != _lib.K1_STREAM:
                continue
            for i in idx:
                bits = self._bits[i]
                key = bits.tobytes()
                if key not in runs_of:
                    hit = self._runs_cache.get(key)
                    if hit is None:
                        buf = np.zeros(3 * len(bits) + 3, dtype=np.int32)
                        alias = C.c_int32(0)
                        n = lib.csg_pitch_runs(bits.ctypes.data, len(bits), self.G, buf.ctypes.data, C.byref(alias))
                        hit = self._runs_cache[key] = (buf[: 3 * n].copy(), n, int(alias.value))
                    runs_of[key] = (runs_len, hit[1], hit[2])
                    runs_tab.append(hit[0])
                    runs_len += hit[1]
        d_runs = self._table(f"{tag}_runs", np.concatenate(runs_tab)) if runs_tab else None
        bits_off, off = {}, 0
        for i in indices:
            bits_off[i] = off
            off += len(self._bits[i])
        tables = {}
        for key, idx in groups.items():
            layout, kern, code = key[0], key[1], self._key_code(key)
            tab = np.zeros(len(idx), dtype=FILE_DESC)
            blocks, max_p, max_e = 0, 1, 1
            for j, i in enumerate(idx):
                f = self.files[i]
                tab[j]["d_cube"] = ptr_of(i)
                tab[j]["sums_off"] = f["sums_off"]
                tab[j]["flags_off"] = f["flags_off"]
                tab[j]["T"], tab[j]["P"], tab[j]["E"] = f["T"], f["P"], f["E"]
                tab[j]["bits_off"] = bits_off[i]
                tab[j]["first_block"] = blocks
                if kern == _lib.K1_STREAM:
                    tab[j]["reserved"] = runs_of[self._bits[i].tobytes()]
                blocks += lib.csg_collapse_blocks(f["T"], f["P"], f["E"], code, layout, kern)
                max_p, max_e = max(max_p, f["P"]), max(max_e, f["E"])
            tables[key] = (self._table(f"{tag}_files_" + "_".join(map(str, key)), tab), len(idx), blocks, max_p, max_e)
        packed = [self._bits[i] for i in indices]
        d_bits = self._table(f"{tag}_bits", np.concatenate(packed) if packed else np.zeros(1, np.uint8))
        return tables, d_runs, d_bits

    def _ensure_outputs_of_k1(self):
        """Room for every registered file's sums and row flags; what is already there survives a growth
        (a device-to-device copy on the stream, ordered after the kernels that wrote it)."""
        need = max(self._sums_elems, 1) * self.dtype.itemsize
        if self.d_sums is None or self.d_sums.nbytes < need:
            old, used = self.d_sums, self._sums_valid_bytes
            self.d_sums = self.ctx.alloc(need if old is None else max(need, 2 * old.nbytes))
            if old is not None and used:
                self.ctx._check(self.ctx.lib.csg_d2d(self.ctx.handle, self.d_sums.ptr, old.ptr, used))
                self.ctx.sync()  # `old` is freed when it goes out of scope
        need = max(self._flags_bytes, 4)
        if self.d_flags is None or self.d_flags.nbytes < need:
            old, used = self.d_flags, self._flags_valid_bytes
            self.d_flags = self.ctx.alloc(need if old is None else max(need, 2 * old.nbytes))
            if old is not None and used:
                self.ctx._check(self.ctx.lib.csg_d2d(self.ctx.handle, self.d_flags.ptr, old.ptr, used))
                self.ctx.sync()

    def _build_file_tables(self):
        """Tables over EVERY file (cubes resident in HBM: the all-at-once path)."""
        for f in self.files:
            if f["T"] > 0 and f["device_ptr"] is None:
                raise CsgError("cube not on the device: call upload_cubes() first")
        self.d_files, self.d_runs, self.d_bits = self._file_tables(range(len(self.files)), lambda i: self.files[i]["device_ptr"])
        self._ensure_outputs_of_k1()
        self._tables_dirty = False

    def _key_code(self, key) -> int:
        """Cube dtype code of a K1 table key (see :meth:`_file_tables`)."""
        return key[3] if len(key) > 3 else self.code

    def _launch_k1(self, tables, d_runs, d_bits):
        for key, (tab, n, blocks, max_p, max_e) in tables.items():
            self.ctx._check(
                self.ctx.lib.csg_collapse(
                    self.ctx.handle, tab.ptr, n, blocks, d_bits.ptr, d_runs.ptr if d_runs is not None else None, self.G,
                    max_p, max_e, self._key_code(key), key[0], key[1], self.d_sums.ptr, self.d_flags.ptr,
                )
            )

    def collapse(self):
        """K1 over every file (one launch per storage layout / kernel / block shape present)."""
        if self._tables_dirty:
            self._build_file_tables()
        self.d_flags.zero()
        self._launch_k1(self.d_files, self.d_runs, self.d_bits)
        self._sums_valid_bytes = self._sums_elems * self.dtype.itemsize
        self._flags_valid_bytes = self._flags_bytes
        self._n_collapsed = len(self.files)

    def collapse_pending(self):
        """Streaming ingest: upload and collapse the files registered since the last call, then forget
        their cubes.  The cubes pass through ONE device staging buffer (stream order: this call's uploads
        wait for the previous call's K1), so HBM holds the sums and flags of everything but the cubes of
        one call only; host arrays are released as soon as the copies are enqueued -- from pinned memory
        (``_lib.PinnedRing``) the copy is asynchronous, and the caller re-uses a slot once the event it
        records after this call has passed.  Returns the number of files collapsed."""
        first = self._n_collapsed
        todo = [i for i in range(first, len(self.files)) if self.files[i]["T"] > 0]
        self._ensure_outputs_of_k1()
        new_flags = self._flags_bytes - self._flags_valid_bytes
        if new_flags > 0:
            self.ctx._check(self.ctx.lib.csg_memset(self.ctx.handle, self.d_flags.ptr + self._flags_valid_bytes, 0, new_flags))
        if todo:
            base = self.files[todo[0]]["cube_off"]
            span = self._cube_bytes - base
            if self.d_stage is None or self.d_stage.nbytes < span:
                self.d_stage = None  # free before the larger allocation
                self.d_stage = self.ctx.alloc(span)
            # the small tables first: their (pageable) uploads wait for the stream, which at this point holds
            # the PREVIOUS call's copies and K1 only -- normally long finished while the host was decoding
            tables, d_runs, d_bits = self._file_tables(todo, lambda i: self.d_stage.ptr + self.files[i]["cube_off"] - base,
                                                       tag="pending")
            for i in todo:
                f = self.files[i]
                if f["host"] is None:
                    raise CsgError("collapse_pending() needs host cubes (device-resident files use collapse())")
                self.d_stage.upload(f["host"], f["cube_off"] - base, keep=False)
            self._launch_k1(tables, d_runs, d_bits)
            for i in todo:
                self.files[i]["host"] = None
        self._sums_valid_bytes = self._sums_elems * self.dtype.itemsize
        self._flags_valid_bytes = self._flags_bytes
        self._n_collapsed = len(self.files)
        self._tables_dirty = True
        return len(todo)

    def mat_off(self, file: int, group: int) -> int:
        """Element offset of the file's energy-major [E][Tp] matrix of one group in the sums buffer."""
        f = self.files[file]
        return f["sums_off"] + group * f["E"] * f["Tp"]

    def sums(self, file: int, group: int = 0) -> np.ndarray:
        """Download one collapsed matrix in numpy's (T, E) orientation (``np.nansum(cube, axis=1)``)."""
        f = self.files[file]
        if f["T"] == 0:
            return np.zeros((0, f["E"]), dtype=self.dtype)
        n = f["E"] * f["Tp"]
        a = self.d_sums.download(self.dtype, n, self.mat_off(file, group) * self.dtype.itemsize)
        return np.ascontiguousarray(a.reshape(f["E"], f["Tp"])[:, : f["T"]].T)

    def flags(self, file: int) -> np.ndarray:
        f = self.files[file]
        return self.d_flags.download(np.uint8, f["T"], f["flags_off"]) if f["T"] else np.zeros(0, np.uint8)

    # ---------------------------------------------------------------- regions
    def _pool_add(self, idx: np.ndarray) -> int:
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        key = idx.tobytes()
        off = self._pool_cache.get(key)
        if off is None:
            off = self._pool_len
            self._pool.append(idx)
            self._pool_len += len(idx)
            self._pool_cache[key] = off
        return off

    def reset_tables(self):
        """Forget every region / panel / window / z slot (the cubes and their sums stay)."""
        self._regions, self._panels, self._pool, self._windows, self._zvals = [], [], [], [], []
        self._pool_len, self._pool_cache = 0, {}
        self._raster_blocks = self._pixels = 0
        self._zvals_dirty = False
        self.d_regions = self.d_panels = self.d_windows = self.d_window_any = None

    def add_region(self, file: int, group: int, cols, *, t0: int = 0, nt: int | None = None, rows=None,
                   want_pct: bool | int = WANT_REDUCTIONS, p_lo: float = 1.0, p_hi: float = 99.0) -> int:
        """``want_pct``: ``WANT_REDUCTIONS`` (or False), ``WANT_PERCENTILES`` (or True) or ``WANT_GEOMETRY``."""
        f = self.files[file]
        cols = np.asarray(cols, dtype=np.int32)
        if rows is not None:
            rows = np.asarray(rows, dtype=np.int32)
            # contiguous runs need no list
            if len(rows) > 0 and np.array_equal(rows, np.arange(rows[0], rows[0] + len(rows), dtype=np.int32)):
                t0, nt, rows = int(rows[0]), len(rows), None
            elif len(rows) == 0:
                t0, nt, rows = 0, 0, None
        if rows is None:
            nt = f["T"] - t0 if nt is None else nt
            rows_off = -1
        else:
            rows_off = self._pool_add(rows)
            t0, nt = 0, len(rows)
        cols_off = self._pool_add(cols) if len(cols) else 0
        self._regions.append(
            RegionRow(mat_off=self.mat_off(file, group), ld=f["Tp"], t0=t0, nt=nt, rows_off=rows_off, cols_off=cols_off,
                      ne=len(cols), want_pct=int(want_pct), reserved=0, p_lo=float(p_lo), p_hi=float(p_hi))
        )
        return len(self._regions) - 1

    def require_stats(self, region: int, want_pct: int):
        """Make K2a compute at least ``want_pct`` for a region, in the order geometry < reductions <
        percentiles; a region never loses what it was already asked for."""
        r = self._regions[region]
        if _WANT_RANK[int(want_pct)] > _WANT_RANK[r.want_pct]:
            self._regions[region] = r._replace(want_pct=int(want_pct))

    def drop_reductions(self, region: int):
        """A region whose reductions no panel reads any more becomes geometry only (percentiles stay)."""
        r = self._regions[region]
        if r.want_pct == WANT_REDUCTIONS:
            self._regions[region] = r._replace(want_pct=WANT_GEOMETRY)

    def zslot(self, value=None) -> ZSlot:
        """A new slot of the per-step z-bound table (``None`` = not given -> percentile bound)."""
        self._zvals.append(np.nan if value is None else float(value))
        self._zvals_dirty = True
        return ZSlot(value, len(self._zvals) - 1)

    def set_zslot(self, slot: int, value):
        value = np.nan if value is None else float(value)
        old = self._zvals[slot]
        if not (old == value or (old != old and value != value)):
            self._zvals[slot] = value
            self._zvals_dirty = True

    def add_window(self, file: int, bit: int, rows) -> int:
        """A zoom window over the K1 row flags: ``rows`` = (t0, nt) or an index array."""
        f = self.files[file]
        if isinstance(rows, tuple):
            t0, nt, rows_off = int(rows[0]), int(rows[1]), -1
        else:
            rows = np.asarray(rows, dtype=np.int32)
            if len(rows) and np.array_equal(rows, np.arange(rows[0], rows[0] + len(rows), dtype=np.int32)):
                t0, nt, rows_off = int(rows[0]), len(rows), -1
            else:
                t0, nt, rows_off = 0, len(rows), (self._pool_add(rows) if len(rows) else -1)
        self._windows.append(WindowRow(flags_off=f["flags_off"], t0=t0, nt=nt, rows_off=rows_off, bit=int(bit)))
        return len(self._windows) - 1

    def run_windows(self):
        """d_window_any[w] = any row of window w holds a non-NaN cell of its group (K1 flags)."""
        if not self._windows:
            return
        self.ctx._check(
            self.ctx.lib.csg_window_any(
                self.ctx.handle, self.d_flags.ptr, self.d_windows.ptr, len(self._windows), self.d_pool.ptr,
                self.d_window_any.ptr,
            )
        )

    def window_any(self) -> np.ndarray:
        """Download the result of :meth:`run_windows`: uint8 per window."""
        if not self._windows:
            return np.zeros(0, np.uint8)
        return self.d_window_any.download(np.uint8, len(self._windows))

    def _pool_array(self) -> np.ndarray:
        if getattr(self, "_pool_flat_len", -1) != self._pool_len:
            self._pool_flat = np.concatenate(self._pool) if self._pool else np.zeros(0, np.int32)
            self._pool_flat_len = self._pool_len
        return self._pool_flat

    def region_energy_index(self, region: int) -> np.ndarray:
        """Energy channel of every image row of a region (lowest energy first)."""
        r = self._regions[region]
        return self._pool_array()[r.cols_off : r.cols_off + r.ne]

    def region_time_ends(self, region: int) -> tuple[int, int]:
        """Time steps of the first and last image column of a region."""
        r = self._regions[region]
        if r.rows_off < 0:
            return r.t0, r.t0 + r.nt - 1
        pool = self._pool_array()
        return int(pool[r.rows_off]), int(pool[r.rows_off + r.nt - 1])

    def add_panel(self, region: int, pct_region: int = -1, log_scale: bool = False, z_min=None, z_max=None,
                  stat_region: int = -1) -> int:
        r = self._regions[region]
        self._panels.append(
            PanelRow(region=region, pct_region=pct_region, log_scale=int(bool(log_scale)), first_block=self._raster_blocks,
                     z_min=np.nan if z_min is None else float(z_min), z_max=np.nan if z_max is None else float(z_max),
                     out_off=self._pixels, stat_region=stat_region, reserved=0,
                     zmin_slot=z_min.slot if isinstance(z_min, ZSlot) else -1,
                     zmax_slot=z_max.slot if isinstance(z_max, ZSlot) else -1)
        )
        self._raster_blocks += self.ctx.lib.csg_raster_blocks(r.ne, r.nt)
        self._pixels += (r.ne * r.nt + 3) & ~3  # every panel starts 16-byte aligned: 128-bit RGBA stores
        return len(self._panels) - 1

    def set_stat_region(self, panel: int, region: int):
        """Take a panel's reductions (safe_vmin, nanmin / nanmax) from ``region`` instead of its own region."""
        self._panels[panel] = self._panels[panel]._replace(stat_region=region)

    def panel_region(self, panel: int) -> int:
        """The region a panel draws."""
        return self._panels[panel].region

    def panel_offset(self, panel: int) -> int:
        """First pixel of a panel in the batch's RGBA / index buffers."""
        return self._panels[panel].out_off

    def panel_shape(self, panel: int) -> tuple[int, int]:
        r = self._regions[self._panels[panel].region]
        return r.ne, r.nt

    def upload_tables(self):
        """Region / panel / index tables -> device (call after the last add_*)."""
        regions = np.array(self._regions, dtype=REGION) if self._regions else np.zeros(0, REGION)
        self.d_regions = self.ctx.to_device(regions) if len(regions) else None
        pool = np.concatenate(self._pool) if self._pool else np.zeros(1, np.int32)
        self.d_pool = self.ctx.to_device(pool)
        self.d_stats = self.ctx.alloc(max(len(regions), 1) * REGION_STATS.itemsize)
        if self._windows:
            self.d_windows = self.ctx.to_device(np.array(self._windows, dtype=FLAG_WINDOW))
            self.d_window_any = self.ctx.alloc(len(self._windows))
        self.upload_panels()

    def upload_panels(self):
        """Panel table -> device.  Panels whose bounds do not depend on the per-step z slots come
        first, so they can be resolved and rasterised before the slot values are known."""
        self.d_panels = self.d_block_panel = None
        self._dev_order = np.zeros(0, np.int64)
        self._n_free = self._blocks_free = 0
        if not self._panels:
            return
        logical = np.array(self._panels, dtype=PANEL)
        free = (logical["zmin_slot"] < 0) & (logical["zmax_slot"] < 0)
        order = np.concatenate([np.flatnonzero(free), np.flatnonzero(~free)])
        dev = logical[order]
        blocks = np.array([self.ctx.lib.csg_raster_blocks(*self.panel_shape(p)) for p in order], dtype=np.int64)
        first = np.concatenate([[0], np.cumsum(blocks)[:-1]])
        dev["first_block"] = first
        # region-stat references stay valid (they index regions, not panels)
        self._dev_order = order
        self._n_free = int(free.sum())
        self._blocks_free = int(blocks[: self._n_free].sum())
        self.d_panels = self.ctx.to_device(dev)
        self.d_block_panel = self.ctx.to_device(np.repeat(np.arange(len(dev), dtype=np.int32), blocks))
        n = len(dev)
        if self.d_norms is None or self.d_norms.nbytes < n * PANEL_NORM.itemsize:
            self.d_norms = self.ctx.alloc(n * PANEL_NORM.itemsize)
        thr_bytes = self.ctx.lib.csg_threshold_bytes(n, self.code)
        if self.d_thr is None or self.d_thr.nbytes < thr_bytes:
            self.d_thr = self.ctx.alloc(thr_bytes)

    # ------------------------------------------------------------------ stages
    def run_stats(self):
        """K2a over every region."""
        if not self._regions:
            return
        self.ctx._check(
            self.ctx.lib.csg_region_stats_run(
                self.ctx.handle, self.d_sums.ptr, self.code, self.d_regions.ptr, len(self._regions), self.d_pool.ptr,
                self.d_stats.ptr,
            )
        )

    def force_exact_stats(self, on: bool = True):
        """Test knob (``csg_region_stats_force_exact``): route every percentile region of later
        :meth:`run_stats` calls on this batch's context through the exact radix-select fallback."""
        self.ctx._check(self.ctx.lib.csg_region_stats_force_exact(self.ctx.handle, int(bool(on))))

    def stats_fallbacks(self) -> int:
        """Regions of the last run_stats() that needed the exact radix-select fallback."""
        n = C.c_int(0)
        self.ctx._check(self.ctx.lib.csg_region_stats_fallbacks(self.ctx.handle, len(self._regions), C.byref(n)))
        return int(n.value)

    def stats(self) -> np.ndarray:
        if not self._regions:
            return np.zeros(0, REGION_STATS)
        return self.d_stats.download(REGION_STATS, len(self._regions))

    def _panel_range(self, part):
        """(first panel, count, first block, block count) in device order: part None = every panel,
        0 = panels free of z slots, 1 = panels that read z slots."""
        n = len(self._panels)
        if part is None:
            return 0, n, 0, self._raster_blocks
        if part == 0:
            return 0, self._n_free, 0, self._blocks_free
        return self._n_free, n - self._n_free, self._blocks_free, self._raster_blocks - self._blocks_free

    def prepare(self, part=None):
        """Resolve panel normalisations on the device (``part``: see :meth:`_panel_range`)."""
        if not self._panels:
            return
        p0, n, _, _ = self._panel_range(part)
        if n == 0:
            return
        if self._zvals and (self._zvals_dirty or self.d_zvals is None) and part != 0:
            vals = np.asarray(self._zvals, dtype=np.float64)
            if self.d_zvals is None or self.d_zvals.nbytes < vals.nbytes:
                self.d_zvals = self.ctx.alloc(max(vals.nbytes * 2, 256))
            self.d_zvals.upload(vals)
            self._zvals_dirty = False
        thr_one = self.ctx.lib.csg_threshold_bytes(1, self.code)
        self.ctx._check(
            self.ctx.lib.csg_panel_prepare(
                self.ctx.handle, self.d_panels.ptr + p0 * PANEL.itemsize, n, self.d_regions.ptr, self.d_stats.ptr,
                self.code, self.d_zvals.ptr if self.d_zvals is not None else None,
                self.d_norms.ptr + p0 * PANEL_NORM.itemsize, self.d_thr.ptr + p0 * thr_one,
            )
        )

    def norms(self) -> np.ndarray:
        """Resolved normalisation of every panel, indexed by panel id."""
        if not self._panels:
            return np.zeros(0, PANEL_NORM)
        return self.by_panel(self.d_norms.download(PANEL_NORM, len(self._panels)))

    def by_panel(self, dev: np.ndarray) -> np.ndarray:
        """Rows of a per-panel table in device order (see :meth:`upload_panels`), reordered by panel id."""
        out = np.empty_like(dev)
        out[self._dev_order] = dev
        return out

    def set_lut(self, lut259: np.ndarray):
        lut = np.ascontiguousarray(lut259, dtype=np.uint8)
        if lut.shape != (259, 4):
            raise ValueError("LUT must be (259, 4) uint8: 256 colours + under + over + bad")
        self.d_lut = self.ctx.to_device(lut)

    def rasterise(self, want_rgba: bool = True, want_index: bool = True, part=None):
        """K3 over the panels of ``part`` (see :meth:`_panel_range`)."""
        if not self._panels:
            return
        if want_rgba and self.d_lut is None:
            raise CsgError("set_lut() before rasterise(want_rgba=True)")
        if want_rgba and (self.d_rgba is None or self.d_rgba.nbytes < self._pixels * 4):
            self.d_rgba = self.ctx.alloc(max(self._pixels, 1) * 4)
        if want_index and (self.d_index is None or self.d_index.nbytes < self._pixels * 2):
            self.d_index = self.ctx.alloc(max(self._pixels, 1) * 2)
        _, n, b0, nb = self._panel_range(part)
        if n == 0 or nb == 0:
            return
        self.ctx._check(
            self.ctx.lib.csg_rasterise(
                self.ctx.handle, self.d_sums.ptr, self.code, self.d_regions.ptr, self.d_pool.ptr, self.d_panels.ptr,
                self.d_norms.ptr, self.d_thr.ptr, len(self._panels), nb, b0, self.d_block_panel.ptr,
                self.d_lut.ptr if self.d_lut is not None else None,
                self.d_rgba.ptr if want_rgba else None, self.d_index.ptr if want_index else None,
            )
        )

    def panel_index(self, panel: int) -> np.ndarray:
        ne, nt = self.panel_shape(panel)
        return self.d_index.download(np.uint16, ne * nt, self.panel_offset(panel) * 2).reshape(ne, nt)

    def panel_rgba(self, panel: int) -> np.ndarray:
        ne, nt = self.panel_shape(panel)
        return self.d_rgba.download(np.uint8, ne * nt * 4, self.panel_offset(panel) * 4).reshape(ne, nt, 4)

    def all_rgba(self) -> np.ndarray:
        return self.d_rgba.download(np.uint8, self._pixels * 4)

    def all_index(self) -> np.ndarray:
        return self.d_index.download(np.uint16, self._pixels)

    @property
    def n_regions(self) -> int:
        return len(self._regions)

    @property
    def n_panels(self) -> int:
        return len(self._panels)

    @property
    def n_windows(self) -> int:
        return len(self._windows)

    @property
    def n_pixels(self) -> int:
        return self._pixels


def collapse_host(cube: np.ndarray, pa_bits: np.ndarray | None = None, n_groups: int = 0, ctx: Context | None = None):
    """``csg_collapse_host``: the drop-in for ``COLLAPSE_FUNCTION(cube, axis=1)``.

    Returns ``(sums[(G+1), T, E], row_flags[T])``; the sums of an 8/16/32-bit integer cube are float64 (exact).
    """
    ctx = ctx or _lib.default_context()
    host, layout, (T, P, E) = classify_cube(np.asarray(cube))
    host = np.ascontiguousarray(host)
    code = np_cube_code(host.dtype)
    sums = np.zeros((n_groups + 1, T, E), dtype=compute_dtype(host.dtype))
    flags = np.zeros(T, dtype=np.uint8)
    bits = np.ascontiguousarray(pa_bits, dtype=np.uint8) if n_groups else None
    ctx._check(
        ctx.lib.csg_collapse_host(
            ctx.handle, host.ctypes.data, T, P, E, code, layout, bits.ctypes.data if bits is not None else None,
            n_groups, sums.ctypes.data, flags.ctypes.data,
        )
    )
    return sums, flags


def nansum(cube, axis: int = 1):
    """GPU ``np.nansum(cube, axis=1)`` with numpy's exact summation order (the
    reference's pluggable ``COLLAPSE_FUNCTION``, ``constants.py:12``).  An 8/16/32-bit integer cube gives
    numpy's int64 (signed) or uint64 (unsigned) sums, converted exactly from the float64 sums of K1."""
    cube = np.asarray(cube)
    if cube.ndim != 3:
        raise ValueError("nansum: expected a 3-D cube")
    if axis != 1:
        cube = np.moveaxis(cube, axis, 1)
    sums, _ = collapse_host(cube)
    if cube.dtype in _lib.INT_CUBE_CODES:
        return sums[0].astype(np.uint64 if cube.dtype.kind == "u" else np.int64)
    return sums[0]


def matrix_percentiles(matrix: np.ndarray, p_lo, p_hi, ctx: Context | None = None) -> tuple[float, float]:
    """``(np.nanpercentile(matrix, p_lo), np.nanpercentile(matrix, p_hi))`` of the flattened
    matrix, selected exactly on the GPU (K2a) in the matrix dtype's arithmetic."""
    ctx = ctx or _lib.default_context()
    m = np.asarray(matrix)
    if m.dtype not in (np.float32, np.float64):
        m = m.astype(np.float64)  # numpy computes integer input in float64
    flat = np.ascontiguousarray(m).reshape(1, -1)
    n = flat.shape[1]
    if n == 0:
        return float("nan"), float("nan")
    d_m = ctx.to_device(flat)
    # one energy row holding every cell
    reg = RegionRow(mat_off=0, ld=n, t0=0, nt=n, rows_off=-1, cols_off=0, ne=1, want_pct=WANT_PERCENTILES, reserved=0,
                    p_lo=float(p_lo), p_hi=float(p_hi))
    d_r = ctx.to_device(np.array([reg], dtype=REGION))
    d_pool = ctx.to_device(np.zeros(1, dtype=np.int32))
    d_out = ctx.alloc(REGION_STATS.itemsize)
    ctx._check(ctx.lib.csg_region_stats_run(ctx.handle, d_m.ptr, np_dtype_code(flat.dtype), d_r.ptr, 1, d_pool.ptr, d_out.ptr))
    st = d_out.download(REGION_STATS, 1)[0]
    return float(st["p_lo"]), float(st["p_hi"])
