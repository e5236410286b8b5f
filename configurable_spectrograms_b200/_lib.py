"""ctypes binding of ``libcsgpu.so`` (C ABI in ``include/csgpu.h``).

There is no CPU fallback: if the shared library is missing or no CUDA device is
usable, :class:`CsgError` is raised -- the product path never computes on the host.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# CSG_LIBRARY: another build of the same ABI (A/B experiments: a kernel variant compiled with a different -D)
LIB_PATH = os.environ.get("CSG_LIBRARY") or os.path.join(HERE, "libcsgpu.so")

ABI_VERSION = 26
F32, F64 = 0, 1
LAYOUT_TPE, LAYOUT_TEP = 0, 1
K1_GENERIC, K1_STREAM = 0, 1
MAX_GROUPS = 7
I_UNDER, I_OVER, I_BAD = 256, 257, 258
NORM_OK, NORM_VMIN_GT_VMAX, NORM_INVALID = 0, 1, 2


class CsgError(RuntimeError):
    """A libcsgpu call failed (message from ``csg_last_error``)."""


# numpy mirrors of the C structs (sizes asserted against the header comments)
FILE_DESC = np.dtype(
    [
        ("d_cube", "<u8"),
        ("sums_off", "<i8"),
        ("flags_off", "<i8"),
        ("T", "<i4"),
        ("P", "<i4"),
        ("E", "<i4"),
        ("bits_off", "<i4"),
        ("first_block", "<i4"),
        ("reserved", "<i4", (3,)),
    ],
    align=True,
)
REGION = np.dtype(
    [
        ("mat_off", "<i8"),
        ("ld", "<i4"),
        ("t0", "<i4"),
        ("nt", "<i4"),
        ("rows_off", "<i4"),
        ("cols_off", "<i4"),
        ("ne", "<i4"),
        ("want_pct", "<i4"),
        ("reserved", "<i4"),
        ("p_lo", "<f8"),
        ("p_hi", "<f8"),
    ],
    align=True,
)
REGION_STATS = np.dtype(
    [
        ("p_lo", "<f8"),
        ("p_hi", "<f8"),
        ("min_pos", "<f8"),
        ("fin_min", "<f8"),
        ("fin_max", "<f8"),
        ("n_valid", "<i8"),
        ("n_nan", "<i4"),
        ("n_neginf", "<i4"),
        ("n_posinf", "<i4"),
        ("n_pos", "<i4"),
    ],
    align=True,
)
PANEL = np.dtype(
    [
        ("region", "<i4"),
        ("pct_region", "<i4"),
        ("log_scale", "<i4"),
        ("first_block", "<i4"),
        ("z_min", "<f8"),
        ("z_max", "<f8"),
        ("out_off", "<i8"),
        ("stat_region", "<i4"),
        ("reserved", "<i4"),
        ("zmin_slot", "<i4"),
        ("zmax_slot", "<i4"),
    ],
    align=True,
)
PANEL_NORM = np.dtype(
    [
        ("vmin", "<f8"),
        ("vmax", "<f8"),
        ("fill_lo", "<f8"),
        ("fill_hi", "<f8"),
        ("t_vmin", "<f8"),
        ("t_range", "<f8"),
        ("status", "<i4"),
        ("degenerate", "<i4"),
        ("c0", "<f4"),
        ("c1", "<f4"),
    ],
    align=True,
)
POOL_ITEM = np.dtype(
    [("mat_off", "<i8"), ("T", "<i4"), ("E", "<i4"), ("inst", "<i4"), ("pos", "<i4")], align=True
)
POOL_QUERY = np.dtype(
    [("inst", "<i4"), ("pos", "<i4"), ("slot", "<i4"), ("bin", "<i4"), ("rank", "<i8"), ("row_total", "<i8")],
    align=True,
)
FLAG_WINDOW = np.dtype(
    [("flags_off", "<i8"), ("t0", "<i4"), ("nt", "<i4"), ("rows_off", "<i4"), ("bit", "<i4")], align=True
)
assert FLAG_WINDOW.itemsize == 24
PNG_TILE = np.dtype(
    [("rgba_off", "<i8"), ("ne", "<i4"), ("nt", "<i4"), ("x", "<i4"), ("y", "<i4"), ("w", "<i4"), ("h", "<i4"),
     ("vline_first", "<i4"), ("vline_count", "<i4"), ("flags", "<i4"), ("row_map", "<i4")], align=True
)
TILE_OVERLAY, TILE_TOP_ORIGIN, TILE_ROW_MAP = 1, 2, 4
PNG_ZERO_SEGMENT = np.dtype([("n_raw", "<i4"), ("len", "<i4"), ("bytes", "u1", (56,))], align=True)
assert PNG_ZERO_SEGMENT.itemsize == 64
PNG_FILE = np.dtype(
    [("path", "<u8"), ("row_first", "<i8"), ("seg_first", "<i8"), ("file_bytes", "<i8"), ("width", "<i4"), ("height", "<i4"),
     ("n_rows", "<i4"), ("segs_per_row", "<i4"), ("status", "<i4"), ("pad", "<i4")], align=True
)
assert PNG_FILE.itemsize == 56
PNG_VLINE = np.dtype([("col", "<i4"), ("half", "<i4"), ("rgba", "<u4"), ("pad", "<i4")], align=True)
PNG_CANVAS = np.dtype(
    [("W", "<i4"), ("H", "<i4"), ("tile_first", "<i4"), ("tile_count", "<i4"), ("background", "<u4"),
     ("seg_first", "<i4"), ("segs_per_row", "<i4"), ("row_first", "<i4")], align=True
)
PNG_TABLES = np.dtype(
    [("lit_code", "<u2", (256,)), ("lit_len", "u1", (256,)), ("len_code", "<u4", (65,)), ("dist_code", "<u4", (129,)),
     ("len_sym", "<u2", (65,)), ("len_len", "u1", (65,)), ("dist_len", "u1", (129,)), ("dist_sym", "u1", (129,)),
     ("eob_len", "u1"), ("eob_code", "<u2"), ("header_bits", "<i4"), ("header", "<u4", (40,))], align=True
)
assert PNG_TILE.itemsize == 48 and PNG_VLINE.itemsize == 16 and PNG_CANVAS.itemsize == 32
POOL_REQUEST = np.dtype([("inst", "<i4"), ("mode", "<i4"), ("p", "<f8")], align=True)
POOL_SEL = np.dtype(
    [("inst", "<i4"), ("pos", "<i4"), ("req", "<i4"), ("active", "<i4"), ("slot", "<i4", (2,)), ("rank", "<i8", (2,)),
     ("prefix", "<u8", (2,)), ("gamma", "<f8")],
    align=True,
)
assert POOL_REQUEST.itemsize == 16 and POOL_SEL.itemsize == 64
assert FILE_DESC.itemsize == 56 and REGION.itemsize == 56 and REGION_STATS.itemsize == 64
assert PANEL.itemsize == 56 and PANEL_NORM.itemsize == 64 and POOL_ITEM.itemsize == 24 and POOL_QUERY.itemsize == 32

_vp, _i, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t

#: every symbol include/csgpu.h declares: (restype, argtypes)
SIGNATURES = {
    "csg_abi_version": (_i, []),
    "csg_device_count": (_i, []),
    "csg_create": (_vp, [_i, _vp]),
    "csg_create_side": (_vp, [_i, _i]),
    "csg_create_with_priority": (_vp, [_i, _i]),
    "csg_wait_for": (_i, [_vp, _vp]),
    "csg_destroy": (None, [_vp]),
    "csg_last_error": (C.c_char_p, [_vp]),
    "csg_sync": (_i, [_vp]),
    "csg_stream_handle": (_vp, [_vp]),
    "csg_device_info": (_i, [_vp, C.c_char_p, _i, C.POINTER(_i), C.POINTER(_sz)]),
    "csg_dev_alloc": (_i, [_vp, _sz, C.POINTER(_vp)]),
    "csg_dev_free": (_i, [_vp, _vp]),
    "csg_dev_trim": (_i, [_vp, C.POINTER(_sz)]),
    "csg_dev_cached": (_i, [_vp, C.POINTER(_sz), C.POINTER(_sz)]),
    "csg_host_alloc": (_i, [_vp, _sz, C.POINTER(_vp)]),
    "csg_host_free": (_i, [_vp, _vp]),
    "csg_host_register": (_i, [_vp, _vp, _sz]),
    "csg_host_unregister": (_i, [_vp, _vp]),
    "csg_h2d": (_i, [_vp, _vp, _vp, _sz]),
    "csg_d2h": (_i, [_vp, _vp, _vp, _sz]),
    "csg_d2d": (_i, [_vp, _vp, _vp, _sz]),
    "csg_memset": (_i, [_vp, _vp, _i, _sz]),
    "csg_d2h_side": (_i, [_vp, _vp, _vp, _sz]),
    "csg_side_join": (_i, [_vp]),
    "csg_side_sync": (_i, [_vp]),
    "csg_timer_start": (_i, [_vp, _i]),
    "csg_timer_stop": (_i, [_vp, _i]),
    "csg_timer_ms": (_i, [_vp, _i, C.POINTER(C.c_float)]),
    "csg_launch_count": (_i64, [_vp]),
    "csg_event_record": (_i, [_vp, _i]),
    "csg_event_sync": (_i, [_vp, _i]),
    "csg_collapse_kernel": (_i, [C.c_int32, C.c_int32, C.c_int32, _i, _i, _vp]),
    "csg_collapse_kernel_for": (_i, [C.c_int32, C.c_int32, C.c_int32, _i, _i, _vp, _i]),
    "csg_pitch_runs": (_i, [_vp, _i, _i, _vp, _vp]),
    "csg_collapse_blocks": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, _i, _i, _i]),
    "csg_sums_elems": (_i64, [C.c_int32, C.c_int32, _i]),
    "csg_collapse": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "csg_window_any": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "csg_collapse_host": (_i, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, _i, _i, _vp, _i, _vp, _vp]),
    "csg_region_stats_run": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "csg_region_stats_fallbacks": (_i, [_vp, _i, C.POINTER(_i)]),
    "csg_region_stats_force_exact": (_i, [_vp, _i]),
    "csg_raster_blocks": (C.c_int32, [C.c_int32, C.c_int32]),
    "csg_threshold_bytes": (_sz, [_i, _i]),
    "csg_panel_prepare": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "csg_rasterise": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "csg_rasterise_blocks_per_sm": (_i, [_vp, _i]),
    "csg_pool_hist_first": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "csg_pool_scan_cols": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp]),
    "csg_pool_slot_payload_bytes": (_sz, [_i, _i]),
    "csg_pool_energy_candidates": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "csg_pool_pack_results": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp, _vp, _i]),
    "csg_pool_reduce_max": (_i, [_vp, _vp, _i, _i, _vp]),
    "csg_png_fixed_tables": (_i, [_vp]),
    "csg_png_set_tables": (_i, [_vp, _vp]),
    "csg_png_count": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _i, _vp, _vp, _i, _vp]),
    "csg_png_max_segment_tiles": (C.c_int32, []),
    "csg_png_slot_bytes": (C.c_int32, []),
    "csg_png_segments": (C.c_int32, [C.c_int32, C.c_int32]),
    "csg_png_encode": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "csg_png_compact": (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    "csg_png_write_files": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i]),
    "csg_peer_create": (_i, [_vp, _i, _i, _sz, _vp, _vp]),
    "csg_peer_mailbox": (_vp, [_vp]),
    "csg_peer_connect_ipc": (_i, [_vp, _vp, _vp]),
    "csg_peer_connect_ptrs": (_i, [_vp, _vp, _vp]),
    "csg_peer_allgather": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "csg_peer_error_word": (_vp, [_vp]),
    "csg_peer_clear_error": (_i, [_vp, _vp]),
    "csg_peer_wait_stats": (_i, [_vp, _vp, _i, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "csg_peer_trace": (_i, [_vp, _vp, _i, _vp, C.POINTER(_i)]),
    "csg_peer_disconnect": (_i, [_vp, _vp]),
    "csg_peer_destroy": (_i, [_vp, _vp]),
    "csg_pool_hist_refine": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp]),
    "csg_pool_scan": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _vp, _vp]),
    "csg_pool_locate": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i]),
    "csg_pool_row_totals": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "csg_pool_sel_init": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "csg_pool_sel_locate": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp]),
    "csg_pool_sel_bounds": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "csg_pool_sel_slots": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _i, _vp, _vp]),
    "csg_pool_sel_assign": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _sz, _i, _i, _i, _vp, _vp]),
    "csg_pool_sel_finish": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp]),
    "csg_pool_base": (_i, [_vp, _vp, _sz, _i, _i, _i, _sz, _vp, _vp]),
}

SIGNATURES.update({
    "csg_cdf_open": (_i, [C.c_char_p, C.POINTER(_vp)]),
    "csg_cdf_close": (None, [_vp]),
    "csg_cdf_var_count": (_i, [_vp]),
    "csg_cdf_var_info": (_i, [_vp, C.c_char_p, _i, _vp]),
    "csg_cdf_read": (_i, [_vp, C.c_char_p, _i64, _i64, _vp, _sz]),
    "csg_cdf_last_error": (C.c_char_p, []),
})
CDF_VAR = np.dtype(
    [("name", "S260"), ("data_type", "<i4"), ("elem_bytes", "<i4"), ("n_dims", "<i4"), ("dims", "<i4", (8,)),
     ("rec_vary", "<i4"), ("compressed", "<i4"), ("row_major", "<i4"), ("n_records", "<i8"), ("values_per_record", "<i8")],
    align=True,
)
assert CDF_VAR.itemsize == 336

_lib = None


def load_library(path: str | None = None):
    """dlopen ``libcsgpu.so`` and bind every declared symbol (no compute, no GPU needed)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise CsgError(
            f"{p} not found: build it with `python -m configurable_spectrograms_b200.build` "
            "(there is no CPU fallback for this path)"
        )
    lib = C.CDLL(p, mode=C.RTLD_LOCAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.csg_abi_version() != ABI_VERSION:
        raise CsgError(f"libcsgpu ABI version {lib.csg_abi_version()} != {ABI_VERSION}: rebuild the library")
    if path is None:
        _lib = lib
    return lib


def np_dtype_code(dtype) -> int:
    dt = np.dtype(dtype)
    if dt == np.float32:
        return F32
    if dt == np.float64:
        return F64
    raise TypeError(f"unsupported cube dtype {dt}: libcsgpu computes in float32 or float64")


class DevBuf:
    """A device allocation owned by a :class:`Context`."""

    __slots__ = ("ctx", "ptr", "nbytes")

    def __init__(self, ctx: "Context", nbytes: int):
        self.ctx = ctx
        self.nbytes = int(nbytes)
        out = _vp()
        ctx._check(ctx.lib.csg_dev_alloc(ctx.handle, max(self.nbytes, 1), C.byref(out)))
        self.ptr = out.value

    def free(self):
        if self.ptr and self.ctx.handle:
            self.ctx.lib.csg_dev_free(self.ctx.handle, self.ptr)
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def upload(self, arr: np.ndarray, offset: int = 0, keep: bool = True):
        """Asynchronous H2D on the context stream.  ``keep=False``: the caller owns the source's lifetime
        (pinned staging slots; pageable sources are staged by the driver before the call returns)."""
        arr = np.ascontiguousarray(arr)
        assert offset + arr.nbytes <= self.nbytes, (offset, arr.nbytes, self.nbytes)
        self.ctx._check(self.ctx.lib.csg_h2d(self.ctx.handle, self.ptr + offset, arr.ctypes.data, arr.nbytes))
        if keep:
            self.ctx._keep(arr)

    def download(self, dtype, count: int, offset: int = 0, sync: bool = True) -> np.ndarray:
        out = np.empty(count, dtype=dtype)
        assert offset + out.nbytes <= self.nbytes, (offset, out.nbytes, self.nbytes)
        self.ctx._check(self.ctx.lib.csg_d2h(self.ctx.handle, out.ctypes.data, self.ptr + offset, out.nbytes))
        if sync:
            self.ctx.sync()
        return out

    def zero(self):
        self.ctx._check(self.ctx.lib.csg_memset(self.ctx.handle, self.ptr, 0, self.nbytes))


class PinnedBuf:
    """Page-locked host memory exposed as a numpy byte array."""

    def __init__(self, ctx: "Context", nbytes: int):
        self.ctx = ctx
        self.nbytes = int(nbytes)
        out = _vp()
        ctx._check(ctx.lib.csg_host_alloc(ctx.handle, max(self.nbytes, 1), C.byref(out)))
        self.ptr = out.value
        self.array = np.ctypeslib.as_array((C.c_uint8 * max(self.nbytes, 1)).from_address(self.ptr))

    def view(self, dtype, count: int, offset: int = 0) -> np.ndarray:
        dt = np.dtype(dtype)
        return self.array[offset : offset + count * dt.itemsize].view(dt)

    def free(self):
        if self.ptr and self.ctx.handle:
            self.array = None
            self.ctx.lib.csg_host_free(self.ctx.handle, self.ptr)
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedRing:
    """Pinned staging slots for streaming ingest (north_star: "cdflib arrays staged into pinned buffers").

    Loader threads decode cubes straight into the current slot (:meth:`alloc` is a thread-safe bump
    allocator handing out numpy views of page-locked memory), the main thread enqueues the asynchronous
    H2D copies + K1 of that chunk and calls :meth:`release`, which records an event on the context
    stream; :meth:`acquire` of the same slot, ``n_slots`` chunks later, waits for that event only -- so
    decoding chunk k+1 overlaps the copies of chunk k and nothing is ever overwritten while in flight.
    """

    FIRST_EVENT = 8  # csg_event slots 8 .. 8 + n_slots - 1 (30 / 31 belong to the pool selector)

    def __init__(self, ctx: "Context", n_slots: int = 3, slot_bytes: int = 1 << 30):
        import threading

        if not 1 <= n_slots <= 16:
            raise ValueError("n_slots must be 1..16")
        self.ctx = ctx
        self.slot_bytes = int(slot_bytes)
        self.limit = self.slot_bytes  # bytes of a slot handed out per chunk (shared_ring may lower it for a call)
        self.slots = [ctx.pinned(self.slot_bytes) for _ in range(n_slots)]
        self._used = [0] * n_slots
        self._in_flight = [False] * n_slots
        self._next = 0
        self._lock = threading.Lock()
        self.overflow_bytes = 0  # cubes that did not fit a slot and went through pageable memory

    def acquire(self) -> int:
        """The next slot, empty and safe to write (blocks until its previous copies have finished)."""
        k = self._next
        self._next = (k + 1) % len(self.slots)
        if self._in_flight[k]:
            self.ctx.event_sync(self.FIRST_EVENT + k)
            self._in_flight[k] = False
        self._used[k] = 0
        return k

    def alloc(self, slot: int, shape, dtype) -> np.ndarray:
        """A C-contiguous array of ``shape`` inside the slot (256-byte aligned); pageable memory when the
        slot is full -- slower to upload, never wrong."""
        dt = np.dtype(dtype)
        n = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
        with self._lock:
            off = (self._used[slot] + 255) & ~255
            if off + n > self.limit:
                self.overflow_bytes += n
                return np.empty(shape, dtype=dt)
            self._used[slot] = off + n
        return self.slots[slot].array[off : off + n].view(dt).reshape(shape)

    def release(self, slot: int):
        """Call after the slot's copies have been enqueued on the context stream."""
        self.ctx.event_record(self.FIRST_EVENT + slot)
        self._in_flight[slot] = True

    def drain(self):
        """Wait until no slot is in flight (the ring itself stays allocated for the next call)."""
        for k, busy in enumerate(self._in_flight):
            if busy:
                self.ctx.event_sync(self.FIRST_EVENT + k)
                self._in_flight[k] = False

    def close(self):
        self.drain()
        for s in self.slots:
            s.free()
        self.slots = []


def shared_ring(ctx: "Context", n_slots: int = 3, slot_bytes: int = 1 << 30) -> PinnedRing:
    """The context's staging ring, allocated on first use and kept: page-locking memory costs about a
    quarter of a second per GB, far more than a streaming call spends anywhere else.  A call that asks for
    larger slots replaces it."""
    ring = ctx.__dict__.get("_ring")
    if ring is not None and (ring.slot_bytes < slot_bytes or len(ring.slots) < n_slots):
        ring.close()
        ring = None
    if ring is None:
        ring = ctx.__dict__["_ring"] = PinnedRing(ctx, n_slots, slot_bytes)
    ring.drain()
    ring.overflow_bytes = 0
    ring._next = 0
    ring.limit = min(int(slot_bytes), ring.slot_bytes)
    return ring


class Context:
    """One GPU context (``csg_ctx``); all work runs on its stream."""

    def __init__(self, device: int = 0, stream: int | None = None, side: bool = False, priority: int | None = None):
        self.lib = load_library()
        self.handle = None
        if self.lib.csg_device_count() <= 0:
            raise CsgError("no CUDA device available: libcsgpu has no CPU fallback")
        # stream: a cudaStream_t handle (e.g. torch.cuda.Stream().cuda_stream); None/0 = own stream;
        # side: a companion context with its own highest-priority stream (see side_context())
        # priority: own stream, that many steps more urgent than the least urgent level (0 = default)
        if side:
            h = self.lib.csg_create_side(int(device), 1)
        elif priority is not None and not stream:
            h = self.lib.csg_create_with_priority(int(device), int(priority))
        else:
            h = self.lib.csg_create(int(device), _vp(stream) if stream else None)
        if not h:
            raise CsgError(self.lib.csg_last_error(None).decode())
        self.handle = h
        self.device = int(device)
        self._alive: list = []

    def side_context(self) -> "Context":
        """The companion context of this one (created on first use): same device, its own
        highest-priority stream -- for work that should overlap this context's kernels."""
        side = self.__dict__.get("_side")
        if side is None:
            side = self._side = Context(self.device, side=True)
        return side

    def background_context(self) -> "Context":
        """A companion context on the LEAST urgent stream: long kernels that should yield to everything else
        (the K4 encoder beside the next chunk's K2a / K3)."""
        background = self.__dict__.get("_background")
        if background is None:
            background = self._background = Context(self.device, priority=0)
        return background

    def wait_for(self, other: "Context"):
        """Everything enqueued on ``other`` so far happens before what this context enqueues next."""
        self._check(self.lib.csg_wait_for(self.handle, other.handle))

    # -- helpers
    def _check(self, status: int):
        if status != 0:
            raise CsgError(self.lib.csg_last_error(self.handle).decode())

    def _keep(self, obj):
        """Hold a host array until the next sync (async H2D source).  Pageable sources are staged
        before cudaMemcpyAsync returns, so the list only has to bridge the call itself."""
        self._alive.append(obj)
        if len(self._alive) > 1024:
            del self._alive[:512]

    def sync(self):
        self._check(self.lib.csg_sync(self.handle))
        self._alive.clear()

    @property
    def stream_handle(self) -> int:
        """The cudaStream_t (as an integer) all of this context's work is enqueued on."""
        return int(self.lib.csg_stream_handle(self.handle) or 0)

    def close(self):
        if self.handle:
            self.lib.csg_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def alloc(self, nbytes: int) -> DevBuf:
        return DevBuf(self, nbytes)

    def pinned(self, nbytes: int) -> PinnedBuf:
        return PinnedBuf(self, nbytes)

    def cached(self) -> tuple[int, int]:
        """(bytes parked in the device block cache, bytes handed out) on this context's device."""
        idle, live = _sz(), _sz()
        self._check(self.lib.csg_dev_cached(self.handle, C.byref(idle), C.byref(live)))
        return int(idle.value), int(live.value)

    def trim(self) -> int:
        """Return every parked device block to the driver; the bytes released."""
        n = _sz()
        self._check(self.lib.csg_dev_trim(self.handle, C.byref(n)))
        return int(n.value)

    def to_device(self, arr: np.ndarray) -> DevBuf:
        arr = np.ascontiguousarray(arr)
        buf = DevBuf(self, arr.nbytes)
        buf.upload(arr)
        return buf

    def device_info(self):
        name = C.create_string_buffer(128)
        sm, mem = _i(), _sz()
        self._check(self.lib.csg_device_info(self.handle, name, 128, C.byref(sm), C.byref(mem)))
        return name.value.decode(), sm.value, mem.value

    def launch_count(self) -> int:
        """Kernels launched by this context and by its side context (if it has one)."""
        n = int(self.lib.csg_launch_count(self.handle))
        side = self.__dict__.get("_side")
        if side is not None:
            n += side.launch_count()
        return n

    def d2h_side(self, host_ptr: int, dev_ptr: int, nbytes: int):
        """Read a result back on the copy-out stream (overlaps later work on the main stream)."""
        self._check(self.lib.csg_d2h_side(self.handle, host_ptr, dev_ptr, nbytes))

    def side_join(self):
        self._check(self.lib.csg_side_join(self.handle))

    def side_sync(self):
        self._check(self.lib.csg_side_sync(self.handle))

    def event_record(self, slot: int):
        self._check(self.lib.csg_event_record(self.handle, slot))

    def event_sync(self, slot: int):
        self._check(self.lib.csg_event_sync(self.handle, slot))

    def timer_start(self, slot: int):
        self._check(self.lib.csg_timer_start(self.handle, slot))

    def timer_stop(self, slot: int):
        self._check(self.lib.csg_timer_stop(self.handle, slot))

    def timer_ms(self, slot: int) -> float:
        ms = C.c_float()
        self._check(self.lib.csg_timer_ms(self.handle, slot, C.byref(ms)))
        return float(ms.value)


_default_ctx: dict[int, Context] = {}


def default_context(device: int = 0) -> Context:
    """Process-wide context per device (created on first use)."""
    ctx = _default_ctx.get(device)
    if ctx is None or ctx.handle is None:
        ctx = Context(device, priority=1)  # one step above background work (see Context.background_context)
        _default_ctx[device] = ctx
    return ctx
