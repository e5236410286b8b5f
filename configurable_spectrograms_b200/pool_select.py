"""Exact order statistics of every prefix pool of an instrument's file sequence.

The reference recomputes ``np.nanpercentile(np.concatenate(blocks so far), p)`` after
every (orbit, instrument) step and keeps a running maximum
(``fast/extrema.py:280-300``).  Here the pooled samples stay in HBM as the collapsed
total matrices; per-file radix-digit histograms are scanned along the file sequence so
one row describes one prefix pool, and the two neighbours of every prefix's percentile
are located digit by digit (``csrc/pool.cu``).  Prefixes that provably cannot hold the
running maximum are dropped between digits, so the refinement passes follow only a
handful of buckets.

Multi-GPU: ranks hold contiguous blocks of the ascending-orbit sequence.  Per digit one
all-gather of each rank's bucket totals gives every rank the counts held by lower
ranks (added on the fly by the locate kernels); one all-gather of [bounds | surviving
(instrument, prefix) lists] keeps the slot tables identical everywhere; one last all-gather
carries the results.  The all-gather itself is an ``exchange`` object (``comm.make_exchange``):
peer mailboxes written over NVLink (``csrc/peer.cu``) or NCCL.

Two drivers over the same kernels: :class:`DevicePoolSelector` (the whole digit loop enqueued on
a stream, no host round trip -- the batch path) and :func:`prefix_percentiles` (host-driven,
any number of candidate buckets -- the fallback when the device slot table overflows, and the
form the gloo tests exercise with a numpy kernel stand-in).
"""

from __future__ import annotations

from collections import namedtuple

import numpy as np

from . import _lib
from ._lib import POOL_QUERY, POOL_REQUEST, POOL_SEL

FIRST_BITS = 11
NEXT_BITS = 10
MAX_SLOTS = 64
_U64MAX = np.iinfo(np.uint64).max


def key_bits(dtype) -> int:
    return 31 if np.dtype(dtype) == np.float32 else 63


def digit_plan(dtype) -> list[tuple[int, int]]:
    """[(shift, bits)] from the most significant digit down to shift 0."""
    total = key_bits(dtype)
    plan = [(total - FIRST_BITS, FIRST_BITS)]
    shift = total - FIRST_BITS
    while shift > 0:
        b = min(NEXT_BITS, shift)
        shift -= b
        plan.append((shift, b))
    return plan


def bits_to_value(bits: np.ndarray, dtype) -> np.ndarray:
    dt = np.dtype(dtype)
    if dt == np.float32:
        return bits.astype(np.uint32).view(np.float32)
    return bits.astype(np.uint64).view(np.float64)


def percentile_ranks(n: np.ndarray, p, dtype):
    """Vectorised numpy ``_get_indexes`` / ``_get_gamma`` in dtype D (n >= 1)."""
    D = np.dtype(dtype).type
    q = D(p) / D(100)
    nm1 = (n - 1).astype(dtype)
    v = nm1 * q
    above = v >= nm1
    below = v < 0
    fl = np.floor(v)
    lo = fl.astype(np.int64)
    hi = lo + 1
    gamma = (v - fl).astype(dtype)
    lo = np.where(above, n - 1, np.where(below, 0, lo))
    hi = np.where(above, n - 1, np.where(below, 0, hi))
    hi = np.minimum(hi, n - 1)
    lo = np.minimum(lo, n - 1)
    gamma = np.where(above | below, D(0), gamma).astype(dtype)
    return lo, hi, gamma


def lerp_vec(a, b, g, dtype):
    """numpy ``_lerp`` rounded after every operation in D (vectorised)."""
    dt = np.dtype(dtype)
    with np.errstate(invalid="ignore", over="ignore"):
        a, b, g = a.astype(dt), b.astype(dt), g.astype(dt)
        d = (b - a).astype(dt)
        r = (a + (d * g).astype(dt)).astype(dt)
        alt = (b - (d * (dt.type(1) - g).astype(dt)).astype(dt)).astype(dt)
    return np.where(g >= 0.5, alt, r)


class _Grow:
    """Grow-only device / pinned scratch so a steady-state step allocates nothing."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.dev: dict[str, _lib.DevBuf] = {}
        self.pin: dict[str, _lib.PinnedBuf] = {}

    def device(self, name: str, nbytes: int) -> _lib.DevBuf:
        buf = self.dev.get(name)
        if buf is None or buf.nbytes < nbytes:
            buf = self.dev[name] = self.ctx.alloc(max(int(nbytes * 1.25), 256))
        return buf

    def pinned(self, name: str, nbytes: int) -> _lib.PinnedBuf:
        buf = self.pin.get(name)
        if buf is None or buf.nbytes < nbytes:
            buf = self.pin[name] = self.ctx.pinned(max(int(nbytes * 1.25), 256))
        return buf

    def put(self, name: str, arr: np.ndarray) -> _lib.DevBuf:
        """Upload a small array through pinned staging into the device buffer ``name`` (on the stream)."""
        arr = np.ascontiguousarray(arr)
        pin = self.pinned(name, arr.nbytes)
        pin.array[: arr.nbytes] = arr.view(np.uint8).reshape(-1)
        dev = self.device(name, arr.nbytes)
        self.ctx._check(self.ctx.lib.csg_h2d(self.ctx.handle, dev.ptr, pin.ptr, arr.nbytes))
        return dev


class GpuPoolBackend:
    """The four pool kernels over a :class:`engine.Batch`'s sums buffer (persistent scratch)."""

    def __init__(self, batch):
        self.batch = batch
        self.ctx = batch.ctx
        self.mem = _Grow(batch.ctx)
        self._items_key = None
        self.n_items = 0

    def _get(self, name: str, dev: _lib.DevBuf, dtype, count: int, sync=True) -> np.ndarray:
        nbytes = np.dtype(dtype).itemsize * count
        pin = self.mem.pinned("get_" + name, nbytes)
        self.ctx._check(self.ctx.lib.csg_d2h(self.ctx.handle, pin.ptr, dev.ptr, nbytes))
        if sync:
            self.ctx.sync()
        return pin.view(dtype, count)

    def set_items(self, items: np.ndarray, n_inst: int, max_pos: int, inst_len: np.ndarray, max_E: int):
        key = (items.tobytes(), n_inst, max_pos, inst_len.tobytes(), max_E)
        self.items = items
        self.n_items = len(items)
        self.n_inst, self.max_pos, self.max_E = n_inst, max(max_pos, 1), max(max_E, 1)
        if key != self._items_key:
            self.d_items = self.mem.put("items", items) if len(items) else None
            self.d_inst_len = self.mem.put("inst_len", np.ascontiguousarray(inst_len, dtype=np.int32))
            self._items_key = key

    def hist_first(self, bits: int):
        nb = 1 << bits
        self.n_slots, self.bits = 1, bits
        nbytes = self.n_inst * self.max_pos * nb * 4
        self.d_hist = self.mem.device("hist0", nbytes)
        self.ctx._check(self.ctx.lib.csg_memset(self.ctx.handle, self.d_hist.ptr, 0, nbytes))
        d_counts = self.mem.device("counts", max(self.n_items, 1) * self.max_E * 4)
        d_npos = self.mem.device("npos", max(self.n_items, 1) * 4)
        if self.n_items:
            self.ctx._check(
                self.ctx.lib.csg_pool_hist_first(
                    self.ctx.handle, self.batch.d_sums.ptr, self.batch.code, self.d_items.ptr, self.n_items,
                    self.max_pos, bits, self.max_E, self.d_hist.ptr, d_counts.ptr, d_npos.ptr, None,
                )
            )
        counts = self._get("counts", d_counts, np.int32, self.n_items * self.max_E, sync=False)
        npos = self._get("npos", d_npos, np.int32, self.n_items)
        return counts.reshape(self.n_items, self.max_E).copy(), npos.copy()

    def hist_refine(self, slot_prefix: np.ndarray, prefix_shift: int, shift: int, bits: int):
        n_slots = slot_prefix.shape[1]
        nb = 1 << bits
        self.n_slots, self.bits = n_slots, bits
        nbytes = self.n_inst * self.max_pos * n_slots * nb * 4
        self.d_hist = self.mem.device("hist1", nbytes)
        self.ctx._check(self.ctx.lib.csg_memset(self.ctx.handle, self.d_hist.ptr, 0, nbytes))
        d_pref = self.mem.put("pref", np.ascontiguousarray(slot_prefix, dtype=np.uint64))
        if self.n_items:
            self.ctx._check(
                self.ctx.lib.csg_pool_hist_refine(
                    self.ctx.handle, self.batch.d_sums.ptr, self.batch.code, self.d_items.ptr, self.n_items,
                    self.max_pos, n_slots, d_pref.ptr, prefix_shift, shift, bits, self.d_hist.ptr,
                )
            )

    def scan(self, want_totals: bool):
        """Inclusive scan along the file sequence; returns this rank's bucket totals when asked."""
        nb = 1 << self.bits
        n = self.n_inst * self.n_slots * nb
        d_tot = self.mem.device("totals", n * 4) if want_totals else None
        self.ctx._check(
            self.ctx.lib.csg_pool_scan(
                self.ctx.handle, self.d_hist.ptr, self.n_inst, self.max_pos, self.d_inst_len.ptr, self.n_slots,
                self.bits, None, d_tot.ptr if d_tot is not None else None,
            )
        )
        if want_totals:
            return self._get("totals", d_tot, np.uint32, n).reshape(self.n_inst, self.n_slots, nb).copy()
        return None

    def locate(self, queries: np.ndarray, base: np.ndarray | None) -> np.ndarray:
        if len(queries) == 0:
            return queries
        d_q = self.mem.put("queries", queries)
        d_base = self.mem.put("base", np.ascontiguousarray(base, dtype=np.uint32)) if base is not None else None
        self.ctx._check(
            self.ctx.lib.csg_pool_locate(
                self.ctx.handle, self.d_hist.ptr, self.max_pos, self.n_slots, self.bits,
                d_base.ptr if d_base is not None else None, d_q.ptr, len(queries),
            )
        )
        return self._get("queries", d_q, POOL_QUERY, len(queries)).copy()


class DevicePoolSelector:
    """The whole digit loop enqueued on the context's stream: no host round trip per digit.

    ``enqueue`` launches histograms, scans, the selection-table kernels of ``csrc/poolsel.cu`` and
    (multi-rank) the exchanges on device buffers, then an asynchronous read-back of the
    few results; ``result`` waits for that read-back only, so kernels enqueued afterwards (K2a)
    overlap the host bookkeeping.  When more than ``N_SLOTS`` distinct key prefixes survive a
    digit the device flags it and the caller falls back to the host-driven ``prefix_percentiles``.
    """

    N_SLOTS = 16
    EVENT_SLOT = 31

    def __init__(self, batch, ctx=None):
        """``ctx``: the context whose stream carries the selection (default: the batch's own; the batch
        step passes the batch context's side context so the digit loop overlaps K2a / K3)."""
        self.batch = batch
        self.ctx = ctx if ctx is not None else batch.ctx
        self.mem = _Grow(self.ctx)
        self._static_key = None
        self._pending = None

    def enqueue(self, dtype, items: np.ndarray, n_inst: int, inst_len: np.ndarray, max_E: int, requests: list[dict],
                comm=None, count_rows: int | None = None, exchange=None, ydev: dict | None = None, dry: bool = False):
        """``count_rows`` (multi-rank): rows of the per-file count table every rank contributes to the
        gather (the largest item count over the ranks); ``result_counts`` then returns every
        rank's rows, rank after rank.

        ``exchange``: the all-gather the ranks meet through (``comm.make_exchange``; built from
        ``comm`` when omitted).  ``ydev``: per-instrument energy tables for the on-device y
        candidates -- ``{"order": int32[n_inst][max_E], "keys": float64[n_inst][max_E],
        "n_keys": int32[n_inst], "limit": int32[n_inst]}`` -- in which case the per-file counts
        are neither gathered nor read back (``result_counts`` is not available)."""
        from .comm import NcclExchange, make_exchange

        comm = comm or SingleRank()
        if exchange is None:
            exchange = self.__dict__.get("_exchange")
            if exchange is None or exchange.size != comm.size:
                exchange = self._exchange = make_exchange(comm, self.ctx)
        self._slot_bytes_needed = self._payload_bytes(np.dtype(dtype), n_inst, max_E, len(items), count_rows, len(requests),
                                                      exchange.size, ydev is not None)
        try:
            exchange.ensure(self._slot_bytes_needed)
        except RuntimeError:
            if exchange.kind != "peer" or not hasattr(comm, "allgather_dev"):
                raise
            # no CUDA IPC here (every rank sees the same handle table, so every rank lands here)
            exchange = self._exchange = NcclExchange(comm, self.ctx)
            exchange.ensure(self._slot_bytes_needed)
        if exchange.kind == "nccl":
            # NCCL is ordered against THIS context's stream: one stream switch for the whole digit loop
            with comm.stream_scope(self.ctx.stream_handle):
                return self._enqueue(dtype, items, n_inst, inst_len, max_E, requests, exchange, count_rows, ydev, dry)
        return self._enqueue(dtype, items, n_inst, inst_len, max_E, requests, exchange, count_rows, ydev, dry)

    def reserve(self, *args, **kwargs):
        """Same arguments as :meth:`enqueue`: allocate every scratch buffer, upload the static
        tables, size the exchange mailboxes -- and launch nothing.  Device allocations order
        kernels of different streams behind each other, so ranks that share ONE process (the
        single-GPU tests) must all reserve before any of them enqueues; one process per GPU
        never needs this."""
        return self.enqueue(*args, dry=True, **kwargs)

    def _payload_bytes(self, D, n_inst, max_E, n_items, count_rows, n_req, R, device_y):
        S = self.N_SLOTS
        bits0 = digit_plan(D)[0][1]
        rows = _count_rows(n_items, R, count_rows)
        sizes = [
            _al(n_inst * ((1 << bits0) + max(int(max_E), 1)) * 4, 16),
            n_inst * S * 1024 * 4,
            int(self.ctx.lib.csg_pool_slot_payload_bytes(n_inst, S)),
            _al((n_req + n_inst + 5) * 8, 16),
        ]
        if not device_y:
            sizes.append(_al(rows * max(int(max_E), 1) * 4, 16))
        return max(sizes)

    def _enqueue(self, dtype, items, n_inst, inst_len, max_E, requests, ex, count_rows, ydev, dry=False):
        """``dry``: allocate / upload every buffer the step needs and launch nothing (see ``reserve``)."""
        ctx, lib, mem = self.ctx, self.ctx.lib, self.mem
        h = ctx.handle

        def run(fn, *args):
            if not dry:
                ctx._check(fn(*args))

        def gather(src_ptr, nbytes):
            return src_ptr if dry else ex.allgather(src_ptr, nbytes)

        def record(slot):
            if not dry:
                ctx.event_record(slot)

        D = np.dtype(dtype)
        code = _lib.np_dtype_code(D)
        plan = digit_plan(D)
        R, S = ex.size, self.N_SLOTS
        n_items, n_req = len(items), len(requests)
        max_pos = max(int(inst_len.max()) if len(inst_len) else 0, 1)
        max_E = max(int(max_E), 1)
        device_y = ydev is not None
        # ---- static tables (re-uploaded only when they change)
        key = (items.tobytes(), n_inst, inst_len.tobytes(), max_E, repr(requests), D.str,
               None if ydev is None else tuple(np.ascontiguousarray(ydev[k]).tobytes() for k in ("order", "keys", "n_keys", "limit")))
        if key != self._static_key:
            reqs = np.zeros(max(n_req, 1), dtype=POOL_REQUEST)
            for r, rq in enumerate(requests):
                reqs[r] = (rq["inst"], 0 if rq["mode"] == "running_max" else 1, float(rq["p"]))
            self.d_items = self.mem.put("items", items) if n_items else None
            self.d_inst_len = self.mem.put("inst_len", np.ascontiguousarray(inst_len, dtype=np.int32))
            self.d_reqs = self.mem.put("reqs", reqs)
            if device_y:
                self.d_order = self.mem.put("y_order", np.ascontiguousarray(ydev["order"], dtype=np.int32))
                self.d_keys = self.mem.put("y_keys", np.ascontiguousarray(ydev["keys"], dtype=np.float64))
                self.d_nkeys = self.mem.put("y_nkeys", np.ascontiguousarray(ydev["n_keys"], dtype=np.int32))
                self.d_limit = self.mem.put("y_limit", np.ascontiguousarray(ydev["limit"], dtype=np.int32))
            self._static_key = key
        shift0, bits0 = plan[0]
        nb0 = 1 << bits0
        hist0 = mem.device("hist0", n_inst * max_pos * nb0 * 4)
        run(lib.csg_memset, h, hist0.ptr, 0, n_inst * max_pos * nb0 * 4)
        rows = _count_rows(n_items, R, count_rows)
        d_counts = mem.device("counts", rows * max_E * 4)
        d_npos = mem.device("npos", max(n_items, 1) * 4)
        d_ehist = None
        if device_y:
            d_ehist = mem.device("ehist", n_inst * max_pos * max_E * 4)
            run(lib.csg_memset, h, d_ehist.ptr, 0, n_inst * max_pos * max_E * 4)
        elif R > 1:
            run(lib.csg_memset, h, d_counts.ptr, 0, rows * max_E * 4)
        sums = self.batch.d_sums.ptr
        if n_items:
            run(lib.csg_pool_hist_first, h, sums, code, self.d_items.ptr, n_items, max_pos, bits0, max_E, hist0.ptr,
                                        d_counts.ptr, d_npos.ptr, d_ehist.ptr if device_y else None)
        n_out = (n_req + n_inst + 5 + 1) & ~1  # doubles, 16-byte multiple
        n_count_rows = 0 if device_y else (n_items if R == 1 else R * rows)
        sizes = [("out", n_out * 8), ("counts", n_count_rows * max_E * 4), ("npos", n_items * 4)]
        pin = mem.pinned("readback", sum(_al(n) for _, n in sizes) + 64)
        views, off = {}, 0
        for name, n in sizes:
            views[name] = (off, n)
            off += _al(n)
        if not device_y:
            # the per-energy positive counts are final here: read them back now so the host can
            # work on the y extrema while the digit loop runs
            if R > 1:  # every rank's per-file counts, gathered on the device
                g = gather(d_counts.ptr, _al(rows * max_E * 4, 16))
                run(lib.csg_d2h, h, pin.ptr + views["counts"][0], g, R * rows * max_E * 4)
                assert _al(rows * max_E * 4, 16) == rows * max_E * 4 or R == 1, "count rows must pack to 16 bytes"
            elif n_items:
                run(lib.csg_d2h, h, pin.ptr + views["counts"][0], d_counts.ptr, n_items * max_E * 4)
            if n_items:
                run(lib.csg_d2h, h, pin.ptr + views["npos"][0], d_npos.ptr, n_items * 4)
            record(self.EVENT_SLOT - 1)
        # ---- level 0: scan, exchange [bucket totals | per-energy totals], lower ranks' base
        e_cols = max_E if device_y else 0
        pay0 = _al(n_inst * (nb0 + e_cols) * 4, 16)
        d_tot = mem.device("totals", max(n_inst * S * 1024 * 4, pay0))
        d_base = mem.device("base", n_inst * S * 1024 * 4) if R > 1 else None
        d_above = mem.device("above", n_inst * 8) if R > 1 else None
        run(lib.csg_pool_scan, h, hist0.ptr, n_inst, max_pos, self.d_inst_len.ptr, 1, bits0, None, d_tot.ptr if R > 1 else None)
        etot_off = n_inst * nb0 * 4
        if device_y:
            run(lib.csg_pool_scan_cols, h, d_ehist.ptr, n_inst, max_pos, self.d_inst_len.ptr, max_E,
                                       d_tot.ptr + etot_off if R > 1 else None)
        g_etot, stride0 = None, pay0 // 4
        if R > 1:
            g0 = gather(d_tot.ptr, pay0)
            run(lib.csg_pool_base, h, g0, stride0, R, ex.rank, n_inst, nb0, d_base.ptr, d_above.ptr)
            g_etot = g0 + etot_off
        d_ycand = None
        if device_y:
            d_ycand = mem.device("ycand", n_inst * 8)
            run(lib.csg_pool_energy_candidates, h, d_ehist.ptr, n_inst, max_pos, max_E, self.d_order.ptr, self.d_keys.ptr,
                                               self.d_nkeys.ptr, self.d_limit.ptr, g_etot, stride0, ex.rank, d_ycand.ptr)
        d_n_after = mem.device("n_after", n_inst * max_pos * 8)
        d_below = mem.device("below", n_inst * 8)
        d_flags = mem.device("flags", 16)
        d_sel = mem.device("sel", max(n_req, 1) * max_pos * POOL_SEL.itemsize)
        slot_pay = int(lib.csg_pool_slot_payload_bytes(n_inst, S))
        d_xbuf = mem.device("slot_payload", slot_pay)  # [64 x int64 bounds | n_inst x S slot lists]
        d_best, d_local = d_xbuf.ptr, d_xbuf.ptr + 64 * 8
        d_table = mem.device("table", n_inst * S * 8)
        d_values = mem.device("values", 64 * 8)
        d_has = mem.device("has", 64 * 4)
        d_out = mem.device("out", n_out * 8)
        d_red = mem.device("out_reduced", n_out * 8)
        base_ptr = d_base.ptr if R > 1 else None
        run(lib.csg_memset, h, d_flags.ptr, 0, 16)
        run(lib.csg_pool_row_totals, h, hist0.ptr, n_inst, max_pos, bits0, base_ptr, d_n_after.ptr, d_below.ptr)
        run(lib.csg_pool_sel_init, h, code, self.d_reqs.ptr, n_req, self.d_inst_len.ptr, max_pos, d_n_after.ptr,
                                  d_below.ptr, d_above.ptr if R > 1 else None, d_sel.ptr)
        run(lib.csg_pool_sel_locate, h, hist0.ptr, max_pos, 1, bits0, base_ptr, d_sel.ptr, n_req, d_flags.ptr)
        prev_shift = shift0
        for shift, bits in plan[1:]:
            nb = 1 << bits
            # bounds + locally pruned slot lists travel together; the global bound is applied after
            run(lib.csg_pool_sel_bounds, h, d_sel.ptr, self.d_reqs.ptr, n_req, max_pos, prev_shift, d_best)
            run(lib.csg_pool_sel_slots, h, d_sel.ptr, self.d_reqs.ptr, n_req, max_pos, prev_shift, d_best, n_inst, S,
                                       d_local, d_flags.ptr)
            g = gather(d_xbuf.ptr, slot_pay) if R > 1 else d_xbuf.ptr
            run(lib.csg_pool_sel_assign, h, d_sel.ptr, self.d_reqs.ptr, n_req, max_pos, prev_shift, g, slot_pay, R, n_inst, S,
                                        d_table.ptr, d_flags.ptr)
            nbytes = n_inst * max_pos * S * nb * 4
            hist1 = mem.device("hist1", nbytes)
            run(lib.csg_memset, h, hist1.ptr, 0, nbytes)
            if n_items:
                run(lib.csg_pool_hist_refine, h, sums, code, self.d_items.ptr, n_items, max_pos, S, d_table.ptr, prev_shift,
                                             shift, bits, hist1.ptr)
            run(lib.csg_pool_scan, h, hist1.ptr, n_inst, max_pos, self.d_inst_len.ptr, S, bits, d_table.ptr,
                                  d_tot.ptr if R > 1 else None)
            if R > 1:
                g = gather(d_tot.ptr, n_inst * S * nb * 4)
                run(lib.csg_pool_base, h, g, n_inst * S * nb, R, ex.rank, n_inst, S * nb, d_base.ptr, None)
            run(lib.csg_pool_sel_locate, h, hist1.ptr, max_pos, S, bits, base_ptr, d_sel.ptr, n_req, d_flags.ptr)
            prev_shift = shift
        run(lib.csg_pool_sel_finish, h, code, d_sel.ptr, n_req, max_pos, d_values.ptr, d_has.ptr)
        # ---- one last payload: [values | y candidates | flags | exchange error], max over the ranks
        run(lib.csg_pool_pack_results, h, d_values.ptr, n_req, d_ycand.ptr if device_y else None, n_inst, d_flags.ptr,
                                      ex.error_ptr, d_out.ptr, n_out)
        src = d_out.ptr
        if R > 1:
            g = gather(d_out.ptr, n_out * 8)
            run(lib.csg_pool_reduce_max, h, g, R, n_out, d_red.ptr)
            src = d_red.ptr
        run(lib.csg_d2h, h, pin.ptr + views["out"][0], src, n_out * 8)
        record(self.EVENT_SLOT)
        if not dry:
            self._last_exchange = ex
            self._pending = _Readback(pin, views, n_req, n_inst, max_E, n_count_rows, device_y)

    def _view(self, name, dt):
        pin, views = self._pending.pin, self._pending.views
        return pin.view(dt, views[name][1] // np.dtype(dt).itemsize, views[name][0])

    def result_counts(self):
        """(counts[n_items][max_E], npos[n_items]) -- available right after the first histogram pass."""
        p = self._pending
        if p.device_y:
            raise _lib.CsgError("per-file counts are not read back when the y candidates are computed on the device")
        self.ctx.event_sync(self.EVENT_SLOT - 1)
        return self._view("counts", np.int32).reshape(p.n_count_rows, p.max_E).copy(), self._view("npos", np.int32).copy()

    def _out(self):
        n_req, n_inst = self._pending.n_req, self._pending.n_inst
        self.ctx.event_sync(self.EVENT_SLOT)
        out = self._view("out", np.float64)
        flags = out[n_req + n_inst : n_req + n_inst + 4]
        if out[n_req + n_inst + 4] != 0:
            ex = self.__dict__.get("_last_exchange")
            if ex is not None and hasattr(ex, "clear_error"):
                ex.clear_error()
            raise _lib.CsgError(f"peer exchange timed out waiting for rank {int(out[n_req + n_inst + 4]) - 1}")
        return out[:n_req], out[n_req : n_req + n_inst], flags

    def result_values(self):
        """One float per request (None: empty pool), or None when the slot table overflowed."""
        values, _, flags = self._out()
        if flags[1]:  # slot overflow: later digits ran on a truncated table, their flags mean nothing
            self.overflows = self.__dict__.get("overflows", 0) + 1
            return None
        if flags[0] or flags[2]:
            raise _lib.CsgError("device pool selection: a rank fell outside its bucket (histogram / scan mismatch)")
        return [float(v) if np.isfinite(v) else None for v in values]

    def result_y_candidates(self):
        """Largest 99 %-coverage energy per instrument over the positions below ``limit`` (None:
        no position took part on any rank).  Only with ``ydev``."""
        _, ycand, _ = self._out()
        return [float(v) if v != -np.inf else None for v in ycand]

    def result(self):
        """(values | None on slot overflow, counts, npos); waits for the read-backs only."""
        counts, npos = self.result_counts()
        return self.result_values(), counts, npos


# where the last DevicePoolSelector.enqueue lands its read-backs (views: {name: (byte offset, bytes)} in pin)
_Readback = namedtuple("_Readback", "pin views n_req n_inst max_E n_count_rows device_y")


def _count_rows(n_items: int, n_ranks: int, count_rows: int | None) -> int:
    """Rows of this rank's per-file count table (several ranks: what every rank adds to the gather)."""
    return max(n_items, 1) if (n_ranks == 1 or count_rows is None) else max(int(count_rows), n_items, 1)


def _al(n: int, a: int = 64) -> int:
    return (int(n) + a - 1) // a * a


class SingleRank:
    rank, size = 0, 1

    def allgather(self, arr: np.ndarray) -> list[np.ndarray]:
        return [arr]

    def allgather_object(self, obj):
        return [obj]


def prefix_percentiles(backend, dtype, items: np.ndarray, n_inst: int, inst_len: np.ndarray, max_E: int,
                       requests: list[dict], comm=None):
    """Resolve percentile requests over prefix pools.

    ``items`` (POOL_ITEM) are this rank's files, ``pos`` = local position in the
    instrument's sequence.  ``requests`` entries::

        {"inst": i, "p": percentile, "mode": "running_max" | "last"}

    ``running_max`` -> max over every prefix of nanpercentile(prefix pool, p) (NaN-free: the
    pool holds finite positives only); ``last`` -> the percentile of the whole pool.
    Returns ``(values, counts, npos)``: one float per request (``None`` when the
    instrument's pool is empty everywhere), the per-item per-energy positive counts and
    per-item positive totals (host side of ``fast/extrema.py:260-264``).
    """
    comm = comm or SingleRank()
    D = np.dtype(dtype)
    plan = digit_plan(D)
    max_pos = int(inst_len.max()) if len(inst_len) else 0
    backend.set_items(items, n_inst, max_pos, inst_len, max_E)

    # ---- digit 0: histograms, positive counts
    shift0, bits0 = plan[0]
    counts, npos = backend.hist_first(bits0)
    n_after = np.zeros((n_inst, max(max_pos, 1)), dtype=np.int64)
    if len(items):
        per = np.zeros((n_inst, max(max_pos, 1)), dtype=np.int64)
        per[items["inst"], items["pos"]] = npos
        n_after = np.cumsum(per, axis=1)
    local_tot = n_after[:, -1].copy() if max_pos else np.zeros(n_inst, np.int64)
    all_tot = comm.allgather(local_tot)
    below = np.sum(all_tot[: comm.rank], axis=0).astype(np.int64) if comm.rank > 0 else np.zeros(n_inst, np.int64)
    grand = np.sum(all_tot, axis=0).astype(np.int64)
    n_after = n_after + below[:, None]

    # ---- queries: (request, pos) pairs -> two rank targets each
    qr, qp, qlo, qhi, qg = [], [], [], [], []
    for r, req in enumerate(requests):
        i = req["inst"]
        L = int(inst_len[i])
        if L == 0:
            continue
        n = n_after[i, :L]
        if req["mode"] == "last":
            holders = [rk for rk in range(comm.size) if all_tot[rk][i] > 0]
            if not holders or holders[-1] != comm.rank:
                continue
            ks = np.array([L - 1])
        else:
            prev = np.concatenate([[below[i]], n[:-1]])
            ks = np.flatnonzero((n > 0) & (n != prev))  # a file without positives repeats the candidate
        if len(ks) == 0:
            continue
        lo, hi, g = percentile_ranks(n[ks], req["p"], D)
        qr.append(np.full(len(ks), r)), qp.append(ks), qlo.append(lo), qhi.append(hi), qg.append(g)
    if qr:
        q_req, q_pos = np.concatenate(qr), np.concatenate(qp)
        q_lo, q_hi, q_gamma = np.concatenate(qlo), np.concatenate(qhi), np.concatenate(qg)
    else:
        q_req = q_pos = q_lo = q_hi = np.zeros(0, np.int64)
        q_gamma = np.zeros(0, D)
    nq = len(q_req)
    req_inst = np.array([r["inst"] for r in requests], dtype=np.int64)
    req_runmax = np.array([r["mode"] == "running_max" for r in requests], dtype=bool)
    q_inst = req_inst[q_req] if nq else np.zeros(0, np.int64)
    t_rank = np.empty(2 * nq, dtype=np.int64)
    t_rank[0::2], t_rank[1::2] = q_lo, q_hi
    t_prefix = np.zeros(2 * nq, dtype=np.uint64)
    t_inst = np.repeat(q_inst, 2)
    t_pos = np.repeat(q_pos, 2)
    active = np.ones(nq, dtype=bool)

    def exchange_base(totals):
        """counts held by lower ranks for every (inst, slot, bin)"""
        if comm.size == 1 or totals is None:
            return None
        allt = comm.allgather(totals)
        if comm.rank == 0:
            return None
        return np.sum(np.stack(allt[: comm.rank]).astype(np.uint64), axis=0).astype(np.uint32)

    prev_shift = None
    for level, (shift, bits) in enumerate(plan):
        if level == 0:
            base = exchange_base(backend.scan(comm.size > 1))
            _locate(backend, base, t_inst, t_pos, np.zeros(2 * nq, np.int64), t_rank, t_prefix, np.repeat(active, 2), bits)
        else:
            act_t = np.repeat(active, 2)
            mine = [np.unique(t_prefix[act_t & (t_inst == i)]) for i in range(n_inst)]
            if comm.size > 1:
                parts = comm.allgather_object(mine)
                mine = [np.unique(np.concatenate([p[i] for p in parts])) for i in range(n_inst)]
            todo = [m for m in mine]
            done_t = ~act_t
            while True:
                n_slots = min(MAX_SLOTS, max((len(v) for v in todo), default=0))
                if n_slots == 0:
                    break
                table = np.full((n_inst, n_slots), _U64MAX, dtype=np.uint64)
                for i in range(n_inst):
                    chunk = todo[i][:n_slots]
                    todo[i] = todo[i][n_slots:]
                    table[i, : len(chunk)] = chunk
                backend.hist_refine(table, prev_shift, shift, bits)
                base = exchange_base(backend.scan(comm.size > 1))
                # slot of every pending target = position of its prefix in its instrument's row
                t_slot = np.full(2 * nq, -1, dtype=np.int64)
                for i in range(n_inst):
                    sel = np.flatnonzero(~done_t & (t_inst == i))
                    if len(sel) == 0:
                        continue
                    row = table[i]
                    s = np.searchsorted(row, t_prefix[sel])
                    s = np.minimum(s, n_slots - 1)
                    hit = row[s] == t_prefix[sel]
                    t_slot[sel[hit]] = s[hit]
                pending = t_slot >= 0
                _locate(backend, base, t_inst, t_pos, t_slot, t_rank, t_prefix, pending, bits)
                done_t |= pending
        prev_shift = shift
        # ---- prune prefixes that cannot hold the running maximum
        if nq:
            sh = np.uint64(shift)
            lo_bound = bits_to_value(t_prefix[0::2] << sh, D).astype(np.float64)
            hi_bound = bits_to_value(((t_prefix[1::2] + np.uint64(1)) << sh) - np.uint64(1), D).astype(np.float64)
        else:
            lo_bound = hi_bound = np.zeros(0)
        best_local = np.full(len(requests), -np.inf)
        if nq:
            sel = active & req_runmax[q_req]
            np.maximum.at(best_local, q_req[sel], lo_bound[sel])
        best = best_local
        if comm.size > 1:
            best = np.max(np.stack(comm.allgather(best_local)), axis=0)
        if nq:
            drop = req_runmax[q_req] & (hi_bound < best[q_req])
            active &= ~drop

    # ---- exact neighbours -> numpy's lerp -> per-request reduction
    local_val = np.full(len(requests), -np.inf)
    local_has = np.zeros(len(requests), dtype=bool)
    if nq and active.any():
        vals = bits_to_value(t_prefix, D)
        sel = np.flatnonzero(active)
        v = lerp_vec(vals[2 * sel], vals[2 * sel + 1], q_gamma[sel], D).astype(np.float64)
        np.maximum.at(local_val, q_req[sel], v)  # "last" requests hold a single query
        local_has[q_req[sel]] = True
    if comm.size > 1:
        parts = comm.allgather(np.concatenate([local_val, local_has.astype(np.float64)]))
        stack = np.stack(parts)
        local_val = stack[:, : len(requests)].max(axis=0)
        local_has = stack[:, len(requests) :].max(axis=0) > 0
    out = [float(local_val[r]) if (local_has[r] and grand[requests[r]["inst"]] > 0) else None for r in range(len(requests))]
    return out, counts, npos


def _locate(backend, base, t_inst, t_pos, t_slot, t_rank, t_prefix, pending, bits):
    idx = np.flatnonzero(pending)
    if len(idx) == 0:
        return
    q = np.zeros(len(idx), dtype=POOL_QUERY)
    q["inst"], q["pos"], q["slot"], q["rank"] = t_inst[idx], t_pos[idx], t_slot[idx], t_rank[idx]
    q["bin"] = -1
    res = backend.locate(q, base)
    if np.any(res["bin"] < 0):
        raise _lib.CsgError("pool_locate: a rank fell outside its bucket (histogram / scan mismatch)")
    t_prefix[idx] = (t_prefix[idx] << np.uint64(bits)) | res["bin"].astype(np.uint64)
    t_rank[idx] = res["rank"]
