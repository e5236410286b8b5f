"""Generic batch plotting (reference ``generic_batch.py``): one ``generic_plot_spectrogram_set``
per item, saved as ``output_dir/<item>/generic.png``, resumable through ``run_batch``.

The reference gives every item to a worker process that collapses, ranks, normalises and draws on its
own.  Here the items of a *group* share one pass over the GPU: their datasets are built on a thread pool
(user code), every cube is uploaded and collapsed as it arrives, then ONE percentile launch and ONE raster
launch serve every panel of the group and the figures are composed and PNG-encoded on the device
(``plotting.SpectrogramGroup``).  ``run_batch`` still sees one future per item: ``GroupedExecutor`` is the
executor it is handed.

Under ``torchrun`` (``torch.distributed`` initialised, several ranks) every rank runs on its own GPU: the
ranks walk the same pending items in rounds, each rank plots its slice of a round, and every rank hands
``run_batch`` every item's status, so every rank returns the full result list.  Rank 0 alone writes the
progress JSON; each rank writes the PNG files of its own items.
"""

from __future__ import annotations

import concurrent.futures
import functools
import os
import threading
from collections.abc import Callable
from concurrent.futures import ThreadPoolExecutor
from typing import Any

from .batch_runner import run_batch
from .comm import TorchComm, block_of, current_device, rank_world
from .constants import PLOTTING_PROGRESS_JSON_PATH
from .figure import close_all_axes_and_clear
from .logging_utils import log_error
from .plotting import SpectrogramGroup, generic_plot_spectrogram_set

__all__ = ["generic_batch_plot", "GroupedExecutor"]

#: ``fig.savefig(out_path, dpi=150)`` (reference ``generic_batch.py:113``)
SAVE_DPI = 150


class GroupedExecutor(concurrent.futures.Executor):
    """An executor whose tasks are whole groups of items: ``submit(fn, item)`` only queues the item; a
    single service thread takes ``group_size`` items at a time and runs ``process_group(items)`` -- which
    returns one result per item -- so the items of a group can share their GPU work.  ``fn`` itself is not
    called (the group function replaces it).

    ``comm`` (a ``comm.TorchComm`` over several ranks): every rank submits the same items in the same order.
    The ranks take them in rounds of up to ``group_size`` items per rank, whose size they agree on through
    ``comm`` (the fewest items any rank has queued, so every rank's round holds the same items); rank r runs
    ``process_group`` on the r-th contiguous slice of a round, the ranks all-gather their results, and every
    rank resolves every future of the round.  Results travel between ranks, so they must pickle."""

    def __init__(self, process_group: Callable[[list], list], group_size: int, comm=None):
        self._process, self._size = process_group, max(1, int(group_size))
        self._comm = comm if comm is not None and comm.size > 1 else None
        self._queue: list = []
        self._lock = threading.Condition()
        self._closed = False
        self._thread = threading.Thread(target=self._serve if self._comm is None else self._serve_ranks, daemon=True)
        self._thread.start()

    def submit(self, fn, item):  # noqa: D102  (Executor API)
        future: concurrent.futures.Future = concurrent.futures.Future()
        with self._lock:
            if self._closed:
                raise RuntimeError("cannot schedule new items after shutdown")
            self._queue.append((item, future))
            self._lock.notify()
        return future

    def _serve(self):
        while True:
            with self._lock:
                while not self._queue and not self._closed:
                    self._lock.wait()
                if not self._queue:
                    return
                # a full group, or whatever is left once nothing more will come
                if len(self._queue) < self._size and not self._closed:
                    self._lock.wait(timeout=0.05)
                take, self._queue = self._queue[: self._size], self._queue[self._size :]
            live = [(item, fut) for item, fut in take if fut.set_running_or_notify_cancel()]
            if not live:
                continue
            try:
                results = self._process([item for item, _f in live])
                for (_item, fut), res in zip(live, results):
                    fut.set_result(res)
            except BaseException as exc:  # a failure of the group machinery fails its items, not the batch
                for _item, fut in live:
                    if not fut.done():
                        fut.set_exception(exc)

    def _serve_ranks(self):
        comm = self._comm
        full = self._size * comm.size
        take: list = []
        try:
            while True:
                with self._lock:
                    while not self._queue and not self._closed:
                        self._lock.wait()
                    if len(self._queue) < full and not self._closed:
                        self._lock.wait(timeout=0.05)
                    offer = (len(self._queue), self._closed)
                offers = comm.allgather_object(offer)
                n = min(full, min(queued for queued, _closed in offers))
                if n == 0:
                    if all(closed for _queued, closed in offers):
                        return
                    continue
                with self._lock:
                    take, self._queue = self._queue[:n], self._queue[n:]
                self._round(take)
                take = []
        except BaseException as exc:  # the exchange itself failed: no rank can resolve these futures any more
            with self._lock:
                left, self._queue = take + self._queue, []
            for _item, fut in left:
                if not fut.done():
                    fut.set_exception(exc)

    def _round(self, take: list):
        """Run this rank's slice of one round; resolve every future of the round from every rank's results."""
        comm = self._comm
        live = [fut.set_running_or_notify_cancel() for _item, fut in take]
        lo, hi = block_of(len(take), comm.rank, comm.size)
        outcome: tuple = ("ok", [])
        try:
            if lo < hi:
                outcome = ("ok", list(self._process([item for item, _f in take[lo:hi]])))
        except BaseException as exc:  # a failure of the group machinery fails its items, not the batch
            outcome = ("error", f"{type(exc).__name__}: {exc}")
        finally:  # every rank joins every round's exchange, with an empty slice or a failed group too
            parts = comm.allgather_object(outcome)
        per = -(-len(take) // comm.size)
        for k, (_item, fut) in enumerate(take):
            if not live[k]:
                continue
            kind, payload = parts[k // per]
            if kind == "ok" and k % per < len(payload):
                fut.set_result(payload[k % per])
            else:
                fut.set_exception(RuntimeError(payload if kind == "error" else "the group returned no result for this item"))

    def shutdown(self, wait=True, *, cancel_futures=False):  # noqa: D102
        with self._lock:
            self._closed = True
            if cancel_futures:
                for _item, fut in self._queue:
                    fut.cancel()
                self._queue = []
            self._lock.notify_all()
        if wait:
            self._thread.join()


def generic_batch_plot(
    items,
    output_dir: str,
    build_datasets_fn: Callable[[Any], list[dict]],
    zoom_center_fn: Callable[[Any], float | None] | None = None,
    zoom_window_seconds: float | None = None,
    vertical_lines_fn: Callable[[Any], list[float] | None] | None = None,
    y_scale: str = "linear",
    z_scale: str = "linear",
    colormap: str = "viridis",
    cusp_marker_style: str = "both",
    cusp_marker_kwargs: dict | None = None,
    max_workers: int = 2,
    progress_json_path: str = PLOTTING_PROGRESS_JSON_PATH,
    ignore_progress_json: bool = False,
    flush_batch_size: int = 10,
    log_flush_batch_size: int | None = None,
    install_signal_handlers: bool = True,
) -> list[tuple[Any, str]]:
    """Plot every item (reference ``:15-129``).  Returns ``[(item, status)]`` with status in
    ``{'ok', 'no_data', 'error'}``.  ``max_workers`` sizes the thread pool that builds the datasets and the
    GPU group (``8 * max_workers`` items share a pass, ``CSG_GENERIC_GROUP`` overrides).

    Under ``torchrun`` the ranks share the items (see the module docstring); every rank passes the same
    ``items`` and returns every item's status."""
    from . import _lib
    from .png import write_figures_device

    os.makedirs(output_dir, exist_ok=True)
    workers = max(1, int(max_workers))
    group_size = max(1, int(os.environ.get("CSG_GENERIC_GROUP", str(8 * workers))))
    _rank, world, dist = rank_world()
    comm, device = None, 0
    if world > 1:
        # the ranks' statuses are host objects: a gloo group keeps them off the GPU collectives' streams.  The
        # device is read here: the executor's service thread, where the groups run, starts on device 0
        comm = TorchComm(dist, group=dist.new_group(backend="gloo"))
        device = current_device()

    def build(item):
        try:
            return build_datasets_fn(item), None
        except Exception as exc:
            return None, exc

    def process_group(items):
        if world > 1:  # launches go to the calling thread's current device, and this thread started on device 0
            import torch

            torch.cuda.set_device(device)
        ctx = _lib.default_context(device)
        group = SpectrogramGroup(colormap, ctx)
        status = ["error"] * len(items)
        figures: dict[int, Any] = {}
        owners: list[int] = []  # which item (position in the group) every planned panel belongs to
        with ThreadPoolExecutor(max_workers=workers) as pool:
            built = list(pool.map(build, items))
        for k, (item, (datasets, failure)) in enumerate(zip(items, built)):
            try:
                if failure is not None:
                    raise failure
                if not datasets:
                    status[k] = "no_data"
                    continue
                before = len(group.pending)
                fig, _canvas = generic_plot_spectrogram_set(
                    datasets, zoom_center=zoom_center_fn(item) if zoom_center_fn else None,
                    zoom_window_seconds=zoom_window_seconds, vertical_lines=vertical_lines_fn(item) if vertical_lines_fn else None,
                    y_scale=y_scale, z_scale=z_scale, colormap=colormap, cusp_marker_style=cusp_marker_style,
                    cusp_marker_kwargs=cusp_marker_kwargs, show=False, _group=group,
                )
                owners += [k] * (len(group.pending) - before)
                figures[k] = fig
                status[k] = "ok"
            except Exception as exc:
                log_error(f"[GENERIC-FAIL] Item {item}: {exc}")
        try:
            for k, failure in zip(owners, group.run()):
                if failure is not None and status[k] == "ok":
                    log_error(f"[GENERIC-FAIL] Item {items[k]}: {failure}")
                    status[k] = "error"
            saves: dict = {}
            for k, fig in figures.items():
                if status[k] != "ok" or fig is None:
                    continue
                item_dir = os.path.join(output_dir, str(items[k]))
                os.makedirs(item_dir, exist_ok=True)
                path = os.path.join(item_dir, "generic.png")
                if any(ax.images for ax in fig.axes):
                    saves.setdefault(group.rgba_ptr(fig), []).append((path, fig))
                else:  # every dataset was filtered out: the reference still saves the (empty) figure
                    fig.savefig(path, dpi=SAVE_DPI)
            for ptr, jobs in saves.items():
                write_figures_device(ctx, ptr, jobs, max_workers=workers, dpi=SAVE_DPI)
        except Exception as exc:
            log_error(f"[GENERIC-FAIL] Group of {len(items)} items: {exc}")
            status = [("error" if k in figures else st) for k, st in enumerate(status)]
        finally:
            for fig in figures.values():
                close_all_axes_and_clear(fig)
        return list(zip(items, status))

    return run_batch(
        items,
        None,
        functools.partial(GroupedExecutor, process_group, group_size, comm),
        progress_json_path=progress_json_path,
        ignore_progress_json=ignore_progress_json,
        flush_batch_size=flush_batch_size,
        log_flush_batch_size=log_flush_batch_size,
        install_signal_handlers=install_signal_handlers,
        _comm=comm,
    )
