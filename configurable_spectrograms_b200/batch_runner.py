"""Resumable fan-out of a worker over items (reference ``batch_runner.py``): same signature,
same progress-JSON schema (``completed_items / errors / no_data / last_index /
schema_version``, items identified by ``repr``), same return value."""

from __future__ import annotations

import concurrent.futures
import json
import os
import signal
from collections.abc import Callable, Iterable
from typing import Any

from .logging_utils import configure_log_batch, flush_log_buffer, log_error, log_message

__all__ = ["run_batch"]


def _sigint_handler(signum, frame) -> None:
    log_message("[INTERRUPT] SIGINT received: flushing progress and stopping.", force_flush=True)
    raise KeyboardInterrupt


def run_batch(
    items: Iterable[Any],
    worker_fn: Callable[[Any], tuple[Any, str]],
    executor_factory: Callable[[], concurrent.futures.Executor],
    progress_json_path: str | None = None,
    ignore_progress_json: bool = False,
    flush_batch_size: int = 10,
    log_flush_batch_size: int | None = None,
    install_signal_handlers: bool = True,
    *,
    _comm=None,
) -> list[tuple[Any, str]]:
    """Run ``worker_fn`` over ``items`` on the executor with resumable progress (reference ``:33-178``).

    Items already listed under ``completed_items`` are skipped; every finished item is filed
    under ``completed_items`` / ``no_data`` / ``errors`` by its status; the JSON is rewritten
    every ``flush_batch_size`` items and once at the end.  Returns ``[(item, status)]``.

    ``_comm`` (internal; a ``comm.TorchComm`` over the ranks of one job whose executors resolve every
    item on every rank): every rank reads the progress JSON, and once all have, rank 0 alone writes it.
    """
    previous_sigint = None
    if install_signal_handlers:
        try:
            previous_sigint = signal.getsignal(signal.SIGINT)
            signal.signal(signal.SIGINT, _sigint_handler)
        except (ValueError, OSError) as exc:
            log_message(f"[WARN] Could not install temporary SIGINT handler: {exc}")
    flush_batch_size = max(1, int(flush_batch_size))
    configure_log_batch(log_flush_batch_size or flush_batch_size)
    state: dict[str, Any] = {"completed_items": [], "errors": [], "no_data": [], "last_index": -1, "schema_version": 1}
    if progress_json_path is not None and not ignore_progress_json and os.path.exists(progress_json_path):
        try:
            with open(progress_json_path) as handle:
                loaded = json.load(handle)
            if isinstance(loaded, dict):
                for key in state:
                    if key in loaded:
                        state[key] = loaded[key]
        except (OSError, json.JSONDecodeError) as exc:
            log_error(f"[PROGRESS] Failed to read existing progress JSON '{progress_json_path}': {exc}")
    writer = _comm is None or _comm.rank == 0
    if _comm is not None and _comm.size > 1:
        _comm.barrier()  # rank 0's first (truncating) write comes after every rank's read
    item_list = list(items)
    done = set(state.get("completed_items", []))
    pending = [item for item in item_list if repr(item) not in done]
    log_message(f"[BATCH] Starting batch run with {len(pending)} pending / {len(item_list)} total items; "
                f"flush_batch_size={flush_batch_size}")
    unwritten = 0

    def flush(force: bool = False) -> None:
        nonlocal unwritten
        if progress_json_path is None or not writer or (unwritten == 0 and not force) or (unwritten < flush_batch_size and not force):
            return
        try:
            with open(progress_json_path, "w") as handle:
                json.dump(state, handle, indent=2)
            unwritten = 0
        except OSError as exc:
            log_error(f"[PROGRESS] Failed writing progress JSON '{progress_json_path}': {exc}")

    results: list[tuple[Any, str]] = []
    try:
        with executor_factory() as executor:
            futures = {executor.submit(worker_fn, item): item for item in pending}
            for fut in concurrent.futures.as_completed(futures):
                original = futures[fut]
                try:
                    ident, status = fut.result()
                except Exception as exc:
                    ident, status = original, "error"
                    log_error(f"[BATCH-FAIL] Item {original} outer exception: {exc}")
                results.append((ident, status))
                bucket = "completed_items" if status == "ok" else ("no_data" if status == "no_data" else "errors")
                state[bucket].append(repr(ident))
                state["last_index"] = len(results) - 1
                unwritten += 1
                flush()
    finally:
        flush(force=True)
        flush_log_buffer(force=True)
        if install_signal_handlers and previous_sigint is not None:
            try:
                signal.signal(signal.SIGINT, previous_sigint)
            except (ValueError, OSError) as exc:
                log_message(f"[WARN] Could not restore original SIGINT handler: {exc}")
    log_message(
        f"[BATCH] Completed batch run: {len(results)} processed (ok={sum(1 for _, s in results if s == 'ok')} "
        f"no_data={sum(1 for _, s in results if s == 'no_data')} error={sum(1 for _, s in results if s == 'error')})",
        force_flush=True,
    )
    return results
