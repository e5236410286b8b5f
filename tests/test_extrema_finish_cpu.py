"""CPU tests of fast.extrema.extrema_finish on a stand-in selector: the slot-overflow fallback in both
y modes, and the refusal to report per-step states from a device-merged selection."""

import types

import numpy as np
import pytest

from configurable_spectrograms_b200._lib import POOL_ITEM
from configurable_spectrograms_b200.fast import extrema as X
from oracle.pool_backend import NumpyPoolBackend
from tests.test_host_logic import _FakeSelector, json_copy

ORDER = ("ees", "eeb", "ies")
N_E = 12


class _OverflowSelector(_FakeSelector):
    """Reports a slot-table overflow: extrema_finish must resolve the values from the host-driven loop."""

    def result_values(self):
        self.overflowed = True
        return None


def _case(rng, energy):
    """Random orbits whose matrices sit in one flat float32 array at their ``mat_off`` offsets:
    ``(sequence, flat, make_shard(selector), {mat_off: matrix})``."""
    orbits, file_meta, mats, chunks, off = [], [], {}, [], 0
    for k in range(int(rng.integers(2, 9))):
        entry = {"orbit": 13000 + 2 * k, "files": {}, "lines": {}}
        for ii, inst in enumerate(ORDER):
            if rng.random() < 0.25:
                continue
            m = rng.gamma(2.0, 3.0, (int(rng.integers(3, 9)), N_E)) * (40.0 if k == 1 else 1.0)
            m[rng.random(m.shape) < 0.3] = 0.0
            if rng.random() < 0.15:
                m[:] = 0.0
            m = m.astype(np.float32)
            entry["files"][inst] = len(file_meta)
            file_meta.append({"energy": energy[ii], "mat_off": off, "T": m.shape[0]})
            mats[off] = m
            chunks.append(m.ravel())
            off += m.size
        orbits.append(entry)
    flat = np.concatenate(chunks) if chunks else np.zeros(0, np.float32)
    sequence = [(o["orbit"], {i: True for i in o["files"]}) for o in orbits]

    def pool_items(steps_by_inst):
        rows, owners, inst_len = [], [], np.zeros(len(ORDER), np.int32)
        for ii, inst in enumerate(ORDER):
            for oi in steps_by_inst.get(inst, []):
                f = orbits[oi]["files"].get(inst)
                if f is None:
                    continue
                rows.append((file_meta[f]["mat_off"], file_meta[f]["T"], N_E, ii, inst_len[ii]))
                owners.append((inst, oi, f))
                inst_len[ii] += 1
        return (np.array(rows, dtype=POOL_ITEM) if rows else np.zeros(0, POOL_ITEM)), inst_len, owners

    def make_shard(selector):
        sh = types.SimpleNamespace(orbits=orbits, file_meta=file_meta, first_orbit_index=0, instrument_order=ORDER)
        sh.batch = types.SimpleNamespace(dtype=np.float32)
        sh.pool_items = pool_items
        sh._pool_selector = selector
        return sh

    return sequence, flat, make_shard, mats


def test_slot_overflow_fallback_through_extrema_finish():
    """With the device slot table overflowed, the values come from prefix_percentiles on the shard's
    cached backend, and the state equals the one from the device values -- per step and merged."""
    rng = np.random.default_rng(23)
    energy = [np.geomspace(30000.0, 4.0, N_E), np.geomspace(5.0, 25000.0, N_E), rng.permutation(np.linspace(1.0, 4000.0, N_E))]
    for trial in range(12):
        sequence, flat, make_shard, mats = _case(rng, energy)
        for ys, zs in (("linear", "log"), ("log", "log")):
            start = {f"{ys}_{zs}_last_orbit": 13000} if trial % 3 == 1 else {}
            for per_step in (True, False):
                states = []
                for selector in (_FakeSelector(mats, ORDER, energy), _OverflowSelector(mats, ORDER, energy)):
                    sh = make_shard(selector)
                    sh._pool_backend = NumpyPoolBackend(flat)
                    pending = X.extrema_enqueue(sh, sequence, ORDER, ys, zs, json_copy(start), max_percentile=99.0,
                                                compute_mins=trial % 2 == 0, per_step=per_step)
                    assert (pending.ydev is None) == per_step
                    states.append(X.extrema_finish(pending))
                assert selector.overflowed
                assert states[1] == states[0], (trial, ys, zs, per_step)


def test_device_merged_finish_refuses_per_step_reports():
    rng = np.random.default_rng(5)
    energy = [np.geomspace(30000.0, 4.0, N_E)] * len(ORDER)
    sequence, _flat, make_shard, mats = _case(rng, energy)
    pending = X.extrema_enqueue(make_shard(_FakeSelector(mats, ORDER, energy)), sequence, ORDER, "linear", "log", {},
                                per_step=False)
    assert pending.ydev is not None
    with pytest.raises(ValueError):
        X.extrema_finish(pending, on_step_done=lambda reuse: None)
