"""CPU tests of the product's host-side bookkeeping (no GPU, no libcsgpu compute): the extrema
walk, the per-step energy candidates and the shard planner's masks, checked against the
reference's own results (tests/golden) with numpy standing in for the device selection."""

import numpy as np

from configurable_spectrograms_b200.fast import extrema as X
from tests.helpers import load_json
from tests.test_oracle import _tree_files


def _brute_energy_candidates(energies, counts):
    """CS/fast/extrema.py:261-278 literally: dict keyed by float(energy), sorted, cumsum, searchsorted."""
    acc, out = {}, []
    for e, c in zip(energies, counts):
        for ev, cnt in zip(e, c):
            if cnt:
                acc[float(ev)] = acc.get(float(ev), 0) + int(cnt)
        if not acc:
            out.append(0.0)
            continue
        ks = np.array(sorted(acc))
        cum = np.cumsum([acc[k] for k in ks])
        idx = min(int(np.searchsorted(cum, 0.99 * cum[-1], side="right")), len(ks) - 1)
        out.append(float(ks[idx]))
    return out


def test_energy_candidates_paths_agree():
    rng = np.random.default_rng(0)
    for dup in (False, True):
        energy = np.sort(rng.uniform(4, 30000, 96))[::-1].copy()
        if dup:
            energy[10:14] = energy[10]
            energy[50] = energy[51]
        n = 17
        counts = rng.integers(0, 40, (n, 96)) * (rng.random((n, 96)) < 0.7)
        counts[3] = 0
        counts[0, 60:] = 0
        shared = X.energy_candidates([energy] * n, counts)
        separate = X.energy_candidates([energy.copy() for _ in range(n)], counts)
        brute = _brute_energy_candidates([energy] * n, counts)
        assert shared == separate == brute
    # files with different tables, and an empty leading pool
    e1, e2 = np.linspace(10, 1000, 12), np.linspace(5, 3000, 9)
    cs = [np.zeros(12, int), rng.integers(0, 9, 12), rng.integers(0, 9, 9), rng.integers(0, 9, 12)]
    es = [e1, e1, e2, e1]
    padded = [np.pad(c, (0, 12 - len(c))) for c in cs]
    assert X.energy_candidates(es, padded) == _brute_energy_candidates(es, cs)


def _numpy_scan(files, order, max_percentile, compute_mins):
    """on_scan for X._walk with numpy standing in for K1/K2b (same semantics as the device path:
    one call per (instrument, orbit index) in sequence order)."""
    pools = {i: [] for i in order}
    counts = {i: ([], []) for i in order}

    def scan(inst, orbit_index, handle):
        _o, per = files[orbit_index]
        if inst in per:
            energy, cube = per[inst]
            with np.errstate(invalid="ignore", over="ignore"):
                c = np.nansum(cube, axis=1)
            m = np.isfinite(c) & (c > 0)
            counts[inst][0].append(energy)
            counts[inst][1].append(m.sum(axis=0))
            if m.any():
                pools[inst].append(c[m])
        ce = X.energy_candidates(*counts[inst])
        cand_e = ce[-1] if ce else 0.0
        cand_z, z_min = 0.0, 0
        if pools[inst]:
            pool = np.concatenate(pools[inst])
            cand_z = float(np.nanpercentile(pool, max_percentile))
            if compute_mins:
                z_min = float(np.nanpercentile(pool, 1))
        return cand_e, cand_z, z_min

    return scan


def test_walk_reproduces_reference_extrema_json():
    files, order = _tree_files()
    gold = load_json("extrema_tree.json")
    sequence = [(o, {i: True for i in per}) for o, per in files]
    totals = {i: sum(1 for _, h in sequence if i in h) for i in order}
    state = {}
    for combo in gold["combos"]:  # CLI order, one shared cache
        steps, totals2 = X.plan_scanned_steps(sequence, order, combo["y"], combo["z"], state)
        assert totals2 == totals
        before = json_copy(state)
        state = X._walk(sequence, order, combo["y"], combo["z"], state, totals, 0.1, -1.0, _numpy_scan(files, order, 99.0, False))
        assert state == combo["extrema"], (combo["y"], combo["z"])
        # the dry run predicted exactly the steps that reached the scan
        seen = {i: [] for i in order}

        def record(inst, oi, handle):
            seen[inst].append(oi)
            return 0.0, 0.0, 0

        X._walk(sequence, order, combo["y"], combo["z"], before, totals, 0.1, -1.0, record)
        assert seen == steps
    st = X._walk(sequence, order, "linear", "linear", {}, totals, 0.1, -1.0, _numpy_scan(files, order, 95.0, True))
    assert st == gold["pool95_mins"]
    st = X._walk(sequence, order, "linear", "log", {}, totals, 0.1, -1.0, _numpy_scan(files, order, 99.0, False))
    assert st == gold["batch_extrema"]


def json_copy(obj):
    import json

    return json.loads(json.dumps(obj))


def test_pitch_angle_bits_closed_intervals():
    from configurable_spectrograms_b200.fast.constants import DEFAULT_PITCH_ANGLE_CATEGORIES
    from configurable_spectrograms_b200.fast.pipeline import pitch_angle_bits, zoom_window

    pa = np.array([0.0, 30.0, 35.0, 40.0, 145.0, 150.0, 210.0, 330.0, 360.0, 365.0, np.nan, -3.0])
    bits, keys = pitch_angle_bits(pa, DEFAULT_PITCH_ANGLE_CATEGORIES)
    assert keys == ["all", "downgoing", "upgoing", "perpendicular"] or len(keys) == 4
    g = {k: (bits >> i) & 1 for i, k in enumerate(keys)}
    all_k, down, up, perp = (g[k] for k in keys)
    assert list(all_k) == [1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0]
    assert list(down) == [1, 1, 0, 0, 0, 0, 0, 1, 1, 0, 0, 0]
    assert list(up) == [0, 0, 0, 0, 0, 1, 1, 0, 0, 0, 0, 0]
    assert list(perp) == [0, 0, 0, 1, 0, 0, 1, 1, 0, 0, 0, 0]  # 210 and 330 sit in two groups; 35 and 145 in none
    assert zoom_window([], 6.25) is None
    assert zoom_window([100.0], 6.25) == (100.0, 375.0)
    assert zoom_window([100.0, 1100.0], 6.25) == (600.0, 1500.0)


def test_walk_chain_fast_path_equals_step_loop():
    """The per-instrument chain shortcut writes exactly what the step-by-step loop writes."""
    rng = np.random.default_rng(9)
    order = ("ees", "eeb", "ies", "ieb")
    for trial in range(30):
        n = int(rng.integers(1, 12))
        sequence = []
        for k in range(n):
            present = {i: True for i in order if rng.random() < 0.8}
            sequence.append((13000 + 3 * k, present))
        totals = {i: sum(1 for _, h in sequence if i in h) for i in order}
        table = {(i, k): (float(rng.uniform(0, 5000)), float(rng.uniform(0, 900)), 0) for i in order for k in range(n)}
        scan = lambda inst, oi, h: table[(inst, oi)]
        for ys, zs in (("linear", "log"), ("log", "log"), ("log", "linear"), ("linear", "linear")):
            start = {} if trial % 3 else {"ees_%s_%s_y_max" % (ys, zs): 77, "ees_%s_%s_z_max" % (ys, zs): 12.5}
            if trial % 5 == 0:
                start[f"{ys}_{zs}_last_orbit"] = 13000  # resume: the first orbit is skipped
            fast = X._walk(sequence, order, ys, zs, json_copy(start), totals, 0.1, -1.0, scan)
            slow = X._walk(sequence, order, ys, zs, json_copy(start), totals, 0.1, -1.0, scan, on_step_done=lambda reuse: None)
            assert fast == slow, (trial, ys, zs)
            assert list(fast) and set(fast) == set(slow)

            # the folded variant: one merge with the largest candidate of the chain's steps
            def folded_scan(inst, oi, h):
                return table[(inst, oi)]

            def range_max(inst, a, b):
                return (max(table[(inst, k)][0] for k in range(a, b + 1)), max(table[(inst, k)][1] for k in range(a, b + 1)),
                        table[(inst, b)][2])

            folded = X._walk(sequence, order, ys, zs, json_copy(start), totals, 0.1, -1.0, folded_scan, range_max=range_max)
            assert folded == slow, (trial, ys, zs)


class _FakeSelector:
    """Stands in for pool_select.DevicePoolSelector on the CPU: answers from the collapsed matrices
    with numpy what the kernels answer on the device (single rank)."""

    def __init__(self, mats, order, energy):
        self.mats, self.order, self.energy = mats, order, energy  # mats[(inst, local orbit index)] = (T, E) sums

    def enqueue(self, dtype, items, n_inst, inst_len, max_E, requests, comm=None, count_rows=None, ydev=None, **_kw):
        self.items, self.requests, self.ydev, self.max_E = items, requests, ydev, max_E

    def _files(self, ii):  # this instrument's files in position order
        rows = [it for it in self.items if it["inst"] == ii]
        return [self.mats[int(it["mat_off"])] for it in sorted(rows, key=lambda it: it["pos"])]

    def result_counts(self):
        counts = np.zeros((len(self.items), self.max_E), np.int32)
        npos = np.zeros(len(self.items), np.int32)
        for k, it in enumerate(self.items):
            m = self.mats[int(it["mat_off"])]
            pos = np.isfinite(m) & (m > 0)
            counts[k, : m.shape[1]] = pos.sum(axis=0)
            npos[k] = pos.sum()
        return counts, npos

    def result_values(self):
        out = []
        for rq in self.requests:
            pool, best, last = [], None, None
            for m in self._files(rq["inst"]):
                pos = m[np.isfinite(m) & (m > 0)]
                if pos.size:
                    pool.append(pos)
                if pool:
                    last = float(np.nanpercentile(np.concatenate(pool), rq["p"]))
                    best = last if best is None else max(best, last)
            out.append(best if rq["mode"] == "running_max" else last)
        return out

    def result_y_candidates(self):
        """csg_pool_energy_candidates: the largest 99 %-coverage energy over the positions below `limit`."""
        out = []
        for ii in range(len(self.order)):
            files = self._files(ii)[: int(self.ydev["limit"][ii])]
            if not files:
                out.append(None)
                continue
            counts = [(np.isfinite(m) & (m > 0)).sum(axis=0) for m in files]
            out.append(max(X.energy_candidates([self.energy[ii]] * len(files), np.asarray(counts))))
        return out


def test_device_merged_extrema_equal_the_per_step_walk():
    """extrema_enqueue(per_step=False) + extrema_finish: one merge per instrument from the largest
    candidates (what the device returns) must give the state of the per-step walk over gathered
    counts -- with missing files at the start of a chain, instruments that "complete" early,
    resumed runs and empty files."""
    import types

    from configurable_spectrograms_b200._lib import POOL_ITEM

    rng = np.random.default_rng(17)
    order = ("ees", "eeb", "ies")
    energy = [np.geomspace(30000.0, 4.0, 12), np.geomspace(5.0, 25000.0, 12), rng.permutation(np.linspace(1.0, 4000.0, 12))]
    for trial in range(25):
        n = int(rng.integers(2, 9))
        orbits, mats, file_meta, files = [], {}, [], []
        for k in range(n):
            entry = {"orbit": 13000 + 2 * k, "files": {}, "lines": {}}
            for ii, inst in enumerate(order):
                if rng.random() < 0.25:
                    continue
                m = rng.gamma(2.0, 3.0, (int(rng.integers(3, 9)), 12)) * (40.0 if k == 1 else 1.0)
                m[rng.random(m.shape) < 0.3] = 0.0
                if rng.random() < 0.15:
                    m[:] = 0.0
                fid = len(files)
                files.append({"T": m.shape[0], "E": 12})
                mats[fid] = m.astype(np.float32)
                file_meta.append({"energy": energy[ii]})
                entry["files"][inst] = fid
            orbits.append(entry)
        sequence = [(o["orbit"], {i: True for i in o["files"]}) for o in orbits]

        def make_shard():
            sh = types.SimpleNamespace(orbits=orbits, file_meta=file_meta, first_orbit_index=0, instrument_order=order)
            sh.batch = types.SimpleNamespace(dtype=np.float32, files=files, mat_off=lambda f, g: f)

            def pool_items(steps_by_inst):
                rows, owners, inst_len = [], [], np.zeros(len(order), np.int32)
                for ii, inst in enumerate(order):
                    pos = 0
                    for oi in steps_by_inst.get(inst, []):
                        f = orbits[oi]["files"].get(inst)
                        if f is None:
                            continue
                        rows.append((f, files[f]["T"], 12, ii, pos))
                        owners.append((inst, oi, f))
                        pos += 1
                    inst_len[ii] = pos
                return (np.array(rows, dtype=POOL_ITEM) if rows else np.zeros(0, POOL_ITEM)), inst_len, owners

            sh.pool_items = pool_items
            sh._pool_selector = _FakeSelector(mats, order, energy)
            return sh

        for ys, zs in (("linear", "log"), ("log", "log")):
            start = {}
            if trial % 4 == 1:
                start[f"{ys}_{zs}_last_orbit"] = 13000  # resume after the first orbit
            if trial % 4 == 2:
                start[f"ees_{ys}_{zs}_y_max"], start[f"ees_{ys}_{zs}_z_max"] = 55, 3.0
            results = []
            for per_step in (True, False):
                sh = make_shard()
                pending = X.extrema_enqueue(sh, sequence, order, ys, zs, json_copy(start), max_percentile=99.0,
                                            compute_mins=trial % 2 == 0, per_step=per_step)
                if not per_step:
                    assert pending.ydev is not None, "the chain preconditions hold for every case generated here"
                results.append(X.extrema_finish(pending))
            assert results[0] == results[1], (trial, ys, zs, results)


def test_mirrored_modules_pass_their_doctests():
    """The mirrors carry the reference's doctest examples (its only known-answer pins, SURVEY.md
    section 4): percentile_utils, fast.extrema, cdf_utils, fast.orbit_discovery."""
    import doctest
    import importlib

    total = 0
    for name in ("percentile_utils", "fast.extrema", "cdf_utils", "fast.orbit_discovery"):
        mod = importlib.import_module("configurable_spectrograms_b200." + name)
        result = doctest.testmod(mod, optionflags=doctest.ELLIPSIS | doctest.NORMALIZE_WHITESPACE)
        assert result.failed == 0, (name, result)
        total += result.attempted
    assert total >= 20
