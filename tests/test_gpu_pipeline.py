"""GPU parity of the planned batch path (ShardPlan / BatchStep / extrema) against what the
UNMODIFIED reference produced (tests/golden/*, captured by tests/golden/make_golden.py) and
against the oracle port of its batch step."""

import json

import numpy as np
import pytest

from oracle import cpu_pipeline as CP
from oracle import restate as R
from tests.helpers import dataset_from_arrays, load_json, load_npz, panels, same_float

pytestmark = pytest.mark.gpu

ORDER = ("ees", "eeb", "ies", "ieb")


@pytest.fixture(scope="module")
def ctx():
    from configurable_spectrograms_b200 import _lib

    return _lib.Context(0)


def _lut():
    return R.lut_with_extremes(np.random.default_rng(3).integers(0, 256, (256, 4), dtype=np.uint8))


def _check_panel(batch, norms, pid, ref, lut, what):
    nm = norms[pid]
    assert nm["status"] == 0, what
    assert same_float(nm["vmin"], ref["vmin"]) and same_float(nm["vmax"], ref["vmax"]), (what, nm["vmin"], ref["vmin"], nm["vmax"], ref["vmax"])
    idx_ref, rgba_ref = R.rasterise(ref, lut)
    got = batch.panel_index(pid)
    assert got.shape == idx_ref.shape, (what, got.shape, idx_ref.shape)
    assert np.array_equal(got, idx_ref), (what, int((got != idx_ref).sum()))
    assert np.array_equal(batch.panel_rgba(pid), rgba_ref), what


def test_pitch_angle_grid_matches_reference_captures(ctx):
    from configurable_spectrograms_b200.fast.pipeline import ShardPlan

    g = load_npz("pa_grid.npz")
    ds = dataset_from_arrays({k[3:]: v for k, v in g.items() if k.startswith("in_")})
    lo, hi = g["cusp_idx"]
    lines = [float(ds["times"][lo]), float(ds["times"][hi])]
    lut = _lut()
    for zs in ("linear", "log"):
        for variant, kw in (("raw", {}), ("given", dict(y_min=0.0, y_max=2900.0, z_min=0.0, z_max=460.0))):
            ref = panels(g, f"{variant}_{zs}")
            shard = ShardPlan(ctx, "linear", zs)
            shard.add_orbit(777, {"ees": ds}, {"ees": lines})
            shard.upload()
            shard.collapse()
            fig = shard.plan_pitch_angle_grid(shard.orbits[0], "ees", variant, **kw)
            shard.run_once(lut, want_index=True)
            assert fig.zoom_needed
            norms = shard.batch.norms()
            assert len(fig.rows) == 4 and len(ref) == 8
            k = 0
            for row in fig.rows:
                for pid in (row.full_panel, row.zoom_panel):
                    _check_panel(shard.batch, norms, pid, ref[k], lut, (zs, variant, row.label, k))
                    k += 1


def test_instrument_grid_matches_reference_captures(ctx):
    from configurable_spectrograms_b200.fast.pipeline import ShardPlan

    g = load_npz("inst_grid.npz")
    ext = json.loads(str(g["extrema_json"]))
    dsets, lines = {}, {}
    for inst in ORDER:
        ds = dataset_from_arrays({k[len(inst) + 4 :]: v for k, v in g.items() if k.startswith(f"in_{inst}_")})
        dsets[inst] = ds
        lines[inst] = [float(ds["times"][40]), float(ds["times"][60])]
    lut = _lut()
    for tag, ge in (("raw", None), ("given", ext)):
        ref = panels(g, tag)
        shard = ShardPlan(ctx, "linear", "log")
        shard.add_orbit(778, dsets, lines)
        shard.upload()
        shard.collapse()
        fig = shard.plan_instrument_grid(shard.orbits[0], tag, global_extrema=ge)
        shard.run_once(lut, want_index=True)
        assert fig.zoom_needed
        norms = shard.batch.norms()
        assert len(ref) == 2 * len(fig.rows)
        k = 0
        for row in fig.rows:
            for pid in (row.full_panel, row.zoom_panel):
                _check_panel(shard.batch, norms, pid, ref[k], lut, (tag, row.label, k))
                k += 1


def _tree():
    import io

    import pandas as pd

    from configurable_spectrograms_b200.cdf_utils import get_timestamps_for_orbit

    tree = load_npz("extrema_tree.npz")
    orbits = sorted({int(k.split("_")[0]) for k in tree if k[0].isdigit()})
    frame = pd.read_csv(io.StringIO(str(tree["csv"])), sep="\t")
    out = []
    for o in orbits:
        dsets, lines = {}, {}
        for inst in ORDER:
            if f"{o}_{inst}_data" not in tree:
                continue
            ds = dataset_from_arrays({v: tree[f"{o}_{inst}_{v}"] for v in ("time_unix", "data", "energy", "pitch_angle")})
            dsets[inst] = ds
            lines[inst] = get_timestamps_for_orbit(frame, o, inst, ds["times"])
        out.append((o, dsets, lines))
    return out


def _tree_shard(ctx, ys, zs, tree):
    from configurable_spectrograms_b200.fast.pipeline import ShardPlan

    shard = ShardPlan(ctx, ys, zs, instrument_order=ORDER)
    shard.first_orbit_index = 0
    for o, dsets, lines in tree:
        shard.add_orbit(o, dsets, lines)
    shard.upload()
    shard.collapse()
    return shard


def test_global_extrema_match_reference_json(ctx):
    """compute_global_extrema's numbers for the four (y, z) combos in CLI order (one shared cache),
    a fresh default-percentile run with mins, and the batch driver's cache -- all from the
    reference itself (tests/golden/extrema_tree.json)."""
    from configurable_spectrograms_b200.fast.extrema import extrema_from_shard

    tree = _tree()
    gold = load_json("extrema_tree.json")
    sequence = [(o, {i: True for i in dsets}) for o, dsets, _ in tree]
    state = {}
    for combo in gold["combos"]:
        shard = _tree_shard(ctx, combo["y"], combo["z"], tree)
        state = extrema_from_shard(shard, sequence, ORDER, combo["y"], combo["z"], state, max_percentile=99.0)
        assert state == combo["extrema"], (combo["y"], combo["z"])
    shard = _tree_shard(ctx, "linear", "linear", tree)
    st = extrema_from_shard(shard, sequence, ORDER, "linear", "linear", {}, max_percentile=95.0, compute_mins=True)
    assert st == gold["pool95_mins"]
    shard = _tree_shard(ctx, "linear", "log", tree)
    st = extrema_from_shard(shard, sequence, ORDER, "linear", "log", {}, max_percentile=99.0)
    assert st == gold["batch_extrema"]


def test_batch_step_matches_oracle_port(ctx, monkeypatch):
    """Every panel of every figure of both submissions of every orbit: bounds, indices, RGBA."""
    from configurable_spectrograms_b200.fast.pipeline import BatchStep, check_norm_status

    monkeypatch.setattr(CP, "NATIVE_LOG", False)
    tree = _tree()
    gold = load_json("extrema_tree.json")
    lut = _lut()
    sequence = [(o, {i: True for i in dsets}) for o, dsets, _ in tree]
    shard = _tree_shard(ctx, "linear", "log", tree)
    step = BatchStep(shard, sequence, max_percentile=99.0, lut259=lut, want_index=True)
    for _ in range(2):  # the second run re-uses the plan and only refreshes the z slots
        state = step.run({})
        step.finish()
        assert state == gold["batch_extrema"]
    b = shard.batch
    norms = b.norms()
    figs = iter(shard.figures)
    n_checked = 0

    def compare(fig, expected, what):
        nonlocal n_checked
        exp = iter(expected)
        need = fig.zoom is not None and fig.zoom_needed
        for row in fig.rows:
            pids = [row.full_panel] + ([row.zoom_panel] if need else [])
            for pid in pids:
                e = next(exp)
                if pid is None:
                    assert e is None, what
                    continue
                try:
                    check_norm_status(norms[pid], str(what))
                except ValueError:
                    assert e is None, what
                    continue
                assert e is not None, what
                assert np.array_equal(b.panel_index(pid), e[0]), (what, row.label)
                assert np.array_equal(b.panel_rgba(pid), e[1]), (what, row.label)
                n_checked += 1
        assert next(exp, "end") == "end", what

    with np.errstate(all="ignore"):
        for o, dsets, lines in tree:
            for extrema in (None, state):
                for inst in ORDER:
                    if inst not in dsets:
                        continue
                    ov = R.extrema_overrides(extrema, inst, "linear", "log")
                    for variant, kw in (("given", dict(y_min=ov[0], y_max=ov[1], z_min=ov[2], z_max=ov[3])), ("raw", {})):
                        fig = next(figs)
                        assert (fig.kind, fig.orbit, fig.instrument, fig.variant) == ("pitch-angle", o, inst, variant)
                        exp = CP.pitch_angle_grid(dsets[inst], lines.get(inst), "log", lut, **kw)
                        compare(fig, exp, (o, inst, variant, extrema is not None))
                first_lines = next((lines.get(i) for i in ORDER if i in dsets), None)
                for variant, ge in (("given", extrema), ("raw", None)):
                    fig = next(figs)
                    assert (fig.kind, fig.orbit, fig.variant) == ("instrument-grid", o, variant)
                    exp = CP.instrument_grid(dsets, first_lines, "log", lut, ge, "linear")
                    compare(fig, exp, (o, "grid", variant, extrema is not None))
    assert next(figs, None) is None
    assert n_checked > 200
