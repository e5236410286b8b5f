"""GPU parity of the reference-shaped host API (plotting.*, fast.plotting.*, fast.process_orbit,
fast.batch_directory, generic_batch) against what the UNMODIFIED reference produced
(tests/golden/*, see tests/golden/make_golden.py)."""

import json
import os

import numpy as np
import pytest

from oracle import restate as R
from tests.helpers import dataset_from_arrays, load_json, load_npz, panels, same_float

pytestmark = pytest.mark.gpu

ORDER = ("ees", "eeb", "ies", "ieb")


def _index_of(ref):
    lut = R.lut_with_extremes(np.zeros((256, 4), np.uint8))
    return R.rasterise(ref, lut)[0]


def _check_axes(ax, ref, what):
    im = ax.images[-1]
    assert same_float(im.vmin, ref["vmin"]) and same_float(im.vmax, ref["vmax"]), (what, im.vmin, ref["vmin"], im.vmax, ref["vmax"])
    assert (im.norm == "log") == (ref["mode"] == "log"), what
    assert np.array_equal(im.index, _index_of(ref)), what
    assert np.array_equal(np.asarray(im.extent, dtype=np.float64), ref["extent"]), (what, im.extent, ref["extent"])


def test_generic_plot_spectrogram_set_matches_reference():
    from configurable_spectrograms_b200.plotting import generic_plot_spectrogram_set

    g = load_npz("generic_set.npz")
    for name in ("f32", "f64", "tep"):
        ds = dataset_from_arrays({k[len(name) + 4 :]: v for k, v in g.items() if k.startswith(f"in_{name}_")})
        for zs in ("linear", "log"):
            ref = panels(g, f"{name}_{zs}")
            fig, canvas = generic_plot_spectrogram_set(
                [{"x": ds["times"], "y": ds["energy"], "data": ds["data"], "label": name}], z_scale=zs, colormap="viridis", show=False
            )
            assert fig is not None and canvas.figure is fig and len(fig.axes) == 1
            _check_axes(fig.axes[0], ref[0], (name, zs))
            assert fig.axes[0].title == name
    ds = dataset_from_arrays({k[7:]: v for k, v in g.items() if k.startswith("in_f32_")})
    ref = panels(g, "f32_zoom_log")
    fig, _ = generic_plot_spectrogram_set(
        [{"x": ds["times"], "y": ds["energy"], "data": ds["data"]}], zoom_center=float(ds["times"][20]),
        zoom_window_seconds=50.0, z_scale="log", show=False,
    )
    _check_axes(fig.axes[0], ref[0], "zoom")
    assert generic_plot_spectrogram_set([]) == (None, None)


def test_make_spectrogram_conventions():
    """(None, None) when everything is filtered out; caller arrays are never modified; matplotlib's
    draw-time error for inverted bounds."""
    from configurable_spectrograms_b200.plotting import make_spectrogram

    rng = np.random.default_rng(3)
    times = 946684800.0 + 2.5 * np.arange(30)
    energy = np.linspace(4.0, 30000.0, 12)
    cube = rng.poisson(3.0, (30, 5, 12)).astype(np.float32)
    keep = cube.copy()
    assert make_spectrogram(times, energy, cube, y_axis_min=-10, y_axis_max=-5) == (None, None)
    ax, x_plot = make_spectrogram(times, energy, cube, y_axis_max=40000, vertical_lines_unix=[float(times[10])])
    assert ax is not None and len(x_plot) == 30 and np.array_equal(cube, keep)
    assert ax.images[-1].rgba.shape == (12, 30, 4)
    assert any(l["kind"] == "vline" for l in ax.lines)
    with pytest.raises(ValueError):  # LogNorm(vmin=50, vmax=10): matplotlib raises when the figure is drawn
        make_spectrogram(times, energy, cube, y_axis_max=40000, z_axis_scale_function="log", z_axis_min=50.0, z_axis_max=10.0)
    # inverted linear bounds fall back to the data range instead (reference plotting.py:313-315)
    ax, _ = make_spectrogram(times, energy, cube, y_axis_max=40000, z_axis_min=50.0, z_axis_max=10.0)
    with np.errstate(invalid="ignore"):
        m = np.nansum(cube, axis=1)
    assert ax.images[-1].vmin == float(m.min()) and ax.images[-1].vmax == float(m.max())
    # integer cubes go through float64 exactly like numpy
    ax, _ = make_spectrogram(times, energy, cube.astype(np.int64), y_axis_max=40000)
    ref = R.panel(times, energy, cube.astype(np.float64), x_min=None, x_max=None, y_max=40000)
    assert same_float(ax.images[-1].vmin, ref["vmin"]) and same_float(ax.images[-1].vmax, ref["vmax"])


def _write_tree(tmp_path):
    tree = load_npz("extrema_tree.npz")
    keys = sorted({k.rsplit("_", 1)[0] for k in tree if k.endswith("_relpath")})
    for stem in keys:
        rel = str(tree[f"{stem}_relpath"])
        path = tmp_path / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_bytes(b"")
        np.savez(str(path) + ".npz", **{v: tree[f"{stem}_{v}"] for v in ("time_unix", "data", "energy", "pitch_angle")})
    (tmp_path / "FAST_Cusp_Indices.csv").write_text(str(tree["csv"]))


def test_pitch_angle_and_instrument_grid_functions(tmp_path, monkeypatch):
    from configurable_spectrograms_b200 import cdf_utils
    from configurable_spectrograms_b200.fast.plotting import FAST_plot_instrument_grid, FAST_plot_pitch_angle_grid

    g = load_npz("pa_grid.npz")
    arrays = {k[3:]: v for k, v in g.items() if k.startswith("in_")}
    d = tmp_path / "one" / "2000" / "01"
    d.mkdir(parents=True)
    path = d / "fa_esa_l2_ees_20000101000000_777_v02.cdf"
    path.write_bytes(b"")
    np.savez(str(path) + ".npz", **arrays)
    import pandas as pd

    frame = pd.DataFrame({"Orbit Number": [777], "ees min Index": [80], "ees Max Index": [92]})
    cdf_utils.orbit_column_cache.clear()
    for zs in ("linear", "log"):
        for variant, kw in (("raw", {}), ("given", dict(y_min=0.0, y_max=2900.0, z_min=0.0, z_max=460.0))):
            ref = panels(g, f"{variant}_{zs}")
            fig, canvas = FAST_plot_pitch_angle_grid(str(path), filtered_orbits_df=frame, orbit_number=777,
                                                     scale_function_z=zs, show=False, colormap="turbo", **kw)
            assert fig is not None and len(fig.axes) == 8
            assert fig.suptitle_text == "Orbit 777 - Pitch Angle ees ESA Spectrograms"
            for k, ax in enumerate(fig.axes):  # row-major: (row, Full), (row, Zoomed)
                _check_axes(ax, ref[k], (zs, variant, k))
            assert fig.axes[0].title == "Full" and fig.axes[1].title == "Zoomed"
            assert [fig.axes[2 * i].yaxis.label.text for i in range(4)] == [
                "All\n(0, 360)", "Downgoing\n(0, 30), (330, 360)", "Upgoing\n(150, 210)", "Perpendicular\n(40, 140), (210, 330)"]
            out = tmp_path / f"pa_{zs}_{variant}.png"
            fig.savefig(str(out), dpi=200)
            assert out.stat().st_size > 1000
    # instrument grid
    g = load_npz("inst_grid.npz")
    ext = json.loads(str(g["extrema_json"]))
    files = {}
    for inst in ORDER:
        p = d / f"fa_esa_l2_{inst}_20000101000000_778_v02.cdf"
        p.write_bytes(b"")
        np.savez(str(p) + ".npz", **{k[len(inst) + 4 :]: v for k, v in g.items() if k.startswith(f"in_{inst}_")})
        files[inst] = str(p)
    cols = {"Orbit Number": [778]}
    for inst in ORDER:
        cols[f"{inst} min Index"], cols[f"{inst} Max Index"] = [40], [60]
    frame = pd.DataFrame(cols)
    cdf_utils.orbit_column_cache.clear()
    for tag, ge in (("raw", None), ("given", ext)):
        ref = panels(g, tag)
        fig, _ = FAST_plot_instrument_grid(files, filtered_orbits_df=frame, orbit_number=778, scale_function_y="linear",
                                           scale_function_z="log", show=False, colormap="viridis", global_extrema=ge)
        assert len(fig.axes) == len(ref)
        for k, ax in enumerate(fig.axes):
            _check_axes(ax, ref[k], (tag, k))
    assert FAST_plot_instrument_grid({}, show=False) == (None, None)


def test_directory_driver_matches_reference_outputs(tmp_path, monkeypatch):
    """FAST_plot_spectrograms_directory on the golden tree: statuses, PNG tree, extrema JSON and
    progress keys as the reference wrote them."""
    from configurable_spectrograms_b200 import cdf_utils, png
    from configurable_spectrograms_b200.fast.batch_directory import FAST_plot_spectrograms_directory

    _write_tree(tmp_path)
    monkeypatch.chdir(tmp_path)
    cdf_utils.filtered_orbits_cache.clear()
    cdf_utils.orbit_column_cache.clear()
    gold = load_json("extrema_tree.json")
    res = FAST_plot_spectrograms_directory(
        "./FAST_data", output_base="./FAST_plots/", y_scale="linear", z_scale="log", colormap="cividis",
        max_processing_percentile=99, max_workers=2, progress_json_path="./progress.json",
    )
    assert sorted((r["orbit"], r["status"]) for r in res) == [tuple(x) for x in gold["batch_status"]]
    pngs = []
    for dirpath, _dirs, fs in os.walk("./FAST_plots"):
        pngs += [os.path.relpath(os.path.join(dirpath, fn), "./FAST_plots") for fn in fs]
    assert sorted(pngs) == gold["batch_pngs"]
    assert json.load(open("./FAST_calculated_extrema.json")) == gold["batch_extrema"]
    prog = json.load(open("./progress.json"))
    assert set(prog) == set(gold["batch_progress"])
    assert prog["linear_log_error_plotting"] == [] and prog["orbit_linear_log_timed_out"] == []
    # (the reference's own last_orbit lags by its unflushed tail: 13004; ours records the true last orbit)
    assert prog["linear_log_last_orbit"] == 13005
    img = png.decode_rgba(open(os.path.join("./FAST_plots", gold["batch_pngs"][0]), "rb").read())
    assert img.ndim == 3 and img.shape[2] == 4 and img.shape[0] > 100
    # the driver's PNGs were composed and encoded on the device (K4); the per-orbit worker composes
    # on the host and encodes with zlib: same files, same pixels
    from configurable_spectrograms_b200.cdf_utils import load_filtered_orbits
    from configurable_spectrograms_b200.fast.orbit_discovery import discover_orbit_files
    from configurable_spectrograms_b200.fast.process_orbit import FAST_process_single_orbit

    files = discover_orbit_files("./FAST_data", ORDER)
    for orbit in (13000, 13002):
        r = FAST_process_single_orbit(orbit, files[orbit], load_filtered_orbits(), 6, "linear", "log", ORDER, "cividis",
                                      "./host_out/", global_extrema=gold["batch_extrema"])
        assert r["status"] == "ok"
        names = sorted(os.listdir(f"./host_out/2000/01/{orbit}"))
        assert names
        for name in names:
            dev_png = open(f"./FAST_plots/2000/01/{orbit}/{name}", "rb").read()
            host_png = open(f"./host_out/2000/01/{orbit}/{name}", "rb").read()
            assert np.array_equal(png.decode_rgba(dev_png), png.decode_rgba(host_png)), name
    # resume: nothing left to do, nothing re-plotted
    again = FAST_plot_spectrograms_directory(
        "./FAST_data", output_base="./FAST_plots/", y_scale="linear", z_scale="log", colormap="cividis",
        max_processing_percentile=99, max_workers=2, progress_json_path="./progress.json",
    )
    assert again == []


def _run_driver(**kw):
    from configurable_spectrograms_b200 import cdf_utils
    from configurable_spectrograms_b200.fast.batch_directory import FAST_plot_spectrograms_directory

    cdf_utils.filtered_orbits_cache.clear()
    cdf_utils.orbit_column_cache.clear()
    args = dict(output_base="./FAST_plots/", y_scale="linear", z_scale="log", colormap="cividis", max_processing_percentile=99,
                max_workers=2, progress_json_path="./progress.json")
    args.update(kw)
    return FAST_plot_spectrograms_directory("./FAST_data", **args)


def _png_tree(base="./FAST_plots"):
    out = []
    for dirpath, _dirs, fs in os.walk(base):
        out += [os.path.relpath(os.path.join(dirpath, fn), base) for fn in fs]
    return sorted(out)


def test_directory_driver_streams_in_small_chunks(tmp_path, monkeypatch):
    """The streaming pipeline with chunks of 2 orbits and pinned slots too small for a chunk (some cubes
    overflow into pageable memory): same statuses, PNG tree, extrema JSON and pixels as one big chunk."""
    from configurable_spectrograms_b200 import png

    _write_tree(tmp_path)
    monkeypatch.chdir(tmp_path)
    gold = load_json("extrema_tree.json")
    monkeypatch.setenv("CSG_CHUNK_ORBITS", "64")
    res = _run_driver(output_base="./big/")
    assert sorted((r["orbit"], r["status"]) for r in res) == [tuple(x) for x in gold["batch_status"]]
    os.remove("./progress.json"), os.remove("./FAST_calculated_extrema.json")
    monkeypatch.setenv("CSG_CHUNK_ORBITS", "2")
    monkeypatch.setenv("CSG_SLOT_BYTES", str(1 << 20))  # 1 MB: two to three of the small test cubes fit, the rest overflow
    flushes = []
    import configurable_spectrograms_b200.fast.batch_directory as BD

    real_write = BD._write_json
    monkeypatch.setattr(BD, "_write_json", lambda path, data: (flushes.append(data.get("linear_log_last_orbit")), real_write(path, data)))
    res = _run_driver(output_base="./small/", flush_batch_size=2)
    assert sorted((r["orbit"], r["status"]) for r in res) == [tuple(x) for x in gold["batch_status"]]
    assert _png_tree("./small") == _png_tree("./big") == gold["batch_pngs"]
    assert json.load(open("./FAST_calculated_extrema.json")) == gold["batch_extrema"]
    # progress reaches the disk chunk by chunk (an interrupt loses at most the chunk in flight)
    assert len(flushes) >= 3 and flushes[0] < flushes[-1] == 13005
    for name in gold["batch_pngs"][::7]:
        a = png.decode_rgba(open(os.path.join("./small", name), "rb").read())
        c = png.decode_rgba(open(os.path.join("./big", name), "rb").read())
        assert np.array_equal(a, c), name


def test_directory_driver_timeouts_and_retry(tmp_path, monkeypatch):
    """Soft timeouts after the fact + one retry (reference batch_directory.py:316-324,422-431,455-514)."""
    _write_tree(tmp_path)
    monkeypatch.chdir(tmp_path)
    res = _run_driver(orbit_timeout_seconds=0, retry_timeouts=False)
    assert res and all(r["status"] == "timeout" and r["timeout_type"] == "orbit" for r in res)
    prog = json.load(open("./progress.json"))
    assert prog["orbit_linear_log_timed_out"] == sorted({r["orbit"] for r in res})
    assert prog["linear_log_error_plotting"] == []
    # with the retry every timed-out orbit is re-run once through FAST_process_single_orbit (whose own soft
    # limits are generous here) and cleared from the list; results collapse to one entry per orbit
    os.remove("./progress.json")
    import configurable_spectrograms_b200.fast.process_orbit as PO

    real = PO.FAST_process_single_orbit
    calls = []

    def patient(*a, **k):  # the retry hands the same limits down; give the re-run a limit it can meet
        calls.append(a[0])
        assert k["orbit_timeout_seconds"] == 0 and k["global_extrema"] is None
        k["orbit_timeout_seconds"] = 600
        return real(*a, **k)

    monkeypatch.setattr(PO, "FAST_process_single_orbit", patient)
    res = _run_driver(orbit_timeout_seconds=0, retry_timeouts=True, output_base="./retry/")
    assert sorted(calls) == sorted({r["orbit"] for r in res})
    assert sorted(r["orbit"] for r in res) == sorted({r["orbit"] for r in res})
    assert all(r["status"] == "ok" for r in res), res
    prog = json.load(open("./progress.json"))
    assert prog["orbit_linear_log_timed_out"] == []


def test_directory_driver_float64_and_mixed_dtypes(tmp_path, monkeypatch):
    """A float64 archive is computed in float64 (numpy's sums, ranks and extrema depend on the dtype):
    extrema JSON against the oracle walk on the same float64 cubes.  One float64 file inside a float32
    archive is refused -- reported as an error of that orbit -- not cast."""
    tree = load_npz("extrema_tree.npz")
    keys = sorted({k.rsplit("_", 1)[0] for k in tree if k.endswith("_relpath")})

    def write(root, dtype_of):
        for stem in keys:
            path = root / str(tree[f"{stem}_relpath"])
            path.parent.mkdir(parents=True, exist_ok=True)
            path.write_bytes(b"")
            arrays = {v: tree[f"{stem}_{v}"] for v in ("time_unix", "data", "energy", "pitch_angle")}
            arrays["data"] = arrays["data"].astype(dtype_of(stem)) * (1.0 + 1e-9 if dtype_of(stem) == np.float64 else 1.0)
            np.savez(str(path) + ".npz", **arrays)
        (root / "FAST_Cusp_Indices.csv").write_text(str(tree["csv"]))

    f64 = tmp_path / "f64"
    f64.mkdir()
    write(f64, lambda stem: np.float64)
    monkeypatch.chdir(f64)
    res = _run_driver()
    assert res and all(r["status"] == "ok" for r in res)
    files = []
    orbits = sorted({int(k.split("_")[0]) for k in keys})
    for o in orbits:
        entry = {}
        for inst in ORDER:
            if f"{o}_{inst}_data" in tree:
                ds = dataset_from_arrays({v: tree[f"{o}_{inst}_{v}"] for v in ("time_unix", "data", "energy", "pitch_angle")})
                entry[inst] = (ds["energy"], ds["data"].astype(np.float64) * (1.0 + 1e-9))
        files.append((o, entry))
    want = R.global_extrema(files, ORDER, "linear", "log", state={}, max_percentile=99.0)
    got = json.load(open("./FAST_calculated_extrema.json"))
    assert got == want
    mixed = tmp_path / "mixed"
    mixed.mkdir()
    odd = next(k for k in keys if k.startswith("13002_ees"))
    write(mixed, lambda stem: np.float64 if stem == odd else np.float32)
    monkeypatch.chdir(mixed)
    res = _run_driver()
    by_orbit = {}
    for r in res:
        by_orbit.setdefault(r["orbit"], set()).add(r["status"])
    assert by_orbit[13002] == {"error"} and all(v == {"ok"} for o, v in by_orbit.items() if o != 13002)
    assert json.load(open("./progress.json"))["linear_log_error_plotting"] == [13002]


def test_directory_driver_reads_binary_cdf_files(tmp_path, monkeypatch):
    """The same golden tree stored as real CDF v3 files (gzip-compressed variables, network byte order) --
    read by the native reader straight into the pinned slots -- gives the reference's outputs."""
    from tests import cdf_writer as W

    tree = load_npz("extrema_tree.npz")
    keys = sorted({k.rsplit("_", 1)[0] for k in tree if k.endswith("_relpath")})
    for stem in keys:
        path = tmp_path / str(tree[f"{stem}_relpath"])
        path.parent.mkdir(parents=True, exist_ok=True)
        W.write_fast_cdf(path, {v: tree[f"{stem}_{v}"] for v in ("time_unix", "data", "energy", "pitch_angle")},
                         encoding=W.NETWORK, gzip=4, records_per_block=8)
    (tmp_path / "FAST_Cusp_Indices.csv").write_text(str(tree["csv"]))
    monkeypatch.chdir(tmp_path)
    gold = load_json("extrema_tree.json")
    res = _run_driver()
    assert sorted((r["orbit"], r["status"]) for r in res) == [tuple(x) for x in gold["batch_status"]]
    assert _png_tree() == gold["batch_pngs"]
    assert json.load(open("./FAST_calculated_extrema.json")) == gold["batch_extrema"]


def test_process_single_orbit_and_generic_batch(tmp_path, monkeypatch):
    from configurable_spectrograms_b200 import cdf_utils
    from configurable_spectrograms_b200.cdf_utils import load_fast_cdf_dataset, load_filtered_orbits
    from configurable_spectrograms_b200.fast.orbit_discovery import discover_orbit_files
    from configurable_spectrograms_b200.fast.process_orbit import FAST_process_single_orbit
    from configurable_spectrograms_b200.generic_batch import generic_batch_plot

    _write_tree(tmp_path)
    monkeypatch.chdir(tmp_path)
    cdf_utils.filtered_orbits_cache.clear()
    cdf_utils.orbit_column_cache.clear()
    gold = load_json("extrema_tree.json")
    frame = load_filtered_orbits()
    files = discover_orbit_files("./FAST_data", ORDER)
    for orbit in (13000, 13003):
        r = FAST_process_single_orbit(orbit, files[orbit], frame, 6, "linear", "log", ORDER, "cividis", "./out/",
                                      global_extrema=gold["batch_extrema"])
        assert r == {"orbit": orbit, "status": "ok", "errors": []}
        got = sorted(os.listdir(f"./out/2000/01/{orbit}"))
        assert got == sorted(os.path.basename(p) for p in gold["batch_pngs"] if f"/{orbit}/" in p)
    # generic batch: items are orbit numbers, one dataset per instrument present
    def build(item):
        return [
            {"x": ds["times"], "y": ds["energy"], "data": ds["data"], "label": inst}
            for inst, ds in ((i, load_fast_cdf_dataset(p)) for i, p in files[item].items())
        ] if item != 13001 else []

    res = generic_batch_plot([13000, 13001, 13002], "./generic_out", build, y_scale="linear", z_scale="log",
                             max_workers=2, progress_json_path="./generic_progress.json", install_signal_handlers=False)
    assert sorted(res) == [(13000, "ok"), (13001, "no_data"), (13002, "ok")]
    assert os.path.exists("./generic_out/13000/generic.png") and not os.path.exists("./generic_out/13001")
    prog = json.load(open("./generic_progress.json"))
    assert sorted(prog["completed_items"]) == ["13000", "13002"] and prog["no_data"] == ["13001"] and prog["schema_version"] == 1
    res = generic_batch_plot([13000, 13001, 13002], "./generic_out", build, max_workers=2,
                             progress_json_path="./generic_progress.json", install_signal_handlers=False)
    assert res == [(13001, "no_data")]  # completed items are skipped on resume


def test_two_gpu_extrema_and_directory_driver(tmp_path):
    """Ranks own contiguous orbit blocks; the NCCL exchange of bucket totals / surviving prefixes
    must reproduce the reference's extrema JSON and PNG tree (skipped on a single-GPU box)."""
    import subprocess
    import sys

    import torch

    n_ranks = int(os.environ.get("CSG_TEST_WORLD", "2"))  # 8: more ranks than the tree has orbits (empty shards)
    if torch.cuda.device_count() < n_ranks:
        pytest.skip(f"needs {n_ranks} GPUs")
    _write_tree(tmp_path)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n_ranks}", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(root, "tests", "multigpu_worker.py"), str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    if r.returncode != 0:  # the whole log in the test's temporary directory (the assertion shows its tails)
        (tmp_path / "multigpu_worker_failure.log").write_text(r.stdout + "\n=====\n" + r.stderr)
    assert r.returncode == 0 and f"MULTIGPU_OK world={n_ranks}" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
