"""8-, 16- and 32-bit integer count cubes collapsed on the GPU at their stored width.

numpy sums such cubes in int64 / uint64 and computes everything after the sums in float64.  K1 reads the
stored type and writes float64 sums, which are exact, so every result equals the one of the same counts
widened to float64 on the host -- bit for bit.  Covered here: the public drop-in against ``np.nansum``
(value and dtype), every integer K1 path at its edges against the widened float64 path (sums and row
flags), the end-to-end plotting paths, the directory driver's staging width, and the mixed-dtype rules."""

import json
import os

import numpy as np
import pytest

from tests.helpers import dataset_from_arrays, load_json, load_npz

pytestmark = pytest.mark.gpu

INT_DTYPES = [np.int8, np.uint8, np.int16, np.uint16, np.int32, np.uint32]
# CDF type codes of the integer types the test CDF writer does not list (CDF_INT1, CDF_UINT2, CDF_UINT4)
EXTRA_CDF_TYPES = {np.dtype(np.int8): 1, np.dtype(np.uint16): 12, np.dtype(np.uint32): 14}
ORDER = ("ees", "eeb", "ies", "ieb")


@pytest.fixture(scope="module")
def ctx():
    from configurable_spectrograms_b200 import _lib

    return _lib.Context(0)


def _counts(rng, shape, dtype, extremes=False):
    info = np.iinfo(dtype)
    if extremes:
        return rng.choice(np.array([info.min, info.max, 0, 1], dtype=dtype), size=shape)
    return rng.integers(info.min, int(info.max) + 1, size=shape, dtype=dtype)


def _bits(rng, P, n_groups):
    """Group 0 empty, 1 every bin, 2 the last bin, the rest random (overlapping) subsets."""
    b = np.zeros(P, np.uint8)
    for g in range(n_groups):
        m = np.zeros(P, bool) if g == 0 else np.ones(P, bool) if g == 1 else (np.arange(P) == P - 1) if g == 2 else rng.random(P) < 0.5
        b |= (m.astype(np.uint8) << g).astype(np.uint8)
    return b


# ------------------------------------------------------------------ the drop-in collapse function


@pytest.mark.parametrize("dtype", INT_DTYPES, ids=lambda d: np.dtype(d).name)
def test_collapse_function_equals_numpy_in_value_and_dtype(dtype):
    from configurable_spectrograms_b200.constants import COLLAPSE_FUNCTION
    from configurable_spectrograms_b200.fast.constants import FAST_COLLAPSE_FUNCTION

    rng = np.random.default_rng(np.dtype(dtype).num)
    cases = {
        "extremes": _counts(rng, (17, 9, 13), dtype, extremes=True),
        "full_range": _counts(rng, (33, 64, 96), dtype),
        "P32768": _counts(rng, (2, 32768, 3), dtype, extremes=True),
        "tep_view": np.ascontiguousarray(_counts(rng, (20, 24, 40), dtype)).transpose(0, 2, 1),
        "slice": _counts(rng, (30, 20, 50), dtype)[::2, 1:19, 3:47],
    }
    info = np.iinfo(dtype)
    cases["all_max"] = np.full((5, 300, 8), info.max, dtype)
    cases["all_min"] = np.full((5, 300, 8), info.min, dtype)
    for name, cube in cases.items():
        for fn in (COLLAPSE_FUNCTION, FAST_COLLAPSE_FUNCTION):
            got, ref = fn(cube, axis=1), np.nansum(cube, axis=1)
            assert got.dtype == ref.dtype and np.array_equal(got, ref), name
    cube = _counts(rng, (6, 11, 14), dtype)
    for axis in (0, 2):
        got, ref = COLLAPSE_FUNCTION(cube, axis=axis), np.nansum(cube, axis=axis)
        assert got.dtype == ref.dtype and np.array_equal(got, ref), axis


# ----------------------------------------------------------------------------- K1 paths at edges

K1_T = (1, 3, 4, 5, 15, 16, 17, 800)
K1_E = (1, 3, 7, 8, 9, 96, 97, 200)
K1_P = (1, 7, 8, 64, 129, 300)


def _widened_pair(ctx, n_groups, files):
    """One float64 batch holding the integer cubes, and per file the (sums, flags) of the cube widened to
    float64 through the existing path, one file per batch; ``files``: (cube, bits) or
    (cube, bits, (device buffer, byte offset)) for a device-resident cube."""
    from configurable_spectrograms_b200.engine import Batch

    b_int, ref = Batch(ctx, np.float64, n_groups=n_groups), []
    for entry in files:
        cube, bits = entry[0], entry[1] if n_groups else None
        if len(entry) > 2:
            buf, off = entry[2]
            b_int.add_file(None, bits, shape=cube.shape, layout=0, device_ptr=buf.ptr + off, cube_dtype=cube.dtype)
        else:
            b_int.add_file(cube, bits)
        b = Batch(ctx, np.float64, n_groups=n_groups)
        b.add_file(cube.astype(np.float64), bits)
        b.upload_cubes()
        b.collapse()
        ref.append(([b.sums(0, g) for g in range(n_groups + 1)], b.flags(0)))
    b_int.upload_cubes()
    b_int.collapse()
    return b_int, ref


def _same_outputs(b_int, ref, n_groups):
    for f, (sums, flags) in enumerate(ref):
        for g in range(n_groups + 1):
            a = b_int.sums(f, g)
            assert a.dtype == np.float64 and np.array_equal(a.view(np.uint64), sums[g].view(np.uint64)), (f, g, b_int.files[f]["T"])
        assert np.array_equal(b_int.flags(f), flags), f


@pytest.mark.parametrize("n_groups", [0, 1, 4, 5, 7])
@pytest.mark.parametrize("dtype", INT_DTYPES, ids=lambda d: np.dtype(d).name)
def test_k1_integer_paths_at_edges(ctx, dtype, n_groups):
    from configurable_spectrograms_b200 import _lib

    rng = np.random.default_rng(100 * np.dtype(dtype).num + n_groups)
    files = []
    # every T, E and P of the edge lists, in C order (stream kernel where E * itemsize allows, else generic)
    # and as transposed (T,E,P) views (row kernel)
    for k, T in enumerate(K1_T):
        for j in range(3):
            E, P = K1_E[(k + 3 * j) % len(K1_E)], K1_P[(2 * k + j) % len(K1_P)]
            if T == 800 and E * P > 20000:
                E, P = 96, 64  # the FAST shape
            cube = _counts(rng, (T, P, E), dtype, extremes=(j == 1))
            files.append((cube, _bits(rng, P, n_groups)))
            tep = np.ascontiguousarray(cube.transpose(0, 2, 1)).transpose(0, 2, 1)
            files.append((tep, _bits(rng, P, n_groups)))
    # every stream-kernel block shape: 16 x (E * itemsize / 16) threads up to 512
    es = np.dtype(dtype).itemsize
    for E in sorted({16 // es, 96, 512 // es}):
        files.append((_counts(rng, (17, 9, E), dtype), _bits(rng, 9, n_groups)))
    b_int, ref = _widened_pair(ctx, n_groups, files)
    kernels = {key[:2] for key in b_int.d_files}
    assert (_lib.LAYOUT_TEP, _lib.K1_STREAM) in kernels and (_lib.LAYOUT_TPE, _lib.K1_GENERIC) in kernels
    if not (es == 1 and n_groups > 4):  # 8-bit cubes with more than 4 groups take the generic kernel
        assert (_lib.LAYOUT_TPE, _lib.K1_STREAM) in kernels
    assert all(len(key) == 4 and key[3] == _lib.INT_CUBE_CODES[np.dtype(dtype)] for key in b_int.d_files)
    _same_outputs(b_int, ref, n_groups)


@pytest.mark.parametrize("dtype", INT_DTYPES, ids=lambda d: np.dtype(d).name)
def test_k1_integer_cube_misaligned_by_one_element(ctx, dtype):
    from configurable_spectrograms_b200 import _lib

    rng = np.random.default_rng(7 + np.dtype(dtype).num)
    es = np.dtype(dtype).itemsize
    cubes = [_counts(rng, (17, 64, 96), dtype), _counts(rng, (5, 7, 9), dtype)]
    bufs = []
    for cube in cubes:
        buf = ctx.alloc(cube.nbytes + 256)
        buf.upload(cube, es)
        bufs.append(buf)
    files = [(c, _bits(rng, c.shape[1], 4), (buf, es)) for c, buf in zip(cubes, bufs)]
    b_int, ref = _widened_pair(ctx, 4, files)
    assert {key[:2] for key in b_int.d_files} == {(_lib.LAYOUT_TPE, _lib.K1_GENERIC)}
    _same_outputs(b_int, ref, 4)


def test_k1_mixed_dtypes_in_one_collapse_pending_call(ctx):
    from configurable_spectrograms_b200.engine import Batch

    rng = np.random.default_rng(11)
    b_int, b_ref = Batch(ctx, np.float64, n_groups=4), Batch(ctx, np.float64, n_groups=4)
    for dtype in (np.int16, np.uint32, np.float64, np.int16, np.uint32, np.float64):
        cube = _counts(rng, (37, 64, 96), dtype) if dtype != np.float64 else rng.poisson(5.0, (37, 64, 96)).astype(np.float64)
        bits = _bits(rng, 64, 4)
        b_int.add_file(cube, bits)
        b_ref.add_file(cube.astype(np.float64), bits)
    assert b_int.collapse_pending() == 6 and b_ref.collapse_pending() == 6
    ref = [([b_ref.sums(f, g) for g in range(5)], b_ref.flags(f)) for f in range(6)]
    _same_outputs(b_int, ref, 4)


# ------------------------------------------------------------------------------------ end to end


@pytest.mark.parametrize("dtype", [np.uint16, np.int32, np.uint8])
def test_make_spectrogram_integer_equals_float64(dtype):
    from configurable_spectrograms_b200.plotting import make_spectrogram

    rng = np.random.default_rng(5)
    times = 946684800.0 + 2.5 * np.arange(300)
    energy = np.linspace(4.0, 30000.0, 96)
    cube = rng.poisson(3.0, (300, 64, 96)).astype(dtype)
    for z in (None, "log"):
        for zoom in (None, (times[150], 120.0)):
            kw = dict(y_axis_max=40000, z_axis_scale_function=z)
            if zoom is not None:
                kw.update(center_timestamp=zoom[0], window_duration_seconds=zoom[1])
            ax_i, x_i = make_spectrogram(times, energy, cube, **kw)
            ax_f, x_f = make_spectrogram(times, energy, cube.astype(np.float64), **kw)
            im_i, im_f = ax_i.images[-1], ax_f.images[-1]
            assert np.array_equal(x_i, x_f)
            assert np.array_equal(im_i.rgba, im_f.rgba) and np.array_equal(im_i.index, im_f.index), (z, zoom)
            assert im_i.vmin == im_f.vmin and im_i.vmax == im_f.vmax, (z, zoom)


def _png_pixels(base):
    from configurable_spectrograms_b200 import png

    out = {}
    for dirpath, _dirs, fs in os.walk(base):
        for fn in fs:
            if fn.endswith(".png"):
                out[os.path.relpath(os.path.join(dirpath, fn), base)] = png.decode_rgba(open(os.path.join(dirpath, fn), "rb").read())
    return out


def test_generic_batch_plot_integer_equals_float64(tmp_path, monkeypatch):
    from configurable_spectrograms_b200.generic_batch import generic_batch_plot

    monkeypatch.chdir(tmp_path)
    rng = np.random.default_rng(9)
    times = 946684800.0 + 2.5 * np.arange(200)
    energy = np.linspace(4.0, 30000.0, 96)
    cubes = {f"item{k}": rng.poisson(2.0 + k, (200, 64, 96)).astype(dt) for k, dt in enumerate((np.uint16, np.int32, np.int8))}

    def run(widen):
        def build(item):
            data = cubes[item].astype(np.float64) if widen else cubes[item]
            return [{"x": times, "y": energy, "data": data, "label": item}]

        tag = "f64" if widen else "int"
        return generic_batch_plot(sorted(cubes), f"./out_{tag}", build, y_scale="linear", z_scale="log", max_workers=1,
                                  progress_json_path=f"./progress_{tag}.json", install_signal_handlers=False)

    run(False)
    run(True)
    got, ref = _png_pixels("./out_int"), _png_pixels("./out_f64")
    assert sorted(got) == sorted(ref) and len(got) == len(cubes)
    for name in ref:
        assert np.array_equal(got[name], ref[name]), name


def _write_cdf_tree(root, int_types):
    """The golden extrema tree as real CDF files whose ``data`` holds integer counts: ``int_types`` cycles
    through the files (None = CDF_DOUBLE).  Returns the cube bytes of every file as stored."""
    from tests import cdf_writer as W

    tree = load_npz("extrema_tree.npz")
    stems = sorted({k.rsplit("_", 1)[0] for k in tree if k.endswith("_relpath")})
    stored = 0
    for n, stem in enumerate(stems):
        path = os.path.join(root, str(tree[f"{stem}_relpath"]))
        os.makedirs(os.path.dirname(path), exist_ok=True)
        arrays = {v: tree[f"{stem}_{v}"] for v in ("time_unix", "data", "energy", "pitch_angle")}
        counts = np.rint(np.nan_to_num(np.asarray(arrays["data"], np.float64), nan=0.0, posinf=0.0, neginf=0.0))
        dt = int_types[n % len(int_types)]
        arrays["data"] = np.clip(counts, 0, 60000).astype(dt if dt is not None else np.float64)
        stored += arrays["data"].nbytes
        W.write_fast_cdf(path, arrays)
    with open(os.path.join(root, "FAST_Cusp_Indices.csv"), "w") as f:
        f.write(str(tree["csv"]))
    return stored


def test_directory_run_of_integer_cdf_files_equals_float64(tmp_path, monkeypatch):
    from configurable_spectrograms_b200 import _lib, cdf_utils, engine
    from configurable_spectrograms_b200.fast.batch_directory import FAST_plot_spectrograms_directory
    from tests import cdf_writer as W

    for dt, code in EXTRA_CDF_TYPES.items():
        monkeypatch.setitem(W.CDF_TYPES, dt, code)

    staged = []
    original = engine.Batch.collapse_pending

    def recording(self):
        for f in self.files[self._n_collapsed :]:
            if f["host"] is not None:
                staged.append((f["host"].dtype, f["host"].nbytes, f["T"] * f["P"] * f["E"]))
        return original(self)

    monkeypatch.setattr(engine.Batch, "collapse_pending", recording)
    results = {}
    for tag, types in (("int", (np.uint16, np.int32)), ("f64", (None,))):
        root = tmp_path / tag
        root.mkdir()
        stored = _write_cdf_tree(str(root), types)
        monkeypatch.chdir(root)
        cdf_utils.filtered_orbits_cache.clear()
        cdf_utils.orbit_column_cache.clear()
        staged.clear()
        res = FAST_plot_spectrograms_directory("./FAST_data", output_base="./FAST_plots/", y_scale="linear", z_scale="log",
                                               colormap="cividis", max_processing_percentile=99, max_workers=2,
                                               progress_json_path="./progress.json")
        ring = _lib.default_context().__dict__.get("_ring")
        assert ring is not None and ring.overflow_bytes == 0, tag
        # every cube went to the device at its stored width: no widening anywhere
        assert {np.dtype(d) for d, _, _ in staged} == {np.dtype(t or np.float64) for t in types}, tag
        assert sum(n for _, n, _ in staged) == stored, tag
        results[tag] = (sorted((r["orbit"], r["status"]) for r in res), json.load(open("./FAST_calculated_extrema.json")),
                        _png_pixels("./FAST_plots"))
    (st_i, ex_i, px_i), (st_f, ex_f, px_f) = results["int"], results["f64"]
    assert st_i == st_f and [s for _, s in st_i].count("ok") >= 1
    assert ex_i == ex_f
    assert sorted(px_i) == sorted(px_f) and px_i
    for name in px_f:
        assert np.array_equal(px_i[name], px_f[name]), name
    assert len(load_json("extrema_tree.json")["batch_pngs"]) == len(px_f)


# ------------------------------------------------------------------------------ mixed-dtype rules


def _dataset(rng, dtype):
    return dataset_from_arrays({"time_unix": 946684800.0 + 2.5 * np.arange(40), "data": rng.poisson(3.0, (40, 64, 96)).astype(dtype),
                                "energy": np.linspace(4.0, 30000.0, 96), "pitch_angle": np.linspace(0.0, 360.0, 64)})


def test_shard_dtype_rules_for_integer_files(ctx):
    from configurable_spectrograms_b200.fast.pipeline import ShardPlan

    rng = np.random.default_rng(3)
    sh = ShardPlan(ctx, dtype=np.float32)
    with pytest.raises(TypeError):
        sh.add_orbit(1, {"ees": _dataset(rng, np.int16)})
    sh = ShardPlan(ctx)
    d16, d64 = _dataset(rng, np.int16), _dataset(rng, np.float64)
    sh.add_orbit(1, {"ees": d16})
    sh.add_orbit(2, {"ees": d64})
    assert sh.batch.dtype == np.float64 and [f["dtype"] for f in sh.batch.files] == [np.dtype(np.int16), np.dtype(np.float64)]
    assert sh.collapse_pending() == 2
    for f, ds in enumerate((d16, d64)):
        assert np.array_equal(sh.batch.sums(f, 0), np.nansum(ds["data"], axis=1).astype(np.float64))
