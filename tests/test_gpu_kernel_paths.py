"""Every compiled body of K1 (collapse), K2a (region stats) and K3 (rasteriser), reached through
``engine.Batch`` and the C ABI at the shapes, alignments and values where such kernels go wrong:
partial tiles, pitch counts off the cp.async ring's 8-bin stages, every block size and group class of
the stream kernel, every output / addressing variant of the rasteriser and its persistent walk across
panels, cells placed exactly on colour boundaries, and the K2a walk's head / vector / tail split and
sampling threshold.  Seeded inputs; every comparison is bit for bit against numpy or
``oracle/restate.py`` (one documented exception: float64 ``log10`` at colour boundaries)."""

import numpy as np
import pytest

from tests.helpers import bits, same_bits, same_float

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from configurable_spectrograms_b200 import _lib

    return _lib.Context(0)


def _bits_from_masks(masks):
    b = np.zeros(len(masks[0]), dtype=np.uint8)
    for g, m in enumerate(masks):
        b |= (m.astype(np.uint8) << g).astype(np.uint8)
    return b


def _lut():
    from oracle import restate as R

    return R.lut_with_extremes(np.random.default_rng(99).integers(0, 256, (256, 4), dtype=np.uint8))


# ------------------------------------------------------------------------------------------------ K1


def _stream_block(dtype, E):
    """Threads per block of the stream kernel: 16 time rows x E / VEC energy chunks of 16 bytes."""
    return 16 * E // (16 // np.dtype(dtype).itemsize)


# Each (dtype, E) picks one block size, and the block size picks the body: up to 384 threads the
# cp.async ring, above it the register-staged loads.  Crossed with n_groups 0 / 3 / 4 / 7 (group
# classes 0, 4 -- with and without a dead group -- and CSG_MAX_GROUPS) these are all 30 instantiations.
K1_CASES = [(np.float32, E) for E in (64, 96, 128, 192, 256)] + [(np.float64, E) for E in (32, 48, 64, 96, 128)]
K1_BLOCKS = [256, 384, 512, 768, 1024]
for _dt in (np.float32, np.float64):
    assert sorted(_stream_block(d, E) for d, E in K1_CASES if d is _dt) == K1_BLOCKS
K1_T = (1, 15, 16, 17, 33)  # partial 16-row tiles; several files per launch (find_file)
K1_P = (1, 7, 8, 9, 16, 17, 64)  # the ring's 8-bin stages and refills, runs ending off a stage boundary


def _k1_masks(rng, P, n_groups):
    """Group 0 holds every bin (copied from the total), 1 none, 2 only the last bin, the rest random."""
    masks = []
    for g in range(n_groups):
        if g == 0:
            m = np.ones(P, bool)
        elif g == 1:
            m = np.zeros(P, bool)
        elif g == 2:
            m = np.arange(P) == P - 1
        else:
            m = rng.random(P) < 0.5
        masks.append(m)
    return masks


def _k1_cube(rng, T, P, E, dtype):
    c = rng.gamma(2.0, 3.0, (T, P, E)).astype(dtype)
    c[rng.random(c.shape) < 0.05] = np.nan
    c[rng.random(c.shape) < 0.02] = -0.0
    n_inf = max(1, c.size // 400)
    c.flat[rng.integers(0, c.size, n_inf)] = np.inf
    c.flat[rng.integers(0, c.size, n_inf)] = -np.inf
    if P >= 2:
        # +1e30 ... small values ... -1e30 down one (t, e) column: the sum keeps only what follows the
        # cancellation, so any order other than the ascending-p chain changes the bits
        n = max(1, T * E // 6)
        t, e = rng.integers(0, T, n), rng.integers(0, E, n)
        p1 = rng.integers(0, P - 1, n)
        p2 = rng.integers(p1 + 1, P)
        c[t, p1, e] = 1e30
        c[t, p2, e] = -1e30
    if T >= 3:
        c[1, :, : E // 2] = -0.0  # sums of -0.0 only: the chain is seeded with +0.0
        c[T // 2] = np.nan  # a time row without a single sample
    return c


def _check_collapse(b, f, cube, masks):
    with np.errstate(invalid="ignore", over="ignore"):
        assert same_bits(b.sums(f, 0), np.nansum(cube, axis=1), zero_sign_insensitive=False), ("total", cube.shape)
        for g, m in enumerate(masks):
            ref = np.nansum(cube[:, m, :], axis=1)
            assert same_bits(b.sums(f, g + 1), ref, zero_sign_insensitive=False), (g, cube.shape)
    nn = ~np.isnan(cube)
    want = nn.any(axis=(1, 2)).astype(np.uint8)
    for g, m in enumerate(masks):
        want |= (nn[:, m, :].any(axis=(1, 2)).astype(np.uint8) << (g + 1)).astype(np.uint8)
    assert np.array_equal(b.flags(f), want), cube.shape


@pytest.mark.parametrize("n_groups", [0, 3, 4, 7])
@pytest.mark.parametrize("dtype,E", K1_CASES, ids=[f"{np.dtype(d).name}-E{E}" for d, E in K1_CASES])
def test_collapse_stream_kernel_every_instantiation(ctx, dtype, E, n_groups):
    from configurable_spectrograms_b200 import _lib
    from configurable_spectrograms_b200.engine import Batch

    assert _stream_block(dtype, E) in K1_BLOCKS
    rng = np.random.default_rng(1000 * E + 10 * n_groups + np.dtype(dtype).itemsize)
    b = Batch(ctx, dtype, n_groups=n_groups)
    files = []
    for T in K1_T:
        for P in K1_P:
            cube = _k1_cube(rng, T, P, E, dtype)
            masks = _k1_masks(rng, P, n_groups)
            files.append((b.add_file(cube, _bits_from_masks(masks) if n_groups else None), cube, masks))
    b.upload_cubes()
    b.collapse()
    for f, cube, _ in files:
        d = b.files[f]
        kern = ctx.lib.csg_collapse_kernel_for(d["T"], d["P"], E, b.code, d["layout"], d["device_ptr"], n_groups)
        assert kern == _lib.K1_STREAM, ("fell back to the generic kernel", cube.shape)
    assert set(b.d_files) == {(_lib.LAYOUT_TPE, _lib.K1_STREAM, E)}, "every file in one stream-kernel launch"
    for f, cube, masks in files:
        _check_collapse(b, f, cube, masks)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_collapse_mixed_block_shapes_in_one_batch(ctx, dtype):
    """E = 64 and E = 96 (two stream-kernel block shapes) and E = 95 (the generic kernel) in one batch:
    three launches that share the sums / flags buffers, each file right."""
    from configurable_spectrograms_b200 import _lib
    from configurable_spectrograms_b200.engine import Batch

    rng = np.random.default_rng(41)
    b = Batch(ctx, dtype, n_groups=4)
    files = []
    for E in (64, 95, 96, 64, 95, 96):
        T, P = int(rng.integers(1, 40)), int(rng.choice(K1_P))
        cube = _k1_cube(rng, T, P, E, dtype)
        masks = _k1_masks(rng, P, 4)
        files.append((b.add_file(cube, _bits_from_masks(masks)), cube, masks))
    b.upload_cubes()
    b.collapse()
    assert set(b.d_files) == {
        (_lib.LAYOUT_TPE, _lib.K1_STREAM, 64),
        (_lib.LAYOUT_TPE, _lib.K1_STREAM, 96),
        (_lib.LAYOUT_TPE, _lib.K1_GENERIC, 0),
    }
    for f, cube, masks in files:
        _check_collapse(b, f, cube, masks)


def test_collapse_host_seven_groups(ctx):
    from configurable_spectrograms_b200.engine import collapse_host

    rng = np.random.default_rng(42)
    for dtype, E in ((np.float32, 96), (np.float64, 48)):
        cube = _k1_cube(rng, 33, 17, E, dtype)
        masks = _k1_masks(rng, 17, 7)
        sums, fl = collapse_host(cube, _bits_from_masks(masks), n_groups=7, ctx=ctx)
        with np.errstate(invalid="ignore", over="ignore"):
            assert same_bits(sums[0], np.nansum(cube, axis=1), zero_sign_insensitive=False)
            for g, m in enumerate(masks):
                assert same_bits(sums[g + 1], np.nansum(cube[:, m, :], axis=1), zero_sign_insensitive=False), g
        nn = ~np.isnan(cube)
        want = nn.any(axis=(1, 2)).astype(np.uint8)
        for g, m in enumerate(masks):
            want |= (nn[:, m, :].any(axis=(1, 2)).astype(np.uint8) << (g + 1)).astype(np.uint8)
        assert np.array_equal(fl, want)


# ------------------------------------------------------------------------------- matrices for K2a / K3


def _matrix_batch(ctx, mats, dtype):
    """A batch whose collapsed matrices are exactly ``mats`` (each (T, E); -0.0 becomes +0.0): the two
    pitch bins of a cell hold (value, 0), or (+inf, -inf) where the value is NaN."""
    from configurable_spectrograms_b200.engine import Batch

    b = Batch(ctx, dtype, 0)
    ids = []
    for M in mats:
        M = np.asarray(M, dtype)
        nan = np.isnan(M)
        cube = np.zeros((M.shape[0], 2, M.shape[1]), dtype)
        cube[:, 0, :] = np.where(nan, np.inf, M)
        cube[:, 1, :] = np.where(nan, -np.inf, 0)
        ids.append(b.add_file(cube))
    b.upload_cubes()
    b.collapse()
    for f, M in zip(ids, mats):
        assert same_bits(b.sums(f), np.asarray(M, dtype))
    return b, ids


def _random_matrix(rng, T, E, dtype):
    M = (rng.gamma(1.5, 40.0, (T, E)) * (rng.random((T, E)) < 0.9)).astype(dtype)  # zeros too
    M[rng.random((T, E)) < 0.03] = np.nan
    M[rng.random((T, E)) < 0.01] = np.inf
    M[rng.random((T, E)) < 0.01] = -np.inf
    M[rng.random((T, E)) < 0.02] *= -1
    M[M == 0] = 0  # +0.0 only: the collapse seeds every sum with +0.0
    return M


# ----------------------------------------------------------------------------------------------- K3


def _oracle_panel(Mr, log, z_min, z_max):
    """make_spectrogram's z handling on a region matrix (ne, nt): percentile bounds of the region itself."""
    from oracle import restate as R

    with np.errstate(invalid="ignore"), np.testing.suppress_warnings() as sup:
        sup.filter(RuntimeWarning)
        zmin, zmax = R.compute_percentile_bounds(Mr, 1, 99, z_min, z_max)
        fp = Mr[np.isfinite(Mr) & (Mr > 0)]
        safe = np.nanmin(fp) if fp.size else 1e-10
        return R.clamp_for_imshow(Mr, "log" if log else "linear", zmin, zmax, safe)


def _oracle_raster(ref, lut):
    """(index, rgba) of the oracle, or None where matplotlib raises (vmin > vmax, invalid log bounds)."""
    from oracle import restate as R

    try:
        with np.errstate(all="ignore"):
            return R.rasterise(ref, lut)
    except ValueError:
        return None


def _check_panels(b, specs, lut, rgba=None, index=None):
    """Every panel's bounds and planes against the oracle; ``specs[p] = (region matrix, log, z_min, z_max)``.
    ``rgba`` / ``index``: whole output planes downloaded once (None: that plane is not checked)."""
    norms = b.norms()
    n_ok = 0
    for p, (Mr, log, zlo, zhi) in enumerate(specs):
        ref = _oracle_panel(Mr, log, zlo, zhi)
        nm = norms[p]
        assert same_float(nm["vmin"], ref["vmin"]) and same_float(nm["vmax"], ref["vmax"]), (p, nm, ref["vmin"], ref["vmax"])
        out = _oracle_raster(ref, lut)
        if out is None:
            assert nm["status"] != 0, p
            continue
        assert nm["status"] == 0, p
        ne, nt = b.panel_shape(p)
        off = b.panel_offset(p)
        if index is not None:
            assert np.array_equal(index[off : off + ne * nt].reshape(ne, nt), out[0]), (p, ne, nt, log, zlo, zhi)
        if rgba is not None:
            assert np.array_equal(rgba[4 * off : 4 * (off + ne * nt)].reshape(ne, nt, 4), out[1]), (p, ne, nt, log, zlo, zhi)
        n_ok += 1
    return n_ok


def _poison(b):
    for buf in (b.d_rgba, b.d_index):
        if buf is not None:
            b.ctx._check(b.ctx.lib.csg_memset(b.ctx.handle, buf.ptr, 0xA5, buf.nbytes))


K3_BOUNDS = [(None, None), (5.0, 300.0), (None, 50.0), (0.0, None), (-20.0, 90.0)]


@pytest.mark.parametrize("addressing", ["t0_aligned", "t0_offset", "rows"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("scale", ["linear", "log"])
def test_rasterise_every_output_and_addressing_variant(ctx, scale, dtype, addressing):
    """RGBA only (the batch path's own 128-bit-store body), index only, and both: each against the oracle,
    and the RGBA-only plane equal to the RGBA of the both-outputs run; small panels whose groups of four
    pixels straddle image rows, and one panel of three chunks with a partial last one."""
    rng = np.random.default_rng({"linear": 1, "log": 2}[scale] * 100 + np.dtype(dtype).itemsize * 10 + len(addressing))
    T, E = 400, 96
    M = _random_matrix(rng, T, E, dtype)
    b, (f,) = _matrix_batch(ctx, [M], dtype)
    log = scale == "log"
    shapes = [(ne, nt) for ne in (1, 3, 74) for nt in (1, 2, 3, 5, 64, 65)] + [(74, 300)]
    specs = []
    for k, (ne, nt) in enumerate(shapes):
        cols = rng.choice(E, ne, replace=False)
        if addressing == "rows":
            rows = np.sort(rng.choice(T, nt, replace=False))
            if nt > 1 and rows[-1] - rows[0] == nt - 1:  # a gap: a contiguous list is planned as a time range
                if rows[-1] + 1 < T:
                    rows[-1] += 1
                else:
                    rows[0] -= 1
            r = b.add_region(f, 0, cols, rows=rows, want_pct=True)
        else:
            t0 = 4 * int(rng.integers(0, (T - nt) // 4)) + (0 if addressing == "t0_aligned" else 1 + k % 3)
            rows = np.arange(t0, t0 + nt)
            r = b.add_region(f, 0, cols, t0=t0, nt=nt, want_pct=True)
        zlo, zhi = K3_BOUNDS[k % len(K3_BOUNDS)]
        b.add_panel(r, -1, log, zlo, zhi)
        specs.append((M[np.ix_(rows, cols)].T, log, zlo, zhi))
    assert b._raster_blocks > len(shapes)  # the last panel spans several chunks
    lut = _lut()
    b.upload_tables()
    b.run_stats()
    b.prepare()
    b.set_lut(lut)
    b.rasterise()  # allocates both planes
    planes = {}
    for want_rgba, want_index in ((True, False), (False, True), (True, True)):
        _poison(b)
        b.rasterise(want_rgba=want_rgba, want_index=want_index)
        planes[(want_rgba, want_index)] = (b.all_rgba(), b.all_index())
    rgba_only, untouched_index = planes[(True, False)]
    untouched_rgba, index_only = planes[(False, True)]
    both_rgba, both_index = planes[(True, True)]
    assert (untouched_index == 0xA5A5).all(), "an RGBA-only run wrote the index plane"
    assert (untouched_rgba == 0xA5).all(), "an index-only run wrote the RGBA plane"
    assert np.array_equal(rgba_only, both_rgba)
    assert np.array_equal(index_only, both_index)
    n_ok = _check_panels(b, specs, lut, rgba=rgba_only, index=index_only)
    assert n_ok >= len(shapes) // 2


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_rasterise_persistent_blocks_walk_many_panels(ctx, dtype):
    """More chunks than the persistent grid holds, so every block walks several chunks of several panels and
    reloads the threshold table at each change; ordinary panels interleaved with degenerate ones (vmin ==
    vmax, NaN bounds) and with panels in error (vmin > vmax) that are skipped.  The same planes, equal to
    the oracle, with csg_rasterise_blocks_per_sm at 0 (as many as fit), 1 and 2."""
    rng = np.random.default_rng(51 + np.dtype(dtype).itemsize)
    _name, sms, _mem = ctx.device_info()
    per_sm = 3 if dtype == np.float32 else 2  # what fits: csg_rasterise's default
    T, E = 600, 96
    M = _random_matrix(rng, T, E, dtype)
    M[:, E - 1] = np.nan  # one energy row of NaN cells only: linear bounds are NaN
    b, (f,) = _matrix_batch(ctx, [M], dtype)
    specs = []
    # (kind, log, z_min, z_max): log (7, 7) is degenerate (vmin == vmax), log (50, 10) an error (vmin > vmax);
    # a linear panel over NaN cells only has NaN bounds; "wide" panels span two chunks
    kinds = [("plain", False, None, None), ("plain", True, None, None), ("plain", True, 7.0, 7.0),
             ("plain", False, 5.0, None), ("nan", False, None, None), ("plain", True, 0.0, 300.0),
             ("plain", True, 50.0, 10.0), ("wide", True, None, None), ("wide", False, None, None)]
    k = 0
    while b._raster_blocks <= 4 * sms * per_sm:
        kind, log, zlo, zhi = kinds[k % len(kinds)]
        k += 1
        ne = 40 if kind == "wide" else int(rng.integers(1, 12))
        nt = int(rng.integers(200, 300))
        t0 = int(rng.integers(0, T - nt))
        cols = np.full(ne, E - 1) if kind == "nan" else rng.choice(E - 1, ne, replace=False)
        r = b.add_region(f, 0, cols, t0=t0, nt=nt, want_pct=True)
        b.add_panel(r, -1, log, zlo, zhi)
        specs.append((M[t0 : t0 + nt][:, cols].T, log, zlo, zhi))
    n_chunks = b._raster_blocks
    lut = _lut()
    b.upload_tables()
    b.run_stats()
    b.prepare()
    b.set_lut(lut)
    norms = b.norms()
    assert (norms["degenerate"] == 1).any() and (norms["degenerate"] == 2).any() and (norms["status"] != 0).any()
    runs = []
    try:
        for setting in (0, 1, 2):
            grid = sms * (min(setting, per_sm) if setting else per_sm)
            assert n_chunks > 3 * grid, (n_chunks, grid)  # every block walks several chunks
            ctx._check(ctx.lib.csg_rasterise_blocks_per_sm(ctx.handle, setting))
            b.rasterise()
            _poison(b)
            b.rasterise()
            runs.append((b.all_rgba(), b.all_index()))
    finally:
        ctx._check(ctx.lib.csg_rasterise_blocks_per_sm(ctx.handle, 0))
    for rgba, index in runs[1:]:
        assert np.array_equal(rgba, runs[0][0]) and np.array_equal(index, runs[0][1])
    n_ok = _check_panels(b, specs, lut, rgba=runs[0][0], index=runs[0][1])
    assert n_ok >= len(specs) // 2


def _bound(z):
    """The value a z bound (a float, None or a ZSlot) holds: None means "take the percentile"."""
    return None if z is None or np.isnan(float(z)) else float(z)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_rasterise_split_by_z_slots_equals_one_call(ctx, dtype):
    """Panels whose bounds live in z slots run as part 1, after the slot-free panels of part 0, at a nonzero
    chunk offset: prepare / rasterise of part 0 then part 1 give the planes and norms of one call, and every
    panel equals the oracle with the slots' values as its bounds."""
    rng = np.random.default_rng(61 + np.dtype(dtype).itemsize)
    T, E = 500, 96
    M = _random_matrix(rng, T, E, dtype)
    b, (f,) = _matrix_batch(ctx, [M], dtype)
    slots = [b.zslot(None), b.zslot(250.0), b.zslot(2.0), b.zslot(0.0)]
    specs = []
    for k in range(24):
        ne, nt = int(rng.integers(1, 40)), int(rng.integers(1, 400))
        t0 = int(rng.integers(0, T - nt + 1))
        cols = rng.choice(E, ne, replace=False)
        log = k % 3 == 1
        if k % 2:  # interleaved: the device order (slot-free panels first) differs from the logical one
            zlo, zhi = slots[(k // 2) % 4], slots[(k // 2 + 1) % 4]
        else:
            zlo, zhi = K3_BOUNDS[k % len(K3_BOUNDS)]
        r = b.add_region(f, 0, cols, t0=t0, nt=nt, want_pct=True)
        b.add_panel(r, -1, log, zlo, zhi)
        specs.append((M[t0 : t0 + nt][:, cols].T, log, _bound(zlo), _bound(zhi)))
    lut = _lut()
    b.upload_tables()
    b.run_stats()
    b.set_lut(lut)
    assert 0 < b._n_free < b.n_panels and 0 < b._blocks_free < b._raster_blocks
    b.prepare(part=0)
    b.rasterise(part=0)  # allocates both planes
    _poison(b)
    b.rasterise(part=0)
    b.prepare(part=1)
    b.rasterise(part=1)
    split = (b.norms(), b.all_rgba(), b.all_index())
    _poison(b)
    b.d_norms.zero()
    b.prepare()
    b.rasterise()
    whole = (b.norms(), b.all_rgba(), b.all_index())
    assert np.array_equal(split[0].view(np.uint8), whole[0].view(np.uint8))
    assert np.array_equal(split[1], whole[1]) and np.array_equal(split[2], whole[2])
    n_ok = _check_panels(b, specs, lut, rgba=split[1], index=split[2])
    assert n_ok >= len(specs) // 2


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_rasterise_linear_panels_with_infinite_range(ctx, dtype):
    """Linear panels whose vmax - vmin is infinite: vmin = -inf (every cell "bad"), vmax = +inf (index 0,
    "bad" where v - vmin overflows), and finite bounds whose difference overflows float64.  Infinite bounds
    also come out of percentiles of regions with a few percent of infinite cells.  The colour is no monotone step function of the value there; the threshold search
    used to gallop forever on such a float32 panel."""
    rng = np.random.default_rng(81 + np.dtype(dtype).itemsize)
    D = np.dtype(dtype).type
    big = D(np.finfo(dtype).max) / D(1.1)
    T, E = 200, 12
    M = _random_matrix(rng, T, E, dtype)
    M[rng.random((T, E)) < 0.05] = -np.inf
    M[:, 0:4][rng.random((T, 4)) < 0.1] = np.inf
    M[:, 4:8] = np.abs(np.nan_to_num(M[:, 4:8], nan=3.0, posinf=5.0, neginf=7.0))
    M[:, 4:8][rng.random((T, 4)) < 0.1] = np.inf
    M[::3, 5] = big  # v - vmin overflows to inf
    M[1::3, 6] = -big / D(4)
    b, (f,) = _matrix_batch(ctx, [M], dtype)
    cases = [  # (cols, z_min, z_max): an infinite bound falls back to nanmin / nanmax of the clamped matrix
        (np.arange(8, 12), -np.inf, None),  # vmin = -inf (NaN and -inf cells)
        (np.arange(0, 4), -np.inf, np.inf),  # both infinite
        (np.arange(4, 8), None, np.inf),  # finite vmin, vmax = +inf
        (np.arange(4, 8), -1e308, 1e308),  # finite bounds, infinite difference
        (np.arange(0, 12), -1e308, 1e308),
    ]
    specs = []
    for cols, zlo, zhi in cases:
        r = b.add_region(f, 0, cols, want_pct=True)
        b.add_panel(r, -1, False, zlo, zhi)
        specs.append((M[:, cols].T, False, zlo, zhi))
    lut = _lut()
    b.upload_tables()
    b.run_stats()
    b.prepare()
    b.set_lut(lut)
    b.rasterise()
    norms = b.norms()
    assert np.isneginf(norms["vmin"][:2]).all() and np.isfinite(norms["vmin"][2]) and np.isposinf(norms["vmax"][2])
    with np.errstate(over="ignore"):
        assert not np.isfinite(norms["vmax"] - norms["vmin"]).any()
    assert _check_panels(b, specs, lut, rgba=b.all_rgba(), index=b.all_index()) == len(cases)
    idx = b.all_index()
    off, (ne, nt) = b.panel_offset(2), b.panel_shape(2)
    assert {0, 258} <= set(np.unique(idx[off : off + ne * nt]))  # both colours of the infinite range occur


# ---- colour boundaries: the 257-entry threshold table and the guess-and-verify lookup


def _keys(a):
    """The device's ordered keys (Key<T>): unsigned integers in the order of the float values."""
    u = bits(a)
    sign = u.dtype.type(1) << u.dtype.type(8 * u.itemsize - 1)
    return np.where(u & sign, ~u, u | sign)


def _from_keys(k, dtype):
    sign = k.dtype.type(1) << k.dtype.type(8 * k.itemsize - 1)
    return np.where(k & sign, k & ~sign, ~k).astype(k.dtype).view(dtype)


def _codes(v, vmin, vmax, log):
    """The oracle's monotone colour code of substituted values: under -1, colours 0..255, over 256."""
    from oracle import restate as R

    x = R.lognorm(v, vmin, vmax) if log else R.normalize(v, vmin, vmax)
    idx = R.colormap_index(x).astype(np.int64)
    assert not (idx == R.I_BAD).any()
    return np.where(idx == R.I_UNDER, -1, np.where(idx == R.I_OVER, 256, idx))


def _host_thresholds(dtype, vmin, vmax, log):
    """thr[k] = the smallest value (of the substituted domain: finite positives for log, [-inf, inf] for
    linear) whose oracle code reaches k, by bisection over the ordered bit patterns; +inf where none does."""
    D = np.dtype(dtype)
    one = lambda v: _keys(np.array([v], D))[0]  # noqa: E731
    dom_lo, dom_hi = (one(0.0) + 1, one(np.inf) - 1) if log else (one(-np.inf), one(np.inf))
    k = np.arange(257)
    code = lambda key: _codes(_from_keys(key, D), vmin, vmax, log)  # noqa: E731
    lo = np.full(257, dom_lo, dom_lo.dtype)
    hi = np.full(257, dom_hi, dom_hi.dtype)
    at_lo = code(lo) >= k
    found = code(hi) >= k
    with np.errstate(over="ignore"):
        while True:  # invariant where active: code(lo) < k <= code(hi)
            active = found & ~at_lo & (hi - lo > 1)
            if not active.any():
                break
            mid = lo + (hi - lo) // 2
            up = code(mid) >= k
            hi = np.where(active & up, mid, hi)
            lo = np.where(active & ~up, mid, lo)
    thr = _from_keys(np.where(at_lo, lo, hi), D).copy()
    thr[~found] = np.inf
    return thr


def _boundary_panels(dtype):
    """(log, z_min, z_max) with awkward bounds: one-ulp ranges, a range over most of the dtype (the in-place
    subtraction overflows to inf), vmin clamped to 1e-10 on log panels."""
    D = np.dtype(dtype).type
    ulp = float(np.nextafter(D(100.0), D(np.inf)))
    huge = 3.0e38 if D is np.float32 else 8.0e307
    return [
        (False, 3.0, 4000.0),
        (False, -50.0, 70.0),
        (False, 100.0, ulp),
        (False, -huge, huge),
        (True, 1.0, 5000.0),
        (True, 100.0, ulp),
        (True, 0.0, 1.0e4),  # max(0, safe_vmin, 1e-10) = 1e-10: the region holds smaller positives
        (True, 1e-30, 1e30),
    ]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_threshold_table_and_lookup_at_colour_boundaries(ctx, dtype):
    """The device's 257 thresholds equal the oracle's own (smallest value whose code reaches k), and a
    matrix of every threshold and its predecessor is coloured like the oracle.  Float64 log panels are the
    exception: CUDA's double log10 and the host's np.log10 may differ in the last bit, so there the table is
    not compared and a boundary cell may take the oracle's index or its neighbour (never "bad" for one and
    not the other).  A float64 log panel one ulp wide has log10(vmin) == log10(vmax): LogNorm masks every
    cell, and so must the rasteriser."""
    from oracle import restate as R

    D = np.dtype(dtype)
    panels = _boundary_panels(dtype)
    mats, expect = [], []
    tiny = np.array([np.nextafter(D.type(0), D.type(1))], D)  # below every vmin: safe_vmin never raises it
    for log, zlo, zhi in panels:
        vmin = max(zlo, 1e-10) if log else zlo
        all_bad = log and np.log10(vmin) == np.log10(zhi)
        if all_bad:  # no thresholds: cells at and around the bounds
            thr = None
            near = np.array([vmin, zhi, 1.0, 1e4], D)
            with np.errstate(over="ignore"):
                vals = np.concatenate([near, np.nextafter(near, D.type(-np.inf)), np.nextafter(near, D.type(np.inf)), tiny])
        else:
            thr = _host_thresholds(dtype, vmin, zhi, log)
            with np.errstate(over="ignore"):
                vals = np.concatenate([thr, np.nextafter(thr, D.type(-np.inf)), tiny])
        n = (len(vals) + 3) // 4 * 4
        vals = np.concatenate([vals, np.full(n - len(vals), vals[0], D)])
        mats.append(vals.reshape(-1, 4))  # (T, 4): every cell of the panel
        expect.append((vmin, thr))
    assert any(t is None for _, t in expect) == (D == np.float64)
    b, ids = _matrix_batch(ctx, mats, dtype)
    specs = []
    for (log, zlo, zhi), f, Mx in zip(panels, ids, mats):
        r = b.add_region(f, 0, np.arange(4), want_pct=True)
        b.add_panel(r, -1, log, zlo, zhi)
        specs.append(Mx.T)
    lut = _lut()
    b.upload_tables()
    b.run_stats()
    b.prepare()
    b.set_lut(lut)
    b.rasterise()
    norms = b.norms()
    n = b.n_panels
    dev = b.d_thr.download(D, n * 264).reshape(n, 264)[:, :257]
    table = b.by_panel(dev)
    for p, ((log, zlo, zhi), (vmin, thr), Mr) in enumerate(zip(panels, expect, specs)):
        nm = norms[p]
        assert nm["status"] == 0 and nm["vmin"] == vmin and nm["vmax"] == zhi, (p, nm)
        inexact_log = log and D == np.float64
        if thr is not None and not inexact_log:
            assert nm["degenerate"] == 0, (p, nm)
            assert same_bits(table[p], thr, zero_sign_insensitive=False), (p, np.flatnonzero(bits(table[p]) != bits(thr)))
        ref = R.clamp_for_imshow(Mr, "log" if log else "linear", zlo, zhi, float(tiny[0]))
        assert ref["vmin"] == vmin and ref["vmax"] == zhi
        idx_ref, rgba_ref = R.rasterise(ref, lut)
        assert (idx_ref == R.I_BAD).all() == (thr is None), p
        got = b.panel_index(p)
        if inexact_log:
            code = lambda i: np.where(i == R.I_UNDER, -1, np.where(i == R.I_OVER, 256, i.astype(np.int64)))  # noqa: E731
            assert np.array_equal(got == R.I_BAD, idx_ref == R.I_BAD), p
            assert (np.abs(code(got) - code(idx_ref)) <= 1).all(), (p, np.argwhere(got != idx_ref)[:8])
        else:
            assert np.array_equal(got, idx_ref), (p, np.argwhere(got != idx_ref)[:8])
            assert np.array_equal(b.panel_rgba(p), rgba_ref), p


# ---------------------------------------------------------------------------------------------- K2a


def _check_region(st, ref, want_pct, pl, ph):
    with np.errstate(invalid="ignore"), np.testing.suppress_warnings() as sup:
        sup.filter(RuntimeWarning)
        some = (~np.isnan(ref)).any()
        elo = float(np.nanpercentile(ref, pl)) if (want_pct and some) else np.nan
        ehi = float(np.nanpercentile(ref, ph)) if (want_pct and some) else np.nan
    assert same_float(st["p_lo"], elo), (st["p_lo"], elo)
    assert same_float(st["p_hi"], ehi), (st["p_hi"], ehi)
    fp = ref[np.isfinite(ref) & (ref > 0)]
    assert st["n_pos"] == fp.size
    assert st["min_pos"] == (fp.min() if fp.size else np.inf)
    fin = ref[np.isfinite(ref)]
    assert st["fin_min"] == (fin.min() if fin.size else np.inf)
    assert st["fin_max"] == (fin.max() if fin.size else -np.inf)
    assert st["n_valid"] == (~np.isnan(ref)).sum()
    assert st["n_nan"] == np.isnan(ref).sum()
    assert st["n_posinf"] == np.isposinf(ref).sum() and st["n_neginf"] == np.isneginf(ref).sum()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_region_stats_walk_and_selection_edges(ctx, dtype):
    """The vector walk's head / vectors / tail split at every t0 residue (rows shorter than the head, V + 1
    cells), row lists, column lists past the 1024 staged in shared memory, cell counts around the 2048 below
    which nothing is sampled, reductions only / geometry only regions between percentile ones, all-NaN and
    all-+inf regions -- every field against numpy, and the same percentiles through the exact select."""
    rng = np.random.default_rng(71 + np.dtype(dtype).itemsize)
    V = 16 // np.dtype(dtype).itemsize
    T, E = 2100, 40
    M = _random_matrix(rng, T, E, dtype)
    c_nan, c_inf = E - 2, E - 1
    M[:, c_nan] = np.nan
    M[:, c_inf] = np.inf
    b, (f,) = _matrix_batch(ctx, [M], dtype)
    pairs = [(0, 100), (1, 99), (50, 50)]
    cases = []  # (cols, rows, want_pct, (p_lo, p_hi))

    def add(cols, rows, want_pct=1):
        cases.append((np.asarray(cols), np.asarray(rows), want_pct, pairs[len(cases) % 3]))

    some = rng.choice(E - 2, 7, replace=False)
    for t0 in range(16, 16 + 2 * V):  # every residue, twice; rows shorter than the head, V + 1 cells
        for nt in sorted({1, 2, V - 1, V + 1, 2 * V + 3, 301}):
            add(some, np.arange(t0, t0 + nt))
    for ne, nt in ((23, 89), (32, 64), (3, 683), (17, 241), (1, 2048), (1, 2049)):  # 2047 2048 2049 4097 2048 2049 cells
        for t0 in (0, 1 + int(rng.integers(0, 4))):
            add(rng.choice(E - 2, ne, replace=ne > E - 2), np.arange(t0, t0 + nt))
    long_cols = rng.integers(0, E - 2, 1500)  # past the shared-memory column list; repeats are legal
    for rows in (np.arange(3, 4), np.arange(5, 8), np.arange(1, 1 + V + 1), np.array([2, 9, 10, 400, 1299])):
        add(long_cols, rows)
    for ne in (1, 5, 33):
        add(rng.choice(E - 2, ne, replace=False), np.sort(rng.choice(T, int(rng.integers(2, 900)), replace=False)))
    add([c_nan] * 3, np.arange(0, 1000))  # all NaN, sampled
    add([c_nan, c_nan], np.arange(7, 12))  # all NaN, small
    add([c_inf] * 2, np.arange(3, 1206))  # all +inf, sampled
    add([c_inf, c_inf, c_inf], np.array([1, 4, 9]))  # all +inf, small
    add(np.r_[some, c_inf], np.arange(1, 600))
    for k in range(0, len(cases), 5):  # reductions only, and geometry only, among the percentile regions
        cols, rows, _, pp = cases[k]
        cases.append((cols, rows, 0, pp))
        cases.append((cols, rows, 2, pp))
    rng.shuffle(cases)
    regs = [b.add_region(f, 0, c, rows=r, want_pct=w, p_lo=pl, p_hi=ph) for c, r, w, (pl, ph) in cases]
    b.upload_tables()
    b.run_stats()
    st = b.stats().copy()
    for r, (cols, rows, w, (pl, ph)) in zip(regs, cases):
        if w == 2:
            continue  # geometry only: no statistics
        ref = M[np.ix_(rows, cols)].T
        try:
            _check_region(st[r], ref, w, pl, ph)
        except AssertionError as exc:
            raise AssertionError(f"region {r}: {len(cols)} cols x rows {rows[:3]}..({len(rows)}), want_pct {w}, "
                                 f"p {pl}/{ph}: {exc}") from None
    b.force_exact_stats(True)
    try:
        b.run_stats()
        exact = b.stats().copy()
        n_pct = sum(1 for r, c in zip(regs, cases) if c[2] == 1 and st[r]["n_valid"] > 0)
        assert b.stats_fallbacks() == n_pct
    finally:
        b.force_exact_stats(False)
    for r, (_, _, w, _) in zip(regs, cases):
        if w == 1:
            assert same_float(exact[r]["p_lo"], st[r]["p_lo"]) and same_float(exact[r]["p_hi"], st[r]["p_hi"]), r
