"""Every path of the pooled-extrema selection (K2b: ``csrc/pool.cu``, ``csrc/poolsel.cu``,
``pool_select.py``) at its edges, through both drivers -- the device digit loop
(``DevicePoolSelector``) and the host-driven descent (``prefix_percentiles`` over
``GpuPoolBackend``) -- against numpy's ``nanpercentile`` of every prefix pool, brute force.

Covered: ``walk_rows`` vector tails and its 64-vector stride, empty energy bands, T = 0; neighbours
that differ only across a radix-digit boundary, subnormals, the float extremes, tiny and all-equal
pools; the clamp and ``gamma >= 0.5`` branches of numpy's rank arithmetic; short, ragged and empty
file sequences; the 16-slot device table at and past its capacity, 64 requests over more than 1024
table entries, the 65th request; the host driver's multi-round refine (more than 64 prefixes in a
digit); the device y candidates beyond one 128-energy chunk; ranks without files and a whole pool
held by the lowest rank; the ABI's argument refusals.

Pools are built exactly: a cube with one pitch bin collapses to itself (K1 seeds its chain with
+0.0, compiles no flush-to-zero, and turns NaN into 0), so ``(T, 1, E)`` cubes put exactly the
chosen values into the pool.  Every comparison is ``==``."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

F32_T = (0, 1, 3, 4, 5, 255, 256, 257, 260)  # float4 tails, T around the 64-vector (256-cell) stride
F64_T = (1, 2, 3, 127, 128, 129, 130)  # double2 tails, T around the 64-vector (128-cell) stride
PASS_E = (1, 2, 3, 4, 5, 97)  # E < kSplit = 4 leaves energy bands empty
EDGE_P = (0.0, 1e-7, 25.0, 50.0, 99.99999, 100.0)


@pytest.fixture(scope="module")
def ctx():
    from configurable_spectrograms_b200 import _lib

    return _lib.Context(0)


# ------------------------------------------------------------------------------------ reference


def _positives(m):
    with np.errstate(invalid="ignore"):
        return m[np.isfinite(m) & (m > 0)]


def _matrix(cube):
    with np.errstate(invalid="ignore", over="ignore"):
        return np.nansum(cube, axis=1)


def _brute(mats, p):
    """numpy over every prefix pool of one instrument's files (position order).

    Returns ``(running max, whole pool, per-prefix values)``: the running maximum of
    ``np.nanpercentile(pool so far, p)`` over the prefixes whose pool grew, the percentile of the
    whole pool, and the value of every prefix (None where the pool did not grow).  None stands for
    an empty pool.  ``p`` goes in as a Python float: an ``np.float64`` would turn numpy's float32
    rank arithmetic into float64 (NEP 50)."""
    p = float(p)
    blocks, best, last, per = [], None, None, []
    for m in mats:
        pos = _positives(m)
        if pos.size == 0:
            per.append(None)
            continue
        blocks.append(pos)
        v = float(np.nanpercentile(np.concatenate(blocks), p))
        best = v if best is None else max(best, v)
        last = v
        per.append(v)
    return best, last, per


def _expected(case, req):
    best, last, _ = _brute([_matrix(c) for c in case.cubes[req["inst"]]], req["p"])
    return best if req["mode"] == "running_max" else last


def _ranks(n, p, dtype):
    from configurable_spectrograms_b200.pool_select import percentile_ranks

    lo, hi, g = percentile_ranks(np.array([n], np.int64), float(p), dtype)
    return int(lo[0]), int(hi[0]), float(g[0])


# ----------------------------------------------------------------------------------- pool cases


class Case:
    """Cubes by instrument, in sequence order (an instrument may have none)."""

    def __init__(self, dtype, n_inst):
        self.dtype = np.dtype(dtype).type
        self.cubes = [[] for _ in range(n_inst)]

    @property
    def n_inst(self):
        return len(self.cubes)

    @property
    def inst_len(self):
        return np.array([len(c) for c in self.cubes], dtype=np.int32)

    @property
    def max_E(self):
        return max([c.shape[2] for cs in self.cubes for c in cs] + [1])

    def add(self, inst, cube):
        assert cube.dtype == self.dtype
        self.cubes[inst].append(cube)

    def add_exact(self, inst, values, rng, E=3):
        """One file whose pool is exactly ``values``, among cells the pool must exclude."""
        self.add(inst, exact_cube(self.dtype, values, rng, E))


def exact_cube(dtype, values, rng, E=3):
    """A (T, 1, E) cube holding ``values`` plus 0.0, -0.0, a negative, NaN and +-inf; NaN fills the rest."""
    D = np.dtype(dtype).type
    cells = np.concatenate([np.asarray(values, dtype=D), np.array([0.0, -0.0, -2.5, np.nan, np.inf, -np.inf], dtype=D)])
    T = -(-len(cells) // E)
    flat = np.full(T * E, np.nan, dtype=D)
    flat[: len(cells)] = cells
    return flat[rng.permutation(T * E)].reshape(T, 1, E)


def wide_cube(rng, dtype, T, P, E, integer=False, scale=1.0):
    """An ordinary cube (P > 1): gamma or Poisson data with NaN, -0.0, negatives and +-inf."""
    c = (rng.poisson(2.0, (T, P, E)) if integer else rng.gamma(2.0, 3.0, (T, P, E))).astype(dtype) * dtype(scale)
    c[rng.random(c.shape) < 0.08] = np.nan
    c[rng.random(c.shape) < 0.04] = -0.0
    c[rng.random(c.shape) < 0.04] = -1.0
    if c.size >= 8:
        c.flat[rng.integers(0, c.size, 2)] = np.inf
        c.flat[rng.integers(0, c.size, 1)] = -np.inf
    return c


def from_key(key, dtype):
    if np.dtype(dtype) == np.float32:
        return np.array([key], np.uint32).view(np.float32)[0]
    return np.array([key], np.uint64).view(np.float64)[0]


def to_key(v, dtype):
    return int(np.array([v], dtype).view(np.uint32 if np.dtype(dtype) == np.float32 else np.uint64)[0])


def digit_boundaries(dtype):
    """Key bits b whose neighbours key / key + 1 straddle a radix digit: 0 (the last bit alone) and
    the lowest bit of every digit above the last."""
    from configurable_spectrograms_b200.pool_select import digit_plan

    return [0] + sorted(s for s, _b in digit_plan(dtype) if s > 0)


def boundary_pair(dtype, b):
    """(lo, hi): adjacent floats whose keys differ in bit 0 only (b = 0) or carry from bits 0..b-1 into bit b."""
    base = to_key(np.dtype(dtype).type(1.37), dtype)
    lo = (base & ~((1 << (b + 1)) - 1)) | ((1 << b) - 1)
    return from_key(lo, dtype), from_key(lo + 1, dtype)


def special_pools(dtype):
    """{name: pool values}: subnormals, the normal minimum, the float maximum, tiny and all-equal pools."""
    D = np.dtype(dtype).type
    fi = np.finfo(dtype)
    nbits = 23 if D is np.float32 else 52
    top_sub = (1 << nbits) - 1
    return {
        "smallest_subnormal": [from_key(1, dtype), from_key(1, dtype), from_key(2, dtype), from_key(3, dtype), D(1.0)],
        "largest_subnormal": [from_key(top_sub - 1, dtype), from_key(top_sub, dtype), D(fi.tiny), D(fi.tiny) * D(2)],
        "max": [D(1.0), np.nextafter(fi.max, D(0)), fi.max, fi.max],
        "all_equal": [D(3.0)] * 9,
        "one_sample": [D(5.0)],
        "two_samples": [D(2.0), D(3.0)],
    }


SPECIAL_P = (0.0, 30.0, 50.0, 70.0, 100.0)


def digit_case(dtype, seed=3):
    """Case 2: one instrument per digit boundary (neighbour pair split over two files, requests whose
    virtual index lands between the pair with gamma below and above 0.5) and one per special pool."""
    D = np.dtype(dtype).type
    rng = np.random.default_rng(seed)
    bnds = digit_boundaries(dtype)
    specials = special_pools(dtype)
    case = Case(dtype, len(bnds) + len(specials))
    reqs = []
    for i, b in enumerate(bnds):
        lo, hi = boundary_pair(dtype, b)
        pool = [lo / D(8), lo / D(4), lo / D(2), lo, hi, hi * D(2), hi * D(4), hi * D(8)]  # lo, hi at ranks 3, 4
        first = rng.permutation(8)[:4]
        case.add_exact(i, [pool[k] for k in first], rng)
        case.add_exact(i, [pool[k] for k in range(8) if k not in first], rng)
        for x in (3.25, 3.75):
            p = 100.0 * x / 7.0
            r_lo, r_hi, g = _ranks(8, p, dtype)
            assert (r_lo, r_hi) == (3, 4) and (0.0 < g < 0.5 if x < 3.5 else g >= 0.5), (b, p, r_lo, r_hi, g)
            reqs.append({"inst": i, "p": p, "mode": "last"})
        reqs.append({"inst": i, "p": 100.0 * 3.75 / 7.0, "mode": "running_max"})
    for j, (name, pool) in enumerate(specials.items()):
        i = len(bnds) + j
        case.add_exact(i, pool, rng)
        reqs += [{"inst": i, "p": p, "mode": "last"} for p in SPECIAL_P]
        reqs.append({"inst": i, "p": 50.0, "mode": "running_max"})
    assert len(reqs) <= 64
    return case, reqs


def edge_case(dtype, seed=4):
    """Case 3: pools of 3 (p = 25: gamma exactly 0.5) and 5 (p = 50: gamma exactly 0) positives over
    several files, and a wide instrument; every edge percentile in both modes."""
    D = np.dtype(dtype).type
    rng = np.random.default_rng(seed)
    case = Case(dtype, 3)
    # b - a rounds (2**m + 1 is not representable): numpy's g >= 0.5 form b - (b-a)(1-g) and the
    # other form a + (b-a)g land on different floats at g = 0.5
    big = D(2.0) ** (24 if D is np.float32 else 53) + D(2)
    case.add_exact(0, [big * D(4)], rng)
    case.add_exact(0, [D(1.0), big], rng)
    case.add_exact(1, [D(4.0), D(0.75)], rng)
    case.add_exact(1, [], rng)
    case.add_exact(1, [D(9.5), D(2.0), D(6.25)], rng)
    for k in range(3):
        case.add(2, wide_cube(rng, D, 6, 2, 3, integer=True, scale=4.0 if k == 1 else 1.0))
    assert _ranks(3, 25.0, dtype)[2] == 0.5 and _ranks(5, 50.0, dtype) == (2, 3, 0.0)
    reqs = [{"inst": i, "p": p, "mode": m} for i in range(3) for p in EDGE_P for m in ("last", "running_max")]
    return case, reqs


def multi_round_case(dtype, n_last=70, seed=1):
    """Case 6: ``n_last`` whole-pool requests with distinct p over a pool spread across ~90 binades,
    so more than 64 distinct key prefixes survive a digit; plus one running-max request."""
    rng = np.random.default_rng(seed)
    case = Case(dtype, 1)
    for _k in range(5):
        c = np.exp(rng.uniform(-30, 30, (50, 1, 6))).astype(dtype)
        c[rng.random(c.shape) < 0.1] = np.nan
        c[0, 0, :3] = np.array([0.0, -4.0, -np.inf], dtype=dtype)
        case.add(0, c)
    reqs = [{"inst": 0, "p": float(p), "mode": "last"} for p in np.linspace(0.5, 99.5, n_last)]
    reqs.append({"inst": 0, "p": 99.0, "mode": "running_max"})
    return case, reqs


# ----------------------------------------------------------------------------------------- drivers


def build_batch(ctx, case):
    """Upload and collapse every cube of ``case``; POOL_ITEM rows in (instrument, position) order."""
    from configurable_spectrograms_b200._lib import POOL_ITEM
    from configurable_spectrograms_b200.engine import Batch

    b = Batch(ctx, case.dtype, 0)
    rows = []
    for i, cubes in enumerate(case.cubes):
        for k, c in enumerate(cubes):
            f = b.add_file(c)
            rows.append((b.mat_off(f, 0), c.shape[0], c.shape[2], i, k))
    b.upload_cubes()
    b.collapse()
    return b, np.array(rows, dtype=POOL_ITEM) if rows else np.zeros(0, POOL_ITEM)


def check_counts(case, counts, npos):
    """Per-file per-energy positive counts and totals, items in (instrument, position) order."""
    j = 0
    for cubes in case.cubes:
        for c in cubes:
            with np.errstate(invalid="ignore"):
                ok = np.isfinite(_matrix(c)) & (_matrix(c) > 0)
            want = np.zeros(counts.shape[1], np.int64)
            want[: c.shape[2]] = ok.sum(axis=0)
            assert np.array_equal(counts[j], want), (j, c.shape)
            assert npos[j] == ok.sum(), (j, c.shape)
            j += 1
    assert j == len(npos)


def run_device(b, case, items, reqs, max_E=None, ydev=None, sel=None):
    """DevicePoolSelector twice (the second run re-uses every scratch buffer): (values, counts, npos)."""
    from configurable_spectrograms_b200.pool_select import DevicePoolSelector

    sel = sel or DevicePoolSelector(b)
    max_E = max_E or case.max_E
    out = []
    for _ in range(2):
        sel.enqueue(case.dtype, items, case.n_inst, case.inst_len, max_E, reqs, ydev=ydev)
        if ydev is None:
            counts, npos = sel.result_counts()
            out.append((sel.result_values(), counts, npos))
        else:
            out.append((sel.result_values(), None, None))
    assert out[0][0] == out[1][0]
    return out[1]


def run_host(b, case, items, reqs, max_E=None, backend=None):
    from configurable_spectrograms_b200.pool_select import GpuPoolBackend, prefix_percentiles

    backend = backend or GpuPoolBackend(b)
    return prefix_percentiles(backend, case.dtype, items, case.n_inst, case.inst_len, max_E or case.max_E, reqs)


def check_values(case, reqs, vals, what):
    assert vals is not None, f"{what}: slot overflow"
    assert len(vals) == len(reqs)
    for r, req in enumerate(reqs):
        want = _expected(case, req)
        assert vals[r] == want, (what, r, req, vals[r], want)


def check_both(ctx, case, reqs):
    b, items = build_batch(ctx, case)
    vals, counts, npos = run_device(b, case, items, reqs)
    check_values(case, reqs, vals, "device")
    check_counts(case, counts, npos)
    vals, counts, npos = run_host(b, case, items, reqs)
    check_values(case, reqs, vals, "host-driven")
    check_counts(case, counts, npos)


def y_reference(energy, cubes):
    """max over the prefixes of the reference's 99 %-coverage energy (None: no file took part)."""
    from configurable_spectrograms_b200.fast.extrema import energy_candidates

    if not cubes:
        return None
    counts = []
    for c in cubes:
        m = _matrix(c)
        with np.errstate(invalid="ignore"):
            counts.append((np.isfinite(m) & (m > 0)).sum(axis=0))
    return max(energy_candidates([energy] * len(cubes), np.asarray(counts)))


def y_tables(energies, max_E, limit):
    n_inst = len(energies)
    order = np.zeros((n_inst, max_E), np.int32)
    keys = np.zeros((n_inst, max_E), np.float64)
    n_keys = np.zeros(n_inst, np.int32)
    for i, e in enumerate(energies):
        o = np.argsort(e, kind="stable")
        order[i, : len(e)], keys[i, : len(e)], n_keys[i] = o, e[o], len(e)
    return {"order": order, "keys": keys, "n_keys": n_keys, "limit": np.asarray(limit, np.int32)}


# ------------------------------------------------------------------------------- 1. first pass


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_first_pass_tails_bands_and_energy_rows(ctx, dtype):
    """One instrument per (T, E): the histogram walk's vector tails, its two-halves 64-vector stride
    and empty energy bands, through the per-energy counts, the per-position energy rows of the
    device y tables, one percentile request each and the y candidates."""
    rng = np.random.default_rng(11 if dtype is np.float32 else 12)
    shapes = [(T, E) for T in (F32_T if dtype is np.float32 else F64_T) for E in PASS_E]
    case = Case(dtype, len(shapes))
    for i, (T, E) in enumerate(shapes):
        case.add(i, wide_cube(rng, dtype, T, 3, E))
    reqs = [{"inst": i, "p": (50.0, 99.0, 1.0)[i % 3], "mode": ("last", "running_max")[i % 2]} for i in range(len(shapes))]
    assert len(reqs) <= 64
    check_both(ctx, case, reqs)
    # the same files with the energy tables on the device: the scanned per-position count rows
    from configurable_spectrograms_b200.pool_select import DevicePoolSelector

    b, items = build_batch(ctx, case)
    max_E = case.max_E
    energies = [rng.permutation(np.geomspace(4.0, 30000.0, E)) for _T, E in shapes]
    ydev = y_tables(energies, max_E, case.inst_len)
    sel = DevicePoolSelector(b)
    vals, _, _ = run_device(b, case, items, reqs, ydev=ydev, sel=sel)
    check_values(case, reqs, vals, "device (y tables)")
    ehist = sel.mem.dev["ehist"].download(np.uint32, case.n_inst * max_E).reshape(case.n_inst, max_E)
    for i, (c,) in enumerate(case.cubes):
        m = _matrix(c)
        with np.errstate(invalid="ignore"):
            want = (np.isfinite(m) & (m > 0)).sum(axis=0)
        assert np.array_equal(ehist[i, : c.shape[2]], want), shapes[i]
        assert not ehist[i, c.shape[2] :].any(), shapes[i]
    ycand = sel.result_y_candidates()
    for i, (c,) in enumerate(case.cubes):
        assert ycand[i] == y_reference(energies[i], [c]), (shapes[i], ycand[i])


# ---------------------------------------------------------------------------- 2. digit boundaries


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_neighbours_across_digit_boundaries_and_float_extremes(ctx, dtype):
    case, reqs = digit_case(dtype)
    check_both(ctx, case, reqs)


# --------------------------------------------------------------------------- 3. percentile edges


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_percentile_edges_both_modes(ctx, dtype):
    case, reqs = edge_case(dtype)
    check_both(ctx, case, reqs)


# ---------------------------------------------------------------------------------- 4. sequences

# (inst_len, positions without positives, position of the storm file)
SEQUENCES = {
    "short": [(1, (), 0), (7, (0, 3, 6), 1), (0, (), None), (8, (0, 4, 7), 5), (9, (0, 5, 8), 7)],
    "long": [(17, (0, 8, 16), 15), (0, (), None), (100, (0, 50, 99), 1), (9, (0, 4, 8), 5), (7, (3,), 6)],
}


def sequence_case(dtype, layout, seed=7):
    rng = np.random.default_rng(seed)
    spec = SEQUENCES[layout]
    case = Case(dtype, len(spec))
    for i, (L, empty, storm) in enumerate(spec):
        for k in range(L):
            c = wide_cube(rng, dtype, int(rng.integers(2, 6)), 2, 3, integer=True, scale=8.0 if k == storm else 1.0)
            if k in empty:
                c[:] = -np.abs(c)  # no positives: NaN, zeros, negatives, -inf
            case.add(i, c)
    reqs = []
    for i in range(len(spec)):
        reqs += [{"inst": i, "p": 99.0, "mode": "running_max"}, {"inst": i, "p": 50.0, "mode": "last"},
                 {"inst": i, "p": 1.0, "mode": "running_max"}]
    return case, reqs


@pytest.mark.parametrize("layout", sorted(SEQUENCES))
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_sequences_short_ragged_and_empty(ctx, dtype, layout):
    """The scan's eight segments over sequences shorter than, equal to, just past and far past 8
    files, ragged across instruments, an instrument with no file (its requests are None), files
    without positives at the first / a middle / the last position, the running maximum reached at
    the first / a middle / the last prefix that grew."""
    case, reqs = sequence_case(dtype, layout)
    reached = set()
    for i, (L, _empty, _storm) in enumerate(SEQUENCES[layout]):
        best, _last, per = _brute([_matrix(c) for c in case.cubes[i]], 99.0)
        if L == 0:
            assert best is None
            continue
        grew = [k for k, v in enumerate(per) if v is not None]
        at = per.index(best)
        reached.add("first" if at == grew[0] else "last" if at == grew[-1] else "middle")
    assert reached == {"first", "middle", "last"}, reached
    for r, req in enumerate(reqs):
        if SEQUENCES[layout][req["inst"]][0] == 0:
            assert _expected(case, req) is None
    check_both(ctx, case, reqs)


# ------------------------------------------------------------------------ 5. slot table, requests


def powers_case(dtype, n_req, seed=5):
    """One file of 40 powers of two (one binade, hence one top-level bucket, per sample); request r
    takes the neighbours at ranks 4r and 4r + 1, so n_req requests need 2 n_req distinct prefixes."""
    rng = np.random.default_rng(seed)
    D = np.dtype(dtype).type
    case = Case(dtype, 1)
    case.add_exact(0, [D(2.0) ** k for k in range(-20, 20)], rng, E=5)
    reqs = []
    for r in range(n_req):
        p = 100.0 * (4 * r + 0.5) / 39.0
        assert _ranks(40, p, dtype)[:2] == (4 * r, 4 * r + 1)
        reqs.append({"inst": 0, "p": p, "mode": "last"})
    return case, reqs


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_device_slot_table_capacity(ctx, dtype):
    """16 distinct prefixes fill the 16-slot table exactly (values); 18 overflow it (None), and the
    host-driven fallback still equals numpy."""
    from configurable_spectrograms_b200.pool_select import DevicePoolSelector

    assert DevicePoolSelector.N_SLOTS == 16
    case, reqs = powers_case(dtype, 8)
    b, items = build_batch(ctx, case)
    vals, _, _ = run_device(b, case, items, reqs)
    check_values(case, reqs, vals, "device, 16 prefixes")
    case, reqs = powers_case(dtype, 9)
    b, items = build_batch(ctx, case)
    sel = DevicePoolSelector(b)
    sel.enqueue(dtype, items, 1, case.inst_len, case.max_E, reqs)
    assert sel.result_values() is None, "18 distinct prefixes cannot fit 16 slots"
    vals, counts, npos = run_host(b, case, items, reqs)
    check_values(case, reqs, vals, "host-driven fallback")
    check_counts(case, counts, npos)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_sixty_four_requests_over_seventeen_positions(ctx, dtype):
    """64 requests (the documented maximum) x 17 positions = 1088 selection entries: the bounds and
    finish kernels' 1024-thread walks wrap.  The pool sits in one narrow key range so the slot table
    never overflows.  A 65th request is refused."""
    from configurable_spectrograms_b200._lib import CsgError
    from configurable_spectrograms_b200.pool_select import DevicePoolSelector

    rng = np.random.default_rng(17)
    D = np.dtype(dtype).type
    ulp = D(2.0) ** (-23 if D is np.float32 else -52)
    spread = 1024 if D is np.float32 else 4  # only the last digit's bits vary
    case = Case(dtype, 1)
    for _k in range(17):
        vals = D(1.0) + rng.integers(0, spread, int(rng.integers(3, 12))).astype(D) * ulp
        case.add_exact(0, vals, rng)
    ps = [float(p) for p in np.linspace(0.0, 100.0, 32)]
    reqs = [{"inst": 0, "p": p, "mode": m} for m in ("running_max", "last") for p in ps]
    assert len(reqs) == 64
    check_both(ctx, case, reqs)
    b, items = build_batch(ctx, case)
    with pytest.raises(CsgError, match="at most 64"):
        DevicePoolSelector(b).enqueue(dtype, items, 1, case.inst_len, case.max_E, reqs + reqs[:1])


# ------------------------------------------------------------------ 6. host-driven multi-round


class CountingBackend:
    """A pool backend that counts the refinement histograms (one per round of each digit)."""

    def __init__(self, inner):
        self.inner, self.refines = inner, 0

    def __getattr__(self, name):
        return getattr(self.inner, name)

    def hist_refine(self, *args):
        self.refines += 1
        return self.inner.hist_refine(*args)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_host_driven_refine_in_several_rounds(ctx, dtype):
    from configurable_spectrograms_b200.pool_select import GpuPoolBackend, digit_plan

    case, reqs = multi_round_case(dtype)
    b, items = build_batch(ctx, case)
    backend = CountingBackend(GpuPoolBackend(b))
    vals, counts, npos = run_host(b, case, items, reqs, backend=backend)
    assert backend.refines > len(digit_plan(dtype)) - 1, "more than 64 prefixes must take more than one round"
    check_values(case, reqs, vals, "host-driven")
    check_counts(case, counts, npos)


# ---------------------------------------------------------------------- 7. device y candidates


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_device_y_candidates_long_tables_ties_and_limits(ctx, dtype):
    """297 energies in a 300-column table (padded rows, two 128-energy chunks and a carry), energies
    in permuted order with ties, a count vector whose cumulative sum hits 0.99 x total exactly
    (searchsorted 'right' takes the next energy), a limit below the sequence and a limit of 0."""
    rng = np.random.default_rng(23)
    D = np.dtype(dtype).type
    max_E = 300
    energies = [
        rng.permutation(np.geomspace(3.0, 40000.0, 297)),
        np.array([40.0, 10.0, 30.0, 20.0, 50.0]),
        rng.permutation(np.repeat(np.linspace(5.0, 900.0, 100), 2)),
        rng.permutation(np.linspace(1.0, 10.0, 6)),
    ]
    case = Case(dtype, 4)
    for k in range(4):
        case.add(0, wide_cube(rng, D, int(rng.integers(3, 9)), 2, 297, scale=6.0 if k == 1 else 1.0))
    # sorted energies 10, 20, 30, 40, 50 hold 50, 49, 0, 1, 0 positives: the cumulative sum is 99.0 at 20 and 30
    assert 0.99 * 100 == 99.0
    c = np.full((50, 1, 5), np.nan, dtype=D)
    c[:, 0, 1] = np.arange(1, 51, dtype=D)
    c[:49, 0, 3] = D(2.5)
    c[49, 0, 3] = D(-1.0)
    c[:, 0, 2] = D(0.0)
    c[7, 0, 0] = D(3.0)
    c[:, 0, 4] = -np.inf
    case.add(1, c)
    for k in range(3):
        case.add(2, wide_cube(rng, D, int(rng.integers(2, 6)), 2, 200, integer=True))
    for k in range(2):
        case.add(3, wide_cube(rng, D, 4, 2, 6))
    limit = np.array([3, 1, 3, 0], np.int32)
    ydev = y_tables(energies, max_E, limit)
    assert ydev["n_keys"][0] < max_E
    reqs = [{"inst": i, "p": p, "mode": m} for i in range(4) for p, m in ((99.0, "running_max"), (1.0, "last"))]
    from configurable_spectrograms_b200.pool_select import DevicePoolSelector

    b, items = build_batch(ctx, case)
    sel = DevicePoolSelector(b)
    vals, _, _ = run_device(b, case, items, reqs, max_E=max_E, ydev=ydev, sel=sel)
    check_values(case, reqs, vals, "device (y tables)")
    ycand = sel.result_y_candidates()
    want = [y_reference(energies[i], case.cubes[i][: limit[i]]) for i in range(4)]
    assert want[1] == 40.0 and want[3] is None
    assert ycand == want, (ycand, want)


# ------------------------------------------------------------------------------------ 8. ranks


def _rank_run(dtype, cubes, n_inst, n_orbits, n_ranks, E, energies, reqs):
    """The device selection over n_ranks in one process (contiguous orbit blocks, peer mailboxes),
    checked on every rank against the single-rank brute force over the global sequence."""
    from configurable_spectrograms_b200 import _lib
    from configurable_spectrograms_b200._lib import POOL_ITEM
    from configurable_spectrograms_b200.comm import SharedPeerGroup
    from configurable_spectrograms_b200.engine import Batch
    from configurable_spectrograms_b200.pool_select import DevicePoolSelector

    per = -(-n_orbits // n_ranks)
    ctxs = [_lib.Context(0) for _ in range(n_ranks)]
    exchanges = SharedPeerGroup(ctxs).members
    runs, keep = [], []
    for r in range(n_ranks):
        lo, hi = r * per, min(n_orbits, (r + 1) * per)
        b = Batch(ctxs[r], dtype, 0)
        mine = [(i, k, b.add_file(cubes[(i, k)])) for k in range(lo, hi) for i in range(n_inst) if (i, k) in cubes]
        b.upload_cubes()
        b.collapse()
        pos = [0] * n_inst
        rows = []
        for i, k, f in mine:
            rows.append((b.mat_off(f, 0), cubes[(i, k)].shape[0], E, i, pos[i]))
            pos[i] += 1
        items = np.array(rows, dtype=POOL_ITEM) if rows else np.zeros(0, POOL_ITEM)
        ydev = y_tables(energies, E, pos)
        runs.append((DevicePoolSelector(b), items, np.array(pos, np.int32), ydev))
        keep.append(b)
    assert any(len(items) == 0 for _s, items, _l, _y in runs) or n_ranks < 4
    for r in range(n_ranks):  # ranks sharing one process: every allocation happens before any launch
        sel, items, inst_len, ydev = runs[r]
        sel.reserve(dtype, items, n_inst, inst_len, E, reqs, exchange=exchanges[r], ydev=ydev)
    for c in ctxs:
        c.sync()
    global_case = Case(dtype, n_inst)
    for k in range(n_orbits):
        for i in range(n_inst):
            if (i, k) in cubes:
                global_case.add(i, cubes[(i, k)])
    want_y = [y_reference(energies[i], global_case.cubes[i]) for i in range(n_inst)]
    for r in range(n_ranks):
        sel, items, inst_len, ydev = runs[r]
        sel.enqueue(dtype, items, n_inst, inst_len, E, reqs, exchange=exchanges[r], ydev=ydev)
    for r in range(n_ranks):
        sel = runs[r][0]
        check_values(global_case, reqs, sel.result_values(), f"rank {r}")
        assert sel.result_y_candidates() == want_y, (r, want_y)
    del runs, keep, exchanges
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_ranks_with_no_files(dtype):
    """4 ranks over 3 orbits: the last rank holds no file at all."""
    rng = np.random.default_rng(31)
    E = 8
    cubes = {(i, k): wide_cube(rng, dtype, int(rng.integers(4, 12)), 3, E, integer=(i == 0), scale=5.0 if k == 1 else 1.0)
             for i in range(2) for k in range(3)}
    energies = [np.geomspace(30000.0, 4.0, E), rng.permutation(np.linspace(1.0, 400.0, E))]
    reqs = [{"inst": i, "p": p, "mode": m} for i in range(2) for p, m in ((99.0, "running_max"), (1.0, "last"), (50.0, "last"))]
    _rank_run(dtype, cubes, 2, 3, 4, E, energies, reqs)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_ranks_pool_held_by_the_lowest_rank(dtype):
    """3 ranks over 6 orbits; every positive of instrument 0 sits on rank 0 (the higher ranks' files
    have none): its whole-pool requests are answered by rank 0 through ``above``, its running-max
    prefixes repeat across ranks 1 and 2."""
    rng = np.random.default_rng(37)
    E = 8
    cubes = {}
    for k in range(6):
        c0 = wide_cube(rng, dtype, int(rng.integers(4, 12)), 3, E, scale=3.0 if k == 1 else 1.0)
        if k >= 2:
            c0[:] = -np.abs(c0)
        cubes[(0, k)] = c0
        cubes[(1, k)] = wide_cube(rng, dtype, int(rng.integers(4, 12)), 3, E, integer=True)
    energies = [rng.permutation(np.geomspace(5.0, 25000.0, E)), np.geomspace(30000.0, 4.0, E)]
    reqs = [{"inst": i, "p": p, "mode": m} for i in range(2) for p, m in ((99.0, "running_max"), (1.0, "last"), (50.0, "last"))]
    _rank_run(dtype, cubes, 2, 6, 3, E, energies, reqs)


# -------------------------------------------------------------------------------- 9. ABI refusals


def test_abi_refuses_out_of_range_arguments(ctx):
    """Each entry point refuses its out-of-range argument with an error status and launches nothing."""
    from configurable_spectrograms_b200._lib import F32, F64

    lib, h = ctx.lib, ctx.handle
    buf = ctx.alloc(1 << 16)
    p = buf.ptr
    calls = {
        "hist_first bits 0": lambda: lib.csg_pool_hist_first(h, p, F32, p, 1, 1, 0, 8, p, p, p, None),
        "hist_first bits 13": lambda: lib.csg_pool_hist_first(h, p, F64, p, 1, 1, 13, 8, p, p, p, None),
        "hist_first max_E 8193": lambda: lib.csg_pool_hist_first(h, p, F32, p, 1, 1, 11, 8193, p, p, p, None),
        "hist_refine n_slots 0": lambda: lib.csg_pool_hist_refine(h, p, F32, p, 1, 1, 0, p, 20, 10, 10, p),
        "hist_refine n_slots 65": lambda: lib.csg_pool_hist_refine(h, p, F64, p, 1, 1, 65, p, 52, 42, 10, p),
        "sel_slots n_slots 0": lambda: lib.csg_pool_sel_slots(h, p, p, 1, 1, 20, p, 1, 0, p, p),
        "sel_slots n_slots 65": lambda: lib.csg_pool_sel_slots(h, p, p, 1, 1, 20, p, 1, 65, p, p),
        "sel_init 65 requests": lambda: lib.csg_pool_sel_init(h, F32, p, 65, p, 1, p, p, None, p),
    }
    ctx.sync()
    for name, call in calls.items():
        n0 = int(lib.csg_launch_count(h))
        assert call() != 0, name
        assert int(lib.csg_launch_count(h)) == n0, name
    ctx.sync()
    buf.free()

