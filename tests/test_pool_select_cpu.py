"""The host-driven pooled-extrema descent (``pool_select.prefix_percentiles``) with the numpy stand-in
for the pool kernels (``oracle/pool_backend.NumpyPoolBackend``), on the edge cases of
``test_gpu_pool_paths.py``: more than 64 distinct prefixes in a digit (several refine rounds),
neighbours split across every radix-digit boundary, subnormals and the float extremes, and the edge
percentiles in both modes.  Every value equals numpy's ``nanpercentile`` of the prefix pools."""

import numpy as np
import pytest

from tests.test_gpu_pool_paths import (
    SEQUENCES,
    CountingBackend,
    _brute,
    _matrix,
    boundary_pair,
    digit_boundaries,
    digit_case,
    edge_case,
    multi_round_case,
    sequence_case,
    to_key,
)


def _run_numpy(case, reqs, backend_wrap=None):
    """prefix_percentiles over the collapsed matrices of ``case`` ((T, E) row-major, one flat array)."""
    from configurable_spectrograms_b200._lib import POOL_ITEM
    from configurable_spectrograms_b200.pool_select import prefix_percentiles
    from oracle.pool_backend import NumpyPoolBackend

    mats, rows, off = [], [], 0
    for i, cubes in enumerate(case.cubes):
        for k, c in enumerate(cubes):
            m = _matrix(c)
            mats.append(m.reshape(-1))
            rows.append((off, m.shape[0], m.shape[1], i, k))
            off += m.size
    flat = np.concatenate(mats) if mats else np.zeros(1, case.dtype)
    items = np.array(rows, dtype=POOL_ITEM)
    backend = NumpyPoolBackend(flat)
    if backend_wrap is not None:
        backend = backend_wrap(backend)
    vals, _counts, _npos = prefix_percentiles(backend, case.dtype, items, case.n_inst, case.inst_len, case.max_E, reqs)
    return vals, backend


def _check(case, reqs, vals):
    for r, req in enumerate(reqs):
        best, last, _ = _brute([_matrix(c) for c in case.cubes[req["inst"]]], req["p"])
        want = best if req["mode"] == "running_max" else last
        assert vals[r] == want, (r, req, vals[r], want)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_host_descent_more_than_64_prefixes_takes_several_rounds(dtype):
    from configurable_spectrograms_b200.pool_select import digit_plan

    case, reqs = multi_round_case(dtype)
    vals, backend = _run_numpy(case, reqs, CountingBackend)
    assert backend.refines > len(digit_plan(dtype)) - 1, "more than 64 prefixes must take more than one round"
    _check(case, reqs, vals)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_host_descent_digit_boundaries_and_float_extremes(dtype):
    case, reqs = digit_case(dtype)
    vals, _ = _run_numpy(case, reqs)
    _check(case, reqs, vals)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_host_descent_percentile_edges(dtype):
    case, reqs = edge_case(dtype)
    vals, _ = _run_numpy(case, reqs)
    _check(case, reqs, vals)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_boundary_pairs_straddle_each_digit(dtype):
    """The neighbour pairs of the digit-boundary cases are adjacent floats whose keys differ in bit 0
    alone or carry into the lowest bit of a digit: 2 digit boundaries for float32, 6 for float64."""
    bnds = digit_boundaries(dtype)
    assert len(bnds) == (3 if dtype is np.float32 else 7)
    for b in bnds:
        lo, hi = boundary_pair(dtype, b)
        kl, kh = to_key(lo, dtype), to_key(hi, dtype)
        assert kh == kl + 1 and (kl ^ kh) == (1 << (b + 1)) - 1, b


@pytest.mark.parametrize("layout", sorted(SEQUENCES))
def test_sequence_cases_reach_the_running_max_where_they_claim(layout):
    """The sequence cases put the running maximum of p = 99 at the first, a middle and the last
    prefix that grew (on the host: the GPU test asserts it too, this keeps the seeds honest)."""
    for dtype in (np.float32, np.float64):
        case, _reqs = sequence_case(dtype, layout)
        reached = set()
        for i, (L, _empty, _storm) in enumerate(SEQUENCES[layout]):
            if L == 0:
                continue
            best, _last, per = _brute([_matrix(c) for c in case.cubes[i]], 99.0)
            grew = [k for k, v in enumerate(per) if v is not None]
            at = per.index(best)
            reached.add("first" if at == grew[0] else "last" if at == grew[-1] else "middle")
        assert reached == {"first", "middle", "last"}, (dtype, layout, reached)
