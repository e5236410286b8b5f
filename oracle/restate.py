"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's hot path.

Nothing under ``oracle/`` is imported by the product package; only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may use it, and only as the checker / reported CPU baseline.

The reference (ev-hansen/Configurable-Spectrograms, ``CS/`` =
``src/configurable_spectrograms/``) is pure Python; its arithmetic lives in
numpy 2.3.5 (installed here, so numpy itself pins ``nansum`` and
``nanpercentile``) and matplotlib 3.11.1 (NOT installable here: ``uv.lock:710``;
``Normalize`` / ``LogNorm`` / ``Colormap.__call__`` are restated from the
published algorithm -- **parity unpinned** at that boundary, see DESIGN.md).

Pinning status
--------------
* ``nansum_*``        : pinned against ``np.nansum`` (tests/test_oracle.py).
* ``nanpercentile``   : pinned against ``np.nanpercentile`` and the reference
                        doctests ``CS/percentile_utils.py:81-85``.
* ``round_extrema``/``extrema_overrides``: pinned by the reference doctests
                        ``CS/percentile_utils.py:32-35``, ``CS/fast/extrema.py:52-56``.
* ``panel_*``/``extrema_*``: pinned against the UNMODIFIED reference run under
                        the stubs in ``oracle/stubs.py`` (golden fixtures in
                        ``tests/golden/``, generator committed beside them).
* ``normalize``/``lognorm``/``colormap_index``: parity unpinned (matplotlib absent).
"""

from __future__ import annotations

import math

import numpy as np

# ----------------------------------------------------------------------------
# R1  np.nansum(axis=1) summation orders (CS/constants.py:12, called at
#     CS/plotting.py:188, CS/fast/plotting.py:128,278, CS/fast/extrema.py:259)
# ----------------------------------------------------------------------------


def nansum_layout_a(cube: np.ndarray, select: np.ndarray | None = None) -> np.ndarray:
    """Layout A: C-contiguous (T,P,E), reduce axis 1 = plain ascending-p chain.

    ``select`` is a boolean (P,) membership mask standing for the reference's
    gather ``data[:, mask, :]`` (``CS/fast/plotting.py:127``); an empty
    selection sums to +0.0 like ``np.nansum`` of a zero-length axis.
    """
    T, P, E = cube.shape
    D = cube.dtype.type
    idx = np.arange(P) if select is None else np.flatnonzero(select)
    if idx.size == 0:
        return np.zeros((T, E), dtype=cube.dtype)
    # the reduction is seeded with the identity +0.0 (np.sum([-0.0]) == +0.0)
    acc = np.zeros((T, E), dtype=cube.dtype)
    with np.errstate(invalid="ignore", over="ignore"):
        for p in idx:
            x = cube[:, p, :]
            acc = (acc + np.where(np.isnan(x), D(0), x)).astype(cube.dtype)
    return acc


def _pairwise_1d(a: np.ndarray) -> np.floating:
    """numpy's pairwise_sum for a contiguous 1-D run (block 128, 8 accumulators)."""
    n = a.shape[0]
    D = a.dtype.type
    if n < 8:
        acc = D(-0.0)  # numpy seeds the short loop with -0.0 so the sign of zero survives
        for i in range(n):
            acc = D(acc + a[i])
        return acc
    if n <= 128:
        r = [D(a[k]) for k in range(8)]
        i = 8
        while i < n - (n % 8):
            for k in range(8):
                r[k] = D(r[k] + a[i + k])
            i += 8
        res = D(D(D(r[0] + r[1]) + D(r[2] + r[3])) + D(D(r[4] + r[5]) + D(r[6] + r[7])))
        while i < n:
            res = D(res + a[i])
            i += 1
        return res
    n2 = n // 2
    n2 -= n2 % 8
    return D(_pairwise_1d(a[:n2]) + _pairwise_1d(a[n2:]))


def nansum_layout_b(cube_tep: np.ndarray, select: np.ndarray | None = None) -> np.ndarray:
    """Layout B: the reduced (pitch) axis is memory-contiguous.

    ``cube_tep`` is the stored (T,E,P) array whose transposed *view*
    (``CS/cdf_utils.py:254-255``) the reference collapses along axis 1.
    A gathered subset (``data[:, mask, :]`` on the view) is a fresh
    C-contiguous (T,P',E) copy, i.e. layout A -- handled by the caller.
    """
    assert select is None
    T, E, P = cube_tep.shape
    z = np.where(np.isnan(cube_tep), cube_tep.dtype.type(0), cube_tep)
    out = np.empty((T, E), dtype=cube_tep.dtype)
    D0 = cube_tep.dtype.type(0)
    with np.errstate(invalid="ignore", over="ignore"):
        for t in range(T):
            for e in range(E):
                out[t, e] = D0 + _pairwise_1d(z[t, e])  # identity seed: -0.0 -> +0.0
    return out


def nansum_layout_b_vec(cube_tep: np.ndarray) -> np.ndarray:
    """Vectorised layout B for n = P <= 128 (same order as :func:`_pairwise_1d`)."""
    T, E, P = cube_tep.shape
    assert 8 <= P <= 128
    z = np.where(np.isnan(cube_tep), cube_tep.dtype.type(0), cube_tep)
    with np.errstate(invalid="ignore", over="ignore"):
        r = [z[..., k].copy() for k in range(8)]
        i = 8
        while i < P - (P % 8):
            for k in range(8):
                r[k] = r[k] + z[..., i + k]
            i += 8
        res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
        while i < P:
            res = res + z[..., i]
            i += 1
        res = res + cube_tep.dtype.type(0)  # identity seed: -0.0 -> +0.0
    return res.astype(cube_tep.dtype)


# ----------------------------------------------------------------------------
# R4  np.nanpercentile(matrix, p) flattened, method "linear", arithmetic in the
#     array dtype (CS/percentile_utils.py:87-88; numpy
#     lib/_function_base_impl.py:_quantile/_lerp, _nanfunctions_impl.py)
# ----------------------------------------------------------------------------


def percentile_rank(n: int, p, dtype) -> tuple[int, int, np.floating]:
    """(lo, hi, gamma) for ``n`` valid samples at percentile ``p`` in dtype ``D``."""
    D = np.dtype(dtype).type
    q = D(p) / D(100)
    v = D(n - 1) * q
    if v >= n - 1:  # numpy clamps both neighbours to the last element
        lo = hi = n - 1
    elif v < 0:
        lo = hi = 0
    else:
        lo = int(np.floor(v))
        hi = lo + 1
    g = D(v - D(lo)) if not (v >= n - 1) else D(v - np.floor(v))
    return lo, min(hi, n - 1), g


def lerp(a, b, g, dtype):
    D = np.dtype(dtype).type
    with np.errstate(invalid="ignore", over="ignore"):
        d = D(D(b) - D(a))
        r = D(D(a) + D(d * D(g)))
        if g >= 0.5:
            r = D(D(b) - D(d * D(D(1) - D(g))))
    return r


def nanpercentile(values: np.ndarray, p) -> float:
    """Restated ``float(np.nanpercentile(values, p))`` (flattened)."""
    a = np.asarray(values).ravel()
    s = np.sort(a[~np.isnan(a)])
    n = s.size
    if n == 0:
        return float("nan")
    lo, hi, g = percentile_rank(n, p, a.dtype)
    return float(lerp(s[lo], s[hi], g, a.dtype))


def compute_percentile_bounds(matrix, low=1, high=99, z_min=None, z_max=None):
    """``CS/percentile_utils.py:47-89``."""
    lo = float(z_min) if z_min is not None else nanpercentile(matrix, low)
    hi = float(z_max) if z_max is not None else nanpercentile(matrix, high)
    return lo, hi


def round_extrema(value, direction: str) -> float:
    """``CS/percentile_utils.py:8-44`` (2-significant-digit ceil/floor)."""
    if value == 0:
        return 0.0
    factor = 10 ** (math.floor(math.log10(abs(value))) - 1)
    if direction == "up":
        return float(math.ceil(value / factor) * factor)
    if direction == "down":
        return float(math.floor(value / factor) * factor)
    raise ValueError(f"Invalid direction: {direction}")


def extrema_overrides(global_extrema, inst, y_scale, z_scale):
    """``CS/fast/extrema.py:26-70``."""
    if not isinstance(global_extrema, dict):
        return None, None, None, None
    k = f"{inst}_{y_scale}_{z_scale}"

    def r(v, d):
        return round_extrema(v, d) if v is not None else None

    return (
        r(global_extrema.get(f"{k}_y_min"), "down"),
        r(global_extrema.get(f"{k}_y_max"), "up"),
        r(global_extrema.get(f"{k}_z_min"), "down"),
        r(global_extrema.get(f"{k}_z_max"), "up"),
    )


# ----------------------------------------------------------------------------
# R3 + R8  make_spectrogram numeric path (CS/plotting.py:183-329)
# ----------------------------------------------------------------------------


def panel(
    x,
    y,
    cube,
    *,
    x_min=None,
    x_max=None,
    center=None,
    window=None,
    y_min=0,
    y_max=4000,
    z_scale=None,
    z_min=None,
    z_max=None,
    collapse_axis=1,
):
    """Numeric result of one ``make_spectrogram`` call.

    Returns ``None`` when the reference returns ``(None, None)``; else a dict
    with the matrix handed to ``imshow`` (E' x T', clamped), ``vmin``, ``vmax``,
    ``mode`` and the surviving x / y axes.
    """
    x = np.asarray(x)
    y = np.asarray(y)
    cube = np.asarray(cube)
    with np.errstate(invalid="ignore", over="ignore"):
        collapsed = np.nansum(cube, axis=collapse_axis)  # :188
    nan_col = ~np.all(np.isnan(collapsed), axis=0)  # :191
    valid = (y >= y_min) & (y <= y_max)  # :192
    keep = nan_col & valid
    collapsed = collapsed[:, keep]
    y = y[keep]
    if collapsed.size == 0 or y.size == 0:  # :196
        return None
    if y[0] > y[-1]:  # :200-202
        y = y[::-1]
        collapsed = collapsed[:, ::-1]
    if center is not None and window is not None:  # :204-210
        half = window / 2
        zm = (x >= center - half) & (x <= center + half)
        x = x[zm]
        collapsed = collapsed[zm, :]
    if x_min is not None or x_max is not None:  # :212-219
        xm = np.ones_like(x, dtype=bool)
        if x_min is not None:
            xm &= x >= x_min
        if x_max is not None:
            xm &= x <= x_max
        x = x[xm]
        collapsed = collapsed[xm, :]
    m = collapsed.T  # :236
    if m.size == 0:  # :255 (the reference raises IndexError earlier at :253 when x is empty)
        return None
    with np.errstate(invalid="ignore"):
        zmin, zmax = compute_percentile_bounds(m, 1, 99, z_min, z_max)  # :259
        fp = m[np.isfinite(m) & (m > 0)]
        safe_vmin = np.nanmin(fp) if fp.size > 0 else 1e-10  # :261-262
    out = clamp_for_imshow(m, z_scale, zmin, zmax, safe_vmin)
    out.update(x=x, y=y, safe_vmin=float(safe_vmin))
    return out


def clamp_for_imshow(m, z_scale, zmin, zmax, safe_vmin):
    """The z clamps of ``make_spectrogram`` (``CS/plotting.py:276-278`` log, ``:307-315`` linear) on the
    matrix handed to ``imshow``, given the percentile bounds and ``safe_vmin`` already resolved."""
    with np.errstate(invalid="ignore"):
        if z_scale == "log":
            zmin = float(max(zmin, safe_vmin, 1e-10))  # :276
            zmax = float(zmax)
            m = np.where(~np.isfinite(m) | (m <= 0), zmin, m)  # :278
            mode = "log"
        else:
            zmin = float(zmin)
            zmax = float(zmax)
            m = np.where(np.isnan(m), zmin, m)  # :310
            m = np.where(np.isneginf(m), zmin, m)
            m = np.where(np.isposinf(m), zmax, m)
            if not (np.isfinite(zmin) and np.isfinite(zmax) and zmax > zmin):  # :313-315
                zmin = float(np.nanmin(m))
                zmax = float(np.nanmax(m))
            mode = "linear"
    return {"matrix": m, "vmin": zmin, "vmax": zmax, "mode": mode}


# ----------------------------------------------------------------------------
# R9  matplotlib Normalize / LogNorm / Colormap.__call__ index math.
#     PARITY UNPINNED: matplotlib 3.11.1 (uv.lock:710-711) is not installed; the
#     algorithm below restates colors.py (Normalize.__call__, the
#     make_norm_from_scale(LogScale, nonpositive="mask") __call__ and
#     Colormap._get_rgba_and_mask) as published.  In-place ``-=``/``/=`` on a
#     float32 array with np.float64 scalars computes in float64 and rounds to
#     float32 (NEP 50), hence the explicit casts.
# ----------------------------------------------------------------------------

I_UNDER, I_OVER, I_BAD = 256, 257, 258


def log10_like(values: np.ndarray, native: bool = False) -> np.ndarray:
    """``np.log10`` in the array dtype.

    numpy's float32 ``log10`` is libm/SVML dependent and not correctly
    rounded; the product defines the transform as the correctly rounded
    float32 of the float64 logarithm, which is what ``native=False`` gives.
    ``native=True`` is whatever this machine's numpy does (flip-count tests).
    """
    with np.errstate(divide="ignore", invalid="ignore"):
        if native or values.dtype == np.float64:
            return np.log10(values)
        return np.log10(values.astype(np.float64)).astype(values.dtype)


def normalize(matrix: np.ndarray, vmin: float, vmax: float) -> np.ndarray:
    D = matrix.dtype
    if vmin == vmax:
        return np.zeros_like(matrix)
    if vmin > vmax:
        raise ValueError("minvalue must be less than or equal to maxvalue")
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        x = (matrix.astype(np.float64) - np.float64(vmin)).astype(D)
        x = (x.astype(np.float64) / (np.float64(vmax) - np.float64(vmin))).astype(D)
    return x


def lognorm(matrix: np.ndarray, vmin: float, vmax: float, native_log: bool = False) -> np.ndarray:
    """Returns the normalised array; invalid (non-finite) entries are NaN (= masked)."""
    D = matrix.dtype
    if vmin > vmax:
        raise ValueError("vmin must be less or equal to vmax")
    if vmin == vmax:
        return np.zeros_like(matrix)
    t = log10_like(matrix, native=native_log)
    with np.errstate(divide="ignore", invalid="ignore"):
        t_vmin, t_vmax = np.log10(np.array([vmin, vmax], dtype=np.float64))
    if not np.isfinite([t_vmin, t_vmax]).all():
        raise ValueError("Invalid vmin or vmax")
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        t = (t.astype(np.float64) - t_vmin).astype(D)
        t = (t.astype(np.float64) / (t_vmax - t_vmin)).astype(D)
    return np.where(np.isfinite(t), t, np.nan).astype(D)


def colormap_index(x: np.ndarray, n: int = 256) -> np.ndarray:
    """``Colormap._get_rgba_and_mask`` index plane (uint16; 256/257/258 = under/over/bad)."""
    with np.errstate(invalid="ignore", over="ignore"):
        xa = x * x.dtype.type(n)
        xa = np.where(xa == n, x.dtype.type(n - 1), xa)
        under = xa < 0
        over = xa >= n
        bad = np.isnan(xa)
        idx = np.where(bad | under | over, 0, xa).astype(np.int64)
    idx[under] = I_UNDER
    idx[over] = I_OVER
    idx[bad] = I_BAD
    return idx.astype(np.uint16)


def lut_with_extremes(lut256: np.ndarray) -> np.ndarray:
    """(259,4) uint8: 256 colours + under (=lut[0]) + over (=lut[255]) + bad (0,0,0,0)."""
    lut = np.zeros((259, 4), dtype=np.uint8)
    lut[:256] = lut256
    lut[I_UNDER] = lut256[0]
    lut[I_OVER] = lut256[255]
    return lut


def rasterise(panel_result: dict, lut259: np.ndarray, native_log: bool = False):
    """(index plane uint16, RGBA uint8) that ``imshow`` would colour at cell resolution."""
    m = panel_result["matrix"]
    if panel_result["mode"] == "log":
        x = lognorm(m, panel_result["vmin"], panel_result["vmax"], native_log=native_log)
    else:
        x = normalize(m, panel_result["vmin"], panel_result["vmax"])
    idx = colormap_index(x)
    return idx, lut259[idx]


# ----------------------------------------------------------------------------
# R5 + R6  compute_global_extrema (CS/fast/extrema.py:73-366) without file IO.
#     ``files`` is the ascending-orbit sequence of
#     (orbit, {inst: (energy(E,), cube(T,P,E))}); ``state`` is the JSON cache dict.
#
#     Control flow restated verbatim, including the quirk that the
#     linear/linear combo re-uses ITS OWN keys from the second orbit on
#     (``ll_y_key in extrema_state`` at :208-224 is true as soon as the first
#     orbit's step has stored them), so on a fresh cache linear/linear scans only
#     the first orbit per instrument, while e.g. linear/log scans every orbit
#     with the running max and stores linear-domain values under its own keys.
# ----------------------------------------------------------------------------


def global_extrema(
    files,
    instrument_order,
    y_scale="linear",
    z_scale="linear",
    state=None,
    max_percentile=95.0,
    compute_mins=False,
    log_floor_cutoff=0.1,
    log_floor_value=-1.0,
):
    from collections import defaultdict

    instrument_order = tuple(instrument_order)
    state = {} if state is None else state

    def safe_log(v):  # :151-161
        if v is None:
            return float(log_floor_value)
        try:
            v = float(v)
        except (TypeError, ValueError):
            return float(log_floor_value)
        if not np.isfinite(v) or v <= log_floor_cutoff:
            return float(log_floor_value)
        return float(np.log10(v))

    orbit_numbers = [o for o, _ in files]
    per_orbit = dict(files)
    counts = {i: defaultdict(int) for i in instrument_order}
    blocks = {i: [] for i in instrument_order}
    totals = {i: sum(1 for o in orbit_numbers if i in per_orbit[o]) for i in instrument_order}
    last_key = f"{y_scale}_{z_scale}_last_orbit"
    lv = state.get(last_key, -1)
    last = int(lv) if isinstance(lv, (int, float)) else -1
    for orbit_index, orbit in enumerate(orbit_numbers):
        if orbit <= last:  # :192
            continue
        for inst in instrument_order:
            kp = f"{inst}_{y_scale}_{z_scale}"
            pk = f"{kp}_extrema_progress"
            pe = state.get(pk)
            if isinstance(pe, dict) and pe.get("complete"):
                continue
            y_log, z_log = y_scale == "log", z_scale == "log"
            lly, llz = f"{inst}_linear_linear_y_max", f"{inst}_linear_linear_z_max"
            llymin, llzmin = f"{inst}_linear_linear_y_min", f"{inst}_linear_linear_z_min"
            if not y_log and lly in state:  # :208-213
                state[f"{kp}_y_max"] = state[lly]
                state[f"{kp}_y_min"] = state.get(llymin, 0)
            elif y_log and lly in state:
                state[f"{kp}_y_max"] = safe_log(state[lly])
                state[f"{kp}_y_min"] = log_floor_value
            if not z_log and llz in state:  # :215-220
                state[f"{kp}_z_max"] = state[llz]
                state[f"{kp}_z_min"] = state.get(llzmin, 0)
            elif z_log and llz in state:
                state[f"{kp}_z_max"] = safe_log(state[llz])
                state[f"{kp}_z_min"] = log_floor_value
            if lly in state and llz in state:  # :222-243
                state[pk] = {"processed_index": max(totals[inst] - 1, -1), "total": totals[inst], "complete": True}
                for i2 in instrument_order:
                    state.pop(f"{i2}_{y_scale}_{z_scale}_last_orbit", None)
                state[last_key] = max(orbit_numbers) if orbit_numbers else -1
                continue
            if inst in per_orbit[orbit]:  # :248-268
                energy, cube = per_orbit[orbit][inst]
                with np.errstate(invalid="ignore", over="ignore"):
                    c = np.nansum(cube, axis=1)
                m = np.isfinite(c) & (c > 0)
                per_bin = m.sum(axis=0)
                for ev, cnt in zip(energy, per_bin, strict=False):
                    if cnt:
                        counts[inst][float(ev)] += int(cnt)
                pos = c[m]
                if pos.size:
                    blocks[inst].append(pos)
            cand_e = 0.0
            if counts[inst]:  # :270-278
                es = sorted(counts[inst].keys())
                cum = np.cumsum(np.array([counts[inst][e] for e in es]))
                target = 0.99 * cum[-1]
                idx = min(np.searchsorted(cum, target, side="right"), len(es) - 1)
                cand_e = float(es[idx])
            cand_z = 0.0
            if blocks[inst]:  # :280-285
                agg = np.concatenate(blocks[inst])
                fp = agg[np.isfinite(agg) & (agg > 0)]
                if fp.size:
                    cand_z = nanpercentile(fp, max_percentile)
            prev_e = state.get(f"{kp}_y_max")
            prev_z = state.get(f"{kp}_z_max")
            me = max(float(prev_e), cand_e) if isinstance(prev_e, (int, float)) else cand_e
            mz = max(float(prev_z), cand_z) if isinstance(prev_z, (int, float)) else cand_z
            me = int(min(4000, math.ceil(me)))  # :299
            mz = float(math.ceil(mz))  # :300
            if compute_mins and blocks[inst]:  # :302-309
                agg = np.concatenate(blocks[inst])
                fp = agg[np.isfinite(agg) & (agg > 0)]
                zmin_store = nanpercentile(fp, 1) if fp.size else 0.0
            else:
                zmin_store = 0
            state[f"{kp}_y_min"] = 0
            state[f"{kp}_y_max"] = me
            state[f"{kp}_z_min"] = zmin_store
            state[f"{kp}_z_max"] = mz
            state[pk] = {
                "processed_index": orbit_index,
                "total": totals[inst],
                "complete": orbit_index + 1 >= totals[inst],
            }
            for i2 in instrument_order:
                state.pop(f"{i2}_{y_scale}_{z_scale}_last_orbit", None)
            state[last_key] = orbit
    return state
