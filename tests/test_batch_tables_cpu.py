"""engine.Batch's descriptor tables without a GPU: the row types follow the ABI mirror dtypes, planned rows
become the structured arrays the kernels read, and the table edits change only the field they own."""

from types import SimpleNamespace

import numpy as np
import pytest

from configurable_spectrograms_b200 import _lib, engine
from configurable_spectrograms_b200.engine import WANT_GEOMETRY, WANT_PERCENTILES, WANT_REDUCTIONS


class _HostContext:
    """What a Batch needs of a Context to plan and hand over its tables: the library's host-only functions,
    and uploads kept as host arrays instead of copied to a device."""

    def __init__(self):
        self.lib = _lib.load_library()

    def to_device(self, arr):
        return np.array(arr, copy=True)

    def alloc(self, nbytes):
        return SimpleNamespace(nbytes=nbytes)


@pytest.fixture
def batch():
    b = engine.Batch(_HostContext(), np.float32, n_groups=1)
    b.add_file(np.zeros((10, 3, 6), np.float32), np.array([1, 0, 1], np.uint8))  # Tp 12: sums of 2 x 6 x 12 -> 192
    b.add_file(np.zeros((7, 3, 5), np.float32), np.array([0, 1, 1], np.uint8))  # Tp 8, flags at 12
    return b


def _rows(table, expected):
    assert len(table) == len(expected)
    for row, want in zip(table, expected):
        for name in table.dtype.names:
            got = row[name]
            assert got == want.get(name, 0) or (np.isnan(got) and np.isnan(want[name])), (name, got, want)


def test_row_types_follow_the_abi_mirror():
    assert engine.RegionRow._fields == _lib.REGION.names
    assert engine.PanelRow._fields == _lib.PANEL.names
    assert engine.WindowRow._fields == _lib.FLAG_WINDOW.names


def test_planned_rows_become_the_kernel_tables(batch):
    b = batch
    r0 = b.add_region(0, 1, [5, 4, 3], want_pct=True, p_lo=2.0, p_hi=98.0)
    r1 = b.add_region(1, 0, [0, 2], rows=[1, 3, 4], want_pct=WANT_GEOMETRY)
    r2 = b.add_region(1, 1, [0, 2], t0=2, nt=3)
    slot = b.zslot(7.5)
    p0 = b.add_panel(r0, -1, True, 1.0, None)
    p1 = b.add_panel(r1, r0, False, None, slot, stat_region=r0)
    p2 = b.add_panel(r2, -1, False, 0.5, 2.5)
    b.add_window(1, 2, [4, 6])
    b.add_window(0, 1, (2, 5))
    b.upload_tables()

    assert b.d_regions.dtype == _lib.REGION and b.d_panels.dtype == _lib.PANEL and b.d_windows.dtype == _lib.FLAG_WINDOW
    assert list(b.d_pool) == [5, 4, 3, 1, 3, 4, 0, 2, 4, 6]  # cols of r0, rows of r1, cols of r1 / r2, window rows
    _rows(b.d_regions, [
        dict(mat_off=72, ld=12, t0=0, nt=10, rows_off=-1, cols_off=0, ne=3, want_pct=WANT_PERCENTILES, p_lo=2.0, p_hi=98.0),
        dict(mat_off=192, ld=8, t0=0, nt=3, rows_off=3, cols_off=6, ne=2, want_pct=WANT_GEOMETRY, p_lo=1.0, p_hi=99.0),
        dict(mat_off=192 + 5 * 8, ld=8, t0=2, nt=3, rows_off=-1, cols_off=6, ne=2, want_pct=WANT_REDUCTIONS, p_lo=1.0, p_hi=99.0),
    ])
    # the device table holds the panels free of z slots first; first_block counts in that order
    blocks = [b.ctx.lib.csg_raster_blocks(*b.panel_shape(p)) for p in (p0, p1, p2)]
    assert blocks[0] > 0 and blocks[1] > 0 and blocks[2] > 0
    assert list(b.d_panels["region"]) == [r0, r2, r1]
    assert list(b.d_block_panel) == [0] * blocks[0] + [1] * blocks[2] + [2] * blocks[1]
    nan = float("nan")
    _rows(b.by_panel(b.d_panels), [
        dict(region=r0, pct_region=-1, log_scale=1, first_block=0, z_min=1.0, z_max=nan, out_off=0, stat_region=-1,
             zmin_slot=-1, zmax_slot=-1),
        dict(region=r1, pct_region=r0, log_scale=0, first_block=blocks[0] + blocks[2], z_min=nan, z_max=7.5, out_off=32,
             stat_region=r0, zmin_slot=-1, zmax_slot=slot.slot),
        dict(region=r2, pct_region=-1, log_scale=0, first_block=blocks[0], z_min=0.5, z_max=2.5, out_off=40,
             stat_region=-1, zmin_slot=-1, zmax_slot=-1),
    ])
    assert [b.panel_offset(p) for p in (p0, p1, p2)] == [0, 32, 40]  # every panel 16-byte aligned
    assert [b.panel_region(p) for p in (p0, p1, p2)] == [r0, r1, r2]
    assert b.n_pixels == 48 and b.n_windows == 2
    _rows(b.d_windows, [dict(flags_off=12, t0=0, nt=2, rows_off=8, bit=2), dict(flags_off=0, t0=2, nt=5, rows_off=-1, bit=1)])


def test_require_stats_only_raises_in_the_documented_order(batch):
    order = [WANT_GEOMETRY, WANT_REDUCTIONS, WANT_PERCENTILES]
    pairs = [(start, asked) for start in range(3) for asked in range(3)]
    ids = [batch.add_region(0, 0, [1, 2], want_pct=order[start]) for start, _asked in pairs]
    batch.upload_tables()
    before = batch.d_regions
    for rid, (_start, asked) in zip(ids, pairs):
        batch.require_stats(rid, order[asked])
    batch.upload_tables()
    after = batch.d_regions
    assert list(after["want_pct"]) == [order[max(start, asked)] for start, asked in pairs]
    after["want_pct"] = before["want_pct"]
    assert after.tobytes() == before.tobytes()
    # a region nobody reads reductions of becomes geometry only; percentile and geometry regions stay
    for rid in ids:
        batch.drop_reductions(rid)
    batch.upload_tables()
    assert list(batch.d_regions["want_pct"]) == [WANT_GEOMETRY if order[max(s, a)] == WANT_REDUCTIONS else order[max(s, a)]
                                                 for s, a in pairs]


def test_set_stat_region_edits_that_field_only(batch):
    regions = [batch.add_region(f, g, [0, 1, 2], want_pct=True) for f in (0, 1) for g in (0, 1)]
    panels = [batch.add_panel(r, -1, bool(r % 2), 1.0, batch.zslot(4.0) if r == 1 else None) for r in regions]
    batch.upload_tables()
    before = batch.by_panel(batch.d_panels)
    batch.set_stat_region(panels[2], regions[0])
    batch.upload_tables()
    after = batch.by_panel(batch.d_panels)
    assert after["stat_region"][panels[2]] == regions[0]
    after["stat_region"][panels[2]] = before["stat_region"][panels[2]]
    assert after.tobytes() == before.tobytes()
