"""K4: figure mosaics composed and DEFLATE-encoded on the device decode (zlib, Pillow) to exactly
the image the host composer builds (figure.SpectrogramFigure.compose -- the oracle of this stage)."""

import io
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from configurable_spectrograms_b200 import _lib

    return _lib.Context(0)


def _twin_figures(rng, flat, specs, grid, lines):
    """The same figure twice: panels as host arrays, and as references into the device buffer; with the
    annotations of a real figure (labels, ticks, colour bars, title, footer, cusp lines and brackets)."""
    from configurable_spectrograms_b200.cusp_marking import draw_cusp_bracket_marker
    from configurable_spectrograms_b200.figure import DeviceRaster, SpectrogramFigure

    figs = []
    n_rows, n_cols = grid
    for device in (False, True):
        fig = SpectrogramFigure(figsize=(12 * n_cols, 3 * n_rows))
        for k, (cell, off, ne, nt) in enumerate(specs):
            ax = fig.add_subplot(n_rows, n_cols, cell)
            host = flat[off : off + ne * nt].view(np.uint8).reshape(ne, nt, 4)
            x0 = 10957.0 + 0.01 * k
            x1 = x0 + nt * 2.5 / 86400.0
            ax.set_xlim(x0 - (0.001 if k % 2 else 0.0), x1 + (0.002 if k % 2 else 0.0))  # odd panels: image inside wider limits
            im = ax.imshow(DeviceRaster(off, ne, nt) if device else host, extent=(x0, x1, 4.0, 4000.0), cmap="turbo",
                           norm="log" if k % 2 == 0 else None, vmin=1.0, vmax=2400.0)
            fig.colorbar(im, ax=ax, label="Counts", ticks=[1, 10, 100, 1000] if k % 2 == 0 else None)
            ax.set_xlabel("Time (UTC)")
            ax.set_ylabel("Energy (eV)", fontsize=14)
            ax.set_yticks([0, 1000, 2000, 3000, 4000])
            ax.set_yticklabels(["0", "1000", "2000", "3000", "4000"])
            ax.xaxis.set_major_formatter("%H:%M:%S" if nt < 40 else "%H:%M")
            ax.tick_params(axis="both", which="major", labelsize=11, length=6)
            if k == 0:
                ax.set_title("Full", fontsize=14)
            marks = []
            for frac, width, colour in lines.get(k, []):
                marks.append(x0 + frac * (x1 - x0))
                ax.axvline(marks[-1], color=colour, linewidth=width)
            if marks:
                draw_cusp_bracket_marker(ax, marks, caption="cusp")
        fig.suptitle(f"Orbit 13000 - figure with {len(specs)} panels", fontsize=16)
        fig.text(0.5, 0.01, "Data timespan: 2000-01-01 00:00:00 to 2000-01-01 00:33:20 UTC", ha="center", va="bottom", fontsize=11)
        fig.tight_layout(rect=(0, 0.06, 1, 0.95))
        figs.append(fig)
    return figs


def test_device_png_and_deferred_files_match_host_compose(ctx):
    from configurable_spectrograms_b200 import png

    rng = np.random.default_rng(12)
    # a colour-mapped look: few distinct colours, flat stretches, plus pure noise panels
    palette = rng.integers(0, 256, 300, dtype=np.uint32) | np.uint32(0xFF000000)
    shapes = [(74, 800), (74, 181), (74, 903), (60, 47), (3, 5), (74, 1500), (1, 1), (96, 2100), (74, 800)]
    offs, parts, pos = [], [], 0
    for i, (ne, nt) in enumerate(shapes):
        if i % 3 == 2:
            px = rng.integers(0, 2**32, ne * nt, dtype=np.uint64).astype(np.uint32)  # incompressible
        else:
            idx = np.clip((rng.normal(0, 1, (ne, nt)).cumsum(axis=1) * 3 + 150).astype(int), 0, 299)
            px = palette[idx].reshape(-1)
        offs.append(pos)
        parts.append(px)
        pos += (ne * nt + 3) & ~3
        parts.append(np.zeros(((ne * nt + 3) & ~3) - ne * nt, np.uint32))
    flat = np.concatenate(parts)
    d_rgba = ctx.to_device(flat)
    layouts = [
        # (grid, [(cell, panel)], {panel position: [(x, linewidth, colour)]})
        # lines: (fraction of the panel's time span, linewidth in points, colour)
        ((4, 2), [(1, 0), (2, 1), (3, 2), (5, 8), (6, 3), (7, 0)], {0: [(0.31, 4, "black"), (0.31, 2, "red")], 1: [(0.5, 4, "red")]}),
        ((1, 1), [(1, 5)], {0: [(1.0, 4, "red"), (0.0, 1, "black")]}),
        ((2, 2), [(1, 4), (4, 6)], {}),
        ((2, 1), [(1, 7), (2, 2)], {0: [(0.53, 4, "red"), (0.53, 1, "black")]}),
        ((1, 1), [], {}),
    ]
    host_figs, dev_figs = [], []
    for grid, cells, lines in layouts:
        specs = [(cell, offs[p], *shapes[p]) for cell, p in cells]
        h, d = _twin_figures(rng, flat, specs, grid, lines)
        host_figs.append(h)
        dev_figs.append(d)
    for budget, dpi in ((160_000, 100), (700, 100), (160_000, 200), (160_000, 37)):  # one group / several groups; three resolutions
        blobs = png.encode_figures_device(ctx, d_rgba.ptr, dev_figs, max_segments=budget, dpi=dpi)
        assert len(blobs) == len(host_figs)
        for blob, fig in zip(blobs, host_figs):
            want = fig.compose(dpi)
            got = png.decode_rgba(blob)
            assert got.shape == want.shape
            assert np.array_equal(got, want)
    # an independent decoder agrees, and the stream is a real zlib stream (Adler-32 verified by zlib)
    from PIL import Image

    for blob, fig in zip(blobs, host_figs):
        im = np.asarray(Image.open(io.BytesIO(blob)).convert("RGBA"))
        assert np.array_equal(im, fig.compose(37))
    # compression at display resolution: repeated lines and stretched cells shrink a lot
    blobs = png.encode_figures_device(ctx, d_rgba.ptr, dev_figs, dpi=200)
    sizes = [len(b) for b in blobs]
    raws = [f.compose(200).nbytes for f in host_figs]
    assert sizes[0] < 0.2 * raws[0]
    assert all(s < 0.5 * r + 2000 for s, r in zip(sizes, raws))
    # ---- deferred mode (the directory driver's): files through the native writer; the last group is completed
    # later, or given up -- after which the context encodes again
    import tempfile

    with tempfile.TemporaryDirectory() as tmp:
        paths = [f"{tmp}/f{k}.png" for k in range(len(dev_figs))]
        for budget in (160_000, 700):  # everything deferred / only the last of several groups
            handle = png.encode_figures_device(ctx, d_rgba.ptr, dev_figs, dpi=100, max_segments=budget, paths=paths, defer=True)
            with pytest.raises(RuntimeError, match="deferred encode is still open"):
                png.encode_figures_device(ctx, d_rgba.ptr, dev_figs[:1], dpi=100)
            for fut in handle.complete():
                fut.result()
            assert handle.complete() == handle.futures  # idempotent
            for path, fig in zip(paths, host_figs):
                assert np.array_equal(png.decode_rgba(open(path, "rb").read()), fig.compose(100))
                os.remove(path)
        handle = png.encode_figures_device(ctx, d_rgba.ptr, dev_figs, dpi=100, paths=paths, defer=True)
        handle.abandon()
        assert handle.complete() == [] and not any(os.path.exists(p) for p in paths)
        blobs = png.encode_figures_device(ctx, d_rgba.ptr, dev_figs, dpi=100)  # the context is free again
        assert np.array_equal(png.decode_rgba(blobs[0]), host_figs[0].compose(100))
