"""The C-ABI boundary without a GPU: the library loads, exports every symbol include/csgpu.h declares,
and the product path fails loudly -- no CPU fallback -- when there is no device or no library."""

import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "csgpu.h")).read()
    return sorted(set(re.findall(r"CSG_API\s+[\w\s\*]+?\b(csg_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from configurable_spectrograms_b200 import _lib

    lib = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 70
    missing = [name for name in declared if not hasattr(lib, name)]
    assert missing == []
    # the ctypes binding table covers the header too, and the ABI versions agree
    assert sorted(_lib.SIGNATURES) == declared
    assert lib.csg_abi_version() == _lib.ABI_VERSION
    header = open(os.path.join(ROOT, "include", "csgpu.h")).read()
    assert f"#define CSG_ABI_VERSION {_lib.ABI_VERSION}" in header


def test_struct_layouts_match_the_header_sizes():
    from configurable_spectrograms_b200 import _lib

    sizes = {"csg_pool_item": (_lib.POOL_ITEM, 24), "csg_pool_query": (_lib.POOL_QUERY, 32), "csg_png_tile": (_lib.PNG_TILE, 48),
             "csg_png_vline": (_lib.PNG_VLINE, 16), "csg_png_canvas": (_lib.PNG_CANVAS, 32), "csg_pool_request": (_lib.POOL_REQUEST, 16),
             "csg_pool_sel": (_lib.POOL_SEL, 64), "csg_cdf_var": (_lib.CDF_VAR, 336), "csg_png_file": (_lib.PNG_FILE, 56),
             "csg_png_zero_segment": (_lib.PNG_ZERO_SEGMENT, 64)}
    header = open(os.path.join(ROOT, "include", "csgpu.h")).read()
    for name, (dtype, nbytes) in sizes.items():
        assert dtype.itemsize == nbytes, name
        assert re.search(r"\}\s*" + name + r"\s*;\s*/\*\s*" + str(nbytes) + " bytes", header), name


def test_no_device_means_an_error_not_a_fallback():
    import torch

    from configurable_spectrograms_b200 import _lib, engine

    if torch.cuda.is_available():
        pytest.skip("this box has a GPU")
    with pytest.raises(_lib.CsgError, match="no CPU fallback"):
        _lib.Context(0)
    with pytest.raises(_lib.CsgError):
        engine.nansum(np.zeros((2, 3, 4), np.float32), axis=1)


def test_missing_library_means_an_error(monkeypatch, tmp_path):
    from configurable_spectrograms_b200 import _lib

    with pytest.raises(_lib.CsgError, match="no CPU fallback"):
        _lib.load_library(str(tmp_path / "libcsgpu.so"))
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libcsgpu.so"))
    monkeypatch.setattr(_lib, "_lib", None)
    with pytest.raises(_lib.CsgError, match="no CPU fallback"):
        _lib.load_library()


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "configurable_spectrograms_b200")
    offenders = []
    for dirpath, _dirs, files in os.walk(pkg):
        for name in files:
            if name.endswith(".py"):
                text = open(os.path.join(dirpath, name)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M):
                    offenders.append(os.path.join(dirpath, name))
    assert offenders == []


def test_bench_reference_arm_prints_one_json_line():
    """``bench.py --impl reference`` (CPU only: the unmodified reference from ``oracle/_ref`` on the host cores
    where it has been copied, else the numpy port of its numeric path) on a one-orbit sample: exit 0, stdout =
    the ONE JSON line of the contract with the reference arm's keys -- the reference's own log lines (it prints
    ``[ERROR] Failed to load progress JSON`` to stdout) go to stderr."""
    import json
    import subprocess
    import sys

    from oracle import ref_driver as RD

    kind = "reference" if RD.available() else "port"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample-orbits", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:2000]
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "orbits/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == kind and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "orbits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["vs_baseline"] is None
