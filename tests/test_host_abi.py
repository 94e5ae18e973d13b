"""CPU-side checks of the drop-in boundary: libsrtb_b200.so loads, exports every symbol
include/srtb_b200.h declares, its host helpers agree with the oracle, and — with no GPU in this
container — the product path fails loudly instead of falling back to a CPU implementation."""
import re
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
HEADER = ROOT / "include" / "srtb_b200.h"


def declared_symbols():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    return sorted(set(re.findall(r"\b(srtb_b200_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import srtb_b200
    lib = srtb_b200.load_library()          # raises if the .so is missing: no fallback
    names = declared_symbols()
    assert len(names) >= 20
    out = subprocess.run(["nm", "-D", "--defined-only", str(srtb_b200.LIB_PATH)], capture_output=True, text=True,
                         check=True).stdout
    exported = set(re.findall(r"\bT (srtb_b200_[a-z0-9_]+)", out))
    assert set(names) <= exported, sorted(set(names) - exported)
    assert set(names) == set(srtb_b200.SYMBOLS), "python binding and header disagree"
    assert b"sm_100a" in lib.srtb_b200_version()


def test_library_is_sm100a_only():
    import srtb_b200
    r = subprocess.run(["cuobjdump", "-lelf", str(srtb_b200.LIB_PATH)], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = set(re.findall(r"sm_\d+a?", r.stdout))
    assert archs == {"sm_100a"}, archs


def test_no_cpu_fallback():
    import torch
    import srtb_b200
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(srtb_b200.SrtbError) as e:
        srtb_b200.Context(0)
    assert "no CPU fallback" in str(e.value)
    assert not hasattr(srtb_b200, "oracle")
    src = (ROOT / "simple-radio-telescope-backend_b200" / "srtb_b200" / "__init__.py").read_text()
    assert "oracle_lib" not in src and "import oracle" not in src


def test_product_never_links_the_oracle():
    import srtb_b200
    out = subprocess.run(["ldd", str(srtb_b200.LIB_PATH)], capture_output=True, text=True).stdout
    assert "srtb_oracle" not in out
    for f in (ROOT / "simple-radio-telescope-backend_b200" / "csrc").glob("*.cu*"):
        assert "oracle" not in f.read_text().lower(), f
    for f in (ROOT / "include").rglob("*.h*"):
        assert "oracle" not in f.read_text().lower(), f


def test_host_helpers_match_oracle(oracle):
    import srtb_b200
    for nc, c in [(1 << 25, 1 << 11), (1 << 23, 1 << 11), (512, 16), (1 << 29, 1 << 11)]:
        assert srtb_b200.norm_coefficient(nc, c) == oracle.norm_coefficient(nc, c)
    for s in ["11-12, 15-90, 233-235, 1176-1177", "", "1418-1422", "1-2-3, 5-6", " 7 - 8 ,9-10", "a-b, 1-2", "3-4,"]:
        assert srtb_b200.eval_rfi_ranges(s) == oracle.eval_rfi_ranges(s), s
    cases = [(11.0, 12.0, 0.0, 1499.0, 1500), (1418.0, 1422.0, 1437.0, -64.0, 1 << 29),
             (1422.0, 1418.0, 1437.0, -64.0, 1 << 12), (100.0, 200.0, 1000.0, 500.0, 4096),
             (1400.0, 1600.0, 1000.0, 500.0, 4096), (1018.0, 1022.0, 1000.0, 400.0, 1 << 25),
             (1000.0, 1500.0, 1000.0, 500.0, 1 << 23)]
    for args in cases:
        assert srtb_b200.rfi_range_to_bins(*args) == oracle.rfi_range_to_bins(*args), args
    for args in [(1 << 26, 1 << 11, 1000.0, 500.0, 1e9, 5.0, True), (1 << 24, 1 << 11, 1000.0, 500.0, 1e9, 56.778, True),
                 (1 << 30, 1 << 11, 1437.0, -64.0, 128e6, -478.80, True), (1 << 30, 1 << 11, 1437.0, -64.0, 128e6, -478.80, False),
                 (1 << 28, 1 << 15, 1000.0, 500.0, 1e9, 100.0, True)]:
        assert srtb_b200.nsamps_reserved(*args) == oracle.nsamps_reserved(*args), args


def test_cpp_pipe_framework():
    """the re-hosted srtb::pipeline framework (include/srtb/pipeline/framework): queues, start_pipe,
    fan-out, tee, loose out, composite_pipe, stop semantics — tests/cpp/test_framework.cpp"""
    d = ROOT / "tests" / "cpp"
    subprocess.run(["make", "-C", str(d), "test_framework"], check=True, capture_output=True)
    r = subprocess.run([str(d / "test_framework")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "framework ok" in r.stdout, r.stderr


def test_cpp_host_next(tmp_path):
    """SURVEY section 8(f) host pieces: cfg loader + expression grammar, NPY writer (tests/cpp/test_host_next.cpp);
    the files it writes are read back with numpy"""
    import numpy as np
    d = ROOT / "tests" / "cpp"
    subprocess.run(["make", "-C", str(d), "test_host_next"], check=True, capture_output=True)
    # the reference's two example .cfg files, stored verbatim under tests/golden, are parsed as they ship
    r = subprocess.run([str(d / "test_host_next"), str(tmp_path), str(ROOT / "tests" / "golden")], capture_output=True,
                       text=True, timeout=120, env={"SRTB_LOG_LEVEL": "1", "PATH": "/usr/bin:/bin"})
    assert r.returncode == 0 and "host next ok" in r.stdout, r.stderr[-2000:]
    a = np.load(tmp_path / "srtb_test.npy")
    assert a.shape == (2, 3) and a.dtype == np.complex64 and a[1, 2] == 5 - 5j
    assert np.load(tmp_path / "srtb_test_1d.npy").tolist() == [1.0, 2.0, 3.0]
