"""bench.py contract checks that need no GPU: the reference arm prints exactly ONE JSON line on stdout with the keys
the driver reads; the GPU arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-1500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-500:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Gsamples/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("Gsamples/s 8-bit baseband") and d["value"] > 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["gpu_launches"] == 0


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True,
                       text=True, timeout=600)
    assert r.returncode != 0 and r.stdout.strip() == ""
    assert "no CUDA device" in r.stderr or "no CPU fallback" in r.stderr


def test_bad_arguments_are_refused_before_any_work():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"],
                  ["--workload", "config5", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--warmup", "0", *extra],
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and r.stdout.strip() == "" and "error:" in r.stderr, extra


@pytest.mark.gpu
def test_dump_outputs_are_reproducible(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same arrays (float32 / float64, <= 64 MiB)"""
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "0",
                            "--workload", "config2", "--secondary", "none", "--no-cpu-baseline", "--stage-iters", "1",
                            "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-1500:]
        assert json.loads(r.stdout)["steps"] == 3
        dumps.append({p.stem: np.load(p) for p in sorted((tmp_path / run).glob("*.npy"))})
    a, b = dumps
    assert {"detect_summary", "signal_count", "series", "spectrum_sample", "spectrum_sample_index"} <= set(a)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert a["detect_summary"].shape == (1, 4) and a["detect_summary"][0, 2] == 1      # one stream, detector enabled
    assert np.abs(a["spectrum_sample"]).sum() > 0
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_both_arms_name_the_same_workload_and_default_is_the_j1644_shape():
    """the driver compares config.workload of the two arms; the default is BASELINE configs[2] (north star)"""
    sys.path.insert(0, str(ROOT))
    import bench
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-1500:]
    d = json.loads([l for l in r.stdout.splitlines() if l.strip()][0])
    assert d["config"]["workload"] == bench.workload_string("config3", bench.WORKLOADS["config3"])
    assert "2^26-sample blocks x2 stream(s)" in d["config"]["workload"] and "DM=562.05" in d["config"]["workload"]


def test_sweep_byte_model():
    """bytes the launched kernels must move per sample (bench.py roofline.chain.sweep_bytes)"""
    sys.path.insert(0, str(ROOT))
    import bench
    # raw-fused first sweep (b/8 + 4), two more R2C sweeps, one-kernel waterfall (8) + its tabulated chirp phases (2)
    assert bench.sweep_bytes_per_sample(bench.WORKLOADS["config2"]) == 1 + 4 + 8 + 8 + 8 + 2
    assert bench.sweep_bytes_per_sample(bench.WORKLOADS["config3"]) == 32    # two interleaved streams: 2 raw bytes per sample
    # packed 2-bit first sweep, three more R2C sweeps, long rows: chirp-on-load sweep + last sweep + column sums
    assert bench.sweep_bytes_per_sample(bench.WORKLOADS["config1"]) == 0.25 + 4 + 24 + 8 + 8 + 4
    # DM sweep: the R2C once, the waterfall group (rows of 2^15: 20 bytes) once per trial
    assert bench.sweep_bytes_per_sample(bench.WORKLOADS["config4"]) == 1 + 4 + 16 + 20 * 21


def test_numa_binding_is_a_no_op_when_the_topology_cannot_be_read():
    """multi-rank runs bind each rank to its GPU's NUMA node; an unknown device or node -1 must change nothing"""
    import os
    sys.path.insert(0, str(ROOT))
    import bench

    class Props:
        pci_domain_id, pci_bus_id, pci_device_id = 0, 0xfe, 0x1f   # no such PCI device

    class FakeTorch:
        class cuda:
            @staticmethod
            def get_device_properties(i):
                return Props()

    before = os.sched_getaffinity(0)
    assert bench.bind_to_gpu_numa_node(FakeTorch, 0) is None
    assert os.sched_getaffinity(0) == before

