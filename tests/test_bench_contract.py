"""The reference arm of bench.py runs without a GPU: its JSON line must keep the contract the
driver parses (metric/unit/impl/e2e/cpu_baseline keys; one line on stdout)."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference",
                          "--gpus", "1", "--steps", "1", "--warmup", "1", "--cpu-batch", "32"],
                         capture_output=True, text=True, timeout=600, cwd=REPO,
                         env={**os.environ, "OMP_NUM_THREADS": "1"})       # as under torchrun
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("samples/sec")
    assert d["unit"] == "samples/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    # the unmodified reference when it is importable (/root/reference or oracle/_ref), else the port
    from oracle.ref_shim import reference_available
    assert cb["kind"] == ("reference" if reference_available() else "port")
    assert cb["value"] == d["value"] and cb["cores"] >= 1 and "batch 32" in cb["sample"]
    assert d["gpu_launches"] == 0 and d["dtype"] == "f32" and d["vs_baseline"] is None


def test_other_ranks_of_the_reference_arm_exit_quietly():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=REPO,
                         env={**os.environ, "RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_falls_back_to_the_port_without_the_reference(tmp_path):
    """Neither /root/reference nor oracle/_ref: the restatement is timed and says so."""
    code = ("import sys, json; sys.argv=['bench.py','--impl','reference','--steps','1','--warmup','0','--cpu-batch','16'];"
            "sys.path.insert(0, %r); import oracle.ref_shim as rs; rs.REFERENCE_DIR='/nonexistent'; rs.REFERENCE_ZIP='/nonexistent';"
            "import runpy; runpy.run_path(%r, run_name='__main__')" % (REPO, os.path.join(REPO, "bench.py")))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
    assert d["cpu_baseline"]["kind"] == "port" and d["value"] > 0


def test_resnet_workload_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--workload",
                          "resnet18", "--image", "32", "--steps", "1", "--warmup", "0", "--cpu-batch", "4"],
                         capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
    assert "ResNet-18" in d["config"]["workload"] and d["value"] > 0


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """--dump-outputs: float32 .npy files of what the last timed step returned, under 64 MB, and
    the same files from a second run with the same arguments."""
    import numpy as np
    dumps = []
    for run in range(2):
        d = tmp_path / ("run%d" % run)
        out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--gpus", "1", "--steps", "3",
                              "--warmup", "1", "--batch", "256", "--no-e2e", "--no-torch-baseline",
                              "--no-cpu-baseline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900, cwd=REPO)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
        assert line["steps"] == 3 and line["warmup"] == 1
        dumps.append({p.name: np.load(p) for p in sorted(d.iterdir())})
    first, second = dumps
    assert set(first) == {"loss_total.npy", "loss_cls.npy", "loss_reg.npy", "output_0.npy", "output_1.npy",
                          "master_weights_sample.npy"}, sorted(first)
    assert sum(a.nbytes for a in first.values()) <= 64 << 20
    assert first["output_0.npy"].size == 256 * 1000 and first["output_1.npy"].size == 256 * 64
    assert first["master_weights_sample.npy"].size == 1 << 22
    for name, a in first.items():
        assert a.dtype == np.float32 and np.isfinite(a).all(), name
        np.testing.assert_array_equal(a, second[name], err_msg=name)
