"""bench.py's contract with the driver, as far as it can be checked without a GPU: both arms describe the workload
with one and the same `config` object, and the reference arm (the reference's own generated C on the host cores)
prints a complete line."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)


def test_workload_config_is_one_function_of_keys_and_world():
    import bench
    a = bench.workload_config(1 << 20, 1)
    assert a["workload"] == "batched X25519 (rfc7748) 2^20 random scalars/points per GPU"
    assert a["keys_per_gpu"] == 1 << 20 and a["keys_total"] == 1 << 20
    assert bench.workload_config(1 << 20, 8)["keys_total"] == 8 << 20
    assert set(a) == {"workload", "keys_per_gpu", "keys_total", "sharding", "l2", "inputs"}
    assert "model" not in a
    # one buffer set once three of them would pass 1 GiB
    assert "3 buffer sets" in a["l2"] and "one buffer set" in bench.workload_config(1 << 24, 1)["l2"]
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"config": workload_config(') == 2          # our arm and the reference arm


def test_dump_rows_are_a_fixed_sample():
    import numpy as np
    import bench
    assert np.array_equal(bench.dump_rows(1000), np.arange(1000))
    a = bench.dump_rows(1 << 20)
    assert a.size == bench.DUMP_ROWS and (np.diff(a) > 0).all() and a[-1] < 1 << 20
    assert np.array_equal(a, bench.dump_rows(1 << 20))
    assert bench.dump_rows(1 << 20, bench.DUMP_ROWS // 8).size == bench.DUMP_ROWS // 8
    assert bench.DUMP_ROWS * 32 * 4 <= 64 << 20


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """--dump-outputs writes the results of the last timed step (here the second of the three rotating input sets);
    every row must equal the plain-C restatement on the same inputs."""
    import numpy as np
    import bench
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    n, steps = 5000, 2
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0",
                        "--keys", str(n), "--no-extra", "--no-cpu-baseline", "--parity-keys", "0",
                        "--dump-outputs", str(tmp_path)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    j = json.loads(r.stdout.strip().splitlines()[-1])
    assert j["steps"] == steps and j["gpu_launches"] == steps
    got = np.load(tmp_path / "x25519_out.npy")
    assert got.dtype == np.float32 and got.shape == (n, 32)
    k, u = bench.make_inputs(n, 7748 + 1000 * ((steps - 1) % 3))
    assert np.array_equal(got.astype(np.uint8), c_oracle.rfc7748_batch("X25519", k, u))


def test_reference_arm_line():
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_X25519.so")):
        pytest.skip("oracle/_ref not built")
    import bench
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--keys", "4096"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-500:]
    j = json.loads(r.stdout.strip().splitlines()[-1])
    assert j["impl"] == "reference" and j["metric"] == "X25519 scalar-mults/s" and j["higher_is_better"] is True
    assert j["config"] == bench.workload_config(4096, 1)
    assert j["cpu_baseline"]["kind"] == "reference" and j["cpu_baseline"]["cores"] >= 1 and j["cpu_baseline"]["value"] == j["value"]
    assert j["e2e"] == {"value": j["value"], "unit": j["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["gpu_launches"] == 0 and j["value"] > 0
