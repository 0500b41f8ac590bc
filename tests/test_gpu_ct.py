"""Dynamic half of the constant-time check (VERDICT r1 item 9): the number of warp instructions each secret-handling
kernel executes must not depend on the secrets.  tools/ct_target.py launches the ladders (per-key and shared-inversion
kernels), both scalar multiplications and the P-256 inversion / square-root kernels on all-zero, all-ones, low-bits and
random inputs of identical shape; `ncu --metrics smsp__inst_executed.sum` counts.  (The static half, tools/ct_audit.py,
runs in the CPU suite.)"""
import csv
import io
import os
import shutil
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
KERNELS = "k_rfc7748|k_ecnmul|k_inv_shared|k_field"


def counts(kind):
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.access(ncu, os.X_OK):
        pytest.skip("ncu not installed or not executable by this user")
    cmd = [ncu, "--metrics", "smsp__inst_executed.sum", "--clock-control", "none", "--csv", "-k", "regex:" + KERNELS,
           sys.executable, os.path.join(ROOT, "tools", "ct_target.py"), kind]
    try:
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    except PermissionError:
        pytest.skip("ncu cannot be run by this user")
    if "ERR_NVGPUCTRPERM" in r.stdout + r.stderr:
        pytest.skip("no permission to read GPU performance counters")
    assert r.returncode == 0 and ("done " + kind) in r.stdout, (r.stdout[-1500:], r.stderr[-1500:])
    txt = r.stdout[r.stdout.index('"ID"'):]
    out = []
    for row in csv.DictReader(io.StringIO(txt)):
        if row.get("Metric Name") == "smsp__inst_executed.sum":
            out.append((row["Kernel Name"].split("(")[0], int(row["Metric Value"].replace(",", ""))))
    return out


def test_executed_instructions_do_not_depend_on_secrets():
    base = counts("random")
    names = [k for k, _ in base]
    assert sum("k_rfc7748" in k for k in names) >= 4 and sum("k_ecnmul" in k for k in names) >= 2
    assert any("k_inv_shared" in k for k in names)
    for kind in ("zero", "ones", "lowbits"):
        got = counts(kind)
        assert [k for k, _ in got] == names
        diff = [(k, a, b) for (k, a), (_, b) in zip(base, got) if a != b]
        assert diff == [], (kind, diff)
