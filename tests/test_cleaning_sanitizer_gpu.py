"""Point-cloud cleaning under compute-sanitizer (memcheck + racecheck) on a tiny cloud (tests/sanitizer_clean_target.py)."""
import os
import shutil
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _sanitizer():
    return shutil.which("compute-sanitizer") or (
        "/usr/local/cuda/bin/compute-sanitizer" if os.path.exists("/usr/local/cuda/bin/compute-sanitizer") else None)


@pytest.mark.parametrize("tool", ["memcheck", "racecheck"])
def test_cleaning_is_clean_under_compute_sanitizer(lib, tool):
    exe = _sanitizer()
    if exe is None:
        pytest.skip("compute-sanitizer not installed")
    # only the library's own kernels (all live in anonymous namespaces of libg2pc.so) are instrumented
    # --report-api-errors no: the CUDA runtime's lazy module loading probes kernels with cuKernelGetFunction and handles
    # the INVALID_HANDLE return itself; memcheck would otherwise count that host-API return code as an error
    cmd = [exe, "--tool", tool, "--kernel-name", "kns=_GLOBAL__N_"] + \
          (["--report-api-errors", "no"] if tool == "memcheck" else []) + ["--print-limit", "5", sys.executable,
           os.path.join(HERE, "sanitizer_clean_target.py")]
    try:
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    except subprocess.TimeoutExpired:
        pytest.skip("compute-sanitizer run exceeded 15 minutes on this box")
    tail = r.stdout[-3000:]
    assert "SANITIZER_TARGET_OK" in r.stdout, tail
    if tool == "racecheck":
        assert "RACECHECK SUMMARY: 0 hazards displayed (0 errors, 0 warnings)" in r.stdout, tail
    else:
        assert "ERROR SUMMARY: 0 errors" in r.stdout, tail
