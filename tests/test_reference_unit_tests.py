"""The reference's OWN MTTKRP unit tests (tests/mttkrp_test.c, ctest): every fixture x every
mode x ONEMODE/TWOMODE/ALLMODE x NOTILE/DENSETILE(all depths), CSF MTTKRP vs the COO gold
mttkrp_stream, abs tol 1e-10, 7 OpenMP threads.

  * reftest_mttkrp_cpu : linked against the reference's kernels (sanity: the oracle build and
                         the golden fixtures are what the reference expects) -- runs anywhere;
  * reftest_mttkrp_gpu : the SAME test objects, but splatt_mttkrp_csf / _alloc_ws / _free_ws
                         resolve from libsplatt_b200.so (objcopy rename, INTEGRATION.md option A):
                         the reference's test-suite judging our CUDA kernels.

Both binaries are built by oracle/build_ref.sh to read their fixtures from
splatt_b200_fixtures/ under the working directory; they are rewritten there from
tests/golden/*.npz and a relocated copy of the binary (tests/util.py) runs in a temporary
directory."""
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import ref
from tests.util import relocated_binary

GOLD = Path(__file__).parent / "golden"
CPU = ref.CLI_PATH.parent / "reftest_mttkrp_cpu"
GPU = ref.CLI_PATH.parent / "reftest_mttkrp_gpu"


def _write_fixtures(fix):
    fix.mkdir()
    for name in ("small", "med", "small4", "med4", "med5"):
        out = fix / f"{name}.tns"
        z = np.load(GOLD / f"{name}.npz")
        ind, vals = z["ind"], z["vals"]
        with open(out, "w") as f:
            for n in range(len(vals)):
                f.write(" ".join(str(int(ind[m][n]) + 1) for m in range(ind.shape[0])))
                f.write(f" {float(vals[n])!r}\n")


def _run(exe, wd):
    _write_fixtures(wd / "splatt_b200_fixtures")
    exe, env = relocated_binary(exe, wd)
    # the tests ask for 7 threads, but their gold (mttkrp_stream) runs before the first
    # omp_set_num_threads call; on a 128-CPU host the default-sized team stalls in libgomp --
    # pin the default team size to what the tests intend
    env["OMP_NUM_THREADS"] = "7"
    try:
        r = subprocess.run([str(exe), "mttkrp"], capture_output=True, text=True, timeout=150, env=env,
                           cwd=wd)
    except subprocess.TimeoutExpired:
        # seen once with a default-sized (128-thread) OpenMP team: every thread asleep inside the
        # reference's CPU gold mttkrp_stream (backtrace: GOMP barrier) -- not a verdict on the kernels
        pytest.skip("the reference's CPU gold stalled in OpenMP on this host")
    m = re.search(r"RESULTS: (\d+) tests \((\d+) ok, (\d+) failed, (\d+) skipped\)", r.stdout)
    assert m, r.stdout[-2000:] + r.stderr[-2000:]
    return tuple(int(x) for x in m.groups()), r.stdout


@pytest.mark.skipif(not CPU.exists(), reason="oracle/_ref/reftest_mttkrp_cpu not built")
def test_reference_mttkrp_unit_tests_cpu(tmp_path):
    (total, ok, failed, skipped), out = _run(CPU, tmp_path)
    assert (total, ok, failed, skipped) == (7, 7, 0, 0), out[-1500:]


@pytest.mark.gpu
@pytest.mark.skipif(not GPU.exists(), reason="oracle/_ref/reftest_mttkrp_gpu not built")
def test_reference_mttkrp_unit_tests_on_libsplatt_b200(tmp_path):
    (total, ok, failed, skipped), out = _run(GPU, tmp_path)
    assert (total, ok, failed, skipped) == (7, 7, 0, 0), out[-1500:]
    for name in ("csf_one_notile", "csf_two_notile", "csf_all_notile", "csf_one_densetile_alldepth",
                 "csf_two_densetile_alldepth", "csf_all_densetile_alldepth"):
        assert re.search(rf"mttkrp:{name} \[OK\]", out), name
