"""BASELINE config 1: the UNMODIFIED reference CLI on a small 3-mode .tns, rank 16, one CPU
thread (reference plumbing, no GPU) -- proves the oracle build is a working SPLATT."""
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import ref
from tests.util import relocated_binary

GOLD = Path(__file__).parent / "golden"


def _write_tns(path, ind, vals):
    with open(path, "w") as f:
        for n in range(len(vals)):
            f.write(" ".join(str(int(ind[m][n]) + 1) for m in range(ind.shape[0])))   # 1-indexed
            f.write(f" {float(vals[n])!r}\n")


@pytest.mark.skipif(not ref.CLI_PATH.exists(), reason="oracle/_ref/splatt not built")
def test_reference_cli_cpd_on_med_fixture(tmp_path):
    z = np.load(GOLD / "med.npz")
    tns = tmp_path / "med.tns"
    _write_tns(tns, z["ind"], z["vals"])
    r = subprocess.run([str(ref.CLI_PATH), "cpd", str(tns), "-r", "16", "-t", "1", "--seed", "1",
                        "--nowrite", "-i", "5"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    out = r.stdout
    assert "DIMS=2425x10816x29567" in out and "NNZ=100000" in out
    fits = [float(x) for x in re.findall(r"fit = ([0-9.]+)", out)]
    assert len(fits) == 5
    assert abs(fits[-1] - 0.00087) < 2e-5          # SURVEY.md 8(c): fit 0.00087 after 5 its
    assert "Final fit" in out


@pytest.mark.skipif(not ref.CLI_PATH.exists(), reason="oracle/_ref/splatt not built")
def test_reference_cli_small_fixture(tmp_path):
    z = np.load(GOLD / "small.npz")
    tns = tmp_path / "small.tns"
    _write_tns(tns, z["ind"], z["vals"])
    r = subprocess.run([str(ref.CLI_PATH), "cpd", str(tns), "-r", "2", "-t", "1", "--seed", "1",
                        "--nowrite", "-i", "3"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    assert "DIMS=2x3x2" in r.stdout and "NNZ=6" in r.stdout


GPU_CLI = ref.CLI_PATH.parent / "splatt_gpu"


@pytest.mark.gpu
@pytest.mark.skipif(not GPU_CLI.exists(), reason="oracle/_ref/splatt_gpu not built")
@pytest.mark.parametrize("gpus", ["one", "list-0,0", "ngpus-2"])
@pytest.mark.parametrize("name,rank", [("med", 16), ("med4", 8), ("med5", 5)])
def test_reference_cli_linked_against_libsplatt_b200(tmp_path, name, rank, gpus):
    """The drop-in, end to end: the UNMODIFIED reference CLI (tt_read, csf_alloc, cpd_als_iterate,
    LAPACK solve -- all reference code) with only its four MTTKRP symbols resolved from
    libsplatt_b200.so (objcopy rename, INTEGRATION.md option A).  Same seed => the GPU-backed run
    prints the same fit trajectory as the pure-CPU run.  `gpus`: one GPU; the single-process
    multi-GPU engine on a device list that names GPU 0 twice (SPLATT_B200_DEVICES=0,0); and
    SPLATT_B200_NGPUS=2 on two real GPUs (gpurun --gpus 2) -- the reference's C host driving
    several GPUs through the unchanged C API (the shape of src/mpi/mpi_cpd.c:627-804)."""
    import torch
    gpu_cli, env = relocated_binary(GPU_CLI, tmp_path)
    if gpus == "list-0,0":
        env["SPLATT_B200_DEVICES"] = "0,0"
    elif gpus == "ngpus-2":
        if torch.cuda.device_count() < 2:
            pytest.skip("needs >= 2 GPUs (gpurun --gpus 2)")
        env["SPLATT_B200_NGPUS"] = "2"
    z = np.load(GOLD / f"{name}.npz")
    tns = tmp_path / f"{name}.tns"
    _write_tns(tns, z["ind"], z["vals"])
    args = ["cpd", str(tns), "-r", str(rank), "-t", "2", "--seed", "3", "--nowrite", "-i", "6",
            "--tol", "0"]
    cpu = subprocess.run([str(ref.CLI_PATH)] + args, capture_output=True, text=True, timeout=300)
    gpu = subprocess.run([str(gpu_cli)] + args, capture_output=True, text=True, timeout=300, env=env)
    assert cpu.returncode == 0 and gpu.returncode == 0, gpu.stderr
    f_cpu = re.findall(r"fit = ([0-9.]+)  delta = ([-+0-9.e]+)", cpu.stdout)
    f_gpu = re.findall(r"fit = ([0-9.]+)  delta = ([-+0-9.e]+)", gpu.stdout)
    assert len(f_cpu) == 6 and len(f_gpu) == 6
    for (a, da), (b, db) in zip(f_cpu, f_gpu):
        assert abs(float(a) - float(b)) <= 1e-5           # printed to 5 decimals
        assert abs(float(da) - float(db)) <= 1e-6 + 1e-3 * abs(float(da))
    final_cpu = float(re.search(r"Final fit: ([0-9.]+)", cpu.stdout).group(1))
    final_gpu = float(re.search(r"Final fit: ([0-9.]+)", gpu.stdout).group(1))
    assert abs(final_cpu - final_gpu) <= 1e-5


@pytest.mark.gpu
@pytest.mark.skipif(not GPU_CLI.exists(), reason="oracle/_ref/splatt_gpu not built")
@pytest.mark.parametrize("name", ["med", "med4"])
def test_reference_bench_harness_on_gpu(tmp_path, name):
    """SURVEY 8(f) #4: the reference's own MTTKRP benchmark driver (`splatt bench -a csf`,
    src/bench.c:133-224 -- it forces ONEMODE + DENSETILE CSFs) running on the GPU engine through
    the same link-time replacement, with `-w` dumping every mode's MTTKRP result
    (csf_mode<N>.mat): the dumps must match the pure-CPU binary's."""
    z = np.load(GOLD / f"{name}.npz")
    tns = tmp_path / f"{name}.tns"
    _write_tns(tns, z["ind"], z["vals"])
    # the CLI seeds rand() with time(NULL) (src/cmds/splatt_bin.c:91): pin time() for both runs so
    # that both binaries draw the same random factor matrices
    shim_c = tmp_path / "time_shim.c"
    shim_c.write_text("#include <time.h>\ntime_t time(time_t * t) { if (t) *t = 1234567; return 1234567; }\n")
    shim = tmp_path / "time_shim.so"
    subprocess.run(["gcc", "-shared", "-fPIC", "-o", str(shim), str(shim_c)], check=True)
    gpu_cli, env = relocated_binary(GPU_CLI, tmp_path)
    env["LD_PRELOAD"] = str(shim)
    outs = {}
    for tag, exe in (("cpu", ref.CLI_PATH), ("gpu", gpu_cli)):
        wd = tmp_path / tag
        wd.mkdir()
        r = subprocess.run([str(exe), "bench", str(tns), "-a", "csf", "-i", "1", "-r", "8", "-t", "2",
                            "-w"], capture_output=True, text=True, timeout=300, cwd=wd, env=env)
        assert r.returncode == 0, r.stderr
        assert "** CSF **" in r.stdout
        outs[tag] = [np.loadtxt(wd / f"csf_mode{m + 1}.mat") for m in range(len(z["dims"]))]
    for m, (a, b) in enumerate(zip(outs["cpu"], outs["gpu"])):
        assert a.shape == b.shape == (int(z["dims"][m]), 8)
        # the dump keeps 9 significant digits
        assert np.allclose(a, b, rtol=1e-7, atol=1e-7), m
