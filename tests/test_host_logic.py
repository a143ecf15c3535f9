"""CPU: host-side logic of the engine that needs no GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import restate
from splatt_b200 import _abi as A

DIMS = [[30, 10, 20], [10, 10, 10], [30, 10, 20, 10], [5, 4, 3, 2, 1], [7, 7, 3, 7, 3, 9],
        [2425, 10816, 29567], [60114, 83826, 23034, 1132, 100], [4, 3, 5, 4, 3, 6, 2, 5]]


def level_orders(lib, dims, alloc):
    d = np.ascontiguousarray(dims, dtype=np.uint64)
    perms = (C.c_int * 64)()
    mp = (C.c_int * 8)()
    n = lib.splatt_b200_level_orders(d.ctypes.data_as(A.idx_p), len(dims), alloc, perms, mp)
    return [[perms[c * 8 + l] for l in range(len(dims))] for c in range(n)], [mp[m] for m in
                                                                             range(len(dims))]


@pytest.mark.parametrize("dims", DIMS)
@pytest.mark.parametrize("alloc", [0, 1, 2])
def test_level_orders_match_restatement(lib, dims, alloc):
    assert level_orders(lib, dims, alloc) == restate.csf_policy(dims, alloc)


@pytest.mark.parametrize("dims", DIMS)
def test_level_orders_match_compiled_reference(lib, refmod, dims):
    """csf_find_mode_order (src/csf.c:694-726) for the orders csf_alloc uses (:770-814)."""
    n = len(dims)
    small = refmod.mode_order(dims, refmod.CSF_SORTED_SMALLFIRST)
    assert level_orders(lib, dims, 0)[0] == [small]
    two, mp = level_orders(lib, dims, 1)
    assert two[0] == small
    assert two[1] == refmod.mode_order(dims, refmod.CSF_SORTED_MINUSONE, small[-1])
    assert mp == [1 if m == small[-1] else 0 for m in range(n)]
    allm, mp = level_orders(lib, dims, 2)
    assert allm == [refmod.mode_order(dims, refmod.CSF_SORTED_MINUSONE, m) for m in range(n)]
    assert mp == list(range(n))
    for which in range(4):
        assert restate.mode_order(dims, which, n - 1) == refmod.mode_order(dims, which, n - 1)


def test_bad_policy_is_rejected(lib):
    assert level_orders(lib, [3, 4, 5], 7) == ([], [0, 0, 0])


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No CPU fallback: a missing extension is an error, not a slow path."""
    monkeypatch.setattr(A, "_lib", None)
    monkeypatch.setattr(A, "LIB_PATH", tmp_path / "nope.so")
    with pytest.raises(RuntimeError, match="no fallback"):
        A.load()


@pytest.mark.parametrize("spec", [((30, 20, 40), 3000), ((12, 10, 14, 8), 2500), ((9, 8, 7, 6, 5), 2000)])
@pytest.mark.parametrize("tile", [(0, 0), (1, 1), (1, 2), (1, 8)])
@pytest.mark.parametrize("alloc", [0, 2])
def test_csf_to_coo_expands_reference_csfs(lib, refmod, spec, tile, alloc):
    """Host side of the device mirror: a reference CSF (untiled, or DENSETILE at any depth,
    built with 7 threads like tests/mttkrp_test.c -- up to 7^nmodes mostly empty tiles) expands
    to exactly the tensor's nonzeros."""
    import time
    from tests.util import random_coo
    dims, inds, vals = random_coo(spec[0], spec[1], seed=4)
    o = refmod.default_opts()
    o[0], o[6], o[7], o[8] = 7, alloc, tile[0], tile[1]
    tt = refmod.RefTensor.from_coo(dims, inds, vals)
    rc = refmod.RefCsf(tt, o)
    n = len(vals)
    for c in range(rc.count):
        out = [np.zeros(n, dtype=np.uint32) for _ in dims]
        ov = np.zeros(n)
        ip = (C.POINTER(C.c_uint32) * len(dims))(*[a.ctypes.data_as(C.POINTER(C.c_uint32)) for a in out])
        t0 = time.time()
        import ctypes as _C
        csf_c = _C.cast(_C.addressof(rc.ptr[c]), _C.POINTER(A.SplattCsf))
        assert lib.splatt_b200_csf_to_coo(csf_c, ip, ov.ctypes.data_as(A.val_p)) == A.SPLATT_SUCCESS
        assert time.time() - t0 < 5.0
        got = sorted(zip(*[a.tolist() for a in out], ov.tolist()))
        want = sorted(zip(*[i.tolist() for i in inds], vals.tolist()))
        assert got == want


@pytest.mark.parametrize("env,want", [
    ({}, []),
    ({"SPLATT_B200_NGPUS": "1"}, []),
    ({"SPLATT_B200_NGPUS": "4"}, [0, 1, 2, 3]),
    ({"SPLATT_B200_DEVICES": "0,2,5"}, [0, 2, 5]),
    ({"SPLATT_B200_DEVICES": "0,0", "SPLATT_B200_NGPUS": "8"}, [0, 0]),     # the list wins
    ({"SPLATT_B200_NGPUS": "99"}, list(range(16))),                          # capped
])
def test_multi_gpu_device_list_from_environment(lib, monkeypatch, env, want):
    """SPLATT_B200_NGPUS / SPLATT_B200_DEVICES: which devices the drop-in symbols drive from one
    process (multi.cu); no variable or one device = the single-GPU path."""
    for k in ("SPLATT_B200_NGPUS", "SPLATT_B200_DEVICES"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    buf = (C.c_int * 16)()
    n = lib.splatt_b200_multi_env_devices(buf, 16)
    assert [buf[i] for i in range(n)] == want


def test_multi_gpu_engine_rejects_bad_arguments(lib):
    """No GPU needed: argument checks come before any CUDA call.  (The build count is
    cumulative over the process, so GPU tests run earlier in the session are allowed for.)"""
    built = lib.splatt_b200_build_count()
    out = C.c_void_p()
    devs = (C.c_int * 1)(0)
    assert lib.splatt_b200_multi_create(None, 1, 8, devs, 1, 0, C.byref(out)) == A.SPLATT_ERROR_BADINPUT
    assert lib.splatt_b200_multi_mttkrp_host(None, 0, None, None) == A.SPLATT_ERROR_BADINPUT
    assert lib.splatt_b200_multi_info(None, None, None, None, None) == A.SPLATT_ERROR_BADINPUT
    lib.splatt_b200_multi_free(None)
    lib.splatt_b200_cache_clear()                       # drops cached mirrors, builds nothing
    assert lib.splatt_b200_build_count() == built


def test_every_environment_switch_is_documented():
    """Every SPLATT_B200_* variable the sources read appears in DESIGN.md (section 9)."""
    import re
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    names = set()
    for f in list((root / "splatt_b200" / "csrc").glob("*.cu*")) + list((root / "splatt_b200").glob("*.py")) \
            + [root / "bench.py"]:
        text = f.read_text()
        names |= set(re.findall(r'getenv\("(SPLATT_B200_[A-Z0-9_]+)"\)', text))
        names |= set(re.findall(r'environ(?:\.get)?[\[(]"(SPLATT_B200_[A-Z0-9_]+)"', text))
    assert len(names) > 10
    design = (root / "DESIGN.md").read_text()
    missing = sorted(n for n in names if n not in design)
    assert not missing, missing
