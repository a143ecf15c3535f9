"""The reference's answers to the calls the tests make, with or without the compiled reference.

The `refmod` fixture (tests/conftest.py) returns this module.  It offers the calls of
oracle/ref.py.  Where the unmodified reference was built into oracle/_ref, every call goes to
it.  Everywhere else each answer comes from this repository -- the plain-C restatement of the
reference in oracle/restate.c, for MTTKRP, CSF construction and CPD-ALS -- and is checked
against what the compiled reference answered to the same call, stored in
tests/golden/reference_calls.npz:

  * small answers (options, ABI facts, mode orders, small CPD results) are stored whole and
    returned as they are;
  * a dense result (an MTTKRP output, a large CPD result) is stored as a fingerprint: Frobenius
    norm, column sums and row-weighted column sums of every matrix;
  * a CSF is stored as the SHA-256 of all its arrays, so it must be bit-identical.

A call the store does not hold fails.  With REFGOLD_RECORD=<file> set and oracle/_ref built, the
answers of the compiled reference are added to the store and written to <file> at exit (run
the CPU and the GPU tests that way, then copy <file> to tests/golden/reference_calls.npz).
Reference CSFs built with SPLATT_DENSETILE have no counterpart here, so a test that needs one
skips where oracle/_ref was not built.
"""
from __future__ import annotations

import atexit
import hashlib
import os
from pathlib import Path

import numpy as np
import pytest

from oracle import ref as _ref_mod
from oracle import restate
from oracle.ref import (CSF_INORDER_MINUSONE, CSF_MODE_CUSTOM, CSF_SORTED_BIGFIRST,  # noqa: F401
                        CSF_SORTED_MINUSONE, CSF_SORTED_SMALLFIRST)

STORE_PATH = Path(__file__).parent / "golden" / "reference_calls.npz"
LIVE = _ref_mod.available()
RECORD = os.environ.get("REFGOLD_RECORD") if LIVE else None
WHOLE_MAX = 8192            # answers up to this many numbers are stored whole

_store = None


def _load():
    global _store
    if _store is None:
        _store = {}
        if STORE_PATH.exists():
            z = np.load(STORE_PATH)
            keys, kinds, offs, data = z["keys"], z["kinds"], z["offsets"], z["data"]
            for i, k in enumerate(keys):
                _store[k.tobytes().hex()] = (int(kinds[i]), data[offs[i]:offs[i + 1]].copy())
    return _store


def _save():
    s = _load()
    keys = sorted(s)
    offs = np.cumsum([0] + [len(s[k][1]) for k in keys])
    np.savez_compressed(RECORD, keys=np.array([list(bytes.fromhex(k)) for k in keys], dtype=np.uint8),
                        kinds=np.array([s[k][0] for k in keys], dtype=np.uint8),
                        offsets=offs.astype(np.int64),
                        data=np.concatenate([s[k][1] for k in keys]) if keys else np.zeros(0))


if RECORD:
    atexit.register(_save)

WHOLE, DENSE, HASH = 0, 1, 2


def _key(*parts) -> str:
    h = hashlib.sha1()
    for p in parts:
        if isinstance(p, np.ndarray):
            h.update(str(p.dtype).encode() + str(p.shape).encode())
            h.update(np.ascontiguousarray(p).tobytes())
        else:
            h.update(repr(p).encode())
        h.update(b"|")
    return h.hexdigest()


def _dense_fp(mats) -> np.ndarray:
    fp = []
    for a in mats:
        a = np.asarray(a, dtype=np.float64)
        w = 1.0 + (np.arange(a.shape[0]) % 13)[:, None]
        fp += [[np.linalg.norm(a)], a.sum(axis=0), (w * a).sum(axis=0)]
    return np.concatenate(fp)


def _check_dense(mats, want, rtol):
    got = _dense_fp(mats)
    assert got.shape == want.shape, "stored reference answer has another shape"
    at = 0
    for a in mats:
        n, r = np.asarray(a).shape
        fro = want[at]
        tol = rtol * max(fro, 1e-300) * np.sqrt(n)
        assert abs(got[at] - fro) <= rtol * max(fro, 1e-300), ("fro", got[at], fro)
        assert np.all(np.abs(got[at + 1:at + 1 + r] - want[at + 1:at + 1 + r]) <= tol), "colsum"
        assert np.all(np.abs(got[at + 1 + r:at + 1 + 2 * r] - want[at + 1 + r:at + 1 + 2 * r])
                      <= 13 * tol), "weighted colsum"
        at += 1 + 2 * r


def _put(key, kind, data):
    _load()[key] = (kind, np.asarray(data, dtype=np.float64).ravel().copy())


def _get(key, what):
    s = _load()
    if key not in s:
        pytest.fail(f"tests/golden/reference_calls.npz holds no reference answer for this {what}; "
                    "record it with the compiled reference (REFGOLD_RECORD, see tests/refgold.py)")
    return s[key]


def _csf_hash(csf) -> np.ndarray:
    """SHA-256 of every array of every CSF.  Nonzeros with equal coordinates may lie in either
    order (that is up to the sort), so the values of such runs are hashed sorted."""
    h = hashlib.sha256()
    for c in range(csf.count):
        a = csf.arrays(c)
        for k in ("nnz", "dims", "dim_perm", "dim_iperm", "nfibs"):
            h.update(repr(a[k]).encode())
        n = len(a["nfibs"])
        fiber = np.repeat(np.arange(a["nfibs"][n - 2]), np.diff(a["fptr"][n - 2]).astype(np.int64))
        vals = a["vals"][np.lexsort((a["vals"], a["fids"][n - 1], fiber))]
        for arr in a["fids"] + a["fptr"] + [vals]:
            h.update(b"none" if arr is None else np.ascontiguousarray(arr).tobytes())
    return np.frombuffer(h.digest(), dtype=np.float64)


def default_opts() -> np.ndarray:
    key = _key("default_opts")
    if LIVE:
        o = _ref_mod.default_opts()
        if RECORD:
            _put(key, WHOLE, o)
        return o
    return _get(key, "default_opts")[1].copy()


def abi_facts():
    key = _key("abi_facts")
    if LIVE:
        f = _ref_mod.abi_facts()
        if RECORD:
            _put(key, WHOLE, f)
        return f
    return [int(x) for x in _get(key, "abi_facts")[1]]


def mode_order(dims, which: int, mode: int = 0):
    key = _key("mode_order", [int(d) for d in dims], int(which), int(mode))
    if LIVE:
        p = _ref_mod.mode_order(dims, which, mode)
        if RECORD:
            _put(key, WHOLE, p)
        return p
    mine = restate.mode_order(dims, which, mode)
    assert mine == [int(x) for x in _get(key, "mode_order")[1]]
    return mine


class RefTensor:
    """A COO tensor; the reference's sptensor_t where oracle/_ref exists."""

    def __init__(self, dims, ind, vals):
        self.dims = [int(d) for d in dims]
        self.nmodes = len(self.dims)
        self.inds = [np.array(i, dtype=np.uint64) for i in ind]
        self.vals = np.array(vals, dtype=np.float64)
        self.nnz = len(self.vals)
        # the key names the tensor as given: the reference's csf_alloc later sorts it in place
        self.key = _key("tensor", self.dims, *self.inds, self.vals)
        self.live = _ref_mod.RefTensor.from_coo(dims, ind, vals) if LIVE else None

    @classmethod
    def from_coo(cls, dims, ind, vals) -> "RefTensor":
        return cls(dims, ind, vals)

    def mttkrp_key(self, mats, mode):
        return _key("mttkrp", self.key, int(mode),
                    *[np.asarray(m, dtype=np.float64) for i, m in enumerate(mats) if i != mode])

    def mttkrp_stream(self, mats, mode: int, nthreads: int = 1) -> np.ndarray:
        key = self.mttkrp_key(mats, mode)
        if LIVE:
            out = self.live.mttkrp_stream(mats, mode, nthreads)
            if RECORD:
                _put(key, DENSE, _dense_fp([out]))
            return out
        out = restate.mttkrp_coo(self.dims, self.inds, self.vals, mats, mode)
        _check_dense([out], _get(key, "MTTKRP")[1], 1e-12)
        return out

    def free(self):
        if self.live is not None:
            self.live.free()


class _OracleCsfs:
    """The CSFs oracle/restate.c builds for a csf_alloc policy, laid out as the array of
    `splatt_csf` the reference's csf_alloc returns (untiled), so that `.ptr` can be handed to
    any function taking `splatt_csf const *`."""

    def __init__(self, tt: RefTensor, alloc: int):
        import ctypes as C
        from splatt_b200 import _abi as A
        perms, _ = restate.csf_policy(tt.dims, alloc)
        self.count = len(perms)
        self._keep = []
        arr = (A.SplattCsf * self.count)()
        n = tt.nmodes

        def p(a, t):
            a = np.ascontiguousarray(a)
            self._keep.append(a)
            return a.ctypes.data_as(t)
        for c, perm in enumerate(perms):
            a = restate.OracleCsf(tt.dims, tt.inds, tt.vals, perm).arrays()
            pt = (A.CsfSparsity * 1)()
            for lv in range(n):
                pt[0].nfibs[lv] = a["nfibs"][lv]
                if a["fids"][lv] is not None:
                    pt[0].fids[lv] = p(a["fids"][lv], A.idx_p)
                if lv < n - 1:
                    pt[0].fptr[lv] = p(a["fptr"][lv], A.idx_p)
            pt[0].vals = p(a["vals"], A.val_p)
            self._keep.append(pt)
            s = arr[c]
            s.nnz, s.nmodes, s.which_tile, s.ntiles, s.ntiled_modes = tt.nnz, n, 0, 1, 0
            for m in range(n):
                s.dims[m] = tt.dims[m]
                s.dim_perm[m] = a["dim_perm"][m]
                s.dim_iperm[a["dim_perm"][m]] = m
                s.tile_dims[m] = 1
            s.pt = C.cast(pt, C.POINTER(A.CsfSparsity))
        self._arr = arr
        self.ptr = C.cast(arr, C.POINTER(A.SplattCsf))

    def free(self):
        pass


class RefCsf:
    """CSF(s) as the reference's csf_alloc builds them."""

    def __init__(self, tt: RefTensor, opts: np.ndarray):
        self.tt = tt
        self.opts = np.array(opts, dtype=np.float64)
        o = self.opts
        tiled = int(o[7]) != 0
        self.key = _key("csf", tt.key, int(o[6]), int(o[7]), int(o[8]), int(o[0]) if tiled else 0)
        if LIVE:
            self.impl = _ref_mod.RefCsf(tt.live, opts)
        elif tiled:
            pytest.skip("a DENSETILE CSF is built by the compiled reference only (oracle/_ref)")
        else:
            self.impl = _OracleCsfs(tt, int(o[6]))
        self.ptr = self.impl.ptr
        self.count = self.impl.count
        self.nmodes = tt.nmodes
        self.dims = list(tt.dims)
        if RECORD and not tiled:
            _put(self.key, HASH, _csf_hash(self))
        elif not LIVE:
            assert _csf_hash(self).tobytes() == _get(self.key, "CSF")[1].tobytes(), \
                "CSF differs from the reference's"

    def arrays(self, c: int = 0, tile: int = 0) -> dict:
        from splatt_b200.api import Csf
        return Csf.arrays(self.impl, c, tile)   # same struct layout

    def mttkrp_csf(self, mats, mode: int, *, warm: int = 0, iters: int = 1, opts=None):
        """The reference's mttkrp_csf; (out, times[s]).  Without oracle/_ref no time is taken."""
        key = self.tt.mttkrp_key(mats, mode)
        if LIVE:
            out, times = self.impl.mttkrp_csf(mats, mode, warm=warm, iters=iters, opts=opts)
            if RECORD:
                _put(key, DENSE, _dense_fp([out]))
            return out, times
        out = restate.mttkrp_coo(self.tt.dims, self.tt.inds, self.tt.vals, mats, mode)
        _check_dense([out], _get(key, "MTTKRP")[1], 1e-12)
        return out, np.zeros(max(iters, 1))[:iters]

    def cpd_als(self, R: int, seed: int, opts=None):
        o = self.opts if opts is None else np.asarray(opts, dtype=np.float64)
        key = _key("cpd", self.tt.key, int(R), int(seed), float(o[1]), float(o[2]), int(o[3]))
        if LIVE:
            fit, lam, facs = self.impl.cpd_als(R, seed, opts)
            if RECORD:
                whole = np.concatenate([[fit], lam] + [f.ravel() for f in facs])
                if whole.size <= WHOLE_MAX:
                    _put(key, WHOLE, whole)
                else:
                    _put(key, DENSE, np.concatenate([[fit], lam, _dense_fp(facs)]))
            return fit, lam, facs
        kind, want = _get(key, "CPD-ALS")
        if kind == WHOLE:
            facs, at = [], 1 + R
            for d in self.dims:
                facs.append(want[at:at + d * R].reshape(d, R).copy())
                at += d * R
            return float(want[0]), want[1:1 + R].copy(), facs
        fit, lam, facs = restate.cpd_als(self.tt.dims, self.tt.inds, self.tt.vals, R, int(o[3]),
                                         float(o[1]), seed)
        assert abs(fit - want[0]) <= 1e-10, (fit, want[0])
        assert np.allclose(lam, want[1:1 + R], rtol=1e-8, atol=1e-12)
        _check_dense(facs, want[1 + R:], 1e-8)
        return fit, lam, facs

    def free(self):
        self.impl.free()
