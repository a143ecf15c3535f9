"""Shared helpers for the test-suite: seeded synthetic tensors and error norms."""
from __future__ import annotations

import os
import re
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent


def random_coo(dims, nnz, seed=0, unique=True, skew=None):
    """Seeded random COO.  unique=True removes duplicate coordinates (the order of
    duplicates inside a CSF leaf is sort-implementation specific).  skew: optional
    list of per-mode Zipf exponents (None = uniform)."""
    rng = np.random.default_rng(seed)
    dims = list(dims)
    inds = []
    for m, d in enumerate(dims):
        if skew is not None and skew[m]:
            p = 1.0 / np.arange(1, d + 1) ** skew[m]
            p /= p.sum()
            perm = rng.permutation(d)
            inds.append(perm[rng.choice(d, size=nnz, p=p)].astype(np.uint64))
        else:
            inds.append(rng.integers(0, d, size=nnz, dtype=np.uint64))
    vals = rng.uniform(0.0, 1.0, size=nnz)
    if unique:
        key = np.zeros(nnz, dtype=np.uint64)
        for m, d in enumerate(dims):
            key = key * np.uint64(d) + inds[m]
        _, first = np.unique(key, return_index=True)
        first.sort()
        inds = [i[first] for i in inds]
        vals = vals[first]
    return dims, inds, vals


def cover_all_slices(dims, inds, vals, seed=1):
    """Append one nonzero per (mode, index) so that no slice is empty."""
    rng = np.random.default_rng(seed)
    extra = [[] for _ in dims]
    for m, d in enumerate(dims):
        missing = np.setdiff1d(np.arange(d, dtype=np.uint64), inds[m])
        for mm, dd in enumerate(dims):
            if mm == m:
                extra[mm].append(missing)
            else:
                extra[mm].append(rng.integers(0, dd, size=len(missing), dtype=np.uint64))
    inds2 = [np.concatenate([inds[m]] + extra[m]) for m in range(len(dims))]
    n_extra = len(inds2[0]) - len(vals)
    vals2 = np.concatenate([vals, rng.uniform(0.0, 1.0, size=n_extra)])
    return dims, inds2, vals2


def factor_mats(dims, R, seed=0):
    """Seeded factors, uniform [-3, 3] like the reference's mat_rand (src/util.c:15-23)."""
    rng = np.random.default_rng(1000 + seed)
    return [np.ascontiguousarray(rng.uniform(-3.0, 3.0, size=(d, R))) for d in dims]


def rel_fro(a, b):
    den = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / (den if den > 0 else 1.0))


def relocated_binary(exe, wd):
    """A copy in `wd` of a binary under oracle/_ref that runs wherever the tree now lies, and
    the environment to run it in.

    Binaries linked by an earlier oracle/build_ref.sh name libsplatt_b200.so by the absolute
    path of the tree they were built in, and read their fixtures from /tmp/splatt_b200_fixtures/.
    In the copy both strings are rewritten in place (same length, NUL-padded): the library by
    file name, found through LD_LIBRARY_PATH, and the fixtures relative to the working
    directory.  Binaries of the current recipe already use both forms and are copied unchanged."""
    data = Path(exe).read_bytes()

    def pad(m, new):
        return new + b"\0" * (len(m.group(0)) - len(new))
    data = re.sub(rb"/[^\0]*/splatt_b200/libsplatt_b200\.so\0",
                  lambda m: pad(m, b"libsplatt_b200.so\0"), data)
    data = re.sub(rb"/tmp/(splatt_b200_fixtures/[^\0]*\0)", lambda m: pad(m, m.group(1)), data)
    out = Path(wd) / Path(exe).name
    out.write_bytes(data)
    out.chmod(0o755)
    paths = [str(ROOT / "splatt_b200")] + [p for p in [os.environ.get("LD_LIBRARY_PATH")] if p]
    return out, dict(os.environ, LD_LIBRARY_PATH=os.pathsep.join(paths))
