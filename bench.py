#!/usr/bin/env python
"""bench.py -- MTTKRP nnz*R/sec per mode on synthetic sparse tensors (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--dump-outputs DIR]

A "step" is one MTTKRP sweep: one MTTKRP per mode of the tensor (the hot path of
one CPD-ALS iteration).  value = nnz_total * R * nmodes / step time = the mean
per-mode throughput, whole-job aggregate over all ranks.

Headline workload (config.workload): BASELINE.json configs[1] at N=1 -- synthetic
uniform 3-mode 10K x 10K x 10K, 10M nonzeros, rank 32, fp64.  For N>1 the per-GPU
work is held fixed (weak scaling): the tensor has 10M*N nonzeros in the same 10K^3
index space, every rank holds an equal-nnz contiguous share of each mode's fiber
stream, and the per-mode sum over ranks happens INSIDE the MTTKRP kernel
(multimem.red over an NVLink multicast mapping, group barrier in the kernel's
tail); `--nccl-exchange` runs kernel + NCCL all-reduce instead.

Timed region: inputs resident in HBM; W warm-up steps, then exactly K steps
enqueued back to back (no host synchronisation inside the region), one CUDA event
pair per step and per mode on the launching stream; L2 flushed (256 MB write)
between steps, outside the per-step events; barrier + synchronize on both sides;
MAX over ranks.  Nothing is re-measured: the one timed region is what is reported.

Also in the JSON line:
  parity_rel_fro   per mode, the summed output of the timed path (fused exchange at
                   N>1) against the reference's own mttkrp_csf (oracle/_ref) on the same
                   tensor, computed on rank 0 outside the timed region.
  named_configs    BASELINE.json configs[3] (100K^3, 100M nnz, R=32) and configs[4]
                   (Zipf 1M x 1M x 1K, 200M nnz, R=64) with the WHOLE tensor fixed and
                   shared by the N ranks (strong scaling): per-mode ms, nnz*R/s, own
                   clocks sample, exchange kind, parity_rel_fro vs the reference.
  e2e              the same sweep through the reference-facing C ABI
                   (splatt_mttkrp_alloc_ws + splatt_mttkrp_csf) with HOST buffers, copies
                   inside the timed region; reported for pageable caller buffers (what the
                   reference's splatt_malloc gives; `value`) and page-locked ones.  At N>1
                   it is the single-process multi-GPU engine behind that same C entry
                   (SPLATT_B200_NGPUS=N), run by rank 0 while the other ranks idle.

`--impl reference` times the reference's own OpenMP mttkrp_csf (oracle/_ref,
compiled unmodified from the reference's sources) on the host cores on the same workload.

`--dump-outputs DIR` writes what the headline workload's timed path computed in its
last step, the summed output of every mode, as DIR/mttkrp_mode<m>.npy (float64,
10000 x 32 each).  Inputs are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

DIM = 10_000
NNZ_PER_GPU = 10_000_000
RANK = 32
NMODES = 3
SEED = 1
FALLBACK_HBM_GBS = 6650.0

NAMED = {
    "4": {"name": "BASELINE.json configs[3]: synthetic uniform 3-mode 100000^3, 100M nnz, rank 32",
          "dims": [100_000] * 3, "nnz": 100_000_000, "rank": 32, "zipf": False, "seed": 3},
    "5": {"name": "BASELINE.json configs[4]: Zipf(1.0) 3-mode 1M x 1M x 1K, 200M nnz, rank 64",
          "dims": [1_000_000, 1_000_000, 1_000], "nnz": 200_000_000, "rank": 64, "zipf": True,
          "seed": 4},
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- workloads
def make_coo_gpu(nnz: int, device, dims=None, seed=SEED, zipf=False):
    """Seeded synthetic COO on the device: mode-0, mode-1, ... index arrays, then values.
    zipf: modes 0 and 1 are Zipf(1.0) ranks (inverse-CDF sampling) sent through a fixed random
    relabelling; the last mode stays uniform (SURVEY 8d, config 5)."""
    import torch
    dims = [DIM] * NMODES if dims is None else dims
    g = torch.Generator(device=device).manual_seed(seed)

    def zipf_idx(d):
        w = 1.0 / torch.arange(1, d + 1, device=device, dtype=torch.float64)
        cdf = torch.cumsum(w / w.sum(), 0)
        u = torch.rand(nnz, device=device, dtype=torch.float64, generator=g)
        r = torch.searchsorted(cdf, u).clamp_(max=d - 1)
        del u
        return torch.randperm(d, device=device, generator=g)[r].to(torch.int32)

    ind = []
    for m, d in enumerate(dims):
        if zipf and m < 2:
            ind.append(zipf_idx(d))
        else:
            ind.append(torch.randint(0, d, (nnz,), device=device, dtype=torch.int32, generator=g))
    vals = torch.rand(nnz, device=device, dtype=torch.float64, generator=g)
    return ind, vals


def make_factors_host(seed=SEED, dims=None, rank=RANK):
    dims = [DIM] * NMODES if dims is None else dims
    rng = np.random.default_rng(1000 + seed)
    return [np.ascontiguousarray(rng.uniform(-3.0, 3.0, size=(d, rank))) for d in dims]


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture."""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


def rel_fro(a, b):
    den = float(np.linalg.norm(b))
    return float(np.linalg.norm(a - b) / (den if den > 0 else 1.0))


# --------------------------------------------------------------------------- reference arm
class ReferenceRun:
    """The reference's own mttkrp_csf on one tensor: CSF(s) built by its csf_alloc, ws and
    thread scratch allocated once per group of calls (the src/cpd.c:285-304 pattern)."""

    def __init__(self, dims, ind_host, vals_host, csf_alloc=1):
        from oracle import ref
        self.ref = ref
        self.dims = list(dims)
        self.o = ref.default_opts()
        self.aff = len(os.sched_getaffinity(0))
        self.o[0] = self.aff
        self.o[6] = csf_alloc
        t0 = time.time()
        self.tt = ref.RefTensor.from_coo(self.dims, ind_host, vals_host)
        self.csf = ref.RefCsf(self.tt, self.o)
        self.alloc_name = {0: "ONEMODE", 1: "TWOMODE", 2: "ALLMODE"}[csf_alloc]
        log(f"[reference] csf_alloc ({self.alloc_name}) {time.time()-t0:.1f}s with {self.aff} threads")

    def sweep(self, mats, threads, warm, iters):
        """Returns (outputs per mode, seconds per sweep [iters])."""
        oo = self.o.copy()
        oo[0] = threads
        res = [self.csf.mttkrp_csf(mats, m, warm=warm, iters=iters, opts=oo)
               for m in range(len(self.dims))]
        return [r[0] for r in res], np.sum(np.stack([r[1] for r in res]), axis=0)

    def best_threads(self, mats, trials=2):
        """The reference gets its best thread count: torchrun exports OMP_NUM_THREADS=1 and
        more threads than physical cores hurts it; on config 2 it privatises its output only
        below 21 threads (src/mttkrp.c:221-236), which is where it is fastest.  Every
        candidate is timed `trials` times (best kept) to keep the pick stable."""
        env = os.environ.get("SPLATT_REF_THREADS")
        if env:
            return int(env), {}
        aff = self.aff
        cands = sorted({t for t in (8, 12, 16, 20, 24, 32, 48, 64, aff // 2, aff) if 1 <= t <= aff})
        trial = {t: float(np.min(self.sweep(mats, t, 1, trials)[1])) for t in cands}
        best = min(trial, key=trial.get)
        log(f"[reference] {self.alloc_name} sweep seconds by thread count: " +
            ", ".join(f"{t}:{trial[t]:.3f}" for t in cands) + f" -> using {best}")
        return best, trial

    def free(self):
        self.csf.free()
        self.tt.free()


def reference_best(dims, ind_host, vals_host, mats, steps, warmup):
    """Time the reference at its best configuration: default TWOMODE and ALLMODE (a legal
    option that turns its slow internal-mode call into a root call), each at its best thread
    count; the faster one is reported.  Returns (seconds per sweep [steps], threads, what)."""
    best = None
    for alloc in (1, 2):
        rr = ReferenceRun(dims, ind_host, vals_host, alloc)
        thr, _ = rr.best_threads(mats)
        _, step_s = rr.sweep(mats, thr, warmup, steps)
        rr.free()
        cand = (float(np.mean(step_s)), step_s, thr, rr.alloc_name)
        if best is None or cand[0] < best[0]:
            best = cand
    return best[1], best[2], best[3]


def port_sweeps(ind_host, vals_host, mats, steps, warmup):
    """Fallback when oracle/_ref is absent: the plain-C restatement (oracle/restate.c,
    COO streaming MTTKRP = the reference's gold mttkrp_stream), one host thread."""
    from oracle import restate
    dims = [DIM] * NMODES
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        for m in range(NMODES):
            restate.mttkrp_coo(dims, ind_host, vals_host, mats, m)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return np.array(times), 1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    try:
        from oracle import ref
        import torch
        nnz = NNZ_PER_GPU * max(args.gpus, 1)
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        ind, vals = make_coo_gpu(nnz, dev)
        ind_h = [i.cpu().numpy().astype(np.uint64) for i in ind]
        vals_h = vals.cpu().numpy()
        del ind, vals
        mats = make_factors_host()
        if ref.available():
            step_s, cores, alloc = reference_best([DIM] * NMODES, ind_h, vals_h, mats, args.steps,
                                                  args.warmup)
            kind, what = "reference", f"reference mttkrp_csf (OpenMP, {alloc}, untiled)"
        else:
            step_s, cores = port_sweeps(ind_h, vals_h, mats, args.steps, min(args.warmup, 1))
            kind, what = "port", "oracle/restate.c COO streaming MTTKRP (oracle/_ref absent)"
        ms = float(np.mean(step_s) * 1e3)
        value = nnz * RANK * NMODES / (ms * 1e-3)
        line = {"metric": "MTTKRP nnz*R/sec per mode", "value": value, "unit": "nnz*R/s",
                "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(args.gpus),
                "cpu_baseline": {"value": value, "unit": "nnz*R/s", "cores": cores,
                                 "kind": kind,
                                 "sample": f"full workload, {args.steps} sweeps x {NMODES} modes, "
                                           + what + "; the faster of TWOMODE / ALLMODE at its "
                                           "fastest thread count"},
                "e2e": {"value": value, "unit": "nnz*R/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
    except Exception as e:  # pragma: no cover
        print(json.dumps({"impl": "reference", "unavailable": f"{type(e).__name__}: {e}"}))
    return 0


def workload_config(n_gpus):
    return {"workload": f"synthetic uniform 3-mode {DIM}^3, {NNZ_PER_GPU} nnz per GPU "
                        f"({NNZ_PER_GPU * max(n_gpus,1)} total), rank {RANK} "
                        "(BASELINE.json configs[1] at N=1)",
            "dims": [DIM] * NMODES, "nnz_total": NNZ_PER_GPU * max(n_gpus, 1), "rank": RANK,
            "step": "one MTTKRP per mode (3 launches; N>1: each followed by the exchange)",
            "partition": "equal-nnz contiguous shares of every mode's fiber stream; the output "
                         "factor is summed over ranks once per mode (see exchange)",
            "l2": "flushed between steps (256 MB write, outside the timed events)",
            "seed": SEED}


def gather_probe_gbs(dev):
    """Measured rate of the access pattern that bounds the kernel at the KERNEL's own shape
    (24 warps/SM, 8 rows in flight): random whole-row fp64 gathers (RANK columns) from a
    DIM-row matrix, nothing else.  The ceiling over all shapes is in profiles/ (probe sweep)."""
    import ctypes as C
    import torch
    from splatt_b200 import _abi as A
    lib = A.load()
    n = 2 * NNZ_PER_GPU                      # one leaf + one parent row per nonzero
    g = torch.Generator(device=dev).manual_seed(7)
    idx = torch.randint(0, DIM, (n,), device=dev, dtype=torch.int32, generator=g)
    mat = torch.rand(DIM, RANK, device=dev, dtype=torch.float64, generator=g)
    sink = torch.zeros(8, device=dev, dtype=torch.float64)
    s = torch.cuda.current_stream().cuda_stream

    def run():
        rc = lib.splatt_b200_gather_probe(C.cast(C.c_void_p(mat.data_ptr()), A.val_p), RANK, RANK,
                                          C.cast(C.c_void_p(idx.data_ptr()), C.POINTER(C.c_uint32)),
                                          n, C.cast(C.c_void_p(sink.data_ptr()), A.val_p),
                                          C.c_void_p(s))
        assert rc == A.SPLATT_SUCCESS
    for _ in range(3):
        run()
    ts = []
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = float(np.median(ts))
    return n * RANK * 8 / (ms * 1e-3) / 1e9, ms


def probe_sweep_best():
    p = ROOT / "profiles" / "r02_probe_sweep_R32.json"
    try:
        return json.loads(p.read_text())["best"]
    except Exception:
        return None


def cpd_iteration_times(S, csf, ind, vals, mats_h, ref_threads=None):
    """CPD-ALS seconds per iteration (the metric's second half): splatt_cpd_als of this
    library (MTTKRP + dense tail on the device) vs the reference's, same tensor, rank and
    iteration count; set-up is removed by differencing two iteration counts."""
    out = {"rank": RANK, "ours_ms": None, "reference_ms": None}
    try:
        def ours(n):
            o = S.default_opts()
            o[3], o[1], o[4] = n, 0.0, 0
            t0 = time.perf_counter()
            S.cpd_als(csf.ptr, RANK, o, seed=SEED)
            return time.perf_counter() - t0
        ours(1)
        # 100 extra iterations (~0.13 s) dwarf the run-to-run noise of the set-up
        out["ours_ms"] = (min(ours(110), ours(110)) - min(ours(10), ours(10))) / 100 * 1e3
    except Exception as e:  # pragma: no cover
        out["ours_error"] = str(e)
    try:
        from oracle import ref
        if ref.available():
            o = ref.default_opts()
            o[1], o[4] = 0.0, 0
            o[0] = ref_threads or int(os.environ.get("SPLATT_REF_THREADS", "16"))
            tt = ref.RefTensor.from_coo([DIM] * NMODES,
                                        [i.cpu().numpy().astype(np.uint64) for i in ind],
                                        vals.cpu().numpy())
            rc = ref.RefCsf(tt, o)

            def theirs(n):
                oo = o.copy()
                oo[3] = n
                t0 = time.perf_counter()
                rc.cpd_als(RANK, SEED, opts=oo)
                return time.perf_counter() - t0
            out["reference_ms"] = (theirs(3) - theirs(1)) / 2 * 1e3
            out["reference_threads"] = int(o[0])
    except Exception as e:  # pragma: no cover
        out["reference_error"] = str(e)
    return out


# --------------------------------------------------------------------------- our arm
class Ctx:
    """Process-group facts + host-side (no GPU work) rendezvous helpers."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self._hb = 0

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def host_wait(self, tag):
        """Ranks != 0 sleep (no GPU work, no spinning collective) until rank 0 posts `tag`;
        used while rank 0 alone works (CPU reference for parity, single-process e2e)."""
        import torch.distributed as dist
        if self.world == 1:
            return
        store = dist.distributed_c10d._get_default_store()
        key = f"splatt_b200_bench/{tag}"
        if self.rank == 0:
            store.set(key, "1")
        else:
            import datetime
            store.wait([key], datetime.timedelta(seconds=1500))

    def max_over_ranks(self, x: float) -> float:
        import torch
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())


class Workload:
    """One tensor sharded over the ranks + the sweep that is timed."""

    def __init__(self, ctx, dims, ind, vals, R, nccl_exchange, seed):
        import torch
        import splatt_b200 as S
        from splatt_b200 import _abi as A
        self.ctx, self.dims, self.R, self.N = ctx, list(dims), R, len(dims)
        self.nnz = int(vals.numel())
        dev = ctx.dev
        t0 = time.time()
        self.T = S.Tensor.from_coo(self.dims, ind, vals, layout=A.LAYOUT_ALLROOT,
                                   shard_rank=ctx.rank, shard_count=ctx.world)
        torch.cuda.synchronize()
        self.build_s = time.time() - t0
        self.mats_h = make_factors_host(seed, self.dims, R)
        self.mats = [torch.from_numpy(m).to(dev) for m in self.mats_h]
        self.outs = [torch.empty((d, R), dtype=torch.float64, device=dev) for d in self.dims]
        self.info = [self.T.mode_info(m, R) for m in range(self.N)]
        self.fx = None
        if ctx.world > 1 and not nccl_exchange:
            from splatt_b200 import parallel
            self.fx = parallel.FusedExchange(self.T, R)
            if not self.fx.available():
                log(f"[rank {ctx.rank}] fused exchange unavailable ({self.fx.error}); NCCL all-reduce")
                self.fx = None
        self.exchange = ("none (single GPU)" if ctx.world == 1 else
                         ("fused: multimem.red.add.f64 into an NVLink multicast buffer, group "
                          "barrier in the kernel's tail" if self.fx.kernel_barrier else
                          "fused: multimem.red.add.f64 into an NVLink multicast buffer + 1 "
                          "symmetric-memory barrier launch")
                         if self.fx is not None else "NCCL all-reduce(sum) after the kernel")

    def sweep(self, events=None, capture=None):
        import torch.distributed as dist
        for m in range(self.N):
            if events is not None:
                events[m][0].record()
            if self.fx is not None:
                buf = self.fx.mttkrp(m, self.mats)  # kernel: reduces into every GPU's buffer + barrier
                if capture is not None:
                    capture[m] = buf[:, :self.R].clone()
                self.fx.release(m)                  # result consumed: re-zero for the next sweep
            else:
                self.T.mttkrp(m, self.mats, self.outs[m])
            if events is not None:
                events[m][1].record()
            if self.ctx.world > 1 and self.fx is None:
                dist.all_reduce(self.outs[m])
            if capture is not None and self.fx is None:
                capture[m] = self.outs[m].clone()

    def outputs_host(self):
        """One sweep of the timed path; the summed outputs on the host (rank 0's copy)."""
        import torch
        cap = [None] * self.N
        self.sweep(capture=cap)
        torch.cuda.synchronize()
        return [c.cpu().numpy() for c in cap]

    def timed(self, flush, steps, warmup, capture=None):
        """W warm-up steps, then K steps back to back; returns per-step ms, per-mode ms lists.
        capture: a list of N slots that receives the outputs of the last step."""
        import torch
        for _ in range(warmup):
            flush.zero_()
            self.sweep()
        self.ctx.barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
              for _ in range(steps)]
        kev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                for _ in range(self.N)] for _ in range(steps)]
        import splatt_b200 as S
        l0 = S.launch_count()
        w0 = time.time()
        for k in range(steps):
            flush.zero_()
            ev[k][0].record()
            # the fused exchange re-zeroes its buffer after every mode, so its result is copied
            # inside the last step; the other paths' outputs are still in place after the loop
            self.sweep(kev[k], capture if k == steps - 1 and self.fx is not None else None)
            ev[k][1].record()
        self.ctx.barrier()
        if capture is not None and self.fx is None:
            for m in range(self.N):
                capture[m] = self.outs[m].clone()
        wall = time.time() - w0
        self.launches = S.launch_count() - l0
        step_ms = [a.elapsed_time(b) for a, b in ev]
        mode_ms = [[kev[k][m][0].elapsed_time(kev[k][m][1]) for k in range(steps)]
                   for m in range(self.N)]
        return step_ms, mode_ms, wall

    def keep_busy(self, flush, seconds):
        """The same sweep loop, untimed, for `seconds`: gives the 100 ms clock sampler a window
        under this workload (the timed region itself is only tens of milliseconds long)."""
        import torch
        t0 = time.time()
        while True:
            for _ in range(20):
                flush.zero_()
                self.sweep()
            torch.cuda.synchronize()
            stop = torch.tensor([1.0 if time.time() - t0 >= seconds else 0.0], device=self.ctx.dev)
            if self.ctx.world > 1:
                import torch.distributed as dist
                dist.all_reduce(stop, op=dist.ReduceOp.MAX)      # every rank leaves together
            if stop.item() > 0.5:
                break

    def free(self):
        import torch
        self.T.free()
        self.fx = None
        self.mats = self.outs = None
        torch.cuda.empty_cache()


def parity_vs_reference(ctx, tag, dims, ind_host, vals_host, mats_h, ours_host):
    """rank 0: the reference's mttkrp_csf (default TWOMODE) on the same tensor vs our summed
    outputs; the other ranks sleep on the store meanwhile."""
    out = None
    if ctx.rank == 0:
        try:
            from oracle import ref
            if ref.available():
                rr = ReferenceRun(dims, ind_host, vals_host, 1)
                t0 = time.time()
                gold, _ = rr.sweep(mats_h, min(rr.aff, 32), 0, 1)
                rr.free()
                out = {"per_mode": [rel_fro(ours_host[m], gold[m]) for m in range(len(dims))],
                       "against": "reference mttkrp_csf (oracle/_ref, TWOMODE) on the same tensor",
                       "reference_seconds": time.time() - t0}
            else:
                out = {"per_mode": None, "against": "oracle/_ref not built"}
        except Exception as e:  # pragma: no cover
            out = {"per_mode": None, "error": f"{type(e).__name__}: {e}"}
    ctx.host_wait(f"parity/{tag}")
    return out


def run_named(ctx, key, args, flush):
    """One named multi-GPU configuration, whole tensor fixed (strong scaling)."""
    import torch
    spec = NAMED[key]
    dims, nnz, R = spec["dims"], spec["nnz"], spec["rank"]
    sampler = ClockSampler(ctx.local_rank).start() if ctx.rank == 0 else None
    ind, vals = make_coo_gpu(nnz, ctx.dev, dims, spec["seed"], spec["zipf"])
    ind_h = vals_h = None
    if ctx.rank == 0:
        ind_h = [i.cpu().numpy().astype(np.uint64) for i in ind]
        vals_h = vals.cpu().numpy()
    wl = Workload(ctx, dims, ind, vals, R, args.nccl_exchange, spec["seed"])
    del ind, vals
    torch.cuda.empty_cache()
    ours = wl.outputs_host()
    steps = args.steps
    step_ms, mode_ms, _ = wl.timed(flush, steps, max(args.warmup, 3))
    ms_per_step = ctx.max_over_ranks(float(np.sum(step_ms))) / steps
    per_mode = [ctx.max_over_ranks(float(np.mean(mode_ms[m]))) for m in range(wl.N)]
    wl.keep_busy(flush, 0.3)
    clocks = sampler.stop() if sampler else None
    par = parity_vs_reference(ctx, f"named{key}", dims, ind_h, vals_h, wl.mats_h, ours)
    rec = None
    if ctx.rank == 0:
        rec = {"workload": spec["name"] + f", whole tensor shared by {ctx.world} GPU(s) "
                                          "(strong scaling)",
               "dims": dims, "nnz_total": nnz, "rank": R, "n_gpus": ctx.world, "steps": steps,
               "ms_per_step": ms_per_step, "per_mode_ms": per_mode,
               "value": nnz * R * wl.N / (ms_per_step * 1e-3), "unit": "nnz*R/s",
               "per_mode_nnzR_per_s": [nnz * R / (t * 1e-3) for t in per_mode],
               "per_mode_ms_includes": "memset + kernel" if wl.fx is None and ctx.world == 1 else
                                       ("kernel incl. exchange and group barrier + re-zero"
                                        if wl.fx is not None else "memset + kernel (all-reduce follows)"),
               "exchange": wl.exchange, "clocks": clocks,
               "parity_rel_fro": par.get("per_mode") if par else None, "parity": par,
               "alg_bytes_local": [i["alg_bytes"] for i in wl.info],
               "nfibs_local": [i["nfibs"] for i in wl.info],
               "build_seconds": wl.build_s, "device_bytes_local": wl.T.device_bytes}
    wl.free()
    return rec


def e2e_c_abi(S, dims, R, ind_h, vals_h, mats_h, steps, ngpus):
    """The sweep through splatt_mttkrp_alloc_ws + splatt_mttkrp_csf with HOST buffers
    (H2D + kernel(s) + D2H + sync inside every call), pageable and page-locked.
    ngpus > 1: SPLATT_B200_NGPUS routes the same C entry to the single-process multi-GPU
    engine."""
    import torch
    res = {}
    o = S.default_opts()
    csf = S.csf_alloc(dims, ind_h, vals_h, o)
    old = os.environ.get("SPLATT_B200_NGPUS")
    if ngpus > 1:
        os.environ["SPLATT_B200_NGPUS"] = str(ngpus)
    try:
        ws = S.MttkrpWorkspace(csf.ptr, R, o)
        N = len(dims)
        for kind in ("pageable", "pinned"):
            if kind == "pinned":
                mats = [torch.from_numpy(m).pin_memory().numpy() for m in mats_h]
                outs = [torch.empty((d, R), dtype=torch.float64).pin_memory().numpy() for d in dims]
            else:
                mats = [np.array(m, copy=True) for m in mats_h]          # plain malloc'ed memory
                outs = [np.empty((d, R), dtype=np.float64) for d in dims]

            def sweep():
                for m in range(N):
                    ws.mttkrp_csf(mats, m, outs[m])
            # warm-up: >= 3 sweeps and >= 0.5 s -- the GPU (clocks, PCIe link state) has been
            # idle through the CPU-side reference runs that precede this phase
            tw, nw = time.perf_counter(), 0
            while nw < 3 or time.perf_counter() - tw < 0.5:
                sweep()
                nw += 1
            t0 = time.perf_counter()
            for _ in range(steps):
                sweep()
            res[kind] = (time.perf_counter() - t0) / steps * 1e3
            res[kind + "_out0"] = outs[0].copy() if kind == "pageable" else None
        ws.free()
    finally:
        if ngpus > 1:
            if old is None:
                os.environ.pop("SPLATT_B200_NGPUS", None)
            else:
                os.environ["SPLATT_B200_NGPUS"] = old
    return res, csf


def run_ours(args):
    import torch
    import torch.distributed as dist
    import splatt_b200 as S

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the CUDA extension is the product, "
                           "there is no CPU fallback")
    # NCCL's own log is left exactly as the environment asks (the driver reads the
    # communicator lines); the JSON line is printed last, after the process group is gone.
    ctx = Ctx()
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    n_gpus = world
    nnz_total = NNZ_PER_GPU * n_gpus
    dims = [DIM] * NMODES
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    sampler = ClockSampler(ctx.local_rank).start() if rank == 0 else None
    # ---- headline workload: identical tensor on every rank, each keeps its share of every stream
    ind, vals = make_coo_gpu(nnz_total, dev)
    wl = Workload(ctx, dims, ind, vals, RANK, args.nccl_exchange, SEED)
    ours_host = wl.outputs_host()          # also warms the GPU up before the W warm-up steps
    last = [None] * NMODES if args.dump_outputs else None
    step_ms, kern_ms, wall_s = wl.timed(flush, args.steps, max(args.warmup, 3), capture=last)
    if last is not None and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for m, out in enumerate(last):
            np.save(os.path.join(args.dump_outputs, f"mttkrp_mode{m}.npy"), out.cpu().numpy())
    del last
    launches = wl.launches
    ms_per_step = ctx.max_over_ranks(float(np.sum(step_ms))) / args.steps
    worst_step = ctx.max_over_ranks(float(np.max(step_ms)))
    best_step = ctx.max_over_ranks(float(np.min(step_ms)))
    value = nnz_total * RANK * NMODES / (ms_per_step * 1e-3)
    wl.keep_busy(flush, 0.6)               # clock samples under this very workload
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["window"] = ("build + warm-up + timed region + 0.6 s of the same sweep loop right "
                            "after it (the timed region alone is shorter than the 100 ms "
                            "sampling period)")
    ind_h = vals_h = None
    if rank == 0:
        ind_h = [i.cpu().numpy().astype(np.uint64) for i in ind]
        vals_h = vals.cpu().numpy()
    parity = parity_vs_reference(ctx, "weak", dims, ind_h, vals_h, wl.mats_h, ours_host)
    info = wl.info
    exchange = wl.exchange
    device_bytes = wl.T.device_bytes
    build_s = wl.build_s
    fused = wl.fx is not None

    # CPD-ALS iteration time at N > 1 (torch.distributed path): sharded MTTKRP + exchange +
    # replicated device tail
    cpd_multi = None
    if world > 1:
        try:
            from splatt_b200 import parallel
            init = [m[:, :RANK].contiguous() for m in wl.mats]
            tt = float((vals * vals).sum().item())
            _, _, _, its = parallel.cpd_als_sharded(wl.T, RANK, init, tt, niters=8, tol=0.0,
                                                    fused=fused)
            cpd_multi = {"rank": RANK,
                         "ours_ms": ctx.max_over_ranks(float(np.median(its[2:]))) * 1e3,
                         "path": "parallel.cpd_als_sharded: shard MTTKRP + exchange + device ALS "
                                 "tail on rank 0, factor broadcast (one process per GPU)"}
        except Exception as e:  # pragma: no cover
            cpd_multi = {"error": f"{type(e).__name__}: {e}"}
    mats_h = wl.mats_h
    wl.free()
    del ind, vals
    torch.cuda.empty_cache()

    # ---- named multi-GPU configurations (strong scaling)
    named = {}
    for key in [k for k in args.named.split(",") if k in NAMED]:
        try:
            named[key] = run_named(ctx, key, args, flush)
        except Exception as e:  # pragma: no cover
            log(f"[rank {rank}] named config {key} failed: {type(e).__name__}: {e}")
            named[key] = {"error": f"{type(e).__name__}: {e}"}
            ctx.host_wait(f"named-fail/{key}")

    # ---- e2e: host buffers through the reference-facing C ABI (rank 0 drives all N GPUs
    # from one process; the other ranks hold no work meanwhile)
    h2d = sum(dims[o] * RANK * 8 for m in range(NMODES) for o in range(NMODES) if o != m)
    d2h = sum(dims[m] * RANK * 8 for m in range(NMODES))
    e2e = csf = None
    del flush
    torch.cuda.empty_cache()
    ctx.barrier()
    if rank == 0:
        try:
            sampler2 = ClockSampler(ctx.local_rank).start()
            ind32 = [i.astype(np.uint32) for i in ind_h]
            res, csf = e2e_c_abi(S, dims, RANK, ind32, vals_h, mats_h, args.steps, world)
            e2e_clocks = sampler2.stop()
            gold0 = parity["per_mode"] if parity else None
            e2e = {"value": nnz_total * RANK * NMODES / (res["pageable"] * 1e-3), "unit": "nnz*R/s",
                   "ms_per_step": res["pageable"],
                   "buffers": "pageable host memory (what the reference's splatt_malloc returns), "
                              "staged through the workspace's page-locked bounce buffers",
                   "pinned": {"value": nnz_total * RANK * NMODES / (res["pinned"] * 1e-3),
                              "ms_per_step": res["pinned"]},
                   "pageable_over_pinned": res["pinned"] / res["pageable"],
                   "h2d_bytes_per_step": h2d * (world if world > 1 else 1), "d2h_bytes_per_step": d2h,
                   "path": "splatt_mttkrp_alloc_ws + splatt_mttkrp_csf (C ABI, host buffers)" +
                           ("" if world == 1 else f", SPLATT_B200_NGPUS={world}: single-process "
                            "multi-GPU engine (factors to every GPU over its own PCIe link, fused "
                            "multicast exchange, result back as one row slice per GPU)"),
                   "parity_rel_fro_mode0_vs_device_path": rel_fro(res["pageable_out0"], ours_host[0]),
                   "clocks": e2e_clocks}
            del gold0
        except Exception as e:  # pragma: no cover
            e2e = {"value": None, "unit": "nnz*R/s", "error": f"{type(e).__name__}: {e}",
                   "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}
    ctx.host_wait("e2e")

    line = None
    if rank == 0:
        # roofline of the dominant kernel: the root-stream kernel of mode 0
        peak, how = hbm_peak()
        k_ms = float(np.mean(kern_ms[0]))
        alg = info[0]["alg_bytes"]
        gather_numbers = {}
        try:
            if world == 1:
                peak_gbs, probe_ms = gather_probe_gbs(dev)
                gb = info[0]["nfibs"][-1] * RANK * 8 + info[0]["nfibs"][-2] * RANK * 8
                gather_numbers = {"achieved_GBps": gb / (k_ms * 1e-3) / 1e9,
                                  "probe_same_shape_GBps": peak_gbs, "probe_ms": probe_ms,
                                  "probe_sweep_best": probe_sweep_best()}
        except Exception as e:  # pragma: no cover
            gather_numbers = {"probe_error": str(e)}
        achieved = alg / (k_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": "mttkrp_stream_kernel<3,16,root> (mode 0)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": how, "alg_bytes_per_launch": alg,
                "launch_ms": k_ms, "traffic": ncu_traffic(),
                "per_mode_ms": [float(np.mean(k)) for k in kern_ms],
                "gather_path": dict(gather_numbers, **{
                    "bytes_per_launch": int(info[0]["nfibs"][-1] * RANK * 8 +
                                            info[0]["nfibs"][-2] * RANK * 8),
                    "note": "factor rows that must cross L2->SM per launch (one leaf row per "
                            "nonzero + one parent row per fiber); the L2->SM return path and the "
                            "L1 data pipe, not HBM, bound the kernel (DESIGN.md 4.1)"}),
                "kernel_share_of_step": float(sum(np.mean(k) for k in kern_ms) / ms_per_step),
                "launch_ms_includes": "memset + kernel" if not fused else
                                      "kernel incl. exchange + in-kernel group barrier + re-zero",
                "note": "alg bytes = 16 B/nnz record stream + 4 B/node upper-level ids + "
                        "3 factor-sized matrices (2 read, 1 written); SURVEY 8(d) at stored widths"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                from oracle import ref
                if ref.available():
                    step_s, cores, alloc = reference_best(dims, ind_h, vals_h, mats_h, 3, 1)
                    cv = nnz_total * RANK * NMODES / float(np.mean(step_s))
                    cpu = {"value": cv, "unit": "nnz*R/s", "cores": cores, "kind": "reference",
                           "sample": "full workload: 3 sweeps x 3 modes after 1 warm-up, reference "
                                     f"mttkrp_csf (OpenMP, {alloc}, untiled; the faster of TWOMODE / "
                                     "ALLMODE) at its fastest thread count among 8..all host threads "
                                     "(cores = that count)"}
                else:
                    step_s, cores = port_sweeps(ind_h, vals_h, mats_h, 1, 0)
                    cv = nnz_total * RANK * NMODES / float(np.mean(step_s))
                    cpu = {"value": cv, "unit": "nnz*R/s", "cores": cores, "kind": "port",
                           "sample": "full workload: 1 sweep x 3 modes, oracle/restate.c COO "
                                     "streaming MTTKRP on one host thread (oracle/_ref absent)"}
            except Exception as e:  # pragma: no cover
                cpu = {"value": None, "unit": "nnz*R/s", "cores": 0, "kind": "reference",
                       "sample": f"failed: {e}"}
        cpd = None
        if not args.no_cpu_baseline and csf is not None:
            try:
                if world == 1:
                    ind_t = [torch.from_numpy(i.astype(np.int64)) for i in ind_h]
                    cpd = cpd_iteration_times(S, csf, ind_t, torch.from_numpy(vals_h), mats_h,
                                              cpu.get("cores") if cpu and cpu.get("value") else None)
                else:
                    # the C entry behind splatt_cpd_als on all N GPUs from one process
                    # (splatt_b200_multi_cpd_als on one engine handle: the tensor is built and
                    # sharded once, two iteration counts are differenced)
                    from splatt_b200 import _abi as A
                    mg = S.MultiGpu(csf.ptr, A.CSF_TWOMODE, RANK, list(range(world)))

                    def ours(n):
                        o = S.default_opts()
                        o[3], o[1], o[4] = n, 0.0, 0
                        t0 = time.perf_counter()
                        fit, _, _ = mg.cpd_als(o, seed=SEED)
                        return time.perf_counter() - t0, fit
                    ours(2)
                    (ta, fit_a) = min(ours(110), ours(110))
                    (tb, _) = min(ours(10), ours(10))
                    cpd = dict(cpd_multi or {}, c_abi_ms=(ta - tb) / 100 * 1e3, c_abi_fit=fit_a,
                               c_abi_multicast=mg.multicast,
                               c_abi_path=f"splatt_b200_multi_cpd_als on {world} GPUs (what "
                                          "splatt_cpd_als runs with SPLATT_B200_NGPUS set): "
                                          "single-process multi-GPU engine, row-partitioned tail")
                    mg.free()
            except Exception as e:  # pragma: no cover
                cpd = dict(cpd_multi or {}, error=f"{type(e).__name__}: {e}")
        line = {"metric": "MTTKRP nnz*R/sec per mode", "value": value, "unit": "nnz*R/s",
                "n_gpus": n_gpus, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(n_gpus),      # identical in both arms
                "exchange": exchange,
                "clocks": clocks,
                "parity_rel_fro": parity.get("per_mode") if parity else None, "parity": parity,
                "step_ms_min": best_step, "step_ms_max": worst_step,
                "e2e": e2e,
                "gpu_launches": int(launches),
                "roofline": roof,
                "cpu_baseline": cpu,
                "named_configs": named,
                "named_config": named.get("4"),
                "cpd_als_iteration": cpd if cpd is not None else cpd_multi,
                "remeasured": False,
                "build_seconds": build_s, "wall_seconds_timed_region": wall_s,
                "device_bytes": device_bytes}
    ctx.host_wait("tail")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if world > 1:
            time.sleep(2.0)          # let the other ranks' NCCL teardown lines out first
        sys.stdout.flush()
        sys.stderr.flush()
        print(json.dumps(line), flush=True)
        # the JSON line must be the LAST line on stdout: with NCCL_DEBUG=INFO the library
        # prints from its exit handlers ("Closing env plugin ...") -- whatever is printed from
        # here on goes to stderr, and the process still ends through the normal interpreter
        # exit (atexit handlers, library destructors)
        os.dup2(sys.stderr.fileno(), sys.stdout.fileno())
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's per-mode outputs of the headline workload "
                         "as DIR/mttkrp_mode<m>.npy")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--nccl-exchange", action="store_true",
                    help="N>1: use kernel + NCCL all-reduce instead of the fused multicast exchange")
    ap.add_argument("--named", default="4,5",
                    help="named multi-GPU configs to run after the headline workload "
                         "(BASELINE.json configs[3] = 4, configs[4] = 5; '' = none)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
