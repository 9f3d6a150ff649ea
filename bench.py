#!/usr/bin/env python
"""bench.py -- headline benchmark of the embedding-similarity hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c1|c2|c3|c4|c5] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: 64 queries, top-10, scored against every
row of the HBM-resident synthetic store (SURVEY.md 8d generator).
  N = 1 : config C2 -- 1 000 000 x 384 fp32 store on one B200 (BASELINE.json configs[1]).
  N > 1 : config C3 -- 100 000 000 x 384 bf16 store row-sharded over N GPUs (100M/N rows each),
          local scan + exact rescoring, ONE ncclAllGather of the per-rank lists, device merge
          (strong scaling: the store is fixed, rows per GPU shrink with N).
One JSON line on stdout (rank 0).  `value` = queries/s with queries and outputs resident in
HBM; `e2e` = the same metric through the public host-buffer API (pinned host queries in, host
results out, copies inside the timed region).  The same line carries, at every N:
  parity      the timed call checked IN THIS RUN: against the binary64 scan of every row (all queries; for N > 1
              against the host merge of the per-shard binary64 scans, and identical lists on every rank), and
              against the CPU oracle on rank 0 (>= 8 queries); a mismatch exits non-zero
  certification  how many timed queries the first pass could not certify and what settled them
  dedup       config C4 (all-pairs, 1M x 768 bf16, threshold 0.9) on the same N GPUs: pairs/s, TFLOP/s per GPU
  streaming   config C5 (4096-row inserts interleaved with single-query top-10 over 10M x 384): p50/p99
  clustered   the main workload on a unit-norm Gaussian-mixture store with non-representable values
  reference_size  (N = 1) config C1, the reference's own size: 5 000 x 384 store, 30 queries, L2 flushed before every step
  cpu_baseline  the oracle port on the box's host cores (bounded sample)
`--impl reference` times the reference's CPU algorithm (oracle port, all host threads) on the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "queries_per_sec_top10_384d"
UNIT = "queries/s"
CONFIGS = {
    # name: (rows_total, dim, store dtype, queries, k, store seed, query seed)
    "c1": (5_000, 384, "f32", 30, 10, 1, 1001),      # the reference's own size (LIMIT 5000 store, 30 benchmark queries)
    "c2": (1_000_000, 384, "f32", 64, 10, 2, 2002),
    "c3": (100_000_000, 384, "bf16", 64, 10, 3, 3003),
    "c5": (10_000_000, 384, "f32", 1, 10, 5, 5005),
}
# all-pairs dedup: rows, dim, dtype, threshold, seed, planted-duplicate period
C4 = (1_000_000, 768, "bf16", 0.9, 4, 100)


def _use_all_host_cores() -> int:
    """torchrun pins OMP_NUM_THREADS=1 in every worker and an OpenMP runtime reads the variable only once, when it is
    initialised -- so the CPU legs (rank 0 only) also set the thread count of the runtime that is already loaded."""
    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)
    try:
        import ctypes
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(cores)
    except Exception:  # pragma: no cover
        pass
    return cores


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
        except Exception:
            pass
    return 1400.0, "fallback (B200_PROFILING.md sustained)"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict):
    """--dump-outputs: writes each array as out_dir/<name>.npy -- integers and float64 as float64, float32 as float32 -- so
    that two builds can be compared output for output.  Arrays share their leading dimension; when together they exceed
    64 MB, a fixed, seeded sample of that dimension (the same rows of every array) is written, with the chosen positions
    as sample_rows.npy."""
    import numpy as np
    arrays = {name: np.asarray(a) for name, a in arrays.items()}
    arrays = {name: a.astype(np.float32 if a.dtype == np.float32 else np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        n = len(next(iter(arrays.values())))
        keep = int((DUMP_LIMIT_BYTES - 4096) / (total / n + 8))     # 8 bytes a row for sample_rows, 4 KB for the headers
        pick = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {name: a[pick] for name, a in arrays.items()}
        arrays["sample_rows"] = pick.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """SM clocks and throttle reasons sampled DURING the timed region (in-process NVML polling,
    ~2 ms period: a subprocess `nvidia-smi -lms` starts too slowly for a region of tens of ms)."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index: int, period_s: float = 0.002):
        # period_s: NVML queries take the driver's resource-manager lock, which memory-management calls (cuMemCreate /
        # cuMemMap of a growing store, cudaMalloc) need as well -- at the 2 ms period a growth step of the streaming record
        # was seen stalling for 100-200 ms behind the sampler, so records with long timed regions poll every 50 ms
        self.period_s = float(period_s)
        self.gpu, self.samples, self.mask, self.smax, self.err = gpu_index, [], 0, None, None
        self._stop = threading.Event()
        self.t = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except Exception:
                    idx = self.gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # pragma: no cover
            self.err = repr(e)
            return self
        self.t = threading.Thread(target=self._poll, daemon=True)
        self.t.start()
        return self

    def _poll(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception as e:
                self.err = repr(e)
                return
            time.sleep(self.period_s)

    def stop(self):
        self._stop.set()
        if self.t:
            self.t.join(timeout=1)
        reasons = sorted(n for bit, n in self.REASONS.items() if self.mask & bit)
        if self.err and not self.samples:
            reasons = ["nvml unavailable: " + self.err]
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.smax,
                "reasons": reasons, "samples": len(self.samples)}


def _ncu_traffic(dt: str, rows_local: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of the scan kernel, per launch, from the committed
    `ncu --set full` capture of this dtype and shard size (profiles/*scan*summary.json); None when no
    capture of exactly this shape exists."""
    pdir = os.path.join(ROOT, "profiles")
    try:
        names = sorted(os.listdir(pdir), reverse=True)     # later rounds first
    except OSError:
        return None
    for name in names:
        if "scan" not in name or not name.endswith("_summary.json"):
            continue
        try:
            d = json.load(open(os.path.join(pdir, name)))
            if int(d.get("rows", -1)) == int(rows_local) and str(d.get("store_dtype", dt)) == dt:
                return float(d["dram_bytes_read"]) + float(d["dram_bytes_write"])
        except Exception:
            continue
    return None


def _ncu_pairs_pipe():
    """Tensor-pipe activity of pairs_tc2_kernel from the committed `ncu --set full` capture (profiles/*pairs*summary.json,
    latest round first): {"pct", "rows", "file"} or None."""
    pdir = os.path.join(ROOT, "profiles")
    try:
        names = sorted((n for n in os.listdir(pdir) if "pairs" in n and n.endswith("_summary.json")), reverse=True)
    except OSError:
        return None
    for name in names:
        try:
            d = json.load(open(os.path.join(pdir, name)))
            if d.get("tensor_pipe_active_pct") is not None:
                return {"pct": float(d["tensor_pipe_active_pct"]), "rows": int(d.get("rows", 0)), "file": "profiles/" + name}
        except Exception:
            continue
    return None


def _ncu_pairs_full_size(rows: int):
    """The committed ncu pass of pairs_tc2_kernel at exactly `rows` rows (profiles/*pairs*summary.json): per-launch DRAM
    traffic, tensor-pipe activity, SM clock under the profiler; None when no capture of this size exists."""
    pdir = os.path.join(ROOT, "profiles")
    try:
        names = sorted((n for n in os.listdir(pdir) if "pairs" in n and n.endswith("_summary.json")), reverse=True)
    except OSError:
        return None
    for name in names:
        try:
            d = json.load(open(os.path.join(pdir, name)))
            if int(d.get("rows", -1)) == int(rows) and d.get("dram_bytes_read") is not None:
                return {"traffic": float(d["dram_bytes_read"]) + float(d.get("dram_bytes_write") or 0.0),
                        "tensor_pipe_active_pct": d.get("tensor_pipe_active_pct"), "tflops_under_ncu": d.get("tflops"),
                        "sm_clock_ghz": d.get("sm_clock_ghz"), "l2_hit_rate_pct": d.get("l2_hit_rate_pct"), "file": "profiles/" + name}
        except Exception:
            continue
    return None


class Ctx:
    """Process-wide state of one bench run (rank, device, communicator)."""

    def __init__(self, args):
        import torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world > 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.comm = None
        self.peer_exchange = False
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            from vidmem_b200.sharded import Communicator
            self.comm = Communicator.from_torch_distributed(self.local_rank)
            self.peer_exchange = bool(args.peer_exchange and self.comm.enable_peer_exchange())

    def barrier(self):
        import torch
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, values):
        import torch
        if self.world == 1:
            return [float(v) for v in values]
        import torch.distributed as dist
        t = torch.tensor(list(values), device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def all_true(self, flag: bool) -> bool:
        return self.max_over_ranks([0.0 if flag else 1.0])[0] == 0.0

    def close(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
            if self.comm is not None:
                self.comm.close()
            dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port (C restatement of the reference's Python loop)
# ---------------------------------------------------------------------------------------------
def cpu_reference_leg(cfg_name: str, steps: int, warmup: int, sample_rows: int):
    """Times the reference algorithm (pre_llm_injector.py:346-388 restated in C, OpenMP over
    queries) on `sample_rows` rows of the same synthetic store; returns (queries/s at the FULL
    store size by linear extrapolation in rows -- the algorithm is a flat loop over rows --,
    ms per sampled step, description)."""
    import numpy as np
    from oracle import oracle, synth
    rows_total, dim, _dt, nq, k, sseed, qseed = CONFIGS[cfg_name]
    sample_rows = min(sample_rows, rows_total)
    X = synth.synth_rows(sseed, 0, sample_rows, dim).astype(np.float64)
    Q = synth.synth_queries(qseed, nq, dim, sseed, rows_total).astype(np.float64)
    oracle.lib()
    for _ in range(warmup):
        oracle.batch_similarities(Q, X, k)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        oracle.batch_similarities(Q, X, k)
        times.append(time.perf_counter() - t0)
    per_step = sum(times) / len(times)
    full = per_step * (rows_total / sample_rows)
    what = "the full store" if sample_rows == rows_total else f"{sample_rows} of {rows_total} rows, time scaled linearly in rows to the full store"
    return nq / full, per_step * 1e3, f"{nq} queries x {sample_rows} rows x {dim}: {what}"


def cpu_interpreter_leg(cfg_name: str, n_queries: int):
    """The reference's own execution model (SURVEY 8d "ref_python"): one interpreter thread, generator expressions over
    Python floats (oracle/pyloop.py restates pre_llm_injector.py:346-388), on `n_queries` queries of the config against
    the full store -- only sensible at C1's size (~60 us per pair).  Its lists must equal the C port's bit for bit."""
    from oracle import oracle, pyloop, synth
    rows_total, dim, _dt, nq, k, sseed, qseed = CONFIGS[cfg_name]
    X = synth.synth_rows(sseed, 0, rows_total, dim)
    Q = synth.synth_queries(qseed, nq, dim, sseed, rows_total)[:n_queries]
    store = {i: [float(v) for v in X[i]] for i in range(rows_total)}
    queries = [[float(v) for v in q] for q in Q]
    t0 = time.perf_counter()
    got = pyloop.batch_similarities(queries, store, k)
    dt = time.perf_counter() - t0
    mode = oracle.SUM_NEUMAIER if sys.version_info >= (3, 12) else oracle.SUM_NAIVE
    same = got == oracle.batch_similarities(Q, X, k, sum_mode=mode)
    return {"value": len(queries) / dt, "unit": UNIT, "cores": 1, "kind": "port (CPython loop)", "us_per_pair": dt / (len(queries) * rows_total) * 1e6,
            "sample": f"{len(queries)} of {nq} queries x {rows_total} rows x {dim}, one interpreter thread", "equals_c_port": bool(same)}


def cpu_blas_leg(cfg_name: str, sample_rows: int):
    """The reference's own vectorised idiom (src/pipeline/prune.py:62,76): sklearn cosine_similarity (BLAS
    sgemm over every host core, store re-normalised on every call) + argpartition/sort for the top-k, on the
    same bounded sample.  Context only: float32, not the bit-exact reference order."""
    import numpy as np
    from sklearn.metrics.pairwise import cosine_similarity
    from oracle import synth
    rows_total, dim, _dt, nq, k, sseed, qseed = CONFIGS[cfg_name]
    sample_rows = min(sample_rows, rows_total)
    X = synth.synth_rows(sseed, 0, sample_rows, dim)
    Q = synth.synth_queries(qseed, nq, dim, sseed, rows_total)
    cosine_similarity(Q[:2], X[:1000])
    t0 = time.perf_counter()
    S = cosine_similarity(Q, X)
    part = np.argpartition(-S, k - 1, axis=1)[:, :k]
    np.take_along_axis(S, part, 1).sort(axis=1)
    dt = time.perf_counter() - t0
    return nq / (dt * rows_total / sample_rows)


def run_reference(args):
    """The reference arm: the reference's own CPU algorithm for this path (the oracle port: the reference is pure
    Python, there is no C source to compile) with every host thread, on our arm's workload.  --steps / --warmup
    are honoured; each step scores the 64-query batch against as many rows of the store as keep the whole run
    inside ~150 s (all of them for C2 on a 16-core box), stated in `sample`."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun pins OMP_NUM_THREADS=1 in every worker; the reference arm is meant to use every host core
    _use_all_host_cores()
    cfg = args.config if args.config in CONFIGS else ("c2" if args.gpus == 1 else "c3")
    cores = os.cpu_count() or 1
    rows_total, dim, dt, nq, k, _, _ = CONFIGS[cfg]
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    if args.cpu_sample_rows:
        sample = args.cpu_sample_rows
    else:
        _q, probe_ms, _d = cpu_reference_leg(cfg, 1, 1, 20000)          # calibrate: ms per 20 000 rows
        budget_ms = 150e3 / (steps + warmup)
        sample = int(min(rows_total, max(20000, 20000 * budget_ms / max(probe_ms, 1e-3))))
        if sample >= rows_total // 2:
            sample = rows_total
    qps, ms, desc = cpu_reference_leg(cfg, steps, warmup, sample)
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{cfg}: {rows_total}x{dim} {dt} store, {nq}-query batch, top-{k} cosine",
                       "timed_sample": desc, "ms_per_step_is": "one timed step over the sampled rows (value is extrapolated to the full store)"},
            "cpu_baseline": {"value": qps, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
            "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def make_queries(store, n_rows: int, nq: int, dim: int, seed: int, dev, world: int = 1):
    """Synthetic query batch for the timed arm (no oracle code on this path): even queries are copies of a
    resident row with every 4th column redrawn, odd queries are independent draws; all values are multiples
    of 1/128 like the store rows.  Under torchrun rank 0's batch is broadcast so every rank scores the same
    queries.  -> float32 CPU tensor [nq, dim]."""
    import torch
    g = torch.Generator(device="cpu").manual_seed(seed)
    ridx = torch.randint(0, max(n_rows, 1), (nq,), generator=g)
    base = store.rows[ridx.to(dev), :dim].float()
    noise = (torch.randint(-127, 128, (nq, dim), generator=g).float() / 128.0).to(dev)
    redraw = (torch.arange(dim, device=dev) % 4 == 0)[None, :] | (torch.arange(nq, device=dev) % 2 == 1)[:, None]
    q = torch.where(redraw, noise, base).contiguous()
    if world > 1:
        import torch.distributed as dist
        dist.broadcast(q, src=0)
    return q.cpu()


def _hash_normal(ids, dim: int, seed: int):
    """Standard-normal [len(ids), dim] tensor that is a pure function of (seed, id, column): splitmix-style integer
    mixing (int64 wrap-around) + Box-Muller, so any rank can produce any row or centre without a shared stream."""
    import math
    import torch
    j = torch.arange(dim, device=ids.device, dtype=torch.int64)
    z = ids.to(torch.int64)[:, None] * -7046029254386353131 + j[None, :] * -4658895280553007687 + (seed * 2654435761 + 12345)
    z = (z ^ (z >> 30)) * -4658895280553007687
    z = (z ^ (z >> 27)) * -7723592293110705685
    z = z ^ (z >> 31)
    u1 = ((z & 0xFFFFFF).to(torch.float32) + 0.5) * (1.0 / 16777216.0)
    u2 = (((z >> 24) & 0xFFFFFF).to(torch.float32) + 0.5) * (1.0 / 16777216.0)
    return torch.sqrt(-2.0 * torch.log(u1)) * torch.cos((2.0 * math.pi) * u2)


def fill_clustered(store, n: int, dim: int, seed: int, per_centre: int, rho: float, row_lo: int = 0):
    """Unit-norm Gaussian-mixture rows written straight into the store's HBM: centre c = global row // per_centre,
    row = normalise(unit(centre_c) + rho * g / sqrt(dim)), g ~ N(0, I) -- `per_centre` near-duplicates per centre
    (cosine between members ~ 1 / (1 + rho^2)); values are NOT representable in bf16 / tf32."""
    import torch
    dev = store.device
    chunk = 1 << 17
    for r0 in range(0, n, chunk):
        m = min(chunk, n - r0)
        rows = torch.arange(row_lo + r0, row_lo + r0 + m, device=dev, dtype=torch.int64)
        uc, inv = torch.unique(rows // per_centre, return_inverse=True)
        cvec = _hash_normal(uc, dim, seed * 2 + 1)
        cvec = cvec / cvec.norm(dim=1, keepdim=True)
        x = cvec[inv] + (rho / dim ** 0.5) * _hash_normal(rows, dim, seed * 2)
        x = x / x.norm(dim=1, keepdim=True)
        store.rows[r0:r0 + m, :dim] = x.to(store.rows.dtype)
        if store.ld > dim:
            store.rows[r0:r0 + m, dim:] = 0


# ---------------------------------------------------------------------------------------------
# parity of the timed call, checked inside the run
# ---------------------------------------------------------------------------------------------
def parity_topk(ctx: Ctx, store, q_dev, k: int, row_lo: int, flags_timed: int, exact_queries: int):
    """(1) the timed call (fast scan + certification, sharded merge for N > 1) against the binary64 scan of every
    row (VM_FLAG_FORCE_EXACT) of the same store: N = 1 directly; N > 1 against the HOST merge (numpy) of the per-shard
    binary64 scans, so neither the fast scan nor the NCCL exchange nor the merge kernel is its own witness;
    (2) N > 1: every rank holds identical lists.  Index lists equal, binary64 scores bit-equal."""
    import numpy as np
    import torch
    import vidmem_b200 as vm
    from vidmem_b200.sharded import merge_lists_host
    nq = q_dev.shape[0]
    got = store.topk_device(q_dev, k, flags=flags_timed & ~vm.VM_FLAG_TIMING, comm=ctx.comm, row_offset=row_lo)
    torch.cuda.synchronize()
    g_idx, g_score, g_count = (t.cpu().numpy().copy() for t in got)
    ne = min(nq, exact_queries)
    t0 = time.perf_counter()
    ex = store.topk_device(q_dev[:ne].contiguous(), k, flags=vm.VM_FLAG_FORCE_EXACT)       # local shard, local rows
    torch.cuda.synchronize()
    exact_s = time.perf_counter() - t0
    e_idx, e_score, e_count = (t.cpu().numpy().copy() for t in ex)
    e_idx = np.where(e_idx >= 0, e_idx + row_lo, e_idx)
    identical = True
    if ctx.world > 1:
        import torch.distributed as dist
        packs = [None] * ctx.world
        dist.all_gather_object(packs, (e_idx, e_score, e_count, g_idx, g_score, g_count))
        e_idx, e_score, e_count = merge_lists_host([(p[0], p[1], p[2]) for p in packs], k)
        identical = all(np.array_equal(p[3], packs[0][3]) and np.array_equal(p[4].view(np.int64), packs[0][4].view(np.int64))
                        and np.array_equal(p[5], packs[0][5]) for p in packs)
    ok = identical and np.array_equal(g_count[:ne], e_count[:ne])
    for qi in range(ne):
        c = int(e_count[qi])
        ok = ok and np.array_equal(g_idx[qi, :c], e_idx[qi, :c]) and np.array_equal(g_score[qi, :c].view(np.int64), e_score[qi, :c].view(np.int64))
    ok = ctx.all_true(bool(ok))
    return {"checked": "timed call vs binary64 scan of every row" + (" (host merge of per-shard exact scans) + identical lists on every rank" if ctx.world > 1 else ""),
            "queries": int(ne), "ok": bool(ok), "identical_across_ranks": bool(identical) if ctx.world > 1 else None,
            "exact_scan_s": round(exact_s, 3)}, (g_idx, g_score, g_count)


def parity_oracle(store, q_host, k: int, n_queries: int, max_rows: int):
    """Rank 0, after the timed region: the default (fast) path over the first `rows` resident rows against the CPU
    oracle's blocked tier (float64 BLAS pre-ranking + bit-exact reference rescoring) on the same rows copied back
    from HBM.  Index lists equal, binary64 scores bit-equal."""
    import numpy as np
    import torch
    from oracle import oracle
    n = min(len(store), max_rows)
    view = store.prefix_view(n) if n < len(store) else store
    try:
        Q = np.ascontiguousarray(q_host[:n_queries], dtype=np.float32)
        idx, score, count = view.topk(Q, k)
        X = store.rows[:n, :store.dim].float().cpu().numpy()
        t0 = time.perf_counter()
        oi, os_, oc = oracle.topk_blocked(Q, X, k)
        dt = time.perf_counter() - t0
        ok = bool(np.array_equal(count, oc.astype(count.dtype)))
        for qi in range(len(Q)):
            c = int(oc[qi])
            ok = ok and np.array_equal(idx[qi, :c], oi[qi, :c]) and np.array_equal(score[qi, :c].view(np.int64), os_[qi, :c].view(np.int64))
        return {"checked": "default path vs CPU oracle (blocked tier, bit-exact rescoring)", "queries": int(len(Q)), "rows": int(n),
                "ok": bool(ok), "oracle_s": round(dt, 2)}
    finally:
        if view is not store:
            view.close()


def parity_oracle_f64(store, q_host, k: int, n_queries: int, max_rows: int):
    """Binary64 store: the default path over the first `rows` resident rows against the CPU oracle's plain reference
    loop (vo_batch_similarities: every query x every row, reference summation order) on the float64 ORIGINALS copied
    back from HBM.  Index lists equal, binary64 scores bit-equal."""
    import numpy as np
    from oracle import oracle
    n = min(len(store), max_rows)
    view = store.prefix_view(n) if n < len(store) else store
    try:
        Q = np.ascontiguousarray(q_host[:n_queries], dtype=np.float64)
        idx, score, count = view.topk(Q, k)
        X = store.rows_exact[:n, :store.dim].cpu().numpy()
        t0 = time.perf_counter()
        ref = oracle.batch_similarities(Q, X, k)
        dt = time.perf_counter() - t0
        ok = all(int(count[qi]) == len(lst) and [int(v) for v in idx[qi, :len(lst)]] == [r for r, _ in lst]
                 and [float(v) for v in score[qi, :len(lst)]] == [sc for _, sc in lst] for qi, lst in enumerate(ref))
        return {"checked": "default path vs CPU oracle (plain reference loop on the float64 originals)", "queries": int(len(Q)),
                "rows": int(n), "ok": bool(ok), "oracle_s": round(dt, 2)}
    finally:
        if view is not store:
            view.close()


# ---------------------------------------------------------------------------------------------
# top-k scorer (C1 / C2 / C3, clustered variant)
# ---------------------------------------------------------------------------------------------
def bench_topk(ctx: Ctx, args, cfg: str, steps: int, warmup: int, variant: str = "iid", with_e2e: bool = True,
               with_parity: bool = True, rows_override=None, store_dtype=None, cluster_rho=None, dump_dir=None):
    """store_dtype "f64" / "f64+bf16": the same workload on a BINARY64 store -- rows kept as float64 originals (here the
    synthetic values times (1 + 1e-9 g), g ~ N(0,1): not representable in fp32 / bf16), the scan streams their rounded
    fp32 / bf16 shadow, every exact step reads the originals; queries are float64 too.
    dump_dir: rank 0 writes the (idx, score, count) lists of the last timed step there."""
    import numpy as np
    import torch
    import vidmem_b200 as vm
    from vidmem_b200.store import EmbeddingStore
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    rows_total, dim, dt, nq, k, sseed, qseed = CONFIGS[cfg]
    if rows_override:
        rows_total = rows_override
    rho = args.cluster_rho if cluster_rho is None else float(cluster_rho)
    row_lo = rows_total * rank // world
    row_hi = rows_total * (rank + 1) // world
    n_local = row_hi - row_lo
    exact_store = store_dtype in ("f64", "f64+bf16")
    if store_dtype:
        dt = "bf16" if store_dtype in ("bf16", "f64+bf16") else "f32"      # what the scan streams
    es = 4 if dt == "f32" else 2

    store = EmbeddingStore(dim, n_local, store_dtype or dt, device=ctx.local_rank)
    if variant == "iid":
        store.synth_fill(sseed, n_local, row0=row_lo)
        store.set_size(n_local)            # binary64 store: the originals start as the widened shadow values
        torch.cuda.synchronize()
        q_pinned = make_queries(store, n_local, nq, dim, qseed, dev, world)
        if exact_store:
            # originals off the fp32 / bf16 grid: relative 1e-9 is far below half an ulp of either shadow type, so the
            # shadow (and its cached norms) IS the rounding of these originals
            for r0 in range(0, n_local, 1 << 17):
                m = min(1 << 17, n_local - r0)
                ids = torch.arange(row_lo + r0, row_lo + r0 + m, device=dev, dtype=torch.int64)
                store.rows_exact[r0:r0 + m, :dim] *= (1.0 + 1e-9 * _hash_normal(ids, dim, sseed + 77).double())
            q_pinned = q_pinned.double() * (1.0 + 1e-9 * torch.randn(q_pinned.shape, generator=torch.Generator().manual_seed(qseed), dtype=torch.float64))
        q_pinned = q_pinned.pin_memory()
    else:
        fill_clustered(store, n_local, dim, sseed, args.cluster_size, rho, row_lo)
        store.set_size(n_local)
        torch.cuda.synchronize()
        # queries: perturbed members of random clusters (so the top-k sits inside a near-duplicate cluster)
        g = torch.Generator(device="cpu").manual_seed(qseed)
        ridx = torch.randint(0, max(n_local, 1), (nq,), generator=g)
        base = store.rows[ridx.to(dev), :dim].float()
        q = base + (rho / dim ** 0.5) * torch.randn((nq, dim), generator=g).to(dev)
        if world > 1:
            import torch.distributed as dist
            dist.broadcast(q, src=0)
        q_pinned = q.cpu().contiguous().pin_memory()
    Q = q_pinned.numpy()
    q_dev = q_pinned.to(dev)
    out = (torch.empty((nq, k), dtype=torch.int64, device=dev), torch.empty((nq, k), dtype=torch.float64, device=dev),
           torch.empty((nq,), dtype=torch.int32, device=dev))
    flags_dev = vm.VM_FLAG_ASYNC | args.flags

    def step_device():
        store.topk_device(q_dev, k, out=out, flags=flags_dev, comm=ctx.comm, row_offset=row_lo)

    parity = None
    if with_parity:
        parity, _ = parity_topk(ctx, store, q_dev, k, row_lo, flags_dev, nq if n_local <= 16_000_000 else 8)

    # ---- leg 1: inputs resident in HBM ------------------------------------------------------
    warm = max(warmup, 3)
    for _ in range(warm):
        step_device()
    ctx.barrier()
    store.counters(reset=True)   # certification counters of the timed region only
    sampler = ClockSampler(ctx.local_rank)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fits_l2 = n_local * dim * es <= 126e6
    ctx.barrier()
    if not fits_l2:
        ev0.record()
        for _ in range(steps):
            step_device()
        ev1.record()
        ctx.barrier()
        dev_ms = ev0.elapsed_time(ev1)
    else:
        # store fits the 126 MB L2: flush it (write a 256 MB buffer) before every step and time the steps one by one
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        dev_ms = 0.0
        for _ in range(steps):
            flush.zero_()
            ev0.record()
            step_device()
            ev1.record()
            ev1.synchronize()
            dev_ms += ev0.elapsed_time(ev1)
        ctx.barrier()
        del flush
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"topk_idx": out[0].cpu(), "topk_score": out[1].cpu(), "topk_count": out[2].cpu()})
    stats = store.last_stats
    launches = int(stats.scan_launches) * steps
    cert = store.counters(reset=True)
    band_kept = band_spilled = None
    if int(stats.scan_kernel) == 2 and int(stats.scan_variant) == 2:
        bk, bs = store.band_keys()
        band_kept, band_spilled = float(bk.mean()), float(bs.mean())
    # scan-kernel time: the same loop once more with VM_FLAG_TIMING -- every step then carries its own CUDA event pair
    # around the scan kernel on the launching stream (an event between two kernels rules out their programmatic
    # overlap, so the timed region above runs without it); the average over the last <= 64 steps is read back
    for _ in range(2):
        store.topk_device(q_dev, k, out=out, flags=flags_dev | vm.VM_FLAG_TIMING, comm=ctx.comm, row_offset=row_lo)
    torch.cuda.synchronize()
    store.avg_scan_ms()
    ctx.barrier()
    if fits_l2:
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    for _ in range(min(steps, 64)):
        if fits_l2:
            flush.zero_()
        store.topk_device(q_dev, k, out=out, flags=flags_dev | vm.VM_FLAG_TIMING, comm=ctx.comm, row_offset=row_lo)
    scan_avg_live, scan_calls = store.avg_scan_ms()
    store.counters(reset=True)
    ctx.barrier()

    # ---- leg 2: end to end through the host-buffer API ----------------------------------------
    e2e_ms = float("nan")
    if with_e2e:
        def step_host():
            return store.topk(q_pinned.numpy(), k, comm=ctx.comm, row_offset=row_lo, flags=args.flags)

        for _ in range(3):
            step_host()
        ctx.barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step_host()
        e1.record()
        ctx.barrier()
        e2e_wall_ms = (time.perf_counter() - t0) * 1e3
        e2e_ms = max(e0.elapsed_time(e1), e2e_wall_ms)  # host-synchronous API: wall clock is the honest number
    clocks = sampler.stop() if rank == 0 else None
    dev_ms, e2e_ms, scan_avg = ctx.max_over_ranks([dev_ms, e2e_ms if with_e2e else 0.0, scan_avg_live])

    oracle_par = None
    if rank == 0 and with_parity and not args.no_cpu_baseline:
        oracle_par = parity_oracle_f64(store, Q, k, 8, 150_000) if exact_store else parity_oracle(store, Q, k, 8, 2_000_000)

    rec = None
    if rank == 0:
        ms_per_step = dev_ms / steps
        peak, peak_src = _peaks()
        alg_bytes = n_local * dim * es + n_local * 4          # store rows once + cached inverse norms
        achieved = alg_bytes / (scan_avg * 1e-3) / 1e9 if scan_avg > 0 else 0.0
        n_q = max(int(cert["queries"]), 1)
        rec = {
            "metric": METRIC, "value": nq / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None,
            "dtype": "tf32" if (dt == "f32" and stats.scan_kernel == 2) else ("f32" if dt == "f32" else "bf16"),
            "data": "synthetic",
            "config": {"workload": f"{cfg}: {rows_total}x{dim} {store_dtype or dt} store" + (f" (binary64 rows + {dt} shadow)" if exact_store else "")
                                   + f", {nq}-query batch, top-{k} cosine, "
                                   f"{'row-sharded over %d GPUs + NCCL all-gather merge' % world if world > 1 else '1 GPU'}",
                       "variant": ("iid: counter-hash integers / 128 (SURVEY 8d)" if variant == "iid" else
                                   f"clustered: unit-norm Gaussian mixture, {args.cluster_size} near-duplicates per centre, "
                                   f"noise rho={rho} (cosine between members ~{1 / (1 + rho ** 2):.4f}), non-representable values"),
                       "rows_per_gpu": n_local,
                       "l2_policy": ("inputs larger than L2 (%.0f MB store per GPU vs 126 MB L2)" % (n_local * dim * es / 1e6))
                       if not fits_l2 else
                       ("store (%.1f MB) fits L2: L2 flushed (256 MB write) before every timed step, steps timed one by one" % (n_local * dim * es / 1e6)),
                       "scan_kernel": {0: "exact_fp64", 1: "simt", 2: "tcgen05"}[int(stats.scan_kernel)],
                       "scan_variant": {0: "lists", 1: "dump", 2: "slabs+bound service"}.get(int(stats.scan_variant), "?"),
                       "scan_ctas": int(stats.scan_ctas), "candidates_per_query": int(stats.candidates),
                       "exact_rescoring": "binary64, reference summation order (Neumaier)",
                       "timing": "cuda events around the K timed steps, max over ranks; roofline.kernel_ms from a second pass of the same "
                                 "loop with one event pair per scan kernel",
                       "exchange": ("peer memory (symmetric buffers, NVLink pull-merge kernel)" if ctx.peer_exchange else
                                    "ncclAllGather + merge kernel") if world > 1 else "none"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": _ncu_traffic(dt, n_local), "kernel": "scan_tc_kernel", "kernel_ms": scan_avg,
                         "kernel_ms_samples": scan_calls, "algorithmic_bytes": alg_bytes, "peak_source": peak_src,
                         "step_frac": alg_bytes / (ms_per_step * 1e-3) / 1e9 / peak},
            "certification": {"queries_timed": int(cert["queries"]), "uncertified": int(cert["uncertified"]),
                              "certified_pct": 100.0 * (1.0 - cert["uncertified"] / n_q),
                              "band_settled": int(cert["band_settled"]), "collect_settled": int(cert["collect_settled"]),
                              "full_rescans": int(cert["full_rescans"]), "bound_violations": int(cert["bound_violations"]),
                              "band_keys_per_query": band_kept, "spilled_keys_per_query": band_spilled,
                              "note": "rank 0's shard; counted on the device over the timed steps (VM_FLAG_ASYNC)"},
            "parity": parity,
            "clocks": clocks,
        }
        if with_e2e:
            rec["e2e"] = {"value": nq / (e2e_ms / steps * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(Q.nbytes),
                          "d2h_bytes_per_step": int(nq * k * 16 + nq * 4 + 4), "ms_per_step": e2e_ms / steps}
        if oracle_par is not None:
            rec["parity"]["oracle"] = oracle_par
            rec["parity"]["ok"] = bool(rec["parity"]["ok"] and oracle_par["ok"])
    store.close()
    del store, q_dev, out
    torch.cuda.empty_cache()
    return rec


def scaling_baseline(ctx: Ctx):
    """C3 (the N > 1 workload) on ONE GPU, so that the N = 2/4/8 lines have a same-workload N = 1 reference."""
    import torch
    import vidmem_b200 as vm
    from vidmem_b200.store import EmbeddingStore
    try:
        r3, d3, dt3, nq3, k3, ss3, qs3 = CONFIGS["c3"]
        s3 = EmbeddingStore(d3, r3, dt3, device=ctx.local_rank)
        s3.synth_fill(ss3, r3)
        s3.set_size(r3)
        q3 = make_queries(s3, r3, nq3, d3, qs3, ctx.dev).to(ctx.dev)
        o3 = (torch.empty((nq3, k3), dtype=torch.int64, device=ctx.dev), torch.empty((nq3, k3), dtype=torch.float64, device=ctx.dev),
              torch.empty((nq3,), dtype=torch.int32, device=ctx.dev))
        for _ in range(3):
            s3.topk_device(q3, k3, out=o3, flags=vm.VM_FLAG_ASYNC)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(10):
            s3.topk_device(q3, k3, out=o3, flags=vm.VM_FLAG_ASYNC)
        a1.record()
        torch.cuda.synchronize()
        ms3 = a0.elapsed_time(a1) / 10
        res = {"workload": f"c3: {r3}x{d3} {dt3} store on ONE GPU, {nq3}-query batch, top-{k3}",
               "value": nq3 / (ms3 * 1e-3), "unit": UNIT, "ms_per_step": ms3,
               "hbm_frac": (r3 * d3 * 2 + r3 * 4) / (ms3 * 1e-3) / 1e9 / _peaks()[0],
               "algorithmic_bytes": r3 * d3 * 2 + r3 * 4, "traffic": _ncu_traffic(dt3, r3)}
        s3.close()
        del s3
        torch.cuda.empty_cache()
        return res
    except Exception as e:  # pragma: no cover - e.g. not enough free HBM
        return {"error": repr(e)}


# ---------------------------------------------------------------------------------------------
# all-pairs dedup (C4)
# ---------------------------------------------------------------------------------------------
def bench_dedup(ctx: Ctx, args, steps: int, warmup: int, rows_override=None, dump_dir=None):
    """Config C4: all-pairs dedup, 1M x 768 bf16 vs itself, threshold 0.9 (planted near-duplicates), on the run's N
    GPUs.  N > 1 goes through vm_pairs_above_sharded: tile grid dealt cyclically, ncclAllGather of counts and hit
    lists, every rank ends with the complete list (inside the timed region); the e2e leg additionally starts from
    rows in rank 0's pinned host memory (H2D + ONE ncclBroadcast) and ends with the pairs on the host.
    dump_dir: rank 0 writes the pair list of the last timed step there."""
    import ctypes as C
    import numpy as np
    import torch
    import vidmem_b200 as vm
    from vidmem_b200 import dedup
    from vidmem_b200.store import EmbeddingStore
    rows, dim, dt, thr, seed, dup = C4
    if rows_override:
        rows = rows_override
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    st = EmbeddingStore(dim, rows, dt, device=ctx.local_rank)
    st.synth_fill(seed, rows, dup_period=dup)               # every rank synthesises the same operand for the resident leg
    torch.cuda.synchronize()
    x = st.rows[:rows]
    cap = 1 << 22
    lib = vm._lib.load()
    oi = torch.empty((cap,), dtype=torch.int64, device=dev); oj = torch.empty_like(oi)
    os_ = torch.empty((cap,), dtype=torch.float32, device=dev); cnt = torch.zeros((1,), dtype=torch.int64, device=dev)

    def step(xt=x, root=-1):
        sp = torch.cuda.current_stream(dev).cuda_stream
        if world == 1:
            vm._lib.check(lib.vm_pairs_above(ctx.local_rank, xt.data_ptr(), vm.VM_BF16, rows, dim, C.c_float(thr), cap, oi.data_ptr(),
                                             oj.data_ptr(), os_.data_ptr(), cnt.data_ptr(), 0, 1, 0, sp))
        else:
            vm._lib.check(lib.vm_pairs_above_sharded(ctx.comm.handle, xt.data_ptr(), vm.VM_BF16, rows, dim, C.c_float(thr), cap,
                                                     oi.data_ptr(), oj.data_ptr(), os_.data_ptr(), cnt.data_ptr(), root, 0, sp))

    def pair_hash():
        m = int(cnt.item())
        h = ((oi[:m] * 1_000_003 + oj[:m]) % 2_147_483_629).sum() if m else torch.zeros((), dtype=torch.int64, device=dev)
        return m, int(h.item())

    warm = max(1, min(warmup, 1))
    for _ in range(warm):
        step()
    ctx.barrier()
    sampler = ClockSampler(ctx.local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    ctx.barrier()
    ms = e0.elapsed_time(e1) / steps
    hits, hsum = pair_hash()
    if dump_dir and rank == 0:
        m = min(hits, cap)
        pi, pj, ps = oi[:m].cpu().numpy(), oj[:m].cpu().numpy(), os_[:m].cpu().numpy()
        order = np.lexsort((pj, pi))                        # (i, j) order, as dedup.pairs_above returns the set
        dump_outputs(dump_dir, {"pairs_i": pi[order], "pairs_j": pj[order], "pairs_score": ps[order]})
    # e2e: rank 0's rows come from pinned host memory every step, pairs go back to the host
    xh = None
    if rank == 0:
        xh = torch.empty((rows, dim), dtype=torch.bfloat16).pin_memory()
        xh.copy_(x[:, :dim].cpu())
    xd = torch.zeros_like(x)
    ctx.barrier()
    e2e_steps = max(1, min(steps, 2))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        if rank == 0:
            xd[:, :dim].copy_(xh, non_blocking=True)
        step(xd, root=0 if world > 1 else -1)
        m = int(cnt.item())
        pi, pj, ps = oi[:m].cpu(), oj[:m].cpu(), os_[:m].cpu()
    ctx.barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    e2e_hits, e2e_hsum = pair_hash()
    clocks = sampler.stop() if rank == 0 else None
    ms, e2e_ms = ctx.max_over_ranks([ms, e2e_ms])

    # ---- parity, in this run --------------------------------------------------------------------
    # (a) N > 1: the sharded pair multiset (count + checksum of i*P+j) == rank 0's own single-GPU pass over the same rows;
    #     the e2e leg (H2D + broadcast) reproduces it
    single_hits = single_hsum = None
    if world > 1:
        if rank == 0:
            vm._lib.check(lib.vm_pairs_above(ctx.local_rank, x.data_ptr(), vm.VM_BF16, rows, dim, C.c_float(thr), cap, oi.data_ptr(),
                                             oj.data_ptr(), os_.data_ptr(), cnt.data_ptr(), 0, 1, 0, torch.cuda.current_stream(dev).cuda_stream))
            single_hits, single_hsum = pair_hash()
        ctx.barrier()
    ok = (hits, hsum) == (e2e_hits, e2e_hsum) and (world == 1 or rank != 0 or (hits, hsum) == (single_hits, single_hsum))
    # (b) rank 0: exact pair-SET equality against the CPU oracle on the first `ns` rows (also the cpu_baseline sample)
    sample = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import oracle
        _use_all_host_cores()
        ns = min(rows, 12288)
        E = x[:ns, :dim].float().cpu().numpy()
        t0 = time.perf_counter()
        ri, rj, _rs = oracle.pairs_above(E, thr)
        dt_s = time.perf_counter() - t0
        gi, gj, _gs = dedup.pairs_above(x[:ns].contiguous(), thr, cap=1 << 20)
        same = len(gi) == len(ri) and np.array_equal(gi, ri) and np.array_equal(gj, rj)
        ok = ok and bool(same)
        sample = {"rows": int(ns), "oracle_pairs": int(len(ri)), "gpu_pairs": int(len(gi)), "set_equal": bool(same),
                  "cpu_pairs_per_s": (ns * (ns - 1) / 2) / dt_s}
    # (c) rank 0, at the FULL size: the emitted list against the generator's definition -- every emitted pair really
    #     exceeds the threshold (binary64 cosine of the regenerated rows), and every planted near-duplicate whose exact
    #     cosine to its parent is clear of the threshold is in the list
    planted_check = None
    if rank == 0 and not args.no_cpu_baseline and hits <= cap:
        from oracle import synth
        m = int(cnt.item())
        pi_, pj_ = oi[:m].cpu().numpy(), oj[:m].cpu().numpy()
        A = synth.synth_rows_at(seed, pi_.astype(np.uint64), dim, dup).astype(np.float64)
        B = synth.synth_rows_at(seed, pj_.astype(np.uint64), dim, dup).astype(np.float64)
        ex = (A * B).sum(1) / np.sqrt((A * A).sum(1) * (B * B).sum(1)) if m else np.zeros(0)
        all_above = bool((ex > thr).all() and (pi_ < pj_).all())
        ids = np.arange(1, rows, dtype=np.uint64)
        with np.errstate(over="ignore"):
            hk = synth.splitmix64(np.array([np.uint64(seed) ^ np.uint64(0xD6E8FEB86659FD93)], dtype=np.uint64))[0]
            hr = synth.splitmix64(hk + ids)
            is_planted = hr % np.uint64(dup) == 0
            planted = ids[is_planted]
            parent = synth.splitmix64(hr[is_planted]) % planted
        P = synth.synth_rows_at(seed, planted, dim, dup).astype(np.float64)
        Pa = synth.synth_rows_at(seed, parent, dim, dup).astype(np.float64)
        cs = (P * Pa).sum(1) / np.sqrt((P * P).sum(1) * (Pa * Pa).sum(1))
        found = set(zip(pi_.tolist(), pj_.tolist()))
        expect = {(int(min(a, b)), int(max(a, b))) for a, b, c in zip(planted, parent, cs) if c > thr + 1e-4}
        planted_check = {"rows": int(rows), "emitted_pairs_all_above_threshold_in_binary64": all_above,
                         "planted_pairs_clear_of_threshold": len(expect), "of_which_found": len(expect & found)}
        ok = ok and all_above and expect <= found
    ok = ctx.all_true(bool(ok))

    rec = None
    if rank == 0:
        pairs = rows * (rows - 1) / 2
        peak, src = _tensor_peak()
        tf = pairs * 2 * dim / (ms * 1e-3) / 1e12 / world      # per GPU
        full = _ncu_pairs_full_size(rows) if world == 1 else None   # the capture is of the single-GPU launch
        rec = {"metric": "dedup_unique_pairs_per_sec", "value": pairs / (ms * 1e-3), "unit": "pairs/s", "n_gpus": world,
               "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
               "scaling": "strong", "dtype": "bf16", "data": "synthetic",
               "config": {"workload": f"c4: all-pairs dedup {rows}x{dim} bf16 vs itself, threshold {thr} (strict), "
                                      f"1/{dup} rows planted near-duplicates, upper triangle dealt over {world} GPU(s)"
                                      + (", ncclAllGather of counts + hit lists inside the timed region" if world > 1 else ""),
                          "hits": hits, "l2_policy": "operand %.0f MB > 126 MB L2" % (rows * dim * 2 / 1e6)},
               "e2e": {"value": pairs / (e2e_ms * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": rows * dim * 2,
                       "d2h_bytes_per_step": hits * 20 + 8, "ms_per_step": e2e_ms,
                       "path": "pinned host rows -> H2D" + (" -> ncclBroadcast" if world > 1 else "") + " -> kernel -> pairs D2H"},
               "gpu_launches": 3 * steps + (1 * steps if world > 1 else 0),
               "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                            "traffic": full["traffic"] if full else None, "kernel": "pairs_tc2_kernel", "kernel_ms": ms, "peak_source": src,
                            "flops_counted": "2*D per unordered pair (upper triangle only), per GPU",
                            "ncu_tensor_pipe_active_pct": _ncu_pairs_pipe(), "ncu_at_this_size": full,
                            "frac_of_nominal_2250": tf / 2250.0},
               "parity": {"ok": bool(ok), "checked": "full-size list vs the generator (every emitted pair above the threshold in binary64, every planted pair found); pair multiset (count + checksum) resident == e2e"
                                                     + (" == single-GPU pass" if world > 1 else "") + "; exact pair-set equality vs CPU oracle on a row sample",
                          "pairs": hits, "checksum": hsum, "single_gpu_pairs": single_hits, "oracle_sample": sample,
                          "full_size_structure": planted_check},
               "clocks": clocks}
        if sample:
            rec["cpu_baseline"] = {"value": sample["cpu_pairs_per_s"], "unit": "pairs/s", "cores": os.cpu_count() or 1, "kind": "port",
                                   "sample": f"{sample['rows']} x {dim} rows all-pairs (pairs/s is size-independent for the O(N^2 D) loop)"}
    st.close()
    del st, x, xd, oi, oj, os_
    torch.cuda.empty_cache()
    return rec


# ---------------------------------------------------------------------------------------------
# streaming (C5)
# ---------------------------------------------------------------------------------------------
def bench_streaming(ctx: Ctx, args, rounds: int, dtype=None, rows_override=None, dump_dir=None):
    """Config C5: streaming mode -- 4096-row inserts interleaved with single-query top-10 lookups over a
    10M x 384 store; p50/p99 latencies (host wall clock around synchronous host-buffer calls).
    N > 1: the store is row-sharded (10M/N rows per rank before the inserts), each 4096-row insert goes to ONE rank
    (round-robin == least-full), every query is a collective vm_topk_sharded call (local scan, ncclAllGather, merge).
    dump_dir: rank 0 writes the lists of the last round's queries there."""
    import numpy as np
    import torch
    import vidmem_b200 as vm
    from vidmem_b200.store import EmbeddingStore
    rows_total, dim, dt, nq, k, sseed, qseed = CONFIGS["c5"]
    if rows_override:
        rows_total = rows_override
    dt = dtype or dt
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    per_round_q = 8
    ins = 4096
    n0 = rows_total * (rank + 1) // world - rows_total * rank // world
    row_base = rank * (1 << 32)                       # global row = rank stride + local row (unique, order by rank then age)
    # growable store: exactly the resident rows are backed at the start, so the timed inserts include the store's
    # growth (new physical HBM mapped behind the resident rows; nothing is copied, addresses stay put)
    st = EmbeddingStore(dim, n0, dt, device=ctx.local_rank, max_capacity=2 * n0 + max(rounds, 64) * ins)
    cap0, base0, bytes0 = st.capacity, st.rows.data_ptr(), st.resident_bytes()
    st.synth_fill(sseed, n0, row0=rows_total * rank // world)
    st.set_size(n0)
    torch.cuda.synchronize()
    qpin = make_queries(st, n0, rounds * per_round_q, dim, qseed, dev, world).pin_memory().numpy()
    g = torch.Generator(device="cpu").manual_seed(sseed + 1)
    new_rows = (torch.randint(-127, 128, (rounds * ins, dim), generator=g).float() / 128.0).pin_memory()
    for w in range(3):
        st.topk(qpin[w:w + 1], k, comm=ctx.comm, row_offset=row_base)
    # one untimed insert on every rank: the first append of a process pays one-time costs that are not the store's (upload
    # staging buffer, lazy loading of the conversion kernels, the driver reclaiming memory the previous record released)
    st.append(new_rows[:ins])
    n_warm = ins
    ctx.barrier()
    sampler = ClockSampler(ctx.local_rank, period_s=0.05)
    if rank == 0:
        sampler.start()
    q_lat, i_lat, last_round = [], [], []
    t_all = time.perf_counter()
    for r in range(rounds):
        if r % world == rank:
            t0 = time.perf_counter()
            st.append(new_rows[r * ins:(r + 1) * ins])          # host -> device, convert, norms; synchronous
            i_lat.append((time.perf_counter() - t0) * 1e3)
        for qi in range(per_round_q):
            t0 = time.perf_counter()
            res = st.topk(qpin[r * per_round_q + qi:r * per_round_q + qi + 1], k, comm=ctx.comm, row_offset=row_base)
            q_lat.append((time.perf_counter() - t0) * 1e3)
            if r == rounds - 1:
                last_round.append(res)
    wall = time.perf_counter() - t_all
    ctx.barrier()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {name: np.concatenate([res[f] for res in last_round])
                                for f, name in enumerate(("topk_idx", "topk_score", "topk_count"))})
    clocks = sampler.stop() if rank == 0 else None
    # the planted row of the last insert must be its own best match (every rank sees the same answer)
    probe = new_rows[(rounds - 1) * ins + 17:(rounds - 1) * ins + 18].numpy()
    pi, ps, pc = st.topk(probe, k, comm=ctx.comm, row_offset=row_base)
    owner = (rounds - 1) % world
    n_owner_before = (rows_total * (owner + 1) // world - rows_total * owner // world) + n_warm + ((rounds - 1) // world) * ins
    ok = int(pc[0]) == k and abs(float(ps[0, 0]) - 1.0) < 1e-12 and int(pi[0, 0]) == owner * (1 << 32) + n_owner_before + 17
    ok = ctx.all_true(bool(ok))
    scan_ms = []
    for qi in range(5):
        st.topk(qpin[qi:qi + 1], k, flags=vm.VM_FLAG_TIMING)
        scan_ms.append(st.last_scan_ms())
    es = 4 if dt == "f32" else 2
    n_now = len(st)
    q50, q99, scan = ctx.max_over_ranks([float(np.percentile(q_lat, 50)), float(np.percentile(q_lat, 99)), sum(scan_ms) / len(scan_ms)])
    ins_all = None
    if world > 1:
        import torch.distributed as dist
        packs = [None] * world
        dist.all_gather_object(packs, i_lat)
        ins_all = [v for p in packs for v in p]
    else:
        ins_all = i_lat
    rec = None
    if rank == 0:
        peak, src = _peaks()
        alg = n_now * dim * es + n_now * 4
        rec = {"metric": "streaming_queries_per_sec_top10_384d", "value": len(q_lat) / (sum(q_lat) * 1e-3), "unit": "queries/s",
               "n_gpus": world, "steps": rounds, "warmup": 3, "ms_per_step": wall * 1e3 / rounds, "higher_is_better": True,
               "scaling": "strong", "dtype": "tf32" if dt == "f32" else "bf16", "data": "synthetic",
               "config": {"workload": f"c5: streaming, {rows_total}x{dim} {dt} store" + (f" row-sharded over {world} GPUs" if world > 1 else "")
                                      + f", {ins}-row inserts interleaved with {per_round_q} single-query top-{k} lookups per insert, "
                                        "host buffers, synchronous calls",
                          "scan_kernel": {0: "exact_fp64", 1: "simt", 2: "tcgen05"}[int(st.last_stats.scan_kernel)],
                          "l2_policy": "inputs larger than L2 (%.0f MB per GPU)" % (n_now * dim * es / 1e6)},
               "latency_ms": {"query_p50": q50, "query_p99": q99, "insert_p50": float(np.percentile(ins_all, 50)),
                              "insert_p99": float(np.percentile(ins_all, 99)), "insert_max": float(max(ins_all)),
                              "inserts": len(ins_all), "queries": len(q_lat)},
               "growth": {"store": "growable (virtual range reserved, physical HBM mapped on demand)", "capacity_rows_before": cap0,
                          "capacity_rows_after": st.capacity, "resident_mb_before": bytes0 / 1e6, "resident_mb_after": st.resident_bytes() / 1e6,
                          "rows_moved": 0, "base_address_unchanged": bool(st.rows.data_ptr() == base0),
                          "note": "rank 0's shard; growth steps (256 MB of HBM mapped behind the resident rows) fall inside the timed "
                                  "inserts; one untimed warm-up insert per rank precedes them"},
               "e2e": {"value": len(q_lat) / (sum(q_lat) * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": ins * dim * 4 + per_round_q * dim * 4,
                       "d2h_bytes_per_step": per_round_q * (k * 16 + 8)},
               "gpu_launches": int(st.last_stats.scan_launches) * len(q_lat) + 2 * len(i_lat),
               "roofline": {"bound": "hbm", "achieved": alg / (scan * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": alg / (scan * 1e-3) / 1e9 / peak, "traffic": _ncu_traffic(dt, n0), "kernel": "scan_tc_kernel", "kernel_ms": scan,
                            "traffic_note": "ncu pass at the store's starting size (%d rows); algorithmic_bytes is the size after the inserts" % n0,
                            "algorithmic_bytes": alg, "peak_source": src},
               "parity": {"ok": bool(ok), "checked": "a row of the last insert is its own exact top-1 (score 1.0, expected global row) on every rank"},
               "clocks": clocks}
    st.close()
    del st
    torch.cuda.empty_cache()
    return rec


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    ctx = Ctx(args)
    rank, world = ctx.rank, ctx.world
    cfg = args.config or ("c2" if world == 1 else "c3")
    failed = []

    def note(name, rec):
        if rec is not None and rec.get("parity") and rec["parity"].get("ok") is False:
            failed.append(name)
        return rec

    if cfg == "c4":
        line = note("dedup", bench_dedup(ctx, args, args.steps, args.warmup, args.rows, dump_dir=args.dump_outputs))
    elif cfg == "c5":
        line = note("streaming", bench_streaming(ctx, args, args.steps, args.c5_dtype, args.rows, dump_dir=args.dump_outputs))
    else:
        line = note("topk", bench_topk(ctx, args, cfg, args.steps, args.warmup, variant=args.variant, rows_override=args.rows,
                                       store_dtype=args.store_dtype, dump_dir=args.dump_outputs))
        full = cfg in ("c2", "c3") and not args.rows and not args.only_main
        if rank == 0 and not args.no_cpu_baseline:
            cores = _use_all_host_cores()                    # torchrun pins OMP_NUM_THREADS to 1 in every worker
            qps, ms, desc = cpu_reference_leg(cfg, 1, 1, args.cpu_sample_rows or 100000)
            line["cpu_baseline"] = {"value": qps, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc}
            try:
                line["cpu_baseline"]["sklearn_blas_value"] = cpu_blas_leg(cfg, args.cpu_sample_rows or 100000)
            except Exception:  # pragma: no cover
                line["cpu_baseline"]["sklearn_blas_value"] = None
        if full:
            clustered = note("clustered", bench_topk(ctx, args, cfg, min(args.steps, 20), 3, variant="clustered", with_e2e=False,
                                                     rows_override=None if world > 1 else None))
            # tight clusters: every query's top-k lies inside ONE cluster of near-identical rows, more of them within the scan's
            # error band than the candidate list holds -> every query is settled from the band (certification.band_settled)
            tight = note("clustered_tight", bench_topk(ctx, args, cfg, min(args.steps, 20), 3, variant="clustered", with_e2e=False,
                                                       cluster_rho=0.05))
            b64 = None
            if world == 1 and cfg == "c2":
                b64 = {sd: note("binary64_" + sd, bench_topk(ctx, args, cfg, min(args.steps, 20), 3, with_e2e=True, store_dtype=sd))
                       for sd in ("f64", "f64+bf16")}
            # sub-records: all-pairs steps of ~0.5 s each capped at 3, streaming rounds kept within 8..64
            dd = note("dedup", bench_dedup(ctx, args, min(args.steps, 3), args.warmup))
            stream = note("streaming", bench_streaming(ctx, args, max(8, min(args.steps, 64))))
            stream_bf16 = note("streaming_bf16", bench_streaming(ctx, args, max(8, min(args.steps, 64)), "bf16"))
            if rank == 0:
                line["clustered"] = {key: clustered[key] for key in ("value", "unit", "ms_per_step", "config", "roofline", "certification", "parity", "clocks")}
                line["clustered"]["vs_iid"] = clustered["value"] / line["value"]
                line["clustered_tight"] = {key: tight[key] for key in ("value", "unit", "ms_per_step", "config", "roofline", "certification", "parity", "clocks")}
                line["clustered_tight"]["vs_iid"] = tight["value"] / line["value"]
                if b64:
                    line["binary64_store"] = {sd: {key: r[key] for key in ("value", "unit", "ms_per_step", "config", "roofline", "certification", "parity", "e2e")}
                                              for sd, r in b64.items()}
                line["dedup"] = dd
                line["streaming"] = stream
                line["streaming_bf16"] = {key: stream_bf16[key] for key in ("value", "unit", "ms_per_step", "config", "latency_ms", "growth", "roofline", "parity")}
            if world == 1 and cfg == "c2":
                # config C1: the reference's OWN size (LIMIT 5000 store, 30 benchmark queries) -- latency-bound, L2 flushed per step
                c1 = note("reference_size", bench_topk(ctx, args, "c1", min(args.steps, 100), 3))
                if rank == 0:
                    line["reference_size"] = {key: c1[key] for key in ("value", "unit", "ms_per_step", "steps", "config", "roofline", "certification",
                                                                       "parity", "e2e", "clocks")}
                    if not args.no_cpu_baseline:
                        qps1, ms1, desc1 = cpu_reference_leg("c1", 3, 1, CONFIGS["c1"][0])
                        line["reference_size"]["cpu_baseline"] = {"value": qps1, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                                                                  "sample": desc1, "ms_per_step": ms1,
                                                                  "python_loop": cpu_interpreter_leg("c1", 3)}
            if world == 1 and cfg == "c2" and not args.no_scaling_baseline:
                line["scaling_baseline"] = scaling_baseline(ctx)
    if rank == 0:
        line["vs_baseline"] = None
        if failed:
            line["parity_failed"] = failed
        print(json.dumps(line), flush=True)
    ctx.close()
    if failed:
        sys.stderr.write("bench.py: PARITY FAILED in " + ", ".join(failed) + "\n")
        sys.exit(3)


def torchrun_argv(gpus: int, argv, port: int):
    """The launch line of the bench contract for N > 1 (one rank per GPU, 127.0.0.1 rendezvous)."""
    return [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={gpus}", "--master-addr", "127.0.0.1",
            "--master-port", str(port), os.path.abspath(__file__), *argv]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps of the main record (c5: insert + query rounds; c4: all-pairs steps of ~0.5 s each at the default "
                         "1M rows, so pass a small --steps with --config c4)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS) + ["c4"])
    ap.add_argument("--variant", default="iid", choices=["iid", "clustered"], help="store contents of the main top-k measurement")
    ap.add_argument("--cluster-size", type=int, default=64, help="clustered variant: near-duplicates per centre")
    ap.add_argument("--cluster-rho", type=float, default=0.2, help="clustered variant: noise norm relative to the centre")
    ap.add_argument("--rows", type=int, default=None, help="override the total row count (debug)")
    ap.add_argument("--flags", type=int, default=0, help="extra VM_FLAG_* bits (debug: 4 = force SIMT, 8 = force tcgen05)")
    ap.add_argument("--cpu-sample-rows", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip every CPU leg (oracle timing and oracle parity)")
    ap.add_argument("--only-main", action="store_true", help="skip the clustered / dedup / streaming sub-records")
    ap.add_argument("--peer-exchange", action="store_true",
                    help="multi-GPU: replace ncclAllGather + merge by the peer-memory pull-merge kernel (symmetric memory)")
    ap.add_argument("--no-scaling-baseline", action="store_true", help="skip the extra C3-on-one-GPU measurement of the N=1 run")
    ap.add_argument("--c5-dtype", default=None, choices=["f32", "bf16"])
    ap.add_argument("--store-dtype", default=None, choices=["f32", "bf16", "f64", "f64+bf16"],
                    help="store dtype override for the top-k configs (f64 / f64+bf16: binary64 store, see DESIGN.md 2)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the main record's timed path returned in its last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.gpus > 1 and args.impl == "ours" and "WORLD_SIZE" not in os.environ:
        # started as plain `python bench.py --gpus N`: re-launch under torchrun, one rank per GPU
        import socket
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        os.execv(sys.executable, torchrun_argv(args.gpus, sys.argv[1:], port))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
