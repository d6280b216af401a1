#!/usr/bin/env python
"""bench.py -- headline metric of the exact-scan hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (mmr_search: scan + top-k) over the whole index for one batch of B
queries.  Workload = BASELINE.json's metric config: exact top-10 over a synthetic 10M x 512 bf16 CLIP-shaped
index (configs[2]'s table; it fits one B200, so N=1 scans all of it; N>1 row-range-shards the SAME table, i.e.
strong scaling, with an NCCL all-gather of the per-shard top-k and a final merge kernel).

Prints ONE JSON line (see the keys below).  `value` = queries/s with inputs resident in HBM (CUDA events, max
over ranks); `e2e` = the same through the host-buffer C-ABI call B200Store.search_* makes (H2D + scan + D2H +
sync per step); `roofline` = algorithmic bytes (rows*dim*2 per launch) / mean launch time vs the measured HBM
peak; `cpu_baseline` = the oracle's numpy flat search on this box's host cores on a bounded sample.
`--impl reference` times that CPU path alone (the reference's scan runs inside lancedb, which is not
installable here: the restated flat search in oracle/ stands in, labelled kind="port").
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# The CPU arm must use every host core it is allowed to: torchrun exports OMP_NUM_THREADS=1 to its children, which
# would silently make the BLAS scan single-threaded.  The BLAS pool is sized when numpy is first imported, so the
# variables are overridden HERE, before that import (and re-checked with threadpoolctl in run_reference).
if "reference" in sys.argv:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(host_cores())

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "queries/sec, exact top-10 over 10Mx512 bf16 (flat cosine scan + top-k)"
BLOCK_ROWS = 250_000      # synthetic table is generated in blocks seeded by (SEED, block id)
SEED = 0x5EED
QSEED = 0xC0FFEE


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f16", "f32"])
    ap.add_argument("--cpu-sample-rows", type=int, default=1_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-store", action="store_true", help="N=1: build the table on the device instead of loading it "
                    "through B200Store.load_arrow (e2e is then the bare host-buffer C call)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "fused", "nccl"],
                    help="N>1: fused = peer-memory stores from the scan kernel + wait/merge kernel; nccl = all-gather + merge")
    ap.add_argument("--sweep", default="8,128,1024", help="extra batch sizes reported under 'sweep' (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy, so two "
                    "builds can be compared output for output (same arguments = same inputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the B200 path's results (the CPU arm may scan a sample of the rows)")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured"
    return 6650.0, 1590.0, "fallback"


def sustained_tensor_peak():
    """cuBLAS bf16 back to back for seconds (power-capped clocks): the denominator for a tensor-bound kernel timed inside a
    long loop (the burst figure is what one isolated launch can reach).  None when the driver file is absent."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            v = json.load(fh).get("bf16_tflops_sustained")
        return float(v) if v else None
    except Exception:
        return None


def load_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return {}


# --------------------------------------------------------------------------------------------- synthetic data
def host_block(block_id: int, n: int, dim: int, out=None) -> np.ndarray:
    """The first n rows of block `block_id` of the synthetic table: normalised N(0,1)^dim in fp32, seeded by
    (SEED, block id).  The generator fills rows in order, so a shorter block is a prefix of a longer one."""
    blk = np.empty((n, dim), dtype=np.float32) if out is None else out
    rng = np.random.default_rng([SEED, block_id])
    rng.standard_normal(out=blk, dtype=np.float32)
    blk /= np.sqrt(np.einsum("ij,ij->i", blk, blk))[:, None]
    return blk


def table_blocks(lo: int, hi: int, dim: int, threads: int):
    """Rows [lo, hi) of the synthetic table as (first row, fp32 rows) pairs, equal to host_table(n)[lo:hi] for every
    n >= hi.  Blocks are generated `threads` at a time, so at most that many are held in host memory."""
    from concurrent.futures import ThreadPoolExecutor

    threads = max(1, threads)
    b0, b1 = lo // BLOCK_ROWS, (hi + BLOCK_ROWS - 1) // BLOCK_ROWS

    def make(b):
        s = b * BLOCK_ROWS
        cs, ce = max(s, lo), min(s + BLOCK_ROWS, hi)
        return cs, host_block(b, ce - s, dim)[cs - s:]

    with ThreadPoolExecutor(threads) as pool:
        for c in range(b0, b1, threads):
            yield from pool.map(make, range(c, min(c + threads, b1)))


def gen_queries(n: int, dim: int):
    rng = np.random.default_rng(QSEED)
    q = rng.standard_normal((n, dim), dtype=np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return q.astype(np.float32)


def build_shard(pkg, lo: int, hi: int, dim: int, dtype: str, device):
    """Rows [lo, hi) of the synthetic table, the same rows host_table generates, narrowed on the device by the L1
    loader B200Store.load_arrow uses (mmr_load_rows_f32_host_scatter): one table whichever way a run loads it."""
    import torch
    tdt = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}[dtype]
    rows = torch.empty((hi - lo, dim), dtype=tdt, device=device)
    for start, blk in table_blocks(lo, hi, dim, min(host_cores(), 8)):
        pkg.ResidentIndex.load_rows_into(rows, blk, dst_offset=start - lo)
    return pkg.ResidentIndex(rows, row_base=lo)


def planted_rows(n_rows: int, bounds, world: int, k: int):
    """k row ordinals for the in-run parity check: first / last row, both sides of every shard boundary, a few more."""
    cand = [0, n_rows - 1]
    for r in range(1, world):
        cand += [bounds[r] - 1, bounds[r]]
    for extra in range(1, 4 * k):
        cand += [n_rows // 2 + 7919 * extra]
    planted = []
    for c in cand:
        if 0 <= c < n_rows and c not in planted:
            planted.append(c)
        if len(planted) == k:
            break
    return sorted(planted)


def dump_outputs(dirname: str, arrays: dict, limit: int = 64 << 20) -> None:
    """Write each [B, ...] result array as dirname/<name>.npy: floats as float32, integers (row ids) as float64, both
    exact.  Above `limit` bytes in all, every array keeps the same seeded sample of its B queries, whose indices go to
    query_index.npy."""
    os.makedirs(dirname, exist_ok=True)
    out = {name: a.astype(np.float32 if a.dtype.kind == "f" else np.float64) for name, a in arrays.items()}
    n = len(next(iter(out.values())))
    per_query = sum(a.nbytes for a in out.values()) // max(n, 1) + 8
    if per_query * n > limit:
        keep = np.sort(np.random.default_rng(SEED).choice(n, limit // per_query, replace=False))
        out = {name: a[keep] for name, a in out.items()}
        out["query_index"] = keep.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock + throttle reasons of GPU `index` while the timed region runs."""

    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                for bit, name in self.BITS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self._nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=1.0)

    def summary(self):
        if not self.samples:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                a, b = [float(x) for x in out.strip().split(",")]
                return {"sm_mhz": a, "sm_max_mhz": b, "reasons": [], "samples": 0}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------- CPU arm
def host_mem_available_gb() -> float:
    try:
        with open("/proc/meminfo") as fh:
            for line in fh:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


def host_table(n: int, dim: int, threads: int) -> np.ndarray:
    """The CPU arm's fp32 table: n unit-norm rows of the same distribution as the GPU arm's synthetic table
    (normalised N(0,1)^dim; the reference stores fp32, lancedb_store.py:33-44), generated block by block from
    (SEED, block id) in `threads` threads.  Only the distribution matters for timing a flat scan."""
    from concurrent.futures import ThreadPoolExecutor

    out = np.empty((n, dim), dtype=np.float32)

    def fill(b):
        s, e = b * BLOCK_ROWS, min((b + 1) * BLOCK_ROWS, n)
        host_block(b, e - s, dim, out=out[s:e])

    with ThreadPoolExecutor(max(1, threads)) as pool:
        list(pool.map(fill, range((n + BLOCK_ROWS - 1) // BLOCK_ROWS)))
    return out


def blas_threads() -> int:
    try:
        from threadpoolctl import threadpool_info
        return max([int(i.get("num_threads", 1)) for i in threadpool_info()] or [1])
    except Exception:
        return -1


class CpuReference:
    """The reference's CPU flat search (restated in oracle/, kind "port": the real one runs inside lancedb/lance, not
    installable here) on this box's host cores.  One object = one resident fp32 table; `search` is one pass."""

    def __init__(self, rows: int, dim: int):
        self.cores = host_cores()
        # the whole table when host memory allows it (10M x 512 fp32 = 20.5 GB), else a bounded sample scaled up
        need_gb = rows * dim * 4 / 1e9
        self.n = rows if host_mem_available_gb() > need_gb + 8.0 else min(rows, 1_000_000)
        self.scale = rows / self.n
        t0 = time.perf_counter()
        self.table = host_table(self.n, dim, self.cores)
        self.gen_s = time.perf_counter() - t0
        self.mode = None

    def _pass(self, q, k, mode):
        from oracle import flat_search as ofs
        if mode == "blas":      # one multi-threaded sgemv/sgemm over the table + partition
            return ofs.flat_search_batch(self.table, q, k) if q.shape[0] > 1 else ofs.flat_search(self.table, q[0], k)
        return ofs.flat_search_threads(self.table, q, k, self.cores)   # row slices on a thread pool

    def calibrate(self, q, k):
        """Pick the faster of the two threadings once (after one untimed pass each)."""
        best = None
        for mode in ("blas", "slices"):
            self._pass(q, k, mode)
            t0 = time.perf_counter()
            self._pass(q, k, mode)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, mode)
        self.mode = best[1]
        return best

    def search(self, q, k):
        return self._pass(q, k, self.mode)

    def describe(self) -> dict:
        whole = self.n * self.scale == self.n
        return {"cores": self.cores, "kind": "port", "blas_threads": blas_threads(), "threading": self.mode,
                "sample": (f"all {self.n} rows per pass" if self.scale == 1.0 else
                           f"first {self.n} rows per pass, time x{self.scale:g} (host memory too small for the fp32 table)"),
                "note": "numpy/OpenBLAS fp32 restatement of the flat search (oracle/), not LanceDB; fp32 rows as the "
                        "reference stores them"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=host_cores())
    except Exception:
        pass
    cpu = CpuReference(args.rows, args.dim)
    qs = gen_queries((args.warmup + args.steps) * args.batch, args.dim).reshape(-1, args.batch, args.dim)
    cpu.calibrate(qs[0], args.k)
    n_warm = max(1, min(args.warmup, 3))
    for i in range(n_warm):
        cpu.search(qs[i % len(qs)], args.k)
    steps = args.steps
    t0 = time.perf_counter()
    for i in range(steps):
        cpu.search(qs[args.warmup + i], args.k)
    dt = (time.perf_counter() - t0) / steps * cpu.scale
    qps = args.batch / dt
    desc = cpu.describe()
    line = {
        "impl": "reference", "metric": METRIC, "value": qps,
        "unit": "queries/s", "n_gpus": args.gpus, "steps": steps, "warmup": n_warm,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.rows}x{args.dim} {args.dtype} unit-norm rows, top-{args.k}, query batch {args.batch}",
                   "note": "CPU arm: the reference's scan lives in lancedb/lance (not installable here); the restated numpy "
                           "flat search scans the fp32 rows the reference stores",
                   "host_threads": desc["cores"], "blas_threads": desc["blas_threads"], "threading": desc["threading"],
                   "table_gen_s": round(cpu.gen_s, 2)},
        "cpu_baseline": dict(desc, value=qps, unit="queries/s"),
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- B200 arm
def run_b200(args):
    import importlib
    import torch
    import torch.distributed as dist

    pkg = importlib.import_module("multimodal-rag-for-image-text-search_b200")
    lib = pkg._native.lib()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the scan has no CPU fallback); use --impl reference for the CPU arm")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    # All queries of the timed loop are staged in HBM before it starts, so consecutive searches may be pipelined with
    # programmatic dependent launch (opt-in contract of the library, see csrc/mmr_b200.cu).
    if os.environ.get("MMR_PDL") is None:
        pkg._native.set_option("MMR_PDL", "1")
    B, k, D, K, W = args.batch, args.k, args.dim, args.steps, args.warmup
    # row-range shard of the one global table
    bounds = pkg.shard_bounds(args.rows, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    esize = 4 if args.dtype == "f32" else 2
    q_host = gen_queries((K + W) * B, D).reshape(K + W, B, D)
    planted = planted_rows(args.rows, bounds, world, k)
    unit_q0 = q_host[0, 0] / np.linalg.norm(q_host[0, 0])

    # N = 1: the table goes the way a deployment loads it -- fp32 rows in the reference's Arrow schema ->
    # B200Store.load_arrow (columnar host copy, scatter loader fp32 -> resident bf16) -- and every number below is taken
    # on that store's resident index; the CPU arm scans the same host table.  N > 1 (one process per GPU): every rank
    # generates its own row range on its GPU (the host could not hold N copies of the fp32 table).
    store, cpu, load_info = None, None, None
    use_store = world == 1 and not args.no_cpu_baseline and not args.no_store
    if use_store:
        cpu = CpuReference(args.rows, D)
        use_store = cpu.scale == 1.0            # the whole table fits host memory
    if use_store:
        import pyarrow as pa
        cpu.table[planted] = unit_q0              # the parity rows are part of the table itself (host AND device copy)
        n = args.rows
        t0 = time.perf_counter()
        one = lambda v: pa.array([v], pa.string()).take(pa.array(np.zeros(n, np.int32)))
        table = pkg.make_arrow_table(pa.array(np.arange(n)).cast(pa.string()), one("bench"), one("doc"), one("image"),
                                     cpu.table, one("{}"))
        t1 = time.perf_counter()
        store = pkg.B200Store(device=device, dtype=args.dtype)
        store.load_arrow("image_collection", table)
        ix = store._image_table.resident()
        torch.cuda.synchronize(device)
        t2 = time.perf_counter()
        load_info = {"api": "B200Store.load_arrow (reference 6-column schema, embedding column used zero-copy) + first resident()",
                     "arrow_table_s": round(t1 - t0, 2), "load_s": round(t2 - t1, 2),
                     "loader_GBs_fp32_source": store._image_table.last_load_gbs,
                     "rows": n, "host_bytes": n * D * 4}
        ix.set_query_precision("auto")            # the device-timed loops below measure the kernel families by batch size
    else:
        ix = build_shard(pkg, lo, hi, D, args.dtype, device)
    q_dev = torch.from_numpy(q_host).to(device)
    out_s = torch.empty((B, k), dtype=torch.float32, device=device)
    out_r = torch.empty((B, k), dtype=torch.int64, device=device)
    sharded = pkg.ShardedIndex(ix, exchange=args.exchange) if world > 1 else None

    def step(i):
        if world > 1:
            return sharded.search(q_dev[i], k)   # local scan -> one packed all-gather -> K4 merge in place
        return ix.search(q_dev[i], k, out=(out_s, out_r))

    # ---- parity inside the bench run: k exact copies of warm-up query 0 are planted on both sides of every shard
    # boundary (and at the table's first / last row); the search must return exactly those rows, in row order, with
    # equal scores, and -- for N > 1 -- the fused peer-memory exchange must equal the NCCL all-gather path bit for bit.
    if not use_store:   # through the store's loader, so both ways of loading hold the same planted rows
        mine = [c for c in planted if lo <= c < hi]
        if mine:
            pkg.ResidentIndex.load_rows_into(ix.rows, np.tile(unit_q0, (len(mine), 1)), dst_rows=np.array(mine) - lo)
    torch.cuda.synchronize(device)
    pq = q_dev[0, :1].contiguous()
    if world > 1:
        fused_s, fused_r = [t.clone() for t in sharded.search(pq, k)]
        nccl = pkg.ShardedIndex(ix, exchange="nccl")
        nccl_s, nccl_r = nccl.search(pq, k)
        torch.cuda.synchronize(device)
        assert torch.equal(fused_r, nccl_r) and torch.equal(fused_s, nccl_s), \
            f"rank {rank}: {sharded.exchange} exchange and NCCL all-gather + merge disagree"
        par_s, par_r = fused_s, fused_r
        del nccl
    else:
        par_s, par_r = [t.clone() for t in ix.search(pq, k)]
    assert par_r[0].cpu().tolist() == planted, f"rank {rank}: planted rows {planted} came back as {par_r[0].cpu().tolist()}"
    assert bool((par_s[0] == par_s[0, 0]).all()) and float(par_s[0, 0]) > 0.99, "planted copies must tie at cosine ~1"
    parity_checked = True

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for i in range(W):
        res = step(i)
    barrier()
    launches0 = lib.mmr_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        barrier()
        ev0.record()
        for i in range(W, W + K):
            res = step(i)
        ev1.record()
        barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = lib.mmr_launch_count() - launches0
    if world > 1:
        t = torch.tensor([ms_total], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / K
    qps = B / (ms_step * 1e-3)
    last_scores, last_rows = res[0].cpu().numpy(), res[1].cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"scores": last_scores, "rows": last_rows})

    # kernel-only pass (no collective) for the roofline of the dominant kernel: one launch per step
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(device)
    ev2.record()
    for i in range(W, W + K):
        ix.search(q_dev[i], k, out=(out_s, out_r))
    ev3.record()
    torch.cuda.synchronize(device)
    per_pass = 8 if args.dtype == "f32" else 4
    n_launch = (B + per_pass - 1) // per_pass if lib.mmr_last_kernel() == 1 else 1  # K2: the scan kernel dominates its 5 launches
    kernel_ms = ev2.elapsed_time(ev3) / (K * n_launch)
    hbm_peak, tf_peak, peak_kind = measured_peaks()
    tf_sustained = sustained_tensor_peak()
    algo_bytes = (hi - lo) * D * esize

    def roof(b, ms_per_pass, n_launches=1):
        """Roofline entry for one pass of b queries over this GPU's rows in ms_per_pass."""
        gbs = algo_bytes / (ms_per_pass * 1e-3) / 1e9
        tfl = 2.0 * b * (hi - lo) * D / (ms_per_pass * 1e-3) / 1e12
        tensor_bound = tfl / tf_peak > gbs / hbm_peak
        out = {"bound": "tensor" if tensor_bound else "hbm",
               "achieved": tfl if tensor_bound else gbs, "peak": tf_peak if tensor_bound else hbm_peak,
               "unit": "TFLOP/s" if tensor_bound else "GB/s",
               "frac": (tfl / tf_peak) if tensor_bound else (gbs / hbm_peak), "traffic": None,
               "peak_kind": f"of {peak_kind}" + (" (cuBLAS bf16 burst)" if tensor_bound else " (copy)"),
               "hbm_GBs": gbs, "tensor_tflops": tfl, "frac_of_nominal_8TBs": gbs / 8000.0,
               **({"frac_of_sustained_tensor_peak": tfl / tf_sustained, "sustained_tensor_peak": tf_sustained}
                  if tensor_bound and tf_sustained else {}),
               "algorithmic_bytes_per_launch": algo_bytes, "algorithmic_flops_per_launch": 2.0 * b * (hi - lo) * D / n_launches}
        return out

    kern = lib.mmr_last_kernel()
    roofline = roof(B, kernel_ms * n_launch, n_launch)
    roofline["kernel"] = {1: "scan_stream_kernel (K1, bulk-copy streaming dot + warp top-k)",
                          2: "scan_umma_kernel (K2, tcgen05/TMEM contraction + fused top-k)",
                          3: "scan_stream_kernel varlen"}.get(kern)
    roofline["kernel_ms"] = kernel_ms
    # dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu --set full
    # capture of this exact workload (profiles/roofline_traffic.json names the .csv each figure was read from)
    traffic = load_traffic().get(f"k{kern}_{args.dtype}_{hi - lo}x{D}_b{B}_k{k}")
    if traffic:
        roofline["traffic"] = traffic["dram_bytes_per_launch"]
        roofline["traffic_source"] = traffic["source"]

    # ---- end to end: the call a user of the drop-in makes, host buffers in, host results out, every step
    e2e = None
    if world == 1 and store is not None:
        # LanceDBStore's own signature: search_image(user_id, query_vec: list of floats, top_k) -> list of dicts
        ix.set_query_precision("f32")                        # the store's serving policy
        qlists = [[q.tolist() for q in q_host[i]] for i in range(W + K)]
        users = ["bench"] * B

        def request(i):
            if B == 1:
                return [store.search_image("bench", qlists[i][0], k)]
            return store.search_image_batch(users, q_host[i], k)

        for i in range(min(W, 5)):
            request(i)
        t0 = time.perf_counter()
        for i in range(W, W + K):
            hits = request(i)
        dt = (time.perf_counter() - t0) / K
        e2e = {"value": B / dt, "unit": "queries/s", "h2d_bytes_per_step": B * D * 4, "d2h_bytes_per_step": B * k * 12,
               "ms_per_step": dt * 1e3,
               "api": "B200Store.search_image(user_id, list_of_floats, top_k) -> list of {chunk_id, score, meta} dicts, on the "
                      f"{args.rows}-row collection loaded with load_arrow" if B == 1 else "B200Store.search_image_batch",
               "transfers": "B <= 2: the query rides in the kernel parameters and the result lands in a mapped pinned mailbox "
                            "(no cudaMemcpy); bytes counted are what crosses PCIe"}
        got_rows = [int(h["chunk_id"]) for h in hits[0]]
        if B <= 2:   # (larger batches: the store scores in fp32, the device loop above used the 16-bit tensor-core queries)
            assert got_rows == last_rows[0].tolist(), "store path and device path disagree on the last step"
        # the bare C call under it (what the store adds on top is Python: list -> ndarray, dict building, json.loads)
        t0 = time.perf_counter()
        for i in range(W, W + K):
            hs, hr = ix.search_host(q_host[i], k)
        e2e["c_abi_ms_per_step"] = (time.perf_counter() - t0) / K * 1e3
        assert B > 2 or (hr == last_rows).all(), "host-buffer path and device path disagree"
        ix.set_query_precision("auto")
    elif world == 1:
        for i in range(min(W, 5)):
            ix.search_host(q_host[i], k)
        t0 = time.perf_counter()
        for i in range(W, W + K):
            hs, hr = ix.search_host(q_host[i], k)
        dt = (time.perf_counter() - t0) / K
        e2e = {"value": B / dt, "unit": "queries/s", "h2d_bytes_per_step": B * D * 4, "d2h_bytes_per_step": B * k * 12,
               "ms_per_step": dt * 1e3, "api": "mmr_search_host (the call B200Store.search_text/search_image make)"}
        assert (hr == last_rows).all(), "host-buffer path and device path disagree"
    else:
        # one process per GPU: host query in, fused exchange, merged host result out (mmr_search_exchange_host)
        barrier()
        for i in range(min(W, 5)):
            sharded.search_host(q_host[i], k)
        barrier()
        t0 = time.perf_counter()
        for i in range(W, W + K):
            hs, hr = sharded.search_host(q_host[i], k)
        dt = torch.tensor([(time.perf_counter() - t0) / K], device=device)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        assert (hr == last_rows).all(), "host-buffer exchange path and device path disagree"
        e2e = {"value": B / float(dt.item()), "unit": "queries/s", "h2d_bytes_per_step": B * D * 4,
               "d2h_bytes_per_step": B * k * 12, "ms_per_step": float(dt.item()) * 1e3,
               "api": "ShardedIndex.search_host (mmr_search_exchange_host: query in the scan kernel's parameters, fused "
                      "peer-memory exchange, merged result + flag in a mapped pinned mailbox)"}

    # optional sweep over other batch sizes (device-resident timing only)
    sweep = []
    for b2 in [int(x) for x in args.sweep.split(",") if x.strip()]:
        if world > 1:
            break
        qd2 = torch.from_numpy(gen_queries(b2 * 8, D).reshape(8, b2, D)).to(device)
        for i in range(3):
            ix.search(qd2[i], k)
        torch.cuda.synchronize(device)
        reps = max(10, min(K, 100))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps):
            ix.search(qd2[i % 8], k)
        e1.record()
        torch.cuda.synchronize(device)
        ms = e0.elapsed_time(e1) / reps
        r2 = roof(b2, ms)
        sweep.append({"batch": b2, "ms_per_step": ms, "queries_per_s": b2 / (ms * 1e-3), "bound": r2["bound"],
                      "frac": r2["frac"], "hbm_GBs": r2["hbm_GBs"], "tensor_tflops": r2["tensor_tflops"],
                      "kernel": lib.mmr_last_kernel()})

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the same CPU path as `--impl reference` (that arm is THE baseline; this is its in-run copy on a ~12 s budget),
        # on the very table the GPU searched
        if cpu is None:
            cpu = CpuReference(args.rows, D)
        cpu.calibrate(q_host[0], k)
        reps, t0 = 0, time.perf_counter()
        while reps < 3 or (time.perf_counter() - t0 < 12.0 and reps < 50):
            cd, ci = cpu.search(q_host[W + reps % K], k)
            reps += 1
        per_pass = (time.perf_counter() - t0) / reps * cpu.scale
        cpu_baseline = dict(cpu.describe(), value=B / per_pass, unit="queries/s", passes=reps, ms_per_pass=per_pass * 1e3)
        if store is not None:
            # oracle parity at full size, inside the run: the CPU flat search over the same 10M fp32 rows vs the GPU result
            i = W + (reps - 1) % K
            gs, gr = [t.cpu().numpy() for t in ix.search(q_dev[i], k)]
            cd, ci = np.atleast_2d(cd), np.atleast_2d(ci)
            tol = 1e-5 if args.dtype == "f32" else 1e-3
            worst = 0.0
            for b in range(B):
                want = {int(r): 1.0 - float(d) for d, r in zip(cd[b], ci[b])}
                kth = min(want.values())
                for sc, r in zip(gs[b], gr[b]):
                    assert int(r) in want or sc <= kth + tol, f"GPU hit {int(r)} ({sc}) is not in the oracle top-{k}"
                    if int(r) in want:
                        worst = max(worst, abs(want[int(r)] - float(sc)))
                missing = [r for r, sc in want.items() if r not in set(gr[b].tolist()) and sc > kth + tol]
                assert not missing, f"oracle hits {missing} missing from the GPU result"
            assert worst <= tol, f"score error {worst} > {tol}"
            cpu_baseline["oracle_parity_at_full_size"] = {"checked": True, "max_abs_score_err": worst, "tolerance": tol}
        del cpu
    if rank == 0:
        line = {
            "metric": METRIC,
            "value": qps, "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": f"{args.rows}x{D} {args.dtype} unit-norm rows, top-{k}, query batch {B}",
                       "parallelism": f"row-range shards x{world}" + (
                           "" if world == 1 else (", NCCL all-gather + merge kernel" if sharded.exchange == "nccl" else
                                                  ", fused exchange: scan kernel stores results into peers over NVLink + wait/merge kernel")),
                       "l2": "index (>= 1.28 GB per GPU) is larger than L2 (126 MB); no flush needed",
                       "rows_per_gpu": hi - lo,
                       "launch": "back-to-back searches on one stream, programmatic dependent launch "
                                 + ("on" if pkg._native.get_option("MMR_PDL") == 1 else "off")},
            "hbm_GBs_aggregate": args.rows * D * esize / (ms_step * 1e-3) / 1e9,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "loader": load_info, "gpu_launches": int(launches),
            "parity_checked": parity_checked,
            "parity": {"planted_rows": planted, "what": "k copies of a query across every shard boundary returned exactly, "
                       "in row order" + ("; fused exchange == NCCL all-gather + merge, bit for bit" if world > 1 else "")},
            "clocks": clocks.summary(), "sweep": sweep or None,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
