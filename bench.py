#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on its config: queries/sec, 10M-doc Zipfian corpus, 3-term AND,
BM25 top-100 (config C2), at 1/2/4/8 B200.

    python bench.py --gpus N --steps K --warmup W            our CUDA path (torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...  the reference's own CPU Enquire::get_mset
    python bench.py --config C3|C5|C4 ...                    the other BASELINE.json configurations (default C2)
    python bench.py ... --dump-outputs DIR                   also write the last timed step's MSets as DIR/*.npy

A "step" is one pass of the hot path over one batch of BATCH synthetic queries.
  value  — whole-job queries/s with the batch's plan already resident in HBM (device-timed with CUDA
           events on the searcher's stream, barrier + synchronize on both sides, max over ranks).
  e2e    — the same metric through the reference-facing C-ABI call (xgm_search_submit/wait) with HOST
           buffers: host planning, H2D of the plan, kernels, D2H of the MSets all inside the timed region.
  roofline — decode+intersect+score kernel: algorithmic bytes (SURVEY.md §8d) / its CUDA-event time.
  cpu_baseline — the compiled reference (oracle/_ref) on the box's host cores, rank 0, N=1 only.
  parity — N=1: the (docid, weight) dump of the compiled reference on the SAME 10M-doc corpus against the CUDA MSets.
N>1 is strong scaling: the same 10M-doc corpus split into N interleaved docid shards (Xapian's own
scheme, backends/multi.h:37-70), every query runs on every shard with global statistics (exchanged per
batch, inside the e2e region), and the per-GPU top-k are merged after one all-to-all: every rank merges
and returns the MSets of its 1/N of the batch (Matcher::merge_mset semantics).
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NDOCS = int(os.environ.get("XGM_BENCH_DOCS", 10_000_000))
VOCAB = int(os.environ.get("XGM_BENCH_VOCAB", 1_000_000))
SEED = 12345
QSEED = 777
TOPRANKS = 1000
UNIT = "queries/s"

# BASELINE.json's configurations (SURVEY.md section 8d).  C2 is the one `metric` is quoted on and the default;
# the others are run with --config and their lines kept under profiles/.
CONFIGS = {
    "C2": dict(metric="queries/sec, 10M-doc 3-term AND BM25 top-100", op="AND", nterms=3, topk=100, batch=4096,
               workload="C2: 10M docs, V=1M Zipf(1) terms, 3-term OP_AND, BM25, get_mset(0,100)",
               kernel="xgm_and_bm3_kernel (decode driver + bitmap intersect + BM25)", ref_queries=1024, parity=1024),
    "C3": dict(metric="queries/sec, 10M-doc 5-term OR BM25 top-1000", op="OR", nterms=5, topk=1000, batch=512,
               workload="C3: 10M docs, V=1M Zipf(1) terms, 5-term OP_OR, BM25, get_mset(0,1000)",
               kernel="xgm_or_tile_kernel + xgm_or3_kernel<phase 1> (bitmap union count, MaxScore candidates, tree-order BM25)", ref_queries=256, parity=200),
    "C5": dict(metric="queries/sec, 10M-doc 2-term AND + multivalue range filter + sort by value, top-100", op="AND",
               nterms=2, topk=100, batch=4096, values=True,
               workload=("C5: 10M docs, OP_FILTER(2-term OP_AND, Xapiand MultipleValueRange(slot 0, [lo, lo+1e4])), "
                         "Multi_MultiValueKeyMaker(slot 1) then relevance, get_mset(0,100)"),
               kernel="xgm_and_bm3_kernel (decode driver + bitmap intersect + range predicate + BM25)",
               ref_queries=1024, parity=256),
    "C4": dict(metric="queries/sec, 100M-doc (8 shards) 3-term AND BM25 top-100", op="AND", nterms=3, topk=100, batch=4096,
               docs=int(os.environ.get("XGM_BENCH_C4_DOCS", 100_000_000)), shards=8,
               workload="C4: 100M docs in 8 interleaved shards, 3-term OP_AND, BM25, get_mset(0,100), two-phase statistics",
               kernel="xgm_and_bm3_kernel (decode driver + bitmap intersect + BM25)", ref_queries=0, parity=0),
}
BATCH_ENV = os.environ.get("XGM_BENCH_BATCH")
REF_Q_ENV = os.environ.get("XGM_BENCH_REF_QUERIES")


def config(name):
    c = dict(CONFIGS[name])
    c["name"] = name
    c.setdefault("docs", NDOCS)
    c.setdefault("values", False)
    if BATCH_ENV:
        c["batch"] = int(BATCH_ENV)
    if REF_Q_ENV:
        c["ref_queries"] = int(REF_Q_ENV)
    return c


def gen_queries(cfg, step: int, n: int):
    """n queries of the configuration: term ranks drawn uniformly from [0, 1000) without repetition
    (SURVEY.md section 8d); C5 adds a range [lo, lo + 1e4] over slot 0."""
    rng = random.Random(QSEED * 1000003 + step)
    out = []
    for _ in range(n):
        t = rng.sample(range(TOPRANKS), cfg["nterms"])
        lo = rng.randrange(0, 990000) if cfg["name"] == "C5" else None
        out.append((t, lo))
    return out


def term_name(r: int) -> str:
    return f"T{r:06d}"


def xgm_query(cfg, q, stats=None, check_at_least=0):
    from xapiand_b200 import xgm
    terms, lo = q
    kw = dict(first=0, maxitems=cfg["topk"], check_at_least=check_at_least, stats=stats)
    if lo is not None:
        # numeric keys of the synthetic index are order-isomorphic to the serialised bytes the reference compares
        kw.update(filter=xgm.FILTER_MULTI_RANGE, filter_slot=0, range_lo=lo, range_hi=lo + 10000,
                  sort_by=xgm.SORT_VAL_REL, sort_slot=1, sort_reverse=False, sort_missing_key=2 ** 64 - 1)
    return xgm.Query(xgm.OP_AND if cfg["op"] == "AND" else xgm.OP_OR, [term_name(t) for t in terms], **kw)


def ref_query_line(cfg, q, check_at_least=0):
    from oracle import oracle as O
    terms, lo = q
    return O.query_line(cfg["op"], [term_name(t) for t in terms], 0, cfg["topk"], check_at_least,
                        mvr=None if lo is None else (0, lo, lo + 10000, 0), keysort=None if lo is None else (1, 0))


# ---------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------

class ClockSampler:
    """SM clock / throttle-reason samples taken DURING the timed regions.  NVML is polled from a thread every
    few milliseconds (the regions last tens of milliseconds; polling faster contends with the CUDA driver
    and slows the host side of the end-to-end loop), plus one sample taken by the main thread while the
    device-resident region's work is queued; `nvidia-smi -lms` is the fallback."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
               (0x4, "sw_power_cap"), (0x80, "hw_power_brake_slowdown"))

    def __init__(self, gpu_index: int, uuid: str | None = None):
        self.gpu = gpu_index
        self.uuid = uuid
        self.samples = []      # (perf_counter, sm_mhz, reason_bits)
        self.windows = []      # [t0, t1] of the timed regions
        self.max_mhz = None
        self.proc = None
        self.rows = []
        self.handle = None
        self.stop_flag = False
        self.thread = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid)
                except Exception:
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.handle = h
            self.nvml = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.handle = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            time.sleep(0.3)
        except Exception:
            self.proc = None

    def sample_now(self):
        if self.handle is None:
            return
        n = self.nvml
        try:
            mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
            try:
                bits = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                bits = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            self.samples.append((time.perf_counter(), mhz, bits))
        except Exception:
            pass

    def _poll(self):
        while not self.stop_flag:
            self.sample_now()
            time.sleep(0.004)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def begin(self):
        self.windows.append([time.perf_counter(), None])

    def end(self):
        self.windows[-1][1] = time.perf_counter()

    def _inside(self, t):
        return any(w[0] <= t <= (w[1] if w[1] is not None else t) for w in self.windows)

    def stop(self):
        self.stop_flag = True
        if self.handle is None and not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml and nvidia-smi unavailable"]}
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            mx = []
            for t, r in self.rows:
                p = [x.strip() for x in r.split(",")]
                if len(p) < 9:
                    continue
                try:
                    mhz = float(p[1]); mx.append(float(p[2]))
                except ValueError:
                    continue
                bits = 0
                for (bit, _), v in zip(self.REASONS[:4], p[5:9]):
                    if v.lower().startswith("active"):
                        bits |= bit
                self.samples.append((t, mhz, bits))
            self.max_mhz = max(mx) if mx else None
        elif self.thread:
            self.thread.join(timeout=1)
        inside = [s for s in self.samples if self._inside(s[0])]
        # the regions are short; if the poller never fell inside one, use the samples bracketing them
        use = inside or self.samples
        bits = 0
        for s in use:
            bits |= s[2]
        reasons = sorted(name for bit, name in self.REASONS if bits & bit)
        return {"sm_mhz": statistics.median(s[1] for s in use) if use else None, "sm_max_mhz": self.max_mhz,
                "samples": len(use), "samples_in_timed_regions": len(inside), "reasons": reasons,
                "source": "nvml" if self.handle is not None else "nvidia-smi"}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the compiled reference's Enquire::get_mset on host cores
# ---------------------------------------------------------------------------------------------

def ref_db_dir(cfg=None):
    base = os.environ.get("XGM_REF_DB_DIR") or ("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp")
    return os.path.join(base, f"xgm_refdb_mv_{NDOCS}_{VOCAB}_{SEED}")


def ref_cores():
    """Host threads the reference arm may use: the scheduler affinity, capped by the cgroup CPU quota
    (a container can see 128 CPUs and be allowed 16)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = int(q) / int(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    n = aff if quota is None else max(1, min(aff, int(quota)))
    return n, {"affinity": aff, "cgroup_quota": quota}


def build_reference_db():
    """The 10M-doc glass DB of C2 / C3 / C5, written by the reference's own WritableDatabase: value slots the way
    Xapiand stores them (--mvalues), so that one DB serves every configuration."""
    from oracle import oracle as O
    if not O.have_reference():
        raise RuntimeError("oracle/_ref missing: the reference was not built (oracle/build_ref.sh)")
    procs = min(ref_cores()[0], 128)
    return O.ref_build_parallel(ref_db_dir(), NDOCS, VOCAB, seed=SEED, procs=procs, mvalues=True)


def run_reference_queries(cfg, dbs, nqueries: int, steps: int, warmup: int, threads: int, dump=False, step0=0,
                          check_at_least=0):
    """Each step = nqueries queries of the workload over all host threads.  Every thread opens its own
    Xapian::Database + Enquire before the first pass (oracle/ref_runner.cc); the wall clock of a pass covers
    Enquire::set_query + get_mset + reading the MSet."""
    from oracle import oracle as O
    work = os.path.join(ref_db_dir(), f"work_{cfg['name']}_{os.getpid()}")
    lines = [ref_query_line(cfg, q, check_at_least) for q in gen_queries(cfg, step0, nqueries)]
    return O.ref_query(dbs, lines, work, threads=threads, repeat=steps, warmup=max(1, warmup), dump=dump)


def single_thread_baseline(cfg, dbs):
    """SURVEY.md section 8(d) asks for the reference at (i) one thread and (ii) all cores: the one-thread leg, on a
    small bounded sample (a few seconds)."""
    n = int(os.environ.get("XGM_BENCH_REF_QUERIES_1T", 256 if cfg["name"] != "C3" else 48))
    try:
        info, _ = run_reference_queries(cfg, dbs, n, 1, 1, 1)
        return {"value": info["qps"], "unit": UNIT, "cores": 1, "p50_ms": info["p50_ms"], "p99_ms": info["p99_ms"],
                "sample": f"1 pass of {n} queries of the same workload, one thread"}
    except Exception as e:  # reported, never required
        return {"value": None, "unit": UNIT, "cores": 1, "sample": f"unavailable: {e}"}


def ref_queries_per_step(cfg, cores):
    """At least 64 queries per thread and step, so that thread start-up and the slowest query's tail do not
    dominate a step."""
    return max(cfg["ref_queries"], 64 * cores)


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = config(args.config)
    if cfg["name"] == "C4":
        print(json.dumps({"impl": "reference", "unavailable": "C4 (100M docs) reference DB is not built inside bench.py"}))
        return 0
    t0 = time.time()
    binfo = build_reference_db()
    cores, cinfo = ref_cores()
    nq = ref_queries_per_step(cfg, cores) if not REF_Q_ENV else cfg["ref_queries"]
    info, _ = run_reference_queries(cfg, binfo["dbs"], nq, args.steps, args.warmup, cores)
    qps = info["qps"]
    ms_per_step = info["wall_s"] / args.steps * 1e3
    sample = (f"{nq} queries/step of the same workload on the full {NDOCS}-doc glass DB "
              f"(built by {binfo['procs']} parallel WritableDatabase writers + Database::compact), "
              f"{cores} threads each with its own Xapian::Database+Enquire opened before the timed passes")
    line = {"impl": "reference", "metric": cfg["metric"], "value": qps, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "docs": NDOCS, "vocab": VOCAB, "queries_per_step": nq,
                       "topk": cfg["topk"]},
            "cpu_baseline": {"value": qps, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample,
                             "cores_detail": cinfo, "p50_ms": info["p50_ms"], "p99_ms": info["p99_ms"],
                             "single_thread": single_thread_baseline(cfg, binfo["dbs"])},
            "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "setup_s": round(time.time() - t0, 1)}
    print(json.dumps(line))
    return 0


def parity_against_reference(cfg, dbs, searcher, cores):
    """BASELINE.md section 3: the (docid, %.17g weight) dump of the compiled reference on the bench corpus itself
    against the CUDA MSets of the same queries — docids identical in order, weights bit-equal."""
    import struct
    from xapiand_b200 import xgm
    n = cfg["parity"]
    if n == 0:
        return None
    out = {"checked": 0, "mismatches": 0, "bounds_approx": 0, "declined": 0, "against": "compiled reference, full corpus"}
    legs = [0] if cfg["name"] != "C3" else [0, NDOCS]  # C3 also with check_at_least = N (SURVEY.md section 8d)
    for cal in legs:
        qs = gen_queries(cfg, 12345, n)
        _, ref = run_reference_queries(cfg, dbs, n, 1, 0, cores, dump=True, step0=12345, check_at_least=cal)
        res = searcher.search([xgm_query(cfg, q, check_at_least=cal) for q in qs])
        for r, m in zip(ref, res):
            out["checked"] += 1
            if m.status != 0:
                out["declined"] += 1
                continue
            same = list(m.docids) == r.docids and all(struct.pack("<d", a) == struct.pack("<d", b) for a, b in zip(m.weights, r.weights))
            same = same and m.matches_upper_bound == r.ub
            if not (m.flags & 1):
                same = same and (m.matches_lower_bound, m.get_matches_estimated()) == (r.lb, r.est)
            else:
                out["bounds_approx"] += 1
            out["mismatches"] += 0 if same else 1
    return out


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------

class CudaArray:
    """Zero-copy view of a raw device pointer for torch.as_tensor (CUDA array interface v2)."""

    def __init__(self, ptr: int, shape, typestr: str):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2}


DUMP_LIMIT = 64 << 20


def mset_arrays(prefix, n, docids, weights, extra=()):
    """One timed path's MSets as float64 arrays: [nq, stride] docids and weights (entries past a query's n set
    to 0, since no docid is 0) plus per-query columns."""
    import numpy as np
    n = np.asarray(n, np.int64)
    keep = np.arange(docids.shape[1])[None, :] < n[:, None]
    out = {f"{prefix}_n": n.astype(np.float64),
           f"{prefix}_docids": np.where(keep, docids, 0).astype(np.float64),
           f"{prefix}_weights": np.where(keep, weights, 0.0).astype(np.float64)}
    for name, col in extra:
        out[f"{prefix}_{name}"] = np.asarray(col, np.float64)
    return out


def dump_outputs(path, arrays, suffix=""):
    """Write DIR/<name><suffix>.npy.  Rows are queries; above DUMP_LIMIT bytes in all, a fixed seeded sample of the
    rows is written, and query_index.npy says which."""
    import numpy as np
    nq = len(next(iter(arrays.values())))
    row_bytes = sum(a[0].nbytes for a in arrays.values()) + 8
    budget = DUMP_LIMIT - 4096 * (len(arrays) + 1)  # room for the .npy headers
    rows = np.arange(nq)
    if nq * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(nq, budget // row_bytes, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, f"query_index{suffix}.npy"), rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}{suffix}.npy"), a[rows])


def ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from xapiand_b200 import xgm

    cfg = config(args.config)
    BATCH, TOPK = cfg["batch"], cfg["topk"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libxgm has no CPU path")
    if cfg["name"] == "C4" and world != cfg["shards"]:
        raise SystemExit(f"--config C4 is the {cfg['shards']}-shard configuration: launch it with --gpus {cfg['shards']}")
    if BATCH % world:
        raise SystemExit("the batch must divide evenly over the ranks")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    t_setup = time.time()
    host_cpus = ref_cores()[0]
    if world > 1:  # N ranks share the box's CPUs: size the library's planner pool accordingly
        os.environ.setdefault("XGM_HOST_THREADS", str(max(1, min(8, host_cpus // world - 1))))
    threads = max(4, (os.cpu_count() or 8) // max(1, world))
    ix = xgm.Index.synthetic(cfg["docs"], VOCAB, seed=SEED, nshards=world, shard=rank, values=cfg["values"],
                             device=local_rank, host_threads=min(64, threads))
    info = ix.info()
    build_s = time.time() - t_setup
    L = xgm.lib()

    # ---- batches: queries marshalled once; for N > 1 their global statistics are filled in per step ----
    nbatches = max(args.warmup, 3) + args.steps + 2
    raw = [gen_queries(cfg, i, BATCH) for i in range(nbatches)]
    batches = [xgm.QueryBatch([xgm_query(cfg, q) for q in qs]) for qs in raw]
    if world > 1:
        # phase 1 of Xapiand's two-phase scheme (src/database/handler.cc:1532-1538, weightinternal.cc:54-72) per batch:
        # local termfreq of every distinct query term (one C call), ONE all-reduce of (termfreqs, doccount,
        # total_length), then the sums go into the batch's statistics blocks.  All of it is inside the e2e region.
        lookup = ix.term_freq_lookup([term_name(r) for r in range(TOPRANKS)])  # every term a query may draw
        term_idx = [np.array([q[0] for q in qs], np.int64) for qs in raw]
        for b in batches:
            b.attach_global_stats()
        # the sums are host data on both sides (term dictionary in, planner out) and 8 KB per batch.  On the NCCL
        # communicator the exchange queued behind the result exchanges of earlier batches (0.8 ms); a gloo all-reduce
        # between 8 local processes took 2.4 ms.  The ranks of one node exchange through shared memory instead
        # (xapiand_b200/shm_exchange.py, ~20 us); ranks on several nodes (or XGM_BENCH_STATS=gloo) keep the gloo group.
        one_node = int(os.environ.get("LOCAL_WORLD_SIZE", world)) == world
        use_shm = one_node and os.environ.get("XGM_BENCH_STATS", "shm") == "shm"
        stats_pg = None if use_shm else dist.new_group(backend="gloo")
        shm = None
        if use_shm:
            from xapiand_b200.shm_exchange import ShmExchange
            shm_name = f"xgm_p1_{os.environ.get('MASTER_PORT', '0')}_{os.getuid()}"
            if rank == 0:
                shm = ShmExchange(shm_name, 0, world, TOPRANKS + 2, create=True)
            dist.barrier()
            if rank != 0:
                shm = ShmExchange(shm_name, rank, world, TOPRANKS + 2)
            dist.barrier()

        pending_stats = {}
        next_xid = [0]

        def local_stats():
            a = np.empty(TOPRANKS + 2, np.int64)
            a[:TOPRANKS] = lookup()
            a[TOPRANKS] = int(info.doccount)
            a[TOPRANKS + 1] = int(info.total_length)
            return a

        def start_stats(bi: int):
            """Phase 1 of batch bi, first half: local termfreqs (one C call) posted / the all-reduce left in flight."""
            if bi in pending_stats or bi >= nbatches:
                return
            if use_shm:
                xid = next_xid[0]
                next_xid[0] += 1
                shm.post(xid, local_stats())
                pending_stats[bi] = xid
            else:
                buf = torch.from_numpy(local_stats())
                pending_stats[bi] = (buf, dist.all_reduce(buf, group=stats_pg, async_op=True))

        def exchange_stats(bi: int):
            """Second half: wait for the sums and write them into the batch's statistics blocks.  The exchange of
            batch bi + 1 is started before returning, so that it overlaps the planning and matching of batch bi."""
            start_stats(bi)
            if use_shm:
                a = shm.collect(pending_stats.pop(bi))
            else:
                buf, work = pending_stats.pop(bi)
                work.wait()
                a = buf.numpy()
            batches[bi].set_global_stats(int(a[TOPRANKS]), int(a[TOPRANKS + 1]), a[:TOPRANKS][term_idx[bi]].astype(np.uint32))
            start_stats(bi + 1)
    else:
        shm = None

        def exchange_stats(bi: int):
            return None

    NSEARCH = int(os.environ.get("XGM_BENCH_NSEARCH", 3))  # batches in flight in the end-to-end loop (host planning / GPU / result scatter overlap)
    searchers = [xgm.Searcher(ix, max_batch=BATCH, max_topk=TOPK) for _ in range(NSEARCH)]
    streams = [torch.cuda.ExternalStream(s.stream(), device=torch.device("cuda", local_rank)) for s in searchers]
    if world > 1:
        for s in searchers:
            s.results_on_device(True)  # the per-shard MSets are exchanged and merged on the device

    # ---- N > 1: the merge.  Rank r owns queries [r*BATCH/N, (r+1)*BATCH/N): one all-to-all moves every shard's
    # top-k of those queries to r (three regions of the result slab: weights | docids | records), r merges them
    # (Matcher::merge_mset, unshard included) and copies ITS slice of the merged MSets to the host. ----
    QL = BATCH // world
    if world > 1:
        xbuf = []
        for s in searchers:
            base, nbytes, off_d, off_c, stride = s.device_slab()
            assert stride == TOPK
            lw = torch.as_tensor(CudaArray(base, (BATCH * TOPK * 8,), "|u1"), device="cuda")
            ld = torch.as_tensor(CudaArray(base + off_d, (BATCH * TOPK * 4,), "|u1"), device="cuda")
            li = torch.as_tensor(CudaArray(base + off_c, (BATCH * 32,), "|u1"), device="cuda")
            gw, gd, gi = torch.empty_like(lw), torch.empty_like(ld), torch.empty_like(li)
            ow = torch.empty(QL * TOPK, dtype=torch.float64, device="cuda")
            od = torch.empty(QL * TOPK, dtype=torch.int32, device="cuda")
            on = torch.empty(QL, dtype=torch.int32, device="cuda")
            xbuf.append((lw, ld, li, gw, gd, gi, ow, od, on))
        host_out = [(torch.empty(QL * TOPK, dtype=torch.float64).pin_memory(),
                     torch.empty(QL * TOPK, dtype=torch.int32).pin_memory(),
                     torch.empty(QL, dtype=torch.int32).pin_memory()) for _ in searchers]

    def merge_step(si: int, to_host: bool):
        lw, ld, li, gw, gd, gi, ow, od, on = xbuf[si]
        with torch.cuda.stream(streams[si]):
            dist.all_to_all_single(gw, lw)
            dist.all_to_all_single(gd, ld)
            dist.all_to_all_single(gi, li)
            st = L.xgm_merge_topk_device(gw.data_ptr(), gd.data_ptr(), gi.data_ptr(), world, QL, TOPK, TOPK,
                                         ow.data_ptr(), od.data_ptr(), on.data_ptr(), searchers[si].stream())
            if st != 0:
                raise RuntimeError(L.xgm_last_error().decode())
            if to_host:
                hw, hd, hn = host_out[si]
                hw.copy_(ow, non_blocking=True)
                hd.copy_(od, non_blocking=True)
                hn.copy_(on, non_blocking=True)

    # ---- warm-up: W steps through the full API (also makes the plan of batch 0 resident) ----
    W = max(args.warmup, 3)
    for w in range(W):
        for si, srch in enumerate(searchers):  # every searcher (staging buffers, worker thread) is warmed up
            bi = w % nbatches
            exchange_stats(bi)
            srch.submit(batches[bi], background=True)
            if world > 1:
                srch.launched()
                merge_step(si, True)
                srch.wait_device()
            else:
                srch.wait_raw()
    exchange_stats(0)
    if world > 1:  # the device-resident loop alternates between two searchers holding the same resident plan
        searchers[1].submit(batches[0])
        searchers[1].wait_device()
        searchers[0].results_on_device(False)
    searchers[0].submit(batches[0])
    _, _, _, inf0 = searchers[0].wait_raw()
    if world > 1:
        searchers[0].results_on_device(True)
    bad = sum(1 for i in range(BATCH) if inf0[i].status != 0)
    if bad:
        raise SystemExit(f"{bad} queries of the bench batch were not answered on the device")
    approx0 = sum(1 for i in range(BATCH) if inf0[i].flags & 1)
    st0 = searchers[0].last_stats()
    barrier()

    # ---- device-resident timed region: K replays of the resident plan ----
    try:
        uuid = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        uuid = None
    sampler = ClockSampler(local_rank, uuid)
    sampler.start()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    match_ms, topk_ms = [], []
    barrier()
    sampler.begin()
    ev0.record(streams[0])
    for k in range(args.steps):
        # N > 1: the exchange + merge of step k (searcher k%2's stream) overlaps the kernels of step k+1
        # (the index's compute stream), consecutive steps being independent batches
        si = k % 2 if world > 1 else 0
        searchers[si].replay()
        if world > 1:
            merge_step(si, False)
    if world > 1:
        tail = torch.cuda.Event()
        tail.record(streams[1])
        streams[0].wait_event(tail)
    ev1.record(streams[0])
    sampler.sample_now()  # the K replays are queued and running
    barrier()
    sampler.end()
    dev_ms = ev0.elapsed_time(ev1)
    dump = {}
    if args.dump_outputs:  # what the last replay left on the device: the slab (N = 1) / the merged MSets (N > 1)
        if world == 1:
            wp, dp, cp, stride = searchers[0].device_results()
            w = torch.as_tensor(CudaArray(wp, (BATCH, stride), "<f8"), device="cuda").cpu().numpy()
            d = torch.as_tensor(CudaArray(dp, (BATCH, stride), "<i4"), device="cuda").cpu().numpy().view(np.uint32)
            cnt = torch.as_tensor(CudaArray(cp, (BATCH, 8), "<i4"), device="cuda").cpu().numpy().view(np.uint32)
            dump.update(mset_arrays("replay", cnt[:, 0], d, w, [("exact_matches", cnt[:, 1])]))  # XgmDevResult n, exact
        else:
            ow, od, on = xbuf[(args.steps - 1) % 2][6:]
            dump.update(mset_arrays("replay", on.cpu().numpy(), od.cpu().numpy().view(np.uint32).reshape(QL, TOPK),
                                    ow.cpu().numpy().reshape(QL, TOPK)))
    # per-launch time of the dominant kernel: K more replays, reading each launch's own events
    for k in range(args.steps):
        searchers[0].replay()
        ls = searchers[0].last_stats()
        match_ms.append(ls.match_kernel_ms)
        topk_ms.append(ls.topk_kernel_ms)
    xchg_ms = None
    if world > 1:  # the exchange + merge alone, for the "what bounds the step" note
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(streams[0])
        for k in range(args.steps):
            merge_step(0, False)
        e1.record(streams[0])
        torch.cuda.synchronize()
        xchg_ms = e0.elapsed_time(e1) / args.steps
    torch.cuda.synchronize()
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    value = BATCH * args.steps / (dev_ms / 1e3)

    # ---- end-to-end timed region: K steps through submit/wait with host buffers, NSEARCH searchers ----
    barrier()
    sampler.begin()
    t0 = time.perf_counter()
    stats_s = 0.0
    wait = (lambda s: s.wait_device()) if world > 1 else (lambda s: s.wait_raw())
    # Software pipeline over NSEARCH searchers.  Batch k is submitted in iteration k (its searcher's worker thread
    # plans + enqueues it); N > 1: its exchange + merge is enqueued two iterations later, when that worker has long
    # finished, so xgm_search_launched never blocks this thread; its results are collected NSEARCH iterations later.
    LAG = 2 if NSEARCH >= 3 else 1
    def finish(j):  # exchange + merge of batch j (N > 1)
        searchers[j % NSEARCH].launched()
        merge_step(j % NSEARCH, True)
    for k in range(args.steps):
        si = k % NSEARCH
        bi = W + 1 + k
        if world > 1 and k >= LAG:
            finish(k - LAG)
        if k >= NSEARCH:
            wait(searchers[si])  # batch k - NSEARCH: scatter (N = 1) / synchronise (N > 1)
        ts = time.perf_counter()
        exchange_stats(bi)  # N > 1: phase-1 statistics of THIS batch (lookups + all-reduce + fill-in)
        stats_s += time.perf_counter() - ts
        searchers[si].submit(batches[bi], background=True)
    if world > 1:
        for j in range(max(0, args.steps - LAG), args.steps):
            finish(j)
    for j in range(max(0, args.steps - NSEARCH), args.steps):
        last = wait(searchers[j % NSEARCH])
    pending = (args.steps - 1) % NSEARCH
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    sampler.end()
    if args.dump_outputs:  # the last step's MSets as the caller holds them: scattered by xgm_search_wait / merged
        if world == 1:
            l_docids, l_weights, l_keys, l_info = last
            inf = np.ctypeslib.as_array(l_info)[:BATCH]
            cols = ["first", "matches_lower_bound", "matches_estimated", "matches_upper_bound", "exact_matches", "status",
                    "flags", "max_possible", "max_attained", "percent_scale_factor"]
            if cfg["values"]:
                keys = np.where(np.arange(TOPK)[None, :] < inf["n"][:, None].astype(np.int64), l_keys.reshape(BATCH, TOPK), 0)
                cols += [("sort_key_hi", keys >> np.uint64(32)), ("sort_key_lo", keys & np.uint64(0xffffffff))]
            dump.update(mset_arrays("e2e", inf["n"], l_docids.reshape(BATCH, TOPK), l_weights.reshape(BATCH, TOPK),
                                    [c if isinstance(c, tuple) else (c, inf[c]) for c in cols]))
        else:
            hw, hd, hn = host_out[pending]
            dump.update(mset_arrays("e2e", hn.numpy(), hd.numpy().view(np.uint32).reshape(QL, TOPK),
                                    hw.numpy().reshape(QL, TOPK)))
    e2e_s = t1 - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    bs = searchers[pending].last_stats()
    h2d, d2h = int(bs.h2d_bytes), int(bs.d2h_bytes)
    if world > 1:
        d2h += QL * TOPK * 12 + QL * 4
    clocks = sampler.stop()
    e2e_value = BATCH * args.steps / e2e_s

    # ---- p50 latency at batch = 1 through the C-ABI (rank-local) ----
    lat = []
    one = xgm.Searcher(ix, max_batch=1, max_topk=TOPK)
    singles = [xgm.QueryBatch([xgm_query(cfg, q)]) for q in gen_queries(cfg, 999, 200)]
    for b in singles[:20]:
        one.submit(b); one.wait_raw()
    for b in singles:
        a = time.perf_counter()
        one.submit(b)
        one.wait_raw()
        lat.append((time.perf_counter() - a) * 1e3)
    lat.sort()

    # ---- roofline of the dominant kernel ----
    peak, peak_src = measured_peak_gbs()
    alg_bytes = int(st0.algorithmic_bytes)
    kern_ms = statistics.mean(match_ms)
    achieved = alg_bytes / 1e9 / (kern_ms / 1e3)
    launches_per_step = int(st0.kernel_launches) + (4 if world > 1 else 0)

    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", f"r2_{cfg['name'].lower()}_match_kernel.json")
    if os.path.exists(tp) and world == 1:
        try:
            prof = json.load(open(tp))
            # the capture is only a cross-reference while the kernel source is the one it was taken from
            import hashlib
            src = open(os.path.join(ROOT, "xapiand_b200", "csrc", "xgm_kernels.cu"), "rb").read()
            if prof.get("queries_per_launch") == BATCH and prof.get("kernels_sha16") == hashlib.sha256(src).hexdigest()[:16]:
                traffic = prof["dram_bytes_read"] + prof["dram_bytes_write"]
                traffic_src = f"profiles/{os.path.basename(tp)} (ncu dram__bytes_read+write of one launch, same kernel source hash)"
        except Exception:
            pass
    step_parts = {"match_kernel_ms": kern_ms, "topk_kernel_ms": statistics.mean(topk_ms), "host_plan_ms": float(bs.host_plan_ms),
                  "host_scatter_ms": float(bs.host_wait_ms)}
    if world > 1:
        step_parts.update(exchange_merge_ms=xchg_ms, stats_exchange_ms=stats_s / args.steps * 1e3)
    bound = max(step_parts, key=lambda k: step_parts[k] or 0.0)
    line = {"metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if cfg["name"] != "C4" else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "docs": cfg["docs"], "vocab": VOCAB, "queries_per_step": BATCH,
                       "topk": TOPK, "shards": world, "shard_docs": int(info.doccount),
                       "cache": "inputs larger than L2: one step streams %.0f MB of posting columns (L2 = 126 MB)" % (alg_bytes / 1e6),
                       "index_bytes": int(info.bytes_docids + info.bytes_wdfs + info.bytes_headers + info.bytes_doclen),
                       "index_build_s": round(build_s, 1),
                       "value_is": "device-resident replay of one planned batch (kernel throughput); e2e is the end-to-end number"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_s / args.steps * 1e3, "p50_ms_batch1": lat[len(lat) // 2],
                    "p99_ms_batch1": lat[int(len(lat) * 0.99)], "distinct_batches": args.steps,
                    "includes": "host planning, H2D of the plan, kernels, D2H of the MSets, result scatter" +
                                ("; per batch the phase-1 statistics exchange, the all-to-all and the merge" if world > 1 else "")},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "hbm", "kernel": cfg["kernel"],
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": traffic_src,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                         "kernel_ms_per_launch": kern_ms},
            "step_breakdown_ms": step_parts, "step_bound_by": bound, "host_cpus": host_cpus,
            "stats_exchange_via": None if world == 1 else ("shared memory (one node)" if use_shm else "gloo all-reduce"),
            "bounds_approx_fraction": approx0 / BATCH,
            "clocks": clocks}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            binfo = build_reference_db()
            cores, cdet = ref_cores()
            nq = ref_queries_per_step(cfg, cores) if not REF_Q_ENV else cfg["ref_queries"]
            cinfo, _ = run_reference_queries(cfg, binfo["dbs"], nq, 3, 1, cores)
            line["cpu_baseline"] = {
                "value": cinfo["qps"], "unit": UNIT, "cores": cores, "kind": "reference", "cores_detail": cdet,
                "sample": (f"3 passes of {nq} queries of the same workload on the full {NDOCS}-doc "
                           f"glass DB, {cores} threads (one Xapian::Database+Enquire each, opened before the timed passes)"),
                "p50_ms": cinfo["p50_ms"], "p99_ms": cinfo["p99_ms"],
                "single_thread": single_thread_baseline(cfg, binfo["dbs"])}
            if not args.no_parity:
                line["parity"] = parity_against_reference(cfg, binfo["dbs"], xgm.Searcher(ix, max_batch=256, max_topk=TOPK), cores)
        except Exception as e:  # the baseline is reported, never required for the GPU numbers
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": ref_cores()[0], "kind": "reference",
                                    "sample": f"unavailable: {e}"}
    if rank == 0:
        print(json.dumps(line))
    if dump:
        dump_outputs(args.dump_outputs, dump, "" if world == 1 else f".rank{rank}")
    if world > 1:
        if shm is not None:
            dist.barrier()
            shm.close()  # rank 0 removes the /dev/shm file
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the dump diff against the compiled reference")
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS), help="BASELINE.json configuration (default C2)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the MSets of the last timed step of each timed path as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return reference_arm(args)
    return ours(args)


if __name__ == "__main__":
    sys.exit(main())
