"""oracle/oracle.py — TEST INFRASTRUCTURE, not product code.

ctypes bindings for the C restatement (oracle/xgm_oracle.c → oracle/libxgm_oracle.so) and a thin
subprocess wrapper around the compiled reference (oracle/_ref/ref_runner, which links the
reference's own Xapian built by oracle/build_ref.sh).  Only tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs may import this module.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libxgm_oracle.so")
REF_DIR = os.path.join(HERE, "_ref")
REF_RUNNER = os.path.join(REF_DIR, "ref_runner")
REF_RUNNER_XGM = os.path.join(REF_DIR, "ref_runner_xgm")  # same driver on libxapian_ref_xgm.so (the xgm shim)

OP_AND, OP_OR = 0, 1
SORT_REL, SORT_VAL_REL, SORT_VAL, SORT_REL_VAL = 0, 1, 2, 3
FILTER_NONE, FILTER_VALUE_RANGE_MIN, FILTER_MULTI_RANGE = 0, 1, 2


def _digest(deps: Sequence[str], recipe: Sequence[str]) -> str:
    import hashlib
    repo = os.path.dirname(HERE)  # the command names paths inside the tree; where the tree lies does not count
    h = hashlib.sha256("\0".join(recipe).replace(repo, "").encode())
    for d in deps:
        with open(d, "rb") as f:
            h.update(hashlib.sha256(f.read()).digest())
    return h.hexdigest()


def stale(target: str, deps: Sequence[str], recipe: Sequence[str]) -> bool:
    """True unless target exists and target.sha256 holds the digest of the contents of deps and of the build
    command it was made from.  Contents, not modification times: a tree that was copied or checked out again
    keeps its build products, while a changed source or flag still rebuilds."""
    try:
        with open(target + ".sha256") as f:
            return not os.path.exists(target) or f.read().strip() != _digest(deps, recipe)
    except OSError:
        return True


def mark_built(target: str, deps: Sequence[str], recipe: Sequence[str]) -> None:
    with open(target + ".sha256", "w") as f:
        f.write(_digest(deps, recipe) + "\n")


def build(force: bool = False) -> str:
    """Compile the C restatement (gcc, no FMA contraction)."""
    src = os.path.join(HERE, "xgm_oracle.c")
    deps = [src, os.path.join(HERE, "xgm_oracle.h"),
            os.path.join(HERE, "..", "xapiand_b200", "csrc", "xgm_corpus.h")]
    cmd = ["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-o", LIB_PATH, src, "-lm"]
    if not force and not stale(LIB_PATH, deps, cmd):
        return LIB_PATH
    subprocess.check_call(cmd)
    mark_built(LIB_PATH, deps, cmd)
    return LIB_PATH


class _Index(C.Structure):
    _fields_ = [("doccount", C.c_uint32), ("lastdocid", C.c_uint32), ("total_length", C.c_uint64),
                ("doclen_lb", C.c_uint32), ("doclen_ub", C.c_uint32),
                ("doclen", C.POINTER(C.c_uint32)), ("nterms", C.c_uint32),
                ("off", C.POINTER(C.c_uint64)), ("docids", C.POINTER(C.c_uint32)),
                ("wdfs", C.POINTER(C.c_uint32)), ("collfreq", C.POINTER(C.c_uint64)),
                ("wdf_ub", C.POINTER(C.c_uint32)), ("names", C.POINTER(C.c_char_p)),
                ("nvals0", C.POINTER(C.c_uint8)), ("vals0", C.POINTER(C.c_uint64)),
                ("val1", C.POINTER(C.c_uint64)), ("has1", C.POINTER(C.c_uint8))]


class _Stats(C.Structure):
    _fields_ = [("collection_size", C.c_uint32), ("total_length", C.c_uint64),
                ("termfreq", C.POINTER(C.c_uint32)), ("maybe_termfreq", C.POINTER(C.c_uint32))]


class _Query(C.Structure):
    _fields_ = [("op", C.c_int), ("nterms", C.c_uint32), ("terms", C.POINTER(C.c_uint32)),
                ("wqf", C.POINTER(C.c_uint32)), ("factors", C.POINTER(C.c_double)), ("first", C.c_uint32),
                ("maxitems", C.c_uint32),
                ("check_at_least", C.c_uint32), ("stats", C.POINTER(_Stats)),
                ("k1", C.c_double), ("k3", C.c_double), ("b", C.c_double), ("min_normlen", C.c_double),
                ("filter", C.c_int), ("range_lo", C.c_uint64), ("range_hi", C.c_uint64),
                ("sort_by", C.c_int), ("sort_slot", C.c_int), ("sort_reverse", C.c_int),
                ("nfilter", C.c_uint32), ("filter_terms", C.POINTER(C.c_uint32)),
                ("nnot", C.c_uint32), ("not_terms", C.POINTER(C.c_uint32)),
                ("nmaybe", C.c_uint32), ("maybe_terms", C.POINTER(C.c_uint32)),
                ("filter_weighted", C.c_int), ("filter_factor", C.c_double),
                ("sort_keymaker", C.c_int), ("sort_missing", C.c_uint64)]


class _MSet(C.Structure):
    _fields_ = [("n", C.c_uint32), ("docids", C.POINTER(C.c_uint32)), ("weights", C.POINTER(C.c_double)),
                ("sortvals", C.POINTER(C.c_uint64)),
                ("matches_lower_bound", C.c_uint32), ("matches_estimated", C.c_uint32),
                ("matches_upper_bound", C.c_uint32), ("known_matching_docs", C.c_uint32),
                ("exact_matches", C.c_uint32),
                ("max_possible", C.c_double), ("max_attained", C.c_double),
                ("percent_scale_factor", C.c_double)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB_PATH)
        L.orc_index_synthetic.restype = C.POINTER(_Index)
        L.orc_index_synthetic.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int]
        L.orc_index_load_flat.restype = C.POINTER(_Index)
        L.orc_index_load_flat.argtypes = [C.c_char_p]
        L.orc_index_free.argtypes = [C.POINTER(_Index)]
        L.orc_index_make_sparse.argtypes = [C.POINTER(_Index), C.c_uint32, C.c_uint32]
        L.orc_query_defaults.argtypes = [C.POINTER(_Query)]
        L.orc_match.argtypes = [C.POINTER(_Index), C.POINTER(_Query), C.POINTER(_MSet)]
        L.orc_merge.argtypes = [C.POINTER(_MSet), C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_int,
                                C.POINTER(_MSet)]
        L.orc_mset_free.argtypes = [C.POINTER(_MSet)]
        L.orc_round_estimate.restype = C.c_uint32
        L.orc_round_estimate.argtypes = [C.c_uint32] * 3
        L.orc_and_order.argtypes = [C.POINTER(C.c_uint32), C.c_uint32, C.POINTER(C.c_uint32)]
        L.orc_or_program.argtypes = [C.POINTER(C.c_uint32), C.c_uint32, C.POINTER(C.c_int32)]
        L.orc_or_program.restype = C.c_uint32
        L.orc_bm25_init.argtypes = [C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_double, C.c_double,
                                    C.c_double, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.orc_bm25_sumpart.restype = C.c_double
        L.orc_bm25_sumpart.argtypes = [C.c_double] * 5 + [C.c_uint32, C.c_uint32]
        L.orc_bm25_maxpart.restype = C.c_double
        L.orc_bm25_maxpart.argtypes = [C.c_double] * 5 + [C.c_uint32, C.c_uint32]
        _lib = L
    return _lib


@dataclass
class MSet:
    docids: np.ndarray
    weights: np.ndarray
    sortvals: np.ndarray
    lb: int = 0
    est: int = 0
    ub: int = 0
    known: int = 0
    exact: int = 0
    max_possible: float = 0.0
    max_attained: float = 0.0
    percent_scale_factor: float = 0.0


@dataclass
class Query:
    op: int
    terms: Sequence[int]
    first: int = 0
    maxitems: int = 10
    check_at_least: int = 0
    wqf: Optional[Sequence[int]] = None
    factors: Optional[Sequence[float]] = None    # OP_SCALE_WEIGHT factor per term (oracle only so far)
    bm25: Optional[tuple] = None                 # (k1, k3, b, min_normlen); None = BM25Weight defaults
    filter: int = FILTER_NONE
    range_lo: int = 0
    range_hi: int = 0
    sort_by: int = SORT_REL
    sort_slot: int = 1
    sort_reverse: bool = False
    # global stats for the two-phase scheme: (collection_size, total_length, [termfreq per term]
    # [, [termfreq per maybe term]])
    stats: Optional[tuple] = None
    # OP_FILTER(q, AND of boolean terms) / OP_AND_NOT(q, OR of terms) / OP_AND_MAYBE(q, OR of terms), AND base only
    filter_terms: Sequence[int] = ()
    not_terms: Sequence[int] = ()
    maybe_terms: Sequence[int] = ()
    # Xapiand's MultipleValueRange as a weighted AND child / Multi_MultiValueKeyMaker sort (see xgm_oracle.h)
    filter_weighted: bool = False
    filter_factor: float = 0.0
    sort_keymaker: bool = False
    sort_missing: int = 0


def _mset_from_c(m: _MSet) -> MSet:
    n = m.n
    out = MSet(
        docids=np.ctypeslib.as_array(m.docids, (n,)).copy() if n else np.zeros(0, np.uint32),
        weights=np.ctypeslib.as_array(m.weights, (n,)).copy() if n else np.zeros(0, np.float64),
        sortvals=np.ctypeslib.as_array(m.sortvals, (n,)).copy() if n else np.zeros(0, np.uint64),
        lb=m.matches_lower_bound, est=m.matches_estimated, ub=m.matches_upper_bound,
        known=m.known_matching_docs, exact=m.exact_matches,
        max_possible=m.max_possible, max_attained=m.max_attained,
        percent_scale_factor=m.percent_scale_factor)
    return out


class Index:
    """Flat posting arrays held by the C oracle."""

    def __init__(self, ptr):
        if not ptr:
            raise RuntimeError("oracle index construction failed")
        self._p = ptr
        self.c = ptr.contents

    @classmethod
    def synthetic(cls, ndocs: int, vocab: int, seed: int = 12345, nshards: int = 1, shard: int = 0,
                  values: bool = False) -> "Index":
        return cls(lib().orc_index_synthetic(ndocs, vocab, seed, nshards, shard, int(values)))

    @classmethod
    def load_flat(cls, path: str) -> "Index":
        return cls(lib().orc_index_load_flat(path.encode()))

    def make_sparse(self, mod0: int, mod1: int):
        """Drop slot values by the rule of `ref_runner build --mvalues-sparse mod0 mod1`."""
        lib().orc_index_make_sparse(self._p, mod0, mod1)

    def close(self):
        if self._p:
            lib().orc_index_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- flat views (zero-copy numpy) -------------------------------------------------
    @property
    def doccount(self): return self.c.doccount
    @property
    def lastdocid(self): return self.c.lastdocid
    @property
    def total_length(self): return self.c.total_length
    @property
    def nterms(self): return self.c.nterms
    @property
    def doclen_lb(self): return self.c.doclen_lb
    @property
    def doclen_ub(self): return self.c.doclen_ub

    def doclen(self) -> np.ndarray:
        return np.ctypeslib.as_array(self.c.doclen, (self.c.lastdocid + 1,))

    def offsets(self) -> np.ndarray:
        return np.ctypeslib.as_array(self.c.off, (self.c.nterms + 1,))

    def all_docids(self) -> np.ndarray:
        n = int(self.offsets()[-1])
        return np.ctypeslib.as_array(self.c.docids, (n,))

    def all_wdfs(self) -> np.ndarray:
        n = int(self.offsets()[-1])
        return np.ctypeslib.as_array(self.c.wdfs, (n,))

    def termfreq(self, t: int) -> int:
        off = self.offsets()
        return int(off[t + 1] - off[t])

    def postings(self, t: int):
        off = self.offsets()
        a, b = int(off[t]), int(off[t + 1])
        return self.all_docids()[a:b], self.all_wdfs()[a:b]

    def wdf_ub(self) -> np.ndarray:
        return np.ctypeslib.as_array(self.c.wdf_ub, (self.c.nterms,))

    def collfreq(self) -> np.ndarray:
        return np.ctypeslib.as_array(self.c.collfreq, (self.c.nterms,))

    def name(self, t: int) -> str:
        return self.c.names[t].decode()

    def values(self):
        if not self.c.nvals0:
            return None
        n = self.c.lastdocid + 1
        return (np.ctypeslib.as_array(self.c.nvals0, (n,)),
                np.ctypeslib.as_array(self.c.vals0, (3 * n,)).reshape(n, 3),
                np.ctypeslib.as_array(self.c.val1, (n,)))

    # ---- matching -----------------------------------------------------------------------
    def match(self, q: Query) -> MSet:
        L = lib()
        cq = _Query()
        L.orc_query_defaults(C.byref(cq))
        terms = (C.c_uint32 * len(q.terms))(*q.terms)
        cq.op = q.op
        cq.nterms = len(q.terms)
        cq.terms = terms
        if q.wqf is not None:
            wqf = (C.c_uint32 * len(q.wqf))(*q.wqf)
            cq.wqf = wqf
        if q.factors is not None:
            fac = (C.c_double * len(q.factors))(*q.factors)
            cq.factors = fac
        if q.bm25 is not None:
            cq.k1, cq.k3, cq.b, cq.min_normlen = [float(x) for x in q.bm25]
        cq.first, cq.maxitems, cq.check_at_least = q.first, q.maxitems, q.check_at_least
        cq.filter, cq.range_lo, cq.range_hi = q.filter, q.range_lo, q.range_hi
        cq.sort_by, cq.sort_slot, cq.sort_reverse = q.sort_by, q.sort_slot, int(q.sort_reverse)
        cq.filter_weighted, cq.filter_factor = int(q.filter_weighted), float(q.filter_factor)
        cq.sort_keymaker, cq.sort_missing = int(q.sort_keymaker), int(q.sort_missing)
        if q.stats is not None:
            tf = (C.c_uint32 * len(q.terms))(*q.stats[2])
            mtf = None
            if len(q.stats) > 3 and q.stats[3] is not None:
                mtf = (C.c_uint32 * len(q.maybe_terms))(*q.stats[3])
            st = _Stats(q.stats[0], q.stats[1], tf, mtf)
            cq.stats = C.pointer(st)
        keep = []
        for name, ts in (("filter", q.filter_terms), ("not", q.not_terms), ("maybe", q.maybe_terms)):
            arr = (C.c_uint32 * max(1, len(ts)))(*ts)
            keep.append(arr)
            setattr(cq, "n" + name, len(ts))
            setattr(cq, name + "_terms", arr)
        m = _MSet()
        rc = L.orc_match(self._p, C.byref(cq), C.byref(m))
        if rc != 0:
            raise RuntimeError("orc_match failed")
        out = _mset_from_c(m)
        L.orc_mset_free(C.byref(m))
        return out


def merge(parts: List[MSet], first: int, maxitems: int, sort_by: int = SORT_REL,
          sort_reverse: bool = False) -> MSet:
    L = lib()
    arr = (_MSet * len(parts))()
    keep = []
    for i, p in enumerate(parts):
        d = np.ascontiguousarray(p.docids, np.uint32)
        w = np.ascontiguousarray(p.weights, np.float64)
        s = np.ascontiguousarray(p.sortvals if len(p.sortvals) == len(d) else np.zeros(len(d), np.uint64), np.uint64)
        keep += [d, w, s]
        arr[i].n = len(d)
        arr[i].docids = d.ctypes.data_as(C.POINTER(C.c_uint32))
        arr[i].weights = w.ctypes.data_as(C.POINTER(C.c_double))
        arr[i].sortvals = s.ctypes.data_as(C.POINTER(C.c_uint64))
        arr[i].matches_lower_bound, arr[i].matches_estimated, arr[i].matches_upper_bound = p.lb, p.est, p.ub
        arr[i].known_matching_docs, arr[i].exact_matches = p.known, p.exact
        arr[i].max_possible, arr[i].max_attained = p.max_possible, p.max_attained
        arr[i].percent_scale_factor = p.percent_scale_factor
    m = _MSet()
    L.orc_merge(arr, len(parts), first, maxitems, sort_by, int(sort_reverse), C.byref(m))
    out = _mset_from_c(m)
    L.orc_mset_free(C.byref(m))
    return out


def convert_to_percent(weight: float, percent_scale_factor: float) -> int:
    """MSet::Internal::convert_to_percent, api/mset.cc:333-365."""
    if percent_scale_factor == 0.0:
        return 100
    if weight <= 0.0:
        return 0
    pct = int(weight * percent_scale_factor + 100.0 * 2.220446049250313e-16)
    return 1 if pct <= 0 else min(pct, 100)


def round_estimate(lb: int, ub: int, est: int) -> int:
    return int(lib().orc_round_estimate(lb, ub, est))


def and_order(termfreqs: Sequence[int]) -> List[int]:
    n = len(termfreqs)
    tf = (C.c_uint32 * n)(*termfreqs)
    out = (C.c_uint32 * n)()
    lib().orc_and_order(tf, n, out)
    return list(out)


def or_program(termfreqs: Sequence[int]) -> List[int]:
    n = len(termfreqs)
    tf = (C.c_uint32 * n)(*termfreqs)
    out = (C.c_int32 * (2 * n))()
    k = lib().orc_or_program(tf, n, out)
    return list(out[:k])


# ------------------------------------------------------------------------------------------
# compiled reference (oracle/_ref) — available wherever oracle/_ref was built or shipped
# ------------------------------------------------------------------------------------------

def have_reference() -> bool:
    return os.path.exists(REF_RUNNER) and os.path.exists(os.path.join(REF_DIR, "libxapian_ref.so"))


def ref_build(out_dir: str, ndocs: int, vocab: int, seed: int = 12345, nshards: int = 1, shard: int = 0,
              values: bool = False, env=None, mvalues: bool = False, sparse=None) -> dict:
    cmd = [REF_RUNNER, "build", "--out", out_dir, "--docs", str(ndocs), "--vocab", str(vocab),
           "--seed", str(seed), "--nshards", str(nshards), "--shard", str(shard)]
    if values:
        cmd.append("--values")
    if mvalues:  # Xapiand's slot encoding: StringList of Serialise::positive keys
        cmd.append("--mvalues")
        if sparse:
            cmd += ["--mvalues-sparse", str(sparse[0]), str(sparse[1])]
    e = dict(os.environ)
    e.setdefault("XAPIAN_FLUSH_THRESHOLD", "200000")
    if env:
        e.update(env)
    return json.loads(subprocess.check_output(cmd, env=e).decode().strip().splitlines()[-1])


def ref_build_parallel(out_dir: str, ndocs: int, vocab: int, seed: int = 12345, procs: int = 8,
                       values: bool = False, compact: bool = True, mvalues: bool = False, nshards: int = 1,
                       shard: int = 0) -> dict:
    """Write the corpus as `procs` contiguous docid-range glass DBs in parallel (one writer process
    each), then Database::compact them into one DB whose docids are the corpus docids.  Returns timing
    info; the result lives in out_dir/db (or out_dir/part*/ when compact=False)."""
    import time
    os.makedirs(out_dir, exist_ok=True)
    marker = os.path.join(out_dir, "READY.json")
    if os.path.exists(marker):
        return json.load(open(marker))
    procs = max(1, min(procs, ndocs))
    per = (ndocs + procs - 1) // procs
    e = dict(os.environ)
    e.setdefault("XAPIAN_FLUSH_THRESHOLD", "200000")
    t0 = time.time()
    ps, parts = [], []
    for i in range(procs):
        a, b = i * per + 1, min(ndocs, (i + 1) * per)
        if a > b:
            break
        d = os.path.join(out_dir, f"part{i:03d}")
        parts.append(d)
        cmd = [REF_RUNNER, "build", "--out", d, "--docs", str(ndocs), "--vocab", str(vocab), "--seed", str(seed),
               "--range-first", str(a), "--range-last", str(b), "--nshards", str(nshards), "--shard", str(shard)]
        if values:
            cmd.append("--values")
        if mvalues:
            cmd.append("--mvalues")
        ps.append(subprocess.Popen(cmd, env=e, stdout=subprocess.DEVNULL))
    for p in ps:
        if p.wait() != 0:
            raise RuntimeError("reference build failed")
    t1 = time.time()
    info = dict(ndocs=ndocs, vocab=vocab, seed=seed, procs=len(parts), build_s=round(t1 - t0, 2))
    if compact and len(parts) > 1:
        cmd = [REF_RUNNER, "compact", "--out", os.path.join(out_dir, "db")]
        for d in parts:
            cmd += ["--db", d]
        subprocess.check_call(cmd, stdout=subprocess.DEVNULL)
        info["compact_s"] = round(time.time() - t1, 2)
        info["dbs"] = [os.path.join(out_dir, "db")]
        import shutil
        for d in parts:
            shutil.rmtree(d, ignore_errors=True)
    else:
        info["dbs"] = parts
    json.dump(info, open(marker, "w"))
    return info


def query_line(op: str, terms: Sequence[str], first: int, maxitems: int, check_at_least: int = 0,
               vr: Optional[tuple] = None, sort: Optional[tuple] = None, filter_terms: Sequence[str] = (),
               not_terms: Sequence[str] = (), maybe_terms: Sequence[str] = (), bm25: Optional[tuple] = None,
               mvr: Optional[tuple] = None, keysort: Optional[tuple] = None) -> str:
    s = f"{op} {first} {maxitems} {check_at_least} {len(terms)} " + " ".join(terms)
    for tag, ts in (("FT", filter_terms), ("NOT", not_terms), ("MAYBE", maybe_terms)):
        if ts:
            s += f" {tag} {len(ts)} " + " ".join(ts)
    if bm25 is not None:  # (k1, k3, b, min_normlen)
        s += " BM25 " + " ".join(repr(float(x)) for x in bm25)
    if vr is not None:
        s += f" VR {vr[0]} {vr[1]} {vr[2]}"
    if mvr is not None:  # (slot, lo, hi, weighted): Xapiand's MultipleValueRange as OP_FILTER right side / OP_AND child
        s += f" {'MVRW' if len(mvr) > 3 and mvr[3] else 'MVR'} {mvr[0]} {mvr[1]} {mvr[2]}"
    if keysort is not None:  # (slot, reverse): Multi_MultiValueKeyMaker{SerialiseKey}, set_sort_by_key_then_relevance
        s += f" KEYSORT {keysort[0]} {int(keysort[1])}"
    if sort is not None:
        s += f" SORT {sort[0]} {int(sort[1])}"
        if len(sort) > 2 and sort[2]:
            s += f" SORTMODE {int(sort[2])}"  # 1 = value only, 2 = relevance then value
    return s


@dataclass
class RefResult:
    docids: List[int] = field(default_factory=list)
    weights: List[float] = field(default_factory=list)
    sort_keys: List[str] = field(default_factory=list)
    percents: List[int] = field(default_factory=list)
    lb: int = 0
    est: int = 0
    ub: int = 0
    max_possible: float = 0.0
    max_attained: float = 0.0
    served: int = -1      # shim runner only: 1 = libxgm answered, 0 = the reference matcher did
    flags: int = 0
    reason: str = ""


def parse_dump(path: str) -> List[RefResult]:
    out: List[RefResult] = []
    with open(path) as f:
        cur = None
        for line in f:
            p = line.split()
            if not p:
                continue
            if p[0] == "Q":
                cur = RefResult(lb=int(p[3]), est=int(p[4]), ub=int(p[5]),
                                max_possible=float(p[6]), max_attained=float(p[7]))
                if len(p) > 10 and p[8].startswith("S"):
                    cur.served, cur.flags, cur.reason = int(p[8][1:]), int(p[9][1:]), p[10]
                out.append(cur)
            else:
                cur.docids.append(int(p[0]))
                cur.weights.append(float(p[1]))
                if p[-1].startswith("p"):
                    cur.percents.append(int(p.pop()[1:]))
                if len(p) > 2:
                    cur.sort_keys.append(p[2])
    return out


def have_shim_reference() -> bool:
    return os.path.exists(REF_RUNNER_XGM) and os.path.exists(os.path.join(REF_DIR, "libxapian_ref_xgm.so"))


def ref_query(dbs: Sequence[str], query_lines: Sequence[str], workdir: str, threads: int = 1,
              twophase: bool = False, repeat: int = 1, warmup: int = 0, dump: bool = True, shim: bool = False,
              env=None):
    """shim=True: the same driver linked against libxapian_ref_xgm.so — Matcher::get_mset tries libxgm first."""
    os.makedirs(workdir, exist_ok=True)
    qf = os.path.join(workdir, "queries.txt")
    with open(qf, "w") as f:
        f.write("\n".join(query_lines) + "\n")
    e = dict(os.environ)
    if shim:
        e.setdefault("XGM_LIB", os.path.join(HERE, "..", "xapiand_b200", "libxgm.so"))
    if env:
        e.update(env)
    cmd = [REF_RUNNER_XGM if shim else REF_RUNNER, "query", "--queries", qf, "--threads", str(threads), "--repeat", str(repeat),
           "--warmup", str(warmup)]
    for d in dbs:
        cmd += ["--db", d]
    if twophase:
        cmd.append("--twophase")
    df = os.path.join(workdir, "dump_xgm.txt" if shim else "dump.txt")
    if dump:
        cmd += ["--dump", df]
    info = json.loads(subprocess.check_output(cmd, env=e).decode().strip().splitlines()[-1])
    return info, (parse_dump(df) if dump else None)
