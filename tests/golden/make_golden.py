"""Generate the golden fixtures in tests/golden/ by running the COMPILED REFERENCE (oracle/_ref:
the reference's own Xapian built from /root/reference/src/xapian by oracle/build_ref.sh) on seeded
synthetic corpora.  Only runs where oracle/_ref exists (this container); the fixtures it writes are
committed so the oracle and the CUDA path can be checked against the reference anywhere.

    python tests/golden/make_golden.py
"""
import json
import os
import random
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def name(r):
    return f"T{r:06d}"


def run_set(tag, ndocs, vocab, queries, nshards=1, twophase=False, values=False, seed=12345):
    tmp = tempfile.mkdtemp(prefix="xgm_golden_")
    try:
        dbs = []
        for s in range(nshards):
            d = os.path.join(tmp, f"s{s}")
            O.ref_build(d, ndocs, vocab, seed=seed, nshards=nshards, shard=s, values=values)
            dbs.append(d)
        lines = []
        for q in queries:
            facs, wq = q.get("factors"), q.get("wqf")
            tnames = [name(t) + ("" if not wq or wq[j] == 1 else f"#{wq[j]}") +
                      ("" if not facs or facs[j] == 1.0 else f"^{facs[j]!r}") for j, t in enumerate(q["terms"])]
            lines.append(O.query_line("TERM" if len(q["terms"]) == 1 else q["op"], tnames,
                                      q["first"], q["maxitems"], q["check_at_least"], vr=q.get("vr"),
                                      sort=(q["sort"] + [q.get("sort_mode", 0)]) if q.get("sort") else None,
                                      bm25=q.get("bm25"),
                                      filter_terms=[name(t) for t in q.get("filter_terms", [])],
                                      not_terms=[name(t) for t in q.get("not_terms", [])],
                                      maybe_terms=[name(t) for t in q.get("maybe_terms", [])]))
        info, res = O.ref_query(dbs, lines, os.path.join(tmp, "w"), twophase=twophase)
        fixture = dict(tag=tag, ndocs=ndocs, vocab=vocab, seed=seed, nshards=nshards, twophase=twophase, values=values,
                       queries=[])
        for q, r in zip(queries, res):
            e = dict(q)
            e["docids"] = r.docids
            e["weights"] = [float(w).hex() for w in r.weights]
            if r.sort_keys:
                e["sort_keys"] = r.sort_keys
            e["percents"] = r.percents
            e.update(lb=r.lb, est=r.est, ub=r.ub, max_possible=float(r.max_possible).hex(),
                     max_attained=float(r.max_attained).hex())
            fixture["queries"].append(e)
        with open(os.path.join(OUT, f"{tag}.json"), "w") as f:
            json.dump(fixture, f, separators=(",", ":"))
        print(tag, len(queries), "queries", os.path.getsize(os.path.join(OUT, f"{tag}.json")), "bytes")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run_mv_set(tag, ndocs, vocab, queries, sparse=(7, 5), seed=12345, db=None, with_slots=True):
    """Xapiand's own multivalue classes (oracle/_ref/libxapiand_mv_ref.so = src/multivalue/range.cc, keymaker.cc …
    compiled from the reference): slots written as StringLists of Serialise::positive keys, MultipleValueRange as
    OP_FILTER right side or weighted OP_AND child, Multi_MultiValueKeyMaker{SerialiseKey} as the sorter.
    db: an existing database of that corpus to query instead of building one; with_slots=False leaves the
    per-document slot bytes out of the fixture (a test that opens the database itself does not need them)."""
    import subprocess
    tmp = tempfile.mkdtemp(prefix="xgm_golden_")
    try:
        d = db or os.path.join(tmp, "db")
        if db is None:
            O.ref_build(d, ndocs, vocab, seed=seed, mvalues=True, sparse=sparse)
        lines = [O.query_line("TERM" if len(q["terms"]) == 1 else "AND", [name(t) for t in q["terms"]], q["first"],
                              q["maxitems"], q["check_at_least"], mvr=q.get("mvr"), keysort=q.get("keysort"))
                 for q in queries]
        info, res = O.ref_query([d], lines, os.path.join(tmp, "w"))
        slots = {}
        for ln in subprocess.check_output([O.REF_RUNNER, "slots", "--db", d]).decode().splitlines() if with_slots else []:
            sl, did, hx = (ln.split() + [""])[:3]
            slots.setdefault(sl, {})[did] = hx
        nums = sorted({v for q in queries if q.get("mvr") for v in q["mvr"][1:3]})
        ser = subprocess.check_output([O.REF_RUNNER, "serialise"] + [str(v) for v in nums]).decode().split()
        fixture = dict(tag=tag, ndocs=ndocs, vocab=vocab, seed=seed, sparse=list(sparse), slots=slots,
                       serialised=dict(zip(map(str, nums), ser)), queries=[])
        for q, r in zip(queries, res):
            e = dict(q)
            e["docids"] = r.docids
            e["weights"] = [float(w).hex() for w in r.weights]
            if r.sort_keys:
                e["sort_keys"] = r.sort_keys
            e["percents"] = r.percents
            e.update(lb=r.lb, est=r.est, ub=r.ub, max_possible=float(r.max_possible).hex(),
                     max_attained=float(r.max_attained).hex())
            fixture["queries"].append(e)
        with open(os.path.join(OUT, f"{tag}.json"), "w") as f:
            json.dump(fixture, f, separators=(",", ":"))
        print(tag, len(queries), "queries", os.path.getsize(os.path.join(OUT, f"{tag}.json")), "bytes")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


#        name                    docs  vocab  seed   ref_build options
GLASS = [("plain_1k",             1000, 300,   5,     {}),
         ("mvalues_sparse_1500",  1500, 600,   12345, dict(mvalues=True, sparse=[7, 5])),
         ("values_2k",            2000, 40,    5,     dict(values=True)),
         ("single_doc",           1,    5,     5,     {})]


def _export_digest(db, flat):
    """Size and SHA-256 of the flat file `ref_runner export` writes by walking db through the public iterators."""
    import hashlib
    import subprocess
    subprocess.check_call([O.REF_RUNNER, "export", "--db", db, "--out", flat], stdout=subprocess.DEVNULL)
    data = open(flat, "rb").read()
    return len(data), hashlib.sha256(data).hexdigest()


def _tar_xz(src_dir, dst):
    """The database directory as a reproducible .tar.xz (sorted members, no owner or time stamps)."""
    import lzma
    import tarfile
    with lzma.open(dst, "wb", preset=9 | lzma.PRESET_EXTREME) as xz, tarfile.open(fileobj=xz, mode="w") as tar:
        for fn in sorted(os.listdir(src_dir)):
            ti = tar.gettarinfo(os.path.join(src_dir, fn), arcname=fn)
            ti.mtime, ti.uid, ti.gid, ti.uname, ti.gname, ti.mode = 0, 0, 0, "", "", 0o644
            with open(os.path.join(src_dir, fn), "rb") as f:
                tar.addfile(ti, f)


def edge_glass_queries(rng, n, topranks, ndocs):
    """AND / OR of 1-5 terms, top-10 or top-100, with and without check_at_least = every document."""
    qs = []
    for i in range(n):
        op = "AND" if i % 2 == 0 else "OR"
        terms = rng.sample(range(topranks), rng.choice([1, 2, 3, 5]))
        qs.append(dict(op=op, terms=terms, first=0, maxitems=rng.choice([10, 100]), check_at_least=rng.choice([0, ndocs])))
    return qs


def run_glass_sets():
    """Glass databases written by the reference, for the tests of the direct glass reader (tests/golden/glass/):
    each database as .tar.xz plus the digest of the reference's own flat export of it (databases.json), the
    reference's MSets on the multivalue database (multivalue_1500.json), and glass_6k.json: the digest of the
    export of a 6000-document database and the reference's MSets on it (weights as the SHA-256 of their
    little-endian float64 bytes, to keep the fixture small)."""
    import hashlib
    import numpy as np
    gdir = os.path.join(OUT, "glass")
    os.makedirs(gdir, exist_ok=True)
    tmp = tempfile.mkdtemp(prefix="xgm_golden_")
    try:
        meta = {}
        for tag, ndocs, vocab, seed, kw in GLASS:
            d = os.path.join(tmp, tag)
            O.ref_build(d, ndocs, vocab, seed=seed, **kw)
            size, sha = _export_digest(d, d + ".flat")
            meta[tag] = dict(ndocs=ndocs, vocab=vocab, seed=seed, **kw, export_bytes=size, export_sha256=sha)
            _tar_xz(d, os.path.join(gdir, f"{tag}.tar.xz"))
            print(tag, os.path.getsize(os.path.join(gdir, f"{tag}.tar.xz")), "bytes")
        with open(os.path.join(gdir, "databases.json"), "w") as f:
            json.dump(meta, f, indent=1)
        mv = meta["mvalues_sparse_1500"]
        run_mv_set("multivalue_1500", mv["ndocs"], mv["vocab"], mv_queries(random.Random(20261017), 80, 60, mv["ndocs"]),
                   sparse=mv["sparse"], seed=mv["seed"], db=os.path.join(tmp, "mvalues_sparse_1500"), with_slots=False)

        ndocs, vocab, seed = 6000, 800, 99
        d = os.path.join(tmp, "edge")
        O.ref_build(d, ndocs, vocab, seed=seed)
        size, sha = _export_digest(d, d + ".flat")
        queries = edge_glass_queries(random.Random(12), 80, 120, ndocs)
        lines = [O.query_line("TERM" if len(q["terms"]) == 1 else q["op"], [name(t) for t in q["terms"]], 0, q["maxitems"],
                              q["check_at_least"]) for q in queries]
        _, res = O.ref_query([d], lines, os.path.join(tmp, "w"))
        for q, r in zip(queries, res):
            q.update(docids=r.docids, weights_sha256=hashlib.sha256(np.asarray(r.weights, "<f8").tobytes()).hexdigest(),
                     lb=r.lb, est=r.est, ub=r.ub, max_possible=float(r.max_possible).hex(),
                     max_attained=float(r.max_attained).hex())
        fixture = dict(tag="glass_6k", ndocs=ndocs, vocab=vocab, seed=seed, export_bytes=size, export_sha256=sha,
                       queries=queries)
        with open(os.path.join(OUT, "glass_6k.json"), "w") as f:
            json.dump(fixture, f, separators=(",", ":"))
        print("glass_6k", os.path.getsize(os.path.join(OUT, "glass_6k.json")), "bytes")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def mv_queries(rng, n, topranks, ndocs):
    qs = []
    for i in range(n):
        nb = rng.choice([1, 2, 2, 3])
        q = dict(terms=rng.sample(range(topranks), nb), first=rng.choice([0, 0, 3]), maxitems=rng.choice([5, 10, 100]),
                 check_at_least=rng.choice([0, 0, ndocs]))
        lo = rng.randrange(0, 950000)
        kind = i % 4
        if kind != 3:  # range source: filter (0, 1) or weighted AND child (2)
            q["mvr"] = [0, lo, lo + rng.choice([5000, 50000, 300000]), 1 if kind == 2 else 0]
        if i % 3 != 1:
            q["keysort"] = [rng.choice([0, 1, 1]), rng.choice([0, 1])]
        qs.append(q)
    return qs


def mixed(rng, n, topranks, ndocs, big_or_items):
    qs = []
    for i in range(n):
        kind = i % 5
        if kind == 0:
            q = dict(op="AND", terms=rng.sample(range(topranks), 3), first=0, maxitems=100, check_at_least=0)
        elif kind == 1:
            q = dict(op="OR", terms=rng.sample(range(topranks), 5), first=0, maxitems=big_or_items, check_at_least=0)
        elif kind == 2:
            q = dict(op="AND", terms=rng.sample(range(topranks), 1), first=0, maxitems=10, check_at_least=0)
        elif kind == 3:
            q = dict(op=rng.choice(["AND", "OR"]), terms=rng.sample(range(topranks), rng.choice([2, 3, 4])),
                     first=rng.choice([0, 3]), maxitems=rng.choice([1, 5, 20, 100]), check_at_least=ndocs)
        else:
            q = dict(op="AND", terms=rng.sample(range(topranks), 2), first=rng.choice([0, 0, 7]),
                     maxitems=rng.choice([10, 30]), check_at_least=0)
        qs.append(q)
    return qs


def ops_queries(rng, n, topranks, ndocs):
    """SURVEY.md §8(f)-1 shapes: OP_FILTER with boolean terms, OP_AND_NOT, OP_AND_MAYBE around an AND base."""
    qs = []
    for _ in range(n):
        nb = rng.choice([1, 2, 2, 3])
        pool = rng.sample(range(topranks), nb + 9)
        nf, nx, nm = rng.choice([0, 0, 1, 2, 3]), rng.choice([0, 0, 1, 2, 3]), rng.choice([0, 0, 1, 2, 3])
        if nf + nx + nm == 0:
            nx = 1
        qs.append(dict(op="AND", terms=pool[:nb], first=rng.choice([0, 0, 3]), maxitems=rng.choice([5, 10, 50, 200]),
                       check_at_least=rng.choice([0, 0, ndocs]), filter_terms=pool[nb:nb + nf],
                       not_terms=pool[nb + 3:nb + 3 + nx], maybe_terms=pool[nb + 6:nb + 6 + nm]))
    return qs


def orops_queries(rng, n, topranks, ndocs):
    """The same groups around an OR base — a free-text OR restricted by boolean terms, the commonest filtered
    search: OP_FILTER(OP_OR(...), terms), OP_AND_NOT, OP_AND_MAYBE (api/queryinternal.cc:2208-2283)."""
    qs = []
    for _ in range(n):
        nb = rng.choice([2, 2, 3, 4, 5])
        pool = rng.sample(range(topranks), nb + 9)
        nf, nx, nm = rng.choice([0, 1, 1, 2]), rng.choice([0, 0, 1, 2, 3]), rng.choice([0, 0, 0, 1, 2])
        if nf + nx + nm == 0:
            nf = 1
        qs.append(dict(op="OR", terms=pool[:nb], first=rng.choice([0, 0, 3]), maxitems=rng.choice([5, 10, 50, 200]),
                       check_at_least=rng.choice([0, 0, ndocs]), filter_terms=pool[nb:nb + nf],
                       not_terms=pool[nb + 3:nb + 3 + nx], maybe_terms=pool[nb + 6:nb + 6 + nm]))
    return qs


def scale_queries(rng, n, topranks, ndocs):
    """OP_SCALE_WEIGHT factors on the leaves of AND / OR queries (Xapiand's _boost); factor 0 = unweighted leaf."""
    qs = []
    for _ in range(n):
        nb = rng.choice([1, 2, 3, 4])
        fac = [rng.choice([1.0, 1.0, 2.0, 0.5, 3.25, 0.0, 1e-3]) for _ in range(nb)]
        if all(f == 0.0 for f in fac):
            fac[0] = 1.5
        qs.append(dict(op=rng.choice(["AND", "OR"]), terms=rng.sample(range(topranks), nb), factors=fac,
                       first=rng.choice([0, 0, 3]), maxitems=rng.choice([5, 10, 50, 200]),
                       check_at_least=rng.choice([0, 0, ndocs])))
    return qs


def regime_queries(rng, n, topranks, ndocs):
    """Intermediate check_at_least (between k+1 and the match count), small k, first > 0, value sorts: the
    regimes where ProtoMSet's min_weight lags (protomset.h:377-398)."""
    qs = []
    for i in range(n):
        nb = rng.choice([1, 2, 3, 4])
        q = dict(op=rng.choice(["AND", "OR"]), terms=rng.sample(range(topranks), nb), first=rng.choice([0, 0, 1, 3, 10]),
                 maxitems=rng.choice([1, 2, 5, 10, 50, 200]),
                 check_at_least=rng.choice([0, 3, 7, 20, 40, 100, 300, 1000, ndocs]))
        if i % 4 == 0:
            q["sort"] = [1, rng.choice([0, 1])]
        qs.append(q)
    return qs


def wqf_queries(rng, n, topranks, ndocs):
    """Within-query frequencies > 1 (Query(term, wqf): the (k3+1)*wqf/(k3+wqf) factor of BM25Weight::init)."""
    qs = []
    for _ in range(n):
        nb = rng.choice([1, 2, 3, 4])
        qs.append(dict(op=rng.choice(["AND", "OR"]), terms=rng.sample(range(topranks), nb),
                       wqf=[rng.choice([1, 1, 2, 3, 7]) for _ in range(nb)], first=rng.choice([0, 0, 3]),
                       maxitems=rng.choice([5, 10, 50]), check_at_least=rng.choice([0, 30, ndocs])))
    return qs


def sortmode_queries(rng, n, topranks, ndocs):
    """set_sort_by_value (mode 1) and set_sort_by_relevance_then_value (mode 2) next to value-then-relevance (0)."""
    qs = []
    for _ in range(n):
        nb = rng.choice([1, 2, 3])
        qs.append(dict(op=rng.choice(["AND", "OR"]), terms=rng.sample(range(topranks), nb), first=rng.choice([0, 0, 3]),
                       maxitems=rng.choice([1, 5, 10, 50, 200]), check_at_least=rng.choice([0, 20, 300, ndocs]),
                       sort=[1, rng.choice([0, 1])], sort_mode=rng.choice([0, 1, 2])))
    return qs


def bm25_queries(rng, n, topranks, ndocs):
    """BM25Weight(k1, 0, k3, b, min_normlen) away from the defaults (k1 = 0 and b = 0 switch the length
    normalisation off, k3 = 0 the wqf factor: bm25weight.cc:46-130), with wqf > 1 mixed in."""
    qs = []
    for _ in range(n):
        nb = rng.choice([1, 2, 3, 4])
        qs.append(dict(op=rng.choice(["AND", "OR"]), terms=rng.sample(range(topranks), nb),
                       wqf=[rng.choice([1, 1, 3]) for _ in range(nb)], first=rng.choice([0, 0, 3]),
                       maxitems=rng.choice([5, 10, 50]), check_at_least=rng.choice([0, 30, ndocs]),
                       bm25=[rng.choice([0.0, 0.5, 1.0, 1.2, 2.0]), rng.choice([0.0, 1.0, 7.0]),
                             rng.choice([0.0, 0.25, 0.5, 0.75, 1.0]), rng.choice([0.0, 0.5, 1.0])]))
    return qs


def main():
    if not O.have_reference():
        raise SystemExit("oracle/_ref not built: run oracle/build_ref.sh (needs /root/reference)")
    if sys.argv[1:] == ["glass"]:
        run_glass_sets()
        return
    if sys.argv[1:] == ["mv"]:
        run_mv_set("multivalue_5k", 5000, 2000, mv_queries(random.Random(20260930), 240, 60, 5000))
        return
    if sys.argv[1:] == ["orops"]:
        run_set("orops_6k", 6000, 900, orops_queries(random.Random(20260931), 240, 120, 6000), seed=11)
        return
    if sys.argv[1:] == ["ops"]:  # only the fixtures added after round 1's first batch
        run_set("ops_6k", 6000, 900, ops_queries(random.Random(20260924), 240, 200, 6000), seed=11)
        run_set("scale_6k", 6000, 900, scale_queries(random.Random(20260925), 200, 200, 6000), seed=11)
        run_set("regimes_6k", 6000, 900, regime_queries(random.Random(20260926), 300, 120, 6000), seed=11, values=True)
        run_set("wqf_6k", 6000, 900, wqf_queries(random.Random(20260927), 150, 150, 6000), seed=11)
        run_set("sortmodes_6k", 6000, 900, sortmode_queries(random.Random(20260928), 200, 100, 6000), seed=11, values=True)
        run_set("bm25_6k", 6000, 900, bm25_queries(random.Random(20260929), 200, 150, 6000), seed=11)
        return
    rng = random.Random(20260923)
    # C1: BASELINE config 1 — 1k docs / 100 terms, every single term top-10, plus mixed shapes
    c1 = [dict(op="AND", terms=[t], first=0, maxitems=10, check_at_least=0) for t in range(100)]
    c1 += mixed(rng, 60, 100, 1000, 50)
    run_set("c1_1k_100", 1000, 100, c1)
    run_set("mid_20k", 20000, 5000, mixed(rng, 120, 400, 20000, 200))
    # Xapiand two-phase scheme over 4 interleaved shards (handler.cc:1485-1551)
    sh = []
    for i in range(60):
        op = "AND" if i % 2 == 0 else "OR"
        k = 3 if op == "AND" else 4
        sh.append(dict(op=op, terms=rng.sample(range(300), k), first=rng.choice([0, 0, 5]), maxitems=rng.choice([10, 100]),
                       check_at_least=rng.choice([0, 20000])))
    run_set("shard4_20k", 20000, 5000, sh, nshards=4, twophase=True)
    run_set("shard2_20k", 20000, 5000, sh[:30], nshards=2, twophase=True)
    # value range filter + sort by value then relevance (stock OP_VALUE_RANGE / set_sort_by_value_then_relevance)
    vq = []
    for i in range(60):
        lo = rng.randrange(0, 900000)
        q = dict(op="AND", terms=rng.sample(range(60), 2), first=0, maxitems=rng.choice([10, 100]),
                 check_at_least=rng.choice([0, 5000]), vr=[0, lo, lo + rng.choice([10000, 100000, 400000])])
        if i % 3 != 2:
            q["sort"] = [1, rng.choice([0, 1])]
        vq.append(q)
    run_set("values_5k", 5000, 2000, vq, values=True)
    run_set("ops_6k", 6000, 900, ops_queries(random.Random(20260924), 240, 200, 6000), seed=11)
    run_set("scale_6k", 6000, 900, scale_queries(random.Random(20260925), 200, 200, 6000), seed=11)
    run_set("regimes_6k", 6000, 900, regime_queries(random.Random(20260926), 300, 120, 6000), seed=11, values=True)
    run_set("wqf_6k", 6000, 900, wqf_queries(random.Random(20260927), 150, 150, 6000), seed=11)
    run_set("sortmodes_6k", 6000, 900, sortmode_queries(random.Random(20260928), 200, 100, 6000), seed=11, values=True)
    run_set("bm25_6k", 6000, 900, bm25_queries(random.Random(20260929), 200, 150, 6000), seed=11)
    run_mv_set("multivalue_5k", 5000, 2000, mv_queries(random.Random(20260930), 240, 60, 5000))
    run_set("orops_6k", 6000, 900, orops_queries(random.Random(20260931), 240, 120, 6000), seed=11)
    run_glass_sets()


if __name__ == "__main__":
    main()
