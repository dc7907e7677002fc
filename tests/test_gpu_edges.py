"""GPU edge cases: hand-made indexes (docid gaps, boolean wdf=0 terms, huge wdf, partial blocks, block
boundaries, terms absent from the index), degenerate get_mset arguments, and the glass → public
iterators → HBM data path against the compiled reference."""
import os
import random
import shutil
import tempfile

import numpy as np
import pytest

from oracle import oracle as O
from tests.flatfile import write_flat
from tests.util import assert_mset_equal
from xapiand_b200 import xgm

pytestmark = pytest.mark.gpu


def make_edge_index(tmp, seed=3):
    rng = np.random.default_rng(seed)
    lastdocid = 9000
    doclen = np.zeros(lastdocid + 1, np.uint32)
    alive = np.sort(rng.choice(np.arange(1, lastdocid + 1), size=7000, replace=False))  # docid gaps
    doclen[alive] = rng.integers(1, 400, size=len(alive))
    terms = []
    def add(name, k, wmax, wzero=False):
        d = np.sort(rng.choice(alive, size=k, replace=False)).astype(np.uint32)
        w = np.zeros(k, np.uint32) if wzero else rng.integers(1, wmax + 1, size=k).astype(np.uint32)
        terms.append((name, d, w))
    add("a127", 127, 3); add("b128", 128, 3); add("c129", 129, 3); add("d1", 1, 5); add("e256", 256, 2)
    add("f_all", len(alive), 4); add("g_bool", 900, 1, wzero=True); add("h_bigwdf", 500, 70000)
    add("i_mid", 3000, 6); add("j_mid", 2500, 6); add("k_rare", 40, 2); add("l_half", 3500, 9)
    # consecutive docids (zero-bit deltas) and one huge gap
    d = np.concatenate([alive[:300], alive[-5:]]).astype(np.uint32)
    terms.append(("m_runs", d, np.ones(len(d), np.uint32)))
    terms.sort(key=lambda t: t[0])
    # a document's length is the sum of its wdfs (plus terms not modelled here): the reference's
    # get_maxpart bound (bm25weight.cc:183-207) relies on doclen >= wdf
    total = np.zeros(lastdocid + 1, np.uint64)
    for _, d, w in terms:
        total[d] += w
    doclen[alive] = (total[alive] + rng.integers(1, 400, size=len(alive)).astype(np.uint64)).astype(np.uint32)
    path = os.path.join(tmp, "edge.flat")
    write_flat(path, doclen, terms)
    return path, [t[0] for t in terms]


@pytest.fixture(scope="module")
def edge():
    tmp = tempfile.mkdtemp(prefix="xgm_edge_")
    path, names = make_edge_index(tmp)
    ix = xgm.Index.load_flat(path)
    orc = O.Index.load_flat(path)
    yield ix, orc, names
    shutil.rmtree(tmp, ignore_errors=True)


def test_edge_roundtrip(edge):
    ix, orc, names = edge
    for t, nm in enumerate(names):
        d, w = ix.decode_term(t)
        rd, rw = orc.postings(t)
        assert np.array_equal(d, rd) and np.array_equal(w, rw), nm
        assert ix.term_stats(nm).term_id == t


def test_edge_queries_all_pairs(edge):
    ix, orc, names = edge
    rng = random.Random(4)
    xq, oq = [], []
    n = len(names)
    for i in range(n):
        for j in range(n):
            if i == j:
                continue
            for op in ("AND", "OR"):
                mi = rng.choice([1, 10, 100])
                cal = rng.choice([0, 0, 9000])
                first = rng.choice([0, 0, 2])
                xq.append(xgm.Query(xgm.OP_AND if op == "AND" else xgm.OP_OR, [names[i], names[j]], first=first,
                                    maxitems=mi, check_at_least=cal))
                oq.append(O.Query(op=O.OP_AND if op == "AND" else O.OP_OR, terms=[i, j], first=first, maxitems=mi,
                                  check_at_least=cal))
    for t in range(n):
        xq.append(xgm.Query(xgm.OP_AND, [names[t]], maxitems=50))
        oq.append(O.Query(op=O.OP_AND, terms=[t], maxitems=50))
    for _ in range(60):
        k = rng.choice([3, 4, 6])
        ts = rng.sample(range(n), k)
        op = rng.choice(["AND", "OR"])
        xq.append(xgm.Query(xgm.OP_AND if op == "AND" else xgm.OP_OR, [names[t] for t in ts], maxitems=30))
        oq.append(O.Query(op=O.OP_AND if op == "AND" else O.OP_OR, terms=ts, maxitems=30))
    s = xgm.Searcher(ix, max_batch=len(xq), max_topk=128)
    res = s.search(xq)
    for i, (m, q) in enumerate(zip(res, oq)):
        ref = orc.match(q)
        assert_mset_equal(m, ref, ctx=f"edge[{i}] {xq[i].terms} op={xq[i].op}", check_counts=not (m.flags & 1))


def test_degenerate_arguments(edge):
    ix, orc, names = edge
    s = xgm.Searcher(ix, max_batch=8, max_topk=64)
    t = names.index("i_mid")
    u = names.index("j_mid")
    cases = [dict(first=0, maxitems=0, check_at_least=0),      # bounds only (matcher.cc:437-461)
             dict(first=0, maxitems=0, check_at_least=50),     # nothing kept but matches counted
             dict(first=40, maxitems=10, check_at_least=0),
             dict(first=100000, maxitems=10, check_at_least=0),  # first beyond the collection
             dict(first=0, maxitems=60, check_at_least=100000)]
    for c in cases:
        m = s.search([xgm.Query(xgm.OP_AND, [names[t], names[u]], **c)])[0]
        ref = orc.match(O.Query(op=O.OP_AND, terms=[t, u], **c))
        assert m.status == 0
        assert list(m.docids) == list(ref.docids), c
        if m.flags & 1:  # pruned / large match set: conservative but valid bounds
            assert m.matches_lower_bound <= ref.lb and m.matches_upper_bound == ref.ub, c
        else:
            assert (m.matches_lower_bound, m.matches_estimated_raw, m.matches_upper_bound) == (ref.lb, ref.est, ref.ub), c
    # OR with an absent leaf behaves like the OR of the others; AND with an absent leaf is empty
    m = s.search([xgm.Query(xgm.OP_AND, [names[t], "zzz_absent"], maxitems=10)])[0]
    assert m.size() == 0 and m.status == 0


def test_unsupported_shapes_are_declined_not_guessed(edge):
    ix, orc, names = edge
    s = xgm.Searcher(ix, max_batch=4, max_topk=16)
    too_many = [names[i % len(names)] + ("" if i < len(names) else "x") for i in range(17)]
    r = s.search([xgm.Query(xgm.OP_AND, too_many, maxitems=5)])[0]
    assert r.status == xgm.E_UNIMPLEMENTED
    r = s.search([xgm.Query(xgm.OP_AND, [names[0], names[0]], maxitems=5)])[0]   # repeated leaf
    assert r.status == xgm.E_UNIMPLEMENTED
    r = s.search([xgm.Query(7, [names[0]], maxitems=5)])[0]                        # unknown operator
    assert r.status == xgm.E_UNIMPLEMENTED


def test_glass_db_through_public_iterators_matches_reference():
    """Drop-in data path: a glass DB written by the reference → `ref_runner export` (Database::allterms_begin /
    postlist_begin / get_doclength, INTEGRATION.md §1) → xgm_index_load_flat → same MSets as the
    reference's Enquire::get_mset on that very DB (tests/golden/glass_6k.json).  The export is the flat file of
    the seeded corpus the DB was built from; it is rewritten here and must match the reference's export (size
    and SHA-256) before it is loaded."""
    import hashlib
    import json
    from tests.golden_util import GOLDEN
    with open(os.path.join(GOLDEN, "glass_6k.json")) as f:
        fx = json.load(f)
    orc = O.Index.synthetic(fx["ndocs"], fx["vocab"], seed=fx["seed"])
    tmp = tempfile.mkdtemp(prefix="xgm_glass_")
    try:
        flat = os.path.join(tmp, "db.flat")
        write_flat(flat, orc.doclen(), [(orc.name(t),) + tuple(orc.postings(t)) for t in range(orc.nterms)])
        data = open(flat, "rb").read()
        assert (len(data), hashlib.sha256(data).hexdigest()) == (fx["export_bytes"], fx["export_sha256"])
        ix = xgm.Index.load_flat(flat)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    qs = [xgm.Query(xgm.OP_AND if q["op"] == "AND" else xgm.OP_OR, [f"T{r:06d}" for r in q["terms"]],
                    maxitems=q["maxitems"], check_at_least=q["check_at_least"]) for q in fx["queries"]]
    s = xgm.Searcher(ix, max_batch=len(qs), max_topk=128)
    for i, (m, r) in enumerate(zip(s.search(qs), fx["queries"])):
        ctx = f"glass[{i}] {r['op']} {r['terms']} maxitems={r['maxitems']} check_at_least={r['check_at_least']}"
        assert m.status == 0
        assert list(m.docids) == r["docids"], ctx
        assert hashlib.sha256(np.asarray(m.weights, "<f8").tobytes()).hexdigest() == r["weights_sha256"], f"{ctx}: weights"
        assert float(m.max_possible).hex() == r["max_possible"]
        assert float(m.max_attained).hex() == r["max_attained"]
        assert m.matches_upper_bound == r["ub"]
        if not (m.flags & 1):
            assert (m.matches_lower_bound, m.get_matches_estimated()) == (r["lb"], r["est"]), ctx


def test_background_submit_matches_synchronous(edge):
    """xgm_search_submit_async: planning + launches on the searcher's worker thread; same MSets, two
    searchers in flight, and a second submit before wait is refused."""
    ix, orc, names = edge
    rng = random.Random(8)
    batches = []
    for b in range(4):
        qs = []
        for _ in range(600):  # >= 512 queries: the threaded planner runs inside the worker
            ts = rng.sample(range(len(names)), rng.choice([1, 2, 3]))
            qs.append(xgm.Query(rng.choice([xgm.OP_AND, xgm.OP_OR]), [names[t] for t in ts], maxitems=rng.choice([5, 40])))
        batches.append(xgm.QueryBatch(qs))
    s0 = xgm.Searcher(ix, max_batch=600, max_topk=64)
    s1 = xgm.Searcher(ix, max_batch=600, max_topk=64)
    sync = [s0.search(b) for b in batches]
    got = [None] * 4
    s0.submit(batches[0], background=True)
    s1.submit(batches[1], background=True)
    with pytest.raises(xgm.XgmError):
        s0.submit(batches[2], background=True)
    s0.launched()
    got[0] = s0.wait()
    s0.submit(batches[2], background=True)
    got[1] = s1.wait()
    s1.submit(batches[3], background=True)
    got[2] = s0.wait()
    got[3] = s1.wait()
    for b in range(4):
        for i, (a, m) in enumerate(zip(sync[b], got[b])):
            assert a.status == m.status and list(a.docids) == list(m.docids), (b, i)
            assert [float(x).hex() for x in a.weights] == [float(x).hex() for x in m.weights], (b, i)
            assert (a.matches_lower_bound, a.matches_estimated_raw, a.matches_upper_bound) == \
                   (m.matches_lower_bound, m.matches_estimated_raw, m.matches_upper_bound), (b, i)


def test_process_exits_after_a_large_batch():
    """Batches of >= 512 queries are planned on the library's helper threads, which stay parked for the life of
    the process: the host program must still exit (a static pool object whose condition variable was destroyed
    at exit() once blocked every Python process that had submitted a large batch)."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, {root!r})\n"
            "from xapiand_b200 import xgm\n"
            "ix = xgm.Index.synthetic(20000, 3000)\n"
            "s = xgm.Searcher(ix, max_batch=640, max_topk=16)\n"
            "r = s.search([xgm.Query(xgm.OP_AND, [i % 50, 50 + i % 40], maxitems=10) for i in range(600)])\n"
            "print(sum(m.status == 0 for m in r))\n").format(root=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=180)
    assert p.returncode == 0 and p.stdout.strip() == "600", p.stderr[-500:]
