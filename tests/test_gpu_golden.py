"""GPU tests against the golden fixtures the COMPILED REFERENCE produced (tests/golden/*.json)."""
import struct

import numpy as np
import pytest

from tests.golden_util import load, sortable_key_to_int
from xapiand_b200 import xgm

pytestmark = pytest.mark.gpu


def bits(x):
    return struct.pack("<d", float(x))


def x_query(q, stats=None, first=None, maxitems=None):
    kw = dict(first=q["first"] if first is None else first, maxitems=q["maxitems"] if maxitems is None else maxitems,
              check_at_least=q["check_at_least"], stats=stats)
    if "vr" in q:
        kw.update(filter=xgm.FILTER_VALUE_RANGE, filter_slot=0, range_lo=q["vr"][1], range_hi=q["vr"][2])
    if "sort" in q:
        kw.update(sort_by=xgm.SORT_VAL_REL, sort_slot=q["sort"][0], sort_reverse=bool(q["sort"][1]))
    return xgm.Query(xgm.OP_AND if q["op"] == "AND" else xgm.OP_OR, q["terms"], **kw)


def check(m, q, ctx, counts=True):
    assert m.status == 0, ctx
    assert list(m.docids) == q["docids"], f"{ctx}: docids"
    assert all(bits(a) == bits(b) for a, b in zip(m.weights, q["weights"])), f"{ctx}: weights not bit-equal"
    assert bits(m.max_attained) == bits(q["max_attained"]), f"{ctx}: max_attained"
    if counts:
        assert bits(m.max_possible) == bits(q["max_possible"]), f"{ctx}: max_possible"
        assert m.matches_upper_bound == q["ub"], f"{ctx}: upper bound"
        if not (m.flags & 1):
            assert (m.matches_lower_bound, m.get_matches_estimated()) == (q["lb"], q["est"]), f"{ctx}: bounds"


@pytest.mark.parametrize("tag", ["c1_1k_100", "mid_20k"])
def test_cuda_matches_reference_single_db(tag):
    fx = load(tag)
    ix = xgm.Index.synthetic(fx["ndocs"], fx["vocab"], fx["seed"])
    s = xgm.Searcher(ix, max_batch=len(fx["queries"]), max_topk=256)
    res = s.search([x_query(q) for q in fx["queries"]])
    for i, (q, m) in enumerate(zip(fx["queries"], res)):
        check(m, q, f"{tag}[{i}] {q['op']} {q['terms']}")


@pytest.mark.parametrize("tag", ["shard4_20k", "shard2_20k"])
def test_cuda_matches_reference_twophase_shards(tag):
    """Xapiand's DocMatcher scheme: per-shard search with global statistics, unshard, merge."""
    fx = load(tag)
    n = fx["nshards"]
    shards = [xgm.Index.synthetic(fx["ndocs"], fx["vocab"], fx["seed"], nshards=n, shard=s) for s in range(n)]
    infos = [ix.info() for ix in shards]
    coll = sum(i.doccount for i in infos)
    tlen = sum(i.total_length for i in infos)
    searchers = [xgm.Searcher(ix, max_batch=len(fx["queries"]), max_topk=256) for ix in shards]
    per_shard = []
    gstats = []
    for q in fx["queries"]:
        gtf = [sum(ix.term_stats(f"T{t:06d}").termfreq for ix in shards) for t in q["terms"]]
        gstats.append((coll, tlen, gtf))
    for si, s in enumerate(searchers):
        res = s.search([x_query(q, stats=gstats[i], first=0, maxitems=q["first"] + q["maxitems"])
                        for i, q in enumerate(fx["queries"])])
        for m in res:
            m.docids = xgm.unshard(m.docids, si, n)
        per_shard.append(res)
    for i, q in enumerate(fx["queries"]):
        merged = xgm.merge_msets([per_shard[si][i] for si in range(n)], q["first"], q["maxitems"])
        check(merged, q, f"{tag}[{i}] {q}")


def test_cuda_matches_reference_value_filter_and_sort():
    fx = load("values_5k")
    ix = xgm.Index.synthetic(fx["ndocs"], fx["vocab"], fx["seed"], values=True)
    s = xgm.Searcher(ix, max_batch=len(fx["queries"]), max_topk=128)
    res = s.search([x_query(q) for q in fx["queries"]])
    for i, (q, m) in enumerate(zip(fx["queries"], res)):
        ctx = f"values[{i}] {q}"
        check(m, q, ctx, counts=False)
        if "sort" in q:
            keys = [sortable_key_to_int(k) for k in q.get("sort_keys", [])]
            mine = list(m.sort_keys)
            for a in range(len(keys) - 1):
                assert (keys[a] < keys[a + 1]) == (mine[a] < mine[a + 1]), ctx
                assert (keys[a] == keys[a + 1]) == (mine[a] == mine[a + 1]), ctx


def test_multi_range_filter_and_sort_variants_against_oracle():
    """Xapiand's MultipleValueRange semantics (src/multivalue/range.cc:351-368) and sort by the
    smallest / largest value of a multi-valued slot (keymaker.cc:67-92), against the oracle."""
    import random
    from oracle import oracle as O
    nd, V = 20000, 3000
    ix = xgm.Index.synthetic(nd, V, values=True)
    orc = O.Index.synthetic(nd, V, values=True)
    rng = random.Random(11)
    xq, oq = [], []
    for i in range(120):
        terms = rng.sample(range(80), 2)
        lo = rng.randrange(0, 950000)
        hi = lo + rng.choice([5000, 50000, 300000])
        use_max = bool(i % 2)
        rev = bool((i // 2) % 2)
        sort = i % 3 != 0
        cal = rng.choice([0, nd])
        xq.append(xgm.Query(xgm.OP_AND, terms, maxitems=rng.choice([10, 100]), check_at_least=cal,
                            filter=xgm.FILTER_MULTI_RANGE, filter_slot=0, range_lo=lo, range_hi=hi,
                            sort_by=xgm.SORT_VAL_REL if sort else xgm.SORT_REL, sort_slot=0, sort_reverse=rev,
                            sort_use_max=use_max))
        oq.append(O.Query(op=O.OP_AND, terms=terms, maxitems=xq[-1].maxitems, check_at_least=cal,
                          filter=O.FILTER_MULTI_RANGE, range_lo=lo, range_hi=hi,
                          sort_by=O.SORT_VAL_REL if sort else O.SORT_REL, sort_slot=2 if use_max else 0, sort_reverse=rev))
    s = xgm.Searcher(ix, max_batch=len(xq), max_topk=128)
    res = s.search(xq)
    for i, (m, q) in enumerate(zip(res, oq)):
        ref = orc.match(q)
        ctx = f"multi[{i}] {xq[i]}"
        assert m.status == 0, ctx
        assert list(m.docids) == list(ref.docids), ctx
        assert np.asarray(m.weights).tobytes() == np.asarray(ref.weights).tobytes(), ctx
        assert m.exact_matches == ref.exact, ctx
        assert bits(m.max_attained) == bits(ref.max_attained), ctx
        if q.sort_by != O.SORT_REL:
            assert list(m.sort_keys) == list(ref.sortvals), ctx


class _CudaArray:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def test_device_merge_matches_reference_twophase():
    """The multi-GPU data path on one GPU: per-shard device results are concatenated exactly as an
    all-gather would lay them out ([part][query][rank]) and merged by xgm_merge_topk_device (unshard +
    Matcher::merge_mset order); checked against the reference's own two-phase run over 4 shards."""
    import torch
    fx = load("shard4_20k")
    n = fx["nshards"]
    qs = [q for q in fx["queries"] if q["first"] == 0]  # the device merge keeps ranks [0, k)
    K = 128
    shards = [xgm.Index.synthetic(fx["ndocs"], fx["vocab"], fx["seed"], nshards=n, shard=s) for s in range(n)]
    infos = [ix.info() for ix in shards]
    coll = sum(i.doccount for i in infos)
    tlen = sum(i.total_length for i in infos)
    nq = len(qs)
    gw, gd, gc, slabs = [], [], [], []
    searchers = []
    for si, ix in enumerate(shards):
        s = xgm.Searcher(ix, max_batch=nq, max_topk=K)
        searchers.append(s)
        batch = []
        for q in qs:
            gtf = [sum(x.term_stats(f"T{t:06d}").termfreq for x in shards) for t in q["terms"]]
            batch.append(x_query(q, stats=(coll, tlen, gtf), first=0, maxitems=q["maxitems"]))
        s.search(batch)
        wptr, dptr, cptr, stride = s.device_results()
        assert stride == K
        gw.append(torch.as_tensor(_CudaArray(wptr, (nq * K,), "<f8"), device="cuda").clone())
        gd.append(torch.as_tensor(_CudaArray(dptr, (nq * K,), "<u4"), device="cuda").view(torch.int32).clone())
        gc.append(torch.as_tensor(_CudaArray(cptr, (nq * 8,), "<u4"), device="cuda").view(torch.int32).clone())
        base, nbytes, off_d, off_c, sstride = s.device_slab()
        assert sstride == K and base == wptr and base + off_d == dptr and base + off_c == cptr
        slabs.append(torch.as_tensor(_CudaArray(base, (nbytes,), "|u1"), device="cuda").clone())
    W, D, Cn = torch.cat(gw), torch.cat(gd), torch.cat(gc)
    ow = torch.zeros(nq * K, dtype=torch.float64, device="cuda")
    od = torch.zeros(nq * K, dtype=torch.int32, device="cuda")
    on = torch.zeros(nq, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    st = xgm.lib().xgm_merge_topk_device(W.data_ptr(), D.data_ptr(), Cn.data_ptr(), n, nq, K, K, ow.data_ptr(),
                                         od.data_ptr(), on.data_ptr(), None)
    assert st == 0, xgm.lib().xgm_last_error()
    torch.cuda.synchronize()
    # the same merge over whole result slabs, as one all-gather lays them out
    G = torch.cat(slabs)
    ow2, od2, on2 = torch.zeros_like(ow), torch.zeros_like(od), torch.zeros_like(on)
    st = xgm.lib().xgm_merge_topk_device_slab(G.data_ptr(), nbytes, off_d, off_c, n, nq, K, K, ow2.data_ptr(),
                                              od2.data_ptr(), on2.data_ptr(), None)
    assert st == 0, xgm.lib().xgm_last_error()
    torch.cuda.synchronize()
    assert torch.equal(on, on2)
    for i in range(nq):
        c = int(on[i])
        assert torch.equal(od[i * K:i * K + c], od2[i * K:i * K + c]) and torch.equal(ow[i * K:i * K + c], ow2[i * K:i * K + c])
    ow, od, on = ow.cpu().numpy().reshape(nq, K), od.cpu().numpy().view(np.uint32).reshape(nq, K), on.cpu().numpy()
    for i, q in enumerate(qs):
        m = q["maxitems"]
        got_n = min(int(on[i]), m)
        assert got_n == len(q["docids"]), f"merge[{i}]"
        assert list(od[i, :got_n]) == q["docids"], f"merge[{i}] docids"
        assert all(bits(a) == bits(b) for a, b in zip(ow[i, :got_n], q["weights"])), f"merge[{i}] weights"


def test_cuda_matches_reference_filter_andnot_andmaybe():
    """SURVEY.md §8(f)-1 on the device: OP_FILTER with boolean terms, OP_AND_NOT
    and OP_AND_MAYBE around an AND base against the compiled reference's MSets (ops_6k fixture)."""
    fx = load("ops_6k")
    ix = xgm.Index.synthetic(fx["ndocs"], fx["vocab"], fx["seed"])
    name = lambda t: f"T{t:06d}"
    qs = [xgm.Query(xgm.OP_AND, [name(t) for t in q["terms"]], first=q["first"], maxitems=q["maxitems"],
                    check_at_least=q["check_at_least"], filter_terms=[name(t) for t in q["filter_terms"]],
                    not_terms=[name(t) for t in q["not_terms"]], maybe_terms=[name(t) for t in q["maybe_terms"]])
          for q in fx["queries"]]
    res = xgm.Searcher(ix, max_batch=len(qs), max_topk=256).search(qs)
    checked = 0
    for i, (q, m) in enumerate(zip(fx["queries"], res)):
        ctx = f"ops[{i}] {q['terms']} F{q['filter_terms']} N{q['not_terms']} M{q['maybe_terms']}"
        assert m.status == 0, ctx
        assert list(m.docids) == q["docids"], ctx
        assert all(bits(a) == bits(b) for a, b in zip(m.weights, q["weights"])), ctx
        assert bits(m.max_possible) == bits(q["max_possible"]) and bits(m.max_attained) == bits(q["max_attained"]), ctx
        assert m.matches_upper_bound == q["ub"], ctx
        if not (m.flags & 1):
            assert (m.matches_lower_bound, m.get_matches_estimated()) == (q["lb"], q["est"]), ctx
        checked += 1
    assert checked == len(qs)


def test_cuda_matches_reference_groups_around_or_base():
    """OP_FILTER with boolean terms and OP_AND_NOT around an OR base (a free-text OR restricted / thinned by
    boolean terms) against the compiled reference's MSets (orops_6k); optional leaves on an OR base are declined."""
    fx = load("orops_6k")
    ix = xgm.Index.synthetic(fx["ndocs"], fx["vocab"], fx["seed"])
    name = lambda t: f"T{t:06d}"
    qs = [xgm.Query(xgm.OP_OR, [name(t) for t in q["terms"]], first=q["first"], maxitems=q["maxitems"],
                    check_at_least=q["check_at_least"], filter_terms=[name(t) for t in q["filter_terms"]],
                    not_terms=[name(t) for t in q["not_terms"]], maybe_terms=[name(t) for t in q["maybe_terms"]])
          for q in fx["queries"]]
    res = xgm.Searcher(ix, max_batch=len(qs), max_topk=256).search(qs)
    served = 0
    for i, (q, m) in enumerate(zip(fx["queries"], res)):
        ctx = f"orops[{i}] {q['terms']} F{q['filter_terms']} N{q['not_terms']} M{q['maybe_terms']}"
        if q["maybe_terms"]:
            assert m.status == xgm.E_UNIMPLEMENTED, ctx
            continue
        assert m.status == 0, ctx
        assert list(m.docids) == q["docids"], ctx
        assert all(bits(a) == bits(b) for a, b in zip(m.weights, q["weights"])), ctx
        assert bits(m.max_possible) == bits(q["max_possible"]) and bits(m.max_attained) == bits(q["max_attained"]), ctx
        assert m.matches_upper_bound == q["ub"], ctx
        if not (m.flags & 1):
            assert (m.matches_lower_bound, m.get_matches_estimated()) == (q["lb"], q["est"]), ctx
        served += 1
    assert served >= 120


@pytest.mark.parametrize("tag", ["wqf_6k", "bm25_6k", "regimes_6k", "sortmodes_6k", "scale_6k"])
def test_cuda_matches_reference_more_regimes(tag):
    """The fixtures added late in round 1 (within-query frequencies, non-default BM25 parameters, intermediate
    check_at_least / first, the three value-sort modes, OP_SCALE_WEIGHT factors) on the device."""
    from oracle import oracle as O
    fx = load(tag)
    ix = xgm.Index.synthetic(fx["ndocs"], fx["vocab"], fx["seed"], values=fx["values"])
    name = lambda t: f"T{t:06d}"
    qs, keep = [], []
    for q in fx["queries"]:
        kw = dict(first=q["first"], maxitems=q["maxitems"], check_at_least=q["check_at_least"])
        if q.get("wqf"):
            kw["wqf"] = q["wqf"]
        if q.get("factors"):
            kw["factors"] = q["factors"]
        if q.get("bm25"):
            if not any(q["bm25"]):
                continue  # all-zero parameters mean "defaults" at the C-ABI
            kw["bm25"] = q["bm25"]
        if q.get("sort"):
            mode = {0: xgm.SORT_VAL_REL, 1: xgm.SORT_VAL, 2: xgm.SORT_REL_VAL}[q.get("sort_mode", 0)]
            kw.update(sort_by=mode, sort_slot=q["sort"][0], sort_reverse=bool(q["sort"][1]))
        qs.append(xgm.Query(xgm.OP_AND if q["op"] == "AND" else xgm.OP_OR, [name(t) for t in q["terms"]], **kw))
        keep.append(q)
    res = xgm.Searcher(ix, max_batch=len(qs), max_topk=256).search(qs)
    declined = 0
    for i, (q, m) in enumerate(zip(keep, res)):
        ctx = f"{tag}[{i}] {q}"
        if m.status == xgm.E_UNIMPLEMENTED and q.get("factors") and q["op"] == "OR" and 0.0 in q["factors"]:
            declined += 1
            continue
        assert m.status == 0, ctx
        assert list(m.docids) == q["docids"], ctx
        assert all(bits(a) == bits(b) for a, b in zip(m.weights, q["weights"])), ctx
        assert bits(m.max_possible) == bits(q["max_possible"]) and bits(m.max_attained) == bits(q["max_attained"]), ctx
        assert m.matches_upper_bound == q["ub"], ctx
        if not (m.flags & 1):
            assert (m.matches_lower_bound, m.get_matches_estimated()) == (q["lb"], q["est"]), ctx
        if not (q["op"] == "OR" and q.get("sort")):  # OR + value sort: percent scale is a documented approximation
            assert [O.convert_to_percent(w, m.percent_scale_factor) for w in m.weights] == q["percents"], ctx
    assert declined < len(keep) // 4



def _check_multivalue(ix, fx, revision):
    from oracle import oracle as O
    key = lambda v: xgm.value_key(bytes.fromhex(fx["serialised"][str(v)]))[0]
    qs = []
    for q in fx["queries"]:
        kw = dict(first=q["first"], maxitems=q["maxitems"], check_at_least=q["check_at_least"], revision=revision)
        if "mvr" in q:
            kw.update(filter=xgm.FILTER_MULTI_RANGE, filter_slot=q["mvr"][0], range_lo=key(q["mvr"][1]),
                      range_hi=key(q["mvr"][2]), filter_weighted=bool(q["mvr"][3]))
        if "keysort" in q:
            slot, rev = q["keysort"]
            kw.update(sort_by=xgm.SORT_VAL_REL, sort_slot=slot, sort_reverse=bool(rev), sort_use_max=bool(rev),
                      sort_missing_key=xgm.value_key(b"" if rev else b"\xff")[0])
        qs.append(xgm.Query(xgm.OP_AND, [f"T{t:06d}" for t in q["terms"]], **kw))
    res = xgm.Searcher(ix, max_batch=len(qs), max_topk=128).search(qs)
    exact_bounds = 0
    for i, (q, m) in enumerate(zip(fx["queries"], res)):
        ctx = f"mv[{i}] {q['terms']} mvr={q.get('mvr')} keysort={q.get('keysort')}"
        check(m, q, ctx)
        exact_bounds += not (m.flags & 1)
        if "keysort" in q:
            got = [xgm.sort_key_bytes(int(k), bool(q["keysort"][1])).hex() for k in m.sort_keys]
            assert got == q.get("sort_keys", []), ctx
        mine = [O.convert_to_percent(w, m.percent_scale_factor) for w in m.weights]
        assert mine == q["percents"], ctx
    assert exact_bounds >= len(qs) * 3 // 4


def test_cuda_matches_xapiand_multivalue_classes():
    """SURVEY.md §8 rows a15 / a16 against Xapiand's REAL classes (multivalue_5k fixture: src/multivalue/range.cc,
    keymaker.cc, serialise_list.h, sortable_serialise.cc compiled from the reference).  The index is built from the
    slot bytes exactly as Xapiand stores them (xgm_builder_add_value_slot_serialised); range bounds and the
    missing-value keys go in as value keys of the reference's serialised bytes; MSetIterator::get_sort_key bytes are
    rebuilt from the device's keys (xgm_sort_key_bytes) and must equal Multi_MultiValueKeyMaker's."""
    from oracle import oracle as O
    fx = load("multivalue_5k")
    orc = O.Index.synthetic(fx["ndocs"], fx["vocab"], fx["seed"])  # the corpus' postings only
    terms = [(orc.name(t),) + tuple(orc.postings(t)) for t in range(orc.nterms)]
    last = orc.lastdocid
    slots = {int(s): [bytes.fromhex(fx["slots"][s].get(str(d), "")) for d in range(last + 1)] for s in fx["slots"]}
    ix = xgm.Index.from_postings(orc.doclen(), terms, serialised_slots=slots, revision=7)
    assert ix.info().revision == 7
    _check_multivalue(ix, fx, 7)
    # a query that names another revision is refused with XGM_E_STALE (→ Xapian::DatabaseModifiedError)
    stale = xgm.Searcher(ix, max_batch=1, max_topk=16).search([xgm.Query(xgm.OP_AND, ["T000001"], revision=8)])
    assert stale[0].status == xgm.E_STALE


def test_direct_glass_reader_index_matches_xapiand_multivalue_classes():
    """SURVEY.md section 8(b) / (f)-3: xgm_index_open reads the glass directory itself (iamglass + the postlist B-tree:
    posting chunks, document lengths, value streams) — the same fixture as above must come out of an index built that
    way from the database the reference wrote, carrying the database's own revision.  The database is
    tests/golden/glass/mvalues_sparse_1500.tar.xz, the reference's MSets on it multivalue_1500.json."""
    import ctypes
    import shutil
    import tempfile
    from tests.golden_util import glass_databases, glass_db
    fx = load("multivalue_1500")
    built = glass_databases()["mvalues_sparse_1500"]
    assert (built["ndocs"], built["vocab"], built["seed"], built["sparse"]) == (fx["ndocs"], fx["vocab"], fx["seed"], fx["sparse"])
    tmp = tempfile.mkdtemp(prefix="xgm_glass_")
    try:
        db = glass_db("mvalues_sparse_1500", tmp + "/db")
        rev = ctypes.c_uint64()
        assert xgm.lib().xgm_glass_revision(db.encode(), ctypes.byref(rev), None, None) == 0
        ix = xgm.Index.open_glass(db)
        assert ix.info().revision == rev.value and ix.info().doccount == fx["ndocs"]
        _check_multivalue(ix, fx, rev.value)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
