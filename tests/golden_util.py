"""Load golden fixtures (written by tests/golden/make_golden.py from the compiled reference)."""
import json
import os

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(tag):
    with open(os.path.join(GOLDEN, f"{tag}.json")) as f:
        fx = json.load(f)
    for q in fx["queries"]:
        q["weights"] = [float.fromhex(w) for w in q["weights"]]
        q["max_possible"] = float.fromhex(q["max_possible"])
        q["max_attained"] = float.fromhex(q["max_attained"])
    return fx


def glass_databases():
    """tests/golden/glass/databases.json: how each stored database was built and the size and SHA-256 of the flat
    file the reference's `ref_runner export` wrote from it."""
    with open(os.path.join(GOLDEN, "glass", "databases.json")) as f:
        return json.load(f)


def glass_db(tag, dest):
    """Unpack the glass database the reference wrote (tests/golden/glass/<tag>.tar.xz) into dest; returns dest."""
    import tarfile
    with tarfile.open(os.path.join(GOLDEN, "glass", f"{tag}.tar.xz")) as tar:
        tar.extractall(dest, filter="data")
    return dest


def sortable_key_to_int(hexkey: str) -> int:
    """Invert Xapian::sortable_serialise for the non-negative integers the fixtures use.
    Positive x = m * 2^e is stored as 0b11 [large-exponent bit, 3-bit or 10-bit exponent] mantissa..
    (src/xapian/api/sortable-serialise.cc); decoding is only needed to compare sort order, so we map the
    byte string to an integer that preserves order instead: zero-padded big-endian bytes."""
    if hexkey == "-":
        return 0
    b = bytes.fromhex(hexkey)
    return int.from_bytes(b.ljust(10, b"\0"), "big")


def fixture_query_line(q) -> str:
    """The oracle/ref_runner query line of a fixture entry (what tests/golden/make_golden.py fed the reference)."""
    from oracle import oracle as O
    name = lambda r: f"T{r:06d}"
    facs, wq = q.get("factors"), q.get("wqf")
    tnames = [name(t) + ("" if not wq or wq[j] == 1 else f"#{wq[j]}") +
              ("" if not facs or facs[j] == 1.0 else f"^{facs[j]!r}") for j, t in enumerate(q["terms"])]
    return O.query_line("TERM" if len(q["terms"]) == 1 else q.get("op", "AND"), tnames, q["first"], q["maxitems"],
                        q["check_at_least"], vr=q.get("vr"),
                        sort=(q["sort"] + [q.get("sort_mode", 0)]) if q.get("sort") else None, bm25=q.get("bm25"),
                        filter_terms=[name(t) for t in q.get("filter_terms", [])],
                        not_terms=[name(t) for t in q.get("not_terms", [])],
                        maybe_terms=[name(t) for t in q.get("maybe_terms", [])],
                        mvr=q.get("mvr"), keysort=q.get("keysort"))
