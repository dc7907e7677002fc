"""CPU tests of the direct glass reader (xapiand_b200/csrc/xgm_glass.cu): `xgm_glass_export_flat` parses
iamglass + postlist.glass itself and must produce, byte for byte, the file `ref_runner export` writes by walking
the same database through the reference's public iterators (allterms / postlist / doclength / valuestream).
The databases were written by the reference (tests/golden/glass/); the size and SHA-256 of the reference's export
of each are stored next to them (tests/golden/make_golden.py glass)."""
import ctypes
import hashlib

import pytest

from tests.golden_util import glass_databases, glass_db
from xapiand_b200 import xgm

DATABASES = glass_databases()


@pytest.mark.parametrize("tag", sorted(DATABASES))
def test_direct_reader_equals_the_reference_iterators(tag, tmp_path):
    ref = DATABASES[tag]
    db = glass_db(tag, str(tmp_path / "db"))
    mine = tmp_path / "mine.flat"
    st = xgm.lib().xgm_glass_export_flat(db.encode(), str(mine).encode())
    assert st == 0, xgm.lib().xgm_last_error()
    data = mine.read_bytes()
    assert (len(data), hashlib.sha256(data).hexdigest()) == (ref["export_bytes"], ref["export_sha256"]), \
        "the export differs from the reference's"
    rev, dc, last = ctypes.c_uint64(), ctypes.c_uint32(), ctypes.c_uint32()
    assert xgm.lib().xgm_glass_revision(db.encode(), ctypes.byref(rev), ctypes.byref(dc), ctypes.byref(last)) == 0
    assert (dc.value, last.value) == (ref["ndocs"], ref["ndocs"]) and rev.value >= 1


def test_reader_rejects_what_is_not_a_glass_database(tmp_path):
    assert xgm.lib().xgm_glass_export_flat(str(tmp_path).encode(), str(tmp_path / "x").encode()) == xgm.E_IO
    (tmp_path / "iamglass").write_bytes(b"not a version file" * 4)
    assert xgm.lib().xgm_glass_export_flat(str(tmp_path).encode(), str(tmp_path / "x").encode()) == xgm.E_IO
