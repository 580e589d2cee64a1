"""search_memories ordering and paging on the device (PackedMemdir.sort_page -> fei_sort_rows) against the oracle listing sorted
by CPython exactly as the reference does (search.py:370-388): exact order, the whole result dicts, and the warning line of a sort
that raises.  Also fei_sort_rows itself on a synthetic corpus of a million records."""
import contextlib
import io
import os

import numpy as np
import pytest

from oracle import memdir_oracle as mo
from tests.memdir_util import build_tree

pytestmark = pytest.mark.gpu

FIELDS = ["Subject", "subject", "Priority", "Tags", "Status", "status", "state", "status_value", "filename", "folder", "id", "unique_id",
          "hostname", "flags", "date", "timestamp", "Due", "Created", "content", "NoSuchField"]
LIMITS = (None, 0, 1, 7)
LONG = "Quarterly planning notes for the infrastructure team, part "

# (folder, name, text): long shared prefixes, proper prefixes, NUL, non-ASCII (4-byte UTF-8 too), empty and absent values,
# duplicate-case keys, a Timestamp header, Due naive / tz-aware / unparseable / absent, timestamp ties
FIXTURE = [
    (".Sortfix", "1700000100.aa01.hosta:2,S", f"Subject: {LONG}one\nPriority: high\nDue: 2024-03-01\n---\nbody alpha"),
    (".Sortfix", "1700000100.aa02.hostb:2,", f"Subject: {LONG}one and more\nPriority: low\nDue: 2024-03-01\n---\nbody alpha two"),
    (".Sortfix", "1700000100.aa03.hosta:2,FS", f"Subject: {LONG}\npriority: High\nDue: 2023-12-31 23:59\n---\n"),
    (".Sortfix", "1700000200.aa04.hostc:2,R", "Subject: ab\x00c\nPriority: \nDue: 2025-01-01\n---\nab\x00c body"),
    (".Sortfix", "1700000200.aa05.hosta:2,", "Subject: ab\x00\nDue: 2025-01-01\n---\nab\x00"),
    (".Sortfix", "1700000300.aa06.hostd:2,P", "Subject: ab\nsubject: shadowed\nSubject: ab last\nDue: 2022-06-01\n---\nab"),
    (".Sortfix", "1700000300.aa07.hosta:2,", "subject: lower first\nSubject: upper second\nDue: 2022-06-01\n---\nzz"),
    (".Sortfix", "1700000400.aa08.hoste:2,", "Subject: é accent\nDue: 2021-01-01\n---\n\U0001F600 grin"),
    (".Sortfix", "1700000400.aa09.hosta:2,S", "Subject: \U0001F600 emoji\nDue: 2021-01-01\n---\n日本語"),
    (".Sortfix", "1700000500.aa10.hostf:2,", "Subject: \nTimestamp: 1700000000\nDue: 2020-02-02\n---\n"),
    (".Sortfix", "1700000500.aa11.hosta:2,", "Priority: mid\nTimestamp: 17\nDue: 2020-02-02\n---\nno subject here"),
    (".Sortfix", "1700000600.aa12.hostg:2,F", f"Subject: {LONG}one\nStatus: active\nDue: 2019-09-09\n---\n{LONG}one"),
    (".Sortmix", "1700000700.bb01.hosta:2,", "Subject: mixed a\nDue: 2024-01-01\n---\nx"),
    (".Sortmix", "1700000700.bb02.hosta:2,", "Subject: mixed b\n---\ny"),
    (".Sortmix", "1700000800.bb03.hostb:2,", "Subject: mixed c\nDue: not a date\n---\nz"),
    (".Sortmix", "1700000800.bb04.hostb:2,", "Subject: mixed d\nDue: 2024-01-01T10:00:00+02:00\n---\nw"),
    (".Sortmix", "1700000900.bb05.hostc:2,", "Subject: mixed e\nDue: 2023-05-05\nStatus: done\n---\nv"),
    (".Sortaware", "1700001000.cc01.hosta:2,", "Subject: aware a\nDue: 2024-01-01T10:00:00+02:00\n---\n"),
    (".Sortaware", "1700001000.cc02.hosta:2,", "Subject: aware b\nDue: 2024-01-01T08:00:00+00:00\n---\n"),
    (".Sortaware", "1700001100.cc03.hosta:2,", "Subject: aware c\nDue: 2023-01-01T08:00:00-05:00\n---\n"),
]


def write_fixture(base):
    for folder, name, text in FIXTURE:
        d = os.path.join(base, folder, "cur")
        for st in ("cur", "new", "tmp"):
            os.makedirs(os.path.join(base, folder, st), exist_ok=True)
        with open(os.path.join(d, name), "w", encoding="utf-8") as f:
            f.write(text)


@pytest.fixture(scope="module")
def tree(gpu, tmp_path_factory):
    base = str(tmp_path_factory.mktemp("memdir_sort") / "Memdir")
    build_tree(base)
    write_fixture(base)
    from fei_b200.memdir_tools import utils as U
    old = U.MEMDIR_BASE
    U.set_memdir_base(base)
    yield base
    U.set_memdir_base(old)


def _query(conds, include_content, sort, rev, limit, offset):
    from fei_b200.memdir_tools.search import SearchQuery
    q = SearchQuery()
    for f, op, v in conds:
        q.add_condition(f, op, v)
    q.with_content(include_content)
    q.set_sort(sort, rev)
    q.set_pagination(limit, offset)
    return q


def _reference_sort(mems, field, rev):
    """search.py:370-382 on the oracle's dicts: (sorted list, printed warning lines)."""
    res = list(mems)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        try:
            res.sort(key=lambda m: mo.lookup(m, field) or "", reverse=rev)
        except Exception as e:
            print(f"Warning: Unable to sort results: {e}")
            res.sort(key=lambda x: x["metadata"]["timestamp"], reverse=True)
    return res, buf.getvalue()


def _warnings(text):
    return [ln for ln in text.splitlines() if ln.startswith("Warning:")]


def check_all(base, folders, statuses, conds, fields, include_content, offsets=(0, 3, None)):
    from fei_b200.memdir_tools.search import search_memories
    with contextlib.redirect_stdout(io.StringIO()):
        mems = mo.listing(base, folders, statuses, include_content)
    mems = [mems[i] for i in mo.run_search(mems, [{"field": f, "operator": op, "value": v} for f, op, v in conds])]
    n_checked = 0
    for field in fields:
        for rev in (False, True):
            want_all, want_out = _reference_sort(mems, field, rev)
            for limit in LIMITS:
                for offset in offsets:
                    off = len(mems) + 2 if offset is None else offset
                    want = want_all[off:None if limit is None else off + limit] if (off or limit) else want_all
                    buf = io.StringIO()
                    with contextlib.redirect_stdout(buf):
                        got = search_memories(_query(conds, include_content, field, rev, limit, off), folders, statuses)
                    ctx = (folders, statuses, conds, field, rev, limit, off, include_content)
                    assert [(m["folder"], m["status"], m["filename"]) for m in got] == \
                        [(m["folder"], m["status"], m["filename"]) for m in want], ctx
                    assert got == want, ctx
                    assert _warnings(buf.getvalue()) == _warnings(want_out), ctx
                    n_checked += 1
    return n_checked


def test_sorted_pages_match_cpython_sort(tree):
    assert check_all(tree, None, None, [], FIELDS, False) > 0


def test_sorted_pages_with_content_and_a_condition(tree):
    check_all(tree, None, None, [("Tags", "has_tag", "python")], ["content", "Subject", "date", "Due"], True)
    check_all(tree, [".Sortfix"], ["cur"], [], ["content", "Subject", "filename"], True)


def test_requested_segments_in_non_listing_order(tree):
    from fei_b200 import packer
    packer.packed()
    folders = [".Sortfix", "", ".Sortmix", ".Projects/AI"]
    check_all(tree, folders, ["new", "cur"], [], ["Subject", "Due", "timestamp", "folder", "status", "id"], False)


def test_single_class_date_headers_and_mixed_class_fallback(tree):
    fields = ["Due", "due", "timestamp", "Timestamp", "Subject"]
    check_all(tree, [".Sortfix"], None, [], fields, False)       # Due on every record: naive datetimes, one class
    check_all(tree, [".Sortaware"], None, [], fields, False)     # tz-aware only
    check_all(tree, [".Sortmix"], None, [], fields, False)       # absent / unparseable / aware / naive: the sort raises


def test_sort_keys_that_raise(tmp_path, gpu):
    """A Due value dateutil overflows on: the key function raises, the list stays as it was, then the newest-first fallback."""
    from fei_b200.memdir_tools import utils as U
    base = str(tmp_path / "Memdir")
    for st in ("cur", "new", "tmp"):
        os.makedirs(os.path.join(base, st), exist_ok=True)
    for k, due in enumerate(["2024-01-01", "99999999999999999999", "2023-01-01", "99999999999999999999"]):
        with open(os.path.join(base, "cur", f"17000000{k % 2}0.dd{k:02d}.host:2,"), "w") as f:
            f.write(f"Subject: s{k}\nDue: {due}\n---\nb")
    old = U.MEMDIR_BASE
    U.set_memdir_base(base)
    try:
        check_all(base, None, None, [], ["Due"], False)
    finally:
        U.set_memdir_base(old)


def test_sorted_pages_after_incremental_sync(gpu, tmp_path):
    from fei_b200 import packer, synth
    from fei_b200.memdir_tools import utils as U
    from fei_b200.memdir_tools.search import search_memories
    base = str(tmp_path / "Memdir")
    synth.write_memdir(base, [synth.record(33, i) for i in range(300)])
    write_fixture(base)
    old = U.MEMDIR_BASE
    U.set_memdir_base(base)
    try:
        first = search_memories(_query([], False, None, False, None, 0))
        assert U.update_memory_flags(first[0]["filename"], first[0]["folder"], first[0]["status"], "FRS")
        assert U.move_memory(first[1]["filename"], first[1]["folder"], ".Archive", first[1]["status"], "cur")
        os.remove(os.path.join(base, ".Sortfix", "cur", "1700000300.aa07.hosta:2,"))
        U.save_memory(".Sortfix", "fresh body", {"Subject": LONG + "one", "Due": "2024-03-01", "Timestamp": "5"}, "P")
        U.save_memory("", "second fresh body", {"Subject": "ab\x00c", "Priority": "high"}, "")
        pm = packer.packed()
        assert pm.identity is False and pm.delta is not None
        check_all(base, None, None, [], ["Subject", "Priority", "filename", "id", "hostname", "flags", "date", "timestamp", "Due", "folder"], False)
        check_all(base, None, None, [], ["content"], True)
        assert packer.packed().identity is False
    finally:
        U.set_memdir_base(old)


def test_paging_materialises_only_the_page(tree, monkeypatch):
    from fei_b200 import packer
    from fei_b200.memdir_tools.search import search_memories
    pm = packer.packed()
    sizes = []
    real = packer.PackedMemdir.materialize
    monkeypatch.setattr(packer.PackedMemdir, "materialize", lambda self, pos, ic: (sizes.append(len(pos)), real(self, pos, ic))[1])
    with contextlib.redirect_stdout(io.StringIO()):
        assert len(search_memories(_query([], True, "Subject", True, 10, 5))) == 10
        assert len(search_memories(_query([], False, None, False, 3, 0))) == 3
    assert sizes == [10, 3] and pm.n > 100


# ----------------------------------------------------------------------------- the C ABI
def _subject(hdr: bytes):
    seen = None
    vals = {}
    for line in hdr.split(b"\n"):
        k, c, v = line.partition(b":")
        if c:
            k = k.strip()
            vals[k] = v.strip()
            if seen is None and k.decode().lower() == "subject":
                seen = k
    return vals[seen] if seen is not None else b""


@pytest.fixture(scope="module")
def synth_corpus(gpu):
    from fei_b200.corpus import Corpus
    n = 1 << 20
    c = Corpus().synth(0x5047, 0, n)
    got = c.fetch(0, n)
    ho = got["hdr_off"].astype(np.int64)
    hdr = got["hdr"].tobytes()
    subj = [_subject(hdr[ho[i]:ho[i + 1]]) for i in range(n)]
    yield c, subj, got["wall"].tolist()
    c.close()


def test_abi_sort_rows_matches_python_stable_sort(synth_corpus):
    from fei_b200 import _abi
    from fei_b200.packer import _slot_prog
    c, subj, wall = synth_corpus
    n = len(subj)
    rng = np.random.default_rng(7)
    rows = rng.permutation(n)[: n - 12345]                   # any order, not every record
    sub = rng.permutation(n)[:150000]                        # bodies average 3.5 kB: sort a slice of the corpus by them
    _h, _ho, body, bo = c.fetch_records(sub)
    bo = bo.astype(np.int64)
    bodies = {int(r): body[bo[k]:bo[k + 1]] for k, r in enumerate(sub.tolist())}
    for name, kw, key, rs in (("Subject", dict(source=_abi.SORT_SLOT, prog=_slot_prog("Subject", 0)), subj, rows),
                              ("body", dict(source=_abi.SORT_BODY), bodies, sub),
                              ("wall", dict(source=_abi.SORT_WALL), wall, rows)):
        m = len(rs)
        for desc in (False, True):
            want = sorted(range(m), key=lambda i: key[rs[i]], reverse=desc)
            got, info = _abi.sort_rows([c], np.zeros(m, np.uint32), rs, descending=desc, **kw)
            assert got.tolist() == want, (name, desc)
            if name != "wall":
                assert info.rounds >= 2, (name, info.rounds)
            page, _ = _abi.sort_rows([c], np.zeros(m, np.uint32), rs, descending=desc, first=m - 5, count=100, **kw)
            assert page.tolist() == want[m - 5:], (name, desc)


def test_abi_sort_rows_edges(synth_corpus):
    import ctypes as C
    from fei_b200 import _abi
    c = synth_corpus[0]
    got, info = _abi.sort_rows([c], np.zeros(0, np.uint32), np.zeros(0, np.uint64), source=_abi.SORT_WALL)
    assert got.size == 0 and info.rounds == 0
    got, info = _abi.sort_rows([c], np.zeros(1, np.uint32), np.array([77], np.uint64), source=_abi.SORT_BODY, descending=True)
    assert got.tolist() == [0]
    got, _ = _abi.sort_rows([c], np.zeros(3, np.uint32), np.array([5, 6, 7], np.uint64), source=_abi.SORT_WALL, first=3, count=10)
    assert got.size == 0
    with pytest.raises(_abi.FeiError) as e:
        _abi.sort_rows([c], np.zeros(2, np.uint32), np.array([1, 2], np.uint64), source=99)
    assert e.value.code == _abi.FEI_E_BADARG
    with pytest.raises(_abi.FeiError) as e:                      # a synthetic corpus has no file names
        _abi.sort_rows([c], np.zeros(2, np.uint32), np.array([1, 2], np.uint64), source=_abi.SORT_NAME)
    assert e.value.code == _abi.FEI_E_BADARG
    with pytest.raises(_abi.FeiError) as e:
        _abi.sort_rows([c], np.array([0, 1], np.uint32), np.array([1, 2], np.uint64), source=_abi.SORT_WALL)
    assert e.value.code == _abi.FEI_E_BADARG
    spec = _abi.SortSpec(_abi.SORT_KEYS, 0, None, 0, None)
    hs = (C.c_void_p * 1)(c.handle)
    rc = _abi.lib().fei_sort_rows(hs, 1, np.zeros(2, np.uint32).ctypes.data, np.array([1, 2], np.uint64).ctypes.data, 2, C.byref(spec), 0, 0, 0, None, None)
    assert rc == _abi.FEI_E_BADARG
