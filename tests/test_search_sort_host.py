"""The host side of search_memories' ordering (no GPU): keys of more than one class make CPython's list.sort raise part way and
leave a partial order, which the reference then re-sorts newest first (search.py:370-382).  packer.python_order replays that on
indices; it must leave the same order and print the same warning as list.sort on the oracle's dicts."""
import contextlib
import io

import pytest

from oracle import memdir_oracle as mo

DUES = ["2024-01-01", None, "not a date", "2024-01-01T10:00:00+02:00", "2023-05-05", "", "2022-02-02 10:00", "2024-01-01",
        "2021-01-01T00:00:00+00:00", None, "2020-01-01"]


def _mems(dues, timestamp_headers=()):
    out = []
    for k, due in enumerate(dues):
        head = f"Subject: s{k}\n" + (f"Due: {due}\n" if due is not None else "")
        if k in timestamp_headers:
            head += f"Timestamp: {900 + k}\n"
        ts = 1700000000 + 10 * (k % 4)                       # ties
        out.append(mo.make_memory(f"{ts}.u{k:03d}.host:2,", "", "cur", head + "---\nbody", False))
    return out


def _reference(mems, field, rev):
    res = list(mems)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        try:
            res.sort(key=lambda m: mo.lookup(m, field) or "", reverse=rev)
        except Exception as e:
            print(f"Warning: Unable to sort results: {e}")
            res.sort(key=lambda x: x["metadata"]["timestamp"], reverse=True)
    return [m["filename"] for m in res], buf.getvalue()


def _ours(mems, field, rev):
    from fei_b200.packer import python_order
    ts = [m["metadata"]["timestamp"] for m in mems]
    err, keys = None, []
    for m in mems:                                            # the key of every result, in list order, as list.sort computes them
        try:
            keys.append(mo.lookup(m, field) or "")
        except Exception as e:
            err = e
            break
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        order = python_order(keys, ts, rev, err)
    return [mems[i]["filename"] for i in order], buf.getvalue()


@pytest.mark.parametrize("rev", [False, True])
@pytest.mark.parametrize("dues,field,ts_hdr", [
    (DUES, "Due", ()),                                        # str / naive / aware: raises part way
    (DUES[:1] + DUES[2:3], "Due", ()),                        # naive and an unparseable (str) value
    ([d for d in DUES if d and "+" not in d and d != "not a date"], "Due", ()),     # one class: no warning
    (DUES, "timestamp", (1, 4, 6)),                           # Timestamp header (str) next to the int metadata
    (["2024-01-01", "99999999999999999999", "2023-01-01"], "Due", ()),             # the key function raises (OverflowError)
])
def test_python_order_matches_list_sort_on_dicts(dues, field, ts_hdr, rev):
    mems = _mems(dues, ts_hdr)
    want, want_out = _reference(mems, field, rev)
    got, got_out = _ours(mems, field, rev)
    assert got == want
    assert got_out == want_out
    if len({type(k) for k in [mo.lookup(m, field) or "" for m in mems if "9999999999" not in str(m["headers"])]}) > 1:
        assert want_out.startswith("Warning: Unable to sort results: ")


def test_ranks_and_key_classes():
    from datetime import datetime, timedelta, timezone
    from fei_b200.packer import _key_class, _ranks
    a = datetime(2024, 1, 1, 10, tzinfo=timezone(timedelta(hours=2)))
    b = datetime(2024, 1, 1, 8, tzinfo=timezone.utc)           # the same instant as a
    assert _ranks([a, b, datetime(2023, 1, 1, tzinfo=timezone.utc)]) == [1, 1, 0]
    assert _ranks(["b", "a\x00", "a", "\U0001F600", "é"]) == [2, 1, 0, 4, 3]
    assert {_key_class(x) for x in (a, b)} == {"aware"}
    assert _key_class(datetime(2024, 1, 1)) == "naive" and _key_class("") == "str" and _key_class(5) == "int"
