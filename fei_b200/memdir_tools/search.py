"""memdir_tools.search on the GPU: same public names and behaviour as the reference
(memdir_tools/search.py): ``SearchQuery``, ``parse_search_args``, ``search_memories``.

``search_memories`` keeps its signature (search.py:337) but the per-record loop
(search.py:361-367 -> _memory_matches_query) runs as CUDA kernels over the packed corpus:
the query is compiled to a predicate program (fei_b200.program), scanned by libfeiscan, and
only the hits of the requested page are materialised as the reference's result dicts: the hits are ordered by
`sort_by` on the device (PackedMemdir.sort_page -> fei_sort_rows) with the reference's semantics (search.py:369-388).
"""
from __future__ import annotations

import calendar
import math
import re
from datetime import datetime, timedelta
from typing import Any, Dict, List, Optional, Sequence, Tuple

import dateutil.parser
import numpy as np

from .. import packer
from ..program import (C_BODY, C_CONST, C_DATE_CMP, C_FLAGS, C_FOLDER_SET, C_NAME, C_RECBITS, C_SLOT, C_STATUS_SET, C_TS_CMP, CMP, MAX_AUX,
                       NAME_DATE_STR, NAME_FILENAME, NAME_HOST, NAME_ID, NAME_TS_STR, Cond, ProgramBuilder, const)
from ..regexc import Pattern, compile_patterns
from . import utils as U

STANDARD_FOLDERS = U.STANDARD_FOLDERS
FLAGS = U.FLAGS
_DATE_HEADERS = ("date", "due", "created", "modified", "deleteddate")
_WORKFLOW = ("active", "pending", "completed", "in-progress", "blocked", "deferred")


class SearchQuery:
    """Conditions + sort + pagination container (reference search.py:21-95)."""

    def __init__(self):
        self.conditions: List[Dict[str, Any]] = []
        self.sort_by = None
        self.sort_reverse = False
        self.limit = None
        self.offset = 0
        self.include_content = False

    def add_condition(self, field: str, operator: str, value: Any) -> "SearchQuery":
        self.conditions.append({"field": field, "operator": operator, "value": value})
        return self

    def set_sort(self, field: str, reverse: bool = False) -> "SearchQuery":
        self.sort_by, self.sort_reverse = field, reverse
        return self

    def set_pagination(self, limit: Optional[int] = None, offset: int = 0) -> "SearchQuery":
        self.limit, self.offset = limit, offset
        return self

    def with_content(self, include: bool = True) -> "SearchQuery":
        self.include_content = include
        return self


def parse_search_args(args_str: str) -> SearchQuery:
    """Query-string grammar of the reference (search.py:392-519), including its quirks:
    the operator alternation makes `>=`/`<=` parse as `>`/`<` with a leading '=' in the value, and
    `sort:` / `limit:` tokens are captured by the field pattern before their own branches."""
    q = SearchQuery()
    tokens = [a or b for a, b in re.findall(r'([^\s"]+)|"([^"]*)"', args_str)]
    words: List[str] = []
    for tok in tokens:
        if tok.startswith("#") and len(tok) > 1:
            q.add_condition("Tags", "has_tag", tok[1:])
            continue
        if tok.startswith("+") and len(tok) > 1 and all(c in "FRSP" for c in tok[1:]):
            for fl in tok[1:]:
                q.add_condition("flags", "has_flag", fl)
            continue
        m = re.match(r"([a-zA-Z_]+)(:|=|!=|>|<|>=|<=)(.+)", tok)
        if m:
            field, op, value = m.groups()
            fl = field.lower()
            if fl in ("status_value", "state"):
                field = "Status"
            elif fl == "status" and value.lower() in _WORKFLOW:
                field = "Status"
            if op == ":":
                op = "has_tag" if field.lower() == "tags" else "has_flag" if field.lower() == "flags" else "contains"
            if value.startswith("/") and value.endswith("/") and len(value) > 2:
                value, op = value[1:-1], "matches"
            if field.lower() == "tags" and op == "has_tag" and "," in value:
                for tag in value.split(","):
                    tag = tag.strip()
                    if tag:
                        q.add_condition("Tags", "has_tag", tag)
            else:
                q.add_condition(field, op, value)
        elif tok.startswith("sort:"):
            f = tok[5:]
            rev = f.startswith("-")
            q.set_sort(f[1:] if rev else f, rev)
        elif tok.startswith("limit:"):
            try:
                q.set_pagination(limit=int(tok[6:]))
            except ValueError:
                pass
        elif tok == "with_content":
            q.with_content(True)
        else:
            words.append(tok)
    if words:
        phrase = " ".join(words)
        q.add_condition("Subject", "contains", phrase)
        q.add_condition("content", "contains", phrase)
    return q


# ----------------------------------------------------------------------------- query compiler
class _Raises:
    """A condition that raises in the reference for every record that reaches it with a non-None value."""

    def __init__(self, exc: Exception, presence: Optional[Cond], exc_of=None):
        self.exc, self.presence = exc, presence
        self.exc_of = exc_of                 # record index -> the exception that record raises (when the records differ in that)


def _string_pattern(op: str, v2: Any, v1_name: str):
    """(Pattern | bool | _Raises-marker, negate) for a str-valued field (search.py:147-239)."""
    if op == "contains":
        return Pattern("contains", str(v2).lower()), False
    if op == "matches":
        try:
            re.compile(str(v2), re.IGNORECASE)
        except re.error:
            return False, False                            # bad regex never matches (search.py:153-154)
        return Pattern("regex", str(v2), re.IGNORECASE), False
    if op == "startswith":
        return Pattern("startswith", str(v2).lower()), False
    if op == "endswith":
        return Pattern("endswith", str(v2).lower()), False
    if op == "has_tag":
        return Pattern("has_tag", str(v2).lower()), False
    if op in ("=", "!="):
        if isinstance(v2, str):
            return Pattern("equals", v2.lower()), op == "!="
        return op == "!=", False                          # str == non-str is False
    if op in (">", "<", ">=", "<="):
        if isinstance(v2, str):
            if v2 == "now" or (v2.startswith("now") and re.match(r"now([+-])(\d+)([dwmy])", v2)):
                return TypeError(f"'{op}' not supported between instances of 'str' and 'datetime.datetime'"), False
            return Pattern({">": "cmp_gt", "<": "cmp_lt", ">=": "cmp_ge", "<=": "cmp_le"}[op], v2), False
        return TypeError(f"'{op}' not supported between instances of 'str' and '{type(v2).__name__}'"), False
    if op == "has_flag":
        return Pattern("exact_contains", str(v2).upper()), False
    return False, False                                    # unknown operator


def _eval_on_strings(values: Sequence[str], op: str, v2: Any) -> List[Any]:
    """Host evaluation of a string operator on a handful of distinct values (folder / status names)."""
    pat, neg = _string_pattern(op, v2, "")
    if isinstance(pat, bool):
        return [pat] * len(values)
    if isinstance(pat, Exception):
        return [pat] * len(values)
    d = compile_patterns([pat])
    return [bool(d.run(v.encode("utf-8")) & 1) != neg for v in values]


def compile_conditions(conditions: Sequence[Dict[str, Any]], include_content: bool, pm: "packer.PackedMemdir") -> List[Any]:
    """Reference conditions -> ordered list of Cond / _Raises (evaluation order of search.py:265-331)."""
    def is_keyword(c):
        return c["field"] == "Subject" and c["operator"] == "contains" and any(
            o["field"] == "content" and o["operator"] == "contains" and o["value"] == c["value"] for o in conditions)
    ordered = [c for c in conditions if is_keyword(c)] + [c for c in conditions if not is_keyword(c)]
    out: List[Any] = []
    for c in ordered:
        out.extend(_compile_one(c["field"], c["operator"], c["value"], include_content, pm))
    return out


def _slot(field: str, mode: int, empty: bool, pat, neg, if_missing: int = 0) -> List[Any]:
    present = Cond(C_SLOT, pattern=Pattern("regex", "", re.IGNORECASE), field=field, mode=mode, empty_if_missing=empty)
    if isinstance(pat, bool):
        # constant verdict, but a missing header (None) is always False (search.py:144-145)
        return [present if pat else const(False)] if not empty else [const(pat)]
    if isinstance(pat, Exception):
        return [_Raises(pat, None if empty else present)]
    return [Cond(C_SLOT, pattern=pat, negate=neg, field=field, mode=mode, empty_if_missing=empty, if_missing=if_missing)]


def _compile_one(field: Any, op: str, v2: Any, include_content: bool, pm) -> List[Any]:
    field = str(field)
    low = field.lower()
    if field in ("Status", "status_value", "state") or low in ("status_value", "state"):
        pat, neg = _string_pattern(op, v2, "Status")
        return _slot("Status", 1, True, pat, neg)                         # headers.get("Status", "")
    if low == "content":
        pat, neg = _string_pattern(op, v2, "content")
        if isinstance(pat, bool):
            return [const(pat)]
        if isinstance(pat, Exception):
            return [_Raises(pat, None)]
        if not include_content:                                           # memory.get("content", "") == "" (search.py:103-104, :363)
            return [const(bool(compile_patterns([pat]).run(b"") & 1) != neg)]
        return [Cond(C_BODY, pattern=pat, negate=neg)]
    if low == "flags":
        pat, neg = _string_pattern(op, v2, "flags")
        if isinstance(pat, bool):
            return [const(pat)]
        if isinstance(pat, Exception):
            return [_Raises(pat, None)]
        return [Cond(C_FLAGS, pattern=pat, negate=neg)]
    if low == "date":
        return _compile_date(op, v2)
    if low in ("id", "filename"):
        pat, neg = _string_pattern(op, v2, low)
        if isinstance(pat, bool):
            return [const(pat)]
        if isinstance(pat, Exception):
            return [_Raises(pat, None)]
        return [Cond(C_NAME, pattern=pat, negate=neg, which=NAME_ID if low == "id" else NAME_FILENAME)]
    if low in ("folder", "status", "maildir_status"):
        names = pm.folders if low == "folder" else U.STANDARD_FOLDERS
        ids = [pm.folder_ids[f] for f in names] if low == "folder" else list(range(len(names)))      # packed folder ids are stable, not positions
        if ids and max(ids) >= 64:
            raise NotImplementedError("folder predicates on more than 64 folders")
        verdicts = _eval_on_strings(names, op, v2)
        if any(isinstance(v, Exception) for v in verdicts):
            return [_Raises(next(v for v in verdicts if isinstance(v, Exception)), None)]
        bits = sum(1 << i for i, v in zip(ids, verdicts) if v)
        return [Cond(C_FOLDER_SET if low == "folder" else C_STATUS_SET, set64=bits)]
    if low in _DATE_HEADERS:
        return _compile_date_header(field, op, v2, pm)
    if low == "timestamp":
        return _compile_timestamp(field, op, v2, pm)
    pat, neg = _string_pattern(op, v2, field)
    if low in ("unique_id", "hostname"):                                  # header first, metadata otherwise (search.py:121-137)
        if isinstance(pat, (bool, Exception)):
            return [const(pat)] if isinstance(pat, bool) else [_Raises(pat, None)]
        return [Cond(C_SLOT, pattern=pat, negate=neg, field=field, mode=0, if_missing=2),
                Cond(C_NAME, pattern=pat, negate=neg, which=NAME_ID if low == "unique_id" else NAME_HOST)]
    return _slot(field, 0, False, pat, neg)


def _compile_date(op: str, v2: Any) -> List[Any]:
    """`date` is datetime.fromtimestamp(ts) (utils.py:94); the operand goes through dateutil (search.py:166-198)."""
    if op not in CMP:                                    # text operators read str(datetime) = "YYYY-MM-DD HH:MM:SS" (search.py:148-163, :237-239)
        pat, neg = _string_pattern(op, v2, "date")
        if isinstance(pat, bool):
            return [const(pat)]
        if isinstance(pat, Exception):
            return [_Raises(pat, None)]
        return [Cond(C_NAME, pattern=pat, negate=neg, which=NAME_DATE_STR)]
    if not isinstance(v2, datetime):
        try:
            v2 = dateutil.parser.parse(str(v2))
        except (ValueError, TypeError, OverflowError):
            return [const(False)]
    if v2.tzinfo is not None and v2.utcoffset() is not None:
        if op == "=":
            return [const(False)]                        # naive == aware is False, != is True
        if op == "!=":
            return [const(True)]
        return [_Raises(TypeError("can't compare offset-naive and offset-aware datetimes"), None)]
    micros = calendar.timegm(v2.timetuple()) * 1000000 + v2.microsecond
    return [Cond(C_DATE_CMP, op=CMP[op], i64=micros)]



def _int_cmp_cond(op: str, v2: Any) -> List[Any]:
    """metadata["timestamp"] (an int) against a non-string operand: Python's int comparison semantics (search.py:166-234)."""
    if isinstance(v2, datetime):
        if op in ("=", "!="):
            return [const(op == "!=")]
        return [_Raises(TypeError(f"'{op}' not supported between instances of 'int' and 'datetime.datetime'"), None)]
    if isinstance(v2, bool):
        v2 = int(v2)
    if isinstance(v2, float):
        if math.isnan(v2):
            return [const(op == "!=")]
        if math.isinf(v2):
            return [const({">": v2 < 0, ">=": v2 < 0, "<": v2 > 0, "<=": v2 > 0, "=": False, "!=": True}[op])]
        if v2 != math.floor(v2):
            if op in ("=", "!="):
                return [const(op == "!=")]
            lo, hi = math.floor(v2), math.ceil(v2)
            op, v2 = (">", lo) if op in (">", ">=") else ("<", hi)
        else:
            v2 = int(v2)
    if not isinstance(v2, int):
        if op in ("=", "!="):
            return [const(op == "!=")]                    # int == <other object> is False
        return [_Raises(TypeError(f"'{op}' not supported between instances of 'int' and '{type(v2).__name__}'"), None)]
    big = (1 << 63) - 1
    if v2 > big or v2 < -big:
        return [const({">": v2 < 0, ">=": v2 < 0, "<": v2 > 0, "<=": v2 > 0, "=": False, "!=": True}[op])]
    return [Cond(C_TS_CMP, op=CMP[op], i64=int(v2))]


def _compile_timestamp(field: str, op: str, v2: Any, pm) -> List[Any]:
    """`timestamp`: a header of that name wins (search.py:121-132), else metadata["timestamp"], an int (search.py:134-137)."""
    absent = Cond(C_SLOT, pattern=Pattern("regex", "", re.IGNORECASE), negate=True, field=field, mode=0, if_missing=1)   # true iff no such header
    pat, neg = _string_pattern(op, v2, field)
    hdr = [const(pat)] if isinstance(pat, bool) else [_Raises(pat, None)] if isinstance(pat, Exception) else None
    if op in ("contains", "matches", "startswith", "endswith", "has_tag", "has_flag"):      # str(value1): same text semantics for both sources
        if hdr is not None:
            return hdr
        return [Cond(C_SLOT, pattern=pat, negate=neg, field=field, mode=0, if_missing=2), Cond(C_NAME, pattern=pat, negate=neg, which=NAME_TS_STR)]
    if op not in CMP:
        return [const(False)]
    # comparison operators: the metadata int and a header string behave differently
    if isinstance(v2, str):
        if op in ("=", "!="):                             # int == str is False; header str == str compares lower-cased
            meta = const(op == "!=")
        else:
            kind = "datetime.datetime" if v2 == "now" or re.match(r"now([+-])(\d+)([dwmy])", v2) else "str"
            meta = _Raises(TypeError(f"'{op}' not supported between instances of 'int' and '{kind}'"), absent)
        if isinstance(meta, _Raises):
            return [meta] + (hdr if hdr is not None else [Cond(C_SLOT, pattern=pat, negate=neg, field=field, mode=0)])
        if hdr is not None and isinstance(pat, bool) and pat == meta.value:
            return [meta]
        if hdr is not None:
            raise NotImplementedError("timestamp condition whose header and metadata forms disagree in kind")
        return [Cond(C_SLOT, pattern=pat, negate=neg, field=field, mode=0, if_missing=2), meta]
    meta = _int_cmp_cond(op, v2)
    # a non-string operand against a header string: str == int is False, str < int raises
    if op in ("=", "!="):
        hdr_c = const(op == "!=")
        if len(meta) == 1 and isinstance(meta[0], Cond) and meta[0].kind == C_CONST and meta[0].value == hdr_c.value:
            return meta
        present = Cond(C_SLOT, pattern=Pattern("regex", "", re.IGNORECASE), negate=(op == "="), field=field, mode=0, if_missing=2)
        return [present] + meta if not isinstance(meta[0], _Raises) else meta
    exc = TypeError(f"'{op}' not supported between instances of 'str' and '{type(v2).__name__}'")
    present = Cond(C_SLOT, pattern=Pattern("regex", "", re.IGNORECASE), field=field, mode=0)
    return [_Raises(exc, present)] + meta


def _parse_dt(value: str):
    """dateutil.parser.parse as search.py:126-130 calls it, plus whether the result depends on today's date (missing
    fields are taken from `default` = today): such values must be parsed again for every query."""
    try:
        a = dateutil.parser.parse(value, default=datetime(2001, 1, 1))
        b = dateutil.parser.parse(value, default=datetime(2002, 2, 2))
    except (ValueError, TypeError, OverflowError):
        return None, False
    return a, a != b


def _judge_value(v1: Any, op: str, v2: Any) -> bool:
    """The reference's comparison of ONE resolved field value with the operand (search.py:141-242), applied on the host to
    the distinct values of a date-like header (a datetime when dateutil could parse it, else the raw string).  May raise TypeError."""
    if op == "contains":
        return str(v2).lower() in str(v1).lower()
    if op == "matches":
        try:
            return re.search(str(v2), str(v1), re.IGNORECASE) is not None
        except re.error:
            return False
    if op == "startswith":
        return str(v1).lower().startswith(str(v2).lower())
    if op == "endswith":
        return str(v1).lower().endswith(str(v2).lower())
    if op == "has_tag":
        return str(v2).lower() in [t.strip() for t in str(v1).lower().split(",")]
    if op == "has_flag":
        return str(v2).upper() in str(v1)
    if op not in CMP:
        return False
    if isinstance(v1, datetime) and not isinstance(v2, datetime):
        try:
            v2 = dateutil.parser.parse(str(v2))
        except (ValueError, TypeError):
            return False
    if op in ("=", "!="):
        if isinstance(v1, str) and isinstance(v2, str):
            return (v1.lower() == v2.lower()) == (op == "=")
        return (v1 == v2) == (op == "=")
    if isinstance(v2, str) and v2.startswith("now"):
        now = datetime.now()
        if v2 == "now":
            v2 = now
        else:
            m = re.match(r"now([+-])(\d+)([dwmy])", v2)
            if m:
                k = int(m.group(2)) * (-1 if m.group(1) == "-" else 1)
                v2 = now + timedelta(days=k * {"d": 1, "w": 7, "m": 30, "y": 365}[m.group(3)])
    return {">": lambda: v1 > v2, "<": lambda: v1 < v2, ">=": lambda: v1 >= v2, "<=": lambda: v1 <= v2}[op]()


def _compile_date_header(field: str, op: str, v2: Any, pm) -> List[Any]:
    """Due / Created / Modified / DeletedDate: the header value goes through dateutil per record (search.py:126-130).  The GPU hands
    back every record's value (fei_corpus_slot_values), the host judges the DISTINCT values with the reference's rules and returns the
    verdicts as aux columns the scan reads (C_RECBITS): one for 'condition holds', one for 'the reference would raise here'."""
    present, inv, distinct = pm.header_values(field)
    ok = np.zeros(len(distinct) + 1, dtype=np.uint8)      # last entry: absent header (None -> False, search.py:144-145)
    bad = np.zeros(len(distinct) + 1, dtype=np.uint8)
    first_exc: Optional[Exception] = None
    excs: Dict[int, Exception] = {}
    for k, text in enumerate(distinct):
        parsed = pm.parsed_dates.get(text)
        if parsed is None:
            parsed = pm.parsed_dates[text] = _parse_dt(text)
        dt, today_dependent = parsed
        if today_dependent:
            dt = dateutil.parser.parse(text)
        try:
            ok[k] = 1 if _judge_value(dt if dt is not None else text, op, v2) else 0
        except TypeError as e:
            bad[k] = 1
            excs[k] = e
            first_exc = first_exc or e
    out: List[Any] = []
    if bad.any():
        out.append(_Raises(first_exc, Cond(C_RECBITS, which=pm.new_aux(bad[inv])), exc_of=lambda i: excs[int(inv[i])]))
    out.append(Cond(C_RECBITS, which=pm.new_aux(ok[inv])))
    return out


# ----------------------------------------------------------------------------- search
def _scan_ranges(pm, conds: List[Cond], ranges: List[Tuple[int, int]]) -> np.ndarray:
    """Ordered hit indices (pack order restricted / re-ordered to the requested segments)."""
    pb = ProgramBuilder()
    pb.add_query(conds)
    hits = pm.scan_hits(pb.build(), 1)[0]
    parts = []
    for a, b in ranges:
        lo, hi = np.searchsorted(hits, a), np.searchsorted(hits, b)
        parts.append(hits[lo:hi])
    return np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)


def search_memories(query: SearchQuery, folders: Optional[List[str]] = None, statuses: Optional[List[str]] = None,
                    debug: bool = False) -> List[Dict[str, Any]]:
    pm = packer.packed()
    with pm.lock:                                        # one snapshot of the packed corpus (and its aux columns) for the whole request
        ranges = pm.ranges(folders, statuses)
        pm.report_skipped(folders, statuses)
        pm.begin_query()
        compiled = compile_conditions(query.conditions, query.include_content, pm)
        conds: List[Cond] = []
        for item in compiled:
            if isinstance(item, _Raises):
                # the reference raises as soon as one record reaches this condition with a value
                probe = conds + ([item.presence] if item.presence is not None else [])
                reached = _scan_ranges(pm, probe or [const(True)], ranges)
                if len(reached):
                    raise (item.exc_of(int(reached[0])) if item.exc_of else item.exc)
                conds.append(const(False))               # nobody reaches it: everything was rejected earlier
                break
            conds.append(item)
        hits = _scan_ranges(pm, conds or [const(True)], ranges)
        page = range(len(hits))                          # the slice of search.py:385-388, as positions in the ordered hits
        if query.offset or query.limit:
            start = query.offset
            end = None if query.limit is None else start + query.limit
            page = page[start:end]
        if query.sort_by:                                # ordered on the device; only the page is materialised
            hits = pm.sort_page(hits, query.sort_by, query.sort_reverse, query.include_content, page.start, len(page))
        else:
            hits = hits[page.start:page.stop]
        return pm.materialize(hits, query.include_content)
