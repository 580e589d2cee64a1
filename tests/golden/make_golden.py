#!/usr/bin/env python3
"""Regenerate the golden fixtures by running the UNMODIFIED reference: a checkout of
github.com/david-strejc/fei, whose path FEI_REFERENCE gives.

Needs that checkout and a built libfeiscan (the seeded record generator); the JSON fixtures
it writes are committed, so the tests never need the reference.  Usage:

    FEI_REFERENCE=/path/to/fei TZ=UTC python tests/golden/make_golden.py [chain] [memdir] [chainsearch] [dropin]

The reference is imported with cwd = a scratch directory (memdir_tools.utils binds
MEMDIR_BASE to os.getcwd() at import, utils.py:16) and HOME = scratch (memorychain.py:49-52).
"""
from __future__ import annotations

import io
import json
import logging
import os
import random
import shutil
import sys
import tempfile
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("FEI_REFERENCE", "")

sys.dont_write_bytecode = True
os.environ.setdefault("TZ", "UTC")


def import_reference(scratch: str):
    if not REF or not os.path.isdir(os.path.join(REF, "memdir_tools")):
        sys.exit("set FEI_REFERENCE to a checkout of the reference (a directory with memdir_tools/)")
    os.environ["HOME"] = scratch
    os.chdir(scratch)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import memdir_tools.utils as ru
    import memdir_tools.search as rs
    import memdir_tools.filter as rf
    import memdir_tools.memorychain as rm
    assert ru.__file__.startswith(REF), ru.__file__
    return ru, rs, rf, rm


# --------------------------------------------------------------------------- chain
def chain_cases():
    """(name, ctor args, post-ctor attribute overrides) for single-block KATs (SURVEY.md 8(c))."""
    md = lambda uid, **kw: dict({"metadata": {"unique_id": uid}}, **kw)
    cases = [
        ("kat1", (1, 1700000000.123456, md("abcd1234"), "0" * 64, "nodeA", "nodeB"), {}),
        ("kat2", (1, 1700000000.0, md("abcd1234"), "0" * 64, "n1", "n2"), {}),
        ("kat3_1e16", (2, 1e16, md("x"), "0", "n1", "n2"), {}),
        ("kat4_int_ts", (3, 1700000000, md("x"), "0", "n1", "n2"), {}),
        ("kat5_0.1+0.2", (4, 0.1 + 0.2, md("x"), "0", "n1", "n2"), {}),
        ("kat6_escapes", (5, 1.5e-7, md('q"uo\\te\n\x01'), "0", "nöde-ü", "节点\U0001F409"), {}),
        ("kat7_task", (6, 1712345678.123456, md("task0001", type="task", task_difficulty="extreme", task_state="accepted"),
                       "ab" * 32, "n1", "n2"), {"nonce": 4242}),
        ("kat8_empty_md", (7, 1.0, {}, "p", "r", "q"), {}),
        ("neg_ts", (8, -12.5, md("m"), "0", "a", "b"), {}),
        ("tiny", (9, 5e-324, md("m"), "0", "a", "b"), {}),
        ("huge", (10, 1.7976931348623157e308, md("m"), "0", "a", "b"), {}),
        ("e15", (11, 1e15, md("m"), "0", "a", "b"), {}),
        ("e-4", (12, 0.0001, md("m"), "0", "a", "b"), {}),
        ("e-5", (13, 0.00001, md("m"), "0", "a", "b"), {}),
        ("123456789012345678", (14, 123456789012345678.0, md("m"), "0", "a", "b"), {}),
        ("bigint_index", (2 ** 70, 1.0, md("m"), "0", "a", "b"), {}),
        ("neg_nonce", (15, 2.5, md("m"), "0", "a", "b"), {"nonce": -7}),
        ("solver_set", (16, 3.25, md("m", type="task"), "0", "a", "b"), {"solver_node": "solver-\x7f- "}),
        ("none_nodes", (17, 4.0, md("m"), "0", None, None), {}),
        ("bool_fields", (18, 4.0, md("m"), "0", True, False), {}),
        ("del_tab", (19, 4.0, md("a\tb\rc\x08d\x0ce/f"), "0", "x", "y"), {}),
        ("nan_ts", (20, float("nan"), md("m"), "0", "a", "b"), {}),
        ("inf_ts", (21, float("-inf"), md("m"), "0", "a", "b"), {}),
        ("negzero", (22, -0.0, md("m"), "0", "a", "b"), {}),
    ]
    rng = random.Random(20240921)
    for k in range(40):
        mant = rng.random() * 10 ** rng.randint(-12, 22)
        ts = rng.choice([mant, float(int(mant)), -mant, round(mant, rng.randint(0, 8))])
        cases.append((f"rand{k}", (100 + k, ts, md("%08x" % rng.getrandbits(32)), "%064x" % rng.getrandbits(256), "n1", "n2"),
                      {"nonce": rng.randint(0, 10 ** 6)}))
    return cases


def make_chain(scratch: str):
    ru, rs, rf, rm = import_reference(scratch)
    out = {"generator": "tests/golden/make_golden.py chain", "reference": "memdir_tools/memorychain.py @ /root/reference",
           "single": [], "chains": []}
    for name, args, over in chain_cases():
        b = rm.MemoryBlock(*args)
        for k, v in over.items():
            setattr(b, k, v)
        idx, ts = args[0], args[1]
        ts_repr = repr(ts)
        out["single"].append({
            "name": name,
            "index": idx, "timestamp_repr": ts_repr, "timestamp_is_int": isinstance(ts, int),
            "memory_data": args[2], "previous_hash": args[3], "responsible_node": args[4], "proposer_node": args[5],
            "nonce": b.nonce, "solver_node": b.solver_node,
            "text": __import__("json").dumps({
                "index": b.index, "timestamp": b.timestamp,
                "memory_id": b.memory_data.get("metadata", {}).get("unique_id", ""),
                "previous_hash": b.previous_hash, "responsible_node": b.responsible_node,
                "proposer_node": b.proposer_node, "task_state": b.task_state, "difficulty": b.difficulty,
                "solver_node": b.solver_node, "nonce": b.nonce}, sort_keys=True),
            "hash": b.calculate_hash(),
        })

    # linked chains validated by the reference's own validate_chain
    sys.path.insert(0, REPO)
    from fei_b200 import synth
    stream = io.StringIO()
    handler = logging.StreamHandler(stream)
    handler.setFormatter(logging.Formatter("%(levelname)s %(message)s"))
    rm.logger.addHandler(handler)
    rm.logger.propagate = False

    def run_validate(blocks):
        ch = object.__new__(rm.MemoryChain)          # __init__ crashes on a fresh HOME (SURVEY 8(c))
        ch.lock = threading.RLock()
        ch.chain = blocks
        stream.seek(0); stream.truncate()
        ok = ch.validate_chain()
        return ok, stream.getvalue().strip()

    n = 300
    specs = synth.chain_specs(seed=0xC4A1, first=0, n=n)
    blocks = []
    prev = "0"
    for s in specs:
        b = rm.MemoryBlock(s["index"], s["timestamp"], s["memory_data"], prev, s["responsible_node"], s["proposer_node"])
        blocks.append(b)
        prev = b.hash
    base = [b.to_dict() for b in blocks]
    ok, log = run_validate(blocks)
    out["chains"].append({"name": "synthetic_300_valid", "seed": 0xC4A1, "n": n, "hashes": [b.hash for b in blocks], "ok": ok, "log": log})

    def variant(name, mutate):
        keys = ("hash", "previous_hash", "nonce", "task_state", "solver_node", "timestamp")
        bl = [rm.MemoryBlock.from_dict(json.loads(json.dumps(d))) for d in base]
        before = [tuple(getattr(b, k) for k in keys) for b in bl]
        mutate(bl)
        ok, log = run_validate(bl)
        out["chains"].append({"name": name, "seed": 0xC4A1, "n": n, "ok": ok, "log": log,
                              "mutated": [dict(i=i, **{k: getattr(bl[i], k) for k in keys})
                                          for i in range(n) if tuple(getattr(bl[i], k) for k in keys) != before[i]]})

    def m_hash(bl): bl[137].hash = bl[137].hash[:-1] + ("0" if bl[137].hash[-1] != "0" else "1")
    def m_link(bl): bl[55].previous_hash = "f" * 64                      # shows up as invalid hash (prev is hashed)
    def m_nonce(bl): bl[200].nonce = 99
    def m_relink_only(bl):                                              # consistent hash, wrong link
        bl[77].previous_hash = "e" * 64
        bl[77].hash = bl[77].calculate_hash()
    def m_genesis(bl): bl[0].hash = "not-a-hash"                        # genesis hash unchecked, but block 1's link breaks
    def m_two(bl):
        bl[250].hash = "x" * 64
        bl[10].timestamp = bl[10].timestamp + 1.0
    def m_solver(bl): bl[33].solver_node = "node-z"                      # vote_on_solution-after-rehash pattern
    def m_short(bl): bl[5].hash = bl[5].hash[:63]
    def m_upper(bl): bl[6].hash = bl[6].hash.upper()
    def m_last(bl): bl[n - 1].hash = "0" * 64
    def m_first(bl): bl[1].nonce = 1
    for nm, fn in [("bad_hash_137", m_hash), ("bad_prev_55", m_link), ("nonce_200", m_nonce), ("relinked_77", m_relink_only),
                   ("genesis_hash", m_genesis), ("two_faults", m_two), ("solver_33", m_solver), ("short_hash_5", m_short),
                   ("upper_hash_6", m_upper), ("last_block", m_last), ("first_checked", m_first)]:
        variant(nm, fn)
    # proof of work: MemoryBlock.mine_block of the reference (memorychain.py:132-143)
    out["mined"] = []
    for k, (diff, start) in enumerate([(1, 0), (2, 0), (3, 0), (2, 5000), (4, 0), (0, 7), (3, 123456)]):
        s = specs[10 + k]
        b = rm.MemoryBlock(s["index"], s["timestamp"], s["memory_data"], "ab" * 32, s["responsible_node"], s["proposer_node"])
        b.nonce = start
        b.hash = b.calculate_hash()
        b.mine_block(diff)
        out["mined"].append({"spec_index": 10 + k, "previous_hash": "ab" * 32, "difficulty": diff, "start_nonce": start, "nonce": b.nonce, "hash": b.hash})
    with open(os.path.join(HERE, "chain_kats.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True, default=str)
    print("wrote chain_kats.json:", len(out["single"]), "single blocks,", len(out["chains"]), "chains")


# --------------------------------------------------------------------------- dropin
DROPIN_MODULES = ("memdir_tools", "memdir_tools.utils", "memdir_tools.search", "memdir_tools.filter", "memdir_tools.memorychain")


def make_dropin(scratch: str):
    """The shape of the package fei_b200.dropin.install() patches: per module the functions, the classes with their methods,
    the other values it defines, and the names it imports from its sibling modules (what install() has to rebind)."""
    import importlib
    import inspect
    import_reference(scratch)
    out = {"generator": "tests/golden/make_golden.py dropin", "modules": {}}
    for name in DROPIN_MODULES:
        mod = importlib.import_module(name)
        entry = {"functions": [], "classes": {}, "values": [], "imports": {}}
        for k, v in vars(mod).items():
            if k.startswith("__") or inspect.ismodule(v):
                continue
            if inspect.isfunction(v) or inspect.isclass(v):
                if v.__module__ == name:
                    if inspect.isclass(v):
                        entry["classes"][k] = [m for m, f in vars(v).items() if inspect.isfunction(f)]
                    else:
                        entry["functions"].append(k)
                elif v.__module__.startswith("memdir_tools."):
                    entry["imports"][k] = v.__module__
            elif not callable(v):
                entry["values"].append(k)
        out["modules"][name] = entry
    with open(os.path.join(HERE, "dropin_layout.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote dropin_layout.json:", ", ".join(f"{m}: {len(e['functions'])} functions, {len(e['classes'])} classes"
                                                 for m, e in out["modules"].items()))


def main():
    what = sys.argv[1:] or ["chain", "memdir", "chainsearch", "dropin"]
    scratch = tempfile.mkdtemp(prefix="fei_golden_")
    try:
        if "chain" in what:
            make_chain(scratch)
        if "memdir" in what:
            from make_golden_memdir import make_memdir
            make_memdir(scratch, import_reference)
        if "chainsearch" in what:
            from make_golden_chainsearch import make_chainsearch
            make_chainsearch()
        if "dropin" in what:
            make_dropin(scratch)
    finally:
        os.chdir(REPO)
        shutil.rmtree(scratch, ignore_errors=True)


if __name__ == "__main__":
    sys.path.insert(0, HERE)
    main()
