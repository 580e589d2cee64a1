"""Helpers shared by the chain tests: rebuild blocks from the golden fixtures."""
import copy

from oracle import chain_oracle as co
from fei_b200 import synth


def ts_of(s):
    if s["timestamp_is_int"]:
        return int(s["timestamp_repr"])
    return float(s["timestamp_repr"])


def single_block(s, cls=co.Block):
    b = cls(s["index"], ts_of(s), copy.deepcopy(s["memory_data"]), s["previous_hash"], s["responsible_node"], s["proposer_node"])
    b.nonce = s["nonce"]
    b.solver_node = s["solver_node"]
    b.hash = s["hash"]
    return b


def base_chain(case, cls=None):
    specs = synth.chain_specs(case["seed"], 0, case["n"])
    return co.build_chain(specs)


def mutated_chain(case):
    chain = base_chain(case)
    for m in case.get("mutated", []):
        b = chain[m["i"]]
        for k in ("hash", "previous_hash", "nonce", "task_state", "solver_node", "timestamp"):
            setattr(b, k, m[k])
    return chain


def expected(case):
    """(ok, first_bad, kind) parsed from the reference's log line."""
    if case["ok"]:
        return True, -1, 0
    words = case["log"].split()
    idx = int(words[2])
    kind = 1 if "invalid hash" in case["log"] else 2
    return False, idx, kind


def chainsearch_golden():
    """tests/golden/chainsearch_golden.json with every block body in place: a body stored as `"content_synth": i` is the body of
    seeded record i (see tests/golden/make_golden_chainsearch.py)."""
    from tests.conftest import load_golden
    g = load_golden("chainsearch_golden.json")
    for b in g["blocks"]:
        md = b["memory_data"]
        if "content_synth" in md:
            body = synth.record(g["synth_seed"], md.pop("content_synth"))["body"].decode()
            b["memory_data"] = {"content": body, **md}
    return g
