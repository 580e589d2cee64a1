"""Chain-memory search part of make_golden.py: the reference's MemorychainConnector.search_memories / search_by_tag
(fei/tools/memorychain_connector.py:273-362) over a fixed chain.  Only the network fetch (get_chain) is replaced by a local list;
the search code runs unmodified.

The fixture keeps the file under 1 MB by storing a body longer than STORED_BODY_MAX characters as `"content_synth": i`, the
index of the seeded record whose body it is; tests/chain_util.chainsearch_golden() puts the body back."""
from __future__ import annotations

import importlib.util
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("FEI_REFERENCE", "")
SEED, N = 0xFE1, 300
STORED_BODY_MAX = 4900

QUERIES = [  # (query, search_content, search_subject, search_tags)
    ("python", True, True, True), ("PYTHON", True, False, False), ("learning", False, True, False), ("docker", False, False, True),
    ("", True, True, True), ("", False, False, True), ("no such words anywhere", True, True, True), ("line\nbreak", True, True, True),
    ("İstanbul", True, True, True), ("i̇stanbul", False, True, False), ("cafÉ", True, True, True), ("x", False, False, False),
    (", ", False, False, True), ("review notes", True, True, True),
]
TAGS = ["python", "#Python", "PYTHON ", " python", "x", "", "#", "İzmir", "machine learning"]


def chain_blocks():
    sys.path.insert(0, REPO)
    from fei_b200 import synth
    blocks = [{"index": 0, "memory_data": {"metadata": {"unique_id": "genesis"}, "headers": {"Subject": "Genesis Block python", "Tags": "system,genesis,python"},
                                             "content": "Initial block of the Memory Chain about python"}}]
    for i in range(N):
        r = synth.record(SEED, i)
        headers = {}
        for line in r["hdr"].decode().strip().split("\n"):
            k, _, v = line.partition(":")
            headers[k.strip()] = v.strip()
        md = {"metadata": {"unique_id": r["uid"], "timestamp": r["ts"]}, "headers": headers, "content": r["body"].decode()}
        blocks.append({"index": i + 1, "memory_data": md})
    extra = [
        {"metadata": {"unique_id": "nohdr"}, "content": "no headers at all, python"},
        {"metadata": {"unique_id": "nocontent"}, "headers": {"Subject": "only a subject about Python", "Tags": " Python , x "}},
        {"headers": {"Subject": "multi\nline\nbreak subject", "Tags": "a,b\n,c"}, "content": "body with --- separators\n---\nand Subject: fake header"},
        {"metadata": {"unique_id": "idot"}, "headers": {"Subject": "İstanbul café", "Tags": "İzmir, x"}, "content": "İ body CAFÉ"},
        {"metadata": {"unique_id": "empty"}, "headers": {"Subject": "", "Tags": ""}, "content": ""},
        {"metadata": {"unique_id": "genesis"}, "headers": {"Subject": "a second genesis id is skipped too, python"}, "content": "python"},
    ]
    for k, md in enumerate(extra):
        blocks.append({"index": N + 1 + k, "memory_data": md})
    return blocks


def make_chainsearch():
    if not REF:
        sys.exit("set FEI_REFERENCE to a checkout of the reference")
    spec = importlib.util.spec_from_file_location("ref_memorychain_connector", os.path.join(REF, "fei", "tools", "memorychain_connector.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    blocks = chain_blocks()
    conn = object.__new__(mod.MemorychainConnector)
    conn.get_chain = lambda: blocks                                   # the HTTP fetch, nothing else
    ident = {id(b["memory_data"]): i for i, b in enumerate(blocks)}
    out = {"generator": "tests/golden/make_golden.py chainsearch", "blocks": blocks, "queries": [], "tags": [], "synth_seed": SEED}
    for q, c, s, t in QUERIES:
        res = conn.search_memories(q, search_content=c, search_subject=s, search_tags=t)
        out["queries"].append({"query": q, "search_content": c, "search_subject": s, "search_tags": t, "result": [ident[id(m)] for m in res]})
    for tag in TAGS:
        res = conn.search_by_tag(tag)
        out["tags"].append({"tag": tag, "result": [ident[id(m)] for m in res]})
    stored = []
    for b in blocks:
        md = b["memory_data"]
        if 1 <= b["index"] <= N and len(md["content"]) > STORED_BODY_MAX:
            md = {"content_synth": b["index"] - 1, **{k: v for k, v in md.items() if k != "content"}}
        stored.append({"index": b["index"], "memory_data": md})
    out["blocks"] = stored
    with open(os.path.join(HERE, "chainsearch_golden.json"), "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote chainsearch_golden.json:", len(blocks), "blocks,", len(out["queries"]), "queries,", len(out["tags"]), "tag lookups")
