"""CPU suite: the oracle (Python + C restatements) against the reference-generated golden
vectors, and the library's host-side canonical-JSON serialiser against the same texts."""
import hashlib
import os

import pytest

from oracle import chain_oracle as co
from tests.chain_util import single_block, base_chain, mutated_chain, expected


def test_fips_vectors():
    assert co.c_sha256_hex(b"abc") == "ba7816bf8f01cfea414140de5dae2223b00361a396177a9cb410ff61f20015ad"
    assert co.c_sha256_hex(b"") == hashlib.sha256(b"").hexdigest()
    two_block = b"abcdbcdecdefdefgefghfghighijhijkijkljklmklmnlmnomnopnopq"
    assert co.c_sha256_hex(two_block) == "248d6a61d20638b8e5c026930c3e6039a33ce45964ff2167f6ecedd419db06c1"
    for n in (55, 56, 63, 64, 65, 119, 120, 127, 128, 359, 1000):
        data = bytes((7 * k + n) & 0xFF for k in range(n))
        assert co.c_sha256_hex(data) == hashlib.sha256(data).hexdigest()


def test_python_oracle_matches_reference_single_blocks(chain_golden):
    for s in chain_golden["single"]:
        b = single_block(s)
        assert co.block_text(b) == s["text"], s["name"]
        assert co.block_hash(b) == s["hash"], s["name"]


def test_c_oracle_matches_reference_single_blocks(chain_golden):
    for s in chain_golden["single"]:
        if s["name"] == "bigint_index":
            continue                      # the C twin takes int64 only
        b = single_block(s)
        text = co.c_block_text(b)
        assert text == s["text"].encode(), s["name"]
        assert co.c_sha256_hex(text) == s["hash"], s["name"]


def test_oracle_chain_hashes_and_verdicts(chain_golden):
    for case in chain_golden["chains"]:
        chain = mutated_chain(case)
        if "hashes" in case:
            assert [b.hash for b in chain] == case["hashes"]
        assert co.validate(chain) == expected(case), case["name"]
        assert co.c_validate(chain) == expected(case), case["name"]


def test_library_serialiser_matches_reference_texts(chain_golden):
    """Host-only entry point of libfeiscan (no GPU): canonical JSON == json.dumps of the reference."""
    from fei_b200.memdir_tools import memorychain as mc
    blocks = [single_block(s) for s in chain_golden["single"]]
    texts = mc.canonical_texts(blocks)
    for s, t in zip(chain_golden["single"], texts):
        assert t == s["text"].encode(), s["name"]


def test_library_serialiser_float_repr_sweep():
    import random
    import struct
    from fei_b200.memdir_tools import memorychain as mc
    rng = random.Random(7)
    vals = [0.0, -0.0, 1.0, 1e22, 1e21, 1e16, 9999999999999998.0, 1e-4, 9.999e-5, 123456.789, 5e-324, 2.2250738585072014e-308]
    for _ in range(3000):
        vals.append(struct.unpack("<d", struct.pack("<Q", rng.getrandbits(64)))[0])
        vals.append(rng.random() * 10 ** rng.randint(-20, 20))
        vals.append(1.7e9 + rng.random() * 1e6)
    blocks = [co.Block(i, v, {"metadata": {"unique_id": "u"}}, "0", "a", "b", hash="") for i, v in enumerate(vals)]
    for b, t in zip(blocks, mc.canonical_texts(blocks)):
        assert t == co.block_text(b).encode()


def test_abi_exports_every_declared_symbol():
    """The C-ABI library loads on a CPU-only box and exports everything include/feiscan.h declares."""
    import re
    from fei_b200 import _abi
    l = _abi.lib()
    assert l.fei_abi_version() == 1
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "feiscan.h")).read()
    declared = set(re.findall(r"\b(fei_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    for name in declared:
        getattr(l, name)
    assert declared == set(_abi.EXPORTS)


def test_oracle_mining_matches_reference(chain_golden):
    from fei_b200 import synth
    for m in chain_golden["mined"]:
        s = synth.block(0xC4A1, m["spec_index"])
        b = co.Block(s["index"], s["timestamp"], s["memory_data"], m["previous_hash"], s["responsible_node"], s["proposer_node"], nonce=m["start_nonce"])
        co.mine(b, m["difficulty"])
        assert (b.nonce, b.hash) == (m["nonce"], m["hash"]), m


def test_native_marshalling_equals_python_marshalling(chain_golden):
    """fei_b200/_fastcols.c (CPython helper) must hand libfeiscan exactly the columns the pure-Python path builds, and step
    aside (None) for anything unusual."""
    import numpy as np
    from fei_b200.memdir_tools import memorychain as mc
    from tests.chain_util import base_chain
    if mc._fastcols is None:
        pytest.skip("_fastcols not built")
    blocks = base_chain(chain_golden["chains"][0])
    plain = []
    for b in blocks:
        m = mc.MemoryBlock(b.index, b.timestamp, b.memory_data, b.previous_hash, b.responsible_node, b.proposer_node)
        m.nonce = b.nonce; m.hash = b.hash
        for k in ("task_state", "difficulty", "solver_node"):
            setattr(m, k, getattr(b, k, None))
        plain.append(m)
    nat = mc.chain_columns_native(plain)
    assert nat is not None
    cols, stored = mc.chain_columns(plain)
    for a, b in zip(nat[0], cols):
        assert a.uniform == b.uniform
        for k in ("num", "blob", "off", "tag"):
            x, y = getattr(a, k), getattr(b, k)
            assert (x is None) == (y is None) and (x is None or np.array_equal(x, y)), k
    hb, ho = mc._str_blob(stored)
    assert np.array_equal(nat[1], hb) and np.array_equal(nat[2], ho)
    # unusual values: the helper declines, the Python path decides
    plain[3].nonce = True
    assert mc.chain_columns_native(plain) is None
    plain[3].nonce = 1 << 70
    assert mc.chain_columns_native(plain) is None
    plain[3].nonce = 0
    plain[5].previous_hash = "\ud800"
    assert mc.chain_columns_native(plain) is None
    plain[5].previous_hash = "0"
    plain[7].memory_data = {"metadata": None}
    assert mc.chain_columns_native(plain) is None
    assert mc.chain_columns_native([co.Block(0, 1.0, {}, "0", "a", "b")]) is None          # __slots__ class: no instance dict


def test_chain_memory_search_oracle_matches_reference():
    """oracle.search_chain_memories / search_chain_by_tag pinned on what the reference's MemorychainConnector returned
    (tests/golden/chainsearch_golden.json, generated by make_golden.py chainsearch)."""
    from tests.chain_util import chainsearch_golden
    g = chainsearch_golden()
    for q in g["queries"]:
        assert co.search_chain_memories(g["blocks"], q["query"], q["search_content"], q["search_subject"], q["search_tags"]) == q["result"], q["query"]
    for t in g["tags"]:
        assert co.search_chain_by_tag(g["blocks"], t["tag"]) == t["result"], t["tag"]
