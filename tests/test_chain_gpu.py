"""GPU parity: SHA-256 link hashes and validate_chain verdicts through the C ABI vs the
reference-generated golden vectors and the oracle."""
import hashlib
import logging

import numpy as np
import pytest

from oracle import chain_oracle as co
from tests.chain_util import single_block, base_chain, mutated_chain, expected

pytestmark = pytest.mark.gpu


def test_single_block_hashes(gpu, chain_golden):
    from fei_b200.memdir_tools import memorychain as mc
    blocks = [single_block(s) for s in chain_golden["single"]]
    _, _, dig = mc.hash_and_validate(blocks, want_digests=True)
    for s, d in zip(chain_golden["single"], dig):
        assert bytes(d).hex() == s["hash"], s["name"]


def test_memoryblock_class_roundtrip(gpu, chain_golden):
    from fei_b200.memdir_tools import memorychain as mc
    s = next(x for x in chain_golden["single"] if x["name"] == "kat7_task")
    b = mc.MemoryBlock(s["index"], float(s["timestamp_repr"]), s["memory_data"], s["previous_hash"], s["responsible_node"], s["proposer_node"])
    b.nonce = s["nonce"]
    assert b.calculate_hash() == s["hash"]
    d = b.to_dict()
    b2 = mc.MemoryBlock.from_dict(d)
    assert b2.hash == b.hash and b2.task_state == "accepted" and b2.difficulty == "extreme"


def test_validate_chain_matches_reference_verdicts(gpu, chain_golden, caplog):
    from fei_b200.memdir_tools import memorychain as mc
    for case in chain_golden["chains"]:
        chain = mutated_chain(case)
        ch = mc.MemoryChain(blocks=chain)
        caplog.clear()
        with caplog.at_level(logging.ERROR, logger="memorychain"):
            ok = ch.validate_chain()
        assert ok == case["ok"], case["name"]
        got = " ".join(f"{r.levelname} {r.getMessage()}" for r in caplog.records)
        assert got == case["log"], case["name"]
        fb, kind, dig = mc.hash_and_validate(chain, want_digests=True)
        assert (fb < 0, fb, kind) == expected(case), case["name"]
        for b, d in zip(chain, dig):
            assert bytes(d).hex() == co.block_hash(b)


def test_message_length_edges(gpu):
    """Padding boundaries: lengths around multiples of 64 and arbitrary stored strings."""
    from fei_b200 import _abi
    import ctypes as C
    msgs = [bytes((i * 31 + k) & 0xFF for k in range(n)) for i, n in enumerate([0, 1, 54, 55, 56, 57, 63, 64, 65, 118, 119, 120, 121, 127, 128, 129, 359, 447, 448, 1000, 4096])]
    hashes = [hashlib.sha256(m).hexdigest().encode() for m in msgs]
    prevs = [b"0"] + hashes[:-1]
    def blob(parts):
        off = np.zeros(len(parts) + 1, dtype=np.uint64); np.cumsum([len(p) for p in parts], out=off[1:])
        return np.frombuffer(b"".join(parts) or b"\0", dtype=np.uint8).copy(), off
    m, mo = blob(msgs); h, ho = blob(hashes); p, po = blob(prevs)
    dig = np.zeros((len(msgs), 32), dtype=np.uint8)
    fb, kind = C.c_int64(), C.c_int32()
    _abi.check(_abi.lib().fei_chain_validate_msgs(_abi.ptr(m), _abi.ptr(mo), _abi.ptr(h), _abi.ptr(ho), _abi.ptr(p), _abi.ptr(po),
                                                 len(msgs), 0, C.byref(fb), C.byref(kind), _abi.ptr(dig)))
    assert fb.value == -1 and kind.value == 0
    for d, hx in zip(dig, hashes):
        assert bytes(d).hex().encode() == hx
    # arbitrary (non-hex) stored strings compare as strings: link ok only if byte-equal
    hashes2 = list(hashes); hashes2[3] = b"weird-hash"
    prevs2 = [b"0"] + hashes2[:-1]
    h, ho = blob(hashes2); p, po = blob(prevs2)
    _abi.check(_abi.lib().fei_chain_validate_msgs(_abi.ptr(m), _abi.ptr(mo), _abi.ptr(h), _abi.ptr(ho), _abi.ptr(p), _abi.ptr(po),
                                                 len(msgs), 0, C.byref(fb), C.byref(kind), None))
    assert (fb.value, kind.value) == (3, 1)          # block 4's link to "weird-hash" is fine, block 3's hash is not


def test_synthetic_chain_1m_properties(gpu):
    """Full-size style run on device-resident data: valid chain -> True; one corruption -> same index;
    digests equal hashlib on the fetched texts (sampled)."""
    from fei_b200 import _abi
    import ctypes as C
    n = 1_000_000                                     # BASELINE configs[3] size
    for corrupt in (-1, 777_777):
        ch = C.c_void_p()
        _abi.check(_abi.lib().fei_chain_create(C.byref(ch)))
        try:
            _abi.check(_abi.lib().fei_chain_synth(ch, 0xC4A1, 0, n, corrupt))
            dig = np.zeros((n, 32), dtype=np.uint8)
            fb, kind, ms = C.c_int64(), C.c_int32(), C.c_float()
            _abi.check(_abi.lib().fei_chain_validate(ch, C.byref(fb), C.byref(kind), _abi.ptr(dig), C.byref(ms)))
            if corrupt < 0:
                assert (fb.value, kind.value) == (-1, 0)
            else:
                assert (fb.value, kind.value) == (corrupt, 1)
            k = 2000
            buf = np.zeros(k * 400, dtype=np.uint8); off = np.zeros(k + 1, dtype=np.uint64)
            hh = np.zeros(k * 64, dtype=np.uint8)
            first = 500_000
            _abi.check(_abi.lib().fei_chain_fetch(ch, first, k, _abi.ptr(buf), buf.size, _abi.ptr(off), _abi.ptr(hh), None))
            for i in range(k):
                text = bytes(buf[int(off[i]):int(off[i + 1])])
                assert hashlib.sha256(text).digest() == bytes(dig[first + i])
            # first 300 blocks are the golden synthetic chain
            specs_chain = co.build_chain(__import__("fei_b200.synth", fromlist=["x"]).chain_specs(0xC4A1, 0, 300))
            for i, b in enumerate(specs_chain):
                assert bytes(dig[i]).hex() == b.hash
        finally:
            _abi.lib().fei_chain_destroy(ch)


def test_receive_chain_update_checks(gpu, chain_golden, caplog):
    """The inline copy of the validation in receive_chain_update (memorychain.py:1059-1078) shares the kernel."""
    from fei_b200.memdir_tools import memorychain as mc
    case = chain_golden["chains"][0]
    chain = base_chain(case)
    dicts = []
    for b in chain:
        d = {"index": b.index, "timestamp": b.timestamp, "memory_data": b.memory_data, "previous_hash": b.previous_hash,
             "responsible_node": b.responsible_node, "proposer_node": b.proposer_node, "nonce": b.nonce, "hash": b.hash}
        if b.memory_data.get("type") == "task":               # what MemoryBlock.to_dict adds for task blocks (:282-291)
            d.update({"difficulty": b.difficulty, "task_state": b.task_state, "solver_node": b.solver_node})
        dicts.append(d)
    local = mc.MemoryChain(blocks=[mc.MemoryBlock.from_dict(d) for d in dicts[:100]])
    assert local.receive_chain_update(dicts[:50]) is False                 # not longer
    assert local.receive_chain_update(dicts) is True and len(local.chain) == len(dicts)
    bad = [dict(d) for d in dicts] + [dict(dicts[-1], index=999, hash="0" * 64)]
    with caplog.at_level(logging.WARNING, logger="memorychain"):
        assert local.receive_chain_update(bad) is False
    assert any("Block 300 has invalid hash" in r.getMessage() for r in caplog.records)
    diverged = [dict(d) for d in dicts]
    diverged[5] = dict(diverged[5], nonce=1)
    other = mc.MemoryChain(blocks=[mc.MemoryBlock.from_dict(d) for d in dicts[:10]])
    caplog.clear()
    with caplog.at_level(logging.WARNING, logger="memorychain"):
        assert other.receive_chain_update(diverged) is False
    assert any("Block 5 has invalid hash" in r.getMessage() for r in caplog.records)


def test_mine_block_matches_reference(gpu, chain_golden):
    """Proof of work on the GPU (fei_chain_mine) finds the same nonce and hash as MemoryBlock.mine_block."""
    from fei_b200 import synth
    from fei_b200.memdir_tools import memorychain as mc
    for m in chain_golden["mined"]:
        s = synth.block(0xC4A1, m["spec_index"])
        b = mc.MemoryBlock(s["index"], s["timestamp"], s["memory_data"], m["previous_hash"], s["responsible_node"], s["proposer_node"])
        b.nonce = m["start_nonce"]
        b.mine_block(m["difficulty"])
        assert (b.nonce, b.hash) == (m["nonce"], m["hash"]), m
        assert b.hash == b.calculate_hash()
    # a harder one, checked against the oracle's definition only
    s = synth.block(0xC4A1, 3)
    b = mc.MemoryBlock(s["index"], s["timestamp"], s["memory_data"], "0" * 64, s["responsible_node"], s["proposer_node"])
    b.mine_block(5)
    assert b.hash.startswith("00000") and b.hash == co.block_hash(b)
    probe = co.Block(s["index"], s["timestamp"], s["memory_data"], "0" * 64, s["responsible_node"], s["proposer_node"])
    for n in range(max(0, b.nonce - 3000), b.nonce):          # no smaller nonce in the window before it
        probe.nonce = n
        assert not co.block_hash(probe).startswith("00000")


def test_build_persist_and_reload_a_chain(gpu, tmp_path):
    """create_genesis_block / add_memory (GPU proof of work) / save_chain / load_chain / serialize_chain (reference :528-594, :1130-1172)."""
    import json
    from fei_b200 import synth
    from fei_b200.memdir_tools import memorychain as mc
    chain = mc.MemoryChain(node_id="node-a", difficulty=3)
    chain.create_genesis_block()
    g = chain.get_latest_block()
    assert g.index == 0 and g.previous_hash == "0" and g.hash.startswith("000") and g.hash == co.block_hash(g)
    with pytest.raises(TypeError):                       # the genesis payload holds a datetime, json.dump refuses it -- as in the reference
        mc.MemoryChain(blocks=chain.chain, chain_file=str(tmp_path / "g.json")).save_chain()
    g.memory_data["metadata"]["date"] = g.memory_data["metadata"]["date"].isoformat()
    chain.chain_file = str(tmp_path / "sub" / "chain.json")          # add_memory persists after every block from here on
    hashes = []
    for i in range(4):
        h = chain.add_memory(synth.block(0xC4A1, 10 + i)["memory_data"], responsible_node="node-b" if i % 2 else None)
        hashes.append(h)
        b = chain.get_latest_block()
        assert b.hash == h and h.startswith("000") and b.index == i + 1 and b.previous_hash == chain.chain[-2].hash
        assert b.responsible_node == ("node-b" if i % 2 else "node-a") and b.proposer_node == "node-a"
        probe = co.Block(b.index, b.timestamp, b.memory_data, b.previous_hash, b.responsible_node, b.proposer_node)
        co.mine(probe, 3)                                # the oracle's nonce loop starts from 0 like MemoryBlock.mine_block
        assert (probe.nonce, probe.hash) == (b.nonce, b.hash)
    assert chain.validate_chain() is True and co.validate(chain.chain) == (True, -1, 0)
    on_disk = json.load(open(chain.chain_file))
    assert on_disk == json.loads(json.dumps(chain.serialize_chain())) and len(on_disk) == 5
    assert open(chain.chain_file).read() == json.dumps(chain.serialize_chain(), indent=2)
    again = mc.MemoryChain(node_id="node-c", chain_file=chain.chain_file)
    assert again.load_chain() is True and [b.hash for b in again.chain] == [g.hash] + hashes and again.validate_chain() is True
    assert mc.MemoryChain(chain_file=str(tmp_path / "missing.json")).load_chain() is False
    (tmp_path / "bad.json").write_text("{not json")
    assert mc.MemoryChain(chain_file=str(tmp_path / "bad.json")).load_chain() is False


def _our_chain(n, seed=0xC4A1):
    from fei_b200 import synth
    from fei_b200.memdir_tools import memorychain as mc
    blocks = []
    for ob in co.build_chain(synth.chain_specs(seed, 0, n)):
        b = mc.MemoryBlock(ob.index, ob.timestamp, ob.memory_data, ob.previous_hash, ob.responsible_node, ob.proposer_node)
        b.nonce = ob.nonce; b.hash = ob.hash
        blocks.append(b)
    return blocks


def test_resident_chain_tracks_mutations(gpu, caplog):
    """MemoryChain keeps a device image of its blocks: a second validate_chain() re-hashes resident data without marshalling a
    block, and every kind of edit (attribute assignment, item assignment, append / pop, a new list) is seen -- the verdict and the
    log line stay the reference's (memorychain.py:596-618)."""
    import ctypes as C
    from fei_b200 import _abi
    from fei_b200.memdir_tools import memorychain as mc
    n = 3000
    ch = mc.MemoryChain(blocks=_our_chain(n))
    r = ch._res
    assert r is not None and r.uploads == 1 and r.marshalled == n          # built when the blocks arrived
    assert ch.validate_chain() and ch.validate_chain() and r.uploads == 1   # resident: nothing marshalled, nothing uploaded
    # the GPU-made canonical JSON equals json.dumps(..., sort_keys=True) of the reference
    off = np.zeros(n + 1, dtype=np.uint64); buf = np.zeros(600 * n, dtype=np.uint8)
    _abi.check(_abi.lib().fei_chain_fetch(r.h, 0, n, _abi.ptr(buf), buf.size, _abi.ptr(off), None, None))
    texts = [bytes(buf[int(off[i]):int(off[i + 1])]) for i in range(n)]
    assert texts == [co.block_text(b).encode() for b in ch.chain]
    with caplog.at_level(logging.ERROR, logger="memorychain"):
        ch.chain[1234].nonce = 5                                            # attribute assignment on a block of the chain
        assert ch.validate_chain() is False and r.uploads == 2 and r.marshalled == n - 1234
        assert caplog.records[-1].getMessage() == "Block 1234 has invalid hash"
        ch.chain[1234].nonce = 0
        assert ch.validate_chain() is True and r.uploads == 3
        ch.chain[2000].memory_data = {"metadata": {"unique_id": "someone-else"}}
        assert ch.validate_chain() is False and caplog.records[-1].getMessage() == "Block 2000 has invalid hash"
        good = _our_chain(n)[2000]
        ch.chain[2000] = good                                               # item assignment
        assert ch.validate_chain() is True
        last = ch.chain.pop()
        assert ch.validate_chain() is True and r.n == n - 1
        last.previous_hash = "0" * 64
        ch.chain.append(last)
        assert ch.validate_chain() is False and caplog.records[-1].getMessage() == f"Block {n - 1} has invalid hash"
        ch.chain = _our_chain(500)                                          # a new list
        assert ch.validate_chain() is True and r.n == 500
        ch.chain[77].hash = "f" * 64                                        # stored hash edited: block 77 invalid, and 78 would have a broken link
        assert ch.validate_chain() is False and caplog.records[-1].getMessage() == "Block 77 has invalid hash"
    # blocks of a foreign class cannot report their mutations: such a chain is marshalled again on every call, never stale
    foreign = co.build_chain(__import__("fei_b200.synth", fromlist=["x"]).chain_specs(0xC4A1, 0, 300))
    ch2 = mc.MemoryChain(blocks=foreign)
    assert ch2.validate_chain() is True
    foreign[100].nonce = 9
    assert ch2.validate_chain() is False and co.validate(foreign) == (False, 100, 1)


def test_gpu_canonical_json_matches_reference_kats(gpu, chain_golden):
    """fei_chain_load_cols: the column form serialised on the GPU (incl. Python's shortest round-trip float repr, ensure_ascii
    escapes, big ints) gives the reference's digests for every golden single-block vector."""
    import ctypes as C
    from fei_b200 import _abi
    from fei_b200.memdir_tools import memorychain as mc
    blocks = [single_block(s) for s in chain_golden["single"]]
    for b in blocks:
        if not isinstance(b.previous_hash, str):
            b.previous_hash = str(b.previous_hash)
    cols, stored = mc.chain_columns(blocks)
    hb, ho = mc._str_blob([s if isinstance(s, str) else "" for s in stored])
    h = C.c_void_p(); _abi.check(_abi.lib().fei_chain_create(C.byref(h)))
    n = len(blocks)
    _abi.check(_abi.lib().fei_chain_load_cols(h, mc._cols_struct(cols), _abi.ptr(hb), _abi.ptr(ho), n, 0))
    dig = np.zeros((n, 32), dtype=np.uint8); fb, kind = C.c_int64(), C.c_int32()
    _abi.check(_abi.lib().fei_chain_validate(h, C.byref(fb), C.byref(kind), _abi.ptr(dig), None))
    off = np.zeros(n + 1, dtype=np.uint64); buf = np.zeros(4096 * n, dtype=np.uint8)
    _abi.check(_abi.lib().fei_chain_fetch(h, 0, n, _abi.ptr(buf), buf.size, _abi.ptr(off), None, None))
    _abi.lib().fei_chain_destroy(h)
    for i, b in enumerate(blocks):
        assert bytes(buf[int(off[i]):int(off[i + 1])]) == mc.canonical_texts([b])[0], chain_golden["single"][i]["name"]
        assert bytes(dig[i]).hex() == co.block_hash(b), chain_golden["single"][i]["name"]


def test_chain_memory_search_matches_reference(gpu):
    """ChainMemorySearch (GPU) vs the reference's MemorychainConnector.search_memories / search_by_tag goldens and the oracle."""
    from tests.chain_util import chainsearch_golden
    from fei_b200.memdir_tools.chain_search import ChainMemorySearch
    g = chainsearch_golden()
    idx = {id(b["memory_data"]): i for i, b in enumerate(g["blocks"])}
    cs = ChainMemorySearch(g["blocks"])
    for q in g["queries"]:
        got = [idx[id(m)] for m in cs.search_memories(q["query"], q["search_content"], q["search_subject"], q["search_tags"])]
        assert got == q["result"] == co.search_chain_memories(g["blocks"], q["query"], q["search_content"], q["search_subject"], q["search_tags"]), q["query"]
    for t in g["tags"]:
        assert [idx[id(m)] for m in cs.search_by_tag(t["tag"])] == t["result"], t["tag"]
    cs.close()
