#!/usr/bin/env python3
"""Cost of ordering and paging search results (fei_sort_rows, PackedMemdir.sort_page); one JSON line on stdout.

  (a) device only: a fei_corpus_synth corpus of --records records, every record a row (the hits of a query matching all);
      sorted by Subject (header, several 7-byte refinement rounds), by date (the wall column) and by Priority; kernel time
      from CUDA events (fei_sort_info.ms), best of --reps, rounds and rows per second;
  (b) end to end on an on-disk tree of --files files: warm search_memories(Tags has_tag python, with_content, limit=10) with and
      without sort_by="Subject", and in the same process the path it replaces (materialise every hit, dict sort, slice),
      the arms alternating.

    python tools/prof_sort.py [--records 10000000] [--files 1000000] [--reps 3]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fei_b200 import _abi, synth                                # noqa: E402


def gpu_identity():
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in out.stdout.strip().split(",")[:2]]
    return name, power


def device_only(n, reps):
    from fei_b200.corpus import Corpus
    from fei_b200.packer import _slot_prog
    c = Corpus().synth(0x5047, 0, n)
    rows = np.arange(n, dtype=np.uint64)
    rc = np.zeros(n, dtype=np.uint32)
    out = {}
    for name, kw in (("Subject", dict(source=_abi.SORT_SLOT, prog=_slot_prog("Subject", 0))), ("date", dict(source=_abi.SORT_WALL)),
                     ("Priority", dict(source=_abi.SORT_SLOT, prog=_slot_prog("Priority", 0)))):
        _abi.sort_rows([c], rc, rows, count=10, **kw)             # warm-up
        best, wall = None, None
        for _ in range(reps):
            t0 = time.perf_counter()
            _, info = _abi.sort_rows([c], rc, rows, count=10, **kw)
            t1 = time.perf_counter()
            if best is None or info.ms < best.ms:
                best, wall = info, (t1 - t0) * 1e3
        out[name] = {"rows": n, "kernel_ms": round(best.ms, 3), "call_ms": round(wall, 3), "rounds": best.rounds,
                     "radix_passes": best.radix_passes, "refined_rows": best.refined_rows, "rows_per_s": round(n / (best.ms / 1e3))}
    c.close()
    return out


def _old_key(mem, field):
    """The removed host sort key (search.py:97-139) for a plain header field."""
    low = field.lower()
    for k, v in mem["headers"].items():
        if k.lower() == low:
            return v
    return None


def end_to_end(n_files, reps):
    from fei_b200 import packer
    from fei_b200.memdir_tools import search as S
    from fei_b200.memdir_tools import utils as U
    tmp = tempfile.mkdtemp(prefix="prof_sort_")
    try:
        base = os.path.join(tmp, "Memdir")
        synth.write_memdir_native(base, 0x5047, 0, n_files)
        U.set_memdir_base(base)

        def query(sort):
            q = S.SearchQuery().add_condition("Tags", "has_tag", "python").with_content(True).set_pagination(10, 0)
            if sort:
                q.set_sort("Subject")
            return q

        def old_path():
            pm = packer.packed()
            with pm.lock:
                q = query(True)
                conds = S.compile_conditions(q.conditions, True, pm)
                hits = S._scan_ranges(pm, conds, pm.ranges(None, None))
                res = pm.materialize(hits, True)
            res.sort(key=lambda x: _old_key(x, "Subject") or "")
            return res[0:10], len(hits)

        arms = {"new_sorted": lambda: S.search_memories(query(True)), "new_unsorted": lambda: S.search_memories(query(False)),
                "old_sorted": lambda: old_path()[0]}
        for f in arms.values():                                  # pack + warm every arm
            f()
        n_hits = old_path()[1]
        assert [m["filename"] for m in arms["new_sorted"]()] == [m["filename"] for m in arms["old_sorted"]()]
        times = {k: [] for k in arms}
        for _ in range(reps):
            for k, f in arms.items():
                t0 = time.perf_counter()
                f()
                times[k].append((time.perf_counter() - t0) * 1e3)
        return {"files": n_files, "hits": n_hits, **{k + "_ms": [round(x, 2) for x in v] for k, v in times.items()}}
    finally:
        packer.drop()
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=10_000_000)
    ap.add_argument("--files", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    _abi.init(0)
    name, power = gpu_identity()
    res = {"gpu": name, "power_limit": power, "device_only": device_only(a.records, a.reps)}
    res["end_to_end"] = end_to_end(a.files, a.reps)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
