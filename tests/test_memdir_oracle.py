"""CPU suite: the Memdir oracle (restated search.py / filter.py / utils.py) against the golden
results recorded from the unmodified reference; host-side query parsing of the product."""
import contextlib
import io

import pytest

from oracle import memdir_oracle as mo
from tests.memdir_util import build_tree, key_of, same_modulo_ties


@pytest.fixture(scope="module")
def tree(tmp_path_factory):
    base = str(tmp_path_factory.mktemp("memdir") / "Memdir")
    g = build_tree(base)
    return base, g


def _conds(c):
    return [{"field": f, "operator": op, "value": v} for f, op, v in c]


def test_listing_order_and_skipped_files(tree):
    base, g = tree
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        mems = mo.listing(base, None, None, True)
    assert same_modulo_ties([key_of(m) for m in mems], g["listing"])
    assert "adv00011" in buf.getvalue() and "Error processing" in buf.getvalue()      # invalid UTF-8 file reported + skipped
    assert sorted(mo.memdir_folders(base)) == sorted(g["folders"])


def test_search_results_match_reference(tree):
    base, g = tree
    for q in g["queries"]:
        with contextlib.redirect_stdout(io.StringIO()):
            mems = mo.listing(base, q["folders"], q["statuses"], q["include_content"])
        got = [key_of(mems[i]) for i in mo.run_search(mems, _conds(q["conditions"]))]
        assert same_modulo_ties(got, q["result"]), q["name"]


def test_raising_queries(tree):
    base, g = tree
    with contextlib.redirect_stdout(io.StringIO()):
        mems = mo.listing(base, None, None, False)
    for q in g["raising"]:
        with pytest.raises(TypeError):
            mo.run_search(mems, _conds(q["conditions"]))


def test_filter_statistics_match_reference(tree):
    from tests.golden.make_golden_memdir import FILTERS_EXTRA
    base, g = tree
    defaults = [
        {"name": "Python Content", "conditions": [("Tags", r"python", False), ("content", r"python|django|flask", True)], "actions": [{"type": "move"}, {"type": "flag"}]},
        {"name": "AI Content", "conditions": [("Tags", r"ai|machine[- ]learning|neural|llm", False)], "actions": [{"type": "move"}]},
        {"name": "Learning Content", "conditions": [("Tags", r"books|reading|learning", False), ("Subject", r"books|read|learning", False)], "actions": [{"type": "move"}]},
        {"name": "High Priority", "conditions": [("Priority", r"high", False)], "actions": [{"type": "flag"}]},
        {"name": "Completed Items", "conditions": [("Status", r"completed|done|archived", False)], "actions": [{"type": "move"}, {"type": "flag"}]},
        {"name": "Trash Items", "conditions": [("Tags", r"trash|delete|remove", False)], "actions": [{"type": "move"}]},
    ]
    filters = [{"name": f["name"], "actions": f["actions"], "conditions": [{"field": a, "pattern": b, "negate": c} for a, b, c in f["conditions"]]}
               for f in defaults + FILTERS_EXTRA]
    for run in g["filters"]:
        statuses = run["statuses"] or ["new"]
        with contextlib.redirect_stdout(io.StringIO()):
            mems = mo.listing(base, None, statuses, True)
        stats = mo.run_filters(mems, filters)
        want = run["stats"]
        for k in ("total_memories", "filters_applied", "actions_taken", "memories_modified"):
            assert stats[k] == want[k], (run["statuses"], k)
        assert sorted(d["memory_id"] for d in stats["details"]) == sorted(d["memory_id"] for d in want["details"])
        by_id = {d["memory_id"]: d for d in want["details"]}
        for d in stats["details"]:
            assert d["filters_applied"] == by_id[d["memory_id"]]["filters_applied"] and d["subject"] == by_id[d["memory_id"]]["subject"]


def test_parse_search_args_matches_reference():
    """Host-side query grammar of the product (fei_b200/memdir_tools/search.py) vs the reference's output."""
    from fei_b200.memdir_tools.search import parse_search_args
    from tests.conftest import load_golden
    for case in load_golden("memdir_golden.json")["parse"]:
        q = parse_search_args(case["input"])
        assert q.conditions == case["conditions"], case["input"]
        assert (q.sort_by, q.sort_reverse, q.limit, q.offset, q.include_content) == \
               (case["sort_by"], case["sort_reverse"], case["limit"], case["offset"], case["include_content"]), case["input"]


def test_public_signatures_match_reference():
    """Drop-in contract: same parameter names, kinds, order and defaults as the reference's entry points."""
    import importlib
    import inspect
    from tests.conftest import load_golden
    sigs = load_golden("memdir_golden.json")["signatures"]
    for name, want in sigs.items():
        mod, _, attr = name.partition(".")
        obj = importlib.import_module(f"fei_b200.memdir_tools.{mod}")
        for part in attr.split("."):
            obj = getattr(obj, part)
        got = [[p.name, int(p.kind), None if p.default is inspect.Parameter.empty else repr(p.default)]
               for p in inspect.signature(obj).parameters.values()]
        if name == "memorychain.MemoryBlock.mine_block":        # ours appends an optional `max_tries`
            got = got[:len(want)]
        assert got == want, (name, got, want)


def _write_stand_in(root, layout):
    """A `memdir_tools` package shaped like the reference (tests/golden/dropin_layout.json, recorded from it): the same modules,
    functions, classes with their methods, values, and names imported between modules; every body is a placeholder."""
    pkg = root / "memdir_tools"
    pkg.mkdir()
    for name, m in layout["modules"].items():
        by_src = {}
        for k, src in m["imports"].items():
            by_src.setdefault(src.rpartition(".")[2], []).append(k)
        lines = [f"from .{src} import {', '.join(names)}" for src, names in by_src.items()]
        lines += [f"def {f}(*args, **kwargs):\n    return None" for f in m["functions"]]
        for c, methods in m["classes"].items():
            lines.append(f"class {c}:\n" + "".join(f"    def {f}(self, *args, **kwargs):\n        return None\n" for f in methods) + "    pass")
        lines += [f"{v} = None" for v in m["values"]]
        (pkg / ("__init__.py" if name == "memdir_tools" else name.rpartition(".")[2] + ".py")).write_text("\n".join(lines) + "\n")


def test_dropin_install_patches_the_reference_package(tmp_path):
    """install() rebinds the entry points of a package laid out like the unmodified reference, including the names other
    modules imported before install(), and leaves everything else alone.  (Running them needs a GPU; the patched functions
    are the ones the gpu suite exercises.)"""
    import os
    import subprocess
    import sys
    from tests.conftest import load_golden
    _write_stand_in(tmp_path, load_golden("dropin_layout.json"))
    code = (
        "import sys, os; d = sys.argv[1]; os.chdir(d); os.environ['HOME'] = d;"
        "sys.path.insert(0, d); sys.path.insert(0, %r); sys.dont_write_bytecode = True;"
        "import memdir_tools as P, memdir_tools.utils as U, memdir_tools.search as S, memdir_tools.filter as F, memdir_tools.memorychain as M;"
        "parse = S.parse_search_args;"
        "import fei_b200.dropin as D; D.install();"
        "assert S.__file__.startswith(d);"
        "assert S.search_memories.__module__ == 'fei_b200.dropin' and F.run_filters.__module__ == 'fei_b200.dropin';"
        "assert F.FilterManager.process_memories.__module__ == 'fei_b200.dropin' and hasattr(F, 'apply_filters');"
        "assert F.MemoryFilter.matches.__module__ == 'fei_b200.dropin';"
        "assert M.MemoryChain.validate_chain.__module__ == 'fei_b200.memdir_tools.memorychain';"
        "assert P.search_memories is S.search_memories and U.search_memories.__module__ == 'fei_b200.dropin';"   # names imported before install() are rebound
        "assert S.parse_search_args is parse and P.parse_search_args is parse; print('patched')"
    ) % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code, str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "patched" in out.stdout, out.stderr[-2000:]


def test_oracle_next_rows_match_reference(tree):
    """The oracle's restatements of the "next" rows (legacy substring search, folder statistics, archiver criteria) against
    the reference-generated goldens; the archiver's single-record host form against the oracle."""
    import contextlib, io
    base, g = tree
    with contextlib.redirect_stdout(io.StringIO()):
        for case in g["legacy"]:
            mems = mo.listing(base, case["folders"], case["statuses"], True)
            res = mo.legacy_search(mems, case["query"], case["headers_only"])
            assert same_modulo_ties([key_of(m) for m in res], case["result"]), case
            assert [("content" in m) for m in res][:4] == case["has_content_key"]
        listing = mo.listing(base, None, None, True)
        from fei_b200.memdir_tools.archiver import MemoryArchiver
        arch = MemoryArchiver()
        for c in g["criteria"]:
            got = [key_of(m) for m in listing if mo.matches_criteria(m, c["criteria"])]
            assert same_modulo_ties(got, c["result"]), c["criteria"]
            assert [arch._memory_matches_criteria(m, c["criteria"]) for m in listing] == [mo.matches_criteria(m, c["criteria"]) for m in listing]
        # folder statistics need the special folders the reference manager creates before it counts (ensure_memdir_structure)
        from fei_b200.memdir_tools import utils as U
        U.set_memdir_base(base); U.ensure_memdir_structure()
        for case in g["folder_stats"]:
            st = mo.folder_stats(base, case["folder_path"], case["include_subfolders"])
            ref = case["stats"]
            for k in ("folder", "total_memories", "memory_counts", "flag_counts"):
                assert st[k] == ref[k], (case["folder_path"], k)
            assert st["tags"] == ref["tags"]
            assert sorted(st["subfolders"], key=lambda x: x["folder"]) == sorted(ref["subfolders"], key=lambda x: x["folder"])
