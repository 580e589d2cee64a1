#!/usr/bin/env python3
"""bench.py — Memdir scan + Memorychain validation on B200 (one JSON line on stdout).

A "step" is one pass of the hot path over one batch of synthetic input:
  primary workload  BASELINE.json configs[2]: 32-pattern batch `content matches` search over a synthetic Memdir
                    (--entries per GPU, default 10M) resident in HBM; every record body is read once for all 32
                    patterns, hit lists are compacted in listing order; with N>1 the record range is sharded
                    and the step ends with the NCCL all-gatherv of the hit lists.
  extra (N=1)       configs[1] multi-field filter (tags+flags+date+body regex) and configs[3] validate_chain
                    over 1M synthetic blocks, each with its own timing.
`value` = whole-job memories/s with inputs resident in HBM; `e2e` = the same scan through the C ABI from pinned
HOST buffers (upload + tiling + scan + hit lists back) on a --e2e-entries batch per step.
`--impl reference` times the reference's CPU algorithm (oracle port: the reference is pure Python) on the host
cores for the same workload on a bounded sample.
"""
from __future__ import annotations

import argparse
import ctypes as C
import datetime
import json
import os
import re
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
os.environ.setdefault("TZ", "UTC")

import numpy as np  # noqa: E402

SEED = 0xFE1
CHAIN_SEED = 0xC4A1
BATCH32 = ["python", "docker|kubernetes", "neural networks", "react", "angular", "rust", "django", "flask", "terraform", "ansible",
           "microservices", "big data", "ci/cd", "git", "aws|azure|gcp", "spring boot", r"vue\.js", r"node\.js", "devops", "security",
           "blockchain", "testing", "databases", "algorithms", "cloud computing", "mobile development", "computer vision",
           "reinforcement learning", "ui/ux", "web development", "data structures", "machine learning"]
METRIC = "memories_per_sec_scanned"


def measured_peak_field(key, default):
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            return json.load(f).get(key, default)
    except Exception:
        return default


def measured_peak():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, device: int):
        self.rows = []
        self.proc = None
        self.device = device

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill(); out = ""
        sm, mx, reasons = [], [], set()
        for line in out.splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- reference arm / cpu baseline
def _oracle_batch_worker(args):
    seed, first, n, patterns = args
    from fei_b200 import synth
    from oracle import memdir_oracle as mo
    mems = [mo.make_memory(r["filename"], r["folder"], r["status"], synth.file_text(r), True)
            for r in (synth.record(seed, first + k) for k in range(n))]
    t0 = time.perf_counter()
    total = 0
    for p in patterns:                               # the reference runs one search_memories per pattern
        total += len(mo.run_search(mems, [{"field": "content", "operator": "matches", "value": p}]))
    return time.perf_counter() - t0, total


def usable_cores() -> int:
    """Cores this process may really use: scheduler affinity capped by the cgroup CPU quota (os.cpu_count() reports the
    whole machine inside a container)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def cpu_scan_rate(sample: int, cores: int):
    """memories/s of the 32-pattern batch on `cores` host processes (match-only, records already parsed)."""
    if cores <= 1:
        dt, _ = _oracle_batch_worker((SEED, 0, sample, BATCH32))
        return sample / dt, dt
    import multiprocessing as mp
    per = max(1, sample // cores)
    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_oracle_batch_worker, [(SEED, i * per, per, BATCH32) for i in range(cores)])
    dt = max(r[0] for r in res)
    return per * cores / dt, dt


def cpu_chain_rate(nblocks: int):
    from fei_b200 import synth
    from oracle import chain_oracle as co
    chain = co.build_chain(synth.chain_specs(CHAIN_SEED, 0, nblocks))
    t0 = time.perf_counter()
    ok = co.validate(chain)
    dt = time.perf_counter() - t0
    assert ok[0]
    return (nblocks - 1) / dt, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = usable_cores()
    use = max(1, min(cores, 64))
    per_step = 1500 * use                               # bounded sample: 1500 records x 32 passes per worker per step
    times = []
    for step in range(args.warmup + args.steps):
        rate, dt = cpu_scan_rate(per_step, use)
        if step >= args.warmup:
            times.append((rate, dt))
    rate = float(np.mean([r for r, _ in times]))
    ms = float(np.mean([d for _, d in times])) * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "memories/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "memdir 32-pattern batch content search (BASELINE configs[2]) on the host CPU: reference algorithm "
                               "(oracle port of search.py:244-335; the reference is pure Python), match-only over parsed records",
                   "entries_per_step": per_step, "patterns": 32},
        "cpu_baseline": {"value": rate, "unit": "memories/s", "cores": use, "kind": "port",
                         "sample": f"{per_step} synthetic records x 32 single-pattern passes per step, {use} processes (harness-parallelised; the reference itself is single-threaded)"},
        "e2e": {"value": rate, "unit": "memories/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ----------------------------------------------------------------------------- our arm
_REAL_STDOUT = None


def quiet_stdout():
    """stdout carries exactly ONE JSON line: anything libraries print there (NCCL's version banner, ...) goes to stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--entries", type=int, default=0, help="synthetic Memdir entries per GPU (default: 10 M; 12.5 M on 8 GPUs = the 100 M-entry cfg5)")
    ap.add_argument("--e2e-entries", type=int, default=1_000_000, help="records per streamed batch of the end-to-end leg")
    ap.add_argument("--e2e-batches", type=int, default=10, help="batches per end-to-end step (10 x 1 M = the 10 M-entry configuration)")
    ap.add_argument("--parity-entries", type=int, default=500_000, help="records per rank of the sharded-vs-unsharded parity run")
    ap.add_argument("--api-files", type=int, default=1_000_000, help="files of the on-disk Memdir for the Python-API extra")
    ap.add_argument("--chain-blocks", type=int, default=1_000_000)
    ap.add_argument("--cpu-sample", type=int, default=60000)
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (one process, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl ours in a single process")
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not args.entries:
        args.entries = 12_500_000 if world >= 8 else 10_000_000
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        dist = dist_mod
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from fei_b200 import _abi
    from fei_b200.corpus import Corpus
    from fei_b200.program import C_BODY, C_DATE_CMP, C_FLAGS, C_SLOT, CMP, Cond, ProgramBuilder, content_batch_program
    from fei_b200.regexc import Pattern
    lib = _abi.lib()
    _abi.init(local)
    info = _abi.device_info()

    def barrier():
        if dist:
            dist.barrier()

    def allmax(x: float) -> float:
        if not dist:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x: float) -> float:
        if not dist:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    if dist:                                           # library-level NCCL communicator (bootstrap; totals; fallback of the mask exchange)
        import torch
        idbuf = np.zeros(_abi.NCCL_ID_BYTES, dtype=np.uint8)
        if rank == 0:
            _abi.check(lib.fei_comm_unique_id(_abi.ptr(idbuf)))
        t = torch.from_numpy(idbuf).cuda()
        dist.broadcast(t, 0)
        idbuf = t.cpu().numpy()
        _abi.check(lib.fei_comm_init(_abi.ptr(idbuf), world, rank))

    # ---- resident corpus shard: records [rank*entries, (rank+1)*entries)
    t0 = time.perf_counter()
    corpus = Corpus().synth(SEED, rank * args.entries, args.entries)
    gen_s = time.perf_counter() - t0
    st = corpus.stats()
    prog = content_batch_program([Pattern("regex", p, re.IGNORECASE) for p in BATCH32])
    nq = 32
    if dist:
        _abi.check(lib.fei_comm_bind_corpus(corpus.handle))
    p2p = bool(lib.fei_comm_is_p2p()) if dist else False

    def step():
        if dist:                                       # the same scan, the mask all-gather of each finished chunk under the next chunk's scan
            tot = np.zeros(32, dtype=np.uint64)
            _abi.check(lib.fei_comm_scan_gather(corpus.handle, prog, len(prog), _abi.ptr(tot)))
            return tot[:nq]
        return corpus.scan_count(prog, nq)             # k_body in chunks + ordered compaction on the side stream; lists stay on the device

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                                # sampled through warm-up (same workload) and the timed region
        time.sleep(0.3)
    for _ in range(args.warmup):
        step()
    barrier()
    wall0 = time.perf_counter()
    dev_ms = body_ms = compact_ms = 0.0
    launches = 0
    touched = 0
    for _ in range(args.steps):
        totals = step()
        tm = corpus.timing()
        dev_ms += tm["total_ms"]; body_ms += tm["body_ms"]; compact_ms += tm["compact_ms"]
        launches += tm["kernel_launches"]; touched = tm["body_bytes_touched"]
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:                              # before anything else scans: the device still holds the last step's lists
        dump_outputs(args.dump_outputs, corpus, nq, totals, lib, _abi)
    step_ms = allmax(wall * 1e3 / args.steps)         # wall between barriers, max over ranks (includes the exchange)
    dev_step_ms = allmax(dev_ms / args.steps)         # CUDA-event time of the scan calls
    total_entries = allsum(float(args.entries))
    value = total_entries / (step_ms * 1e-3)
    local_hits = corpus.scan_count(prog, nq) if dist else totals
    hits_sum_ok = True
    if dist:                                           # the gathered totals are the sum of the shards' own counts
        import torch
        t = torch.from_numpy(local_hits.astype(np.int64)).cuda()
        dist.all_reduce(t)
        hits_sum_ok = bool((t.cpu().numpy().astype(np.uint64) == totals).all())

    peak, peak_src = measured_peak()
    body_ms_avg = body_ms / args.steps
    algo_bytes = st["body_bytes"] + 8 * st["n"] + 4 * st["n"]       # body text + (record id, length) + hit mask written
    achieved = algo_bytes / (body_ms_avg * 1e-3) / 1e9
    traffic = ncu_traffic_per_entry()
    roofline = {"bound": "hbm", "kernel": "k_body<direct,acc64>", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": int(algo_bytes), "kernel_ms": body_ms_avg,
                "kernel_ms_note": "CUDA events on the compute stream around the kernel's one launch per step (a gate kernel on a second stream "
                                  "releases the compaction of each finished run of windows while it is still scanning); kernel launches per step incl. "
                                  "gates and compaction: %d" % (launches // max(1, args.steps)),
                "bytes_per_memory": algo_bytes / max(1, st["n"]),
                "traffic": int(traffic["bytes_per_entry"] * st["n"]) if traffic else None,
                "traffic_source": (traffic["source"] + ", scaled linearly with entries") if traffic else "no capture",
                "note": "body-only batch: header bytes are not needed by this query and are not read; "
                        "SURVEY 8(d)'s 3626 B/memory figure includes ~152 B of header text"}

    workload = "memdir-32pattern-batch (BASELINE configs[2]): 32 `content matches` regexes, one pass; per step: hit masks + ordered per-query hit lists on the device"
    exchange_how = None
    if world > 1:
        exchange_how = ("the warp that completes a 4096-record window stores its hit masks into every rank's buffer from inside the scan kernel (peer memory over NVLink, CUDA IPC)"
                        if p2p and lib.fei_comm_last_exchange_in_kernel() else
                        "a finished chunk's masks leave with peer-memory copies (copy engines, CUDA IPC) under the next chunk's scan" if p2p else
                        "a finished chunk's masks leave with a grouped ncclBroadcast under the next chunk's scan")
        workload = ("memdir-32pattern-batch over %d range shards (BASELINE configs[4] / cfg5 batch leg): every rank scans its shard (masks + ordered local lists, the "
                    "single-GPU work) and the step ENDS when every rank holds the hit masks of all shards (rank-major = global listing order) and the global "
                    "per-query totals; masks are the wire format because 97-100 %% of the records hit (8 B/hit lists would be 16x larger); the exchange is "
                    "fused into the scan: %s" % (world, exchange_how))
    line = {
        "metric": METRIC, "value": value, "unit": "memories/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload,
                   "entries_per_gpu": args.entries, "entries_total": int(total_entries), "patterns": 32,
                   "corpus_bytes_per_gpu": int(st["body_bytes"] + st["hdr_bytes"]), "parallelism": f"range-shard x{world}",
                   "per_gpu_work_note": "10 M entries per GPU up to 4 GPUs, 12.5 M on 8 (= the 100 M-entry cfg5); memories/s per GPU does not depend on the shard size",
                   "l2": "inputs (tens of GB per GPU) are far larger than the 126 MB L2; no flush needed"},
        "device_ms_per_step": dev_step_ms, "roofline": roofline, "gpu_launches": int(launches),
        "sm_count": info["sm_count"], "corpus_gen_s": gen_s,
        "hits_per_query_min_max": [int(min(totals)), int(max(totals))],
    }
    if clocks is not None:
        line["clocks"] = clocks

    # ---- parity: what the timed steps computed, held against independent computations
    parity = {"gathered_totals_equal_sum_of_shard_counts": hits_sum_ok} if dist else {}
    parity.update(run_parity(args, rank, world, dist, corpus, prog, nq, lib, _abi))
    line["parity"] = parity
    if dist:
        line["multi_gpu"] = run_multi_extra(args, rank, world, dist, corpus, st, lib, _abi, barrier, allmax, step_ms, step)

    # end-to-end through the C ABI from pinned host buffers, every rank on its own batches (own PCIe link)
    barrier()
    e2e = run_e2e(args, corpus, prog, nq, lib, _abi, barrier)
    barrier()
    e2e_ms = allmax(e2e["ms_per_step"])
    e2e_entries = allsum(float(e2e["entries_per_step"]))
    e2e.update({"value": e2e_entries / (e2e_ms * 1e-3), "ms_per_step": e2e_ms, "entries_per_step": int(e2e_entries),
                "h2d_bytes_per_step": int(allsum(float(e2e["h2d_bytes_per_step"]))), "d2h_bytes_per_step": int(allsum(float(e2e["d2h_bytes_per_step"]))),
                "h2d_gbs_measured_min_over_ranks": -allmax(-e2e["h2d_gbs_measured"])})
    line["e2e"] = e2e
    if rank == 0 and world == 1:
        rate, dt = cpu_scan_rate(args.cpu_sample, 1)
        line["cpu_baseline"] = {"value": rate, "unit": "memories/s", "cores": 1, "kind": "port",
                                "sample": f"{args.cpu_sample} synthetic records x 32 single-pattern passes (oracle port of search.py:244-335, match-only), {dt:.1f} s",
                                "host_cores_available": usable_cores(), "host_cores_reported": os.cpu_count()}
        if not args.no_extra:
            try:
                line["extra"] = run_extra(args, corpus, st, peak, lib, _abi)
            except Exception as e:                                 # an extra must not cost the headline line
                import traceback
                line["extra"] = {"error": f"{type(e).__name__}: {e}", "traceback": traceback.format_exc()[-1500:]}
    if dist:
        lib.fei_comm_destroy()
        dist.destroy_process_group()
    if rank == 0:
        emit(line)
    return 0


def ncu_traffic_per_entry():
    """dram__bytes_read + dram__bytes_write per entry of the headline kernel, from the latest `ncu --set full` capture summarised
    under profiles/ (profiles/traffic.json, written by tools/ncu_summary.py --traffic)."""
    try:
        with open(os.path.join(REPO, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return {"bytes_per_entry": float(t["k_body"]["dram_bytes"]) / float(t["k_body"]["entries"]), "source": t["k_body"]["source"]}
    except Exception:
        return None


def batch_cfg2_program(n_total: int):
    """The cfg-2 multi-field query: Tags has_tag python AND flags has_flag F AND date > median AND content matches react|angular."""
    from fei_b200.program import C_BODY, C_DATE_CMP, C_FLAGS, C_SLOT, CMP, Cond, ProgramBuilder
    from fei_b200.regexc import Pattern
    median_ts = 1700000000 + (n_total // 2) // 4
    pb = ProgramBuilder()
    pb.add_query([
        Cond(C_FLAGS, pattern=Pattern("exact_contains", "F")),
        Cond(C_DATE_CMP, op=CMP[">"], i64=median_ts * 1000000),
        Cond(C_SLOT, pattern=Pattern("has_tag", "python"), field="Tags", mode=0),
        Cond(C_BODY, pattern=Pattern("regex", r"react|angular", re.IGNORECASE)),
    ])
    return pb.build()


DUMP_SAMPLE = 1 << 17


def dump_outputs(out_dir, corpus, nq, totals, lib, _abi):
    """What the last timed step hands its caller, as float64 .npy files (every value is an integer below 2**53):
      hit_counts                 [nq]     hits per query
      hit_list_checksums         [nq, 4]  order-sensitive checksums (A, S) of each ordered hit list, in 32-bit halves: A hi, A lo, S hi, S lo
      hit_list_sample_positions  [K]      a fixed seeded sample of K list positions
      hit_list_sample            [nq, K]  the record index at each sampled position of each ordered list, -1 past its end
    The full lists (about 2.5 GB at 10 M entries) are reduced to checksums plus the sample: about 34 MB in all."""
    os.makedirs(out_dir, exist_ok=True)
    counts = np.asarray(totals[:nq], dtype=np.uint64)
    a, s = corpus.list_checksums(nq)
    lo = np.uint64(0xFFFFFFFF)
    checks = np.stack([a >> np.uint64(32), a & lo, s >> np.uint64(32), s & lo], axis=1)
    lists = [np.empty(max(1, int(c)), dtype=np.uint64) for c in counts]
    ptrs = (C.c_void_p * 32)(*[lst.ctypes.data for lst in lists])
    cap = np.zeros(32, dtype=np.uint64)
    cap[:nq] = counts
    _abi.check(lib.fei_scan_fetch_hits(corpus.handle, nq, ptrs, _abi.ptr(cap)))   # copies the resident lists; no scan
    pos = np.sort(np.random.default_rng(SEED).choice(corpus.n, size=min(DUMP_SAMPLE, corpus.n), replace=False))
    sample = np.full((nq, pos.size), -1.0)
    for q in range(nq):
        inside = pos < int(counts[q])
        sample[q, inside] = lists[q][pos[inside]]
    del lists
    for name, arr in (("hit_counts", counts), ("hit_list_checksums", checks), ("hit_list_sample_positions", pos), ("hit_list_sample", sample)):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(arr, dtype=np.float64))


def run_parity(args, rank, world, dist, corpus, prog, nq, lib, _abi):
    """(1) one GPU: the chunked scan against a single-launch scan of the same corpus (order-sensitive checksums of all 32 lists) and
    three 300-record windows of the bench corpus against the oracle (the CPU restatement of the reference, used as the checker);
    (2) N GPUs: a sharded scan + gather of P x N records against an UNSHARDED scan of the same global range on rank 0: per-query totals
    and order-sensitive checksums of the global ordered lists, for the 32-pattern batch (dense wire format) and the cfg-2 query
    (sparse: grouped-broadcast all-gatherv of the lists)."""
    from fei_b200.corpus import Corpus
    out = {}
    if world == 1:
        corpus.scan_count(prog, nq)
        a1, s1 = corpus.list_checksums(nq)
        os.environ["FEI_SCAN_CHUNKS"] = "1"
        c1 = corpus.scan_count(prog, nq)
        a2, s2 = corpus.list_checksums(nq)
        os.environ.pop("FEI_SCAN_CHUNKS")
        out["chunked_scan_equals_single_launch"] = bool((a1 == a2).all() and (s1 == s2).all())
        try:
            from fei_b200 import synth
            from oracle import memdir_oracle as mo
            masks = corpus.scan_masks(prog)
            ok, checked = True, 0
            for start in (0, corpus.n // 3, max(0, corpus.n - 300)):
                recs = [synth.record(SEED, corpus.global_base + start + k) for k in range(min(300, corpus.n - start))]
                mems = [mo.make_memory(r["filename"], r["folder"], r["status"], synth.file_text(r), True) for r in recs]
                for q, p in enumerate(BATCH32):
                    want = set(mo.run_search(mems, [{"field": "content", "operator": "matches", "value": p}]))
                    got = {k for k in range(len(recs)) if (int(masks[start + k]) >> q) & 1}
                    ok = ok and want == got
                checked += len(recs)
            out["sampled_windows_vs_oracle"] = {"records": checked, "patterns": 32, "equal": bool(ok)}
        except Exception as e:                                     # the oracle is test infrastructure; its absence must not cost the line
            out["sampled_windows_vs_oracle"] = {"error": f"{type(e).__name__}: {e}"}
        return out
    P = args.parity_entries
    pc = Corpus().synth(SEED, rank * P, P)
    full = Corpus().synth(SEED, 0, P * world) if rank == 0 else None
    _abi.check(lib.fei_comm_bind_corpus(pc.handle))
    res = {}
    for name, pr, q_n in (("batch32_dense", prog, nq), ("cfg2_query_sparse", batch_cfg2_program(P * world), 1)):
        gt = np.zeros(32, dtype=np.uint64); ga = np.zeros(32, dtype=np.uint64); gs = np.zeros(32, dtype=np.uint64)
        if name == "batch32_dense":
            tot = np.zeros(32, dtype=np.uint64)
            _abi.check(lib.fei_comm_scan_gather(pc.handle, pr, len(pr), _abi.ptr(tot)))
        else:
            pc.scan_count(pr, q_n)
            tot = np.zeros(32, dtype=np.uint64)
            _abi.check(lib.fei_comm_allgather_hits(pc.handle, q_n, None, None, _abi.ptr(tot), None))
        _abi.check(lib.fei_comm_gathered_checksum(q_n, _abi.ptr(gt), _abi.ptr(ga), _abi.ptr(gs)))
        if rank == 0:
            cnt = full.scan_count(pr, q_n)
            fa, fs = full.list_checksums(q_n)
            res[name] = {"entries_total": P * world, "queries": q_n,
                         "totals_equal": bool((cnt == tot[:q_n]).all() and (cnt == gt[:q_n]).all()),
                         "ordered_list_checksums_equal": bool((fa == ga[:q_n]).all() and (fs == gs[:q_n]).all()),
                         "hits": [int(cnt.min()), int(cnt.max())]}
        dist.barrier()
    pc.close()
    if full is not None:
        full.close()
    _abi.check(lib.fei_comm_bind_corpus(corpus.handle))
    out["sharded_vs_unsharded"] = res
    return out


def run_multi_extra(args, rank, world, dist, corpus, st, lib, _abi, barrier, allmax, step_ms, step):
    """cfg5's other leg and the list form of the result: (a) the cfg-2 query on the full shards, exchanged with the sparse grouped-
    broadcast all-gatherv of the compacted lists; (b) the GLOBAL ordered lists of the 32-pattern batch materialised on every rank
    from the gathered masks (what a caller that wants indices rather than masks pays on top of a step)."""
    out = {}
    n_total = args.entries * world
    step(); barrier()                                   # the gathered masks of the batch are the last exchange on every rank again
    gl = np.zeros(32, dtype=np.uint64); lms = C.c_float()
    vals = []
    for _ in range(3):
        _abi.check(lib.fei_comm_global_lists(32, _abi.ptr(gl), C.byref(lms)))
        vals.append(lms.value)
    lists_ms = allmax(float(np.mean(vals[1:])))
    out["global_ordered_lists"] = {"build_ms": lists_ms, "ms_per_step_including_lists": step_ms + lists_ms,
                                   "value_including_lists": n_total / ((step_ms + lists_ms) * 1e-3), "unit": "memories/s",
                                   "list_bytes_per_rank": int(gl.sum()) * 8,
                                   "note": "32 global ordered index lists built on every rank's device from the gathered masks (k_count / k_scan_blocks / k_emit over the rank segments)"}
    pr = batch_cfg2_program(n_total)
    tot = np.zeros(32, dtype=np.uint64)

    def sparse_step():
        corpus.scan_count(pr, 1)
        _abi.check(lib.fei_comm_allgather_hits(corpus.handle, 1, None, None, _abi.ptr(tot), None))
    for _ in range(3):
        sparse_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(10):
        sparse_step()
    barrier()
    ms = allmax((time.perf_counter() - t0) * 1e3 / 10)
    out["cfg2_query_sparse_allgatherv"] = {"ms_per_step": ms, "value": n_total / (ms * 1e-3), "unit": "memories/s", "hits_total": int(tot[0]),
                                           "wire": "counts all-gather + one grouped ncclBroadcast per (rank, query) list segment",
                                           "query": "Tags has_tag python AND flags has_flag F AND date > median AND content matches react|angular"}
    return out


def run_e2e(args, corpus, prog, nq, lib, _abi, barrier):
    """Streaming end to end: `batches` batches of raw records (file contents: header text + '---' + body, as read from disk) go from
    pinned host memory through fei_corpus_load_raw (H2D on the copy stream, then UTF-8 validation / newline folding / split / strip /
    tiling / header directory kernels) and fei_scan_hits (k_body + compaction + 32 ordered hit lists D2H).  Two corpus handles
    rotate, each with its own load stream: batch k+2 is being copied while batch k+1 runs through the pack kernels and batch k is
    scanned and its hits travel back."""
    from concurrent.futures import ThreadPoolExecutor
    from fei_b200.corpus import Corpus
    n = min(args.e2e_entries, corpus.n)
    nb = max(1, args.e2e_batches)
    host = corpus.fetch(0, n)                           # canonical host arrays of the first n records
    hdr, ho, body, bo = host["hdr"].tobytes(), host["hdr_off"], host["body"].tobytes(), host["body_off"]
    parts = []
    for i in range(n):                                  # the file as create_memory_content writes it (utils.py:129-132)
        parts.append(hdr[int(ho[i]):int(ho[i + 1])]); parts.append(b"---\n"); parts.append(body[int(bo[i]):int(bo[i + 1])])
    raw = np.frombuffer(b"".join(parts), dtype=np.uint8).copy()
    raw_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum((ho[1:] - ho[:-1]) + 4 + (bo[1:] - bo[:-1]), out=raw_off[1:])
    del parts, hdr, body
    arrays = {"n": n, "global_base": 0, "raw": raw, "raw_off": raw_off, "ts": host["ts"], "wall": host["wall"], "flags8": host["flags8"],
              "fsb": (host["fsb"] & np.uint32(0x00FFFFFF))}
    pinned = []
    keys = ("raw", "raw_off", "ts", "wall", "flags8", "fsb")
    for k in keys:
        a = arrays[k]
        if lib.fei_host_register(a.ctypes.data, a.nbytes) == 0:
            pinned.append(a)
    h2d = sum(arrays[k].nbytes for k in keys)
    bw_h2d, bw_d2h = C.c_float(), C.c_float()
    barrier()                                           # every rank measures its link while the others use theirs
    _abi.check(lib.fei_host_copy_bench(raw.ctypes.data, min(raw.nbytes, 1 << 30), 3, C.byref(bw_h2d), C.byref(bw_d2h)))
    barrier()
    cs = [Corpus(), Corpus(), Corpus()]                # two batches can be in the load pipeline (one copying, one in the pack kernels) while a third is scanned
    bufs = [np.zeros(n, dtype=np.uint64) for _ in range(nq)]
    for b in bufs:
        if lib.fei_host_register(b.ctypes.data, b.nbytes) == 0:
            pinned.append(b)
    ptrs = (C.c_void_p * 32)(*[b.ctypes.data for b in bufs])
    cap = np.zeros(32, dtype=np.uint64); cap[:nq] = n
    nh = np.zeros(32, dtype=np.uint64)
    pool = ThreadPoolExecutor(2)

    def load(c):
        assert c.load_raw(arrays).all()

    def one_step():
        d2h = 0
        futs = {k: pool.submit(load, cs[k % 3]) for k in range(min(2, nb))}
        for k in range(nb):
            futs.pop(k).result()
            if k + 2 < nb:
                futs[k + 2] = pool.submit(load, cs[(k + 2) % 3])        # handle (k+2)%3 == (k-1)%3: its scan finished in the previous iteration
            _abi.check(lib.fei_scan_hits(cs[k % 3].handle, prog, len(prog), ptrs, _abi.ptr(cap), _abi.ptr(nh)))
            d2h += int(nh[:nq].sum()) * 8
        return d2h
    one_step()                                          # warm-up: allocations, first-touch
    times = []
    d2h = 0
    for _ in range(2):
        barrier()
        t0 = time.perf_counter()
        d2h = one_step()
        times.append(time.perf_counter() - t0)
    pool.shutdown()
    stage = np.zeros(3, dtype=np.float32)
    stages_all = []
    for back in range(min(3, nb) - 1, -1, -1):                      # the last three batches of the step, oldest first (one per handle)
        _abi.check(lib.fei_corpus_last_load_timing(cs[(nb - 1 - back) % 3].handle, _abi.ptr(stage)))
        stages_all.append({"batch": nb - 1 - back, "text_h2d_ms": float(stage[0]), "pack_kernels_ms": float(stage[1]), "text_h2d_gbs": float(stage[2])})
    for a in pinned:
        lib.fei_host_unregister(a.ctypes.data)
    for c in cs:
        c.close()
    dt = float(np.mean(times))
    return {"value": n * nb / dt, "unit": "memories/s", "entries_per_step": n * nb, "batches_per_step": nb, "ms_per_step": dt * 1e3,
            "h2d_bytes_per_step": int(h2d) * nb, "d2h_bytes_per_step": int(d2h),
            "h2d_gbs_achieved": h2d * nb / dt / 1e9, "h2d_gbs_measured": float(bw_h2d.value), "d2h_gbs_measured": float(bw_d2h.value),
            "frac_of_measured_h2d": (h2d * nb / dt / 1e9) / float(bw_h2d.value) if bw_h2d.value else None,
            "last_batch_device_stages": {"text_h2d_ms": float(stage[0]), "pack_kernels_ms": float(stage[1]), "text_h2d_gbs": float(stage[2]),
                                         "note": "CUDA events on the batch's load stream; the copy runs while the previous batch is packed and the one before it is scanned"},
            "last_three_batches_device_stages": stages_all,
            "path": "pinned host buffers of raw file contents -> fei_corpus_load_raw (H2D + ingest + tiling + header directory, copy stream) "
                    "|| fei_scan_hits of the previous batch (k_body + compaction + 32 ordered hit lists D2H, compute stream); "
                    "%d batches of %d records per step (the same pinned batch is re-sent: every batch is copied, packed and scanned anew)" % (nb, n)}


def api_on_disk(n_files: int):
    """The drop-in entry points end to end on an on-disk Memdir of n_files files (page-cached): cold = native listing + multi-threaded
    reads + GPU pack + scan; warm = the packed corpus is reused (inotify says nothing changed); then one new file (incremental
    sync), a snapshot save / restore, and the oracle (the reference's algorithm on one host core) on a sub-tree for the per-file rate."""
    import contextlib, io, shutil, tempfile
    from fei_b200 import packer, synth
    from fei_b200.memdir_tools import filter as gfilter, search as gsearch, utils as gutils
    from oracle import memdir_oracle as mo
    scratch = tempfile.mkdtemp(prefix="feiscan_bench_")
    try:
        base = os.path.join(scratch, "Memdir")
        t0 = time.perf_counter()
        synth.write_memdir_native(base, SEED, 0, n_files)
        write_s = time.perf_counter() - t0
        gutils.set_memdir_base(base)
        q = gsearch.SearchQuery(); q.add_condition("content", "matches", r"kubernetes.*docker|docker.*kubernetes"); q.add_condition("Tags", "has_tag", "python")
        q.with_content(True)
        q0 = gsearch.SearchQuery(); q0.add_condition("content", "matches", r"quagga.*zebra")          # no hits: the cost without materialisation
        sink = io.StringIO()
        with contextlib.redirect_stdout(sink):
            t0 = time.perf_counter(); cold = gsearch.search_memories(q); cold_s = time.perf_counter() - t0
            pm = packer.packed()
            cold_stages = dict(pm.timing)
            warm, warm0 = [], []
            for _ in range(5):
                t0 = time.perf_counter(); res = gsearch.search_memories(q); warm.append(time.perf_counter() - t0)
                t0 = time.perf_counter(); gsearch.search_memories(q0.with_content(True)); warm0.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); stats = gfilter.apply_filters(dry_run=True); filt_first_s = time.perf_counter() - t0     # compiles the filters' automata
            t0 = time.perf_counter(); stats = gfilter.apply_filters(dry_run=True); filt_s = time.perf_counter() - t0
            gutils.save_memory(".Projects/AI", "fresh body about kubernetes and docker", {"Tags": "python,new", "Subject": "fresh"}, "P")
            t0 = time.perf_counter(); res2 = gsearch.search_memories(q); inc_s = time.perf_counter() - t0
            inc = {"ms": inc_s * 1e3, "files_read": pm.files_read, "windows_packed": pm.windows_packed, "hits": len(res2)}
            snap = os.path.join(scratch, "snap")
            t0 = time.perf_counter(); pm.save_snapshot(snap); save_s = time.perf_counter() - t0
            snap_bytes = os.path.getsize(snap + ".corpus")
            packer.drop()
            t0 = time.perf_counter(); pm2 = packer.PackedMemdir.from_snapshot(base, snap); load_s = time.perf_counter() - t0
            packer._cache[base] = pm2
            t0 = time.perf_counter(); res3 = gsearch.search_memories(q); resync_s = time.perf_counter() - t0
            snapshot = {"bytes": snap_bytes, "save_s": save_s, "restore_s": load_s, "restore_gbs_device_events": pm2.snapshot_gbs,
                        "restore_gbs_wall": snap_bytes / load_s / 1e9, "first_query_after_restore_s": resync_s, "files_read_after_restore": pm2.files_read,
                        "hits": len(res3)}
            sub_f, sub_s = [".Projects/AI"], ["new"]
            t0 = time.perf_counter()
            mems = mo.listing(base, sub_f, sub_s, True)
            want = mo.run_search(mems, [{"field": f, "operator": op, "value": v} for f, op, v in (("content", "matches", r"kubernetes.*docker|docker.*kubernetes"), ("Tags", "has_tag", "python"))])
            cpu_s = time.perf_counter() - t0
            sub = gsearch.search_memories(q, sub_f, sub_s)
        assert len(cold) == len(res) and len(res2) == len(res) + 1 and len(res3) == len(res2)
        assert [m["filename"] for m in sub] == [mems[i]["filename"] for i in want], "API result differs from the oracle on the sub-tree"
        return {"files": n_files, "write_tree_s": write_s, "query": "content matches kubernetes.*docker|docker.*kubernetes AND Tags has_tag python (with_content)",
                "search_memories_cold_s": cold_s, "cold_stages": cold_stages, "search_memories_warm_ms": float(np.median(warm)) * 1e3, "hits": len(res),
                "search_memories_warm_no_hits_ms": float(np.median(warm0)) * 1e3,
                "materialisation_ms_per_1k_hits": (float(np.median(warm)) - float(np.median(warm0))) * 1e3 / max(1, len(res)) * 1000,
                "apply_filters_default_dry_run_first_ms": filt_first_s * 1e3, "apply_filters_default_dry_run_warm_ms": filt_s * 1e3,
                "apply_filters_stats": {k: stats.get(k) for k in ("total_memories", "filters_applied", "actions_taken", "memories_modified")},
                "incremental_one_new_file": inc, "snapshot": snapshot, "host_cores": usable_cores(), "read_threads": packer.READ_THREADS,
                "cpu_oracle_subtree": {"files": len(mems), "s": cpu_s, "memories_per_s": len(mems) / cpu_s,
                                       "note": "oracle: lists, reads, parses and matches every file of the sub-tree on one host core, as the reference does on every call"},
                "memories_per_s_warm": n_files / float(np.median(warm)), "memories_per_s_cold": n_files / cold_s}
    finally:
        packer.drop()
        shutil.rmtree(scratch, ignore_errors=True)


def run_extra(args, corpus, st, peak, lib, _abi):
    from fei_b200.program import C_BODY, C_DATE_CMP, C_FLAGS, C_SLOT, CMP, Cond, ProgramBuilder
    from fei_b200.regexc import Pattern
    out = {}
    # ---- configs[1]: multi-field filter: Tags has_tag python AND flags has_flag F AND date > median AND content matches react|angular
    median_ts = 1700000000 + (corpus.global_base + corpus.n // 2) // 4
    pb = ProgramBuilder()
    pb.add_query([
        Cond(C_FLAGS, pattern=Pattern("exact_contains", "F")),
        Cond(C_DATE_CMP, op=CMP[">"], i64=median_ts * 1000000),
        Cond(C_SLOT, pattern=Pattern("has_tag", "python"), field="Tags", mode=0),
        Cond(C_BODY, pattern=Pattern("regex", r"react|angular", re.IGNORECASE)),
    ])
    prog = pb.build()
    for _ in range(3):
        corpus.scan_count(prog, 1)
    ms = []; tm = None
    for _ in range(5):
        cnt = corpus.scan_count(prog, 1)
        tm = corpus.timing(); ms.append(tm["total_ms"])
    t = float(np.mean(ms)) * 1e-3
    head_bytes = 20 * st["n"] + 4 * st["n"]          # meta columns (wall, flags8, fsb) + alive mask; header text is read for survivors only
    out["cfg2_multi_field_filter"] = {
        "metric": METRIC, "value": corpus.n / t, "unit": "memories/s", "entries": corpus.n, "ms": t * 1e3, "hits": int(cnt[0]),
        "head_ms": tm["head_ms"], "body_ms": tm["body_ms"], "compact_ms": tm["compact_ms"],
        "roofline": {"bound": "hbm", "kernel": "k_head_meta+k_head_parse", "achieved": head_bytes / (tm["head_ms"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": head_bytes / (tm["head_ms"] * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": int(head_bytes),
                     "note": "k_head_meta + k_head_parse: meta columns are streamed for every record, header text and body tiles are read only for records that "
                             "survive the earlier predicates (as the reference short-circuits); at this size the pass is launch/latency bound, not HBM bound. "
                             "body tile bytes touched: %d" % tm["body_bytes_touched"]},
        "query": "Tags has_tag python AND flags has_flag F AND date > median AND content matches react|angular",
    }
    # ---- header-only filters over every record (what FilterManager.process_memories runs): three one-field filters in one pass
    pb = ProgramBuilder()
    pb.add_query([Cond(C_SLOT, pattern=Pattern("has_tag", "python"), field="Tags", mode=0)])
    pb.add_query([Cond(C_SLOT, pattern=Pattern("contains", "learning"), field="Subject", mode=0)])
    pb.add_query([Cond(C_SLOT, pattern=Pattern("equals", "high"), field="Priority", mode=0), Cond(C_FLAGS, pattern=Pattern("exact_contains", "F"))])
    progh = pb.build()
    for _ in range(3):
        corpus.scan_count(progh, 3)
    ms = []; tmh = None
    for _ in range(5):
        cnth = corpus.scan_count(progh, 3)
        tmh = corpus.timing(); ms.append(tmh["total_ms"])
    th = float(np.mean(ms)) * 1e-3
    # per record: 20 B meta + 12 B work-list entry written and read + per field (2 B length + the value's 16-byte units, ~32 B) + 4 B alive mask
    hdr_bytes = st["n"] * (20 + 24 + 3 * 34 + 4)
    out["header_filters_3_fields"] = {
        "metric": METRIC, "value": corpus.n / th, "unit": "memories/s", "entries": corpus.n, "ms": th * 1e3, "head_ms": tmh["head_ms"],
        "hits": [int(x) for x in cnth[:3]],
        "roofline": {"bound": "hbm", "kernel": "k_head_meta+k_head_parse", "achieved": hdr_bytes / (tmh["head_ms"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": hdr_bytes / (tmh["head_ms"] * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": int(hdr_bytes),
                     "note": "header fields are read from the value columns built at pack time (hdir.cu): coalesced 16-byte units per record; "
                             "the pass is instruction / latency bound (three short automaton runs per record), not HBM bound"},
        "query": "3 filters in one pass: Tags has_tag python | Subject contains learning | Priority = high AND flags has_flag F",
    }
    # ---- configs[0] at full corpus size: one regex over every body (the common search_memories call)
    pb = ProgramBuilder()
    pb.add_query([Cond(C_BODY, pattern=Pattern("regex", r"kubernetes.*docker|docker.*kubernetes", re.IGNORECASE))])
    prog1 = pb.build()
    for _ in range(3):
        corpus.scan_count(prog1, 1)
    ms = []; bms = []
    for _ in range(5):
        cnt1 = corpus.scan_count(prog1, 1)
        tm1 = corpus.timing(); ms.append(tm1["total_ms"]); bms.append(tm1["body_ms"])
    t1 = float(np.mean(ms)) * 1e-3; b1 = float(np.mean(bms)) * 1e-3
    body_bytes = st["body_bytes"] + 12 * st["n"]
    read1 = int(tm1["body_bytes_read"]) + 12 * st["n"]        # bytes the kernel really requested (early stop per group)
    out["cfg1_single_regex_full_corpus"] = {
        "metric": METRIC, "value": corpus.n / t1, "unit": "memories/s", "entries": corpus.n, "ms": t1 * 1e3, "body_ms": b1 * 1e3, "hits": int(cnt1[0]),
        "roofline": {"bound": "hbm", "kernel": "k_body_sticky", "achieved": read1 / b1 / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": read1 / b1 / 1e9 / peak, "bytes_read_per_launch": read1,
                     "algorithmic_bytes_full_read": int(body_bytes), "algorithmic_rate_GBps": body_bytes / b1 / 1e9,
                     "tile_bytes_of_groups_entered": int(tm1["body_bytes_touched"]),
                     "note": "single-pattern automaton is 'sticky': a group stops being read once all 32 of its records have matched, "
                             "so `achieved` counts the bytes really requested (kernel counter), not the full corpus"},
        "query": "content matches kubernetes.*docker|docker.*kubernetes",
    }
    # same kernel on a pattern that never matches: no early exit, every body byte goes through the DFA
    pb = ProgramBuilder()
    pb.add_query([Cond(C_BODY, pattern=Pattern("regex", r"quagga.*zebra|zebra.*quagga", re.IGNORECASE))])
    prog0 = pb.build()
    for _ in range(3):
        corpus.scan_count(prog0, 1)
    bms = []
    for _ in range(5):
        cnt0 = corpus.scan_count(prog0, 1)
        bms.append(corpus.timing()["body_ms"])
    b0 = float(np.mean(bms)) * 1e-3
    out["single_regex_no_match_full_read"] = {
        "metric": METRIC, "value": corpus.n / b0, "unit": "memories/s (kernel only)", "entries": corpus.n, "body_ms": b0 * 1e3, "hits": int(cnt0[0]),
        "roofline": {"bound": "hbm", "kernel": "k_body_sticky", "achieved": body_bytes / b0 / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": body_bytes / b0 / 1e9 / peak, "algorithmic_bytes_per_launch": int(body_bytes)},
        "query": "content matches quagga.*zebra|zebra.*quagga (no record matches: no early exit)",
    }
    # ---- the drop-in entry points end to end on an on-disk Memdir: search_memories() and apply_filters() of the reference-shaped
    #      Python API (cold = listing + reading + packing + upload + scan; warm = the packed corpus is reused), next to the oracle
    #      (the reference's algorithm: list, read, parse and match every file on one host core)
    try:
        out["python_api_on_disk"] = api_on_disk(args.api_files)
    except Exception as e:                                     # a full scratch disk must not cost the headline line
        out["python_api_on_disk"] = {"error": f"{type(e).__name__}: {e}"}
    # ---- configs[3]: validate_chain over synthetic blocks resident on the device
    ch = C.c_void_p()
    _abi.check(lib.fei_chain_create(C.byref(ch)))
    t0 = time.perf_counter()
    _abi.check(lib.fei_chain_synth(ch, CHAIN_SEED, 0, args.chain_blocks, -1))
    build_s = time.perf_counter() - t0
    fb, kind, kms = C.c_int64(), C.c_int32(), C.c_float()
    for _ in range(3):
        _abi.check(lib.fei_chain_validate(ch, C.byref(fb), C.byref(kind), None, C.byref(kms)))
    ms = []
    for _ in range(10):
        _abi.check(lib.fei_chain_validate(ch, C.byref(fb), C.byref(kind), None, C.byref(kms)))
        ms.append(kms.value)
    t = float(np.mean(ms)) * 1e-3
    nb = args.chain_blocks
    info = _abi.device_info() if hasattr(_abi, "device_info") else {}
    sm_mhz_max = float(measured_peak_field("sm_max_mhz", 1965.0))
    alu_nominal = float(info.get("sm_count", 148)) * 64 * sm_mhz_max * 1e6
    tops, mb_ms = C.c_float(), C.c_float()
    _abi.check(lib.fei_microbench_alu(5, C.byref(tops), C.byref(mb_ms)))       # LOP3 / SHF issue rate of this chip, measured now
    alu_peak = float(tops.value) * 1e12
    cpu_rate, cpu_dt = cpu_chain_rate(min(nb, 50_000))
    out["cfg4_validate_chain"] = {
        "metric": "sha256_chain_blocks_per_sec", "value": (nb - 1) / t, "unit": "chain blocks/s", "blocks": nb, "kernel_ms": t * 1e3,
        "compression_blocks_per_sec": (nb - 1) * 6 / t, "valid": fb.value == -1, "chain_build_s_host": build_s,
        "roofline": {"bound": "int32-issue (not HBM)", "achieved": 493.0 * (nb - 1) / t / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": 493.0 * (nb - 1) / t / 1e9 / peak, "bytes_per_block": 493,
                     "note": "SHA-256 is integer-ALU bound: ~13k 32-bit ops per chain block (6 compressions); HBM fraction is expected to be low"},
        # the bound that applies: ALU-pipe issue (IADD3 / LOP3 / SHF / PRMT run at 64 lanes per clock per SM).  1300 = ALU-pipe
        # instructions per compression in the kernel's SASS (profiles/r1_sass_evidence.txt); ncu reports the pipe 95 % busy.
        "roofline_alu": {"bound": "int32 ALU pipe", "achieved": (nb - 1) * 6 * 1300 / t / 1e12, "unit": "T lane-ops/s",
                         "peak": alu_peak / 1e12, "frac": (nb - 1) * 6 * 1300 / t / alu_peak,
                         "peak_source": "measured: fei_microbench_alu (8 independent LOP3 + SHF chains per thread, %d SMs x 8 CTAs x 256 threads, best of 5, %.3f ms)" % (info.get("sm_count", 148), mb_ms.value),
                         "peak_nominal": alu_nominal / 1e12, "peak_nominal_source": "sm_count x 64 lanes x %.0f MHz (max SM clock)" % sm_mhz_max,
                         "alu_instr_per_compression": 1300, "ncu": "profiles/r1e_k_sha256_validate_1M.txt"},
        "cpu_baseline": {"value": cpu_rate, "unit": "chain blocks/s", "cores": 1, "kind": "port",
                         "sample": f"validate_chain oracle (json.dumps + hashlib, memorychain.py:596-618) over {min(nb, 50_000)} blocks, {cpu_dt:.2f} s"},
    }
    lib.fei_chain_destroy(ch)
    # ---- the same path end to end through the reference-shaped Python API: MemoryChain over nb reference-shaped MemoryBlock objects.
    #      The chain keeps a device image of its blocks (typed columns -> GPU canonical JSON -> SHA-ready blocks), built when the
    #      blocks arrive; validate_chain() re-hashes resident data; an edited block is marshalled again together with its successors.
    from fei_b200 import synth
    from fei_b200.memdir_tools import memorychain as mc
    nb_api = nb
    ch2 = C.c_void_p()
    _abi.check(lib.fei_chain_create(C.byref(ch2)))
    _abi.check(lib.fei_chain_synth(ch2, CHAIN_SEED, 0, nb_api, -1))
    hh = np.zeros(64 * nb_api, dtype=np.uint8); moff = np.zeros(nb_api + 1, dtype=np.uint64)
    _abi.check(lib.fei_chain_fetch(ch2, 0, nb_api, None, 0, _abi.ptr(moff), _abi.ptr(hh), None))
    lib.fei_chain_destroy(ch2)
    hashes = hh.tobytes().decode()
    t0 = time.perf_counter()
    blocks = []                                                            # reference-shaped MemoryBlock objects (plain instance attributes)
    for i, sp in enumerate(synth.chain_specs(CHAIN_SEED, 0, nb_api)):
        b = mc.MemoryBlock(sp["index"], sp["timestamp"], sp["memory_data"], "0" if i == 0 else hashes[64 * i - 64:64 * i], sp["responsible_node"], sp["proposer_node"])
        b.hash = hashes[64 * i:64 * i + 64]
        blocks.append(b)
    objects_s = time.perf_counter() - t0
    t0 = time.perf_counter(); chain_obj = mc.MemoryChain(blocks=blocks); construct_s = time.perf_counter() - t0
    t0 = time.perf_counter(); ok_first = chain_obj.validate_chain(); first_s = time.perf_counter() - t0
    ts = []
    for _ in range(5):
        t0 = time.perf_counter(); ok = chain_obj.validate_chain(); ts.append(time.perf_counter() - t0)
    chain_obj.chain[nb_api // 2].nonce = 7
    t0 = time.perf_counter(); ok_edit = chain_obj.validate_chain(); edit_s = time.perf_counter() - t0
    chain_obj.chain[nb_api // 2].nonce = 0
    os.environ["FEI_CHAIN_RESIDENT"] = "0"
    t0 = time.perf_counter(); ok_oneshot = mc.MemoryChain(blocks=blocks).validate_chain(); oneshot_s = time.perf_counter() - t0
    os.environ.pop("FEI_CHAIN_RESIDENT")
    out["cfg4_validate_chain"]["e2e_python_api"] = {
        "blocks": nb_api, "valid": bool(ok_first and ok), "unit": "chain blocks/s",
        "build_python_block_objects_s": objects_s,
        "chain_construction_s": construct_s, "chain_construction_blocks_per_s": nb_api / construct_s,
        "first_validate_blocks_per_s": (nb_api - 1) / first_s, "first_validate_ms": first_s * 1e3,
        "value": (nb_api - 1) / min(ts), "resident_validate_ms": min(ts) * 1e3,
        "validate_after_editing_the_middle_block": {"ms": edit_s * 1e3, "verdict": bool(ok_edit), "blocks_marshalled_again": nb_api - nb_api // 2},
        "one_shot_validate_without_device_image_blocks_per_s": (nb_api - 1) / oneshot_s, "one_shot_valid": bool(ok_oneshot),
        "path": "MemoryChain(blocks=...): attribute marshal (CPython helper _fastcols) -> typed columns H2D -> k_json_size / k_json_write (canonical JSON incl. "
                "shortest float repr on the GPU) -> padding / link kernels; validate_chain(): k_sha256_validate over the resident image"}
    return out


if __name__ == "__main__":
    sys.exit(main())
