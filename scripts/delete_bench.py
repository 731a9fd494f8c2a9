"""Cost of tombstones: an untouched collection (A) against the same collection with rows deleted (B), timed alternately
(A B A B ...) in one process, plus compaction against a device-to-device copy of the same bytes.

For every point: ms per call (CUDA events around one search_device call, median over --reps), the path taken,
queries_rescanned and, on the one-kernel search, rows rescored per query (-1 = the in-kernel exact scan).  Parity on every
timed call: B's ids and score bits equal those of a compacted copy of B (C), after mapping C's ids back through the
survivors, compared on the device.  The templated corpus (16 384-row topic runs) is searched with the queries' own topic
runs deleted.  The card's name and power limit are read (read-only nvidia-smi query) in the same run.

    python scripts/delete_bench.py [--rows 10000000] [--out profiles/r04/deletes.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import ragfin_b200  # noqa: E402
from ragfin_b200.synthetic import synth_rows, synth_topic_rows  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def build(rows, dim, seed, topics=0, dtype="bf16"):
    idx = ragfin_b200.Index(dim, dtype, capacity=rows, device=0)
    for r in range(0, rows, 1_000_000):
        m = min(1_000_000, rows - r)
        if topics:
            idx.add_synthetic_topics(seed, r, m, topics, 3)
        else:
            idx.add_synthetic(seed, r, m)
    torch.cuda.synchronize()
    return idx


def timed(idx, q, k):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = idx.search_device(q, k)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def describe(idx, nq):
    st = idx.stats()
    d = {"path": st["path"], "queries_rescanned": st["queries_rescanned"]}
    if st["path"] == 3:
        _, resc = idx.fused_counts(nq)
        d["rows_rescored"] = [int(v) for v in resc]
    return d


def measure(a, b, c, survivors_dev, q, k, reps):
    """Warm-up, then reps rounds of A, B in turn; every B result is checked against C's."""
    for idx in (x for x in (a, b, c) if x is not None):
        for _ in range(3):
            idx.search_device(q, k)
    torch.cuda.synchronize()
    ms = {"A": [], "B": []}
    parity = True
    for _ in range(reps):
        if a is not None:
            t, _ = timed(a, q, k)
            ms["A"].append(t)
        t, (bi, bs) = timed(b, q, k)
        ms["B"].append(t)
        ci, cs = c.search_device(q, k)
        mapped = torch.where(ci >= 0, survivors_dev[ci.clamp(min=0)], ci)
        parity &= bool(torch.equal(bi, mapped) and torch.equal(bs.view(torch.int32), cs.view(torch.int32)))
    res = {}
    for name, idx in (("A", a), ("B", b)):
        if idx is None:
            continue
        timed(idx, q, k)
        res[name] = {"ms_median": round(statistics.median(ms[name]), 4), "ms_min": round(min(ms[name]), 4), **describe(idx, q.shape[0])}
    if "A" in res:
        res["B_over_A"] = round(res["B"]["ms_median"] / res["A"]["ms_median"], 4)
    return res, parity


def compaction(idx, rows, dim):
    """ragfin_compact (host clock around the synchronous call: prefix on the host, allocation, gather kernel, free) next to a
    device-to-device copy of the whole matrix (torch copy_ -> cudaMemcpyAsync), both as (bytes read + bytes written) / time;
    plus the gather kernel alone (CUDA events of ragfin_profile): the call also allocates the new matrix and frees the old one."""
    ld = (dim + 7) // 8 * 8
    live = idx.live_count
    idx.profile(True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    survivors = idx.compact()
    t_compact = time.perf_counter() - t0
    kernel_ms, _ = idx.profile_read()
    idx.profile(False)
    moved = (rows + live) * ld * 2
    src = torch.empty(rows * ld, dtype=torch.bfloat16, device="cuda")
    dst = torch.empty_like(src)
    src.fill_(1.0)
    dst.copy_(src)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    t_copy = e0.elapsed_time(e1) * 1e-3
    del src, dst
    torch.cuda.empty_cache()
    r = {"rows": rows, "live": live, "compact_s": round(t_compact, 4), "compact_gb_s": round(moved / t_compact / 1e9, 1),
         "compact_kernel_s": round(kernel_ms * 1e-3, 5), "compact_kernel_gb_s": round(moved / (kernel_ms * 1e-3) / 1e9, 1),
         "d2d_copy_s": round(t_copy, 4), "d2d_copy_gb_s": round(2 * rows * ld * 2 / t_copy / 1e9, 1)}
    r["compact_over_copy_rate"] = round(r["compact_gb_s"] / r["d2d_copy_gb_s"], 3)
    r["compact_kernel_over_copy_rate"] = round(r["compact_kernel_gb_s"] / r["d2d_copy_gb_s"], 3)
    return survivors, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--frac", type=float, default=0.01)
    ap.add_argument("--out", default="profiles/r04/deletes.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    report = {"gpu": gpu_info(), "rows": a.rows, "dim": a.dim, "dtype": "bf16", "deleted_fraction": a.frac, "reps": a.reps,
              "timing": "CUDA events around one search_device call, median; A and B alternate", "points": []}
    dead = np.flatnonzero(np.random.default_rng(77).random(a.rows) < a.frac)
    A, B, C = build(a.rows, a.dim, 1234), build(a.rows, a.dim, 1234), build(a.rows, a.dim, 1234)
    B.delete(dead)
    C.delete(dead)
    survivors, report["compaction"] = compaction(C, a.rows, a.dim)
    print(json.dumps(report["compaction"]), flush=True)
    surv = torch.from_numpy(survivors).cuda()
    parity_all = True
    for nq, k in ((1, 10), (16, 10), (128, 10), (4096, 10), (1, 100), (1, 1000)):
        q = torch.from_numpy(synth_rows(4321, 0, nq, a.dim)).cuda()
        res, parity = measure(A, B, C, surv, q, k, a.reps)
        parity_all &= parity
        report["points"].append({"corpus": "synthetic", "nq": nq, "k": k, "parity_vs_compacted": parity, **res})
        print(json.dumps(report["points"][-1]), flush=True)
    for idx in (A, B, C):
        idx.close()
    del surv
    torch.cuda.empty_cache()
    # templated corpus: the query's own topic run deleted (16 384 near-duplicates that would otherwise all qualify)
    topic_rows = 16384
    # TA: the same corpus untouched (its answers differ: the query's own run is there), timed for the path it takes
    TA, T, TC = (build(a.rows, a.dim, 1234, topics=topic_rows) for _ in range(3))
    run = np.arange(7 * topic_rows, 8 * topic_rows)
    T.delete(run)
    TC.delete(run)
    surv = torch.from_numpy(TC.compact()).cuda()
    q = torch.from_numpy(synth_topic_rows(1234, 7 * topic_rows + 11, 1, a.dim, topic_rows, 2)).cuda()
    for fused in (True, False):
        for idx in (TA, T, TC):
            idx.set_fused(fused)
        res, parity = measure(TA, T, TC, surv, q, 10, a.reps)
        parity_all &= parity
        report["points"].append({"corpus": "templated, query's topic run deleted", "fused": fused, "nq": 1, "k": 10,
                                 "parity_vs_compacted": parity, **res})
        print(json.dumps(report["points"][-1]), flush=True)
    report["parity_all"] = parity_all
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print("parity B == compacted B on every timed call:", parity_all)


if __name__ == "__main__":
    main()
