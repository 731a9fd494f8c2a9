"""Grouping search (group_by) against the plain search of the same queries, timed alternately (grouped, plain, grouped, ...)
in one process, median of --reps calls each.

Collections: 10M x 768 synthetic rows in bf16 and f32+f16, and the templated corpus (16 384-row topic runs, bf16).
Code layouts: runs of 16 rows (625 000 groups: a document's chunks), 1 000 random groups, and on the templated corpus its
16 384-row runs.  k = 10 and 100, batches 1 / 16 / 128.  Each point: ms per call (CUDA events around one search_device call),
stats path and queries_rescanned.

Every timed grouped call is checked against the engine's plain exact search of the same queries with k' = 16 384: that list
is an exact prefix of each query's ordering, so when it holds at least k distinct groups its first k distinct groups, each at
its first row, are the grouped answer (ids and score bits compared).  Where it holds fewer (the templated runs), the query
is recorded as not checkable at this size instead of passing.  The card's name and power limit are read in the same run.

Targets (from the large-k pipeline's cost, not measured beforehand): batch 1, k = 10, runs of 16 at most 1.3x the plain
search of the same call; batch 16 at most 2x.  Batch 128 is reported without a target.

    python scripts/group_bench.py [--rows 10000000] [--reps 5] [--out profiles/r05/grouped.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import ragfin_b200  # noqa: E402
from ragfin_b200.synthetic import synth_rows  # noqa: E402

KP = 16384   # the plain exact list the answers are checked against


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def build(rows, dim, seed, dtype, topics=0):
    idx = ragfin_b200.Index(dim, dtype, capacity=rows, device=0)
    for r in range(0, rows, 1_000_000):
        m = min(1_000_000, rows - r)
        if topics:
            idx.add_synthetic_topics(seed, r, m, topics, 3)
        else:
            idx.add_synthetic(seed, r, m)
    torch.cuda.synchronize()
    return idx


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def check(got, plain_kp, codes, k):
    """Per query: True (matches the first k distinct groups of the exact k' list), False (differs) or None (the list holds
    fewer than k distinct groups: not checkable at this size)."""
    gi, gs = (t.cpu().numpy() for t in got)
    pi, ps = plain_kp
    out = []
    for i in range(len(gi)):
        rows = pi[i][pi[i] >= 0]
        _, first = np.unique(codes[rows], return_index=True)
        first = np.sort(first)
        if len(first) < k:
            out.append(None)
            continue
        sel = first[:k]
        out.append(bool(np.array_equal(gi[i], rows[sel]) and np.array_equal(gs[i].view(np.uint32), ps[i][sel].view(np.uint32))))
    return out


def run_points(idx, label, queries, layouts, ks, batches, reps, dev):
    res = []
    for lname, codes in layouts:
        ng = int(codes.max()) + 1
        gd = torch.from_numpy(codes).to(dev)
        for nb in batches:
            q = queries[:nb]
            kp = idx.search_device(q, KP)
            torch.cuda.synchronize()
            plain_kp = tuple(t.cpu().numpy() for t in kp)
            for k in ks:
                idx.search_device(q, k, group_by=gd, n_groups=ng)   # warm-up of both shapes
                idx.search_device(q, k)
                torch.cuda.synchronize()
                tg, tp, checks, rescanned = [], [], [], []
                for _ in range(reps):
                    ms, got = timed(lambda: idx.search_device(q, k, group_by=gd, n_groups=ng))
                    st = idx.stats()
                    tg.append(ms)
                    rescanned.append(st["queries_rescanned"])
                    assert st["path"] == 2, st
                    checks += check(got, plain_kp, codes, k)
                    ms, _ = timed(lambda: idx.search_device(q, k))
                    tp.append(ms)
                n_bad = sum(c is False for c in checks)
                p = {"collection": label, "layout": lname, "n_groups": ng, "batch": nb, "k": k,
                     "grouped_ms": statistics.median(tg), "plain_ms": statistics.median(tp),
                     "ratio": statistics.median(tg) / statistics.median(tp), "grouped_ms_all": tg, "plain_ms_all": tp,
                     "queries_rescanned": max(rescanned), "checked_calls_queries": sum(c is True for c in checks),
                     "not_checkable_queries": sum(c is None for c in checks), "mismatched_queries": n_bad}
                if nb == 1 and k == 10 and lname == "runs of 16":
                    p["target"] = "<= 1.3x plain"
                    p["target_met"] = p["ratio"] <= 1.3
                elif nb == 16:
                    p["target"] = "<= 2x plain"
                    p["target_met"] = p["ratio"] <= 2.0
                print(json.dumps({k_: v for k_, v in p.items() if not k_.endswith("_all")}), flush=True)
                assert n_bad == 0, p
                res.append(p)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="profiles/r05/grouped.json")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = gpu_info()
    print(json.dumps(info), flush=True)
    rng = np.random.default_rng(5)
    layouts = [("runs of 16", (np.arange(a.rows) // 16).astype(np.int32)),
               ("1000 random groups", rng.integers(0, 1000, a.rows).astype(np.int32))]
    queries = torch.from_numpy(synth_rows(4242, 0, 128, a.dim)).to(dev)
    points = []
    for dtype in ("bf16", "f32+f16"):
        idx = build(a.rows, a.dim, 4241, dtype)
        points += run_points(idx, f"{a.rows} x {a.dim} {dtype}", queries, layouts, (10, 100), (1, 16, 128), a.reps, dev)
        idx.close()
        torch.cuda.empty_cache()
    topic = 16384
    idx = build(a.rows, a.dim, 4243, "bf16", topics=topic)
    # queries near the centres of 128 different topic runs (noise 2^-2): their own run is 16 384 near-duplicates
    from ragfin_b200.synthetic import synth_topic_rows
    runs = rng.choice(a.rows // topic, 128, replace=False)
    tq = np.concatenate([synth_topic_rows(4243, int(r) * topic + 7, 1, a.dim, topic, 2, synth_rows) for r in runs])
    tlay = [("templated runs of 16384", (np.arange(a.rows) // topic).astype(np.int32))]
    points += run_points(idx, f"{a.rows} x {a.dim} bf16 templated", torch.from_numpy(tq).to(dev), tlay, (10, 100), (1, 16, 128), a.reps, dev)
    idx.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"gpu": info, "script": "scripts/group_bench.py", "reps": a.reps, "points": points}, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
