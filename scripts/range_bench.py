"""Range search (radius < score <= range_filter) against the plain search on the same collection, timed alternately
(range, plain with the one-kernel search on, plain with it off, range, ...) in one process.

Collections: 10M x 768 bf16 and one f32+f16 line (synthetic rows), and the templated corpus (16 384-row topic runs).
Cases, k = 10 and 100, batches 1 / 16 / 128 / 4096:
  floor      radius = the median over the batch of each query's 1000th score (about 1 000 rows per query in the window)
  ceiling    range_filter = the median of each query's 1000th score (each query's top ~1 000 rows excluded)
  templated  range_filter 0.02 under the lowest score of the query's own topic run (16 384 near-duplicates excluded)
For every point: ms per call (CUDA events around one search_device call, median over --reps), path, queries_rescanned.
Parity on every timed call: ids and score bits equal the exact answer over the window as the ENGINE's own plain search
gives it (not an external oracle, out of reach at 10M x 768; the plain search is checked against the oracle by the test
suite): one exact plain search per point with a larger k, its hits restricted to the window (the script checks that this
list reaches past the window's k-th row) - or, on the templated corpus, a filtered search without the query's topic run,
after checking that every row outside the run scores at most range_filter.  The card's name and power limit are read in the same run.

    python scripts/range_bench.py [--rows 10000000] [--out profiles/r04/range.json]
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


def window_ref(ids, sc, k, radius, rf):
    """Top k of an exact plain answer restricted to radius < s <= rf; checks that the list covers the window's k-th row."""
    r32, f32 = np.float32(radius), np.float32(rf)
    out_i = np.full((len(ids), k), -1, np.int64)
    out_s = np.full((len(ids), k), -np.inf, np.float32)
    for q in range(len(ids)):
        ok = (sc[q] > r32) & (sc[q] <= f32) & (ids[q] >= 0)
        sel = np.flatnonzero(ok)[:k]
        exhausted = ids[q, -1] < 0 or sc[q, -1] <= r32
        assert len(sel) == k or exhausted, f"reference list too short for query {q}"
        out_i[q, :len(sel)], out_s[q, :len(sel)] = ids[q, sel], sc[q, sel]
    return out_i, out_s


def same(got, want):
    gi, gs = got[0].cpu().numpy(), got[1].cpu().numpy()
    return bool(np.array_equal(gi, want[0]) and np.array_equal(gs.view(np.uint32), want[1].view(np.uint32)))


def measure(idx, q, k, radius, rf, want, reps):
    plain = lambda: idx.search_device(q, k)   # noqa: E731
    rng = lambda: idx.search_device(q, k, radius=radius, range_filter=rf)   # noqa: E731
    t = {"range": [], "plain_fused": [], "plain_nofused": []}
    parity, stats = True, None
    for rep in range(reps + 1):           # rep 0 warms every shape up
        idx.set_fused(True)
        ms, out = timed(rng)
        st = idx.stats()
        parity &= same(out, want)
        if rep:
            t["range"].append(ms)
            stats = {"path": st["path"], "queries_rescanned": st["queries_rescanned"]}
        ms, _ = timed(plain)
        if rep:
            t["plain_fused"].append(ms)
        idx.set_fused(False)
        ms, _ = timed(plain)
        if rep:
            t["plain_nofused"].append(ms)
    idx.set_fused(True)
    med = {key: statistics.median(v) for key, v in t.items()}
    return {"ms": med, "range_over_plain_fused": med["range"] / med["plain_fused"],
            "range_over_plain_nofused": med["range"] / med["plain_nofused"], "parity": parity, **stats}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batches", default="1,16,128,4096")
    ap.add_argument("--out", default="profiles/r04/range.json")
    a = ap.parse_args()
    batches = [int(b) for b in a.batches.split(",")]
    report = {"gpu": gpu_info(), "rows": a.rows, "dim": a.dim, "reps": a.reps, "points": []}
    print(json.dumps(report["gpu"]), flush=True)
    qall = torch.from_numpy(synth_rows(4242, 0, max(batches), a.dim)).cuda()
    for dtype, ks, bs in (("bf16", (10, 100), batches), ("f32+f16", (10,), batches)):
        idx = build(a.rows, a.dim, 4141, dtype)
        for k in ks:
            for nq in bs:
                q = qall[:nq].contiguous()
                ids, sc = (t.cpu().numpy() for t in idx.search_device(q, 1000))
                cut = float(np.median(sc[:, 999]))
                wide_i, wide_s = (t.cpu().numpy() for t in idx.search_device(q, 4096))
                for case, radius, rf in (("floor", cut, None), ("ceiling", None, cut)):
                    want = window_ref(wide_i, wide_s, k, -np.inf if radius is None else radius, np.inf if rf is None else rf)
                    p = {"dtype": dtype, "case": case, "k": k, "batch": nq, **measure(idx, q, k, radius, rf, want, a.reps)}
                    report["points"].append(p)
                    print(json.dumps(p), flush=True)
        idx.close()
        torch.cuda.empty_cache()
    # templated corpus: each query is a noisy copy of a run's centre, range_filter under that run
    topic_rows = 16384
    idx = build(a.rows, a.dim, 700, "bf16", topics=topic_rows)
    n_topics = a.rows // topic_rows
    for nq in batches:
        if nq > n_topics:
            continue
        rng = np.random.default_rng(nq)
        topics = rng.choice(n_topics - 1, nq, replace=False)
        q = torch.from_numpy(np.stack([idx.read_rows(int(t) * topic_rows + 7, 1)[0] for t in topics])).cuda()
        q = q + 0.01 * torch.from_numpy(synth_rows(4343, 0, nq, a.dim)).cuda()
        def run_of(t):
            run = np.zeros(len(idx), bool)
            run[int(t) * topic_rows:(int(t) + 1) * topic_rows] = True
            return run
        rf = np.inf
        for i, t in enumerate(topics):           # the lowest score of each query's own run sets range_filter
            _, rs = idx.search(q[i:i + 1].cpu().numpy(), topic_rows, allow=run_of(t))
            rf = min(rf, float(rs.min()) - 0.02)
        rf = float(np.float32(rf))
        want_i = np.full((nq, 100), -1, np.int64)
        want_s = np.full((nq, 100), -np.inf, np.float32)
        for i, t in enumerate(topics):           # the best rows without the run: the answer, once nothing else is above rf
            oi, os_ = idx.search(q[i:i + 1].cpu().numpy(), 100, allow=~run_of(t))
            assert os_[0, 0] <= np.float32(rf), "a row outside the run scores above range_filter"
            want_i[i], want_s[i] = oi[0], os_[0]
        for k in (10, 100):
            p = {"dtype": "bf16", "case": "templated", "k": k, "batch": nq,
                 **measure(idx, q, k, None, rf, (want_i[:, :k].copy(), want_s[:, :k].copy()), a.reps)}
            report["points"].append(p)
            print(json.dumps(p), flush=True)
    idx.close()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
