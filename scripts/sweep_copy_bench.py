"""f32 vs f32+f16 vs bf16 collections built from the same seed, timed alternately (A B C A B C ...) in one process.

For every point: ms per call (CUDA events, median), dominant-kernel ms (ragfin_profile, in a separate profiled pass), sweep
GB/s (bytes of the matrix the sweep streams over the dominant-kernel time), rows rescored by the one-kernel search and
queries_rescanned; plus each type's ingest rate, and a parity check: the ids and score bits of f32+f16 equal those of f32 on
every timed call, compared on the device.  The card's name and power limit are read (read-only nvidia-smi query) in the same
run and written beside the numbers.

    python scripts/sweep_copy_bench.py [--rows 10000000] [--out profiles/r03/sweep_copy.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import ragfin_b200  # noqa: E402
from ragfin_b200.synthetic import synth_rows, synth_topic_rows  # noqa: E402

TYPES = ("f32", "f32+f16", "bf16")
SWEEP_BYTES = {"f32": 4, "f32+f16": 2, "bf16": 2}   # bytes per element the tensor-core sweep streams


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def build(dtype, rows, dim, seed, topics=0):
    idx = ragfin_b200.Index(dim, dtype, capacity=rows, device=0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for r in range(0, rows, 1_000_000):
        m = min(1_000_000, rows - r)
        if topics:
            idx.add_synthetic_topics(seed, r, m, topics, 3)
        else:
            idx.add_synthetic(seed, r, m)
    torch.cuda.synchronize()
    return idx, rows / (time.perf_counter() - t0)


def measure(idxs, q, k, reps, rows, dim):
    """One point: warm-up, then reps rounds of one timed call per type in turn; then a profiled pass."""
    res = {t: {"ms": []} for t in idxs}
    parity = True
    for t in idxs:
        for _ in range(3):
            idxs[t].search_device(q, k)
    torch.cuda.synchronize()
    for _ in range(reps):
        outs = {}
        for t in idxs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            outs[t] = idxs[t].search_device(q, k)
            e1.record()
            torch.cuda.synchronize()
            res[t]["ms"].append(e0.elapsed_time(e1))
        if "f32" in outs and "f32+f16" in outs:
            a, b = outs["f32"], outs["f32+f16"]
            parity &= bool(torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32)))
    nq = q.shape[0]
    for t, idx in idxs.items():
        st = idx.stats()
        r = res[t]
        r["ms_median"] = round(statistics.median(r["ms"]), 4)
        r["ms_min"] = round(min(r["ms"]), 4)
        r["path"] = st["path"]
        r["queries_rescanned"] = st["queries_rescanned"]
        if st["path"] == 3:
            _, resc = idx.fused_counts(nq)
            r["rows_rescored"] = [int(v) for v in resc]
        idx.profile(True)
        for _ in range(5):
            idx.search_device(q, k)
        kms, launches = idx.profile_read()
        idx.profile(False)
        if launches:
            per = kms / 5
            r["kernel_ms"] = round(per, 4)
            r["sweep_gb_s"] = round(rows * ((dim + 7) // 8 * 8) * SWEEP_BYTES[t] / (per * 1e-3) / 1e9, 1)
        del r["ms"]
    return res, parity


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--config1-rows", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="profiles/r03/sweep_copy.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    report = {"gpu": gpu_info(), "dim": a.dim, "reps": a.reps, "timing": "CUDA events around one search_device call, median",
              "ingest_rows_per_s": {}, "points": []}
    parity_all = True

    def run_points(idxs, rows, points, label):
        nonlocal parity_all
        for nq, k, qfn in points:
            q = torch.from_numpy(qfn(nq)).cuda()
            res, parity = measure(idxs, q, k, a.reps, rows, a.dim)
            parity_all &= parity
            report["points"].append({"corpus": label, "rows": rows, "nq": nq, "k": k, "parity_f32_f32f16": parity, "by_type": res})
            print(json.dumps(report["points"][-1]), flush=True)

    qrand = lambda nq: synth_rows(4321, 0, nq, a.dim)
    idxs = {}
    for t in TYPES:
        idxs[t], rate = build(t, a.rows, a.dim, 1234)
        report["ingest_rows_per_s"][t] = round(rate)
    run_points(idxs, a.rows, [(1, 10, qrand), (16, 10, qrand), (128, 10, qrand), (4096, 10, qrand), (1, 100, qrand), (1, 1000, qrand)],
               "synthetic")
    for idx in idxs.values():
        idx.close()
    idxs = {t: build(t, a.config1_rows, a.dim, 1234)[0] for t in TYPES}
    run_points(idxs, a.config1_rows, [(1024, 10, qrand)], "config1")
    for idx in idxs.values():
        idx.close()
    topic_rows = 6000
    qtopic = lambda nq: synth_topic_rows(1234, 7 * topic_rows + 11, nq, a.dim, topic_rows, 2)
    idxs = {t: build(t, a.rows, a.dim, 1234, topics=topic_rows)[0] for t in TYPES}
    run_points(idxs, a.rows, [(1, 10, qtopic)], "templated")
    for idx in idxs.values():
        idx.close()
    report["parity_f32_f32f16_all"] = parity_all
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print("parity f32 == f32+f16 on every timed call:", parity_all)


if __name__ == "__main__":
    main()
