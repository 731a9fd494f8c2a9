"""One-kernel search with the int8 tile filter on and off, alternated in one process, on the bench corpus (10M x 768 bf16)
and the templated corpus: ms per call (CUDA events over back-to-back pipelined searches), tiles read in 16 bits and screened,
the bytes a search really reads and the rate that gives, and ids / score bits of both arms compared on every timed call.
Also the one-time build of the int8 copy.  Writes profiles/r06/i8_sweep.json (or --out).  Needs the GPU."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ragfin_b200  # noqa: E402
from ragfin_b200.synthetic import synth_rows  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def arm(idx, on, q, k, steps):
    """steps back-to-back searches of one arm; returns (ms per call, last outputs of every call, tiles of the last call)."""
    idx.set_sweep_copy(on)
    for i in range(3):
        idx.search_device(q[i % len(q)], k)
    torch.cuda.synchronize()
    outs = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        outs.append(idx.search_device(q[i % len(q)], k))
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, [(a.cpu().numpy(), b.cpu().numpy()) for a, b in outs], idx.fused_tiles()


def shape(idx, n, ld, q, k, steps, rounds):
    res = {"on_ms": [], "off_ms": []}
    equal = True
    for _ in range(rounds):
        ms_on, o_on, tiles = arm(idx, True, q, k, steps)
        ms_off, o_off, _ = arm(idx, False, q, k, steps)
        res["on_ms"].append(ms_on)
        res["off_ms"].append(ms_off)
        equal = equal and all(np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
                              for a, b in zip(o_on, o_off))
    t16, t8 = tiles
    ld8 = (ld + 15) // 16 * 16
    # bytes of the last int8 search: int8 tiles + their side data, 16-bit tiles (first tiles and refined ones)
    real = t8 * 256 * (ld8 + 8) + t16 * 256 * ld * 2
    ms_on = float(np.median(res["on_ms"]))
    res.update({"on_ms_median": ms_on, "off_ms_median": float(np.median(res["off_ms"])),
                "speedup": float(np.median(res["off_ms"])) / ms_on, "tiles_16bit": t16, "tiles_int8": t8,
                "bytes_per_search": real, "tb_per_s": real / (ms_on * 1e-3) / 1e12, "bytes_16bit_sweep": n * ld * 2,
                "ids_and_score_bits_equal_every_call": equal})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06", "i8_sweep.json"))
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    ld = (a.dim + 7) // 8 * 8
    out = {"gpu": gpu_info(), "rows": a.rows, "dim": a.dim, "dtype": "bf16", "steps": a.steps, "rounds": a.rounds, "shapes": {}}
    idx = ragfin_b200.Index(a.dim, "bf16", capacity=a.rows, device=0)
    for r in range(0, a.rows, 1_000_000):
        idx.add_synthetic(1, r, min(1_000_000, a.rows - r))
    idx.set_pipelined(True)
    q1 = torch.from_numpy(synth_rows(2, 0, 4, a.dim)).to(dev)
    # one-time build: the first search with the copy on, minus a search with it
    idx.set_sweep_copy(True)
    torch.cuda.synchronize()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record(); idx.search_device(q1[:1], 10); e1.record(); idx.search_device(q1[:1], 10); e2.record()
    torch.cuda.synchronize()
    out["copy_build_ms"] = e0.elapsed_time(e1) - e1.elapsed_time(e2)
    out["copy_bytes"] = a.rows * ((ld + 15) // 16 * 16 + 8)
    for nb, k in ((1, 10), (4, 10), (16, 10), (1, 100)):
        qs = [torch.from_numpy(synth_rows(3 + i, 0, nb, a.dim)).to(dev) for i in range(4)]
        out["shapes"][f"b{nb}_k{k}"] = shape(idx, a.rows, ld, qs, k, a.steps, a.rounds)
        print(f"b{nb} k{k}", json.dumps(out["shapes"][f"b{nb}_k{k}"])[:300], flush=True)
    idx.close()
    # templated corpus (bench.py's clustered regime): runs of 16 384 near-duplicates
    topic = 16_384
    cidx = ragfin_b200.Index(a.dim, "bf16", capacity=a.rows, device=0)
    for r in range(0, a.rows, 1_000_000):
        cidx.add_synthetic_topics(1, r, min(1_000_000, a.rows - r), topic_rows=topic, noise_shift=3)
    cidx.set_pipelined(True)
    rows = cidx.read_rows(topic * 7 + 11, 1).astype(np.float32)
    qs = [torch.from_numpy(rows + synth_rows(10 + i, 0, 1, a.dim) / 4).to(dev) for i in range(4)]
    out["shapes"]["templated_b1_k10"] = shape(cidx, a.rows, ld, qs, 10, a.steps, a.rounds)
    print("templated", json.dumps(out["shapes"]["templated_b1_k10"])[:300], flush=True)
    cidx.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
