#!/usr/bin/env python
"""bench.py - exact cosine top-k throughput on a synthetic 10M x 768 bf16 corpus (BASELINE.json).

A "step" is one pass of the hot path over one batch of synthetic queries: one exact top-k search
of `--batch` queries over the whole corpus.  With --gpus N the corpus is row-sharded over N ranks
(one process per GPU, torchrun), each rank searches its shard and the per-rank hits are exchanged
and reduced (<= 16 queries: inside the search kernel, by NVLink peer stores; else push / merge
kernels or NCCL all-gather + reduce kernel): total work is fixed, so scaling = "strong".

  value     queries/s with the queries already resident in HBM: K back-to-back searches on one stream,
            CUDA events around the K steps, max over ranks.  Pipelining is switched on (Index.set_pipelined: the
            one-kernel search is launched with programmatic stream serialization, so consecutive searches of
            resident queries overlap - throughput, not latency; the library's default is off)
  e2e       queries/s through the public host API, one synchronous call per step: pinned host queries ->
            H2D -> search [+ exchange + reduce] -> D2H of (ids, scores)  (latency-bound: no pipelining)
  roofline  dominant kernel (<= 16 queries: the whole search, HBM; large batch: the tensor-core sweep), timed
            live with CUDA events recorded by the library around every launch, in a second pass of the same
            K steps (events between launches would serialise what the timed pass pipelines)
  parity_check  after every timed regime, at every N: the timed batches and a needle batch re-run through
            the same call and verified against the oracle (see parity_check below)
  regimes   batch 4096 (tensor-bound), clustered (templated corpus), ingest (K1)
  cpu_baseline  the reference's CPU retrieval path (oracle/fast_cpu.py port) on this box's cores, over the
            whole corpus when the host has the memory

`--impl reference` times only that CPU path (rank 0), same metric and the same `config` object (job_config); what an
arm did on that config (search path, exchange, pipelining, rescans) is printed beside it under `run`.
`--dump-outputs DIR` writes the ids and scores of the last timed search of each batch size as .npy files.  Every input is
generated from a fixed seed, so the same arguments give the same files and two builds can be compared output for output.
Clocks and throttle reasons are sampled through NVML during the timed regions; a region that saw hw_slowdown,
hw_thermal_slowdown or sw_thermal_slowdown is rejected and measured once more (`clocks.remeasured_after`); sw_power_cap
is kept and reported.
Inputs are far larger than L2 (15.36 GB corpus vs 126 MB), so no L2 flush is needed between steps.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark may run from a read-only tree: no __pycache__ next to the sources

METRIC = "exact top-k queries/sec at 10Mx768"
SEED_CORPUS, SEED_QUERY = 1234, 1235


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="queries per search call")
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--dtype", default="bf16", choices=["f32", "bf16", "f16"])
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--also-batch", type=int, default=4096,
                    help="second regime measured in the same run and reported under 'regimes' (0 = off)")
    ap.add_argument("--gemm-cluster", type=int, default=0, help="tcgen05 path cluster size: 0 auto, 1, 2 or 4")
    ap.add_argument("--gemm-variant", type=int, default=-1, help="tcgen05 kernel of the multi-kernel path: 0 auto, 1 streaming, 2 A-stationary, 3 swapped roles for <= 16 queries, 4 2-SM MMA pairs (-1 = library default)")
    ap.add_argument("--cpu-rows", type=int, default=0,
                    help="rows of the CPU baseline sample (0 = the whole corpus when MemAvailable >= 1.3 x rows*dim*4, else 2M rows, extrapolated)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-regimes", action="store_true", help="skip the clustered-corpus and ingest legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the ids (as float64) and scores (float32) of the last timed search of "
                         "each batch size as DIR/<name>.npy, at most 64 MB in all (a fixed sample of queries beyond that)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return a


DUMP_BYTES = 64_000_000


def dump_outputs(d, results):
    """results: (name, ids [nq, k] int64, scores [nq, k] fp32) per timed batch size.  ids are written as float64 (exact)
    so that every file is floating point; queries beyond the byte budget are sampled with a fixed seed, and the sampled
    query positions are written as <name>_queries.npy."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    per = DUMP_BYTES // max(1, len(results)) - 3 * 1024          # 3 files, npy headers included
    for name, ids, scores in results:
        nq, k = ids.shape
        keep = max(1, per // (12 * k + 8))                          # float64 id + float32 score per hit, float64 query position
        if nq > keep:
            rows = np.sort(np.random.default_rng(0).choice(nq, keep, replace=False))
            ids, scores = ids[rows], scores[rows]
            np.save(os.path.join(d, f"{name}_queries.npy"), rows.astype(np.float64))
        np.save(os.path.join(d, f"{name}_ids.npy"), ids.astype(np.float64))
        np.save(os.path.join(d, f"{name}_scores.npy"), scores.astype(np.float32))


def workload_name(a):
    rows = f"{a.rows // 1_000_000}M" if a.rows % 1_000_000 == 0 else str(a.rows)
    return f"synthetic {rows}x{a.dim} {a.dtype} corpus, batch-{a.batch} queries, k={a.k}"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            m = json.load(f)
        return {"hbm": m["hbm_gbs"], "bf16": m["bf16_tflops"], "bf16_sustained": m.get("bf16_tflops_sustained"),
                "source": "MEASURED_PEAKS.json"}
    return {"hbm": 6650.0, "bf16": 1590.0, "bf16_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


# ----------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi DURING the timed region
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """Polls NVML in-process (about every 2 ms) while the timed region runs, so that even a three-step
    batch-1 region (7 ms) is sampled; falls back to an `nvidia-smi -lms` child if NVML is unavailable."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []
        self.sm, self.mx, self.reasons, self.power = [], [], set(), []
        self.stop_flag = threading.Event()
        self.thread = None
        self.nvml = None

    def _nvml_handle(self):
        import pynvml
        import torch
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.gpu]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.gpu
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)

    def _poll(self, pynvml, h):
        bits = {pynvml.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                pynvml.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                pynvml.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                pynvml.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"}
        try:
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)))
        except Exception:
            pass
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                for b, nm in bits.items():
                    if r & b:
                        self.reasons.add(nm)
                self.power.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1e3)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            pynvml, h = self._nvml_handle()
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll, args=(pynvml, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None,
                    "reasons": sorted(self.reasons), "source": "nvml, 2 ms poll over the timed regions"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(self.NAMES, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 20"}


# ----------------------------------------------------------------------------------------------
# CPU baseline (oracle port; the only place bench.py executes oracle/)
# ----------------------------------------------------------------------------------------------
def mem_available_bytes():
    try:
        with open("/proc/meminfo") as f:
            for ln in f:
                if ln.startswith("MemAvailable:"):
                    return int(ln.split()[1]) * 1024
    except OSError:
        pass
    return 0


def cpu_corpus(a, rows):
    """fp32 normalised rows [rows, dim] of the synthetic corpus as a torch CPU tensor, generated block by block with the C
    oracle (what a CPU Milvus would hold: bf16 / fp16 corpora are up-cast, SURVEY.md 8d)."""
    import numpy as np
    import torch
    from oracle import c_oracle
    out = torch.empty((rows, a.dim), dtype=torch.float32)
    o = out.numpy()
    blk = 500_000
    for r0 in range(0, rows, blk):
        m = min(blk, rows - r0)
        o[r0:r0 + m] = c_oracle.normalize_rows(c_oracle.synth_rows(SEED_CORPUS, r0, m, a.dim), "f32")
    return out


def cpu_baseline(a, budget_s: float, steps: int | None = None, warmup: int = 1):
    import numpy as np
    import torch
    from oracle import c_oracle, fast_cpu
    c_oracle.build()
    # all host threads: torchrun exports OMP_NUM_THREADS=1 to its workers, which would make the N > 1 reference arm scalar
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if torch.get_num_threads() < ncpu:
        torch.set_num_threads(ncpu)
    # the whole corpus when the host can hold it in fp32 (BASELINE.md 3: 30.7 GB at 10M x 768), else a slice, scaled linearly
    full_bytes = a.rows * a.dim * 4
    rows = a.rows if (a.cpu_rows <= 0 and mem_available_bytes() >= 1.3 * full_bytes) else min(a.cpu_rows if a.cpu_rows > 0 else 2_000_000, a.rows)
    extrapolated = rows < a.rows
    nq = a.batch if a.batch <= 64 else 64           # bounded sample of the query batch
    t_gen = time.perf_counter()
    stored = cpu_corpus(a, rows)
    t_gen = time.perf_counter() - t_gen
    q = c_oracle.synth_rows(SEED_QUERY, 0, nq * 4, a.dim)
    for i in range(warmup):
        fast_cpu.fast_topk(stored, q[(i % 4) * nq:(i % 4 + 1) * nq], a.k)
    times, t_end, i = [], time.perf_counter() + budget_s, 0
    while (steps is None and time.perf_counter() < t_end) or (steps is not None and i < steps):
        t0 = time.perf_counter()
        last = fast_cpu.fast_topk(stored, q[(i % 4) * nq:(i % 4 + 1) * nq], a.k)
        times.append(time.perf_counter() - t0)
        i += 1
        if steps is None and i >= 400:
            break
    per_call = statistics.median(times)
    qps = nq / per_call * (rows / a.rows)            # linear in corpus rows (brute force); factor 1 when not extrapolated
    sample = (f"{nq} of {a.batch} queries per call over " +
              (f"the whole {a.rows}-row corpus held as fp32 ({full_bytes / 1e9:.1f} GB)" if not extrapolated else
               f"a {rows}-row fp32 slice of the {a.rows}-row corpus; throughput scaled by {rows}/{a.rows} (linear in rows)") +
              f", {len(times)} calls, median")
    return {"value": qps, "unit": "queries/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample,
            "extrapolated": extrapolated, "rows_timed": rows, "corpus_build_s": round(t_gen, 1),
            "ms_per_call_on_sample": per_call * 1e3}, last


def job_config(a, world):
    """The workload both arms are measured on: printed identically by `--impl ours` and `--impl reference`."""
    return {"workload": workload_name(a), "rows": a.rows, "dim": a.dim, "k": a.k, "batch": a.batch,
            "parallelism": f"row-shard x{world}" if world > 1 else "single GPU",
            "l2": "inputs (corpus shard) larger than L2; no flush needed"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # every step is one search of the batch (at most 64 of its queries) over the corpus
    base, (ids, scores) = cpu_baseline(a, budget_s=0.0, steps=a.steps, warmup=a.warmup)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, [(f"batch_{a.batch}", ids, scores)])
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": "queries/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": a.batch / base["value"] * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": job_config(a, a.gpus),      # our arm's config, key for key (the reference arm runs "on your arm's config")
        "run": {"note": "reference CPU retrieval path (Milvus/knowhere brute-force COSINE restated: oracle/fast_cpu.py), "
                        "rank 0's host cores only; the corpus is held as fp32 in host memory, far larger than any cache"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def run_ours(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    import ragfin_b200
    from ragfin_b200.sharded import ShardedSearcher, shard_bounds
    from ragfin_b200.synthetic import synth_rows

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- corpus: this rank's row shard of the synthetic matrix, generated + ingested on device
    row0, n_local = shard_bounds(a.rows, world, rank)
    idx = ragfin_b200.Index(a.dim, a.dtype, capacity=max(n_local, 1), device=local)
    t0 = time.perf_counter()
    for r in range(0, n_local, 1_000_000):
        idx.add_synthetic(SEED_CORPUS, row0 + r, min(1_000_000, n_local - r))
    idx.set_id_base(row0)
    idx.set_gemm_cluster(a.gemm_cluster)
    idx.set_pipelined(True)   # the value pass: queries resident in HBM before the timed region, nothing produces them between searches
    if a.gemm_variant >= 0:
        idx.set_gemm_variant(a.gemm_variant)
    torch.cuda.synchronize()
    ingest_s = time.perf_counter() - t0
    searcher = ShardedSearcher.for_index(idx)
    peaks = measured_peaks()
    esize = 4 if a.dtype == "f32" else 2
    ld = (a.dim + 7) // 8 * 8
    shard_rows = shard_bounds(a.rows, world, 0)[1]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(batch, steps, warmup):
        """One regime: device-resident timing (value), host end-to-end timing (e2e), live kernel timing (roofline)."""
        nbatches = 4
        q_host = torch.from_numpy(synth_rows(SEED_QUERY, 0, nbatches * batch, a.dim)).view(nbatches, batch, a.dim).pin_memory()
        q_dev = q_host.to(dev)
        out_ids = torch.empty((batch, a.k), dtype=torch.int64).pin_memory()
        out_sc = torch.empty((batch, a.k), dtype=torch.float32).pin_memory()
        q_stage = torch.empty((batch, a.dim), dtype=torch.float32, device=dev)

        fused_sharded = world > 1 and searcher.exchange is not None and searcher.fused_ok(batch, a.k)

        q_batches = [q_host[b] for b in range(nbatches)]   # the caller's own pinned buffers, handed over as they are

        def e2e_step(i):
            if world == 1:   # the C-ABI host call: H2D + search + D2H + sync inside ragfin_search_host
                idx.search(q_batches[i % nbatches], a.k, out_ids=out_ids, out_scores=out_sc)
            elif fused_sharded:   # ragfin_search_sharded_host: pinned staging, one kernel per GPU (sweep + exchange + reduce), one sync
                searcher.search_host(q_batches[i % nbatches], a.k, out_ids=out_ids, out_scores=out_sc)
            else:
                q_stage.copy_(q_host[i % nbatches], non_blocking=True)
                ids, sc = searcher.search(q_stage, a.k)
                out_ids.copy_(ids, non_blocking=True)
                out_sc.copy_(sc, non_blocking=True)
                torch.cuda.current_stream().synchronize()

        for i in range(warmup):
            searcher.search(q_dev[i % nbatches], a.k)
        for i in range(max(1, warmup // 2)):
            e2e_step(i)
        st = idx.stats()
        # kernels of ours per step: the search's own launches; sharded without the one-kernel path: + push / merge kernels
        # (peer memory) or + the reduce kernel after NCCL's all-gather
        launches_per_step = st["launches"] + (0 if world == 1 or fused_sharded else 2 if searcher.exchange is not None else 1)

        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        # value: K back-to-back searches, nothing between the launches (the one-kernel search is launched with programmatic
        # stream serialization: the next search's CTAs take over SMs as this one's finish; an event between two launches
        # would serialise them)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            last = searcher.search(q_dev[i % nbatches], a.k)
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        last = (last[0].cpu().numpy(), last[1].cpu().numpy()) if a.dump_outputs else None
        # roofline: the same K steps once more with the library's event pair around every launch of the dominant kernel
        # (serialised by those events: per-launch durations, not throughput)
        idx.profile(True)
        barrier()
        evp0, evp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        evp0.record()
        for i in range(steps):
            searcher.search(q_dev[i % nbatches], a.k)
        evp1.record()
        barrier()
        ms_prof = evp0.elapsed_time(evp1)
        kern_ms, kern_n = idx.profile_read()
        idx.profile(False)

        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            e2e_step(i)
        barrier()
        e2e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3], dtype=torch.float64, device=dev)
        clocks = sampler.stop() if rank == 0 else None
        kern = torch.tensor([kern_ms / max(kern_n, 1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(kern, op=dist.ReduceOp.MAX)
        ms, e2e_ms, kern_avg_ms = float(ms.item()), float(e2e_ms.item()), float(kern.item())
        launches_of_kernel_per_step = kern_n / max(steps, 1)
        # intensity of one pass = 2*nq*N*D flops over N*ld*esize bytes; below the ridge (peak flops / peak bytes,
        # ~257 queries for bf16) the tensor-core kernel is HBM-bound like the scan
        ridge = peaks["bf16"] * 1e12 / (peaks["hbm"] * 1e9)
        if st["path"] == 0 or 2.0 * batch / esize < ridge:   # algorithmic bytes = one pass over the shard per launch
            alg = shard_rows * ld * esize
            achieved = alg / (kern_avg_ms * 1e-3) / 1e9
            # <= 16 queries run the swapped-role kernel unless a variant is forced (csrc/gemm_rows.cuh)
            kname = ("scan_topk_kernel" if st["path"] == 0 else "sweep_fused_kernel" if st["path"] == 3 else
                     "gemm_rows_kernel" if batch <= 16 and a.gemm_variant in (-1, 0, 3) else "gemm_topk_kernel")
            roof = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": achieved / peaks["hbm"], "algorithmic_bytes_per_launch": alg,
                    "frac_of_nominal_8TBps": achieved / 8000.0}
        else:                 # tensor-bound GEMM: algorithmic flops = 2 * nq * shard rows * dim per launch
            alg = 2.0 * batch * shard_rows * a.dim
            achieved = alg / (kern_avg_ms * 1e-3) / 1e12
            roof = {"bound": "tensor", "kernel": "gemm_pair_kernel" if a.gemm_variant in (-1, 0, 3, 4) and batch > 128 else "gemm_topk_kernel", "achieved": achieved, "peak": peaks["bf16"],
                    "unit": "TFLOP/s", "frac": achieved / peaks["bf16"], "algorithmic_flops_per_launch": alg,
                    "frac_of_sustained_peak": achieved / peaks["bf16_sustained"] if peaks.get("bf16_sustained") else None}
        roof.update({"kernel_ms_avg": kern_avg_ms, "kernel_launches_timed": kern_n, "peak_source": peaks["source"],
                     "kernel_share_of_step": kern_avg_ms * launches_of_kernel_per_step / (ms_prof / steps),
                     "kernel_timing": "a second pass of the same steps with an event pair around every launch of the kernel (%.4f ms per step: "
                                      "the events serialise launches that the timed pass pipelines)" % (ms_prof / steps),
                     # DRAM bytes of the same kernel from the committed ncu --set full capture of this workload on ONE GPU
                     # (profiles/traffic.json): a profile figure, not a measurement of this run; null for shards
                     "traffic": load_traffic(a, batch) if world == 1 else None,
                     "traffic_source": "profiles/traffic.json (ncu --set full capture of this workload, not this run)" if world == 1 else None})
        return {
            "value": batch * steps / (ms * 1e-3), "unit": "queries/s", "batch": batch, "steps": steps,
            "ms_per_step": ms / steps, "clocks": clocks,
            "e2e": {"value": batch * steps / (e2e_ms * 1e-3), "unit": "queries/s", "ms_per_step": e2e_ms / steps,
                    "h2d_bytes_per_step": batch * a.dim * 4, "d2h_bytes_per_step": batch * a.k * 12},
            "gpu_launches": launches_per_step * steps, "roofline": roof,
            "queries_rescanned_last_step": st["queries_rescanned"], "last_step_outputs": last,
            "search_path": {0: "scan + finalize", 1: "tensor-core sweep, multi-kernel", 2: "large k", 3: "one kernel (sweep_fused)"}.get(st["path"]),
            "exchange": None if world == 1 else ("in-kernel peer stores (ragfin_search_sharded)" if fused_sharded else
                                                 "peer-memory push / merge kernels" if searcher.exchange is not None else "nccl all-gather + reduce kernel"),
        }

    def throttled(m):
        reasons = (m.get("clocks") or {}).get("reasons") or []
        return any(r in reasons for r in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"))

    def measure_checked(batch, steps, warmup):
        """A region that saw a hardware / thermal slowdown is rejected and measured once more (sw_power_cap is kept and
        reported); rank 0 samples the clocks, so it decides for every rank."""
        m = measure(batch, steps, warmup)
        redo = torch.tensor([1 if (rank == 0 and throttled(m)) else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.broadcast(redo, 0)
        if int(redo.item()):
            rejected = (m.get("clocks") or {}).get("reasons")
            m = measure(batch, steps, warmup)
            m["remeasured_after"] = rejected
        return m

    def parity_check(batch):
        """Correctness of the path that was just timed, OUTSIDE the timed region, on the (sharded) result as every rank sees
        it: the timed query batches re-run through the same call plus one needle batch; rank 0 verifies with the oracle
          order      score descending, ties to the lower id
          scores     every returned score bit-equal to the oracle's canonical score of that row (row regenerated on the host)
          needles    queries that are copies of corpus rows planted in EVERY shard come back first with their global id
          sample     a random 200k-row sample (oracle-scored) holds no row that beats the k-th hit of the checked queries
          agree      every rank holds the same merged result (hash compared over the ranks)."""
        from oracle import c_oracle
        nbatches = 4
        q_all = synth_rows(SEED_QUERY, 0, nbatches * batch, a.dim).reshape(nbatches, batch, a.dim)
        # positions checked inside a batch: everything for small batches, else 2 per 128-query tile (every tile of the batch)
        if batch <= 16:
            pos = list(range(batch))
        else:
            pos = sorted({min(batch - 1, t * 128 + (37 * t + 5) % 128) for t in range((batch + 127) // 128)} |
                         {min(batch - 1, t * 128 + (91 * t + 64) % 128) for t in range((batch + 127) // 128)})
        # needle rows: one in every shard (none on a shard boundary), as queries at the checked positions of one extra batch
        needle_rows = []
        for w in range(world):
            r0, cnt = shard_bounds(a.rows, world, w)
            if cnt > 0:
                needle_rows += [r0 + cnt // 3, r0 + (2 * cnt) // 3]
        needle_batches = []
        for c0 in range(0, len(needle_rows), len(pos)):
            qb = q_all[1 % nbatches].copy()
            chunk = needle_rows[c0:c0 + len(pos)]
            for p_, r in zip(pos, chunk):
                qb[p_] = c_oracle.synth_rows(SEED_CORPUS, r, 1, a.dim)[0]
            needle_batches.append((qb, dict(zip(pos, chunk))))
        runs = [(q_all[i], {}) for i in range(nbatches if batch <= 16 else 1)] + needle_batches
        results = []
        agree = True
        for qb, needles in runs:
            ids, sc = searcher.search(torch.from_numpy(qb).to(dev), a.k)
            torch.cuda.synchronize()
            ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
            if world > 1:   # every rank must hold the same merged result
                import hashlib
                hsh = int.from_bytes(hashlib.blake2b(ids.tobytes() + sc.tobytes(), digest_size=8).digest(), "little") >> 1
                t = torch.tensor([hsh, -hsh], dtype=torch.int64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                agree &= int(t[0].item()) == -int(t[1].item())
            results.append((qb, needles, ids, sc))
        if rank != 0:
            return None
        t0 = time.perf_counter()
        fails, checked, n_needles = [], 0, 0
        rng = np.random.default_rng(7)
        nblk, blk_rows = 100, 2000
        starts = rng.integers(0, max(1, a.rows - blk_rows), size=nblk)
        sample = [(int(s0), c_oracle.normalize_rows(c_oracle.synth_rows(SEED_CORPUS, int(s0), min(blk_rows, a.rows - int(s0)), a.dim), a.dtype)) for s0 in starts]
        sample_queries = 0
        for qb, needles, ids, sc in results:
            qhat = c_oracle.normalize_rows(qb[pos], "f32")
            for j, p_ in enumerate(pos):
                i_, s_ = ids[p_], sc[p_]
                checked += 1
                keff = min(a.k, a.rows)
                if (i_[:keff] < 0).any() or (i_[:keff] >= a.rows).any():
                    fails.append(f"q{p_}: id out of range"); continue
                for x in range(keff - 1):
                    if not (s_[x] > s_[x + 1] or (s_[x] == s_[x + 1] and i_[x] < i_[x + 1])):
                        fails.append(f"q{p_}: order at {x}"); break
                rows_ = np.concatenate([c_oracle.synth_rows(SEED_CORPUS, int(r), 1, a.dim) for r in i_[:keff]])
                want = c_oracle.exact_scores(c_oracle.normalize_rows(rows_, a.dtype), qhat[j])
                if not np.array_equal(want.view(np.uint32), s_[:keff].view(np.uint32)):
                    fails.append(f"q{p_}: score bits differ from the oracle's")
                if p_ in needles:
                    n_needles += 1
                    if int(i_[0]) != needles[p_] or abs(float(s_[0]) - 1.0) > 1e-2:
                        fails.append(f"needle row {needles[p_]} came back as {int(i_[0])} ({float(s_[0]):.6f})")
                if sample_queries < 12 and (j % max(1, len(pos) // 4) == 0):   # sample property on a few queries of every run
                    sample_queries += 1
                    kth_s, kth_i, have = s_[keff - 1], i_[keff - 1], set(i_[:keff].tolist())
                    for s0, blk in sample:
                        ssc = c_oracle.exact_scores(blk, qhat[j])
                        rws = np.arange(s0, s0 + blk.shape[0])
                        better = (ssc > kth_s) | ((ssc == kth_s) & (rws < kth_i))
                        if not set(rws[better].tolist()) <= have:
                            fails.append(f"q{p_}: a sampled row near {s0} beats the k-th hit"); break
        return {"ok": not fails and agree, "queries": checked, "needles": n_needles, "needle_shards": world,
                "sample_rows": nblk * blk_rows, "sample_queries": sample_queries, "ranks_agree": agree,
                "failures": fails[:5], "check_s": round(time.perf_counter() - t0, 1),
                "how": "timed batches + needle batch re-run through the timed call after the timed region; rank 0 checks order, "
                       "score bits == oracle canonical score of the regenerated rows, needles (copies of corpus rows in every "
                       "shard) first with their global id, no row of a 200k-row oracle-scored sample beats the k-th hit; "
                       "result hash equal on every rank"}

    def ingest_leg():
        """K1 (L2-normalise + cast at ingest, "chunking_storing (1).py":379-396) on one rank: rows/s and GB/s of
        4 * dim (fp32 read) + esize * ld (stored write) bytes per row, kernel time from the library's events.
        device: source already in HBM (the N2 device feed); host: pinned source through the double-buffered staging."""
        if rank != 0:
            return None
        n_dev, n_host = 2_000_000, 500_000
        per_row = 4 * a.dim + esize * ld
        out = {"bytes_per_row": per_row, "kernel": "ingest_vec_kernel" if a.dim % 4 == 0 and ld <= 1024 else "ingest_kernel"}
        src = torch.randn((n_dev, a.dim), dtype=torch.float32, device=dev,
                          generator=torch.Generator(device=dev).manual_seed(SEED_CORPUS + 1))
        tmp = ragfin_b200.Index(a.dim, a.dtype, capacity=3 * n_dev, device=local)
        tmp.add(src)                                    # warm-up (first launch, clocks)
        tmp.profile(True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(2):
            tmp.add(src)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        kms, kn = tmp.profile_read()
        tmp.profile(False)
        out["device"] = {"rows": 2 * n_dev, "kernel_ms": kms, "launches": kn, "gbps": 2 * n_dev * per_row / (kms * 1e-3) / 1e9,
                         "frac_of_hbm_peak": 2 * n_dev * per_row / (kms * 1e-3) / 1e9 / peaks["hbm"], "rows_per_s": 2 * n_dev / (kms * 1e-3),
                         "wall_ms_through_the_api": wall * 1e3}
        tmp.close()
        del src
        hsrc = torch.randn((n_host, a.dim), dtype=torch.float32, generator=torch.Generator().manual_seed(SEED_CORPUS + 2)).pin_memory()
        tmp = ragfin_b200.Index(a.dim, a.dtype, capacity=2 * n_host, device=local)
        tmp.add(hsrc.numpy())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tmp.add(hsrc.numpy())
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        out["host"] = {"rows": n_host, "wall_ms": wall * 1e3, "h2d_gbps": n_host * a.dim * 4 / wall / 1e9, "rows_per_s": n_host / wall,
                       "note": "pinned host source, H2D of slice i + 1 overlaps K1 on slice i (PCIe-bound)"}
        tmp.close()
        return out

    def clustered_leg(batch, iid_ms):
        """The same search over a corpus with the structure of templated text (the reference's chunks are templates filled
        with each quarter's figures): contiguous runs of `topic_rows` near-duplicate rows in topic order
        (ragfin_add_synthetic_topics), queries aimed at single topics.  A strided sample never sees the topic, thousands of
        rows sit within a hair of the k-th score: the case that sends a static-threshold design to its exact fallback."""
        from oracle import c_oracle
        from ragfin_b200.synthetic import synth_topic_rows
        topic_rows, shift, seed = 16384, 3, SEED_CORPUS + 77
        cidx = ragfin_b200.Index(a.dim, a.dtype, capacity=max(n_local, 1), device=local)
        for r in range(0, n_local, 1_000_000):
            cidx.add_synthetic_topics(seed, row0 + r, min(1_000_000, n_local - r), topic_rows, shift)
        cidx.set_id_base(row0)
        csearch = ShardedSearcher.for_index(cidx)
        rows_fn = lambda sd, r0, m, d: c_oracle.synth_rows(sd, r0, m, d)
        nb = 8
        n_topics = max(1, a.rows // topic_rows)
        targets = [((2 * i + 1) * n_topics // (2 * nb * batch)) % n_topics for i in range(nb * batch)]     # spread over the corpus (every shard)
        from ragfin_b200.synthetic import TOPIC_SEED_OFFSET
        # a query = its topic's centre + fresh noise at twice the corpus amplitude (not a copy of any row)
        qh = np.concatenate([c_oracle.synth_rows(seed + TOPIC_SEED_OFFSET, t, 1, a.dim) +
                             c_oracle.synth_rows(seed + 4242, i, 1, a.dim) * np.float32(2.0 ** -(shift - 1)) for i, t in enumerate(targets)]).astype(np.float32)
        qd = torch.from_numpy(qh).to(dev).view(nb, batch, a.dim)
        steps = max(10, min(a.steps, 50))
        for i in range(3):
            csearch.search(qd[i % nb], a.k)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            csearch.search(qd[i % nb], a.k)
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms.item()) / steps
        resc, appended = 0, []
        results = []
        for i in range(nb):
            ids, sc = csearch.search(qd[i], a.k)
            torch.cuda.synchronize()
            st = cidx.stats()
            resc += max(0, st["queries_rescanned"])
            if st["path"] == 3:
                appended += cidx.fused_counts(batch)[0].tolist()
            results.append((ids.cpu().numpy(), sc.cpu().numpy()))
        t = torch.tensor([resc], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        resc = int(t.item())
        out = None
        if rank == 0:
            fails, checked = [], 0
            for i, (ids, sc) in enumerate(results):
                qhat = c_oracle.normalize_rows(qh[i * batch:(i + 1) * batch], "f32")
                for j in range(min(batch, 4)):
                    t_q = targets[i * batch + j]
                    i_, s_ = ids[j], sc[j]
                    checked += 1
                    if not all(s_[x] > s_[x + 1] or (s_[x] == s_[x + 1] and i_[x] < i_[x + 1]) for x in range(a.k - 1)):
                        fails.append(f"q{i}.{j}: order")
                    # the whole target topic, rebuilt on the host and scored by the oracle: its top-k IS the answer
                    blk = c_oracle.normalize_rows(synth_topic_rows(seed, t_q * topic_rows, min(topic_rows, a.rows - t_q * topic_rows), a.dim, topic_rows, shift, rows_fn), a.dtype)
                    ssc = c_oracle.exact_scores(blk, qhat[j])
                    order = np.lexsort((np.arange(len(ssc)), -ssc.astype(np.float64)))[:a.k]
                    want_ids = order + t_q * topic_rows
                    if not (np.array_equal(i_, want_ids) and np.array_equal(s_.view(np.uint32), ssc[order].view(np.uint32))):
                        fails.append(f"q{i}.{j}: differs from the oracle's top-k of topic {t_q}")
            out = {"ms_per_step": ms, "value": batch / (ms * 1e-3), "unit": "queries/s", "batch": batch, "steps": steps,
                   "vs_iid_time": ms / iid_ms, "queries_rescanned": resc,
                   "rows_appended_per_query": {"mean": float(np.mean(appended)) if appended else None, "max": int(max(appended)) if appended else None},
                   "corpus": f"{a.rows} rows in runs of {topic_rows} near-duplicates (centre + noise / {2 ** shift}; cosine ~0.98 inside a run), topic order",
                   "queries": "one topic each (its centre + noise / %d), topics spread over every shard" % 2 ** (shift - 1),
                   "parity_check": {"ok": not fails, "queries": checked, "failures": fails[:5],
                                    "how": "ids and score bits equal to the oracle's exact top-k over the query's whole topic (16384 rows rebuilt on the host)"}}
        if csearch.exchange is not None:
            csearch.exchange.close()
        cidx.close()
        return out

    main = measure_checked(a.batch, a.steps, a.warmup)
    main["parity_check"] = parity_check(a.batch)
    last = main.pop("last_step_outputs")
    outputs = [(f"batch_{a.batch}",) + last] if last else []
    other = None
    if a.also_batch and a.also_batch != a.batch:
        other = measure_checked(a.also_batch, max(5, a.steps // 10), a.warmup)
        other["parity_check"] = parity_check(a.also_batch)
        last = other.pop("last_step_outputs")
        if last:
            outputs.append((f"batch_{a.also_batch}",) + last)
    if a.dump_outputs and rank == 0:   # every rank holds the same merged result
        dump_outputs(a.dump_outputs, outputs)
    def side_leg(fn, *args):
        """The side regimes must not cost the headline line: on one GPU a failure is reported in place of the leg's figures
        (with several ranks it propagates - a rank that skipped a leg would leave the others waiting in its collectives)."""
        if world > 1:
            return fn(*args)
        try:
            return fn(*args)
        except Exception as e:                                     # noqa: BLE001 - reported, never hidden
            try:
                torch.cuda.synchronize()
            except Exception:                                      # noqa: BLE001
                pass
            return {"error": f"{type(e).__name__}: {e}"[:400]}

    clustered = side_leg(clustered_leg, a.batch, main["ms_per_step"]) if not a.no_extra_regimes else None
    ingest = side_leg(ingest_leg) if (world == 1 and not a.no_extra_regimes) else None

    if rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": "queries/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": a.dtype, "data": "synthetic",
            "config": job_config(a, world),
            # what THIS arm did on that config (kept out of `config` so that both arms print the same config object)
            "run": {"ingest_s": round(ingest_s, 2), "queries_rescanned_last_step": main["queries_rescanned_last_step"],
                    "search_path": main["search_path"], "exchange": main["exchange"],
                    "pipelined": "value: ragfin_set_pipelined(1), consecutive searches of one stream overlap (queries resident before the "
                                 "timed region); e2e: one synchronous call at a time"},
            "clocks": dict(main["clocks"] or {}, **({"remeasured_after": main["remeasured_after"]} if "remeasured_after" in main else {})),
            "e2e": main["e2e"], "gpu_launches": main["gpu_launches"], "roofline": main["roofline"],
            "parity_check": main["parity_check"],
        }
        if other is not None:
            line["regimes"] = {f"batch_{other['batch']}": other}
        if clustered is not None:
            line.setdefault("regimes", {})["clustered"] = clustered
        if ingest is not None:
            line.setdefault("regimes", {})["ingest"] = ingest
        if world == 1 and not a.no_cpu_baseline:
            del idx
            try:
                line["cpu_baseline"] = cpu_baseline(a, budget_s=15.0)[0]
            except Exception as e:                                 # noqa: BLE001 - e.g. the host cannot hold the fp32 corpus
                line["cpu_baseline"] = {"value": None, "unit": "queries/s", "kind": "port", "error": f"{type(e).__name__}: {e}"[:400]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def load_traffic(a, batch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    ncu --set full capture of this workload (profiles/traffic.json), else null."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        t = json.load(f)
    return t.get(f"{a.rows}x{a.dim}:{a.dtype}:b{batch}:k{a.k}")


def main():
    a = parse_args()
    if a.gpus > 1 and "WORLD_SIZE" not in os.environ:   # convenience: self-launch under torchrun
        port = 29500 + os.getpid() % 2000
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
