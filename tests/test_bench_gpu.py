"""bench.py --dump-outputs on the engine: the files hold what the last timed search of each batch size returned, equal to
the oracle's exact top-k of that step's queries (ids, and score bits)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_last_timed_step(tmp_path, coracle):
    rows, dim, k, steps = 30000, 384, 10, 3
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(rows), "--dim", str(dim), "--k", str(k),
                        "--steps", str(steps), "--warmup", "1", "--also-batch", "256", "--no-cpu-baseline", "--no-extra-regimes",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == steps and line["parity_check"]["ok"]
    sys.path.insert(0, ROOT)
    try:
        import bench
    finally:
        sys.path.pop(0)
    x = coracle.normalize_rows(coracle.synth_rows(bench.SEED_CORPUS, 0, rows, dim), "bf16")
    # batch 1 runs `steps` timed searches, batch 256 max(5, steps // 10); step i searches query batch i % 4
    for batch, last in ((1, steps - 1), (256, 4)):
        q = coracle.synth_rows(bench.SEED_QUERY, 0, 4 * batch, dim)[(last % 4) * batch:(last % 4 + 1) * batch]
        want_ids, want_sc = coracle.cosine_topk(q, x, k)
        ids, sc = np.load(tmp_path / f"batch_{batch}_ids.npy"), np.load(tmp_path / f"batch_{batch}_scores.npy")
        assert ids.dtype == np.float64 and sc.dtype == np.float32
        assert np.array_equal(ids, want_ids.astype(np.float64)), batch
        assert np.array_equal(sc.view(np.uint32), want_sc.view(np.uint32)), batch
