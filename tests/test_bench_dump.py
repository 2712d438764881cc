"""GPU: bench.py --dump-outputs writes what its last timed step computed -- the step's result as bench.py reports it,
and posterior and sets that match the FP64 oracle -- as finite float32/float64 .npy files within 64 MB."""
import json
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(oracle, tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, "bench.py", "--workload", "c4s", "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                        "--no-peaks", "--no-lipschitz-steps", "--no-reference-configs", "--dump-outputs", str(out)],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    cfg = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])["config"]
    files = sorted(out.glob("*.npy"))
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    d = {f.stem: np.load(f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in d.values())
    assert np.all(d["expander_per_value"][d["expander_per_idx"] < 0] == 0.0)          # no candidate: 0, not the sentinel
    assert int(d["n_safe"]) == cfg["n_safe"] and int(d["n_unsafe"]) == cfg["n_unsafe"] and int(d["n_min"]) == cfg["n_min"]
    assert int(d["expander_n_hit"]) == cfg["n_hit"] and int(d["x_new_idx"]) == cfg["x_new_idx"]
    import sbo_b200  # noqa: F401
    from sbo_b200 import workloads
    ds, lo, hi, pts, beta = workloads.c4(pts_per_dim=16, n=128)          # bench.py's c4s
    idx = d["point_index"].astype(np.int64)
    assert idx.size == np.prod(pts)                                       # a grid this small is dumped whole
    mo, vo = oracle.posterior_chol(oracle.make_grid(lo, hi, pts)[idx], ds)
    assert np.max(np.abs(d["posterior_mean"] - mo)) <= 1e-9 * np.max(np.abs(mo))
    assert np.max(np.abs(d["posterior_var"] - vo)) <= 1e-9 * np.max(ds["Y_std"]) ** 2
    lcb, _ = oracle.bounds(mo, vo, beta)
    assert np.array_equal(d["safe_mask"].astype(bool), oracle.safe_mask(lcb))
    assert np.array_equal(d["unsafe_mask"].astype(bool), oracle.unsafe_mask(lcb))
    assert d["minimizer_mask"].sum() == cfg["n_min"]
