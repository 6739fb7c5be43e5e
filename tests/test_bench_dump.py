"""bench.py --dump-outputs: the arrays written are the state after exactly `warmup + steps` MD steps of the timed path."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps, warmup):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "c2", "--steps", str(steps),
                        "--warmup", str(warmup), "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == steps and d["warmup"] == warmup
    assert sorted(os.listdir(out_dir)) == ["c2_coords.npy", "c2_velocities.npy"]
    x, v = np.load(out_dir / "c2_coords.npy"), np.load(out_dir / "c2_velocities.npy")
    assert x.shape == v.shape == (d["config"]["n_atoms"], 3) and x.dtype == v.dtype == np.float32
    assert np.isfinite(x).all() and np.isfinite(v).all()
    return x.astype(np.float64), v.astype(np.float64)


def test_dump_is_state_after_warmup_plus_timed_steps(tmp_path):
    # 5 + 4 and 3 + 6 steps end in the same state (bit for bit on a B200); had the dump been taken after the profiled run that
    # follows the timed steps (as many steps again), the two would be 2 steps apart: 2.8e-3 nm and 7.2e-3 nm/ps on a B200
    import bench
    box = bench.workload("c2", np.float32)[0]["box"]
    xa, va = _bench(tmp_path / "a", steps=4, warmup=5)
    xb, vb = _bench(tmp_path / "b", steps=6, warmup=3)
    d = xa - xb
    d -= box * np.round(d / box)
    print(f"[bench dump] 5+4 vs 3+6 steps: max|dx| = {np.abs(d).max():.2e} nm, max|dv| = {np.abs(va - vb).max():.2e} nm/ps")
    assert np.abs(d).max() < 1e-4
    assert np.abs(va - vb).max() < 1e-3
