"""bench.py on the GPU (-m gpu): --steps sets what is timed, and --dump-outputs holds what the last timed step computed, in
float32/float64, within 64 MB, agreeing with the oracle on a sample."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_steps_and_dump_outputs(oracle_built, tmp_path):
    from openmmgridforce_b200 import workloads as W
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    steps, windows = 2, 2
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                          "--windows", str(windows), "--no-extras", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["run"]["timed_steps"] == windows * steps        # counted from the evaluations enqueued in the timed windows
    assert {v["timed_steps"] for v in line["e2e"]["variants"].values()} == {steps}
    assert sorted(os.listdir(tmp_path)) == ["energies.npy", "forces.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    en, f = np.load(tmp_path / "energies.npy"), np.load(tmp_path / "forces.npy")
    assert en.dtype == np.float64 and f.dtype == np.float32 and f.shape == (en.shape[0], b.N_ATOMS, 3)
    # every window starts at pose set 0 and the sets alternate: the last of 2 steps evaluates set 1, not the canonical set 0
    w, sets, _ = b.pose_sets(W, 0, 1, True, 2)
    pos = sets[(steps - 1) % len(sets)]
    assert en.shape[0] == pos.shape[0]
    pick = np.sort(np.random.default_rng(0).choice(pos.shape[0], 512, replace=False))
    port = oracle_built.PortOracle(w.counts, w.spacing, w.origin, w.grids, w.scaling, oob_k=w.oob_k)
    ge_ref, f_ref = port.execute_batched(pos[pick], n_threads=os.cpu_count() or 1)
    e_ref = ge_ref.sum(axis=1)
    bound = np.maximum(1e-6 * np.abs(e_ref), 6e-8 * W.mixed_energy_bound(w, pos[pick]))
    assert (np.abs(en[pick] - e_ref) <= bound).all()
    assert np.abs(f[pick] - f_ref).max() <= 1e-5 * np.abs(f_ref).max()
