"""bench.py contract checks.  Without a GPU: the reference arm (CPU restatement on the host cores) prints one JSON line whose
`config.workload` names the size it REALLY ran, with the keys a reader of the result line needs; box grids of the multi-GPU layout; argument
checks.  On the GPU: --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_labels_what_it_ran():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-size", "16"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-600:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "DOF/s" and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert "16^3 = 4096 DOFs" in d["config"]["workload"] and "200^3" not in d["config"]["workload"]  # the size it ran, not the GPU arm's
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "16^3" in cb["sample"]
    assert cb["scaling"][-1]["edge"] == 16 and cb["scaling"][-1]["dofs"] == 4096
    assert d["e2e"] == {"value": d["value"], "unit": "DOF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert abs(d["value"] - 4096 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]


def test_reference_arm_on_other_ranks_is_silent(monkeypatch):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_box_grids_cover_every_rank_evenly():
    from geneo4petsc_b200 import dist
    for world in (1, 2, 4, 8):
        for subs in (1, 2, 8, 27):
            K, g, sub_rank = dist.box_grid(world, subs)
            assert K[0] * K[1] * K[2] == world * subs and g[0] * g[1] * g[2] == world
            assert np.bincount(sub_rank, minlength=world).tolist() == [subs] * world
            for rank in range(world):  # the kept region of a rank contains the lower corner of each of its boxes
                lo, hi = dist.keep_region(97, K, g, rank, subs)
                assert np.all(lo >= 0) and np.all(hi <= 97) and np.all(lo < hi)
                for b in np.flatnonzero(sub_rank == rank):
                    b3 = (b % K[0], (b // K[0]) % K[1], b // (K[0] * K[1]))
                    first = [-(-b3[a] * 97 // K[a]) for a in range(3)]
                    assert all(lo[a] <= first[a] < hi[a] for a in range(3))


def test_bench_rejects_runs_without_timed_steps():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_solution(tmp_path):
    """--dump-outputs DIR: x of the last timed step (all rows at this size, ids in x_index) and [its, rnorm, reason], float64;
    the same arguments give the same inputs, so two runs agree to the solver's tolerance."""
    runs = []
    for k in range(2):
        d = tmp_path / ("run%d" % k)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--size", "16", "--steps", "2", "--warmup", "1",
                            "--e2e-steps", "1", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=900, cwd=tmp_path)
        assert r.returncode == 0, r.stderr[-800:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        runs.append({name: np.load(d / (name + ".npy")) for name in ("x", "x_index", "ksp")})
    for out in runs:
        assert all(v.dtype == np.float64 for v in out.values())
        np.testing.assert_array_equal(out["x_index"], np.arange(16 ** 3))
        # b = A (1..N); CG stops at 1e-5 on the preconditioned residual: ~2e-3 absolute error on every row
        assert np.linalg.norm(out["x"] - (out["x_index"] + 1.0)) <= 1e-4 * np.linalg.norm(out["x_index"] + 1.0)
        assert out["ksp"][0] >= 1 and out["ksp"][2] > 0
    np.testing.assert_allclose(runs[0]["x"], runs[1]["x"], rtol=1e-8)
    assert runs[0]["ksp"][0] == runs[1]["ksp"][0]
