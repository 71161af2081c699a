"""Same-pattern update vs refactor vs fresh setup on the bench's N=1 workload: 200^3 Laplacian, 8 box subdomains, geneo
ASM,1 tau 0.1, CG rtol 1e-5.  Problem A has --kappa 2 lin, problem B --kappa 50 lin (same mesh, same partition).

Two 200^3 preconditioners do not fit one GPU together, so everything runs in sequence in one process:
setup(A) (also warms the process: its first upload is slow) -> update(B) -> refactor() -> CG -> destroy -> setup(B) -> CG.
Prints one JSON line (and writes it to --out when given)."""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import geneo4petsc_b200 as g  # noqa: E402
from geneo4petsc_b200 import dist  # noqa: E402

OPTS = ["-geneo_lvl", "ASM,1", "-geneo_tau", "0.1"]


def gpu_name_and_power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, limit = [s.strip() for s in out[0].split(",")]
        return name, limit
    except Exception as e:  # (the numbers are still printed; without the card they are not worth much)
        return "unknown (%s)" % e, "unknown"


def problem(size, kappa):
    prob = g.Problem()
    K, _, sub_rank = dist.box_grid(1, 8)
    edge = dist.generate_boxed(prob, "laplacian", "--dim 3 --size %d --inpEps 0.0001 --kappa %s lin" % (size, kappa), K)
    dist.decompose_owned(prob, len(sub_rank), sub_rank, 0, True, 0)
    return prob, edge


def timed(fn):
    t = time.perf_counter()
    fn()  # (the result is dropped: setup / update / refactor return the PC, which must not outlive `del pc`)
    return time.perf_counter() - t  # (every call below ends in a device synchronisation)


def solve(pc):
    b = pc.make_rhs()
    r = pc.ksp_solve(b, ksp="cg", rtol=1e-5, atol=1e-50)
    return r["its"], r["reason"], r["x"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if g.device_count() < 1:
        raise SystemExit("update_target.py: no CUDA device -- the library has no CPU fallback")
    pa, edge = problem(a.size, "2")
    pb, _ = problem(a.size, "50")
    n = edge ** 3
    v = np.sin(np.arange(n) * 0.37)

    pc = g.GeneoPC(OPTS)
    t_setup_a = timed(lambda: pc.setup(pa))
    c0 = g.counters()
    t_update = timed(lambda: pc.update(pb))
    c1 = g.counters()
    numeric_in_update = pc.timers()["numeric"]
    t_refactor = timed(pc.refactor)
    its_u, reason_u, x_u = solve(pc)
    ne_u = pc.info()["nE"]
    av_u = pc.mult(v)
    del pc
    gc.collect()

    fresh = g.GeneoPC(OPTS)
    t_fresh = timed(lambda: fresh.setup(pb))
    its_f, reason_f, x_f = solve(fresh)
    ne_f = fresh.info()["nE"]
    av_f = fresh.mult(v)
    name, limit = gpu_name_and_power_limit()
    res = {
        "workload": "laplacian3d %d^3, 8 box subdomains, geneo ASM,1 tau=0.1, CG rtol 1e-5; A: --kappa 2 lin, B: --kappa 50 lin" % edge,
        "gpu": name, "power_limit": limit,
        "setup_A_s": round(t_setup_a, 3),
        "update_s": round(t_update, 3),
        "update_numeric_s": round(numeric_in_update, 3),
        "update_values_s": round(t_update - numeric_in_update, 3),
        "update_h2d_bytes": c1["h2d"] - c0["h2d"],
        "update_launches": c1["launches"] - c0["launches"],
        "refactor_s": round(t_refactor, 3),
        "fresh_setup_s": round(t_fresh, 3),
        "updated": {"its": its_u, "reason": reason_u, "nE": ne_u},
        "fresh": {"its": its_f, "reason": reason_f, "nE": ne_f},
        "x_rel_diff": float(np.linalg.norm(x_u - x_f) / np.linalg.norm(x_f)),
        "mult_bitwise_equal": bool(np.array_equal(av_u, av_f)),
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
