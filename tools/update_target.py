"""Same-pattern update vs refactor vs fresh setup on the bench's N=1 workload: 200^3 Laplacian, 8 box subdomains, geneo
ASM,1 tau 0.1, CG rtol 1e-5.  Problem A has --kappa 2 lin, problem B --kappa 50 lin (same mesh, same partition).

Two 200^3 preconditioners do not fit one GPU together, so everything runs in sequence in one process:
setup(A) (also warms the process: its first upload is slow) -> update(B) -> refactor() -> CG -> destroy -> setup(B) -> CG.
Prints one JSON line (and writes it to --out when given).

Under `python -m torch.distributed.run --nproc-per-node N` it runs the bench's weak-scaling unit instead: one process per
GPU, edge weak_edge(size, N) as in bench.py, 8 box subdomains per GPU, and the same sequence with setup_dist (the fresh
setup includes the rank layout and the halo request exchange, which the update keeps).  Every time is the slowest rank's;
the update is split into the host rebuild of the rank layout, the value placement (uploads, device checks, the vote of the
ranks) and the numeric setup.  --dist runs this sequence with one process too (under torch.distributed.run
--nproc-per-node 1): a rank's own share of the update at the weak-scaling unit's size, without the halo traffic."""
import argparse
import gc
import json
import math
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


def weak_edge(size, world):
    # bench.py's weak-scaling rule (the reference's, incl. its float truncation)
    return size if world == 1 else int(math.floor((float(size) ** 3 * world) ** (1.0 / 3.0) + 1e-9))


def main_dist(a, rank, world, local):
    import torch
    import torch.distributed as tdist
    torch.cuda.set_device(local)
    tdist.init_process_group("gloo")  # rendezvous and the result gather only; the data path is the library's NCCL
    edge = weak_edge(a.size, world)
    K, rg, sub_rank = dist.box_grid(world, 8)
    lo, hi = dist.keep_region(edge, K, rg, rank, 8) if world > 1 else (None, None)
    args = "--dim 3 --size %d --inpEps 0.0001 --kappa %%s lin" % edge

    def problem_dist(kappa):
        prob = g.Problem()
        assert dist.generate_boxed(prob, "laplacian", args % kappa, K, lo, hi) == edge
        dist.decompose_owned(prob, len(sub_rank), sub_rank, rank, True, 0)
        return prob

    def setup_dist(prob):
        pc = g.GeneoPC(OPTS)
        lay = dist.Layout(prob, rank, world, sub_rank)
        lay.exchange_requests(tdist)
        return dist.setup_dist(pc, prob, lay, dist.nccl_unique_id(tdist, rank))

    def timed_all(fn):  # every rank starts together; the caller reports the slowest rank
        tdist.barrier()
        return timed(fn)

    def solve_dist(pc):
        n_own, n_loc = dist.local_sizes(pc)
        owned = pc.layout.owned
        ones, b, x = (torch.zeros(n_loc, dtype=torch.float64, device="cuda") for _ in range(3))
        ones[:n_own] = torch.from_numpy(owned.astype(np.float64) + 1.0).cuda()
        pc.mult_device(ones.data_ptr(), b.data_ptr())  # b = A (1..N), as bench.py
        r = pc.ksp_solve_device(b.data_ptr(), x.data_ptr(), ksp="cg", rtol=1e-5, atol=1e-50)
        v = torch.zeros_like(x)
        v[:n_own] = torch.from_numpy(np.sin(owned * 0.37)).cuda()
        pc.mult_device(v.data_ptr(), b.data_ptr())
        torch.cuda.synchronize()
        return r["its"], r["reason"], x[:n_own].cpu().numpy(), b[:n_own].cpu().numpy()

    pa, pb = problem_dist("2"), problem_dist("50")
    box = {}
    t_setup_a = timed_all(lambda: box.update(pc=setup_dist(pa)))
    pc = box.pop("pc")
    c0 = g.counters()
    t_update = timed_all(lambda: pc.update(pb))
    c1 = g.counters()
    tm = pc.timers()
    t_refactor = timed_all(pc.refactor)
    its_u, reason_u, x_u, av_u = solve_dist(pc)
    ne_u = pc.info()["nE"]
    del pc
    gc.collect()
    t_fresh = timed_all(lambda: box.update(pc=setup_dist(pb)))
    fresh = box.pop("pc")
    its_f, reason_f, x_f, av_f = solve_dist(fresh)
    ne_f = fresh.info()["nE"]
    name, limit = gpu_name_and_power_limit()
    mine = dict(setup_A_s=t_setup_a, update_s=t_update, update_layout_s=tm["update_layout"], update_numeric_s=tm["numeric"],
                update_values_s=t_update - tm["update_layout"] - tm["numeric"], refactor_s=t_refactor, fresh_setup_s=t_fresh,
                h2d=c1["h2d"] - c0["h2d"], launches=c1["launches"] - c0["launches"], bitwise=bool(np.array_equal(av_u, av_f)),
                dx2=float(np.sum((x_u - x_f) ** 2)), x2=float(np.sum(x_f ** 2)))
    everyone = [None] * world
    tdist.all_gather_object(everyone, mine)
    del fresh
    tdist.destroy_process_group()
    if rank != 0:
        return
    slowest = {k: round(max(o[k] for o in everyone), 3) for k in mine if k.endswith("_s")}
    res = {
        "workload": "laplacian3d %d^3 on %d GPU(s) through setup_dist (weak scaling, bench.py's edge), %d box subdomains (8 per GPU), geneo ASM,1 "
                    "tau=0.1, CG rtol 1e-5; A: --kappa 2 lin, B: --kappa 50 lin; times: slowest rank" % (edge, world, len(sub_rank)),
        "gpu": name, "power_limit": limit, "world": world,
        **slowest,
        "update_h2d_bytes": sum(o["h2d"] for o in everyone),
        "update_h2d_bytes_max_rank": max(o["h2d"] for o in everyone),
        "update_launches_max_rank": max(o["launches"] for o in everyone),
        "updated": {"its": its_u, "reason": reason_u, "nE": ne_u},
        "fresh": {"its": its_f, "reason": reason_f, "nE": ne_f},
        "x_rel_diff": math.sqrt(sum(o["dx2"] for o in everyone) / sum(o["x2"] for o in everyone)),
        "mult_bitwise_equal": all(o["bitwise"] for o in everyone),
    }
    emit(res, a.out)


def emit(res, out):
    line = json.dumps(res)
    print(line)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(line + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=200)
    ap.add_argument("--out", default=None)
    ap.add_argument("--dist", action="store_true", help="the multi-GPU sequence also with one process (one rank's share of it)")
    a = ap.parse_args()
    if g.device_count() < 1:
        raise SystemExit("update_target.py: no CUDA device -- the library has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 or a.dist:
        return main_dist(a, int(os.environ["RANK"]), world, int(os.environ.get("LOCAL_RANK", "0")))
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
    emit(res, a.out)


if __name__ == "__main__":
    main()
