"""Same-pattern update of a multi-GPU preconditioner (geneo_pc_update on a PC from geneo_pc_setup_dist): every rank passes
its own problem, built like the setup's from the same partition and sub_rank; afterwards each rank holds what a fresh
setup_dist on the new problems builds -- the owned operator rows bit for bit, the same coarse space, applies and
iterations --, and a problem rejected on one rank only makes every rank fail and keep its previous preconditioner.

The two-rank tests need 2 GPUs (one process per GPU, spawned like tests/test_gpu_dist.py).  The one-rank tests run the
same multi-GPU code path (rank layout, owned-row placement, vote) with world = 1 on a single GPU."""
import os
import queue
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

EDGE = 32
LAP = "--dim 3 --size %d --inpEps 0.0001 --kappa %%s lin" % EDGE
HEAT = "--dim 3 --size %d --inpEps 0.0001 --kappa 100. minmax --lbd 1. --dt %%s" % EDGE
# name -> (kind, (args of problem 1, args of problem 2), -geneo_lvl, extra options, ksp, partition)
CASES = {
    "asm_box": ("laplacian", (LAP % "2.", LAP % "50."), "ASM,1", [], "cg", "box"),
    "soras2_box": ("laplacian", (LAP % "2.", LAP % "50."), "SORAS,2", ["-geneo_optim", "0.5"], "gmres", "box"),
    "hybrid_box": ("laplacian", (LAP % "2.", LAP % "50."), "ASM,H1", [], "gmres", "box"),
    "asm_metis": ("laplacian", (LAP % "2.", LAP % "50."), "ASM,1", [], "cg", "metis"),
    "heat_box": ("heat", (HEAT % "0.1", HEAT % "0.05"), "ASM,1", [], "cg", "box"),
}
METIS_PARTS = 6


def _opts(case):
    lvl, extra = CASES[case][2], CASES[case][3]
    tau = "0.1" if lvl.endswith("2") else "0.2"
    return ["-geneo_lvl", lvl, "-geneo_tau", tau, "-els2_eps_tol", "1e-10"] + list(extra)


def _problem(g, dist, case, which, world, rank, overlap=0, decompose=True):
    """Problem 1 or 2 of `case` as rank `rank` of `world` builds it; returns (problem, sub_rank)."""
    kind, args, partition = CASES[case][0], CASES[case][1][which - 1], CASES[case][5]
    if partition == "box":
        K, grid, sub_rank = dist.box_grid(world)
        lo, hi = dist.keep_region(EDGE, K, grid, rank) if world > 1 else (None, None)
        prob = g.Problem()
        dist.generate_boxed(prob, kind, args, K, lo, hi)
        if decompose:
            dist.decompose_owned(prob, len(sub_rank), sub_rank, rank, True, overlap)
        return prob, sub_rank
    prob = g.Problem().generate(kind, args)
    return prob, dist.metis_problem(prob, METIS_PARTS, world, rank)


def _setup(g, dist, tdist, opts, prob, sub_rank, world, rank):
    lay = dist.Layout(prob, rank, world, sub_rank)
    if world > 1:
        lay.exchange_requests(tdist)
    uid = dist.nccl_unique_id(tdist, rank) if world > 1 else None
    return dist.setup_dist(g.GeneoPC(opts), prob, lay, uid)


def _state(pc, ksp, n_sub):
    """What this rank's part of the preconditioner gives: A x and M^-1 x on the owned rows, the coarse space, a solve."""
    import torch
    from geneo4petsc_b200 import dist
    owned = pc.layout.owned
    n_own, n_loc = dist.local_sizes(pc)
    xg = np.random.default_rng(11).standard_normal(EDGE ** 3)
    x = torch.zeros(n_loc, dtype=torch.float64, device="cuda")
    x[:n_own] = torch.from_numpy(xg[owned]).cuda()
    y = torch.zeros_like(x)
    pc.mult_device(x.data_ptr(), y.data_ptr())
    torch.cuda.synchronize()
    ax = y[:n_own].cpu().numpy()
    pc.apply_device(x.data_ptr(), y.data_ptr())
    torch.cuda.synchronize()
    mx = y[:n_own].cpu().numpy()
    ones = torch.zeros_like(x)
    ones[:n_own] = torch.from_numpy(owned.astype(np.float64) + 1.0).cuda()
    b, sol = torch.zeros_like(x), torch.zeros_like(x)
    pc.mult_device(ones.data_ptr(), b.data_ptr())
    r = pc.ksp_solve_device(b.data_ptr(), sol.data_ptr(), ksp=ksp, rtol=1e-8, atol=1e-50)
    torch.cuda.synchronize()
    subs = [(pc.sub_info(s), np.sort(pc.sub_eigenvalues(s))) for s in range(n_sub)]
    return dict(owned=owned.copy(), xg=xg, ax=ax, mx=mx, sol=sol[:n_own].cpu().numpy(), its=r["its"], reason=r["reason"],
                nE=pc.info()["nE"], subs=subs)


def _assert_same_state(u, f):
    """u: the updated PC, f: a fresh setup_dist on the same problems (this rank's parts)."""
    assert np.array_equal(u["owned"], f["owned"])
    assert np.array_equal(u["ax"], f["ax"])  # the owned operator rows bit for bit
    assert u["nE"] == f["nE"]
    for (a, ea), (b, eb) in zip(u["subs"], f["subs"]):
        for k in ("estim", "nev", "neg", "perturbed"):
            assert a[k] == b[k], (k, a, b)
        np.testing.assert_allclose(ea, eb, rtol=1e-9, atol=1e-14)
    assert np.linalg.norm(u["mx"] - f["mx"]) <= 1e-9 * np.linalg.norm(f["mx"])
    assert u["reason"] > 0 and f["reason"] > 0 and abs(u["its"] - f["its"]) <= 1, (u["its"], f["its"])


def _assert_matches_single_gpu(g, dist, case, gathered):
    """The gathered multi-GPU result against the single-GPU setup of problem 2 on the same partition (tolerances of
    test_gpu_dist.test_two_gpu_solve_matches_single_gpu)."""
    kind, args, lvl, ksp, partition = CASES[case][0], CASES[case][1][1], CASES[case][2], CASES[case][4], CASES[case][5]
    n = EDGE ** 3
    if partition == "box":
        K, _, sub_rank = dist.box_grid(len(gathered))
        ref = g.Problem()
        dist.generate_boxed(ref, kind, args, K)
        eptr, eidx, _ = ref.mesh()
        first = eidx[eptr[:-1]]
        i, j, l = first % EDGE, (first // EDGE) % EDGE, first // (EDGE * EDGE)
        ep = ((i * K[0]) // EDGE + K[0] * ((j * K[1]) // EDGE + K[1] * ((l * K[2]) // EDGE))).astype(np.int32)
        ref.decompose(len(sub_rank), True, 0, elem_part=ep)
    else:
        ref = g.Problem().generate(kind, args)
        ref.decompose(METIS_PARTS, True, 0)
        assert np.array_equal(ref.partition()[0], gathered[0]["partition"])
    pc1 = g.GeneoPC(_opts(case)).setup(ref)
    xg = gathered[0]["xg"]
    ax1, mx1 = pc1.mult(xg), pc1.apply(xg)
    r1 = pc1.ksp_solve(pc1.make_rhs(), ksp=ksp, rtol=1e-8, atol=1e-50)
    ax_d, mx_d, sol_d = np.zeros(n), np.zeros(n), np.zeros(n)
    for o in gathered:
        ax_d[o["owned"]] = o["ax"]; mx_d[o["owned"]] = o["mx"]; sol_d[o["owned"]] = o["sol"]
    np.testing.assert_allclose(ax_d, ax1, rtol=1e-11, atol=1e-11)
    assert all(pc1.info()["nE"] == o["nE"] for o in gathered)
    tol = 1e-4 if lvl.endswith("2") else 1e-6
    assert np.linalg.norm(mx_d - mx1) <= tol * np.linalg.norm(mx1), np.linalg.norm(mx_d - mx1) / np.linalg.norm(mx1)
    assert all(o["reason"] > 0 for o in gathered) and r1["reason"] > 0
    assert abs(gathered[0]["its"] - r1["its"]) <= 1, (gathered[0]["its"], r1["its"])
    assert np.linalg.norm(sol_d - r1["x"]) <= 1e-6 * np.linalg.norm(r1["x"])


def _update_case(case, world, rank, tdist):
    """setup_dist(p1) -> update(p2) against a fresh setup_dist(p2), then (ASM box) the round trip back to p1."""
    import geneo4petsc_b200 as g
    from geneo4petsc_b200 import dist
    ksp = CASES[case][4]
    p1, sr1 = _problem(g, dist, case, 1, world, rank)
    p2, sr2 = _problem(g, dist, case, 2, world, rank)
    assert np.array_equal(sr1, sr2)
    if CASES[case][5] == "metis":
        assert np.array_equal(p1.partition()[0], p2.partition()[0])  # one partition for both problems
    n_sub = int(np.sum(np.asarray(sr1) == rank))
    pc = _setup(g, dist, tdist, _opts(case), p1, sr1, world, rank)
    layout = pc.layout
    s1 = _state(pc, ksp, n_sub)
    assert pc.update(p2) is pc
    assert pc.problem is p2 and pc.layout is layout  # the new problem is kept alive, the layout stays the setup's
    u = _state(pc, ksp, n_sub)
    assert not np.array_equal(u["ax"], s1["ax"])
    fresh = _setup(g, dist, tdist, _opts(case), p2, sr2, world, rank)
    _assert_same_state(u, _state(fresh, ksp, n_sub))
    del fresh
    if case == "asm_box":
        pc.update(p1)
        back = _state(pc, ksp, n_sub)
        assert np.array_equal(back["ax"], s1["ax"])
        assert np.linalg.norm(back["mx"] - s1["mx"]) <= 1e-9 * np.linalg.norm(s1["mx"])
    u["partition"] = p2.partition()[0] if CASES[case][5] == "metis" else None
    del u["subs"]
    gathered = [u]
    if world > 1:
        gathered = [None] * world
        tdist.all_gather_object(gathered, u)
    if rank == 0:
        _assert_matches_single_gpu(g, dist, case, gathered)
    del pc


def _rejections(world, rank, tdist):
    """A problem only some ranks cannot use: every rank raises, keeps its preconditioner and still solves as before."""
    import geneo4petsc_b200 as g
    from geneo4petsc_b200 import dist
    case = "asm_box"
    p1, sr = _problem(g, dist, case, 1, world, rank)
    pc = _setup(g, dist, tdist, _opts(case), p1, sr, world, rank)
    n_sub = int(np.sum(np.asarray(sr) == rank))
    s0 = _state(pc, "cg", n_sub)
    # (rejecting rank, its problem, its own message); with one rank both come from rank 0
    bad = [(world - 1, lambda: _problem(g, dist, case, 2, world, rank, overlap=1)[0], "node"),
           (0, lambda: _problem(g, dist, case, 2, world, rank, decompose=False)[0], "no decomposed problem")]
    for who, make, own in bad:
        prob = make() if rank == who else _problem(g, dist, case, 2, world, rank)[0]
        with pytest.raises(g.GeneoError) as e:
            pc.update(prob)
        msg = str(e.value)
        if rank == who:
            assert own in msg, msg
        else:
            assert "rejected by rank %d" % who in msg, msg
        s = _state(pc, "cg", n_sub)
        assert np.array_equal(s["ax"], s0["ax"])
        assert np.linalg.norm(s["mx"] - s0["mx"]) <= 1e-12 * np.linalg.norm(s0["mx"])
        assert s["reason"] > 0 and s["its"] == s0["its"]
    del pc


def _worker(rank, world, port, what, case, q):
    try:
        import faulthandler
        faulthandler.dump_traceback_later(200, exit=True)  # a rank stuck in a collective shows where, then dies
        sys.path.insert(0, ROOT)
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        import torch
        import torch.distributed as tdist
        torch.cuda.set_device(rank)
        tdist.init_process_group("gloo", rank=rank, world_size=world)  # rendezvous only; the data path is the library's NCCL
        if what == "update":
            _update_case(case, world, rank, tdist)
        else:
            _rejections(world, rank, tdist)
        tdist.barrier()
        tdist.destroy_process_group()
        q.put((rank, "ok"))
    except BaseException as e:  # noqa: BLE001  (pytest.raises failures are BaseException subclasses)
        import traceback
        q.put((rank, "fail: %s\n%s" % (e, traceback.format_exc())))


def _two_ranks(what, case, port_offset):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 28700 + (os.getpid() % 500) + port_offset
    procs = [ctx.Process(target=_worker, args=(r, 2, port, what, case, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = []
    try:
        for _ in procs:
            res.append(q.get(timeout=400))
            assert res[-1][1] == "ok", res[-1]  # report the first failure at once: the other rank is then stuck in a collective
    except queue.Empty:
        pytest.fail("a rank did not answer; got %r" % (res,))
    finally:
        for p in procs:
            p.join(timeout=5)
            if p.is_alive():
                p.kill()


def _one_rank():
    import torch
    if torch.cuda.device_count() < 1:
        pytest.skip("needs a GPU")
    torch.cuda.set_device(0)


@pytest.mark.parametrize("case", list(CASES))
def test_two_gpu_update_equals_fresh_setup(case):
    _two_ranks("update", case, list(CASES).index(case))


def test_two_gpu_rejection_on_one_rank_leaves_every_rank_intact():
    _two_ranks("reject", None, len(CASES))


@pytest.mark.parametrize("case", list(CASES))
def test_one_rank_update_equals_fresh_setup(case):
    _one_rank()
    _update_case(case, 1, 0, None)


def test_one_rank_rejections_leave_the_preconditioner_intact():
    _one_rank()
    _rejections(1, 0, None)
