"""Blocks of right-hand sides (PCMatApply / KSPMatSolve with CG): apply_block against apply column by column for every PC
variant, block widths that are and are not multiples of 8, and lock-step block CG against ksp_solve(b_j, "cg") column by
column -- on a single-GPU PC, after re-setups, and on a multi-GPU PC with one rank (one GPU) and with two ranks (2 GPUs,
spawned like tests/test_gpu_dist.py).  The argument checks that need no set-up PC run without a GPU."""
import os
import queue
import sys

import numpy as np
import pytest

import geneo4petsc_b200 as g
from oracle import geneo_oracle as go

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
NPARTS = 4
WIDTHS = (1, 5, 8, 13, 16)
VARIANTS = [("ASM,0", []), ("ASM,1", []), ("RAS,1", []), ("SRAS,1", []), ("ORAS,1", ["-geneo_optim", "0.5"]),
            ("SORAS,2", ["-geneo_optim", "0.5"]), ("ASM,H1", []), ("ASM,E1", [])]


def _mesh(heat=False, kappa=2.0):
    if heat:
        return go.gen_grid(3, 12, 1e-4, 100.0, "minmax", heat=True)
    return go.gen_grid(3, 12, 1e-4, kappa, "lin")


def _problem(mesh, part=None):
    p = g.Problem().set_mesh(mesh.nb_node, mesh.elem_ptr, mesh.elem_idx, mesh.mat_val)
    if part is None:
        return p.decompose(NPARTS, True, 0)
    return p.decompose(NPARTS, True, 0, elem_part=part[0], node_part=part[1])


def _pc(lvl, extra=(), mesh=None):
    tau = "0.1" if lvl.endswith("2") else "0.3"
    p = _problem(mesh if mesh is not None else _mesh())
    return g.GeneoPC(["-geneo_lvl", lvl, "-geneo_tau", tau, "-els2_eps_tol", "1e-10"] + list(extra)).setup(p)


def _assert_block_apply(pc, X):
    Y = pc.apply_block(X)
    assert Y.shape == X.shape
    for j in range(X.shape[1]):
        y = pc.apply(X[:, j])
        assert np.linalg.norm(Y[:, j] - y) <= 1e-9 * np.linalg.norm(y), (j, np.linalg.norm(Y[:, j] - y) / np.linalg.norm(y))


def _assert_block_cg(pc, B, rtol=1e-10):
    r = pc.ksp_solve_block(B, ksp="cg", rtol=rtol)
    for j in range(B.shape[1]):
        s = pc.ksp_solve(B[:, j], ksp="cg", rtol=rtol)
        assert r["reason"][j] == s["reason"], (j, r["reason"][j], s["reason"])
        assert abs(int(r["its"][j]) - s["its"]) <= 1, (j, r["its"][j], s["its"])
        assert np.linalg.norm(r["x"][:, j] - s["x"]) <= 1e-6 * np.linalg.norm(s["x"]), j
    return r


# ---- argument checks (no device needed) -------------------------------------------------------------------------------
def test_block_calls_before_setup_have_no_context():
    """Checked before anything touches the device: the same message with or without a GPU."""
    pc = g.GeneoPC()
    with pytest.raises(g.GeneoError, match="without context"):
        pc.apply_block(np.ones((10, 3)))
    with pytest.raises(g.GeneoError, match="without context"):
        pc.ksp_solve_block(np.ones((10, 3)), ksp="cg")


def test_block_calls_reject_an_empty_block_and_gmres():
    """k < 1 and a Krylov method other than CG are refused before the context is looked at."""
    pc = g.GeneoPC()
    with pytest.raises(g.GeneoError, match="k must be at least 1"):
        pc.apply_block(np.ones((10, 0)))
    with pytest.raises(g.GeneoError, match="k must be at least 1"):
        pc.ksp_solve_block(np.ones((10, 0)), ksp="cg")
    with pytest.raises(g.GeneoError, match="cg only"):
        pc.ksp_solve_block(np.ones((10, 3)), ksp="gmres")


# ---- single GPU -------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("lvl,extra", VARIANTS)
def test_block_apply_matches_apply(lvl, extra):
    pc = _pc(lvl, extra)
    n = pc.info()["nbDof"]
    rng = np.random.default_rng(5)
    for k in WIDTHS:
        _assert_block_apply(pc, rng.standard_normal((n, k)))
    assert pc.stats()["applies"] >= sum(WIDTHS)


@gpu
def test_block_apply_edge_cases():
    import torch
    pc = _pc("ASM,1")
    n = pc.info()["nbDof"]
    X = np.random.default_rng(7).standard_normal((n, 11))
    X[:, 3] = 0.
    Y = pc.apply_block(X)
    assert not Y[:, 3].any()  # a zero column gives a zero column
    # device entry point: X is not written, rows n..ldy-1 of Y are not written
    k, ldx, ldy = 11, n + 3, n + 5
    dX = torch.zeros((k, ldx), dtype=torch.float64, device="cuda")  # column-major (ldx, k)
    dX[:, :n] = torch.from_numpy(X.T.copy()).cuda()
    dX[:, n:] = 7.0
    dX0 = dX.clone()
    dY = torch.full((k, ldy), -3.0, dtype=torch.float64, device="cuda")
    pc.apply_block_device(dX.data_ptr(), dY.data_ptr(), k, ldx, ldy)
    torch.cuda.synchronize()
    assert torch.equal(dX, dX0)
    assert bool((dY[:, n:] == -3.0).all())
    Yd = dY[:, :n].cpu().numpy().T
    assert np.linalg.norm(Yd - Y) <= 1e-12 * np.linalg.norm(Y)
    with pytest.raises(g.GeneoError, match="leading dimension"):
        pc.apply_block_device(dX.data_ptr(), dY.data_ptr(), k, n - 1, ldy)
    with pytest.raises(g.GeneoError, match="leading dimension"):
        pc.ksp_solve_block_device(dX.data_ptr(), dY.data_ptr(), k, ldx, n - 1)


def _rhs_block(pc, k, seed):
    n = pc.info()["nbDof"]
    B = np.random.default_rng(seed).standard_normal((n, k))
    B[:, 1] = 0.
    B[:, 2] = pc.make_rhs()
    return B


@gpu
@pytest.mark.parametrize("case", ["ASM,1", "ASM,E1", "heat"])
@pytest.mark.parametrize("k", [8, 11])
def test_block_cg_matches_cg(case, k):
    pc = _pc("ASM,1", mesh=_mesh(heat=True)) if case == "heat" else _pc(case)
    r = _assert_block_cg(pc, _rhs_block(pc, k, 13))
    assert r["reason"][1] > 0 and r["its"][1] == 0 and all(r["reason"] > 0)


@gpu
def test_block_after_refactor_and_update():
    m1, m2 = _mesh(kappa=2.0), _mesh(kappa=50.0)
    p1 = _problem(m1)
    p2 = _problem(m2, part=p1.partition())
    pc = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.3", "-els2_eps_tol", "1e-10"]).setup(p1)
    X = np.random.default_rng(9).standard_normal((m1.nb_node, 9))
    _assert_block_apply(pc, X)
    pc.refactor()
    _assert_block_apply(pc, X)
    pc.update(p2)
    _assert_block_apply(pc, X)
    _assert_block_cg(pc, X[:, :3])


# ---- multi-GPU PC (geneo_pc_setup_dist): one rank on one GPU, two ranks on two GPUs -----------------------------------
DIST_EDGE = 16
DIST_ARGS = "--dim 3 --size %d --inpEps 0.0001 --kappa 2. lin" % DIST_EDGE


def _dist_pc(g, dist, tdist, lvl, world, rank):
    K, grid, sub_rank = dist.box_grid(world)
    lo, hi = dist.keep_region(DIST_EDGE, K, grid, rank) if world > 1 else (None, None)
    prob = g.Problem()
    dist.generate_boxed(prob, "laplacian", DIST_ARGS, K, lo, hi)
    dist.decompose_owned(prob, len(sub_rank), sub_rank, rank, True, 0)
    lay = dist.Layout(prob, rank, world, sub_rank)
    if world > 1:
        lay.exchange_requests(tdist)
    uid = dist.nccl_unique_id(tdist, rank) if world > 1 else None
    return dist.setup_dist(g.GeneoPC(["-geneo_lvl", lvl, "-geneo_tau", "0.2", "-els2_eps_tol", "1e-10"]), prob, lay, uid)


def _dist_check(pc):
    """Block apply and block CG on the rank's [owned | ghost] columns against the single-vector device entry points
    (collective: every rank makes the same calls in the same order)."""
    import torch
    from geneo4petsc_b200 import dist
    n_own, n_loc = dist.local_sizes(pc)
    owned = pc.layout.owned
    k = 11
    rng = np.random.default_rng(21)
    Xg = rng.standard_normal((DIST_EDGE ** 3, k))
    X = torch.zeros((k, n_loc), dtype=torch.float64, device="cuda")
    X[:, :n_own] = torch.from_numpy(Xg[owned].T.copy()).cuda()
    X[:, 4] = 0.
    Y = torch.zeros_like(X)
    pc.apply_block_device(X.data_ptr(), Y.data_ptr(), k, n_loc, n_loc)
    y = torch.zeros(n_loc, dtype=torch.float64, device="cuda")
    for j in range(k):
        x = X[j].clone()
        pc.apply_device(x.data_ptr(), y.data_ptr())
        torch.cuda.synchronize()
        a, b = Y[j, :n_own].cpu().numpy(), y[:n_own].cpu().numpy()
        assert np.linalg.norm(a - b) <= 1e-9 * np.linalg.norm(b), (j, np.linalg.norm(a - b), np.linalg.norm(b))
    kb = 9
    B = torch.zeros((kb, n_loc), dtype=torch.float64, device="cuda")
    ones = torch.zeros(n_loc, dtype=torch.float64, device="cuda")
    ones[:n_own] = torch.from_numpy(owned.astype(np.float64) + 1.0).cuda()
    for j in range(kb):
        if j == 1:
            continue  # a zero column
        xs = ones * (j + 1) if j == 0 else X[j].clone()
        pc.mult_device(xs.data_ptr(), B[j].data_ptr())
    Xb = torch.zeros_like(B)
    r = pc.ksp_solve_block_device(B.data_ptr(), Xb.data_ptr(), kb, n_loc, n_loc, ksp="cg", rtol=1e-10)
    torch.cuda.synchronize()
    for j in range(kb):
        b, sol = B[j].clone(), torch.zeros(n_loc, dtype=torch.float64, device="cuda")
        s = pc.ksp_solve_device(b.data_ptr(), sol.data_ptr(), ksp="cg", rtol=1e-10)
        torch.cuda.synchronize()
        xs, xb = sol[:n_own].cpu().numpy(), Xb[j, :n_own].cpu().numpy()
        assert r["reason"][j] == s["reason"] and abs(int(r["its"][j]) - s["its"]) <= 1, (j, r["its"][j], s["its"])
        assert np.linalg.norm(xb - xs) <= 1e-6 * np.linalg.norm(xs), j
    assert r["its"][1] == 0 and all(r["reason"] > 0)


@gpu
@pytest.mark.parametrize("lvl", ["ASM,1", "ASM,E1"])
def test_block_on_a_one_rank_multi_gpu_pc(lvl):
    from geneo4petsc_b200 import dist
    pc = _dist_pc(g, dist, None, lvl, 1, 0)
    _dist_check(pc)


def _worker(rank, world, port, lvl, q):
    try:
        import faulthandler
        faulthandler.dump_traceback_later(150, exit=True)  # a rank stuck in a collective shows where, then dies
        sys.path.insert(0, ROOT)
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        import torch
        import torch.distributed as tdist
        import geneo4petsc_b200 as gg
        from geneo4petsc_b200 import dist
        torch.cuda.set_device(rank)
        tdist.init_process_group("gloo", rank=rank, world_size=world)
        pc = _dist_pc(gg, dist, tdist, lvl, world, rank)
        _dist_check(pc)
        tdist.barrier()
        del pc
        tdist.destroy_process_group()
        q.put((rank, "ok"))
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, "fail: %s\n%s" % (e, traceback.format_exc())))


@gpu
@pytest.mark.parametrize("lvl", ["ASM,1", "ASM,E1"])
def test_block_on_two_gpus(lvl):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 30300 + (os.getpid() % 500) + (0 if lvl == "ASM,1" else 1)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, lvl, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = []
    try:
        for _ in procs:
            res.append(q.get(timeout=240))
            assert res[-1][1] == "ok", res[-1]
    except queue.Empty:
        pytest.fail("a rank did not answer; got %r" % (res,))
    finally:
        for p in procs:
            p.join(timeout=5)
            if p.is_alive():
                p.kill()
