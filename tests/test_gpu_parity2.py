"""GPU parity tests, part 2 (round 2): BASELINE configs[0] (2-D Laplacian, 4 METIS subdomains, CG), the rest of the option
matrix (-geneo_no_syl, -geneo_cst, -geneo_gamma, -geneo_cut), null-pivot semantics on floating subdomains, span(Z) instead
of M^-1 x for the clustered GenEO-2 spectrum, the shared reference ordering of box subdomains, repeated setup on one
handle, and a larger oracle comparison.  Every comparison with the oracle also asserts that no pivot was perturbed."""
import numpy as np
import pytest

import geneo4petsc_b200 as g
from oracle import geneo_oracle as go

pytestmark = pytest.mark.gpu


def _problem(mesh, nparts, dual=True, overlap=0):
    return g.Problem().set_mesh(mesh.nb_node, mesh.elem_ptr, mesh.elem_idx, mesh.mat_val).decompose(nparts, dual, overlap)


def _oracle(mesh, p, nparts, opt, dual=True, overlap=0, **kw):
    return go.run_case(mesh, nparts, opt, dual=dual, overlap=overlap, part=p.partition(), **kw)


def _assert_counts(pc, rep, nparts, eig_rtol=1e-6):
    assert pc.info()["nE"] == rep.pc.e.shape[0]
    for s in range(nparts):
        si = pc.sub_info(s)
        assert si["perturbed"] == 0, (s, si)  # a perturbed pivot of A - tau B would falsify the inertia count
        assert si["nev"] == rep.pc.sub[s].z.shape[1] and si["estim"] == rep.pc.sub[s].estim, (s, si, rep.pc.sub[s].estim)
        np.testing.assert_allclose(np.sort(pc.sub_eigenvalues(s)), np.sort(np.array(rep.pc.sub[s].eigvals)), rtol=eig_rtol, atol=1e-12)


@pytest.mark.parametrize("size", [10, 100])
def test_c1_2d_laplacian_4_metis_subdomains_cg(size):
    """BASELINE configs[0] = tst/laplacian: `--dim 2 --size S --kappa 2. lin --inpEps 0.0001`, 4 subdomains --metisDual,
    -geneo_lvl ASM,1 -geneo_tau 0.1, CG with rtol = atol = 1e-5 (tst/laplacian/laplacianRun.sh:30,140)."""
    mesh = go.gen_grid(2, size, 1e-4, 2.0, "lin")
    p = _problem(mesh, 4)
    pc = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.1"]).setup(p)
    assert pc.name == "geneo1ASM"
    rep = _oracle(mesh, p, 4, go.GenEOOptions(lvl1="ASM", lvl2="1", tau=0.1), ksp="cg", rtol=1e-5, atol=1e-5)
    x = np.random.default_rng(0).standard_normal(mesh.nb_node)
    np.testing.assert_allclose(pc.mult(x), rep.a @ x, rtol=1e-12, atol=1e-12)
    _assert_counts(pc, rep, 4)
    b = pc.make_rhs()
    np.testing.assert_allclose(b, rep.b, rtol=1e-12, atol=1e-12 * np.abs(rep.b).max())  # (b = A (1..N): cancellation in the rows)
    r = pc.ksp_solve(b, ksp="cg", rtol=1e-5, atol=1e-5)
    assert r["reason"] > 0 and rep.ksp.converged
    assert abs(r["its"] - rep.ksp.its) <= 1, (r["its"], rep.ksp.its)
    # (the KSP tests the PRECONDITIONED residual, like the reference: the true one is whatever the oracle reaches too)
    assert np.linalg.norm(rep.a @ r["x"] - b) <= max(10 * rep.true_rel_res, 1e-4) * np.linalg.norm(b)


@pytest.mark.parametrize("lvl,extra,okw", [
    ("ASM,1", ["-geneo_no_syl"], dict(no_syl=True)),
    ("SORAS,2", ["-geneo_cst"], dict(cst=True)),
    ("SORAS,2", ["-geneo_gamma", "5"], dict(gamma=5.0)),
    ("SORAS,2", ["-geneo_cst", "-geneo_gamma", "3", "-geneo_cut", "6"], dict(cst=True, gamma=3.0, cut=6)),
    ("ASM,1", ["-geneo_cut", "3"], dict(cut=3)),
])
def test_remaining_option_matrix(lvl, extra, okw):
    """-geneo_no_syl (src/geneo.cpp:2434), -geneo_cst (:2415), -geneo_gamma, -geneo_cut: the rest of the 58-combination
    matrix of tst/laplacian/laplacianRun.sh:31-58."""
    mesh, nparts = go.gen_grid(3, 12, 1e-4, 2.0, "lin"), 4
    p = _problem(mesh, nparts)
    l1, l2 = lvl.split(",")
    tau = 0.3 if l2 == "1" else 0.1
    argv = ["-geneo_lvl", lvl, "-geneo_tau", str(tau), "-geneo_optim", "0.5", "-els2_eps_tol", "1e-9"] + extra
    pc = g.GeneoPC(argv).setup(p)
    rep = _oracle(mesh, p, nparts, go.GenEOOptions(lvl1=l1, lvl2=l2, tau=tau, optim=0.5, **okw), ksp="gmres", rtol=1e-6, atol=1e-6)
    _assert_counts(pc, rep, nparts)
    for s in range(nparts):
        si = pc.sub_info(s)
        if l2 == "2" and not okw.get("cst"):
            assert abs(si["tauLoc"] - rep.pc.sub[s].tau_loc) < 1e-12 and abs(si["gammaLoc"] - rep.pc.sub[s].gamma_loc) < 1e-9
    r = pc.ksp_solve(pc.make_rhs(), ksp="gmres", rtol=1e-6, atol=1e-6)
    assert r["reason"] > 0 and abs(r["its"] - rep.ksp.its) <= 1, (r["its"], rep.ksp.its)


def _principal_angle_sines(z1, z2):
    q1, _ = np.linalg.qr(z1)
    q2, _ = np.linalg.qr(z2)
    c = np.clip(np.linalg.svd(q1.T @ q2, compute_uv=False), 0.0, 1.0)
    return np.sqrt(1.0 - c ** 2)


def test_geneo2_span_of_z_matches_the_oracle():
    """Q = Z E^-1 Z^T only depends on span(Z_i).  For GenEO-2 the (A_neu, A_rob) spectrum clusters at the threshold, so
    M^-1 x is compared loosely elsewhere (1e-4); here the invariant itself: with the default eigen tolerance every kept
    eigen-direction well inside the threshold lies in the oracle's span to 1e-5 (sines of the principal angles), and with a
    tight tolerance the whole span does to 1e-7."""
    mesh, nparts = go.gen_grid(3, 12, 1e-4, 2.0, "lin"), 4
    p = _problem(mesh, nparts)
    rep = _oracle(mesh, p, nparts, go.GenEOOptions(lvl1="SORAS", lvl2="2", tau=0.1, optim=0.5), ksp="gmres", rtol=1e-6)
    tight = g.GeneoPC(["-geneo_lvl", "SORAS,2", "-geneo_tau", "0.1", "-geneo_optim", "0.5", "-els2_eps_tol", "1e-10"]).setup(p)
    loose = g.GeneoPC(["-geneo_lvl", "SORAS,2", "-geneo_tau", "0.1", "-geneo_optim", "0.5"]).setup(p)
    for s in range(nparts):
        zo = rep.pc.sub[s].z
        assert tight.sub_z(s).shape == zo.shape == loose.sub_z(s).shape
        assert _principal_angle_sines(tight.sub_z(s), zo).max() < 1e-7
        assert _principal_angle_sines(loose.sub_z(s), zo).max() < 2e-3  # default tolerance: residual 1e-4 next to a cluster
    x = np.random.default_rng(3).standard_normal(mesh.nb_node)
    yo = rep.pc.apply(x)
    assert np.linalg.norm(tight.apply(x) - yo) <= 1e-8 * np.linalg.norm(yo)


def test_floating_subdomains_null_pivot_semantics():
    """--inpEps 0: the Neumann matrix of a subdomain that does not touch the Dirichlet face is singular (constant kernel).
    The reference leans on MUMPS null-pivot detection with a huge fixation (ICNTL(24)=1, CNTL(5)=1e20, src/geneo.cpp:81-83)
    and on the Nicolaides rule (:897-944) to put the constant vector into Z exactly once.  Same here: the solve converges to
    (1..N), E is positive definite, and the floating subdomains report a Nicolaides vector."""
    mesh, nparts = go.gen_grid(3, 12, 0.0, 1.0, ""), 4
    p = _problem(mesh, nparts)
    pc = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.2"]).setup(p)
    info = pc.info()
    einv = pc.coarse_inverse()
    assert np.isfinite(einv).all()
    w = np.linalg.eigvalsh(0.5 * (einv + einv.T))
    assert w.min() > 0, w.min()  # no duplicated constant vector: E (hence E^-1) is SPD
    assert info["nicolaides"] >= 1
    b = pc.make_rhs()
    r = pc.ksp_solve(b, ksp="cg", rtol=1e-8, atol=1e-50)
    assert r["reason"] > 0
    np.testing.assert_allclose(r["x"], np.arange(1, mesh.nb_node + 1.0), rtol=1e-4)


def test_setup_twice_on_one_handle():
    """PCSetUp repeated on the same PC with a NEW problem (other pattern, other size): nothing of the first one may survive
    (the forest held raw pointers into the old plans)."""
    m1, m2 = go.gen_grid(3, 10, 1e-4, 2.0, "lin"), go.gen_grid(3, 12, 1e-4)
    p1, p2 = _problem(m1, 3), _problem(m2, 4)
    pc = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.3", "-els2_eps_tol", "1e-10"])
    pc.setup(p1)
    x1 = np.random.default_rng(7).standard_normal(m1.nb_node)
    y1 = pc.apply(x1)
    pc.setup(p2)
    fresh = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.3", "-els2_eps_tol", "1e-10"]).setup(p2)
    x2 = np.random.default_rng(8).standard_normal(m2.nb_node)
    assert pc.info()["nE"] == fresh.info()["nE"]
    assert np.linalg.norm(pc.apply(x2) - fresh.apply(x2)) <= 1e-10 * np.linalg.norm(fresh.apply(x2))
    pc.setup(p1)
    assert np.linalg.norm(pc.apply(x1) - y1) <= 1e-10 * np.linalg.norm(y1)


def test_sequential_and_pipelined_numeric_setup_agree(monkeypatch):
    """The pipelined numeric setup (independent factorizations on several streams, eigen-solves overlapped) computes what
    the one-after-the-other path computes."""
    mesh, nparts = go.gen_grid(3, 16, 1e-4, 2.0, "lin"), 6
    p = _problem(mesh, nparts)
    argv = ["-geneo_lvl", "ASM,1", "-geneo_tau", "0.3", "-els2_eps_tol", "1e-10"]
    x = np.random.default_rng(4).standard_normal(mesh.nb_node)
    monkeypatch.setenv("GENEO_PIPELINE", "0")
    seq = g.GeneoPC(argv).setup(p)
    monkeypatch.setenv("GENEO_PIPELINE", "1")
    pip = g.GeneoPC(argv).setup(p)
    assert [seq.sub_info(s)["nev"] for s in range(nparts)] == [pip.sub_info(s)["nev"] for s in range(nparts)]
    assert [seq.sub_info(s)["neg"] for s in range(nparts)] == [pip.sub_info(s)["neg"] for s in range(nparts)] == [0] * nparts
    ys, yp = seq.apply(x), pip.apply(x)
    assert np.linalg.norm(ys - yp) <= 1e-9 * np.linalg.norm(ys)
    pip.refactor()
    assert np.linalg.norm(pip.apply(x) - yp) <= 1e-9 * np.linalg.norm(yp)


def test_box_subdomains_share_one_ordering():
    """Box partition of a structured grid: the 8 subdomains inherit the reference nested dissection of their bounding box
    (one METIS call instead of eight).  Same preconditioner as with one ordering per subdomain; factor size within 15 %."""
    from geneo4petsc_b200 import dist
    edge = 56  # 8 boxes of 28^3 (+ one interface plane) >= 20 000 nodes: the sharing rule applies
    outs = []
    for reuse in ("1", "0"):
        prob = g.Problem()
        K, rg, sub_rank = dist.box_grid(1, 8)
        assert dist.generate_boxed(prob, "laplacian", "--dim 3 --size %d --inpEps 0.0001" % edge, K) == edge
        dist.decompose_owned(prob, 8, sub_rank, 0, True, 0)
        pc = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.1", "-els2_eps_tol", "1e-10", "-geneo_ordering_reuse", reuse]).setup(prob)
        b = pc.make_rhs()
        r = pc.ksp_solve(b, ksp="cg", rtol=1e-8, atol=1e-50)
        assert r["reason"] > 0
        xe = np.arange(1, edge ** 3 + 1.0)
        assert np.linalg.norm(r["x"] - xe) <= 1e-6 * np.linalg.norm(xe)
        outs.append((pc.info()["nE"], r["its"], pc.stats()["factor_bytes"], pc.factor_stats()["ordering_reuse_s"],
                     pc.apply(np.sin(np.arange(edge ** 3) * 0.1))))
    assert outs[0][0] == outs[1][0] and abs(outs[0][1] - outs[1][1]) <= 1
    assert outs[0][2] <= 1.15 * outs[1][2]
    assert np.linalg.norm(outs[0][4] - outs[1][4]) <= 1e-8 * np.linalg.norm(outs[1][4])


@pytest.mark.slow
def test_80_cubed_against_the_oracle():
    """512 000 DOFs, 8 METIS subdomains (64 000 DOFs each): iteration count, coarse dimension, eigen-counts and eigenvalues
    against the oracle (scipy SuperLU / ARPACK; ~1 min of CPU)."""
    mesh, nparts = go.gen_grid(3, 80, 1e-4), 8
    p = _problem(mesh, nparts)
    pc = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.1"]).setup(p)
    rep = _oracle(mesh, p, nparts, go.GenEOOptions(lvl1="ASM", lvl2="1", tau=0.1), ksp="cg", rtol=1e-5, workers=8)
    _assert_counts(pc, rep, nparts)
    r = pc.ksp_solve(pc.make_rhs(), ksp="cg", rtol=1e-5, atol=1e-50)
    assert r["reason"] > 0 and abs(r["its"] - rep.ksp.its) <= 1, (r["its"], rep.ksp.its)
    assert np.linalg.norm(r["x"] - rep.ksp.x) <= 1e-4 * np.linalg.norm(rep.ksp.x)


def test_check_and_debug_files(tmp_path, monkeypatch):
    """-geneo_chk log / -geneo_dbg log,2 (src/geneo.cpp:2438-2480): the per-subdomain diagnostics the reference writes next to
    the run -- SPD check through the inertia (:782-840), rank of Z through the diagonal of R (:173-247), partition of unity
    (:988-997), eigenvalue / Sylvester-inertia logs (:344-349, :547-551), the timing log at destroy (:2189-2216)."""
    monkeypatch.chdir(tmp_path)
    mesh, nparts = go.gen_grid(3, 12, 1e-4, 2.0, "lin"), 4
    p = _problem(mesh, nparts)
    pc = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.3", "-geneo_chk", "log", "-geneo_dbg", "log,2"]).setup(p)
    rep = _oracle(mesh, p, nparts, go.GenEOOptions(lvl1="ASM", lvl2="1", tau=0.3), ksp="cg", rtol=1e-6)
    for s in range(nparts):
        spd = (tmp_path / ("check%d.SPD.ADir.log" % s)).read_text()
        assert "ADir - inertia: nbNegEV 0, nbNullEV 0, nbPosEV %d" % pc.sub_info(s)["n"] in spd
        r = np.loadtxt(tmp_path / ("check%d.setup.Z.R" % s), ndmin=2)
        assert r.shape == (pc.sub_info(s)["nev"],) * 2 and np.all(np.abs(np.diag(r)) > 1e-12)
        ev = (tmp_path / ("debug%d.setup.Z.ev.log" % s)).read_text()
        assert "Z - nb of eigen values: %d" % pc.sub_info(s)["nev"] in ev
        syl = (tmp_path / ("debug%d.setup.tau.sylvester.inertia.log" % s)).read_text()
        assert "=> estim %d" % rep.pc.sub[s].estim in syl and "nbNegEV %d," % rep.pc.sub[s].estim in syl
    pc.ksp_solve(pc.make_rhs(), ksp="cg", rtol=1e-6)
    del pc
    import gc
    gc.collect()
    t = (tmp_path / "debug0.timing.log").read_text()
    assert "lvl1SetupMinvTimeLoc" in t and "lvl2SetupEigTimeLoc" in t and " ms" in t
    # a matrix that is not SPD is caught by the check (the reference aborts, src/geneo.cpp:829-832)
    ids = [p.sub_nodes(s)[0] for s in range(nparts)]
    bad = [(ids[s], p.sub_matrix(s, 0) * (-1.0 if s == 1 else 1.0), p.sub_matrix(s, 1) * (-1.0 if s == 1 else 1.0)) for s in range(nparts)]
    q = g.Problem().set_subdomains(mesh.nb_node, bad)
    with pytest.raises(g.GeneoError, match="not SPD"):
        g.GeneoPC(["-geneo_lvl", "ASM,0", "-geneo_chk", "log"]).setup(q)
