"""GPU parity tests: the CUDA path (through the C ABI of include/geneo_b200.h) against the oracle on the same seeded
inputs, against the reference's tst/dummy goldens (tests/golden/dummy_goldens.json) and through size-independent
properties.  Tolerances: partition / eigen-counts / dim E identical; eigenvalues 1e-6 relative; iteration counts +-1;
final true relative residual <= 10 x rtol (the KSP tests the PRECONDITIONED norm, like the reference)."""
import numpy as np
import pytest

import geneo4petsc_b200 as g
from oracle import geneo_oracle as go
from tests._cases import golden_config

pytestmark = pytest.mark.gpu


def _problem(mesh, nparts, dual=True, overlap=0):
    return g.Problem().set_mesh(mesh.nb_node, mesh.elem_ptr, mesh.elem_idx, mesh.mat_val).decompose(nparts, dual, overlap)


def _oracle(mesh, p, nparts, opt, dual=True, overlap=0, **kw):
    return go.run_case(mesh, nparts, opt, dual=dual, overlap=overlap, part=p.partition(), **kw)


def test_dmma_tile_gemm_is_correct():
    for n in (64, 200, 513):
        rate, err = g.microbench(0, n, 1)
        assert err < 1e-10 * n, (n, err)


@pytest.fixture(scope="module")
def lap3d():
    return go.gen_grid(3, 12, 1e-4, 2.0, "lin")


@pytest.mark.parametrize("lvl", ["ASM,0", "ASM,1", "RAS,1", "SRAS,1", "ASM,H1", "ASM,E1", "SORAS,0", "SORAS,2", "SORAS,H2", "SORAS,E2", "ORAS,1"])
def test_apply_matches_oracle(lap3d, lvl):
    mesh, nparts = lap3d, 4
    p = _problem(mesh, nparts)
    l1, l2 = lvl.split(",")
    # GenEO-2 scales tau by the maximal multiplicity (tauLoc = k tau): keep the coarse space a small part of the spectrum.
    # Eigenvalues cluster near 1 for the (A_neu, A_rob) pencil, so individual eigenvectors next to the threshold are
    # ill-conditioned: a tight eigen tolerance makes the comparison with the dense oracle meaningful.
    tau = 0.3 if l2 in ("1", "H1", "E1") else 0.1
    argv = ["-geneo_lvl", lvl, "-geneo_tau", str(tau), "-geneo_optim", "0.5"]
    if l2 in ("2", "H2", "E2"):
        argv += ["-els2_eps_tol", "1e-8"]
    pc = g.GeneoPC(argv).setup(p)
    rep = _oracle(mesh, p, nparts, go.GenEOOptions(lvl1=l1, lvl2=l2, tau=tau, optim=0.5), ksp="cg", rtol=1e-6)
    rng = np.random.default_rng(0)
    x = rng.standard_normal(mesh.nb_node)
    np.testing.assert_allclose(pc.mult(x), rep.a @ x, rtol=1e-12, atol=1e-12)
    info = pc.info()
    if l2 != "0":
        assert info["nE"] == rep.pc.e.shape[0]
        for s in range(nparts):
            si = pc.sub_info(s)
            assert si["nev"] == rep.pc.sub[s].z.shape[1] and si["estim"] == rep.pc.sub[s].estim
            mine, ref = np.sort(pc.sub_eigenvalues(s)), np.sort(np.array(rep.pc.sub[s].eigvals))
            np.testing.assert_allclose(mine, ref, rtol=1e-6, atol=1e-12)
    y, yo = pc.apply(x), rep.pc.apply(x)
    # default eigen tolerance 1e-4 on the residual (reference: 1e-3, src/geneo.cpp:658): span(Z) agrees to ~1e-5
    assert np.linalg.norm(y - yo) <= 1e-4 * np.linalg.norm(yo)
    if lvl == "ASM,1":  # with a tight eigen tolerance the preconditioner is the oracle's to 1e-8
        pc2 = g.GeneoPC(["-geneo_lvl", lvl, "-geneo_tau", str(tau), "-els2_eps_tol", "1e-10"]).setup(p)
        y2 = pc2.apply(x)
        assert np.linalg.norm(y2 - yo) <= 1e-8 * np.linalg.norm(yo)


@pytest.mark.parametrize("ksp", ["cg", "gmres"])
@pytest.mark.parametrize("lvl,dual,overlap", [("ASM,1", True, 0), ("ASM,1", False, 1), ("ASM,H1", True, 1), ("ASM,E1", True, 0),
                                              ("SORAS,2", True, 0), ("ASM,0", True, 0)])
def test_ksp_iterations_match_oracle(lap3d, ksp, lvl, dual, overlap):
    if ksp == "cg" and lvl.startswith("ASM,E"):
        pytest.skip("efficient hybrid is not symmetric: GMRES only")
    mesh, nparts = lap3d, 4
    p = _problem(mesh, nparts, dual, overlap)
    l1, l2 = lvl.split(",")
    pc = g.GeneoPC(["-geneo_lvl", lvl]).setup(p)
    b = pc.make_rhs()
    rep = _oracle(mesh, p, nparts, go.GenEOOptions(lvl1=l1, lvl2=l2), dual=dual, overlap=overlap, ksp=ksp, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(b, rep.b, rtol=1e-12)
    r = pc.ksp_solve(b, ksp=ksp, rtol=1e-6, atol=1e-6)
    assert r["reason"] > 0 and rep.ksp.converged
    assert abs(r["its"] - rep.ksp.its) <= 1, (r["its"], rep.ksp.its)
    true_res = np.linalg.norm(rep.a @ r["x"] - b) / np.linalg.norm(b)
    assert true_res <= max(10 * rep.true_rel_res, 1e-5)
    np.testing.assert_allclose(r["history"][0], rep.ksp.history[0], rtol=1e-4)


def test_coarse_space_identities(lap3d):
    """Q A Z = Z  and  symmetric PC (size-independent properties)."""
    mesh, nparts = lap3d, 4
    p = _problem(mesh, nparts)
    pc = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.3"]).setup(p)
    nodes0, _ = p.sub_nodes(0)
    z0 = pc.sub_z(0)
    v = np.zeros(mesh.nb_node)
    v[nodes0] = z0[:, 0]
    import torch
    dv = torch.tensor(pc.mult(v), device="cuda")
    out = torch.zeros_like(dv)
    pc.apply_q_device(dv.data_ptr(), out.data_ptr())
    torch.cuda.synchronize()
    np.testing.assert_allclose(out.cpu().numpy(), v, atol=1e-8 * np.abs(v).max())
    rng = np.random.default_rng(1)
    a, b = rng.standard_normal(mesh.nb_node), rng.standard_normal(mesh.nb_node)
    assert abs(a @ pc.apply(b) - b @ pc.apply(a)) <= 1e-9 * abs(a @ pc.apply(b))


def test_dummy_goldens_through_the_cuda_path(dummy_goldens, dummy_inputs):
    """The reference's own 8-DOF goldens: b, converged x, nnz count, PC name -- every geneo configuration."""
    n_ok = 0
    for name, gd in sorted(dummy_goldens["goldens"].items()):
        cfg = golden_config(gd)
        if cfg is None:
            continue
        eps = 1.0 if gd["input"] == "tridiag" else 1e-4
        p = g.Problem().read_file(dummy_inputs / (gd["input"] + ".inp"), eps).decompose(2, cfg["dual"], cfg["overlap"])
        argv = ["-geneo_lvl", "%s,%s" % (cfg["lvl1"], cfg["lvl2"])] + (["-geneo_cut", "10"] if gd["input"] == "tridiag" else [])
        if cfg["offload"]:
            argv.append("-geneo_offload")
        pc = g.GeneoPC(argv).setup(p)
        b = go.read_rhs_file(str(dummy_inputs / "B.inp"), 8) if gd["input"] == "identity" else pc.make_rhs()
        np.testing.assert_allclose(b, gd["b"], atol=1e-12)
        r = pc.ksp_solve(b, ksp="gmres", rtol=1e-12, atol=1e-12)
        assert r["reason"] > 0, name
        np.testing.assert_allclose(r["x"], gd["x"], atol=2e-5)
        assert gd["info"][2].startswith("INFO: %s pc" % pc.name)
        assert ("nnz coefs %d," % p.sizes()["nnz"]) in gd["info"][0]
        n_ok += 1
    assert n_ok == 80


def test_heat_high_contrast(lap3d):
    mesh = go.gen_grid(3, 12, 1e-4, 100.0, "minmax", heat=True)
    p = _problem(mesh, 4)
    pc = g.GeneoPC(["-geneo_lvl", "ASM,1"]).setup(p)
    rep = _oracle(mesh, p, 4, go.GenEOOptions(), ksp="cg", rtol=1e-6, atol=1e-6)
    r = pc.ksp_solve(pc.make_rhs(), ksp="cg", rtol=1e-6, atol=1e-6)
    assert r["reason"] > 0
    assert abs(r["its"] - rep.ksp.its) <= max(1, int(0.1 * rep.ksp.its))
    assert pc.info()["nE"] == rep.pc.e.shape[0]


def test_larger_case_roundtrip():
    """64k DOFs, 8 subdomains: solution of A x = A (1..N) is (1..N); eigen-counts equal the oracle's inertia counts."""
    mesh = go.gen_grid(3, 40, 1e-4)
    p = _problem(mesh, 8)
    pc = g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.2"]).setup(p)
    b = pc.make_rhs()
    r = pc.ksp_solve(b, ksp="cg", rtol=1e-10, atol=1e-50)
    assert r["reason"] > 0
    np.testing.assert_allclose(r["x"], np.arange(1, mesh.nb_node + 1.0), rtol=1e-5)
    rep = _oracle(mesh, p, 8, go.GenEOOptions(tau=0.2), ksp="cg", rtol=1e-10, atol=1e-50)
    assert [pc.sub_info(s)["nev"] for s in range(8)] == [s.z.shape[1] for s in rep.pc.sub]
    assert abs(r["its"] - rep.ksp.its) <= 1


def test_predecomposed_input_gives_the_same_preconditioner(lap3d):
    """The PETSc plug-in's view of the input (local Neumann matrices + local-to-global maps, geneo_problem_set_subdomain)
    yields the same PC as the driver's mesh path."""
    mesh = lap3d
    p = _problem(mesh, 4, dual=False, overlap=1)
    subs = [(p.sub_nodes(s)[0], p.sub_matrix(s, 0)) for s in range(4)]
    q = g.Problem().set_subdomains(mesh.nb_node, subs)
    x = np.random.default_rng(5).standard_normal(mesh.nb_node)
    y = [g.GeneoPC(["-geneo_lvl", "ASM,1", "-geneo_tau", "0.3", "-els2_eps_tol", "1e-10"]).setup(pr).apply(x) for pr in (p, q)]
    assert np.linalg.norm(y[0] - y[1]) <= 1e-8 * np.linalg.norm(y[0])


def test_thick_restart_reaches_the_same_eigenpairs():
    """A Krylov basis far too small for the wanted pairs (-els2_eps_ncv) forces several thick restarts (block
    Krylov-Schur); counts and eigenvalues must not change (oracle: dense eigh of the pencil, src/geneo.cpp:626-744)."""
    mesh, nparts = go.gen_grid(3, 16, 1e-4, 2.0, "lin"), 2
    p = _problem(mesh, nparts)
    # the gap of the pencil at tau is 1.6e-3 (subdomain 0): a Ritz vector next to it is accurate to ~ tol / gap, so the
    # 1e-7 asked of M^-1 x below needs a residual tolerance of 1e-10 (1e-9 leaves ~1e-7, i.e. pass or fail by rounding)
    base = ["-geneo_lvl", "ASM,1", "-geneo_tau", "0.45", "-els2_eps_tol", "1e-10"]
    pc_ref = g.GeneoPC(base).setup(p)
    pc_small = g.GeneoPC(base + ["-els2_eps_ncv", "80"]).setup(p)  # 36 + 2 guard pairs wanted from an 80-column basis
    rep = _oracle(mesh, p, nparts, go.GenEOOptions(lvl1="ASM", lvl2="1", tau=0.45), ksp="cg", rtol=1e-6)
    for s in range(nparts):
        a, bb = pc_ref.sub_info(s), pc_small.sub_info(s)
        assert a["nev"] == bb["nev"] == rep.pc.sub[s].z.shape[1] and a["nev"] >= 20, (a, bb)
        assert bb["eigDim"] <= 80 and bb["eigSteps"] > a["eigSteps"]  # the small basis really restarted
        ref = np.sort(np.array(rep.pc.sub[s].eigvals))
        np.testing.assert_allclose(np.sort(pc_small.sub_eigenvalues(s)), ref, rtol=1e-6, atol=1e-12)
        np.testing.assert_allclose(np.sort(pc_ref.sub_eigenvalues(s)), ref, rtol=1e-6, atol=1e-12)
    x = np.random.default_rng(1).standard_normal(mesh.nb_node)
    y, yo = pc_small.apply(x), rep.pc.apply(x)
    assert np.linalg.norm(y - yo) <= 1e-7 * np.linalg.norm(yo)


def test_level_profile_covers_the_whole_factor():
    """geneo_pc_level_profile: one timestamped PC-apply solve; the per-phase bytes add up to the factor read twice."""
    mesh = go.gen_grid(3, 14, 1e-4, 2.0, "lin")
    p = _problem(mesh, 4)
    pc = g.GeneoPC(["-geneo_lvl", "ASM,0"]).setup(p)
    us, by, it = pc.level_profile()
    assert len(us) == len(by) == len(it) and len(us) % 2 == 0 and (us >= 0).all() and it.sum() > 0
    st = pc.stats()
    assert by.sum() <= st["trisolve_bytes"] and by.sum() >= 0.8 * st["trisolve_bytes"]  # (the rest: row indices, vectors)


@pytest.mark.parametrize("lvl,ksp", [("ASM,1", "gmres"), ("SORAS,2", "gmres"), ("ASM,1", "cg")])
def test_graph_laplacian_matches_oracle(lvl, ksp):
    """BASELINE configs[3]: the irregular graph Laplacian of tst/graph (arguments of tst/graph/graphRun.sh:144) from the
    product's generator (bit-exact to the reference's own one: test_host.py), METIS partition, GenEO + GMRES / CG."""
    gen = g.Problem().generate("graph", "--size 400 --level 3 --noGround --inpEps 0.0001")
    ep, ei, em = gen.mesh()
    npe = np.diff(ep)
    mesh = go.Mesh(gen.sizes()["nb_node"], ep.astype(np.int64), ei.astype(np.int64),
                   np.concatenate([[0], np.cumsum(npe * npe)]).astype(np.int64), np.asarray(em, dtype=np.float64))
    nparts = 4
    p = _problem(mesh, nparts)
    l1, l2 = lvl.split(",")
    argv = ["-geneo_lvl", lvl, "-geneo_tau", "0.1"]
    if l2 == "2":
        argv += ["-geneo_optim", "0.02", "-els2_eps_tol", "1e-8"]
    pc = g.GeneoPC(argv).setup(p)
    rep = _oracle(mesh, p, nparts, go.GenEOOptions(lvl1=l1, lvl2=l2, tau=0.1, optim=0.02 if l2 == "2" else 0.0), ksp=ksp, rtol=1e-6, atol=1e-6)
    x = np.random.default_rng(5).standard_normal(mesh.nb_node)
    np.testing.assert_allclose(pc.mult(x), rep.a @ x, rtol=1e-12, atol=1e-12)
    assert pc.info()["nE"] == rep.pc.e.shape[0]
    for s in range(nparts):
        si = pc.sub_info(s)
        assert si["nev"] == rep.pc.sub[s].z.shape[1] and si["estim"] == rep.pc.sub[s].estim
        np.testing.assert_allclose(np.sort(pc.sub_eigenvalues(s)), np.sort(np.array(rep.pc.sub[s].eigvals)), rtol=1e-6, atol=1e-12)
    r = pc.ksp_solve(pc.make_rhs(), ksp=ksp, rtol=1e-6, atol=1e-6)
    assert r["reason"] > 0 and abs(r["its"] - rep.ksp.its) <= 1, (r["its"], rep.ksp.its)
    assert np.linalg.norm(r["x"] - rep.ksp.x) <= 1e-4 * np.linalg.norm(rep.ksp.x)


def test_block16_eigensolver_uses_the_16_rhs_solve(lap3d):
    """-els2_eps_block 16: the Lanczos block goes through k_solve_ring<16> (two DMMAs per factor fragment); counts and
    eigenvalues are those of the dense oracle, and the preconditioner is the one of the default block of 8."""
    mesh, nparts = lap3d, 4
    p = _problem(mesh, nparts)
    base = ["-geneo_lvl", "ASM,1", "-geneo_tau", "0.3", "-els2_eps_tol", "1e-10"]
    pc8 = g.GeneoPC(base + ["-els2_eps_block", "8"]).setup(p)
    pc16 = g.GeneoPC(base + ["-els2_eps_block", "16"]).setup(p)
    rep = _oracle(mesh, p, nparts, go.GenEOOptions(lvl1="ASM", lvl2="1", tau=0.3), ksp="cg", rtol=1e-6)
    for s in range(nparts):
        assert pc16.sub_info(s)["nev"] == rep.pc.sub[s].z.shape[1]
        np.testing.assert_allclose(np.sort(pc16.sub_eigenvalues(s)), np.sort(np.array(rep.pc.sub[s].eigvals)), rtol=1e-6, atol=1e-12)
    x = np.random.default_rng(2).standard_normal(mesh.nb_node)
    y8, y16, yo = pc8.apply(x), pc16.apply(x), rep.pc.apply(x)
    assert np.linalg.norm(y16 - yo) <= 1e-8 * np.linalg.norm(yo)
    assert np.linalg.norm(y16 - y8) <= 1e-8 * np.linalg.norm(y8)


def test_cli_reproduces_the_reference_logs(dummy_goldens, dummy_inputs):
    """The PETSc-free driver (geneo4petsc_b200/geneo4PETSc) run with the command lines of tst/dummy/dummy.sh against the
    reference's golden logs: local matrices, B, the converged X, and the INFO lines (only the solver names after L1 / L2
    differ: ldlt / blocklanczos instead of mumps / arpack)."""
    import os
    import re
    import subprocess
    from tests._cases import driver_command, parse_driver_log
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "geneo4petsc_b200", "geneo4PETSc")
    names = ["tridiag-pc=geneoASM1-metis=dual", "tridiag-pc=geneoASMH1-metis=dual-opt=overlap1", "tridiag-pc=geneoSORAS2-metis=dual",
             "tridiag-pc=geneoSORASE2-metis=dual-opt=offload", "identity-pc=geneoASM0-metis=dual", "identity-pc=geneoASME1-metis=dual",
             "identity-pc=geneoSORASH2-metis=dual-opt=overlap1", "tridiag-pc=geneoSORAS0-metis=dual"]

    def norm(line):
        line = re.sub(r"L1 \S+", "L1 *", line)
        return re.sub(r"L2 .*$", "L2 *", line)

    for name in names:
        g = dummy_goldens["goldens"][name]
        r = subprocess.run([exe] + driver_command(name, g, dummy_inputs), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (name, r.stdout[-400:], r.stderr[-400:])
        got = parse_driver_log(r.stdout)
        assert got["mats"] == g["mats"], name
        np.testing.assert_allclose(got["b"], g["b"], rtol=1e-6, err_msg=name)
        np.testing.assert_allclose(got["x"], g["x"], rtol=1e-5, atol=1e-9, err_msg=name)
        assert [norm(l) for l in got["info"]] == [norm(l) for l in g["info"]], (name, got["info"], g["info"])
