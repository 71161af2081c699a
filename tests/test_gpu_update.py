"""Same-pattern value update (geneo_pc_update, PCSetUp with SAME_NONZERO_PATTERN): after update(p2) the preconditioner is
the one a fresh setup on p2 builds -- the operator bit for bit, the same coarse space, the same applies and iterations --
and an update that does not match the setup's partition, node sets or patterns is rejected with the previous
preconditioner left intact.  The second problem of every pair is decomposed with the first one's partition, and the test
asserts first that the two decompositions have the same node sets and matrix patterns."""
import numpy as np
import pytest
import scipy.sparse as sp

import geneo4petsc_b200 as g
from oracle import geneo_oracle as go

gpu = pytest.mark.gpu
NPARTS = 4


def _problem(mesh, nparts=NPARTS, part=None):
    p = g.Problem().set_mesh(mesh.nb_node, mesh.elem_ptr, mesh.elem_idx, mesh.mat_val)
    if part is None:
        return p.decompose(nparts, True, 0)
    return p.decompose(nparts, True, 0, elem_part=part[0], node_part=part[1])


def _pair(heat=False):
    """Two problems on one mesh with one partition: only the values differ (kappa 2 -> 50, or heat dt 0.1 -> 0.05)."""
    if heat:
        m1 = go.gen_grid(3, 12, 1e-4, 100.0, "minmax", heat=True, dt=0.1)
        m2 = go.gen_grid(3, 12, 1e-4, 100.0, "minmax", heat=True, dt=0.05)
    else:
        m1, m2 = go.gen_grid(3, 12, 1e-4, 2.0, "lin"), go.gen_grid(3, 12, 1e-4, 50.0, "lin")
    p1 = _problem(m1)
    p2 = _problem(m2, part=p1.partition())
    _assert_same_patterns(p1, p2)
    return m1, m2, p1, p2


def _assert_same_patterns(p1, p2):
    for s in range(NPARTS):
        assert np.array_equal(p1.sub_nodes(s)[0], p2.sub_nodes(s)[0])
        for which in (0, 1):
            a, b = p1.sub_matrix(s, which), p2.sub_matrix(s, which)
            assert np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices), (s, which)
            assert not np.array_equal(a.data, b.data), (s, which)


def _argv(lvl, extra=()):
    tau = "0.1" if lvl.endswith("2") else "0.3"
    return ["-geneo_lvl", lvl, "-geneo_tau", tau, "-els2_eps_tol", "1e-10"] + list(extra)


def _ksp(lvl):
    return "cg" if lvl.startswith("ASM") else "gmres"


def _assert_same_pc(pc, fresh, lvl, nb_node):
    x = np.random.default_rng(11).standard_normal(nb_node)
    assert np.array_equal(pc.mult(x), fresh.mult(x))  # the operator bit for bit
    assert pc.info()["nE"] == fresh.info()["nE"]
    for s in range(NPARTS):
        a, b = pc.sub_info(s), fresh.sub_info(s)
        for k in ("estim", "nev", "neg", "perturbed"):
            assert a[k] == b[k], (s, k, a, b)
        np.testing.assert_allclose(np.sort(pc.sub_eigenvalues(s)), np.sort(fresh.sub_eigenvalues(s)), rtol=1e-9, atol=1e-14)
    y, yf = pc.apply(x), fresh.apply(x)
    assert np.linalg.norm(y - yf) <= 1e-9 * np.linalg.norm(yf)
    b = fresh.make_rhs()
    r, rf = pc.ksp_solve(b, ksp=_ksp(lvl), rtol=1e-6), fresh.ksp_solve(b, ksp=_ksp(lvl), rtol=1e-6)
    assert r["reason"] > 0 and rf["reason"] > 0 and abs(r["its"] - rf["its"]) <= 1, (r["its"], rf["its"])


@gpu
@pytest.mark.parametrize("lvl,extra,heat", [
    ("ASM,1", [], False),
    ("RAS,1", [], False),
    ("ORAS,1", ["-geneo_optim", "0.5"], False),
    ("SORAS,2", ["-geneo_optim", "0.5"], False),
    ("ASM,E1", [], False),
    ("ASM,1", [], True),
])
def test_update_equals_fresh_setup(lvl, extra, heat):
    m1, m2, p1, p2 = _pair(heat)
    pc = g.GeneoPC(_argv(lvl, extra)).setup(p1)
    pc.update(p2)
    fresh = g.GeneoPC(_argv(lvl, extra)).setup(p2)
    _assert_same_pc(pc, fresh, lvl, m2.nb_node)


@gpu
def test_updated_values_match_the_oracle():
    """The updated preconditioner against the oracle on the second problem: the values are right on their own, not only
    the ones the fresh-setup path would produce."""
    m1, m2, p1, p2 = _pair()
    pc = g.GeneoPC(_argv("ASM,1")).setup(p1).update(p2)
    rep = go.run_case(m2, NPARTS, go.GenEOOptions(lvl1="ASM", lvl2="1", tau=0.3), ksp="cg", rtol=1e-6, atol=1e-6, part=p1.partition())
    x = np.random.default_rng(2).standard_normal(m2.nb_node)
    np.testing.assert_allclose(pc.mult(x), rep.a @ x, rtol=1e-12, atol=1e-12)
    assert pc.info()["nE"] == rep.pc.e.shape[0]
    for s in range(NPARTS):
        si = pc.sub_info(s)
        assert si["perturbed"] == 0 and si["nev"] == rep.pc.sub[s].z.shape[1] and si["estim"] == rep.pc.sub[s].estim, (s, si)
        np.testing.assert_allclose(np.sort(pc.sub_eigenvalues(s)), np.sort(np.array(rep.pc.sub[s].eigvals)), rtol=1e-6, atol=1e-12)
    r = pc.ksp_solve(pc.make_rhs(), ksp="cg", rtol=1e-6, atol=1e-6)
    assert r["reason"] > 0 and rep.ksp.converged and abs(r["its"] - rep.ksp.its) <= 1, (r["its"], rep.ksp.its)


@gpu
def test_update_round_trip():
    m1, m2, p1, p2 = _pair()
    pc = g.GeneoPC(_argv("ASM,1")).setup(p1)
    x = np.random.default_rng(5).standard_normal(m1.nb_node)
    y0, a0 = pc.apply(x), pc.mult(x)
    pc.update(p2)
    assert not np.array_equal(pc.mult(x), a0)
    pc.update(p1)
    assert np.array_equal(pc.mult(x), a0)
    assert np.linalg.norm(pc.apply(x) - y0) <= 1e-9 * np.linalg.norm(y0)


@gpu
@pytest.mark.parametrize("pipeline", ["0", "1"])
def test_update_on_both_numeric_paths(monkeypatch, pipeline):
    monkeypatch.setenv("GENEO_PIPELINE", pipeline)
    m1, m2, p1, p2 = _pair()
    pc = g.GeneoPC(_argv("ASM,1")).setup(p1).update(p2)
    _assert_same_pc(pc, g.GeneoPC(_argv("ASM,1")).setup(p2), "ASM,1", m2.nb_node)


def _subs(p):
    return [[p.sub_nodes(s)[0], p.sub_matrix(s, 0), p.sub_matrix(s, 1)] for s in range(NPARTS)]


def _move_entry(a, dir_pattern):
    """A copy of CSR `a` with one off-diagonal entry moved to a column of its row outside `dir_pattern` (same nnz)."""
    a = a.tocsr().copy()
    for r in range(a.shape[0]):
        cols = a.indices[a.indptr[r]:a.indptr[r + 1]]
        taken = set(dir_pattern.indices[dir_pattern.indptr[r]:dir_pattern.indptr[r + 1]])
        free = [c for c in range(a.shape[1]) if c not in taken]
        off = [t for t in range(a.indptr[r], a.indptr[r + 1]) if a.indices[t] != r]
        if free and off:
            a.indices[off[0]] = free[0]
            a.has_sorted_indices = False
            a.sort_indices()
            return a
    raise AssertionError("no entry to move")


def _move_to_another_row(a):
    """A copy of CSR `a` with the last entry of row 0 moved to the end of row 1 (same nnz, row lengths differ)."""
    a = a.tocsr()
    ptr, idx, val = a.indptr.copy(), a.indices.copy(), a.data.copy()
    rows = [list(zip(idx[ptr[r]:ptr[r + 1]], val[ptr[r]:ptr[r + 1]])) for r in range(a.shape[0])]
    _, v = rows[0].pop()
    free = next(k for k in range(a.shape[1]) if k not in {e[0] for e in rows[1]})
    rows[1] = sorted(rows[1] + [(free, v)])
    ptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])])
    return sp.csr_matrix((np.array([e[1] for r in rows for e in r]), np.array([e[0] for r in rows for e in r], dtype=np.int32), ptr),
                         shape=a.shape)


def _with_duplicate(a):
    """CSR arrays of `a` whose first row with two entries repeats its first column (same nnz)."""
    a = a.tocsr()
    ptr, idx, val = a.indptr.copy(), a.indices.copy(), a.data.copy()
    r = next(r for r in range(a.shape[0]) if ptr[r + 1] - ptr[r] >= 2)
    idx[ptr[r] + 1] = idx[ptr[r]]
    return sp.csr_matrix((val, idx, ptr), shape=a.shape)


@gpu
def test_rejected_updates_leave_the_preconditioner_intact():
    m1, m2, p1, p2 = _pair()
    pc = g.GeneoPC(_argv("ASM,1")).setup(p1)
    x = np.random.default_rng(9).standard_normal(m1.nb_node)
    a0, y0 = pc.mult(x), pc.apply(x)

    def rejected(make, match):
        with pytest.raises(g.GeneoError, match=match):
            pc.update(make())
        assert np.array_equal(pc.mult(x), a0)
        assert np.linalg.norm(pc.apply(x) - y0) <= 1e-12 * np.linalg.norm(y0)

    rejected(lambda: g.Problem(), "without a decomposed problem")
    rejected(lambda: _problem(m2, NPARTS - 1), "subdomains")
    ep, npart = p1.partition()
    rejected(lambda: _problem(m2, part=((ep + 1) % NPARTS, (npart + 1) % NPARTS)), "node")

    def extra_dir_entry():
        subs = _subs(p2)
        d = subs[0][2].tolil()
        r, c = next((r, c) for r in range(d.shape[0]) for c in (0, d.shape[0] - 1) if d[r, c] == 0)
        d[r, c] = 1.0
        subs[0][2] = d.tocsr()
        return g.Problem().set_subdomains(m2.nb_node, subs)
    rejected(extra_dir_entry, "A_dir has")

    def moved_dir_entry():
        subs = _subs(p2)
        subs[1][2] = _move_entry(subs[1][2], subs[1][2])
        return g.Problem().set_subdomains(m2.nb_node, subs)
    rejected(moved_dir_entry, "A_dir entries outside")

    def neu_outside_dir():
        subs = _subs(p2)
        subs[2][1] = _move_entry(subs[2][1], subs[2][2])
        return g.Problem().set_subdomains(m2.nb_node, subs)
    rejected(neu_outside_dir, "A_neu entries outside the A_dir pattern")

    def moved_to_another_row():
        subs = _subs(p2)
        subs[3][2] = _move_to_another_row(subs[3][2])
        return g.Problem().set_subdomains(m2.nb_node, subs)
    rejected(moved_to_another_row, "A_dir rows whose length differs")

    # A duplicate column never reaches the update: building the pre-decomposed problem refuses it.  The PC is untouched.
    with pytest.raises(g.GeneoError, match="duplicate column"):
        subs = _subs(p2)
        subs[0][1] = _with_duplicate(subs[0][1])
        g.Problem().set_subdomains(m2.nb_node, subs)
    assert np.array_equal(pc.mult(x), a0)

    # the same matrices through the pre-decomposed input: accepted, and the operator is the first problem's again
    pc.update(g.Problem().set_subdomains(m2.nb_node, _subs(p1)))
    assert np.array_equal(pc.mult(x), a0)
    assert np.linalg.norm(pc.apply(x) - y0) <= 1e-9 * np.linalg.norm(y0)


@gpu
def test_failed_numeric_setup_leaves_no_context(tmp_path, monkeypatch):
    """The values pass every check but the new A_dir of subdomain 1 is negative definite: -geneo_chk stops the numeric
    setup, and the half-updated preconditioner refuses to apply."""
    monkeypatch.chdir(tmp_path)  # (-geneo_chk writes its logs to the working directory)
    m1, m2, p1, p2 = _pair()
    pc = g.GeneoPC(["-geneo_lvl", "ASM,0", "-geneo_chk", "log"]).setup(p1)
    bad = _subs(p1)
    bad[1][1], bad[1][2] = -bad[1][1], -bad[1][2]
    with pytest.raises(g.GeneoError, match="not SPD"):
        pc.update(g.Problem().set_subdomains(m1.nb_node, bad))
    with pytest.raises(g.GeneoError, match="without context"):
        pc.apply(np.ones(m1.nb_node))


def test_update_before_setup_has_no_context():
    """Checked before anything touches the device: the same message with or without a GPU."""
    with pytest.raises(g.GeneoError, match="without context"):
        g.GeneoPC().update(g.Problem())
