"""CPU-side tests of the product's HOST logic (no device needed): C-ABI exports, generators, decomposition parity with
the oracle, symbolic analysis (validated by a numpy emulation of the device numeric phase), small dense eigen-solver."""
import os

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.linalg as sla

import geneo4petsc_b200 as g
from geneo4petsc_b200._lib import header_functions
from oracle import geneo_oracle as go
from tests import _emul


def test_library_exports_every_declared_symbol():
    names = header_functions()
    assert len(names) >= 40
    for f in names:
        assert hasattr(g.lib, f), "missing export " + f


def test_no_cpu_fallback_without_device():
    if g.device_count() > 0:
        pytest.skip("a device is present")
    p = g.Problem().generate("laplacian", "--dim 2 --size 6").decompose(2)
    with pytest.raises(g.GeneoError, match="no CUDA device"):
        g.GeneoPC().setup(p)
    with pytest.raises(g.GeneoError):
        g.microbench(1, 1024)


def test_level_probe_rejects_a_block_width_without_a_solve_kernel():
    """microbench kind 100 * nlev + nr: the solve kernels exist for nr = 1, 8 and 16 only.  The kind is checked before the
    device is touched, so the same error comes with or without a GPU."""
    with pytest.raises(g.GeneoError, match="nr must be 1, 8 or 16"):
        g.microbench(102, 128, 1)


@pytest.mark.parametrize("kind,args,kw", [
    ("laplacian", "--dim 3 --size 9 --kappa 2. lin --inpEps 0.0001", dict(dim=3, size=9, inp_eps=1e-4, kappa_max=2.0, interp="lin")),
    ("laplacian", "--dim 2 --size 11 --weakScaling 3 --kappa 5. quad", dict(dim=2, size=11, weak=3, kappa_max=5.0, interp="quad")),
    ("laplacian", "--dim 1 --size 7", dict(dim=1, size=7)),
    ("heat", "--dim 3 --size 7 --kappa 100. minmax --lbd 1. --dt 0.1", dict(dim=3, size=7, kappa_max=100.0, interp="minmax", heat=True)),
])
def test_structured_generator_matches_reference_element_sequence(kind, args, kw):
    p = g.Problem().generate(kind, args)
    ep, ei, em = p.mesh()
    m = go.gen_grid(**kw)  # itself checked bit-exact against the reference's own generator (test_oracle_props.py)
    assert p.sizes()["nb_node"] == m.nb_node and p.sizes()["nb_elem"] == m.nb_elem
    assert np.array_equal(ep, m.elem_ptr) and np.array_equal(ei, m.elem_idx) and np.array_equal(em, m.mat_val)


def test_bad_options_are_rejected():
    for bad in (["-geneo_lvl", "FOO,1"], ["-geneo_lvl", "ASM,9"], ["-geneo_tau", "1.5"], ["-geneo_tau", "abc"],
                ["-geneo_lvl", "SORAS,2", "-geneo_gamma", "0.5"], ["-geneo_lvl"], ["-geneo_ordering", "2"],
                ["-geneo_ordering", "-1"]):
        with pytest.raises(g.GeneoError):
            g.GeneoPC(bad)
    with pytest.raises(g.GeneoError, match="ordering must be 0"):
        g.Symbolic(sp.identity(40, format="csr"), ordering=2)
    assert g.GeneoPC(["-geneo_lvl", "SORAS,H2"]).name == "geneo2HSORAS"
    assert g.GeneoPC().name == "geneo1ASM"
    assert g.GeneoPC(["-geneo_lvl", "RAS,E1"]).name == "geneo1ERAS"
    assert g.GeneoPC(["-geneo_lvl", "ASM,0"]).name == "geneo0ASM"


@pytest.mark.parametrize("dual,overlap,nparts", [(True, 0, 4), (False, 0, 3), (True, 1, 4), (False, 2, 2), (True, 0, 1)])
def test_decomposition_matches_oracle(dual, overlap, nparts):
    mesh = go.gen_grid(3, 8, 1e-4, 3.0, "lin")
    p = g.Problem().set_mesh(mesh.nb_node, mesh.elem_ptr, mesh.elem_idx, mesh.mat_val).decompose(nparts, dual, overlap)
    ep, npart = p.partition()
    oe, on = go.metis_partition(mesh, nparts, dual)
    assert np.array_equal(ep, oe) and np.array_equal(npart, on)  # same METIS build, same options => identical partition
    dec = go.decompose(mesh, nparts, oe, on, dual, overlap)
    nnz = 0
    for s in range(nparts):
        nodes, mult = p.sub_nodes(s)
        assert np.array_equal(nodes, dec.nodes[s])
        assert np.array_equal(mult, dec.node_mult[dec.nodes[s]])
        for q in range(nparts):
            assert np.array_equal(p.sub_intersect(s, q), dec.intersect[s][q])
        a_neu = go.local_neumann(mesh, dec, s)
        mine = p.sub_matrix(s, 0)
        assert abs(mine - a_neu).max() < 1e-13
        nnz += mine.nnz
    a = go.assemble_global(mesh.nb_node, dec, [go.local_neumann(mesh, dec, s) for s in range(nparts)])
    for s in range(nparts):
        nodes = dec.nodes[s]
        a_dir = a[nodes][:, nodes]
        assert abs(p.sub_matrix(s, 1) - a_dir).max() < 1e-12
    assert p.sizes()["nnz"] == nnz


def test_explicit_partition_is_honoured():
    mesh = go.gen_grid(2, 8)
    epart = (np.arange(mesh.nb_elem) % 3).astype(np.int32)
    p = g.Problem().set_mesh(mesh.nb_node, mesh.elem_ptr, mesh.elem_idx, mesh.mat_val).decompose(3, True, 0, elem_part=epart)
    assert np.array_equal(p.partition()[0], epart)
    dec = go.decompose(mesh, 3, epart, np.zeros(mesh.nb_node, dtype=int), True, 0)
    for s in range(3):
        assert np.array_equal(p.sub_nodes(s)[0], dec.nodes[s])


def _grid_matrix(n, dim):
    mesh = go.gen_grid(dim, n, 1e-2)
    part = go.metis_partition(mesh, 1, True)
    dec = go.decompose(mesh, 1, part[0], part[1], True, 0)
    return go.local_neumann(mesh, dec, 0)


@pytest.mark.parametrize("n,dim,nb,ordering,amalg", [(6, 3, 8, 1, True), (9, 3, 16, 1, True), (12, 2, 128, 1, True),
                                                     (7, 3, 8, 0, False), (10, 3, 32, 1, False), (30, 1, 8, 1, True)])
def test_symbolic_structures_drive_a_correct_factorization(n, dim, nb, ordering, amalg):
    a = _grid_matrix(n, dim).tocsr()
    a.sort_indices()
    sym = g.Symbolic(a, nb=nb, ordering=ordering, amalgamate=amalg)
    fr = sym.fronts
    assert sorted(sym.perm.tolist()) == list(range(a.shape[0]))
    assert fr[:, _emul.F_K].sum() == a.shape[0] and fr[:, _emul.F_K].max() <= nb
    par = fr[:, _emul.F_PARENT]
    has_par = par >= 0
    assert np.all(fr[has_par, _emul.F_LEVEL] + 1 == fr[par[has_par], _emul.F_LEVEL])  # children exactly one level below
    L, neg = _emul.factorize(sym, a.data)
    assert neg == 0
    rng = np.random.default_rng(0)
    b = rng.standard_normal(a.shape[0])
    x = _emul.solve(sym, L, b)
    assert np.linalg.norm(a @ x - b) <= 1e-9 * np.linalg.norm(b)
    # inertia of an indefinite shift (Sylvester): compare with the exact eigenvalue count
    # (a few eigenvalues below the shift, like A_neu - tau B in GenEO: the block LDL^T does not pivot across pivot blocks,
    #  so a shift deep inside the spectrum -- hundreds of sign changes -- is outside its contract)
    w = sla.eigvalsh(a.toarray())
    nbelow = min(5, len(w) // 4)
    shift = 0.5 * (w[nbelow - 1] + w[nbelow])
    s = (a - shift * sp.identity(a.shape[0])).tocsr()
    s.sort_indices()
    assert np.array_equal(s.indices, a.indices)
    _, neg = _emul.factorize(sym, s.data)
    assert neg == int(np.sum(w < shift))


def test_symbolic_dense_matrix_is_one_chain():
    n = 70
    rng = np.random.default_rng(1)
    m = rng.standard_normal((n, n))
    e = m @ m.T + n * np.eye(n)
    a = sp.csr_matrix(e)
    sym = g.Symbolic(a, nb=16, ordering=0, amalgamate=False)
    assert sym.info["nsuper"] == 1 and sym.info["nfronts"] == 5 and sym.info["nlevels"] == 5
    L, neg = _emul.factorize(sym, a.data)
    x = _emul.solve(sym, L, np.ones(n))
    np.testing.assert_allclose(e @ x, np.ones(n), rtol=1e-10)


def test_host_sym_eig_matches_lapack():
    rng = np.random.default_rng(3)
    for n in (1, 2, 5, 40, 130):
        a = rng.standard_normal((n, n))
        a = a + a.T
        w, v = g.host_sym_eig(a)
        np.testing.assert_allclose(w, np.linalg.eigvalsh(a), atol=1e-11 * max(1, n))
        np.testing.assert_allclose(a @ v, v * w, atol=1e-10 * max(1, n))


def test_predecomposed_input_matches_mesh_decomposition():
    """initGenEOPC's view (local Neumann matrices + local-to-global maps) gives back the same multiplicities,
    intersections and Dirichlet matrices as the driver's own decomposition."""
    import geneo4petsc_b200 as g
    for dual, overlap in ((True, 0), (False, 1)):
        p = g.Problem().generate("laplacian", "--dim 3 --size 9 --inpEps 0.0001 --kappa 2. lin").decompose(4, dual, overlap)
        subs = [(p.sub_nodes(s)[0], p.sub_matrix(s, 0)) for s in range(4)]
        q = g.Problem().set_subdomains(p.sizes()["nb_node"], subs)
        assert q.sizes()["nnz"] == p.sizes()["nnz"]
        for s in range(4):
            np.testing.assert_array_equal(q.sub_nodes(s)[1], p.sub_nodes(s)[1])
            for t in range(4):
                np.testing.assert_array_equal(q.sub_intersect(s, t), p.sub_intersect(s, t))
            d = (q.sub_matrix(s, 1) - p.sub_matrix(s, 1)).tocoo()
            assert d.nnz == 0 or np.abs(d.data).max() <= 1e-12 * np.abs(p.sub_matrix(s, 1).data).max()


def test_nested_dissection_is_deterministic_across_threads():
    """The library's ND calls use a thread-local rand() (glibc's is one locked, shared stream): orderings computed
    concurrently on different threads must equal the one computed alone (symbolic.cpp)."""
    import threading
    import scipy.sparse as sp
    from geneo4petsc_b200.api import Symbolic
    s = 14
    eye, t = sp.identity(s, format="csr"), sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(s, s), format="csr")
    a = (sp.kron(sp.kron(t, eye), eye) + sp.kron(sp.kron(eye, t), eye) + sp.kron(sp.kron(eye, eye), t)).tocsr()
    ref = Symbolic(a)
    out = [None] * 4

    def work(i):
        out[i] = Symbolic(a)

    ths = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    [th.start() for th in ths]
    [th.join() for th in ths]
    for o in out:
        assert np.array_equal(o.perm, ref.perm) and o.info["lSize"] == ref.info["lSize"]


def test_chain_panels_share_the_update_matrix_of_their_child():
    """Front::inplace: panel p+1 of a supernode works on the trailing block of panel p's update matrix (chain arena)."""
    import scipy.sparse as sp
    from geneo4petsc_b200.api import Symbolic
    s = 10
    eye, t = sp.identity(s, format="csr"), sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(s, s), format="csr")
    a = (sp.kron(sp.kron(t, eye), eye) + sp.kron(sp.kron(eye, t), eye) + sp.kron(sp.kron(eye, eye), t)).tocsr()
    sym = Symbolic(a, nb=8)  # narrow panels: long chains
    fr = sym.fronts
    inpl = np.nonzero(fr[:, 15] == 1)[0]
    assert len(inpl) > 10 and sym.info["cArena"] > 0
    for f in inpl:
        c = f - 1
        assert fr[c, 5] == 1 and fr[c, 3] == f and fr[f, 6] == 1          # chain link, only child
        assert fr[f, 14] == fr[c, 14] == 2 and fr[f, 13] == fr[c, 13]      # same arena, same leading dimension
        assert fr[f, 9] == fr[c, 9] + fr[f, 1] * (fr[c, 13] + 1)           # trailing block
        m = fr[f, 2] - fr[f, 1]
        assert fr[f, 9] + (m - 1) * fr[f, 13] + m <= sym.info["cArena"]


def test_cli_dumps_the_local_matrices_of_the_reference_goldens(dummy_goldens, dummy_inputs):
    """geneo4PETSc (this repo's PETSc-free driver, csrc/cli.cpp) with the command lines of tst/dummy/dummy.sh: the
    `--verbose 2` dump of the MATIS operator (partition + overlap + 1/mult weighting) is the reference's, in PETSc's own
    ASCII layout.  Runs without a GPU: the dump precedes the (device) setup, which then fails loudly on a CPU-only box."""
    import os
    import subprocess
    from tests._cases import driver_command, golden_config, parse_driver_log
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(ROOT, "geneo4petsc_b200", "geneo4PETSc")
    assert os.path.exists(exe), "CLI not built (python __graft_entry__.py)"
    checked = 0
    for name, g in sorted(dummy_goldens["goldens"].items()):
        cfg = golden_config(g)
        if cfg is None or not cfg["dual"]:  # nodal goldens: this METIS build mirrors the two labels (SURVEY 8c), tested elsewhere
            continue
        r = subprocess.run([exe] + driver_command(name, g, dummy_inputs), capture_output=True, text=True, timeout=120)
        got = parse_driver_log(r.stdout)
        assert got["mats"] == g["mats"], name
        assert r.stdout.startswith("The matrix A is:\nMat Object: 2 MPI processes\n  type: is\n  Mat Object: 1 MPI processes\n    type: seqaij\nrow 0:")
        if r.returncode != 0:  # CPU-only box
            assert "no CUDA device" in r.stderr and "INFO:" not in r.stdout
        checked += 1
    assert checked == 40


def test_cli_rejects_bad_command_lines():
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "geneo4petsc_b200", "geneo4PETSc")
    for args, msg in ((["--inpEps"], "invalid command line"), ([], "no input"), (["--inpFileA", "a", "--inpLibA", "b", "c"], "several input"),
                      (["--inpFileA", "x.inp", "-pc_type", "bjacobi"], "PETSc built-in"), (["--bogus"], "invalid command line")):
        r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=60)
        assert r.returncode == 1 and msg in r.stderr, (args, r.stderr)
    r = subprocess.run([exe, "--help"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and "usage: geneo4PETSc" in r.stderr


def test_chain_pairs_cover_every_update_exactly_once():
    """Front::pair (rank-256 trailing updates): pairs are (first, second) = consecutive panels of an in-place chain; the
    first only updates the strip its successor assembles, the second applies both panels to the trailing block.  The
    numpy emulation of the device phase (tests/_emul.py) factorizes with exactly these roles and must still solve."""
    from geneo4petsc_b200.api import Symbolic
    s = 9
    eye, t = sp.identity(s, format="csr"), sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(s, s), format="csr")
    a = (sp.kron(sp.kron(t, eye), eye) + sp.kron(sp.kron(eye, t), eye) + sp.kron(sp.kron(eye, eye), t) + 0.1 * sp.identity(s ** 3)).tocsr()
    sym = Symbolic(a, nb=6)  # panels of 6 columns (not a multiple of the 64-wide device tile): long chains, ragged strips
    fr = sym.fronts
    first, second = np.nonzero(fr[:, 16] == 1)[0], np.nonzero(fr[:, 16] == 2)[0]
    assert len(first) > 5 and np.array_equal(first + 1, second)
    for f in first:
        assert fr[f, 5] == 1 and fr[f, 3] == f + 1 and fr[f + 1, 15] == 1 and fr[f + 1, 4] == fr[f, 4] + 1
    L, neg = _emul.factorize(sym, a.data)
    assert neg == 0
    b = np.random.default_rng(4).standard_normal(a.shape[0])
    x = _emul.solve(sym, L, b)
    assert np.linalg.norm(a @ x - b) <= 1e-10 * np.linalg.norm(b)


def test_cli_loads_getinput_plugins_like_the_reference(tmp_path):
    """--inpLibA L A: the driver dlopens any library exporting the reference's getInput() (src/geneo4PETSc.cpp:75-96).  Here L
    is tests/plugins/gen_web.cpp, an irregular graph Laplacian; the local matrices the driver dumps must be those of the
    oracle's decomposition of the mesh the same library returns."""
    import os
    import subprocess
    from tests._cases import parse_driver_log
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib = str(tmp_path / "libgenweb.so")
    cxx = "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"  # shared libstdc++: std::vector crosses dlopen (oracle/Makefile)
    subprocess.run([cxx, "-O2", "-std=c++11", "-fPIC", "-shared", "-o", lib, os.path.join(root, "tests", "plugins", "gen_web.cpp")],
                   check=True)
    args = "--size 300 --inpEps 0.0001"
    r = subprocess.run([os.path.join(root, "geneo4petsc_b200", "geneo4PETSc"), "--inpLibA", lib, args.replace(" ", "#"), "--nbPart", "3",
                        "--verbose", "2", "-pc_type", "geneo"], capture_output=True, text=True, timeout=120)
    got = parse_driver_log(r.stdout)
    mesh = go.plugin_input(lib, args)
    p = g.Problem().set_mesh(mesh.nb_node, mesh.elem_ptr, mesh.elem_idx, mesh.mat_val).decompose(3, True, 0)
    ep, npart = p.partition()
    dec = go.decompose(mesh, 3, ep, npart, True, 0)
    assert len(got["mats"]) == 3
    for s in range(3):
        a = go.local_neumann(mesh, dec, s).toarray()
        dense = np.zeros(a.shape)
        for rr, ent in got["mats"][s]:
            for c, v in ent:
                dense[rr, c] = v
        np.testing.assert_allclose(dense, a, rtol=1e-5, atol=1e-12)  # the dump prints 6 significant digits


@pytest.mark.parametrize("args", ["--size 400 --level 3 --noGround --inpEps 0.0001", "--size 16 --level 2 --inpEps 0.001",
                                  "--size 9 --level 0 --noGround", "--size 25 --level 1 --weakScaling 4"])
def test_graph_generator_matches_the_reference_plugin(args):
    """The product's closed-form graph generator (mesh.cpp generate_graph, BASELINE configs[3]) against the reference's own
    tst/graph/graph.cpp compiled into oracle/_ref: same node count, element sequence and element matrices, bit for bit."""
    try:
        ref = go.ref_generator("graph", args)
    except FileNotFoundError:
        pytest.skip("oracle/_ref/libgengraph.so not built (needs /root/reference at build time)")
    p = g.Problem().generate("graph", args)
    ep, ei, em = p.mesh()
    assert p.sizes()["nb_node"] == ref.nb_node
    assert np.array_equal(ep, ref.elem_ptr) and np.array_equal(ei, ref.elem_idx) and np.array_equal(em, ref.mat_val)


def _box_matrix(d):
    def T(s):
        return sp.diags([-1., 2.2, -1.], [-1, 0, 1], shape=(s, s), format="csr")

    def I(s):
        return sp.identity(s, format="csr")
    a, b, c = d
    m = (sp.kron(sp.kron(I(c), I(b)), T(a)) + sp.kron(sp.kron(I(c), T(b)), I(a)) + sp.kron(sp.kron(T(c), I(b)), I(a))).tocsr()
    m.sort_indices()
    return m


def test_box_subdomains_inherit_the_reference_ordering():
    """One nested dissection of the bounding box serves every (nearly) full box inside it: the induced permutation of a
    smaller box is a valid ordering (the numpy emulation of the device phase factorizes and solves with it) and its fill
    stays close to the box's own METIS ordering."""
    from geneo4petsc_b200.api import box_ordering
    ext = np.array([13, 12, 11])
    rank = box_ordering(ext, threads=2)
    assert sorted(rank.tolist()) == list(range(int(ext.prod())))
    for d in ((13, 12, 11), (12, 12, 11), (13, 11, 10)):
        a = _box_matrix(d)
        x = np.arange(d[0] * d[1] * d[2])
        c0, c1, c2 = x % d[0], (x // d[0]) % d[1], x // (d[0] * d[1])
        perm = np.argsort(rank[c0 + ext[0] * (c1 + ext[1] * c2)], kind="stable").astype(np.int32)
        sym = g.Symbolic(a, nb=16, perm=perm)
        own = g.Symbolic(a, nb=16)
        assert np.array_equal(sym.perm, sym.perm) and sorted(sym.perm.tolist()) == list(range(a.shape[0]))
        assert sym.info["lSize"] <= 1.35 * own.info["lSize"]
        L, neg = _emul.factorize(sym, a.data)
        assert neg == 0
        b = np.random.default_rng(1).standard_normal(a.shape[0])
        assert np.linalg.norm(a @ _emul.solve(sym, L, b) - b) <= 1e-9 * np.linalg.norm(b)


def test_host_preparation_fast_and_general_paths_agree():
    """The cold setup permutes the values of a subdomain and builds the scatter map of its factor in ONE pass when the rows
    are sorted and the pattern symmetric (transposed positions, a second thread for the ordering-independent part), and
    falls back to sorting rows + binary searches otherwise: same permuted matrix, same scattered factor, and the same
    entries of an UNSYMMETRIC-valued input are read (row perm[i], column perm[j] for i >= j)."""
    from geneo4petsc_b200.api import host_prepare_probe
    a = _box_matrix((9, 8, 7)).tocsr()
    a.sort_indices()
    rng = np.random.default_rng(5)
    a.data = a.data * (1.0 + 0.1 * rng.standard_normal(a.nnz))  # symmetric pattern, unsymmetric values
    perm = g.Symbolic(a, nb=16).perm.copy()
    sym = g.Symbolic(a, nb=16, perm=perm)
    lsize = sym.info["lSize"]
    L0 = np.zeros(lsize)
    L0[sym.asm_dst] = a.data[sym.asm_src]
    assert len(np.unique(sym.asm_dst)) == len(sym.asm_dst) == (a.nnz + a.shape[0]) // 2
    _, d0, s0 = host_prepare_probe(a, perm, nb=16, helper=False, scatter_len=lsize)
    _, d1, s1 = host_prepare_probe(a, perm, nb=16, helper=True, scatter_len=lsize)
    _, d2, s2 = host_prepare_probe(a, perm, nb=16, helper=2, scatter_len=lsize)  # general path forced
    # the same matrix with the columns of every row in random order (analysis entry point only: subdomain matrices are
    # validated to have sorted rows)
    b = a.copy()
    for r in range(b.shape[0]):
        lo, hi = b.indptr[r], b.indptr[r + 1]
        o = rng.permutation(hi - lo)
        b.indices[lo:hi] = b.indices[lo:hi][o]
        b.data[lo:hi] = b.data[lo:hi][o]
    b.has_sorted_indices = False
    assert d0 == d1 == d2
    assert np.array_equal(s0, L0) and np.array_equal(s1, L0) and np.array_equal(s2, L0)
    symu = g.Symbolic(b, nb=16, perm=perm)  # analysis entry point on unsorted rows: binary-search scatter map
    Lu = np.zeros(lsize)
    Lu[symu.asm_dst] = b.data[symu.asm_src]
    assert np.array_equal(Lu, L0)
    # METIS inside the probe (no inherited ordering)
    _, d3 = host_prepare_probe(a, None, nb=16, helper=True)
    _, d4 = host_prepare_probe(a, None, nb=16, helper=False)
    assert d3 == d4


def test_reference_plot_script_parses_the_cli_log():
    """tst/plot.py (the reference's post-processing, :56-116) must read the logs of the PETSc-free driver: its own `job` parser
    is imported from /root/reference (matplotlib stubbed out) and fed a log of geneo4petsc_b200/geneo4PETSc captured on the B200
    box (tests/golden/cli_tridiag_geneo1ASM.log, --timing --cmdLine)."""
    import importlib.util
    import sys
    import types
    ref = "/root/reference/tst/plot.py"
    if not os.path.exists(ref):
        pytest.skip("reference tree not present")
    saved = {k: sys.modules.get(k) for k in ("matplotlib", "matplotlib.pyplot", "mpl_toolkits", "mpl_toolkits.mplot3d")}
    try:
        for name in saved:
            sys.modules[name] = types.ModuleType(name)
        sys.modules["mpl_toolkits.mplot3d"].Axes3D = object
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
        spec = importlib.util.spec_from_file_location("geneo_ref_plot", ref)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    log = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cli_tridiag_geneo1ASM.log")
    lines = open(log).readlines()
    first = next(i for i, ln in enumerate(lines) if ln.startswith("INFO:"))
    lines = [ln for ln in lines[first:] if ln[0:3] != "WRNG" and len(ln.split()) > 0]  # plot.py:215-216
    j = mod.job()
    j.buildJob("tridiag-ws=1-np=2-tol=1e-12-metis=dual-ksp=gmres-pc=geneoASM1.log", lines)
    assert (j.nbDOF, j.nbCoef, j.metis, j.overlap, j.ksp, j.pc) == (8, 23, "dual", "0", "gmres", "geneo1ASM")
    assert j.L1 == "ldlt" and j.tau == "0.10" and j.L2 == "blocklanczos+ldlt" and j.gamma is None and not j.offload
    assert (j.estimDimE, j.estimDimEMin, j.estimDimEMax, j.realDimE, j.realDimEMin, j.realDimEMax, j.nicolaides) == (0, 0, 0, 2, 1, 1, 2)
    assert j.nbIt == 6 and j.setUpSolve > 0 and j.itSolve > 0 and abs(j.solve - (j.setUpSolve + j.itSolve)) < 1e-4
    assert j.getSurfName() == "metis=dual-overlap=0-ksp=gmres-pc=geneo1ASM-L1=ldlt-tau=0.10-L2=blocklanczos+ldlt-distribE"


def test_decomposition_and_layout_digests_are_pinned():
    """SHA-256 of everything the decomposition and the rank layouts produce (index sets, multiplicities, intersections,
    weighted Neumann / Dirichlet matrices, owned rows of A, ghosts) over 22 small configurations -- box partitions seen by
    single ranks of 1/2/4/8-GPU runs, METIS dual / nodal parts with overlap 0..2, parts grouped onto 2 and 3 ranks, the
    graph generator.  The digests were written by the triplet-list implementation the oracle comparisons pinned
    (tools/host_decomp_digest.py); the row-wise assembly on dense node ids has to reproduce them to the bit."""
    import importlib.util
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("host_decomp_digest", os.path.join(root, "tools", "host_decomp_digest.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    want = json.load(open(os.path.join(root, "tests", "golden", "decomposition_digests.json")))
    got = mod.run()
    assert set(got) == set(want)
    assert [k for k in got if got[k] != want[k]] == []


def test_decomposition_of_a_mesh_that_does_not_hold_every_node_id():
    """A (sub-)mesh whose elements use only part of the global node ids -- what every rank of a multi-GPU run holds -- goes
    through the dense node index: the same subdomains, multiplicities, intersections and matrices as the mesh renumbered
    from zero, with the global ids shifted."""
    mesh = go.gen_grid(2, 6, 1e-2)
    ep, ei, em = np.asarray(mesh.elem_ptr), np.asarray(mesh.elem_idx), np.asarray(mesh.mat_val)
    p = g.Problem().set_mesh(mesh.nb_node + 8, ep, ei + 3, em)  # 3 unused ids in front, 5 behind
    q = g.Problem().set_mesh(mesh.nb_node, ep, ei, em)
    for prob in (p, q):
        prob.decompose(3, True, 1)
    for s in range(3):
        a, ma = p.sub_nodes(s)
        b, mb = q.sub_nodes(s)
        assert np.array_equal(a, b + 3) and np.array_equal(ma, mb)
        for which in (0, 1):
            A, B = p.sub_matrix(s, which), q.sub_matrix(s, which)
            assert np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices) and np.array_equal(A.data, B.data)
        for t in range(3):
            assert np.array_equal(p.sub_intersect(s, t), q.sub_intersect(s, t))

