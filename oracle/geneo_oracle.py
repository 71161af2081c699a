"""
geneo_oracle.py -- CPU restatement of geneo4PETSc's GenEO hot path.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module.
The product (geneo4petsc_b200/) never does: it fails loudly when its CUDA library is missing.

What is restated (every function cites the reference file:line it follows, paths relative to /root/reference):
  * text input reader                          src/geneo4PETSc.cpp:98-194
  * METIS partition (through oracle_shim)      src/geneo4PETSc.cpp:381-421
  * decomposition / overlap / multiplicities   src/geneo4PETSc.cpp:196-379
  * weighted local Neumann matrices, RHS       src/geneo4PETSc.cpp:447-494, 643-715, 807-835
  * GenEO setup (D, A_dir, A_rob, pencils, Sylvester count, eigenpairs, Nicolaides, Z, E)
                                               src/geneo.cpp:965-1000, 1613-1670, 1234-1366, 502-533, 626-744, 842-963
  * local tau / gamma (GenEO-2)                src/geneo.cpp:1097-1232
  * PC apply (additive / hybrid / eff. hybrid; ASM/RAS/SRAS/ORAS/SORAS)
                                               src/geneo.cpp:1435-1542, 1902-2098
  * outer Krylov: PETSc-faithful left-preconditioned CG and GMRES(m) with the KSPConvergedDefault rule
                                               call site src/geneo4PETSc.cpp:1240 (PETSc itself is a third-party
                                               dependency absent from /root/reference: PETSc >= 3.10.3, see DESIGN.md)

Third-party arithmetic the reference delegates to and that is NOT in /root/reference (PETSc, SLEPc/ARPACK, MUMPS) is
replaced by scipy (SuperLU `splu`, ARPACK `eigsh(sigma=0)`, LAPACK `eigh`).

Parity pinning: the 84 goldens of tst/dummy pin local matrices, RHS and solution (tests/golden/dummy_*.json, checked by
tests/test_oracle_golden.py).  Eigenvalues, eigen-counts, dim E and iteration counts are pinned by NOTHING in the
reference tree ("parity unpinned" for those, see DESIGN.md); for them this oracle is the definition of "reference".
"""
from __future__ import annotations

import ctypes
import math
import os
import subprocess
import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np
import scipy.linalg as sla
import scipy.sparse as sp
import scipy.sparse.linalg as spla

_HERE = os.path.dirname(os.path.abspath(__file__))
_SHIM = None


def _shim():
    """Load (building if needed) oracle/_build/liboracle_shim.so."""
    global _SHIM
    if _SHIM is not None:
        return _SHIM
    path = os.path.join(_HERE, "_build", "liboracle_shim.so")
    if not os.path.exists(path):
        subprocess.check_call(["make", "-C", _HERE, "shim"], stdout=subprocess.DEVNULL)
    lib = ctypes.CDLL(path)
    lib.oracle_get_input.restype = ctypes.c_int
    lib.oracle_metis_part.restype = ctypes.c_int
    lib.oracle_free.restype = None
    lib.oracle_free.argtypes = [ctypes.c_void_p]
    _SHIM = lib
    return lib


# ---------------------------------------------------------------------------------------------------------------------
# Mesh = list of elements (CSR) + one dense row-major matrix per element.
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class Mesh:
    nb_node: int
    elem_ptr: np.ndarray  # int64 [nb_elem+1]
    elem_idx: np.ndarray  # int64 [elem_ptr[-1]]
    mat_ptr: np.ndarray  # int64 [nb_elem+1]  offsets into mat_val (n_e*n_e per element)
    mat_val: np.ndarray  # float64

    @property
    def nb_elem(self) -> int:
        return len(self.elem_ptr) - 1


def _mesh_from_lists(elems: List[List[int]], mats: List[List[float]], nb_node: int) -> Mesh:
    elem_ptr = np.zeros(len(elems) + 1, dtype=np.int64)
    mat_ptr = np.zeros(len(elems) + 1, dtype=np.int64)
    for e, (d, m) in enumerate(zip(elems, mats)):
        elem_ptr[e + 1] = elem_ptr[e] + len(d)
        mat_ptr[e + 1] = mat_ptr[e] + len(m)
    elem_idx = np.array([i for d in elems for i in d], dtype=np.int64)
    mat_val = np.array([v for m in mats for v in m], dtype=np.float64)
    return Mesh(nb_node, elem_ptr, elem_idx, mat_ptr, mat_val)


def read_input_file(path: str, inp_eps: float = 1e-4) -> Mesh:
    """Text format A.  Follows src/geneo4PETSc.cpp:98-142 (readLineFile) and :144-194 (readInputFile)."""
    elems, mats, nodes = [], [], set()
    with open(path) as f:
        for line in f:
            line = line.lstrip()
            if not line or line[0] in "%#":
                continue
            dofs, vals, fill_dof = [], [], True
            for tok in line.split():
                if tok == "-":
                    fill_dof = False
                    continue
                if fill_dof:
                    dofs.append(int(tok))
                else:
                    vals.append(float(tok))
            if not vals:  # default matrix, :130-138
                n = len(dofs)
                for i in range(n):
                    for j in range(n):
                        vals.append(1.0 + inp_eps if i == j else -1.0 / float(n - 1))
            if len(vals) != len(dofs) ** 2:
                raise ValueError("bad matrix in file")
            elems.append(dofs)
            mats.append(vals)
            nodes.update(dofs)
    nb_node = len(nodes)
    if max(nodes) + 1 != nb_node:
        raise ValueError("bad node set")
    return _mesh_from_lists(elems, mats, nb_node)


def read_rhs_file(path: str, n: int) -> np.ndarray:
    """Text format B.  Follows src/geneo4PETSc.cpp:836-861 (missing value defaults to 1.)."""
    b = np.zeros(n)
    with open(path) as f:
        for line in f:
            line = line.lstrip()
            if not line or line[0] in "%#":
                continue
            t = line.split()
            b[int(t[0])] = float(t[1]) if len(t) > 1 else 1.0
    return b


def ref_generator(kind: str, args: str) -> Mesh:
    """Run the reference's OWN generator (oracle/_ref/libgen<kind>.so, built from tst/<kind>/*.cpp) -- the
    `--inpLibA L A` path of src/geneo4PETSc.cpp:75-96."""
    path = os.path.join(_HERE, "_ref", "libgen%s.so" % kind)
    if not os.path.exists(path):
        raise FileNotFoundError(path + " (run `make -C oracle ref` where /root/reference exists)")
    return plugin_input(path, args)


def plugin_input(path: str, args: str) -> Mesh:
    """The mesh of any library exporting the reference's getInput() plug-in ABI, called with `args`."""
    lib = _shim()
    ne, nn = ctypes.c_uint32(), ctypes.c_uint32()
    p_ptr, p_idx = ctypes.POINTER(ctypes.c_uint32)(), ctypes.POINTER(ctypes.c_uint32)()
    p_val = ctypes.POINTER(ctypes.c_double)()
    n_idx, n_val = ctypes.c_uint64(), ctypes.c_uint64()
    rc = lib.oracle_get_input(path.encode(), args.encode(), ctypes.byref(ne), ctypes.byref(nn), ctypes.byref(p_ptr),
                              ctypes.byref(p_idx), ctypes.byref(n_idx), ctypes.byref(p_val), ctypes.byref(n_val))
    if rc != 0:
        raise RuntimeError("getInput of %s failed" % path)
    elem_ptr = np.ctypeslib.as_array(p_ptr, shape=(ne.value + 1,)).astype(np.int64)
    elem_idx = np.ctypeslib.as_array(p_idx, shape=(max(n_idx.value, 1),))[: n_idx.value].astype(np.int64)
    mat_val = np.ctypeslib.as_array(p_val, shape=(max(n_val.value, 1),))[: n_val.value].copy()
    for p in (p_ptr, p_idx, p_val):
        lib.oracle_free(ctypes.cast(p, ctypes.c_void_p))
    npe = np.diff(elem_ptr)
    mat_ptr = np.concatenate([[0], np.cumsum(npe * npe)]).astype(np.int64)
    return Mesh(int(nn.value), elem_ptr, elem_idx, mat_ptr, mat_val)


# ---- numpy restatement of the reference generators (vectorised; checked against ref_generator in tests) -------------
def _kappa_1d(interp: str, alpha: float, beta: float, x: np.ndarray) -> np.ndarray:
    """tst/laplacian/laplacianServices.cpp:27-40 (computeKappa)."""
    if interp == "quad":
        return alpha * x * x + beta
    if interp == "lin":
        return alpha * x + beta
    if interp == "minmax":
        k = np.ones_like(x)
        k[x >= beta] = alpha
        k[x >= 2.0 * beta] = 1.0
        return k
    return np.ones_like(x)


def grid_size(dim: int, size: int, weak: int = 1) -> int:
    """tst/laplacian/laplacian.cpp:101-105 (float truncation of sqrt/cbrt reproduced)."""
    if dim == 1:
        return size * weak
    if dim == 2:
        return int(math.sqrt(size * size * weak))
    return int(np.cbrt(float(size * size * size * weak)))


def gen_grid(dim: int = 3, size: int = 4, inp_eps: float = 1e-4, kappa_max: float = 1.0, interp: str = "",
             weak: int = 1, heat: bool = False, lbd: float = 1.0, dt: float = 0.1) -> Mesh:
    """Laplacian (tst/laplacian/laplacian.cpp:56-188) and heat (tst/heat/heat.cpp:117-261) meshes of 2-node edge
    elements + 1-node Dirichlet elements, emitted in the SAME ORDER as the reference loops (d3, d2, d1, then for
    nd=1..3: [BC element at offset -1 of the last dimension], edge to the +1 neighbour)."""
    n = grid_size(dim, size, weak)
    n1, n2, n3 = n, (n if dim >= 2 else 1), (n if dim >= 3 else 1)
    xmax = float(n - 1)
    alpha, beta = 0.0, 1.0  # laplacianServices.cpp:7-25 (initLaplacian)
    if interp == "quad":
        alpha = (kappa_max - beta) / (xmax * xmax)
    elif interp == "lin":
        alpha = (kappa_max - beta) / xmax
    elif interp == "minmax":
        alpha, beta = kappa_max, xmax / 3.0
    d3, d2, d1 = np.meshgrid(np.arange(n3), np.arange(n2), np.arange(n1), indexing="ij")
    d1, d2, d3 = d1.ravel(), d2.ravel(), d3.ravel()  # central points in loop order
    c = d1 + n1 * d2 + n1 * n2 * d3
    kap = (_kappa_1d(interp, alpha, beta, d1.astype(float)) * _kappa_1d(interp, alpha, beta, d2.astype(float))
           * _kappa_1d(interp, alpha, beta, d3.astype(float)))
    npts = len(c)
    # slots per central point, in emission order: nd=1:+1, nd=2:(BC if dim==2), +1, nd=3:(BC if dim==3), +1 ; (dim==1: BC first)
    slots = []  # (mask, second node or -1)
    if dim == 1:
        slots.append((d1 == 0, None))
    slots.append((d1 + 1 < n1, c + 1))
    if dim == 2:
        slots.append((d2 == 0, None))
    slots.append((d2 + 1 < n2, c + n1))
    if dim == 3:
        slots.append((d3 == 0, None))
    slots.append((d3 + 1 < n3, c + n1 * n2))
    ns = len(slots)
    valid = np.stack([m for m, _ in slots], axis=1)  # [npts, ns]
    is_bc = np.array([nb is None for _, nb in slots])
    second = np.stack([np.full(npts, -1) if nb is None else nb for _, nb in slots], axis=1)
    first = np.repeat(c[:, None], ns, axis=1)
    kap2 = np.repeat(kap[:, None], ns, axis=1)
    bc2 = np.repeat(is_bc[None, :], npts, axis=0)
    v = valid.ravel()
    first, second, kap2, bc2 = first.ravel()[v], second.ravel()[v], kap2.ravel()[v], bc2.ravel()[v]
    ne = len(first)
    npe = np.where(bc2, 1, 2)
    elem_ptr = np.concatenate([[0], np.cumsum(npe)]).astype(np.int64)
    elem_idx = np.empty(elem_ptr[-1], dtype=np.int64)
    elem_idx[elem_ptr[:-1]] = first
    elem_idx[elem_ptr[:-1][~bc2] + 1] = second[~bc2]
    mat_ptr = np.concatenate([[0], np.cumsum(npe * npe)]).astype(np.int64)
    mat_val = np.empty(mat_ptr[-1])
    dg = (1.0 + inp_eps) * kap2  # laplacianServices.cpp:79-91
    og = -1.0 * kap2
    if heat:  # heat.cpp:53-59, 109: lbd*laplacian + inertia/dt
        dg = lbd * dg + (1.0 / 3.0) / dt
        og = lbd * og + (1.0 / 6.0) / dt
    o = mat_ptr[:-1]
    mat_val[o[bc2]] = dg[bc2]
    oo = o[~bc2]
    mat_val[oo] = dg[~bc2]
    mat_val[oo + 1] = og[~bc2]
    mat_val[oo + 2] = og[~bc2]
    mat_val[oo + 3] = dg[~bc2]
    return Mesh(int(npts), elem_ptr, elem_idx, mat_ptr, mat_val)


# ---------------------------------------------------------------------------------------------------------------------
# Partition + decomposition
# ---------------------------------------------------------------------------------------------------------------------
def metis_partition(mesh: Mesh, nb_part: int, dual: bool = True) -> Tuple[np.ndarray, np.ndarray]:
    """src/geneo4PETSc.cpp:381-421."""
    lib = _shim()
    epart = np.zeros(mesh.nb_elem, dtype=np.int64)
    npart = np.zeros(mesh.nb_node, dtype=np.int64)
    eptr = np.ascontiguousarray(mesh.elem_ptr, dtype=np.int64)
    eind = np.ascontiguousarray(mesh.elem_idx, dtype=np.int64)
    rc = lib.oracle_metis_part(ctypes.c_int(1 if dual else 0), ctypes.c_int64(mesh.nb_elem), ctypes.c_int64(mesh.nb_node),
                               eptr.ctypes.data_as(ctypes.c_void_p), eind.ctypes.data_as(ctypes.c_void_p),
                               ctypes.c_int64(nb_part), epart.ctypes.data_as(ctypes.c_void_p),
                               npart.ctypes.data_as(ctypes.c_void_p))
    if rc != 0:
        raise RuntimeError("METIS KO")
    return epart, npart


@dataclass
class Decomposition:
    nb_part: int
    nodes: List[np.ndarray]  # sorted global node ids of each domain (std::set order)
    elems: List[np.ndarray]  # sorted global element ids of each domain
    node_mult: np.ndarray  # per global node
    elem_mult: np.ndarray  # per global element
    intersect: List[List[np.ndarray]]  # intersect[p][q] = LOCAL indices (in p) of nodes shared with q


def decompose(mesh: Mesh, nb_part: int, elem_part: np.ndarray, node_part: np.ndarray, dual: bool = True,
              overlap: int = 0) -> Decomposition:
    """src/geneo4PETSc.cpp:196-215 (element partition from node partition), :238-269 (overlap layers),
    :292-379 (domains, multiplicities, pairwise intersections in local indices)."""
    ne, nn = mesh.nb_elem, mesh.nb_node
    npe = np.diff(mesh.elem_ptr)
    e_of_idx = np.repeat(np.arange(ne), npe)
    inc = sp.csr_matrix((np.ones(len(mesh.elem_idx), dtype=np.int32), (e_of_idx, mesh.elem_idx)), shape=(ne, nn))
    inc_t = inc.T.tocsr()
    nodes, elems = [], []
    node_mult = np.zeros(nn, dtype=np.int64)
    elem_mult = np.zeros(ne, dtype=np.int64)
    for p in range(nb_part):
        if dual:
            in_p = (elem_part == p)
        else:  # an element belongs to p if one of its nodes does (:203-211)
            in_p = (inc @ (node_part == p).astype(np.int32)) > 0
        for _ in range(overlap):  # :244-269 : add every element sharing a node with the current element set
            touched = (inc_t @ in_p.astype(np.int32)) > 0
            in_p = in_p | ((inc @ touched.astype(np.int32)) > 0)
        ep = np.flatnonzero(in_p)
        np_ = np.flatnonzero((inc_t @ in_p.astype(np.int32)) > 0)
        elems.append(ep)
        nodes.append(np_)
        elem_mult[ep] += 1
        node_mult[np_] += 1
    intersect = []
    for p in range(nb_part):
        row = []
        for q in range(nb_part):
            if p == q:
                row.append(np.zeros(0, dtype=np.int64))
                continue
            glob = np.intersect1d(nodes[p], nodes[q], assume_unique=True)
            row.append(np.searchsorted(nodes[p], glob).astype(np.int64))
        intersect.append(row)
    return Decomposition(nb_part, nodes, elems, node_mult, elem_mult, intersect)


def local_neumann(mesh: Mesh, dec: Decomposition, p: int) -> sp.csr_matrix:
    """A_neu,p = sum_e (1/elemIdxMult[e]) K_e in local numbering (rank in the sorted node set).
    src/geneo4PETSc.cpp:447-494 (buildDomain weighting :473-476), :643-715 (preallocate/fill, ADD_VALUES)."""
    nodes, ep = dec.nodes[p], dec.elems[p]
    n = len(nodes)
    s, t = mesh.elem_ptr[ep], mesh.elem_ptr[ep + 1]
    npe = t - s
    rows, cols, vals = [], [], []
    for k in np.unique(npe):  # group elements by size
        sel = ep[npe == k]
        idx = mesh.elem_idx[mesh.elem_ptr[sel][:, None] + np.arange(k)[None, :]]  # [m,k] global
        loc = np.searchsorted(nodes, idx)
        m = mesh.mat_val[mesh.mat_ptr[sel][:, None] + np.arange(k * k)[None, :]].reshape(-1, k, k)
        m = m * (1.0 / dec.elem_mult[sel].astype(float))[:, None, None]
        rows.append(np.repeat(loc[:, :, None], k, axis=2).ravel())
        cols.append(np.repeat(loc[:, None, :], k, axis=1).ravel())
        vals.append(m.ravel())
    a = sp.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n)).tocsr()
    a.sum_duplicates()
    a.sort_indices()
    return a


def assemble_global(nb_dof: int, dec: Decomposition, a_neu: List[sp.csr_matrix]) -> sp.csr_matrix:
    """A = sum_i R_i^T A_neu,i R_i  (MatConvert MATIS->MATAIJ, src/geneo.cpp:1692)."""
    rows, cols, vals = [], [], []
    for p, a in enumerate(a_neu):
        c = a.tocoo()
        rows.append(dec.nodes[p][c.row])
        cols.append(dec.nodes[p][c.col])
        vals.append(c.data)
    g = sp.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(nb_dof, nb_dof)).tocsr()
    g.sum_duplicates()
    g.sort_indices()
    return g


# ---------------------------------------------------------------------------------------------------------------------
# GenEO preconditioner
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class GenEOOptions:
    """Defaults: src/geneo.cpp:2649-2662.  Grammar of -geneo_lvl: :2349-2369."""
    lvl1: str = "ASM"  # ASM | RAS | SRAS | ORAS | SORAS
    lvl2: str = "1"  # 0 | 1 | H1 | E1 | 2 | H2 | E2
    optim: float = 0.0
    tau: float = 0.1
    gamma: float = 10.0
    cst: bool = False
    cut: int = -1
    no_syl: bool = False
    offload: bool = False  # semantically a no-op here (coarse problem replicated)
    eps_tol: float = 1e-3  # src/geneo.cpp:658
    dense_max: int = 1500  # oracle knob: below this size the pencil is solved densely (ground truth)

    def flags(self):
        l1 = self.lvl1
        ras = l1 in ("RAS", "SRAS", "ORAS", "SORAS")
        sras = l1 in ("SRAS", "SORAS")
        oras = l1 in ("ORAS", "SORAS")
        lvl2 = {"0": 0, "1": 1, "H1": 1, "E1": 1, "2": 2, "H2": 2, "E2": 2}[self.lvl2]
        hybrid = self.lvl2 in ("H1", "E1", "H2", "E2")
        eff = self.lvl2 in ("E1", "E2")
        return l1 == "ASM", ras, sras, oras, lvl2, hybrid, eff

    def name(self) -> str:
        """src/geneo.cpp:2245-2268 (buildGenEOName)."""
        _, _, _, _, lvl2, hybrid, eff = self.flags()
        return "geneo%d%s%s" % (lvl2, ("E" if eff else "H") if hybrid else "", self.lvl1)


def inertia(m: sp.spmatrix) -> Tuple[int, int, int]:
    """(#neg, #zero, #pos) eigenvalues of the symmetric matrix m.  Stands for MUMPS LDL^T + MatGetInertia
    (src/geneo.cpp:452-500).  Dense LDL^T (Bunch-Kaufman) for small sizes, exact eigenvalues as a cross-check path;
    sparse LU sign count otherwise (diag(U) signs = signs of the LDL^T pivots when no row exchange occurs)."""
    n = m.shape[0]
    if n <= 3000:
        w = sla.eigvalsh(m.toarray())
        tol = 0.0
        return int(np.sum(w < -tol)), int(np.sum(w == 0.0)), int(np.sum(w > tol))
    lu = spla.splu(sp.csc_matrix(m), diag_pivot_thresh=0.0, permc_spec="MMD_AT_PLUS_A",
                   options=dict(SymmetricMode=True))
    d = lu.U.diagonal()
    # Row permutation parity is irrelevant for the count when perm_r == perm_c (symmetric pivoting).
    if not np.array_equal(lu.perm_r, lu.perm_c):
        w = spla.eigsh(m, k=min(n - 1, 200), sigma=0.0, which="LM", return_eigenvectors=False)
        neg = int(np.sum(w < 0))
        return neg, 0, n - neg
    return int(np.sum(d < 0)), int(np.sum(d == 0)), int(np.sum(d > 0))


def _gen_eig_small(a: sp.spmatrix, b: sp.spmatrix, nev: int, which: str, dense_max: int, tol: float):
    """nev eigenpairs of A x = lambda B x closest to 0 ('tau': shift-invert sigma=0, EPS_TARGET_MAGNITUDE,
    src/geneo.cpp:635-650) or largest ('gamma': EPS_LARGEST_MAGNITUDE, :652-656)."""
    n = a.shape[0]
    nev = max(1, min(nev, n))
    if n <= dense_max or nev >= n - 1:
        w, v = sla.eigh(a.toarray(), b.toarray())
        order = np.argsort(np.abs(w)) if which == "tau" else np.argsort(-np.abs(w))
        sel = order[:nev]
        return w[sel], v[:, sel]
    ncv = min(n - 1, max(2 * nev + 1, 20))
    if which == "tau":
        w, v = spla.eigsh(sp.csc_matrix(a), k=nev, M=sp.csc_matrix(b), sigma=0.0, which="LM", tol=tol * 1e-3, ncv=ncv)
        order = np.argsort(np.abs(w))
    else:
        w, v = spla.eigsh(sp.csc_matrix(a), k=nev, M=sp.csc_matrix(b), which="LM", tol=tol * 1e-3, ncv=ncv)
        order = np.argsort(-np.abs(w))
    return w[order], v[:, order]


@dataclass
class SubdomainSetup:
    n: int
    a_neu: sp.csr_matrix
    a_dir: sp.csr_matrix
    a_rob: Optional[sp.csr_matrix]
    d: np.ndarray
    solve_l1: object  # callable x -> M^{-1} x
    z: Optional[np.ndarray] = None  # n x nev  (already D-weighted)
    eigvals: List[float] = field(default_factory=list)
    estim: int = 0
    nicolaides: int = 0
    tau_loc: float = -1.0
    gamma_loc: float = -1.0


class GenEOOracle:
    """Two-level GenEO Schwarz preconditioner, CPU restatement.  One object holds ALL subdomains (the reference holds
    one per MPI rank, src/geneo4PETSc.cpp:604)."""

    def __init__(self, nb_dof: int, dec: Decomposition, a_neu: List[sp.csr_matrix], opt: GenEOOptions,
                 a_glob: Optional[sp.csr_matrix] = None):
        self.n = nb_dof
        self.dec = dec
        self.opt = opt
        self.a_neu = a_neu
        self.a = a_glob if a_glob is not None else assemble_global(nb_dof, dec, a_neu)
        self.sub: List[SubdomainSetup] = []
        self.timers: Dict[str, float] = {}
        self.z_off = None
        self.e = None
        self.e_lu = None
        # One worker thread per subdomain stands for the reference's one MPI rank per subdomain (src/geneo4PETSc.cpp:604);
        # SuperLU / ARPACK / LAPACK release the GIL inside scipy.  1 = serial (tests).
        self.workers = 1

    def _map(self, fn, items):
        if self.workers <= 1 or len(items) <= 1:
            return [fn(i) for i in items]
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=self.workers) as ex:
            return list(ex.map(fn, items))

    # ---- setup: src/geneo.cpp:1672-1843 (setUpGenEOPC) ---------------------------------------------------------------
    def setup(self, b: Optional[np.ndarray] = None):
        opt = self.opt
        asm, ras, sras, oras, lvl2, hybrid, eff = opt.flags()
        t0 = time.perf_counter()

        def one(p):
            nodes = self.dec.nodes[p]
            a_dir = self.a[nodes][:, nodes].tocsr()  # MatCreateSubMatrices, :1699
            a_dir.sort_indices()
            mult = self.dec.node_mult[nodes]
            d = 1.0 / mult.astype(float)  # createPartitionOfUnity :977-980
            a_rob = None
            if oras:  # createRobinMatrix :1613-1670
                a_rob = a_dir.copy()
                if abs(opt.optim) > np.finfo(float).eps:
                    border = np.flatnonzero(mult > 1)
                    if len(border):
                        sub = self.a_neu[p][border][:, border].tocoo()
                        add = sp.coo_matrix((sub.data, (border[sub.row], border[sub.col])), shape=a_dir.shape)
                        a_rob = (a_rob + opt.optim * add).tocsr()
            m1 = a_rob if oras else a_dir  # setUpLevel1 :137-143
            lu = spla.splu(sp.csc_matrix(m1))
            return SubdomainSetup(len(nodes), self.a_neu[p], a_dir, a_rob, d, lu.solve)

        self.sub.extend(self._map(one, list(range(self.dec.nb_part))))
        self.timers["l1_setup"] = time.perf_counter() - t0
        self.x0 = np.zeros(self.n)
        if lvl2:
            self._setup_level2()
            if eff and b is not None:  # :1601-1603
                self.x0 = self.apply_q(b)
        return self

    def _local_tau(self, p: int) -> float:
        """src/geneo.cpp:1097-1118."""
        if self.opt.cst:
            return self.opt.tau
        k = int(self.dec.node_mult[self.dec.nodes[p]].max())
        t = k * self.opt.tau
        return 0.9 if t >= 1.0 else t

    def _local_gamma(self, p: int) -> float:
        """src/geneo.cpp:1120-1232.  NB the reference's connectivity quirk is reproduced: C_pq = 0 when the
        intersection is NOT empty and 1 when it is empty (:1143-1145)."""
        g = self.opt.gamma
        if self.opt.cst:
            return g
        P = self.dec.nb_part
        c = np.zeros((P, P))
        for r in range(P):
            for q in range(P):
                c[r, q] = 1.0 if r == q else (0.0 if len(self.dec.intersect[r][q]) else 1.0)
        f = 1.0 / c.sum(axis=1)
        m = c * f[:, None] * f[None, :]
        w = sla.eigvalsh(m)
        lam = w[np.argmax(np.abs(w))]
        g = g / lam * f[p] * f[p]
        return 1.1 if g <= 1.0 else g

    def _eigen_local_problem(self, s: SubdomainSetup, a, b, param: float, pb: str, cut: int):
        """src/geneo.cpp:842-963 (eigenLocalProblem) + :502-533 (Sylvester estimate) + :626-722 (solve + filter)."""
        opt = self.opt
        nev = 1  # SLEPc default nev when nothing is requested
        if not opt.no_syl:
            neg, _, pos = inertia((a - param * b).tocsr())
            est = neg if pb == "tau" else pos
            est = min(est, s.n)
            if cut > 0:
                est = min(est, cut)
            s.estim += est
            if est > 0:
                nev = est
        if cut > 0 and nev > cut:
            nev = cut
        w, v = _gen_eig_small(a, b, nev, pb, opt.dense_max, opt.eps_tol)
        keep = (w <= param) if pb == "tau" else (w >= param)
        vals, vecs = list(w[keep]), [v[:, i] for i in np.flatnonzero(keep)]
        if pb == "tau":  # Nicolaides :897-944
            eps = np.finfo(float).eps
            if len(vals) > 0 and min(vals) >= eps:
                one = np.ones(s.n)
                ratio = abs(float(one @ (a @ one)) / float(one @ (b @ one)))
                if ratio <= np.finfo(np.float32).eps:
                    vals.append(0.0)
                    vecs.append(one)
                    s.nicolaides += 1
        return vals, vecs

    def _setup_level2(self):
        """src/geneo.cpp:1234-1366 (buildCoarseSpaceWithGenEO), :249-286 / :355-407 (Z), :1028-1066 (E)."""
        opt = self.opt
        _, _, _, _, lvl2, _, _ = opt.flags()
        cut = opt.cut
        if lvl2 == 2 and cut >= 2:
            cut = cut // 2  # :1275
        t0 = time.perf_counter()

        def one(p):
            s = self.sub[p]
            dd = sp.diags(s.d)
            dadird = (dd @ s.a_dir @ dd).tocsr()  # :1243-1246
            vals, vecs = [], []
            if lvl2 == 1:
                vals, vecs = self._eigen_local_problem(s, s.a_neu, dadird, opt.tau, "tau", cut)
            else:
                if s.a_rob is None:
                    raise ValueError("GenEO-2 requires an optimised level 1 (ORAS/SORAS)")
                s.tau_loc = self._local_tau(p)
                v1, e1 = self._eigen_local_problem(s, s.a_neu, s.a_rob, s.tau_loc, "tau", cut)
                s.gamma_loc = self._local_gamma(p)
                v2, e2 = self._eigen_local_problem(s, dadird, s.a_rob, s.gamma_loc, "gamma", cut)
                vals, vecs = v1 + v2, e1 + e2
            if not vecs:  # :1305-1314
                vals, vecs = [0.0], [np.ones(s.n)]
                s.nicolaides += 1
            s.eigvals = vals
            s.z = np.stack(vecs, axis=1) * s.d[:, None]  # fillZE2L :261

        self._map(one, list(range(len(self.sub))))
        self.timers["l2_eig"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        nev = [s.z.shape[1] for s in self.sub]
        self.z_off = np.concatenate([[0], np.cumsum(nev)]).astype(int)  # :363-375
        rows, cols, vals = [], [], []
        for p, s in enumerate(self.sub):
            nodes = self.dec.nodes[p]
            rows.append(np.repeat(nodes, nev[p]))
            cols.append(np.tile(np.arange(self.z_off[p], self.z_off[p + 1]), s.n))
            vals.append(s.z.ravel())
        self.zmat = sp.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))),
                                  shape=(self.n, self.z_off[-1])).tocsr()
        self.e = (self.zmat.T @ (self.a @ self.zmat)).toarray()  # MatPtAP :1033
        self.e_lu = sla.lu_factor(self.e)
        self.timers["l2_ze"] = time.perf_counter() - t0

    # ---- apply -------------------------------------------------------------------------------------------------------
    def apply_q(self, x: np.ndarray) -> np.ndarray:
        """Q = Z E^-1 Z^T, src/geneo.cpp:1435-1517."""
        w = self.zmat.T @ x
        w = sla.lu_solve(self.e_lu, w)
        return self.zmat @ w

    def _level1(self, x: np.ndarray) -> np.ndarray:
        """restrict, [D], M^-1, [D], prolong-add.  src/geneo.cpp:1980-2025, 1845-1900."""
        _, ras, sras, _, _, _, _ = self.opt.flags()
        out = np.zeros(self.n)

        def one(p):
            s = self.sub[p]
            xl = x[self.dec.nodes[p]]
            if ras:
                xl = xl * s.d
            xl = s.solve_l1(xl)
            if sras:
                xl = xl * s.d
            return xl

        for p, xl in enumerate(self._map(one, list(range(len(self.sub))))):  # summed in subdomain order
            np.add.at(out, self.dec.nodes[p], xl)
        return out

    def apply(self, x: np.ndarray) -> np.ndarray:
        """src/geneo.cpp:2051-2098 (applyGenEOPC), :1962-2038 (applyLevel1), :1902-1945 (projectOnFineSpace)."""
        _, _, _, _, lvl2, hybrid, eff = self.opt.flags()
        y = np.zeros(self.n)
        if lvl2 and not eff:
            y = self.apply_q(x)
        xx = x.copy()
        if hybrid and not eff:
            xx = xx - self.a @ y  # (I - P^T) x = x - A Q x
        xx = self._level1(xx)
        if hybrid:
            xx = xx - self.apply_q(self.a @ xx)  # (I - P)
        return y + xx


# ---------------------------------------------------------------------------------------------------------------------
# PETSc-faithful Krylov (left preconditioning, preconditioned residual norm, KSPConvergedDefault)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class KSPResult:
    x: np.ndarray
    its: int
    rnorm: float
    reason: str
    history: List[float]

    @property
    def converged(self) -> bool:
        return self.reason.startswith("KSP_CONVERGED")


def _ttol(pc, b, rnorm0, rtol, atol, guess_nonzero):
    """KSPConvergedDefault at iteration 0 with a non-zero initial guess: the reference norm is ||M^-1 b||
    (the driver always sets KSPSetInitialGuessNonzero, src/geneo4PETSc.cpp:1348)."""
    if guess_nonzero:
        snorm = float(np.linalg.norm(pc(b)))
        if snorm == 0.0:
            snorm = rnorm0
    else:
        snorm = rnorm0
    return max(rtol * snorm, atol), snorm


def ksp_cg(a, pc, b, x0, rtol=1e-5, atol=1e-50, dtol=1e5, max_it=10000, guess_nonzero=True) -> KSPResult:
    """PETSc KSPCG, KSP_NORM_PRECONDITIONED (default), single reduction off."""
    x = x0.copy()
    r = b - a @ x if guess_nonzero else b.copy()
    z = pc(r)
    dp = float(np.linalg.norm(z))
    hist = [dp]
    ttol, rn0 = _ttol(pc, b, dp, rtol, atol, guess_nonzero)

    def test(rn):
        if rn != rn:
            return "KSP_DIVERGED_NANORINF"
        if rn <= ttol:
            return "KSP_CONVERGED_ATOL" if rn < atol else "KSP_CONVERGED_RTOL"
        if rn >= dtol * rn0:
            return "KSP_DIVERGED_DTOL"
        return ""

    reason = test(dp)
    if reason:
        return KSPResult(x, 0, dp, reason, hist)
    beta = float(z @ r)
    p = None
    betaold = 1.0
    i = 0
    while i < max_it:
        if beta == 0.0:
            return KSPResult(x, i, dp, "KSP_CONVERGED_ATOL", hist)
        if i > 0 and beta * betaold < 0.0:
            return KSPResult(x, i, dp, "KSP_DIVERGED_INDEFINITE_PC", hist)
        p = z.copy() if i == 0 else z + (beta / betaold) * p
        w = a @ p
        dpi = float(p @ w)
        betaold = beta
        if dpi <= 0.0:
            return KSPResult(x, i + 1, dp, "KSP_DIVERGED_INDEFINITE_MAT", hist)
        al = beta / dpi
        x = x + al * p
        r = r - al * w
        z = pc(r)
        dp = float(np.linalg.norm(z))
        hist.append(dp)
        reason = test(dp)
        if reason:
            return KSPResult(x, i + 1, dp, reason, hist)
        beta = float(z @ r)
        i += 1
    return KSPResult(x, i, dp, "KSP_DIVERGED_ITS", hist)


def ksp_gmres(a, pc, b, x0, rtol=1e-5, atol=1e-50, dtol=1e5, max_it=10000, restart=30, guess_nonzero=True) -> KSPResult:
    """PETSc KSPGMRES: left preconditioning, classical Gram-Schmidt without refinement, restart `restart`,
    convergence on the recurrence estimate of ||M^-1 r||, happy-breakdown tolerance 1e-30."""
    n = len(b)
    x = x0.copy()
    its = 0
    hist = []
    ttol = rn0 = None
    reason = ""
    while True:
        r = pc(b - a @ x) if (guess_nonzero or its > 0) else pc(b)
        res = float(np.linalg.norm(r))
        if ttol is None:
            ttol, rn0 = _ttol(pc, b, res, rtol, atol, guess_nonzero)
            hist.append(res)

        def test(rn):
            if rn != rn:
                return "KSP_DIVERGED_NANORINF"
            if rn <= ttol:
                return "KSP_CONVERGED_ATOL" if rn < atol else "KSP_CONVERGED_RTOL"
            if rn >= dtol * rn0:
                return "KSP_DIVERGED_DTOL"
            return ""

        reason = test(res)
        if reason or its >= max_it:
            break
        if res == 0.0:
            reason = "KSP_CONVERGED_ATOL"
            break
        v = np.zeros((restart + 1, n))
        h = np.zeros((restart + 1, restart))
        cs, sn, g = np.zeros(restart), np.zeros(restart), np.zeros(restart + 1)
        v[0] = r / res
        g[0] = res
        k = 0
        while k < restart and its < max_it:
            w = pc(a @ v[k])
            hk = v[: k + 1] @ w  # VecMDot
            w = w - hk @ v[: k + 1]  # VecMAXPY
            h[: k + 1, k] = hk
            tt = float(np.linalg.norm(w))
            hapbnd = min(abs(tt / g[k]) if g[k] != 0.0 else 1e-30, 1e-30)  # KSPGMRESCycle: haptol = 1e-30
            happy = tt < hapbnd
            if not happy:
                v[k + 1] = w / tt
            h[k + 1, k] = tt
            for j in range(k):  # apply previous rotations
                t1 = h[j, k]
                h[j, k] = cs[j] * t1 + sn[j] * h[j + 1, k]
                h[j + 1, k] = -sn[j] * t1 + cs[j] * h[j + 1, k]
            den = math.hypot(h[k, k], h[k + 1, k])
            if den == 0.0:
                reason = "KSP_DIVERGED_BREAKDOWN"
                break
            cs[k], sn[k] = h[k, k] / den, h[k + 1, k] / den
            h[k, k] = den
            h[k + 1, k] = 0.0
            g[k + 1] = -sn[k] * g[k]
            g[k] = cs[k] * g[k]
            res = abs(g[k + 1])
            k += 1
            its += 1
            hist.append(res)
            reason = test(res)
            if reason:
                break
            if happy:
                reason = "KSP_CONVERGED_HAPPY_BREAKDOWN"
                break
        if k > 0:  # build solution
            y = sla.solve_triangular(h[:k, :k], g[:k])
            x = x + y @ v[:k]
        if reason:
            break
        if its >= max_it:
            reason = "KSP_DIVERGED_ITS"
            break
    if not reason:
        reason = "KSP_DIVERGED_ITS"
    return KSPResult(x, its, res, reason, hist)


# ---------------------------------------------------------------------------------------------------------------------
# Driver-level restatement: src/geneo4PETSc.cpp:1283-1394 (solve) = createA + createB + KSPSetUp + KSPSolve
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class SolveReport:
    dec: Decomposition
    a: sp.csr_matrix
    b: np.ndarray
    pc: GenEOOracle
    ksp: KSPResult
    nnz_loc: int
    setup_s: float
    solve_s: float
    true_rel_res: float


def run_case(mesh: Mesh, nb_part: int, opt: GenEOOptions, dual: bool = True, overlap: int = 0, ksp: str = "gmres",
             rtol: float = 1e-5, atol: float = 1e-50, max_it: int = 10000, restart: int = 30,
             b: Optional[np.ndarray] = None, part: Optional[Tuple[np.ndarray, np.ndarray]] = None,
             workers: int = 1) -> SolveReport:
    if part is None:
        part = metis_partition(mesh, nb_part, dual)
    dec = decompose(mesh, nb_part, part[0], part[1], dual, overlap)
    a_neu = [local_neumann(mesh, dec, p) for p in range(nb_part)]
    a = assemble_global(mesh.nb_node, dec, a_neu)
    if b is None:  # createB :820-831
        b = a @ np.arange(1, mesh.nb_node + 1, dtype=float)
    t0 = time.perf_counter()
    pc = GenEOOracle(mesh.nb_node, dec, a_neu, opt, a)
    pc.workers = workers
    pc.setup(b)
    t1 = time.perf_counter()
    fn = ksp_cg if ksp == "cg" else ksp_gmres
    kw = dict(rtol=rtol, atol=atol, max_it=max_it)
    if ksp != "cg":
        kw["restart"] = restart
    res = fn(a, pc.apply, b, pc.x0, **kw)
    t2 = time.perf_counter()
    tr = float(np.linalg.norm(a @ res.x - b) / np.linalg.norm(b))
    return SolveReport(dec, a, b, pc, res, int(sum(m.nnz for m in a_neu)), t1 - t0, t2 - t1, tr)
