"""Thin ctypes mirror of include/geneo_b200.h.  Names follow the reference's interface (hdr/geneo.hpp, hdr/geneo_c.h,
src/geneo4PETSc.cpp): Problem = the driver's partitionAndDecompose state, GeneoPC = geneoContext + KSP."""
import ctypes as C

import numpy as np

from ._lib import load

lib = load()
_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)
_u32p = C.POINTER(C.c_uint32)
_f64p = C.POINTER(C.c_double)
lib.geneo_last_error.restype = C.c_char_p
lib.geneo_ksp_reason_name.restype = C.c_char_p

KSP_REASONS = {2: "KSP_CONVERGED_RTOL", 3: "KSP_CONVERGED_ATOL", 7: "KSP_CONVERGED_HAPPY_BREAKDOWN", -3: "KSP_DIVERGED_ITS",
               -4: "KSP_DIVERGED_DTOL", -5: "KSP_DIVERGED_BREAKDOWN", -8: "KSP_DIVERGED_INDEFINITE_PC",
               -9: "KSP_DIVERGED_NANORINF", -10: "KSP_DIVERGED_INDEFINITE_MAT"}


class GeneoError(RuntimeError):
    pass


def _chk(rc):
    if rc != 0:
        raise GeneoError(lib.geneo_last_error().decode())


def _p(a, t):
    return a.ctypes.data_as(t) if a is not None else None


def device_count():
    return int(lib.geneo_device_count())


def counters():
    """{launches, h2d, d2h}: kernel launches and host<->device bytes issued by the library so far."""
    c = np.zeros(3, dtype=np.int64)
    _chk(lib.geneo_counters(_p(c, _i64p)))
    return dict(launches=int(c[0]), h2d=int(c[1]), d2h=int(c[2]))


def profile_dump(path):
    _chk(lib.geneo_profile_dump(str(path).encode()))


def host_sym_eig(a):
    a = np.array(a, dtype=np.float64, order="C")
    n = a.shape[0]
    w = np.zeros(n)
    _chk(lib.geneo_host_sym_eig(C.c_int(n), _p(a, _f64p), _p(w, _f64p)))
    return w, a


def microbench(kind, n, reps=5):
    r = np.zeros(2)
    _chk(lib.geneo_microbench(C.c_int(kind), C.c_int(n), C.c_int(reps), _p(r, _f64p)))
    return float(r[0]), float(r[1])


class Problem:
    """Input mesh + METIS partition + overlapping decomposition (src/geneo4PETSc.cpp:571-641)."""

    def __init__(self):
        self.h = C.c_void_p()
        _chk(lib.geneo_problem_create(C.byref(self.h)))

    def __del__(self):
        if getattr(self, "h", None) and self.h:
            lib.geneo_problem_destroy(self.h)
            self.h = None

    def set_mesh(self, nb_node, elem_ptr, elem_idx, elem_mat):
        ep = np.ascontiguousarray(elem_ptr, dtype=np.uint32)
        ei = np.ascontiguousarray(elem_idx, dtype=np.uint32)
        em = np.ascontiguousarray(elem_mat, dtype=np.float64)
        _chk(lib.geneo_problem_set_mesh(self.h, C.c_uint32(nb_node), C.c_uint32(len(ep) - 1), _p(ep, _u32p), _p(ei, _u32p), _p(em, _f64p)))
        return self

    def generate(self, kind, args):
        _chk(lib.geneo_problem_generate(self.h, kind.encode(), args.encode()))
        return self

    def read_file(self, path, inp_eps=1e-4):
        _chk(lib.geneo_problem_read_file(self.h, str(path).encode(), C.c_double(inp_eps)))
        return self

    def decompose(self, nb_part, dual=True, overlap=0, elem_part=None, node_part=None):
        ep = None if elem_part is None else np.ascontiguousarray(elem_part, dtype=np.int32)
        npart = None if node_part is None else np.ascontiguousarray(node_part, dtype=np.int32)
        _chk(lib.geneo_problem_decompose(self.h, C.c_int(nb_part), C.c_int(1 if dual else 0), C.c_int(overlap), _p(ep, _i32p), _p(npart, _i32p)))
        return self

    def set_subdomains(self, nb_dof, subs):
        """Pre-decomposed input: subs = [(global_ids ascending, A_neu scipy CSR[, A_dir scipy CSR]), ...] (initGenEOPC's view)."""
        _chk(lib.geneo_problem_begin_subdomains(self.h, C.c_int64(nb_dof), C.c_int(len(subs))))
        for s, item in enumerate(subs):
            ids = np.ascontiguousarray(item[0], dtype=np.int32)
            mats = []
            for m in item[1:3]:
                m = m.tocsr()
                mats += [np.ascontiguousarray(m.indptr, dtype=np.int64), np.ascontiguousarray(m.indices, dtype=np.int32),
                         np.ascontiguousarray(m.data, dtype=np.float64)]
            while len(mats) < 6:
                mats.append(None)
            _chk(lib.geneo_problem_set_subdomain(self.h, C.c_int(s), C.c_int64(len(ids)), _p(ids, _i32p), _p(mats[0], _i64p),
                                                 _p(mats[1], _i32p), _p(mats[2], _f64p), _p(mats[3], _i64p), _p(mats[4], _i32p),
                                                 _p(mats[5], _f64p)))
        _chk(lib.geneo_problem_end_subdomains(self.h))
        return self

    def sizes(self):
        v = [C.c_int64() for _ in range(4)]
        _chk(lib.geneo_problem_sizes(self.h, *[C.byref(x) for x in v]))
        return dict(nb_node=v[0].value, nb_elem=v[1].value, nb_part=v[2].value, nnz=v[3].value)

    def mesh(self):
        s = self.sizes()
        ni, nm = C.c_int64(), C.c_int64()
        _chk(lib.geneo_problem_mesh_sizes(self.h, C.byref(ni), C.byref(nm)))
        ep = np.zeros(s["nb_elem"] + 1, dtype=np.int64)
        ei = np.zeros(ni.value, dtype=np.int32)
        em = np.zeros(nm.value)
        _chk(lib.geneo_problem_get_mesh(self.h, _p(ep, _i64p), _p(ei, _i32p), _p(em, _f64p)))
        return ep, ei, em

    def partition(self):
        s = self.sizes()
        ep = np.zeros(s["nb_elem"], dtype=np.int32)
        npart = np.zeros(s["nb_node"], dtype=np.int32)
        _chk(lib.geneo_problem_get_partition(self.h, _p(ep, _i32p), _p(npart, _i32p)))
        return ep, npart

    def sub_sizes(self, s):
        v = np.zeros(4, dtype=np.int64)
        _chk(lib.geneo_problem_sub_sizes(self.h, C.c_int(s), _p(v, _i64p)))
        return v

    def sub_nodes(self, s):
        n = int(self.sub_sizes(s)[0])
        nodes, mult = np.zeros(n, dtype=np.int32), np.zeros(n, dtype=np.int32)
        _chk(lib.geneo_problem_sub_nodes(self.h, C.c_int(s), _p(nodes, _i32p), _p(mult, _i32p)))
        return nodes, mult

    def sub_intersect(self, s, q):
        cnt = C.c_int64()
        _chk(lib.geneo_problem_sub_intersect(self.h, C.c_int(s), C.c_int(q), None, C.c_int64(0), C.byref(cnt)))
        idx = np.zeros(cnt.value, dtype=np.int32)
        if cnt.value:
            _chk(lib.geneo_problem_sub_intersect(self.h, C.c_int(s), C.c_int(q), _p(idx, _i32p), C.c_int64(cnt.value), C.byref(cnt)))
        return idx

    def sub_matrix(self, s, which):
        """which = 0: weighted Neumann matrix, 1: Dirichlet matrix; returns a scipy CSR."""
        import scipy.sparse as sp
        sz = self.sub_sizes(s)
        n, nnz = int(sz[0]), int(sz[2 + which])
        ptr, idx, val = np.zeros(n + 1, dtype=np.int64), np.zeros(nnz, dtype=np.int32), np.zeros(nnz)
        _chk(lib.geneo_problem_sub_matrix(self.h, C.c_int(s), C.c_int(which), _p(ptr, _i64p), _p(idx, _i32p), _p(val, _f64p)))
        return sp.csr_matrix((val, idx, ptr), shape=(n, n))


class GeneoPC:
    """geneoContext + the KSP that drives it.  Usage mirrors the reference driver (src/geneo4PETSc.cpp:1328-1369):
    create -> set_from_options(argv) -> setup(problem) -> ksp_solve(b)."""
    TIMER_NAMES = ["lvl1SetupMinv", "lvl2SetupTauLoc", "lvl2SetupTauSyl", "lvl2SetupTauEig", "lvl2SetupGammaLoc",
                   "lvl2SetupGammaSyl", "lvl2SetupGammaEig", "lvl2SetupSyl", "lvl2SetupEig", "lvl2SetupZ", "lvl2SetupE",
                   "lvl1Apply", "lvl1ApplyScatter", "lvl1ApplyMinv", "lvl1ApplyGather", "lvl1ApplyPrjFS", "lvl2Apply",
                   "lvl2ApplyZt", "lvl2ApplyEinv", "lvl2ApplyZ", "symbolic", "operator", "setup", "upload", "numeric",
                   "update_layout"]

    def __init__(self, options=None):
        self.h = C.c_void_p()
        _chk(lib.geneo_pc_create(C.byref(self.h)))
        self.problem = None
        if options:
            self.set_from_options(options)

    def __del__(self):
        if getattr(self, "h", None) and self.h:
            lib.geneo_pc_destroy(self.h)
            self.h = None

    def set_from_options(self, argv):
        if isinstance(argv, str):
            argv = argv.split()
        arr = (C.c_char_p * len(argv))(*[a.encode() for a in argv])
        _chk(lib.geneo_pc_set_from_options(self.h, C.c_int(len(argv)), arr))
        return self

    def setup(self, problem):
        self.problem = problem  # borrowed by the library: keep it alive
        _chk(lib.geneo_pc_setup(self.h, problem.h))
        return self

    def refactor(self):
        """Numeric setup again on the device-resident matrices (same pattern)."""
        _chk(lib.geneo_pc_refactor(self.h))
        return self

    def update(self, problem):
        """PCSetUp with SAME_NONZERO_PATTERN: the values of `problem` (same partition, node sets and patterns as the last
        setup) replace the resident ones, then the numeric setup runs.  A mismatch raises and leaves the PC as it was."""
        self.problem = problem  # borrowed by the library: keep it alive
        _chk(lib.geneo_pc_update(self.h, problem.h))
        return self

    def level_profile(self):
        """(us, bytes, items) per phase of one level-1 solve: forward levels leaves-first, then backward root-first."""
        n = C.c_int()
        _chk(lib.geneo_pc_level_profile(self.h, None, None, None, C.c_int(0), C.byref(n)))
        us, by, it = np.zeros(n.value), np.zeros(n.value), np.zeros(n.value, dtype=np.int64)
        _chk(lib.geneo_pc_level_profile(self.h, _p(us, _f64p), _p(by, _f64p), _p(it, _i64p), C.c_int(n.value), C.byref(n)))
        return us, by, it

    def kernel_time(self):
        """(ms, launches) of the level-1 solve kernel since the last call (needs -geneo_kernel_timing)."""
        ms, n = C.c_double(), C.c_int64()
        _chk(lib.geneo_pc_kernel_time(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    @property
    def name(self):
        buf = C.create_string_buffer(64)
        _chk(lib.geneo_pc_name(self.h, buf, C.c_int(64)))
        return buf.value.decode()

    def info(self):
        i, r = np.zeros(16, dtype=np.int64), np.zeros(4)
        _chk(lib.geneo_pc_info(self.h, _p(i, _i64p), _p(r, _f64p)))
        keys = ["nbDof", "nbPart", "lvl2", "hybrid", "effHybrid", "lvl1ORAS", "offload", "noSyl", "estimDimE", "estimMin",
                "estimMax", "realDimE", "realMin", "realMax", "nicolaides", "nE"]
        d = {k: int(v) for k, v in zip(keys, i)}
        d.update(tau=r[0], gamma=r[1], optim=r[2])
        return d

    def timers(self):
        t = np.zeros(len(self.TIMER_NAMES))
        _chk(lib.geneo_pc_timers(self.h, _p(t, _f64p), C.c_int(len(t))))
        return dict(zip(self.TIMER_NAMES, t.tolist()))

    def stats(self):
        s = np.zeros(8)
        _chk(lib.geneo_pc_stats(self.h, _p(s, _f64p)))
        keys = ["factor_bytes", "factor_nnz", "factor_flops", "trisolve_bytes", "apply_bytes", "spmv_bytes", "applies", "sum_ni"]
        return dict(zip(keys, s.tolist()))

    def factor_stats(self):
        """every numeric factorization of the last (re-)setup: device seconds, flops, count; host seconds of the shared ordering."""
        s = np.zeros(4)
        _chk(lib.geneo_pc_factor_stats(self.h, _p(s, _f64p)))
        return dict(seconds=s[0], flops=s[1], count=int(s[2]), ordering_reuse_s=s[3])

    def factor_bench(self):
        """(seconds, flops) of the level-1 factorizations run once more, alone on the device (CUDA events)."""
        s = np.zeros(2)
        _chk(lib.geneo_pc_factor_bench(self.h, _p(s, _f64p)))
        return float(s[0]), float(s[1])

    def sub_info(self, s):
        i, r = np.zeros(8, dtype=np.int64), np.zeros(2)
        _chk(lib.geneo_pc_sub_info(self.h, C.c_int(s), _p(i, _i64p), _p(r, _f64p)))
        keys = ["n", "nev", "estim", "nicolaides", "eigSteps", "eigDim", "neg", "perturbed"]
        d = {k: int(v) for k, v in zip(keys, i)}
        d.update(tauLoc=r[0], gammaLoc=r[1])
        return d

    def sub_eigenvalues(self, s):
        cnt = C.c_int()
        _chk(lib.geneo_pc_sub_eigenvalues(self.h, C.c_int(s), None, C.c_int(0), C.byref(cnt)))
        v = np.zeros(cnt.value)
        if cnt.value:
            _chk(lib.geneo_pc_sub_eigenvalues(self.h, C.c_int(s), _p(v, _f64p), C.c_int(cnt.value), C.byref(cnt)))
        return v

    def sub_z(self, s):
        si = self.sub_info(s)
        z = np.zeros((si["n"], si["nev"]))
        _chk(lib.geneo_pc_sub_z(self.h, C.c_int(s), _p(z, _f64p)))
        return z

    def coarse_inverse(self):
        ne = self.info()["nE"]
        e = np.zeros((ne, ne))
        _chk(lib.geneo_pc_coarse_matrix(self.h, _p(e, _f64p)))
        return e

    # host-buffer entry points (what a PETSc caller sees)
    def apply(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.zeros_like(x)
        _chk(lib.geneo_pc_apply(self.h, _p(x, _f64p), _p(y, _f64p)))
        return y

    def mult(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.zeros_like(x)
        _chk(lib.geneo_mult(self.h, _p(x, _f64p), _p(y, _f64p)))
        return y

    def make_rhs(self):
        b = np.zeros(self.info()["nbDof"])
        _chk(lib.geneo_make_rhs(self.h, _p(b, _f64p)))
        return b

    def ksp_solve(self, b, ksp="gmres", rtol=1e-5, atol=1e-50, dtol=1e5, max_it=10000, restart=30):
        b = np.ascontiguousarray(b, dtype=np.float64)
        x = np.zeros_like(b)
        out, rn, hist = np.zeros(3, dtype=np.int64), C.c_double(), np.zeros(max_it + 2)
        _chk(lib.geneo_ksp_solve(self.h, ksp.encode(), _p(b, _f64p), _p(x, _f64p), C.c_double(rtol), C.c_double(atol),
                                 C.c_double(dtol), C.c_int(max_it), C.c_int(restart), _p(out, _i64p), C.byref(rn),
                                 _p(hist, _f64p), C.c_int(len(hist))))
        return dict(x=x, its=int(out[0]), reason=int(out[1]), reason_name=KSP_REASONS.get(int(out[1]), "?"),
                    rnorm=rn.value, history=hist[: int(out[2])].copy())

    def apply_block(self, X):
        """PCMatApply: Y = M^-1 X for the k columns of X, shape (n, k) (or (n,)); 8 columns per pass over the factors."""
        X = np.asarray(X, dtype=np.float64)
        Xf = np.asfortranarray(X[:, None] if X.ndim == 1 else X)
        Y = np.zeros(Xf.shape, order="F")
        _chk(lib.geneo_pc_apply_block(self.h, C.c_int(Xf.shape[1]), _p(Xf, _f64p), C.c_int64(Xf.shape[0]), _p(Y, _f64p),
                                      C.c_int64(Y.shape[0])))
        return Y.reshape(X.shape)

    def ksp_solve_block(self, B, ksp="cg", rtol=1e-5, atol=1e-50, dtol=1e5, max_it=10000):
        """KSPMatSolve with lock-step CG on the k columns of B, shape (n, k): each column as ksp_solve(B[:, j], "cg")."""
        B = np.asarray(B, dtype=np.float64)
        Bf = np.asfortranarray(B[:, None] if B.ndim == 1 else B)
        k = Bf.shape[1]
        X = np.zeros(Bf.shape, order="F")
        out, rn = np.zeros(2 * max(k, 1), dtype=np.int64), np.zeros(max(k, 1))
        _chk(lib.geneo_ksp_solve_block(self.h, (ksp or "").encode(), C.c_int(k), _p(Bf, _f64p), C.c_int64(Bf.shape[0]),
                                       _p(X, _f64p), C.c_int64(X.shape[0]), C.c_double(rtol), C.c_double(atol), C.c_double(dtol),
                                       C.c_int(max_it), _p(out, _i64p), _p(rn, _f64p)))
        return dict(x=X.reshape(B.shape), **self._block_result(out, rn, k))

    @staticmethod
    def _block_result(out, rn, k):
        its, reason = out[0:2 * k:2].astype(int), out[1:2 * k:2].astype(int)
        return dict(its=its, reason=reason, reason_name=[KSP_REASONS.get(int(r), "?") for r in reason], rnorm=rn[:k].copy())

    # device-pointer entry points (torch tensors' data_ptr())
    def apply_block_device(self, dx_ptr, dy_ptr, k, ldx, ldy):
        _chk(lib.geneo_pc_apply_block_device(self.h, C.c_int(k), C.c_void_p(dx_ptr), C.c_int64(ldx), C.c_void_p(dy_ptr),
                                             C.c_int64(ldy)))

    def ksp_solve_block_device(self, db_ptr, dx_ptr, k, ldb, ldx, ksp="cg", rtol=1e-5, atol=1e-50, dtol=1e5, max_it=10000):
        out, rn = np.zeros(2 * max(k, 1), dtype=np.int64), np.zeros(max(k, 1))
        _chk(lib.geneo_ksp_solve_block_device(self.h, (ksp or "").encode(), C.c_int(k), C.c_void_p(db_ptr), C.c_int64(ldb),
                                              C.c_void_p(dx_ptr), C.c_int64(ldx), C.c_double(rtol), C.c_double(atol),
                                              C.c_double(dtol), C.c_int(max_it), _p(out, _i64p), _p(rn, _f64p)))
        return self._block_result(out, rn, k)

    def apply_device(self, dx_ptr, dy_ptr):
        _chk(lib.geneo_pc_apply_device(self.h, C.c_void_p(dx_ptr), C.c_void_p(dy_ptr)))

    def apply_q_device(self, dx_ptr, dy_ptr):
        _chk(lib.geneo_pc_apply_q_device(self.h, C.c_void_p(dx_ptr), C.c_void_p(dy_ptr)))

    def mult_device(self, dx_ptr, dy_ptr):
        _chk(lib.geneo_mult_device(self.h, C.c_void_p(dx_ptr), C.c_void_p(dy_ptr)))

    def ksp_solve_device(self, db_ptr, dx_ptr, ksp="gmres", rtol=1e-5, atol=1e-50, dtol=1e5, max_it=10000, restart=30):
        out, rn, hist = np.zeros(3, dtype=np.int64), C.c_double(), np.zeros(max_it + 2)
        _chk(lib.geneo_ksp_solve_device(self.h, ksp.encode(), C.c_void_p(db_ptr), C.c_void_p(dx_ptr), C.c_double(rtol),
                                        C.c_double(atol), C.c_double(dtol), C.c_int(max_it), C.c_int(restart),
                                        _p(out, _i64p), C.byref(rn), _p(hist, _f64p), C.c_int(len(hist))))
        return dict(its=int(out[0]), reason=int(out[1]), reason_name=KSP_REASONS.get(int(out[1]), "?"), rnorm=rn.value,
                    history=hist[: int(out[2])].copy())


def box_ordering(dims, stencil=((1, 0, 0), (0, 1, 0), (0, 0, 1)), threads=1):
    """rank[x + d0 (y + d1 z)] of the reference nested dissection of a box (host only)."""
    d = np.ascontiguousarray(dims, dtype=np.int32)
    st = np.ascontiguousarray(stencil, dtype=np.int32).reshape(-1, 3)
    rank = np.zeros(int(d[0]) * int(d[1]) * int(d[2]), dtype=np.int32)
    _chk(lib.geneo_box_ordering(_p(d, _i32p), C.c_int(len(st)), _p(st, _i32p), C.c_int(threads), _p(rank, _i32p)))
    return rank


class Symbolic:
    """Host-only view of the symbolic analysis (test hook)."""

    def __init__(self, a_csr, nb=128, ordering=1, amalgamate=True, perm=None):
        a = a_csr.tocsr()
        self.n = a.shape[0]
        ptr = np.ascontiguousarray(a.indptr, dtype=np.int64)
        idx = np.ascontiguousarray(a.indices, dtype=np.int32)
        self.h = C.c_void_p()
        if perm is not None:    # caller-supplied permutation (new -> old)
            pp = np.ascontiguousarray(perm, dtype=np.int32)
            _chk(lib.geneo_symbolic_create_perm(C.c_int(self.n), _p(ptr, _i64p), _p(idx, _i32p), C.c_int(nb),
                                                C.c_int(1 if amalgamate else 0), _p(pp, _i32p), C.byref(self.h)))
        else:
            _chk(lib.geneo_symbolic_create(C.c_int(self.n), _p(ptr, _i64p), _p(idx, _i32p), C.c_int(nb), C.c_int(ordering),
                                           C.c_int(1 if amalgamate else 0), C.byref(self.h)))
        i, r = np.zeros(11, dtype=np.int64), np.zeros(1)
        _chk(lib.geneo_symbolic_info(self.h, _p(i, _i64p), _p(r, _f64p)))
        keys = ["n", "nfronts", "nlevels", "lSize", "uArena", "wArena", "nRowIdx", "nRel", "nAsm", "nsuper", "cArena"]
        self.info = {k: int(v) for k, v in zip(keys, i)}
        self.info["flops"] = float(r[0])
        self.perm = np.zeros(self.n, dtype=np.int32)
        self.fronts = np.zeros((self.info["nfronts"], 17), dtype=np.int64)
        self.row_idx = np.zeros(self.info["nRowIdx"], dtype=np.int32)
        self.rel = np.zeros(max(1, self.info["nRel"]), dtype=np.int32)
        self.asm_src = np.zeros(self.info["nAsm"], dtype=np.int64)
        self.asm_dst = np.zeros(self.info["nAsm"], dtype=np.int64)
        _chk(lib.geneo_symbolic_get(self.h, _p(self.perm, _i32p), _p(self.fronts, _i64p), _p(self.row_idx, _i32p),
                                    _p(self.rel, _i32p), _p(self.asm_src, _i64p), _p(self.asm_dst, _i64p)))

    def __del__(self):
        if getattr(self, "h", None) and self.h:
            lib.geneo_symbolic_destroy(self.h)
            self.h = None


def host_prepare_probe(a_csr, perm=None, nb=128, helper=False, scatter_len=0, sort=True):
    """Per-subdomain host preparation of a symmetric CSR matrix (host only): (stage seconds, digest[, scattered factor])."""
    a = a_csr.tocsr()
    if sort:
        a.sort_indices()
    n = a.shape[0]
    ptr = np.ascontiguousarray(a.indptr, dtype=np.int64)
    idx = np.ascontiguousarray(a.indices, dtype=np.int32)
    val = np.ascontiguousarray(a.data, dtype=np.float64)
    sec = np.zeros(4)
    dig = C.c_uint64(0)
    pp = None if perm is None else np.ascontiguousarray(perm, dtype=np.int32)
    out = np.zeros(scatter_len) if scatter_len else None
    _chk(lib.geneo_host_prepare_probe(C.c_int(n), _p(ptr, _i64p), _p(idx, _i32p), _p(val, _f64p),
                                      None if pp is None else _p(pp, _i32p), C.c_int(nb), C.c_int(int(helper)),
                                      _p(sec, _f64p), C.byref(dig), None if out is None else _p(out, _f64p),
                                      C.c_int64(scatter_len)))
    return (sec, int(dig.value)) if out is None else (sec, int(dig.value), out)
