/*
 * geneo_b200.h -- C ABI of libgeneob200.so: a B200-native (sm_100a) drop-in for the data-parallel hot path of
 * geneo4PETSc (two-level GenEO Schwarz preconditioner + the preconditioned Krylov iteration it drives).
 *
 * Plain pointers and sizes only (no PETSc, no torch, no C++ types).  Every entry point returns 0 on success and a
 * non-zero code on failure; geneo_last_error() then holds the message (the reference returns PetscErrorCode through
 * CHKERRQ and aborts through SETERRABT, src/geneo.cpp:74).  There is NO CPU fallback: every numeric entry point fails
 * loudly when no CUDA device is present.  Entry points are NOT re-entrant (same as the reference, SURVEY.md 8b).
 *
 * Each entry point cites the reference interface it replaces (paths relative to the reference tree).
 * The PETSc-facing adapter that re-exports createGenEOPC / PCGenEOSetup / initGenEOPC on top of this ABI cannot be compiled in
 * this image (no petsc.h, no MPI): INTEGRATION.md section 2 holds the translation unit a maintainer adds on the reference
 * side; the pre-decomposed input it feeds (geneo_problem_begin_subdomains / _set_subdomain / _end_subdomains) and the PETSc-free
 * driver with the reference's command line (geneo4petsc_b200/csrc/cli.cpp -> geneo4petsc_b200/geneo4PETSc) are built and tested.
 */
#ifndef GENEO_B200_H
#define GENEO_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct geneo_problem_s* geneo_problem_t; /* mesh + partition + decomposition (driver half, src/geneo4PETSc.cpp) */
typedef struct geneo_pc_s* geneo_pc_t;           /* geneoContext (hdr/geneo.hpp:46-138)                                  */

const char* geneo_last_error(void);
int geneo_version(void);
int geneo_device_count(void); /* number of visible CUDA devices (0 on a CPU-only host) */

/* ------------------------------------------------------------------------------------------------------------------
 * Driver half: input, partition, decomposition            (src/geneo4PETSc.cpp:571-641 partitionAndDecompose)
 * ------------------------------------------------------------------------------------------------------------------ */
int geneo_problem_create(geneo_problem_t* out);
int geneo_problem_destroy(geneo_problem_t p);
/* The getInput() plug-in ABI (src/geneo4PETSc.cpp:81-85, :1522-1543) flattened: elemPtr[nbElem+1], elemIdx[elemPtr[nbElem]],
 * elemMat = the dense row-major n_e x n_e matrices of all elements back to back. */
int geneo_problem_set_mesh(geneo_problem_t p, uint32_t nbNode, uint32_t nbElem, const uint32_t* elemPtr,
                           const uint32_t* elemIdx, const double* elemMat);
/* --inpLibA replacement for the reference's own generators: kind = "laplacian" (tst/laplacian/laplacian.cpp:56-188),
 * "heat" (tst/heat/heat.cpp:117-261) or "graph" (tst/graph/graph.cpp:38-205); args uses the plug-ins' own grammar
 * ("--size S --dim D --kappa K interp ...", "--size S --level L --noGround ..."). */
int geneo_problem_generate(geneo_problem_t p, const char* kind, const char* args);
/* --inpFileA (src/geneo4PETSc.cpp:144-194). */
int geneo_problem_read_file(geneo_problem_t p, const char* path, double inpEps);
/* METIS partition (src/geneo4PETSc.cpp:381-445) unless elemPart/nodePart are given, then decompose (:292-379) with
 * `overlap` layers (:238-290) and assemble the weighted Neumann matrices (:447-494, :643-715) and the Dirichlet
 * matrices R_i A R_i^T (src/geneo.cpp:1699).  nbPart replaces "mpirun -n" (src/geneo4PETSc.cpp:604). */
int geneo_problem_decompose(geneo_problem_t p, int nbPart, int metisDual, int overlap, const int32_t* elemPart,
                            const int32_t* nodePart);
/* The METIS partition alone (src/geneo4PETSc.cpp:381-445), without the decomposition: elemPart[nbElem], nodePart[nbNode]. */
int geneo_problem_partition(geneo_problem_t p, int nbPart, int metisDual, int32_t* elemPart, int32_t* nodePart);
/* Pre-decomposed input -- what the PETSc plug-in itself receives (initGenEOPC, hdr/geneo.hpp:30-35; PCGenEOSetup,
 * hdr/geneo_c.h:10): per subdomain the local-to-global map (ISLocalToGlobalMapping; ascending, the reference's local
 * numbering src/geneo4PETSc.cpp:485-489), the local Neumann matrix of the MATIS (MatISGetLocalMat, src/geneo.cpp:1714)
 * and optionally the Dirichlet matrix (pcADirLoc).  end_subdomains derives the multiplicities (dofIdxMultLoc), the
 * intersections (intersectLoc) and any missing A_dir,i = R_i A R_i^T (MatConvert + MatCreateSubMatrices, :1692-1699). */
int geneo_problem_begin_subdomains(geneo_problem_t p, int64_t nbDof, int nbPart);
int geneo_problem_set_subdomain(geneo_problem_t p, int s, int64_t n, const int32_t* globalIds, const int64_t* neuPtr,
                                const int32_t* neuIdx, const double* neuVal, const int64_t* dirPtr /* may be NULL */,
                                const int32_t* dirIdx, const double* dirVal);
int geneo_problem_end_subdomains(geneo_problem_t p);
int geneo_problem_sizes(geneo_problem_t p, int64_t* nbNode, int64_t* nbElem, int64_t* nbPart, int64_t* nnzNeuTotal);
int geneo_problem_get_mesh(geneo_problem_t p, int64_t* elemPtr, int32_t* elemIdx, double* elemMat); /* sizes from _mesh_sizes */
int geneo_problem_mesh_sizes(geneo_problem_t p, int64_t* nIdx, int64_t* nMat);
int geneo_problem_get_partition(geneo_problem_t p, int32_t* elemPart, int32_t* nodePart);
/* subdomain s: sizes = {nbNodeLoc, nbElemLoc, nnz(A_neu), nnz(A_dir)} */
int geneo_problem_sub_sizes(geneo_problem_t p, int s, int64_t sizes[4]);
int geneo_problem_sub_nodes(geneo_problem_t p, int s, int32_t* nodes, int32_t* mult);
int geneo_problem_sub_intersect(geneo_problem_t p, int s, int q, int32_t* idx, int64_t cap, int64_t* count);
/* which = 0: A_neu (MatISGetLocalMat, src/geneo.cpp:1714), 1: A_dir (:1699) */
int geneo_problem_sub_matrix(geneo_problem_t p, int s, int which, int64_t* ptr, int32_t* idx, double* val);

/* ------------------------------------------------------------------------------------------------------------------
 * Preconditioner                                             (hdr/geneo_c.h:9-10, hdr/geneo.hpp:30-41)
 * ------------------------------------------------------------------------------------------------------------------ */
int geneo_pc_create(geneo_pc_t* out);                                        /* createGenEOPC, src/geneo.cpp:2639-2728    */
int geneo_pc_set_from_options(geneo_pc_t pc, int argc, const char* const* argv); /* setUpGenEOPCFromOptions, :2329-2514  */
/* initGenEOPC (:2591-2632) + setUpGenEOPC (:1672-1843) for every subdomain of a decomposed problem held by this process */
int geneo_pc_setup(geneo_pc_t pc, geneo_problem_t p);
/* applyGenEOPC (:2051-2098).  Host buffers of length nbDof (copied in and out); x is not modified. */
int geneo_pc_apply(geneo_pc_t pc, const double* x, double* y);
int geneo_pc_apply_device(geneo_pc_t pc, const double* dx, double* dy);     /* same with device pointers            */
int geneo_pc_apply_q_device(geneo_pc_t pc, const double* dx, double* dy);   /* applyQ, :1435-1542                   */
/* PCMatApply: Y = M^-1 X for k >= 1 columns, every variant geneo_pc_apply supports (applyGenEOPC, :2051-2098, column by
 * column).  X and Y are column-major (PETSc MATDENSE) with leading dimensions ldx, ldy >= the vector length (nbDof, or
 * nLoc of geneo_pc_local_sizes on a multi-GPU PC, where the call is collective with local [owned | ghost] columns).
 * 8 columns go through one pass over the level-1 factors; k need not be a multiple of 8.  X is not modified; rows
 * between the vector length and ldy of Y are not written.  Each column agrees with geneo_pc_apply to rounding (the
 * 8-column kernels sum in another order).  Fails with a message when k < 1, before setup ("without context"), or when a
 * leading dimension is below the vector length. */
int geneo_pc_apply_block(geneo_pc_t pc, int k, const double* X, int64_t ldx, double* Y, int64_t ldy);
int geneo_pc_apply_block_device(geneo_pc_t pc, int k, const double* dX, int64_t ldx, double* dY, int64_t ldy);
/* PCSetUp again with an unchanged non-zero pattern: every factorization, eigen-solve, Z and E recomputed from the
 * matrices already resident in HBM (no host analysis, no upload).  setUpGenEOPC is re-entered the same way when PETSc
 * flags the operator as changed (src/geneo.cpp:1672-1843). */
int geneo_pc_refactor(geneo_pc_t pc);
/* PCSetUp again after the operator's VALUES changed and its pattern did not (PETSc's SAME_NONZERO_PATTERN: time steps
 * with a new dt, Newton steps, coefficient updates), re-entering setUpGenEOPC (src/geneo.cpp:1672-1843) without its
 * pattern work: the ordering, the symbolic analysis, the operator's layout and the uploaded plans of the last
 * geneo_pc_setup / geneo_pc_setup_dist are kept; the new A_neu / A_dir values are uploaded, placed on the device, and the
 * numeric setup (every factorization, eigen-solve, Z and E) runs.  The PC is then what a fresh setup on p would give.
 * p must be decomposed with the same nbPart as the last setup, every subdomain with the same node set and the same A_neu
 * and A_dir patterns; only the values may differ.  Fails with a message when the PC is not set up or p is not decomposed.
 * What is checked of the input: the partition and every node set exactly; A_dir exactly (row by row: same length, every
 * entry in the setup's pattern, none twice); A_neu by its number of entries, each inside its row of the setup's A_dir
 * pattern, none twice.  On one process each A_neu entry must also lie in the operator's pattern and the A_neu of all
 * subdomains together must reach every entry of the operator; an A_neu entry moved within those bounds is accepted, and
 * the result is then still exactly what a fresh geneo_pc_setup on p builds (same operator layout, same values).
 * On a PC set up with geneo_pc_setup_dist the call is COLLECTIVE: every rank calls it with its own problem, built the way
 * the setup's was (geneo_problem_generate_boxed + geneo_problem_decompose_owned, or the same METIS grouping) from the same
 * partition and sub_rank.  The operator's owned rows are re-assembled from the rank's mesh by the layout code of
 * geneo_layout_create; the rank's owned and ghost node lists must come out as at the setup (so the halo plan and the NCCL
 * communicator stay), and every owned row must have the operator's pattern.  The operator, A_dir, A_neu and the Robin
 * values are then bit for bit those of a fresh geneo_pc_setup_dist on the new problems.  All ranks vote on the checks:
 * either every rank updates or every rank fails, a rank whose input was rejected with its own reason, the others with a
 * message naming that rank.
 * All checks run before any resident value is overwritten: after a rejected update the PC still holds the previous
 * preconditioner.  If the numeric setup itself fails (e.g. -geneo_chk finds the new A_dir not SPD), the PC is left
 * without context until the next successful setup or update. */
int geneo_pc_update(geneo_pc_t pc, geneo_problem_t p);
/* With -geneo_kernel_timing: CUDA-event time (ms) and launch count of the level-1 solve kernel since the last call. */
int geneo_pc_kernel_time(geneo_pc_t pc, double* ms, int64_t* launches);
/* Diagnostic: one level-1 solve (the PC-apply kernel) with a device timestamp after every level barrier.  Phase p < nlev
 * is the forward sweep of level p (leaves first), then the backward sweep from the root down.  us[p] = duration,
 * bytes[p] = factor bytes streamed, nitems[p] = work items; *nphases = 2 * nlev (arrays may be NULL / shorter: cap). */
int geneo_pc_level_profile(geneo_pc_t pc, double* us, double* bytes, int64_t* nitems, int cap, int* nphases);
/* process-wide counters: {kernel launches, host->device bytes, device->host bytes} issued by this library so far */
int geneo_counters(int64_t c[3]);
/* GENEO_PROFILE=1 in the environment: per-launch-site CUDA-event times accumulated so far -> CSV, then reset */
int geneo_profile_dump(const char* path);
int geneo_pc_destroy(geneo_pc_t pc);                                         /* destroyGenEOPC, :2217-2243           */
/* geneoContext fields the driver reads (src/geneo4PETSc.cpp:928-986, 1123-1225) */
int geneo_pc_name(geneo_pc_t pc, char* buf, int cap);                        /* gCtx->name                           */
/* ints = {nbDof, nbPart, lvl2, hybrid, effHybrid, lvl1ORAS, offload, noSyl, estimDimE, estimMin, estimMax, realDimE,
 *         realMin, realMax, nicolaides, nE}                                                                          */
int geneo_pc_info(geneo_pc_t pc, int64_t ints[16], double reals[4] /* tau, gamma, optim, reserved */);
/* timers (seconds), same order as hdr/geneo.hpp:115-123 then extras; see abi.cpp for the index list */
int geneo_pc_timers(geneo_pc_t pc, double* t, int cap);
/* stats = {factor bytes, factor nnz, factor flops, tri-solve algorithmic bytes per apply, apply algorithmic bytes,
 *          SpMV algorithmic bytes, number of applies so far, sum n_i} */
int geneo_pc_stats(geneo_pc_t pc, double stats[8]);
/* every numeric factorization of the last (re-)setup: out = {device seconds, flops (symbolic: sum k^3/3 + m k^2 + m^2 k),
 * number of factorizations, host seconds spent on the shared reference ordering of the cold setup} */
int geneo_pc_factor_stats(geneo_pc_t pc, double out[4]);
/* Measurement: the level-1 factorizations of every local subdomain once more (same values, same factors), alone on the
 * device, timed with CUDA events: out = {seconds, flops}. */
int geneo_pc_factor_bench(geneo_pc_t pc, double out[2]);
int geneo_pc_sub_info(geneo_pc_t pc, int s, int64_t ints[8] /* n, nev, estim, nicolaides, eigSteps, eigDim, neg, perturbed */,
                      double reals[2] /* tauLoc, gammaLoc */);
int geneo_pc_sub_eigenvalues(geneo_pc_t pc, int s, double* vals, int cap, int* count);
/* Z_s in the subdomain's natural local numbering, row-major n x nev (for parity checks of span(Z)) */
int geneo_pc_sub_z(geneo_pc_t pc, int s, double* z);
int geneo_pc_coarse_matrix(geneo_pc_t pc, double* einv /* nE x nE row-major, E^-1 */);

/* ------------------------------------------------------------------------------------------------------------------
 * Operator and Krylov solve                                   (src/geneo4PETSc.cpp:807-835 createB, :1233-1281)
 * ------------------------------------------------------------------------------------------------------------------ */
int geneo_mult(geneo_pc_t pc, const double* x, double* y);                   /* MatMult(MATIS), host buffers          */
int geneo_mult_device(geneo_pc_t pc, const double* dx, double* dy);
int geneo_make_rhs(geneo_pc_t pc, double* b);                                /* b = A (1,2,...,N)^T, :820-831         */
/* KSPSolve with left preconditioning, preconditioned-norm convergence test, non-zero initial guess flagged
 * (x0 = Q b for the efficient hybrid variants, 0 otherwise: src/geneo.cpp:1601-1607, src/geneo4PETSc.cpp:1348).
 * ksp = "cg" | "gmres".  Host buffers.  out = {iterations, reason (PETSc KSPConvergedReason values), nb history} */
int geneo_ksp_solve(geneo_pc_t pc, const char* ksp, const double* b, double* x, double rtol, double atol, double dtol,
                    int maxIt, int restart, int64_t out[3], double* rnorm, double* history, int histCap);
int geneo_ksp_solve_device(geneo_pc_t pc, const char* ksp, const double* db, double* dx, double rtol, double atol,
                           double dtol, int maxIt, int restart, int64_t out[3], double* rnorm, double* history, int histCap);
/* KSPMatSolve with KSPCG: k >= 1 right-hand sides B (column-major, ldb) solved in lock step, 8 columns per block SpMV and
 * block PC apply (pseudo-block CG).  Every column runs geneo_ksp_solve's CG recurrence -- same initial guess, reference
 * norm, convergence test and breakdown checks -- and stops on its own; X (column-major, ldx) receives the solutions.
 * ksp must be "cg" (block GMRES is not provided).  out[2 j] = iterations, out[2 j + 1] = reason, rnorm[j] = final
 * preconditioned residual norm of column j (either may be NULL).  Argument checks as geneo_pc_apply_block, ksp first. */
int geneo_ksp_solve_block(geneo_pc_t pc, const char* ksp, int k, const double* B, int64_t ldb, double* X, int64_t ldx,
                          double rtol, double atol, double dtol, int maxIt, int64_t* out, double* rnorm);
int geneo_ksp_solve_block_device(geneo_pc_t pc, const char* ksp, int k, const double* dB, int64_t ldb, double* dX, int64_t ldx,
                                 double rtol, double atol, double dtol, int maxIt, int64_t* out, double* rnorm);
const char* geneo_ksp_reason_name(int reason);

/* ------------------------------------------------------------------------------------------------------------------
 * Multi-GPU: one process per GPU (replaces the MPI layer under PETSc VecScatter / MatMult(MATIS) / VecDot:
 * src/geneo.cpp:1850-1852, 1881-1883, 1931-1935; one MPI rank per subdomain at src/geneo4PETSc.cpp:604 becomes
 * several subdomains per GPU).  Every rank decomposes the SAME partition and assembles only its subdomains; a rank
 * owns the rows of the nodes whose lowest-numbered subdomain it holds; local vectors are [owned | ghost].
 * The caller provides the rendezvous (torch.distributed in bench.py/tests): the halo requests (ghost ids grouped by
 * owner, geneo_layout_get) are exchanged by the caller and fed back through geneo_layout_set_send; the NCCL unique id
 * of rank 0 (geneo_nccl_unique_id) is broadcast by the caller.  All later calls are collective over the ranks.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct geneo_layout_s* geneo_layout_t;
/* Structured generator + BOX partition (boxK boxes per axis, element -> box of its lower node) for runs where METIS on
 * the global mesh does not fit one rank; optionally only the SUB-mesh with a node inside [keepLo, keepHi) (node
 * coordinates, global node ids kept).  The partition is stored in the problem (elemPart = NULL in decompose_owned). */
int geneo_problem_generate_boxed(geneo_problem_t p, const char* kind, const char* args, const int32_t boxK[3],
                                 const int32_t keepLo[3] /* may be NULL */, const int32_t keepHi[3], int32_t* edge);
/* like geneo_problem_decompose with an explicit partition, assembling matrices only for subRank[p] == rank */
int geneo_problem_decompose_owned(geneo_problem_t p, int nbPart, int metisDual, int overlap, const int32_t* elemPart,
                                  const int32_t* nodePart, const int32_t* subRank, int rank);
int geneo_layout_create(geneo_problem_t p, int rank, int world, const int32_t* subRank, geneo_layout_t* out); /* host only */
int geneo_layout_destroy(geneo_layout_t l);
int geneo_layout_sizes(geneo_layout_t l, int64_t out[4] /* nOwn, nGhost, nnz(owned rows of A), world */);
int geneo_layout_get(geneo_layout_t l, int32_t* owned, int32_t* ghost, int64_t* ghostPtr /* [world+1] */);
int geneo_layout_matrix(geneo_layout_t l, int64_t* ptr, int32_t* idx, double* val); /* owned rows of A, local columns */
int geneo_layout_set_send(geneo_layout_t l, int peer, const int32_t* globalIds, int64_t n);
int geneo_nccl_unique_id(void* out128);
int geneo_pc_setup_dist(geneo_pc_t pc, geneo_problem_t p, geneo_layout_t l, const void* ncclUid128);
int geneo_pc_local_sizes(geneo_pc_t pc, int64_t out[2] /* nOwn, nLoc: lengths of the vectors the device entry points take */);
int geneo_allreduce_sum(geneo_pc_t pc, double* h, int n); /* host array, in place (statistics) */

/* ------------------------------------------------------------------------------------------------------------------
 * Host-only test hooks (no device needed): symbolic analysis of a CSR pattern, dense symmetric eigen-solver
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct geneo_symbolic_s* geneo_symbolic_t;
/* ordering: 0 natural, 1 METIS nested dissection */
int geneo_symbolic_create(int n, const int64_t* ptr, const int32_t* idx, int nb, int ordering, int amalgamate,
                          geneo_symbolic_t* out);
/* same with a caller-supplied permutation (new -> old) */
int geneo_symbolic_create_perm(int n, const int64_t* ptr, const int32_t* idx, int nb, int amalgamate, const int32_t* perm,
                               geneo_symbolic_t* out);
/* reference nested dissection of a box of grid points (symbolic.hpp box_reference_ordering): rank[dims[0]*dims[1]*dims[2]] */
int geneo_box_ordering(const int32_t dims[3], int nst, const int32_t* stencil, int threads, int32_t* rank);
int geneo_symbolic_destroy(geneo_symbolic_t s);
/* ints = {n, nfronts, nlevels, lSize, uArena, wArena, nRowIdx, nRel, nAsm, nsuper, cArena} ; reals = {flops} */
int geneo_symbolic_info(geneo_symbolic_t s, int64_t ints[11], double reals[1]);
/* fronts: 17 int64 per front = {col0,k,h,parent,level,chain,nchild,rowOff,lOff,uOff,wOff,relOff,ld,uLd,uArena,inplace,pair} */
int geneo_symbolic_get(geneo_symbolic_t s, int32_t* perm, int64_t* fronts, int32_t* rowIdx, int32_t* rel, int64_t* asmSrc,
                       int64_t* asmDst);
/* the whole per-subdomain host preparation (analysis, values permuted to the solver order, scatter map, work lists of
 * every factorization level) of a symmetric CSR matrix taken as A_dir = A_neu; perm may be NULL (METIS).
 * helper & 1: the ordering-independent part runs on a second thread, as in a cold setup with spare cores;
 * helper & 2: force the general path (row sorts + binary searches) that unsymmetric patterns take.
 * scatterOut (optional, scatterLen = factor size of the analysis): the factor array as the assembly kernel fills it.
 * seconds = {analysis, permuted values, work lists, 0}; digest = hash of everything produced (regression checks) */
int geneo_host_prepare_probe(int n, const int64_t* ptr, const int32_t* idx, const double* val, const int32_t* perm, int nb, int helper,
                             double seconds[4], uint64_t* digest, double* scatterOut, int64_t scatterLen);
int geneo_host_sym_eig(int n, double* a /* row-major in, eigenvectors (columns) out */, double* w);
/* eigenvalues + selected rows of the eigenvector matrix (the Rayleigh-Ritz shortcut of the block Lanczos solver):
 * yrows[t * n + j] = component rows[t] of the eigenvector of w[j]; a is destroyed */
int geneo_host_sym_eig_rows(int n, double* a, const int32_t* rows, int nrows, double* w, double* yrows);
/* microbenchmarks on the device (first-run calibration): kind 0 = DMMA 64x64-tile GEMM C=AB^T (M=N=K=n) TFLOP/s,
 * kind 1 = device copy GB/s over n doubles, kind 2 = solve-kernel streaming over ~2 GB of synthetic n x 128 panels at a
 * single level (result[0] = algorithmic GB/s, result[1] = ms per solve), kind 100 * nlev + nr (nlev >= 1, nr = 1, 8 or 16;
 * any other nr is rejected) = level-latency probe of the nr-column solve over nlev levels of `reps` n x 128 panels each
 * (same results as kind 2).  result[0] = rate, result[1] = max abs error vs a reference (kind 0). */
int geneo_microbench(int kind, int n, int reps, double result[2]);

#ifdef __cplusplus
}
#endif
#endif
