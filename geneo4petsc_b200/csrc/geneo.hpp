// geneo.hpp -- the two-level GenEO Schwarz preconditioner and the preconditioned Krylov iteration it drives,
// device-resident.  Host-side mirror of the reference's plug-in interface (hdr/geneo.hpp:46-138 geneoContext,
// src/geneo.cpp:1672-1843 setUpGenEOPC, :2051-2098 applyGenEOPC, :2329-2514 options, :2245-2268 name).
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "comm.hpp"
#include "eigen.hpp"
#include "kernels.hpp"
#include "ldlt.hpp"
#include "mesh.hpp"

namespace geneo {

// Same parameters, names and defaults as geneoContext (hdr/geneo.hpp:54-70; defaults src/geneo.cpp:2649-2662).
struct GeneoOptions {
  bool lvl1ASM = true, lvl1RAS = false, lvl1SRAS = false, lvl1ORAS = false;
  int lvl2 = 1;
  bool hybrid = false, effHybrid = false;
  double optim = 0., tau = 0.1, gamma = 10.;
  bool cst = false;
  int cut = -1;
  bool noSyl = false, offload = false;
  int debug = 0;                // -geneo_dbg F,D : D = 1 timing log, D = 2 + per-subdomain eigenvalue / inertia logs (src/geneo.cpp:2189, 726, 547)
  bool check = false;           // -geneo_chk F   : partition of unity, SPD (inertia), rank of Z (src/geneo.cpp:988, 782-840, 173-247)
  std::string debugFmt = "log", checkFmt = "log";  // log | bin | mat (only the text logs are written; matrices: CLI --verbose 2)
  // knobs of the sub-solvers (stand for the reference's -dls1_/-syl2_/-els2_/-dcs2_ PETSc option prefixes)
  int nb = 128;          // LDL^T panel width
  int ordering = 1;      // 1 METIS NodeND, 0 natural
  bool orderingReuse = true;  // structured problems: box subdomains share one nested dissection (-geneo_ordering_reuse 0|1)
  double epsTol = 1e-4;  // -els2_eps_tol (block Lanczos residual tolerance; reference default 1e-3, src/geneo.cpp:658)
  int epsBlock = 0;      // block size of the Lanczos eigen-solver (-els2_eps_block); 0: 8
  bool releaseWorkspace = false;  // free the factorization / eigen-solver workspaces after every setup
  int epsMaxDim = 0;     // -els2_eps_ncv like bound on the Krylov dimension (0 = automatic)
  double pivRel = 1e-14; // null-pivot threshold relative to max |a_ij| (stands for MUMPS CNTL(3), ICNTL(24) = 1, CNTL(5) = 1e20)
  bool timing = false;   // synchronise and time every apply phase (reference timers hdr/geneo.hpp:115-123)
  bool kernelTiming = false;  // CUDA-event pairs around the level-1 solve kernel (bench.py roofline leg), no host sync

  // Parse "-geneo_lvl ASM,1 -geneo_tau 0.1 ..." (grammar of src/geneo.cpp:2338-2481).  Unknown tokens are ignored
  // (they belong to the caller: PETSc options DB in the reference).  Returns 0, or 1 + message on a bad value.
  int parse(int argc, const char* const* argv, std::string& err);
  std::string name() const;  // buildGenEOName
};

struct SubdomainState {
  int id = 0, n = 0, nev = 0, prevNev = 0;
  int64_t off = 0;   // into the concatenated subdomain vectors
  int zoff = 0;      // into the coarse vector
  std::shared_ptr<LdltPlan> plan;
  std::unique_ptr<LdltFactor> L1;
  DevBuf<int> gidx;       // rank-local index of solver-order row k
  DevBuf<double> d;       // partition of unity, solver order
  DevBuf<double> Z;       // n x nev row-major, solver order, already D-weighted
  CsrDev pat;             // permuted pattern of A_dir; pat.val = A_dir values
  DevBuf<double> vNeu, vRob;
  DevBuf<double> vB, vS;  // D A_dir D and A_neu - tau B (values on the A_dir pattern), kept between re-setups
  std::vector<double> eigvals;
  int estim = 0, nicolaides = 0, eigSteps = 0, eigDim = 0, negL1 = 0, perturbed = 0;
  int sylNeg[2] = {0, 0}, sylNull[2] = {0, 0}, sylEstim[2] = {0, 0}, nKept[2] = {0, 0};  // per pencil (tau, gamma): inertia of A - theta B, kept pairs
  double tauLoc = -1., gammaLoc = -1.;
  int maxMult = 1;
  double anorm = 0.;  // max |a_ij| of A_dir (scale of the static pivot threshold)
  int64_t neuNnz = 0; // entries of the A_neu input (check_values: a same-pattern update has as many)
};

struct KspResult {
  int its = 0, reason = 0;
  double rnorm = 0.;
  std::vector<double> history;
};
// PETSc KSPConvergedReason values used here
enum { KSP_CONVERGED_RTOL = 2, KSP_CONVERGED_ATOL = 3, KSP_CONVERGED_HAPPY_BREAKDOWN = 7, KSP_DIVERGED_ITS = -3,
       KSP_DIVERGED_DTOL = -4, KSP_DIVERGED_BREAKDOWN = -5, KSP_DIVERGED_INDEFINITE_PC = -8, KSP_DIVERGED_NANORINF = -9,
       KSP_DIVERGED_INDEFINITE_MAT = -10 };
const char* ksp_reason_name(int reason);

class GeneoPC {
 public:
  GeneoOptions opt;
  int nbDof = 0;      // global size
  int nLoc = 0;       // length of the vectors held by this process (== nbDof on one GPU)
  int nOwn = 0;       // leading entries owned by this process (dots/norms run over these)
  int nbPart = 0;
  SellMatrix A;       // operator, sum_i R_i^T A_neu,i R_i
  std::vector<SubdomainState> subs;
  int nE = 0;
  cudaStream_t st = 0;

  // reference timers (hdr/geneo.hpp:115-123), seconds
  double lvl1SetupMinvTime = 0., lvl2SetupSylTime = 0., lvl2SetupEigTime = 0., lvl2SetupZTime = 0., lvl2SetupETime = 0.;
  double lvl2SetupTauLocTime = 0., lvl2SetupTauSylTime = 0., lvl2SetupTauEigTime = 0.;
  double lvl2SetupGammaLocTime = 0., lvl2SetupGammaSylTime = 0., lvl2SetupGammaEigTime = 0.;
  double lvl1ApplyTime = 0., lvl1ApplyScatterTime = 0., lvl1ApplyMinvTime = 0., lvl1ApplyGatherTime = 0.;
  double lvl1ApplyPrjFSTime = 0., lvl2ApplyTime = 0., lvl2ApplyZtTime = 0., lvl2ApplyEinvTime = 0., lvl2ApplyZTime = 0.;
  double symbolicTime = 0., operatorTime = 0., setupTime = 0., uploadTime = 0., numericTime = 0., orderingReuseTime = 0.;
  double updateLayoutTime = 0.;  // last same-pattern update of a multi-GPU PC: host rebuild of the rank's layout
  int estimDimE = 0, realDimE = 0, nicolaides = 0;
  int64_t factorBytes = 0, factorNnz = 0, applyCount = 0;
  double factorFlops = 0.;
  // every numeric factorization of the last (re-)setup (A_dir/A_rob, A_neu - tau B, A_neu, ...): device seconds (each call
  // ends with a stream synchronisation), flops from the symbolic analysis, number of factorizations
  double allFactorSeconds = 0., allFactorFlops = 0.;
  int allFactorCount = 0;
  std::string infoL2;
  std::vector<int> nevGlobal, estimGlobal;  // per subdomain (global ids), known on every rank

  GeneoPC();
  ~GeneoPC();
  // Single GPU (layout == nullptr): every subdomain of `dec` is local.  Multi-GPU: the subdomains with
  // layout->subRank[p] == rank are local, vectors are [owned | ghost] (RankLayout), comm holds the NCCL plumbing.
  void setup(const Decomposition& dec, const RankLayout* layout = nullptr, const void* ncclUid = nullptr);
  Comm comm;
  // Multi-GPU setup (layout given): the rank's place and the layout's node lists, which a same-pattern update must reproduce
  // for the local numbering, the halo send lists and comm to stay valid.  `dist` is false after a single-GPU setup.
  struct DistKeys {
    bool dist = false;
    int rank = 0, world = 1;
    std::vector<int> subRank, owned, ghost;
    std::vector<int64_t> ghostPtr;
  } distKeys;
  // Numeric half of the setup again (every factorization, eigen-solve, Z, E) on the matrices already resident in HBM:
  // PCSetUp with an unchanged non-zero pattern.  setup() = host analysis + uploads + numeric_setup().
  void numeric_setup();
  // PCSetUp with SAME_NONZERO_PATTERN and new values, in three steps: check_values() uploads the A_dir / A_neu values of
  // `dec` -- same partition, node sets and patterns as the last setup() -- locates them in the resident pattern and checks
  // them on the device without writing any resident value (on a mismatch it throws and the preconditioner is left as it
  // was); commit_values() puts them in place (A_dir, A_neu, the Robin values, the operator, the pivot scale);
  // numeric_setup() must follow before the next apply.
  // On one process the operator is re-summed from the A_neu values.  On a multi-GPU PC (`layout`: the rank's layout rebuilt
  // from the new problem) the operator's owned rows are the layout's, placed into a fresh value buffer (op).
  struct PendingValues {
    struct Sub { DevBuf<double> dir, neu; DevBuf<int64_t> slot; double anorm = 0.; };  // slot: operator entry of A_neu q, or -1
    std::vector<Sub> subs;
    DevBuf<double> op;  // multi-GPU: the operator's new values, SELL layout of A
  };
  void check_values(const Decomposition& dec, PendingValues& nv, const RankLayout* layout = nullptr);
  // Multi-GPU PC, collective: every rank passes its own problem (null when it has none, `dec` null when it is not
  // decomposed).  Rebuilds the rank's layout from `mesh` / `dec` as setup's caller did (build_rank_layout), requires the
  // setup's owned / ghost lists, then check_values().  Every rank's verdict goes into one vote: either all ranks return with their pending values or all throw
  // (a rejecting rank with its own reason, the others naming it), so no rank commits while another one rejects.
  void check_values_dist(const Mesh* mesh, const Decomposition* dec, PendingValues& nv);
  void commit_values(PendingValues& nv);
  void numeric_begin();
  void numeric_end();
  // accumulated CUDA-event time of the level-1 solve kernel since the last call (ms) and its number of launches
  void kernel_time(double* ms, int64_t* launches);
  void level_profile(std::vector<double>& us, std::vector<double>& bytes, std::vector<int64_t>& nitems);
  void apply(const double* x, double* y);                 // device pointers, length nLoc; x is not modified
  void applyQ(const double* x, double* y);                // y = Z E^-1 Z^T x
  void mult(const double* x, double* y);                  // y = A x on the owned rows (ghosts of x refreshed first)
  void mult_sub(const double* x, const double* b, double* y);  // y = b - A x
  void initial_guess(const double* b, double* x0);        // x0 = Q b (efficient hybrid) or 0 (src/geneo.cpp:1601-1607)
  KspResult solve_cg(const double* b, double* x, double rtol, double atol, double dtol, int maxIt);
  KspResult solve_gmres(const double* b, double* x, double rtol, double atol, double dtol, int maxIt, int restart);
  // Blocks of k right-hand sides (PCMatApply / KSPMatSolve), device pointers, column-major with leading dimensions >= nLoc.
  // 8 columns at a time go through one pass over the level-1 factors (the 8-column solve kernel); k need not be a multiple
  // of 8 (the last chunk is zero-padded).  Rows nLoc..ld-1 of the outputs are not written.
  // apply_block: Y = M^-1 X, every variant apply() supports; X is not written.
  void apply_block(int k, const double* X, int64_t ldx, double* Y, int64_t ldy);
  // solve_cg_block: lock-step (pseudo-block) CG.  Every column runs solve_cg's recurrence from initial_guess()'s x0 (which
  // it computes itself) with its own convergence test; a column that stops is frozen.  X receives the solutions.
  std::vector<KspResult> solve_cg_block(int k, const double* B, int64_t ldb, double* X, int64_t ldx, double rtol, double atol,
                                        double dtol, int maxIt);
  double dot(const double* x, const double* y);
  double norm(const double* x) { return std::sqrt(dot(x, x)); }
  // algorithmic bytes of one PC apply (SURVEY.md 8d) and of its dominant kernel family (factor sweeps)
  double apply_algo_bytes() const;
  double trisolve_algo_bytes() const;
  void copy_einv(double* out) const;  // nE x nE row-major E^-1 to the host
  void factor_bench(double* seconds, double* flops);  // the level-1 factorizations once more, alone on the device (CUDA events)
  void write_timing_log() const;      // -geneo_dbg F,1: <debugNN>.timing.log, the reference's timer list (src/geneo.cpp:2189-2216)
  void run_checks_and_dumps();        // -geneo_chk / -geneo_dbg F,2 after a (re-)setup

 private:
  void numeric_subdomain(SubdomainState& s, LdltWorkspace& ws);
  void numeric_pipeline();
  bool use_pipeline() const;
  int eigen_local_problem(SubdomainState& s, const double* vA, const double* vB, double param, bool tauPb, int cut,
                          LdltWorkspace& ws, std::vector<double>& vals, std::vector<DevBuf<double>>& vecs,
                          std::vector<int>& counts);
  // where an eigen-solve runs: the library's stream and workspace (sequential path) or one of the pipeline's eigen threads
  struct EigCtx { cudaStream_t st = 0; EigWorkspace* ws = nullptr; double* scal = nullptr; struct GroupSolver* grp = nullptr; int member = -1; };
  int eigen_finish(SubdomainState& s, const LdltFactor& fac, const double* vA, const double* vB, double param, bool tauPb, int est,
                   int cut, std::vector<double>& vals, std::vector<DevBuf<double>>& vecs, std::vector<int>& counts, const EigCtx& cx);
  int eig_block(int est, int cut) const;  // Lanczos block of a pencil that wants est pairs
  int sylvester_estimate(SubdomainState& s, int neg, int perturbedS, bool tauPb, int cut);
  void assemble_z(SubdomainState& s, std::vector<double>& vals, std::vector<DevBuf<double>>& vecs, std::vector<int>& counts, cudaStream_t zs);
  void account_subdomain(const SubdomainState& s);
  double local_gamma(const SubdomainState& s) const;
  struct Lane;
  std::vector<std::unique_ptr<struct GroupSolver>> groupSolvers;  // lock-step block solves of the pencils of a lane group
  std::vector<std::unique_ptr<Lane>> lanes;  // streams + workspaces of the pipelined numeric setup, kept between re-setups
  void build_coarse();
  void level1(const double* xin, double* yout, bool addQ);
  SolveForest forest;
  // workspaces kept between (re-)setups: update arenas + transient factor, block-Lanczos buffers (-geneo_release_workspace frees them)
  LdltWorkspace factorWs;
  EigWorkspace eigWs;
  std::vector<char> connectivity;  // nbPart x nbPart: 1 when the intersection of two subdomains is EMPTY (src/geneo.cpp:1143-1145)
  std::vector<cudaEvent_t> ktEvents;  // kernelTiming: pairs
  size_t ktUsed = 0;
  DevBuf<double> Xall, Yall, w, w2, Einv, t1, t2, t3, scal;
  DevBuf<int> gidxAll;
  DevBuf<double> dAll;
  DevBuf<int64_t> pullPtr, pullPos;
  int64_t nAll = 0;
  // row-major 8-column blocks of the block apply, allocated on the first block call and kept (re-sized when a setup changes
  // nAll / nLoc): the caller's columns in and out (bIn, bOut), the hybrid variants' intermediates (bT1, bT2), the
  // concatenated subdomain blocks (bXall, bYall), the coarse vectors Z^T X and E^-1 Z^T X (bW, bW2)
  DevBuf<double> bIn, bOut, bT1, bT2, bXall, bYall, bW, bW2;
  void ensure_block();
  void level1_8(double* x, double* y, bool addQ);  // x, y: nLoc x 8; the ghost rows of x are refreshed
  void applyQ8(double* x, double* y);               // y may be x
  void apply8(double* x, double* y);                // y != x
  void mult8(double* x, double* y);                 // owned rows of y = A x
  void mult_sub8(double* x, const double* b, double* y);  // owned rows of y = b - A x
  void coarse8();                                    // bW2 = E^-1 Z^T bXall (nE x 8, allreduced over the ranks)
  void cg8(const double* b, double* x, unsigned active, double rtol, double atol, double dtol, int maxIt, KspResult* res);
  std::vector<cudaStream_t> streams;
  std::vector<cudaEvent_t> events;
  cudaEvent_t evFork = nullptr;
};

// host-only test hook (geneo.cu): per-subdomain host preparation of a symmetric CSR matrix, stage stopwatches + digest
void host_prepare_probe(int n, const int64_t* ptr, const int* idx, const double* val, const int* userPerm, int nb, int helper,
                        double seconds[4], uint64_t* digest, double* scatterOut, int64_t scatterLen);

}  // namespace geneo
