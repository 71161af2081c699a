// ldlt.hpp -- device-resident block LDL^T multifrontal factorization + solves (replaces MUMPS LU/Cholesky:
// reference call sites src/geneo.cpp:94-124, 452-500, 766-776, 1044-1066; solve phase :1995, :1486-1493).
#pragma once
#include <memory>
#include "common.hpp"
#include "symbolic.hpp"

namespace geneo {

struct FrontDev {  // device copy of what the kernels need from symbolic.hpp:Front
  int64_t lOff, uOff, wOff, rowOff, relOff;
  int k, h, ld, parent, nchild;
  int uLd, uArena, inplace, pair;
};
struct UArenas { double* a[3]; };  // ping-pong arenas 0/1 + chain arena 2 (Front::uArena)

struct WorkItem { int f, a, b; };
class SolveForest;

// Pattern-level object: symbolic analysis + device work lists.  Shared by every numeric factorization that uses
// the same sparsity pattern (A_dir, A_neu expanded to the A_dir pattern, A_neu - tau*B).
class LdltPlan {
 public:
  LdltPlan(int n, const int64_t* ptr, const int* idx, const SymbolicOptions& opt);
  explicit LdltPlan(Symbolic&& s);  // symbolic analysis done elsewhere (e.g. on a host worker thread)
  struct HostOnly {};
  LdltPlan(Symbolic&& s, HostOnly);  // work lists built too, but nothing uploaded: no CUDA call (worker threads); then upload()
  void upload();
  Symbolic sym;
  // device-resident schedule
  DevBuf<FrontDev> dFronts;
  DevBuf<int> dRowIdx, dRel;
  DevBuf<int64_t> dAsmSrc, dAsmDst;
  DevBuf<WorkItem> dItems;  // all item lists, concatenated
  struct Range { int64_t off = 0; int cnt = 0; };
  std::vector<Range> eaddItems, diagItems, diagSmallItems, copyItems, panelItems, schurItems;  // per level (factor)
  std::vector<Range> schur2Items;  // per level: trailing updates of the second panels of chain pairs (K = two panels)
  std::vector<int64_t> levelU;                                                 // doubles of the ping-pong arena used per level
  std::vector<std::vector<std::pair<int64_t, int64_t>>> levelChainZero;        // (offset, doubles) of the chain blocks born at a level
  DevBuf<int> dPerm;                                                           // new -> old
  size_t plan_bytes() const;
  // single-factor solve forest (eigen-solver, coarse operator): a property of the PATTERN, built once and shared by
  // every numeric factor of this plan (the transient factors of a re-setup reuse it: no item lists are rebuilt)
  mutable std::shared_ptr<SolveForest> selfForest;
  mutable const double* selfL = nullptr;
 private:
  void build_device();
  void build_host();
  std::vector<FrontDev> hostFronts_;
  std::vector<WorkItem> hostItems_;
};

// ---- level-scheduled solves over a forest of factors (one persistent cooperative kernel) -----------------------------
struct ForestSub { const double* L; const FrontDev* fronts; const int* rowIdx; int64_t xoff; };
// item of the ring-buffered NR = 1 kernel (48 bytes): lOff / rowOff point at the tile origin (row r0, column c0) of the
// panel and at rowIdx[r0]; nrows x nc is the extent of the item; the first kdiag rows are pivot rows (forward: D^-1 rows
// that go to Y[ydiag + i]; backward: masked); xcol = first pivot column of the item in the subdomain's permuted numbering
struct RingItem { int64_t lOff, rowOff; int sub, ld, nrows, nc, kdiag, xcol, ydiag, pad; };
class SolveForest {
 public:
  // plans[s] solves rows [xoff[s], xoff[s]+n_s) of the concatenated (permuted) vectors
  void build(const std::vector<const LdltPlan*>& plans, const std::vector<int64_t>& xoff);
  void set_factors(const std::vector<const double*>& L, cudaStream_t st);
  // X (forward sweep, overwritten) -> Y (result); row-major blocks with leading dimension ldx, columns j0..j0+nr-1;
  // nr = 8 or 16, or nr = 1 with ldx = 1
  void solve(double* X, double* Y, int ldx, int j0, int nr, cudaStream_t st) const;
  // NR = 1 solve with a device timestamp after every level barrier: us[p] = duration of phase p (forward levels bottom-up,
  // then backward levels top-down), bytes[p] = factor bytes streamed in it, nitems[p] = ring items
  void solve_profile(double* X, double* Y, int nr, std::vector<double>& us, std::vector<double>& bytes, std::vector<int64_t>& nitems) const;
  int nlev = 0;
  int64_t ntot = 0;
 private:
  void build_ring(int which) const;  // which = 0: NR = 1 item lists, 1: NR = 8 (built on first use)
  std::vector<const LdltPlan*> plans_;
  std::vector<int64_t> xoff_;
  std::vector<ForestSub> hSubs;
  DevBuf<ForestSub> dSubs;
  // ring kernels (NR = 1 and NR = 8): their own item lists (spans chosen per level) and ranges, built on first use
  mutable DevBuf<RingItem> dRing[2];
  mutable DevBuf<int64_t> dRingRanges[2];
  mutable std::vector<double> ringBytes_[2];  // per phase (2 * nlev)
  mutable std::vector<int64_t> ringCount_[2];
  mutable bool ringBuilt[2] = {false, false};
  int ringGrid[2] = {1, 1};
};

struct FactorStats { int neg = 0, perturbed = 0; double seconds = 0.; };

// Shared scratch for numeric factorizations (two ping-pong update arenas + the per-level panel scratch).
struct LdltWorkspace {
  DevBuf<double> u0, u1, uc;     // ping-pong update arenas, chain arena
  DevBuf<double> w0, w1;         // per-level scratch of the unscaled panels, by level parity (a chain pair reads the previous level's)
  DevBuf<double> spareL;  // storage of the transient factors (inertia / shift-invert), recycled between subdomains
  DevBuf<int> counters;  // [0] negative pivots, [1] perturbed pivots
  void ensure(const Symbolic& s);
};

class LdltFactor {
 public:
  explicit LdltFactor(std::shared_ptr<LdltPlan> plan) : plan_(plan) {}
  // vals: device array aligned with the plan's input CSR pattern.  pivTol: a |pivot| below it is a null pivot, fixed to 1e34 pivTol (MUMPS CNTL(5) semantics).
  FactorStats factorize(const double* dVals, double pivTol, LdltWorkspace& ws, cudaStream_t st);
  // Solve in the PERMUTED ordering: X (n x ldx row-major block, columns j0..j0+nr-1) is overwritten by the forward
  // sweep, the result lands in Y (same layout).  nr in {8, 16}, or nr = 1 with ldx = 1.
  void solve_permuted(double* X, double* Y, int ldx, int j0, int nr, cudaStream_t st) const;
  const LdltPlan& plan() const { return *plan_; }
  std::shared_ptr<LdltPlan> plan_ptr() const { return plan_; }
  DevBuf<double> L;
  void release() { if (plan_->selfL == L.p) plan_->selfL = nullptr; L.release(); }
 private:
  std::shared_ptr<LdltPlan> plan_;
};

// One numeric factorization to be enqueued: F->L receives the factor of `vals` (device array aligned with the plan's input
// pattern); everything runs on `st` with the scratch of `ws`.  hostCounters (2 ints, ideally pinned: {negative, perturbed
// pivots}) are written when the stream reaches the end of the job -- nothing here synchronises.
struct FactorJob {
  LdltFactor* F = nullptr;
  const double* vals = nullptr;
  double pivTol = 0.;
  LdltWorkspace* ws = nullptr;
  cudaStream_t st = 0;
  int* hostCounters = nullptr;
};
// Enqueue several INDEPENDENT factorizations, level by level round-robin over the jobs (levels aligned at the roots, where
// the long serial chains of big fronts are), each job on its own stream with its own workspace: the device overlaps the
// latency-bound kernels of one job (pivot-block inversions, small levels, launch tails) with the DMMA tiles of the others.
// Two jobs may share stream + workspace (they then simply run back to back).  Launch only: no host synchronisation.
void factorize_enqueue(std::vector<FactorJob>& jobs);

double solve_stream_bench(int nf, int h, int k, int reps, double* gbps, int nlev = 1, int nr = 1);  // ms per solve; synthetic one-level forest

// DGEMM self-test hooks (microbenchmarks / parity tests of the DMMA tile kernel).
void dgemm_nt_device(int M, int N, int K, const double* A, int lda, const double* B, int ldb, double* C, int ldc,
                     int mode /*0: C=AB^T, 1: C-=AB^T*/, cudaStream_t st);

}  // namespace geneo
