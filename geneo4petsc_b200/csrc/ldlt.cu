// ldlt.cu -- numeric block LDL^T multifrontal factorization and level-scheduled solves on sm_100a.
//
// Factorization kernels (all batched over one schedule level, work lists precomputed on the host, see symbolic.hpp):
//   k_assemble      scatter the input CSR values (lower triangle, permuted) into the panels
//   k_extend_add    child update matrix -> parent panel / parent update matrix (relative indices); along a supernode chain
//                   only the parent's panel columns: the update matrix itself stays in place (Front::inplace)
//   k_diag_invert   one CTA per front: symmetric sweep inversion of the k x k pivot block held in REGISTERS
//                   (8x8 per thread, 256 threads), pivot signs give the inertia (Sylvester, src/geneo.cpp:452-500)
//   k_copy_panel    W = F21 (unscaled panel, needed by the Schur product)
//   k_panel / k_schur / k_schur2   64x64 tiles of  L21 = W * D^-1 ,  U -= L21 * W^T  and (second panel of a chain pair)
//                   U -= [L21_prev | L21] [W_prev | W]^T  on the FP64 tensor pipe (mma.sync.m8n8k4.f64 -- FP64 has no
//                   tcgen05 path), operands global -> shared with cp.async, double-buffered, 5 CTAs per SM
// Solve kernels:
//   k_solve_ring<1 | 8 | 16>   ONE persistent cooperative launch per solve over a forest of factors; the factor tiles stream
//                   through warp-private cp.async rings that run ahead of the arithmetic across items and level barriers
//                   (HBM-bound by design); 8 / 16 right-hand sides use DMMA fragments
#include "ldlt.hpp"

#include <cooperative_groups.h>

#include <algorithm>

namespace geneo {
namespace cg = cooperative_groups;

// =====================================================================================================================
// DMMA 64x64 tile:  C (+)= A * B^T,  A: M x K (col-major, lda), B: N x K (col-major, ldb), C: M x N (col-major, ldc)
// =====================================================================================================================
namespace {

constexpr int TS = 64;     // tile edge
constexpr int KC = 16;     // K chunk per stage
constexpr int SLD = 68;    // padded smem leading dimension (conflict-free 64-bit fragment loads)
constexpr int GEMM_THREADS = 128;
// cp.async pipeline depth of the DMMA tile kernels: 2 stages allow 5 CTAs per SM, 3 only 4 -- measured: 27.1 vs 24.6
// TFLOP/s on the rank-128 update, occupancy beats depth
constexpr int GEMM_STAGES = 2;

__device__ __forceinline__ void dmma8x8x4(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

constexpr int GEMM_SMEM = GEMM_STAGES * 2 * KC * SLD * 8;  // bytes of dynamic shared memory per CTA
static_assert(GEMM_SMEM <= 48 * 1024, "the tile kernels launch without raising their dynamic shared memory limit");

// 8-byte asynchronous copy global -> shared; srcBytes = 0 zero-fills (rows / columns outside the matrix)
__device__ __forceinline__ void cp_async8(double* smem, const double* gmem, int srcBytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem), "r"(srcBytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit_g() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_g() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// C (+)= A B^T on one 64x64 tile.  All 128 threads of the CTA call this with identical arguments.  The operands travel
// global -> shared with cp.async through a GEMM_STAGES-deep ring (no register staging: 4-5 CTAs per SM keep the DMMA pipe
// fed while another CTA is in its prologue or read-modify-writing its C tile); one __syncthreads per K chunk.
// The K dimension may come in TWO segments (A | A2)(B | B2)^T with their own leading dimensions (K2 = 0: one segment): the
// rank-256 trailing update of a chain pair multiplies the panels of two consecutive fronts in one pass over the C tile.
__device__ void gemm_tile_nt(const double* __restrict__ A, int lda, int M, const double* __restrict__ B, int ldb,
                             int N, int K, double* __restrict__ C, int ldc, int mode, double* smem,
                             const double* __restrict__ A2 = nullptr, int lda2 = 0, const double* __restrict__ B2 = nullptr,
                             int ldb2 = 0, int K2 = 0) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp & 1, wn = warp >> 1;
  const int lr = tid & 63;   // row loaded by this thread
  const int lk = tid >> 6;   // first k column loaded by this thread (0/1), stride 2
  if (mode == 1) {  // the C tile is read-modify-written at the very end: pull it into L2 now, behind the whole product
    const int col = tid >> 1;
    if (col < N) {
      const double* cp = C + (size_t)col * ldc + (tid & 1) * 32;
      if ((tid & 1) * 32 < M) asm volatile("prefetch.global.L2 [%0];" ::"l"(cp));
      if ((tid & 1) * 32 + 16 < M) asm volatile("prefetch.global.L2 [%0];" ::"l"(cp + 16));
    }
  }
  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.;

  const int nch1 = (K + KC - 1) / KC;
  const int nch = nch1 + (K2 + KC - 1) / KC;
  const bool aok = lr < M, bok = lr < N;
  auto issue = [&](int ch) {  // chunk ch -> stage ch % GEMM_STAGES
    double* a = smem + (ch % GEMM_STAGES) * (2 * KC * SLD);
    double* b = a + KC * SLD;
    const bool seg2 = ch >= nch1;
    const double* Ar = (seg2 ? A2 : A) + (aok ? lr : 0);
    const double* Br = (seg2 ? B2 : B) + (bok ? lr : 0);
    const int la = seg2 ? lda2 : lda, lb = seg2 ? ldb2 : ldb, Ks = seg2 ? K2 : K, k0 = (seg2 ? ch - nch1 : ch) * KC;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int kl = lk + 2 * i, kk = k0 + kl;
      const bool kok = kk < Ks;
      cp_async8(a + kl * SLD + lr, Ar + (size_t)(kok ? kk : 0) * la, (aok && kok) ? 8 : 0);
      cp_async8(b + kl * SLD + lr, Br + (size_t)(kok ? kk : 0) * lb, (bok && kok) ? 8 : 0);
    }
  };
#pragma unroll
  for (int s = 0; s < GEMM_STAGES - 1; s++) {
    if (s < nch) issue(s);
    cp_async_commit_g();
  }
  for (int ch = 0; ch < nch; ch++) {
    cp_async_wait_g<GEMM_STAGES - 2>();  // chunk ch has landed (this thread's copies) ...
    __syncthreads();                     // ... everybody's; and everybody is done with the stage refilled below
    if (ch + GEMM_STAGES - 1 < nch) issue(ch + GEMM_STAGES - 1);
    cp_async_commit_g();
    const double* a = smem + (ch % GEMM_STAGES) * (2 * KC * SLD);
    const double* b = a + KC * SLD;
#pragma unroll
    for (int k4 = 0; k4 < KC / 4; k4++) {
      double fa[4], fb[4];
      const int krow = (k4 * 4 + (lane & 3)) * SLD;
#pragma unroll
      for (int i = 0; i < 4; i++) {
        fa[i] = a[krow + wm * 32 + i * 8 + (lane >> 2)];
        fb[i] = b[krow + wn * 32 + i * 8 + (lane >> 2)];
      }
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) dmma8x8x4(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
    }
  }
  cp_async_wait_g<0>();
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int row = wm * 32 + i * 8 + (lane >> 2);
      const int col = wn * 32 + j * 8 + 2 * (lane & 3);
      if (row < M) {
#pragma unroll
        for (int e = 0; e < 2; e++)
          if (col + e < N) {
            double* p = C + row + (size_t)(col + e) * ldc;
            if (mode == 0) *p = acc[i][j][e];
            else *p -= acc[i][j][e];
          }
      }
    }
}

__global__ void __launch_bounds__(GEMM_THREADS) k_dgemm_nt(int M, int N, int K, const double* A, int lda,
                                                           const double* B, int ldb, double* C, int ldc, int mode) {
  extern __shared__ __align__(16) double gsm[];
  const int ti = blockIdx.x, tj = blockIdx.y;
  gemm_tile_nt(A + ti * TS, lda, min(TS, M - ti * TS), B + tj * TS, ldb, min(TS, N - tj * TS), K,
               C + ti * TS + (size_t)tj * TS * ldc, ldc, mode, gsm);
}

// =====================================================================================================================
// Factorization kernels
// =====================================================================================================================
__global__ void k_assemble(int64_t cnt, const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                           const double* __restrict__ vals, double* __restrict__ L) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < cnt; t += (int64_t)gridDim.x * blockDim.x)
    L[dst[t]] = vals[src[t]];
}

constexpr int EADD_COLS = 8;     // columns per item: 8 independent loads / updates in flight per thread
constexpr int EADD_ROWS = 256;   // one row per thread
__global__ void __launch_bounds__(256) k_extend_add(const WorkItem* __restrict__ items, const FrontDev* __restrict__ fr,
                                                    const int* __restrict__ relArr, double* __restrict__ L, UArenas ua) {
  const WorkItem it = items[blockIdx.x];
  const FrontDev F = fr[it.f];
  const FrontDev P = fr[F.parent];
  const int m = F.h - F.k, pk = P.k, ph = P.ld;
  const int r = it.b * EADD_ROWS + threadIdx.x;
  const int c0 = it.a * EADD_COLS;
  if (r >= m || r < c0) return;  // lower triangle of the child's update matrix
  const int cld = F.uLd, pld = P.uLd;
  const double* Uc = ua.a[F.uArena] + F.uOff + r + (size_t)c0 * cld;
  double* Up = ua.a[P.uArena] + P.uOff;
  double* Lp = L + P.lOff;
  const int* rel = F.relOff >= 0 ? relArr + F.relOff : nullptr;
  const bool atomic = P.nchild > 1;
  const bool panelOnly = P.inplace != 0;  // the parent's update matrix IS the trailing block of this one: nothing to move
  const int pr = rel ? rel[r] : r;
  const int nc = min(EADD_COLS, min(m, r + 1) - c0);  // columns c0 .. min(r, m-1)
  double v[EADD_COLS];
#pragma unroll
  for (int c = 0; c < EADD_COLS; c++)
    if (c < nc) v[c] = __ldg(Uc + (size_t)c * cld);
#pragma unroll
  for (int c = 0; c < EADD_COLS; c++)
    if (c < nc) {
      const int pc = rel ? rel[c0 + c] : c0 + c;
      if (pc >= pk && panelOnly) continue;
      double* dst = (pc < pk) ? (Lp + pr + (size_t)pc * ph) : (Up + (pr - pk) + (size_t)(pc - pk) * pld);
      if (atomic) atomicAdd(dst, v[c]);
      else *dst += v[c];
    }
}

// One CTA (TD*TD threads) per front.  Thread (ti,tj) owns the strided E x E sub-block i = ti+TD*ii, j = tj+TD*jj of the
// pivot block (padded to KB = TD*E with the identity) in REGISTERS.  Symmetric sweep operator: after sweeping every pivot
// the block holds -F11^-1; the pivots met on the way are the D of the LDL^T factorization (their signs give the
// inertia).  Per pivot every element gets ONE fused multiply-add (a -= c_i * (c_j / d)); the pivot row and column are
// patched afterwards by the few threads that own them.  <128,16>: k <= 128, 256 threads; <32,8>: k <= 32, 64 threads
// (small fronts are the vast majority: many of them are resident per SM).
template <int KB, int TD>
__global__ void __launch_bounds__(TD * TD) k_diag_invert(const WorkItem* __restrict__ items, const FrontDev* __restrict__ fr,
                                                        double* __restrict__ L, double pivTol, int* __restrict__ counters) {
  constexpr int E = KB / TD;
  __shared__ double cbuf[2][KB];
  const WorkItem it = items[blockIdx.x];
  const FrontDev F = fr[it.f];
  const int k = F.k, h = F.ld;
  double* P = L + F.lOff;
  const int ti = threadIdx.x % TD, tj = threadIdx.x / TD;
  double a[E][E];
#pragma unroll
  for (int ii = 0; ii < E; ii++)
#pragma unroll
    for (int jj = 0; jj < E; jj++) {
      const int i = ti + TD * ii, j = tj + TD * jj;
      double v = (i == j) ? 1. : 0.;
      if (i < k && j < k) v = (i >= j) ? P[i + (size_t)j * h] : P[j + (size_t)i * h];
      a[ii][jj] = v;
    }
  if (tj == 0) {  // publish column 0
#pragma unroll
    for (int ii = 0; ii < E; ii++) cbuf[0][ti + TD * ii] = a[ii][0];
  }
  __syncthreads();
  int neg = 0, pert = 0;
  for (int p = 0; p < k; p++) {
    const double* cb = cbuf[p & 1];
    double d = cb[p];
    // Null pivot (|d| < pivTol = 1e-14 max|a_ij|): fixed to a HUGE positive value, 1e20 max|a_ij| -- the semantics of MUMPS
    // ICNTL(24) = 1 with CNTL(5) = 1e20, which the reference sets for every local solver (src/geneo.cpp:81-83): the
    // corresponding solution component becomes 0 (a floating subdomain's constant mode is then supplied by the Nicolaides
    // rule, src/geneo.cpp:897-944, instead of appearing twice).  Counted apart, neither negative nor positive (MUMPS INFOG(28)).
    if (!(fabs(d) >= pivTol)) { d = pivTol * 1e34; pert++; }
    else if (d < 0.) neg++;
    const double rinv = 1. / d;
    double ci[E], cjr[E];
#pragma unroll
    for (int q = 0; q < E; q++) { ci[q] = cb[ti + TD * q]; cjr[q] = cb[tj + TD * q] * rinv; }
#pragma unroll
    for (int ii = 0; ii < E; ii++)
#pragma unroll
      for (int jj = 0; jj < E; jj++) a[ii][jj] = fma(-ci[ii], cjr[jj], a[ii][jj]);
    const int pt = p % TD, pq = p / TD;
    if (ti == pt) {  // row p: a[p][j] = c_j / d  (and the pivot itself: -1/d)
#pragma unroll
      for (int ii = 0; ii < E; ii++)
        if (ii == pq) {
#pragma unroll
          for (int jj = 0; jj < E; jj++) a[ii][jj] = (tj + TD * jj == p) ? -rinv : cjr[jj];
        }
    }
    if (tj == pt) {  // column p: a[i][p] = c_i / d
#pragma unroll
      for (int jj = 0; jj < E; jj++)
        if (jj == pq) {
#pragma unroll
          for (int ii = 0; ii < E; ii++) a[ii][jj] = (ti + TD * ii == p) ? -rinv : ci[ii] * rinv;
        }
    }
    // publish column p+1 for the next sweep
    const int pn = p + 1;
    if (pn < k && tj == pn % TD) {
      double* nb = cbuf[pn & 1];
      const int jn = pn / TD;
#pragma unroll
      for (int ii = 0; ii < E; ii++) {
        double v = 0.;
#pragma unroll
        for (int q = 0; q < E; q++)
          if (q == jn) v = a[ii][q];
        nb[ti + TD * ii] = v;
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int ii = 0; ii < E; ii++)
#pragma unroll
    for (int jj = 0; jj < E; jj++) {
      const int i = ti + TD * ii, j = tj + TD * jj;
      if (i < k && j < k) P[i + (size_t)j * h] = -a[ii][jj];
    }
  if (threadIdx.x == 0 && (neg | pert)) {
    if (neg) atomicAdd(&counters[0], neg);
    if (pert) atomicAdd(&counters[1], pert);
  }
}

constexpr int COPY_ROWS = 256;   // one row per thread
constexpr int COPY_COLS = 16;    // independent loads in flight per thread; a tall thin panel near the root still fills the chip
__global__ void __launch_bounds__(256) k_copy_panel(const WorkItem* __restrict__ items, const FrontDev* __restrict__ fr,
                                                    const double* __restrict__ L, double* __restrict__ W) {
  const WorkItem it = items[blockIdx.x];
  const FrontDev F = fr[it.f];
  const int m = F.h - F.k, k = F.k, h = F.ld;
  const int r = it.a * COPY_ROWS + threadIdx.x;
  if (r >= m) return;
  const int c0 = it.b * COPY_COLS;
  const double* src = L + F.lOff + k + r + (size_t)c0 * h;
  double* dst = W + F.wOff + r + (size_t)c0 * m;
  double v[COPY_COLS];
#pragma unroll
  for (int c = 0; c < COPY_COLS; c++)
    if (c0 + c < k) v[c] = __ldg(src + (size_t)c * h);
#pragma unroll
  for (int c = 0; c < COPY_COLS; c++)
    if (c0 + c < k) dst[(size_t)c * m] = v[c];
}

__global__ void __launch_bounds__(GEMM_THREADS) k_panel(const WorkItem* __restrict__ items,
                                                        const FrontDev* __restrict__ fr, double* __restrict__ L,
                                                        const double* __restrict__ W) {
  extern __shared__ __align__(16) double gsm[];
  const WorkItem it = items[blockIdx.x];
  const FrontDev F = fr[it.f];
  const int m = F.h - F.k, k = F.k, h = F.ld;
  double* P = L + F.lOff;
  // L21[ti rows, tj cols] = W[ti rows, :] * Dinv[tj rows, :]^T   (Dinv symmetric)
  gemm_tile_nt(W + F.wOff + it.a * TS, m, min(TS, m - it.a * TS), P + it.b * TS, h, min(TS, k - it.b * TS), k,
               P + k + it.a * TS + (size_t)it.b * TS * h, h, 0, gsm);
}

__global__ void __launch_bounds__(GEMM_THREADS, 5) k_schur(const WorkItem* __restrict__ items,
                                                        const FrontDev* __restrict__ fr, const double* __restrict__ L,
                                                        const double* __restrict__ W, UArenas ua) {
  extern __shared__ __align__(16) double gsm[];
  const WorkItem it = items[blockIdx.x];
  const FrontDev F = fr[it.f];
  const int m = F.h - F.k, k = F.k, h = F.ld;
  // first panel of a chain pair: EXACTLY the columns the next panel assembles (its k' pivot columns, not rounded up to the
  // tile: the rank-256 update of the next level covers everything from column k' on)
  const int ncols = F.pair == 1 ? min(m, fr[it.f + 1].k) : m;
  // U[ti, tj] -= L21[ti rows, :] * W[tj rows, :]^T   (lower triangle of tiles only)
  gemm_tile_nt(L + F.lOff + k + it.a * TS, h, min(TS, m - it.a * TS), W + F.wOff + it.b * TS, m,
               min(TS, ncols - it.b * TS), k, ua.a[F.uArena] + F.uOff + it.a * TS + (size_t)it.b * TS * F.uLd, F.uLd, 1, gsm);
}

// Second panel of a chain pair: U -= [L21_prev(rows below this panel's pivots) | L21] [W_prev(same rows) | W]^T, K = k_prev + k.
// The first panel of the pair only updated the strip of U this panel assembled (its own k pivot columns).
__global__ void __launch_bounds__(GEMM_THREADS, 5) k_schur2(const WorkItem* __restrict__ items, const FrontDev* __restrict__ fr,
                                                         const double* __restrict__ L, const double* __restrict__ Wcur,
                                                         const double* __restrict__ Wprev, UArenas ua) {
  extern __shared__ __align__(16) double gsm[];
  const WorkItem it = items[blockIdx.x];
  const FrontDev F = fr[it.f];
  const FrontDev Pf = fr[it.f - 1];
  const int m = F.h - F.k, k = F.k, pm = Pf.h - Pf.k;
  gemm_tile_nt(L + Pf.lOff + Pf.k + k + it.a * TS, Pf.ld, min(TS, m - it.a * TS), Wprev + Pf.wOff + k + it.b * TS, pm,
               min(TS, m - it.b * TS), Pf.k, ua.a[F.uArena] + F.uOff + it.a * TS + (size_t)it.b * TS * F.uLd, F.uLd, 1, gsm,
               L + F.lOff + k + it.a * TS, F.ld, Wcur + F.wOff + it.b * TS, m, k);
}

// =====================================================================================================================
// Solve: ONE persistent cooperative kernel per solve over a FOREST of factors (all local subdomains at once).
//
//   forward + diagonal (fused):  [ y1 ; x2 ] (+,-)= P[:, c0:c1] * x1[c0:c1]   over ALL h rows of the panel: the first k rows
//                                are D^-1 (-> Y += ...), the rest are L21 (-> X[rows] -= ...): one uniform GEMV stream.
//   backward:                    y1[c0:c1] -= L21[:, c0:c1]^T * y2
//
// Levels are separated by grid-wide barriers instead of kernel launches: one launch and 2*levels barriers per solve.
// =====================================================================================================================
constexpr int MAX_SMEM_SUBS = 64;

// ---------------------------------------------------------------------------------------------------------------------
// Ring-buffered streaming solve: NR = 1 (the preconditioner application) and NR = 8 (block solves of the eigen-solver
// and of the coarse operator).
//
// The factor does not depend on the sweep (only x / y do), so its tiles are moved by cp.async into a warp-private ring
// of shared-memory stages that runs AHEAD of the arithmetic -- across item boundaries and across the grid barriers that
// separate the levels.  HBM keeps streaming while a level drains, while the barrier is in flight and while the first x / y
// values of the next level are fetched from L2; the barrier only gates the consumption of a stage, never its transfer.
//
//   item (RingItem)  forward : 64 rows x nc columns (nc <= 128: a span of 32-column groups chosen per level on the host)
//                    backward: up to 512 rows x nc <= 16 (NR = 1) / 32 (NR = 8) columns (row span chosen per level)
//   chunk            64 rows x 8 columns = one ring stage: 8 x 16-byte cp.async per lane (4 KB per warp) plus the 64 row
//                    indices of the tile (first column chunk of a row tile only)
//   ring             RING_S stages per warp; RING_S-1 chunks (8 KB) in flight per warp, 128 KB per SM, 19 MB per chip
//                    = the HBM latency-bandwidth product with margin for one barrier
//   schedule         static: item j of phase p belongs to warp (j mod #warps); the producer side of a warp walks the same
//                    sequence RING_S-1 chunks ahead of its consumer side and hands the item records over through a small
//                    shared-memory record ring, so no thread ever waits on an item record.
//   NR = 1           FP64 FMA, x broadcast by shuffles, one butterfly transpose-reduction per backward item
//   NR = 8           the 8 right-hand sides are the N dimension of mma.sync.m8n8k4.f64 (FP64 tensor pipe): forward
//                    C[8 rows x 8 rhs] += L[8 rows x 4 cols] X[4 cols x 8 rhs], backward C[8 cols x 8 rhs] += L^T Y2;
//                    the stage keeps a column stride of 68 doubles so that both fragment reads are bank-conflict free.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int RING_CH = 8;                     // columns per chunk
constexpr int RING_RS = 8;                     // item records in flight per warp (> stages, power of two)
constexpr int RING_MAXPH = 512;                // phases whose (offset, count) are kept in shared memory
template <int W, int STAGES, int CSTRIDE, int BC> struct RingCfgT {
  static constexpr int WARPS = W, S = STAGES, CS = CSTRIDE, BWD_COLS = BC;  // CS: column stride of a stage in doubles
  static constexpr int STAGE = RING_CH * CSTRIDE * 8 + 256;                 // tile + 64 row indices
  static constexpr int WARP_BYTES = STAGES * STAGE + RING_RS * 48;
  static constexpr int SMEM = W * WARP_BYTES;
};
template <int NR> struct RingCfg;
template <> struct RingCfg<1> : RingCfgT<16, 3, 64, 16> {};  // 16 warps x 3 stages: 128 KB in flight per SM, <= 128 registers
template <> struct RingCfg<8> : RingCfgT<12, 4, 68, 32> {};  // 12 warps x 4 stages: 144 KB in flight per SM, <= 168 registers
// NR = 16 walks the item lists of NR = 8 with two DMMAs per L fragment.  8 warps = 2 per SM sub-partition: the register file
// of a sub-partition (16 K registers) then allows 255 registers per thread (10 or 12 warps put 3 on one sub-partition: 168);
// 6 stages keep 160 KB in flight per SM.
template <> struct RingCfg<16> : RingCfgT<8, 6, 68, 32> {};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }
__device__ __forceinline__ long long gtimer() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }

// a RingItem travels as three int4: a = {lOff, rowOff}, b = {sub, ld, nrows, nc}, c = {kdiag, xcol, ydiag, pad}
struct RingRec { int4 a, b, c; };
__device__ __forceinline__ RingRec load_ring_item(const RingItem* p) {
  const int4* q = reinterpret_cast<const int4*>(p);
  RingRec r;
  r.a = __ldg(q); r.b = __ldg(q + 1); r.c = __ldg(q + 2);
  return r;
}
__device__ __forceinline__ int64_t rec_i64(int lo, int hi) { return (int64_t)(((unsigned long long)(unsigned)hi << 32) | (unsigned)lo); }

template <int NR>
__global__ void __launch_bounds__(RingCfg<NR>::WARPS * 32, 1)
k_solve_ring(const ForestSub* __restrict__ subs, int nsubs, const RingItem* __restrict__ items,
             const int64_t* __restrict__ ranges, int nlev, int64_t ntot, double* __restrict__ X, double* __restrict__ Y,
             int ldx, long long* __restrict__ tstamp) {
  constexpr int CS = RingCfg<NR>::CS;
  constexpr int RING_S = RingCfg<NR>::S;
  constexpr int TILE_BYTES = RING_CH * CS * 8;
  constexpr int STAGE = RingCfg<NR>::STAGE;
  constexpr int BWD_COLS = RingCfg<NR>::BWD_COLS;
  cg::grid_group grid = cg::this_grid();
  extern __shared__ __align__(16) unsigned char ringmem[];
  __shared__ ForestSub sSubs[MAX_SMEM_SUBS];
  __shared__ unsigned sOff[RING_MAXPH];  // item lists are far below 2^32 records
  __shared__ int sCnt[RING_MAXPH];
  const int nph = 2 * nlev;
  const bool phSmem = nph <= RING_MAXPH;
  for (int t = threadIdx.x; t < min(nsubs, MAX_SMEM_SUBS); t += blockDim.x) sSubs[t] = subs[t];
  if (phSmem)
    for (int p = threadIdx.x; p < nph; p += blockDim.x) {  // phases 0..nlev-1 forward (level p), then backward from the root
      const bool b = p >= nlev;
      const int l = b ? (2 * nlev - 1 - p) : p;
      sOff[p] = (unsigned)ranges[(b ? 2 * nlev : 0) + l];
      sCnt[p] = (int)ranges[(b ? 3 * nlev : nlev) + l];
    }
  if (NR > 1)  // fragments read whole stages: never let a NaN pattern of uninitialised shared memory into a product
    for (int t = threadIdx.x; t < RingCfg<NR>::SMEM / 16; t += blockDim.x) reinterpret_cast<int4*>(ringmem)[t] = make_int4(0, 0, 0, 0);
  const bool inSmem = nsubs <= MAX_SMEM_SUBS;
  const int lane = threadIdx.x & 31;
  unsigned char* wmem = ringmem + (threadIdx.x >> 5) * RingCfg<NR>::WARP_BYTES;
  int4* recRing = reinterpret_cast<int4*>(wmem + RING_S * STAGE);
  // consecutive items of a phase go to different SMs: a level with few items still uses every SM's LSU / L1 / RED path
  const int64_t gw = (int64_t)(threadIdx.x >> 5) * gridDim.x + blockIdx.x;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < ntot * NR; t += (int64_t)gridDim.x * blockDim.x)
    Y[(t / NR) * ldx + (t % NR)] = 0.;
  __syncthreads();
  auto phase_range = [&](int p, int64_t& off, int64_t& cnt) {
    if (phSmem) { off = sOff[p]; cnt = sCnt[p]; return; }
    const bool b = p >= nlev;
    const int l = b ? (2 * nlev - 1 - p) : p;
    off = __ldg(ranges + (b ? 2 * nlev : 0) + l);
    cnt = __ldg(ranges + (b ? 3 * nlev : nlev) + l);
  };

  // ---------------- producer side (warp-uniform state) ----------------
  int pp = 0;             // phase of the next record to fetch
  int64_t pi = gw;        // index of that record inside its phase
  RingRec nrec;           // fetched ahead
  bool nvalid = false;
  auto fetch_next = [&](int budget) {  // looks at no more than `budget` phases: never a long scan on somebody's critical path
    while (pp < nph && budget-- > 0) {
      int64_t off, cnt;
      phase_range(pp, off, cnt);
      if (pi < cnt) {
        nrec = load_ring_item(items + off + pi);
        nvalid = true;
        pi += nw;
        return;
      }
      pp++;
      pi = gw;
    }
  };
  const double* psrc = nullptr;  // per lane: first element of this lane's two rows in the current column chunk
  const int* pidx = nullptr;
  int pld = 0, pnrows = 0, pnc = 0, pQ = 1, pT = 0, pt = 0, pcq = 0;
  bool pactive = false;
  unsigned pm = 0;              // records handed over so far
  unsigned pcount = 0;          // chunks produced so far
  unsigned ccount = 0;          // chunks consumed so far
  int pstage = 0, cstage = 0;   // = pcount % RING_S, ccount % RING_S
  auto top_up = [&]() {         // keep the ring full: RING_S stages in use, the current one included
    while (pcount - ccount < RING_S) {
      if (!pactive) {
        if (!nvalid) { fetch_next(8); if (!nvalid) break; }
        const ForestSub& S = inSmem ? sSubs[nrec.b.x] : subs[nrec.b.x];
        psrc = S.L + rec_i64(nrec.a.x, nrec.a.y);
        pidx = S.rowIdx + rec_i64(nrec.a.z, nrec.a.w);
        pld = nrec.b.y; pnrows = nrec.b.z; pnc = nrec.b.w;
        pQ = (pnc + RING_CH - 1) / RING_CH;
        pT = (pnrows + 63) >> 6;
        pt = 0; pcq = 0;
        pactive = true;
        if (lane < 3) recRing[(pm & (RING_RS - 1)) * 3 + lane] = lane == 0 ? nrec.a : lane == 1 ? nrec.b : nrec.c;
        pm++;
        nvalid = false;
        fetch_next(2);  // the following record travels while this item streams
      }
      unsigned char* st = wmem + pstage * STAGE;
      const int r = pt * 64 + 2 * lane;
      const bool rowok = r < pnrows;
      const double* src = psrc + (size_t)(pcq * RING_CH) * pld + (rowok ? r : 0);
      double* dst = reinterpret_cast<double*>(st) + 2 * lane;
      const int ncc = pnc - pcq * RING_CH;
      if (ncc >= RING_CH) {
#pragma unroll
        for (int u = 0; u < RING_CH; u++) cp_async16(dst + u * CS, src + (size_t)u * pld);
      } else {
#pragma unroll
        for (int u = 0; u < RING_CH - 1; u++)
          if (u < ncc) cp_async16(dst + u * CS, src + (size_t)u * pld);  // warp-uniform predicate
      }
      if (pcq == 0) {
        int* di = reinterpret_cast<int*>(st + TILE_BYTES) + 2 * lane;
        if (rowok) cp_async4(di, pidx + r);
        if (r + 1 < pnrows) cp_async4(di + 1, pidx + r + 1);
      }
      cp_async_commit();
      pcount++;
      pstage = pstage + 1 == RING_S ? 0 : pstage + 1;
      if (++pcq == pQ) { pcq = 0; if (++pt == pT) pactive = false; }
    }
  };
  auto acquire = [&]() -> const unsigned char* {  // next chunk of this warp's stream, landed
    if (NR > 1) __syncwarp();                     // every lane is done with the stage that is about to be refilled
    do top_up(); while (pcount == ccount);
    const unsigned ahead = pcount - ccount - 1;   // groups committed after the one needed now
    if (RING_S > 5 && ahead >= 5) cp_async_wait<5>();
    else if (RING_S > 4 && ahead >= 4) cp_async_wait<4>();
    else if (RING_S > 3 && ahead >= 3) cp_async_wait<3>();
    else if (ahead >= 2) cp_async_wait<2>();
    else if (ahead == 1) cp_async_wait<1>();
    else cp_async_wait<0>();
    if (NR > 1) __syncwarp();                     // fragments read what OTHER lanes copied
    return wmem + cstage * STAGE;
  };
  auto release = [&]() { ccount++; cstage = cstage + 1 == RING_S ? 0 : cstage + 1; };
  top_up();

  // ---------------- consumer side ----------------
  unsigned cm = 0;
  grid.sync();
  if (tstamp && blockIdx.x == 0 && threadIdx.x == 0) tstamp[0] = gtimer();
  for (int p = 0; p < nph; p++) {
    const bool bwd = p >= nlev;
    int64_t off, cnt;
    phase_range(p, off, cnt);
    double xn[NR == 1 ? 4 : 8];  // x1 of the NEXT forward item of this phase, fetched during the last chunk of the current one
    bool havex = false;
    for (int64_t i = gw; i < cnt; i += nw) {
      while (pm == cm) top_up();  // (only after a long idle stretch can a warp find its record not handed over yet)
      __syncwarp();
      const int4* rr = recRing + (cm & (RING_RS - 1)) * 3;
      const int4 rb = rr[1], rc = rr[2];
      cm++;
      const ForestSub& S = inSmem ? sSubs[rb.x] : subs[rb.x];
      const int nc = rb.w, nrows = rb.z, kd = rc.x, xcol = rc.y, ydiag = rc.z;
      const int Q = (nc + RING_CH - 1) / RING_CH;
      if constexpr (NR == 1) {
        if (!bwd) {
          // [ y1 ; x2 ] (+,-)= P[r0:r0+64, c0:c0+nc] * x1
          double xv[4];
          if (havex) {
#pragma unroll
            for (int g = 0; g < 4; g++) xv[g] = xn[g];
          } else {
            const double* x1 = X + (S.xoff + xcol);
#pragma unroll
            for (int g = 0; g < 4; g++) xv[g] = (g * 32 + lane < nc) ? __ldcg(x1 + g * 32 + lane) : 0.;
          }
          havex = false;
          double a0 = 0., a1 = 0.;
          int row0 = 0, row1 = 0;
          for (int q = 0; q < Q; q++) {
            const unsigned char* st = acquire();
            if (q == 0) {
              const int2 ri = *reinterpret_cast<const int2*>(st + TILE_BYTES + 8 * lane);
              row0 = ri.x; row1 = ri.y;
            }
            if (q == Q - 1 && i + nw < cnt) {  // the next item's record has been handed over by now (RING_S >= 2)
              __syncwarp();
              const int4* r2 = recRing + (cm & (RING_RS - 1)) * 3;
              const int4 b2 = r2[1], c2 = r2[2];
              const double* x2 = X + ((inSmem ? sSubs[b2.x] : subs[b2.x]).xoff + c2.y);
#pragma unroll
              for (int g = 0; g < 4; g++) xn[g] = (g * 32 + lane < b2.w) ? __ldcg(x2 + g * 32 + lane) : 0.;
              havex = true;
            }
            const double2* tb = reinterpret_cast<const double2*>(st) + lane;
            const int ncc = nc - q * RING_CH;
            const double xg = (q >> 2) == 0 ? xv[0] : (q >> 2) == 1 ? xv[1] : (q >> 2) == 2 ? xv[2] : xv[3];
            const int cb = (q & 3) * RING_CH;
            if (ncc >= RING_CH) {
#pragma unroll
              for (int u = 0; u < RING_CH; u++) {
                const double2 v = tb[u * 32];
                const double xc = __shfl_sync(0xffffffffu, xg, cb + u);
                a0 += v.x * xc;
                a1 += v.y * xc;
              }
            } else {
#pragma unroll
              for (int u = 0; u < RING_CH - 1; u++)
                if (u < ncc) {
                  const double2 v = tb[u * 32];
                  const double xc = __shfl_sync(0xffffffffu, xg, cb + u);
                  a0 += v.x * xc;
                  a1 += v.y * xc;
                }
            }
            release();
          }
          const int r = 2 * lane;
          if (r < nrows) {
            if (r < kd) atomicAdd(Y + (S.xoff + ydiag + r), a0);
            else atomicAdd(X + (S.xoff + row0), -a0);
          }
          if (r + 1 < nrows) {
            if (r + 1 < kd) atomicAdd(Y + (S.xoff + ydiag + r + 1), a1);
            else atomicAdd(X + (S.xoff + row1), -a1);
          }
        } else {
          // y1[c0:c0+nc] -= L21[rows, c0:c0+nc]^T * y2[rows]      (nc <= 16, rows in tiles of 64)
          double acc[BWD_COLS];
#pragma unroll
          for (int u = 0; u < BWD_COLS; u++) acc[u] = 0.;
          const int T = (nrows + 63) >> 6;
          for (int t = 0; t < T; t++) {
            double y0 = 0., y1 = 0.;
#pragma unroll
            for (int cq = 0; cq < BWD_COLS / RING_CH; cq++) {
              if (cq < Q) {  // warp-uniform
                const unsigned char* st = acquire();
                if (cq == 0) {
                  const int r = t * 64 + 2 * lane;
                  const int2 ri = *reinterpret_cast<const int2*>(st + TILE_BYTES + 8 * lane);
                  if (r >= kd && r < nrows) y0 = __ldcg(Y + (S.xoff + ri.x));
                  if (r + 1 >= kd && r + 1 < nrows) y1 = __ldcg(Y + (S.xoff + ri.y));
                }
                const double2* tb = reinterpret_cast<const double2*>(st) + lane;
                const int ncc = nc - cq * RING_CH;
#pragma unroll
                for (int u = 0; u < RING_CH; u++)
                  if (u < ncc) {
                    const double2 v = tb[u * 32];
                    acc[cq * RING_CH + u] += v.x * y0 + v.y * y1;
                  }
                release();
              }
            }
          }
#pragma unroll
          for (int q = 0; q < BWD_COLS; q++) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], 16);
#pragma unroll
          for (int o = BWD_COLS / 2; o >= 1; o >>= 1) {
            const bool upper = (lane & o) != 0;
#pragma unroll
            for (int i2 = 0; i2 < o; i2++) {
              const double send = upper ? acc[i2] : acc[i2 + o];
              const double keep = upper ? acc[i2 + o] : acc[i2];
              acc[i2] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
          }
          if (lane < BWD_COLS && lane < nc) atomicAdd(&Y[S.xoff + xcol + lane], -acc[0]);
        }
      } else {
        // ---------------- NR = 8 H (H = 1, 2): FP64 tensor-core fragments; lane = 4 g + t ----------------
        constexpr int H = NR / 8;  // groups of 8 right-hand sides: every L fragment read from shared memory feeds H DMMAs
        const int g = lane >> 2, t4 = lane & 3;
        if (!bwd) {
          // C[row rb*8+g][rhs 2 t4 + e] += sum_cols L[row][col] X[col][rhs];  B fragment: X[col 4 ks + t4][rhs g]
          auto load_x = [&](const ForestSub& S2, int xc2, int nc2, int grp, int hh, double (&xf)[8]) {
            const double* xb = X + (size_t)(S2.xoff + xc2 + grp * 32) * ldx + 8 * hh + g;
#pragma unroll
            for (int ks = 0; ks < 8; ks++) {
              const int c = grp * 32 + ks * 4 + t4;
              xf[ks] = c < nc2 ? __ldcg(xb + (size_t)(ks * 4 + t4) * ldx) : 0.;
            }
          };
          double xf[H][8];
          if (H == 1 && havex) {
#pragma unroll
            for (int ks = 0; ks < 8; ks++) xf[0][ks] = xn[ks];
          } else {
#pragma unroll
            for (int hh = 0; hh < H; hh++) load_x(S, xcol, nc, 0, hh, xf[hh]);
          }
          havex = false;
          double acc[H][8][2];
#pragma unroll
          for (int hh = 0; hh < H; hh++)
#pragma unroll
            for (int b8 = 0; b8 < 8; b8++) acc[hh][b8][0] = acc[hh][b8][1] = 0.;
          int ridx[8];
          for (int q = 0; q < Q; q++) {
            if (q > 0 && (q & 3) == 0) {  // next group of 32 columns
#pragma unroll
              for (int hh = 0; hh < H; hh++) load_x(S, xcol, nc, q >> 2, hh, xf[hh]);
            }
            const unsigned char* st = acquire();
            if (q == 0) {
              const int* ip = reinterpret_cast<const int*>(st + TILE_BYTES);
#pragma unroll
              for (int b8 = 0; b8 < 8; b8++) ridx[b8] = ip[b8 * 8 + g];
            }
            if (H == 1 && q == Q - 1 && i + nw < cnt) {
              const int4* r2 = recRing + (cm & (RING_RS - 1)) * 3;
              const int4 b2 = r2[1], c2 = r2[2];
              load_x(inSmem ? sSubs[b2.x] : subs[b2.x], c2.y, b2.w, 0, 0, xn);
              havex = true;
            }
            const double* tb = reinterpret_cast<const double*>(st);
            const int ncc = nc - q * RING_CH;
#pragma unroll
            for (int ks = 0; ks < 2; ks++) {
              const int col = ks * 4 + t4;
              const double* ap = tb + col * CS + g;
              const bool ok = col < ncc;
              double a[8];
#pragma unroll
              for (int b8 = 0; b8 < 8; b8++) a[b8] = ok ? ap[b8 * 8] : 0.;
#pragma unroll
              for (int hh = 0; hh < H; hh++) {
                const double bfrag = (q & 1) ? ((q & 2) ? xf[hh][6 + ks] : xf[hh][2 + ks]) : ((q & 2) ? xf[hh][4 + ks] : xf[hh][ks]);
#pragma unroll
                for (int b8 = 0; b8 < 8; b8++) dmma8x8x4(acc[hh][b8][0], acc[hh][b8][1], a[b8], bfrag);
              }
            }
            release();
          }
#pragma unroll
          for (int b8 = 0; b8 < 8; b8++) {
            const int r = b8 * 8 + g;
            if (r < nrows) {
              double* d = (r < kd) ? Y + (size_t)(S.xoff + ydiag + r) * ldx + 2 * t4 : X + (size_t)(S.xoff + ridx[b8]) * ldx + 2 * t4;
              const double sg = (r < kd) ? 1. : -1.;
#pragma unroll
              for (int hh = 0; hh < H; hh++) {
                atomicAdd(d + 8 * hh, sg * acc[hh][b8][0]);
                atomicAdd(d + 8 * hh + 1, sg * acc[hh][b8][1]);
              }
            }
          }
        } else {
          // C[col cq*8+g][rhs 2 t4 + e] += sum_rows L[row][col] Y2[row][rhs];  A fragment: L[row 4 ks + t4][col g],
          // B fragment: Y2[row 4 ks + t4][rhs g]
          double acc[H][BWD_COLS / 8][2];
#pragma unroll
          for (int hh = 0; hh < H; hh++)
#pragma unroll
            for (int c8 = 0; c8 < BWD_COLS / 8; c8++) acc[hh][c8][0] = acc[hh][c8][1] = 0.;
          const int T = (nrows + 63) >> 6;
          for (int t = 0; t < T; t++) {
            double yf[H][16];
#pragma unroll
            for (int cq = 0; cq < BWD_COLS / RING_CH; cq++) {
              if (cq < Q) {  // warp-uniform
                const unsigned char* st = acquire();
                if (cq == 0) {
                  const int* ip = reinterpret_cast<const int*>(st + TILE_BYTES);
#pragma unroll
                  for (int ks = 0; ks < 16; ks++) {
                    const int r = t * 64 + ks * 4 + t4;
                    const bool ok = r >= kd && r < nrows;
                    const double* yp = Y + (size_t)(S.xoff + (ok ? ip[ks * 4 + t4] : 0)) * ldx + g;
#pragma unroll
                    for (int hh = 0; hh < H; hh++) yf[hh][ks] = ok ? __ldcg(yp + 8 * hh) : 0.;
                  }
                }
                const double* ap = reinterpret_cast<const double*>(st) + g * CS + t4;
#pragma unroll
                for (int ks = 0; ks < 16; ks++) {
                  const double a = ap[ks * 4];
#pragma unroll
                  for (int hh = 0; hh < H; hh++) dmma8x8x4(acc[hh][cq][0], acc[hh][cq][1], a, yf[hh][ks]);
                }
                release();
              }
            }
          }
#pragma unroll
          for (int c8 = 0; c8 < BWD_COLS / 8; c8++) {
            const int c = c8 * 8 + g;
            if (c < nc) {
              double* d = Y + (size_t)(S.xoff + xcol + c) * ldx + 2 * t4;
#pragma unroll
              for (int hh = 0; hh < H; hh++) {
                atomicAdd(d + 8 * hh, -acc[hh][c8][0]);
                atomicAdd(d + 8 * hh + 1, -acc[hh][c8][1]);
              }
            }
          }
        }
      }
    }
    top_up();  // idle warps keep scanning ahead / prefetching here, off everybody's critical path
    if (p + 1 < nph) {
      grid.sync();
      if (tstamp && blockIdx.x == 0 && threadIdx.x == 0) tstamp[p + 1] = gtimer();
    }
  }
  cp_async_wait<0>();
  if (tstamp && blockIdx.x == 0 && threadIdx.x == 0) tstamp[nph] = gtimer();
}

}  // namespace

void dgemm_nt_device(int M, int N, int K, const double* A, int lda, const double* B, int ldb, double* C, int ldc,
                     int mode, cudaStream_t st) {
  dim3 grid((M + TS - 1) / TS, (N + TS - 1) / TS);
  k_dgemm_nt<<<GENEO_TICK(grid), GEMM_THREADS, GEMM_SMEM, st>>>(M, N, K, A, lda, B, ldb, C, ldc, mode);
  CUDA_CHECK(cudaGetLastError());
}

// =====================================================================================================================
// Plan: symbolic + work lists
// =====================================================================================================================
LdltPlan::LdltPlan(int n, const int64_t* ptr, const int* idx, const SymbolicOptions& opt) {
  symbolic_analyze(n, ptr, idx, opt, sym);
  build_device();
}
LdltPlan::LdltPlan(Symbolic&& s) : sym(std::move(s)) { build_device(); }
LdltPlan::LdltPlan(Symbolic&& s, HostOnly) : sym(std::move(s)) { build_host(); }

void LdltPlan::build_device() {
  build_host();
  upload();
}

// work lists of every level (host only: safe on a worker thread, no CUDA call)
void LdltPlan::build_host() {
  const int nf = (int)sym.fronts.size();
  std::vector<FrontDev>& fd = hostFronts_;
  fd.assign(nf, FrontDev());
  for (int f = 0; f < nf; f++) {
    const Front& F = sym.fronts[f];
    fd[f] = FrontDev{F.lOff, F.uOff, F.wOff, F.rowOff, F.relOff, F.k, F.h, F.ld, F.parent, F.nchild, F.uLd, F.uArena, F.inplace, F.pair};
  }
  std::vector<WorkItem>& items = hostItems_;
  items.clear();
  auto begin = [&](Range& r) { r.off = (int64_t)items.size(); };
  auto end = [&](Range& r) { r.cnt = (int)((int64_t)items.size() - r.off); };
  const int nl = sym.nlevels;
  eaddItems.resize(nl); diagItems.resize(nl); diagSmallItems.resize(nl); copyItems.resize(nl); panelItems.resize(nl); schurItems.resize(nl);
  schur2Items.resize(nl);
  levelU.assign(nl, 0);
  levelChainZero.assign(nl, {});
  for (int l = 0; l < nl; l++) {
    const int* lf = &sym.levelFronts[sym.levelPtr[l]];
    const int cnt = sym.levelPtr[l + 1] - sym.levelPtr[l];
    for (int t = 0; t < cnt; t++) {
      const Front& F = sym.fronts[lf[t]];
      const int64_t m = F.m();
      if (m > 0 && !F.inplace) {
        if (F.uArena == 2) levelChainZero[l].emplace_back(F.uOff, m * m);
        else levelU[l] = std::max(levelU[l], F.uOff + m * m);
      }
    }
    // extend-add: children are the fronts of level l-1 (their parents are all at level l)
    begin(eaddItems[l]);
    if (l > 0) {
      const int* cf = &sym.levelFronts[sym.levelPtr[l - 1]];
      const int cc = sym.levelPtr[l] - sym.levelPtr[l - 1];
      for (int t = 0; t < cc; t++) {
        const Front& C = sym.fronts[cf[t]];
        // a chain link only adds its first k_parent columns to the parent's panel (the rest stays in place)
        const int ncols = (C.parent >= 0 && sym.fronts[C.parent].inplace) ? std::min(C.m(), sym.fronts[C.parent].k) : C.m();
        for (int cb = 0; cb * EADD_COLS < ncols; cb++)
          for (int rb = (cb * EADD_COLS) / EADD_ROWS; rb * EADD_ROWS < C.m(); rb++) items.push_back(WorkItem{cf[t], cb, rb});
      }
    }
    end(eaddItems[l]);
    begin(diagItems[l]);   // pivot blocks wider than 32 columns: 256-thread CTAs
    for (int t = 0; t < cnt; t++)
      if (sym.fronts[lf[t]].k > 32) items.push_back(WorkItem{lf[t], 0, 0});
    end(diagItems[l]);
    begin(diagSmallItems[l]);  // k <= 32: 64-thread CTAs
    for (int t = 0; t < cnt; t++)
      if (sym.fronts[lf[t]].k <= 32) items.push_back(WorkItem{lf[t], 0, 0});
    end(diagSmallItems[l]);
    begin(copyItems[l]);
    for (int t = 0; t < cnt; t++)
      for (int rb = 0; rb * COPY_ROWS < sym.fronts[lf[t]].m(); rb++)
        for (int cb = 0; cb * COPY_COLS < sym.fronts[lf[t]].k; cb++) items.push_back(WorkItem{lf[t], rb, cb});
    end(copyItems[l]);
    begin(panelItems[l]);
    for (int t = 0; t < cnt; t++) {
      const Front& F = sym.fronts[lf[t]];
      for (int ti = 0; ti * TS < F.m(); ti++)
        for (int tj = 0; tj * TS < F.k; tj++) items.push_back(WorkItem{lf[t], ti, tj});
    }
    end(panelItems[l]);
    begin(schurItems[l]);
    for (int t = 0; t < cnt; t++) {
      const Front& F = sym.fronts[lf[t]];
      if (F.pair == 2) continue;
      // first of a chain pair: only the column tiles the next panel assembles; the rest waits for the rank-256 update
      const int ncolTiles = F.pair == 1 ? (std::min(F.m(), sym.fronts[lf[t] + 1].k) + TS - 1) / TS : (F.m() + TS - 1) / TS;
      for (int ti = 0; ti * TS < F.m(); ti++)
        for (int tj = 0; tj <= ti && tj < ncolTiles; tj++) items.push_back(WorkItem{lf[t], ti, tj});
    }
    end(schurItems[l]);
    begin(schur2Items[l]);
    for (int t = 0; t < cnt; t++) {
      const Front& F = sym.fronts[lf[t]];
      if (F.pair != 2) continue;
      for (int ti = 0; ti * TS < F.m(); ti++)
        for (int tj = 0; tj <= ti; tj++) items.push_back(WorkItem{lf[t], ti, tj});
    }
    end(schur2Items[l]);
  }

}

void LdltPlan::upload() {
  dFronts.upload(hostFronts_);
  dRowIdx.upload(sym.rowIdx);
  if (!sym.rel.empty()) dRel.upload(sym.rel);
  dAsmSrc.upload(sym.asmSrc);
  dAsmDst.upload(sym.asmDst);
  dItems.upload(hostItems_);
  dPerm.upload(sym.perm);
  CUDA_CHECK(::geneo::sync_stream(0));
  // the host copies of the big arrays are no longer needed
  std::vector<int64_t>().swap(sym.asmSrc);
  std::vector<int64_t>().swap(sym.asmDst);
  std::vector<WorkItem>().swap(hostItems_);
  std::vector<FrontDev>().swap(hostFronts_);
}

size_t LdltPlan::plan_bytes() const {
  return dFronts.bytes() + dRowIdx.bytes() + dRel.bytes() + dAsmSrc.bytes() + dAsmDst.bytes() + dItems.bytes() +
         dPerm.bytes();
}

void LdltWorkspace::ensure(const Symbolic& s) {
  if ((int64_t)u0.n < s.uArena) { u0.alloc((size_t)s.uArena); u1.alloc((size_t)s.uArena); }
  if ((int64_t)uc.n < s.cArena) uc.alloc((size_t)s.cArena);
  if ((int64_t)w0.n < s.wArena) { w0.alloc((size_t)s.wArena); w1.alloc((size_t)s.wArena); }
  if (counters.n < 2) counters.alloc(2);
}

namespace {
void factor_prepare(FactorJob& J) {
  const LdltPlan& P = J.F->plan();
  const Symbolic& S = P.sym;
  J.ws->ensure(S);
  if ((int64_t)J.F->L.n < S.lSize) J.F->L.alloc((size_t)S.lSize);  // a recycled (larger) buffer is fine
  CUDA_CHECK(cudaMemsetAsync(J.F->L.p, 0, (size_t)S.lSize * sizeof(double), J.st));
  J.ws->counters.zero(J.st);
  const int64_t cnt = (int64_t)P.dAsmSrc.n;
  const int grid = (int)std::min<int64_t>((cnt + 255) / 256, 148 * 16);
  if (cnt) k_assemble<<<GENEO_TICK(grid), 256, 0, J.st>>>(cnt, P.dAsmSrc.p, P.dAsmDst.p, J.vals, J.F->L.p);
  CUDA_CHECK(cudaGetLastError());
}

void factor_level(FactorJob& J, int l) {
  const LdltPlan& P = J.F->plan();
  LdltWorkspace& ws = *J.ws;
  cudaStream_t st = J.st;
  double* Lp = J.F->L.p;
  const double pivTol = J.pivTol;
  const WorkItem* items = P.dItems.p;
  const UArenas ua{{ws.u0.p, ws.u1.p, ws.uc.p}};
  double* Ucur = (l & 1) ? ws.u1.p : ws.u0.p;
  double* Wcur = (l & 1) ? ws.w1.p : ws.w0.p;
  const double* Wprev = (l & 1) ? ws.w0.p : ws.w1.p;
  if (P.levelU[l] > 0) CUDA_CHECK(cudaMemsetAsync(Ucur, 0, (size_t)P.levelU[l] * sizeof(double), st));
  for (auto& z : P.levelChainZero[l]) CUDA_CHECK(cudaMemsetAsync(ws.uc.p + z.first, 0, (size_t)z.second * sizeof(double), st));
  if (P.eaddItems[l].cnt)
    k_extend_add<<<GENEO_TICK(P.eaddItems[l].cnt), 256, 0, st>>>(items + P.eaddItems[l].off, P.dFronts.p, P.dRel.p, Lp, ua);
  if (P.diagItems[l].cnt)
    k_diag_invert<128, 16><<<GENEO_TICK(P.diagItems[l].cnt), 256, 0, st>>>(items + P.diagItems[l].off, P.dFronts.p, Lp, pivTol, ws.counters.p);
  if (P.diagSmallItems[l].cnt)
    k_diag_invert<32, 8><<<GENEO_TICK(P.diagSmallItems[l].cnt), 64, 0, st>>>(items + P.diagSmallItems[l].off, P.dFronts.p, Lp, pivTol, ws.counters.p);
  if (P.copyItems[l].cnt)
    k_copy_panel<<<GENEO_TICK(P.copyItems[l].cnt), 256, 0, st>>>(items + P.copyItems[l].off, P.dFronts.p, Lp, Wcur);
  if (P.panelItems[l].cnt)
    k_panel<<<GENEO_TICK(P.panelItems[l].cnt), GEMM_THREADS, GEMM_SMEM, st>>>(items + P.panelItems[l].off, P.dFronts.p, Lp, Wcur);
  if (P.schurItems[l].cnt)
    k_schur<<<GENEO_TICK(P.schurItems[l].cnt), GEMM_THREADS, GEMM_SMEM, st>>>(items + P.schurItems[l].off, P.dFronts.p, Lp, Wcur, ua);
  if (P.schur2Items[l].cnt)
    k_schur2<<<GENEO_TICK(P.schur2Items[l].cnt), GEMM_THREADS, GEMM_SMEM, st>>>(items + P.schur2Items[l].off, P.dFronts.p, Lp, Wcur, Wprev, ua);
  CUDA_CHECK(cudaGetLastError());
}
}  // namespace

void factorize_enqueue(std::vector<FactorJob>& jobs) {
  int gmax = 0;
  for (auto& J : jobs) { factor_prepare(J); gmax = std::max(gmax, J.F->plan().sym.nlevels); }
  for (int g = 0; g < gmax; g++)
    for (auto& J : jobs) {
      const int l = g - (gmax - J.F->plan().sym.nlevels);  // roots aligned
      if (l >= 0) factor_level(J, l);
    }
  for (auto& J : jobs)
    if (J.hostCounters) CUDA_CHECK(cudaMemcpyAsync(J.hostCounters, J.ws->counters.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, J.st));
}

FactorStats LdltFactor::factorize(const double* dVals, double pivTol, LdltWorkspace& ws, cudaStream_t st) {
  FactorStats stats;
  const double t0 = now_s();
  HostProfScope hp("factorize: host side total");
  int h[2] = {0, 0};
  std::vector<FactorJob> jobs(1);
  jobs[0].F = this; jobs[0].vals = dVals; jobs[0].pivTol = pivTol; jobs[0].ws = &ws; jobs[0].st = st; jobs[0].hostCounters = h;
  factorize_enqueue(jobs);
  CUDA_CHECK(::geneo::sync_stream(st));
  stats.neg = h[0];
  stats.perturbed = h[1];
  stats.seconds = now_s() - t0;
  return stats;
}

struct RingLaunch { const void* fn; int warps, smem, bwdCols; };
static RingLaunch ring_launch(int which) {  // which = 0: NR = 1, 1: NR = 8, 2: NR = 16 (shares the item lists of NR = 8)
  static const RingLaunch table[3] = {
      {(const void*)k_solve_ring<1>, RingCfg<1>::WARPS, RingCfg<1>::SMEM, RingCfg<1>::BWD_COLS},
      {(const void*)k_solve_ring<8>, RingCfg<8>::WARPS, RingCfg<8>::SMEM, RingCfg<8>::BWD_COLS},
      {(const void*)k_solve_ring<16>, RingCfg<16>::WARPS, RingCfg<16>::SMEM, RingCfg<16>::BWD_COLS}};
  return table[which];
}

// =====================================================================================================================
// SolveForest
// =====================================================================================================================
void SolveForest::build(const std::vector<const LdltPlan*>& plans, const std::vector<int64_t>& xoff) {
  const int ns = (int)plans.size();
  plans_ = plans;
  xoff_ = xoff;
  nlev = 0;
  ntot = 0;
  for (int s = 0; s < ns; s++) { nlev = std::max(nlev, plans[s]->sym.nlevels); ntot = std::max<int64_t>(ntot, xoff[s] + plans[s]->sym.n); }
  ringBuilt[0] = ringBuilt[1] = false;
  hSubs.assign(ns, ForestSub{nullptr, nullptr, nullptr, 0});
  for (int s = 0; s < ns; s++) { hSubs[s].fronts = plans[s]->dFronts.p; hSubs[s].rowIdx = plans[s]->dRowIdx.p; hSubs[s].xoff = xoff[s]; }
  dSubs.alloc(ns);
  CUDA_CHECK(::geneo::sync_stream(0));
  int dev = 0, nsm = 0;
  CUDA_CHECK(cudaGetDevice(&dev));
  CUDA_CHECK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
  for (int which = 0; which < 3; which++) {
    const RingLaunch rl = ring_launch(which);
    int nb = 0;
    CUDA_CHECK(cudaFuncSetAttribute(rl.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, rl.smem));
    CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rl.fn, rl.warps * 32, rl.smem));
    if (which < 2) ringGrid[which] = std::max(1, nb) * nsm;
    else ringGrid[1] = std::min(ringGrid[1], std::max(1, nb) * nsm);  // NR = 16 walks the NR = 8 lists on the SAME cooperative grid:
                                                                        // it must fit both kernels (the warp -> item mapping is
                                                                        // computed in the kernel from its own block size)
  }
}

// Item lists of the ring kernel.  Per level the host picks the span of an item from the amount of work in the level: a
// level with many tiles per warp gets wide (forward: up to all 128 columns of a panel) / tall (backward: up to 512 rows)
// items -- fewer records, x / y fetches and atomics per byte --, a level near the root gets the finest tiles so that every
// warp of the chip has something to stream.
void SolveForest::build_ring(int which) const {
  HostProfScope hp("forest build (ring)");
  const int ns = (int)plans_.size();
  const int warps = ring_launch(which).warps;
  const int RING_BWD_COLS = ring_launch(which).bwdCols;
  const int64_t nw = (int64_t)ringGrid[which] * warps;
  std::vector<RingItem> items;
  std::vector<int64_t> ranges(4 * (size_t)nlev, 0);
  std::vector<double>& ringBytes = ringBytes_[which];
  std::vector<int64_t>& ringCount = ringCount_[which];
  ringBytes.assign(2 * (size_t)nlev, 0.);
  ringCount.assign(2 * (size_t)nlev, 0);
  auto by_size = [](const RingItem& a, const RingItem& b) { return (int64_t)a.nrows * a.nc > (int64_t)b.nrows * b.nc; };
  auto pow2_floor = [](int64_t v, int lo, int hi) { int r = lo; while (2 * r <= hi && 2 * (int64_t)r <= v) r *= 2; return r; };
  for (int l = 0; l < nlev; l++) {  // forward + diagonal: every row of the panel
    int64_t tiles = 0;
    double bytes = 0.;
    for (int s = 0; s < ns; s++) {
      const Symbolic& S = plans_[s]->sym;
      if (l >= S.nlevels) continue;
      for (int t = S.levelPtr[l]; t < S.levelPtr[l + 1]; t++) {
        const Front& F = S.fronts[S.levelFronts[t]];
        tiles += (int64_t)((F.h + 63) / 64) * ((F.k + 31) / 32);
        bytes += 8. * F.h * F.k;
      }
    }
    // 32 is the floor for the block solves too: wider floors measured slower (8 x 100^3 eigen-solves: 3.25 / 3.30 / 3.48 s at 32 / 64 / 128)
    const int cspan = 32 * pow2_floor(tiles / (4 * nw), 1, 4);
    ranges[l] = (int64_t)items.size();
    for (int s = 0; s < ns; s++) {
      const Symbolic& S = plans_[s]->sym;
      if (l >= S.nlevels) continue;
      for (int t = S.levelPtr[l]; t < S.levelPtr[l + 1]; t++) {
        const Front& F = S.fronts[S.levelFronts[t]];
        for (int r0 = 0; r0 < F.h; r0 += 64)
          for (int c0 = 0; c0 < F.k; c0 += cspan)
            items.push_back(RingItem{F.lOff + (int64_t)c0 * F.ld + r0, F.rowOff + r0, s, F.ld, std::min(64, F.h - r0),
                                     std::min(cspan, F.k - c0), std::max(0, std::min(64, F.k - r0)), F.col0 + c0, F.col0 + r0, 0});
      }
    }
    ranges[nlev + l] = (int64_t)items.size() - ranges[l];
    std::stable_sort(items.begin() + ranges[l], items.end(), by_size);
    ringBytes[l] = bytes;
    ringCount[l] = ranges[nlev + l];
  }
  for (int l = 0; l < nlev; l++) {  // backward: the L21 rows, tiles start at the even row k & ~1 (row k-1 masked by kdiag)
    int64_t tiles = 0;
    double bytes = 0.;
    for (int s = 0; s < ns; s++) {
      const Symbolic& S = plans_[s]->sym;
      if (l >= S.nlevels) continue;
      for (int t = S.levelPtr[l]; t < S.levelPtr[l + 1]; t++) {
        const Front& F = S.fronts[S.levelFronts[t]];
        if (F.m() == 0) continue;
        tiles += (int64_t)((F.h - (F.k & ~1) + 63) / 64) * ((F.k + RING_BWD_COLS - 1) / RING_BWD_COLS);
        bytes += 8. * F.m() * F.k;
      }
    }
    const int rspan = 64 * pow2_floor(tiles / (2 * nw), 1, 8);
    ranges[2 * nlev + l] = (int64_t)items.size();
    for (int s = 0; s < ns; s++) {
      const Symbolic& S = plans_[s]->sym;
      if (l >= S.nlevels) continue;
      for (int t = S.levelPtr[l]; t < S.levelPtr[l + 1]; t++) {
        const Front& F = S.fronts[S.levelFronts[t]];
        if (F.m() == 0) continue;
        const int rstart = F.k & ~1;
        for (int r0 = rstart; r0 < F.h; r0 += rspan)
          for (int c0 = 0; c0 < F.k; c0 += RING_BWD_COLS)
            items.push_back(RingItem{F.lOff + (int64_t)c0 * F.ld + r0, F.rowOff + r0, s, F.ld, std::min(rspan, F.h - r0),
                                     std::min(RING_BWD_COLS, F.k - c0), std::max(0, F.k - r0), F.col0 + c0, 0, 0});
      }
    }
    ranges[3 * nlev + l] = (int64_t)items.size() - ranges[2 * nlev + l];
    std::stable_sort(items.begin() + ranges[2 * nlev + l], items.end(), by_size);
    ringBytes[2 * nlev - 1 - l] = bytes;  // phase order: backward runs from the root down
    ringCount[2 * nlev - 1 - l] = ranges[3 * nlev + l];
  }
  dRing[which].upload(items);
  dRingRanges[which].upload(ranges);
  CUDA_CHECK(::geneo::sync_stream(0));
  ringBuilt[which] = true;
}

void SolveForest::set_factors(const std::vector<const double*>& L, cudaStream_t st) {
  GENEO_CHECK(L.size() == hSubs.size(), "forest: wrong number of factors");
  for (size_t s = 0; s < L.size(); s++) hSubs[s].L = L[s];
  CUDA_CHECK(cudaMemcpyAsync(dSubs.p, hSubs.data(), sizeof(ForestSub) * hSubs.size(), cudaMemcpyHostToDevice, st));
  CUDA_CHECK(::geneo::sync_stream(st));
}

void SolveForest::solve(double* X, double* Y, int ldx, int j0, int nr, cudaStream_t st) const {
  GENEO_CHECK((nr == 1 && ldx == 1) || nr == 8 || nr == 16, "forest solve: nr must be 1 (with ldx = 1), 8 or 16");
  double* Xp = X + j0;
  double* Yp = Y + j0;
  const ForestSub* subs = dSubs.p;
  int nsubs = (int)hSubs.size();
  int nl = nlev;
  int64_t nt = ntot;
  const int which = nr == 1 ? 0 : 1;
  if (!ringBuilt[which]) build_ring(which);
  const RingItem* ritems = dRing[which].p;
  const int64_t* rranges = dRingRanges[which].p;
  long long* ts = nullptr;
  void* a1[] = {(void*)&subs, (void*)&nsubs, (void*)&ritems, (void*)&rranges, (void*)&nl, (void*)&nt, (void*)&Xp, (void*)&Yp,
                (void*)&ldx, (void*)&ts};
  (void)GENEO_TICK(0);
  const RingLaunch rl = ring_launch(nr == 16 ? 2 : which);
  CUDA_CHECK(cudaLaunchCooperativeKernel(rl.fn, dim3(ringGrid[which]), dim3(rl.warps * 32), a1, rl.smem, st));
}

void SolveForest::solve_profile(double* X, double* Y, int nr, std::vector<double>& us, std::vector<double>& bytes,
                                std::vector<int64_t>& nitems) const {
  GENEO_CHECK(nr == 1 || nr == 8, "solve_profile: nr must be 1 or 8");
  const int which = nr == 1 ? 0 : 1;
  if (!ringBuilt[which]) build_ring(which);
  const ForestSub* subs = dSubs.p;
  int nsubs = (int)hSubs.size();
  const RingItem* ritems = dRing[which].p;
  const int64_t* rranges = dRingRanges[which].p;
  int nl = nlev;
  int64_t nt = ntot;
  int ldx = nr;
  DevBuf<long long> dts((size_t)2 * nlev + 1);
  long long* ts = dts.p;
  void* a1[] = {(void*)&subs, (void*)&nsubs, (void*)&ritems, (void*)&rranges, (void*)&nl, (void*)&nt, (void*)&X, (void*)&Y,
                (void*)&ldx, (void*)&ts};
  (void)GENEO_TICK(0);
  const RingLaunch rl = ring_launch(which);
  CUDA_CHECK(cudaLaunchCooperativeKernel(rl.fn, dim3(ringGrid[which]), dim3(rl.warps * 32), a1, rl.smem, 0));
  CUDA_CHECK(::geneo::sync_stream(0));
  std::vector<long long> h = dts.to_host();
  us.resize(2 * (size_t)nlev);
  for (int p = 0; p < 2 * nlev; p++) us[p] = 1e-3 * (double)(h[p + 1] - h[p]);
  bytes = ringBytes_[which];
  nitems = ringCount_[which];
}

// Synthetic streaming benchmark of the solve kernel: nf independent h x k panels at ONE level (no level effects, no
// small fronts): what fraction of the HBM bandwidth do the forward / backward tiles reach on their own?
double solve_stream_bench(int nf, int h, int k, int reps, double* gbps, int nlev, int nr) {
  // nlev levels of nf independent h x k panels each (level l front f: rows/cols disjoint from everything else)
  Symbolic S;
  const int nt = nf * nlev;
  S.n = nt * h;
  S.nb = 128;
  S.fronts.resize(nt);
  S.rowIdx.resize((size_t)nt * h);
  for (int64_t i = 0; i < (int64_t)nt * h; i++) S.rowIdx[i] = (int)i;
  int64_t lOff = 0;
  for (int f = 0; f < nt; f++) {
    Front& F = S.fronts[f];
    F.col0 = f * h; F.k = k; F.h = h; F.ld = (h + 1) & ~1; F.parent = -1; F.level = f / nf; F.rowOff = (int64_t)f * h; F.lOff = lOff;
    lOff += (int64_t)F.ld * k;
  }
  S.lSize = lOff;
  S.nlevels = nlev;
  S.levelPtr.resize(nlev + 1);
  for (int l = 0; l <= nlev; l++) S.levelPtr[l] = l * nf;
  S.levelFronts.resize(nt);
  for (int f = 0; f < nt; f++) S.levelFronts[f] = f;
  S.perm.resize(S.n); S.iperm.resize(S.n);
  for (int i = 0; i < S.n; i++) S.perm[i] = S.iperm[i] = i;
  S.frontOfCol.assign(S.n, 0);
  auto plan = std::make_shared<LdltPlan>(std::move(S));
  DevBuf<double> L((size_t)lOff), X((size_t)nt * h * nr), Y((size_t)nt * h * nr);
  CUDA_CHECK(cudaMemset(L.p, 0, L.bytes()));
  CUDA_CHECK(cudaMemset(X.p, 0, X.bytes()));
  SolveForest F;
  F.build({plan.get()}, {0});
  F.set_factors({L.p}, 0);
  for (int i = 0; i < 2; i++) F.solve(X.p, Y.p, nr, 0, nr, 0);
  cudaEvent_t e0, e1;
  CUDA_CHECK(cudaEventCreate(&e0)); CUDA_CHECK(cudaEventCreate(&e1));
  CUDA_CHECK(cudaEventRecord(e0, 0));
  for (int i = 0; i < reps; i++) F.solve(X.p, Y.p, nr, 0, nr, 0);
  CUDA_CHECK(cudaEventRecord(e1, 0));
  CUDA_CHECK(cudaEventSynchronize(e1));
  float ms = 0.f;
  CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  const double bytes = (double)nt * 8. * (2. * (double)(h - k) * k + (double)k * k);
  if (gbps) *gbps = bytes * reps / (ms * 1e-3) / 1e9;
  return ms / reps;
}

void LdltFactor::solve_permuted(double* X, double* Y, int ldx, int j0, int nr, cudaStream_t st) const {
  GENEO_CHECK(L.p != nullptr, "solve before factorize");
  const LdltPlan& P = *plan_;
  if (!P.selfForest) {
    P.selfForest = std::make_shared<SolveForest>();
    P.selfForest->build({plan_.get()}, {0});
    P.selfL = nullptr;
  }
  if (P.selfL != L.p) { P.selfForest->set_factors({L.p}, st); P.selfL = L.p; }
  P.selfForest->solve(X, Y, ldx, j0, nr, st);
}

}  // namespace geneo
