// symbolic.hpp -- host symbolic analysis for the block LDL^T multifrontal solver that replaces MUMPS
// (reference call sites: src/geneo.cpp:94-124 directLocalSolve, :452-500 getInertia, :746-780 buildEigenSolver).
//
// Design (B200-first, see DESIGN.md "Sparse LDL^T"):
//   * fill-reducing ordering: METIS NodeND on the host, the natural order, or a permutation from the caller (the reference
//     box ordering shared by the subdomains of a structured problem);
//   * elimination tree, postorder, Gilbert-Ng-Peyton column counts, supernodes with relaxed amalgamation;
//   * every supernode is cut into PANELS ("fronts") of at most NB pivot columns, chained in the assembly tree, so that
//     each front needs exactly one dense NBxNB pivot-block inversion, one panel product and one Schur GEMM;
//   * fronts are levelled top-down (level = height - depth): a child is always exactly one level below its parent, so
//     update matrices live in two ping-pong arenas and every level is ONE batched launch per kernel;
//   * the factor is stored as block LDL^T:  panel f (h x k, column-major, ld = h) holds D_f^{-1} (k x k, full) on top
//     of the unit-lower block L21 = F21 D_f^{-1} (m x k).  Triangular solves then contain no triangular kernel at all:
//     forward = rectangular GEMV scatter, diagonal = dense k x k GEMV, backward = transposed GEMV gather.
#pragma once
#include <cstdint>
#include <vector>

namespace geneo {

struct Front {
  int col0 = 0;        // first pivot column (permuted numbering)
  int k = 0;           // pivot columns (<= NB)
  int h = 0;           // rows of the panel = k + m
  int ld = 0;          // leading dimension of the panel in the factor array: h rounded up to even (16-byte columns)
  int parent = -1;     // parent front, -1 for a root
  int level = 0;       // schedule level (children are at level-1)
  int chain = 0;       // 1 if the parent is the next panel of the same supernode (identity relative indices)
  int nchild = 0;
  int64_t rowOff = 0;  // into Symbolic::rowIdx (h entries, ascending, first k = own columns)
  int64_t lOff = 0;    // into the factor value array (ld*k doubles)
  int64_t uOff = -1;   // into update arena `uArena`; the update matrix is m x m (lower triangle used) with leading dimension uLd
  int uLd = 0;         // leading dimension of the update matrix storage
  int uArena = 0;      // 0/1: ping-pong arena of parity (level & 1) -- consumed by the next level; 2: chain arena
  int pair = 0;        // rank-256 trailing updates along a chain: 1 = first of a pair (only the strip of its update matrix
                       // that the next panel assembles is updated at its own level), 2 = second of a pair (its Schur
                       // update applies BOTH panels at once: K = k_prev + k, one read-modify-write of the update matrix
                       // for two panels); 0 = ordinary rank-k update
  int inplace = 0;     // 1: non-first panel of a supernode -- its update matrix IS the trailing block of its (only)
                       // child's update matrix (same storage, uOff = child.uOff + k (uLd + 1)): nothing is copied or
                       // zeroed along a supernode chain, the child only adds its first k columns to this panel
  int64_t wOff = -1;   // into the per-level scratch holding the unscaled panel F21 (m*k doubles, ld = m)
  int64_t relOff = -1; // into Symbolic::rel (m entries: position of update row i in the parent's row list); -1 if chain
  int m() const { return h - k; }
};

struct Symbolic {
  int n = 0, nb = 128;
  std::vector<int> perm;   // new -> old
  std::vector<int> iperm;  // old -> new
  std::vector<Front> fronts;
  std::vector<int> rowIdx;
  std::vector<int> rel;
  std::vector<int> frontOfCol;  // permuted column -> front
  int nlevels = 0;
  std::vector<int> levelPtr;    // [nlevels+1] into levelFronts
  std::vector<int> levelFronts; // fronts sorted by level
  int64_t lSize = 0;            // doubles in the factor
  int64_t uArena = 0;           // doubles in EACH of the two ping-pong update arenas
  int64_t cArena = 0;           // doubles in the chain arena (update matrices that live for a whole supernode chain)
  int64_t wArena = 0;           // doubles in the per-level panel scratch
  // scatter of the input values into the factor array: for t < asmSrc.size(): L[asmDst[t]] = val[asmSrc[t]]
  std::vector<int64_t> asmSrc;  // index into the input CSR value array (lower triangle entries after permutation)
  std::vector<int64_t> asmDst;
  // statistics
  int nsuper = 0;
  double flops = 0.;            // sum_f k^3/3 + m k^2 + m^2 k
  int64_t nnzRowIdx = 0;
  int maxK = 0, maxH = 0;
};

struct SymbolicOptions {
  int nb = 128;        // panel width
  int ordering = 1;    // 0 natural, 1 METIS NodeND, 3 caller-supplied permutation (userPerm)
  const int* userPerm = nullptr;  // ordering == 3: new -> old, length n
  bool amalgamate = true;
  int subtreeCols = 64; // subtrees of the assembly tree with at most this many columns are merged into one dense front
  bool skipAsm = false;  // leave asmSrc / asmDst empty: the caller builds the scatter map itself (symbolic_asm_map, or
                         // fused with its own pass over the matrix as GeneoPC's host preparation does)
  int ndDepth = 0;     // top levels of the nested dissection done here (METIS_ComputeVertexSeparator) with the two halves
                       // ordered by concurrent threads: 2^ndDepth threads per matrix; 0 = plain METIS_NodeND
};

// Reference nested dissection of a dims[0] x dims[1] x dims[2] box of grid points coupled through `stencil` (nst integer
// offsets, 3 ints each; both signs need not be listed).  rank[x + dims[0] (y + dims[1] z)] = position of the point in the
// elimination order.  ANY subset of the box inherits a valid nested-dissection ordering by sorting its points by rank
// (induced separators): the subdomains of a structured problem that fit into one bounding box share ONE METIS call instead
// of one each -- the host wall of the cold setup (MUMPS analysis in the reference, src/geneo.cpp:99-110).
void box_reference_ordering(const int dims[3], int nst, const int* stencil, int ndDepth, std::vector<int>& rank);

// ptr/idx: CSR pattern of a structurally symmetric n x n matrix (both triangles; column order irrelevant).
void symbolic_analyze(int n, const int64_t* ptr, const int* idx, const SymbolicOptions& opt, Symbolic& s);

// tT[t] = position of the entry (c, r) for the entry t = (r, c).  Needs sorted rows and a symmetric pattern: returns false
// (tT unspecified) otherwise.  ndiag (optional) = number of diagonal entries present.
bool transpose_positions(int n, const int64_t* ptr, const int* idx, std::vector<int64_t>& tT, int64_t* ndiag);

// Scatter map of an analysed matrix (asmSrc = positions in the INPUT value array).  Entry (i, j), i >= j, of P A P^T takes
// the value stored in row perm[i] of the input.  With tT (transpose_positions) the map is built front by front with one
// table lookup per entry; without it, row by row with a binary search per entry.
void symbolic_asm_map(int n, const int64_t* ptr, const int* idx, const std::vector<int64_t>* tT, Symbolic& s);

}  // namespace geneo
