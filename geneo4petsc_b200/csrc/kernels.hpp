// kernels.hpp -- HBM-bound building blocks: SELL-32 SpMV, CSR SpMM, fused BLAS-1, gather/scatter (restrict/prolong),
// tall-skinny Gram / block updates.  Replaces PETSc MatMult / Vec* / VecScatter on the hot path
// (reference call sites: src/geneo4PETSc.cpp:1240,1354; src/geneo.cpp:1850-1852,1881-1883,1931-1944,1469-1513).
#pragma once
#include "common.hpp"

namespace geneo {

// Sliced ELLPACK, slice height 32 (one warp per slice, one thread per row, column-major inside the slice so every
// warp load is one contiguous 256-byte (values) / 128-byte (indices) transaction).
struct SellMatrix {
  int n = 0, nslices = 0;
  int64_t nnz = 0;        // true nonzeros (for algorithmic byte counts)
  int64_t stored = 0;     // stored entries incl. padding
  DevBuf<int64_t> sliceOff;  // [nslices+1]
  DevBuf<int> col;
  DevBuf<double> val;
  DevBuf<int> rowLen;     // [n] true entries of every row (padding carries column = row and value 0: not searchable)
  void build(const CsrHost& a, cudaStream_t st);
  // algorithmic bytes of one SpMV (CSR formula of SURVEY.md 8d): nnz*12 + (n+1)*4 + 16*n
  double algo_bytes() const { return (double)nnz * 12. + ((double)n + 1.) * 4. + 16. * (double)n; }
};
void sell_spmv(const SellMatrix& A, const double* x, double* y, cudaStream_t st);              // y = A x
void sell_spmv_sub(const SellMatrix& A, const double* x, const double* b, double* y, cudaStream_t st);  // y = b - A x

// Y[:, 0:8] = A X[:, 0:8] (row-major blocks, ld 8) -- used by the coarse operator assembly W = A (R_j^T Z_j) and the block
// PC apply / block CG
void sell_spmm8(const SellMatrix& A, const double* X, double* Y, cudaStream_t st);

struct CsrDev {
  int n = 0;
  int64_t nnz = 0;
  DevBuf<int64_t> ptr;
  DevBuf<int> idx;
  DevBuf<double> val;
  void upload_pattern(const CsrHost& a, cudaStream_t st);
};
// Y[:, 0:nr] = A X[:, 0:nr] for row-major blocks (ldx, ldy); ptr/idx/val device CSR.
void csr_spmm(int n, const int64_t* ptr, const int* idx, const double* val, const double* X, int ldx, double* Y, int ldy,
              int nr, cudaStream_t st);

// ---- BLAS-1 (device results in `out`, one double per reduction, zeroed by the call) --------------------------------
void vec_dot(int n, const double* x, const double* y, double* out, cudaStream_t st);
void vec_dot2(int n, const double* x, const double* y, const double* z, double* out, cudaStream_t st);  // out[0]=x.y out[1]=z.z
void vec_axpy(int n, double a, const double* x, double* y, cudaStream_t st);                  // y += a x
void vec_aypx(int n, double a, const double* x, double* y, cudaStream_t st);                  // y = x + a y
void vec_axpby(int n, double a, const double* x, double b, double* y, cudaStream_t st);       // y = a x + b y
void vec_cg_update(int n, double a, const double* p, const double* w, double* x, double* r, cudaStream_t st);  // x+=a p; r-=a w
void vec_scale(int n, double a, double* x, cudaStream_t st);
void vec_set(int n, double a, double* x, cudaStream_t st);
void vec_iota(int n, double first, double* x, cudaStream_t st);                               // x[i] = first + i
void vec_mdot(int n, int nv, const double* V, int64_t ldv, const double* w, double* out, cudaStream_t st);   // out[j] = V_j . w
void vec_maxpy(int n, int nv, const double* V, int64_t ldv, const double* coef, double* w, cudaStream_t st); // w -= sum coef_j V_j (coef on device)

// ---- restrict / prolong ---------------------------------------------------------------------------------------------
// out[k*ld + j] = scale? scale[k]*x[idx[k]] : x[idx[k]]  (restrict + permutation (+ partition of unity))
void gather_rows(int64_t cnt, const int* idx, const double* scale, const double* x, double* out, cudaStream_t st);
// y[g] (=|+=) sum_{e in [ptr[g],ptr[g+1])} t[pos[e]]     (deterministic pull-prolong)
void pull_sum(int n, const int64_t* ptr, const int64_t* pos, const double* t, double* y, bool accumulate, cudaStream_t st);

// block versions (row-major n x 8 blocks): G[idx[k]*8 + c] = Z[k*ldz + c0 + c] (c < nc, other columns zero) and
// out[k*8 + c] = G[idx[k]*8 + c]
void scatter_rows8(int n, const int* idx, const double* Z, int ldz, int c0, int nc, double* G, cudaStream_t st);
void gather_rows8(int n, const int* idx, const double* G, double* out, cudaStream_t st);

// ---- blocks of 8 right-hand sides (GeneoPC::apply_block / solve_cg_block): row-major n x 8 blocks ---------------------
// B[i*8 + c] = X[c*ldx + i] for c < nc, 0 for nc <= c < 8 (column-major with leading dimension ldx -> row-major block)
void pack_cols8(int64_t n, int nc, const double* X, int64_t ldx, double* B, cudaStream_t st);
// Y[c*ldy + i] = B[i*8 + c] for c < nc (rows i >= n of Y are not written)
void unpack_cols8(int64_t n, int nc, const double* B, double* Y, int64_t ldy, cudaStream_t st);
// y[g*8 + c] = sum_{e in [ptr[g],ptr[g+1])} t[pos[e]*8 + c]   (pull_sum per column, same order)
void pull_sum8(int n, const int64_t* ptr, const int64_t* pos, const double* t, double* y, cudaStream_t st);
// per-column dots over n rows (out zeroed by the call): out[c] = x_c . y_c ; with z: also out[8 + c] = z_c . z_c
void dot_cols8(int n, const double* x, const double* y, const double* z, double* out, cudaStream_t st);
struct Coef8 { double v[8]; };  // one coefficient per column, passed by value
// columns c with bit c of mask set: x_c += a_c p_c, r_c -= a_c w_c
void cg_update8(int n, Coef8 a, unsigned mask, const double* p, const double* w, double* x, double* r, cudaStream_t st);
// columns c with bit c of mask set: p_c = z_c + b_c p_c
void aypx8(int n, Coef8 b, unsigned mask, const double* z, double* p, cudaStream_t st);

// ---- tall-skinny dense --------------------------------------------------------------------------------------------
// G[p x q] (row-major, ldg) += X[:,0:p]^T Y[:,0:q]   (n rows; caller zeroes G)
void ts_gram(int n, const double* X, int ldx, int p, const double* Y, int ldy, int q, double* G, int ldg, cudaStream_t st);
// W[:,0:q] = beta*W + alpha * Q[:,0:p] C[p x q]      (C row-major ldc, on device)
void ts_update(int n, const double* Q, int ldq, int p, const double* C, int ldc, int q, double* W, int ldw, double alpha,
               double beta, cudaStream_t st);
// coarse helpers on one subdomain block: w[c] = sum_k Z[k*ldz+c] * x[k] ; t[k] = a*t[k]*(d?d[k]:1) + sum_c Z[k*ldz+c] w[c]
void zt_x(int n, int nev, const double* Z, int ldz, const double* x, double* w, cudaStream_t st);
void z_w_add(int n, int nev, const double* Z, int ldz, const double* w, const double* d, double* t, cudaStream_t st);
void dense_gemv(int m, int n, const double* A, int lda, const double* x, double* y, cudaStream_t st);  // y = A x (row-major A)
// dst[r*ldd + j] = src[r*lds + j], j < ncols (row-major blocks; replaces pitched cudaMemcpy2D, which moves 8*ncols bytes per DMA row)
void copy_cols(int64_t n, const double* src, int lds, double* dst, int ldd, int ncols, cudaStream_t st);
void vec_pointwise(int64_t n, const double* d, double* x, cudaStream_t st);                   // x *= d
void rows_scale(int n, int ld, const double* d, double* Z, cudaStream_t st);                  // Z[k*ld + c] *= d[k]
// values of B = D A D on the pattern of A: out[nz] = d[row] * val[nz] * d[col] ; and out = a - tau*b
void csr_scale_sym(int n, const int64_t* ptr, const int* idx, const double* val, const double* d, double* out, cudaStream_t st);
void vals_axpby(int64_t nnz, const double* a, double tau, const double* b, double* out, cudaStream_t st);  // out = a - tau b
void csr_sum_all(int64_t nnz, const double* val, double* out, cudaStream_t st);               // out[0] = sum(val) (zeroed by the call)

// ---- same-pattern value update (GeneoPC::check_values / commit_values) -----------------------------------------------
// One thread per input row.  The locate kernels write no value the preconditioner uses: the located values land in fresh
// buffers and every mismatch is counted into cnt[UPD_*] (one set of counters per subdomain, read back once).  The
// duplicate counters are a defensive check: the library's own inputs cannot carry a duplicate column (the pre-decomposed
// input refuses one when the problem is built, the decomposition never makes one).
enum { UPD_NODES, UPD_DIR_ROW, UPD_DIR_OUTSIDE, UPD_DIR_DUP, UPD_NEU_OUTSIDE, UPD_NEU_DUP, UPD_NEU_NOT_IN_A, UPD_ANORM, UPD_SLOTS };
// iperm[perm[k]] = k; cnt[UPD_NODES] += (gidx[k] != nodes[perm[k]])
void update_nodes(int n, const int* perm, const int* gidx, const int* nodes, int* iperm, unsigned long long* cnt, cudaStream_t st);
// input CSR (ptr, idx, val) of A_dir, natural order -> dir[q] on the permuted pattern (patPtr, patIdx; rows sorted by column).
// Every row must have the stored row's length; hits (zeroed by the caller) bit 0 marks a filled q (duplicates).
void update_locate_dir(int n, int64_t nnz, const int64_t* ptr, const int* idx, const double* val, const int* iperm,
                       const int64_t* patPtr, const int* patIdx, int* hits, double* dir, unsigned long long* cnt, cudaStream_t st);
// input CSR of A_neu -> neu[q] (zeroed by the caller) on the same pattern and, per q, the slot of the operator A it adds to
// (row gidx[k], column gidx[kc]; slot[q] stays -1 off the A_neu pattern); cover[slot] = 1 marks the operator's entries reached.
// slot == nullptr (multi-GPU, where gidx is rank-local and A holds only the owned rows): no operator lookup, cover unused.
void update_locate_neu(int n, int64_t nnz, const int64_t* ptr, const int* idx, const double* val, const int* iperm, const int* gidx,
                       const int64_t* patPtr, const int* patIdx, int* hits, const SellMatrix& A, double* neu, int64_t* slot,
                       unsigned char* cover, unsigned long long* cnt, cudaStream_t st);
// *cnt += number of true entries of A that no A_neu entry reached
void update_cover_check(const SellMatrix& A, const unsigned char* cover, unsigned long long* cnt, cudaStream_t st);
// Multi-GPU: the owned rows (ptr, idx, val: CSR, A.n rows, local columns sorted) must have A's row lengths and columns
// position by position; their values go to the same slots of `out` (A.val's layout, padding zeroed by the caller).
// *cnt += rows that differ.
void update_owned_rows(const SellMatrix& A, int64_t nnz, const int64_t* ptr, const int* idx, const double* val, double* out,
                       unsigned long long* cnt, cudaStream_t st);
// *out = bits of max |v| (atomicMax on the bit pattern: exact, order-free; NaN ignored like std::max(amax, NaN) does)
void update_absmax(int64_t nnz, const double* v, unsigned long long* out, cudaStream_t st);
// A.val[slot[q]] += neu[q] where slot[q] >= 0 (a subdomain reaches every slot at most once: no atomics)
void update_sell_add(int64_t nnz, const int64_t* slot, const double* neu, SellMatrix& A, cudaStream_t st);
// Robin values (createRobinMatrix): rob[q] = dir[q] + optim * neu[q] where row and column are shared (d < 1), dir[q] elsewhere
void update_robin(int n, const int64_t* ptr, const int* idx, const double* d, const double* dir, const double* neu, double optim,
                  double* rob, cudaStream_t st);

}  // namespace geneo
