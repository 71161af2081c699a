// kernels.cu -- see kernels.hpp.  sm_100a.  Everything here is HBM-bound: coalesced, vectorised where alignment is
// known, grid sized as a multiple of the 148 SMs, warp-shuffle reductions.
#include "kernels.hpp"

#include <algorithm>

namespace geneo {
namespace {

constexpr int NSM = 148;

inline int grid_for(int64_t n, int threads, int perSm = 8) {
  int64_t g = (n + threads - 1) / threads;
  return (int)std::max<int64_t>(1, std::min<int64_t>(g, (int64_t)NSM * perSm));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block reduction of NV values per thread, result atomically added to out[0..NV)
template <int NV>
__device__ __forceinline__ void block_reduce_atomic(double (&v)[NV], double* out) {
  __shared__ double sh[NV][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int q = 0; q < NV; q++) {
    v[q] = warp_sum(v[q]);
    if (lane == 0) sh[q][warp] = v[q];
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int q = 0; q < NV; q++) {
      double s = lane < nw ? sh[q][lane] : 0.;
      s = warp_sum(s);
      if (lane == 0) atomicAdd(out + q, s);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// SELL-32 SpMV
// ---------------------------------------------------------------------------------------------------------------
template <bool SUB>
__global__ void __launch_bounds__(256) k_sell_spmv(int n, int nslices, const int64_t* __restrict__ sliceOff,
                                                   const int* __restrict__ col, const double* __restrict__ val,
                                                   const double* __restrict__ x, const double* __restrict__ b,
                                                   double* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  for (int s = blockIdx.x * wpb + (threadIdx.x >> 5); s < nslices; s += gridDim.x * wpb) {
    const int64_t o0 = sliceOff[s], o1 = sliceOff[s + 1];
    const int width = (int)((o1 - o0) >> 5);
    const int* c = col + o0 + lane;
    const double* v = val + o0 + lane;
    double a0 = 0., a1 = 0.;
    int j = 0;
    for (; j + 4 <= width; j += 4) {
      const int c0 = c[(j + 0) * 32], c1 = c[(j + 1) * 32], c2 = c[(j + 2) * 32], c3 = c[(j + 3) * 32];
      const double v0 = v[(j + 0) * 32], v1 = v[(j + 1) * 32], v2 = v[(j + 2) * 32], v3 = v[(j + 3) * 32];
      a0 += v0 * __ldg(x + c0);
      a1 += v1 * __ldg(x + c1);
      a0 += v2 * __ldg(x + c2);
      a1 += v3 * __ldg(x + c3);
    }
    for (; j < width; j++) a0 += v[j * 32] * __ldg(x + c[j * 32]);
    const int row = s * 32 + lane;
    if (row < n) y[row] = SUB ? (b[row] - (a0 + a1)) : (a0 + a1);
  }
}

__global__ void __launch_bounds__(256) k_sell_spmm8(int n, int nslices, const int64_t* __restrict__ sliceOff,
                                                    const int* __restrict__ col, const double* __restrict__ val,
                                                    const double* __restrict__ X, double* __restrict__ Y) {
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  for (int s = blockIdx.x * wpb + (threadIdx.x >> 5); s < nslices; s += gridDim.x * wpb) {
    const int64_t o0 = sliceOff[s], o1 = sliceOff[s + 1];
    const int width = (int)((o1 - o0) >> 5);
    double acc[8] = {0., 0., 0., 0., 0., 0., 0., 0.};
    for (int j = 0; j < width; j++) {
      const int c = col[o0 + j * 32 + lane];
      const double v = val[o0 + j * 32 + lane];
      const double2* xr = reinterpret_cast<const double2*>(X + (size_t)c * 8);
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const double2 xv = __ldg(xr + q);
        acc[2 * q] += v * xv.x;
        acc[2 * q + 1] += v * xv.y;
      }
    }
    const int row = s * 32 + lane;
    if (row < n) {
      double2* yr = reinterpret_cast<double2*>(Y + (size_t)row * 8);
#pragma unroll
      for (int q = 0; q < 4; q++) yr[q] = make_double2(acc[2 * q], acc[2 * q + 1]);
    }
  }
}
__global__ void k_scatter_rows8(int n, const int* __restrict__ idx, const double* __restrict__ Z, int ldz, int c0, int nc,
                                double* __restrict__ G) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < (int64_t)n * 8; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = t >> 3;
    const int c = (int)(t & 7);
    G[(size_t)idx[k] * 8 + c] = c < nc ? Z[(size_t)k * ldz + c0 + c] : 0.;
  }
}
__global__ void k_gather_rows8(int n, const int* __restrict__ idx, const double* __restrict__ G, double* __restrict__ out) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < (int64_t)n * 8; t += (int64_t)gridDim.x * blockDim.x)
    out[t] = G[(size_t)idx[t >> 3] * 8 + (t & 7)];
}

template <int NRT>
__global__ void __launch_bounds__(256) k_csr_spmm(int n, const int64_t* __restrict__ ptr, const int* __restrict__ idx,
                                                  const double* __restrict__ val, const double* __restrict__ X, int ldx,
                                                  double* __restrict__ Y, int ldy) {
  // NRT threads per row (one per right-hand side)
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t row = t / NRT;
  const int j = (int)(t % NRT);
  if (row >= n) return;
  double acc = 0.;
  for (int64_t q = ptr[row]; q < ptr[row + 1]; q++) acc += val[q] * X[(size_t)idx[q] * ldx + j];
  Y[(size_t)row * ldy + j] = acc;
}

// ---------------------------------------------------------------------------------------------------------------
// BLAS-1
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dot(int n, const double* __restrict__ x, const double* __restrict__ y,
                                             double* out) {
  double v[1] = {0.};
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    v[0] += x[i] * y[i];
  block_reduce_atomic<1>(v, out);
}
__global__ void __launch_bounds__(256) k_dot2(int n, const double* __restrict__ x, const double* __restrict__ y,
                                              const double* __restrict__ z, double* out) {
  double v[2] = {0., 0.};
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    v[0] += x[i] * y[i];
    const double zz = z[i];
    v[1] += zz * zz;
  }
  block_reduce_atomic<2>(v, out);
}
__global__ void k_axpby(int n, double a, const double* __restrict__ x, double b, double* __restrict__ y) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = a * x[i] + b * y[i];
}
__global__ void k_axpy(int n, double a, const double* __restrict__ x, double* __restrict__ y) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    y[i] += a * x[i];
}
__global__ void k_cg_update(int n, double a, const double* __restrict__ p, const double* __restrict__ w,
                            double* __restrict__ x, double* __restrict__ r) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    x[i] += a * p[i];
    r[i] -= a * w[i];
  }
}
__global__ void k_scale(int n, double a, double* __restrict__ x) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] *= a;
}
__global__ void k_set(int n, double a, double step, double* __restrict__ x) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    x[i] = a + step * (double)i;
}
// out[j] = V_j . w for j < nv : every CTA streams w once and all basis vectors (VecMDot)
__global__ void __launch_bounds__(256) k_mdot(int n, int nv, const double* __restrict__ V, int64_t ldv,
                                              const double* __restrict__ w, double* out) {
  for (int j0 = 0; j0 < nv; j0 += 4) {
    double v[4] = {0., 0., 0., 0.};
    const int nj = min(4, nv - j0);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
      const double wi = w[i];
      for (int q = 0; q < nj; q++) v[q] += V[(j0 + q) * ldv + i] * wi;
    }
    __syncthreads();
    block_reduce_atomic<4>(v, out + j0);  // out has room for nv rounded up to 4
    __syncthreads();
  }
}
__global__ void __launch_bounds__(256) k_maxpy(int n, int nv, const double* __restrict__ V, int64_t ldv,
                                               const double* __restrict__ coef, double* __restrict__ w) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double s = w[i];
    for (int j = 0; j < nv; j++) s -= coef[j] * V[j * ldv + i];
    w[i] = s;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// restrict / prolong
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_gather(int64_t cnt, const int* __restrict__ idx, const double* __restrict__ scale,
                         const double* __restrict__ x, double* __restrict__ out) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < cnt; k += (int64_t)gridDim.x * blockDim.x) {
    double v = __ldg(x + idx[k]);
    if (scale) v *= scale[k];
    out[k] = v;
  }
}
__global__ void k_pull_sum(int n, const int64_t* __restrict__ ptr, const int64_t* __restrict__ pos,
                           const double* __restrict__ t, double* __restrict__ y, bool accumulate) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
    double s = accumulate ? y[g] : 0.;
    for (int64_t e = ptr[g]; e < ptr[g + 1]; e++) s += __ldg(t + pos[e]);
    y[g] = s;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// tall-skinny dense
// ---------------------------------------------------------------------------------------------------------------
// G (p x q) += X^T Y  for tall-skinny row-major blocks (the Gram products of the block Lanczos eigen-solver: X = B Q with up
// to a few hundred columns, Y = one block of 8).  The long dimension is the K of mma.sync.m8n8k4.f64: a warp walks 4-row
// steps of its CTA's row range, A fragment = X[4 rows][8 columns]^T straight from global memory (4 rows x 64 bytes per
// load, 8 loads = 512 contiguous bytes per row), B fragment = Y[4 rows][8 columns]; 8 accumulator fragments per warp
// (64 columns of X per CTA), summed over the 8 warps through shared memory, one atomicAdd per entry and CTA.
constexpr int TG_PCOLS = 64;   // columns of X per CTA (8 fragments)
__device__ __forceinline__ void dmma_f64(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
// QT = 8-column tiles of Y per CTA (1 or 2): a block of 16 shares every X fragment between two B fragments, so X -- the
// n x dim basis, the only big operand -- is read once per Gram product whatever the Lanczos block.
template <int QT>
__global__ void __launch_bounds__(256) k_ts_gram(int n, const double* __restrict__ X, int ldx, int p,
                                                 const double* __restrict__ Y, int ldy, int q, double* G, int ldg,
                                                 int rowsPerCta) {
  __shared__ double red[8][8][64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int p0 = blockIdx.x * TG_PCOLS, q0 = blockIdx.y * 8 * QT;
  const int64_t r0 = (int64_t)blockIdx.z * rowsPerCta;
  const int64_t r1 = min((int64_t)n, r0 + rowsPerCta);
  double acc[QT][8][2];
#pragma unroll
  for (int qt = 0; qt < QT; qt++)
#pragma unroll
    for (int pb = 0; pb < 8; pb++) acc[qt][pb][0] = acc[qt][pb][1] = 0.;
  for (int64_t r = r0 + 4 * warp; r < r1; r += 32) {
    const int64_t row = r + t;
    const bool rok = row < r1;
    const double* xr = X + (size_t)(rok ? row : r0) * ldx + p0 + g;
    double yb[QT];
#pragma unroll
    for (int qt = 0; qt < QT; qt++) yb[qt] = (rok && q0 + qt * 8 + g < q) ? __ldg(Y + (size_t)row * ldy + q0 + qt * 8 + g) : 0.;
    double a[8];
#pragma unroll
    for (int pb = 0; pb < 8; pb++) a[pb] = (rok && p0 + pb * 8 + g < p) ? __ldg(xr + pb * 8) : 0.;
#pragma unroll
    for (int qt = 0; qt < QT; qt++)
#pragma unroll
      for (int pb = 0; pb < 8; pb++) dmma_f64(acc[qt][pb][0], acc[qt][pb][1], a[pb], yb[qt]);
  }
#pragma unroll
  for (int qt = 0; qt < QT; qt++) {
    if (qt > 0) __syncthreads();
#pragma unroll
    for (int pb = 0; pb < 8; pb++) { red[warp][pb][2 * lane] = acc[qt][pb][0]; red[warp][pb][2 * lane + 1] = acc[qt][pb][1]; }
    __syncthreads();
    for (int e = threadIdx.x; e < 8 * 64; e += 256) {
      const int pb = e >> 6, f = e & 63;  // fragment entry f of lane f/2: C[m = (f/2) >> 2][n = 2 ((f/2) & 3) + (f & 1)]
      double sum = 0.;
#pragma unroll
      for (int w = 0; w < 8; w++) sum += red[w][pb][f];
      const int ln = f >> 1;
      const int pc = p0 + pb * 8 + (ln >> 2), qc = q0 + qt * 8 + 2 * (ln & 3) + (f & 1);
      if (pc < p && qc < q && sum != 0.) atomicAdd(&G[(size_t)pc * ldg + qc], sum);
    }
  }
}

// W[r, 0:q] = beta W[r, 0:q] + alpha sum_p Q[r,p] C[p, 0:q],  q <= 8.  One thread per row (128 rows per CTA); Q tiles of
// 128 rows x 32 columns go through shared memory so that the global reads are coalesced 256-byte row segments and the
// per-row reads are conflict-free (leading dimension 33); C (p x 8) sits in shared memory and is read as a broadcast.
constexpr int TSU_ROWS = 128, TSU_COLS = 32;
template <int QW>  // columns of W per pass (8 or 16): Q is read once per pass
__global__ void __launch_bounds__(TSU_ROWS) k_ts_update(int n, const double* __restrict__ Q, int ldq, int p,
                                                        const double* __restrict__ C, int ldc, int q, double* __restrict__ W,
                                                        int ldw, double alpha, double beta) {
  extern __shared__ double sm[];
  double* sC = sm;                     // [p][QW]
  double* tile = sm + (size_t)p * QW;  // [TSU_ROWS][TSU_COLS + 1]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int e = tid; e < p * QW; e += TSU_ROWS) {
    const int pp = e / QW, jj = e % QW;
    sC[e] = jj < q ? C[(size_t)pp * ldc + jj] : 0.;
  }
  const int64_t r0 = (int64_t)blockIdx.x * TSU_ROWS;
  double acc[QW];
#pragma unroll
  for (int j = 0; j < QW; j++) acc[j] = 0.;
  for (int pb = 0; pb < p; pb += TSU_COLS) {
    __syncthreads();
    // warp w loads rows w*32 .. w*32+31 of the tile, lane = column
#pragma unroll 8
    for (int rr = 0; rr < 32; rr++) {
      const int64_t r = r0 + warp * 32 + rr;
      tile[(warp * 32 + rr) * (TSU_COLS + 1) + lane] = (r < n && pb + lane < p) ? Q[(size_t)r * ldq + pb + lane] : 0.;
    }
    __syncthreads();
    const int pc = min(TSU_COLS, p - pb);
    const double* trow = tile + tid * (TSU_COLS + 1);
    for (int pp = 0; pp < pc; pp++) {
      const double a = trow[pp];
      const double* c = sC + (size_t)(pb + pp) * QW;
#pragma unroll
      for (int j = 0; j < QW; j++) acc[j] += a * c[j];
    }
  }
  const int64_t r = r0 + tid;
  if (r < n) {
    double* w = W + (size_t)r * ldw;
#pragma unroll
    for (int j = 0; j < QW; j++)
      if (j < q) w[j] = (beta == 0. ? 0. : beta * w[j]) + alpha * acc[j];
  }
}

// w[c] += sum_k Z[k,c] x[k]  : block handles a row chunk; thread (c lanes within a row) ; nev <= 32*? generic loop
__global__ void __launch_bounds__(256) k_zt_x(int n, int nev, const double* __restrict__ Z, int ldz,
                                              const double* __restrict__ x, double* w) {
  // thread t handles column c = t % nevPad for rows r = t / nevPad + stride
  __shared__ double sh[256];
  int nevPad = 1;
  while (nevPad < nev) nevPad <<= 1;
  if (nevPad > 256) nevPad = 256;
  for (int c0 = 0; c0 < nev; c0 += nevPad) {
    const int c = c0 + (threadIdx.x % nevPad);
    const int rlane = threadIdx.x / nevPad, rstride = 256 / nevPad;
    double acc = 0.;
    if (c < nev)
      for (int64_t r = (int64_t)blockIdx.x * rstride + rlane; r < n; r += (int64_t)gridDim.x * rstride)
        acc += Z[(size_t)r * ldz + c] * x[r];
    sh[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < nevPad) {
      double s = 0.;
      for (int q = 0; q < rstride; q++) s += sh[q * nevPad + threadIdx.x];
      if (c0 + threadIdx.x < nev) atomicAdd(&w[c0 + threadIdx.x], s);
    }
    __syncthreads();
  }
}
__global__ void __launch_bounds__(256) k_z_w_add(int n, int nev, const double* __restrict__ Z, int ldz,
                                                 const double* __restrict__ w, const double* __restrict__ d,
                                                 double* __restrict__ t) {
  // one warp per 32/nevGroup rows would be ideal; simple version: warp per row group, lanes over columns
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < n; r += nwarps) {
    double acc = 0.;
    for (int c = lane; c < nev; c += 32) acc += Z[(size_t)r * ldz + c] * w[c];
    acc = warp_sum(acc);
    if (lane == 0) t[r] = t[r] * (d ? d[r] : 1.) + acc;
  }
}
__global__ void __launch_bounds__(256) k_dense_gemv(int m, int n, const double* __restrict__ A, int lda,
                                                    const double* __restrict__ x, double* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= m) return;
  double acc = 0.;
  for (int c = lane; c < n; c += 32) acc += A[(size_t)row * lda + c] * x[c];
  acc = warp_sum(acc);
  if (lane == 0) y[row] = acc;
}
__global__ void k_pointwise(int64_t n, const double* __restrict__ d, double* __restrict__ x) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] *= d[i];
}
__global__ void k_rows_scale(int64_t tot, int ld, const double* __restrict__ d, double* __restrict__ Z) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < tot; i += (int64_t)gridDim.x * blockDim.x) Z[i] *= d[i / ld];
}
__global__ void k_csr_scale_sym(int n, const int64_t* __restrict__ ptr, const int* __restrict__ idx,
                                const double* __restrict__ val, const double* __restrict__ d, double* __restrict__ out) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const double dr = d[r];
    for (int64_t q = ptr[r]; q < ptr[r + 1]; q++) out[q] = dr * val[q] * d[idx[q]];
  }
}
__global__ void k_vals_axpby(int64_t nnz, const double* __restrict__ a, double tau, const double* __restrict__ b,
                             double* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = a[i] - tau * b[i];
}
__global__ void __launch_bounds__(256) k_sum_all(int64_t nnz, const double* __restrict__ v, double* out) {
  double s[1] = {0.};
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) s[0] += v[i];
  block_reduce_atomic<1>(s, out);
}

// ---------------------------------------------------------------------------------------------------------------
// same-pattern value update
// ---------------------------------------------------------------------------------------------------------------
// position of `key` among a[base + j * stride], j < len (ascending), or -1
__device__ __forceinline__ int64_t find_sorted(const int* __restrict__ a, int64_t base, int64_t len, int stride, int key) {
  int64_t lo = 0, hi = len;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[base + mid * stride] < key) lo = mid + 1;
    else hi = mid;
  }
  return (lo < len && a[base + lo * stride] == key) ? base + lo * stride : -1;
}
__global__ void k_update_nodes(int n, const int* __restrict__ perm, const int* __restrict__ gidx, const int* __restrict__ nodes,
                               int* __restrict__ iperm, unsigned long long* cnt) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const int r = perm[k];
    iperm[r] = (int)k;
    if (gidx[k] != nodes[r]) atomicAdd(cnt + UPD_NODES, 1ull);
  }
}
__global__ void k_update_locate_dir(int n, int64_t nnz, const int64_t* __restrict__ ptr, const int* __restrict__ idx,
                                    const double* __restrict__ val, const int* __restrict__ iperm, const int64_t* __restrict__ patPtr,
                                    const int* __restrict__ patIdx, int* __restrict__ hits, double* __restrict__ dir,
                                    unsigned long long* cnt) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const int k = iperm[r];
    const int64_t a = ptr[r], b = ptr[r + 1], p0 = patPtr[k], len = patPtr[k + 1] - p0;
    if (a < 0 || b > nnz || b - a != len) { atomicAdd(cnt + UPD_DIR_ROW, 1ull); continue; }
    for (int64_t t = a; t < b; t++) {
      const int c = idx[t];
      const int64_t q = (c >= 0 && c < n) ? find_sorted(patIdx, p0, len, 1, iperm[c]) : -1;
      if (q < 0) atomicAdd(cnt + UPD_DIR_OUTSIDE, 1ull);
      else if (atomicOr(hits + q, 1) & 1) atomicAdd(cnt + UPD_DIR_DUP, 1ull);
      else dir[q] = val[t];
    }
  }
}
__global__ void k_update_locate_neu(int n, int64_t nnz, const int64_t* __restrict__ ptr, const int* __restrict__ idx,
                                    const double* __restrict__ val, const int* __restrict__ iperm, const int* __restrict__ gidx,
                                    const int64_t* __restrict__ patPtr, const int* __restrict__ patIdx, int* __restrict__ hits,
                                    const int64_t* __restrict__ sliceOff, const int* __restrict__ col, const int* __restrict__ rowLen,
                                    double* __restrict__ neu, int64_t* __restrict__ slot, unsigned char* __restrict__ cover,
                                    unsigned long long* cnt) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const int k = iperm[r];
    const int64_t a = ptr[r], b = ptr[r + 1], p0 = patPtr[k], len = patPtr[k + 1] - p0;
    if (a < 0 || b < a || b > nnz) { atomicAdd(cnt + UPD_NEU_OUTSIDE, 1ull); continue; }
    const int g = gidx[k];  // row of the operator: slice g / 32, lane g % 32, entry j at sliceOff + 32 j + lane
    const int64_t base = slot ? sliceOff[g >> 5] + (g & 31) : 0;
    const int glen = slot ? rowLen[g] : 0;
    for (int64_t t = a; t < b; t++) {
      const int c = idx[t];
      const int kc = (c >= 0 && c < n) ? iperm[c] : -1;
      const int64_t q = kc >= 0 ? find_sorted(patIdx, p0, len, 1, kc) : -1;
      if (q < 0) { atomicAdd(cnt + UPD_NEU_OUTSIDE, 1ull); continue; }
      if (atomicOr(hits + q, 2) & 2) { atomicAdd(cnt + UPD_NEU_DUP, 1ull); continue; }
      if (!slot) { neu[q] = val[t]; continue; }  // no operator lookup (multi-GPU: the operator rows come from the layout)
      const int64_t sl = find_sorted(col, base, glen, 32, gidx[kc]);
      if (sl < 0) { atomicAdd(cnt + UPD_NEU_NOT_IN_A, 1ull); continue; }
      neu[q] = val[t];
      slot[q] = sl;
      cover[sl] = 1;
    }
  }
}
__global__ void k_update_cover(int n, const int64_t* __restrict__ sliceOff, const int* __restrict__ rowLen,
                               const unsigned char* __restrict__ cover, unsigned long long* cnt) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t base = sliceOff[g >> 5] + (g & 31);
    int miss = 0;
    for (int j = 0; j < rowLen[g]; j++) miss += cover[base + 32 * (int64_t)j] == 0;
    if (miss) atomicAdd(cnt, (unsigned long long)miss);
  }
}
// one thread per owned row g: the input row (ptr, idx, val) must have the operator row's length and, position by position,
// its columns (both sorted by local column); its values go to the same slots of `out`
__global__ void k_update_owned_rows(int n, int64_t nnz, const int64_t* __restrict__ ptr, const int* __restrict__ idx,
                                    const double* __restrict__ val, const int64_t* __restrict__ sliceOff, const int* __restrict__ col,
                                    const int* __restrict__ rowLen, double* __restrict__ out, unsigned long long* cnt) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t a = ptr[g], b = ptr[g + 1], base = sliceOff[g >> 5] + (g & 31);
    const int len = rowLen[g];
    if (a < 0 || b > nnz || b - a != len) { atomicAdd(cnt, 1ull); continue; }
    bool same = true;
    for (int j = 0; j < len; j++) {
      const int64_t o = base + 32 * (int64_t)j;
      same = same && idx[a + j] == col[o];
      out[o] = val[a + j];
    }
    if (!same) atomicAdd(cnt, 1ull);
  }
}
__global__ void __launch_bounds__(256) k_update_absmax(int64_t nnz, const double* __restrict__ v, unsigned long long* out) {
  __shared__ unsigned long long sh[8];
  unsigned long long m = 0;  // bit patterns of non-negative doubles order like the values
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) {
    const double a = fabs(v[i]);
    if (a == a) m = max(m, (unsigned long long)__double_as_longlong(a));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) m = max(m, sh[w]);
    atomicMax(out, m);
  }
}
__global__ void k_update_sell_add(int64_t nnz, const int64_t* __restrict__ slot, const double* __restrict__ neu, double* __restrict__ val) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = slot[q];
    if (s >= 0) val[s] += neu[q];
  }
}
__global__ void k_update_robin(int n, const int64_t* __restrict__ ptr, const int* __restrict__ idx, const double* __restrict__ d,
                               const double* __restrict__ dir, const double* __restrict__ neu, double optim, double* __restrict__ rob) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const bool shared = d[k] < 1.;  // d = 1 / multiplicity
    for (int64_t q = ptr[k]; q < ptr[k + 1]; q++)  // (rounded product, then sum: the host's v += optim * vNeu, no FMA)
      rob[q] = (shared && d[idx[q]] < 1.) ? __dadd_rn(dir[q], __dmul_rn(optim, neu[q])) : dir[q];
  }
}

// ---------------------------------------------------------------------------------------------------------------
// blocks of 8 right-hand sides.  Element t of a row-major n x 8 block is column t & 7; every grid stride below is a multiple
// of 8, so a thread stays on the column threadIdx.x & 7.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double coef_of(const Coef8& a, int c) {  // a.v[c] without dynamic indexing (no local memory)
  double v = 0.;
#pragma unroll
  for (int q = 0; q < 8; q++) v = q == c ? a.v[q] : v;
  return v;
}
__global__ void k_pack_cols8(int64_t n, int nc, const double* __restrict__ X, int64_t ldx, double* __restrict__ B) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n * 8; t += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(t & 7);
    B[t] = c < nc ? X[c * ldx + (t >> 3)] : 0.;
  }
}
__global__ void k_unpack_cols8(int64_t n, int nc, const double* __restrict__ B, double* __restrict__ Y, int64_t ldy) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n * 8; t += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(t & 7);
    if (c < nc) Y[c * ldy + (t >> 3)] = B[t];
  }
}
__global__ void k_pull_sum8(int n, const int64_t* __restrict__ ptr, const int64_t* __restrict__ pos, const double* __restrict__ t,
                            double* __restrict__ y) {
  for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < (int64_t)n * 8; u += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = u >> 3;
    const int c = (int)(u & 7);
    double s = 0.;
    for (int64_t e = ptr[g]; e < ptr[g + 1]; e++) s += __ldg(t + pos[e] * 8 + c);
    y[u] = s;
  }
}
// out[c] += sum x_c y_c (and out[8 + c] += sum z_c z_c): lanes l, l ^ 8, l ^ 16, l ^ 24 share a column
template <bool ZZ>
__global__ void __launch_bounds__(256) k_dot_cols8(int64_t tot, const double* __restrict__ x, const double* __restrict__ y,
                                                   const double* __restrict__ z, double* out) {
  __shared__ double sh[2][8][8];
  double a = 0., b = 0.;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < tot; t += (int64_t)gridDim.x * blockDim.x) {
    a += x[t] * y[t];
    if (ZZ) {
      const double zz = z[t];
      b += zz * zz;
    }
  }
  a += __shfl_xor_sync(0xffffffffu, a, 8);
  a += __shfl_xor_sync(0xffffffffu, a, 16);
  if (ZZ) {
    b += __shfl_xor_sync(0xffffffffu, b, 8);
    b += __shfl_xor_sync(0xffffffffu, b, 16);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane < 8) { sh[0][warp][lane] = a; sh[1][warp][lane] = b; }
  __syncthreads();
  if (threadIdx.x < 8) {
    double sa = 0., sb = 0.;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) { sa += sh[0][w][threadIdx.x]; sb += sh[1][w][threadIdx.x]; }
    atomicAdd(out + threadIdx.x, sa);
    if (ZZ) atomicAdd(out + 8 + threadIdx.x, sb);
  }
}
__global__ void k_cg_update8(int64_t tot, Coef8 a, unsigned mask, const double* __restrict__ p, const double* __restrict__ w,
                             double* __restrict__ x, double* __restrict__ r) {
  const int c = threadIdx.x & 7;
  if (!((mask >> c) & 1u)) return;
  const double ac = coef_of(a, c);
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < tot; t += (int64_t)gridDim.x * blockDim.x) {
    x[t] += ac * p[t];
    r[t] -= ac * w[t];
  }
}
__global__ void k_aypx8(int64_t tot, Coef8 b, unsigned mask, const double* __restrict__ z, double* __restrict__ p) {
  const int c = threadIdx.x & 7;
  if (!((mask >> c) & 1u)) return;
  const double bc = coef_of(b, c);
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < tot; t += (int64_t)gridDim.x * blockDim.x)
    p[t] = z[t] + bc * p[t];
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
void SellMatrix::build(const CsrHost& a, cudaStream_t st) {
  n = a.n;
  nnz = a.nnz();
  nslices = (n + 31) / 32;
  std::vector<int64_t> off(nslices + 1, 0);
  for (int s = 0; s < nslices; s++) {
    int64_t w = 0;
    for (int r = s * 32; r < std::min(n, s * 32 + 32); r++) w = std::max<int64_t>(w, a.ptr[r + 1] - a.ptr[r]);
    off[s + 1] = off[s] + w * 32;
  }
  stored = off[nslices];
  std::vector<int> c((size_t)stored);
  std::vector<double> v((size_t)stored, 0.);
  for (int s = 0; s < nslices; s++) {
    const int64_t w = (off[s + 1] - off[s]) / 32;
    for (int l = 0; l < 32; l++) {
      const int r = s * 32 + l;
      const int64_t len = r < n ? a.ptr[r + 1] - a.ptr[r] : 0;
      for (int64_t j = 0; j < w; j++) {
        const int64_t o = off[s] + j * 32 + l;
        if (j < len) { c[o] = a.idx[a.ptr[r] + j]; v[o] = a.val[a.ptr[r] + j]; }
        else { c[o] = r < n ? r : 0; v[o] = 0.; }
      }
    }
  }
  std::vector<int> len(n);
  for (int r = 0; r < n; r++) len[r] = (int)(a.ptr[r + 1] - a.ptr[r]);
  sliceOff.upload(off, st);
  col.upload(c, st);
  val.upload(v, st);
  rowLen.upload(len, st);
  CUDA_CHECK(::geneo::sync_stream(st));
}

void sell_spmv(const SellMatrix& A, const double* x, double* y, cudaStream_t st) {
  const int grid = std::max(1, std::min((A.nslices + 7) / 8, NSM * 8));
  k_sell_spmv<false><<<GENEO_TICK(grid), 256, 0, st>>>(A.n, A.nslices, A.sliceOff.p, A.col.p, A.val.p, x, nullptr, y);
  CUDA_CHECK(cudaGetLastError());
}
void sell_spmv_sub(const SellMatrix& A, const double* x, const double* b, double* y, cudaStream_t st) {
  const int grid = std::max(1, std::min((A.nslices + 7) / 8, NSM * 8));
  k_sell_spmv<true><<<GENEO_TICK(grid), 256, 0, st>>>(A.n, A.nslices, A.sliceOff.p, A.col.p, A.val.p, x, b, y);
  CUDA_CHECK(cudaGetLastError());
}

void sell_spmm8(const SellMatrix& A, const double* X, double* Y, cudaStream_t st) {
  const int grid = std::max(1, std::min((A.nslices + 7) / 8, NSM * 8));
  k_sell_spmm8<<<GENEO_TICK(grid), 256, 0, st>>>(A.n, A.nslices, A.sliceOff.p, A.col.p, A.val.p, X, Y);
  CUDA_CHECK(cudaGetLastError());
}
void scatter_rows8(int n, const int* idx, const double* Z, int ldz, int c0, int nc, double* G, cudaStream_t st) {
  if (n) k_scatter_rows8<<<GENEO_TICK(grid_for((int64_t)n * 8, 256)), 256, 0, st>>>(n, idx, Z, ldz, c0, nc, G);
}
void gather_rows8(int n, const int* idx, const double* G, double* out, cudaStream_t st) {
  if (n) k_gather_rows8<<<GENEO_TICK(grid_for((int64_t)n * 8, 256)), 256, 0, st>>>(n, idx, G, out);
}

void CsrDev::upload_pattern(const CsrHost& a, cudaStream_t st) {
  n = a.n;
  nnz = a.nnz();
  ptr.upload(a.ptr, st);
  idx.upload(a.idx, st);
  val.upload(a.val, st);
  CUDA_CHECK(::geneo::sync_stream(st));
}

void csr_spmm(int n, const int64_t* ptr, const int* idx, const double* val, const double* X, int ldx, double* Y, int ldy,
              int nr, cudaStream_t st) {
  const int64_t tot = (int64_t)n * nr;
  const int grid = (int)((tot + 255) / 256);
  switch (nr) {
    case 1: k_csr_spmm<1><<<GENEO_TICK(grid), 256, 0, st>>>(n, ptr, idx, val, X, ldx, Y, ldy); break;
    case 2: k_csr_spmm<2><<<GENEO_TICK(grid), 256, 0, st>>>(n, ptr, idx, val, X, ldx, Y, ldy); break;
    case 4: k_csr_spmm<4><<<GENEO_TICK(grid), 256, 0, st>>>(n, ptr, idx, val, X, ldx, Y, ldy); break;
    case 8: k_csr_spmm<8><<<GENEO_TICK(grid), 256, 0, st>>>(n, ptr, idx, val, X, ldx, Y, ldy); break;
    case 16: k_csr_spmm<16><<<GENEO_TICK(grid), 256, 0, st>>>(n, ptr, idx, val, X, ldx, Y, ldy); break;
    case 32: k_csr_spmm<32><<<GENEO_TICK(grid), 256, 0, st>>>(n, ptr, idx, val, X, ldx, Y, ldy); break;
    default: GENEO_CHECK(false, "csr_spmm: nr must be a power of two <= 32");
  }
  CUDA_CHECK(cudaGetLastError());
}

void vec_dot(int n, const double* x, const double* y, double* out, cudaStream_t st) {
  CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(double), st));
  k_dot<<<GENEO_TICK(grid_for(n, 256, 4)), 256, 0, st>>>(n, x, y, out);
}
void vec_dot2(int n, const double* x, const double* y, const double* z, double* out, cudaStream_t st) {
  CUDA_CHECK(cudaMemsetAsync(out, 0, 2 * sizeof(double), st));
  k_dot2<<<GENEO_TICK(grid_for(n, 256, 4)), 256, 0, st>>>(n, x, y, z, out);
}
void vec_axpy(int n, double a, const double* x, double* y, cudaStream_t st) { k_axpy<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, a, x, y); }
void vec_aypx(int n, double a, const double* x, double* y, cudaStream_t st) { k_axpby<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, 1., x, a, y); }
void vec_axpby(int n, double a, const double* x, double b, double* y, cudaStream_t st) { k_axpby<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, a, x, b, y); }
void vec_cg_update(int n, double a, const double* p, const double* w, double* x, double* r, cudaStream_t st) {
  k_cg_update<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, a, p, w, x, r);
}
void vec_scale(int n, double a, double* x, cudaStream_t st) { k_scale<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, a, x); }
void vec_set(int n, double a, double* x, cudaStream_t st) { k_set<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, a, 0., x); }
void vec_iota(int n, double first, double* x, cudaStream_t st) { k_set<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, first, 1., x); }
void vec_mdot(int n, int nv, const double* V, int64_t ldv, const double* w, double* out, cudaStream_t st) {
  CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(double) * (size_t)((nv + 3) / 4 * 4), st));
  k_mdot<<<GENEO_TICK(grid_for(n, 256, 4)), 256, 0, st>>>(n, nv, V, ldv, w, out);
}
void vec_maxpy(int n, int nv, const double* V, int64_t ldv, const double* coef, double* w, cudaStream_t st) {
  k_maxpy<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, nv, V, ldv, coef, w);
}
void gather_rows(int64_t cnt, const int* idx, const double* scale, const double* x, double* out, cudaStream_t st) {
  if (cnt) k_gather<<<GENEO_TICK(grid_for(cnt, 256)), 256, 0, st>>>(cnt, idx, scale, x, out);
}
void pull_sum(int n, const int64_t* ptr, const int64_t* pos, const double* t, double* y, bool accumulate, cudaStream_t st) {
  k_pull_sum<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, ptr, pos, t, y, accumulate);
}
void ts_gram(int n, const double* X, int ldx, int p, const double* Y, int ldy, int q, double* G, int ldg, cudaStream_t st) {
  if (n <= 0 || p <= 0 || q <= 0) return;
  const bool wide = q > 8;  // two 8-column tiles of Y per CTA: X is read once for a block of 16
  const int tp = (p + TG_PCOLS - 1) / TG_PCOLS, tq = wide ? (q + 15) / 16 : 1;
  int nz = std::max(1, std::min((n + 255) / 256, std::max(1, NSM * 8 / (tp * tq))));
  int rowsPerCta = ((n + nz - 1) / nz + 31) / 32 * 32;
  nz = (n + rowsPerCta - 1) / rowsPerCta;
  dim3 grid(tp, tq, nz);
  if (wide) k_ts_gram<2><<<GENEO_TICK(grid), 256, 0, st>>>(n, X, ldx, p, Y, ldy, q, G, ldg, rowsPerCta);
  else k_ts_gram<1><<<GENEO_TICK(grid), 256, 0, st>>>(n, X, ldx, p, Y, ldy, q, G, ldg, rowsPerCta);
  CUDA_CHECK(cudaGetLastError());
}
void ts_update(int n, const double* Q, int ldq, int p, const double* C, int ldc, int q, double* W, int ldw, double alpha,
               double beta, cudaStream_t st) {
  // C chunk (192 x 8 or 96 x 16 doubles) + the Q tile stay below 48 KB of shared memory
  const int grid = (n + TSU_ROWS - 1) / TSU_ROWS;
  if (n <= 0) return;
  for (int j0 = 0; j0 < q;) {
    const bool wide = q - j0 > 8;  // 16 columns per pass: Q is read once for a block of 16
    const int QW = wide ? 16 : 8, PCHUNK = wide ? 96 : 192;
    const int qc = std::min(QW, q - j0);
    for (int p0 = 0; p0 < std::max(p, 1); p0 += PCHUNK) {
      const int pc = std::max(0, std::min(PCHUNK, p - p0));
      const size_t smem = ((size_t)pc * QW + (size_t)TSU_ROWS * (TSU_COLS + 1)) * sizeof(double);
      if (wide) k_ts_update<16><<<GENEO_TICK(grid), TSU_ROWS, smem, st>>>(n, Q + p0, ldq, pc, C + (size_t)p0 * ldc + j0, ldc, qc, W + j0, ldw,
                                                                          alpha, p0 == 0 ? beta : 1.);
      else k_ts_update<8><<<GENEO_TICK(grid), TSU_ROWS, smem, st>>>(n, Q + p0, ldq, pc, C + (size_t)p0 * ldc + j0, ldc, qc, W + j0, ldw, alpha,
                                                                    p0 == 0 ? beta : 1.);
    }
    j0 += QW;
  }
  CUDA_CHECK(cudaGetLastError());
}
void zt_x(int n, int nev, const double* Z, int ldz, const double* x, double* w, cudaStream_t st) {
  if (nev == 0) return;
  int nevPad = 1;
  while (nevPad < nev) nevPad <<= 1;
  nevPad = std::min(nevPad, 256);
  const int rstride = 256 / nevPad;
  const int grid = std::max(1, std::min((n + rstride * 8 - 1) / (rstride * 8), NSM * 4));
  k_zt_x<<<GENEO_TICK(grid), 256, 0, st>>>(n, nev, Z, ldz, x, w);
  CUDA_CHECK(cudaGetLastError());
}
void z_w_add(int n, int nev, const double* Z, int ldz, const double* w, const double* d, double* t, cudaStream_t st) {
  const int grid = std::max(1, std::min((n + 7) / 8, NSM * 8));
  k_z_w_add<<<GENEO_TICK(grid), 256, 0, st>>>(n, nev, Z, ldz, w, d, t);
  CUDA_CHECK(cudaGetLastError());
}
void dense_gemv(int m, int n, const double* A, int lda, const double* x, double* y, cudaStream_t st) {
  if (m == 0) return;
  k_dense_gemv<<<GENEO_TICK((m + 7) / 8), 256, 0, st>>>(m, n, A, lda, x, y);
  CUDA_CHECK(cudaGetLastError());
}
__global__ void k_copy_cols(int64_t n, const double* __restrict__ src, int lds, double* __restrict__ dst, int ldd, int ncols) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n * ncols; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / ncols;
    const int j = (int)(t % ncols);
    dst[r * ldd + j] = src[r * lds + j];
  }
}
void copy_cols(int64_t n, const double* src, int lds, double* dst, int ldd, int ncols, cudaStream_t st) {
  if (n * ncols == 0) return;
  k_copy_cols<<<GENEO_TICK(grid_for(n * ncols, 256)), 256, 0, st>>>(n, src, lds, dst, ldd, ncols);
  CUDA_CHECK(cudaGetLastError());
}
void vec_pointwise(int64_t n, const double* d, double* x, cudaStream_t st) { k_pointwise<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, d, x); }
void rows_scale(int n, int ld, const double* d, double* Z, cudaStream_t st) {
  const int64_t tot = (int64_t)n * ld;
  if (tot) k_rows_scale<<<GENEO_TICK(grid_for(tot, 256)), 256, 0, st>>>(tot, ld, d, Z);
}
void csr_scale_sym(int n, const int64_t* ptr, const int* idx, const double* val, const double* d, double* out, cudaStream_t st) {
  k_csr_scale_sym<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, ptr, idx, val, d, out);
}
void vals_axpby(int64_t nnz, const double* a, double tau, const double* b, double* out, cudaStream_t st) {
  k_vals_axpby<<<GENEO_TICK(grid_for(nnz, 256)), 256, 0, st>>>(nnz, a, tau, b, out);
}
void csr_sum_all(int64_t nnz, const double* val, double* out, cudaStream_t st) {
  CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(double), st));
  k_sum_all<<<GENEO_TICK(grid_for(nnz, 256, 4)), 256, 0, st>>>(nnz, val, out);
}

void update_nodes(int n, const int* perm, const int* gidx, const int* nodes, int* iperm, unsigned long long* cnt, cudaStream_t st) {
  k_update_nodes<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, perm, gidx, nodes, iperm, cnt);
  CUDA_CHECK(cudaGetLastError());
}
void update_locate_dir(int n, int64_t nnz, const int64_t* ptr, const int* idx, const double* val, const int* iperm,
                       const int64_t* patPtr, const int* patIdx, int* hits, double* dir, unsigned long long* cnt, cudaStream_t st) {
  k_update_locate_dir<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, nnz, ptr, idx, val, iperm, patPtr, patIdx, hits, dir, cnt);
  CUDA_CHECK(cudaGetLastError());
}
void update_locate_neu(int n, int64_t nnz, const int64_t* ptr, const int* idx, const double* val, const int* iperm, const int* gidx,
                       const int64_t* patPtr, const int* patIdx, int* hits, const SellMatrix& A, double* neu, int64_t* slot,
                       unsigned char* cover, unsigned long long* cnt, cudaStream_t st) {
  k_update_locate_neu<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, nnz, ptr, idx, val, iperm, gidx, patPtr, patIdx, hits,
                                                                    A.sliceOff.p, A.col.p, A.rowLen.p, neu, slot, cover, cnt);
  CUDA_CHECK(cudaGetLastError());
}
void update_cover_check(const SellMatrix& A, const unsigned char* cover, unsigned long long* cnt, cudaStream_t st) {
  k_update_cover<<<GENEO_TICK(grid_for(A.n, 256)), 256, 0, st>>>(A.n, A.sliceOff.p, A.rowLen.p, cover, cnt);
  CUDA_CHECK(cudaGetLastError());
}
void update_owned_rows(const SellMatrix& A, int64_t nnz, const int64_t* ptr, const int* idx, const double* val, double* out,
                       unsigned long long* cnt, cudaStream_t st) {
  k_update_owned_rows<<<GENEO_TICK(grid_for(A.n, 256)), 256, 0, st>>>(A.n, nnz, ptr, idx, val, A.sliceOff.p, A.col.p, A.rowLen.p, out, cnt);
  CUDA_CHECK(cudaGetLastError());
}
void update_absmax(int64_t nnz, const double* v, unsigned long long* out, cudaStream_t st) {
  k_update_absmax<<<GENEO_TICK(grid_for(nnz, 256, 4)), 256, 0, st>>>(nnz, v, out);
  CUDA_CHECK(cudaGetLastError());
}
void update_sell_add(int64_t nnz, const int64_t* slot, const double* neu, SellMatrix& A, cudaStream_t st) {
  k_update_sell_add<<<GENEO_TICK(grid_for(nnz, 256)), 256, 0, st>>>(nnz, slot, neu, A.val.p);
  CUDA_CHECK(cudaGetLastError());
}
void update_robin(int n, const int64_t* ptr, const int* idx, const double* d, const double* dir, const double* neu, double optim,
                  double* rob, cudaStream_t st) {
  k_update_robin<<<GENEO_TICK(grid_for(n, 256)), 256, 0, st>>>(n, ptr, idx, d, dir, neu, optim, rob);
  CUDA_CHECK(cudaGetLastError());
}

void pack_cols8(int64_t n, int nc, const double* X, int64_t ldx, double* B, cudaStream_t st) {
  if (n == 0) return;
  k_pack_cols8<<<GENEO_TICK(grid_for(n * 8, 256)), 256, 0, st>>>(n, nc, X, ldx, B);
  CUDA_CHECK(cudaGetLastError());
}
void unpack_cols8(int64_t n, int nc, const double* B, double* Y, int64_t ldy, cudaStream_t st) {
  if (n == 0) return;
  k_unpack_cols8<<<GENEO_TICK(grid_for(n * 8, 256)), 256, 0, st>>>(n, nc, B, Y, ldy);
  CUDA_CHECK(cudaGetLastError());
}
void pull_sum8(int n, const int64_t* ptr, const int64_t* pos, const double* t, double* y, cudaStream_t st) {
  if (n == 0) return;
  k_pull_sum8<<<GENEO_TICK(grid_for((int64_t)n * 8, 256)), 256, 0, st>>>(n, ptr, pos, t, y);
  CUDA_CHECK(cudaGetLastError());
}
void dot_cols8(int n, const double* x, const double* y, const double* z, double* out, cudaStream_t st) {
  CUDA_CHECK(cudaMemsetAsync(out, 0, (z ? 16 : 8) * sizeof(double), st));
  if (n == 0) return;
  const int64_t tot = (int64_t)n * 8;
  if (z) k_dot_cols8<true><<<GENEO_TICK(grid_for(tot, 256, 4)), 256, 0, st>>>(tot, x, y, z, out);
  else k_dot_cols8<false><<<GENEO_TICK(grid_for(tot, 256, 4)), 256, 0, st>>>(tot, x, y, nullptr, out);
  CUDA_CHECK(cudaGetLastError());
}
void cg_update8(int n, Coef8 a, unsigned mask, const double* p, const double* w, double* x, double* r, cudaStream_t st) {
  if (n == 0 || mask == 0) return;
  const int64_t tot = (int64_t)n * 8;
  k_cg_update8<<<GENEO_TICK(grid_for(tot, 256)), 256, 0, st>>>(tot, a, mask, p, w, x, r);
  CUDA_CHECK(cudaGetLastError());
}
void aypx8(int n, Coef8 b, unsigned mask, const double* z, double* p, cudaStream_t st) {
  if (n == 0 || mask == 0) return;
  const int64_t tot = (int64_t)n * 8;
  k_aypx8<<<GENEO_TICK(grid_for(tot, 256)), 256, 0, st>>>(tot, b, mask, z, p);
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace geneo
