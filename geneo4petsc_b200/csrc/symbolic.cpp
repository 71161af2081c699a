// symbolic.cpp -- see symbolic.hpp.  Host only.
#include "symbolic.hpp"

#include <dlfcn.h>

#include <algorithm>
#include <numeric>
#include <string>
#include <thread>

#include "common.hpp"

namespace geneo {

typedef int64_t midx_t;
extern "C" int METIS_SetDefaultOptions(midx_t* options);
extern "C" int METIS_NodeND(midx_t* nvtxs, midx_t* xadj, midx_t* adjncy, midx_t* vwgt, midx_t* options, midx_t* perm,
                            midx_t* iperm);

extern "C" int METIS_ComputeVertexSeparator(midx_t* nvtxs, midx_t* xadj, midx_t* adjncy, midx_t* vwgt, midx_t* options,
                                           midx_t* sepsize, midx_t* part);

// ---------------------------------------------------------------------------------------------------------------------
// METIS draws its random permutations from rand(): glibc serialises rand() behind one process-wide lock, so nested
// dissections of different subdomains running on different threads spend most of their time in futex calls (measured:
// 8 concurrent orderings of 10^6-vertex graphs take as long as 8 serial ones, 64 % system time) -- and they perturb each
// other's random streams.  Inside the nested-dissection calls of THIS library rand()/srand() resolve (hidden visibility,
// bound at link time, nothing exported) to a thread-local generator; everywhere else -- in particular in the k-way mesh
// partition whose result is pinned by the reference's goldens -- they forward to the C library.
// ---------------------------------------------------------------------------------------------------------------------
namespace {
thread_local bool t_nd_rng = false;
thread_local uint64_t t_nd_state = 0x9E3779B97F4A7C15ull;
struct NdRngScope {
  bool old;
  NdRngScope() : old(t_nd_rng) { t_nd_rng = true; }
  ~NdRngScope() { t_nd_rng = old; }
};
}  // namespace
extern "C" __attribute__((visibility("hidden"))) int rand(void) {
  if (!t_nd_rng) {
    static int (*real)(void) = reinterpret_cast<int (*)(void)>(dlsym(RTLD_DEFAULT, "rand"));
    return real();
  }
  uint64_t x = t_nd_state;  // xorshift64*
  x ^= x >> 12; x ^= x << 25; x ^= x >> 27;
  t_nd_state = x;
  return (int)((x * 2685821657736338717ull) >> 33);  // 31 bits, like RAND_MAX = 2^31 - 1
}
extern "C" __attribute__((visibility("hidden"))) void srand(unsigned seed) {
  if (!t_nd_rng) {
    static void (*real)(unsigned) = reinterpret_cast<void (*)(unsigned)>(dlsym(RTLD_DEFAULT, "srand"));
    real(seed);
    return;
  }
  t_nd_state = ((uint64_t)seed + 1) * 0x9E3779B97F4A7C15ull;
}

namespace {

struct NdGraph { std::vector<midx_t> xadj, adj; int n() const { return (int)xadj.size() - 1; } };

// Nested dissection with the top `depth` levels done here so that the two halves can be ordered concurrently
// (METIS_NodeND is serial; its own recursion does exactly this: separator last, halves recursively).  order: new -> old.
void nd_recursive(NdGraph& g, int depth, std::vector<int>& order) {
  NdRngScope rngScope;
  const int n = g.n();
  midx_t options[40];
  METIS_SetDefaultOptions(options);
  midx_t nv = n;
  if (depth <= 0 || n < 20000) {
    std::vector<midx_t> p(n), ip(n);
    order.resize(n);
    if (g.adj.empty()) { std::iota(order.begin(), order.end(), 0); return; }
    const double tNd = now_s();
    const int rc = METIS_NodeND(&nv, g.xadj.data(), g.adj.data(), NULL, options, p.data(), ip.data());
    GENEO_CHECK(rc == 1, "METIS_NodeND failed");
    if (getenv("GENEO_ND_TIMING")) fprintf(stderr, "nd: leaf NodeND of %d vertices: %.3f s\n", n, now_s() - tNd);
    for (int i = 0; i < n; i++) order[i] = (int)p[i];
    return;
  }
  std::vector<midx_t> part(n);
  midx_t sep = 0;
  const double tSep = now_s();
  const int rc = METIS_ComputeVertexSeparator(&nv, g.xadj.data(), g.adj.data(), NULL, options, &sep, part.data());
  GENEO_CHECK(rc == 1, "METIS_ComputeVertexSeparator failed");
  if (getenv("GENEO_ND_TIMING")) fprintf(stderr, "nd: separator of %d vertices (depth left %d): %d vertices, %.3f s\n", n, depth, (int)sep, now_s() - tSep);
  std::vector<int> ids[3];
  for (int i = 0; i < n; i++) ids[part[i] < 0 || part[i] > 2 ? 2 : part[i]].push_back(i);
  if (ids[0].empty() || ids[1].empty()) { nd_recursive(g, 0, order); return; }
  std::vector<int> loc(n, -1);
  NdGraph sub[2];
  for (int s = 0; s < 2; s++) {
    for (size_t t = 0; t < ids[s].size(); t++) loc[ids[s][t]] = (int)t;
    sub[s].xadj.assign(ids[s].size() + 1, 0);
    for (size_t t = 0; t < ids[s].size(); t++) {
      const int v = ids[s][t];
      for (midx_t e = g.xadj[v]; e < g.xadj[v + 1]; e++)
        if (part[g.adj[e]] == s) sub[s].adj.push_back(loc[g.adj[e]]);
      sub[s].xadj[t + 1] = (midx_t)sub[s].adj.size();
    }
  }
  { NdGraph().xadj.swap(g.xadj); std::vector<midx_t>().swap(g.adj); }  // the parent graph is no longer needed
  std::vector<int> ord[2];
  std::string err;
  std::thread th([&]() { try { nd_recursive(sub[0], depth - 1, ord[0]); } catch (std::exception& e) { err = e.what(); } });
  nd_recursive(sub[1], depth - 1, ord[1]);
  th.join();
  GENEO_CHECK(err.empty(), err);
  order.clear();
  order.reserve(n);
  for (int s = 0; s < 2; s++)
    for (int v : ord[s]) order.push_back(ids[s][v]);
  for (int v : ids[2]) order.push_back(v);
}

// Elimination tree of P A P^T (Liu, path compression).  Row j of the permuted matrix = row perm[j] of the input.
void etree(int n, const int64_t* ptr, const int* idx, const std::vector<int>& perm, const std::vector<int>& iperm,
           std::vector<int>& parent) {
  parent.assign(n, -1);
  std::vector<int> anc(n, -1);
  for (int j = 0; j < n; j++) {
    const int jo = perm[j];
    for (int64_t t = ptr[jo]; t < ptr[jo + 1]; t++) {
      int i = iperm[idx[t]];
      while (i != -1 && i < j) {
        int next = anc[i];
        anc[i] = j;
        if (next == -1) parent[i] = j;
        i = next;
      }
    }
  }
}

void postorder(int n, const std::vector<int>& parent, std::vector<int>& post) {
  std::vector<int> head(n, -1), next(n, -1), stack;
  for (int j = n - 1; j >= 0; j--)
    if (parent[j] != -1) { next[j] = head[parent[j]]; head[parent[j]] = j; }
  post.clear();
  post.reserve(n);
  stack.reserve(64);
  for (int r = 0; r < n; r++) {
    if (parent[r] != -1) continue;
    stack.push_back(r);
    while (!stack.empty()) {
      int p = stack.back();
      int c = head[p];
      if (c == -1) { post.push_back(p); stack.pop_back(); }
      else { head[p] = next[c]; stack.push_back(c); }
    }
  }
}

// Column counts of the Cholesky factor (Gilbert, Ng, Peyton 1994), skeleton-matrix / row-subtree leaves.
void colcounts(int n, const int64_t* ptr, const int* idx, const std::vector<int>& perm, const std::vector<int>& iperm,
               const std::vector<int>& parent, const std::vector<int>& post, std::vector<int>& cc) {
  std::vector<int> first(n, -1), maxfirst(n, -1), prevleaf(n, -1), anc(n);
  std::vector<int64_t> delta(n, 0);
  for (int k = 0; k < n; k++) {
    int j = post[k];
    delta[j] = (first[j] == -1) ? 1 : 0;  // j is a leaf of the etree
    for (; j != -1 && first[j] == -1; j = parent[j]) first[j] = k;
  }
  for (int i = 0; i < n; i++) anc[i] = i;
  for (int k = 0; k < n; k++) {
    const int j = post[k];
    if (parent[j] != -1) delta[parent[j]]--;
    const int jo = perm[j];
    for (int64_t t = ptr[jo]; t < ptr[jo + 1]; t++) {
      const int i = iperm[idx[t]];
      if (i <= j || first[j] <= maxfirst[i]) continue;  // j is not a leaf of the i-th row subtree
      maxfirst[i] = first[j];
      const int jprev = prevleaf[i];
      prevleaf[i] = j;
      if (jprev == -1) { delta[j]++; continue; }  // first leaf
      int q = jprev;
      while (q != anc[q]) q = anc[q];
      for (int s = jprev; s != q;) { int sp = anc[s]; anc[s] = q; s = sp; }
      delta[j]++;
      delta[q]--;  // q = least common ancestor of jprev and j
    }
    if (parent[j] != -1) anc[j] = parent[j];
  }
  for (int k = 0; k < n; k++) {  // accumulate up the tree in postorder (children before parents)
    const int j = post[k];
    if (parent[j] != -1) delta[parent[j]] += delta[j];
  }
  cc.resize(n);
  for (int j = 0; j < n; j++) cc[j] = (int)delta[j];
}

}  // namespace

void box_reference_ordering(const int dims[3], int nst, const int* stencil, int ndDepth, std::vector<int>& rank) {
  const int64_t n64 = (int64_t)dims[0] * dims[1] * dims[2];
  GENEO_CHECK(n64 > 0 && n64 < 2147483647, "reference box: bad dimensions");
  const int n = (int)n64;
  // symmetric closure of the stencil, without the origin and without duplicates
  std::vector<int> off;
  auto have = [&](int a, int b, int c) {
    for (size_t t = 0; t < off.size(); t += 3) if (off[t] == a && off[t + 1] == b && off[t + 2] == c) return true;
    return false;
  };
  for (int t = 0; t < nst; t++)
    for (int sg = -1; sg <= 1; sg += 2) {
      const int a = sg * stencil[3 * t], b = sg * stencil[3 * t + 1], c = sg * stencil[3 * t + 2];
      if ((a | b | c) == 0 || have(a, b, c)) continue;
      off.push_back(a); off.push_back(b); off.push_back(c);
    }
  NdGraph g;
  g.xadj.assign((size_t)n + 1, 0);
  g.adj.reserve((size_t)n * (off.size() / 3));
  for (int z = 0; z < dims[2]; z++)
    for (int y = 0; y < dims[1]; y++)
      for (int x = 0; x < dims[0]; x++) {
        const int v = x + dims[0] * (y + dims[1] * z);
        for (size_t t = 0; t < off.size(); t += 3) {
          const int a = x + off[t], b = y + off[t + 1], c = z + off[t + 2];
          if (a < 0 || a >= dims[0] || b < 0 || b >= dims[1] || c < 0 || c >= dims[2]) continue;
          g.adj.push_back(a + dims[0] * (b + dims[1] * c));
        }
        g.xadj[(size_t)v + 1] = (midx_t)g.adj.size();
      }
  std::vector<int> order;
  if (g.adj.empty()) { order.resize(n); std::iota(order.begin(), order.end(), 0); }
  else nd_recursive(g, ndDepth, order);
  GENEO_CHECK((int)order.size() == n, "reference box: nested dissection lost vertices");
  rank.assign(n, 0);
  for (int i = 0; i < n; i++) rank[order[i]] = i;
}

void symbolic_analyze(int n, const int64_t* ptr, const int* idx, const SymbolicOptions& opt, Symbolic& S) {
  const double tStart = now_s();
  (void)tStart;
  S = Symbolic();
  S.n = n;
  S.nb = opt.nb;
  GENEO_CHECK(n > 0, "empty matrix");
  GENEO_CHECK(opt.nb >= 1 && opt.nb <= 128, "panel width must be in [1,128]");

  // ---- 1. fill-reducing ordering ------------------------------------------------------------------------------------
  std::vector<int> perm(n), iperm(n);
  bool useMetis = opt.ordering == 1 && n > 32;
  if (useMetis) {
    std::vector<midx_t> xadj(n + 1, 0), adj;
    adj.reserve(ptr[n]);
    for (int i = 0; i < n; i++) {
      for (int64_t t = ptr[i]; t < ptr[i + 1]; t++)
        if (idx[t] != i) adj.push_back(idx[t]);
      xadj[i + 1] = (midx_t)adj.size();
    }
    if (adj.empty()) useMetis = false;
    else {
      NdGraph g;
      g.xadj.swap(xadj);
      g.adj.swap(adj);
      std::vector<int> order;
      nd_recursive(g, opt.ndDepth, order);
      GENEO_CHECK((int)order.size() == n, "nested dissection lost vertices");
      for (int i = 0; i < n; i++) { perm[i] = order[i]; iperm[order[i]] = i; }
    }
  }
  if (opt.ordering == 3) {
    GENEO_CHECK(opt.userPerm != nullptr, "ordering 3 needs a permutation");
    std::fill(iperm.begin(), iperm.end(), -1);
    for (int i = 0; i < n; i++) {
      const int o = opt.userPerm[i];
      GENEO_CHECK(o >= 0 && o < n && iperm[o] < 0, "user permutation is not a permutation");
      perm[i] = o; iperm[o] = i;
    }
  } else if (!useMetis) { std::iota(perm.begin(), perm.end(), 0); std::iota(iperm.begin(), iperm.end(), 0); }

  const bool tm = getenv("GENEO_SYM_TIMING") != nullptr;
  double tq = now_s();
  auto lap = [&](const char* what) { if (tm) { const double t = now_s(); fprintf(stderr, "symbolic n=%d %s %.3fs\n", n, what, t - tq); tq = t; } };
  lap("ordering");
  // ---- 2. etree, postorder, column counts; relabel so that the ordering IS a postorder -----------------------------
  std::vector<int> parent, post, cc;
  etree(n, ptr, idx, perm, iperm, parent);
  postorder(n, parent, post);
  GENEO_CHECK((int)post.size() == n, "postorder failed");
  colcounts(n, ptr, idx, perm, iperm, parent, post, cc);
  {
    std::vector<int> ipost(n), perm2(n), parent2(n), cc2(n);
    for (int k = 0; k < n; k++) ipost[post[k]] = k;
    for (int k = 0; k < n; k++) {
      perm2[k] = perm[post[k]];
      parent2[k] = parent[post[k]] == -1 ? -1 : ipost[parent[post[k]]];
      cc2[k] = cc[post[k]];
    }
    perm.swap(perm2); parent.swap(parent2); cc.swap(cc2);
    for (int k = 0; k < n; k++) iperm[perm[k]] = k;
  }

  lap("etree+colcounts");
  // ---- 3. supernodes (maximal: same structure as the next column) + relaxed amalgamation ----------------------------
  std::vector<int> snFirst, snK, snH;
  for (int j = 0; j < n; j++) {
    bool join = j > 0 && parent[j - 1] == j && cc[j] == cc[j - 1] - 1;
    if (join) snK.back()++;
    else { snFirst.push_back(j); snK.push_back(1); snH.push_back(cc[j]); }
  }
  int ns = (int)snFirst.size();
  std::vector<int> snOf(n);
  for (int s = 0; s < ns; s++)
    for (int j = snFirst[s]; j < snFirst[s] + snK[s]; j++) snOf[j] = s;
  std::vector<int> snParent(ns);
  for (int s = 0; s < ns; s++) {
    int last = snFirst[s] + snK[s] - 1;
    snParent[s] = parent[last] == -1 ? -1 : snOf[parent[last]];
  }
  std::vector<int> alive(ns, 1);
  if (opt.amalgamate) {
    std::vector<int> prev(ns), mergedInto(ns, -1);
    std::vector<double> zeros(ns, 0.);
    for (int s = 0; s < ns; s++) prev[s] = s - 1;
    auto rootOf = [&](int s) { while (s != -1 && mergedInto[s] != -1) s = mergedInto[s]; return s; };
    // columns in the whole subtree of every supernode: small subtrees become ONE dense front (the GPU prefers a few
    // thousand fronts of a few KB to hundreds of thousands of tiny ones; they hold ~5 % of the factor)
    std::vector<int> subCols(ns, 0);
    for (int s = 0; s < ns; s++) {
      subCols[s] += snK[s];
      if (snParent[s] != -1) subCols[snParent[s]] += subCols[s];
    }
    for (int s = 0; s < ns; s++) {
      while (true) {
        int c = prev[s];
        if (c < 0) break;
        if (rootOf(snParent[c]) != s) break;  // the supernode just before s is not one of its children
        const double kc = snK[c], hc = snH[c], ks = snK[s], hs = snH[s];
        const double newk = kc + ks, newh = kc + hs;
        const double z = zeros[c] + zeros[s] + kc * (newh - hc);
        const double total = newk * newh - newk * (newk - 1.) / 2.;
        const double frac = z / total;
        bool merge = (newk <= 4) || (newk <= 16 && frac < 0.8) || (newk <= 48 && frac < 0.1) || (frac < 0.05) ||
                     (subCols[s] <= opt.subtreeCols);
        if (!merge) break;
        snFirst[s] = snFirst[c]; snK[s] = (int)newk; snH[s] = (int)newh; zeros[s] = z;
        alive[c] = 0; mergedInto[c] = s; prev[s] = prev[c];
      }
    }
    for (int s = 0; s < ns; s++)
      if (alive[s]) snParent[s] = rootOf(snParent[s]);
  }
  // compact
  std::vector<int> newId(ns, -1), fFirst, fK, fPar;
  for (int s = 0; s < ns; s++)
    if (alive[s]) { newId[s] = (int)fFirst.size(); fFirst.push_back(snFirst[s]); fK.push_back(snK[s]); }
  for (int s = 0; s < ns; s++)
    if (alive[s]) fPar.push_back(snParent[s] == -1 ? -1 : newId[snParent[s]]);
  ns = (int)fFirst.size();
  S.nsuper = ns;
  for (int s = 0; s < ns; s++)
    for (int j = fFirst[s]; j < fFirst[s] + fK[s]; j++) snOf[j] = s;

  // ---- 4. row structure of every supernode (own columns, then the sorted union of A-entries and children rows) -------
  std::vector<int64_t> snRowOff(ns + 1, 0);
  std::vector<int>& rowIdx = S.rowIdx;
  {
    std::vector<int> chHead(ns, -1), chNext(ns, -1), mark(n, -1);
    for (int s = ns - 1; s >= 0; s--)
      if (fPar[s] != -1) { chNext[s] = chHead[fPar[s]]; chHead[fPar[s]] = s; }
    std::vector<int> below;
    for (int s = 0; s < ns; s++) {
      const int c0 = fFirst[s], c1 = c0 + fK[s];
      below.clear();
      for (int j = c0; j < c1; j++) {
        const int jo = perm[j];
        for (int64_t t = ptr[jo]; t < ptr[jo + 1]; t++) {
          const int i = iperm[idx[t]];
          if (i >= c1 && mark[i] != s) { mark[i] = s; below.push_back(i); }
        }
      }
      for (int c = chHead[s]; c != -1; c = chNext[c]) {
        for (int64_t t = snRowOff[c] + fK[c]; t < snRowOff[c + 1]; t++) {
          const int i = rowIdx[t];
          if (i >= c1 && mark[i] != s) { mark[i] = s; below.push_back(i); }
        }
      }
      std::sort(below.begin(), below.end());
      for (int j = c0; j < c1; j++) rowIdx.push_back(j);
      rowIdx.insert(rowIdx.end(), below.begin(), below.end());
      snRowOff[s + 1] = (int64_t)rowIdx.size();
    }
  }
  S.nnzRowIdx = (int64_t)rowIdx.size();

  lap("supernodes+rowidx");
  // ---- 5. cut supernodes into panels (fronts) ------------------------------------------------------------------------
  const int NB = opt.nb;
  std::vector<int> firstFrontOfSn(ns), lastFrontOfSn(ns);
  S.frontOfCol.assign(n, -1);
  for (int s = 0; s < ns; s++) {
    const int hs = (int)(snRowOff[s + 1] - snRowOff[s]);
    const int np = (fK[s] + NB - 1) / NB;
    firstFrontOfSn[s] = (int)S.fronts.size();
    for (int p = 0; p < np; p++) {
      Front f;
      const int off = p * NB;
      f.col0 = fFirst[s] + off;
      f.k = std::min(NB, fK[s] - off);
      f.h = hs - off;
      f.ld = (f.h + 1) & ~1;
      f.rowOff = snRowOff[s] + off;
      f.chain = (p + 1 < np) ? 1 : 0;
      const int id = (int)S.fronts.size();
      for (int j = f.col0; j < f.col0 + f.k; j++) S.frontOfCol[j] = id;
      S.fronts.push_back(f);
    }
    lastFrontOfSn[s] = (int)S.fronts.size() - 1;
  }
  const int nf = (int)S.fronts.size();
  for (int s = 0; s < ns; s++) {
    for (int f = firstFrontOfSn[s]; f < lastFrontOfSn[s]; f++) S.fronts[f].parent = f + 1;
    S.fronts[lastFrontOfSn[s]].parent = (fPar[s] == -1) ? -1 : firstFrontOfSn[fPar[s]];
  }
  // relative indices of the last panel of every supernode into the first panel of the parent supernode
  for (int f = 0; f < nf; f++) {
    Front& F = S.fronts[f];
    if (F.parent == -1 || F.chain) { if (F.parent == -1) GENEO_CHECK(F.m() == 0, "root front with update rows"); continue; }
    const Front& P = S.fronts[F.parent];
    F.relOff = (int64_t)S.rel.size();
    const int* mine = &rowIdx[F.rowOff + F.k];
    const int* par = &rowIdx[P.rowOff];
    int q = 0;
    for (int i = 0; i < F.m(); i++) {
      while (q < P.h && par[q] < mine[i]) q++;
      GENEO_CHECK(q < P.h && par[q] == mine[i], "symbolic: child row missing in parent front");
      S.rel.push_back(q);
    }
  }
  for (int f = 0; f < nf; f++)
    if (S.fronts[f].parent != -1) S.fronts[S.fronts[f].parent].nchild++;

  // ---- 6. top-down levels, arenas, offsets ---------------------------------------------------------------------------
  std::vector<int> depth(nf, 0);
  int maxDepth = 0;
  for (int f = nf - 1; f >= 0; f--) {
    if (S.fronts[f].parent != -1) depth[f] = depth[S.fronts[f].parent] + 1;
    maxDepth = std::max(maxDepth, depth[f]);
  }
  S.nlevels = maxDepth + 1;
  S.levelPtr.assign(S.nlevels + 1, 0);
  for (int f = 0; f < nf; f++) { S.fronts[f].level = maxDepth - depth[f]; S.levelPtr[S.fronts[f].level + 1]++; }
  for (int l = 0; l < S.nlevels; l++) S.levelPtr[l + 1] += S.levelPtr[l];
  S.levelFronts.resize(nf);
  {
    std::vector<int> pos(S.levelPtr.begin(), S.levelPtr.end() - 1);
    for (int f = 0; f < nf; f++) S.levelFronts[pos[S.fronts[f].level]++] = f;
  }
  int64_t lOff = 0;
  for (int f = 0; f < nf; f++) {
    Front& F = S.fronts[f];
    F.lOff = lOff;
    lOff += (int64_t)F.ld * F.k;
    const double k = F.k, m = F.m();
    S.flops += k * k * k / 3. + m * k * k + m * m * k;
    S.maxK = std::max(S.maxK, F.k);
    S.maxH = std::max(S.maxH, F.h);
  }
  S.lSize = lOff;
  // Update matrices.  91 % of the update volume of a 3-D problem sits in supernode CHAINS (panel p+1 of a supernode is the
  // only parent of panel p, identity relative indices): there the parent's update matrix is the trailing block of the
  // child's, so it stays where it is (in the chain arena, for the life of the chain) -- no extend-add, no memset, one
  // read-modify-write per panel instead of four passes.  Everything else ping-pongs between two arenas by level parity.
  struct Live { int64_t off, size; int lEnd; };
  std::vector<Live> live;
  for (int l = 0; l < S.nlevels; l++) {
    int64_t u = 0, w = 0;
    live.erase(std::remove_if(live.begin(), live.end(), [&](const Live& b) { return b.lEnd < l; }), live.end());
    for (int t = S.levelPtr[l]; t < S.levelPtr[l + 1]; t++) {
      const int f = S.levelFronts[t];
      Front& F = S.fronts[f];
      const int64_t m = F.m();
      if (m > 0) {
        F.wOff = w; w += m * F.k;
        w = (w + 15) & ~(int64_t)15;  // 128-byte alignment of every scratch panel / fresh update matrix
        const bool inplace = f > 0 && S.fronts[f - 1].chain && S.fronts[f - 1].parent == f;
        if (inplace) {
          const Front& C = S.fronts[f - 1];
          F.inplace = 1;
          F.uArena = C.uArena;
          F.uLd = C.uLd;
          F.uOff = C.uOff + (int64_t)F.k * ((int64_t)C.uLd + 1);
        } else if (F.chain) {  // first panel of a chain: lives until the tree parent of the last panel
          int last = f;
          while (S.fronts[last].chain) last++;
          const int lEnd = S.fronts[last].level + 1;
          const int64_t size = (m * m + 15) & ~(int64_t)15;
          std::sort(live.begin(), live.end(), [](const Live& a, const Live& b) { return a.off < b.off; });
          int64_t off = 0;
          for (const Live& b : live) {
            if (b.off - off >= size) break;
            off = std::max(off, b.off + b.size);
          }
          live.push_back(Live{off, size, lEnd});
          F.uArena = 2; F.uLd = (int)m; F.uOff = off;
          S.cArena = std::max(S.cArena, off + size);
        } else {
          F.uArena = l & 1; F.uLd = (int)m; F.uOff = u;
          u += m * m;
          u = (u + 15) & ~(int64_t)15;
        }
      }
    }
    S.uArena = std::max(S.uArena, u);
    S.wArena = std::max(S.wArena, w);
  }

  for (int f = 0; f < nf; f++) {  // chains start at a fresh front followed by in-place panels: pair them up two by two
    if (!(S.fronts[f].chain && !S.fronts[f].inplace && S.fronts[f].m() > 0)) continue;
    int last = f;
    while (S.fronts[last].chain) last++;
    for (int i = f; i + 1 <= last; i += 2) {
      if (!S.fronts[i + 1].inplace) break;
      S.fronts[i].pair = 1;
      S.fronts[i + 1].pair = 2;
    }
  }

  lap("fronts+levels");
  // ---- 7. scatter map of the input values (lower triangle of P A P^T) into the panels --------------------------------
  S.perm = perm;
  S.iperm = iperm;
  if (!opt.skipAsm) {
    std::vector<int64_t> tT;
    const bool haveT = transpose_positions(n, ptr, idx, tT, nullptr);
    symbolic_asm_map(n, ptr, idx, haveT ? &tT : nullptr, S);
  }
  lap("asm map");
}

bool transpose_positions(int n, const int64_t* ptr, const int* idx, std::vector<int64_t>& tT, int64_t* ndiag) {
  tT.resize((size_t)ptr[n]);
  std::vector<int64_t> next(ptr, ptr + n);
  int64_t nd = 0;
  for (int r = 0; r < n; r++)
    for (int64_t t = ptr[r]; t < ptr[r + 1]; t++) {
      const int c = idx[t];
      if (c < 0 || c >= n) return false;
      const int64_t q = next[c];  // rows run in ascending order: the next unused entry of row c must be the column r
      if (q >= ptr[c + 1] || idx[q] != r) return false;
      tT[t] = q;
      next[c] = q + 1;
      nd += (c == r);
    }
  if (ndiag) *ndiag = nd;
  return true;
}

void symbolic_asm_map(int n, const int64_t* ptr, const int* idx, const std::vector<int64_t>* tTp, Symbolic& S) {
  const std::vector<int>& perm = S.perm;
  const std::vector<int>& iperm = S.iperm;
  const std::vector<int>& rowIdx = S.rowIdx;
  S.asmSrc.clear();
  S.asmDst.clear();
  if (tTp && (int64_t)tTp->size() == ptr[n]) {
    const std::vector<int64_t>& tT = *tTp;
    S.asmSrc.reserve(ptr[n] / 2 + n);
    S.asmDst.reserve(ptr[n] / 2 + n);
    std::vector<int> where(n, 0);  // position of a row in the current front (checked: stale entries are harmless)
    for (const Front& F : S.fronts) {
      const int* rows = &rowIdx[F.rowOff];
      for (int q = 0; q < F.h; q++) where[rows[q]] = q;
      for (int j = F.col0; j < F.col0 + F.k; j++) {
        const int jo = perm[j];
        const int64_t colBase = F.lOff + (int64_t)(j - F.col0) * F.ld;
        for (int64_t t = ptr[jo]; t < ptr[jo + 1]; t++) {  // row perm[j]: the transposed entries of column j
          const int i = iperm[idx[t]];
          if (i < j) continue;
          const int pos = where[i];
          GENEO_CHECK(pos < F.h && rows[pos] == i, "symbolic: matrix entry outside the predicted structure");
          S.asmSrc.push_back(tT[t]);
          S.asmDst.push_back(colBase + pos);
        }
      }
    }
    return;
  }
  S.asmSrc.reserve(ptr[n] / 2 + n);
  S.asmDst.reserve(ptr[n] / 2 + n);
  for (int ro = 0; ro < n; ro++) {
    const int i = iperm[ro];
    for (int64_t t = ptr[ro]; t < ptr[ro + 1]; t++) {
      const int j = iperm[idx[t]];
      if (i < j) continue;  // entry (i,j) with i >= j goes to column j
      const Front& F = S.fronts[S.frontOfCol[j]];
      int pos;
      if (i < F.col0 + F.k) pos = i - F.col0;
      else {
        const int* b = &rowIdx[F.rowOff + F.k];
        const int* e = &rowIdx[F.rowOff + F.h];
        const int* it = std::lower_bound(b, e, i);
        GENEO_CHECK(it != e && *it == i, "symbolic: matrix entry outside the predicted structure");
        pos = F.k + (int)(it - b);
      }
      S.asmSrc.push_back(t);
      S.asmDst.push_back(F.lOff + pos + (int64_t)(j - F.col0) * F.ld);
    }
  }
}

}  // namespace geneo
