// abi.cpp -- the C ABI of include/geneo_b200.h (thin: argument checking, host<->device staging, error capture).
#include "geneo_b200.h"

#include <algorithm>
#include <cstring>
#include <memory>
#include <string>

#include "dense_host.hpp"
#include "geneo.hpp"

namespace geneo { int profile_dump(const char* path); }
using namespace geneo;

struct geneo_problem_s {
  Mesh mesh;
  Decomposition dec;
  std::vector<int> elemPart, nodePart;
  bool decomposed = false, dual = true;
  int overlap = 0;
};
struct geneo_pc_s {
  GeneoPC pc;
  bool ready = false;
  bool dist = false;  // set up by geneo_pc_setup_dist
  const geneo_problem_s* prob = nullptr;  // borrowed (like pcA / pcMap in the reference, src/geneo.cpp:2221-2230)
};
struct geneo_symbolic_s { Symbolic s; };
struct geneo_layout_s { RankLayout L; };

static thread_local std::string g_err;
#define ABI_TRY try {
#define ABI_CATCH                                                 \
  } catch (std::exception & e) { g_err = e.what(); return 1; }    \
  catch (...) { g_err = "geneo_b200: unknown error"; return 1; }  \
  return 0;
#define ABI_REQ(c, m) do { if (!(c)) { g_err = std::string("geneo_b200: ") + (m); return 1; } } while (0)

extern "C" {

const char* geneo_last_error(void) { return g_err.c_str(); }
int geneo_version(void) { return 100; }
int geneo_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// ---- problem ---------------------------------------------------------------------------------------------------------
int geneo_problem_create(geneo_problem_t* out) { ABI_TRY ABI_REQ(out, "null output"); *out = new geneo_problem_s(); ABI_CATCH }
int geneo_problem_destroy(geneo_problem_t p) { ABI_TRY delete p; ABI_CATCH }

int geneo_problem_set_mesh(geneo_problem_t p, uint32_t nbNode, uint32_t nbElem, const uint32_t* elemPtr,
                           const uint32_t* elemIdx, const double* elemMat) {
  ABI_TRY
  ABI_REQ(p && elemPtr && elemIdx && elemMat, "null argument");
  ABI_REQ(nbNode > 0 && nbElem > 0, "empty input");  // src/geneo4PETSc.cpp:593
  Mesh& m = p->mesh;
  m = Mesh();
  m.nbNode = (int)nbNode;
  m.elemPtr.assign(elemPtr, elemPtr + nbElem + 1);
  m.elemIdx.assign(elemIdx, elemIdx + elemPtr[nbElem]);
  for (int v : m.elemIdx) ABI_REQ(v >= 0 && v < (int)nbNode, "bad element node index");
  m.finalize();
  m.matVal.assign(elemMat, elemMat + m.matPtr.back());
  p->decomposed = false;
  ABI_CATCH
}
int geneo_problem_generate(geneo_problem_t p, const char* kind, const char* args) {
  ABI_TRY
  ABI_REQ(p && kind && args, "null argument");
  const std::string k(kind);
  ABI_REQ(k == "laplacian" || k == "heat" || k == "graph", "unknown generator (laplacian | heat | graph)");
  if (k == "graph") {
    GraphGenOptions go;
    ABI_REQ(parse_graph_args(args, go) == 0, "invalid generator command line");
    generate_graph(go, p->mesh);
  } else {
    GridGenOptions o;
    o.heat = (k == "heat");
    ABI_REQ(parse_gen_args(args, o) == 0, "invalid generator command line");
    generate_grid(o, p->mesh);
  }
  p->decomposed = false;
  ABI_CATCH
}
int geneo_problem_generate_boxed(geneo_problem_t p, const char* kind, const char* args, const int32_t boxK[3],
                                 const int32_t keepLo[3], const int32_t keepHi[3], int32_t* edge) {
  ABI_TRY
  ABI_REQ(p && kind && args && boxK, "null argument");
  GridGenOptions o;
  const std::string k(kind);
  ABI_REQ(k == "laplacian" || k == "heat", "unknown generator (laplacian | heat)");
  o.heat = (k == "heat");
  ABI_REQ(parse_gen_args(args, o) == 0, "invalid generator command line");
  for (int a = 0; a < 3; a++) {
    o.boxK[a] = boxK[a];
    if (keepLo && keepHi) { o.keepLo[a] = keepLo[a]; o.keepHi[a] = keepHi[a]; }
  }
  generate_grid(o, p->mesh, &p->elemPart);  // the box partition of the generated (sub-)mesh is kept for decompose_owned
  p->nodePart.clear();
  p->decomposed = false;
  if (edge) *edge = grid_edge(o);
  ABI_CATCH
}
int geneo_problem_read_file(geneo_problem_t p, const char* path, double inpEps) {
  ABI_TRY
  ABI_REQ(p && path, "null argument");
  ABI_REQ(read_input_file(path, inpEps, p->mesh) == 0, "read input file KO");
  p->decomposed = false;
  ABI_CATCH
}
int geneo_problem_decompose(geneo_problem_t p, int nbPart, int metisDual, int overlap, const int32_t* elemPart,
                            const int32_t* nodePart) {
  ABI_TRY
  ABI_REQ(p && p->mesh.nbNode > 0, "no mesh");
  ABI_REQ(nbPart >= 1 && overlap >= 0, "bad partition count / overlap");
  const int ne = p->mesh.nbElem(), nn = p->mesh.nbNode;
  p->dual = metisDual != 0;
  p->overlap = overlap;
  if ((p->dual && elemPart) || (!p->dual && nodePart)) {
    p->elemPart.assign(ne, 0); p->nodePart.assign(nn, 0);
    if (elemPart) p->elemPart.assign(elemPart, elemPart + ne);
    if (nodePart) p->nodePart.assign(nodePart, nodePart + nn);
  } else {
    ABI_REQ(metis_partition(p->mesh, nbPart, p->dual, p->elemPart, p->nodePart) == 0, "partition KO");
  }
  decompose(p->mesh, nbPart, p->elemPart, p->nodePart, p->dual, overlap, std::vector<char>(), p->dec);
  p->decomposed = true;
  ABI_CATCH
}
int geneo_problem_partition(geneo_problem_t p, int nbPart, int metisDual, int32_t* elemPart, int32_t* nodePart) {
  ABI_TRY
  ABI_REQ(p && p->mesh.nbNode > 0 && nbPart >= 1, "no mesh");
  std::vector<int> ep, np_;
  ABI_REQ(metis_partition(p->mesh, nbPart, metisDual != 0, ep, np_) == 0, "partition KO");
  if (elemPart) std::copy(ep.begin(), ep.end(), elemPart);
  if (nodePart) std::copy(np_.begin(), np_.end(), nodePart);
  ABI_CATCH
}
// ---- pre-decomposed input (the PETSc plug-in's view: initGenEOPC / PCGenEOSetup) -----------------------------------------
static void csr_from_c(int n, const int64_t* ptr, const int32_t* idx, const double* val, CsrHost& a) {
  if (ptr[0] != 0) throw Error("geneo_b200: local matrix: row pointer must start at 0");
  for (int r = 0; r < n; r++)
    if (ptr[r + 1] < ptr[r]) throw Error("geneo_b200: local matrix: row pointer is not monotone");
  for (int64_t t = 0; t < ptr[n]; t++)
    if (idx[t] < 0 || idx[t] >= n) throw Error("geneo_b200: local matrix: column index outside [0, n)");
  a.n = a.ncols = n;
  a.ptr.assign(ptr, ptr + n + 1);
  a.idx.assign(idx, idx + ptr[n]);
  a.val.assign(val, val + ptr[n]);
  for (int r = 0; r < n; r++) {  // sorted columns are assumed downstream
    bool sorted = true;
    for (int64_t t = a.ptr[r] + 1; t < a.ptr[r + 1]; t++) sorted = sorted && a.idx[t - 1] < a.idx[t];
    if (sorted) continue;
    std::vector<std::pair<int, double>> row;
    for (int64_t t = a.ptr[r]; t < a.ptr[r + 1]; t++) row.emplace_back(a.idx[t], a.val[t]);
    std::sort(row.begin(), row.end());
    for (size_t k = 1; k < row.size(); k++)
      if (row[k].first == row[k - 1].first) throw Error("geneo_b200: duplicate column in a local matrix row");
    for (size_t k = 0; k < row.size(); k++) { a.idx[a.ptr[r] + k] = row[k].first; a.val[a.ptr[r] + k] = row[k].second; }
  }
}
int geneo_problem_begin_subdomains(geneo_problem_t p, int64_t nbDof, int nbPart) {
  ABI_TRY
  ABI_REQ(p && nbDof > 0 && nbDof < 2147483647 && nbPart >= 1, "bad sizes");
  p->mesh = Mesh();
  p->dec = Decomposition();
  p->dec.nbNode = (int)nbDof; p->dec.nbPart = nbPart; p->dec.nbElem = 0;
  p->dec.subs.assign(nbPart, Subdomain());
  p->elemPart.clear(); p->nodePart.clear();
  p->decomposed = false;
  ABI_CATCH
}
int geneo_problem_set_subdomain(geneo_problem_t p, int s, int64_t n, const int32_t* globalIds, const int64_t* neuPtr,
                                const int32_t* neuIdx, const double* neuVal, const int64_t* dirPtr, const int32_t* dirIdx,
                                const double* dirVal) {
  ABI_TRY
  ABI_REQ(p && s >= 0 && s < (int)p->dec.subs.size() && n > 0 && globalIds && neuPtr && neuIdx && neuVal, "bad argument");
  Subdomain& S = p->dec.subs[s];
  S = Subdomain();
  S.id = s;
  S.nodes.assign(globalIds, globalIds + n);
  for (int64_t l = 0; l < n; l++) {
    ABI_REQ(globalIds[l] >= 0 && globalIds[l] < p->dec.nbNode, "subdomain: global id out of range");
    ABI_REQ(l == 0 || globalIds[l - 1] < globalIds[l], "subdomain: global ids must be sorted ascending (the reference's local numbering)");
  }
  csr_from_c((int)n, neuPtr, neuIdx, neuVal, S.aNeu);
  if (dirPtr && dirIdx && dirVal) csr_from_c((int)n, dirPtr, dirIdx, dirVal, S.aDir);
  ABI_CATCH
}
int geneo_problem_end_subdomains(geneo_problem_t p) {
  ABI_TRY
  ABI_REQ(p && !p->dec.subs.empty(), "no subdomains");
  finish_predecomposed(p->dec);
  p->decomposed = true;
  ABI_CATCH
}

int geneo_problem_sizes(geneo_problem_t p, int64_t* nbNode, int64_t* nbElem, int64_t* nbPart, int64_t* nnz) {
  ABI_TRY
  ABI_REQ(p, "null argument");
  if (nbNode) *nbNode = p->mesh.nbNode;
  if (nbElem) *nbElem = p->mesh.nbElem();
  if (nbPart) *nbPart = p->decomposed ? p->dec.nbPart : 0;
  if (nnz) *nnz = p->decomposed ? p->dec.nnzNeuTotal : 0;
  ABI_CATCH
}
int geneo_problem_mesh_sizes(geneo_problem_t p, int64_t* nIdx, int64_t* nMat) {
  ABI_TRY
  ABI_REQ(p, "null argument");
  if (nIdx) *nIdx = (int64_t)p->mesh.elemIdx.size();
  if (nMat) *nMat = (int64_t)p->mesh.matVal.size();
  ABI_CATCH
}
int geneo_problem_get_mesh(geneo_problem_t p, int64_t* elemPtr, int32_t* elemIdx, double* elemMat) {
  ABI_TRY
  ABI_REQ(p, "null argument");
  if (elemPtr) std::copy(p->mesh.elemPtr.begin(), p->mesh.elemPtr.end(), elemPtr);
  if (elemIdx) std::copy(p->mesh.elemIdx.begin(), p->mesh.elemIdx.end(), elemIdx);
  if (elemMat) std::copy(p->mesh.matVal.begin(), p->mesh.matVal.end(), elemMat);
  ABI_CATCH
}
int geneo_problem_get_partition(geneo_problem_t p, int32_t* elemPart, int32_t* nodePart) {
  ABI_TRY
  ABI_REQ(p && p->decomposed, "not decomposed");
  if (elemPart) std::copy(p->elemPart.begin(), p->elemPart.end(), elemPart);
  if (nodePart) std::copy(p->nodePart.begin(), p->nodePart.end(), nodePart);
  ABI_CATCH
}
int geneo_problem_sub_sizes(geneo_problem_t p, int s, int64_t sizes[4]) {
  ABI_TRY
  ABI_REQ(p && p->decomposed && s >= 0 && s < p->dec.nbPart, "bad subdomain");
  const Subdomain& S = p->dec.subs[s];
  sizes[0] = (int64_t)S.nodes.size(); sizes[1] = (int64_t)S.elems.size(); sizes[2] = S.aNeu.nnz(); sizes[3] = S.aDir.nnz();
  ABI_CATCH
}
int geneo_problem_sub_nodes(geneo_problem_t p, int s, int32_t* nodes, int32_t* mult) {
  ABI_TRY
  ABI_REQ(p && p->decomposed && s >= 0 && s < p->dec.nbPart, "bad subdomain");
  const Subdomain& S = p->dec.subs[s];
  if (nodes) std::copy(S.nodes.begin(), S.nodes.end(), nodes);
  if (mult) std::copy(S.mult.begin(), S.mult.end(), mult);
  ABI_CATCH
}
int geneo_problem_sub_intersect(geneo_problem_t p, int s, int q, int32_t* idx, int64_t cap, int64_t* count) {
  ABI_TRY
  ABI_REQ(p && p->decomposed && s >= 0 && s < p->dec.nbPart && q >= 0 && q < p->dec.nbPart, "bad subdomain");
  const std::vector<int>& v = p->dec.subs[s].intersect[q];
  if (count) *count = (int64_t)v.size();
  if (idx) std::copy(v.begin(), v.begin() + std::min<int64_t>(cap, (int64_t)v.size()), idx);
  ABI_CATCH
}
int geneo_problem_sub_matrix(geneo_problem_t p, int s, int which, int64_t* ptr, int32_t* idx, double* val) {
  ABI_TRY
  ABI_REQ(p && p->decomposed && s >= 0 && s < p->dec.nbPart, "bad subdomain");
  const CsrHost& a = which == 0 ? p->dec.subs[s].aNeu : p->dec.subs[s].aDir;
  if (ptr) std::copy(a.ptr.begin(), a.ptr.end(), ptr);
  if (idx) std::copy(a.idx.begin(), a.idx.end(), idx);
  if (val) std::copy(a.val.begin(), a.val.end(), val);
  ABI_CATCH
}

// ---- preconditioner ---------------------------------------------------------------------------------------------------
int geneo_pc_create(geneo_pc_t* out) { ABI_TRY ABI_REQ(out, "null output"); *out = new geneo_pc_s(); ABI_CATCH }
int geneo_pc_destroy(geneo_pc_t pc) { ABI_TRY delete pc; dev_cache_flush(); /* parked device blocks go back to the driver */ ABI_CATCH }
int geneo_pc_set_from_options(geneo_pc_t pc, int argc, const char* const* argv) {
  ABI_TRY
  ABI_REQ(pc, "GenEO preconditioner is invalid");
  std::string err;
  if (pc->pc.opt.parse(argc, argv, err) != 0) { g_err = "geneo_b200: " + err; return 1; }
  ABI_CATCH
}
int geneo_pc_setup(geneo_pc_t pc, geneo_problem_t p) {
  ABI_TRY
  ABI_REQ(pc, "GenEO preconditioner is invalid");
  ABI_REQ(p && p->decomposed, "GenEO preconditioner without a decomposed problem");
  require_device();
  pc->prob = p;
  pc->dist = false;
  pc->pc.setup(p->dec);
  pc->ready = true;
  ABI_CATCH
}
// ---- multi-GPU ---------------------------------------------------------------------------------------------------------
int geneo_problem_decompose_owned(geneo_problem_t p, int nbPart, int metisDual, int overlap, const int32_t* elemPart,
                                  const int32_t* nodePart, const int32_t* subRank, int rank) {
  ABI_TRY
  ABI_REQ(p && p->mesh.nbNode > 0 && subRank, "null argument");
  ABI_REQ(nbPart >= 1, "bad number of partitions");
  const bool stored = metisDual && !elemPart && (int)p->elemPart.size() == p->mesh.nbElem();  // from generate_boxed
  ABI_REQ(stored || (metisDual && elemPart) || (!metisDual && nodePart), "decompose_owned needs an explicit partition (identical on every rank)");
  p->dual = metisDual != 0;
  p->overlap = overlap;
  if (!stored) {
    p->elemPart.clear(); p->nodePart.clear();
    if (elemPart) p->elemPart.assign(elemPart, elemPart + p->mesh.nbElem());
    if (nodePart) p->nodePart.assign(nodePart, nodePart + p->mesh.nbNode);
  }
  std::vector<char> owner(nbPart, 0);
  for (int q = 0; q < nbPart; q++) owner[q] = subRank[q] == rank;
  decompose(p->mesh, nbPart, p->elemPart, p->nodePart, p->dual, overlap, owner, p->dec);
  p->decomposed = true;
  ABI_CATCH
}
int geneo_layout_create(geneo_problem_t p, int rank, int world, const int32_t* subRank, geneo_layout_t* out) {
  ABI_TRY
  ABI_REQ(p && p->decomposed && subRank && out, "layout needs a decomposed problem");
  std::unique_ptr<geneo_layout_s> l(new geneo_layout_s());
  std::vector<int> sr(subRank, subRank + p->dec.nbPart);
  build_rank_layout(p->mesh, p->dec, sr, rank, world, l->L);
  *out = l.release();
  ABI_CATCH
}
int geneo_layout_destroy(geneo_layout_t l) { ABI_TRY delete l; ABI_CATCH }
int geneo_layout_sizes(geneo_layout_t l, int64_t out[4]) {
  ABI_TRY
  ABI_REQ(l && out, "null argument");
  out[0] = l->L.nOwn(); out[1] = l->L.nGhost(); out[2] = l->L.A.nnz(); out[3] = l->L.world;
  ABI_CATCH
}
int geneo_layout_get(geneo_layout_t l, int32_t* owned, int32_t* ghost, int64_t* ghostPtr) {
  ABI_TRY
  ABI_REQ(l, "null argument");
  if (owned) std::copy(l->L.owned.begin(), l->L.owned.end(), owned);
  if (ghost) std::copy(l->L.ghost.begin(), l->L.ghost.end(), ghost);
  if (ghostPtr) std::copy(l->L.ghostPtr.begin(), l->L.ghostPtr.end(), ghostPtr);
  ABI_CATCH
}
int geneo_layout_matrix(geneo_layout_t l, int64_t* ptr, int32_t* idx, double* val) {
  ABI_TRY
  ABI_REQ(l && ptr && idx && val, "null argument");
  const CsrHost& a = l->L.A;
  std::copy(a.ptr.begin(), a.ptr.end(), ptr);
  std::copy(a.idx.begin(), a.idx.end(), idx);
  std::copy(a.val.begin(), a.val.end(), val);
  ABI_CATCH
}
int geneo_layout_set_send(geneo_layout_t l, int peer, const int32_t* globalIds, int64_t n) {
  ABI_TRY
  ABI_REQ(l && peer >= 0 && peer < l->L.world && (n == 0 || globalIds), "bad argument");
  std::vector<int>& s = l->L.sendIdx[peer];
  s.resize((size_t)n);
  for (int64_t i = 0; i < n; i++) {
    const int g = globalIds[i];
    ABI_REQ(g >= 0 && g < l->L.nbNode, "halo request outside the mesh");
    const int li = l->L.local(g);
    ABI_REQ(li >= 0 && li < l->L.nOwn(), "halo request for a node this rank does not own");
    s[i] = li;
  }
  ABI_CATCH
}
int geneo_nccl_unique_id(void* out128) { ABI_TRY ABI_REQ(out128, "null argument"); require_device(); Comm::unique_id(out128); ABI_CATCH }
int geneo_pc_setup_dist(geneo_pc_t pc, geneo_problem_t p, geneo_layout_t l, const void* ncclUid128) {
  ABI_TRY
  ABI_REQ(pc && p && p->decomposed && l, "GenEO preconditioner without a decomposed problem / layout");
  require_device();
  pc->prob = p;
  pc->dist = true;
  pc->pc.setup(p->dec, &l->L, ncclUid128);
  pc->ready = true;
  ABI_CATCH
}
int geneo_pc_local_sizes(geneo_pc_t pc, int64_t out[2]) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && out, "GenEO preconditioner without context");
  out[0] = pc->pc.nOwn; out[1] = pc->pc.nLoc;
  ABI_CATCH
}
int geneo_allreduce_sum(geneo_pc_t pc, double* h, int n) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && h, "GenEO preconditioner without context");
  pc->pc.comm.allreduce_sum_host(h, n, pc->pc.st);
  ABI_CATCH
}

int geneo_profile_dump(const char* path) { ABI_TRY ABI_REQ(path, "null argument"); ABI_REQ(profile_dump(path) == 0, "cannot write the profile"); ABI_CATCH }

int geneo_pc_refactor(geneo_pc_t pc) {
  ABI_TRY
  ABI_REQ(pc && pc->ready, "GenEO preconditioner without context");
  pc->pc.numeric_setup();
  ABI_CATCH
}
int geneo_pc_update(geneo_pc_t pc, geneo_problem_t p) {
  ABI_TRY
  ABI_REQ(pc && pc->ready, "GenEO preconditioner without context");
  GeneoPC::PendingValues nv;
  if (pc->dist) {  // collective: a problem this rank cannot use is its vote against the update, not an early return
    pc->pc.check_values_dist(p ? &p->mesh : nullptr, p && p->decomposed ? &p->dec : nullptr, nv);
  } else {
    ABI_REQ(p && p->decomposed, "GenEO preconditioner without a decomposed problem");
    require_device();
    pc->pc.check_values(p->dec, nv);  // throws on any mismatch before a resident value changes: the PC stays as it was
  }
  pc->ready = false;                // from here on values and factors disagree until the numeric setup has completed
  pc->prob = p;
  pc->pc.commit_values(nv);
  pc->pc.numeric_setup();
  pc->ready = true;
  ABI_CATCH
}
int geneo_pc_kernel_time(geneo_pc_t pc, double* ms, int64_t* launches) {
  ABI_TRY
  ABI_REQ(pc && pc->ready, "GenEO preconditioner without context");
  pc->pc.kernel_time(ms, launches);
  ABI_CATCH
}
int geneo_pc_level_profile(geneo_pc_t pc, double* us, double* bytes, int64_t* nitems, int cap, int* nphases) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && nphases, "GenEO preconditioner without context");
  std::vector<double> u, b;
  std::vector<int64_t> c;
  pc->pc.level_profile(u, b, c);
  *nphases = (int)u.size();
  for (int i = 0; i < (int)u.size() && i < cap; i++) {
    if (us) us[i] = u[i];
    if (bytes) bytes[i] = b[i];
    if (nitems) nitems[i] = c[i];
  }
  ABI_CATCH
}
int geneo_counters(int64_t c[3]) {
  ABI_TRY
  ABI_REQ(c, "null argument");
  c[0] = (int64_t)g_kernel_launches.load(); c[1] = (int64_t)g_h2d_bytes; c[2] = (int64_t)g_d2h_bytes;
  ABI_CATCH
}
static int stage_apply(geneo_pc_t pc, const double* x, double* y, int what) {
  GeneoPC& g = pc->pc;
  DevBuf<double> dx(g.nLoc), dy(g.nLoc);
  dx.upload(x, g.nLoc, g.st);
  if (what == 0) g.apply(dx.p, dy.p);
  else g.mult(dx.p, dy.p);
  dy.download(y, g.nLoc, g.st);
  return 0;
}
int geneo_pc_apply(geneo_pc_t pc, const double* x, double* y) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && x && y, "GenEO preconditioner without context");
  stage_apply(pc, x, y, 0);
  ABI_CATCH
}
int geneo_pc_apply_device(geneo_pc_t pc, const double* dx, double* dy) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && dx && dy, "GenEO preconditioner without context");
  pc->pc.apply(dx, dy);
  ABI_CATCH
}
int geneo_pc_apply_q_device(geneo_pc_t pc, const double* dx, double* dy) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && dx && dy && pc->pc.opt.lvl2 >= 1, "GenEO preconditioner without coarse space");
  pc->pc.applyQ(dx, dy);
  ABI_CATCH
}
// ---- blocks of right-hand sides ----------------------------------------------------------------------------------------
// k and ksp are checked before the context, ld once the vector length is known
#define BLOCK_REQ(pc, k, a, b, ld1, ld2)                                                                          \
  ABI_REQ((k) >= 1, "block of right-hand sides: k must be at least 1");                                       \
  ABI_REQ(pc && pc->ready && (a) && (b), "GenEO preconditioner without context");                            \
  ABI_REQ((ld1) >= pc->pc.nLoc && (ld2) >= pc->pc.nLoc, "block of right-hand sides: leading dimension below the vector length")
static void block_ksp_check(const char* ksp) {
  const std::string k(ksp ? ksp : "(null)");
  if (k != "cg") throw Error("geneo_b200: block solve: unsupported -ksp_type " + k + " (cg only; no block GMRES)");
}
static void block_report(const std::vector<KspResult>& r, int64_t* out, double* rnorm) {
  for (size_t j = 0; j < r.size(); j++) {
    if (out) { out[2 * j] = r[j].its; out[2 * j + 1] = r[j].reason; }
    if (rnorm) rnorm[j] = r[j].rnorm;
  }
}
// host column-major blocks go through the device 8 columns at a time: what = 0 apply, 1 CG solve
static void stage_block(geneo_pc_t pc, int what, int k, const double* X, int64_t ldx, double* Y, int64_t ldy, double rtol,
                        double atol, double dtol, int maxIt, int64_t* out, double* rnorm) {
  GeneoPC& g = pc->pc;
  const size_t n = (size_t)g.nLoc;
  DevBuf<double> dx(n * 8), dy(n * 8);
  for (int j0 = 0; j0 < k; j0 += 8) {
    const int nc = std::min(8, k - j0);
    for (int c = 0; c < nc; c++) h2d_staged(dx.p + c * n, X + (size_t)(j0 + c) * ldx, n * sizeof(double), g.st);
    g_h2d_bytes += nc * n * sizeof(double);
    if (what == 0) g.apply_block(nc, dx.p, (int64_t)n, dy.p, (int64_t)n);
    else block_report(g.solve_cg_block(nc, dx.p, (int64_t)n, dy.p, (int64_t)n, rtol, atol, dtol, maxIt), out ? out + 2 * j0 : nullptr,
                      rnorm ? rnorm + j0 : nullptr);
    for (int c = 0; c < nc; c++)
      CUDA_CHECK(cudaMemcpyAsync(Y + (size_t)(j0 + c) * ldy, dy.p + c * n, n * sizeof(double), cudaMemcpyDeviceToHost, g.st));
    g_d2h_bytes += nc * n * sizeof(double);
    CUDA_CHECK(::geneo::sync_stream(g.st));
  }
}
int geneo_pc_apply_block(geneo_pc_t pc, int k, const double* X, int64_t ldx, double* Y, int64_t ldy) {
  ABI_TRY
  BLOCK_REQ(pc, k, X, Y, ldx, ldy);
  stage_block(pc, 0, k, X, ldx, Y, ldy, 0., 0., 0., 0, nullptr, nullptr);
  ABI_CATCH
}
int geneo_pc_apply_block_device(geneo_pc_t pc, int k, const double* dX, int64_t ldx, double* dY, int64_t ldy) {
  ABI_TRY
  BLOCK_REQ(pc, k, dX, dY, ldx, ldy);
  pc->pc.apply_block(k, dX, ldx, dY, ldy);
  ABI_CATCH
}

int geneo_pc_name(geneo_pc_t pc, char* buf, int cap) {
  ABI_TRY
  ABI_REQ(pc && buf && cap > 0, "null argument");
  const std::string n = pc->pc.opt.name();
  strncpy(buf, n.c_str(), cap - 1);
  buf[cap - 1] = 0;
  ABI_CATCH
}
int geneo_pc_info(geneo_pc_t pc, int64_t ints[16], double reals[4]) {
  ABI_TRY
  ABI_REQ(pc, "null argument");
  const GeneoPC& g = pc->pc;
  int emin = 0, emax = 0, rmin = 0, rmax = 0;
  if (g.opt.lvl2 >= 1 && !g.nevGlobal.empty()) {  // over ALL subdomains (known on every rank)
    emin = *std::min_element(g.estimGlobal.begin(), g.estimGlobal.end()); emax = *std::max_element(g.estimGlobal.begin(), g.estimGlobal.end());
    rmin = *std::min_element(g.nevGlobal.begin(), g.nevGlobal.end()); rmax = *std::max_element(g.nevGlobal.begin(), g.nevGlobal.end());
  }
  const int64_t v[16] = {g.nbDof, g.nbPart, g.opt.lvl2, g.opt.hybrid, g.opt.effHybrid, g.opt.lvl1ORAS, g.opt.offload,
                         g.opt.noSyl, g.estimDimE, emin, emax, g.realDimE, rmin, rmax, g.nicolaides, g.nE};
  for (int i = 0; i < 16; i++) ints[i] = v[i];
  if (reals) { reals[0] = g.opt.tau; reals[1] = g.opt.gamma; reals[2] = g.opt.optim; reals[3] = 0.; }
  ABI_CATCH
}
int geneo_pc_timers(geneo_pc_t pc, double* t, int cap) {
  ABI_TRY
  ABI_REQ(pc && t, "null argument");
  const GeneoPC& g = pc->pc;
  const double v[] = {g.lvl1SetupMinvTime,                                                          // 0
                      g.lvl2SetupTauLocTime, g.lvl2SetupTauSylTime, g.lvl2SetupTauEigTime,          // 1-3
                      g.lvl2SetupGammaLocTime, g.lvl2SetupGammaSylTime, g.lvl2SetupGammaEigTime,    // 4-6
                      g.lvl2SetupSylTime, g.lvl2SetupEigTime, g.lvl2SetupZTime, g.lvl2SetupETime,   // 7-10
                      g.lvl1ApplyTime, g.lvl1ApplyScatterTime, g.lvl1ApplyMinvTime, g.lvl1ApplyGatherTime,  // 11-14
                      g.lvl1ApplyPrjFSTime, g.lvl2ApplyTime, g.lvl2ApplyZtTime, g.lvl2ApplyEinvTime, g.lvl2ApplyZTime,  // 15-19
                      g.symbolicTime, g.operatorTime, g.setupTime, g.uploadTime, g.numericTime,    // 20-24
                      g.updateLayoutTime};                                                          // 25
  const int n = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < std::min(n, cap); i++) t[i] = v[i];
  ABI_CATCH
}
int geneo_pc_stats(geneo_pc_t pc, double stats[8]) {
  ABI_TRY
  ABI_REQ(pc && pc->ready, "GenEO preconditioner without context");
  const GeneoPC& g = pc->pc;
  double nall = 0.;
  for (auto& s : g.subs) nall += s.n;
  stats[0] = (double)g.factorBytes; stats[1] = (double)g.factorNnz; stats[2] = g.factorFlops;
  stats[3] = g.trisolve_algo_bytes(); stats[4] = g.apply_algo_bytes(); stats[5] = g.A.algo_bytes();
  stats[6] = (double)g.applyCount; stats[7] = nall;
  ABI_CATCH
}
int geneo_pc_factor_stats(geneo_pc_t pc, double out[4]) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && out, "GenEO preconditioner without context");
  out[0] = pc->pc.allFactorSeconds; out[1] = pc->pc.allFactorFlops; out[2] = (double)pc->pc.allFactorCount; out[3] = pc->pc.orderingReuseTime;
  ABI_CATCH
}
int geneo_pc_factor_bench(geneo_pc_t pc, double out[2]) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && out, "GenEO preconditioner without context");
  pc->pc.factor_bench(&out[0], &out[1]);
  ABI_CATCH
}
int geneo_pc_sub_info(geneo_pc_t pc, int s, int64_t ints[8], double reals[2]) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && s >= 0 && s < (int)pc->pc.subs.size(), "bad subdomain");
  const SubdomainState& S = pc->pc.subs[s];
  const int64_t v[8] = {S.n, S.nev, S.estim, S.nicolaides, S.eigSteps, S.eigDim, S.negL1, S.perturbed};
  for (int i = 0; i < 8; i++) ints[i] = v[i];
  if (reals) { reals[0] = S.tauLoc; reals[1] = S.gammaLoc; }
  ABI_CATCH
}
int geneo_pc_sub_eigenvalues(geneo_pc_t pc, int s, double* vals, int cap, int* count) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && s >= 0 && s < (int)pc->pc.subs.size(), "bad subdomain");
  const std::vector<double>& e = pc->pc.subs[s].eigvals;
  if (count) *count = (int)e.size();
  if (vals) std::copy(e.begin(), e.begin() + std::min<size_t>(cap, e.size()), vals);
  ABI_CATCH
}
int geneo_pc_sub_z(geneo_pc_t pc, int s, double* z) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && z && s >= 0 && s < (int)pc->pc.subs.size(), "bad subdomain");
  const SubdomainState& S = pc->pc.subs[s];
  ABI_REQ(S.nev > 0, "no coarse space");
  std::vector<double> zp = S.Z.to_host(pc->pc.st);
  const std::vector<int>& perm = S.plan->sym.perm;  // solver row k = natural row perm[k]
  for (int k = 0; k < S.n; k++)
    for (int c = 0; c < S.nev; c++) z[(size_t)perm[k] * S.nev + c] = zp[(size_t)k * S.nev + c];
  ABI_CATCH
}
int geneo_pc_coarse_matrix(geneo_pc_t pc, double* einv) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && einv && pc->pc.nE > 0, "no coarse space");
  pc->pc.copy_einv(einv);
  ABI_CATCH
}

// ---- operator / Krylov -------------------------------------------------------------------------------------------------
int geneo_mult(geneo_pc_t pc, const double* x, double* y) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && x && y, "GenEO preconditioner without context");
  stage_apply(pc, x, y, 1);
  ABI_CATCH
}
int geneo_mult_device(geneo_pc_t pc, const double* dx, double* dy) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && dx && dy, "GenEO preconditioner without context");
  pc->pc.mult(dx, dy);
  ABI_CATCH
}
int geneo_make_rhs(geneo_pc_t pc, double* b) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && b, "GenEO preconditioner without context");
  GeneoPC& g = pc->pc;
  DevBuf<double> dx(g.nLoc), dy(g.nLoc);
  vec_iota(g.nLoc, 1., dx.p, g.st);
  g.mult(dx.p, dy.p);
  dy.download(b, g.nLoc, g.st);
  ABI_CATCH
}
static int ksp_run(geneo_pc_t pc, const char* ksp, const double* db, double* dx, double rtol, double atol, double dtol,
                   int maxIt, int restart, int64_t out[3], double* rnorm, double* history, int histCap) {
  GeneoPC& g = pc->pc;
  const std::string k(ksp ? ksp : "gmres");
  if (k != "cg" && k != "gmres") throw Error("geneo_b200: unsupported -ksp_type " + k + " (cg | gmres)");
  g.initial_guess(db, dx);
  KspResult r = (k == "cg") ? g.solve_cg(db, dx, rtol, atol, dtol, maxIt) : g.solve_gmres(db, dx, rtol, atol, dtol, maxIt, restart);
  if (out) { out[0] = r.its; out[1] = r.reason; out[2] = (int64_t)r.history.size(); }
  if (rnorm) *rnorm = r.rnorm;
  if (history) for (size_t i = 0; i < r.history.size() && (int)i < histCap; i++) history[i] = r.history[i];
  return 0;
}
int geneo_ksp_solve_device(geneo_pc_t pc, const char* ksp, const double* db, double* dx, double rtol, double atol,
                           double dtol, int maxIt, int restart, int64_t out[3], double* rnorm, double* history, int histCap) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && db && dx, "GenEO preconditioner without context");
  ksp_run(pc, ksp, db, dx, rtol, atol, dtol, maxIt, restart, out, rnorm, history, histCap);
  CUDA_CHECK(::geneo::sync_stream(pc->pc.st));
  ABI_CATCH
}
int geneo_ksp_solve(geneo_pc_t pc, const char* ksp, const double* b, double* x, double rtol, double atol, double dtol,
                    int maxIt, int restart, int64_t out[3], double* rnorm, double* history, int histCap) {
  ABI_TRY
  ABI_REQ(pc && pc->ready && b && x, "GenEO preconditioner without context");
  GeneoPC& g = pc->pc;
  DevBuf<double> db(g.nLoc), dx(g.nLoc);
  db.upload(b, g.nLoc, g.st);
  ksp_run(pc, ksp, db.p, dx.p, rtol, atol, dtol, maxIt, restart, out, rnorm, history, histCap);
  dx.download(x, g.nLoc, g.st);
  ABI_CATCH
}
int geneo_ksp_solve_block(geneo_pc_t pc, const char* ksp, int k, const double* B, int64_t ldb, double* X, int64_t ldx,
                          double rtol, double atol, double dtol, int maxIt, int64_t* out, double* rnorm) {
  ABI_TRY
  block_ksp_check(ksp);
  BLOCK_REQ(pc, k, B, X, ldb, ldx);
  stage_block(pc, 1, k, B, ldb, X, ldx, rtol, atol, dtol, maxIt, out, rnorm);
  ABI_CATCH
}
int geneo_ksp_solve_block_device(geneo_pc_t pc, const char* ksp, int k, const double* dB, int64_t ldb, double* dX, int64_t ldx,
                                 double rtol, double atol, double dtol, int maxIt, int64_t* out, double* rnorm) {
  ABI_TRY
  block_ksp_check(ksp);
  BLOCK_REQ(pc, k, dB, dX, ldb, ldx);
  block_report(pc->pc.solve_cg_block(k, dB, ldb, dX, ldx, rtol, atol, dtol, maxIt), out, rnorm);
  ABI_CATCH
}
const char* geneo_ksp_reason_name(int reason) { return ksp_reason_name(reason); }

// ---- host-only hooks ---------------------------------------------------------------------------------------------------
int geneo_symbolic_create(int n, const int64_t* ptr, const int32_t* idx, int nb, int ordering, int amalgamate,
                          geneo_symbolic_t* out) {
  ABI_TRY
  ABI_REQ(ptr && idx && out && n > 0, "null argument");
  ABI_REQ(ordering == 0 || ordering == 1, "ordering must be 0 (natural) or 1 (METIS)");
  geneo_symbolic_s* s = new geneo_symbolic_s();
  SymbolicOptions o;
  o.nb = nb; o.ordering = ordering; o.amalgamate = amalgamate != 0;
  try { symbolic_analyze(n, ptr, idx, o, s->s); } catch (...) { delete s; throw; }
  *out = s;
  ABI_CATCH
}
int geneo_symbolic_create_perm(int n, const int64_t* ptr, const int32_t* idx, int nb, int amalgamate, const int32_t* perm,
                               geneo_symbolic_t* out) {
  ABI_TRY
  ABI_REQ(ptr && idx && out && perm && n > 0, "null argument");
  geneo_symbolic_s* s = new geneo_symbolic_s();
  SymbolicOptions o;
  o.nb = nb; o.ordering = 3; o.amalgamate = amalgamate != 0; o.userPerm = perm;
  try { symbolic_analyze(n, ptr, idx, o, s->s); } catch (...) { delete s; throw; }
  *out = s;
  ABI_CATCH
}
int geneo_box_ordering(const int32_t dims[3], int nst, const int32_t* stencil, int threads, int32_t* rank) {
  ABI_TRY
  ABI_REQ(dims && rank && (nst == 0 || stencil), "null argument");
  int depth = 0;
  while ((2 << depth) <= threads && depth < 5) depth++;
  std::vector<int> r;
  const int d[3] = {dims[0], dims[1], dims[2]};
  box_reference_ordering(d, nst, stencil, depth, r);
  std::copy(r.begin(), r.end(), rank);
  ABI_CATCH
}
int geneo_symbolic_destroy(geneo_symbolic_t s) { ABI_TRY delete s; ABI_CATCH }
int geneo_symbolic_info(geneo_symbolic_t s, int64_t ints[11], double reals[1]) {
  ABI_TRY
  ABI_REQ(s, "null argument");
  const Symbolic& S = s->s;
  const int64_t v[11] = {S.n, (int64_t)S.fronts.size(), S.nlevels, S.lSize, S.uArena, S.wArena, (int64_t)S.rowIdx.size(),
                         (int64_t)S.rel.size(), (int64_t)S.asmSrc.size(), S.nsuper, S.cArena};
  for (int i = 0; i < 11; i++) ints[i] = v[i];
  if (reals) reals[0] = S.flops;
  ABI_CATCH
}
int geneo_symbolic_get(geneo_symbolic_t s, int32_t* perm, int64_t* fronts, int32_t* rowIdx, int32_t* rel, int64_t* asmSrc,
                       int64_t* asmDst) {
  ABI_TRY
  ABI_REQ(s, "null argument");
  const Symbolic& S = s->s;
  if (perm) std::copy(S.perm.begin(), S.perm.end(), perm);
  if (fronts)
    for (size_t f = 0; f < S.fronts.size(); f++) {
      const Front& F = S.fronts[f];
      const int64_t v[17] = {F.col0, F.k, F.h, F.parent, F.level, F.chain, F.nchild, F.rowOff, F.lOff, F.uOff, F.wOff, F.relOff, F.ld,
                             F.uLd, F.uArena, F.inplace, F.pair};
      std::copy(v, v + 17, fronts + 17 * f);
    }
  if (rowIdx) std::copy(S.rowIdx.begin(), S.rowIdx.end(), rowIdx);
  if (rel) std::copy(S.rel.begin(), S.rel.end(), rel);
  if (asmSrc) std::copy(S.asmSrc.begin(), S.asmSrc.end(), asmSrc);
  if (asmDst) std::copy(S.asmDst.begin(), S.asmDst.end(), asmDst);
  ABI_CATCH
}
int geneo_host_sym_eig_rows(int n, double* a, const int32_t* rows, int nrows, double* w, double* yrows) {
  ABI_TRY
  ABI_REQ(a && w && yrows && rows && n >= 0 && nrows >= 0, "null argument");
  for (int t = 0; t < nrows; t++) ABI_REQ(rows[t] >= 0 && rows[t] < n, "row index out of range");
  sym_eig_rows(n, a, rows, nrows, w, yrows);
  ABI_CATCH
}
int geneo_host_prepare_probe(int n, const int64_t* ptr, const int32_t* idx, const double* val, const int32_t* perm, int nb, int helper,
                             double seconds[4], uint64_t* digest, double* scatterOut, int64_t scatterLen) {
  ABI_TRY
  ABI_REQ(ptr && idx && val && seconds && digest && n > 0, "null argument");
  host_prepare_probe(n, ptr, idx, val, perm, nb, helper, seconds, digest, scatterOut, scatterLen);
  ABI_CATCH
}
int geneo_host_sym_eig(int n, double* a, double* w) { ABI_TRY ABI_REQ(a && w && n >= 0, "null argument"); sym_eig(n, a, w); ABI_CATCH }

int geneo_microbench(int kind, int n, int reps, double result[2]) {
  ABI_TRY
  // checked before anything touches the device: a bad kind allocates no synthetic forest
  ABI_REQ(kind < 100 || kind % 100 == 1 || kind % 100 == 8 || kind % 100 == 16,
          "microbench kind 100*nlev + nr: nr must be 1, 8 or 16");
  require_device();
  ABI_REQ(result && n > 0 && reps > 0, "bad argument");
  cudaEvent_t e0, e1;
  CUDA_CHECK(cudaEventCreate(&e0));
  CUDA_CHECK(cudaEventCreate(&e1));
  float ms = 0.f;
  result[0] = result[1] = 0.;
  if (kind == 2) {  // solve-kernel streaming: n = panel height h; about 2 GB of 128-column panels at one level
    const int k = 128, h = std::max(n, k);
    const int nf = (int)std::max<int64_t>(8, (int64_t)(2.0e9 / ((double)h * k * 8.)));
    double gb = 0.;
    result[1] = solve_stream_bench(nf, h, k, reps, &gb);  // ms per solve (forward + backward)
    result[0] = gb;                                       // algorithmic GB/s
  } else if (kind >= 100) {  // level-latency probe: kind = 100*nlev + nr; nlev levels of `reps` fronts of n x 128 each
    const int nlev = kind / 100, nr = kind % 100;
    double gb = 0.;
    result[1] = solve_stream_bench(reps, std::max(n, 128), 128, 5, &gb, nlev, nr);
    result[0] = gb;
  } else if (kind == 3) {  // the Schur-update shape: C (n x n) -= A (n x 128) B (n x 128)^T, C streamed from HBM
    const int K = 128;
    DevBuf<double> A((size_t)n * K), B((size_t)n * K), C((size_t)n * n);
    A.zero(); B.zero(); C.zero();
    dgemm_nt_device(n, n, K, A.p, n, B.p, n, C.p, n, 1, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaEventRecord(e0));
    for (int r = 0; r < reps; r++) dgemm_nt_device(n, n, K, A.p, n, B.p, n, C.p, n, 1, 0);
    CUDA_CHECK(cudaEventRecord(e1));
    CUDA_CHECK(cudaEventSynchronize(e1));
    CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    result[0] = 2. * (double)n * n * K * reps / (ms * 1e-3) / 1e12;
    result[1] = ms / reps;
  } else if (kind == 0) {
    std::vector<double> hA((size_t)n * n), hB((size_t)n * n);
    for (size_t i = 0; i < hA.size(); i++) { hA[i] = (double)((i * 2654435761u) % 1000) / 1000. - 0.5; hB[i] = (double)((i * 40503u) % 1000) / 1000. - 0.5; }
    DevBuf<double> A, B, C((size_t)n * n);
    A.upload(hA); B.upload(hB);
    dgemm_nt_device(n, n, n, A.p, n, B.p, n, C.p, n, 0, 0);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaEventRecord(e0));
    for (int r = 0; r < reps; r++) dgemm_nt_device(n, n, n, A.p, n, B.p, n, C.p, n, 0, 0);
    CUDA_CHECK(cudaEventRecord(e1));
    CUDA_CHECK(cudaEventSynchronize(e1));
    CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    result[0] = 2. * (double)n * n * n * reps / (ms * 1e-3) / 1e12;
    std::vector<double> hC = C.to_host();
    double err = 0.;
    for (int t = 0; t < 64; t++) {  // spot check 64 entries against a host dot product
      const int i = (t * 7919) % n, j = (t * 104729) % n;
      double s = 0.;
      for (int k = 0; k < n; k++) s += hA[i + (size_t)k * n] * hB[j + (size_t)k * n];
      err = std::max(err, std::fabs(s - hC[i + (size_t)j * n]));
    }
    result[1] = err;
  } else {
    DevBuf<double> A((size_t)n), B((size_t)n);
    A.zero(); B.zero();
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaEventRecord(e0));
    for (int r = 0; r < reps; r++) CUDA_CHECK(cudaMemcpyAsync(B.p, A.p, (size_t)n * 8, cudaMemcpyDeviceToDevice, 0));
    CUDA_CHECK(cudaEventRecord(e1));
    CUDA_CHECK(cudaEventSynchronize(e1));
    CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    result[0] = 2. * (double)n * 8. * reps / (ms * 1e-3) / 1e9;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  ABI_CATCH
}

}  // extern "C"
