// geneo.cu -- see geneo.hpp.
#include "geneo.hpp"

#include <algorithm>
#include <array>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstring>
#include <sstream>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>

#include "dense_host.hpp"

namespace geneo {

std::atomic<unsigned long long> g_kernel_launches{0};
unsigned long long g_h2d_bytes = 0, g_d2h_bytes = 0;

// ---- in-library launch profiler (GENEO_PROFILE=1) -----------------------------------------------------------------------
bool g_profile = getenv("GENEO_PROFILE") != nullptr;
namespace {
struct ProfRec { const char* file; int line; cudaEvent_t ev; double host; };
std::vector<ProfRec> g_prof;
}  // namespace
void profile_tick(const char* file, int line) {
  if (g_prof.size() >= 400000) return;
  ProfRec r{file, line, nullptr, now_s()};
  if (cudaEventCreate(&r.ev) != cudaSuccess) return;
  cudaEventRecord(r.ev, 0);
  g_prof.push_back(r);
}
// ---- stream-ordered device block cache (common.hpp) -------------------------------------------------------------------
namespace {
struct CachedBlock { void* p; size_t cap; };
// (never destroyed: DevBufs with static storage duration may be released after any other static object)
std::vector<CachedBlock>& g_dev_cache = *new std::vector<CachedBlock>();
size_t g_dev_cache_bytes = 0;
std::mutex& g_dev_cache_mtx = *new std::mutex();
constexpr size_t DEV_CACHE_LIMIT = (size_t)16 << 30;  // bytes of freed blocks the cache keeps at most
}  // namespace
void dev_cache_flush() {
  std::lock_guard<std::mutex> lk(g_dev_cache_mtx);
  for (auto& b : g_dev_cache) cudaFree(b.p);
  g_dev_cache.clear();
  g_dev_cache_bytes = 0;
}
void* dev_alloc(size_t bytes, size_t* cap) {
  const size_t want = (bytes + 511) & ~(size_t)511;
  {
    std::lock_guard<std::mutex> lk(g_dev_cache_mtx);
    int best = -1;
    for (int i = 0; i < (int)g_dev_cache.size(); i++) {
      const size_t c = g_dev_cache[i].cap;
      if (c >= want && c <= want + want / 4 + (1u << 20) && (best < 0 || c < g_dev_cache[best].cap)) best = i;
    }
    if (best >= 0) {
      void* p = g_dev_cache[best].p;
      *cap = g_dev_cache[best].cap;
      g_dev_cache_bytes -= *cap;
      g_dev_cache[best] = g_dev_cache.back();
      g_dev_cache.pop_back();
      return p;
    }
  }
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {  // out of memory with blocks parked in the cache: give them back and try again
    cudaGetLastError();
    dev_cache_flush();
    e = cudaMalloc(&p, want);
  }
  if (e != cudaSuccess) throw Error(std::string("geneo_b200: cudaMalloc of ") + std::to_string(want) + " bytes failed: " + cudaGetErrorString(e));
  *cap = want;
  return p;
}
void dev_free(void* p, size_t cap) {
  if (!p) return;
  std::lock_guard<std::mutex> lk(g_dev_cache_mtx);
  if (cap > DEV_CACHE_LIMIT / 2 || g_dev_cache_bytes + cap > DEV_CACHE_LIMIT || g_dev_cache.size() >= 256) {
    cudaFree(p);
    return;
  }
  g_dev_cache.push_back(CachedBlock{p, cap});
  g_dev_cache_bytes += cap;
}

void h2d_staged(void* dst, const void* src, size_t bytes, cudaStream_t st) {
  constexpr size_t CH = (size_t)32 << 20;
  if (bytes < ((size_t)4 << 20)) {
    CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    return;
  }
  static std::mutex mtx;
  static char* pin[2] = {nullptr, nullptr};
  static cudaEvent_t ev[2];
  static bool used[2] = {false, false};
  std::lock_guard<std::mutex> lk(mtx);
  if (!pin[0]) {
    for (int i = 0; i < 2; i++) {
      CUDA_CHECK(cudaHostAlloc((void**)&pin[i], CH, cudaHostAllocDefault));
      CUDA_CHECK(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
    }
  }
  int slot = 0;
  for (size_t off = 0; off < bytes; off += CH, slot ^= 1) {
    const size_t len = std::min(CH, bytes - off);
    if (used[slot]) CUDA_CHECK(cudaEventSynchronize(ev[slot]));  // the DMA that last read this bounce buffer is done
    {  // one core copies ~5 GB/s into the bounce buffer, PCIe 5 moves 25+: split the chunk over a few threads
      const int nt = len >= ((size_t)8 << 20) ? 4 : 1;
      const char* sp = static_cast<const char*>(src) + off;
      char* dp = pin[slot];
      std::thread th[3];
      for (int t = 1; t < nt; t++) th[t - 1] = std::thread([=]() { const size_t a = len * t / nt, b = len * (t + 1) / nt; memcpy(dp + a, sp + a, b - a); });
      memcpy(dp, sp, len / nt);
      for (int t = 1; t < nt; t++) th[t - 1].join();
    }
    CUDA_CHECK(cudaMemcpyAsync(static_cast<char*>(dst) + off, pin[slot], len, cudaMemcpyHostToDevice, st));
    CUDA_CHECK(cudaEventRecord(ev[slot], st));
    used[slot] = true;
  }
}

thread_local double g_sync_wait_s = 0.;
namespace {
const bool g_hostprof = getenv("GENEO_HOSTPROF") != nullptr;
struct HostProfRec { std::string name; double s = 0.; long n = 0; };
std::vector<HostProfRec> g_hostprof_recs;
}  // namespace
void host_prof_add(const char* name, double seconds) {
  if (!g_hostprof) return;
  for (auto& r : g_hostprof_recs) if (r.name == name) { r.s += seconds; r.n++; return; }
  g_hostprof_recs.push_back(HostProfRec{name, seconds, 1});
}
void host_prof_report(const char* title) {
  if (!g_hostprof) return;
  fprintf(stderr, "HOSTPROF %s: sync-wait %.3f s\n", title, g_sync_wait_s);
  for (auto& r : g_hostprof_recs) fprintf(stderr, "HOSTPROF   %-28s %9.3f s  %7ld calls\n", r.name.c_str(), r.s, r.n);
  g_hostprof_recs.clear();
  g_sync_wait_s = 0.;
}
int profile_dump(const char* path) {
  FILE* f = fopen(path, "w");
  if (!f) return 1;
  cudaEvent_t last;
  cudaEventCreate(&last);
  cudaEventRecord(last, 0);
  cudaDeviceSynchronize();
  const double hostEnd = now_s();
  struct Agg { long n = 0; double gpu = 0., host = 0.; };
  std::vector<std::pair<std::string, Agg>> agg;
  auto find = [&](const std::string& k) -> Agg& {
    for (auto& a : agg) if (a.first == k) return a.second;
    agg.emplace_back(k, Agg());
    return agg.back().second;
  };
  for (size_t i = 0; i < g_prof.size(); i++) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, g_prof[i].ev, i + 1 < g_prof.size() ? g_prof[i + 1].ev : last);
    const double h = (i + 1 < g_prof.size() ? g_prof[i + 1].host : hostEnd) - g_prof[i].host;
    const char* b = strrchr(g_prof[i].file, '/');
    Agg& a = find(std::string(b ? b + 1 : g_prof[i].file) + ":" + std::to_string(g_prof[i].line));
    a.n++; a.gpu += ms; a.host += 1e3 * h;
  }
  fprintf(f, "site,launches,gpu_ms_until_next_launch,host_ms_until_next_launch\n");
  for (auto& a : agg) fprintf(f, "%s,%ld,%.3f,%.3f\n", a.first.c_str(), a.second.n, a.second.gpu, a.second.host);
  fclose(f);
  for (auto& r : g_prof) cudaEventDestroy(r.ev);
  cudaEventDestroy(last);
  g_prof.clear();
  return 0;
}

// =====================================================================================================================
// Options
// =====================================================================================================================
int GeneoOptions::parse(int argc, const char* const* argv, std::string& err) {
  auto need = [&](int a, const char* o) -> const char* {
    if (a + 1 >= argc || !argv[a + 1]) { err = std::string("invalid option ") + o; return nullptr; }
    return argv[a + 1];
  };
  auto num = [&](const char* s, double& v, const char* o) -> bool {
    std::stringstream ss(s);
    ss >> v;
    if (!ss) { err = std::string("invalid option ") + o + ", bad " + s; return false; }
    return true;
  };
  for (int a = 0; a < argc; a++) {
    if (!argv[a]) continue;
    const std::string o = argv[a];
    if (o == "-geneo_lvl") {
      const char* v = need(a, "-geneo_lvl"); if (!v) return 1;
      std::string s(v);
      const size_t c = s.find(',');
      if (c == std::string::npos) { err = "invalid option -geneo_lvl"; return 1; }
      const std::string l1 = s.substr(0, c), l2 = s.substr(c + 1);
      if (l1 == "ASM") lvl1ASM = true;
      else if (l1 == "RAS") lvl1RAS = true;
      else if (l1 == "SRAS") lvl1RAS = lvl1SRAS = true;
      else if (l1 == "ORAS") lvl1RAS = lvl1ORAS = true;
      else if (l1 == "SORAS") lvl1RAS = lvl1SRAS = lvl1ORAS = true;
      else { err = "invalid option -geneo_lvl, unknown " + l1; return 1; }
      if (l2 == "0") lvl2 = 0;
      else if (l2 == "1") lvl2 = 1;
      else if (l2 == "H1") { lvl2 = 1; hybrid = true; }
      else if (l2 == "E1") { lvl2 = 1; hybrid = true; effHybrid = true; }
      else if (l2 == "2") lvl2 = 2;
      else if (l2 == "H2") { lvl2 = 2; hybrid = true; }
      else if (l2 == "E2") { lvl2 = 2; hybrid = true; effHybrid = true; }
      else { err = "invalid option -geneo_lvl, unknown " + l2; return 1; }
      a++;
    } else if (o == "-geneo_optim") { const char* v = need(a, "-geneo_optim"); if (!v || !num(v, optim, "-geneo_optim")) return 1; a++; }
    else if (o == "-geneo_tau") { const char* v = need(a, "-geneo_tau"); if (!v || !num(v, tau, "-geneo_tau")) return 1; a++; }
    else if (o == "-geneo_gamma") { const char* v = need(a, "-geneo_gamma"); if (!v || !num(v, gamma, "-geneo_gamma")) return 1; a++; }
    else if (o == "-geneo_cut") { double c; const char* v = need(a, "-geneo_cut"); if (!v || !num(v, c, "-geneo_cut")) return 1; cut = (int)c; a++; }
    else if (o == "-geneo_cst") cst = true;
    else if (o == "-geneo_release_workspace") releaseWorkspace = true;
    else if (o == "-geneo_no_syl") noSyl = true;
    else if (o == "-geneo_offload") offload = true;
    else if (o == "-geneo_dbg") {
      const char* v = need(a, "-geneo_dbg"); if (!v) return 1;
      std::string s(v);
      const size_t c = s.find(',');
      if (c == std::string::npos) { err = "invalid option -geneo_dbg"; return 1; }
      const std::string f = s.substr(0, c);
      if (f != "log" && f != "bin" && f != "mat") { err = "invalid option -geneo_dbg, unknown " + f; return 1; }
      double d; if (!num(s.substr(c + 1).c_str(), d, "-geneo_dbg")) return 1;
      debug = (int)d; debugFmt = f; a++;
    } else if (o == "-geneo_chk") {
      const char* v = need(a, "-geneo_chk"); if (!v) return 1;
      std::string f(v);
      if (f != "log" && f != "bin" && f != "mat") { err = "invalid option -geneo_chk, unknown " + f; return 1; }
      check = true; checkFmt = f; a++;
    } else if (o == "-els2_eps_tol") { const char* v = need(a, "-els2_eps_tol"); if (!v || !num(v, epsTol, "-els2_eps_tol")) return 1; a++; }
    else if (o == "-els2_eps_block") { double c; const char* v = need(a, "-els2_eps_block"); if (!v || !num(v, c, "-els2_eps_block")) return 1; epsBlock = (int)c; a++; }
    else if (o == "-els2_eps_ncv") { double c; const char* v = need(a, "-els2_eps_ncv"); if (!v || !num(v, c, "-els2_eps_ncv")) return 1; epsMaxDim = (int)c; a++; }
    else if (o == "-geneo_nb") { double c; const char* v = need(a, "-geneo_nb"); if (!v || !num(v, c, "-geneo_nb")) return 1; nb = (int)c; a++; }
    else if (o == "-geneo_ordering") { double c; const char* v = need(a, "-geneo_ordering"); if (!v || !num(v, c, "-geneo_ordering")) return 1; ordering = (int)c; a++; }
    else if (o == "-geneo_ordering_reuse") { double c; const char* v = need(a, "-geneo_ordering_reuse"); if (!v || !num(v, c, "-geneo_ordering_reuse")) return 1; orderingReuse = c != 0.; a++; }
    else if (o == "-geneo_timing") timing = true;
    else if (o == "-geneo_kernel_timing") kernelTiming = true;
  }
  // consistency (src/geneo.cpp:2486-2488)
  if (lvl2 >= 1 && tau <= 0.) { err = "GenEO preconditioner: tau must be > 0."; return 1; }
  if (lvl2 >= 1 && tau >= 1.) { err = "GenEO preconditioner: tau must be < 1."; return 1; }
  if (lvl2 >= 2 && gamma <= 1.) { err = "GenEO preconditioner: gamma must be > 1."; return 1; }
  if (nb < 8 || nb > 128) { err = "-geneo_nb must be in [8,128]"; return 1; }
  if (ordering != 0 && ordering != 1) { err = "-geneo_ordering must be 0 (natural) or 1 (METIS)"; return 1; }
  return 0;
}

std::string GeneoOptions::name() const {
  std::string nm = "geneo";
  nm += (lvl2 == 0) ? "0" : (lvl2 == 1 ? "1" : "2");
  if (hybrid) nm += effHybrid ? "E" : "H";
  std::string l1;
  if (lvl1ASM) l1 = "ASM";
  if (lvl1RAS) l1 = "RAS";
  if (lvl1SRAS) l1 = "SRAS";
  if (lvl1ORAS) l1 = "ORAS";
  if (lvl1SRAS && lvl1ORAS) l1 = "SORAS";
  return nm + l1;
}

const char* ksp_reason_name(int r) {
  switch (r) {
    case KSP_CONVERGED_RTOL: return "KSP_CONVERGED_RTOL";
    case KSP_CONVERGED_ATOL: return "KSP_CONVERGED_ATOL";
    case KSP_CONVERGED_HAPPY_BREAKDOWN: return "KSP_CONVERGED_HAPPY_BREAKDOWN";
    case KSP_DIVERGED_ITS: return "KSP_DIVERGED_ITS";
    case KSP_DIVERGED_DTOL: return "KSP_DIVERGED_DTOL";
    case KSP_DIVERGED_BREAKDOWN: return "KSP_DIVERGED_BREAKDOWN";
    case KSP_DIVERGED_INDEFINITE_PC: return "KSP_DIVERGED_INDEFINITE_PC";
    case KSP_DIVERGED_NANORINF: return "KSP_DIVERGED_NANORINF";
    case KSP_DIVERGED_INDEFINITE_MAT: return "KSP_DIVERGED_INDEFINITE_MAT";
    default: return "KSP_CONVERGED_ITERATING";
  }
}

// =====================================================================================================================
// Setup
// =====================================================================================================================
namespace {

struct HostPrep {  // everything the host prepares for one subdomain (worker thread)
  Symbolic sym;
  std::shared_ptr<LdltPlan> plan;  // symbolic + the work lists of every level, not uploaded yet
  CsrHost patP;                 // permuted pattern of A_dir with its values
  std::vector<double> vNeuP, vRobP, dP;
  std::vector<int> gidx;
  std::vector<int> userPerm;    // ordering inherited from the reference box (see plan_ordering_reuse); empty: METIS on this subdomain
  double anorm = 0.;
  int maxMult = 1;
  double stageS[4] = {0., 0., 0., 0.};  // symbolic analysis, permuted values, work lists, (spare)
  std::string err;
};

// Structured problems (Decomposition::grid known): subdomains that fill their common bounding box share ONE nested
// dissection -- the reference ordering of that box, restricted to each subdomain (symbolic.hpp box_reference_ordering).
// Box partitions at 8 subdomains per GPU and 8 ranks per node otherwise spend 20 s of host time in 64 METIS calls.
// Multi-GPU: rank 0 orders the box with every core of the node and the ranks receive it over NCCL.
void plan_ordering_reuse(const Decomposition& dec, const std::vector<const Subdomain*>& mine, const GeneoOptions& opt, Comm& comm,
                         unsigned hwAll, cudaStream_t st, std::vector<HostPrep>& prep) {
  if (opt.ordering != 1 || !opt.orderingReuse || dec.grid[0] <= 0) return;
  const int P = (int)mine.size();
  const int64_t n1 = dec.grid[0], n12 = (int64_t)dec.grid[0] * std::max(1, dec.grid[1]);
  auto coord = [&](int g, int c[3]) { c[0] = (int)(g % n1); c[1] = (int)((g / n1) % std::max(1, dec.grid[1])); c[2] = (int)(g / n12); };
  std::vector<std::array<int, 3>> lo(P), ext(P);
  double ref[4] = {0., 0., 0., 0.};  // max extents, number of candidate subdomains
  for (int p = 0; p < P; p++) {
    int l[3] = {INT32_MAX, INT32_MAX, INT32_MAX}, h[3] = {-1, -1, -1}, c[3];
    for (int g : mine[p]->nodes) { coord(g, c); for (int a = 0; a < 3; a++) { l[a] = std::min(l[a], c[a]); h[a] = std::max(h[a], c[a]); } }
    for (int a = 0; a < 3; a++) { lo[p][a] = l[a]; ext[p][a] = h[a] - l[a] + 1; }
    // a candidate is (nearly) a full box: induced separators of a ragged METIS part cost ~1.5x the flops of its own ordering
    const double box = (double)ext[p][0] * ext[p][1] * ext[p][2];
    if ((double)mine[p]->nodes.size() >= 0.97 * box && mine[p]->nodes.size() >= 20000) {
      for (int a = 0; a < 3; a++) ref[a] = std::max(ref[a], (double)ext[p][a]);
      ref[3] += 1.;
    }
  }
  if (comm.active()) {  // global maximum of the extents through a one-hot sum
    std::vector<double> all(4 * (size_t)comm.world, 0.);
    for (int a = 0; a < 4; a++) all[4 * (size_t)comm.rank + a] = ref[a];
    comm.allreduce_sum_host(all.data(), (int)all.size(), st);
    for (int a = 0; a < 4; a++) ref[a] = 0.;
    for (int r = 0; r < comm.world; r++) {
      for (int a = 0; a < 3; a++) ref[a] = std::max(ref[a], all[4 * (size_t)r + a]);
      ref[3] += all[4 * (size_t)r + 3];
    }
  }
  if (ref[3] < 2.) return;  // nothing to share
  const int dims[3] = {(int)ref[0], (int)ref[1], (int)ref[2]};
  const int64_t nref = (int64_t)dims[0] * dims[1] * dims[2];
  std::vector<int> rank;
  if (comm.rank == 0) {
    // stencil of the operator: coordinate offsets met in the rows of the first local subdomain (capped: a wide stencil
    // means this is not a nearest-neighbour grid problem and the reference box would not be representative)
    std::vector<int> sten;
    const Subdomain& S = *mine[0];
    bool ok = true;
    for (int r = 0; r < S.aDir.n && ok; r++) {
      int cr[3], cc[3];
      coord(S.nodes[r], cr);
      for (int64_t t = S.aDir.ptr[r]; t < S.aDir.ptr[r + 1]; t++) {
        coord(S.nodes[S.aDir.idx[t]], cc);
        const int d[3] = {cc[0] - cr[0], cc[1] - cr[1], cc[2] - cr[2]};
        if ((d[0] | d[1] | d[2]) == 0) continue;
        bool have = false;
        for (size_t q = 0; q < sten.size() && !have; q += 3) have = sten[q] == d[0] && sten[q + 1] == d[1] && sten[q + 2] == d[2];
        if (!have) { sten.push_back(d[0]); sten.push_back(d[1]); sten.push_back(d[2]); }
        if (sten.size() > 3 * 64) { ok = false; break; }
      }
    }
    if (ok && !sten.empty()) {
      int depth = 0;
      while ((2u << depth) <= hwAll && depth < 4) depth++;
      box_reference_ordering(dims, (int)(sten.size() / 3), sten.data(), depth, rank);
    }
  }
  if (comm.active()) {  // broadcast from rank 0 (a sum with zeros elsewhere; ranks < 2^31 are exact in FP64); [0] = valid flag
    DevBuf<double> d((size_t)nref + 1);
    std::vector<double> h((size_t)nref + 1, 0.);
    if (comm.rank == 0 && !rank.empty()) { h[0] = 1.; for (int64_t i = 0; i < nref; i++) h[(size_t)i + 1] = rank[(size_t)i]; }
    d.upload(h, st);
    comm.allreduce_sum(d.p, (int)(nref + 1), st);
    d.download(h.data(), (size_t)nref + 1, st);
    if (h[0] < 0.5) return;
    if (comm.rank != 0) { rank.resize((size_t)nref); for (int64_t i = 0; i < nref; i++) rank[(size_t)i] = (int)h[(size_t)i + 1]; }
  }
  if (rank.empty()) return;
  std::vector<int> slot((size_t)nref);
  for (int p = 0; p < P; p++) {
    const Subdomain& S = *mine[p];
    const double box = (double)ext[p][0] * ext[p][1] * ext[p][2];
    if (!((double)S.nodes.size() >= 0.97 * box && S.nodes.size() >= 20000)) continue;
    std::fill(slot.begin(), slot.end(), -1);
    for (int l = 0; l < (int)S.nodes.size(); l++) {
      int c[3];
      coord(S.nodes[l], c);
      slot[(size_t)rank[(size_t)(c[0] - lo[p][0]) + (size_t)dims[0] * ((size_t)(c[1] - lo[p][1]) + (size_t)dims[1] * (size_t)(c[2] - lo[p][2]))]] = l;
    }
    prep[p].userPerm.reserve(S.nodes.size());
    for (int64_t i = 0; i < nref; i++) if (slot[(size_t)i] >= 0) prep[p].userPerm.push_back(slot[(size_t)i]);
  }
}

void prepare_subdomain(const Subdomain& S, const GeneoOptions& opt, int ndDepth, HostPrep& H, bool helper, bool forceGeneral = false) {
  const int n = (int)S.nodes.size();
  SymbolicOptions so;
  so.nb = opt.nb;
  so.ordering = opt.ordering;
  so.ndDepth = ndDepth;
  so.skipAsm = true;
  if (!H.userPerm.empty()) { so.ordering = 3; so.userPerm = H.userPerm.data(); }
  const bool ptm = getenv("GENEO_PREP_TIMING") != nullptr;
  double tq = now_s(), tl = tq;
  auto lap = [&](const char* what) { if (ptm) { const double t = now_s(); fprintf(stderr, "prepare n=%d %s %.3fs\n", n, what, t - tl); tl = t; } };
  const int64_t nnz = S.aDir.nnz();
  // ---- everything that does not depend on the ordering (a second thread when the cores allow it): positions of the
  //      transposed entries, A_neu expanded to the A_dir pattern, and the first touch of the large output arrays (fresh
  //      pages cost about as much as the passes that fill them)
  std::vector<int64_t> tT, asmSrc, asmDst;
  std::vector<double> neuExp;
  bool haveT = false;
  std::string sideErr;
  auto side = [&]() {
    try {
      int64_t ndiag = 0;
      haveT = nnz > 0 && !forceGeneral && transpose_positions(n, S.aDir.ptr.data(), S.aDir.idx.data(), tT, &ndiag);
      if (!haveT) std::vector<int64_t>().swap(tT);
      neuExp.assign((size_t)nnz, 0.);
      for (int r = 0; r < n; r++) {
        int64_t q = S.aDir.ptr[r];
        for (int64_t t = S.aNeu.ptr[r]; t < S.aNeu.ptr[r + 1]; t++) {
          while (q < S.aDir.ptr[r + 1] && S.aDir.idx[q] < S.aNeu.idx[t]) q++;
          GENEO_CHECK(q < S.aDir.ptr[r + 1] && S.aDir.idx[q] == S.aNeu.idx[t], "A_neu entry outside the A_dir pattern");
          neuExp[q] = S.aNeu.val[t];
        }
      }
      H.patP.n = H.patP.ncols = n;
      H.patP.ptr.assign(n + 1, 0);
      H.patP.idx.resize((size_t)nnz);
      H.patP.val.resize((size_t)nnz);
      H.vNeuP.resize((size_t)nnz);
      if (haveT) {  // symmetric pattern: as many entries below the diagonal as above
        asmSrc.resize((size_t)(ndiag + (nnz - ndiag) / 2));
        asmDst.resize(asmSrc.size());
      }
    } catch (std::exception& e) { sideErr = e.what(); }
  };
  std::thread sideThread;
  if (helper) sideThread = std::thread(side);
  try {
    symbolic_analyze(n, S.aDir.ptr.data(), S.aDir.idx.data(), so, H.sym);
  } catch (...) {
    if (sideThread.joinable()) sideThread.join();
    throw;
  }
  H.stageS[0] = now_s() - tq; tq = now_s();
  lap("analysis");
  if (sideThread.joinable()) sideThread.join();
  else side();
  if (!sideErr.empty()) throw Error(sideErr);
  lap(helper ? "wait for the side thread" : "transposed positions, A_neu, first touch");
  const std::vector<int>& perm = H.sym.perm;
  const std::vector<int>& iperm = H.sym.iperm;
  if (haveT) {
    // Sorted rows, symmetric pattern: ONE pass over the matrix in the new row order fills P A P^T through the transposed
    // entries -- every row comes out sorted by new column without a sort -- and, the rows running front by front, the
    // scatter map of the lower triangle with it (position of a row in the front of column k: one table lookup).
    Symbolic& Y = H.sym;
    std::vector<int64_t> fill(n);
    for (int k = 0; k < n; k++) H.patP.ptr[k + 1] = H.patP.ptr[k] + (S.aDir.ptr[perm[k] + 1] - S.aDir.ptr[perm[k]]);
    for (int k = 0; k < n; k++) fill[k] = H.patP.ptr[k];
    // with a second thread: the A_neu values take the same walk on their own (the random writes are the cost)
    std::thread neuThread;
    auto neuWalk = [&]() {
      std::vector<int64_t> fill2(H.patP.ptr.begin(), H.patP.ptr.end() - 1);
      for (int k = 0; k < n; k++) {
        const int ro = perm[k];
        for (int64_t t = S.aDir.ptr[ro]; t < S.aDir.ptr[ro + 1]; t++) H.vNeuP[(size_t)fill2[iperm[S.aDir.idx[t]]]++] = neuExp[(size_t)tT[t]];
      }
    };
    if (helper) neuThread = std::thread(neuWalk);
    struct Join { std::thread& t; ~Join() { if (t.joinable()) t.join(); } } joinNeu{neuThread};
    const bool neuHere = !helper;
    std::vector<int> where(n, 0);
    double amax = 0.;
    int64_t w = 0;
    int kNext = 0;
    const int64_t wMax = (int64_t)asmSrc.size();
    for (const Front& F : Y.fronts) {
      GENEO_CHECK(F.col0 == kNext, "host preparation: fronts do not cover the columns in order");
      kNext = F.col0 + F.k;
      const int* rows = &Y.rowIdx[F.rowOff];
      for (int q = 0; q < F.h; q++) where[rows[q]] = q;
      for (int k = F.col0; k < F.col0 + F.k; k++) {
        const int ro = perm[k];
        const int64_t colBase = F.lOff + (int64_t)(k - F.col0) * F.ld;
        for (int64_t t = S.aDir.ptr[ro]; t < S.aDir.ptr[ro + 1]; t++) {
          const int i = iperm[S.aDir.idx[t]];
          const int64_t q = fill[i]++;
          const int64_t src = tT[t];  // the entry (idx[t], ro) of the input = entry (i, k) of the permuted matrix
          const double v = S.aDir.val[src];
          H.patP.idx[q] = k;
          H.patP.val[q] = v;
          if (neuHere) H.vNeuP[q] = neuExp[src];
          amax = std::max(amax, std::fabs(v));
          if (i >= k) {
            const int pos = where[i];
            GENEO_CHECK(pos < F.h && rows[pos] == i && w < wMax, "symbolic: matrix entry outside the predicted structure");
            asmSrc[(size_t)w] = q;
            asmDst[(size_t)w] = colBase + pos;
            w++;
          }
        }
      }
    }
    if (neuThread.joinable()) neuThread.join();
    GENEO_CHECK(kNext == n && w == wMax, "host preparation: scatter map lost entries");
    H.anorm = std::max(H.anorm, amax);
    Y.asmSrc.swap(asmSrc);
    Y.asmDst.swap(asmDst);
    lap("permuted values + scatter map");
  } else {
    // general input (unsorted rows or an unsymmetric pattern): sort every permuted row, binary searches for the scatter map
    symbolic_asm_map(n, S.aDir.ptr.data(), S.aDir.idx.data(), nullptr, H.sym);
    std::vector<int64_t> origToPerm((size_t)nnz);
    std::vector<std::pair<int, int64_t>> row;
    for (int k = 0; k < n; k++) {
      const int ro = perm[k];
      row.clear();
      for (int64_t t = S.aDir.ptr[ro]; t < S.aDir.ptr[ro + 1]; t++) row.emplace_back(iperm[S.aDir.idx[t]], t);
      std::sort(row.begin(), row.end());
      int64_t q = H.patP.ptr[k];
      for (auto& e : row) {
        H.patP.idx[q] = e.first;
        H.patP.val[q] = S.aDir.val[e.second];
        H.vNeuP[q] = neuExp[e.second];
        origToPerm[e.second] = q;
        H.anorm = std::max(H.anorm, std::fabs(S.aDir.val[e.second]));
        q++;
      }
      H.patP.ptr[k + 1] = q;
    }
    for (auto& s : H.sym.asmSrc) s = origToPerm[s];
    lap("permuted values + scatter map (general input)");
  }
  std::vector<double>().swap(neuExp);
  std::vector<int64_t>().swap(tT);
  H.dP.resize(n);
  H.gidx.resize(n);
  for (int k = 0; k < n; k++) {
    H.dP[k] = 1.0 / ((double)S.mult[perm[k]]);  // createPartitionOfUnity, src/geneo.cpp:977-980
    H.gidx[k] = S.nodes[perm[k]];
    H.maxMult = std::max(H.maxMult, S.mult[perm[k]]);
  }
  if (opt.lvl1ORAS) {  // createRobinMatrix, src/geneo.cpp:1613-1670 (done sparsely: no dense border x border buffer)
    H.vRobP = H.patP.val;
    if (std::fabs(opt.optim) > DBL_EPSILON)
      for (int k = 0; k < n; k++) {
        if (S.mult[perm[k]] <= 1) continue;
        for (int64_t q = H.patP.ptr[k]; q < H.patP.ptr[k + 1]; q++)
          if (S.mult[perm[H.patP.idx[q]]] > 1) H.vRobP[q] += opt.optim * H.vNeuP[q];
      }
  }
  lap("partition of unity, Robin");
  H.stageS[1] = now_s() - tq; tq = now_s();
  // the work lists of every factorization level are host work too: built here, uploaded by the thread that owns the device
  H.plan = std::make_shared<LdltPlan>(std::move(H.sym), LdltPlan::HostOnly{});
  H.stageS[2] = now_s() - tq;
}

}  // namespace

// Host-only test hook: the per-subdomain host preparation (analysis, permuted values, scatter map, work lists) of a plain
// symmetric CSR matrix taken as A_dir = A_neu, with its stage stopwatches and a digest of everything it produced.
void host_prepare_probe(int n, const int64_t* ptr, const int* idx, const double* val, const int* userPerm, int nb, int helper,
                        double seconds[4], uint64_t* digest, double* scatterOut, int64_t scatterLen) {
  Subdomain S;
  S.nodes.resize(n); for (int i = 0; i < n; i++) S.nodes[i] = i;
  S.mult.assign(n, 1);
  S.aDir.n = S.aDir.ncols = n;
  S.aDir.ptr.assign(ptr, ptr + n + 1);
  S.aDir.idx.assign(idx, idx + ptr[n]);
  S.aDir.val.assign(val, val + ptr[n]);
  S.aNeu = S.aDir;
  GeneoOptions opt;
  opt.nb = nb;
  opt.lvl1ORAS = true;
  opt.optim = 0.5;
  HostPrep H;
  if (userPerm) H.userPerm.assign(userPerm, userPerm + n);
  prepare_subdomain(S, opt, 0, H, (helper & 1) != 0, (helper & 2) != 0);
  for (int a = 0; a < 4; a++) seconds[a] = H.stageS[a];
  uint64_t h = 1469598103934665603ull;
  auto mix = [&](const void* p, size_t bytes) {
    const unsigned char* c = (const unsigned char*)p;
    // 8 bytes at a time (FNV-like; the arrays are large)
    size_t i = 0;
    for (; i + 8 <= bytes; i += 8) { uint64_t v; memcpy(&v, c + i, 8); h = (h ^ v) * 1099511628211ull; }
    for (; i < bytes; i++) h = (h ^ c[i]) * 1099511628211ull;
  };
  const Symbolic& Y = H.plan->sym;
  mix(H.patP.ptr.data(), H.patP.ptr.size() * 8); mix(H.patP.idx.data(), H.patP.idx.size() * 4);
  mix(H.patP.val.data(), H.patP.val.size() * 8); mix(H.vNeuP.data(), H.vNeuP.size() * 8);
  mix(H.vRobP.data(), H.vRobP.size() * 8); mix(H.dP.data(), H.dP.size() * 8); mix(H.gidx.data(), H.gidx.size() * 4);
  mix(Y.perm.data(), Y.perm.size() * 4); mix(Y.rowIdx.data(), Y.rowIdx.size() * 4); mix(Y.rel.data(), Y.rel.size() * 4);
  // the scatter map as a set of (src, dst) pairs: order-independent sum of a pair hash
  uint64_t acc = 0;
  for (size_t t = 0; t < Y.asmSrc.size(); t++) {
    uint64_t v = (uint64_t)Y.asmSrc[t] * 0x9E3779B97F4A7C15ull ^ ((uint64_t)Y.asmDst[t] + 0x7F4A7C15ull) * 0xC2B2AE3D27D4EB4Full;
    v ^= v >> 29; v *= 0xBF58476D1CE4E5B9ull; v ^= v >> 32;
    acc += v;
  }
  mix(&acc, 8);
  const uint64_t na = Y.asmSrc.size();
  mix(&na, 8);
  for (const Front& F : Y.fronts) {
    const int64_t q[8] = {F.col0, F.k, F.h, F.parent, F.lOff, F.uOff, F.wOff, F.relOff};
    mix(q, sizeof(q));
  }
  *digest = h;
  if (scatterOut) {  // what the assembly kernel would write: the factor array holding the scattered lower triangle
    GENEO_CHECK(scatterLen == Y.lSize, "host_prepare_probe: scatterLen must be the factor size of the analysis");
    std::fill(scatterOut, scatterOut + scatterLen, 0.);
    for (size_t t = 0; t < Y.asmSrc.size(); t++) scatterOut[Y.asmDst[t]] = H.patP.val[(size_t)Y.asmSrc[t]];
  }
}

// one lane of the pipelined numeric setup (numeric_pipeline): a stream, its update arenas and a transient factor
struct GeneoPC::Lane {
  cudaStream_t st = nullptr;
  LdltWorkspace ws;
  DevBuf<double> T;          // transient factor (S, then A_neu) of the subdomain currently in the lane
  int* hc = nullptr;         // pinned: {neg, perturbed} of S, of A_neu, of A_dir
  cudaStream_t est = nullptr;  // the eigen-solve of the lane's subdomain: stream, Lanczos buffers, scalar scratch
  EigWorkspace eig;
  DevBuf<double> scal;
  ~Lane() { if (st) cudaStreamDestroy(st); if (est) cudaStreamDestroy(est); if (hc) cudaFreeHost(hc); }
};

// Lock-step block solves of the pencils of one lane group (EigOptions::solve): every member (one host thread each) hands in
// its right-hand side block; the last one to arrive launches ONE forest solve over the group's shift-invert factors.  A
// single 100^3 factor keeps the solve kernel in its level barriers (1.5 TB/s); four of them stream.  The group dissolves
// when its first member is done: the others finish their last steps alone.
struct GroupSolver {
  SolveForest forest;
  std::vector<const LdltPlan*> plans;
  std::vector<int64_t> off;      // first row of every member in the concatenated buffers
  DevBuf<double> xs, w;          // (sum n_i) x ld, row-major
  int ld = 0;
  cudaStream_t st = nullptr;
  std::vector<cudaEvent_t> evIn;
  cudaEvent_t evOut[2] = {nullptr, nullptr};
  std::mutex m;
  std::condition_variable cv;
  int members = 0, arrived = 0;
  long gen = 0, refused = 0;
  bool on = false;
  ~GroupSolver() {
    for (auto e : evIn) if (e) cudaEventDestroy(e);
    for (auto e : evOut) if (e) cudaEventDestroy(e);
    if (st) cudaStreamDestroy(st);
  }
  bool solve(int i, int j0, int nr, cudaStream_t ist) {
    CUDA_CHECK(cudaEventRecord(evIn[i], ist));
    std::unique_lock<std::mutex> lk(m);
    if (!on) { refused++; return false; }
    const long my = gen;
    if (++arrived == members) {
      try {
        for (int q = 0; q < members; q++) CUDA_CHECK(cudaStreamWaitEvent(st, evIn[q], 0));
        forest.solve(xs.p, w.p, ld, j0, nr, st);
        CUDA_CHECK(cudaEventRecord(evOut[my & 1], st));
      } catch (...) { on = false; arrived = 0; cv.notify_all(); throw; }
      arrived = 0;
      gen++;
      cv.notify_all();
    } else {
      cv.wait(lk, [&]() { return gen != my || !on; });
      if (gen == my) { arrived--; return false; }  // dissolved while waiting: solve alone
    }
    lk.unlock();
    CUDA_CHECK(cudaStreamWaitEvent(ist, evOut[my & 1], 0));
    return true;
  }
  void leave() {
    std::lock_guard<std::mutex> lk(m);
    on = false;
    cv.notify_all();
  }
};

GeneoPC::GeneoPC() {}
// The pipelined numeric setup needs a single level-2 pencil (GenEO-1) or none; GenEO-2, the launch profiler (events on ONE
// stream) and GENEO_PIPELINE=0 take the sequential path.
bool GeneoPC::use_pipeline() const {
  if (opt.lvl2 == 2 || g_profile || subs.empty()) return false;
  if (const char* e = getenv("GENEO_PIPELINE")) return atoi(e) != 0;
  return true;
}
GeneoPC::~GeneoPC() {
  try { write_timing_log(); } catch (...) {}
  for (auto s : streams) cudaStreamDestroy(s);
  for (auto e : events) cudaEventDestroy(e);
  for (auto e : ktEvents) cudaEventDestroy(e);
  if (evFork) cudaEventDestroy(evFork);
}

double GeneoPC::dot(const double* x, const double* y) {
  vec_dot(nOwn, x, y, scal.p, st);
  comm.allreduce_sum(scal.p, 1, st);
  double h = 0.;
  CUDA_CHECK(cudaMemcpyAsync(&h, scal.p, sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_CHECK(::geneo::sync_stream(st));
  return h;
}

void GeneoPC::mult(const double* x, double* y) {
  comm.halo_forward(const_cast<double*>(x), 1, st);  // only the ghost copies of x are written
  sell_spmv(A, x, y, st);
}
void GeneoPC::mult_sub(const double* x, const double* b, double* y) {
  comm.halo_forward(const_cast<double*>(x), 1, st);
  sell_spmv_sub(A, x, b, y, st);
}

void GeneoPC::setup(const Decomposition& dec, const RankLayout* layout, const void* ncclUid) {
  require_device();
  const double tSetup0 = now_s();
  // PCSetUp may be repeated on the same PC with a NEW problem / pattern: nothing of the previous one may survive (the
  // solve forest holds raw pointers into the old plans, subs[p].L1 is bound to the old plan, comm to the old layout)
  CUDA_CHECK(::geneo::sync_stream(st));
  subs.clear();
  groupSolvers.clear();
  lanes.clear();
  forest = SolveForest();
  factorWs = LdltWorkspace();
  eigWs.release();
  comm.reset();
  nE = 0; applyCount = 0; ktUsed = 0;
  nevGlobal.clear(); estimGlobal.clear();
  nbDof = dec.nbNode;
  nLoc = nOwn = nbDof;
  nbPart = dec.nbPart;
  scal.alloc(1024);
  std::vector<const Subdomain*> mine;
  distKeys = DistKeys();
  if (layout) {
    distKeys.dist = true;
    distKeys.rank = layout->rank;
    distKeys.world = layout->world;
    distKeys.subRank = layout->subRank;
    distKeys.owned = layout->owned;
    distKeys.ghost = layout->ghost;
    distKeys.ghostPtr = layout->ghostPtr;
    nOwn = layout->nOwn();
    nLoc = nOwn + layout->nGhost();
    for (auto& S : dec.subs)
      if (layout->subRank[S.id] == layout->rank) {
        GENEO_CHECK(S.aNeu.n > 0, "multi-GPU setup: a local subdomain has no matrices");
        mine.push_back(&S);
      }
    comm.init(layout->rank, layout->world, ncclUid, *layout, st);
  } else {
    for (auto& S : dec.subs)
      if (S.aNeu.n > 0) mine.push_back(&S);
    GENEO_CHECK((int)mine.size() == dec.nbPart, "single-process setup needs every subdomain's matrices");
  }
  auto localIndex = [&](int g) -> int { return layout ? layout->local(g) : g; };
  if (opt.lvl2 == 2 && !opt.lvl1ORAS)
    throw Error("geneo_b200: GenEO-2 needs an optimised level 1 (ORAS/SORAS) -- untested/unsupported in the reference too");

  double t0 = now_s();
  // ---- pipeline: worker threads do the host analysis of the subdomains IN ORDER (a few at a time, each one using the
  //      other cores for the top levels of its nested dissection) while this thread uploads and runs the whole numeric
  //      phase of every subdomain that is ready -> the device factorizes subdomain p while the host orders p+1, p+2.
  t0 = now_s();
  const int P = (int)mine.size();
  std::vector<HostPrep> prep(P);
  subs.resize(P);
  nAll = 0;
  for (int p = 0; p < P; p++) { subs[p].id = mine[p]->id; subs[p].n = (int)mine[p]->nodes.size(); subs[p].off = nAll; nAll += subs[p].n; }
  connectivity.assign((size_t)dec.nbPart * dec.nbPart, 0);
  for (int r = 0; r < dec.nbPart; r++)
    for (int q = 0; q < dec.nbPart; q++) connectivity[(size_t)r * dec.nbPart + q] = dec.subs[r].intersect[q].empty() ? 1 : 0;
  if (layout && comm.active()) {  // a rank only knows the intersections of ITS subdomains: rows are summed over the ranks
    std::vector<double> c((size_t)dec.nbPart * dec.nbPart, 0.);
    for (int r = 0; r < dec.nbPart; r++)
      if (layout->subRank[r] == layout->rank)
        for (int q = 0; q < dec.nbPart; q++) c[(size_t)r * dec.nbPart + q] = connectivity[(size_t)r * dec.nbPart + q];
    comm.allreduce_sum_host(c.data(), (int)c.size(), st);
    for (size_t t = 0; t < c.size(); t++) connectivity[t] = c[t] > 0.5 ? 1 : 0;
  }
  // host threads of THIS process: all cores, divided by the ranks sharing the node (torchrun exports LOCAL_WORLD_SIZE)
  unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  if (const char* e = getenv("GENEO_HOST_THREADS")) hw = (unsigned)std::max(1, atoi(e));
  else if (const char* e2 = getenv("LOCAL_WORLD_SIZE")) hw = std::max(1u, hw / (unsigned)std::max(1, atoi(e2)));
  int inFlight = std::max(1, std::min(P, hw >= 8 ? 2 : 1));  // subdomains analysed concurrently
  int ndDepth = 0;
  while ((unsigned)(inFlight << (ndDepth + 1)) <= hw && ndDepth < 4) ndDepth++;
  std::mutex mtx;
  std::condition_variable cv;
  std::vector<char> ready(P, 0);
  std::atomic<int> ticket(0);
  std::vector<std::thread> pool;
  std::string orchErr;
  bool sideThreads = false;
  // The shared reference ordering (one METIS call for all box subdomains) and then the analysis workers are started from
  // an orchestrating thread: this thread assembles and uploads the operator meanwhile.  Single process only -- with
  // several ranks the ordering is a collective on the library's stream and stays on this thread.
  auto orchestrate = [&]() {
    try {
      const double tr = now_s();
      const unsigned hwAll = getenv("GENEO_HOST_THREADS") ? hw : std::max(1u, std::thread::hardware_concurrency());
      plan_ordering_reuse(dec, mine, opt, comm, hwAll, st, prep);
      orderingReuseTime = now_s() - tr;
      int nInherit = 0;
      for (auto& H : prep) nInherit += H.userPerm.empty() ? 0 : 1;
      if (nInherit == P) { inFlight = std::max(1, std::min<int>(P, (int)hw)); ndDepth = 0; }  // no METIS call left: one thread per subdomain
      sideThreads = (unsigned)(2 * inFlight) <= hw;  // a second thread per subdomain for the ordering-independent part
    } catch (std::exception& e) { orchErr = e.what(); }
    for (int w = 0; w < inFlight; w++)
      pool.emplace_back([&]() {
        for (;;) {
          const int p = ticket.fetch_add(1);
          if (p >= P) break;
          if (!orchErr.empty()) prep[p].err = orchErr;
          else try { prepare_subdomain(*mine[p], opt, ndDepth, prep[p], sideThreads); } catch (std::exception& e) { prep[p].err = e.what(); }
          { std::lock_guard<std::mutex> lk(mtx); ready[p] = 1; }
          cv.notify_all();
        }
      });
  };
  std::thread orch;
  struct Joiner {
    std::thread& o; std::vector<std::thread>& t;
    ~Joiner() { if (o.joinable()) o.join(); for (auto& x : t) if (x.joinable()) x.join(); }
  } joiner{orch, pool};
  if (layout && comm.active()) orchestrate();
  else orch = std::thread(orchestrate);

  // (assembled by this thread while the workers are already busy with the first subdomains)
  // ---- operator A = sum_i R_i^T A_neu,i R_i  (MatConvert MATIS->AIJ, src/geneo.cpp:1692), SELL-32 on the device ------
  t0 = now_s();
  if (layout) {
    A.build(layout->A, st);  // owned rows, assembled from the elements (mesh.cpp build_rank_layout)
  } else {
    CsrHost g;
    g.n = g.ncols = nLoc;
    std::vector<int64_t> cnt(nLoc + 1, 0);
    for (auto* S : mine)
      for (int l = 0; l < S->aNeu.n; l++) cnt[S->nodes[l] + 1] += S->aNeu.ptr[l + 1] - S->aNeu.ptr[l];
    for (int i = 0; i < nLoc; i++) cnt[i + 1] += cnt[i];
    std::vector<int> ci((size_t)cnt[nLoc]);
    std::vector<double> cv((size_t)cnt[nLoc]);
    {
      std::vector<int64_t> pos(cnt.begin(), cnt.end() - 1);
      for (auto* S : mine)
        for (int l = 0; l < S->aNeu.n; l++) {
          int64_t& p = pos[S->nodes[l]];
          for (int64_t t = S->aNeu.ptr[l]; t < S->aNeu.ptr[l + 1]; t++) { ci[p] = S->nodes[S->aNeu.idx[t]]; cv[p] = S->aNeu.val[t]; p++; }
        }
    }
    // sort + merge every row (a node shared by subdomains gets one partial row from each): rows are independent, so the
    // pass is split over the host threads (it is on the critical path of the cold setup: the device waits for A)
    g.ptr.assign(nLoc + 1, 0);
    const int nth = (int)std::max(1u, std::min(hw, 32u));
    auto for_rows = [&](auto&& fn) {
      std::vector<std::thread> ths;
      for (int t = 0; t < nth; t++)
        ths.emplace_back([&, t]() {
          const int i0 = (int)((int64_t)nLoc * t / nth), i1 = (int)((int64_t)nLoc * (t + 1) / nth);
          fn(i0, i1);
        });
      for (auto& th : ths) th.join();
    };
    for_rows([&](int i0, int i1) {  // pass 1: sort each row segment in place, merge duplicates to its front, count
      std::vector<std::pair<int, double>> row;
      for (int i = i0; i < i1; i++) {
        row.clear();
        for (int64_t t = cnt[i]; t < cnt[i + 1]; t++) row.emplace_back(ci[t], cv[t]);
        std::stable_sort(row.begin(), row.end(), [](const std::pair<int, double>& a, const std::pair<int, double>& b) { return a.first < b.first; });
        int64_t w = cnt[i];
        for (size_t k = 0; k < row.size();) {
          const int c = row[k].first;
          double sum = 0.;
          while (k < row.size() && row[k].first == c) { sum += row[k].second; k++; }
          ci[w] = c; cv[w] = sum; w++;
        }
        g.ptr[i + 1] = w - cnt[i];
      }
    });
    for (int i = 0; i < nLoc; i++) g.ptr[i + 1] += g.ptr[i];
    g.idx.resize((size_t)g.ptr[nLoc]); g.val.resize((size_t)g.ptr[nLoc]);
    for_rows([&](int i0, int i1) {  // pass 2: compact
      for (int i = i0; i < i1; i++) {
        const int64_t len = g.ptr[i + 1] - g.ptr[i];
        std::copy(ci.begin() + cnt[i], ci.begin() + cnt[i] + len, g.idx.begin() + g.ptr[i]);
        std::copy(cv.begin() + cnt[i], cv.begin() + cnt[i] + len, g.val.begin() + g.ptr[i]);
      }
    });
    A.build(g, st);
  }
  operatorTime = now_s() - t0;


  numeric_begin();
  const bool pipelined = use_pipeline();
  LdltWorkspace& ws = factorWs;
  std::vector<int> gAll((size_t)nAll);
  std::vector<double> dA((size_t)nAll);
  double waitHost = 0., tUp = 0., tNum = 0.;
  for (int p = 0; p < P; p++) {
    {
      const double tw = now_s();
      std::unique_lock<std::mutex> lk(mtx);
      cv.wait(lk, [&]() { return ready[p] != 0; });
      waitHost += now_s() - tw;
    }
    HostPrep& H = prep[p];
    if (!H.err.empty()) throw Error(H.err);
    const double tu = now_s();
    SubdomainState& s = subs[p];
    for (int k = 0; k < s.n; k++) {
      const int li = localIndex(H.gidx[k]);
      GENEO_CHECK(li >= 0, "multi-GPU layout: a subdomain node is neither owned nor ghost");
      H.gidx[k] = li;
      gAll[s.off + k] = li;
      dA[s.off + k] = H.dP[k];
    }
    s.maxMult = H.maxMult;
    s.anorm = H.anorm;
    s.neuNnz = mine[p]->aNeu.nnz();
    s.plan = H.plan;
    s.plan->upload();
    s.pat.upload_pattern(H.patP, st);
    s.vNeu.upload(H.vNeuP, st);
    if (opt.lvl1ORAS) s.vRob.upload(H.vRobP, st);
    s.gidx.upload(H.gidx, st);
    s.d.upload(H.dP, st);
    CUDA_CHECK(::geneo::sync_stream(st));
    H = HostPrep();  // free host memory early
    tUp += now_s() - tu;
    if (!pipelined) {  // one subdomain after the other: the device factorizes p while the host still orders p+1, p+2
      const double tn = now_s();
      numeric_subdomain(s, ws);
      tNum += now_s() - tn;
    }
  }
  if (pipelined) {
    const double tn = now_s();
    numeric_pipeline();
    tNum += now_s() - tn;
  }
  if (opt.releaseWorkspace) { factorWs = LdltWorkspace(); eigWs.release(); groupSolvers.clear(); lanes.clear(); }
  symbolicTime = waitHost;  // time this thread spent WAITING for the host analysis (the rest of it was hidden behind the device)
  uploadTime = tUp;

  // ---- concatenated subdomain layout, pull-prolong structure ---------------------------------------------------------------
  t0 = now_s();
  {
    std::vector<int64_t> pp(nLoc + 1, 0);
    for (int64_t t = 0; t < nAll; t++) pp[gAll[t] + 1]++;
    for (int i = 0; i < nLoc; i++) pp[i + 1] += pp[i];
    std::vector<int64_t> ps((size_t)nAll);
    std::vector<int64_t> cur(pp.begin(), pp.end() - 1);
    for (int64_t t = 0; t < nAll; t++) ps[cur[gAll[t]]++] = t;  // ascending subdomain id inside every row: deterministic sums
    gidxAll.upload(gAll, st);
    dAll.upload(dA, st);
    pullPtr.upload(pp, st);
    pullPos.upload(ps, st);
    CUDA_CHECK(::geneo::sync_stream(st));
  }
  Xall.alloc((size_t)nAll); Yall.alloc((size_t)nAll);
  t1.alloc(nLoc); t2.alloc(nLoc); t3.alloc(nLoc);
  uploadTime += now_s() - t0;
  const double te = now_s();
  numeric_end();
  numericTime = tNum + (now_s() - te);
  setupTime = now_s() - tSetup0;
}

void GeneoPC::numeric_begin() {
  lvl1SetupMinvTime = lvl2SetupSylTime = lvl2SetupEigTime = lvl2SetupZTime = lvl2SetupETime = 0.;
  lvl2SetupTauLocTime = lvl2SetupTauSylTime = lvl2SetupTauEigTime = 0.;
  lvl2SetupGammaLocTime = lvl2SetupGammaSylTime = lvl2SetupGammaEigTime = 0.;
  estimDimE = realDimE = nicolaides = 0;
  factorBytes = factorNnz = 0;
  factorFlops = 0.;
  allFactorSeconds = allFactorFlops = 0.;
  allFactorCount = 0;
  for (auto& s : subs) {
    s.prevNev = std::max(s.prevNev, s.nev);  // (sizes the memory reserve of the next pipelined setup)
    s.estim = s.nicolaides = s.eigSteps = s.eigDim = s.negL1 = s.perturbed = 0;
    s.nev = 0;
  }
}

void GeneoPC::numeric_end() {
  HostProfScope hpEnd("numeric_end");
  if (comm.active()) {  // the driver prints GLOBAL dimensions (src/geneo4PETSc.cpp:971-986 reduces them over the ranks)
    double g[3] = {(double)estimDimE, (double)realDimE, (double)nicolaides};
    comm.allreduce_sum_host(g, 3, st);
    estimDimE = (int)std::lround(g[0]); realDimE = (int)std::lround(g[1]); nicolaides = (int)std::lround(g[2]);
  }
  if (opt.lvl2 == 0) {
    nevGlobal.assign(nbPart, 0);
    estimGlobal.assign(nbPart, 0);
  }
  {  // the forest of all level-1 factors
    std::vector<const LdltPlan*> plans;
    std::vector<int64_t> xoff;
    std::vector<const double*> Ls;
    for (auto& s : subs) { plans.push_back(s.plan.get()); xoff.push_back(s.off); Ls.push_back(s.L1->L.p); }
    const double tf = now_s();
    if (forest.nlev == 0) forest.build(plans, xoff);
    forest.set_factors(Ls, st);
    if (getenv("GENEO_COLD_TIMING")) fprintf(stderr, "COLD rank %d: level-1 forest %.3f s\n", comm.rank, now_s() - tf);
  }
  if (opt.lvl2 >= 1) {
    const double te = now_s();
    build_coarse();
    lvl2SetupETime = now_s() - te;
    if (getenv("GENEO_COLD_TIMING")) fprintf(stderr, "COLD rank %d: coarse operator %.3f s\n", comm.rank, lvl2SetupETime);
    infoL2 = "blocklanczos ldlt";
  }
  CUDA_CHECK(::geneo::sync_stream(st));
  if (opt.check || opt.debug >= 2) run_checks_and_dumps();
}

// ---- -geneo_chk / -geneo_dbg (diagnostics; file names follow the reference: one prefix per subdomain = per MPI rank there) -----
namespace {
std::string diag_prefix(const char* what, int id, int nbPart) {
  const int w = (int)std::to_string(nbPart).size();
  std::string r = std::to_string(id);
  while ((int)r.size() < w) r = "0" + r;
  return std::string(what) + r;
}
}  // namespace

void GeneoPC::run_checks_and_dumps() {
  for (auto& s : subs) {
    if (opt.debug >= 2) {
      const std::string pre = diag_prefix("debug", s.id, nbPart);
      if (opt.lvl2 >= 1) {
        FILE* f = fopen((pre + ".setup.Z.ev.log").c_str(), "w");  // src/geneo.cpp:344-349
        if (f) {
          fprintf(f, "\nZ - nb of eigen values: %d\n", (int)s.eigvals.size());
          for (size_t e = 0; e < s.eigvals.size(); e++) fprintf(f, "Z - eigen value %d: %.17g\n", (int)e, s.eigvals[e]);
          fclose(f);
        }
        const char* pb[2] = {"tau", "gamma"};
        for (int q = 0; q < (opt.lvl2 == 2 ? 2 : 1); q++) {
          if (opt.noSyl) continue;
          f = fopen((pre + ".setup." + pb[q] + ".sylvester.inertia.log").c_str(), "w");  // :547-551
          if (!f) continue;
          fprintf(f, "\nnbNegEV %d, nbNullEV %d, nbPosEV %d => estim %d\n", s.sylNeg[q], s.sylNull[q], s.n - s.sylNeg[q] - s.sylNull[q], s.sylEstim[q]);
          fclose(f);
        }
      }
    }
    if (opt.check) {
      const std::string pre = diag_prefix("check", s.id, nbPart);
      // partition of unity (src/geneo.cpp:988-997): min D > 0
      std::vector<double> d = s.d.to_host(st);
      double dmin = d.empty() ? 1. : *std::min_element(d.begin(), d.end());
      if (std::fabs(dmin) <= DBL_EPSILON) throw Error("geneo_b200: GenEO - check D: bad partition of unity, min " + std::to_string(dmin));
      // SPD of the level-1 matrix through the inertia of its factorization (checkSPD, :782-840: the inertia half)
      {
        const char* info = opt.lvl1ORAS ? "ARob" : "ADir";
        FILE* f = fopen((pre + ".SPD." + info + ".log").c_str(), "w");
        if (f) {
          fprintf(f, "\n%s - inertia: nbNegEV %d, nbNullEV %d, nbPosEV %d\n", info, s.negL1, 0, s.n - s.negL1);
          fclose(f);
        }
        if (s.negL1 > 0) throw Error("geneo_b200: GenEO - check SPD: not SPD (inertia - negative or null eigen value found)");
      }
      // rank of Z_i (checkRank, :173-247): Z = Q R by modified Gram-Schmidt with refinement on the host, diag(R) != 0
      if (opt.lvl2 >= 1 && s.nev > 0) {
        std::vector<double> z = s.Z.to_host(st);  // n x nev row-major
        const int n = s.n, k = s.nev;
        std::vector<double> R((size_t)k * k, 0.), col(n);
        for (int j = 0; j < k; j++) {
          for (int pass = 0; pass < 2; pass++)
            for (int i = 0; i < j; i++) {
              double dot = 0.;
              for (int r = 0; r < n; r++) dot += z[(size_t)r * k + i] * z[(size_t)r * k + j];
              R[(size_t)i * k + j] += dot;
              for (int r = 0; r < n; r++) z[(size_t)r * k + j] -= dot * z[(size_t)r * k + i];
            }
          double nrm = 0.;
          for (int r = 0; r < n; r++) nrm += z[(size_t)r * k + j] * z[(size_t)r * k + j];
          nrm = std::sqrt(nrm);
          R[(size_t)j * k + j] = nrm;
          if (nrm > 0.) for (int r = 0; r < n; r++) z[(size_t)r * k + j] /= nrm;
        }
        FILE* f = fopen((pre + ".setup.Z.R").c_str(), "w");
        if (f) {
          for (int i = 0; i < k; i++) { for (int j = 0; j < k; j++) fprintf(f, "%.10e ", R[(size_t)i * k + j]); fprintf(f, "\n"); }
          fclose(f);
        }
        for (int j = 0; j < k; j++)
          if (std::fabs(R[(size_t)j * k + j]) <= DBL_EPSILON)
            throw Error("geneo_b200: GenEO - check rank: Z = Q*R with R(" + std::to_string(j) + ", " + std::to_string(j) + ") = " + std::to_string(R[(size_t)j * k + j]));
      }
    }
  }
}

void GeneoPC::write_timing_log() const {
  if (opt.debug < 1) return;
  for (auto& s : subs) {
    FILE* f = fopen((diag_prefix("debug", s.id, nbPart) + ".timing.log").c_str(), "w");
    if (!f) continue;
    const struct { const char* n; double v; } T[] = {
        {"lvl1SetupMinvTimeLoc", lvl1SetupMinvTime}, {"lvl1ApplyTimeLoc", lvl1ApplyTime}, {"lvl1ApplyScatterTimeLoc", lvl1ApplyScatterTime},
        {"lvl1ApplyMinvTimeLoc", lvl1ApplyMinvTime}, {"lvl1ApplyGatherTimeLoc", lvl1ApplyGatherTime}, {"lvl1ApplyPrjFSTimeLoc", lvl1ApplyPrjFSTime},
        {"lvl2SetupTauLocTimeLoc", lvl2SetupTauLocTime}, {"lvl2SetupTauSylTimeLoc", lvl2SetupTauSylTime}, {"lvl2SetupTauEigTimeLoc", lvl2SetupTauEigTime},
        {"lvl2SetupGammaLocTimeLoc", lvl2SetupGammaLocTime}, {"lvl2SetupGammaSylTimeLoc", lvl2SetupGammaSylTime},
        {"lvl2SetupGammaEigTimeLoc", lvl2SetupGammaEigTime}, {"lvl2SetupSylTimeLoc", lvl2SetupSylTime}, {"lvl2SetupEigTimeLoc", lvl2SetupEigTime},
        {"lvl2SetupZTimeLoc", lvl2SetupZTime}, {"lvl2SetupETimeLoc", lvl2SetupETime}, {"lvl2ApplyTimeLoc", lvl2ApplyTime},
        {"lvl2ApplyZtTimeLoc", lvl2ApplyZtTime}, {"lvl2ApplyEinvTimeLoc", lvl2ApplyEinvTime}, {"lvl2ApplyZTimeLoc", lvl2ApplyZTime}};
    for (auto& t : T) fprintf(f, "%-26s%g ms\n", t.n, 1e3 * t.v);  // (this GPU holds every local subdomain: the timers are per process)
    fclose(f);
  }
}

void GeneoPC::numeric_setup() {
  const double tNum0 = now_s();
  numeric_begin();
  if (use_pipeline()) numeric_pipeline();
  else for (auto& s : subs) numeric_subdomain(s, factorWs);
  if (opt.releaseWorkspace) { factorWs = LdltWorkspace(); eigWs.release(); groupSolvers.clear(); lanes.clear(); }
  numeric_end();
  numericTime = now_s() - tNum0;
  host_prof_add("numeric_setup total", numericTime);
  host_prof_report("numeric_setup");
}

// Same-pattern update.  Everything the setup derived from the pattern stays: plans (dPerm), the permuted A_dir pattern,
// gidx, d, the operator's SELL layout, lanes and workspaces.  Per subdomain the new CSR matrices go up through one staging
// set sized for the largest subdomain and are located on the device in the setup's pattern; the values land in fresh
// buffers (PendingValues), and the counters of every check are read back once.  Only commit_values() writes resident values.
// With a layout (multi-GPU) gidx is rank-local and the operator holds only the owned rows, assembled from the elements:
// node ids are compared in the layout's local numbering, A_neu is not located in the operator, and the layout's owned rows
// are checked against the operator's pattern and placed into nv.op instead.
void GeneoPC::check_values(const Decomposition& dec, PendingValues& nv, const RankLayout* layout) {
  require_device();
  const int P = (int)subs.size();
  GENEO_CHECK(P > 0 && (layout != nullptr) == distKeys.dist, "update: the preconditioner is not set up for this kind of update");
  auto fail = [](const std::string& m) { throw Error("geneo_b200: same-pattern update: " + m); };
  if (dec.nbPart != nbPart)
    fail("the problem has " + std::to_string(dec.nbPart) + " subdomains, the preconditioner was set up with " + std::to_string(nbPart));
  if (dec.nbNode != nbDof)
    fail("the problem has " + std::to_string(dec.nbNode) + " DOFs, the preconditioner was set up with " + std::to_string(nbDof));
  int nMax = 0;
  int64_t zMax = 0;
  for (int p = 0; p < P; p++) {
    const Subdomain& S = dec.subs[subs[p].id];
    const SubdomainState& s = subs[p];
    const std::string sub = "subdomain " + std::to_string(s.id) + ": ";
    if (S.id != s.id || (int)S.nodes.size() != s.n) fail(sub + "the node set differs from the setup's (another partition?)");
    if (S.aNeu.n != s.n || S.aDir.n != s.n) fail(sub + "no matrices on this process");
    if (S.aDir.nnz() != s.pat.nnz)
      fail(sub + "A_dir has " + std::to_string(S.aDir.nnz()) + " entries, the pattern of the setup " + std::to_string(s.pat.nnz));
    if (S.aNeu.nnz() != s.neuNnz)
      fail(sub + "A_neu has " + std::to_string(S.aNeu.nnz()) + " entries, the pattern of the setup " + std::to_string(s.neuNnz));
    nMax = std::max(nMax, s.n);
    zMax = std::max(zMax, s.pat.nnz);
  }
  if (layout) zMax = std::max<int64_t>(zMax, layout->A.nnz());  // the staging set carries the owned rows too
  CUDA_CHECK(::geneo::sync_stream(st));
  DevBuf<int64_t> dPtr((size_t)std::max(nMax, layout ? nOwn : 0) + 1);
  DevBuf<int> dIdx((size_t)zMax), dNodes((size_t)nMax), dIperm((size_t)nMax), hits((size_t)zMax);
  DevBuf<double> dVal((size_t)zMax);
  DevBuf<unsigned long long> cnt((size_t)P * UPD_SLOTS + 1);  // + the operator entries no A_neu reached / owned rows that differ
  DevBuf<unsigned char> cover(layout ? 0 : (size_t)A.stored);
  cnt.zero(st);
  cover.zero(st);
  nv.subs.clear();
  nv.subs.resize(P);
  std::vector<int> local;
  for (int p = 0; p < P; p++) {
    const Subdomain& S = dec.subs[subs[p].id];
    SubdomainState& s = subs[p];
    const int n = s.n;
    const int64_t nnz = s.pat.nnz, nnzNeu = s.neuNnz;
    unsigned long long* c = cnt.p + (size_t)p * UPD_SLOTS;
    PendingValues::Sub& w = nv.subs[p];
    w.dir.alloc((size_t)nnz);
    w.neu.alloc((size_t)nnz);
    w.neu.zero(st);
    if (!layout) {
      w.slot.alloc((size_t)nnz);
      CUDA_CHECK(cudaMemsetAsync(w.slot.p, 0xff, (size_t)nnz * sizeof(int64_t), st));  // -1: off the A_neu pattern
    }
    CUDA_CHECK(cudaMemsetAsync(hits.p, 0, (size_t)nnz * sizeof(int), st));
    if (layout) {  // gidx holds local indices: compare against the new layout's numbering of the node ids
      local.resize((size_t)n);
      for (int l = 0; l < n; l++) local[l] = layout->local(S.nodes[l]);
      dNodes.upload(local.data(), (size_t)n, st);
    } else {
      dNodes.upload(S.nodes.data(), (size_t)n, st);
    }
    update_nodes(n, s.plan->dPerm.p, s.gidx.p, dNodes.p, dIperm.p, c, st);
    dPtr.upload(S.aDir.ptr.data(), (size_t)n + 1, st);
    dIdx.upload(S.aDir.idx.data(), (size_t)nnz, st);
    dVal.upload(S.aDir.val.data(), (size_t)nnz, st);
    update_locate_dir(n, nnz, dPtr.p, dIdx.p, dVal.p, dIperm.p, s.pat.ptr.p, s.pat.idx.p, hits.p, w.dir.p, c, st);
    update_absmax(nnz, w.dir.p, c + UPD_ANORM, st);
    dPtr.upload(S.aNeu.ptr.data(), (size_t)n + 1, st);
    dIdx.upload(S.aNeu.idx.data(), (size_t)nnzNeu, st);
    dVal.upload(S.aNeu.val.data(), (size_t)nnzNeu, st);
    update_locate_neu(n, nnzNeu, dPtr.p, dIdx.p, dVal.p, dIperm.p, s.gidx.p, s.pat.ptr.p, s.pat.idx.p, hits.p, A, w.neu.p, w.slot.p,
                      cover.p, c, st);
  }
  if (layout) {
    const CsrHost& R = layout->A;
    GENEO_CHECK(R.n == nOwn, "update: the rebuilt layout has another number of owned rows");
    nv.op.alloc(A.val.n);
    nv.op.zero(st);  // the padding of the SELL layout
    dPtr.upload(R.ptr.data(), (size_t)R.n + 1, st);
    dIdx.upload(R.idx.data(), (size_t)R.nnz(), st);
    dVal.upload(R.val.data(), (size_t)R.nnz(), st);
    update_owned_rows(A, R.nnz(), dPtr.p, dIdx.p, dVal.p, nv.op.p, cnt.p + (size_t)P * UPD_SLOTS, st);
  } else {
    update_cover_check(A, cover.p, cnt.p + (size_t)P * UPD_SLOTS, st);
  }
  const std::vector<unsigned long long> h = cnt.to_host(st);  // the only read-back
  static const char* what[UPD_ANORM] = {
      "node ids differ from the setup's", "A_dir rows whose length differs from the setup's", "A_dir entries outside the setup's pattern",
      "duplicate A_dir entries", "A_neu entries outside the A_dir pattern", "duplicate A_neu entries",
      "A_neu entries outside the operator's pattern"};
  for (int p = 0; p < P; p++)
    for (int e = 0; e < UPD_ANORM; e++)
      if (h[(size_t)p * UPD_SLOTS + e])
        fail("subdomain " + std::to_string(subs[p].id) + ": " + std::to_string(h[(size_t)p * UPD_SLOTS + e]) + " " + what[e]);
  if (h[(size_t)P * UPD_SLOTS])
    fail(std::to_string(h[(size_t)P * UPD_SLOTS]) +
         (layout ? " owned rows of the operator differ from the setup's pattern" : " entries of the operator are in no subdomain's A_neu"));
  for (int p = 0; p < P; p++) memcpy(&nv.subs[p].anorm, &h[(size_t)p * UPD_SLOTS + UPD_ANORM], sizeof(double));
}

void GeneoPC::check_values_dist(const Mesh* mesh, const Decomposition* dec, PendingValues& nv) {
  GENEO_CHECK(distKeys.dist, "update: the preconditioner is not set up on several GPUs");
  const DistKeys& K = distKeys;
  std::string err;
  try {
    auto fail = [](const std::string& m) { throw Error("geneo_b200: same-pattern update: " + m); };
    if (!mesh || !dec) fail("this rank has no decomposed problem");
    if (dec->nbPart != nbPart)
      fail("the problem has " + std::to_string(dec->nbPart) + " subdomains, the preconditioner was set up with " + std::to_string(nbPart));
    const double t0 = now_s();
    RankLayout L;
    build_rank_layout(*mesh, *dec, K.subRank, K.rank, K.world, L);
    updateLayoutTime = now_s() - t0;
    if (L.owned != K.owned || L.ghost != K.ghost || L.ghostPtr != K.ghostPtr)
      fail("the rank's owned / ghost nodes differ from the setup's (another partition or sub_rank?)");
    check_values(*dec, nv, &L);
  } catch (std::exception& e) {
    err = e.what();
  }
  std::vector<double> vote((size_t)K.world, 0.);  // 1 where a rank rejects the update
  vote[K.rank] = err.empty() ? 0. : 1.;
  comm.allreduce_sum_host(vote.data(), K.world, st);
  if (!err.empty()) throw Error(err);
  for (int q = 0; q < K.world; q++)
    if (vote[q] > 0.5)
      throw Error("geneo_b200: same-pattern update rejected by rank " + std::to_string(q) +
                  " (its own message gives the reason); the preconditioner is left as it was");
}

// The checked values replace the resident ones.  Operator, one process: zero, then + A_neu,p subdomain by subdomain in
// ascending order -- the host merge of setup() sums 0 + a_1 + a_2 ... in the same order, so A, mult() and everything
// downstream match a fresh setup bit for bit.  Multi-GPU: the owned rows placed by check_values (no sum) become A's values.
void GeneoPC::commit_values(PendingValues& nv) {
  GENEO_CHECK(nv.subs.size() == subs.size(), "commit_values: the pending values do not belong to this preconditioner");
  GENEO_CHECK(!distKeys.dist || nv.op.n == A.val.n, "commit_values: the pending operator does not belong to this preconditioner");
  if (distKeys.dist) A.val = std::move(nv.op);
  else CUDA_CHECK(cudaMemsetAsync(A.val.p, 0, A.val.bytes(), st));
  for (size_t p = 0; p < subs.size(); p++) {
    SubdomainState& s = subs[p];
    PendingValues::Sub& w = nv.subs[p];
    s.anorm = w.anorm;
    s.pat.val = std::move(w.dir);
    s.vNeu = std::move(w.neu);
    if (!distKeys.dist) update_sell_add(s.pat.nnz, w.slot.p, s.vNeu.p, A, st);
    if (opt.lvl1ORAS) {  // createRobinMatrix, as prepare_subdomain does it
      if ((int64_t)s.vRob.n != s.pat.nnz) s.vRob.alloc((size_t)s.pat.nnz);
      if (std::fabs(opt.optim) > DBL_EPSILON) update_robin(s.n, s.pat.ptr.p, s.pat.idx.p, s.d.p, s.pat.val.p, s.vNeu.p, opt.optim, s.vRob.p, st);
      else CUDA_CHECK(cudaMemcpyAsync(s.vRob.p, s.pat.val.p, s.pat.val.bytes(), cudaMemcpyDeviceToDevice, st));
    }
  }
  CUDA_CHECK(::geneo::sync_stream(st));
}

void GeneoPC::level_profile(std::vector<double>& us, std::vector<double>& bytes, std::vector<int64_t>& nitems) {
  CUDA_CHECK(::geneo::sync_stream(st));
  Xall.zero(st);
  CUDA_CHECK(::geneo::sync_stream(st));
  forest.solve_profile(Xall.p, Yall.p, 1, us, bytes, nitems);
}

void GeneoPC::kernel_time(double* ms, int64_t* launches) {
  CUDA_CHECK(::geneo::sync_stream(st));
  double tot = 0.;
  for (size_t i = 0; i + 1 < ktUsed; i += 2) {
    float t = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&t, ktEvents[i], ktEvents[i + 1]));
    tot += t;
  }
  if (ms) *ms = tot;
  if (launches) *launches = (int64_t)(ktUsed / 2);
  ktUsed = 0;
}

// getLocalGenEOGamma, src/geneo.cpp:1120-1232 (connectivity quirk reproduced)
double GeneoPC::local_gamma(const SubdomainState& s) const {
  const int NP = nbPart;
  std::vector<double> C((size_t)NP * NP, 0.), F(NP, 0.), wv(NP);
  for (int r = 0; r < NP; r++)
    for (int q = 0; q < NP; q++)
      C[(size_t)r * NP + q] = (r == q) ? 1. : (connectivity[(size_t)r * NP + q] ? 1. : 0.);
  for (int r = 0; r < NP; r++) { double sum = 0.; for (int q = 0; q < NP; q++) sum += C[(size_t)r * NP + q]; F[r] = 1. / sum; }
  for (int r = 0; r < NP; r++) for (int q = 0; q < NP; q++) C[(size_t)r * NP + q] *= F[r] * F[q];
  sym_eig(NP, C.data(), wv.data());
  double lam = wv[0];
  for (int r = 0; r < NP; r++) if (std::fabs(wv[r]) > std::fabs(lam)) lam = wv[r];
  double gl = opt.gamma / lam * F[s.id] * F[s.id];
  if (gl <= 1.) gl = 1.1;
  return gl;
}

// Z_s = D [v_1 ... v_nev]  (fillZE2L, src/geneo.cpp:249-272); empty => constant vector (:1305-1314)
void GeneoPC::assemble_z(SubdomainState& s, std::vector<double>& vals, std::vector<DevBuf<double>>& vecs, std::vector<int>& counts,
                         cudaStream_t zs) {
  int nev = 0;
  for (int c : counts) nev += c;
  const double tz = now_s();
  if (nev == 0) {
    s.nev = 1;
    s.Z.alloc((size_t)s.n);
    CUDA_CHECK(cudaMemcpyAsync(s.Z.p, s.d.p, sizeof(double) * s.n, cudaMemcpyDeviceToDevice, zs));  // D * 1
    s.eigvals.assign(1, 0.);
    s.nicolaides += 1;
  } else {
    s.nev = nev;
    s.Z.alloc((size_t)s.n * nev);
    int c0 = 0;
    for (size_t b = 0; b < vecs.size(); b++) {
      const int nc = counts[b];
      if (nc == 0) continue;
      copy_cols(s.n, vecs[b].p, nc, s.Z.p + c0, nev, nc, zs);
      c0 += nc;
    }
    rows_scale(s.n, nev, s.d.p, s.Z.p, zs);  // Z = D V
    s.eigvals = vals;
  }
  CUDA_CHECK(::geneo::sync_stream(zs));
  {  // (several eigen threads of a lane group end here)
    static std::mutex zTimerMtx;
    std::lock_guard<std::mutex> lk(zTimerMtx);
    lvl2SetupZTime += now_s() - tz;
  }
}

// every factorization and eigen-solve of one subdomain, one after the other on the library's stream (level 2 first: its
// factors are transient).  GenEO-2 and the fallback of the pipelined path (numeric_pipeline).
void GeneoPC::numeric_subdomain(SubdomainState& s, LdltWorkspace& ws) {
  HostProfScope hpSub("numeric_subdomain");
  const double pivTol = opt.pivRel * std::max(s.anorm, 1e-300);
  if (opt.lvl2 >= 1) {
    std::vector<double> vals;
    std::vector<DevBuf<double>> vecs;
    std::vector<int> counts;
    int cut = opt.cut;
    if (opt.lvl2 == 2 && cut >= 2) cut = cut / 2;  // src/geneo.cpp:1275
    HostProfScope hpL2("numeric_subdomain: level 2");
    if ((int64_t)s.vB.n < s.pat.nnz) s.vB.alloc((size_t)s.pat.nnz);
    csr_scale_sym(s.n, s.pat.ptr.p, s.pat.idx.p, s.pat.val.p, s.d.p, s.vB.p, st);  // D A_dir D, src/geneo.cpp:1243-1246
    if (opt.lvl2 == 1) {
      eigen_local_problem(s, s.vNeu.p, s.vB.p, opt.tau, true, cut, ws, vals, vecs, counts);
    } else {
      double tl = opt.tau;  // getLocalGenEOTau, src/geneo.cpp:1097-1118
      if (!opt.cst) { tl = s.maxMult * opt.tau; if (tl >= 1.) tl = 0.9; s.tauLoc = tl; }
      eigen_local_problem(s, s.vNeu.p, s.vRob.p, tl, true, cut, ws, vals, vecs, counts);
      double gl = opt.gamma;
      if (!opt.cst) { gl = local_gamma(s); s.gammaLoc = gl; }
      eigen_local_problem(s, s.vB.p, s.vRob.p, gl, false, cut, ws, vals, vecs, counts);
    }
    assemble_z(s, vals, vecs, counts, st);
  }
  // level 1: factor A_dir (or A_rob), src/geneo.cpp:126-148
  const double tl1 = now_s();
  if (!s.L1) s.L1.reset(new LdltFactor(s.plan));  // a re-factorization overwrites the resident factor in place
  HostProfScope hp("lvl1 factorize");
  FactorStats fs = s.L1->factorize(opt.lvl1ORAS ? s.vRob.p : s.pat.val.p, pivTol, ws, st);
  allFactorSeconds += fs.seconds; allFactorFlops += s.plan->sym.flops; allFactorCount++;
  s.negL1 = fs.neg;
  s.perturbed += fs.perturbed;
  lvl1SetupMinvTime += now_s() - tl1;
  account_subdomain(s);
}

void GeneoPC::account_subdomain(const SubdomainState& s) {
  factorBytes += (int64_t)s.L1->L.bytes();
  factorNnz += s.plan->sym.lSize;
  factorFlops += s.plan->sym.flops;
  estimDimE += s.estim;
  realDimE += s.nev;
  nicolaides += s.nicolaides;
}

// Measurement hook (bench.py roofline_factorization): every level-1 matrix factorized once more -- same values, same result,
// written over the resident factors -- through the lanes of the pipelined setup, and NOTHING else on the device: the
// factorization kernels timed alone with CUDA events (start on lane 0 with every lane waiting for it, stop after every lane).
void GeneoPC::factor_bench(double* seconds, double* flops) {
  GENEO_CHECK(!subs.empty() && subs[0].L1, "factor_bench before setup");
  const int P = (int)subs.size();
  CUDA_CHECK(cudaDeviceSynchronize());
  double fl = 0.;
  for (auto& s : subs) fl += s.plan->sym.flops;
  cudaEvent_t e0, e1;
  CUDA_CHECK(cudaEventCreate(&e0));
  CUDA_CHECK(cudaEventCreate(&e1));
  float ms = 0.f;
  if (lanes.empty()) {  // sequential path
    CUDA_CHECK(cudaEventRecord(e0, st));
    for (auto& s : subs) s.L1->factorize(opt.lvl1ORAS ? s.vRob.p : s.pat.val.p, opt.pivRel * std::max(s.anorm, 1e-300), factorWs, st);
    CUDA_CHECK(cudaEventRecord(e1, st));
    CUDA_CHECK(cudaEventSynchronize(e1));
  } else {
    const int NL = (int)lanes.size();
    for (int j = 0; j < NL; j++)
      for (int p = j; p < P; p += NL) lanes[j]->ws.ensure(subs[p].plan->sym);
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaEventRecord(e0, lanes[0]->st));
    for (int j = 1; j < NL; j++) CUDA_CHECK(cudaStreamWaitEvent(lanes[j]->st, e0, 0));
    for (int g0 = 0; g0 < P; g0 += NL) {
      std::vector<FactorJob> jobs;
      for (int p = g0; p < std::min(P, g0 + NL); p++) {
        FactorJob J;
        J.F = subs[p].L1.get(); J.vals = opt.lvl1ORAS ? subs[p].vRob.p : subs[p].pat.val.p;
        J.pivTol = opt.pivRel * std::max(subs[p].anorm, 1e-300);
        J.ws = &lanes[p - g0]->ws; J.st = lanes[p - g0]->st;
        jobs.push_back(J);
      }
      factorize_enqueue(jobs);
    }
    std::vector<cudaEvent_t> done(NL, nullptr);
    for (int j = 1; j < NL; j++) {
      CUDA_CHECK(cudaEventCreateWithFlags(&done[j], cudaEventDisableTiming));
      CUDA_CHECK(cudaEventRecord(done[j], lanes[j]->st));
      CUDA_CHECK(cudaStreamWaitEvent(lanes[0]->st, done[j], 0));
    }
    CUDA_CHECK(cudaEventRecord(e1, lanes[0]->st));
    CUDA_CHECK(cudaEventSynchronize(e1));
    for (int j = 1; j < NL; j++) cudaEventDestroy(done[j]);
  }
  CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (seconds) *seconds = 1e-3 * ms;
  if (flops) *flops = fl;
}

// estimateNumberOfEigenValues (src/geneo.cpp:502-533) from the inertia of A - param B (Sylvester)
int GeneoPC::sylvester_estimate(SubdomainState& s, int neg, int perturbedS, bool tauPb, int cut) {
  // tau problem: #eigenvalues below tau = negative pivots; gamma problem: #above gamma = positive pivots (zero / perturbed
  // pivots are neither: the reference counts pcNbPosEV)
  int est = tauPb ? neg : (s.n - neg - perturbedS);
  est = std::max(0, std::min(est, s.n));
  if (cut > 0 && est > cut) est = cut;
  s.estim += est;
  s.perturbed += perturbedS;
  const int q = tauPb ? 0 : 1;
  s.sylNeg[q] = neg; s.sylNull[q] = perturbedS; s.sylEstim[q] = est;
  return est;
}

// eigenLocalProblem (src/geneo.cpp:842-963) + estimateNumberOfEigenValues (:502-533) + eigenLocalSolve (:626-722)
int GeneoPC::eigen_local_problem(SubdomainState& s, const double* vA, const double* vB, double param, bool tauPb, int cut,
                                 LdltWorkspace& ws, std::vector<double>& vals, std::vector<DevBuf<double>>& vecs,
                                 std::vector<int>& counts) {
  HostProfScope hpElp("eigen_local_problem");
  const int64_t nnz = s.pat.nnz;
  const double pivTol = opt.pivRel * std::max(s.anorm, 1e-300);
  int est = 0;
  LdltFactor tmp(s.plan);
  tmp.L = std::move(ws.spareL);  // cudaMalloc/cudaFree of a multi-GB factor per factorization costs more than the kernels
  if (!opt.noSyl) {
    const double t0 = now_s();
    if ((int64_t)s.vS.n < nnz) s.vS.alloc((size_t)nnz);
    vals_axpby(nnz, vA, param, vB, s.vS.p, st);  // A - param B, src/geneo.cpp:511-515
    HostProfScope hp("syl factorize");
    FactorStats fs = tmp.factorize(s.vS.p, pivTol, ws, st);
    allFactorSeconds += fs.seconds; allFactorFlops += s.plan->sym.flops; allFactorCount++;
    est = sylvester_estimate(s, fs.neg, fs.perturbed, tauPb, cut);
    const double dt = now_s() - t0;
    lvl2SetupSylTime += dt;
    (tauPb ? lvl2SetupTauSylTime : lvl2SetupGammaSylTime) += dt;
  }
  int got = 0;
  if (opt.noSyl || est > 0) {
    const double t0 = now_s();
    {  // shift-invert factor: A (tau problem: T = A^-1 B) or B (gamma problem: T = B^-1 A, self-adjoint in the A inner product)
      HostProfScope hp("eig factorize");
      FactorStats f2 = tmp.factorize(tauPb ? vA : vB, pivTol, ws, st);
      allFactorSeconds += f2.seconds; allFactorFlops += s.plan->sym.flops; allFactorCount++;
    }
    EigCtx cx;
    cx.st = st; cx.ws = &eigWs; cx.scal = scal.p;
    got = eigen_finish(s, tmp, vA, vB, param, tauPb, est, cut, vals, vecs, counts, cx);
    const double dt = now_s() - t0;
    lvl2SetupEigTime += dt;
    (tauPb ? lvl2SetupTauEigTime : lvl2SetupGammaEigTime) += dt;
  }
  ws.spareL = std::move(tmp.L);
  tmp.release();
  return got;
}

// Block Lanczos with the shift-invert factor `fac`, threshold filter (src/geneo.cpp:713-714), Nicolaides rule (:897-944).
int GeneoPC::eig_block(int est, int cut) const {
  int nev = est > 0 ? est : 1;
  if (cut > 0 && nev > cut) nev = cut;
  const int guard = (!opt.noSyl && (cut <= 0 || nev < cut)) ? 2 : 0;
  // Block of 8 by default.  -els2_eps_block 16 sends 16 right-hand sides per pass over the factor (k_solve_ring<16>),
  // but measured on 8 x 80^3 the wider block needs a 45-60 % larger Krylov space for the same pairs (13-16 steps of 16
  // against 18-19 steps of 8): 1.13 s against 0.93 s for the eight eigen-solves.
  // A pencil that wants many pairs (high-contrast heat: 100-250 per subdomain) is bound by the passes over the basis, one per
  // step whatever the block: there the block of 16 (fewer, fatter steps) wins.
  return opt.epsBlock > 0 ? opt.epsBlock : (nev + guard >= 64 ? 16 : 8);
}

int GeneoPC::eigen_finish(SubdomainState& s, const LdltFactor& fac, const double* vA, const double* vB, double param, bool tauPb,
                          int est, int cut, std::vector<double>& vals, std::vector<DevBuf<double>>& vecs, std::vector<int>& counts,
                          const EigCtx& cx) {
  cudaStream_t st = cx.st;  // (shadows the library's stream: everything below runs where the caller says)
  const int n = s.n;
  const int64_t nnz = s.pat.nnz;
  int nev = est > 0 ? est : 1;  // SLEPc default when nothing is requested
  if (cut > 0 && nev > cut) nev = cut;
  // Two guard pairs beyond the Sylvester estimate: the threshold filter below decides what is kept, so a pivot of
  // A - theta B whose sign is lost to rounding (no pivoting across pivot blocks) cannot drop a genuine GenEO vector.
  const int guard = (!opt.noSyl && (cut <= 0 || nev < cut)) ? 2 : 0;
  EigOptions eo;
  eo.block = eig_block(est, cut);
  eo.tol = opt.epsTol; eo.maxDim = opt.epsMaxDim; eo.invert = tauPb;
  eo.ws = cx.ws;
  if (cx.grp && cx.member >= 0) {  // this pencil's block solves ride on the group's forest solve
    GroupSolver* G = cx.grp;
    const int mi = cx.member;
    eo.xsExt = G->xs.p + (size_t)G->off[mi] * G->ld;
    eo.wExt = G->w.p + (size_t)G->off[mi] * G->ld;
    eo.solve = [G, mi](int j0, int nr, cudaStream_t ist) { return G->solve(mi, j0, nr, ist); };
    eo.leave = [G]() { G->leave(); };
  }
  {  // fail with a message, not with a 100 GB cudaMalloc: tau = 0.4 on a 100^3 subdomain asks for thousands of pairs
    const int want = std::min(nev + guard, n);
    const double maxDim = eo.maxDim > 0 ? eo.maxDim : std::max(4 * want + 8 * eo.block, 128);
    const double need = 8. * (double)n * (2. * std::min<double>(maxDim, n) + 2. * want) - (double)(cx.ws ? cx.ws->Q.cap + cx.ws->BQ.cap : 0);
    size_t freeB = 0, totB = 0;
    CUDA_CHECK(cudaMemGetInfo(&freeB, &totB));
    if (need > (double)freeB)
      throw Error("geneo_b200: the eigen-solve of subdomain " + std::to_string(s.id) + " wants " + std::to_string(want) + " pairs of a pencil of order " +
                  std::to_string(n) + ": its Lanczos basis and Ritz vectors need " + std::to_string((long long)(need / 1e9)) + " GB, " +
                  std::to_string((long long)(freeB / 1e9)) + " GB are free -- lower -geneo_tau or cap the count with -geneo_cut");
  }
  EigResult er;
  {
    HostProfScope hp("eig block_lanczos");
    block_lanczos(n, fac, s.pat.ptr.p, s.pat.idx.p, tauPb ? vB : vA, std::min(nev + guard, n), eo, er, st);
  }
  if (er.nconv < (int)er.lambda.size())
    fprintf(stderr, "WRNG: geneo_b200: eigen solve of subdomain %d converged %d/%d pairs (dim %d)\n", s.id, er.nconv,
            (int)er.lambda.size(), er.dim);
  s.eigSteps += er.steps;
  s.eigDim = std::max(s.eigDim, er.dim);
  // keep lambda <= tau (tau) / >= gamma (gamma): src/geneo.cpp:713-714.  Candidates are a prefix (sorted); like the
  // reference (which only walks EPSGetConverged pairs, :700-722) a pair whose residual did not reach the tolerance is not kept.
  std::vector<double> lam;
  std::vector<int> keepIdx;
  for (size_t i = 0; i < er.lambda.size(); i++) {
    const bool keep = tauPb ? (er.lambda[i] <= param) : (er.lambda[i] >= param);
    if (!keep) break;
    if (cut > 0 && (int)lam.size() >= cut) break;  // -geneo_cut caps what is kept (src/geneo.cpp:532, 871-879)
    const bool conv = er.nconv >= (int)er.lambda.size() || i >= er.resid.size() || er.resid[i] <= eo.tol;
    if (!conv) continue;
    lam.push_back(er.lambda[i]);
    keepIdx.push_back((int)i);
  }
  const int got = (int)lam.size();
  DevBuf<double> X;
  if (got > 0) {
    X.alloc((size_t)n * got);
    bool prefix = true;
    for (int q = 0; q < got; q++) prefix = prefix && keepIdx[q] == q;
    if (prefix) copy_cols(n, er.vecs.p, (int)er.lambda.size(), X.p, got, got, st);
    else for (int q = 0; q < got; q++) copy_cols(n, er.vecs.p + keepIdx[q], (int)er.lambda.size(), X.p + q, got, 1, st);
    CUDA_CHECK(::geneo::sync_stream(st));
  }
  // Nicolaides (src/geneo.cpp:897-944): add the constant vector when eigenvalues were kept, none is ~0 and 1 is in ker(A)
  bool addOne = false;
  if (tauPb && got > 0 && *std::min_element(lam.begin(), lam.end()) >= DBL_EPSILON) {
    double num = 0., den = 0.;
    csr_sum_all(nnz, vA, cx.scal, st);
    CUDA_CHECK(cudaMemcpyAsync(&num, cx.scal, sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(::geneo::sync_stream(st));
    csr_sum_all(nnz, vB, cx.scal, st);
    CUDA_CHECK(cudaMemcpyAsync(&den, cx.scal, sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(::geneo::sync_stream(st));
    if (std::fabs(num / den) <= (double)FLT_EPSILON) addOne = true;
  }
  s.nKept[tauPb ? 0 : 1] = got;
  if (got > 0) { vals.insert(vals.end(), lam.begin(), lam.end()); vecs.push_back(std::move(X)); counts.push_back(got); }
  if (addOne) {
    DevBuf<double> one((size_t)n);
    vec_set(n, 1., one.p, st);
    CUDA_CHECK(::geneo::sync_stream(st));
    vals.push_back(0.);
    vecs.push_back(std::move(one));
    counts.push_back(1);
    s.nicolaides += 1;
  }
  return got;
}

// =====================================================================================================================
// Pipelined numeric setup (one level-2 pencil or none): the three factorizations of every subdomain -- S = A_neu - tau B
// (inertia), A_neu (shift-invert factor of the eigen-solve), A_dir / A_rob (the resident level-1 factor) -- are enqueued by a
// helper thread on a few LANES (stream + update arenas + transient factor), level by level round-robin over the lanes, so
// that independent factorizations overlap on the device; this thread runs the host-driven block Lanczos of subdomain p on
// the library's stream as soon as p's shift-invert factor is there -- the latency-bound eigen-solve hides behind the
// DMMA tiles of the other lanes.  Dependencies: CUDA events between streams, two host flags per subdomain between the threads.
// =====================================================================================================================
void GeneoPC::numeric_pipeline() {
  const double tCold0 = now_s();
  static const bool coldTiming = getenv("GENEO_COLD_TIMING") != nullptr;
  const int P = (int)subs.size();
  const bool l2 = opt.lvl2 >= 1, syl = l2 && !opt.noSyl;
  // ---- lanes: as many as fit next to the resident factors (each lane = update arenas + one transient factor) -------------
  int64_t maxL = 0, maxArena = 0, sumL = 0;
  for (auto& s : subs) {
    const Symbolic& S = s.plan->sym;
    maxL = std::max(maxL, S.lSize);
    maxArena = std::max(maxArena, 2 * S.uArena + S.cArena + 2 * S.wArena);
    if (!s.L1 || (int64_t)s.L1->L.n < S.lSize) sumL += S.lSize;
  }
  // How many lanes?  Each costs its update arenas + a transient factor (17.8 GB at 100^3); what the eigen-solves and the
  // coarse vectors will need next to them (Lanczos bases 2 n maxDim, Z_i = n nev_i) depends on the eigen-counts, which a FIRST
  // setup does not know (a heat subdomain wants 200+ pairs, a Laplacian one 10): two lanes then, which already give most of
  // the overlap (8 factorizations: 2.06 s on one lane, 1.87 s on two, 1.82 s on four); a re-setup sizes the reserve from
  // the eigen-counts of the previous one and takes up to four.
  int prevMaxNev = 0;
  double zGrowth = 0.;
  for (auto& s : subs) {
    prevMaxNev = std::max(prevMaxNev, s.prevNev);
    zGrowth += std::max(0., 8. * (double)s.n * std::max(s.prevNev, 1) - (double)s.Z.cap);
  }
  const bool history = l2 && prevMaxNev > 0;
  int want = std::min(P, (history || !l2) ? 4 : 2);
  {
    size_t freeB = 0, totB = 0;
    CUDA_CHECK(cudaMemGetInfo(&freeB, &totB));
    int64_t have = 0;  // what the existing lanes already hold
    double eigHave = 0.;
    for (auto& L : lanes) {
      have += (int64_t)(L->T.cap + L->ws.u0.cap + L->ws.u1.cap + L->ws.uc.cap + L->ws.w0.cap + L->ws.w1.cap);
      eigHave += (double)(L->eig.Q.cap + L->eig.BQ.cap);
    }
    eigHave += (double)(eigWs.Q.cap + eigWs.BQ.cap);
    const double perLane = 8. * ((l2 ? (double)maxL : 0.) + (double)maxArena);
    int64_t nmax = 0;
    for (auto& s : subs) nmax = std::max<int64_t>(nmax, s.n);
    auto eig_need = [&](int lanesNow) {  // one Lanczos workspace per lane (lock-step group) or one shared one, + Ritz vectors
      const int b = eig_block(prevMaxNev, opt.cut);
      const double maxDim = opt.epsMaxDim > 0 ? opt.epsMaxDim : std::max(4 * (prevMaxNev + 2) + 8 * b, 128);
      const double one = 8. * (double)nmax * (2. * maxDim + 8. * b + 2. * (prevMaxNev + 2));
      return one * lanesNow;
    };
    while (want > 1) {
      const double reserve = history ? std::max(0., eig_need(want) - eigHave) + zGrowth + 0.05 * (double)totB
                                     : std::max(6e9, 0.15 * (double)totB);
      // resident factors still to come, the reserve, the lanes
      if (perLane * want <= (double)freeB + (double)have - 8. * (double)sumL - reserve) break;
      want--;
    }
  }
  while ((int)lanes.size() > want) lanes.pop_back();
  while ((int)lanes.size() < want) {
    lanes.emplace_back(new Lane());
    CUDA_CHECK(cudaStreamCreateWithFlags(&lanes.back()->st, cudaStreamNonBlocking));
    CUDA_CHECK(cudaStreamCreateWithFlags(&lanes.back()->est, cudaStreamNonBlocking));
    CUDA_CHECK(cudaHostAlloc((void**)&lanes.back()->hc, 6 * sizeof(int), cudaHostAllocDefault));
    lanes.back()->scal.alloc(16);
  }
  const int NL = (int)lanes.size();
  // every allocation of the concurrent region happens here, before it starts (the block cache is stream-ordered on ONE stream)
  for (auto& s : subs) {
    if (!s.L1) s.L1.reset(new LdltFactor(s.plan));
    if ((int64_t)s.L1->L.n < s.plan->sym.lSize) s.L1->L.alloc((size_t)s.plan->sym.lSize);
    if (l2 && (int64_t)s.vB.n < s.pat.nnz) s.vB.alloc((size_t)s.pat.nnz);
    if (syl && (int64_t)s.vS.n < s.pat.nnz) s.vS.alloc((size_t)s.pat.nnz);
  }
  for (int j = 0; j < NL; j++) {
    for (int p = j; p < P; p += NL) lanes[j]->ws.ensure(subs[p].plan->sym);
    if (l2 && (int64_t)lanes[j]->T.n < maxL) lanes[j]->T.alloc((size_t)maxL);
  }
  CUDA_CHECK(cudaDeviceSynchronize());
  const double tCold1 = now_s();

  std::vector<cudaEvent_t> evS(P, nullptr), evN(P, nullptr), evD(P, nullptr);
  for (int p = 0; p < P; p++) {
    CUDA_CHECK(cudaEventCreateWithFlags(&evS[p], cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&evN[p], cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&evD[p], cudaEventDisableTiming));
  }
  struct EvGuard { std::vector<cudaEvent_t>*a, *b, *c; ~EvGuard() { for (auto* v : {a, b, c}) for (auto e : *v) if (e) cudaEventDestroy(e); } } evGuard{&evS, &evN, &evD};
  std::vector<std::unique_ptr<LdltFactor>> tmpF(P);
  // pinned landing zone of the level-1 counters (a device -> pageable copy would block the enqueueing thread)
  struct PinnedInts { int* p = nullptr; ~PinnedInts() { if (p) cudaFreeHost(p); } } hcDpin;
  CUDA_CHECK(cudaHostAlloc((void**)&hcDpin.p, 2 * (size_t)P * sizeof(int), cudaHostAllocDefault));
  int* hcD = hcDpin.p;
  std::fill(hcD, hcD + 2 * (size_t)P, 0);
  std::mutex mtx;
  std::condition_variable cv;
  std::vector<char> enqueued(P, 0), eigDone(P, 0);  // helper -> main: S and A_neu of p are enqueued; main -> helper: p's lane is free
  std::string helperErr;
  bool abortAll = false;
  int dev = 0;
  CUDA_CHECK(cudaGetDevice(&dev));
  const double tPipe0 = now_s();

  std::thread helper([&]() {
    try {
      CUDA_CHECK(cudaSetDevice(dev));
      for (int g0 = 0; g0 < P; g0 += NL) {
        const int g1 = std::min(P, g0 + NL);
        std::vector<FactorJob> jobs;
        if (l2) {
          for (int p = g0; p < g1; p++) {  // the lane's previous tenant must be through with its eigen-solve
            if (p - NL >= 0) {
              std::unique_lock<std::mutex> lk(mtx);
              cv.wait(lk, [&]() { return eigDone[p - NL] != 0 || abortAll; });
              if (abortAll) return;
            }
            Lane& L = *lanes[p - g0];
            SubdomainState& s = subs[p];
            tmpF[p].reset(new LdltFactor(s.plan));
            tmpF[p]->L = std::move(L.T);
            csr_scale_sym(s.n, s.pat.ptr.p, s.pat.idx.p, s.pat.val.p, s.d.p, s.vB.p, L.st);  // B = D A_dir D, src/geneo.cpp:1243-1246
            if (syl) vals_axpby(s.pat.nnz, s.vNeu.p, opt.tau, s.vB.p, s.vS.p, L.st);          // S = A_neu - tau B, :511-515
          }
          if (syl) {
            jobs.clear();
            for (int p = g0; p < g1; p++) {
              Lane& L = *lanes[p - g0];
              FactorJob J;
              J.F = tmpF[p].get(); J.vals = subs[p].vS.p; J.pivTol = opt.pivRel * std::max(subs[p].anorm, 1e-300);
              J.ws = &L.ws; J.st = L.st; J.hostCounters = L.hc;
              jobs.push_back(J);
            }
            factorize_enqueue(jobs);
            for (int p = g0; p < g1; p++) CUDA_CHECK(cudaEventRecord(evS[p], lanes[p - g0]->st));
          }
          jobs.clear();
          for (int p = g0; p < g1; p++) {
            Lane& L = *lanes[p - g0];
            FactorJob J;
            J.F = tmpF[p].get(); J.vals = subs[p].vNeu.p; J.pivTol = opt.pivRel * std::max(subs[p].anorm, 1e-300);
            J.ws = &L.ws; J.st = L.st; J.hostCounters = L.hc + 2;
            jobs.push_back(J);
          }
          factorize_enqueue(jobs);
          for (int p = g0; p < g1; p++) CUDA_CHECK(cudaEventRecord(evN[p], lanes[p - g0]->st));
          { std::lock_guard<std::mutex> lk(mtx); for (int p = g0; p < g1; p++) enqueued[p] = 1; }
          cv.notify_all();
        }
        jobs.clear();
        for (int p = g0; p < g1; p++) {
          Lane& L = *lanes[p - g0];
          FactorJob J;
          J.F = subs[p].L1.get(); J.vals = opt.lvl1ORAS ? subs[p].vRob.p : subs[p].pat.val.p;
          J.pivTol = opt.pivRel * std::max(subs[p].anorm, 1e-300);
          J.ws = &L.ws; J.st = L.st; J.hostCounters = nullptr;  // (copied to hcD[p] below: the lane's next tenant reuses L.hc)
          jobs.push_back(J);
        }
        factorize_enqueue(jobs);
        for (int p = g0; p < g1; p++) {
          Lane& L = *lanes[p - g0];
          CUDA_CHECK(cudaMemcpyAsync(&hcD[2 * (size_t)p], L.ws.counters.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, L.st));
          CUDA_CHECK(cudaEventRecord(evD[p], L.st));
        }
      }
    } catch (std::exception& e) {
      std::lock_guard<std::mutex> lk(mtx);
      helperErr = e.what();
      abortAll = true;
    }
    cv.notify_all();
  });
  struct Joiner { std::thread& t; std::mutex& m; std::condition_variable& c; bool& ab; ~Joiner() { { std::lock_guard<std::mutex> lk(m); ab = true; } c.notify_all(); if (t.joinable()) t.join(); } } joiner{helper, mtx, cv, abortAll};

  // ---- the eigen-solves, one lane group at a time: the pencils of a group run in LOCK-STEP (one host thread each, one
  //      forest solve per step over the group's shift-invert factors) while the helper keeps the lanes busy with the
  //      level-1 factorizations of this group and the S / A_neu factorizations of the next one
  if ((int)groupSolvers.size() < (P + NL - 1) / NL) groupSolvers.resize((P + NL - 1) / NL);
  bool mainAbort = false;
  for (int g0 = 0; l2 && g0 < P && !mainAbort; g0 += NL) {
    const int g1 = std::min(P, g0 + NL);
    std::vector<int> est(g1 - g0, 0);
    for (int p = g0; p < g1; p++) {
      {
        std::unique_lock<std::mutex> lk(mtx);
        cv.wait(lk, [&]() { return enqueued[p] != 0 || abortAll; });
        if (abortAll && !enqueued[p]) { mainAbort = true; break; }
      }
      if (syl) {
        const double t0 = now_s();
        CUDA_CHECK(cudaEventSynchronize(evS[p]));
        est[p - g0] = sylvester_estimate(subs[p], lanes[p - g0]->hc[0], lanes[p - g0]->hc[1], true, opt.cut);
        lvl2SetupSylTime += now_s() - t0; lvl2SetupTauSylTime += now_s() - t0;
      }
    }
    if (mainAbort) break;
    const double t0 = now_s();
    for (int p = g0; p < g1; p++) CUDA_CHECK(cudaEventSynchronize(evN[p]));
    std::vector<int> act;  // members with an eigen-solve to do
    for (int p = g0; p < g1; p++)
      if (opt.noSyl || est[p - g0] > 0) act.push_back(p);
    // Do the Lanczos buffers of all members fit at once?  (basis + its B image: 2 n maxDim doubles per pencil -- 20 GB for a
    // heat subdomain that wants 200 pairs.)  If not, the pencils run one after the other on the library's stream, as in
    // the sequential path, and share one workspace.
    bool threaded = act.size() >= 2 && !g_hostprof;
    if (threaded) {
      double need = 0.;
      for (int p : act) {
        const int b = eig_block(est[p - g0], opt.cut);
        const int nev = std::max(1, est[p - g0]) + 2;
        const double maxDim = opt.epsMaxDim > 0 ? opt.epsMaxDim : std::max(4 * nev + 8 * b, 128);
        need += 8. * subs[p].n * (2. * maxDim + 8. * b) - (double)(lanes[p - g0]->eig.Q.cap + lanes[p - g0]->eig.BQ.cap);
      }
      size_t freeB = 0, totB = 0;
      CUDA_CHECK(cudaMemGetInfo(&freeB, &totB));
      if (need > (double)freeB - 3e9) threaded = false;
    }
    // group solver: same Lanczos block for everybody, at least two pencils
    GroupSolver* grp = nullptr;
    bool uniform = threaded;
    for (size_t a = 1; a < act.size() && uniform; a++)
      uniform = eig_block(est[act[a] - g0], opt.cut) == eig_block(est[act[0] - g0], opt.cut) && subs[act[a]].n > 64;
    if (uniform && subs[act[0]].n > 64) {
      std::unique_ptr<GroupSolver>& slot = groupSolvers[g0 / NL];
      std::vector<const LdltPlan*> plans;
      for (int p : act) plans.push_back(subs[p].plan.get());
      const int ld = (eig_block(est[act[0] - g0], opt.cut) + 7) / 8 * 8;
      if (!slot || slot->plans != plans) {
        slot.reset(new GroupSolver());
        slot->plans = plans;
        int64_t o = 0;
        for (int p : act) { slot->off.push_back(o); o += subs[p].n; }
        slot->forest.build(plans, slot->off);
        CUDA_CHECK(cudaStreamCreateWithFlags(&slot->st, cudaStreamNonBlocking));
        slot->evIn.assign(act.size(), nullptr);
        for (auto& e : slot->evIn) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : slot->evOut) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      }
      grp = slot.get();
      const size_t rows = (size_t)(grp->off.back() + subs[act.back()].n);
      if (grp->xs.n < rows * ld) { grp->xs.alloc(rows * ld); grp->w.alloc(rows * ld); }
      grp->ld = ld;
      grp->members = (int)act.size();
      grp->arrived = 0;
      grp->gen = grp->refused = 0;
      grp->on = true;
      std::vector<const double*> Ls;
      for (int p : act) Ls.push_back(tmpF[p]->L.p);
      grp->forest.set_factors(Ls, grp->st);
    }    std::vector<std::vector<double>> gvals(g1 - g0);
    std::vector<std::vector<DevBuf<double>>> gvecs(g1 - g0);
    std::vector<std::vector<int>> gcounts(g1 - g0);
    std::vector<std::string> gerr(g1 - g0);
    std::vector<std::thread> eth;
    for (size_t a = 0; a < act.size(); a++) {
      const int p = act[a];
      auto work = [&, a, p]() {
        try {
          CUDA_CHECK(cudaSetDevice(dev));
          Lane& L = *lanes[p - g0];
          EigCtx cx;
          if (threaded) { cx.st = L.est; cx.ws = &L.eig; cx.scal = L.scal.p; cx.grp = grp; cx.member = grp ? (int)a : -1; }
          else { cx.st = st; cx.ws = &eigWs; cx.scal = scal.p; }
          eigen_finish(subs[p], *tmpF[p], subs[p].vNeu.p, subs[p].vB.p, opt.tau, true, est[p - g0], opt.cut, gvals[p - g0], gvecs[p - g0],
                       gcounts[p - g0], cx);
          assemble_z(subs[p], gvals[p - g0], gvecs[p - g0], gcounts[p - g0], cx.st);
          CUDA_CHECK(cudaStreamSynchronize(cx.st));
        } catch (std::exception& e) {
          gerr[p - g0] = e.what();
          if (grp) grp->leave();
        }
      };
      if (threaded) eth.emplace_back(work);
      else work();
    }
    for (auto& t : eth) t.join();
    for (auto& e : gerr) if (!e.empty()) throw Error(e);
    for (int p = g0; p < g1; p++)
      if (std::find(act.begin(), act.end(), p) == act.end()) assemble_z(subs[p], gvals[p - g0], gvecs[p - g0], gcounts[p - g0], st);  // constant vector
    if (grp) CUDA_CHECK(cudaStreamSynchronize(grp->st));
    if (getenv("GENEO_DEBUG_GROUP"))
      fprintf(stderr, "DEBUG group %d: %d pencils, threaded %d, group solver %d, combined solves %ld, solo after dissolve %ld, %.3f s\n", g0 / NL,
              (int)act.size(), (int)threaded, grp ? 1 : 0, grp ? grp->gen : 0, grp ? grp->refused : 0, now_s() - t0);
    lvl2SetupEigTime += now_s() - t0; lvl2SetupTauEigTime += now_s() - t0;
    {
      std::lock_guard<std::mutex> lk(mtx);
      for (int p = g0; p < g1; p++) {
        lanes[p - g0]->T = std::move(tmpF[p]->L);
        subs[p].plan->selfL = nullptr;  // the plan's single-factor forest must re-read the factor pointer next time
        eigDone[p] = 1;
      }
    }
    cv.notify_all();
  }
  { std::lock_guard<std::mutex> lk(mtx); if (!helperErr.empty()) abortAll = true; }
  helper.join();
  if (!helperErr.empty()) throw Error(helperErr);
  const double tl1 = now_s();
  for (int p = 0; p < P; p++) {
    CUDA_CHECK(cudaEventSynchronize(evD[p]));
    subs[p].negL1 = hcD[2 * (size_t)p];
    subs[p].perturbed += hcD[2 * (size_t)p + 1];
  }
  for (auto& L : lanes) CUDA_CHECK(cudaStreamSynchronize(L->st));
  lvl1SetupMinvTime += now_s() - tl1;
  for (int p = 0; p < P; p++) {
    account_subdomain(subs[p]);
    allFactorFlops += subs[p].plan->sym.flops * (1 + (l2 ? 1 : 0) + (syl ? 1 : 0));
    allFactorCount += 1 + (l2 ? 1 : 0) + (syl ? 1 : 0);
  }
  allFactorSeconds += now_s() - tPipe0;  // span of the factorization pipeline (the eigen-solves run inside it)
  if (coldTiming)
    fprintf(stderr, "COLD rank %d: pipeline allocations (lanes %d, resident factors, value buffers) %.3f s, pipeline %.3f s\n", comm.rank, NL,
            tCold1 - tCold0, now_s() - tCold1);
}

// Z offsets (all_gather of nev_i, src/geneo.cpp:363-375), E = Z^T A Z (MatPtAP :1033), E^-1 (dcs2_, :1059-1065)
void GeneoPC::build_coarse() {
  const int P = (int)subs.size();
  // all_gather of nev_i (src/geneo.cpp:363) -> global column offsets of Z
  std::vector<double> tmp(2 * (size_t)nbPart, 0.);
  for (auto& s : subs) { tmp[s.id] = s.nev; tmp[nbPart + s.id] = s.estim; }
  comm.allreduce_sum_host(tmp.data(), 2 * nbPart, st);
  nevGlobal.assign(nbPart, 0);
  estimGlobal.assign(nbPart, 0);
  std::vector<int> zoffGlobal(nbPart + 1, 0), localOf(nbPart, -1);
  for (int q = 0; q < nbPart; q++) {
    nevGlobal[q] = (int)std::lround(tmp[q]);
    estimGlobal[q] = (int)std::lround(tmp[nbPart + q]);
    zoffGlobal[q + 1] = zoffGlobal[q] + nevGlobal[q];
  }
  nE = zoffGlobal[nbPart];
  for (int p = 0; p < P; p++) { subs[p].zoff = zoffGlobal[subs[p].id]; localOf[subs[p].id] = p; }
  const int nEp = (nE + 7) / 8 * 8;
  DevBuf<double> dE((size_t)nE * nE);
  dE.zero(st);
  DevBuf<double> G((size_t)nLoc * 8), Wg((size_t)nLoc * 8);
  int nmax = 0;
  for (auto& s : subs) nmax = std::max(nmax, s.n);
  DevBuf<double> Gi((size_t)std::max(1, nmax) * 8);
  for (int j = 0; j < nbPart; j++) {  // every rank walks the GLOBAL list of subdomains in lockstep (halo exchanges are collective)
    const int jl = localOf[j];
    for (int c0 = 0; c0 < nevGlobal[j]; c0 += 8) {
      const int nc = std::min(8, nevGlobal[j] - c0);
      G.zero(st);
      if (jl >= 0) scatter_rows8(subs[jl].n, subs[jl].gidx.p, subs[jl].Z.p, subs[jl].nev, c0, nc, G.p, st);
      if (comm.active()) {  // R_j^T Z_j lives on the owner rows: ghost parts go to their owners, then to every copy
        comm.halo_reverse_add(G.p, 8, st);
        comm.halo_forward(G.p, 8, st);
      }
      sell_spmm8(A, G.p, Wg.p, st);
      comm.halo_forward(Wg.p, 8, st);
      for (int i = 0; i < P; i++) {
        SubdomainState& si = subs[i];
        gather_rows8(si.n, si.gidx.p, Wg.p, Gi.p, st);
        // E[zoff_i + a, zoff_j + c0 + c] += sum_k Z_i[k,a] * Gi[k,c]
        ts_gram(si.n, si.Z.p, si.nev, si.nev, Gi.p, 8, nc, dE.p + (size_t)si.zoff * nE + zoffGlobal[j] + c0, nE, st);
      }
    }
  }
  comm.allreduce_sum(dE.p, nE * nE, st);  // every block row was computed by exactly one rank
  std::vector<double> hE = dE.to_host(st);
  for (int i = 0; i < nE; i++)
    for (int j = i + 1; j < nE; j++) hE[(size_t)i * nE + j] = hE[(size_t)j * nE + i] = 0.5 * (hE[(size_t)i * nE + j] + hE[(size_t)j * nE + i]);
  // dense block LDL^T of E with the same device kernels (one chain of panels), then E^-1 by solving for the identity
  CsrHost pe;
  pe.n = pe.ncols = nE;
  pe.ptr.resize(nE + 1);
  pe.idx.resize((size_t)nE * nE);
  for (int i = 0; i <= nE; i++) pe.ptr[i] = (int64_t)i * nE;
  for (int i = 0; i < nE; i++) for (int j = 0; j < nE; j++) pe.idx[(size_t)i * nE + j] = j;
  SymbolicOptions so;
  so.nb = opt.nb; so.ordering = 0; so.amalgamate = false;
  auto plan = std::make_shared<LdltPlan>(nE, pe.ptr.data(), pe.idx.data(), so);
  LdltFactor LE(plan);
  LdltWorkspace ws;
  // Symmetric equilibration E' = S E S, S = diag(E_ii)^-1/2 (MUMPS scales by default too): with a 10^6 coefficient contrast
  // the diagonal of E spans 12 orders of magnitude (tiny GenEO eigenvalues next to Nicolaides vectors of stiff
  // subdomains) and the null-pivot test, relative to max |E_ii|, would throw genuine coarse modes away.
  std::vector<double> sc(nE, 1.);
  for (int i = 0; i < nE; i++) {
    const double dii = hE[(size_t)i * nE + i];
    sc[i] = dii > 0. ? 1. / std::sqrt(dii) : 1.;
  }
  for (int i = 0; i < nE; i++)
    for (int j = 0; j < nE; j++) hE[(size_t)i * nE + j] *= sc[i] * sc[j];
  dE.upload(hE, st);
  FactorStats fs = LE.factorize(dE.p, opt.pivRel, ws, st);  // (unit diagonal after scaling)
  if (fs.neg > 0 || fs.perturbed > 0)
    fprintf(stderr, "WRNG: geneo_b200: coarse operator E is not positive definite (neg %d, null pivots %d)\n", fs.neg, fs.perturbed);
  // E^-1 = S E'^-1 S: solve for the columns of S, then scale the rows
  std::vector<double> hI((size_t)nE * nEp, 0.);
  for (int i = 0; i < nE; i++) hI[(size_t)i * nEp + i] = sc[i];
  DevBuf<double> dI, dS;
  dI.upload(hI, st);
  dS.upload(sc, st);
  Einv.alloc((size_t)nE * nEp);
  Einv.zero(st);
  for (int j0 = 0; j0 < nEp; j0 += 8) LE.solve_permuted(dI.p, Einv.p, nEp, j0, 8, st);
  if (nE > 0) rows_scale(nE, nEp, dS.p, Einv.p, st);
  w.alloc(nEp); w2.alloc(nEp);
  CUDA_CHECK(::geneo::sync_stream(st));
}

// =====================================================================================================================
// Apply
// =====================================================================================================================
void GeneoPC::applyQ(const double* x, double* y) {  // src/geneo.cpp:1435-1517
  const int P = (int)subs.size();
  comm.halo_forward(const_cast<double*>(x), 1, st);
  gather_rows(nAll, gidxAll.p, nullptr, x, Xall.p, st);
  w.zero(st);
  for (int p = 0; p < P; p++) zt_x(subs[p].n, subs[p].nev, subs[p].Z.p, subs[p].nev, Xall.p + subs[p].off, w.p + subs[p].zoff, st);
  comm.allreduce_sum(w.p, nE, st);  // coarse gather: every rank gets the whole Z^T x (E^-1 is replicated)
  dense_gemv(nE, nE, Einv.p, (nE + 7) / 8 * 8, w.p, w2.p, st);
  Yall.zero(st);
  for (int p = 0; p < P; p++) z_w_add(subs[p].n, subs[p].nev, subs[p].Z.p, subs[p].nev, w2.p + subs[p].zoff, nullptr, Yall.p + subs[p].off, st);
  pull_sum(nLoc, pullPtr.p, pullPos.p, Yall.p, y, false, st);
  comm.halo_reverse_add(y, 1, st);
}

// restrict, [D], M^-1, [D], (+ Z E^-1 Z^T fused when addQ), prolong-add.  src/geneo.cpp:1980-2025, 1845-1900.
void GeneoPC::level1(const double* xin, double* yout, bool addQ) {
  const int P = (int)subs.size();
  double tt = 0.;
  auto tic = [&]() { if (opt.timing) { CUDA_CHECK(::geneo::sync_stream(st)); tt = now_s(); } };
  auto toc = [&](double& acc) { if (opt.timing) { CUDA_CHECK(::geneo::sync_stream(st)); acc += now_s() - tt; } };
  tic();
  comm.halo_forward(const_cast<double*>(xin), 1, st);
  gather_rows(nAll, gidxAll.p, nullptr, xin, Xall.p, st);
  toc(lvl1ApplyScatterTime);
  if (addQ) {
    tic();
    w.zero(st);
    for (int p = 0; p < P; p++) zt_x(subs[p].n, subs[p].nev, subs[p].Z.p, subs[p].nev, Xall.p + subs[p].off, w.p + subs[p].zoff, st);
    comm.allreduce_sum(w.p, nE, st);
    toc(lvl2ApplyZtTime);
    tic();
    dense_gemv(nE, nE, Einv.p, (nE + 7) / 8 * 8, w.p, w2.p, st);
    toc(lvl2ApplyEinvTime);
  }
  tic();
  if (opt.lvl1RAS) vec_pointwise(nAll, dAll.p, Xall.p, st);  // D before the solve, src/geneo.cpp:1991-1993
  if (opt.kernelTiming) {
    while (ktEvents.size() < ktUsed + 2) { cudaEvent_t e; CUDA_CHECK(cudaEventCreate(&e)); ktEvents.push_back(e); }
    CUDA_CHECK(cudaEventRecord(ktEvents[ktUsed], st));
  }
  forest.solve(Xall.p, Yall.p, 1, 0, 1, st);  // every local subdomain in ONE persistent cooperative kernel
  if (opt.kernelTiming) { CUDA_CHECK(cudaEventRecord(ktEvents[ktUsed + 1], st)); ktUsed += 2; }
  toc(lvl1ApplyMinvTime);
  if (addQ || opt.lvl1SRAS) {
    tic();
    for (int p = 0; p < P; p++)
      z_w_add(subs[p].n, addQ ? subs[p].nev : 0, subs[p].Z.p, subs[p].nev, addQ ? w2.p + subs[p].zoff : nullptr,
              opt.lvl1SRAS ? subs[p].d.p : nullptr, Yall.p + subs[p].off, st);
    toc(addQ ? lvl2ApplyZTime : lvl1ApplyMinvTime);
  }
  tic();
  pull_sum(nLoc, pullPtr.p, pullPos.p, Yall.p, yout, false, st);
  comm.halo_reverse_add(yout, 1, st);
  toc(lvl1ApplyGatherTime);
}

void GeneoPC::apply(const double* x, double* y) {  // applyGenEOPC, src/geneo.cpp:2051-2098
  applyCount++;
  double t0 = 0.;
  if (opt.timing) { CUDA_CHECK(::geneo::sync_stream(st)); t0 = now_s(); }
  if (opt.lvl2 == 0) level1(x, y, false);
  else if (!opt.hybrid) level1(x, y, true);                         // y = Q x + sum R^T [D] M^-1 [D] R x
  else if (!opt.effHybrid) {
    applyQ(x, t1.p);                                                // t1 = Q x
    mult_sub(t1.p, x, t2.p);                                        // t2 = x - A Q x = (I - P^T) x
    level1(t2.p, t3.p, false);
    mult(t3.p, t2.p);
    applyQ(t2.p, y);                                                // y = Q A t3
    vec_axpby(nLoc, 1., t3.p, -1., y, st);                          // y = (I - P) t3
    vec_axpy(nLoc, 1., t1.p, y, st);                                // y += Q x
  } else {
    level1(x, t3.p, false);
    mult(t3.p, t2.p);
    applyQ(t2.p, y);
    vec_axpby(nLoc, 1., t3.p, -1., y, st);
  }
  if (opt.timing) { CUDA_CHECK(::geneo::sync_stream(st)); lvl1ApplyTime += now_s() - t0; }
}

void GeneoPC::initial_guess(const double* b, double* x0) {
  if (opt.lvl2 >= 1 && opt.effHybrid) applyQ(b, x0);
  else CUDA_CHECK(cudaMemsetAsync(x0, 0, sizeof(double) * nLoc, st));
}

void GeneoPC::copy_einv(double* out) const {
  const int nEp = (nE + 7) / 8 * 8;
  std::vector<double> h = Einv.to_host(st);
  for (int i = 0; i < nE; i++)
    for (int j = 0; j < nE; j++) out[(size_t)i * nE + j] = h[(size_t)i * nEp + j];
}

// =====================================================================================================================
// Block apply: the steps of applyQ / level1 / apply on row-major nLoc x 8 blocks, 8 columns per pass over the factors
// =====================================================================================================================
void GeneoPC::ensure_block() {
  const size_t nb = (size_t)nLoc * 8, na = (size_t)nAll * 8, nw = (size_t)(nE + 7) / 8 * 8 * 8;
  if (bIn.n != nb) { bIn.alloc(nb); bOut.alloc(nb); bT1.alloc(nb); bT2.alloc(nb); }
  if (bXall.n != na) { bXall.alloc(na); bYall.alloc(na); }
  if (bW.n != std::max<size_t>(nw, 8)) { bW.alloc(std::max<size_t>(nw, 8)); bW2.alloc(std::max<size_t>(nw, 8)); }
}

void GeneoPC::coarse8() {
  const int nEp = (nE + 7) / 8 * 8;
  bW.zero(st);
  for (auto& s : subs) ts_gram(s.n, s.Z.p, s.nev, s.nev, bXall.p + (size_t)s.off * 8, 8, 8, bW.p + (size_t)s.zoff * 8, 8, st);
  comm.allreduce_sum(bW.p, nE * 8, st);
  ts_update(nE, Einv.p, nEp, nE, bW.p, 8, 8, bW2.p, 8, 1., 0., st);
}

void GeneoPC::applyQ8(double* x, double* y) {
  comm.halo_forward(x, 8, st);
  gather_rows8((int)nAll, gidxAll.p, x, bXall.p, st);
  coarse8();
  for (auto& s : subs)  // (beta 0: a subdomain without coarse vectors gets zero rows)
    ts_update(s.n, s.Z.p, s.nev, s.nev, bW2.p + (size_t)s.zoff * 8, 8, 8, bYall.p + (size_t)s.off * 8, 8, 1., 0., st);
  pull_sum8(nLoc, pullPtr.p, pullPos.p, bYall.p, y, st);
  comm.halo_reverse_add(y, 8, st);
}

void GeneoPC::level1_8(double* x, double* y, bool addQ) {
  comm.halo_forward(x, 8, st);
  gather_rows8((int)nAll, gidxAll.p, x, bXall.p, st);
  if (addQ) coarse8();
  if (opt.lvl1RAS) rows_scale((int)nAll, 8, dAll.p, bXall.p, st);
  forest.solve(bXall.p, bYall.p, 8, 0, 8, st);  // every local subdomain, 8 columns, in one launch of the 8-column kernel
  for (auto& s : subs) {
    double* ys = bYall.p + (size_t)s.off * 8;
    if (opt.lvl1SRAS) rows_scale(s.n, 8, s.d.p, ys, st);
    if (addQ && s.nev > 0) ts_update(s.n, s.Z.p, s.nev, s.nev, bW2.p + (size_t)s.zoff * 8, 8, 8, ys, 8, 1., 1., st);
  }
  pull_sum8(nLoc, pullPtr.p, pullPos.p, bYall.p, y, st);
  comm.halo_reverse_add(y, 8, st);
}

void GeneoPC::mult8(double* x, double* y) {
  comm.halo_forward(x, 8, st);
  sell_spmm8(A, x, y, st);
}
void GeneoPC::mult_sub8(double* x, const double* b, double* y) {
  mult8(x, y);
  vec_axpby(A.n * 8, 1., b, -1., y, st);
}

void GeneoPC::apply8(double* x, double* y) {
  const int n8 = nLoc * 8;
  if (opt.lvl2 == 0) level1_8(x, y, false);
  else if (!opt.hybrid) level1_8(x, y, true);
  else if (!opt.effHybrid) {
    applyQ8(x, bT1.p);                  // t1 = Q x
    mult_sub8(bT1.p, x, bT2.p);         // t2 = x - A Q x
    level1_8(bT2.p, y, false);          // y = t3
    mult8(y, bT2.p);
    applyQ8(bT2.p, bT2.p);              // t2 = Q A t3
    vec_axpby(n8, -1., bT2.p, 1., y, st);  // y = (I - P) t3
    vec_axpy(n8, 1., bT1.p, y, st);        // y += Q x
  } else {
    level1_8(x, y, false);
    mult8(y, bT2.p);
    applyQ8(bT2.p, bT2.p);
    vec_axpby(n8, -1., bT2.p, 1., y, st);
  }
}

void GeneoPC::apply_block(int k, const double* X, int64_t ldx, double* Y, int64_t ldy) {
  GENEO_CHECK(k >= 1 && ldx >= nLoc && ldy >= nLoc, "block apply: k >= 1 and leading dimensions >= the vector length");
  ensure_block();
  for (int j0 = 0; j0 < k; j0 += 8) {
    const int nc = std::min(8, k - j0);
    pack_cols8(nLoc, nc, X + (size_t)j0 * ldx, ldx, bIn.p, st);
    apply8(bIn.p, bOut.p);
    unpack_cols8(nLoc, nc, bOut.p, Y + (size_t)j0 * ldy, ldy, st);
  }
  applyCount += k;
}

double GeneoPC::trisolve_algo_bytes() const {
  double b = 0.;
  for (auto& s : subs)
    for (auto& F : s.plan->sym.fronts) {
      const double k = F.k, m = F.m();
      b += 8. * (2. * m * k + k * k) + 2. * 4. * m + 8. * 4. * (k + m);  // factor once fwd + once bwd, D^-1 once, indices, x/y
    }
  return b;
}
double GeneoPC::apply_algo_bytes() const {
  double b = trisolve_algo_bytes();
  double nz = 0.;
  for (auto& s : subs) nz += (double)s.n * s.nev;
  b += 6. * 8. * (double)nAll + 4. * (double)nAll;
  if (opt.lvl2 >= 1) b += 2. * 8. * nz + 8. * (double)nE * nE;
  b += 2. * 8. * (double)nLoc;
  return b;
}

// =====================================================================================================================
// Krylov: PETSc-faithful left-preconditioned CG and GMRES(m)
// =====================================================================================================================
namespace {
struct ConvTest {  // KSPConvergedDefault
  double ttol = 0., rnorm0 = 0., atol = 0., dtol = 0.;
  int operator()(double rn) const {
    if (rn != rn) return KSP_DIVERGED_NANORINF;
    if (rn <= ttol) return rn < atol ? KSP_CONVERGED_ATOL : KSP_CONVERGED_RTOL;
    if (rn >= dtol * rnorm0) return KSP_DIVERGED_DTOL;
    return 0;
  }
};
}  // namespace

KspResult GeneoPC::solve_cg(const double* b, double* x, double rtol, double atol, double dtol, int maxIt) {
  KspResult R;
  DevBuf<double> r(nLoc), z(nLoc), p(nLoc), wv(nLoc);
  mult_sub(x, b, r.p);  // non-zero initial guess is ALWAYS flagged (src/geneo4PETSc.cpp:1348)
  apply(r.p, z.p);
  double dp = norm(z.p);
  R.history.push_back(dp);
  ConvTest conv;
  {  // reference norm ||M^-1 b|| (guess non-zero)
    apply(b, wv.p);
    double sn = norm(wv.p);
    if (sn == 0.) sn = dp;
    conv.ttol = std::max(rtol * sn, atol); conv.rnorm0 = sn; conv.atol = atol; conv.dtol = dtol;
  }
  R.rnorm = dp;
  R.reason = conv(dp);
  if (R.reason) return R;
  double beta = dot(z.p, r.p), betaold = 1.;
  int i = 0;
  while (i < maxIt) {
    if (beta == 0.) { R.reason = KSP_CONVERGED_ATOL; R.its = i; return R; }
    if (i > 0 && beta * betaold < 0.) { R.reason = KSP_DIVERGED_INDEFINITE_PC; R.its = i; return R; }
    if (i == 0) CUDA_CHECK(cudaMemcpyAsync(p.p, z.p, sizeof(double) * nLoc, cudaMemcpyDeviceToDevice, st));
    else vec_aypx(nLoc, beta / betaold, z.p, p.p, st);  // p = z + b p
    mult(p.p, wv.p);
    const double dpi = dot(p.p, wv.p);
    betaold = beta;
    if (dpi <= 0.) { R.reason = KSP_DIVERGED_INDEFINITE_MAT; R.its = i + 1; return R; }
    const double a = beta / dpi;
    vec_cg_update(nLoc, a, p.p, wv.p, x, r.p, st);
    apply(r.p, z.p);
    vec_dot2(nOwn, z.p, r.p, z.p, scal.p, st);  // beta = z.r and ||z||^2 in one pass
    comm.allreduce_sum(scal.p, 2, st);
    double h[2];
    CUDA_CHECK(cudaMemcpyAsync(h, scal.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(::geneo::sync_stream(st));
    dp = std::sqrt(h[1]);
    R.history.push_back(dp);
    R.rnorm = dp;
    R.its = i + 1;
    R.reason = conv(dp);
    if (R.reason) return R;
    beta = h[0];
    i++;
  }
  R.reason = KSP_DIVERGED_ITS;
  R.its = i;
  return R;
}

KspResult GeneoPC::solve_gmres(const double* b, double* x, double rtol, double atol, double dtol, int maxIt, int restart) {
  KspResult R;
  restart = std::max(1, std::min(restart, maxIt));
  size_t freeB = 0, totB = 0;
  CUDA_CHECK(cudaMemGetInfo(&freeB, &totB));
  const size_t need = (size_t)(restart + 1) * nLoc * sizeof(double);
  if (need > freeB * 0.9) {  // the reference's test scripts use -ksp_gmres_restart 1000; clamp to what fits
    restart = (int)std::max<size_t>(2, (size_t)(freeB * 0.9 / ((double)nLoc * sizeof(double))) - 1);
    fprintf(stderr, "WRNG: geneo_b200: GMRES restart clamped to %d (device memory)\n", restart);
  }
  DevBuf<double> V((size_t)(restart + 1) * nLoc), t(nLoc), wv(nLoc), coef(restart + 8);
  std::vector<double> H((size_t)(restart + 1) * restart, 0.), cs(restart), sn(restart), g(restart + 1), hk(restart + 8), y(restart);
  ConvTest conv;
  bool haveTol = false;
  int its = 0;
  double res = 0.;
  int reason = 0;
  while (true) {
    mult_sub(x, b, t.p);
    apply(t.p, V.p);  // r = M^-1 (b - A x)
    res = norm(V.p);
    if (!haveTol) {
      apply(b, wv.p);
      double s0 = norm(wv.p);
      if (s0 == 0.) s0 = res;
      conv.ttol = std::max(rtol * s0, atol); conv.rnorm0 = s0; conv.atol = atol; conv.dtol = dtol;
      haveTol = true;
      R.history.push_back(res);
    }
    reason = conv(res);
    if (reason || its >= maxIt) break;
    if (res == 0.) { reason = KSP_CONVERGED_ATOL; break; }
    vec_scale(nLoc, 1. / res, V.p, st);
    std::fill(g.begin(), g.end(), 0.);
    g[0] = res;
    int k = 0;
    while (k < restart && its < maxIt) {
      double* vk = V.p + (size_t)k * nLoc;
      double* vn = V.p + (size_t)(k + 1) * nLoc;
      mult(vk, t.p);
      apply(t.p, vn);  // w = M^-1 A v_k
      vec_mdot(nOwn, k + 1, V.p, nLoc, vn, coef.p, st);  // classical Gram-Schmidt, no refinement (PETSc default)
      comm.allreduce_sum(coef.p, k + 1, st);
      vec_maxpy(nLoc, k + 1, V.p, nLoc, coef.p, vn, st);
      CUDA_CHECK(cudaMemcpyAsync(hk.data(), coef.p, sizeof(double) * (k + 1), cudaMemcpyDeviceToHost, st));
      const double tt = norm(vn);
      for (int j = 0; j <= k; j++) H[(size_t)j * restart + k] = hk[j];
      double hap = g[k] != 0. ? std::fabs(tt / g[k]) : 1e-30;
      if (hap > 1e-30) hap = 1e-30;
      const bool happy = tt < hap;
      if (!happy) vec_scale(nLoc, 1. / tt, vn, st);
      H[(size_t)(k + 1) * restart + k] = tt;
      for (int j = 0; j < k; j++) {
        const double t1v = H[(size_t)j * restart + k];
        H[(size_t)j * restart + k] = cs[j] * t1v + sn[j] * H[(size_t)(j + 1) * restart + k];
        H[(size_t)(j + 1) * restart + k] = -sn[j] * t1v + cs[j] * H[(size_t)(j + 1) * restart + k];
      }
      const double den = std::hypot(H[(size_t)k * restart + k], H[(size_t)(k + 1) * restart + k]);
      if (den == 0.) { reason = KSP_DIVERGED_BREAKDOWN; break; }
      cs[k] = H[(size_t)k * restart + k] / den;
      sn[k] = H[(size_t)(k + 1) * restart + k] / den;
      H[(size_t)k * restart + k] = den;
      H[(size_t)(k + 1) * restart + k] = 0.;
      g[k + 1] = -sn[k] * g[k];
      g[k] = cs[k] * g[k];
      res = std::fabs(g[k + 1]);
      k++;
      its++;
      R.history.push_back(res);
      reason = conv(res);
      if (reason) break;
      if (happy) { reason = KSP_CONVERGED_HAPPY_BREAKDOWN; break; }
    }
    if (k > 0) {  // x += V y,  H y = g
      for (int i = k - 1; i >= 0; i--) {
        double s = g[i];
        for (int j = i + 1; j < k; j++) s -= H[(size_t)i * restart + j] * y[j];
        y[i] = s / H[(size_t)i * restart + i];
      }
      for (int i = 0; i < k; i++) hk[i] = -y[i];
      CUDA_CHECK(cudaMemcpyAsync(coef.p, hk.data(), sizeof(double) * k, cudaMemcpyHostToDevice, st));
      vec_maxpy(nLoc, k, V.p, nLoc, coef.p, x, st);
      CUDA_CHECK(::geneo::sync_stream(st));
    }
    if (reason) break;
    if (its >= maxIt) { reason = KSP_DIVERGED_ITS; break; }
  }
  if (!reason) reason = KSP_DIVERGED_ITS;
  R.its = its;
  R.rnorm = res;
  R.reason = reason;
  return R;
}

std::vector<KspResult> GeneoPC::solve_cg_block(int k, const double* B, int64_t ldb, double* X, int64_t ldx, double rtol,
                                               double atol, double dtol, int maxIt) {
  GENEO_CHECK(k >= 1 && ldb >= nLoc && ldx >= nLoc, "block CG: k >= 1 and leading dimensions >= the vector length");
  ensure_block();
  std::vector<KspResult> res(k);
  for (int j0 = 0; j0 < k; j0 += 8) {  // bIn = b, bOut = x of the chunk (apply8 leaves both alone)
    const int nc = std::min(8, k - j0);
    pack_cols8(nLoc, nc, B + (size_t)j0 * ldb, ldb, bIn.p, st);
    if (opt.lvl2 >= 1 && opt.effHybrid) applyQ8(bIn.p, bOut.p);  // initial_guess: x0 = Q b, or 0
    else bOut.zero(st);
    cg8(bIn.p, bOut.p, (1u << nc) - 1u, rtol, atol, dtol, maxIt, res.data() + j0);
    unpack_cols8(nLoc, nc, bOut.p, X + (size_t)j0 * ldx, ldx, st);
  }
  CUDA_CHECK(::geneo::sync_stream(st));
  return res;
}

// solve_cg on the columns set in `active` (the others are zero padding), all of them in lock step: one block SpMV and one
// block PC apply per iteration, the per-column dots in one pass and one host read-back each.  A column that stops is
// frozen (its x and r are not written again) and keeps the its / reason / rnorm solve_cg would have returned.
void GeneoPC::cg8(const double* b, double* x, unsigned active, double rtol, double atol, double dtol, int maxIt, KspResult* res) {
  const int nc = 32 - __builtin_clz(active);
  DevBuf<double> r((size_t)nLoc * 8), z((size_t)nLoc * 8), p((size_t)nLoc * 8), wv((size_t)nLoc * 8);
  double h[16];
  auto readback = [&](int cnt) {
    comm.allreduce_sum(scal.p, cnt, st);
    CUDA_CHECK(cudaMemcpyAsync(h, scal.p, cnt * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(::geneo::sync_stream(st));
  };
  mult_sub8(x, b, r.p);  // non-zero initial guess, as solve_cg
  apply8(r.p, z.p);
  dot_cols8(nOwn, z.p, r.p, z.p, scal.p, st);  // beta = z.r and ||z||^2
  double zr[8], zz[8];
  readback(16);
  for (int c = 0; c < 8; c++) { zr[c] = h[c]; zz[c] = h[8 + c]; }
  apply8(const_cast<double*>(b), wv.p);  // reference norm ||M^-1 b|| (b's ghost rows are refreshed, its owned rows kept)
  applyCount += 2 * nc;
  dot_cols8(nOwn, wv.p, wv.p, nullptr, scal.p, st);
  readback(8);
  ConvTest conv[8];
  double beta[8], betaold[8];
  for (int c = 0; c < 8; c++) {
    beta[c] = 0.;
    betaold[c] = 1.;
    if (!((active >> c) & 1u)) continue;
    KspResult& R = res[c];
    const double dp = std::sqrt(zz[c]);
    double sn = std::sqrt(h[c]);
    if (sn == 0.) sn = dp;
    conv[c].ttol = std::max(rtol * sn, atol); conv[c].rnorm0 = sn; conv[c].atol = atol; conv[c].dtol = dtol;
    R.history.push_back(dp);
    R.rnorm = dp;
    R.reason = conv[c](dp);
    if (R.reason) active &= ~(1u << c);
    beta[c] = zr[c];
  }
  auto stop = [&](int c, int reason, int its) { res[c].reason = reason; res[c].its = its; active &= ~(1u << c); };
  int i = 0;
  while (active) {
    for (int c = 0; c < 8; c++) {
      if (!((active >> c) & 1u)) continue;
      if (i >= maxIt) stop(c, KSP_DIVERGED_ITS, i);
      else if (beta[c] == 0.) stop(c, KSP_CONVERGED_ATOL, i);
      else if (i > 0 && beta[c] * betaold[c] < 0.) stop(c, KSP_DIVERGED_INDEFINITE_PC, i);
    }
    if (!active) break;
    Coef8 cf{};
    for (int c = 0; c < 8; c++) cf.v[c] = beta[c] / betaold[c];
    if (i == 0) CUDA_CHECK(cudaMemcpyAsync(p.p, z.p, sizeof(double) * nLoc * 8, cudaMemcpyDeviceToDevice, st));
    else aypx8(nLoc, cf, active, z.p, p.p, st);  // p = z + b p
    mult8(p.p, wv.p);
    dot_cols8(nOwn, p.p, wv.p, nullptr, scal.p, st);
    readback(8);
    for (int c = 0; c < 8; c++) {
      if (!((active >> c) & 1u)) continue;
      betaold[c] = beta[c];
      if (h[c] <= 0.) stop(c, KSP_DIVERGED_INDEFINITE_MAT, i + 1);
      else cf.v[c] = beta[c] / h[c];
    }
    cg_update8(nLoc, cf, active, p.p, wv.p, x, r.p, st);
    if (!active) break;
    apply8(r.p, z.p);
    applyCount += __builtin_popcount(active);
    dot_cols8(nOwn, z.p, r.p, z.p, scal.p, st);
    readback(16);
    for (int c = 0; c < 8; c++) {
      if (!((active >> c) & 1u)) continue;
      KspResult& R = res[c];
      const double dp = std::sqrt(h[8 + c]);
      R.history.push_back(dp);
      R.rnorm = dp;
      R.its = i + 1;
      R.reason = conv[c](dp);
      if (R.reason) active &= ~(1u << c);
      beta[c] = h[c];
    }
    i++;
  }
}

}  // namespace geneo
