// comm.cu -- see comm.hpp.
#include "comm.hpp"

#include <dlfcn.h>

#include <cstring>

namespace geneo {
namespace {

// minimal NCCL ABI (nccl.h 2.x): opaque comm, 128-byte unique id, enums as ints
struct NcclUid { char internal[128]; };
typedef void* ncclComm_t;
enum { ncclSuccess = 0 };
enum { ncclFloat64 = 8 };  // ncclDataType_t: int8 0, uint8 1, int32 2, uint32 3, int64 4, uint64 5, f16 6, f32 7, f64 8
enum { ncclSum = 0 };
struct Api {
  int (*GetUniqueId)(NcclUid*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, NcclUid, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
};
Api& api() {
  static Api a;
  if (a.ok) return a;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);  // the copy torch already loaded, if any
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) throw Error(std::string("geneo_b200: cannot load libnccl.so.2 for the multi-GPU path: ") + dlerror());
  auto sym = [&](const char* n) { void* p = dlsym(h, n); if (!p) throw Error(std::string("geneo_b200: libnccl lacks ") + n); return p; };
  a.GetUniqueId = (decltype(a.GetUniqueId))sym("ncclGetUniqueId");
  a.CommInitRank = (decltype(a.CommInitRank))sym("ncclCommInitRank");
  a.AllReduce = (decltype(a.AllReduce))sym("ncclAllReduce");
  a.Send = (decltype(a.Send))sym("ncclSend");
  a.Recv = (decltype(a.Recv))sym("ncclRecv");
  a.GroupStart = (decltype(a.GroupStart))sym("ncclGroupStart");
  a.GroupEnd = (decltype(a.GroupEnd))sym("ncclGroupEnd");
  a.GetErrorString = (decltype(a.GetErrorString))sym("ncclGetErrorString");
  a.ok = true;
  return a;
}
#define NCCL_CHECK(call)                                                                                     \
  do {                                                                                                       \
    int r__ = (call);                                                                                        \
    if (r__ != ncclSuccess)                                                                                  \
      throw Error(std::string("geneo_b200: NCCL error ") + api().GetErrorString(r__) + " in " #call " at " + \
                  __FILE__ + ":" + std::to_string(__LINE__));                                                \
  } while (0)

// buf[t*width + c] = x[idx[t]*width + c]
__global__ void k_pack_rows(int64_t cnt, int width, const int* __restrict__ idx, const double* __restrict__ x,
                            double* __restrict__ buf) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < cnt * width; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / width;
    const int c = (int)(t - r * width);
    buf[t] = x[(int64_t)idx[r] * width + c];
  }
}
// y[idx[t]*width + c] += buf[t*width + c].  A row may appear once per peer, so the adds of different peers are issued
// as separate launches (peer order = rank order): the sum order is deterministic.
__global__ void k_unpack_add_rows(int64_t cnt, int width, const int* __restrict__ idx, const double* __restrict__ buf,
                                  double* __restrict__ y) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < cnt * width; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / width;
    const int c = (int)(t - r * width);
    y[(int64_t)idx[r] * width + c] += buf[t];
  }
}
inline int grid_for(int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, 148 * 8)); }

}  // namespace

// One NCCL communicator per PROCESS and (rank, world), shared by every preconditioner the process sets up -- the way MPI
// hands the reference one PETSC_COMM_WORLD for all its PCs.  ncclCommInitRank and the lazily established peer connections of
// the first send / recv / allreduce cost seconds on 8 GPUs; a second PCSetUp in the same job must not pay them again.
namespace {
struct SharedComm { int rank, world; ncclComm_t c; };
std::vector<SharedComm>& shared_comms() { static std::vector<SharedComm>* v = new std::vector<SharedComm>(); return *v; }
}  // namespace

void Comm::reset() {
  comm_ = nullptr;
  rank = 0; world = 1; nOwn = nGhost = 0; bufWidth_ = 0;
  sendPtr_.clear(); recvPtr_.clear();
}

void Comm::unique_id(void* out128) {
  NcclUid id;
  NCCL_CHECK(api().GetUniqueId(&id));
  std::memcpy(out128, &id, sizeof(id));
}

void Comm::init(int rank_, int world_, const void* uid128, const RankLayout& L, cudaStream_t st) {
  reset();
  rank = rank_; world = world_;
  nOwn = L.nOwn(); nGhost = L.nGhost();
  if (world <= 1) return;
  GENEO_CHECK(uid128 != nullptr, "multi-GPU setup without an NCCL unique id");
  ncclComm_t c = nullptr;
  for (auto& sc : shared_comms())
    if (sc.rank == rank && sc.world == world) c = sc.c;  // (every rank takes the same branch: they all set up the same sequence of PCs)
  if (!c) {
    NcclUid id;
    std::memcpy(&id, uid128, sizeof(id));
    NCCL_CHECK(api().CommInitRank(&c, world, id, rank));
    shared_comms().push_back(SharedComm{rank, world, c});
  }
  comm_ = c;
  sendPtr_.assign(world + 1, 0);
  recvPtr_.assign(L.ghostPtr.begin(), L.ghostPtr.end());
  std::vector<int> idx;
  for (int q = 0; q < world; q++) {
    idx.insert(idx.end(), L.sendIdx[q].begin(), L.sendIdx[q].end());
    sendPtr_[q + 1] = (int64_t)idx.size();
  }
  if (idx.empty()) idx.push_back(0);
  dSendIdx_.upload(idx, st);
  CUDA_CHECK(::geneo::sync_stream(st));
  ensure(1);
}

void Comm::ensure(int width) {
  if (width <= bufWidth_) return;
  bufWidth_ = width;
  sendBuf_.alloc((size_t)std::max<int64_t>(1, sendPtr_[world]) * width);
  recvBuf_.alloc((size_t)std::max<int64_t>(1, sendPtr_[world]) * width);
}

void Comm::allreduce_sum(double* d, int n, cudaStream_t st) {
  if (!active() || n <= 0) return;
  NCCL_CHECK(api().AllReduce(d, d, (size_t)n, ncclFloat64, ncclSum, (ncclComm_t)comm_, st));
}

void Comm::allreduce_sum_host(double* h, int n, cudaStream_t st) {
  if (!active() || n <= 0) return;
  if ((int)tmp_.n < n) tmp_.alloc((size_t)n);
  CUDA_CHECK(cudaMemcpyAsync(tmp_.p, h, sizeof(double) * n, cudaMemcpyHostToDevice, st));
  allreduce_sum(tmp_.p, n, st);
  CUDA_CHECK(cudaMemcpyAsync(h, tmp_.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
  CUDA_CHECK(::geneo::sync_stream(st));
}

void Comm::halo_forward(double* x, int width, cudaStream_t st) {
  if (!active()) return;
  ensure(width);
  const int64_t ns = sendPtr_[world];
  if (ns) k_pack_rows<<<GENEO_TICK(grid_for(ns * width)), 256, 0, st>>>(ns, width, dSendIdx_.p, x, sendBuf_.p);
  NCCL_CHECK(api().GroupStart());
  for (int q = 0; q < world; q++) {
    if (q == rank) continue;
    const int64_t s = sendPtr_[q + 1] - sendPtr_[q], r = recvPtr_[q + 1] - recvPtr_[q];
    if (s) NCCL_CHECK(api().Send(sendBuf_.p + sendPtr_[q] * width, (size_t)(s * width), ncclFloat64, q, (ncclComm_t)comm_, st));
    if (r) NCCL_CHECK(api().Recv(x + ((int64_t)nOwn + recvPtr_[q]) * width, (size_t)(r * width), ncclFloat64, q, (ncclComm_t)comm_, st));  // ghosts are grouped by owner: no unpack
    bytesSent += s * width * 8;
  }
  NCCL_CHECK(api().GroupEnd());
}

void Comm::halo_reverse_add(double* y, int width, cudaStream_t st) {
  if (!active()) return;
  ensure(width);
  NCCL_CHECK(api().GroupStart());
  for (int q = 0; q < world; q++) {
    if (q == rank) continue;
    const int64_t s = sendPtr_[q + 1] - sendPtr_[q], r = recvPtr_[q + 1] - recvPtr_[q];
    if (r) NCCL_CHECK(api().Send(y + ((int64_t)nOwn + recvPtr_[q]) * width, (size_t)(r * width), ncclFloat64, q, (ncclComm_t)comm_, st));  // ghost partial sums, contiguous per owner: no pack
    if (s) NCCL_CHECK(api().Recv(recvBuf_.p + sendPtr_[q] * width, (size_t)(s * width), ncclFloat64, q, (ncclComm_t)comm_, st));
    bytesSent += r * width * 8;
  }
  NCCL_CHECK(api().GroupEnd());
  for (int q = 0; q < world; q++) {
    const int64_t s = sendPtr_[q + 1] - sendPtr_[q];
    if (q == rank || !s) continue;
    k_unpack_add_rows<<<GENEO_TICK(grid_for(s * width)), 256, 0, st>>>(s, width, dSendIdx_.p + sendPtr_[q], recvBuf_.p + sendPtr_[q] * width, y);
  }
}

}  // namespace geneo
