// comm.hpp -- multi-GPU plumbing of the hot path: one process per GPU, NCCL over NVLink/NVSwitch (SURVEY.md 8e).
// Replaces the MPI layer under PETSc's VecScatter / MatMult(MATIS) / VecDot (reference call sites
// src/geneo.cpp:1850-1852, 1881-1883, 1931-1935; src/geneo4PETSc.cpp:1240): exactly three exchange steps exist --
//   (1) halo forward (owner -> ghost copies) / reverse-add (ghost partial sums -> owner),
//   (2) allreduce of Krylov dots / norms and of the coarse vector Z^T x (E^-1 is replicated),
//   (3) allreduce of E and of the nev_i at setup.
// libnccl is dlopen'ed (the torch-bundled or the system one): the library has no link-time dependency on it and a
// single-GPU process never touches it.
#pragma once
#include <vector>
#include "common.hpp"
#include "mesh.hpp"

namespace geneo {

class Comm {
 public:
  int rank = 0, world = 1;
  bool active() const { return world > 1; }
  void reset();  // back to the single-process state (the process-wide communicator stays for the next init)
  static void unique_id(void* out128);  // ncclGetUniqueId (rank 0), to be broadcast by the caller
  void init(int rank, int world, const void* uid128, const RankLayout& L, cudaStream_t st);
  void allreduce_sum(double* d, int n, cudaStream_t st);      // in place, device buffer
  void allreduce_sum_host(double* h, int n, cudaStream_t st); // small host arrays (setup statistics)
  // x: [nOwn | nGhost] rows of `width` doubles (row-major).  forward: ghosts <- owners' values.
  void halo_forward(double* x, int width, cudaStream_t st);
  // reverse: owners += ghost partial sums (ghost rows are left untouched)
  void halo_reverse_add(double* y, int width, cudaStream_t st);
  int nOwn = 0, nGhost = 0;
  int64_t bytesSent = 0;  // per-process NVLink traffic issued (statistics)
 private:
  void* comm_ = nullptr;  // ncclComm_t: the process-wide communicator of (rank, world), never destroyed
  std::vector<int64_t> sendPtr_, recvPtr_;  // [world+1]: rows sent to / received from each peer
  DevBuf<int> dSendIdx_;
  DevBuf<double> sendBuf_, recvBuf_, tmp_;
  void ensure(int width);
  int bufWidth_ = 0;
};

}  // namespace geneo
