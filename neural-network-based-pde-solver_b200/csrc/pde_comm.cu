// pde_comm.cu — the exchange step of the data-parallel loss step as ONE kernel over NVLink peer
// memory (SURVEY.md §8e, §8f-4).
//
// What is exchanged is tiny — [grad | dE | sums], 12 803 floats = 51 KB for config 2 — so the cost
// of an all-reduce is launch + protocol latency, not bandwidth.  pde_allreduce_oneshot is a
// flag-in-data ("low latency") push protocol with a single one-way NVLink trip on the critical path:
//
//   push    : every 32-bit word of the rank's vector is stored, paired with the call number, as one
//             8-byte word into the slot [parity][source rank][i] of EVERY peer (8-byte stores are
//             single-copy atomic, so the flag can never be seen without its data; no fence, no
//             separate signal, no copy-in)
//   reduce  : the rank polls its own (local) slots until the W-1 flags of an element carry the call
//             number and adds the values in rank order 0..W-1 — the same order on every rank, so the
//             replicated parameters stay bit-identical and the result does not depend on arrival order
//
// Slots are double buffered by call parity.  No end-of-call barrier is needed: parity p is rewritten
// two calls later, and a rank only gets there after its call in between has completed, which needed
// every peer's data of that call, which the peer pushes only after it has finished reading parity p.
// The call counter lives in device memory, so the kernel is CUDA-graph replayable; elements are
// independent, so any number of blocks can run (the last one to finish advances the counter).
//
// Lockstep requirement and failure reporting.  Like any collective, every rank must make the same sequence of
// calls.  A rank waits for its peers' words for at most the exchange timeout (pde_set_exchange_timeout, default
// 600 s, 0 = wait for ever; host-side skew such as a checkpoint on one rank or a first-call module load is
// therefore harmless).  If the wait does expire the rank poisons ITS result with NaN and increments an error
// word in its own control block; the peers, which did receive this rank's words, cannot know, so the host side
// must look: pde_exchange_errors() reads the word (comm.NvlinkAllReduce.check() raises on it, and the fused
// trainer / bench.py call that at every point where they synchronise anyway).
//
// Peer buffers are plain cudaMalloc allocations shared with CUDA IPC handles (pde_peer_alloc /
// pde_peer_open); the handles travel through torch.distributed's object collectives once at set-up.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <atomic>

#include "../../include/pde_b200.h"
#include "pde_comm.cuh"
#include "pde_launch.h"

namespace {

using namespace pde::comm;
constexpr int COMM_THREADS = 256, COMM_MAX_BLOCKS = 16;
std::atomic<long long> g_spin_limit{600ll * 2000000000ll};   // clock64 ticks; <= 0: no timeout

// Thread = one element.
template <typename T>
__global__ void __launch_bounds__(COMM_THREADS) allreduce_oneshot_kernel(const CommArgs a) {
  constexpr int WPE = sizeof(T) / 4;
  const uint32_t call = *a.seq + 1u;
  T* buf = static_cast<T*>(a.buf);
  const long long n = a.n_words / WPE;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    buf[i] = exchange_element<T>(a, i, buf[i], call);
  finish_call(a, call);
}

}  // namespace

namespace pde {
int comm_fill_args(const pde_peers* peers, int32_t dtype, int64_t n, int64_t slot_elems, void* seq, comm::CommArgs* out) {
  if (!peers || !seq || !out) return PDE_ERR_INVALID;
  if (dtype != PDE_F32 && dtype != PDE_F64) return PDE_ERR_INVALID;
  if (peers->world < 1 || peers->world > PDE_MAX_PEERS || peers->rank < 0 || peers->rank >= peers->world) return PDE_ERR_INVALID;
  if (n < 1 || n > slot_elems) return PDE_ERR_INVALID;
  comm::CommArgs& a = *out;
  a.rank = peers->rank; a.world = peers->world;
  for (int p = 0; p < PDE_MAX_PEERS; ++p) {
    a.base[p] = p < peers->world ? static_cast<unsigned char*>(peers->base[p]) : nullptr;
    if (p < peers->world && !a.base[p]) return PDE_ERR_INVALID;
  }
  const int wpe = dtype == PDE_F64 ? 2 : 1;
  a.n_words = n * wpe; a.slot_words = slot_elems * wpe; a.is_f64 = dtype == PDE_F64;
  a.buf = nullptr; a.seq = static_cast<uint32_t*>(seq);
  a.spin_limit = g_spin_limit.load(std::memory_order_relaxed);
  return PDE_OK;
}
}  // namespace pde

extern "C" {

int pde_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64) {
  if (!ptr || !handle64 || bytes == 0) return PDE_ERR_INVALID;
  void* p = nullptr;
  if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return PDE_ERR_CUDA; }
  if (cudaMemset(p, 0, bytes) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) { cudaFree(p); cudaGetLastError(); return PDE_ERR_CUDA; }
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, p) != cudaSuccess) { cudaFree(p); cudaGetLastError(); return PDE_ERR_CUDA; }
  static_assert(sizeof(h) == 64, "CUDA IPC handle size");
  memcpy(handle64, &h, 64);
  *ptr = p;
  return PDE_OK;
}

int pde_peer_open(const unsigned char* handle64, void** ptr) {
  if (!ptr || !handle64) return PDE_ERR_INVALID;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  void* p = nullptr;
  if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); return PDE_ERR_CUDA; }
  *ptr = p;
  return PDE_OK;
}

int pde_peer_close(void* ptr) {
  if (!ptr) return PDE_ERR_INVALID;
  if (cudaIpcCloseMemHandle(ptr) != cudaSuccess) { cudaGetLastError(); return PDE_ERR_CUDA; }
  return PDE_OK;
}

int pde_peer_free(void* ptr) {
  if (!ptr) return PDE_ERR_INVALID;
  if (cudaFree(ptr) != cudaSuccess) { cudaGetLastError(); return PDE_ERR_CUDA; }
  return PDE_OK;
}

int pde_peer_bytes(int32_t dtype, int64_t slot_elems, size_t* bytes) {
  if (!bytes || slot_elems < 1 || (dtype != PDE_F32 && dtype != PDE_F64)) return PDE_ERR_INVALID;
  const size_t words = (size_t)slot_elems * (dtype == PDE_F64 ? 2 : 1);
  *bytes = (size_t)CTRL_BYTES + 2 * (size_t)PDE_MAX_PEERS * words * 8;   // (value, flag) pairs, per parity and source rank
  return PDE_OK;
}

int pde_allreduce_oneshot(const pde_peers* peers, int32_t dtype, void* buf, int64_t n, int64_t slot_elems, void* seq,
                          void* stream) {
  if (!buf) return PDE_ERR_INVALID;
  CommArgs a;
  int rc = pde::comm_fill_args(peers, dtype, n, slot_elems, seq, &a);
  if (rc) return rc;
  a.buf = buf;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  long long g = (n + COMM_THREADS - 1) / COMM_THREADS;
  const int grid = (int)(g < 1 ? 1 : (g > COMM_MAX_BLOCKS ? COMM_MAX_BLOCKS : g));
  if (dtype == PDE_F32) allreduce_oneshot_kernel<float><<<grid, COMM_THREADS, 0, st>>>(a);
  else allreduce_oneshot_kernel<double><<<grid, COMM_THREADS, 0, st>>>(a);
  pde::count_launch(1);
  return cudaGetLastError() == cudaSuccess ? PDE_OK : PDE_ERR_CUDA;
}

int pde_set_exchange_timeout(double seconds) {
  if (!(seconds >= 0.0) || seconds > 1.0e6) return PDE_ERR_INVALID;
  g_spin_limit.store((long long)(seconds * 2.0e9), std::memory_order_relaxed);   // clock64 ticks at <= 2 GHz; 0 = no timeout
  return PDE_OK;
}

int pde_exchange_errors(const pde_peers* peers, uint32_t* timeouts, void* stream) {
  if (!peers || !timeouts || peers->rank < 0 || peers->rank >= PDE_MAX_PEERS || !peers->base[peers->rank]) return PDE_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uint32_t* word = static_cast<const uint32_t*>(peers->base[peers->rank]) + CTRL_ERR_WORD;
  if (cudaMemcpyAsync(timeouts, word, sizeof(uint32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess) { cudaGetLastError(); return PDE_ERR_CUDA; }
  if (cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); return PDE_ERR_CUDA; }
  return PDE_OK;
}

}  // extern "C"
