// b200ddp.cu — libb200ddp.so: B200 (sm_100a) data plane for the `local_cuda` TorchX scheduler.
//
// What lives here (see include/b200ddp.h for the ABI and DESIGN.md for the rationale):
//   * rendezvous: POSIX-shm control block + exchange of ONE symmetric arena per rank, either as CUDA VMM allocations
//     shared by file descriptor and bound into an NVSwitch MULTICAST object (b2_vmm.h), or - when the driver / fabric
//     does not offer that - as cudaMalloc + CUDA IPC
//     (replaces c10d TCPStore + ncclCommInitRank on the reference path,
//      torchx/distributed/__init__.py:217-222 -> torch.distributed.init_process_group)
//   * the DDP gradient-bucket allreduce as ONE fused kernel per bucket
//     (replaces the 4-launch cast -> div -> ncclAllReduce -> copy sequence of
//      torch/distributed/algorithms/ddp_comm_hooks/default_hooks.py:57-93)
//       - one-shot        : push compressed message to every peer, one flag barrier, reduce locally   (b2_kernels.cuh)
//       - two-shot        : push-scatter -> reduce own slice -> pull-gather, single pass              (b2_kernels.cuh)
//       - two-shot, piped : the same three phases as warp-specialised roles over K chunks            (b2_pipe.cuh)
//       - NVLS, piped     : cast -> multimem.ld_reduce / multimem.st through the switch -> widen      (b2_pipe.cuh)
//   * broadcast / barrier on the same fabric (DDP init + BN-buffer sync, dist.barrier()).
//
// Memory model: every cross-GPU hand-off is  data stores -> bar.sync -> st.release.sys(flag)
// on the producer and  ld.acquire.sys(flag) -> bar.sync -> data loads  on the consumer, with a
// monotonically increasing sequence number instead of flag resets (no ABA, no reset races).
// All peer waits are bounded: a CTA that waits longer than `timeout_ns` records B2_ETIMEOUT in a
// host-mapped status word and carries on, so a dead peer can never hang the GPU.
//
// No tensor cores: the path is a pure bandwidth-bound reduction (1 add per 2-4 bytes moved).

#include "b2_dev.cuh"
#include "b2_kernels.cuh"
#include "b2_pipe.cuh"
#include "b2_ll.cuh"
#include "b2_vmm.h"

#include <errno.h>
#include <fcntl.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

#include <atomic>
#include <map>
#include <mutex>
#include <new>
#include <string>

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char tmp[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(tmp, sizeof(tmp), fmt, ap);
  va_end(ap);
  g_err = tmp;
  return code;
}

#define B2_CUDA(expr)                                                                         \
  do {                                                                                        \
    cudaError_t e__ = (expr);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return fail(B2_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, \
                  __LINE__);                                                                  \
  } while (0)

struct DeviceGuard {  // the library never leaves the caller's current device changed
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

double now_s() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec + 1e-9 * ts.tv_nsec;
}

// ---- shm control block (multi-process rendezvous) ----------------------------------------------
constexpr uint64_t kShmMagic = 0x42323030444451ull;  // "B200DDQ": layout 2

struct ShmSlot {
  cudaIpcMemHandle_t handle;  // cudaMalloc backend only
  int device;        // the rank's ordinal in ITS OWN numbering (CUDA_VISIBLE_DEVICES may differ between ranks)
  char bus_id[24];   // PCI bus id: the identity that is comparable across processes
  int pid;
  int cap_vmm;       // this rank can build its arena from VMM objects and pass file descriptors
  int cap_mc;        // ... and its device supports NVSwitch multicast
  unsigned long long arena_bytes;
  std::atomic<uint32_t> hello;  // 1 once cap_* are valid (backend agreement happens before any allocation)
  std::atomic<uint32_t> ready;  // 1 once handle/device/pid/arena_bytes are valid and the fd socket is bound
  char pad[64];
};

struct ShmBlock {
  std::atomic<uint64_t> magic;
  uint64_t epoch;
  int world;
  std::atomic<int> mapped;     // ranks that have mapped every peer arena
  std::atomic<int> departed;   // ranks that have finished using peer memory (destroy handshake)
  std::atomic<int> mc_added;   // multicast: ranks past cuMulticastAddDevice
  std::atomic<int> mc_bound;   // ... past cuMulticastBindMem
  std::atomic<int> mc_mapped;  // ... past mapping the multicast object
  std::atomic<int> mc_fail;    // any rank failed a multicast step: everybody drops the NVLS path
  ShmSlot slot[B2_MAX_WORLD];
};

// the multicast mapping of an in-process world is shared by its ranks
struct LocalMc {
  vmm::Mapping map;
  int refs = 0;
};

}  // namespace

struct b2_comm {
  CommDev d{};
  int device = -1;
  bool local_world = false;    // created by b2_comm_create_local (no IPC, no shm)
  bool use_vmm = false;        // arena built from VMM objects (else cudaMalloc [+ CUDA IPC])
  bool peer_is_ipc[B2_MAX_WORLD] = {};
  uint8_t* arena_of[B2_MAX_WORLD] = {};  // arena_of[r] = rank r's arena as mapped in this process
  void* arena = nullptr;       // this rank's arena: [xbar flags | pipeline flags | stage0 | stage1]
  size_t arena_bytes = 0;
  size_t stage_bytes = 0;
  vmm::Mapping own;                  // VMM backend: my physical allocation + its mapping
  vmm::Mapping peers[B2_MAX_WORLD];  // VMM backend, multi-process: imported peer allocations
  vmm::Mapping mc;                   // VMM backend, multi-process: the multicast object
  LocalMc* local_mc = nullptr;       // VMM backend, in-process world
  uint32_t* counters = nullptr;  // cudaMalloc'ed: opseq, done
  unsigned long long* trace_dev = nullptr;  // cudaMalloc'ed on demand: kMaxCtas * 8 stamps
  uint32_t* status_host = nullptr;
  // tuning (identical on every rank: they come from the same environment / the same b2_comm_set_param calls)
  int max_ctas = 0;                 // 0 = heuristic
  size_t oneshot_max_wire_bytes = 0;  // AUTO: one-shot up to this many wire bytes
  size_t pipe_min_wire_bytes = 0;     // AUTO: the pipelined kernels from this many wire bytes
  size_t nvls_min_wire_bytes = 0;     // AUTO: NVLS (when available and the mode allows it) from this many wire bytes
  int nvls_min_world = 4;             // AUTO: NVLS only pays once (1 + 1/W) < 2 (W-1)/W, i.e. W >= 4
  size_t ll_min_wire_bytes = 0;       // AUTO: the barrier-free LL two-shot from this many wire bytes (above the one-shot range) ...
  size_t ll_max_wire_bytes = 0;       // ... up to (excluding) this many
  size_t pipe_chunk_bytes = 0;        // target wire bytes of one pipeline chunk (per rank)
  uint64_t launches = 0;
  int last_algo = 0;                  // B2_ALGO_* of the most recent allreduce launch (what AUTO picked)
  ShmBlock* shm = nullptr;
  std::string shm_path;
};

namespace {

size_t env_size(const char* name, size_t dflt) {
  const char* s = getenv(name);
  if (!s || !*s) return dflt;
  char* end = nullptr;
  unsigned long long v = strtoull(s, &end, 10);
  return end == s ? dflt : static_cast<size_t>(v);
}

// Largest message (in wire bytes) for which one-shot beats two-shot, from the measured sweeps in profiles/
// (8xB200 NVSwitch): one-shot moves (W-1)x the payload per rank but needs one barrier instead of two, so the
// crossover falls quickly with W.  At W=2 both move the same bytes and one-shot wins until HBM traffic dominates.
size_t default_oneshot_max(int world) {
  if (world <= 2) return 16u << 20;
  if (world <= 4) return 2u << 20;
  return 512u << 10;
}

// What B2_ALGO_AUTO resolves to for one launch (DESIGN.md 2.6).  Pure: the same inputs give the same answer on every rank.
struct AutoPolicy {
  size_t oneshot_max, ll_min, ll_max, pipe_min, nvls_min;
  int nvls_min_world;
};

AutoPolicy default_policy(int world) {
  AutoPolicy p;
  p.oneshot_max = env_size("B2_ONESHOT_MAX_BYTES", default_oneshot_max(world));
  p.pipe_min = env_size("B2_PIPE_MIN_BYTES", ~static_cast<size_t>(0));
  p.nvls_min = env_size("B2_NVLS_MIN_BYTES", 64u << 20);
  p.nvls_min_world = static_cast<int>(env_size("B2_NVLS_MIN_WORLD", 8));
  p.ll_min = env_size("B2_LL_MIN_BYTES", world >= 3 ? 0 : ~static_cast<size_t>(0));
  p.ll_max = env_size("B2_LL_MAX_BYTES", 8u << 20);
  return p;
}

int auto_algo(const AutoPolicy& p, int world, int mode, size_t wire_bytes, bool multicast, bool fits_oneshot) {
  // fp32-wire NVLS would let the switch pick the fp32 summation order; AUTO keeps that mode on the rank-order kernels
  if (multicast && mode != B2_F32 && world >= p.nvls_min_world && wire_bytes >= p.nvls_min) return B2_ALGO_NVLS;
  if (wire_bytes <= p.oneshot_max && fits_oneshot) return B2_ALGO_ONESHOT;
  if (wire_bytes >= p.ll_min && wire_bytes < p.ll_max) return B2_ALGO_TWOSHOT_LL;
  if (wire_bytes >= p.pipe_min) return B2_ALGO_TWOSHOT_PIPE;
  return B2_ALGO_TWOSHOT;
}

// Arena layout for a given world size; fills d.*_off / d.slice_cap and arena_bytes (before backend rounding).
void layout(b2_comm* c, int world, size_t stage_bytes) {
  size_t cap = stage_bytes / (world + 1);
  cap &= ~static_cast<size_t>(255);
  c->stage_bytes = cap * (world + 1);
  c->d.slice_cap = cap;
  c->d.flag_off = 0;
  c->d.pflag_off = kXbarFlagBytes;
  c->d.stage_off[0] = kFlagRegionBytes;
  c->d.stage_off[1] = kFlagRegionBytes + c->stage_bytes;
  c->arena_bytes = kFlagRegionBytes + 2 * c->stage_bytes;
  // the sentinel-managed buffers (LL two-shot recv/out, NVLS out): 2W regions per parity
  const size_t ll_bytes = 2 * static_cast<size_t>(world) * cap;
  c->d.ll_off[0] = c->arena_bytes;
  c->d.ll_off[1] = c->arena_bytes + ll_bytes;
  c->arena_bytes += 2 * ll_bytes;
  c->d.llflag_off = 32u << 10;  // inside the xbar flag region, past its kMaxCtas slots
}

// Everything of a rank except the arena itself.
int init_rank(b2_comm* c, int rank, int world, int device, size_t stage_bytes) {
  c->device = device;
  c->d.rank = rank;
  c->d.world = world;
  if (stage_bytes == 0) stage_bytes = env_size("B2_STAGE_MB", kDefaultStageBytes >> 20) << 20;
  if (stage_bytes < (static_cast<size_t>(world + 1) << 12))
    return fail(B2_EINVAL, "stage_bytes=%zu too small for world=%d", stage_bytes, world);
  c->d.timeout_ns = env_size("B2_TIMEOUT_MS", kDefaultTimeoutNs / 1000000ull) * 1000000ull;
  layout(c, world, stage_bytes);
  c->max_ctas = static_cast<int>(env_size("B2_MAX_CTAS", 0));
  // AUTO thresholds from the measured sweeps (profiles/r02_sweep_w8.md, r02_pipeline_and_ll_w2.md), in wire bytes:
  //   one-shot            up to default_oneshot_max(world)
  //   LL two-shot         from there to 8 MiB at W >= 3 (2-16 MiB fp32 buckets at W=8: 5-9 % ahead of the single-pass kernel;
  //                       at W=2 one-shot covers that range and LL loses above it: off)
  //   single-pass two-shot  above that (the DDP 25 MiB buckets: equal in isolation, and the kernel with no extra local
  //                       traffic when backward competes for HBM inside the training step)
  //   NVLS                from 64 MiB at W = 8 (128 MiB-1 GiB fp32: 245 / 336 / 1281 us against 268 / 397 / 1542 us two-shot and
  //                       357 / 394 / 1330 us ncclAllReduce); the switch's arithmetic, bit-identical to NCCL's NVLS (DESIGN.md 2.4)
  //   pipelined two-shot  never (explicit choice only)
  const AutoPolicy pol = default_policy(world);
  c->oneshot_max_wire_bytes = pol.oneshot_max;
  c->pipe_min_wire_bytes = pol.pipe_min;
  c->nvls_min_wire_bytes = pol.nvls_min;
  c->nvls_min_world = pol.nvls_min_world;
  c->ll_min_wire_bytes = pol.ll_min;
  c->ll_max_wire_bytes = pol.ll_max;
  c->pipe_chunk_bytes = env_size("B2_PIPE_CHUNK_KB", 2048) << 10;
  B2_CUDA(cudaSetDevice(device));
  B2_CUDA(cudaMalloc(&c->counters, 256));
  B2_CUDA(cudaMemset(c->counters, 0, 256));
  c->d.opseq = c->counters;
  c->d.done = c->counters + 32;  // a different 128 B line
  B2_CUDA(cudaHostAlloc(&c->status_host, 64, cudaHostAllocMapped | cudaHostAllocPortable));
  memset(c->status_host, 0, 64);
  void* sdev = nullptr;
  B2_CUDA(cudaHostGetDevicePointer(&sdev, c->status_host, 0));
  c->d.status = static_cast<uint32_t*>(sdev);
  return B2_OK;
}

// This rank's arena.  VMM backend: a shareable physical allocation mapped for `devices` (the rank's own device in the
// one-process-per-GPU case, every device of the world for an in-process world).  Legacy backend: cudaMalloc.
int alloc_arena(b2_comm* c, bool use_vmm, bool multicast, const int* devices, int ndev) {
  B2_CUDA(cudaSetDevice(c->device));
  c->use_vmm = use_vmm;
  if (use_vmm) {
    const size_t gran = vmm::arena_granularity(c->device, c->d.world, multicast);
    c->arena_bytes = (c->arena_bytes + gran - 1) / gran * gran;
    const CUmemAllocationProp prop = vmm::alloc_prop(c->device);
    const CUresult r = vmm::driver().MemCreate(&c->own.handle, c->arena_bytes, &prop, 0);
    if (r != CUDA_SUCCESS) return fail(B2_ECUDA, "cuMemCreate(%zu bytes): %s", c->arena_bytes, vmm::errstr(r).c_str());
    const std::string e = vmm::map_handle(&c->own, c->arena_bytes, gran, devices, ndev);
    if (!e.empty()) return fail(B2_ECUDA, "mapping this rank's arena: %s", e.c_str());
    c->arena = reinterpret_cast<void*>(c->own.va);
  } else {
    B2_CUDA(cudaMalloc(&c->arena, c->arena_bytes));
  }
  B2_CUDA(cudaMemset(c->arena, 0, kFlagRegionBytes));
  B2_CUDA(cudaMemset(static_cast<uint8_t*>(c->arena) + c->d.ll_off[0], 0xFF, 4 * static_cast<size_t>(c->d.world) * c->d.slice_cap));
  B2_CUDA(cudaDeviceSynchronize());
  c->arena_of[c->d.rank] = static_cast<uint8_t*>(c->arena);
  return B2_OK;
}

void rotate_peers(b2_comm* c) {
  for (int jj = 0; jj < c->d.world; ++jj) c->d.peer[jj] = c->arena_of[(c->d.rank + jj) % c->d.world];
}

void free_rank_resources(b2_comm* c) {
  if (c->device >= 0) cudaSetDevice(c->device);
  if (c->use_vmm) {
    if (c->local_mc && --c->local_mc->refs == 0) {
      vmm::unmap_release(&c->local_mc->map);
      delete c->local_mc;
    }
    c->local_mc = nullptr;
    vmm::unmap_release(&c->mc);
    for (int r = 0; r < B2_MAX_WORLD; ++r) vmm::unmap_release(&c->peers[r]);
    vmm::unmap_release(&c->own);
  } else if (c->arena) {
    cudaFree(c->arena);
  }
  if (c->counters) cudaFree(c->counters);
  if (c->trace_dev) cudaFree(c->trace_dev);
  c->trace_dev = nullptr;
  if (c->status_host) cudaFreeHost(c->status_host);
  c->arena = nullptr;
  c->counters = nullptr;
  c->status_host = nullptr;
}

int grid_for(const b2_comm* c, unsigned long long vecs_per_cta_dim, int unroll) {
  // Enough CTAs that each thread has work, capped so the collective leaves SMs to the backward
  // pass it overlaps with.  Deterministic in (n, world, max_ctas) => identical on every rank.
  // Default cap: 64 CTAs; 128 once 64 CTAs would each loop more than twice (from ~16 MiB fp32 buckets at W=8), where the
  // sweeps in profiles/r01_sweep_w*.jsonl show the 128-CTA grid 3-6 % faster.  One CTA per SM (512 threads, <= 128 regs).
  const int dflt = vecs_per_cta_dim > 64ull * kThreads * static_cast<unsigned long long>(unroll) * 2ull ? 128 : 64;
  const int cap = c->max_ctas > 0 ? (c->max_ctas > kMaxCtas ? kMaxCtas : c->max_ctas) : dflt;
  unsigned long long per = static_cast<unsigned long long>(kThreads) * unroll;
  unsigned long long g = (vecs_per_cta_dim + per - 1) / per;
  if (g < 1) g = 1;
  if (g > static_cast<unsigned long long>(cap)) g = cap;
  return static_cast<int>(g);
}

int unroll_for_world(int w) { return w >= 5 ? 1 : (w >= 3 ? 2 : (w >= 2 ? 4 : 8)); }

// Pipelined kernels: grid g, K chunks, cell = vecs of one (chunk, CTA) cell of a slice (multiple of 32, so every warp
// access is a whole 512 B line group).  Deterministic in (Ls, wire bytes, tuning) => identical on every rank.
struct PipePlan {
  int grid;
  int K;
  unsigned long long cell;
};

PipePlan plan_pipe(const b2_comm* c, unsigned long long Ls, size_t wire_bytes) {
  const unsigned long long units = (Ls + 31) / 32;  // 32-vec units in a slice
  const int cap = c->max_ctas > 0 ? (c->max_ctas > kMaxCtas ? kMaxCtas : c->max_ctas)
                                  : (wire_bytes >= (8u << 20) ? 128 : 64);
  unsigned long long g = units < static_cast<unsigned long long>(cap) ? units : cap;
  if (g < 1) g = 1;
  unsigned long long K = c->pipe_chunk_bytes ? (wire_bytes + c->pipe_chunk_bytes / 2) / c->pipe_chunk_bytes : 1;
  if (K < 1) K = 1;
  if (K > static_cast<unsigned long long>(kMaxChunks)) K = kMaxChunks;
  const unsigned long long per_cta_units = (units + g - 1) / g;
  if (K > per_cta_units) K = per_cta_units;
  const unsigned long long cell_units = (units + g * K - 1) / (g * K);
  PipePlan p;
  p.grid = static_cast<int>(g);
  p.K = static_cast<int>(K);
  p.cell = cell_units * 32;
  return p;
}

template <int MODE, int W>
cudaError_t launch_oneshot(const CommDev& d, const Src& src, int grid, void* buf, unsigned long long n, float scale,
                           cudaStream_t s) {
  k_oneshot<MODE, W><<<grid, kThreads, 0, s>>>(d, src, buf, n, scale);
  return cudaGetLastError();
}
template <int MODE, int W>
cudaError_t launch_twoshot(const CommDev& d, const Src& src, int grid, void* buf, unsigned long long n, float scale,
                           cudaStream_t s) {
  k_twoshot<MODE, W><<<grid, kThreads, 0, s>>>(d, src, buf, n, scale);
  return cudaGetLastError();
}
template <int MODE, int W>
cudaError_t launch_ll(const CommDev& d, const Src& src, int grid, void* buf, unsigned long long n, float scale, cudaStream_t s) {
  k_ll<MODE, W><<<grid, kThreads, 0, s>>>(d, src, buf, n, scale);
  return cudaGetLastError();
}
template <int MODE, int W, int ALG>
cudaError_t launch_pipe(const CommDev& d, const Src& src, const PipePlan& p, void* buf, unsigned long long n, float scale,
                        cudaStream_t s) {
  k_pipe<MODE, W, ALG><<<p.grid, kThreads, 0, s>>>(d, src, buf, n, scale, p.K, p.cell);
  return cudaGetLastError();
}

// kind: one of B2_ALGO_ONESHOT / TWOSHOT / TWOSHOT_PIPE / NVLS
template <int MODE>
cudaError_t launch_by_world(const CommDev& d, const Src& src, int kind, int grid, const PipePlan& p, void* buf,
                            unsigned long long n, float scale, cudaStream_t s) {
#define B2_CASE(Wv)                                                                                  \
  case Wv:                                                                                           \
    switch (kind) {                                                                                  \
      case B2_ALGO_ONESHOT:                                                                          \
        return launch_oneshot<MODE, Wv>(d, src, grid, buf, n, scale, s);                                  \
      case B2_ALGO_TWOSHOT:                                                                          \
        return launch_twoshot<MODE, Wv>(d, src, grid, buf, n, scale, s);                                  \
      case B2_ALGO_TWOSHOT_PIPE:                                                                     \
        return launch_pipe<MODE, Wv, pl::kP2p>(d, src, p, buf, n, scale, s);                            \
      case B2_ALGO_TWOSHOT_LL:                                                                       \
        return launch_ll<MODE, Wv>(d, src, grid, buf, n, scale, s);                                  \
      default:                                                                                       \
        return launch_pipe<MODE, Wv, pl::kNvls>(d, src, p, buf, n, scale, s);                           \
    }
  switch (d.world) {
    B2_CASE(2)
    B2_CASE(3)
    B2_CASE(4)
    B2_CASE(5)
    B2_CASE(6)
    B2_CASE(7)
    B2_CASE(8)
    default:
      return cudaErrorInvalidValue;
  }
#undef B2_CASE
}

template <int MODE>
cudaError_t launch_local(const Src& src, void* buf, unsigned long long n, float scale, cudaStream_t s) {
  // TMA-staged path for 16 B-aligned buckets.  Measured on B200 (profiles/r01_local_pass_tma_vs_plain.jsonl): the ring
  // needs several tiles per CTA to pay for its prologue - slower than the plain kernel below 25 MiB, equal to 168 MiB,
  // ahead from 512 MiB - so it is the default from 256 MiB up.  B2_LOCAL_TMA_MIN_MB moves the threshold (0 = always
  // for >= 1 MiB, e.g. for the parity tests), B2_LOCAL_TMA=0 disables it.
  static const bool use_tma = env_size("B2_LOCAL_TMA", 1) != 0;
  static const unsigned long long tma_min = env_size("B2_LOCAL_TMA_MIN_MB", 256) << 20;
  const unsigned long long nbytes = n * (MODE == B2_BF16 ? 2 : 4);
  if (use_tma && src.nseg == 0 && (reinterpret_cast<uintptr_t>(buf) & 15u) == 0 && nbytes >= (1ull << 20) && nbytes >= tma_min) {
    const unsigned long long ntiles = nbytes / tma::kTileBytes;
    unsigned long long g = ntiles < 148ull * 2 ? ntiles : 148ull * 2;  // persistent: 2 CTAs (2 x 64 KiB rings) per SM
    constexpr int kSmem = tma::kStages * tma::kTileBytes;
    static std::atomic<unsigned> configured{0};  // bit d: the 64 KiB opt-in has been set on device d
    int devno = 0;
    cudaGetDevice(&devno);
    if (!(configured.load(std::memory_order_relaxed) & (1u << (devno & 31)))) {
      const cudaError_t attr = cudaFuncSetAttribute(k_local_pass_tma<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
      if (attr != cudaSuccess) return attr;
      configured.fetch_or(1u << (devno & 31), std::memory_order_relaxed);
    }
    k_local_pass_tma<MODE><<<static_cast<int>(g), tma::kTmaThreads, kSmem, s>>>(buf, n, scale);
    return cudaGetLastError();
  }
  const unsigned long long V = (n + 7) / 8;
  unsigned long long g = (V + kThreads * 4ull - 1) / (kThreads * 4ull);
  if (g < 1) g = 1;
  if (g > 148ull * 4) g = 148ull * 4;  // 4 resident CTAs per SM keep ~64 KiB of loads in flight per SM
  k_local_pass<MODE><<<static_cast<int>(g), kThreads, 0, s>>>(src, buf, n, scale);
  return cudaGetLastError();
}

cudaError_t launch_mode(const CommDev& d, const Src& src, int mode, int kind, int grid, const PipePlan& p, void* buf,
                        unsigned long long n, float scale, cudaStream_t s) {
  switch (mode) {
    case B2_F32_WIRE_BF16:
      return launch_by_world<B2_F32_WIRE_BF16>(d, src, kind, grid, p, buf, n, scale, s);
    case B2_F32:
      return launch_by_world<B2_F32>(d, src, kind, grid, p, buf, n, scale, s);
    default:
      return launch_by_world<B2_BF16>(d, src, kind, grid, p, buf, n, scale, s);
  }
}

const Src kNoSrc = {};  // nseg == 0: the collective reads the bucket itself

int local_pass_impl(const Src& src, void* buf, size_t n_elems, int mode, float scale, int device, void* stream) {
  if (n_elems == 0) return B2_OK;
  if (!buf) return fail(B2_EINVAL, "b2_local_pass: null buffer");
  DeviceGuard g(device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t e;
  switch (mode) {
    case B2_F32_WIRE_BF16:
      e = launch_local<B2_F32_WIRE_BF16>(src, buf, n_elems, scale, s);
      break;
    case B2_F32:
      e = launch_local<B2_F32>(src, buf, n_elems, scale, s);
      break;
    case B2_BF16:
      e = launch_local<B2_BF16>(src, buf, n_elems, scale, s);
      break;
    default:
      return fail(B2_EINVAL, "unknown mode %d", mode);
  }
  if (e != cudaSuccess) return fail(B2_ECUDA, "k_local_pass launch: %s", cudaGetErrorString(e));
  return B2_OK;
}

size_t elem_bytes(int mode) { return mode == B2_BF16 ? 2 : 4; }
size_t wire_vec_bytes(int mode) { return mode == B2_F32 ? 32 : 16; }

unsigned next_creation_index(const char* shm_name, uint64_t epoch) {
  static std::mutex mu;
  static std::map<std::string, unsigned> seen;
  std::lock_guard<std::mutex> lock(mu);
  return seen[std::string(shm_name) + "#" + std::to_string(epoch)]++;
}

bool wait_count(std::atomic<int>& ctr, int target, std::atomic<int>* abort_flag, double deadline) {
  while (ctr.load(std::memory_order_acquire) < target) {
    if (abort_flag && abort_flag->load(std::memory_order_acquire)) return false;
    if (now_s() > deadline) return false;
    usleep(200);
  }
  return true;
}

// Multi-process multicast bring-up (after every rank has mapped every peer arena).  Any failure on any rank sets
// sb->mc_fail and every rank drops the NVLS path together; the P2P mappings are unaffected.
void setup_multicast(b2_comm* c, int sock, const std::string& sock_base, int stash_mc_fd, double deadline) {
  ShmBlock* sb = c->shm;
  const int W = c->d.world, rank = c->d.rank;
  const vmm::Driver& drv = vmm::driver();
  std::string why;
  int mc_fd = stash_mc_fd;
  bool ok = true;
  if (rank == 0) {
    const CUmulticastObjectProp mp = vmm::mc_prop(W, c->arena_bytes);
    CUresult r = drv.MulticastCreate(&c->mc.handle, &mp);
    if (r != CUDA_SUCCESS) {
      why = "cuMulticastCreate: " + vmm::errstr(r);
      ok = false;
    }
    int fd = -1;
    if (ok) {
      r = drv.MemExportToShareableHandle(&fd, c->mc.handle, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0);
      if (r != CUDA_SUCCESS) {
        why = "export of the multicast object: " + vmm::errstr(r);
        ok = false;
      }
    }
    for (int p = 1; p < W && ok; ++p) ok = vmm::send_fd(sock, sock_base, p, fd, vmm::FdMsg{0, 1}, &why);
    if (fd >= 0) close(fd);
  } else {
    while (mc_fd < 0 && ok) {
      if (sb->mc_fail.load(std::memory_order_acquire) || now_s() > deadline) {
        ok = false;
        why = "rank 0 could not create the multicast object";
        break;
      }
      vmm::FdMsg msg{};
      std::string w2;
      const int fd = vmm::recv_fd(sock, &msg, 100, &w2);
      if (fd >= 0 && msg.kind == 1) mc_fd = fd;
      else if (fd >= 0) close(fd);
    }
    if (ok) {
      const CUresult r = drv.MemImportFromShareableHandle(&c->mc.handle, reinterpret_cast<void*>(static_cast<uintptr_t>(mc_fd)),
                                                          CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR);
      if (r != CUDA_SUCCESS) {
        why = "import of the multicast object: " + vmm::errstr(r);
        ok = false;
      }
    }
    if (mc_fd >= 0) close(mc_fd);
  }
  CUdevice cudev = 0;
  if (ok && drv.DeviceGet(&cudev, c->device) != CUDA_SUCCESS) ok = false;
  if (ok) {
    const CUresult r = drv.MulticastAddDevice(c->mc.handle, cudev);
    if (r != CUDA_SUCCESS) {
      why = "cuMulticastAddDevice: " + vmm::errstr(r);
      ok = false;
    }
  }
  if (!ok) sb->mc_fail.store(1, std::memory_order_release);
  sb->mc_added.fetch_add(1, std::memory_order_acq_rel);
  ok = wait_count(sb->mc_added, W, nullptr, deadline) && !sb->mc_fail.load(std::memory_order_acquire) && ok;
  if (ok) {  // every device is in the team: binding cannot block
    const CUresult r = drv.MulticastBindMem(c->mc.handle, 0, c->own.handle, 0, c->arena_bytes, 0);
    if (r != CUDA_SUCCESS) {
      why = "cuMulticastBindMem: " + vmm::errstr(r);
      ok = false;
      sb->mc_fail.store(1, std::memory_order_release);
    }
  }
  sb->mc_bound.fetch_add(1, std::memory_order_acq_rel);
  ok = wait_count(sb->mc_bound, W, nullptr, deadline) && !sb->mc_fail.load(std::memory_order_acquire) && ok;
  if (ok) {
    const size_t gran = vmm::arena_granularity(c->device, W, true);
    const std::string e = vmm::map_handle(&c->mc, c->arena_bytes, gran, &c->device, 1);
    if (!e.empty()) {
      why = "mapping the multicast object: " + e;
      ok = false;
      sb->mc_fail.store(1, std::memory_order_release);
    }
  }
  sb->mc_mapped.fetch_add(1, std::memory_order_acq_rel);
  ok = wait_count(sb->mc_mapped, W, nullptr, deadline) && !sb->mc_fail.load(std::memory_order_acquire) && ok;
  if (ok) {
    c->d.mc = reinterpret_cast<uint8_t*>(c->mc.va);
  } else {
    vmm::unmap_release(&c->mc);
    c->d.mc = nullptr;
    if (!why.empty() && env_size("B2_VERBOSE", 0)) fprintf(stderr, "[b200ddp] rank %d: NVLS disabled: %s\n", rank, why.c_str());
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int b2_version(void) { return B2_ABI_VERSION; }

const char* b2_last_error(void) { return g_err.c_str(); }

int b2_comm_create_local(b2_comm_t** out, int world, const int* devices, size_t stage_bytes) {
  if (!out || !devices || world < 1 || world > B2_MAX_WORLD)
    return fail(B2_EINVAL, "b2_comm_create_local: bad arguments (world=%d)", world);
  int prev = -1;
  cudaGetDevice(&prev);
  b2_comm* cs[B2_MAX_WORLD] = {};
  int rc = B2_OK;
  // distinct devices -> VMM arenas visible to every device of the world (+ one multicast object); repeated devices
  // (all ranks on one GPU, the single-GPU parity topology) -> plain cudaMalloc, no multicast
  bool distinct = world > 1;
  for (int a = 0; a < world; ++a)
    for (int b = a + 1; b < world; ++b)
      if (devices[a] == devices[b]) distinct = false;
  bool use_vmm = distinct && env_size("B2_VMM", 1) != 0;
  bool use_mc = use_vmm && env_size("B2_NVLS", 1) != 0;
  for (int r = 0; r < world && use_vmm; ++r) {
    const vmm::Caps cp = vmm::caps(devices[r]);
    use_vmm = use_vmm && cp.vmm;
    use_mc = use_mc && cp.multicast;
  }
  use_mc = use_mc && use_vmm;
  for (int r = 0; r < world && rc == B2_OK; ++r) {
    cs[r] = new (std::nothrow) b2_comm();
    if (!cs[r]) {
      rc = fail(B2_ESYS, "out of host memory");
      break;
    }
    cs[r]->local_world = true;
    rc = init_rank(cs[r], r, world, devices[r], stage_bytes);
  }
  for (int a = 0; a < world && rc == B2_OK; ++a) {
    for (int b = 0; b < world && rc == B2_OK; ++b) {
      if (devices[a] == devices[b]) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, devices[a], devices[b]);
      if (!can) {
        rc = fail(B2_ENOPEER, "device %d cannot access device %d over P2P", devices[a], devices[b]);
        break;
      }
      cudaSetDevice(devices[a]);
      cudaError_t e = cudaDeviceEnablePeerAccess(devices[b], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
      } else if (e != cudaSuccess) {
        rc = fail(B2_ECUDA, "cudaDeviceEnablePeerAccess(%d->%d): %s", devices[a], devices[b],
                  cudaGetErrorString(e));
      }
    }
  }
  for (int r = 0; r < world && rc == B2_OK; ++r) rc = alloc_arena(cs[r], use_vmm, use_mc, devices, use_vmm ? world : 1);
  if (rc == B2_OK && use_mc) {
    // one multicast object over the W allocations, mapped once for all devices of the world
    const vmm::Driver& drv = vmm::driver();
    LocalMc* lm = new (std::nothrow) LocalMc();
    bool ok = lm != nullptr;
    if (ok) {
      const CUmulticastObjectProp mp = vmm::mc_prop(world, cs[0]->arena_bytes);
      ok = drv.MulticastCreate(&lm->map.handle, &mp) == CUDA_SUCCESS;
      for (int r = 0; r < world && ok; ++r) {
        CUdevice dv;
        ok = drv.DeviceGet(&dv, devices[r]) == CUDA_SUCCESS && drv.MulticastAddDevice(lm->map.handle, dv) == CUDA_SUCCESS;
      }
      for (int r = 0; r < world && ok; ++r)
        ok = drv.MulticastBindMem(lm->map.handle, 0, cs[r]->own.handle, 0, cs[r]->arena_bytes, 0) == CUDA_SUCCESS;
      if (ok) ok = vmm::map_handle(&lm->map, cs[0]->arena_bytes, vmm::arena_granularity(devices[0], world, true), devices, world).empty();
      if (ok) {
        lm->refs = world;
        for (int r = 0; r < world; ++r) {
          cs[r]->local_mc = lm;
          cs[r]->d.mc = reinterpret_cast<uint8_t*>(lm->map.va);
        }
      } else {
        vmm::unmap_release(&lm->map);
        delete lm;
      }
    }
  }
  if (rc == B2_OK) {
    for (int a = 0; a < world; ++a)
      for (int b = 0; b < world; ++b) cs[a]->arena_of[b] = static_cast<uint8_t*>(cs[b]->arena);
    for (int r = 0; r < world; ++r) {
      rotate_peers(cs[r]);
      out[r] = cs[r];
    }
  } else {
    std::string keep = g_err;
    for (int r = 0; r < world; ++r)
      if (cs[r]) {
        free_rank_resources(cs[r]);
        delete cs[r];
      }
    g_err = keep;
  }
  if (prev >= 0) cudaSetDevice(prev);
  return rc;
}

int b2_comm_create(b2_comm_t** out, int rank, int world, int device, const char* shm_name,
                   uint64_t epoch, size_t stage_bytes, int timeout_ms) {
  if (!out || world < 1 || world > B2_MAX_WORLD || rank < 0 || rank >= world || device < 0)
    return fail(B2_EINVAL, "b2_comm_create: bad arguments (rank=%d world=%d device=%d)", rank, world,
                device);
  if (world > 1 && (!shm_name || !*shm_name))
    return fail(B2_EINVAL, "b2_comm_create: shm_name is required when world > 1");
  const double deadline = now_s() + (timeout_ms > 0 ? timeout_ms : 120000) * 1e-3;
  int prev = -1;
  cudaGetDevice(&prev);
  b2_comm* c = new (std::nothrow) b2_comm();
  if (!c) return fail(B2_ESYS, "out of host memory");
  int rc = init_rank(c, rank, world, device, stage_bytes);
  int sock = -1;
  std::string sock_base;
  if (rc == B2_OK && world == 1) rc = alloc_arena(c, false, false, &device, 1);
  if (rc == B2_OK && world > 1) {
    // <name>.e<epoch>.c<n>: n counts this process's communicators on (name, epoch).  Every rank creates its
    // communicators in the same order, so n agrees across ranks, and a second communicator (init_pg + DDP, two DDP
    // modules) can never open the control block of the first one while rank 0 has not unlinked it yet.
    char path[256];
    snprintf(path, sizeof(path), "%s%s.e%llu.c%u", shm_name[0] == '/' ? "" : "/", shm_name,
             static_cast<unsigned long long>(epoch), next_creation_index(shm_name, epoch));
    c->shm_path = path;
    sock_base = std::string("b2fd") + path;
    int fd = shm_open(path, O_CREAT | O_RDWR, 0600);
    if (fd < 0) rc = fail(B2_ESYS, "shm_open(%s): %s", path, strerror(errno));
    if (rc == B2_OK && ftruncate(fd, sizeof(ShmBlock)) != 0)
      rc = fail(B2_ESYS, "ftruncate(%s): %s", path, strerror(errno));
    if (rc == B2_OK) {
      void* m = mmap(nullptr, sizeof(ShmBlock), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
      if (m == MAP_FAILED)
        rc = fail(B2_ESYS, "mmap(%s): %s", path, strerror(errno));
      else
        c->shm = static_cast<ShmBlock*>(m);
    }
    if (fd >= 0) close(fd);
  }
  if (rc == B2_OK && world > 1) {
    ShmBlock* sb = c->shm;
    ShmSlot& me = sb->slot[rank];
    // ---- 1. agree on the backend before anybody allocates -------------------------------------------------
    vmm::Caps cp;
    if (env_size("B2_VMM", 1) != 0) cp = vmm::caps(device);
    if (cp.vmm) {
      std::string why;
      sock = vmm::sock_open(sock_base, rank, &why);
      if (sock < 0) cp = vmm::Caps();  // no way to pass file descriptors: stay on CUDA IPC
    }
    if (env_size("B2_NVLS", 1) == 0) cp.multicast = false;
    me.cap_vmm = cp.vmm ? 1 : 0;
    me.cap_mc = cp.multicast ? 1 : 0;
    me.device = device;
    memset(me.bus_id, 0, sizeof(me.bus_id));
    cudaDeviceGetPCIBusId(me.bus_id, sizeof(me.bus_id), device);
    if (rank == 0) {
      sb->epoch = epoch;
      sb->world = world;
      sb->magic.store(kShmMagic, std::memory_order_release);
    }
    me.hello.store(1, std::memory_order_release);
    bool use_vmm = true, use_mc = true;
    for (int r = 0; r < world && rc == B2_OK; ++r) {
      while (sb->slot[r].hello.load(std::memory_order_acquire) != 1) {
        if (now_s() > deadline) {
          rc = fail(B2_ETIMEOUT, "rendezvous timed out waiting for rank %d on %s", r, c->shm_path.c_str());
          break;
        }
        usleep(200);
      }
      use_vmm = use_vmm && sb->slot[r].cap_vmm != 0;
      use_mc = use_mc && sb->slot[r].cap_mc != 0;
    }
    // a multicast team is a set of DISTINCT devices: ranks sharing a GPU (functional tests) stay on the P2P kernels
    for (int a = 0; a < world && rc == B2_OK; ++a)
      for (int b = a + 1; b < world; ++b)
        if (strncmp(sb->slot[a].bus_id, sb->slot[b].bus_id, sizeof(sb->slot[a].bus_id)) == 0) use_mc = false;
    use_mc = use_mc && use_vmm;
    // ---- 2. allocate and publish ---------------------------------------------------------------------------
    if (rc == B2_OK) rc = alloc_arena(c, use_vmm, use_mc, &device, 1);
    if (rc == B2_OK) {
      if (!use_vmm) {
        cudaError_t e = cudaIpcGetMemHandle(&me.handle, c->arena);
        if (e != cudaSuccess) rc = fail(B2_ECUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
      }
      me.pid = static_cast<int>(getpid());
      me.arena_bytes = c->arena_bytes;
      if (rc == B2_OK) me.ready.store(1, std::memory_order_release);
    }
    for (int r = 0; r < world && rc == B2_OK; ++r) {
      while (sb->slot[r].ready.load(std::memory_order_acquire) != 1) {
        if (now_s() > deadline) {
          rc = fail(B2_ETIMEOUT, "rendezvous timed out waiting for rank %d on %s", r, c->shm_path.c_str());
          break;
        }
        usleep(200);
      }
    }
    // ---- 3. map every peer's arena -------------------------------------------------------------------------
    int stash_mc_fd = -1;
    for (int r = 0; r < world && rc == B2_OK; ++r) {
      if (r == rank) continue;
      const ShmSlot& ps = sb->slot[r];
      if (ps.arena_bytes != c->arena_bytes) {
        rc = fail(B2_EINVAL, "rank %d uses arena_bytes=%llu, this rank %zu (stage size must match)", r,
                  ps.arena_bytes, c->arena_bytes);
        break;
      }
      // Resolve the peer's GPU in THIS process's numbering by bus id.  If it is not visible here (each "node" of a
      // multi-node-on-one-box job gets its own CUDA_VISIBLE_DEVICES) the P2P query is impossible, but an IPC / imported
      // mapping of an invisible peer's memory can still be opened, so we just try.
      int peer_local = -1;
      if (cudaDeviceGetByPCIBusId(&peer_local, ps.bus_id) != cudaSuccess) {
        cudaGetLastError();
        peer_local = -1;
      }
      if (peer_local >= 0 && peer_local != device) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, device, peer_local);
        if (!can) {
          rc = fail(B2_ENOPEER, "device %d cannot access rank %d's device %s over P2P", device, r, ps.bus_id);
          break;
        }
      }
      if (!use_vmm) {
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, ps.handle, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
          rc = fail(B2_ECUDA, "cudaIpcOpenMemHandle(rank %d, device %d): %s", r, ps.device,
                    cudaGetErrorString(e));
          break;
        }
        c->arena_of[r] = static_cast<uint8_t*>(p);
        c->peer_is_ipc[r] = true;
      }
    }
    if (rc == B2_OK && use_vmm) {
      const vmm::Driver& drv = vmm::driver();
      std::string why;
      int fd = -1;
      CUresult r0 = drv.MemExportToShareableHandle(&fd, c->own.handle, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0);
      if (r0 != CUDA_SUCCESS) rc = fail(B2_ECUDA, "cuMemExportToShareableHandle: %s", vmm::errstr(r0).c_str());
      for (int p = 0; p < world && rc == B2_OK; ++p) {
        if (p == rank) continue;
        if (!vmm::send_fd(sock, sock_base, p, fd, vmm::FdMsg{rank, 0}, &why)) rc = fail(B2_ESYS, "%s", why.c_str());
      }
      if (fd >= 0) close(fd);
      int got = 0;
      const size_t gran = vmm::arena_granularity(device, world, use_mc);
      while (rc == B2_OK && got < world - 1) {
        if (now_s() > deadline) {
          rc = fail(B2_ETIMEOUT, "rendezvous timed out receiving peer arenas (%d/%d)", got, world - 1);
          break;
        }
        vmm::FdMsg msg{};
        const int pfd = vmm::recv_fd(sock, &msg, 200, &why);
        if (pfd < 0) continue;
        if (msg.kind == 1) {  // rank 0 is already at the multicast step
          stash_mc_fd = pfd;
          continue;
        }
        if (msg.src_rank < 0 || msg.src_rank >= world || msg.src_rank == rank || c->peers[msg.src_rank].handle) {
          close(pfd);
          continue;
        }
        vmm::Mapping& pm = c->peers[msg.src_rank];
        CUresult r1 = drv.MemImportFromShareableHandle(&pm.handle, reinterpret_cast<void*>(static_cast<uintptr_t>(pfd)),
                                                       CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR);
        close(pfd);
        if (r1 != CUDA_SUCCESS) {
          rc = fail(B2_ECUDA, "cuMemImportFromShareableHandle(rank %d): %s", msg.src_rank, vmm::errstr(r1).c_str());
          break;
        }
        const std::string e = vmm::map_handle(&pm, c->arena_bytes, gran, &device, 1);
        if (!e.empty()) {
          rc = fail(B2_ECUDA, "mapping rank %d's arena: %s", msg.src_rank, e.c_str());
          break;
        }
        c->arena_of[msg.src_rank] = reinterpret_cast<uint8_t*>(pm.va);
        ++got;
      }
    }
    if (rc == B2_OK) {
      sb->mapped.fetch_add(1, std::memory_order_acq_rel);
      if (!wait_count(sb->mapped, world, nullptr, deadline))
        rc = fail(B2_ETIMEOUT, "rendezvous timed out waiting for peers to map (%d/%d)", sb->mapped.load(), world);
    }
    // ---- 4. NVLS: one multicast object over all arenas -----------------------------------------------------
    if (rc == B2_OK && use_mc) setup_multicast(c, sock, sock_base, stash_mc_fd, deadline);
    else if (stash_mc_fd >= 0) close(stash_mc_fd);
    // everyone holds its mappings now: the name can go (the memory lives until the last munmap)
    if (rc == B2_OK && rank == 0) shm_unlink(c->shm_path.c_str());
  }
  if (sock >= 0) close(sock);
  if (rc != B2_OK) {
    std::string keep = g_err;
    for (int r = 0; r < world; ++r)
      if (c->peer_is_ipc[r]) cudaIpcCloseMemHandle(c->arena_of[r]);
    if (c->shm) munmap(c->shm, sizeof(ShmBlock));
    if (rank == 0 && !c->shm_path.empty()) shm_unlink(c->shm_path.c_str());
    free_rank_resources(c);
    delete c;
    g_err = keep;
  } else {
    rotate_peers(c);
    *out = c;
  }
  if (prev >= 0) cudaSetDevice(prev);
  return rc;
}

int b2_comm_destroy(b2_comm_t* c) {
  if (!c) return B2_OK;
  int prev = -1;
  cudaGetDevice(&prev);
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  if (c->shm) {
    // nobody frees its arena while a peer may still have kernels reading it
    ShmBlock* sb = c->shm;
    sb->departed.fetch_add(1, std::memory_order_acq_rel);
    const double deadline = now_s() + 10.0;
    while (sb->departed.load(std::memory_order_acquire) < c->d.world && now_s() < deadline) usleep(200);
    for (int r = 0; r < c->d.world; ++r)
      if (c->peer_is_ipc[r]) cudaIpcCloseMemHandle(c->arena_of[r]);
    munmap(c->shm, sizeof(ShmBlock));
  }
  free_rank_resources(c);
  delete c;
  if (prev >= 0) cudaSetDevice(prev);
  return B2_OK;
}

int b2_comm_rank(const b2_comm_t* c) { return c ? c->d.rank : B2_EINVAL; }
int b2_comm_world(const b2_comm_t* c) { return c ? c->d.world : B2_EINVAL; }
int b2_comm_device(const b2_comm_t* c) { return c ? c->device : B2_EINVAL; }

int b2_comm_caps(const b2_comm_t* c) {
  if (!c) return B2_EINVAL;
  return (c->use_vmm ? B2_CAP_VMM : 0) | (c->d.mc != nullptr ? B2_CAP_MULTICAST : 0);
}

int b2_comm_set_timeout_ms(b2_comm_t* c, int timeout_ms) {
  if (!c || timeout_ms <= 0) return fail(B2_EINVAL, "b2_comm_set_timeout_ms: bad arguments");
  c->d.timeout_ns = static_cast<unsigned long long>(timeout_ms) * 1000000ull;
  return B2_OK;
}

int b2_comm_set_max_ctas(b2_comm_t* c, int max_ctas) {
  if (!c || max_ctas < 0) return fail(B2_EINVAL, "b2_comm_set_max_ctas: bad arguments");
  c->max_ctas = max_ctas;
  return B2_OK;
}

int b2_comm_set_param(b2_comm_t* c, const char* name, long long value) {
  if (!c || !name || value < 0) return fail(B2_EINVAL, "b2_comm_set_param: bad arguments");
  const std::string k(name);
  if (k == "oneshot_max_bytes") c->oneshot_max_wire_bytes = static_cast<size_t>(value);
  else if (k == "pipe_min_bytes") c->pipe_min_wire_bytes = static_cast<size_t>(value);
  else if (k == "nvls_min_bytes") c->nvls_min_wire_bytes = static_cast<size_t>(value);
  else if (k == "nvls_min_world") c->nvls_min_world = static_cast<int>(value);
  else if (k == "ll_min_bytes") c->ll_min_wire_bytes = static_cast<size_t>(value);
  else if (k == "ll_max_bytes") c->ll_max_wire_bytes = static_cast<size_t>(value);
  else if (k == "pipe_chunk_bytes") c->pipe_chunk_bytes = static_cast<size_t>(value);
  else if (k == "max_ctas") c->max_ctas = static_cast<int>(value);
  else return fail(B2_EINVAL, "b2_comm_set_param: unknown parameter '%s'", name);
  return B2_OK;
}

int b2_comm_status(const b2_comm_t* c) {
  if (!c) return fail(B2_EINVAL, "null communicator");
  const uint32_t s = *reinterpret_cast<volatile uint32_t*>(c->status_host);
  if (s == 0) return B2_OK;
  return fail(-static_cast<int>(s), "rank %d: a kernel gave up waiting for a peer (code %d)", c->d.rank,
              -static_cast<int>(s));
}

uint64_t b2_comm_launch_count(const b2_comm_t* c) { return c ? c->launches : 0; }

int b2_comm_last_algo(const b2_comm_t* c) { return c ? c->last_algo : B2_EINVAL; }

int b2_auto_algo(int world, int mode, size_t n_elems, int has_multicast) {
  if (world < 1 || world > B2_MAX_WORLD || (mode != B2_F32_WIRE_BF16 && mode != B2_F32 && mode != B2_BF16))
    return fail(B2_EINVAL, "b2_auto_algo: bad arguments (world=%d mode=%d)", world, mode);
  if (world == 1 || n_elems == 0) return B2_ALGO_AUTO;  // no collective: the local pass
  const size_t wire = (n_elems + 7) / 8 * wire_vec_bytes(mode);
  return auto_algo(default_policy(world), world, mode, wire, has_multicast != 0, true);
}

int b2_comm_trace(b2_comm_t* c, int enable, uint64_t* out, int max_ctas) {
  if (!c) return fail(B2_EINVAL, "null communicator");
  DeviceGuard g(c->device);
  if (enable && !c->trace_dev) B2_CUDA(cudaMalloc(&c->trace_dev, sizeof(unsigned long long) * kMaxCtas * 8));
  if (out && max_ctas > 0 && c->trace_dev) {
    const int n = max_ctas < kMaxCtas ? max_ctas : kMaxCtas;
    B2_CUDA(cudaMemcpy(out, c->trace_dev, sizeof(unsigned long long) * n * 8, cudaMemcpyDeviceToHost));
  }
  if (enable) B2_CUDA(cudaMemset(c->trace_dev, 0, sizeof(unsigned long long) * kMaxCtas * 8));  // no stale CTAs
  c->d.trace = enable ? c->trace_dev : nullptr;
  return B2_OK;
}

int b2_local_pass(void* buf, size_t n_elems, int mode, float scale, int device, void* stream) {
  return local_pass_impl(kNoSrc, buf, n_elems, mode, scale, device, stream);
}

static int allreduce_impl(b2_comm_t* c, Src& src, void* buf, size_t n_elems, int mode, float scale, int algo, void* stream) {
  if (!c) return fail(B2_EINVAL, "null communicator");
  if (mode != B2_F32_WIRE_BF16 && mode != B2_F32 && mode != B2_BF16)
    return fail(B2_EINVAL, "unknown mode %d", mode);
  if (algo != B2_ALGO_AUTO && algo != B2_ALGO_ONESHOT && algo != B2_ALGO_TWOSHOT && algo != B2_ALGO_TWOSHOT_PIPE &&
      algo != B2_ALGO_NVLS && algo != B2_ALGO_TWOSHOT_LL)
    return fail(B2_EINVAL, "unknown algo %d", algo);
  if (n_elems == 0) return B2_OK;
  if (!buf) return fail(B2_EINVAL, "b2_allreduce: null buffer");
  if (*reinterpret_cast<volatile uint32_t*>(c->status_host) != 0)
    return fail(B2_ESTATE, "communicator poisoned by an earlier peer-wait timeout");
  const int W = c->d.world;
  if (W == 1) {
    if (mode == B2_F32 && scale == 1.0f && src.nseg == 0) return B2_OK;  // identity
    int rc = local_pass_impl(src, buf, n_elems, mode, scale, c->device, stream);
    if (rc == B2_OK) c->launches++;
    return rc;
  }
  if (algo == B2_ALGO_NVLS && c->d.mc == nullptr)
    return fail(B2_ENOTSUP, "B2_ALGO_NVLS: this communicator has no multicast mapping (b2_comm_caps)");
  DeviceGuard g(c->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t wvb = wire_vec_bytes(mode);
  const size_t cap_vecs = c->d.slice_cap / wvb;  // vecs one region can hold
  const int U = unroll_for_world(W);
  uint8_t* p = static_cast<uint8_t*>(buf);
  size_t left = n_elems;
  while (left > 0) {
    const unsigned long long V_left = (left + 7) / 8;
    const size_t wire_left = V_left * wvb;
    int kind;
    if (algo == B2_ALGO_AUTO) {
      AutoPolicy pol{c->oneshot_max_wire_bytes, c->ll_min_wire_bytes, c->ll_max_wire_bytes, c->pipe_min_wire_bytes,
                     c->nvls_min_wire_bytes, c->nvls_min_world};
      kind = auto_algo(pol, W, mode, wire_left, c->d.mc != nullptr, V_left <= cap_vecs);
    } else {
      kind = algo;
    }
    const bool oneshot = kind == B2_ALGO_ONESHOT;
    const unsigned long long max_vecs = oneshot ? cap_vecs : cap_vecs * W;
    const unsigned long long V = V_left < max_vecs ? V_left : max_vecs;
    const size_t n = V == V_left ? left : static_cast<size_t>(V) * 8;
    const unsigned long long Ls = (V + W - 1) / W;
    const PipePlan plan = plan_pipe(c, Ls, V * wvb);
    const int grid = grid_for(c, oneshot ? V : Ls, U);
    const cudaError_t e = launch_mode(c->d, src, mode, kind, grid, plan, p, n, scale, s);
    if (e != cudaSuccess) return fail(B2_ECUDA, "allreduce kernel launch: %s", cudaGetErrorString(e));
    c->launches++;
    c->last_algo = kind;
    p += n * elem_bytes(mode);
    src.off += n;
    left -= n;
  }
  return B2_OK;
}

int b2_allreduce(b2_comm_t* c, void* buf, size_t n_elems, int mode, float scale, int algo, void* stream) {
  Src src = kNoSrc;
  return allreduce_impl(c, src, buf, n_elems, mode, scale, algo, stream);
}

int b2_allreduce_gather(b2_comm_t* c, void* out, size_t n_elems, const b2_segment_t* segments, int n_segments, int mode,
                        float scale, int algo, void* stream) {
  if (n_elems == 0) return B2_OK;
  if (!segments) return fail(B2_EINVAL, "b2_allreduce_gather: null segment table");
  if (n_segments <= 0 || n_segments > B2_MAX_SEGMENTS)
    return fail(B2_EINVAL, "b2_allreduce_gather: need 1..%d segments (got %d)", B2_MAX_SEGMENTS, n_segments);
  Src src;
  src.nseg = n_segments;
  src.off = 0;
  unsigned long long at = 0;
  for (int i = 0; i < n_segments; ++i) {
    if (segments[i].begin != at)
      return fail(B2_EINVAL, "b2_allreduce_gather: segment %d does not continue the bucket at element %llu", i, at);
    if (segments[i].end <= at) return fail(B2_EINVAL, "b2_allreduce_gather: segment %d is empty", i);
    if (!segments[i].src) return fail(B2_EINVAL, "b2_allreduce_gather: segment %d has a null src", i);
    src.ptr[i] = segments[i].src;
    src.begin[i] = at;
    at = segments[i].end;
  }
  if (at != n_elems) return fail(B2_EINVAL, "b2_allreduce_gather: segments cover %llu elements, bucket has %zu", at, n_elems);
  for (int i = n_segments; i <= B2_MAX_SEGMENTS; ++i) src.begin[i] = at;
  for (int i = n_segments; i < B2_MAX_SEGMENTS; ++i) src.ptr[i] = nullptr;
  return allreduce_impl(c, src, out, n_elems, mode, scale, algo, stream);
}

int b2_broadcast(b2_comm_t* c, void* buf, size_t bytes, int root, void* stream) {
  if (!c) return fail(B2_EINVAL, "null communicator");
  if (root < 0 || root >= c->d.world) return fail(B2_EINVAL, "b2_broadcast: root %d out of range", root);
  if (bytes == 0 || c->d.world == 1) return B2_OK;
  if (!buf) return fail(B2_EINVAL, "b2_broadcast: null buffer");
  if (*reinterpret_cast<volatile uint32_t*>(c->status_host) != 0)
    return fail(B2_ESTATE, "communicator poisoned by an earlier peer-wait timeout");
  DeviceGuard g(c->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t cap = c->stage_bytes & ~static_cast<size_t>(15);
  uint8_t* p = static_cast<uint8_t*>(buf);
  size_t left = bytes;
  while (left > 0) {
    const size_t n = left < cap ? left : cap;
    const int grid = grid_for(c, (n + 15) / 16, 1);
    k_broadcast<<<grid, kThreads, 0, s>>>(c->d, p, n, root);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(B2_ECUDA, "broadcast kernel launch: %s", cudaGetErrorString(e));
    c->launches++;
    p += n;
    left -= n;
  }
  return B2_OK;
}

int b2_barrier(b2_comm_t* c, void* stream) {
  if (!c) return fail(B2_EINVAL, "null communicator");
  if (c->d.world == 1) return B2_OK;
  if (*reinterpret_cast<volatile uint32_t*>(c->status_host) != 0)
    return fail(B2_ESTATE, "communicator poisoned by an earlier peer-wait timeout");
  DeviceGuard g(c->device);
  k_barrier<<<1, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(c->d);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(B2_ECUDA, "barrier kernel launch: %s", cudaGetErrorString(e));
  c->launches++;
  return B2_OK;
}

}  // extern "C"
