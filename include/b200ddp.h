/*
 * b200ddp.h — C ABI of libb200ddp.so, the B200-native data plane behind the
 * `local_cuda` TorchX scheduler.
 *
 * This is the drop-in boundary for the data-parallel hot path.  The reference
 * (meta-pytorch/torchx) has no native code: its `dist.ddp` component only builds a
 * `torchrun` command line (torchx/components/dist.py:261-308) and the gradient
 * allreduce is executed by third-party torch + NCCL.  The entry points below are
 * therefore exactly the operations the reference's workers reach through
 * `torch.distributed` on this path, each citing the interface it replaces:
 *
 *   b2_comm_create     <- dist.init_process_group("nccl")   torchx/distributed/__init__.py:217-222
 *                         (TCPStore rendezvous + ncclCommInitRank; here: POSIX-shm control block +
 *                          CUDA-IPC exchange of one symmetric arena per rank over NVSwitch)
 *   b2_allreduce       <- the DDP bucket comm hook          torch/distributed/algorithms/ddp_comm_hooks/default_hooks.py:18-93
 *                         (`buf.to(bf16).div_(W)` -> ncclAllReduce(SUM) -> `buf.copy_()`, 4 launches; here ONE fused kernel)
 *                         and `dist.all_reduce`             torchx/schedulers/test/train.py:35,
 *                                                           torchx/examples/apps/compute_world_size/module/util.py:37
 *   b2_allreduce_gather <- the Reducer's bucket copy-in fused into the hook (reducer.cpp mark_variable_ready_dense)
 *   b2_broadcast       <- DDP init / per-forward buffer sync torch/nn/parallel/distributed.py:881-890, 2176-2243
 *   b2_barrier         <- dist.barrier()                     torchx/distributed/__init__.py:268,274,297,303
 *   b2_comm_destroy    <- dist.destroy_process_group()
 *
 * Conventions: plain pointers and sizes only (no torch types); every function returns
 * B2_OK (0) or a negative B2_E* code and never throws across the ABI; the text of the
 * last error on the calling thread is available from b2_last_error().  All device work
 * is enqueued asynchronously on the caller's CUDA stream (`stream` is a cudaStream_t
 * passed as void*; NULL = the legacy default stream).  A communicator is a single
 * stream-ordered sequence of collectives (like an NCCL communicator): all ranks must
 * issue the same operations in the same order, and calls on one communicator must not
 * be issued concurrently from several host threads.
 */
#ifndef B200DDP_H_
#define B200DDP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_ABI_VERSION 2
#define B2_MAX_WORLD 8 /* one NVSwitch domain: 8 x B200 */

/* ---- return codes ---------------------------------------------------------------- */
#define B2_OK 0
#define B2_EINVAL (-1)   /* bad argument (null pointer, rank >= world, unknown dtype ...) */
#define B2_ECUDA (-2)    /* a CUDA runtime call failed; see b2_last_error() */
#define B2_ESYS (-3)     /* shm_open/mmap/... failed */
#define B2_ETIMEOUT (-4) /* rendezvous or an in-kernel peer wait timed out */
#define B2_ENOPEER (-5)  /* two ranks' devices cannot reach each other over P2P */
#define B2_ESTATE (-6)   /* communicator is poisoned by an earlier failure */
#define B2_ENOTSUP (-7)  /* the requested algorithm needs a capability this communicator lacks (b2_comm_caps) */

/* ---- element / wire formats ------------------------------------------------------ */
/* The arithmetic of every mode is fixed so results are bit-reproducible run to run and
 * independent of timing:   c_r = wire(scale * x_r) ;  s = ((c_0 + c_1) + ...) + c_{W-1} in fp32,
 * rank order ;  out = round(s).  See oracle/allreduce_oracle.c for the exact rounding points. */
#define B2_F32_WIRE_BF16 0 /* fp32 bucket, bf16 on the wire, fp32 result holding bf16-representable values
                              (== torch bf16_compress_hook semantics)                                   */
#define B2_F32 1           /* fp32 bucket, fp32 on the wire (== DDP default: pre-divide then SUM)         */
#define B2_BF16 2          /* bf16 bucket, bf16 on the wire, fp32 accumulate, one final rounding          */

/* ---- algorithm selection --------------------------------------------------------- */
#define B2_ALGO_AUTO 0
#define B2_ALGO_ONESHOT 1      /* push whole message to every peer, one flag barrier, reduce locally                  */
#define B2_ALGO_TWOSHOT 2      /* push-scatter (fused cast) -> reduce own slice -> pull-gather (fused cast), one pass */
#define B2_ALGO_TWOSHOT_PIPE 3 /* the same three phases as warp-specialised roles pipelined over K chunks             */
#define B2_ALGO_NVLS 4         /* cast -> multimem.ld_reduce + multimem.st through the NVSwitch -> widen, pipelined;
                                  needs B2_CAP_MULTICAST.  The switch sums the W contributions with fp32 accumulation
                                  and rounds once; its summation order is the switch's, see DESIGN.md 2.4              */
#define B2_ALGO_TWOSHOT_LL 5   /* barrier-free two-shot: push-scatter -> reduce as contributions arrive -> push the result
                                  to every rank -> widen as slices arrive; arrival is read off the data itself (sentinel-
                                  filled buffers), no flag barrier and no fence on the data path; rank-order arithmetic   */

/* ---- capabilities (b2_comm_caps) -------------------------------------------------- */
#define B2_CAP_VMM 1       /* arena is a CUDA VMM allocation shared by file descriptor (else cudaMalloc + CUDA IPC) */
#define B2_CAP_MULTICAST 2 /* arena is bound into an NVSwitch multicast object on every rank: NVLS is available    */

typedef struct b2_comm b2_comm_t; /* opaque */

/* Library / ABI version (B2_ABI_VERSION this header was written for). */
int b2_version(void);

/* Text of the last error raised on the calling thread ("" if none). Never NULL. */
const char* b2_last_error(void);

/*
 * Create this rank's communicator.  All `world` ranks (one process per GPU) call this with the
 * same `shm_name` (a POSIX shm object name such as "/b2_<app_id>", handed out by the launcher
 * through the B2_SHM_NAME environment variable) and the same `epoch` (the launcher's restart
 * counter: a re-launched gang uses a new epoch so survivors never map a dead peer's memory).
 * `device` is the CUDA ordinal this rank is pinned to.  `stage_bytes` is the per-rank size of ONE
 * of the two symmetric staging buffers (0 = default 512 MiB); messages larger than what fits are
 * chunked internally.  `timeout_ms` bounds the rendezvous (0 = default 120 s).
 */
int b2_comm_create(b2_comm_t** out, int rank, int world, int device, const char* shm_name,
                   uint64_t epoch, size_t stage_bytes, int timeout_ms);

/*
 * Create `world` communicators inside ONE process (out[0..world-1]), rank i on devices[i].
 * Devices may repeat (all ranks on one GPU): this is the single-GPU parity-test topology.  With
 * distinct devices it uses cudaDeviceEnablePeerAccess instead of CUDA IPC.
 */
int b2_comm_create_local(b2_comm_t** out, int world, const int* devices, size_t stage_bytes);

int b2_comm_destroy(b2_comm_t* comm);

int b2_comm_rank(const b2_comm_t* comm);
int b2_comm_world(const b2_comm_t* comm);
int b2_comm_device(const b2_comm_t* comm);

/* Bitmask of B2_CAP_* this communicator ended up with (identical on every rank), or B2_EINVAL. */
int b2_comm_caps(const b2_comm_t* comm);

/* In-kernel peer-wait timeout (default 600 s, NCCL's default for the same situation; B2_TIMEOUT_MS env overrides at
 * create time).  A kernel that gives up records B2_ETIMEOUT for b2_comm_status() and poisons the communicator. */
int b2_comm_set_timeout_ms(b2_comm_t* comm, int timeout_ms);

/* Upper bound on CTAs one collective may occupy (default: tuned per message size; 0 restores it).
 * Must be set identically on every rank. */
int b2_comm_set_max_ctas(b2_comm_t* comm, int max_ctas);

/*
 * What B2_ALGO_AUTO resolves to for a message of `n_elems` elements in `mode` on `world` ranks with the library's default
 * thresholds (and the B2_* environment overrides); `has_multicast` = the communicator would have B2_CAP_MULTICAST.  Pure
 * function, no GPU needed: lets a caller (and the CPU test-suite) see the policy table of DESIGN.md 2.6.  Messages larger
 * than a staging buffer are cut into several launches, each resolved on its own size.  world == 1: B2_ALGO_AUTO (local pass).
 */
int b2_auto_algo(int world, int mode, size_t n_elems, int has_multicast);

/*
 * Tuning knobs of the AUTO algorithm choice and of the pipelined kernels; must be set identically on every rank.
 *   "oneshot_max_bytes"  one-shot up to this many wire bytes           (env B2_ONESHOT_MAX_BYTES)
 *   "pipe_min_bytes"     pipelined two-shot from this many wire bytes   (env B2_PIPE_MIN_BYTES)
 *   "nvls_min_bytes"     NVLS from this many wire bytes                 (env B2_NVLS_MIN_BYTES)
 *   "nvls_min_world"     NVLS from this world size                      (env B2_NVLS_MIN_WORLD)
 *   "ll_min_bytes"       barrier-free LL two-shot from this many wire bytes (env B2_LL_MIN_BYTES) ...
 *   "ll_max_bytes"       ... up to (excluding) this many                (env B2_LL_MAX_BYTES)
 *   "pipe_chunk_bytes"   target wire bytes per pipeline chunk           (env B2_PIPE_CHUNK_KB, in KiB)
 *   "max_ctas"           same as b2_comm_set_max_ctas
 */
int b2_comm_set_param(b2_comm_t* comm, const char* name, long long value);

/*
 * Non-blocking health check: B2_OK, or B2_ETIMEOUT if any kernel of this communicator gave up
 * waiting for a peer (its output is then undefined).  Reads a host-mapped status word; does not
 * synchronise the device.
 */
int b2_comm_status(const b2_comm_t* comm);

/* Number of kernels this communicator has launched so far (for bench.py's gpu_launches). */
uint64_t b2_comm_launch_count(const b2_comm_t* comm);

/* B2_ALGO_* of the most recent multi-rank allreduce launch of this communicator (what B2_ALGO_AUTO resolved to; 0 if none). */
int b2_comm_last_algo(const b2_comm_t* comm);

/*
 * Measurement aid (tools/sweep_allreduce.py --trace): when enabled, every CTA of a collective records %globaltimer at
 * its phase boundaries, 8 u64 slots per CTA.  Single-pass kernels: start, scatter/push done, barrier 1 passed, reduce
 * done, barrier 2 passed, gather done.  Pipelined kernels (one stamp per role group): role A start, role A done (all
 * chunks), role B passed its first wait, role B done, role C passed its first wait, role C done.  Calling with a
 * non-NULL `out` first copies the stamps of the most recent collective for CTAs [0, max_ctas) (synchronously; call
 * after a stream sync), then applies `enable`.
 */
int b2_comm_trace(b2_comm_t* comm, int enable, uint64_t* out, int max_ctas);

/*
 * In-place averaged/scaled SUM allreduce of `n_elems` elements at device pointer `buf`
 * (any device allocation of this rank; it does not need to be symmetric memory):
 *      buf[i] <- round( sum_{r=0..W-1} wire( scale * buf_r[i] ) )
 * `mode` is one of B2_F32_WIRE_BF16 / B2_F32 / B2_BF16, `algo` one of B2_ALGO_*.
 * scale is normally 1/W (DDP gradient averaging).  n_elems == 0 is a no-op.
 */
int b2_allreduce(b2_comm_t* comm, void* buf, size_t n_elems, int mode, float scale, int algo,
                 void* stream);

/*
 * The same collective with the INPUT gathered straight from the per-parameter gradient tensors instead of from the
 * bucket: replaces the Reducer's copy-in pass (torch/csrc/distributed/c10d/reducer.cpp, mark_variable_ready_dense ->
 * bucket_view.copy_(grad); with gradient_as_bucket_view the copy still happens whenever autograd produced the gradient
 * elsewhere, torch/nn/parallel/distributed.py:589-600) - 8 bytes per element and one multi-tensor launch per bucket.
 *      out[i] <- round( sum_r wire( scale * segment_r(i)[i - begin] ) ),   i in [0, n_elems)
 * `segments`: HOST array of 1..B2_MAX_SEGMENTS entries in bucket order and without gaps: segment k covers bucket elements
 * [begin, end) and reads them from the DEVICE pointer `src` (this rank's tensor of the bucket's dtype, dense in the
 * bucket's element order; it may alias `out`).  The table is copied into the kernel parameters by this call: it need not
 * outlive it.  `out` is this rank's bucket.  More parameters than B2_MAX_SEGMENTS: B2_EINVAL (copy in, then b2_allreduce).
 * A NULL table, an empty segment, a NULL `src`, a gap or a table that does not cover exactly n_elems: B2_EINVAL.
 */
#define B2_MAX_SEGMENTS 128
typedef struct b2_segment {
  const void* src;
  uint64_t begin;
  uint64_t end;
} b2_segment_t;

int b2_allreduce_gather(b2_comm_t* comm, void* out, size_t n_elems, const b2_segment_t* segments, int n_segments,
                        int mode, float scale, int algo, void* stream);

/* Broadcast `bytes` bytes at `buf` from rank `root` to every rank (bit-exact copy). */
int b2_broadcast(b2_comm_t* comm, void* buf, size_t bytes, int root, void* stream);

/* Device-side barrier across all ranks, ordered on `stream`. */
int b2_barrier(b2_comm_t* comm, void* stream);

/*
 * Local (no peers) building block, also the W==1 fast path of b2_allreduce: applies
 * x <- round(wire(scale*x)) to `n_elems` elements on `device`.  Exposed so the single-GPU
 * roofline of the fused cast/scale pass can be measured without a communicator.
 */
int b2_local_pass(void* buf, size_t n_elems, int mode, float scale, int device, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200DDP_H_ */
