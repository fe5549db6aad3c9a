// Internal declarations shared by the translation units of libedb.so.
// Not part of the C-ABI (that is include/edb.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "edb.h"

namespace edb {

constexpr int kMaxWorld = 64;
constexpr int kMaxGroup = EDB_MAX_GROUP;
constexpr int kMaxGroups = EDB_MAX_GROUPS;

// ---- flag area at the start of every rank's slab --------------------------------------------
// One 1 KiB block (128 x u64) per group slot.  All counters are monotonically increasing
// sequence numbers ("epochs"), never reset, so the same kernel parameters stay valid across
// CUDA-graph replays.
constexpr size_t kFlagBlockBytes = 1024;
constexpr size_t kFlagAreaBytes = 64 * 1024;           // kMaxGroups blocks + spare
constexpr size_t kScratchBytes = 40u << 20;             // per-rank scratch: low-latency packet buffers
// Low-latency ("LL") small-message protocol: 8-byte packets {4 B payload, 4 B epoch} pushed into
// the receivers' scratch with single 8-byte stores, so data and flag become visible together and
// an op needs no fence, no flag round trip and no peer reads (NCCL's LL idea).  Per group slot
// (first kLLGroups slots): 2 parities x kMaxGroup sources x kLLCapacity packets.
constexpr int kLLGroups = 4;
constexpr size_t kLLCapacity = 65536;                  // packets per (parity, source) = 256 KiB payload
constexpr size_t kLLBytesPerGroup = 2 * 8 * kLLCapacity * 8;  // 8 MiB
constexpr size_t kUserOffset = kFlagAreaBytes + kScratchBytes;

enum FlagWord : int {
  F_READY = 0,    // [0..7]   READY[p]  : peer p staged its data for op q          (written by p)
  F_DONE = 8,     // [8..15]  DONE[p]   : peer p finished reading my data of op q  (written by p)
  F_READY2 = 16,  // [16..23] READY2[p] : second phase of two-shot ops             (written by p)
  F_SEQ = 24,     // last op number completed locally                              (written by me)
  F_CNT_A = 25,   // last-block counters
  F_CNT_B = 26,
  F_CNT_C = 27,
  F_ERR = 28,     // != 0: a spin wait timed out (value = op number)
  F_LLSEQ = 29,   // sequence number of the low-latency ops of this group
  F_CNT_LL = 30,  // last-block counter of the LL kernels
  F_ERRHOST = 31, // device pointer of the pinned host error record (written once at edb_init)
  // ---- epoch protocol (edb_epoch_barrier + the fused / push kernels) --------------------------
  // One group-wide barrier per phase of the step instead of a handshake per op: between two
  // barriers peers may read this rank's symmetric operands / write its receive slots freely.
  F_EPOCH = 48,      // [48..55] ARRIVED[p]: member p reached barrier number e   (written by p)
  F_EPOCH_SEQ = 56,  // barriers completed locally                                 (written by me)
  F_AGSEQ = 57,      // launch number of the AG+GEMM kernels (local chunk-flag epochs)
  F_AGCNT = 58,      // CTAs of the current AG+GEMM launch that have read F_AGSEQ
  F_AGDONE = 59,     // comm CTAs of the current launch that have finished
  F_AGCHUNK = 64,    // [64..71] local: peer shard c is in the gathered buffer (launch number)
  F_AGTILE = 72,     // [72..79] comm CTAs done with shard c
  // push protocol of the stand-alone collectives (edb_*_push, epoch mode): every member writes its
  // contribution straight into the consumers' static buffers and raises ONE one-way flag per peer
  F_PUSHFLAG = 80,   // [80..87] PUSHED[p]: member p's data of push-op q has landed here (written by p)
  F_PUSHSEQ = 88,    // push-ops completed locally
  F_CNT_P = 89,      // last-block counters of the push kernels
  F_CNT_P2 = 90,
};

struct Group {
  int n = 0, me = -1, slot = -1;
  int ranks[kMaxGroup];
};

struct Runtime {
  bool inited = false;
  int rank = 0, world = 1, device = 0, sm_count = 148;
  char* heap = nullptr;
  size_t heap_bytes = 0;
  size_t bump = kUserOffset;
  char* peer_heap[kMaxWorld] = {};
  bool peer_is_ipc[kMaxWorld] = {};
  Group groups[kMaxGroups];
  int ngroups = 0;
  // options
  int64_t allreduce_oneshot_bytes = 512 * 1024;
  int64_t copy_ctas_per_sm = 4;
  int64_t comm_ctas = 16;
  int64_t spin_timeout_ms = 120000;  // fatal when exceeded (NCCL-watchdog-like; EDB_SPIN_TIMEOUT_MS)
  uint64_t* host_err = nullptr;      // pinned + mapped: {flag, op, kind, -}; survives a trapped context
  uint64_t* host_err_dev = nullptr;  // device alias of host_err
  int64_t ll_max_bytes = 128 * 1024;  // payload per rank up to which the LL protocol is used (0 = off)
  int64_t gemm_force_bn = 0;  // tuning aid: 128 / 256 overrides the tile-width heuristic
  int64_t gemm_splitk = 1;   // 1: split K over idle SMs when the tiles fill at most half of them
  int64_t push_sync = 1;     // how push-GEMM CTAs retire (GemmParams::push_sync); 1 measured == 0
  int64_t gemm_cluster = 2;  // 2: pair CTAs in clusters and multicast the B tile; 1: off
};

Runtime& rt();
int set_error(int code, const char* fmt, ...);
int cuda_check(cudaError_t e, const char* what);
void count_launch();

#define EDB_CUDA(call)                                  \
  do {                                                  \
    int _rc = ::edb::cuda_check((call), #call);         \
    if (_rc) return _rc;                                \
  } while (0)

#define EDB_REQUIRE(cond, ...)                                        \
  do {                                                                \
    if (!(cond)) return ::edb::set_error(EDB_E_INVALID, __VA_ARGS__); \
  } while (0)

inline char* ll_region(char* heap, int slot) {
  return heap + kFlagAreaBytes + (size_t)slot * kLLBytesPerGroup;
}
inline uint64_t* flag_block(char* heap, int slot) {
  return reinterpret_cast<uint64_t*>(heap + (size_t)slot * kFlagBlockBytes);
}

// ---- kernel-side descriptors ------------------------------------------------------------------

struct Box {
  const char* src;
  char* dst;
  int64_t inner;    // contiguous bytes per row
  int64_t ext[4];   // outer extents, ext[0] slowest; unused dims = 1
  int64_t sstr[4];  // byte strides
  int64_t dstr[4];
  int32_t vec;      // bytes per access: 16, 8, 4, 2 or 1
  int32_t peer;     // group index whose READY flag gates this box; -1 = none (local)
};

struct FlagCtx {
  uint64_t* local;            // my flag block of this group
  uint64_t* peer[kMaxGroup];  // every member's flag block (peer[me] == local)
  int n, me;
  int n_war;                  // number of local flag blocks to check for write-after-read
  uint64_t* war_block[kMaxGroups];
  uint8_t war_n[kMaxGroups];
  uint8_t war_me[kMaxGroups];
  uint64_t timeout_ns;
};

constexpr int kMaxBoxes = 18;

struct GatherDesc {
  FlagCtx f;
  int n_in;     // boxes [0, n_in) are the local copy-in phase
  int n_boxes;  // boxes [n_in, n_boxes) are pulled after the READY flags
  Box box[kMaxBoxes];
};

struct ReduceDesc {
  FlagCtx f;
  int has_in;  // copy `in` first
  Box in;
  // reduction geometry: n_src sources with identical layout
  const char* src[kMaxGroup];
  char* dst;
  int64_t inner;  // bytes per row (source dtype)
  int64_t ext[4];
  int64_t sstr[4];
  int64_t dstr[4];  // destination byte strides (destination dtype)
  int n_src;
  int dtype, out_dtype, redop;
  float scale;
  // two-shot all-reduce: after reducing my part into dst (which lives in my stage2), pull the
  // other parts from the peers' stage2 into final_dst
  int two_shot;
  int n_pull;
  Box pull[kMaxGroup];
};

// host helpers (edb_reshard.cu)
int make_box(Box* out, const void* src, const int64_t* src_strides, void* dst,
             const int64_t* dst_strides, const int64_t* extents, int ndim, int elem_size, int peer);
int fill_flagctx(FlagCtx* f, int gid);
int grid_for_bytes(size_t bytes, int threads, int max_ctas_per_sm);
// edb_ll.cu: low-latency path; returns -1 when the op is not eligible (caller uses the flag path)
int ll_try(int gid, int mode, void* dst, const void* src, int64_t in_bytes, int64_t outer,
           int64_t row_bytes, int dtype, int redop, float scale, cudaStream_t st);

inline size_t dtype_size(int dt) {
  switch (dt) {
    case EDB_F32: return 4;
    case EDB_BF16: return 2;
    case EDB_F16: return 2;
    case EDB_F64: return 8;
    case EDB_I32: return 4;
    case EDB_I64: return 8;
  }
  return 0;
}

// ---- device helpers ---------------------------------------------------------------------------

__device__ __forceinline__ uint64_t ld_acquire_sys(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint64_t* p, uint64_t v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_relaxed_gpu(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint64_t ld_acquire_gpu(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(uint64_t* p, uint64_t v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// A wait on a peer timed out: the peer is lost or more than `spin_timeout_ms` behind.  Carrying on
// would reduce / copy stale peer data and publish the op as done, so the timeout is FATAL (what
// NCCL's watchdog does for the reference): record {op, flag word, 1} in the pinned host error
// record (readable after the context is gone: edb_health()), then trap, which fails this kernel
// and every later CUDA call of the process.  `err_word` = the local flag block's F_ERR word.
static __device__ __noinline__ void fatal_timeout(uint64_t* err_word, uint64_t target, int what) {
  if (err_word) {
    atomicMax((unsigned long long*)err_word, (unsigned long long)target);
    volatile uint64_t* host = reinterpret_cast<volatile uint64_t*>(err_word[F_ERRHOST - F_ERR]);
    if (host) {
      host[1] = target;
      host[2] = (uint64_t)what;
      host[0] = 1;
      __threadfence_system();
    }
  }
  printf("edb: wait on a peer timed out (op/epoch %llu, kind %d) - aborting\n",
         (unsigned long long)target, what);
  asm volatile("trap;");
}

// Spin until *flag >= target (system scope acquire); fatal on timeout (see fatal_timeout).
__device__ __forceinline__ bool spin_wait_sys(const uint64_t* flag, uint64_t target,
                                              uint64_t timeout_ns, uint64_t* err_word) {
  if (ld_acquire_sys(flag) >= target) return true;
  uint64_t t0 = globaltimer_ns();
  while (ld_acquire_sys(flag) < target) {
    __nanosleep(64);
    if (globaltimer_ns() - t0 > timeout_ns) fatal_timeout(err_word, target, 1);
  }
  return true;
}

// ---- flag protocol ---------------------------------------------------------------------------------

// Returns the op number of this launch after the write-after-read guard.
__device__ __forceinline__ uint64_t begin_op(const FlagCtx& f, uint64_t* s_q) {
  if (threadIdx.x == 0) *s_q = ld_relaxed_gpu(f.local + F_SEQ) + 1;
  // one thread per (group of this rank, member): every group's readers must be done
  for (int i = threadIdx.x; i < f.n_war * kMaxGroup; i += blockDim.x) {
    const int b = i >> 3, p = i & 7;
    if (p < f.war_n[b] && p != f.war_me[b]) {
      const uint64_t* blk = f.war_block[b];
      const uint64_t seq = ld_relaxed_gpu(blk + F_SEQ);
      spin_wait_sys(blk + F_DONE + p, seq, f.timeout_ns, f.local + F_ERR);
    }
  }
  __syncthreads();
  return *s_q;
}

// Grid-wide "everyone arrived" (no wait): the last CTA to arrive publishes `q` to word
// `flag_base + me` of every member's flag block (its own included).
__device__ __forceinline__ void grid_signal(const FlagCtx& f, int cnt_word, int flag_base,
                                            uint64_t q, int* s_last, unsigned n_ctas) {
  // One fence per CTA, not per thread: bar.sync orders every thread's writes before thread 0's
  // system-scope fence (PTX causality order is cumulative through barriers; this is the pattern of
  // a cooperative-groups grid sync).  A membar.sys in all 256 threads of every CTA cost several
  // microseconds per op.
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    const unsigned long long prev =
        atomicAdd(reinterpret_cast<unsigned long long*>(f.local + cnt_word), 1ULL);
    const int last = (prev == (unsigned long long)n_ctas - 1);
    if (last) {
      f.local[cnt_word] = 0;
      __threadfence_system();  // acquire side: the other CTAs' fenced writes precede the flag
    }
    *s_last = last;
  }
  __syncthreads();
  if (*s_last && threadIdx.x < f.n) st_release_sys(f.peer[threadIdx.x] + flag_base + f.me, q);
}

__device__ __forceinline__ void wait_flag(const FlagCtx& f, int flag_base, int p, uint64_t q) {
  if (threadIdx.x == 0) spin_wait_sys(f.local + flag_base + p, q, f.timeout_ns, f.local + F_ERR);
  __syncthreads();
}

__device__ __forceinline__ void finish_op(const FlagCtx& f, uint64_t q, int* s_last,
                                          unsigned n_ctas) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();  // covers the whole CTA's writes (see grid_signal)
    const unsigned long long prev =
        atomicAdd(reinterpret_cast<unsigned long long*>(f.local + F_CNT_B), 1ULL);
    const int last = (prev == (unsigned long long)n_ctas - 1);
    if (last) {
      f.local[F_CNT_B] = 0;
      __threadfence_system();
    }
    *s_last = last;
  }
  __syncthreads();
  if (*s_last) {
    if (threadIdx.x < f.n && threadIdx.x != f.me)
      st_release_sys(f.peer[threadIdx.x] + F_DONE + f.me, q);
    if (threadIdx.x == 0) st_release_gpu(f.local + F_SEQ, q);
  }
}

// ---- epoch protocol ------------------------------------------------------------------------------
// Group-wide barrier executed by ONE CTA (>= 32 threads): thread p signals member p and waits for
// it.  The system-scope fence + release stores order everything this rank did earlier on the
// stream (kernel boundaries included: its stores into peer memory, its reads of peer memory)
// before the signal; the acquire loads order the peers' work before whatever follows here.
__device__ __forceinline__ void epoch_barrier_cta(const FlagCtx& f, uint64_t* s_e) {
  if (threadIdx.x == 0) {
    *s_e = ld_relaxed_gpu(f.local + F_EPOCH_SEQ) + 1;
    __threadfence_system();
  }
  __syncthreads();
  const uint64_t e = *s_e;
  if ((int)threadIdx.x < f.n && (int)threadIdx.x != f.me) {
    st_release_sys(f.peer[threadIdx.x] + F_EPOCH + f.me, e);
    const uint64_t* flag = f.local + F_EPOCH + threadIdx.x;
    if (ld_acquire_sys(flag) < e) {
      const uint64_t t0 = globaltimer_ns();
      while (ld_acquire_sys(flag) < e) {
        __nanosleep(32);
        if (globaltimer_ns() - t0 > f.timeout_ns) fatal_timeout(f.local + F_ERR, e, 2);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) st_release_gpu(f.local + F_EPOCH_SEQ, e);
}

}  // namespace edb
