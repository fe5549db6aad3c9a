// Dense bf16 GEMM on Blackwell 5th-gen tensor cores (tcgen05 + TMEM + TMA), the compute half of
// the sharded-op kernel dispatch: the aten.mm.default nodes of the sharded FX graph
// (Linear fwd / dgrad / wgrad; SURVEY.md §8 a14) land here.
//
//   C[M,N] (bf16) = A · B, fp32 accumulation in tensor memory.
//     A: K-major  ([M,K] row-major)  or MN-major (stored [K,M])
//     B: K-major  ([N,K] row-major, i.e. nn.Linear weight) or MN-major (stored [K,N])
//
// Structure (one persistent CTA per SM, 192 threads):
//   warp 0      : TMA producer   — cp.async.bulk.tensor tiles of A and B into a 4/6-stage smem ring
//   warp 1      : MMA issuer     — one elected lane issues tcgen05.mma (128 x BN x 16), accumulators
//                                  live in TMEM, double-buffered so the epilogue of tile i overlaps
//                                  the main loop of tile i+1; also owns TMEM alloc/dealloc
//   warps 2..5  : epilogue       — tcgen05.ld TMEM -> registers -> bf16 -> 16-byte global stores
// Synchronisation is mbarrier-only (full/empty per smem stage, full/empty per TMEM stage).
//
// Shared-memory tiles use the canonical 128-byte-swizzle UMMA layouts, written by TMA with
// CU_TENSOR_MAP_SWIZZLE_128B and described to the tensor core with matching smem descriptors
// (K-major: SBO = 1024 B; MN-major: one 64-element atom per TMA box, LBO = atom stride).
#include <cuda.h>
#include <cuda_bf16.h>

#include "edb_internal.cuh"

namespace edb {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 bytes = one swizzle atom
constexpr int UMMA_K = 16;
constexpr int kGemmThreads = 192;
constexpr int kSmemABytes = BM * BK * 2;  // 16 KiB

// CL = 1: one CTA computes a 128 x BN tile.  CL = 2: a CTA pair computes a 256 x BN tile with
// tcgen05.mma.cta_group::2 — each CTA stages its own 128 rows of A and HALF of the B tile, so a
// stage is 16 KiB + BN*64 B instead of 16 KiB + BN*128 B: more stages in flight (the 1-CTA kernel
// is bound by TMA latency x stage depth: 62% tensor-pipe at 8192^3) and 1.5x less L2->SM traffic.
template <int BN, int CL = 1> struct TileCfg {
  static constexpr int kSmemBBytes = (BN / CL) * BK * 2;
  static constexpr int kStageBytes = kSmemABytes + kSmemBBytes;
  static constexpr int kStages = (CL == 2) ? ((BN == 256) ? 6 : 8) : ((BN == 256) ? 4 : 6);
  static constexpr int kTmemCols = 2 * BN;  // two accumulator stages
  static constexpr int kEpiBufBytes = BM * 64 * 2;  // one 128 x 64 bf16 store box (128B swizzle)
  static constexpr int kEpiBufs = 2;
  static constexpr int kSmemBytes =
      kStages * kStageBytes + kEpiBufs * kEpiBufBytes + 1024 /*align*/ + 256 /*barriers*/;
};

// ---- PTX wrappers ------------------------------------------------------------------------------------

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t addr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(addr), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin on an mbarrier phase.  A watchdog turns a protocol bug into a trap (kernel error) instead
// of a hung GPU: 4 s is ~1000x the longest legitimate wait of any role in these kernels.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  if (mbar_try_wait(addr, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(addr, parity)) {
    if ((++spins & 0xfff) == 0 && globaltimer_ns() - t0 > 4000000000ull) {
      printf("edb gemm watchdog: block %d thread %d stuck on barrier %u parity %u\n", blockIdx.x,
             threadIdx.x, addr, parity);
      asm volatile("trap;");
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* smem,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4}], [%2];" ::"r"(smem_u32(smem)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem, int c0,
                                             int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
      "r"(smem_u32(smem)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_store_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N> __device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void epi_bar_sync() {
  asm volatile("bar.sync 1, 128;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_mcast(const CUtensorMap* map, uint64_t* bar, void* smem,
                                                  int c0, int c1, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // shared::cluster address of the same offset in CTA rank 0
__device__ __forceinline__ void tma_load_2d_2sm(const CUtensorMap* map, uint64_t* leader_bar,
                                                void* smem, int c0, int c1) {
  // executed by both CTAs of the pair; the transaction bytes update the LEADER's barrier
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem)),
      "l"(map), "r"(smem_u32(leader_bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_on_leader(uint64_t* bar) {
  asm volatile(
      "{\n"
      ".reg .b32 raddr;\n"
      "mapa.shared::cluster.u32 raddr, %0, 0;\n"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [raddr];\n"
      "}\n" ::"r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(dst_smem)),
               "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols)
               : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(dst_smem)),
               "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols)
               : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
          smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- descriptors -------------------------------------------------------------------------------------

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4   [16,30) leading byte offset >> 4   [32,46) stride byte offset >> 4
//   [46,48) version = 1 (sm_100)   [61,64) layout type: 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// Instruction descriptor for kind::f16 (cute::UMMA::InstrDescriptor bit layout):
//   [4,6) D format: 1 = F32   [7,10) A format: 1 = BF16   [10,13) B format: 1 = BF16
//   [15] A major: 0 = K, 1 = MN   [16] B major   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc(int m, int n, bool a_mn, bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct GemmParams {
  __nv_bfloat16* C;
  const __nv_bfloat16* bias;  // optional [N] row vector added in the epilogue (aten.addmm)
  int64_t ldc;
  int M, N, K;
  int m_tiles, n_tiles;
  // split-K (MODE_PLAIN only): work unit = (tile, k-slice); every slice writes its fp32 partial
  // tile to `partial` [splits][M][ldp] and k_splitk_reduce sums the slices in a fixed order
  int splits, kb_per_split;
  float* partial;
  int64_t ldp;
  // push mode (MODE_PLAIN, edb_gemm_push_bf16): row block m of C belongs to group member
  // m / push_mtc and is TMA-stored into that member's receive slot (store map cm.m[owner]) instead
  // of C; m_rot rotates the m order so that the ranks do not all push to the same owner at once
  int push_n, push_mtc, m_rot;
  // how a pushing CTA retires: 2 = wait for the completion of its TMA stores + system-scope fence,
  // 1 = completion only, 0 = only until the staging smem has been read (grid completion then
  // covers the stores, as it does for every ordinary TMA-store epilogue)
  int push_sync;
  // fused elementwise epilogue with a second operand `aux` [M, N] bf16 (row stride ld_aux):
  //   EPI_ADD      C = bf16(acc + bias + aux)                  (residual add behind a Linear)
  //   EPI_GELU_BWD C = bf16(acc * gelu'(aux)), tanh approximation, ATen's formula in fp32
  //                (aten.gelu_backward(grad = this GEMM, self = aux): the dgrad GEMM of the MLP's
  //                second Linear produces d(pre-activation) directly)
  const __nv_bfloat16* aux;
  int64_t ld_aux;
  int epi_op;
};
enum { EPI_NONE = 0, EPI_ADD = 1, EPI_GELU_BWD = 2 };

__device__ __forceinline__ float gelu_tanh_grad(float x) {
  // at::native GeluBackwardCUDAKernelImpl, approximate == 'tanh' (opmath = float)
  const float kBeta = 0.7978845608028654f;  // sqrt(2) * (2/sqrt(pi)) * 0.5
  const float kKappa = 0.044715f;
  const float x_sq = x * x;
  const float inner = kBeta * (x + kKappa * x_sq * x);
  // tanh and sech^2 from ONE exponential: e = exp(-2|u|) (ex2.approx, rel. error 2^-22),
  // tanh = sign(u)(1-e)/(1+e), 1 - tanh^2 = 4e/(1+e)^2.  (tanh.approx.f32 is one MUFU op cheaper but
  // its 2^-11 error is absolute near saturation: 1 - t*t then loses everything for |x| > 3 and the
  // gradient of a saturated unit came out as ~3 % of dy instead of ~0.  tanhf costs more than the
  // main loop: 16.7 M evaluations per MLP dgrad GEMM sit on the four epilogue warps.)
  const float au = fabsf(inner);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-2.885390081777927f * au));  // 2 / ln 2
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  const float t = copysignf((1.0f - e) * r, inner);
  const float tanh_d = 4.0f * e * r * r;
  const float left = 0.5f * x, right = 1.0f + t;
  const float left_d = 0.5f * right;
  const float inner_d = kBeta * (1.0f + 3.0f * kKappa * x_sq);
  return left_d + left * tanh_d * inner_d;
}

// Fusion modes of the GEMM kernel
//   MODE_PLAIN : C = A.B
//   MODE_AG    : B (weights, [N,K] K-major) is sharded S(0) over the group; a few "comm" CTAs pull the
//                peer shards over NVLink with TMA bulk copies into the local gathered buffer while
//                the MMA CTAs start on the local shard and pick up chunks as their flags arrive
//                (all_gather_end -> aten.mm of the sharded graph in one kernel).  No handshake with
//                the peers inside the kernel: an edb_epoch_barrier earlier on the stream made every
//                member's shard final, and the next barrier comes before anybody overwrites it.
//                Only the local chunk flags (comm CTAs -> MMA CTAs) remain.
enum { MODE_PLAIN = 0, MODE_AG = 1 };
constexpr int kMaxPfItems = 4;
constexpr int kPfSlots = 12, kPfDepth = 8;  // 16 KiB slots of the prefetch ring / loads in flight

struct FusedArgs {
  FlagCtx f;
  int n_comm;  // MODE_AG: number of comm CTAs at the start of the grid
  // MODE_AG
  const char* shard_src[kMaxGroup];  // member p's shard (peer mapped); [me] is local
  char* full_dst;                    // local gathered buffer
  int64_t shard_bytes;
  int ag_rows;        // rows of B per shard (N / n)
  int ag_first_tile;  // n-tile containing the first row of my shard
  // all-gather PREFETCH riding on a plain GEMM (edb_gemm_pf_bf16): the first pf_ctas CTAs of the
  // grid do no MMA work; they copy, for each item and each group member p, the byte range
  // [src_off, src_off + bytes) of p's symmetric heap into local dst_off + p * dst_stride — the
  // operand of a LATER kernel (next layer's weight), so nobody in this kernel waits for the data
  // and the consumer is an ordinary GEMM.  Epoch protocol: the sources are final since the last
  // edb_epoch_barrier.
  int pf_ctas, pf_items, pf_n;
  const char* pf_heap[kMaxGroup];  // members' heaps (peer mapped), [pf_me] = local
  char* pf_local;
  uint64_t pf_src[kMaxPfItems], pf_dst[kMaxPfItems];
  int64_t pf_bytes[kMaxPfItems], pf_stride[kMaxPfItems];
  // pf_sstride: member p's source is at pf_src + p * pf_sstride (0: the same offset everywhere).
  // With pf_sstride == pf_stride and pf_src == pf_dst every member's shard LIVES in its slot of
  // the gathered buffer: nothing to copy for the own range (pf_inplace), n-1 remote ranges only.
  int64_t pf_sstride[kMaxPfItems];
  int pf_inplace[kMaxPfItems];
};

struct CMaps {
  CUtensorMap m[kMaxGroup];  // push: store map of member p's receive slot [me]; MODE_AG: m[0] = local shard
};

template <int MODE>
__device__ __forceinline__ void tile_coords(int t, const GemmParams& p, const FusedArgs& fa,
                                            int& m_blk, int& n_blk) {
  if (MODE == MODE_AG) {
    // n-tiles in rotated order starting at the tile that holds my own shard (needs no transfer),
    // then in the order the comm CTAs pull the peers' shards; a tile may span several shards (see
    // the producer)
    const int ni = t / p.m_tiles;
    n_blk = (fa.ag_first_tile + ni) % p.n_tiles;
    m_blk = t - ni * p.m_tiles;
  } else {
    m_blk = (t % p.m_tiles + p.m_rot) % p.m_tiles;
    n_blk = t / p.m_tiles;
  }
}

__device__ __forceinline__ void bulk_load(void* smem, const void* gsrc, uint32_t bytes,
                                          uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(smem)),
      "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
               "r"(smem_u32(smem)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() {
  asm volatile("fence.proxy.async;" ::: "memory");
}
__device__ __forceinline__ void spin_wait_gpu(const uint64_t* flag, uint64_t target) {
  if (ld_acquire_gpu(flag) >= target) return;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (ld_acquire_gpu(flag) < target) {
    __nanosleep(32);
    if ((++spins & 0xfff) == 0 && globaltimer_ns() - t0 > 4000000000ull) {
      printf("edb fused gemm watchdog: block %d stuck on chunk flag\n", blockIdx.x);
      asm volatile("trap;");
    }
  }
}

// Prefetch CTA (see FusedArgs::pf_*): one thread drives a TMA bulk-copy ring peer HBM -> smem ->
// local HBM over the 16 KiB blocks of all (item, member) ranges; block b belongs to CTA
// b % pf_ctas, so the CTAs stream neighbouring blocks and every range finishes at about the same
// time.  No flags: the consumer is a later kernel on the stream.
__device__ __forceinline__ void pf_role(const FusedArgs& fa, uint8_t* smem, int idx, int nctas) {
  constexpr int S = kPfSlots, D = kPfDepth, SLOT = 16384;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S * SLOT);
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) mbar_init(&full[s], 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  // flat block numbering: item-major, member-major inside an item, remote members first
  uint32_t n_load = 0, n_store = 0;
  struct Cur { int it, k; int64_t blk; };
  auto advance = [&](Cur& c) {
    // move to the next block owned by this CTA; returns false at the end
    while (c.it < fa.pf_items) {
      const int64_t nblk = (fa.pf_bytes[c.it] + SLOT - 1) / SLOT;
      const int members = fa.pf_inplace[c.it] ? fa.pf_n - 1 : fa.pf_n;  // own range last / skipped
      if (c.k < members && c.blk < nblk) return true;
      if (c.k < members) c.blk -= nblk;  // keep the round-robin phase across ranges
      if (++c.k >= members) {
        c.k = 0;
        ++c.it;
      }
    }
    return false;
  };
  Cur ld = {0, 0, (int64_t)idx}, stc = {0, 0, (int64_t)idx};
  bool more = advance(ld);
  int inflight = 0;
  while (more || inflight > 0) {
    if (more && inflight < D) {
      const uint32_t slot = n_load % S;
      if (n_load >= (uint32_t)S) tma_store_wait_read<S - D - 1>();
      const int p = (fa.f.me + 1 + ld.k) % fa.pf_n;  // own range last (a local copy)
      const int64_t off = ld.blk * SLOT;
      const int64_t left = fa.pf_bytes[ld.it] - off;
      const uint32_t bytes = (uint32_t)(left < SLOT ? left : SLOT);
      mbar_expect_tx(&full[slot], bytes);
      bulk_load(smem + slot * SLOT,
                fa.pf_heap[p] + fa.pf_src[ld.it] + (int64_t)p * fa.pf_sstride[ld.it] + off, bytes,
                &full[slot]);
      ++n_load;
      ++inflight;
      ld.blk += nctas;
      more = advance(ld);
      continue;
    }
    // oldest load -> store
    advance(stc);
    const uint32_t slot = n_store % S;
    mbar_wait(&full[slot], (n_store / S) & 1);
    const int p = (fa.f.me + 1 + stc.k) % fa.pf_n;
    const int64_t off = stc.blk * SLOT;
    const int64_t left = fa.pf_bytes[stc.it] - off;
    const uint32_t bytes = (uint32_t)(left < SLOT ? left : SLOT);
    bulk_store(fa.pf_local + fa.pf_dst[stc.it] + (int64_t)p * fa.pf_stride[stc.it] + off,
               smem + slot * SLOT, bytes);
    tma_store_commit();
    ++n_store;
    --inflight;
    stc.blk += nctas;
  }
  tma_store_wait_all();
}

__global__ void __launch_bounds__(32, 1) k_ag_prefetch(const __grid_constant__ FusedArgs fa) {
  extern __shared__ uint8_t pf_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(pf_smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  pf_role(fa, smem, (int)blockIdx.x, (int)gridDim.x);
}

// MODE_AG comm CTA: one thread drives a TMA bulk-copy ring  peer HBM -> smem -> local HBM, ONE
// software pipeline over the blocks of all shards — no drain between shards (a drain costs a load +
// store latency per shard, ~4 us x (n-1) at n = 8) and no flag traffic with the peers at all.  A
// shard is announced to the MMA CTAs once `wait_group` proves its last store complete, which lags
// kLag stores behind.
__device__ __forceinline__ void ag_comm_role(const FusedArgs& fa, uint8_t* smem, int comm_idx,
                                             uint64_t q) {
  constexpr int S = 8, D = 5, SLOT = 16384, kLag = 2;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S * SLOT);
  const FlagCtx& f = fa.f;
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) mbar_init(&full[s], 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  const int64_t per = ((fa.shard_bytes + fa.n_comm - 1) / fa.n_comm + SLOT - 1) / SLOT * SLOT;
  const int64_t lo = (int64_t)comm_idx * per;
  const int64_t hi = lo + per < fa.shard_bytes ? lo + per : fa.shard_bytes;
  const int nblk = hi > lo ? (int)((hi - lo + SLOT - 1) / SLOT) : 0;
  const int total = nblk * f.n;
  auto announce = [&](int k) {
    const int c = (f.me + k) % f.n;
    const unsigned long long prev =
        atomicAdd(reinterpret_cast<unsigned long long*>(f.local + F_AGTILE + c), 1ULL);
    if (prev == (unsigned long long)fa.n_comm - 1) {
      f.local[F_AGTILE + c] = 0;
      __threadfence();
      st_release_gpu(f.local + F_AGCHUNK + c, q);
    }
  };
  if (nblk == 0) {
    for (int k = 0; k < f.n; ++k) announce(k);  // nothing to move for this CTA: still counted
  } else {
    uint32_t n_load = 0, n_store = 0;
    int next_announce = 0;  // shards [0, next_announce) have been announced
    for (int g = 0; g < total + D; ++g) {
      if (g < total) {
        const int k = g / nblk, i = g - k * nblk;
        const int c = (f.me + k) % f.n;
        const uint32_t slot = n_load % S;
        if (n_load >= (uint32_t)S) tma_store_wait_read<S - D - 1>();
        const int64_t left = hi - lo - (int64_t)i * SLOT;
        const uint32_t bytes = (uint32_t)(left < SLOT ? left : SLOT);
        mbar_expect_tx(&full[slot], bytes);
        bulk_load(smem + slot * SLOT, fa.shard_src[c] + lo + (int64_t)i * SLOT, bytes, &full[slot]);
        ++n_load;
      }
      if (g >= D) {
        const int j = g - D;
        const int k = j / nblk, i = j - k * nblk;
        const int c = (f.me + k) % f.n;
        const uint32_t slot = n_store % S;
        mbar_wait(&full[slot], (n_store / S) & 1);
        const int64_t left = hi - lo - (int64_t)i * SLOT;
        const uint32_t bytes = (uint32_t)(left < SLOT ? left : SLOT);
        bulk_store(fa.full_dst + (int64_t)c * fa.shard_bytes + lo + (int64_t)i * SLOT,
                   smem + slot * SLOT, bytes);
        tma_store_commit();
        ++n_store;
        // shard `next_announce` ended with store number (next_announce + 1) * nblk: once kLag more
        // stores have been committed, wait_group<kLag> proves it complete
        if ((int)n_store - kLag >= (next_announce + 1) * nblk) {
          asm volatile("cp.async.bulk.wait_group %0;" ::"n"(kLag) : "memory");
          fence_proxy_async_all();
          __threadfence();
          while ((int)n_store - kLag >= (next_announce + 1) * nblk) announce(next_announce++);
        }
      }
    }
    tma_store_wait_all();
    fence_proxy_async_all();
    __threadfence();
    while (next_announce < f.n) announce(next_announce++);
  }
  // advance the launch number once every CTA of this launch has read the old one
  const unsigned long long prev =
      atomicAdd(reinterpret_cast<unsigned long long*>(f.local + F_AGDONE), 1ULL);
  if (prev == (unsigned long long)fa.n_comm - 1) {
    f.local[F_AGDONE] = 0;
    while (ld_acquire_gpu(f.local + F_AGCNT) < (uint64_t)gridDim.x) __nanosleep(64);
    f.local[F_AGCNT] = 0;
    st_release_gpu(f.local + F_AGSEQ, q);
  }
}

// ---- kernel ------------------------------------------------------------------------------------------

// CL = 2: thread-block cluster of two CTAs = one 256 x BN tile computed with cta_group::2 UMMA.
// Both CTAs run the TMA producer (own 128 rows of A + own half of B, transaction bytes counted on
// the leader's `full` barrier) and the epilogue (own 128 accumulator rows in own TMEM); only the
// leader (cluster rank 0) issues the MMAs and multicasts `commit` to both CTAs' barriers.
// (A multicast-only variant of this cluster shape was measured first: +4%, TMA multicast does not
// save L2 reads at cluster size 2 — profiles/r01_gemm_vs_cublas_v3_cluster_multicast.log.)
template <int BN, bool A_KMAJOR, bool B_KMAJOR, int MODE, int CL>
__global__ void __launch_bounds__(kGemmThreads, 1)
    k_gemm_bf16(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                const __grid_constant__ CUtensorMap tmap_c, const GemmParams p,
                const __grid_constant__ FusedArgs fa, const __grid_constant__ CMaps cm) {
  using Cfg = TileCfg<BN, CL>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  __shared__ uint64_t s_q;
  uint64_t q = 0;
  const int n_gemm_ctas = (int)gridDim.x - (MODE == MODE_AG ? fa.n_comm : fa.pf_ctas);

  if (MODE == MODE_AG) {
    if (threadIdx.x == 0) {
      s_q = ld_relaxed_gpu(fa.f.local + F_AGSEQ) + 1;
      atomicAdd(reinterpret_cast<unsigned long long*>(fa.f.local + F_AGCNT), 1ULL);
    }
    __syncthreads();
    q = s_q;
    // the comm CTAs are the producers the MMA CTAs spin on: they get the LOWEST block indices so
    // that they are scheduled first even when the grid is not fully co-resident
    if ((int)blockIdx.x < fa.n_comm) {
      ag_comm_role(fa, smem, (int)blockIdx.x, q);
      return;
    }
  }
  if (MODE == MODE_PLAIN && fa.pf_ctas > 0 && (int)blockIdx.x < fa.pf_ctas) {
    // prefetch CTAs (whole clusters when CL == 2): lowest block indices, no part in the GEMM
    pf_role(fa, smem, (int)blockIdx.x, fa.pf_ctas);
    return;
  }
  const int cta = (int)blockIdx.x - (MODE == MODE_AG ? fa.n_comm : fa.pf_ctas);

  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * kSmemABytes;
  uint8_t* smem_epi = smem + kStages * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_epi + Cfg::kEpiBufs * Cfg::kEpiBufBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kStages;
  uint64_t* tmem_full = bars + 2 * kStages;
  uint64_t* tmem_empty = bars + 2 * kStages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int k_blocks = (p.K + BK - 1) / BK;
  // work units: single tiles (CL == 1) or vertical tile pairs handled by one cluster (CL == 2)
  const int crank = (CL == 2) ? (int)cluster_ctarank() : 0;
  const int pm_tiles = (CL == 2) ? (p.m_tiles + 1) / 2 : p.m_tiles;
  const int num_tiles = pm_tiles * p.n_tiles;
  const int num_units = (MODE == MODE_PLAIN) ? num_tiles * p.splits : num_tiles;
  const int unit0 = (CL == 2) ? cta / 2 : cta;
  const int unit_stride = (CL == 2) ? n_gemm_ctas / 2 : n_gemm_ctas;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_a);
    prefetch_tmap(&tmap_b);
    prefetch_tmap(&tmap_c);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < kStages; ++s) {
        mbar_init(&full_bar[s], 1);
        mbar_init(&empty_bar[s], 1);
      }
      for (int s = 0; s < 2; ++s) {
        mbar_init(&tmem_full[s], 1);
        mbar_init(&tmem_empty[s], 4 * CL);  // one arrive per epilogue warp (of both CTAs if CL == 2)
      }
      fence_barrier_init();
    }
    __syncwarp();
    if (CL == 2) tmem_alloc_2cta(tmem_slot, Cfg::kTmemCols);
    else tmem_alloc(tmem_slot, Cfg::kTmemCols);
  }
  tcgen05_fence_before();
  __syncthreads();
  if (CL == 2) cluster_sync_all();  // the peer's barriers exist before anything is multicast at them
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int ready_chunk = -1;
      for (int u = unit0; u < num_units; u += unit_stride) {
        const int t = (MODE == MODE_PLAIN) ? u % num_tiles : u;
        int kb0 = 0, kb1 = k_blocks;
        if (MODE == MODE_PLAIN && p.splits > 1) {
          kb0 = (u / num_tiles) * p.kb_per_split;
          kb1 = kb0 + p.kb_per_split < k_blocks ? kb0 + p.kb_per_split : k_blocks;
        }
        int m_blk, n_blk;
        if (CL == 2) {
          m_blk = 2 * ((t % pm_tiles + p.m_rot) % pm_tiles) + crank;
          n_blk = t / pm_tiles;
        } else {
          tile_coords<MODE>(t, p, fa, m_blk, n_blk);
        }
        const CUtensorMap* bmap = &tmap_b;
        int b_row = n_blk * BN;
        if (MODE == MODE_AG) {
          const int c_lo = (n_blk * BN) / fa.ag_rows, c_hi = (n_blk * BN + BN - 1) / fa.ag_rows;
          if (c_lo == fa.f.me && c_hi == fa.f.me) {
            bmap = &cm.m[0];  // entirely inside my own shard: no transfer needed
            b_row = n_blk * BN - fa.f.me * fa.ag_rows;
          } else if (n_blk != ready_chunk) {
            for (int c = c_lo; c <= c_hi; ++c)
              spin_wait_gpu(fa.f.local + F_AGCHUNK + c, q);
            fence_proxy_async_all();
            ready_chunk = n_blk;
          }
        }
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem_a + stage * kSmemABytes;
          uint8_t* sb = smem_b + stage * Cfg::kSmemBBytes;
          if (CL == 2) {
            // both CTAs' loads complete on the leader's barrier, which expects both stages' bytes
            if (crank == 0) mbar_expect_tx(&full_bar[stage], 2 * Cfg::kStageBytes);
            if (A_KMAJOR) {
              tma_load_2d_2sm(&tmap_a, &full_bar[stage], sa, kb * BK, m_blk * BM);
            } else {
#pragma unroll
              for (int h = 0; h < BM / 64; ++h)
                tma_load_2d_2sm(&tmap_a, &full_bar[stage], sa + h * (64 * BK * 2),
                                m_blk * BM + h * 64, kb * BK);
            }
            const int b_half = b_row + crank * (BN / 2);
            if (B_KMAJOR) {
              tma_load_2d_2sm(bmap, &full_bar[stage], sb, kb * BK, b_half);
            } else {
#pragma unroll
              for (int h = 0; h < BN / 128; ++h)
                tma_load_2d_2sm(bmap, &full_bar[stage], sb + h * (64 * BK * 2), b_half + h * 64,
                                kb * BK);
            }
            if (++stage == kStages) {
              stage = 0;
              phase ^= 1;
            }
            continue;
          }
          mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
          if (A_KMAJOR) {
            tma_load_2d(&tmap_a, &full_bar[stage], sa, kb * BK, m_blk * BM);
          } else {
            // MN-major: one 64(m) x 64(k) swizzle atom column per box
#pragma unroll
            for (int h = 0; h < BM / 64; ++h)
              tma_load_2d(&tmap_a, &full_bar[stage], sa + h * (64 * BK * 2), m_blk * BM + h * 64,
                          kb * BK);
          }
          if (B_KMAJOR) {
            tma_load_2d(bmap, &full_bar[stage], sb, kb * BK, b_row);
          } else {
#pragma unroll
            for (int h = 0; h < BN / 64; ++h)
              tma_load_2d(bmap, &full_bar[stage], sb + h * (64 * BK * 2), b_row + h * 64, kb * BK);
          }
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1 && (CL == 1 || crank == 0)) {
    // ===== MMA issuer (leader CTA only when CL == 2) =====
    constexpr uint32_t idesc = make_idesc(BM * CL, BN, !A_KMAJOR, !B_KMAJOR);
    int stage = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (int u = unit0; u < num_units; u += unit_stride) {
      int kb0 = 0, kb1 = k_blocks;
      if (MODE == MODE_PLAIN && p.splits > 1) {
        kb0 = (u / num_tiles) * p.kb_per_split;
        kb1 = kb0 + p.kb_per_split < k_blocks ? kb0 + p.kb_per_split : k_blocks;
      }
      mbar_wait(&tmem_empty[as], aphase ^ 1);
      tcgen05_fence_after();
      const uint32_t tmem_d = tmem_base + as * BN;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        if (lane == 0) {
          const uint32_t a_addr = smem_u32(smem_a + stage * kSmemABytes);
          const uint32_t b_addr = smem_u32(smem_b + stage * Cfg::kSmemBBytes);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            uint64_t da, db;
            if (A_KMAJOR) da = make_smem_desc(a_addr + k * UMMA_K * 2, 0, 1024);
            else da = make_smem_desc(a_addr + k * UMMA_K * 128, 64 * BK * 2, 1024);
            if (B_KMAJOR) db = make_smem_desc(b_addr + k * UMMA_K * 2, 0, 1024);
            else db = make_smem_desc(b_addr + k * UMMA_K * 128, 64 * BK * 2, 1024);
            if (CL == 2) umma_f16_2cta(tmem_d, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            else umma_f16(tmem_d, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          // free the smem stage when these MMAs retire (in both CTAs of a pair)
          if (CL == 2) {
            umma_commit_2cta(&empty_bar[stage], (uint16_t)3);
            if (kb == kb1 - 1) umma_commit_2cta(&tmem_full[as], (uint16_t)3);
          } else {
            umma_commit(&empty_bar[stage]);
            if (kb == kb1 - 1) umma_commit(&tmem_full[as]);
          }
        }
        __syncwarp();
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (++as == 2) {
        as = 0;
        aphase ^= 1;
      }
    }
  } else if (warp >= 2) {
    // ===== epilogue warps 2..5: TMEM -> registers -> bf16 -> swizzled smem -> TMA store =====
    const int quad = warp & 3;            // TMEM lane quadrant this warp may access
    const int row_in_tile = quad * 32 + lane;
    const bool issuer = (warp == 2 && lane == 0);
    int as = 0;
    uint32_t aphase = 0;
    int ebuf = 0;
    for (int u = unit0; u < num_units; u += unit_stride) {
      const int t = (MODE == MODE_PLAIN) ? u % num_tiles : u;
      int m_blk, n_blk;
      if (CL == 2) {
        m_blk = 2 * ((t % pm_tiles + p.m_rot) % pm_tiles) + crank;
        n_blk = t / pm_tiles;
      } else {
        tile_coords<MODE>(t, p, fa, m_blk, n_blk);
      }
      if (MODE == MODE_PLAIN && p.splits > 1) {
        // split-K: this unit's fp32 partial goes straight from registers to the workspace (one
        // 256-byte run per thread and chunk); k_splitk_reduce adds the slices, bias and rounds
        mbar_wait(&tmem_full[as], aphase);
        tcgen05_fence_after();
        const int64_t r = (int64_t)m_blk * BM + row_in_tile;
        float* prow = p.partial + ((int64_t)(u / num_tiles) * p.M + r) * p.ldp;
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 64) {
          uint32_t v[64];
          const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN + c0);
          tmem_ld_32x32b_x32(taddr, v);
          tmem_ld_32x32b_x32(taddr + 32, v + 32);
          tmem_ld_wait();
          if (c0 + 64 >= BN) {
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (CL == 2) mbar_arrive_on_leader(&tmem_empty[as]);
              else mbar_arrive(&tmem_empty[as]);
            }
          }
          const int col0 = n_blk * BN + c0;
          if (r < p.M) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int col = col0 + 4 * j;
              if (col < p.ldp)  // ldp = N rounded up to 4: whole float4 groups only
                *reinterpret_cast<uint4*>(prow + col) =
                    make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
          }
        }
        if (++as == 2) {
          as = 0;
          aphase ^= 1;
        }
        continue;
      }
      const CUtensorMap* cmap = &tmap_c;
      int c_row = m_blk * BM;
      if (MODE == MODE_PLAIN && p.push_n > 0) {
        const int owner = m_blk / p.push_mtc;
        cmap = &cm.m[owner];
        c_row = (m_blk - owner * p.push_mtc) * BM;
      }
      // fused elementwise epilogue: this thread's 64 aux values of a chunk (one 128-byte row
      // segment) are requested one chunk AHEAD — the first one before the accumulator is even
      // complete — so that their latency hides behind the main loop / the previous chunk
      const bool has_aux = (MODE == MODE_PLAIN && p.epi_op != EPI_NONE);
      const int64_t arow_i = (int64_t)m_blk * BM + row_in_tile;
      const __nv_bfloat16* arow = has_aux ? p.aux + arow_i * p.ld_aux + (int64_t)n_blk * BN : nullptr;
      uint4 anext[8];
      auto load_aux = [&](int c0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (arow_i < p.M && n_blk * BN + c0 + 8 * j < p.N)
            anext[j] = __ldg(reinterpret_cast<const uint4*>(arow + c0 + 8 * j));
          else
            anext[j] = make_uint4(0, 0, 0, 0);
        }
      };
      if (has_aux) load_aux(0);
      mbar_wait(&tmem_full[as], aphase);
      tcgen05_fence_after();
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 64) {
        uint32_t v[64];
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN + c0);
        tmem_ld_32x32b_x32(taddr, v);
        tmem_ld_32x32b_x32(taddr + 32, v + 32);
        uint4 acur[8];
        if (has_aux) {
#pragma unroll
          for (int j = 0; j < 8; ++j) acur[j] = anext[j];
          if (c0 + 64 < BN) load_aux(c0 + 64);
        }
        tmem_ld_wait();
        if (c0 + 64 >= BN) {
          // all of this warp's accumulator columns are in registers: hand the TMEM stage back
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (CL == 2) mbar_arrive_on_leader(&tmem_empty[as]);
            else mbar_arrive(&tmem_empty[as]);
          }
        }
        // the staging buffer we are about to overwrite must have been read by its TMA store
        if (issuer) tma_store_wait_read<Cfg::kEpiBufs - 1>();
        epi_bar_sync();
        uint8_t* buf = smem_epi + ebuf * Cfg::kEpiBufBytes;
        uint8_t* rowp = buf + row_in_tile * 128;
        if (p.bias != nullptr) {
          const int col0 = n_blk * BN + c0;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (col0 + 8 * j < p.N) {  // N % 8 == 0 whenever a bias is passed
              const uint4 braw = __ldg(reinterpret_cast<const uint4*>(p.bias + col0 + 8 * j));
              const __nv_bfloat162* bb = reinterpret_cast<const __nv_bfloat162*>(&braw);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float2 f = __bfloat1622float2(bb[e]);
                v[8 * j + 2 * e] = __float_as_uint(__uint_as_float(v[8 * j + 2 * e]) + f.x);
                v[8 * j + 2 * e + 1] = __float_as_uint(__uint_as_float(v[8 * j + 2 * e + 1]) + f.y);
              }
            }
          }
        }
        if (has_aux) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const __nv_bfloat162* aa = reinterpret_cast<const __nv_bfloat162*>(&acur[j]);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = __bfloat1622float2(aa[e]);
              float x0 = __uint_as_float(v[8 * j + 2 * e]), x1 = __uint_as_float(v[8 * j + 2 * e + 1]);
              if (p.epi_op == EPI_ADD) {
                x0 += f.x;
                x1 += f.y;
              } else {
                // ATen multiplies the bf16-rounded GEMM result: reproduce that rounding
                x0 = __bfloat162float(__float2bfloat16_rn(x0)) * gelu_tanh_grad(f.x);
                x1 = __bfloat162float(__float2bfloat16_rn(x1)) * gelu_tanh_grad(f.y);
              }
              v[8 * j + 2 * e] = __float_as_uint(x0);
              v[8 * j + 2 * e + 1] = __float_as_uint(x1);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          uint4 o;
          __nv_bfloat162 h0 = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 0]), __uint_as_float(v[8 * j + 1]));
          __nv_bfloat162 h1 = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 2]), __uint_as_float(v[8 * j + 3]));
          __nv_bfloat162 h2 = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
          __nv_bfloat162 h3 = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7]));
          o.x = *reinterpret_cast<uint32_t*>(&h0);
          o.y = *reinterpret_cast<uint32_t*>(&h1);
          o.z = *reinterpret_cast<uint32_t*>(&h2);
          o.w = *reinterpret_cast<uint32_t*>(&h3);
          // 128-byte swizzle: 16-byte chunk j of row r lives at chunk (j ^ (r & 7))
          *reinterpret_cast<uint4*>(rowp + ((j ^ (row_in_tile & 7)) << 4)) = o;
        }
        fence_proxy_async();
        epi_bar_sync();
        if (issuer) {
          tma_store_2d(cmap, buf, n_blk * BN + c0, c_row);
          tma_store_commit();
        }
        ebuf ^= 1;
      }
      if (++as == 2) {
        as = 0;
        aphase ^= 1;
      }
    }
    if (issuer) {
      if (MODE == MODE_PLAIN && p.push_n > 0 && p.push_sync == 0) {
        tma_store_wait_read<0>();
      } else {
        tma_store_wait_all();
        if (MODE == MODE_PLAIN && p.push_n > 0 && p.push_sync >= 2) {
          // the tiles went into peer memory: make them visible system-wide before this CTA retires
          // (the next edb_epoch_barrier on the stream then orders them before its signal)
          fence_proxy_async_all();
          __threadfence_system();
        }
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (CL == 2) cluster_sync_all();  // nobody leaves while the peer may still signal its barriers
  if (warp == 1) {
    tcgen05_fence_after();
    if (CL == 2) tmem_dealloc_2cta(tmem_base, Cfg::kTmemCols);
    else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---- deferred reduce-scatter: reduce the receive slots of many pushed GEMMs in one launch -----------
// An edb_epoch_barrier earlier on the stream made every slot complete: purely local memory traffic.
constexpr int kRsMaxItems = 160;
constexpr int kRsFinishThreads = 256;
constexpr int64_t kRsFinishChunkVecs = 4096;  // 64 KiB of bf16 per slot and work unit

template <typename Out>
__device__ __forceinline__ void rs_store(Out* out, int64_t i, const float* acc) {
  if (sizeof(Out) == 4) {
    float4* o = reinterpret_cast<float4*>(out) + 2 * i;
    o[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    o[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  } else {
    uint4 o;
    __nv_bfloat162 h0 = __floats2bfloat162_rn(acc[0], acc[1]);
    __nv_bfloat162 h1 = __floats2bfloat162_rn(acc[2], acc[3]);
    __nv_bfloat162 h2 = __floats2bfloat162_rn(acc[4], acc[5]);
    __nv_bfloat162 h3 = __floats2bfloat162_rn(acc[6], acc[7]);
    o.x = *reinterpret_cast<uint32_t*>(&h0);
    o.y = *reinterpret_cast<uint32_t*>(&h1);
    o.z = *reinterpret_cast<uint32_t*>(&h2);
    o.w = *reinterpret_cast<uint32_t*>(&h3);
    reinterpret_cast<uint4*>(out)[i] = o;
  }
}

struct RsFinishItem {
  const char* recv;     // n slots of chunk_bytes (local)
  void* dst;            // [chunk_bytes / 2] elements of out_dtype
  int64_t chunk_bytes;
};
struct RsFinishDesc {
  int n;  // group size = number of slots
  int n_items;
  float scale;
  int out_dtype;
  int first_unit[kRsMaxItems + 1];
  RsFinishItem it[kRsMaxItems];
};

// NSRC > 0: group size known at compile time, so that exactly NSRC x U 16-byte loads are in flight
// per thread (8 for every instantiation: the slots are read once, nothing is reused, the kernel
// lives on memory-level parallelism); NSRC == 0: any group size, one vector at a time.
template <int NSRC>
__global__ void __launch_bounds__(kRsFinishThreads, 4)
    k_rs_finish(const __grid_constant__ RsFinishDesc d) {
  const int total_units = d.first_unit[d.n_items];
  const int n = NSRC > 0 ? NSRC : d.n;
  constexpr int MAXS = NSRC > 0 ? NSRC : kMaxGroup;
  constexpr int U = NSRC > 0 ? (8 / NSRC > 0 ? 8 / NSRC : 1) : 1;
  for (int u = blockIdx.x; u < total_units; u += gridDim.x) {
    int lo = 0, hi = d.n_items;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (d.first_unit[mid] <= u) lo = mid;
      else hi = mid;
    }
    const char* recv = d.it[lo].recv;
    void* dst = d.it[lo].dst;
    const int64_t chunk_bytes = d.it[lo].chunk_bytes;
    const int64_t nvec = chunk_bytes / 16;
    const int64_t v0 = (int64_t)(u - d.first_unit[lo]) * kRsFinishChunkVecs;
    const int64_t v1 = v0 + kRsFinishChunkVecs < nvec ? v0 + kRsFinishChunkVecs : nvec;
    for (int64_t i0 = v0 + threadIdx.x; i0 < v1; i0 += U * kRsFinishThreads) {
      uint4 raw[U][MAXS];
#pragma unroll
      for (int uu = 0; uu < U; ++uu) {
        const int64_t i = i0 + uu * kRsFinishThreads;
        if (i < v1) {
#pragma unroll
          for (int sidx = 0; sidx < MAXS; ++sidx)
            if (sidx < n)
              raw[uu][sidx] = __ldcs(reinterpret_cast<const uint4*>(recv + (int64_t)sidx * chunk_bytes + i * 16));
        }
      }
#pragma unroll
      for (int uu = 0; uu < U; ++uu) {
        const int64_t i = i0 + uu * kRsFinishThreads;
        if (i >= v1) break;
        float acc[8];
#pragma unroll
        for (int sidx = 0; sidx < MAXS; ++sidx) {
          if (sidx < n) {
            const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw[uu][sidx]);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 v = __bfloat1622float2(h[e]);
              if (sidx == 0) {
                acc[2 * e] = v.x;
                acc[2 * e + 1] = v.y;
              } else {
                acc[2 * e] += v.x;
                acc[2 * e + 1] += v.y;
              }
            }
          }
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] *= d.scale;
        if (d.out_dtype == EDB_F32) rs_store<float>(static_cast<float*>(dst), i, acc);
        else rs_store<__nv_bfloat16>(static_cast<__nv_bfloat16*>(dst), i, acc);
      }
    }
  }
}

// push mode: row r of C belongs to member r / rows_per and goes to base[owner] + (r % rows_per) * ldc
struct PushDst {
  int n;
  int64_t rows_per, row_rot;
  __nv_bfloat16* base[kMaxGroup];
};

__global__ void __launch_bounds__(256)
    k_splitk_reduce(__nv_bfloat16* __restrict__ C, int64_t ldc, const float* __restrict__ partial,
                    int64_t ldp, int splits, int M, int N, const __nv_bfloat16* __restrict__ bias,
                    const __grid_constant__ PushDst pd) {
  const int64_t groups_per_row = ldp / 4;
  const int64_t total = (int64_t)M * groups_per_row;
  const int64_t slice = (int64_t)M * ldp;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / groups_per_row;
    const int c = (int)(i - r * groups_per_row) * 4;
    if (pd.n > 0) r = (r + pd.row_rot) % M;  // start at the next member's rows (no incast)
    const float* src = partial + r * ldp + c;
    float4 acc = *reinterpret_cast<const float4*>(src);
    for (int s = 1; s < splits; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(src + s * slice);
      acc.x += v.x;
      acc.y += v.y;
      acc.z += v.z;
      acc.w += v.w;
    }
    float o[4] = {acc.x, acc.y, acc.z, acc.w};
    __nv_bfloat16* dst = C + r * ldc + c;
    if (pd.n > 0) {
      const int64_t owner = r / pd.rows_per;
      dst = pd.base[owner] + (r - owner * pd.rows_per) * ldc + c;
    }
    if (c + 3 < N) {
      // whole group inside the row: one 8-byte store (ldc % 8 == 0 and c % 4 == 0 => aligned)
      if (bias) {
#pragma unroll
        for (int e = 0; e < 4; ++e) o[e] += __bfloat162float(bias[c + e]);
      }
      __nv_bfloat162 h0 = __floats2bfloat162_rn(o[0], o[1]);
      __nv_bfloat162 h1 = __floats2bfloat162_rn(o[2], o[3]);
      uint2 v;
      v.x = *reinterpret_cast<uint32_t*>(&h0);
      v.y = *reinterpret_cast<uint32_t*>(&h1);
      *reinterpret_cast<uint2*>(dst) = v;
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (c + e < N) {
          if (bias) o[e] += __bfloat162float(bias[c + e]);
          dst[e] = __float2bfloat16_rn(o[e]);
        }
      }
    }
  }
}

// ---- host side ---------------------------------------------------------------------------------------

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// 2-D bf16 tensor map: `inner` contiguous elements, `outer` rows `ld` elements apart.
static int make_tmap(CUtensorMap* map, const void* base, int64_t inner, int64_t outer, int64_t ld,
                     int box_inner, int box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(EDB_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS)
    return set_error(EDB_E_CUDA, "cuTensorMapEncodeTiled failed (%d) inner=%lld outer=%lld ld=%lld",
                     (int)rc, (long long)inner, (long long)outer, (long long)ld);
  return EDB_OK;
}

template <int BN, bool AK, bool BK_, int MODE, int CL>
static int launch_gemm_cl(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc,
                          const GemmParams& p, const FusedArgs& fa, const CMaps& cm, int grid,
                          cudaStream_t st) {
  using Cfg = TileCfg<BN, CL>;
  static bool configured = false;
  auto kern = k_gemm_bf16<BN, AK, BK_, MODE, CL>;
  if (!configured) {
    EDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured = true;
  }
  if (CL == 1) {
    kern<<<grid, kGemmThreads, Cfg::kSmemBytes, st>>>(ta, tb, tc, p, fa, cm);
  } else {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    EDB_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, p, fa, cm));
  }
  count_launch();
  return cuda_check(cudaGetLastError(), "k_gemm_bf16 launch");
}

template <int BN, bool AK, bool BK_>
static int launch_gemm_plain(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc,
                             const GemmParams& p, const FusedArgs& fa, const CMaps& cm, int grid,
                             cudaStream_t st, int cl) {
  if (cl == 2) return launch_gemm_cl<BN, AK, BK_, MODE_PLAIN, 2>(ta, tb, tc, p, fa, cm, grid, st);
  return launch_gemm_cl<BN, AK, BK_, MODE_PLAIN, 1>(ta, tb, tc, p, fa, cm, grid, st);
}

static int dispatch_gemm_plain(int bn, bool a_k, bool b_k, const CUtensorMap& ta,
                               const CUtensorMap& tb, const CUtensorMap& tc, const GemmParams& p,
                               const FusedArgs& fa, const CMaps& cm, int grid, cudaStream_t st,
                               int cl) {
  const int key = (bn == 256 ? 4 : 0) | (a_k ? 2 : 0) | (b_k ? 1 : 0);
  switch (key) {
    case 7: return launch_gemm_plain<256, true, true>(ta, tb, tc, p, fa, cm, grid, st, cl);
    case 6: return launch_gemm_plain<256, true, false>(ta, tb, tc, p, fa, cm, grid, st, cl);
    case 5: return launch_gemm_plain<256, false, true>(ta, tb, tc, p, fa, cm, grid, st, cl);
    case 4: return launch_gemm_plain<256, false, false>(ta, tb, tc, p, fa, cm, grid, st, cl);
    case 3: return launch_gemm_plain<128, true, true>(ta, tb, tc, p, fa, cm, grid, st, cl);
    case 2: return launch_gemm_plain<128, true, false>(ta, tb, tc, p, fa, cm, grid, st, cl);
    case 1: return launch_gemm_plain<128, false, true>(ta, tb, tc, p, fa, cm, grid, st, cl);
    default: return launch_gemm_plain<128, false, false>(ta, tb, tc, p, fa, cm, grid, st, cl);
  }
}

static int pick_bn(int64_t M, int64_t N, int sms) {
  // 128-wide tiles need 128 B/cycle of operand traffic per SM (A 16 KiB + B 16 KiB per 256 MMA
  // cycles) and run at ~half the rate of 256-wide ones (96 B/cycle) even when they quantise better
  // into waves (measured: profiles/r01_gemm_tile_cluster_sweep.log), so 256 unless N is tiny.
  (void)M;
  (void)sms;
  return N <= 128 ? 128 : 256;
}

static int check_operands(const void* A, const void* B, const void* C, const void* bias, int64_t M,
                          int64_t N, int64_t K, int64_t lda, int64_t ldb, int64_t ldc,
                          const char* who) {
  if (M <= 0 || N <= 0 || K <= 0) return set_error(EDB_E_UNSUPPORTED, "%s: empty problem", who);
  if (M > 0x7fffffff || N > 0x7fffffff || K > 0x7fffffff)
    return set_error(EDB_E_UNSUPPORTED, "%s: dimension too large", who);
  if (((uintptr_t)A | (uintptr_t)B | (uintptr_t)C) & 15)
    return set_error(EDB_E_UNSUPPORTED, "%s: base pointers must be 16-byte aligned", who);
  // TMA: global strides must be multiples of 16 bytes; extents (M, N, K) may be anything — boxes
  // that run past an extent are zero-filled on load and clipped on store.
  if ((lda | ldb | ldc) & 7)
    return set_error(EDB_E_UNSUPPORTED, "%s: lda/ldb/ldc must be multiples of 8", who);
  if (bias && ((N & 7) || ((uintptr_t)bias & 15)))
    return set_error(EDB_E_UNSUPPORTED, "%s: bias needs N %% 8 == 0 and 16-byte alignment", who);
  return EDB_OK;
}

// fp32 workspace of split-K GEMMs: one slab per (device, stream) pair, allocated on first use
// (outside any stream capture: the compiled step always runs eagerly once before it is captured).
constexpr size_t kSplitKBytes = (size_t)64 << 20;
struct SplitKSlab {
  int device;
  cudaStream_t stream;
  float* ptr;
};
static SplitKSlab g_splitk[16];
static int g_splitk_n = 0;

static float* splitk_workspace(cudaStream_t st) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  for (int i = 0; i < g_splitk_n; ++i)
    if (g_splitk[i].device == dev && g_splitk[i].stream == st) return g_splitk[i].ptr;
  if (g_splitk_n == 16) return nullptr;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
    cudaGetLastError();
    return nullptr;  // cannot allocate while capturing: this launch runs unsplit
  }
  float* ptr = nullptr;
  if (cudaMalloc(&ptr, kSplitKBytes) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  g_splitk[g_splitk_n++] = {dev, st, ptr};
  return ptr;
}

static int sm_count_now() {
  Runtime& r = rt();
  if (!r.inited) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess)
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    r.sm_count = sms;
  }
  return r.sm_count;
}

}  // namespace edb

using namespace edb;

extern "C" {

// push: NULL, or the receive slots of the group members (C rows are spread over them)
struct PushSpec {
  int n, me;
  int64_t rows_per;          // M / n, a multiple of BM
  char* slot[kMaxGroup];     // member p's receive slot for MY rows: [rows_per, N] bf16, ld = N
};

// pf: NULL, or the all-gather prefetch that rides on this GEMM
// epi: NULL, or the fused elementwise epilogue
struct EpiSpec {
  int op;
  const void* aux;
  int64_t ld_aux;
};

struct PfSpec {
  int gid, n_items;
  const uint64_t* src_offs;
  const uint64_t* dst_offs;
  const int64_t* bytes;
  const int64_t* dst_strides;
  const int64_t* src_strides;  // may be NULL (all 0)
};

static int fill_prefetch(FusedArgs* fa, const PfSpec* pf, int want_ctas) {
  Runtime& r = rt();
  if (!r.inited) return set_error(EDB_E_STATE, "runtime not initialised (call edb_init)");
  if (pf->gid < 0 || pf->gid >= r.ngroups) return set_error(EDB_E_INVALID, "bad group id %d", pf->gid);
  if (pf->n_items < 0 || pf->n_items > kMaxPfItems)
    return set_error(EDB_E_UNSUPPORTED, "prefetch: at most %d items per launch", kMaxPfItems);
  const Group& g = r.groups[pf->gid];
  fa->f.n = g.n;
  fa->f.me = g.me;
  fa->pf_n = g.n;
  fa->pf_items = pf->n_items;
  fa->pf_local = r.heap;
  for (int p = 0; p < g.n; ++p) fa->pf_heap[p] = r.peer_heap[g.ranks[p]];
  int64_t blocks = 0;
  for (int i = 0; i < pf->n_items; ++i) {
    const int64_t b = pf->bytes[i], st = pf->dst_strides[i];
    if (b <= 0 || (b & 15) || (pf->src_offs[i] & 15) || (pf->dst_offs[i] & 15) || (st & 15) || st < b)
      return set_error(EDB_E_INVALID, "prefetch item %d: ranges must be 16-byte aligned, stride >= bytes", i);
    if (pf->src_offs[i] < kUserOffset || pf->src_offs[i] + (uint64_t)b > r.heap_bytes ||
        pf->dst_offs[i] < kUserOffset ||
        pf->dst_offs[i] + (uint64_t)st * (g.n - 1) + (uint64_t)b > r.heap_bytes)
      return set_error(EDB_E_INVALID, "prefetch item %d: symmetric range out of bounds", i);
    const int64_t sst = pf->src_strides ? pf->src_strides[i] : 0;
    if (sst < 0 || (sst & 15) ||
        pf->src_offs[i] + (uint64_t)sst * (g.n - 1) + (uint64_t)b > r.heap_bytes)
      return set_error(EDB_E_INVALID, "prefetch item %d: bad source stride", i);
    fa->pf_src[i] = pf->src_offs[i];
    fa->pf_dst[i] = pf->dst_offs[i];
    fa->pf_bytes[i] = b;
    fa->pf_stride[i] = st;
    fa->pf_sstride[i] = sst;
    fa->pf_inplace[i] = (sst == st && pf->src_offs[i] == pf->dst_offs[i]) ? 1 : 0;
    blocks += (b + 16383) / 16384 * (fa->pf_inplace[i] ? g.n - 1 : g.n);
  }
  int ctas = want_ctas;
  if (blocks < ctas) ctas = (int)blocks;
  ctas &= ~1;  // whole clusters when the GEMM runs CTA pairs
  if (ctas < 2 && blocks > 0) ctas = 2;
  fa->pf_ctas = pf->n_items > 0 ? ctas : 0;
  return EDB_OK;
}

static int gemm_plain_impl(void* C, const void* A, const void* B, const void* bias, int64_t M,
                           int64_t N, int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int a_kmajor,
                           int b_kmajor, void* stream, const PushSpec* push,
                           const PfSpec* pf = nullptr, const EpiSpec* epi = nullptr) {
  int rc = check_operands(A, B, C, bias, M, N, K, lda, ldb, ldc, "edb_gemm_bf16");
  if (rc) return rc;
  const int sms = sm_count_now();
  int bn = pick_bn(M, N, sms);
  if (rt().gemm_force_bn == 128 || rt().gemm_force_bn == 256) bn = (int)rt().gemm_force_bn;
  // CTA pairs (cta_group::2) whenever there are at least two tile rows (push: an even number, so
  // that no pair has a phantom tile whose owner index would be out of range)
  int cl = (rt().gemm_cluster >= 2 && M > BM) ? 2 : 1;
  if (push && ((M / BM) & 1)) cl = 1;
  CUtensorMap ta, tb, tc;
  if (a_kmajor) rc = make_tmap(&ta, A, K, M, lda, BK, BM);
  else rc = make_tmap(&ta, A, M, K, lda, 64, BK);
  if (rc) return rc;
  if (b_kmajor) rc = make_tmap(&tb, B, K, N, ldb, BK, bn / cl);
  else rc = make_tmap(&tb, B, N, K, ldb, 64, BK);
  if (rc) return rc;
  rc = make_tmap(&tc, C, N, push ? push->rows_per : M, ldc, 64, BM);
  if (rc) return rc;
  GemmParams p;
  p.C = static_cast<__nv_bfloat16*>(C);
  p.bias = static_cast<const __nv_bfloat16*>(bias);
  p.ldc = ldc;
  p.M = (int)M;
  p.N = (int)N;
  p.K = (int)K;
  p.m_tiles = (int)((M + BM - 1) / BM);
  p.n_tiles = (int)((N + bn - 1) / bn);
  p.push_n = 0;
  p.push_mtc = 1;
  p.m_rot = 0;
  p.push_sync = (int)rt().push_sync;
  p.aux = nullptr;
  p.ld_aux = 0;
  p.epi_op = EPI_NONE;
  if (epi && epi->op != EPI_NONE) {
    if (epi->op != EPI_ADD && epi->op != EPI_GELU_BWD)
      return set_error(EDB_E_INVALID, "edb_gemm_epi_bf16: unknown epilogue op %d", epi->op);
    if ((N & 7) || ((uintptr_t)epi->aux & 15) || (epi->ld_aux & 7) || epi->ld_aux < N || !epi->aux)
      return set_error(EDB_E_UNSUPPORTED,
                       "edb_gemm_epi_bf16: aux needs N %% 8 == 0, 16-byte alignment, ld %% 8 == 0");
    p.aux = static_cast<const __nv_bfloat16*>(epi->aux);
    p.ld_aux = epi->ld_aux;
    p.epi_op = epi->op;
  }
  FusedArgs fa;
  memset(&fa, 0, sizeof(fa));
  CMaps cm;
  memset(&cm, 0, sizeof(cm));
  PushDst pd;
  memset(&pd, 0, sizeof(pd));
  int sms_gemm = sms;  // SMs left to the GEMM when prefetch CTAs ride along
  if (pf && pf->n_items > 0) {
    int want = (int)rt().comm_ctas;
    if (want < 2) want = 2;
    if (want > sms / 4) want = sms / 4;
    rc = fill_prefetch(&fa, pf, want);
    if (rc) return rc;
    sms_gemm = sms - fa.pf_ctas;
  }
  if (push) {
    p.push_n = push->n;
    p.push_mtc = (int)(push->rows_per / BM);
    // start with the rows of the next member, end with my own (a local store)
    const int first_m = ((push->me + 1) % push->n) * p.push_mtc;
    p.m_rot = (cl == 2) ? first_m / 2 : first_m;
    pd.n = push->n;
    pd.rows_per = push->rows_per;
    pd.row_rot = (int64_t)first_m * BM;
    for (int q = 0; q < push->n; ++q) {
      rc = make_tmap(&cm.m[q], push->slot[q], N, push->rows_per, N, 64, BM);
      if (rc) return rc;
      pd.base[q] = reinterpret_cast<__nv_bfloat16*>(push->slot[q]);
    }
  }
  p.splits = 1;
  p.kb_per_split = 0;
  p.partial = nullptr;
  p.ldp = (N + 3) / 4 * 4;
  cudaStream_t st = (cudaStream_t)stream;
  // split-K: when the tiles occupy at most half of the SMs and K is long (weight gradients:
  // M, N = layer widths, K = tokens), slices of K go to the idle SMs.  Each slice keeps >= 8
  // k-blocks so that the pipeline fill and the fp32 partial traffic stay small against the MMAs.
  const int units = (cl == 2 ? ((p.m_tiles + 1) / 2) : p.m_tiles) * p.n_tiles;
  const int ctas = units * cl;
  const int k_blocks = (int)((K + BK - 1) / BK);
  if (rt().gemm_splitk && 2 * ctas <= sms_gemm && k_blocks >= 16 && p.epi_op == EPI_NONE) {
    int splits = sms_gemm / ctas;
    if (splits > k_blocks / 8) splits = k_blocks / 8;
    if (splits > 8) splits = 8;
    while (splits > 1 && (size_t)splits * (size_t)M * (size_t)p.ldp * sizeof(float) > kSplitKBytes)
      --splits;
    if (splits > 1) {
      float* ws = splitk_workspace(st);
      if (ws != nullptr) {
        p.kb_per_split = (k_blocks + splits - 1) / splits;
        p.splits = (k_blocks + p.kb_per_split - 1) / p.kb_per_split;  // no empty slice
        p.partial = ws;
      }
    }
  }
  int grid;
  if (cl == 2) {
    const int pairs = units * p.splits;
    const int clusters = pairs < sms_gemm / 2 ? pairs : sms_gemm / 2;
    grid = 2 * clusters;
  } else {
    const int tiles = units * p.splits;
    grid = tiles < sms_gemm ? tiles : sms_gemm;
  }
  grid += fa.pf_ctas;
  rc = dispatch_gemm_plain(bn, a_kmajor != 0, b_kmajor != 0, ta, tb, tc, p, fa, cm, grid, st, cl);
  if (rc || p.splits == 1) return rc;
  const int64_t groups = (int64_t)M * (p.ldp / 4);
  int rgrid = (int)((groups + 255) / 256);
  if (rgrid > 4 * sms) rgrid = 4 * sms;
  k_splitk_reduce<<<rgrid, 256, 0, st>>>(p.C, ldc, p.partial, p.ldp, p.splits, (int)M, (int)N, p.bias,
                                        pd);
  count_launch();
  return cuda_check(cudaGetLastError(), "k_splitk_reduce launch");
}

int edb_gemm_bf16(void* C, const void* A, const void* B, const void* bias, int64_t M, int64_t N,
                  int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int a_kmajor, int b_kmajor,
                  int accumulate_into_c, void* stream) {
  if (accumulate_into_c) return set_error(EDB_E_UNSUPPORTED, "edb_gemm_bf16: accumulate_into_c");
  return gemm_plain_impl(C, A, B, bias, M, N, K, lda, ldb, ldc, a_kmajor, b_kmajor, stream, nullptr);
}

int edb_gemm_pf_bf16(void* C, const void* A, const void* B, const void* bias, int64_t M, int64_t N,
                     int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int a_kmajor, int b_kmajor,
                     int gid, int n_items, const uint64_t* src_offs, const uint64_t* dst_offs,
                     const int64_t* bytes, const int64_t* dst_strides, const int64_t* src_strides,
                     void* stream) {
  PfSpec pf = {gid, n_items, src_offs, dst_offs, bytes, dst_strides, src_strides};
  return gemm_plain_impl(C, A, B, bias, M, N, K, lda, ldb, ldc, a_kmajor, b_kmajor, stream, nullptr,
                         n_items > 0 ? &pf : nullptr);
}

int edb_gemm_epi_bf16(void* C, const void* A, const void* B, const void* bias, const void* aux,
                      int64_t ld_aux, int epi_op, int64_t M, int64_t N, int64_t K, int64_t lda,
                      int64_t ldb, int64_t ldc, int a_kmajor, int b_kmajor, int gid, int n_items,
                      const uint64_t* src_offs, const uint64_t* dst_offs, const int64_t* bytes,
                      const int64_t* dst_strides, const int64_t* src_strides, void* stream) {
  PfSpec pf = {gid, n_items, src_offs, dst_offs, bytes, dst_strides, src_strides};
  EpiSpec epi = {epi_op, aux, ld_aux};
  return gemm_plain_impl(C, A, B, bias, M, N, K, lda, ldb, ldc, a_kmajor, b_kmajor, stream, nullptr,
                         n_items > 0 ? &pf : nullptr, &epi);
}

int edb_ag_prefetch(int gid, int n_items, const uint64_t* src_offs, const uint64_t* dst_offs,
                    const int64_t* bytes, const int64_t* dst_strides, const int64_t* src_strides,
                    void* stream) {
  if (n_items <= 0) return EDB_OK;
  Runtime& r = rt();
  static bool configured = false;
  const int smem = kPfSlots * 16384 + 1024 + 128;
  if (!configured) {
    EDB_CUDA(cudaFuncSetAttribute(k_ag_prefetch, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  for (int done = 0; done < n_items; done += kMaxPfItems) {
    const int k = n_items - done < kMaxPfItems ? n_items - done : kMaxPfItems;
    PfSpec pf = {gid, k, src_offs + done, dst_offs + done, bytes + done, dst_strides + done,
                 src_strides ? src_strides + done : nullptr};
    FusedArgs fa;
    memset(&fa, 0, sizeof(fa));
    // nothing else needs the SMs: one CTA per SM (1 thread each drives a 5-deep 16 KiB ring)
    int rc = fill_prefetch(&fa, &pf, r.sm_count);
    if (rc) return rc;
    if (fa.pf_ctas == 0) continue;
    k_ag_prefetch<<<fa.pf_ctas, 32, smem, (cudaStream_t)stream>>>(fa);
    count_launch();
    rc = cuda_check(cudaGetLastError(), "k_ag_prefetch launch");
    if (rc) return rc;
  }
  return EDB_OK;
}

int edb_gemm_push_bf16(int gid, uint64_t recv_off, const void* A, const void* B, int64_t M,
                       int64_t N, int64_t K, int64_t lda, int64_t ldb, int a_kmajor, int b_kmajor,
                       void* stream) {
  Runtime& r = rt();
  if (!r.inited) return set_error(EDB_E_STATE, "runtime not initialised (call edb_init)");
  if (gid < 0 || gid >= r.ngroups) return set_error(EDB_E_INVALID, "bad group id %d", gid);
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  if (M % n || (M / n) % BM)
    return set_error(EDB_E_UNSUPPORTED, "edb_gemm_push_bf16: rows per rank must be a multiple of 128");
  if (N & 7) return set_error(EDB_E_UNSUPPORTED, "edb_gemm_push_bf16: N must be a multiple of 8");
  const int64_t rows = M / n;
  const size_t chunk_bytes = (size_t)rows * N * 2;
  if (recv_off < kUserOffset || recv_off + chunk_bytes * n > r.heap_bytes || (recv_off & 1023))
    return set_error(EDB_E_INVALID, "edb_gemm_push_bf16: bad symmetric offset");
  PushSpec ps;
  memset(&ps, 0, sizeof(ps));
  ps.n = n;
  ps.me = me;
  ps.rows_per = rows;
  for (int q = 0; q < n; ++q)
    ps.slot[q] = r.peer_heap[g.ranks[q]] + recv_off + (size_t)me * chunk_bytes;
  // C itself is never written in push mode; my own slot stands in for the checks / the unused map
  return gemm_plain_impl(ps.slot[me], A, B, nullptr, M, N, K, lda, ldb, N, a_kmajor, b_kmajor, stream,
                         &ps);
}

int edb_ag_gemm_epoch_bf16(int gid, void* C, const void* A, const void* bias, uint64_t b_shard_off,
                           uint64_t b_full_off, int64_t M, int64_t N, int64_t K, int64_t lda,
                           int64_t ldc, void* stream) {
  FusedArgs fa;
  memset(&fa, 0, sizeof(fa));
  int rc = fill_flagctx(&fa.f, gid);
  if (rc) return rc;
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  if (N % n) return set_error(EDB_E_UNSUPPORTED, "edb_ag_gemm_epoch_bf16: N %% group size != 0");
  const int64_t rows = N / n;
  int bn = 0;
  if (N % 256 == 0) bn = 256;
  else if (N % 128 == 0) bn = 128;
  else return set_error(EDB_E_UNSUPPORTED, "edb_ag_gemm_epoch_bf16: N=%lld not a multiple of 128",
                        (long long)N);
  if (rows % 8)
    return set_error(EDB_E_UNSUPPORTED, "edb_ag_gemm_epoch_bf16: shard rows %lld not a multiple of 8",
                     (long long)rows);
  if (K & 7) return set_error(EDB_E_UNSUPPORTED, "edb_ag_gemm_epoch_bf16: K must be a multiple of 8");
  const size_t shard_bytes = (size_t)rows * K * 2;
  if (b_shard_off < kUserOffset || b_shard_off + shard_bytes > r.heap_bytes || (b_shard_off & 15) ||
      b_full_off < kUserOffset || b_full_off + shard_bytes * n > r.heap_bytes || (b_full_off & 1023))
    return set_error(EDB_E_INVALID, "edb_ag_gemm_epoch_bf16: bad symmetric offsets");
  const char* shard = r.heap + b_shard_off;
  char* full = r.heap + b_full_off;
  rc = check_operands(A, full, C, bias, M, N, K, lda, K, ldc, "edb_ag_gemm_epoch_bf16");
  if (rc) return rc;
  CUtensorMap ta, tb, tc;
  rc = make_tmap(&ta, A, K, M, lda, BK, BM);
  if (rc) return rc;
  rc = make_tmap(&tb, full, K, N, K, BK, bn);
  if (rc) return rc;
  rc = make_tmap(&tc, C, N, M, ldc, 64, BM);
  if (rc) return rc;
  CMaps cm;
  memset(&cm, 0, sizeof(cm));
  rc = make_tmap(&cm.m[0], shard, K, rows, K, BK, bn);
  if (rc) return rc;
  GemmParams p;
  p.C = static_cast<__nv_bfloat16*>(C);
  p.bias = static_cast<const __nv_bfloat16*>(bias);
  p.ldc = ldc;
  p.M = (int)M;
  p.N = (int)N;
  p.K = (int)K;
  p.m_tiles = (int)((M + BM - 1) / BM);
  p.n_tiles = (int)(N / bn);
  p.splits = 1;
  p.kb_per_split = 0;
  p.partial = nullptr;
  p.ldp = 0;
  p.push_n = 0;
  p.push_mtc = 1;
  p.m_rot = 0;
  p.push_sync = 0;
  p.aux = nullptr;
  p.ld_aux = 0;
  p.epi_op = EPI_NONE;
  const int sms = r.sm_count;
  int n_comm = (int)r.comm_ctas;
  if (n_comm < 1) n_comm = 1;
  if (n_comm > sms / 4) n_comm = sms / 4;
  if (n == 1) n_comm = 1;
  fa.n_comm = n_comm;
  for (int pidx = 0; pidx < n; ++pidx) fa.shard_src[pidx] = r.peer_heap[g.ranks[pidx]] + b_shard_off;
  fa.shard_src[me] = shard;
  fa.full_dst = full;
  fa.shard_bytes = (int64_t)shard_bytes;
  fa.ag_rows = (int)rows;
  fa.ag_first_tile = (int)(((int64_t)me * rows) / bn);
  const int tiles = p.m_tiles * p.n_tiles;
  int gemm_ctas = sms - n_comm;
  if (gemm_ctas > tiles) gemm_ctas = tiles;
  // A and B are K-major (C = A.Bᵀ, nn.Linear fwd): the only layout this kernel is built for
  if (bn == 256)
    return launch_gemm_cl<256, true, true, MODE_AG, 1>(ta, tb, tc, p, fa, cm, gemm_ctas + n_comm,
                                                       (cudaStream_t)stream);
  return launch_gemm_cl<128, true, true, MODE_AG, 1>(ta, tb, tc, p, fa, cm, gemm_ctas + n_comm,
                                                     (cudaStream_t)stream);
}

int edb_rs_finish_local(int gid, int n_items, void* const* dsts, const uint64_t* recv_offs,
                        const int64_t* chunk_bytes, float post_scale, int out_dtype, void* stream) {
  if (n_items <= 0) return EDB_OK;
  if (out_dtype != EDB_BF16 && out_dtype != EDB_F32)
    return set_error(EDB_E_UNSUPPORTED, "edb_rs_finish_local: out dtype must be bf16 or f32");
  Runtime& r = rt();
  if (!r.inited) return set_error(EDB_E_STATE, "runtime not initialised (call edb_init)");
  if (gid < 0 || gid >= r.ngroups) return set_error(EDB_E_INVALID, "bad group id %d", gid);
  const int n = r.groups[gid].n;
  cudaStream_t st = (cudaStream_t)stream;
  int done = 0;
  while (done < n_items) {
    RsFinishDesc d;
    d.n = n;
    d.scale = post_scale;
    d.out_dtype = out_dtype;
    d.first_unit[0] = 0;
    int k = 0;
    int64_t units = 0;
    for (; done < n_items && k < kRsMaxItems; ++done, ++k) {
      const int64_t cb = chunk_bytes[done];
      if (cb <= 0 || (cb & 15) || ((uintptr_t)dsts[done] & 15))
        return set_error(EDB_E_INVALID, "edb_rs_finish_local: item %d: chunk bytes / dst alignment", done);
      if (recv_offs[done] < kUserOffset || recv_offs[done] + (uint64_t)cb * n > r.heap_bytes ||
          (recv_offs[done] & 15))
        return set_error(EDB_E_INVALID, "edb_rs_finish_local: item %d: bad symmetric offset", done);
      d.it[k].recv = r.heap + recv_offs[done];
      d.it[k].dst = dsts[done];
      d.it[k].chunk_bytes = cb;
      units += (cb / 16 + kRsFinishChunkVecs - 1) / kRsFinishChunkVecs;
      if (units > 0x7fffffffLL) return set_error(EDB_E_UNSUPPORTED, "edb_rs_finish_local: too much work");
      d.first_unit[k + 1] = (int)units;
    }
    d.n_items = k;
    int grid = (int)(units < 4LL * r.sm_count ? units : 4LL * r.sm_count);
    switch (n) {
      case 2: k_rs_finish<2><<<grid, kRsFinishThreads, 0, st>>>(d); break;
      case 4: k_rs_finish<4><<<grid, kRsFinishThreads, 0, st>>>(d); break;
      case 8: k_rs_finish<8><<<grid, kRsFinishThreads, 0, st>>>(d); break;
      default: k_rs_finish<0><<<grid, kRsFinishThreads, 0, st>>>(d); break;
    }
    count_launch();
    const int rc = cuda_check(cudaGetLastError(), "k_rs_finish launch");
    if (rc) return rc;
  }
  return EDB_OK;
}

}  // extern "C"
