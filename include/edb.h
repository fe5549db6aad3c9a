/*
 * edb.h — C-ABI of the easydist-b200 runtime (libedb.so).
 *
 * This is the drop-in boundary for the reshard / redistribute hot path of
 * alibaba/easydist's PyTorch backend.  Every entry point replaces one of the ten
 * Python callables the reference inserts into the sharded FX graph
 * (easydist/torch/passes/sharding.py:94-168) or the NCCL/funcol call underneath it.
 * The reference has no FFI for this path (it is pure Python over
 * torch.ops.c10d_functional.*); the binding a maintainer would add is the ctypes
 * shim shown in INTEGRATION.md (and implemented in easydist_b200/_lib.py).
 *
 * Conventions
 *   - one process per GPU; the library holds one runtime per process
 *   - every function returns 0 on success, non-zero on error; the message of the
 *     last error of the calling thread is returned by edb_last_error()
 *   - plain pointers and sizes only; `stream` is a cudaStream_t passed as void*
 *     (NULL = legacy default stream); all work is stream-ordered and CUDA-graph
 *     capturable: no host synchronisation, no allocation, static peer pointers
 *   - "symmetric heap": one cudaMalloc'd slab per rank, the same size on every
 *     rank, mapped into every peer with CUDA IPC.  A symmetric buffer is named by
 *     its byte offset in the slab; the same offset names the matching buffer on
 *     every rank of a group
 *   - shapes are int64 row-major (contiguous) extents; `elem_size` in bytes
 *   - `gid` is a group handle from edb_group_create (ranks of one mesh dim, in
 *     mesh-coordinate order, exactly the `group` list the reference passes)
 */
#ifndef EDB_H_
#define EDB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EDB_VERSION 100          /* 0.1.0 */
#define EDB_MAX_GROUP 8          /* ranks per group (one NVSwitch domain) */
#define EDB_MAX_GROUPS 16        /* groups per process */
#define EDB_IPC_HANDLE_BYTES 64  /* sizeof(cudaIpcMemHandle_t) */

/* dtype codes (reductions need the arithmetic type; pure data movement only needs elem_size) */
enum edb_dtype { EDB_F32 = 0, EDB_BF16 = 1, EDB_F16 = 2, EDB_F64 = 3, EDB_I32 = 4, EDB_I64 = 5 };
/* reduce ops: the reference's reduce_map, sharding.py:68-73 */
enum edb_redop { EDB_SUM = 0, EDB_MAX = 1, EDB_MIN = 2, EDB_AVG = 3 };

/* ---- runtime ---------------------------------------------------------------------------- */

int edb_version(void);
/* message of the last failing call on this thread ("" if none) */
const char* edb_last_error(void);

/* Bind the process to `device`, allocate the symmetric heap (`heap_bytes`, rounded up to 2 MiB)
 * and zero its flag area.  Replaces: the process-group bootstrap the user does with
 * init_process_group("nccl") + easydist/torch/device_mesh.py:129-150 set_device_mesh. */
int edb_init(int rank, int world, int device, size_t heap_bytes);
int edb_finalize(void);
int edb_is_initialized(void);
/* 0 while healthy.  A wait on a peer that exceeds "spin_timeout_ms" is fatal (the kernel records
 * the op in a pinned host word and traps — like the NCCL watchdog aborting the reference's
 * process — instead of continuing with stale peer data); afterwards this returns EDB_E_STATE with
 * the details in edb_last_error(), even though the CUDA context is gone. */
int edb_health(void);
/* base address / size of the local heap; `user_offset` = first byte usable by edb_symm_alloc */
int edb_heap_info(void** base, size_t* bytes, size_t* user_offset);

/* CUDA-IPC bootstrap: export my slab handle (64 bytes), attach every peer's.  The exchange of
 * the 64-byte blobs is done by the host language over whatever it has (torch.distributed
 * all_gather_object here; same role as ProcessGroupNCCL's ncclUniqueId exchange over the c10d
 * store).  Mechanism also used by the reference in tensorfield/csrc/allocator_interface.cpp:106-110. */
int edb_ipc_export(void* handle_out);
int edb_ipc_attach(int peer_rank, const void* handle);
/* testing aid for single-process multi-"rank" loopback: peer slab = pointer in this process */
int edb_attach_local(int peer_rank, void* base);

/* Create the group of `n` global `ranks` (mesh-dim order).  `slot` selects the group's flag block
 * in the slab and must be the same number on every member (the mesh-dim index, or any agreed id
 * < EDB_MAX_GROUPS).  Replaces funcol's _expand_group(group, tag) (sharding.py:95). */
int edb_group_create(const int* ranks, int n, int slot, int* gid_out);
int edb_group_info(int gid, int* n_out, int* my_index_out);

/* Deterministic bump allocator over the symmetric heap (same call sequence on every rank =>
 * same offsets).  edb_symm_reset(mark) rewinds to a previous edb_symm_mark(). */
int edb_symm_alloc(size_t bytes, size_t align, uint64_t* offset_out);
int edb_symm_mark(uint64_t* mark_out);
int edb_symm_reset(uint64_t mark);

/* ---- local reshard ops (no peer traffic) ------------------------------------------------- */

/* scatter_wrapper (sharding.py:122-123): dst = contiguous(chunk(src, num_chunks, dim)[index]).
 * torch.chunk semantics: block = ceil(shape[dim]/num_chunks); trailing chunks may be short/empty;
 * `dst_extent_out` (may be NULL) receives the dst extent along `dim`. */
int edb_scatter(void* dst, const void* src, const int64_t* shape, int ndim, int dim,
                int num_chunks, int index, int elem_size, int64_t* dst_extent_out, void* stream);

/* copy_wrapper (sharding.py:126-127): dst[0:bytes] = src[0:bytes] (both contiguous, same dtype). */
int edb_copy(void* dst, const void* src, size_t bytes, void* stream);

/* Generic strided N-D box copy (local): dst and src are base pointers, strides in BYTES.
 * Used for Partition boxes (sharding.py:336-474) that stay on the rank. */
int edb_box_copy_local(void* dst, const int64_t* dst_strides, const void* src,
                       const int64_t* src_strides, const int64_t* extents, int ndim, int elem_size,
                       void* stream);

/* ---- collectives over peer memory --------------------------------------------------------- */

/* all_gather_start/end (sharding.py:105-119): out = concat over group ranks of `src` along `dim`.
 * `src`: this rank's shard, contiguous, shape `local_shape`.  The result is written to the
 * symmetric buffer at `dst_off` (shape: local_shape with [dim] multiplied by n); each rank copies
 * its shard into its own slot and pulls the other slots from the peers' buffers. */
int edb_all_gather(int gid, uint64_t dst_off, const void* src, const int64_t* local_shape, int ndim,
                   int dim, int elem_size, void* stream);

/* reduce_scatter_start/end (sharding.py:130-152): dst = reduce_op over ranks of `src`, chunk
 * `my_index` along `dim` (shape[dim] % n must be 0, as the reference asserts).  `src` (full-shape
 * partial value) is first staged at symmetric offset `stage_off` (pass src == NULL when the
 * producer already wrote it there); every rank then pulls its chunk from every peer's stage and
 * reduces in rank order 0..n-1 with fp32 accumulation (f64 for f64, exact for ints).
 * out = reduce * post_scale, cast to `out_dtype` (EDB_AVG multiplies by 1/n after the sum). */
int edb_reduce_scatter(int gid, void* dst, uint64_t stage_off, const void* src,
                       const int64_t* shape, int ndim, int dim, int dtype, int redop,
                       float post_scale, int out_dtype, void* stream);

/* all_reduce_start/end (sharding.py:94-102).  One-shot (every rank reduces every peer's stage)
 * up to `edb_set_option("allreduce_oneshot_bytes")`, two-shot (reduce-scatter into `stage2_off`,
 * then all-gather) above.  `dst` may be any device pointer (contiguous, numel elements). */
int edb_all_reduce(int gid, void* dst, uint64_t stage_off, uint64_t stage2_off, const void* src,
                   int64_t numel, int dtype, int redop, void* stream);

/* all_to_all_start/end (sharding.py:155-163): S(gather_dim) -> S(scatter_dim).
 * dst = chunk(all_gather(src, gather_dim), n, scatter_dim)[my_index], moving only 1/n of what the
 * reference's all-gather implementation moves.  `src` is staged at `stage_off` (src==NULL: already
 * there); dst is a plain device pointer (contiguous result). */
int edb_all_to_all(int gid, void* dst, uint64_t stage_off, const void* src,
                   const int64_t* local_shape, int ndim, int gather_dim, int scatter_dim,
                   int elem_size, void* stream);

/* Partition P2P redistribution (do_p2p_comm_wrapper, sharding.py:595-612): after `src` (this
 * rank's source partition, contiguous, `src_shape`) is staged at `stage_off`, copy `nbox` boxes
 * into `dst` (contiguous, `dst_shape`).  Box b comes from group member peer[b] and is given in the
 * coordinates of that member's source partition (src_start), of my destination partition
 * (dst_start) and its extents; 3*ndim int64 per box, all members must pass the same ndim. */
int edb_box_exchange(int gid, void* dst, const int64_t* dst_shape, uint64_t stage_off,
                     const void* src, const int64_t* src_shape, int ndim, int elem_size, int nbox,
                     const int* peer, const int64_t* src_start, const int64_t* dst_start,
                     const int64_t* extents, const int64_t* peer_src_shapes, void* stream);

/* Halo exchange for S(dim) with halo width w (metashard/halo.py:33-55 halo_padding): dst =
 * concat(prev_rank.src[-w:], src, next_rank.src[:w]) along dim (edges only have one neighbour).
 * The reference discovers halo shardings but never lowers them; semantics follow halo_padding. */
int edb_halo_exchange(int gid, void* dst, uint64_t stage_off, const void* src,
                      const int64_t* local_shape, int ndim, int dim, int halo, int elem_size,
                      void* stream);

/* ---- dense compute on the path (sharded-op kernel dispatch) ------------------------------- */

/* C[M,N] (bf16, row-major, ldc) = A·B (+ bias) with fp32 accumulation on tcgen05 tensor cores.
 *   a_kmajor: A is [M,K] row-major (lda = elements between rows)   else A is stored [K,M] (lda between k rows)
 *   b_kmajor: B is [N,K] row-major (i.e. C = A·Bᵀ, nn.Linear fwd)  else B is stored [K,N] (ldb between k rows)
 * Replaces the aten.mm.default nodes of the sharded graph (Linear fwd / dgrad / wgrad;
 * easydist/torch/passes/fix_bias.py turns addmm into mm+add first).
 *   bias: NULL, or a bf16 row vector [N] added to every row in the epilogue (aten.addmm.default)
 * Requirements: 16-byte aligned bases, lda/ldb/ldc multiples of 8 elements (TMA stride rule);
 * M, N, K themselves are arbitrary (tail boxes are zero-filled / clipped).  Returns
 * EDB_E_UNSUPPORTED (=2) for shapes it does not cover so the host can dispatch elsewhere. */
int edb_gemm_bf16(void* C, const void* A, const void* B, const void* bias, int64_t M, int64_t N,
                  int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int a_kmajor, int b_kmajor,
                  int accumulate_into_c, void* stream);

/* edb_gemm_bf16 with a fused elementwise epilogue over a second operand aux[M, N] (bf16, row
 * stride ld_aux; N % 8 == 0) — "no separate elementwise kernel on the critical path":
 *   epi_op 1 (add)      : C = bf16(A.B + bias + aux)        x + Linear(y): the residual adds of the
 *                         transformer block (aten.add.Tensor behind aten.addmm in the traced graph)
 *   epi_op 2 (gelu_bwd) : C = bf16(bf16(A.B) * gelu'(aux))  aten.gelu_backward(grad = A.B, self = aux,
 *                         approximate = 'tanh') with ATen's fp32 formula
 * Optionally carries an all-gather prefetch like edb_gemm_pf_bf16 (n_items may be 0). */
int edb_gemm_epi_bf16(void* C, const void* A, const void* B, const void* bias, const void* aux,
                      int64_t ld_aux, int epi_op, int64_t M, int64_t N, int64_t K, int64_t lda,
                      int64_t ldb, int64_t ldc, int a_kmajor, int b_kmajor, int gid, int n_items,
                      const uint64_t* src_offs, const uint64_t* dst_offs, const int64_t* bytes,
                      const int64_t* dst_strides, const int64_t* src_strides, void* stream);

/* ---- epoch protocol: one group barrier per phase of the step instead of a handshake per op ----
 *
 * The per-op protocol above costs several dependent system-scope round trips per collective
 * (WAR guard, READY, DONE: ~18 us per fused op at n=2..8), which is what the reference pays per
 * NCCL call as launch + rendezvous latency (sharding.py:94-152, serialized on one stream by
 * CUDA_DEVICE_MAX_CONNECTIONS=1, easydist/torch/__init__.py:53).  A train step has only two
 * points where ranks really depend on each other: (1) before the optimizer — every gradient
 * contribution has arrived and nobody still reads the old parameters; (2) after it — the new
 * parameter shards are final.  `edb_epoch_barrier` is that rendezvous (one 32-thread kernel,
 * monotonic epoch words, CUDA-graph capturable); between two barriers the *_epoch / push kernels
 * below read peers' symmetric operands and write peers' receive slots with no flag traffic. */

/* Group-wide barrier on `stream`: returns (in stream order) once every member has reached its own
 * call.  Everything a member did before its barrier — including its stores into peer memory — is
 * visible to every member after it (system-scope fence + release / acquire). */
int edb_epoch_barrier(int gid, void* stream);

/* All-gather fused into the consuming GEMM: B (weights [N,K], K-major) is sharded S(0) over the
 * group, shard (N/n rows) resident at symmetric offset `b_shard_off` on every rank.  The kernel's
 * copy CTAs pull the peer shards into the local gathered buffer `b_full_off` while the MMA CTAs
 * start on the local shard and consume the others as the copy CTAs announce them (local flags
 * only).  C[M,N] = A[M,K]·B_fullᵀ.  (all_gather_end -> aten.mm pattern, SURVEY App. B)
 * The caller guarantees, with an edb_epoch_barrier earlier on every member's stream, that all
 * shards at `b_shard_off` are final, and that nobody modifies its shard before the next barrier. */
int edb_ag_gemm_epoch_bf16(int gid, void* C, const void* A, const void* bias, uint64_t b_shard_off,
                           uint64_t b_full_off, int64_t M, int64_t N, int64_t K, int64_t lda,
                           int64_t ldc, void* stream);

/* The stand-alone collectives as PUSHES (epoch mode; what the compiled graphs use for every reshard
 * edge with static buffers).  Preconditions: the destination / receive buffers named by the
 * symmetric offsets are dedicated to this graph node, and an edb_epoch_barrier separates the last
 * reader of the previous step from this call (the compiled step ends with one).  Then no
 * write-after-read guard and no READY/DONE handshake is needed: every member stores its contribution
 * straight into the consumers' buffers over NVLink and raises one flag per peer; the consumer polls
 * its own memory.  Results are identical to the flag-protocol entry points above (same rank-order
 * fp32 accumulation).  <= "ll_max_bytes" the low-latency packet path is taken as before.
 *   all_gather_push    : dst_off = the gathered result on every member (as edb_all_gather)
 *   all_to_all_push    : dst_off = the RESULT (symmetric, contiguous, shape of edb_all_to_all's dst)
 *   reduce_scatter_push: recv_off = n receive slots (total input bytes); dst = local result
 *   all_reduce_push    : out_off = the result on every member; recv_off = n * bytes (one-shot: bytes
 *                        <= "allreduce_oneshot_bytes" or numel not divisible) else bytes (two-shot:
 *                        reduce-scatter push + in-place all-gather push) */
int edb_all_gather_push(int gid, uint64_t dst_off, const void* src, const int64_t* local_shape,
                        int ndim, int dim, int elem_size, void* stream);
int edb_all_to_all_push(int gid, uint64_t dst_off, const void* src, const int64_t* local_shape,
                        int ndim, int gather_dim, int scatter_dim, int elem_size, void* stream);
int edb_reduce_scatter_push(int gid, void* dst, uint64_t recv_off, const void* src,
                            const int64_t* shape, int ndim, int dim, int dtype, int redop,
                            float post_scale, int out_dtype, void* stream);
int edb_all_reduce_push(int gid, uint64_t out_off, uint64_t recv_off, const void* src, int64_t numel,
                        int dtype, int redop, void* stream);

/* All-gather as a PREFETCH (the way the zero3 / auto-SPMD parameter gathers run in epoch mode).
 * An item names a byte range that exists at the same symmetric offset on every member (a
 * parameter shard, or part of one): for every member p the range [src_off, src_off + bytes) of
 * p's heap is copied to the local heap at dst_off + p * dst_stride (dst_stride = bytes gives the
 * dim-0 all-gather of all_gather_start, sharding.py:105-119).  Sources must be final since the
 * last edb_epoch_barrier and stay untouched until the next one.
 *   edb_ag_prefetch   : stand-alone launch (whole GPU; start of the step, before the first GEMM)
 *   edb_gemm_pf_bf16  : edb_gemm_bf16 whose grid carries "comm_ctas" extra CTAs doing the copy
 *                       while the others run the GEMM — the gathered operand belongs to a LATER
 *                       kernel, so neither side waits for the other: the all-gather of layer i+1
 *                       costs layer i a few SMs and no time (<= 4 items per launch).
 *
 * `src_strides` (may be NULL = all 0): member p's source range starts at src_off + p*src_stride.
 * With src_stride == dst_stride and src_off == dst_off every member's shard lives IN PLACE in its
 * own slot of the gathered buffer (the optimizer updates it there): the own range needs no copy
 * and only the n-1 remote ranges move — the layout the zero3 lowering uses. */
int edb_ag_prefetch(int gid, int n_items, const uint64_t* src_offs, const uint64_t* dst_offs,
                    const int64_t* bytes, const int64_t* dst_strides, const int64_t* src_strides,
                    void* stream);
int edb_gemm_pf_bf16(void* C, const void* A, const void* B, const void* bias, int64_t M, int64_t N,
                     int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int a_kmajor, int b_kmajor,
                     int gid, int n_items, const uint64_t* src_offs, const uint64_t* dst_offs,
                     const int64_t* bytes, const int64_t* dst_strides, const int64_t* src_strides,
                     void* stream);

/* GEMM whose result is reduce-scattered over its rows, push half: C = A.B (operand layouts as
 * edb_gemm_bf16, incl. cta_group::2 pairs and split-K); row block [p*M/n, (p+1)*M/n) is stored
 * straight into member p's receive slot [me] at symmetric `recv_off` (n slots of (M/n)*N*2 bytes
 * on every member, dedicated to this GEMM) over NVLink, next member's rows first, own rows last.
 * No flags: after the next edb_epoch_barrier every slot of every member is complete, and
 * edb_rs_finish_local may reduce them; the slots may be overwritten again after the barrier that
 * follows that reduction.  (aten.mm -> reduce_scatter_start(avg) of the zero2/zero3 graphs,
 * compile_dp.py:101-118, with the gradient scale + cast fused into the reduction.) */
int edb_gemm_push_bf16(int gid, uint64_t recv_off, const void* A, const void* B, int64_t M,
                       int64_t N, int64_t K, int64_t lda, int64_t ldb, int a_kmajor, int b_kmajor,
                       void* stream);

/* Reduce the receive slots of n_items pushed GEMMs in ONE launch: dsts[i][j] = out_dtype(
 * post_scale * sum over members s in rank order (fp32) of slot_s[j]); purely local memory traffic
 * (the barrier in front made the slots complete). */
int edb_rs_finish_local(int gid, int n_items, void* const* dsts, const uint64_t* recv_offs,
                        const int64_t* chunk_bytes, float post_scale, int out_dtype, void* stream);

/* LayerNorm over the last dimension — aten.native_layer_norm / native_layer_norm_backward nodes of
 * the sharded graph (SURVEY.md App. B lists 8+8 per step in config 1).  x, y, dy, dx: [rows, H]
 * contiguous, dtype bf16 or f32 (w, b, dw, db: [H], same dtype; b/dw/db may be NULL);
 * mean, rstd: [rows] f32.  HBM-streaming kernels: one warp per row, 16-byte vector accesses, shuffle
 * reductions; backward keeps the column partials of dw/db in registers and finishes them in a
 * fixed order (deterministic).  `workspace`: edb_layer_norm_bwd_workspace(H) bytes of scratch.
 * Supported H: multiples of 256 (bf16) / 128 (f32) up to 2048 / 1024; else EDB_E_UNSUPPORTED. */
int edb_layer_norm_fwd(void* y, void* mean, void* rstd, const void* x, const void* w, const void* b,
                       int64_t rows, int64_t H, float eps, int dtype, void* stream);
int edb_layer_norm_bwd(void* dx, void* dw, void* db, const void* dy, const void* x, const void* mean,
                       const void* rstd, const void* w, void* workspace, int64_t rows, int64_t H,
                       int dtype, void* stream);
/* same with the gradient accumulation that follows in the graph fused in: dx = T(T(dx) + add_in)
 * (aten.add.Tensor(native_layer_norm_backward(...)[0], residual_grad)); add_in: [rows, H] or NULL */
int edb_layer_norm_bwd_add(void* dx, void* dw, void* db, const void* dy, const void* x,
                           const void* mean, const void* rstd, const void* w, const void* add_in,
                           void* workspace, int64_t rows, int64_t H, int dtype, void* stream);
int edb_layer_norm_bwd_workspace(int64_t H, size_t* bytes_out);

/* Column sums out[c] = sum_r x[r, c] of a [rows, cols] matrix with row stride `ld` (elements):
 * the bias gradients `aten.sum.dim_IntList(dy, [0], True)` of the sharded graph.  bf16 or f32, fp32
 * accumulation in a fixed order (deterministic).  `workspace`: edb_colsum_workspace(cols) bytes. */
int edb_colsum(void* out, const void* x, void* workspace, int64_t rows, int64_t cols, int64_t ld,
               int dtype, void* stream);
int edb_colsum_workspace(int64_t cols, size_t* bytes_out);

/* Cross-entropy over the last dimension of logits [rows, vocab] (row stride `ld` elements, bf16 or
 * f32) — the `_log_softmax -> nll_loss_forward` / `nll_loss_backward -> _log_softmax_backward_data`
 * chains that end the traced train step (weight=None; reduction 1 = mean, 2 = sum; ignore_index as
 * in aten.nll_loss_forward).  Forward: one pass, online max / sum-exp in fp32; writes the fp32 scalars
 * `loss`, `total_weight` (= number of non-ignored rows) and per-row logsumexp `lse` [rows]
 * (`row_loss` [rows]: scratch).  Backward: dlogits[r, j] = c * (softmax(x_r)[j] - [j == target_r]),
 * c = *grad_out / *total_weight (mean) or *grad_out (sum), 0 for ignored rows, written in the logits
 * dtype with row stride `ld_out` (padding columns [vocab, ld_out) zeroed) so the LM-head GEMMs can
 * consume it without staging.  Rows reduced in a fixed order (deterministic). */
int edb_cross_entropy_fwd(float* loss, float* total_weight, float* lse, float* row_loss,
                          const void* logits, int64_t ld, const int64_t* target, int64_t rows,
                          int64_t vocab, int64_t ignore_index, int reduction, int dtype, void* stream);
int edb_cross_entropy_bwd(void* dlogits, int64_t ld_out, const void* logits, int64_t ld,
                          const int64_t* target, const float* lse, const float* grad_out,
                          const float* total_weight, int64_t rows, int64_t vocab,
                          int64_t ignore_index, int reduction, int dtype, void* stream);

/* Fused multi-tensor SGD-momentum step — the optimizer region of the compiled train step
 * (torch.optim.SGD(momentum, foreach=True) traces to `_foreach_mul_(bufs, mu)`,
 * `_foreach_add_(bufs, grads, alpha=grad_alpha)`, `_foreach_add_(params, bufs, alpha=neg_lr)`; the
 * reference keeps the optimizer inside the compiled graph: easydist/torch/compile_dp.py:201-260).
 * For each of the n tensors (host arrays of device pointers and element counts, all of `dtype` bf16
 * or f32, 16-byte aligned, contiguous):  m = mu*m + grad_alpha*g;  p = p + neg_lr*m, in one pass, with
 * the rounding of the three ATen ops reproduced (bit-identical result). */
int edb_sgd_momentum(int n, void* const* params, const void* const* grads, void* const* bufs,
                     const int64_t* numels, float mu, float grad_alpha, float neg_lr, int dtype,
                     void* stream);

/* ---- options / introspection --------------------------------------------------------------- */

/* integer options: "allreduce_oneshot_bytes", "copy_ctas_per_sm", "comm_ctas", "spin_timeout_ms",
 * "ll_max_bytes", "gemm_cluster", "gemm_force_bn", "gemm_splitk" */
int edb_set_option(const char* name, int64_t value);
int edb_get_option(const char* name, int64_t* value_out);
/* number of kernels this library has launched since load (all entry points) */
uint64_t edb_launch_count(void);

#define EDB_OK 0
#define EDB_E_INVALID 1
#define EDB_E_UNSUPPORTED 2
#define EDB_E_CUDA 3
#define EDB_E_STATE 4

#ifdef __cplusplus
}
#endif
#endif /* EDB_H_ */
