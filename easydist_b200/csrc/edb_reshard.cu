// Reshard / redistribute kernels of libedb.so: every edge the reference lowers to a functional
// collective (easydist/torch/passes/sharding.py:94-163) is here ONE kernel that moves bytes with
// peer-to-peer loads over NVLink/NVSwitch and synchronises with epoch flags in the symmetric heap.
//
// Data movement is expressed as strided "boxes" (Box in edb_internal.cuh); the host side of each
// entry point turns (shape, dim, group) into a handful of boxes, collapsing dimensions so that the
// inner run is as long as possible and 16-byte vector accesses are used whenever alignment allows.
//
// Protocol of one collective `q` in a group (all counters are monotonically increasing):
//   0. WAR guard: wait DONE[p] >= SEQ of every group this rank is in (peers finished reading what
//      they pulled from me in earlier ops) before overwriting symmetric memory.
//   1. copy-in: my contribution -> my symmetric buffer.
//   2. last CTA to finish copy-in: READY[me] = q in every peer's flag block (release.sys).
//   3. per peer p: wait READY[p] >= q (acquire.sys), pull/reduce p's data with plain loads.
//   4. last CTA to finish: DONE[me] = q at every peer, SEQ = q locally.
// Nothing here needs the host, so the kernels are CUDA-graph capturable and the parameters of a
// captured launch stay valid on replay.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>

#include "edb_internal.cuh"

namespace edb {

constexpr int kThreads = 256;

// ---- box copy ------------------------------------------------------------------------------------

template <int V> struct VecT;
template <> struct VecT<16> { typedef uint4 type; };
template <> struct VecT<8> { typedef uint2 type; };
template <> struct VecT<4> { typedef uint32_t type; };
template <> struct VecT<2> { typedef uint16_t type; };
template <> struct VecT<1> { typedef uint8_t type; };

__device__ __forceinline__ void box_offsets(const Box& b, uint32_t r, int64_t& so, int64_t& dof) {
  so = 0;
  dof = 0;
#pragma unroll
  for (int k = 3; k >= 0; --k) {
    const uint32_t e = (uint32_t)b.ext[k];
    if (e > 1) {
      const uint32_t idx = r % e;
      r /= e;
      so += (int64_t)idx * b.sstr[k];
      dof += (int64_t)idx * b.dstr[k];
    }
  }
}

template <int V>
__device__ __forceinline__ void copy_box_v(const Box& b, uint64_t tid, uint64_t nthr) {
  typedef typename VecT<V>::type T;
  const uint64_t row_vecs = (uint64_t)b.inner / V;
  const uint64_t rows = (uint64_t)b.ext[0] * b.ext[1] * b.ext[2] * b.ext[3];
  const uint64_t total = rows * row_vecs;
  constexpr int U = 4;
  if (rows == 1) {
    const T* __restrict__ s = reinterpret_cast<const T*>(b.src);
    T* __restrict__ d = reinterpret_cast<T*>(b.dst);
    uint64_t i = tid;
    for (; i + (U - 1) * nthr < total; i += U * nthr) {
      T v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = s[i + u * nthr];
#pragma unroll
      for (int u = 0; u < U; ++u) d[i + u * nthr] = v[u];
    }
    for (; i < total; i += nthr) d[i] = s[i];
    return;
  }
  const bool small = total < 0xffffffffull;
  uint64_t i = tid;
  for (; i + (U - 1) * nthr < total; i += U * nthr) {
    T v[U];
    char* dp[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint64_t ii = i + u * nthr;
      uint64_t r, c;
      if (small) {
        const uint32_t r32 = (uint32_t)ii / (uint32_t)row_vecs;
        r = r32;
        c = (uint32_t)ii - r32 * (uint32_t)row_vecs;
      } else {
        r = ii / row_vecs;
        c = ii - r * row_vecs;
      }
      int64_t so, dof;
      box_offsets(b, (uint32_t)r, so, dof);
      v[u] = *reinterpret_cast<const T*>(b.src + so + c * V);
      dp[u] = b.dst + dof + c * V;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) *reinterpret_cast<T*>(dp[u]) = v[u];
  }
  for (; i < total; i += nthr) {
    uint64_t r = i / row_vecs, c = i - r * row_vecs;
    int64_t so, dof;
    box_offsets(b, (uint32_t)r, so, dof);
    *reinterpret_cast<T*>(b.dst + dof + c * V) = *reinterpret_cast<const T*>(b.src + so + c * V);
  }
}

__device__ __forceinline__ void copy_box(const Box& b, uint64_t tid, uint64_t nthr) {
  switch (b.vec) {
    case 16: copy_box_v<16>(b, tid, nthr); break;
    case 8: copy_box_v<8>(b, tid, nthr); break;
    case 4: copy_box_v<4>(b, tid, nthr); break;
    case 2: copy_box_v<2>(b, tid, nthr); break;
    default: copy_box_v<1>(b, tid, nthr); break;
  }
}

// ---- kernels -----------------------------------------------------------------------------------------

__global__ void __launch_bounds__(kThreads) k_local_copy(const __grid_constant__ GatherDesc d) {
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t nthr = (uint64_t)gridDim.x * blockDim.x;
  for (int b = 0; b < d.n_boxes; ++b) copy_box(d.box[b], tid, nthr);
}

__global__ void __launch_bounds__(kThreads) k_gather(const __grid_constant__ GatherDesc d) {
  __shared__ uint64_t s_q;
  __shared__ int s_last;
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t nthr = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t q = begin_op(d.f, &s_q);
  for (int b = 0; b < d.n_in; ++b) copy_box(d.box[b], tid, nthr);
  grid_signal(d.f, F_CNT_A, F_READY, q, &s_last, gridDim.x);
  for (int b = d.n_in; b < d.n_boxes; ++b) {
    const int p = d.box[b].peer;
    if (p >= 0 && p != d.f.me) wait_flag(d.f, F_READY, p, q);
    copy_box(d.box[b], tid, nthr);
  }
  finish_op(d.f, q, &s_last, gridDim.x);
}

// ---- push protocol (epoch mode) ---------------------------------------------------------------
// The destination buffers are static per graph node and an edb_epoch_barrier separates two steps, so
// nobody reads or writes them concurrently with the next step's push: no write-after-read guard, no
// READY/DONE handshake — data first, then one flag per peer (system-scope release), and the
// consumer polls its own memory.

// All CTAs of the launch have written their share: the last one to arrive raises the flags.
// Returns true in that CTA.
__device__ __forceinline__ bool push_signal(const FlagCtx& f, uint64_t q, int* s_last,
                                            unsigned n_ctas) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();  // covers the CTA's stores into peer memory (see grid_signal)
    const unsigned long long prev =
        atomicAdd(reinterpret_cast<unsigned long long*>(f.local + F_CNT_P), 1ULL);
    const int last = (prev == (unsigned long long)n_ctas - 1);
    if (last) {
      f.local[F_CNT_P] = 0;
      __threadfence_system();
    }
    *s_last = last;
  }
  __syncthreads();
  if (*s_last && (int)threadIdx.x < f.n && (int)threadIdx.x != f.me)
    st_release_sys(f.peer[threadIdx.x] + F_PUSHFLAG + f.me, q);
  return *s_last != 0;
}

__device__ __forceinline__ void push_wait(const FlagCtx& f, uint64_t q) {
  if ((int)threadIdx.x < f.n && (int)threadIdx.x != f.me)
    spin_wait_sys(f.local + F_PUSHFLAG + threadIdx.x, q, f.timeout_ns, f.local + F_ERR);
  __syncthreads();
}

// all-gather / all-to-all / any box scatter as a push: every box writes into a member's buffer
__global__ void __launch_bounds__(kThreads) k_push(const __grid_constant__ GatherDesc d) {
  __shared__ uint64_t s_q;
  __shared__ int s_last;
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t nthr = (uint64_t)gridDim.x * blockDim.x;
  if (threadIdx.x == 0) s_q = ld_relaxed_gpu(d.f.local + F_PUSHSEQ) + 1;
  __syncthreads();
  const uint64_t q = s_q;
  for (int b = 0; b < d.n_boxes; ++b) copy_box(d.box[b], tid, nthr);
  if (push_signal(d.f, q, &s_last, gridDim.x)) {
    // only this CTA stays until every member's data is here; the others are done
    push_wait(d.f, q);
    if (threadIdx.x == 0) st_release_gpu(d.f.local + F_PUSHSEQ, q);
  }
}

__global__ void __launch_bounds__(32) k_epoch_barrier(const __grid_constant__ FlagCtx f) {
  __shared__ uint64_t s_e;
  epoch_barrier_cta(f, &s_e);
}

// ---- reductions ------------------------------------------------------------------------------------

template <typename T> struct Conv;
template <> struct Conv<float> {
  typedef float acc;
  static __device__ __forceinline__ float to(float v) { return v; }
  static __device__ __forceinline__ float from(float v) { return v; }
};
template <> struct Conv<__nv_bfloat16> {
  typedef float acc;
  static __device__ __forceinline__ float to(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ __nv_bfloat16 from(float v) { return __float2bfloat16_rn(v); }
};
template <> struct Conv<__half> {
  typedef float acc;
  static __device__ __forceinline__ float to(__half v) { return __half2float(v); }
  static __device__ __forceinline__ __half from(float v) { return __float2half_rn(v); }
};
template <> struct Conv<double> {
  typedef double acc;
  static __device__ __forceinline__ double to(double v) { return v; }
  static __device__ __forceinline__ double from(double v) { return v; }
};
template <> struct Conv<int32_t> {
  typedef int32_t acc;
  static __device__ __forceinline__ int32_t to(int32_t v) { return v; }
  static __device__ __forceinline__ int32_t from(int32_t v) { return v; }
};
template <> struct Conv<int64_t> {
  typedef int64_t acc;
  static __device__ __forceinline__ int64_t to(int64_t v) { return v; }
  static __device__ __forceinline__ int64_t from(int64_t v) { return v; }
};

template <int OP, typename A> __device__ __forceinline__ A combine(A a, A b) {
  if (OP == EDB_MAX) return a > b ? a : b;
  if (OP == EDB_MIN) return a < b ? a : b;
  return a + b;
}

template <typename A> __device__ __forceinline__ A apply_scale(A v, float s) { return v; }
template <> __device__ __forceinline__ float apply_scale<float>(float v, float s) { return v * s; }
template <> __device__ __forceinline__ double apply_scale<double>(double v, float s) {
  return v * (double)s;
}

template <typename In, typename Out, int OP>
__device__ __forceinline__ void reduce_rows(const ReduceDesc& d, char* dst_b, uint64_t tid,
                                            uint64_t nthr, bool vec) {
  typedef typename Conv<In>::acc A;
  constexpr int EPV = 16 / sizeof(In);
  const uint64_t rows = (uint64_t)d.ext[0] * d.ext[1] * d.ext[2] * d.ext[3];
  const bool scaled = (d.scale != 1.0f);
  Box geo;  // only ext/sstr/dstr are used by box_offsets
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    geo.ext[k] = d.ext[k];
    geo.sstr[k] = d.sstr[k];
    geo.dstr[k] = d.dstr[k];
  }
  if (vec) {
    const uint64_t row_vecs = (uint64_t)d.inner / 16;
    const uint64_t total = rows * row_vecs;
    for (uint64_t i = tid; i < total; i += nthr) {
      uint64_t r = 0, c = i;
      int64_t so = 0, dof = 0;
      if (rows > 1) {
        r = i / row_vecs;
        c = i - r * row_vecs;
        box_offsets(geo, (uint32_t)r, so, dof);
      }
      uint4 raw[kMaxGroup];
#pragma unroll
      for (int p = 0; p < kMaxGroup; ++p)
        if (p < d.n_src) raw[p] = *reinterpret_cast<const uint4*>(d.src[p] + so + c * 16);
      A acc[EPV];
      {
        const In* e = reinterpret_cast<const In*>(&raw[0]);
#pragma unroll
        for (int j = 0; j < EPV; ++j) acc[j] = Conv<In>::to(e[j]);
      }
#pragma unroll
      for (int p = 1; p < kMaxGroup; ++p)
        if (p < d.n_src) {
          const In* e = reinterpret_cast<const In*>(&raw[p]);
#pragma unroll
          for (int j = 0; j < EPV; ++j) acc[j] = combine<OP, A>(acc[j], Conv<In>::to(e[j]));
        }
      Out o[EPV];
#pragma unroll
      for (int j = 0; j < EPV; ++j)
        o[j] = Conv<Out>::from((typename Conv<Out>::acc)(scaled ? apply_scale<A>(acc[j], d.scale)
                                                                : acc[j]));
      constexpr int OB = EPV * sizeof(Out);  // 16 or 32 (or 8 for f32->bf16)
      char* dp = d.dst + dof + c * OB;
      if (OB == 32) {
        reinterpret_cast<uint4*>(dp)[0] = reinterpret_cast<const uint4*>(o)[0];
        reinterpret_cast<uint4*>(dp)[1] = reinterpret_cast<const uint4*>(o)[1];
      } else if (OB == 16) {
        *reinterpret_cast<uint4*>(dp) = *reinterpret_cast<const uint4*>(o);
      } else {
        *reinterpret_cast<uint2*>(dp) = *reinterpret_cast<const uint2*>(o);
      }
      if (dst_b) {
        char* dq = dst_b + dof + c * OB;
        if (OB == 32) {
          reinterpret_cast<uint4*>(dq)[0] = reinterpret_cast<const uint4*>(o)[0];
          reinterpret_cast<uint4*>(dq)[1] = reinterpret_cast<const uint4*>(o)[1];
        } else if (OB == 16) {
          *reinterpret_cast<uint4*>(dq) = *reinterpret_cast<const uint4*>(o);
        } else {
          *reinterpret_cast<uint2*>(dq) = *reinterpret_cast<const uint2*>(o);
        }
      }
    }
  } else {
    const uint64_t row_el = (uint64_t)d.inner / sizeof(In);
    const uint64_t total = rows * row_el;
    for (uint64_t i = tid; i < total; i += nthr) {
      uint64_t r = 0, c = i;
      int64_t so = 0, dof = 0;
      if (rows > 1) {
        r = i / row_el;
        c = i - r * row_el;
        box_offsets(geo, (uint32_t)r, so, dof);
      }
      A acc = Conv<In>::to(*reinterpret_cast<const In*>(d.src[0] + so + c * sizeof(In)));
      for (int p = 1; p < d.n_src; ++p)
        acc = combine<OP, A>(acc,
                             Conv<In>::to(*reinterpret_cast<const In*>(d.src[p] + so + c * sizeof(In))));
      if (scaled) acc = apply_scale<A>(acc, d.scale);
      const Out o = Conv<Out>::from((typename Conv<Out>::acc)acc);
      *reinterpret_cast<Out*>(d.dst + dof + c * sizeof(Out)) = o;
      if (dst_b) *reinterpret_cast<Out*>(dst_b + dof + c * sizeof(Out)) = o;
    }
  }
}

struct ReduceLaunch {
  ReduceDesc d;
  char* dst_b;  // optional second destination (two-shot: final dst of my own part)
  int vec;
  int push;     // k_push_reduce: d.pull[] are pushes into the members' receive slots
};

template <typename In, typename Out, int OP>
__global__ void __launch_bounds__(kThreads, 3) k_reduce(const __grid_constant__ ReduceLaunch L) {
  __shared__ uint64_t s_q;
  __shared__ int s_last;
  const ReduceDesc& d = L.d;
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t nthr = (uint64_t)gridDim.x * blockDim.x;
  const bool multi = d.f.n > 1;
  uint64_t q = 0;
  if (multi) {
    q = begin_op(d.f, &s_q);
    if (d.has_in) copy_box(d.in, tid, nthr);
    grid_signal(d.f, F_CNT_A, F_READY, q, &s_last, gridDim.x);
    if (threadIdx.x < d.f.n && threadIdx.x != d.f.me)
      spin_wait_sys(d.f.local + F_READY + threadIdx.x, q, d.f.timeout_ns, d.f.local + F_ERR);
    __syncthreads();
  }
  reduce_rows<In, Out, OP>(d, L.dst_b, tid, nthr, L.vec != 0);
  if (multi) {
    if (d.two_shot) {
      grid_signal(d.f, F_CNT_C, F_READY2, q, &s_last, gridDim.x);
      for (int b = 0; b < d.n_pull; ++b) {
        wait_flag(d.f, F_READY2, d.pull[b].peer, q);
        copy_box(d.pull[b], tid, nthr);
      }
    }
    finish_op(d.f, q, &s_last, gridDim.x);
  }
}

// reduce-scatter / one-shot all-reduce as a push: my chunk for member p goes into p's receive slot
// [me] (d.pull[] = the pushes, own slot included), then every CTA reduces its share of the n
// local slots in rank order
template <typename In, typename Out, int OP>
__global__ void __launch_bounds__(kThreads, 3) k_push_reduce(const __grid_constant__ ReduceLaunch L) {
  __shared__ uint64_t s_q;
  __shared__ int s_last;
  const ReduceDesc& d = L.d;
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t nthr = (uint64_t)gridDim.x * blockDim.x;
  if (threadIdx.x == 0) s_q = ld_relaxed_gpu(d.f.local + F_PUSHSEQ) + 1;
  __syncthreads();
  const uint64_t q = s_q;
  for (int b = 0; b < d.n_pull; ++b) copy_box(d.pull[b], tid, nthr);
  push_signal(d.f, q, &s_last, gridDim.x);
  push_wait(d.f, q);
  reduce_rows<In, Out, OP>(d, L.dst_b, tid, nthr, L.vec != 0);
  // the op number advances when every CTA is through (they all read it at the start)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned long long prev =
        atomicAdd(reinterpret_cast<unsigned long long*>(d.f.local + F_CNT_P2), 1ULL);
    if (prev == (unsigned long long)gridDim.x - 1) {
      d.f.local[F_CNT_P2] = 0;
      __threadfence();
      st_release_gpu(d.f.local + F_PUSHSEQ, q);
    }
  }
}

// ---- host helpers --------------------------------------------------------------------------------

// Kernels whose CTAs spin on flags written by other CTAs (of this or a peer GPU) must be fully
// co-resident, otherwise resident CTAs wait forever for CTAs that cannot be scheduled.  The grid
// is therefore capped by the occupancy of the exact kernel being launched.
int grid_for_bytes(size_t bytes, int threads, int max_ctas_per_sm) {
  Runtime& r = rt();
  const size_t per_cta = (size_t)threads * 16 * 4;
  size_t want = (bytes + per_cta - 1) / per_cta;
  int64_t per_sm = std::max<int64_t>(1, r.copy_ctas_per_sm);
  if (max_ctas_per_sm > 0 && per_sm > max_ctas_per_sm) per_sm = max_ctas_per_sm;
  const size_t cap = (size_t)r.sm_count * (size_t)per_sm;
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  return (int)want;
}

template <typename K> static int occupancy_of(K kernel) {
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, kThreads, 0) != cudaSuccess || n < 1)
    n = 1;
  return n;
}

static int pick_vec(uintptr_t bits) {
  if ((bits & 15) == 0) return 16;
  if ((bits & 7) == 0) return 8;
  if ((bits & 3) == 0) return 4;
  if ((bits & 1) == 0) return 2;
  return 1;
}

// Build a Box from N-D extents (elements) and byte strides, collapsing dimensions.
int make_box(Box* out, const void* src, const int64_t* src_strides, void* dst,
             const int64_t* dst_strides, const int64_t* extents, int ndim, int elem_size,
             int peer) {
  if (ndim > 16) return set_error(EDB_E_UNSUPPORTED, "make_box: ndim %d too large", ndim);
  int64_t e[17], ss[17], ds[17];
  int m = 0;
  for (int i = 0; i < ndim; ++i) {
    if (extents[i] == 1) continue;
    e[m] = extents[i];
    ss[m] = src_strides[i];
    ds[m] = dst_strides[i];
    ++m;
  }
  // innermost "byte" dimension
  e[m] = elem_size;
  ss[m] = 1;
  ds[m] = 1;
  ++m;
  // merge adjacent dims (outer i, inner i+1) when both sides are contiguous across them
  int64_t fe[17], fs[17], fd[17];
  int k = 0;
  fe[0] = e[0];
  fs[0] = ss[0];
  fd[0] = ds[0];
  for (int i = 1; i < m; ++i) {
    if (fs[k] == ss[i] * e[i] && fd[k] == ds[i] * e[i]) {
      fe[k] *= e[i];
      fs[k] = ss[i];
      fd[k] = ds[i];
    } else {
      ++k;
      fe[k] = e[i];
      fs[k] = ss[i];
      fd[k] = ds[i];
    }
  }
  ++k;  // number of merged dims; last one is the inner run when its strides are 1
  Box b;
  memset(&b, 0, sizeof(b));
  b.src = static_cast<const char*>(src);
  b.dst = static_cast<char*>(dst);
  b.peer = peer;
  int outer = k;
  if (fs[k - 1] == 1 && fd[k - 1] == 1) {
    b.inner = fe[k - 1];
    outer = k - 1;
  } else {
    b.inner = 1;  // cannot happen (the byte dim always has stride 1) but stay safe
  }
  if (outer > 4)
    return set_error(EDB_E_UNSUPPORTED, "make_box: %d non-mergeable outer dims (max 4)", outer);
  for (int i = 0; i < 4; ++i) {
    b.ext[i] = 1;
    b.sstr[i] = 0;
    b.dstr[i] = 0;
  }
  uintptr_t bits = (uintptr_t)b.src | (uintptr_t)b.dst | (uintptr_t)b.inner;
  int64_t rows = 1;
  for (int i = 0; i < outer; ++i) {
    const int slot = 4 - outer + i;
    b.ext[slot] = fe[i];
    b.sstr[slot] = fs[i];
    b.dstr[slot] = fd[i];
    bits |= (uintptr_t)fs[i] | (uintptr_t)fd[i];
    rows *= fe[i];
  }
  if (rows >= 0xffffffffll)
    return set_error(EDB_E_UNSUPPORTED, "make_box: too many rows (%lld)", (long long)rows);
  b.vec = pick_vec(bits);
  *out = b;
  return EDB_OK;
}

static void contiguous_strides(const int64_t* shape, int ndim, int elem_size, int64_t* strides) {
  int64_t s = elem_size;
  for (int i = ndim - 1; i >= 0; --i) {
    strides[i] = s;
    s *= shape[i];
  }
}

static int64_t numel_of(const int64_t* shape, int ndim) {
  int64_t n = 1;
  for (int i = 0; i < ndim; ++i) n *= shape[i];
  return n;
}

int fill_flagctx(FlagCtx* f, int gid) {
  Runtime& r = rt();
  if (!r.inited) return set_error(EDB_E_STATE, "runtime not initialised (call edb_init)");
  if (gid < 0 || gid >= r.ngroups) return set_error(EDB_E_INVALID, "bad group id %d", gid);
  const Group& g = r.groups[gid];
  memset(f, 0, sizeof(*f));
  f->n = g.n;
  f->me = g.me;
  f->local = flag_block(r.heap, g.slot);
  for (int p = 0; p < g.n; ++p) f->peer[p] = flag_block(r.peer_heap[g.ranks[p]], g.slot);
  f->n_war = r.ngroups;  // <= kMaxGroups by construction (edb_group_create)
  for (int i = 0; i < r.ngroups; ++i) {
    f->war_block[i] = flag_block(r.heap, r.groups[i].slot);
    f->war_n[i] = (uint8_t)r.groups[i].n;
    f->war_me[i] = (uint8_t)r.groups[i].me;
  }
  f->timeout_ns = (uint64_t)r.spin_timeout_ms * 1000000ull;
  return EDB_OK;
}

static int check_symm(uint64_t off, size_t bytes, const char* what) {
  Runtime& r = rt();
  if (off < kUserOffset || off + bytes > r.heap_bytes || (off & 15))
    return set_error(EDB_E_INVALID, "%s: symmetric range [%llu, +%zu) invalid", what,
                     (unsigned long long)off, bytes);
  return EDB_OK;
}

static size_t box_bytes(const Box& b) {
  return (size_t)(b.inner * b.ext[0] * b.ext[1] * b.ext[2] * b.ext[3]);
}

static int launch_gather(const GatherDesc& d, bool flags, cudaStream_t st, bool push = false) {
  size_t bytes = 0;
  for (int b = 0; b < d.n_boxes; ++b) bytes += box_bytes(d.box[b]);
  static const int occ_gather = occupancy_of(k_gather);
  static const int occ_push = occupancy_of(k_push);
  const int grid = grid_for_bytes(bytes, kThreads, push ? occ_push : (flags ? occ_gather : 0));
  if (push) k_push<<<grid, kThreads, 0, st>>>(d);
  else if (flags) k_gather<<<grid, kThreads, 0, st>>>(d);
  else k_local_copy<<<grid, kThreads, 0, st>>>(d);
  count_launch();
  return cuda_check(cudaGetLastError(), "reshard kernel launch");
}

template <typename In, typename Out, int OP>
static void launch_reduce_kernel(const ReduceLaunch& L, size_t bytes, cudaStream_t st) {
  if (L.push) {
    static const int occ_p = occupancy_of(k_push_reduce<In, Out, OP>);
    const int grid = grid_for_bytes(bytes, kThreads, occ_p);
    k_push_reduce<In, Out, OP><<<grid, kThreads, 0, st>>>(L);
    return;
  }
  static const int occ = occupancy_of(k_reduce<In, Out, OP>);
  const int grid = grid_for_bytes(bytes, kThreads, occ);
  k_reduce<In, Out, OP><<<grid, kThreads, 0, st>>>(L);
}

template <typename In, typename Out>
static int launch_reduce_op(const ReduceLaunch& L, size_t bytes, cudaStream_t st) {
  switch (L.d.redop) {
    case EDB_SUM:
    case EDB_AVG: launch_reduce_kernel<In, Out, EDB_SUM>(L, bytes, st); break;
    case EDB_MAX: launch_reduce_kernel<In, Out, EDB_MAX>(L, bytes, st); break;
    case EDB_MIN: launch_reduce_kernel<In, Out, EDB_MIN>(L, bytes, st); break;
    default: return set_error(EDB_E_INVALID, "bad reduce op %d", L.d.redop);
  }
  count_launch();
  return cuda_check(cudaGetLastError(), "reduce kernel launch");
}

static int launch_reduce(ReduceLaunch& L, cudaStream_t st) {
  ReduceDesc& d = L.d;
  const size_t in_es = dtype_size(d.dtype), out_es = dtype_size(d.out_dtype);
  if (!in_es || !out_es) return set_error(EDB_E_INVALID, "bad dtype %d/%d", d.dtype, d.out_dtype);
  // vector path: every source/destination address and stride 16-byte friendly
  uintptr_t bits = (uintptr_t)d.inner;
  for (int p = 0; p < d.n_src; ++p) bits |= (uintptr_t)d.src[p];
  for (int k = 0; k < 4; ++k) bits |= (uintptr_t)d.sstr[k];
  const size_t obytes = 16 / in_es * out_es;  // bytes written per 16-byte input vector
  uintptr_t obits = (uintptr_t)d.dst | (uintptr_t)L.dst_b;
  for (int k = 0; k < 4; ++k) obits |= (uintptr_t)d.dstr[k];
  const size_t oalign = obytes >= 16 ? 16 : obytes;
  L.vec = ((bits & 15) == 0 && (obits & (oalign - 1)) == 0) ? 1 : 0;
  size_t bytes = (size_t)(d.inner * d.ext[0] * d.ext[1] * d.ext[2] * d.ext[3]) * d.n_src +
                 (d.has_in ? box_bytes(d.in) : 0);
  if (L.push)
    for (int b = 0; b < d.n_pull; ++b) bytes += box_bytes(d.pull[b]);
  const size_t grid = bytes;  // the launcher sizes the grid from the byte count + occupancy
  const int key = d.dtype * 16 + d.out_dtype;
  switch (key) {
    case EDB_F32 * 16 + EDB_F32: return launch_reduce_op<float, float>(L, grid, st);
    case EDB_F32 * 16 + EDB_BF16: return launch_reduce_op<float, __nv_bfloat16>(L, grid, st);
    case EDB_BF16 * 16 + EDB_BF16: return launch_reduce_op<__nv_bfloat16, __nv_bfloat16>(L, grid, st);
    case EDB_BF16 * 16 + EDB_F32: return launch_reduce_op<__nv_bfloat16, float>(L, grid, st);
    case EDB_F16 * 16 + EDB_F16: return launch_reduce_op<__half, __half>(L, grid, st);
    case EDB_F16 * 16 + EDB_F32: return launch_reduce_op<__half, float>(L, grid, st);
    case EDB_F64 * 16 + EDB_F64: return launch_reduce_op<double, double>(L, grid, st);
    case EDB_I32 * 16 + EDB_I32: return launch_reduce_op<int32_t, int32_t>(L, grid, st);
    case EDB_I64 * 16 + EDB_I64: return launch_reduce_op<int64_t, int64_t>(L, grid, st);
  }
  return set_error(EDB_E_UNSUPPORTED, "reduce: dtype %d -> %d not supported", d.dtype, d.out_dtype);
}

}  // namespace edb

using namespace edb;

extern "C" {

int edb_copy(void* dst, const void* src, size_t bytes, void* stream) {
  if (bytes == 0) return EDB_OK;
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  const int64_t ext[1] = {(int64_t)bytes}, str[1] = {1};
  int rc = make_box(&d.box[0], src, str, dst, str, ext, 1, 1, -1);
  if (rc) return rc;
  d.n_in = 0;
  d.n_boxes = 1;
  return launch_gather(d, false, (cudaStream_t)stream);
}

int edb_box_copy_local(void* dst, const int64_t* dst_strides, const void* src,
                       const int64_t* src_strides, const int64_t* extents, int ndim, int elem_size,
                       void* stream) {
  if (numel_of(extents, ndim) == 0) return EDB_OK;
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  int rc = make_box(&d.box[0], src, src_strides, dst, dst_strides, extents, ndim, elem_size, -1);
  if (rc) return rc;
  d.n_boxes = 1;
  return launch_gather(d, false, (cudaStream_t)stream);
}

int edb_scatter(void* dst, const void* src, const int64_t* shape, int ndim, int dim, int num_chunks,
                int index, int elem_size, int64_t* dst_extent_out, void* stream) {
  EDB_REQUIRE(ndim >= 1 && ndim <= 16 && dim >= 0 && dim < ndim, "edb_scatter: bad dim %d/%d", dim,
              ndim);
  EDB_REQUIRE(num_chunks >= 1 && index >= 0 && index < num_chunks, "edb_scatter: bad chunk %d/%d",
              index, num_chunks);
  // torch.chunk: block = ceil(size/chunks); chunk i = [i*block, min(size,(i+1)*block))
  const int64_t size = shape[dim];
  const int64_t block = (size + num_chunks - 1) / num_chunks;
  const int64_t lo = std::min(size, block * index), hi = std::min(size, block * (index + 1));
  if (dst_extent_out) *dst_extent_out = hi - lo;
  int64_t ext[16], sstr[16], dstr[16], oshape[16];
  for (int i = 0; i < ndim; ++i) ext[i] = oshape[i] = shape[i];
  ext[dim] = oshape[dim] = hi - lo;
  if (numel_of(ext, ndim) == 0) return EDB_OK;
  contiguous_strides(shape, ndim, elem_size, sstr);
  contiguous_strides(oshape, ndim, elem_size, dstr);
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  int rc = make_box(&d.box[0], static_cast<const char*>(src) + lo * sstr[dim], sstr, dst, dstr, ext,
                    ndim, elem_size, -1);
  if (rc) return rc;
  d.n_boxes = 1;
  return launch_gather(d, false, (cudaStream_t)stream);
}

int edb_all_gather(int gid, uint64_t dst_off, const void* src, const int64_t* local_shape, int ndim,
                   int dim, int elem_size, void* stream) {
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  int rc = fill_flagctx(&d.f, gid);
  if (rc) return rc;
  EDB_REQUIRE(ndim >= 1 && ndim <= 16 && dim >= 0 && dim < ndim, "edb_all_gather: bad dim %d/%d",
              dim, ndim);
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  int64_t outer = 1, rowb = elem_size;
  for (int i = 0; i < dim; ++i) outer *= local_shape[i];
  for (int i = dim; i < ndim; ++i) rowb *= local_shape[i];
  const size_t total = (size_t)outer * rowb * n;
  if (total == 0) return EDB_OK;
  rc = check_symm(dst_off, total, "edb_all_gather");
  if (rc) return rc;
  char* out_me = r.heap + dst_off;
  {
    const int ll = ll_try(gid, /*LL_ALL_GATHER*/ 1, out_me, src, outer * rowb, outer, rowb, 0, 0, 1.0f,
                          (cudaStream_t)stream);
    if (ll >= 0) return ll;
  }
  const int64_t ext[2] = {outer, rowb};
  const int64_t s_src[2] = {rowb, 1}, s_out[2] = {rowb * n, 1};
  rc = make_box(&d.box[0], src, s_src, out_me + (int64_t)me * rowb, s_out, ext, 2, 1, -1);
  if (rc) return rc;
  d.n_in = 1;
  int nb = 1;
  for (int k = 1; k < n; ++k) {
    const int p = (me + k) % n;
    const char* out_p = r.peer_heap[g.ranks[p]] + dst_off;
    rc = make_box(&d.box[nb], out_p + (int64_t)p * rowb, s_out, out_me + (int64_t)p * rowb, s_out,
                  ext, 2, 1, p);
    if (rc) return rc;
    ++nb;
  }
  d.n_boxes = nb;
  return launch_gather(d, n > 1, (cudaStream_t)stream);
}

int edb_all_to_all(int gid, void* dst, uint64_t stage_off, const void* src,
                   const int64_t* local_shape, int ndim, int gather_dim, int scatter_dim,
                   int elem_size, void* stream) {
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  int rc = fill_flagctx(&d.f, gid);
  if (rc) return rc;
  EDB_REQUIRE(ndim >= 1 && ndim <= 16 && gather_dim >= 0 && gather_dim < ndim && scatter_dim >= 0 &&
                  scatter_dim < ndim && gather_dim != scatter_dim,
              "edb_all_to_all: bad dims g=%d s=%d ndim=%d", gather_dim, scatter_dim, ndim);
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  EDB_REQUIRE(local_shape[scatter_dim] % n == 0,
              "edb_all_to_all: scatter dim size %lld not divisible by group size %d",
              (long long)local_shape[scatter_dim], n);
  const int64_t total = numel_of(local_shape, ndim) * elem_size;
  if (total == 0) return EDB_OK;
  if (n > 1) {
    rc = check_symm(stage_off, (size_t)total, "edb_all_to_all");
    if (rc) return rc;
  }
  int64_t oshape[16], ext[16], sstr[16], dstr[16];
  for (int i = 0; i < ndim; ++i) oshape[i] = ext[i] = local_shape[i];
  const int64_t cs = local_shape[scatter_dim] / n;
  oshape[gather_dim] = local_shape[gather_dim] * n;
  oshape[scatter_dim] = cs;
  ext[scatter_dim] = cs;
  contiguous_strides(local_shape, ndim, elem_size, sstr);
  contiguous_strides(oshape, ndim, elem_size, dstr);
  int nb = 0;
  if (src && n > 1) {
    const int64_t e1[1] = {total}, s1[1] = {1};
    rc = make_box(&d.box[nb++], src, s1, r.heap + stage_off, s1, e1, 1, 1, -1);
    if (rc) return rc;
  }
  d.n_in = nb;
  const char* my_src = src ? static_cast<const char*>(src) : r.heap + stage_off;
  for (int k = 0; k < n; ++k) {
    const int p = (me + k) % n;
    const char* sp = (p == me) ? my_src : r.peer_heap[g.ranks[p]] + stage_off;
    rc = make_box(&d.box[nb++], sp + (int64_t)me * cs * sstr[scatter_dim], sstr,
                  static_cast<char*>(dst) + (int64_t)p * local_shape[gather_dim] * dstr[gather_dim],
                  dstr, ext, ndim, elem_size, p == me ? -1 : p);
    if (rc) return rc;
  }
  d.n_boxes = nb;
  return launch_gather(d, n > 1, (cudaStream_t)stream);
}

int edb_halo_exchange(int gid, void* dst, uint64_t stage_off, const void* src,
                      const int64_t* local_shape, int ndim, int dim, int halo, int elem_size,
                      void* stream) {
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  int rc = fill_flagctx(&d.f, gid);
  if (rc) return rc;
  EDB_REQUIRE(ndim >= 1 && ndim <= 16 && dim >= 0 && dim < ndim, "edb_halo_exchange: bad dim");
  EDB_REQUIRE(halo >= 0 && halo <= local_shape[dim],
              "edb_halo_exchange: halo %d larger than shard extent %lld (halo.py raises too)", halo,
              (long long)local_shape[dim]);
  EDB_REQUIRE(src != nullptr, "edb_halo_exchange: src required");
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  const int64_t total = numel_of(local_shape, ndim) * elem_size;
  if (total == 0) return EDB_OK;
  if (n > 1) {
    rc = check_symm(stage_off, (size_t)total, "edb_halo_exchange");
    if (rc) return rc;
  }
  const bool has_prev = me > 0 && halo > 0, has_next = me < n - 1 && halo > 0;
  int64_t oshape[16], ext[16], sstr[16], dstr[16];
  for (int i = 0; i < ndim; ++i) oshape[i] = ext[i] = local_shape[i];
  oshape[dim] = local_shape[dim] + (has_prev ? halo : 0) + (has_next ? halo : 0);
  contiguous_strides(local_shape, ndim, elem_size, sstr);
  contiguous_strides(oshape, ndim, elem_size, dstr);
  int nb = 0;
  if (n > 1) {
    const int64_t e1[1] = {total}, s1[1] = {1};
    rc = make_box(&d.box[nb++], src, s1, r.heap + stage_off, s1, e1, 1, 1, -1);
    if (rc) return rc;
  }
  d.n_in = nb;
  char* out = static_cast<char*>(dst);
  const int64_t head = has_prev ? halo : 0;
  rc = make_box(&d.box[nb++], src, sstr, out + head * dstr[dim], dstr, ext, ndim, elem_size, -1);
  if (rc) return rc;
  ext[dim] = halo;
  if (has_prev) {
    const char* sp = r.peer_heap[g.ranks[me - 1]] + stage_off;
    rc = make_box(&d.box[nb++], sp + (local_shape[dim] - halo) * sstr[dim], sstr, out, dstr, ext,
                  ndim, elem_size, me - 1);
    if (rc) return rc;
  }
  if (has_next) {
    const char* sp = r.peer_heap[g.ranks[me + 1]] + stage_off;
    rc = make_box(&d.box[nb++], sp, sstr, out + (head + local_shape[dim]) * dstr[dim], dstr, ext,
                  ndim, elem_size, me + 1);
    if (rc) return rc;
  }
  d.n_boxes = nb;
  return launch_gather(d, n > 1, (cudaStream_t)stream);
}

int edb_box_exchange(int gid, void* dst, const int64_t* dst_shape, uint64_t stage_off,
                     const void* src, const int64_t* src_shape, int ndim, int elem_size, int nbox,
                     const int* peer, const int64_t* src_start, const int64_t* dst_start,
                     const int64_t* extents, const int64_t* peer_src_shapes, void* stream) {
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  int rc = fill_flagctx(&d.f, gid);
  if (rc) return rc;
  EDB_REQUIRE(ndim >= 1 && ndim <= 16, "edb_box_exchange: bad ndim %d", ndim);
  EDB_REQUIRE(nbox >= 0 && nbox <= kMaxBoxes - 1, "edb_box_exchange: %d boxes (max %d)", nbox,
              kMaxBoxes - 1);
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  const int64_t total = src ? numel_of(src_shape, ndim) * elem_size : 0;
  int nb = 0;
  if (total > 0 && n > 1) {
    rc = check_symm(stage_off, (size_t)total, "edb_box_exchange");
    if (rc) return rc;
    const int64_t e1[1] = {total}, s1[1] = {1};
    rc = make_box(&d.box[nb++], src, s1, r.heap + stage_off, s1, e1, 1, 1, -1);
    if (rc) return rc;
  }
  d.n_in = nb;
  int64_t dstr[16], sstr[16];
  contiguous_strides(dst_shape, ndim, elem_size, dstr);
  for (int b = 0; b < nbox; ++b) {
    const int p = peer[b];
    EDB_REQUIRE(p >= 0 && p < n, "edb_box_exchange: box %d from member %d of %d", b, p, n);
    const int64_t* pshape = peer_src_shapes + (size_t)p * ndim;
    contiguous_strides(pshape, ndim, elem_size, sstr);
    const int64_t* ss = src_start + (size_t)b * ndim;
    const int64_t* ds = dst_start + (size_t)b * ndim;
    const int64_t* ex = extents + (size_t)b * ndim;
    if (numel_of(ex, ndim) == 0) continue;
    int64_t so = 0, dof = 0;
    for (int i = 0; i < ndim; ++i) {
      EDB_REQUIRE(ss[i] >= 0 && ss[i] + ex[i] <= pshape[i] && ds[i] >= 0 &&
                      ds[i] + ex[i] <= dst_shape[i],
                  "edb_box_exchange: box %d out of bounds in dim %d", b, i);
      so += ss[i] * sstr[i];
      dof += ds[i] * dstr[i];
    }
    const char* sp = (p == me) ? static_cast<const char*>(src) : r.peer_heap[g.ranks[p]] + stage_off;
    EDB_REQUIRE(sp != nullptr, "edb_box_exchange: local box without src");
    rc = make_box(&d.box[nb++], sp + so, sstr, static_cast<char*>(dst) + dof, dstr, ex, ndim,
                  elem_size, p == me ? -1 : p);
    if (rc) return rc;
  }
  d.n_boxes = nb;
  if (n == 1 && nb == 0) return EDB_OK;
  return launch_gather(d, n > 1, (cudaStream_t)stream);
}

int edb_reduce_scatter(int gid, void* dst, uint64_t stage_off, const void* src,
                       const int64_t* shape, int ndim, int dim, int dtype, int redop,
                       float post_scale, int out_dtype, void* stream) {
  ReduceLaunch L;
  memset(&L, 0, sizeof(L));
  ReduceDesc& d = L.d;
  int rc = fill_flagctx(&d.f, gid);
  if (rc) return rc;
  EDB_REQUIRE(ndim >= 1 && ndim <= 16 && dim >= 0 && dim < ndim, "edb_reduce_scatter: bad dim");
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  // the reference asserts divisibility (sharding.py:136-137)
  EDB_REQUIRE(shape[dim] % n == 0,
              "edb_reduce_scatter: input dimension %d (%lld) must be a multiple of group_size %d",
              dim, (long long)shape[dim], n);
  const size_t es = dtype_size(dtype), oes = dtype_size(out_dtype);
  EDB_REQUIRE(es && oes, "edb_reduce_scatter: bad dtype");
  EDB_REQUIRE(!(redop == EDB_AVG && (dtype == EDB_I32 || dtype == EDB_I64)),
              "edb_reduce_scatter: avg on integer dtype");
  int64_t outer = 1, inner_el = 1;
  for (int i = 0; i < dim; ++i) outer *= shape[i];
  for (int i = dim + 1; i < ndim; ++i) inner_el *= shape[i];
  const int64_t c = shape[dim] / n;
  const int64_t chunk_b = c * inner_el * (int64_t)es;
  const int64_t total = outer * chunk_b * n;
  if (total == 0) return EDB_OK;
  if (src && out_dtype == dtype) {
    const float sc = post_scale * (redop == EDB_AVG ? 1.0f / (float)n : 1.0f);
    const int ll = ll_try(gid, /*LL_REDUCE_SCATTER*/ 2, dst, src, total, outer, chunk_b, dtype, redop,
                          sc, (cudaStream_t)stream);
    if (ll >= 0) return ll;
  }
  if (n > 1 || !src) {
    rc = check_symm(stage_off, (size_t)total, "edb_reduce_scatter");
    if (rc) return rc;
  }
  if (src && n > 1) {
    const int64_t e1[1] = {total}, s1[1] = {1};
    rc = make_box(&d.in, src, s1, r.heap + stage_off, s1, e1, 1, 1, -1);
    if (rc) return rc;
    d.has_in = 1;
  }
  const char* my_src = src ? static_cast<const char*>(src) : r.heap + stage_off;
  for (int p = 0; p < n; ++p) {
    const char* base = (p == me) ? my_src : r.peer_heap[g.ranks[p]] + stage_off;
    d.src[p] = base + (int64_t)me * chunk_b;
  }
  d.n_src = n;
  d.dst = static_cast<char*>(dst);
  d.inner = chunk_b;
  for (int k = 0; k < 4; ++k) {
    d.ext[k] = 1;
    d.sstr[k] = 0;
    d.dstr[k] = 0;
  }
  EDB_REQUIRE(outer < 0xffffffffll, "edb_reduce_scatter: too many rows");
  d.ext[3] = outer;
  d.sstr[3] = chunk_b * n;
  d.dstr[3] = c * inner_el * (int64_t)oes;
  d.dtype = dtype;
  d.out_dtype = out_dtype;
  d.redop = redop;
  d.scale = post_scale * (redop == EDB_AVG ? 1.0f / (float)n : 1.0f);
  return launch_reduce(L, (cudaStream_t)stream);
}

int edb_all_reduce(int gid, void* dst, uint64_t stage_off, uint64_t stage2_off, const void* src,
                   int64_t numel, int dtype, int redop, void* stream) {
  ReduceLaunch L;
  memset(&L, 0, sizeof(L));
  ReduceDesc& d = L.d;
  int rc = fill_flagctx(&d.f, gid);
  if (rc) return rc;
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  const size_t es = dtype_size(dtype);
  EDB_REQUIRE(es, "edb_all_reduce: bad dtype %d", dtype);
  EDB_REQUIRE(!(redop == EDB_AVG && (dtype == EDB_I32 || dtype == EDB_I64)),
              "edb_all_reduce: avg on integer dtype");
  const int64_t total = numel * (int64_t)es;
  if (total == 0) return EDB_OK;
  if (src) {
    const int ll = ll_try(gid, /*LL_ALL_REDUCE*/ 0, dst, src, total, 1, total, dtype, redop,
                          redop == EDB_AVG ? 1.0f / (float)n : 1.0f, (cudaStream_t)stream);
    if (ll >= 0) return ll;
  }
  if (n > 1 || !src) {
    rc = check_symm(stage_off, (size_t)total, "edb_all_reduce");
    if (rc) return rc;
  }
  if (src && n > 1) {
    const int64_t e1[1] = {total}, s1[1] = {1};
    rc = make_box(&d.in, src, s1, r.heap + stage_off, s1, e1, 1, 1, -1);
    if (rc) return rc;
    d.has_in = 1;
  }
  const char* my_src = src ? static_cast<const char*>(src) : r.heap + stage_off;
  d.n_src = n;
  d.dtype = d.out_dtype = dtype;
  d.redop = redop;
  d.scale = (redop == EDB_AVG ? 1.0f / (float)n : 1.0f);
  for (int k = 0; k < 4; ++k) {
    d.ext[k] = 1;
    d.sstr[k] = 0;
    d.dstr[k] = 0;
  }
  const bool two_shot = n > 1 && total > r.allreduce_oneshot_bytes;
  if (!two_shot) {
    for (int p = 0; p < n; ++p)
      d.src[p] = (p == me) ? my_src : r.peer_heap[g.ranks[p]] + stage_off;
    d.dst = static_cast<char*>(dst);
    d.inner = total;
    return launch_reduce(L, (cudaStream_t)stream);
  }
  rc = check_symm(stage2_off, (size_t)total, "edb_all_reduce(stage2)");
  if (rc) return rc;
  const int64_t epv = 16 / (int64_t)es;
  int64_t chunk = (numel + n - 1) / n;
  chunk = (chunk + epv - 1) / epv * epv;
  const int64_t chunk_b = chunk * (int64_t)es;
  auto part_lo = [&](int p) { return std::min<int64_t>(total, (int64_t)p * chunk_b); };
  auto part_hi = [&](int p) { return std::min<int64_t>(total, (int64_t)(p + 1) * chunk_b); };
  const int64_t lo = part_lo(me), hi = part_hi(me);
  for (int p = 0; p < n; ++p)
    d.src[p] = ((p == me) ? my_src : r.peer_heap[g.ranks[p]] + stage_off) + lo;
  d.dst = r.heap + stage2_off + lo;
  L.dst_b = static_cast<char*>(dst) + lo;
  d.inner = hi - lo;
  if (d.inner == 0) {  // nothing to reduce on this rank: keep the kernel in the protocol
    d.ext[3] = 0;
  }
  d.two_shot = 1;
  int np = 0;
  for (int k = 1; k < n; ++k) {
    const int p = (me + k) % n;
    const int64_t plo = part_lo(p), phi = part_hi(p);
    if (phi <= plo) continue;
    const int64_t e1[1] = {phi - plo}, s1[1] = {1};
    rc = make_box(&d.pull[np], r.peer_heap[g.ranks[p]] + stage2_off + plo, s1,
                  static_cast<char*>(dst) + plo, s1, e1, 1, 1, p);
    if (rc) return rc;
    ++np;
  }
  d.n_pull = np;
  return launch_reduce(L, (cudaStream_t)stream);
}

int edb_all_gather_push(int gid, uint64_t dst_off, const void* src, const int64_t* local_shape,
                        int ndim, int dim, int elem_size, void* stream) {
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  int rc = fill_flagctx(&d.f, gid);
  if (rc) return rc;
  EDB_REQUIRE(ndim >= 1 && ndim <= 16 && dim >= 0 && dim < ndim, "edb_all_gather_push: bad dim %d/%d",
              dim, ndim);
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  if (n <= 1) return edb_all_gather(gid, dst_off, src, local_shape, ndim, dim, elem_size, stream);
  int64_t outer = 1, rowb = elem_size;
  for (int i = 0; i < dim; ++i) outer *= local_shape[i];
  for (int i = dim; i < ndim; ++i) rowb *= local_shape[i];
  const size_t total = (size_t)outer * rowb * n;
  if (total == 0) return EDB_OK;
  rc = check_symm(dst_off, total, "edb_all_gather_push");
  if (rc) return rc;
  {
    const int ll = ll_try(gid, /*LL_ALL_GATHER*/ 1, r.heap + dst_off, src, outer * rowb, outer, rowb, 0,
                          0, 1.0f, (cudaStream_t)stream);
    if (ll >= 0) return ll;
  }
  const int64_t ext[2] = {outer, rowb};
  const int64_t s_src[2] = {rowb, 1}, s_out[2] = {rowb * n, 1};
  int nb = 0;
  for (int k = 0; k < n; ++k) {  // own buffer first, then the peers starting with the next one
    const int p = (me + k) % n;
    char* out_p = r.peer_heap[g.ranks[p]] + dst_off;
    if (p == me && out_p + (int64_t)me * rowb == static_cast<const char*>(src) && outer == 1)
      continue;  // in-place gather: my part already sits in my buffer
    rc = make_box(&d.box[nb], src, s_src, out_p + (int64_t)me * rowb, s_out, ext, 2, 1, -1);
    if (rc) return rc;
    ++nb;
  }
  d.n_in = 0;
  d.n_boxes = nb;
  return launch_gather(d, true, (cudaStream_t)stream, true);
}

int edb_all_to_all_push(int gid, uint64_t dst_off, const void* src, const int64_t* local_shape,
                        int ndim, int gather_dim, int scatter_dim, int elem_size, void* stream) {
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  int rc = fill_flagctx(&d.f, gid);
  if (rc) return rc;
  EDB_REQUIRE(ndim >= 1 && ndim <= 16 && gather_dim >= 0 && gather_dim < ndim && scatter_dim >= 0 &&
                  scatter_dim < ndim && gather_dim != scatter_dim && src != nullptr,
              "edb_all_to_all_push: bad dims g=%d s=%d ndim=%d", gather_dim, scatter_dim, ndim);
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  EDB_REQUIRE(local_shape[scatter_dim] % n == 0,
              "edb_all_to_all_push: scatter dim size %lld not divisible by group size %d",
              (long long)local_shape[scatter_dim], n);
  const int64_t total = numel_of(local_shape, ndim) * elem_size;
  if (total == 0) return EDB_OK;
  rc = check_symm(dst_off, (size_t)total, "edb_all_to_all_push");
  if (rc) return rc;
  int64_t oshape[16], ext[16], sstr[16], dstr[16];
  for (int i = 0; i < ndim; ++i) oshape[i] = ext[i] = local_shape[i];
  const int64_t cs = local_shape[scatter_dim] / n;
  oshape[gather_dim] = local_shape[gather_dim] * n;
  oshape[scatter_dim] = cs;
  ext[scatter_dim] = cs;
  contiguous_strides(local_shape, ndim, elem_size, sstr);
  contiguous_strides(oshape, ndim, elem_size, dstr);
  int nb = 0;
  for (int k = 0; k < n; ++k) {
    const int p = (me + k) % n;
    // chunk p of my tensor along scatter_dim lands at index `me` along gather_dim of p's result
    rc = make_box(&d.box[nb++], static_cast<const char*>(src) + (int64_t)p * cs * sstr[scatter_dim],
                  sstr,
                  r.peer_heap[g.ranks[p]] + dst_off +
                      (int64_t)me * local_shape[gather_dim] * dstr[gather_dim],
                  dstr, ext, ndim, elem_size, -1);
    if (rc) return rc;
  }
  d.n_in = 0;
  d.n_boxes = nb;
  return launch_gather(d, true, (cudaStream_t)stream, true);
}

// shared by reduce_scatter_push and the one-shot all_reduce_push: `pieces` = n (reduce-scatter: my
// tensor is cut into n chunks along dim, chunk p goes to member p) or 1 (all-reduce: everybody gets
// my whole tensor); slot s of the local receive buffer holds member s's contribution
static int push_reduce_impl(int gid, void* dst, uint64_t recv_off, const void* src, int64_t outer,
                            int64_t chunk_b, bool scatter, int dtype, int redop, float scale,
                            int out_dtype, const char* who, cudaStream_t st) {
  ReduceLaunch L;
  memset(&L, 0, sizeof(L));
  ReduceDesc& d = L.d;
  int rc = fill_flagctx(&d.f, gid);
  if (rc) return rc;
  Runtime& r = rt();
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  const int64_t slot_b = outer * chunk_b;  // bytes of one member's contribution to one receiver
  rc = check_symm(recv_off, (size_t)slot_b * n, who);
  if (rc) return rc;
  EDB_REQUIRE(outer < 0xffffffffll, "%s: too many rows", who);
  const int64_t ext[2] = {outer, chunk_b};
  const int64_t s_src[2] = {scatter ? chunk_b * n : chunk_b, 1}, s_slot[2] = {chunk_b, 1};
  for (int k = 0; k < n; ++k) {
    const int p = (me + 1 + k) % n;  // peers first, own slot last
    const char* sp = static_cast<const char*>(src) + (scatter ? (int64_t)p * chunk_b : 0);
    rc = make_box(&d.pull[k], sp, s_src, r.peer_heap[g.ranks[p]] + recv_off + (int64_t)me * slot_b,
                  s_slot, ext, 2, 1, -1);
    if (rc) return rc;
  }
  d.n_pull = n;
  for (int s = 0; s < n; ++s) d.src[s] = r.heap + recv_off + (int64_t)s * slot_b;
  d.n_src = n;
  d.dst = static_cast<char*>(dst);
  d.inner = slot_b;  // the slots are contiguous: one long row
  for (int k = 0; k < 4; ++k) {
    d.ext[k] = 1;
    d.sstr[k] = 0;
    d.dstr[k] = 0;
  }
  d.dtype = dtype;
  d.out_dtype = out_dtype;
  d.redop = redop;
  d.scale = scale;
  L.push = 1;
  return launch_reduce(L, st);
}

int edb_reduce_scatter_push(int gid, void* dst, uint64_t recv_off, const void* src,
                            const int64_t* shape, int ndim, int dim, int dtype, int redop,
                            float post_scale, int out_dtype, void* stream) {
  Runtime& r = rt();
  if (!r.inited) return set_error(EDB_E_STATE, "runtime not initialised (call edb_init)");
  if (gid < 0 || gid >= r.ngroups) return set_error(EDB_E_INVALID, "bad group id %d", gid);
  const int n = r.groups[gid].n;
  if (n <= 1 || src == nullptr)
    return edb_reduce_scatter(gid, dst, recv_off, src, shape, ndim, dim, dtype, redop, post_scale,
                              out_dtype, stream);
  EDB_REQUIRE(ndim >= 1 && ndim <= 16 && dim >= 0 && dim < ndim, "edb_reduce_scatter_push: bad dim");
  EDB_REQUIRE(shape[dim] % n == 0,
              "edb_reduce_scatter_push: input dimension %d (%lld) must be a multiple of group_size %d",
              dim, (long long)shape[dim], n);
  const size_t es = dtype_size(dtype);
  EDB_REQUIRE(es && dtype_size(out_dtype), "edb_reduce_scatter_push: bad dtype");
  EDB_REQUIRE(!(redop == EDB_AVG && (dtype == EDB_I32 || dtype == EDB_I64)),
              "edb_reduce_scatter_push: avg on integer dtype");
  int64_t outer = 1, inner_el = 1;
  for (int i = 0; i < dim; ++i) outer *= shape[i];
  for (int i = dim + 1; i < ndim; ++i) inner_el *= shape[i];
  const int64_t chunk_b = shape[dim] / n * inner_el * (int64_t)es;
  if (outer * chunk_b == 0) return EDB_OK;
  if (out_dtype == dtype) {
    const float sc = post_scale * (redop == EDB_AVG ? 1.0f / (float)n : 1.0f);
    const int ll = ll_try(gid, /*LL_REDUCE_SCATTER*/ 2, dst, src, outer * chunk_b * n, outer, chunk_b,
                          dtype, redop, sc, (cudaStream_t)stream);
    if (ll >= 0) return ll;
  }
  return push_reduce_impl(gid, dst, recv_off, src, outer, chunk_b, true, dtype, redop,
                          post_scale * (redop == EDB_AVG ? 1.0f / (float)n : 1.0f), out_dtype,
                          "edb_reduce_scatter_push", (cudaStream_t)stream);
}

int edb_all_reduce_push(int gid, uint64_t out_off, uint64_t recv_off, const void* src, int64_t numel,
                        int dtype, int redop, void* stream) {
  Runtime& r = rt();
  if (!r.inited) return set_error(EDB_E_STATE, "runtime not initialised (call edb_init)");
  if (gid < 0 || gid >= r.ngroups) return set_error(EDB_E_INVALID, "bad group id %d", gid);
  const Group& g = r.groups[gid];
  const int n = g.n, me = g.me;
  const size_t es = dtype_size(dtype);
  EDB_REQUIRE(es && src != nullptr, "edb_all_reduce_push: bad dtype %d / src", dtype);
  EDB_REQUIRE(!(redop == EDB_AVG && (dtype == EDB_I32 || dtype == EDB_I64)),
              "edb_all_reduce_push: avg on integer dtype");
  const int64_t total = numel * (int64_t)es;
  if (total == 0) return EDB_OK;
  int rc = check_symm(out_off, (size_t)total, "edb_all_reduce_push");
  if (rc) return rc;
  char* out = r.heap + out_off;
  if (n <= 1) return edb_copy(out, src, (size_t)total, stream);
  const float scale = redop == EDB_AVG ? 1.0f / (float)n : 1.0f;
  {
    const int ll = ll_try(gid, /*LL_ALL_REDUCE*/ 0, out, src, total, 1, total, dtype, redop, scale,
                          (cudaStream_t)stream);
    if (ll >= 0) return ll;
  }
  const int64_t per = 16 / (int64_t)es * n;
  // one-shot moves (n-1) x the tensor per rank, two-shot 2(n-1)/n x in two launches: with two
  // members the volumes are equal, so the single launch wins up to much larger tensors
  const int64_t thr = r.allreduce_oneshot_bytes * (n == 2 ? 8 : 1);
  const bool two_shot = total > thr && numel % per == 0;
  if (!two_shot)  // everybody receives everybody's tensor (receive buffer: n * total bytes)
    return push_reduce_impl(gid, out, recv_off, src, 1, total, false, dtype, redop, scale, dtype,
                            "edb_all_reduce_push", (cudaStream_t)stream);
  // two-shot: reduce-scatter push (my reduced chunk lands in place, at out + me*chunk), then an
  // in-place all-gather push of the chunks
  const int64_t chunk_b = total / n;
  rc = push_reduce_impl(gid, out + (int64_t)me * chunk_b, recv_off, src, 1, chunk_b, true, dtype,
                        redop, scale, dtype, "edb_all_reduce_push", (cudaStream_t)stream);
  if (rc) return rc;
  const int64_t shp[1] = {chunk_b};
  return edb_all_gather_push(gid, out_off, out + (int64_t)me * chunk_b, shp, 1, 0, 1, stream);
}

int edb_epoch_barrier(int gid, void* stream) {
  FlagCtx f;
  int rc = fill_flagctx(&f, gid);
  if (rc) return rc;
  if (f.n <= 1) return EDB_OK;
  k_epoch_barrier<<<1, 32, 0, (cudaStream_t)stream>>>(f);
  count_launch();
  return cuda_check(cudaGetLastError(), "k_epoch_barrier launch");
}

}  // extern "C"
