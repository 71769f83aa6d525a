// tb_common.cuh — context, workspace buffers, error plumbing and the device-wide primitives
// (3-phase scans, stable LSD radix sort) shared by the collapse and coverage pipelines.
// sm_100a only. No CPU fallback: every entry point fails when CUDA fails.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../include/tiebrush_b200.h"

#define TB_CUDA(call)                                                                                  \
  do {                                                                                                 \
    cudaError_t e__ = (call);                                                                          \
    if (e__ != cudaSuccess) {                                                                          \
      ctx->set_error("CUDA error %s at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return 1;                                                                                        \
    }                                                                                                  \
  } while (0)

struct DevBuf {  // grow-only device buffer
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() { return (T*)p; }
};

struct HostBuf {  // grow-only pinned host buffer
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
  template <class T> T* as() { return (T*)p; }
};

enum { TB_NBUF = 52, TB_NBAMBUF = 28 };

struct tb_ctx {
  int device = 0;
  int n_samples = 0;
  int mode = 0;
  uint32_t flag_mask = 0;
  int max_nh = TB_NO_MAX_NH;
  int min_qual = -1;
  int keep_bits = 0;
  int collapse_same = 0;
  int sm_count = 148;
  size_t smem_optin = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[16] = {};
  int profiling = 0;
  float last_ms[16] = {};   // per-stage device times of the last call (see tb_last_kernel_ms)
  int64_t launches = 0;
  int64_t last_heavy = 0;   // slots redone by the full-size tile launch in the last collapse call
  int last_yd_path = 0;     // YD stage of the last collapse call: 0 parallel (frontier + link bitmaps), 1 sequential lists
  int64_t last_yd_stat[4] = {};   // YD stage of the last collapse call: members | sub-chains | compact length | 1024-group blocks
  int last_path = 0;        // front end of the last collapse call: 0 tile, 1 ordered (by options), 2 ordered (table overflow fallback)
  int64_t last_ord_deep = 0;   // ordered front end, last call: start positions handled by the warp kernel
  int last_cov_exact = 0;   // last coverage call took the exact ordered-double path (weights that are not multiples of 2^-20)
  int last_tile_gen = 0;    // 1 once a collapse call has run the tile kernel (col_tile_kernel)
  int64_t last_tile_slots = 0;   // slots of the last tile-path call that used the heavy list (256-thread geometry)
  int64_t last_tile_runs[3] = {0, 0, 0};   // last tile-path call: records streamed, heads probed, full-warp probe batches
  std::string err;
  DevBuf buf[TB_NBUF];   // workspace slots (see the enum in each pipeline)
  DevBuf in_stage[20];   // device copies of host input arrays
  DevBuf out_stage[9];   // device output arrays when the caller wants host results: runs in 0..3, junction rows in 4..8
  HostBuf pinned[2];     // small pinned readback areas
  // multi-GPU (shard.cu): NCCL communicator of this context's rank, workspace, statistics of the last sharded call
  void* comm = nullptr; int rank = 0; int world = 1;
  cudaStream_t gather_stream = nullptr;   // second stream: ordered gather overlapped with the windows
  DevBuf shard_buf[19];
  int64_t shard_stat[8] = {};   // lead records received | sent | ranks received from | bytes sent (halo) | seam records | bytes moved by the gather
  int64_t stream_windows = 0;   // windows of the last tc_coverage_stream / tc_shard_coverage call
  // BAM decode (bgzf.cu): workspace, and the bundle tc_coverage_bam holds for its next call: records [bam_from, bam_from +
  // bam_held) of column set bam_set, whose CIGAR words start at bam_cbase (bam_hcig words)
  DevBuf bam_buf[TB_NBAMBUF];
  HostBuf bam_pinned;
  int bam_set = 0;
  int64_t bam_from = 0, bam_held = 0;
  uint32_t bam_cbase = 0, bam_hcig = 0;
  void set_error(const char* fmt, ...);
};

extern std::string g_tb_global_error;

static inline unsigned tb_grid_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// a host input array on the device (device arrays and NULL pass through)
template <class T>
static int tb_stage_in(tb_ctx* ctx, DevBuf& b, const T* src, size_t count, int on_device, const T** out) {
  if (on_device || src == nullptr) { *out = src; return 0; }
  TB_CUDA(b.ensure(count * sizeof(T) + 16));
  TB_CUDA(cudaMemcpyAsync(b.p, src, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  *out = (const T*)b.p;
  return 0;
}

// tc_coverage_stream's view of one window (coverage.cu): the record that follows the window in the stream, and how many
// records of the window were processed (all but the last bundle when that record continues it)
struct CovExt { int has_next; int32_t next_tid, next_pos; int64_t consumed; };

// -------------------------------------------------------------------------------------------------
// small device helpers
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t tb_mix64(uint64_t x) {  // splitmix64 finalizer
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ULL;
  x ^= x >> 27; x *= 0x94d049bb133111ebULL;
  x ^= x >> 31;
  return x;
}

// shuffles for arbitrary trivially-copyable T (word by word)
template <class T>
__device__ __forceinline__ T tb_shfl_up(T v, int d) {
  static_assert(sizeof(T) % 4 == 0, "T must be a multiple of 4 bytes");
  union { T t; uint32_t w[sizeof(T) / 4]; } u; u.t = v;
#pragma unroll
  for (int k = 0; k < (int)(sizeof(T) / 4); ++k) u.w[k] = __shfl_up_sync(0xffffffffu, u.w[k], d);
  return u.t;
}
template <class T>
__device__ __forceinline__ T tb_shfl_down(T v, int d) {
  static_assert(sizeof(T) % 4 == 0, "T must be a multiple of 4 bytes");
  union { T t; uint32_t w[sizeof(T) / 4]; } u; u.t = v;
#pragma unroll
  for (int k = 0; k < (int)(sizeof(T) / 4); ++k) u.w[k] = __shfl_down_sync(0xffffffffu, u.w[k], d);
  return u.t;
}

__device__ __forceinline__ int tb_lane() { return threadIdx.x & 31; }
__device__ __forceinline__ int tb_warp() { return threadIdx.x >> 5; }

// -------------------------------------------------------------------------------------------------
// Device-wide scan, 3 phases (block reduce -> single-block scan of block aggregates -> block downsweep).
// Op must provide:  typedef T;  static T identity();  static T combine(T a, T b)  (associative).
// Reads the input twice; used for O(window span) and O(records) arrays that are small next to the
// record streams. Block = 256 threads x 8 items.
// -------------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

template <class Op>
__device__ __forceinline__ typename Op::T tb_block_reduce(typename Op::T v, typename Op::T* s_warp /*[32]*/) {
  typedef typename Op::T T;
  // ascending distances keep the operands in element order (lane l ends with v_l + ... + v_{l+2d-1}), which matters for
  // non-commutative operators such as the segmented maximum; lane 0 holds the warp total
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    T o = tb_shfl_down(v, d);
    v = Op::combine(v, o);
  }
  __syncthreads();
  if (tb_lane() == 0) s_warp[tb_warp()] = v;
  __syncthreads();
  T r = Op::identity();
  int nw = blockDim.x >> 5;
  for (int w = 0; w < nw; ++w) r = Op::combine(r, s_warp[w]);
  return r;  // every thread gets the block total (order-preserving: warp order == element order)
}

// exclusive scan of one value per thread across the block; returns the exclusive prefix, *total gets block total.
// Two levels: inclusive scan inside every warp, then warp 0 scans the (<= 32) warp totals with shuffles.
// s_warp holds 33 elements. Operand order is preserved (non-commutative operators are fine).
template <class Op>
__device__ __forceinline__ typename Op::T tb_block_exscan(typename Op::T v, typename Op::T* s_warp /*[33]*/, typename Op::T* total) {
  typedef typename Op::T T;
  const int lane = tb_lane(), warp = tb_warp();
  T inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    T o = tb_shfl_up(inc, d);
    if (lane >= d) inc = Op::combine(o, inc);
  }
  __syncthreads();  // s_warp may still be read from a previous call
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int nw = blockDim.x >> 5;
    T x = lane < nw ? s_warp[lane] : Op::identity();
    T xi = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      T o = tb_shfl_up(xi, d);
      if (lane >= d) xi = Op::combine(o, xi);
    }
    T xe = tb_shfl_up(xi, 1);
    if (lane == 0) xe = Op::identity();
    s_warp[lane] = xe;              // exclusive prefix of the warp totals
    if (lane == 31) s_warp[32] = xi;  // block total (identity padding on the right)
  }
  __syncthreads();
  T exc = tb_shfl_up(inc, 1);
  if (lane == 0) exc = Op::identity();
  if (total) *total = s_warp[32];
  return Op::combine(s_warp[warp], exc);
}

template <class Op, class InF>
__global__ void __launch_bounds__(SCAN_THREADS) tb_scan_reduce_kernel(InF in, int64_t n, typename Op::T* block_agg) {
  typedef typename Op::T T;
  __shared__ T s_warp[33];
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  T acc = Op::identity();
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    int64_t i = base + k;
    if (i < n) acc = Op::combine(acc, in(i));
  }
  T tot = tb_block_reduce<Op>(acc, s_warp);
  if (threadIdx.x == 0) block_agg[blockIdx.x] = tot;
}

// single block: exclusive scan of block aggregates in place; total written to agg[nblocks]
template <class Op>
__global__ void __launch_bounds__(1024) tb_scan_spine_kernel(typename Op::T* agg, int64_t nblocks) {
  typedef typename Op::T T;
  __shared__ T s_warp[33];
  __shared__ T s_carry;
  if (threadIdx.x == 0) s_carry = Op::identity();
  __syncthreads();
  for (int64_t base = 0; base < nblocks; base += blockDim.x) {
    int64_t i = base + threadIdx.x;
    T v = (i < nblocks) ? agg[i] : Op::identity();
    T tot;
    T exc = tb_block_exscan<Op>(v, s_warp, &tot);
    T carry = s_carry;
    if (i < nblocks) agg[i] = Op::combine(carry, exc);
    __syncthreads();
    if (threadIdx.x == 0) s_carry = Op::combine(carry, tot);
    __syncthreads();
  }
  if (threadIdx.x == 0) agg[nblocks] = s_carry;
}

// downsweep: out(i, exclusive_prefix, inclusive_prefix)
template <class Op, class InF, class OutF>
__global__ void __launch_bounds__(SCAN_THREADS) tb_scan_down_kernel(InF in, int64_t n, const typename Op::T* block_pre, OutF out) {
  typedef typename Op::T T;
  __shared__ T s_warp[33];
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  T v[SCAN_ITEMS];
  T acc = Op::identity();
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    int64_t i = base + k;
    v[k] = (i < n) ? in(i) : Op::identity();
    acc = Op::combine(acc, v[k]);
  }
  T exc = tb_block_exscan<Op>(acc, s_warp, (T*)nullptr);
  T run = Op::combine(block_pre[blockIdx.x], exc);
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    int64_t i = base + k;
    T inc = Op::combine(run, v[k]);
    if (i < n) out(i, run, inc);
    run = inc;
  }
}

// -------------------------------------------------------------------------------------------------
// Decoupled look-back (single-pass device-wide prefixes): a tile publishes one 64-bit state word,
// 2 flag bits | 62-bit payload: first its own aggregate (LB_AGG), then its inclusive prefix (LB_INC)
// once its look-back over the predecessors is done. Tiles must take their ids from a ticket counter
// so that every predecessor of a running tile is itself running or finished. The spin is bounded
// and reports through *fail instead of hanging the device.
// -------------------------------------------------------------------------------------------------
constexpr unsigned long long LB_AGG = 1ULL << 62, LB_INC = 2ULL << 62, LB_MASK = (1ULL << 62) - 1ULL;

__device__ __forceinline__ unsigned long long lb_load(const unsigned long long* p) { return *reinterpret_cast<const volatile unsigned long long*>(p); }
__device__ __forceinline__ void lb_store(unsigned long long* p, unsigned long long v) { *reinterpret_cast<volatile unsigned long long*>(p) = v; }

// exclusive prefix (max or sum of the 62-bit payloads) of the tiles before `tile`; called by one whole warp
template <bool IS_MAX>
__device__ unsigned long long lb_lookback(const unsigned long long* st, long long tile, long long* fail) {
  const int lane = threadIdx.x & 31;
  unsigned long long acc = 0;   // identity of both operators (payloads are non-negative)
  int spins = 0;
  for (long long idx = tile - 1; idx >= 0; idx -= 32) {
    const long long j = idx - lane;
    unsigned long long w = j >= 0 ? lb_load(&st[j]) : LB_INC;   // before the first tile: an inclusive identity
    while (__any_sync(0xffffffffu, (w >> 62) == 0)) {
      if (++spins > (1 << 22)) { *fail = 1; break; }
      if ((w >> 62) == 0) w = lb_load(&st[j]);
    }
    const unsigned inc = __ballot_sync(0xffffffffu, (w >> 62) == 2);
    const int first = inc ? __ffs(inc) - 1 : 32;
    unsigned long long v = lane <= first ? (w & LB_MASK) : 0ULL;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, d);
      v = IS_MAX ? (v > o ? v : o) : v + o;
    }
    acc = IS_MAX ? (acc > v ? acc : v) : acc + v;
    if (inc) break;
  }
  return acc;
}


struct OpSumU32 { typedef uint32_t T; __host__ __device__ static T identity() { return 0; } __host__ __device__ static T combine(T a, T b) { return a + b; } };
struct OpSumI64 { typedef long long T; __host__ __device__ static T identity() { return 0; } __host__ __device__ static T combine(T a, T b) { return a + b; } };
struct OpMaxU64 { typedef unsigned long long T; __host__ __device__ static T identity() { return 0; } __host__ __device__ static T combine(T a, T b) { return a > b ? a : b; } };

static inline int64_t tb_scan_blocks(int64_t n) { return (n + SCAN_TILE - 1) / SCAN_TILE; }

// host driver; `agg` must hold tb_scan_blocks(n)+1 elements of Op::T. After the call agg[nblocks] = grand total.
template <class Op, class InF, class OutF>
static inline cudaError_t tb_device_scan(tb_ctx* ctx, InF in, int64_t n, typename Op::T* agg, OutF out) {
  int64_t nb = tb_scan_blocks(n);
  if (nb == 0) {
    tb_scan_spine_kernel<Op><<<1, 1024, 0, ctx->stream>>>(agg, 0);
    ctx->launches += 1;
    return cudaGetLastError();
  }
  tb_scan_reduce_kernel<Op, InF><<<(unsigned)nb, SCAN_THREADS, 0, ctx->stream>>>(in, n, agg);
  tb_scan_spine_kernel<Op><<<1, 1024, 0, ctx->stream>>>(agg, nb);
  tb_scan_down_kernel<Op, InF, OutF><<<(unsigned)nb, SCAN_THREADS, 0, ctx->stream>>>(in, n, agg, out);
  ctx->launches += 3;
  return cudaGetLastError();
}

// -------------------------------------------------------------------------------------------------
// Stable LSD radix sort of (u64 key, u32 value) pairs, 8 bits per pass, hand-written:
//   pass = per-block digit histogram -> device scan of the (digit-major) table -> stable scatter.
// Stability inside a block: each warp owns a contiguous sub-tile and walks it in order with
// __match_any_sync ranks; per-warp digit counters are prefix-summed across warps.
// -------------------------------------------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_STEPS = 8;                       // 32-element steps per warp
constexpr int RS_TILE = RS_THREADS * RS_STEPS;    // 2048 elements per block

static __global__ void __launch_bounds__(RS_THREADS) tb_rs_hist_kernel(const uint64_t* __restrict__ keys, int64_t n, int shift,
                                                                uint32_t* __restrict__ table, int64_t nblocks) {
  __shared__ uint32_t cnt[256];
  cnt[threadIdx.x] = 0;
  __syncthreads();
  int64_t base = (int64_t)blockIdx.x * RS_TILE;
  for (int s = 0; s < RS_STEPS; ++s) {
    int64_t i = base + (int64_t)tb_warp() * (RS_STEPS * 32) + s * 32 + tb_lane();
    if (i < n) atomicAdd(&cnt[(keys[i] >> shift) & 0xff], 1u);
  }
  __syncthreads();
  table[(int64_t)threadIdx.x * nblocks + blockIdx.x] = cnt[threadIdx.x];
}

static __global__ void __launch_bounds__(RS_THREADS) tb_rs_scatter_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                                   int64_t n, int shift, const uint32_t* __restrict__ table_scanned,
                                                                   int64_t nblocks, uint64_t* __restrict__ okeys, uint32_t* __restrict__ ovals) {
  __shared__ uint32_t cnt[RS_WARPS][256];
  for (int w = 0; w < RS_WARPS; ++w) cnt[w][threadIdx.x] = 0;
  __syncthreads();
  int64_t wbase = (int64_t)blockIdx.x * RS_TILE + (int64_t)tb_warp() * (RS_STEPS * 32);
  uint64_t k[RS_STEPS];
  uint32_t v[RS_STEPS];
  const unsigned lt = (1u << tb_lane()) - 1u;
  // phase a: per-warp digit counts
#pragma unroll
  for (int s = 0; s < RS_STEPS; ++s) {
    int64_t i = wbase + s * 32 + tb_lane();
    bool ok = i < n;
    k[s] = ok ? keys[i] : 0;
    v[s] = ok ? vals[i] : 0;
    unsigned d = ok ? (unsigned)((k[s] >> shift) & 0xff) : 256u;
    unsigned peers = __match_any_sync(0xffffffffu, d);
    if (ok && (peers & lt) == 0) cnt[tb_warp()][d] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  // phase b: thread d turns counts into starting offsets per warp
  {
    unsigned d = threadIdx.x;
    uint32_t run = table_scanned[(int64_t)d * nblocks + blockIdx.x];
    for (int w = 0; w < RS_WARPS; ++w) { uint32_t c = cnt[w][d]; cnt[w][d] = run; run += c; }
  }
  __syncthreads();
  // phase c: stable scatter
#pragma unroll
  for (int s = 0; s < RS_STEPS; ++s) {
    int64_t i = wbase + s * 32 + tb_lane();
    bool ok = i < n;
    unsigned d = ok ? (unsigned)((k[s] >> shift) & 0xff) : 256u;
    unsigned peers = __match_any_sync(0xffffffffu, d);
    if (ok) {
      uint32_t dst = cnt[tb_warp()][d] + __popc(peers & lt);
      okeys[dst] = k[s];
      ovals[dst] = v[s];
    }
    __syncwarp();
    if (ok && (peers & lt) == 0) cnt[tb_warp()][d] += __popc(peers);
    __syncwarp();
  }
}

struct RsTableIn { const uint32_t* t; __device__ uint32_t operator()(int64_t i) const { return t[i]; } };
struct RsTableOut { uint32_t* t; __device__ void operator()(int64_t i, uint32_t exc, uint32_t) const { t[i] = exc; } };

// Sorts n pairs by key bits [lo_bit, hi_bit). keys/vals are ping-ponged with kalt/valt; returns in *res_k/*res_v
// the buffers holding the result. table: 256*nblocks u32; agg: scan aggregates (tb_scan_blocks(256*nblocks)+1 u32).
static inline cudaError_t tb_radix_sort(tb_ctx* ctx, uint64_t* keys, uint32_t* vals, uint64_t* kalt, uint32_t* valt, int64_t n,
                                        int lo_bit, int hi_bit, uint32_t* table, uint32_t* agg, uint64_t** res_k, uint32_t** res_v) {
  int64_t nb = (n + RS_TILE - 1) / RS_TILE;
  uint64_t* ck = keys; uint32_t* cv = vals; uint64_t* ok = kalt; uint32_t* ov = valt;
  for (int shift = lo_bit; shift < hi_bit && n > 0; shift += 8) {
    tb_rs_hist_kernel<<<(unsigned)nb, RS_THREADS, 0, ctx->stream>>>(ck, n, shift, table, nb);
    ctx->launches += 1;
    RsTableIn tin{table}; RsTableOut tout{table};
    cudaError_t e = tb_device_scan<OpSumU32>(ctx, tin, 256 * nb, agg, tout);
    if (e != cudaSuccess) return e;
    tb_rs_scatter_kernel<<<(unsigned)nb, RS_THREADS, 0, ctx->stream>>>(ck, cv, n, shift, table, nb, ok, ov);
    ctx->launches += 1;
    uint64_t* tk = ck; ck = ok; ok = tk;
    uint32_t* tv = cv; cv = ov; ov = tv;
  }
  *res_k = ck; *res_v = cv;
  return cudaGetLastError();
}
static inline size_t tb_radix_table_elems(int64_t n) { return (size_t)256 * (size_t)((n + RS_TILE - 1) / RS_TILE) + 8; }
static inline size_t tb_radix_agg_elems(int64_t n) { return (size_t)tb_scan_blocks(256 * ((n + RS_TILE - 1) / RS_TILE)) + 8; }

// -------------------------------------------------------------------------------------------------
// CIGAR walk shared by both pipelines: GSamRecord::setupCoordinates (reference src/GSam.cpp:351-417)
// -------------------------------------------------------------------------------------------------
#define TB_OP_M 0
#define TB_OP_I 1
#define TB_OP_D 2
#define TB_OP_N 3
#define TB_OP_S 4
#define TB_OP_H 5
#define TB_OP_P 6
#define TB_OP_EQ 7
#define TB_OP_X 8
