// shard.cu — tiecov over long streams and over several GPUs (SURVEY §8e; reference counterparts: the bundle invariant
// src/tiecov.cpp:443-481, the global junction counter :92-94, and tiewrap.py:42-123, the reference's only parallel mode).
//
//   tc_coverage_stream   one coordinate-sorted stream slice, cut into windows of at most `window` records AT BUNDLE HEADS: a
//                        window whose last bundle is continued by the record behind it leaves that bundle to the next
//                        window (CovExt, coverage.cu), so every window holds whole bundles and the concatenated outputs are
//                        those of one pass. Works on device-resident and on host arrays (one H2D copy per window).
//   tc_shard_coverage    one rank's part of a run that is sharded by coordinate over the GPUs of a box, one process (or
//                        thread) per GPU. A bundle belongs to the rank that holds its first record: the records a rank
//                        holds of a bundle that was opened further left (its "lead") travel to that owner over NCCL
//                        (ncclAllGather of the open-bundle state: maximum (tid,end) key and lead sizes; grouped
//                        ncclSend / ncclRecv of the lead records' columns), the owner processes them with the rest of the
//                        bundle. Every rank then works on whole bundles only: no stitching, results identical to one GPU.
//   tc_shard_gather      ordered gather of the per-rank runs / junction rows on rank 0 (ncclAllGather of the counts,
//                        grouped ncclSend / ncclRecv of the rows); the junction numbering base of every rank
//                        (JUNC%08d is a global counter, tiecov.cpp:92-94) is the prefix sum of the counts.
//
// NCCL is loaded at run time (dlopen of libnccl.so.2: inside a PyTorch process that is the library torch already
// mapped); a single-GPU run never touches it.
#include <dlfcn.h>
#include <nccl.h>
#include <algorithm>
#include <functional>
#include "tc_columns.cuh"

int tc_coverage_impl(tb_ctx* ctx, const tc_soa_in* in, tc_runs_out* runs, tc_juncs_out* juncs, const int32_t* yx, CovExt* ext);

namespace {

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  std::string err;
  bool load() {
    if (lib) return true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) { lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
    if (!lib) { err = std::string("cannot load libnccl.so.2: ") + dlerror(); return false; }
#define TB_NCCL_SYM(field, name) do { *(void**)(&field) = dlsym(lib, name); if (!field) { err = std::string("libnccl lacks ") + name; lib = nullptr; return false; } } while (0)
    TB_NCCL_SYM(GetUniqueId, "ncclGetUniqueId"); TB_NCCL_SYM(CommInitRank, "ncclCommInitRank"); TB_NCCL_SYM(CommDestroy, "ncclCommDestroy");
    TB_NCCL_SYM(GetErrorString, "ncclGetErrorString"); TB_NCCL_SYM(AllGather, "ncclAllGather"); TB_NCCL_SYM(Send, "ncclSend");
    TB_NCCL_SYM(Recv, "ncclRecv"); TB_NCCL_SYM(GroupStart, "ncclGroupStart"); TB_NCCL_SYM(GroupEnd, "ncclGroupEnd");
#undef TB_NCCL_SYM
    return true;
  }
};
NcclApi g_nccl;

#define TB_NCCL(call)                                                                                           \
  do {                                                                                                          \
    ncclResult_t r__ = (call);                                                                                  \
    if (r__ != ncclSuccess) { ctx->set_error("NCCL error %s at %s:%d: %s", #call, __FILE__, __LINE__, g_nccl.GetErrorString(r__)); return 1; } \
  } while (0)

// workspace slots of this file in ctx->shard_buf: SB_TAIL (the leads received from the right) and SB_SEAM (the seam window)
// are record sets of 8 slots each (tc_alloc_records)
enum { SB_GATHER = 0, SB_SEND, SB_GROUND, SB_TAIL, SB_SEAM = SB_TAIL + 8, SB_COUNT_ = SB_SEAM + 8 };
static_assert(SB_COUNT_ <= (int)(sizeof(tb_ctx::shard_buf) / sizeof(DevBuf)), "raise tb_ctx::shard_buf");

// ---- open-bundle state of a slice: maximum (tid << 32 | end) key over its records. Only the records of the LAST reference
// id can hold it (tids never decrease), so a one-thread binary search finds where they start and the reduction reads
// that part only. ----
__global__ void shard_last_tid_kernel(int64_t n, const int32_t* __restrict__ tid, long long* __restrict__ start) {
  const int32_t t = tid[n - 1];
  int64_t lo = 0, hi = n - 1;   // first i with tid[i] == t
  while (lo < hi) { const int64_t mid = lo + ((hi - lo) >> 1); if (tid[mid] >= t) hi = mid; else lo = mid + 1; }
  *start = lo;
}
__global__ void __launch_bounds__(256) shard_maxkey_kernel(int64_t n, const long long* __restrict__ start, const int32_t* __restrict__ tid, const int32_t* __restrict__ pos,
                                                           const uint32_t* __restrict__ cig_off, const uint32_t* __restrict__ cigar, unsigned long long* __restrict__ out) {
  unsigned long long m = 0;
  for (int64_t i = *start + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int l = 0;
    for (uint32_t c = cig_off[i]; c < cig_off[i + 1]; ++c) { const uint32_t w = cigar[c]; if ((0x18Du >> (w & 0xf)) & 1u) l += (int)(w >> 4); }
    const unsigned long long key = ((unsigned long long)(uint32_t)tid[i] << 32) | (uint32_t)(pos[i] + l);
    m = key > m ? key : m;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) { const unsigned long long o = __shfl_xor_sync(0xffffffffu, m, d); m = o > m ? o : m; }
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// ---- lead of a slice: the records before its first bundle head, given the open-bundle state `ein` of everything left of
// it. Chunks of LEAD_BLOCKS x 1024 records, three small kernels per chunk (a lead can be 10^6 records in a deep stream:
// one block walking it would take milliseconds): block maxima of the keys -> their exclusive prefix maximum (one block,
// seeded with the carry of the chunks before) -> every block rescans its records against that carry and the first head of
// the chunk wins an atomicMin. state[0] = carry (in/out), state[1] = first head (or -1). ----
constexpr int LEAD_BLOCKS = 4096;
__device__ __forceinline__ unsigned long long shard_key(int64_t i, const int32_t* tid, const int32_t* pos, const uint32_t* cig_off, const uint32_t* cigar) {
  int l = 0;
  for (uint32_t c = cig_off[i]; c < cig_off[i + 1]; ++c) { const uint32_t w = cigar[c]; if ((0x18Du >> (w & 0xf)) & 1u) l += (int)(w >> 4); }
  return ((unsigned long long)(uint32_t)tid[i] << 32) | (uint32_t)(pos[i] + l);
}
__global__ void __launch_bounds__(1024) shard_lead_max_kernel(int64_t base, int64_t n, const int32_t* __restrict__ tid, const int32_t* __restrict__ pos,
                                                              const uint32_t* __restrict__ cig_off, const uint32_t* __restrict__ cigar, unsigned long long* __restrict__ bmax) {
  __shared__ unsigned long long s_w[33];
  const int64_t i = base + (int64_t)blockIdx.x * 1024 + threadIdx.x;
  const unsigned long long key = i < n ? shard_key(i, tid, pos, cig_off, cigar) : 0ULL;
  const unsigned long long tot = tb_block_reduce<OpMaxU64>(key, s_w);
  if (threadIdx.x == 0) bmax[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(1024) shard_lead_scan_kernel(unsigned long long* __restrict__ bmax, int nblocks, unsigned long long* __restrict__ state) {
  __shared__ unsigned long long s_w[33];
  unsigned long long carry = state[0];
  for (int b0 = 0; b0 < nblocks; b0 += 1024) {
    const int b = b0 + (int)threadIdx.x;
    const unsigned long long v = b < nblocks ? bmax[b] : 0ULL;
    unsigned long long tot;
    const unsigned long long exc = tb_block_exscan<OpMaxU64>(v, s_w, &tot);
    if (b < nblocks) bmax[b] = exc > carry ? exc : carry;   // maximum key of everything before block b
    carry = tot > carry ? tot : carry;
    __syncthreads();
  }
  if (threadIdx.x == 0) state[0] = carry;
}
__global__ void __launch_bounds__(1024) shard_lead_head_kernel(int64_t base, int64_t n, const int32_t* __restrict__ tid, const int32_t* __restrict__ pos,
                                                               const uint32_t* __restrict__ cig_off, const uint32_t* __restrict__ cigar,
                                                               const unsigned long long* __restrict__ bpre, unsigned long long* __restrict__ state) {
  __shared__ unsigned long long s_w[33];
  const int64_t i = base + (int64_t)blockIdx.x * 1024 + threadIdx.x;
  const unsigned long long key = i < n ? shard_key(i, tid, pos, cig_off, cigar) : 0ULL;
  const unsigned long long exc = tb_block_exscan<OpMaxU64>(key, s_w, (unsigned long long*)nullptr);
  const unsigned long long carry = bpre[blockIdx.x];
  const unsigned long long run = exc > carry ? exc : carry;
  if (i < n) {
    const bool head = run == 0 || tid[i] != (int)(run >> 32) || (pos[i] + 1) > (int)(uint32_t)run;   // tiecov.cpp:443
    if (head) atomicMin(&state[1], (unsigned long long)i);
  }
}

// see tc_copy_records. The source's first offset is read here, so a piece whose offsets arrived from another rank needs no
// host round trip.
__global__ void __launch_bounds__(256) tc_copy_records_kernel(TcRecords src, int64_t from, int64_t m, TcRecords dst, int64_t r, uint32_t w, uint32_t words) {
  const uint32_t c0 = src.cig_off[from];
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k <= m || k < (int64_t)words; k += (int64_t)gridDim.x * blockDim.x) {
    if (k <= m) dst.cig_off[r + k] = src.cig_off[from + k] - c0 + w;
    if (k < m) {
      const int64_t s = from + k, d = r + k;
      if (src.tid && dst.tid) dst.tid[d] = src.tid[s];
      if (src.pos && dst.pos) dst.pos[d] = src.pos[s];
      if (src.yc && dst.yc) dst.yc[d] = src.yc[s];
      if (src.strand && dst.strand) dst.strand[d] = src.strand[s];
      if (src.end && dst.end) dst.end[d] = src.end[s];
      if (src.yx && dst.yx) dst.yx[d] = src.yx[s];
    }
    if (k < (int64_t)words) dst.cigar[w + k] = src.cigar[c0 + k];
  }
}

// n rows of a column set to (send) or from a peer, one ncclSend / ncclRecv per column the set has; inside the caller's group
static int nccl_rows(tb_ctx* ctx, const TcCols& c, int64_t n, bool send, int peer, cudaStream_t st) {
  ncclComm_t comm = (ncclComm_t)ctx->comm;
  for (int i = 0; i < c.n; ++i) {
    if (!c.p[i]) continue;
    if (send) TB_NCCL(g_nccl.Send(c.p[i], (size_t)n * c.size[i], ncclUint8, peer, comm, st));
    else TB_NCCL(g_nccl.Recv(c.p[i], (size_t)n * c.size[i], ncclUint8, peer, comm, st));
  }
  return 0;
}

// n records to or from a peer: the row columns, the n + 1 offsets at c.cig_off, then `words` CIGAR words at c.cigar
static int nccl_records(tb_ctx* ctx, const TcRecords& c, int64_t n, int64_t words, bool send, int peer, cudaStream_t st) {
  if (nccl_rows(ctx, tc_cols(c), n, send, peer, st)) return 1;
  ncclComm_t comm = (ncclComm_t)ctx->comm;
  if (send) {
    TB_NCCL(g_nccl.Send(c.cig_off, (size_t)(n + 1) * 4, ncclUint8, peer, comm, st));
    TB_NCCL(g_nccl.Send(c.cigar, (size_t)words * 4, ncclUint8, peer, comm, st));
  } else {
    TB_NCCL(g_nccl.Recv(c.cig_off, (size_t)(n + 1) * 4, ncclUint8, peer, comm, st));
    TB_NCCL(g_nccl.Recv(c.cigar, (size_t)words * 4, ncclUint8, peer, comm, st));
  }
  return 0;
}

// ---- ordered gather overlapped with the windows (tc_shard_coverage_gather) ------------------------------------------------
// Rank 0's output arrays are cut into `world` regions of equal capacity; the rows of rank r arrive in region r in the order
// they are produced. After every window a rank takes part in one ROUND on a second stream: ncclAllGather of {new runs, new
// junction rows, done} (the only host wait of the round: the previous round's transfers have long finished), then one
// grouped ncclSend / ncclRecv of the new rows, which travels while the next window computes. Ranks that run out of windows
// keep answering rounds with zero rows until every rank is done.
struct GatherState {
  tc_runs_out* all_runs = nullptr; tc_juncs_out* all_juncs = nullptr;   // rank 0 only
  int64_t cap_r = 0, cap_j = 0;            // region capacity per rank
  int64_t sent_r = 0, sent_j = 0;          // rows of this rank already handed over
  std::vector<int64_t> got_r, got_j;       // rows per rank so far (every rank tracks them: they come with the allgather)
  bool all_done = false;
  int rounds = 0;
  int64_t bytes = 0;
};

// One ordered transfer of rows to rank 0, cr[r] / cj[r] from rank r (this rank's start at gs.sent_*). Rank 0 places them
// by layout: `regions` puts rank r's at r * cap + got[r] (tc_shard_coverage_gather), otherwise they follow each other in rank
// order (tc_shard_gather). Rank 0 copies its own rows (unless they are already in place) and receives the others'; every
// other rank sends. Adds the bytes that crossed NCCL to gs.bytes and the rows to gs.got_* / gs.sent_*.
static int gather_rows(tb_ctx* ctx, GatherState& gs, const tc_runs_out* runs, const tc_juncs_out* juncs, const std::vector<int64_t>& cr,
                       const std::vector<int64_t>& cj, bool regions, cudaStream_t st) {
  const int W = ctx->comm ? ctx->world : 1, R = ctx->comm ? ctx->rank : 0;
  std::vector<int64_t> br(W), bj(W);   // first row of rank r on rank 0
  for (int r = 0; r < W; ++r) {
    br[r] = regions ? r * gs.cap_r + gs.got_r[r] : (r ? br[r - 1] + cr[r - 1] : 0);
    bj[r] = regions ? r * gs.cap_j + gs.got_j[r] : (r ? bj[r - 1] + cj[r - 1] : 0);
  }
  if (R == 0) {
    if (gs.all_runs && runs) TB_CUDA(tc_copy_rows(tc_at(*gs.all_runs, br[0]), tc_at(*runs, gs.sent_r), cr[0], cudaMemcpyDeviceToDevice, st));
    if (gs.all_juncs && juncs) TB_CUDA(tc_copy_rows(tc_at(*gs.all_juncs, bj[0]), tc_at(*juncs, gs.sent_j), cj[0], cudaMemcpyDeviceToDevice, st));
  }
  if (W > 1) {
    TB_NCCL(g_nccl.GroupStart());
    for (int r = 1; r < W; ++r) {
      if (R != 0 && r != R) continue;   // rank 0 receives from every rank, the others send their own rows
      const tc_runs_out* rs = R ? runs : gs.all_runs;
      const tc_juncs_out* js = R ? juncs : gs.all_juncs;
      const int64_t ro = R ? gs.sent_r : br[r], jo = R ? gs.sent_j : bj[r];
      if (rs && cr[r] > 0 && nccl_rows(ctx, tc_cols(tc_at(*rs, ro)), cr[r], R != 0, R ? 0 : r, st)) return 1;
      if (js && cj[r] > 0 && nccl_rows(ctx, tc_cols(tc_at(*js, jo)), cj[r], R != 0, R ? 0 : r, st)) return 1;
      gs.bytes += cr[r] * 20 + cj[r] * 21;
    }
    TB_NCCL(g_nccl.GroupEnd());
  }
  for (int r = 0; r < W; ++r) { gs.got_r[r] += cr[r]; gs.got_j[r] += cj[r]; }
  gs.sent_r += cr[R]; gs.sent_j += cj[R];
  return 0;
}

static int gather_round(tb_ctx* ctx, GatherState& gs, const tc_runs_out* runs, const tc_juncs_out* juncs, bool done) {
  const int W = ctx->comm ? ctx->world : 1, R = ctx->comm ? ctx->rank : 0;
  cudaStream_t gst = ctx->gather_stream;
  const int64_t new_r = (runs ? runs->n_runs : 0) - gs.sent_r, new_j = (juncs ? juncs->n_juncs : 0) - gs.sent_j;
  std::vector<unsigned long long> h(4 * (size_t)W, 0ULL);
  if (W > 1) {
    ncclComm_t comm = (ncclComm_t)ctx->comm;
    DevBuf* SB = ctx->shard_buf;
    TB_CUDA(SB[SB_GROUND].ensure(sizeof(unsigned long long) * 4 * (size_t)(W + 1)));
    TB_CUDA(ctx->pinned[1].ensure(sizeof(unsigned long long) * 8 * (size_t)(W + 1)));
    unsigned long long* d_mine = SB[SB_GROUND].as<unsigned long long>();
    unsigned long long* d_all = d_mine + 4;
    unsigned long long* h_all = ctx->pinned[1].as<unsigned long long>();
    h_all[0] = (unsigned long long)new_r; h_all[1] = (unsigned long long)new_j; h_all[2] = done ? 1ULL : 0ULL; h_all[3] = 0;
    TB_CUDA(cudaMemcpyAsync(d_mine, h_all, sizeof(unsigned long long) * 4, cudaMemcpyHostToDevice, gst));
    TB_NCCL(g_nccl.AllGather(d_mine, d_all, 4, ncclUint64, comm, gst));
    TB_CUDA(cudaMemcpyAsync(h_all + 4, d_all, sizeof(unsigned long long) * 4 * W, cudaMemcpyDeviceToHost, gst));
    TB_CUDA(cudaStreamSynchronize(gst));
    for (int i = 0; i < 4 * W; ++i) h[i] = h_all[4 + i];
  } else {
    h[0] = (unsigned long long)new_r; h[1] = (unsigned long long)new_j; h[2] = done ? 1ULL : 0ULL;
  }
  bool all = true;
  for (int r = 0; r < W; ++r) {
    if (!h[4 * r + 2]) all = false;
    if (gs.got_r[r] + (int64_t)h[4 * r] > gs.cap_r || gs.got_j[r] + (int64_t)h[4 * r + 1] > gs.cap_j) {
      ctx->set_error("tc_shard_coverage_gather: region of rank %d too small (%lld runs / %lld junction rows per rank)", r, (long long)gs.cap_r, (long long)gs.cap_j);
      return 1;
    }
  }
  std::vector<int64_t> cr(W), cj(W);
  for (int r = 0; r < W; ++r) { cr[r] = (int64_t)h[4 * r]; cj[r] = (int64_t)h[4 * r + 1]; }
  if (gather_rows(ctx, gs, runs, juncs, cr, cj, true, gst)) return 1;
  gs.all_done = all;
  gs.rounds++;
  return 0;
}

}  // namespace

// One stream slice in windows cut at bundle heads. `skip` leading records are not processed (they belong to a bundle that
// another rank owns). next = {tid, pos} of the record that follows the slice in the stream (host values), or NULL.
// Outputs are appended to runs / juncs (n_runs / n_juncs on entry = rows already there). *consumed = records processed.
// yx (tc_coverage_bam): the YX column of `in`; runs then receives the sample heat-map rows (tc_sample_window) and juncs is NULL.
int tc_stream_impl(tb_ctx* ctx, const tc_soa_in* in, int64_t skip, int64_t window, const int32_t* next, tc_runs_out* runs, tc_juncs_out* juncs, int64_t* consumed,
                   const std::function<int()>* after_window = nullptr, const int32_t* yx = nullptr) {
  TB_CUDA(cudaSetDevice(ctx->device));
  const int64_t n = in->n;
  if (window < 1024) window = 1024;
  if (window >= (1LL << 31)) window = (1LL << 31) - 1;
  int64_t w0 = skip;
  float ms_acc[3] = {0.f, 0.f, 0.f};
  while (w0 < n) {
    int64_t wlen = std::min(window, n - w0);
    for (;;) {
      const int64_t w1 = w0 + wlen;
      CovExt ext; memset(&ext, 0, sizeof(ext));
      uint32_t c01[2] = {0, 0};
      int32_t nx[2] = {0, 0};
      if (in->on_device) {
        TB_CUDA(cudaMemcpyAsync(&c01[0], in->cig_off + w0, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        TB_CUDA(cudaMemcpyAsync(&c01[1], in->cig_off + w1, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (w1 < n) {
          TB_CUDA(cudaMemcpyAsync(&nx[0], in->tid + w1, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
          TB_CUDA(cudaMemcpyAsync(&nx[1], in->pos + w1, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        }
        TB_CUDA(cudaStreamSynchronize(ctx->stream));
      } else {
        c01[0] = in->cig_off[w0]; c01[1] = in->cig_off[w1];
        if (w1 < n) { nx[0] = in->tid[w1]; nx[1] = in->pos[w1]; }
      }
      if (w1 < n) { ext.has_next = 1; ext.next_tid = nx[0]; ext.next_pos = nx[1]; }
      else if (next) { ext.has_next = 1; ext.next_tid = next[0]; ext.next_pos = next[1]; }
      const TcRecords wc = tc_at(tc_records(*in, yx), w0);
      const tc_soa_in sub = tc_window(wc, wlen, (int64_t)(c01[1] - c01[0]), in->on_device);
      tc_runs_out r; tc_juncs_out j;   // the rows after those already in runs / juncs
      if (runs) { r = tc_at(*runs, runs->n_runs); r.capacity -= runs->n_runs; r.n_runs = 0; }
      if (juncs) { j = tc_at(*juncs, juncs->n_juncs); j.capacity -= juncs->n_juncs; j.n_juncs = 0; }
      const int rc = tc_coverage_impl(ctx, &sub, runs ? &r : nullptr, juncs ? &j : nullptr, wc.yx, &ext);
      if (rc == 3) {   // one bundle spans the window
        if (w1 >= n) { *consumed = w0; goto done; }   // ... and the slice: the caller joins it with what follows
        wlen = std::min(wlen * 2, n - w0);
        continue;
      }
      if (rc) return rc;
      if (runs) runs->n_runs += r.n_runs;
      if (juncs) juncs->n_juncs += j.n_juncs;
      ms_acc[0] += ctx->last_ms[6]; ms_acc[1] += ctx->last_ms[1]; ms_acc[2] += ctx->last_ms[7];
      ctx->stream_windows++;
      if (after_window) { const int rc2 = (*after_window)(); if (rc2) return rc2; }
      if (ext.consumed < wlen && w1 >= n) { *consumed = w0 + ext.consumed; goto done; }   // the open tail belongs with the records behind the slice
      w0 += ext.consumed;
      break;
    }
  }
  *consumed = n;
done:
  ctx->last_ms[6] = ms_acc[0]; ctx->last_ms[1] = ms_acc[1]; ctx->last_ms[7] = ms_acc[2];   // sums over the windows of this call
  return 0;
}

void tc_copy_records(tb_ctx* ctx, cudaStream_t st, const TcRecords& src, int64_t from, int64_t m, const TcRecords& dst, int64_t r, uint32_t w,
                     uint32_t words) {
  const int64_t work = std::max<int64_t>(m + 1, words);
  tc_copy_records_kernel<<<(unsigned)std::min<int64_t>((work + 255) / 256, 4096), 256, 0, st>>>(src, from, m, dst, r, w, words);
  ctx->launches++;
}

extern "C" {

int tb_comm_unique_id(void* id128) {
  if (!g_nccl.load()) { g_tb_global_error = "tb_comm_unique_id: " + g_nccl.err; return 1; }
  ncclUniqueId id;
  const ncclResult_t r = g_nccl.GetUniqueId(&id);
  if (r != ncclSuccess) { g_tb_global_error = std::string("tb_comm_unique_id: ") + g_nccl.GetErrorString(r); return 1; }
  memcpy(id128, &id, sizeof(id));
  return 0;
}

int tb_comm_init(tb_ctx* ctx, int rank, int world, const void* id128) {
  if (!ctx) return 1;
  if (!g_nccl.load()) { ctx->set_error("tb_comm_init: %s", g_nccl.err.c_str()); return 1; }
  if (world < 1 || rank < 0 || rank >= world) { ctx->set_error("tb_comm_init: rank %d of %d", rank, world); return 1; }
  TB_CUDA(cudaSetDevice(ctx->device));
  ncclUniqueId id; memcpy(&id, id128, sizeof(id));
  ncclComm_t comm = nullptr;
  TB_NCCL(g_nccl.CommInitRank(&comm, world, id, rank));
  ctx->comm = (void*)comm; ctx->rank = rank; ctx->world = world;
  return 0;
}

int tb_comm_destroy(tb_ctx* ctx) {
  if (!ctx || !ctx->comm) return 0;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  g_nccl.CommDestroy((ncclComm_t)ctx->comm);
  ctx->comm = nullptr; ctx->world = 1; ctx->rank = 0;
  return 0;
}

int tb_comm_rank(tb_ctx* ctx) { return ctx ? ctx->rank : -1; }
int tb_comm_world(tb_ctx* ctx) { return ctx ? ctx->world : -1; }

int tc_coverage_stream(tb_ctx* ctx, const tc_soa_in* in, int64_t window, const int32_t* next_tid_pos, tc_runs_out* runs, tc_juncs_out* juncs, int64_t* consumed) {
  if (!ctx) return 1;
  if (!in || (!runs && !juncs) || !consumed) { ctx->set_error("tc_coverage_stream: in, consumed and one of runs / juncs are required"); return 1; }
  ctx->err.clear();
  if (runs) runs->n_runs = 0;
  if (juncs) juncs->n_juncs = 0;
  ctx->stream_windows = 0;
  return tc_stream_impl(ctx, in, 0, window, next_tid_pos, runs, juncs, consumed);
}

static int shard_coverage_impl(tb_ctx* ctx, const tc_soa_in* segs, int n_segs, int64_t window, tc_runs_out* runs, tc_juncs_out* juncs, GatherState* gs) {
  if (!ctx) return 1;
  if (!segs || n_segs < 1 || (!runs && !juncs)) { ctx->set_error("tc_shard_coverage: segments and one of runs / juncs are required"); return 1; }
  ctx->err.clear();
  TB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // ONE host-resident segment (the command-line tool's case) is copied to the device first; several segments must be resident
  tc_soa_in dseg;
  if (!segs[0].on_device) {
    if (n_segs != 1) { ctx->set_error("tc_shard_coverage: host arrays are accepted as ONE segment; several segments must be device resident"); return 1; }
    tc_soa_in h = segs[0];
    dseg = h; dseg.on_device = 1;
    if (h.n > 0) {   // staged in in_stage[8..16): tc_coverage_impl stages its windows in [0, 8)
      h.n_cig = (int64_t)(h.cig_off[h.n] - h.cig_off[0]);
      if (tc_stage_window(ctx, ctx->in_stage + 8, h, nullptr, &dseg, nullptr)) return 1;
      TB_CUDA(cudaStreamSynchronize(st));
    }
    segs = &dseg;
  }
  for (int s = 0; s < n_segs; ++s) if (!segs[s].on_device) { ctx->set_error("tc_shard_coverage: segments must be all host (one) or all device resident"); return 1; }
  if (runs) runs->n_runs = 0;
  if (juncs) juncs->n_juncs = 0;
  ctx->stream_windows = 0;
  memset(ctx->shard_stat, 0, sizeof(ctx->shard_stat));
  const int W = ctx->comm ? ctx->world : 1, R = ctx->comm ? ctx->rank : 0;
  const tc_soa_in& first = segs[0];
  const tc_soa_in& last = segs[n_segs - 1];
  int64_t n_local = 0;
  for (int s = 0; s < n_segs; ++s) n_local += segs[s].n;
  int64_t lead = 0, tail_n = 0, tail_words = 0;
  TcRecords tail{};   // the leads received from the ranks on the right, in rank order
  int32_t tail_next[2] = {0, 0};
  DevBuf* SB = ctx->shard_buf;
  cudaEvent_t e0 = ctx->ev[12], e1 = ctx->ev[13];
  if (ctx->profiling) TB_CUDA(cudaEventRecord(e0, st));
  if (W > 1) {
    ncclComm_t comm = (ncclComm_t)ctx->comm;
    // ---- 1. open-bundle state of every rank: allgather of {max key of the last segment, first record key, records} ----
    TB_CUDA(SB[SB_GATHER].ensure(sizeof(unsigned long long) * 8 * (size_t)(W + 1)));
    TB_CUDA(ctx->pinned[1].ensure(sizeof(unsigned long long) * 8 * (size_t)(W + 1)));
    unsigned long long* d_mine = SB[SB_GATHER].as<unsigned long long>();
    unsigned long long* d_all = d_mine + 8;
    unsigned long long* h_all = ctx->pinned[1].as<unsigned long long>();
    TB_CUDA(cudaMemsetAsync(d_mine, 0, sizeof(unsigned long long) * 8, st));
    if (last.n > 0) {
      long long* d_start = (long long*)(d_mine + 5);
      shard_last_tid_kernel<<<1, 1, 0, st>>>(last.n, last.tid, d_start);
      shard_maxkey_kernel<<<148u * 8u, 256, 0, st>>>(last.n, d_start, last.tid, last.pos, last.cig_off, last.cigar, d_mine);
      ctx->launches += 2;
    }
    {
      unsigned long long h_mine[3] = {0, 0, (unsigned long long)n_local};
      if (first.n > 0) {
        int32_t tp[2];
        TB_CUDA(cudaMemcpyAsync(&tp[0], first.tid, 4, cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaMemcpyAsync(&tp[1], first.pos, 4, cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaStreamSynchronize(st));
        h_mine[1] = ((unsigned long long)(uint32_t)tp[0] << 32) | (uint32_t)tp[1];
      }
      TB_CUDA(cudaMemcpyAsync(d_mine + 1, &h_mine[1], sizeof(unsigned long long) * 2, cudaMemcpyHostToDevice, st));
    }
    TB_NCCL(g_nccl.AllGather(d_mine, d_all, 4, ncclUint64, comm, st));
    TB_CUDA(cudaMemcpyAsync(h_all, d_all, sizeof(unsigned long long) * 4 * W, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    unsigned long long ein = 0;
    for (int r = 0; r < R; ++r) if (h_all[4 * r + 2] > 0 && h_all[4 * r] > ein) ein = h_all[4 * r];
    std::vector<unsigned long long> firstkey(W), nrec(W);
    for (int r = 0; r < W; ++r) { firstkey[r] = h_all[4 * r + 1]; nrec[r] = h_all[4 * r + 2]; }
    // ---- 2. my lead; allgather of {lead, lead CIGAR words, has a head, records of the first segment} ----
    uint32_t lead_c[2] = {0, 0};
    if (first.n > 0 && ein != 0) {
      TB_CUDA(SB[SB_SEND].ensure(sizeof(unsigned long long) * (LEAD_BLOCKS + 8)));
      unsigned long long* d_bmax = SB[SB_SEND].as<unsigned long long>();
      unsigned long long* d_state = d_mine + 6;   // [carry, first head]
      unsigned long long h_state[2] = {ein, ~0ULL};
      TB_CUDA(cudaMemcpyAsync(d_state, h_state, sizeof(h_state), cudaMemcpyHostToDevice, st));
      lead = first.n;   // no head at all: the whole slice continues a bundle opened further left
      for (int64_t base = 0; base < first.n; base += (int64_t)LEAD_BLOCKS * 1024) {
        const int nb = (int)std::min<int64_t>(LEAD_BLOCKS, (first.n - base + 1023) / 1024);
        shard_lead_max_kernel<<<nb, 1024, 0, st>>>(base, first.n, first.tid, first.pos, first.cig_off, first.cigar, d_bmax);
        shard_lead_scan_kernel<<<1, 1024, 0, st>>>(d_bmax, nb, d_state);
        shard_lead_head_kernel<<<nb, 1024, 0, st>>>(base, first.n, first.tid, first.pos, first.cig_off, first.cigar, d_bmax, d_state);
        ctx->launches += 3;
        TB_CUDA(cudaMemcpyAsync(h_state, d_state, sizeof(h_state), cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaStreamSynchronize(st));
        if (h_state[1] != ~0ULL) { lead = (int64_t)h_state[1]; break; }
      }
      if (lead == first.n && n_segs > 1) { ctx->set_error("tc_shard_coverage: the first segment of rank %d lies inside one bundle; segments of a rank must end at reference-id boundaries", R); return 1; }
      if (lead > 0) {
        TB_CUDA(cudaMemcpyAsync(&lead_c[0], first.cig_off, 4, cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaMemcpyAsync(&lead_c[1], first.cig_off + lead, 4, cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaStreamSynchronize(st));
      }
    }
    {
      unsigned long long h2[4] = {(unsigned long long)lead, (unsigned long long)(lead_c[1] - lead_c[0]), (unsigned long long)(n_local > 0 && lead < n_local ? 1 : 0), (unsigned long long)first.n};
      TB_CUDA(cudaMemcpyAsync(d_mine, h2, sizeof(h2), cudaMemcpyHostToDevice, st));
    }
    TB_NCCL(g_nccl.AllGather(d_mine, d_all, 4, ncclUint64, comm, st));
    TB_CUDA(cudaMemcpyAsync(h_all, d_all, sizeof(unsigned long long) * 4 * W, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    std::vector<long long> leads(W), lwords(W), hashead(W);
    for (int r = 0; r < W; ++r) { leads[r] = (long long)h_all[4 * r]; lwords[r] = (long long)h_all[4 * r + 1]; hashead[r] = (long long)h_all[4 * r + 2]; }
    // ---- 3. who sends to whom: the lead of rank r goes to the nearest rank on its left that holds a bundle head ----
    int owner = -1;
    if (lead > 0) { for (int r = R - 1; r >= 0; --r) if (hashead[r]) { owner = r; break; } }
    if (lead > 0 && owner < 0) { ctx->set_error("tc_shard_coverage: rank %d has a lead but no rank on its left holds a bundle head", R); return 1; }
    std::vector<int> from;
    if (hashead[R]) {
      for (int r = R + 1; r < W; ++r) {
        if (nrec[r] == 0) continue;
        if (leads[r] > 0) from.push_back(r);
        if (hashead[r]) break;
      }
    }
    for (int r : from) { tail_n += leads[r]; tail_words += lwords[r]; }
    if (!from.empty()) { const unsigned long long fk = firstkey[from[0]]; tail_next[0] = (int32_t)(fk >> 32); tail_next[1] = (int32_t)(uint32_t)fk; }
    if (tail_words >= (1LL << 32) || tail_n >= (1LL << 31)) { ctx->set_error("tc_shard_coverage: %lld lead records do not fit one window", (long long)tail_n); return 1; }
    if (tail_n > 0) {
      TB_CUDA(tc_alloc_records(SB + SB_TAIL, tail_n, tail_words + 4, false, &tail));
      TB_CUDA(SB[SB_SEND].ensure(sizeof(uint32_t) * (tail_n + from.size() + 1)));
    }
    // ---- 4. the halo exchange proper: one grouped send / receive of the lead records' columns. No `end` column: the
    // seam window that takes the leads is processed from the CIGARs ----
    TB_NCCL(g_nccl.GroupStart());
    if (lead > 0) {
      TcRecords lr = tc_records(first);
      lr.end = nullptr;
      lr.cigar += lead_c[0];
      if (nccl_records(ctx, lr, lead, lead_c[1] - lead_c[0], true, owner, st)) return 1;
      ctx->shard_stat[1] = lead; ctx->shard_stat[3] = (int64_t)lead * 17 + 4 + (int64_t)(lead_c[1] - lead_c[0]) * 4;
    }
    {
      int64_t ro = 0, wo = 0; size_t piece = 0;
      for (int r : from) {
        // the leads + 1 offsets of piece p land in a scratch area at [ro + p, ...) and are rebased into the tail below
        TcRecords dst = tc_at(tail, ro);
        dst.cig_off = SB[SB_SEND].as<uint32_t>() + ro + piece;
        dst.cigar = tail.cigar + wo;
        if (nccl_records(ctx, dst, leads[r], lwords[r], false, r, st)) return 1;
        ro += leads[r]; wo += lwords[r]; ++piece;
      }
    }
    TB_NCCL(g_nccl.GroupEnd());
    ctx->shard_stat[0] = tail_n; ctx->shard_stat[2] = (int64_t)from.size();
    // ---- 5. received offsets -> offsets into the tail arena, piece by piece ----
    int64_t ro = 0, wo = 0; size_t piece = 0;
    for (int r : from) {
      TcRecords src{};
      src.cig_off = SB[SB_SEND].as<uint32_t>() + ro + piece;
      tc_copy_records(ctx, st, src, 0, leads[r], tail, ro, (uint32_t)wo, 0);
      ro += leads[r]; wo += lwords[r]; ++piece;
    }
  }
  if (ctx->profiling) TB_CUDA(cudaEventRecord(e1, st));
  // ---- 6. this rank's whole bundles, segment by segment ----
  int64_t consumed_last = last.n;
  float ms_sum[3] = {0.f, 0.f, 0.f};   // K6 / K7 / K8 device time over every window of the call
  std::function<int()> round_cb = [&]() -> int { return gather_round(ctx, *gs, runs, juncs, false); };
  const std::function<int()>* cb = gs ? &round_cb : nullptr;
  for (int s = 0; s < n_segs; ++s) {
    const bool is_last = s == n_segs - 1;
    int64_t consumed = 0;
    const int64_t skip = s == 0 ? lead : 0;
    if (skip >= segs[s].n) { if (is_last) consumed_last = segs[s].n; continue; }
    const int rc = tc_stream_impl(ctx, &segs[s], skip, window, (is_last && tail_n > 0) ? tail_next : nullptr, runs, juncs, &consumed, cb);
    if (rc) return rc;
    ms_sum[0] += ctx->last_ms[6]; ms_sum[1] += ctx->last_ms[1]; ms_sum[2] += ctx->last_ms[7];
    if (is_last) consumed_last = consumed;
    else if (consumed < segs[s].n) { ctx->set_error("tc_shard_coverage: segment %d of rank %d ends inside a bundle; segments of a rank must end at reference-id boundaries", s, R); return 1; }
  }
  // ---- 7. the seam: what the last segment left open + the leads received from the right ----
  const int64_t open_n = (lead >= last.n && n_segs == 1) ? 0 : last.n - consumed_last;
  if (open_n + tail_n > 0 && !(open_n == 0 && tail_n == 0)) {
    if (open_n > 0 && tail_n == 0) {   // cannot happen: the stream leaves a tail only when told that something follows
      ctx->set_error("tc_shard_coverage: open tail without a continuation (internal error)"); return 1;
    }
    const int64_t sn = open_n + tail_n;
    uint32_t oc[2] = {0, 0};
    if (open_n > 0) {
      TB_CUDA(cudaMemcpyAsync(&oc[0], last.cig_off + consumed_last, 4, cudaMemcpyDeviceToHost, st));
      TB_CUDA(cudaMemcpyAsync(&oc[1], last.cig_off + last.n, 4, cudaMemcpyDeviceToHost, st));
      TB_CUDA(cudaStreamSynchronize(st));
    }
    const int64_t ow = (int64_t)(oc[1] - oc[0]), sw = ow + tail_words;
    TcRecords sc;   // like the tail, without `end`
    TB_CUDA(tc_alloc_records(SB + SB_SEAM, sn, sw + 4, false, &sc));
    if (open_n > 0) tc_copy_records(ctx, st, tc_records(last), consumed_last, open_n, sc, 0, 0, (uint32_t)ow);
    tc_copy_records(ctx, st, tail, 0, tail_n, sc, open_n, (uint32_t)ow, (uint32_t)tail_words);
    const tc_soa_in seam = tc_window(sc, sn, sw);
    int64_t consumed = 0;
    const int rc = tc_stream_impl(ctx, &seam, 0, std::max<int64_t>(window, sn), nullptr, runs, juncs, &consumed, cb);
    if (rc) return rc;
    ms_sum[0] += ctx->last_ms[6]; ms_sum[1] += ctx->last_ms[1]; ms_sum[2] += ctx->last_ms[7];
    ctx->shard_stat[4] = sn;
  }
  ctx->last_ms[6] = ms_sum[0]; ctx->last_ms[1] = ms_sum[1]; ctx->last_ms[7] = ms_sum[2];
  if (gs) {   // hand over what is left and answer rounds until every rank is done
    for (int guard = 0; !gs->all_done; ++guard) {
      if (guard > (1 << 20)) { ctx->set_error("tc_shard_coverage_gather: the ranks did not agree on the end of the gather (internal error)"); return 1; }
      if (gather_round(ctx, *gs, runs, juncs, true)) return 1;
    }
    TB_CUDA(cudaStreamSynchronize(ctx->gather_stream));
  }
  if (ctx->profiling) {
    TB_CUDA(cudaStreamSynchronize(st));
    float ms = 0;
    if (cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) ctx->last_ms[9] = ms;
    (void)cudaGetLastError();
  }
  return 0;
}

int tc_shard_coverage(tb_ctx* ctx, const tc_soa_in* segs, int n_segs, int64_t window, tc_runs_out* runs, tc_juncs_out* juncs) {
  return shard_coverage_impl(ctx, segs, n_segs, window, runs, juncs, nullptr);
}

// tc_shard_coverage with the ordered gather folded into the window loop (see GatherState). region (host, [4 * world], every
// rank): for rank r the offset and count of its runs, then of its junction rows, inside all_runs / all_juncs on rank 0; the
// ordered result is region 0, region 1, ... The junction numbering base of rank r is the sum of the junction counts before it.
int tc_shard_coverage_gather(tb_ctx* ctx, const tc_soa_in* segs, int n_segs, int64_t window, tc_runs_out* runs, tc_juncs_out* juncs,
                             tc_runs_out* all_runs, tc_juncs_out* all_juncs, int64_t* region) {
  if (!ctx) return 1;
  if (!runs || !juncs || !region) { ctx->set_error("tc_shard_coverage_gather: runs, juncs and region are required"); return 1; }
  const int W = ctx->comm ? ctx->world : 1, R = ctx->comm ? ctx->rank : 0;
  if (R == 0 && (!all_runs || !all_juncs)) { ctx->set_error("tc_shard_coverage_gather: rank 0 needs all_runs and all_juncs"); return 1; }
  TB_CUDA(cudaSetDevice(ctx->device));
  if (!ctx->gather_stream) TB_CUDA(cudaStreamCreateWithFlags(&ctx->gather_stream, cudaStreamNonBlocking));
  GatherState gs;
  gs.all_runs = R == 0 ? all_runs : nullptr; gs.all_juncs = R == 0 ? all_juncs : nullptr;
  // every rank must use the same region sizes: rank 0's capacities travel with the first allgather of the halo exchange?
  // simpler: the caller passes the SAME capacities on every rank (all_* structs with NULL arrays elsewhere)
  if (!all_runs || !all_juncs) { ctx->set_error("tc_shard_coverage_gather: every rank passes all_runs / all_juncs (capacities; arrays may be NULL except on rank 0)"); return 1; }
  gs.cap_r = all_runs->capacity / W; gs.cap_j = all_juncs->capacity / W;
  gs.got_r.assign(W, 0); gs.got_j.assign(W, 0);
  const int rc = shard_coverage_impl(ctx, segs, n_segs, window, runs, juncs, &gs);
  if (rc) return rc;
  int64_t tr = 0, tj = 0;
  for (int r = 0; r < W; ++r) {
    region[4 * r] = r * gs.cap_r; region[4 * r + 1] = gs.got_r[r]; region[4 * r + 2] = r * gs.cap_j; region[4 * r + 3] = gs.got_j[r];
    tr += gs.got_r[r]; tj += gs.got_j[r];
  }
  if (R == 0) { all_runs->n_runs = tr; all_juncs->n_juncs = tj; }
  ctx->shard_stat[5] = gs.bytes; ctx->shard_stat[6] = gs.rounds;
  return 0;
}

int64_t tc_shard_stat(tb_ctx* ctx, int which) { return (ctx && which >= 0 && which < 8) ? ctx->shard_stat[which] : -1; }

// ordered gather on rank 0. all_runs / all_juncs (rank 0 only; device arrays) receive the rows of rank 0, 1, ... in that
// order; junc_base[r] (host, [world+1], every rank) = junctions of the ranks before r.
int tc_shard_gather(tb_ctx* ctx, const tc_runs_out* runs, const tc_juncs_out* juncs, tc_runs_out* all_runs, tc_juncs_out* all_juncs, int64_t* junc_base) {
  if (!ctx) return 1;
  ctx->err.clear();
  TB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int W = ctx->comm ? ctx->world : 1, R = ctx->comm ? ctx->rank : 0;
  const int64_t nr = runs ? runs->n_runs : 0, nj = juncs ? juncs->n_juncs : 0;
  std::vector<int64_t> cr(W, 0), cj(W, 0);
  cr[R] = nr; cj[R] = nj;
  ncclComm_t comm = (ncclComm_t)ctx->comm;
  DevBuf* SB = ctx->shard_buf;
  if (W > 1) {
    TB_CUDA(SB[SB_GATHER].ensure(sizeof(unsigned long long) * 8 * (size_t)(W + 1)));
    TB_CUDA(ctx->pinned[1].ensure(sizeof(unsigned long long) * 8 * (size_t)(W + 1)));
    unsigned long long* d_mine = SB[SB_GATHER].as<unsigned long long>();
    unsigned long long* d_all = d_mine + 8;
    unsigned long long* h_all = ctx->pinned[1].as<unsigned long long>();
    unsigned long long h2[2] = {(unsigned long long)nr, (unsigned long long)nj};
    TB_CUDA(cudaMemcpyAsync(d_mine, h2, sizeof(h2), cudaMemcpyHostToDevice, st));
    TB_NCCL(g_nccl.AllGather(d_mine, d_all, 2, ncclUint64, comm, st));
    TB_CUDA(cudaMemcpyAsync(h_all, d_all, sizeof(unsigned long long) * 2 * W, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    for (int r = 0; r < W; ++r) { cr[r] = (int64_t)h_all[2 * r]; cj[r] = (int64_t)h_all[2 * r + 1]; }
  }
  if (junc_base) { junc_base[0] = 0; for (int r = 0; r < W; ++r) junc_base[r + 1] = junc_base[r] + cj[r]; }
  int64_t tr = 0, tj = 0;
  for (int r = 0; r < W; ++r) { tr += cr[r]; tj += cj[r]; }
  if (R == 0) {
    if (all_runs) { if (all_runs->capacity < tr) { ctx->set_error("tc_shard_gather: runs capacity %lld < %lld", (long long)all_runs->capacity, (long long)tr); return 1; } all_runs->n_runs = tr; }
    if (all_juncs) { if (all_juncs->capacity < tj) { ctx->set_error("tc_shard_gather: junction capacity %lld < %lld", (long long)all_juncs->capacity, (long long)tj); return 1; } all_juncs->n_juncs = tj; }
  }
  GatherState gs;
  gs.all_runs = all_runs; gs.all_juncs = all_juncs;
  gs.got_r.assign(W, 0); gs.got_j.assign(W, 0);
  if (gather_rows(ctx, gs, runs, juncs, cr, cj, false, st)) return 1;
  if (W > 1) ctx->shard_stat[5] = gs.bytes;   // bytes over NVLink in the gather
  TB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

}  // extern "C"
