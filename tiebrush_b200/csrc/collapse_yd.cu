// collapse_yd.cu — the YD tag: GSegList::processRead / mergeRead (src/tiebrush.cpp:151-250) driven by flushPData
// (src/tiebrush.cpp:512-524) over the collapsed groups in output order.
//
// The reference keeps, per (sample, strand list) — a "chain" — a linked list of merged exon segments; for every emitted
// group and every sample that contributed to it, processRead returns the distance d from the read start back to the
// start of the segment that reaches it, and YD = max of d over those samples (and over YD tags carried by
// TieBrush-made inputs). The list is a sequential state machine with binding quirks (touching segments are not merged;
// when the merge cursor runs off the list the current and all later exons are silently dropped, SURVEY §9.4).
//
// PARALLEL FORMULATION (default). Reading the list code closely gives two facts (checked against a literal model of the
// list on randomised chains, and through the oracle in tests/):
//   (1) which exons enter the list depends on ONE scalar per chain, the frontier E = largest end of any exon kept so
//       far: a read at x with E < x finds only dead nodes, empties the list and appends all its exons ("bulk"); otherwise
//       exon j >= 2 is kept iff its start <= max(E, ends of the read's earlier kept exons) — else the cursor runs off the
//       list and it and all later exons are dropped. E never decreases.
//   (2) the list is the interval union of the kept exons, and links left of x are final when the read at x arrives
//       (later reads start at >= x). With link[p] = "some kept exon contains p and p+1", d = the number of consecutive
//       set links ending at x-1 (0 if link[x-1] is clear). Reads sharing a start get the same d (the reference's
//       last_pos cache).
//   So: Y1 group descriptors + union bitmap U of all exon positions; Y2 rank(U) gives compact coordinates (runs of links
//   are preserved: a link at p implies p+1 is covered); Y3-Y5 chain member lists by a stable counting scatter over the
//   sample bitsets, cut into independent sub-chains where a member starts beyond every earlier end of its chain (the
//   count pass also keeps each chain's largest end per block of groups, a scan turns those into prefix maxima, and the
//   scatter runs the head test in registers as it writes the members; one stream compaction of the head bits);
//   Y6 the frontier recurrence per sub-chain (one scalar, lane-parallel; long sub-chains are walked by a whole warp with
//   prefetch) -> kept-exon count per member; Y7 kept exons OR their links into the chain's bitmap; Y8 prefix max of
//   "last clear link" over 512-bit blocks; Y9 one lookup per member, atomicMax into the group.
//
// SEQUENTIAL FALLBACK. The literal list (sorted arrays in shared memory, dead nodes dropped eagerly) per sub-chain:
// used when a representative has a degenerate exon (N directly followed by N, SURVEY §9.7), more than 255 exons, an
// exon reaching beyond the union bitmap, or when TB_YD_PATH=seq is set (tests run both).
#include <stdlib.h>
#include "collapse_internal.cuh"

namespace {

constexpr int YD_INLINE_EX = 3;   // exons kept in the descriptor; longer chains are decoded from the CIGAR
struct __align__(16) GDesc {      // 32 bytes; coordinates 1-based genomic (desc) or compact (cdesc)
  int32_t start;                  // start of the representative (== first exon start)
  uint32_t meta;                  // n_exons (low 16) | strand char << 16
  int32_t e0, s1, e1, s2, e2;     // first three exons: [start,e0] [s1,e1] [s2,e2]
  int32_t zend;                   // end of the last exon
};
enum { YS_FALLBACK = 8, YS_LC = 9 };   // status slots used by this file (CS_* occupy 0..6)
constexpr int64_t YD_U_SLACK = 1 << 22;  // union bitmap extends this far beyond the last start position

__device__ __forceinline__ void yd_set_bits32(uint32_t* bm, int64_t lo, int64_t hi) {  // set bits [lo,hi]
  for (int64_t w = lo >> 5; w <= (hi >> 5); ++w) {
    const int b0 = w == (lo >> 5) ? (int)(lo & 31) : 0, b1 = w == (hi >> 5) ? (int)(hi & 31) : 31;
    const uint32_t mask = (b1 == 31 ? 0xffffffffu : ((1u << (b1 + 1)) - 1u)) & ~((1u << b0) - 1u);
    if ((bm[w] & mask) != mask) atomicOr(&bm[w], mask);
  }
}
__device__ __forceinline__ void yd_set_bits64(unsigned long long* bm, int64_t lo, int64_t hi) {  // set bits [lo,hi]
  for (int64_t w = lo >> 6; w <= (hi >> 6); ++w) {
    const int b0 = w == (lo >> 6) ? (int)(lo & 63) : 0, b1 = w == (hi >> 6) ? (int)(hi & 63) : 63;
    const unsigned long long mask = (b1 == 63 ? ~0ULL : ((1ULL << (b1 + 1)) - 1ULL)) & ~((1ULL << b0) - 1ULL);
    if ((bm[w] & mask) != mask) atomicOr(&bm[w], mask);
  }
}

// Y1: descriptor per group (genomic coordinates), group end, strand; union bitmap of exon positions (bit = coordinate - ubase)
__global__ void __launch_bounds__(256) yd_desc_kernel(ColIn in, const uint32_t* __restrict__ rep, int64_t G, GDesc* __restrict__ desc,
                                                      uint32_t* __restrict__ gend, uint32_t* __restrict__ gstart, uint8_t* __restrict__ gstrand,
                                                      uint32_t* __restrict__ U, int64_t ubits, long long* __restrict__ status) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const uint32_t r = rep[g];
  const int pos = in.pos[r];
  const int ubase = in.pos_lo + 1;
  ExonIter it; it.init(in.cigar, in.cig_off[r], in.cig_off[r + 1], pos);
  GDesc d; d.start = pos + 1; d.e0 = d.s1 = d.e1 = d.s2 = d.e2 = 0;
  int s, e, ne = 0; bool bad = false;
  while (it.next(s, e)) {
    if (ne == 0) d.e0 = e;
    else if (ne == 1) { d.s1 = s; d.e1 = e; }
    else if (ne == 2) { d.s2 = s; d.e2 = e; }
    if (e < s) bad = true;                                   // degenerate exon (N directly after N)
    else if (U) { if ((int64_t)e - ubase >= ubits) bad = true; else yd_set_bits32(U, (int64_t)s - ubase, (int64_t)e - ubase); }
    ++ne;
  }
  if (ne > 255) bad = true;
  if (bad) status[YS_FALLBACK] = 1;
  const uint8_t sc = in.strand[r];
  d.meta = (uint32_t)(ne > 0xffff ? 0xffff : ne) | ((uint32_t)sc << 16);
  d.zend = pos + it.l;
  desc[g] = d;
  gend[g] = (uint32_t)(pos + it.l);
  gstart[g] = (uint32_t)(pos + 1);
  gstrand[g] = sc;
}

// Y2: compact coordinates. rank(p) = number of covered positions before p.
struct UPopIn { const uint32_t* U; __device__ uint32_t operator()(int64_t w) const { return (uint32_t)__popc(U[w]); } };
struct UPopOut { uint32_t* r; __device__ void operator()(int64_t w, uint32_t exc, uint32_t) const { r[w] = exc; } };
__device__ __forceinline__ int32_t yd_rank(const uint32_t* __restrict__ U, const uint32_t* __restrict__ rankpre, int64_t bit) {
  const int64_t w = bit >> 5;
  return (int32_t)(rankpre[w] + (uint32_t)__popc(U[w] & ((1u << (bit & 31)) - 1u)));
}
__global__ void __launch_bounds__(256) yd_compact_kernel(const GDesc* __restrict__ desc, int64_t G, const uint32_t* __restrict__ U,
                                                         const uint32_t* __restrict__ rankpre, int ubase, GDesc* __restrict__ cdesc) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  GDesc d = desc[g];
  const int ne = (int)(d.meta & 0xffffu);
  d.start = yd_rank(U, rankpre, (int64_t)d.start - ubase);
  d.e0 = yd_rank(U, rankpre, (int64_t)d.e0 - ubase);
  if (ne >= 2) { d.s1 = yd_rank(U, rankpre, (int64_t)d.s1 - ubase); d.e1 = yd_rank(U, rankpre, (int64_t)d.e1 - ubase); }
  if (ne >= 3) { d.s2 = yd_rank(U, rankpre, (int64_t)d.s2 - ubase); d.e2 = yd_rank(U, rankpre, (int64_t)d.e2 - ubase); }
  d.zend = yd_rank(U, rankpre, (int64_t)d.zend - ubase);
  cdesc[g] = d;
}

// ---- Y3-Y5: chain member lists and their sub-chain heads ---------------------------------------------------------------
// A member heads a sub-chain when it is its chain's first, or when its start lies beyond every earlier end of the chain
// (and beyond the carried frontier). The test runs in GENOMIC coordinates on both paths: on the parallel path every group
// start and end and every carried frontier is a covered position, and rank() is strictly increasing over covered
// positions, so the answer is the one of the compact coordinates. The member pass therefore needs neither the compact
// coordinates nor the path choice (known only at the host sync after the count).
constexpr int YD_BLOCK = 1024;   // groups per counting block
// key of a chain's largest end (group end, raised to the carried frontier) in the prefix-maximum table: chain ids ascend
// in the chain-major table, so the plain prefix maximum is the segmented one; 0 = no member of the chain so far
__device__ __forceinline__ unsigned long long yd_end_key(int c, uint32_t e) { return ((unsigned long long)(c + 1) << 32) | e; }
// per (chain, block of groups): members, and the key of their largest end (0 without members); chain c = side*k + sample,
// tables are chain-major: blkcnt[c*nblk + b]. seed: carried frontier per chain (genomic, -1 = none), nullptr without carry.
__global__ void __launch_bounds__(128) yd_count_kernel(const uint32_t* __restrict__ bits, uint32_t W, int k, int64_t G, const uint8_t* __restrict__ gstrand,
                                                      const uint32_t* __restrict__ gend, const int32_t* __restrict__ seed,
                                                      uint32_t* __restrict__ blkcnt, unsigned long long* __restrict__ blkkey, int64_t nblk) {
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (warp >= nblk * W) return;
  const int64_t b = warp / W; const uint32_t w = (uint32_t)(warp % W);
  const int lane = tb_lane();
  const int64_t g0 = b * YD_BLOCK, g1 = (g0 + YD_BLOCK < G) ? g0 + YD_BLOCK : G;
  uint32_t cf = 0, cr = 0, mf = 0, mr = 0;
  for (int64_t base = g0; base < g1; base += 32) {
    const int64_t g = base + lane;
    uint32_t word = 0, ge = 0; uint8_t sc = 0;
    if (g < g1) { word = bits[(uint64_t)g * W + w]; if (word) { sc = gstrand[g]; ge = gend[g]; } }
    unsigned any = __ballot_sync(0xffffffffu, word != 0);
    while (any) {
      const int q = __ffs(any) - 1; any &= any - 1;
      const uint32_t wq = __shfl_sync(0xffffffffu, word, q);
      const int sq = __shfl_sync(0xffffffffu, (int)sc, q);
      const uint32_t eq = __shfl_sync(0xffffffffu, ge, q);
      if ((wq >> lane) & 1u) {
        if (sq != '-') { ++cf; mf = eq > mf ? eq : mf; }
        if (sq != '+') { ++cr; mr = eq > mr ? eq : mr; }
      }
    }
  }
  const int s = (int)(w * 32 + lane);
  if (s < k) {
    const int cfw = s, crv = k + s;
    if (seed) {
      if (seed[cfw] >= 0 && (uint32_t)seed[cfw] > mf) mf = (uint32_t)seed[cfw];
      if (seed[crv] >= 0 && (uint32_t)seed[crv] > mr) mr = (uint32_t)seed[crv];
    }
    blkcnt[(int64_t)cfw * nblk + b] = cf; blkkey[(int64_t)cfw * nblk + b] = cf ? yd_end_key(cfw, mf) : 0ULL;
    blkcnt[(int64_t)crv * nblk + b] = cr; blkkey[(int64_t)crv * nblk + b] = cr ? yd_end_key(crv, mr) : 0ULL;
  }
}
struct CntIn { const uint32_t* c; __device__ unsigned long long operator()(int64_t i) const { return c[i]; } };
struct CntOut { unsigned long long* o; __device__ void operator()(int64_t i, unsigned long long exc, unsigned long long) const { o[i] = exc; } };
struct OpSumU64 { typedef unsigned long long T; __host__ __device__ static T identity() { return 0; } __host__ __device__ static T combine(T a, T b) { return a + b; } };
// exclusive prefix maximum of the end keys, in place: every element is read by the thread that later overwrites it
struct EndMaxIn { const unsigned long long* t; __device__ unsigned long long operator()(int64_t i) const { return t[i]; } };
struct EndMaxOut { unsigned long long* t; __device__ void operator()(int64_t i, unsigned long long exc, unsigned long long) const { t[i] = exc; } };
__global__ void __launch_bounds__(128) yd_colbase_kernel(const unsigned long long* __restrict__ blkoff, const unsigned long long* __restrict__ total, int64_t nblk,
                                                         int nchains, unsigned long long* __restrict__ colbase) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < nchains) colbase[c] = blkoff[(int64_t)c * nblk];
  if (c == nchains) colbase[c] = *total;
}
// stable scatter of the members into the chain lists: mem[i] = (group id, head | chain << 1), one 8-byte store per member
// (the lanes of a warp write 32 different chains, so every store instruction costs a sector per lane). Each lane owns two
// chains (the sample's two strand lists) and carries their running end key in a register, from the prefix maximum of the
// earlier blocks.
__global__ void __launch_bounds__(128) yd_scatter_kernel(const uint32_t* __restrict__ bits, uint32_t W, int k, int64_t G, const uint8_t* __restrict__ gstrand,
                                                        const uint32_t* __restrict__ gstart, const uint32_t* __restrict__ gend, const int32_t* __restrict__ seed,
                                                        const unsigned long long* __restrict__ blkoff, const unsigned long long* __restrict__ blkpre, int64_t nblk,
                                                        uint2* __restrict__ mem) {
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (warp >= nblk * W) return;
  const int64_t b = warp / W; const uint32_t w = (uint32_t)(warp % W);
  const int lane = tb_lane();
  const int s = (int)(w * 32 + lane);
  const int64_t g0 = b * YD_BLOCK, g1 = (g0 + YD_BLOCK < G) ? g0 + YD_BLOCK : G;
  const int cf = s, cr = k + s;
  unsigned long long pf = 0, pr = 0, runf = 0, runr = 0;
  uint32_t sf = 0, sr = 0;   // carried frontiers (0 = none: every end key is above it)
  if (s < k) {
    pf = blkoff[(int64_t)cf * nblk + b]; pr = blkoff[(int64_t)cr * nblk + b];
    runf = blkpre[(int64_t)cf * nblk + b]; runr = blkpre[(int64_t)cr * nblk + b];
    if (seed) { sf = seed[cf] > 0 ? (uint32_t)seed[cf] : 0u; sr = seed[cr] > 0 ? (uint32_t)seed[cr] : 0u; }
  }
  const unsigned long long hf = (unsigned long long)(cf + 1) << 32, hr = (unsigned long long)(cr + 1) << 32;
  for (int64_t base = g0; base < g1; base += 32) {
    const int64_t g = base + lane;
    uint32_t word = 0, gs = 0, ge = 0; uint8_t sc = 0;
    if (g < g1) { word = bits[(uint64_t)g * W + w]; if (word) { sc = gstrand[g]; gs = gstart[g]; ge = gend[g]; } }
    unsigned any = __ballot_sync(0xffffffffu, word != 0);
    while (any) {
      const int q = __ffs(any) - 1; any &= any - 1;
      const uint32_t wq = __shfl_sync(0xffffffffu, word, q);
      const int sq = __shfl_sync(0xffffffffu, (int)sc, q);
      const uint32_t sx = __shfl_sync(0xffffffffu, gs, q), ex = __shfl_sync(0xffffffffu, ge, q);
      if ((wq >> lane) & 1u) {
        // head: first member of the chain (no key of this chain yet), or a start beyond every earlier end and the seed
        if (sq != '-') {
          const bool h = runf < hf || sx > (uint32_t)runf;
          mem[pf++] = make_uint2((uint32_t)(base + q), (h ? 1u : 0u) | ((uint32_t)cf << 1));
          const unsigned long long key = hf | (ex > sf ? ex : sf);
          runf = key > runf ? key : runf;
        }
        if (sq != '+') {
          const bool h = runr < hr || sx > (uint32_t)runr;
          mem[pr++] = make_uint2((uint32_t)(base + q), (h ? 1u : 0u) | ((uint32_t)cr << 1));
          const unsigned long long key = hr | (ex > sr ? ex : sr);
          runr = key > runr ? key : runr;
        }
      }
    }
  }
}

// Y5: list of the sub-chain heads by one stream compaction of the head bits. heads[nsub] = n_members closes the last
// sub-chain; work[0] (the work-unit counter of the frontier / sequential kernels) starts at 0 and work[1] = nsub.
struct HeadIn { const uint2* mem; __device__ uint32_t operator()(int64_t i) const { return mem[i].y & 1u; } };
struct HeadOut {
  uint32_t* heads; int64_t n; unsigned long long* work;
  __device__ void operator()(int64_t i, uint32_t exc, uint32_t inc) const {
    if (inc != exc) heads[exc] = (uint32_t)i;
    if (i == n - 1) { heads[inc] = (uint32_t)n; work[0] = 0; work[1] = inc; }
  }
};

constexpr int YD_WARPS = 8;
constexpr uint32_t YD_LONG = 16;     // sub-chains longer than this are walked by the whole warp

// ---- Y6: frontier recurrence -> kept-exon count per member -----------------------------------------------------------
struct Frontier {
  int E;
  __device__ __forceinline__ void reset() { E = -1; }
  // returns the number of kept exons of the read described by d (compact coordinates). Reads with more than three exons
  // continue over the CIGAR (genomic coordinates mapped through rank()).
  __device__ __forceinline__ uint32_t step(const ColIn& in, const GDesc& d, uint32_t rep, const uint32_t* U, const uint32_t* rankpre) {
    const int ne = (int)(d.meta & 0xffffu);
    if (E < d.start) { E = d.zend; return (uint32_t)ne; }   // bulk: the list is empty when the read is merged
    int cur = max(E, d.e0); uint32_t r = 1;
    if (ne >= 2 && d.s1 <= cur) {
      r = 2; cur = max(cur, d.e1);
      if (ne >= 3 && d.s2 <= cur) {
        r = 3; cur = max(cur, d.e2);
        if (ne > YD_INLINE_EX) {
          const int ubase = in.pos_lo + 1;
          ExonIter it; it.init(in.cigar, in.cig_off[rep], in.cig_off[rep + 1], in.pos[rep]);
          int s, e, j = 0;
          while (it.next(s, e)) {
            if (j++ < YD_INLINE_EX) continue;
            if (yd_rank(U, rankpre, (int64_t)s - ubase) > cur) break;
            ++r; cur = max(cur, (int)yd_rank(U, rankpre, (int64_t)e - ubase));
          }
        }
      }
    }
    E = cur;
    return r;
  }
};

// for a read with more than YD_INLINE_EX exons: index of the last exon whose (compact) start is <= frontier, and its end
__device__ __noinline__ int yd_reach(const ColIn& in, uint32_t rep, int frontier, const uint32_t* U, const uint32_t* rankpre, int* e_out) {
  const int ubase = in.pos_lo + 1;
  ExonIter it; it.init(in.cigar, in.cig_off[rep], in.cig_off[rep + 1], in.pos[rep]);
  int s, e, j = -1, last_e = 0;
  while (it.next(s, e)) {
    if (j >= 0 && yd_rank(U, rankpre, (int64_t)s - ubase) > frontier) break;
    ++j; last_e = yd_rank(U, rankpre, (int64_t)e - ubase);
  }
  *e_out = last_e;
  return j;
}

// links of the first `r` exons of a read into the chain bitmap that starts at bit `base` (exon [s,t] sets links s..t-1)
__device__ __forceinline__ void yd_emit_links(const ColIn& in, const GDesc& d, uint32_t r, uint32_t rep, const uint32_t* U, const uint32_t* rankpre,
                                              unsigned long long* bm, int64_t base) {
  if (d.e0 > d.start) yd_set_bits64(bm, base + d.start, base + d.e0 - 1);
  if (r >= 2 && d.e1 > d.s1) yd_set_bits64(bm, base + d.s1, base + d.e1 - 1);
  if (r >= 3 && d.e2 > d.s2) yd_set_bits64(bm, base + d.s2, base + d.e2 - 1);
  if (r > (uint32_t)YD_INLINE_EX) {
    const int ubase = in.pos_lo + 1;
    ExonIter it; it.init(in.cigar, in.cig_off[rep], in.cig_off[rep + 1], in.pos[rep]);
    int s, e; uint32_t j = 0;
    while (j < r && it.next(s, e)) {
      if (j++ < (uint32_t)YD_INLINE_EX) continue;
      const int64_t cs = yd_rank(U, rankpre, (int64_t)s - ubase), ce = yd_rank(U, rankpre, (int64_t)e - ubase);
      if (ce > cs) yd_set_bits64(bm, base + cs, base + ce - 1);
    }
  }
}

// Y6: frontier recurrence -> kept-exon count per member.
// The member array (all chains back to back, sub-chain heads flagged) is cut into work units that start at sub-chain
// heads (first head at or after a multiple of YD_UNIT members), so a unit needs no state from outside. Persistent warps
// pull units and walk them 32 members per step, YD_PF steps of descriptors in flight. Within a step the frontier is
// resolved by iterating "classes -> segmented prefix max -> classes" to its fixed point (see the kernel); the common
// classes (later exons of a spliced read dropped; or everything reached after a spanning read) settle in 1-2 scans.
constexpr int YD_PF = 4;
constexpr uint32_t YD_UNIT = 2048;
__global__ void __launch_bounds__(256) yd_unit_kernel(const uint32_t* __restrict__ heads, const unsigned long long* __restrict__ nsub_p, uint32_t n_members,
                                                      uint32_t nunits, uint32_t* __restrict__ ustart) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t nsub = (uint32_t)*nsub_p;
  if (u > nunits) return;
  if (u == nunits) { ustart[u] = n_members; return; }
  const uint32_t target = u * YD_UNIT;
  uint32_t lo = 0, hi = nsub;   // first h in [0,nsub] with heads[h] >= target (heads[nsub] = n_members)
  while (lo < hi) { const uint32_t mid = lo + ((hi - lo) >> 1); if (heads[mid] >= target) hi = mid; else lo = mid + 1; }
  ustart[u] = heads[lo];
}

// asynchronous global -> shared copies (LDGSTS): the gathers of the software pipeline below land in shared memory
// without holding registers, so the loop body exists once (no unrolled register queues) and stays inside the
// instruction cache
__device__ __forceinline__ void yd_cp_async8(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void yd_cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void yd_cp_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void yd_cp_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// frontier after member i, kept when i is the last member of chain c (the carry_out of the parallel path needs it)
__device__ __forceinline__ void yd_note_frontier(const uint2* mem, uint32_t i, uint32_t c, uint32_t n_members, int E, int32_t* efin) {
  if (i + 1 == n_members || (mem[i + 1].y >> 1) != c) efin[c] = E;
}

constexpr int YD_FWARPS = 4;   // warps per CTA of the frontier kernel (6 KB of shared-memory rings each)
// CARRY: lists carried into the window (seed) and / or the final frontiers wanted (efin); the instantiation without
// them is the kernel of a plain tb_collapse_window call
template <bool CARRY>
__global__ void __launch_bounds__(YD_FWARPS * 32) yd_frontier_kernel(ColIn in, const GDesc* __restrict__ cdesc, const uint32_t* __restrict__ rep,
                                                                    const uint2* __restrict__ mem,
                                                                    const uint32_t* __restrict__ ustart, uint32_t nunits, unsigned long long* work,
                                                                    const uint32_t* __restrict__ U, const uint32_t* __restrict__ rankpre,
                                                                    unsigned long long* __restrict__ bm, int64_t lpad, int32_t* __restrict__ mstart,
                                                                    const int32_t* __restrict__ seed, int32_t* __restrict__ efin, uint32_t n_members) {
  // two-stage pipeline per warp: member ids (group, head flag) are fetched 2*YD_PF steps ahead, descriptors YD_PF steps
  // ahead, so each of the two dependent gathers has YD_PF steps to land. A lane only ever reads ring entries it
  // requested itself (except in the replay, which synchronises the warp first).
  __shared__ __align__(16) GDesc s_ring[YD_FWARPS][YD_PF][32];
  __shared__ __align__(8) uint2 s_mem[YD_FWARPS][2 * YD_PF][32];   // (group id, head | chain << 1)
  __shared__ uint8_t s_r[YD_FWARPS][32];
  const int wl = tb_warp(), lane = tb_lane();
  for (;;) {
    unsigned long long u = 0;
    if (lane == 0) u = atomicAdd(&work[0], 1ULL);
    u = __shfl_sync(0xffffffffu, u, 0);
    if (u >= nunits) break;
    const uint32_t a = ustart[u], b = ustart[u + 1];
    if (a >= b) continue;
    Frontier F; F.reset();
    // prologue: ids of steps 0..2*YD_PF-1, then descriptors of steps 0..YD_PF-1 (one group each)
#pragma unroll
    for (int p = 0; p < 2 * YD_PF; ++p) {
      const uint32_t idx = a + (uint32_t)p * 32u + lane;
      if (idx < b) yd_cp_async8(&s_mem[wl][p][lane], mem + idx);
    }
    yd_cp_commit();
    yd_cp_wait<0>();
#pragma unroll
    for (int p = 0; p < YD_PF; ++p) {
      if (a + (uint32_t)p * 32u + lane < b) {
        const GDesc* src = cdesc + s_mem[wl][p][lane].x;
        yd_cp_async16(&s_ring[wl][p][lane], src); yd_cp_async16(reinterpret_cast<char*>(&s_ring[wl][p][lane]) + 16, reinterpret_cast<const char*>(src) + 16);
      }
      yd_cp_commit();
    }
    uint32_t step = 0;
#pragma unroll 1
    for (uint32_t cb = a; cb < b; cb += 32u, ++step) {
      const int slot = (int)(step % YD_PF), islot = (int)(step % (2 * YD_PF)), nslot = (int)((step + YD_PF) % (2 * YD_PF));
      yd_cp_wait<YD_PF - 1>();   // this step's descriptors and the ids of step + YD_PF have landed
      const int cnt = (int)((b - cb) < 32u ? (b - cb) : 32u);
      const bool live = lane < cnt;
      GDesc dm; dm.start = 0; dm.meta = 0; dm.e0 = dm.s1 = dm.e1 = dm.s2 = dm.e2 = dm.zend = 0;
      uint32_t g = 0; int head = 0;
      if (live) { dm = s_ring[wl][slot][lane]; g = s_mem[wl][islot][lane].x; head = (int)(s_mem[wl][islot][lane].y & 1u); }
      const int ne = (int)(dm.meta & 0xffffu);
      // For a frontier E >= start the step is  E' = max(E, end of the last exon whose start <= E)  and exactly the
      // exons up to that one are kept (exon starts lie beyond the previous exon's end); for E < start every exon is
      // kept and E' = last end. So, GIVEN each member's class (bulk, or index jx of the exon that E reaches), the
      // frontier is a segmented prefix max of one value per member. Guess the classes (heads: bulk, others: jx = 0,
      // i.e. later exons dropped), scan, re-derive the classes from the frontier each member then sees, and repeat
      // until nothing changes: a fixed point satisfies the recurrence member by member, hence is the exact result.
      int jx = 0; bool bulk = head != 0;
      int contrib = live ? (bulk ? dm.zend : dm.e0) : -1;
      if (CARRY && seed && live && head) {   // a chain's first member after a cut: its step starts from the carried frontier
        const int E0 = seed[s_mem[wl][islot][lane].y >> 1];
        if (E0 >= dm.start) {
          bulk = false;
          if (ne <= YD_INLINE_EX) {
            jx = (ne >= 3 && E0 >= dm.s2) ? 2 : ((ne >= 2 && E0 >= dm.s1) ? 1 : 0);
            contrib = jx == 2 ? dm.e2 : (jx == 1 ? dm.e1 : dm.e0);
          } else jx = yd_reach(in, rep[g], E0, U, rankpre, &contrib);
          contrib = max(contrib, E0);
        }
      }
      int e_after = F.E, e_lane = -1;
      bool replay = false;
#pragma unroll 1
      for (int iter = 0;; ++iter) {
        int v = contrib, h = head;
#pragma unroll
        for (int dd = 1; dd < 32; dd <<= 1) {
          const int v2 = __shfl_up_sync(0xffffffffu, v, dd), h2 = __shfl_up_sync(0xffffffffu, h, dd);
          if (lane >= dd) { if (!h) v = max(v, v2); h |= h2; }
        }
        if (!h) v = max(v, F.E);                     // no head at or before this lane: the carried sub-chain continues
        int pm = __shfl_up_sync(0xffffffffu, v, 1);
        if (lane == 0) pm = F.E;
        bool nb = bulk; int nj = jx, nc = contrib;
        if (live && !head) {
          nb = pm < dm.start;
          if (nb) { nj = 0; nc = dm.zend; }
          else if (ne <= YD_INLINE_EX) {
            nj = (ne >= 3 && pm >= dm.s2) ? 2 : ((ne >= 2 && pm >= dm.s1) ? 1 : 0);
            nc = nj == 2 ? dm.e2 : (nj == 1 ? dm.e1 : dm.e0);
          } else nj = yd_reach(in, rep[g], pm, U, rankpre, &nc);
        }
        const bool changed = nb != bulk || nj != jx;
        bulk = nb; jx = nj; contrib = nc;
        if (!__any_sync(0xffffffffu, changed)) { e_after = __shfl_sync(0xffffffffu, v, cnt - 1); e_lane = v; break; }
        if (iter >= 8) { replay = true; break; }
      }
      uint32_t r = bulk ? (uint32_t)ne : (uint32_t)jx + 1u;
      if (replay) {   // no fixed point within a few rounds: one lane walks the step in order (ring entries of all lanes)
        __syncwarp();
        if (lane == 0) {
          for (int t = 0; t < cnt; ++t) {
            const GDesc& d = s_ring[wl][slot][t];
            const uint32_t fl = s_mem[wl][islot][t].y;
            if (fl & 1u) { F.reset(); if (CARRY && seed) F.E = seed[fl >> 1]; }
            const uint32_t rr = ((d.meta & 0xffffu) > (uint32_t)YD_INLINE_EX) ? rep[s_mem[wl][islot][t].x] : 0u;
            s_r[wl][t] = (uint8_t)F.step(in, d, rr, U, rankpre);
            if (CARRY && efin) yd_note_frontier(mem, cb + (uint32_t)t, fl >> 1, n_members, F.E, efin);
          }
        }
        F.E = __shfl_sync(0xffffffffu, F.E, 0);
        __syncwarp();
        r = s_r[wl][lane];
        __syncwarp();
      } else {
        F.E = e_after;
        if (CARRY && efin && live) yd_note_frontier(mem, cb + lane, s_mem[wl][islot][lane].y >> 1, n_members, e_lane, efin);
      }
      // Y7 fused: the kept exons OR their links into the chain's bitmap; compact start per member for the lookup
      if (live) {
        const int64_t base = (int64_t)(s_mem[wl][islot][lane].y >> 1) * lpad;
        yd_emit_links(in, dm, r, r > (uint32_t)YD_INLINE_EX ? rep[g] : 0u, U, rankpre, bm, base);
        mstart[cb + lane] = dm.start;
      }
      // refill: descriptors of step + YD_PF into this step's ring slot, ids of step + 2*YD_PF into this step's id slot
      {
        const uint32_t idx = cb + 32u * YD_PF + lane;
        if (idx < b) {
          const GDesc* src = cdesc + s_mem[wl][nslot][lane].x;
          yd_cp_async16(&s_ring[wl][slot][lane], src); yd_cp_async16(reinterpret_cast<char*>(&s_ring[wl][slot][lane]) + 16, reinterpret_cast<const char*>(src) + 16);
        }
        const uint32_t idx2 = cb + 32u * 2 * YD_PF + lane;
        if (idx2 < b) yd_cp_async8(&s_mem[wl][islot][lane], mem + idx2);
        yd_cp_commit();
      }
    }
    yd_cp_wait<0>();
  }
}

// ---- Y8: position of the last clear link before every 512-bit block ---------------------------------------------------
struct OpMaxI64 { typedef long long T; __host__ __device__ static T identity() { return -1; } __host__ __device__ static T combine(T a, T b) { return a > b ? a : b; } };
struct LastZeroIn {   // highest clear bit of block b (global bit index), -1 if the block is all ones
  const unsigned long long* bm;
  __device__ long long operator()(int64_t b) const {
    for (int w = 7; w >= 0; --w) {
      const unsigned long long z = ~bm[b * 8 + w];
      if (z) return (b * 8 + w) * 64 + (63 - __clzll((long long)z));
    }
    return -1;
  }
};
struct LastZeroOut { long long* lz; __device__ void operator()(int64_t b, long long exc, long long) const { lz[b] = exc; } };

// ---- Y9: d = number of consecutive set links ending at start-1 --------------------------------------------------------
// last clear bit below bit q (global index) of the link bitmaps: the block's words, then the prefix over earlier blocks
__device__ __forceinline__ long long yd_clear_below(const unsigned long long* __restrict__ bm, const long long* __restrict__ lz, int64_t q) {
  int64_t w = q >> 6; const int b = (int)(q & 63);
  unsigned long long zeros = ~bm[w] & ((1ULL << b) - 1ULL);
  const int64_t wb = w & ~7LL;   // first word of the 512-bit block
  for (;;) {
    if (zeros) return w * 64 + (63 - __clzll((long long)zeros));
    if (w == wb) return lz[wb >> 3];
    --w; zeros = ~bm[w];
  }
}
// ext (carried lists only): a run of links that reaches the chain's first bit continues the carried node that began before
// the window, ext[chain] positions further down
__global__ void __launch_bounds__(256) yd_lookup_kernel(const int32_t* __restrict__ mstart, const uint2* __restrict__ mem, int64_t n_members,
                                                        const unsigned long long* __restrict__ bm,
                                                        const long long* __restrict__ lz, int64_t lpad, int32_t* __restrict__ yd,
                                                        const int32_t* __restrict__ ext) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_members) return;
  const int x = mstart[i];
  if (x <= 0) {
    if (ext && x == 0) { const int32_t d = ext[mem[i].y >> 1]; if (d > 0) atomicMax(&yd[mem[i].x], d); }
    return;
  }
  const uint2 m = mem[i];
  const uint32_t g = m.x;
  const int64_t base = (int64_t)(m.y >> 1) * lpad;
  const int64_t q = base + x - 1;
  if (!((bm[q >> 6] >> (q & 63)) & 1ULL)) return;
  long long z = yd_clear_below(bm, lz, q);
  if (z < base - 1) z = base - 1;   // cannot happen (every chain's region ends with clear padding); keeps d bounded
  long long d = q - z;
  if (ext && z == base - 1) d += ext[m.y >> 1];
  if (d > 0) atomicMax(&yd[g], (int32_t)d);
}

// ---- carried lists (tb_collapse_window_carry) ---------------------------------------------------------------------------
// Carry-in: chain c's list starts as the carried nodes that are still alive (end >= ubase, the window's first start). On
// the parallel path that is what a first member of the chain made of those nodes would leave behind (all appended to an
// empty list, links only inside a node): their positions enter U, their links enter the chain's bitmap, the chain's
// frontier starts at the last node's end, and the one node that may begin below ubase is cut at ubase with the cut-off
// length kept in ext[c]. On the sequential path the nodes are loaded into the list itself.
__device__ __forceinline__ int yd_seg_chain(const long long* __restrict__ coff, int nchains, long long q) {   // last c with coff[c] <= q
  int lo = 0, hi = nchains;
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (coff[mid] <= q) lo = mid; else hi = mid; }
  return lo;
}
__global__ void __launch_bounds__(256) yd_carry_u_kernel(const int32_t* __restrict__ cs, const int32_t* __restrict__ ce, int64_t nin, int ubase,
                                                         uint32_t* __restrict__ U, int64_t ubits, long long* __restrict__ status) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nin || ce[q] < ubase) return;
  const int s = max(cs[q], ubase), e = ce[q];
  if ((int64_t)e - ubase >= ubits) { status[YS_FALLBACK] = 1; return; }
  yd_set_bits32(U, (int64_t)s - ubase, (int64_t)e - ubase);
}
// U == nullptr: sequential path, genomic seeds
__global__ void __launch_bounds__(128) yd_carry_seed_kernel(const long long* __restrict__ coff, const int32_t* __restrict__ cs, const int32_t* __restrict__ ce,
                                                            int nchains, int ubase, const uint32_t* __restrict__ U, const uint32_t* __restrict__ rankpre,
                                                            int32_t* __restrict__ seed, int32_t* __restrict__ ext, int32_t* __restrict__ efin) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nchains) return;
  const long long a = coff[c], b = coff[c + 1];
  int32_t sd = -1, x = 0;
  if (b > a && ce[b - 1] >= ubase) {
    sd = U ? yd_rank(U, rankpre, (int64_t)ce[b - 1] - ubase) : ce[b - 1];
    for (long long q = a; q < b; ++q)
      if (ce[q] >= ubase) { if (cs[q] < ubase) x = ubase - cs[q]; break; }
  }
  seed[c] = sd; ext[c] = x;
  if (efin) efin[c] = sd;
}
__global__ void __launch_bounds__(256) yd_carry_links_kernel(const long long* __restrict__ coff, const int32_t* __restrict__ cs, const int32_t* __restrict__ ce,
                                                             int64_t nin, int nchains, int ubase, const uint32_t* __restrict__ U,
                                                             const uint32_t* __restrict__ rankpre, unsigned long long* __restrict__ bm, int64_t lpad) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nin || ce[q] < ubase) return;
  const int64_t base = (int64_t)yd_seg_chain(coff, nchains, q) * lpad;
  const int64_t a = yd_rank(U, rankpre, (int64_t)max(cs[q], ubase) - ubase), b = yd_rank(U, rankpre, (int64_t)ce[q] - ubase);
  if (b > a) yd_set_bits64(bm, base + a, base + b - 1);
}

// Carry-out, canonical form for B = pos_hi + 1: nodes with end >= B that cover two positions or more, and the last node
// when its end >= B. A chain reserves its slots with one atomicAdd; past the capacity only the count is kept.
__device__ __forceinline__ bool yd_keep_node(int32_t s, int32_t e, bool last, int32_t B) { return e >= B && (e > s || last); }
__device__ __forceinline__ long long yd_reserve(long long* ometa, int nchains, int c, long long cnt) {
  const long long slot = (long long)atomicAdd((unsigned long long*)&ometa[2 * nchains], (unsigned long long)cnt);
  ometa[2 * c] = slot; ometa[2 * c + 1] = cnt;
  return slot;
}
__device__ __forceinline__ void yd_put(int32_t* os, int32_t* oe, int64_t cap, long long at, int32_t s, int32_t e) {
  if (at < cap) { os[at] = s; oe[at] = e; }
}
// compact coordinate -> genomic offset from ubase: the a-th set bit of U
__device__ int64_t yd_select(const uint32_t* __restrict__ U, const uint32_t* __restrict__ rankpre, int64_t nuw, int64_t a) {
  int64_t lo = 0, hi = nuw - 1;
  while (lo < hi) { const int64_t mid = (lo + hi + 1) >> 1; if ((int64_t)rankpre[mid] <= a) lo = mid; else hi = mid - 1; }
  uint32_t w = U[lo];
  for (int64_t r = a - (int64_t)rankpre[lo]; r > 0; --r) w &= w - 1;
  return lo * 32 + __ffs((int)w) - 1;
}
// first bit >= p (chain-relative) that is set (want = true) or clear, or lim
__device__ int64_t yd_next_bit(const unsigned long long* __restrict__ bm, int64_t base, int64_t p, int64_t lim, bool want) {
  while (p < lim) {
    const int64_t gq = base + p, w = gq >> 6;
    const unsigned long long word = (want ? bm[w] : ~bm[w]) & (~0ULL << (gq & 63));
    if (word) { const int64_t r = w * 64 + __ffsll((long long)word) - 1 - base; return r < lim ? r : lim; }
    p = (w + 1) * 64 - base;
  }
  return lim;
}
struct YdParOut {   // what the extraction on the parallel path reads
  const unsigned long long* bm; const long long* lz; int64_t lpad;
  const uint32_t* U; const uint32_t* rankpre; int64_t nuw; int ubase; int64_t bbit;   // bbit = B - ubase (< the bits of U)
  const int32_t* ext; const int32_t* efin;
};
// nodes of chain c on the parallel path: the maximal runs of links ending at or beyond cB - 1, then the last node [E, E]
// when the link below the frontier E is clear; written from slot `at` when write is set. Returns the node count.
__device__ long long yd_par_nodes(const YdParOut& P, int c, bool write, long long at, int32_t* os, int32_t* oe, int64_t cap) {
  const int64_t E = P.efin[c], cB = yd_rank(P.U, P.rankpre, P.bbit);   // cB: compact coordinate of the first covered position >= B
  if (E < cB) return 0;
  const int64_t base = (int64_t)c * P.lpad, p0 = cB > 0 ? cB - 1 : 0;
  long long cnt = 0;
  auto gend = [&](int64_t a) -> int32_t { return (int32_t)(P.ubase + yd_select(P.U, P.rankpre, P.nuw, a)); };
  auto gstart = [&](int64_t a) -> int32_t { return (a == 0 && P.ext[c] > 0) ? P.ubase - P.ext[c] : gend(a); };
  int64_t p = p0;
  bool last_linked = false;
  while (p < E) {
    p = yd_next_bit(P.bm, base, p, E, true);
    if (p >= E) break;
    int64_t r0 = p;
    if (p == p0 && p > 0 && ((P.bm[(base + p - 1) >> 6] >> ((base + p - 1) & 63)) & 1ULL)) {   // the run began before the scan
      long long z = yd_clear_below(P.bm, P.lz, base + p);
      r0 = z < base ? 0 : z + 1 - base;
    }
    const int64_t q = yd_next_bit(P.bm, base, p, E, false);   // links r0..q-1: node [r0, q]
    if (write) yd_put(os, oe, cap, at + cnt, gstart(r0), gend(q));
    ++cnt;
    last_linked = q == E;
    p = q;
  }
  if (!last_linked) { if (write) yd_put(os, oe, cap, at + cnt, gstart(E), gend(E)); ++cnt; }
  return cnt;
}
// one thread per chain: chains without members in this window pass their carried nodes on (re-filtered against B);
// on the parallel path the others are read from the link bitmaps (the sequential path wrote them from its lists)
__global__ void __launch_bounds__(128) yd_carry_out_kernel(int nchains, const unsigned long long* __restrict__ colbase, const long long* __restrict__ coff,
                                                           const int32_t* __restrict__ cs, const int32_t* __restrict__ ce, int32_t B, bool parallel,
                                                           YdParOut P, int32_t* __restrict__ os, int32_t* __restrict__ oe, int64_t cap,
                                                           long long* __restrict__ ometa) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nchains) return;
  if (colbase[c + 1] == colbase[c]) {
    long long cnt = 0;
    const long long a = coff ? coff[c] : 0, b = coff ? coff[c + 1] : 0;
    for (long long q = a; q < b; ++q) cnt += yd_keep_node(cs[q], ce[q], q == b - 1, B);
    const long long at = yd_reserve(ometa, nchains, c, cnt);
    long long j = 0;
    for (long long q = a; q < b; ++q) if (yd_keep_node(cs[q], ce[q], q == b - 1, B)) yd_put(os, oe, cap, at + j++, cs[q], ce[q]);
  } else if (parallel) {
    const long long cnt = yd_par_nodes(P, c, false, 0, os, oe, cap);
    yd_par_nodes(P, c, true, yd_reserve(ometa, nchains, c, cnt), os, oe, cap);
  }
}
// everything the sequential kernel needs for the carry
struct YdSeqCarry {
  const long long* coff; const int32_t* cs; const int32_t* ce;   // carry_in, nullptr = lists start empty
  const unsigned long long* colbase; const uint2* mem; int nchains; int ubase;
  int32_t B; int32_t* os; int32_t* oe; int64_t cap; long long* ometa;   // os == nullptr: no carry_out
};

// ---- sequential fallback: the literal list ------------------------------------------------------------------------------
// one segment list; node q lives at st[q*32], en[q*32] (the lane offset is folded into the pointers)
struct SegArr {
  int n; uint32_t last_pos; int last_dist; int cap;
  uint32_t* st; uint32_t* en;
  __device__ __forceinline__ uint32_t& S(int q) { return st[q << 5]; }
  __device__ __forceinline__ uint32_t& E(int q) { return en[q << 5]; }
  __device__ void reset() { n = 0; last_pos = 0; last_dist = -1; }
  __device__ void erase(int a, int b) {  // remove [a,b)
    const int d = b - a; if (d <= 0) return;
    for (int q = b; q < n; ++q) { S(q - d) = S(q); E(q - d) = E(q); }
    n -= d;
  }
  __device__ bool insert(int at, uint32_t s, uint32_t e) {
    if (n >= cap) return false;
    for (int q = n; q > at; --q) { S(q) = S(q - 1); E(q) = E(q - 1); }
    S(at) = s; E(at) = e; ++n; return true;
  }
  // mergeRead :167-219 over an exon source; returns false on capacity overflow
  template <class Src>
  __device__ bool merge(Src& src) {
    int s, e;
    if (n == 0) {
      while (src.next(s, e)) { if (n >= cap) return false; S(n) = (uint32_t)s; E(n) = (uint32_t)e; ++n; }
      return true;
    }
    int cur = 0;
    while (src.next(s, e)) {
      const uint32_t es = (uint32_t)s, ee = (uint32_t)e;
      while (cur < n) {
        if (ee < S(cur)) { if (!insert(cur, es, ee)) return false; ++cur; break; }  // inserted before the cursor node, which is now at cur
        if (es <= E(cur)) {
          if (es < S(cur)) S(cur) = es;
          if (ee > E(cur)) E(cur) = ee;
          const int nx = cur + 1;
          while (nx < n && S(nx) <= E(cur)) {
            const uint32_t nend = E(nx);
            erase(nx, nx + 1);
            if (nend > E(cur)) { E(cur) = nend; break; }
          }
          break;
        }
        ++cur;
      }
      if (cur >= n) return true;  // cursor ran off the list: this and all later exons are dropped (reference behaviour)
    }
    return true;
  }
  // the carried nodes of one chain that are still alive; false on capacity overflow
  __device__ __noinline__ bool seed(const int32_t* cs, const int32_t* ce, long long a, long long b, int ubase) {
    for (long long q = a; q < b; ++q) {
      if (ce[q] < ubase) continue;
      if (n >= cap) return false;
      S(n) = (uint32_t)cs[q]; E(n) = (uint32_t)ce[q]; ++n;
    }
    return true;
  }
  // the list in canonical carry form
  __device__ __noinline__ void export_carry(uint32_t c, const YdSeqCarry& k) {
    long long cnt = 0;
    for (int q = 0; q < n; ++q) cnt += yd_keep_node((int32_t)S(q), (int32_t)E(q), q == n - 1, k.B);
    const long long at = yd_reserve(k.ometa, k.nchains, (int)c, cnt);
    long long j = 0;
    for (int q = 0; q < n; ++q) if (yd_keep_node((int32_t)S(q), (int32_t)E(q), q == n - 1, k.B)) yd_put(k.os, k.oe, k.cap, at + j++, (int32_t)S(q), (int32_t)E(q));
  }
  // processRead :221-250
  template <class Src>
  __device__ int process(Src& src, uint32_t rstart, bool& ok) {
    if (last_pos == rstart) { ok = merge(src) && ok; return last_dist; }
    int d = 0, prev = -1;
    for (int q = 0; q < n && S(q) < rstart; ++q) prev = q;
    if (prev >= 0) {
      if (E(prev) >= rstart) d = (int)(rstart - S(prev));
      if (d == 0) erase(0, prev + 1);
      else erase(0, prev);  // eager drop of the inert nodes before prev
    }
    last_pos = rstart; last_dist = d;
    ok = merge(src) && ok;
    return d;
  }
};

struct InlineExons {  // exon source over a descriptor
  int start, ne, i; int e0, s1, e1, s2, e2;
  __device__ bool next(int& s, int& e) {
    if (i >= ne) return false;
    if (i == 0) { s = start; e = e0; } else if (i == 1) { s = s1; e = e1; } else { s = s2; e = e2; }
    ++i; return true;
  }
};

__device__ __forceinline__ int yd_step(const ColIn& in, SegArr& L, const GDesc& d, uint32_t r, bool& ok) {
  const int ne = (int)(d.meta & 0xffffu);
  if (ne <= YD_INLINE_EX) { InlineExons src{d.start, ne, 0, d.e0, d.s1, d.e1, d.s2, d.e2}; return L.process(src, (uint32_t)d.start, ok); }
  ExonIter it; it.init(in.cigar, in.cig_off[r], in.cig_off[r + 1], d.start - 1);
  return L.process(it, (uint32_t)d.start, ok);
}

constexpr int YD_CAP_SMEM = 24;      // live nodes per list in shared memory
constexpr int YD_CAP_GLOBAL = 4096;  // live nodes per list in the global-memory repeat

template <bool SMEM, bool CARRY>   // CARRY: lists seeded from / exported to a carry (ca); false = plain tb_collapse_window
__global__ void __launch_bounds__(YD_WARPS * 32) yd_chain_kernel(ColIn in, const GDesc* __restrict__ desc, const uint32_t* __restrict__ rep,
                                                                const uint2* __restrict__ mem, const uint32_t* __restrict__ heads,
                                                                unsigned long long* work, int32_t* __restrict__ yd, uint32_t* gscratch, long long* status,
                                                                YdSeqCarry ca) {
  extern __shared__ __align__(16) uint32_t s_dyn[];   // SMEM: YD_WARPS * 2 * YD_CAP_SMEM * 32 words of lists
  __shared__ GDesc s_desc[YD_WARPS][32];
  __shared__ uint32_t s_g[YD_WARPS][32];
  __shared__ int s_d[YD_WARPS][32];
  const int wl = tb_warp(), lane = tb_lane();
  const int cap = SMEM ? YD_CAP_SMEM : YD_CAP_GLOBAL;
  uint32_t* base = SMEM ? &s_dyn[(size_t)wl * 2 * YD_CAP_SMEM * 32] : gscratch + ((size_t)blockIdx.x * YD_WARPS + wl) * 2 * (size_t)YD_CAP_GLOBAL * 32;
  SegArr L; L.cap = cap; L.st = base + lane; L.en = base + (size_t)cap * 32 + lane;
  SegArr L0; L0.cap = cap; L0.st = base; L0.en = base + (size_t)cap * 32;   // lane 0's list, used by the cooperative walk
  const unsigned long long nsub = work[1];
  bool ok = true;
  for (;;) {
    unsigned long long j0 = 0;
    if (lane == 0) j0 = atomicAdd(&work[0], 32ULL);
    j0 = __shfl_sync(0xffffffffu, j0, 0);
    if (j0 >= nsub) break;
    const unsigned long long j = j0 + lane;
    uint32_t c0 = 0, c1 = 0;
    if (j < nsub) { c0 = heads[j]; c1 = heads[j + 1]; }
    const uint32_t len = c1 - c0;
    const uint32_t ch = (CARRY && len > 0) ? ca.mem[c0].y >> 1 : 0u;
    if (len > 0 && len <= YD_LONG) {   // short sub-chains: one per lane
      L.reset();
      if (CARRY && ca.coff && c0 == ca.colbase[ch]) ok = L.seed(ca.cs, ca.ce, ca.coff[ch], ca.coff[ch + 1], ca.ubase) && ok;
      for (uint32_t i = c0; i < c1; ++i) {
        const uint32_t g = mem[i].x;
        const int dist = yd_step(in, L, desc[g], rep[g], ok);
        if (dist > 0) atomicMax(&yd[g], dist);
      }
      if (CARRY && ca.os && c1 == ca.colbase[ch + 1]) L.export_carry(ch, ca);
    }
    unsigned longs = __ballot_sync(0xffffffffu, len > YD_LONG);
    while (longs) {                    // long sub-chains: the whole warp walks them one after the other
      const int q = __ffs(longs) - 1; longs &= longs - 1;
      const uint32_t a = __shfl_sync(0xffffffffu, c0, q), b = __shfl_sync(0xffffffffu, c1, q);
      const uint32_t chq = __shfl_sync(0xffffffffu, ch, q);
      L0.reset();
      if (CARRY && lane == 0 && ca.coff && a == ca.colbase[chq]) ok = L0.seed(ca.cs, ca.ce, ca.coff[chq], ca.coff[chq + 1], ca.ubase) && ok;
      uint32_t gnext = 0; GDesc dnext; dnext.start = 0; dnext.meta = 0; dnext.e0 = dnext.s1 = dnext.e1 = dnext.s2 = dnext.e2 = dnext.zend = 0;
      if (a + lane < b) { gnext = mem[a + lane].x; dnext = desc[gnext]; }
      for (uint32_t cb = a; cb < b; cb += 32) {
        const uint32_t g = gnext;
        s_desc[wl][lane] = dnext; s_g[wl][lane] = gnext;
        __syncwarp();
        if (cb + 32 + lane < b) { gnext = mem[cb + 32 + lane].x; dnext = desc[gnext]; }   // prefetch the next batch
        if (lane == 0) {
          const int cnt = (int)((b - cb) < 32u ? (b - cb) : 32u);
          for (int t = 0; t < cnt; ++t) {
            const GDesc& d = s_desc[wl][t];
            const uint32_t rr = ((d.meta & 0xffffu) > (uint32_t)YD_INLINE_EX) ? rep[s_g[wl][t]] : 0u;
            s_d[wl][t] = yd_step(in, L0, d, rr, ok);
          }
        }
        __syncwarp();
        if (cb + lane < b) { const int dist = s_d[wl][lane]; if (dist > 0) atomicMax(&yd[g], dist); }
        __syncwarp();
      }
      if (CARRY && lane == 0 && ca.os && b == ca.colbase[chq + 1]) L0.export_carry(chq, ca);
    }
  }
  if (!ok) status[CS_YD_OVERFLOW] = 1;
}

__global__ void __launch_bounds__(256) yd_combine_kernel(int32_t* __restrict__ yd, const int32_t* __restrict__ ydc, int64_t G) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < G) { const int32_t a = yd[g], b = ydc[g]; yd[g] = a > b ? a : b; }   // max(carried YD tags, chain distance); 0 = no tag
}
__global__ void yd_store_lc_kernel(const uint32_t* tot, long long* status) { status[YS_LC] = *tot; }

}  // namespace

int col_yd(tb_ctx* ctx, const ColIn& in, const ColGeom& g, const ColGroups& grp, int64_t G, const YdCarry& cy) {
  cudaStream_t st = ctx->stream;
  DevBuf* B = ctx->buf;
  const uint32_t W = g.W; const int k = g.k; const int nchains = 2 * k;
  const int64_t nblk = (G + YD_BLOCK - 1) / YD_BLOCK;
  const char* env = getenv("TB_YD_PATH");
  bool parallel = !(env && env[0] == 's');
  const int64_t ubits = (int64_t)g.S + YD_U_SLACK;
  const int64_t nuw = (ubits + 31) / 32 + 1;
  const int ubase = in.pos_lo + 1;
  TB_CUDA(B[XB_GDESC].ensure(sizeof(GDesc) * (size_t)G * 2));
  TB_CUDA(B[XB_YDPM].ensure(sizeof(uint32_t) * (size_t)G * 2 + (size_t)G + 64));
  TB_CUDA(B[XB_YDBLK].ensure(sizeof(uint32_t) * ((size_t)nblk * nchains + nchains) + sizeof(uint64_t) * (2 * (size_t)nblk * nchains + nchains + 16)));
  TB_CUDA(B[XB_WORK].ensure(256));
  TB_CUDA(B[XB_YDC].ensure(sizeof(int32_t) * (size_t)G));
  GDesc* desc = B[XB_GDESC].as<GDesc>();
  GDesc* cdesc = desc + G;
  uint32_t* gend = B[XB_YDPM].as<uint32_t>();
  uint32_t* gstart = gend + G;
  uint8_t* gstrand = (uint8_t*)(gstart + G);
  unsigned long long* blkoff = B[XB_YDBLK].as<unsigned long long>();            // [nchains*nblk] exclusive member offsets, chain-major
  unsigned long long* blkkey = blkoff + (size_t)nblk * nchains;                 // [nchains*nblk] end keys, then their exclusive prefix maxima
  unsigned long long* colbase = blkkey + (size_t)nblk * nchains;                // [nchains+1]
  uint32_t* blkcnt = (uint32_t*)(colbase + nchains + 16);                       // [nchains*nblk]
  int32_t* gseed = (int32_t*)(blkcnt + (size_t)nblk * nchains);                 // [nchains] carried frontier, genomic
  unsigned long long* work = B[XB_WORK].as<unsigned long long>() + 8;           // the tile kernel's slot counter sits at +0
  int32_t* ydc = B[XB_YDC].as<int32_t>();
  long long* h_status = ctx->pinned[0].as<long long>();
  uint32_t* U = nullptr; uint32_t* rankpre = nullptr;
  if (parallel) {
    TB_CUDA(B[XB_YDU].ensure(sizeof(uint32_t) * (size_t)nuw * 2 + 64));
    U = B[XB_YDU].as<uint32_t>(); rankpre = U + nuw;
    TB_CUDA(cudaMemsetAsync(U, 0, sizeof(uint32_t) * (size_t)nuw, st));
  }
  TB_CUDA(cudaMemsetAsync(ydc, 0, sizeof(int32_t) * (size_t)G, st));
  TB_CUDA(cudaMemsetAsync(g.d_status + YS_FALLBACK, 0, 2 * sizeof(long long), st));
  if (cy.out) TB_CUDA(cudaMemsetAsync(cy.ometa + 2 * nchains, 0, sizeof(long long), st));
  int64_t agg_need = tb_scan_blocks((int64_t)nblk * nchains); if (tb_scan_blocks(nuw) > agg_need) agg_need = tb_scan_blocks(nuw);
  TB_CUDA(B[XB_AGG].ensure((size_t)(agg_need + 8) * sizeof(uint64_t)));
  // ---- Y1, Y2 ----
  yd_desc_kernel<<<tb_grid_for(G, 256), 256, 0, st>>>(in, grp.rep, G, desc, gend, gstart, gstrand, U, ubits, g.d_status);
  ctx->launches++;
  if (parallel && cy.in && cy.nin > 0) {   // carried nodes take part in the compact coordinates
    yd_carry_u_kernel<<<tb_grid_for(cy.nin, 256), 256, 0, st>>>(cy.cs, cy.ce, cy.nin, ubase, U, ubits, g.d_status);
    ctx->launches++;
  }
  if (parallel) {
    TB_CUDA((tb_device_scan<OpSumU32>(ctx, UPopIn{U}, nuw, B[XB_AGG].as<uint32_t>(), UPopOut{rankpre})));
    yd_store_lc_kernel<<<1, 1, 0, st>>>(B[XB_AGG].as<uint32_t>() + tb_scan_blocks(nuw), g.d_status);
    ctx->launches++;
  }
  // ---- Y3: member counts -> offsets; largest ends -> per-chain prefix maxima (head test in genomic coordinates, see Y3-Y5) ----
  if (cy.in) {
    yd_carry_seed_kernel<<<tb_grid_for(nchains, 128), 128, 0, st>>>(cy.coff, cy.cs, cy.ce, nchains, ubase, nullptr, nullptr, gseed, cy.ext, nullptr);
    ctx->launches++;
  }
  const int64_t nwarps = nblk * W;
  yd_count_kernel<<<tb_grid_for(nwarps * 32, 128), 128, 0, st>>>(grp.bits, W, k, G, gstrand, gend, cy.in ? gseed : nullptr, blkcnt, blkkey, nblk);
  ctx->launches++;
  TB_CUDA((tb_device_scan<OpSumU64>(ctx, CntIn{blkcnt}, (int64_t)nblk * nchains, B[XB_AGG].as<unsigned long long>(), CntOut{blkoff})));
  yd_colbase_kernel<<<tb_grid_for(nchains + 1, 128), 128, 0, st>>>(blkoff, B[XB_AGG].as<unsigned long long>() + tb_scan_blocks((int64_t)nblk * nchains), nblk, nchains, colbase);
  ctx->launches++;
  TB_CUDA((tb_device_scan<OpMaxU64>(ctx, EndMaxIn{blkkey}, (int64_t)nblk * nchains, B[XB_AGG].as<unsigned long long>(), EndMaxOut{blkkey})));
  // member count, compact length and the fallback flag are only known on the device
  TB_CUDA(cudaMemcpyAsync(h_status, g.d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
  TB_CUDA(cudaMemcpyAsync(h_status + 16, colbase + nchains, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  TB_CUDA(cudaStreamSynchronize(st));
  const int64_t n_members = h_status[16];
  if (n_members >= (1LL << 32)) { ctx->set_error("tb_collapse_window: %lld chain members exceed the 32-bit YD index", (long long)n_members); return 1; }
  if (h_status[YS_FALLBACK]) parallel = false;
  const int64_t Lc = h_status[YS_LC];
  ctx->last_yd_path = parallel ? 0 : 1;
  ctx->last_yd_stat[0] = n_members; ctx->last_yd_stat[1] = 0; ctx->last_yd_stat[2] = parallel ? Lc : 0; ctx->last_yd_stat[3] = nblk;
  if (cy.in) {
    yd_carry_seed_kernel<<<tb_grid_for(nchains, 128), 128, 0, st>>>(cy.coff, cy.cs, cy.ce, nchains, ubase, parallel ? U : nullptr, rankpre, cy.seed, cy.ext,
                                                                  parallel && cy.out ? cy.efin : nullptr);
    ctx->launches++;
  } else if (parallel && cy.out) {
    TB_CUDA(cudaMemsetAsync(cy.efin, 0xff, sizeof(int32_t) * (size_t)nchains, st));
  }
  const int32_t* seed = cy.in ? cy.seed : nullptr;
  YdParOut pout; memset(&pout, 0, sizeof(pout));
  if (n_members > 0) {
    TB_CUDA(B[XB_YDCHAIN].ensure(sizeof(uint2) * ((size_t)n_members + 32)));
    TB_CUDA(B[XB_BHEAD].ensure(sizeof(uint32_t) * ((size_t)n_members + 32)));
    const int64_t lpad = ((Lc + 1 + 511) / 512) * 512;            // bits per chain, at least one clear padding bit
    const int64_t nwords = lpad / 64 * nchains, nblocks512 = nwords / 8;
    TB_CUDA(B[XB_AGG].ensure((size_t)(tb_scan_blocks(nblocks512 > n_members ? nblocks512 : n_members) + 8) * sizeof(uint64_t)));
    uint2* mem = B[XB_YDCHAIN].as<uint2>(); uint32_t* heads = B[XB_BHEAD].as<uint32_t>();
    yd_scatter_kernel<<<tb_grid_for(nwarps * 32, 128), 128, 0, st>>>(grp.bits, W, k, G, gstrand, gstart, gend, cy.in ? gseed : nullptr, blkoff, blkkey, nblk,
                                                                     mem);
    ctx->launches++;
    // ---- Y5: sub-chain heads ----
    TB_CUDA((tb_device_scan<OpSumU32>(ctx, HeadIn{mem}, n_members, B[XB_AGG].as<uint32_t>(), HeadOut{heads, n_members, work})));
    if (parallel) {
      yd_compact_kernel<<<tb_grid_for(G, 256), 256, 0, st>>>(desc, G, U, rankpre, ubase, cdesc);
      ctx->launches++;
    }
    if (parallel) {
      // ---- Y6-Y9 ----
      TB_CUDA(B[XB_YDKEPT].ensure(sizeof(int32_t) * (size_t)n_members + 128));
      TB_CUDA(B[XB_YDBM].ensure(sizeof(uint64_t) * (size_t)nwords + 64));
      TB_CUDA(B[XB_YDLZ].ensure(sizeof(int64_t) * (size_t)nblocks512 + 64));
      int32_t* mstart = B[XB_YDKEPT].as<int32_t>();
      unsigned long long* bm = B[XB_YDBM].as<unsigned long long>();
      long long* lz = B[XB_YDLZ].as<long long>();
      TB_CUDA(cudaMemsetAsync(bm, 0, sizeof(uint64_t) * (size_t)nwords, st));
      if (cy.in && cy.nin > 0) {
        yd_carry_links_kernel<<<tb_grid_for(cy.nin, 256), 256, 0, st>>>(cy.coff, cy.cs, cy.ce, cy.nin, nchains, ubase, U, rankpre, bm, lpad);
        ctx->launches++;
      }
      const uint32_t nunits = (uint32_t)((n_members + YD_UNIT - 1) / YD_UNIT);
      TB_CUDA(B[XB_YDUNIT].ensure(sizeof(uint32_t) * ((size_t)nunits + 2)));
      uint32_t* ustart = B[XB_YDUNIT].as<uint32_t>();
      yd_unit_kernel<<<tb_grid_for((int64_t)nunits + 1, 256), 256, 0, st>>>(heads, work + 1, (uint32_t)n_members, nunits, ustart);
      (seed || cy.out ? yd_frontier_kernel<true> : yd_frontier_kernel<false>)<<<(unsigned)ctx->sm_count * 16, YD_FWARPS * 32, 0, st>>>(in, cdesc, grp.rep, mem, ustart, nunits, work, U, rankpre, bm, lpad, mstart,
                                                                                  seed, cy.out ? cy.efin : nullptr, (uint32_t)n_members);
      ctx->launches++;
      ctx->launches += 2;
      TB_CUDA((tb_device_scan<OpMaxI64>(ctx, LastZeroIn{bm}, nblocks512, B[XB_AGG].as<long long>(), LastZeroOut{lz})));
      yd_lookup_kernel<<<tb_grid_for(n_members, 256), 256, 0, st>>>(mstart, mem, n_members, bm, lz, lpad, ydc, cy.in ? cy.ext : nullptr);
      ctx->launches++;
      pout = YdParOut{bm, lz, lpad, U, rankpre, nuw, ubase, (int64_t)cy.bout - ubase, cy.ext, cy.efin};
      if (cy.out && !cy.in) TB_CUDA(cudaMemsetAsync(cy.ext, 0, sizeof(int32_t) * (size_t)nchains, st));
    } else {
      YdSeqCarry ca{cy.in ? cy.coff : nullptr, cy.cs, cy.ce, colbase, mem, nchains, ubase, cy.bout, cy.out ? cy.os : nullptr, cy.oe, cy.cap, cy.ometa};
      const size_t smem = (size_t)YD_WARPS * 2 * YD_CAP_SMEM * 32 * sizeof(uint32_t);
      const bool carry = cy.in || cy.out;
      auto chain_smem = carry ? yd_chain_kernel<true, true> : yd_chain_kernel<true, false>;
      TB_CUDA(cudaFuncSetAttribute(chain_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      chain_smem<<<(unsigned)ctx->sm_count * 4, YD_WARPS * 32, smem, st>>>(in, desc, grp.rep, mem, heads, work, ydc, nullptr, g.d_status, ca);
      ctx->launches++;
      TB_CUDA(cudaMemcpyAsync(h_status, g.d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
      TB_CUDA(cudaStreamSynchronize(st));
      if (h_status[CS_YD_OVERFLOW]) {
        // a list outgrew shared memory (its later distances are wrong): repeat everything with lists in global memory
        const unsigned grid2 = (unsigned)ctx->sm_count;
        TB_CUDA(B[XB_YDSCRATCH].ensure((size_t)grid2 * YD_WARPS * 2 * YD_CAP_GLOBAL * 32 * sizeof(uint32_t)));
        TB_CUDA(cudaMemsetAsync(ydc, 0, sizeof(int32_t) * (size_t)G, st));
        TB_CUDA(cudaMemsetAsync(work, 0, sizeof(unsigned long long), st));
        TB_CUDA(cudaMemsetAsync(g.d_status + CS_YD_OVERFLOW, 0, sizeof(long long), st));
        if (cy.out) TB_CUDA(cudaMemsetAsync(cy.ometa + 2 * nchains, 0, sizeof(long long), st));
        (carry ? yd_chain_kernel<false, true> : yd_chain_kernel<false, false>)<<<grid2, YD_WARPS * 32, 0, st>>>(in, desc, grp.rep, mem, heads, work, ydc, B[XB_YDSCRATCH].as<uint32_t>(), g.d_status, ca);
        ctx->launches++;
        TB_CUDA(cudaMemcpyAsync(h_status, g.d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaStreamSynchronize(st));
        if (h_status[CS_YD_OVERFLOW]) { ctx->set_error("tb_collapse_window: YD segment list exceeded %d live nodes", YD_CAP_GLOBAL); return 1; }
      }
    }
  }
  if (cy.out) {
    yd_carry_out_kernel<<<tb_grid_for(nchains, 128), 128, 0, st>>>(nchains, colbase, cy.in ? cy.coff : nullptr, cy.cs, cy.ce, cy.bout, parallel && n_members > 0,
                                                                   pout, cy.os, cy.oe, cy.cap, cy.ometa);
    ctx->launches++;
  }
  yd_combine_kernel<<<tb_grid_for(G, 256), 256, 0, st>>>(grp.yd, ydc, G);
  ctx->launches++;
  if (n_members > 0) {   // sub-chain count for tb_last_yd_stat
    TB_CUDA(cudaMemcpyAsync(h_status + 17, work + 1, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    ctx->last_yd_stat[1] = h_status[17];
  }
  return 0;
}
