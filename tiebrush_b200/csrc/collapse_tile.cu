// collapse_tile.cu — fast front end of the collapse: position-partitioned shared-memory hash tiles.
//
// Used when grouping is order independent (no -F, no -A, no TieBrush-made inputs, no --store-frac): then the
// reference's per-position sorted list (src/tiebrush.cpp:438-499) is simply the set of distinct keys in key order,
// YC is a count, YX a distinct-sample count and the representative is the first member in merge order
// (src/tmerge.h:28-50; closed form: min over members of (E, fidx, index-in-file), SURVEY §9.2).
//
//   slots      slot m = the start positions whose first merged rank P[p] lies in [mT,(m+1)T). Only the LAST position of a
//              slot can hold >= T records, so a slot is < T records of ordinary positions plus, possibly, one pile-up
//              position that is processed as a second sub-tile in "single position" mode.
//   table      every start position owns a private open-addressing region of the shared-memory table, placed at
//              floor(1.25 * (P[p]-rank0)) and sized >= its record count: regions are laid out in position order, a group
//              can never overflow its region (groups <= records), and the final order needs sorting only INSIDE a position.
//   streaming  persistent CTAs pull slots; each warp owns a contiguous range of the slot's file-major record list
//              (k slices, located by the per-(slot,file) offsets), so loads are coalesced and the per-file running
//              maximum of `end` that defines the merge order is a warp-local segmented scan with a register carry.
//              A record probes its region: tag compare in shared memory, then its real key bytes against the owner's
//              (grouping never rests on the hash). Only the first record of a run of identical neighbours inside a
//              32-record warp step probes, for the whole run; these run heads are queued in registers and probe 32 at a
//              time. Heads of one file hitting one group are merged with match_any: one representative atomicMin and
//              one sample-bit atomicOr (both rarely), plus each head's count atomic.
//   epilogue   occupied entries are compacted in region (= position) order, ranked inside their position by
//              (strand, end, mode key) with the reference's comparator, and written to the staging arrays.
#include <limits.h>
#include "collapse_internal.cuh"

namespace {

constexpr unsigned long long EMPTY64 = ~0ULL;

struct TileParams {
  uint32_t T, M, ecap, W, cap_records, heavy_records;
  const uint32_t* P; const uint32_t* slotpos; const uint32_t* off;
  uint32_t* gcount; uint32_t* st_rep; float* st_yc; uint32_t* st_yx; uint32_t* st_bits;
  long long* status; unsigned int* slot_counter; uint64_t seed;
  uint32_t* heavy_list;        // launch 1: slots whose pile-up position overflowed this launch's table are appended here ...
  const uint32_t* slot_list;   // launch 2 (one CTA per SM, full-size table): ... and redone from this list
  uint32_t n_list;
};

// ---------------------------------------------------------------------------------------------------
// C3: first position of every slot: slotpos[m] = first p with P[p] >= m*T
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) col_slotpos_kernel(const uint32_t* __restrict__ P, uint32_t span, uint32_t T, uint32_t M, uint32_t* __restrict__ slotpos) {
  uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m > M) return;
  if (m == M) { slotpos[M] = span; return; }
  const unsigned long long target = (unsigned long long)m * T;  // < n = P[span]
  uint32_t lo = 0, hi = span;  // first p in [0,span] with P[p] >= target
  while (lo < hi) { uint32_t mid = lo + ((hi - lo) >> 1); if ((unsigned long long)P[mid] >= target) hi = mid; else lo = mid + 1; }
  slotpos[m] = lo;
}

// ---------------------------------------------------------------------------------------------------
// C4: off[m][f] = first record of run f that falls in a slot >= m
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) col_off_init_kernel(uint32_t* __restrict__ off, const long long* __restrict__ run_off, int k, uint64_t total) {
  uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= total) return;
  int f = (int)(x % (uint64_t)k);
  off[x] = (uint32_t)run_off[f + 1];
}

// A record whose position differs from its predecessor's moves its file's cursor into a later slot only when the two
// positions lie in different slots — one record in ~T/k — so the slots are compared first and the file is looked up
// (binary search over the k run offsets) only for those records and at the k-1 run boundaries. Run starts themselves are
// written by col_off_heads_kernel.
__global__ void __launch_bounds__(256) col_off_kernel(ColIn in, const long long* __restrict__ run_off, const uint32_t* __restrict__ P, uint32_t T,
                                                      uint32_t* __restrict__ off, long long* __restrict__ status) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= in.n || i == 0) return;
  const int32_t p = in.pos[i];
  const uint32_t rel = (uint32_t)(p - in.pos_lo);
  if (rel >= in.span) return;  // already reported by C1
  const int32_t pp = in.pos[i - 1];
  if (pp == p) return;
  int64_t sprev = 0, scur = 0;
  if (pp < p) {
    const uint32_t prel = (uint32_t)(pp - in.pos_lo);
    if (prel >= in.span) return;
    sprev = (int64_t)(P[prel] / T); scur = (int64_t)(P[rel] / T);
    if (scur <= sprev) return;                 // same slot: nothing moves
  }
  int lo = 0, hi = in.k;                       // run containing i: last f with run_off[f] <= i
  while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (run_off[mid] <= i) lo = mid; else hi = mid; }
  const int f = lo;
  if (i == run_off[f]) return;                 // a run start: col_off_heads_kernel
  if (pp > p) { status[CS_ERR] = ERR_UNSORTED; atomicMin((unsigned long long*)&status[CS_ERRIDX], (unsigned long long)i); return; }
  for (int64_t s = sprev + 1; s <= scur; ++s) off[(uint64_t)s * in.k + f] = (uint32_t)i;
}

// a record that starts its run but has the same position as the last record of the previous run was skipped above
__global__ void __launch_bounds__(128) col_off_heads_kernel(ColIn in, const long long* __restrict__ run_off, const uint32_t* __restrict__ P, uint32_t T,
                                                            uint32_t* __restrict__ off) {
  int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= in.k) return;
  const int64_t i = run_off[f];
  if (i >= run_off[f + 1]) return;
  const uint32_t rel = (uint32_t)(in.pos[i] - in.pos_lo);
  if (rel >= in.span) return;
  const int64_t scur = (int64_t)(P[rel] / T);
  for (int64_t s = 0; s <= scur; ++s) off[(uint64_t)s * in.k + f] = (uint32_t)i;
}

// ---------------------------------------------------------------------------------------------------
// C5: the tile kernel
// ---------------------------------------------------------------------------------------------------
template <int THREADS>
struct TileSmem {
  unsigned long long* word;   // [E]  streaming: tag32<<32 | owner record ; epilogue: 64-bit sort key
  unsigned long long* rep;    // [E]  streaming: min over members of (E-pos)<<32 | record ; epilogue: owner<<32 | rep
  uint32_t* cnt;              // [E]
  uint32_t* bits;             // [E*W]
  uint32_t* a;                // [k]  slice begin of the current sub-tile
  uint32_t* b;                // [k]  slice end
  uint32_t* c;                // [k]  scratch (slot-level slice end while a pile-up sub-tile is split off)
  uint32_t* soff;             // [k+1] exclusive prefix of slice lengths
  uint16_t* rbase;            // [E]  region base of the entry's position (segment id in the epilogue)
  uint16_t* occ;              // [E]  compacted entry indices
  uint16_t* tmp;              // [E]  epilogue: rank inside the position (bits 0-12) | saturated key (14) | tied (15)
};

static size_t tile_smem_bytes(uint32_t k, uint32_t E, uint32_t W) {
  return (size_t)E * (8 + 8 + 4 + 4 * (size_t)W + 2 + 2 + 2) + (size_t)(6 * k + 1) * 4 + 64;
}

// 64-bit epilogue sort key: strand(2) | ref_len(30) | key length(8, saturated) | first key word, byte order of memcmp (24).
// It is a monotone prefix of the reference's order (strand, end, mode compare); ties are settled by tb_mode_cmp.
__device__ unsigned long long tile_sort_key(const ColIn& in, uint32_t o, unsigned sc) {
  const uint32_t c0 = in.cig_off[o], c1 = in.cig_off[o + 1];
  const int pos = in.pos[o];
  uint32_t reflen, len8, w24;
  if (in.mode == TB_MODE_EXON) {
    ExonIter it; it.init(in.cigar, c0, c1, pos);
    int s, e, nex = 0, e0 = 0;
    while (it.next(s, e)) { if (nex == 0) e0 = e; ++nex; }
    reflen = (uint32_t)it.l;
    len8 = nex > 255 ? 255u : (uint32_t)nex;
    uint32_t d = (uint32_t)(e0 - pos);               // first exon end - pos (its start is pos+1 for every record of the position)
    w24 = d > 0xffffffu ? 0xffffffu : d;
  } else {
    reflen = (uint32_t)tb_ref_len(in.cigar, c0, c1);
    uint32_t a = c0, b = c1;
    if (in.mode == TB_MODE_CLIP) tb_clip_range(in.cigar, a, b);
    const uint32_t nc = b - a;
    len8 = nc > 255 ? 255u : nc;
    w24 = nc ? (__byte_perm(in.cigar[a], 0, 0x0123) >> 8) : 0u;
  }
  return ((unsigned long long)sc << 62) | ((unsigned long long)(reflen & 0x3fffffffu) << 32) | ((unsigned long long)len8 << 24) | w24;
}

// Bytes [off, off+6) of the comparison string that FOLLOWS the 64-bit sort key, big-endian in the low 48 bits (zero beyond
// its end). The string continues the reference's order exactly: default / -P / -L: the rest of the memcmp over the raw
// little-endian CIGAR words (byte 3 of the first word onwards; equal n_cigar is part of the key), then for -L the MD tag as
// one presence byte (absent < present, cmpFull :298-302) and its characters (strcmp); -E: the exon coordinates as big-endian
// integers (first exon end, then start,end of every later exon; equal exon count is part of the key).
__device__ __noinline__ unsigned long long tile_tail_chunk(const ColIn& in, uint32_t o, uint32_t off) {
  const uint32_t c0 = in.cig_off[o], c1 = in.cig_off[o + 1];
  unsigned long long v = 0;
  if (in.mode == TB_MODE_EXON) {
    const uint32_t first = off >> 2, last = (off + 5) >> 2;   // integers of the stream touched by the chunk: first..last (<= first+2)
    uint32_t vals[3] = {0u, 0u, 0u};
    ExonIter it; it.init(in.cigar, c0, c1, in.pos[o]);
    int sx, ex; uint32_t j = 0;
    while (it.next(sx, ex)) {   // exon j holds stream integers 2j-1 (start, j > 0) and 2j (end)
      if (j > 0 && 2 * j - 1 >= first && 2 * j - 1 <= first + 2) vals[2 * j - 1 - first] = (uint32_t)sx;
      if (2 * j >= first && 2 * j <= first + 2) vals[2 * j - first] = (uint32_t)ex;
      if (2 * j >= last) break;
      ++j;
    }
#pragma unroll
    for (uint32_t bi = 0; bi < 6; ++bi) {
      const uint32_t t = off + bi;
      v = (v << 8) | ((vals[(t >> 2) - first] >> ((3u - (t & 3u)) * 8u)) & 0xffu);
    }
    return v;
  }
  uint32_t a = c0, b = c1;
  if (in.mode == TB_MODE_CLIP) tb_clip_range(in.cigar, a, b);
  const uint32_t nc = b - a, ncb = nc ? 4u * nc - 3u : 0u;   // CIGAR bytes after the three the sort key holds
  uint32_t m0 = 0, m1 = 0;
  if (in.mode == TB_MODE_FULL) { m0 = in.md_off[o]; m1 = in.md_off[o + 1]; }
  for (uint32_t bi = 0; bi < 6; ++bi) {
    const uint32_t t = off + bi;
    uint32_t byte = 0;
    if (t < ncb) { const uint32_t g = t + 3u; byte = (in.cigar[a + (g >> 2)] >> ((g & 3u) * 8u)) & 0xffu; }
    else if (in.mode == TB_MODE_FULL && m1 > m0) {
      const uint32_t u = t - ncb;
      if (u == 0) byte = 1u;
      else if (m0 + u - 1u < m1) byte = in.md[m0 + u - 1u];
    }
    v = (v << 8) | byte;
  }
  return v;
}

// is record i (own CIGAR range [c0,c1)) the same alignment as the table owner o? Same position by construction, same
// strand by the tag. Identical raw CIGARs decide every mode but -L at once (identical CIGAR at one position => identical
// clipped CIGAR and identical exon chain); -L then compares the MD bytes inline. Only records whose raw CIGARs differ
// (or whose MD lengths differ) go through the general comparator, which is exact for every mode.
// The inline part: identical raw CIGAR words [c0,c1) vs [o0,o1) and, in -L, identical MD bytes. True is exact for every
// mode; false only means "not decided here".
__device__ __forceinline__ bool tile_same_raw(const ColIn& in, uint32_t i, uint32_t c0, uint32_t c1, uint32_t o, uint32_t o0, uint32_t o1) {
  const uint32_t nc = c1 - c0;
  bool same_cigar = (o1 - o0 == nc);
  if (same_cigar)
    for (uint32_t q = 0; q < nc; ++q) if (in.cigar[c0 + q] != in.cigar[o0 + q]) { same_cigar = false; break; }
  if (!same_cigar) return false;
  if (in.mode != TB_MODE_FULL) return true;
  const uint32_t ma = in.md_off[i], na = in.md_off[i + 1] - ma, mb = in.md_off[o], nb = in.md_off[o + 1] - mb;
  if (na != nb) return false;
  for (uint32_t q = 0; q < na; ++q) if (in.md[ma + q] != in.md[mb + q]) return false;
  return true;
}

__device__ __forceinline__ bool tile_same_key(const ColIn& in, uint32_t i, uint32_t c0, uint32_t c1, uint32_t o) {
  if (tile_same_raw(in, i, c0, c1, o, in.cig_off[o], in.cig_off[o + 1])) return true;
  if (in.mode == TB_MODE_CIGAR) return false;
  return tb_mode_cmp(in, i, o) == 0;
}

// MODE >= 0 fixes the merge strategy at compile time (the default CIGAR mode gets its own instantiation: every mode branch
// of the record parser / verifier / sort key folds away); MODE < 0 reads it from the window descriptor.
template <int THREADS, int MODE>
__device__ uint32_t tile_process(const ColIn& in_, const TileParams& tp, TileSmem<THREADS>& sm, uint32_t n_sub, uint32_t rankbase, bool single,
                                 uint64_t outbase, uint32_t* s_scan,
                                 volatile uint32_t* s_flags /*[0]=kept [1]=overflow [2]=ngroups; whole launch: [4]=records [5]=heads [6]=batches*/) {
  constexpr int NW = THREADS / 32;
  ColIn in = in_;
  if (MODE >= 0) in.mode = MODE;
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t E = tp.ecap, W = tp.W, k = (uint32_t)in.k;
  // ---- exclusive prefix of the slice lengths ----
  {
    uint32_t carry = 0;
    for (uint32_t base = 0; base < k; base += THREADS) {
      const uint32_t f = base + tid;
      const uint32_t c = f < k ? sm.b[f] - sm.a[f] : 0u;
      uint32_t tot;
      const uint32_t exc = tb_block_exscan<OpSumU32>(c, s_scan, &tot);
      if (f < k) sm.soff[f] = carry + exc;
      carry += tot;
    }
    if (tid == 0) sm.soff[k] = carry;
  }
  uint32_t E_used = single ? E : ((5u * n_sub) >> 2) + 1u;
  if (E_used > E) E_used = E;
  for (uint32_t s = tid; s < E_used; s += THREADS) { sm.word[s] = EMPTY64; sm.rep[s] = EMPTY64; sm.cnt[s] = 0; }
  {  // bitsets: 16-byte stores (the array starts 16-byte aligned: E is a multiple of 64)
    uint4* b4 = reinterpret_cast<uint4*>(sm.bits);
    const uint32_t n4 = (E_used * W + 3) >> 2;
    for (uint32_t s = tid; s < n4; s += THREADS) b4[s] = make_uint4(0u, 0u, 0u, 0u);
  }
  if (tid == 0) { s_flags[0] = 0; s_flags[1] = 0; s_flags[2] = 0; }
  __syncthreads();

  // ---- stream this warp's contiguous range of the file-major record list ----
  const uint32_t j0 = (uint32_t)(((unsigned long long)n_sub * warp) / NW), j1 = (uint32_t)(((unsigned long long)n_sub * (warp + 1)) / NW);
  uint32_t carry_f = 0xffffffffu; int carry_pos = INT_MIN; int carry_max = 0;
  uint32_t my_kept = 0;
  uint32_t f_lo = 0;   // file of the first record of the next step (warp-uniform)
  if (j0 < j1) {
    uint32_t lo = 0, hi = k;
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (sm.soff[mid] <= j0) lo = mid; else hi = mid; }
    f_lo = lo;
    // look-back: if the range starts inside a (file,position) run, the running maximum of the part before it is needed
    if (j0 > sm.soff[f_lo]) {
      const uint32_t slo = sm.a[f_lo];
      const uint32_t i0 = slo + (j0 - sm.soff[f_lo]);
      const int p = in.pos[i0];
      if (in.pos[i0 - 1] == p) {
        int mx = 0;
        for (uint32_t top = i0; top > slo;) {
          const bool ok = lane < top - slo;
          const uint32_t idx = ok ? top - 1 - lane : slo;
          const bool same = ok && in.pos[idx] == p;
          const int rl = same ? tb_ref_len(in.cigar, in.cig_off[idx], in.cig_off[idx + 1]) : 0;
          const unsigned notsame = __ballot_sync(0xffffffffu, !same);
          const unsigned first = notsame ? (unsigned)(__ffs(notsame) - 1) : 32u;
          if (lane < first) mx = max(mx, rl);
          if (first < 32u) break;
          top -= 32;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, d));
        carry_f = f_lo; carry_pos = p; carry_max = mx;
      }
    }
  }
  // Runs of identical neighbours: a passing record that is the same alignment as the record in the lane before it (same
  // file, hence record i-1; same position, strand, tag and raw CIGAR words, and in -L the same MD bytes) is a member
  // of that lane's run; it neither probes nor merges. The run's first record, its head, carries the weight 1 + members,
  // and keeps its own (E, index), the smallest of the run (the running maximum E is non-decreasing along it). Runs end at
  // a warp step, so lane 0 is always a head. Heads queue in registers (lane q holds queue entry q) until 32 are pending
  // and then probe the table as one full warp; the rest is flushed by extra steps past the range's end.
  const uint32_t glimit = E - (E >> 3);
  uint32_t q_i = 0, q_tag = 0, q_rel = 0, q_fw = 0; int q_E = 0;   // this lane's queue entry
  uint32_t npend = 0;                                                           // queued heads (warp-uniform)
  uint32_t n_heads = 0, n_batches = 0;                                          // statistics (warp-uniform)
  uint32_t jb = j0;
  for (; jb < j1 || npend; jb += 32) {
    if (single && s_flags[2] > glimit) { s_flags[1] = 1; break; }   // warp-uniform (broadcast read)
    const uint32_t j = jb + lane;
    const bool valid = j < j1;
    uint32_t f = 0xfffffffeu, i = 0, c0 = 0, c1 = 0, h1 = 0; int pos = INT_MIN + 1 + (int)lane, reflen = 0; bool pass = false; unsigned sc = 0;
    if (valid) {
      f = f_lo;                                   // slices are contiguous in j: walk forward from the step's first file
      while (sm.soff[f + 1] <= j) ++f;
      i = sm.a[f] + (j - sm.soff[f]);
      pos = in.pos[i];
      c0 = in.cig_off[i]; c1 = in.cig_off[i + 1];
      const uint16_t fl = in.flag[i]; const uint8_t mq = in.mapq[i]; const uint16_t nh = in.nh[i];
      sc = tb_strand_code(in.strand[i]);
      pass = tb_passes_options(in, fl, mq, nh);
    }
    // parse: reference length and key hash. Outside -E the CIGAR walk is one warp-uniform loop, so every word is compared
    // with the same word of the previous lane's record on the way (same_words: the raw CIGARs are identical).
    const uint32_t nc = c1 - c0;
    bool same_words = __shfl_up_sync(0xffffffffu, nc, 1) == nc;
    if (in.mode == TB_MODE_EXON) {
      uint32_t h2;
      if (valid) tb_parse_record32(in, i, pos, c0, c1, reflen, h1, h2);
    } else {
      uint32_t a = c0, b = c1;
      if (in.mode == TB_MODE_CLIP && valid) tb_clip_range(in.cigar, a, b);
      h1 = 0x9876543u ^ (b - a);
      const uint32_t nmax = __reduce_max_sync(0xffffffffu, nc);
      for (uint32_t q = 0; q < nmax; ++q) {
        const uint32_t c = c0 + q;
        const uint32_t w = q < nc ? in.cigar[c] : 0u;
        same_words &= __shfl_up_sync(0xffffffffu, w, 1) == w;
        if (q < nc && tb_op_ref(w & 0xf)) reflen += (int)(w >> 4);
        if (c >= a && c < b) { h1 = (h1 ^ w) * 0x9E3779B1u; h1 ^= h1 >> 15; }
      }
      if (in.mode == TB_MODE_FULL && valid) {   // the MD tag, as tb_parse_record32 folds it
        const uint32_t m0 = in.md_off[i], m1 = in.md_off[i + 1];
        h1 = (h1 ^ (uint32_t)(m1 > m0)) * 0x9E3779B1u; h1 ^= h1 >> 15;
        uint32_t acc = 0, nb = 0;
        for (uint32_t q = m0; q < m1; ++q) {
          const uint32_t ch = in.md[q];
          if (ch == 0) break;
          acc = (acc << 8) | ch;
          if (++nb == 4) { h1 = (h1 ^ acc) * 0x9E3779B1u; h1 ^= h1 >> 15; acc = 0; nb = 0; }
        }
        h1 = (h1 ^ (acc ^ (nb << 29))) * 0x9E3779B1u; h1 ^= h1 >> 15;
      }
    }
    // segmented inclusive max-scan of ref_len over (file,position) runs == the running max that orders the reference's
    // priority queue (SURVEY §9.2); records the filters drop still take part (they delay the records behind them)
    uint32_t f_prev = __shfl_up_sync(0xffffffffu, f, 1); int pos_prev = __shfl_up_sync(0xffffffffu, pos, 1);
    if (lane == 0) { f_prev = carry_f; pos_prev = carry_pos; }
    int h = (!valid || f != f_prev || pos != pos_prev) ? 1 : 0;
    int v = valid ? reflen : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v2 = __shfl_up_sync(0xffffffffu, v, d), h2s = __shfl_up_sync(0xffffffffu, h, d);
      if ((int)lane >= d) { if (!h) v = max(v, v2); h |= h2s; }
    }
    if (!h) v = max(v, carry_max);
    const int Erel = v;
    carry_f = __shfl_sync(0xffffffffu, f, 31); carry_pos = __shfl_sync(0xffffffffu, pos, 31); carry_max = __shfl_sync(0xffffffffu, Erel, 31);
    f_lo = carry_f;   // only meaningful while lane 31 is valid, i.e. while another step follows

    // ---- run detection: slot-independent hash of the key, compared with the previous lane's as a pre-filter ----
    const uint32_t tag = (sc << 30) | (tb_mix32(h1 ^ ((uint32_t)reflen * 0x9E3779B1u) ^ (uint32_t)tp.seed) >> 2);
    const unsigned passm = __ballot_sync(0xffffffffu, pass);
    my_kept += pass;
    const uint32_t tag_u = __shfl_up_sync(0xffffffffu, tag, 1), c0_u = __shfl_up_sync(0xffffffffu, c0, 1);
    bool member = pass && lane > 0 && ((passm >> (lane - 1)) & 1u) && f == f_prev && pos == pos_prev && tag == tag_u && same_words;
    if (member && in.mode == TB_MODE_EXON)   // the walk above did not compare; record i-1's words end where record i's begin
      member = tile_same_raw(in, i, c0, c1, i - 1, c0_u, c0);
    if (member && in.mode == TB_MODE_FULL) {   // -L: the MD bytes as well (record i-1's end where record i's begin)
      const uint32_t ma = in.md_off[i], na = in.md_off[i + 1] - ma, mb = in.md_off[i - 1];
      if (ma - mb != na) member = false;
      for (uint32_t q = 0; member && q < na; ++q) member = in.md[ma + q] == in.md[mb + q];
    }
    const unsigned memm = __ballot_sync(0xffffffffu, member);
    const unsigned headm = passm & ~memm;
    const uint32_t nh = __popc(headm);
    // ---- append the heads to the queue: lane q takes the head of rank (q - npend) mod 32 ----
    const uint32_t r = (lane - npend) & 31u;
    uint32_t src = 0;   // lane of the r-th set bit of headm (r < nh)
#pragma unroll
    for (uint32_t w = 16; w; w >>= 1)
      if ((uint32_t)__popc(headm & ((1u << (src + w)) - 1u)) <= r) src += w;
    const uint32_t weight = __ffsll(~((unsigned long long)memm >> (lane + 1)));   // 1 + the members that follow
    const uint32_t g_i = __shfl_sync(0xffffffffu, i, src), g_tag = __shfl_sync(0xffffffffu, tag, src);
    const uint32_t g_rel = __shfl_sync(0xffffffffu, (uint32_t)(pos - in.pos_lo), src), g_fw = __shfl_sync(0xffffffffu, f | (weight << 26), src);
    const int g_E = __shfl_sync(0xffffffffu, Erel, src);
    if (lane >= npend) { q_i = g_i; q_tag = g_tag; q_rel = g_rel; q_fw = g_fw; q_E = g_E; }
    const uint32_t tot = npend + nh;
    if (tot == 0 || (tot < 32 && jb + 32 < j1)) { npend = tot; continue; }   // warp-uniform: not full, and more records follow

    // ---- probe the queued heads as one warp (all 32 lanes unless this is the range's last batch) ----
    const bool live = lane < tot;
    const uint32_t qf = q_fw & 0x3ffffffu;
    n_heads += tot < 32 ? tot : 32u; n_batches += tot >= 32;
    uint32_t s = 0;
    bool placed = false;
    if (live) {
      uint32_t base = 0, size = E;
      if (!single) {
        const uint32_t Pa = tp.P[q_rel] - rankbase, Pb = tp.P[q_rel + 1] - rankbase;
        base = (5u * Pa) >> 2; size = ((5u * Pb) >> 2) - base;
      }
      s = base + __umulhi(q_tag << 2, size);   // the tag's 30 hash bits also pick the first entry
      const unsigned long long mine = ((unsigned long long)q_tag << 32) | q_i;
      for (uint32_t t = 0; t < size; ++t) {
        unsigned long long w = sm.word[s];
        if (w == EMPTY64) {
          w = atomicCAS(&sm.word[s], EMPTY64, mine);
          if (w == EMPTY64) { sm.rbase[s] = (uint16_t)base; atomicAdd((uint32_t*)&s_flags[2], 1u); placed = true; break; }
        }
        if ((uint32_t)(w >> 32) == q_tag) {
          const uint32_t o = (uint32_t)w;  // owner: compare the real keys
          if (o == q_i || tile_same_key(in, q_i, in.cig_off[q_i], in.cig_off[q_i + 1], o)) { placed = true; break; }
        }
        if (++s == base + size) s = base;
      }
      if (!placed) s_flags[1] = 1;
    }
    // merge the heads of one file that hit one group: queue order is stream order, so the lowest lane has the smallest
    // (E, index) of them. Each head adds its own weight to the count (a warp reduction over the match_any groups would
    // run once per distinct group mask).
    const uint32_t mkey = placed ? (s | (qf << 13)) : (0x80000000u | lane);
    const unsigned peers = __match_any_sync(0xffffffffu, mkey);
    if (placed) atomicAdd(&sm.cnt[s], q_fw >> 26);
    if (placed && (int)lane == __ffs(peers) - 1) {
      const unsigned long long repkey = ((unsigned long long)(uint32_t)q_E << 32) | q_i;
      if (repkey < sm.rep[s]) atomicMin(&sm.rep[s], repkey);
      const uint32_t bi = s * W + (qf >> 5), bit = 1u << (qf & 31);
      if (!(sm.bits[bi] & bit)) atomicOr(&sm.bits[bi], bit);
    }
    // heads beyond the batch stay queued: lane q < tot - 32 took rank q + 32 - npend, exactly the first of them
    q_i = g_i; q_tag = g_tag; q_rel = g_rel; q_fw = g_fw; q_E = g_E;
    npend = tot > 32 ? tot - 32 : 0u;
  }
  if (lane == 0) {
    atomicAdd((uint32_t*)&s_flags[4], min(jb, j1) - j0);
    atomicAdd((uint32_t*)&s_flags[5], n_heads);
    atomicAdd((uint32_t*)&s_flags[6], n_batches);
  }
  if (my_kept) atomicAdd((uint32_t*)&s_flags[0], my_kept);
  __syncthreads();
  if (s_flags[1]) return 0xffffffffu;   // block-uniform: table overflow (single-position mode only)

  // ---- epilogue A: compact the occupied entries in region (= position) order. Each warp owns a contiguous chunk of the
  // table: ballot counts, one block-wide scan of the NW warp totals, ballot ranks (two barriers per sub-tile) ----
  uint32_t G = 0;
  {
    const uint32_t chunk = (((E_used + NW - 1) / NW) + 31u) & ~31u;
    const uint32_t e0 = warp * chunk, e1 = min(E_used, e0 + chunk);
    uint32_t mine = 0;
    for (uint32_t eb = e0; eb < e1; eb += 32) {
      const uint32_t e = eb + lane;
      mine += __popc(__ballot_sync(0xffffffffu, e < e1 && sm.word[e] != EMPTY64));
    }
    uint32_t tot;
    uint32_t base = tb_block_exscan<OpSumU32>(lane == 0 ? mine : 0u, s_scan, &tot);   // lane 0 of warp w: entries before the warp's chunk
    base = __shfl_sync(0xffffffffu, base, 0);
    for (uint32_t eb = e0; eb < e1; eb += 32) {
      const uint32_t e = eb + lane;
      const bool occf = e < e1 && sm.word[e] != EMPTY64;
      const unsigned bal = __ballot_sync(0xffffffffu, occf);
      if (occf) sm.occ[base + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)e;
      base += __popc(bal);
    }
    G = tot;
  }
  __syncthreads();
  // ---- epilogue B: sort keys ----
  for (uint32_t r = tid; r < G; r += THREADS) {
    const uint32_t e = sm.occ[r];
    const unsigned long long w = sm.word[e];
    const uint32_t o = (uint32_t)w; const unsigned sc = (unsigned)(w >> 62);
    sm.word[e] = tile_sort_key(in, o, sc);
    sm.rep[e] = ((unsigned long long)o << 32) | (uint32_t)sm.rep[e];
  }
  __syncthreads();
  // ---- epilogue C: rank inside the position. Ranks come from the 64-bit keys in shared memory; groups whose keys tie are
  // refined by re-keying with (rank so far, next 6 bytes of the comparison string) — one global read per tied group and
  // round instead of one comparator call per tied PAIR (a pile-up position in -L mode holds hundreds of groups that differ
  // only in MD) — and only what still ties after TILE_REFINE rounds goes through the general comparator ----
  constexpr int TILE_REFINE = 6;
  for (int round = 0;; ++round) {
    int any_tie = 0;
    for (uint32_t r = tid; r < G; r += THREADS) {
      const uint32_t e = sm.occ[r];
      const uint16_t rb = sm.rbase[e];
      const unsigned long long ki = sm.word[e];
      uint32_t rank = 0, ties = 0;
      if (single) {   // one position: every entry is compared, with no region test
#pragma unroll 4
        for (uint32_t q = 0; q < G; ++q) {
          const unsigned long long kq = sm.word[sm.occ[q]];
          rank += kq < ki; ties += kq == ki;
        }
        --ties;   // the entry itself
      } else {        // the entries of the position: the neighbours with the same region base
        for (uint32_t q = r; q > 0;) {
          const uint32_t eq = sm.occ[--q];
          if (sm.rbase[eq] != rb) break;
          const unsigned long long kq = sm.word[eq];
          rank += kq < ki; ties += kq == ki;
        }
        for (uint32_t q = r + 1; q < G; ++q) {
          const uint32_t eq = sm.occ[q];
          if (sm.rbase[eq] != rb) break;
          const unsigned long long kq = sm.word[eq];
          rank += kq < ki; ties += kq == ki;
        }
      }
      uint16_t sat = round == 0 ? ((((uint32_t)(ki >> 24) & 0xffu) == 255u) ? 0x4000u : 0u) : (sm.tmp[e] & 0x4000u);
      sm.tmp[e] = (uint16_t)(rank | sat | (ties ? 0x8000u : 0u));
      any_tie |= (ties != 0 && !sat);
    }
    if (round >= TILE_REFINE || in.mode == TB_MODE_CIGAR) { __syncthreads(); break; }   // default mode: ties are rare, one round
    if (!__syncthreads_or(any_tie)) break;
    for (uint32_t r = tid; r < G; r += THREADS) {
      const uint32_t e = sm.occ[r];
      const uint32_t t = sm.tmp[e];
      unsigned long long chunk = 0;
      if ((t & 0xC000u) == 0x8000u) chunk = tile_tail_chunk(in, (uint32_t)(sm.rep[e] >> 32), (uint32_t)round * 6u);
      sm.word[e] = ((unsigned long long)(t & 0x1fffu) << 48) | chunk;
    }
    __syncthreads();
  }
  for (uint32_t r = tid; r < G; r += THREADS) {
    const uint32_t e = sm.occ[r];
    const uint16_t rb = sm.rbase[e];
    const uint32_t t = sm.tmp[e];
    const bool tied = (t & 0x8000u) != 0;
    uint32_t rank = t & 0x1fffu, a = (single && !tied) ? 0u : r;   // a: first entry of the position (0 in single mode)
    const unsigned long long ki = sm.word[e];
    const uint32_t oi = (uint32_t)(sm.rep[e] >> 32);
    while (a > 0) {
      const uint32_t eq = sm.occ[a - 1];
      if (!single && sm.rbase[eq] != rb) break;
      --a;
      if (tied && sm.word[eq] == ki && tb_mode_cmp(in, (uint32_t)(sm.rep[eq] >> 32), oi) < 0) ++rank;
    }
    if (tied)
      for (uint32_t q = r + 1; q < G; ++q) {
        const uint32_t eq = sm.occ[q];
        if (!single && sm.rbase[eq] != rb) break;
        if (sm.word[eq] == ki && tb_mode_cmp(in, (uint32_t)(sm.rep[eq] >> 32), oi) < 0) ++rank;
      }
    const uint64_t o = outbase + a + rank;
    tp.st_rep[o] = (uint32_t)sm.rep[e];
    tp.st_yc[o] = (float)sm.cnt[e];
    uint32_t yx = 0;
    for (uint32_t w = 0; w < W; ++w) { const uint32_t bw = sm.bits[e * W + w]; yx += __popc(bw); tp.st_bits[o * W + w] = bw; }
    tp.st_yx[o] = yx;
  }
  return G;
}

// slot descriptor handed from the prefetching thread to the block
struct SlotMeta { uint32_t m, rank0, rank1, p0, p1; };

template <int THREADS, int MODE>
__global__ void __launch_bounds__(THREADS, 1024 / THREADS) col_tile_kernel(ColIn in, TileParams tp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint32_t s_scan[33];
  __shared__ uint32_t s_flags[8];
  __shared__ SlotMeta s_meta[2];
  __shared__ uint32_t s_pbig;
  const uint32_t E = tp.ecap, W = tp.W, k = (uint32_t)in.k, tid = threadIdx.x;
  TileSmem<THREADS> sm;
  sm.word = (unsigned long long*)smem_raw;
  sm.rep = sm.word + E;
  sm.cnt = (uint32_t*)(sm.rep + E);
  sm.bits = sm.cnt + E;
  uint32_t* ab = sm.bits + (size_t)E * W;          // [2][2k] double-buffered slice bounds (next slot's are prefetched)
  sm.c = ab + 4 * (size_t)k;
  sm.soff = sm.c + k;
  sm.rbase = (uint16_t*)(sm.soff + k + 1);
  sm.occ = sm.rbase + E;
  sm.tmp = sm.occ + E;
  uint32_t kept_total = 0;   // thread 0 only
  auto fetch_meta = [&](SlotMeta& d) {   // one thread: claim the next slot and read its geometry
    SlotMeta t; t.m = atomicAdd(tp.slot_counter, 1u); t.rank0 = t.rank1 = t.p0 = t.p1 = 0;
    if (tp.slot_list) t.m = t.m < tp.n_list ? tp.slot_list[t.m] : tp.M;
    if (t.m < tp.M) { t.p0 = tp.slotpos[t.m]; t.p1 = tp.slotpos[t.m + 1]; t.rank0 = tp.P[t.p0]; t.rank1 = tp.P[t.p1]; }
    d = t;
  };
  auto load_bounds = [&](const SlotMeta& d, uint32_t* dst) {   // all threads: per-file slices of a slot
    if (d.m < tp.M) for (uint32_t f = tid; f < k; f += THREADS) { dst[f] = tp.off[(uint64_t)d.m * k + f]; dst[k + f] = tp.off[(uint64_t)(d.m + 1) * k + f]; }
  };
  if (tid == 0) { fetch_meta(s_meta[0]); fetch_meta(s_meta[1]); s_flags[4] = 0; s_flags[5] = 0; s_flags[6] = 0; }
  __syncthreads();
  load_bounds(s_meta[0], ab);
  for (uint32_t it = 0;; ++it) {
    __syncthreads();
    const SlotMeta cur = s_meta[it & 1], nxt = s_meta[(it + 1) & 1];
    if (cur.m >= tp.M) break;
    sm.a = ab + (size_t)(it & 1) * 2 * k; sm.b = sm.a + k;
    load_bounds(nxt, ab + (size_t)((it + 1) & 1) * 2 * k);   // overlaps with this slot's work
    __syncthreads();                                          // everybody has read s_meta[it&1]
    if (tid == THREADS - 1) fetch_meta(s_meta[it & 1]);       // slot it+2; its latency hides behind this slot
    const uint32_t m = cur.m, rank0 = cur.rank0, rank1 = cur.rank1, p0 = cur.p0, p1 = cur.p1;
    const uint32_t n_t = rank1 - rank0;
    if (n_t == 0) { if (tid == 0) tp.gcount[m] = 0; continue; }
    uint32_t G = 0, kept_slot = 0;   // kept_slot: thread 0 only
    bool overflow = false;
    if (n_t <= tp.cap_records) {
      G = tile_process<THREADS, MODE>(in, tp, sm, n_t, rank0, false, rank0, s_scan, s_flags);
      overflow = G == 0xffffffffu;
      if (tid == 0) kept_slot = s_flags[0];
    } else {
      // the last position of the slot is a pile-up: split it off
      if (tid == 0) {
        uint32_t lo = p0, hi = p1;  // last p in [p0,p1) with P[p] < rank1 (the last non-empty position)
        while (hi - lo > 1) { const uint32_t mid = lo + ((hi - lo) >> 1); if (tp.P[mid] < rank1) lo = mid; else hi = mid; }
        s_pbig = lo;
      }
      __syncthreads();
      const uint32_t pbig = s_pbig;
      const uint32_t rb = tp.P[pbig];
      // A very deep pile-up (tens of thousands of alignments at one start) almost always holds more distinct alignments than
      // this launch's small table: streaming it until the table overflows is wasted work. Send the slot straight to the
      // full-size launch (a performance shortcut only: that launch computes the same groups).
      if (tp.heavy_list && tp.heavy_records && rank1 - rb > tp.heavy_records) {   // block-uniform
        if (tid == 0) { tp.gcount[m] = 0; tp.heavy_list[atomicAdd((unsigned long long*)&tp.status[CS_NHEAVY], 1ULL)] = m; }
        continue;
      }
      const int big_pos = (int)pbig + in.pos_lo;
      for (uint32_t f = tid; f < k; f += THREADS) {  // first record of the slice at the pile-up position
        uint32_t lo = sm.a[f], hi = sm.b[f];
        while (lo < hi) { const uint32_t mid = lo + ((hi - lo) >> 1); if (in.pos[mid] >= big_pos) hi = mid; else lo = mid + 1; }
        sm.c[f] = sm.b[f]; sm.b[f] = lo;
      }
      __syncthreads();
      uint32_t G1 = 0;
      if (rb > rank0) {
        G1 = tile_process<THREADS, MODE>(in, tp, sm, rb - rank0, rank0, false, rank0, s_scan, s_flags);
        overflow = G1 == 0xffffffffu;
        if (tid == 0) kept_slot = s_flags[0];
      }
      if (!overflow) {
        __syncthreads();
        for (uint32_t f = tid; f < k; f += THREADS) { sm.a[f] = sm.b[f]; sm.b[f] = sm.c[f]; }
        __syncthreads();
        const uint32_t G2 = tile_process<THREADS, MODE>(in, tp, sm, rank1 - rb, rb, true, (uint64_t)rank0 + G1, s_scan, s_flags);
        overflow = G2 == 0xffffffffu;
        if (tid == 0) kept_slot += s_flags[0];
        G = G1 + G2;
      }
    }
    if (overflow) {   // block-uniform
      if (tid == 0) {
        tp.gcount[m] = 0;
        if (tp.heavy_list) tp.heavy_list[atomicAdd((unsigned long long*)&tp.status[CS_NHEAVY], 1ULL)] = m;   // redone by the full-size launch
        else tp.status[CS_TABLE_OVERFLOW] = 1;
      }
      continue;
    }
    if (tid == 0) kept_total += kept_slot;
    if (tid == 0) tp.gcount[m] = G;
  }
  if (tid == 0 && kept_total) atomicAdd((unsigned long long*)&tp.status[CS_NKEPT], (unsigned long long)kept_total);
  if (tid == 0 && s_flags[4]) {
    atomicAdd((unsigned long long*)&tp.status[CS_TILE_RECORDS], (unsigned long long)s_flags[4]);
    atomicAdd((unsigned long long*)&tp.status[CS_TILE_HEADS], (unsigned long long)s_flags[5]);
    atomicAdd((unsigned long long*)&tp.status[CS_TILE_BATCHES], (unsigned long long)s_flags[6]);
  }
}

// ---------------------------------------------------------------------------------------------------
// C6: compaction of the staged groups
// ---------------------------------------------------------------------------------------------------
struct GcIn { const uint32_t* c; __device__ uint32_t operator()(int64_t i) const { return c[i]; } };
struct GcOut { uint32_t* b; __device__ void operator()(int64_t i, uint32_t exc, uint32_t) const { b[i] = exc; } };

__global__ void __launch_bounds__(128) col_compact_kernel(TileParams tp, const uint32_t* __restrict__ gbase, uint32_t* __restrict__ o_rep,
                                                          float* __restrict__ o_yc, uint32_t* __restrict__ o_yx, int32_t* __restrict__ o_yd,
                                                          uint32_t* __restrict__ o_bits, int64_t capacity) {
  const uint32_t m = blockIdx.x;
  const uint32_t G = tp.gcount[m];
  if (G == 0) return;
  const uint64_t src = tp.P[tp.slotpos[m]];
  const uint64_t dst = gbase[m];
  for (uint32_t r = threadIdx.x; r < G; r += blockDim.x) {
    if ((int64_t)(dst + r) >= capacity) break;
    o_rep[dst + r] = tp.st_rep[src + r];
    o_yc[dst + r] = tp.st_yc[src + r];
    o_yx[dst + r] = tp.st_yx[src + r];
    o_yd[dst + r] = 0;
  }
  for (uint64_t x = threadIdx.x; x < (uint64_t)G * tp.W; x += blockDim.x) {
    if ((int64_t)(dst + x / tp.W) >= capacity) break;
    o_bits[dst * tp.W + x] = tp.st_bits[src * tp.W + x];
  }
}

__global__ void col_store_total_kernel(const uint32_t* tot, long long* status) { status[CS_NGROUPS] = *tot; }

}  // namespace

int col_front_tile(tb_ctx* ctx, const ColIn& in, const ColGeom& g, ColGroups& out, int64_t* n_groups, int64_t* n_kept) {
  cudaStream_t st = ctx->stream;
  DevBuf* B = ctx->buf;
  const int64_t n = g.n; const int k = g.k; const uint32_t W = g.W, S = g.S;
  // ---- geometry: CTAs of 256 threads, 4 of them per SM, each with a quarter of the opt-in shared memory for its table;
  // one 1024-thread CTA per SM when the 256-thread table does not fit k ----
  int threads = 256;
  const int ctas_per_sm = 1024 / threads;
  const size_t smem_sm = ctx->smem_optin ? ctx->smem_optin + 1024 : 233472;   // shared memory per SM (opt-in per block + 1 KB reserved)
  const size_t smem_limit = smem_sm / ctas_per_sm - 1024 - 512;               // per CTA: minus the reserved KB and the static part
  uint32_t E = 8192;   // region bases are u16 and the match key keeps 13 bits for the entry
  while (E > 64 && tile_smem_bytes((uint32_t)k, E, W) > smem_limit) E -= 64;
  if (tile_smem_bytes((uint32_t)k, E, W) > smem_limit) {
    threads = 1024;   // fall through to the single-CTA geometry below
    const size_t lim1 = smem_sm - 1024 - 512;
    E = 8192;
    while (E > 64 && tile_smem_bytes((uint32_t)k, E, W) > lim1) E -= 64;
    if (tile_smem_bytes((uint32_t)k, E, W) > lim1) { ctx->set_error("tb_collapse_window: %d samples do not fit the shared-memory group table", k); return 1; }
  }
  const uint32_t cap_records = (uint32_t)(((uint64_t)(E - 1) * 4) / 5);   // floor(1.25*n)+1 <= E
  // full-size table of the second launch (pile-up positions, slots the first launch deferred)
  const size_t lim_full = smem_sm - 1024 - 512;
  uint32_t E_full = 8192;
  while (E_full > 64 && tile_smem_bytes((uint32_t)k, E_full, W) > lim_full) E_full -= 64;
  const uint32_t cap_full = (uint32_t)(((uint64_t)(E_full - 1) * 4) / 5);
  // slot size: a slot holds < T records of ordinary positions plus its last position; a slot that outgrows the table
  // splits that last position off as a pile-up sub-tile (tile kernel), so any T <= cap_records is correct. Larger T =
  // fewer, fuller slots (less per-slot work), but more slots that need the split; 7/8 of the table.
  const uint32_t T = (uint32_t)(((uint64_t)cap_records * 7) / 8);
  if (T < 8) { ctx->set_error("tb_collapse_window: %d samples leave no room for a shared-memory tile", k); return 1; }
  const uint32_t M = (uint32_t)((n + T - 1) / T);
  ctx->last_tile_gen = 1;

  TB_CUDA(B[XB_SLOTPOS].ensure(sizeof(uint32_t) * ((size_t)M + 2)));
  TB_CUDA(B[XB_OFF].ensure(sizeof(uint32_t) * ((size_t)M + 1) * k));
  TB_CUDA(B[XB_GCOUNT].ensure(sizeof(uint32_t) * ((size_t)M + 2)));
  TB_CUDA(B[XB_GBASE].ensure(sizeof(uint32_t) * ((size_t)M + 2)));
  TB_CUDA(B[XB_ST_REP].ensure(sizeof(uint32_t) * n));
  TB_CUDA(B[XB_ST_YC].ensure(sizeof(float) * n));
  TB_CUDA(B[XB_ST_YX].ensure(sizeof(uint32_t) * n));
  TB_CUDA(B[XB_ST_BITS].ensure(sizeof(uint32_t) * (size_t)n * W));
  TB_CUDA(B[XB_WORK].ensure(256));
  TB_CUDA(B[XB_AGG].ensure((size_t)(tb_scan_blocks((int64_t)M + 2) + 8) * sizeof(uint64_t)));

  // ---- C3, C4 ----
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[5], st));
  col_slotpos_kernel<<<tb_grid_for((int64_t)M + 1, 256), 256, 0, st>>>(g.P, S, T, M, B[XB_SLOTPOS].as<uint32_t>());
  const uint64_t off_total = ((uint64_t)M + 1) * k;
  col_off_init_kernel<<<tb_grid_for((int64_t)off_total, 256), 256, 0, st>>>(B[XB_OFF].as<uint32_t>(), g.d_runoff, k, off_total);
  col_off_kernel<<<tb_grid_for(n, 256), 256, 0, st>>>(in, g.d_runoff, g.P, T, B[XB_OFF].as<uint32_t>(), g.d_status);
  col_off_heads_kernel<<<tb_grid_for(k, 128), 128, 0, st>>>(in, g.d_runoff, g.P, T, B[XB_OFF].as<uint32_t>());
  ctx->launches += 4;
  // ---- C5 ----
  TileParams tp; memset(&tp, 0, sizeof(tp));
  tp.T = T; tp.M = M; tp.ecap = E; tp.W = W; tp.cap_records = cap_records; tp.P = g.P; tp.slotpos = B[XB_SLOTPOS].as<uint32_t>(); tp.off = B[XB_OFF].as<uint32_t>();
  tp.gcount = B[XB_GCOUNT].as<uint32_t>(); tp.st_rep = B[XB_ST_REP].as<uint32_t>(); tp.st_yc = B[XB_ST_YC].as<float>();
  tp.st_yx = B[XB_ST_YX].as<uint32_t>(); tp.st_bits = B[XB_ST_BITS].as<uint32_t>(); tp.status = g.d_status; tp.seed = 0x243F6A8885A308D3ULL;
  tp.slot_counter = B[XB_WORK].as<unsigned int>();
  tp.heavy_records = 24u * E;
  auto launch = [&](int thr, const TileParams& t, unsigned nslots) -> cudaError_t {
    const size_t smem = tile_smem_bytes((uint32_t)k, t.ecap, W);
    const unsigned want = (unsigned)ctx->sm_count * (1024u / (unsigned)thr);
    const unsigned grid = nslots < want ? nslots : want;
    cudaError_t e = cudaMemsetAsync(t.slot_counter, 0, 64, st);
    if (e != cudaSuccess) return e;
#define TB_TILE_LAUNCH(T, M)                                                                                                     \
  do {                                                                                                                           \
    if ((e = cudaFuncSetAttribute(col_tile_kernel<T, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e; \
    col_tile_kernel<T, M><<<grid, T, smem, st>>>(in, t);                                                                        \
  } while (0)
    const bool dflt = in.mode == TB_MODE_CIGAR;
    if (thr == 1024) { if (dflt) TB_TILE_LAUNCH(1024, TB_MODE_CIGAR); else TB_TILE_LAUNCH(1024, -1); }
    else {   // the default geometry has one instantiation per merge strategy
      switch (in.mode) {
        case TB_MODE_CIGAR: TB_TILE_LAUNCH(256, TB_MODE_CIGAR); break;
        case TB_MODE_FULL: TB_TILE_LAUNCH(256, TB_MODE_FULL); break;
        case TB_MODE_CLIP: TB_TILE_LAUNCH(256, TB_MODE_CLIP); break;
        case TB_MODE_EXON: TB_TILE_LAUNCH(256, TB_MODE_EXON); break;
        default: TB_TILE_LAUNCH(256, -1); break;
      }
    }
#undef TB_TILE_LAUNCH
    ctx->launches++;
    return cudaGetLastError();
  };
  // launch 1: every slot, small position-partitioned tables, several CTAs per SM. Slots it cannot finish (a pile-up position
  // with more distinct alignments than the table holds) go to the heavy list; launch 2 redoes those slots with the
  // full-size table, one CTA per SM. With the single-CTA geometry launch 1 already has the full-size table.
  if (threads != 1024) {
    TB_CUDA(B[XB_HEAVY].ensure(sizeof(uint32_t) * ((size_t)M + 1)));
    tp.heavy_list = B[XB_HEAVY].as<uint32_t>();
  }
  long long* h_status = ctx->pinned[0].as<long long>();
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[0], st));
  TB_CUDA(launch(threads, tp, M));
  if (tp.heavy_list) {
    TB_CUDA(cudaMemcpyAsync(h_status, g.d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    const int64_t nheavy = h_status[CS_NHEAVY];
    ctx->last_heavy = nheavy;
    ctx->last_tile_slots = (int64_t)M;
    if (nheavy > 0 && !h_status[CS_TABLE_OVERFLOW]) {
      TileParams t2 = tp;
      t2.ecap = E_full; t2.cap_records = cap_full;
      t2.slot_list = tp.heavy_list; t2.n_list = (uint32_t)nheavy; t2.heavy_list = nullptr;
      TB_CUDA(launch(1024, t2, (unsigned)nheavy));
    }
  } else ctx->last_heavy = 0;
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[1], st));
  // ---- C6 ----
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[6], st));
  TB_CUDA((tb_device_scan<OpSumU32>(ctx, GcIn{tp.gcount}, (int64_t)M, B[XB_AGG].as<uint32_t>(), GcOut{B[XB_GBASE].as<uint32_t>()})));
  col_store_total_kernel<<<1, 1, 0, st>>>(B[XB_AGG].as<uint32_t>() + tb_scan_blocks(M), g.d_status);
  ctx->launches++;
  TB_CUDA(cudaMemcpyAsync(h_status, g.d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
  TB_CUDA(cudaStreamSynchronize(st));
  if (ctx->profiling) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]) == cudaSuccess) ctx->last_ms[0] = ms;
    if (cudaEventElapsedTime(&ms, ctx->ev[5], ctx->ev[0]) == cudaSuccess) ctx->last_ms[3] = ms;
    (void)cudaGetLastError();
  }
  for (int q = 0; q < 3; ++q) ctx->last_tile_runs[q] = h_status[CS_TILE_RECORDS + q];
  if (h_status[CS_ERR] == ERR_UNSORTED) { ctx->set_error("tb_collapse_window: run not coordinate-sorted at record %lld", h_status[CS_ERRIDX]); return 1; }
  if (h_status[CS_TABLE_OVERFLOW]) return 2;
  const int64_t G = h_status[CS_NGROUPS];
  *n_groups = G; *n_kept = h_status[CS_NKEPT];
  if (G > out.capacity) { ctx->set_error("tb_collapse_window: output capacity %lld < %lld groups", (long long)out.capacity, (long long)G); return 1; }
  if (G == 0) return 0;
  TB_CUDA(B[XB_BITS].ensure(sizeof(uint32_t) * (size_t)G * W));
  out.bits = B[XB_BITS].as<uint32_t>();
  col_compact_kernel<<<M, 128, 0, st>>>(tp, B[XB_GBASE].as<uint32_t>(), out.rep, out.yc, out.yx, out.yd, out.bits, G);
  ctx->launches++;
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[7], st));
  return 0;
}
