// tb_record.cuh — the reference's record model on the device, shared by every collapse kernel:
//   GSamRecord::setupCoordinates (src/GSam.cpp:351-417)  -> ExonIter / ref_len
//   passes_options (src/tiebrush.cpp:532-541)            -> passes_options
//   cmpFlags / cmpCigar / cmpFull / cmpCigarClip / cmpExons (src/tiebrush.cpp:275-345) -> mode_cmp(_flags)
#pragma once
#include "tb_common.cuh"

struct ColIn {
  int64_t n; int k; int mode; uint32_t flag_mask; int max_nh; int min_qual; int keep_bits; int collapse_same;
  const int32_t* pos; const uint16_t* flag; const uint8_t* mapq; const uint8_t* strand; const uint16_t* nh;
  const uint32_t* cig_off; const uint32_t* cigar; const uint32_t* md_off; const uint8_t* md;
  const uint64_t* qhash; const float* yc_in; const int32_t* yx_in; const int32_t* yd_in;
  int32_t pos_lo; uint32_t span;
};

// does this CIGAR op consume the reference? (M, D, N, =, X)
__device__ __forceinline__ bool tb_op_ref(uint32_t op) { return (0x18Du >> op) & 1u; }

__device__ __forceinline__ int tb_ref_len(const uint32_t* __restrict__ cigar, uint32_t c0, uint32_t c1) {
  int l = 0;
  for (uint32_t c = c0; c < c1; ++c) { uint32_t w = cigar[c]; if (tb_op_ref(w & 0xf)) l += (int)(w >> 4); }
  return l;
}

struct ExonIter {  // yields the exon chain of one record (1-based inclusive coordinates)
  const uint32_t* cig; uint32_t c, c1; int pos, l, exstart; bool intron, ins, done;
  __device__ void init(const uint32_t* cigar, uint32_t c0, uint32_t cend, int p) { cig = cigar; c = c0; c1 = cend; pos = p; l = 0; exstart = p; intron = ins = false; done = false; }
  __device__ bool next(int& s, int& e) {
    if (done) return false;
    while (c < c1) {
      uint32_t w = cig[c++]; uint32_t op = w & 0xf; int len = (int)(w >> 4);
      switch (op) {
        case TB_OP_M: case TB_OP_EQ: case TB_OP_X: case TB_OP_D: l += len; intron = false; ins = false; break;
        case TB_OP_N: {
          bool emit = (!ins || !intron);
          int es = exstart + 1, ee = pos + l;
          l += len; exstart = pos + l; intron = true;
          if (emit) { s = es; e = ee; return true; }
          break;
        }
        case TB_OP_S: case TB_OP_H: intron = false; ins = false; break;
        case TB_OP_I: ins = true; break;
        default: break;
      }
    }
    done = true; s = exstart + 1; e = pos + l; return true;
  }
};

__device__ __forceinline__ uint64_t tb_fold(uint64_t h, uint64_t w) { h = (h ^ w) * 0x9E3779B97F4A7C15ULL; return h ^ (h >> 29); }
__device__ __forceinline__ unsigned tb_strand_code(uint8_t c) { return c == '+' ? 0u : (c == '-' ? 1u : 2u); }  // '+'(43) < '-'(45) < '.'(46)

// clipped range for -P: strip leading then trailing soft clips (cmpCigarClip :321-328)
__device__ __forceinline__ void tb_clip_range(const uint32_t* cig, uint32_t& a, uint32_t& b) {
  while (a < b && (cig[a] & 0xf) == TB_OP_S) ++a;
  while (b > a && (cig[b - 1] & 0xf) == TB_OP_S) --b;
}

// one pass over the record's CIGAR: reference length and the hash of the mode key
__device__ __forceinline__ void tb_parse_record(const ColIn& in, int64_t i, int pos, uint32_t c0, uint32_t c1, int& reflen, uint64_t& khash) {
  int l = 0;
  uint64_t h;
  if (in.mode == TB_MODE_EXON) {
    ExonIter it; it.init(in.cigar, c0, c1, pos);
    int s, e, nex = 0; h = 0x1234567ULL;
    while (it.next(s, e)) { h = tb_fold(h, ((uint64_t)(uint32_t)s << 32) | (uint32_t)e); ++nex; }
    h = tb_fold(h, (uint64_t)nex);
    l = it.l;
  } else {
    uint32_t a = c0, b = c1;
    if (in.mode == TB_MODE_CLIP) tb_clip_range(in.cigar, a, b);
    h = tb_fold(0x9876543ULL, (uint64_t)(b - a));
    for (uint32_t c = c0; c < c1; ++c) {
      uint32_t w = in.cigar[c];
      if (tb_op_ref(w & 0xf)) l += (int)(w >> 4);
      if (c >= a && c < b) h = tb_fold(h, w);
    }
    if (in.mode == TB_MODE_FULL) {
      uint32_t m0 = in.md_off[i], m1 = in.md_off[i + 1];
      h = tb_fold(h, (uint64_t)(m1 > m0));
      for (uint32_t q = m0; q < m1; ++q) { uint8_t ch = in.md[q]; if (ch == 0) break; h = tb_fold(h, ch); }
    }
  }
  reflen = l; khash = h;
}


// 32-bit variant for the tile kernel (64-bit multiplies cost four IMADs each): two independent running hashes
__device__ __forceinline__ uint32_t tb_mix32(uint32_t x) { x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16; return x; }
__device__ __forceinline__ void tb_fold2(uint32_t& h1, uint32_t& h2, uint32_t w) {
  h1 = (h1 ^ w) * 0x9E3779B1u; h1 ^= h1 >> 15;
  h2 = (h2 + w) * 0x85EBCA77u; h2 ^= h2 >> 13;
}
__device__ __forceinline__ void tb_parse_record32(const ColIn& in, int64_t i, int pos, uint32_t c0, uint32_t c1, int& reflen, uint32_t& h1o, uint32_t& h2o) {
  int l = 0;
  uint32_t h1, h2;
  if (in.mode == TB_MODE_EXON) {
    ExonIter it; it.init(in.cigar, c0, c1, pos);
    int s, e, nex = 0; h1 = 0x1234567u; h2 = 0x89abcdefu;
    while (it.next(s, e)) { tb_fold2(h1, h2, (uint32_t)s); tb_fold2(h1, h2, (uint32_t)e); ++nex; }
    tb_fold2(h1, h2, (uint32_t)nex);
    l = it.l;
  } else {
    uint32_t a = c0, b = c1;
    if (in.mode == TB_MODE_CLIP) tb_clip_range(in.cigar, a, b);
    h1 = 0x9876543u ^ (b - a); h2 = 0x3c6ef372u + (b - a);
    for (uint32_t c = c0; c < c1; ++c) {
      const uint32_t w = in.cigar[c];
      if (tb_op_ref(w & 0xf)) l += (int)(w >> 4);
      if (c >= a && c < b) tb_fold2(h1, h2, w);
    }
    if (in.mode == TB_MODE_FULL) {
      const uint32_t m0 = in.md_off[i], m1 = in.md_off[i + 1];
      tb_fold2(h1, h2, (uint32_t)(m1 > m0));
      uint32_t acc = 0, nb = 0;   // bytes up to the NUL, four per fold
      for (uint32_t q = m0; q < m1; ++q) {
        const uint32_t ch = in.md[q];
        if (ch == 0) break;
        acc = (acc << 8) | ch;
        if (++nb == 4) { tb_fold2(h1, h2, acc); acc = 0; nb = 0; }
      }
      tb_fold2(h1, h2, acc ^ (nb << 29));
    }
  }
  reflen = l; h1o = h1; h2o = h2;
}

// exact mode comparison of two records, sign as in the reference's cmp* functions (cmpFlags NOT applied)
static __device__ __noinline__ int tb_mode_cmp(const ColIn& in, uint32_t ia, uint32_t ib) {
  uint32_t a0 = in.cig_off[ia], a1 = in.cig_off[ia + 1], b0 = in.cig_off[ib], b1 = in.cig_off[ib + 1];
  if (in.mode == TB_MODE_EXON) {
    ExonIter x, y; x.init(in.cigar, a0, a1, in.pos[ia]); y.init(in.cigar, b0, b1, in.pos[ib]);
    int na = 0, nb = 0, s, e;  // exon counts first (cmpExons :337)
    { ExonIter t = x; while (t.next(s, e)) ++na; }
    { ExonIter t = y; while (t.next(s, e)) ++nb; }
    if (na != nb) return na - nb;
    int sa, ea, sb, eb;
    while (x.next(sa, ea)) { y.next(sb, eb); if (sa != sb) return sa - sb; if (ea != eb) return ea - eb; }
    return 0;
  }
  if (in.mode == TB_MODE_CLIP) { tb_clip_range(in.cigar, a0, a1); tb_clip_range(in.cigar, b0, b1); }
  int na = (int)(a1 - a0), nb = (int)(b1 - b0);
  if (na != nb) return na - nb;
  for (int q = 0; q < na; ++q) {
    uint32_t wa = in.cigar[a0 + q], wb = in.cigar[b0 + q];
    if (wa != wb) {  // memcmp over little-endian bytes == numeric order of the byte-reversed words
      uint32_t ra = __byte_perm(wa, 0, 0x0123), rb = __byte_perm(wb, 0, 0x0123);
      return ra < rb ? -1 : 1;
    }
  }
  if (in.mode == TB_MODE_FULL) {
    uint32_t ma = in.md_off[ia], mae = in.md_off[ia + 1], mb = in.md_off[ib], mbe = in.md_off[ib + 1];
    bool pa = mae > ma, pb = mbe > mb;
    if (!pa || !pb) { if (pa == pb) return 0; return pa ? 1 : -1; }
    for (;; ++ma, ++mb) {  // strcmp
      uint8_t ca = ma < mae ? in.md[ma] : 0, cb = mb < mbe ? in.md[mb] : 0;
      if (ca != cb) return (int)ca - (int)cb;
      if (ca == 0) return 0;
    }
  }
  return 0;
}

// the reference's cmp* including cmpFlags (:275-283): different masked flags compare as "1" in BOTH directions
__device__ __forceinline__ int tb_mode_cmp_flags(const ColIn& in, uint32_t ia, uint32_t ib) {
  if (in.flag_mask != 0 && ((in.flag_mask & in.flag[ia]) != (in.flag_mask & in.flag[ib]))) return 1;
  return tb_mode_cmp(in, ia, ib);
}

__device__ __forceinline__ bool tb_passes_options(const ColIn& in, uint16_t fl, uint8_t mq, uint16_t nh) {  // tiebrush.cpp:532-541
  if (!(in.keep_bits & TB_KEEP_SUPP) && (fl & 0x800)) return false;
  if (!(in.keep_bits & TB_KEEP_SECONDARY) && (fl & 0x100)) return false;
  if (!(in.keep_bits & TB_KEEP_UNMAP) && (fl & 0x4)) return false;
  if ((int)mq < in.min_qual) return false;
  if ((int)nh > in.max_nh) return false;
  return true;
}

// workspace slots in ctx->buf used by the collapse pipeline (coverage.cu has its own numbering; calls never overlap)
enum {
  XB_HIST = 0,   // u32 [S+2]  counts, then exclusive scan P
  XB_AGG,        // scan aggregates
  XB_STATUS,     // i64 [16]
  XB_SLOTPOS,    // u32 [M+2]  first position of every slot
  XB_OFF,        // u32 [(M+1)*k] per (slot,file) first record
  XB_RUNOFF,     // i64 [k+1]
  XB_MERGED,     // u8  [k]
  XB_GCOUNT,     // u32 [M+1]
  XB_GBASE,      // u32 [M+1]
  XB_ST_REP,     // u32 [n] staged (indexed by merged rank)
  XB_ST_YC,      // f32 [n]
  XB_ST_YX,      // u32 [n]
  XB_ST_BITS,    // u32 [n*W]
  XB_ST_YD,      // i32 [n]   ordered path only: max of carried YD tags
  XB_BITS,       // u32 [G*W] compacted
  XB_GDESC,      // YD: group descriptors
  XB_BHEAD,      // YD: bundle heads
  XB_YDPM,       // YD: group ends, starts and strands (genomic)
  XB_WORK,       // small device counters
  XB_YDC,        // YD: chain distances per group
  XB_YDSCRATCH,  // YD: global-memory lists of the repeat launch
  XB_YDBLK, XB_YDCHAIN, XB_YDU, XB_YDKEPT, XB_YDBM, XB_YDLZ, XB_YDUNIT, XB_HEAVY,   // YD: per-block member counts, chain members (group id, head flag | chain)
  XB_ORD_KEY, XB_ORD_KEY2, XB_ORD_VAL, XB_ORD_VAL2, XB_ORD_REFLEN, XB_ORD_TABLE, XB_ORD_AGG,   // ordered path: merge-order sort
  XB_ORD_LIST, XB_ORD_GREP, XB_ORD_GYC, XB_ORD_GYX, XB_ORD_GYD, XB_ORD_VALID, XB_ORD_GBITS,                // ordered path: per-position group lists
  XB_META_DICT,   // u64 [256] dictionary of the packed wire format
  XB_ORD_DEEP,    // ordered path: counter + list of the deep start positions
  XB_YDCARRY,     // YD carry: device copy of carry_in, per-chain seed / ext / final frontier
  XB_YDCOUT,      // YD carry: carry_out area (per-chain slots, cursor, segments)
  XB_COUNT_
};
static_assert(XB_COUNT_ <= TB_NBUF, "raise TB_NBUF");

enum { CS_ERR = 0, CS_ERRIDX, CS_NKEPT, CS_NGROUPS, CS_TABLE_OVERFLOW, CS_NBUNDLES, CS_YD_OVERFLOW, CS_NHEAVY, CS_N_ };   // 8-10: YD (YS_*)
enum { CS_TILE_RECORDS = 11, CS_TILE_HEADS, CS_TILE_BATCHES };   // tile kernel statistics of the collapse call
enum { ERR_POS_RANGE = 1, ERR_UNSORTED = 2 };
