// bgzf.cu — BAM bytes to tiecov's columns on the device: BGZF inflate and BAM record parse (SAM spec §4.1, §4.2).
//
//   host scan     one read of every BGZF header / footer (magic, XLEN, BSIZE, CRC32, ISIZE): the compressed span of each
//                 block and, by an exclusive prefix sum of ISIZE, where its output goes. An incomplete block at the end of
//                 the buffer is left to the next call.
//   B1 inflate    one warp per block (DEFLATE stored / fixed / dynamic), straight into its place in one contiguous buffer.
//                 Every lane runs the same serial Huffman decode (uniform control flow, broadcast loads); the warp shares
//                 the table build and the back-reference copies. Then the CRC32 of the block's output: every lane takes a
//                 32nd of it, the lane CRCs are joined by crc32_combine (zlib's GF(2) form) in a shuffle tree.
//   B2 walk       one thread per block walks the block_size chain from the block's first byte, guessing that a record
//                 starts there (htslib starts a new block whenever the next record would not fit). The guess of block b is
//                 proven when the chain of b-1 ended exactly on b's first byte; from the first block where that fails, one
//                 thread re-walks the chain from the true entry, block after block, reusing every walk that started on it.
//   B3 records    one thread per block lists its records' offsets; then one thread per record parses the fixed fields, the
//                 CIGAR and the aux tags (YC, YX, XS, ts; every aux type is walked, CG refused), drops unmapped records,
//                 and a device scan of (kept, n_cigar) places the kept records' columns and CIGAR words.
//
// Errors: a device status word per stage keeps the first error (atomicMin of offset << 8 | code); kernels bound-check
// every read and write against their buffers whatever the bytes say, and never trap.
#include <functional>
#include <algorithm>
#include "tc_columns.cuh"

int tc_stream_impl(tb_ctx* ctx, const tc_soa_in* in, int64_t skip, int64_t window, const int32_t* next, tc_runs_out* runs, tc_juncs_out* juncs,
                   int64_t* consumed, const std::function<int()>* after_window, const int32_t* yx);

namespace {

enum {   // ctx->bam_buf slots
  BZ_COMP = 0,   // u8  compressed bytes of the complete blocks
  BZ_BLK,        // BlkDesc [nb]
  BZ_U,          // u8  inflated bytes, all blocks back to back (+8 bytes of slack)
  BZ_WALK,       // Walk [nb]
  BZ_RBASE,      // u32 [nb] first record of every block (exclusive scan of the walk counts)
  BZ_AGG,        // scan aggregates
  BZ_ROFF,       // i64 [records] uncompressed offset of every record
  BZ_REC,        // Rec [records]
  BZ_STATUS,     // u64 [8]
  BZ_COLS,       // two record sets (ping-pong for tc_coverage_bam's held bundle): 8 slots each from here (tc_alloc_records)
  BZ_COUNT_ = BZ_COLS + 16
};
static_assert((int)BZ_COUNT_ <= (int)TB_NBAMBUF, "bam_buf too small");
// status words
enum { S_INFLATE = 0, S_WALK, S_PARSE, S_BREAK, S_TAIL, S_UNMAPPED, S_N_ };
// inflate error codes
enum { E_BTYPE = 1, E_CODE, E_DIST, E_LENGTH, E_CRC, E_TRUNC, E_STORED, E_LENS };
// parse error codes
enum { P_BSIZE = 1, P_FIELDS, P_AUX, P_CG, P_REFID };

struct BlkDesc { int64_t coff, cdata, uoff; int32_t clen, isize; uint32_t crc; int32_t pad; };   // coff: header byte in the input
struct Walk { int64_t o, e; uint32_t c; int32_t reason; };   // reason: 0 reached the block end, 1 record runs past the data, 2 bad block_size
struct Rec { int32_t tid, pos, end, yx; float yc; uint32_t ncig; int64_t cig_src; uint8_t strand, kept, pad[6]; };

// ---------------------------------------------------------------------------------------------------------------------
// B1: inflate
// ---------------------------------------------------------------------------------------------------------------------
constexpr int INF_WARPS = 4, INF_THREADS = 32 * INF_WARPS;
constexpr int LFAST = 10, DFAST = 8;   // bits resolved by one shared-memory lookup; longer codes take the canonical walk

__constant__ uint16_t c_lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_clorder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct Huff {   // canonical code: counts per length, symbols in code order, and a LFAST / DFAST-bit direct table
  uint16_t count[16];
  uint16_t first[16];   // first canonical code of every length
  uint16_t offs[16];    // index in sym of the first symbol of every length
  uint16_t next[16];    // build scratch
};

struct WarpSmem {
  uint16_t lfast[1 << LFAST];
  uint16_t dfast[1 << DFAST];
  uint16_t lsym[288];
  uint16_t dsym[32];
  Huff lh, dh;
  uint8_t lens[320];
};

struct Bits {
  const uint8_t* src; int64_t p, end; uint64_t buf; int cnt; int bad;
  __device__ __forceinline__ void refill() { while (cnt <= 56 && p < end) { buf |= (uint64_t)src[p++] << cnt; cnt += 8; } }
  __device__ __forceinline__ uint32_t get(int n) {
    if (n == 0) return 0;
    if (cnt < n) refill();
    if (cnt < n) { bad = 1; return 0; }
    const uint32_t v = (uint32_t)(buf & ((1ull << n) - 1ull));
    buf >>= n; cnt -= n;
    return v;
  }
};

// builds the code of `n` lengths in s->lens[lo..lo+n) into h / sym / fast (fast may be null); whole warp; 0 = ok
__device__ __forceinline__ int huff_build(WarpSmem* s, int lo, int n, Huff* h, uint16_t* sym, uint16_t* fast, int fastb) {
  const int lane = tb_lane();
  int err = 0;
  if (lane == 0) {
    for (int l = 0; l < 16; ++l) h->count[l] = 0;
    for (int i = 0; i < n; ++i) h->count[s->lens[lo + i]]++;
    int left = 1;
    for (int l = 1; l < 16 && !err; ++l) { left <<= 1; left -= h->count[l]; if (left < 0) err = 1; }   // over-subscribed
    h->offs[1] = 0; h->first[1] = 0;
    int code = 0;
    for (int l = 1; l < 15; ++l) { h->offs[l + 1] = h->offs[l] + h->count[l]; code = (code + h->count[l]) << 1; h->first[l + 1] = (uint16_t)code; }
    if (!err) {
      for (int l = 1; l < 16; ++l) h->next[l] = h->offs[l];
      for (int i = 0; i < n; ++i) if (s->lens[lo + i]) sym[h->next[s->lens[lo + i]]++] = (uint16_t)i;
    }
  }
  err = __shfl_sync(0xffffffffu, err, 0);
  __syncwarp();
  if (err || !fast) return err;
  for (int i = lane; i < (1 << fastb); i += 32) fast[i] = 0;
  __syncwarp();
  const int nsym = h->offs[15] + h->count[15];
  for (int k = lane; k < nsym; k += 32) {
    const int v = sym[k];
    const int l = s->lens[lo + v];
    if (l > fastb) continue;
    const uint32_t code = h->first[l] + (uint32_t)(k - h->offs[l]);
    const uint32_t rev = __brev(code) >> (32 - l);
    for (uint32_t j = rev; j < (1u << fastb); j += (1u << l)) fast[j] = (uint16_t)(v | (l << 9));
  }
  __syncwarp();
  return 0;
}

// one symbol; -1 = invalid code or no bits left
__device__ __forceinline__ int huff_decode(Bits& b, const Huff* h, const uint16_t* sym, const uint16_t* fast, int fastb) {
  if (b.cnt < 15) b.refill();
  if (fast) {
    const uint16_t e = fast[b.buf & ((1u << fastb) - 1u)];
    const int l = e >> 9;
    if (e && l <= b.cnt) { b.buf >>= l; b.cnt -= l; return e & 511; }
  }
  int code = 0, first = 0, index = 0;   // canonical walk, one bit at a time (puff's decode)
  for (int l = 1; l < 16; ++l) {
    if (b.cnt == 0) return -1;
    code |= (int)(b.buf & 1u); b.buf >>= 1; b.cnt--;
    const int c = h->count[l];
    if (code - c < first) return sym[index + (code - first)];
    index += c; first += c; first <<= 1; code <<= 1;
  }
  return -1;
}

__device__ __forceinline__ uint32_t crc_mult(uint32_t a, uint32_t b) {   // a * b mod P, reflected (zlib multmodp)
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
    m >>= 1;
    b = (b & 1) ? (b >> 1) ^ 0xedb88320u : b >> 1;
  }
  return p;
}
__device__ __forceinline__ uint32_t crc_combine(uint32_t crc1, uint32_t crc2, uint32_t len2) {   // crc32 of A||B from crc(A), crc(B), |B|
  uint32_t x = 1u << 31;            // x^0
  uint32_t sq = 1u << 23;           // x^8 (one byte)
  while (len2) { if (len2 & 1) x = crc_mult(sq, x); sq = crc_mult(sq, sq); len2 >>= 1; }
  return crc_mult(x, crc1) ^ crc2;
}

__global__ void __launch_bounds__(INF_THREADS, 8) bgzf_inflate_kernel(const uint8_t* __restrict__ comp, const BlkDesc* __restrict__ blk, int64_t nb,
                                                                  uint8_t* out, unsigned long long* __restrict__ status) {
  __shared__ WarpSmem sm[INF_WARPS];
  __shared__ uint32_t crctab[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ 0xedb88320u : c >> 1;
    crctab[i] = c;
  }
  __syncthreads();
  const int64_t b = (int64_t)blockIdx.x * INF_WARPS + tb_warp();
  if (b >= nb) return;
  const int lane = tb_lane();
  WarpSmem* s = &sm[tb_warp()];
  const BlkDesc d = blk[b];
  const int64_t obase = d.uoff, oend = d.uoff + d.isize;
  int64_t o = obase;
  Bits bits{comp, d.cdata, d.cdata + d.clen, 0, 0, 0};
  int err = 0, last = 0;
  while (!last && !err) {
    last = (int)bits.get(1);
    const uint32_t type = bits.get(2);
    if (bits.bad) { err = E_TRUNC; break; }
    if (type == 0) {   // stored: realign on the byte stream
      bits.get(bits.cnt & 7);
      bits.p -= bits.cnt >> 3; bits.buf = 0; bits.cnt = 0;
      if (bits.p + 4 > bits.end) { err = E_TRUNC; break; }
      const uint32_t len = comp[bits.p] | (uint32_t)comp[bits.p + 1] << 8, nlen = comp[bits.p + 2] | (uint32_t)comp[bits.p + 3] << 8;
      bits.p += 4;
      if (len != (~nlen & 0xffffu)) { err = E_STORED; break; }
      if (bits.p + len > bits.end) { err = E_TRUNC; break; }
      if (o + len > oend) { err = E_LENGTH; break; }
      for (uint32_t k = lane; k < len; k += 32) out[o + k] = comp[bits.p + k];
      bits.p += len; o += len;
      __syncwarp();
      continue;
    }
    if (type == 3) { err = E_BTYPE; break; }
    int nlen = 288, ndist = 30;
    if (type == 1) {
      for (int i = lane; i < 320; i += 32) s->lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
      __syncwarp();
    } else {
      nlen = (int)bits.get(5) + 257; ndist = (int)bits.get(5) + 1;
      const int ncode = (int)bits.get(4) + 4;
      if (bits.bad) { err = E_TRUNC; break; }
      if (nlen > 286 || ndist > 30) { err = E_LENS; break; }
      if (lane == 0) for (int i = 0; i < 19; ++i) s->lens[c_clorder[i]] = 0;
      __syncwarp();
      for (int i = 0; i < ncode; ++i) { const uint32_t v = bits.get(3); if (lane == 0) s->lens[c_clorder[i]] = (uint8_t)v; }
      __syncwarp();
      if (bits.bad) { err = E_TRUNC; break; }
      if (huff_build(s, 0, 19, &s->lh, s->lsym, nullptr, 0)) { err = E_LENS; break; }
      // the code lengths of both codes, read with the code-length code (kept in lsym / lh until the real code replaces it)
      uint8_t tmp_prev = 0;
      int idx = 0;
      __shared__ uint8_t ltmp[INF_WARPS][320];
      uint8_t* lt = ltmp[tb_warp()];
      while (idx < nlen + ndist) {
        const int sy = huff_decode(bits, &s->lh, s->lsym, nullptr, 0);
        if (sy < 0) { err = bits.cnt == 0 && bits.p >= bits.end ? E_TRUNC : E_CODE; break; }
        if (sy < 16) { if (lane == 0) lt[idx] = (uint8_t)sy; tmp_prev = (uint8_t)sy; ++idx; continue; }
        int rep; uint8_t v = 0;
        if (sy == 16) { if (idx == 0) { err = E_LENS; break; } v = tmp_prev; rep = 3 + (int)bits.get(2); }
        else if (sy == 17) rep = 3 + (int)bits.get(3);
        else rep = 11 + (int)bits.get(7);
        if (bits.bad) { err = E_TRUNC; break; }
        if (idx + rep > nlen + ndist) { err = E_LENS; break; }
        if (lane == 0) for (int k = 0; k < rep; ++k) lt[idx + k] = v;
        idx += rep; tmp_prev = v;
      }
      __syncwarp();
      if (err) break;
      for (int i = lane; i < 320; i += 32) s->lens[i] = i < nlen ? lt[i] : (i >= 288 && i - 288 < ndist ? lt[nlen + i - 288] : 0);
      __syncwarp();
      if (s->lens[256] == 0) { err = E_LENS; break; }
    }
    // literal / length code in lens[0..nlen), distance code in lens[288..288+ndist)
    if (huff_build(s, 0, nlen, &s->lh, s->lsym, s->lfast, LFAST) || huff_build(s, 288, ndist, &s->dh, s->dsym, s->dfast, DFAST)) { err = E_LENS; break; }
    for (;;) {
      const int sy = huff_decode(bits, &s->lh, s->lsym, s->lfast, LFAST);
      if (sy < 0) { err = (bits.p >= bits.end && bits.cnt < 15) ? E_TRUNC : E_CODE; break; }
      if (sy < 256) {
        if (o >= oend) { err = E_LENGTH; break; }
        if (lane == 0) out[o] = (uint8_t)sy;
        ++o;
        continue;
      }
      if (sy == 256) break;
      const int li = sy - 257;
      if (li >= 29) { err = E_CODE; break; }
      const int len = c_lbase[li] + (int)bits.get(c_lext[li]);
      const int ds = huff_decode(bits, &s->dh, s->dsym, s->dfast, DFAST);
      if (ds < 0 || ds >= 30) { err = ds < 0 && bits.p >= bits.end ? E_TRUNC : E_CODE; break; }
      const int64_t dist = c_dbase[ds] + (int)bits.get(c_dext[ds]);
      if (bits.bad) { err = E_TRUNC; break; }
      if (dist > o - obase) { err = E_DIST; break; }
      if (o + len > oend) { err = E_LENGTH; break; }
      const int step = dist < 32 ? (int)dist : 32;
      __syncwarp();
      for (int j = 0; j < len; j += step) {
        const int k = j + lane;
        if (lane < step && k < len) out[o + k] = out[o + k - dist];
        __syncwarp();
      }
      o += len;
    }
    __syncwarp();
  }
  if (!err && o != oend) err = E_LENGTH;
  if (err) {
    if (lane == 0) atomicMin(status + S_INFLATE, ((unsigned long long)b << 8) | (unsigned long long)err);
    return;
  }
  // CRC32 of [obase, oend): a contiguous slice per lane, joined left to right in a shuffle tree
  const int64_t n = oend - obase, per = (n + 31) / 32;
  const int64_t a0 = obase + (int64_t)lane * per < oend ? obase + (int64_t)lane * per : oend;
  const int64_t a1 = a0 + per < oend ? a0 + per : oend;
  uint32_t c = 0xffffffffu;
  for (int64_t k = a0; k < a1; ++k) c = crctab[(c ^ out[k]) & 0xff] ^ (c >> 8);
  c ^= 0xffffffffu;
  uint32_t len = (uint32_t)(a1 - a0);
  for (int dlt = 1; dlt < 32; dlt <<= 1) {
    const uint32_t c2 = __shfl_down_sync(0xffffffffu, c, dlt), l2 = __shfl_down_sync(0xffffffffu, len, dlt);
    if ((lane & (2 * dlt - 1)) == 0) { c = crc_combine(c, c2, l2); len += l2; }
  }
  if (lane == 0 && c != d.crc) atomicMin(status + S_INFLATE, ((unsigned long long)b << 8) | (unsigned long long)E_CRC);
}

// ---------------------------------------------------------------------------------------------------------------------
// B2: record boundaries
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_u32(const uint8_t* u, int64_t p) { return u[p] | (uint32_t)u[p + 1] << 8 | (uint32_t)u[p + 2] << 16 | (uint32_t)u[p + 3] << 24; }
__device__ __forceinline__ uint16_t ld_u16(const uint8_t* u, int64_t p) { return (uint16_t)(u[p] | u[p + 1] << 8); }

// the block_size chain from t while it starts records inside [.., bend); every record it counts lies inside [0, U)
__device__ Walk walk_chain(const uint8_t* u, int64_t U, int64_t t, int64_t bend) {
  Walk w{t, t, 0, 0};
  int64_t p = t;
  while (p < bend) {
    if (p + 4 > U) { w.reason = 1; break; }
    const uint32_t bs = ld_u32(u, p);
    if (bs < 32) { w.reason = 2; break; }
    if (p + 4 + (int64_t)bs > U) { w.reason = 1; break; }
    p += 4 + (int64_t)bs;
    w.c++;
  }
  w.e = p;
  return w;
}

__global__ void walk_guess_kernel(const uint8_t* __restrict__ u, int64_t U, const BlkDesc* __restrict__ blk, int64_t nb, int64_t skip, Walk* __restrict__ walk,
                                  unsigned long long* __restrict__ status) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  const int64_t bend = blk[b].uoff + blk[b].isize;
  const Walk w = walk_chain(u, U, b == 0 ? skip : blk[b].uoff, bend);
  walk[b] = w;
  const int64_t next = b + 1 < nb ? blk[b + 1].uoff : U;
  if (w.reason != 0 || w.e != next) atomicMin(status + S_BREAK, (unsigned long long)b);
}

// one thread: from the first block whose chain did not end on the next block's first byte, follow the true chain
__global__ void walk_fix_kernel(const uint8_t* __restrict__ u, int64_t U, const BlkDesc* __restrict__ blk, int64_t nb, Walk* __restrict__ walk,
                                unsigned long long* __restrict__ status) {
  const unsigned long long b0 = status[S_BREAK];
  if (b0 >= (unsigned long long)nb) { status[S_TAIL] = (unsigned long long)U; return; }
  int64_t t = walk[b0].o;
  int64_t tail = -1;
  for (int64_t b = (int64_t)b0; b < nb; ++b) {
    if (tail >= 0) { walk[b].c = 0; walk[b].o = walk[b].e = tail; walk[b].reason = 0; continue; }
    Walk w = walk[b];
    if (w.o != t) { w = walk_chain(u, U, t, blk[b].uoff + blk[b].isize); walk[b] = w; }
    if (w.reason == 2) { atomicMin(status + S_WALK, ((unsigned long long)w.e << 8) | P_BSIZE); tail = w.e; walk[b].reason = 0; continue; }
    if (w.reason == 1) { tail = w.e; walk[b].reason = 0; continue; }
    t = w.e;
  }
  status[S_TAIL] = (unsigned long long)(tail >= 0 ? tail : t);
}

struct WalkCountIn { const Walk* w; __device__ uint32_t operator()(int64_t i) const { return w[i].c; } };
struct WalkBaseOut { uint32_t* base; __device__ void operator()(int64_t i, uint32_t exc, uint32_t) const { base[i] = exc; } };

__global__ void record_offsets_kernel(const uint8_t* __restrict__ u, const Walk* __restrict__ walk, const uint32_t* __restrict__ base, int64_t nb,
                                      int64_t* __restrict__ roff) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  int64_t p = walk[b].o;
  const uint32_t c = walk[b].c, r0 = base[b];
  for (uint32_t k = 0; k < c; ++k) { roff[r0 + k] = p; p += 4 + (int64_t)ld_u32(u, p); }
}

// ---------------------------------------------------------------------------------------------------------------------
// B3: one thread per record
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int aux_fixed_size(uint8_t t) {
  switch (t) {
    case 'A': case 'c': case 'C': return 1;
    case 's': case 'S': return 2;
    case 'i': case 'I': case 'f': return 4;
    case 'd': return 8;
    default: return 0;
  }
}

// bam_aux2f / bam_aux2i of the value at u[v] of type t (known to lie inside the record)
__device__ double aux_num(const uint8_t* u, int64_t v, uint8_t t, bool as_float) {
  switch (t) {
    case 'c': return (double)(int8_t)u[v];
    case 'C': return (double)u[v];
    case 's': return (double)(int16_t)ld_u16(u, v);
    case 'S': return (double)ld_u16(u, v);
    case 'i': return (double)(int32_t)ld_u32(u, v);
    case 'I': return (double)ld_u32(u, v);
    case 'f': return as_float ? (double)__uint_as_float(ld_u32(u, v)) : 0.0;
    case 'd': return as_float ? __longlong_as_double((long long)((uint64_t)ld_u32(u, v) | (uint64_t)ld_u32(u, v + 4) << 32)) : 0.0;
    default: return 0.0;
  }
}

__global__ void __launch_bounds__(256) parse_kernel(const uint8_t* __restrict__ u, const int64_t* __restrict__ roff, int64_t n, Rec* __restrict__ rec,
                                                   unsigned long long* __restrict__ status) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t r = roff[i];
  const int64_t rend = r + 4 + (int64_t)ld_u32(u, r);   // inside the data (record walk)
  Rec o; memset(&o, 0, sizeof(o));
  auto fail = [&](int code) { atomicMin(status + S_PARSE, ((unsigned long long)r << 8) | (unsigned long long)code); rec[i] = o; };
  const int32_t refid = (int32_t)ld_u32(u, r + 4), pos = (int32_t)ld_u32(u, r + 8);
  const int l_qn = u[r + 12];
  const int ncig = ld_u16(u, r + 16), flag = ld_u16(u, r + 18);
  const int32_t l_seq = (int32_t)ld_u32(u, r + 20);
  if (l_seq < 0) { fail(P_FIELDS); return; }
  const int64_t cig = r + 36 + l_qn;
  const int64_t aux = cig + 4 * (int64_t)ncig + ((int64_t)l_seq + 1) / 2 + l_seq;
  if (aux > rend) { fail(P_FIELDS); return; }
  int64_t yc_v = -1, yx_v = -1, xs_v = -1, ts_v = -1;
  uint8_t yc_t = 0, yx_t = 0, xs_t = 0, ts_t = 0;
  for (int64_t a = aux; a < rend;) {
    if (a + 3 > rend) { fail(P_AUX); return; }
    const uint8_t t0 = u[a], t1 = u[a + 1], ty = u[a + 2];
    const int64_t v = a + 3;
    int64_t next;
    const int fs = aux_fixed_size(ty);
    if (fs) next = v + fs;
    else if (ty == 'Z' || ty == 'H') {
      int64_t z = v;
      while (z < rend && u[z] != 0) ++z;
      if (z >= rend) { fail(P_AUX); return; }
      next = z + 1;
    } else if (ty == 'B') {
      if (v + 5 > rend) { fail(P_AUX); return; }
      const int es = aux_fixed_size(u[v]);
      if (es == 0 || es == 8 || u[v] == 'A') { fail(P_AUX); return; }
      next = v + 5 + (int64_t)es * (int64_t)ld_u32(u, v + 1);
    } else { fail(P_AUX); return; }
    if (next > rend) { fail(P_AUX); return; }
    if (t0 == 'C' && t1 == 'G') { fail(P_CG); return; }
    if (t0 == 'Y' && t1 == 'C' && yc_v < 0) { yc_v = v; yc_t = ty; }
    else if (t0 == 'Y' && t1 == 'X' && yx_v < 0) { yx_v = v; yx_t = ty; }
    else if (t0 == 'X' && t1 == 'S' && xs_v < 0) { xs_v = v; xs_t = ty; }
    else if (t0 == 't' && t1 == 's' && ts_v < 0) { ts_v = v; ts_t = ty; }
    a = next;
  }
  o.kept = (flag & 4) ? 0 : 1;   // tiecov.cpp:436-438
  if (!o.kept) { atomicAdd(status + S_UNMAPPED, 1ull); rec[i] = o; return; }
  if (refid < 0) { fail(P_REFID); return; }
  o.tid = refid; o.pos = pos; o.ncig = (uint32_t)ncig; o.cig_src = cig;
  int rl = 0;
  for (int k = 0; k < ncig; ++k) { const uint32_t w = ld_u32(u, cig + 4 * k); if ((0x18Du >> (w & 0xf)) & 1u) rl += (int)(w >> 4); }   // tb_op_ref
  o.end = pos + rl;
  o.yc = yc_v >= 0 ? (float)aux_num(u, yc_v, yc_t, true) : 1.0f;                 // tiecov.cpp:482-485
  o.yx = yx_v >= 0 ? (int32_t)(int64_t)aux_num(u, yx_v, yx_t, false) : 1;         // tiecov.cpp:495
  // spliceStrand (GSam.cpp:464-475): XS of type A / Z when not empty, else ts flipped on the reverse strand
  uint8_t c = 0;
  if (xs_v >= 0 && (xs_t == 'A' || xs_t == 'Z') && u[xs_v] != 0) c = u[xs_v];
  if (c == 0 && ts_v >= 0 && (ts_t == 'A' || ts_t == 'Z')) {
    const uint8_t m = u[ts_v];
    if (m == '+' || m == '-') c = (flag & 16) ? (m == '+' ? '-' : '+') : m;
  }
  o.strand = (c == '+' || c == '-') ? c : '.';
  rec[i] = o;
}

struct KeepIn { const Rec* rec; __device__ long long operator()(int64_t i) const { return rec[i].kept ? (1LL << 32) | (long long)rec[i].ncig : 0LL; } };
struct KeepOut {   // places record i's columns and CIGAR words after the `held` records already in the set
  const Rec* rec; const uint8_t* u; TcRecords c; int64_t held; uint32_t held_cig; int64_t n;
  __device__ void operator()(int64_t i, long long exc, long long inc) const {
    const Rec& x = rec[i];
    if (x.kept) {
      const int64_t d = held + (exc >> 32);
      const uint32_t co = held_cig + (uint32_t)(exc & 0xffffffffLL);
      c.tid[d] = x.tid; c.pos[d] = x.pos; c.end[d] = x.end; c.yc[d] = x.yc; c.yx[d] = x.yx; c.strand[d] = x.strand; c.cig_off[d] = co;
      for (uint32_t k = 0; k < x.ncig; ++k) c.cigar[co + k] = ld_u32(u, x.cig_src + 4 * k);
    }
    if (i == n - 1) c.cig_off[held + (inc >> 32)] = held_cig + (uint32_t)(inc & 0xffffffffLL);
  }
};

const char* inflate_msg(int code) {
  switch (code) {
    case E_BTYPE: return "invalid DEFLATE block type";
    case E_CODE: return "invalid Huffman code";
    case E_DIST: return "back-reference distance before the start of the block";
    case E_LENGTH: return "inflated length differs from ISIZE";
    case E_CRC: return "CRC32 of the inflated bytes differs from the footer";
    case E_TRUNC: return "DEFLATE data ends early";
    case E_STORED: return "stored block LEN / NLEN mismatch";
    default: return "invalid Huffman code lengths";
  }
}
const char* parse_msg(int code) {
  switch (code) {
    case P_BSIZE: return "block_size below the 32-byte fixed part";
    case P_FIELDS: return "read name / CIGAR / SEQ / QUAL run past the record";
    case P_AUX: return "aux field runs past the record or has an unknown type";
    case P_CG: return "CIGAR stored in the CG tag (records with more than 65535 operations are not supported)";
    default: return "mapped record (flag without 0x4) with refID < 0";
  }
}

// record set k of ctx->bam_buf, as sized by the last bam_decode that wrote it
TcRecords column_set(tb_ctx* ctx, int k) {
  TcRecords c;
  tc_alloc_records(ctx->bam_buf + BZ_COLS + 8 * k, 0, 0, true, &c);
  return c;
}

}  // namespace


// Decodes the complete blocks of `in` into column set 1 - ctx->bam_set. The first `held` records of that set are the bundle
// tc_coverage_bam holds from its last call (copied from ctx->bam_set), the kept records of this chunk follow them.
// *set / *n_out / *ncig_out: the set written, its records and CIGAR words. Fills st (resume_* included). 0 = ok.
static int bam_decode(tb_ctx* ctx, const tb_bgzf_in* in, int64_t held, const char* fn, int* set_out, int64_t* n_out, uint32_t* ncig_out, tb_bgzf_stat* st) {
  TB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  memset(st, 0, sizeof(*st));
  if (in->n_bytes < 0 || (in->n_bytes > 0 && !in->data) || in->skip < 0) {
    ctx->set_error("%s: invalid input (n_bytes %lld, skip %lld)", fn, (long long)in->n_bytes, (long long)in->skip); return 1;
  }
  // ---- host scan of the block headers / footers ----
  const uint8_t* h = in->data;
  std::vector<BlkDesc> blk;
  int64_t p = 0, U = 0;
  while (p < in->n_bytes) {
    const int64_t rem = in->n_bytes - p;
    if (rem < 18) break;
    if (h[p] != 0x1f || h[p + 1] != 0x8b || h[p + 2] != 8 || h[p + 3] != 4) {
      ctx->set_error("%s: BGZF block at byte offset %lld: bad gzip header (magic 1f 8b 08 and FLG 04 expected)", fn, (long long)p); return 1;
    }
    const int xlen = h[p + 10] | h[p + 11] << 8;
    if (rem < 12 + xlen) break;
    int bsize = -1;
    for (int x = 0; x + 4 <= xlen;) {
      const int slen = h[p + 12 + x + 2] | h[p + 12 + x + 3] << 8;
      if (h[p + 12 + x] == 'B' && h[p + 12 + x + 1] == 'C' && slen == 2 && x + 6 <= xlen) { bsize = h[p + 12 + x + 4] | h[p + 12 + x + 5] << 8; break; }
      x += 4 + slen;
    }
    if (bsize < 0) { ctx->set_error("%s: BGZF block at byte offset %lld: no BC subfield (BSIZE) in the gzip extra field", fn, (long long)p); return 1; }
    const int64_t total = (int64_t)bsize + 1;
    if (total < 12 + xlen + 8) { ctx->set_error("%s: BGZF block at byte offset %lld: BSIZE %d shorter than its header and footer", fn, (long long)p, bsize); return 1; }
    if (rem < total) break;
    auto le32 = [&](int64_t q) { return (uint32_t)h[q] | (uint32_t)h[q + 1] << 8 | (uint32_t)h[q + 2] << 16 | (uint32_t)h[q + 3] << 24; };
    BlkDesc d;
    d.coff = p; d.cdata = p + 12 + xlen; d.clen = (int32_t)(total - 12 - xlen - 8);
    d.crc = le32(p + total - 8);
    const uint32_t isize = le32(p + total - 4);
    if (isize > 65536) { ctx->set_error("%s: BGZF block at byte offset %lld: ISIZE %u above 64 KiB", fn, (long long)p, isize); return 1; }
    d.isize = (int32_t)isize; d.uoff = U; d.pad = 0;
    blk.push_back(d);
    U += isize; p += total;
  }
  const int64_t complete = p;
  if (in->last && complete < in->n_bytes) { ctx->set_error("%s: truncated BGZF block at byte offset %lld (no data follows)", fn, (long long)complete); return 1; }
  if (U >= (1LL << 32)) { ctx->set_error("%s: %lld inflated bytes in one call (at most 4 GiB: pass smaller chunks)", fn, (long long)U); return 1; }
  const int64_t nb = (int64_t)blk.size();
  st->blocks = nb; st->bytes_in = complete; st->bytes_out = U;
  if (nb > 0 && in->skip > blk[0].isize) { ctx->set_error("%s: skip %lld beyond the first block's %d inflated bytes", fn, (long long)in->skip, blk[0].isize); return 1; }
  if (nb == 0 && in->last && in->skip > 0) { ctx->set_error("%s: skip %lld but no block follows", fn, (long long)in->skip); return 1; }
  // uncompressed offset -> (byte offset of the block that holds it, offset inside that block)
  auto where = [&](int64_t uo, int64_t* bo, int64_t* within) {
    int64_t b = std::upper_bound(blk.begin(), blk.end(), uo, [](int64_t v, const BlkDesc& x) { return v < x.uoff; }) - blk.begin() - 1;
    if (b < 0) b = 0;
    while (b > 0 && blk[b].isize == 0) --b;
    *bo = blk[b].coff; *within = uo - blk[b].uoff;
  };
  DevBuf* B = ctx->bam_buf;
  TB_CUDA(B[BZ_STATUS].ensure(sizeof(unsigned long long) * 8));
  TB_CUDA(ctx->bam_pinned.ensure(sizeof(unsigned long long) * 8));
  unsigned long long* d_st = B[BZ_STATUS].as<unsigned long long>();
  unsigned long long* h_st = ctx->bam_pinned.as<unsigned long long>();
  int64_t nrec = 0, tail = U;
  const uint8_t* du = nullptr;
  if (nb > 0) {
    // ---- B1 ----
    TB_CUDA(B[BZ_COMP].ensure((size_t)complete + 8));
    TB_CUDA(B[BZ_BLK].ensure(sizeof(BlkDesc) * nb));
    TB_CUDA(B[BZ_U].ensure((size_t)U + 8));
    du = B[BZ_U].as<uint8_t>();
    TB_CUDA(cudaMemcpyAsync(B[BZ_COMP].p, h, (size_t)complete, cudaMemcpyHostToDevice, s));
    TB_CUDA(cudaMemcpyAsync(B[BZ_BLK].p, blk.data(), sizeof(BlkDesc) * nb, cudaMemcpyHostToDevice, s));
    for (int k = 0; k < 8; ++k) h_st[k] = 0;
    h_st[S_INFLATE] = h_st[S_WALK] = h_st[S_PARSE] = h_st[S_BREAK] = ~0ull;
    TB_CUDA(cudaMemcpyAsync(d_st, h_st, sizeof(unsigned long long) * 8, cudaMemcpyHostToDevice, s));
    if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[14], s));
    bgzf_inflate_kernel<<<tb_grid_for(nb, INF_WARPS), INF_THREADS, 0, s>>>(B[BZ_COMP].as<uint8_t>(), B[BZ_BLK].as<BlkDesc>(), nb, B[BZ_U].as<uint8_t>(), d_st);
    ctx->launches++;
    TB_CUDA(cudaGetLastError());
    if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[15], s));
    TB_CUDA(cudaMemcpyAsync(h_st, d_st, sizeof(unsigned long long) * 8, cudaMemcpyDeviceToHost, s));
    TB_CUDA(cudaStreamSynchronize(s));
    if (ctx->profiling) { float ms = 0; if (cudaEventElapsedTime(&ms, ctx->ev[14], ctx->ev[15]) == cudaSuccess) ctx->last_ms[10] = ms; }
    if (h_st[S_INFLATE] != ~0ull) {
      ctx->set_error("%s: BGZF block at byte offset %lld: %s", fn, (long long)blk[h_st[S_INFLATE] >> 8].coff, inflate_msg((int)(h_st[S_INFLATE] & 0xff)));
      return 1;
    }
    // ---- B2 ----
    if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[14], s));
    TB_CUDA(B[BZ_WALK].ensure(sizeof(Walk) * nb));
    TB_CUDA(B[BZ_RBASE].ensure(sizeof(uint32_t) * (nb + 1)));
    Walk* walk = B[BZ_WALK].as<Walk>();
    walk_guess_kernel<<<tb_grid_for(nb, 128), 128, 0, s>>>(du, U, B[BZ_BLK].as<BlkDesc>(), nb, in->skip, walk, d_st);
    walk_fix_kernel<<<1, 1, 0, s>>>(du, U, B[BZ_BLK].as<BlkDesc>(), nb, walk, d_st);
    ctx->launches += 2;
    TB_CUDA(B[BZ_AGG].ensure(sizeof(long long) * (tb_scan_blocks(nb) + 8)));
    TB_CUDA((tb_device_scan<OpSumU32>(ctx, WalkCountIn{walk}, nb, B[BZ_AGG].as<uint32_t>(), WalkBaseOut{B[BZ_RBASE].as<uint32_t>()})));
    uint32_t nrec_u = 0;
    TB_CUDA(cudaMemcpyAsync(&nrec_u, B[BZ_AGG].as<uint32_t>() + tb_scan_blocks(nb), sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    TB_CUDA(cudaMemcpyAsync(h_st, d_st, sizeof(unsigned long long) * 8, cudaMemcpyDeviceToHost, s));
    TB_CUDA(cudaStreamSynchronize(s));
    if (h_st[S_WALK] != ~0ull) {
      const int64_t uo = (int64_t)(h_st[S_WALK] >> 8);
      int64_t bo, w; where(uo, &bo, &w);
      ctx->set_error("%s: BAM record at inflated offset %lld (BGZF block at byte offset %lld, +%lld): %s", fn, (long long)uo, (long long)bo, (long long)w, parse_msg(P_BSIZE));
      return 1;
    }
    tail = (int64_t)h_st[S_TAIL];
    nrec = nrec_u;
  }
  if (in->last && tail != U) {
    int64_t bo, w; where(tail, &bo, &w);
    ctx->set_error("%s: BAM record at inflated offset %lld (BGZF block at byte offset %lld, +%lld) runs past the end of the data (no data follows)", fn,
                   (long long)tail, (long long)bo, (long long)w);
    return 1;
  }
  if (nb == 0) { st->resume_byte = in->last ? in->n_bytes : 0; st->resume_skip = in->last ? 0 : in->skip; }
  else if (tail == U) { st->resume_byte = complete; st->resume_skip = 0; }
  else { int64_t bo, w; where(tail, &bo, &w); st->resume_byte = bo; st->resume_skip = w; }
  // ---- B3 ----
  if (nrec > 0) {
    TB_CUDA(B[BZ_ROFF].ensure(sizeof(int64_t) * nrec));
    TB_CUDA(B[BZ_REC].ensure(sizeof(Rec) * nrec));
    record_offsets_kernel<<<tb_grid_for(nb, 128), 128, 0, s>>>(du, B[BZ_WALK].as<Walk>(), B[BZ_RBASE].as<uint32_t>(), nb, B[BZ_ROFF].as<int64_t>());
    parse_kernel<<<tb_grid_for(nrec, 256), 256, 0, s>>>(du, B[BZ_ROFF].as<int64_t>(), nrec, B[BZ_REC].as<Rec>(), d_st);
    ctx->launches += 2;
    TB_CUDA(cudaGetLastError());
    TB_CUDA(cudaMemcpyAsync(h_st, d_st, sizeof(unsigned long long) * 8, cudaMemcpyDeviceToHost, s));
    TB_CUDA(cudaStreamSynchronize(s));
    if (h_st[S_PARSE] != ~0ull) {
      const int64_t uo = (int64_t)(h_st[S_PARSE] >> 8);
      int64_t bo, w; where(uo, &bo, &w);
      ctx->set_error("%s: BAM record at inflated offset %lld (BGZF block at byte offset %lld, +%lld): %s", fn, (long long)uo, (long long)bo, (long long)w,
                     parse_msg((int)(h_st[S_PARSE] & 0xff)));
      return 1;
    }
    st->unmapped = (int64_t)h_st[S_UNMAPPED];
  }
  st->records = nrec - st->unmapped;
  // ---- columns: the held records, then the kept records of this chunk. Sized from the ISIZE sum: a CIGAR word takes 4
  // inflated bytes, so U / 4 bounds this chunk's words ----
  const int set = 1 - ctx->bam_set;
  const uint32_t held_cig = held > 0 ? ctx->bam_hcig : 0;
  const int64_t cap_cig = (int64_t)held_cig + U / 4 + 1;
  if (cap_cig >= (1LL << 32)) { ctx->set_error("%s: %lld CIGAR words exceed the 32-bit offsets of one column set (pass smaller chunks)", fn, (long long)cap_cig); return 1; }
  TcRecords c;
  TB_CUDA(tc_alloc_records(B + BZ_COLS + 8 * set, held + nrec + 1, cap_cig, true, &c));
  if (held > 0) tc_copy_records(ctx, s, column_set(ctx, ctx->bam_set), ctx->bam_from, held, c, 0, 0, held_cig);
  long long tot = 0;
  if (nrec > 0) {
    TB_CUDA(B[BZ_AGG].ensure(sizeof(long long) * (tb_scan_blocks(nrec) + 8)));
    TB_CUDA((tb_device_scan<OpSumI64>(ctx, KeepIn{B[BZ_REC].as<Rec>()}, nrec, B[BZ_AGG].as<long long>(), KeepOut{B[BZ_REC].as<Rec>(), du, c, held, held_cig, nrec})));
    TB_CUDA(cudaMemcpyAsync(&tot, B[BZ_AGG].as<long long>() + tb_scan_blocks(nrec), sizeof(long long), cudaMemcpyDeviceToHost, s));
  } else if (held == 0) {
    TB_CUDA(cudaMemsetAsync(c.cig_off, 0, sizeof(uint32_t), s));
  }
  if (ctx->profiling && nb > 0) TB_CUDA(cudaEventRecord(ctx->ev[15], s));
  TB_CUDA(cudaStreamSynchronize(s));
  if (ctx->profiling && nb > 0) { float ms = 0; if (cudaEventElapsedTime(&ms, ctx->ev[14], ctx->ev[15]) == cudaSuccess) ctx->last_ms[11] = ms; }
  *set_out = set;
  *n_out = held + (int64_t)(tot >> 32);
  *ncig_out = held_cig + (uint32_t)(tot & 0xffffffffLL);
  return 0;
}

static void set_columns(tb_ctx* ctx, int set, int64_t n, uint32_t ncig, tc_soa_in* cols, const int32_t** yx) {
  const TcRecords c = column_set(ctx, set);
  *cols = tc_window(c, n, ncig);
  if (yx) *yx = c.yx;
}

extern "C" {

int tc_bam_columns(tb_ctx* ctx, const tb_bgzf_in* in, tc_soa_in* cols, const int32_t** yx, tb_bgzf_stat* st) {
  if (!ctx) return 1;
  if (!in || !cols || !st) { ctx->set_error("tc_bam_columns: in, cols and st are required"); return 1; }
  ctx->err.clear();
  ctx->bam_held = 0;   // the columns of this call replace whatever tc_coverage_bam held
  int set; int64_t n; uint32_t ncig;
  const int rc = bam_decode(ctx, in, 0, "tc_bam_columns", &set, &n, &ncig, st);
  if (rc) return rc;
  ctx->bam_set = set;
  set_columns(ctx, set, n, ncig, cols, yx);
  return 0;
}

int tc_coverage_bam(tb_ctx* ctx, const tb_bgzf_in* in, int64_t window, tc_runs_out* runs, tc_juncs_out* juncs, tc_runs_out* sample_rows, tb_bgzf_stat* st) {
  if (!ctx) return 1;
  if (!in || !st || (!runs && !juncs && !sample_rows)) { ctx->set_error("tc_coverage_bam: in, st and one of runs / juncs / sample_rows are required"); return 1; }
  ctx->err.clear();
  if (runs) runs->n_runs = 0;
  if (juncs) juncs->n_juncs = 0;
  if (sample_rows) sample_rows->n_runs = 0;
  ctx->stream_windows = 0;
  if (in->first) ctx->bam_held = 0;
  int set; int64_t n; uint32_t ncig;
  int rc = bam_decode(ctx, in, ctx->bam_held, "tc_coverage_bam", &set, &n, &ncig, st);
  if (rc) return rc;
  // a bundle has at most 2 runs (or heat-map rows) per M block and one junction per N op
  st->need_rows = 2 * (int64_t)ncig + 16;
  if ((runs && runs->capacity < st->need_rows) || (sample_rows && sample_rows->capacity < st->need_rows) || (juncs && juncs->capacity < (int64_t)ncig + 16)) {
    ctx->set_error("tc_coverage_bam: row capacity too small (%lld rows and %lld junctions needed); the call may be repeated with the same input", (long long)st->need_rows,
                   (long long)ncig + 16);
    return 5;
  }
  tc_soa_in cols; const int32_t* yx = nullptr;
  set_columns(ctx, set, n, ncig, &cols, &yx);
  // the open bundle at the end of the chunk waits for the records of the next call: a next record at {last tid, -1}
  // continues it whatever its end
  int32_t nx[2] = {0, -1};
  if (!in->last && n > 0) {
    TB_CUDA(cudaMemcpyAsync(&nx[0], cols.tid + n - 1, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    TB_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  const int32_t* next = in->last ? nullptr : nx;
  int64_t consumed = 0, consumed_s = 0;
  int exact = 0;
  if (n > 0 && (runs || juncs)) {
    rc = tc_stream_impl(ctx, &cols, 0, window, next, runs, juncs, &consumed, nullptr, nullptr);
    if (rc) return rc;
    exact = ctx->last_cov_exact;
  }
  if (n > 0 && sample_rows) {
    rc = tc_stream_impl(ctx, &cols, 0, window, next, sample_rows, nullptr, &consumed_s, nullptr, yx);
    if (rc) return rc;
    if ((runs || juncs) && consumed_s != consumed) { ctx->set_error("tc_coverage_bam: the heat-map and the coverage windows disagree (internal error)"); return 1; }
    consumed = consumed_s;
    ctx->last_cov_exact = exact;
  }
  ctx->bam_set = set;
  ctx->bam_from = consumed;
  ctx->bam_held = n - consumed;
  ctx->bam_cbase = 0;
  if (ctx->bam_held > 0) {
    TB_CUDA(cudaMemcpyAsync(&ctx->bam_cbase, cols.cig_off + consumed, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    TB_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  ctx->bam_hcig = ncig - ctx->bam_cbase;
  return 0;
}

}  // extern "C"
