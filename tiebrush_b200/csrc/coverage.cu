// coverage.cu — tiecov's hot path on the device (reference src/tiecov.cpp:62-120, 194-241, 435-528).
//
//   K6  bundle breaks   : prefix-max of (tid,end) over the record stream; a record opens a bundle iff its
//                         tid differs from, or its start exceeds, the running max end   (tiecov.cpp:443);
//                         three streaming passes with the `end` column (cbk_*_kernel), one pass with decoupled
//                         look-back without it (cov_bundle_kernel)
//   K7  coverage        : difference array over BUNDLE-COMPACTED coordinates (gaps between bundles are
//                         skipped; one sentinel cell closes each bundle), +w at every M-block start and
//                         -w one past its end, 64-bit fixed-point atomics                (addCov :194-223)
//   K8  bedgraph runs   : scan of the difference array -> change points -> stream compaction of the
//                         non-zero-depth runs; runs never join across bundles     (flushCoverage :226-241)
//   -s  sample heat-map : per compacted cell the float32 running mean of YX over its covering records in stream order,
//                         ceil, runs of equal value (addMean / discretize / flushCoverage :155-185, 277-309): tc_sample_window
//   K9  junctions       : intron (start,end,strand) keys reduced in a device hash table (fingerprint CAS,
//                         min/max verified, so exactness never rests on the hash), then radix-sorted
//                         into print order                                   (addJunction/flushJuncs :100-120)
//
// Weights: YC is float32 on disk (SURVEY §9.5); the reference accumulates doubles. Here every weight is
// converted once to 2^-20 fixed point (exact for all integer-valued YC and for dyadic fractions) and
// summed in int64, which equals the reference's double sum whenever that sum is exact.
#include "tb_common.cuh"

namespace {

constexpr double COV_FX_SCALE = 1048576.0;

enum {  // workspace slots in ctx->buf
  CB_KEY = 0,     // u64 [2*tiles+8] look-back tile states of K6 (max chain, count chain) + ticket
  CB_BID,         // u32 [n]   bundle id per record
  CB_BSTART,      // i32 [n]   bundle start (1-based)   (indexed by bundle)
  CB_BEND,        // i32 [n]
  CB_BTID,        // i32 [n]
  CB_BBASE,       // i64 [n+1] compact base offset per bundle
  CB_AGG,         // scan aggregates (max of all uses)
  CB_STATUS,      // i64 [16]  device status block
  CB_DIFF,        // i64 [L]
  CB_CPPOS,       // i64 [Kmax]
  CB_CPDEPTH,     // i64 [Kmax]
  CB_JTAG,        // u64 [JCAP]
  CB_JKMIN,       // u64 [JCAP]
  CB_JKMAX,       // u64 [JCAP]
  CB_JTID,        // i32 [2*JCAP] (min, max)
  CB_JVAL,        // i64 [JCAP]
  CB_JKEYS,       // u64 [J] compacted
  CB_JIDX,        // u32 [J]
  CB_JKEYS2,      // u64 [J]
  CB_JIDX2,       // u32 [J]
  CB_RSTABLE,     // radix sort table
  CB_RSAGG,
  CB_TIDKEYS,     // u64 [J]
  CB_TIDKEYS2,
  CB_PMEND,       // u32 [n]  exact path: inclusive prefix maximum of the record ends (1-based), monotone inside a tid (junc_exact_kernel)
  CB_RFIRST,      // u32 [n]  first record of every bundle (cov_tail_kernel, junc_exact_kernel)
  CB_IOFF,        // u32 [n+1] ordered walks: first item of every record
  CB_IKEY, CB_IKEY2, CB_IVAL, CB_IVAL2,   // u64 / u32 [items] tile id | item index (radix sort ping-pong)
  CB_ILO, CB_IHI, CB_IREC,                // u32 [items] first / last cell of the item, its record
  CB_COUNT_
};

// status block layout (int64 each)
enum { ST_ERRIDX = 0, ST_NBUNDLES, ST_DENSE_LEN, ST_NCHANGE, ST_NRUNS, ST_NJUNC, ST_JOVERFLOW, ST_RUNOVERFLOW, ST_INEXACT, ST_LBFAIL, ST_N_,
       ST_TAIL_END = 12, ST_TAIL_TID = 13, ST_TAIL_FIRST = 14 };   // slot 10 (ST_N_) is the junction compaction counter; 12-14: last bundle of the window
static_assert(ST_N_ < ST_TAIL_END, "status slots overlap");

struct CovIn {
  int64_t n;
  const int32_t* tid; const int32_t* pos; const float* yc; const uint8_t* strand;
  const uint32_t* cig_off; const uint32_t* cigar;
  const int32_t* end;   // optional (tc_soa_in.end): 0-based exclusive end of every record; K6 then never touches the CIGARs
};

// ---- K6: bundles in ONE pass over the records (decoupled look-back) -----------------------------------------------
// A record opens a bundle iff its tid differs from, or its start exceeds, the running maximum end of everything before
// it (tiecov.cpp:443): with key = tid << 32 | end that is a test against the exclusive prefix maximum of the keys, and the
// bundle id is the inclusive prefix count of such heads. Both prefixes are carried across tiles of 2048 records by
// single-word tile states (2 flag bits | 62-bit payload; aggregate first, inclusive prefix once the tile's own look-back
// is done): the max chain resolves first, the head count of a tile follows from it, then the count chain. Tiles take
// tickets in launch order, so every predecessor of a running tile is itself running or finished (forward progress);
// the spin is bounded and reports through ST_LBFAIL instead of hanging. The head of bundle b also closes bundle b-1:
// its exclusive prefix maximum IS that bundle's end (a bundle starts beyond every earlier end of its tid).
// Reads every input field once (27 B per record) and writes the bundle id (4 B); no key / prefix arrays.
constexpr int CBK_THREADS = 256, CBK_ITEMS = 16, CBK_TILE = CBK_THREADS * CBK_ITEMS, CBK_MINB = 2;
// VEC: the per-record columns are 16-byte aligned, so a thread fetches its CBK_ITEMS consecutive records with 128-bit loads
// (a warp request then covers 512 contiguous bytes instead of 32 scattered sectors)
template <bool VEC>
__global__ void __launch_bounds__(CBK_THREADS, CBK_MINB) cov_bundle_kernel(CovIn in, int check_ops, unsigned long long* __restrict__ st_max,
                                                                 unsigned long long* __restrict__ st_cnt, unsigned long long* __restrict__ ticket,
                                                                 uint32_t* __restrict__ bid, int32_t* __restrict__ bstart, int32_t* __restrict__ bend,
                                                                 int32_t* __restrict__ btid, uint32_t* __restrict__ pmend, uint32_t* __restrict__ rfirst,
                                                                 long long* __restrict__ status) {
  __shared__ unsigned long long s_scan64[33];
  __shared__ uint32_t s_scan32[33];
  __shared__ unsigned long long s_tile, s_pa, s_pb;
  if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1ULL);
  __syncthreads();
  const long long tile = (long long)s_tile;
  const int64_t base = tile * CBK_TILE + (int64_t)threadIdx.x * CBK_ITEMS;
  unsigned long long key[CBK_ITEMS]; int pos[CBK_ITEMS], tidv[CBK_ITEMS];
  uint32_t coff[CBK_ITEMS + 1]; float ycv[CBK_ITEMS];   // coff: CIGAR offsets
  const bool full = base + CBK_ITEMS <= in.n;
  if (VEC && full) {
    static_assert(CBK_ITEMS % 4 == 0, "128-bit loads");
#pragma unroll
    for (int q = 0; q < CBK_ITEMS / 4; ++q) {
      const int4 p = *reinterpret_cast<const int4*>(in.pos + base + 4 * q), t = *reinterpret_cast<const int4*>(in.tid + base + 4 * q);
      const uint4 c = *reinterpret_cast<const uint4*>(in.cig_off + base + 4 * q);
      const float4 y = *reinterpret_cast<const float4*>(in.yc + base + 4 * q);
      pos[4 * q] = p.x; pos[4 * q + 1] = p.y; pos[4 * q + 2] = p.z; pos[4 * q + 3] = p.w;
      tidv[4 * q] = t.x; tidv[4 * q + 1] = t.y; tidv[4 * q + 2] = t.z; tidv[4 * q + 3] = t.w;
      coff[4 * q] = c.x; coff[4 * q + 1] = c.y; coff[4 * q + 2] = c.z; coff[4 * q + 3] = c.w;
      ycv[4 * q] = y.x; ycv[4 * q + 1] = y.y; ycv[4 * q + 2] = y.z; ycv[4 * q + 3] = y.w;
    }
    coff[CBK_ITEMS] = in.cig_off[base + CBK_ITEMS];
  } else {
#pragma unroll
    for (int k = 0; k < CBK_ITEMS; ++k) {
      const int64_t i = base + k;
      pos[k] = 0; tidv[k] = 0; coff[k] = 0; ycv[k] = 0.f;
      if (i < in.n) { pos[k] = in.pos[i]; tidv[k] = in.tid[i]; coff[k] = in.cig_off[i]; ycv[k] = in.yc[i]; }
    }
    coff[CBK_ITEMS] = 0;
#pragma unroll
    for (int k = 0; k < CBK_ITEMS; ++k) if (base + k < in.n) coff[k + 1] = in.cig_off[base + k + 1];
  }
  unsigned long long tm = 0;
#pragma unroll
  for (int k = 0; k < CBK_ITEMS; ++k) {
    const int64_t i = base + k;
    key[k] = 0;
    if (i < in.n) {
      const uint32_t c0 = coff[k], c1 = coff[k + 1];
      int l = 0;
      bool bad = check_ops && (c1 - c0 >= 256u);  // tiecov.cpp:198 uint8_t loop counter never terminates
      for (uint32_t c = c0; c < c1; ++c) {
        const uint32_t w = in.cigar[c];
        const uint32_t op = w & 0xf, len = w >> 4;
        if (op == TB_OP_M || op == TB_OP_D || op == TB_OP_N || op == TB_OP_EQ || op == TB_OP_X) l += (int)len;
        if (check_ops && !(op == TB_OP_M || op == TB_OP_I || op == TB_OP_D || op == TB_OP_N || op == TB_OP_S)) bad = true;
      }
      if (bad) atomicMin((unsigned long long*)&status[ST_ERRIDX], (unsigned long long)i);
      key[k] = ((unsigned long long)(uint32_t)tidv[k] << 32) | (uint32_t)(pos[k] + l);
      const float sc = ycv[k] * (float)COV_FX_SCALE;
      if (sc != truncf(sc)) status[ST_INEXACT] = 1;  // benign race: any writer stores 1
      tm = key[k] > tm ? key[k] : tm;
    }
  }
  // ---- max chain ----
  unsigned long long tot;
  const unsigned long long texc = tb_block_exscan<OpMaxU64>(tm, s_scan64, &tot);
  if (threadIdx.x == 0) lb_store(&st_max[tile], LB_AGG | tot);
  if (threadIdx.x < 32) {
    const unsigned long long pa = lb_lookback<true>(st_max, tile, &status[ST_LBFAIL]);
    if (threadIdx.x == 0) { s_pa = pa; lb_store(&st_max[tile], LB_INC | (pa > tot ? pa : tot)); }
  }
  __syncthreads();
  unsigned long long run = s_pa > texc ? s_pa : texc;   // exclusive prefix maximum at this thread's first record
  // ---- heads ----
  const unsigned long long run0 = run; uint32_t headm = 0, hc = 0;
#pragma unroll
  for (int k = 0; k < CBK_ITEMS; ++k) {
    const int64_t i = base + k;
    if (i < in.n) {
      const bool h = i == 0 || tidv[k] != (int)(run >> 32) || (pos[k] + 1) > (int)(uint32_t)run;   // tiecov.cpp:443
      if (h) { headm |= 1u << k; ++hc; }
      run = key[k] > run ? key[k] : run;
    }
  }
  // ---- count chain ----
  uint32_t htot;
  const uint32_t hexc = tb_block_exscan<OpSumU32>(hc, s_scan32, &htot);
  if (threadIdx.x == 0) lb_store(&st_cnt[tile], LB_AGG | (unsigned long long)htot);
  if (threadIdx.x < 32) {
    const unsigned long long pb = lb_lookback<false>(st_cnt, tile, &status[ST_LBFAIL]);
    if (threadIdx.x == 0) { s_pb = pb; lb_store(&st_cnt[tile], LB_INC | (pb + htot)); }
  }
  __syncthreads();
  uint32_t cnt = (uint32_t)s_pb + hexc;   // heads before this thread's first record
  run = run0;
#pragma unroll
  for (int k = 0; k < CBK_ITEMS; ++k) {
    const int64_t i = base + k;
    if (i >= in.n) break;
    if (headm & (1u << k)) {
      const uint32_t b = cnt++;
      bstart[b] = pos[k] + 1; btid[b] = tidv[k];
      if (b > 0) bend[b - 1] = (int)(uint32_t)run;   // this head closes the previous bundle
      if (rfirst) rfirst[b] = (uint32_t)i;
    }
    bid[i] = cnt - 1;
    run = key[k] > run ? key[k] : run;
    if (pmend) pmend[i] = (uint32_t)run;
    if (i == in.n - 1) { bend[cnt - 1] = (int)(uint32_t)run; status[ST_NBUNDLES] = cnt; }
  }
}

// ---- K6 with the end column: three streaming passes instead of two look-back chains -------------------------------
// With GSamRecord::end supplied there is no CIGAR walk in K6 and the single pass above spends its time waiting on the
// look-back chains (16 % issue slots, 18 % of the DRAM peak in ncu). Reading the small columns again is cheaper:
//   P1  maximum key of every tile of 4096 records (tid, end: 8 B per record)            -> device scan: tile prefixes
//   P2  heads from the exclusive prefix maximum (pos, tid, end, yc: 16 B per record): per thread a 16-bit head mask,
//       per tile the head count; a head parks the end of the bundle it closes in its own bid slot  -> device scan
//   P3  bundle ids from the masks alone (0.125 B per record read, 4 B written as 128-bit stores); only the heads touch
//       pos / tid / the parked end to write bstart, btid, bend and rfirst.
// 28 B per record in three coalesced passes, no inter-CTA waiting. Same outputs as cov_bundle_kernel (which stays for
// inputs without the end column and for the pmend pass of the exact path).
struct TileU64In { const unsigned long long* p; __device__ unsigned long long operator()(int64_t i) const { return p[i]; } };
struct TileU64Exc { unsigned long long* p; __device__ void operator()(int64_t i, unsigned long long exc, unsigned long long) const { p[i] = exc; } };
struct TileU32In { const uint32_t* p; __device__ uint32_t operator()(int64_t i) const { return p[i]; } };
struct TileU32Exc { uint32_t* p; __device__ void operator()(int64_t i, uint32_t exc, uint32_t) const { p[i] = exc; } };

template <bool VEC>
__global__ void __launch_bounds__(CBK_THREADS) cbk_tilemax_kernel(CovIn in, unsigned long long* __restrict__ tmax) {
  __shared__ unsigned long long s_red[CBK_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * CBK_TILE + (int64_t)threadIdx.x * CBK_ITEMS;
  unsigned long long tm = 0;
  if (VEC && base + CBK_ITEMS <= in.n) {
#pragma unroll
    for (int q = 0; q < CBK_ITEMS / 4; ++q) {
      const int4 t = *reinterpret_cast<const int4*>(in.tid + base + 4 * q);
      const uint4 e = *reinterpret_cast<const uint4*>(in.end + base + 4 * q);
      const unsigned long long k0 = ((unsigned long long)(uint32_t)t.x << 32) | e.x, k1 = ((unsigned long long)(uint32_t)t.y << 32) | e.y,
                               k2 = ((unsigned long long)(uint32_t)t.z << 32) | e.z, k3 = ((unsigned long long)(uint32_t)t.w << 32) | e.w;
      const unsigned long long a = k0 > k1 ? k0 : k1, b = k2 > k3 ? k2 : k3, c = a > b ? a : b;
      tm = c > tm ? c : tm;
    }
  } else {
#pragma unroll
    for (int k = 0; k < CBK_ITEMS; ++k)
      if (base + k < in.n) {
        const unsigned long long key = ((unsigned long long)(uint32_t)in.tid[base + k] << 32) | (uint32_t)in.end[base + k];
        tm = key > tm ? key : tm;
      }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) { const unsigned long long o = __shfl_xor_sync(0xffffffffu, tm, d); tm = o > tm ? o : tm; }
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = tm;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < CBK_THREADS / 32; ++w) tm = s_red[w] > tm ? s_red[w] : tm;
    tmax[blockIdx.x] = tm;
  }
}

template <bool VEC>
__global__ void __launch_bounds__(CBK_THREADS) cbk_heads_kernel(CovIn in, const unsigned long long* __restrict__ tpre, uint16_t* __restrict__ masks,
                                                                uint32_t* __restrict__ theads, uint32_t* bid, long long* __restrict__ status) {
  static_assert(CBK_ITEMS <= 16, "16-bit head masks");
  __shared__ unsigned long long s_scan64[33];
  __shared__ uint32_t s_red[CBK_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * CBK_TILE + (int64_t)threadIdx.x * CBK_ITEMS;
  int pos[CBK_ITEMS], tidv[CBK_ITEMS]; uint32_t endv[CBK_ITEMS]; float ycv[CBK_ITEMS];
  if (VEC && base + CBK_ITEMS <= in.n) {
#pragma unroll
    for (int q = 0; q < CBK_ITEMS / 4; ++q) {
      const int4 p = *reinterpret_cast<const int4*>(in.pos + base + 4 * q), t = *reinterpret_cast<const int4*>(in.tid + base + 4 * q);
      const uint4 e = *reinterpret_cast<const uint4*>(in.end + base + 4 * q);
      const float4 y = *reinterpret_cast<const float4*>(in.yc + base + 4 * q);
      pos[4 * q] = p.x; pos[4 * q + 1] = p.y; pos[4 * q + 2] = p.z; pos[4 * q + 3] = p.w;
      tidv[4 * q] = t.x; tidv[4 * q + 1] = t.y; tidv[4 * q + 2] = t.z; tidv[4 * q + 3] = t.w;
      endv[4 * q] = e.x; endv[4 * q + 1] = e.y; endv[4 * q + 2] = e.z; endv[4 * q + 3] = e.w;
      ycv[4 * q] = y.x; ycv[4 * q + 1] = y.y; ycv[4 * q + 2] = y.z; ycv[4 * q + 3] = y.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < CBK_ITEMS; ++k) {
      const int64_t i = base + k;
      pos[k] = 0; tidv[k] = 0; endv[k] = 0; ycv[k] = 0.f;
      if (i < in.n) { pos[k] = in.pos[i]; tidv[k] = in.tid[i]; endv[k] = (uint32_t)in.end[i]; ycv[k] = in.yc[i]; }
    }
  }
  unsigned long long tm = 0; bool inexact = false;
#pragma unroll
  for (int k = 0; k < CBK_ITEMS; ++k)
    if (base + k < in.n) {
      const unsigned long long key = ((unsigned long long)(uint32_t)tidv[k] << 32) | endv[k];
      tm = key > tm ? key : tm;
      const float sc = ycv[k] * (float)COV_FX_SCALE;
      inexact |= sc != truncf(sc);
    }
  if (inexact) status[ST_INEXACT] = 1;  // benign race: any writer stores 1
  const unsigned long long texc = tb_block_exscan<OpMaxU64>(tm, s_scan64, (unsigned long long*)nullptr);
  const unsigned long long tp = tpre[blockIdx.x];
  unsigned long long run = tp > texc ? tp : texc;   // exclusive prefix maximum at this thread's first record
  uint32_t headm = 0;
#pragma unroll
  for (int k = 0; k < CBK_ITEMS; ++k) {
    const int64_t i = base + k;
    if (i < in.n) {
      const bool h = i == 0 || tidv[k] != (int)(run >> 32) || (pos[k] + 1) > (int)(uint32_t)run;   // tiecov.cpp:443
      if (h) { headm |= 1u << k; bid[i] = (uint32_t)run; }   // parked for P3: the end of the bundle this head closes
      const unsigned long long key = ((unsigned long long)(uint32_t)tidv[k] << 32) | endv[k];
      run = key > run ? key : run;
    }
  }
  masks[(int64_t)blockIdx.x * CBK_THREADS + threadIdx.x] = (uint16_t)headm;
  uint32_t hc = __popc(headm);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) hc += __shfl_xor_sync(0xffffffffu, hc, d);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = hc;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < CBK_THREADS / 32; ++w) hc += s_red[w];
    theads[blockIdx.x] = hc;
  }
}

__global__ void __launch_bounds__(CBK_THREADS) cbk_write_kernel(CovIn in, const uint16_t* __restrict__ masks, const uint32_t* __restrict__ thbase,
                                                                const unsigned long long* __restrict__ tpre, const unsigned long long* __restrict__ tmax,
                                                                uint32_t* bid, int32_t* __restrict__ bstart, int32_t* __restrict__ bend,
                                                                int32_t* __restrict__ btid, uint32_t* __restrict__ rfirst, long long* __restrict__ status) {
  __shared__ uint32_t s_scan32[33];
  const int64_t base = (int64_t)blockIdx.x * CBK_TILE + (int64_t)threadIdx.x * CBK_ITEMS;
  const uint32_t headm = masks[(int64_t)blockIdx.x * CBK_THREADS + threadIdx.x];
  const uint32_t hexc = tb_block_exscan<OpSumU32>((uint32_t)__popc(headm), s_scan32, (uint32_t*)nullptr);
  uint32_t cnt = thbase[blockIdx.x] + hexc;   // heads before this thread's first record
  uint32_t ids[CBK_ITEMS];
#pragma unroll
  for (int k = 0; k < CBK_ITEMS; ++k) {
    const int64_t i = base + k;
    if (headm & (1u << k)) {
      const uint32_t b = cnt++;
      bstart[b] = in.pos[i] + 1; btid[b] = in.tid[i];
      if (b > 0) bend[b - 1] = (int)bid[i];   // parked by P2; this head closes the previous bundle
      if (rfirst) rfirst[b] = (uint32_t)i;
    }
    ids[k] = cnt - 1;
  }
  if (base + CBK_ITEMS <= in.n) {
#pragma unroll
    for (int q = 0; q < CBK_ITEMS / 4; ++q)
      *reinterpret_cast<uint4*>(bid + base + 4 * q) = make_uint4(ids[4 * q], ids[4 * q + 1], ids[4 * q + 2], ids[4 * q + 3]);
  } else {
#pragma unroll
    for (int k = 0; k < CBK_ITEMS; ++k) if (base + k < in.n) bid[base + k] = ids[k];
  }
  if (base < in.n && in.n - 1 < base + CBK_ITEMS) {   // the thread of the last record: close the last bundle
    const unsigned long long a = tpre[blockIdx.x], b = tmax[blockIdx.x], fin = a > b ? a : b;
    uint32_t last = 0;
#pragma unroll
    for (int k = 0; k < CBK_ITEMS; ++k) if (base + k == in.n - 1) last = ids[k];
    bend[last] = (int)(uint32_t)fin; status[ST_NBUNDLES] = (long long)last + 1;
  }
}

struct BLenIn {
  const int32_t* bstart; const int32_t* bend; const long long* status;
  __device__ long long operator()(int64_t b) const {
    if (b >= status[ST_NBUNDLES]) return 0;
    long long len = (long long)bend[b] - bstart[b] + 1;
    if (len < 0) len = 0;
    return len + 1;  // + sentinel cell one past the bundle end
  }
};
struct BBaseOut { long long* base; __device__ void operator()(int64_t b, long long exc, long long) const { base[b] = exc; } };

__global__ void cov_publish_kernel(const long long* len_total, long long* status) { status[ST_DENSE_LEN] = *len_total; }

// ---- K7 + K9 insert ---------------------------------------------------------------------------------
// Junction table: open addressing on the full 64-bit key (start<<33 | end<<2 | strand code; code 3 never occurs, so ~0 is
// a safe EMPTY) claimed by CAS, the reference id claimed by a second CAS (-1 = not yet written), the value added with a
// RED. Equality is decided on the real key and tid, never on a hash.
struct JTable {
  unsigned long long* key; int32_t* tid; long long* val;
  uint32_t mask; uint64_t seed;
};
constexpr unsigned long long J_EMPTY = ~0ULL;

__device__ __forceinline__ void junc_insert(const JTable& jt, int tid, unsigned long long k64, long long w, long long* status) {
  const unsigned long long h = tb_mix64(k64 ^ tb_mix64((unsigned long long)(uint32_t)tid + jt.seed));
  uint32_t s = (uint32_t)(h >> 20) & jt.mask;
  for (uint32_t probe = 0; probe <= jt.mask; ++probe) {
    unsigned long long cur = jt.key[s];
    if (cur == J_EMPTY) {
      cur = atomicCAS(&jt.key[s], J_EMPTY, k64);
      if (cur == J_EMPTY) { atomicAdd((unsigned long long*)&status[ST_NJUNC], 1ULL); cur = k64; }
    }
    if (cur == k64) {
      int t = jt.tid[s];
      if (t == -1) { t = atomicCAS(&jt.tid[s], -1, tid); if (t == -1) t = tid; }
      if (t == tid) { atomicAdd((unsigned long long*)&jt.val[s], (unsigned long long)w); return; }
      // same coordinates on another reference: a different junction, keep probing. The slot claim above counted a new
      // junction only when this thread created the key; a (key, other tid) pair is created further down the probe.
    }
    s = (s + 1) & jt.mask;
  }
  status[ST_JOVERFLOW] = 1;
}

__device__ __forceinline__ unsigned strand_code(uint8_t c) { return c == '+' ? 0u : (c == '-' ? 1u : 2u); }  // '+' < '-' < '.'
__device__ __forceinline__ uint8_t strand_char(unsigned c) { return c == 0 ? '+' : (c == 1 ? '-' : '.'); }

// Segmented inclusive prefix sum over runs of adjacent lanes (`head` marks the first lane of a run).
__device__ __forceinline__ long long cov_seg_prefix(bool head_in, long long val) {
  const unsigned lane = threadIdx.x & 31;
  int h = (lane == 0 || head_in) ? 1 : 0;
  long long v = val;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const long long v2 = __shfl_up_sync(0xffffffffu, v, d); const int h2 = __shfl_up_sync(0xffffffffu, h, d);
    if ((int)lane >= d) { if (!h) v += v2; h |= h2; }
  }
  return v;
}

// K7 geometry: a CTA owns COV_RPT*256 consecutive records and a shared-memory tile of COV_TILE difference cells that
// starts at the compact coordinate of its first record. The stream is coordinate sorted, so nearly every update of the
// CTA (M-block starts and ends within ~COV_TILE bases of the first start) lands in the tile; blocks behind a long intron
// fall outside and go to global memory directly. A cell is an exact 64-bit two's-complement sum kept as two 32-bit
// words: native 32-bit shared atomics on the low word, the carry / borrow it reports folded into the high word (64-bit
// shared atomicAdd is a CAS loop on sm_100). Junction weights are pre-aggregated the same way in a small shared hash
// table. The flush issues one global RED per NON-ZERO cell / occupied junction slot: an order of magnitude fewer global
// atomics than one per update, and none of them contended inside the CTA. The kernel waits on memory more than it
// issues, so the geometry buys occupancy: 2048 cells (28 KB of shared memory per CTA with the lists) and a 40-register
// cap keep 6 CTAs = 48 warps per SM; 4096 cells / 5 CTAs measured 13 % slower on the C4 stream, 7 or 8 CTAs spill.
constexpr int COV_THREADS = 256;
constexpr int COV_RPT = 16;
constexpr int COV_TILE = 2048;
constexpr int COV_JSLOTS = 256;
constexpr int COV_MINB = 6;
constexpr int COV_BATCH = 4;
static_assert(COV_RPT % COV_BATCH == 0, "COV_RPT must be a multiple of COV_BATCH");

__device__ __forceinline__ void cov_cell_add(uint32_t* lo, uint32_t* hi, uint32_t c, long long w) {   // cell c += w
  const uint32_t wl = (uint32_t)(unsigned long long)w, wh = (uint32_t)((unsigned long long)w >> 32);
  const uint32_t old = atomicAdd(&lo[c], wl);
  const uint32_t add_hi = wh + ((uint32_t)(old + wl) < old ? 1u : 0u);
  if (add_hi) atomicAdd(&hi[c], add_hi);
}

struct CovSmem {
  uint32_t lo[COV_TILE], hi[COV_TILE];
  unsigned long long jkey[COV_JSLOTS]; uint32_t jlo[COV_JSLOTS], jhi[COV_JSLOTS];
  uint16_t list[COV_THREADS * COV_RPT];   // per warp: its records, grouped by CIGAR length class
};

// What a record's updates go through: the CTA's shared tile of difference cells and its small junction table, global
// memory for whatever falls outside.
struct CovTile {
  CovSmem* sm; long long cell0; int tid0; long long* diff; JTable jt; long long* status;
  __device__ __forceinline__ void cell(long long c, long long w) const {
    const unsigned long long rel = (unsigned long long)(c - cell0);
    if (rel < (unsigned long long)COV_TILE) cov_cell_add(sm->lo, sm->hi, (uint32_t)rel, w);
    else atomicAdd((unsigned long long*)&diff[c], (unsigned long long)w);
  }
  __device__ __forceinline__ void junction(int tid, unsigned long long k64, long long w) const {
    if (tid == tid0) {
      uint32_t s = (uint32_t)(tb_mix64(k64) >> 40) & (COV_JSLOTS - 1);
#pragma unroll 1
      for (int probe = 0; probe < 8; ++probe) {
        unsigned long long cur = sm->jkey[s];
        if (cur == J_EMPTY) { cur = atomicCAS(&sm->jkey[s], J_EMPTY, k64); if (cur == J_EMPTY) cur = k64; }
        if (cur == k64) { cov_cell_add(sm->jlo, sm->jhi, s, w); return; }
        s = (s + 1) & (COV_JSLOTS - 1);
      }
    }
    junc_insert(jt, tid, k64, w, status);
  }
};

// setupCoordinates' state (GSam.cpp:351-417) plus the pending -w of the coverage walk, advanced one CIGAR word at a time.
struct CovWalk {
  int l = 0, exstart, nclosed = 0, last_end = 0;
  bool intron = false, ins = false;
  long long pend = -1;   // difference cell of the pending -w (one past the last M block), -1 = none
  // the switch of setupCoordinates / addCov as predicated arithmetic (lanes of a warp sit on different ops):
  //   M,=,X,D : l += len, intron = ins = false      N : close the exon (unless ins && intron), l += len, intron = true
  //   S,H     : intron = ins = false                I : ins = true                  M alone adds coverage
  __device__ __forceinline__ void step(const CovTile& t, uint32_t cw, int pos, int tid, unsigned sc, long long shift, long long w,
                                       int do_cov, int do_junc, int check_ops, int64_t i) {
    const uint32_t op = cw & 0xf; const int len = (int)(cw >> 4);
    if (check_ops && !((0x1Fu >> op) & 1u)) atomicMin((unsigned long long*)&t.status[ST_ERRIDX], (unsigned long long)i);   // M I D N S only (tiecov.cpp:219-220)
    if (op == TB_OP_M) {
      if (do_cov && len > 0 && w != 0) {
        const long long a = (long long)(pos + l + 1) + shift;
        if (pend != a) {       // the -w closing an M block cancels against the +w opening the next when they touch (M I M)
          if (pend >= 0) t.cell(pend, -w);
          t.cell(a, w);
        }
        pend = a + len;
      }
    } else if (op == TB_OP_N) {
      if (!ins || !intron) {
        if (do_junc && nclosed > 0)
          t.junction(tid, ((unsigned long long)(uint32_t)(last_end + 1) << 33) | ((unsigned long long)(uint32_t)exstart << 2) | sc, w);
        last_end = pos + l; nclosed++;
      }
      exstart = pos + l + len;
    }
    const bool refc = (0x18Du >> op) & 1u;            // M(0) D(2) N(3) =(7) X(8) consume the reference
    const bool known = (0x1BFu >> op) & 1u;           // M I D N S H = X: the ops the reference's switch names
    l += refc ? len : 0;
    if (known) {
      ins = (op == TB_OP_I) || (op == TB_OP_N && ins);
      intron = (op == TB_OP_N) || (op == TB_OP_I && intron);
    }
  }
  __device__ __forceinline__ void finish(const CovTile& t, int tid, unsigned sc, long long w, int do_junc) {
    if (pend >= 0) t.cell(pend, -w);
    if (do_junc && nclosed > 0)   // the junction that ends at the last exon
      t.junction(tid, ((unsigned long long)(uint32_t)(last_end + 1) << 33) | ((unsigned long long)(uint32_t)exstart << 2) | sc, w);
  }
};

// One warp walks its list: 32 entries per step, neighbours in the list being neighbours in the stream with the same
// CIGAR length, so the lanes of a step run the same number of words (a step that straddles two classes aside). The fixed
// columns are loaded together, then the first three CIGAR words and the bundle base together; longer CIGARs load the
// rest word by word. One loop for every length: the code stays small enough for the instruction cache.
__device__ __forceinline__ void cov_walk_list(const CovIn& in, const uint32_t* __restrict__ bid, const int32_t* __restrict__ bstart,
                                              const long long* __restrict__ bbase, const uint16_t* list, unsigned cnt, unsigned lane,
                                              int64_t wrec0, const CovTile& t, int do_cov, int do_junc, int check_ops) {
#pragma unroll 1
  for (unsigned e0 = 0; e0 < cnt; e0 += 32) {
    const unsigned e = e0 + lane;
    bool on = e < cnt;
    int64_t i = 0; uint32_t c0 = 0, nc = 0, b = 0; int pos = 0, tid = 0; float yc = 0.f; unsigned st = 0;
    if (on) {
      const unsigned slot = list[e];
      i = wrec0 + (int64_t)(slot >> 5) * COV_THREADS + (slot & 31);
      c0 = in.cig_off[i]; nc = in.cig_off[i + 1] - c0;
      pos = in.pos[i]; tid = in.tid[i]; yc = in.yc[i]; st = in.strand[i]; b = bid[i];
    }
    uint32_t cw0 = 0, cw1 = 0, cw2 = 0; long long shift = 0;
    if (on) {
      shift = bbase[b] - (long long)bstart[b];   // compact index of 1-based coordinate x is x + shift
      cw0 = in.cigar[c0];
      if (nc > 1u) cw1 = in.cigar[c0 + 1];
      if (nc > 2u) cw2 = in.cigar[c0 + 2];
    }
    long long w = on ? (long long)rintf(yc * (float)COV_FX_SCALE) : 0;
    // Adjacent list entries that are the same alignment (pile-ups of an uncollapsed or synthetic stream) would all hit the
    // same shared cells: sum their weights in registers by one segmented prefix sum and let the last of the run issue the
    // updates. The comparison is on registers (neighbour lane by shuffle); skipped when the step has no such pair.
    bool dup;
    {
      const int ppos = __shfl_up_sync(0xffffffffu, pos, 1), ptid = __shfl_up_sync(0xffffffffu, tid, 1);
      const unsigned pst = __shfl_up_sync(0xffffffffu, st, 1), pnc = __shfl_up_sync(0xffffffffu, nc, 1);
      const uint32_t pc0 = __shfl_up_sync(0xffffffffu, c0, 1);
      const uint32_t pw0 = __shfl_up_sync(0xffffffffu, cw0, 1), pw1 = __shfl_up_sync(0xffffffffu, cw1, 1), pw2 = __shfl_up_sync(0xffffffffu, cw2, 1);
      dup = on && lane > 0 && ppos == pos && ptid == tid && pst == st && pnc == nc && pw0 == cw0 && pw1 == cw1 && pw2 == cw2;   // (an idle lane has nc 0)
      if (dup)
        for (uint32_t q = 3; q < nc; ++q) if (in.cigar[pc0 + q] != in.cigar[c0 + q]) { dup = false; break; }
    }
    if (__any_sync(0xffffffffu, dup)) {
      w = cov_seg_prefix(!dup, w);
      const int next_dup = __shfl_down_sync(0xffffffffu, (int)dup, 1);
      if (lane != 31 && next_dup) on = false;   // not the last record of its run inside this step
    }
    if (!on) continue;
    const unsigned sc = strand_code((uint8_t)st);
    CovWalk wk; wk.exstart = pos;
    if (check_ops && nc >= 256u) atomicMin((unsigned long long*)&t.status[ST_ERRIDX], (unsigned long long)i);   // tiecov.cpp:198
#pragma unroll 1
    for (uint32_t q = 0; q < nc; ++q) {
      const uint32_t cw = q == 0 ? cw0 : (q == 1 ? cw1 : (q == 2 ? cw2 : in.cigar[c0 + q]));
      wk.step(t, cw, pos, tid, sc, shift, w, do_cov, do_junc, check_ops, i);
    }
    wk.finish(t, tid, sc, w, do_junc);
  }
}

// K7. A CTA owns COV_RPT*256 consecutive records, a warp every eighth group of 32 of them. A lane's warp pays for the
// longest CIGAR among its 32 records, and the C4 stream mixes 1-, 3- and 5-word CIGARs evenly, so each warp first SORTS
// its 512 records by CIGAR length class (1, 3, 2, 4, 5 words, longer) into its own shared list — classes counted and
// ranked with match / redux warp primitives on six 10-bit counters packed in two registers, no atomics, no CTA barrier —
// and then walks the classes one after another (cov_walk_list).
__global__ void __launch_bounds__(COV_THREADS, COV_MINB) cov_accumulate_kernel(CovIn in, const uint32_t* __restrict__ bid, const int32_t* __restrict__ bstart,
                                                                     const long long* __restrict__ bbase, long long* __restrict__ diff,
                                                                     int do_cov, int do_junc, JTable jt, long long* __restrict__ status, int check_ops) {
  __shared__ CovSmem sm;
  static_assert(COV_RPT * 3 <= 64 && COV_RPT * 32 < 1024, "class word / packed counters sized for <= 21 rounds");
  const int64_t rec0 = (int64_t)blockIdx.x * (COV_THREADS * COV_RPT);
  for (int c = threadIdx.x; c < COV_TILE; c += COV_THREADS) { sm.lo[c] = 0; sm.hi[c] = 0; }
  for (int c = threadIdx.x; c < COV_JSLOTS; c += COV_THREADS) { sm.jkey[c] = J_EMPTY; sm.jlo[c] = 0; sm.jhi[c] = 0; }
  CovTile t; t.sm = &sm; t.diff = diff; t.jt = jt; t.status = status;
  {
    const uint32_t b0 = bid[rec0];
    t.cell0 = (long long)in.pos[rec0] + 1 + bbase[b0] - (long long)bstart[b0];
    t.tid0 = in.tid[rec0];
  }
  __syncthreads();
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint16_t* list = sm.list + warp * (32 * COV_RPT);
  // ---- classes, in list order: 0 = 1 CIGAR word, 1 = 3 words, then 2 / 4 / 5 words and longer; 7 = nothing to do
  // (past the end, or an empty CIGAR) ----
  unsigned long long cls = 0;
  uint32_t tot_lo = 0, tot_hi = 0;           // packed 10-bit counters: classes 0-2 | classes 3-5 (warp-uniform)
  auto packed = [](unsigned c, uint32_t& lo, uint32_t& hi) { lo = c < 3 ? 1u << (10 * c) : 0u; hi = (c >= 3 && c < 6) ? 1u << (10 * (c - 3)) : 0u; };
#pragma unroll 1
  for (int r0 = 0; r0 < COV_RPT; r0 += COV_BATCH) {
    uint32_t a0[COV_BATCH], a1[COV_BATCH];
#pragma unroll
    for (int k = 0; k < COV_BATCH; ++k) {
      const int64_t i = rec0 + (int64_t)(r0 + k) * COV_THREADS + threadIdx.x;
      a0[k] = 0; a1[k] = 0;
      if (i < in.n) { a0[k] = in.cig_off[i]; a1[k] = in.cig_off[i + 1]; }
    }
#pragma unroll
    for (int k = 0; k < COV_BATCH; ++k) {
      const uint32_t nc = a1[k] - a0[k];
      const unsigned c = nc == 0 ? 7u : (nc <= 5u ? (0x43120u >> (4 * (nc - 1u))) & 0xfu : 5u);
      cls |= (unsigned long long)c << (3 * (r0 + k));
      uint32_t lo, hi; packed(c, lo, hi);
      tot_lo += __reduce_add_sync(0xffffffffu, lo); tot_hi += __reduce_add_sync(0xffffffffu, hi);
    }
  }
  unsigned cnt[6], base[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) cnt[k] = ((k < 3 ? tot_lo : tot_hi) >> (10 * (k % 3))) & 1023u;
  base[0] = 0;
#pragma unroll
  for (int k = 1; k < 6; ++k) base[k] = base[k - 1] + cnt[k - 1];
  uint32_t run_lo = base[0] | (base[1] << 10) | (base[2] << 20), run_hi = base[3] | (base[4] << 10) | (base[5] << 20);   // next free entry of every class
#pragma unroll 4
  for (int r = 0; r < COV_RPT; ++r) {
    const unsigned c = (unsigned)(cls >> (3 * r)) & 7u;
    const unsigned peers = __match_any_sync(0xffffffffu, c);
    if (c < 6u) {
      const unsigned at = ((c < 3u ? run_lo : run_hi) >> (10 * (c < 3u ? c : c - 3u))) & 1023u;
      list[at + __popc(peers & ((1u << lane) - 1u))] = (uint16_t)((r << 5) | lane);
    }
    uint32_t lo, hi; packed(c, lo, hi);
    run_lo += __reduce_add_sync(0xffffffffu, lo); run_hi += __reduce_add_sync(0xffffffffu, hi);
  }
  __syncwarp();
  const int64_t wrec0 = rec0 + warp * 32;
  cov_walk_list(in, bid, bstart, bbase, list, base[5] + cnt[5], lane, wrec0, t, do_cov, do_junc, check_ops);
  __syncthreads();
  if (do_cov)
    for (int c = threadIdx.x; c < COV_TILE; c += COV_THREADS) {
      const unsigned long long v = ((unsigned long long)sm.hi[c] << 32) | sm.lo[c];
      if (v) atomicAdd((unsigned long long*)&diff[t.cell0 + c], v);
    }
  if (do_junc)
    for (int c = threadIdx.x; c < COV_JSLOTS; c += COV_THREADS) {
      const unsigned long long k64 = sm.jkey[c];
      if (k64 != J_EMPTY) junc_insert(jt, t.tid0, k64, (long long)(((unsigned long long)sm.jhi[c] << 32) | sm.jlo[c]), status);
    }
}

// ---- K8: change points and runs --------------------------------------------------------------------
struct SumNz { long long sum; long long nz; };
struct OpSumNz {
  typedef SumNz T;
  __host__ __device__ static T identity() { return SumNz{0, 0}; }
  __host__ __device__ static T combine(T a, T b) { return SumNz{a.sum + b.sum, a.nz + b.nz}; }
};
struct DiffIn {
  const long long* d;
  __device__ SumNz operator()(int64_t i) const { long long v = d[i]; return SumNz{v, v != 0 ? 1 : 0}; }
};
struct ChangeOut {
  const long long* d; long long* cppos; long long* cpdepth;
  __device__ void operator()(int64_t i, SumNz exc, SumNz inc) const {
    if (inc.nz != exc.nz) { cppos[exc.nz] = i; cpdepth[exc.nz] = inc.sum; }
  }
};

// ---- ordered per-cell walks in O(covered bases): tiecov -s and the exact path of fractional weights -------------------
// tiecov -s (sample heat-map, src/tiecov.cpp:155-185, 277-323): per base the float32 running mean of YX over the covering
// records IN STREAM ORDER (first += (YX - first) / second; second++), then ceil; the arithmetic is the reference's,
// operation by operation (IEEE single: subtract, divide, add; nothing to contract). Exact path, for weights that are not
// multiples of 2^-20 (YC written by `tiebrush --store-frac`: 1/3, 1/5 ...): the reference adds each record's weight to a
// double per base IN STREAM ORDER (addCov, src/tiecov.cpp:194-223), and the rounding of that sum depends on the order; the
// cell keeps the bit pattern of the double.
// A cell must not visit every record that MIGHT cover it (all records of the bundle whose running maximum end reaches the
// cell: a spliced read "covers" its whole intron this way). Instead every M block of every record becomes one ITEM per
// 256-cell tile it touches (first cell, last cell, record), emitted in stream order; a stable radix sort by tile keeps that
// order inside a tile; one CTA per tile then folds its items in order, each thread one cell — a cell only ever sees
// records that cover its tile.
constexpr int OW_TILE = 256;
template <bool EMIT>
__global__ void __launch_bounds__(256) ow_items_kernel(CovIn in, const uint32_t* __restrict__ bid, const int32_t* __restrict__ bstart,
                                                       const long long* __restrict__ bbase, uint32_t* __restrict__ cnt_or_off,
                                                       unsigned long long* __restrict__ ikey, uint32_t* __restrict__ ival, uint32_t* __restrict__ ilo,
                                                       uint32_t* __restrict__ ihi, uint32_t* __restrict__ irec) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= in.n) return;
  const uint32_t b = bid[i];
  const long long shift = bbase[b] - (long long)bstart[b];   // compact cell of 1-based coordinate g is g + shift
  int p = in.pos[i] + 1;
  uint32_t items = 0, w = EMIT ? cnt_or_off[i] : 0u;
  const uint32_t c1 = in.cig_off[i + 1];
  for (uint32_t c = in.cig_off[i]; c < c1; ++c) {
    const uint32_t cw = in.cigar[c];
    const uint32_t op = cw & 0xf; const int len = (int)(cw >> 4);
    if (op == TB_OP_M) {
      if (len > 0) {
        const long long x0 = (long long)p + shift, x1 = x0 + len - 1;
        for (long long t = x0 / OW_TILE; t <= x1 / OW_TILE; ++t) {
          if (EMIT) {
            const long long lo = t * OW_TILE > x0 ? t * OW_TILE : x0, hi = (t + 1) * OW_TILE - 1 < x1 ? (t + 1) * OW_TILE - 1 : x1;
            ikey[w] = (unsigned long long)t; ival[w] = w; ilo[w] = (uint32_t)lo; ihi[w] = (uint32_t)hi; irec[w] = (uint32_t)i;
            ++w;
          }
          ++items;
        }
      }
      p += len;
    } else if (op == TB_OP_D || op == TB_OP_N) p += len;
  }
  if (!EMIT) cnt_or_off[i] = items;
}
struct IcntIn { const uint32_t* c; __device__ uint32_t operator()(int64_t i) const { return c[i]; } };
struct IoffOut { uint32_t* o; int64_t n; __device__ void operator()(int64_t i, uint32_t exc, uint32_t inc) const { o[i] = exc; if (i == n - 1) o[n] = inc; } };

// MEAN = true: tiecov -s, float32 running mean of YX then ceil (addMean, tiecov.cpp:155-185); false: double sum of yc (addCov)
template <bool MEAN>
__global__ void __launch_bounds__(OW_TILE) ow_cells_kernel(const unsigned long long* __restrict__ skey, const uint32_t* __restrict__ sval, int64_t n_items,
                                                           const uint32_t* __restrict__ ilo, const uint32_t* __restrict__ ihi, const uint32_t* __restrict__ irec,
                                                           const int32_t* __restrict__ yx, const float* __restrict__ yc, long long* __restrict__ cell, int64_t L) {
  __shared__ uint32_t s_lo[OW_TILE], s_hi[OW_TILE];
  __shared__ float s_w[OW_TILE];
  __shared__ long long s_range[2];
  const long long t = blockIdx.x;
  if (threadIdx.x < 2) {   // [first, last) item of this tile in the sorted list
    const unsigned long long want = (unsigned long long)t + threadIdx.x;
    long long lo = 0, hi = n_items;
    while (lo < hi) { const long long mid = lo + ((hi - lo) >> 1); if (skey[mid] >= want) hi = mid; else lo = mid + 1; }
    s_range[threadIdx.x] = lo;
  }
  __syncthreads();
  const long long j0 = s_range[0], j1 = s_range[1];
  const long long x = t * OW_TILE + threadIdx.x;
  float mean = 0.f; unsigned long long cnt = 1; double sum = 0.0;
  for (long long base = j0; base < j1; base += OW_TILE) {
    const long long j = base + threadIdx.x;
    __syncthreads();
    if (j < j1) {
      const uint32_t it = sval[j];
      s_lo[threadIdx.x] = ilo[it]; s_hi[threadIdx.x] = ihi[it];
      const uint32_t r = irec[it];
      s_w[threadIdx.x] = MEAN ? (float)yx[r] : yc[r];
    }
    __syncthreads();
    const int m = (int)((j1 - base) < OW_TILE ? (j1 - base) : OW_TILE);
    for (int q = 0; q < m; ++q) {
      if ((uint32_t)x >= s_lo[q] && (uint32_t)x <= s_hi[q]) {
        if (MEAN) { mean += (s_w[q] - mean) / (float)cnt; ++cnt; }
        else sum += (double)s_w[q];
      }
    }
  }
  if (x < L) cell[x] = MEAN ? (long long)(unsigned long long)ceilf(mean) : __double_as_longlong(sum);
}
struct ChgIn {
  const long long* v;
  __device__ uint32_t operator()(int64_t x) const { return v[x] != (x ? v[x - 1] : 0) ? 1u : 0u; }
};
struct ChgOut {
  const long long* v; long long* cppos; long long* cpdepth;
  __device__ void operator()(int64_t x, uint32_t exc, uint32_t inc) const { if (inc != exc) { cppos[exc] = x; cpdepth[exc] = v[x]; } }
};
__global__ void cov_store_nchange_kernel(const uint32_t* tot, long long* status) { status[ST_NCHANGE] = *tot; }

// last bundle of the window: its end, reference id and first record (the caller decides whether the record that follows the
// window continues it — then the bundle is left to the next window, tc_coverage_stream)
__global__ void cov_tail_kernel(const int32_t* bend, const int32_t* btid, const uint32_t* rfirst, long long* status) {
  const long long nb = status[ST_NBUNDLES];
  if (nb < 1) return;
  status[ST_TAIL_END] = bend[nb - 1]; status[ST_TAIL_TID] = btid[nb - 1]; status[ST_TAIL_FIRST] = rfirst[nb - 1];
}
__global__ void cov_set_nbundles_kernel(long long* status, long long nb) { status[ST_NBUNDLES] = nb; }

struct RunValidIn {
  const long long* cpdepth; const long long* status;
  __device__ uint32_t operator()(int64_t k) const {
    long long K = status[ST_NCHANGE];
    return (k + 1 < K && cpdepth[k] != 0) ? 1u : 0u;
  }
};
struct RunOut {
  const long long* cppos; const long long* cpdepth; long long* status;
  const long long* bbase; const int32_t* bstart; const int32_t* btid;
  int32_t* o_tid; int32_t* o_start; int32_t* o_end; double* o_val; long long capacity; double scale;
  __device__ void operator()(int64_t k, uint32_t exc, uint32_t inc) const {
    if (inc == exc) return;
    if ((long long)exc >= capacity) { status[ST_RUNOVERFLOW] = 1; return; }
    long long c = cppos[k], c2 = cppos[k + 1];
    long long B = status[ST_NBUNDLES];
    long long lo = 0, hi = B;  // last bundle with base <= c
    while (hi - lo > 1) { long long m = (lo + hi) >> 1; if (bbase[m] <= c) lo = m; else hi = m; }
    long long off = (long long)bstart[lo] - 1 - bbase[lo];
    o_tid[exc] = btid[lo];
    o_start[exc] = (int32_t)(c + off);
    o_end[exc] = (int32_t)(c2 + off);
    o_val[exc] = scale > 0.0 ? (double)cpdepth[k] / scale : __longlong_as_double(cpdepth[k]);
  }
};

__global__ void cov_store_total_kernel(const SumNz* tot, const uint32_t* nruns, long long* status) {
  if (tot) status[ST_NCHANGE] = tot->nz;
  if (nruns) status[ST_NRUNS] = *nruns;
}

// ---- K9 extraction ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) junc_init_kernel(JTable jt, uint32_t cap) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= cap) return;
  jt.key[s] = J_EMPTY; jt.tid[s] = -1; jt.val[s] = 0;
}

__global__ void __launch_bounds__(256) junc_compact_kernel(JTable jt, uint32_t cap, unsigned long long* __restrict__ keys, uint32_t* __restrict__ idx,
                                                           unsigned long long* __restrict__ counter, long long* __restrict__ status) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= cap) return;
  if (jt.key[s] == J_EMPTY) return;
  unsigned long long k = atomicAdd(counter, 1ULL);
  keys[k] = jt.key[s];
  idx[k] = s;
}

__global__ void __launch_bounds__(256) junc_tidkey_kernel(JTable jt, const uint32_t* __restrict__ idx, int64_t J, unsigned long long* __restrict__ tkeys) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= J) return;
  tkeys[k] = (unsigned long long)(uint32_t)jt.tid[idx[k]];
}

__global__ void __launch_bounds__(256) junc_emit_kernel(JTable jt, const uint32_t* __restrict__ idx, int64_t J, int32_t* o_tid, int32_t* o_start,
                                                        int32_t* o_end, uint8_t* o_strand, double* o_val) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= J) return;
  uint32_t s = idx[k];
  unsigned long long key = jt.key[s];
  o_tid[k] = jt.tid[s];
  o_start[k] = (int32_t)(key >> 33);
  o_end[k] = (int32_t)((key >> 2) & 0x7fffffffULL);
  o_strand[k] = strand_char((unsigned)(key & 3));
  o_val[k] = (double)jt.val[s] / COV_FX_SCALE;
}

// EXACT junction values for weights that are not multiples of 2^-20: the reference adds each record's weight to a double per
// junction in stream order (addJunction, src/tiecov.cpp:100-112). One thread per emitted junction row walks the records of
// its bundle that start before the junction and reach beyond it, re-runs the exon state machine of setupCoordinates on each
// and adds (double)yc when the record has this very junction on this strand.
__global__ void __launch_bounds__(128) junc_exact_kernel(CovIn in, int64_t NB, const int32_t* __restrict__ btid, const int32_t* __restrict__ bstart,
                                                         const uint32_t* __restrict__ rfirst, const uint32_t* __restrict__ pmend, int64_t J,
                                                         const int32_t* __restrict__ o_tid, const int32_t* __restrict__ o_start, const int32_t* __restrict__ o_end,
                                                         const uint8_t* __restrict__ o_strand, double* __restrict__ o_val) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= J) return;
  const int tid = o_tid[k], js = o_start[k], je = o_end[k];
  const unsigned sc = strand_code(o_strand[k]);
  int64_t lo = 0, hi = NB;   // last bundle with (tid, start) <= (tid, js)
  while (hi - lo > 1) { const int64_t m = (lo + hi) >> 1; if (btid[m] < tid || (btid[m] == tid && bstart[m] <= js)) lo = m; else hi = m; }
  const uint32_t r0 = rfirst[lo], r1 = lo + 1 < NB ? rfirst[lo + 1] : (uint32_t)in.n;
  uint32_t a = r0, z = r1;   // first record whose running maximum end reaches beyond the junction
  while (a < z) { const uint32_t m = a + ((z - a) >> 1); if (pmend[m] > (uint32_t)je) z = m; else a = m + 1; }
  const uint32_t first = a;
  a = first; z = r1;         // first record that starts at or after the junction
  while (a < z) { const uint32_t m = a + ((z - a) >> 1); if (in.pos[m] + 1 >= js) z = m; else a = m + 1; }
  const uint32_t last = a;
  double sum = 0.0;
  for (uint32_t i = first; i < last; ++i) {
    if (strand_code(in.strand[i]) != sc) continue;
    const int pos = in.pos[i];
    int l = 0, exstart = pos, nclosed = 0, last_end = 0;
    bool intron = false, ins = false, hit = false;
    const uint32_t c1 = in.cig_off[i + 1];
    for (uint32_t c = in.cig_off[i]; c < c1 && !hit; ++c) {
      const uint32_t cw = in.cigar[c];
      const uint32_t op = cw & 0xf; const int len = (int)(cw >> 4);
      if (op == TB_OP_N) {
        if (!ins || !intron) {
          if (nclosed > 0 && last_end + 1 == js && exstart == je) hit = true;
          last_end = pos + l; nclosed++;
        }
        exstart = pos + l + len;
      }
      const bool refc = (0x18Du >> op) & 1u;
      const bool known = (0x1BFu >> op) & 1u;
      l += refc ? len : 0;
      if (known) {
        ins = (op == TB_OP_I) || (op == TB_OP_N && ins);
        intron = (op == TB_OP_N) || (op == TB_OP_I && intron);
      }
      if (last_end + 1 > js) break;   // the exons closed so far already end beyond the junction's start
    }
    if (!hit && nclosed > 0 && last_end + 1 == js && exstart == je) hit = true;   // the junction that ends at the last exon
    if (hit) sum += (double)in.yc[i];
  }
  o_val[k] = sum;
}

static inline unsigned grid_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

template <class T>
static int stage_in(tb_ctx* ctx, DevBuf& b, const T* src, size_t count, int on_device, const T** out) {
  if (on_device || src == nullptr) { *out = src; return 0; }
  TB_CUDA(b.ensure(count * sizeof(T) + 16));
  TB_CUDA(cudaMemcpyAsync(b.p, src, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  *out = (const T*)b.p;
  return 0;
}

}  // namespace

int tc_coverage_impl(tb_ctx* ctx, const tc_soa_in* hin, tc_runs_out* runs, tc_juncs_out* juncs, const int32_t* yx_in, CovExt* ext) {
  TB_CUDA(cudaSetDevice(ctx->device));
  int64_t n = hin->n;   // records processed: all of the window, or (tc_coverage_stream) all but its open last bundle
  if (runs) runs->n_runs = 0;
  if (juncs) juncs->n_juncs = 0;
  if (n == 0) return 0;
  if (n >= (1LL << 31)) { ctx->set_error("tc_coverage_window: n=%lld too large for one window", (long long)n); return 1; }
  const bool sample = yx_in != nullptr;   // tiecov -s: runs = rows of the sample heat-map (value = ceil of the running mean of YX)
  const int do_cov = runs != nullptr, do_junc = juncs != nullptr && !sample;
  cudaStream_t st = ctx->stream;

  // ---- inputs on the device ----
  CovIn in; in.n = n;
  int64_t ncig = hin->n_cig;
  if (stage_in(ctx, ctx->in_stage[0], hin->tid, (size_t)n, hin->on_device, &in.tid)) return 1;
  if (stage_in(ctx, ctx->in_stage[1], hin->pos, (size_t)n, hin->on_device, &in.pos)) return 1;
  if (stage_in(ctx, ctx->in_stage[2], hin->yc, (size_t)n, hin->on_device, &in.yc)) return 1;
  if (stage_in(ctx, ctx->in_stage[3], hin->strand, (size_t)n, hin->on_device, &in.strand)) return 1;
  if (stage_in(ctx, ctx->in_stage[4], hin->cig_off, (size_t)n + 1, hin->on_device, &in.cig_off)) return 1;
  {
    // host arrays: a window of a longer stream keeps its absolute CIGAR offsets (tc_coverage_stream): copy the window's
    // words only and bias the device pointer so that cigar[cig_off[i]] still lands on them
    const uint32_t cbase = (!hin->on_device && n > 0) ? hin->cig_off[0] : 0u;
    const uint32_t* staged = nullptr;
    if (stage_in(ctx, ctx->in_stage[5], hin->cigar ? hin->cigar + cbase : nullptr, (size_t)ncig, hin->on_device, &staged)) return 1;
    in.cigar = staged - cbase;
  }
  in.end = nullptr;
  if (hin->end) { if (stage_in(ctx, ctx->in_stage[7], hin->end, (size_t)n, hin->on_device, &in.end)) return 1; }
  const int32_t* d_yx = nullptr;
  if (sample) { if (stage_in(ctx, ctx->in_stage[6], yx_in, (size_t)n, hin->on_device, &d_yx)) return 1; }

  DevBuf* B = ctx->buf;
  TB_CUDA(B[CB_RFIRST].ensure(sizeof(uint32_t) * n));
  uint32_t* d_pmend = nullptr;   // set and filled only when the exact path turns out to be needed
  uint32_t* d_rfirst = B[CB_RFIRST].as<uint32_t>();
  TB_CUDA(B[CB_KEY].ensure(sizeof(uint64_t) * (2 * (size_t)((n + CBK_TILE - 1) / CBK_TILE) + 16)));
  TB_CUDA(B[CB_BID].ensure(sizeof(uint32_t) * n));
  TB_CUDA(B[CB_BSTART].ensure(sizeof(int32_t) * n));
  TB_CUDA(B[CB_BEND].ensure(sizeof(int32_t) * n));
  TB_CUDA(B[CB_BTID].ensure(sizeof(int32_t) * n));
  TB_CUDA(B[CB_BBASE].ensure(sizeof(int64_t) * (n + 1)));
  TB_CUDA(B[CB_STATUS].ensure(sizeof(int64_t) * 16));
  TB_CUDA(ctx->pinned[0].ensure(sizeof(int64_t) * 16));
  long long* d_status = B[CB_STATUS].as<long long>();
  long long* h_status = ctx->pinned[0].as<long long>();
  {
    long long init[16]; memset(init, 0, sizeof(init)); init[ST_ERRIDX] = -1;  // as u64: max
    memcpy(h_status, init, sizeof(init));
    TB_CUDA(cudaMemcpyAsync(d_status, h_status, sizeof(init), cudaMemcpyHostToDevice, st));
    TB_CUDA(cudaStreamSynchronize(st));  // h_status is reused for readback below
  }
  // ---- K6 ----
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[8], st));
  auto launch_k6 = [&](bool use_end) -> int {
    const int64_t ntiles = (n + CBK_TILE - 1) / CBK_TILE;
    const bool vec = (((uintptr_t)in.pos | (uintptr_t)in.tid | (uintptr_t)in.cig_off | (uintptr_t)in.yc | (uintptr_t)in.end) & 15u) == 0;
    if (use_end) {   // three streaming passes (see cbk_tilemax_kernel)
      const int64_t sb = tb_scan_blocks(ntiles) + 8;
      TB_CUDA(B[CB_KEY].ensure(sizeof(uint64_t) * ((size_t)ntiles * (3 + CBK_THREADS / 4) + (size_t)sb + 16)));
      unsigned long long* tmax = B[CB_KEY].as<unsigned long long>();
      unsigned long long* tpre = tmax + ntiles;
      unsigned long long* agg = tpre + ntiles;
      uint32_t* theads = reinterpret_cast<uint32_t*>(agg + sb);
      uint32_t* thbase = theads + ntiles;
      uint16_t* masks = reinterpret_cast<uint16_t*>(thbase + ntiles);
      if (vec) cbk_tilemax_kernel<true><<<(unsigned)ntiles, CBK_THREADS, 0, st>>>(in, tmax);
      else cbk_tilemax_kernel<false><<<(unsigned)ntiles, CBK_THREADS, 0, st>>>(in, tmax);
      TB_CUDA((tb_device_scan<OpMaxU64>(ctx, TileU64In{tmax}, ntiles, agg, TileU64Exc{tpre})));
      if (vec) cbk_heads_kernel<true><<<(unsigned)ntiles, CBK_THREADS, 0, st>>>(in, tpre, masks, theads, B[CB_BID].as<uint32_t>(), d_status);
      else cbk_heads_kernel<false><<<(unsigned)ntiles, CBK_THREADS, 0, st>>>(in, tpre, masks, theads, B[CB_BID].as<uint32_t>(), d_status);
      TB_CUDA((tb_device_scan<OpSumU32>(ctx, TileU32In{theads}, ntiles, reinterpret_cast<uint32_t*>(agg), TileU32Exc{thbase})));
      cbk_write_kernel<<<(unsigned)ntiles, CBK_THREADS, 0, st>>>(in, masks, thbase, tpre, tmax, B[CB_BID].as<uint32_t>(), B[CB_BSTART].as<int32_t>(),
                                                              B[CB_BEND].as<int32_t>(), B[CB_BTID].as<int32_t>(), d_rfirst, d_status);
      ctx->launches += 3;
      return 0;
    }
    unsigned long long* st_max = B[CB_KEY].as<unsigned long long>();
    unsigned long long* st_cnt = st_max + ntiles;
    unsigned long long* ticket = st_cnt + ntiles;
    TB_CUDA(cudaMemsetAsync(st_max, 0, sizeof(uint64_t) * (2 * (size_t)ntiles + 8), st));
    auto* k6 = vec ? cov_bundle_kernel<true> : cov_bundle_kernel<false>;
    k6<<<(unsigned)ntiles, CBK_THREADS, 0, st>>>(in, do_cov, st_max, st_cnt, ticket, B[CB_BID].as<uint32_t>(), B[CB_BSTART].as<int32_t>(),
                                                 B[CB_BEND].as<int32_t>(), B[CB_BTID].as<int32_t>(), d_pmend, d_rfirst, d_status);
    ctx->launches++;
    return 0;
  };
  // -s ignores the end column: the accumulate kernel does not run on -s, so the look-back K6 (which walks the CIGARs) is
  // the only kernel there that rejects unsupported ops
  const bool has_end = in.end != nullptr && !sample;
  if (launch_k6(has_end)) return 1;
  if (ext) { cov_tail_kernel<<<1, 1, 0, st>>>(B[CB_BEND].as<int32_t>(), B[CB_BTID].as<int32_t>(), d_rfirst, d_status); ctx->launches++; }
  // the bundle count decides the size of the next scan
  TB_CUDA(cudaMemcpyAsync(h_status, d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
  TB_CUDA(cudaStreamSynchronize(st));
  if (h_status[ST_LBFAIL]) { ctx->set_error("tc_coverage_window: bundle scan did not make progress (internal error)"); return 1; }
  if (ext) {
    // tc_coverage_stream: the record that follows the window continues its last bundle -> leave that bundle to the next window
    ext->consumed = n;
    if (ext->has_next && ext->next_tid == (int32_t)h_status[ST_TAIL_TID] && (long long)ext->next_pos + 1 <= h_status[ST_TAIL_END]) {
      if (h_status[ST_NBUNDLES] <= 1) { ext->consumed = 0; return 3; }   // one bundle spans the whole window: the caller enlarges it
      const int64_t keep = h_status[ST_TAIL_FIRST];
      ext->consumed = keep;
      cov_set_nbundles_kernel<<<1, 1, 0, st>>>(d_status, h_status[ST_NBUNDLES] - 1);
      ctx->launches++;
      h_status[ST_NBUNDLES] -= 1;
      in.n = keep;
    }
  }
  const int64_t n_full = n;
  n = in.n;
  // weights that are not multiples of 2^-20 (YC of `tiebrush --store-frac`): the fixed-point sums would differ from the
  // reference's ordered double sums -> exact path (one ordered walk per cell / per junction). Never silent.
  const bool exact = !sample && h_status[ST_INEXACT] != 0;
  ctx->last_cov_exact = exact ? 1 : 0;
  if (exact) {
    TB_CUDA(B[CB_PMEND].ensure(sizeof(uint32_t) * n_full));
    d_pmend = B[CB_PMEND].as<uint32_t>();
    const int64_t nb_keep = h_status[ST_NBUNDLES];
    const int64_t n_eff = n;
    in.n = n_full; n = n_full;
    if (launch_k6(false)) return 1;     // second run: also the running maximum of the ends (pmend) for junc_exact_kernel (walks the CIGARs: op check)
    in.n = n_eff; n = n_eff;
    cov_set_nbundles_kernel<<<1, 1, 0, st>>>(d_status, nb_keep);
    ctx->launches++;
  }
  const int64_t NB = h_status[ST_NBUNDLES];
  size_t agg_bytes = (size_t)(tb_scan_blocks(n > 2 * ncig + 16 ? n : 2 * ncig + 16) + 8) * sizeof(SumNz);
  TB_CUDA(B[CB_AGG].ensure(agg_bytes));
  TB_CUDA((tb_device_scan<OpSumI64>(ctx, BLenIn{B[CB_BSTART].as<int32_t>(), B[CB_BEND].as<int32_t>(), d_status}, NB,
                                    B[CB_AGG].as<long long>(), BBaseOut{B[CB_BBASE].as<long long>()})));
  cov_publish_kernel<<<1, 1, 0, st>>>(B[CB_AGG].as<long long>() + tb_scan_blocks(NB), d_status);
  ctx->launches++;
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[9], st));
  TB_CUDA(cudaMemcpyAsync(h_status, d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
  TB_CUDA(cudaStreamSynchronize(st));
  if (h_status[ST_ERRIDX] != -1) {
    ctx->set_error("ERROR: unknown opcode in CIGAR of record %lld (tiecov supports only M,I,D,N,S; n_cigar<256)", h_status[ST_ERRIDX]);
    return 2;
  }
  const int64_t L = h_status[ST_DENSE_LEN];
  {
    int64_t m = L > n ? L : n; if (2 * ncig + 16 > m) m = 2 * ncig + 16;
    TB_CUDA(B[CB_AGG].ensure((size_t)(tb_scan_blocks(m) + 8) * sizeof(SumNz)));
  }

  // ---- junction table ----
  JTable jt; memset(&jt, 0, sizeof(jt));
  uint32_t jcap = 1024;
  if (do_junc) {
    int64_t want = 2 * ncig; if (want > (1 << 22)) want = 1 << 22;
    while ((int64_t)jcap < want) jcap <<= 1;
  }
  uint64_t seed = 0x9e3779b97f4a7c15ULL;
  const bool cells = sample || (exact && do_cov);   // a per-cell value array takes the place of the difference array
  if (cells) {
    TB_CUDA(B[CB_DIFF].ensure(sizeof(int64_t) * (L + 1)));
    if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[0], st));
    if (L >= (1LL << 32)) { ctx->set_error("tc_coverage_window: %lld cells do not fit the 32-bit item lists (smaller windows)", (long long)L); return 1; }
    TB_CUDA(B[CB_IOFF].ensure(sizeof(uint32_t) * (n + 2)));
    uint32_t* ioff = B[CB_IOFF].as<uint32_t>();
    ow_items_kernel<false><<<grid_for(n, 256), 256, 0, st>>>(in, B[CB_BID].as<uint32_t>(), B[CB_BSTART].as<int32_t>(), B[CB_BBASE].as<long long>(), ioff,
                                                            nullptr, nullptr, nullptr, nullptr, nullptr);
    TB_CUDA(B[CB_AGG].ensure((size_t)(tb_scan_blocks(n) + 8) * sizeof(SumNz)));
    TB_CUDA((tb_device_scan<OpSumU32>(ctx, IcntIn{ioff}, n, B[CB_AGG].as<uint32_t>(), IoffOut{ioff, n})));
    uint32_t n_items_u = 0;
    TB_CUDA(cudaMemcpyAsync(&n_items_u, ioff + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    const int64_t NI = n_items_u;
    const int64_t nalloc = NI > 0 ? NI : 1;
    TB_CUDA(B[CB_IKEY].ensure(sizeof(uint64_t) * nalloc)); TB_CUDA(B[CB_IKEY2].ensure(sizeof(uint64_t) * nalloc));
    TB_CUDA(B[CB_IVAL].ensure(sizeof(uint32_t) * nalloc)); TB_CUDA(B[CB_IVAL2].ensure(sizeof(uint32_t) * nalloc));
    TB_CUDA(B[CB_ILO].ensure(sizeof(uint32_t) * nalloc)); TB_CUDA(B[CB_IHI].ensure(sizeof(uint32_t) * nalloc)); TB_CUDA(B[CB_IREC].ensure(sizeof(uint32_t) * nalloc));
    ow_items_kernel<true><<<grid_for(n, 256), 256, 0, st>>>(in, B[CB_BID].as<uint32_t>(), B[CB_BSTART].as<int32_t>(), B[CB_BBASE].as<long long>(), ioff,
                                                           B[CB_IKEY].as<unsigned long long>(), B[CB_IVAL].as<uint32_t>(), B[CB_ILO].as<uint32_t>(),
                                                           B[CB_IHI].as<uint32_t>(), B[CB_IREC].as<uint32_t>());
    ctx->launches += 2;
    const int64_t ntile = (L + OW_TILE - 1) / OW_TILE;
    int bits = 1; while ((1LL << bits) < ntile + 1) ++bits;
    uint64_t* rk = B[CB_IKEY].as<uint64_t>(); uint32_t* rv = B[CB_IVAL].as<uint32_t>();
    if (NI > 0) {
      TB_CUDA(B[CB_RSTABLE].ensure(sizeof(uint32_t) * tb_radix_table_elems(NI)));
      TB_CUDA(B[CB_RSAGG].ensure(sizeof(uint32_t) * tb_radix_agg_elems(NI)));
      TB_CUDA(tb_radix_sort(ctx, B[CB_IKEY].as<uint64_t>(), B[CB_IVAL].as<uint32_t>(), B[CB_IKEY2].as<uint64_t>(), B[CB_IVAL2].as<uint32_t>(), NI, 0, bits,
                            B[CB_RSTABLE].as<uint32_t>(), B[CB_RSAGG].as<uint32_t>(), &rk, &rv));
    }
    if (sample)
      ow_cells_kernel<true><<<(unsigned)ntile, OW_TILE, 0, st>>>((const unsigned long long*)rk, rv, NI, B[CB_ILO].as<uint32_t>(), B[CB_IHI].as<uint32_t>(), B[CB_IREC].as<uint32_t>(),
                                                                d_yx, in.yc, B[CB_DIFF].as<long long>(), L);
    else
      ow_cells_kernel<false><<<(unsigned)ntile, OW_TILE, 0, st>>>((const unsigned long long*)rk, rv, NI, B[CB_ILO].as<uint32_t>(), B[CB_IHI].as<uint32_t>(), B[CB_IREC].as<uint32_t>(),
                                                                 d_yx, in.yc, B[CB_DIFF].as<long long>(), L);
    ctx->launches++;
    if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[1], st));
  }
  const int acc_cov = do_cov && !cells;   // the accumulate kernel still finds the junction keys on the exact path
  if (!sample && (acc_cov || do_junc))
  for (int attempt = 0;; ++attempt) {
    if (do_junc) {
      TB_CUDA(B[CB_JTAG].ensure(sizeof(uint64_t) * jcap));
      TB_CUDA(B[CB_JTID].ensure(sizeof(int32_t) * jcap));
      TB_CUDA(B[CB_JVAL].ensure(sizeof(int64_t) * jcap));
      jt.key = B[CB_JTAG].as<unsigned long long>(); jt.tid = B[CB_JTID].as<int32_t>(); jt.val = B[CB_JVAL].as<long long>();
      jt.mask = jcap - 1; jt.seed = seed;
      junc_init_kernel<<<grid_for(jcap, 256), 256, 0, st>>>(jt, jcap);
      ctx->launches++;
    }
    if (acc_cov) {
      TB_CUDA(B[CB_DIFF].ensure(sizeof(int64_t) * (L + 1)));
      TB_CUDA(cudaMemsetAsync(B[CB_DIFF].p, 0, sizeof(int64_t) * (L + 1), st));
    }
    // ---- K7 (+K9 insert): the dominant kernel ----
    if (ctx->profiling && !cells) TB_CUDA(cudaEventRecord(ctx->ev[0], st));
    cov_accumulate_kernel<<<grid_for(n, COV_THREADS * COV_RPT), COV_THREADS, 0, st>>>(in, B[CB_BID].as<uint32_t>(), B[CB_BSTART].as<int32_t>(), B[CB_BBASE].as<long long>(),
                                                           B[CB_DIFF].as<long long>(), acc_cov, do_junc, jt, d_status, (has_end && do_cov) ? 1 : 0);
    ctx->launches++;
    if (ctx->profiling && !cells) TB_CUDA(cudaEventRecord(ctx->ev[1], st));
    if (!do_junc) break;
    TB_CUDA(cudaMemcpyAsync(h_status, d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    bool overflow = h_status[ST_JOVERFLOW] != 0 || h_status[ST_NJUNC] * 2 > (int64_t)jcap;
    if (!overflow) break;
    if (attempt > 8 || jcap >= (1u << 30)) { ctx->set_error("junction table overflow (%lld distinct junctions)", h_status[ST_NJUNC]); return 1; }
    jcap <<= 2;
    h_status[ST_JOVERFLOW] = 0; h_status[ST_NJUNC] = 0;
    TB_CUDA(cudaMemcpyAsync(d_status, h_status, sizeof(int64_t) * 16, cudaMemcpyHostToDevice, st));
    TB_CUDA(cudaStreamSynchronize(st));
  }

  // ---- K8 ----
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[10], st));
  if (do_cov) {
    // change points: at most one per non-zero difference cell, and no more than two per M block
    int64_t kmax = 2 * ncig + 16; if (L + 1 < kmax) kmax = L + 1;
    TB_CUDA(B[CB_CPPOS].ensure(sizeof(int64_t) * kmax));
    TB_CUDA(B[CB_CPDEPTH].ensure(sizeof(int64_t) * kmax));
    long long* d_diff = B[CB_DIFF].as<long long>();
    long long* cppos = B[CB_CPPOS].as<long long>();
    long long* cpdepth = B[CB_CPDEPTH].as<long long>();
    if (cells) {
      TB_CUDA((tb_device_scan<OpSumU32>(ctx, ChgIn{d_diff}, L, B[CB_AGG].as<uint32_t>(), ChgOut{d_diff, cppos, cpdepth})));
      cov_store_nchange_kernel<<<1, 1, 0, st>>>(B[CB_AGG].as<uint32_t>() + tb_scan_blocks(L), d_status);
    } else {
      TB_CUDA((tb_device_scan<OpSumNz>(ctx, DiffIn{d_diff}, L, B[CB_AGG].as<SumNz>(), ChangeOut{d_diff, cppos, cpdepth})));
      cov_store_total_kernel<<<1, 1, 0, st>>>(B[CB_AGG].as<SumNz>() + tb_scan_blocks(L), nullptr, d_status);
    }
    ctx->launches++;
    // the number of change points is only known on the device
    TB_CUDA(cudaMemcpyAsync(h_status, d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    if (h_status[ST_ERRIDX] != -1) {   // found by K7 when the packer supplied the ends (K6 did not walk the CIGARs)
      ctx->set_error("ERROR: unknown opcode in CIGAR of record %lld (tiecov supports only M,I,D,N,S; n_cigar<256)", h_status[ST_ERRIDX]);
      return 2;
    }
    const int64_t K = h_status[ST_NCHANGE];
    // output staging
    int64_t cap = runs->capacity;
    int32_t *o_tid = runs->tid, *o_start = runs->start0, *o_end = runs->end0; double* o_val = runs->value;
    int64_t stage_cap = cap < K ? cap : K;
    if (stage_cap < 1) stage_cap = 1;
    if (!runs->on_device) {
      TB_CUDA(ctx->out_stage[0].ensure(sizeof(int32_t) * stage_cap)); TB_CUDA(ctx->out_stage[1].ensure(sizeof(int32_t) * stage_cap));
      TB_CUDA(ctx->out_stage[2].ensure(sizeof(int32_t) * stage_cap)); TB_CUDA(ctx->out_stage[3].ensure(sizeof(double) * stage_cap));
      o_tid = ctx->out_stage[0].as<int32_t>(); o_start = ctx->out_stage[1].as<int32_t>(); o_end = ctx->out_stage[2].as<int32_t>();
      o_val = ctx->out_stage[3].as<double>();
    }
    RunOut ro{cppos, cpdepth, d_status, B[CB_BBASE].as<long long>(), B[CB_BSTART].as<int32_t>(), B[CB_BTID].as<int32_t>(),
              o_tid, o_start, o_end, o_val, stage_cap, sample ? 1.0 : (cells ? 0.0 : COV_FX_SCALE)};
    TB_CUDA((tb_device_scan<OpSumU32>(ctx, RunValidIn{cpdepth, d_status}, K, B[CB_AGG].as<uint32_t>(), ro)));
    cov_store_total_kernel<<<1, 1, 0, st>>>(nullptr, B[CB_AGG].as<uint32_t>() + tb_scan_blocks(K), d_status);
    ctx->launches++;
  }
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[11], st));
  TB_CUDA(cudaMemcpyAsync(h_status, d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
  TB_CUDA(cudaStreamSynchronize(st));
  if (ctx->profiling) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]) == cudaSuccess) ctx->last_ms[1] = ms;
    if (cudaEventElapsedTime(&ms, ctx->ev[8], ctx->ev[9]) == cudaSuccess) ctx->last_ms[6] = ms;
    if (cudaEventElapsedTime(&ms, ctx->ev[10], ctx->ev[11]) == cudaSuccess) ctx->last_ms[7] = ms;
  }
  if (do_cov) {
    if (h_status[ST_RUNOVERFLOW] || h_status[ST_NRUNS] > runs->capacity) {
      ctx->set_error("tc_coverage_window: runs capacity %lld too small (%lld runs)", (long long)runs->capacity, h_status[ST_NRUNS]);
      return 1;
    }
    runs->n_runs = h_status[ST_NRUNS];
    if (!runs->on_device && runs->n_runs > 0) {
      size_t r = (size_t)runs->n_runs;
      TB_CUDA(cudaMemcpyAsync(runs->tid, ctx->out_stage[0].p, sizeof(int32_t) * r, cudaMemcpyDeviceToHost, st));
      TB_CUDA(cudaMemcpyAsync(runs->start0, ctx->out_stage[1].p, sizeof(int32_t) * r, cudaMemcpyDeviceToHost, st));
      TB_CUDA(cudaMemcpyAsync(runs->end0, ctx->out_stage[2].p, sizeof(int32_t) * r, cudaMemcpyDeviceToHost, st));
      TB_CUDA(cudaMemcpyAsync(runs->value, ctx->out_stage[3].p, sizeof(double) * r, cudaMemcpyDeviceToHost, st));
    }
  }
  // ---- K9 extraction: compact, verify, sort (start,end,strand) then stable by tid ----
  if (do_junc) {
    int64_t J = h_status[ST_NJUNC];
    if (J > juncs->capacity) { ctx->set_error("tc_coverage_window: junction capacity %lld too small (%lld)", (long long)juncs->capacity, (long long)J); return 1; }
    if (J > 0) {
      TB_CUDA(B[CB_JKEYS].ensure(sizeof(uint64_t) * J)); TB_CUDA(B[CB_JKEYS2].ensure(sizeof(uint64_t) * J));
      TB_CUDA(B[CB_JIDX].ensure(sizeof(uint32_t) * J)); TB_CUDA(B[CB_JIDX2].ensure(sizeof(uint32_t) * J));
      TB_CUDA(B[CB_TIDKEYS].ensure(sizeof(uint64_t) * J)); TB_CUDA(B[CB_TIDKEYS2].ensure(sizeof(uint64_t) * J));
      TB_CUDA(B[CB_RSTABLE].ensure(sizeof(uint32_t) * tb_radix_table_elems(J)));
      TB_CUDA(B[CB_RSAGG].ensure(sizeof(uint32_t) * tb_radix_agg_elems(J)));
      unsigned long long* counter = (unsigned long long*)(d_status + ST_N_);
      TB_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), st));
      junc_compact_kernel<<<grid_for(jcap, 256), 256, 0, st>>>(jt, jcap, B[CB_JKEYS].as<unsigned long long>(), B[CB_JIDX].as<uint32_t>(), counter, d_status);
      ctx->launches++;
      uint64_t* rk; uint32_t* rv;
      TB_CUDA(tb_radix_sort(ctx, B[CB_JKEYS].as<uint64_t>(), B[CB_JIDX].as<uint32_t>(), B[CB_JKEYS2].as<uint64_t>(), B[CB_JIDX2].as<uint32_t>(), J, 0, 64,
                            B[CB_RSTABLE].as<uint32_t>(), B[CB_RSAGG].as<uint32_t>(), &rk, &rv));
      // stable second sort by tid (31 significant bits)
      uint32_t* other_v = (rv == B[CB_JIDX].as<uint32_t>()) ? B[CB_JIDX2].as<uint32_t>() : B[CB_JIDX].as<uint32_t>();
      junc_tidkey_kernel<<<grid_for(J, 256), 256, 0, st>>>(jt, rv, J, B[CB_TIDKEYS].as<unsigned long long>());
      ctx->launches++;
      uint64_t* rk2; uint32_t* rv2;
      TB_CUDA(tb_radix_sort(ctx, B[CB_TIDKEYS].as<uint64_t>(), rv, B[CB_TIDKEYS2].as<uint64_t>(), other_v, J, 0, 32,
                            B[CB_RSTABLE].as<uint32_t>(), B[CB_RSAGG].as<uint32_t>(), &rk2, &rv2));
      int32_t *o_tid = juncs->tid, *o_start = juncs->start, *o_end = juncs->end; uint8_t* o_strand = juncs->strand; double* o_val = juncs->value;
      if (!juncs->on_device) {
        TB_CUDA(ctx->out_stage[4].ensure(sizeof(int32_t) * 3 * J)); TB_CUDA(ctx->out_stage[5].ensure(J)); TB_CUDA(ctx->out_stage[6].ensure(sizeof(double) * J));
        o_tid = ctx->out_stage[4].as<int32_t>(); o_start = o_tid + J; o_end = o_start + J; o_strand = ctx->out_stage[5].as<uint8_t>(); o_val = ctx->out_stage[6].as<double>();
      }
      junc_emit_kernel<<<grid_for(J, 256), 256, 0, st>>>(jt, rv2, J, o_tid, o_start, o_end, o_strand, o_val);
      ctx->launches++;
      if (exact) {   // ordered double sums replace the fixed-point values
        junc_exact_kernel<<<grid_for(J, 128), 128, 0, st>>>(in, NB, B[CB_BTID].as<int32_t>(), B[CB_BSTART].as<int32_t>(), d_rfirst, d_pmend, J,
                                                           o_tid, o_start, o_end, o_strand, o_val);
        ctx->launches++;
      }
      if (!juncs->on_device) {
        TB_CUDA(cudaMemcpyAsync(juncs->tid, o_tid, sizeof(int32_t) * J, cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaMemcpyAsync(juncs->start, o_start, sizeof(int32_t) * J, cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaMemcpyAsync(juncs->end, o_end, sizeof(int32_t) * J, cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaMemcpyAsync(juncs->strand, o_strand, (size_t)J, cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaMemcpyAsync(juncs->value, o_val, sizeof(double) * J, cudaMemcpyDeviceToHost, st));
      }
      TB_CUDA(cudaMemcpyAsync(h_status, d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
    }
    TB_CUDA(cudaStreamSynchronize(st));
    juncs->n_juncs = J;
  }
  TB_CUDA(cudaStreamSynchronize(st));
  return 0;
}
