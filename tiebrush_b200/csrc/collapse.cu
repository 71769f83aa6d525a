// collapse.cu — driver of tiebrush's hot path on the device (tb_collapse_window): k-way merge of the per-sample
// sorted runs, grouping of duplicate alignments per start position, YC / YX / YD and the representative
// (reference src/tmerge.cpp:331-344, src/tmerge.h:28-50, src/tiebrush.cpp:275-345, 350-541).
//
//   C1 histogram   cnt[pos-pos_lo] += run length   (one RED per run of equal positions inside a warp)
//   C2 scan        P[p] = #records with pos < p    (merged-order rank of every start position: the flush boundary of
//                                                   flushPData, tiebrush.cpp:577-585, is a change of start position)
//   front end      collapse_tile.cu (order-independent grouping, the fast path) or collapse_ordered.cu (exact
//                  emulation of the reference's sorted-list search for -F / -A / TieBrush-made inputs / --store-frac,
//                  and the fallback when one position holds more distinct alignments than a shared-memory table)
//   C7 YD          collapse_yd.cu
#include "collapse_internal.cuh"

namespace {

// C1: histogram of start positions. Runs are coordinate sorted, so equal positions are adjacent: the first lane of
// every run of equal positions inside a warp adds the run length (pile-ups would otherwise serialise on one address).
__global__ void __launch_bounds__(256) col_hist_kernel(ColIn in, uint32_t* __restrict__ cnt, long long* __restrict__ status) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31;
  long long rel = -1 - (long long)lane;   // distinct sentinels for lanes past the end
  bool ok = false;
  if (i < in.n) {
    rel = (long long)in.pos[i] - in.pos_lo;
    ok = rel >= 0 && rel < (long long)in.span;
    if (!ok) { status[CS_ERR] = ERR_POS_RANGE; atomicMin((unsigned long long*)&status[CS_ERRIDX], (unsigned long long)i); rel = -1 - (long long)lane; }
    else if ((in.keep_bits & TB_KEEP_UNMAP) && (in.flag[i] & 0x4)) {
      // the reference aborts on a real unmapped read under -M (GVec invalid index in flushPData, SURVEY §9.4): parity is an error
      status[CS_ERR] = 3; atomicMin((unsigned long long*)&status[CS_ERRIDX], (unsigned long long)i);
    }
  }
  const long long prev = __shfl_up_sync(0xffffffffu, rel, 1);
  const bool head = lane == 0 || prev != rel;
  const unsigned heads = __ballot_sync(0xffffffffu, head);
  if (head && ok) {
    const unsigned after = heads & ~((2u << lane) - 1u);          // heads above this lane
    const unsigned next = after ? (unsigned)(__ffs(after) - 1) : 32u;
    atomicAdd(&cnt[rel], next - lane);
  }
}

// compact wire format (tb_soa_in.n_cigar8 / cigar16 / cigar_ext): rebuild the wide CIGAR columns on the device
struct Nc8In { const uint8_t* c; __device__ uint32_t operator()(int64_t i) const { return c[i]; } };
struct OffOut {
  uint32_t* off; int64_t n;
  __device__ void operator()(int64_t i, uint32_t exc, uint32_t inc) const { off[i] = exc; if (i == n - 1) off[n] = inc; }
};
struct EscIn { const uint16_t* c; __device__ uint32_t operator()(int64_t j) const { return (c[j] >> 4) == 0xFFFu ? 1u : 0u; } };
struct ExpandOut {
  const uint16_t* c; const uint32_t* ext; uint32_t* out;
  __device__ void operator()(int64_t j, uint32_t exc, uint32_t inc) const {
    const uint32_t w = c[j];
    const uint32_t len = inc != exc ? ext[exc] : (w >> 4);   // escaped length = the next entry of cigar_ext, in op order
    out[j] = (w & 0xfu) | (len << 4);
  }
};

// compact wire format: a scan total against what the packer declared (status[CS_ERR] = code on mismatch)
__global__ void col_check_total_kernel(const uint32_t* tot, unsigned long long want, long long* status, int code) {
  if ((unsigned long long)*tot != want) { status[CS_ERR] = code; status[CS_ERRIDX] = (long long)*tot; }
}

// packed wire format of the fixed columns (tb_soa_in.pos_d8 / meta8): rebuilt on the device by scans
struct PosEscIn { const uint8_t* d; __device__ uint32_t operator()(int64_t i) const { return d[i] >= 254 ? 1u : 0u; } };
struct PosValOut {   // delta (or absolute position) of every record; escaped ones take the next entry of pos_ext
  const uint8_t* d; const int32_t* ext; int32_t* val;
  __device__ void operator()(int64_t i, uint32_t exc, uint32_t) const { val[i] = d[i] >= 254 ? ext[exc] : (int32_t)d[i]; }
};
struct SegT { int32_t v; int32_t abs; };
struct OpSegSum {   // running sum that restarts at absolute entries (non-commutative, associative)
  typedef SegT T;
  __host__ __device__ static T identity() { return SegT{0, 0}; }
  __host__ __device__ static T combine(T a, T b) { return b.abs ? b : SegT{a.v + b.v, a.abs}; }
};
struct SegIn { const uint8_t* d; const int32_t* val; __device__ SegT operator()(int64_t i) const { return SegT{val[i], d[i] == 255 ? 1 : 0}; } };
struct SegOut { int32_t* pos; __device__ void operator()(int64_t i, SegT, SegT inc) const { pos[i] = inc.v; } };
struct MetaEscIn { const uint8_t* m; __device__ uint32_t operator()(int64_t i) const { return m[i] == 255 ? 1u : 0u; } };
struct MetaOut {
  const uint8_t* m; const unsigned long long* dict; const unsigned long long* ext;
  uint16_t* flag; uint8_t* mapq; uint8_t* strand; uint16_t* nh;
  __device__ void operator()(int64_t i, uint32_t exc, uint32_t) const {
    const unsigned long long t = m[i] == 255 ? ext[exc] : dict[m[i]];
    flag[i] = (uint16_t)t; mapq[i] = (uint8_t)(t >> 16); strand[i] = (uint8_t)(t >> 24); nh[i] = (uint16_t)(t >> 32);
  }
};

struct HistIn { const uint32_t* c; __device__ uint32_t operator()(int64_t i) const { return c[i]; } };
struct HistOut { uint32_t* p; __device__ void operator()(int64_t i, uint32_t exc, uint32_t) const { p[i] = exc; } };

// ---- YD carry (tb_collapse_window_carry), host side -----------------------------------------------------------------------
// carry_in re-filtered against B without any device work (a window with no records or no groups)
int yd_carry_pass_host(tb_ctx* ctx, const tb_soa_in* hin, const tb_yd_carry* cin, tb_yd_carry* cout) {
  const int nchains = 2 * hin->n_files;
  const int32_t B = hin->pos_hi + 1;
  auto keep = [&](int64_t q, int64_t b) { return cin->seg_end[q] >= B && (cin->seg_end[q] > cin->seg_start[q] || q == b - 1); };
  int64_t tot = 0;
  if (cin)
    for (int c = 0; c < nchains; ++c)
      for (int64_t q = cin->chain_off[c], b = cin->chain_off[c + 1]; q < b; ++q) tot += keep(q, b);
  cout->n_segs = tot;
  if (tot > cout->capacity) { ctx->set_error("tb_collapse_window_carry: carry_out capacity %lld < %lld segments", (long long)cout->capacity, (long long)tot); return 1; }
  cout->tid = hin->tid; cout->pos_hi = hin->pos_hi;
  int64_t j = 0;
  for (int c = 0; c < nchains; ++c) {
    cout->chain_off[c] = j;
    if (cin)
      for (int64_t q = cin->chain_off[c], b = cin->chain_off[c + 1]; q < b; ++q)
        if (keep(q, b)) { cout->seg_start[j] = cin->seg_start[q]; cout->seg_end[j] = cin->seg_end[q]; ++j; }
  }
  cout->chain_off[nchains] = j;
  return 0;
}

}  // namespace

int tb_collapse_impl(tb_ctx* ctx, const tb_soa_in* hin, tb_groups_out* out, const tb_yd_carry* cin, tb_yd_carry* cout) {
  TB_CUDA(cudaSetDevice(ctx->device));
  const int64_t n = hin->n;
  const int k = hin->n_files;
  out->n_groups = 0; out->n_kept = 0;
  if (cin && cin->tid != hin->tid) cin = nullptr;   // the reference empties the lists at a tid change (tiebrush.cpp:586-589)
  if (n == 0) return cout ? yd_carry_pass_host(ctx, hin, cin, cout) : 0;
  if (n >= (1LL << 31)) { ctx->set_error("tb_collapse_window: n=%lld too large for one window (< 2^31)", (long long)n); return 1; }
  if (k < 1 || k > ctx->n_samples) { ctx->set_error("tb_collapse_window: n_files=%d but the context was created for %d samples", k, ctx->n_samples); return 1; }
  bool any_merged = false;
  if (hin->file_merged) for (int f = 0; f < k; ++f) any_merged |= hin->file_merged[f] != 0;
  if (any_merged && (!hin->yc_in || !hin->yx_in || !hin->yd_in)) { ctx->set_error("tb_collapse_window: TieBrush-made inputs need yc_in/yx_in/yd_in"); return 1; }
  if (ctx->collapse_same && !hin->qhash) { ctx->set_error("tb_collapse_window: -A needs qhash"); return 1; }
  if (ctx->mode == TB_MODE_FULL && (!hin->md_off || !hin->md)) { ctx->set_error("tb_collapse_window: -L needs md_off/md"); return 1; }
  if (hin->pos_hi <= hin->pos_lo) { ctx->set_error("tb_collapse_window: pos_lo/pos_hi not set"); return 1; }
  if (out->capacity < 1) { ctx->set_error("tb_collapse_window: zero output capacity"); return 1; }
  for (int f = 0; f < k; ++f) if (hin->run_off[f] > hin->run_off[f + 1]) { ctx->set_error("tb_collapse_window: run_off not monotone"); return 1; }
  if (hin->run_off[0] != 0 || hin->run_off[k] != n) { ctx->set_error("tb_collapse_window: run_off must span [0,n]"); return 1; }
  cudaStream_t st = ctx->stream;
  DevBuf* B = ctx->buf;
  const bool ordered = ctx->flag_mask != 0 || ctx->collapse_same || any_merged || (ctx->keep_bits & TB_STORE_FRAC);

  ColIn in; memset(&in, 0, sizeof(in));
  in.n = n; in.k = k; in.mode = ctx->mode; in.flag_mask = ctx->flag_mask; in.max_nh = ctx->max_nh; in.min_qual = ctx->min_qual; in.keep_bits = ctx->keep_bits;
  in.collapse_same = ctx->collapse_same;
  in.pos_lo = hin->pos_lo; in.span = (uint32_t)(hin->pos_hi - hin->pos_lo);
  TB_CUDA(B[XB_STATUS].ensure(sizeof(int64_t) * 16));
  TB_CUDA(ctx->pinned[0].ensure(1024));
  long long* d_status = B[XB_STATUS].as<long long>();
  long long* h_status = ctx->pinned[0].as<long long>();
  memset(h_status, 0, sizeof(int64_t) * 16); h_status[CS_ERRIDX] = -1;
  TB_CUDA(cudaMemcpyAsync(d_status, h_status, sizeof(int64_t) * 16, cudaMemcpyHostToDevice, st));
  const int dev = hin->on_device;
  if (!hin->pos && !hin->pos_d8) { ctx->set_error("tb_collapse_window: neither pos nor pos_d8 given"); return 1; }
  if (!(hin->flag && hin->mapq && hin->strand && hin->nh) && !(hin->meta8 && (hin->meta_dict || hin->n_meta_dict == 0) && (hin->meta_ext || hin->n_meta_ext == 0))) {
    ctx->set_error("tb_collapse_window: neither flag / mapq / strand / nh nor meta8 (+ meta_dict, meta_ext) given"); return 1;
  }
  if (hin->pos) { if (tb_stage_in(ctx, ctx->in_stage[0], hin->pos, (size_t)n, dev, &in.pos)) return 1; }
  else {   // positions = running sum of the per-record differences, restarted at absolute entries
    const uint8_t* d8 = nullptr; const int32_t* pext = nullptr;
    if (tb_stage_in(ctx, ctx->in_stage[16], hin->pos_d8, (size_t)n, dev, &d8)) return 1;
    if (hin->n_pos_ext > 0) { if (tb_stage_in(ctx, ctx->in_stage[17], hin->pos_ext, (size_t)hin->n_pos_ext, dev, &pext)) return 1; }
    TB_CUDA(ctx->in_stage[0].ensure(sizeof(int32_t) * (size_t)n + 16));
    TB_CUDA(B[XB_AGG].ensure((size_t)(tb_scan_blocks(n) + 8) * sizeof(uint64_t)));
    int32_t* dpos = ctx->in_stage[0].as<int32_t>();
    TB_CUDA((tb_device_scan<OpSumU32>(ctx, PosEscIn{d8}, n, B[XB_AGG].as<uint32_t>(), PosValOut{d8, pext, dpos})));
    col_check_total_kernel<<<1, 1, 0, st>>>(B[XB_AGG].as<uint32_t>() + tb_scan_blocks(n), (unsigned long long)hin->n_pos_ext, d_status, 6);
    TB_CUDA((tb_device_scan<OpSegSum>(ctx, SegIn{d8, dpos}, n, B[XB_AGG].as<SegT>(), SegOut{dpos})));
    ctx->launches++;
    in.pos = dpos;
  }
  if (hin->flag && hin->mapq && hin->strand && hin->nh) {
    if (tb_stage_in(ctx, ctx->in_stage[1], hin->flag, (size_t)n, dev, &in.flag)) return 1;
    if (tb_stage_in(ctx, ctx->in_stage[2], hin->mapq, (size_t)n, dev, &in.mapq)) return 1;
    if (tb_stage_in(ctx, ctx->in_stage[3], hin->strand, (size_t)n, dev, &in.strand)) return 1;
    if (tb_stage_in(ctx, ctx->in_stage[4], hin->nh, (size_t)n, dev, &in.nh)) return 1;
  } else {   // dictionary-coded (flag, mapq, strand, nh)
    if (hin->n_meta_dict < 0 || hin->n_meta_dict > 255) { ctx->set_error("tb_collapse_window: n_meta_dict %d out of range (0..255)", hin->n_meta_dict); return 1; }
    const uint8_t* m8 = nullptr; const uint64_t* mext = nullptr;
    if (tb_stage_in(ctx, ctx->in_stage[18], hin->meta8, (size_t)n, dev, &m8)) return 1;
    if (hin->n_meta_ext > 0) { if (tb_stage_in(ctx, ctx->in_stage[19], hin->meta_ext, (size_t)hin->n_meta_ext, dev, &mext)) return 1; }
    TB_CUDA(ctx->in_stage[1].ensure(sizeof(uint16_t) * (size_t)n + 16)); TB_CUDA(ctx->in_stage[2].ensure((size_t)n + 16));
    TB_CUDA(ctx->in_stage[3].ensure((size_t)n + 16)); TB_CUDA(ctx->in_stage[4].ensure(sizeof(uint16_t) * (size_t)n + 16));
    TB_CUDA(B[XB_META_DICT].ensure(sizeof(uint64_t) * 256));
    uint64_t dict_h[256]; memset(dict_h, 0, sizeof(dict_h));
    if (hin->n_meta_dict > 0) memcpy(dict_h, hin->meta_dict, sizeof(uint64_t) * (size_t)hin->n_meta_dict);
    TB_CUDA(cudaMemcpyAsync(B[XB_META_DICT].p, dict_h, sizeof(dict_h), cudaMemcpyHostToDevice, st));
    TB_CUDA(B[XB_AGG].ensure((size_t)(tb_scan_blocks(n) + 8) * sizeof(uint64_t)));
    TB_CUDA((tb_device_scan<OpSumU32>(ctx, MetaEscIn{m8}, n, B[XB_AGG].as<uint32_t>(),
                                      MetaOut{m8, B[XB_META_DICT].as<unsigned long long>(), (const unsigned long long*)mext, ctx->in_stage[1].as<uint16_t>(),
                                              ctx->in_stage[2].as<uint8_t>(), ctx->in_stage[3].as<uint8_t>(), ctx->in_stage[4].as<uint16_t>()})));
    col_check_total_kernel<<<1, 1, 0, st>>>(B[XB_AGG].as<uint32_t>() + tb_scan_blocks(n), (unsigned long long)hin->n_meta_ext, d_status, 7);
    ctx->launches++;
    in.flag = ctx->in_stage[1].as<uint16_t>(); in.mapq = ctx->in_stage[2].as<uint8_t>(); in.strand = ctx->in_stage[3].as<uint8_t>(); in.nh = ctx->in_stage[4].as<uint16_t>();
  }
  if (!hin->cig_off && !hin->n_cigar8) { ctx->set_error("tb_collapse_window: neither cig_off nor n_cigar8 given"); return 1; }
  if (!hin->cigar && !(hin->cigar16 && (hin->cigar_ext || hin->n_ext == 0))) { ctx->set_error("tb_collapse_window: neither cigar nor cigar16 (+cigar_ext) given"); return 1; }
  if (hin->cig_off) { if (tb_stage_in(ctx, ctx->in_stage[5], hin->cig_off, (size_t)n + 1, dev, &in.cig_off)) return 1; }
  else {   // offsets = exclusive scan of the per-record op counts
    const uint8_t* n8 = nullptr;
    if (tb_stage_in(ctx, ctx->in_stage[13], hin->n_cigar8, (size_t)n, dev, &n8)) return 1;
    TB_CUDA(ctx->in_stage[5].ensure(sizeof(uint32_t) * ((size_t)n + 1) + 16));
    TB_CUDA(B[XB_AGG].ensure((size_t)(tb_scan_blocks(n) + 8) * sizeof(uint64_t)));
    TB_CUDA((tb_device_scan<OpSumU32>(ctx, Nc8In{n8}, n, B[XB_AGG].as<uint32_t>(), OffOut{ctx->in_stage[5].as<uint32_t>(), n})));
    in.cig_off = ctx->in_stage[5].as<uint32_t>();
    // the packer's n_cig must be the sum of the per-record op counts (otherwise the arena would be read out of bounds)
    col_check_total_kernel<<<1, 1, 0, st>>>(B[XB_AGG].as<uint32_t>() + tb_scan_blocks(n), (unsigned long long)hin->n_cig, d_status, 4);
    ctx->launches++;
  }
  if (hin->cigar) { if (tb_stage_in(ctx, ctx->in_stage[6], hin->cigar, (size_t)hin->n_cig, dev, &in.cigar)) return 1; }
  else {   // 16-bit ops widened to BAM words, escaped lengths taken from cigar_ext in op order
    const uint16_t* c16 = nullptr; const uint32_t* ext = nullptr;
    if (tb_stage_in(ctx, ctx->in_stage[14], hin->cigar16, (size_t)hin->n_cig, dev, &c16)) return 1;
    if (hin->n_ext > 0) { if (tb_stage_in(ctx, ctx->in_stage[15], hin->cigar_ext, (size_t)hin->n_ext, dev, &ext)) return 1; }
    TB_CUDA(ctx->in_stage[6].ensure(sizeof(uint32_t) * ((size_t)hin->n_cig + 4) + 16));
    TB_CUDA(B[XB_AGG].ensure((size_t)(tb_scan_blocks(hin->n_cig) + 8) * sizeof(uint64_t)));
    TB_CUDA((tb_device_scan<OpSumU32>(ctx, EscIn{c16}, hin->n_cig, B[XB_AGG].as<uint32_t>(), ExpandOut{c16, ext, ctx->in_stage[6].as<uint32_t>()})));
    in.cigar = ctx->in_stage[6].as<uint32_t>();
    // every escaped length (field 0xFFF) takes one entry of cigar_ext, in op order
    col_check_total_kernel<<<1, 1, 0, st>>>(B[XB_AGG].as<uint32_t>() + tb_scan_blocks(hin->n_cig), (unsigned long long)hin->n_ext, d_status, 5);
    ctx->launches++;
  }
  if (ctx->mode == TB_MODE_FULL) {
    if (tb_stage_in(ctx, ctx->in_stage[7], hin->md_off, (size_t)n + 1, dev, &in.md_off)) return 1;
    if (tb_stage_in(ctx, ctx->in_stage[8], hin->md, (size_t)hin->n_md, dev, &in.md)) return 1;
  }
  if (ctx->collapse_same) { if (tb_stage_in(ctx, ctx->in_stage[9], hin->qhash, (size_t)n, dev, &in.qhash)) return 1; }
  if (any_merged) {
    if (tb_stage_in(ctx, ctx->in_stage[10], hin->yc_in, (size_t)n, dev, &in.yc_in)) return 1;
    if (tb_stage_in(ctx, ctx->in_stage[11], hin->yx_in, (size_t)n, dev, &in.yx_in)) return 1;
    if (tb_stage_in(ctx, ctx->in_stage[12], hin->yd_in, (size_t)n, dev, &in.yd_in)) return 1;
  }

  const uint32_t W = (uint32_t)((k + 31) / 32);
  const uint32_t S = in.span;
  TB_CUDA(B[XB_HIST].ensure(sizeof(uint32_t) * ((size_t)S + 2)));
  TB_CUDA(B[XB_RUNOFF].ensure(sizeof(int64_t) * (k + 1)));
  TB_CUDA(cudaMemcpyAsync(B[XB_RUNOFF].p, hin->run_off, sizeof(int64_t) * (k + 1), cudaMemcpyHostToDevice, st));
  const uint8_t* d_merged = nullptr;
  if (any_merged) {
    TB_CUDA(B[XB_MERGED].ensure((size_t)k));
    TB_CUDA(cudaMemcpyAsync(B[XB_MERGED].p, hin->file_merged, (size_t)k, cudaMemcpyHostToDevice, st));
    d_merged = B[XB_MERGED].as<uint8_t>();
  }
  YdCarry cy;
  const int nchains = 2 * k;
  if (cin || cout) {   // device copy of carry_in; areas for the seeds and for carry_out
    cy.in = cin != nullptr; cy.out = cout != nullptr;
    cy.nin = cin ? cin->n_segs : 0;
    cy.bout = hin->pos_hi + 1;
    cy.cap = cout ? cout->capacity : 0;
    TB_CUDA(B[XB_YDCARRY].ensure(sizeof(int64_t) * (nchains + 1) + sizeof(int32_t) * (3 * (size_t)nchains + 2 * (size_t)cy.nin) + 64));
    long long* coff = B[XB_YDCARRY].as<long long>();
    cy.seed = (int32_t*)(coff + nchains + 1); cy.ext = cy.seed + nchains; cy.efin = cy.ext + nchains;
    if (cin) {
      int32_t* cs = cy.efin + nchains; int32_t* ce = cs + cy.nin;
      TB_CUDA(cudaMemcpyAsync(coff, cin->chain_off, sizeof(int64_t) * (nchains + 1), cudaMemcpyHostToDevice, st));
      if (cy.nin > 0) {
        TB_CUDA(cudaMemcpyAsync(cs, cin->seg_start, sizeof(int32_t) * (size_t)cy.nin, cudaMemcpyHostToDevice, st));
        TB_CUDA(cudaMemcpyAsync(ce, cin->seg_end, sizeof(int32_t) * (size_t)cy.nin, cudaMemcpyHostToDevice, st));
      }
      cy.coff = coff; cy.cs = cs; cy.ce = ce;
    }
    if (cout) {
      TB_CUDA(B[XB_YDCOUT].ensure(sizeof(int64_t) * (2 * (size_t)nchains + 1) + sizeof(int32_t) * 2 * (size_t)cy.cap + 64));
      cy.ometa = B[XB_YDCOUT].as<long long>();
      cy.os = (int32_t*)(cy.ometa + 2 * nchains + 1); cy.oe = cy.os + cy.cap;
    }
  }
  TB_CUDA(cudaStreamSynchronize(st));  // h_status and the caller's small host arrays may be reused from here on
  {
    int64_t mx = (int64_t)S + 2; if (n > mx) mx = n;
    TB_CUDA(B[XB_AGG].ensure((size_t)(tb_scan_blocks(mx) + 8) * sizeof(uint64_t)));
  }
  uint32_t* d_hist = B[XB_HIST].as<uint32_t>();
  // ---- C1, C2 ----
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[4], st));
  TB_CUDA(cudaMemsetAsync(d_hist, 0, sizeof(uint32_t) * ((size_t)S + 2), st));
  col_hist_kernel<<<tb_grid_for(n, 256), 256, 0, st>>>(in, d_hist, d_status);
  ctx->launches++;
  TB_CUDA((tb_device_scan<OpSumU32>(ctx, HistIn{d_hist}, (int64_t)S + 1, B[XB_AGG].as<uint32_t>(), HistOut{d_hist})));
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[5], st));
  // the position checks must be known before the front ends index P[] by position
  TB_CUDA(cudaMemcpyAsync(h_status, d_status, sizeof(int64_t) * 16, cudaMemcpyDeviceToHost, st));
  TB_CUDA(cudaStreamSynchronize(st));
  if (ctx->profiling) { float ms = 0; if (cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]) == cudaSuccess) ctx->last_ms[2] = ms; }
  if (h_status[CS_ERR] == ERR_POS_RANGE) { ctx->set_error("tb_collapse_window: record %lld has pos outside [pos_lo,pos_hi)", h_status[CS_ERRIDX]); return 1; }
  if (h_status[CS_ERR] == 4) { ctx->set_error("tb_collapse_window: compact wire format: n_cigar8 sums to %lld ops but n_cig = %lld", h_status[CS_ERRIDX], (long long)hin->n_cig); return 1; }
  if (h_status[CS_ERR] == 5) { ctx->set_error("tb_collapse_window: compact wire format: cigar16 holds %lld escaped lengths but n_ext = %lld", h_status[CS_ERRIDX], (long long)hin->n_ext); return 1; }
  if (h_status[CS_ERR] == 6) { ctx->set_error("tb_collapse_window: packed wire format: pos_d8 holds %lld escaped entries but n_pos_ext = %lld", h_status[CS_ERRIDX], (long long)hin->n_pos_ext); return 1; }
  if (h_status[CS_ERR] == 7) { ctx->set_error("tb_collapse_window: packed wire format: meta8 holds %lld escaped entries but n_meta_ext = %lld", h_status[CS_ERRIDX], (long long)hin->n_meta_ext); return 1; }
  if (h_status[CS_ERR] == 3) { ctx->set_error("tb_collapse_window: unmapped record %lld kept by -M: the reference aborts here (GVec invalid index)", h_status[CS_ERRIDX]); return 1; }

  ColGeom g; g.n = n; g.k = k; g.W = W; g.S = S; g.P = d_hist; g.d_runoff = B[XB_RUNOFF].as<long long>(); g.d_merged = d_merged; g.d_status = d_status;
  ColGroups grp; memset(&grp, 0, sizeof(grp));
  grp.capacity = out->capacity;
  grp.rep = out->rep_index; grp.yc = out->yc; grp.yx = out->yx; grp.yd = out->yd;
  if (!out->on_device) {
    const size_t cap = (size_t)(out->capacity < n ? out->capacity : n);
    TB_CUDA(ctx->out_stage[0].ensure(sizeof(uint32_t) * cap)); TB_CUDA(ctx->out_stage[1].ensure(sizeof(float) * cap));
    TB_CUDA(ctx->out_stage[2].ensure(sizeof(uint32_t) * cap)); TB_CUDA(ctx->out_stage[3].ensure(sizeof(int32_t) * cap));
    grp.rep = ctx->out_stage[0].as<uint32_t>(); grp.yc = ctx->out_stage[1].as<float>(); grp.yx = ctx->out_stage[2].as<uint32_t>(); grp.yd = ctx->out_stage[3].as<int32_t>();
    grp.capacity = (int64_t)cap;
  }
  int64_t G = 0, kept = 0;
  int rc = 2;
  ctx->last_path = ordered ? 1 : 0;
  if (!ordered) rc = col_front_tile(ctx, in, g, grp, &G, &kept);
  if (rc == 2) {
    if (!ordered) {  // a start position with more distinct alignments than one shared-memory table: exact path for the window
      ctx->last_path = 2;
      memset(h_status, 0, sizeof(int64_t) * 16); h_status[CS_ERRIDX] = -1;
      TB_CUDA(cudaMemcpyAsync(d_status, h_status, sizeof(int64_t) * 16, cudaMemcpyHostToDevice, st));
      TB_CUDA(cudaStreamSynchronize(st));
    }
    rc = col_front_ordered(ctx, in, g, grp, &G, &kept);
  }
  if (rc) return 1;
  if (G > out->capacity) { ctx->set_error("tb_collapse_window: output capacity %lld < %lld groups", (long long)out->capacity, (long long)G); return 1; }
  out->n_kept = kept;
  out->n_groups = G;
  if (G == 0) return cout ? yd_carry_pass_host(ctx, hin, cin, cout) : 0;
  // ---- C7: YD ----
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[2], st));
  if (col_yd(ctx, in, g, grp, G, cy)) return 1;
  if (ctx->profiling) TB_CUDA(cudaEventRecord(ctx->ev[3], st));
  if (!out->on_device) {
    TB_CUDA(cudaMemcpyAsync(out->rep_index, grp.rep, sizeof(uint32_t) * G, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaMemcpyAsync(out->yc, grp.yc, sizeof(float) * G, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaMemcpyAsync(out->yx, grp.yx, sizeof(uint32_t) * G, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaMemcpyAsync(out->yd, grp.yd, sizeof(int32_t) * G, cudaMemcpyDeviceToHost, st));
  }
  std::vector<long long> ometa;
  std::vector<int32_t> oseg;
  if (cout) {   // the carried lists come back in the order the chains reserved their slots
    ometa.resize(2 * (size_t)nchains + 1);
    TB_CUDA(cudaMemcpyAsync(ometa.data(), cy.ometa, sizeof(int64_t) * ometa.size(), cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    const int64_t tot = ometa[2 * nchains];
    cout->n_segs = tot;
    if (tot > cout->capacity) { ctx->set_error("tb_collapse_window_carry: carry_out capacity %lld < %lld segments", (long long)cout->capacity, (long long)tot); return 1; }
    oseg.resize(2 * (size_t)tot + 2);
    if (tot > 0) {
      TB_CUDA(cudaMemcpyAsync(oseg.data(), cy.os, sizeof(int32_t) * (size_t)tot, cudaMemcpyDeviceToHost, st));
      TB_CUDA(cudaMemcpyAsync(oseg.data() + tot, cy.oe, sizeof(int32_t) * (size_t)tot, cudaMemcpyDeviceToHost, st));
    }
  }
  TB_CUDA(cudaStreamSynchronize(st));
  if (cout) {
    const int64_t tot = ometa[2 * nchains];
    int64_t j = 0;
    for (int c = 0; c < nchains; ++c) {
      cout->chain_off[c] = j;
      for (int64_t q = ometa[2 * c], e = q + ometa[2 * c + 1]; q < e; ++q, ++j) { cout->seg_start[j] = oseg[q]; cout->seg_end[j] = oseg[tot + q]; }
    }
    cout->chain_off[nchains] = j;
    cout->tid = hin->tid; cout->pos_hi = hin->pos_hi;
  }
  if (ctx->profiling) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ctx->ev[6], ctx->ev[7]) == cudaSuccess) ctx->last_ms[4] = ms;
    if (cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]) == cudaSuccess) ctx->last_ms[5] = ms;
    (void)cudaGetLastError();   // an event that was not recorded on this path (ordered front end) leaves an error behind
  }
  return 0;
}
