// tc_columns.cuh — tiecov's column sets, each listed once: the records of a window (tc_soa_in, plus the YX column of
// tiecov -s), the coverage rows (tc_runs_out) and the junction rows (tc_juncs_out). Every path that stages, slices,
// exchanges or gathers tiecov data goes through tc_fields, so a column added here travels everywhere.
#pragma once
#include <type_traits>
#include "tb_common.cuh"

// a record set: the row columns, then the CSR pair (cig_off [n + 1] into cigar). end and yx may be NULL.
struct TcRecords {
  int32_t *tid, *pos; float* yc; uint8_t* strand; int32_t *end, *yx;
  uint32_t *cig_off, *cigar;
};

// the row columns of each set, in the order they travel. The CSR pair of a record set is not a row column: its offsets
// need a rebase wherever records move (tc_copy_records).
template <class F> void tc_fields(tc_runs_out& r, F&& f) { f(r.tid); f(r.start0); f(r.end0); f(r.value); }
template <class F> void tc_fields(tc_juncs_out& j, F&& f) { f(j.tid); f(j.start); f(j.end); f(j.strand); f(j.value); }
template <class F> void tc_fields(TcRecords& c, F&& f) { f(c.tid); f(c.pos); f(c.yc); f(c.strand); f(c.end); f(c.yx); }

// a set's columns as (pointer, element size); a column the set does not have is a NULL pointer
struct TcCols { int n = 0; char* p[8]; size_t size[8]; };
template <class S> TcCols tc_cols(S s) {
  TcCols c;
  tc_fields(s, [&](auto* q) { c.p[c.n] = (char*)q; c.size[c.n++] = sizeof(*q); });
  return c;
}

// the set from row k on (a record set keeps its absolute CIGAR offsets, so `cigar` is shared)
template <class S> S tc_at(S s, int64_t k) {
  tc_fields(s, [&](auto*& q) { if (q) q += k; });
  return s;
}
inline TcRecords tc_at(TcRecords c, int64_t k) {
  c = tc_at<TcRecords>(c, k);
  c.cig_off += k;
  return c;
}

inline TcRecords tc_records(const tc_soa_in& w, const int32_t* yx = nullptr) {
  return TcRecords{(int32_t*)w.tid, (int32_t*)w.pos, (float*)w.yc, (uint8_t*)w.strand, (int32_t*)w.end, (int32_t*)yx,
                   (uint32_t*)w.cig_off, (uint32_t*)w.cigar};
}
inline tc_soa_in tc_window(const TcRecords& c, int64_t n, int64_t n_cig, int on_device = 1) {
  tc_soa_in w; memset(&w, 0, sizeof(w));
  w.n = n; w.tid = c.tid; w.pos = c.pos; w.yc = c.yc; w.strand = c.strand; w.end = c.end;
  w.cig_off = c.cig_off; w.cigar = c.cigar; w.on_device = on_device; w.n_cig = n_cig;
  return w;
}

// n rows from src to dst (kind: the direction); a column that either side lacks, or that both share, is skipped
template <class S> cudaError_t tc_copy_rows(const S& dst, const S& src, int64_t n, cudaMemcpyKind kind, cudaStream_t st) {
  const TcCols d = tc_cols(dst), s = tc_cols(src);
  for (int i = 0; i < d.n; ++i) {
    if (n <= 0 || !d.p[i] || !s.p[i] || d.p[i] == s.p[i]) continue;
    const cudaError_t e = cudaMemcpyAsync(d.p[i], s.p[i], d.size[i] * (size_t)n, kind, st);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// device arrays for `cap` rows of the columns `s` has, column i in slots[i]; `s` then points at them (the device stand-in
// of a host output set)
template <class S> cudaError_t tc_alloc_rows(DevBuf* slots, S& s, int64_t cap) {
  cudaError_t e = cudaSuccess;
  int i = 0;
  tc_fields(s, [&](auto*& q) {
    using T = std::remove_reference_t<decltype(*q)>;
    DevBuf& b = slots[i++];
    if (!q || e != cudaSuccess) return;
    e = b.ensure(sizeof(T) * (size_t)cap);
    q = b.as<T>();
  });
  return e;
}

// a record set in slots[0..8) with room for n records and `words` CIGAR words; end / yx only when with_end_yx
inline cudaError_t tc_alloc_records(DevBuf* slots, int64_t n, int64_t words, bool with_end_yx, TcRecords* c) {
  cudaError_t e = cudaSuccess;
  auto col = [&](int i, size_t bytes) { if (e == cudaSuccess) e = slots[i].ensure(bytes); return slots[i].p; };
  const size_t r = (size_t)n;
  c->tid = (int32_t*)col(0, 4 * r); c->pos = (int32_t*)col(1, 4 * r); c->yc = (float*)col(2, 4 * r); c->strand = (uint8_t*)col(3, r);
  c->end = with_end_yx ? (int32_t*)col(4, 4 * r) : nullptr;
  c->yx = with_end_yx ? (int32_t*)col(5, 4 * r) : nullptr;
  c->cig_off = (uint32_t*)col(6, 4 * (r + 1)); c->cigar = (uint32_t*)col(7, 4 * (size_t)words);
  return e;
}

// the device copy of a record window, column i in slots[i] (device windows pass through). A host window of a longer stream
// keeps its absolute CIGAR offsets: only its n_cig words are copied, and the device `cigar` is biased so that
// cigar[cig_off[i]] still lands on them.
inline int tc_stage_window(tb_ctx* ctx, DevBuf* slots, const tc_soa_in& h, const int32_t* yx, tc_soa_in* d, const int32_t** d_yx) {
  const size_t n = (size_t)h.n;
  TcRecords c = tc_records(h, yx);
  int i = 0, rc = 0;
  tc_fields(c, [&](auto*& q) {
    using T = std::remove_reference_t<decltype(*q)>;
    const T* out = nullptr;
    if (!rc) rc = tb_stage_in(ctx, slots[i], (const T*)q, n, h.on_device, &out);
    q = (T*)out;
    ++i;
  });
  const uint32_t cbase = (!h.on_device && n > 0) ? h.cig_off[0] : 0u;
  const uint32_t *off = nullptr, *words = nullptr;
  if (rc || tb_stage_in(ctx, slots[6], h.cig_off, n + 1, h.on_device, &off) ||
      tb_stage_in(ctx, slots[7], h.cigar ? h.cigar + cbase : nullptr, (size_t)h.n_cig, h.on_device, &words)) return 1;
  c.cig_off = (uint32_t*)off; c.cigar = (uint32_t*)words - cbase;
  *d = tc_window(c, h.n, h.n_cig);
  if (d_yx) *d_yx = c.yx;
  return 0;
}

// records [from, from + m) of src to rows [r, r + m) of dst on stream st: the row columns both sets have, the m + 1 offsets
// rebased so that src's first CIGAR word lands on word w of dst, and `words` CIGAR words (0 when they are already in place).
// One launch (shard.cu).
void tc_copy_records(tb_ctx* ctx, cudaStream_t st, const TcRecords& src, int64_t from, int64_t m, const TcRecords& dst, int64_t r, uint32_t w,
                     uint32_t words);
