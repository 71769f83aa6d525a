/*
 * yd_carry_oracle.c — TEST INFRASTRUCTURE ONLY: the oracle's collapse (oracle/tb_oracle.c, included unchanged) with the
 * YD segment lists carried across a window cut, the reference semantics tb_collapse_window_carry is checked against.
 *
 * tbo_collapse_carry runs the main loop of tbo_collapse (src/tiebrush.cpp:557-601 for one window) with the per-sample
 * lists fsegs / rsegs seeded from a carry instead of empty, and exports the lists the window leaves behind in the
 * canonical form of include/tiebrush_b200.h: for B = pos_hi + 1, the nodes with end >= B that cover two positions or
 * more, and the list's last node when its end >= B. A carry whose tid differs from the window's is ignored (the
 * reference empties the lists at a tid change, tiebrush.cpp:586-589).
 */
#include "../oracle/tb_oracle.c"

static void seglist_seed(seglist* L, const int32_t* s, const int32_t* e, int64_t a, int64_t b) { /* the carried nodes, as they are */
  segnode** tail = &L->head;
  for (int64_t q = a; q < b; q++) { *tail = newnode((uint32_t)s[q], (uint32_t)e[q], NULL); tail = &(*tail)->next; }
}

/* canonical carry of one list for B; writes at most `room` nodes, returns how many there are */
static int64_t seglist_export(const seglist* L, uint32_t B, int32_t* s, int32_t* e, int64_t room) {
  int64_t c = 0;
  for (const segnode* p = L->head; p; p = p->next) {
    if (p->end < B || (p->end == p->start && p->next)) continue;
    if (c < room) { s[c] = (int32_t)p->start; e[c] = (int32_t)p->end; }
    c++;
  }
  return c;
}

/* returns 0 ok, 1 group capacity, 2 cout->capacity too small (cout->n_segs = segments needed), 3 malformed carry */
int tbo_collapse_carry(const tb_soa_in* in, const tbo_opts* o, const tb_yd_carry* cin, tb_groups_out* out, tb_yd_carry* cout) {
  if (in->on_device || out->on_device) return -1;
  int64_t n = in->n; int k = in->n_files;
  if (cin && cin->tid != in->tid) cin = NULL;
  if (cin) {
    if (cin->n_chains != 2 * k || in->pos_lo < cin->pos_hi || cin->chain_off[0] != 0 || cin->chain_off[2 * k] != cin->n_segs) return 3;
    for (int c = 0; c < 2 * k; c++)
      for (int64_t q = cin->chain_off[c]; q < cin->chain_off[c + 1]; q++)
        if (cin->seg_end[q] < cin->seg_start[q] || (q > cin->chain_off[c] && cin->seg_start[q] <= cin->seg_end[q - 1])) return 3;
  }
  if (cout && cout->n_chains != 2 * k) return 3;
  col_state S; memset(&S, 0, sizeof(S));
  S.in = in; S.o = o; S.out = out;
  out->n_groups = 0; out->n_kept = 0;
  S.rec = (rec_t*)malloc(sizeof(rec_t) * (size_t)(n > 0 ? n : 1));
  int64_t nex_cap = (int64_t)in->cig_off[n] + n + 1;
  S.exons = (seg_t*)malloc(sizeof(seg_t) * (size_t)nex_cap);
  int64_t eo = 0;
  for (int64_t i = 0; i < n; i++) {
    uint32_t nc = in->cig_off[i + 1] - in->cig_off[i];
    S.rec[i].ex_off = (int)eo;
    if (in->flag[i] & 0x4) { S.rec[i].start = 0; S.rec[i].end = 0; S.rec[i].n_ex = 0; continue; }
    S.rec[i].n_ex = setup_coordinates(in->pos[i], in->cigar + in->cig_off[i], nc, S.exons + eo, &S.rec[i].start, &S.rec[i].end);
    eo += S.rec[i].n_ex;
  }
  S.cc.in = in; S.cc.o = o; S.cc.rec = S.rec; S.cc.exons = S.exons;
  S.fsegs = (seglist*)calloc((size_t)(k > 0 ? k : 1), sizeof(seglist));
  S.rsegs = (seglist*)calloc((size_t)(k > 0 ? k : 1), sizeof(seglist));
  for (int f = 0; f < k; f++) { seglist_reset(&S.fsegs[f]); seglist_reset(&S.rsegs[f]); }
  if (cin)
    for (int f = 0; f < k; f++) {
      seglist_seed(&S.fsegs[f], cin->seg_start, cin->seg_end, cin->chain_off[f], cin->chain_off[f + 1]);
      seglist_seed(&S.rsegs[f], cin->seg_start, cin->seg_end, cin->chain_off[k + f], cin->chain_off[k + f + 1]);
    }
  head_t* heap = (head_t*)malloc(sizeof(head_t) * (size_t)(k > 0 ? k : 1)); int hn = 0;
  int64_t* cursor = (int64_t*)malloc(sizeof(int64_t) * (size_t)(k > 0 ? k : 1));
  for (int f = 0; f < k; f++) {
    cursor[f] = in->run_off[f];
    if (cursor[f] < in->run_off[f + 1]) { int64_t i = cursor[f]++; head_t h = { S.rec[i].start, S.rec[i].end, f, i }; heap_push(heap, &hn, h); }
  }
  int64_t prev_pos = -1; int rc = 0;
  while (hn > 0) {
    head_t h = heap_pop(heap, &hn);
    int f = h.fidx;
    if (cursor[f] < in->run_off[f + 1]) { int64_t i = cursor[f]++; head_t nh = { S.rec[i].start, S.rec[i].end, f, i }; heap_push(heap, &hn, nh); }
    if (!passes_options(&S, h.idx)) continue;
    out->n_kept++;
    int64_t pos = (int64_t)S.rec[h.idx].start;
    if (pos != prev_pos) { if (flush_pdata(&S)) { rc = 1; break; } prev_pos = pos; }
    add_pdata(&S, h.idx, f);
  }
  if (!rc && flush_pdata(&S)) rc = 1;
  if (!rc && cout) {
    const uint32_t B = (uint32_t)in->pos_hi + 1;
    int64_t tot = 0;
    cout->tid = in->tid; cout->pos_hi = in->pos_hi;
    for (int c = 0; c < 2 * k; c++) {
      const seglist* L = c < k ? &S.fsegs[c] : &S.rsegs[c - k];
      int64_t room = cout->capacity - tot; if (room < 0) room = 0;
      int64_t at = tot < cout->capacity ? tot : 0;
      cout->chain_off[c] = tot;
      tot += seglist_export(L, B, cout->seg_start + at, cout->seg_end + at, room);
    }
    cout->chain_off[2 * k] = tot;
    cout->n_segs = tot;
    if (tot > cout->capacity) rc = 2;
  }
  for (int gi = 0; gi < S.nlist; gi++) { free(S.list[gi]->samples); free(S.list[gi]); }
  for (int f = 0; f < k; f++) { seglist_clear(&S.fsegs[f]); seglist_clear(&S.rsegs[f]); }
  free(S.fsegs); free(S.rsegs); free(heap); free(cursor); free(S.list); free(S.rec); free(S.exons);
  return rc;
}
