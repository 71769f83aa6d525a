"""Coordinate sharding of the hot path over the GPUs of one box (SURVEY.md §8e), one process per GPU.

The path shards by reference-coordinate range: a collapse group never spans a (tid,start)
(SPData::operator<, src/tiebrush.cpp:438-457), tiecov state never spans a bundle (src/tiecov.cpp:443).
Records are assigned to a shard by START position. What crosses a shard edge:

  tiebrush  nothing but the YD segment lists (GSegList, src/tiebrush.cpp:122-253). They are provably empty after
            the first read past a *coverage gap* (processRead frees every node when d==0, :237-242), so a shard
            starts its input at the last gap at or before its cut and drops the groups before the cut
            (`collapse_sharded`): exact, no collective on the data path.
  tiecov    reads that start in shard g and reach into g+1.. (the halo). `coverage_sharded` all-gathers those few
            records (one small message per rank), every rank prepends the ones that reach its range, computes its
            window and clips the bedGraph runs to its range. A run that was cut in two by the edge is stitched
            when both halves carry the same value and the bundle continues across the edge (runs never join across
            bundles, tiecov.cpp:226-241). Junction rows are per bundle (flushJuncs, tiecov.cpp:114-120): the rows
            of a bundle that spans an edge are reduced by key and re-sorted at the ordered gather, which also
            restores the global JUNC%08d numbering (tiecov.cpp:92-94).

Collectives (torch.distributed; NCCL over NVLink on the GPU box, gloo in the CPU tests): one variable-size
all_gather for the halo, one for the ordered gather of the (small) outputs. The per-record work itself runs through
`compute` = api.Context.coverage_window / collapse_window, i.e. the CUDA path; this module is host-side edge logic only.
"""
from __future__ import annotations

import numpy as np

from . import sam

_REF_OPS = (0, 2, 3, 7, 8)          # M D N = X consume the reference (GSam.cpp:351-417)
COV_COLS = ("tid", "pos", "yc", "strand")


# --------------------------------------------------------------------------------------------------
# geometry helpers (numpy, host)
# --------------------------------------------------------------------------------------------------
def ref_end(cols) -> np.ndarray:
    """0-based exclusive end of every record (== GSamRecord::end, 1-based inclusive)."""
    cig = np.asarray(cols["cigar"]).astype(np.int64)
    off = np.asarray(cols["cig_off"]).astype(np.int64)
    ref = np.where(np.isin(cig & 0xF, _REF_OPS), cig >> 4, 0)
    cs = np.concatenate([[0], np.cumsum(ref)])
    return np.asarray(cols["pos"]).astype(np.int64) + (cs[off[1:]] - cs[off[:-1]])


def _key(tid, pos):
    return (np.asarray(tid).astype(np.int64) << 32) | np.asarray(pos).astype(np.int64)


def bundle_heads(tid, pos, end, e_before=None) -> np.ndarray:
    """head[i] = record i opens a new tiecov bundle (tiecov.cpp:443: tid change or start > b_end).
    `e_before` = (tid, end) already open to the left of record 0 (the halo), or None."""
    n = len(pos)
    if n == 0:
        return np.zeros(0, bool)
    k = _key(tid, end)
    pm = np.maximum.accumulate(k)
    head = np.ones(n, bool)
    head[1:] = _key(tid[1:], pos[1:]) >= pm[:-1]          # same tid and pos >= max end so far, or a later tid
    if e_before is not None:
        open_k = int(_key(e_before[0], e_before[1]))
        pm2 = np.maximum(pm, open_k)
        head[0] = int(_key(tid[0], pos[0])) >= open_k
        head[1:] = _key(tid[1:], pos[1:]) >= pm2[:-1]
    return head


def cov_cuts(cols, n_shards: int) -> list[tuple[int, int]]:
    """n_shards-1 cut keys (tid,pos) balancing records; all records of one (tid,pos) stay together."""
    key = _key(cols["tid"], cols["pos"])
    n = len(key)
    cuts = []
    for g in range(1, n_shards):
        i = min(n, (g * n) // n_shards)
        if i >= n:
            cuts.append((1 << 30, 0))
            continue
        i = int(np.searchsorted(key, key[i], side="left"))     # back to the first record of that position
        cuts.append((int(key[i] >> 32), int(key[i] & 0xFFFFFFFF)))
    return cuts


def cov_slice(cols, lo, hi):
    """Records with lo <= (tid,pos) < hi of a coordinate-sorted coverage stream (None = open end)."""
    key = _key(cols["tid"], cols["pos"])
    a = 0 if lo is None else int(np.searchsorted(key, (lo[0] << 32) | lo[1], side="left"))
    b = len(key) if hi is None else int(np.searchsorted(key, (hi[0] << 32) | hi[1], side="left"))
    return _cov_take(cols, np.arange(a, b, dtype=np.int64))


def _cov_take(cols, idx):
    out = {k: np.asarray(cols[k])[idx] for k in COV_COLS}
    out["cig_off"], out["cigar"] = sam._gather_csr(np.asarray(cols["cig_off"]), np.asarray(cols["cigar"]), idx)
    return out


def _cov_concat(parts):
    parts = [p for p in parts if len(p["pos"])]
    if not parts:
        return dict(tid=np.zeros(0, np.int32), pos=np.zeros(0, np.int32), yc=np.zeros(0, np.float32), strand=np.zeros(0, np.uint8),
                    cig_off=np.zeros(1, np.uint32), cigar=np.zeros(0, np.uint32))
    out = {k: np.concatenate([p[k] for p in parts]) for k in COV_COLS}
    offs, base = [np.zeros(1, np.uint32)], 0
    for p in parts:
        offs.append((p["cig_off"][1:].astype(np.int64) + base).astype(np.uint32))
        base += int(p["cig_off"][-1])
    out["cig_off"] = np.concatenate(offs)
    out["cigar"] = np.concatenate([p["cigar"] for p in parts])
    return out


# --------------------------------------------------------------------------------------------------
# collectives: variable-size all_gather of int64 vectors
# --------------------------------------------------------------------------------------------------
def _dist():
    import torch.distributed as dist
    return dist if (dist.is_available() and dist.is_initialized()) else None


def _comm_device(group=None):
    import torch
    d = _dist()
    if d is not None and d.get_backend(group) == "nccl":
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def allgather_var(vec: np.ndarray, group=None) -> list[np.ndarray]:
    """All ranks contribute an int64 vector of any length; everyone gets the list in rank order.
    Two collectives: lengths, then payloads padded to the longest."""
    import torch
    d = _dist()
    vec = np.ascontiguousarray(vec, dtype=np.int64)
    if d is None or d.get_world_size(group) == 1:
        return [vec]
    dev = _comm_device(group)
    world = d.get_world_size(group)
    ln = torch.tensor([len(vec)], dtype=torch.int64, device=dev)
    lens = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
    d.all_gather(lens, ln, group=group)
    lens = [int(x.item()) for x in lens]
    m = max(max(lens), 1)
    pay = torch.zeros(m, dtype=torch.int64, device=dev)
    if len(vec):
        pay[: len(vec)] = torch.from_numpy(vec).to(dev)
    got = [torch.zeros(m, dtype=torch.int64, device=dev) for _ in range(world)]
    d.all_gather(got, pay, group=group)
    return [g[:l].cpu().numpy() for g, l in zip(got, lens)]


def _pack_cov(cols) -> np.ndarray:
    """Coverage records -> one int64 vector: n, n_cig, then the columns (values widened / bit-cast)."""
    n = len(cols["pos"])
    ncig = int(cols["cig_off"][-1]) if n else 0
    return np.concatenate([
        np.asarray([n, ncig], np.int64), cols["tid"].astype(np.int64), cols["pos"].astype(np.int64),
        cols["yc"].astype(np.float32).view(np.uint32).astype(np.int64), cols["strand"].astype(np.int64),
        cols["cig_off"].astype(np.int64), cols["cigar"][:ncig].astype(np.int64)])


def _unpack_cov(v: np.ndarray):
    n, ncig = int(v[0]), int(v[1])
    o = 2
    tid = v[o:o + n].astype(np.int32); o += n
    pos = v[o:o + n].astype(np.int32); o += n
    yc = v[o:o + n].astype(np.uint32).view(np.float32); o += n
    strand = v[o:o + n].astype(np.uint8); o += n
    cig_off = v[o:o + n + 1].astype(np.uint32); o += n + 1
    cigar = v[o:o + ncig].astype(np.uint32)
    return dict(tid=tid, pos=pos, yc=yc, strand=strand, cig_off=cig_off, cigar=cigar)


# --------------------------------------------------------------------------------------------------
# tiecov
# --------------------------------------------------------------------------------------------------
def _reduce_rows(rows):
    """Junction rows (tid,start,end,strand,value) of ONE bundle gathered from several shards -> reduced by key and
    sorted like CJunc::operator< (start, end, strand char; tiecov.cpp:62-89)."""
    tid, s, e, st, v = rows
    if len(s) == 0:
        return rows
    order = np.lexsort((st, e, s))
    tid, s, e, st, v = tid[order], s[order], e[order], st[order], v[order]
    new = np.ones(len(s), bool)
    new[1:] = (s[1:] != s[:-1]) | (e[1:] != e[:-1]) | (st[1:] != st[:-1])
    idx = np.nonzero(new)[0]
    return tid[idx], s[idx], e[idx], st[idx], np.add.reduceat(v, idx)


def _cat_rows(parts, width):
    if not parts:
        dts = (np.int32, np.int32, np.int32, np.uint8, np.float64) if width == 5 else (np.int32, np.int32, np.int32, np.float64)
        return tuple(np.zeros(0, dt) for dt in dts)
    return tuple(np.concatenate([np.asarray(p[c]) for p in parts]) for c in range(width))


def coverage_shard_local(compute, own, lo, hi, halo_in):
    """The per-rank part of the sharded tiecov: window = halo + own records, runs clipped to [lo,hi), junction rows of
    own records split into (rows of the bundle that continues from the left | the rest), plus the edge descriptors
    the ordered gather needs. `compute(cols, want_runs, want_juncs)` is the device call."""
    n_own = len(own["pos"])
    cont = len(halo_in["pos"]) > 0
    window = _cov_concat([halo_in, own])
    runs = tuple(np.asarray(a) for a in compute(window, True, False)["runs"]) if len(window["pos"]) else _cat_rows([], 4)
    rt, rs, re_, rv = (a.copy() for a in runs)
    if lo is not None:
        m = rt == lo[0]
        rs[m] = np.maximum(rs[m], lo[1])
    if hi is not None:
        m = rt == hi[0]
        re_[m] = np.minimum(re_[m], hi[1])
        keep = ~((rt > hi[0]))
    else:
        keep = np.ones(len(rt), bool)
    keep &= rs < re_
    runs = (rt[keep], rs[keep], re_[keep], rv[keep])
    # ---- junctions: own records only (a halo record was counted by the rank that owns it) ----
    juncs = tuple(np.asarray(a) for a in compute(own, False, True)["juncs"]) if n_own else _cat_rows([], 5)
    n_head = n_tail = 0
    beyond = False
    if n_own:
        e_own = ref_end(own)
        e_before = None
        if cont:
            e_before = (int(halo_in["tid"][0]), int(ref_end(halo_in).max()))
        head = bundle_heads(own["tid"], own["pos"], e_own, e_before)
        hidx = np.nonzero(head)[0]
        beyond = len(hidx) > 0
        jkey = _key(juncs[0], juncs[1] - 1)                   # 0-based first intron base: inside its record, inside its bundle
        if cont:
            # the bundle continuing from the left ends where the first own bundle head starts
            x_end = int(_key(own["tid"][hidx[0]], own["pos"][hidx[0]])) if beyond else np.iinfo(np.int64).max
            n_head = int(np.searchsorted(jkey, x_end, side="left")) if beyond else len(jkey)
            merged = _reduce_rows(tuple(a[:n_head] for a in juncs))   # own-only bundles inside it were split: re-join
            juncs = tuple(np.concatenate([m, a[n_head:]]) for m, a in zip(merged, juncs))
            n_head = len(merged[0])
        if beyond:
            last = int(_key(own["tid"][hidx[-1]], own["pos"][hidx[-1]]))
            jkey = _key(juncs[0], juncs[1] - 1)
            n_tail = int(len(jkey) - max(n_head, np.searchsorted(jkey, last, side="left")))
            # own-only bundles inside the last true bundle are already whole (no halo joins them), but the last true bundle may
            # consist of several own-only bundles only if a halo record bridges them, which is the head bundle: nothing to do
    meta = dict(n_own=n_own, cont=int(cont), beyond=int(beyond), n_head=n_head, n_tail=n_tail)
    return runs, juncs, meta


def _assemble(parts, cuts):
    """Ordered gather on the host: parts[g] = (runs, juncs, meta) of rank g."""
    out_runs = []
    for g, (runs, _, meta) in enumerate(parts):
        if len(runs[0]) == 0:
            continue
        runs = tuple(a.copy() for a in runs)
        if out_runs and meta["cont"] and g > 0:
            p = out_runs[-1]
            ct, cp = cuts[g - 1]
            if p[0][-1] == ct and p[2][-1] == cp and runs[0][0] == ct and runs[1][0] == cp and p[3][-1] == runs[3][0]:
                p[2][-1] = runs[2][0]                         # one run cut in two by the edge
                runs = tuple(a[1:] for a in runs)
        if len(runs[0]):
            out_runs.append(runs)
    runs = _cat_rows(out_runs, 4)
    out_j, open_rows = [], None

    def flush():
        nonlocal open_rows
        if open_rows is not None:
            out_j.append(open_rows[0] if len(open_rows) == 1 else _reduce_rows(_cat_rows(open_rows, 5)))
        open_rows = None

    for runs_g, juncs, meta in parts:
        if meta["n_own"] == 0:
            continue
        h = meta["n_head"]
        if meta["cont"]:
            if open_rows is None:
                open_rows = []
            open_rows.append(tuple(a[:h] for a in juncs))
        if meta["beyond"]:
            flush()
            t = meta["n_tail"]
            nj = len(juncs[0])
            out_j.append(tuple(a[h:nj - t] for a in juncs))
            open_rows = [tuple(a[nj - t:] for a in juncs)]
    flush()
    return runs, _cat_rows(out_j, 5)


def coverage_sharded(compute, own, lo, hi, cuts, group=None):
    """Sharded tiecov -c/-j. Every rank passes the records it owns (start in [lo,hi), coordinate-sorted) and the list of
    all cuts; returns (runs, juncs) in the reference's print order on rank 0 and (None, None) elsewhere.
    compute(cols, want_runs, want_juncs) -> dict(runs=(tid,start0,end0,value), juncs=(tid,start,end,strand,value))."""
    d = _dist()
    rank = d.get_rank(group) if d else 0
    world = d.get_world_size(group) if d else 1
    e_own = ref_end(own) if len(own["pos"]) else np.zeros(0, np.int64)
    # ---- halo: own records reaching past this shard's upper edge ----
    if hi is not None and len(e_own):
        far = np.nonzero((own["tid"] == hi[0]) & (e_own > hi[1]))[0]
    else:
        far = np.zeros(0, np.int64)
    sent = allgather_var(_pack_cov(_cov_take(own, far)), group)
    halo = []
    if lo is not None:
        for g in range(rank):
            c = _unpack_cov(sent[g])
            if len(c["pos"]):
                m = np.nonzero((c["tid"] == lo[0]) & (ref_end(c) > lo[1]))[0]
                halo.append(_cov_take(c, m))
    halo_in = _cov_concat(halo)
    if len(halo_in["pos"]) > 1:
        order = np.argsort(halo_in["pos"], kind="stable")
        halo_in = _cov_take(halo_in, order)
    runs, juncs, meta = coverage_shard_local(compute, own, lo, hi, halo_in)
    # ---- ordered gather ----
    hdr = np.asarray([meta["n_own"], meta["cont"], meta["beyond"], meta["n_head"], meta["n_tail"], len(runs[0]), len(juncs[0])], np.int64)
    pay = np.concatenate([hdr, runs[0].astype(np.int64), runs[1].astype(np.int64), runs[2].astype(np.int64),
                          runs[3].astype(np.float64).view(np.int64), juncs[0].astype(np.int64), juncs[1].astype(np.int64),
                          juncs[2].astype(np.int64), juncs[3].astype(np.int64), juncs[4].astype(np.float64).view(np.int64)])
    got = allgather_var(pay, group)
    if rank != 0:
        return None, None
    parts = []
    for v in got:
        n_own, cont, beyond, n_head, n_tail, nr, nj = (int(x) for x in v[:7])
        o = 7
        r = []
        for dt in (np.int32, np.int32, np.int32):
            r.append(v[o:o + nr].astype(dt)); o += nr
        r.append(v[o:o + nr].copy().view(np.float64)); o += nr
        j = []
        for dt in (np.int32, np.int32, np.int32, np.uint8):
            j.append(v[o:o + nj].astype(dt)); o += nj
        j.append(v[o:o + nj].copy().view(np.float64)); o += nj
        parts.append((tuple(r), tuple(j), dict(n_own=n_own, cont=cont, beyond=beyond, n_head=n_head, n_tail=n_tail)))
    assert len(parts) == world
    return _assemble(parts, cuts)


# --------------------------------------------------------------------------------------------------
# tiebrush
# --------------------------------------------------------------------------------------------------
def _file_slices(cols, run_off, lo, hi):
    """Per-file index ranges of records with lo <= pos < hi in a file-major window (one tid)."""
    pos = np.asarray(cols["pos"])
    idx, off = [], [0]
    for f in range(len(run_off) - 1):
        a, b = int(run_off[f]), int(run_off[f + 1])
        x = a + int(np.searchsorted(pos[a:b], lo, side="left"))
        y = a + int(np.searchsorted(pos[a:b], hi, side="left"))
        idx.append(np.arange(x, y, dtype=np.int64))
        off.append(off[-1] + (y - x))
    return np.concatenate(idx) if idx else np.zeros(0, np.int64), np.asarray(off, np.int64)


def collapse_cuts(cols, run_off, n_shards: int) -> list[int]:
    """n_shards-1 start-position cuts balancing the records of a file-major window."""
    pos = np.sort(np.asarray(cols["pos"]), kind="stable")
    n = len(pos)
    return [int(pos[min(n - 1, (g * n) // n_shards)]) if n else 0 for g in range(1, n_shards)]


def gap_at_or_before(cols, run_off, cut: int) -> int:
    """Largest coordinate c <= cut such that no record of any file with pos < c ends after c (a coverage gap of the union
    of all samples). Every per-sample YD list is emptied by the first read at or past such a coordinate
    (tiebrush.cpp:237-242), so a shard whose input starts there reproduces YD exactly."""
    pos = np.asarray(cols["pos"]).astype(np.int64)
    m = pos < cut
    if not m.any():
        return cut
    p, e = pos[m], ref_end(cols)[m]
    order = np.argsort(p, kind="stable")
    p, e = p[order], e[order]
    pm = np.maximum.accumulate(e)
    if pm[-1] <= cut:
        return cut
    ok = np.nonzero(p[1:] >= pm[:-1])[0]                    # record j+1 starts at or past everything before it
    return int(p[ok[-1] + 1]) if len(ok) else int(p[0])


def collapse_shard_local(compute, cols, run_off, lo, hi, extra=()):
    """One rank of the sharded tiebrush: collapse the slice [gap_at_or_before(lo), hi) and keep the groups whose start is
    >= lo. `compute(sub_cols, sub_run_off)` is the device call (api.Context.collapse_window). Returns rep_index into
    the ORIGINAL window, yc, yx, yd, n_kept (records of [lo,hi) that passed the filters cannot be told apart from the
    look-back ones by the device call, so n_kept is recomputed by the caller if needed)."""
    pos = np.asarray(cols["pos"])
    lo_eff = lo if lo is None else gap_at_or_before(cols, run_off, lo)
    idx, sub_off = _file_slices(cols, run_off, np.iinfo(np.int32).min if lo_eff is None else lo_eff, np.iinfo(np.int32).max if hi is None else hi)
    if len(idx) == 0:
        z = np.zeros(0, np.int64)
        return dict(rep_index=z, yc=np.zeros(0, np.float32), yx=np.zeros(0, np.uint32), yd=np.zeros(0, np.int32))
    sub = sam.take(cols, idx)
    for k in extra:
        sub[k] = cols[k]
    res = compute(sub, sub_off)
    rep = idx[np.asarray(res["rep_index"]).astype(np.int64)]
    keep = np.ones(len(rep), bool) if lo is None else pos[rep] >= lo
    return dict(rep_index=rep[keep], yc=np.asarray(res["yc"])[keep], yx=np.asarray(res["yx"])[keep], yd=np.asarray(res["yd"])[keep])


def collapse_cut_windows(compute, cols, run_off, cuts, yd_carry, pos_range=None, extra=()):
    """Collapse one file-major window (one tid) as a sequence of windows cut at the start positions `cuts` (0-based; a
    window holds the records with cut_i <= pos < cut_i+1), the YD lists carried from each window to the next. No coverage
    gap is needed at a cut. `compute(sub_cols, sub_run_off, pos_range=(lo, hi), yd_carry=carry)` is the call of one window
    (api.Context.collapse_window, or the oracle) and returns the lists it leaves behind as "yd_carry". `yd_carry` = the
    carry the first window starts from (the result of the previous tid, or an empty one). `pos_range` = (lo, hi) of the
    whole window, default (min pos, max pos + 1). Returns the concatenated groups with rep_index into `cols`, n_kept, the
    final yd_carry and the carried segments per cut (`carried`)."""
    pos = np.asarray(cols["pos"])
    if pos_range is None:
        pos_range = (int(pos.min()), int(pos.max()) + 1) if len(pos) else (0, 1)
    lo, hi = int(pos_range[0]), int(pos_range[1])
    bounds = [lo] + sorted({int(c) for c in cuts if lo < int(c) < hi}) + [hi]
    reps, ycs, yxs, yds, carried, kept = [], [], [], [], [], 0
    for a, b in zip(bounds[:-1], bounds[1:]):
        idx, sub_off = _file_slices(cols, run_off, a, b)
        sub = sam.take(cols, idx)
        for k in extra:
            sub[k] = cols[k]
        res = compute(sub, sub_off, pos_range=(a, b), yd_carry=yd_carry)
        yd_carry = res["yd_carry"]
        carried.append(int(yd_carry["chain_off"][-1]))
        reps.append(idx[np.asarray(res["rep_index"]).astype(np.int64)])
        ycs.append(np.asarray(res["yc"])); yxs.append(np.asarray(res["yx"])); yds.append(np.asarray(res["yd"]))
        kept += int(res["n_kept"])
    return dict(rep_index=np.concatenate(reps), yc=np.concatenate(ycs).astype(np.float32), yx=np.concatenate(yxs).astype(np.uint32),
                yd=np.concatenate(yds).astype(np.int32), n_kept=kept, yd_carry=yd_carry, carried=carried)


def collapse_sharded(compute, cols, run_off, cuts, group=None):
    """Sharded tiebrush over one window every rank can read (each rank slices its own coordinate range, as a host
    reader with a BAM index would). Ordered gather of the groups on rank 0."""
    d = _dist()
    rank = d.get_rank(group) if d else 0
    world = d.get_world_size(group) if d else 1
    lo = None if rank == 0 else cuts[rank - 1]
    hi = None if rank == world - 1 else cuts[rank]
    r = collapse_shard_local(compute, cols, run_off, lo, hi)
    g = len(r["rep_index"])
    pay = np.concatenate([np.asarray([g], np.int64), r["rep_index"].astype(np.int64), r["yc"].astype(np.float32).view(np.uint32).astype(np.int64),
                          r["yx"].astype(np.int64), r["yd"].astype(np.int64)])
    got = allgather_var(pay, group)
    if rank != 0:
        return None
    reps, ycs, yxs, yds = [], [], [], []
    for v in got:
        g = int(v[0])
        reps.append(v[1:1 + g]); ycs.append(v[1 + g:1 + 2 * g].astype(np.uint32).view(np.float32))
        yxs.append(v[1 + 2 * g:1 + 3 * g].astype(np.uint32)); yds.append(v[1 + 3 * g:1 + 4 * g].astype(np.int32))
    return dict(rep_index=np.concatenate(reps), yc=np.concatenate(ycs), yx=np.concatenate(yxs), yd=np.concatenate(yds))


# --------------------------------------------------------------------------------------------------
# tiecov -s (sample heat-map) over coordinate shards
# --------------------------------------------------------------------------------------------------
def sample_shard_local(compute, cols, lo, hi):
    """One rank of the sharded tiecov -s over a stream every rank can read. The running mean of a base folds ALL records
    covering it in stream order, and those lie in the base's own bundle, so the rank computes from the head of the bundle
    that is open at `lo` up to `hi` and keeps the part of every row inside [lo, hi). `compute(cols)` -> rows
    (tid, start0, end0, ival) of whole bundles, cols incl. `yx`. Returns (rows, lo_inside_bundle)."""
    key = _key(cols["tid"], cols["pos"])
    n = len(key)
    a = 0 if lo is None else int(np.searchsorted(key, (lo[0] << 32) | lo[1], side="left"))
    b = n if hi is None else int(np.searchsorted(key, (hi[0] << 32) | hi[1], side="left"))
    empty = tuple(np.zeros(0, dt) for dt in (np.int32, np.int32, np.int32, np.uint64))
    end = ref_end(cols)
    head = bundle_heads(np.asarray(cols["tid"]), np.asarray(cols["pos"]), end)
    # Is a bundle open at `lo`? Decided from the running maximum end of the records BEFORE the cut (0-based exclusive end
    # > lo's position on lo's tid), not from the first record at or after it: the bundle may reach beyond the cut without
    # any further record of it starting there, and then its bases in [lo, bundle end) belong to this rank all the same.
    inside = False
    if lo is not None and a > 0:
        pm_before = int(np.max(_key(cols["tid"], end)[:a]))      # keys grow with tid, so the maximum sits on the last tid
        inside = (pm_before >> 32) == lo[0] and (pm_before & 0xFFFFFFFF) > lo[1]
    if a >= b and not inside:
        return empty, inside
    a0 = a
    if inside:
        a0 = a - 1
        while not head[a0]:
            a0 -= 1
        # records [a0, a) open the bundle; if the first record at or after the cut starts a NEW bundle it is simply the next
        # bundle of this rank's window
    if a0 >= b:
        return empty, inside
    idx = np.arange(a0, b, dtype=np.int64)
    sub = _cov_take(cols, idx)
    sub["yx"] = np.asarray(cols["yx"])[idx]
    t, s, e, v = (np.asarray(x) for x in compute(sub))
    # clip to [lo, hi): a row is kept for the part whose 0-based positions start at or after lo (records before lo belong to
    # the left neighbour's range), and nothing can reach beyond this rank's last record start + its span except through
    # records starting before hi, which are all here; positions >= hi on the same tid belong to the right neighbour
    s = s.astype(np.int64).copy(); e = e.astype(np.int64).copy()
    if lo is not None:
        on = t == lo[0]
        s[on] = np.maximum(s[on], lo[1])
        keep = (t > lo[0]) | (on & (e > s))
    else:
        keep = np.ones(len(t), bool)
    if hi is not None:
        on = t == hi[0]
        e[on] = np.minimum(e[on], hi[1])
        keep &= (t < hi[0]) | (on & (e > s))
    return (t[keep].astype(np.int32), s[keep].astype(np.int32), e[keep].astype(np.int32), v[keep].astype(np.uint64)), inside


def _stitch_sample(parts):
    """Rank-ordered rows; a row that ends exactly where the next rank's first row starts, same tid and value, is one row of
    the unsharded output iff the cut fell inside a bundle (rows never join across bundles, tiecov.cpp:293-309)."""
    out = [[], [], [], []]
    for rows, inside in parts:
        t, s, e, v = rows
        last = next((i for i in range(len(out[0]) - 1, -1, -1) if len(out[0][i])), None)   # a rank may have contributed no row
        if len(t) and last is not None and inside:
            lt, ls, le, lv = out[0][last], out[1][last], out[2][last], out[3][last]
            if lt[-1] == t[0] and le[-1] == s[0] and lv[-1] == v[0]:
                le[-1] = e[0]
                t, s, e, v = t[1:], s[1:], e[1:], v[1:]
        for q, x in zip(out, (t, s, e, v)):
            q.append(np.array(x, copy=True))
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)
    return cat(out[0], np.int32), cat(out[1], np.int32), cat(out[2], np.int32), cat(out[3], np.uint64)


def sample_sharded(compute, cols, cuts, group=None):
    """Sharded tiecov -s: rank g owns the coordinate range [cuts[g-1], cuts[g]) of a stream all ranks can read; rows are
    gathered in rank order (one variable-size all_gather) and stitched at the cuts. Every rank returns the full rows."""
    d = _dist()
    rank = d.get_rank(group) if d is not None else 0
    bounds = [None] + list(cuts) + [None]
    rows, inside = sample_shard_local(compute, cols, bounds[rank], bounds[rank + 1])
    vec = np.concatenate([[len(rows[0]), int(inside)], rows[0].astype(np.int64), rows[1].astype(np.int64), rows[2].astype(np.int64),
                          rows[3].astype(np.int64)]).astype(np.int64)
    parts = []
    for v in allgather_var(vec, group):
        m, ins = int(v[0]), bool(v[1])
        body = v[2:]
        parts.append(((body[:m].astype(np.int32), body[m:2 * m].astype(np.int32), body[2 * m:3 * m].astype(np.int32), body[3 * m:4 * m].astype(np.uint64)), ins))
    return _stitch_sample(parts)
