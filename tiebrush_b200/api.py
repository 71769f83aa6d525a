"""Host-side Python mirror of the hot-path interface, one level above the C ABI.

`Context` plays the role of the reference's global option state (struct Options / mrgStrategy,
src/tiebrush.cpp:89-100); `collapse_window` stands where main()'s loop calls TInputFiles::next +
passes_options + addPData + flushPData (tiebrush.cpp:570-592) and `coverage_window` where tiecov's
loop calls addCov / flushCoverage / addJunction / flushJuncs (tiecov.cpp:435-528).

Column dicts use the tiebrush_b200.sam.to_columns layout. Values may be numpy arrays (host path:
the library copies host<->device inside the call) or torch CUDA tensors (device-resident path)."""
from __future__ import annotations

import ctypes as C
import numpy as np

from . import _lib

NO_MAX_NH = 0x7FFFFFFF


class TieBrushError(RuntimeError):
    pass


def compact_cigar_columns(cig_off, cigar):
    """Host packer of the compact wire format: (n_cigar8, cigar16, cigar_ext) from the wide CSR columns (numpy or torch)."""
    if _is_torch(cigar):   # chunked, 32-bit arithmetic on the bit patterns: a full-size window has 2.7e9 CIGAR words
        import torch
        n = int(cig_off.shape[0]) - 1
        n8 = torch.empty(n, dtype=torch.uint8, device=cigar.device)
        step = 1 << 27
        for a0 in range(0, n, step):
            a1 = min(n, a0 + step)
            d = cig_off[a0 + 1:a1 + 1] - cig_off[a0:a1]          # wraps correctly in int32 (u32 bit patterns)
            if int(d.max()) >= 256 or int(d.min()) < 0:
                raise ValueError("a record with >= 256 CIGAR ops needs the wide format")
            n8[a0:a1] = d.to(torch.uint8)
        m = int(cigar.shape[0])
        c16 = torch.empty(m, dtype=torch.int16, device=cigar.device)
        exts = []
        for a0 in range(0, m, step):
            w = cigar[a0:a0 + step]
            ln = (w >> 4) & 0x0FFFFFFF
            esc = ln >= 0xFFF
            c16[a0:a0 + step] = ((w & 0xF) | (torch.where(esc, torch.full_like(ln, 0xFFF), ln) << 4)).to(torch.int16)
            exts.append(ln[esc])
        return n8, c16, torch.cat(exts) if exts else torch.empty(0, dtype=torch.int32, device=cigar.device)
    off = np.asarray(cig_off).astype(np.int64); w = np.asarray(cigar).astype(np.int64)
    nc = off[1:] - off[:-1]
    if len(nc) and nc.max() >= 256:
        raise ValueError("a record with >= 256 CIGAR ops needs the wide format")
    ln = w >> 4
    esc = ln >= 0xFFF
    c16 = ((w & 0xF) | (np.where(esc, 0xFFF, ln) << 4)).astype(np.uint16)
    return nc.astype(np.uint8), c16, ln[esc].astype(np.uint32)


def _is_torch(a):
    return hasattr(a, "data_ptr")


def _ptr(a):
    if a is None:
        return None
    if _is_torch(a):
        return a.data_ptr()
    return a.ctypes.data


def _host(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def pack_fixed_columns(cols, run_off, max_dict=255):
    """Host packer of the packed wire format of the fixed columns (include/tiebrush_b200.h): pos -> pos_d8 (+ pos_ext),
    (flag, mapq, strand, nh) -> meta8 (+ meta_dict, meta_ext). numpy or torch columns in, same kind out (meta_dict always
    numpy). What a host packer would fill directly; here built from the wide columns."""
    pos = cols["pos"]
    tor = _is_torch(pos)
    n = int(pos.shape[0])
    starts = np.asarray(run_off[:-1], np.int64)
    starts = starts[starts < n]
    if tor:
        import torch
        dev = pos.device
        d = torch.empty(n, dtype=torch.int64, device=dev)
        d[0:1] = 0
        d[1:] = pos[1:].to(torch.int64) - pos[:-1].to(torch.int64)
        is_start = torch.zeros(n, dtype=torch.bool, device=dev)
        is_start[torch.as_tensor(starts, device=dev)] = True
        esc = is_start | (d >= 254) | (d < 0)
        absolute = is_start | (d < 0)
        d8 = torch.where(absolute, 255, torch.where(esc, 254, d)).to(torch.uint8)
        ext = torch.where(absolute, pos.to(torch.int64), d)[esc].to(torch.int32)
        del d, is_start, esc, absolute
        tup = (cols["flag"].to(torch.int64) & 0xffff) | ((cols["mapq"].to(torch.int64) & 0xff) << 16) | ((cols["strand"].to(torch.int64) & 0xff) << 24) | ((cols["nh"].to(torch.int64) & 0xffff) << 32)
        samp = tup[:: max(1, n // 4_000_000)]
        vals, cnts = torch.unique(samp, return_counts=True)
        order = torch.argsort(cnts, descending=True)[:max_dict]
        dict_sorted = torch.sort(vals[order]).values
        idx = torch.searchsorted(dict_sorted, tup).clamp(max=max(len(dict_sorted) - 1, 0))
        hit = dict_sorted[idx] == tup if len(dict_sorted) else torch.zeros(n, dtype=torch.bool, device=dev)
        m8 = torch.where(hit, idx, 255).to(torch.uint8)
        mext = tup[~hit]
        return dict(pos_d8=d8, pos_ext=ext, meta8=m8, meta_ext=mext, meta_dict=dict_sorted.cpu().numpy().astype(np.uint64))
    pos64 = np.asarray(pos).astype(np.int64)
    d = np.zeros(n, np.int64)
    d[1:] = pos64[1:] - pos64[:-1]
    is_start = np.zeros(n, bool); is_start[starts] = True
    absolute = is_start | (d < 0)
    esc = absolute | (d >= 254)
    d8 = np.where(absolute, 255, np.where(esc, 254, d)).astype(np.uint8)
    ext = np.where(absolute, pos64, d)[esc].astype(np.int32)
    tup = (np.asarray(cols["flag"]).astype(np.uint64) & 0xffff) | ((np.asarray(cols["mapq"]).astype(np.uint64) & 0xff) << np.uint64(16)) | \
          ((np.asarray(cols["strand"]).astype(np.uint64) & 0xff) << np.uint64(24)) | ((np.asarray(cols["nh"]).astype(np.uint64) & 0xffff) << np.uint64(32))
    vals, cnts = np.unique(tup, return_counts=True)
    dict_sorted = np.sort(vals[np.argsort(-cnts, kind="stable")[:max_dict]])
    if len(dict_sorted):
        idx = np.minimum(np.searchsorted(dict_sorted, tup), len(dict_sorted) - 1)
        hit = dict_sorted[idx] == tup
    else:
        idx, hit = np.zeros(n, np.int64), np.zeros(n, bool)
    m8 = np.where(hit, idx, 255).astype(np.uint8)
    return dict(pos_d8=d8, pos_ext=ext, meta8=m8, meta_ext=tup[~hit].astype(np.uint64), meta_dict=dict_sorted.astype(np.uint64))


def empty_yd_carry(n_samples):
    """The YD carry a stream starts from: no lists (what tb_collapse_window assumes). Pass it, or the yd_carry of the
    previous window's result, as collapse_window(..., yd_carry=)."""
    return dict(tid=-1, pos_hi=0, chain_off=np.zeros(2 * n_samples + 1, np.int64), seg_start=np.zeros(0, np.int32),
                seg_end=np.zeros(0, np.int32))


class Context:
    def __init__(self, device=0, n_samples=1, mode=0, flag_mask=0, max_nh=NO_MAX_NH, min_qual=-1, keep_bits=0, collapse_same=0):
        self.lib = _lib.load()
        self.h = self.lib.tb_create(device, n_samples, mode, flag_mask, max_nh, min_qual, keep_bits, collapse_same)
        if not self.h:
            raise TieBrushError(self.lib.tb_last_error(None).decode())
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.tb_destroy(self.h)
            self.h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _err(self):
        return self.lib.tb_last_error(self.h).decode()

    def set_stream(self, cuda_stream_ptr):
        self.lib.tb_set_stream(self.h, cuda_stream_ptr)

    def set_profiling(self, on=True):
        self.lib.tb_set_profiling(self.h, int(on))

    def last_kernel_ms(self, which):
        return float(self.lib.tb_last_kernel_ms(self.h, which))

    def launch_count(self):
        return int(self.lib.tb_launch_count(self.h))

    def last_heavy_slots(self):
        return int(self.lib.tb_last_heavy_slots(self.h))

    def last_ord_deep(self):
        """Ordered front end, last call: start positions handled by the one-warp-per-position kernel."""
        return int(self.lib.tb_last_ord_deep(self.h))

    def last_tile_gen(self):
        """1 once a collapse call has run the tile kernel (col_tile_kernel, the only generation), 0 before."""
        return int(self.lib.tb_last_tile_gen(self.h))

    def last_tile_stats(self):
        """Tile statistics: multi_pass, deferred_records and deferred_slots are always 0; slots is the slot count of the
        last tile-path call that ran the 256-thread geometry (0 before any)."""
        return dict(zip(("multi_pass", "deferred_records", "deferred_slots", "slots"), (int(self.lib.tb_last_tile_stat(self.h, i)) for i in range(4))))

    def last_yd_path(self):
        """0 parallel YD formulation, 1 sequential segment lists."""
        return int(self.lib.tb_last_yd_path(self.h))

    def last_yd_stats(self):
        """YD stage of the last collapse call: chain members, sub-chains, compact length Lc (0 on the sequential path), 1024-group blocks."""
        return dict(zip(("n_members", "n_subchains", "lc", "nblk"), (int(self.lib.tb_last_yd_stat(self.h, i)) for i in range(4))))

    def last_path(self):
        """0 tile path, 1 ordered path (by options), 2 ordered path (table-overflow fallback)."""
        return int(self.lib.tb_last_path(self.h))

    # ------------------------------------------------------------------------------------------
    def collapse_window(self, cols, run_off, tid=0, file_merged=None, pos_range=None, out=None, yd_carry=None):
        """One window of tiebrush. Returns dict(rep_index, yc, yx, yd, n_kept, n_groups).
        yd_carry: the YD lists carried in from the window before (empty_yd_carry(k), or the "yd_carry" of the previous
        result); the window may then start at any start position, not only at a coverage gap. The result then holds the
        lists this window leaves behind under "yd_carry" (dict of numpy arrays: tid, pos_hi, chain_off, seg_start,
        seg_end; chain c = side * k + sample). Without it the call is tb_collapse_window, unchanged."""
        first = cols["pos"] if cols.get("pos") is not None else cols["pos_d8"]
        dev = _is_torch(first)
        n = int(first.shape[0])
        run_off = _host(run_off, np.int64)
        k = len(run_off) - 1
        keep = []  # keep converted arrays alive

        def col(name, dt):
            a = cols.get(name)
            if a is None:
                return None
            if not dev:
                a = _host(a, dt)
            keep.append(a)
            return a

        pos, flag, mapq = col("pos", np.int32), col("flag", np.uint16), col("mapq", np.uint8)
        strand, nh = col("strand", np.uint8), col("nh", np.uint16)
        cig_off, cigar = col("cig_off", np.uint32), col("cigar", np.uint32)
        # compact wire format of the CIGAR columns (see include/tiebrush_b200.h); used when the wide column is absent
        n8, c16, cext = col("n_cigar8", np.uint8), col("cigar16", np.uint16), col("cigar_ext", np.uint32)
        # packed wire format of the fixed columns (pos_d8 / meta8, see include/tiebrush_b200.h); used when the wide column is absent
        pd8, pext = col("pos_d8", np.uint8), col("pos_ext", np.int32)
        m8, mext = col("meta8", np.uint8), col("meta_ext", np.uint64)
        mdict = _host(cols["meta_dict"], np.uint64) if cols.get("meta_dict") is not None else None   # always host memory
        keep.append(mdict)
        md_off, md = col("md_off", np.uint32), col("md", np.uint8)
        qh = col("qhash", np.uint64)
        fm = _host(file_merged, np.uint8) if file_merged is not None else None
        yc_in = col("yc_in", np.float32) if fm is not None else None
        yx_in = col("yx_in", np.int32) if fm is not None else None
        yd_in = col("yd_in", np.int32) if fm is not None else None
        n_cig = int(cols["n_cig"]) if "n_cig" in cols else (int(cig_off[-1]) if (n and cig_off is not None) else (int(c16.shape[0]) if c16 is not None else 0))
        n_ext = int(cext.shape[0]) if cext is not None else 0
        n_md = int(cols["n_md"]) if "n_md" in cols else (int(md_off[-1]) if (md_off is not None and n) else 0)
        if pos_range is None:
            if dev:
                raise ValueError("pos_range=(lo,hi) is required for device-resident windows")
            if pos is None:
                raise ValueError("pos_range=(lo,hi) is required with the packed wire format")
            pos_range = (int(pos.min()), int(pos.max()) + 1) if n else (0, 0)
        sin = _lib.SoaIn(n, k, tid, _ptr(run_off), _ptr(fm), _ptr(pos), _ptr(flag), _ptr(mapq), _ptr(strand), _ptr(nh),
                         _ptr(cig_off), _ptr(cigar), _ptr(md_off), _ptr(md), _ptr(qh), _ptr(yc_in), _ptr(yx_in), _ptr(yd_in),
                         1 if dev else 0, n_cig, n_md, pos_range[0], pos_range[1], _ptr(n8), _ptr(c16), _ptr(cext), n_ext,
                         _ptr(pd8), _ptr(pext), int(pext.shape[0]) if pext is not None else 0, _ptr(m8), _ptr(mdict),
                         int(mdict.shape[0]) if mdict is not None else 0, _ptr(mext), int(mext.shape[0]) if mext is not None else 0)
        cap = max(n, 1)
        if out is None:
            if dev:
                import torch
                d = first.device
                out = dict(rep_index=torch.empty(cap, dtype=torch.int32, device=d), yc=torch.empty(cap, dtype=torch.float32, device=d),
                           yx=torch.empty(cap, dtype=torch.int32, device=d), yd=torch.empty(cap, dtype=torch.int32, device=d))
            else:
                out = dict(rep_index=np.empty(cap, np.uint32), yc=np.empty(cap, np.float32), yx=np.empty(cap, np.uint32), yd=np.empty(cap, np.int32))
        o = _lib.GroupsOut(int(out["rep_index"].shape[0]), 0, 0, _ptr(out["rep_index"]), _ptr(out["yc"]), _ptr(out["yx"]), _ptr(out["yd"]),
                           1 if _is_torch(out["rep_index"]) else 0)
        if yd_carry is None:
            rc = self.lib.tb_collapse_window(self.h, C.byref(sin), C.byref(o))
            if rc != 0:
                raise TieBrushError(self._err())
        else:
            ci = {key: _host(yd_carry[key], dt) for key, dt in (("chain_off", np.int64), ("seg_start", np.int32), ("seg_end", np.int32))}
            cin = _lib.YdCarry(int(yd_carry["tid"]), int(yd_carry["pos_hi"]), len(ci["chain_off"]) - 1, len(ci["seg_start"]),
                               int(ci["chain_off"][-1]), _ptr(ci["chain_off"]), _ptr(ci["seg_start"]), _ptr(ci["seg_end"]))
            cap = max(4096, 2 * len(ci["seg_start"]) + 8 * k)
            while True:   # a carry_out too small for the lists: the call says how many there are
                co = dict(chain_off=np.zeros(2 * k + 1, np.int64), seg_start=np.zeros(cap, np.int32), seg_end=np.zeros(cap, np.int32))
                cout = _lib.YdCarry(0, 0, 2 * k, cap, 0, _ptr(co["chain_off"]), _ptr(co["seg_start"]), _ptr(co["seg_end"]))
                rc = self.lib.tb_collapse_window_carry(self.h, C.byref(sin), C.byref(cin), C.byref(o), C.byref(cout))
                if rc == 0 or int(cout.n_segs) <= cap:
                    break
                cap = int(cout.n_segs)
            if rc != 0:
                raise TieBrushError(self._err())
            m = int(cout.n_segs)
            carry = dict(tid=int(cout.tid), pos_hi=int(cout.pos_hi), chain_off=co["chain_off"], seg_start=co["seg_start"][:m], seg_end=co["seg_end"][:m])
        g = int(o.n_groups)
        res = dict(rep_index=out["rep_index"][:g], yc=out["yc"][:g], yx=out["yx"][:g], yd=out["yd"][:g], n_kept=int(o.n_kept), n_groups=g)
        if yd_carry is not None:
            res["yd_carry"] = carry
        return res

    # ------------------------------------------------------------------------------------------
    def sample_window(self, cols, cap_rows=None):
        """tiecov -s of one window (whole bundles): rows (tid, start0, end0, ival) of the sample-count heat-map; `cols` needs
        tid, pos, yc, strand, cig_off, cigar as for coverage_window plus yx (YX tag, 1 when absent). Host columns only."""
        n = int(cols["pos"].shape[0])
        keep = [_host(cols[k], dt) for k, dt in (("tid", np.int32), ("pos", np.int32), ("yc", np.float32), ("strand", np.uint8),
                                                 ("cig_off", np.uint32), ("cigar", np.uint32), ("yx", np.int32))]
        tid, pos, yc, strand, cig_off, cigar, yx = keep
        n_cig = int(cig_off[-1]) if n else 0
        cin = _lib.CovIn(n, _ptr(tid), _ptr(pos), _ptr(yc), _ptr(strand), _ptr(cig_off), _ptr(cigar), 0, n_cig)
        cap = cap_rows if cap_rows is not None else 2 * n_cig + 16
        rt, rs, re, rv = np.empty(cap, np.int32), np.empty(cap, np.int32), np.empty(cap, np.int32), np.empty(cap, np.float64)
        rows = _lib.RunsOut(cap, 0, _ptr(rt), _ptr(rs), _ptr(re), _ptr(rv), 0)
        rc = self.lib.tc_sample_window(self.h, C.byref(cin), _ptr(yx), C.byref(rows))
        if rc == 2:
            raise ValueError(self._err())
        if rc != 0:
            raise TieBrushError(self._err())
        r = int(rows.n_runs)
        return rt[:r], rs[:r], re[:r], rv[:r].astype(np.uint64)

    def coverage_window(self, cols, want_runs=True, want_juncs=True, cap_runs=None, cap_juncs=None, out=None):
        """One window of tiecov -c/-j. Returns dict(runs=(tid,start0,end0,value), juncs=(tid,start,end,strand,value))."""
        dev = _is_torch(cols["pos"])
        n = int(cols["pos"].shape[0])
        keep = []

        def col(name, dt):
            a = cols[name]
            if not dev:
                a = _host(a, dt)
            keep.append(a)
            return a

        tid, pos, yc = col("tid", np.int32), col("pos", np.int32), col("yc", np.float32)
        strand, cig_off, cigar = col("strand", np.uint8), col("cig_off", np.uint32), col("cigar", np.uint32)
        n_cig = int(cols["n_cig"]) if "n_cig" in cols else (int(cig_off[-1]) if n else 0)
        end = cols.get("end")
        if end is not None:
            end = end if dev else _host(end, np.int32)
            keep.append(end)
        cin = _lib.CovIn(n, _ptr(tid), _ptr(pos), _ptr(yc), _ptr(strand), _ptr(cig_off), _ptr(cigar), 1 if dev else 0, n_cig, _ptr(end))
        capr = cap_runs if cap_runs is not None else 2 * n_cig + 16
        capj = cap_juncs if cap_juncs is not None else n_cig + 16
        if out is None:
            if dev:
                import torch
                d = cols["pos"].device
                i32 = lambda m: torch.empty(m, dtype=torch.int32, device=d)
                out = dict(r_tid=i32(capr), r_start=i32(capr), r_end=i32(capr), r_val=torch.empty(capr, dtype=torch.float64, device=d),
                           j_tid=i32(capj), j_start=i32(capj), j_end=i32(capj), j_strand=torch.empty(capj, dtype=torch.uint8, device=d),
                           j_val=torch.empty(capj, dtype=torch.float64, device=d))
            else:
                out = dict(r_tid=np.empty(capr, np.int32), r_start=np.empty(capr, np.int32), r_end=np.empty(capr, np.int32), r_val=np.empty(capr, np.float64),
                           j_tid=np.empty(capj, np.int32), j_start=np.empty(capj, np.int32), j_end=np.empty(capj, np.int32),
                           j_strand=np.empty(capj, np.uint8), j_val=np.empty(capj, np.float64))
        odev = 1 if _is_torch(out["r_tid"]) else 0
        runs = _lib.RunsOut(int(out["r_tid"].shape[0]), 0, _ptr(out["r_tid"]), _ptr(out["r_start"]), _ptr(out["r_end"]), _ptr(out["r_val"]), odev)
        juncs = _lib.JuncsOut(int(out["j_tid"].shape[0]), 0, _ptr(out["j_tid"]), _ptr(out["j_start"]), _ptr(out["j_end"]), _ptr(out["j_strand"]),
                              _ptr(out["j_val"]), odev)
        rc = self.lib.tc_coverage_window(self.h, C.byref(cin), C.byref(runs) if want_runs else None, C.byref(juncs) if want_juncs else None)
        if rc == 2:
            raise ValueError(self._err())
        if rc != 0:
            raise TieBrushError(self._err())
        r, j = int(runs.n_runs), int(juncs.n_juncs)
        return dict(runs=(out["r_tid"][:r], out["r_start"][:r], out["r_end"][:r], out["r_val"][:r]),
                    juncs=(out["j_tid"][:j], out["j_start"][:j], out["j_end"][:j], out["j_strand"][:j], out["j_val"][:j]),
                    n_runs=r, n_juncs=j)


# ---------------------------------------------------------------------------------------------------------------------
# tiecov over long streams / several GPUs (csrc/shard.cu): thin ctypes plumbing, no logic of its own
# ---------------------------------------------------------------------------------------------------------------------
def _cov_in(cols, keep):
    """tc_soa_in for a column dict (numpy or torch); `keep` collects the arrays that must outlive the call."""
    dev = _is_torch(cols["pos"])
    n = int(cols["pos"].shape[0])
    arrs = []
    for name, dt in (("tid", np.int32), ("pos", np.int32), ("yc", np.float32), ("strand", np.uint8), ("cig_off", np.uint32), ("cigar", np.uint32)):
        a = cols[name]
        if not dev:
            a = _host(a, dt)
        keep.append(a)
        arrs.append(a)
    n_cig = int(cols["n_cig"]) if "n_cig" in cols else (int(arrs[4][-1]) - int(arrs[4][0]) if n else 0)
    end = cols.get("end")
    if end is not None:
        if not dev:
            end = _host(end, np.int32)
        keep.append(end)
    return _lib.CovIn(n, *[_ptr(a) for a in arrs], 1 if dev else 0, n_cig, _ptr(end))


def cov_out_buffers(cap_runs, cap_juncs, device=None):
    """Output arrays of a coverage call (torch on `device`, or numpy when device is None)."""
    if device is not None:
        import torch
        i32 = lambda m: torch.empty(m, dtype=torch.int32, device=device)
        return dict(r_tid=i32(cap_runs), r_start=i32(cap_runs), r_end=i32(cap_runs), r_val=torch.empty(cap_runs, dtype=torch.float64, device=device),
                    j_tid=i32(cap_juncs), j_start=i32(cap_juncs), j_end=i32(cap_juncs), j_strand=torch.empty(cap_juncs, dtype=torch.uint8, device=device),
                    j_val=torch.empty(cap_juncs, dtype=torch.float64, device=device))
    return dict(r_tid=np.empty(cap_runs, np.int32), r_start=np.empty(cap_runs, np.int32), r_end=np.empty(cap_runs, np.int32), r_val=np.empty(cap_runs, np.float64),
                j_tid=np.empty(cap_juncs, np.int32), j_start=np.empty(cap_juncs, np.int32), j_end=np.empty(cap_juncs, np.int32),
                j_strand=np.empty(cap_juncs, np.uint8), j_val=np.empty(cap_juncs, np.float64))


def _out_structs(out):
    odev = 1 if _is_torch(out["r_tid"]) else 0
    runs = _lib.RunsOut(int(out["r_tid"].shape[0]), 0, _ptr(out["r_tid"]), _ptr(out["r_start"]), _ptr(out["r_end"]), _ptr(out["r_val"]), odev)
    juncs = _lib.JuncsOut(int(out["j_tid"].shape[0]), 0, _ptr(out["j_tid"]), _ptr(out["j_start"]), _ptr(out["j_end"]), _ptr(out["j_strand"]), _ptr(out["j_val"]), odev)
    return runs, juncs


def _rows(out, r, j):
    return dict(runs=(out["r_tid"][:r], out["r_start"][:r], out["r_end"][:r], out["r_val"][:r]),
                juncs=(out["j_tid"][:j], out["j_start"][:j], out["j_end"][:j], out["j_strand"][:j], out["j_val"][:j]), n_runs=r, n_juncs=j)


def _coverage_stream(self, cols, window, out, next_tid_pos=None):
    """tc_coverage_stream: one slice in windows cut at bundle heads. Returns the rows and `consumed`."""
    keep = []
    cin = _cov_in(cols, keep)
    runs, juncs = _out_structs(out)
    nx = None
    if next_tid_pos is not None:
        nx = (C.c_int32 * 2)(int(next_tid_pos[0]), int(next_tid_pos[1]))
    consumed = C.c_int64(0)
    rc = self.lib.tc_coverage_stream(self.h, C.byref(cin), int(window), nx, C.byref(runs), C.byref(juncs), C.byref(consumed))
    if rc == 2:
        raise ValueError(self._err())
    if rc != 0:
        raise TieBrushError(self._err())
    res = _rows(out, int(runs.n_runs), int(juncs.n_juncs))
    res["consumed"] = int(consumed.value)
    res["windows"] = int(self.lib.tc_stream_windows(self.h))
    return res


def _comm_unique_id():
    buf = (C.c_ubyte * 128)()
    lib = _lib.load()
    if lib.tb_comm_unique_id(buf) != 0:
        raise TieBrushError(lib.tb_last_error(None).decode())
    return bytes(buf)


def _comm_init(self, rank, world, unique_id):
    buf = (C.c_ubyte * 128).from_buffer_copy(unique_id)
    if self.lib.tb_comm_init(self.h, int(rank), int(world), buf) != 0:
        raise TieBrushError(self._err())


def _shard_coverage(self, segs, window, out):
    """tc_shard_coverage over this rank's device-resident segments (list of column dicts). Collective."""
    keep = []
    arr = (_lib.CovIn * len(segs))(*[_cov_in(s, keep) for s in segs])
    runs, juncs = _out_structs(out)
    rc = self.lib.tc_shard_coverage(self.h, arr, len(segs), int(window), C.byref(runs), C.byref(juncs))
    if rc == 2:
        raise ValueError(self._err())
    if rc != 0:
        raise TieBrushError(self._err())
    res = _rows(out, int(runs.n_runs), int(juncs.n_juncs))
    res["windows"] = int(self.lib.tc_stream_windows(self.h))
    res["stats"] = dict(zip(("lead_received", "lead_sent", "ranks_received_from", "halo_bytes_sent", "seam_records"),
                            (int(self.lib.tc_shard_stat(self.h, i)) for i in range(5))))
    return res


def _shard_gather(self, local, all_out, world):
    """tc_shard_gather: ordered gather of `local` (result of shard_coverage, device rows) into `all_out` on rank 0. Collective."""
    lr = _lib.RunsOut(int(local["n_runs"]), int(local["n_runs"]), *[_ptr(a) for a in local["runs"]], 1)
    lj = _lib.JuncsOut(int(local["n_juncs"]), int(local["n_juncs"]), *[_ptr(a) for a in local["juncs"]], 1)
    base = (C.c_int64 * (world + 1))()
    if all_out is not None:
        ar, aj = _out_structs(all_out)
        rc = self.lib.tc_shard_gather(self.h, C.byref(lr), C.byref(lj), C.byref(ar), C.byref(aj), base)
    else:
        rc = self.lib.tc_shard_gather(self.h, C.byref(lr), C.byref(lj), None, None, base)
    if rc != 0:
        raise TieBrushError(self._err())
    res = dict(junc_base=[int(x) for x in base], gather_bytes=int(self.lib.tc_shard_stat(self.h, 5)))
    if all_out is not None:
        res.update(_rows(all_out, int(ar.n_runs), int(aj.n_juncs)))
    return res


def _shard_coverage_gather(self, segs, window, out, all_out, cap_runs_all, cap_juncs_all, world):
    """tc_shard_coverage_gather: this rank's windows with the ordered gather on rank 0 overlapped (one round per window on a
    second stream). `all_out` = rank 0's arrays (capacity cap_*_all, cut into `world` regions), None elsewhere; every rank
    passes the same capacities. Returns the local rows, the regions [(runs offset, runs, juncs offset, juncs)] and, on rank 0,
    the gathered rows per region."""
    keep = []
    arr = (_lib.CovIn * len(segs))(*[_cov_in(s, keep) for s in segs])
    runs, juncs = _out_structs(out)
    if all_out is not None:
        ar, aj = _out_structs(all_out)
        ar.capacity, aj.capacity = int(cap_runs_all), int(cap_juncs_all)
    else:
        ar = _lib.RunsOut(int(cap_runs_all), 0, None, None, None, None, 1)
        aj = _lib.JuncsOut(int(cap_juncs_all), 0, None, None, None, None, None, 1)
    region = (C.c_int64 * (4 * world))()
    rc = self.lib.tc_shard_coverage_gather(self.h, arr, len(segs), int(window), C.byref(runs), C.byref(juncs), C.byref(ar), C.byref(aj), region)
    if rc == 2:
        raise ValueError(self._err())
    if rc != 0:
        raise TieBrushError(self._err())
    res = _rows(out, int(runs.n_runs), int(juncs.n_juncs))
    res["windows"] = int(self.lib.tc_stream_windows(self.h))
    res["stats"] = dict(zip(("lead_received", "lead_sent", "ranks_received_from", "halo_bytes_sent", "seam_records", "gather_bytes", "gather_rounds"),
                            (int(self.lib.tc_shard_stat(self.h, i)) for i in range(7))))
    res["regions"] = [tuple(int(region[4 * r + q]) for q in range(4)) for r in range(world)]
    res["total_runs"] = sum(x[1] for x in res["regions"]); res["total_juncs"] = sum(x[3] for x in res["regions"])
    if all_out is not None:
        cat = lambda keys, oi, ci: tuple((torch_cat if _is_torch(all_out[keys[0]]) else np.concatenate)([all_out[kk][x[oi]:x[oi] + x[ci]] for x in res["regions"]]) for kk in keys)
        import functools
        try:
            import torch
            torch_cat = torch.cat
        except Exception:   # pragma: no cover
            torch_cat = None
        res["gathered_runs"] = lambda: cat(("r_tid", "r_start", "r_end", "r_val"), 0, 1)
        res["gathered_juncs"] = lambda: cat(("j_tid", "j_start", "j_end", "j_strand", "j_val"), 2, 3)
    return res


Context.coverage_stream = _coverage_stream
Context.shard_coverage_gather = _shard_coverage_gather
Context.comm_init = _comm_init
Context.shard_coverage = _shard_coverage
Context.shard_gather = _shard_gather
Context.last_cov_exact = lambda self: int(self.lib.tc_last_exact(self.h))
comm_unique_id = _comm_unique_id
