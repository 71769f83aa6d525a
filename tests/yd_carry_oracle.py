"""TEST INFRASTRUCTURE ONLY — ctypes binding of tests/yd_carry_oracle.c: the oracle's collapse with the YD segment lists
seeded from a carry and the lists left behind exported (tbo_collapse_carry). The shared library is compiled on first use
into a temporary directory, so the tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle.oracle import _In, _Opts, _Out, _c, _p

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "yd_carry_oracle.c"), os.path.join(ROOT, "oracle", "tb_oracle.c"), os.path.join(ROOT, "include", "tiebrush_b200.h")]


class Carry(C.Structure):
    _fields_ = [("tid", C.c_int32), ("pos_hi", C.c_int32), ("n_chains", C.c_int32), ("capacity", C.c_int64), ("n_segs", C.c_int64),
                ("chain_off", C.c_void_p), ("seg_start", C.c_void_p), ("seg_end", C.c_void_p)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha1(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"tb_yd_carry_oracle_{os.getuid()}_{h}.so")
        if not os.path.exists(path):
            tmp = path + f".{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-Wall", "-o", tmp, SOURCES[0], "-lm"])
            os.replace(tmp, path)
        _lib = C.CDLL(path)
        _lib.tbo_collapse_carry.restype = C.c_int
    return _lib


def empty_carry(n_samples):
    """A YD carry with no lists (what the first window of a stream starts from)."""
    return dict(tid=-1, pos_hi=0, chain_off=np.zeros(2 * n_samples + 1, np.int64), seg_start=np.zeros(0, np.int32), seg_end=np.zeros(0, np.int32))


def collapse(cols: dict, run_off, yd_carry, pos_range=None, tid=0, mode=0, flag_mask=0, max_nh=0x7FFFFFFF, min_qual=-1, keep_bits=0,
             collapse_same=0, file_merged=None):
    """Oracle collapse of one window whose YD lists start from `yd_carry` (a dict like empty_carry() or the yd_carry of an
    earlier result). `pos_range` = the window's (pos_lo, pos_hi), default (min pos, max pos + 1). Returns dict(rep_index, yc,
    yx, yd, n_kept, yd_carry) like oracle.oracle.collapse plus the lists this window leaves behind."""
    n = len(cols["pos"])
    run_off = _c(run_off, np.int64)
    k = len(run_off) - 1
    a = dict(pos=_c(cols["pos"], np.int32), flag=_c(cols["flag"], np.uint16), mapq=_c(cols["mapq"], np.uint8),
             strand=_c(cols["strand"], np.uint8), nh=_c(cols["nh"], np.uint16), cig_off=_c(cols["cig_off"], np.uint32),
             cigar=_c(cols["cigar"], np.uint32))
    md_off = _c(cols["md_off"], np.uint32) if "md_off" in cols else np.zeros(n + 1, np.uint32)
    md = _c(cols["md"], np.uint8) if "md" in cols else np.zeros(0, np.uint8)
    qh = _c(cols["qhash"], np.uint64) if "qhash" in cols else None
    fm = _c(file_merged, np.uint8) if file_merged is not None else None
    yc_in = _c(cols["yc_in"], np.float32) if (fm is not None and "yc_in" in cols) else None
    yx_in = _c(cols["yx_in"], np.int32) if (fm is not None and "yx_in" in cols) else None
    yd_in = _c(cols["yd_in"], np.int32) if (fm is not None and "yd_in" in cols) else None
    if pos_range is None:
        pos_range = (int(a["pos"].min()), int(a["pos"].max()) + 1) if n else (0, 1)
    sin = _In(n, k, tid, _p(run_off), _p(fm), _p(a["pos"]), _p(a["flag"]), _p(a["mapq"]), _p(a["strand"]), _p(a["nh"]),
              _p(a["cig_off"]), _p(a["cigar"]), _p(md_off), _p(md), _p(qh), _p(yc_in), _p(yx_in), _p(yd_in), 0,
              int(a["cig_off"][-1]) if n else 0, int(md_off[-1]) if n else 0, int(pos_range[0]), int(pos_range[1]))
    cap = max(n, 1)
    rep = np.zeros(cap, np.uint32); yc = np.zeros(cap, np.float32); yx = np.zeros(cap, np.uint32); yd = np.zeros(cap, np.int32)
    out = _Out(cap, 0, 0, _p(rep), _p(yc), _p(yx), _p(yd), 0)
    o = _Opts(mode, flag_mask, max_nh, min_qual, keep_bits, collapse_same)
    ci = {key: _c(yd_carry[key], dt) for key, dt in (("chain_off", np.int64), ("seg_start", np.int32), ("seg_end", np.int32))}
    cin = Carry(int(yd_carry["tid"]), int(yd_carry["pos_hi"]), len(ci["chain_off"]) - 1, len(ci["seg_start"]), int(ci["chain_off"][-1]),
                _p(ci["chain_off"]), _p(ci["seg_start"]), _p(ci["seg_end"]))
    ccap = 64
    while True:
        co = dict(chain_off=np.zeros(2 * k + 1, np.int64), seg_start=np.zeros(ccap, np.int32), seg_end=np.zeros(ccap, np.int32))
        cout = Carry(0, 0, 2 * k, ccap, 0, _p(co["chain_off"]), _p(co["seg_start"]), _p(co["seg_end"]))
        rc = lib().tbo_collapse_carry(C.byref(sin), C.byref(o), C.byref(cin), C.byref(out), C.byref(cout))
        if rc != 2:
            break
        ccap = int(cout.n_segs)
    if rc != 0:
        raise RuntimeError(f"tbo_collapse_carry rc={rc}")
    m, g = int(cout.n_segs), out.n_groups
    return dict(rep_index=rep[:g].copy(), yc=yc[:g].copy(), yx=yx[:g].copy(), yd=yd[:g].copy(), n_kept=int(out.n_kept),
                yd_carry=dict(tid=int(cout.tid), pos_hi=int(cout.pos_hi), chain_off=co["chain_off"], seg_start=co["seg_start"][:m].copy(),
                              seg_end=co["seg_end"][:m].copy()))
