"""Shared test plumbing: golden-case loading and window-by-window drivers for either implementation."""
from __future__ import annotations

import os
import numpy as np

from tiebrush_b200 import sam

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
OPT_NAMES = ("mode", "flag_mask", "max_nh", "min_qual", "keep_bits", "collapse_same")
_cache = {}


def _npz(name):
    if name not in _cache:
        _cache[name] = np.load(os.path.join(GOLDEN, name), allow_pickle=False)
    return _cache[name]


def case_names(npz_name):
    z = _npz(npz_name)
    return sorted({k.split("/")[1] for k in z.files if k.startswith("case/")})


def _input_files(z, inkey, with_tags):
    pre = f"in/{inkey}/"
    cols = {k[len(pre):]: z[k] for k in z.files if k.startswith(pre)}
    foff = cols.pop("file_off")
    n = len(cols["pos"])
    for k in ("yc_in", "yx_in", "yd_in"):
        if k not in cols:
            cols[k] = np.zeros(n, np.float32 if k == "yc_in" else np.int32)
    cols["has_yc"] = np.zeros(n, np.bool_)
    return [sam.take(cols, np.arange(foff[i], foff[i + 1])) for i in range(len(foff) - 1)]


def load_collapse_case(npz_name, case):
    z = _npz(npz_name)
    pre = f"case/{case}/"
    inkey = str(z[pre + "inkey"][0])
    files = _input_files(z, inkey, True)
    files = [files[i] for i in z[pre + "files"]]
    opts = dict(zip(OPT_NAMES, (int(v) for v in z[pre + "opts"])))
    fm = z[pre + "file_merged"] if (pre + "file_merged") in z.files else None
    exp = dict(tid=z[pre + "out/tid"], lhash=z[pre + "out/lhash"], yc=z[pre + "out/yc"], yx=z[pre + "out/yx"],
               yd=z[pre + "out/yd"], n_kept=int(z[pre + "out/n_kept"][0]))
    return files, opts, fm, exp


def run_collapse(collapse_fn, files, opts, file_merged=None):
    """Drive `collapse_fn(cols, run_off, tid=, file_merged=, **opts)` over one window per reference id."""
    o_tid, o_lh, o_yc, o_yx, o_yd, kept = [], [], [], [], [], 0
    for tid, cols, run_off, _src in sam.split_windows_by_tid(files):
        r = collapse_fn(cols, run_off, tid=tid, file_merged=file_merged, **opts)
        g = len(r["rep_index"])
        o_tid.append(np.full(g, tid, np.int32))
        o_lh.append(cols["lhash"][r["rep_index"].astype(np.int64)])
        o_yc.append(r["yc"]); o_yx.append(r["yx"]); o_yd.append(r["yd"])
        kept += r["n_kept"]
    cat = lambda xs, dt: np.concatenate(xs) if xs else np.zeros(0, dt)
    return dict(tid=cat(o_tid, np.int32), lhash=cat(o_lh, np.uint64), yc=cat(o_yc, np.float32),
                yx=cat(o_yx, np.uint32), yd=cat(o_yd, np.int32), n_kept=kept)


def assert_collapse_equal(got, exp, what=""):
    assert got["n_kept"] == exp["n_kept"], f"{what}: n_kept {got['n_kept']} != {exp['n_kept']}"
    assert len(got["lhash"]) == len(exp["lhash"]), f"{what}: groups {len(got['lhash'])} != {len(exp['lhash'])}"
    for k in ("tid", "lhash", "yx", "yd"):
        bad = np.nonzero(got[k].astype(np.int64) != exp[k].astype(np.int64))[0] if k != "lhash" else np.nonzero(got[k] != exp[k])[0]
        assert len(bad) == 0, f"{what}: {k} differs at {bad[:5]} got {got[k][bad[:5]]} exp {exp[k][bad[:5]]}"
    # the golden YC went through htslib's SAM text ("%g", 6 significant digits): integers are exact, fractional values
    # (--store-frac) are compared after the same rendering
    gyc = np.asarray([np.float32(float("%g" % v)) for v in got["yc"]], np.float32) if len(got["yc"]) else np.zeros(0, np.float32)
    bad = np.nonzero(gyc.view(np.uint32) != exp["yc"].astype(np.float32).view(np.uint32))[0]
    assert len(bad) == 0, f"{what}: yc differs at {bad[:5]} got {got['yc'][bad[:5]]} exp {exp['yc'][bad[:5]]}"


_AUX_INT = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I"}
_SEQ2 = [a + b for a in "=ACMGRSVTWYHKDBN" for b in "=ACMGRSVTWYHKDBN"]   # one byte of BAM SEQ = two bases
_QUAL33 = bytes((q + 33) & 0xFF for q in range(256))


def bam_sam_text(path):
    """A BAM file as the SAM text htslib prints for it (`htsfile -c`): header, then one line per record. BGZF is a series of
    gzip members, so the gzip module reads it; the record layout is the one of the SAM/BAM specification, section 4.2."""
    import gzip
    import struct
    b = gzip.open(path, "rb").read()
    assert b[:4] == b"BAM\1", f"{path}: not a BAM file"
    l_text = struct.unpack_from("<i", b, 4)[0]
    lines = [b[8:8 + l_text].rstrip(b"\0").decode().rstrip("\n")]
    o = 8 + l_text
    n_ref = struct.unpack_from("<i", b, o)[0]
    o += 4
    names = []
    for _ in range(n_ref):
        ln = struct.unpack_from("<i", b, o)[0]
        names.append(b[o + 4:o + 3 + ln].decode())
        o += 8 + ln
    while o < len(b):
        bs, tid, pos, l_qn, mapq, _bin, n_cig, flag, l_seq, ntid, npos, tlen = struct.unpack_from("<iiiBBHHHiiii", b, o)
        end, o = o + 4 + bs, o + 36
        qname = b[o:o + l_qn - 1].decode()
        o += l_qn
        cig = sam.cigar_str(struct.unpack_from(f"<{n_cig}I", b, o))
        o += 4 * n_cig
        seq = "".join([_SEQ2[x] for x in b[o:o + (l_seq + 1) // 2]])[:l_seq] if l_seq else "*"
        o += (l_seq + 1) // 2
        qual = "*" if (l_seq == 0 or b[o] == 0xFF) else b[o:o + l_seq].translate(_QUAL33).decode("latin-1")
        o += l_seq
        f = [qname, str(flag), names[tid] if tid >= 0 else "*", str(pos + 1), str(mapq), cig,
             "*" if ntid < 0 else ("=" if ntid == tid else names[ntid]), str(npos + 1), str(tlen), seq, qual]
        while o < end:
            tag, t = b[o:o + 2].decode(), chr(b[o + 2])
            o += 3
            if t == "A":
                f.append(f"{tag}:A:{chr(b[o])}"); o += 1
            elif t in _AUX_INT:
                v = struct.unpack_from(_AUX_INT[t], b, o)[0]
                f.append(f"{tag}:i:{v}"); o += struct.calcsize(_AUX_INT[t])
            elif t == "f":
                f.append(f"{tag}:f:{struct.unpack_from('<f', b, o)[0]:g}"); o += 4
            elif t == "d":
                f.append(f"{tag}:d:{struct.unpack_from('<d', b, o)[0]:g}"); o += 8
            elif t in "ZH":
                z = b.index(b"\0", o)
                f.append(f"{tag}:{t}:{b[o:z].decode()}"); o = z + 1
            elif t == "B":
                st, cnt = chr(b[o]), struct.unpack_from("<i", b, o + 1)[0]
                fmt = "<f" if st == "f" else _AUX_INT[st]
                w = struct.calcsize(fmt)
                vals = [struct.unpack_from(fmt, b, o + 5 + w * k)[0] for k in range(cnt)]
                f.append(f"{tag}:B:{st}" + "".join(f",{v:g}" if st == "f" else f",{v}" for v in vals)); o += 5 + w * cnt
            else:
                raise ValueError(f"{path}: aux type {t!r}")
        lines.append("\t".join(f))
    return "\n".join(lines) + "\n"


# The reference's own test data (test/t1/t1s[0-9].bam, test/t2/t2s[0-9].bam) and what the compiled, unmodified reference
# makes of it: md5 of the record text of `tiebrush -o o.bam <files>` (`htsfile -c o.bam | grep -v '^@' | md5sum`), of the
# bedGraph and junction BED of `tiecov -c -j` on the t1+t2 output, and the counts of its summary line.
FIXTURES = os.path.join(GOLDEN, "fixtures")
REF_MD5 = {"t1": "db674977026be7f2832fe9869ed40376", "t2": "27f7b93a789a9cddb06dca63449d32af", "t12": "50320443e9d380da6bc6c46b1fa90d85",
           "cov": "8d1b0c70113a233095742cec61bb8129", "junc": "61427ff301f9ea70d48d5fbff20db7e2"}
REF_COUNTS = {"t1": (416922, 3479), "t2": (242910, 8179), "t12": (659832, 9491)}   # (input records kept, records written)


def fixture_inputs(which):
    """The sample BAMs of the fixture sets `which` (e.g. ["t1", "t2"]): (per-file columns, SAM header lines, input line by
    line hash). Decoded once per process."""
    key = ("fixtures",) + tuple(which)
    if key not in _cache:
        paths = [os.path.join(FIXTURES, t, f"{t}s{i}.bam") for t in which for i in range(10)]
        for p in paths:
            if p not in _cache:
                _cache[p] = bam_sam_text(p)
        texts = [_cache[p] for p in paths]
        header = [ln for ln in texts[0].split("\n") if ln.startswith("@")]
        ids = sam.parse_sam("\n".join(header))[1]
        files = [sam.to_columns(sam.parse_sam(t, ids)[0]) for t in texts]
        lines = {}
        for t in texts:
            for ln in t.split("\n"):
                if ln and ln[0] != "@":
                    lines.setdefault(sam.line_hash(ln.split("\t")), ln)
        _cache[key] = (files, header, lines)
    return _cache[key]


def collapsed_records(got, lines):
    """The SAM record lines tiebrush writes for the groups of run_collapse(): the representative's line with YC (float),
    YX and, when non-zero, YD appended, as htslib prints them."""
    return ["\t".join([lines[int(lh)], f"YC:f:{float(yc):g}", f"YX:i:{int(yx)}"] + ([f"YD:i:{int(yd)}"] if int(yd) > 0 else []))
            for lh, yc, yx, yd in zip(got["lhash"], got["yc"], got["yx"], got["yd"])]


def md5_text(lines):
    import hashlib
    return hashlib.md5(("\n".join(lines) + "\n").encode()).hexdigest()


def coverage_input(header, records):
    """tiecov's view of a collapsed file: columns of its mapped records, weight YC (1 where the tag is absent)."""
    R, ids = sam.parse_sam("\n".join(header + records) + "\n")
    cols = sam.to_columns(R)
    keep = np.nonzero((cols["flag"] & 4) == 0)[0]
    sub = sam.take(cols, keep)
    sub["yc"] = np.where(cols["has_yc"], cols["yc_in"], np.float32(1)).astype(np.float32)[keep]
    return sub, {v: k for k, v in ids.items()}


def coverage_files(got, names):
    """The bytes of tiecov's -c bedGraph and -j junction BED for coverage rows `got` (the formats of tiecov.cpp)."""
    bg = "track type=bedGraph\n" + "".join(f"{names[int(t)]}\t{int(s)}\t{int(e)}\t{float(v):.3f}\n" for t, s, e, v in zip(*got["runs"]))
    bed = "track name=junctions\n" + "".join(f"{names[int(t)]}\t{int(s) - 1}\t{int(e)}\tJUNC{i + 1:08d}\t{float(v):.3f}\t{chr(int(c))}\n"
                                             for i, (t, s, e, c, v) in enumerate(zip(*got["juncs"])))
    return bg, bed


def load_coverage_case(case):
    z = _npz("coverage.npz")
    pre = f"{case}/"
    cols = {k[len(pre) + 3:]: z[k] for k in z.files if k.startswith(pre + "in/")}
    keep = (cols["flag"] & 4) == 0  # tiecov.cpp:436-438
    n = len(cols["pos"])
    full = dict(cols)
    for k in sam.PER_RECORD:
        if k not in full:
            full[k] = np.zeros(n, np.int32)
    sub = sam.take({**full, "md_off": np.zeros(n + 1, np.uint32), "md": np.zeros(0, np.uint8)}, np.nonzero(keep)[0])
    sub["yc"] = cols["yc"][keep]
    runs = tuple(z[pre + "runs/" + k] for k in ("tid", "start0", "end0", "milli"))
    juncs = tuple(z[pre + "juncs/" + k] for k in ("tid", "start0", "end", "num", "milli", "strand"))
    return sub, runs, juncs


def coverage_case_names():
    z = _npz("coverage.npz")
    return sorted({k.split("/")[0] for k in z.files})


def milli(v):
    """'%.3f' rendering of a double as integer thousandths (exact for the integer-valued sums used here)."""
    return np.asarray([int(round(float(f"{x:.3f}") * 1000)) for x in v], np.int64)


def assert_coverage_equal(got, runs, juncs, what=""):
    gt, gs, ge, gv = got["runs"]
    assert len(gt) == len(runs[0]), f"{what}: runs {len(gt)} != {len(runs[0])}"
    assert (gt == runs[0]).all() and (gs == runs[1]).all() and (ge == runs[2]).all(), f"{what}: run coords differ"
    assert (milli(gv) == runs[3]).all(), f"{what}: run values differ"
    jt, js, je, jc, jv = got["juncs"]
    assert len(jt) == len(juncs[0]), f"{what}: juncs {len(jt)} != {len(juncs[0])}"
    assert (jt == juncs[0]).all() and (js - 1 == juncs[1]).all() and (je == juncs[2]).all(), f"{what}: junc coords differ"
    assert (np.arange(1, len(jt) + 1) == juncs[3]).all()
    assert (milli(jv) == juncs[4]).all() and (jc == juncs[5]).all(), f"{what}: junc values/strands differ"
