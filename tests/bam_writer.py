"""Test-only BGZF + BAM writer (SAM spec §4.1-4.2): the files the device decoder is checked on, in every block layout and
DEFLATE variant a writer may produce. Nothing here is used by the library."""
from __future__ import annotations

import struct
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

HTS_BLOCK = 0xff00                     # htslib's BGZF_BLOCK_SIZE: the inflated bytes one block holds at most
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
VARIANTS = {"stored": (0, zlib.Z_DEFAULT_STRATEGY), "l1": (1, zlib.Z_DEFAULT_STRATEGY), "l6": (6, zlib.Z_DEFAULT_STRATEGY),
            "l9": (9, zlib.Z_DEFAULT_STRATEGY), "fixed": (6, zlib.Z_FIXED), "huffman": (6, zlib.Z_HUFFMAN_ONLY), "rle": (6, zlib.Z_RLE)}
_INT = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I"}
_CIG = {c: i for i, c in enumerate("MIDNSHP=X")}
_NT = {c: i for i, c in enumerate("=ACMGRSVTWYHKDBN")}


def bgzf_block(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    """One BGZF block (a gzip member with the BC subfield) holding `data` (at most 64 KiB)."""
    assert len(data) <= 65536
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    body = co.compress(data) + co.flush()
    bsize = 12 + 6 + len(body) + 8 - 1
    assert bsize < 65536, "block does not compress into 64 KiB"
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", bsize) + body
            + struct.pack("<II", zlib.crc32(data) & 0xffffffff, len(data)))


def header_bytes(text, names, lengths):
    t = text.encode()
    out = [b"BAM\1", struct.pack("<i", len(t)), t, struct.pack("<i", len(names))]
    for nm, ln in zip(names, lengths):
        out += [struct.pack("<i", len(nm) + 1), nm.encode() + b"\0", struct.pack("<i", ln)]
    return b"".join(out)


def tag_bytes(tag, typ, val):
    """One aux field: A / c C s S i I / f / d / Z / H, or B as (subtype, list)."""
    t = tag.encode() + typ.encode()
    if typ == "A":
        return t + val.encode()
    if typ in _INT:
        return t + struct.pack(_INT[typ], val)
    if typ == "f":
        return t + struct.pack("<f", val)
    if typ == "d":
        return t + struct.pack("<d", val)
    if typ in "ZH":
        return t + val.encode() + b"\0"
    sub, vals = val
    return t + sub.encode() + struct.pack("<i", len(vals)) + b"".join(struct.pack("<f" if sub == "f" else _INT[sub], v) for v in vals)


def record_bytes(tid, pos, flag, cigar, tags=(), qname="r", mapq=60, seq=None, qual=None, l_seq=0):
    """One BAM record. cigar: packed words (len << 4 | op); seq: a base string (else l_seq bases of N); tags: (tag, type, value)."""
    if seq is None:
        seq = "N" * l_seq
    l_seq = len(seq)
    sb = bytearray((l_seq + 1) // 2)
    for i, c in enumerate(seq):
        sb[i >> 1] |= _NT[c] << (4 if i % 2 == 0 else 0)
    qb = bytes(qual) if qual is not None else b"\xff" * l_seq
    qn = qname.encode() + b"\0"
    body = struct.pack("<iiBBHHHiiii", tid, pos, len(qn), mapq, 4680, len(cigar), flag, l_seq, -1, -1, 0) + qn \
        + struct.pack(f"<{len(cigar)}I", *cigar) + bytes(sb) + qb + b"".join(tag_bytes(*t) for t in tags)
    return struct.pack("<i", len(body)) + body


def record_from_sam(fields, ids):
    """A SAM text line (split on tabs) as BAM record bytes."""
    cig = []
    if fields[5] != "*":
        num = ""
        for c in fields[5]:
            if c.isdigit():
                num += c
            else:
                cig.append(int(num) << 4 | _CIG[c]); num = ""
    tags = []
    for t in fields[11:]:
        tag, typ, v = t[:2], t[3], t[5:]
        if typ == "i":
            x = int(v)
            tags.append((tag, "i" if -2**31 <= x < 2**31 else "I", x))
        elif typ in "fd":
            tags.append((tag, typ, float(v)))
        elif typ == "B":
            p = v.split(",")
            tags.append((tag, "B", (p[0], [float(x) if p[0] == "f" else int(x) for x in p[1:]])))
        else:
            tags.append((tag, typ, v))
    seq = None if fields[9] == "*" else fields[9]
    qual = None if fields[10] == "*" else bytes(ord(c) - 33 for c in fields[10])
    tid = ids[fields[2]] if fields[2] != "*" else -1
    rec = record_bytes(tid, int(fields[3]) - 1, int(fields[1]), cig, tags, qname=fields[0], mapq=int(fields[4]), seq=seq, qual=qual)
    nxt = tid if fields[6] == "=" else (ids[fields[6]] if fields[6] != "*" else -1)
    return rec[:24] + struct.pack("<iii", nxt, int(fields[7]) - 1, int(fields[8])) + rec[36:]


def blocks(header, records, layout="htslib", cut=None):
    """The inflated payloads of the blocks of a file. htslib: the header flushed on its own, then a new block whenever the
    next record would not fit in HTS_BLOCK bytes (records larger than that span blocks); fixed: every `cut` bytes of the whole
    stream (the header and records span blocks)."""
    if layout == "fixed":
        s = header + b"".join(records)
        return [s[i:i + cut] for i in range(0, len(s), cut)]
    out = [header[i:i + HTS_BLOCK] for i in range(0, len(header), HTS_BLOCK)]
    cur = bytearray()
    for r in records:
        if cur and len(cur) + len(r) > HTS_BLOCK:
            out.append(bytes(cur)); cur = bytearray()
        cur += r
        while len(cur) > HTS_BLOCK:
            out.append(bytes(cur[:HTS_BLOCK])); cur = cur[HTS_BLOCK:]
    if cur:
        out.append(bytes(cur))
    return out


def bgzf_file(payloads, variant="l6", empty_every=0, eof=True, threads=8):
    """BGZF bytes of the payloads: one block each (compressed on `threads` threads: zlib releases the GIL), an empty block
    after every `empty_every` of them when non-zero, the 28-byte EOF marker when `eof`."""
    level, strategy = VARIANTS[variant]
    with ThreadPoolExecutor(threads) as ex:
        bl = list(ex.map(lambda d: bgzf_block(d, level, strategy), payloads))
    if empty_every:
        bl = [b for i, x in enumerate(bl) for b in ([x, bgzf_block(b"", level, strategy)] if (i + 1) % empty_every == 0 else [x])]
    return b"".join(bl) + (EOF_BLOCK if eof else b"")


def columns_records(cols, l_seq=0):
    """Records of coverage columns (tid, pos, cig_off, cigar; optional flag / yc / yx / strand), numpy-vectorised for files
    of millions of records. Every record has the qname "q<8 digits>", l_seq (even) bases of SEQ and QUAL and the tags NH:C:1,
    XS:A:<strand>, YC:f and YX:i. Returns (flat record bytes, record ends)."""
    n = len(cols["pos"])
    off = np.asarray(cols["cig_off"], np.int64)
    ncig = off[1:] - off[:-1]
    fixed = 36 + 10 + (l_seq + 1) // 2 + l_seq
    aux = 4 + 4 + 7 + 7                    # NH:C, XS:A, YC:f, YX:i
    size = fixed + 4 * ncig + aux
    ends = np.cumsum(size)
    starts = ends - size
    buf = np.zeros(int(ends[-1]) if n else 0, np.uint8)

    def put(rel, arr, dtype):
        b = np.ascontiguousarray(arr, dtype).view(np.uint8).reshape(n, -1)
        idx = starts[:, None] + rel + np.arange(b.shape[1])[None, :]
        buf[idx] = b

    put(0, size - 4, "<i4")
    put(4, cols["tid"], "<i4"); put(8, cols["pos"], "<i4")
    put(12, np.full(n, 10, np.uint8), "u1"); put(13, np.full(n, 60, np.uint8), "u1"); put(14, np.full(n, 4680, np.uint16), "<u2")
    put(16, ncig, "<u2"); put(18, np.asarray(cols.get("flag", np.zeros(n)), np.uint16), "<u2"); put(20, np.full(n, l_seq, np.int32), "<i4")
    put(24, np.full(n, -1, np.int32), "<i4"); put(28, np.full(n, -1, np.int32), "<i4"); put(32, np.zeros(n, np.int32), "<i4")
    digits = (np.arange(n, dtype=np.int64)[:, None] // (10 ** np.arange(7, -1, -1))[None, :]) % 10
    q = np.concatenate([np.full((n, 1), ord("q")), digits + ord("0"), np.zeros((n, 1))], 1).astype(np.uint8)
    buf[starts[:, None] + 36 + np.arange(10)[None, :]] = q
    # CIGAR words: word w of record r at starts[r] + 46 + 4 * (w - off[r])
    rec_of = np.repeat(np.arange(n), ncig)
    wpos = starts[rec_of] + 46 + 4 * (np.arange(int(off[-1] - off[0])) - (off[:-1][rec_of] - off[0]))
    cw = np.asarray(cols["cigar"], np.uint32)[int(off[0]):int(off[-1])].view(np.uint8).reshape(-1, 4)
    buf[wpos[:, None] + np.arange(4)[None, :]] = cw
    sq = starts + 46 + 4 * ncig
    if l_seq:
        buf[sq[:, None] + np.arange((l_seq + 1) // 2)[None, :]] = 0x12        # "AC" pairs
        buf[(sq + (l_seq + 1) // 2)[:, None] + np.arange(l_seq)[None, :]] = 30
    a = sq + (l_seq + 1) // 2 + l_seq
    strand = np.asarray(cols.get("strand", np.full(n, ord("."), np.uint8)), np.uint8)
    yc = np.asarray(cols.get("yc", np.ones(n, np.float32)), np.float32)
    yx = np.asarray(cols.get("yx", np.ones(n, np.int32)), np.int32)
    for k, v in enumerate(b"NHC"):
        buf[a + k] = v
    buf[a + 3] = 1
    for k, v in enumerate(b"XSA"):
        buf[a + 4 + k] = v
    buf[a + 7] = strand
    for k, v in enumerate(b"YCf"):
        buf[a + 8 + k] = v
    b4 = yc.view(np.uint8).reshape(n, 4)
    buf[(a + 11)[:, None] + np.arange(4)[None, :]] = b4
    for k, v in enumerate(b"YXi"):
        buf[a + 15 + k] = v
    buf[(a + 18)[:, None] + np.arange(4)[None, :]] = yx.view(np.uint8).reshape(n, 4)
    return buf, ends


def columns_payloads(header, buf, ends):
    """htslib-style block payloads of a flat record buffer (record ends `ends`): a new block whenever the next record would
    not fit in HTS_BLOCK bytes."""
    out = [header[i:i + HTS_BLOCK] for i in range(0, len(header), HTS_BLOCK)]
    s, n = 0, len(ends)
    mv = memoryview(buf)
    while s < len(buf):
        k = int(np.searchsorted(ends, s + HTS_BLOCK, side="right"))   # records ending within the block
        e = int(ends[k - 1]) if k > 0 and ends[k - 1] > s else min(s + HTS_BLOCK, len(buf))
        out.append(bytes(mv[s:e]))
        s = e
    return out
