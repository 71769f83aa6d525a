"""CPU checks of the test-only BAM writer (tests/bam_writer.py) and of api.read_bam_header: in every block layout and
DEFLATE variant the files decode with zlib (helpers.bam_sam_text) into the records that were written, and the header
reader finds where the records start."""
import zlib

import numpy as np
import pytest

import bam_writer as W
import helpers as H

LAYOUTS = ["htslib", "fixed1000", "long", "empty_noeof"]


def synthetic_file(layout, variant, seed=3, n=400):
    """(BAM bytes, record bytes, header text, (flag, tid, pos, CIGAR words, tags) per record) of a small seeded stream on two references with unmapped records,
    tags of every aux type around the ones tiecov reads, and for `long` a record larger than a block."""
    rng = np.random.default_rng(seed)
    text = "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:c0\tLN:1000000\n@SQ\tSN:c1\tLN:2000000\n@CO\tSAMPLE:a\n"
    names = ["c0", "c1"]
    recs, meta = [], []
    tid, pos = 0, 100
    for i in range(n):
        if i == n // 2:
            tid, pos = 1, 50
        pos += int(rng.integers(0, 60))
        unm = rng.random() < 0.1
        flag = 4 if unm else int(rng.choice([0, 16]))
        m1 = int(rng.integers(10, 60))
        cig = [(m1 << 4) | 0] + ([(int(rng.integers(50, 3000)) << 4) | 3, (int(rng.integers(10, 60)) << 4) | 0] if rng.random() < 0.5 else [])
        tags = [("RG", "Z", "grp%d" % (i % 3)), ("XB", "B", ("s", [1, -2, 3]))]
        k = i % 9
        yct = "fdcCsSiI"[k] if k < 8 else None
        if yct:
            v = {"f": 2.5, "d": 3.25, "c": -2, "C": 200, "s": -300, "S": 60000, "i": 70000, "I": 3000000000}[yct]
            tags.append(("YC", yct, v))
        if i % 4:
            tags.append(("YX", "cCsSiI"[i % 6], int(rng.integers(1, 100))))
        xs = i % 7
        if xs == 0:
            tags.append(("XS", "A", "+-"[i % 2]))
        elif xs == 1:
            tags.append(("XS", "Z", "-"))
        elif xs == 2:
            tags.append(("XS", "A", "x"))
        elif xs == 3:
            tags.append(("ts", "A", "+-"[(i // 7) % 2]))
        tags.append(("ZZ", "H", "1AE3"))
        seq = "ACGT" * 10
        if layout == "long" and i == n // 3:
            seq = "ACGT" * 20000
            tags.append(("BB", "B", ("I", list(range(5000)))))
        r = W.record_bytes(tid if not unm else (tid if i % 2 else -1), pos if not unm else (pos if i % 2 else -1), flag, cig if not unm else [],
                           tags, qname=f"r{i}", seq=seq, qual=bytes([20] * len(seq)))
        recs.append(r)
        meta.append((flag, tid, pos, cig, tags))
    hdr = W.header_bytes(text, names, [1000000, 2000000])
    if layout == "fixed1000":
        pl = W.blocks(hdr, recs, "fixed", cut=1000)
    else:
        pl = W.blocks(hdr, recs)
    data = W.bgzf_file(pl, variant, empty_every=3 if layout == "empty_noeof" else 0, eof=layout != "empty_noeof")
    return data, recs, text, meta


@pytest.mark.parametrize("variant", list(W.VARIANTS))
@pytest.mark.parametrize("layout", LAYOUTS)
def test_writer_files_decode_into_the_written_records(tmp_path, layout, variant):
    from tiebrush_b200 import api
    data, recs, text, _ = synthetic_file(layout, variant)
    p = tmp_path / "x.bam"
    p.write_bytes(data)
    assert _inflate_from(data, 0) == W.header_bytes(text, ["c0", "c1"], [1000000, 2000000]) + b"".join(recs)
    body = [ln.split("\t") for ln in H.bam_sam_text(str(p)).split("\n") if ln and ln[0] != "@"]
    assert [f[0] for f in body] == [f"r{i}" for i in range(len(recs))]
    ids = {"c0": 0, "c1": 1}
    for f, r in zip(body, recs):   # integer tags come back as type i: compare the fixed part and the CIGAR / SEQ / QUAL
        b = W.record_from_sam(f, ids)
        assert b[4:36] == r[4:36] and f[5] != "" and b[36:36 + 40] == r[36:36 + 40]
    h = api.read_bam_header(str(p))
    assert h["names"] == ["c0", "c1"] and h["lengths"] == [1000000, 2000000] and h["n_samples"] == 1 and h["text"] == text
    # the records start where the header reader says: inflate from that block, drop `skip` bytes
    raw = _inflate_from(data, h["block_offset"])
    assert raw[h["skip"]:] == b"".join(recs)
    if layout != "fixed1000":
        assert h["skip"] == 0


def _inflate_from(data, off):
    out, o = bytearray(), off
    while o < len(data):
        bsize = int.from_bytes(data[o + 16:o + 18], "little")
        out += zlib.decompress(data[o + 18:o + bsize + 1 - 8], -15)
        o += bsize + 1
    return bytes(out)


def test_columns_records_equal_the_scalar_encoder():
    from tiebrush_b200 import synth
    cols = synth.to_host(synth.coverage_stream(500, seed=2, n_tx=10, chroms=2))
    cols["yx"] = np.arange(500, dtype=np.int32) % 7 + 1
    buf, ends = W.columns_records(cols, l_seq=150)
    starts = np.concatenate([[0], ends[:-1]])
    off = cols["cig_off"]
    for i in (0, 1, 250, 499):
        r = W.record_bytes(int(cols["tid"][i]), int(cols["pos"][i]), 0, list(cols["cigar"][off[i]:off[i + 1]]),
                           [("NH", "C", 1), ("XS", "A", chr(cols["strand"][i])), ("YC", "f", float(cols["yc"][i])), ("YX", "i", int(cols["yx"][i]))],
                           qname="q%08d" % i, seq="AC" * 75, qual=bytes([30] * 150))
        assert bytes(buf[starts[i]:ends[i]]) == r
    pl = W.columns_payloads(b"hdr", buf, ends)
    assert b"".join(pl[1:]) == bytes(buf) and all(len(x) <= W.HTS_BLOCK for x in pl)
