"""BAM bytes to tiecov's outputs on the device (csrc/bgzf.cu): BGZF inflate and record parse against the columns that were
written, the reference's own BAMs, its md5s and heat-map goldens, chunking invariance, and clean errors on malformed input."""
import hashlib
import os
import struct

import numpy as np
import pytest

import bam_writer as W
import helpers as H
from test_bam_writer import LAYOUTS, synthetic_file

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from tiebrush_b200 import api
    with api.Context(device=0) as c:
        yield c


def _np(cols):
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in cols.items()}


def _columns(ctx, data, skip):
    cols, st = ctx.bam_columns(data, skip, last=True)
    c = _np(cols)
    c["cig_off"] = c["cig_off"].view(np.uint32); c["cigar"] = c["cigar"].view(np.uint32)
    return c, st


def _expected(meta):
    from tiebrush_b200 import sam
    ex = dict(tid=[], pos=[], end=[], yc=[], yx=[], strand=[], cig_off=[0], cigar=[])
    for flag, tid, pos, cig, tags in meta:
        if flag & 4:
            continue
        t = {}
        for name, typ, v in tags:
            t.setdefault(name, (typ, v))
        ex["tid"].append(tid); ex["pos"].append(pos)
        ex["end"].append(pos + sum(w >> 4 for w in cig if (w & 15) in (0, 2, 3, 7, 8)))
        ex["yc"].append(np.float32(t["YC"][1]) if "YC" in t else np.float32(1))
        ex["yx"].append(int(t["YX"][1]) if "YX" in t else 1)
        ex["strand"].append(ord(sam.splice_strand(t, flag)))
        ex["cigar"] += cig; ex["cig_off"].append(len(ex["cigar"]))
    dt = dict(tid=np.int32, pos=np.int32, end=np.int32, yc=np.float32, yx=np.int32, strand=np.uint8, cig_off=np.uint32, cigar=np.uint32)
    return {k: np.asarray(v, dt[k]) for k, v in ex.items()}


def _assert_cols(got, exp, keys=("tid", "pos", "end", "yx", "strand", "cig_off", "cigar")):
    for k in keys:
        assert np.array_equal(got[k], exp[k]), k
    assert np.array_equal(got["yc"].view(np.uint32), exp["yc"].astype(np.float32).view(np.uint32)), "yc"


@pytest.mark.parametrize("variant", list(W.VARIANTS))
@pytest.mark.parametrize("layout", LAYOUTS)
def test_bam_columns_equal_the_written_records(ctx, layout, variant):
    from tiebrush_b200 import api
    data, recs, text, meta = synthetic_file(layout, variant)
    import tempfile
    with tempfile.NamedTemporaryFile(suffix=".bam") as f:
        f.write(data); f.flush()
        h = api.read_bam_header(f.name)
    got, st = _columns(ctx, data[h["block_offset"]:], h["skip"])
    exp = _expected(meta)
    assert st["unmapped"] == sum(1 for m in meta if m[0] & 4) and st["records"] == len(exp["pos"])
    assert st["resume_byte"] == len(data) - h["block_offset"]
    _assert_cols(got, exp)


@pytest.mark.parametrize("name", [f"t{t}s{i}" for t in (1, 2) for i in range(10)])
def test_fixture_bams_decode_into_the_fixture_columns(ctx, name):
    from tiebrush_b200 import api
    path = os.path.join(H.FIXTURES, name[:2], name + ".bam")
    files, _, _ = H.fixture_inputs([name[:2]])
    c = files[int(name[3:])]
    keep = (c["flag"] & 4) == 0
    h = api.read_bam_header(path)
    data = open(path, "rb").read()
    got, st = _columns(ctx, data[h["block_offset"]:], h["skip"])
    assert st["records"] == int(keep.sum())
    for k in ("tid", "pos", "strand"):
        assert np.array_equal(got[k], np.asarray(c[k])[keep]), k
    yc = np.where(c["has_yc"], c["yc_in"], np.float32(1)).astype(np.float32)[keep]
    assert np.array_equal(got["yc"], yc) and np.array_equal(got["yx"], np.asarray(c["yx_in"])[keep])
    off = np.asarray(c["cig_off"], np.int64)
    cig = np.concatenate([np.asarray(c["cigar"])[off[i]:off[i + 1]] for i in np.nonzero(keep)[0]] or [np.zeros(0, np.uint32)]).astype(np.uint32)
    assert np.array_equal(got["cigar"], cig)


def _collapsed_bam(tmp_path, layout):
    """The t1+t2 collapse of the reference's fixtures as a BAM file (the records tiebrush writes, test writer)."""
    from tiebrush_b200 import api
    files, header, lines = H.fixture_inputs(["t1", "t2"])
    with api.Context(device=0, n_samples=len(files)) as c:
        got = H.run_collapse(lambda cols, run_off, **kw: c.collapse_window(cols, run_off, tid=kw["tid"], file_merged=kw["file_merged"]), files, {})
    records = H.collapsed_records(got, lines)
    sq = [ln for ln in header if ln.startswith("@SQ")]
    names = [next(f[3:] for f in ln.split("\t") if f.startswith("SN:")) for ln in sq]
    lens = [int(next(f[3:] for f in ln.split("\t") if f.startswith("LN:"))) for ln in sq]
    ids = {n: i for i, n in enumerate(names)}
    recs = [W.record_from_sam(r.split("\t"), ids) for r in records]
    hdr = W.header_bytes("\n".join(header) + "\n", names, lens)
    pl = W.blocks(hdr, recs) if layout == "htslib" else W.blocks(hdr, recs, "fixed", cut=7777)
    p = tmp_path / f"t12_{layout}.bam"
    p.write_bytes(W.bgzf_file(pl, "l6"))
    return str(p), header, records


@pytest.mark.parametrize("layout", ["htslib", "fixed"])
def test_coverage_bam_has_the_reference_md5(ctx, tmp_path, layout):
    path, header, records = _collapsed_bam(tmp_path, layout)
    got = ctx.coverage_bam(path, chunk_bytes=50_000)
    bg, bed = H.coverage_files(got, got["header"]["names"])
    assert hashlib.md5(bg.encode()).hexdigest() == H.REF_MD5["cov"]
    assert hashlib.md5(bed.encode()).hexdigest() == H.REF_MD5["junc"]


@pytest.mark.parametrize("case", ["t1", "t2"])
def test_coverage_bam_sample_heatmap_golden(ctx, tmp_path, case):
    z = np.load(os.path.join(H.GOLDEN, "sample_heatmap.npz"))
    tid, pos, off, cig, yx = (z[f"{case}/in/{k}"] for k in ("tid", "pos", "cig_off", "cigar", "yx_in"))
    ntid = int(tid.max()) + 1
    names = [f"chr{i}" for i in range(ntid)]
    text = "@HD\tVN:1.0\tSO:coordinate\n" + "".join(f"@SQ\tSN:{n}\tLN:500000000\n" for n in names) + "".join(f"@CO\tSAMPLE:s{i}\n" for i in range(10))
    recs = [W.record_bytes(int(tid[i]), int(pos[i]), 0, [int(w) for w in cig[off[i]:off[i + 1]]], [("YX", "i", int(yx[i]))], qname=f"r{i}")
            for i in range(len(pos))]
    p = tmp_path / "s.bam"
    p.write_bytes(W.bgzf_file(W.blocks(W.header_bytes(text, names, [500000000] * ntid), recs)))
    got = ctx.coverage_bam(str(p), want_runs=False, want_juncs=False, want_sample=True, chunk_bytes=30_000)
    assert got["header"]["n_samples"] == 10
    t, s, e, iv = got["sample"]
    assert np.array_equal(t, z[f"{case}/out/tid"]) and np.array_equal(s, z[f"{case}/out/start"])
    assert np.array_equal(e, z[f"{case}/out/end"]) and np.array_equal(iv, z[f"{case}/out/ival"])


def _stream_bam(tmp_path, n, seed, frac=False, layout="htslib"):
    from tiebrush_b200 import synth
    host = synth.to_host(synth.coverage_stream(n, seed=seed, n_tx=40, chroms=3))
    rng = np.random.default_rng(seed)
    host["yx"] = rng.integers(1, 61, n).astype(np.int32)
    if frac:
        host["yc"] = (rng.integers(1, 40, n).astype(np.float32) / rng.choice(np.asarray([3, 5, 7], np.float32), n)).astype(np.float32)
    buf, ends = W.columns_records(host, l_seq=150)
    names = ["c0", "c1", "c2"]
    hdr = W.header_bytes("@HD\tVN:1.6\n" + "".join(f"@SQ\tSN:{x}\tLN:300000000\n" for x in names), names, [300000000] * 3)
    pl = W.columns_payloads(hdr, buf, ends) if layout == "htslib" else W.blocks(hdr, [bytes(buf)], "fixed", cut=9000)
    p = tmp_path / f"s{seed}.bam"
    p.write_bytes(W.bgzf_file(pl, "l6"))
    return str(p), host


def _rows_equal(got, exp):
    for a, b in zip(got["runs"] + got["juncs"], exp["runs"] + exp["juncs"]):
        assert np.array_equal(np.asarray(a), np.asarray(b))


@pytest.mark.parametrize("chunk", [None, 100_000, "block", 997, 20_001])
def test_coverage_bam_is_the_same_for_every_chunk_size(ctx, tmp_path, chunk):
    """Whole file, 100 KB, one block at a time, chunks that end inside the header (fixed cuts: the header spans blocks) and
    inside blocks; a small window too. Rows equal tc_coverage_stream on the generator's columns and the oracle (-c / -j),
    and sample_window / the oracle (-s)."""
    from oracle import oracle
    from tiebrush_b200 import api
    path, host = _stream_bam(tmp_path, 30000, 5, layout="fixed" if chunk in ("block", 997) else "htslib")
    data = open(path, "rb").read()
    cb = len(data) + 1 if chunk is None else (int.from_bytes(data[16:18], "little") + 1 if chunk == "block" else chunk)
    got = ctx.coverage_bam(path, want_sample=True, chunk_bytes=cb, window=1024 if chunk == 20_001 else 1 << 22)
    exp = oracle.coverage(host)
    _rows_equal(got, exp)
    cap = 2 * int(host["cig_off"][-1]) + 16
    ref = ctx.coverage_stream(host, 1 << 22, api.cov_out_buffers(cap, cap))
    _rows_equal(got, ref)
    sw, so = ctx.sample_window(host), oracle.sample_heatmap(host)
    for a, b, c in zip(got["sample"], sw, so):
        assert np.array_equal(a, b) and np.array_equal(np.asarray(a), c)


def test_coverage_bam_fractional_yc_takes_the_exact_path(ctx, tmp_path):
    from oracle import oracle
    path, host = _stream_bam(tmp_path, 20000, 7, frac=True, layout="fixed")
    got = ctx.coverage_bam(path, chunk_bytes=40_000)
    assert ctx.last_cov_exact() == 1
    _rows_equal(got, oracle.coverage(host))


def test_coverage_bam_bundle_over_many_chunks(ctx, tmp_path):
    """One deep bundle (every record overlaps the next) across many small chunks, small windows."""
    from oracle import oracle
    n = 6000
    cols = dict(tid=np.zeros(n, np.int32), pos=(np.arange(n) * 10).astype(np.int32), cig_off=np.arange(n + 1, dtype=np.uint32),
                cigar=np.full(n, (150 << 4) | 0, np.uint32), yc=np.ones(n, np.float32), strand=np.full(n, ord("+"), np.uint8))
    buf, ends = W.columns_records(cols, l_seq=150)
    hdr = W.header_bytes("@SQ\tSN:c0\tLN:1000000\n", ["c0"], [1000000])
    p = tmp_path / "deep.bam"
    p.write_bytes(W.bgzf_file(W.columns_payloads(hdr, buf, ends)))
    got = ctx.coverage_bam(str(p), chunk_bytes=20_000, window=1024)
    _rows_equal(got, oracle.coverage(cols))


def _corrupt(data, what):
    b = bytearray(data)
    o = 0
    bsize = lambda q: int.from_bytes(b[q + 16:q + 18], "little")
    o = bsize(0) + 1                                  # second block: the first record block of an htslib file
    if what == "magic":
        b[o] = 0x1e
    elif what == "crc":
        b[o + bsize(o) + 1 - 8] ^= 0x01
    elif what == "isize":
        b[o + bsize(o) + 1 - 4] ^= 0x01
    elif what == "huffman":
        b[o + 18 + 1] ^= 0xff                         # inside the dynamic header's code length codes
    elif what == "truncated":
        b = b[:-(28 + 20)]                            # no EOF marker and the last block cut short
    return bytes(b), o


@pytest.mark.parametrize("what", ["magic", "crc", "isize", "huffman", "truncated", "block_size"])
def test_malformed_input_returns_an_error_and_the_context_stays_usable(ctx, tmp_path, what):
    from tiebrush_b200 import api
    data, recs, text, meta = synthetic_file("htslib", "l6")
    h_off = int.from_bytes(data[16:18], "little") + 1
    if what == "block_size":
        # the last record claims more bytes than the file holds
        body = b"".join(recs[:-1]) + struct.pack("<i", len(recs[-1]) + 100) + recs[-1][4:]
        hdr = W.header_bytes(text, ["c0", "c1"], [1000000, 2000000])
        bad, boff = W.bgzf_file(W.blocks(hdr, [body])), None
    else:
        bad, boff = _corrupt(data, what)
    with pytest.raises(api.TieBrushError) as e:
        ctx.bam_columns(bad[h_off:], 0, last=True)
    msg = str(e.value)
    if what in ("magic", "crc", "isize", "huffman"):
        assert f"byte offset {boff - h_off}" in msg, msg
    else:
        assert "byte offset" in msg, msg
    good, _ = _columns(ctx, data[h_off:], 0)
    _assert_cols(good, _expected(meta))


def test_cg_tag_and_unmapped_refid_are_refused(ctx):
    from tiebrush_b200 import api
    hdr = W.header_bytes("@SQ\tSN:c0\tLN:1000\n", ["c0"], [1000])
    for tags, tid, flag, word in (([("CG", "B", ("I", [160]))], 0, 0, "CG"), ([], -1, 0, "refID")):
        rec = W.record_bytes(tid, 5, flag, [(10 << 4) | 0], tags)
        data = W.bgzf_file([hdr, rec])
        with pytest.raises(api.TieBrushError, match=word):
            ctx.bam_columns(data[len(W.bgzf_block(hdr)):], 0, last=True)


def test_coverage_bam_at_scale(ctx, tmp_path):
    """1e7 records: rows equal tc_coverage_stream on the same columns (count and properties on all rows, oracle on a prefix
    of whole bundles)."""
    from oracle import oracle
    from tiebrush_b200 import api, synth
    n = 10_000_000
    host = synth.to_host(synth.coverage_stream(n, seed=11, n_tx=20000, chroms=4))
    buf, ends = W.columns_records(host, l_seq=0)
    names = [f"c{i}" for i in range(4)]
    hdr = W.header_bytes("".join(f"@SQ\tSN:{x}\tLN:300000000\n" for x in names), names, [300000000] * 4)
    p = tmp_path / "big.bam"
    p.write_bytes(W.bgzf_file(W.columns_payloads(hdr, buf, ends), "l1", threads=16))
    del buf
    got = ctx.coverage_bam(str(p), chunk_bytes=64 << 20)
    assert got["stat"]["records"] == n
    cap = 2 * int(host["cig_off"][-1]) + 16
    ref = ctx.coverage_stream(host, 1 << 22, api.cov_out_buffers(cap, cap // 2))
    assert got["n_runs"] == ref["n_runs"] and got["n_juncs"] == ref["n_juncs"]
    _rows_equal(got, ref)
    t, s, e, v = got["runs"]
    assert (e > s).all() and (v > 0).all()
    cut = synth.bundle_cut(host, 200_000)
    exp = oracle.coverage(synth.take_prefix(host, cut))
    r = len(exp["runs"][0])
    for a, b in zip(got["runs"], exp["runs"]):
        assert np.array_equal(np.asarray(a)[:r], b)
