"""The ordered collapse front end (collapse_ordered.cu) against the oracle, where its results depend on record order and on
the probe order of the list search: deep start positions on both sides of the thread / warp kernel switch, more than 32
samples, file boundaries that share a start position, empty files, window spans that need every radix digit pass, and
every option that routes to this path (-F, -A, --store-frac, TieBrush-made inputs) plus the table-overflow fallback.

Every window runs three ways: with the default kernel switch (positions of at least 96 records go to the one-warp-per-
position kernel), with TB_ORD_DEEP=1 (every position on the warp kernel) and with TB_ORD_DEEP=0 (every position on the
one-thread kernel). Each run must equal the oracle bit for bit, and reports the path and the warp-kernel positions it
took, so that a case cannot pass on a path it did not run."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DEFAULT_DEEP = 96
OP_M, OP_I, OP_D, OP_N, OP_S = 0, 1, 2, 3, 4
NH_VALUES = np.array([0, 1, 2, 3, 7, 65535], np.uint16)
MAPQ_VALUES = np.array([0, 1, 60], np.uint8)
STRANDS = np.frombuffer(b"+-.", np.uint8)
MD_POOL = [b"75", b"12G62", b"0C74", b"30^AC45"]


def _cigar_pool(rng, m):
    """m distinct CIGARs (lists of BAM words). Every other entry is a twin of the one before it with the same reference
    length but different ops (an I inserted into an M block, or a D turned into an N), so ord_less has to break ties on
    the ops; some introns are long (over 4095, the escape of the compact CIGAR format, and up to 200 kb)."""
    pool, seen = [], set()
    while len(pool) < m:
        words = []
        if rng.random() < 0.2:
            words.append((int(rng.integers(1, 20)) << 4) | OP_S)
        for b in range(int(rng.integers(1, 4))):
            if b:
                words.append((int(rng.choice([40, 300, 5000, 200_000])) << 4) | OP_N)
            a = int(rng.integers(10, 60))
            if rng.random() < 0.25:
                words += [(a << 4) | OP_M, (int(rng.integers(1, 4)) << 4) | OP_D, (int(rng.integers(5, 30)) << 4) | OP_M]
            else:
                words.append((a << 4) | OP_M)
        if rng.random() < 0.2:
            words.append((int(rng.integers(1, 20)) << 4) | OP_S)
        twin = list(words)
        d = [j for j, w in enumerate(twin) if w & 0xF == OP_D]
        if d:
            twin[d[0]] = (twin[d[0]] & ~0xF) | OP_N
        else:
            j = next(j for j, w in enumerate(twin) if w & 0xF == OP_M)
            ln = twin[j] >> 4
            twin[j:j + 1] = [((ln // 2) << 4) | OP_M, (2 << 4) | OP_I, ((ln - ln // 2) << 4) | OP_M]
        for c in (words, twin):
            if tuple(c) not in seen and len(pool) < m:
                seen.add(tuple(c))
                pool.append(c)
    return pool


def build_window(rng, k, sites, merged=None, with_md=False, nh=None, flag_or=0):
    """File-major host columns and run_off of one window. `sites` is a list of (start position, records[, files[, pool]]):
    that many records start there, spread over `files` (default: all k). Within a file the records are in position order
    and, at one position, in random order. Per position: a pool of 2-50 distinct CIGARs drawn with skewed weights (or
    `pool` CIGARs drawn uniformly), 1-3 QNAME
    hashes per (file, position) so the -A skip rule fires often, and flag bits that -F 16 / 83 / 1040 mask, both pair
    orders, 0x100 and 0x800. `merged` (per-file 0/1) adds TieBrush-made yc_in / yx_in / yd_in columns."""
    recs = []
    for si, site in enumerate(sites):
        p, d = int(site[0]), int(site[1])
        files = np.asarray(site[2] if len(site) > 2 else np.arange(k))
        if len(site) > 3:
            cig = _cigar_pool(rng, site[3])
            w = np.ones(len(cig))
        else:
            cig = _cigar_pool(rng, int(rng.integers(2, 51)))
            w = 1.0 / np.arange(1, len(cig) + 1)
        ci = rng.choice(len(cig), d, p=w / w.sum())
        f = rng.choice(files, d)
        npool = rng.integers(1, 4, k)
        recs.append(dict(pos=np.full(d, p, np.int32), f=f, cig=[cig[c] for c in ci], ci=ci,
                         qhash=(np.uint64(4 * si + 1) + rng.integers(0, npool[f]).astype(np.uint64)).astype(np.uint64)))
    pos = np.concatenate([r["pos"] for r in recs])
    f = np.concatenate([r["f"] for r in recs])
    cig = [c for r in recs for c in r["cig"]]
    n = len(pos)
    flag = np.zeros(n, np.uint16)
    for bit, pr in ((0x1, 0.5), (0x2, 0.4), (0x10, 0.4), (0x400, 0.15), (0x100, 0.05), (0x800, 0.05)):
        flag |= np.where(rng.random(n) < pr, bit, 0).astype(np.uint16)
    flag |= rng.choice(np.array([0, 0x40, 0x80], np.uint16), n)
    flag |= np.uint16(flag_or)
    cols = dict(pos=pos, flag=flag, mapq=rng.choice(MAPQ_VALUES, n, p=[0.1, 0.1, 0.8]),
                strand=rng.choice(STRANDS, n), nh=nh(n) if nh else rng.choice(NH_VALUES, n, p=[0.1, 0.5, 0.15, 0.1, 0.1, 0.05]),
                qhash=np.concatenate([r["qhash"] for r in recs]))
    if merged is not None:
        cols["yc_in"] = rng.choice(np.array([0, 1, 1 / 3, 2.5, 4096, 1e6], np.float32), n)
        cols["yx_in"] = rng.integers(1, k + 1, n).astype(np.int32)
        cols["yd_in"] = rng.choice(np.array([0, 0, 1, 7, 100_000], np.int32), n)
    order = np.lexsort((rng.random(n), pos, f))      # file-major, position order inside a file, random inside a position
    out = {key: v[order] for key, v in cols.items()}
    ncig = np.array([len(cig[i]) for i in order])
    out["cig_off"] = np.concatenate([[0], np.cumsum(ncig)]).astype(np.uint32)
    out["cigar"] = np.array([wd for i in order for wd in cig[i]], np.uint32)
    if with_md:
        md = [MD_POOL[int(x)] + b"\0" for x in rng.integers(0, len(MD_POOL), n)]
        out["md_off"] = np.concatenate([[0], np.cumsum([len(s) for s in md])]).astype(np.uint32)
        out["md"] = np.frombuffer(b"".join(md), np.uint8).copy()
    run_off = np.searchsorted(f[order], np.arange(k + 1)).astype(np.int64)
    return out, run_off


def check_ordered(monkeypatch, cols, run_off, opts, file_merged=None, path=1, expect_groups=True):
    """The window through the GPU with the default kernel switch, TB_ORD_DEEP=1 and TB_ORD_DEEP=0; each run equal to the
    oracle. Returns the warp-kernel position count of the default run."""
    from oracle import oracle
    from tiebrush_b200 import api
    k = len(run_off) - 1
    exp = oracle.collapse(cols, run_off, file_merged=file_merged, **opts)
    assert (len(exp["rep_index"]) > 0) == expect_groups and (exp["n_kept"] > 0) == expect_groups
    depth = np.unique(cols["pos"], return_counts=True)[1]
    deep_default = None
    with api.Context(device=0, n_samples=k, **opts) as ctx:
        for setting, want_deep in ((None, int((depth >= DEFAULT_DEEP).sum())), ("1", len(depth)), ("0", 0)):
            if setting is None:
                monkeypatch.delenv("TB_ORD_DEEP", raising=False)
            else:
                monkeypatch.setenv("TB_ORD_DEEP", setting)
            got = ctx.collapse_window(cols, run_off, file_merged=file_merged)
            assert ctx.last_path() == path, setting
            assert ctx.last_ord_deep() == want_deep, setting
            assert got["n_kept"] == exp["n_kept"], setting
            for key in ("rep_index", "yc", "yx", "yd"):
                assert np.array_equal(np.asarray(got[key]), exp[key]), (setting, key)
            if setting is None:
                deep_default = ctx.last_ord_deep()
    return deep_default


# option sets that route to the ordered path: Context options, builder flags
OPTIONS = {
    "F16": (dict(flag_mask=16), {}),
    "F83": (dict(flag_mask=83), {}),
    "F83_L": (dict(flag_mask=83, mode=1), dict(with_md=True)),
    "F83_P": (dict(flag_mask=83, mode=2), {}),
    "F83_E": (dict(flag_mask=83, mode=3), {}),
    "F1040_E": (dict(flag_mask=1040, mode=3), {}),
    "A": (dict(collapse_same=1), {}),
    "A_keep_sec_supp": (dict(collapse_same=1, keep_bits=2 | 1), {}),
    "frac": (dict(keep_bits=8), {}),
    "frac_keep_sec_F16": (dict(keep_bits=2 | 8, flag_mask=16), {}),
    "merged_all": ({}, dict(merged="all")),
    "merged_mixed": ({}, dict(merged="mixed")),
    "merged_mixed_F16": (dict(flag_mask=16), dict(merged="mixed")),
}


def _file_merged(kind, k):
    if kind is None:
        return None
    return np.ones(k, np.uint8) if kind == "all" else (np.arange(k) % 2 == 0).astype(np.uint8)   # "mixed": even files merged


def _run_case(monkeypatch, rng, k, sites, opt_name, **build):
    opts, extra = OPTIONS[opt_name]
    fm = _file_merged(extra.get("merged"), k)
    cols, run_off = build_window(rng, k, sites, merged=fm, with_md=extra.get("with_md", False), **build)
    return check_ordered(monkeypatch, cols, run_off, opts, file_merged=fm)


def _filler(rng, lo, hi, count, k, max_depth=20):
    """Shallow positions (one-thread kernel) around the interesting ones."""
    return [(int(p), int(rng.integers(1, max_depth + 1)), rng.choice(k, int(rng.integers(1, k + 1)), replace=False))
            for p in rng.choice(np.arange(lo, hi), count, replace=False)]


@pytest.mark.parametrize("opt_name", list(OPTIONS))
@pytest.mark.parametrize("depth", [1, 95, 96, 97, 1000, 20000])
def test_deep_position_vs_oracle(depth, opt_name, monkeypatch):
    """One position of `depth` records among shallow ones: the kernel switch at 96 records, and deep pile-ups."""
    rng = np.random.default_rng([depth, list(OPTIONS).index(opt_name)])
    k = 12
    sites = _filler(rng, 10_000, 10_400, 40, k) + [(10_500, depth)] + _filler(rng, 10_501, 10_900, 40, k)
    _run_case(monkeypatch, rng, k, sites, opt_name)


@pytest.mark.parametrize("opt_name", ["A", "frac", "F83", "F1040_E", "merged_mixed"])
@pytest.mark.parametrize("k", [1, 31, 32, 33, 64, 65, 100])
def test_many_samples_vs_oracle(k, opt_name, monkeypatch):
    """k samples (bitset words W = 1 .. 4). Samples 0 and k-1, and every seventh one, hold no record except at the deep
    position, so their bits come from the warp kernel alone."""
    rng = np.random.default_rng([k, 7, list(OPTIONS).index(opt_name)])
    lonely = sorted({0, k - 1} | set(range(3, k, 7)))
    rest = np.array([f for f in range(k) if f not in lonely]) if len(lonely) < k else np.arange(k)
    sites = [(int(p), int(rng.integers(1, 30)), rng.choice(rest, int(rng.integers(1, len(rest) + 1)), replace=False))
             for p in rng.choice(np.arange(50_000, 51_000), 60, replace=False)]
    sites.append((51_000, 40 * k + 100))
    sites.append((51_001, 150, rest))
    deep = _run_case(monkeypatch, rng, k, sites, opt_name)
    assert deep == 2


def _chain_sites(rng, k, empty):
    """File f holds start positions q_f .. q_{f+1}: the last records of file f and the first of the next non-empty file
    share position q_{f+1}. Files in `empty` hold nothing (first, last, and between two files sharing a position)."""
    live = [f for f in range(k) if f not in empty]
    q = 20_000 + 37 * np.arange(len(live) + 1)
    sites = []
    for j, f in enumerate(live):
        sites.append((int(q[j]) + 5, int(rng.integers(1, 40)), [f]))
        sites.append((int(q[j]) + 20, int(rng.integers(90, 110)), [f]))
    for j in range(len(live) + 1):
        owners = [live[x] for x in (j - 1, j) if 0 <= x < len(live)]
        sites.append((int(q[j]), 130 if j % 2 else 40, owners))
    return sites


@pytest.mark.parametrize("opt_name", ["frac", "A", "F83", "merged_mixed"])
@pytest.mark.parametrize("empty", [(), (0,), (8,), (4,), (0, 4, 5, 8)])
def test_file_boundary_positions_vs_oracle(empty, opt_name, monkeypatch):
    """The merge-order key (position, running maximum of the reference end) restarts at every (file, position): a file
    that starts at the position where the previous one ends must not inherit its running maximum."""
    rng = np.random.default_rng([len(empty), sum(empty), list(OPTIONS).index(opt_name), 3])
    _run_case(monkeypatch, rng, 9, _chain_sites(rng, 9, set(empty)), opt_name)


@pytest.mark.parametrize("opt_name", ["frac", "F16", "A"])
@pytest.mark.parametrize("span", [1, (1 << 16) - 1, (1 << 16) + 1, 250_000_000])
def test_window_span_vs_oracle(span, opt_name, monkeypatch):
    """Window spans of 1 position, 2^16 - 1, 2^16 + 1 and about chr1: the sort key has 32 + ceil(log2 span) bits, so
    these take 5, 6, 7 and 8 radix passes."""
    rng = np.random.default_rng([span, list(OPTIONS).index(opt_name)])
    k = 6
    lo = 100
    if span == 1:
        sites = [(lo, 3000)]
    else:
        mid = rng.choice(np.arange(lo + 1, lo + span - 1), min(span - 2, 50), replace=False)
        sites = [(lo, 200)] + [(int(p), int(rng.integers(1, 120))) for p in mid] + [(lo + span - 1, 150)]
    _run_case(monkeypatch, rng, k, sites, opt_name)


@pytest.mark.parametrize("name,opts,build", [
    ("N", dict(max_nh=2, keep_bits=8), dict(nh=lambda n: np.full(n, 3, np.uint16))),
    ("Q", dict(min_qual=61, flag_mask=16), {}),
    ("secondary", dict(collapse_same=1), dict(flag_or=0x100)),
    ("supplementary", dict(keep_bits=2 | 8), dict(flag_or=0x800)),
])
def test_fully_filtered_window(name, opts, build, monkeypatch):
    """Every record dropped by -N / -Q / the flag bits: no group, nothing kept, but the deep positions (counted over
    all records) still go to the warp kernel."""
    rng = np.random.default_rng(len(name))
    k = 5
    cols, run_off = build_window(rng, k, _filler(rng, 300, 400, 30, k) + [(500, 400)], **build)
    assert check_ordered(monkeypatch, cols, run_off, opts, expect_groups=False) == 1


def test_table_overflow_fallback_many_samples(monkeypatch):
    """Default options, 65 samples (W = 2): a position with more distinct alignments than a shared-memory table sends the
    window from the tile path to the ordered path (last_path 2)."""
    rng = np.random.default_rng(65)
    k = 65
    sites = _filler(rng, 1_000, 1_900, 100, k, max_depth=150) + [(2_000, 13_000, np.arange(k), 20_000)]
    cols, run_off = build_window(rng, k, sites)
    assert check_ordered(monkeypatch, cols, run_off, {}, path=2) >= 2


def test_c3_shaped_exon_mode_f83_vs_oracle(monkeypatch):
    """The benchmark's -E -F 83 leg at a reduced size: 100 samples of paired reads on chr1, a few transcripts so that
    start positions pile up to thousands of records. The whole window against the oracle."""
    from tiebrush_b200 import synth
    cols, run_off, pr = synth.cohort_window(100, 50_000, seed=4, n_tx=2, device="cpu", paired=True)
    host = synth.to_host(cols)
    depth = np.unique(host["pos"], return_counts=True)[1]
    assert depth.max() >= 2000 and (depth >= 1000).sum() > 1000
    deep = check_ordered(monkeypatch, host, run_off, dict(mode=3, flag_mask=83))
    assert deep > 2000
