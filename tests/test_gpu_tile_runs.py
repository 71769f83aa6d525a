"""The tile front end (collapse_tile.cu) on windows built out of runs of identical neighbours, against the oracle.

Inside a 32-record warp step, a record that is the same alignment as the record before it in the same file joins that
record's run; only the run's first record (its head) probes the group table, with the run's length as its weight, and
the heads of a warp are queued until 32 of them probe as one full warp. These windows put runs where that bookkeeping
can break: lengths around one and two warp steps, runs that cross a warp's range (inside one file and start position,
so the range's look-back maximum is involved), both sides of a slot's pile-up split, records the filters drop at the
start, middle and end of a run, neighbours that differ only in strand or (with -L) MD, CIGARs that differ but are
equal under -P / -E, 1 to 70 samples, a position deep enough for the full-size relaunch, and one with more distinct
alignments than the largest table (sent to the ordered path). Every window must equal the oracle bit for bit, and the
tile statistics must show fewer heads than records."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

OP_M, OP_I, OP_D, OP_N, OP_S = 0, 1, 2, 3, 4


def _w(n, op):
    return (n << 4) | op


# reference lengths 50, 40, 550, 52, 49, 50, 40, 40: entries 5 and 7 equal entries 0 and 1 under -P and -E (soft clips
# only), entry 6 has entry 1's reference length with other ops
POOL = [
    [_w(50, OP_M)],
    [_w(10, OP_S), _w(40, OP_M)],
    [_w(20, OP_M), _w(500, OP_N), _w(30, OP_M)],
    [_w(30, OP_M), _w(2, OP_D), _w(20, OP_M)],
    [_w(25, OP_M), _w(1, OP_I), _w(24, OP_M)],
    [_w(7, OP_S), _w(50, OP_M)],
    [_w(40, OP_M)],
    [_w(3, OP_S), _w(40, OP_M), _w(6, OP_S)],
]
MD_POOL = [b"50", b"12G37", b"0C49", b"30^AC18"]
RUN_LENS = [1, 2, 3, 31, 32, 33, 64, 65]
# a record the options may drop: (flag, mapq, nh)
DROPS = [(0x100, 60, 1), (0x800, 60, 1), (0, 0, 1), (0, 60, 3)]


def _position_runs(rng, depth, k, pool=None, run_lens=RUN_LENS):
    """`depth` records at one start position as a list of (file, runs), each run a list of record tuples
    (cigar, strand, md, flag, mapq, nh). A run goes to one file whole; the next run often repeats the alignment with the
    other strand, another MD or the -P / -E twin of its CIGAR, and a run may hold a record the filters drop."""
    out, n, prev = [], 0, None
    npool = len(POOL) if pool is None else pool
    while n < depth:
        L = int(min(rng.choice(run_lens), depth - n))
        ci, st, mi = int(rng.integers(npool)), int(rng.integers(2)), int(rng.integers(len(MD_POOL)))
        if prev is not None and rng.random() < 0.5:
            ci, st, mi = prev
            what = rng.integers(3)
            if what == 0:
                st ^= 1
            elif what == 1:
                mi = (mi + 1) % len(MD_POOL)
            elif ci in (0, 1, 5, 7) and pool is None:
                ci = {0: 5, 5: 0, 1: 7, 7: 1}[ci]
        rec = (ci, st, mi, 0, 60, 1)
        run = [rec] * L
        if rng.random() < 0.4:
            at = int(rng.choice([0, L // 2, L - 1]))
            fl, mq, nh = DROPS[int(rng.integers(len(DROPS)))]
            run[at] = (ci, st, mi, fl, mq, nh)
        f = int(rng.integers(k)) if rng.random() < 0.7 or prev is None else out[-1][0]
        out.append((f, run))
        n += L
        prev = (ci, st, mi)
    return out


def build_window(rng, k, sites, big_pool=None, run_lens=RUN_LENS):
    """File-major host columns and run_off. `sites` is a list of (start position, depth); within a file, records keep
    the order their runs were drawn in. `big_pool` (n) draws CIGARs from n distinct ones instead of POOL."""
    pool = POOL if big_pool is None else [[_w(10 + c % 90, OP_M), _w(100 + c // 90, OP_N), _w(30, OP_M)] for c in range(big_pool)]
    per_file = [[] for _ in range(k)]
    for p, depth in sorted(sites):
        for f, run in _position_runs(rng, depth, k, big_pool, run_lens):
            per_file[f] += [(p,) + r for r in run]
    recs = [r for f in range(k) for r in per_file[f]]
    run_off = np.concatenate([[0], np.cumsum([len(x) for x in per_file])]).astype(np.int64)
    n = len(recs)
    a = np.array([r[:7] for r in recs], np.int64).reshape(n, 7)
    cols = dict(pos=a[:, 0].astype(np.int32), flag=a[:, 4].astype(np.uint16), mapq=a[:, 5].astype(np.uint8),
                strand=np.frombuffer(b"+-", np.uint8)[a[:, 2]], nh=a[:, 6].astype(np.uint16),
                qhash=np.arange(n, dtype=np.uint64))
    cig = [pool[c] for c in a[:, 1]]
    cols["cig_off"] = np.concatenate([[0], np.cumsum([len(c) for c in cig])]).astype(np.uint32)
    cols["cigar"] = np.array([w for c in cig for w in c], np.uint32)
    md = [MD_POOL[m] + b"\0" for m in a[:, 3]]
    cols["md_off"] = np.concatenate([[0], np.cumsum([len(s) for s in md])]).astype(np.uint32)
    cols["md"] = np.frombuffer(b"".join(md), np.uint8).copy()
    return cols, run_off


def check_tile(cols, run_off, opts, path=0):
    """The window through the GPU equals the oracle; the tile path ran and its statistics are consistent."""
    from oracle import oracle
    from tiebrush_b200 import api
    k = len(run_off) - 1
    n = len(cols["pos"])
    exp = oracle.collapse(cols, run_off, **opts)
    with api.Context(device=0, n_samples=k, **opts) as ctx:
        got = ctx.collapse_window(cols, run_off)
        assert ctx.last_path() == path
        assert got["n_kept"] == exp["n_kept"]
        for key in ("rep_index", "yc", "yx", "yd"):
            assert np.array_equal(np.asarray(got[key]), exp[key]), key
        st = ctx.last_tile_stats()
        heavy = ctx.last_heavy_slots()
    if path != 0:
        return st, heavy, exp
    # every record is streamed at least once (slots redone by the full-size launch twice, or once if sent there directly)
    assert st["records"] >= n
    assert 0 < st["heads"] <= st["records"]
    assert st["heads"] <= exp["n_kept"] + st["records"] - n   # heads are passing records; redone slots probe again
    assert 32 * st["batches"] <= st["heads"]
    return st, heavy, exp


def _slot_records(k):
    """Records per slot T of the 256-thread geometry (col_front_tile), assuming the B200's 227 KB of opt-in shared
    memory per block. Only used to line a slot up with a position; the tests hold whatever it returns."""
    W = (k + 31) // 32
    limit = (227 * 1024 + 1024) // 4 - 1024 - 512
    E = 8192
    while E > 64 and E * (26 + 4 * W) + (6 * k + 1) * 4 + 64 > limit:
        E -= 64
    return ((E - 1) * 4 // 5) * 7 // 8


OPTS = {
    "default": {},
    "L": dict(mode=1),
    "P": dict(mode=2),
    "E": dict(mode=3),
    "N": dict(max_nh=2),
    "Q": dict(min_qual=10),
    "S": dict(keep_bits=1),
}


@pytest.mark.parametrize("opt", list(OPTS))
@pytest.mark.parametrize("k", [1, 32, 33, 70])
def test_runs_vs_oracle(k, opt):
    """Shallow positions, an ordinary position of 1000 records (several warps' ranges), then the last ordinary position
    of a slot right before a pile-up of 4000 records (the single-position sub-tile), then more shallow positions."""
    rng = np.random.default_rng([k, list(OPTS).index(opt)])
    shallow = lambda lo, hi, c: [(int(p), int(rng.integers(1, 80))) for p in rng.choice(np.arange(lo, hi), c, replace=False)]
    sites = shallow(1000, 1400, 30) + [(1500, 1000)] + shallow(1501, 1900, 20)
    pad = -sum(d for _, d in sites) % _slot_records(k)   # position 2000 starts a slot, so 2001 is that slot's pile-up
    sites += ([(1999, pad)] if pad else []) + [(2000, 300), (2001, 4000)] + shallow(2002, 2400, 30)
    cols, run_off = build_window(rng, k, sites)
    st, _, exp = check_tile(cols, run_off, OPTS[opt])
    assert st["heads"] < exp["n_kept"]   # the runs were found


@pytest.mark.parametrize("k", [1, 12])
def test_one_position_runs_across_warps(k):
    """A window of one start position: every warp's range starts inside the same (file, position) run of records."""
    rng = np.random.default_rng([k, 99])
    cols, run_off = build_window(rng, k, [(777, 1200)])
    st, _, exp = check_tile(cols, run_off, {})
    assert st["heads"] < exp["n_kept"]


def test_heavy_relaunch_runs():
    """A pile-up of 60000 records goes straight to the full-size launch."""
    rng = np.random.default_rng(5)
    k = 12
    sites = [(int(p), int(rng.integers(1, 50))) for p in rng.choice(np.arange(100, 400), 40, replace=False)] + [(500, 60000)]
    cols, run_off = build_window(rng, k, sites)
    st, heavy, exp = check_tile(cols, run_off, dict(mode=2))
    assert heavy >= 1
    assert st["heads"] < exp["n_kept"] and st["batches"] > 0


def test_more_alignments_than_the_table_fall_back():
    """A position with more distinct alignments than the full-size table holds: the window goes to the ordered path."""
    rng = np.random.default_rng(6)
    k = 8
    sites = [(int(p), int(rng.integers(1, 50))) for p in rng.choice(np.arange(100, 400), 40, replace=False)] + [(500, 150000)]
    cols, run_off = build_window(rng, k, sites, big_pool=60000, run_lens=[1, 1, 2, 33])
    deep = (cols["pos"] == 500) & ((cols["flag"] & 0x900) == 0)
    co = cols["cig_off"]
    keys = {(tuple(cols["cigar"][co[i]:co[i + 1]]), int(cols["strand"][i])) for i in np.nonzero(deep)[0]}
    assert len(keys) > 8192   # more groups than any table has entries
    check_tile(cols, run_off, {}, path=2)
