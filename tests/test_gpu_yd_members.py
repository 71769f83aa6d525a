"""GPU checks of the YD chain members and their sub-chain heads (count pass with block end maxima, prefix maxima, scatter
with the head test, head list) on the shapes that pass must get right: one unbroken chain over many 1024-group blocks,
chains with no member in whole blocks, one and several 32-sample bit words, strand '.' groups, and a carried frontier
above every end of the first block. Groups against the oracle on both YD paths; member and sub-chain counts
(Context.last_yd_stats) against a numpy model of the head rule."""
from collections import defaultdict

import numpy as np
import pytest

import yd_carry_oracle as YO

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["par", "seq"])
def yd_path(request, monkeypatch):
    monkeypatch.setenv("TB_YD_PATH", request.param)
    return request.param


def ref_len(cigar):
    import re
    return sum(int(n) for n, op in re.findall(r"(\d+)([MIDNSHP=X])", cigar) if op in "MDN=X")


def window(samples):
    """File-major window from per-sample lists of (1-based pos, CIGAR, strand '+' / '-' / '.'); '.' = no XS tag."""
    from tiebrush_b200 import sam
    parts = []
    for s, recs in enumerate(samples):
        text = "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:chr1\tLN:1000000\n"
        for i, (p, c, st) in enumerate(sorted(recs)):
            tag = f"\tXS:A:{st}" if st != "." else ""
            text += f"s{s}r{i}\t0\tchr1\t{p}\t60\t{c}\t*\t0\t0\t*\t*{tag}\tNH:i:1\n"
        R, _ = sam.parse_sam(text)
        parts.append(sam.to_columns(R))
    cols = sam.concat(parts)
    run_off = np.cumsum([0] + [len(p["pos"]) for p in parts]).astype(np.int64)
    return cols, run_off


def model_stats(samples, rep_keys, seed=None):
    """Chain members and sub-chains of groups in output order (rep_keys: (1-based pos, CIGAR, strand) per group): member of
    chain c = side * k + sample when the sample holds the group and the strand fits the side; a member heads a sub-chain when
    it is its chain's first or starts beyond every earlier end of the chain and the carried frontier seed[c]."""
    k = len(samples)
    holders = defaultdict(set)
    for s, recs in enumerate(samples):
        for r in recs:
            holders[r].add(s)
    chains = defaultdict(list)
    for key in rep_keys:
        p, c, st = key
        for s in sorted(holders[key]):
            if st != "-":
                chains[s].append((p, p + ref_len(c) - 1))
            if st != "+":
                chains[k + s].append((p, p + ref_len(c) - 1))
    n_sub = 0
    for c, mem in chains.items():
        run = None
        for st, en in mem:
            n_sub += run is None or st > run
            sd = (seed or {}).get(c, -1)
            run = max(en, sd, -1 if run is None else run)
    return sum(len(m) for m in chains.values()), n_sub


def rep_keys_of(cols, rep):
    from tiebrush_b200 import sam
    out = []
    for r in np.asarray(rep).astype(np.int64):
        cig = sam.cigar_str(cols["cigar"][int(cols["cig_off"][r]):int(cols["cig_off"][r + 1])])
        out.append((int(cols["pos"][r]) + 1, cig, chr(int(cols["strand"][r]))))
    return out


def check_vs_oracle(got, exp):
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), np.asarray(exp[key])), key


def long_stretch(k=3, n_pos=4000):
    """Every sample holds every group: one covered stretch of 3 * n_pos groups, no sub-chain head after the first."""
    recs = []
    for p in range(1000, 1000 + n_pos):
        recs += [(p, "100M", "."), (p, "40M10N60M", "+"), (p, "30M20N70M", "+")]
    return [list(recs) for _ in range(k)]


def empty_blocks():
    """Sample 0 fills ~6 blocks; samples 1 and 2 have members only before and after them. Sample 1's first read reaches
    past the filler (its late members are no heads), sample 2's does not (its first late member is a head)."""
    s0 = [(p, c, "+") for p in range(1000, 4000) for c in ("100M", "60M")]
    s1 = [(990, "50M5000N50M", "+"), (4500, "100M", "+"), (4600, "100M", "+")]
    s2 = [(995, "100M", "-"), (4500, "100M", "-"), (4550, "70M", "-")]
    return [s0, s1, s2]


@pytest.mark.parametrize("build", [long_stretch, empty_blocks])
def test_members_and_heads_vs_oracle_and_model(build, yd_path):
    from oracle import oracle
    from tiebrush_b200 import api
    samples = build()
    cols, run_off = window(samples)
    with api.Context(device=0, n_samples=len(samples)) as ctx:
        got = ctx.collapse_window(cols, run_off)
        stats = ctx.last_yd_stats()
        assert ctx.last_yd_path() == (0 if yd_path == "par" else 1)
    check_vs_oracle(got, oracle.collapse(cols, run_off))
    assert stats["nblk"] == (got["n_groups"] + 1023) // 1024
    assert (stats["n_members"], stats["n_subchains"]) == model_stats(samples, rep_keys_of(cols, got["rep_index"]))
    assert (stats["lc"] > 0) == (yd_path == "par")
    if build is long_stretch:
        assert stats["nblk"] >= 10 and stats["n_subchains"] == 2 * len(samples)


@pytest.mark.parametrize("k", [1, 31, 33, 100])
def test_bit_words_vs_oracle(k, yd_path):
    from oracle import oracle
    from tiebrush_b200 import api, synth
    cols, run_off, _ = synth.cohort_window(k, max(200, 40000 // k), seed=k, n_tx=12, device="cpu")
    host = synth.to_host(cols)
    with api.Context(device=0, n_samples=k) as ctx:
        got = ctx.collapse_window(host, run_off)
        stats = ctx.last_yd_stats()
    check_vs_oracle(got, oracle.collapse(host, run_off))
    assert stats["n_members"] > got["n_groups"] and 0 < stats["n_subchains"] < stats["n_members"]


def test_carried_frontier_above_the_first_block(yd_path):
    """Window 1 ends with a long spliced read of sample 0 (its list's frontier reaches 30199); window 2 starts with more
    than a block of groups that all end below it, then a read beyond it. Sample 1's carried node is dead at the cut."""
    from oracle import oracle
    from tiebrush_b200 import api, shard
    dense = [(p, c, "+") for p in range(1000, 2500) for c in ("100M", "60M")]
    samples = [[(100, "50M30000N50M", "+")] + dense + [(40000, "100M", "+")], [(100, "80M", "+")] + dense]
    cols, run_off = window(samples)
    whole = oracle.collapse(cols, run_off)
    exp = shard.collapse_cut_windows(lambda s, o, pos_range, yd_carry: YO.collapse(s, o, yd_carry=yd_carry, pos_range=pos_range),
                                     cols, run_off, [999], YO.empty_carry(2))
    carries = []
    with api.Context(device=0, n_samples=2) as ctx:
        def one(s, o, pos_range, yd_carry):
            r = ctx.collapse_window(s, o, pos_range=pos_range, yd_carry=yd_carry)
            carries.append(yd_carry)
            return r
        got = shard.collapse_cut_windows(one, cols, run_off, [999], api.empty_yd_carry(2))
        stats = ctx.last_yd_stats()
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), np.asarray(whole[key])), key
        assert np.array_equal(np.asarray(got[key]), np.asarray(exp[key])), key
    # the second window's chains: sample 0 starts from the carried frontier 30199, sample 1's carried node ends below it
    cin = carries[1]
    seed = {c: int(cin["seg_end"][cin["chain_off"][c + 1] - 1]) for c in range(4) if cin["chain_off"][c + 1] > cin["chain_off"][c]}
    seed = {c: e for c, e in seed.items() if e >= 1000}
    assert seed == {0: 30199}
    n0 = int(np.count_nonzero(np.asarray(cols["pos"]) < 999))
    sub_keys = [key for key in rep_keys_of(cols, got["rep_index"]) if key[0] >= 1000]
    sub_samples = [[r for r in recs if r[0] >= 1000] for recs in samples]
    assert len(sub_keys) > 1024 and n0 == 2
    assert (stats["n_members"], stats["n_subchains"]) == model_stats(sub_samples, sub_keys, seed)
    assert stats["n_subchains"] == 3   # sample 0: the first member and the read beyond the frontier; sample 1: one sub-chain
