"""CPU checks of the YD carry (tb_collapse_window_carry): the oracle, cut into windows at start positions with no coverage
gap and the YD lists carried across every cut (and into the next reference id), reproduces the compiled reference's
goldens and fixture md5s; the ctypes struct matches the header."""
import os
import re

import numpy as np
import pytest

import helpers as H
import yd_carry_oracle as YO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cut_positions(cols, pattern, seed=0):
    """Cuts at start positions of a window: every start position, every `n`-th, or a seeded random subset."""
    u = np.unique(np.asarray(cols["pos"]))
    if pattern == "every":
        return u[1:]
    if isinstance(pattern, int):
        return u[pattern::pattern]
    rng = np.random.default_rng(seed)
    return u[1:][rng.random(len(u) - 1) < 0.3]


def carried_collapse(compute, pattern, k, log=None):
    """A collapse_fn for helpers.run_collapse: every per-tid window is cut by `pattern` and collapsed window by window with
    `compute(cols, run_off, tid=, file_merged=, yd_carry=, pos_range=, **opts)`; the carry goes on into the next tid."""
    from tiebrush_b200 import shard
    state = dict(carry=YO.empty_carry(k), n=0)

    def fn(cols, run_off, tid=0, file_merged=None, **opts):
        one = lambda sub, off, pos_range, yd_carry: compute(sub, off, tid=tid, file_merged=file_merged, yd_carry=yd_carry, pos_range=pos_range, **opts)
        r = shard.collapse_cut_windows(one, cols, run_off, cut_positions(cols, pattern, seed=tid + 7 * state["n"]), state["carry"])
        state["carry"] = r["yd_carry"]
        state["n"] += 1
        if log is not None:
            log.extend(r["carried"])
        return r
    return fn


def oracle_collapse(cols, run_off, **kw):
    return YO.collapse(cols, run_off, **kw)


@pytest.mark.parametrize("pattern", ["every", 7, "random"])
@pytest.mark.parametrize("npz", ["collapse_random.npz", "collapse_fixture.npz", "collapse_merged.npz"])
def test_oracle_carry_reproduces_goldens(npz, pattern):
    carried = []
    for case in H.case_names(npz):
        files, opts, fm, exp = H.load_collapse_case(npz, case)
        got = H.run_collapse(carried_collapse(oracle_collapse, pattern, len(files), carried), files, opts, fm)
        H.assert_collapse_equal(got, exp, f"{case} cut {pattern}")
    assert sum(carried) > 0   # lists really crossed the cuts


@pytest.mark.parametrize("name,which", [("t1", ["t1"]), ("t2", ["t2"]), ("t12", ["t1", "t2"])])
def test_oracle_carry_every_50_positions_matches_reference_md5(name, which):
    files, header, lines = H.fixture_inputs(which)
    got = H.run_collapse(carried_collapse(oracle_collapse, 50, len(files)), files, {})
    assert (got["n_kept"], len(got["lhash"])) == H.REF_COUNTS[name]
    assert H.md5_text(H.collapsed_records(got, lines)) == H.REF_MD5[name]


def test_carry_matters_in_the_oracle():
    """The same cuts with an empty carry at every cut give a different YD somewhere: the carry is what makes them exact."""
    from oracle import oracle
    from tiebrush_b200 import shard, synth
    k = 6
    cols, run_off, _ = synth.cohort_window(k, 3000, seed=21, n_tx=4, device="cpu")
    host = synth.to_host(cols)
    whole = oracle.collapse(host, run_off)
    cuts = cut_positions(host, 5)
    ok = shard.collapse_cut_windows(lambda s, o, pos_range, yd_carry: YO.collapse(s, o, yd_carry=yd_carry, pos_range=pos_range),
                                    host, run_off, cuts, YO.empty_carry(k))
    lost = shard.collapse_cut_windows(lambda s, o, pos_range, yd_carry: YO.collapse(s, o, yd_carry=YO.empty_carry(k), pos_range=pos_range),
                                      host, run_off, cuts, YO.empty_carry(k))
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(ok[key], whole[key]), key
    assert max(ok["carried"]) > 0
    assert not np.array_equal(lost["yd"], whole["yd"])


def survey_9_4_case(with_a):
    """SURVEY §9.4's hand-built chain: A = 100M at 100 (1-based), B = 30M100N20M at 150, C = 10M at 285, one sample,
    '+' strand. Window 1 holds A and B, window 2 holds C."""
    from tiebrush_b200 import sam
    text = "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:chr1\tLN:100000\n"
    recs = ([("a", 100, "100M")] if with_a else []) + [("b", 150, "30M100N20M"), ("c", 285, "10M")]
    text += "".join(f"{q}\t0\tchr1\t{p}\t60\t{c}\t*\t0\t0\t*\t*\tXS:A:+\tNH:i:1\n" for q, p, c in recs)
    R, _ = sam.parse_sam(text)
    cols = sam.to_columns(R)
    return cols, np.asarray([0, len(cols["pos"])], np.int64)


@pytest.mark.parametrize("with_a,yd_c", [(True, 0), (False, 5)])
def test_oracle_survey_9_4_case_cut_between_b_and_c(with_a, yd_c):
    from oracle import oracle
    from tiebrush_b200 import shard
    cols, run_off = survey_9_4_case(with_a)
    whole = oracle.collapse(cols, run_off)
    cut = shard.collapse_cut_windows(lambda s, o, pos_range, yd_carry: YO.collapse(s, o, yd_carry=yd_carry, pos_range=pos_range),
                                     cols, run_off, [200], YO.empty_carry(1))
    assert np.array_equal(cut["yd"], whole["yd"])
    assert int(cut["yd"][-1]) == yd_c


def test_yd_carry_struct_matches_the_header_field_order():
    from tiebrush_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "tiebrush_b200.h")).read()
    body = hdr[:hdr.index("} tb_yd_carry;")]
    body = body[body.rindex("typedef struct {"):]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [n for n in re.findall(r"([A-Za-z_][A-Za-z0-9_]*)\s*(?:,|;)", body) if n not in ("typedef", "struct")]
    assert names == [f[0] for f in _lib.YdCarry._fields_]
    assert "tb_collapse_window_carry" in _lib.SYMBOLS
