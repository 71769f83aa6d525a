"""GPU checks of tb_collapse_window_carry: windows cut at start positions without a coverage gap, the YD lists carried
across the cuts, give the groups of one call and of the compiled reference; every carry_out equals the oracle's."""
import numpy as np
import pytest

import helpers as H
import yd_carry_oracle as YO
from test_yd_carry import carried_collapse, cut_positions, survey_9_4_case

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["par", "seq"])
def yd_path(request, monkeypatch):
    monkeypatch.setenv("TB_YD_PATH", request.param)
    return request.param


def gpu_carry_fn(k, opts):
    """compute() of one cut window on one context per (k, opts)."""
    from tiebrush_b200 import api
    ctxs = {}

    def fn(cols, run_off, tid=0, file_merged=None, yd_carry=None, pos_range=None, **o):
        key = tuple(sorted(o.items()))
        if key not in ctxs:
            ctxs[key] = api.Context(device=0, n_samples=k, **o)
        return ctxs[key].collapse_window(cols, run_off, tid=tid, file_merged=file_merged, pos_range=pos_range, yd_carry=yd_carry)
    return fn


@pytest.mark.parametrize("npz,pattern", [("collapse_random.npz", 7), ("collapse_fixture.npz", "random"), ("collapse_merged.npz", "every")])
def test_carry_goldens(npz, pattern, yd_path):
    carried = []
    for case in H.case_names(npz):
        files, opts, fm, exp = H.load_collapse_case(npz, case)
        got = H.run_collapse(carried_collapse(gpu_carry_fn(len(files), opts), pattern, len(files), carried), files, opts, fm)
        H.assert_collapse_equal(got, exp, f"{case} cut {pattern}")
    assert sum(carried) > 0


@pytest.mark.parametrize("name,which", [("t1", ["t1"]), ("t2", ["t2"]), ("t12", ["t1", "t2"])])
def test_carry_fixture_bams_against_reference_md5(name, which, yd_path):
    files, header, lines = H.fixture_inputs(which)
    got = H.run_collapse(carried_collapse(gpu_carry_fn(len(files), {}), 50, len(files)), files, {})
    assert (got["n_kept"], len(got["lhash"])) == H.REF_COUNTS[name]
    assert H.md5_text(H.collapsed_records(got, lines)) == H.REF_MD5[name]


def _recording(compute, log):
    def fn(sub, off, pos_range, yd_carry):
        r = compute(sub, off, pos_range=pos_range, yd_carry=yd_carry)
        log.append(r["yd_carry"])
        return {kk: (v.cpu().numpy() if hasattr(v, "cpu") else v) for kk, v in r.items()}
    return fn


def _assert_carries_equal(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        for key in ("tid", "pos_hi"):
            assert int(x[key]) == int(y[key]), (i, key)
        for key in ("chain_off", "seg_start", "seg_end"):
            assert np.array_equal(np.asarray(x[key]), np.asarray(y[key])), (i, key, x[key][:8], y[key][:8])


def _cut_and_compare(ctx, host, run_off, cuts, exp, opts, k):
    from oracle import oracle
    from tiebrush_b200 import api, shard
    glog, olog = [], []
    got = shard.collapse_cut_windows(_recording(lambda s, o, pos_range, yd_carry: ctx.collapse_window(s, o, pos_range=pos_range, yd_carry=yd_carry), glog),
                                     host, run_off, cuts, api.empty_yd_carry(k))
    ref = shard.collapse_cut_windows(_recording(lambda s, o, pos_range, yd_carry: YO.collapse(s, o, yd_carry=yd_carry, pos_range=pos_range, **opts), olog),
                                     host, run_off, cuts, YO.empty_carry(k))
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), np.asarray(exp[key])), key
        assert np.array_equal(np.asarray(ref[key]), np.asarray(exp[key])), key
    assert got["n_kept"] == exp["n_kept"]
    _assert_carries_equal(glog, olog)
    return got


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
@pytest.mark.parametrize("n_tx,k,reads", [(40, 12, 20000), (2000, 40, 5000), (3, 5, 30000), (150, 1000, 300)])
def test_carry_synthetic_vs_single_call_and_oracle(mode, n_tx, k, reads, yd_path):
    from oracle import oracle
    from tiebrush_b200 import api, shard, synth
    cols, run_off, pr = synth.cohort_window(k, reads, seed=3, n_tx=n_tx, device="cpu", with_md=(mode == 1))
    host = synth.to_host(cols)
    if mode == 1:
        host["md_off"], host["md"] = synth.md_columns(cols)
    exp = oracle.collapse(host, run_off, mode=mode)
    with api.Context(device=0, n_samples=k, mode=mode) as ctx:
        one = ctx.collapse_window(host, run_off)
        for key in ("rep_index", "yc", "yx", "yd"):
            assert np.array_equal(np.asarray(one[key]), exp[key]), key
        carried = 0
        for n in (2, 7):
            got = _cut_and_compare(ctx, host, run_off, shard.collapse_cuts(host, run_off, n), exp, dict(mode=mode), k)
            carried += sum(got["carried"][:-1])
        assert ctx.last_yd_path() == (0 if yd_path == "par" else 1)
    assert carried > 0


def test_carry_one_window_per_position(yd_path):
    from oracle import oracle
    from tiebrush_b200 import api, synth
    k = 6
    cols, run_off, pr = synth.cohort_window(k, 400, seed=8, n_tx=5, device="cpu")
    host = synth.to_host(cols)
    exp = oracle.collapse(host, run_off)
    with api.Context(device=0, n_samples=k) as ctx:
        got = _cut_and_compare(ctx, host, run_off, cut_positions(host, "every"), exp, {}, k)
    assert max(got["carried"]) > 0


def test_carry_crosses_yd_paths(monkeypatch):
    """A carry made on the sequential path and fed to the parallel one, and the reverse, gives the same groups."""
    from oracle import oracle
    from tiebrush_b200 import api, shard, synth
    k = 12
    cols, run_off, pr = synth.cohort_window(k, 20000, seed=13, n_tx=40, device="cpu")
    host = synth.to_host(cols)
    exp = oracle.collapse(host, run_off)
    cuts = shard.collapse_cuts(host, run_off, 6)
    for first in ("seq", "par"):
        state = dict(i=0)
        with api.Context(device=0, n_samples=k) as ctx:
            def fn(s, o, pos_range, yd_carry):
                monkeypatch.setenv("TB_YD_PATH", first if state["i"] % 2 == 0 else ("par" if first == "seq" else "seq"))
                state["i"] += 1
                return ctx.collapse_window(s, o, pos_range=pos_range, yd_carry=yd_carry)
            got = shard.collapse_cut_windows(fn, host, run_off, cuts, api.empty_yd_carry(k))
        for key in ("rep_index", "yc", "yx", "yd"):
            assert np.array_equal(got[key], exp[key]), (first, key)


@pytest.mark.parametrize("opts", [dict(flag_mask=16), dict(collapse_same=1), dict(keep_bits=8), dict(max_nh=2, min_qual=1, mode=3), dict(keep_bits=2 | 8, flag_mask=16)])
def test_carry_options(opts, yd_path):
    from oracle import oracle
    from tiebrush_b200 import api, shard, synth
    k = 7
    cols, run_off, pr = synth.cohort_window(k, 15000, seed=11, n_tx=25, device="cpu", paired=True)
    host = synth.to_host(cols)
    if opts.get("collapse_same"):   # -A: records 2i and 2i+1 share a read name
        host["qhash"] = (np.arange(len(host["pos"])) // 2).astype(np.uint64)
    exp = oracle.collapse(host, run_off, **opts)
    with api.Context(device=0, n_samples=k, **opts) as ctx:
        _cut_and_compare(ctx, host, run_off, shard.collapse_cuts(host, run_off, 7), exp, opts, k)


def _torch(a):
    import torch
    a = np.ascontiguousarray(a)
    sig = {np.dtype(np.uint32): np.int32, np.dtype(np.uint16): np.int16, np.dtype(np.uint64): np.int64}
    return torch.as_tensor(a.view(sig.get(a.dtype, a.dtype))).cuda()


@pytest.mark.parametrize("fmt", ["device", "packed", "packed_device"])
def test_carry_device_columns_and_packed_wire(fmt, yd_path):
    from oracle import oracle
    from tiebrush_b200 import api, shard, synth
    k = 12
    cols, run_off, pr = synth.cohort_window(k, 15000, seed=23, n_tx=200, device="cpu")
    host = synth.to_host(cols)
    exp = oracle.collapse(host, run_off)

    with api.Context(device=0, n_samples=k) as ctx:
        glog = []

        def one(s, o, pos_range, yd_carry):   # every cut window packed / moved to the device on its own
            d = {kk: s[kk] for kk in ("pos", "flag", "mapq", "strand", "nh", "cig_off", "cigar")}
            if fmt != "device":
                n8, c16, ext = api.compact_cigar_columns(d["cig_off"], d["cigar"])
                d = dict(api.pack_fixed_columns(d, o, max_dict=255), n_cigar8=n8, cigar16=c16, cigar_ext=ext)
            if fmt != "packed":
                d = {kk: (v if kk == "meta_dict" else _torch(v)) for kk, v in d.items()}
            r = ctx.collapse_window(d, o, pos_range=pos_range, yd_carry=yd_carry)
            glog.append(r["yd_carry"])
            return {kk: (v.cpu().numpy().view(np.uint32) if kk in ("rep_index", "yx") and hasattr(v, "cpu") else (v.cpu().numpy() if hasattr(v, "cpu") else v))
                    for kk, v in r.items()}
        got = shard.collapse_cut_windows(one, host, run_off, shard.collapse_cuts(host, run_off, 5), api.empty_yd_carry(k))
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), exp[key]), key
    assert sum(len(c["seg_start"]) for c in glog[:-1]) > 0


@pytest.mark.parametrize("with_a,yd_c", [(True, 0), (False, 5)])
def test_carry_survey_9_4_case(with_a, yd_c, yd_path):
    from tiebrush_b200 import api, shard
    cols, run_off = survey_9_4_case(with_a)
    with api.Context(device=0, n_samples=1) as ctx:
        whole = ctx.collapse_window(cols, run_off)
        cut = shard.collapse_cut_windows(lambda s, o, pos_range, yd_carry: ctx.collapse_window(s, o, pos_range=pos_range, yd_carry=yd_carry),
                                         cols, run_off, [200], api.empty_yd_carry(1))
    assert np.array_equal(cut["yd"], np.asarray(whole["yd"]))
    assert int(cut["yd"][-1]) == yd_c


def test_carry_is_what_makes_the_cut_exact(yd_path):
    """Some cuts carry non-empty lists, and the same cuts with an empty carry give a different YD on some group."""
    from tiebrush_b200 import api, shard, synth
    k = 6
    cols, run_off, _ = synth.cohort_window(k, 3000, seed=21, n_tx=4, device="cpu")
    host = synth.to_host(cols)
    cuts = cut_positions(host, 5)
    with api.Context(device=0, n_samples=k) as ctx:
        whole = ctx.collapse_window(host, run_off)
        ok = shard.collapse_cut_windows(lambda s, o, pos_range, yd_carry: ctx.collapse_window(s, o, pos_range=pos_range, yd_carry=yd_carry),
                                        host, run_off, cuts, api.empty_yd_carry(k))
        lost = shard.collapse_cut_windows(lambda s, o, pos_range, yd_carry: ctx.collapse_window(s, o, pos_range=pos_range, yd_carry=api.empty_yd_carry(k)),
                                          host, run_off, cuts, api.empty_yd_carry(k))
    assert max(ok["carried"]) > 0
    assert np.array_equal(ok["yd"], np.asarray(whole["yd"]))
    assert not np.array_equal(lost["yd"], np.asarray(whole["yd"]))


def test_carry_errors():
    """Every rule of tb_collapse_window_carry: non-zero return with a message, nothing written."""
    from tiebrush_b200 import api, synth
    k = 4
    cols, run_off, pr = synth.cohort_window(k, 2000, seed=2, n_tx=10, device="cpu")
    host = synth.to_host(cols)
    lo, hi = pr
    good = dict(tid=0, pos_hi=lo, chain_off=np.zeros(2 * k + 1, np.int64), seg_start=np.zeros(0, np.int32), seg_end=np.zeros(0, np.int32))

    def segs(s, e):
        c = dict(good)
        c["seg_start"], c["seg_end"] = np.asarray(s, np.int32), np.asarray(e, np.int32)
        c["chain_off"] = np.asarray([0] + [len(s)] * (2 * k), np.int64)
        return c
    bad = [(dict(good, pos_hi=lo + 1), "pos_lo"),
           (dict(good, chain_off=np.zeros(2 * k + 3, np.int64)), "n_chains"),
           (segs([lo + 5, lo + 1], [lo + 9, lo + 3]), "overlap or are unsorted"),
           (segs([lo + 1, lo + 5], [lo + 6, lo + 9]), "overlap or are unsorted"),
           (segs([lo + 9], [lo + 5]), "end < start")]
    with api.Context(device=0, n_samples=k) as ctx:
        for carry, msg in bad:
            with pytest.raises(api.TieBrushError, match=msg):
                ctx.collapse_window(host, run_off, pos_range=pr, yd_carry=carry)
        # touching segments are allowed; a different tid means the lists start empty
        ctx.collapse_window(host, run_off, pos_range=pr, yd_carry=segs([lo + 1, lo + 5], [lo + 4, lo + 9]))
        r = ctx.collapse_window(host, run_off, pos_range=pr, yd_carry=dict(segs([1], [2]), tid=5, pos_hi=hi + 10))
        assert r["yd_carry"]["tid"] == 0 and r["yd_carry"]["pos_hi"] == hi
    # a carry_out that is too small: the call reports the segments it needs and writes no carry
    import ctypes as C
    from tiebrush_b200 import _lib
    lib = _lib.load()
    with api.Context(device=0, n_samples=k) as ctx:
        from tiebrush_b200 import sam, shard
        sub_hi = int(np.median(host["pos"]))
        idx, off = shard._file_slices(host, run_off, lo, sub_hi)
        sub = sam.take(host, idx)
        need = len(ctx.collapse_window(sub, off, pos_range=(lo, sub_hi), yd_carry=api.empty_yd_carry(k))["yd_carry"]["seg_start"])
        assert need > 0
        keep = [np.ascontiguousarray(sub[kk], dt) for kk, dt in (("pos", np.int32), ("flag", np.uint16), ("mapq", np.uint8), ("strand", np.uint8),
                                                                  ("nh", np.uint16), ("cig_off", np.uint32), ("cigar", np.uint32))]
        ro = np.asarray(off, np.int64)
        p = lambda a: a.ctypes.data
        n = len(keep[0])
        sin = _lib.SoaIn(n, k, 0, p(ro), None, p(keep[0]), p(keep[1]), p(keep[2]), p(keep[3]), p(keep[4]), p(keep[5]), p(keep[6]),
                         None, None, None, None, None, None, 0, int(keep[5][-1]), 0, lo, sub_hi)
        outs = [np.zeros(n, np.uint32), np.zeros(n, np.float32), np.zeros(n, np.uint32), np.zeros(n, np.int32)]
        o = _lib.GroupsOut(n, 0, 0, *[p(a) for a in outs], 0)
        co, cs, ce = np.full(2 * k + 1, -7, np.int64), np.zeros(1, np.int32), np.zeros(1, np.int32)
        cout = _lib.YdCarry(0, 0, 2 * k, 0, 0, p(co), p(cs), p(ce))
        assert lib.tb_collapse_window_carry(ctx.h, C.byref(sin), None, C.byref(o), C.byref(cout)) != 0
        assert "capacity" in ctx._err() and int(cout.n_segs) == need and (co == -7).all()
        cout.n_chains = 2 * k + 2
        assert lib.tb_collapse_window_carry(ctx.h, C.byref(sin), None, C.byref(o), C.byref(cout)) != 0
        assert "n_chains" in ctx._err()
