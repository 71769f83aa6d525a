"""GPU parity tests (through the C ABI): tiecov coverage / junction / bedgraph kernels vs the oracle and
vs golden outputs of the compiled reference."""
import os

import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from tiebrush_b200 import api
    with api.Context(device=0) as c:
        yield c


@pytest.mark.parametrize("case", H.coverage_case_names())
def test_coverage_golden(ctx, case):
    cols, runs, juncs = H.load_coverage_case(case)
    got = ctx.coverage_window(cols)
    H.assert_coverage_equal(got, runs, juncs, case)


@pytest.mark.parametrize("case", H.coverage_case_names()[:4])
def test_coverage_matches_oracle_exactly(ctx, case):
    from oracle import oracle
    cols, _, _ = H.load_coverage_case(case)
    got, exp = ctx.coverage_window(cols), oracle.coverage(cols)
    for a, b in zip(got["runs"], exp["runs"]):
        assert np.array_equal(a, b)
    for a, b in zip(got["juncs"], exp["juncs"]):
        assert np.array_equal(a, b)


def test_coverage_only_runs_or_only_juncs(ctx):
    cols, runs, juncs = H.load_coverage_case(H.coverage_case_names()[0])
    r = ctx.coverage_window(cols, want_juncs=False)
    assert r["n_runs"] == len(runs[0]) and r["n_juncs"] == 0
    j = ctx.coverage_window(cols, want_runs=False)
    assert j["n_juncs"] == len(juncs[0]) and j["n_runs"] == 0


def test_coverage_rejects_unsupported_ops(ctx):
    cols = dict(tid=np.zeros(2, np.int32), pos=np.asarray([10, 12], np.int32), yc=np.ones(2, np.float32),
                strand=np.asarray([ord(".")] * 2, np.uint8), cig_off=np.asarray([0, 1, 2], np.uint32),
                cigar=np.asarray([(5 << 4) | 0, (5 << 4) | 7], np.uint32))
    with pytest.raises(ValueError):
        ctx.coverage_window(cols)
    # junction-only runs never look at the ops (addCov is not called, tiecov.cpp:486-488)
    assert ctx.coverage_window(cols, want_runs=False)["n_juncs"] == 0


def test_coverage_empty(ctx):
    cols = dict(tid=np.zeros(0, np.int32), pos=np.zeros(0, np.int32), yc=np.zeros(0, np.float32), strand=np.zeros(0, np.uint8),
                cig_off=np.zeros(1, np.uint32), cigar=np.zeros(0, np.uint32))
    r = ctx.coverage_window(cols)
    assert r["n_runs"] == 0 and r["n_juncs"] == 0


def test_coverage_device_resident_large_random(ctx):
    """Size-independent properties on a large synthetic stream kept in HBM: total covered weight is conserved,
    runs are sorted, disjoint, never zero, and adjacent equal-valued runs only meet at bundle edges."""
    import torch
    from tiebrush_b200 import synth
    cols = synth.coverage_stream(n=2_000_000, seed=7, device="cuda")
    out = ctx.coverage_window(cols)
    t, s, e, v = (x.cpu().numpy() for x in out["runs"])
    assert len(t) > 0 and (v != 0).all() and (e > s).all()
    same = t[1:] == t[:-1]
    assert (s[1:][same] >= e[:-1][same]).all()
    total = float(((e - s).astype(np.float64) * v).sum())
    assert total == synth.covered_weight(cols)
    # against the oracle on a prefix that the CPU finishes quickly (cut at a bundle boundary)
    from oracle import oracle
    host = synth.to_host(cols)
    cut = synth.bundle_cut(host, 200_000)
    sub = synth.take_prefix(host, cut)
    exp = oracle.coverage(sub)
    got = ctx.coverage_window(sub)
    for a, b in zip(got["runs"], exp["runs"]):
        assert np.array_equal(np.asarray(a), b)
    for a, b in zip(got["juncs"], exp["juncs"]):
        assert np.array_equal(np.asarray(a), b)


def test_coverage_c4_scale_properties_and_oracle_prefix():
    """BASELINE C4 shape: a whole-genome (24 chromosomes) collapsed stream resident in HBM, 2e8 records in one window
    (TB_TEST_FULL=0: 2e7). Size-independent properties over the whole output — the covered weight sum(YC x M bases) is
    conserved by the runs, runs are sorted / disjoint / non-zero, junction rows are sorted and positive — and bit-exact
    equality with the oracle on a whole-bundle prefix of the same stream."""
    import os
    import torch
    from oracle import oracle
    from tiebrush_b200 import api, synth
    n = 20_000_000 if os.environ.get("TB_TEST_FULL") == "0" else 200_000_000
    cols = synth.coverage_stream(n, seed=3, chroms=24, device="cuda")
    with api.Context(device=0, n_samples=1) as c4:
        out = c4.coverage_window(cols)
        t, s, e, v = out["runs"]
        assert out["n_runs"] > 1000 and bool((v != 0).all()) and bool((e > s).all())
        same = t[1:] == t[:-1]
        assert bool((t[1:] >= t[:-1]).all()) and bool((s[1:][same] >= e[:-1][same]).all())
        total = float(((e - s).to(torch.float64) * v).sum().item())
        # covered weight on the device: per-record M bases (segment sum over the CIGAR arena) x YC
        cig = cols["cigar"].to(torch.int64) & 0xFFFFFFFF
        mlen = (cig >> 4) * ((cig & 0xF) == 0)
        cs = torch.zeros(mlen.numel() + 1, dtype=torch.int64, device="cuda"); cs[1:] = torch.cumsum(mlen, 0)
        off = cols["cig_off"].to(torch.int64) & 0xFFFFFFFF
        per_rec = cs[off[1:]] - cs[off[:-1]]
        assert total == float((per_rec.to(torch.float64) * cols["yc"].to(torch.float64)).sum().item())
        jt, js, je, jstrand, jv = out["juncs"]
        assert out["n_juncs"] > 100 and bool((jv > 0).all()) and bool((je >= js).all())
        sj = jt[1:] == jt[:-1]
        assert bool((jt[1:] >= jt[:-1]).all()) and bool((js[1:][sj] >= js[:-1][sj]).all())
        # oracle on a whole-bundle prefix (first bundle boundary after 200k records)
        H = 4_000_000
        head = {k: cols[k][:H].cpu() for k in ("tid", "pos", "yc", "strand")}
        head["cig_off"] = cols["cig_off"][:H + 1].cpu(); head["cigar"] = cols["cigar"][: int(off[H].item())].cpu()
        host = synth.to_host(head)
        cut = synth.bundle_cut(host, 200_000)
        assert cut < H
        sub = synth.take_prefix(host, cut)
        exp = oracle.coverage(sub)
        nr, nj = len(exp["runs"][0]), len(exp["juncs"][0])
        for a, b in zip(out["runs"], exp["runs"]):
            assert np.array_equal(a[:nr].cpu().numpy(), b)
        # junction rows of the prefix: same (tid,start,end,strand,value) multiset restricted to the prefix's coordinates
        got = c4.coverage_window(sub)
        for a, b in zip(got["juncs"], exp["juncs"]):
            assert np.array_equal(np.asarray(a), b)
        assert nj > 0


def test_coverage_unaligned_columns_take_the_scalar_path(ctx):
    """The bundle kernels' 128-bit loads need 16-byte aligned columns. Device columns of a window cut at an arbitrary record
    offset are not aligned: here every column starts one element past an aligned buffer, and the result must still equal
    the oracle, once without the end column (look-back K6) and once with it (the three streaming passes)."""
    import torch
    from oracle import oracle
    from tiebrush_b200 import synth
    cols = synth.coverage_stream(60_001, seed=21, n_tx=40, chroms=3, device="cuda")
    cols["end"] = synth.end_column(cols)
    exp = oracle.coverage(synth.to_host(cols))

    def unaligned(a):   # 4 bytes (strand: 1 byte) past the buffer's aligned start
        buf = torch.empty(a.numel() + 1, dtype=a.dtype, device=a.device)
        buf[1:] = a
        return buf[1:]
    for with_end in (False, True):
        moved = ("tid", "pos", "yc", "strand", "cig_off") + (("end",) if with_end else ())
        win = {k: v for k, v in cols.items() if k != "end"}
        win.update({k: unaligned(cols[k]) for k in moved})
        assert all(win[k].data_ptr() % 16 != 0 for k in moved)
        got = ctx.coverage_window(win)
        for a, b in zip(got["runs"] + got["juncs"], exp["runs"] + exp["juncs"]):
            assert np.array_equal(a.cpu().numpy(), b)


@pytest.mark.parametrize("case", ["t1", "t2"])
def test_sample_heatmap_golden(ctx, case):
    """tiecov -s on the device against the reference's own fixtures (columns 1-4 of test/t{1,2}/t{1,2}.sample.bedgraph)."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sample_heatmap.npz"))
    cols = {k: z[f"{case}/in/{k}"] for k in ("tid", "pos", "cig_off", "cigar")}
    n = len(cols["pos"])
    cols.update(yx=z[f"{case}/in/yx_in"], yc=np.ones(n, np.float32), strand=np.full(n, ord("."), np.uint8))
    t, s, e, iv = ctx.sample_window(cols)
    assert np.array_equal(t, z[f"{case}/out/tid"]) and np.array_equal(s, z[f"{case}/out/start"])
    assert np.array_equal(e, z[f"{case}/out/end"]) and np.array_equal(iv, z[f"{case}/out/ival"])


@pytest.mark.parametrize("n,n_tx,chroms,seed", [(40_000, 30, 2, 1), (120_000, 400, 3, 2), (30_000, 3, 1, 3)])
def test_sample_heatmap_matches_oracle(ctx, n, n_tx, chroms, seed):
    """tiecov -s: float32 running mean of YX per base in stream order, ceil, runs — device against the oracle, bit for bit
    (spliced reads, deep pile-ups, several chromosomes, YX from 1 to 60)."""
    from oracle import oracle
    from tiebrush_b200 import synth
    cols = synth.to_host(synth.coverage_stream(n, seed=seed, n_tx=n_tx, chroms=chroms))
    cols["yx"] = np.random.default_rng(seed).integers(1, 61, size=n).astype(np.int32)
    got, exp = ctx.sample_window(cols), oracle.sample_heatmap(cols)
    assert len(exp[0]) > 100
    for a, b in zip(got, exp):
        assert np.array_equal(np.asarray(a), b)


# ---- long streams: windows cut at bundle heads (tc_coverage_stream) -------------------------------------------------
def _same_rows(a, b):
    assert a["n_runs"] == b["n_runs"] and a["n_juncs"] == b["n_juncs"]
    for x, y in zip(a["runs"] + a["juncs"], b["runs"] + b["juncs"]):
        x = x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)
        y = y.cpu().numpy() if hasattr(y, "cpu") else np.asarray(y)
        assert np.array_equal(x, y)


@pytest.mark.parametrize("window", [1024, 5000, 70000])
@pytest.mark.parametrize("where", ["host", "device"])
def test_coverage_stream_equals_one_window(ctx, window, where):
    """The stream cut into small windows at bundle heads gives the rows of one window (= the oracle), host and device arrays."""
    import torch
    from oracle import oracle
    from tiebrush_b200 import api, synth
    cols = synth.coverage_stream(60000, seed=4, n_tx=60, chroms=3, device="cuda" if where == "device" else "cpu")
    host = synth.to_host(cols)
    exp = oracle.coverage(host)
    src = cols if where == "device" else host
    cap = 2 * int(host["cig_off"][-1]) + 16
    out = api.cov_out_buffers(cap, cap, device="cuda" if where == "device" else None)
    got = ctx.coverage_stream(src, window, out)
    assert got["consumed"] == len(host["pos"]) and (got["windows"] >= 5 if window < 20000 else got["windows"] >= 1)
    _same_rows(got, dict(runs=exp["runs"], juncs=exp["juncs"], n_runs=len(exp["runs"][0]), n_juncs=len(exp["juncs"][0])))


def test_coverage_stream_leaves_the_open_bundle(ctx):
    """A slice that ends inside a bundle: with the following record given, that bundle is left to the caller."""
    from oracle import oracle
    from tiebrush_b200 import api, synth
    host = synth.to_host(synth.coverage_stream(30000, seed=6, n_tx=20, chroms=1))
    n = len(host["pos"])
    cut = n // 2
    while synth.bundle_cut(host, cut) == cut:     # move the cut inside a bundle
        cut += 1
    part = synth.take_prefix(host, cut)
    cap = 2 * int(host["cig_off"][-1]) + 16
    got = ctx.coverage_stream(part, 4096, api.cov_out_buffers(cap, cap), next_tid_pos=(host["tid"][cut], host["pos"][cut]))
    prev_head = got["consumed"]
    assert prev_head < cut and synth.bundle_cut(host, prev_head) == prev_head and synth.bundle_cut(host, prev_head + 1) > cut
    exp = oracle.coverage(synth.take_prefix(host, prev_head))
    _same_rows(got, dict(runs=exp["runs"], juncs=exp["juncs"], n_runs=len(exp["runs"][0]), n_juncs=len(exp["juncs"][0])))


# ---- weights that are not multiples of 2^-20 (tiebrush --store-frac): exact ordered double sums -------------------------
@pytest.mark.parametrize("with_end", [False, True], ids=["no_end", "end"])
@pytest.mark.parametrize("seed", [1, 2])
def test_coverage_fractional_yc_takes_the_exact_path(ctx, seed, with_end):
    """YC = 1/3, 1/5, 1/7 ... (float32): fixed point would round every weight; the device sums doubles in stream order like
    the reference (tiecov.cpp:194-223, :100-112) and says so. With the end column K6 first runs its three streaming passes,
    then the look-back pass for the running maximum of the ends that the exact junction walk needs."""
    from oracle import oracle
    from tiebrush_b200 import synth
    cols = synth.coverage_stream(40000, seed=seed, n_tx=25, chroms=2)
    if with_end:
        cols["end"] = synth.end_column(cols)
    host = synth.to_host(cols)
    rng = np.random.default_rng(seed)
    host["yc"] = (rng.integers(1, 40, len(host["pos"])).astype(np.float32) / rng.choice(np.asarray([3, 5, 7, 9, 11], np.float32), len(host["pos"]))).astype(np.float32)
    got, exp = ctx.coverage_window(host), oracle.coverage(host)
    assert ctx.last_cov_exact() == 1
    for a, b in zip(got["runs"] + got["juncs"], exp["runs"] + exp["juncs"]):
        assert np.array_equal(np.asarray(a), b)
    host["yc"] = np.ones_like(host["yc"])
    ctx.coverage_window(host)
    assert ctx.last_cov_exact() == 0


# ---- the optional `end` column (GSamRecord::end from the host packer): K6 never walks a CIGAR ------------------------------
@pytest.mark.parametrize("where", ["host", "device"])
def test_coverage_with_end_column_equals_without(ctx, where):
    import torch
    from oracle import oracle
    from tiebrush_b200 import api, synth
    cols = synth.coverage_stream(50000, seed=8, n_tx=40, chroms=3, device="cuda" if where == "device" else "cpu")
    cols["end"] = synth.end_column(cols)
    host = synth.to_host(cols)
    exp = oracle.coverage(host)
    src = cols if where == "device" else host
    got = ctx.coverage_window(src)
    for a, b in zip(got["runs"] + got["juncs"], exp["runs"] + exp["juncs"]):
        assert np.array_equal(a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a), b)
    cap = 2 * int(host["cig_off"][-1]) + 16
    st = ctx.coverage_stream(src, 3000, api.cov_out_buffers(cap, cap, device="cuda" if where == "device" else None))
    _same_rows(st, dict(runs=exp["runs"], juncs=exp["juncs"], n_runs=len(exp["runs"][0]), n_juncs=len(exp["juncs"][0])))


def test_coverage_with_end_column_still_rejects_unsupported_ops(ctx):
    cols = dict(tid=np.zeros(2, np.int32), pos=np.asarray([10, 12], np.int32), yc=np.ones(2, np.float32),
                strand=np.asarray([ord(".")] * 2, np.uint8), cig_off=np.asarray([0, 1, 2], np.uint32),
                cigar=np.asarray([(5 << 4) | 0, (5 << 4) | 7], np.uint32), end=np.asarray([15, 17], np.int32))
    with pytest.raises(ValueError):
        ctx.coverage_window(cols)
    assert ctx.coverage_window(cols, want_runs=False)["n_juncs"] == 0
