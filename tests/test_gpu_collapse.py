"""GPU parity tests (through the C ABI): merge + collapse kernels vs golden outputs of the compiled reference
and vs the oracle on seeded synthetic cohorts."""
import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu


def gpu_collapse(cols, run_off, tid=0, file_merged=None, **opts):
    from tiebrush_b200 import api
    k = len(run_off) - 1
    with api.Context(device=0, n_samples=k, **opts) as ctx:
        return ctx.collapse_window(cols, run_off, tid=tid, file_merged=file_merged)


@pytest.mark.parametrize("case", H.case_names("collapse_random.npz"))
def test_collapse_random(case):
    files, opts, fm, exp = H.load_collapse_case("collapse_random.npz", case)
    H.assert_collapse_equal(H.run_collapse(gpu_collapse, files, opts, fm), exp, case)


@pytest.mark.parametrize("case", H.case_names("collapse_fixture.npz"))
def test_collapse_fixture(case):
    files, opts, fm, exp = H.load_collapse_case("collapse_fixture.npz", case)
    H.assert_collapse_equal(H.run_collapse(gpu_collapse, files, opts, fm), exp, case)


@pytest.mark.parametrize("case", H.case_names("collapse_merged.npz"))
def test_collapse_merged(case):
    files, opts, fm, exp = H.load_collapse_case("collapse_merged.npz", case)
    H.assert_collapse_equal(H.run_collapse(gpu_collapse, files, opts, fm), exp, case)


@pytest.mark.parametrize("name,which", [("t1", ["t1"]), ("t2", ["t2"]), ("t12", ["t1", "t2"])])
def test_fixture_bams_against_reference_md5(name, which):
    """The reference's own sample BAMs (tests/golden/fixtures) through the GPU collapse: the records tiebrush would write
    from its groups have the md5 of the compiled reference's output; for t1+t2 also the bytes of tiecov -c -j on them."""
    from tiebrush_b200 import api
    files, header, lines = H.fixture_inputs(which)
    got = H.run_collapse(gpu_collapse, files, {})
    assert (got["n_kept"], len(got["lhash"])) == H.REF_COUNTS[name]
    records = H.collapsed_records(got, lines)
    assert H.md5_text(records) == H.REF_MD5[name]
    if name == "t12":
        import hashlib
        cols, names = H.coverage_input(header, records)
        with api.Context(device=0) as ctx:
            bg, bed = H.coverage_files(ctx.coverage_window(cols), names)
        assert hashlib.md5(bg.encode()).hexdigest() == H.REF_MD5["cov"]
        assert hashlib.md5(bed.encode()).hexdigest() == H.REF_MD5["junc"]


@pytest.fixture(params=["par", "seq"])
def yd_path(request, monkeypatch):
    """Both YD implementations: the parallel formulation (frontier + link bitmaps) and the sequential segment lists."""
    monkeypatch.setenv("TB_YD_PATH", request.param)
    return request.param


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
@pytest.mark.parametrize("n_tx,k,reads", [(40, 12, 20000), (2000, 40, 5000), (3, 5, 30000), (150, 1000, 300), (300, 100, 3000)])
def test_collapse_synthetic_vs_oracle(mode, n_tx, k, reads, yd_path):
    """Seeded synthetic cohorts (deep pile-ups when n_tx is tiny) against the oracle, bit for bit, in every merge strategy.
    No start position holds more distinct alignments than the full-size table, so every window stays on the tile path."""
    from oracle import oracle
    from tiebrush_b200 import api, synth
    cols, run_off, pr = synth.cohort_window(k, reads, seed=3, n_tx=n_tx, device="cpu", with_md=(mode == 1))
    host = synth.to_host(cols)
    if mode == 1:
        host["md_off"], host["md"] = synth.md_columns(cols)
    with api.Context(device=0, n_samples=k, mode=mode) as ctx:
        got = ctx.collapse_window(host, run_off)
        assert ctx.last_path() == 0 and ctx.last_tile_gen() == 1
        assert ctx.last_yd_path() == (0 if yd_path == "par" else 1)
    exp = oracle.collapse(host, run_off, mode=mode)
    assert got["n_kept"] == exp["n_kept"]
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), exp[key]), key


def test_collapse_full_mode_synthetic_vs_oracle():
    """-L (CIGAR + MD) on a synthetic cohort with MD strings."""
    from oracle import oracle
    from tiebrush_b200 import synth
    cols, run_off, pr = synth.cohort_window(10, 20000, seed=9, n_tx=30, device="cpu", with_md=True)
    host = synth.to_host(cols)
    host["md_off"], host["md"] = synth.md_columns(cols)
    got = gpu_collapse(host, run_off, mode=1)
    exp = oracle.collapse(host, run_off, mode=1)
    assert got["n_kept"] == exp["n_kept"]
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), exp[key]), key


@pytest.mark.parametrize("opts", [dict(max_nh=1), dict(min_qual=30), dict(max_nh=3, min_qual=1, mode=3), dict(flag_mask=16),
                                  dict(flag_mask=16, mode=3, max_nh=2), dict(keep_bits=2 | 8)])
def test_collapse_filters_and_ordered_path_synthetic_vs_oracle(opts):
    """-N/-Q filters on the tile path; -F and --store-frac on the ordered path (exact list emulation), paired flags."""
    from oracle import oracle
    from tiebrush_b200 import api, synth
    k = 7
    cols, run_off, pr = synth.cohort_window(k, 15000, seed=11, n_tx=25, device="cpu", paired=True)
    host = synth.to_host(cols)
    with api.Context(device=0, n_samples=k, **opts) as ctx:
        got = ctx.collapse_window(host, run_off)
        assert ctx.last_path() == (1 if ("flag_mask" in opts or opts.get("keep_bits", 0) & 8) else 0)
    exp = oracle.collapse(host, run_off, **opts)
    assert got["n_kept"] == exp["n_kept"]
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), exp[key]), key


def test_collapse_table_overflow_falls_back_to_ordered_path():
    """One start position with more distinct alignments than a shared-memory table holds: the window is redone by the
    exact path and still matches the oracle."""
    from oracle import oracle
    from tiebrush_b200 import api
    rng = np.random.default_rng(5)
    k, per = 3, 4000
    n = k * per
    a = rng.integers(1, 400, n); b = rng.integers(1, 400, n)
    cigar = np.stack([(a << 4) | 0, np.full(n, (1 << 4) | 1), (b << 4) | 0], 1).astype(np.uint32).reshape(-1)
    pos = np.full(n, 1000, np.int32)
    pos[:: 7] = 990  # a second, ordinary position in front
    order = np.concatenate([f * per + np.argsort(pos[f * per:(f + 1) * per], kind="stable") for f in range(k)])
    cols = dict(pos=pos[order], flag=np.zeros(n, np.uint16), mapq=np.full(n, 60, np.uint8), strand=np.full(n, ord("+"), np.uint8),
                nh=np.ones(n, np.uint16), cig_off=(np.arange(n + 1) * 3).astype(np.uint32), cigar=cigar.reshape(n, 3)[order].reshape(-1))
    run_off = np.arange(k + 1, dtype=np.int64) * per
    with api.Context(device=0, n_samples=k) as ctx:
        got = ctx.collapse_window(cols, run_off)
        assert ctx.last_path() == 2
    exp = oracle.collapse(cols, run_off)
    assert got["n_groups"] == len(exp["rep_index"]) > 8000
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), exp[key]), key


def test_collapse_heavy_position_uses_full_size_table():
    """A pile-up position with more distinct alignments than a quarter-SM table holds (but fewer than a full-SM one) is
    redone by the second tile launch and stays on the tile path."""
    from oracle import oracle
    from tiebrush_b200 import api
    rng = np.random.default_rng(15)
    k, per = 3, 6000
    n = k * per
    a = rng.integers(1, 60, n); b = rng.integers(1, 60, n)     # ~3400 distinct (a,b) pairs at the pile-up position
    cigar = np.stack([(a << 4) | 0, np.full(n, (1 << 4) | 2), (b << 4) | 0], 1).astype(np.uint32)
    pos = np.where(rng.random(n) < 0.95, 7000, rng.integers(6000, 8000, n)).astype(np.int32)
    order = np.concatenate([f * per + np.argsort(pos[f * per:(f + 1) * per], kind="stable") for f in range(k)])
    cols = dict(pos=pos[order], flag=np.zeros(n, np.uint16), mapq=np.full(n, 60, np.uint8), strand=np.full(n, ord("-"), np.uint8),
                nh=np.ones(n, np.uint16), cig_off=(np.arange(n + 1) * 3).astype(np.uint32), cigar=cigar[order].reshape(-1))
    run_off = np.arange(k + 1, dtype=np.int64) * per
    with api.Context(device=0, n_samples=k) as ctx:
        got = ctx.collapse_window(cols, run_off)
        assert ctx.last_path() == 0 and ctx.last_heavy_slots() >= 1
    exp = oracle.collapse(cols, run_off)
    assert got["n_groups"] == len(exp["rep_index"]) > 3000
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), exp[key]), key


def test_collapse_pileup_position_single_mode():
    """A pile-up position (more records than a tile) with few distinct alignments stays on the tile path."""
    from oracle import oracle
    from tiebrush_b200 import api
    rng = np.random.default_rng(6)
    k, per = 5, 6000
    n = k * per
    a = rng.integers(40, 60, n)
    cigar = np.stack([(a << 4) | 0, np.full(n, (300 << 4) | 3), ((150 - a) << 4) | 0], 1).astype(np.uint32)
    pos = np.where(rng.random(n) < 0.9, 5000, rng.integers(4000, 6000, n)).astype(np.int32)
    order = np.concatenate([f * per + np.argsort(pos[f * per:(f + 1) * per], kind="stable") for f in range(k)])
    cols = dict(pos=pos[order], flag=np.zeros(n, np.uint16), mapq=np.full(n, 60, np.uint8),
                strand=rng.choice(np.frombuffer(b"+-.", np.uint8), n), nh=np.ones(n, np.uint16),
                cig_off=(np.arange(n + 1) * 3).astype(np.uint32), cigar=cigar[order].reshape(-1))
    run_off = np.arange(k + 1, dtype=np.int64) * per
    with api.Context(device=0, n_samples=k) as ctx:
        got = ctx.collapse_window(cols, run_off)
        assert ctx.last_path() == 0
    exp = oracle.collapse(cols, run_off)
    assert got["n_kept"] == exp["n_kept"]
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), exp[key]), key


def test_yd_many_exons_and_degenerate_exons():
    """Representatives with more than three exons (decoded from the CIGAR by the YD kernels) stay on the parallel YD
    path; a degenerate exon (N directly followed by N, GSam.cpp:376-388) sends the window to the sequential lists."""
    from oracle import oracle
    from tiebrush_b200 import api
    rng = np.random.default_rng(8)
    k, per = 4, 3000
    n = k * per

    def make(degenerate):
        cigs, pos = [], []
        for i in range(n):
            nb = int(rng.integers(1, 7))
            words = []
            for b in range(nb):
                words.append((int(rng.integers(5, 40)) << 4) | 0)
                if b < nb - 1:
                    words.append((int(rng.choice([1, 30, 80, 200])) << 4) | 3)
                    if degenerate and rng.random() < 0.02:
                        words.append((int(rng.integers(1, 9)) << 4) | 3)
            cigs.append(words); pos.append(int(rng.integers(1000, 3000)))
        pos = np.asarray(pos, np.int32)
        order = np.concatenate([f * per + np.argsort(pos[f * per:(f + 1) * per], kind="stable") for f in range(k)])
        off = np.zeros(n + 1, np.uint32); off[1:] = np.cumsum([len(cigs[i]) for i in order])
        cigar = np.asarray([w for i in order for w in cigs[i]], np.uint32)
        return dict(pos=pos[order], flag=np.zeros(n, np.uint16), mapq=np.full(n, 60, np.uint8),
                    strand=rng.choice(np.frombuffer(b"+-.", np.uint8), n), nh=np.ones(n, np.uint16), cig_off=off, cigar=cigar)

    run_off = np.arange(k + 1, dtype=np.int64) * per
    for degenerate in (False, True):
        cols = make(degenerate)
        with api.Context(device=0, n_samples=k) as ctx:
            got = ctx.collapse_window(cols, run_off)
            assert ctx.last_yd_path() == (1 if degenerate else 0)
        exp = oracle.collapse(cols, run_off)
        for key in ("rep_index", "yc", "yx", "yd"):
            assert np.array_equal(np.asarray(got[key]), exp[key]), (degenerate, key)


def test_collapse_device_resident_properties():
    """BASELINE-shaped cohort kept in HBM: size-independent properties (sum YC == records kept, reps are
    members with the right position order, YX <= min(k, YC)) plus oracle equality on the host copy."""
    import torch
    from oracle import oracle
    from tiebrush_b200 import api, synth
    k, reads = 50, 40000
    cols, run_off, pr = synth.cohort_window(k, reads, seed=5, n_tx=500, device="cuda")
    with api.Context(device=0, n_samples=k) as ctx:
        got = ctx.collapse_window(cols, run_off, pos_range=pr)
    rep = got["rep_index"].cpu().numpy().view(np.uint32); yc = got["yc"].cpu().numpy(); yx = got["yx"].cpu().numpy().view(np.uint32)
    assert got["n_kept"] == k * reads and float(yc.sum()) == k * reads
    pos = cols["pos"].cpu().numpy()
    assert (np.diff(pos[rep]) >= 0).all()
    assert (yx <= np.minimum(k, yc)).all() and (yx >= 1).all()
    host = synth.to_host(cols)
    exp = oracle.collapse(host, run_off)
    assert np.array_equal(rep, exp["rep_index"]) and np.array_equal(yc, exp["yc"]) and np.array_equal(yx, exp["yx"])
    assert np.array_equal(got["yd"].cpu().numpy(), exp["yd"])


def _device_prefix_slice(cols, run_off, hi):
    """Records of every file with pos < hi (a coordinate prefix of the window), gathered on the device, returned as host columns."""
    import torch
    dev = cols["pos"].device
    parts, new_off = [], [0]
    for f in range(len(run_off) - 1):
        a, b = int(run_off[f]), int(run_off[f + 1])
        c = a + int(torch.searchsorted(cols["pos"][a:b], torch.tensor([hi], device=dev, dtype=cols["pos"].dtype))[0])
        parts.append(torch.arange(a, c, device=dev))
        new_off.append(new_off[-1] + (c - a))
    idx = torch.cat(parts)
    sub = {k: cols[k][idx].cpu().numpy() for k in ("pos", "flag", "mapq", "strand", "nh")}
    sub["flag"] = sub["flag"].view(np.uint16); sub["nh"] = sub["nh"].view(np.uint16)
    c0 = cols["cig_off"][idx].long() & 0xffffffff
    ln = (cols["cig_off"][idx + 1].long() & 0xffffffff) - c0
    off = torch.zeros(len(idx) + 1, dtype=torch.long, device=dev); off[1:] = torch.cumsum(ln, 0)
    rep = torch.repeat_interleave(torch.arange(len(idx), device=dev), ln)
    src = c0[rep] + (torch.arange(int(off[-1]), device=dev) - off[:-1][rep])
    sub["cigar"] = cols["cigar"][src].cpu().numpy().view(np.uint32)
    sub["cig_off"] = off.cpu().numpy().astype(np.uint32)
    return sub, np.asarray(new_off, np.int64), idx


def test_collapse_baseline_size_properties_and_oracle_prefix():
    """BASELINE C2 shape (100 samples on chr1, default mode) resident in HBM at the FULL configured size, 100 x 10M reads =
    1e9 alignments (about 11 s on a B200; TB_TEST_FULL=0 shrinks it to 100 x 2M). Size-independent properties over the whole output (sum YC == records, YX bounds,
    representatives in position order and inside their own position, YD >= 0) and bit-exact equality with the oracle
    on a coordinate prefix of the same window (a prefix needs no state from the rest: groups and YD only look left)."""
    import os
    import torch
    from oracle import oracle
    from tiebrush_b200 import api, synth
    k = 100
    reads = 2_000_000 if os.environ.get("TB_TEST_FULL") == "0" else 10_000_000
    cols, run_off, pr = synth.cohort_window(k, reads, seed=0, device="cuda")
    n = k * reads
    out = dict(rep_index=torch.empty(n, dtype=torch.int32, device="cuda"), yc=torch.empty(n, dtype=torch.float32, device="cuda"),
               yx=torch.empty(n, dtype=torch.int32, device="cuda"), yd=torch.empty(n, dtype=torch.int32, device="cuda"))
    with api.Context(device=0, n_samples=k) as ctx:
        got = ctx.collapse_window(cols, run_off, pos_range=pr, out=out)
        assert ctx.last_path() == 0 and ctx.last_yd_path() == 0
    G = got["n_groups"]
    rep = out["rep_index"][:G].long() & 0xffffffff
    yc, yx, yd = out["yc"][:G], out["yx"][:G], out["yd"][:G]
    assert got["n_kept"] == n
    assert int(yc.to(torch.float64).sum().item()) == n
    assert bool((yx >= 1).all()) and bool((yx.to(torch.float32) <= torch.clamp(yc, max=float(k))).all()) and bool((yd >= 0).all())
    rpos = cols["pos"][rep]
    assert bool((rpos[1:] >= rpos[:-1]).all())
    # oracle on a prefix of ~2M records
    first = cols["pos"][: reads]
    hi = int(first[min(reads - 1, max(1, (2_000_000 // k)))].item())
    sub, sub_off, idx = _device_prefix_slice(cols, run_off, hi)
    exp = oracle.collapse(sub, sub_off)
    Gs = len(exp["rep_index"])
    assert Gs > 1000 and bool((rpos[:Gs] < hi).all()) and (G == Gs or int(rpos[Gs].item()) >= hi)
    assert np.array_equal(idx[torch.as_tensor(exp["rep_index"].astype(np.int64), device="cuda")].cpu().numpy(), rep[:Gs].cpu().numpy())
    assert np.array_equal(yc[:Gs].cpu().numpy(), exp["yc"]) and np.array_equal(yx[:Gs].cpu().numpy().view(np.uint32), exp["yx"])
    assert np.array_equal(yd[:Gs].cpu().numpy(), exp["yd"])


@pytest.mark.parametrize("mode", [0, 3])
def test_collapse_compact_wire_format_equals_wide(mode):
    """n_cigar8 + cigar16 (+ cigar_ext for lengths >= 4095, here the long introns) must give exactly the wide-format result,
    from host buffers and from device-resident tensors."""
    import torch
    from oracle import oracle
    from tiebrush_b200 import api, synth
    k = 16
    cols, run_off, pr = synth.cohort_window(k, 20000, seed=17, n_tx=300, device="cpu")
    host = synth.to_host(cols)
    n8, c16, ext = api.compact_cigar_columns(host["cig_off"], host["cigar"])
    assert len(ext) > 0 and c16.dtype == np.uint16 and n8.dtype == np.uint8
    compact = {kk: host[kk] for kk in ("pos", "flag", "mapq", "strand", "nh")}
    compact.update(n_cigar8=n8, cigar16=c16, cigar_ext=ext)
    exp = oracle.collapse(host, run_off, mode=mode)
    with api.Context(device=0, n_samples=k, mode=mode) as ctx:
        wide = ctx.collapse_window(host, run_off)
        got = ctx.collapse_window(compact, run_off)
        dcols = {kk: torch.as_tensor(v.view(np.int16) if v.dtype == np.uint16 else (v.view(np.int32) if v.dtype == np.uint32 else v)).cuda() for kk, v in compact.items()}
        dgot = ctx.collapse_window(dcols, run_off, pos_range=pr)
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), exp[key]), key
        assert np.array_equal(np.asarray(got[key]), np.asarray(wide[key])), key
        G = dgot["n_groups"]
        assert np.array_equal(dgot[key][:G].cpu().numpy().view(np.asarray(exp[key]).dtype), exp[key]), key


def test_compact_wire_format_is_validated():
    """ADVICE r1: a packer whose n_cig / cigar_ext do not match the per-record op counts gets an error, not an out-of-bounds read."""
    from tiebrush_b200 import api, synth
    cols, run_off, pr = synth.cohort_window(6, 3000, seed=2, n_tx=20, device="cpu")
    host = synth.to_host(cols)
    n8, c16, ext = api.compact_cigar_columns(host["cig_off"], host["cigar"])
    compact = {k: host[k] for k in ("pos", "flag", "mapq", "strand", "nh")}
    with api.Context(device=0, n_samples=6) as ctx:
        bad = dict(compact, n_cigar8=n8.copy(), cigar16=c16, cigar_ext=ext)
        bad["n_cigar8"][5] += 1                                  # op counts no longer sum to n_cig
        with pytest.raises(api.TieBrushError, match="n_cigar8 sums to"):
            ctx.collapse_window(bad, run_off)
        if len(ext):
            bad = dict(compact, n_cigar8=n8, cigar16=c16, cigar_ext=ext[:-1].copy())   # one escaped length short
            with pytest.raises(api.TieBrushError, match="escaped lengths"):
                ctx.collapse_window(bad, run_off)
        ok = ctx.collapse_window(dict(compact, n_cigar8=n8, cigar16=c16, cigar_ext=ext), run_off)
        assert ok["n_groups"] > 0


@pytest.mark.parametrize("mode,name", [(3, "-E"), (1, "-L")])
def test_collapse_c3_full_size_properties_and_oracle_prefix(mode, name):
    """BASELINE C3 at its configured size: the C2 cohort (100 x 10M reads, chr1) in -E and -L modes with -N 5 -Q 1
    (TB_TEST_FULL=0 shrinks it to 100 x 2M). Size-independent properties over the whole output (sum YC == records that pass the
    filters, counted independently on the device; YX bounds; representatives pass the filters and come in position order) and
    bit-exact equality with the oracle on a coordinate prefix. VERDICT r1 item 5c."""
    import os
    import torch
    from oracle import oracle
    from tiebrush_b200 import api, synth
    k = 100
    reads = 2_000_000 if os.environ.get("TB_TEST_FULL") == "0" else 10_000_000
    cols, run_off, pr = synth.cohort_window(k, reads, seed=0, device="cuda", with_md=(mode == 1))
    if mode == 1:
        cols["md_off"], cols["md"], cols["n_md"] = synth.md_columns_torch(cols)
        del cols["md_mm"], cols["md_a"]
    n = k * reads
    out = dict(rep_index=torch.empty(n, dtype=torch.int32, device="cuda"), yc=torch.empty(n, dtype=torch.float32, device="cuda"),
               yx=torch.empty(n, dtype=torch.int32, device="cuda"), yd=torch.empty(n, dtype=torch.int32, device="cuda"))
    with api.Context(device=0, n_samples=k, mode=mode, max_nh=5, min_qual=1) as ctx:
        got = ctx.collapse_window(cols, run_off, pos_range=pr, out=out)
        assert ctx.last_path() == 0
    G = got["n_groups"]
    passes = ((cols["nh"].to(torch.int32) & 0xffff) <= 5) & (cols["mapq"].to(torch.int32) >= 1)
    kept = int(passes.sum().item())
    assert 0 < kept < n and got["n_kept"] == kept
    rep = out["rep_index"][:G].long() & 0xffffffff
    yc, yx, yd = out["yc"][:G], out["yx"][:G], out["yd"][:G]
    assert int(yc.to(torch.float64).sum().item()) == kept
    assert bool((yx >= 1).all()) and bool((yx.to(torch.float32) <= torch.clamp(yc, max=float(k))).all()) and bool((yd >= 0).all())
    assert bool(passes[rep].all())
    rpos = cols["pos"][rep]
    assert bool((rpos[1:] >= rpos[:-1]).all())
    sub, sub_off = synth.prefix_slice(cols, run_off, 1_500_000)
    hi = int(sub["pos"].max()) + 1
    exp = oracle.collapse(sub, sub_off, mode=mode, max_nh=5, min_qual=1)
    Gs = len(exp["rep_index"])
    assert Gs > 1000 and bool((rpos[:Gs] < hi).all()) and (G == Gs or int(rpos[Gs].item()) >= hi)
    # representatives compared through (file, index in file): the prefix keeps every file's order
    sub_file = np.searchsorted(sub_off, exp["rep_index"].astype(np.int64), side="right") - 1
    glob = np.asarray(run_off)[sub_file] + (exp["rep_index"].astype(np.int64) - sub_off[sub_file])
    assert np.array_equal(glob, rep[:Gs].cpu().numpy())
    assert np.array_equal(yc[:Gs].cpu().numpy(), exp["yc"]) and np.array_equal(yx[:Gs].cpu().numpy().view(np.uint32), exp["yx"])
    assert np.array_equal(yd[:Gs].cpu().numpy(), exp["yd"])


@pytest.mark.parametrize("mode,max_dict", [(0, 255), (3, 255), (0, 3)])
def test_collapse_packed_wire_format_equals_wide(mode, max_dict):
    """pos_d8 (+ pos_ext: run starts, large gaps) and meta8 (+ dictionary, escapes when the dictionary is too small) with the
    compact CIGAR columns must give exactly the wide-format result, from host buffers and from device-resident tensors."""
    import torch
    from oracle import oracle
    from tiebrush_b200 import api, synth
    k = 12
    cols, run_off, pr = synth.cohort_window(k, 15000, seed=23, n_tx=200, device="cpu")
    host = synth.to_host(cols)
    n8, c16, ext = api.compact_cigar_columns(host["cig_off"], host["cigar"])
    pk = api.pack_fixed_columns(host, run_off, max_dict=max_dict)
    assert len(pk["pos_ext"]) >= k and (len(pk["meta_ext"]) > 0) == (max_dict < 10)
    packed = dict(pk, n_cigar8=n8, cigar16=c16, cigar_ext=ext)
    exp = oracle.collapse(host, run_off, mode=mode)
    with api.Context(device=0, n_samples=k, mode=mode) as ctx:
        got = ctx.collapse_window(packed, run_off, pos_range=pr)
        tpk = api.pack_fixed_columns({kk: (v.cuda() if hasattr(v, "cuda") else v) for kk, v in cols.items()}, run_off, max_dict=max_dict)
        dcols = dict(tpk, n_cigar8=torch.as_tensor(n8).cuda(), cigar16=torch.as_tensor(c16.view(np.int16)).cuda(), cigar_ext=torch.as_tensor(ext.view(np.int32)).cuda())
        dgot = ctx.collapse_window(dcols, run_off, pos_range=pr)
        bad = dict(packed, pos_ext=pk["pos_ext"][:-1].copy())
        with pytest.raises(api.TieBrushError, match="pos_d8 holds"):
            ctx.collapse_window(bad, run_off, pos_range=pr)
    for key in ("rep_index", "yc", "yx", "yd"):
        assert np.array_equal(np.asarray(got[key]), exp[key]), key
        G = dgot["n_groups"]
        assert np.array_equal(dgot[key][:G].cpu().numpy().view(np.asarray(exp[key]).dtype), exp[key]), key
