"""CPU tests: the C restatement (oracle/tb_oracle.c) against golden vectors produced by the UNMODIFIED
compiled reference (tests/golden/make_golden.py). This is what pins the oracle."""
import hashlib
import os

import numpy as np
import pytest

import helpers as H
from oracle import oracle
from tiebrush_b200 import sam


@pytest.mark.parametrize("case", H.case_names("collapse_random.npz"))
def test_collapse_random(case):
    files, opts, fm, exp = H.load_collapse_case("collapse_random.npz", case)
    H.assert_collapse_equal(H.run_collapse(oracle.collapse, files, opts, fm), exp, case)


@pytest.mark.parametrize("case", H.case_names("collapse_fixture.npz"))
def test_collapse_fixture(case):
    files, opts, fm, exp = H.load_collapse_case("collapse_fixture.npz", case)
    H.assert_collapse_equal(H.run_collapse(oracle.collapse, files, opts, fm), exp, case)


@pytest.mark.parametrize("case", H.case_names("collapse_merged.npz"))
def test_collapse_merged(case):
    files, opts, fm, exp = H.load_collapse_case("collapse_merged.npz", case)
    H.assert_collapse_equal(H.run_collapse(oracle.collapse, files, opts, fm), exp, case)


@pytest.mark.parametrize("case", H.coverage_case_names())
def test_coverage(case):
    cols, runs, juncs = H.load_coverage_case(case)
    H.assert_coverage_equal(oracle.coverage(cols), runs, juncs, case)


def test_coverage_rejects_unsupported_ops():
    cols = dict(tid=np.zeros(1, np.int32), pos=np.asarray([10], np.int32), yc=np.ones(1, np.float32),
                strand=np.asarray([ord(".")], np.uint8), cig_off=np.asarray([0, 1], np.uint32),
                cigar=np.asarray([(5 << 4) | 7], np.uint32))
    with pytest.raises(ValueError):
        oracle.coverage(cols)


def test_full_fixtures_against_reference_md5():
    """All 20 sample BAMs of the reference's own tests (tests/golden/fixtures): the oracle's collapsed records, and its
    tiecov -c -j files on them, byte for byte what the compiled reference wrote (md5 of its outputs, helpers.REF_MD5)."""
    files, header, lines = H.fixture_inputs(["t1", "t2"])
    got = H.run_collapse(oracle.collapse, files, {})
    assert (got["n_kept"], len(got["lhash"])) == H.REF_COUNTS["t12"]
    records = H.collapsed_records(got, lines)
    assert H.md5_text(records) == H.REF_MD5["t12"]
    cols, names = H.coverage_input(header, records)
    cov = oracle.coverage(cols)
    assert len(cov["runs"][0]) == 9043 and len(cov["juncs"][0]) == 18
    bg, bed = H.coverage_files(cov, names)
    assert hashlib.md5(bg.encode()).hexdigest() == H.REF_MD5["cov"]
    assert hashlib.md5(bed.encode()).hexdigest() == H.REF_MD5["junc"]


def test_sample_heatmap_oracle_matches_the_reference_binary(tmp_path):
    """Groundwork for SURVEY §8f.2 (tiecov -s): the C restatement of addMean / discretize / normalize / flushCoverage against
    the UNMODIFIED reference binary on a TieBrush-made BAM (needs oracle/_ref, i.e. a container with /root/reference)."""
    import subprocess
    import sys
    ref = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref")
    if not all(os.path.exists(os.path.join(ref, b)) for b in ("tiebrush", "tiecov", "htsfile")):
        pytest.skip("reference binaries not built here")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import test_gpu_host_cli as T
    from oracle import oracle
    from tiebrush_b200 import sam
    paths = T._write_sams(str(tmp_path), k=5, reads=2500, seed=4, n_tx=15)
    bam = str(tmp_path / "c.bam")
    T._run([os.path.join(ref, "tiebrush"), "-o", bam] + paths)
    T._run([os.path.join(ref, "tiecov"), "-s", str(tmp_path / "s"), bam])
    text = subprocess.run([os.path.join(ref, "htsfile"), "-c", bam], capture_output=True, text=True, check=True).stdout
    n_samples = sum(1 for ln in text.split("\n") if ln.startswith("@CO\tSAMPLE:"))
    R, ids = sam.parse_sam(text)
    cols = sam.to_columns(R)
    cols["yx"] = cols["yx_in"]
    names = {v: k for k, v in ids.items()}
    t, s, e, iv = oracle.sample_heatmap(cols)
    got = [f"{names[int(a)]}\t{int(b)}\t{int(c)}\t{int(d)}\t{float(oracle.heatmap_value(int(d), n_samples)):f}" for a, b, c, d in zip(t, s, e, iv)]
    exp = [ln for ln in open(str(tmp_path / "s.bedgraph")).read().split("\n") if ln and not ln.startswith("track")]
    assert n_samples == 5 and len(exp) > 20
    assert got == exp


@pytest.mark.parametrize("case", ["t1", "t2"])
def test_sample_heatmap_oracle_matches_the_reference_fixtures(case):
    """tiecov -s groundwork: the oracle reproduces columns 1-4 of the reference's own test/t{1,2}/t{1,2}.sample.bedgraph from the
    committed columns of test/t{1,2}/t{1,2}.bam (tests/golden/make_golden_sample.py)."""
    from oracle import oracle
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sample_heatmap.npz"))
    cols = {k: z[f"{case}/in/{k}"] for k in ("tid", "pos", "cig_off", "cigar")}
    cols["yx"] = z[f"{case}/in/yx_in"]
    t, s, e, iv = oracle.sample_heatmap(cols)
    assert int(z[f"{case}/n_samples"][0]) == 10 and len(t) > 50
    assert np.array_equal(t, z[f"{case}/out/tid"]) and np.array_equal(s, z[f"{case}/out/start"])
    assert np.array_equal(e, z[f"{case}/out/end"]) and np.array_equal(iv, z[f"{case}/out/ival"])
