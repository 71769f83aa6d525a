#!/usr/bin/env python
"""bench.py — throughput of the tiebrush merge+collapse hot path (and tiecov coverage) on B200.

Contract: `python bench.py --gpus N --steps K --warmup W` (N>1 under torch.distributed.run, one rank per
GPU) prints ONE JSON line from rank 0. A step = one pass of the hot path over one synthetic cohort window
(BASELINE.json configs[1]: 100 RNA-seq samples x 10 M spliced 150-bp reads on chr1, default CIGAR mode)
with the inputs resident in HBM; `e2e` is the same call through the C ABI with HOST (pinned) buffers, the
host->device and device->host copies inside the timed region. `--impl reference` times the unmodified
reference binary (oracle/_ref/tiebrush, single-threaded as shipped) on a bounded sample of the same cohort.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--samples", type=int, default=int(os.environ.get("TB_BENCH_SAMPLES", 100)))
    ap.add_argument("--reads", type=int, default=int(os.environ.get("TB_BENCH_READS", 10_000_000)), help="reads per sample")
    ap.add_argument("--mode", type=int, default=0, help="0 default CIGAR, 1 -L (CIGAR+MD), 2 -P (clip), 3 -E (exon boundaries)")
    ap.add_argument("--max-nh", type=int, default=0x7fffffff, help="-N (C3 filters)")
    ap.add_argument("--min-qual", type=int, default=-1, help="-Q")
    ap.add_argument("--flag-mask", type=int, default=0, help="-F (uses the paired-end cohort so the mask has bits to bite on)")
    ap.add_argument("--cov-records", type=int, default=int(os.environ.get("TB_BENCH_COV", 2_000_000_000)),
                    help="records of the tiecov leg = BASELINE config C4: ONE whole-genome collapsed stream of this many records, "
                         "split in stream order over the GPUs (strong scaling; 0 = skip)")
    ap.add_argument("--cov-window", type=int, default=int(os.environ.get("TB_BENCH_COV_WINDOW", 0)),
                    help="records per tiecov window (cut at bundle heads); 0 = a quarter of the rank's slice (>= 4 windows per GPU: 5e8 records "
                         "each on 1 GPU, 6.25e7 on 8), at most 5e8")
    ap.add_argument("--cov-no-end", action="store_true", help="tiecov leg without the optional `end` column (the bundle kernel walks the CIGARs)")
    ap.add_argument("--cov-e2e-records", type=int, default=int(os.environ.get("TB_BENCH_COV_E2E", 250_000_000)),
                    help="records per rank of the tiecov end-to-end leg (host buffers; a prefix of the rank's slice)")
    ap.add_argument("--cov-cpu-sample", type=int, default=int(os.environ.get("TB_BENCH_COV_CPU", 2_000_000)),
                    help="records of the stream written as SAM for the reference tiecov binary (CPU baseline of the tiecov leg)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--wire", default="packed", choices=["packed", "compact", "wide"],
                    help="host column format of the e2e leg: packed = pos_d8 + meta8 (+ dictionary / escapes) and the compact CIGAR columns, "
                         "compact = wide fixed columns + n_cigar8 + cigar16 (+cigar_ext), wide = cig_off + cigar (u32)")
    ap.add_argument("--e2e-windows", type=int, default=int(os.environ.get("TB_BENCH_E2E_WINDOWS", 8)),
                    help="end-to-end leg: the window is handed over as this many coordinate sub-windows cut at coverage gaps (as the host tool "
                         "cuts them), two in flight on two contexts so that the copies of one overlap the kernels of the other (1 = one call)")
    ap.add_argument("--cpu-sample", type=int, default=int(os.environ.get("TB_BENCH_CPU_SAMPLE", 20_000_000)),
                    help="records of the cohort fed to the CPU baseline (bounded sample)")
    ap.add_argument("--cli-reads", type=int, default=int(os.environ.get("TB_BENCH_CLI_READS", 50_000)),
                    help="reads per sample file of the host command-line leg (0 = skip)")
    ap.add_argument("--ref-reads", type=int, default=int(os.environ.get("TB_BENCH_REF_READS", 50_000)),
                    help="--impl reference: reads per sample file written as SAM for the reference binary")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned (collapse groups, tiecov runs / junctions) as "
                         "DIR/<name>.npy: a fixed, seeded sample of rows, at most 64 MB in all, so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_ROWS = 1 << 18   # rows sampled per output table: the three tables stay under 64 MB as float64


def dump_table(out_dir, prefix, count, columns):
    """Writes a fixed, seeded sample of `count` rows of `columns` [(name, array, np dtype)] as out_dir/<prefix>_<name>.npy, the
    sampled row numbers as <prefix>_row.npy and the row count as <prefix>_count.npy. The sample depends on `count` alone, so
    two builds that return the same rows write the same files. Integer columns go out as float64 (exact below 2^53)."""
    os.makedirs(out_dir, exist_ok=True)
    rows = np.arange(count, dtype=np.int64) if count <= DUMP_ROWS else \
        np.sort(np.random.default_rng(12345).choice(count, DUMP_ROWS, replace=False))
    np.save(os.path.join(out_dir, f"{prefix}_count.npy"), np.asarray([count], np.float64))
    np.save(os.path.join(out_dir, f"{prefix}_row.npy"), rows.astype(np.float64))
    for name, a, dt in columns:
        if hasattr(a, "cpu"):   # device tensor: gather the sample there, copy only it
            import torch
            a = a[torch.from_numpy(rows).to(a.device)].cpu().numpy()
        else:
            a = np.asarray(a)[rows]
        np.save(os.path.join(out_dir, f"{prefix}_{name}.npy"), a.astype(dt))


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu_index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) > 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) > 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_per_record(kernel):
    """DRAM bytes per record of `kernel` from the committed ncu --set full capture (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return float(json.load(open(p))[kernel]["bytes_per_record"])
    except Exception:
        return None


def host_slice_sample(host, run_off, target):
    """A coordinate slice [lo,hi) of the window holding ~target records: all files, whole positions."""
    n = len(host["pos"])
    if target >= n:
        return host, run_off
    # pick the cut from the first run's quantile, then slice every run by coordinate
    frac = target / n
    r0 = host["pos"][run_off[0]:run_off[1]]
    hi = int(r0[min(len(r0) - 1, int(len(r0) * frac))])
    from tiebrush_b200 import sam
    idx, new_off = [], [0]
    for f in range(len(run_off) - 1):
        a, b = int(run_off[f]), int(run_off[f + 1])
        c = a + int(np.searchsorted(host["pos"][a:b], hi, side="left"))
        idx.append(np.arange(a, c, dtype=np.int64))
        new_off.append(new_off[-1] + (c - a))
    idx = np.concatenate(idx)
    sub = {k: host[k][idx] for k in ("pos", "flag", "mapq", "strand", "nh")}
    sub["cig_off"], sub["cigar"] = sam._gather_csr(host["cig_off"], host["cigar"], idx)
    if "md_off" in host:
        sub["md_off"], sub["md"] = sam._gather_csr(host["md_off"], host["md"], idx)
    return sub, np.asarray(new_off, np.int64)


def write_sam_files(host, run_off, tmpdir):
    """Materialise a (small) window as one SAM file per sample for the reference binary."""
    from tiebrush_b200 import sam
    paths = []
    hdr = "@HD\tVN:1.0\tSO:coordinate\n@SQ\tSN:chr1\tLN:248956422\n"
    for f in range(len(run_off) - 1):
        a, b = int(run_off[f]), int(run_off[f + 1])
        lines = [hdr]
        for i in range(a, b):
            cig = sam.cigar_str(host["cigar"][host["cig_off"][i]:host["cig_off"][i + 1]])
            tags = f"NH:i:{int(host['nh'][i])}"
            s = chr(int(host["strand"][i]))
            if s != ".":
                tags += f"\tXS:A:{s}"
            lines.append(f"s{f}.{i}\t{int(host['flag'][i])}\tchr1\t{int(host['pos'][i]) + 1}\t{int(host['mapq'][i])}\t{cig}\t*\t0\t0\t*\t*\t{tags}\n")
        p = os.path.join(tmpdir, f"s{f}.sam")
        with open(p, "w") as fh:
            fh.write("".join(lines))
        paths.append(p)
    return paths


def to_bam_files(sam_paths):
    """SAM text -> BAM with oracle/_ref/hts_tool (the reference's vendored htslib); None when the tool is not built."""
    tool = os.path.join(ROOT, "oracle", "_ref", "hts_tool")
    if not os.path.exists(tool):
        return None
    out = []
    for p in sam_paths:
        b = p[:-4] + ".bam"
        if subprocess.run([tool, "tobam", p, b], capture_output=True).returncode != 0:
            return None
        os.remove(p)
        out.append(b)
    return out


def run_reference_arm(args):
    """Times the UNMODIFIED reference binary (single-threaded, as shipped) on a bounded sample: K steps of
    `tiebrush -o out.bam s0.bam ... s{k-1}.bam`, wall clock around the process. Beside the headline (-O2, 1 thread, BAM in /
    BAM out) SURVEY §8d's other baselines are taken once each: the -O0 -g build that the reference's CMakeLists.txt:49
    produces, the reference's own parallel driver tiewrap.py on all host cores, and a decode-only pass over the inputs."""
    from tiebrush_b200 import synth
    refdir = os.path.join(ROOT, "oracle", "_ref")
    ref = os.path.join(refdir, "tiebrush")
    line = {"impl": "reference", "metric": "alignments_collapsed_per_sec", "unit": "alignments/s", "higher_is_better": True,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "dtype": "u32", "data": "synthetic", "scaling": "weak",
            "vs_baseline": None}
    if not os.path.exists(ref):
        line["unavailable"] = "oracle/_ref/tiebrush not built (needs /root/reference at build time)"
        print(json.dumps(line)); return
    cols, run_off, _ = synth.cohort_window(args.samples, args.ref_reads, seed=0, device="cpu")
    host = synth.to_host(cols)
    n = len(host["pos"])
    nproc = len(os.sched_getaffinity(0))
    extra = {}
    with tempfile.TemporaryDirectory() as tmp:
        paths = write_sam_files(host, run_off, tmp)
        bams = to_bam_files(paths)
        fmt = "BAM"
        if bams is None:
            bams, fmt = write_sam_files(host, run_off, tmp), "SAM text (oracle/_ref/hts_tool missing)"
        times = []
        for it in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            r = subprocess.run([ref, "-o", os.path.join(tmp, "o.bam")] + bams, capture_output=True, text=True)
            dt = time.perf_counter() - t0
            if r.returncode != 0:
                line["unavailable"] = "reference binary failed: " + r.stderr[:200]
                print(json.dumps(line)); return
            if it >= args.warmup:
                times.append(dt)

        def once(cmd, **kw):
            t0 = time.perf_counter()
            r = subprocess.run(cmd, capture_output=True, text=True, **kw)
            return (time.perf_counter() - t0) if r.returncode == 0 else None, r

        o0 = os.path.join(refdir, "tiebrush_O0")
        if os.path.exists(o0):
            dt, _ = once([o0, "-o", os.path.join(tmp, "o0.bam")] + bams)
            if dt:
                extra["O0_build"] = {"value": n / dt, "unit": "alignments/s", "cores": 1, "seconds": dt,
                                     "what": "-O0 -g build of the same sources (what the reference's CMakeLists.txt:49 produces), 1 run"}
        tw = os.path.join(refdir, "tiewrap.py")
        if os.path.exists(tw):
            bsz = max(2, -(-len(bams) // nproc))
            dt, r = once([sys.executable, tw, "-t", str(nproc), "-b", str(bsz), "-o", os.path.join(tmp, "tw.bam")] + bams)
            if dt:
                extra["tiewrap_all_cores"] = {"value": n / dt, "unit": "alignments/s", "cores": nproc, "batch_size": bsz, "seconds": dt,
                                              "what": f"the reference's own parallel mode: tiewrap.py -t {nproc} -b {bsz} (batch tree of tiebrush -O2 processes), 1 run"}
        tool = os.path.join(refdir, "hts_tool")
        if os.path.exists(tool) and fmt == "BAM":
            dt, r = once([tool, "decode"] + bams)
            if dt:
                extra["decode_only"] = {"value": n / dt, "unit": "alignments/s", "cores": 1, "seconds": dt,
                                        "what": "sam_read1 loop over the same BAM inputs (htslib sam.c), no collapse, no output: the host decode share"}
    ms = 1000.0 * float(np.mean(times))
    v = n / (ms / 1000.0)
    line.update({"value": v, "ms_per_step": ms,
                 "config": {"workload": f"C2 cohort model (100 samples x 10M reads chr1, default mode); bounded sample: {args.samples} {fmt} files x {args.ref_reads} reads",
                            "records_per_step": n, "host_cores_available": nproc},
                 "cpu_baseline": {"value": v, "unit": "alignments/s", "cores": 1, "kind": "reference",
                                  "sample": f"{args.samples} files x {args.ref_reads} reads of the C2 cohort model as {fmt}, reference tiebrush -O2, 1 thread (the reference is single-threaded)",
                                  **extra},
                 "e2e": {"value": v, "unit": "alignments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(line))


def run_host_cli(args):
    """tiebrush_gpu (reference main loop replaced by the window packer + tb_collapse_window) on SAM files of the cohort."""
    import re
    from tiebrush_b200 import synth
    exe = os.path.join(ROOT, "tiebrush_b200", "host", "_build", "tiebrush_gpu")
    if not os.path.exists(exe):
        return {"unavailable": "tiebrush_b200/host/_build/tiebrush_gpu not built (needs /root/reference at build time)"}
    cols, run_off, _ = synth.cohort_window(args.samples, args.cli_reads, seed=0, device="cpu")
    host = synth.to_host(cols)
    n = len(host["pos"])
    with tempfile.TemporaryDirectory() as tmp:
        paths = write_sam_files(host, run_off, tmp)
        bams = to_bam_files(paths)
        fmt = "BAM"
        if bams is None:
            bams, fmt = write_sam_files(host, run_off, tmp), "SAM"
        paths = bams
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            r = subprocess.run([exe, "-o", os.path.join(tmp, "o.bam")] + paths, capture_output=True, text=True, env=dict(os.environ, TB_TIMING="1"))
            dt = time.perf_counter() - t0
            if r.returncode != 0:
                return {"unavailable": "tiebrush_gpu failed: " + r.stderr[-200:]}
            if best is None or dt < best[0]:
                best = (dt, r.stderr)
    m = re.search(r"total ([0-9.]+) s \| decode\+merge ([0-9.]+) \| pack ([0-9.]+) \| device \(H2D\+kernels\+D2H\) ([0-9.]+) \| tag\+write ([0-9.]+) \| windows (\d+)", best[1])
    out = {"value": n / best[0], "unit": "alignments/s", "wall_s": best[0], "records": n,
           "sample": f"{args.samples} {fmt} files x {args.cli_reads} reads of the C2 cohort model (same sample as --impl reference), {fmt} in / BAM out, best of 3, process start to exit"}
    if m:
        out.update({"in_process_s": float(m.group(1)), "decode_merge_s": float(m.group(2)), "pack_s": float(m.group(3)),
                    "device_s": float(m.group(4)), "tag_write_s": float(m.group(5)), "windows": int(m.group(6))})
    return out


def write_cov_sam(cols, path, n_contigs):
    """A prefix of the collapsed stream as SAM text (YC:i tags) for the reference tiecov binary."""
    from tiebrush_b200 import sam, synth
    lens, _, _ = synth.genome_layout(1000)
    hdr = "@HD\tVN:1.0\tSO:coordinate\n" + "".join(f"@SQ\tSN:ctg{c}\tLN:{int(lens[c])}\n" for c in range(n_contigs))
    off, cig = cols["cig_off"], cols["cigar"]
    with open(path, "w") as fh:
        fh.write(hdr)
        buf = []
        for i in range(len(cols["pos"])):
            c = sam.cigar_str(cig[off[i]:off[i + 1]])
            s = chr(int(cols["strand"][i]))
            tags = f"YC:i:{int(cols['yc'][i])}" + (f"\tXS:A:{s}" if s != "." else "")
            buf.append(f"r{i}\t0\tctg{int(cols['tid'][i])}\t{int(cols['pos'][i]) + 1}\t60\t{c}\t*\t0\t0\t*\t*\t{tags}\n")
            if len(buf) >= 100000:
                fh.write("".join(buf)); buf = []
        fh.write("".join(buf))


def gap_cut_subwindows(cols, run_off, pr, S, dev):
    """The file-major window as S coordinate sub-windows cut where NO read of any sample covers the cut coordinate (the rule of
    the host tool, tiebrush_gpu_main.cpp: groups never span a start position and the YD segment lists are empty after a gap,
    so the sub-windows are independent and their outputs concatenate to the window's). Returns [(cols_s, run_off_s, (lo, hi))]."""
    import torch
    k = len(run_off) - 1
    lo = int(pr[0])
    span = int(pr[1]) - lo + 400000
    cover = torch.zeros(span + 2, dtype=torch.int32, device=dev)
    offs = []
    for f in range(k):
        a, b = int(run_off[f]), int(run_off[f + 1])
        o = cols["cig_off"][a:b + 1].to(torch.int64) & 0xFFFFFFFF
        offs.append(o)
        c0, c1 = int(o[0]), int(o[-1])
        cig = cols["cigar"][c0:c1].to(torch.int64) & 0xFFFFFFFF
        op = cig & 0xF
        ref = torch.where((op == 0) | (op == 2) | (op == 3) | (op == 7) | (op == 8), cig >> 4, torch.zeros_like(cig))
        cs = torch.zeros(c1 - c0 + 1, dtype=torch.int64, device=dev)
        cs[1:] = torch.cumsum(ref, 0)
        rl = cs[o[1:] - c0] - cs[o[:-1] - c0]
        p = cols["pos"][a:b].to(torch.int64) - lo
        ones = torch.ones(b - a, dtype=torch.int32, device=dev)
        cover.index_add_(0, p, ones)
        cover.index_add_(0, (p + rl).clamp(max=span), -ones)
        del cig, op, ref, cs, rl, p, ones
    depth = torch.cumsum(cover, 0, dtype=torch.int32)
    del cover
    # records that start before every coordinate (for balancing the cuts by records, not by coordinate)
    starts = torch.zeros(span + 2, dtype=torch.int32, device=dev)
    for f in range(k):
        a, b = int(run_off[f]), int(run_off[f + 1])
        starts.index_add_(0, cols["pos"][a:b].to(torch.int64) - lo, torch.ones(b - a, dtype=torch.int32, device=dev))
    cum = torch.cumsum(starts, 0, dtype=torch.int64)     # cum[x] = records with pos - lo <= x
    del starts
    n_all = int(cum[-1].item())
    cuts, prev_cnt, prev_x = [], 0, 0
    W_ = 20_000_000
    for s_ in range(1, S):
        target = prev_cnt + (n_all - prev_cnt) // (S - s_ + 1)      # re-balanced after a stretch that could not be cut
        x = int(torch.searchsorted(cum, torch.tensor([target], device=dev, dtype=torch.int64))[0].item())
        x = min(max(x, prev_x + 1), span)
        cand = []
        zf = (depth[x:x + W_] == 0).nonzero()
        if len(zf):
            cand.append(x + int(zf[0].item()))
        a0 = max(prev_x + 1, x - W_)
        zb = (depth[a0:x + 1] == 0).nonzero()
        if len(zb):
            cand.append(a0 + int(zb[-1].item()))
        cand = [c for c in cand if prev_x < c < span]
        if not cand:
            continue
        best = min(cand, key=lambda c: abs(int(cum[c - 1].item()) - target))
        cnt = int(cum[best - 1].item())           # records with pos - lo < best
        if cnt <= prev_cnt or cnt >= n_all:
            continue
        cuts.append(lo + best); prev_cnt, prev_x = cnt, best
    del depth, cum
    bounds = [lo] + [c for c in cuts if c < int(pr[1])] + [int(pr[1])]
    subs = []
    for s_ in range(len(bounds) - 1):
        b0 = torch.tensor([bounds[s_], bounds[s_ + 1]], device=dev, dtype=cols["pos"].dtype)
        parts = {kk: [] for kk in ("pos", "flag", "mapq", "strand", "nh", "cig_off", "cigar")}
        ro, base = [0], 0
        for f in range(k):
            a, b = int(run_off[f]), int(run_off[f + 1])
            i0, i1 = (int(v) for v in torch.searchsorted(cols["pos"][a:b], b0))
            for kk in ("pos", "flag", "mapq", "strand", "nh"):
                parts[kk].append(cols[kk][a + i0:a + i1])
            o = offs[f]
            c0, c1 = int(o[i0]), int(o[i1])
            parts["cig_off"].append(o[i0:i1] - c0 + base)
            parts["cigar"].append(cols["cigar"][c0:c1])
            base += c1 - c0
            ro.append(ro[-1] + (i1 - i0))
        sub = {kk: torch.cat(v) for kk, v in parts.items() if kk != "cig_off"}
        sub["cig_off"] = torch.cat(parts["cig_off"] + [torch.tensor([base], device=dev, dtype=torch.int64)]).to(torch.int32)
        sub["n_cig"] = base
        subs.append((sub, np.asarray(ro, np.int64), (bounds[s_], bounds[s_ + 1])))
    return subs


def pin_wire(api, sub, run_off, wire):
    """Pinned host arrays of one (sub-)window in the wire format; returns (host dict, bytes)."""
    import torch
    wc = dict(sub)
    names = ("pos", "flag", "mapq", "strand", "nh", "cig_off", "cigar")
    if wire in ("compact", "packed"):
        wc["n_cigar8"], wc["cigar16"], wc["cigar_ext"] = api.compact_cigar_columns(sub["cig_off"], sub["cigar"])
        names = ("pos", "flag", "mapq", "strand", "nh", "n_cigar8", "cigar16", "cigar_ext")
    meta_dict = None
    if wire == "packed":
        pk = api.pack_fixed_columns(sub, run_off)
        meta_dict = pk.pop("meta_dict")
        wc.update(pk)
        names = ("pos_d8", "pos_ext", "meta8", "meta_ext", "n_cigar8", "cigar16", "cigar_ext")
    host, nbytes = {}, 0
    for name in names:
        t = wc[name]
        ht = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        ht.copy_(t)
        host[name] = ht.numpy().view({"cig_off": np.uint32, "cigar": np.uint32, "flag": np.uint16, "nh": np.uint16, "cigar16": np.uint16, "cigar_ext": np.uint32, "meta_ext": np.uint64}.get(name, ht.numpy().dtype))
        nbytes += ht.numel() * ht.element_size()
    host["n_cig"] = int(sub["n_cig"])
    if meta_dict is not None:
        host["meta_dict"] = meta_dict
        nbytes += meta_dict.nbytes
    return host, nbytes


def run_tiecov_leg(args, rank, world, local, dev, stream, peak, barrier, dist):
    import torch
    from tiebrush_b200 import api, synth
    R = args.cov_records
    a, b = rank * R // world, (rank + 1) * R // world
    t_gen = time.perf_counter()
    # the segments carry the `end` column a host packer has for free (GSamRecord::end): the bundle kernel then reads 16 B per record
    segs, mbases = synth.genome_slice(R, a, b, seed=0, device=dev, with_end=not args.cov_no_end)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    n_local = b - a
    if args.cov_window <= 0:
        args.cov_window = int(min(500_000_000, max(1 << 20, -(-n_local // 4))))
    ncig_local = sum(int(s["n_cig"]) for s in segs)
    cctx = api.Context(device=local, n_samples=1)
    cctx.set_stream(stream.cuda_stream); cctx.set_profiling(True)
    if world > 1:   # one NCCL communicator of the library's own per rank; the id travels over torch.distributed
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(api.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        cctx.comm_init(rank, world, idt.cpu().numpy().tobytes())
    # rows: a run needs a covered base of its own, so deep streams have few per record (0.15 at 2e9), shallow ones up to ~0.5
    capr, capj = int(1.0 * n_local) + (1 << 22), int(0.05 * n_local) + (1 << 22)
    out_local = api.cov_out_buffers(capr, capj, device=dev)
    if world > 1 and rank == 0:
        all_out = api.cov_out_buffers(world * capr, world * capj, device=dev)
    else:
        all_out = out_local if rank == 0 else None

    cap_all_r, cap_all_j = world * capr, world * capj   # rank 0: one region per rank (the same capacities on every rank)

    def step():
        # this rank's windows with the ordered gather folded in: after every window the new rows travel to rank 0's region
        # of this rank on a second stream while the next window computes
        loc = cctx.shard_coverage_gather(segs, args.cov_window, out_local, all_out, cap_all_r, cap_all_j, world)
        ms = [cctx.last_kernel_ms(i) for i in (6, 1, 7, 9)]
        g = {"gather_bytes": loc["stats"]["gather_bytes"], "rounds": loc["stats"]["gather_rounds"]}
        return loc, g, ms

    for _ in range(max(1, args.warmup)):
        loc, g, ms = step()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = cctx.launch_count()
    barrier()
    with torch.cuda.stream(stream):
        c0.record(stream)
        for _ in range(args.steps):
            loc, g, ms = step()
        c1.record(stream)
    barrier()
    launches = cctx.launch_count() - l0
    cov_ms = c0.elapsed_time(c1) / args.steps
    if args.dump_outputs and rank == 0:   # the rows of the whole stream, gathered on rank 0 by the last step
        f64, f32 = np.float64, np.float32
        dump_table(args.dump_outputs, "tiecov_runs", loc["total_runs"],
                   list(zip(("tid", "start", "end", "value"), loc["gathered_runs"](), (f64, f64, f64, f64))))
        dump_table(args.dump_outputs, "tiecov_juncs", loc["total_juncs"],
                   list(zip(("tid", "start", "end", "strand", "value"), loc["gathered_juncs"](), (f64, f64, f64, f32, f64))))
    tot = torch.tensor([float(mbases), float(loc["n_runs"]), float(loc["n_juncs"]), float(loc["stats"]["halo_bytes_sent"]),
                        float(loc["stats"]["lead_sent"]), float(g["gather_bytes"]) if rank else 0.0], device=dev, dtype=torch.float64)
    tmax = torch.tensor([cov_ms, ms[3]], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    cov_ms = float(tmax[0].item())
    mb_tot, runs_tot, juncs_tot = float(tot[0].item()), int(tot[1].item()), int(tot[2].item())
    if rank == 0:
        assert loc["total_runs"] == runs_tot and loc["total_juncs"] == juncs_tot, "gathered rows != rows produced"
    a_cov = n_local * (19 + 4 * ncig_local / max(n_local, 1)) + 16 * loc["n_runs"] + 16 * loc["n_juncs"]   # this rank's algorithmic bytes (SURVEY §8d)
    acc_ms = max(ms[1], 1e-6)
    line = {"metric": "coverage_bases_per_sec", "value": mb_tot / (cov_ms / 1000.0), "unit": "bases/s", "records_per_sec": R / (cov_ms / 1000.0),
            "ms_per_step": cov_ms, "n_gpus": world, "scaling": "strong", "steps": args.steps,
            "config": {"workload": f"C4: tiecov -c -j on ONE synthetic collapsed whole-genome stream of {R} records (96 contigs, Zipf YC), split in stream order over {world} GPU(s), windows of <= {args.cov_window} records cut at bundle heads",
                       "records": R, "records_per_gpu": n_local, "end_column": not args.cov_no_end, "windows_per_gpu": loc["windows"], "gen_seconds": t_gen,
                       "l2": "inputs (27 B/record, GBs per GPU) exceed the 126 MB L2; no flush needed"},
            "runs": runs_tot, "juncs": juncs_tot, "gpu_launches": int(launches),
            "exchange": {"halo_ms_max": float(tmax[1].item()), "lead_records_moved": int(tot[4].item()), "halo_bytes": int(tot[3].item()),
                         "gather_bytes": int(tot[5].item()), "gather_rounds": int(g["rounds"]),
                         "collectives": "ncclAllGather x2 (open-bundle state, lead sizes) + grouped ncclSend/ncclRecv (lead records); per window, on a second stream: ncclAllGather (new row counts) + grouped ncclSend/ncclRecv (the window's rows into this rank's region on rank 0), overlapped with the next window" if world > 1 else "none (1 GPU)"},
            "roofline": {"bound": "hbm", "kernel": "cov_accumulate_kernel", "achieved": a_cov / (acc_ms / 1000.0) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": a_cov / (acc_ms / 1000.0) / 1e9 / peak, "kernel_ms": float(acc_ms), "algorithmic_bytes": float(a_cov),
                         "traffic": (lambda t: None if t is None else t * n_local)(traffic_per_record("cov_accumulate_kernel")),
                         "traffic_source": "ncu dram bytes per record (profiles/traffic.json) x records of rank 0",
                         "note": "rank 0: sum of the kernel's launches over its windows"},
            "stage_ms": dict(zip(("bundles", "accumulate", "runs", "halo_exchange"), [float(x) for x in ms]))}
    # ---- end to end: the same call with HOST (pinned) buffers, H2D per window and D2H of the rows inside the timed region ----
    if not args.no_e2e and args.cov_e2e_records > 0 and segs:
        ne = min(args.cov_e2e_records, int(segs[0]["pos"].shape[0]))
        seg = segs[0]
        w1 = int(seg["cig_off"][ne].item()) & 0xFFFFFFFF
        host, h2d = {}, 0
        for name, cnt in (("tid", ne), ("pos", ne), ("yc", ne), ("strand", ne), ("cig_off", ne + 1), ("cigar", w1)):   # no `end` over PCIe: the device derives it
            ht = torch.empty(cnt, dtype=seg[name].dtype, pin_memory=True)
            ht.copy_(seg[name][:cnt])
            host[name] = ht.numpy().view({"cig_off": np.uint32, "cigar": np.uint32}.get(name, ht.numpy().dtype))
            h2d += ht.numel() * ht.element_size()
        host["n_cig"] = w1
        mb_e = float(synth.m_bases(dict(cigar=seg["cigar"][:w1])))
        ecap_r, ecap_j = int(1.0 * ne) + (1 << 22), int(0.05 * ne) + (1 << 22)
        pin = lambda m, dt: torch.empty(m, dtype=dt, pin_memory=True).numpy()
        hout = dict(r_tid=pin(ecap_r, torch.int32), r_start=pin(ecap_r, torch.int32), r_end=pin(ecap_r, torch.int32), r_val=pin(ecap_r, torch.float64),
                    j_tid=pin(ecap_j, torch.int32), j_start=pin(ecap_j, torch.int32), j_end=pin(ecap_j, torch.int32), j_strand=pin(ecap_j, torch.uint8),
                    j_val=pin(ecap_j, torch.float64))
        del out_local, all_out
        torch.cuda.empty_cache()
        r2 = cctx.coverage_stream(host, args.cov_window, hout)
        es = args.steps
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with torch.cuda.stream(stream):
            g0.record(stream)
            for _ in range(es):
                r2 = cctx.coverage_stream(host, args.cov_window, hout)
            g1.record(stream)
        barrier()
        e_ms = g0.elapsed_time(g1) / es
        et = torch.tensor([e_ms], device=dev, dtype=torch.float64); eb = torch.tensor([mb_e, float(h2d), float(20 * r2["n_runs"] + 21 * r2["n_juncs"])], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(et, op=dist.ReduceOp.MAX); dist.all_reduce(eb, op=dist.ReduceOp.SUM)
        line["e2e"] = {"value": float(eb[0].item()) / (float(et[0].item()) / 1000.0), "unit": "bases/s", "ms_per_step": float(et[0].item()),
                       "h2d_bytes_per_step": int(eb[1].item()), "d2h_bytes_per_step": int(eb[2].item()), "steps": es,
                       "sample": f"the first {ne} records of every rank's slice through tc_coverage_stream with pinned host arrays ({r2['windows']} windows; H2D per window and D2H of the rows inside the timed region)"}
        del host, hout
    # ---- CPU baseline of this leg: the UNMODIFIED reference tiecov binary on a bounded prefix of the same stream (rank 0, N = 1) ----
    ref = os.path.join(ROOT, "oracle", "_ref", "tiecov")
    if rank == 0 and world == 1 and args.cov_cpu_sample > 0 and segs and os.path.exists(ref):
        ns = min(args.cov_cpu_sample, int(segs[0]["pos"].shape[0]))
        w1 = int(segs[0]["cig_off"][ns].item()) & 0xFFFFFFFF
        sub = {k: segs[0][k][:ns].cpu().numpy() for k in ("tid", "pos", "yc", "strand")}
        sub["cig_off"] = segs[0]["cig_off"][:ns + 1].cpu().numpy().view(np.uint32); sub["cigar"] = segs[0]["cigar"][:w1].cpu().numpy().view(np.uint32)
        mb_s = float(synth.m_bases(dict(cigar=segs[0]["cigar"][:w1])))
        with tempfile.TemporaryDirectory() as tmp:
            sp = os.path.join(tmp, "c.sam")
            write_cov_sam(sub, sp, 96)
            best = None
            for _ in range(2):
                t0 = time.perf_counter()
                r = subprocess.run([ref, "-c", os.path.join(tmp, "o.cov"), "-j", os.path.join(tmp, "o.j"), sp], capture_output=True, text=True)
                dt = time.perf_counter() - t0
                if r.returncode == 0 and (best is None or dt < best):
                    best = dt
        if best:
            line["cpu_baseline"] = {"value": mb_s / best, "unit": "bases/s", "records_per_sec": ns / best, "cores": 1, "kind": "reference",
                                    "sample": f"the first {ns} records of the same stream as SAM text, reference tiecov -c -j (-O2, single-threaded as shipped), best of 2, process start to exit ({best:.2f} s)"}
    cctx.close()
    del segs
    return line


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        if rank == 0:
            run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    from tiebrush_b200 import api, synth
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # keep this rank's host threads (and so its first-touch / pinned allocations) on the CPUs next to its GPU: with one
    # process per GPU the host->device copies of the e2e leg otherwise cross the socket interconnect
    numa = "unset"
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        numa = f"nvml cpu affinity, {len(os.sched_getaffinity(0))} cpus"
    except Exception as ex:   # not fatal: only the e2e leg's copy rate depends on it
        numa = f"unset ({type(ex).__name__})"
    if world > 1:
        # keep stdout to the ONE JSON line: NCCL prints its version banner there when NCCL_DEBUG=VERSION
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(device=dev)
    peak, peak_src = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- tiecov leg = BASELINE config C4: coverage + junctions + bedGraph runs of ONE collapsed whole-genome stream, split in
    #      stream order over the ranks (strong scaling). Timed region per step: halo exchange over NCCL (open-bundle state
    #      allgather, lead records to the owner of the bundle), per-rank windows cut at bundle heads, ordered gather on rank 0.
    tiecov_line = None
    if args.cov_records > 0:
        tiecov_line = run_tiecov_leg(args, rank, world, local, dev, stream, peak, barrier, dist)
        torch.cuda.empty_cache()

    k, reads = args.samples, args.reads
    n = k * reads
    # ---- synthetic cohort straight into HBM; rank r owns an independent coordinate shard (weak scaling) ----
    t_gen = time.perf_counter()
    # ONE cohort whatever the number of GPUs (strong scaling): every rank draws the same window and keeps its coordinate shard,
    # cut where no read of any sample covers the cut (groups never span a start position, YD lists are empty after a gap:
    # the shards are independent and their outputs concatenate to the window's); the groups are gathered on rank 0 over NCCL
    # inside the timed region. -L keeps independent per-rank windows (the MD arena is not re-cut here).
    strong = world > 1 and args.mode != 1
    cols, run_off, pr = synth.cohort_window(k, reads, seed=0 if strong else rank, device=dev, with_md=(args.mode == 1), paired=(args.flag_mask != 0))
    if args.mode == 1:
        cols["md_off"], cols["md"], cols["n_md"] = synth.md_columns_torch(cols)
        del cols["md_mm"], cols["md_a"]
    n_total = n if (strong or world == 1) else world * n
    if strong:
        subs = gap_cut_subwindows(cols, run_off, pr, world, dev)
        del cols
        if rank < len(subs):
            cols, run_off, pr = subs[rank]
        else:   # fewer gaps than ranks (tiny inputs): this rank idles
            cols, run_off, pr = subs[-1]
            cols = {kk: (v[:0] if hasattr(v, "shape") and kk != "cig_off" else v) for kk, v in cols.items()}
            cols["cig_off"] = torch.zeros(1, dtype=torch.int32, device=dev); cols["n_cig"] = 0
            run_off = np.zeros(k + 1, np.int64)
        del subs
        torch.cuda.empty_cache()
        n = int(cols["pos"].shape[0])
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    n_cig = cols["n_cig"]
    ctx = api.Context(device=local, n_samples=k, mode=args.mode, flag_mask=args.flag_mask, max_nh=args.max_nh, min_qual=args.min_qual)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_profiling(True)
    out = dict(rep_index=torch.empty(n, dtype=torch.int32, device=dev), yc=torch.empty(n, dtype=torch.float32, device=dev),
               yx=torch.empty(n, dtype=torch.int32, device=dev), yd=torch.empty(n, dtype=torch.int32, device=dev))

    gat = None
    if strong:   # rank 0's arrays for the ordered gather of the groups (rep_index | yc | yx | yd), sized from the first run
        cnt_t = torch.zeros(world, dtype=torch.int64, device=dev)

    def gather_groups(g_local):
        """ordered gather of this step's groups on rank 0: all_gather of the counts, one batch of NCCL send / recv"""
        nonlocal gat
        mine = torch.tensor([g_local], dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(cnt_t, mine)
        counts = [int(x) for x in cnt_t.tolist()]
        ops = []
        if rank == 0:
            tot = sum(counts)
            if gat is None or gat["rep_index"].shape[0] < tot:
                gat = {kk: torch.empty(tot + 1024, dtype=v.dtype, device=dev) for kk, v in out.items()}
            off = 0
            for r_, c_ in enumerate(counts):
                if r_ == 0:
                    for kk in out:
                        gat[kk][:c_].copy_(out[kk][:c_], non_blocking=True)
                elif c_ > 0:
                    ops += [dist.P2POp(dist.irecv, gat[kk][off:off + c_], r_) for kk in ("rep_index", "yc", "yx", "yd")]
                off += c_
        elif g_local > 0:
            ops = [dist.P2POp(dist.isend, out[kk][:g_local], 0) for kk in ("rep_index", "yc", "yx", "yd")]
        if ops:
            for w_ in dist.batch_isend_irecv(ops):
                w_.wait()
        return sum(counts)

    def step_dev():
        r_ = ctx.collapse_window(cols, run_off, pos_range=pr, out=out) if n > 0 else {"n_groups": 0, "n_kept": 0}
        if strong:
            r_["groups_all_ranks"] = gather_groups(r_["n_groups"])
        return r_

    for _ in range(args.warmup):
        res = step_dev()
    G = res["n_groups"] if args.warmup else 0
    sampler = ClockSampler(local); sampler.start()
    barrier()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kms, stages = [], []
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(args.steps):
            res = step_dev()
            kms.append(ctx.last_kernel_ms(0))
            stages.append([ctx.last_kernel_ms(i) for i in (2, 3, 0, 4, 5)])
        e1.record(stream)
    barrier()
    launches = ctx.launch_count() - l0
    ms_total = e0.elapsed_time(e1)
    G = res["n_groups"]
    if args.dump_outputs and rank == 0:   # the groups of the last step (of every rank when the cohort is sharded)
        # no name may keep `out` alive here: the e2e leg below frees it to make room for its own buffers
        g_all = res["groups_all_ranks"] if strong else G
        dump_table(args.dump_outputs, "collapse", g_all, [(kk, (gat if strong else out)[kk][:g_all], np.float32 if kk == "yc" else np.float64)
                                                          for kk in ("rep_index", "yc", "yx", "yd")])
        if not strong:
            np.save(os.path.join(args.dump_outputs, "collapse_n_kept.npy"), np.asarray([res["n_kept"]], np.float64))
    if world > 1:
        t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    per_rank = None
    if world > 1:   # who is the slowest: records, groups and device time of the collapse call alone, per rank
        mine = torch.tensor([float(n), float(G), float(np.mean([sum(x) for x in stages]))], device=dev, dtype=torch.float64)
        allr = torch.zeros(3 * world, device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(allr, mine)
        a_ = allr.cpu().numpy().reshape(world, 3)
        per_rank = {"records": [int(x) for x in a_[:, 0]], "groups": [int(x) for x in a_[:, 1]], "kernel_ms": [round(float(x), 3) for x in a_[:, 2]]}
    ms_step = ms_total / args.steps
    value = n_total / (ms_step / 1000.0)
    clocks = sampler
    # ---- roofline of the dominant kernel (collapse tile kernel) ----
    cbar = n_cig / n
    mbar = (int(cols["n_md"]) / n) if (args.mode == 1 and "n_md" in cols) else 0.0
    a_col = n * (30 + 4 * cbar + mbar) + 12 * G     # SURVEY §8d algorithmic bytes (m = mean MD bytes, -L only)
    kernel_ms = float(np.mean(kms))
    roof_kernel = "col_tile_kernel"
    if kernel_ms <= 0.0:   # ordered front end (-F / -A / TieBrush-made inputs / --store-frac): no tile kernel ran; quote the whole step
        kernel_ms, roof_kernel = ms_step, "whole step (ordered front end, col_ordered_kernel dominant)"
    achieved = a_col / (kernel_ms / 1000.0) / 1e9
    roofline = {"bound": "hbm", "kernel": roof_kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (lambda t: None if (t is None or roof_kernel != "col_tile_kernel" or args.mode != 0) else t * n)(traffic_per_record("col_tile_kernel")),
                "traffic_source": "ncu dram__bytes_read.sum+dram__bytes_write.sum per record at 100x2M (profiles/traffic.json) x records of this launch",
                "peak_source": peak_src, "kernel_ms": kernel_ms, "algorithmic_bytes": a_col,
                "layout_bytes": n * (14 + 4 * cbar) + 16 * G}
    line = {"metric": "alignments_collapsed_per_sec", "value": value, "unit": "alignments/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if (strong or world == 1) else "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"{'C2' if (args.mode == 0 and args.flag_mask == 0 and args.min_qual < 0 and args.max_nh == 0x7fffffff) else 'C3'}: {k} RNA-seq samples x {reads} spliced 150bp reads on chr1, tiebrush mode {args.mode} (0=default CIGAR, 1=-L, 2=-P, 3=-E)"
                                   + (f", -N {args.max_nh}" if args.max_nh != 0x7fffffff else "") + (f", -Q {args.min_qual}" if args.min_qual >= 0 else "")
                                   + (f", -F {args.flag_mask}" if args.flag_mask else "") + (f"; the ONE cohort sharded by coordinate (cuts at coverage gaps) over {world} GPUs, groups gathered on rank 0 over NCCL" if strong else ", one window per GPU"),
                       "front_end_path": int(ctx.last_path()) if hasattr(ctx, "last_path") else None,
                       "tile_gen": int(ctx.last_tile_gen()), "heavy_slots": int(ctx.last_heavy_slots()), "tile_stats": ctx.last_tile_stats(),
                       "records_per_step": n_total, "records_per_step_per_gpu": n, "groups_out": int(res.get("groups_all_ranks", G)), "groups_this_rank": G, "mean_cigar_ops": cbar, "l2": "inputs (>=20 GB at full size) exceed the 126 MB L2; no flush needed",
                       "parallelism": (f"one cohort, coordinate shards x{world} cut at coverage gaps; all_gather of the group counts + batched NCCL send/recv of the groups to rank 0 per step" if strong else f"coordinate shards x{world}, no data-path collective"), "gen_seconds": t_gen, "host_affinity": numa},
            "roofline": roofline, "gpu_launches": int(launches), **({"per_rank": per_rank} if per_rank else {}),
            "stage_ms": dict(zip(("hist_scan", "slots_offsets", "tile", "compaction", "yd"), [float(x) for x in np.mean(np.asarray(stages), 0)]))}
    if tiecov_line is not None:
        line["tiecov"] = tiecov_line

    # the CPU baseline's bounded sample is cut from the device-resident window before the e2e leg frees it
    cpu_sub = None
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        cpu_sub = synth.prefix_slice(cols, run_off, args.cpu_sample)
    # ---- end to end through the C ABI with host buffers ----
    host = None
    if not args.no_e2e:
        host = {}
        h2d = 0
        ok = 1
        try:   # pinned host copies of every input column (25 GB per rank at full size): all ranks must succeed, or all skip
            del out, res   # 16 GB of device output columns at full size: not needed by the host-buffer leg
            out = res = None
            torch.cuda.empty_cache()
            wire_cols = dict(cols)
            names = ("pos", "flag", "mapq", "strand", "nh", "cig_off", "cigar")
            if args.wire in ("compact", "packed"):   # what a host packer would fill directly; built here from the wide columns
                wire_cols["n_cigar8"], wire_cols["cigar16"], wire_cols["cigar_ext"] = api.compact_cigar_columns(cols["cig_off"], cols["cigar"])
                names = ("pos", "flag", "mapq", "strand", "nh", "n_cigar8", "cigar16", "cigar_ext")
            meta_dict = None
            if args.wire == "packed":
                pk = api.pack_fixed_columns(cols, run_off)
                meta_dict = pk.pop("meta_dict")
                wire_cols.update(pk)
                names = ("pos_d8", "pos_ext", "meta8", "meta_ext", "n_cigar8", "cigar16", "cigar_ext")
            for name in names + (("md_off", "md") if args.mode == 1 else ()):
                t = wire_cols[name]
                ht = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                ht.copy_(t)
                host[name] = ht.numpy().view({"cig_off": np.uint32, "cigar": np.uint32, "md_off": np.uint32, "flag": np.uint16, "nh": np.uint16, "cigar16": np.uint16, "cigar_ext": np.uint32, "meta_ext": np.uint64}.get(name, ht.numpy().dtype))
                h2d += ht.numel() * ht.element_size()
            cap = max(G + 1024, 1)
            hout_t = dict(rep_index=torch.empty(cap, dtype=torch.int32, pin_memory=True), yc=torch.empty(cap, dtype=torch.float32, pin_memory=True),
                          yx=torch.empty(cap, dtype=torch.int32, pin_memory=True), yd=torch.empty(cap, dtype=torch.int32, pin_memory=True))
            # the same window as coordinate sub-windows cut at coverage gaps (what the host tool hands over), packed and pinned
            subs_host = []
            if args.e2e_windows > 1 and args.mode != 1:
                for sub, ro_s, pr_s in gap_cut_subwindows(cols, run_off, pr, args.e2e_windows, dev):
                    hs, nb = pin_wire(api, sub, ro_s, args.wire)
                    ns = int(ro_s[-1])
                    capg = int(0.5 * ns) + (1 << 20)
                    ho = dict(rep_index=torch.empty(capg, dtype=torch.int32, pin_memory=True).numpy().view(np.uint32), yc=torch.empty(capg, dtype=torch.float32, pin_memory=True).numpy(),
                              yx=torch.empty(capg, dtype=torch.int32, pin_memory=True).numpy().view(np.uint32), yd=torch.empty(capg, dtype=torch.int32, pin_memory=True).numpy())
                    subs_host.append((hs, ro_s, pr_s, ho, nb, ns))
                    del sub
                torch.cuda.empty_cache()
        except (RuntimeError, MemoryError) as ex:
            ok = 0
            e2e_err = str(ex)[:200]
        if world > 1:
            t = torch.tensor([ok], device=dev, dtype=torch.int32)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ok = int(t.item())
        if not ok:
            host = None
            line["e2e"] = {"unavailable": "host buffers for the end-to-end leg could not be prepared on every rank" + (": " + e2e_err if "e2e_err" in dir() else "")}
        else:
            host["n_cig"] = n_cig
            if meta_dict is not None:
                host["meta_dict"] = meta_dict
                h2d += meta_dict.nbytes
            if args.mode == 1:
                host["n_md"] = int(cols["n_md"])
            # the device-resident copy is not needed any more: the host path stages its own (full size: 25 GB each)
            del cols, out, res, wire_cols
            torch.cuda.empty_cache()
            hout = {kk: v.numpy().view(np.uint32) if kk in ("rep_index", "yx") else v.numpy() for kk, v in hout_t.items()}
            es = args.steps
            ctx.collapse_window(host, run_off, pos_range=pr, out=hout)  # warm the staging buffers
            barrier()
            t0 = time.perf_counter()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                g0.record(stream)
                for _ in range(es):
                    r2 = ctx.collapse_window(host, run_off, pos_range=pr, out=hout)
                g1.record(stream)
            barrier()
            e2e_ms = g0.elapsed_time(g1) / es
            if world > 1:
                t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                e2e_ms = float(t.item())
            single = {"ms_per_step": e2e_ms, "value": n_total / (e2e_ms / 1000.0), "h2d_bytes_per_step": int(h2d), "what": "ONE tb_collapse_window call on the whole window of this rank: every copy before the first kernel"}
            g_tot = r2["n_groups"]
            n_sw = 1
            if subs_host:
                # ---- pipelined hand-over: sub-windows alternate between two contexts (two host threads, two streams): the
                # host->device copies of one sub-window overlap the kernels of the other ----
                import threading
                host = None
                stream2 = torch.cuda.Stream(device=dev)
                ctx2 = api.Context(device=local, n_samples=k, mode=args.mode, flag_mask=args.flag_mask, max_nh=args.max_nh, min_qual=args.min_qual)
                ctx2.set_stream(stream2.cuda_stream)
                pair = ((ctx, stream), (ctx2, stream2))
                n_sw = len(subs_host)
                res_sw = [None] * n_sw

                def work(ci, e_end):
                    c, st_ = pair[ci]
                    for i in range(ci, n_sw, 2):
                        hs, ro_s, pr_s, ho, _, _ = subs_host[i]
                        res_sw[i] = c.collapse_window(hs, ro_s, pos_range=pr_s, out=ho)
                    if e_end is not None:
                        e_end.record(st_)

                def one_step(e_ends):
                    th = [threading.Thread(target=work, args=(ci, e_ends[ci] if e_ends else None)) for ci in range(2)]
                    for t_ in th: t_.start()
                    for t_ in th: t_.join()

                one_step(None)   # warm both contexts' staging buffers
                barrier()
                t0 = time.perf_counter()
                ms_steps = []
                for _ in range(es):
                    ea, eb, e0 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                    torch.cuda.synchronize()
                    e0.record(stream)
                    stream2.wait_event(e0)
                    one_step((ea, eb))
                    torch.cuda.synchronize()
                    ms_steps.append(max(e0.elapsed_time(ea), e0.elapsed_time(eb)))
                barrier()
                e2e_ms = float(np.mean(ms_steps))
                if world > 1:
                    t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    e2e_ms = float(t.item())
                h2d = sum(x[4] for x in subs_host)
                g_tot = sum(r_["n_groups"] for r_ in res_sw)
                assert g_tot == r2["n_groups"], f"sub-windows gave {g_tot} groups, the one window {r2['n_groups']}"
                ctx2.close()
            d2h = 16 * g_tot + 128 * n_sw
            if world > 1:   # whole-job byte counts
                t = torch.tensor([float(h2d), float(d2h)], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
                h2d, d2h = int(t[0].item()), int(t[1].item())
            line["e2e"] = {"value": n_total / (e2e_ms / 1000.0), "unit": "alignments/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                           "ms_per_step": e2e_ms, "steps": es, "wall_ms_per_step": 1000.0 * (time.perf_counter() - t0) / es,
                           "windows": n_sw, "hand_over": ("%d coordinate sub-windows cut at coverage gaps, two in flight on two contexts / streams (copies of one overlap the kernels of the other)" % n_sw) if n_sw > 1 else "one call",
                           "single_call": single,
                           "wire_format": args.wire + {"packed": " (pos_d8 + meta8 with dictionary / escapes, n_cigar8 + cigar16 + cigar_ext; the device rebuilds every wide column inside the timed region)",
                                                       "compact": " (n_cigar8 + cigar16 + cigar_ext; the device rebuilds cig_off / cigar inside the timed region)", "wide": " (cig_off + cigar u32)"}[args.wire]}
    sampler.stop_flag.set(); sampler.join(timeout=3)
    line["clocks"] = clocks.summary()

    # ---- CPU baseline: the oracle port on a bounded coordinate slice of the same window (rank 0, N=1 only) ----
    if cpu_sub is not None:
        from oracle import oracle
        sub, sub_off = cpu_sub
        t0 = time.perf_counter()
        ro = oracle.collapse(sub, sub_off, mode=args.mode)
        dt = time.perf_counter() - t0
        ns = len(sub["pos"])
        line["cpu_baseline"] = {"value": ns / dt, "unit": "alignments/s", "cores": 1, "kind": "port",
                                "sample": f"coordinate slice of the same window: {ns} records of all {k} samples ({dt:.1f} s); C port of the reference algorithm (oracle/tb_oracle.c), no BAM decode"}
    # ---- the reference's command line over the C ABI (tiebrush_b200/host), same bounded SAM sample as --impl reference:
    #      wall time with host decode / pack / device / tag+write broken out (rank 0, N=1 only) ----
    if rank == 0 and world == 1 and args.cli_reads > 0:
        line["host_cli"] = run_host_cli(args)
    if rank == 0:
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
