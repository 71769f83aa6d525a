"""BAM decode on the device: a seeded synthetic collapsed BAM (synth.coverage_stream, 150-bp SEQ / QUAL, NH / XS / YC / YX
tags, htslib-style blocks at zlib level 6) through tc_bam_columns and tc_coverage_bam, beside single-core zlib inflate of
the same bytes and tc_coverage_stream on the pre-decoded host columns. Writes one JSON line to <out>/bam_decode_bench.json.

    python tools/bam_decode_bench.py --records 5000000 --out out/
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=5_000_000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--chunk-mb", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="out")
    a = ap.parse_args()
    import torch
    import bam_writer as W
    from tiebrush_b200 import api, synth
    n = a.records
    t0 = time.perf_counter()
    host = synth.to_host(synth.coverage_stream(n, seed=a.seed, n_tx=20000, chroms=4))
    host["yx"] = np.random.default_rng(a.seed).integers(1, 61, n).astype(np.int32)
    buf, ends = W.columns_records(host, l_seq=150)
    names = [f"c{i}" for i in range(4)]
    hdr = W.header_bytes("@HD\tVN:1.6\tSO:coordinate\n" + "".join(f"@SQ\tSN:{x}\tLN:300000000\n" for x in names), names, [300000000] * 4)
    payloads = W.columns_payloads(hdr, buf, ends)
    data = W.bgzf_file(payloads, "l6", threads=os.cpu_count() or 8)
    t_build = time.perf_counter() - t0
    inflated = len(buf) + len(hdr)
    del buf, ends
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "synthetic.bam")
        with open(path, "wb") as f:
            f.write(data)
        h = api.read_bam_header(path)
        body = data[h["block_offset"]:]
        # single-core zlib inflate of the same blocks
        t0 = time.perf_counter()
        o = 0
        while o < len(data):
            bs = int.from_bytes(data[o + 16:o + 18], "little") + 1
            zlib.decompress(data[o + 18:o + bs - 8], -15)
            o += bs
        t_zlib = time.perf_counter() - t0
        with api.Context(device=0) as ctx:
            ctx.set_profiling(True)
            inf, prs, wall = [], [], []
            for _ in range(a.reps + 1):       # the first pass warms up (module load, buffer growth)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                cols, st = ctx.bam_columns(body, h["skip"], last=True)
                torch.cuda.synchronize()
                wall.append(time.perf_counter() - t0)
                inf.append(ctx.last_kernel_ms(10)); prs.append(ctx.last_kernel_ms(11))
                del cols
            inf, prs, wall = inf[1:], prs[1:], wall[1:]
            ctx.set_profiling(False)
            e2e = []
            for _ in range(a.reps + 1):
                t0 = time.perf_counter()
                got = ctx.coverage_bam(path, chunk_bytes=a.chunk_mb << 20)
                e2e.append(time.perf_counter() - t0)
            e2e = e2e[1:]
            cap = 2 * int(host["cig_off"][-1]) + 16
            out = api.cov_out_buffers(cap, cap // 2)
            st_t = []
            for _ in range(a.reps + 1):
                t0 = time.perf_counter()
                ref = ctx.coverage_stream(host, 1 << 22, out)
                st_t.append(time.perf_counter() - t0)
            st_t = st_t[1:]
            same = got["n_runs"] == ref["n_runs"] and got["n_juncs"] == ref["n_juncs"] and all(
                np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(got["runs"] + got["juncs"], ref["runs"] + ref["juncs"]))
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
    except Exception as e:   # the line still says what was measured
        gpu = f"unknown ({e})"
    med = lambda x: float(np.median(x))
    res = dict(metric="bam_decode", gpu=gpu, records=n, bam_bytes=len(data), inflated_bytes=inflated, blocks=int(st["blocks"]),
               build_s=round(t_build, 2),
               inflate_ms=round(med(inf), 3), inflate_gb_s=round(inflated / (med(inf) * 1e-3) / 1e9, 2),
               parse_ms=round(med(prs), 3), parse_records_s=round(n / (med(prs) * 1e-3), 0),
               bam_columns_wall_ms=round(med(wall) * 1e3, 2),
               coverage_bam_s=round(med(e2e), 4), coverage_bam_records_s=round(n / med(e2e), 0), chunk_mb=a.chunk_mb,
               zlib_1core_s=round(t_zlib, 3), zlib_1core_gb_s=round(inflated / t_zlib / 1e9, 3),
               coverage_stream_host_cols_s=round(med(st_t), 4), coverage_stream_records_s=round(n / med(st_t), 0),
               rows_equal_coverage_stream=bool(same), runs=int(got["n_runs"]), juncs=int(got["n_juncs"]),
               timing=dict(inflate_parse="CUDA events around the kernels, median of %d passes after one warm-up" % a.reps,
                           e2e="host clock around Context.coverage_bam(path) (file in the page cache, rows copied to the host)",
                           stream="host clock around coverage_stream on pinned-free numpy columns (H2D per window inside)"))
    line = json.dumps(res)
    print(line)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bam_decode_bench.json"), "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
