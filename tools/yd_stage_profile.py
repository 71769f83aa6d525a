"""Per-kernel budget of the YD stage (C7) of one collapse step of the bench cohort (100 samples x 10M reads, the C2 window).
Warm-up collapses, a few plain steps timed with the library's stage events (stage_ms.yd), then ONE step under torch.profiler
(CUDA activities) in a run of its own. Every kernel and memset between the start of yd_desc_kernel and the end of
yd_combine_kernel belongs to the stage. Per kernel: device time, launches, and the bytes the code requests, from the shapes
(groups G, chain members, sub-chains, compact length Lc, 1024-group blocks; Context.last_yd_stats()), per member or per
group. Gathers are counted at their useful size, not at the 32-byte sector each one costs. Records the card name and
power limit. Prints one JSON object (and writes it to --out when given).
Run on a GPU: python tools/yd_stage_profile.py --out yd_stage.json"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def byte_model(name, s):
    """(unit, bytes per unit) the kernel `name` requests at the shapes `s`; None when not modelled (tiny launches)."""
    G, M, W, T = s["groups"], s["n_members"], s["W"], s["nblk"] * s["nchains"]
    per_g = lambda b: ("group", b)
    per_m = lambda b: ("member", b)
    if name == "yd_desc_kernel":   # rep, pos, cig_off pair, CIGAR ops, strand; descriptor, genomic end / start, strand
        return per_g(4 + 4 + 8 + 4 * s["cig_ops_per_record"] + 1 + 32 + 4 + 4 + 1)
    if name.startswith("tb_scan") and "UPopIn" in name:   # union bitmap word (reduce, down) and its rank prefix
        return ("U word", 4 if "reduce" in name else 8)
    if name == "yd_count_kernel":   # every word-warp reads its bit word, the strand and (fused pass) the group end
        return per_g(W * (4 + 1 + (4 if s["fused"] else 0)) + (T * (8 if s["fused"] else 4)) / G)
    if name.startswith("tb_scan") and ("CntIn" in name or "EndMaxIn" in name):   # one (chain, block) table entry
        return ("table entry", 4 if "reduce" in name else (12 if "CntIn" in name else 8))
    if name == "yd_scatter_kernel":   # bits, strand (+ start / end) per word-warp; group id (+ flag) per member
        if s["fused"]:
            return per_m(4 + 4 + (G * W * (4 + 1 + 8) + T * 12) / M)
        return per_m(4 + (G * W * (4 + 1) + T * 8) / M)
    if name == "yd_fill_mchain_kernel":
        return per_m(2)
    if name == "yd_compact_kernel":   # descriptor in / out, 5-7 rank lookups (U word + prefix) (+ compact end / start)
        return per_g(32 + 32 + 6 * 8 + (0 if s["fused"] else 8))
    if name == "yd_heads_kernel":   # group id, chain id, gathered end and start; flag; head slot
        return per_m(4 + 2 + 4 + 4 + 4 + 4 * s["n_subchains"] / M)
    if name.startswith("tb_scan") and "HeadIn" in name:   # flag read (reduce, down); head slot
        return per_m(4 if "reduce" in name else 4 + 4 * s["n_subchains"] / M)
    if name == "yd_frontier_kernel":   # group id, flag, gathered descriptor, compact start (link words not counted)
        return per_m(4 + 4 + 32 + 4)
    if name.startswith("tb_scan") and "LastZeroIn" in name:   # 512-bit link block (+ its prefix)
        return ("512-bit block", 64 if "reduce" in name else 72)
    if name == "yd_lookup_kernel":   # compact start, flag, group id, gathered link word (+ block prefix), atomicMax
        return per_m(4 + 4 + 4 + 8 + 4)
    if name == "yd_combine_kernel":
        return per_g(12)
    return None


def short_name(full):
    """kernel name without arguments; scans keep their input functor, the frontier its template argument"""
    base = re.sub(r"^void\s+", "", full.replace("(anonymous namespace)::", "")).split("(")[0]
    m = re.match(r"([A-Za-z_0-9:]+)(<.*>)?$", base)
    if not m:
        return base
    head = m.group(1).split("::")[-1]
    targs = m.group(2) or ""
    if head.startswith("tb_scan"):
        fn = re.findall(r"\b(\w+In)\b", targs)
        op = re.findall(r"\b(Op\w+)", targs)
        return f"{head}[{fn[0] if fn else (op[0] if op else '')}]"
    if targs:
        return f"{head}{targs}"
    return head


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=100)
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per sample")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5, help="plain steps timed with the stage events (before the profiled step)")
    ap.add_argument("--out", default=None, help="also write the JSON object to this file")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    from tiebrush_b200 import api, synth
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
    k = args.samples
    dev = torch.device("cuda", 0)
    cols, run_off, pr = synth.cohort_window(k, args.reads, seed=0, device=dev)
    n = int(cols["pos"].shape[0])
    out = dict(rep_index=torch.empty(n, dtype=torch.int32, device=dev), yc=torch.empty(n, dtype=torch.float32, device=dev),
               yx=torch.empty(n, dtype=torch.int32, device=dev), yd=torch.empty(n, dtype=torch.int32, device=dev))
    res = dict(gpu=gpu, samples=k, reads_per_sample=args.reads, records=n, yd_path_env=os.environ.get("TB_YD_PATH", ""))
    with api.Context(device=0, n_samples=k) as ctx:
        ctx.set_profiling(True)
        for _ in range(args.warmup):
            r = ctx.collapse_window(cols, run_off, pos_range=pr, out=out)
        yd_ms, step_ms = [], []
        for _ in range(args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = ctx.collapse_window(cols, run_off, pos_range=pr, out=out)
            e1.record()
            torch.cuda.synchronize()
            yd_ms.append(ctx.last_kernel_ms(5)); step_ms.append(e0.elapsed_time(e1))
        stats = ctx.last_yd_stats()
        l0 = ctx.launch_count()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            r = ctx.collapse_window(cols, run_off, pos_range=pr, out=out)
            torch.cuda.synchronize()
        launches = ctx.launch_count() - l0
        yd_path = ctx.last_yd_path()
    G = int(r["n_groups"])
    W = (k + 31) // 32
    shapes = dict(groups=G, W=W, nchains=2 * k, cig_ops_per_record=cols["n_cig"] / max(n, 1), **stats)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    evs = [e for e in trace.get("traceEvents", []) if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memset", "gpu_memcpy")]
    evs.sort(key=lambda e: e["ts"])
    t_a = min(e["ts"] for e in evs if "yd_desc_kernel" in e["name"])
    t_b = max(e["ts"] + e["dur"] for e in evs if "yd_combine_kernel" in e["name"])
    stage = [e for e in evs if e["ts"] >= t_a and e["ts"] + e["dur"] <= t_b]
    shapes["fused"] = not any("yd_heads_kernel" in e["name"] for e in stage)
    rows = {}
    for e in stage:
        nm = short_name(e["name"]) if e["cat"] == "kernel" else e["cat"]
        row = rows.setdefault(nm, dict(kernel=nm, ms=0.0, launches=0))
        row["ms"] += e["dur"] / 1e3
        row["launches"] += 1
    u_words = (pr[1] - pr[0] + (1 << 22)) // 32 + 1   # union bitmap: the window's positions plus the slack for exon ends
    blocks512 = (stats["lc"] + 1 + 511) // 512 * 2 * k if stats["lc"] else None   # link bitmaps: one padded region per chain
    units = {"group": G, "member": stats["n_members"], "table entry": stats["nblk"] * 2 * k, "U word": u_words, "512-bit block": blocks512}
    for nm, row in rows.items():
        bm = byte_model(nm.split("<")[0] if not nm.startswith("tb_scan") else nm, shapes)
        if bm is None:
            continue
        unit, b = bm
        row["bytes_per"] = unit
        row["bytes_per_unit"] = round(float(b), 2)
        cnt = units.get(unit)
        if cnt:
            row["gb"] = round(cnt * b / 1e9, 3)
            row["gb_per_s"] = round(cnt * b / 1e9 / (row["ms"] / 1e3), 1) if row["ms"] > 0 else None
    table = sorted(rows.values(), key=lambda x: -x["ms"])
    for row in table:
        row["ms"] = round(row["ms"], 3)
    res.update(yd_path=yd_path, shapes=shapes, plain_steps=dict(ms_per_step=[round(x, 2) for x in step_ms], yd_ms=[round(x, 3) for x in yd_ms],
                                                                   yd_ms_mean=round(float(np.mean(yd_ms)), 3), ms_per_step_mean=round(float(np.mean(step_ms)), 2)),
               profiled_step=dict(launches=launches, yd_kernel_ms_sum=round(sum(x["ms"] for x in table), 3), yd_span_ms=round((t_b - t_a) / 1e3, 3)),
               kernels=table)
    txt = json.dumps(res)
    print(txt)
    if args.out:
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
