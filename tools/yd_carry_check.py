"""YD carry at scale (tb_collapse_window_carry): one file-major synthetic cohort held in HBM, collapsed
  (a) as one call,
  (b) as N windows cut at record-balanced start positions with the YD lists carried across the cuts (no gap needed),
  (c) as the gap-cut windows of bench.py (independent windows, no carry),
and the concatenated groups compared. Per call: YD stage ms (tb_last_kernel_ms(5)), kernel launches, carried segments.
Prints one JSON object (and writes it to --out when given). Run on the GPU: python tools/yd_carry_check.py --samples 100 --reads 2000000"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_cut_windows(cols, run_off, bounds):
    """Device-resident sub-windows [bounds[i], bounds[i+1]) of a file-major window: per file one contiguous slice."""
    import torch
    k = len(run_off) - 1
    dev = cols["pos"].device
    offs = [cols["cig_off"][int(run_off[f]):int(run_off[f + 1]) + 1].to(torch.int64) & 0xFFFFFFFF for f in range(k)]
    subs = []
    for a0, b0 in zip(bounds[:-1], bounds[1:]):
        bt = torch.tensor([a0, b0], device=dev, dtype=cols["pos"].dtype)
        parts = {kk: [] for kk in ("pos", "flag", "mapq", "strand", "nh", "cig_off", "cigar")}
        ro, base = [0], 0
        for f in range(k):
            a, b = int(run_off[f]), int(run_off[f + 1])
            i0, i1 = (int(v) for v in torch.searchsorted(cols["pos"][a:b], bt))
            for kk in ("pos", "flag", "mapq", "strand", "nh"):
                parts[kk].append(cols[kk][a + i0:a + i1])
            c0, c1 = int(offs[f][i0]), int(offs[f][i1])
            parts["cig_off"].append(offs[f][i0:i1] - c0 + base)
            parts["cigar"].append(cols["cigar"][c0:c1])
            base += c1 - c0
            ro.append(ro[-1] + (i1 - i0))
        sub = {kk: torch.cat(v) for kk, v in parts.items() if kk != "cig_off"}
        sub["cig_off"] = torch.cat(parts["cig_off"] + [torch.tensor([base], device=dev, dtype=torch.int64)]).to(torch.int32)
        sub["n_cig"] = base
        subs.append((sub, np.asarray(ro, np.int64), (a0, b0), [int(x) for x in ro]))
    return subs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=100)
    ap.add_argument("--reads", type=int, default=2_000_000, help="reads per sample")
    ap.add_argument("--windows", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions of every variant (after one warm-up)")
    ap.add_argument("--out", default=None, help="also write the JSON object to this file")
    args = ap.parse_args()
    import torch
    from tiebrush_b200 import api, shard, synth
    import bench
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
    k = args.samples
    dev = torch.device("cuda", 0)
    cols, run_off, pr = synth.cohort_window(k, args.reads, seed=0, device=dev)
    n = int(cols["pos"].shape[0])
    host_pos = cols["pos"].cpu().numpy()
    cuts = shard.collapse_cuts({"pos": host_pos}, run_off, args.windows)
    del host_pos
    carry_subs = device_cut_windows(cols, run_off, [int(pr[0])] + cuts + [int(pr[1])])
    gap_subs = bench.gap_cut_subwindows(cols, run_off, pr, args.windows, dev)
    res = dict(gpu=gpu, samples=k, reads_per_sample=args.reads, records=n, windows=args.windows)
    with api.Context(device=0, n_samples=k) as ctx:
        ctx.set_profiling(True)

        def run(variant):
            """One pass of a variant: groups (host), YD ms / launches / carried segments per call, wall ms."""
            calls, reps, ycs, yxs, yds = [], [], [], [], []
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if variant == "one":
                items = [(cols, run_off, pr, None)]
            elif variant == "carry":
                items = [(s, ro, p, True) for s, ro, p, _ in carry_subs]
            else:
                items = [(s, ro, p, None) for s, ro, p in gap_subs]
            carry = api.empty_yd_carry(k)
            base = 0
            for s, ro, p, use in items:
                l0 = ctx.launch_count()
                r = ctx.collapse_window(s, ro, pos_range=p, yd_carry=carry if use else None)
                c = dict(yd_ms=ctx.last_kernel_ms(5), launches=ctx.launch_count() - l0, groups=r["n_groups"])
                if use:
                    carry = r["yd_carry"]
                    c["carried_segments"] = int(carry["chain_off"][-1])
                calls.append(c)
                reps.append(r["rep_index"].cpu().numpy().view(np.uint32).astype(np.int64) + base)
                ycs.append(r["yc"].cpu().numpy()); yxs.append(r["yx"].cpu().numpy()); yds.append(r["yd"].cpu().numpy())
                base += int(s["pos"].shape[0])
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
            return calls, wall, [np.concatenate(x) for x in (reps, ycs, yxs, yds)]

        out = {}
        for variant in ("one", "carry", "gap"):
            run(variant)   # warm-up
            walls = []
            for _ in range(args.reps):
                calls, wall, groups = run(variant)
                walls.append(wall)
            out[variant] = (calls, walls, groups)
    # groups: rep_index of the cut variants indexes the concatenated sub-windows; compare through the record position and
    # the per-group tags, which identify a group uniquely together with its order
    pos = cols["pos"].cpu().numpy()
    def key(variant, subs):
        calls, walls, (rep, yc, yx, yd) = out[variant]
        if variant == "one":
            p = pos[rep]
        else:
            p = np.concatenate([s[0]["pos"].cpu().numpy() for s in subs])[rep]
        return p, yc, yx, yd
    one = key("one", None)
    for variant, subs in (("carry", carry_subs), ("gap", gap_subs)):
        got = key(variant, subs)
        res[f"{variant}_groups_equal_one_call"] = bool(all(len(a) == len(b) and np.array_equal(a, b) for a, b in zip(one, got)))
    for variant in ("one", "carry", "gap"):
        calls, walls, _ = out[variant]
        res[variant] = dict(calls=len(calls), wall_ms=[round(w, 2) for w in walls], yd_ms_per_call=[round(c["yd_ms"], 3) for c in calls],
                            yd_ms_sum=round(sum(c["yd_ms"] for c in calls), 3), launches_per_call=[c["launches"] for c in calls],
                            groups_per_call=[c["groups"] for c in calls])
        if variant == "carry":
            res[variant]["carried_segments_per_cut"] = [c["carried_segments"] for c in calls[:-1]]
    res["gap_windows_found"] = len(gap_subs)
    txt = json.dumps(res)
    print(txt)
    if args.out:
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
