"""Runs of identical neighbours in the synthetic cohort, on the CPU: what the tile kernel's run heads should save.

For S samples of `synth.cohort_window` (the benchmark's per-sample distribution) it prints, as one JSON line:
  dup_frac         records identical to the previous record of the same sample (same position, strand and raw CIGAR):
                   the records that join a run instead of probing the group table
  heads_per_step   run heads per 32-record step of a sample's list (a run never crosses a step; the kernel's steps are
                   cut at warp ranges rather than at multiples of 32, which changes this a little), mean and the share of
                   steps with at most 4 heads
  depth classes    share of records at start positions deeper than one slot (the single-position sub-tile) and deeper
                   than the heavy threshold (the full-size relaunch), depths scaled to the 100 x 10M cohort,
                   plus the median number of distinct alignments per position in each class
Filters are not applied (the default options keep every record of the synthetic cohort).

  python tools/tile_run_stats.py --samples 3 --reads 10000000
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tiebrush_b200 import synth  # noqa: E402


def tile_geometry(k, smem_optin=227 * 1024):
    """(E, T, heavy_records) of the tile kernel's 256-thread geometry for k samples (col_front_tile)."""
    W = (k + 31) // 32
    limit = (smem_optin + 1024) // 4 - 1024 - 512
    E = 8192
    while E > 64 and E * (26 + 4 * W) + (6 * k + 1) * 4 + 64 > limit:
        E -= 64
    return E, ((E - 1) * 4 // 5) * 7 // 8, 24 * E


def key_hash(host):
    """64-bit hash of (position, strand, raw CIGAR words) per record."""
    off = host["cig_off"].astype(np.int64)
    cig = host["cigar"].astype(np.uint64)
    n = len(off) - 1
    rec = np.repeat(np.arange(n), np.diff(off))
    j = (np.arange(len(cig)) - off[rec]).astype(np.uint64)
    with np.errstate(over="ignore"):
        mixed = (cig + np.uint64(0x9E3779B97F4A7C15) * (j + np.uint64(1))) * np.uint64(0xBF58476D1CE4E5B9)
        mixed ^= mixed >> np.uint64(31)
        h = np.zeros(n, np.uint64)
        nz = np.diff(off) > 0
        h[nz] = np.add.reduceat(mixed, off[:-1][nz])
        h ^= host["pos"].astype(np.uint64) * np.uint64(0x94D049BB133111EB)
        h ^= host["strand"].astype(np.uint64) << np.uint64(56)
        h += np.diff(off).astype(np.uint64) << np.uint64(48)
    return h


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--samples", type=int, default=3)
    ap.add_argument("--reads", type=int, default=2_000_000, help="reads per sample")
    ap.add_argument("--cohort", type=int, default=100, help="samples of the cohort the depths are scaled to")
    ap.add_argument("--cohort-reads", type=int, default=10_000_000, help="reads per sample of that cohort")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    S, R = args.samples, args.reads
    cols, run_off, _ = synth.cohort_window(S, R, seed=args.seed, device="cpu")
    host = synth.to_host(cols)
    n = len(host["pos"])
    h = key_hash(host)
    file_of = np.repeat(np.arange(S), np.diff(run_off))
    dup = np.zeros(n, bool)
    dup[1:] = (h[1:] == h[:-1]) & (file_of[1:] == file_of[:-1])
    # 32-record steps of every sample's list: a record at a step's first lane is always a head
    idx_in_file = np.arange(n) - run_off[file_of]
    head = ~dup | (idx_in_file % 32 == 0)
    step_id = file_of.astype(np.int64) * ((R + 31) // 32) + idx_in_file // 32
    heads_per_step = np.bincount(step_id, weights=head)[np.unique(step_id)]
    # depth classes at the cohort size
    E, T, heavy = tile_geometry(args.cohort)
    pos_u, pos_inv, depth = np.unique(host["pos"], return_inverse=True, return_counts=True)
    scaled = depth * (args.cohort / S) * (args.cohort_reads / R)
    rec_scaled = scaled[pos_inv]
    groups = np.unique(np.stack([pos_inv, h.view(np.int64)]), axis=1)[0]
    gpp = np.bincount(groups, minlength=len(pos_u))
    out = dict(samples=S, reads_per_sample=R, records=n, cohort=args.cohort, cohort_reads=args.cohort_reads, table_entries=E, slot_records=T,
               heavy_records=heavy,
               dup_frac=round(float(dup.mean()), 4),
               heads_per_step_mean=round(float(heads_per_step.mean()), 2),
               steps_le4_heads=round(float((heads_per_step <= 4).mean()), 4),
               head_ratio=round(float(head.mean()), 4),
               records_deeper_than_slot=round(float((rec_scaled > T).mean()), 4),
               records_deeper_than_heavy=round(float((rec_scaled > heavy).mean()), 4),
               median_groups_deeper_than_slot=int(np.median(gpp[scaled > T])) if (scaled > T).any() else 0,
               median_groups_deeper_than_heavy=int(np.median(gpp[scaled > heavy])) if (scaled > heavy).any() else 0)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
