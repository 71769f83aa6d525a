/*
 * tiebrush_b200.h — C ABI of the B200-native TieBrush / TieCov hot path.
 *
 * The reference (alevar/tiebrush) has no plugin or FFI surface: its two tools are monolithic main()s.
 * The seam this library sits behind is the pair of call sites inside the two hot loops
 * (SURVEY.md §8b):
 *
 *   tiebrush:  TInputFiles::next()                      src/tmerge.cpp:331-344   (k-way merge)
 *              passes_options()                         src/tiebrush.cpp:532-541 (filters)
 *              addPData() / flushPData()                src/tiebrush.cpp:477-530 (collapse, YC/YX/YD)
 *   tiecov:    bundle logic                             src/tiecov.cpp:443-481
 *              addCov() / flushCoverage(FILE*)          src/tiecov.cpp:194-241
 *              addJunction() / flushJuncs()             src/tiecov.cpp:100-120
 *
 * Everything crossing the boundary is a plain pointer + size. No torch / STL types.
 * Arrays are struct-of-arrays; `on_device` says whether the per-record arrays are host pointers
 * (the library copies them from the caller's buffers on its stream with cudaMemcpyAsync: page-locked
 * buffers travel at PCIe rate, pageable ones at what the driver's bounce buffers give; a caller that wants
 * copies to overlap kernels hands over smaller windows on two contexts, as bench.py's e2e leg does) or
 * device pointers (already resident in HBM; no copy). Small descriptor arrays (run_off, file_merged,
 * meta_dict) are always host memory.
 *
 * Error convention mirrors the reference's GError (gclib/GBase.cpp:31-53): a call returns non-zero,
 * tb_last_error() gives the message, the caller prints it to stderr and exits 1.
 * There is NO CPU fallback anywhere behind this ABI: without a CUDA device tb_create() fails.
 */
#ifndef TIEBRUSH_B200_H_
#define TIEBRUSH_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* merge strategy: enum TMrgStrategy, src/tiebrush.cpp:82-87 */
#define TB_MODE_CIGAR 0 /* default: same CIGAR            (cmpCigar     :306-312) */
#define TB_MODE_FULL  1 /* -L/--full: same CIGAR and MD   (cmpFull      :285-304) */
#define TB_MODE_CLIP  2 /* -P/--clip: CIGAR w/o end S ops (cmpCigarClip :314-332) */
#define TB_MODE_EXON  3 /* -E/--exon: same exon chain     (cmpExons     :334-345) */

/* keep_bits: struct Options, src/tiebrush.cpp:89-98 */
#define TB_KEEP_SUPP      1 /* -S / --keep-supp      keep flag 0x800 */
#define TB_KEEP_SECONDARY 2 /* --keep-secondary      keep flag 0x100 */
#define TB_KEEP_UNMAP     4 /* -M / --keep-unmap     (the reference aborts on a real unmapped read; so does tb_collapse_window) */
#define TB_STORE_FRAC     8 /* --store-frac          YC += 1/NH, summed in double in the reference's arrival order */

#define TB_NO_MAX_NH 0x7fffffff /* Options.max_nh default MAX_INT */

typedef struct tb_ctx tb_ctx;

/* One collapse window: every record, of every input file, whose (tid,start) lies in the window.
 * FILE-MAJOR layout: records of input file f (command-line order = sample index, tmerge.h:26
 * `fidx`) occupy [run_off[f], run_off[f+1]) and appear in file order, i.e. coordinate-sorted by pos;
 * the index inside the run is the record's order in its file. The device performs the k-way merge
 * (tmerge.cpp:331-344) itself from these sorted runs.
 * A window must hold ALL records of each (tid,start) it touches, for every file — including records
 * the filters will drop: they still delay the records queued behind them (SURVEY §9.2). */
typedef struct {
  int64_t  n;              /* records in the window (< 2^31)                                   */
  int32_t  n_files;        /* k                                                                */
  int32_t  tid;            /* reference id shared by all records (bam1_core_t.tid)             */
  const int64_t* run_off;  /* [n_files+1], HOST memory                                         */
  const uint8_t* file_merged; /* [n_files] HOST; 1 = file made by TieBrush (tbMerged,
                                 tmerge.cpp:69-77); NULL = none                                */
  /* per-record arrays, length n */
  const int32_t*  pos;     /* bam1_core_t.pos, 0-based                                         */
  const uint16_t* flag;    /* bam1_core_t.flag                                                 */
  const uint8_t*  mapq;    /* bam1_core_t.qual                                                 */
  const uint8_t*  strand;  /* GSamRecord::spliceStrand() result: '+', '-' or '.' (GSam.cpp:464) */
  const uint16_t* nh;      /* NH tag, 0 when absent, saturated at 65535 (tiebrush.cpp:537)      */
  const uint32_t* cig_off; /* [n+1] word offsets into `cigar`; n_cigar = cig_off[i+1]-cig_off[i] */
  const uint32_t* cigar;   /* packed BAM CIGAR words (len<<4|op), arena of cig_off[n] words      */
  const uint32_t* md_off;  /* TB_MODE_FULL only, [n+1] byte offsets into `md`; a record with     */
  const uint8_t*  md;      /*   md_off[i+1]==md_off[i] has NO MD tag, else bytes incl. the NUL    */
  const uint64_t* qhash;   /* collapse_same (-A) only: 64-bit hash of QNAME, else NULL           */
  const float*    yc_in;   /* records of merged files: YC tag as float (0 = absent); else NULL   */
  const int32_t*  yx_in;   /*   YX tag (1 when absent)                                           */
  const int32_t*  yd_in;   /*   YD tag (0 when absent)                                           */
  int32_t  on_device;      /* 0: arrays above are host pointers; 1: device pointers              */
  int64_t  n_cig;          /* words in `cigar` (== cig_off[n]); the packer knows it, the device need not sync */
  int64_t  n_md;           /* bytes in `md` (== md_off[n]), 0 when unused                         */
  int32_t  pos_lo, pos_hi; /* every record has pos in [pos_lo, pos_hi): the window the packer cut  */
  /* Optional COMPACT WIRE FORMAT of the two CIGAR columns (host->device copies are the end-to-end bound: 24.8 -> 17.4 bytes
   * per alignment on the synthetic cohort). Either replaces its wide counterpart when that one is NULL; the device
   * rebuilds cig_off / cigar before anything else runs, so results are identical by construction.
   *   n_cigar8  [n]       ops per record (every record < 256 ops)                       replaces cig_off
   *   cigar16   [n_cig]   op | len << 4 per op, len < 4095; len field 0xFFF = the length  replaces cigar
   *   cigar_ext [n_ext]   is the next entry of cigar_ext (full 28-bit lengths, in op order) */
  const uint8_t*  n_cigar8;
  const uint16_t* cigar16;
  const uint32_t* cigar_ext;
  int64_t  n_ext;
  /* PACKED WIRE FORMAT of the fixed columns (optional, round 2: 14 -> 3 bytes per alignment over PCIe; with the compact
   * CIGAR columns a spliced 150-bp read costs ~8.4 bytes instead of 24.8). Each group replaces its wide columns when those
   * are NULL; the device rebuilds pos / flag / mapq / strand / nh first, so results are identical by construction.
   *   pos_d8    [n]  0..253 = pos minus the pos of the previous record of the same file; 254 = that difference is the next
   *                  entry of pos_ext; 255 = the next entry of pos_ext is the ABSOLUTE pos (mandatory for the first record
   *                  of every file's run, allowed anywhere)
   *   pos_ext   [n_pos_ext]  in record order
   *   meta8     [n]  0..254 = index into meta_dict; 255 = the next entry of meta_ext
   *   meta_dict [n_meta_dict <= 255], HOST memory; an entry = flag | mapq << 16 | strand << 24 | (uint64)nh << 32
   *   meta_ext  [n_meta_ext]  same encoding, in record order */
  const uint8_t*  pos_d8;
  const int32_t*  pos_ext;
  int64_t  n_pos_ext;
  const uint8_t*  meta8;
  const uint64_t* meta_dict;
  int32_t  n_meta_dict;
  const uint64_t* meta_ext;
  int64_t  n_meta_ext;
} tb_soa_in;

/* Collapsed groups of one window in FINAL OUTPUT ORDER (flushPData order, tiebrush.cpp:501-530).
 * The caller keeps the raw records of the window, and for group g writes record rep_index[g]
 * with tags YC:f=yc[g], YX=yx[g] and, when yd[g]>0, YD=yd[g] (else YD removed). */
typedef struct {
  int64_t   capacity;   /* in : entries the arrays below can hold (n is always enough)          */
  int64_t   n_groups;   /* out: groups written (outCounter)                                      */
  int64_t   n_kept;     /* out: records that passed the filters (inCounter, tiebrush.cpp:573)    */
  uint32_t* rep_index;  /* out: window index of the representative record                        */
  float*    yc;         /* out: (float)accYC — bam_aux_update_float writes type 'f'              */
  uint32_t* yx;         /* out: popcount(samples)+accYX                                          */
  int32_t*  yd;         /* out: max upstream bundle extent, 0 = no tag                           */
  int32_t   on_device;  /* 0: host arrays; 1: device arrays                                      */
} tb_groups_out;

/* The YD segment lists (GSegList, tiebrush.cpp:122-253) carried from one collapse window to the next, so that a window
 * may begin at any start position instead of only at a coverage gap. One list per chain: chain c = side * n_samples +
 * sample, side 0 = the '+' list (fsegs), side 1 = the '-' list (rsegs). All arrays are HOST memory.
 * Canonical form, with B = pos_hi + 1 (the smallest 1-based start the next window can hold): the nodes [s, e] (1-based,
 * inclusive, in list order) with e >= B that cover at least two positions or are the list's last node. Nothing else of
 * the lists can change a later distance (merge order, groups, filters and the processRead cache never cross a cut
 * between two start positions). */
typedef struct {
  int32_t  tid;        /* reference id of the lists; -1 = none                                    */
  int32_t  pos_hi;     /* pos_hi of the window that produced them                                 */
  int32_t  n_chains;   /* 2 * n_samples, chain c = side * n_samples + sample                      */
  int64_t  capacity;   /* entries seg_start / seg_end can hold (carry_out)                        */
  int64_t  n_segs;     /* segments; on a capacity error: the number needed                        */
  int64_t* chain_off;  /* [n_chains + 1] segments of chain c: [chain_off[c], chain_off[c+1])      */
  int32_t* seg_start;  /* 1-based, inclusive; canonical form above                                */
  int32_t* seg_end;
} tb_yd_carry;

/* One coverage window: records of a coordinate-sorted (collapsed or raw) stream, unmapped records
 * already dropped (tiecov.cpp:436-438). A window must hold whole bundles (tiecov.cpp:443). */
typedef struct {
  int64_t  n;
  const int32_t*  tid;     /* non-decreasing                                                   */
  const int32_t*  pos;     /* 0-based, non-decreasing within a tid                             */
  const float*    yc;      /* YC tag through bam_aux2f, 1.0 when absent (tiecov.cpp:482-485)    */
  const uint8_t*  strand;  /* spliceStrand(): '+','-','.' (only used for junctions)             */
  const uint32_t* cig_off; /* [n+1]                                                             */
  const uint32_t* cigar;
  int32_t  on_device;
  int64_t  n_cig;          /* words in `cigar` (== cig_off[n]) */
  const int32_t*  end;     /* OPTIONAL, may be NULL: 0-based exclusive end of every record = GSamRecord::end as the host computed
                              it (GSam.cpp:351-417; the north star lists `end` among the packed fields). With it the bundle
                              kernel reads 16 instead of 27 bytes per record and never walks a CIGAR                     */
} tc_soa_in;

/* bedGraph runs, in file order: "chr\tstart0\tend0\t%.3f" (tiecov.cpp:226-241) */
typedef struct {
  int64_t  capacity;
  int64_t  n_runs;     /* out */
  int32_t* tid;
  int32_t* start0;     /* 0-based inclusive */
  int32_t* end0;       /* 0-based exclusive */
  double*  value;
  int32_t  on_device;
} tc_runs_out;

/* junctions in print order (tid,start,end,strand char); print as
 * "chr\t(start-1)\tend\tJUNC%08d\t%.3f\t%c" (tiecov.cpp:91-95) */
typedef struct {
  int64_t  capacity;
  int64_t  n_juncs;    /* out */
  int32_t* tid;
  int32_t* start;      /* exon[i-1].end+1, 1-based */
  int32_t* end;        /* exon[i].start-1          */
  uint8_t* strand;
  double*  value;
  int32_t  on_device;
} tc_juncs_out;

/* ---- lifecycle --------------------------------------------------------------------------- */
/* replaces the globals `options`, `mrgStrategy` (tiebrush.cpp:89-100). Returns NULL on failure;
 * tb_last_error(NULL) then holds the reason. */
tb_ctx* tb_create(int device, int n_samples, int mode, uint32_t flag_mask /* -F */,
                  int max_nh /* -N */, int min_qual /* -Q */, int keep_bits, int collapse_same /* -A */);
void        tb_destroy(tb_ctx*);
const char* tb_last_error(tb_ctx*);

/* Use an externally created CUDA stream (cudaStream_t passed as void*); NULL restores the context's
 * own stream. Lets a caller time calls with its own events. */
int   tb_set_stream(tb_ctx*, void* cuda_stream);
void* tb_get_stream(tb_ctx*);
int   tb_sync(tb_ctx*);

/* ---- tiebrush: merge + collapse of one window --------------------------------------------- */
/* replaces TInputFiles::next + passes_options + addPData + flushPData for the window */
int tb_collapse_window(tb_ctx*, const tb_soa_in* in, tb_groups_out* out);

/* tb_collapse_window for a window cut at any start position: the YD lists start from carry_in (NULL = empty, as in
 * tb_collapse_window) and the lists this window leaves behind are written to carry_out (NULL = not wanted) in the
 * canonical form for B = in->pos_hi + 1. Feeding each window the carry_out of the window before it gives the groups of
 * one call over their union. Rules (a violation returns non-zero with a message and writes nothing):
 *   - carry_in->tid != in->tid: the lists start empty (the reference resets them at a tid change, tiebrush.cpp:586-589);
 *   - on the same tid, in->pos_lo < carry_in->pos_hi is an error (the windows would overlap);
 *   - n_chains != 2 * in->n_files is an error (carry_in and carry_out alike);
 *   - chain_off must be non-decreasing from 0 to n_segs; within a chain the segments must have end >= start, be sorted
 *     and must not overlap (touching segments are allowed);
 *   - carry_out->capacity too small: error, and carry_out->n_segs is set to the number of segments needed (the groups
 *     of `out` are valid; call again with a larger carry_out).
 * A window with no records or no groups returns carry_in re-filtered against its own pos_hi. Host or device columns
 * and the compact / packed wire formats work as in tb_collapse_window. Both YD implementations seed the lists and
 * extract them on the device; without a carry nothing is added to tb_collapse_window's work. */
int tb_collapse_window_carry(tb_ctx*, const tb_soa_in* in, const tb_yd_carry* carry_in, tb_groups_out* out,
                             tb_yd_carry* carry_out);

/* ---- tiecov: coverage, junctions, bedgraph runs of one window ------------------------------ */
/* replaces addCov + flushCoverage + addJunction + flushJuncs; runs / juncs may each be NULL
 * (tiecov without -c / without -j). Returns 2 and an error naming the record for CIGAR ops the
 * reference aborts on (tiecov.cpp:219-220). */
int tc_coverage_window(tb_ctx*, const tc_soa_in* in, tc_runs_out* runs, tc_juncs_out* juncs);

/* ---- tiecov -s: sample heat-map of one window (SURVEY §8f.2) -------------------------------- */
/* replaces addMean + discretize + flushCoverage(pair vector) (tiecov.cpp:155-185, 277-309). `yx` [n] = YX tag of every
 * record (1 when absent, tiecov.cpp:495), host or device like the other columns. rows: runs of equal, non-zero
 * ceil(running mean of YX) per bundle, in file order; value[i] is that integer. The caller prints
 * "chr\tstart0\tend0\t%ld\t%f" with hval = ((float)value / n_samples) * (1.5f - 0.1f) + 0.1f (normalize, :311-318),
 * n_samples = number of @CO SAMPLE lines of the header (load_sample_info, commons.h). */
int tc_sample_window(tb_ctx*, const tc_soa_in* in, const int32_t* yx, tc_runs_out* rows);

/* ---- tiecov over a long stream: windows cut at bundle heads -------------------------------- */
/* `in` = one coordinate-sorted slice (host or device arrays) of any length whose CIGAR arena fits 32-bit offsets. It is
 * processed in windows of at most `window` records; a window whose last bundle is continued by the record behind it
 * leaves that bundle to the next window, so the concatenated rows are those of ONE pass of the reference's loop
 * (tiecov.cpp:435-528). next_tid_pos = {tid, pos} of the record that follows the slice in the stream, or NULL: when it
 * continues the slice's last bundle that bundle is left unprocessed and *consumed < in->n tells the caller where to
 * resume (prepend the rest to the next slice). Rows are written from index 0 of runs / juncs. */
int tc_coverage_stream(tb_ctx*, const tc_soa_in* in, int64_t window, const int32_t* next_tid_pos,
                       tc_runs_out* runs, tc_juncs_out* juncs, int64_t* consumed);

/* ---- several GPUs: one context per GPU, sharded by reference coordinate (SURVEY §8e) ------- */
/* The reference's only parallel mode is tiewrap.py's batch tree (tiewrap.py:42-123); its main loops are sequential. Here a
 * coordinate-sorted stream is split in stream order over `world` ranks (one process or thread per GPU). NCCL carries
 * the open-bundle state (ncclAllGather), the records of a bundle that a cut separated from its head (grouped ncclSend /
 * ncclRecv to the rank that holds the head) and the final ordered gather; everything else is local.
 * tb_comm_unique_id: rank 0 fills 128 bytes (ncclUniqueId) that the launcher distributes; tb_comm_init: every rank,
 * collectively. libnccl.so.2 is loaded at run time; single-GPU use never needs it. */
int tb_comm_unique_id(void* id128);
int tb_comm_init(tb_ctx*, int rank, int world, const void* id128);
int tb_comm_destroy(tb_ctx*);
int tb_comm_rank(tb_ctx*);
int tb_comm_world(tb_ctx*);
/* This rank's slice of the stream as n_segs DEVICE-resident segments in stream order (a rank cuts its slice into segments
 * only at reference-id boundaries; the cuts BETWEEN ranks are arbitrary). Collective. On return runs / juncs hold the rows
 * of the bundles whose first record this rank holds, in stream order: the concatenation over the ranks equals the
 * single-GPU output row for row. Without a communicator (or world 1) it is tc_coverage_stream over the segments. */
int tc_shard_coverage(tb_ctx*, const tc_soa_in* segs, int n_segs, int64_t window, tc_runs_out* runs, tc_juncs_out* juncs);
/* Ordered gather on rank 0 (collective): all_runs / all_juncs (device arrays, rank 0 only, may be NULL elsewhere) receive
 * the rows of rank 0, 1, ... ; junc_base (host, [world+1], every rank) = junctions of the ranks before r, the offset of
 * the global JUNC%08d counter (tiecov.cpp:92-94). */
int tc_shard_gather(tb_ctx*, const tc_runs_out* runs, const tc_juncs_out* juncs, tc_runs_out* all_runs, tc_juncs_out* all_juncs,
                    int64_t* junc_base);
/* tc_shard_coverage with the ordered gather OVERLAPPED with the windows: rank 0's arrays are cut into `world` regions of
 * equal capacity (all_runs->capacity / world rows each), the rows of rank r arrive in region r while rank r is still
 * computing its later windows (one ncclAllGather of the new row counts and one grouped ncclSend / ncclRecv per window, on a
 * second stream). Every rank passes all_runs / all_juncs with the SAME capacities (their arrays may be NULL except on rank
 * 0). region (host, [4 * world], every rank) = for rank r: offset and count of its runs, offset and count of its junction
 * rows; the ordered result is region 0, region 1, ... (not contiguous). Collective. */
int tc_shard_coverage_gather(tb_ctx*, const tc_soa_in* segs, int n_segs, int64_t window, tc_runs_out* runs, tc_juncs_out* juncs,
                             tc_runs_out* all_runs, tc_juncs_out* all_juncs, int64_t* region);
/* Statistics of the last tc_shard_coverage / tc_shard_gather call: 0 lead records received, 1 lead records sent, 2 ranks
 * received from, 3 bytes sent in the halo exchange, 4 records of the seam window, 5 bytes this rank moved in the gather, 6 gather rounds (tc_shard_coverage_gather). */
int64_t tc_shard_stat(tb_ctx*, int which);
/* Windows the last tc_coverage_stream / tc_shard_coverage call processed. */
int64_t tc_stream_windows(tb_ctx*);
/* 1 when the last coverage call took the exact path: some weight was not a multiple of 2^-20 (YC written by `tiebrush
 * --store-frac`), so coverage and junction values were summed as doubles in stream order like the reference does
 * (tiecov.cpp:194-223, :100-112) instead of in 2^-20 fixed point. */
int tc_last_exact(tb_ctx*);

/* ---- measurement helpers ------------------------------------------------------------------ */
/* Kernels launched by this library since the context was created (for bench.py's gpu_launches). */
int64_t tb_launch_count(tb_ctx*);
/* Front end the last tb_collapse_window call ran: 0 = shared-memory tile path (order-independent grouping),
 * 1 = ordered path chosen by the options (-F, -A, TieBrush-made inputs, --store-frac: exact emulation of the reference's
 * per-position sorted-list search in merge order), 2 = ordered path as fallback (a start position with more distinct
 * alignments than one shared-memory table). */
int tb_last_path(tb_ctx*);
/* YD stage of the last tb_collapse_window call: 0 = parallel formulation (frontier recurrence + link bitmaps),
 * 1 = sequential segment lists (degenerate exons / more than 255 exons in a representative, or TB_YD_PATH=seq). */
int tb_last_yd_path(tb_ctx*);
/* Sizes of the YD stage of the last tb_collapse_window call: 0 chain members (one per group, sample and strand list),
 * 1 sub-chains (independent runs of a chain's members), 2 compact length Lc (covered positions; 0 on the sequential
 * path), 3 blocks of 1024 groups the member lists are counted in. -1 for another `which`. */
int64_t tb_last_yd_stat(tb_ctx*, int which);
/* Tile slots of the last call that were redone by the full-size-table launch (pile-up positions with more distinct
 * alignments than a quarter-SM table holds). */
int64_t tb_last_heavy_slots(tb_ctx*);
/* Start positions of the last ordered-path call (tb_last_path() 1 or 2) handed to the one-warp-per-position kernel: those
 * with at least TB_ORD_DEEP records (default 96, counting records the filters drop; 0 sends every position to the
 * one-thread kernel). */
int64_t tb_last_ord_deep(tb_ctx*);
/* Tile kernel generation: 1 once a tb_collapse_window call has run the tile front end (col_tile_kernel, the only
 * generation), 0 before. */
int tb_last_tile_gen(tb_ctx*);
/* Tile statistics: 0, 1 and 2 are always 0; 3 is the number of slots of the last tile-path call that ran the 256-thread
 * geometry (0 before any such call). -1 for another `which`. */
int64_t tb_last_tile_stat(tb_ctx*, int which);
/* Device time in ms of one stage of the last call, measured with CUDA events on the launching stream
 * (enabled by tb_set_profiling(ctx,1)):
 *   0 collapse tile kernel (dominant)      1 coverage accumulate kernel (dominant)
 *   2 collapse C1+C2 histogram+scan        3 collapse C3+C4 slots + run offsets
 *   4 collapse C6 compaction               5 collapse C7 YD (descriptors, bundles, chains)
 *   6 coverage K6 bundles                  7 coverage K8 runs      8 coverage K9 junction extraction
 *   9 tc_shard_coverage: halo exchange (allgathers + send / receive of the lead records)
 * After tc_coverage_stream / tc_shard_coverage, 1, 6 and 7 are sums over the windows of the call. */
int   tb_set_profiling(tb_ctx*, int on);
float tb_last_kernel_ms(tb_ctx*, int which);

const char* tb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* TIEBRUSH_B200_H_ */
