// collapse_internal.cuh — stage interfaces of the collapse pipeline (collapse.cu drives them).
#pragma once
#include "tb_record.cuh"

struct ColGeom {
  int64_t n; int k; uint32_t W;       // records, files, 32-bit words per sample bitset
  uint32_t S;                         // window span in positions
  const uint32_t* P;                  // [S+1] merged-order rank of every position (exclusive scan of the histogram)
  const long long* d_runoff;          // [k+1] device copy of run_off
  const uint8_t* d_merged;            // [k] device copy of file_merged (or nullptr)
  long long* d_status;                // CS_* block
};

// dense group outputs of a front end, in final order
struct ColGroups {
  int64_t capacity;
  uint32_t* rep; float* yc; uint32_t* yx; int32_t* yd;   // yd is pre-set by the front end (0, or the carried YD tag maximum)
  uint32_t* bits;                                        // [G*W] direct-sample bitsets (XB_BITS)
};

// YD lists carried across a window cut (tb_collapse_window_carry), device side; a default-constructed value = no carry.
// Chains are c = side * k + sample. The output area is filled in the order the chains reserve their slots; the host
// puts it into chain order.
struct YdCarry {
  bool in = false;                 // lists seeded from carry_in (same tid)
  bool out = false;                // lists wanted back
  int64_t nin = 0;                 // carried segments
  const long long* coff = nullptr; // [nchains+1] carry_in offsets
  const int32_t* cs = nullptr;     // [nin] carry_in segments, 1-based inclusive
  const int32_t* ce = nullptr;
  int32_t* seed = nullptr;         // [nchains] frontier the chain starts from (compact on the parallel path), -1 = none
  int32_t* ext = nullptr;          // [nchains] parallel path: how far the first live carried node reaches below the window
  int32_t* efin = nullptr;         // [nchains] parallel path: frontier after the chain's last member
  int32_t bout = 0;                // B of carry_out = pos_hi + 1
  int64_t cap = 0;                 // entries of os / oe
  int32_t* os = nullptr; int32_t* oe = nullptr;
  long long* ometa = nullptr;      // [2*nchains] first slot and count per chain, then the slot cursor
};

// Fast path: shared-memory hash tiles. Returns 0 ok, 1 error, 2 = group table overflow (caller falls back to the ordered path).
int col_front_tile(tb_ctx* ctx, const ColIn& in, const ColGeom& g, ColGroups& out, int64_t* n_groups, int64_t* n_kept);
// Exact path: sequential emulation of the reference's per-position sorted list, in merge order.
int col_front_ordered(tb_ctx* ctx, const ColIn& in, const ColGeom& g, ColGroups& out, int64_t* n_groups, int64_t* n_kept);
// YD chains over the dense groups.
int col_yd(tb_ctx* ctx, const ColIn& in, const ColGeom& g, const ColGroups& grp, int64_t G, const YdCarry& cy);
