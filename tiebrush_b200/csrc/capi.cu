// capi.cu — extern "C" entry points of libtiebrush_b200.so (include/tiebrush_b200.h).
#include <stdarg.h>
#include "tb_common.cuh"

std::string g_tb_global_error;

void tb_ctx::set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap; va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  err = buf;
}

int tc_coverage_impl(tb_ctx* ctx, const tc_soa_in* in, tc_runs_out* runs, tc_juncs_out* juncs, const int32_t* yx, CovExt* ext);
int tb_collapse_impl(tb_ctx* ctx, const tb_soa_in* in, tb_groups_out* out, const tb_yd_carry* cin, tb_yd_carry* cout);

// the rules of tb_collapse_window_carry (include/tiebrush_b200.h) for one carry; nonzero = error set
static int yd_carry_invalid(tb_ctx* ctx, const tb_soa_in* in, const tb_yd_carry* c, const char* what) {
  const int nchains = 2 * in->n_files;
  if (c->n_chains != nchains) { ctx->set_error("tb_collapse_window_carry: %s has n_chains %d, the window has %d (2 * n_files)", what, c->n_chains, nchains); return 1; }
  if (!c->chain_off) { ctx->set_error("tb_collapse_window_carry: %s has no chain_off", what); return 1; }
  return 0;
}

static void global_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap; va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_tb_global_error = buf;
}

extern "C" int tb_comm_destroy(tb_ctx* ctx);

extern "C" {

const char* tb_version(void) { return "tiebrush_b200 0.1 (sm_100a)"; }

tb_ctx* tb_create(int device, int n_samples, int mode, uint32_t flag_mask, int max_nh, int min_qual, int keep_bits, int collapse_same) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    global_error("tb_create: no CUDA device (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "count=0");
    return nullptr;
  }
  if (device < 0 || device >= ndev) { global_error("tb_create: device %d out of range (0..%d)", device, ndev - 1); return nullptr; }
  if (mode < 0 || mode > 3) { global_error("tb_create: unknown merge strategy %d", mode); return nullptr; }
  if (max_nh >= 65535 && max_nh != TB_NO_MAX_NH) { global_error("tb_create: -N %d exceeds the saturating u16 NH column (use < 65535)", max_nh); return nullptr; }
  if (n_samples < 1 || n_samples > 65535) { global_error("tb_create: n_samples %d out of range (1..65535)", n_samples); return nullptr; }
  if ((e = cudaSetDevice(device)) != cudaSuccess) { global_error("tb_create: cudaSetDevice: %s", cudaGetErrorString(e)); return nullptr; }
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) { global_error("tb_create: %s", cudaGetErrorString(e)); return nullptr; }
  if (prop.major < 10) { global_error("tb_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); return nullptr; }
  tb_ctx* ctx = new tb_ctx();
  ctx->device = device; ctx->n_samples = n_samples; ctx->mode = mode; ctx->flag_mask = flag_mask; ctx->max_nh = max_nh;
  ctx->min_qual = min_qual; ctx->keep_bits = keep_bits; ctx->collapse_same = collapse_same;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
    global_error("tb_create: cudaStreamCreate: %s", cudaGetErrorString(e)); delete ctx; return nullptr;
  }
  ctx->stream = ctx->own_stream;
  for (int i = 0; i < 16; ++i) cudaEventCreate(&ctx->ev[i]);
  return ctx;
}

void tb_destroy(tb_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (auto& b : ctx->buf) b.release();
  for (auto& b : ctx->in_stage) b.release();
  for (auto& b : ctx->out_stage) b.release();
  for (auto& b : ctx->pinned) b.release();
  for (auto& b : ctx->shard_buf) b.release();
  for (auto& b : ctx->bam_buf) b.release();
  ctx->bam_pinned.release();
  tb_comm_destroy(ctx);
  if (ctx->gather_stream) cudaStreamDestroy(ctx->gather_stream);
  for (int i = 0; i < 16; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
}

const char* tb_last_error(tb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_tb_global_error.c_str(); }

int tb_set_stream(tb_ctx* ctx, void* s) { if (!ctx) return 1; ctx->stream = s ? (cudaStream_t)s : ctx->own_stream; return 0; }
void* tb_get_stream(tb_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int tb_sync(tb_ctx* ctx) {
  if (!ctx) return 1;
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) { ctx->set_error("tb_sync: %s", cudaGetErrorString(e)); return 1; }
  return 0;
}
int64_t tb_launch_count(tb_ctx* ctx) { return ctx ? ctx->launches : 0; }
int tb_last_path(tb_ctx* ctx) { return ctx ? ctx->last_path : -1; }
int tb_last_yd_path(tb_ctx* ctx) { return ctx ? ctx->last_yd_path : -1; }
int64_t tb_last_yd_stat(tb_ctx* ctx, int which) { return (ctx && which >= 0 && which < 4) ? ctx->last_yd_stat[which] : -1; }
int64_t tb_last_heavy_slots(tb_ctx* ctx) { return ctx ? ctx->last_heavy : -1; }
int64_t tb_last_ord_deep(tb_ctx* ctx) { return ctx ? ctx->last_ord_deep : -1; }
int64_t tc_stream_windows(tb_ctx* ctx) { return ctx ? ctx->stream_windows : -1; }
int tc_last_exact(tb_ctx* ctx) { return ctx ? ctx->last_cov_exact : -1; }
int tb_last_tile_gen(tb_ctx* ctx) { return ctx ? ctx->last_tile_gen : -1; }
int64_t tb_last_tile_stat(tb_ctx* ctx, int which) { return (ctx && which >= 0 && which < 4) ? (which == 3 ? ctx->last_tile_slots : ctx->last_tile_runs[which]) : -1; }
int tb_set_profiling(tb_ctx* ctx, int on) { if (!ctx) return 1; ctx->profiling = on; return 0; }
float tb_last_kernel_ms(tb_ctx* ctx, int which) { return (ctx && which >= 0 && which < 16) ? ctx->last_ms[which] : 0.f; }

int tb_collapse_window(tb_ctx* ctx, const tb_soa_in* in, tb_groups_out* out) {
  if (!ctx) return 1;
  if (!in || !out) { ctx->set_error("tb_collapse_window: null argument"); return 1; }
  ctx->err.clear();
  return tb_collapse_impl(ctx, in, out, nullptr, nullptr);
}

int tb_collapse_window_carry(tb_ctx* ctx, const tb_soa_in* in, const tb_yd_carry* cin, tb_groups_out* out, tb_yd_carry* cout) {
  if (!ctx) return 1;
  if (!in || !out) { ctx->set_error("tb_collapse_window_carry: null argument"); return 1; }
  ctx->err.clear();
  if (in->n_files < 1) { ctx->set_error("tb_collapse_window_carry: n_files=%d", in->n_files); return 1; }
  if ((cin || cout) && in->pos_hi <= in->pos_lo) { ctx->set_error("tb_collapse_window_carry: pos_lo/pos_hi not set"); return 1; }
  if (cin) {
    if (yd_carry_invalid(ctx, in, cin, "carry_in")) return 1;
    const int nchains = 2 * in->n_files;
    if (cin->n_segs < 0 || cin->chain_off[0] != 0 || cin->chain_off[nchains] != cin->n_segs) {
      ctx->set_error("tb_collapse_window_carry: carry_in chain_off must run from 0 to n_segs (%lld)", (long long)cin->n_segs); return 1;
    }
    if (cin->n_segs > 0 && (!cin->seg_start || !cin->seg_end)) { ctx->set_error("tb_collapse_window_carry: carry_in has no segments"); return 1; }
    for (int c = 0; c < nchains; ++c) {
      if (cin->chain_off[c + 1] < cin->chain_off[c]) { ctx->set_error("tb_collapse_window_carry: carry_in chain_off decreases at chain %d", c); return 1; }
      for (int64_t q = cin->chain_off[c]; q < cin->chain_off[c + 1]; ++q) {
        if (cin->seg_end[q] < cin->seg_start[q]) { ctx->set_error("tb_collapse_window_carry: carry_in segment %lld has end < start", (long long)q); return 1; }
        if (q > cin->chain_off[c] && cin->seg_start[q] <= cin->seg_end[q - 1]) {
          ctx->set_error("tb_collapse_window_carry: carry_in segments %lld and %lld of chain %d overlap or are unsorted", (long long)q - 1, (long long)q, c); return 1;
        }
      }
    }
    if (cin->tid == in->tid && in->pos_lo < cin->pos_hi) {
      ctx->set_error("tb_collapse_window_carry: pos_lo %d lies before the carried lists' pos_hi %d", in->pos_lo, cin->pos_hi); return 1;
    }
  }
  if (cout) {
    if (yd_carry_invalid(ctx, in, cout, "carry_out")) return 1;
    if (cout->capacity < 0 || (cout->capacity > 0 && (!cout->seg_start || !cout->seg_end))) { ctx->set_error("tb_collapse_window_carry: carry_out has no room"); return 1; }
  }
  return tb_collapse_impl(ctx, in, out, cin, cout);
}

int tc_coverage_window(tb_ctx* ctx, const tc_soa_in* in, tc_runs_out* runs, tc_juncs_out* juncs) {
  if (!ctx) return 1;
  if (!in || (!runs && !juncs)) { ctx->set_error("tc_coverage_window: at least one of runs/juncs required"); return 1; }
  ctx->err.clear();
  return tc_coverage_impl(ctx, in, runs, juncs, nullptr, nullptr);
}

int tc_sample_window(tb_ctx* ctx, const tc_soa_in* in, const int32_t* yx, tc_runs_out* rows) {
  if (!ctx) return 1;
  if (!in || !yx || !rows || (in->n > 0 && !in->yc)) { ctx->set_error("tc_sample_window: in (with yc), yx and rows are required"); return 1; }
  ctx->err.clear();
  return tc_coverage_impl(ctx, in, rows, nullptr, yx, nullptr);
}

}  // extern "C"
