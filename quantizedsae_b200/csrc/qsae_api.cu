// C ABI (include/qsae_b200.h): argument validation, workspace carving, launch sequencing and
// the host-buffer pipeline. No torch types, no exceptions across the boundary.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <new>

#include "../../include/qsae_b200.h"
#include "kernels.h"

using namespace qsae;

namespace qsae {
namespace {
std::atomic<unsigned long long> g_launches{0};
Tuning g_tuning;
bool g_tuning_loaded = false;
int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}
}  // namespace
void reload_tuning() {
  Tuning t;
  t.encode_cluster = env_int("QSAE_ENCODE_CLUSTER", -1);
  t.encode_range = env_int("QSAE_ENCODE_RANGE", 1);
  t.encode_range_pair = env_int("QSAE_ENCODE_RANGE_PAIR", 1);
  t.encode_specialised = env_int("QSAE_ENCODE_SPECIALISED", 1);
  t.prior_prep = env_int("QSAE_PRIOR_PREP", 1);
  t.merge_tier = env_int("QSAE_MERGE_TIER", 0);
  t.sample_div = env_int("QSAE_SAMPLE_DIV", 16);
  if (t.sample_div < 8) t.sample_div = 8;   // the plan samples only when H >= 8 n_sample
  t.dense_step_fused = env_int("QSAE_DENSE_STEP_FUSED", 1);
  t.decode_pair = env_int("QSAE_DECODE_PAIR", -1);
  t.peer_timeout_ms = env_int("QSAE_PEER_TIMEOUT_MS", 20000);
  t.debug_large = getenv("QSAE_DEBUG_LARGE") != nullptr;
  t.debug_pipeline = getenv("QSAE_DEBUG_PIPELINE") != nullptr;
  g_tuning = t;
  g_tuning_loaded = true;
}
void count_launches(int n) { g_launches.fetch_add(static_cast<unsigned long long>(n), std::memory_order_relaxed); }
const Tuning& tuning() {
  if (!g_tuning_loaded) reload_tuning();
  return g_tuning;
}
}  // namespace qsae

namespace {

thread_local char g_err[512] = "";
// optional CUDA events recorded immediately around the fused encoder kernel (bench.py roofline)
thread_local cudaEvent_t g_enc_ev_start = nullptr;
thread_local cudaEvent_t g_enc_ev_stop = nullptr;
// optional per-stage events of qsae_encode_topk / qsae_bsae_forward (qsae_set_stage_events)
thread_local cudaEvent_t g_stage_ev[QSAE_N_STAGE_EVENTS] = {nullptr};
thread_local int g_stage_n = 0;
// qsae_set_unordered_topk: block-level selections (k > QSAE_MAX_K, candidate merges) emit unordered winner sets
thread_local int g_unordered_topk = 0;
inline void stage_mark(int i, cudaStream_t st) {
  if (i < g_stage_n && g_stage_ev[i] != nullptr) cudaEventRecord(g_stage_ev[i], st);
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
int launch_status(const char* what, const char* err) {
  if (err == nullptr) {
    count_launches(1);
    return QSAE_OK;
  }
  return fail(QSAE_ERR_CUDA, "%s: %s", what, err);
}
inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
// carves `bytes` from a workspace at `off` and returns their offset; the next region starts at the aligned end
size_t take(size_t& off, size_t bytes, size_t align = 256) {
  const size_t start = off;
  off = align_up(off + bytes, align);
  return start;
}

int num_sms() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// One fused-kernel + merge stage over a dictionary of H rows.
struct StagePlan {
  int H, k_sel, n_splits, nsub, n_tiles, tiles_per_split, mode, cap, range_g, range_pair;
  size_t cand_off, cnt_off, thr_off, end;
};

enum StageKind { kStageClassBound = 0, kStagePriorMain = 1, kStageSamplePre = 2 };

// The survivor lists of a sweep from `base` on: [B][nsub][cap] entries {float bits, int32 column}, then the counts
// [B][nsub], then the thresholds [B][nsub].
void place_lists(int B, size_t base, StagePlan* sp) {
  const size_t lists = static_cast<size_t>(B) * sp->nsub;
  sp->cand_off = align_up(base, 256);
  sp->cnt_off = sp->cand_off + lists * sp->cap * 8;
  sp->thr_off = sp->cnt_off + lists * 4;
  sp->end = align_up(sp->thr_off + lists * 4, 256);
}

// allow_range (prior-threshold sweeps): the range schedule at small batches; D: width of the contraction (the pair
// variant exists for D = 512 only)
void plan_stage(int B, int H, int k_sel, StageKind kind, size_t base, StagePlan* sp, bool allow_range = false, int D = 0) {
  sp->H = H;
  sp->k_sel = k_sel;
  sp->range_g = 0;
  sp->range_pair = 0;
  sp->n_tiles = (H + kEncBN - 1) / kEncBN;
  sp->n_splits = encode_pick_splits(B, H, num_sms());
  if (kind == kStageSamplePre && (B + kEncBM - 1) / kEncBM >= num_sms()) sp->n_splits = 1;  // enough row blocks
  if (kind == kStageSamplePre && sp->n_splits > 4) sp->n_splits = 4;   // the prior kernel sorts at most 8 x kTopM values per row
  sp->tiles_per_split = (sp->n_tiles + sp->n_splits - 1) / sp->n_splits;
  sp->nsub = sp->n_splits * 2;
  if (kind == kStageSamplePre) {
    sp->mode = 5;   // register-resident class top-2, no survivor buffers: cand region = the kept values
    sp->cap = 0;
    // Large batches stay on the (1 split, row block) grid: the range schedule shortened the pre-pass but doubled the
    // values the prior kernel reads, no gain (profiles/r2s3_measurements.md 3f)
    sp->cand_off = align_up(base, 256);
    sp->cnt_off = sp->thr_off = sp->cand_off;
    sp->end = align_up(sp->cand_off + static_cast<size_t>(B) * sp->nsub * kTopM * 4, 256);
    return;
  }
  if (kind == kStagePriorMain) {
    sp->mode = 4;
    sp->cap = 512;
    // small batches: one CTA per SM over contiguous tile ranges instead of the (split, row block) grid; a list then
    // covers ~1 / nsub of a row's latents (a few dozen survivors), so 256 entries are plenty (a full list is cut
    // exactly in the kernel, as always)
    int range_nsub = 0, range_pair = 0;
    const int g = allow_range ? encode_pick_range(B, H, num_sms(), &range_nsub, D > 448 ? &range_pair : nullptr) : 0;
    if (g > 0) {
      sp->range_g = g;
      sp->range_pair = range_pair;
      sp->nsub = range_nsub;
      sp->cap = 256;
    }
  } else {
    encode_pick_mode(k_sel, &sp->mode, &sp->cap);
    if (sp->tiles_per_split * (kEncBN / 2) <= 448) sp->cap = 512;  // a sub-stream this short cannot fill more
  }
  place_lists(B, base, sp);
}

// Prior threshold = m-th largest pre-activation over a sample of n_sample of the H latents.
// It is too high for a row exactly when >= m sampled latents fall inside the row's top
// (k_sel - 1); that count is ~Binomial(k_sel - 1, n_sample / H). Pick the smallest m whose tail
// probability is below 1e-7 per row (such rows are detected by count and rescued exactly).
int choose_prior_rank(int k_sel, double r) {
  const int n = k_sel - 1;
  if (n <= 0) return 1;
  double pmf = pow(1.0 - r, n), cdf = pmf;
  for (int j = 1; j <= n; ++j) {
    if (1.0 - cdf < 1e-7) return j;
    pmf *= static_cast<double>(n - j + 1) / j * r / (1.0 - r);
    cdf += pmf;
  }
  return n + 1;
}

struct EncodePlan {
  int k_sel, m;
  bool use_prior;
  StagePlan main, pre;
  size_t x_off, prior_off, counters_off, rescue_rows_off, ovf_rows_off, rescue_z_off, total;
};

// shapes the tensor-core encoder takes (b_sae, t_sae): B, H > 0; D a multiple of 8 in [8, 512]
int check_encode_shape(int B, int H, int D) {
  if (B <= 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "B and H must be positive (B=%d H=%d)", B, H);
  if (D < 8 || D > 512 || (D % 8) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "D must be a multiple of 8 in [8, 512], got %d", D);
  return QSAE_OK;
}

int plan_encode(int B, int H, int D, int k, int exact, int n_sample, EncodePlan* pl) {
  const int rc = check_encode_shape(B, H, D);
  if (rc != QSAE_OK) return rc;
  if (k < 1) return fail(QSAE_ERR_INVALID_ARGUMENT, "k must be >= 1, got %d", k);
  if (k > H) return fail(QSAE_ERR_K_OUT_OF_RANGE, "selected index k out of range (k=%d > H=%d)", k, H);
  if (k > kMaxK) return fail(QSAE_ERR_INVALID_ARGUMENT, "k=%d exceeds QSAE_MAX_K=%d on the warp-level path", k, kMaxK);
  int k_sel = k;
  if (exact) {
    k_sel = k + QSAE_RESCORE_MARGIN;
    if (k_sel > kMaxK) k_sel = kMaxK;
    if (k_sel > H) k_sel = H;
  }
  pl->k_sel = k_sel;
  pl->use_prior = false;
  pl->m = 0;
  if (n_sample >= 256 && H >= 8 * static_cast<long long>(n_sample)) {
    const int m = choose_prior_rank(k_sel, static_cast<double>(n_sample) / H);
    // the warp merge holds 512 survivors per row in registers; the prior pays while mean + sigma of the survivor
    // count (m / r, sqrt(m) / r) stays inside (k_sel <= 128 at r = 1 / 16), above that the class-bound modes take over
    const bool fits = (m + sqrt(static_cast<double>(m))) * (static_cast<double>(H) / n_sample) <= 512.0;
    if (m <= kPriorMaxRank && m <= n_sample && fits) {
      pl->use_prior = true;
      pl->m = m;
    }
  }
  size_t off = 0;
  pl->x_off = take(off, static_cast<size_t>(B) * D * 2, 1024);
  plan_stage(B, H, k_sel, pl->use_prior ? kStagePriorMain : kStageClassBound, off, &pl->main, true, D);
  off = pl->main.end;
  pl->counters_off = take(off, 256);
  pl->rescue_rows_off = take(off, static_cast<size_t>(B) * 4);
  if (pl->use_prior) {
    pl->prior_off = take(off, static_cast<size_t>(B) * 4);
    pl->ovf_rows_off = take(off, static_cast<size_t>(B) * 4);
    pl->rescue_z_off = take(off, static_cast<size_t>(kRescueSlots) * H * 4);
    plan_stage(B, n_sample, pl->m, kStageSamplePre, off, &pl->pre);
    off = pl->pre.end;
  }
  pl->total = off;
  return QSAE_OK;
}

EncodeLaunch stage_launch(const StagePlan& sp, int B, int D, int act, const float* bias, uint8_t* ws) {
  EncodeLaunch el{};
  el.B = B; el.H = sp.H; el.D = D; el.k_sel = sp.k_sel;
  el.n_splits = sp.n_splits; el.tiles_per_split = sp.tiles_per_split; el.n_tiles = sp.n_tiles;
  el.nsub = sp.nsub; el.range_g = sp.range_g; el.range_pair = sp.range_pair;
  el.act = act; el.mode = sp.mode; el.cap = sp.cap; el.bias = bias;
  el.cand = ws + sp.cand_off;
  el.cand_cnt = reinterpret_cast<int*>(ws + sp.cnt_off);
  el.cand_thr = reinterpret_cast<float*>(ws + sp.thr_off);
  return el;
}

// Merge of the survivor lists the sweep `el` has just written: k_sel kept per row, the first k_out emitted.
// x_f32, w_f32, bias: the fp32 operands of the exact re-scoring and rescue (or null).
SelectLaunch merge_launch(const EncodeLaunch& el, int k_sel, int k_out, int exact, const float* x_f32, const float* w_f32,
                          const float* bias, float* out_vals, int32_t* out_idx, int32_t* out_flags) {
  SelectLaunch sl{};
  sl.B = el.B; sl.H = el.H; sl.D = el.D; sl.k_sel = k_sel; sl.k_out = k_out; sl.nsub = el.nsub; sl.cap = el.cap;
  sl.act = el.act; sl.exact = exact;
  sl.cand = el.cand; sl.cand_cnt = el.cand_cnt; sl.cand_thr = el.cand_thr;
  sl.x_f32 = x_f32; sl.w_f32 = w_f32; sl.bias = bias;
  sl.out_vals = out_vals; sl.out_idx = out_idx; sl.out_flags = out_flags;
  return sl;
}

// Exact recomputation of the rows the merge `sl` put on its rescue list, into the same outputs
RescueLaunch rescue_launch(const SelectLaunch& sl, const uint16_t* x_bf16, const uint16_t* w_bf16) {
  RescueLaunch rl{};
  rl.B = sl.B; rl.H = sl.H; rl.D = sl.D; rl.k_sel = sl.k_sel; rl.k_out = sl.k_out; rl.act = sl.act; rl.exact = sl.exact;
  rl.x_bf16 = x_bf16; rl.w_bf16 = w_bf16; rl.x_f32 = sl.x_f32; rl.w_f32 = sl.w_f32; rl.bias = sl.bias;
  rl.rescue_count = sl.rescue_count; rl.rescue_rows = sl.rescue_rows;
  rl.out_vals = sl.out_vals; rl.out_idx = sl.out_idx; rl.out_flags = sl.out_flags;
  return rl;
}

int next_pow2_host(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// ---- k > QSAE_MAX_K (e.g. the reference default k = int(0.002 H) = 2097 at H = 2^20, sae/binary.py:94) -----------
// Prior path: top-m over the sampled dictionary rows (class-bound sweep + block merge, m <= QSAE_MAX_K) gives the
// row's threshold; the full sweep keeps everything above it (threshold-only mode, no in-kernel cut); the block-level
// merge radix-selects k_sel of the ~m H / n_sample survivors; rows whose count check fails (or whose lists filled up)
// are recomputed exactly. Dense path (no usable sample): dense pre-activations in row chunks + dense radix select.
struct LargePlan {
  int k_sel, m, chunk_rows;
  bool use_prior;
  StagePlan main, pre, dense;
  size_t x_off, counters_off, rescue_rows_off, pre_vals_off, pre_idx_off, scratch_off, z_off, total;
};

int plan_encode_large(int B, int H, int D, int k, int exact, int n_sample, LargePlan* lp) {
  const int rc = check_encode_shape(B, H, D);
  if (rc != QSAE_OK) return rc;
  if (k > H) return fail(QSAE_ERR_K_OUT_OF_RANGE, "selected index k out of range (k=%d > H=%d)", k, H);
  if (k > kMaxKLarge) return fail(QSAE_ERR_INVALID_ARGUMENT, "k=%d exceeds QSAE_MAX_K_LARGE=%d", k, kMaxKLarge);
  // re-scoring margin: the density of pre-activations around the k-th largest grows with k, so the number of
  // candidates inside the bf16 rounding band does too (k / 4 covers 4 x the band on Gaussian-like rows)
  int k_sel = exact ? k + (k / 4 > QSAE_RESCORE_MARGIN ? k / 4 : QSAE_RESCORE_MARGIN) : k;
  if (k_sel > H) k_sel = H;
  lp->k_sel = k_sel;
  lp->use_prior = false;
  lp->m = 0;
  lp->chunk_rows = 0;
  const int ksort = next_pow2_host(k_sel);
  size_t off = 0;
  lp->x_off = take(off, static_cast<size_t>(B) * D * 2, 1024);
  if (n_sample >= 256 && H >= 8 * static_cast<long long>(n_sample)) {
    const double r = static_cast<double>(n_sample) / H;
    const int m = choose_prior_rank(k_sel, r);
    if (m <= kMaxK && m <= n_sample) {
      plan_stage(B, H, 0, kStagePriorMain, off, &lp->main);
      // survivors of a row = rank of the m-th largest sample value in the full row: mean m / r, standard
      // deviation ~ sqrt(m) / r (negative binomial); a list holds 1 / nsub of them (+ Poisson spread).
      // Lists sized for mean + 7 sigma of both: a filled list costs an exact recomputation of the row.
      const double per_list = (m + 7.0 * sqrt(static_cast<double>(m))) / r / lp->main.nsub;
      int cap = next_pow2_host(static_cast<int>(per_list + 7.0 * sqrt(per_list)) + 64);
      if (cap < 256) cap = 256;
      while (cap > 256 && (static_cast<size_t>(lp->main.nsub) * cap + ksort) * 8 > kSelectSmemBudget) cap >>= 1;
      if ((static_cast<size_t>(lp->main.nsub) * cap + ksort) * 8 <= kSelectSmemBudget &&
          static_cast<long long>(lp->main.nsub) * (cap - 32) >= k_sel) {
        lp->use_prior = true;
        lp->m = m;
        lp->main.cap = cap;
        place_lists(B, off, &lp->main);
      }
    }
  }
  if (lp->use_prior) {
    off = lp->main.end;
    lp->counters_off = take(off, 256);
    lp->rescue_rows_off = take(off, static_cast<size_t>(B) * 4);
    lp->pre_vals_off = take(off, static_cast<size_t>(B) * lp->m * 4);
    lp->pre_idx_off = take(off, static_cast<size_t>(B) * lp->m * 4);
    lp->scratch_off = take(off, rescue_large_scratch_bytes(H, num_sms()));
    plan_stage(B, n_sample, lp->m, kStageClassBound, off, &lp->pre);
    off = lp->pre.end;
  } else {
    // dense pre-activations in row chunks of at most ~1 GB
    long long rows = (1ll << 30) / (static_cast<long long>(H) * 4);
    rows = rows / kEncBM * kEncBM;
    if (rows < kEncBM) rows = kEncBM;
    if (rows > B) rows = B;
    lp->chunk_rows = static_cast<int>(rows);
    lp->z_off = take(off, static_cast<size_t>(rows) * H * 4);
    plan_stage(static_cast<int>(rows), H, 1, kStageClassBound, off, &lp->dense);
    off = lp->dense.end;
  }
  lp->total = off;
  return QSAE_OK;
}

int encode_topk_large(const float* x_f32, const uint16_t* w_bf16, const float* w_f32, const float* b_enc,
                      const uint16_t* w_sample, const float* b_sample, int n_sample, int B, int H, int D, int k, int act,
                      int exact, float* out_vals, int32_t* out_idx, int32_t* out_flags, void* workspace,
                      size_t workspace_bytes, cudaStream_t st) {
  LargePlan lp;
  int rc = plan_encode_large(B, H, D, k, exact, n_sample, &lp);
  if (rc != QSAE_OK) return rc;
  if (workspace_bytes < lp.total)
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "encode_topk: workspace %zu < %zu bytes", workspace_bytes, lp.total);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  uint16_t* x_bf16 = reinterpret_cast<uint16_t*>(ws + lp.x_off);

  if (!lp.use_prior) {
    // ---- dense path
    if (!exact) {
      rc = launch_status("cast x", cast_bf16_launch(x_f32, x_bf16, static_cast<size_t>(B) * D, st));
      if (rc != QSAE_OK) return rc;
    }
    float* z = reinterpret_cast<float*>(ws + lp.z_off);
    for (int r0 = 0; r0 < B; r0 += lp.chunk_rows) {
      const int rows = (B - r0 < lp.chunk_rows) ? (B - r0) : lp.chunk_rows;
      if (exact) {
        rc = launch_status("encode_dense", encode_dense_launch(x_f32 + static_cast<size_t>(r0) * D, nullptr, rows, w_f32,
                                                               b_enc, H, D, act, z, st));
      } else {
        EncodeLaunch el = stage_launch(lp.dense, rows, D, act, b_enc, ws);   // the chunk's split plan, possibly fewer rows
        el.debug_z = z;
        rc = launch_status("encode_topk kernel (dense dump)",
                           encode_topk_launch(x_bf16 + static_cast<size_t>(r0) * D, w_bf16, el, st));
      }
      if (rc != QSAE_OK) return rc;
      rc = launch_status("select_dense", select_dense_launch(z, rows, H, k, num_sms(), out_vals + static_cast<size_t>(r0) * k,
                                                             out_idx + static_cast<size_t>(r0) * k, st));
      if (rc != QSAE_OK) return rc;
    }
    if (out_flags != nullptr) {
      cudaError_t ce = cudaMemsetAsync(out_flags, 0, static_cast<size_t>(B) * 4, st);
      if (ce != cudaSuccess) return fail(QSAE_ERR_CUDA, "encode_topk: %s", cudaGetErrorString(ce));
    }
    return QSAE_OK;
  }

  // ---- prior path
  int* counters = reinterpret_cast<int*>(ws + lp.counters_off);   // [0] rescue rows, [1] sweep overflow flag
  int32_t* rescue_rows = reinterpret_cast<int32_t*>(ws + lp.rescue_rows_off);
  float* pre_vals = reinterpret_cast<float*>(ws + lp.pre_vals_off);
  int32_t* pre_idx = reinterpret_cast<int32_t*>(ws + lp.pre_idx_off);
  cudaError_t ce = cudaMemsetAsync(counters, 0, 4 * sizeof(int), st);
  if (ce != cudaSuccess) return fail(QSAE_ERR_CUDA, "encode_topk: %s", cudaGetErrorString(ce));
  rc = launch_status("cast x", cast_bf16_launch(x_f32, x_bf16, static_cast<size_t>(B) * D, st));
  if (rc != QSAE_OK) return rc;
  // 1. ordered top-m over the sampled rows (tensor-core values: the same arithmetic as the full sweep)
  {
    const EncodeLaunch pe = stage_launch(lp.pre, B, D, act, b_sample, ws);
    rc = launch_status("encode_topk kernel (sample top-m)", encode_topk_launch(x_bf16, w_sample, pe, st));
    if (rc != QSAE_OK) return rc;
    const SelectLaunch sl = merge_launch(pe, lp.m, lp.m, 0, nullptr, nullptr, nullptr, pre_vals, pre_idx, nullptr);
    rc = launch_status("select_topk kernel (sample top-m)", select_topk_launch(sl, st));
    if (rc != QSAE_OK) return rc;
  }
  // 2. full sweep, everything >= the row's m-th largest sample value
  EncodeLaunch el = stage_launch(lp.main, B, D, act, b_enc, ws);
  el.k_sel = 0;
  el.prior = pre_vals + (lp.m - 1); el.prior_stride = lp.m;
  el.overflow = counters + 1;
  if (g_enc_ev_start) cudaEventRecord(g_enc_ev_start, st);
  rc = launch_status("encode_topk kernel", encode_topk_launch(x_bf16, w_bf16, el, st));
  if (g_enc_ev_stop) cudaEventRecord(g_enc_ev_stop, st);
  if (rc != QSAE_OK) return rc;
  // 3. block-per-row merge (radix select), count check
  SelectLaunch sl = merge_launch(el, lp.k_sel, k, exact, x_f32, w_f32, b_enc, out_vals, out_idx, out_flags);
  sl.rescue_count = counters; sl.rescue_rows = rescue_rows; sl.check_count = 1;
  sl.unsorted = g_unordered_topk;
  rc = launch_status("select_topk kernel", select_topk_launch(sl, st));
  if (rc != QSAE_OK) return rc;
  if (tuning().debug_large) {   // diagnostics: survivor statistics of this call (synchronises)
    cudaStreamSynchronize(st);
    int h_counters[4];
    cudaMemcpy(h_counters, counters, sizeof(h_counters), cudaMemcpyDeviceToHost);
    const size_t nl = static_cast<size_t>(B) * lp.main.nsub;
    int* h_cnt = static_cast<int*>(malloc(nl * sizeof(int)));
    cudaMemcpy(h_cnt, el.cand_cnt, nl * sizeof(int), cudaMemcpyDeviceToHost);
    long long tot = 0; int mx = 0, row_min = 1 << 30, row_max = 0;
    for (int r = 0; r < B; ++r) {
      int rs = 0;
      for (int s2 = 0; s2 < lp.main.nsub; ++s2) { const int c = h_cnt[static_cast<size_t>(r) * lp.main.nsub + s2]; rs += c; if (c > mx) mx = c; }
      tot += rs; if (rs < row_min) row_min = rs; if (rs > row_max) row_max = rs;
    }
    fprintf(stderr, "[qsae large] k=%d k_sel=%d m=%d nsub=%d cap=%d: survivors/row mean %.1f min %d max %d, largest list %d; rescued rows %d, sweep overflow %d\n",
            k, lp.k_sel, lp.m, lp.main.nsub, lp.main.cap, static_cast<double>(tot) / B, row_min, row_max, mx, h_counters[0], h_counters[1]);
    free(h_cnt);
  }
  // 4. failed rows: exact recomputation
  return launch_status("rescue kernel (large k)",
                       rescue_large_launch(rescue_launch(sl, x_bf16, w_bf16), ws + lp.scratch_off, num_sms(), st));
}

}  // namespace

extern "C" {

int qsae_abi_version(void) { return QSAE_ABI_VERSION; }
const char* qsae_last_error(void) { return g_err; }

int qsae_check_device(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(QSAE_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10) return fail(QSAE_ERR_UNSUPPORTED_DEVICE, "need an sm_100 device, found sm_%d%d", major, minor);
  return QSAE_OK;
}

int qsae_set_encode_kernel_events(void* start_event, void* stop_event) {
  g_enc_ev_start = reinterpret_cast<cudaEvent_t>(start_event);
  g_enc_ev_stop = reinterpret_cast<cudaEvent_t>(stop_event);
  return QSAE_OK;
}

unsigned long long qsae_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int qsae_default_sample_rows(int H) {
  if (H < 8192) return 0;
  return ((H / tuning().sample_div + 255) / 256) * 256;
}

int qsae_reload_tuning(void) {
  reload_tuning();
  return QSAE_OK;
}

int qsae_set_unordered_topk(int on) {
  g_unordered_topk = on != 0 ? 1 : 0;
  return QSAE_OK;
}

int qsae_set_stage_events(void* const* events, int n) {
  if (n < 0 || n > QSAE_N_STAGE_EVENTS || (n > 0 && !events)) return fail(QSAE_ERR_INVALID_ARGUMENT, "set_stage_events: 0 <= n <= %d", QSAE_N_STAGE_EVENTS);
  g_stage_n = n;
  for (int i = 0; i < n; ++i) g_stage_ev[i] = reinterpret_cast<cudaEvent_t>(events[i]);
  return QSAE_OK;
}

int qsae_cast_f32_to_bf16(const float* src, uint16_t* dst, size_t n, void* stream) {
  if (!src || !dst) return fail(QSAE_ERR_INVALID_ARGUMENT, "cast: null pointer");
  if (n == 0) return QSAE_OK;
  return launch_status("cast_f32_to_bf16", cast_bf16_launch(src, dst, n, S(stream)));
}

int qsae_pack_bitplanes(const float* logits, int H, int D, int n_bits, uint8_t* packed, double* stats,
                        void* stream) {
  if (!logits || !packed) return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_bitplanes: null pointer");
  if (H <= 0 || D <= 0 || n_bits < 1 || n_bits > 8)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_bitplanes: need H,D > 0 and 1 <= n_bits <= 8");
  if (n_bits <= 4 && (D % 2) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_bitplanes: nibble packing needs an even D");
  return launch_status("pack_bitplanes", pack_bitplanes_launch(logits, H, D, n_bits, packed, stats, S(stream)));
}

int qsae_dequant_soft(const float* logits, int H, int D, int n_bits, float* rows, void* stream) {
  if (!logits || !rows) return fail(QSAE_ERR_INVALID_ARGUMENT, "dequant_soft: null pointer");
  if (H <= 0 || D <= 0 || n_bits < 1 || n_bits > 30)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "dequant_soft: bad shape");
  return launch_status("dequant_soft", dequant_soft_launch(logits, H, D, n_bits, rows, S(stream)));
}

int qsae_transpose_f32(const float* src, int R, int C, float* dst, void* stream) {
  if (!src || !dst || R <= 0 || C <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "transpose: bad argument");
  return launch_status("transpose", transpose_launch(src, R, C, dst, S(stream)));
}

int qsae_encode_topk_workspace_bytes(int B, int H, int D, int k, int n_sample, size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  size_t need = 0;
  for (int exact = 0; exact < 2; ++exact) {
    for (int pass = 0; pass < 2; ++pass) {  // with and without the sampled prior
      size_t total = 0;
      if (k > kMaxK) {
        LargePlan lp;
        int rc = plan_encode_large(B, H, D, k, exact, pass ? n_sample : 0, &lp);
        if (rc != QSAE_OK) return rc;
        total = lp.total;
      } else {
        EncodePlan pl;
        int rc = plan_encode(B, H, D, k, exact, pass ? n_sample : 0, &pl);
        if (rc != QSAE_OK) return rc;
        total = pl.total;
      }
      if (total > need) need = total;
    }
  }
  *bytes = need;
  return QSAE_OK;
}

int qsae_prepare_encoder_sample(const uint16_t* w_bf16, const float* b_enc, int H, int D, int n_sample,
                                uint16_t* w_sample, float* b_sample, void* stream) {
  if (!w_bf16 || !b_enc || !w_sample || !b_sample) return fail(QSAE_ERR_INVALID_ARGUMENT, "prepare_encoder_sample: null pointer");
  if (n_sample < 1 || n_sample > H || D < 1) return fail(QSAE_ERR_INVALID_ARGUMENT, "prepare_encoder_sample: need 1 <= n_sample <= H");
  return launch_status("sample_rows", sample_rows_launch(w_bf16, b_enc, H, D, n_sample, w_sample, b_sample, S(stream)));
}

}  // extern "C"

namespace {
// Decode that the merge kernels of the prior path may fuse (qsae_bsae_forward): packed int4 dictionary, D == 512.
struct FusedDecode {
  const uint32_t* packed;
  float scale;
  const float* bias;
  float* recon;
  bool done;   // out: the reconstruction was written by the merge / tail kernels
};

int encode_topk_impl(const float* x_f32, const uint16_t* w_bf16, const float* w_f32, const float* b_enc,
                     const uint16_t* w_sample, const float* b_sample, int n_sample,
                     int B, int H, int D, int k, int act, int exact, float* out_vals, int32_t* out_idx,
                     int32_t* out_flags, void* workspace, size_t workspace_bytes, void* stream,
                     FusedDecode* fd = nullptr) {
  if (B == 0) return QSAE_OK;
  if (!x_f32 || !w_bf16 || !b_enc || !out_vals || !out_idx || !workspace)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "encode_topk: null pointer");
  if (exact && !w_f32) return fail(QSAE_ERR_INVALID_ARGUMENT, "encode_topk: exact mode needs w_f32");
  if (act != QSAE_ACT_NONE && act != QSAE_ACT_RELU)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "encode_topk: unknown activation %d", act);
  if (!w_sample || !b_sample) n_sample = 0;
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0 || (reinterpret_cast<uintptr_t>(w_bf16) & 15) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "encode_topk: workspace must be 256-byte and w_bf16 16-byte aligned");
  if (k > kMaxK && k <= H)
    return encode_topk_large(x_f32, w_bf16, w_f32, b_enc, w_sample, b_sample, n_sample, B, H, D, k, act, exact, out_vals,
                             out_idx, out_flags, workspace, workspace_bytes, S(stream));
  EncodePlan pl;
  int rc = plan_encode(B, H, D, k, exact, n_sample, &pl);
  if (rc != QSAE_OK) return rc;
  if (workspace_bytes < pl.total)
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "encode_topk: workspace %zu < %zu bytes", workspace_bytes, pl.total);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  uint16_t* x_bf16 = reinterpret_cast<uint16_t*>(ws + pl.x_off);
  cudaStream_t st = S(stream);

  int* counters = reinterpret_cast<int*>(ws + pl.counters_off);   // [0] rescue rows, [1] merge overflow rows
  int32_t* rescue_rows = reinterpret_cast<int32_t*>(ws + pl.rescue_rows_off);
  stage_mark(0, st);
  // small batches on the prior path: cast, sample pre-pass, prior and the counter reset are ONE launch
  const int prep_ns = pl.use_prior ? prior_prep_pick_ns(B, D, n_sample, pl.m, num_sms()) : 0;
  if (prep_ns == 0) {
    rc = launch_status("cast x", cast_bf16_launch(x_f32, x_bf16, static_cast<size_t>(B) * D, st));
    if (rc != QSAE_OK) return rc;
    cudaError_t ce = cudaMemsetAsync(counters, 0, kPriorCounters * sizeof(int), st);
    if (ce != cudaSuccess) return fail(QSAE_ERR_CUDA, "encode_topk: %s", cudaGetErrorString(ce));
  }

  if (!pl.use_prior) {
    // ---- class-bound path: one sweep, block-per-row merge
    const EncodeLaunch el = stage_launch(pl.main, B, D, act, b_enc, ws);
    if (g_enc_ev_start) cudaEventRecord(g_enc_ev_start, st);
    rc = launch_status("encode_topk kernel", encode_topk_launch(x_bf16, w_bf16, el, st));
    if (g_enc_ev_stop) cudaEventRecord(g_enc_ev_stop, st);
    if (rc != QSAE_OK) return rc;
    SelectLaunch sl = merge_launch(el, pl.k_sel, k, exact, x_f32, w_f32, b_enc, out_vals, out_idx, out_flags);
    if (exact) { sl.rescue_count = counters; sl.rescue_rows = rescue_rows; }   // uncertified rows only (the bound itself is exact)
    rc = launch_status("select_topk kernel", select_topk_launch(sl, st));
    if (rc != QSAE_OK || !exact) return rc;
    // exact mode: a row whose fp32 re-scoring could not certify the selection is recomputed exactly, as on the
    // prior path (round 1 left such rows flagged with their bf16-chosen candidates)
    return launch_status("rescue kernel", rescue_rows_launch(rescue_launch(sl, x_bf16, w_bf16), num_sms(), st));
  }

  // ---- prior-threshold path
  float* prior = reinterpret_cast<float*>(ws + pl.prior_off);
  int32_t* ovf_rows = reinterpret_cast<int32_t*>(ws + pl.ovf_rows_off);
  if (prep_ns > 0) {
    // 1. cast + sample pre-pass + prior in one cluster launch (prior_prep_kernel)
    PrepLaunch pp{};
    pp.B = B; pp.D = D; pp.n_sample = n_sample; pp.act = act; pp.m = pl.m; pp.ns = prep_ns;
    pp.x_f32 = x_f32; pp.x_bf16 = x_bf16; pp.bias = b_sample; pp.prior = prior; pp.zero_counters = counters;
    rc = launch_status("prior_prep kernel", prior_prep_launch(w_sample, pp, st));
    if (rc != QSAE_OK) return rc;
  } else {
    // 1. pre-pass: the fused kernel over the sampled dictionary rows, top list kept in registers
    EncodeLaunch pe = stage_launch(pl.pre, B, D, act, b_sample, ws);
    pe.top_out = reinterpret_cast<float*>(ws + pl.pre.cand_off);
    rc = launch_status("encode_topk kernel (sample pre-pass)", encode_topk_launch(x_bf16, w_sample, pe, st));
    if (rc != QSAE_OK) return rc;
    rc = launch_status("prior kernel", prior_from_top_launch(pe.top_out, B, pl.pre.nsub, pl.m, prior, st));
    if (rc != QSAE_OK) return rc;
  }
  stage_mark(1, st);
  // 2. full sweep against the prior
  EncodeLaunch el = stage_launch(pl.main, B, D, act, b_enc, ws);
  el.prior = prior; el.prior_stride = 1;
  if (g_enc_ev_start) cudaEventRecord(g_enc_ev_start, st);
  rc = launch_status("encode_topk kernel", encode_topk_launch(x_bf16, w_bf16, el, st));
  if (g_enc_ev_stop) cudaEventRecord(g_enc_ev_stop, st);
  if (rc != QSAE_OK) return rc;
  stage_mark(2, st);
  // 3. merge (warp per row; rows with too many survivors go through the block kernel)
  SelectLaunch sl = merge_launch(el, pl.k_sel, k, exact, x_f32, w_f32, b_enc, out_vals, out_idx, out_flags);
  sl.rescue_count = counters; sl.rescue_rows = rescue_rows; sl.check_count = 1;
  // warp per row: up to 512 survivors in registers (the expected count is ~32 m); rows with more take a two-pass
  // prefilter inside the same warp (round 1 had a second launch with 32 keys per lane for them: 25 us at B = 4096
  // for ~4 % of the rows, more than the first tier). When the caller decodes with the packed int4 dictionary the
  // warp that has just sorted a row also decodes it.
  if (fd != nullptr && D == 512 && k <= 128 && (reinterpret_cast<uintptr_t>(fd->packed) & 15) == 0 &&
      ((reinterpret_cast<uintptr_t>(fd->recon) | reinterpret_cast<uintptr_t>(fd->bias)) & 15) == 0) {
    sl.dec_kind = 1; sl.dec_packed = fd->packed; sl.dec_scale = fd->scale; sl.dec_bias = fd->bias; sl.dec_recon = fd->recon;
    fd->done = true;
  }
  // keys per lane: the survivors of the prior threshold are negative-binomial, m / r on average with a spread of
  // sqrt(m) / r (r = n_sample / H). Large batches (many waves of merge warps, issue-bound) take the smallest tier
  // that holds mean + 3 sigma: 12 keys per lane at k = 32 (267 vs 285 us at B = 65536); one wave of warps
  // (B <= 8192) is latency-bound and faster with 16 (28.7 vs 34.8 us at B = 4096).
  int tier = 16;
  if (tuning().merge_tier > 0) tier = tuning().merge_tier;
  else if (n_sample > 0 && pl.m > 0 && B > 8192) {
    const double inv_r = static_cast<double>(H) / n_sample;
    const double need = (pl.m + 3.0 * sqrt(static_cast<double>(pl.m))) * inv_r;
    tier = need <= 256.0 ? 8 : (need <= 384.0 ? 12 : 16);
  }
  if (32 * tier < pl.k_sel) tier = 16;
  rc = launch_status("select_small kernel", select_small_launch(sl, tier, nullptr, nullptr, num_sms(), counters + 1, ovf_rows, st));
  if (rc != QSAE_OK) return rc;
  stage_mark(3, st);
  // tail, one launch: rows the warp merge could not hold (floods of equal values) through the block-per-row select,
  // rows whose prior failed the count check through the exact recomputation; both decoded there when fused
  RescueLaunch rl = rescue_launch(sl, x_bf16, w_bf16);
  rl.z_scratch = reinterpret_cast<float*>(ws + pl.rescue_z_off); rl.slot_done = counters + 4;
  rc = launch_status("select_tail kernel", select_tail_launch(sl, rl, counters + 1, ovf_rows, num_sms(), st));
  stage_mark(4, st);
  if (tuning().debug_large) {   // diagnostics (synchronises): rows that took the tail kernel
    cudaStreamSynchronize(st);
    int h[4] = {0, 0, 0, 0};
    cudaMemcpy(h, counters, sizeof(h), cudaMemcpyDeviceToHost);
    fprintf(stderr, "[qsae prior path] B=%d k_sel=%d m=%d nsub=%d cap=%d: %d rows recomputed exactly, %d rows through the block select\n",
            B, pl.k_sel, pl.m, pl.main.nsub, pl.main.cap, h[0], h[1]);
    if (h[0] > 0 && h[0] <= 8) {
      int32_t rr[8];
      cudaMemcpy(rr, rescue_rows, h[0] * sizeof(int32_t), cudaMemcpyDeviceToHost);
      for (int i = 0; i < h[0]; ++i) fprintf(stderr, "  rescued row %d\n", rr[i]);
    }
  }
  return rc;
}
}  // namespace

extern "C" {

int qsae_prior_prep(const float* x_f32, const uint16_t* w_sample, const float* b_sample, int n_sample, int B, int D,
                    int act, int m, uint16_t* x_bf16, float* prior, int* ns_out, void* stream) {
  if (B == 0) return QSAE_OK;
  if (!x_f32 || !w_sample || !b_sample || !x_bf16 || !prior) return fail(QSAE_ERR_INVALID_ARGUMENT, "prior_prep: null pointer");
  const int ns = prior_prep_pick_ns(B, D, n_sample, m, num_sms());
  if (ns_out) *ns_out = ns;
  if (ns == 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "prior_prep: no single-launch variant for B=%d D=%d n_sample=%d m=%d", B, D, n_sample, m);
  PrepLaunch pp{};
  pp.B = B; pp.D = D; pp.n_sample = n_sample; pp.act = act; pp.m = m; pp.ns = ns;
  pp.x_f32 = x_f32; pp.x_bf16 = x_bf16; pp.bias = b_sample; pp.prior = prior;
  return launch_status("prior_prep kernel", prior_prep_launch(w_sample, pp, S(stream)));
}

int qsae_encode_topk(const float* x_f32, const uint16_t* w_bf16, const float* w_f32, const float* b_enc,
                     const uint16_t* w_sample, const float* b_sample, int n_sample,
                     int B, int H, int D, int k, int act, int exact, float* out_vals, int32_t* out_idx,
                     int32_t* out_flags, void* workspace, size_t workspace_bytes, void* stream) {
  return encode_topk_impl(x_f32, w_bf16, w_f32, b_enc, w_sample, b_sample, n_sample, B, H, D, k, act, exact, out_vals,
                          out_idx, out_flags, workspace, workspace_bytes, stream);
}

int qsae_bsae_forward(const float* x_f32, const uint16_t* w_bf16, const float* w_f32, const float* b_enc,
                      const uint16_t* w_sample, const float* b_sample, int n_sample, int B, int H, int D, int k,
                      int exact, const uint8_t* packed, int n_bits, float qstep, const float* dec_bias,
                      float* out_vals, int32_t* out_idx, int32_t* out_flags, float* recon, void* workspace,
                      size_t workspace_bytes, void* stream) {
  if (B == 0) return QSAE_OK;
  if (!packed || !recon) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_forward: null pointer");
  if (n_bits < 1 || n_bits > 8) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_forward: 1 <= n_bits <= 8");
  FusedDecode fd = {reinterpret_cast<const uint32_t*>(packed), qstep, dec_bias, recon, false};
  int rc = encode_topk_impl(x_f32, w_bf16, w_f32, b_enc, w_sample, b_sample, n_sample, B, H, D, k, QSAE_ACT_NONE, exact,
                            out_vals, out_idx, out_flags, workspace, workspace_bytes, stream, n_bits <= 4 ? &fd : nullptr);
  if (rc != QSAE_OK) return rc;
  if (fd.done) return QSAE_OK;
  if (n_bits <= 4) rc = qsae_decode_int4(out_vals, out_idx, B, k, packed, H, D, qstep, dec_bias, recon, stream);
  else rc = qsae_decode_int8(out_vals, out_idx, B, k, reinterpret_cast<const int8_t*>(packed), H, D, qstep, dec_bias, recon,
                             stream);
  stage_mark(5, S(stream));
  return rc;
}

int qsae_encode_dense_tc(const float* x_f32, const uint16_t* w_bf16, const float* b_enc, int B, int H, int D,
                         int act, float* z, void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return QSAE_OK;
  if (!x_f32 || !w_bf16 || !b_enc || !z || !workspace) return fail(QSAE_ERR_INVALID_ARGUMENT, "encode_dense_tc: null pointer");
  EncodePlan pl;
  int rc = plan_encode(B, H, D, 1, 0, 0, &pl);
  if (rc != QSAE_OK) return rc;
  if (workspace_bytes < pl.total) return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "encode_dense_tc: workspace %zu < %zu", workspace_bytes, pl.total);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  uint16_t* x_bf16 = reinterpret_cast<uint16_t*>(ws + pl.x_off);
  rc = launch_status("cast x", cast_bf16_launch(x_f32, x_bf16, static_cast<size_t>(B) * D, S(stream)));
  if (rc != QSAE_OK) return rc;
  EncodeLaunch el = stage_launch(pl.main, B, D, act, b_enc, ws);
  el.debug_z = z;
  return launch_status("encode_topk kernel (dense dump)", encode_topk_launch(x_bf16, w_bf16, el, S(stream)));
}

// ---------------------------------------------------------------------------------------------
// q_sae
// ---------------------------------------------------------------------------------------------
int qsae_pack_matryoshka(const float* weight, const float* weight_mirror, int H, int D, const int* level_start,
                         const float* level_factor, int n_levels, uint32_t* packed, float* scale, void* stream) {
  if (!weight || !weight_mirror || !level_start || !level_factor || !packed || !scale)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_matryoshka: null pointer");
  if (H <= 0 || D <= 0 || (D % 16) != 0 || n_levels < 1 || n_levels > 32)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_matryoshka: need D %% 16 == 0 and 1 <= n_levels <= 32");
  return launch_status("pack_matryoshka", pack_matryoshka_launch(weight, weight_mirror, H, D, level_start, level_factor,
                                                                 n_levels, packed, scale, S(stream)));
}

namespace {
struct MatPlan { StagePlan st; size_t x_off, prior_off, scratch_off, total; };
constexpr float kActiveThreshold = 8.940697e-08f;  // sigmoid(z) > 0.5 in fp32 <=> z >= 1.5 * 2^-24
int plan_matryoshka(int B, int H, int D, MatPlan* mp) {
  if (B <= 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "B and H must be positive");
  if (D < 16 || D > 512 || (D % 16) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka: D must be a multiple of 16 in [16, 512], got %d", D);
  size_t off = 0;
  mp->x_off = take(off, static_cast<size_t>(B) * D * 2, 1024);
  mp->prior_off = take(off, static_cast<size_t>(B) * 4);
  plan_stage(B, H, 0, kStagePriorMain, off, &mp->st, true, D);
  // every active latent is kept: largest buffers. Range schedule: more, shorter lists per row (the same capacity per row)
  mp->st.cap = mp->st.range_g > 0 ? kCandCapMax / 2 : kCandCapMax;
  place_lists(B, off, &mp->st);
  off = mp->st.end;
  mp->scratch_off = take(off, decode_matryoshka_scratch_bytes(num_sms()));
  mp->total = off;
  return QSAE_OK;
}
}  // namespace

int qsae_matryoshka_workspace_bytes(int B, int H, int D, size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  MatPlan mp;
  int rc = plan_matryoshka(B, H, D, &mp);
  if (rc != QSAE_OK) return rc;
  *bytes = mp.total;
  return QSAE_OK;
}

int qsae_max_row_norm(const float* w_f32, int H, int D, float* out, void* stream) {
  if (!w_f32 || !out || H <= 0 || D <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "max_row_norm: bad argument");
  return launch_status("max_row_norm", max_row_norm_launch(w_f32, H, D, out, S(stream)));
}

int qsae_decode_matryoshka_lists_workspace_bytes(size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  *bytes = align_up(decode_matryoshka_scratch_bytes(num_sms()), 256);
  return QSAE_OK;
}

int qsae_decode_matryoshka_lists(const int32_t* lists, const int32_t* counts, int cap, int B, const uint32_t* packed,
                                 const float* scale, const int* level_start, int n_levels, int H, int D,
                                 const float* dec_bias, float* result, unsigned long long* level_count,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return QSAE_OK;
  if (!lists || !counts || !packed || !scale || !level_start || !result || !level_count || !workspace)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "decode_matryoshka_lists: null pointer");
  if (n_levels < 1 || n_levels > 8 || (D % 16) != 0 || D > 512 || cap < 1)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "decode_matryoshka_lists: need 1 <= n_levels <= 8, D %% 16 == 0, D <= 512");
  if (workspace_bytes < decode_matryoshka_scratch_bytes(num_sms()))
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "decode_matryoshka_lists: workspace too small");
  cudaError_t ce = cudaMemsetAsync(level_count, 0, static_cast<size_t>(n_levels) * sizeof(unsigned long long), S(stream));
  if (ce != cudaSuccess) return fail(QSAE_ERR_CUDA, "decode_matryoshka_lists: %s", cudaGetErrorString(ce));
  return launch_status("decode_matryoshka", decode_matryoshka_launch(lists, counts, 1, cap, B, packed, scale, level_start,
                                                                     n_levels, H, D, dec_bias, result, level_count,
                                                                     nullptr, nullptr, nullptr, 0.f, 0, workspace, num_sms(),
                                                                     S(stream)));
}

int qsae_matryoshka_forward(const float* x_f32, const uint16_t* w_bf16, const float* w_f32, const float* w_norm_max,
                            const float* b_enc, const uint32_t* packed,
                            const float* scale, const int* level_start, int n_levels, const float* dec_bias,
                            int B, int H, int D, float* result, unsigned long long* level_count, int* overflow,
                            void* workspace, size_t workspace_bytes, void* stream) {
  return qsae_matryoshka_forward_active(x_f32, w_bf16, w_f32, w_norm_max, b_enc, packed, scale, level_start, n_levels,
                                        dec_bias, B, H, D, result, level_count, overflow, nullptr, 0, nullptr, nullptr,
                                        workspace, workspace_bytes, stream);
}

int qsae_matryoshka_forward_active(const float* x_f32, const uint16_t* w_bf16, const float* w_f32,
                                   const float* w_norm_max, const float* b_enc, const uint32_t* packed,
                                   const float* scale, const int* level_start, int n_levels, const float* dec_bias,
                                   int B, int H, int D, float* result, unsigned long long* level_count, int* overflow,
                                   int32_t* active_idx, int active_cap, int32_t* active_cnt, float* residual_out,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return QSAE_OK;
  if (residual_out != nullptr && (reinterpret_cast<uintptr_t>(residual_out) & 15) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward: residual_out must be 16-byte aligned");
  if (active_idx != nullptr && (active_cap < 1 || active_cnt == nullptr))
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward: active list export needs active_cap >= 1 and active_cnt");
  if (!x_f32 || !w_bf16 || !b_enc || !packed || !scale || !level_start || !result || !level_count || !overflow || !workspace)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward: null pointer");
  if (n_levels < 1 || n_levels > 8) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward: 1 <= n_levels <= 8");
  const int exact = (w_f32 != nullptr) ? 1 : 0;
  if (exact && !w_norm_max) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward: exact mode needs w_norm_max");
  MatPlan mp;
  int rc = plan_matryoshka(B, H, D, &mp);
  if (rc != QSAE_OK) return rc;
  if (workspace_bytes < mp.total)
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "matryoshka_forward: workspace %zu < %zu bytes", workspace_bytes, mp.total);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  uint16_t* x_bf16 = reinterpret_cast<uint16_t*>(ws + mp.x_off);
  float* thr = reinterpret_cast<float*>(ws + mp.prior_off);
  cudaStream_t st = S(stream);
  cudaError_t ce = cudaMemsetAsync(level_count, 0, static_cast<size_t>(n_levels) * sizeof(unsigned long long), st);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(overflow, 0, sizeof(int), st);
  if (ce != cudaSuccess) return fail(QSAE_ERR_CUDA, "matryoshka_forward: %s", cudaGetErrorString(ce));
  if (exact) {
    rc = launch_status("row_threshold", row_threshold_launch(x_f32, B, D, w_norm_max, kActiveThreshold, thr, st));
    if (rc != QSAE_OK) return rc;
  }
  rc = launch_status("cast x", cast_bf16_launch(x_f32, x_bf16, static_cast<size_t>(B) * D, st));
  if (rc != QSAE_OK) return rc;
  EncodeLaunch el = stage_launch(mp.st, B, D, QSAE_ACT_NONE, b_enc, ws);
  el.prior = exact ? thr : nullptr; el.prior_stride = 1; el.prior_const = kActiveThreshold;   // per-row band, or one constant threshold (by value)
  el.overflow = overflow;
  rc = launch_status("encode kernel (threshold)", encode_topk_launch(x_bf16, w_bf16, el, st));
  if (rc != QSAE_OK) return rc;
  if (active_idx != nullptr) {   // empty slots read as -1
    ce = cudaMemsetAsync(active_idx, 0xFF, static_cast<size_t>(B) * active_cap * sizeof(int32_t), st);
    if (ce != cudaSuccess) return fail(QSAE_ERR_CUDA, "matryoshka_forward: %s", cudaGetErrorString(ce));
  }
  return launch_status("decode_matryoshka", decode_matryoshka_launch(el.cand, el.cand_cnt, mp.st.nsub, mp.st.cap, B, packed,
                                                                     scale, level_start, n_levels, H, D, dec_bias, result,
                                                                     level_count, x_f32, w_f32, b_enc, kActiveThreshold,
                                                                     exact, ws + mp.scratch_off, num_sms(), st, active_idx,
                                                                     active_cap, active_cnt, residual_out ? x_f32 : nullptr,
                                                                     residual_out, overflow));
}

// ---------------------------------------------------------------------------------------------
// analysis consumers over sparse active lists (scripts/analysis/dynamic_analysis.py)
// ---------------------------------------------------------------------------------------------
int qsae_activation_counts(const int32_t* idx, const float* vals, int B, int cap, int H, unsigned long long* counts,
                           void* stream) {
  if (B < 0 || cap < 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "activation_counts: bad shape");
  if (B == 0 || cap == 0) return QSAE_OK;
  if (!idx || !counts) return fail(QSAE_ERR_INVALID_ARGUMENT, "activation_counts: null pointer");
  return launch_status("activation_counts", activation_counts_launch(idx, vals, B, cap, H, counts, S(stream)));
}

int qsae_coactivation(const int32_t* idx, const float* vals, int B, int cap, int H, int32_t* cooc, void* stream) {
  if (B < 0 || cap < 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "coactivation: bad shape");
  if (cap > 2048) return fail(QSAE_ERR_INVALID_ARGUMENT, "coactivation: at most 2048 list entries per row, got %d", cap);
  if (B == 0 || cap == 0) return QSAE_OK;
  if (!idx || !cooc) return fail(QSAE_ERR_INVALID_ARGUMENT, "coactivation: null pointer");
  return launch_status("coactivation", coactivation_launch(idx, vals, B, cap, H, cooc, S(stream)));
}

int qsae_coactivation_dense(const uint16_t* mask, int K, int H, int32_t* cooc, long long* counts, void* stream) {
  if (K < 0 || H <= 0 || (H % 8) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "coactivation_dense: K >= 0 and H a positive multiple of 8 (K=%d H=%d)", K, H);
  if (K > (1 << 24))
    return fail(QSAE_ERR_INVALID_ARGUMENT, "coactivation_dense: at most 2^24 rows per call (the fp32 counts are exact to "
                "2^24), got %d", K);
  if (K == 0) return QSAE_OK;
  if (!mask || !cooc) return fail(QSAE_ERR_INVALID_ARGUMENT, "coactivation_dense: null pointer");
  if (((reinterpret_cast<uintptr_t>(mask) | reinterpret_cast<uintptr_t>(cooc)) & 15) || (reinterpret_cast<uintptr_t>(counts) & 7))
    return fail(QSAE_ERR_INVALID_ARGUMENT, "coactivation_dense: mask and cooc must be 16-byte aligned, counts 8-byte");
  return launch_status("coactivation_dense", coactivation_dense_launch(mask, K, H, cooc, counts, num_sms(), S(stream)));
}

int qsae_sq_error_accumulate(const float* a, const float* b, size_t n, double* out, void* stream) {
  if (n == 0) return QSAE_OK;
  if (!a || !b || !out) return fail(QSAE_ERR_INVALID_ARGUMENT, "sq_error: null pointer");
  return launch_status("sq_error", sq_error_launch(a, b, n, out, S(stream)));
}

int qsae_compact_dense(const float* dense, int B, int H, int mode, float thr, int cap, int32_t* idx, float* vals, int32_t* pairs,
                       int32_t* cnt, void* stream) {
  if (B < 0 || H <= 0 || cap < 0 || (mode != 0 && mode != 1)) return fail(QSAE_ERR_INVALID_ARGUMENT, "compact_dense: bad arguments");
  if (B == 0) return QSAE_OK;
  if (!dense || !cnt) return fail(QSAE_ERR_INVALID_ARGUMENT, "compact_dense: null pointer");
  return launch_status("compact_dense", compact_dense_launch(dense, B, H, mode, thr, cap, idx, vals, pairs, cnt, S(stream)));
}

// ---------------------------------------------------------------------------------------------
// training-side pieces adjacent to the forward (SURVEY 8f-4; train.cu)
// ---------------------------------------------------------------------------------------------
int qsae_rows_scatter_add(const float* coef, const int32_t* idx, const float* src, int B, int k, int D, int H, float scale,
                          float* dst, float* dst_col, void* stream) {
  if (B < 0 || k < 0 || D <= 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "rows_scatter_add: bad shape");
  if (B == 0 || k == 0) return QSAE_OK;
  if (!idx || !src || !dst) return fail(QSAE_ERR_INVALID_ARGUMENT, "rows_scatter_add: null pointer");
  if ((D % 4) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "rows_scatter_add: src / dst must be 16-byte aligned");
  return launch_status("rows_scatter_add", rows_scatter_add_launch(coef, idx, src, B, k, D, H, scale, dst, dst_col, S(stream)));
}

int qsae_rows_gather_dot(const float* g, const float* rows, const int32_t* idx, int B, int k, int D, int H, float scale,
                         float* out, void* stream) {
  if (B < 0 || k < 0 || D <= 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "rows_gather_dot: bad shape");
  if (B == 0 || k == 0) return QSAE_OK;
  if (!g || !rows || !idx || !out) return fail(QSAE_ERR_INVALID_ARGUMENT, "rows_gather_dot: null pointer");
  if ((D % 4) == 0 && ((reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(rows)) & 15) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "rows_gather_dot: g / rows must be 16-byte aligned");
  return launch_status("rows_gather_dot", rows_gather_dot_launch(g, rows, idx, B, k, D, H, scale, out, S(stream)));
}

int qsae_column_sum(const float* src, int R, int C, float scale, float* out, void* stream) {
  if (R < 0 || C < 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "column_sum: bad shape");
  if (R == 0 || C == 0) return QSAE_OK;
  if (!src || !out) return fail(QSAE_ERR_INVALID_ARGUMENT, "column_sum: null pointer");
  return launch_status("column_sum", column_sum_launch(src, R, C, scale, out, S(stream)));
}

int qsae_bsae_logit_grad(const float* logits, const float* G, int H, int D, int n_bits, const float* gp_dev, float gp_host,
                         int accumulate, float* grad_logits, void* stream) {
  if (H <= 0 || D <= 0 || n_bits < 1 || n_bits > 16) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_logit_grad: bad shape");
  if (!logits || !grad_logits) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_logit_grad: null pointer");
  return launch_status("bsae_logit_grad",
                       bsae_logit_grad_launch(logits, G, H, D, n_bits, gp_dev, gp_host, accumulate, grad_logits, S(stream)));
}

static int check_levels(const char* who, const int* level_start, int n_levels, int H) {
  if (!level_start || n_levels < 1 || n_levels > 8) return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: 1..8 levels", who);
  if (level_start[0] != 0 || level_start[n_levels] != H) return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: level_start must span [0, H]", who);
  for (int i = 0; i < n_levels; ++i)
    if (level_start[i + 1] < level_start[i]) return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: level_start must be non-decreasing", who);
  return QSAE_OK;
}

int qsae_matryoshka_backward_scatter(const int32_t* active_idx, int B, int cap, int H, int D, const float* const* grad_levels,
                                     const int* level_start, int n_levels, float* M, int32_t* z2, void* stream) {
  if (B < 0 || cap < 0 || H <= 0 || D <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_scatter: bad shape");
  int rc = check_levels("matryoshka_backward_scatter", level_start, n_levels, H);
  if (rc != QSAE_OK) return rc;
  if (B == 0 || cap == 0) return QSAE_OK;
  if (!active_idx || !grad_levels || !M || !z2) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_scatter: null pointer");
  for (int i = 0; i < n_levels; ++i)
    if (!grad_levels[i] || ((D % 4) == 0 && (reinterpret_cast<uintptr_t>(grad_levels[i]) & 15) != 0))
      return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_scatter: grad_levels[%d] null or not 16-byte aligned", i);
  return launch_status("matryoshka_backward_scatter",
                       matryoshka_scatter_launch(active_idx, B, cap, H, D, grad_levels, level_start, n_levels, M, z2, S(stream)));
}

int qsae_matryoshka_backward_finish(const float* w, const float* w_mirror, const float* M, const int32_t* z2, const float* alpha,
                                    const int* level_start, int n_levels, int H, int D, float c, int joint_bits, float* grad_w,
                                    float* grad_w_mirror, void* stream) {
  if (H <= 0 || D <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_finish: bad shape");
  int rc = check_levels("matryoshka_backward_finish", level_start, n_levels, H);
  if (rc != QSAE_OK) return rc;
  if (!w || !w_mirror || !alpha || !grad_w || !grad_w_mirror || (!M && !z2))
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_finish: null pointer");
  return launch_status("matryoshka_backward_finish",
                       matryoshka_grad_finish_launch(w, w_mirror, M, z2, alpha, level_start, n_levels, H, D, c, joint_bits,
                                                     grad_w, grad_w_mirror, S(stream)));
}

namespace {
// workspace of the dense STE backward: n_parts bf16 parts, each the n_levels level gradients stacked [n_levels B, D]
int plan_matryoshka_backward_dense(int B, int D, int n_levels, int exact, size_t* part_bytes, size_t* total) {
  if (B < 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_dense: negative batch");
  if (D < 16 || D > 512 || (D % 16) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_dense: D must be a multiple of 16 in [16, 512], got %d", D);
  if (n_levels < 1 || n_levels > 8) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_dense: 1..8 levels, got %d", n_levels);
  *part_bytes = align_up(static_cast<size_t>(n_levels) * B * D * 2, 1024);
  *total = (exact ? 3 : 1) * *part_bytes;
  return QSAE_OK;
}
}  // namespace

int qsae_matryoshka_backward_dense_workspace_bytes(int B, int D, int n_levels, int exact, size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  size_t part = 0;
  return plan_matryoshka_backward_dense(B, D, n_levels, exact, &part, bytes);
}

int qsae_matryoshka_backward_dense(const uint16_t* mask, int B, int H, int D, const float* const* grad_levels,
                                   const int* level_start, int n_levels, const float* w, const float* w_mirror,
                                   const float* alpha, int exact, float* grad_w, float* grad_w_mirror, int32_t* z2,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  size_t part = 0, total = 0;
  int rc = plan_matryoshka_backward_dense(B, D, n_levels, exact, &part, &total);
  if (rc != QSAE_OK) return rc;
  if (H <= 0 || (H % 8) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_dense: H must be a positive multiple of 8, got %d", H);
  rc = check_levels("matryoshka_backward_dense", level_start, n_levels, H);
  if (rc != QSAE_OK) return rc;
  if (!w || !w_mirror || !alpha || !grad_w || !grad_w_mirror || !z2)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_dense: null pointer");
  cudaStream_t st = S(stream);
  cudaError_t e = cudaMemsetAsync(z2, 0, static_cast<size_t>(H) * 4, st);
  if (e != cudaSuccess) return fail(QSAE_ERR_CUDA, "matryoshka_backward_dense: %s", cudaGetErrorString(e));
  if (B == 0) return QSAE_OK;
  if (!mask || !grad_levels || !workspace) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_dense: null pointer");
  if (workspace_bytes < total)
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "matryoshka_backward_dense: workspace %zu < %zu bytes", workspace_bytes, total);
  uintptr_t align16 = reinterpret_cast<uintptr_t>(mask) | reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(w_mirror) |
                      reinterpret_cast<uintptr_t>(grad_w) | reinterpret_cast<uintptr_t>(grad_w_mirror);
  for (int i = 0; i < n_levels; ++i) {
    if (!grad_levels[i]) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_dense: grad_levels[%d] is null", i);
    align16 |= reinterpret_cast<uintptr_t>(grad_levels[i]);
  }
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0 || (align16 & 15) != 0 || (reinterpret_cast<uintptr_t>(alpha) & 3) != 0 ||
      (reinterpret_cast<uintptr_t>(z2) & 3) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_backward_dense: workspace must be 1024-byte aligned, the mask, gradients, "
                "weights and .grad buffers 16-byte aligned");
  // the bf16 parts of every level gradient, stacked per part: part i, level l at ws + i part + l B D
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const int np = exact ? 3 : 1;
  const size_t nbd = static_cast<size_t>(B) * D;
  uint16_t* gp[3];
  for (int i = 0; i < 3; ++i) gp[i] = reinterpret_cast<uint16_t*>(ws + (i < np ? i : 0) * part);
  for (int l = 0; l < n_levels; ++l) {
    const size_t off = static_cast<size_t>(l) * nbd;
    rc = launch_status("matryoshka_backward_dense (gradient parts)",
                       exact ? split_bf16x3_launch(grad_levels[l], gp[0] + off, gp[1] + off, gp[2] + off, nbd, st)
                             : cast_bf16_launch(grad_levels[l], gp[0] + off, nbd, st));
    if (rc != QSAE_OK) return rc;
  }
  rc = launch_status("matryoshka_backward_dense (z2)", mask_column_count_launch(mask, B, H, z2, st));
  if (rc != QSAE_OK) return rc;
  const uint16_t* gpc[3] = {gp[0], gp[1], gp[2]};
  return launch_status("matryoshka_backward_dense (product)",
                       matryoshka_ste_dense_launch(mask, B, H, D, gpc, np, level_start, n_levels, w, w_mirror, alpha, grad_w,
                                                   grad_w_mirror, num_sms(), st));
}

int qsae_rigl_workspace_bytes(size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  *bytes = align_up(rigl_workspace_bytes(num_sms()), 256);
  return QSAE_OK;
}

static int check_rigl(const char* who, const float* weight, const float* mask, int D, int H, void* ws, size_t ws_bytes) {
  if (D <= 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: bad shape", who);
  if (static_cast<unsigned long long>(D) * static_cast<unsigned long long>(H) >= 0xffffffffull)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: D * H must be below 2^32", who);
  if (!weight || !mask || !ws) return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: null pointer", who);
  if (ws_bytes < align_up(rigl_workspace_bytes(num_sms()), 256)) return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "%s: workspace too small", who);
  return QSAE_OK;
}

int qsae_rigl_init_mask(float* weight, float* mask, int D, int H, unsigned long long n_inactive, void* workspace,
                        size_t workspace_bytes, void* stream) {
  int rc = check_rigl("rigl_init_mask", weight, mask, D, H, workspace, workspace_bytes);
  if (rc != QSAE_OK) return rc;
  const char* e = rigl_init_mask_launch(weight, mask, D, H, n_inactive, workspace, num_sms(), S(stream));
  return e ? fail(QSAE_ERR_CUDA, "rigl_init_mask: %s", e) : QSAE_OK;
}

int qsae_rigl_update_mask(float* weight, float* mask, const float* a_mean, const float* d_mean, int D, int H,
                          unsigned long long n_drop, unsigned long long n_grow, void* workspace, size_t workspace_bytes,
                          void* stream) {
  int rc = check_rigl("rigl_update_mask", weight, mask, D, H, workspace, workspace_bytes);
  if (rc != QSAE_OK) return rc;
  const char* e = rigl_update_mask_launch(weight, mask, a_mean, d_mean, D, H, n_drop, n_grow, workspace, num_sms(), S(stream));
  return e ? fail(QSAE_ERR_CUDA, "rigl_update_mask: %s", e) : QSAE_OK;
}

int qsae_mul_inplace(float* a, const float* b, size_t n, void* stream) {
  if (n == 0) return QSAE_OK;
  if (!a || !b) return fail(QSAE_ERR_INVALID_ARGUMENT, "mul_inplace: null pointer");
  return launch_status("mul_inplace", mul_inplace_launch(a, b, n, S(stream)));
}

// ---------------------------------------------------------------------------------------------
// t_sae
// ---------------------------------------------------------------------------------------------
int qsae_split_bf16(const float* src, uint16_t* hi, uint16_t* lo, size_t n, void* stream) {
  if (!src || !hi) return fail(QSAE_ERR_INVALID_ARGUMENT, "split_bf16: null pointer");
  if (n == 0) return QSAE_OK;
  return launch_status("split_bf16", split_bf16_launch(src, hi, lo, n, S(stream)));
}

int qsae_pack_ternary(const float* w, int D, int H, float threshold, uint16_t* t_bf16, int8_t* t_rows, void* stream) {
  if (!w || (!t_bf16 && !t_rows)) return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_ternary: null pointer");
  if (D <= 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_ternary: bad shape");
  return launch_status("pack_ternary", pack_ternary_launch(w, D, H, threshold, t_bf16, t_rows, S(stream)));
}

static int check_dense_decode(const char* who, int B, int K, int N) {
  if (B < 0 || K <= 0 || N <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: bad shape", who);
  if ((K % 8) != 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: the contraction length must be a multiple of 8, got %d", who, K);
  if ((N % 4) != 0 || N > 512) return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: output width must be a multiple of 4, <= 512, got %d", who, N);
  return QSAE_OK;
}

int qsae_decode_dense_workspace_bytes(int B, int K, int N, size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  int rc = check_dense_decode("decode_dense", B, K, N);
  if (rc != QSAE_OK) return rc;
  *bytes = align_up(dense_decode_workspace_bytes(B > 0 ? B : 1, K, N, num_sms()), 256);
  return QSAE_OK;
}

int qsae_decode_dense(const uint16_t* a_hi, const uint16_t* a_lo, const uint16_t* b_t, int B, int K, int N,
                      const float* bias, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_dense_decode("decode_dense", B, K, N);
  if (rc != QSAE_OK || B == 0) return rc;
  if (!a_hi || !b_t || !out || !workspace) return fail(QSAE_ERR_INVALID_ARGUMENT, "decode_dense: null pointer");
  if ((reinterpret_cast<uintptr_t>(a_hi) & 15) || (reinterpret_cast<uintptr_t>(a_lo) & 15) ||
      (reinterpret_cast<uintptr_t>(b_t) & 15) || (reinterpret_cast<uintptr_t>(workspace) & 15))
    return fail(QSAE_ERR_INVALID_ARGUMENT, "decode_dense: operands must be 16-byte aligned");
  const size_t need = dense_decode_workspace_bytes(B, K, N, num_sms());
  if (workspace_bytes < need) return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "decode_dense: workspace %zu < %zu bytes", workspace_bytes, need);
  if (g_enc_ev_start) cudaEventRecord(g_enc_ev_start, S(stream));
  rc = launch_status("dense_decode", dense_decode_launch(a_hi, a_lo, K, b_t, K, B, K, N, bias, nullptr, out, workspace, num_sms(), S(stream)));
  if (g_enc_ev_stop) cudaEventRecord(g_enc_ev_stop, S(stream));
  return rc;
}

namespace {
// Dense pre-activations (+ activation) on the tensor cores.
//   w_mid == w_lo == nullptr: one pass over bf16(x) and w_hi (fast mode; encode_dense_tc_launch).
//   otherwise: fp32-accurate product through 8 + 8 + 8-bit operand splits, x = xh + xm + xl and
//   W = wh + wm + wl (both exact), keeping the six partial products above 2^-24 in ONE launch
//   (encode_dense_split_kernel: both operands streamed, one accumulator, outputs written once).
// x_parts: workspace for the bf16 part(s) of x, 3 * align_up(B * D * 2, 1024) bytes in split mode.
// step: act == 2 only (EncodeLaunch::step_*): the q_sae dense path's A operand written by the epilogue.
struct StepOperand {
  float thr; const float* scale; const int* level_start; int n_levels; unsigned long long* level_count;
  uint16_t* mask; int mask_pitch;   // or null: activity mask (EncodeLaunch::step_mask)
};
int dense_encode_tc(const float* x_f32, const uint16_t* w_hi, const uint16_t* w_mid, const uint16_t* w_lo,
                    const float* b_enc, int B, int H, int D, int act, uint8_t* x_parts, float* out_f32, uint16_t* out_hi,
                    uint16_t* out_lo, cudaStream_t st, const StepOperand* step = nullptr) {
  EncodeLaunch el{};
  el.B = B; el.H = H; el.D = D; el.act = act; el.bias = b_enc;
  if (act == 2) {
    if (!step) return fail(QSAE_ERR_INVALID_ARGUMENT, "dense encoder: step operand without its description");
    el.step_thr = step->thr; el.step_scale = step->scale; el.step_level_start = step->level_start;
    el.step_n_levels = step->n_levels; el.step_level_count = step->level_count;
    el.step_mask = step->mask; el.step_mask_pitch = step->mask_pitch;
  }
  el.n_tiles = (H + kEncBN - 1) / kEncBN;
  el.n_splits = encode_pick_splits(B, H, num_sms());
  el.tiles_per_split = (el.n_tiles + el.n_splits - 1) / el.n_splits;
  const size_t xn = static_cast<size_t>(B) * D;
  const size_t xstride = align_up(xn * 2, 1024);
  uint16_t* xh = reinterpret_cast<uint16_t*>(x_parts);
  if (!w_mid || !w_lo) {
    int rc = launch_status("cast x", cast_bf16_launch(x_f32, xh, xn, st));
    if (rc != QSAE_OK) return rc;
    if (g_enc_ev_start) cudaEventRecord(g_enc_ev_start, st);
    rc = launch_status("encode kernel (dense)", encode_dense_tc_launch(xh, w_hi, el, out_f32, out_hi, out_lo, st));
    if (g_enc_ev_stop) cudaEventRecord(g_enc_ev_stop, st);
    return rc;
  }
  uint16_t* xm = reinterpret_cast<uint16_t*>(x_parts + xstride);
  uint16_t* xl = reinterpret_cast<uint16_t*>(x_parts + 2 * xstride);
  int rc = launch_status("split x", split_bf16x3_launch(x_f32, xh, xm, xl, xn, st));
  if (rc != QSAE_OK) return rc;
  const uint16_t* xp[3] = {xh, xm, xl};
  const uint16_t* wp[3] = {w_hi, w_mid, w_lo};
  if (g_enc_ev_start) cudaEventRecord(g_enc_ev_start, st);
  rc = launch_status("encode kernel (dense, split operands)", encode_dense_split_launch(xp, wp, 3, el, out_f32, out_hi, out_lo, num_sms(), st));
  if (g_enc_ev_stop) cudaEventRecord(g_enc_ev_stop, st);
  return rc;
}
}  // namespace

namespace {
struct TsaePlan { size_t x_off, hi_off, lo_off, dec_off, total; };
int plan_tsae(int B, int H, int D, int exact, TsaePlan* tp) {
  const int rc = check_encode_shape(B, H, D);
  if (rc != QSAE_OK) return rc;
  if ((H % 8) != 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "t_sae: hidden_dim must be a multiple of 8, got %d", H);
  tp->x_off = 0;
  tp->hi_off = (exact ? 3 : 1) * align_up(static_cast<size_t>(B) * D * 2, 1024);
  tp->lo_off = align_up(tp->hi_off + static_cast<size_t>(B) * H * 2, 1024);
  tp->dec_off = exact ? align_up(tp->lo_off + static_cast<size_t>(B) * H * 2, 1024) : tp->lo_off;
  tp->total = align_up(tp->dec_off + dense_decode_workspace_bytes(B, H, D, num_sms()), 256);
  return QSAE_OK;
}
}  // namespace

int qsae_tsae_workspace_bytes(int B, int H, int D, int exact, size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  TsaePlan tp;
  int rc = plan_tsae(B, H, D, exact, &tp);
  if (rc != QSAE_OK) return rc;
  *bytes = tp.total;
  return QSAE_OK;
}

int qsae_split_bf16x3(const float* src, uint16_t* hi, uint16_t* mid, uint16_t* lo, size_t n, void* stream) {
  if (!src || !hi) return fail(QSAE_ERR_INVALID_ARGUMENT, "split_bf16x3: null pointer");
  if (n == 0) return QSAE_OK;
  return launch_status("split_bf16x3", split_bf16x3_launch(src, hi, mid, lo, n, S(stream)));
}

int qsae_tsae_forward(const float* x_f32, const uint16_t* w_hi, const uint16_t* w_mid, const uint16_t* w_lo,
                      const float* b_enc, const uint16_t* t_bf16, int B, int H, int D, int exact, float* h_out,
                      float* recon, void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return QSAE_OK;
  if (!x_f32 || !w_hi || !b_enc || !t_bf16 || !h_out || !recon || !workspace)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "tsae_forward: null pointer");
  if (exact && (!w_mid || !w_lo)) return fail(QSAE_ERR_INVALID_ARGUMENT, "tsae_forward: exact mode needs the three parts of W");
  TsaePlan tp;
  int rc = plan_tsae(B, H, D, exact, &tp);
  if (rc != QSAE_OK) return rc;
  if (workspace_bytes < tp.total)
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "tsae_forward: workspace %zu < %zu bytes", workspace_bytes, tp.total);
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0 || (reinterpret_cast<uintptr_t>(h_out) & 15) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "tsae_forward: workspace must be 1024-byte and h_out 16-byte aligned");
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  uint16_t* h_hi = reinterpret_cast<uint16_t*>(ws + tp.hi_off);
  uint16_t* h_lo = exact ? reinterpret_cast<uint16_t*>(ws + tp.lo_off) : nullptr;
  cudaStream_t st = S(stream);
  rc = dense_encode_tc(x_f32, w_hi, exact ? w_mid : nullptr, exact ? w_lo : nullptr, b_enc, B, H, D, QSAE_ACT_RELU,
                       ws + tp.x_off, h_out, h_hi, h_lo, st);
  if (rc != QSAE_OK) return rc;
  return launch_status("dense_decode", dense_decode_launch(h_hi, h_lo, H, t_bf16, H, B, H, D, nullptr, nullptr, recon,
                                                           ws + tp.dec_off, num_sms(), st));
}

// ---- t_sae backward (training.py: _TernarySAEFn)
int qsae_pack_ternary_t(const float* w, int D, int H, float threshold, uint16_t* t_t_bf16, void* stream) {
  if (!w || !t_t_bf16) return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_ternary_t: null pointer");
  if (D <= 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_ternary_t: bad shape");
  return launch_status("pack_ternary_t", pack_ternary_launch(w, D, H, threshold, nullptr, nullptr, S(stream), t_t_bf16));
}

int qsae_wgrad(const uint16_t* const* a_parts, const uint16_t* const* b_parts, int n_parts, int M, int N, int K, int a_kmajor,
               float* c, void* stream) {
  if (!a_parts || !b_parts || !c) return fail(QSAE_ERR_INVALID_ARGUMENT, "wgrad: null pointer");
  if (n_parts != 1 && n_parts != 3) return fail(QSAE_ERR_INVALID_ARGUMENT, "wgrad: n_parts must be 1 or 3, got %d", n_parts);
  if (M <= 0 || N <= 0 || K <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "wgrad: bad shape M=%d N=%d K=%d", M, N, K);
  if ((N % 8) != 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "wgrad: N must be a multiple of 8, got %d", N);
  if (a_kmajor ? (K % 8) != 0 : (M % 8) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "wgrad: %s must be a multiple of 8 (row pitch of A), got %d", a_kmajor ? "K" : "M",
                a_kmajor ? K : M);
  uintptr_t bits = reinterpret_cast<uintptr_t>(c);
  for (int i = 0; i < n_parts; ++i) {
    if (!a_parts[i] || !b_parts[i]) return fail(QSAE_ERR_INVALID_ARGUMENT, "wgrad: null operand part");
    bits |= reinterpret_cast<uintptr_t>(a_parts[i]) | reinterpret_cast<uintptr_t>(b_parts[i]);
  }
  if (bits & 15) return fail(QSAE_ERR_INVALID_ARGUMENT, "wgrad: operands and output must be 16-byte aligned");
  return launch_status("wgrad", wgrad_launch(a_parts, b_parts, n_parts, M, N, K, a_kmajor != 0, c, num_sms(), S(stream)));
}

namespace {
// workspace of the backward: bf16 parts of g, x [B, D]; the bf16 parts of gz, h [B, H] and (exact mode) fp32 gz
struct TsaeBwdPlan { size_t bd, bh, g_off, x_off, gz_off, gzp_off, hp_off, total; };
int plan_tsae_backward(int B, int H, int D, int exact, TsaeBwdPlan* bp) {
  TsaePlan tp;
  int rc = plan_tsae(B > 0 ? B : 1, H, D, exact, &tp);   // the forward's shape limits
  if (rc != QSAE_OK) return rc;
  const int np = exact ? 3 : 1;
  bp->bd = align_up(static_cast<size_t>(B) * D * 2, 1024);
  bp->bh = align_up(static_cast<size_t>(B) * H * 2, 1024);
  bp->g_off = 0;
  bp->x_off = bp->g_off + np * bp->bd;
  bp->gz_off = bp->x_off + np * bp->bd;
  bp->gzp_off = bp->gz_off + (exact ? align_up(static_cast<size_t>(B) * H * 4, 1024) : 0);   // fp32 gz: exact only
  bp->hp_off = bp->gzp_off + np * bp->bh;
  bp->total = bp->hp_off + np * bp->bh;
  return QSAE_OK;
}
}  // namespace

int qsae_tsae_backward_workspace_bytes(int B, int H, int D, int exact, size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  if (B < 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "tsae_backward: negative batch");
  TsaeBwdPlan bp;
  int rc = plan_tsae_backward(B, H, D, exact, &bp);
  if (rc != QSAE_OK) return rc;
  *bytes = bp.total;
  return QSAE_OK;
}

int qsae_tsae_backward(const float* x, const float* h, const float* g_recon, const float* g_h, const uint16_t* t_t_bf16,
                       const float* mask, const uint16_t* w_hi, const uint16_t* w_mid, const uint16_t* w_lo, int B, int H, int D,
                       int exact, float* grad_w_enc, float* grad_b_enc, float* grad_w_dec, float* grad_x, void* workspace,
                       size_t workspace_bytes, void* stream) {
  if (B < 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "tsae_backward: negative batch");
  TsaeBwdPlan bp;
  int rc = plan_tsae_backward(B, H, D, exact, &bp);
  if (rc != QSAE_OK) return rc;
  if (!grad_w_enc || !grad_b_enc || !grad_w_dec) return fail(QSAE_ERR_INVALID_ARGUMENT, "tsae_backward: null gradient pointer");
  cudaStream_t st = S(stream);
  const size_t nbd = static_cast<size_t>(B) * D, nbh = static_cast<size_t>(B) * H, nhd = static_cast<size_t>(H) * D;
  if (B == 0) {   // nothing to contract: zero gradients
    cudaError_t e = cudaMemsetAsync(grad_w_enc, 0, nhd * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(grad_b_enc, 0, static_cast<size_t>(H) * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(grad_w_dec, 0, nhd * 4, st);
    return e == cudaSuccess ? QSAE_OK : fail(QSAE_ERR_CUDA, "tsae_backward: %s", cudaGetErrorString(e));
  }
  if (!x || !h || !g_recon || !t_t_bf16 || !workspace) return fail(QSAE_ERR_INVALID_ARGUMENT, "tsae_backward: null pointer");
  if (grad_x && (!w_hi || (exact && (!w_mid || !w_lo))))
    return fail(QSAE_ERR_INVALID_ARGUMENT, "tsae_backward: grad_x needs the parts of W_enc (three in exact mode)");
  if (workspace_bytes < bp.total)
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "tsae_backward: workspace %zu < %zu bytes", workspace_bytes, bp.total);
  const uintptr_t align16 = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(h) | reinterpret_cast<uintptr_t>(g_recon) |
                            reinterpret_cast<uintptr_t>(g_h) | reinterpret_cast<uintptr_t>(t_t_bf16) |
                            reinterpret_cast<uintptr_t>(grad_w_enc) | reinterpret_cast<uintptr_t>(grad_w_dec) |
                            reinterpret_cast<uintptr_t>(grad_x) | reinterpret_cast<uintptr_t>(w_hi) |
                            reinterpret_cast<uintptr_t>(w_mid) | reinterpret_cast<uintptr_t>(w_lo);
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0 || (align16 & 15) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "tsae_backward: workspace must be 1024-byte and tensors 16-byte aligned");
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const int np = exact ? 3 : 1;
  uint16_t *gp[3], *xp[3], *gzp[3], *hp[3];
  for (int i = 0; i < 3; ++i) {
    const int j = i < np ? i : 0;
    gp[i] = reinterpret_cast<uint16_t*>(ws + bp.g_off + j * bp.bd);
    xp[i] = reinterpret_cast<uint16_t*>(ws + bp.x_off + j * bp.bd);
    gzp[i] = reinterpret_cast<uint16_t*>(ws + bp.gzp_off + j * bp.bh);
    hp[i] = reinterpret_cast<uint16_t*>(ws + bp.hp_off + j * bp.bh);
  }
  float* gz = reinterpret_cast<float*>(ws + bp.gz_off);
  auto parts = [&](const char* what, const float* src, uint16_t* const* dst, size_t n) {
    return launch_status(what, exact ? split_bf16x3_launch(src, dst[0], dst[1], dst[2], n, st) : cast_bf16_launch(src, dst[0], n, st));
  };
  // gz = (g T + g_h) * 1[h > 0]: the dense encoder over g (M = B, K = D) against T^T [H, D] with the ReLU-backward
  // epilogue, which also sums gz per column into grad_b_enc. Fast mode writes only bf16(gz), the operand of the
  // weight GEMMs; exact mode writes fp32 gz, the source of its three-part split.
  rc = parts("split g", g_recon, gp, nbd);
  if (rc != QSAE_OK) return rc;
  // grad b_enc = sum_b gz: column sums from the same epilogue (atomics)
  cudaError_t e = cudaMemsetAsync(grad_b_enc, 0, static_cast<size_t>(H) * 4, st);
  if (e != cudaSuccess) return fail(QSAE_ERR_CUDA, "tsae_backward: %s", cudaGetErrorString(e));
  EncodeLaunch el{};
  el.B = B; el.H = H; el.D = D; el.act = 3; el.bias = nullptr; el.gate = h; el.gate_add = g_h; el.gate_colsum = grad_b_enc;
  el.n_tiles = (H + kEncBN - 1) / kEncBN;
  el.n_splits = 1;
  el.tiles_per_split = el.n_tiles;
  const uint16_t* wt[1] = {t_t_bf16};
  const uint16_t* gpc[3] = {gp[0], gp[1], gp[2]};
  rc = launch_status("encode kernel (dense, ReLU backward)",
                     encode_dense_split_launch(gpc, wt, np, el, exact ? gz : nullptr, exact ? nullptr : gzp[0], nullptr,
                                               num_sms(), st, 1));
  if (rc != QSAE_OK) return rc;
  if (exact) {
    rc = launch_status("split gz", split_bf16x3_launch(gz, gzp[0], gzp[1], gzp[2], nbh, st));
    if (rc != QSAE_OK) return rc;
  }
  rc = parts("split h", h, hp, nbh);
  if (rc != QSAE_OK) return rc;
  rc = parts("split x", x, xp, nbd);
  if (rc != QSAE_OK) return rc;
  const uint16_t* gzc[3] = {gzp[0], gzp[1], gzp[2]};
  const uint16_t* xc[3] = {xp[0], xp[1], xp[2]};
  const uint16_t* hc[3] = {hp[0], hp[1], hp[2]};
  // grad W_enc [H, D] = gz^T x;  grad W_dec [D, H] = g^T h (already in decoder.weight's layout), then * mask
  rc = launch_status("wgrad (encoder)", wgrad_launch(gzc, xc, np, H, D, B, false, grad_w_enc, num_sms(), st));
  if (rc != QSAE_OK) return rc;
  rc = launch_status("wgrad (decoder)", wgrad_launch(gpc, hc, np, D, H, B, false, grad_w_dec, num_sms(), st));
  if (rc != QSAE_OK) return rc;
  if (mask) {
    rc = launch_status("mul_inplace", mul_inplace_launch(grad_w_dec, mask, nhd, st));
    if (rc != QSAE_OK) return rc;
  }
  if (grad_x) {   // grad x [B, D] = gz W_enc: gz is the K-major A (K = H), W_enc [H, D] the MN-major B
    const uint16_t* wc[3] = {w_hi, exact ? w_mid : w_hi, exact ? w_lo : w_hi};
    rc = launch_status("wgrad (input)", wgrad_launch(gzc, wc, np, B, D, H, true, grad_x, num_sms(), st));
  }
  return rc;
}

// ---- baseline_sae backward: deterministic, latent-major (csrc/train.cu)
namespace {
int check_baseline_backward(int B, int H, int D, int k) {
  if (B < 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "baseline_backward: negative batch");
  const int rc = check_encode_shape(B > 0 ? B : 1, H, D);   // the forward's shape rules
  if (rc != QSAE_OK) return rc;
  if (k < 1) return fail(QSAE_ERR_INVALID_ARGUMENT, "k must be >= 1, got %d", k);
  if (k > H) return fail(QSAE_ERR_K_OUT_OF_RANGE, "selected index k out of range (k=%d > H=%d)", k, H);
  if (static_cast<long long>(B) * k > 0x7fffffffLL)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "baseline_backward: B k = %lld entries exceed 2^31 - 1", static_cast<long long>(B) * k);
  return QSAE_OK;
}
}  // namespace

int qsae_baseline_backward_workspace_bytes(int B, int H, int D, int k, size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  const int rc = check_baseline_backward(B, H, D, k);
  if (rc != QSAE_OK) return rc;
  *bytes = baseline_backward_workspace_bytes(B, H, D, k);
  return QSAE_OK;
}

int qsae_baseline_backward(const float* x, const float* vals, const int32_t* idx, const float* g_recon, const float* g_h,
                           const float* g_vals, const float* w_enc, const float* dec_rows, int B, int H, int D, int k,
                           float* grad_w_enc, float* grad_b_enc, float* grad_w_dec, float* grad_b_dec, float* grad_x,
                           void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_baseline_backward(B, H, D, k);
  if (rc != QSAE_OK) return rc;
  if (g_h && g_vals) return fail(QSAE_ERR_INVALID_ARGUMENT, "baseline_backward: pass the latent gradient as g_h or g_vals, not both");
  if (!grad_w_enc || !grad_b_enc || !grad_w_dec || !grad_b_dec)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "baseline_backward: null gradient pointer");
  cudaStream_t st = S(stream);
  const size_t nhd = static_cast<size_t>(H) * D;
  if (B == 0) {   // nothing selected: zero gradients
    cudaError_t e = cudaMemsetAsync(grad_w_enc, 0, nhd * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(grad_b_enc, 0, static_cast<size_t>(H) * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(grad_w_dec, 0, nhd * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(grad_b_dec, 0, static_cast<size_t>(D) * 4, st);
    return e == cudaSuccess ? QSAE_OK : fail(QSAE_ERR_CUDA, "baseline_backward: %s", cudaGetErrorString(e));
  }
  if (!x || !vals || !idx || !g_recon || !dec_rows || !workspace) return fail(QSAE_ERR_INVALID_ARGUMENT, "baseline_backward: null pointer");
  if (grad_x && !w_enc) return fail(QSAE_ERR_INVALID_ARGUMENT, "baseline_backward: grad_x needs W_enc");
  const size_t need = baseline_backward_workspace_bytes(B, H, D, k);
  if (workspace_bytes < need)
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "baseline_backward: workspace %zu < %zu bytes", workspace_bytes, need);
  const uintptr_t align16 = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(g_recon) |
                            reinterpret_cast<uintptr_t>(w_enc) | reinterpret_cast<uintptr_t>(dec_rows) |
                            reinterpret_cast<uintptr_t>(grad_w_enc) | reinterpret_cast<uintptr_t>(grad_x) |
                            reinterpret_cast<uintptr_t>(workspace);
  if ((align16 & 15) != 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "baseline_backward: workspace and row-major tensors must be 16-byte aligned");
  const char* err = baseline_backward_launch(x, vals, idx, g_recon, g_h, g_vals, w_enc, dec_rows, B, H, D, k, grad_w_enc,
                                             grad_b_enc, grad_w_dec, grad_b_dec, grad_x, workspace, st);
  return err == nullptr ? QSAE_OK : fail(QSAE_ERR_CUDA, "baseline_backward: %s", err);
}

// ---- b_sae backward: deterministic, latent-major, the logit chain rule fused in (csrc/train.cu)
namespace {
int check_bsae_backward(int B, int H, int D, int k, int n_bits) {
  if (B < 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_backward: negative batch");
  const int rc = check_encode_shape(B > 0 ? B : 1, H, D);   // the forward's shape rules
  if (rc != QSAE_OK) return rc;
  if (n_bits < 1 || n_bits > 8) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_backward: 1 <= n_bits <= 8, got %d", n_bits);
  if (k < 1) return fail(QSAE_ERR_INVALID_ARGUMENT, "k must be >= 1, got %d", k);
  if (k > H) return fail(QSAE_ERR_K_OUT_OF_RANGE, "selected index k out of range (k=%d > H=%d)", k, H);
  if (k > kMaxKLarge) return fail(QSAE_ERR_INVALID_ARGUMENT, "k=%d exceeds QSAE_MAX_K_LARGE=%d", k, kMaxKLarge);
  if (static_cast<long long>(B) * k > 0x7fffffffLL)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_backward: B k = %lld entries exceed 2^31 - 1", static_cast<long long>(B) * k);
  return QSAE_OK;
}
}  // namespace

int qsae_bsae_backward_workspace_bytes(int B, int H, int D, int k, int n_bits, size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  const int rc = check_bsae_backward(B, H, D, k, n_bits);
  if (rc != QSAE_OK) return rc;
  *bytes = baseline_backward_workspace_bytes(B, H, D, k);   // the same regions as the baseline_sae backward
  return QSAE_OK;
}

int qsae_bsae_backward(const float* x, const float* vals, const int32_t* idx, const float* g_recon, const float* soft_rows,
                       const float* logits, float q, const float* gp_dev, float gp_host, const float* w_enc, int B, int H,
                       int D, int k, int n_bits, float* grad_w_enc, float* grad_b_enc, float* grad_logits, float* grad_b_dec,
                       float* grad_x, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_bsae_backward(B, H, D, k, n_bits);
  if (rc != QSAE_OK) return rc;
  if (!grad_w_enc || !grad_b_enc || !grad_logits || !grad_b_dec)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_backward: null gradient pointer");
  if (!logits) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_backward: null pointer");
  const uintptr_t align16 = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(g_recon) |
                            reinterpret_cast<uintptr_t>(soft_rows) | reinterpret_cast<uintptr_t>(logits) |
                            reinterpret_cast<uintptr_t>(w_enc) | reinterpret_cast<uintptr_t>(grad_w_enc) |
                            reinterpret_cast<uintptr_t>(grad_logits) | reinterpret_cast<uintptr_t>(grad_x) |
                            reinterpret_cast<uintptr_t>(workspace);
  if ((align16 & 15) != 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_backward: workspace and row-major tensors must be 16-byte aligned");
  cudaStream_t st = S(stream);
  if (B == 0) {   // nothing selected: zero encoder / bias gradients, the polarize-only logit gradient
    const size_t nhd = static_cast<size_t>(H) * D;
    cudaError_t e = cudaMemsetAsync(grad_w_enc, 0, nhd * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(grad_b_enc, 0, static_cast<size_t>(H) * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(grad_b_dec, 0, static_cast<size_t>(D) * 4, st);
    if (e != cudaSuccess) return fail(QSAE_ERR_CUDA, "bsae_backward: %s", cudaGetErrorString(e));
    return launch_status("bsae_backward", bsae_logit_grad_launch(logits, nullptr, H, D, n_bits, gp_dev, gp_host, 0, grad_logits, st));
  }
  if (!x || !vals || !idx || !g_recon || !soft_rows || !workspace) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_backward: null pointer");
  if (grad_x && !w_enc) return fail(QSAE_ERR_INVALID_ARGUMENT, "bsae_backward: grad_x needs W_enc");
  const size_t need = baseline_backward_workspace_bytes(B, H, D, k);
  if (workspace_bytes < need)
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "bsae_backward: workspace %zu < %zu bytes", workspace_bytes, need);
  const char* err = bsae_backward_launch(x, vals, idx, g_recon, soft_rows, logits, q, gp_dev, gp_host, w_enc, B, H, D, k, n_bits,
                                         grad_w_enc, grad_b_enc, grad_logits, grad_b_dec, grad_x, workspace, st);
  return err == nullptr ? QSAE_OK : fail(QSAE_ERR_CUDA, "bsae_backward: %s", err);
}

// ---- q_sae dense fallback: any activity level (an untrained model is ~50 % active), level sums as GEMMs
int qsae_unpack_matryoshka_t(const uint32_t* packed, int H, int D, uint16_t* t_bf16, void* stream) {
  if (!packed || !t_bf16 || H <= 0 || D <= 0 || (D % 16) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "unpack_matryoshka_t: bad argument");
  return launch_status("unpack_matryoshka_t", unpack_matryoshka_t_launch(packed, H, D, t_bf16, S(stream)));
}

namespace {
struct MatDensePlan { size_t x_off, z_off, hi_off, lo_off, cnt_off, dec_off, total; };
int plan_matryoshka_dense(int B, int H, int D, MatDensePlan* mp) {
  if (B <= 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "B and H must be positive");
  if (D < 16 || D > 512 || (D % 16) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka: D must be a multiple of 16 in [16, 512], got %d", D);
  if ((H % 8) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka dense path: hidden_dim must be a multiple of 8, got %d (the A "
                "operand and T^T rows are not padded to 16 bytes; other hidden_dim values have the sparse path only)", H);
  const size_t bh = static_cast<size_t>(B) * H;
  mp->x_off = 0;
  mp->z_off = 3 * align_up(static_cast<size_t>(B) * D * 2, 1024);   // room for the three bf16 parts of x
  mp->hi_off = align_up(mp->z_off + bh * 4, 1024);
  mp->lo_off = align_up(mp->hi_off + bh * 2, 1024);
  mp->cnt_off = align_up(mp->lo_off + bh * 2, 1024);
  mp->dec_off = align_up(mp->cnt_off + matryoshka_dense_operand_scratch_bytes(), 1024);
  mp->total = align_up(mp->dec_off + 16 * static_cast<size_t>(B) * D * sizeof(float), 256);   // up to 16 K splits
  return QSAE_OK;
}
}  // namespace

int qsae_matryoshka_dense_workspace_bytes(int B, int H, int D, size_t* bytes) {
  if (!bytes) return fail(QSAE_ERR_INVALID_ARGUMENT, "workspace query: null pointer");
  MatDensePlan mp;
  int rc = plan_matryoshka_dense(B, H, D, &mp);
  if (rc != QSAE_OK) return rc;
  *bytes = mp.total;
  return QSAE_OK;
}

namespace {
// mask (or null): the activity mask of the forward's own decisions, bf16 [B, >= H] rows of mask_pitch elements
int matryoshka_forward_dense_impl(const float* x_f32, const uint16_t* w_hi, const uint16_t* w_mid, const uint16_t* w_lo,
                                  const float* b_enc, const uint16_t* t_bf16, const float* scale, const int* level_start_dev,
                                  const int* level_start_host, int n_levels, const float* dec_bias, int B, int H, int D,
                                  float* result, unsigned long long* level_count, uint16_t* mask, int mask_pitch,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return QSAE_OK;
  if (!x_f32 || !b_enc || !t_bf16 || !scale || !level_start_dev || !level_start_host || !result || !level_count || !workspace)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward_dense: null pointer");
  if (!w_hi) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward_dense: no encoder weights");
  if (n_levels < 1 || n_levels > 32) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward_dense: 1 <= n_levels <= 32");
  for (int i = 1; i <= n_levels; ++i) {
    if (level_start_host[i] <= level_start_host[i - 1])
      return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka dense path: level boundaries must be increasing");
  }
  if (level_start_host[0] != 0 || level_start_host[n_levels] != H)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka dense path: levels must cover [0, H)");
  MatDensePlan mp;
  int rc = plan_matryoshka_dense(B, H, D, &mp);
  if (rc != QSAE_OK) return rc;
  if (workspace_bytes < mp.total)
    return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "matryoshka_forward_dense: workspace %zu < %zu bytes", workspace_bytes, mp.total);
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward_dense: workspace must be 1024-byte aligned");
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  float* z = reinterpret_cast<float*>(ws + mp.z_off);
  uint16_t* a_hi = reinterpret_cast<uint16_t*>(ws + mp.hi_off);
  uint16_t* a_lo = reinterpret_cast<uint16_t*>(ws + mp.lo_off);
  cudaStream_t st = S(stream);
  cudaError_t ce = cudaMemsetAsync(level_count, 0, static_cast<size_t>(n_levels) * sizeof(unsigned long long), st);
  if (ce != cudaSuccess) return fail(QSAE_ERR_CUDA, "matryoshka_forward_dense: %s", cudaGetErrorString(ce));
  // 1. dense pre-activations on the tensor cores: one bf16 pass, or the fp32-accurate split product when
  //    the mid / lo parts of W are given (exact activity decisions for any fp32 operands)
  // 2. A = active * scale, split into bf16 hi / lo; activity counts per level -- written by the encoder's
  //    epilogue itself when the level boundaries are multiples of 128 (the fp32 pre-activations never reach
  //    HBM: 1.07 GB of traffic and two launches less at B = 4096, H = 32768), else by a streaming kernel
  bool fuse_step = tuning().dense_step_fused != 0;
  for (int i = 0; i <= n_levels; ++i) fuse_step = fuse_step && (level_start_host[i] % 128) == 0;
  if (fuse_step) {
    const StepOperand so = {kActiveThreshold, scale, level_start_dev, n_levels, level_count, mask, mask_pitch};
    rc = dense_encode_tc(x_f32, w_hi, w_mid, w_lo, b_enc, B, H, D, 2, ws + mp.x_off, nullptr, a_hi, a_lo, st, &so);
    if (rc != QSAE_OK) return rc;
  } else {
    rc = dense_encode_tc(x_f32, w_hi, w_mid, w_lo, b_enc, B, H, D, QSAE_ACT_NONE, ws + mp.x_off, z, nullptr, nullptr, st);
    if (rc != QSAE_OK) return rc;
    rc = launch_status("matryoshka_dense_operand",
                       matryoshka_dense_operand_launch(z, B, H, scale, kActiveThreshold, level_start_dev, n_levels, a_hi, a_lo,
                                                       level_count, ws + mp.cnt_off, st, mask, mask_pitch));
    if (rc != QSAE_OK) return rc;
  }
  // 3. one GEMM per level over its K range, outputs accumulated level by level (:121-129). A TMA base address must be
  //    16-byte aligned, so the ranges end at the cuts floor8(level_start[i + 1]); a level whose range is empty after
  //    the cut has no GEMM. When a boundary is off the 8-grid, a last kernel adds each level's leftover columns
  //    [cut, level_start[i + 1]) to that level alone and fills the levels without a GEMM (matryoshka.cu)
  const size_t bd = static_cast<size_t>(B) * D;
  int k0 = 0, prev = -1;
  bool tail = false;
  for (int i = 0; i < n_levels; ++i) {
    const int cut = level_start_host[i + 1] & ~7;
    tail = tail || cut != level_start_host[i + 1];
    if (cut == k0) continue;
    rc = launch_status("dense_decode (level)",
                       dense_decode_launch(a_hi + k0, a_lo + k0, H, t_bf16 + k0, H, B, cut - k0, D, prev < 0 ? dec_bias : nullptr,
                                           prev < 0 ? nullptr : result + prev * bd, result + i * bd, ws + mp.dec_off,
                                           num_sms(), st));
    if (rc != QSAE_OK) return rc;
    k0 = cut;
    prev = i;
  }
  if (tail)
    rc = launch_status("matryoshka_dense_tail", matryoshka_dense_tail_launch(a_hi, a_lo, t_bf16, level_start_dev, n_levels, B,
                                                                             H, D, dec_bias, result, st));
  return rc;
}
}  // namespace

int qsae_matryoshka_forward_dense(const float* x_f32, const uint16_t* w_hi, const uint16_t* w_mid, const uint16_t* w_lo,
                                  const float* b_enc,
                                  const uint16_t* t_bf16, const float* scale, const int* level_start_dev,
                                  const int* level_start_host, int n_levels, const float* dec_bias, int B, int H, int D,
                                  float* result, unsigned long long* level_count, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  return matryoshka_forward_dense_impl(x_f32, w_hi, w_mid, w_lo, b_enc, t_bf16, scale, level_start_dev, level_start_host,
                                       n_levels, dec_bias, B, H, D, result, level_count, nullptr, 0, workspace,
                                       workspace_bytes, stream);
}

int qsae_matryoshka_forward_dense_active(const float* x_f32, const uint16_t* w_hi, const uint16_t* w_mid, const uint16_t* w_lo,
                                         const float* b_enc, const uint16_t* t_bf16, const float* scale,
                                         const int* level_start_dev, const int* level_start_host, int n_levels,
                                         const float* dec_bias, int B, int H, int D, float* result,
                                         unsigned long long* level_count, uint16_t* active_mask, int mask_pitch,
                                         int mask_col, void* workspace, size_t workspace_bytes, void* stream) {
  if (!active_mask) return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward_dense_active: null mask");
  if (mask_col < 0 || mask_col + H > mask_pitch || (mask_pitch % 8) != 0 || (mask_col % 8) != 0 ||
      (reinterpret_cast<uintptr_t>(active_mask) & 15) != 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "matryoshka_forward_dense_active: the mask needs 16-byte aligned rows and columns "
                "(pitch %d, column %d, H %d: multiples of 8, column + H <= pitch)", mask_pitch, mask_col, H);
  return matryoshka_forward_dense_impl(x_f32, w_hi, w_mid, w_lo, b_enc, t_bf16, scale, level_start_dev, level_start_host,
                                       n_levels, dec_bias, B, H, D, result, level_count, active_mask + mask_col, mask_pitch,
                                       workspace, workspace_bytes, stream);
}

int qsae_residual_update(const float* residual, const float* recon, size_t n, float* out, void* stream) {
  if (n == 0) return QSAE_OK;
  if (!residual || !recon || !out) return fail(QSAE_ERR_INVALID_ARGUMENT, "residual_update: null pointer");
  if ((reinterpret_cast<uintptr_t>(residual) | reinterpret_cast<uintptr_t>(recon) | reinterpret_cast<uintptr_t>(out)) & 15)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "residual_update: buffers must be 16-byte aligned");
  return launch_status("residual_update", residual_update_launch(residual, recon, n, out, S(stream)));
}

int qsae_encode_dense_f32(const float* x_f32, const int32_t* rows, int R, const float* w_f32,
                          const float* b_enc, int H, int D, int act, float* z, void* stream) {
  if (R == 0) return QSAE_OK;
  if (!x_f32 || !w_f32 || !z || R < 0 || H <= 0 || D <= 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "encode_dense: bad argument");
  return launch_status("encode_dense", encode_dense_launch(x_f32, rows, R, w_f32, b_enc, H, D, act, z, S(stream)));
}

int qsae_topk_dense_workspace_bytes(int R, int H, int k, size_t* bytes) {
  if (!bytes || R < 0 || H <= 0 || k < 1) return fail(QSAE_ERR_INVALID_ARGUMENT, "topk_dense workspace: bad argument");
  *bytes = align_up(static_cast<size_t>(R) * kDenseCap * 8 + static_cast<size_t>(R) * 4, 256);
  return QSAE_OK;
}

int qsae_topk_dense(const float* z, int R, int H, int k, float* out_vals, int32_t* out_idx,
                    void* workspace, size_t workspace_bytes, void* stream) {
  if (R == 0) return QSAE_OK;
  if (!z || !out_vals || !out_idx || !workspace) return fail(QSAE_ERR_INVALID_ARGUMENT, "topk_dense: null pointer");
  if (k < 1) return fail(QSAE_ERR_INVALID_ARGUMENT, "k must be >= 1, got %d", k);
  if (k > H) return fail(QSAE_ERR_K_OUT_OF_RANGE, "selected index k out of range (k=%d > H=%d)", k, H);
  if (k > kMaxKLarge) return fail(QSAE_ERR_INVALID_ARGUMENT, "k=%d exceeds QSAE_MAX_K_LARGE=%d", k, kMaxKLarge);
  if (k > kMaxK)   // block-level radix select straight from the dense rows (no workspace)
    return launch_status("select_dense", select_dense_launch(z, R, H, k, num_sms(), out_vals, out_idx, S(stream)));
  size_t need = 0;
  qsae_topk_dense_workspace_bytes(R, H, k, &need);
  if (workspace_bytes < need) return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "topk_dense: workspace %zu < %zu", workspace_bytes, need);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  void* cand = ws;
  int* cnt = reinterpret_cast<int*>(ws + static_cast<size_t>(R) * kDenseCap * 8);
  int rc = launch_status("dense_candidates", dense_candidates_launch(z, R, H, k, cand, cnt, S(stream)));
  if (rc != QSAE_OK) return rc;
  SelectLaunch sl{};
  sl.B = R; sl.H = H; sl.D = 0; sl.k_sel = k; sl.k_out = k; sl.nsub = 1; sl.cap = kDenseCap;
  sl.cand = cand; sl.cand_cnt = cnt; sl.out_vals = out_vals; sl.out_idx = out_idx;
  return launch_status("select_topk kernel", select_topk_launch(sl, S(stream)));
}

static int check_decode(const char* who, const float* vals, const int32_t* idx, const void* dict,
                        float* recon, int B, int k, int H, int D, int d_mult) {
  if (!vals || !idx || !dict || !recon) return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: null pointer", who);
  if (B < 0 || k < 0 || H <= 0 || D <= 0 || (D % d_mult) != 0 || D > 1024)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "%s: need D %% %d == 0, D <= 1024 (D=%d)", who, d_mult, D);
  return QSAE_OK;
}

int qsae_decode_int4(const float* vals, const int32_t* idx, int B, int k, const uint8_t* packed, int H,
                     int D, float scale, const float* bias, float* recon, void* stream) {
  int rc = check_decode("decode_int4", vals, idx, packed, recon, B, k, H, D, 8);
  if (rc != QSAE_OK || B == 0) return rc;
  if ((reinterpret_cast<uintptr_t>(bias) | reinterpret_cast<uintptr_t>(recon)) & 15)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "decode_int4: bias and recon must be 16-byte aligned");
  return launch_status("decode_int4", decode_int4_launch(vals, idx, B, k, packed, H, D, scale, bias, recon, 0, S(stream)));
}

int qsae_decode_int8(const float* vals, const int32_t* idx, int B, int k, const int8_t* rows, int H,
                     int D, float scale, const float* bias, float* recon, void* stream) {
  int rc = check_decode("decode_int8", vals, idx, rows, recon, B, k, H, D, 4);
  if (rc != QSAE_OK || B == 0) return rc;
  return launch_status("decode_int8", decode_int8_launch(vals, idx, B, k, rows, H, D, scale, bias, recon, 0, S(stream)));
}

int qsae_decode_rows_f32(const float* vals, const int32_t* idx, int B, int k, const float* rows, int H,
                         int D, float scale, const float* bias, float* recon, void* stream) {
  int rc = check_decode("decode_rows_f32", vals, idx, rows, recon, B, k, H, D, 4);
  if (rc != QSAE_OK || B == 0) return rc;
  return launch_status("decode_rows_f32", decode_f32_launch(vals, idx, B, k, rows, H, D, scale, bias, recon, 0, S(stream)));
}

// ---------------------------------------------------------------------------------------------
// dictionary-sharded b_sae (SURVEY 8e): merge of gathered per-shard candidates, range-restricted decode
// ---------------------------------------------------------------------------------------------
int qsae_pack_candidates(const float* vals, const int32_t* idx, size_t n, void* out, void* stream) {
  if (n == 0) return QSAE_OK;
  if (!vals || !idx || !out) return fail(QSAE_ERR_INVALID_ARGUMENT, "pack_candidates: null pointer");
  return launch_status("pack_candidates", pack_candidates_launch(vals, idx, n, out, S(stream)));
}

int qsae_merge_candidates_workspace_bytes(int B, size_t* bytes) {
  if (!bytes || B < 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "merge_candidates workspace: bad argument");
  *bytes = align_up(256 + static_cast<size_t>(B > 0 ? B : 1) * 4, 256);
  return QSAE_OK;
}

}  // extern "C"

namespace {
int merge_candidates_impl(const void* cand_all, const void* const* list_bases, int n_shards, int B, int k_in,
                          int shard_latents, int k_out, float* out_vals, int32_t* out_idx, int32_t* incomplete,
                          void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return QSAE_OK;
  if ((!cand_all && !list_bases) || !out_vals || !out_idx || !workspace)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "merge_candidates: null pointer");
  if (n_shards < 1 || n_shards > 32 || k_in < 1 || k_out < 1 || shard_latents < 1)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "merge_candidates: need 1 <= n_shards <= 32, k_in, k_out >= 1");
  if (k_out > kMaxKLarge) return fail(QSAE_ERR_INVALID_ARGUMENT, "k=%d exceeds QSAE_MAX_K_LARGE=%d", k_out, kMaxKLarge);
  if (static_cast<long long>(n_shards) * k_in < k_out)
    return fail(QSAE_ERR_K_OUT_OF_RANGE, "selected index k out of range (k=%d > %d candidates)", k_out, n_shards * k_in);
  size_t need = 0;
  qsae_merge_candidates_workspace_bytes(B, &need);
  if (workspace_bytes < need) return fail(QSAE_ERR_WORKSPACE_TOO_SMALL, "merge_candidates: workspace %zu < %zu", workspace_bytes, need);
  cudaStream_t st = S(stream);
  int* counters = static_cast<int*>(workspace);
  int32_t* ovf_rows = reinterpret_cast<int32_t*>(static_cast<uint8_t*>(workspace) + 256);
  cudaError_t ce = cudaMemsetAsync(counters, 0, 2 * sizeof(int), st);
  if (ce != cudaSuccess) return fail(QSAE_ERR_CUDA, "merge_candidates: %s", cudaGetErrorString(ce));
  SelectLaunch sl{};
  sl.B = B; sl.H = n_shards * shard_latents; sl.k_sel = k_out; sl.k_out = k_out; sl.nsub = n_shards; sl.cap = k_in;
  sl.cand = cand_all;                 // [n_shards][B][k_in] entries, every list full
  sl.list_bases = list_bases;         // or one [B][k_in] list array per shard, in that shard's (peer) memory
  sl.row_stride = 1; sl.sub_stride = B; sl.sub_col_offset = shard_latents;
  sl.out_vals = out_vals; sl.out_idx = out_idx;
  sl.unsorted = g_unordered_topk;
  // every row has exactly n_shards * k_in candidates: pick the tier that holds them
  const long long n_cand = static_cast<long long>(n_shards) * k_in;
  if (incomplete != nullptr) {   // truncated lists (k_in < the shards' full candidate count): completeness check
    ce = cudaMemsetAsync(incomplete, 0, sizeof(int32_t), st);
    if (ce != cudaSuccess) return fail(QSAE_ERR_CUDA, "merge_candidates: %s", cudaGetErrorString(ce));
    sl.incomplete = incomplete;
  }
  if (n_cand > 1024 || k_out > kMaxK || incomplete != nullptr)
    return launch_status("select_topk kernel", select_topk_launch(sl, st));
  const int tier = n_cand <= 256 ? 8 : (n_cand <= 512 ? 16 : 32);
  return launch_status("select_small kernel", select_small_launch(sl, tier, nullptr, nullptr, num_sms(), counters + 1, ovf_rows, st));
}
}  // namespace

extern "C" {

int qsae_merge_candidates(const void* cand_all, int n_shards, int B, int k_in, int shard_latents, int k_out,
                          float* out_vals, int32_t* out_idx, int32_t* incomplete, void* workspace, size_t workspace_bytes,
                          void* stream) {
  if (B > 0 && !cand_all) return fail(QSAE_ERR_INVALID_ARGUMENT, "merge_candidates: null pointer");
  return merge_candidates_impl(cand_all, nullptr, n_shards, B, k_in, shard_latents, k_out, out_vals, out_idx, incomplete,
                               workspace, workspace_bytes, stream);
}

int qsae_merge_candidates_peer(const void* const* list_bases, int n_shards, int B, int k_in, int shard_latents, int k_out,
                               float* out_vals, int32_t* out_idx, int32_t* incomplete, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (B > 0 && !list_bases) return fail(QSAE_ERR_INVALID_ARGUMENT, "merge_candidates_peer: null pointer");
  return merge_candidates_impl(nullptr, list_bases, n_shards, B, k_in, shard_latents, k_out, out_vals, out_idx, incomplete,
                               workspace, workspace_bytes, stream);
}

// ---- peer buffers (cudaMalloc + CUDA IPC) and the flag protocol ---------------------------------------------------------
int qsae_peer_alloc(size_t bytes, void** ptr) {
  if (!ptr || bytes == 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "peer_alloc: bad argument");
  cudaError_t e = cudaMalloc(ptr, bytes);   // on the CURRENT device: callers select it first (sharded.PeerExchange does)
  if (e == cudaSuccess) e = cudaMemset(*ptr, 0, bytes);
  if (e != cudaSuccess) return fail(QSAE_ERR_CUDA, "peer_alloc: %s", cudaGetErrorString(e));
  return QSAE_OK;
}

int qsae_peer_free(void* ptr) {
  if (!ptr) return QSAE_OK;
  cudaError_t e = cudaFree(ptr);
  return e == cudaSuccess ? QSAE_OK : fail(QSAE_ERR_CUDA, "peer_free: %s", cudaGetErrorString(e));
}

int qsae_peer_export(const void* ptr, unsigned char* handle64) {
  if (!ptr || !handle64) return fail(QSAE_ERR_INVALID_ARGUMENT, "peer_export: null pointer");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, const_cast<void*>(ptr));
  if (e != cudaSuccess) return fail(QSAE_ERR_CUDA, "peer_export: %s", cudaGetErrorString(e));
  memcpy(handle64, &h, 64);
  return QSAE_OK;
}

int qsae_peer_import(const unsigned char* handle64, void** ptr) {
  if (!handle64 || !ptr) return fail(QSAE_ERR_INVALID_ARGUMENT, "peer_import: null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return fail(QSAE_ERR_CUDA, "peer_import: %s", cudaGetErrorString(e));
  return QSAE_OK;
}

int qsae_peer_close(void* ptr) {
  if (!ptr) return QSAE_OK;
  cudaError_t e = cudaIpcCloseMemHandle(ptr);
  return e == cudaSuccess ? QSAE_OK : fail(QSAE_ERR_CUDA, "peer_close: %s", cudaGetErrorString(e));
}

int qsae_peer_signal(void* const* targets, int n, unsigned value, void* stream) {
  if (!targets) return fail(QSAE_ERR_INVALID_ARGUMENT, "peer_signal: null pointer");
  return launch_status("peer_signal", peer_signal_launch(reinterpret_cast<unsigned* const*>(targets), n, value, S(stream)));
}

int qsae_peer_wait(const unsigned* flags, int n, unsigned value, int32_t* timed_out, void* stream) {
  if (!flags || !timed_out) return fail(QSAE_ERR_INVALID_ARGUMENT, "peer_wait: null pointer");
  return launch_status("peer_wait", peer_wait_launch(flags, n, value, timed_out, S(stream)));
}

int qsae_reduce_partials_peer(const float* const* partial_bases, int n_shards, int row_begin, int rows, int D, float* out,
                              void* stream) {
  if (rows == 0) return QSAE_OK;
  if (!partial_bases || !out || n_shards < 1 || rows < 0 || row_begin < 0 || D <= 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "reduce_partials_peer: bad argument");
  return launch_status("reduce_partials_peer",
                       reduce_partials_peer_launch(partial_bases, n_shards, row_begin, rows, D, out, S(stream)));
}

int qsae_decode_int4_range(const float* vals, const int32_t* idx, int B, int k, const uint8_t* packed_shard,
                           int shard_latents, int idx_begin, int D, float scale, const float* bias, float* recon,
                           void* stream) {
  int rc = check_decode("decode_int4_range", vals, idx, packed_shard, recon, B, k, shard_latents, D, 8);
  if (rc != QSAE_OK || B == 0) return rc;
  if ((reinterpret_cast<uintptr_t>(bias) | reinterpret_cast<uintptr_t>(recon)) & 15)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "decode_int4_range: bias and recon must be 16-byte aligned");
  return launch_status("decode_int4", decode_int4_launch(vals, idx, B, k, packed_shard, shard_latents, D, scale, bias, recon,
                                                         idx_begin, S(stream), true));
}

int qsae_decode_int8_range(const float* vals, const int32_t* idx, int B, int k, const int8_t* rows_shard,
                           int shard_latents, int idx_begin, int D, float scale, const float* bias, float* recon,
                           void* stream) {
  int rc = check_decode("decode_int8_range", vals, idx, rows_shard, recon, B, k, shard_latents, D, 4);
  if (rc != QSAE_OK || B == 0) return rc;
  return launch_status("decode_int8", decode_int8_launch(vals, idx, B, k, rows_shard, shard_latents, D, scale, bias, recon,
                                                         idx_begin, S(stream)));
}

int qsae_densify(const float* vals, const int32_t* idx, int B, int k, int H, float* dense, void* stream) {
  if (B == 0) return QSAE_OK;
  if (!vals || !idx || !dense || B < 0 || k < 0 || H <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "densify: bad argument");
  return launch_status("densify", densify_launch(vals, idx, B, k, H, dense, S(stream)));
}

// --------------------------------------------------------------------------------------------
// host-buffer pipeline
// --------------------------------------------------------------------------------------------
struct qsae_bsae_plan {
  int H, D, n_bits, k, chunk;
  float qstep;
  const float* w_f32;
  const float* b_enc;
  const float* dec_bias;
  uint16_t* w_bf16;
  uint8_t* packed;
  uint16_t* w_sample;
  float* b_sample;
  int n_sample;
  int x_is_bf16, recon_mode;      // host formats (qsae_bsae_plan_set_io)
  int next_slot;                  // chunks go round the slots across calls
  static constexpr int kSlots = 4;
  struct Slot {
    cudaStream_t stream;
    float* x;
    uint16_t* x16;                // bf16 host input lands here and is widened on the device
    void* ws;
    size_t ws_bytes;
    float* vals;
    int32_t* idx;
    float* recon;
    uint16_t* recon16;            // bf16 host output
  } slot[kSlots];
  struct Pending {
    bool active;
    bool used[kSlots];
    cudaEvent_t done[kSlots];     // recorded on a slot's stream after the call's last operation there
  } pending[QSAE_MAX_PENDING];
};

void qsae_bsae_plan_destroy(qsae_bsae_plan* p) {
  if (!p) return;
  for (int s = 0; s < qsae_bsae_plan::kSlots; ++s) {
    auto& sl = p->slot[s];
    if (sl.stream) { cudaStreamSynchronize(sl.stream); cudaStreamDestroy(sl.stream); }
    cudaFree(sl.x); cudaFree(sl.x16); cudaFree(sl.ws); cudaFree(sl.vals); cudaFree(sl.idx); cudaFree(sl.recon); cudaFree(sl.recon16);
  }
  for (int t = 0; t < QSAE_MAX_PENDING; ++t)
    for (int s = 0; s < qsae_bsae_plan::kSlots; ++s)
      if (p->pending[t].done[s]) cudaEventDestroy(p->pending[t].done[s]);
  cudaFree(p->w_bf16);
  cudaFree(p->packed);
  cudaFree(p->w_sample);
  cudaFree(p->b_sample);
  delete p;
}

int qsae_bsae_plan_create(const float* w_enc, const float* b_enc, const float* logits, const float* dec_bias,
                          int H, int D, int n_bits, float gamma, int k, int max_chunk_rows,
                          qsae_bsae_plan** out) {
  if (!w_enc || !b_enc || !logits || !dec_bias || !out) return fail(QSAE_ERR_INVALID_ARGUMENT, "plan_create: null pointer");
  if (max_chunk_rows <= 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "plan_create: max_chunk_rows must be positive");
  if (n_bits < 1 || n_bits > 8) return fail(QSAE_ERR_INVALID_ARGUMENT, "plan_create: 1 <= n_bits <= 8");
  size_t ws_bytes = 0;
  const int n_sample = qsae_default_sample_rows(H);
  int rc = qsae_encode_topk_workspace_bytes(max_chunk_rows, H, D, k, n_sample, &ws_bytes);
  if (rc != QSAE_OK) return rc;
  qsae_bsae_plan* p = new (std::nothrow) qsae_bsae_plan();
  if (!p) return fail(QSAE_ERR_CUDA, "plan_create: out of host memory");
  memset(p, 0, sizeof(*p));
  p->H = H; p->D = D; p->n_bits = n_bits; p->k = k; p->chunk = max_chunk_rows;
  p->qstep = gamma / static_cast<float>(1 << (n_bits - 1));
  p->w_f32 = w_enc; p->b_enc = b_enc; p->dec_bias = dec_bias;
  const size_t packed_bytes = n_bits <= 4 ? static_cast<size_t>(H) * D / 2 : static_cast<size_t>(H) * D;
  p->n_sample = n_sample;
  cudaError_t e = cudaMalloc(&p->w_bf16, static_cast<size_t>(H) * D * 2);
  if (e == cudaSuccess) e = cudaMalloc(&p->packed, packed_bytes);
  if (e == cudaSuccess && n_sample > 0) e = cudaMalloc(&p->w_sample, static_cast<size_t>(n_sample) * D * 2);
  if (e == cudaSuccess && n_sample > 0) e = cudaMalloc(&p->b_sample, static_cast<size_t>(n_sample) * 4);
  for (int s = 0; s < qsae_bsae_plan::kSlots && e == cudaSuccess; ++s) {
    auto& sl = p->slot[s];
    sl.ws_bytes = ws_bytes;
    e = cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&sl.x, static_cast<size_t>(max_chunk_rows) * D * 4);
    if (e == cudaSuccess) e = cudaMalloc(&sl.x16, static_cast<size_t>(max_chunk_rows) * D * 2);
    if (e == cudaSuccess) e = cudaMalloc(&sl.ws, ws_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&sl.vals, static_cast<size_t>(max_chunk_rows) * k * 4);
    if (e == cudaSuccess) e = cudaMalloc(&sl.idx, static_cast<size_t>(max_chunk_rows) * k * 4);
    if (e == cudaSuccess) e = cudaMalloc(&sl.recon, static_cast<size_t>(max_chunk_rows) * D * 4);
    if (e == cudaSuccess) e = cudaMalloc(&sl.recon16, static_cast<size_t>(max_chunk_rows) * D * 2);
  }
  for (int t = 0; t < QSAE_MAX_PENDING && e == cudaSuccess; ++t)
    for (int s = 0; s < qsae_bsae_plan::kSlots && e == cudaSuccess; ++s)
      e = cudaEventCreateWithFlags(&p->pending[t].done[s], cudaEventDisableTiming);
  if (e != cudaSuccess) {
    qsae_bsae_plan_destroy(p);
    return fail(QSAE_ERR_CUDA, "plan_create: %s", cudaGetErrorString(e));
  }
  cudaStream_t st = p->slot[0].stream;
  rc = qsae_cast_f32_to_bf16(w_enc, p->w_bf16, static_cast<size_t>(H) * D, st);
  if (rc == QSAE_OK) rc = qsae_pack_bitplanes(logits, H, D, n_bits, p->packed, nullptr, st);
  if (rc == QSAE_OK && n_sample > 0)
    rc = qsae_prepare_encoder_sample(p->w_bf16, b_enc, H, D, n_sample, p->w_sample, p->b_sample, st);
  if (rc == QSAE_OK && (e = cudaStreamSynchronize(st)) != cudaSuccess)
    rc = fail(QSAE_ERR_CUDA, "plan_create: %s", cudaGetErrorString(e));
  if (rc != QSAE_OK) { qsae_bsae_plan_destroy(p); return rc; }
  *out = p;
  return QSAE_OK;
}

int qsae_bsae_plan_set_io(qsae_bsae_plan* p, int x_is_bf16, int recon_mode) {
  if (!p || recon_mode < 0 || recon_mode > 2) return fail(QSAE_ERR_INVALID_ARGUMENT, "plan_set_io: bad argument");
  for (int t = 0; t < QSAE_MAX_PENDING; ++t)
    if (p->pending[t].active) return fail(QSAE_ERR_INVALID_ARGUMENT, "plan_set_io: batches are still in flight");
  p->x_is_bf16 = x_is_bf16 != 0;
  p->recon_mode = recon_mode;
  return QSAE_OK;
}

}  // extern "C"

namespace {
// Enqueue one batch on the plan's slot streams. ramp: the synchronous call starts with small chunks so that the
// copy-out leg begins early; a stream of batches overlaps across calls instead and uses full chunks.
int enqueue_batch(qsae_bsae_plan* p, const void* x_host, int B, float* vals_host, int32_t* idx_host, void* recon_host,
                  bool ramp, bool* used) {
  int rc = QSAE_OK;
  int c = 0;
  // Chunk schedule of the synchronous call: the device -> host copy of the results is the longest leg (B * (8 k + 4 D)
  // bytes over PCIe), and it cannot start before the first chunk has been copied in and computed. So the first chunks
  // are small (2048 rows, doubling) to start the output stream early, the rest are as large as the plan allows because
  // the kernels are more efficient on large batches (the compute leg must stay ahead of the copy-out leg).
  int next_rows = (!ramp || p->chunk < 2048) ? p->chunk : 2048;
  const bool trace = ramp && tuning().debug_pipeline != 0;   // diagnostics: per-chunk event timeline on stderr
  constexpr int kTraceMax = 64;
  cudaEvent_t tev[kTraceMax][4];
  int trows[kTraceMax];
  if (trace) {
    for (int i = 0; i < kTraceMax; ++i) for (int j = 0; j < 4; ++j) cudaEventCreate(&tev[i][j]);
  }
  const size_t x_elem = p->x_is_bf16 ? 2 : 4;
  for (int r0 = 0, rows = 0; r0 < B && rc == QSAE_OK; r0 += rows, ++c) {
    const int si = p->next_slot;
    p->next_slot = (p->next_slot + 1) % qsae_bsae_plan::kSlots;
    auto& sl = p->slot[si];
    used[si] = true;
    rows = (B - r0 < next_rows) ? (B - r0) : next_rows;
    next_rows = (next_rows * 2 < p->chunk) ? next_rows * 2 : p->chunk;
    if (trace && c < kTraceMax) { trows[c] = rows; cudaEventRecord(tev[c][0], sl.stream); }
    cudaStream_t st = sl.stream;  // stream order protects the slot's buffers from its previous use
    const size_t n_x = static_cast<size_t>(rows) * p->D;
    cudaError_t e = cudaMemcpyAsync(p->x_is_bf16 ? static_cast<void*>(sl.x16) : static_cast<void*>(sl.x),
                                    static_cast<const uint8_t*>(x_host) + static_cast<size_t>(r0) * p->D * x_elem, n_x * x_elem,
                                    cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) { rc = fail(QSAE_ERR_CUDA, "forward_host H2D: %s", cudaGetErrorString(e)); break; }
    if (p->x_is_bf16) {
      rc = launch_status("upcast x", upcast_bf16_launch(sl.x16, sl.x, n_x, st));
      if (rc != QSAE_OK) break;
    }
    if (trace && c < kTraceMax) cudaEventRecord(tev[c][1], st);
    rc = qsae_bsae_forward(sl.x, p->w_bf16, p->w_f32, p->b_enc, p->w_sample, p->b_sample, p->n_sample, rows, p->H, p->D,
                           p->k, 0, p->packed, p->n_bits, p->qstep, p->dec_bias, sl.vals, sl.idx, nullptr, sl.recon, sl.ws,
                           sl.ws_bytes, st);
    if (rc != QSAE_OK) break;
    if (trace && c < kTraceMax) cudaEventRecord(tev[c][2], st);
    e = cudaMemcpyAsync(vals_host + static_cast<size_t>(r0) * p->k, sl.vals, static_cast<size_t>(rows) * p->k * 4,
                        cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(idx_host + static_cast<size_t>(r0) * p->k, sl.idx, static_cast<size_t>(rows) * p->k * 4,
                          cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && p->recon_mode == 0)
      e = cudaMemcpyAsync(static_cast<float*>(recon_host) + static_cast<size_t>(r0) * p->D, sl.recon, n_x * 4,
                          cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && p->recon_mode == 1) {
      rc = launch_status("cast recon", cast_bf16_launch(sl.recon, sl.recon16, n_x, st));
      if (rc != QSAE_OK) break;
      e = cudaMemcpyAsync(static_cast<uint16_t*>(recon_host) + static_cast<size_t>(r0) * p->D, sl.recon16, n_x * 2,
                          cudaMemcpyDeviceToHost, st);
    }
    if (e != cudaSuccess) rc = fail(QSAE_ERR_CUDA, "forward_host D2H: %s", cudaGetErrorString(e));
    if (trace && c < kTraceMax) cudaEventRecord(tev[c][3], st);
  }
  if (trace) {
    for (int s = 0; s < qsae_bsae_plan::kSlots; ++s) cudaStreamSynchronize(p->slot[s].stream);
    const int nc = c < kTraceMax ? c : kTraceMax;
    for (int i = 0; i < nc && rc == QSAE_OK; ++i) {
      float t[4] = {0.f, 0.f, 0.f, 0.f};
      for (int j = 0; j < 4; ++j) cudaEventElapsedTime(&t[j], tev[0][0], tev[i][j]);
      fprintf(stderr, "[qsae pipeline] chunk %2d rows %6d: start %.3f  h2d done %.3f  compute done %.3f  d2h done %.3f ms\n", i,
              trows[i], t[0], t[1], t[2], t[3]);
    }
    for (int i = 0; i < kTraceMax; ++i) for (int j = 0; j < 4; ++j) cudaEventDestroy(tev[i][j]);
  }
  return rc;
}
}  // namespace

extern "C" {

int qsae_bsae_forward_host(qsae_bsae_plan* p, const float* x_host, int B, float* vals_host,
                           int32_t* idx_host, float* recon_host) {
  if (!p || !x_host || !vals_host || !idx_host || (!recon_host && p && p->recon_mode != 2) || B < 0)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "forward_host: bad argument");
  bool used[qsae_bsae_plan::kSlots] = {false, false, false, false};
  int rc = enqueue_batch(p, x_host, B, vals_host, idx_host, recon_host, true, used);
  for (int s = 0; s < qsae_bsae_plan::kSlots; ++s) {
    cudaError_t e = cudaStreamSynchronize(p->slot[s].stream);
    if (e != cudaSuccess && rc == QSAE_OK) rc = fail(QSAE_ERR_CUDA, "forward_host sync: %s", cudaGetErrorString(e));
  }
  return rc;
}

int qsae_bsae_submit_host(qsae_bsae_plan* p, const void* x_host, int B, float* vals_host, int32_t* idx_host,
                          void* recon_host, int* ticket) {
  if (!p || !x_host || !vals_host || !idx_host || (!recon_host && p && p->recon_mode != 2) || B < 0 || !ticket)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "submit_host: bad argument");
  int t = -1;
  for (int i = 0; i < QSAE_MAX_PENDING; ++i)
    if (!p->pending[i].active) { t = i; break; }
  if (t < 0) return fail(QSAE_ERR_INVALID_ARGUMENT, "submit_host: %d batches already in flight; wait for one first", QSAE_MAX_PENDING);
  auto& pd = p->pending[t];
  for (int s = 0; s < qsae_bsae_plan::kSlots; ++s) pd.used[s] = false;
  int rc = enqueue_batch(p, x_host, B, vals_host, idx_host, recon_host, false, pd.used);
  for (int s = 0; s < qsae_bsae_plan::kSlots; ++s) {
    if (!pd.used[s]) continue;
    cudaError_t e = cudaEventRecord(pd.done[s], p->slot[s].stream);
    if (e != cudaSuccess && rc == QSAE_OK) rc = fail(QSAE_ERR_CUDA, "submit_host: %s", cudaGetErrorString(e));
  }
  pd.active = true;   // also after an error: the caller waits (and thereby drains) what was enqueued
  *ticket = t;
  return rc;
}

int qsae_bsae_wait_host(qsae_bsae_plan* p, int ticket) {
  if (!p || ticket < 0 || ticket >= QSAE_MAX_PENDING || !p->pending[ticket].active)
    return fail(QSAE_ERR_INVALID_ARGUMENT, "wait_host: unknown ticket %d", ticket);
  auto& pd = p->pending[ticket];
  int rc = QSAE_OK;
  for (int s = 0; s < qsae_bsae_plan::kSlots; ++s) {
    if (!pd.used[s]) continue;
    cudaError_t e = cudaEventSynchronize(pd.done[s]);
    if (e != cudaSuccess && rc == QSAE_OK) rc = fail(QSAE_ERR_CUDA, "wait_host: %s", cudaGetErrorString(e));
  }
  pd.active = false;
  return rc;
}

}  // extern "C"
