// Internal declarations shared by the .cu files behind the C ABI (include/qsae_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace qsae {

constexpr int kEncBM = 128;        // rows of x per CTA
constexpr int kEncBN = 256;        // latents per accumulator tile
constexpr int kCandCapMax = 1024;  // largest per-(row, sub-stream) survivor buffer
constexpr int kDenseCap = 256;     // survivor buffer of the dense top-k kernel
constexpr int kMaxSplits = 8;      // max CTAs sharing one row block along the latent axis
constexpr int kMaxK = 224;         // == QSAE_MAX_K: largest k of the warp-level selection paths
constexpr int kMaxKLarge = 4096;   // == QSAE_MAX_K_LARGE: largest k of the block-level (radix select) paths
constexpr size_t kSelectSmemBudget = 200 * 1024;   // shared memory of the block-per-row select kernels
constexpr int kTopM = 64;          // values a thread keeps in the sample pre-pass (mode 5): top 2 of 32 column classes
constexpr int kPriorMaxRank = 32;
constexpr int kRescueSlots = 8;    // rows the tail kernel recomputes with the whole grid at a time (scratch: one dense row each)
constexpr int kPriorCounters = 4 + kRescueSlots;   // ints zeroed per call: [0] rescue rows, [1] block-select rows, [4..] slot tickets  // largest rank m of the prior threshold among a row's nsub * kTopM kept values

// Tuning / diagnostic switches, read ONCE from the environment (never on a launch path); qsae_reload_tuning()
// re-reads them (tests and tuning experiments that change the environment of a live process).
struct Tuning {
  int encode_cluster;     // QSAE_ENCODE_CLUSTER: 0 / 1 / 2 forces the cluster variant (-1 = automatic; dense: 0 / 2)
  int encode_range;       // QSAE_ENCODE_RANGE: 0 keeps the (split, row block) grid at small batches
  int encode_range_pair;  // QSAE_ENCODE_RANGE_PAIR: 1 = cta_group::2 pairs on the range schedule (sparse sweeps)
  int encode_specialised; // QSAE_ENCODE_SPECIALISED: 0 = prior-threshold sweeps on the generic kernel (all modes compiled in)
  int merge_tier;         // QSAE_MERGE_TIER: 8 / 12 / 16 forces the keys per lane of the warp merge (0 = from the expected survivor count)
  int sample_div;         // QSAE_SAMPLE_DIV: the sampled prior works on H / sample_div of the latents
  int prior_prep;         // QSAE_PRIOR_PREP: 0 keeps the separate cast / pre-pass / prior kernels
  int dense_step_fused;   // QSAE_DENSE_STEP_FUSED: 0 = q_sae dense path writes fp32 pre-activations and runs the separate operand kernel
  int decode_pair;        // QSAE_DECODE_PAIR: 0 / 1 forces the decoder GEMM variant (-1 = automatic)
  int peer_timeout_ms;    // QSAE_PEER_TIMEOUT_MS: bound of a peer-memory flag wait (default 20000)
  int debug_large;        // QSAE_DEBUG_LARGE: survivor statistics of the large-k path on stderr (synchronises)
  int debug_pipeline;     // QSAE_DEBUG_PIPELINE: per-chunk event timeline of the host-buffer pipeline on stderr
};
const Tuning& tuning();
void reload_tuning();
// kernels launched by this library in this process (qsae_launch_count): the C-ABI wrappers count one per *_launch
// call, launchers that start further kernels add them here
void count_launches(int n);

struct EncodeLaunch {
  int B, H, D;
  int k_sel;            // survivors that must be retained per row (k, or k + rescore margin)
  int n_splits;         // grid.x
  int nsub;             // survivor lists per row: 2 n_splits, or the range schedule's 2 x max pieces per row block
  int range_g;          // > 0: range schedule (encode_topk_sm100.cu) with this many CTAs (or CTA pairs) instead of the (split, row block) grid
  int range_pair;       // range schedule over cta_group::2 pairs (range_g pairs, 2 range_g CTAs)
  int tiles_per_split;  // in units of kEncBN latents
  int n_tiles;          // ceil(H / kEncBN)
  int act;              // 0 none, 1 relu; dense epilogue only: 2 = step operand, out = (z >= step_thr) ? step_scale[col] : 0,
                        // 3 = ReLU backward, out = (acc + gate_add) * (gate > 0) (streamed-operand kernel, no bias)
  int mode;             // epilogue bound: 0 bisection only, 1/2/3 class maxima, 4 prior (see .cu)
  int cap;              // entries per survivor buffer
  const float* bias;    // [H]
  const float* prior;   // mode 4: per-row threshold at prior[row * prior_stride]; null: prior_const for every row
  int prior_stride;
  float prior_const;
  int* overflow;        // mode 4 with k_sel <= 0 (threshold only): set to 1 when a buffer filled up
  float* top_out;       // mode 5: [B][n_splits*2][kTopM] the two largest values of each column class, per sub-stream
  void* cand;           // [B][n_splits*2][cap] {float bits, int32 column}
  int* cand_cnt;        // [B][n_splits*2]
  float* cand_thr;      // [B][n_splits*2] inclusive lower bound of the row's k_sel-th largest value
  int cluster;          // 0 single CTA, 1 TMA-multicast pair, 2 cta_group::2 pair (set by the launcher)
  int dense_flags;      // dense epilogue outputs: 1 fp32, 2 bf16 hi, 4 bf16 lo (set by the launcher)
  float* out_f32;       // dense epilogue: [B, H] row-major outputs (set by the launcher)
  uint16_t* out_hi;
  uint16_t* out_lo;
  // act == 2 (q_sae dense path: the A operand of the level GEMMs written straight from the encoder epilogue)
  float step_thr;
  const float* step_scale;            // [H]
  const int* step_level_start;        // [step_n_levels + 1] device, multiples of 128
  int step_n_levels;
  unsigned long long* step_level_count;   // [step_n_levels] += active (row, latent) pairs per level
  uint16_t* step_mask;                // or null: bf16 activity mask, 1.0 where z >= step_thr; row r at step_mask + r * pitch
  int step_mask_pitch;                // elements, a multiple of 8
  // act == 3 (t_sae backward: gz = (g T + g_h) * 1[h > 0] straight from the accumulator of g T)
  const float* gate;      // [B, H] the forward's ReLU output h
  const float* gate_add;  // [B, H] d loss / d h, or null
  float* gate_colsum;     // [H] += column sums of the output (the bias gradient), or null
  float* debug_z;       // optional dense [B, H] dump of the accumulator (+bias, act); diagnostics only
};

// encode_topk_sm100.cu
int encode_pick_splits(int B, int H, int num_sms);
// range schedule for this shape: CTAs to launch (0 = keep the (split, row block) grid) and lists per row
int encode_pick_range(int B, int H, int num_sms, int* nsub, int* pair = nullptr);
void encode_pick_mode(int k_sel, int* mode, int* cap);
const char* encode_topk_launch(const uint16_t* x_bf16, const uint16_t* w_bf16, EncodeLaunch p,
                               cudaStream_t stream);

// Prior of the sampled-threshold path in ONE launch for small batches (replaces cast + sample pre-pass + prior
// kernel): clusters of `ns` CTAs per 128-row block convert x to bf16 (shared memory operand + the global copy the
// sweep reads), contract it against their share of the sampled dictionary rows on the tensor cores, keep one running
// maximum per (thread, column mod 32) class, exchange the maxima through distributed shared memory and write
// prior[row] = m-th largest class maximum (a lower bound of the m-th largest sampled pre-activation).
struct PrepLaunch {
  int B, D, n_sample, act, m;
  int ns;                  // CTAs per row block = cluster size: 2 or 4
  const float* x_f32;      // [B, D]
  uint16_t* x_bf16;        // [B, D] out
  const float* bias;       // [n_sample] bias of the sampled rows
  float* prior;            // [B] out
  int* zero_counters;      // kPriorCounters ints cleared by the first block (saves the memset node), or null
};
// ns for this shape, 0 = use the separate kernels (large batches, narrow inputs)
int prior_prep_pick_ns(int B, int D, int n_sample, int m, int num_sms);
const char* prior_prep_launch(const uint16_t* w_sample, const PrepLaunch& p, cudaStream_t stream);

// dense epilogue variant (t_sae fast mode, q_sae dense path): h = act(x W^T + b) from one bf16 product, written as fp32
// and/or bf16 hi (+ lo) [B, H]; x tile resident, W streamed (single CTAs or cta_group::2 pairs, p.range_g ignored)
const char* encode_dense_tc_launch(const uint16_t* x_bf16, const uint16_t* w_bf16, EncodeLaunch p, float* out_f32,
                                   uint16_t* out_hi, uint16_t* out_lo, cudaStream_t stream);
// the fp32-accurate product (x and W as three bf16 parts each, six partial products) in ONE launch: both operands
// stream through the ring, every product lands in the same TMEM accumulator, the output is written once
// (p.bias / p.act applied; p.n_tiles as for encode_dense_tc_launch; a range schedule over num_sms / 2 CTA pairs)
// n_parts = 1: only the bf16 product x_parts[0] w_parts[0] (fast-mode t_sae backward) on the same schedule
// n_w_parts = 1 with n_parts = 3: the three x parts against ONE W part (exact when W is bf16-representable, e.g. ternary)
const char* encode_dense_split_launch(const uint16_t* const* x_parts, const uint16_t* const* w_parts, int n_parts, EncodeLaunch p,
                                      float* out_f32, uint16_t* out_hi, uint16_t* out_lo, int num_sms, cudaStream_t stream,
                                      int n_w_parts = 0);
// src -> three bf16 parts with hi + mid + lo == src exactly (24 mantissa bits); mid / lo may be null
const char* split_bf16x3_launch(const float* src, uint16_t* hi, uint16_t* mid, uint16_t* lo, size_t n, cudaStream_t stream);

// dense_decode_sm100.cu: out[B, N] = (a_hi (+ a_lo))[B, K] * b_t[N, K]^T (+ bias), bf16 in, fp32 accumulate
int dense_decode_pick_splits(int B, int K, int num_sms);
size_t dense_decode_workspace_bytes(int B, int K, int N, int num_sms);
// lda / ldb: row pitches in elements (a K sub-range of a wider matrix keeps the full pitch);
// prev: optional [B, N] added to the result (cumulative per-level outputs)
const char* dense_decode_launch(const uint16_t* a_hi, const uint16_t* a_lo, int lda, const uint16_t* b_t, int ldb, int B,
                                int K, int N, const float* bias, const float* prev, float* out, void* workspace,
                                int num_sms, cudaStream_t stream);

// wgrad_sm100.cu: c[M, N] = sum_k A(k, m) B(k, n) over K rows (the batch), bf16 parts, fp32 accumulation.
// b_parts: row-major [K, N]; a_parts: row-major [K, M], or [M, K] when a_kmajor. n_parts = 1 (one product) or 3 (the six
// products of three-part splits above 2^-24, one accumulator). N and the row pitch of A multiples of 8; c [M, N] fp32,
// overwritten.
// cooc[H, H] int32 += M^T M of a bf16 0/1 mask M [K, H] (K <= 2^24, H % 8 == 0), upper-triangle tiles only, each
// product element added to cooc[m, n] and, for n > m, to cooc[n, m] (one writer per element, no atomics);
// counts[h] += the diagonal (or null)
const char* coactivation_dense_launch(const uint16_t* mask, int K, int H, int32_t* cooc, long long* counts, int num_sms,
                                      cudaStream_t stream);
const char* wgrad_launch(const uint16_t* const* a_parts, const uint16_t* const* b_parts, int n_parts, int M, int N, int K,
                         bool a_kmajor, float* c, int num_sms, cudaStream_t stream);
// q_sae STE backward from a dense activity mask: grad_w[h, :] += alpha[h] (mask[:, h]^T g_level(h)) s'(w[h, :]), the same
// for the mirror. mask bf16 0/1 [B, H] (H % 8 == 0); g_parts: n_parts (1 or 3) bf16 parts, each the n_levels level
// gradients stacked [n_levels B, D] (D % 16 == 0); level_start host [n_levels + 1]. One writer per element, no atomics.
const char* matryoshka_ste_dense_launch(const uint16_t* mask, int B, int H, int D, const uint16_t* const* g_parts, int n_parts,
                                        const int* level_start, int n_levels, const float* w, const float* w_mirror,
                                        const float* alpha, float* grad_w, float* grad_w_mirror, int num_sms,
                                        cudaStream_t stream);

// select_topk.cu
struct SelectLaunch {
  int B, H, D, k_sel, k_out, nsub, cap, act, exact;
  const void* cand;       // as above
  const int* cand_cnt;
  const float* cand_thr;  // may be null
  const float* x_f32;     // [B, D]   (exact only)
  const float* w_f32;     // [H, D]   (exact only)
  const float* bias;      // [H]      (exact only)
  float* out_vals;        // [B, k_out]
  int32_t* out_idx;       // [B, k_out]
  int32_t* out_flags;     // [B] or null
  int* rescue_count;      // rows that need the exact recomputation (failed count check, uncertified in exact mode) ...
  int32_t* rescue_rows;   // ... are appended here (capacity B) and their output left to the rescue kernel
  int check_count;        // prior mode: the threshold is only probably valid, so a row with fewer than k_sel
                          // survivors (or a list that filled up) is sent to the rescue list
  // Layout of the survivor lists: list (row, s) starts at entry (row * row_stride + s * sub_stride) * cap.
  // 0 / 0 = the fused encoder's layout [B][nsub][cap]. Gathered per-shard candidates are [nsub][B][cap].
  long long row_stride, sub_stride;
  int sub_col_offset;     // column of an entry of list s is stored_col + s * sub_col_offset (dictionary shards)
  int unsorted;           // block-level select (k > 224), fast mode: emit the k winners as a set, in no particular order
  // Truncated candidate lists (dictionary shards send fewer than k candidates each): *incomplete is set to 1 when,
  // for some row, every entry of some list was selected -- entries that list's owner did not send could then
  // belong to the row's true top-k. Block-per-row kernel only; null = lists are complete, no check.
  int* incomplete;
  // Lists that live in peer memory (dictionary shards, CUDA IPC): list s of row r starts at
  // list_bases[s] + r * cap entries (device array of nsub pointers); null = the cand / stride layout above.
  const void* const* list_bases;
  // Fused decode (prior path of qsae_bsae_forward): the warp / block that has just selected a row also decodes it,
  // recon[row, :] = dec_scale * sum_j v_j * dict[i_j, :] + dec_bias (sae/binary.py:38). dec_kind 0 = off,
  // 1 = packed int4 dictionary with D == 512 (one uint2 per lane), k_out <= 128.
  int dec_kind;
  const uint32_t* dec_packed;   // [H, D / 8] words
  float dec_scale;
  const float* dec_bias;        // [D] or null
  float* dec_recon;             // [B, D]
};

// rescue.cu: exact per-row top-k for the rows listed by the merge kernel (persistent small grid,
// returns immediately when the list is empty)
struct RescueLaunch {
  int B, H, D, k_sel, k_out, act, exact;
  const uint16_t* x_bf16;  // [B, D]
  const uint16_t* w_bf16;  // [H, D]
  const float* x_f32;      // exact only
  const float* w_f32;      // exact only
  const float* bias;       // [H]
  const int* rescue_count;
  const int32_t* rescue_rows;
  float* out_vals;
  int32_t* out_idx;
  int32_t* out_flags;      // may be null
  // tail kernel only: the first kRescueSlots listed rows are recomputed by the WHOLE grid (every block scores its
  // slice of the dictionary into z_scratch[slot][H], the last block to finish selects): one row costs tens of
  // microseconds instead of milliseconds on a single block. null: every row block-per-row (rescue_one_row).
  float* z_scratch;        // [kRescueSlots, H]
  int* slot_done;          // [kRescueSlots] tickets, zero on entry
};
const char* rescue_rows_launch(const RescueLaunch& p, int num_sms, cudaStream_t stream);

// pack.cu: gather a stratified pseudo-random sample of dictionary rows (prior-threshold pre-pass)
const char* sample_rows_launch(const uint16_t* w_bf16, const float* bias, int H, int D, int n_sample,
                               uint16_t* w_sample, float* b_sample, cudaStream_t stream);
const char* select_topk_launch(const SelectLaunch& p, cudaStream_t stream);
// ordered top-k of every row of a dense [R, H] matrix, any k <= kMaxKLarge (block-level radix select)
const char* select_dense_launch(const float* z, int R, int H, int k, int num_sms, float* out_vals, int32_t* out_idx,
                                cudaStream_t stream);
// large-k counterpart of rescue_rows_launch (k_out <= kMaxKLarge); scratch: rescue_large_scratch_bytes
size_t rescue_large_scratch_bytes(int H, int num_sms);
const char* rescue_large_launch(const RescueLaunch& p, void* scratch, int num_sms, cudaStream_t stream);
// warp-per-row merge for small survivor counts (prior mode / gathered shard candidates). tier = keys per
// lane (8 / 16 / 32: rows with up to 256 / 512 / 1024 survivors); rows that do not fit are appended to
// ovf_rows / ovf_count for the next tier. rows == nullptr: every row of the batch; else the device-side list
// rows[0, *count) on a persistent grid.
const char* select_small_launch(const SelectLaunch& p, int tier, const int* count, const int32_t* rows, int num_sms,
                                int* ovf_count, int32_t* ovf_rows, cudaStream_t stream);
const char* select_topk_list_launch(const SelectLaunch& p, const int* count, const int32_t* rows, int num_sms,
                                    cudaStream_t stream);
// Tail of the prior path in ONE launch (persistent grid, returns at once when both lists are empty): rows the
// warp-level merge could not hold (ovf_rows[0, *ovf_count): block-per-row radix select) and rows whose prior
// failed the count check (r.rescue_rows[0, *r.rescue_count): exact recomputation); a row the block select wants
// recomputed is recomputed by the same block. Every row handled here is also decoded when p.dec_kind != 0.
const char* select_tail_launch(const SelectLaunch& p, const RescueLaunch& r, const int* ovf_count,
                               const int32_t* ovf_rows, int num_sms, cudaStream_t stream);
// prior[row] = m-th largest of the row's nsub * kTopM pre-pass values
const char* prior_from_top_launch(const float* top, int B, int nsub, int m, float* prior, cudaStream_t stream);
// survivors from a dense [R, H] matrix (one sub-stream per row, buffers of kDenseCap entries)
const char* dense_candidates_launch(const float* z, int R, int H, int k, void* cand, int* cand_cnt,
                                    cudaStream_t stream);

// pack.cu
const char* cast_bf16_launch(const float* src, uint16_t* dst, size_t n, cudaStream_t stream);
// bf16 -> float32 (exact)
const char* upcast_bf16_launch(const uint16_t* src, float* dst, size_t n, cudaStream_t stream);
const char* pack_bitplanes_launch(const float* logits, int H, int D, int n_bits, uint8_t* packed,
                                  double* stats, cudaStream_t stream);
const char* dequant_soft_launch(const float* logits, int H, int D, int n_bits, float* rows,
                                cudaStream_t stream);
const char* transpose_launch(const float* src, int R, int C, float* dst, cudaStream_t stream);
// out = (r - recon) * 2 (rq_sae residual step)
const char* residual_update_launch(const float* r, const float* recon, size_t n, float* out, cudaStream_t stream);
// src -> hi = bf16(src), lo = bf16(src - hi) (lo may be null)
const char* split_bf16_launch(const float* src, uint16_t* hi, uint16_t* lo, size_t n, cudaStream_t stream);
// t_sae decoder.weight [D, H] -> sign(w) * (|w| >= threshold): bf16 [D, H] and/or int8 rows [H, D]
// t_t_bf16: the same T transposed, bf16 [H, D] (K-major B operand of the t_sae backward's g T); may be null
const char* pack_ternary_launch(const float* w, int D, int H, float threshold, uint16_t* t_bf16, int8_t* t_rows,
                                cudaStream_t stream, uint16_t* t_t_bf16 = nullptr);

// decode.cu
// idx_offset: the dictionary holds latents [idx_offset, idx_offset + H); other entries are skipped
const char* decode_int4_launch(const float* vals, const int32_t* idx, int B, int k,
                               const uint8_t* packed, int H, int D, float scale, const float* bias,
                               float* recon, int idx_offset, cudaStream_t stream, bool skip_unowned = false);
const char* decode_int8_launch(const float* vals, const int32_t* idx, int B, int k,
                               const int8_t* rows, int H, int D, float scale, const float* bias,
                               float* recon, int idx_offset, cudaStream_t stream);
const char* decode_f32_launch(const float* vals, const int32_t* idx, int B, int k, const float* rows,
                              int H, int D, float scale, const float* bias, float* recon, int idx_offset,
                              cudaStream_t stream);
// (vals, idx) [n] -> interleaved {float bits, column} entries, the survivor-list format of the merge kernels
const char* pack_candidates_launch(const float* vals, const int32_t* idx, size_t n, void* out, cudaStream_t stream);
const char* densify_launch(const float* vals, const int32_t* idx, int B, int k, int H, float* dense,
                           cudaStream_t stream);

// matryoshka.cu
const char* pack_matryoshka_launch(const float* w, const float* wm, int H, int D, const int* level_start,
                                   const float* level_factor, int n_levels, uint32_t* packed, float* scale,
                                   cudaStream_t stream);
const char* decode_matryoshka_launch(const void* cand, const int* cand_cnt, int nsub, int cap, int B,
                                     const uint32_t* packed, const float* scale, const int* level_start,
                                     int n_levels, int H, int D, const float* bias, float* result,
                                     unsigned long long* level_count, const float* x_f32, const float* w_f32,
                                     const float* b_enc, float thr_value, int exact, void* scratch, int num_sms,
                                     cudaStream_t stream, int32_t* active_idx = nullptr, int active_cap = 0,
                                     int* active_cnt = nullptr, const float* resid_in = nullptr, float* resid_out = nullptr,
                                     const int* poison_flag = nullptr);
// scratch of decode_matryoshka_launch (per-warp activity counts before the final sum)
size_t decode_matryoshka_scratch_bytes(int num_sms);
// packed 2-bit codes [H, D/16] -> T^T as bf16 [D, H] with entries {-2, 0, +2} (B operand of the dense level GEMMs)
const char* unpack_matryoshka_t_launch(const uint32_t* packed, int H, int D, uint16_t* t_bf16, cudaStream_t stream);
// z [B, H] -> a = (z >= thr) * scale[h] split into bf16 hi / lo [B, H]; level_count[l] += active entries of level l;
// mask (or null): bf16 1.0 / 0.0 = (z >= thr), row b at mask + b * mask_pitch (a multiple of 8 elements)
const char* matryoshka_dense_operand_launch(const float* z, int B, int H, const float* scale, float thr,
                                            const int* level_start, int n_levels, uint16_t* a_hi, uint16_t* a_lo,
                                            unsigned long long* level_count, void* scratch, cudaStream_t stream,
                                            uint16_t* mask = nullptr, int mask_pitch = 0);
size_t matryoshka_dense_operand_scratch_bytes();
const char* matryoshka_dense_tail_launch(const uint16_t* a_hi, const uint16_t* a_lo, const uint16_t* t_bf16,
                                        const int* level_start, int n_levels, int B, int H, int D, const float* bias,
                                        float* result, cudaStream_t stream);
const char* max_row_norm_launch(const float* w, int H, int D, float* out, cudaStream_t stream);
const char* row_threshold_launch(const float* x, int B, int D, const float* wmax, float thr_value, float* thr,
                                 cudaStream_t stream);

// analysis.cu: statistics over sparse active lists idx [B, cap] (entry < 0 = empty; with vals: active iff value > 0)
const char* activation_counts_launch(const int32_t* idx, const float* vals, int B, int cap, int H,
                                     unsigned long long* counts, cudaStream_t stream);
const char* coactivation_launch(const int32_t* idx, const float* vals, int B, int cap, int H, int32_t* cooc,
                                cudaStream_t stream);
const char* sq_error_launch(const float* a, const float* b, size_t n, double* out, cudaStream_t stream);
const char* compact_dense_launch(const float* dense, int B, int H, int mode, float thr, int cap, int32_t* idx, float* vals,
                                 int32_t* pairs, int32_t* cnt, cudaStream_t stream);

// train.cu: training-side kernels adjacent to the forward (SURVEY 8f-4)
const char* rows_scatter_add_launch(const float* coef, const int32_t* idx, const float* src, int B, int k, int D, int H,
                                    float scale, float* dst, float* dst_col, cudaStream_t stream);
const char* rows_gather_dot_launch(const float* g, const float* rows, const int32_t* idx, int B, int k, int D, int H,
                                   float scale, float* out, cudaStream_t stream);
const char* column_sum_launch(const float* src, int R, int C, float scale, float* out, cudaStream_t stream);
const char* bsae_logit_grad_launch(const float* logits, const float* G, int H, int D, int n_bits, const float* gp_dev,
                                   float gp_host, int accumulate, float* grad, cudaStream_t stream);
const char* matryoshka_scatter_launch(const int32_t* idx, int B, int cap, int H, int D, const float* const* g_levels,
                                      const int* level_start, int n_levels, float* M, int32_t* z2, cudaStream_t stream);
const char* matryoshka_grad_finish_launch(const float* W, const float* Wm, const float* M, const int32_t* z2,
                                          const float* alpha, const int* level_start, int n_levels, int H, int D, float c,
                                          int joint_bits, float* gW, float* gWm, cudaStream_t stream);
// z2[h] += number of rows b with mask[b, h] != 0 (bf16 mask [B, H], H % 8 == 0, 16-byte aligned rows; integer atomics)
const char* mask_column_count_launch(const uint16_t* mask, int B, int H, int32_t* z2, cudaStream_t stream);
size_t rigl_workspace_bytes(int sms);
const char* rigl_init_mask_launch(float* weight, float* mask, int D, int H, unsigned long long n_inactive, void* ws, int sms,
                                  cudaStream_t stream);
const char* rigl_update_mask_launch(float* weight, float* mask, const float* amean, const float* dmean, int D, int H,
                                    unsigned long long n_drop, unsigned long long n_grow, void* ws, int sms,
                                    cudaStream_t stream);
const char* mul_inplace_launch(float* a, const float* b, size_t n, cudaStream_t stream);
// baseline_sae backward (deterministic, latent-major): gradients of both Linear layers, b_dec and (gx != null) x
size_t baseline_backward_workspace_bytes(int B, int H, int D, int k);
const char* baseline_backward_launch(const float* x, const float* vals, const int32_t* idx, const float* g,
                                     const float* g_h, const float* g_vals, const float* w_enc, const float* dec_rows, int B,
                                     int H, int D, int k, float* gWe, float* gbe, float* gWd, float* gbd, float* gx, void* workspace,
                                     cudaStream_t stream);
// the same over one shard's latents [idx_begin, idx_begin + H_shard) (no g_h, no grad x); grad b_dec over all of g;
// workspace of baseline_backward_workspace_bytes(B, H_shard, D, k)
const char* baseline_backward_range_launch(const float* x, const float* vals, const int32_t* idx, const float* g,
                                           const float* g_vals, const float* rows_shard, int B, int H_shard, int idx_begin, int D,
                                           int k, float* gWe, float* gbe, float* gWd, float* gbd, void* workspace,
                                           cudaStream_t stream);
// b_sae backward (deterministic, latent-major, the logit chain rule fused in): gradients of the encoder Linear, the bit
// logits, b_dec and (gx != null) x; workspace of baseline_backward_workspace_bytes(B, H, D, k)
const char* bsae_backward_launch(const float* x, const float* vals, const int32_t* idx, const float* g, const float* soft_rows,
                                 const float* logits, float q, const float* gp_dev, float gp_host, const float* w_enc, int B,
                                 int H, int D, int k, int n_bits, float* gWe, float* gbe, float* glog, float* gbd, float* gx,
                                 void* workspace, cudaStream_t stream);

// peer.cu: flag-based exchange over CUDA IPC peer memory (dictionary-sharded forward)
const char* peer_signal_launch(unsigned* const* targets, int n, unsigned value, cudaStream_t stream);
const char* peer_wait_launch(const unsigned* flags, int n, unsigned value, int* timed_out, cudaStream_t stream);
const char* reduce_partials_peer_launch(const float* const* bases, int n, int row_begin, int rows, int D, float* out,
                                        cudaStream_t stream);

// encode_dense.cu
const char* encode_dense_launch(const float* x, const int32_t* rows, int R, const float* w,
                                const float* bias, int H, int D, int act, float* z,
                                cudaStream_t stream);

inline const char* cuda_err(cudaError_t e) { return e == cudaSuccess ? nullptr : cudaGetErrorString(e); }

}  // namespace qsae
