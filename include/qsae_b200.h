/*
 * qsae_b200.h -- C ABI of libqsae_b200.so: the B200 (sm_100a) forward hot path of
 * ASSERT-KTH/QuantizedSAE (b_sae / baseline_sae / q_sae / t_sae).
 *
 * The reference has no FFI of its own: its boundary is the Python nn.Module API
 * (src/quantized_sae/sae/*.py). Each entry point below replaces a group of eager ATen ops
 * inside one reference forward; the citation says which. quantizedsae_b200/sae/*.py mirrors
 * the nn.Module API on top of these calls (via ctypes, quantizedsae_b200/_lib.py) and
 * INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - plain C types only: device (or, where stated, host) pointers, sizes, a CUDA stream
 *     handle passed as void* (cudaStream_t / CUstream; NULL = legacy default stream);
 *   - every function returns 0 on success or a negative qsae_status; the message for the
 *     calling thread is available from qsae_last_error();
 *   - no hidden device allocation: scratch memory is caller-provided, its size comes from
 *     the matching *_workspace_bytes() query;
 *   - all launches are asynchronous on the given stream; nothing synchronises the device
 *     except the *_host() pipeline entry, which returns after its last copy has landed;
 *   - row-major everywhere; "bf16" buffers are raw uint16_t bit patterns.
 */
#ifndef QSAE_B200_H
#define QSAE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QSAE_ABI_VERSION 1

typedef enum qsae_status {
  QSAE_OK = 0,
  QSAE_ERR_INVALID_ARGUMENT = -1,   /* bad shape / null pointer / unsupported size          */
  QSAE_ERR_WORKSPACE_TOO_SMALL = -2,
  QSAE_ERR_CUDA = -3,               /* a CUDA runtime / driver call failed                   */
  QSAE_ERR_UNSUPPORTED_DEVICE = -4, /* not an sm_100 device                                  */
  QSAE_ERR_K_OUT_OF_RANGE = -5      /* k > H (torch.topk raises RuntimeError here)           */
} qsae_status;

/* encoder epilogue applied before selection (reference: none for b_sae/baseline,
 * ReLU for t_sae -- sae/binary.py:82-84, sae/baseline.py:8-10, sae/ternary.py:95-98) */
typedef enum qsae_act { QSAE_ACT_NONE = 0, QSAE_ACT_RELU = 1 } qsae_act;

int qsae_abi_version(void);
const char* qsae_last_error(void);
/* 0 if the current device is sm_100 (B200), QSAE_ERR_UNSUPPORTED_DEVICE otherwise */
int qsae_check_device(void);

/* ---------------------------------------------------------------------------------------
 * One-time weight preparation (cached by the host modules per parameter version)
 * ------------------------------------------------------------------------------------- */

/* float32 -> bf16 (round to nearest even). Used for encoder.0.weight [H,D] and for x.
 * Replaces nothing in the reference (which is fp32 throughout); it is the operand format of
 * the tcgen05 encoder. n = number of elements. */
int qsae_cast_f32_to_bf16(const float* src, uint16_t* dst, size_t n, void* stream);

/* binary_decoder.quantized_int_weights() (sae/binary.py:49-58) fused with packing:
 *   bit_i = sigmoid(logit) > 0.5 ; int_w = sum_i bit_i * c_i, c = [1,2,..,-2^(n-1)].
 * logits [H, D*n_bits] (bit i of feature d at column d*n_bits+i, LSB first, sign bit last).
 * n_bits <= 4: packed [H, D/2] bytes, feature 2j in the low nibble of byte j (two's complement)
 * n_bits  > 4: packed [H, D] int8.
 * stats (device, 2 doubles, optional, must be zeroed by the caller):
 *   stats[0] += sum p(1-p)2^i  (numerator of polarize_loss, sae/binary.py:41-42)
 *   stats[1]  = max |p - bit|  (how far the soft forward is from the hard dictionary)     */
int qsae_pack_bitplanes(const float* logits, int H, int D, int n_bits, uint8_t* packed,
                        double* stats, void* stream);

/* binary_decoder.quantized_int_weights_continuous() (sae/binary.py:60-69), i.e. the soft
 * effective weights of the reference forward (sae/binary.py:26-35): rows [H, D] float32. */
int qsae_dequant_soft(const float* logits, int H, int D, int n_bits, float* rows, void* stream);

/* [R, C] float32 -> [C, R] float32. baseline_sae keeps decoder.weight as [D, H]
 * (sae/baseline.py:12); the sparse decoder gathers feature rows, so it needs [H, D]. */
int qsae_transpose_f32(const float* src, int R, int C, float* dst, void* stream);

/* ---------------------------------------------------------------------------------------
 * Encoder + per-row top-k  (nn.Linear + Tensor.topk: sae/binary.py:92-94,
 * sae/baseline.py:23-36, sae/ternary.py:102-114)
 *
 * z = x W^T + b on the tcgen05 tensor cores (bf16 operands, fp32 accumulate in TMEM); the
 * per-row selection runs in the GEMM epilogue straight out of TMEM, so the dense [B,H]
 * pre-activation never reaches HBM. Output is ordered by (value desc, index asc).
 *
 * exact = 0: values are the tensor-core results. They equal the fp32 reference up to fp32
 *            accumulation order when x and W are bf16-representable (benchmark precondition).
 * With a sampled dictionary (qsae_prepare_encoder_sample) the call first scores only the
 * sampled rows and uses each row's m-th largest sample value as a prior threshold for the full
 * sweep (m chosen so that it is too high with probability < 1e-7 per row); the merge verifies
 * the threshold by counting survivors and a rescue kernel recomputes a failing row exactly, so
 * the result is the exact top-k either way -- the prior only removes survivor traffic.
 * exact = 1: the bf16 pass selects k+QSAE_RESCORE_MARGIN candidates per row, which are
 *            re-scored in fp32 from x_f32 / w_f32 and re-selected; flags[b] == 1 marks a row
 *            whose selection could not be certified against bf16 rounding (see DESIGN.md).
 * Limits: D % 8 == 0, 8 <= D <= 512, 1 <= k <= QSAE_MAX_K_LARGE, k <= H.
 * k <= QSAE_MAX_K runs on the warp-level selection kernels (the b_sae / baseline defaults: 65 and 32
 * at H = 32768). Larger k -- the reference default k = int(0.002 H) = 2097 at H = 2^20, or 262 per
 * shard of an 8-way dictionary split (sae/binary.py:94) -- takes the block-level path: ordered top-m
 * of the sampled rows (m <= QSAE_MAX_K) as the row threshold, a threshold-only sweep (no in-kernel cut),
 * a block-per-row radix select over the ~m H / n_sample survivors, and an exact dense recomputation of
 * any row whose survivor count check fails. Without a usable sample the call falls back to dense
 * pre-activations in row chunks + a dense radix select (small dictionaries only; not a throughput path).
 * ------------------------------------------------------------------------------------- */
#define QSAE_MAX_K 224
#define QSAE_MAX_K_LARGE 4096
#define QSAE_RESCORE_MARGIN 16

/* n_sample: rows of the sampled dictionary that will be passed to qsae_encode_topk (0 = none) */
int qsae_encode_topk_workspace_bytes(int B, int H, int D, int k, int n_sample, size_t* bytes);

/* Gather a stratified pseudo-random sample of n_sample dictionary rows (and their biases) for
 * the prior-threshold pre-pass of qsae_encode_topk. One-time, per weight version.
 * Recommended: n_sample = qsae_default_sample_rows(H) (H / 16 rounded up to a multiple of 256, for H >= 8192). */
int qsae_prepare_encoder_sample(const uint16_t* w_bf16, const float* b_enc, int H, int D, int n_sample,
                                uint16_t* w_sample /* [n_sample, D] */, float* b_sample /* [n_sample] */,
                                void* stream);

/* Rows of the stratified encoder sample the sampled-prior path works best with for a dictionary of H latents
 * (0: the dictionary is too small to sample; the class-bound path is used). H / QSAE_SAMPLE_DIV rounded up to whole
 * 256-row tiles. What qsae_bsae_plan_create and the Python modules pass to qsae_prepare_encoder_sample. */
int qsae_default_sample_rows(int H);

/* Kernels this library has launched in this process (all threads, monotonic): what bench.py reports as gpu_launches. */
unsigned long long qsae_launch_count(void);

/* Tuning / diagnostic switches (QSAE_ENCODE_CLUSTER, QSAE_ENCODE_RANGE, QSAE_PRIOR_PREP, QSAE_SAMPLE_DIV,
 * QSAE_DENSE_STEP_FUSED, QSAE_DECODE_PAIR, QSAE_DEBUG_*; INTEGRATION.md lists them all) are
 * read from the environment once, on first use, never on a
 * launch path. A process that changes them afterwards (tests, tuning runs) calls this to re-read them. */
int qsae_reload_tuning(void);

/* Large selections (k > QSAE_MAX_K through qsae_encode_topk, and qsae_merge_candidates[_peer]) spend most of their
 * instructions sorting the winners into (value desc, index asc) order. The reference only ever uses the winners as a set
 * (mask / scatter into the dense latent, sae/binary.py:96-99; the decoder sums them): with on != 0 the calling thread's
 * subsequent fast-mode (exact = 0) large selections emit the same k winners in no particular order. Exact mode and
 * the warp-level paths (k <= QSAE_MAX_K) always sort. Thread-local; off by default. */
int qsae_set_unordered_topk(int on);

/* Measurement hook: per-stage events of the sampled-prior path of qsae_encode_topk / qsae_bsae_forward, recorded in
 * stream order by the calling thread's next calls: [0] start, [1] prior ready (cast + sample pre-pass + prior),
 * [2] sweep done, [3] merge (+ fused decode) done, [4] tail kernel done, [5] separate decode done (when not fused).
 * events: n cudaEvent_t handles (n <= QSAE_N_STAGE_EVENTS; entries may be NULL); n = 0 switches it off. */
#define QSAE_N_STAGE_EVENTS 6
int qsae_set_stage_events(void* const* events, int n);

/* Prior thresholds of the sampled path on their own (the first launch of qsae_encode_topk for small batches; exposed
 * for tests and tuning): x -> bf16 (x_bf16 [B, D], out), contraction against the sampled rows on the tensor cores,
 * prior[b] = m-th largest per-class maximum of row b's sampled pre-activations, a lower bound of the row's m-th
 * largest sampled value. *ns_out = CTAs per 128-row block used (2 or 4); returns QSAE_ERR_INVALID_ARGUMENT when the
 * shape has no such launch (large batches and widths other than 256 / 512 use the separate kernels). */
int qsae_prior_prep(const float* x_f32, const uint16_t* w_sample, const float* b_sample, int n_sample, int B, int D,
                    int act, int m, uint16_t* x_bf16, float* prior, int* ns_out, void* stream);

/* Measurement hook: when both are non-NULL (cudaEvent_t), the calling thread's next
 * qsae_encode_topk calls record them on their stream immediately before / after the fused
 * encoder kernel, so a caller can time the dominant kernel alone. NULL, NULL switches it off. */
int qsae_set_encode_kernel_events(void* start_event, void* stop_event);

int qsae_encode_topk(const float* x_f32,      /* [B, D] device                              */
                     const uint16_t* w_bf16,   /* [H, D] from qsae_cast_f32_to_bf16          */
                     const float* w_f32,       /* [H, D] original weights; may be NULL if !exact */
                     const float* b_enc,       /* [H]                                        */
                     const uint16_t* w_sample, /* [n_sample, D] or NULL: sampled rows of w_bf16 */
                     const float* b_sample,    /* [n_sample] or NULL                          */
                     int n_sample,             /* 0 = no prior-threshold pre-pass             */
                     int B, int H, int D, int k, int act, int exact,
                     float* out_vals,          /* [B, k]                                     */
                     int32_t* out_idx,         /* [B, k]                                     */
                     int32_t* out_flags,       /* [B] or NULL                                */
                     void* workspace, size_t workspace_bytes, void* stream);

/* BinarySAE.forward on device buffers in one call (sae/binary.py:91-103): qsae_encode_topk followed by the sparse
 * decode of the packed dictionary (qsae_pack_bitplanes; n_bits <= 4: nibbles, else int8 rows),
 * recon = qstep * sum_j v_j dict[idx_j, :] + dec_bias. Same workspace as qsae_encode_topk.
 * (Measured and rejected: decoding a row inside the merge warp that has just sorted it. The merged kernel took
 * exactly the sum of the two, 325 us vs 154 + 171 us at B = 65536: the row phases of the resident warps do not
 * interleave enough to hide the merge's list latency behind the decode's integer work.) */
int qsae_bsae_forward(const float* x_f32, const uint16_t* w_bf16, const float* w_f32, const float* b_enc,
                      const uint16_t* w_sample, const float* b_sample, int n_sample, int B, int H, int D, int k,
                      int exact, const uint8_t* packed, int n_bits, float qstep, const float* dec_bias /* [D] or NULL */,
                      float* out_vals /* [B, k] */, int32_t* out_idx /* [B, k] */, int32_t* out_flags /* [B] or NULL */,
                      float* recon /* [B, D] */, void* workspace, size_t workspace_bytes, void* stream);

/* Exact fp32 CUDA-core encoder for a few rows: z[r, :] = x[rows[r], :] W^T + b (+act), dense
 * [R, H] output. Fallback for rows flagged by qsae_encode_topk(exact=1) and GPU-side
 * cross-check in the tests. Not a throughput path. */
int qsae_encode_dense_f32(const float* x_f32, const int32_t* rows /* [R] or NULL = 0..R-1 */,
                          int R, const float* w_f32, const float* b_enc, int H, int D, int act,
                          float* z /* [R, H] */, void* stream);

/* Diagnostic: the tensor-core encoder with its accumulator (+bias, +act) dumped densely to
 * z [B, H] instead of being consumed by the selection. Same kernel, same pipeline; used by the
 * tests to check the tcgen05 GEMM itself against an fp32 matmul. Workspace as for
 * qsae_encode_topk. Not a product path (it writes the matrix the product path avoids). */
int qsae_encode_dense_tc(const float* x_f32, const uint16_t* w_bf16, const float* b_enc, int B, int H,
                         int D, int act, float* z, void* workspace, size_t workspace_bytes,
                         void* stream);

/* Per-row top-k of a dense [R, H] matrix, same ordering rule. out_* are [R, k]. */
int qsae_topk_dense_workspace_bytes(int R, int H, int k, size_t* bytes);
int qsae_topk_dense(const float* z, int R, int H, int k, float* out_vals, int32_t* out_idx,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Sparse decoders: recon[b,:] = scale * sum_j vals[b,j] * dict[idx[b,j], :] + bias
 * (replace the dense latent.matmul(int_weights) of sae/binary.py:38 and the dense
 * nn.Linear decode of sae/baseline.py:29). idx < 0 entries are skipped.
 * ------------------------------------------------------------------------------------- */
int qsae_decode_int4(const float* vals, const int32_t* idx, int B, int k,
                     const uint8_t* packed /* [H, D/2] */, int H, int D, float scale,
                     const float* bias /* [D] or NULL */, float* recon /* [B, D] */, void* stream);
int qsae_decode_int8(const float* vals, const int32_t* idx, int B, int k,
                     const int8_t* rows /* [H, D] */, int H, int D, float scale,
                     const float* bias, float* recon, void* stream);
int qsae_decode_rows_f32(const float* vals, const int32_t* idx, int B, int k,
                         const float* rows /* [H, D] */, int H, int D, float scale,
                         const float* bias, float* recon, void* stream);

/* ---------------------------------------------------------------------------------------
 * q_sae: QuantizedMatryoshkaDecoder (sae/quantized_matryoshka.py:47-143)
 * ------------------------------------------------------------------------------------- */
/* weight / weight_mirror [H, D] fp32 -> T = sign(sigmoid(w) >= 0.5) + sign(sigmoid(w_m) >= 0.5) in
 * {-2, 0, +2}, packed 2 bits per entry ([H, D/16] uint32: bit0 non-zero, bit1 negative), and
 * scale[h] = level_factor[level(h)] / (||T[h,:]||_2 + 1e-8)   (:67-91).
 * level_start: device int[n_levels + 1] (first latent of each level, then H);
 * level_factor: device float[n_levels] = 2^(n_bits - i - 2) * quant_step. D % 16 == 0. */
int qsae_pack_matryoshka(const float* weight, const float* weight_mirror, int H, int D,
                         const int* level_start, const float* level_factor, int n_levels,
                         uint32_t* packed, float* scale, void* stream);

int qsae_matryoshka_workspace_bytes(int B, int H, int D, size_t* bytes);

/* QuantizedMatryoshkaSAE.forward (:217-220): encoder (Linear + Sigmoid, active <=> sigmoid(z) > 0.5)
 * fused with the collection of each row's active latents, then the sparse level decoder:
 * result[i, b, :] = bias + sum_{h active, level(h) <= i} scale[h] * T[h, :]     (cumulative, :121-129)
 * level_count[i]  = number of active latents of level i over the batch (latent_group[i] * B).
 * *overflow is set to 1 when a row had more active latents than the sparse path holds
 * (1024 per sub-stream); active latents were then dropped and the caller must use a dense path. So that the flag
 * may be read lazily (no host synchronisation per forward), every output of such a call -- result, and the residual
 * of qsae_matryoshka_forward_active -- is NaN: a wrong reconstruction can never be used unnoticed. */
int qsae_matryoshka_forward(const float* x_f32, const uint16_t* w_bf16,
                            const float* w_f32 /* [H,D] or NULL: exact fp32 activity decisions */,
                            const float* w_norm_max /* device scalar from qsae_max_row_norm; exact only */,
                            const float* b_enc, const uint32_t* packed, const float* scale,
                            const int* level_start, int n_levels, const float* dec_bias /* [D] or NULL */,
                            int B, int H, int D, float* result /* [n_levels, B, D] */,
                            unsigned long long* level_count /* [n_levels] */, int* overflow,
                            void* workspace, size_t workspace_bytes, void* stream);

/* The same forward, additionally exporting each row's active latents for the analysis consumers
 * (_activation_mask of scripts/analysis/dynamic_analysis.py:30-73 without the dense [B, H] mask):
 * active_idx [B, active_cap] int32, unordered, empty slots = -1; active_cnt [B] = number of active latents of the
 * row (entries beyond active_cap are counted but not stored). NULL active_idx = plain forward.
 * residual_out [B, D] or NULL: (x - result[n_levels - 1]) * 2, the input of the next rq_sae stage
 * (sae/residual_quantized.py:67), written by the level decoder from the reconstruction it still holds in
 * registers instead of a separate pass (qsae_residual_update). Must not alias x_f32. */
int qsae_matryoshka_forward_active(const float* x_f32, const uint16_t* w_bf16, const float* w_f32,
                                   const float* w_norm_max, const float* b_enc, const uint32_t* packed,
                                   const float* scale, const int* level_start, int n_levels, const float* dec_bias,
                                   int B, int H, int D, float* result, unsigned long long* level_count, int* overflow,
                                   int32_t* active_idx, int active_cap, int32_t* active_cnt, float* residual_out,
                                   void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Analysis consumers over sparse active lists (scripts/analysis/dynamic_analysis.py:317-440).
 * idx [B, cap] int32: latent indices of a row, entries < 0 or >= H are empty; vals [B, cap] or NULL: when
 * given, an entry is active iff its value is > 0 (b_sae / baseline: `latent > 0`, :44-50).
 * qsae_activation_counts: counts[h] += rows in which h is active                (:341, mask.sum(0))
 * qsae_coactivation:      cooc[i * H + j] += rows in which i and j are both active, i == j included
 *                         (:344-345, mask^T mask as int32); cap <= 2048
 * qsae_sq_error_accumulate: *out += sum (a - b)^2 in float64                     (:96-100)
 * All three accumulate into caller-zeroed device buffers, so a data loader's batches add up.
 * ------------------------------------------------------------------------------------- */
int qsae_activation_counts(const int32_t* idx, const float* vals, int B, int cap, int H,
                           unsigned long long* counts /* [H] */, void* stream);
int qsae_coactivation(const int32_t* idx, const float* vals, int B, int cap, int H, int32_t* cooc /* [H, H] */,
                      void* stream);
int qsae_sq_error_accumulate(const float* a, const float* b, size_t n, double* out /* device scalar */, void* stream);
/* The same statistics from a dense activity mask, for rows whose active sets are too long for the lists (a q_sae at
 * high activity; qsae_matryoshka_forward_dense_active writes the mask): cooc[i * H + j] += sum_k M[k, i] M[k, j] for
 * mask [K, H] bf16 0.0 / 1.0, row-major, and counts[h] += sum_k M[k, h] (counts may be NULL). A tcgen05 product over
 * the tiles of the upper triangle; each element is added to cooc[m, n] and cooc[n, m] by one thread, so there are no
 * atomics, the result is bit-deterministic and cooc is complete and symmetric after every call (list and mask batches
 * may add into the same matrix in any order). H % 8 == 0, K <= 2^24 (fp32 accumulation of 0/1 products is exact there);
 * mask and cooc 16-byte aligned. */
int qsae_coactivation_dense(const uint16_t* mask /* [K, H] */, int K, int H, int32_t* cooc /* [H, H] */,
                            long long* counts /* [H] or NULL */, void* stream);

/* Dense [B, H] latents (what the reference hands to its decoders: sae/binary.py:24, sae/quantized_matryoshka.py:47)
 * -> sparse per-row lists, ascending latent order. mode 0: entries != 0; mode 1: entries > thr (q_sae activity, :99).
 * Any of idx [B, cap] (-1 padded), vals [B, cap] (0 padded), pairs [B, cap, 2] (the list format of
 * qsae_decode_matryoshka_lists) may be NULL; cnt [B] counts every hit, stored or not (cap = 0: count only). */
int qsae_compact_dense(const float* dense, int B, int H, int mode, float thr, int cap, int32_t* idx, float* vals,
                       int32_t* pairs, int32_t* cnt, void* stream);

/* Dense path of the same forward, for any activity level (the sparse path reports *overflow when a row
 * has more active latents than its survivor lists hold -- e.g. an untrained model, ~50 % active):
 * dense pre-activations, A = (sigmoid(z) > 0.5) * scale as bf16 hi + lo, and one tcgen05 GEMM per level
 * over that level's range of the latent axis with T^T [D, H] in bf16, outputs accumulated level by level.
 * w_mid / w_lo given (qsae_split_bf16x3 of the encoder weight): fp32-accurate pre-activations through the
 * split passes described at qsae_tsae_forward; else one bf16 pass. level_start is needed on the device (counts) and on the host (GEMM ranges);
 * boundaries and H must be multiples of 8. */
int qsae_unpack_matryoshka_t(const uint32_t* packed /* [H, D/16] */, int H, int D, uint16_t* t_bf16 /* [D, H] */,
                             void* stream);
int qsae_matryoshka_dense_workspace_bytes(int B, int H, int D, size_t* bytes);
int qsae_matryoshka_forward_dense(const float* x_f32, const uint16_t* w_hi, const uint16_t* w_mid, const uint16_t* w_lo,
                                  const float* b_enc,
                                  const uint16_t* t_bf16, const float* scale, const int* level_start_dev,
                                  const int* level_start_host, int n_levels, const float* dec_bias, int B, int H,
                                  int D, float* result /* [n_levels, B, D] */,
                                  unsigned long long* level_count /* [n_levels] */, void* workspace,
                                  size_t workspace_bytes, void* stream);
/* The same forward, also writing its activity mask: active_mask[b * mask_pitch + mask_col + h] = 1.0 (bf16) where
 * latent h of row b is active (sigmoid(z) > 0.5, the decision that forms A; a latent with a zero decoder scale is still
 * active), else 0.0. mask_pitch and mask_col are multiples of 8 with mask_col + H <= mask_pitch, so the stages of an
 * rq_sae can write side by side into one [B, sum of stage widths] mask. Input for qsae_coactivation_dense. */
int qsae_matryoshka_forward_dense_active(const float* x_f32, const uint16_t* w_hi, const uint16_t* w_mid,
                                         const uint16_t* w_lo, const float* b_enc, const uint16_t* t_bf16,
                                         const float* scale, const int* level_start_dev, const int* level_start_host,
                                         int n_levels, const float* dec_bias, int B, int H, int D,
                                         float* result /* [n_levels, B, D] */,
                                         unsigned long long* level_count /* [n_levels] */,
                                         uint16_t* active_mask /* [B, mask_pitch] */, int mask_pitch, int mask_col,
                                         void* workspace, size_t workspace_bytes, void* stream);

/* rq_sae (ResidualQuantizedSAE.forward, sae/residual_quantized.py:53-69): a cascade of one-bit q_saes, each
 * run with qsae_matryoshka_forward (n_levels = 1) on the residual of the previous stage;
 * this is the step between stages (:67): out = (residual - recon) * 2. out may alias residual. */
int qsae_residual_update(const float* residual, const float* recon, size_t n, float* out, void* stream);

/* max_h ||w[h,:]||_2 -> *out (device float). With w_f32 given, qsae_matryoshka_forward lowers each
 * row's sweep threshold by the bound 2^-8 ||x_b|| max_h||w_h|| on |z_bf16 - z_fp32| and decides
 * activity from an fp32 re-scoring, so the active set equals the fp32 reference's for any input. */
int qsae_max_row_norm(const float* w_f32, int H, int D, float* out, void* stream);

/* The level decoder alone, for callers that already hold the active latents:
 * lists [B, cap, 2] int32 (second component = latent index), counts [B]. */
int qsae_decode_matryoshka_lists_workspace_bytes(size_t* bytes);
int qsae_decode_matryoshka_lists(const int32_t* lists, const int32_t* counts, int cap, int B,
                                 const uint32_t* packed, const float* scale, const int* level_start,
                                 int n_levels, int H, int D, const float* dec_bias, float* result,
                                 unsigned long long* level_count, void* workspace, size_t workspace_bytes,
                                 void* stream);

/* ---------------------------------------------------------------------------------------
 * t_sae: TernarySparseAutoencoder / STEWeights (sae/ternary.py:41-52, :116-122)
 *   h = relu(x W^T + b)  -- DENSE [B, H], returned to the caller (no top-k in the reference forward)
 *   recon = h T^T,  T = sign(Wd) * (|Wd| >= 0.5),  Wd = decoder.weight [D, H], no decoder bias
 * Two chained tensor-core GEMMs; the second takes h as bf16 hi (+ lo) and the exact ternary T.
 * ------------------------------------------------------------------------------------- */
/* STEWeights hard weights (sae/ternary.py:46-49). t_bf16 [D, H] (B operand of qsae_decode_dense /
 * qsae_tsae_forward) and/or t_rows [H, D] int8 (gather layout for qsae_decode_int8); either may be NULL. */
int qsae_pack_ternary(const float* w /* [D, H] */, int D, int H, float threshold, uint16_t* t_bf16,
                      int8_t* t_rows, void* stream);

/* hi = bf16(src), lo = bf16(src - hi) (lo may be NULL): hi + lo carries 16 mantissa bits of src. */
int qsae_split_bf16(const float* src, uint16_t* hi, uint16_t* lo, size_t n, void* stream);
/* hi + mid + lo == src exactly (8 + 8 + 8 mantissa bits). The exact modes of the dense encoder take the
 * encoder weight in this form (one-time, cached per weight version); mid / lo may be NULL. */
int qsae_split_bf16x3(const float* src, uint16_t* hi, uint16_t* mid, uint16_t* lo, size_t n, void* stream);

/* out[B, N] = (a_hi (+ a_lo))[B, K] * b_t[N, K]^T (+ bias): the dense F.linear(h, hard_weights) of
 * sae/ternary.py:52 on the tcgen05 tensor cores (bf16 operands, fp32 accumulation in TMEM, split-K
 * with a fixed-order reduction: deterministic). K % 8 == 0, N % 4 == 0, N <= 512. */
int qsae_decode_dense_workspace_bytes(int B, int K, int N, size_t* bytes);
int qsae_decode_dense(const uint16_t* a_hi /* [B, K] */, const uint16_t* a_lo /* [B, K] or NULL */,
                      const uint16_t* b_t /* [N, K] */, int B, int K, int N, const float* bias /* [N] or NULL */,
                      float* out /* [B, N] */, void* workspace, size_t workspace_bytes, void* stream);

/* TernarySparseAutoencoder.forward (sae/ternary.py:116-122).
 * exact = 0: h from the tcgen05 encoder (bf16 operands: equals the fp32 reference up to accumulation
 *            order when x and W are bf16-representable), written as fp32 (h_out) and bf16 by TMA stores
 *            from the GEMM epilogue; recon from one pass over bf16(h) (relative error <= 2^-9 per term).
 * exact = 1: any fp32 operands. x and W are split exactly into three bf16 parts each and the six partial
 *            products above 2^-24 are accumulated on the tensor cores in ONE launch (both operands streamed,
 *            all six products into the same TMEM accumulator, smallest first); recon from two accumulating
 *            passes over the hi/lo split of h (2^-17 per term).
 * H % 8 == 0, D % 8 == 0, 8 <= D <= 512. */
int qsae_tsae_workspace_bytes(int B, int H, int D, int exact, size_t* bytes);
int qsae_tsae_forward(const float* x_f32, const uint16_t* w_hi /* [H, D]: bf16(W) */,
                      const uint16_t* w_mid, const uint16_t* w_lo /* [H, D] from qsae_split_bf16x3; exact = 1 */,
                      const float* b_enc,
                      const uint16_t* t_bf16 /* [D, H] from qsae_pack_ternary */, int B, int H, int D, int exact,
                      float* h_out /* [B, H] */, float* recon /* [B, D] */, void* workspace,
                      size_t workspace_bytes, void* stream);

/* t_t_bf16 [H, D] = T^T as bf16 (exact: the entries are ternary), the B operand of the backward's g T. */
int qsae_pack_ternary_t(const float* w /* [D, H] */, int D, int H, float threshold, uint16_t* t_t_bf16, void* stream);

/* Weight-gradient GEMM on the tensor cores: c[M, N] = sum_k A(k, m) B(k, n), a contraction over K batch rows.
 * b_parts: host array of n_parts device pointers, row-major bf16 [K, N]. a_parts: row-major bf16 [K, M]
 * (a_kmajor = 0), or [M, K] (a_kmajor = 1, then K % 8 == 0). Both MN-major operands are read as they are, no
 * transposes. n_parts = 1: one bf16 product; n_parts = 3: the operands are three-part splits
 * (qsae_split_bf16x3) and the six products above 2^-24 go into one fp32 accumulator (fp32-accurate products).
 * N % 8 == 0 and M % 8 == 0 (a_kmajor = 0) or K % 8 == 0 (a_kmajor = 1); any K >= 1 (TMA zero-fills the tail).
 * c [M, N] fp32 is overwritten. */
int qsae_wgrad(const uint16_t* const* a_parts, const uint16_t* const* b_parts, int n_parts, int M, int N, int K,
               int a_kmajor, float* c, void* stream);

/* Backward of TernarySparseAutoencoder.forward (what torch autograd computes on the reference, training.py):
 *   gz = (g T + g_h) * 1[h > 0]            g = d loss / d recon [B, D], g_h = d loss / d h [B, H] or NULL
 *   grad_w_enc = gz^T x [H, D]    grad_b_enc = sum_b gz [H]    grad_w_dec = mask * (g^T h) [D, H] (mask NULL: 1)
 *   grad_x = gz W_enc [B, D] (NULL: not computed; w_hi / w_mid / w_lo are then unused)
 * gz comes from the dense encoder kernel with a ReLU-backward epilogue (g T never reaches memory), which also sums it
 * per column into grad_b_enc; the three weight products are qsae_wgrad GEMMs. exact = 1: g, gz, h, x (and W_enc: w_mid / w_lo from qsae_split_bf16x3) as three
 * bf16 parts, fp32-accurate products; exact = 0: one bf16 product each. grad_b_enc is a column sum with atomics
 * (not bit-deterministic); everything else is. Outputs are overwritten. h, x, g, g_h, gradients 16-byte aligned.
 * Same shape limits as qsae_tsae_forward; B may be 0 (zero gradients). */
int qsae_tsae_backward_workspace_bytes(int B, int H, int D, int exact, size_t* bytes);
int qsae_tsae_backward(const float* x /* [B, D] */, const float* h /* [B, H] forward output */,
                       const float* g_recon /* [B, D] */, const float* g_h /* [B, H] or NULL */,
                       const uint16_t* t_t_bf16 /* [H, D] from qsae_pack_ternary_t */, const float* mask /* [D, H] or NULL */,
                       const uint16_t* w_hi, const uint16_t* w_mid, const uint16_t* w_lo /* [H, D], grad_x only */,
                       int B, int H, int D, int exact, float* grad_w_enc /* [H, D] */, float* grad_b_enc /* [H] */,
                       float* grad_w_dec /* [D, H] */, float* grad_x /* [B, D] or NULL */, void* workspace,
                       size_t workspace_bytes, void* stream);

/* Backward of BaselineSparseAutoencoder.forward (Linear -> top-k -> scatter -> Linear; what torch autograd computes on
 * the reference). With g = d loss / d recon [B, D], the forward's top-k (vals, idx) [B, k] and
 *   gv[b,j] = <g[b,:], W_dec[:, idx[b,j]]> + g_h[b, idx[b,j]]    (g_h: dense [B, H], or g_vals [B, k]; at most one)
 *   grad_w_enc[h,:] = sum gv x[b,:] [H, D]   grad_b_enc[h] = sum gv [H]   grad_w_dec[:,h] = sum v g[b,:] [D, H]
 * over the rows b that selected h; grad_b_dec = sum_b g [D]; grad_x = gv W_enc [B, D] over the kept entries (NULL: not
 * computed, w_enc unused). dec_rows [H, D] = W_dec^T (qsae_transpose_f32). The entries are grouped by latent with a
 * stable sort, so each output element has one writer and a fixed summation order: every output is bit-deterministic.
 * Latents no row selected get exact zeros. Outputs are overwritten. Caller workspace, one stream, no host
 * synchronisation (CUDA-graph capturable). Same shape rules as qsae_encode_topk (D a multiple of 8 in [8, 512],
 * 1 <= k <= H), B k < 2^31; B may be 0 (zero gradients). x, g_recon, w_enc, dec_rows, grad_w_enc, grad_x and the
 * workspace 16-byte aligned. */
int qsae_baseline_backward_workspace_bytes(int B, int H, int D, int k, size_t* bytes);
int qsae_baseline_backward(const float* x /* [B, D] */, const float* vals, const int32_t* idx /* [B, k] */,
                           const float* g_recon /* [B, D] */, const float* g_h /* [B, H] or NULL */,
                           const float* g_vals /* [B, k] or NULL */, const float* w_enc /* [H, D], grad_x only */,
                           const float* dec_rows /* [H, D] */, int B, int H, int D, int k, float* grad_w_enc /* [H, D] */,
                           float* grad_b_enc /* [H] */, float* grad_w_dec /* [D, H] */, float* grad_b_dec /* [D] */,
                           float* grad_x /* [B, D] or NULL */, void* workspace, size_t workspace_bytes, void* stream);

/* One shard's part of qsae_baseline_backward in the dictionary-sharded baseline_sae: the shard owns the latents
 * [idx_begin, idx_begin + H_shard) and holds their decoder rows rows_shard [H_shard, D] (its decoder.weight^T); idx
 * holds global indices, and an entry outside the range is skipped. The owned entries are compacted in row-major order
 * before they are grouped by latent, so every latent's sums run over the same entries in the same order as in
 * qsae_baseline_backward: grad_w_enc [H_shard, D], grad_b_enc [H_shard] and grad_w_dec [D, H_shard] (row stride
 * H_shard) are bit-equal to the matching slices of its outputs for the same (vals, idx, g_recon, g_vals), and
 * grad_b_dec [D] (over all of g_recon) to its grad_b_dec. No g_h, no grad_x. k counts winners over the whole
 * dictionary and may exceed H_shard (1 <= k <= QSAE_MAX_K_LARGE); B k < 2^31; idx_begin >= 0; H_shard >= 1 and D as
 * in qsae_encode_topk; B may be 0 (zero gradients). x, g_recon, rows_shard, grad_w_enc and the workspace 16-byte
 * aligned. Caller workspace, one stream, no host synchronisation. */
int qsae_baseline_backward_range_workspace_bytes(int B, int H_shard, int D, int k, size_t* bytes);
int qsae_baseline_backward_range(const float* x /* [B, D] */, const float* vals, const int32_t* idx /* [B, k] */,
                                 const float* g_recon /* [B, D] */, const float* g_vals /* [B, k] or NULL */,
                                 const float* rows_shard /* [H_shard, D] */, int B, int H_shard, int idx_begin, int D, int k,
                                 float* grad_w_enc /* [H_shard, D] */, float* grad_b_enc /* [H_shard] */,
                                 float* grad_w_dec /* [D, H_shard] */, float* grad_b_dec /* [D] */, void* workspace,
                                 size_t workspace_bytes, void* stream);

/* Bit-deterministic backward of BinarySAE.forward under its soft (sigmoid) dictionary (sae/binary.py:24-47, 91-103).
 * With g = d loss / d recon [B, D], the forward's top-k (vals, idx) [B, k], q the quantization step and
 *   gv[b,j] = q <g[b,:], soft_rows[idx[b,j], :]>,   G[h,:] = q sum v g[b,:]   (d loss / d int_w)
 *   grad_w_enc[h,:] = sum gv x[b,:] [H, D]   grad_b_enc[h] = sum gv [H]   over the rows b that selected h;
 *   grad_logits[h, d n + i] = (G[h,d] c_i + gp 2^i (1 - 2p) / (H D n)) p (1 - p)   [H, D n]   (qsae_bsae_logit_grad's
 *   formula and bits for the same G; gp_dev / gp_host as there);   grad_b_dec = sum_b g [D];
 *   grad_x = gv W_enc [B, D] over the kept entries (NULL: not computed, w_enc unused).
 * soft_rows [H, D] is the soft dictionary (qsae_dequant_soft of logits). The entries are grouped by latent with a stable
 * sort; each output element has one writer and a fixed summation order, so every output is bit-deterministic. G never
 * reaches memory. Latents no row selected get exact zeros in grad_w_enc / grad_b_enc and the polarize-only logit
 * gradient. Outputs are overwritten. Caller workspace, one stream, no host synchronisation (CUDA-graph capturable).
 * Shape rules of qsae_encode_topk (D a multiple of 8 in [8, 512], 1 <= k <= min(H, QSAE_MAX_K_LARGE)), 1 <= n_bits <= 8,
 * B k < 2^31; B may be 0. x, g_recon, soft_rows, logits, w_enc, grad_w_enc, grad_logits, grad_x and the workspace
 * 16-byte aligned. */
int qsae_bsae_backward_workspace_bytes(int B, int H, int D, int k, int n_bits, size_t* bytes);
int qsae_bsae_backward(const float* x /* [B, D] */, const float* vals, const int32_t* idx /* [B, k] */,
                       const float* g_recon /* [B, D] */, const float* soft_rows /* [H, D] */,
                       const float* logits /* [H, D*n_bits] */, float q, const float* gp_dev, float gp_host,
                       const float* w_enc /* [H, D], grad_x only */, int B, int H, int D, int k, int n_bits,
                       float* grad_w_enc /* [H, D] */, float* grad_b_enc /* [H] */, float* grad_logits /* [H, D*n_bits] */,
                       float* grad_b_dec /* [D] */, float* grad_x /* [B, D] or NULL */, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Dictionary-sharded b_sae (2^20-latent dictionaries over G GPUs; SURVEY.md 8e). Shard g owns the
 * latents [g * shard_latents, (g + 1) * shard_latents) of nn.Linear / binary_decoder
 * (sae/binary.py:82-84, :24-38); x is replicated. Per forward:
 *   qsae_encode_topk on the shard          -> local top-k (values, shard-local indices)
 *   qsae_pack_candidates + all-gather      -> [G][B][k] {value, local index} entries on every rank
 *   qsae_merge_candidates                  -> global top-k (value desc, global index asc), identical on
 *                                             every rank: Tensor.topk over the full dictionary (:94)
 *   qsae_decode_int4_range                 -> partial reconstruction from the winners this shard owns
 *   reduce-scatter(sum) of the partials    -> rows of latent.matmul(int_weights) (:38)
 * The two collectives are issued by the host side (NCCL via torch.distributed); these entry points
 * are the compute steps between them.
 * ------------------------------------------------------------------------------------- */
/* (vals, idx)[n] -> n interleaved {float32 bits, int32 index} 8-byte entries (one all-gather operand) */
int qsae_pack_candidates(const float* vals, const int32_t* idx, size_t n, void* out, void* stream);

int qsae_merge_candidates_workspace_bytes(int B, size_t* bytes);
/* cand_all: [n_shards][B][k_in] entries, shard-local indices; entry (s, b, j) stands for the global
 * latent s * shard_latents + index. out_*: [B, k_out], k_out <= n_shards * k_in, k_out <= QSAE_MAX_K_LARGE.
 * incomplete (device int32, or NULL): for TRUNCATED lists -- every shard sent only its k_in < k_out best
 * candidates (a shard owns ~k_out / n_shards of the winners, so k_out / n_shards + 6 sigma is almost always
 * enough and cuts the all-gather and the merge input by ~n_shards / 1.5). *incomplete is set to 1 when, for
 * some row, ALL k_in entries of some shard were selected: that shard may hold further winners it did not send,
 * and the caller must repeat the exchange with the shards' full candidate lists. 0 = the result is the exact
 * global top-k. Every rank merges the same gathered tensor, so all ranks see the same flag. */
int qsae_merge_candidates(const void* cand_all, int n_shards, int B, int k_in, int shard_latents, int k_out,
                          float* out_vals, int32_t* out_idx, int32_t* incomplete, void* workspace,
                          size_t workspace_bytes, void* stream);

/* qsae_decode_int4 / qsae_decode_int8 restricted to the latents [idx_begin, idx_begin + shard_latents)
 * held in `packed_shard` / `rows_shard` (global indices in idx; others are skipped). */
/* ---- the same exchange over peer memory instead of NCCL (one process per GPU, NVLink / NVSwitch) ----------------
 * Every rank owns one buffer (qsae_peer_alloc: cudaMalloc, zeroed) that its peers map through CUDA IPC
 * (qsae_peer_export -> 64-byte handle, sent to the peers by the host side; qsae_peer_import / qsae_peer_close).
 * A rank writes its candidate lists / partial reconstructions into ITS OWN buffer and then raises a sequence flag
 * in every consumer's buffer (qsae_peer_signal: targets[g] = address of this rank's flag inside rank g's buffer);
 * a consumer polls its own flags (qsae_peer_wait: flags[g] >= value for all g; bounded, ~2 s, then *timed_out = 1)
 * and reads the data straight from peer memory inside the consuming kernel:
 *   qsae_merge_candidates_peer: as qsae_merge_candidates, list s of row r at list_bases[s] + r * k_in entries
 *   qsae_reduce_partials_peer:  out[r, :] = sum_g partial_g[row_begin + r, :] (fixed order, deterministic)
 * list_bases / partial_bases / targets are DEVICE arrays of n_shards pointers. */
int qsae_peer_alloc(size_t bytes, void** ptr);
int qsae_peer_free(void* ptr);
int qsae_peer_export(const void* ptr, unsigned char* handle64);
int qsae_peer_import(const unsigned char* handle64, void** ptr);
int qsae_peer_close(void* ptr);
int qsae_peer_signal(void* const* targets, int n, unsigned value, void* stream);
int qsae_peer_wait(const unsigned* flags, int n, unsigned value, int32_t* timed_out, void* stream);
int qsae_merge_candidates_peer(const void* const* list_bases, int n_shards, int B, int k_in, int shard_latents, int k_out,
                               float* out_vals, int32_t* out_idx, int32_t* incomplete, void* workspace,
                               size_t workspace_bytes, void* stream);
int qsae_reduce_partials_peer(const float* const* partial_bases, int n_shards, int row_begin, int rows, int D, float* out,
                              void* stream);

int qsae_decode_int4_range(const float* vals, const int32_t* idx, int B, int k, const uint8_t* packed_shard,
                           int shard_latents, int idx_begin, int D, float scale, const float* bias,
                           float* recon, void* stream);
int qsae_decode_int8_range(const float* vals, const int32_t* idx, int B, int k, const int8_t* rows_shard,
                           int shard_latents, int idx_begin, int D, float scale, const float* bias,
                           float* recon, void* stream);
/* qsae_decode_rows_f32 restricted to the latents [idx_begin, idx_begin + shard_latents) whose fp32 rows
 * [shard_latents, D] are in `rows_shard` (the dictionary-sharded baseline_sae's transposed decoder columns).
 * rows_shard, bias and recon must be 16-byte aligned (recon may be a slot of a peer-exchange buffer). */
int qsae_decode_rows_f32_range(const float* vals, const int32_t* idx, int B, int k, const float* rows_shard,
                               int shard_latents, int idx_begin, int D, float scale, const float* bias,
                               float* recon, void* stream);

/* latent * mask (sae/binary.py:96-99) / zeros_like + scatter_ (sae/baseline.py:38-39):
 * dense [B, H] float32 from the sparse form. Zero-fills `dense` first. */
int qsae_densify(const float* vals, const int32_t* idx, int B, int k, int H, float* dense,
                 void* stream);

/* ---------------------------------------------------------------------------------------
 * End-to-end b_sae forward on HOST buffers (the reference-facing call of bench.py's e2e leg):
 * chunks the batch, overlaps H2D copy / kernels / D2H copy on internal streams, returns when
 * the outputs are in host memory. Weights stay device-resident in a prepared handle.
 * ------------------------------------------------------------------------------------- */
typedef struct qsae_bsae_plan qsae_bsae_plan;

int qsae_bsae_plan_create(const float* w_enc_f32_dev /* [H,D] */, const float* b_enc_dev /* [H] */,
                          const float* dec_logits_dev /* [H, D*n_bits] */,
                          const float* dec_bias_dev /* [D] */, int H, int D, int n_bits,
                          float gamma, int k, int max_chunk_rows, qsae_bsae_plan** plan);
void qsae_bsae_plan_destroy(qsae_bsae_plan* plan);
/* x_host [B,D] float32 (pinned for full overlap); outputs: vals/idx [B,k], recon [B,D] on host */
int qsae_bsae_forward_host(qsae_bsae_plan* plan, const float* x_host, int B, float* vals_host,
                           int32_t* idx_host, float* recon_host);

/* The same forward as a stream of batches: submit enqueues the H2D copies, kernels and D2H copies of one batch and
 * returns at once with a ticket; wait blocks until that batch's outputs are in host memory. Several batches may be
 * in flight (up to QSAE_MAX_PENDING tickets; submit fails with QSAE_ERR_INVALID_ARGUMENT when all are taken), so the
 * copy-in of batch i + 1 overlaps the kernels of batch i and the copy-out of batch i - 1. Host buffers must stay
 * valid (and should be pinned) until the ticket has been waited for. Tickets complete in submission order. */
#define QSAE_MAX_PENDING 8
int qsae_bsae_submit_host(qsae_bsae_plan* plan, const void* x_host, int B, float* vals_host, int32_t* idx_host,
                          void* recon_host, int* ticket);
int qsae_bsae_wait_host(qsae_bsae_plan* plan, int ticket);

/* Host-side formats of the plan's calls (both entry points), to cut PCIe bytes when the caller can accept it:
 * x_is_bf16 != 0: x_host holds bfloat16 (2 bytes per element; exact for bf16-representable activations);
 * recon_mode 0: float32 reconstruction (default), 1: bfloat16 (rounded to nearest), 2: none (recon_host ignored).
 * Values / indices are always float32 / int32. */
int qsae_bsae_plan_set_io(qsae_bsae_plan* plan, int x_is_bf16, int recon_mode);

/* ---------------------------------------------------------------------------------------
 * Training-side pieces adjacent to the forward (SURVEY 8f-4). The reference gets them from eager autograd over
 * dense [B, H] latents; these work on the sparse forward quantities. Gradient outputs ACCUMULATE (+=) unless stated,
 * like torch's .grad. Sums that join by atomics agree with a serial sum to fp32 rounding (order not fixed).
 * ------------------------------------------------------------------------------------- */

/* dst[idx[b,j], :] += scale * coef[b,j] * src[b, :]; dst_col[idx[b,j]] += scale * coef[b,j] (dst_col may be NULL).
 * coef NULL = 1. idx [B,k] int32, entries < 0 or >= H are skipped. The sparse outer product of
 *   d loss / d int_w   = q * sparse_latent^T @ grad_recon      (backward of sae/binary.py:38)
 *   d loss / d W_enc   = grad_z^T @ x, d loss / d b_enc        (backward of the encoder Linear under the top-k mask, :92-99) */
int qsae_rows_scatter_add(const float* coef, const int32_t* idx, const float* src /* [B,D] */, int B, int k, int D, int H,
                          float scale, float* dst /* [H,D] */, float* dst_col /* [H] or NULL */, void* stream);
/* out[b,j] = scale * <g[b,:], rows[idx[b,j], :]> (written, not accumulated; 0 for skipped entries):
 *   d loss / d latent at the k kept positions = q * grad_recon @ int_w^T restricted to the mask (sae/binary.py:38,99) */
int qsae_rows_gather_dot(const float* g /* [B,D] */, const float* rows /* [H,D] */, const int32_t* idx, int B, int k, int D,
                         int H, float scale, float* out /* [B,k] */, void* stream);
/* out[c] += scale * sum_r src[r,c]: bias gradients; with scale = 1/R the batch means of STEWeights.update_mask
 * (sae/ternary.py:74-75) */
int qsae_column_sum(const float* src, int R, int C, float scale, float* out /* [C] */, void* stream);
/* Chain rule through the sigmoid bits + gradient of polarize_loss (sae/binary.py:26-43):
 *   grad_logits[h, d n + i] (=|+=) (G[h,d] c_i + gp 2^i (1 - 2p) / (H D n)) p (1 - p),  p = sigmoid(logit), c = [1,2,..,-2^(n-1)]
 * G [H,D] = d loss / d int_w (NULL = polarize term only); gp_dev: device scalar holding the upstream gradient of
 * polarize_loss (polarize_lambda under the reference trainer, training/trainer.py:150), NULL = use gp_host.
 * accumulate 0: overwrite, 1: += */
int qsae_bsae_logit_grad(const float* logits, const float* G, int H, int D, int n_bits, const float* gp_dev, float gp_host,
                         int accumulate, float* grad_logits /* [H, D*n_bits] */, void* stream);

/* STE backward of QuantizedMatryoshkaDecoder.forward wrt weight / weight_mirror (sae/quantized_matryoshka.py:94-121,
 * joint_gradient = False) and apply_secant_grad (:145-190), over the active lists exported by
 * qsae_matryoshka_forward_active.
 * step 1 (scatter): M[h,:] += grad_levels[level(h)][b,:] for every active (b,h); z2[h] += 1      (M, z2 caller-zeroed)
 * step 2 (finish):  grad_w[h,d]  += (alpha[h] M[h,d] - sec[h] Bsign(w[h,d])) s'(w[h,d]), same for the mirror, with
 *                   sec[h] = c m z2[h] alpha[h]^2 (c = 1/B/D; m = n_bits - level if joint_bits = n_bits > 0, else 1);
 *                   M NULL = secant term only (apply_secant_grad), z2 NULL = STE term only (loss.backward()). */
int qsae_matryoshka_backward_scatter(const int32_t* active_idx, int B, int cap, int H, int D,
                                     const float* const* grad_levels /* host array of n_levels device pointers [B,D] */,
                                     const int* level_start /* host, n_levels + 1 */, int n_levels, float* M /* [H,D] */,
                                     int32_t* z2 /* [H] */, void* stream);
int qsae_matryoshka_backward_finish(const float* w, const float* w_mirror, const float* M, const int32_t* z2,
                                    const float* alpha /* [H] scale_vector */, const int* level_start /* host */,
                                    int n_levels, int H, int D, float c, int joint_bits, float* grad_w, float* grad_w_mirror,
                                    void* stream);

/* The same STE term at any activity, from the bf16 0/1 activity mask [B, H] of qsae_matryoshka_forward_dense (an
 * untrained q_sae has ~50 % of its latents active, far more than the active lists hold):
 *   grad_w[h,d] += alpha[h] M[h,d] s'(w[h,d]), same for the mirror,  M[h,:] = sum_b mask[b,h] grad_levels[level(h)][b,:]
 *   z2[h] = sum_b mask[b,h]  (WRITTEN, exact int32; the input of the secant step, qsae_matryoshka_backward_finish)
 * M is a tensor-core product mask^T g per level whose epilogue applies the STE factor (M never reaches memory); every
 * element of the .grad buffers has one writer, so the result is bit-deterministic. exact != 0: the gradients enter as
 * three bf16 parts (fp32-accurate; the mask is exact in bf16), exact = 0: one bf16 part. Workspace: the bf16 parts of
 * the level gradients (qsae_matryoshka_backward_dense_workspace_bytes), 1024-byte aligned. No host synchronisation.
 * Limits: H % 8 == 0, D % 16 == 0 and D <= 512, 1..8 levels; mask, gradients, weights and .grad 16-byte aligned.
 * B == 0 zeroes z2 and leaves the gradients untouched. */
int qsae_matryoshka_backward_dense_workspace_bytes(int B, int D, int n_levels, int exact, size_t* bytes);
int qsae_matryoshka_backward_dense(const uint16_t* mask /* bf16 [B, H] */, int B, int H, int D,
                                   const float* const* grad_levels /* host array of n_levels device pointers [B,D] */,
                                   const int* level_start /* host, n_levels + 1 */, int n_levels, const float* w,
                                   const float* w_mirror, const float* alpha /* [H] scale_vector */, int exact,
                                   float* grad_w, float* grad_w_mirror, int32_t* z2 /* [H] */, void* workspace,
                                   size_t workspace_bytes, void* stream);

/* RigL mask maintenance of STEWeights (sae/ternary.py:27-90); weight, mask [D,H] float32 (mask holds 0 / 1), both
 * updated in place; exact order statistics by a three-pass radix select on the device, no host synchronisation.
 * Ties at a cut that torch.topk leaves unspecified are resolved by the lowest flat index.
 * qsae_rigl_init_mask:   the n_inactive smallest |w| -> mask 0; weight *= mask                          (:27-39)
 * qsae_rigl_update_mask: drop every active |w| <= the n_drop-th smallest active |w|; grow the n_grow largest
 *                        |d_mean[d]| |a_mean[h]| among inactive positions; weight *= mask                (:54-87)
 *                        a_mean [H] / d_mean [D] = batch means of input_activations / output_grad (NULL: no grow step)
 * qsae_mul_inplace:      a *= b (mask_grad, :89-90) */
int qsae_rigl_workspace_bytes(size_t* bytes);
int qsae_rigl_init_mask(float* weight, float* mask, int D, int H, unsigned long long n_inactive, void* workspace,
                        size_t workspace_bytes, void* stream);
int qsae_rigl_update_mask(float* weight, float* mask, const float* a_mean, const float* d_mean, int D, int H,
                          unsigned long long n_drop, unsigned long long n_grow, void* workspace, size_t workspace_bytes,
                          void* stream);
int qsae_mul_inplace(float* a, const float* b, size_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* QSAE_B200_H */
