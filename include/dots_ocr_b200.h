/*
 * dots_ocr_b200.h -- C ABI of libdots_ocr_b200.so: hand-written sm_100a kernels for the
 * dots.ocr page-parsing hot path (ViT encode -> LLM prefill -> greedy decode).
 *
 * The reference (rednote-hilab/dots.ocr) has no FFI of its own: its seam is the Python call
 * `self.model.generate(**inputs, max_new_tokens=N)` (dots_ocr/parser.py:110) whose arithmetic
 * lives in HF remote code + torch/cuBLAS/flash-attn binaries.  Each entry point below replaces
 * one of those library kernels; the citation names the reference-side operator it stands in for
 * ([V] = vllm/model_executor/models/dots_ocr.py, [Q] = transformers/models/qwen2/modeling_qwen2.py,
 * [G] = transformers/generation/utils.py -- the in-container mirrors SURVEY.md cites).
 *
 * Conventions: plain C types only; every pointer is a DEVICE pointer owned by the caller unless
 * stated otherwise; `stream` is a cudaStream_t passed as void*; return 0 on success, negative on
 * error (text via dots_last_error(), thread-local); no allocation and no synchronisation inside
 * any call; bf16 tensors are row-major with explicit row pitch in ELEMENTS.
 */
#ifndef DOTS_OCR_B200_H
#define DOTS_OCR_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define DOTS_ABI_VERSION 2

#if defined(__GNUC__)
#define DOTS_API __attribute__((visibility("default")))
#else
#define DOTS_API
#endif

/* GEMM epilogues (rounding points follow HF eager: every nn.Linear output is rounded to bf16) */
#define DOTS_EPI_STORE 0         /* out = bf16(acc) */
#define DOTS_EPI_BIAS 1          /* out = bf16(acc + bias[n]) */
#define DOTS_EPI_BIAS_GELU 2     /* out = bf16(gelu_erf(bf16(acc + bias[n])))          [V]:196-212 */
#define DOTS_EPI_RESIDUAL 3      /* out = bf16(bf16(acc) + residual[m, n])             [V]:466,472  [Q]:302,308 */
#define DOTS_EPI_SWIGLU 4        /* W rows interleaved per 128: [64 gate | 64 up];
                                    out[m, N/2] = bf16(bf16(silu(bf16 g)) * bf16 u)     [V]:334-356  [Q]:46-48 */
#define DOTS_EPI_F32_PARTIAL_T 5 /* internal: swap-AB split-K partials */
#define DOTS_EPI_BF16_T 6        /* internal: swap-AB transposed bf16 store */
#define DOTS_EPI_SWIGLU_T 7      /* internal: swap-AB gate|up GEMM with fused SwiGLU */
#define DOTS_EPI_ROPE 8          /* internal (dots_gemm_bf16_rope): ViT q|k|v projection + 2-D rotary embedding */

DOTS_API const char* dots_last_error(void);
DOTS_API int dots_abi_version(void);
DOTS_API int dots_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Programmatic dependent launch between consecutive kernels of a stream (default on): weight prefetch, barrier
 * setup and TMEM allocation of kernel N+1 overlap the tail of kernel N.  0 = plain stream order. */
DOTS_API int dots_set_pdl(int enable);

/* 1: large prefill GEMMs run on CTA pairs (tcgen05 cta_group::2, 256 x 256 tiles per 2-CTA cluster); 0: one CTA per tile. */
DOTS_API int dots_set_gemm_pair(int enable);

/* ---- dense contractions (tcgen05 / TMEM / TMA) -------------------------------------------- */

/* out[M, N(/2)] = epilogue(A[M, K] * W[N, K]^T).  Replaces every nn.Linear / Conv2d-as-GEMM on the
 * prefill side: [V]:287 qkv, :315 proj, :334-356 fc1|fc3,fc2, :405-415 patch embed, :196-212 merger;
 * [Q]:217-219 q/k/v (fused, +bias), :243 o_proj, :46-48 gate|up, down.  K, N, pitches % 8 == 0. */
DOTS_API int dots_gemm_bf16(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo,
                   int M, int N, int K, int epilogue, const void* bias, const void* residual, long long ldr,
                   void* stream);

/* ViT q|k|v projection with the 2-D rotary embedding fused into the epilogue ([V]:287 + :295-302): the first rope_cols columns
 * (q heads then k heads, 128 wide each) are rotated NeoX-style in fp32 after the bf16 rounding of the Linear output -- bit-identical
 * to dots_gemm_bf16(STORE) followed by dots_vit_rope_apply, without that kernel's read-modify-write pass over q and k.
 * cos_t / sin_t: [M, 64] fp32 from dots_vit_rope_table. */
DOTS_API int dots_gemm_bf16_rope(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int M, int N,
                        int K, const float* cos_t, const float* sin_t, int rope_cols, void* stream);

/* Decode-time skinny GEMM (batch <= 256 rows), swap-AB so the weight matrix is the 128-row tensor-core
 * operand and streams from HBM once.  Either
 *   partial != NULL: partial[s][b][n] (fp32, s < splits) = sum over the s-th K slice, or
 *   out_bf16 != NULL (splits must be 1): out_bf16[b, n] = bf16(acc (+ bias[n])).
 * Replaces the M = batch nn.Linear calls of one decode step ([Q]:217-219, 243, 46-48, 474-475). */
DOTS_API int dots_gemm_skinny_bf16(const void* X, long long ldx, const void* W, long long ldw, float* partial,
                          void* out_bf16, long long ldo, const void* bias, int batch, int N, int K, int splits,
                          void* stream);

/* Decode gate|up projection with SwiGLU fused: act[b, I] = bf16(bf16(silu(bf16 g)) * bf16 u), W = interleaved gate|up weight
 * [2I, K] as for DOTS_EPI_SWIGLU.  Replaces dots_gemm_skinny_bf16 + dots_decode_swiglu for one decode step ([Q]:46-48). */
DOTS_API int dots_gemm_skinny_swiglu_bf16(const void* X, long long ldx, const void* W, long long ldw, void* act, long long ld_act,
                                 int batch, int two_i, int K, void* stream);

/* ---- attention ------------------------------------------------------------------------------ */

/* Variable-length fused attention, head_dim 128.  q/k/v are token-major with per-token strides
 * (elements) so they may alias a fused qkv buffer.  causal=0: ViT bidirectional per image
 * ([V]:304-310, flash_attn_varlen_func); causal=1: LLM prefill, GQA ([Q]:161-183,227-241). */
DOTS_API int dots_attn_varlen_fwd(const void* q, long long q_stride, const void* k, long long k_stride, const void* v,
                         long long v_stride, void* out, long long o_stride, const int* cu_seqlens, int n_seqs,
                         int max_seqlen, int n_q_heads, int n_kv_heads, int head_dim, int causal,
                         float softmax_scale, void* stream);

/* Same contract on the tcgen05 tensor cores (S = QK^T and O += PV accumulate in TMEM, K/V tiles arrive by TMA,
 * two 128-row query tiles per CTA ping-pong between the tensor pipe and the softmax warps).  total_tokens =
 * cu_seqlens[n_seqs] (rows of the q/k/v/out buffers; bounds the TMA maps).  Token strides % 8 == 0. */
DOTS_API int dots_attn_varlen_fwd_tc(const void* q, long long q_stride, const void* k, long long k_stride, const void* v,
                            long long v_stride, void* out, long long o_stride, const int* cu_seqlens, int n_seqs,
                            int max_seqlen, long long total_tokens, int n_q_heads, int n_kv_heads, int head_dim,
                            int causal, float softmax_scale, void* stream);

/* KV CACHE LAYOUT (all entry points that touch k_cache / v_cache): [batch, n_kv_heads, ctx_max, 128] bf16 with ctx_max % 64 == 0;
 * inside each (sequence, kv head) stripe the keys are stored in 64-key tiles of 16 KB whose byte order is the shared-memory image
 * the decode attention kernel consumes -- [dims 0-63 | dims 64-127][64 keys][128-byte row, 16-byte chunks XOR-swizzled by key & 7]
 * (ops.kv_tile / ops.kv_untile convert) -- so that one tile is ONE contiguous bulk copy instead of 128 row requests.
 *
 * One-token-per-sequence attention over the KV cache [batch, n_kv_heads, ctx_max, 128]
 * (replaces DynamicCache + sdpa/flash decode, transformers/cache_utils.py:102-120, [Q]:227-241).
 * ctx_len[b] = number of visible keys (current token's key already appended).
 * part_o [batch, n_q_heads, n_splits, 128] fp32 and part_ml [batch, n_q_heads, n_splits, 2] fp32 are
 * scratch, required when n_splits > 1. */
DOTS_API int dots_attn_decode(const void* q, const void* k_cache, const void* v_cache, const int* ctx_len, void* out,
                     float* part_o, float* part_ml, int batch, int n_q_heads, int n_kv_heads, int head_dim,
                     long long ctx_max, int n_splits, float softmax_scale, void* stream);

/* dots_attn_decode with the QKV finalize fused in front: the current token's q/k/v arrive as the split-K fp32 partials
 * qkv_partial [qkv_splits][batch][(n_q_heads + 2 n_kv_heads) * 128] of dots_gemm_skinny_bf16; the kernel reduces them in split
 * order, adds qkv_bias, applies HF's bf16 RoPE at pos[b] ([Q]:102-146), appends k, v at cache[b, :, pos[b]]
 * (cache_utils.py:119-120) and attends with q held in shared memory.  Requires ctx_len[b] == pos[b] + 1.
 * out_tile_rows > 0: `out` is written k-block-tiled with that many rows per tile (see the decode-projection section); 0: row-major. */
DOTS_API int dots_attn_decode_fused(const float* qkv_partial, int qkv_splits, const void* qkv_bias, const int* pos,
                           const float* inv_freq, void* k_cache, void* v_cache, const int* ctx_len, void* out,
                           int out_tile_rows, float* part_o, float* part_ml, int batch, int n_q_heads, int n_kv_heads,
                           int head_dim, long long ctx_max, int n_splits, float softmax_scale, void* stream);

/* dots_attn_decode_fused with the current token's q|k|v as the bf16 row [batch][(n_q_heads + 2 n_kv_heads) * 128] written by
 * dots_decode_gemm_qkv (bias already added): RoPE at pos[b] + KV append + attention.  out_tile_rows > 0: `out` is written in the
 * k-block-tiled activation layout (the B operand of dots_decode_gemm_resnorm) with that many rows per tile; 0: row-major. */
DOTS_API int dots_attn_decode_qkv(const void* qkv_bf16, const int* pos, const float* inv_freq, void* k_cache, void* v_cache,
                         const int* ctx_len, void* out, int out_tile_rows, float* part_o, float* part_ml, int batch,
                         int n_q_heads, int n_kv_heads, int head_dim, long long ctx_max, int n_splits, float softmax_scale,
                         void* stream);

/* 1 (default): 2..4 key splits of a (sequence, kv head) run as one thread-block cluster and are merged through distributed
 * shared memory by the leader CTA (no partial buffers, no combine launch); 0: always the combine kernel. */
DOTS_API int dots_set_decode_cluster(int enable);

/* TEST ONLY: fault injection that a parity test must detect (tests/test_bench_config_gpu.py).  0 = off; 1 = the decode
 * attention kernel drops the P*V contribution of the first 64-key tile of every sequence; 2 = of every other key tile. */
DOTS_API int dots_debug_set_fault(int code);

/* DIAGNOSTIC: arm (device buffer of u64: [0] = record counter, set to 0; [1] = capacity in records; then 3 words per record) or disarm
 * (NULL) the timeline instrumentation of the decode kernels (tools/decode_timeline.py). */
DOTS_API int dots_debug_set_trace(void* device_buffer);

/* ---- HBM-bound elementwise / reduction kernels ------------------------------------------------ */

/* pixel_values [rows, cols] fp32 (or bf16) -> bf16 [rows, ldo] zero-padded ([V]:586 `.to(dtype)`). */
DOTS_API int dots_cast_pad_bf16(const void* in, int in_is_bf16, long long rows, int cols, void* out, int ldo, void* stream);

/* GPU half of the image processor: uint8 RGB page [H, W, 3] (already smart-resized; H, W multiples of patch * merge) ->
 * rescale + normalise + patchify -> bf16 rows [H/patch * W/patch, ldo] in 2x2-merge token order, zero-padded to ldo.
 * mean255 / std255 are HOST pointers to 3 floats each (255 * CLIP mean / std).  Bit-identical to the host fp32 processor
 * followed by dots_cast_pad_bf16 ([C] image_processing_qwen2_vl.py:148-232). */
DOTS_API int dots_patchify_u8(const void* img_hwc, int H, int W, int patch, int merge, const float* mean255, const float* std255,
                     void* out, int ldo, void* stream);

/* Page resize on the GPU: uint8 RGB [H, W, 3] -> [rh, rw, 3], bicubic + antialias, bit-identical to the resize of the stock image
 * processor (torchvision resize on uint8 = Pillow's integer algorithm; [C] image_processing_qwen2_vl.py:148-232; reference entry
 * dots_ocr/utils/image_utils.py:116-138).  Horizontal pass then vertical pass with a uint8 intermediate `tmp` [H, rw, 3] (needed only
 * when both axes change).  Tap tables per axis are DEVICE arrays built by dots_ocr_b200/resize.py: xmin / xsize [out] int32, w [out,
 * ksize] int16 fixed point with `prec` fractional bits. */
DOTS_API int dots_resize_bicubic_u8(const void* img_hwc, int H, int W, void* tmp, void* out, int rh, int rw, const int* xmin_x,
                           const int* xsize_x, const short* w_x, int ksize_x, int prec_x, const int* xmin_y, const int* xsize_y,
                           const short* w_y, int ksize_y, int prec_y, void* stream);

/* RMSNorm, fp32 statistics: out = bf16(bf16(x * rsqrt(mean x^2 + eps)) * w)   ([Q]:258-263, [V]:450,456,518). */
DOTS_API int dots_rmsnorm(const void* x, long long ldx, const void* w, void* out, long long ldo, long long rows, int cols,
                 float eps, void* stream);

/* LayerNorm with affine (PatchMerger.ln_q, [V]:190-191). */
DOTS_API int dots_layernorm(const void* x, long long ldx, const void* w, const void* b, void* out, long long ldo,
                   long long rows, int cols, float eps, void* stream);

/* ViT 2-D rotary table: cos/sin [total_tokens, 64] fp32 from per-image grids (h, w) in 2x2-merge token
 * order ([V]:163-174, 536-568).  grid_hw is [n_img, 2]; cu_seqlens [n_img + 1]; inv_freq [32]. */
DOTS_API int dots_vit_rope_table(const int* cu_seqlens, const int* grid_hw, int n_img, const float* inv_freq, int half,
                        int merge, float* cos_t, float* sin_t, int total_tokens, void* stream);

/* In-place NeoX rotate-half (fp32 math) on the q and k thirds of qkv [S, 3*heads*128] ([V]:295-302). */
DOTS_API int dots_vit_rope_apply(void* qkv, long long ld, int S, int heads, int head_dim, const float* cos_t,
                        const float* sin_t, void* stream);

/* LLM prefill: 1-D RoPE (bf16 arithmetic like HF, [Q]:102-146) in place on q,k of qkv [T, (nq+2nkv)*128]
 * and append k, v at cache[seq_of_tok[t], :, positions[t]]  (cache_utils.py:119-120). */
DOTS_API int dots_llm_rope_kv_append(void* qkv, long long ld, int T, int n_q_heads, int n_kv_heads, int head_dim,
                            const int* positions, const int* seq_of_tok, const float* inv_freq, void* k_cache,
                            void* v_cache, long long ctx_max, void* stream);

/* masked_scatter bookkeeping: slots[t] = rank of token t among ids == image_token_id, else -1. */
DOTS_API int dots_image_slots(const long long* ids, int T, long long image_token_id, int* slots, int* count_out, void* stream);

/* out[t] = slots[t] >= 0 ? img_embeds[slots[t]] : table[ids[t]]   (embed_tokens + masked_scatter, SURVEY M1). */
DOTS_API int dots_embed_scatter(const long long* ids, const int* slots, const void* table, const void* img_embeds, void* out,
                       int T, int H, long long vocab, void* stream);

DOTS_API int dots_gather_rows(const void* src, long long lds, const int* rows, void* out, long long ldo, int n, int cols,
                     void* stream);

/* Greedy step: argmax over bf16 logits in fp32, lowest index wins ties ([G]:2762,2793); finished rows emit
 * pad, ANY of the stop ids marks a row finished ([G]:2796-2805 with generation_config.eos_token_id a list);
 * appends to out_ids[b, step[b]] and advances step/pos/ctx_len.  stop_ids is a HOST pointer to n_stops <=
 * DOTS_MAX_STOP_IDS ids (copied into the launch; n_stops == 0 disables stopping).  forced_ids (optional)
 * overrides the chosen token (teacher forcing for parity tests).  Nullable: out_ids, step, pos, ctx_len,
 * finished, forced_ids. */
#define DOTS_MAX_STOP_IDS 4
DOTS_API int dots_argmax_advance(const void* logits, long long ldl, int batch, int vocab, long long* next_ids,
                        long long* out_ids, long long out_ld, int* step, int* pos, int* ctx_len, int* finished,
                        const long long* stop_ids, int n_stops, long long pad_id, const long long* forced_ids,
                        long long forced_ld, void* stream);

/* Sampled step with per-row parameters, then the bookkeeping of dots_argmax_advance (same arguments, same nullability).
 * temperature[batch] (f32), top_p[batch] (f32), top_k[batch] (i32), seed[batch] (u64) are DEVICE arrays, read at run time
 * (a captured decode graph picks up rewritten values).  Per row, on the logits in fp32, in HF's warper order:
 * temperature < 1e-5 -> greedy, bit-identical to dots_argmax_advance; top_k > 0 keeps l >= the k-th largest l (ties kept);
 * top_p < 1 keeps, among those, every l whose softmax(l / T) mass of strictly larger logits is < top_p (ties with the last
 * kept value kept); the token is argmax over the kept set of l / T - log(-log u), u from Philox4x32-10 with key = seed[b]
 * and counter = (index >> 2, step[b], 0, 0), word index & 3, u = ((x >> 8) + 0.5) * 2^-24.  A row's token depends only on
 * its logits, parameters, seed and step. */
DOTS_API int dots_sample_advance(const void* logits, long long ldl, int batch, int vocab, long long* next_ids,
                        long long* out_ids, long long out_ld, int* step, int* pos, int* ctx_len, int* finished,
                        const long long* stop_ids, int n_stops, long long pad_id, const long long* forced_ids,
                        long long forced_ld, const float* temperature, const float* top_p, const int* top_k,
                        const unsigned long long* seed, void* stream);

/* ---- decode-step fused finalize kernels (split-K reduce + HF rounding points) ------------------ */
/* First kernel of a decode step: resid = embed[ids]; normed = RMSNorm(resid) * w; also zeroes counters[0..n_counters) -- the
 * rendezvous counters of this step's dots_decode_gemm_resnorm launches (counters may be NULL with n_counters == 0).
 * tile_rows = 32 / 64: normed is written k-block-tiled with that many rows per tile; 0: row-major [batch, H]. */
DOTS_API int dots_decode_embed_rmsnorm(const long long* ids, const void* table, long long vocab, const void* w, void* resid,
                              void* normed, int batch, int H, float eps, unsigned int* counters, int n_counters, int tile_rows,
                              void* stream);
/* tile_rows > 0: normed is written k-block-tiled (rows per tile); 0: row-major. */
DOTS_API int dots_decode_residual_rmsnorm(const float* partial, int splits, void* resid, const void* w, void* normed,
                                 int batch, int H, float eps, int tile_rows, void* stream);
DOTS_API int dots_decode_qkv_rope_append(const float* partial, int splits, const void* bias, const int* pos,
                                const float* inv_freq, void* q_out, void* k_cache, void* v_cache, long long ctx_max,
                                int batch, int n_q_heads, int n_kv_heads, int head_dim, void* stream);
DOTS_API int dots_decode_swiglu(const float* partial, int splits, void* act, int batch, int inter, void* stream);

/* ---- decode-step projections over PRE-TILED operands, split-K reduction on chip ----------------------------------------
 * Operand layouts (host helpers: ops.tile_weight / ops.tile_rows / ops.untile_rows; device: tiled_row_off in csrc/ptx.cuh):
 *   Wt  weights [N, K] as [ceil(N/128)][ceil(K/64)] contiguous 16 KB blobs, each the K-major SWIZZLE_128B shared-memory image of a
 *       128-row x 64-column tile (zero padded);
 *   Xt  activations [batch, K] as [ceil(K/64)] blobs of R x 128 B (R = 32 for batch <= 32, else 64), same swizzle.
 * One ring stage of these GEMMs is ONE 1-D bulk copy per operand: a tensor-map copy of 128-byte rows tops out near 40 GB/s per SM
 * on B200 (one L2 request per row), a bulk copy streams > 100 GB/s per SM (profiles/microbench_r2.md). */

/* q|k|v projection of one decode step, batch <= 64: out[b, n] = bf16(X[b, :] . W[n, :] + bias[n])  ([Q]:217-219, fused
 * q|k|v weight), out row-major with pitch ldo.  K is split over the 8 CTAs of a cluster per 128-row weight tile and reduced
 * through distributed shared memory in split order (deterministic). */
DOTS_API int dots_decode_gemm_qkv(const void* Xt, const void* Wt, const void* bias, void* out, long long ldo, int batch, int N,
                         int K, void* stream);

/* o_proj / down_proj of one decode step with everything up to the next GEMM's input fused, batch <= 64:
 *   x = bf16(bf16(X . W^T) + resid);  resid = x (row-major [batch, N]);  normed_t = bf16(bf16(x * rsqrt(mean x^2 + eps)) * ln_w),
 * written k-block-tiled ([Q]:243,302-308 and :46-48,308 + :258-263).  stats: scratch [ceil(N/128)][64] fp32; counter: one uint32
 * that is ZERO when the kernel starts (the kernel's CTAs rendezvous on it once; dots_decode_embed_rmsnorm re-zeroes a block of
 * counters at the start of every step).  All ceil(N/128) clusters must be co-resident (checked: dots_decode_gemm_max_clusters). */
DOTS_API int dots_decode_gemm_resnorm(const void* Xt, const void* Wt, void* resid, const void* ln_w, void* normed_t, float* stats,
                             unsigned int* counter, int batch, int N, int K, float eps, void* stream);

/* gate|up projection + SwiGLU of one decode step, batch <= 64 (no split-K: 2I/128 tiles cover the SMs).  Wt = tiled interleaved
 * gate|up weight [2I, K] (as DOTS_EPI_SWIGLU); act_t [batch, I] = bf16(bf16(silu(bf16 g)) * bf16 u), written k-block-tiled. */
DOTS_API int dots_decode_gemm_swiglu(const void* Xt, const void* Wt, void* act_t, int batch, int two_i, int K, void* stream);

/* Split-K partials over tiled operands: partial[s][b][n] fp32 (dots_gemm_skinny_bf16 with bulk-copied operands). */
DOTS_API int dots_decode_gemm_partial(const void* Xt, const void* Wt, float* partial, int batch, int N, int K, int splits, void* stream);

/* Ring depths (2..8 stages of 16 KB weights + batch-tile activations) of the decode GEMM families: split-K partial GEMMs (additionally
 * capped by the k-blocks one CTA owns), gate|up + SwiGLU, lm_head.  Defaults 6 / 5 / 4 (measured best at batch 64). */
DOTS_API int dots_set_decode_stages(int partial, int swiglu, int head);

/* lm_head of one decode step, batch <= 64: out[b, n] = bf16(X . W^T), row-major.  x_tile_rows = 32 / 64: X is k-block-tiled;
 * x_tile_rows = 0: X is row-major with pitch ldx (first token after prefill). */
DOTS_API int dots_decode_gemm_head(const void* X, long long ldx, int x_tile_rows, const void* Wt, void* out_bf16, long long ldo,
                          int batch, int N, int K, void* stream);

/* Number of 8-CTA clusters of dots_decode_gemm_resnorm the current device keeps resident at once. */
DOTS_API int dots_decode_gemm_max_clusters(int batch, int* out);

/* ---- SM partitions (two phases of the page pipeline side by side on one GPU) -------------------
 * dots_partition_create splits the current device's SMs into a first group of `sms_first` SMs (a multiple of 8; it keeps the
 * thread-block-cluster guarantees, so the CTA-pair prefill GEMMs go there) and the rest, as two CUDA green contexts, and returns
 * one non-blocking stream in each (usable wherever this header takes a `void* stream`, and by the CUDA runtime of the caller) plus
 * the SM counts the driver actually provisioned.  Kernels launched into such a stream run on its SMs only.  One partition per
 * device; dots_partition_destroy synchronises the device and releases it (safe to call when none exists).
 * dots_set_sm_count(n): the persistent kernels launched next (by this host thread's calls, on the current device) size their
 * grids for n SMs instead of the whole device; 0 restores the device count.  Set it to a partition's count before feeding that
 * partition's stream. */
DOTS_API int dots_partition_create(int sms_first, void** stream_first, void** stream_rest, int* n_first, int* n_rest);
DOTS_API int dots_partition_destroy(void);
DOTS_API int dots_set_sm_count(int n);

/* ---- CUDA-graph helpers (the decode step is captured once and replayed) ----------------------- */
DOTS_API int dots_graph_begin(void* stream);
DOTS_API int dots_graph_end(void* stream, void** graph_exec_out);
DOTS_API int dots_graph_launch(void* graph_exec, void* stream);
DOTS_API int dots_graph_destroy(void* graph_exec);

#ifdef __cplusplus
}
#endif
#endif /* DOTS_OCR_B200_H */
