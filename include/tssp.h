/* tssp.h -- C ABI of the B200-native 2SSP ViT calibration/pruning hot path (libtssp_b200.so).
 *
 * The reference (zvezdvv/2ssp-X-vit) has no FFI: its hot path is eager PyTorch inside src/vit_pruning.py.
 * Each entry point below replaces the body of one reference function (cited per function as
 * reference file:line relative to the reference repo root); the Python shim in 2ssp-x-vit_b200/api.py keeps the
 * reference's own signatures and calls these through ctypes. INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; tssp_last_error() gives the message
 *     (thread-local). No C++ exception crosses this boundary. There is no CPU fallback.
 *   - pointers are caller-owned. `*_on_host` flags say whether a buffer is host (ideally pinned) or device
 *     memory. HOST input buffers (pixels, labels) are copied on the engine's own copy stream, double-buffered so
 *     the transfer of one batch runs under the kernels of the previous one, and the call returns only after those
 *     copies have completed: a host buffer may be freed or overwritten as soon as the call returns (a
 *     DataLoader(pin_memory=True) batch needs no further care). DEVICE input buffers are read by kernels enqueued on
 *     `stream` and must stay valid until that work has run, as with any stream-ordered API.
 *   - `stream` is a cudaStream_t passed as void*; all kernels are enqueued on it (per-batch chains as one CUDA graph
 *     launch), calls return without waiting for them unless they hand results back to host memory.
 *   - all device memory is allocated in tssp_create(); no allocation happens afterwards.
 *   - entry points are serialised by a library-wide lock (safe to call from several threads; one process per GPU
 *     is the intended use). Engine entry points run on the engine's device and restore the caller's current device.
 *   - matrices are row-major with PyTorch layouts (nn.Linear weight = [out_features, in_features]).
 */
#ifndef TSSP_H_
#define TSSP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSSP_MAX_BLOCKS 64
#define TSSP_ABI_VERSION 2

typedef struct tssp_engine* tssp_handle_t;

/* Model anatomy, as discovered by the reference's _get_encoder/_gather_mlp_pairs walkers
 * (src/vit_pruning.py:28-75) on an HF ViTForImageClassification or a timm VisionTransformer, and the options of the timm
 * VisionTransformer models beyond plain ViT (timm vision_transformer.py: VisionTransformer._pos_embed, LayerScale,
 * Block.forward, pre_norm, act_layer). Zero is the plain-ViT behaviour of every option, so a zeroed struct with the model's
 * shape filled in describes a ViT with one CLS token.
 * Tokens per image T = (image_size / patch_size)^2 + 1 + dist_token + register_tokens must lie in [32, 1025]: ViT-x/16 up
 * to 512x512 (T = 1025), ViT-x/8 up to 256x256, ViT-x/14 up to 448x448; tssp_create rejects other shapes (DINOv2 at its
 * native 518x518: T = 1370) and invalid options before it touches a device. */
#define TSSP_MAX_REGISTER_TOKENS 7
#define TSSP_FFN_GELU 0        /* erf GELU (nn.GELU(), HF "gelu") */
#define TSSP_FFN_QUICK_GELU 1  /* QuickGELU, x * sigmoid(1.702 x) (timm QuickGELU); needs score_point = 1 */
typedef struct tssp_config {
    int32_t n_blocks;                      /* B: encoder blocks */
    int32_t hidden;                        /* D: 192 (DeiT-Ti, ViT-Ti) or a multiple of 128, <= 1024 */
    int32_t heads;                         /* D / heads must be 64 */
    int32_t image_size;                    /* H = W, multiple of patch_size */
    int32_t patch_size;                    /* P: any size dividing image_size; the patch vector C_in*P*P is zero padded
                                              to a multiple of 8 inside the engine (P = 14: 588 -> 592) */
    int32_t channels;                      /* C_in (3) */
    int32_t n_classes;                     /* classifier outputs (0: no head, logits/eval unavailable) */
    int32_t head_hidden;                   /* 0: Linear head; >0: Sequential(Linear(D,h,bias=False), GELU, Linear(h,C))
                                              (experiments/vit_pruning/auto_2ssp.py:559-566) */
    int32_t max_images;                    /* batch capacity of the workspace */
    int32_t score_point;                   /* 0: hook after GELU (HF layer.intermediate, src/vit_pruning.py:130)
                                              1: hook before GELU (timm mlp.fc1, src/vit_pruning.py:135) */
    int32_t cache_blocks;                  /* 1: allocate the Stage-2 pre-block activation cache */
    float ln_eps;                          /* LayerNorm eps of the module (1e-12 HF, 1e-6 timm norms) */
    int32_t dist_token;                    /* 1: DeiT distillation token after CLS (transformers DeiTEmbeddings.forward:
                                              [CLS, distillation token, patches] + positions; timm
                                              VisionTransformerDistilled). With a distillation head the logits are
                                              (cls_head(row 0) + dist_head(row 1)) / 2, the eval-mode output of
                                              DeiTForImageClassificationWithTeacher and of timm's distilled models; a
                                              Sequential head cannot be combined with one. Without it
                                              (DeiTForImageClassification) the head reads the CLS row only. */
    int32_t register_tokens;               /* R timm register tokens after CLS (reg_token [1, R, D]), 0..7; not with
                                              dist_token. The classifier reads the CLS row. */
    int32_t pos_patches_only;              /* 0: pos table [T, D] covers the prefix rows (ViT, DeiT, DINOv2);
                                              1: pos table [G^2, D] for the patches only, the prefix rows get no
                                              position (timm no_embed_class: DeiT-III, DINOv2 with registers) */
    int32_t layer_scale;                   /* 1: every block scales its attention and MLP outputs by ls1.gamma /
                                              ls2.gamma before the residual add: x += gamma * (proj(a) + b), in fp32 */
    int32_t pre_norm;                      /* 1: a LayerNorm (timm norm_pre, eps = ln_eps) over every token after the
                                              position embedding and before block 0 (timm CLIP image towers) */
    int32_t ffn_act;                       /* TSSP_FFN_GELU or TSSP_FFN_QUICK_GELU: the activation between fc1 and fc2 of
                                              every block (a Sequential classification head keeps erf GELU) */
    int32_t ffn_dims[TSSP_MAX_BLOCKS];     /* F per block (intermediate width; may differ after Stage-1) */
    int32_t attn_present[TSSP_MAX_BLOCKS]; /* 0: this block's attention is already a bypass module */
} tssp_config_t;

/* The table of fp32 device pointers handed to tssp_load_weights(): the TSSP_W_GLOBAL_COUNT global entries, then
 * TSSP_BW_COUNT entries per block, always TSSP_W_GLOBAL_COUNT + n_blocks * TSSP_BW_COUNT pointers. The entries of an
 * option the config does not enable must be NULL. Q/K/V may alias one fused timm qkv weight (rows [0:D],[D:2D],[2D:3D],
 * experiments/vit_pruning/auto_2ssp.py:436-440). */
enum tssp_weight_index {
    TSSP_W_PATCH_W = 0, /* [D, C_in*P*P]  Conv2d weight flattened */
    TSSP_W_PATCH_B,     /* [D] */
    TSSP_W_CLS,         /* [D] */
    TSSP_W_POS,         /* [T, D], or [G^2, D] with pos_patches_only */
    TSSP_W_FINAL_LN_W,  /* [D] */
    TSSP_W_FINAL_LN_B,  /* [D] */
    TSSP_W_HEAD0_W,     /* [head_hidden, D] or NULL */
    TSSP_W_HEAD_W,      /* [C, D] or [C, head_hidden] */
    TSSP_W_HEAD_B,      /* [C] or NULL */
    TSSP_W_DIST_TOKEN,  /* dist_token: [D] distillation token (required) */
    TSSP_W_HEAD_DIST_W, /* dist_token: [C, D] distillation head, or NULL: the classifier reads the CLS row only */
    TSSP_W_HEAD_DIST_B, /* dist_token: [C] or NULL */
    TSSP_W_REG_TOKENS,  /* register_tokens > 0: [R, D] (row-major reg_token[0]) */
    TSSP_W_NORM_PRE_W,  /* pre_norm: [D] */
    TSSP_W_NORM_PRE_B,  /* pre_norm: [D] */
    TSSP_W_GLOBAL_COUNT
};
enum tssp_block_weight_index {
    TSSP_BW_LN1_W = 0, TSSP_BW_LN1_B,
    TSSP_BW_Q_W, TSSP_BW_Q_B, TSSP_BW_K_W, TSSP_BW_K_B, TSSP_BW_V_W, TSSP_BW_V_B, /* [D,D] / [D] (bias may be NULL) */
    TSSP_BW_PROJ_W, TSSP_BW_PROJ_B,
    TSSP_BW_LN2_W, TSSP_BW_LN2_B,
    TSSP_BW_FC1_W, TSSP_BW_FC1_B, /* [F, D] / [F] */
    TSSP_BW_FC2_W, TSSP_BW_FC2_B, /* [D, F] / [D] */
    TSSP_BW_LS1, TSSP_BW_LS2,     /* layer_scale: [D] gammas of the attention branch (NULL for a block without
                                     attention) and of the MLP branch */
    TSSP_BW_COUNT
};

int tssp_abi_version(void);
const char* tssp_last_error(void);

int tssp_create(const tssp_config_t* cfg, int device, tssp_handle_t* out);

/* Pixel input format of an engine's batch entry points (tssp_s1_batch, tssp_forward_logits, tssp_eval_batch,
 * tssp_s2_batch). TSSP_PIXELS_F32 (the default): `pixels` is fp32 [n, C, H, W], fed to the patch embedding as it is.
 * TSSP_PIXELS_U8: `pixels` is uint8 [n, C, H, W] (the bytes a JPEG decoder produces; C <= 4), read through the same
 * `const float*` parameter, and every pixel is normalised on the device as x = (float(u) * rescale - mean[c]) / std[c]
 * in IEEE fp32, one rounding per operation: the bits of the fp32 batch normalised that way on the host, at a quarter of
 * the host-to-device bytes. A device-resident uint8 batch must be 8-byte aligned when the patch size is a multiple of
 * 8, 2-byte aligned when it is even. Host uint8 batches follow the same lifetime rule as fp32 ones. */
#define TSSP_PIXELS_F32 0
#define TSSP_PIXELS_U8 1
#define TSSP_MAX_PIXEL_CHANNELS 4
typedef struct tssp_pixel_input {
    int32_t format; /* TSSP_PIXELS_F32 or TSSP_PIXELS_U8 */
    float rescale;  /* U8: multiplies every byte first (1/255 for the usual [0, 1] scaling) */
    float mean[TSSP_MAX_PIXEL_CHANNELS]; /* U8: per channel, entries past the model's channels are ignored */
    float std[TSSP_MAX_PIXEL_CHANNELS];  /* U8: per channel, > 0 */
} tssp_pixel_input_t;
/* Sets the format of the following batches. Under U8 the values must be finite, std > 0 and the model's channels in
 * [1, 4]; an invalid input is refused and the engine keeps its previous format. Needs no new device memory (a uint8 batch
 * is staged in the fp32 slots) and no new graph captures (the patch extraction runs outside the captured chains). */
int tssp_set_pixel_input(tssp_handle_t h, const tssp_pixel_input_t* input);
int tssp_destroy(tssp_handle_t h);
/* tssp_destroy parks the engine's device buffers in a per-process pool (exact-size reuse by the next tssp_create; capped
 * by TSSP_POOL_MB, default 16384, 0 = no pool); this returns all parked buffers to the driver. */
int tssp_trim_pool(void);

/* Packs the model's fp32 parameters into the engine's bf16 operand / fp32 vector arenas. */
int tssp_load_weights(tssp_handle_t h, const float* const* table, int n_entries, void* stream);
/* Re-packs one block's FFN after Stage-1 width pruning (new_F <= original F). */
int tssp_update_ffn(tssp_handle_t h, int block, int new_F, const float* fc1_w, const float* fc1_b,
                    const float* fc2_w, void* stream);
/* Marks blocks whose attention submodule has been replaced by a bypass (src/vit_pruning.py:500-504). */
int tssp_set_attention(tssp_handle_t h, const int32_t* present);

/* ---- Stage 1: activation-magnitude scores -- replaces _compute_ffn_activation_importance and its hook
 *      (src/vit_pruning.py:111-201, hook :143-158). Score sums are kept on the device across batches:
 *      sum_b[j] += sum_img sqrt(sum_tok a[img,tok,j]^2). The caller divides by the image count (:200). */
int tssp_s1_reset(tssp_handle_t h, void* stream);
/* img_norms (optional, device, [n][sum_b F_b] fp32): per-image norms of this batch, for GPU-count-invariant
 * reductions across data-parallel ranks. */
/* pixels: fp32 [n, C, H, W], or uint8 under TSSP_PIXELS_U8 (tssp_set_pixel_input) */
int tssp_s1_batch(tssp_handle_t h, const float* pixels, int n, int pixels_on_host, float* img_norms, void* stream);
/* scores: [sum_b F_b] fp32, blocks concatenated. Synchronises `stream` when out_on_host. */
int tssp_s1_scores(tssp_handle_t h, float* scores, int out_on_host, void* stream);

/* ---- forward / top-1 -- replaces the forward + argmax/compare of evaluate_top1 (src/vit_pruning.py:325-373).
 *      skip_attn (optional, [B]): 1 = evaluate with that block's attention removed (zero bypass).
 *      pixels: fp32 [n, C, H, W], or uint8 under TSSP_PIXELS_U8 (tssp_set_pixel_input), here and in tssp_eval_batch. */
int tssp_forward_logits(tssp_handle_t h, const float* pixels, int n, int pixels_on_host, const int32_t* skip_attn,
                        float* logits, int out_on_host, void* stream);
/* adds the number of correct top-1 predictions of this batch to *correct (device uint64). */
int tssp_eval_batch(tssp_handle_t h, const float* pixels, const int64_t* labels, int n, int on_host,
                    const int32_t* skip_attn, unsigned long long* correct_dev, void* stream);

/* ---- Stage 2: attention-removal search -- replaces the deepcopy-and-evaluate loop of
 *      prune_vit_attention_blocks (src/vit_pruning.py:463-497) and of
 *      Auto2SSPInterface._compute_att_depth_importance (pruning_srp-main/mask_conjunction.py:327-357).
 *      One baseline pass caches the activations entering every block; candidate i re-runs only blocks i..B-1.
 *      counts[0] = baseline correct, counts[1+i] = correct with block i's attention removed, accumulated over
 *      batches; cand_mask ([B] or NULL = all): only candidates with a non-zero entry are evaluated (sharding
 *      across ranks); run_baseline is a set of flags: TSSP_S2_COUNT_BASELINE (1) adds the baseline pass to counts[0]
 *      (0 leaves counts[0] untouched; the cache pass still runs), TSSP_S2_WITH_SCORES (2) makes the baseline pass also
 *      accumulate the Stage-1 score sums of the batch exactly as tssp_s1_batch would (call tssp_s1_reset first, read
 *      them with tssp_s1_scores): fit() of mask_conjunction.py:359-362 runs both passes over the same images.
 *      pixels: fp32 [n, C, H, W], or uint8 under TSSP_PIXELS_U8 (tssp_set_pixel_input). */
#define TSSP_S2_COUNT_BASELINE 1
#define TSSP_S2_WITH_SCORES 2
int tssp_s2_reset(tssp_handle_t h, void* stream);
int tssp_s2_batch(tssp_handle_t h, const float* pixels, const int64_t* labels, int n, int on_host,
                  const int32_t* cand_mask, int run_baseline, void* stream);
int tssp_s2_counts(tssp_handle_t h, int64_t* counts_host, void* stream); /* [B+1]; synchronises */

/* ---- Stage 1 neuron gather -- replaces W_int[keep], B_int[keep], W_out[:, keep] + clone()
 *      (src/vit_pruning.py:297-299). fp32 device pointers; keep: device int64 [k], ascending. Bit-exact. */
int tssp_ffn_gather(const float* fc1_w, const float* fc1_b, const float* fc2_w, int F, int D, const int64_t* keep,
                    int k, float* fc1_w_out, float* fc1_b_out, float* fc2_w_out, void* stream);
/* The same for n_blocks blocks in ONE launch (the per-block loop of src/vit_pruning.py:246-311 after its selection
 * step): HOST arrays of length n_blocks holding device pointers / sizes; fc1_b and fc1_b_out may be NULL (no bias) or
 * hold NULL entries. Blocks may have different F and k; D is the model's hidden size. */
int tssp_ffn_gather_batch(int n_blocks, const float* const* fc1_w, const float* const* fc1_b, const float* const* fc2_w,
                          const int32_t* F, int D, const int64_t* const* keep, const int32_t* k, float* const* fc1_w_out,
                          float* const* fc1_b_out, float* const* fc2_w_out, void* stream);

/* ---- kernel-level entry points (used by the parity tests and by the engine itself) ---- */
/* C[M,N] = A[M,K] * W[N,K]^T with a fused epilogue; mode: 0 bf16(acc+bias), 1 bf16 gelu, 2 bf16 gelu + score
 * partials, 3 same with pre-activation scores, 4 fp32 (reduce_add: C += ...), 7 bf16 quickgelu(acc+bias), 8 the same with
 * pre-activation score partials (those of mode 3 for the same operands). A, W bf16; lda/ldw/ldc in elements.
 * K is a multiple of 8; past K the operands' tiles are zero filled, so any such K works (the padded patch vector). */
int tssp_op_gemm(int mode, const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
                 const float* bias, float* partials, int ldp, int tokens_per_image, int reduce_add, void* stream);
/* the QKV form (mode 5): bf16 C = A W^T + bias, and rownorm[m][c] = sum of squares of the fp32 values of columns
 * [64c, 64c+64) of row m (|q|^2, |k|^2 per head for the attention kernel) for c < rownorm_chunks */
/* the LayerScale form (mode 6): fp32 C (=|+=) col_scale[c] * (A W^T + bias)[., c] */
int tssp_op_gemm_scaled(const void* A, int lda, const void* W, int ldw, float* C, int ldc, int M, int N, int K, const float* bias,
                        const float* col_scale, int reduce_add, void* stream);
int tssp_op_gemm_rownorm(const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K, const float* bias,
                         float* rownorm, int ld_rownorm, int rownorm_chunks, void* stream);
int tssp_op_score_finish(const float* partials, int ldp, float* norms, int ldn, int n_img, int T, int F,
                         float* scores, void* stream);
int tssp_op_layernorm(const float* x, int64_t in_stride, const float* gamma, const float* beta, void* out_bf16,
                      int rows, int D, float eps, void* stream);
/* the same LayerNorm with fp32 rows of pitch out_stride (a multiple of 4, >= D); out_f32 may be x (in place). Rounded to
 * bf16, its output is tssp_op_layernorm's bit for bit. */
int tssp_op_layernorm_f32(const float* x, int64_t in_stride, const float* gamma, const float* beta, float* out_f32,
                          int64_t out_stride, int rows, int D, float eps, void* stream);
/* ctx[n*T, D] = softmax(Q K^T / 8) V per (image, head) from the fused qkv[n*T, 3D]; head_dim 64, 16 <= T <= 1025
 * (up to 208 padded keys one kernel holds a whole key row, beyond that a second one streams keys in tiles of 128). */
int tssp_op_attention(const void* qkv_bf16, void* ctx_bf16, int n_img, int T, int heads, int D, void* stream);
/* out[n * T, Kp] with T = (H/P)^2 + prefix_tokens and Kp = round_up(C*P*P, 8): prefix_tokens (1..8) zero rows ahead of
 * every image's patches, columns past C*P*P zero (the padded patch vector of patch sizes that are not a multiple of 8).
 * input NULL or of format TSSP_PIXELS_F32: pixels are fp32 [n_img, C, H, W]. TSSP_PIXELS_U8: pixels are uint8
 * [n_img, C, H, W], C in [1, 4], normalised with input's rescale, mean and std as under tssp_set_pixel_input: bit for bit
 * the fp32 form of the image (float(u) * rescale - mean) / std; they must be 8-byte aligned when P is a multiple of 8,
 * 2-byte aligned when P is even. */
int tssp_op_im2col(const void* pixels, void* out_bf16, int n_img, int C, int H, int W, int P, int prefix_tokens,
                   const tssp_pixel_input_t* input, void* stream);
int tssp_op_cast_bf16(const float* in, int rows, int cols, int ld_in, void* out_bf16, int rows_pad, int cols_pad,
                      int ld_out, void* stream);
int tssp_op_argmax_count(const float* logits, int ld, int n, int C, const int64_t* labels, int32_t* preds,
                         unsigned long long* correct_dev, void* stream);
/* ---- mask builders over the score tables of several methods (SURVEY 8(f) #3). All arrays are DEVICE pointers:
 * scores f64 [n_files][n_blocks][ld] (block b uses its first widths[b] <= max_width <= ld entries, neuron j at index j;
 * the doubles are the JSON values), widths / k / counts int32 [n_blocks], rmax / ranks int32, sums f64, mask uint8
 * [n_blocks][ld] (1 = prune). Comparison and integer work plus IEEE double adds in file order: bit-identical to the
 * reference scripts. The callers' scalar control flow (rounding, growth of the selection fraction) stays on the host. */

/* rank[r][j] = position of j in a stable ascending sort of row r: replaces sorted(keys, key=(value, (i, j))) of
 * manual-experiments/consensus_mask.py:232-236 and sorted(items, key=value) of aggregate_and_mask-summation.py:256 */
int tssp_op_stable_rank_f64(const double* values, int rows, int cols, int ld, int32_t* ranks, void* stream);
/* ranks of every (file, block) row -> ranks_ws [n_files][n_blocks][ld]; rmax[b][j] = max over files (j is in every
 * file's bottom-k set iff rmax < k: consensus_mask.py:228-241); sums[b][j] = v_0 + v_1 + ... in file order (:281-285) */
int tssp_mask_consensus_prepare(const double* scores, int n_files, int n_blocks, const int32_t* widths, int max_width,
                                int ld, int32_t* ranks_ws, int32_t* rmax, double* sums, void* stream);
/* counts[b] = |{j : rmax[b][j] < k[b]}|, the size of the intersection probed by consensus_mask.py:245-256 */
int tssp_mask_count_less(const int32_t* rmax, int n_blocks, const int32_t* widths, int ld, const int32_t* k,
                         int32_t* counts, void* stream);
/* final mask (consensus_mask.py:263-296): the intersection {rmax < k[b]} when it has <= k_common members, else its
 * k_common members of smallest mean over files, ties by neuron index */
int tssp_mask_consensus_select(const int32_t* rmax, const double* sums, int n_files, int n_blocks, const int32_t* widths,
                               int max_width, int ld, const int32_t* k, int k_common, uint8_t* mask, void* stream);
/* summation builder (aggregate_and_mask-summation.py:138-157, 208-269): sums over files, then the
 * min(k_common, widths[b]) smallest sums of every block, ties by neuron index; ranks_ws int32 [n_blocks][ld] */
int tssp_mask_summation(const double* scores, int n_files, int n_blocks, const int32_t* widths, int max_width, int ld,
                        int k_common, double* sums, int32_t* ranks_ws, uint8_t* mask, void* stream);
/* raw min-max normalisation (manual-experiments/normalize_scores.py:44-73): minmax[0..1] = min, max over all n values,
 * out[i] = (v - min) / (max - min), 0 when max == min */
int tssp_op_minmax_normalize_f64(const double* values, long long n, double* minmax, double* out, void* stream);

/* ---- score file text -- replaces the json.dump of experiments/vit_pruning/auto_2ssp.py:769-786 (HOST arrays, no GPU work):
 * writes the bytes of json.dumps({"ffn": {"<b>:<j>": float(score)}}, indent=2) for the concatenated fp32 scores of
 * n_blocks blocks (widths[b] neurons each) into out. Returns the number of bytes written; when out is NULL or cap is
 * too small, the capacity to provide; -1 on a bad argument. Floats are CPython's repr of the exact double (shortest
 * round-trip digits, same fixed / scientific rule), non-finite values as json.dumps prints them. */
long long tssp_format_ffn_scores(const float* scores, const int32_t* widths, int n_blocks, char* out, long long cap);

/* diagnostics: the attention kernel's CTA 0 / chain 0 writes clock64() stamps (16 slots per query tile, first 16 tiles)
 * into device_buf (>= 256 int64) on every launch until called again with NULL. */
int tssp_debug_attention_trace(long long* device_buf);
/* the same for the GEMM kernel: CTA 0 writes 16 clock64() stamps per tile for its first 24 tiles (MMA thread, TMA thread,
 * epilogue warp 0; layout in csrc/gemm_tcgen05.cuh) into device_buf (>= 384 int64) on every launch until NULL. */
int tssp_debug_gemm_trace(long long* device_buf);
/* GEMM tile form for all following calls: 0 = chosen per problem by wave count (default), 1 = single-CTA 128x256 tiles,
 * 2 = CTA-pair 256x256 tiles (tcgen05 cta_group::2). Same results either way up to fp32 summation order inside the
 * tensor core; exists for A/B measurement and so that the parity tests can cover both forms. */
int tssp_set_gemm_form(int ctas);
/* 1 (default; TSSP_GRAPHS=0 in the environment starts with 0): the per-batch launch chains of tssp_s1_batch,
 * tssp_forward_logits, tssp_eval_batch and tssp_s2_batch are captured once per shape into CUDA graphs and replayed;
 * 0: every kernel is launched individually. Same kernels, same arguments, same bits; exists for A/B measurement and
 * for the parity tests. */
int tssp_set_graphs(int on);
/* number of kernels launched by this library since load (bench.py's gpu_launches; a replayed chain counts its kernels) */
unsigned long long tssp_launch_count(void);
/* number of launch chains captured into CUDA graphs since load (tests: a steady-state loop must not re-capture) */
unsigned long long tssp_graph_capture_count(void);
/* Per-kernel-class device timing (CUDA events on the launching stream) between begin and end.
 * Classes: 0 fc1(+GELU+score) 1 qkv 2 proj 3 fc2 4 patch-embed 5 head 6 attention 7 layernorm 8 score finisher 9 misc.
 * tssp_profile_end synchronises the device; arrays need >= TSSP_PROFILE_CLASSES entries. */
#define TSSP_PROFILE_CLASSES 10
int tssp_profile_begin(void);
int tssp_profile_end(double* ms_per_class, unsigned long long* launches_per_class, int n_classes);

#ifdef __cplusplus
}
#endif
#endif /* TSSP_H_ */
