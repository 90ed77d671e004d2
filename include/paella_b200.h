/* paella_b200 — C ABI of the B200-native Paella hot path.
 *
 * The reference (dome272/Paella @ e1ab72b) has no FFI layer: its boundary is the
 * Python class surface (SURVEY.md §8b).  This header is the C ABI the Python
 * mirror in paella_b200/ binds with ctypes; each entry point names the reference
 * code it replaces.  Conventions:
 *   - every pointer is a DEVICE pointer unless the name says `host`;
 *   - no function allocates or frees caller memory; scratch comes in as `workspace`;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*), no hidden syncs;
 *   - return 0 on success, non-zero on error with the text in pb200_last_error();
 *   - there is NO CPU fallback anywhere.
 * Layout: "NCHW"/"NHWC" as named; activations inside the library are channels-last.
 */
#ifndef PAELLA_B200_H
#define PAELLA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB200_ABI_VERSION 2

const char* pb200_last_error(void);
int pb200_abi_version(void);
/* multiprocessor count / max threads per SM of the current device (they fix PyTorch's Philox launch policy). */
int pb200_device_info(int* sm_count, int* max_threads_per_sm);

/* Measurement hooks used by bench.py: number of kernel launches the library has made so far, and optional
 * CUDA-event bracketing of every launch by kernel family (report: JSON {family: {launches, ms, work}},
 * work = algorithmic FLOPs for GEMM-shaped kernels, bytes otherwise). */
long long pb200_launch_count(void);
int pb200_profile_enable(int on);
int pb200_profile_report(char* buf, long long cap);

/* ------------------------------------------------------------------------------------------
 * Random streams and the resample step.  `seed`/`offset` are the (seed, philox offset) of the
 * torch CUDA generator BEFORE the op; each op consumes pb200_philox_offset_increment(numel)
 * offsets, exactly like the torch op it replaces, so a caller that advances the torch
 * generator by that amount stays on the reference's random stream.
 * ------------------------------------------------------------------------------------------ */
/* philox offsets one distribution kernel over `numel` elements consumes
 * (ATen/native/cuda/DistributionTemplates.h:50-62). */
int64_t pb200_philox_offset_increment(int64_t numel);

/* torch.randint(0, num_labels, size) -> int64   [ref/src/utils.py:37] */
int pb200_randint(int64_t* out, int64_t numel, int64_t num_labels, uint64_t seed, uint64_t offset, void* stream);

/* torch.rand(numel) fp32 in [0,1)               [the draw inside ref/src/modules.py:279] */
int pb200_rand(float* out, int64_t numel, uint64_t seed, uint64_t offset, void* stream);

/* torch.multinomial(p, 1)[:, 0] for p fp32 [rows, k] row-major; BIT-EXACT with torch given the
 * same generator state (argmax_k p/q, q = Tensor.exponential_(1))   [ref/src/utils.py:49-50] */
int pb200_multinomial(const float* p, int64_t rows, int64_t k, uint64_t seed, uint64_t offset, int64_t* out,
                      void* stream);

/* The whole resample expression of ref/src/utils.py:45-50 on reference-layout logits:
 *   l = logits_c*cfg + logits_u*(1-cfg)   (logits_u may be NULL: no guidance)
 *   p = softmax(l * (1/temperature), dim=1);  token = multinomial(p)
 * logits_*: fp32 NCHW [B, K, HW].  out: int64 [B, HW].
 * mode 0 = multinomial, 1 = argmax of logits (notebook `mode='argmax'`).
 * Same arithmetic as torch op-by-op except the softmax denominator's summation order. */
int pb200_resample_logits(const float* logits_c, const float* logits_u, int64_t batch, int64_t k, int64_t hw,
                          double cfg, double temperature, int mode, uint64_t seed, uint64_t offset, int64_t* out,
                          void* stream);

/* `quant` sampling mode (notebook cell 3; ref/src_distributed/train.py:155-156): e = softmax(l/T) @ codebook,
 * token = nearest code of e.  logits as above; codebook fp32 [k, c_latent]; no random draw. */
int pb200_resample_quant(const float* logits_c, const float* logits_u, int64_t batch, int64_t k, int64_t hw, double cfg,
                         double temperature, const float* codebook, int c_latent, int64_t* out, void* stream);

/* Paella.add_noise(x, t, random_x=...)            [ref/src/modules.py:277-283]
 *   mask = (rand_like(x.float()) <= t[:,None,None]); x*(1-mask) + random_x*mask
 * x, random_x, out: int64 [B, HW]; t: fp32 [B]; mask_out: int64 [B, HW] or NULL.
 * random_x == NULL -> randint_like(x, 0, num_labels) drawn AFTER the mask draw (second offset block). */
int pb200_add_noise(const int64_t* x, const int64_t* random_x, const float* t, int64_t batch, int64_t hw,
                    int64_t num_labels, uint64_t seed, uint64_t offset, int64_t* out, int64_t* mask_out,
                    void* stream);

/* ------------------------------------------------------------------------------------------
 * Vector quantiser (torchtools.nn.VectorQuantize; call sites ref/src/vqgan.py:94,104).
 * ------------------------------------------------------------------------------------------ */
/* nearest code (first minimum of |c|^2+|x|^2-2x.c, fp32 fma chain — oracle/vq_nearest.c).
 * x: fp32 [n, c] (channels-last vectors); codebook fp32 [k, c], c <= 8; idx: int64 [n]. */
int pb200_vq_nearest(const float* x, int64_t n, int c, const float* codebook, int k, int64_t* idx, void* stream);
/* idx2vq: out[n, c] = codebook[idx[n]] (channels-last). */
int pb200_vq_gather(const int64_t* idx, int64_t n, const float* codebook, int k, int c, float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Tensor-core GEMM (tcgen05, TMA-fed, TMEM accumulators): C[M,N] = A[M,K] . W[N,K]^T (+epilogue)
 * A, W: fp16 row-major (K contiguous), K % 8 == 0.  Used by every 1x1-conv / Linear of the path;
 * exported for unit tests.
 * ------------------------------------------------------------------------------------------ */
enum pb200_epilogue {
    PB200_EPI_F16 = 0,        /* out fp16 [M,ldo]   = acc + bias                                        */
    PB200_EPI_F32 = 1,        /* out fp32 [M,ldo]   = acc + bias                                        */
    PB200_EPI_GELU_F16 = 2,   /* out fp16 = gelu_erf(acc + bias); sqsum[row/rows_per_sample, n] += out^2 */
    PB200_EPI_RESID_F32 = 3,  /* out fp32 = ((acc + bias)*alpha + resid) [* (1+film_a) + film_b]         */
    PB200_EPI_UNPATCH_F32 = 4,/* out fp32 NHWC [B,2h,2w,cout]: col=(dy,dx,co), row=(b,y,x); bias[col]    */
    PB200_EPI_NCHW_F32 = 5,   /* out fp32 [B, N, hw]: row=(b,p) -> out[b][n][p]; acc + bias              */
    /* LayerNorm folded across two GEMMs (the AttnBlock's pre-norm, ref/src/modules.py:78): the producer also emits
     * the fp16 copy of its output row and the row statistics, the consumer multiplies the UN-normalised fp16 rows and
     * normalises in its epilogue:  LN(x) W^T = rstd * (x W^T - mean * rowsum(W)). */
    PB200_EPI_RESID_LN_F32 = 6, /* RESID_F32 + out16[M,ldo] = fp16(out - s); ln_stat[row] += (sum (out-s), sum (out-s)^2),
                                 * s = ln_shift[row] (0 if NULL).  LayerNorm is invariant under a per-row shift, so any s
                                 * is exact; an s near the row mean keeps the fp16 rounding of the copy relative to the row's
                                 * SPREAD instead of its offset (the executor passes the mean the previous AttnBlock saw). */
    PB200_EPI_F16_LN = 7       /* out fp16 = rstd[row]*(acc - mean'[row]*ln_wsum[n]) + bias, (mean', rstd) of the shifted
                                 * rows from ln_stat; if ln_mean_out: ln_mean_out[row] = ln_shift[row] + mean' (true mean) */
};

typedef struct pb200_gemm_epilogue {
    int mode;                  /* enum pb200_epilogue */
    const float* bias;         /* [N] or NULL */
    void* out;
    int64_t ldo;               /* leading dimension of out in elements (F16/F32/GELU/RESID) */
    const float* resid;        /* RESID: fp32 [M, ldr] (may alias out) */
    int64_t ldr;
    float alpha;               /* RESID: scale on (acc+bias); 1.0 for the denoiser */
    uint64_t* sqsum;           /* GELU: [M/rows_per_sample, N] sum of out^2 in 2^-24 fixed point (integer atomics:
                                  order-independent, hence run-to-run deterministic), or NULL */
    int rows_per_sample;       /* GELU/RESID(film)/NCHW: rows of one sample */
    const float* film;         /* RESID: fp32 [B, film_ld]: a = film[b, film_off + n], b = film[b, film_off + N + n]; or NULL */
    int64_t film_ld;
    int64_t film_off;
    int remap_in, remap_out;   /* F16/F32: out_row = (row/remap_in)*remap_out + row%remap_in; 0 = identity */
    int up_h, up_w, up_cout;   /* UNPATCH: coarse grid and output channels */
    void* out16;               /* RESID_LN: fp16 [M, ldo] copy of out */
    int64_t* ln_stat;          /* RESID_LN (accumulated, caller zeroes) / F16_LN (read): [M][2] = (sum x * 2^20, sum x^2 * 2^16)
                                  over the ln_c columns of a row, fixed point (integer atomics: order-independent) */
    const float* ln_wsum;      /* F16_LN: [N] row sums of the fp16 weight matrix */
    int ln_c;                  /* F16_LN: number of columns the statistics cover (= K of this GEMM) */
    const float* ln_shift;     /* RESID_LN / F16_LN: fp32 [M] per-row shift the producer subtracted, or NULL (= 0) */
    float* ln_mean_out;        /* F16_LN: fp32 [M] true row mean (shift + mean of the shifted row), or NULL */
    const void* a_scale;       /* RESID / RESID_LN: fp16 [M / rows_per_sample, a_scale_ld] per-(sample, k) factors multiplied into
                                  the A operand on its way to the tensor core (GlobalResponseNorm folded into the GEMM that
                                  consumes it: A'[m,k] = A[m,k] * a_scale[m / rows_per_sample, k]), or NULL.  Needs M > 128,
                                  K % 64 == 0 and rows_per_sample dividing 128 (>= 16) or a multiple of 128 */
    int64_t a_scale_ld;
} pb200_gemm_epilogue;

int pb200_gemm_f16(const void* a, int64_t lda, const void* w, int64_t ldw, int64_t m, int64_t n, int64_t k,
                   const pb200_gemm_epilogue* epi, void* stream);
/* Host-side tile plan pb200_gemm_f16 would use for an [m,k] x [n,k]^T problem on `sm_count` multiprocessors (0 = the
 * current device, or 148 without one): BLOCK_N, whether the 2-SM (cta_group::2) kernel runs it, and the column width
 * of the narrow tail tiles (0 = none).  Pure arithmetic, no device work. */
int pb200_gemm_plan(int64_t m, int64_t n, int64_t k, int sm_count, int* block_n, int* two_sm, int* tail_block_n);

/* ------------------------------------------------------------------------------------------
 * Block-level kernels: what the reference's building-block modules (ref/src/modules.py:7-106)
 * run when they are called on their own, outside a Paella (inside one the model executor below
 * launches the same kernels from its plan).  Activations are channels-last rows [batch*positions, c]
 * unless named NCHW; "16" pointers are fp16.
 * ------------------------------------------------------------------------------------------ */
/* nn.LayerNorm over the last dim: y = (x-mean)/sqrt(var+eps) [*weight + bias]; exactly one of out32/out16.
 * LayerNorm2d = this between the two layout changes below   [ref/src/modules.py:22-27] */
int pb200_layernorm(const float* x, int64_t rows, int c, float eps, const float* weight, const float* bias, float* out32,
                    void* out16, void* stream);
/* x.permute(0,2,3,1) / x.permute(0,3,1,2) on fp32 [batch, c, hw] <-> [batch, hw, c]   [ref/src/modules.py:27,58-61] */
int pb200_nchw_to_nhwc(const float* in, int batch, int c, int hw, float* out, void* stream);
int pb200_nhwc_to_nchw(const float* in, int batch, int c, int hw, float* out, void* stream);
/* fp32 -> fp16 GEMM operand, optionally through SiLU (AttnBlock.kv_mapper[0])   [ref/src/modules.py:71-74] */
int pb200_cast_f16(const float* x, int64_t n, int silu, void* out16, void* stream);
/* ResBlock front: depthwise k x k conv over cat[x, skip] (groups = c, zero padding k/2) + bias + LayerNorm2d(no
 * affine, eps 1e-6) -> fp16 [batch*h*w, c].  x fp32 NHWC [batch,h,w,c]; skip NHWC [batch,h,w,c] or NULL;
 * w_packed fp32 [k*k][per][c] (per = 2 with skip: concatenated input channels 2g, 2g+1 feed output g)
 * [ref/src/modules.py:46-47,57-58] */
int pb200_dwconv_ln(const float* x, const float* skip, const float* w_packed, const float* bias, int batch, int h, int w,
                    int c, int k, void* out16, void* stream);
/* GlobalResponseNorm in place on the fp16 hidden [batch, rows_per_sample, n] of a PB200_EPI_GELU_F16 GEMM whose
 * epilogue accumulated sqsum (2^-24 fixed point); zeroes zero_per_sample entries per sample of sqsum_next;
 * scale_scratch = caller-owned fp32 [batch, n] (the per-sample multipliers 1 + gamma * Nx, written then read)
 * [ref/src/modules.py:30-40] */
int pb200_grn_f16(void* h16, int batch, int rows_per_sample, int n, const uint64_t* sqsum, uint64_t* sqsum_next,
                  int zero_per_sample, const float* gamma, const float* beta, float* scale_scratch, void* stream);
/* GlobalResponseNorm.forward on an fp32 NHWC tensor [batch, rows_per_sample, n]; stat = scratch [batch, n]
 * [ref/src/modules.py:37-40] */
int pb200_grn_f32(const float* x, int batch, int rows_per_sample, int n, const float* gamma, const float* beta, float* stat,
                  float* out, void* stream);
/* TimestepBlock: x[r, j] = x*(1 + film[r/rows_per_sample, film_off + j]) + film[.., film_off + n + j] in place
 * [ref/src/modules.py:104-106] */
int pb200_film_apply(float* x, int64_t rows, int n, int rows_per_sample, const float* film, int64_t film_ld, int64_t film_off,
                     void* stream);
/* Attention core of nn.MultiheadAttention / CustomMultiheadAttention after the in-projection:
 * qkv16 [batch*positions, 3*embed] = q | k_self | v_self, ckv16 [batch, s_max, 2*embed] = k_cond | v_cond
 * (kv_len[batch] valid rows, NULL = s_max); keys = [self ; cond] if self_attn else cond; optional post-softmax
 * attn_weights on the last n_weights keys of samples [0, weighted_batch); out16 [batch*positions, embed]
 * [ref/src/modules.py:12-19, ref/utils/alter_attention.py:19-36] */
int pb200_attention(const void* qkv16, const void* ckv16, const int* kv_len, void* out16, int batch, int positions, int s_max,
                    int embed, int nhead, int self_attn, const float* attn_weights, int n_weights, int weighted_batch,
                    void* stream);

/* ------------------------------------------------------------------------------------------
 * Denoiser (ref/src/modules.py:109-283, ref/utils/modules.py) as an opaque handle.
 * ------------------------------------------------------------------------------------------ */
#define PB200_MAX_LEVELS 4

typedef struct pb200_paella_config {   /* constructor kwargs of Paella, ref/src/modules.py:110-112 */
    int c_in, c_out, num_labels, c_r, patch_size, c_cond;
    int n_levels;
    int c_hidden[PB200_MAX_LEVELS];
    int nhead[PB200_MAX_LEVELS];
    int blocks[PB200_MAX_LEVELS];
    char level_config[PB200_MAX_LEVELS][8];   /* e.g. "CT", "CTA" */
    int clip_embd, byt5_embd, clip_seq_len, kernel_size, self_attn;
} pb200_paella_config;

typedef struct pb200_paella pb200_paella;     /* opaque */

/* Build the layer plan (host only).  Weights live in a caller-owned device blob of
 * pb200_paella_weight_bytes() bytes, filled by pb200_paella_load_param(); the blob is
 * position-independent, so one rank can fill it and broadcast it (NCCL) to the others. */
int pb200_paella_create(const pb200_paella_config* cfg, pb200_paella** out);
void pb200_paella_destroy(pb200_paella* m);
int64_t pb200_paella_weight_bytes(const pb200_paella* m);
int pb200_paella_bind_weights(pb200_paella* m, void* weight_blob);
/* number / names of the state-dict entries the plan consumes (reference key names). */
int pb200_paella_num_params(const pb200_paella* m);
const char* pb200_paella_param_name(const pb200_paella* m, int i);
int64_t pb200_paella_param_numel(const pb200_paella* m, int i);
/* convert one reference-layout fp32 parameter (device pointer) into the packed blob. */
int pb200_paella_load_param(pb200_paella* m, const char* name, const float* src, int64_t numel, void* stream);

/* conditioning for `batch` samples: byt5 fp32 [B, L, byt5_embd]; clip / clip_image fp32
 * [B, clip_embd] or NULL; n_clip_image images (list-valued clip_image, ref/utils/modules.py:228-235,
 * laid out [n_img, B, clip_embd]).  Sequence length S = L + clip_seq_len*(has_clip + n_clip_image). */
typedef struct pb200_cond {
    const float* byt5; int byt5_len;
    const float* clip;
    const float* clip_image; int n_clip_image;
} pb200_cond;

/* scratch sizes for a forward over `batch_total` samples on an H x W token grid whose
 * conditioning sequences are at most `s_max` long. */
int64_t pb200_paella_workspace_bytes(const pb200_paella* m, int batch_total, int h, int w, int s_max);
/* bytes of the per-call conditioning cache (c_embed + every AttnBlock's cond K/V). */
int64_t pb200_paella_cond_cache_bytes(const pb200_paella* m, int batch_total, int s_max);

/* gen_c_embeddings + every AttnBlock's kv_mapper and K/V projection of the conditioning rows
 * (x- and t-independent) for samples [batch_offset, batch_offset + batch) of the cache. */
int pb200_paella_prepare_cond(pb200_paella* m, const pb200_cond* cond, int batch, int batch_offset, int batch_total,
                              int s_max, void* cond_cache, void* workspace, int64_t workspace_bytes, void* stream);

/* gen_r_embedding: r fp32 [B] -> fp32 [B, c_r]   (ref/src/modules.py:212-221) */
int pb200_paella_r_embedding(const float* r, int batch, int c_r, float* out, void* stream);
/* gen_c_embeddings: -> fp32 [B, S, c_cond], S = byt5_len + clip_seq_len*(has_clip + n_clip_image)   (ref/src/modules.py:223-232) */
int pb200_paella_c_embeddings(pb200_paella* m, const pb200_cond* cond, int batch, float* out, void* workspace,
                              int64_t workspace_bytes, void* stream);

/* Paella.forward up to out_mapper's LayerNorm: tokens int64 [Bt,H,W], r fp32 [Bt] ->
 * features fp32 [Bt*H*W, c_out] (rows (b,y,x)).  attn_weights fp32 [n_attn_weights] or NULL scales
 * the last n key columns after the softmax for samples [0, attn_weights_batch)
 * (ref/utils/alter_attention.py:23-34; the notebook passes it on the conditional forward only).
 * cond_cache was prepared for cache_slots sample slots (the batch_total of pb200_paella_prepare_cond); kv_slot int32
 * [batch_total] names the slot each sample attends to (NULL: slot i for sample i, cache_slots == batch_total) -- samples
 * with identical conditioning, e.g. the unconditional half of a CFG batch, share one slot and its K/V is read once.
 * cfg_pairs = 1: the classifier-free-guidance batch of ref/src/utils.py:42-45 -- tokens [Bt/2,H,W] and r [Bt/2] are
 * given once, sample i + Bt/2 is sample i under the unconditional rows of the conditioning cache.  The blocks before
 * the first AttnBlock do not see the conditioning and are evaluated once per pair (identical arithmetic). */
int pb200_paella_features(pb200_paella* m, const int64_t* tokens, const float* r, int batch_total, int cfg_pairs, int h, int w,
                          const void* cond_cache, int cache_slots, const int* kv_slot, int s_max, const float* attn_weights,
                          int n_attn_weights,
                          int attn_weights_batch, float* features, void* workspace, int64_t workspace_bytes,
                          void* stream);

/* out_mapper on features -> logits fp32 NCHW [B, num_labels, H*W]   (ref/src/modules.py:184-187,274) */
int pb200_paella_logits(pb200_paella* m, const float* features, int batch, int hw, float* logits_nchw,
                        void* workspace, int64_t workspace_bytes, void* stream);

/* Fused out_mapper + CFG + temperature + multinomial (ref/src/utils.py:44-50): logits never reach HBM.
 *   features: fp32 [(2B or B)*HW, c_out]: conditional rows first, then unconditional rows (if cfg_on).
 *   tokens_out int64 [B*HW].  Gumbel-max in the log domain on torch's Philox stream:
 *   argmax_k( l_k/T - log q_k ), q_k the same Exp(1) draw torch.multinomial would use. */
int pb200_paella_sample_tokens(pb200_paella* m, const float* features, int batch, int hw, int cfg_on, double cfg,
                               double temperature, uint64_t seed, uint64_t offset, int64_t* tokens_out,
                               void* workspace, int64_t workspace_bytes, void* stream);
/* Masked (inpainting) form of pb200_paella_sample_tokens: tokens_inout int64 [B*HW] holds the known tokens on entry;
 * rows with mask[row] != 0 (uint8 [B*HW], 1 = regenerate) receive exactly the token pb200_paella_sample_tokens would
 * write there for the same (seed, offset); rows with mask 0 are not written.  Work scales with the rows to regenerate. */
int pb200_paella_sample_tokens_masked(pb200_paella* m, const float* features, int batch, int hw, int cfg_on, double cfg,
                                      double temperature, uint64_t seed, uint64_t offset, const uint8_t* mask,
                                      int64_t* tokens_inout, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * VQGAN (ref/src/vqgan.py:45-107).
 * ------------------------------------------------------------------------------------------ */
typedef struct pb200_vqgan_config {   /* VQModel kwargs, ref/src/vqgan.py:46-47 */
    int levels, bottleneck_blocks, c_hidden, c_latent, codebook_size;
    float scale_factor;
} pb200_vqgan_config;

typedef struct pb200_vqgan pb200_vqgan;

int pb200_vqgan_create(const pb200_vqgan_config* cfg, pb200_vqgan** out);
void pb200_vqgan_destroy(pb200_vqgan* m);
int64_t pb200_vqgan_weight_bytes(const pb200_vqgan* m);
int pb200_vqgan_bind_weights(pb200_vqgan* m, void* weight_blob);
int pb200_vqgan_num_params(const pb200_vqgan* m);
const char* pb200_vqgan_param_name(const pb200_vqgan* m, int i);
int64_t pb200_vqgan_param_numel(const pb200_vqgan* m, int i);
int pb200_vqgan_load_param(pb200_vqgan* m, const char* name, const float* src, int64_t numel, void* stream);
int64_t pb200_vqgan_workspace_bytes(const pb200_vqgan* m, int batch, int img_h, int img_w);

/* VQModel.encode: img fp32 NCHW [B,3,H,W] -> latents fp32 NCHW [B,c_latent,H/4,W/4] (pre-quantisation,
 * NOT divided by scale_factor), quantised latents (same shape) and indices int64 [B,H/4,W/4]. */
int pb200_vqgan_encode(pb200_vqgan* m, const float* img, int batch, int img_h, int img_w, float* latents_nchw,
                       float* quantised_nchw, int64_t* indices, void* workspace, int64_t workspace_bytes,
                       void* stream);
/* VQModel.decode_indices (indices != NULL) or VQModel.decode on NCHW latents already multiplied by
 * scale_factor (latents_nchw != NULL) -> img fp32 NCHW [B,3,4h,4w]. */
int pb200_vqgan_decode(pb200_vqgan* m, const int64_t* indices, const float* latents_nchw, int batch, int h, int w,
                       float* img, void* workspace, int64_t workspace_bytes, void* stream);

/* One codec ResBlock on its own (ref/src/vqgan.py:36-42) -- what `vqgan.ResBlock.forward` runs outside a VQModel; inside
 * one, encode/decode run the same kernels from the plan.  x_nhwc fp32 [B,h,w,c] is updated in place; dw_w9 = the depthwise
 * kernel as [9][c] fp32 (tap-major), w1 [4c,c] / w2 [c,4c] fp16 row-major, gammas_host = the 6 scalars (HOST memory). */
int64_t pb200_vqgan_resblock_workspace_bytes(int batch, int h, int w, int c);
int pb200_vqgan_resblock(float* x_nhwc, int batch, int h, int w, int c, const float* dw_w9, const float* dw_bias,
                         const void* w1_f16, const float* b1, const void* w2_f16, const float* b2, const float* gammas_host,
                         void* workspace, int64_t workspace_bytes, void* stream);

/* Experiment kept for the record (measured slower than the two GEMMs, see csrc/vq_mlp.cu): the ResBlock MLP in one tcgen05
 * kernel, x[rows, c] += alpha * (GELU(a16 W1^T + b1) W2^T + b2) with the 4c-wide hidden kept in TMEM / shared memory.
 * c in {384, 192}, rows >= 256.  The codec uses it only with PB200_VQ_MLP_FUSED=1. */
int pb200_vq_mlp_fused(const void* a16, int64_t rows, int c, const void* w1_f16, const float* b1, const void* w2_f16,
                       const float* b2, float* x, float alpha, void* stream);

/* Output forms of the decoder's last kernel (out_block: 1x1 conv + PixelShuffle, ref/src/vqgan.py:86-89), fused with what
 * the reference's callers do next (ref/src_distributed/train.py:168-171 `decode_indices(x).clamp(0, 1)`, then
 * torchvision.utils.save_image's `mul(255).add_(0.5).clamp_(0, 255).to(uint8)` on an HWC view):
 *   PB200_IMG_F32_NCHW          fp32 [B,3,4h,4w], unclamped               == pb200_vqgan_decode
 *   PB200_IMG_F32_NCHW_CLAMP01  fp32 [B,3,4h,4w], clamp(0,1)
 *   PB200_IMG_U8_NHWC           uint8 [B,4h,4w,3] = trunc(clamp(v,0,1)*255 + 0.5)   */
enum { PB200_IMG_F32_NCHW = 0, PB200_IMG_F32_NCHW_CLAMP01 = 1, PB200_IMG_U8_NHWC = 2 };
int pb200_vqgan_decode_ex(pb200_vqgan* m, const int64_t* indices, const float* latents_nchw, int batch, int h, int w,
                          void* img, int img_mode, void* workspace, int64_t workspace_bytes, void* stream);
/* decode_ex of indices int64 [B,h,w] composited into an original image: where pixel_mask (uint8 [B,4h,4w]) is 0 the
 * output pixel is orig_img (fp32 NCHW [B,3,4h,4w]) put through the same img_mode conversion, elsewhere the decoded
 * pixel.  The compositing happens in the decoder's last kernel (inpainting with the untouched pixels pasted back). */
int pb200_vqgan_decode_composite(pb200_vqgan* m, const int64_t* indices, int batch, int h, int w, const float* orig_img,
                                 const uint8_t* pixel_mask, void* img, int img_mode, void* workspace,
                                 int64_t workspace_bytes, void* stream);

/* Re-read the host-mirrored scalars (the six ResBlock gammas, kernel arguments) from the bound weight blob.  Needed when
 * the blob was filled by anything other than pb200_vqgan_load_param on this handle (NCCL broadcast, a packed file,
 * cudaMemcpy).  bind_weights marks them stale and encode/decode refresh lazily (one stream synchronisation), so calling
 * this is only required when the blob CONTENT changes under an already-bound pointer.  Synchronises `stream`. */
int pb200_vqgan_sync_params(pb200_vqgan* m, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PAELLA_B200_H */
