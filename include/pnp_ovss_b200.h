/*
 * pnp_ovss_b200.h -- C ABI of libpnp_ovss_b200.so: the PnP-OVSS mask-extraction hot path as sm_100a CUDA.
 *
 * The reference (letitiabanana/PnP-OVSS) is pure Python and has no FFI of its own; each entry point below
 * names the reference lines whose arithmetic it replaces.  Shorthands:
 *   DRV  = PnP_OVSS_0514_updated_segmentation.py        DRVC = PnP_OVSS_0514_updated_segmentation_coco.py
 *   BITM = Files to replace for BLIP/blip_image_text_matching.py     MED = Files to replace for BLIP/med.py
 *
 * Conventions (every function):
 *   - every pointer is a DEVICE pointer on the current CUDA device unless the parameter is documented "host";
 *   - the caller owns every buffer; nothing is allocated, freed or cached inside the library;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*) and the call returns immediately;
 *   - return value: PNP_OK (0) or a negative code; no exception crosses the boundary;
 *   - tensors are dense, row-major, fp32 unless stated; shapes are written [outer, ..., inner];
 *   - one process per GPU (DRV:1439 mp.spawn).  Every entry point except pnp_profile_* may be called from several host threads
 *     at once, each on its own stream (pipeline.py issues the buckets of a ragged batch that way).  Process-global state is limited
 *     to: the in-situ profiler (pnp_profile_*, off by default, single-threaded use only) and the per-kernel "allow > 48 KB of
 *     dynamic shared memory" function attribute (granted once per kernel at the device maximum, under a mutex).  The library reads
 *     no environment variables.  No data is cached between calls.
 *   - exception to "returns immediately": pnp_lattice_finish synchronises the stream (it reads the vertex count back).
 */
#ifndef PNP_OVSS_B200_H
#define PNP_OVSS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *pnp_stream_t; /* cudaStream_t */

#define PNP_OK 0
#define PNP_ERR_INVALID_ARGUMENT (-1) /* bad shape / null pointer / unsupported size */
#define PNP_ERR_WORKSPACE (-2)        /* workspace smaller than the *_workspace_bytes() answer */
#define PNP_ERR_CUDA_BASE (-1000)     /* -(1000 + cudaError_t) for launch failures */

#define PNP_ABI_VERSION 1

int pnp_abi_version(void);
/* Static string for a return code (never NULL). */
const char *pnp_error_string(int code);
/* Compute capability the kernels were compiled for (100 for sm_100a). */
int pnp_compiled_sm(void);

/* ------------------------------------------------------------------------------------------------------
 * (a) block-8 cross-attention softmax, fused with capture of the attention map and of its gradient
 *     replaces MED:267-283 (scores/sqrt(64) + mask -> nn.Softmax -> save_attention_map + register_hook)
 * ---------------------------------------------------------------------------------------------------- */

/* probs[b,h,t,:] = softmax_k(scores[b,h,t,:] * scale + key_mask[b,:]).
 * scores, probs [B,heads,T,K]; key_mask [B,K] additive (the extended encoder_attention_mask of MED:269-271)
 * or NULL.  probs may alias scores. */
int pnp_xattn_softmax_fwd(const float *scores, const float *key_mask, float *probs, int B, int heads, int T,
                          int K, float scale, pnp_stream_t stream);

/* Backward of the above fused with the GradCAM product of BITM:415-433 for ONE head.
 *   dscores = probs * (dprobs - sum_k(probs*dprobs)) * scale                (autograd of MED:267-274)
 *   gradcam[b,t-1,p] = probs[b,head,t,p+1] * max(dprobs[b,head,t,p+1],0) * token_mask[b,t]   for t >= 1
 * probs, dprobs, dscores [B,heads,T,K]; token_mask int64 [B,token_mask_stride] (the max_length=500 padded
 * attention_mask, BITM:415-416), token_mask_stride >= T; gradcam [B,T-1,K-1] (= [B,T-1,P,P]).
 * dscores == NULL: only the GradCAM of `head` is produced (frozen-weights mode, SURVEY 7.4).
 * gradcam == NULL: plain softmax backward.  dscores may alias dprobs. */
int pnp_xattn_softmax_bwd_gradcam(const float *probs, const float *dprobs, float *dscores,
                                  const int64_t *token_mask, int token_mask_stride, float *gradcam, int B,
                                  int heads, int T, int K, float scale, int head, pnp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (b) token -> class merge; replaces DRV:810-853 (Mean_over_filtered_label_tokens) and its twin DRV:656-701
 * ---------------------------------------------------------------------------------------------------- */

/* class_maps[b,c,:] = (sum_{i<seg_len[b,c]} gradcam[b, row_offset + seg_start[b,c] + i, :]) / seg_div[b,c]
 * summed in token order, fp32.  seg_len == 0 -> zeros.  The host builds (seg_start, seg_len, seg_div) from
 * the WordPiece strings exactly as the reference loop walks them (seg_div = word length, or 1 where the
 * reference never divides: single-piece words and a split word in last position).
 * gradcam [B,Tm,PP] (Tm = T-1 rows: ENC row already dropped), row_offset = 3 ("a picture of");
 * seg_* [B,C] (int32 / int32 / fp32); class_maps [B,C,PP]. */
int pnp_token_merge(const float *gradcam, const int32_t *seg_start, const int32_t *seg_len, const float *seg_div,
                    float *class_maps, int B, int Tm, int PP, int C, int row_offset, pnp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (c) one round of Salience DropOut; replaces DRV:589-603 (pixel zeroing), DRV:623-635 (cell zeroing),
 *     DRV:638-647 (top-save_len selection) and DRV:716-721 (accumulation, round 0 counted twice)
 * ---------------------------------------------------------------------------------------------------- */

/* For every image b (one CTA each):
 *   pred = gradcam[b] with the n_prev already-chosen cells zeroed            -> ensemble_r (optional)
 *   agg  = round == 0 ? pred + pred : agg + pred                              (optional)
 *   score[p] = sum_{t in [row_lo,row_hi)} gradcam[b,t,p] (sequential fp32), chosen cells := 0
 *   new = the save_len largest scores (ties: larger index ranks higher, = a stable ascending argsort's tail)
 *   chosen[b, n_prev : n_prev+save_len] = new (ascending score order)
 *   imgs[b,:,16r:16r+16,16c:16c+16] = 0 and norm_imgs[b,16r:16r+16,16c:16c+16,:] = 0 for the new cells
 * gradcam, ensemble_r, agg [B,Tm,P*P]; chosen int32 [B,chosen_stride]; imgs [B,3,S,S] or NULL; norm_imgs
 * [B,S,S,3] or NULL; S = P*patch.  Requires P*P <= 1024 and save_len <= 32. */
int pnp_salience_dropout_round(const float *gradcam, float *ensemble_r, float *agg, int32_t *chosen,
                               int chosen_stride, int n_prev, float *imgs, float *norm_imgs, int B, int Tm,
                               int P, int patch, int row_lo, int row_hi, int save_len, int round,
                               pnp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (d) threshold + bilinear upsample (+ Scale_0_1) + background channel; replaces DRV:348-380 / DRV:424-455,
 *     DRV:1078-1094 (Scale_0_1), DRVC:512-541
 * ---------------------------------------------------------------------------------------------------- */

size_t pnp_threshold_upsample_workspace_bytes(int B, int C, int P);
/* class_maps [B,C,P,P] -> out [B,C',H,W] with C' = C + with_background (background first).
 * Per class: keep x where (x-min)/(max-min) >= threshold (NaN compares false), bilinear align_corners=True
 * to HxW, optional per-channel min-max rescale, background = (max over classes == 0). */
int pnp_threshold_upsample(const float *class_maps, float *out, void *workspace, size_t workspace_bytes, int B,
                           int C, int P, int H, int W, float threshold, int rescale, int with_background,
                           pnp_stream_t stream);

/* Gaussian blur + min-max; replaces DRV:1149-1153 (scipy.ndimage.gaussian_filter, mode='reflect',
 * truncate=4, axis 0 then axis 1, float32 between passes) called per channel from DRV:1005-1011.
 * in, out [n_maps,H,W] (out may NOT alias in); minmax [n_maps,2] receives (min, max) of each blurred map
 * (NaN if the map holds a NaN).  normalize != 0 additionally rewrites out = (out-min)/(max-min) in place;
 * normalize == 0 leaves that to the consumer (pnp_crf_unary_from_maps folds it in). */
size_t pnp_gaussian_blur_workspace_bytes(int n_maps, int H, int W, double sigma);
int pnp_gaussian_blur(const float *in, float *out, float *minmax, void *workspace, size_t workspace_bytes,
                      int n_maps, int H, int W, double sigma, int normalize, pnp_stream_t stream);

/* Fused low-rank form of the whole (d) group for a batch whose maps are blurred (--postprocess blur / blur+crf):
 * threshold (DRV:425-433) -> bilinear upsample (DRV:435-437) -> [Scale_0_1] -> background channel (DRV:446-455) ->
 * Gaussian blur + min-max of every channel (DRV:1005-1011, 1149-1153) -> one of
 *   unary  [B,N,Cp]   -log(clip(softmax_c(maps), 1e-5, 1)), pixel-major, Cp = 4*ceil(C'/4), padding 0 (DRV:1057-1063)
 *   labels [B,N]      argmax_c(maps), first maximum, NaN counts as maximum (blur-only mode, DRV:1018-1025)
 *   maps_out [B,C',H,W]  the normalised blurred maps themselves (what `blurring` returns per channel)
 * (any subset; at least one).  minmax_out (optional) [B*C',2] receives (min, max) of every blurred channel.
 * Upsample and blur are linear and separable, so a class channel is A_y m A_x^T with A = G_sigma U (H x P, W x P): no
 * full-resolution input or intermediate exists; Scale_0_1 is affine per channel and cancels in the min-max that follows
 * the blur, so `rescale` only enters the background test.  The background indicator is evaluated at full resolution with
 * the arithmetic of pnp_threshold_upsample and blurred tap by tap like pnp_gaussian_blur.  class_maps [B,C,P,P], P <= 32. */
size_t pnp_lowrank_blur_workspace_bytes(int B, int C, int P, int H, int W, double sigma, int with_background);
int pnp_lowrank_blur_unary(const float *class_maps, float *unary, int32_t *labels, float *maps_out, float *minmax_out,
                           void *workspace, size_t workspace_bytes, int B, int C, int P, int H, int W, float threshold,
                           int rescale, int with_background, double sigma, pnp_stream_t stream);
/* The same over a batch whose images have DIFFERENT class counts (DRV:340-347: every image brings its own caption classes):
 * class_maps is padded to C classes, image b really has n_classes[b] <= C of them (device int32 [B]; NULL = all C).  The channels
 * an image does not have are dead: value -inf in maps_out, never the argmax, and unary +inf -- as are the padding channels up to
 * Cp -- so a mean-field inference over all Cp channels (pnp_crf_inference with C = Cp) keeps their Q at exactly 0 and every
 * real channel gets bit for bit what a per-image run with the exact class count gives.  Scale_0_1's one-class quirk
 * (DRV:1079-1080) is applied per image. */
int pnp_lowrank_blur_unary_padded(const float *class_maps, const int32_t *n_classes, float *unary, int32_t *labels,
                                  float *maps_out, float *minmax_out, void *workspace, size_t workspace_bytes, int B, int C,
                                  int P, int H, int W, float threshold, int rescale, int with_background, double sigma,
                                  pnp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (e) dense-CRF mean-field inference on permutohedral lattices; replaces the pydensecrf calls of
 *     DRV:1030-1074 (DenseCRF2D / addPairwiseGaussian / addPairwiseBilateral / inference)
 * ---------------------------------------------------------------------------------------------------- */

/* A lattice lives in caller-owned device memory; this host struct just records where.  `shared` lattices
 * (spatial: features depend on (H,W) only) hold ONE image's lattice that is applied to every image of a
 * batch; non-shared ones (bilateral) hold n_images independent lattices with globally numbered vertices. */
typedef struct pnp_lattice {
    int d;             /* feature dimension: 2 (x,y) or 5 (x,y,r,g,b) */
    int n_images;      /* images embedded (1 when shared) */
    int n_pixels;      /* pixels per image, H*W */
    int shared;        /* 1: one lattice reused by every image of a batch */
    int n_vertices;    /* M: filled by pnp_lattice_finish (host copy of the device count) */
    int max_row;       /* longest CSR row, filled by pnp_lattice_finish (statistics) */
    int vertex_stride; /* allocated vertex capacity = n_images*n_pixels*(d+1) */
    int width;         /* image width W (n_pixels = H*W), filled by pnp_lattice_build */
    /* device arrays */
    int32_t *offset;   /* [n_images*n_pixels, d+1] vertex id, 0-based, numbered in first-touch order */
    float *bary;       /* [n_images*n_pixels, d+1] barycentric weights */
    int32_t *nbr;      /* [d+1, vertex_stride, 2] blur neighbours +1 (0 = none) */
    int32_t *row_ptr;  /* [vertex_stride+1] CSR over vertices (entries of vertex v: row_ptr[v]..row_ptr[v+1]) */
    int32_t *csr_pix;  /* [n_images*n_pixels*(d+1)] lattice pixel of each entry, ascending inside a row */
    float *csr_w;      /* [n_images*n_pixels*(d+1)] barycentric weight of each entry */
    float *csr_norm;   /* [n_images*n_pixels*(d+1)] norm[csr_pix] in CSR order (sequential read instead of a gather) */
    float *norm;       /* [n_images*n_pixels] 1/sqrt(K 1 + 1e-20) (NORMALIZE_SYMMETRIC) */
    int32_t *counters; /* [8] device: 0 = M, 1 = key-range overflow flag, 2 = longest row */
} pnp_lattice;

/* Bytes of persistent storage a lattice needs, and of scratch needed while building it. */
size_t pnp_lattice_storage_bytes(int d, int n_images, int n_pixels);
size_t pnp_lattice_build_workspace_bytes(int d, int n_images, int n_pixels);
/* Carve `storage` (device, >= pnp_lattice_storage_bytes, 256-byte aligned) into the arrays of *lat (host). */
int pnp_lattice_init(pnp_lattice *lat, void *storage, size_t storage_bytes, int d, int n_images, int n_pixels,
                     int shared);
/* Enqueue the whole build: embed pixels (elevate, round, rank, barycentric), hash-insert the d+1 simplex
 * vertices per pixel with warp-level de-duplication, number vertices in first-touch order (identical to the
 * insertion order of densecrf's sequential hash table), blur-neighbour lookup, CSR by vertex (rows sorted by
 * pixel so the splat sums in the same order as the sequential reference), and the symmetric normalisation.
 * Features: (x/sx, y/sy) and, when rgb != NULL (uint8 [n_images,H,W,3]), (r/sr, g/sg, b/sb).
 * d must be 2 (rgb == NULL) or 5 (rgb != NULL). */
int pnp_lattice_build(pnp_lattice *lat, const uint8_t *rgb, int H, int W, float sx, float sy, float sr,
                      float sg, float sb, void *workspace, size_t workspace_bytes, pnp_stream_t stream);
/* Synchronises `stream`, reads the counters back into lat->n_vertices / max_row.  Returns
 * PNP_ERR_INVALID_ARGUMENT if a lattice coordinate did not fit the packed hash key. */
int pnp_lattice_finish(pnp_lattice *lat, pnp_stream_t stream);

/* Unary from class maps: p = softmax_c((maps[c]-min_c)/(max_c-min_c)) (DRV:1057 after DRV:1151-1152),
 * U = -log(clip(p,1e-5,1)) (pydensecrf.utils.unary_from_softmax).  maps [B,C,N] channel-major;
 * minmax [B*C,2] or NULL (maps used as they are); unary [B,N,Cp] pixel-major, Cp = 4*ceil(C/4), padding
 * channels 0. */
size_t pnp_crf_unary_workspace_bytes(int B, int C, int N); /* 0 for C <= 32 */
int pnp_crf_unary_from_maps(const float *maps, const float *minmax, float *unary, void *workspace,
                            size_t workspace_bytes, int B, int C, int N, pnp_stream_t stream);
/* Layout helpers for the pydensecrf-shaped API: [B,C,N] <-> [B,N,Cp] (padding channels written as 0). */
int pnp_crf_pack_cn_to_nc(const float *src_cn, float *dst_nc, int B, int C, int N, pnp_stream_t stream);
int pnp_crf_unpack_nc_to_cn(const float *src_nc, float *dst_cn, int B, int C, int N, pnp_stream_t stream);

/* Scratch for filtering / inference with B images of Cp channels over the given (finished) lattices:
 * two vertex-value buffers per lattice. */
size_t pnp_crf_scratch_bytes(const pnp_lattice *const *lattices, int n_kernels, int B, int Cp);

/* y = K x (normalized == 0) or y = norm . K (norm . x) (normalized != 0) for one lattice; x, y [B,N,Cp],
 * y may alias x.  Test/diagnostic entry point; the same kernels are the building blocks of the inference. */
int pnp_crf_filter(const pnp_lattice *lat, const float *x, float *y, void *scratch, size_t scratch_bytes, int B,
                   int Cp, int normalized, pnp_stream_t stream);

/* Mean-field inference (DenseCRF::inference with Potts compatibilities):
 *   Q = softmax(-U); n_iter times: Q = softmax(-U + sum_k weights[k] * K_k Q).
 * unary, Q [B,N,Cp]; labels (optional, int32 [B,N]) = first argmax over the C real channels of the final Q.
 * lattices/weights: host arrays of n_kernels (<= 4) entries. */
int pnp_crf_inference(const pnp_lattice *const *lattices, const float *weights, int n_kernels,
                      const float *unary, float *Q, void *scratch, size_t scratch_bytes, int32_t *labels, int B,
                      int C, int Cp, int n_iter, pnp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (f) argmax + relabel + confusion matrix; replaces DRV:387 / DRV:1073 (argmax), DRV:390-399 / 468-480
 *     (sequential relabel, passed here as its composed LUT), DRV:1106-1112 (_fast_hist)
 * ---------------------------------------------------------------------------------------------------- */

/* labels[b,p] = first argmax_c maps[b,c,p] (NaN counts as maximum, like torch/numpy). maps [B,C,N]. */
int pnp_argmax_channels(const float *maps, int32_t *labels, int B, int C, int N, pnp_stream_t stream);

/* hist[n*gt + lut[b,label]] += 1 for every pixel with 0 <= gt < n_class (gt is float32 like the reference's
 * ground truth, truncated toward zero as .astype(int) does).  labels int32 [B,N]; lut int32 [B,lut_stride]
 * (NULL: identity); pred_out (optional) float32 [B,N] receives the relabelled map; hist int64 [n,n],
 * ACCUMULATED into (zero it first).  Pixels whose relabelled id is outside [0,n) are counted in
 * *bad_count (device int32, optional) instead. */
int pnp_confusion_accumulate(const int32_t *labels, const float *gt, const int32_t *lut, int lut_stride,
                             float *pred_out, int64_t *hist, int32_t *bad_count, int B, int N, int n_class,
                             pnp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (f)1 model pass (SURVEY 8f.1; BITM:386-404 drives VIT:93-119 / MED:201-228): operand preparation for
 *      fp32-grade GEMMs on the TF32 tensor cores.  The dense contractions themselves stay torch's (cuBLAS);
 *      y = x W^T runs as ONE TF32 GEMM of depth 3K on [x_hi | x_lo | x_hi] x [W_hi | W_hi | W_lo]^T, where
 *      hi = the operand rounded to TF32 (10 explicit mantissa bits) and lo = operand - hi (exact in fp32).
 * ---------------------------------------------------------------------------------------------------- */

/* out3[m, 0:K] = hi(x[m,:]), out3[m, K:2K] = x - hi, out3[m, 2K:3K] = hi.  x [M,K], out3 [M,3K]; K % 4 == 0,
 * 16-byte aligned pointers. */
int pnp_tf32_split3(const float *x, float *out3, long long M, int K, pnp_stream_t stream);
/* Same split of GELU(x + bias) (exact erf form, VIT:35-40 Mlp / nn.GELU); bias [K] or NULL. */
int pnp_gelu_tf32_split3(const float *x, const float *bias, float *out3, long long M, int K,
                         pnp_stream_t stream);
/* y = LayerNorm(x') * gamma + beta over the last dimension (biased variance, eps inside the sqrt: nn.LayerNorm
 * of VIT:70-71), where x' = x, or x + residual (+ residual_bias [K]) when residual != NULL -- in which case
 * x' is also written to x_out when x_out != NULL (x_out may alias x).  y goes to out3 as the [hi | lo | hi]
 * split ([M,3K]) and/or to out1 unsplit ([M,K]); at least one of them.  K % 4 == 0, K <= 2048. */
int pnp_layernorm_tf32_split3(const float *x, const float *residual, const float *residual_bias, float *x_out,
                              const float *gamma, const float *beta, float eps, float *out3, float *out1,
                              long long M, int K, pnp_stream_t stream);

/* The same three producers for the "3xFP16" form: x = h + l 2^-11 with h = fp16(x), l = fp16((x - h) 2^11), written as fp16
 * [h * hi_scale | l | h] ([M,3K] halves).  Against a weight operand [W_h 2^b | W_h | W_l] with hi_scale * 2^b = 2^11, ONE fp16
 * tensor-core GEMM with fp32 accumulation yields 2^11 * (x W^T) at fp32-grade accuracy; the consumer takes the factor back
 * through in_scale / residual_scale (x is multiplied by in_scale before anything else; the residual by residual_scale).
 * *overflow_flag (device int, optional) is set to 1 when a value does not fit fp16 (|x| * hi_scale > 65504, inf or NaN):
 * the caller checks it once per run and falls back to the TF32 form.  K % 4 == 0; out3 8-byte aligned. */
int pnp_fp16_split3(const float *x, float in_scale, float hi_scale, uint16_t *out3, int *overflow_flag, long long M,
                    int K, pnp_stream_t stream);
int pnp_gelu_fp16_split3(const float *x, float in_scale, const float *bias, float hi_scale, uint16_t *out3,
                         int *overflow_flag, long long M, int K, pnp_stream_t stream);
/* ld_out3 = row stride of out3 in halves: 3K, or 3K + 8 to append the bias columns [bias_one, 1, 0 x 6] to every row -- against
 * the weight rows [b_h 2^11 / bias_one, b_l, 0 x 6] (b = b_h + b_l 2^-11) the GEMM then adds the layer's bias by itself. */
int pnp_layernorm_fp16_split3(const float *x, const float *residual, float residual_scale,
                              const float *residual_bias, float *x_out, const float *gamma, const float *beta,
                              float eps, float hi_scale, uint16_t *out3, int ld_out3, float bias_one, float *out1,
                              int *overflow_flag, long long M, int K, pnp_stream_t stream);

/* Encoder self-attention softmax(Q K^T * softmax_scale) V (VIT:93-119) at fp32-grade accuracy on the fp16 tensor cores: every
 * operand split as above, each product as three fp16 products with fp32 accumulation (main term and corrections apart), online
 * softmax in fp32; nothing of size L x L touches HBM.  The main kernel issues tcgen05.mma with its accumulators in tensor memory
 * (csrc/attention.cu).  qkv [B,L,3,H,D] fp32 exactly as the fused qkv GEMM leaves it (each value times 1/in_scale, in_scale a
 * power of two; 1 for a plain projection); out [B,L,H*D] fp32, unscaled.  D must be 64.  The workspace holds the fp16 (hi, lo)
 * split of k and v. */
size_t pnp_attention_fp16x3_workspace_bytes(int B, int L, int H, int D);
/* out and / or out3 (at least one): out3 [B*L, 3*H*D] fp16 is the [h * out3_hi_scale | l | h] operand split of the output
 * (pnp_fp16_split3's layout), written straight from the accumulators for the projection GEMM that follows.
 * *overflow_flag (device int, optional) is set to 1, and never cleared, when the result may not be fp32-grade: a k or v value
 * times in_scale, or a q value times in_scale * softmax_scale * log2(e), outside fp16's range (or NaN); a row whose scores reach
 * 2^11 in magnitude in the exp2 domain (about 1420 in natural units, scores = q.k * softmax_scale), where the bf16 row bound the
 * softmax subtracts is too coarse for the fp16 (hi, lo) pairs of the probabilities; or, with out3, an output times out3_hi_scale
 * outside fp16's range.  Below that magnitude the result is fp32-grade whatever the spread of a row's scores. */
int pnp_attention_fp16x3(const float *qkv, float in_scale, float softmax_scale, float *out, uint16_t *out3,
                         float out3_hi_scale, void *workspace, size_t workspace_bytes, int *overflow_flag, int B, int L,
                         int H, int D, pnp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * In-situ kernel timing for bench.py's roofline (the one piece of process-global state in the library):
 * between start and stop, every launch of a kernel class whose bit is set in kernel_mask is bracketed by
 * CUDA events recorded on the launch's own stream.  Kernel ids: 1 softmax_fwd, 2 softmax_bwd_gradcam,
 * 3 token_merge, 4 salience_dropout_round, 5 threshold_prep, 6 upsample_write, 7 blur_vertical,
 * 8 blur_horizontal, 9 blur_normalize, 10 lattice_build (all of it), 11 crf_unary, 12 crf_splat_bilateral,
 * 13 crf_blur_axis_bilateral, 14 crf_meanfield_update, 15 argmax_channels, 16 confusion, 17 crf_splat_spatial,
 * 18 crf_blur_axis_spatial, 19 tf32_split3, 20 gelu_tf32_split3, 21 layernorm_tf32_split3, 22 lowrank_blur,
 * 23 lowrank_unary, 24 background_blur, 25 attention_fp16x3 (pnp_profile_kernel_name() is authoritative).
 * ---------------------------------------------------------------------------------------------------- */
int pnp_profile_num_kernels(void); /* ids are 1 .. pnp_profile_num_kernels()-1 */
int pnp_profile_start(unsigned kernel_mask);
/* Waits for the recorded events; total_ms[id] / n_launches[id] for id < n_ids (host arrays). */
int pnp_profile_stop(float *total_ms, int *n_launches, int n_ids);
const char *pnp_profile_kernel_name(int kernel_id);
/* enabled != 0: time only launches enqueued on `stream` (kernels overlapped on other streams are skipped). */
int pnp_profile_filter_stream(pnp_stream_t stream, int enabled);

#ifdef __cplusplus
}
#endif
#endif /* PNP_OVSS_B200_H */
