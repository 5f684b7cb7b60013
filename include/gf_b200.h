/*
 * gf_b200.h — C ABI of the B200-native GaussianFormer hot path.
 *
 * Plain pointers and sizes only (no torch types).  Every pointer is a DEVICE pointer unless it
 * says "host".  Every entry point is asynchronous on the given stream and returns a GF_* status;
 * gf_last_error() gives the message for the calling thread.  The library never allocates or
 * frees device memory: scratch is a caller-provided workspace whose size comes from the matching
 * *_workspace_bytes() query (the reference instead grows torch byte tensors through
 * std::function callbacks — model/head/localagg/local_aggregate.cu:27-33,58-63).
 *
 * What each entry point replaces in the reference (paths relative to the reference tree):
 *
 *   gf_splat_forward   LocalAggregator::Aggregator::forward
 *                        model/head/localagg/src/aggregator.h:24-41, src/aggregator_impl.cu:152-252
 *                        model/head/localagg_prob/src/aggregator.h (variant = GF_SPLAT_PROB)
 *                        model/head/localagg_prob_fast/src/auxiliary.h:8-20 (radii_axes = 3)
 *                      plus, when the *_int / radii pointers are NULL, the host preparation of
 *                        model/head/localagg/local_aggregate/__init__.py:137-143
 *   gf_splat_backward  LocalAggregator::Aggregator::backward
 *                        model/head/localagg/src/aggregator.h:43-61, src/aggregator_impl.cu:256-307
 *                        model/head/localagg_prob/src/backward.cu:24-123 (variant = GF_SPLAT_PROB)
 *   gf_daf_forward     deformable_aggregation()
 *                        model/encoder/gaussian_encoder/ops/src/deformable_aggregation.cpp:4-18
 *                        .../ops/src/deformable_aggregation_cuda.cu:262-284
 *   gf_daf_backward    deformable_aggregation_grad()
 *                        .../ops/src/deformable_aggregation.cpp:20-38, ..._cuda.cu:287-313
 *
 *   gf_daf_fused_*     no native counterpart in the reference: the op call above together with the PyTorch code
 *                      around it in DeformableFeatureAggregation.forward
 *                        model/encoder/gaussian_encoder/deformable_module.py:213-228 (masked joint softmax of
 *                        the weights) and :242 (sum over the key points) -- an opt-in entry point (SURVEY.md 8f-2)
 *
 * The ABI is a superset of those boundaries: explicit stream, explicit class count C (the
 * reference hard-codes NUM_CHANNELS 18, model/head/localagg/src/config.h:15), 64-bit safe sizes,
 * caller-owned workspace and an int status.
 */
#ifndef GF_B200_H_
#define GF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GF_ABI_VERSION 2

/* status codes */
#define GF_OK 0
#define GF_ERR_INVALID_ARG 1   /* bad shape / NULL pointer / unsupported combination */
#define GF_ERR_WORKSPACE 2     /* workspace NULL, misaligned or smaller than *_workspace_bytes() */
#define GF_ERR_CUDA 3          /* a CUDA runtime call failed (message has cudaGetErrorString) */
#define GF_ERR_UNSUPPORTED 4   /* e.g. class count outside the compiled range */

/* splat variants */
#define GF_SPLAT_BASE 0        /* local_aggregate:            logits                       */
#define GF_SPLAT_PROB 1        /* local_aggregate_prob(_fast): logits, bin_logits, density  */

/* bits of the device-side status word (gf_splat_read_flags) — the conditions the reference's
 * Python wrapper asserts on (local_aggregate/__init__.py:138,140,142) */
#define GF_FLAG_POINT_OUT_OF_GRID 1u
#define GF_FLAG_MEAN_OUT_OF_GRID 2u
#define GF_FLAG_RADIUS_LT_1 4u
#define GF_FLAG_GENERIC_PATH 256u /* informational: points were not in canonical voxel order */

typedef void *gf_stream_t; /* a cudaStream_t (NULL = legacy default stream) */

typedef struct gf_splat_desc {
    int32_t G;          /* Gaussians (P in the reference) */
    int32_t N;          /* query points */
    int32_t C;          /* classes / channels (18 for nuScenes-SurroundOcc) */
    int32_t H, W, D;    /* voxel grid */
    int32_t variant;    /* GF_SPLAT_BASE | GF_SPLAT_PROB */
    int32_t radii_axes; /* 1: one radius per Gaussian, 3: per-axis radii (prob_fast) */
    int32_t cov_stride; /* floats per Gaussian in `cov`: 6 = (xx,yy,zz,xy,yz,xz); 9 = row-major
                           3x3 from which entries [0,4,8,1,5,2] are taken (__init__.py:143) */
    /* host-preparation parameters, used when points_int / means_int / radii are NULL */
    float pc_min[3];
    float grid_size;
    float scale_multiplier;
    int32_t radii_min;  /* <=0: no clamp (base variant); >=1: radii.clamp(min) (prob variants) */
    /* ---- ABI 2: explicit batch (the reference op is per sample, local_aggregate/__init__.py:128; SURVEY.md 8b/8e) ---- */
    int32_t batch;      /* samples per call, B >= 1 (0 is read as 1).  Every input / output / gradient tensor carries a
                           leading dimension B with dense strides ([B,N,3], [B,G,3], [B,G], [B,G,C], [B,N,C], ...); all B
                           samples are processed by ONE grid per kernel, and the workspace is B times the B = 1 size */
    int32_t pts_shared; /* != 0: pts / points_int are ONE [N,3] array shared by every sample of the batch (the voxel
                           centres of the occupancy grid, dataset/transform_3d.py:487-499) instead of [B,N,3] */
} gf_splat_desc;

/* Inputs of both passes.  points_int / means_int / radii mirror the reference's native
 * boundary; pass NULL to have them derived on the device from pts / means / scales exactly as
 * the reference's Python wrapper does (fp32 subtract, fp32 divide, truncate; ceil for radii). */
typedef struct gf_splat_inputs {
    const float *pts;         /* [N,3] */
    const int32_t *points_int;/* [N,3] or NULL */
    const float *means;       /* [G,3] */
    const int32_t *means_int; /* [G,3] or NULL */
    const float *opacities;   /* [G] */
    const float *semantics;   /* [G,C] */
    const float *cov;         /* [G,cov_stride] inverse covariance */
    const int32_t *radii;     /* [G] or [G,3], or NULL */
    const float *scales;      /* [G,3]; read when radii == NULL or cov == NULL */
    /* ---- ABI 2: head pre-op fusion (SURVEY.md 8f-1) ---- */
    const float *rotations;   /* [G,4] quaternions (w,x,y,z), any norm > 0, or NULL.  With cov == NULL the inverse
                                 covariance is built on the device as R^T diag(1/s^2) R from scales and rotations -- the
                                 closed form of GaussianHead.prepare_gaussian_args' Cov = (S R)^T (S R),
                                 Cov.cpu().inverse().cuda() (model/head/gaussian_head.py:111-119; quaternion -> matrix
                                 as model/utils/utils.py:20-66) -- inside the pack kernel */
} gf_splat_inputs;

typedef struct gf_splat_outputs {
    float *logits;      /* [N,C]; may be NULL when logits_cn, argmax or ce_partials is requested instead */
    float *bin_logits;  /* [N]  (prob only) */
    float *density;     /* [N]  (prob only) */
    float *probability; /* [N]  (prob only; saved for backward like the reference) */
    uint8_t *argmax;    /* [N]  optional, NULL = off: class with the largest logit per point (lowest
                           index on ties) — the `argmax(dim=1)` of GaussianHead.forward
                           (model/head/gaussian_head.py:185) fused into the render epilogue */
    /* ---- ABI 2: post-op fusion toward the loss (SURVEY.md 8f-3); all optional, NULL = off ---- */
    float *logits_cn;   /* [C,N] per sample: the logits class-major, i.e. the `semantics[None].transpose(1, 2)` /
                           `[1, C, N]` layout GaussianHead hands to the loss (gaussian_head.py:165-175), written by the
                           render epilogue; `logits` may then be NULL (inference: the [N,C] copy never exists) */
    const uint8_t *labels;      /* [N] per sample: target class per point, 255 = ignore (loss/occupancy_loss.py:113-127) */
    const float *class_weights; /* [C] (shared by the batch) or NULL = all ones */
    float *ce_partials; /* [gf_splat_ce_partials(desc), 2] fully overwritten: per render CTA (sum_n w[y_n] * nll_n,
                           sum_n w[y_n]) of CE_ssc_loss = nn.CrossEntropyLoss(weight, ignore_index=255, 'mean')
                           (loss/occupancy_loss.py:164-178) over the CTA's points; loss = sum(col 0) / sum(col 1).
                           Needs labels; tile path only (N == H*W*D, canonical order) */
} gf_splat_outputs;

typedef struct gf_splat_grads {
    /* upstream */
    const float *logits_grad;     /* [N,C] */
    const float *bin_logits_grad; /* [N] (prob only) */
    const float *density_grad;    /* [N] (prob only) */
    /* saved forward outputs (prob only) */
    const float *logits;          /* [N,C] */
    const float *bin_logits;      /* [N] */
    const float *probability;     /* [N] */
    /* results: fully overwritten */
    float *means_grad;            /* [G,3] */
    float *opacity_grad;          /* [G] */
    float *semantics_grad;        /* [G,C] */
    float *cov_grad;              /* cov_stride 6: [G,6] in (xx,yy,zz,xy,yz,xz) order; cov_stride 9: [G,9] row-major
                                     3x3, entries [0,4,8,1,5,2] carry the gradient, [3,6,7] are written as 0.
                                     May be NULL when in->cov == NULL (scales + rotations input) */
    /* ---- ABI 2: gradients of the fused pre-op (in->cov == NULL, in->rotations != NULL); fully overwritten ---- */
    float *scales_grad;           /* [G,3] through Sigma^-1 only (the radii are detached, __init__.py:134) */
    float *rotations_grad;        /* [G,4] w.r.t. the un-normalised quaternion */
} gf_splat_grads;

typedef struct gf_daf_desc {
    int32_t batch;      /* B */
    int32_t num_cams;   /* M */
    int32_t num_feat;   /* F = sum_l h_l*w_l */
    int32_t num_embeds; /* C */
    int32_t num_scale;  /* L */
    int32_t num_pts;    /* P */
    int32_t num_groups; /* Gr, divides C */
} gf_daf_desc;

#define GF_DAF_MAX_LEVELS 8

/* feature_maps_format (ops/deformable_aggregation.py:78-117, forward direction): L maps
 * [B*M, C, h_l, w_l] (contiguous) <-> one channels-last table [B*M, F, C], F = sum_l h_l*w_l,
 * level l occupying rows [sum_{k<l} h_k*w_k, ...).  The reference builds it with reshape + cat +
 * permute and leaves the transposing copy to every later .contiguous(). */
typedef struct gf_daf_format_desc {
    int32_t batch_cams; /* B*M */
    int32_t num_embeds; /* C */
    int32_t num_scale;  /* L <= GF_DAF_MAX_LEVELS */
    int32_t hw[GF_DAF_MAX_LEVELS]; /* h_l*w_l */
} gf_daf_format_desc;

int gf_abi_version(void);
const char *gf_last_error(void);

/* number of classes the splat kernels were compiled for: returns how many values were written
 * to out[] (at most cap). */
int gf_splat_supported_classes(int32_t *out, int cap);

size_t gf_splat_forward_workspace_bytes(const gf_splat_desc *desc);
/* rows of out->ce_partials for this desc (render CTAs of the tile path x batch); 0 when the tile path does not apply */
int gf_splat_ce_partials(const gf_splat_desc *desc);
size_t gf_splat_backward_workspace_bytes(const gf_splat_desc *desc);

int gf_splat_forward(const gf_splat_desc *desc, const gf_splat_inputs *in,
                     const gf_splat_outputs *out, void *workspace, size_t workspace_bytes,
                     gf_stream_t stream);

int gf_splat_backward(const gf_splat_desc *desc, const gf_splat_inputs *in,
                      const gf_splat_grads *grads, void *workspace, size_t workspace_bytes,
                      gf_stream_t stream);

/* Copies the status word of the last gf_splat_forward that used `workspace` to *host_flags
 * (GF_FLAG_* bits) and synchronises the stream.  The reference raises AssertionError from Python
 * for the same conditions. */
int gf_splat_read_flags(const void *workspace, gf_stream_t stream, uint32_t *host_flags);

/* out[B,P,C] is fully overwritten. */
int gf_daf_forward(const gf_daf_desc *desc, const float *mc_ms_feat, const int32_t *spatial_shape,
                   const int32_t *scale_start_index, const float *sample_location,
                   const float *weights, float *output, gf_stream_t stream);

/* Accumulates (+=) into the three gradient buffers like the reference's atomics do; the caller
 * zero-fills them first (ops/deformable_aggregation.py:55-57). */
int gf_daf_backward(const gf_daf_desc *desc, const float *mc_ms_feat, const int32_t *spatial_shape,
                    const int32_t *scale_start_index, const float *sample_location,
                    const float *weights, const float *grad_output, float *grad_mc_ms_feat,
                    float *grad_sampling_location, float *grad_weights, gf_stream_t stream);

/* One pass over the data in either direction: inverse == 0 gathers the L maps into `table`
 * (fully overwritten); inverse != 0 scatters `table` back into the L maps (fully overwritten; this is the
 * gradient of the forward direction).  maps[l] are device pointers, the array itself lives on the host. */
int gf_daf_format(const gf_daf_format_desc *desc, float *const *maps, float *table, int inverse,
                  gf_stream_t stream);

/* ---- fused caller path of the deformable aggregation (opt-in; the entry points above stay the drop-in) ----
 *
 * For every anchor a (num_pts = A * pts_per_anchor sampling points per batch element, anchor-major) and
 * group g, with e running over the anchor's (key point k, camera m, level l) entries:
 *
 *   on_e   = point_mask[b,a,k,m] (or 1 if NULL)  &  weight_mask[b,a,k,m,l,g] (or 1 if NULL)
 *   w_e    = on_e ? exp(logit_e) / sum_{e' on} exp(logit_e') : 0        (all weights 0 when no entry is on)
 *   out[b,a,c] = sum_k gf_daf_forward(...)[b, a*K + k, c]  evaluated with the weights w
 *
 * which is deformable_module.py:213-228 + :242 (weights[~mask] = -inf; weights[all_miss] = 0; softmax over the
 * flattened (k, m, l) axis; * (1 - all_miss); DAF.apply; .sum(dim=2)).  Masks are bytes (0 / non-zero; a
 * torch.bool tensor).  `stats` [B, A, Gr, 2] receives (max * log2(e), 1 / sum) per anchor and group and is what
 * the backward needs besides the forward output.  Supported when gf_daf_fused_supported() != 0:
 * num_embeds % 128 == 0, groups a power of two that divides num_embeds / 4 into power-of-two runs,
 * num_cams * num_scale <= 32; other shapes return GF_ERR_UNSUPPORTED (use the unfused entry points). */
typedef struct gf_daf_fused_desc {
    gf_daf_desc d;
    int32_t pts_per_anchor; /* K; d.num_pts % K == 0 */
} gf_daf_fused_desc;

int gf_daf_fused_supported(const gf_daf_fused_desc *desc);

/* output [B, A, C] and stats [B, A, Gr, 2] are fully overwritten. */
int gf_daf_fused_forward(const gf_daf_fused_desc *desc, const float *mc_ms_feat, const int32_t *spatial_shape,
                         const int32_t *scale_start_index, const float *sample_location,
                         const float *weight_logits, const uint8_t *point_mask, const uint8_t *weight_mask,
                         float *output, float *stats, gf_stream_t stream);

/* grad_weight_logits [B, A, K, M, L, Gr] is fully overwritten; grad_mc_ms_feat and grad_sampling_location are
 * accumulated into (+=) like gf_daf_backward: the caller zero-fills them. */
int gf_daf_fused_backward(const gf_daf_fused_desc *desc, const float *mc_ms_feat, const int32_t *spatial_shape,
                          const int32_t *scale_start_index, const float *sample_location,
                          const float *weight_logits, const uint8_t *point_mask, const uint8_t *weight_mask,
                          const float *stats, const float *output, const float *grad_output,
                          float *grad_mc_ms_feat, float *grad_sampling_location, float *grad_weight_logits,
                          gf_stream_t stream);

/* ---- occupancy loss: weighted cross-entropy + Lovász-softmax, value and gradient (no counterpart in the native
 * reference: OccupancyLoss.loss_voxel, loss/occupancy_loss.py:102-149, with CE_ssc_loss :164-178 / CE_wo_softmax
 * :180-183 and lovasz_softmax(classes='present', per_image=False), loss/utils/lovasz_softmax.py:157-204) ----
 *
 * All B*N points form ONE pooled set.  A point takes part when mask[i] != 0 (or mask == NULL) and, with ignore_empty,
 * labels[i] != empty_label.  Of those:
 *   CE      = sum w[y] nll / sum w[y] over y < C, y != ignore_index; nll = -log_softmax(pred)[y] (use_softmax) or
 *             -log(clamp(pred[y], 1e-6, 1 - 1e-6)); NaN (0/0) when no point is left, as in torch
 *   Lovász  = mean over the classes present in the set {y != lovasz_ignore} (255 labels stay in it as background) of
 *             sum_i e_(i) dJ_i, e = |[y = c] - q_c| sorted in descending order, q = softmax(pred) or pred; 0 without a
 *             present class.  Equal errors are ordered by point index (a stable sort; the reference leaves their order
 *             to torch.sort).  dJ is computed in closed form from integer counts.  q is expected in [0, 1]; errors
 *             above 1 are treated as 1
 *   loss3   = [ce_weight * CE + lovasz_weight * Lovász, ce_weight * CE, lovasz_weight * Lovász]
 *   grad    = d loss3[0] / d pred (torch's subgradients: abs'(0) = 0, clamp passes the gradient on [lo, hi]); 0 for
 *             points that take no part
 * Labels that are neither < C nor ignore_index contribute nothing and set GF_OCC_LABEL_OUT_OF_RANGE in *status.
 * Loss and gradient are bit-identical between calls (fixed-order fp64 sums, no floating-point atomics). */
#define GF_OCC_LABEL_OUT_OF_RANGE 1u

typedef struct gf_occ_loss_desc {
    int32_t B, N, C;        /* pred [B, N, C] row-major (the splat's logits layout); C in 16..20 */
    int32_t use_softmax;    /* != 0: pred are logits (GaussianFormer-1); 0: probabilities (GaussianFormer-2) */
    int32_t ignore_index;   /* CE ignore label, 0..255 (255 in the reference) */
    int32_t lovasz_ignore;  /* label left out of the Lovász set, -1 = none (17 in the shipped configs) */
    int32_t ignore_empty;   /* != 0: points labelled empty_label take no part */
    int32_t empty_label;
    float ce_weight;        /* loss_voxel_ce_weight */
    float lovasz_weight;    /* loss_voxel_lovasz_weight */
    int32_t lovasz;         /* != 0: compute the Lovász term (use_lovasz_loss) */
} gf_occ_loss_desc;

size_t gf_occ_loss_workspace_bytes(const gf_occ_loss_desc *desc);

/* pred [B,N,C] fp32, labels [B,N] uint8, mask [B,N] uint8 or NULL, class_weights [C] or NULL (ones).  loss3 [3] and
 * grad_pred [B,N,C] (NULL: no gradient) are fully overwritten, as is *status (device word, may be NULL).  The
 * workspace needs no initialisation. */
int gf_occ_loss_forward(const gf_occ_loss_desc *desc, const float *pred, const uint8_t *labels, const uint8_t *mask,
                        const float *class_weights, float *loss3, float *grad_pred, uint32_t *status, void *workspace,
                        size_t workspace_bytes, gf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GF_B200_H_ */
