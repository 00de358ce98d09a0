/*
 * libmte -- B200-native (sm_100a) depth-edge hot path of MindTheEdge, C ABI.
 *
 * This header is the drop-in boundary.  The reference (liortalker/MindTheEdge)
 * is pure Python and has no FFI; each entry point below names the reference
 * function (file:line, relative to the reference root) whose arithmetic it
 * replaces.  INTEGRATION.md shows the ctypes stub a reference maintainer would
 * add at each of the three Python seams (edge-loss head, depth->edges,
 * bsds_metric matcher/thinner).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *     planes are dense row-major, images stacked along the leading axis
 *   - every call is asynchronous on `stream`; nothing allocates, nothing
 *     synchronises, no global mutable state (re-entrant; one workspace per
 *     in-flight call)
 *   - `workspace` must hold at least the matching *_workspace_bytes() and its
 *     first MTE_WS_HEADER_BYTES (64 KB: tickets, queues, the loss accumulators)
 *     must be zero before the FIRST use (kernels leave them zero again), see
 *     mte_workspace_init
 *   - return value: 0 = OK, < 0 = argument error (mte_error_string), > 0 =
 *     cudaError_t of the launch
 */
#ifndef MTE_H_
#define MTE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MTE_VERSION 200
#define MTE_MAX_SCALES 4
#define MTE_MAX_THRESHOLDS 254
#define MTE_WS_HEADER_BYTES 65536

typedef struct CUstream_st *mte_stream_t; /* == cudaStream_t */

enum {
    MTE_OK = 0,
    MTE_ERR_NULL = -1,      /* required pointer is NULL */
    MTE_ERR_SHAPE = -2,     /* non-positive or inconsistent shape */
    MTE_ERR_WORKSPACE = -3, /* workspace too small */
    MTE_ERR_ARG = -4,       /* attribute out of range */
    MTE_ERR_ALIGN = -5,     /* pointer not aligned to its element type */
    MTE_ERR_NOT_NESTED = -6 /* threshold list is not monotone where it must be */
};

enum { MTE_F32 = 0, MTE_F64 = 1, MTE_U8 = 2 };

int mte_version(void);
const char *mte_error_string(int code);
/* zero the workspace header (cudaMemsetAsync) */
int mte_workspace_init(void *workspace, size_t bytes, mte_stream_t stream);

/* ------------------------------------------------------------------------
 * (1) Training edge loss.
 * Replaces GradLoss.forward + GradLayer.forward + comp_cross_entropy
 * (packnet_code/packnet_sfm/losses/grad_loss.py:65-95, 122-159, 161-219) and
 * the autograd backward of that chain; with several scales it also replaces
 * the per-scale loop of compute_edge_loss_with_all_scales
 * (packnet_code/packnet_sfm/models/SemiSupEdgeModel.py:164-198).
 * ------------------------------------------------------------------------ */
typedef struct {
    const float *pred;   /* [B,1,h,w] predicted depth (prob map if !is_grad)   */
    const float *edge;   /* [B,1,H,W] soft edge labels in [0,1]                */
    const float *normal; /* [B,1,H,W] edge-normal angle in radians, or NULL    */
    const float *mask;   /* [B,1,H,W] validity mask, or NULL                   */
    float *grad_map;     /* out [B,1,H,W] |directional gradient| (NULL = skip) */
    float *grad_pred;    /* bwd out [B,1,h,w] d loss / d pred                  */
    uint8_t *stash;      /* optional [B,1,H,W]: the forward records 1 byte/px (picked
                            direction + sign of the response); a backward that is given
                            the same stash and grad_map skips the stencil recompute   */
    int32_t B, h, w, H, W;
    float scale_weight;  /* this scale's share of the total (e.g. 0.25)        */
} mte_loss_scale_t;

typedef struct {
    int32_t is_grad;        /* grad_loss.py:129 */
    int32_t is_sigmoid;     /* grad_loss.py:134 */
    int32_t pred_is_inverse;/* fuse inv2depth (utils/depth.py:104-121): pred = 1/clamp(inv,1e-6) */
    float sigmoid_thresh;   /* grad_loss.py:122 (4) */
    float weight;           /* depth_edges_loss_weight, grad_loss.py:158 */
    float pos_to_neg;       /* depth_edges_loss_pos_to_neg_weight, grad_loss.py:212 */
} mte_loss_attrs_t;

size_t mte_edge_loss_workspace_bytes(const mte_loss_scale_t *scales_host, int n_scales);
size_t mte_edge_loss_ctx_bytes(const mte_loss_scale_t *scales_host, int n_scales);
/* loss_out: device float[1 + n_scales] = {sum_s scale_weight_s*loss_s, loss_0, ...}
 * ctx: device buffer carried to the backward (per-image alpha, normalisers).   */
int mte_edge_loss_fwd(const mte_loss_scale_t *scales_host, int n_scales, const mte_loss_attrs_t *attrs_host,
                      float *loss_out, void *ctx, void *workspace, size_t workspace_bytes, mte_stream_t stream);
/* grad_loss: device float[1 + n_scales] upstream gradients w.r.t. loss_out
 * (entry 0 applies to every scale through scale_weight, entry 1+s to scale s). */
int mte_edge_loss_bwd(const mte_loss_scale_t *scales_host, int n_scales, const mte_loss_attrs_t *attrs_host,
                      const float *grad_loss, const void *ctx, void *workspace, size_t workspace_bytes,
                      mte_stream_t stream);

/* One-pass variant for the shipped configuration (is_grad, normals, no mask, prediction at the target size, W % 4
 * == 0, 16-byte aligned planes -- mte_edge_loss_fused_supported says whether a call qualifies): ONE launch produces
 * loss_out, grad_map AND grad_pred.  The class balance alpha_b depends only on the targets (grad_loss.py:169-178), so
 * it is computed in a pre-phase of the same kernel and d loss / d pred is emitted with the forward, for the upstream
 * gradient the caller expects: expected_grad_loss is a DEVICE float[1 + n_scales] (same meaning as grad_loss of
 * mte_edge_loss_bwd) or NULL = {1, 0, ...} (loss.backward()).  The autograd backward is then
 * mte_edge_loss_grad_rescale: it compares the actual upstream gradient (device float[1 + n_scales]) with the factor
 * recorded in ctx, returns at once when they agree and rescales grad_pred in place otherwise; expected_out (optional
 * device float[1 + n_scales]) receives the actual gradient, to be passed as the next step's expectation.
 * Replaces the same reference code as mte_edge_loss_fwd + mte_edge_loss_bwd; 20 B/px of HBM traffic instead of 34. */
int mte_edge_loss_fused_supported(const mte_loss_scale_t *scales_host, int n_scales, const mte_loss_attrs_t *attrs_host);
int mte_edge_loss_fwd_grad(const mte_loss_scale_t *scales_host, int n_scales, const mte_loss_attrs_t *attrs_host,
                           const float *expected_grad_loss, float *loss_out, void *ctx, void *workspace,
                           size_t workspace_bytes, mte_stream_t stream);
int mte_edge_loss_grad_rescale(const mte_loss_scale_t *scales_host, int n_scales, const float *grad_loss, void *ctx,
                               float *expected_out, mte_stream_t stream);

/* Alternative loss types of GradLoss.forward (grad_loss.py:143-156; attention_loss2,
 * losses/attention_loss.py:21-49), single scale, prediction already at the target
 * size.  They build on the fused forward's side outputs: grad_map (the |directional
 * response|, or the map itself when !is_grad) and stash.  loss_types is a bit set;
 * MTE_LOSS_DICE is added to a base type (alone it is an error, as in the reference);
 * with MTE_LOSS_CE, ce_loss points at loss_out[0] of mte_edge_loss_fwd (same weight)
 * and the caller runs mte_edge_loss_bwd first, then this backward with accumulate=1.
 * loss_out: device float[2] (both = weight * loss); ctx: device float[4]. */
enum { MTE_LOSS_CE = 1, MTE_LOSS_ATTENTION = 2, MTE_LOSS_SPATIAL = 4, MTE_LOSS_DICE = 8 };
size_t mte_edge_loss_alt_workspace_bytes(int B, int H, int W);
int mte_edge_loss_alt_fwd(const float *grad_map, const float *edge, const float *mask, int B, int H, int W,
                          int loss_types, int is_sigmoid, float sigmoid_thresh, float weight, const float *ce_loss,
                          float *loss_out, float *ctx, void *workspace, size_t workspace_bytes, mte_stream_t stream);
int mte_edge_loss_alt_bwd(const float *grad_map, const float *edge, const float *mask, const uint8_t *stash,
                          const float *pred, int B, int H, int W, int loss_types, int is_grad, int is_sigmoid,
                          int pred_is_inverse, float sigmoid_thresh, float weight, const float *grad_loss,
                          const float *ctx, float *grad_pred, int accumulate, void *workspace,
                          size_t workspace_bytes, mte_stream_t stream);

/* Target preparation from the on-disk encoding (SURVEY.md 8f rank 2).
 * mte_decode_normals: u8 PNG value -> angle, (360.*(v/255.) - 180)*(pi/180) in float64 then
 * float32 (packnet_code/packnet_sfm/datasets/gta_dataset.py:413, 421).
 * mte_edge_resize_preserve: resize_depth_preserve (datasets/augmentations.py:58-100) of u8
 * edge maps [B,h,w] to [B,H,W] (last valid source pixel in raster order wins) followed by
 * the "/255 if max > 1" rule of resize_sample (:193-199), on the max of each resized
 * map, and the float32 cast. */
int mte_decode_normals(const uint8_t *normal_u8, float *theta_out, size_t n, mte_stream_t stream);
size_t mte_edge_resize_workspace_bytes(int B);
int mte_edge_resize_preserve(const uint8_t *edge_u8, int B, int h, int w, float *edge_out, int H, int W,
                             void *workspace, size_t workspace_bytes, mte_stream_t stream);

/* ------------------------------------------------------------------------
 * (2a) Depth -> edges for evaluation.
 * Replaces the array part of edge_from_depth (edge.py:81-88, twin
 * packnet_code/packnet_sfm/utils/edge.py:74-83): clamp, *255/max_depth, uint8,
 * cv2.Canny(u8, low, high) (aperture 3, L1 norm), for T threshold pairs at once.
 * ------------------------------------------------------------------------ */
size_t mte_canny_workspace_bytes(int n_images, int H, int W, int n_pairs);
/* depth: [N,H,W] of depth_dtype (MTE_F32|MTE_F64|MTE_U8; U8 = already quantised,
 * the bare cv2.Canny call of models/model_wrapper.py:399-401).
 * edges: out [T,N,H,W] uint8 in {0,255}, or NULL.
 * levels: out [N,H,W] uint8 = index of the first pair (pairs must then be nested,
 *         strictest first) at which the pixel is an edge, 255 = never; or NULL. */
int mte_canny_from_depth(const void *depth, int depth_dtype, int n_images, int H, int W, double min_depth,
                         double max_depth, const int32_t *lows_host, const int32_t *highs_host, int n_pairs,
                         uint8_t *edges, uint8_t *levels, void *workspace, size_t workspace_bytes,
                         mte_stream_t stream);

/* Resize of predicted depth to the GT size in front of the Canny sweep:
 * cv2.resize(depth, (W, H), interpolation=cv2.INTER_LINEAR) of edge.py:76-78 (twin
 * packnet_code/packnet_sfm/utils/edge.py:76-78), bit-exact against the opencv-python 4.13.0 wheel with its IPP
 * HAL on (DESIGN.md section 2).  src: [N,h,w] of dtype, dst: out [N,H,W] of the same dtype; src and dst must not
 * overlap.  Takes MTE_F32 with h, w >= 2 only: MTE_F64 (or any other dtype) is MTE_ERR_ARG and a one-row or
 * one-column source MTE_ERR_SHAPE, the inputs whose cv2.resize arithmetic is not pinned.  Both pointers must be
 * 4-byte aligned (MTE_ERR_ALIGN).  The same shape is a device-to-device copy.  No workspace. */
int mte_resize_linear(const void *src, int dtype, int n_images, int h, int w, void *dst, int H, int W,
                      mte_stream_t stream);

/* ------------------------------------------------------------------------
 * (2b) DEE annotation post-process.
 * normals : infer_edge_estimation.py:193-199 (= :244-250)
 * nms     : non_max_suppression, packnet_code/packnet_sfm/utils/tools.py:9-46
 * hyst    : hysteresis + DFS,    packnet_code/packnet_sfm/utils/tools.py:49-92
 * ------------------------------------------------------------------------ */
size_t mte_dee_workspace_bytes(int n_images, int H, int W);
/* prob [N,H,W] f32.  normals_out u8 [N,H,W] or NULL.  edges_out [N,H,W] of
 * out_dtype (MTE_F32|MTE_F64) or NULL.  do_nms / do_hyst choose the stages (the
 * reference's cfg.datasets.test.{nms,hysteresis}); in_dtype is the dtype the
 * reference would have seen at the hysteresis input when do_nms == 0. */
int mte_dee_postprocess(const void *prob, int in_dtype, int n_images, int H, int W, int do_nms, int do_hyst,
                        double t_low, double t_high, uint8_t *normals_out, void *edges_out, int out_dtype,
                        void *workspace, size_t workspace_bytes, mte_stream_t stream);

/* ------------------------------------------------------------------------
 * (3) Precision / recall counts.
 * mte_pr_counts replaces evaluate_boundaries (eval_depth_edges.py:67-145) for a
 * batch of images with one GT map each (the only shipped use, :213) including
 * the crop of _pred_eval (:195-197, :206-208) and the per-image sum of
 * pr_evaluation (:298-301).  The matcher replaces py-bsds500
 * correspond_pixels (call sites eval_depth_edges.py:50-52, 130-132); the
 * thinner replaces py-bsds500 thin.binary_thin (:45, :125).
 * ------------------------------------------------------------------------ */
size_t mte_pr_workspace_bytes(int n_images, int H, int W, int n_thresholds, double max_dist);
/* workspace of mte_pr_counts with apply_thinning = 1: the above plus a slab of
 * thinned bit planes (about 64 MB at most, less for small batches) */
size_t mte_pr_thin_workspace_bytes(int n_images, int H, int W, int n_thresholds, double max_dist);
/* pred: [N,H,W] of pred_dtype:
 *   MTE_F32/MTE_F64 strength map, thresholded as pred >= thresholds[t] (in fp64)
 *   MTE_U8          level plane from mte_canny_from_depth: edge at t iff level <= t
 * gt: [N,H,W] u8, non-zero = boundary.  crop = {x0,x1,y0,y1} or NULL: the
 * window [y0:y1, x0:x1] with python slice semantics, as the reference crops:
 * a negative bound counts from the end of its axis (b + dim), bounds are then
 * clamped to [0, dim], and x1 <= x0 or y1 <= y0 is an empty window.
 * max_dist: matching radius max_dist * sqrt(h^2 + w^2) px of the h x w window
 * (as correspond_pixels); a radius of 32 px or more is MTE_ERR_ARG.
 * counts: device int64[T,4] in the order
 * count_r,sum_r,count_p,sum_p, ACCUMULATED into (zero it first).
 * apply_thinning: 0 = match the binarised window as it is; 1 = thin it first
 * (evaluate_boundaries' default, eval_depth_edges.py:125): the window is cut
 * out of the plane BEFORE it is thinned, so thinning zero-pads at the crop
 * border, not at the plane border, and runs to convergence; sum_p is then the
 * size of the thinned set.  Thresholds may come in any order and repeat (row t
 * of counts belongs to thresholds[t]); the workspace must hold
 * mte_pr_thin_workspace_bytes.  Any other value is MTE_ERR_ARG. */
int mte_pr_counts(const void *pred, int pred_dtype, const uint8_t *gt, int n_images, int H, int W,
                  const int32_t *crop_host, const double *thresholds_host, int n_thresholds, double max_dist,
                  int apply_thinning, int64_t *counts, void *workspace, size_t workspace_bytes,
                  mte_stream_t stream);
/* The same counts per image, from the same single launch chain: counts is a
 * device int64[N,T,4], row (i, t) holding image i's count_r,sum_r,count_p,sum_p
 * for thresholds[t] (or level t), ACCUMULATED into as above.  Arguments,
 * argument checks, workspace queries and return codes are those of
 * mte_pr_counts; summed over i the rows equal its output bit for bit (every
 * row has one writer per call, so they are deterministic).  An empty crop
 * leaves the rows untouched.  These are the per-image EvalResult counts of
 * _pred_eval (eval_depth_edges.py:179-230) before pr_evaluation sums them. */
int mte_pr_counts_per_image(const void *pred, int pred_dtype, const uint8_t *gt, int n_images, int H, int W,
                            const int32_t *crop_host, const double *thresholds_host, int n_thresholds,
                            double max_dist, int apply_thinning, int64_t *counts, void *workspace,
                            size_t workspace_bytes, mte_stream_t stream);

size_t mte_match_workspace_bytes(int n_problems, int h, int w, double max_dist);
/* a,b: [P,h,w] u8 boundary maps.  match_a/match_b: out [P,h,w] u8 (1 = matched)
 * or NULL.  count: device int64[P].  max_dist as in mte_pr_counts (radius
 * max_dist * sqrt(h^2 + w^2) px; 32 px or more is MTE_ERR_ARG). */
int mte_correspond_pixels(const uint8_t *a, const uint8_t *b, int n_problems, int h, int w, double max_dist,
                          uint8_t *match_a, uint8_t *match_b, int64_t *count, void *workspace,
                          size_t workspace_bytes, mte_stream_t stream);

size_t mte_thin_workspace_bytes(int n_images, int H, int W);
int mte_binary_thin(const uint8_t *in, uint8_t *out, int n_images, int H, int W, int max_iter, void *workspace,
                    size_t workspace_bytes, mte_stream_t stream);

/* ------------------------------------------------------------------------
 * In-training "light" metric: chamfer_distance
 * (packnet_code/packnet_sfm/utils/edge.py:20-62; called per Canny setting in
 * both directions by compute_edge_metrics, models/model_wrapper.py:434-440)
 * for a batch of u8 edge maps (set = value/255 > 0.5).
 * out: device double[N,4] = {sum over pred px of the Euclidean distance to the
 *      nearest gt px (exact EDT, as scipy.ndimage.distance_transform_edt),
 *      #pred px, #pred px with distance < thresh, 0}.
 * cond_out: optional int8 [N,H,W]: -1 = not a pred px, 1 = closer than thresh,
 *      0 = not (the third return value of the reference), or NULL.
 * Limits: 1 <= H <= 65,533 (column distances are u16) and 1 <= W <= 24,576
 *      (one row of them sits in shared memory); anything else is MTE_ERR_SHAPE.
 * An image without any GT px measures from (-1, 0), as scipy's EDT does.
 * ------------------------------------------------------------------------ */
size_t mte_chamfer_workspace_bytes(int n_images, int H, int W);
int mte_chamfer_counts(const uint8_t *pred, const uint8_t *gt, int n_images, int H, int W, double thresh,
                       double *out, int8_t *cond_out, void *workspace, size_t workspace_bytes, mte_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MTE_H_ */
