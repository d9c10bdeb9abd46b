/*
 * gsvc_rast.h — C-ABI of libgsvc_rast.so, the B200-native (sm_100a) orthographic TSW Gaussian
 * rasterizer that replaces GSVC's external CUDA extension
 *   diff_gaussian_rasterization.cuda_ortho_gaussian_rasterizer
 * (github.com/actcwlf/ortho_diff_gaussian_rasterization, /root/reference/README.md:52).
 *
 * The reference binds that extension at exactly two call sites:
 *   rasterizer(means3D, means2D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp)
 *       /root/reference/ortho_gaussian_renderer/renderer.py:85-98      → gsvc_rast_forward* / gsvc_rast_backward
 *   rasterizer.visible_filter(means3D, scales, rotations, cov3D_precomp)
 *       /root/reference/ortho_gaussian_renderer/preprocess.py:99-104   → gsvc_rast_visible_filter
 * with the settings block built at renderer.py:63-83 / preprocess.py:58-79 → gsvc_rast_settings.
 *
 * Conventions: plain pointers and sizes only.  Every array pointer is DEVICE memory on the current
 * CUDA device unless its name ends in `_host`.  All float arrays are fp32, densely packed,
 * row-major ([P,3] = 3 consecutive floats per Gaussian).  `stream` is a cudaStream_t passed as
 * void* (NULL = legacy default stream).  Every function returns 0 (or a non-negative count) on
 * success and a negative gsvc_rast_status on failure; gsvc_rast_last_error() then returns a
 * thread-local message.  The library never calls cudaMalloc on these paths: scratch comes from the
 * caller (sizes from gsvc_rast_*_bytes) so it can live in the host framework's caching allocator.
 */
#ifndef GSVC_RAST_H
#define GSVC_RAST_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GSVC_RAST_API __attribute__((visibility("default")))
#else
#define GSVC_RAST_API
#endif

#define GSVC_RAST_ABI_VERSION 5
#define GSVC_RAST_TILE 16 /* tile edge in pixels; tile ids are row-major over ceil(W/16) x ceil(H/16) */
#define GSVC_RAST_MAX_VIEWS 16 /* views per batched call (gsvc_rast_*_views) */

typedef enum gsvc_rast_status {
    GSVC_RAST_OK = 0,
    GSVC_RAST_ERR_INVALID = -1,  /* bad argument (null pointer, exclusive-or rules of renderer.py:90-98 violated) */
    GSVC_RAST_ERR_CUDA = -2,     /* a CUDA runtime call or kernel launch failed */
    GSVC_RAST_ERR_CAPACITY = -3, /* binning buffer too small for num_rendered (retry with a larger one) */
    GSVC_RAST_ERR_OVERFLOW = -4  /* num_rendered does not fit 32-bit tile ranges */
} gsvc_rast_status;

/* The 13 fields of GaussianRasterizationSettings (renderer.py:63-83), in the same order. */
typedef struct gsvc_rast_settings {
    int32_t image_height;
    int32_t image_width;
    float x_min;
    float y_min;
    float scale;
    float threshold;          /* TSW slab half-thickness: |view z| > threshold is culled */
    const float *bg;          /* device [3] (pipeline/train.py:328 keeps it on the GPU) */
    float scale_modifier;
    const float *viewmatrix;  /* device 4x4; logical V[r][c] at viewmatrix[r*vm_stride_r + c*vm_stride_c] —
                                 the reference passes a NON-contiguous permuted tensor (renderer.py:77) */
    int64_t vm_stride_r;
    int64_t vm_stride_c;
    int32_t sh_degree;
    float campos[3];          /* host values: the reference keeps campos on the CPU (frame.py:41) */
    int32_t prefiltered;
    int32_t debug;            /* non-zero: synchronise and check for errors after every kernel */
} gsvc_rast_settings;

GSVC_RAST_API int gsvc_rast_abi_version(void);
GSVC_RAST_API const char *gsvc_rast_last_error(void);

/* Scratch sizes in bytes.  geom: per-Gaussian state (P Gaussians, sh_M SH coefficients or 0);
 * image: per-tile / per-pixel state; binning: per-instance state for `capacity` tile instances. */
GSVC_RAST_API size_t gsvc_rast_geom_bytes(int32_t P, int32_t sh_M);
GSVC_RAST_API size_t gsvc_rast_image_bytes(int32_t image_width, int32_t image_height);
GSVC_RAST_API size_t gsvc_rast_image_bytes_views(int32_t image_width, int32_t image_height, int32_t n_views);
GSVC_RAST_API size_t gsvc_rast_binning_bytes(int64_t capacity);
GSVC_RAST_API size_t gsvc_rast_backward_scratch_bytes(int32_t P); /* per-Gaussian gradient accumulators of the blend backward */

/*
 * visible_filter (preprocess.py:99-104): radii[P] int32, 0 = culled (slab / degenerate / off-image).
 * Exactly one of (scales, rotations) or cov3D_precomp ([P,6] xx,xy,xz,yy,yz,zz) must be non-NULL.
 * [range_lo, range_hi) (SURVEY.md §8f row f4, slab-ordered anchors): the caller promises that anchors outside this
 * index range are outside the TSW slab — e.g. anchors kept z-sorted in intervals as the reference's stream codec
 * stores them (utils/encodings.py:827-862) — and the kernel gives them radius 0 without reading them, so the filter
 * costs O(slab) reads.  Anchors inside the range get the exact test.  (0, 0) = no range: every anchor is read.
 */
GSVC_RAST_API int gsvc_rast_visible_filter(const gsvc_rast_settings *st, int32_t P, const float *means3D, const float *scales,
                             const float *rotations, const float *cov3D_precomp, int32_t *radii, int32_t range_lo,
                             int32_t range_hi, void *stream);

/*
 * visible_filter fused with the compaction its caller does next (SURVEY.md §8f row f2): prefilter_voxel returns
 * `radii_pure > 0` (preprocess.py:108) and generate_neural_gaussians indexes every per-anchor tensor with that
 * boolean mask (guassian.py:147-153) — a nonzero pass plus a host synchronisation.  This entry point writes the
 * ascending indices of the visible anchors (exactly nonzero's order): the filter kernel leaves one ballot word per
 * warp and one count per CTA, a single-CTA scan and a write kernel finish the job (no spinning, deterministic), and
 * publishes their count to `count_slot_host` with the ticket protocol of gsvc_rast_forward_launch (read it with
 * gsvc_rast_wait_count: no stream synchronisation).  radii may be NULL.  visible_indices [P] int32 (first `count`
 * entries valid).  scratch: gsvc_rast_compact_scratch_bytes(P) bytes; its first 64-bit word holds the count on
 * the device afterwards.
 */
GSVC_RAST_API size_t gsvc_rast_compact_scratch_bytes(int32_t P);
GSVC_RAST_API int gsvc_rast_visible_filter_compact(const gsvc_rast_settings *st, int32_t P, const float *means3D,
                             const float *scales, const float *rotations, const float *cov3D_precomp, int32_t *radii,
                             int32_t *visible_indices, void *scratch, uint64_t *count_slot_host, uint32_t ticket,
                             int32_t range_lo, int32_t range_hi, void *stream);

/*
 * Forward, launch form (no host synchronisation): preprocess → tile counting → tile scan →
 * instance scatter → per-tile depth sort → front-to-back blend, all enqueued on `stream`.
 * Exactly one of shs ([P,sh_M,3]) / colors_precomp ([P,3]); exactly one of (scales,rotations) /
 * cov3D_precomp.  `binning` holds `capacity` instances (capacity 0 / binning NULL: only the
 * preprocess and scan stages run).
 * num_rendered: `count_slot_host` (may be NULL) is ONE 64-bit word of pinned host memory that the
 * device can address (cudaHostAlloc / torch pin_memory under UVA).  The scan kernel stores
 * (ticket & 0xFFFFFF) << 40 | num_rendered into it the moment the scan ends — well before the blend
 * finishes — so gsvc_rast_wait_count() returns early and the caller can go on enqueueing work.
 * The caller MUST check num_rendered <= capacity; if not, out_color is invalid and
 * gsvc_rast_forward_render must be re-run with a larger binning buffer (geom/image stay valid).
 * `bwd_scratch` (optional): gsvc_rast_backward_scratch_bytes(P) bytes that a later gsvc_rast_backward will
 * use; the preprocess kernel zeroes the entries of the visible Gaussians on the fly (nobody reads the others),
 * which saves the backward a memset launch (pass scratch_is_zero = 1 there).
 * Outputs: out_color [3,H,W], radii [P].
 * All kernels of the chain are launched with programmatic dependent launch (their launch latency and
 * prologue overlap the predecessor's tail).
 */
GSVC_RAST_API int gsvc_rast_forward_launch(const gsvc_rast_settings *st, int32_t P, int32_t sh_M, const float *means3D,
                             const float *shs, const float *colors_precomp, const float *opacities,
                             const float *scales, const float *rotations, const float *cov3D_precomp,
                             void *geom, void *image, void *binning, int64_t capacity, void *bwd_scratch,
                             float *out_color, int32_t *radii, uint64_t *count_slot_host, uint32_t ticket,
                             void *stream);

/* Wait (spin on the pinned word, no stream synchronisation) until the launch with this ticket has
 * published num_rendered; returns it, or a negative status. */
GSVC_RAST_API int64_t gsvc_rast_wait_count(const uint64_t *count_slot_host, uint32_t ticket, void *stream);

/* Re-run the instance scatter / sort / blend stages on existing geom+image state. */
GSVC_RAST_API int gsvc_rast_forward_render(const gsvc_rast_settings *st, int32_t P, const void *geom, void *image, void *binning,
                             int64_t capacity, float *out_color, void *stream);

/*
 * Forward, allocator-callback form (the shape of the upstream binding: three opaque buffers
 * resized through a callback).  `alloc(user, which, bytes)` must return device memory of at least
 * `bytes` (which: 0 geom, 1 binning, 2 image).  Synchronises `stream` once to size the binning
 * buffer exactly.  Returns num_rendered (>= 0) or a negative status.
 */
typedef void *(*gsvc_rast_alloc_fn)(void *user, int32_t which, size_t bytes);
GSVC_RAST_API int64_t gsvc_rast_forward(const gsvc_rast_settings *st, int32_t P, int32_t sh_M, const float *means3D,
                          const float *shs, const float *colors_precomp, const float *opacities,
                          const float *scales, const float *rotations, const float *cov3D_precomp,
                          gsvc_rast_alloc_fn alloc, void *user, float *out_color, int32_t *radii, void *stream);

/*
 * Backward of the forward above.  dL_dout [3,H,W]; geom/image/binning are the buffers the forward
 * filled; `capacity` the instance capacity the binning buffer was laid out with (the value passed to
 * gsvc_rast_forward_launch / _render; max(num_rendered, 1) after gsvc_rast_forward).  Gradient outputs (any may be NULL when the matching input was
 * not given): dL_dmeans3D [P,3], dL_dmeans2D [P,3] (columns 0,1 = dL/dpixel * (0.5 W, 0.5 H), column 2 = 0),
 * dL_dcolors [P,3], dL_dopacities [P], dL_dscales [P,3], dL_drotations [P,4], dL_dcov3D [P,6],
 * dL_dshs [P,sh_M,3].  All outputs are fully overwritten (zeros for culled Gaussians).
 * `dL_packed` (optional, colors_precomp + scale/rotation inputs only): [P,14] rows of
 * (means3D 3, colours 3, opacity 1, scales 3, rotation 4) written INSTEAD of those five dense arrays — the
 * buffer the frame-sharded NCCL all-reduce sums, so no pack pass is needed (SURVEY.md §5).
 * `scratch`: gsvc_rast_backward_scratch_bytes(P) bytes of device memory; scratch_is_zero = 1 promises it is
 * all-zero on entry (as gsvc_rast_forward_launch's bwd_scratch leaves it; a backward dirties it, so a second
 * backward over the same state must pass 0), 0 makes the call clear it first.
 */
GSVC_RAST_API int gsvc_rast_backward(const gsvc_rast_settings *st, int32_t P, int32_t sh_M, int64_t capacity,
                       const float *means3D, const float *shs, const float *colors_precomp, const float *scales,
                       const float *rotations, const float *cov3D_precomp, const int32_t *radii, const void *geom,
                       const void *image, const void *binning, void *scratch, int32_t scratch_is_zero,
                       const float *dL_dout, float *dL_dmeans3D,
                       float *dL_dmeans2D, float *dL_dcolors, float *dL_dopacities, float *dL_dscales,
                       float *dL_drotations, float *dL_dcov3D, float *dL_dshs, float *dL_packed,
                       void *stream);

/*
 * Batched views ("toast" rendering, SURVEY.md §8f row f1).  The reference renders every frame twice — front
 * view, then the x-mirrored back view — flips the second image and averages (pipeline/train.py:353-387,
 * utils/report_utils.py:303-314), and a training iteration does this for two frames: 4 full rasterizer calls on
 * the SAME Gaussians.  These entry points rasterize up to GSVC_RAST_MAX_VIEWS views of one Gaussian set in ONE
 * kernel chain (virtual Gaussian v*P+g, virtual tile v*T+t), blend view v into output image views[v].out_image
 * (mirrored in x if flip_x, scaled by weight; views sharing an image are summed), and the backward returns the
 * parameter gradients SUMMED over the views — exactly what autograd accumulates across the reference's calls.
 * `st` supplies everything the views share (image size, x_min/y_min/scale, threshold, bg, scale_modifier,
 * sh_degree, debug); its viewmatrix/campos are ignored.  Sizes: geom gsvc_rast_geom_bytes(P*n_views, sh_M),
 * image gsvc_rast_image_bytes_views(W,H,n_views), scratch gsvc_rast_backward_scratch_bytes(P*n_views).
 * Outputs: out_color [n_out,3,H,W], radii [n_views,P]; dL_dout [n_out,3,H,W]; dL_dmeans2D [n_views,P,3];
 * every other gradient as in gsvc_rast_backward.  num_rendered (count slot) is the total over the views.
 */
typedef struct gsvc_rast_view {
    const float *viewmatrix;  /* device 4x4, strides as in gsvc_rast_settings */
    int64_t vm_stride_r;
    int64_t vm_stride_c;
    float campos[3];
    int32_t out_image;        /* 0..n_out-1 */
    int32_t flip_x;           /* non-zero: the view lands in (and takes its gradient from) the image mirrored in x */
    float weight;             /* out[out_image] += weight * view */
} gsvc_rast_view;

GSVC_RAST_API int gsvc_rast_forward_views_launch(const gsvc_rast_settings *st, int32_t n_views,
                             const gsvc_rast_view *views_host, int32_t n_out, int32_t P, int32_t sh_M,
                             const float *means3D, const float *shs, const float *colors_precomp,
                             const float *opacities, const float *scales, const float *rotations,
                             const float *cov3D_precomp, void *geom, void *image, void *binning, int64_t capacity,
                             void *bwd_scratch, float *out_color, int32_t *radii, uint64_t *count_slot_host,
                             uint32_t ticket, void *stream);
GSVC_RAST_API int gsvc_rast_forward_views_render(const gsvc_rast_settings *st, int32_t n_views,
                             const gsvc_rast_view *views_host, int32_t n_out, int32_t P, const void *geom,
                             void *image, void *binning, int64_t capacity, float *out_color, void *stream);
GSVC_RAST_API int gsvc_rast_backward_views(const gsvc_rast_settings *st, int32_t n_views, const gsvc_rast_view *views_host,
                             int32_t n_out, int32_t P, int32_t sh_M, int64_t capacity, const float *means3D,
                             const float *shs, const float *colors_precomp, const float *scales,
                             const float *rotations, const float *cov3D_precomp, const int32_t *radii,
                             const void *geom, const void *image, const void *binning, void *scratch,
                             int32_t scratch_is_zero, const float *dL_dout, float *dL_dmeans3D, float *dL_dmeans2D,
                             float *dL_dcolors, float *dL_dopacities, float *dL_dscales, float *dL_drotations,
                             float *dL_dcov3D, float *dL_dshs, float *dL_packed, void *stream);

/*
 * Deterministic blend backward (docs/SPEC.md U14): bit-identical gradients on every run.  The atomic backward adds the
 * sums of every (8x8 block, Gaussian) hit into the Gaussian's accumulator in whatever order the hits land.  These
 * forms store each hit's sums into a slot of `partials` and add every Gaussian's slots in a fixed order (the tiles of
 * its rectangle row-major, then the four blocks of a tile), in double, rounded once.  `partials`:
 * gsvc_rast_backward_partials_bytes(capacity) bytes of device memory, any content (the call clears the part it needs:
 * 4 bytes per instance); 144 bytes per instance of capacity in all.  A NULL or too small buffer is
 * GSVC_RAST_ERR_INVALID before any CUDA work.  `scratch` is fully overwritten, whatever scratch_is_zero says.
 * Each _det entry point takes its twin's arguments plus (partials, partials_bytes) and is otherwise the same call.
 * What stays order-dependent: the forward of a batch that maps three or more views onto one output image (its atomic
 * adds onto the zeroed image), and the exchange's sum over the ranks.
 */
GSVC_RAST_API size_t gsvc_rast_backward_partials_bytes(int64_t capacity);
GSVC_RAST_API int gsvc_rast_backward_views_det(const gsvc_rast_settings *st, int32_t n_views,
                             const gsvc_rast_view *views_host, int32_t n_out, int32_t P, int32_t sh_M, int64_t capacity,
                             const float *means3D, const float *shs, const float *colors_precomp, const float *scales,
                             const float *rotations, const float *cov3D_precomp, const int32_t *radii,
                             const void *geom, const void *image, const void *binning, void *scratch,
                             int32_t scratch_is_zero, const float *dL_dout, float *dL_dmeans3D, float *dL_dmeans2D,
                             float *dL_dcolors, float *dL_dopacities, float *dL_dscales, float *dL_drotations,
                             float *dL_dcov3D, float *dL_dshs, float *dL_packed, void *partials, size_t partials_bytes,
                             void *stream);

/*
 * Batched views over per-view Gaussian sets ("ragged" batches, docs/SPEC.md "Binning").  The reference regenerates its
 * neural Gaussians on every render() call (ortho_gaussian_renderer/guassian.py:147-246: per-view visibility mask,
 * embeddings from the view's camera, training noise), so every view of a training iteration or a decoded frame has a
 * set of its own, of its own size.  These entry points take the views' sets concatenated in view order: counts_host
 * [n_views] (host memory, each >= 0, sum <= 2^31 - 1) in place of P, view v owning rows off_v .. off_v + counts[v] - 1,
 * off_v = counts[0] + ... + counts[v-1].  Row r is rendered in its own view only; the virtual Gaussian is r itself
 * (point_list and export_keys carry r), tiles are v*T+t as for the shared-set batch, and the view map is the same.
 * Per view, the image, radii and instance count are bit-identical to a single-view call on that view's own set.
 * Every per-Gaussian array has sum(counts) rows: inputs, radii [sum], dL_dmeans2D [sum,3] and every parameter gradient,
 * each row its own view's gradient (nothing is summed over views).  Sizes: geom gsvc_rast_geom_bytes(sum, sh_M), image
 * gsvc_rast_image_bytes_views(W,H,n_views), scratch gsvc_rast_backward_scratch_bytes(sum).  No packed gradient and no
 * exchange.  Other arguments as the _views entry points.
 */
GSVC_RAST_API int gsvc_rast_forward_ragged_launch(const gsvc_rast_settings *st, int32_t n_views,
                             const gsvc_rast_view *views_host, int32_t n_out, const int32_t *counts_host, int32_t sh_M,
                             const float *means3D, const float *shs, const float *colors_precomp,
                             const float *opacities, const float *scales, const float *rotations,
                             const float *cov3D_precomp, void *geom, void *image, void *binning, int64_t capacity,
                             void *bwd_scratch, float *out_color, int32_t *radii, uint64_t *count_slot_host,
                             uint32_t ticket, void *stream);
GSVC_RAST_API int gsvc_rast_forward_ragged_render(const gsvc_rast_settings *st, int32_t n_views,
                             const gsvc_rast_view *views_host, int32_t n_out, const int32_t *counts_host,
                             const void *geom, void *image, void *binning, int64_t capacity, float *out_color,
                             void *stream);
GSVC_RAST_API int gsvc_rast_backward_ragged(const gsvc_rast_settings *st, int32_t n_views, const gsvc_rast_view *views_host,
                             int32_t n_out, const int32_t *counts_host, int32_t sh_M, int64_t capacity,
                             const float *means3D, const float *shs, const float *colors_precomp, const float *scales,
                             const float *rotations, const float *cov3D_precomp, const int32_t *radii,
                             const void *geom, const void *image, const void *binning, void *scratch,
                             int32_t scratch_is_zero, const float *dL_dout, float *dL_dmeans3D, float *dL_dmeans2D,
                             float *dL_dcolors, float *dL_dopacities, float *dL_dscales, float *dL_drotations,
                             float *dL_dcov3D, float *dL_dshs, void *stream);
GSVC_RAST_API int gsvc_rast_backward_ragged_det(const gsvc_rast_settings *st, int32_t n_views,
                             const gsvc_rast_view *views_host, int32_t n_out, const int32_t *counts_host, int32_t sh_M,
                             int64_t capacity, const float *means3D, const float *shs, const float *colors_precomp,
                             const float *scales, const float *rotations, const float *cov3D_precomp,
                             const int32_t *radii, const void *geom, const void *image, const void *binning,
                             void *scratch, int32_t scratch_is_zero, const float *dL_dout, float *dL_dmeans3D,
                             float *dL_dmeans2D, float *dL_dcolors, float *dL_dopacities, float *dL_dscales,
                             float *dL_drotations, float *dL_dcov3D, float *dL_dshs, void *partials,
                             size_t partials_bytes, void *stream);

/*
 * Densification statistic of the step at the rasterizer boundary.  The reference calls
 * GaussianModel.training_statis once per rendered view (pipeline/train.py:559-565); per view it takes the norm of
 * the screen-space gradient of the Gaussians that were drawn — `torch.norm(viewspace_points.grad[radii > 0, :2])`,
 * scene/gaussian_model.py:1311 — and adds it, and a count of 1, into per-offset accumulators (:1313-1314).  This is
 * the rasterizer-side half for all views of a step in one stream pass:
 *     stats[g*stride + 0] (+)= sum_v [radii[v*P+g] > 0] * |dL_dmeans2D[v][g][0:2]|
 *     stats[g*stride + 1] (+)= sum_v [radii[v*P+g] > 0]
 * dL_dmeans2D [n_views,P,3] and radii [n_views,P] as gsvc_rast_backward_views / gsvc_rast_forward_views_launch write
 * them (n_views = 1: the single-view call's [P,3] and [P]).  accumulate = 0 overwrites, 1 adds.  Under frame
 * sharding the [P,2] rows are summed over the ranks with the gradients (gsvc_b200/sharding.py), which gives every
 * rank the statistic of ALL the step's views: densification decisions stay identical across ranks.
 */
GSVC_RAST_API int gsvc_rast_densify_stats(int32_t n_views, int32_t P, const float *dL_dmeans2D, const int32_t *radii,
                            float *stats, int64_t stride, int32_t accumulate, void *stream);

/*
 * Sum all-reduce of a rank-sharded step's fp32 buffer (the packed [P,14] parameter gradients, optionally followed by
 * the [P,2] densification statistic) through the NVSwitch — the one exchange step of the frame-sharded training
 * loop (what DistributedDataParallel's gradient all-reduce would be for /root/reference/pipeline/train.py:462; the
 * reference itself trains on one GPU).  ONE kernel launch per rank, no NCCL.  Rank r owns the r-th slice of the
 * buffer: it obtains the slice's sum over the ranks and writes it into every rank's buffer, either
 *   - through the MULTICAST mapping of the buffers (multicast != NULL): multimem.ld_reduce / multimem.st — the
 *     switch adds and replicates, each GPU's links carry the buffer once out and once in; or
 *   - with peer loads and stores over NVLink (multicast == NULL, buffers != NULL; 2, 4 or 8 ranks).
 *   multicast     the buffer's address in the multicast mapping of a symmetric allocation every rank of the node
 *                 has made with the same size (e.g. torch.distributed._symmetric_memory: handle.multicast_ptr);
 *                 16-byte aligned; NULL selects the peer path
 *   buffers       device array of `world` pointers: buffers[q] = rank q's buffer as mapped into THIS process
 *                 (handle.buffer_ptrs_dev); may be NULL when multicast is given
 *   signal_pads   device array of `world` pointers: signal_pads[q] = rank q's zero-initialised signal pad as mapped
 *                 into THIS process (handle.signal_pad_ptrs_dev), each at least world * 4 bytes
 *   state         GSVC_RAST_EXCHANGE_STATE_WORDS zeroed 32-bit words of this rank's OWN device memory, private to this
 *                 buffer (the CTAs of the launch meet there); zero again when the kernel has completed — except the
 *                 LAST word, which counts waits that gave up: every wait of the exchange is bounded (~20 s), so a
 *                 rank that never arrives leaves a wrong buffer and a non-zero count instead of a spinning GPU
 *   numel         floats in the buffer, a multiple of 4
 *   n_ctas        CTAs of the launch (all of them must be co-resident: <= 4 * SM count)
 * On return of the kernel every rank's buffer holds the sum over the ranks, bit-identical on all of them (one adder
 * per element).  Every rank must make the call (it is a collective); the pad words are back to zero afterwards, so
 * the launch can be captured in a CUDA graph and replayed.
 */
#define GSVC_RAST_EXCHANGE_MAX_CHUNKS 62
#define GSVC_RAST_EXCHANGE_STATE_WORDS (2 + GSVC_RAST_EXCHANGE_MAX_CHUNKS + 1)
GSVC_RAST_API int gsvc_rast_switch_allreduce(void *multicast, void *buffers, void *signal_pads, void *state, int32_t rank,
                               int32_t world, int64_t numel, int32_t n_ctas, void *stream);

/*
 * The backward of a batch of views WITH the exchange of a frame-sharded step in the same launches: the per-Gaussian
 * backward writes the packed [P,14] rows (dL_packed, required) of THIS rank's frames, and the first `n_ctas` CTAs of
 * that same kernel sum the rows over the ranks — chunk by chunk, while the other CTAs are still computing the later
 * chunks — so the call ends with the all-reduced buffer in place on every rank (bit-identical) and most of the transfer
 * hidden under the computation.  dL_packed must be this rank's part of a symmetric allocation as for
 * gsvc_rast_switch_allreduce (same meaning of multicast / buffers / signal_pads / rank / world; the pads must hold
 * world * (1 + chunks) words); P must be even.
 *   state        GSVC_RAST_EXCHANGE_STATE_WORDS zeroed 32-bit words of this rank's own device memory (as above)
 *   n_ctas       CTAs of the exchange role (128 threads each: one coordinator + the movers; 0 selects 65)
 *   chunk_rows   Gaussians per chunk, a multiple of 128 (0 selects ~1/4 of P); the same on every rank
 * Every rank must make the call with the same P.  All other arguments as gsvc_rast_backward_views.
 */
typedef struct gsvc_rast_exchange {
    void *multicast;     /* dL_packed through the multicast mapping, or NULL: peer loads and stores */
    void *buffers;       /* device array of `world` pointers: every rank's dL_packed as mapped here */
    void *signal_pads;   /* device array of `world` pointers: every rank's signal pad as mapped here */
    void *state;
    int32_t rank;
    int32_t world;
    int32_t n_ctas;
    int32_t chunk_rows;
} gsvc_rast_exchange;

GSVC_RAST_API int gsvc_rast_backward_views_exchange(const gsvc_rast_settings *st, int32_t n_views,
                             const gsvc_rast_view *views_host, int32_t n_out, int32_t P, int32_t sh_M, int64_t capacity,
                             const float *means3D, const float *shs, const float *colors_precomp, const float *scales,
                             const float *rotations, const float *cov3D_precomp, const int32_t *radii, const void *geom,
                             const void *image, const void *binning, void *scratch, int32_t scratch_is_zero,
                             const float *dL_dout, float *dL_dmeans2D, float *dL_packed,
                             const gsvc_rast_exchange *exchange, void *stream);
/* the deterministic form (gsvc_rast_backward_views_det); the sum over the ranks is not part of its promise */
GSVC_RAST_API int gsvc_rast_backward_views_exchange_det(const gsvc_rast_settings *st, int32_t n_views,
                             const gsvc_rast_view *views_host, int32_t n_out, int32_t P, int32_t sh_M, int64_t capacity,
                             const float *means3D, const float *shs, const float *colors_precomp, const float *scales,
                             const float *rotations, const float *cov3D_precomp, const int32_t *radii, const void *geom,
                             const void *image, const void *binning, void *scratch, int32_t scratch_is_zero,
                             const float *dL_dout, float *dL_dmeans2D, float *dL_packed,
                             const gsvc_rast_exchange *exchange, void *partials, size_t partials_bytes, void *stream);

/*
 * Stage exports for bit-exact parity tests (not used on the hot path).
 * keys: sorted_keys [R] = (tile << 32) | depth_key, point_list [R], ranges [T,2] (untouched tiles 0,0).
 * geom: depth [P], xy [P,2], conic_opacity [P,4], rgb [P,3], rect [P,4] int32 (minx,miny,maxx,maxy tiles).
 * image: final_T [H,W], n_contrib [H,W].  Any output pointer may be NULL.
 * For state made by a batched call pass its n_views (keys then carry the virtual tile v*T+t, point_list the
 * virtual Gaussian v*P+g, ranges is [n_views*T,2], final_T / n_contrib are [n_views,H,W]; export_geom takes
 * P*n_views); 1 otherwise.
 */
GSVC_RAST_API int gsvc_rast_export_keys(const gsvc_rast_settings *st, int32_t n_views, int64_t capacity, const void *image,
                          const void *binning, uint64_t *sorted_keys, uint32_t *point_list, uint32_t *ranges, void *stream);
GSVC_RAST_API int gsvc_rast_export_geom(int32_t P, int32_t sh_M, const void *geom, float *depth, float *xy, float *conic_opacity,
                          float *rgb, int32_t *rect, void *stream);
GSVC_RAST_API int gsvc_rast_export_image(const gsvc_rast_settings *st, int32_t n_views, const void *image, float *final_T,
                           uint32_t *n_contrib, void *stream);

/*
 * Optional per-stage device timing (tracing aid; used by bench.py for the roofline numbers).
 * gsvc_rast_stage_timing(1) makes every later call (any thread) bracket each stage with CUDA
 * events on the launching stream (no host synchronisation); gsvc_rast_stage_times() waits for them
 * and writes the MEAN duration of each stage in milliseconds over the calls made since the previous
 * query (the last 256 at most; -1 if the stage did not run):
 *   [0] preprocess  [1] tile_scan  [2] scatter  [3] sort_tiles  [4] render_forward
 *   [5] render_backward  [6] preprocess_backward  [7] visible_filter
 * Returns the number of stages (8).
 */
#define GSVC_RAST_NUM_STAGES 8
GSVC_RAST_API int gsvc_rast_stage_timing(int32_t enable);
GSVC_RAST_API int gsvc_rast_stage_times(float *ms_host);

/* Launches whose instance capacity was exceeded since the last reset (current device): their output is invalid.
 * Only launches enqueued while gsvc_rast_count_overflows(1) is in effect on the calling thread are counted — the
 * caller sets it around the launches it captures into a CUDA graph, whose replays nobody re-runs; an eager forward
 * detects an overflow from num_rendered and re-runs by itself.  gsvc_rast_overflow_events synchronises `stream`. */
GSVC_RAST_API int gsvc_rast_count_overflows(int32_t enable);
GSVC_RAST_API int64_t gsvc_rast_overflow_events(int32_t reset, void *stream);

/* Number of kernel launches issued by this library (all threads) since the last reset
 * (bench.py reports it as gpu_launches). */
GSVC_RAST_API int64_t gsvc_rast_launch_count(int32_t reset);

/*
 * Fused epilogue of the neural-Gaussian generator (SURVEY.md 8f row f2): everything
 * /root/reference/ortho_gaussian_renderer/guassian.py does between its four per-anchor MLPs and the rasterizer call —
 * the boolean-mask gathers of the visible anchors' rows (:147-153), opacity * mask and the opacity > 0 selection
 * (:251-258), the repeat / cat / mask-index / split of a [N_vis*K, 22] tensor (:275-281), scaling = s[3:6] *
 * sigmoid(.), rot = normalize(.), xyz = clamp(anchor + (offset + neural_offset) * s[0:3]) (:285-293) — as one marking
 * pass, the filter's compaction scan and one writing pass.
 *   visible_indices [n_vis] ascending anchor rows (gsvc_rast_visible_filter_compact), or NULL when the per-anchor
 *       inputs are already gathered ([n_vis, ...]);
 *   anchor [N,3], grid_offsets [N,K,3], grid_scaling [N,6], masks [N,K]: the model's (activated) per-anchor tensors;
 *   neural_opacity [n_vis,K], color [n_vis,K*3], scale_rot [n_vis,K*7], neural_offset [n_vis,K*3]: the MLP outputs;
 *   bound_min / bound_max [3] (device): the clamp of guassian.py:293.
 * Outputs, rows in the reference's order (anchor-major, offset-minor, selected ones only), each with room for
 * n_vis*K rows: xyz [.,3], color_out [.,3], opacity_out [.], scaling_out [.,3], rot_out [.,4]; plus, per (anchor,
 * offset): neural_opacity_full [n_vis*K] (= opacity * mask, what the reference returns as `neural_opacity`),
 * selection_mask [n_vis*K] (uint8, its `mask`) and rank [n_vis*K] (compact row or -1; the backward reads it).
 * The number of selected Gaussians is published like num_rendered: ticket << 40 | count in count_slot_host
 * (gsvc_rast_wait_count).  scratch: gsvc_gen_epilogue_scratch_bytes(n_vis, K) bytes.
 *
 * gsvc_gen_epilogue_backward: gradients w.r.t. the MLP outputs ([n_vis,...] like the inputs) and, per VISIBLE anchor,
 * w.r.t. anchor [n_vis,3], grid_offsets [n_vis,K,3], grid_scaling [n_vis,6], masks [n_vis,K] (the caller scatters
 * these rows to the full tensors: the gather's backward).  dL_dnop_full may be NULL.  One pass, no atomics.
 */
GSVC_RAST_API size_t gsvc_gen_epilogue_scratch_bytes(int32_t n_vis, int32_t K);
GSVC_RAST_API int gsvc_gen_epilogue_forward(int32_t n_vis, int32_t K, const int32_t *visible_indices, const float *anchor,
                                            const float *grid_offsets, const float *grid_scaling, const float *masks,
                                            const float *neural_opacity, const float *color, const float *scale_rot,
                                            const float *neural_offset, const float *bound_min, const float *bound_max,
                                            float *xyz, float *color_out, float *opacity_out, float *scaling_out,
                                            float *rot_out, float *neural_opacity_full, uint8_t *selection_mask,
                                            int32_t *rank, void *scratch, uint64_t *count_slot_host, uint32_t ticket,
                                            void *stream);
GSVC_RAST_API int gsvc_gen_epilogue_backward(int32_t n_vis, int32_t K, const int32_t *visible_indices, const float *anchor,
                                             const float *grid_offsets, const float *grid_scaling, const float *masks,
                                             const float *neural_opacity, const float *scale_rot,
                                             const float *neural_offset, const float *bound_min, const float *bound_max,
                                             const int32_t *rank, const float *dL_dxyz, const float *dL_dcolor,
                                             const float *dL_dopacity, const float *dL_dscaling, const float *dL_drot,
                                             const float *dL_dnop_full, float *d_neural_opacity, float *d_color,
                                             float *d_scale_rot, float *d_neural_offset, float *d_anchor,
                                             float *d_grid_offsets, float *d_grid_scaling, float *d_masks, void *stream);

/*
 * Photometric training loss (docs/SPEC.md "Photometric loss", decision U9): the L1 + D-SSIM term of the reference's
 * iteration (pipeline/train.py:407-444, the upstream 3DGS ssim of utils/loss_utils.py:41-72), fused.  For each image n
 * of x = image, y = target, both [n_images,3,H,W] fp32:
 *     loss[n] = (1 - lambda) * mean|x - y| + lambda * (1 - mean S)        means over the image's 3*H*W values
 *     S = (2 mu_x mu_y + C1)(2 sigma_xy + C2) / ((mu_x^2 + mu_y^2 + C1)(sigma_x^2 + sigma_y^2 + C2))
 * with the moments taken per channel through the 11x11 Gaussian window (sigma 1.5) with zero padding of 5 (F.conv2d
 * semantics), C1 = 0.01^2, C2 = 0.03^2.  lambda_dssim in [0, 1] (upstream default 0.2; 0 = L1, 1 = 1 - SSIM).
 *   gsvc_rast_loss_forward   writes loss [n_images] (device).  scratch: gsvc_rast_loss_scratch_bytes(n_images, H, W)
 *                            bytes for the per-CTA partial sums (their per-image sum runs in a fixed order: the result
 *                            is bit-reproducible).  Two launches.
 *   gsvc_rast_loss_backward  writes dL_dimage [n_images,3,H,W] = dL_dloss[n] * d loss[n] / d image, dL_dloss [n_images]
 *                            read on the device (no host synchronisation).  It recomputes the moments from image and
 *                            target (the forward leaves nothing behind) and needs no scratch.  One launch, no atomics.
 * The target gets no gradient.  d|x - y|/dx is 0 where x == y.
 */
GSVC_RAST_API size_t gsvc_rast_loss_scratch_bytes(int32_t n_images, int32_t H, int32_t W);
GSVC_RAST_API int gsvc_rast_loss_forward(int32_t n_images, int32_t H, int32_t W, const float *image, const float *target,
                                         float lambda_dssim, float *loss, void *scratch, void *stream);
GSVC_RAST_API int gsvc_rast_loss_backward(int32_t n_images, int32_t H, int32_t W, const float *image,
                                          const float *target, float lambda_dssim, const float *dL_dloss,
                                          float *dL_dimage, void *stream);

/*
 * Frame quality metrics (docs/SPEC.md "Evaluation metrics", decision U10): the PSNR / SSIM / MS-SSIM of an evaluation
 * loop, on the device.  For each image n of x = image, y = target, both [n_images,3,H,W] fp32, with x clamped to
 * [0, 1] on read and y read as given (data range 1):
 *     psnr    = 10 log10(1 / mse), mse = mean (x - y)^2 over the image's 3*H*W values (summed in double); +inf if 0
 *     ssim    = mean S, S as in the loss block above (zero padding of 5, 11x11 window, sigma 1.5)
 *     ms_ssim = mean_c prod_{l<4} relu(cs_{l,c})^{w_l} * relu(ssim_{4,c})^{w_4},  w = (0.0448, 0.2856, 0.3001, 0.2363,
 *               0.1333): pytorch_msssim's ms_ssim(data_range=1).  Per level l and channel c, cs and ssim are the means of
 *               (2 sigma_xy + C2) / (sigma_x^2 + sigma_y^2 + C2) and of S over the VALID (unpadded) window positions;
 *               level l+1 is avg_pool2d(level l, 2, stride 2, padding (h % 2, w % 2)) of x and y.  NaN unless
 *               min(H, W) > 160.
 *   gsvc_rast_quality  writes quality [n_images,3] = (psnr, ssim, ms_ssim) (device).  scratch:
 *                      gsvc_rast_quality_scratch_bytes(n_images, H, W) bytes for the pooled levels 1-4 (a third of the
 *                      pixels of an image pair) and the per-CTA partial sums, which are summed per image in a fixed
 *                      order: the results are bit-reproducible.  Six launches (two when min(H, W) <= 160), no atomics,
 *                      no host synchronisation.
 */
GSVC_RAST_API size_t gsvc_rast_quality_scratch_bytes(int32_t n_images, int32_t H, int32_t W);
GSVC_RAST_API int gsvc_rast_quality(int32_t n_images, int32_t H, int32_t W, const float *image, const float *target,
                                    float *quality /* [n_images,3]: psnr, ssim, ms_ssim */, void *scratch, void *stream);

/*
 * 8-bit frame export (docs/SPEC.md "8-bit frame export", decision U11): composed frames to the bytes an image writer
 * takes.  image is [n_images,3,H,W] fp32 (planar, as render_toast / the views chain write it); out is [n_images,H,W,3]
 * uint8, RGB interleaved, row 0 first, device-addressable.  Every value x becomes
 *     q = uint8(min(max(fl(fl(x * 255) + 0.5), 0), 255))      truncated; NaN -> 0, +inf -> 255, -inf -> 0
 * with the product and the sum rounded separately (never fused): torchvision's save_image arithmetic.  One launch, no
 * scratch, no atomics, no host synchronisation (capturable in a CUDA graph).  n_images, H, W >= 1, image and out non-
 * NULL and n_images * H * W * 3 within a 64-bit index, else GSVC_RAST_ERR_INVALID before any CUDA work.  Fastest
 * when H * W % 4 == 0, image is 16-byte and out 4-byte aligned; any other size or alignment is handled too.
 */
GSVC_RAST_API int gsvc_rast_frames_rgb8(int32_t n_images, int32_t H, int32_t W, const float *image,
                                        uint8_t *out /* [n_images,H,W,3], device-addressable */, void *stream);

/*
 * 8-bit source frames as targets (docs/SPEC.md "8-bit source frames", decision U12): the loss and quality calls above
 * with the target read from a cube of 8-bit frames instead of an fp32 [n_images,3,H,W] tensor.  frames is
 * [n_frames,H,W,3] uint8, RGB interleaved, row 0 first (what frames_rgb8 writes and np.array(PIL.Image) holds), device-
 * addressable, any alignment.  Image n is compared with frame frame_index[n] (frame_index: [n_images] int32 on the
 * device, read by the kernels, so a captured graph picks new frames through an in-place write), or with frame n when
 * frame_index is NULL (then n_images <= n_frames).  A byte q reads as y = fl(q / 255), one correctly rounded division
 * (torchvision's to_tensor): every result equals the fp32 call's with that target, bit for bit.  An index outside
 * [0, n_frames) is never dereferenced: that image's loss and quality row are NaN and its dL_dimage is 0; the other
 * images are unaffected.  Scratch sizes, launch counts and the size and lambda rules are those of the fp32 calls; a
 * NULL pointer, n_frames < 1, a NULL frame_index with n_images > n_frames or n_frames * H * W * 3 beyond a 64-bit index
 * is GSVC_RAST_ERR_INVALID too, before any CUDA work.
 */
GSVC_RAST_API int gsvc_rast_loss_forward_rgb8(int32_t n_images, int32_t H, int32_t W, const float *image,
                                              const uint8_t *frames /* [n_frames,H,W,3] */, int32_t n_frames,
                                              const int32_t *frame_index /* [n_images] device, or NULL */,
                                              float lambda_dssim, float *loss, void *scratch, void *stream);
GSVC_RAST_API int gsvc_rast_loss_backward_rgb8(int32_t n_images, int32_t H, int32_t W, const float *image,
                                               const uint8_t *frames, int32_t n_frames, const int32_t *frame_index,
                                               float lambda_dssim, const float *dL_dloss, float *dL_dimage,
                                               void *stream);
GSVC_RAST_API int gsvc_rast_quality_rgb8(int32_t n_images, int32_t H, int32_t W, const float *image,
                                         const uint8_t *frames, int32_t n_frames, const int32_t *frame_index,
                                         float *quality /* [n_images,3] */, void *scratch, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GSVC_RAST_H */
