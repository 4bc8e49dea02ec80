/*
 * rodygs_b200 — C ABI of the B200-native dynamic-splatting hot path.
 *
 * This is the drop-in boundary for the native module the reference imports as
 * `diff_gauss_pose` (un-vendored submodule, /root/reference/.gitmodules:1-4).
 * The reference reaches that module only through
 *   GaussianRasterizationSettings(...)      /root/reference/src/trainer/renderer.py:50-63
 *   GaussianRasterizer(...)(means3D=...)    /root/reference/src/trainer/renderer.py:65-101
 * (twins at src/model/rodygs_static.py:221-281 and src/evaluator/eval.py:118-176);
 * upstream binds it with pybind11 (`_C.rasterize_gaussians`,
 * `_C.rasterize_gaussians_backward`).  The entry points below are what that
 * binding would call instead; rodygs_b200/_lib.py loads them with ctypes.
 *
 * Conventions
 *  - plain C: raw device pointers, sizes, a cudaStream_t passed as void*.
 *  - every function returns 0 on success; otherwise a negative RDG_E_* code and
 *    rdg_last_error() (thread-local) describes the failure.
 *  - the library owns no device memory; every buffer (inputs, outputs,
 *    workspaces) is allocated by the caller (torch's caching allocator).
 *  - all launches go to the given stream; no call synchronises the host.
 *  - matrices are passed the way the reference passes them: "glm storage",
 *    i.e. the 16 floats of M^T row-major == M column-major
 *    (renderer.py:57 `projection_matrix.transpose(0, 1)`, :97-99 viewmatrix).
 *  - float = IEEE binary32 everywhere.
 */
#ifndef RODYGS_B200_H
#define RODYGS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RDG_ABI_VERSION 8
#define RDG_TILE 16
#define RDG_NUM_BASIS_MAX 16

enum {
    RDG_OK = 0,
    RDG_E_ARG = -1,      /* bad argument (null pointer, size, unsupported option) */
    RDG_E_CUDA = -2,     /* a CUDA runtime call / launch failed */
    RDG_E_CAPACITY = -3  /* workspace smaller than rdg_*_workspace_bytes() says */
};

/* One set of Gaussians.  For the drop-in boundary (already activated, already
 * concatenated tensors: renderer.py:88-100) only `st` is used with
 * n_dynamic = 0 and raw = 0.  For the fused path (raw parameters, static and
 * dynamic models never concatenated: replaces rodygs.py:68-113 +
 * rodygs_static.py:82-105 + rodygs_dynamic.py:122-138) `st` is the static
 * model, `dy` the dynamic one, raw = 1. */
typedef struct RdgSet {
    const float* xyz;       /* [n,3] */
    const float* scaling;   /* [n,3]  raw: log-scale; activated: scale */
    const float* rotation;  /* [n,4]  (r,x,y,z) raw: un-normalised */
    const float* opacity;   /* [n,1]  raw: logit; activated: opacity */
    const float* sh_dc;     /* [n, sh_dc_stride]   first 3 floats = degree-0 coefficients (r,g,b) */
    const float* sh_rest;   /* [n, sh_rest_stride] first 3*(K-1) floats = higher coefficients, coefficient-major */
    int32_t sh_dc_stride;   /* floats between consecutive Gaussians (3 for _features_dc, 48 for a cat'ed [n,16,3]) */
    int32_t sh_rest_stride; /* 45 for _features_rest, 48 for a cat'ed [n,16,3] (pointer = base + 3) */
} RdgSet;

typedef struct RdgScene {
    int64_t n_static;
    int64_t n_dynamic;
    RdgSet st;
    RdgSet dy;
    int32_t raw;                 /* 1: apply exp / normalize / sigmoid inside the kernel */
    const float* colors_precomp; /* [N,3] or NULL; if set, SH is ignored (renderer.py:78-83) */
    /* time-conditioned deformation of the dynamic set (raw = 1 only) */
    int32_t use_deform;          /* rodygs.py:69-73 `use_deform` */
    int32_t num_basis;           /* <= RDG_NUM_BASIS_MAX */
    int32_t num_times;           /* T */
    const float* motion_coeff;   /* [n_dynamic, num_basis]  (_motion_coeff [n,1,K]) */
    const int32_t* time_ind;     /* [n_dynamic] birth-frame index (gaussian_to_time_ind) */
    const float* basis_t;        /* [num_basis,7]  B(t) for this view's time */
    const float* table;          /* [T,num_basis,7] B at every training time (get_total_motion_table) */
    float spatial_lr_scale;
    /* optional CSR of the dynamic Gaussians by birth frame (built once per time_ind by the host:
     * frame_order = stable argsort(time_ind) [n_dynamic], frame_offsets [T+1]).  With it the backward
     * pass reduces dL/dtable per frame without atomics on the hot path; without it (NULL) it falls
     * back to shared-memory atomics. */
    const int32_t* frame_order;
    const int32_t* frame_offsets;
} RdgScene;

typedef struct RdgView {
    int32_t height, width;
    float tanfovx, tanfovy;
    float scale_modifier;
    int32_t sh_degree;           /* 0..3 */
    int32_t enable_cov_grad;     /* pose gradient through the covariance path */
    int32_t enable_sh_grad;      /* pose gradient through the camera position (SH view direction) */
    const float* viewmatrix;     /* device, 16 floats, glm storage */
    const float* projmatrix;     /* device, 16 floats, glm storage (perspective only, renderer.py:57) */
    const float* bg;             /* device, 3 floats */
} RdgView;

/* Per-Gaussian screen-space state written by preprocess, read by binning,
 * blend and the backward pass.  All arrays have N = n_static + n_dynamic rows. */
typedef struct RdgGeom {
    int32_t* radii;          /* [N]   0 = culled */
    uint32_t* tiles_touched; /* [N] */
    float* p0;               /* [N,4] px, py, conic A, conic B */
    float* p1;               /* [N,4] conic C, opacity, r, g */
    float* p2;               /* [N,2] b, view-space depth */
    uint8_t* clamped;        /* [N]   bit c set = channel c clamped at 0 */
    float* dbg_activated;    /* optional [N,11] (xyz, scale, quat, opacity) as used by the kernel; NULL to skip */
    uint32_t* tile_count;    /* optional [tiles+1]: preprocess counts the Gaussians touching each tile (zeroed inside);
                              * required by rdg_bin_tiles */
} RdgGeom;

/* Tile-binning result. */
typedef struct RdgBins {
    uint64_t* keys_sorted;   /* [D_cap] (tile << 32) | float_bits(depth) */
    uint32_t* vals_sorted;   /* [D_cap] Gaussian id */
    uint32_t* ranges;        /* [tiles,2] [start,end) */
    uint32_t* point_offsets; /* [N] inclusive scan of tiles_touched */
    uint32_t* num_rendered;  /* [2]: [0] = D (sum tiles_touched), [1] = 1 if D > D_cap (nothing past D_cap is written) */
    uint64_t* keys_unsorted; /* optional [D_cap] for tests; NULL to use workspace */
    uint32_t* vals_unsorted; /* optional [D_cap] */
    /* Region lists, written by rdg_blend_fwd and read back by rdg_blend_bwd (required by both).  A region is a 16x8-pixel
     * half tile (the unit one warp blends); region r of tile t holds, in depth order, the entries of the tile's list
     * whose alpha >= 1/255 ellipse can reach it, with the 8-bit mask of the 4x4-pixel sub-tiles it reaches:
     *   region_ids  [2 * region_stride]  entry k of region (t, r) at r * region_stride + ranges[t][0] + k
     *   region_masks[2 * region_stride]  same indexing
     *   region_count[2 * tiles]          entries of region (t, r) at 2 t + r
     * region_stride >= D_cap.  RdgImage.n_contrib counts positions of the REGION list. */
    uint32_t* region_ids;
    uint8_t* region_masks;
    uint32_t* region_count;
    int64_t region_stride;
} RdgBins;

typedef struct RdgImage {
    float* color;        /* [3,H,W] */
    float* depth;        /* [1,H,W] */
    float* alpha;        /* [1,H,W] */
    float* final_T;      /* [H,W] */
    uint32_t* n_contrib; /* [H,W] */
} RdgImage;

/* Gradients w.r.t. one RdgSet (same shapes/strides as the inputs). NULL = skip. */
typedef struct RdgSetGrad {
    float* xyz; float* scaling; float* rotation; float* opacity; float* sh_dc; float* sh_rest;
} RdgSetGrad;

typedef struct RdgSceneGrad {
    RdgSetGrad st;
    RdgSetGrad dy;
    float* colors_precomp;   /* [N,3] or NULL */
    float* means2D;          /* [N,3] gradient sink (renderer.py:38-44), per NDC unit; z column = 0 */
    float* viewmatrix;       /* [16] glm storage, accumulated (+=): zero it before the call */
    float* motion_coeff;     /* [n_dynamic,num_basis] */
    float* table;            /* [T,num_basis,7] accumulated (+=) */
    float* basis_t;          /* [num_basis,7]   accumulated (+=) */
    float* g7_scratch;       /* [n_dynamic,8] scratch, required when scene.frame_order is set */
    int32_t models;          /* 0 or 3: both models; 1: the static model only; 2: the dynamic model only.
                              * The data-parallel step calls rdg_preprocess_bwd once per model (or per part of a model) so that the
                              * all-reduce of the ranges already written runs under the next launch (viewmatrix accumulates). */
    int32_t part, parts;     /* parts > 1: only the part-th of `parts` equal pieces of the selected chunk range (256-Gaussian chunks:
                              * piece boundaries are multiples of 256 rows of the model); 0 / 0 = everything */
    int32_t dtable_mode;     /* dL/dtable + dL/dB(t) reduction over the birth-frame CSR (needs every dynamic part's g7 rows):
                              * 0 = after the dynamic model's last part (default), 1 = skip, 2 = ONLY it (no per-Gaussian kernel) */
    uint32_t* sm_queue;      /* optional device scratch, 4 uint32, ZERO on first use (the kernel leaves it zero): with the "sm_reserve"
                              * tunable > 0 the persistent kernel then runs SM-partitioned - CTAs that land on the reserved SMs exit,
                              * the others draw chunks from this counter - so that a collective on another stream finds free SMs */
    float* dcolor;           /* optional [N,3]: dL/d(rgb) of every Gaussian after the SH clamp mask (zeros when it is not
                              * visible) - the 12-byte factors from which rdg_sh_grad_views rebuilds dL/dSH of all views
                              * of a data-parallel step; pass st/dy.sh_dc = sh_rest = NULL with it to skip the dSH rows */
} RdgSceneGrad;

int rdg_abi_version(void);
const char* rdg_last_error(void);
/* number of kernels this library has launched in this process (bench.py's `gpu_launches`). */
uint64_t rdg_launch_count(void);
/* A/B switches and test knobs of the launchers (process-wide; initial value from the environment variable RDG_<NAME>):
 *   "pre_grid_cap" > 0: cap on the persistent grid of the two preprocess kernels (tests: forces many chunks per CTA)
 *   "dtable_v1"    1: first version of the dL/dtable reduction
 *   "diff_smem"    1 (default): the preprocess kernels keep B(t) - table rows in shared memory when num_times <= 140;
 *                  0: every dynamic Gaussian gathers its 448-byte table row from global memory
 *   "sm_reserve"   n > 0: rdg_preprocess_bwd and rdg_sh_grad_views size their persistent grids for 148 - n SMs, leaving the rest
 *                  to a collective (NCCL) that runs beside them on another stream (their CTAs take the whole register file)
 *   "deterministic" 1: rdg_preprocess_bwd runs its kernels with one CTA so that the cross-CTA float atomics of dL/dV,
 *                  dL/dtable and dL/dB(t) land in a fixed order (test mode, slow; pair it with rdg_blend_bwd_deterministic)
 *   "l2_prefetch"  1: the persistent per-Gaussian kernels prefetch the next chunk's parameter rows into L2 with
 *                  cp.async.bulk.prefetch.L2 while the current chunk is computed (measured neutral at config 4: 0.218 / 0.396 ms
 *                  against 0.215 / 0.400 ms for the forward / backward kernel - off by default)
 *   "ar_unroll"    2 / 4 (default) / 8: 16-byte vectors each thread of rdg_allreduce_multimem keeps in flight
 * Returns RDG_E_ARG for an unknown name. */
int rdg_set_tunable(const char* name, int32_t value);

/* ---- forward ------------------------------------------------------------ */

/* deformation + activations + EWA projection + SH->RGB (SURVEY.md §8 a2-a7). */
int rdg_preprocess_fwd(const RdgScene* scene, const RdgView* view, const RdgGeom* geom, void* stream);

/* bytes of scratch rdg_bin needs for N Gaussians and at most d_cap duplicates. */
int64_t rdg_bin_workspace_bytes(int64_t n, int64_t d_cap, int32_t height, int32_t width);

/* Same result (sorted values, sorted keys, ranges, duplicate count) as rdg_bin, computed the B200 way:
 * per-tile counts come from preprocess (geom->tile_count), a tiny scan turns them into tile segments
 * (= the ranges), instances are dropped into their tile's segment with one returning atomic each and
 * every tile is then sorted by (depth bits, Gaussian id) inside ONE CTA in shared memory - two passes
 * over the duplicates in HBM instead of ten.  bins->point_offsets / keys_unsorted / vals_unsorted are not
 * produced (they only exist in the emission order of rdg_bin); bins->keys_sorted may be NULL. */
int64_t rdg_bin_tiles_workspace_bytes(int64_t n, int64_t d_cap, int32_t height, int32_t width);
int rdg_bin_tiles(int64_t n, const RdgGeom* geom, int32_t height, int32_t width, int64_t d_cap,
                  const RdgBins* bins, void* workspace, int64_t workspace_bytes, void* stream);

/* scan + duplicateWithKeys + radix sort + identifyTileRanges (§8 a8). */
int rdg_bin(int64_t n, const RdgGeom* geom, int32_t height, int32_t width, int64_t d_cap,
            const RdgBins* bins, void* workspace, int64_t workspace_bytes, void* stream);

/* front-to-back alpha blend of colour, depth and alpha (§8 a9).  Two launches: the region lists (bins->region_*), then
 * the blend itself. */
int rdg_blend_fwd(int64_t n, const RdgGeom* geom, const RdgBins* bins, const RdgView* view,
                  const RdgImage* out, void* stream);

/* ---- backward ------------------------------------------------------------- */

/* reverse-order blend backward (§8 a10): accumulates per-Gaussian screen-space
 * gradients into acc [N,12] = (dpx, dpy, dA, dB, dC, dopacity, dr, dg, db, ddepth, 0, 0);
 * acc must be zeroed by the caller.  dL_dcolor/depth/alpha may be NULL. */
int rdg_blend_bwd(int64_t n, const RdgGeom* geom, const RdgBins* bins, const RdgView* view,
                  const RdgImage* fwd, const float* dL_dcolor, const float* dL_ddepth,
                  const float* dL_dalpha, float* acc, void* stream);

/* Run-to-run reproducible variant of rdg_blend_bwd (test mode: two passes over the lists).  rdg_blend_bwd sums the
 * per-(Gaussian, region) partial gradients with float atomics, whose order - hence the last bits of acc - changes from run
 * to run.  Here the partials are summed as 64-bit integers: pass 1 takes the largest magnitude of every accumulator
 * (atomicMax), pass 2 adds round(partial * 2^(40 - exponent of that maximum)) with integer atomics, which are exact and
 * order-independent, and a last kernel converts back to float (resolution 2^-40 of the largest partial; up to 2^22
 * partials per accumulator).  acc is overwritten.  scratch: rdg_blend_bwd_deterministic_scratch_bytes(n) bytes, 8-byte
 * aligned, contents irrelevant. */
int64_t rdg_blend_bwd_deterministic_scratch_bytes(int64_t n);
int rdg_blend_bwd_deterministic(int64_t n, const RdgGeom* geom, const RdgBins* bins, const RdgView* view,
                                const RdgImage* fwd, const float* dL_dcolor, const float* dL_ddepth,
                                const float* dL_dalpha, float* acc, void* scratch, int64_t scratch_bytes, void* stream);

/* acc -> parameter gradients (+ pose, + deformation) (§8 a10, App. A.7). */
int rdg_preprocess_bwd(const RdgScene* scene, const RdgView* view, const RdgGeom* geom,
                       const float* acc, const RdgSceneGrad* grads, void* stream);

/* The 12-byte factors of dL/dSH straight from the blend backward's accumulators (acc rows 6..8, clamp mask applied), so that
 * their all-gather can start before rdg_preprocess_bwd runs.  dcolor [N,3]. */
int rdg_dcolor_from_acc(int64_t n, const float* acc, const uint8_t* clamped, float* dcolor, void* stream);
/* ... and written through an NVLink-switch MULTICAST mapping of this rank's block of the gathered buffer (symmetric memory:
 * dcolor_mc = multicast address + block offset, 16-byte aligned): multimem.st replicates every store to all ranks, so the
 * all-gather of the factors happens inside the kernel that produces them.  The caller orders it with a cross-rank barrier
 * before the gathered buffer is read.  Needs NVSwitch multicast support (NVLS); use rdg_dcolor_from_acc + copies otherwise. */
int rdg_dcolor_multicast(int64_t n, const float* acc, const uint8_t* clamped, float* dcolor_mc, void* stream);

/* dL/dSH of all views of a data-parallel step from its rank-1 factors (SURVEY.md §8e): for every Gaussian
 *   dL/dSH[k][c] = scale * sum_v Y_k(normalize(x(t_v) - campos_v)) * dcolor[v][c],
 * with x(t_v) the (deformed, scene.raw) mean at view v's time.  viewmatrices [V,16] glm storage, basis_ts [V,K,7]
 * (B(t_v), needed when scene.use_deform), dcolor [V,N,3] as written by rdg_preprocess_bwd through
 * RdgSceneGrad.dcolor (gathered from all ranks).  Overwrites grad_*->sh_dc / sh_rest; V <= 16.  sm_queue: NULL, or 4 uint32 of
 * device scratch for the SM-partitioned mode (RdgSceneGrad.sm_queue). */
int rdg_sh_grad_views(const RdgScene* scene, int32_t sh_degree, int32_t n_views, const float* viewmatrices,
                      const float* basis_ts, const float* dcolor, float scale, const RdgSetGrad* grad_static,
                      const RdgSetGrad* grad_dynamic, uint32_t* sm_queue, void* stream);

/* The same sum over views fused into its consumer: torch.optim.Adam (eps as given, no weight decay) over the f_dc / f_rest
 * groups (src/trainer/rodygs_static.py:118-123) of one or both models, the gradient of each 256-Gaussian chunk rebuilt in
 * shared memory from the gathered factors - dL/dSH (81 % of the gradient buffer) is never written to HBM.  Updates
 * scene->st / dy.sh_dc [n,3] and sh_rest [n,45] IN PLACE (contiguous, 16-byte aligned) and the four moment tensors of
 * RdgShAdam.  `scale` multiplies the gradient (1 / views, times any loss scale).  Run it BEFORE the Adam step that moves the
 * means / motion coefficients the directions are evaluated from. */
typedef struct RdgShAdam {
    float* exp_avg_dc;      /* [n,3]  */
    float* exp_avg_sq_dc;   /* [n,3]  */
    float* exp_avg_rest;    /* [n,45] */
    float* exp_avg_sq_rest; /* [n,45] */
    float lr_dc;            /* feature_lr */
    float lr_rest;          /* feature_lr / 20 */
    int32_t step;           /* this optimiser's step count, >= 1 (bias correction); 0: leave this model alone */
    int32_t reserved;
} RdgShAdam;
int rdg_sh_adam_views(const RdgScene* scene, int32_t sh_degree, int32_t n_views, const float* viewmatrices,
                      const float* basis_ts, const float* dcolor, float scale, const RdgShAdam* adam_static,
                      const RdgShAdam* adam_dynamic, float beta1, float beta2, float eps, void* stream);

/* In-switch all-reduce (sum * scale) of a float range that every rank holds at the same offset of a symmetric-memory buffer:
 * mc_range = the NVLink-switch multicast address of the range (16-byte aligned, n_floats % 4 == 0).  Rank `rank` of `world`
 * reduces its 1 / world slice with multimem.ld_reduce and broadcasts it with multimem.st; `ctas` x 512 threads (0: 32 CTAs).
 * The caller puts a cross-rank barrier on the stream before (all ranks' values written) and after (all slices landed).  Needs
 * NVSwitch multicast (NVLS); the fallback is the NCCL all-reduce of the same range. */
int rdg_allreduce_multimem(float* mc_range, int64_t n_floats, int32_t rank, int32_t world, float scale, int32_t ctas, void* stream);
/* ... of up to 8 ranges of the same buffer in one launch (the structure-of-arrays fields of one slice of Gaussians):
 * offsets / lens in floats from mc_base (host arrays), every range 16-byte aligned and a multiple of 4 floats. */
int rdg_allreduce_multimem_ranges(float* mc_base, const int64_t* offsets, const int64_t* lens, int32_t n_ranges, int32_t rank,
                                  int32_t world, float scale, int32_t ctas, void* stream);

/* ---- losses ----------------------------------------------------------------- */

int64_t rdg_l1_dssim_workspace_bytes(int32_t channels, int32_t height, int32_t width);

/* loss = w_l1 * mean|x-y| + w_dssim * (1 - mean SSIM(x,y))   (loss_utils.py:19-20,57-97;
 * losses.py:61-107).  out_loss (device, 3 floats) = {loss, l1, ssim}.  dL_dpred [C,H,W] receives d loss / d pred (may be NULL: forward only). */
int rdg_l1_dssim(const float* pred, const float* gt, int32_t channels, int32_t height, int32_t width,
                 float w_l1, float w_dssim, float* out_loss, float* dL_dpred,
                 void* workspace, int64_t workspace_bytes, void* stream);

/* Optional terms that ride on the photometric pass of rdg_losses (NULL pointers / zero weights = off):
 * the global Pearson depth regulariser (losses.py:110-129, loss_utils.py:100-117) and the benchmark's
 * alpha regulariser w * mean(1 - alpha) (SURVEY.md §8 a12). */
typedef struct RdgLossTerms {
    const float* depth;      /* [1,H,W] rendered depth */
    const float* gt_depth;   /* [1,H,W] */
    float w_pearson;         /* weight applied to the gradient written to dL_ddepth */
    float pearson_eps;       /* 1e-6 in the reference */
    float* dL_ddepth;        /* [1,H,W] overwritten with w_pearson * d(1 - Pearson)/d depth; may be NULL */
    const float* alpha;      /* [1,H,W] rendered alpha */
    float w_alpha;
    float* dL_dalpha;        /* [1,H,W] overwritten with -w_alpha / (H W); may be NULL */
    /* LocalPearsonDepthLoss (losses.py:132-182): mean over n_local_boxes boxes of 1 - Pearson(depth, gt_depth) inside the box,
     * weight w_local (0.15 in every reference config); its gradient is ADDED to the global term in dL_ddepth within the same
     * passes.  Boxes: device int32 [n,4] = (row0, col0, rows, cols); the reference draws row0 / col0 with torch.randint on the
     * device every iteration (:149-150).  NULL / 0 = off.  Uses depth / gt_depth / pearson_eps / dL_ddepth from above
     * (w_pearson may be 0). */
    const int32_t* local_boxes;
    int32_t n_local_boxes;   /* <= 256 */
    float w_local;
} RdgLossTerms;

/* The whole per-iteration loss stage in three launches: rdg_l1_dssim plus the optional terms above.
 * out_loss (device, 8 floats) = {photometric loss, l1, ssim, 1 - Pearson (global), w_alpha * mean(1 - alpha),
 *                                mean_b (1 - Pearson_b) (local boxes), -, -};
 * entries of disabled terms are left untouched.  Workspace as for rdg_l1_dssim. */
int rdg_losses(const float* pred, const float* gt, int32_t channels, int32_t height, int32_t width,
               float w_l1, float w_dssim, const RdgLossTerms* extra, float* out_loss, float* dL_dpred,
               void* workspace, int64_t workspace_bytes, void* stream);

/* 1 - Pearson(pred, gt) with the unbiased std (loss_utils.py:100-117), over n_boxes boxes
 * given as (row0, col0, rows, cols) int32 quadruples on the device; box 0 = the whole image
 * gives GlobalPearsonDepthLoss, 128x128 boxes give LocalPearsonDepthLoss (losses.py:110-182).
 * out_loss[b] = per-box loss; dL_dpred (+=) receives sum_b box_weight[b] * d loss_b / d pred
 * and must be zeroed (or hold another gradient) before the call.
 * stats: device scratch, 8 doubles per box. */
int rdg_pearson(const float* pred, const float* gt, int32_t height, int32_t width,
                const int32_t* boxes, const float* box_weight, int32_t n_boxes, float eps,
                float* out_loss, float* dL_dpred, double* stats, void* stream);

/* w * mean(1 - alpha) over n pixels: out_loss[0] += that value, dL_dalpha[i] = -w / n.
 * Benchmark-only regulariser of BASELINE.json config 4 ("depth+alpha regularisers");
 * the reference itself has no alpha consumer (SURVEY.md §8 a12). */
int rdg_alpha_reg(const float* alpha, int64_t n, float weight, float* out_loss, float* dL_dalpha, void* stream);

/* ---- optimiser (next row, SURVEY.md §8 f1) ------------------------------------ */

/* In-place Adam over a flat fp32 parameter range (rodygs_static.py:106-149 uses
 * torch.optim.Adam, eps 1e-15, one lr per group). step >= 1. */
int rdg_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
             float lr, float beta1, float beta2, float eps, int32_t step, float grad_scale, void* stream);

/* All parameter groups of one optimiser in ONE launch over the flat buffers (same arithmetic as rdg_adam):
 * groups[k] = float range [begin, end) of param / grad / exp_avg / exp_avg_sq with its own learning rate
 * (xyz, f_dc, f_rest = feature_lr / 20, opacity, scaling, rotation: rodygs_static.py:106-141; motion_coeff:
 * rodygs_dynamic.py:92-123).  begin must be a multiple of 4 floats; n_groups <= 16. */
typedef struct RdgAdamGroup {
    int64_t begin;
    int64_t end;
    float lr;
    int32_t reserved;
} RdgAdamGroup;
int rdg_adam_groups(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, const RdgAdamGroup* groups,
                    int32_t n_groups, float beta1, float beta2, float eps, int32_t step, float grad_scale, void* stream);

/* ---- densification (next row, SURVEY.md §8 f2) ---------------------------------- */

/* Per-iteration statistics of the model being trained (src/trainer/rodygs.py:316-341,
 * src/trainer/rodygs_static.py:317-319): for every row with radii > 0,
 * max_radii2D = max(max_radii2D, radii), grad_accum += |means2D_grad[:, :2]|, denom += 1.
 * radii / means2D_grad point at the first row of that model inside the concatenated scene. */
int rdg_densify_stats(int64_t n, const int32_t* radii, const float* means2D_grad, float* max_radii2D,
                      float* grad_accum, float* denom, void* stream);

/* densify_and_prune (src/trainer/rodygs_static.py:285-301 with :170-283,303-315;
 * src/trainer/rodygs_dynamic.py:150-197) as one stream compaction.
 * rdg_densify_plan evaluates clone / split / prune on the n rows of one model and writes
 *   counts[4] (device) = {A survivors, B clones, C kept split parents, S split-selected};
 *   the new model has A + B + 2 C rows in the reference's final order [A | B | children copy 0 | copy 1];
 *   map[3 n]  : entry j of the first A + B + 2 C = source row | kind << 30, kind 0 survivor, 1 clone, 2 / 3 split child;
 *   split_rank[n] : rank of a split-selected row among the S (else -1) - child copy c of that row takes the
 *                   noise row c * S + rank, the row layout of the reference's torch.normal call (:182-184).
 * use_screen_size: the reference's `max_screen_size` is not None (iteration > opacity_reset_interval). */
int64_t rdg_densify_workspace_bytes(int64_t n);
int rdg_densify_plan(int64_t n, const float* scaling, int32_t scaling_width, const float* opacity,
                     const float* grad_accum, const float* denom, float grad_threshold, float percent_dense,
                     float extent, float min_opacity, int32_t use_screen_size, uint32_t* map,
                     int32_t* split_rank, int32_t* counts, void* workspace, int64_t workspace_bytes, void* stream);

enum RdgDensifyMode {
    RDG_DENSIFY_COPY = 0,     /* dst[j] = src[map[j]]                                   (parameters, time, time index) */
    RDG_DENSIFY_MOMENT = 1,   /* survivors keep the row, new rows get 0                  (Adam exp_avg / exp_avg_sq, utils.py:34-95) */
    RDG_DENSIFY_XYZ = 2,      /* split children: R(q) (noise * exp(scaling)) + xyz      (rodygs_static.py:182-195) */
    RDG_DENSIFY_SCALING = 3   /* split children: log(exp(scaling) / (0.8 * 2))           (:187-189) */
};
typedef struct RdgDensifyField {
    const void* src;          /* [n, width] 32-bit elements */
    void* dst;                /* [n_new, width] */
    int32_t width;
    int32_t mode;             /* RdgDensifyMode */
} RdgDensifyField;

/* Moves every field of the n_new = A + B + 2 C new rows in one pass (a warp per row).
 * noise [2 S, 3]: unit normal samples; xyz / scaling / rotation: the ORIGINAL tensors (inputs of the split formula). */
int rdg_densify_apply(int64_t n_new, const uint32_t* map, const int32_t* split_rank, const int32_t* counts,
                      const float* noise, const RdgDensifyField* fields, int32_t n_fields, const float* xyz,
                      const float* scaling, int32_t scaling_width, const float* rotation, void* stream);

/* reset_opacity (src/trainer/rodygs_static.py:150-159): opacity = inverse_sigmoid(min(sigmoid(opacity), cap)),
 * Adam moments of the group zeroed (src/trainer/utils.py:15-32; may be NULL). */
int rdg_reset_opacity(int64_t n, float* opacity, float cap, float* exp_avg, float* exp_avg_sq, void* stream);

/* ---- motion regularisers (SURVEY.md section 8, row f4) ------------------------------------------------------- */

/* MotionL1Loss + MotionSparsityLoss (src/trainer/losses.py:364-379) over coeff [n, num_basis] (= _motion_coeff
 * [n, 1, num_basis]) in one pass.  loss_parts[0] = mean |c|, loss_parts[1] = mean(|c| / (max_b |c| + 1e-7)).
 * d_coeff (may be NULL) receives w_l1 * dL1/dc + w_sparsity * dSparsity/dc; added to its contents when accumulate != 0.
 * workspace: 16 bytes (two doubles), 8-byte aligned. */
int rdg_motion_coeff_reg(int64_t n, int32_t num_basis, const float* coeff, float w_l1, float w_sparsity,
                         float* loss_parts, float* d_coeff, int32_t accumulate, void* workspace, void* stream);

/* MotionBasisRegularizaiton.forward (src/trainer/losses.py:499-525) on table [num_times, num_basis, 7], degree 0
 * (velocity; every reference config) or negative (term disabled).  loss_parts[0] = translation term,
 * loss_parts[1] = rotation term = mean(reg_coeff[b] * || I - (R(q[t+1]) - R(q[t])) ||_F) - the reference differences the
 * rotation MATRICES (derivate_motion never passes is_rot, :493-497).  reg_coeff [num_basis]: the normalised weights of
 * coeff_bank[freq_div_mode] (:387-489).  d_table (may be NULL) += grad_scale * dLoss/dtable.  workspace as above. */
int rdg_motion_basis_reg(int32_t num_times, int32_t num_basis, const float* table, const float* reg_coeff,
                         int32_t transl_degree, int32_t rot_degree, float grad_scale, float* loss_parts,
                         float* d_table, void* workspace, void* stream);

/* pytorch3d.ops.knn_points(p[None], p[None], K) of src/trainer/losses.py:238-239: for each of the n points the K
 * nearest of the same n points (itself included), squared distances ascending; exact (grid search with a proven
 * stopping rule, not approximate); exact ties towards the lower index.  idx [n, K] int32, dist2 [n, K].
 * No host synchronisation; workspace 256-byte aligned, rdg_knn_workspace_bytes(n) bytes. */
int64_t rdg_knn_workspace_bytes(int64_t n);
int rdg_knn(int64_t n, const float* points, int32_t K, int32_t* idx, float* dist2, void* workspace,
            int64_t workspace_bytes, void* stream);

/* simple-knn's distCUDA2 (src/model/rodygs_static.py:130-133, initial scales): out[i] = ((b0 + b1) + b2) / 3 in
 * float32, b ascending, the squared distances from point i to its 3 nearest OTHER points.  The point itself is skipped
 * by index, not by distance: an exact duplicate counts as a neighbour at distance 0.  Same distance contract and
 * exactness as rdg_knn.  n >= 4 (RDG_E_ARG below); out [n]; workspace as rdg_knn (rdg_knn_workspace_bytes(n)). */
int rdg_knn3_mean_dist2(int64_t n, const float* points, float* out, void* workspace, int64_t workspace_bytes,
                        void* stream);

/* Backward of dist2[i, k] = |p_i - p_idx[i,k]|^2 (rdg_knn's output) for upstream gradient d_dist2 [n, K]:
 *   d_query[i] = sum_k 2 g_ik (p_i - p_j)   overwritten, row-local, no atomics;
 *   d_ref[j]  -= 2 g_ik (p_i - p_j)          float atomics, ADDED to what d_ref holds (the caller zeroes it).
 * Either output may be NULL (the side that needs no gradient).  idx [n, K] int32. */
int rdg_knn_dist2_bwd(int64_t n, int32_t K, const float* points, const int32_t* idx, const float* d_dist2, float* d_query,
                      float* d_ref, void* stream);

/* RigidityLoss.forward, modes "surface" and "distance_preserving" (src/trainer/losses.py:216-361), value and
 * gradient.  The n rows are the reference's random sample (`indice`, :228-232) gathered by the caller:
 *   points = (xyz + pred_translation)[indice], canon = xyz[indice], coeff = _motion_coeff[indice],
 *   frame_indices = the torch.randint draw of :297-301, nn_idx / nn_dist2 = rdg_knn(points, K).
 * loss_parts[0] = surface term, loss_parts[1] = distance-preserving term (the loss is their sum).
 * d_points / d_canon / d_coeff are overwritten with the gradient of that sum; d_table [num_times, num_basis, 7] is
 * added to (rows frame_indices, columns 0..2).  Mode "coeff" (no reference config uses it) is not built. */
typedef struct RdgRigidity {
    int64_t n;
    int32_t K, num_basis, n_frames;
    int32_t mode_surface, mode_distance;
    float eps;                        /* CharbonnierLoss eps, 1e-6 */
    const float* points;              /* [n, 3] */
    const float* canon;               /* [n, 3] */
    const float* coeff;               /* [n, num_basis] */
    const float* table;               /* [num_times, num_basis, 7] */
    const int32_t* frame_indices;     /* [n_frames] */
    const int32_t* nn_idx;            /* [n, K] */
    const float* nn_dist2;            /* [n, K] */
    float* loss_parts;                /* [2] */
    float* d_points;                  /* [n, 3] */
    float* d_canon;                   /* [n, 3] */
    float* d_coeff;                   /* [n, num_basis] */
    float* d_table;                   /* [num_times, num_basis, 7], accumulated */
} RdgRigidity;
int64_t rdg_rigidity_workspace_bytes(int64_t n, int32_t K, int32_t n_frames);
int rdg_rigidity(const RdgRigidity* args, void* workspace, int64_t workspace_bytes, void* stream);

/* Flat-buffer trainer glue for RigidityLoss: gather the sampled rows (`indice` [n] int32, no repeats - random.sample,
 * losses.py:228-232) and deform them, points = xyz[i] + spatial_lr_scale * sum_b c_ib (basis_t_b - table[time_ind[i]]_b)[:3]
 * (src/model/rodygs_dynamic.py:122-138), canon = xyz[i], coeff_s = coeff[i]; the fused render path never materialises
 * pred_translation. */
int rdg_rigidity_sample(int64_t n, int32_t num_basis, const int32_t* indice, const float* xyz, const float* coeff,
                        const int32_t* time_ind, const float* basis_t, const float* table, float spatial_lr_scale,
                        float* points, float* canon, float* coeff_s, void* stream);
/* ... and its backward: grad_scale * (d_points, d_canon, d_coeff_s of rdg_rigidity; the last two may be NULL) is ADDED to
 * the rows `indice` of d_xyz / d_coeff and, through the deformation, to d_basis_t [num_basis, 7] and d_table. */
int rdg_rigidity_sample_bwd(int64_t n, int32_t num_basis, int32_t num_times, const int32_t* indice, const float* coeff,
                            const int32_t* time_ind, const float* basis_t, const float* table, float spatial_lr_scale,
                            float grad_scale, const float* d_points, const float* d_canon, const float* d_coeff_s,
                            float* d_xyz, float* d_coeff, float* d_basis_t, float* d_table, void* stream);

/* ---- time embedding + motion-basis MLP (SURVEY.md section 8, row a1) ------------------------------------------- */

/* TimestepEmbedder.forward (src/model/rodygs_dynamic.py:202-220) + MLPBasisNetwork.batch_inference / forward
 * (:296-327) for a batch of `rows` times: timenet emb_dim -> width -> width -> width/2, then num_basis heads
 * width/2 -> width/4 -> out_dim (7 = 3 translation + 4 rotation).  The trainer asks for rows = 1 + T (the query time t
 * first, then the T training times), so B(t) [num_basis, 7] and the table [T, num_basis, 7] come from ONE launch.
 *
 * params: ONE packed fp32 buffer, PyTorch [out, in] row-major blocks in this order
 *   timenet.0.weight [W,E] | timenet.0.bias [W] | timenet.2.weight [W,W] | timenet.2.bias [W] |
 *   timenet.4.weight [W/2,W] | timenet.4.bias [W/2] |
 *   basis_xyz.{k}.basis.0.weight stacked over k [nb,W/4,W/2] | ....basis.0.bias [nb,W/4] |
 *   basis_xyz.{k}.basis.2.weight [nb,out,W/4] | ....basis.2.bias [nb,out]            (rdg_basis_mlp_param_count floats)
 * Either `emb` [rows, emb_dim] (what batch_embedding, :290-294, returns) or `times` [rows] with `freqs_pi` [(emb_dim-1)/2]
 * (= freq_bands * pi, :205-212) so that the embedding is evaluated in the kernel.
 * saved (may be NULL for inference): [rows, rdg_basis_mlp_saved_floats()] the embedding and every pre-activation,
 * the only state the backward needs.  activation: 0 = nn.GELU() (erf form), 1 = nn.ReLU. */
typedef struct RdgBasisMlp {
    int32_t emb_dim, width, num_basis, out_dim, activation, rows;
    const float* params;
    const float* emb;        /* [rows, emb_dim] or NULL */
    const float* times;      /* [rows] (used when emb == NULL) */
    const float* freqs_pi;   /* [(emb_dim - 1) / 2] */
    float* basis;            /* out [rows, num_basis, out_dim] */
    float* basis_row0;       /* NULL, or: row 0 goes here [num_basis, out_dim] and rows 1.. to basis[0 .. rows-2] - the
                                trainer keeps B(t) and the table in different slices of its flat buffer */
    float* saved;            /* out (fwd) / in (bwd) [rows, saved_floats] */
} RdgBasisMlp;
int64_t rdg_basis_mlp_param_count(int32_t emb_dim, int32_t width, int32_t num_basis, int32_t out_dim);
int64_t rdg_basis_mlp_saved_floats(int32_t emb_dim, int32_t width, int32_t num_basis);
int rdg_basis_mlp_fwd(const RdgBasisMlp* args, void* stream);
/* Backward of the above (what loss.backward(), src/trainer/rodygs.py:310, runs through the MLP): d_basis
 * [rows, num_basis, out_dim] -> d_params (packed like params; overwritten, or added to when accumulate != 0).
 * d_basis_row0: NULL, or the gradient of row 0 (then d_basis holds rows 1.., like basis_row0 above).
 * Two launches, no atomics: the result is deterministic.  args->basis is not read. */
int64_t rdg_basis_mlp_bwd_workspace_bytes(int32_t rows, int32_t emb_dim, int32_t width, int32_t num_basis);
int rdg_basis_mlp_bwd(const RdgBasisMlp* args, const float* d_basis, const float* d_basis_row0, float* d_params,
                      int32_t accumulate, void* workspace, int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RODYGS_B200_H */
