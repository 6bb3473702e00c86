/*
 * mi3d.h -- C ABI of the B200-native Make-It-3D SDS-step hot path (libmi3d.so).
 *
 * Drop-in boundary (SURVEY.md 8b): these entry points are what the reference's pybind module `_raymarching`
 * (raymarching/src/bindings.cpp:5-23, raymarching/src/raymarching.h:7-22), its third-party tiny-cuda-nn
 * encoder (nerf/network_tcnn.py:54-65,107) and its diffusers U-Net / VAE calls (nerf/sd.py:117-174,212-220)
 * would bind instead.  Conventions for every function:
 *   - plain pointers are DEVICE pointers unless named *_host or documented otherwise; sizes are element counts
 *   - returns 0 on success, a cudaError_t value or MI3D_ERR_ARG (1000001) otherwise; never throws
 *   - never allocates device memory and never synchronises; work is enqueued on `stream`
 *     (pass torch.cuda.current_stream().cuda_stream); scratch comes from the caller, sized by *_workspace_bytes()
 *   - re-entrant; no global mutable state besides one-time kernel attribute setup
 *   - all floating-point tensors are fp32 contiguous, exactly as the reference wrappers pass them
 *     (custom_fwd(cast_inputs=torch.float32), raymarching/raymarching.py:33,175,252)
 */
#ifndef MI3D_H
#define MI3D_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* mi3d_stream_t; /* cudaStream_t */

/* ------------------------------------------------------------------------------------------------------
 * B1: ray-march operators  (replace raymarching/src/raymarching.cu, called from raymarching/raymarching.py)
 * ------------------------------------------------------------------------------------------------------ */

/* replaces near_far_from_aabb, raymarching.cu:92-160 (wrapper raymarching.py:31-61) */
int mi3d_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N, float min_near,
                            float* nears, float* fars, mi3d_stream_t stream);

/* replaces morton3D / morton3D_invert, raymarching.cu:214-258 (raymarching.py:95-142) */
int mi3d_morton3D(const int* coords, uint32_t N, int* indices, mi3d_stream_t stream);
int mi3d_morton3D_invert(const int* indices, uint32_t N, int* coords, mi3d_stream_t stream);

/* replaces packbits, raymarching.cu:268-300 (raymarching.py:144-170).  n_bytes = C*H^3/8.
 * thresh_dev (nullable) is a device scalar: effective threshold = min(thresh, *thresh_dev) -- this is
 * renderer.py:630 `min(self.mean_density, self.density_thresh)` without the .item() host sync. */
int mi3d_packbits(const float* grid, uint32_t n_bytes, float thresh, const float* thresh_dev, uint8_t* bitfield,
                  mi3d_stream_t stream);

/* replaces march_rays_train, raymarching.cu:312-493 (raymarching.py:173-247).
 *  - nears/fars: precomputed [N] (B1 behaviour) or NULL, in which case the slab test against aabb[6] with
 *    min_near is fused into the kernel (optionally written to nears_out/fars_out, nullable).
 *  - noises: [N] U[0,1) (raymarching.py:226) or NULL -> in-kernel Philox keyed by (seed, ray id).
 *  - rays[n] = (n, offset, count): compaction is ordered by ray id (deterministic), not by atomic arrival.
 *  - counter[0] += EMITTED samples, counter[1] += N (caller zeroes it like renderer.py:504).
 *  - M = capacity of xyzs/dirs/deltas in rows; rays that do not fit write nothing (raymarching.cu:416).  Because
 *    offsets are ordered by ray id the emitted samples are always the contiguous prefix [0, counter[0]) -- on overflow
 *    counter[0] is the offset of the first dropped ray, not the uncapped total the reference adds (raymarching.cu:405):
 *    nothing is zero-filled here, so consumers must never see the unwritten rows.
 *  - workspace: mi3d_march_rays_train_workspace_bytes(N) bytes (zero-filled internally). */
size_t mi3d_march_rays_train_workspace_bytes(uint32_t N);
int mi3d_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* density_bitfield, float bound,
                          float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                          const float* nears, const float* fars, const float* aabb, float min_near,
                          float* nears_out, float* fars_out, const float* noises, uint64_t seed,
                          float* xyzs, float* dirs, float* deltas, int* rays, int* counter,
                          void* workspace, mi3d_stream_t stream);

/* Ray generation (replaces get_rays, nerf/utils.py:51-116, for the N = -1 "every pixel" mode training uses, provider.py:297).
 * A batch holds n_views * rays_per_view rays: batch ray i belongs to view i / rays_per_view and to the row-major pixel
 * (i % rays_per_view) * pixel_stride + pixel_phase of that view.  stride 1 / phase 0 / rays_per_view = H*W is one full image;
 * stride G / phase r deals every G-th pixel of each of G views to rank r (ray-parallel render, DESIGN.md section 5).
 * cams: DEVICE [n_views][16] fp32 = rows 0..2 of the cam2world pose (3x4 row-major, R | t) followed by fx, fy, cx, cy. */
typedef struct {
    const float* cams;
    uint32_t n_views;
    uint32_t H, W;
    uint32_t rays_per_view;
    uint32_t pixel_stride, pixel_phase;
} mi3d_raygen;
/* rays_o / rays_d [N,3], depth_scale [N] (each nullable), N = n_views * rays_per_view */
int mi3d_get_rays(const mi3d_raygen* rg, uint32_t N, float* rays_o, float* rays_d, float* depth_scale, mi3d_stream_t stream);
/* mi3d_march_rays_train with the rays generated inside the kernel (no rays_o / rays_d tensors; near/far always fused):
 * depth_scale_out [N] nullable.  The Philox march jitter (noises == NULL) is keyed by (view, pixel), not by the batch index. */
int mi3d_march_rays_train_cam(const mi3d_raygen* rg, float* depth_scale_out, const uint8_t* density_bitfield, float bound,
                              float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                              const float* aabb, float min_near, float* nears_out, float* fars_out, const float* noises,
                              uint64_t seed, float* xyzs, float* dirs, float* deltas, int* rays, int* counter,
                              void* workspace, mi3d_stream_t stream);

/* Optional fused epilogue of NeRFRenderer.run_cuda (nerf/renderer.py:553-570):
 *   image_out = image + (1 - ws) * bg ;  depth_out = (depth + (1 - ws) * max_depth) * depth_scale */
typedef struct {
    const float* bg_color;    /* device [3] or NULL -> bg_scalar (renderer.py:554-555 default 1) */
    float bg_scalar;
    float max_depth;          /* opt.max_depth, main.py:91 */
    const float* depth_scale; /* device [N] or NULL */
    uint32_t rays_per_view;   /* > 0: multi-view batch, bg_color is [n_views][3] and ray n uses row n / rays_per_view; 0: one colour */
} mi3d_epilogue;

/* replaces composite_rays_train_forward, raymarching.cu:501-590 (raymarching.py:250-281).
 * ep == NULL -> plain B1 behaviour (image_out/depth_out ignored). */
int mi3d_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* deltas, const int* rays,
                                      uint32_t M, uint32_t N, float T_thresh, float* weights_sum, float* depth,
                                      float* image, const mi3d_epilogue* ep, float* image_out, float* depth_out,
                                      mi3d_stream_t stream);

/* replaces composite_rays_train_backward, raymarching.cu:602-696 (raymarching.py:283-300).
 * grad_image is w.r.t. image (ep == NULL) or image_out (ep != NULL); grad_depth (nullable) is w.r.t. depth_out and
 * only reaches sigmas through (1 - ws) * max_depth, like autograd does in the reference (raymarching.py:287).
 * zero_tail != 0 writes zeros to samples after the early-out so the outputs need no pre-zeroing. */
int mi3d_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_image, const float* grad_depth,
                                       const float* sigmas, const float* rgbs, const float* deltas, const int* rays,
                                       const float* weights_sum, const float* image, uint32_t M, uint32_t N,
                                       float T_thresh, const mi3d_epilogue* ep, float* grad_sigmas, float* grad_rgbs,
                                       int zero_tail, mi3d_stream_t stream);

/* replaces march_rays / composite_rays (inference), raymarching.cu:907-1022, :1024-1125 (raymarching.py:368-470) */
int mi3d_march_rays(uint32_t n_alive, uint32_t n_step, const int* rays_alive, const float* rays_t, const float* rays_o,
                    const float* rays_d, float bound, float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H,
                    const uint8_t* density_bitfield, const float* nears, const float* fars, float* xyzs, float* dirs,
                    float* deltas, const float* noises, mi3d_stream_t stream);
int mi3d_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int* rays_alive, float* rays_t,
                        const float* sigmas, const float* rgbs, const float* normals, const float* deltas,
                        float* weights_sum, float* depth, float* image, float* normal, mi3d_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * B2: field  (replaces tinycudann.Encoding + nerf/network_tcnn.py MLP / common_forward / normal / forward)
 * ------------------------------------------------------------------------------------------------------ */

/* Multiresolution hash grid geometry (tiny-cuda-nn HashGrid as configured at nerf/network_tcnn.py:54-65):
 * level l owns entries [offsets[l], offsets[l]+sizes[l]) of the flat fp32 table `encoder.params`
 * (2 features per entry, entry-major). */
typedef struct {
    uint32_t n_levels;
    uint32_t n_entries;
    uint32_t offsets[16];
    uint32_t sizes[16];
    uint32_t ress[16];
    float scales[16];
} mi3d_hashgrid;

/* HOST helper: fills *out (host struct, passed by pointer to the calls below). */
int mi3d_hashgrid_make(uint32_t n_levels, uint32_t base_resolution, double per_level_scale, uint32_t log2_hashmap_size,
                       mi3d_hashgrid* out);

/* stand-alone encoder: replaces tcnn.Encoding.forward / backward as called at nerf/network_tcnn.py:107.
 * x [E,3] in [0,1]; out / grad_out [E, 2*n_levels]; grad_table accumulates (+=). hg is a HOST pointer. */
int mi3d_hashgrid_forward(const float* x, uint32_t E, const float* table, const mi3d_hashgrid* hg, float* out, mi3d_stream_t stream);
int mi3d_hashgrid_backward(const float* x, uint32_t E, const float* grad_out, const mi3d_hashgrid* hg, float* grad_table, mi3d_stream_t stream);

/* sigma_net = MLP(32, 4, 64, 3) (nerf/network_tcnn.py:67, :13-32): PyTorch nn.Linear layout [out][in], biases on */
typedef struct { const float *w1, *b1, *w2, *b2, *w3, *b3; } mi3d_mlp;
typedef struct { float *w1, *b1, *w2, *b2, *w3, *b3; } mi3d_mlp_grad;

enum { MI3D_SHADING_ALBEDO = 0, MI3D_SHADING_LAMBERTIAN = 1, MI3D_SHADING_TEXTURELESS = 2, MI3D_SHADING_NORMAL = 3 };
/* kernel family of the fused field.  TCGEN05 (default): tcgen05 split-precision tiles; the backward chain kernel issues the
 * table-gradient REDs itself (LSU-bound RED stream under the latency-bound MMA chain; = _FUSED_SCATTER).  _SPLIT_SCATTER: the
 * round-1 pipeline with a separate full-occupancy scatter kernel (A/B arm).  _SINGLE_E: fused scatter, but the encoding operand of the
 * chain kernel single-buffered (the default alternates consecutive evaluations between the two column halves of its tile; A/B arm).
 * FFMA = the register-tiled fp32 kernels. */
enum { MI3D_FIELD_IMPL_TCGEN05 = 0, MI3D_FIELD_IMPL_FFMA = 1, MI3D_FIELD_IMPL_TCGEN05_FUSED_SCATTER = 2, MI3D_FIELD_IMPL_TCGEN05_SPLIT_SCATTER = 3,
       MI3D_FIELD_IMPL_TCGEN05_SINGLE_E = 4 };

typedef struct {
    float bound;          /* opt.bound */
    float blob_density;   /* opt.blob_density (main.py:56) */
    float blob_radius;    /* opt.blob_radius  (main.py:57) */
    int n_evals;          /* 1: sigma/albedo only; 7: + 6-tap finite-difference normal (network_tcnn.py:115-138);
                             13: + the perturbed normal of the smoothness loss (renderer.py:521-524) */
    int shading;          /* MI3D_SHADING_* (network_tcnn.py:146-170) */
    float ambient_ratio;
    const float* light_d; /* device [3] (multi-view batches: [n_views][3]), needed unless shading == albedo */
    int impl;             /* MI3D_FIELD_IMPL_* (explicit: the library reads no environment variables) */
    float scatter_agg_scale; /* tuning knob of the fused scatter: REDs of hash-grid levels with scale below this are warp-aggregated; 0 = library default (100) */
} mi3d_field_cfg;

/* Multi-view batches (several camera views' rays in one march: ray-parallel multi-GPU render, or several views per GPU).
 * Samples are emitted in ray order, hence grouped by view.  DEVICE table, written by mi3d_render_forward (phase SHADE):
 *   rows [bounds[s], bounds[s+1]),  s <  n_views : the samples of view s in this batch
 *                                   s >= n_views : zero rows of view s - n_views evaluated here (the reference pads every view's
 *                                                  sample list to the next multiple of 128 with xyz = dir = 0 rows that take part
 *                                                  in the loss means, raymarching.py:237-241; exactly one rank owns a view's)
 *   mpad[v] : padded sample count of the WHOLE view v, summed over all ranks -- the denominator of its loss means. */
#define MI3D_MAX_VIEWS 8
typedef struct {
    uint32_t n_views;
    uint32_t bounds[2 * MI3D_MAX_VIEWS + 1];
    uint32_t mpad[MI3D_MAX_VIEWS];
} mi3d_view_segs;

typedef struct {
    const float* xyzs;         /* [cap,3] sample positions (output of mi3d_march_rays_train) */
    const float* dirs;         /* [cap,3] or NULL */
    const int* counter;        /* device: counter[0] = number of valid rows M; NULL -> m_fixed */
    uint32_t m_fixed;
    uint32_t align;            /* 128 reproduces the zero-row padding of raymarching.py:237-241 in the loss means; 0 = none */
    uint32_t cap;              /* rows allocated in every per-sample buffer */
    const float* smooth_noise; /* [cap,3] N(0,1) (renderer.py:522) or NULL -> in-kernel Philox(seed,row) */
    uint64_t seed;
    /* optional encoding cache shared by one forward and the backward(s) that follow it: fp32 [enc_cache_tiles][13][128][32]
     * (mi3d_field_enc_cache_bytes).  mi3d_field_forward stores the hash-grid encodings of the first enc_cache_tiles 128-row tiles of
     * every evaluation point there; mi3d_field_backward, when enc_cache_valid != 0, reads them back instead of re-gathering the
     * table (same table, same samples: the caller vouches for it).  Rows beyond the cache are re-gathered.  NULL = off. */
    float* enc_cache;
    uint32_t enc_cache_tiles;
    uint32_t enc_cache_valid;
    /* multi-view batch: DEVICE table (NULL = one view: counter / m_fixed / align above describe the rows) and its view count.
     * With segs, loss_orient / loss_smooth / grad_loss_* are [n_views] arrays and loss_partials holds
     * 2 * n_views * mi3d_field_grid_ctas(0) floats.  tcgen05 kernels only. */
    const mi3d_view_segs* segs;
    uint32_t n_views;
    uint32_t noise_mode;       /* in-kernel smoothness perturbation keyed by 0: (seed, row)  1: (seed, sample position) */
} mi3d_field_io;
size_t mi3d_field_enc_cache_bytes(uint32_t tiles);

/* number of CTAs the persistent field kernels launch; loss_partials must hold 2 * mi3d_field_grid_ctas(0) floats */
int mi3d_field_grid_ctas(int backward);

/* Fused replacement of NeRFNetwork.forward (+ the regularisers of run_cuda):
 *   sigmas[row], rgbs[row,3], normals[row,3] (nullable), tape[row,16] (nullable; needed for backward),
 *   loss_orient / loss_smooth: device scalars (nullable), means over the padded row count like the reference. */
int mi3d_field_forward(const mi3d_field_io* io, const float* table, const mi3d_hashgrid* hg, const mi3d_mlp* mlp,
                       const mi3d_field_cfg* cfg, float* sigmas, float* rgbs, float* normals, float* tape,
                       float* loss_partials, float* loss_orient, float* loss_smooth, mi3d_stream_t stream);

/* Backward of the above: accumulates (+=) into grad_table [2*n_entries] and grad_mlp.  grad_* inputs are nullable
 * (treated as zero); grad_loss_* are device scalars.  No gradient w.r.t. positions (the reference requests none). */
int mi3d_field_backward(const mi3d_field_io* io, const float* table, const mi3d_hashgrid* hg, const mi3d_mlp* mlp,
                        const mi3d_field_cfg* cfg, const float* tape, const float* grad_sigmas, const float* grad_rgbs,
                        const float* grad_normals, const float* grad_loss_orient, const float* grad_loss_smooth,
                        float* grad_table, const mi3d_mlp_grad* grad_mlp, void* workspace, mi3d_stream_t stream);
/* workspace (nullable): mi3d_field_backward_workspace_bytes() bytes of scratch.  When given, the backward runs per chunk of 1 048 576
 * samples: encodings come from io->enc_cache or from a full-occupancy gather kernel into the scratch, then the tensor-core chain kernel
 * runs and issues the table-gradient REDs itself (cfg->impl = _SPLIT_SCATTER: a separate full-occupancy scatter kernel instead).
 * When NULL the chain kernel also gathers in-kernel (slower: its eight gather warps are starved); the Python host always passes scratch. */
size_t mi3d_field_backward_workspace_bytes(void);

/* ------------------------------------------------------------------------------------------------------
 * Fused render step: the training branch of NeRFRenderer.run_cuda (nerf/renderer.py:481-524,553-583) as one call per
 * direction (SURVEY.md 8b "mi3d_render_fwd / mi3d_render_bwd").  Sequences the kernels behind the B1 / B2 entry points
 * above over one caller-owned workspace; see csrc/render.cu for the multi-view / ray-parallel protocol.
 * ------------------------------------------------------------------------------------------------------ */
typedef struct {
    /* rays: explicit tensors, or generated in the march kernel from cameras when rays_o == NULL */
    const float* rays_o;          /* [N,3] */
    const float* rays_d;          /* [N,3] */
    const float* depth_scale;     /* [N] or NULL (explicit rays only; generated rays carry their own) */
    const mi3d_raygen* raygen;    /* HOST struct (its cams pointer is a device pointer) */
    uint32_t N;
    uint32_t n_views;             /* views in the batch, 1..MI3D_MAX_VIEWS; view of ray i = i / (N / n_views) */
    /* occupancy grid + march (renderer.py:481-508; min_near is the wrapper default 0.2, raymarching.py:34) */
    const uint8_t* density_bitfield;
    uint32_t C, H;
    float bound, dt_gamma;
    uint32_t max_steps;
    float min_near;
    const float* aabb;            /* device [6] */
    const float* noises;          /* [N] or NULL -> Philox(seed) */
    uint64_t seed;
    /* compositing + epilogue (renderer.py:553-570) */
    float T_thresh;
    const float* bg_color;        /* device [n_views][3] or NULL -> bg_scalar */
    float bg_scalar;
    float max_depth;
    /* regularisers (renderer.py:513-524) */
    const float* smooth_noise;    /* [cap,3] or NULL -> Philox(seed + 1) */
    uint32_t noise_mode;          /* mi3d_field_io.noise_mode */
    /* ray-parallel multi-rank render */
    const int* all_counts;        /* DEVICE [n_ranks][n_views]: every rank's ws->view_counts, all-gathered; NULL = this rank holds whole views */
    uint32_t n_ranks;
    uint32_t pad_view_mask;       /* bit v set: this rank evaluates the 128-alignment zero rows of view v (exactly one rank per view) */
} mi3d_render_args;

typedef struct {                  /* filled by mi3d_render_workspace_carve; all DEVICE pointers into the caller's blob */
    uint32_t N, cap, n_views;     /* cap = min(N * max_steps, max_samples) + 128 * n_views rows */
    float *xyzs, *dirs, *deltas, *sigmas, *rgbs, *tape, *g_sigmas, *g_rgbs;        /* per sample */
    int *rays, *counter;                                                            /* [N,3], [2]: counter[0] = emitted samples */
    float *nears, *fars, *ws_raw, *depth_raw, *image_raw, *depth_scale;             /* per ray */
    void* scan_ws;
    float* loss_partials;
    int* view_counts;             /* [MI3D_MAX_VIEWS] this rank's samples per view (written by phase MARCH of multi-view batches) */
    mi3d_view_segs* segs;
    float* enc_cache;
    uint32_t enc_cache_tiles;
    size_t bytes;
} mi3d_render_ws;

size_t mi3d_render_workspace_bytes(uint32_t N, uint32_t max_steps, uint32_t max_samples /* 0 = N * max_steps */, uint32_t n_views,
                                   uint32_t enc_cache_tiles);
int mi3d_render_workspace_carve(void* base, uint32_t N, uint32_t max_steps, uint32_t max_samples, uint32_t n_views,
                                uint32_t enc_cache_tiles, mi3d_render_ws* out);

enum { MI3D_RENDER_PHASE_MARCH = 1, MI3D_RENDER_PHASE_SHADE = 2, MI3D_RENDER_PHASE_ALL = 3 };
/* image [N,3], depth [N], weights_sum [N]; loss_orient / loss_smooth: device scalars (one view, single rank) or [n_views] arrays
 * of this rank's SHARE of every view's mean (multi-view: sum them over ranks).  phases: MARCH | SHADE; a multi-rank caller runs
 * MARCH, all-gathers ws->view_counts into args->all_counts, then runs SHADE. */
int mi3d_render_forward(const mi3d_render_args* args, const float* table, const mi3d_hashgrid* hg, const mi3d_mlp* mlp,
                        const mi3d_field_cfg* cfg, const mi3d_render_ws* ws, int phases, float* image, float* depth,
                        float* weights_sum, float* loss_orient, float* loss_smooth, mi3d_stream_t stream);
/* grad_image [N,3] required; grad_depth / grad_weights_sum [N] and grad_loss_* (scalars or [n_views]) nullable.  Accumulates (+=)
 * into grad_table / grad_mlp.  enc_cache_valid: the workspace still holds this forward's encodings. */
int mi3d_render_backward(const mi3d_render_args* args, const float* table, const mi3d_hashgrid* hg, const mi3d_mlp* mlp,
                         const mi3d_field_cfg* cfg, const mi3d_render_ws* ws, const float* grad_image, const float* grad_depth,
                         const float* grad_weights_sum, const float* grad_loss_orient, const float* grad_loss_smooth,
                         float* grad_table, const mi3d_mlp_grad* grad_mlp, void* bwd_workspace, int enc_cache_valid,
                         mi3d_stream_t stream);

/* Evaluation renderer (SURVEY.md 8f-2): the alive-ray loop of NeRFRenderer.run_cuda's non-training branch (nerf/renderer.py:526-551:
 * march_rays -> field -> composite_rays until every ray is terminated or max_steps is reached) in ONE call, all loop state on the
 * device (no per-iteration host synchronisation; the reference compacts the alive list with a boolean mask every iteration).
 * Outputs [N], [N], [N,3], [N,3] are (re)initialised inside and carry the background mix / depth fix-up of renderer.py:553-570.
 * done_flag_host (nullable): int in pinned, device-accessible HOST memory; lets the host stop enqueueing iterations early. */
typedef struct {
    const float* rays_o;          /* [N,3] */
    const float* rays_d;          /* [N,3] */
    const float* depth_scale;     /* [N] or NULL */
    uint32_t N;
    const uint8_t* density_bitfield;
    uint32_t C, H;
    float bound, dt_gamma;
    uint32_t max_steps;           /* 1024 in the reference's eval calls */
    float min_near;               /* 0.2 (wrapper default, raymarching.py:34) */
    const float* aabb;            /* device [6]: aabb_infer */
    float T_thresh;               /* 1e-4 (renderer.py:483 default passed to composite_rays) */
    int perturb;                  /* jitter the first march iteration */
    uint64_t seed;
    const float* bg_color;        /* device [3] or NULL -> bg_scalar */
    float bg_scalar;
    float max_depth;
} mi3d_render_eval_args;
size_t mi3d_render_eval_workspace_bytes(uint32_t N);
int mi3d_render_eval(const mi3d_render_eval_args* args, const float* table, const mi3d_hashgrid* hg, const mi3d_mlp* mlp,
                     const mi3d_field_cfg* cfg, void* workspace, int* done_flag_host, float* weights_sum, float* depth, float* image,
                     float* normal, mi3d_stream_t stream);

/* Replaces NeRFRenderer.update_extra_state (nerf/renderer.py:587-637): density_grid [C,H^3] EMA-max update from the
 * field at jittered cell centres, mean density (device scalar out), bitfield repack.  jitter: [C,H^3,3] U[0,1) or NULL
 * (Philox).  workspace: mi3d_density_grid_workspace_bytes(C,H). */
size_t mi3d_density_grid_workspace_bytes(uint32_t C, uint32_t H);
int mi3d_density_grid_update(float* density_grid, uint8_t* density_bitfield, uint32_t C, uint32_t H, float bound,
                             float decay, float density_thresh, const float* table, const mi3d_hashgrid* hg,
                             const mi3d_mlp* mlp, const mi3d_field_cfg* cfg, const float* jitter, uint64_t seed,
                             float* mean_density_out, void* workspace, mi3d_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * Parameter update that follows the hot path (SURVEY.md 8f-1): nn.utils.clip_grad_norm(max_norm) (nerf/utils.py:984) +
 * Adan.step() with its own global-norm clip (optimizer.py:102-198) + _single_tensor_adan (optimizer.py:201-256) in one
 * elementwise kernel over a flat (shard of a) parameter vector.  The global gradient norm stays on the device.
 * ------------------------------------------------------------------------------------------------------ */
typedef struct {
    double lr;              /* group['lr'] (python floats of the reference are doubles; the host folds them in double) */
    double beta1, beta2, beta3, eps, weight_decay;     /* (0.98, 0.92, 0.99), 1e-8, 2e-5 (main.py:132) */
    float max_grad_norm;    /* Adan's global clip, 5.0; 0 = off */
    float clip_grad_norm;   /* Trainer's clip_grad_norm max_norm, 10; 0 = off */
    int no_prox;
    int step;               /* group['step'] AFTER the increment: 1 on the first call */
    int reset_prev;         /* != 0: treat neg_pre_grad as missing (optimizer.py:160) */
} mi3d_adan_cfg;
/* out (+)= sum(g[i]^2), deterministic (fixed-order partials, fp64 fold).  g 16-byte aligned.  workspace: mi3d_sumsq_workspace_bytes(). */
size_t mi3d_sumsq_workspace_bytes(void);
int mi3d_sumsq(const float* g, uint64_t n, float* out, int accumulate, void* workspace, mi3d_stream_t stream);
/* total_sumsq: DEVICE scalar = squared L2 norm of ALL gradients of the model before any clipping (every rank passes the global
 * value).  grad is rescaled in place like the reference does (p.grad ends up clipped); all state tensors are updated in place. */
int mi3d_adan_step(float* param, float* grad, float* exp_avg, float* exp_avg_sq, float* exp_avg_diff, float* neg_pre_grad, uint64_t n,
                   const float* total_sumsq, const mi3d_adan_cfg* cfg, mi3d_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * B3: Stable-Diffusion guidance  (replaces the diffusers/cuDNN/cuBLAS calls behind nerf/sd.py:117-174, :212-220)
 * ------------------------------------------------------------------------------------------------------ */

/* The one tensor-core tile kernel (tcgen05.mma + TMEM accumulators + TMA operand staging) exposed directly:
 *   out[M,N] = alpha * A[M,K] . B[N,K]^T + bias[N] (+ residual[M,N]);  A, B fp16 K-major; out fp16 or fp32.
 * Stands in for the cuBLAS GEMM under every nn.Linear of diffusers' UNet2DConditionModel / AutoencoderKL
 * (nerf/sd.py:146, :217).  M % 128 == 0, K % 64 == 0, N % block_n == 0 (block_n in {64,128,160,256}; 0 = auto).
 * epi_mode: 0 plain, 1 GEGLU (rows of B interleaved value/gate; out is [M, N/2]), 2 transposed store (out is [N, M]). */
int mi3d_gemm_f16(const void* a, const void* b, void* out, int out_is_f32, int M, int N, int K, int block_n, float alpha,
                  const float* bias, const void* residual, int epi_mode, mi3d_stream_t stream);

/* Split-K form used for the deep U-Net levels (M = 128 .. 512 rows, K up to 23 040): `splits` K-ranges per output tile run on
 * different SMs and meet by fp32 RED in ws ([M][N] floats, zeroed inside); bias / residual / fp16 conversion happen in a
 * second pass.  fp16 output, plain epilogue only. */
int mi3d_gemm_f16_splitk(const void* a, const void* b, void* out, int M, int N, int K, int block_n, int splits, float alpha,
                         const float* bias, const void* residual, void* ws, mi3d_stream_t stream);

/* Fused multi-head attention, head_dim 64 (stands in for diffusers' attention processor inside BasicTransformerBlock.attn1 /
 * .attn2, nerf/sd.py:146): o = softmax(q k^T / 8) v per (batch, head), scores kept in TMEM / shared memory.
 * q [B*T, ldq], k and v [B*Tk, ldk / ldv], o [B*T, ldo], fp16, head h at columns [64h, 64h+64); only the first Tk_valid keys of
 * every batch take part (77 of the 128 padded text rows for cross attention).  All ld % 8 == 0. */
int mi3d_flash_attn_f16(const void* q, const void* k, const void* v, void* o, int B, int T, int Tk, int Tk_valid, int heads,
                        int ldq, int ldk, int ldv, int ldo, mi3d_stream_t stream);

/* Implicit-GEMM 3x3 stride-1 pad-1 convolution on the same kernel (stands in for the cuDNN conv under diffusers'
 * ResnetBlock2D / Downsample2D / Upsample2D): x [N,H,W,Cin] fp16 NHWC, w [Cout][3][3][Cin] fp16, y [N,H,W,Cout] fp16. */
/* test path: out[M,N] (fp32) = A[M,K] . Bt[K,N], B consumed as an MN-major UMMA operand */
int mi3d_gemm_f16_bt(const void* a, const void* bt, void* out, int M, int N, int K, int block_n, mi3d_stream_t stream);

int mi3d_conv3x3_f16(const void* x, const void* w, void* y, int Nimg, int H, int W, int Cin, int Cout, int block_n,
                     const float* bias, const void* residual, mi3d_stream_t stream);

/* Stable-Diffusion engine: a statically planned launch list over the tile kernel above + memory-bound kernels.
 * Configuration mirrors diffusers' UNet2DConditionModel / AutoencoderKL config.json fields that nerf/sd.py:41,53 load. */
typedef struct {
    int in_ch, out_ch;        /* 4, 4 */
    int n_levels;             /* len(block_out_channels): 4 for SD-2.0-base; 0 = no U-Net in this engine */
    int block_out[4];         /* 320, 640, 1280, 1280 */
    int layers_per_block;     /* 2 */
    int heads[4];             /* 5, 10, 20, 20 (head_dim 64) */
    int cross_dim;            /* 1024 */
    int ctx_len;              /* 77 text tokens */
    int groups;               /* 32 */
    int latent_hw;            /* 64 (nerf/sd.py:124 always feeds 512x512 -> 64x64 latents) */
    int batch;                /* 2 = [uncond, text] (nerf/sd.py:143) */
} mi3d_unet_cfg;

typedef struct {
    int in_ch, latent_ch;     /* 3, 4 */
    int n_levels;             /* 4; 0 = no VAE in this engine */
    int block_out[4];         /* 128, 256, 512, 512 */
    int layers_per_block;     /* 2 */
    int groups;               /* 32 */
    int image_hw;             /* 512 */
    int decoder;              /* != 0: also plan the decoder (mi3d_sd_decode; the denoise side branch of nerf/sd.py:153-159) */
} mi3d_vae_cfg;

typedef struct mi3d_sd* mi3d_sd_t;

/* HOST: bytes of device workspace the engine needs (weights + activations + tapes; nothing else is ever allocated) */
size_t mi3d_sd_workspace_bytes(const mi3d_unet_cfg* unet, const mi3d_vae_cfg* vae);
/* HOST: plans the launch lists inside `workspace` (device memory owned by the caller); NULL on failure */
mi3d_sd_t mi3d_sd_create(const mi3d_unet_cfg* unet, const mi3d_vae_cfg* vae, void* workspace, size_t workspace_bytes);
void mi3d_sd_destroy(mi3d_sd_t h);

/* Parameters are enumerated by their diffusers state_dict names ("down_blocks.0.resnets.0.conv1.weight", VAE names are
 * prefixed as in AutoencoderKL: "encoder....", "quant_conv...."; a '#...' suffix marks a derived copy of the base tensor).
 * load: src = fp32 DEVICE tensor in the diffusers layout; partner_src = the matching ".bias" for GEGLU proj weights. */
int mi3d_sd_num_params(mi3d_sd_t h);
const char* mi3d_sd_param_name(mi3d_sd_t h, int i);
long long mi3d_sd_param_numel(mi3d_sd_t h, int i);
int mi3d_sd_param_shape(mi3d_sd_t h, int i, int* shape4); /* returns rank */
int mi3d_sd_load_param(mi3d_sd_t h, int i, const float* src, const float* partner_src, mi3d_stream_t stream);

/* replaces nerf/sd.py:124 (F.interpolate to 512) + :133,212-220 (encode_imgs: vae.encode(2x-1).latent_dist.sample()*0.18215)
 * pred_rgb [1,3,H,W] fp32 in [0,1]; eps_posterior, latents [1,4,h,w] fp32 (h = image_hw/8). */
int mi3d_sd_encode(mi3d_sd_t h, const float* pred_rgb, int H, int W, const float* eps_posterior, float* latents, mi3d_stream_t stream);
/* the autograd half of latents.backward(gradient=grad) (nerf/sd.py:171): d latents -> d pred_rgb, weights frozen */
int mi3d_sd_encode_backward(mi3d_sd_t h, const float* grad_latents, const float* eps_posterior, int H, int W, float* grad_pred_rgb,
                            mi3d_stream_t stream);
/* replaces nerf/sd.py:138-170: scheduler.add_noise, unet([x,x], t, text_embeddings).sample, CFG (text + gs*(text-uncond)),
 * w = 1 - alphas[t], grad = nan_to_num(w*(noise_pred - noise)).  t: DEVICE int64 scalar; alphas_cumprod: DEVICE fp32 [1000];
 * text_embeddings fp32 [2,77,cross_dim] (uncond first); noise_pred / grad (nullable) fp32 [1,4,h,w]. */
int mi3d_sd_unet_sds(mi3d_sd_t h, const float* latents, const float* noise, const long long* t, const float* alphas_cumprod,
                     const float* text_embeddings, float guidance_scale, float* noise_pred, float* grad, mi3d_stream_t stream);
/* The "denoise" side branch of train_step (nerf/sd.py:153-159), taken on non-large views when t <= 0.4 T:
 * replaces scheduler.step (DDIM, eta 0, t -> t-1; fp32 [1,4,h,w], n = 4*h*w elements) and decode_latents (nerf/sd.py:201-210:
 * vae.decode(latents / 0.18215) -> (x/2 + 0.5).clamp(0,1); imgs fp32 [1,3,image_hw,image_hw]).  Forward only, like the reference. */
int mi3d_sd_ddim_step(const float* noise_pred, const float* latents_noisy, const long long* t, const float* alphas_cumprod,
                      float* prev_sample, int n, mi3d_stream_t stream);
int mi3d_sd_decode(mi3d_sd_t h, const float* latents, float* imgs, mi3d_stream_t stream);
/* live timing of the tensor-core tile kernel: enable=1 starts recording CUDA events around every launch; enable=0 stops and
 * returns the summed kernel time (ms) and launch count (HOST pointers; synchronises on the recorded events). */
int mi3d_sd_profile(mi3d_sd_t h, int enable, float* gemm_ms_host, int* launches_host);
/* same, and (enable=0) also writes one text line per timed launch to dump_path_host: "M N K block_n splits conv batch epi ms" */
int mi3d_sd_profile_dump(mi3d_sd_t h, int enable, float* gemm_ms_host, int* launches_host, const char* dump_path_host);
/* CUDA-graph replay of the three static launch lists (U-Net, VAE encode, VAE input-gradient): from its third call on a list is
 * one cudaGraphLaunch.  `stream` of the run calls must then be capturable (not the legacy default stream).  Off by default at the
 * C level; nerf/sd.py turns it on together with an engine-owned stream.  mi3d_sd_graph_replays: lists currently instantiated. */
int mi3d_sd_set_graph_replay(mi3d_sd_t h, int enable);
int mi3d_sd_graph_replays(mi3d_sd_t h);
/* debug tap: device pointer + size of a named intermediate ("unet.mid", "vae.grad_in", ...) */
int mi3d_sd_debug_tensor(mi3d_sd_t h, const char* name, void** ptr, size_t* bytes);

/* ------------------------------------------------------------------------------------------------------
 * B4: refine-stage point renderer  (replaces pytorch3d rasterize_points + compositing.alpha_composite as called by
 *     render_point, nerf/refine_utils.py:306-333)
 * ------------------------------------------------------------------------------------------------------
 * Square S x S image.  pts_ndc [P,3]: NDC x, y (pixel (row i, column j) has centre (-1 + (2 (S-1-j) + 1) / S, same for i)) and
 * camera depth z; points with z < 0 or a non-finite coordinate are skipped.  A point is a candidate of a pixel when its squared
 * NDC distance d <= radius^2; each pixel keeps the K (1..16) candidates of smallest (z, point index), ascending:
 * idx [S,S,K] int32 (-1 = empty), dists [S,S,K] fp32 (d; -1 = empty).  With a_k = 1 - sqrt(clamp(0.1 d_k / radius^2, 1e-3, 1)),
 * T_0 = 1, T_k+1 = T_k (1 - a_k):  out [C,S,S] = sum_k T_k a_k feats[idx_k].  Background is 0.
 * workspace: mi3d_point_render_workspace_bytes(P, S, K, radius) bytes (tile lists; 0 = bad arguments).
 * backward: g_feats [P,C] (overwritten) from g_out [C,S,S] and the forward's idx / dists; deterministic, no atomics. */
size_t mi3d_point_render_workspace_bytes(uint32_t P, uint32_t S, uint32_t K, float radius);
int mi3d_point_render_forward(const float* pts_ndc, const float* feats, uint32_t P, uint32_t C, uint32_t S, uint32_t K, float radius,
                              int* idx, float* dists, float* out, void* workspace, size_t workspace_bytes, mi3d_stream_t stream);
int mi3d_point_render_backward(const float* g_out, const float* pts_ndc, const int* idx, const float* dists, uint32_t P, uint32_t C,
                               uint32_t S, uint32_t K, float radius, float* g_feats, mi3d_stream_t stream);

/* unit-test entry for the hand-written kind::tf32 tiles of the field kernels (3-term split, K-major / MN-major operands):
 * mode 0: d[128,N] = a[128,K] . b[N,K]^T ; mode 1: d = a[K,128]^T . b[K,N] ; mode 2: d = a[128,K] . b[K,N].  fp32 in/out. */
int mi3d_tf32_tile_test(const float* a, const float* b, float* d, int N, int K, int mode, mi3d_stream_t stream);

const char* mi3d_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MI3D_H */
