/* plenoctree_b200.h — C ABI of the B200-native NeRF-SH hot path.
 *
 * The reference (sxyu/plenoctree) has no FFI layer of its own: its boundary for this path is a
 * set of Python call signatures (SURVEY.md §8b).  Each entry point below is what a binding for
 * one of those call sites would call; the reference interface it replaces is cited as
 * file:line relative to the reference tree.  INTEGRATION.md shows the ctypes stubs.
 *
 * Conventions
 *   - every pointer named *_dev is a CUDA device pointer on the current device, *_host is host
 *     memory; `stream` is a cudaStream_t passed as void* (NULL = default stream);
 *   - all functions return 0 on success, non-zero on error; pob_last_error() returns a
 *     thread-local message for the last failure (never NULL);
 *   - nothing here falls back to the CPU: without a CUDA device every compute call fails.
 *   - precision: POB_PREC_FP16 = fp16 operands / fp32 accumulate on tcgen05 (the numerics class
 *     of the reference's TF32-default XLA GPU path); POB_PREC_FP16X3 = error-compensated 3-pass
 *     split (fp32-class accuracy, 1/3 of the tensor throughput).
 */
#ifndef PLENOCTREE_B200_H
#define PLENOCTREE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define POB_PREC_FP16 1
#define POB_PREC_FP16X3 3

/* ---------------------------------------------------------------------------------------------
 * Library / device
 * ------------------------------------------------------------------------------------------- */
int pob_abi_version(void);
const char* pob_last_error(void);
/* number of SMs of the current CUDA device (persistent-grid size); <0 on error */
int pob_sm_count(void);

/* Instrumentation used by bench.py: number of kernels this library has launched so far, and
 * optional CUDA-event timing per kernel class.  pob_timing_read fills ms_out[5] / launches_out[5] for
 * {mlp_fwd, mlp_bwd, mlp_wgrad, per-ray render stages, optimiser (reduce, Adam, pack)} and returns 5;
 * it synchronises with the recorded events. */
long long pob_launch_count(void);
void pob_timing_enable(int on);
int pob_timing_read(double* ms_out, long long* launches_out);

/* ---------------------------------------------------------------------------------------------
 * Parameters of one MLP (MLP_0 coarse / MLP_1 fine; nerf_sh/nerf/models.py:83-104).
 * Flat fp32 layout = Dense_0..Dense_9 in order, each kernel [in,out] row-major then bias [out]
 * (nerf_sh/nerf/model_utils.py:60-93; Dense index mapping octree/nerf/models.py:79-102).
 * ------------------------------------------------------------------------------------------- */
/* number of fp32 parameters of one MLP for SH degree sh_deg (-1 = plain RGB head, 3 channels) */
int64_t pob_param_count(int sh_deg);
/* byte size of the packed tensor-core operand blob of one MLP */
int64_t pob_packed_bytes(int sh_deg);
/* flat fp32 parameters -> packed blob (fp16 hi/lo forward images, transposed images, biases) */
int pob_pack_weights(const float* flat_dev, int sh_deg, void* packed_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * NerfModel.eval_points_raw(points, viewdirs=None, coarse=False) -> (raw_rgb[M,3K], raw_sigma[M,1])
 *   JAX:   nerf_sh/nerf/models.py:143-181      torch twin: octree/nerf/models.py:211-252
 * raw_rgb_dev may be NULL (sigma only: octree/extraction.py:271,316 discard rgb).
 * ------------------------------------------------------------------------------------------- */
int pob_eval_points_raw(const void* packed_dev, int sh_deg, const float* points_dev, int64_t m,
                        float* raw_rgb_dev, float* raw_sigma_dev, int precision, void* stream);

/* NerfModel.eval_points(points, viewdirs) -> (rgb[M,3], sigma[M,1])  (models.py:183-214):
 * eval_sh at the per-point view direction, sigmoid / relu.  out_rgbs_dev: [M,4] = (r,g,b,sigma). */
int pob_eval_points(const void* packed_dev, int sh_deg, const float* points_dev,
                    const float* viewdirs_dev, int64_t m, float* out_rgbs_dev, int precision,
                    void* stream);

/* Dense-grid sweep of octree.extraction (auto_scale / step1: octree/extraction.py:244-320).
 * Evaluates raw sigma (and optionally raw SH coefficients) at the voxel centres
 *   ((i + 0.5)/reso - offset[a]) / scale[a]
 * of the slab ix in [x0, x0+nx), iy in [0,ny), iz in [0,nz), flattened x-major like
 * torch.meshgrid(xx,yy,zz).reshape(3,-1).T.  No host grid, no H2D copies. */
int pob_eval_grid(const void* packed_dev, int sh_deg, int reso, int x0, int nx, int ny, int nz,
                  const float offset[3], const float scale[3], float* raw_rgb_dev,
                  float* raw_sigma_dev, int precision, void* stream);

/* Anti-aliasing pass of octree.extraction step2 (octree/extraction.py:355-394, SH data formats): the caller
 * provides samples_per_cell points per leaf (tree[inds].sample(S), [n_cells*S, 3], cell-major);
 * out_dev [n_cells, 3K+1] = mean over the S samples of cat([raw_rgb, raw_sigma], -1)  (:391-393). */
int pob_eval_cells_mean(const void* packed_dev, int sh_deg, const float* points_dev, int64_t n_cells,
                        int samples_per_cell, float* out_dev, int precision, void* stream);

/* Host-buffer convenience form of pob_eval_points_raw (H2D, kernel, D2H inside the call);
 * the e2e arm of bench.py times this. */
int pob_eval_points_raw_host(const void* packed_dev, int sh_deg, const float* points_host,
                             int64_t m, float* raw_rgb_host, float* raw_sigma_host,
                             int precision);

/* ---------------------------------------------------------------------------------------------
 * Per-ray stages (exposed individually for parity tests; pob_render_rays chains them).
 * ------------------------------------------------------------------------------------------- */
/* model_utils.sample_along_rays (nerf_sh/nerf/model_utils.py:104-142).  z_base[n_samples] is the
 * un-jittered table near*(1-t)+far*t (or the lindisp form) built by the host with the reference
 * expression; t_rand [n_rays,n_samples] in [0,1) replaces random.uniform (NULL = randomized False). */
int pob_sample_coarse(const float* z_base_dev, const float* t_rand_dev, int n_rays, int n_samples,
                      float* z_out_dev, void* stream);

/* The random draws of one randomized training step in ONE launch (replaces jax.random.uniform at
 * nerf_sh/nerf/model_utils.py:137 (t_rand [n_t] ~ U[0,1)), :262 (u [n_u] ~ U[0,1)) and nerf_sh/train.py:79
 * (sp_points [n_sp] ~ U[-radius, radius))): Philox4x32-10 keyed by `seed`, counter = (index, stream, step).  The
 * threefry streams of the reference cannot be reproduced without JAX; parity tests inject their own draws.
 * step_dev (device float, or NULL) overrides `step`, so that a replayed CUDA graph draws fresh numbers. */
int pob_draw_uniforms(uint64_t seed, float step, const float* step_dev, float* t_rand_dev, int64_t n_t,
                      float* u_dev, int64_t n_u, float* sp_points_dev, int64_t n_sp, float sp_radius, void* stream);
/* model_utils.volumetric_rendering (model_utils.py:176-222).  rgbs [n_rays,n_samples,4] = (rgb, sigma)
 * after activations; outputs comp_rgb [n_rays,3], disp, acc [n_rays], weights [n_rays,n_samples]
 * (disp / acc / weights may be NULL). */
int pob_composite(const float* rgbs_dev, const float* z_dev, const float* dirs_dev, int n_rays, int n_samples,
                  int white_bkgd, float* out_rgb_dev, float* out_disp_dev, float* out_acc_dev,
                  float* out_weights_dev, void* stream);
/* reverse-mode of pob_composite composed with the MSE of loss_fn (nerf_sh/train.py:86-96) and with
 * sigmoid'/relu': g_out [n_rays,n_samples,4] = d/d(pre-activation rgb after eval_sh, raw sigma) of
 * gscale/2 * sum (comp_rgb - pixels)^2;  sq_err_sum_dev (may be NULL) += sum (comp_rgb - pixels)^2. */
int pob_composite_bwd(const float* rgbs_dev, const float* z_dev, const float* dirs_dev, const float* comp_rgb_dev,
                      const float* pixels_dev, int n_rays, int n_samples, int white_bkgd, float gscale,
                      float* g_out_dev, float* sq_err_sum_dev, void* stream);
/* model_utils.sample_pdf (model_utils.py:225-314): inverse-CDF resampling from weights[...,1:-1] over the
 * mid-point bins, then the sorted union with the coarse depths.  u: [n_fine] table (u_per_ray = 0,
 * randomized False: linspace(0, 1-eps)) or [n_rays,n_fine] uniforms.  z_out [n_rays, n_coarse+n_fine]. */
int pob_sample_pdf(const float* z_coarse_dev, const float* weights_dev, const float* u_dev, int u_per_ray,
                   int n_rays, int n_coarse, int n_fine, float* z_out_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * NerfModel.__call__(rng_0, rng_1, rays, randomized) -> [(rgb,disp,acc)_coarse, (rgb,disp,acc)_fine]
 *   nerf_sh/nerf/models.py:216-348   (callers: train.py:70, utils.render_image utils.py:331-381)
 * ------------------------------------------------------------------------------------------- */
typedef struct pob_render_config {
  int sh_deg;               /* flag sh_deg            (nerf_sh/nerf/utils.py:135) */
  int num_coarse_samples;   /* flag num_coarse_samples (utils.py:126)             */
  int num_fine_samples;     /* flag num_fine_samples   (utils.py:130); 0 = single level */
  int white_bkgd;           /* flag white_bkgd */
  int max_rays;             /* capacity of the workspace in rays per call */
  int sparsity_npoints;     /* flag sparsity_npoints (training workspace only) */
  /* model_utils.add_gaussian_noise (nerf_sh/nerf/model_utils.py:317-332; flag noise_std, utils.py:137-142):
   * optional per-sample normal draws ALREADY multiplied by noise_std, added to raw sigma before relu at the
   * coarse [n_rays, Nc] and fine [n_rays, Nc+Nf] level; NULL = off (randomized False or noise_std None). */
  const float* sigma_noise_coarse_dev;
  const float* sigma_noise_fine_dev;
} pob_render_config;

/* bytes of device scratch the render (training=0) / training (training=1) calls need */
int64_t pob_workspace_bytes(const pob_render_config* cfg, int training);

/* out_coarse / out_fine: [n_rays,5] = (r,g,b,disp,acc).  t_rand NULL = randomized False.
 * z_fine_dev (normally NULL): [n_rays, Nc+Nf] sorted depths that replace the sample_pdf stage — lets a
 * caller (and the parity tests) pin the fine-level sample positions. */
int pob_render_rays(const pob_render_config* cfg, const void* packed_coarse_dev, const void* packed_fine_dev,
                    const float* origins_dev, const float* directions_dev, const float* viewdirs_dev,
                    int n_rays, const float* z_base_dev, const float* t_rand_dev, const float* u_dev,
                    int u_per_ray, const float* z_fine_dev, float* out_coarse_dev, float* out_fine_dev,
                    void* workspace_dev, int precision, void* stream);

/* ---------------------------------------------------------------------------------------------
 * train_step (nerf_sh/train.py:51-121), split at the gradient all-reduce:
 *   pob_loss_and_grad = jax.value_and_grad(loss_fn)   (train.py:66-116)
 *   [caller: all-reduce-mean of grad_flat over ranks   (train.py:117) ]
 *   pob_adam_update   = optimizer.apply_gradient       (train.py:119) + operand re-pack
 * ------------------------------------------------------------------------------------------- */
typedef struct pob_train_hparams {
  float sparsity_weight;    /* flag sparsity_weight (utils.py:191) ; 0 disables the term */
  float sparsity_length;    /* flag sparsity_length */
  float loss_scale;         /* power-of-two scale applied to the fp16 gradient chain, divided out of grad_flat */
} pob_train_hparams;

/* grad_flat [num_mlps * pob_param_count] (MLP_0 then MLP_1, reference flat order), per-rank gradient of
 *   mean((rgb_f-px)^2) + mean((rgb_c-px)^2) + sparsity_weight*(1-mean(exp(-len*relu(sigma(p)))))
 * stats [8] (device): [0] sum (rgb_fine-px)^2, [1] sum (rgb_coarse-px)^2, [2] sum exp(-len*relu(sigma)). */
int pob_loss_and_grad(const pob_render_config* cfg, const pob_train_hparams* hp, const void* packed_coarse_dev,
                      const void* packed_fine_dev, const float* origins_dev, const float* directions_dev,
                      const float* viewdirs_dev, const float* pixels_dev, int n_rays, const float* z_base_dev,
                      const float* t_rand_dev, const float* u_dev, int u_per_ray, const float* z_fine_dev,
                      const float* sp_points_dev, float* grad_flat_dev, float* stats_dev, void* workspace_dev,
                      void* stream);

/* flax.optim.Adam (beta1 .9, beta2 .999, eps 1e-8; nerf_sh/nerf/models.py:44) on the flat buffers of
 * num_mlps MLPs, g = grad*grad_mult + weight_decay_coef*param, then re-packs the operand blobs.
 * `step` = number of updates already applied (flax optimizer.state.step).  lr_step_dev (device float[2] = {lr,
 * step}, or NULL) overrides the two host values, so that a captured CUDA graph of the step can be replayed with a
 * new learning rate and step count. */
int pob_adam_update(int sh_deg, int num_mlps, float* params_dev, const float* grads_dev, float* m_dev,
                    float* v_dev, float lr, float step, const float* lr_step_dev, float grad_mult,
                    float weight_decay_coef, void* packed_coarse_dev, void* packed_fine_dev, void* stream);

/* Profiling aid: pob_eval_points_raw (sigma only, FP16) that also records clock64() stamps of CTA 0 into
 * trace_dev[3][256] (role 0 = MMA issuer, 1/2 = first epilogue warp of tile X/Y); scripts/trace_summary.py.
 * save_*_dev (all or none; sized like the training workspace: 512 KB, 16 KB and 4 KB per 128 samples) turn
 * on the training-mode stores so their cost shows in the trace. */
int pob_debug_trace_fwd(const void* packed_dev, int sh_deg, const float* points_dev, int64_t m,
                        float* raw_sigma_dev, unsigned long long* trace_dev, void* save_h_dev,
                        void* save_e_dev, void* save_mask_dev, void* stream);

/* Profiling aid: one mlp_bwd launch (dgrad chain, FP16) on caller-provided inputs — per-sample gradients g_dev
 * [m,4], view directions [m,3], relu masks (4 KB per 128 samples and layer), dZ / dO destinations sized like the
 * training workspace — recording clock64() stamps of CTA 0 into trace_dev[2][256] (role 0 = MMA issuer, 1 = first
 * epilogue warp of tile X); scripts/trace_bwd.py. */
int pob_debug_trace_bwd(const void* packed_dev, int sh_deg, int64_t m, const float* g_dev, const float* viewdirs_dev,
                        const void* mask_dev, void* save_dz_dev, void* save_do_dev, unsigned long long* trace_dev,
                        void* stream);

/* ---------------------------------------------------------------------------------------------
 * PlenOctree side (SURVEY.md §8 rows a13-middle and a15).  These entry points stand where the
 * reference calls the third-party `svox` extension (absent from the reference tree; the oracle
 * restates its published algorithm, parity unpinned — see oracle/octree_oracle.py):
 *   svox.N3Tree / N3TreeView          octree/extraction.py:330-394,489-509
 *   svox.VolumeRenderer.render_persp  octree/optimization.py:174-229, octree/nerf/utils.py:448-498
 *   svox _C.grid_weight_render        octree/extraction.py:181-214
 * Tree layout (svox N3Tree, keys of tree.npz: octree/compression.py:75-95):
 *   data  [n_nodes, N, N, N, data_dim] fp32, sigma is the LAST channel (octree/extraction.py:391),
 *         SH coefficients channel-major c*K + k before it (same order as raw_rgb of eval_points_raw);
 *   child [n_nodes, N, N, N] int32: index of the child node minus the index of this node, 0 = leaf;
 *   world -> tree coordinates: p * invradius + offset in [0,1]^3.
 * ------------------------------------------------------------------------------------------- */
#define POB_OCTREE_RGBA 0 /* data_dim 4: colour = sigmoid(data[0:3])                              */
#define POB_OCTREE_SH 1   /* data_dim 3K+1: colour = sigmoid(sum_k Y_k(viewdir) * data[c*K+k])    */

typedef struct pob_octree {
  const float* data_dev;
  const int32_t* child_dev;
  int64_t n_nodes;
  int N;          /* branch factor per axis (flag tree_branch_n, octree/extraction.py:100) */
  int data_dim;
  int basis_dim;  /* K */
  int format;     /* POB_OCTREE_* */
  float offset[3];
  float invradius[3];
} pob_octree;

/* svox RenderOptions as VolumeRenderer fills them: step_size = flag renderer_step_size
 * (octree/nerf/utils.py:211-215), background_brightness 1, and sigma_thresh = stop_thresh = 1e-2 when
 * fast=True (evaluation without --no_early_stop, octree/nerf/utils.py:472), 0 otherwise. */
typedef struct pob_octree_opts {
  float step_size;
  float background_brightness;
  float sigma_thresh;
  float stop_thresh;
} pob_octree_opts;

/* perspective camera: c2w = first three rows of the camera-to-world matrix, row-major [3][4]
 * (svox CameraSpec: octree/extraction.py:194-199).  16 floats, also the element type of camera arrays. */
typedef struct pob_camera {
  float c2w[12];
  float fx, fy;
  float width, height;
} pob_camera;

/* VolumeRenderer.forward(rays) / render_persp(c2w, width, height, fx): composite the tree along rays.
 * Either explicit rays (origins/dirs/vdirs [n_rays,3], cam NULL) or a pixel-row slab [row0, row0+nrows) of a
 * perspective camera (cam != NULL, ray pointers ignored; out is [nrows*width, 3] row-major).
 * counters_dev (may be NULL): [2] += {leaf visits, contributing leaf visits} for the roofline accounting. */
int pob_octree_render(const pob_octree* tree, const pob_octree_opts* opts, const float* origins_dev,
                      const float* dirs_dev, const float* vdirs_dev, int64_t n_rays, const pob_camera* cam,
                      int row0, int nrows, float* out_rgb_dev, unsigned long long* counters_dev, void* stream);

/* reverse mode of the above for an upstream gradient grad_out [n,3]: grad_data_dev (same shape as data,
 * ACCUMULATED into) += d<grad_out, rgb>/d data.  Thresholds are ignored like in svox's backward. */
int pob_octree_render_backward(const pob_octree* tree, const pob_octree_opts* opts, const float* origins_dev,
                               const float* dirs_dev, const float* vdirs_dev, int64_t n_rays, const pob_camera* cam,
                               int row0, int nrows, const float* grad_out_dev, float* grad_data_dev, void* stream);

/* One training image of octree.optimization (octree/optimization.py:201-207) in one launch:
 *   im = render_persp(c2w); mse = mean((clamp(im,0,1) - gt)^2); mse.backward()
 * over the pixel rows [row0,row0+nrows): grad_data += grad_scale * d sum((clamp(im)-gt)^2) / d data,
 * *sq_err_sum_dev += sum((clamp(im)-gt)^2)  (grad_scale = 1/(H*W*3) gives the reference's mean);
 * gt_rgb_dev [nrows*width,3]; out_rgb_dev (may be NULL) receives the rendered slab. */
int pob_octree_train_persp(const pob_octree* tree, const pob_octree_opts* opts, const pob_camera* cam, int row0,
                           int nrows, const float* gt_rgb_dev, float grad_scale, float* grad_data_dev,
                           double* sq_err_sum_dev, float* out_rgb_dev, void* stream);

/* torch.optim.SGD(lr, momentum 0).step() fused with zero_grad (octree/optimization.py:187-189,205-208):
 * data -= lr * grad; grad = 0, touching only entries whose gradient is non-zero. */
int pob_octree_sgd_step(float* data_dev, float* grad_dev, int64_t n, float lr, void* stream);

/* torch.optim.Adam(lr, eps) (betas 0.9 / 0.999, no weight decay; octree/optimization.py:190-193, the `--nosgd` branch)
 * fused with zero_grad: m, v are the caller's moment buffers (same shape as data), `step` = updates already applied. */
int pob_octree_adam_step(float* data_dev, float* grad_dev, float* m_dev, float* v_dev, int64_t n, float lr, float step,
                         float eps, void* stream);

/* N3Tree.__getitem__(points): packed leaf index node*N^3 + (i*N + j)*N + k of the leaf holding each world
 * point (points clamped into the volume like svox). */
int pob_octree_query(const pob_octree* tree, const float* points_dev, int64_t n, int64_t* leaf_index_dev,
                     void* stream);

/* calculate_grid_weights (octree/extraction.py:181-214): march all pixels of n_cams cameras (cams_dev: device
 * array of pob_camera) through the dense sigma grid [reso]^3 and max-accumulate the per-voxel compositing
 * weight into max_weight_dev (caller zero-initialises; all cameras in one launch, no per-camera grids).
 * hit_dev (may be NULL): uint8 [reso]^3 set to 1 where any ray contributed. */
int pob_grid_weight_render(const float* sigma_grid_dev, int reso, const pob_camera* cams_dev, int n_cams,
                           int max_width, int max_height, const float offset[3], const float invradius[3],
                           const pob_octree_opts* opts, float* max_weight_dev, uint8_t* hit_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Test bench for the tcgen05 descriptor conventions (tests/test_umma_probe.py).
 * Runs `nops` tcgen05.mma (kind::f16, M=128) on two shared-memory images and returns the
 * [128 x out_cols] fp32 accumulator.
 * ------------------------------------------------------------------------------------------- */
int pob_umma_probe(const void* a_img_dev, uint32_t a_bytes, const void* b_img_dev,
                   uint32_t b_bytes, uint32_t b_off, const uint64_t* adesc_dev,
                   const uint64_t* bdesc_dev, const uint32_t* dcol_dev, const uint32_t* accum_dev,
                   int nops, uint32_t idesc, int out_cols, float* out_dev, void* stream);

/* CTA-pair variant (tcgen05 cta_group::2, cluster of two CTAs, M = 256 in idesc): CTA r stages
 * a_img + r*a_bytes and b_img + r*b_bytes (its 128 A rows and its half of the B rows) at the same
 * shared-memory offsets; returns the [256 x out_cols] accumulator (rows 128r.. from CTA r). */
int pob_umma_probe_pair(const void* a_img_dev, uint32_t a_bytes, const void* b_img_dev,
                        uint32_t b_bytes, uint32_t b_off, const uint64_t* adesc_dev,
                        const uint64_t* bdesc_dev, const uint32_t* dcol_dev, const uint32_t* accum_dev,
                        int nops, uint32_t idesc, int out_cols, float* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PLENOCTREE_B200_H */
