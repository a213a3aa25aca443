// kernels.h — internal launch interface between the C-ABI (capi.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pob {

// ---- packed weights of one MLP (device pointers; produced by launch_pack_weights) ----------
struct MlpPacked {
  const uint8_t* w_hi;    // forward slot images, fp16 "hi" part  (fwd_image_bytes(NH))
  const uint8_t* w_lo;    // forward slot images, fp16 residual   (same layout)
  const uint8_t* wt_hi;   // dgrad slot images (transposed weights), fp16
  const float* bias;      // [8*256 + MAX_NH]: trunk biases then heads bias in packed order
};

enum SrcMode : int { SRC_POINTS = 0, SRC_RAYS = 1, SRC_GRID = 2 };
enum OutMode : int { OUT_RAW = 0, OUT_SIGMA = 1, OUT_RGBS = 2, OUT_CELL_MEAN = 3 };

struct FwdParams {
  // ---- sample source ----
  int src_mode;
  long long M;                 // number of samples (rows)
  const float* points;         // SRC_POINTS: [M,3]
  const float* origins;        // SRC_RAYS:   [R,3]
  const float* directions;     //             [R,3]
  const float* zvals;          //             [R, n_per_ray]
  int n_per_ray;
  // SRC_RAYS may carry `M - M_rays` free points behind the ray samples (the sparsity-loss points of the training
  // step ride on the main level's launches instead of three 40-CTA launches of their own): rows [M_rays, M)
  long long M_rays;            // SRC_RAYS: R * n_per_ray (== M when there are no extra points)
  const float* extra_points;   // [M - M_rays, 3]
  const float* viewdirs;       // OUT_RGBS: [R,3] (SRC_RAYS) or [M,3] (SRC_POINTS)
  const float* sigma_noise;    // OUT_RGBS, optional [M]: added to raw sigma before relu (model_utils.py:317-332)
  // SRC_GRID: voxel centres ((i + 0.5)/reso - offset)/scale, x-major flattening (ix,iy,iz)
  int g_reso;                  // arange length the reference normalises by
  int g_x0, g_nx, g_ny, g_nz;  // slab: ix in [g_x0, g_x0+g_nx), iy in [0,g_ny), iz in [0,g_nz)
  float g_offset[3], g_scale[3];
  // ---- model ----
  MlpPacked w;
  int sh_deg;                  // -1: 3 raw rgb channels, K = 1
  int K;                       // (sh_deg+1)^2
  int NH;                      // padded heads width, multiple of 16, <= 80
  // ---- outputs ----
  int out_mode;
  float* out_rgb;              // OUT_RAW: [M, 3K] (reference channel-major order c*K+k)
  float* out_sigma;            // OUT_RAW / OUT_SIGMA: [M]
  float4* out_rgbs;            // OUT_RGBS: [M] (sigmoid(rgb), relu(sigma))
  float* out_cell;             // OUT_CELL_MEAN: [M / cell_S, 3K+1] += mean over the cell's samples of
  int cell_S;                  //   cat([raw_rgb, raw_sigma]) (octree/extraction.py:391-393); zeroed by caller
  // ---- training saves (fast mode only; null = off) ----
  uint8_t* save_h;             // [ntile][8][64 KB] activation tile images h_0..h_7
  uint8_t* save_e;             // [ntile][16 KB]   posenc tile images
  uint32_t* save_mask;         // [8][ntile*128][8] relu masks (bit i of word c = col 32c+i)
  // ---- optional cycle trace of CTA 0 (debug/profiling; null = off): [3 roles][256] clock64 stamps
  unsigned long long* trace;
};

// padded heads width for K spherical-harmonic coefficients per channel
inline int heads_width(int K) { return ((1 + 3 * K) + 15) / 16 * 16; }
// bytes of one forward weight image (hi or lo)
inline size_t fwd_image_bytes(int NH) { return size_t(66) * 16384 + size_t(9) * NH * 64; }
// bytes of one dgrad weight image: heads (ceil(NH/32) slots) + layers 7..1 (8 slots each)
inline size_t bwd_image_bytes(int NH) { return size_t((NH + 31) / 32 + 7 * 8) * 16384; }

// precision: 1 = single fp16 pass (10-bit mantissa operands, fp32 accumulate; CTA pairs, cta_group::2),
//            3 = error-compensated 3-pass split (hi*hi + lo*hi + hi*lo; single CTAs)
cudaError_t launch_mlp_fwd(const FwdParams& p, int nsplit, int num_sms, cudaStream_t stream);

// flat fp32 parameters of one MLP in reference order (Dense_0..Dense_9: kernel [in,out] then
// bias) -> packed images.  `nparams` = param_count(K).
cudaError_t launch_pack_weights(const float* flat, int K, uint8_t* w_hi, uint8_t* w_lo,
                                uint8_t* wt_hi, float* bias, cudaStream_t stream);

cudaError_t launch_umma_probe(const void* a_img, uint32_t a_bytes, const void* b_img,
                              uint32_t b_bytes, uint32_t b_off, const uint64_t* adesc,
                              const uint64_t* bdesc, const uint32_t* dcol, const uint32_t* accum,
                              int nops, uint32_t idesc, int out_cols, float* out,
                              cudaStream_t stream);
cudaError_t launch_umma_probe_pair(const void* a_img, uint32_t a_bytes, const void* b_img,
                              uint32_t b_bytes, uint32_t b_off, const uint64_t* adesc,
                              const uint64_t* bdesc, const uint32_t* dcol, const uint32_t* accum,
                              int nops, uint32_t idesc, int out_cols, float* out,
                              cudaStream_t stream);


// ---- render.cu ------------------------------------------------------------------------------
cudaError_t launch_sample_coarse(const float* z_base, const float* t_rand, int R, int N, float* z_out,
                                 cudaStream_t st);
cudaError_t launch_composite_fwd(const float4* rgbs, const float* z, const float* dirs, int R, int N,
                                 int white_bkgd, float* out_rgb, float* out_disp, float* out_acc,
                                 float* out_weights, cudaStream_t st);
cudaError_t launch_composite_bwd(const float4* rgbs, const float* z, const float* dirs,
                                 const float* comp_rgb, const float* pixels, int R, int N, int white_bkgd,
                                 float gscale, float4* G, float* sq_err_sum, cudaStream_t st);
cudaError_t launch_sample_pdf(const float* z_c, const float* weights, const float* u, int u_per_ray, int R,
                              int Nc, int Nf, float* z_out, cudaStream_t st);
// t_rand [n_t], u [n_u] ~ U[0,1), sp [n_sp] ~ U[-radius, radius): Philox4x32-10 keyed by seed, counter (index, stream, step);
// step_dev (device float, optional) overrides `step` so that a captured graph draws fresh numbers on every replay
cudaError_t launch_draw_uniforms(unsigned long long seed, float step, const float* step_dev, float* t_rand,
                                 long long n_t, float* u, long long n_u, float* sp, long long n_sp, float sp_radius,
                                 cudaStream_t st);
// rgbs[i].w = relu(sigma) of the sparsity points (as the OUT_RGBS epilogue leaves it); G[i] = (0,0,0, dL/dsigma_raw)
cudaError_t launch_sparsity_grad(const float4* rgbs, int n, float length, float coef, float4* G,
                                 float* exp_sum, cudaStream_t st);

// ---- mlp_bwd.cu -----------------------------------------------------------------------------
struct BwdParams {
  long long M;
  const float4* G;          // [M] (d pre_r, d pre_g, d pre_b, d sigma_raw), loss-scaled
  const float* viewdirs;    // [R,3] (n_per_ray > 0) or [M,3] (n_per_ray == 0)
  int n_per_ray;
  long long M_rays;         // rows [M_rays, M) are free points (sigma gradient only): no view direction
  MlpPacked w;
  int sh_deg, K, NH;
  const uint32_t* mask;     // [8][Mpad][8] from mlp_fwd
  uint8_t* save_dz;         // [ntile][8][64 KB]
  uint8_t* save_do;         // [ntile][32 KB]
  unsigned long long* trace;   // optional cycle trace of CTA 0 (null = off): [2 roles][256] clock64 stamps
};
cudaError_t launch_mlp_bwd(const BwdParams& p, int num_sms, cudaStream_t stream);   // CTA pairs

// ---- mlp_wgrad.cu ---------------------------------------------------------------------------
constexpr int WG_PARTIAL_FLOATS = 65536 + 256;
constexpr int WG_MAX_CTAS = 160;
constexpr int WG_NUM_ROLES = 10;
struct WgradSegment {
  const uint8_t *h, *dz, *e, *d_o;
};
struct WgradParams {
  WgradSegment seg;         // one level's tile arrays (its sparsity points ride behind the ray samples)
  long long seg_tiles;
  int NH;
  float* partials;          // [num_ctas][WG_PARTIAL_FLOATS]
  short cta_role[WG_MAX_CTAS], cta_index[WG_MAX_CTAS], cta_count[WG_MAX_CTAS];
};
// role -> [first CTA, count]; fills the per-CTA tables of `p`; returns number of CTAs to launch
int wgrad_assign_roles(WgradParams& p, int num_sms, int role_start[WG_NUM_ROLES],
                       int role_count[WG_NUM_ROLES]);
cudaError_t launch_mlp_wgrad(const WgradParams& p, int num_ctas, cudaStream_t stream);

// ---- optim.cu -------------------------------------------------------------------------------
// partials of one wgrad launch -> flat gradient of one MLP (reference layout), times inv_scale
cudaError_t launch_reduce_grads(const float* partials, const int role_start[WG_NUM_ROLES],
                                const int role_count[WG_NUM_ROLES], int K, float inv_scale,
                                float* grad_flat, cudaStream_t stream);
// flax.optim.Adam.apply_gradient on a flat buffer; grad is multiplied by grad_mult first
// lr_step_dev (optional, device [2] = {lr, step}) overrides the host lr / step: a captured graph replays with new values
cudaError_t launch_adam(float* param, const float* grad, float* m, float* v, long long n, float lr,
                        float step, const float* lr_step_dev, float beta1, float beta2, float eps, float grad_mult,
                        float weight_decay_coef, cudaStream_t stream);

// ---- flat parameter layout of one MLP (reference order) -------------------------------------
// Dense_i kernel is [in,out] row-major (flax), followed by its bias [out].
struct FlatLayout {
  int w_off[10], b_off[10], in_dim[10], out_dim[10], total;
};
inline FlatLayout flat_layout(int K) {
  FlatLayout L;
  int off = 0;
  for (int i = 0; i < 10; ++i) {
    int in = (i == 0) ? 63 : (i == 5 ? 319 : 256);
    int out = (i < 8) ? 256 : (i == 8 ? 1 : 3 * K);
    L.in_dim[i] = in;
    L.out_dim[i] = out;
    L.w_off[i] = off;
    off += in * out;
    L.b_off[i] = off;
    off += out;
  }
  L.total = off;
  return L;
}

}  // namespace pob
