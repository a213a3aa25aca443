// pipeline.cu — host-side sequencing of the kernels into the two reference-level operations:
//   pob_render_rays    = NerfModel.__call__            (nerf_sh/nerf/models.py:216-348)
//   pob_loss_and_grad  = value_and_grad(loss_fn)       (nerf_sh/train.py:66-116)
//   pob_adam_update    = optimizer.apply_gradient      (nerf_sh/train.py:119) + operand re-pack
// Everything is enqueued on the caller's stream; nothing synchronises with the host.
#include <cstring>
#include <string>

#include "../../include/plenoctree_b200.h"
#include "capi_util.h"
#include "common.cuh"
#include "kernels.h"

namespace {

using namespace pob;

struct Level {
  // sizes
  long long M;        // samples
  long long tiles;    // padded to an even number of 128-row tiles
  // buffers
  float* z;           // [R,N]
  float4* rgbs;       // [M]
  float* weights;     // [R,N]
  float* comp;        // [R,3]
  float* disp;        // [R]
  float* acc;         // [R]
  float4* G;          // [M]
  uint8_t *H, *E, *DZ, *DO;
  uint32_t* mask;
};

struct Workspace {
  Level lv[2];        // coarse, fine; in training the LAST level also carries the sparsity points behind its rays
  float* partials[2]; // wgrad partials of the two MLPs' launches
  size_t total;
};

size_t up(size_t x) { return (x + 1023) / 1024 * 1024; }

// tiles are scheduled four at a time (one CTA pair x two tiles): every per-tile array is padded to that unit
long long tiles_for(long long M) { return padded_rows(M) / TILE_M; }

// deterministic carve of the caller-provided workspace
Workspace carve(const pob_render_config& c, int training, uint8_t* base) {
  Workspace w;
  memset(&w, 0, sizeof(w));
  size_t off = 0;
  auto take = [&](size_t bytes) {
    uint8_t* p = base ? base + off : nullptr;
    off += up(bytes);
    return p;
  };
  const long long R = c.max_rays;
  const int Ns[2] = {c.num_coarse_samples, c.num_fine_samples > 0 ? c.num_coarse_samples + c.num_fine_samples : 0};
  const int last = c.num_fine_samples > 0 ? 1 : 0;
  for (int l = 0; l < 2; ++l) {
    Level& L = w.lv[l];
    const long long Mr = R * Ns[l];                                    // ray samples
    L.M = Mr + ((training && l == last) ? c.sparsity_npoints : 0);     // + sparsity points (train.py:77-83)
    L.tiles = tiles_for(L.M);
    if (Mr == 0) continue;
    L.z = (float*)take(sizeof(float) * Mr);
    L.rgbs = (float4*)take(sizeof(float4) * L.M);
    L.weights = (float*)take(sizeof(float) * Mr);
    L.comp = (float*)take(sizeof(float) * 3 * R);
    L.disp = (float*)take(sizeof(float) * R);
    L.acc = (float*)take(sizeof(float) * R);
    if (training) {
      L.G = (float4*)take(sizeof(float4) * L.M);
      L.H = take(size_t(L.tiles) * NUM_TRUNK * A_TILE_BYTES);
      L.E = take(size_t(L.tiles) * E_TILE_BYTES);
      L.DZ = take(size_t(L.tiles) * NUM_TRUNK * A_TILE_BYTES);
      L.DO = take(size_t(L.tiles) * 2 * A_CHUNK_BYTES);
      L.mask = (uint32_t*)take(size_t(NUM_TRUNK) * L.tiles * TILE_M * 8 * sizeof(uint32_t));
    }
  }
  if (training) {
    for (int i = 0; i < 2; ++i) w.partials[i] = (float*)take(sizeof(float) * WG_MAX_CTAS * WG_PARTIAL_FLOATS);
  }
  w.total = off;
  return w;
}

int check_cfg(const char* where, const pob_render_config* c) {
  if (!c) return pob_fail(where, "config is NULL");
  if (c->sh_deg < -1 || c->sh_deg > 4) return pob_fail(where, "sh_deg must be in [-1, 4]");
  if (c->num_coarse_samples < 3 || c->num_coarse_samples > 256)
    return pob_fail(where, "num_coarse_samples must be in [3, 256]");
  if (c->num_fine_samples < 0 || c->num_coarse_samples + c->num_fine_samples > 256)
    return pob_fail(where, "num_coarse_samples + num_fine_samples must be <= 256");
  if (c->max_rays <= 0) return pob_fail(where, "max_rays must be positive");
  if (c->sparsity_npoints < 0) return pob_fail(where, "sparsity_npoints must be >= 0");
  return 0;
}

FwdParams ray_fwd_params(const void* packed, int sh_deg, const float* o, const float* d, const float* v,
                         const float* z, int R, int N, float4* out) {
  FwdParams p = pob_base_params(packed, sh_deg);
  p.src_mode = SRC_RAYS;
  p.M = (long long)R * N;
  p.M_rays = p.M;
  p.origins = o;
  p.directions = d;
  p.viewdirs = v;
  p.zvals = z;
  p.n_per_ray = N;
  p.out_mode = OUT_RGBS;
  p.out_rgbs = out;
  return p;
}

// forward of both levels; fills comp/disp/acc (and rgbs, weights, z) of the workspace levels
int forward_levels(const char* where, const pob_render_config& c, Workspace& w, const void* pk_c,
                   const void* pk_f, const float* o, const float* d, const float* v, int R,
                   const float* z_base, const float* t_rand, const float* u, int u_per_ray,
                   const float* z_fine, int precision, bool save, cudaStream_t st,
                   const float* sp_points = nullptr, long long sp_n = 0) {
  const int sms = pob_sm_count_cached();
  const int Nc = c.num_coarse_samples, Nf = c.num_fine_samples;
  Level& C = w.lv[0];
  { pob_count_launch(1); PobPhaseTimer _t(POB_PH_RENDER, st); POB_CUDA(where, launch_sample_coarse(z_base, t_rand, R, Nc, C.z, st)); }
  {
    FwdParams p = ray_fwd_params(pk_c, c.sh_deg, o, d, v, C.z, R, Nc, C.rgbs);
    p.sigma_noise = c.sigma_noise_coarse_dev;
    if (Nf == 0 && sp_n > 0) {     // single-level model: the sparsity points ride on this launch
      p.M += sp_n;
      p.extra_points = sp_points;
    }
    if (save) {
      p.save_h = C.H;
      p.save_e = C.E;
      p.save_mask = C.mask;
    }
    { pob_count_launch(1); PobPhaseTimer _t(POB_PH_FWD, st); POB_CUDA(where, launch_mlp_fwd(p, precision, sms, st)); }
  }
  { pob_count_launch(1); PobPhaseTimer _t(POB_PH_RENDER, st); POB_CUDA(where, launch_composite_fwd(C.rgbs, C.z, d, R, Nc, c.white_bkgd, C.comp, C.disp, C.acc, C.weights, st)); }
  if (Nf > 0) {
    Level& F = w.lv[1];
    if (z_fine)
      POB_CUDA(where, cudaMemcpyAsync(F.z, z_fine, sizeof(float) * size_t(R) * (Nc + Nf),
                                      cudaMemcpyDeviceToDevice, st));
    else
      { pob_count_launch(1); PobPhaseTimer _t(POB_PH_RENDER, st); POB_CUDA(where, launch_sample_pdf(C.z, C.weights, u, u_per_ray, R, Nc, Nf, F.z, st)); }
    FwdParams p = ray_fwd_params(pk_f, c.sh_deg, o, d, v, F.z, R, Nc + Nf, F.rgbs);
    p.sigma_noise = c.sigma_noise_fine_dev;
    if (sp_n > 0) {                // the sparsity points ride behind the fine level's ray samples (same MLP)
      p.M += sp_n;
      p.extra_points = sp_points;
    }
    if (save) {
      p.save_h = F.H;
      p.save_e = F.E;
      p.save_mask = F.mask;
    }
    { pob_count_launch(1); PobPhaseTimer _t(POB_PH_FWD, st); POB_CUDA(where, launch_mlp_fwd(p, precision, sms, st)); }
    { pob_count_launch(1); PobPhaseTimer _t(POB_PH_RENDER, st); POB_CUDA(where, launch_composite_fwd(F.rgbs, F.z, d, R, Nc + Nf, c.white_bkgd, F.comp, F.disp, F.acc,
                                         F.weights, st)); }
  }
  return 0;
}

__global__ void pack_outputs_kernel(const float* comp, const float* disp, const float* acc, int R, float* out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  out[5 * r + 0] = comp[3 * r + 0];
  out[5 * r + 1] = comp[3 * r + 1];
  out[5 * r + 2] = comp[3 * r + 2];
  out[5 * r + 3] = disp[r];
  out[5 * r + 4] = acc[r];
}

}  // namespace

extern "C" {

int64_t pob_workspace_bytes(const pob_render_config* cfg, int training) {
  if (check_cfg("pob_workspace_bytes", cfg)) return -1;
  return (int64_t)carve(*cfg, training, nullptr).total;
}

int pob_render_rays(const pob_render_config* cfg, const void* packed_coarse_dev, const void* packed_fine_dev,
                    const float* origins_dev, const float* directions_dev, const float* viewdirs_dev,
                    int n_rays, const float* z_base_dev, const float* t_rand_dev, const float* u_dev,
                    int u_per_ray, const float* z_fine_dev, float* out_coarse_dev, float* out_fine_dev,
                    void* workspace_dev, int precision, void* stream) {
  const char* where = "pob_render_rays";
  if (int e = check_cfg(where, cfg)) return e;
  if (int e = pob_check_common(where, packed_coarse_dev, cfg->sh_deg, precision)) return e;
  if (n_rays < 0 || n_rays > cfg->max_rays) return pob_fail(where, "n_rays exceeds cfg->max_rays");
  if (n_rays == 0) return 0;
  if (!origins_dev || !directions_dev || !viewdirs_dev || !z_base_dev || !workspace_dev || !out_coarse_dev)
    return pob_fail(where, "NULL pointer");
  if (cfg->num_fine_samples > 0 && (!packed_fine_dev || (!u_dev && !z_fine_dev) || !out_fine_dev))
    return pob_fail(where, "fine level needs packed_fine, u (or z_fine) and out_fine");
  cudaStream_t st = (cudaStream_t)stream;
  Workspace w = carve(*cfg, 0, (uint8_t*)workspace_dev);
  if (int e = forward_levels(where, *cfg, w, packed_coarse_dev, packed_fine_dev, origins_dev, directions_dev,
                             viewdirs_dev, n_rays, z_base_dev, t_rand_dev, u_dev, u_per_ray, z_fine_dev,
                             precision, false, st))
    return e;
  const unsigned grid = (n_rays + 255) / 256;
  pob_count_launch(cfg->num_fine_samples > 0 ? 2 : 1);
  pack_outputs_kernel<<<grid, 256, 0, st>>>(w.lv[0].comp, w.lv[0].disp, w.lv[0].acc, n_rays, out_coarse_dev);
  if (cfg->num_fine_samples > 0)
    pack_outputs_kernel<<<grid, 256, 0, st>>>(w.lv[1].comp, w.lv[1].disp, w.lv[1].acc, n_rays, out_fine_dev);
  POB_CUDA(where, cudaGetLastError());
  return 0;
}

int pob_loss_and_grad(const pob_render_config* cfg, const pob_train_hparams* hp, const void* packed_coarse_dev,
                      const void* packed_fine_dev, const float* origins_dev, const float* directions_dev,
                      const float* viewdirs_dev, const float* pixels_dev, int n_rays, const float* z_base_dev,
                      const float* t_rand_dev, const float* u_dev, int u_per_ray, const float* z_fine_dev,
                      const float* sp_points_dev, float* grad_flat_dev, float* stats_dev, void* workspace_dev,
                      void* stream) {
  const char* where = "pob_loss_and_grad";
  if (int e = check_cfg(where, cfg)) return e;
  if (!hp) return pob_fail(where, "hparams is NULL");
  if (int e = pob_check_common(where, packed_coarse_dev, cfg->sh_deg, POB_PREC_FP16)) return e;
  if (n_rays <= 0 || n_rays > cfg->max_rays) return pob_fail(where, "n_rays out of range");
  if (!origins_dev || !directions_dev || !viewdirs_dev || !pixels_dev || !z_base_dev || !workspace_dev ||
      !grad_flat_dev || !stats_dev)
    return pob_fail(where, "NULL pointer");
  const int Nc = cfg->num_coarse_samples, Nf = cfg->num_fine_samples;
  if (Nf > 0 && (!packed_fine_dev || (!u_dev && !z_fine_dev)))
    return pob_fail(where, "fine level needs packed_fine and u (or z_fine)");
  const bool sparsity = hp->sparsity_weight > 0.f && cfg->sparsity_npoints > 0;
  if (sparsity && !sp_points_dev) return pob_fail(where, "sparsity term needs sp_points");
  if (!(hp->loss_scale > 0.f)) return pob_fail(where, "loss_scale must be positive");
  cudaStream_t st = (cudaStream_t)stream;
  const int sms = pob_sm_count_cached();
  const int K = cfg->sh_deg < 0 ? 1 : (cfg->sh_deg + 1) * (cfg->sh_deg + 1);
  const int P = flat_layout(K).total;
  Workspace w = carve(*cfg, 1, (uint8_t*)workspace_dev);
  POB_CUDA(where, cudaMemsetAsync(stats_dev, 0, 8 * sizeof(float), st));
  // The sparsity points (train.py:77-83: eval_points_raw of the fine MLP on uniform points) ride behind the ray
  // samples of the last level: same MLP, same launches, rows [n_rays * N, n_rays * N + sp_n) of its arrays.
  const long long sp_n = sparsity ? cfg->sparsity_npoints : 0;
  if (int e = forward_levels(where, *cfg, w, packed_coarse_dev, packed_fine_dev, origins_dev, directions_dev,
                             viewdirs_dev, n_rays, z_base_dev, t_rand_dev, u_dev, u_per_ray, z_fine_dev,
                             POB_PREC_FP16, true, st, sp_points_dev, sp_n))
    return e;
  const float gscale = hp->loss_scale * 2.0f / (3.0f * float(n_rays));
  Level& C = w.lv[0];
  Level& F = w.lv[1];
  Level& LAST = Nf > 0 ? F : C;
  const long long Mr_last = (long long)n_rays * (Nf > 0 ? Nc + Nf : Nc);
  // ---- upstream gradients ----
  { pob_count_launch(1); PobPhaseTimer _t(POB_PH_RENDER, st); POB_CUDA(where, launch_composite_bwd(C.rgbs, C.z, directions_dev, C.comp, pixels_dev, n_rays, Nc,
                                       cfg->white_bkgd, gscale, C.G, stats_dev + (Nf > 0 ? 1 : 0), st)); }
  if (Nf > 0)
    { pob_count_launch(1); PobPhaseTimer _t(POB_PH_RENDER, st); POB_CUDA(where, launch_composite_bwd(F.rgbs, F.z, directions_dev, F.comp, pixels_dev, n_rays, Nc + Nf,
                                         cfg->white_bkgd, gscale, F.G, stats_dev + 0, st)); }
  if (sparsity) {
    const float coef = hp->loss_scale * hp->sparsity_weight * hp->sparsity_length / float(sp_n);
    { pob_count_launch(1); PobPhaseTimer _t(POB_PH_RENDER, st); POB_CUDA(where, launch_sparsity_grad(LAST.rgbs + Mr_last, int(sp_n), hp->sparsity_length, coef,
                                                                                                    LAST.G + Mr_last, stats_dev + 2, st)); }
  }
  // ---- backward: per MLP one dgrad launch, then ONE wgrad launch over its saved dZ / h tiles ----
  // MLP_0 (coarse level only) first: its branch of the graph is independent of MLP_1's (stop_gradient,
  // model_utils.py:286), so grad_flat[0 : P) is final before the 3x larger MLP_1 backward starts.
  const int NH = heads_width(K);
  for (int mlp = 0; mlp < (Nf > 0 ? 2 : 1); ++mlp) {
    Level& L = mlp == 0 ? C : F;
    const long long Mr = (long long)n_rays * (mlp == 0 ? Nc : Nc + Nf);
    const long long Mm = Mr + (&L == &LAST ? sp_n : 0);
    const void* pk = mlp == 0 ? packed_coarse_dev : packed_fine_dev;
    BwdParams b;
    memset(&b, 0, sizeof(b));
    b.M = Mm;
    b.M_rays = Mr;
    b.G = L.G;
    b.viewdirs = viewdirs_dev;
    b.n_per_ray = mlp == 0 ? Nc : Nc + Nf;
    FwdParams base = pob_base_params(pk, cfg->sh_deg);
    b.w = base.w;
    b.sh_deg = cfg->sh_deg;
    b.K = base.K;
    b.NH = base.NH;
    b.mask = L.mask;
    b.save_dz = L.DZ;
    b.save_do = L.DO;
    { pob_count_launch(); PobPhaseTimer _t(POB_PH_BWD, st); POB_CUDA(where, launch_mlp_bwd(b, sms, st)); }
    WgradParams g;
    memset(&g, 0, sizeof(g));
    g.seg = WgradSegment{L.H, L.DZ, L.E, L.DO};
    g.seg_tiles = tiles_for(Mm);
    g.NH = NH;
    g.partials = w.partials[mlp];
    int rs[WG_NUM_ROLES], rc[WG_NUM_ROLES];
    const int nctas = wgrad_assign_roles(g, sms, rs, rc);
    { pob_count_launch(); PobPhaseTimer _t(POB_PH_WGRAD, st); POB_CUDA(where, launch_mlp_wgrad(g, nctas, st)); }
    { pob_count_launch(); PobPhaseTimer _t(POB_PH_OPTIM, st); POB_CUDA(where, launch_reduce_grads(w.partials[mlp], rs, rc, K, 1.0f / hp->loss_scale,
                                        grad_flat_dev + size_t(mlp) * P, st)); }
  }
  return 0;
}

int pob_adam_update(int sh_deg, int num_mlps, float* params_dev, const float* grads_dev, float* m_dev,
                    float* v_dev, float lr, float step, const float* lr_step_dev, float grad_mult,
                    float weight_decay_coef, void* packed_coarse_dev, void* packed_fine_dev, void* stream) {
  const char* where = "pob_adam_update";
  if (sh_deg < -1 || sh_deg > 4) return pob_fail(where, "sh_deg must be in [-1, 4]");
  if (num_mlps < 1 || num_mlps > 2) return pob_fail(where, "num_mlps must be 1 or 2");
  if (!params_dev || !grads_dev || !m_dev || !v_dev || !packed_coarse_dev || (num_mlps == 2 && !packed_fine_dev))
    return pob_fail(where, "NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int K = sh_deg < 0 ? 1 : (sh_deg + 1) * (sh_deg + 1);
  const long long P = flat_layout(K).total;
  { pob_count_launch(1); PobPhaseTimer _t(POB_PH_OPTIM, st); POB_CUDA(where, launch_adam(params_dev, grads_dev, m_dev, v_dev, P * num_mlps, lr, step, lr_step_dev, 0.9f, 0.999f, 1e-8f,
                              grad_mult, weight_decay_coef, st)); }
  if (int e = pob_pack_weights(params_dev, sh_deg, packed_coarse_dev, stream)) return e;
  if (num_mlps == 2)
    if (int e = pob_pack_weights(params_dev + P, sh_deg, packed_fine_dev, stream)) return e;
  return 0;
}

}  // extern "C"
