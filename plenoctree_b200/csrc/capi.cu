// capi.cu — extern "C" entry points declared in include/plenoctree_b200.h.
#include <cstdio>
#include <cstring>
#include <string>

#include "../../include/plenoctree_b200.h"
#include "capi_util.h"
#include "common.cuh"
#include "kernels.h"

static thread_local std::string g_err = "";

int pob_fail(const char* where, const char* what) {
  g_err = std::string(where) + ": " + what;
  return 1;
}
int pob_cuda_fail(const char* where, cudaError_t e) { return pob_fail(where, cudaGetErrorString(e)); }

// ---- instrumentation ---------------------------------------------------------------------------
#include <atomic>
#include <vector>
static std::atomic<long long> g_launches{0};
void pob_count_launch(int n) { g_launches += n; }
static bool g_timing = false;
struct TimedSlot {
  int phase;
  cudaEvent_t a, b;
};
static std::vector<TimedSlot> g_slots;
static double g_phase_ms[POB_PH_COUNT] = {0, 0, 0, 0, 0};
static long long g_phase_n[POB_PH_COUNT] = {0, 0, 0, 0, 0};
PobPhaseTimer::PobPhaseTimer(int phase, cudaStream_t s) : slot(-1), st(s) {
  if (!g_timing) return;
  TimedSlot t;
  t.phase = phase;
  cudaEventCreate(&t.a);
  cudaEventCreate(&t.b);
  cudaEventRecord(t.a, st);
  g_slots.push_back(t);
  slot = int(g_slots.size()) - 1;
}
PobPhaseTimer::~PobPhaseTimer() {
  if (slot >= 0) cudaEventRecord(g_slots[slot].b, st);
}
static void drain_slots() {
  for (auto& t : g_slots) {
    cudaEventSynchronize(t.b);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) {
      g_phase_ms[t.phase] += ms;
      g_phase_n[t.phase] += 1;
    }
    cudaEventDestroy(t.a);
    cudaEventDestroy(t.b);
  }
  g_slots.clear();
}

namespace {

int fail(const char* where, const char* what) { return pob_fail(where, what); }
int cuda_fail(const char* where, cudaError_t e) { return pob_cuda_fail(where, e); }

int K_of(int sh_deg) { return sh_deg < 0 ? 1 : (sh_deg + 1) * (sh_deg + 1); }

bool valid_deg(int sh_deg) { return sh_deg >= -1 && sh_deg <= 4; }

int g_sm_count = -1;
int sm_count() {
  if (g_sm_count > 0) return g_sm_count;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return -2;  // sm_100a only
  g_sm_count = n;
  return n;
}

// packed blob layout of one MLP
struct BlobLayout {
  size_t w_hi, w_lo, wt_hi, bias, total;
};
BlobLayout blob_layout(int K) {
  const int NH = pob::heads_width(K);
  auto up = [](size_t x) { return (x + 1023) / 1024 * 1024; };
  BlobLayout b;
  b.w_hi = 0;
  b.w_lo = up(b.w_hi + pob::fwd_image_bytes(NH));
  b.wt_hi = up(b.w_lo + pob::fwd_image_bytes(NH));
  b.bias = up(b.wt_hi + pob::bwd_image_bytes(NH));
  b.total = up(b.bias + (8 * 256 + pob::MAX_NH) * sizeof(float));
  return b;
}
pob::MlpPacked packed_view(const void* blob, int K) {
  const BlobLayout b = blob_layout(K);
  const uint8_t* p = static_cast<const uint8_t*>(blob);
  pob::MlpPacked w;
  w.w_hi = p + b.w_hi;
  w.w_lo = p + b.w_lo;
  w.wt_hi = p + b.wt_hi;
  w.bias = reinterpret_cast<const float*>(p + b.bias);
  return w;
}

int check_common(const char* where, const void* packed, int sh_deg, int precision) {
  if (!valid_deg(sh_deg)) return fail(where, "sh_deg must be in [-1, 4]");
  if (!packed) return fail(where, "packed weights pointer is NULL");
  if (precision != POB_PREC_FP16 && precision != POB_PREC_FP16X3)
    return fail(where, "precision must be POB_PREC_FP16 or POB_PREC_FP16X3");
  int n = sm_count();
  if (n == -2) return fail(where, "device is not compute capability 10.x (sm_100a build)");
  if (n <= 0) return fail(where, "no CUDA device");
  return 0;
}

pob::FwdParams base_params(const void* packed, int sh_deg) {
  pob::FwdParams p;
  memset(&p, 0, sizeof(p));
  p.sh_deg = sh_deg;
  p.K = K_of(sh_deg);
  p.NH = pob::heads_width(p.K);
  p.w = packed_view(packed, p.K);
  return p;
}

}  // namespace

int pob_sm_count_cached() { return sm_count(); }
int pob_check_common(const char* where, const void* packed, int sh_deg, int precision) {
  return check_common(where, packed, sh_deg, precision);
}
pob::FwdParams pob_base_params(const void* packed, int sh_deg) { return base_params(packed, sh_deg); }

extern "C" {

// 5: pob_loss_and_grad without its MLP_0 event, pob_debug_trace_fwd / _bwd without debug flags;
// 4: pob_loss_and_grad(MLP_0 event), pob_adam_update(lr_step_dev); 3: CTA-pair kernels
int pob_abi_version(void) { return 5; }

long long pob_launch_count(void) { return g_launches.load(); }

void pob_timing_enable(int on) {
  drain_slots();
  g_timing = on != 0;
  for (int i = 0; i < POB_PH_COUNT; ++i) {
    g_phase_ms[i] = 0;
    g_phase_n[i] = 0;
  }
}

int pob_timing_read(double* ms_out, long long* launches_out) {
  drain_slots();
  for (int i = 0; i < POB_PH_COUNT; ++i) {
    if (ms_out) ms_out[i] = g_phase_ms[i];
    if (launches_out) launches_out[i] = g_phase_n[i];
  }
  return POB_PH_COUNT;
}
const char* pob_last_error(void) { return g_err.c_str(); }
int pob_sm_count(void) { return sm_count(); }

int64_t pob_param_count(int sh_deg) {
  if (!valid_deg(sh_deg)) return -1;
  return pob::flat_layout(K_of(sh_deg)).total;
}
int64_t pob_packed_bytes(int sh_deg) {
  if (!valid_deg(sh_deg)) return -1;
  return (int64_t)blob_layout(K_of(sh_deg)).total;
}

int pob_pack_weights(const float* flat_dev, int sh_deg, void* packed_dev, void* stream) {
  if (!valid_deg(sh_deg)) return fail("pob_pack_weights", "sh_deg must be in [-1, 4]");
  if (!flat_dev || !packed_dev) return fail("pob_pack_weights", "NULL pointer");
  const int K = K_of(sh_deg);
  const BlobLayout b = blob_layout(K);
  uint8_t* p = static_cast<uint8_t*>(packed_dev);
  pob_count_launch();
  PobPhaseTimer _t(POB_PH_OPTIM, (cudaStream_t)stream);
  POB_CUDA("pob_pack_weights",
           pob::launch_pack_weights(flat_dev, K, p + b.w_hi, p + b.w_lo, p + b.wt_hi,
                                    reinterpret_cast<float*>(p + b.bias), (cudaStream_t)stream));
  return 0;
}

int pob_eval_points_raw(const void* packed_dev, int sh_deg, const float* points_dev, int64_t m,
                        float* raw_rgb_dev, float* raw_sigma_dev, int precision, void* stream) {
  if (int e = check_common("pob_eval_points_raw", packed_dev, sh_deg, precision)) return e;
  if (m < 0) return fail("pob_eval_points_raw", "negative point count");
  if (m == 0) return 0;
  if (!points_dev || !raw_sigma_dev) return fail("pob_eval_points_raw", "NULL pointer");
  pob::FwdParams p = base_params(packed_dev, sh_deg);
  p.src_mode = pob::SRC_POINTS;
  p.M = m;
  p.points = points_dev;
  p.out_mode = raw_rgb_dev ? pob::OUT_RAW : pob::OUT_SIGMA;
  p.out_rgb = raw_rgb_dev;
  p.out_sigma = raw_sigma_dev;
  pob_count_launch();
  PobPhaseTimer _t(POB_PH_FWD, (cudaStream_t)stream);
  POB_CUDA("pob_eval_points_raw",
           pob::launch_mlp_fwd(p, precision, sm_count(), (cudaStream_t)stream));
  return 0;
}

int pob_debug_trace_fwd(const void* packed_dev, int sh_deg, const float* points_dev, int64_t m,
                        float* raw_sigma_dev, unsigned long long* trace_dev, void* save_h_dev,
                        void* save_e_dev, void* save_mask_dev, void* stream) {
  if (int e = check_common("pob_debug_trace_fwd", packed_dev, sh_deg, POB_PREC_FP16)) return e;
  if (!points_dev || !raw_sigma_dev || !trace_dev || m <= 0) return fail("pob_debug_trace_fwd", "bad arguments");
  pob::FwdParams p = base_params(packed_dev, sh_deg);
  p.src_mode = pob::SRC_POINTS;
  p.M = m;
  p.points = points_dev;
  p.out_mode = pob::OUT_SIGMA;
  p.out_sigma = raw_sigma_dev;
  p.trace = trace_dev;
  p.save_h = static_cast<uint8_t*>(save_h_dev);
  p.save_e = static_cast<uint8_t*>(save_e_dev);
  p.save_mask = static_cast<uint32_t*>(save_mask_dev);
  POB_CUDA("pob_debug_trace_fwd", pob::launch_mlp_fwd(p, 1, sm_count(), (cudaStream_t)stream));
  return 0;
}

int pob_debug_trace_bwd(const void* packed_dev, int sh_deg, int64_t m, const float* g_dev, const float* viewdirs_dev,
                        const void* mask_dev, void* save_dz_dev, void* save_do_dev, unsigned long long* trace_dev,
                        void* stream) {
  if (int e = check_common("pob_debug_trace_bwd", packed_dev, sh_deg, POB_PREC_FP16)) return e;
  if (!g_dev || !viewdirs_dev || !mask_dev || !save_dz_dev || !save_do_dev || m <= 0)
    return fail("pob_debug_trace_bwd", "bad arguments");
  pob::FwdParams base = base_params(packed_dev, sh_deg);
  pob::BwdParams b;
  memset(&b, 0, sizeof(b));
  b.M = m;
  b.G = reinterpret_cast<const float4*>(g_dev);
  b.viewdirs = viewdirs_dev;
  b.n_per_ray = 0;
  b.M_rays = m;
  b.w = base.w;
  b.sh_deg = sh_deg;
  b.K = base.K;
  b.NH = base.NH;
  b.mask = static_cast<const uint32_t*>(mask_dev);
  b.save_dz = static_cast<uint8_t*>(save_dz_dev);
  b.save_do = static_cast<uint8_t*>(save_do_dev);
  b.trace = trace_dev;
  POB_CUDA("pob_debug_trace_bwd", pob::launch_mlp_bwd(b, sm_count(), (cudaStream_t)stream));
  return 0;
}

int pob_eval_points(const void* packed_dev, int sh_deg, const float* points_dev,
                    const float* viewdirs_dev, int64_t m, float* out_rgbs_dev, int precision,
                    void* stream) {
  if (int e = check_common("pob_eval_points", packed_dev, sh_deg, precision)) return e;
  if (m < 0) return fail("pob_eval_points", "negative point count");
  if (m == 0) return 0;
  if (!points_dev || !out_rgbs_dev) return fail("pob_eval_points", "NULL pointer");
  if (sh_deg >= 0 && !viewdirs_dev)
    return fail("pob_eval_points", "viewdirs required when sh_deg >= 0 (models.py:199)");
  pob::FwdParams p = base_params(packed_dev, sh_deg);
  p.src_mode = pob::SRC_POINTS;
  p.M = m;
  p.points = points_dev;
  p.viewdirs = viewdirs_dev ? viewdirs_dev : points_dev;
  p.out_mode = pob::OUT_RGBS;
  p.out_rgbs = reinterpret_cast<float4*>(out_rgbs_dev);
  pob_count_launch();
  PobPhaseTimer _t(POB_PH_FWD, (cudaStream_t)stream);
  POB_CUDA("pob_eval_points",
           pob::launch_mlp_fwd(p, precision, sm_count(), (cudaStream_t)stream));
  return 0;
}

int pob_eval_cells_mean(const void* packed_dev, int sh_deg, const float* points_dev, int64_t n_cells,
                        int samples_per_cell, float* out_dev, int precision, void* stream) {
  if (int e = check_common("pob_eval_cells_mean", packed_dev, sh_deg, precision)) return e;
  if (n_cells < 0 || samples_per_cell <= 0) return fail("pob_eval_cells_mean", "bad sizes");
  if (n_cells == 0) return 0;
  if (!points_dev || !out_dev) return fail("pob_eval_cells_mean", "NULL pointer");
  pob::FwdParams p = base_params(packed_dev, sh_deg);
  p.src_mode = pob::SRC_POINTS;
  p.M = n_cells * (int64_t)samples_per_cell;
  p.points = points_dev;
  p.out_mode = pob::OUT_CELL_MEAN;
  p.out_cell = out_dev;
  p.cell_S = samples_per_cell;
  POB_CUDA("pob_eval_cells_mean",
           cudaMemsetAsync(out_dev, 0, sizeof(float) * n_cells * (3 * p.K + 1), (cudaStream_t)stream));
  pob_count_launch();
  PobPhaseTimer _t(POB_PH_FWD, (cudaStream_t)stream);
  POB_CUDA("pob_eval_cells_mean",
           pob::launch_mlp_fwd(p, precision, sm_count(), (cudaStream_t)stream));
  return 0;
}

int pob_eval_grid(const void* packed_dev, int sh_deg, int reso, int x0, int nx, int ny, int nz,
                  const float offset[3], const float scale[3], float* raw_rgb_dev,
                  float* raw_sigma_dev, int precision, void* stream) {
  if (int e = check_common("pob_eval_grid", packed_dev, sh_deg, precision)) return e;
  if (reso <= 0 || (reso & (reso - 1)))
    return fail("pob_eval_grid", "reso must be a power of two (extraction.py:246,290)");
  if (x0 < 0 || nx < 0 || ny < 0 || nz < 0 || x0 + nx > reso || ny > reso || nz > reso)
    return fail("pob_eval_grid", "slab out of range");
  if (!offset || !scale || !raw_sigma_dev) return fail("pob_eval_grid", "NULL pointer");
  const long long m = (long long)nx * ny * nz;
  if (m == 0) return 0;
  pob::FwdParams p = base_params(packed_dev, sh_deg);
  p.src_mode = pob::SRC_GRID;
  p.M = m;
  p.g_reso = reso;
  p.g_x0 = x0;
  p.g_nx = nx;
  p.g_ny = ny;
  p.g_nz = nz;
  for (int a = 0; a < 3; ++a) {
    p.g_offset[a] = offset[a];
    p.g_scale[a] = scale[a];
  }
  p.out_mode = raw_rgb_dev ? pob::OUT_RAW : pob::OUT_SIGMA;
  p.out_rgb = raw_rgb_dev;
  p.out_sigma = raw_sigma_dev;
  pob_count_launch();
  PobPhaseTimer _t(POB_PH_FWD, (cudaStream_t)stream);
  POB_CUDA("pob_eval_grid",
           pob::launch_mlp_fwd(p, precision, sm_count(), (cudaStream_t)stream));
  return 0;
}

int pob_eval_points_raw_host(const void* packed_dev, int sh_deg, const float* points_host,
                             int64_t m, float* raw_rgb_host, float* raw_sigma_host,
                             int precision) {
  if (int e = check_common("pob_eval_points_raw_host", packed_dev, sh_deg, precision)) return e;
  if (m <= 0) return m == 0 ? 0 : fail("pob_eval_points_raw_host", "negative point count");
  if (!points_host || !raw_sigma_host) return fail("pob_eval_points_raw_host", "NULL pointer");
  const int K = K_of(sh_deg);
  float *d_pts = nullptr, *d_rgb = nullptr, *d_sig = nullptr;
  cudaStream_t st = 0;
  int rc = 0;
  do {
    if (cudaMalloc(&d_pts, sizeof(float) * 3 * m) != cudaSuccess ||
        cudaMalloc(&d_sig, sizeof(float) * m) != cudaSuccess ||
        (raw_rgb_host && cudaMalloc(&d_rgb, sizeof(float) * 3 * K * m) != cudaSuccess)) {
      rc = fail("pob_eval_points_raw_host", "cudaMalloc failed");
      break;
    }
    if (cudaMemcpyAsync(d_pts, points_host, sizeof(float) * 3 * m, cudaMemcpyHostToDevice, st) !=
        cudaSuccess) {
      rc = fail("pob_eval_points_raw_host", "H2D copy failed");
      break;
    }
    rc = pob_eval_points_raw(packed_dev, sh_deg, d_pts, m, d_rgb, d_sig, precision, st);
    if (rc) break;
    if (raw_rgb_host)
      cudaMemcpyAsync(raw_rgb_host, d_rgb, sizeof(float) * 3 * K * m, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(raw_sigma_host, d_sig, sizeof(float) * m, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = cuda_fail("pob_eval_points_raw_host", e);
  } while (0);
  cudaFree(d_pts);
  cudaFree(d_rgb);
  cudaFree(d_sig);
  return rc;
}

int pob_sample_coarse(const float* z_base_dev, const float* t_rand_dev, int n_rays, int n_samples,
                      float* z_out_dev, void* stream) {
  if (!z_base_dev || !z_out_dev) return fail("pob_sample_coarse", "NULL pointer");
  if (n_rays < 0 || n_samples < 1) return fail("pob_sample_coarse", "bad sizes");
  pob_count_launch();
  POB_CUDA("pob_sample_coarse",
           pob::launch_sample_coarse(z_base_dev, t_rand_dev, n_rays, n_samples, z_out_dev, (cudaStream_t)stream));
  return 0;
}

int pob_draw_uniforms(uint64_t seed, float step, const float* step_dev, float* t_rand_dev, int64_t n_t,
                      float* u_dev, int64_t n_u, float* sp_points_dev, int64_t n_sp, float sp_radius, void* stream) {
  if (n_t < 0 || n_u < 0 || n_sp < 0) return fail("pob_draw_uniforms", "negative size");
  if ((n_t && !t_rand_dev) || (n_u && !u_dev) || (n_sp && !sp_points_dev))
    return fail("pob_draw_uniforms", "NULL pointer");
  if (sm_count() <= 0) return fail("pob_draw_uniforms", "no sm_100 CUDA device (there is no CPU fallback)");
  pob_count_launch();
  POB_CUDA("pob_draw_uniforms", pob::launch_draw_uniforms(seed, step, step_dev, t_rand_dev, n_t, u_dev, n_u,
                                                          sp_points_dev, n_sp, sp_radius, (cudaStream_t)stream));
  return 0;
}

int pob_composite(const float* rgbs_dev, const float* z_dev, const float* dirs_dev, int n_rays, int n_samples,
                  int white_bkgd, float* out_rgb_dev, float* out_disp_dev, float* out_acc_dev,
                  float* out_weights_dev, void* stream) {
  if (!rgbs_dev || !z_dev || !dirs_dev || !out_rgb_dev) return fail("pob_composite", "NULL pointer");
  if (n_rays < 0 || n_samples < 1 || n_samples > 256) return fail("pob_composite", "n_samples must be in [1,256]");
  pob_count_launch();
  POB_CUDA("pob_composite",
           pob::launch_composite_fwd(reinterpret_cast<const float4*>(rgbs_dev), z_dev, dirs_dev, n_rays, n_samples,
                                     white_bkgd, out_rgb_dev, out_disp_dev, out_acc_dev, out_weights_dev,
                                     (cudaStream_t)stream));
  return 0;
}

int pob_composite_bwd(const float* rgbs_dev, const float* z_dev, const float* dirs_dev, const float* comp_rgb_dev,
                      const float* pixels_dev, int n_rays, int n_samples, int white_bkgd, float gscale,
                      float* g_out_dev, float* sq_err_sum_dev, void* stream) {
  if (!rgbs_dev || !z_dev || !dirs_dev || !comp_rgb_dev || !pixels_dev || !g_out_dev)
    return fail("pob_composite_bwd", "NULL pointer");
  if (n_rays < 0 || n_samples < 1 || n_samples > 256) return fail("pob_composite_bwd", "n_samples must be in [1,256]");
  pob_count_launch();
  POB_CUDA("pob_composite_bwd",
           pob::launch_composite_bwd(reinterpret_cast<const float4*>(rgbs_dev), z_dev, dirs_dev, comp_rgb_dev,
                                     pixels_dev, n_rays, n_samples, white_bkgd, gscale,
                                     reinterpret_cast<float4*>(g_out_dev), sq_err_sum_dev, (cudaStream_t)stream));
  return 0;
}

int pob_sample_pdf(const float* z_coarse_dev, const float* weights_dev, const float* u_dev, int u_per_ray,
                   int n_rays, int n_coarse, int n_fine, float* z_out_dev, void* stream) {
  if (!z_coarse_dev || !weights_dev || !u_dev || !z_out_dev) return fail("pob_sample_pdf", "NULL pointer");
  if (n_coarse < 3 || n_fine < 1 || n_coarse + n_fine > 256)
    return fail("pob_sample_pdf", "need n_coarse >= 3 and n_coarse + n_fine <= 256");
  pob_count_launch();
  POB_CUDA("pob_sample_pdf", pob::launch_sample_pdf(z_coarse_dev, weights_dev, u_dev, u_per_ray, n_rays, n_coarse,
                                                    n_fine, z_out_dev, (cudaStream_t)stream));
  return 0;
}

int pob_umma_probe(const void* a_img_dev, uint32_t a_bytes, const void* b_img_dev,
                   uint32_t b_bytes, uint32_t b_off, const uint64_t* adesc_dev,
                   const uint64_t* bdesc_dev, const uint32_t* dcol_dev, const uint32_t* accum_dev,
                   int nops, uint32_t idesc, int out_cols, float* out_dev, void* stream) {
  if (sm_count() <= 0) return fail("pob_umma_probe", "no sm_100 CUDA device");
  if (a_bytes % 16 || b_bytes % 16 || b_off % 1024 || b_off < a_bytes ||
      (size_t)b_off + b_bytes > 200 * 1024)
    return fail("pob_umma_probe", "bad image sizes/offsets");
  if (out_cols <= 0 || out_cols > 512) return fail("pob_umma_probe", "out_cols out of range");
  POB_CUDA("pob_umma_probe",
           pob::launch_umma_probe(a_img_dev, a_bytes, b_img_dev, b_bytes, b_off, adesc_dev,
                                  bdesc_dev, dcol_dev, accum_dev, nops, idesc, out_cols, out_dev,
                                  (cudaStream_t)stream));
  return 0;
}

int pob_umma_probe_pair(const void* a_img_dev, uint32_t a_bytes, const void* b_img_dev,
                        uint32_t b_bytes, uint32_t b_off, const uint64_t* adesc_dev,
                        const uint64_t* bdesc_dev, const uint32_t* dcol_dev, const uint32_t* accum_dev,
                        int nops, uint32_t idesc, int out_cols, float* out_dev, void* stream) {
  if (sm_count() <= 0) return fail("pob_umma_probe_pair", "no sm_100 CUDA device");
  if (a_bytes % 16 || b_bytes % 16 || b_off % 1024 || b_off < a_bytes ||
      (size_t)b_off + b_bytes > 200 * 1024)
    return fail("pob_umma_probe_pair", "bad image sizes/offsets");
  if (out_cols <= 0 || out_cols > 512) return fail("pob_umma_probe_pair", "out_cols out of range");
  POB_CUDA("pob_umma_probe_pair",
           pob::launch_umma_probe_pair(a_img_dev, a_bytes, b_img_dev, b_bytes, b_off, adesc_dev,
                                       bdesc_dev, dcol_dev, accum_dev, nops, idesc, out_cols, out_dev,
                                       (cudaStream_t)stream));
  return 0;
}

}  // extern "C"
