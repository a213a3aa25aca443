// octree.cu — PlenOctree kernels: volume renderer forward / backward (SURVEY §8 row a15), fused
// render + MSE-gradient + scatter training pass, SGD, point query, dense-grid weight render
// (octree.extraction masking_mode "weight").
//
// These replace the third-party svox extension the reference calls (octree/optimization.py:174-229,
// octree/extraction.py:181-214, octree/nerf/utils.py:448-498).  The arithmetic follows svox's published
// per-ray march (oracle/octree_oracle.py restates it).  Everything that decides WHERE a ray samples (ray set-up,
// positions, cell exits, step lengths) is written with __fmul_rn / __fadd_rn so that it rounds exactly like the
// float32 oracle and a ray never lands in a different leaf than the oracle's; the shading arithmetic (SH dot
// products, exp, sigmoid, compositing sums) may contract to FMA and uses the fast exp / reciprocal — the march is
// instruction-issue bound (ncu: sm__throughput 73-79 %, DRAM 5 %), so instruction count is what matters.
//
// Thread mapping (B200-first, not svox's thread-per-ray): a *group* of G = 4 lanes owns one ray (see G below).
// All lanes of a group walk the tree together (same-address loads broadcast), lane l owns basis functions l, l+G,
// ...: the 3K coefficient gather of a contributing leaf is three coalesced segments per group instead of 3K
// strided scalar loads per thread, the dot products finish with log2(G) shuffles, and the backward scatter issues
// coalesced RED.ADD.F32.  Pixels are tiled per CTA so that neighbouring rays share L1 lines.
#include <cstdint>

#include "../../include/plenoctree_b200.h"
#include "capi_util.h"
#include "common.cuh"

namespace pob {
namespace {

// Safety caps (never reached by a valid tree / positive step): a corrupt child array or a step that underflows
// against t must not hang the device.  A march visits one leaf per iteration (a few thousand for a depth-10 tree);
// the cap only has to exceed sqrt(3) / step_size for the smallest step the reference's configurations use
// (renderer_step_size 1e-5, octree/config/syn_sh16.json:16,22,24), since every iteration advances by >= step_size.
constexpr int MAX_MARCH_STEPS = 1 << 20;
constexpr int MAX_TREE_DEPTH = 40;

// Lanes per ray (group width G).  The march is instruction-issue bound and every lane of a group repeats the walk,
// so fewer lanes per ray = fewer instructions per ray.  Measured 800x800 / depth-8 SH16: 16 lanes 4.1 ms, 8 lanes
// 2.25 ms, 4 lanes 1.65 ms.  (2 lanes: 1.52 ms render but 4.7 ms training pass — not kept.)
constexpr int G = 4;
constexpr int RAYS_PER_CTA = 256 / G;
// perspective camera: each CTA renders an 8 x 8 pixel tile
constexpr int PIX_TILE_W = 8, PIX_TILE_H = RAYS_PER_CTA / PIX_TILE_W;

struct TreeDev {
  const float* data;
  const int32_t* child;
  int N, D, K, rgba;
  float off[3], inv[3];
};

struct Opts {
  float step, bg, sigma_thresh, stop_thresh;
};

struct Cam {
  float c2w[12];
  float fx, fy, width, height;
};

struct RaySrc {
  const float* o;   // explicit rays (world): origins / dirs / vdirs [n,3]; null -> perspective camera
  const float* d;
  const float* v;
  Cam cam;
  int row0;         // first pixel row of the slab this launch renders
  int nrows;
  long long n;      // number of rays (explicit) / pixels in the slab
};

struct Ray {
  float o[3], d[3], invd[3], vdir[3];
  float delta_scale, tmin, tmax;
  bool hit;
};

__device__ __forceinline__ void dda_unit(const float* cen, const float* invd, float& tmin, float& tmax) {
  tmin = 0.0f;
  tmax = 1e9f;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float t1 = __fmul_rn(-cen[i], invd[i]);
    const float t2 = __fadd_rn(t1, invd[i]);
    tmin = fmaxf(tmin, fminf(t1, t2));
    tmax = fminf(tmax, fmaxf(t1, t2));
  }
}

// persp pixel -> world ray (svox render_image_kernel: no +0.5 pixel centre; README.md:184)
__device__ __forceinline__ void cam_ray(const Cam& c, int ix, int iy, float* o, float* d) {
  float x = __fsub_rn(float(ix), __fmul_rn(0.5f, c.width)) / c.fx;
  float y = -__fsub_rn(float(iy), __fmul_rn(0.5f, c.height)) / c.fy;
  float z = -1.0f;
  const float nrm = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)));
  x = x / nrm;
  y = y / nrm;
  z = z / nrm;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    d[a] = __fadd_rn(__fadd_rn(__fmul_rn(c.c2w[4 * a + 0], x), __fmul_rn(c.c2w[4 * a + 1], y)),
                     __fmul_rn(c.c2w[4 * a + 2], z));
    o[a] = c.c2w[4 * a + 3];
  }
}

// transform_coord + _get_delta_scale + unit-cube intersection (svox trace_ray prologue)
__device__ __forceinline__ void setup_ray(const float* off, const float* inv, const float* ow, const float* dw,
                                          const float* vw, Ray& r) {
  float nrm2 = 0.f;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    r.o[a] = __fadd_rn(off[a], __fmul_rn(inv[a], ow[a]));
    r.d[a] = __fmul_rn(dw[a], inv[a]);
    r.vdir[a] = vw[a];
  }
  nrm2 = __fadd_rn(__fadd_rn(__fmul_rn(r.d[0], r.d[0]), __fmul_rn(r.d[1], r.d[1])), __fmul_rn(r.d[2], r.d[2]));
  r.delta_scale = 1.0f / sqrtf(nrm2);
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    r.d[a] = __fmul_rn(r.d[a], r.delta_scale);
    r.invd[a] = 1.0f / __fadd_rn(r.d[a], 1e-9f);
  }
  dda_unit(r.o, r.invd, r.tmin, r.tmax);
  r.hit = !(r.tmax < 0.f || r.tmin > r.tmax);
}

// svox query_single_from_root: pos in [0,1]^3 -> flat leaf index; pos becomes the position inside the leaf
__device__ __forceinline__ long long query_leaf(const int32_t* __restrict__ child, int N, float* pos, float& cube) {
  const float fN = float(N);
#pragma unroll
  for (int a = 0; a < 3; ++a) pos[a] = fmaxf(0.0f, fminf(1.0f - 1e-6f, pos[a]));
  long long node = 0;
  cube = fN;
  long long idx = 0;
  for (int level = 0; level < MAX_TREE_DEPTH; ++level) {
    int u[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      pos[a] = __fmul_rn(pos[a], fN);
      const float fl = floorf(pos[a]);
      u[a] = int(fl);
      pos[a] = __fsub_rn(pos[a], fl);
    }
    idx = ((node * N + u[0]) * N + u[1]) * N + u[2];
    const int skip = __ldg(child + idx);
    if (skip == 0) return idx;
    cube = cube * fN;
    node += skip;
  }
  return idx;
}

__device__ __forceinline__ unsigned group_mask() {
  const unsigned lane = threadIdx.x & 31;
  return ((1u << G) - 1u) << (lane / G * G);
}

__device__ __forceinline__ float group_sum(float v, unsigned mask) {
#pragma unroll
  for (int s = G / 2; s > 0; s >>= 1) v += __shfl_xor_sync(mask, v, s, G);
  return v;
}

__device__ __forceinline__ float sigmoidf(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }

// ---- leaf lookup with a per-ray path cache --------------------------------------------------------------
// Consecutive samples of a ray fall into neighbouring leaves that share most of their ancestors, yet svox walks
// down from the root for every sample (depth x dependent L2 loads).  For N = 2 the cell digits of a point are the
// binary digits of its coordinates (x*2 and x - floor(x) are exact in fp32), so the walk can resume below the deepest
// ancestor shared with the previous sample: lane k of the group keeps the node entered at level k (the otherwise
// idle lanes are the stack), the shared depth is a count-leading-zeros of the XOR of the integer coordinates, and
// the position inside the leaf is frac(x * 2^(depth+1)) — bit-identical to the iterated form.  Other branch
// factors, and levels deeper than 22, use the plain walk.
struct Marcher {
  unsigned pq0, pq1, pq2;
  static constexpr int PW = 8 / G;   // path registers per lane: levels l, l+G, ... are cached
  static constexpr int CACHED = G * PW;
  int pdepth;     // depth of the previous leaf, -1 = no previous sample
  int path[PW];   // lane l, register j: node entered at level l + j*G (level 0: root)

  __device__ __forceinline__ void init() {
    pdepth = -1;
#pragma unroll
    for (int j = 0; j < PW; ++j) path[j] = 0;
    pq0 = pq1 = pq2 = 0;
  }

  // leaf holding origin + t * dir; returns its flat index and the march length to its exit (+ step)
  // (leaf indices fit 32 bits: n_nodes * N^3 < 2^32 is checked on the host)
  __device__ __forceinline__ unsigned locate(const TreeDev& T, const Ray& r, float step, float t, int l, unsigned mask,
                                             float& delta_t) {
    float pos[3], cube, inv_cube = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a) pos[a] = __fadd_rn(r.o[a], __fmul_rn(t, r.d[a]));
    unsigned idx;
    bool pow2 = false;
    if (T.N == 2) {
      pow2 = true;
#pragma unroll
      for (int a = 0; a < 3; ++a) pos[a] = fmaxf(0.0f, fminf(1.0f - 1e-6f, pos[a]));
      const unsigned q0 = __float2uint_rz(pos[0] * 8388608.0f);
      const unsigned q1 = __float2uint_rz(pos[1] * 8388608.0f);
      const unsigned q2 = __float2uint_rz(pos[2] * 8388608.0f);
      int s = 0, node = 0;
      if (pdepth >= 0) {
        const unsigned diff = (q0 ^ pq0) | (q1 ^ pq1) | (q2 ^ pq2);
        const int c = diff ? __clz(int(diff << 9)) : 23;
        s = min(min(c, pdepth), CACHED - 1);
        int sel = path[0];
#pragma unroll
        for (int j = 1; j < PW; ++j)
          if (s / G == j) sel = path[j];
        node = __shfl_sync(mask, sel, s % G, G);
      }
      pq0 = q0;
      pq1 = q1;
      pq2 = q2;
      int k = s;
      idx = 0;
      bool leaf = false;
      for (; k <= 22; ++k) {
        const int sh = 22 - k;
        idx = unsigned(node) * 8u + ((((q0 >> sh) & 1u) << 2) | (((q1 >> sh) & 1u) << 1) | ((q2 >> sh) & 1u));
        const int skip = __ldg(T.child + idx);
        if (skip == 0) {
          leaf = true;
          break;
        }
        node += skip;
        if (l == (k + 1) % G) {
#pragma unroll
          for (int j = 0; j < PW; ++j)
            if ((k + 1) / G == j) path[j] = node;
        }
      }
      if (leaf) {
        pdepth = k;
        cube = __int_as_float((127 + k + 1) << 23);       // 2^(k+1)
        inv_cube = __int_as_float((127 - k - 1) << 23);   // 2^-(k+1), exact
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          const float sc = pos[a] * cube;
          pos[a] = sc - floorf(sc);
        }
      } else {
        // deeper than the 23 cached digits: finish with the plain walk from `node`
        pdepth = 22;
        cube = 8388608.0f;
        pow2 = false;   // the exit length below falls back to the division
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          const float sc = pos[a] * cube;
          pos[a] = sc - floorf(sc);
        }
        for (int level = 23; level < MAX_TREE_DEPTH; ++level) {
          int u[3];
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            pos[a] = pos[a] * 2.0f;
            const float fl = floorf(pos[a]);
            u[a] = int(fl);
            pos[a] = pos[a] - fl;
          }
          cube = cube * 2.0f;
          idx = unsigned(node) * 8u + unsigned(u[0] * 4 + u[1] * 2 + u[2]);
          const int skip = __ldg(T.child + idx);
          if (skip == 0) break;
          node += skip;
        }
      }
    } else {
      idx = unsigned(query_leaf(T.child, T.N, pos, cube));
    }
    float smin, smax;
    dda_unit(pos, r.invd, smin, smax);
    // cube is a power of two for N = 2: multiplying by its (exact) reciprocal equals the IEEE division
    const float len = pow2 ? __fmul_rn(__fsub_rn(smax, smin), inv_cube) : __fsub_rn(smax, smin) / cube;
    delta_t = __fadd_rn(len, step);
    return idx;
  }
};

// ---- forward march of one ray by one lane group -------------------------------------------------------
// Software-pipelined: the loads of the current leaf (sigma and this lane's three coefficients, issued
// unconditionally) are in flight while the next leaf is located; the march itself never depends on the data.
template <int KPL>
__device__ __forceinline__ void trace_forward(const TreeDev& T, const Opts& O, const Ray& r, const float* basis_l, int l,
                                              unsigned mask, float* out, unsigned& visits, unsigned& hits) {
  if (!r.hit) {
    out[0] = out[1] = out[2] = O.bg;
    return;
  }
  out[0] = out[1] = out[2] = 0.f;
  float light = 1.0f;
  float t = r.tmin;
  const int K = T.K, D = T.D;
  if (!(t < r.tmax)) {
    out[0] = out[1] = out[2] = O.bg;  // light = 1
    return;
  }
  Marcher m;
  m.init();
  float delta_t;
  unsigned idx = m.locate(T, r, O.step, t, l, mask, delta_t);
  for (int it = 0; it < MAX_MARCH_STEPS; ++it) {
    const float* __restrict__ val = T.data + size_t(idx) * unsigned(D);
    const float sigma = __ldg(val + D - 1);
    float c0[KPL], c1[KPL], c2[KPL];  // lane l owns basis functions l, l+G, ...
#pragma unroll
    for (int j = 0; j < KPL; ++j) {
      const int k = l + j * G;
      c0[j] = c1[j] = c2[j] = 0.f;
      if (k < K) {
        c0[j] = __ldg(val + k);
        c1[j] = __ldg(val + K + k);
        c2[j] = __ldg(val + 2 * K + k);
      }
    }
    const float t_next = t + delta_t;
    const bool more = t_next < r.tmax;
    float delta_n = 0.f;
    unsigned idx_n = 0;
    if (more) idx_n = m.locate(T, r, O.step, t_next, l, mask, delta_n);
    ++visits;
    if (sigma > O.sigma_thresh) {
      ++hits;
      const float att = __expf(-delta_t * r.delta_scale * sigma);
      const float weight = light * (1.0f - att);
      float p0 = 0.f, p1 = 0.f, p2 = 0.f;
#pragma unroll
      for (int j = 0; j < KPL; ++j) {
        p0 += basis_l[j] * c0[j];
        p1 += basis_l[j] * c1[j];
        p2 += basis_l[j] * c2[j];
      }
      p0 = group_sum(p0, mask);
      p1 = group_sum(p1, mask);
      p2 = group_sum(p2, mask);
      out[0] += weight * sigmoidf(p0);
      out[1] += weight * sigmoidf(p1);
      out[2] += weight * sigmoidf(p2);
      light *= att;
      if (light <= O.stop_thresh) {
        const float scale = 1.0f / (1.0f - light);
        out[0] *= scale;
        out[1] *= scale;
        out[2] *= scale;
        return;
      }
    }
    if (!more) break;
    t = t_next;
    idx = idx_n;
    delta_t = delta_n;
  }
  out[0] += light * O.bg;
  out[1] += light * O.bg;
  out[2] += light * O.bg;
}

// ---- backward march: colour and density gradients in one pass ---------------------------------------
// accum enters as sum_j w_j (c_j . g) + T_end * bg * sum(g) = g . out (svox computes it with an extra march:
// trace_ray_backward pass 1); every contributing leaf then peels its own term off.
template <int KPL>
__device__ __forceinline__ void trace_backward(const TreeDev& T, const Opts& O, const Ray& r, const float* basis_l, int l,
                                               unsigned mask, const float* g, float accum,
                                               float* __restrict__ grad) {
  if (!r.hit) return;
  float light = 1.0f;
  float t = r.tmin;
  const int K = T.K, D = T.D;
  if (!(t < r.tmax)) return;
  Marcher m;
  m.init();
  float delta_t;
  unsigned idx = m.locate(T, r, O.step, t, l, mask, delta_t);
  for (int it = 0; it < MAX_MARCH_STEPS; ++it) {
    const float* __restrict__ val = T.data + size_t(idx) * unsigned(D);
    const float sigma = __ldg(val + D - 1);
    float c0[KPL], c1[KPL], c2[KPL];  // lane l owns basis functions l, l+G, ...
#pragma unroll
    for (int j = 0; j < KPL; ++j) {
      const int k = l + j * G;
      c0[j] = c1[j] = c2[j] = 0.f;
      if (k < K) {
        c0[j] = __ldg(val + k);
        c1[j] = __ldg(val + K + k);
        c2[j] = __ldg(val + 2 * K + k);
      }
    }
    const float t_next = t + delta_t;
    const bool more = t_next < r.tmax;
    float delta_n = 0.f;
    unsigned idx_n = 0;
    if (more) idx_n = m.locate(T, r, O.step, t_next, l, mask, delta_n);
    if (sigma > 0.0f) {
      const float att = __expf(-delta_t * r.delta_scale * sigma);
      const float weight = light * (1.0f - att);
      float p0 = 0.f, p1 = 0.f, p2 = 0.f;
#pragma unroll
      for (int j = 0; j < KPL; ++j) {
        p0 += basis_l[j] * c0[j];
        p1 += basis_l[j] * c1[j];
        p2 += basis_l[j] * c2[j];
      }
      p0 = group_sum(p0, mask);
      p1 = group_sum(p1, mask);
      p2 = group_sum(p2, mask);
      const float s0 = sigmoidf(p0), s1 = sigmoidf(p1), s2 = sigmoidf(p2);
      float* gv = grad + size_t(idx) * unsigned(D);
      const float t0 = weight * s0 * (1.0f - s0) * g[0];
      const float t1 = weight * s1 * (1.0f - s1) * g[1];
      const float t2 = weight * s2 * (1.0f - s2) * g[2];
#pragma unroll
      for (int j = 0; j < KPL; ++j) {
        const int k = l + j * G;
        if (k < K) {
          atomicAdd(gv + k, basis_l[j] * t0);
          atomicAdd(gv + K + k, basis_l[j] * t1);
          atomicAdd(gv + 2 * K + k, basis_l[j] * t2);
        }
      }
      const float total = s0 * g[0] + s1 * g[1] + s2 * g[2];
      light *= att;
      accum -= weight * total;
      if (l == 0) atomicAdd(gv + D - 1, delta_t * r.delta_scale * (total * light - accum));
    }
    if (!more) break;
    t = t_next;
    idx = idx_n;
    delta_t = delta_n;
  }
}

// ---- ray fetch: lane group -> ray index (pixel tiles for the perspective camera) --------------------------
__device__ __forceinline__ bool fetch_ray(const RaySrc& S, const TreeDev& T, Ray& r, long long& out_index) {
  const int grp = threadIdx.x / G;
  float o[3], d[3];
  if (S.o != nullptr) {
    const long long i = (long long)blockIdx.x * RAYS_PER_CTA + grp;
    if (i >= S.n) return false;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      o[a] = __ldg(S.o + 3 * i + a);
      d[a] = __ldg(S.d + 3 * i + a);
    }
    float v[3] = {__ldg(S.v + 3 * i), __ldg(S.v + 3 * i + 1), __ldg(S.v + 3 * i + 2)};
    setup_ray(T.off, T.inv, o, d, v, r);
    out_index = i;
    return true;
  }
  const int W = int(S.cam.width);
  const int tiles_x = (W + PIX_TILE_W - 1) / PIX_TILE_W;
  const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
  const int ix = tx * PIX_TILE_W + grp % PIX_TILE_W;
  const int iyl = ty * PIX_TILE_H + grp / PIX_TILE_W;  // row inside the slab
  if (ix >= W || iyl >= S.nrows) return false;
  cam_ray(S.cam, ix, S.row0 + iyl, o, d);
  setup_ray(T.off, T.inv, o, d, d, r);
  out_index = (long long)iyl * W + ix;
  return true;
}

template <int KPL>
__device__ __forceinline__ void lane_basis(const TreeDev& T, const Ray& r, int l, float* bl) {
  if (T.rgba) {
#pragma unroll
    for (int j = 0; j < KPL; ++j) bl[j] = 1.0f;
    return;
  }
  float b[25];
  const int deg = T.K >= 25 ? 4 : T.K >= 16 ? 3 : T.K >= 9 ? 2 : T.K >= 4 ? 1 : 0;
  sh_basis(deg, r.vdir[0], r.vdir[1], r.vdir[2], b);
#pragma unroll
  for (int j = 0; j < KPL; ++j) {
    const int want = l + j * G;
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < 25; ++k)
      if (k == want && k < T.K) v = b[k];
    bl[j] = v;
  }
}

// The kernels keep the group width as their first template argument (always G), so that their names
// (octree_render_kernel<4, KPL>, ...) stay those of the recorded profiles.  KPL = basis functions per lane.
template <int GW, int KPL>
__global__ void __launch_bounds__(256) octree_render_kernel(TreeDev T, Opts O, RaySrc S, float* __restrict__ out_rgb,
                                                            unsigned long long* __restrict__ counters) {
  static_assert(GW == G, "one group width");
  Ray r;
  long long oi;
  if (!fetch_ray(S, T, r, oi)) return;
  const int l = threadIdx.x % G;
  const unsigned mask = group_mask();
  float bl[KPL];
  lane_basis<KPL>(T, r, l, bl);
  float out[3];
  unsigned visits = 0, hits = 0;
  trace_forward<KPL>(T, O, r, bl, l, mask, out, visits, hits);
  if (l < 3) out_rgb[3 * oi + l] = l == 0 ? out[0] : l == 1 ? out[1] : out[2];
  if (counters != nullptr && l == 0) {
    atomicAdd(counters + 0, (unsigned long long)visits);
    atomicAdd(counters + 1, (unsigned long long)hits);
  }
}

// VolumeRenderer backward for an upstream gradient d loss / d rgb  (svox trace_ray_backward)
template <int GW, int KPL>
__global__ void __launch_bounds__(256) octree_backward_kernel(TreeDev T, Opts O, RaySrc S,
                                                              const float* __restrict__ grad_out,
                                                              float* __restrict__ grad_data) {
  static_assert(GW == G, "one group width");
  Ray r;
  long long oi;
  if (!fetch_ray(S, T, r, oi)) return;
  const int l = threadIdx.x % G;
  const unsigned mask = group_mask();
  float bl[KPL];
  lane_basis<KPL>(T, r, l, bl);
  float out[3];
  unsigned visits = 0, hits = 0;
  Opts Of = O;
  Of.sigma_thresh = 0.f;
  Of.stop_thresh = 0.f;
  trace_forward<KPL>(T, Of, r, bl, l, mask, out, visits, hits);
  float g[3] = {__ldg(grad_out + 3 * oi), __ldg(grad_out + 3 * oi + 1), __ldg(grad_out + 3 * oi + 2)};
  const float accum = g[0] * out[0] + g[1] * out[1] + g[2] * out[2];
  trace_backward<KPL>(T, Of, r, bl, l, mask, g, accum, grad_data);
}

// One training pass over a camera slab (octree/optimization.py:201-207 minus the optimiser):
//   im = render_persp(c2w); mse = mean((clamp(im,0,1) - gt)^2); mse.backward()
// g = grad_scale * 2 * (clamp(im) - gt) inside the clamp range, 0 outside (torch.clamp's gradient).
template <int GW, int KPL>
__global__ void __launch_bounds__(256) octree_train_kernel(TreeDev T, Opts O, RaySrc S, const float* __restrict__ gt,
                                                           float grad_scale, float* __restrict__ grad_data,
                                                           double* __restrict__ sq_err_sum,
                                                           float* __restrict__ out_rgb) {
  static_assert(GW == G, "one group width");
  Ray r;
  long long oi;
  const bool have = fetch_ray(S, T, r, oi);
  float err = 0.f;
  if (have) {
    const int l = threadIdx.x % G;
    const unsigned mask = group_mask();
    float bl[KPL];
    lane_basis<KPL>(T, r, l, bl);
    float out[3];
    unsigned visits = 0, hits = 0;
    trace_forward<KPL>(T, O, r, bl, l, mask, out, visits, hits);
    float g[3];
    float accum = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float cl = fminf(fmaxf(out[c], 0.0f), 1.0f);
      const float diff = cl - __ldg(gt + 3 * oi + c);
      err += diff * diff;
      g[c] = (out[c] >= 0.0f && out[c] <= 1.0f) ? grad_scale * (2.0f * diff) : 0.0f;
      accum += g[c] * out[c];
    }
    if (out_rgb != nullptr && l < 3) out_rgb[3 * oi + l] = l == 0 ? out[0] : l == 1 ? out[1] : out[2];
    if (g[0] != 0.f || g[1] != 0.f || g[2] != 0.f) trace_backward<KPL>(T, O, r, bl, l, mask, g, accum, grad_data);
    if (l != 0) err = 0.f;
  }
  // CTA reduction of the squared error (one double atomic per CTA)
  __shared__ float s_err[8];
  __syncwarp();
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) err += __shfl_xor_sync(0xffffffffu, err, s);
  if ((threadIdx.x & 31) == 0) s_err[threadIdx.x >> 5] = err;
  __syncthreads();
  if (threadIdx.x == 0 && sq_err_sum != nullptr) {
    float tot = 0.f;
    for (int w = 0; w < 8; ++w) tot += s_err[w];
    atomicAdd(sq_err_sum, double(tot));
  }
}

// torch.optim.SGD(momentum=0).step() + zero_grad fused: data -= lr * grad; grad = 0 (octree/optimization.py:205-208)
__global__ void octree_sgd_kernel(float* __restrict__ data, float* __restrict__ grad, long long n, float lr) {
  const long long n4 = n / 4;
  const long long stride = (long long)gridDim.x * blockDim.x;
  float4* d4 = reinterpret_cast<float4*>(data);
  float4* g4 = reinterpret_cast<float4*>(grad);
  // four independent 16-byte gradient loads in flight per thread (the pass is a pure HBM stream)
  for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < n4; i0 += 4 * stride) {
    float4 g[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = i0 + u * stride;
      g[u] = i < n4 ? __ldcs(g4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = i0 + u * stride;
      if (g[u].x != 0.f || g[u].y != 0.f || g[u].z != 0.f || g[u].w != 0.f) {
        float4 d = d4[i];
        d.x = d.x - lr * g[u].x;
        d.y = d.y - lr * g[u].y;
        d.z = d.z - lr * g[u].z;
        d.w = d.w - lr * g[u].w;
        d4[i] = d;
        g4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  }
  for (long long i = n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float g = grad[i];
    if (g != 0.f) {
      data[i] = data[i] - lr * g;
      grad[i] = 0.f;
    }
  }
}

// N3Tree.__getitem__(points) (svox query_vertical): world points -> packed leaf index node*N^3 + (i*N+j)*N+k
__global__ void octree_query_kernel(TreeDev T, const float* __restrict__ pts, long long n, long long* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float pos[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) pos[a] = __fadd_rn(T.off[a], __fmul_rn(T.inv[a], __ldg(pts + 3 * i + a)));
  float cube;
  out[i] = query_leaf(T.child, T.N, pos, cube);
}

// svox grid_trace_ray for every pixel of every camera in ONE launch; weights are max-reduced straight into the
// output grid (the reference keeps a per-camera grid and runs torch.max over 2^27 voxels per camera,
// octree/extraction.py:199-212).  Weights are >= 0, so the float max is an integer atomicMax on the bit pattern.
__global__ void __launch_bounds__(256) grid_weight_kernel(const float* __restrict__ sigma, int reso, const Cam* __restrict__ cams,
                                                          float off0, float off1, float off2, float inv0, float inv1,
                                                          float inv2, Opts O, float* __restrict__ wmax,
                                                          uint8_t* __restrict__ hit) {
  const Cam c = cams[blockIdx.y];
  const int W = int(c.width), H = int(c.height);
  const int tiles_x = (W + 15) / 16;
  const int ix = (blockIdx.x % tiles_x) * 16 + (threadIdx.x & 15);
  const int iy = (blockIdx.x / tiles_x) * 16 + (threadIdx.x >> 4);
  if (ix >= W || iy >= H) return;
  float o[3], d[3];
  cam_ray(c, ix, iy, o, d);
  const float off[3] = {off0, off1, off2}, inv[3] = {inv0, inv1, inv2};
  Ray r;
  setup_ray(off, inv, o, d, d, r);
  if (!r.hit) return;
  float light = 1.0f;
  float t = r.tmin;
  const float fres = float(reso);
  for (int it = 0; t < r.tmax && it < MAX_MARCH_STEPS; ++it) {
    float pos[3];
    int u[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      pos[a] = __fadd_rn(r.o[a], __fmul_rn(t, r.d[a]));
      pos[a] = fmaxf(0.0f, fminf(1.0f - 1e-6f, pos[a]));
      pos[a] = __fmul_rn(pos[a], fres);
      const float fl = floorf(pos[a]);
      u[a] = int(fl);
      pos[a] = __fsub_rn(pos[a], fl);
    }
    float smin, smax;
    dda_unit(pos, r.invd, smin, smax);
    const float delta_t = __fadd_rn(__fsub_rn(smax, smin) / fres, O.step);
    const long long idx = ((long long)u[0] * reso + u[1]) * reso + u[2];
    const float s = __ldg(sigma + idx);
    if (s > O.sigma_thresh) {
      const float att = __expf(-delta_t * r.delta_scale * s);
      const float weight = light * (1.0f - att);
      light *= att;
      if (weight > wmax[idx]) atomicMax(reinterpret_cast<int*>(wmax + idx), __float_as_int(weight));
      if (hit != nullptr) hit[idx] = 1;
      if (light <= O.stop_thresh) return;
    }
    t += delta_t;
  }
}

}  // namespace
}  // namespace pob

// ---------------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------------
namespace {

using namespace pob;

int tree_dev(const char* where, const pob_octree* t, TreeDev& T) {
  if (!t) return pob_fail(where, "tree is NULL");
  if (!t->data_dev || !t->child_dev) return pob_fail(where, "tree data/child pointer is NULL");
  if (t->N < 2 || t->N > 8) return pob_fail(where, "tree branch factor N must be in [2, 8]");
  if (t->n_nodes < 1) return pob_fail(where, "tree has no nodes");
  if (double(t->n_nodes) * t->N * t->N * t->N >= 4294967296.0) return pob_fail(where, "tree too large (leaf index must fit 32 bits)");
  const int K = t->basis_dim;
  if (t->format == POB_OCTREE_RGBA) {
    if (K != 1 || t->data_dim != 4) return pob_fail(where, "RGBA trees have data_dim 4");
  } else if (t->format == POB_OCTREE_SH) {
    if (!(K == 1 || K == 4 || K == 9 || K == 16 || K == 25)) return pob_fail(where, "SH basis_dim must be 1,4,9,16,25");
    if (t->data_dim != 3 * K + 1) return pob_fail(where, "data_dim must be 3*basis_dim + 1 (sigma last)");
  } else {
    return pob_fail(where, "unsupported data format (RGBA and SH only; SG is out of scope)");
  }
  T.data = t->data_dev;
  T.child = t->child_dev;
  T.N = t->N;
  T.D = t->data_dim;
  T.K = K;
  T.rgba = t->format == POB_OCTREE_RGBA;
  for (int a = 0; a < 3; ++a) {
    T.off[a] = t->offset[a];
    T.inv[a] = t->invradius[a];
  }
  if (pob_sm_count_cached() <= 0) return pob_fail(where, "no sm_100 CUDA device (there is no CPU fallback)");
  return 0;
}

int opts_dev(const char* where, const pob_octree_opts* o, Opts& O) {
  if (!o) return pob_fail(where, "options are NULL");
  // every march iteration advances by at least step_size (unit cube): below sqrt(3) / MAX_MARCH_STEPS a diagonal ray
  // would run into the iteration cap and composite the background through the unmarched remainder
  if (!(o->step_size >= 2e-6f))
    return pob_fail(where, "step_size must be >= 2e-6 (the march is capped at 2^20 iterations per ray)");
  O.step = o->step_size;
  O.bg = o->background_brightness;
  O.sigma_thresh = o->sigma_thresh;
  O.stop_thresh = o->stop_thresh;
  return 0;
}

// basis functions per lane: K = 1 or 4 -> 1, 9 -> 3, 16 -> 4, 25 -> 7
#define POB_OCTREE_DISPATCH(KERNEL, K, ...)                                      \
  do {                                                                           \
    if ((K) <= 4) KERNEL<G, 1><<<blocks, 256, 0, st>>>(__VA_ARGS__);             \
    else if ((K) <= 12) KERNEL<G, 3><<<blocks, 256, 0, st>>>(__VA_ARGS__);       \
    else if ((K) <= 16) KERNEL<G, 4><<<blocks, 256, 0, st>>>(__VA_ARGS__);       \
    else KERNEL<G, 7><<<blocks, 256, 0, st>>>(__VA_ARGS__);                      \
  } while (0)

int ray_src(const char* where, const float* o, const float* d, const float* v, long long n, const pob_camera* cam,
            int row0, int nrows, RaySrc& S, unsigned& blocks) {
  S.o = o;
  S.d = d;
  S.v = v;
  S.row0 = 0;
  S.nrows = 0;
  S.n = n;
  if (cam == nullptr) {
    if (!o || !d || !v) return pob_fail(where, "ray pointers are NULL");
    if (n < 0) return pob_fail(where, "negative ray count");
    blocks = unsigned((n + RAYS_PER_CTA - 1) / RAYS_PER_CTA);
    return 0;
  }
  S.o = S.d = S.v = nullptr;
  for (int i = 0; i < 12; ++i) S.cam.c2w[i] = cam->c2w[i];
  S.cam.fx = cam->fx;
  S.cam.fy = cam->fy;
  S.cam.width = cam->width;
  S.cam.height = cam->height;
  const int W = int(cam->width), H = int(cam->height);
  if (W < 1 || H < 1 || !(cam->fx > 0.f) || !(cam->fy > 0.f)) return pob_fail(where, "bad camera");
  if (row0 < 0 || nrows < 0 || row0 + nrows > H) return pob_fail(where, "pixel-row slab outside the image");
  S.row0 = row0;
  S.nrows = nrows;
  S.n = (long long)nrows * W;
  blocks = unsigned(((W + PIX_TILE_W - 1) / PIX_TILE_W) * ((nrows + PIX_TILE_H - 1) / PIX_TILE_H));
  return 0;
}

}  // namespace

extern "C" {

int pob_octree_render(const pob_octree* tree, const pob_octree_opts* opts, const float* origins_dev,
                      const float* dirs_dev, const float* vdirs_dev, int64_t n_rays, const pob_camera* cam,
                      int row0, int nrows, float* out_rgb_dev, unsigned long long* counters_dev, void* stream) {
  const char* W = "pob_octree_render";
  TreeDev T;
  Opts O;
  RaySrc S;
  unsigned blocks = 0;
  if (int rc = tree_dev(W, tree, T)) return rc;
  if (int rc = opts_dev(W, opts, O)) return rc;
  if (int rc = ray_src(W, origins_dev, dirs_dev, vdirs_dev, n_rays, cam, row0, nrows, S, blocks)) return rc;
  if (!out_rgb_dev) return pob_fail(W, "output pointer is NULL");
  if (blocks == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  pob_count_launch();
  POB_OCTREE_DISPATCH(octree_render_kernel, T.K, T, O, S, out_rgb_dev, counters_dev);
  POB_CUDA(W, cudaGetLastError());
  return 0;
}

int pob_octree_render_backward(const pob_octree* tree, const pob_octree_opts* opts, const float* origins_dev,
                               const float* dirs_dev, const float* vdirs_dev, int64_t n_rays, const pob_camera* cam,
                               int row0, int nrows, const float* grad_out_dev, float* grad_data_dev, void* stream) {
  const char* W = "pob_octree_render_backward";
  TreeDev T;
  Opts O;
  RaySrc S;
  unsigned blocks = 0;
  if (int rc = tree_dev(W, tree, T)) return rc;
  if (int rc = opts_dev(W, opts, O)) return rc;
  if (int rc = ray_src(W, origins_dev, dirs_dev, vdirs_dev, n_rays, cam, row0, nrows, S, blocks)) return rc;
  if (!grad_out_dev || !grad_data_dev) return pob_fail(W, "gradient pointer is NULL");
  if (blocks == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  pob_count_launch();
  POB_OCTREE_DISPATCH(octree_backward_kernel, T.K, T, O, S, grad_out_dev, grad_data_dev);
  POB_CUDA(W, cudaGetLastError());
  return 0;
}

int pob_octree_train_persp(const pob_octree* tree, const pob_octree_opts* opts, const pob_camera* cam, int row0,
                           int nrows, const float* gt_rgb_dev, float grad_scale, float* grad_data_dev,
                           double* sq_err_sum_dev, float* out_rgb_dev, void* stream) {
  const char* W = "pob_octree_train_persp";
  TreeDev T;
  Opts O;
  RaySrc S;
  unsigned blocks = 0;
  if (int rc = tree_dev(W, tree, T)) return rc;
  if (int rc = opts_dev(W, opts, O)) return rc;
  if (!cam) return pob_fail(W, "camera is NULL");
  if (O.sigma_thresh != 0.f || O.stop_thresh != 0.f)
    return pob_fail(W, "training renders with sigma_thresh = stop_thresh = 0 (svox fast=False)");
  if (int rc = ray_src(W, nullptr, nullptr, nullptr, 0, cam, row0, nrows, S, blocks)) return rc;
  if (!gt_rgb_dev || !grad_data_dev) return pob_fail(W, "gt / gradient pointer is NULL");
  if (blocks == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  pob_count_launch();
  POB_OCTREE_DISPATCH(octree_train_kernel, T.K, T, O, S, gt_rgb_dev, grad_scale, grad_data_dev, sq_err_sum_dev,
                      out_rgb_dev);
  POB_CUDA(W, cudaGetLastError());
  return 0;
}

int pob_octree_sgd_step(float* data_dev, float* grad_dev, int64_t n, float lr, void* stream) {
  const char* W = "pob_octree_sgd_step";
  if (!data_dev || !grad_dev) return pob_fail(W, "NULL pointer");
  if (n < 0) return pob_fail(W, "negative size");
  const int sms = pob_sm_count_cached();
  if (sms <= 0) return pob_fail(W, "no sm_100 CUDA device (there is no CPU fallback)");
  if ((reinterpret_cast<uintptr_t>(data_dev) | reinterpret_cast<uintptr_t>(grad_dev)) & 15)
    return pob_fail(W, "data / grad must be 16-byte aligned");
  if (n == 0) return 0;
  pob_count_launch();
  octree_sgd_kernel<<<sms * 16, 256, 0, (cudaStream_t)stream>>>(data_dev, grad_dev, n, lr);
  POB_CUDA(W, cudaGetLastError());
  return 0;
}

int pob_octree_adam_step(float* data_dev, float* grad_dev, float* m_dev, float* v_dev, int64_t n, float lr, float step,
                         float eps, void* stream) {
  const char* W = "pob_octree_adam_step";
  if (!data_dev || !grad_dev || !m_dev || !v_dev) return pob_fail(W, "NULL pointer");
  if (n < 0) return pob_fail(W, "negative size");
  if (pob_sm_count_cached() <= 0) return pob_fail(W, "no sm_100 CUDA device (there is no CPU fallback)");
  if (n == 0) return 0;
  pob_count_launch();
  POB_CUDA(W, pob::launch_adam(data_dev, grad_dev, m_dev, v_dev, n, lr, step, nullptr, 0.9f, 0.999f, eps, 1.0f,
                               0.0f, (cudaStream_t)stream));
  POB_CUDA(W, cudaMemsetAsync(grad_dev, 0, size_t(n) * sizeof(float), (cudaStream_t)stream));
  return 0;
}

int pob_octree_query(const pob_octree* tree, const float* points_dev, int64_t n, int64_t* leaf_index_dev,
                     void* stream) {
  const char* W = "pob_octree_query";
  TreeDev T;
  if (int rc = tree_dev(W, tree, T)) return rc;
  if (!points_dev || !leaf_index_dev) return pob_fail(W, "NULL pointer");
  if (n <= 0) return n < 0 ? pob_fail(W, "negative size") : 0;
  pob_count_launch();
  octree_query_kernel<<<unsigned((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      T, points_dev, n, reinterpret_cast<long long*>(leaf_index_dev));
  POB_CUDA(W, cudaGetLastError());
  return 0;
}

int pob_grid_weight_render(const float* sigma_grid_dev, int reso, const pob_camera* cams_dev, int n_cams,
                           int max_width, int max_height, const float offset[3], const float invradius[3],
                           const pob_octree_opts* opts, float* max_weight_dev, uint8_t* hit_dev, void* stream) {
  const char* W = "pob_grid_weight_render";
  Opts O;
  if (int rc = opts_dev(W, opts, O)) return rc;
  if (!sigma_grid_dev || !cams_dev || !max_weight_dev) return pob_fail(W, "NULL pointer");
  if (reso < 1 || reso > 2048) return pob_fail(W, "reso must be in [1, 2048]");
  if (n_cams < 0 || n_cams > 65535) return pob_fail(W, "n_cams must be in [0, 65535] per call");
  if (max_width < 1 || max_height < 1) return pob_fail(W, "bad image size");
  if (pob_sm_count_cached() <= 0) return pob_fail(W, "no sm_100 CUDA device (there is no CPU fallback)");
  if (n_cams == 0) return 0;
  dim3 grid(unsigned(((max_width + 15) / 16) * ((max_height + 15) / 16)), unsigned(n_cams));
  pob_count_launch();
  grid_weight_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      sigma_grid_dev, reso, reinterpret_cast<const Cam*>(cams_dev), offset[0], offset[1], offset[2], invradius[0],
      invradius[1], invradius[2], O, max_weight_dev, hit_dev);
  POB_CUDA(W, cudaGetLastError());
  return 0;
}

}  // extern "C"
