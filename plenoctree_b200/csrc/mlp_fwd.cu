// mlp_fwd.cu — fused NeRF-SH point evaluator for sm_100a.
//
// One persistent CTA per SM evaluates   posenc(x) -> 8 x (Dense256 + ReLU, skip-concat into
// layer 5) -> [sigma | SH coefficient] heads -> (optionally) eval_sh at the view direction +
// sigmoid/relu   for 256 samples per iteration, without the activations ever leaving the SM:
//
//   reference path                                      this kernel
//   -------------------------------------------------   ------------------------------------
//   model_utils.posenc      (model_utils.py:145-173)    epilogue warps -> E tile (smem, fp16)
//   model_utils.MLP         (model_utils.py:30-94)      tcgen05.mma, fp32 accum in TMEM,
//                                                       bias+ReLU epilogue TMEM->regs->smem
//   sh.eval_sh + sigmoid/relu (sh.py:54-109,            heads epilogue (registers)
//                              models.py:269-281)
//   NerfModel.eval_points_raw (models.py:143-181)       OUT_RAW / OUT_SIGMA
//
// Warp roles (320 threads): warps 0-3 = epilogue group 0 (tile X), warps 4-7 = epilogue group 1
// (tile Y), warp 8 = weight producer (cp.async.bulk ring in 64 KB of shared memory), warp 9 = MMA issuer.
// Both tiles consume every streamed weight slot, TMEM holds the two 128x256 fp32 accumulators
// (512 columns).
//
// NSPLIT = 1 (fp16) runs as a CTA pair: two CTAs of a cluster (one TPC) run ONE tcgen05.mma.cta_group::2 stream
// over FOUR tiles (512 samples per iteration).  Every MMA has M = 256 (128 rows of tile X or Y from each CTA),
// N = 256, and reads only HALF of the weight slot from each CTA's shared memory: per CTA and MMA the operand
// fetch drops from 12 KB to 8 KB and the weight stream from 16 KB to 8 KB per slot.  That matters because the
// shared-memory / L1 data pipe (128 B/clk) is what a single-CTA fp16 kernel saturated: operand fetch 96 B/clk +
// weight fill 31 B/clk during the MMA phase, before the training variant adds its 128 KB of activation stores
// per layer step (profiles/r2_*; DESIGN.md section 6).  Only the leader CTA (cluster rank 0) issues MMAs; the
// peer's warp 9 relays "my half-slot has landed" to the leader, the peer's epilogue warps arrive on the
// leader's a_ready barriers through the cluster address map, and every commit is multicast to both CTAs.
//
// NSPLIT = 3 (fp16x3) runs on single CTAs and evaluates ONE tile per iteration with error-compensated fp16
// operands (x = hi + lo; hi*hi + lo*hi + hi*lo), using the second tile's buffers for the residual parts; its ring
// holds 4 x 16 KB slots, hi and lo images in turn.
#include "common.cuh"
#include "kernels.h"

namespace pob {

namespace {

constexpr int NUM_EPI_WARPS = 8;
constexpr int PRODUCER_WARP = 8;
constexpr int MMA_WARP = 9;
constexpr int FWD_THREADS = 320;

// dynamic smem map
constexpr uint32_t SM_A0 = 0;
constexpr uint32_t SM_A1 = SM_A0 + A_TILE_BYTES;
constexpr uint32_t SM_E0 = SM_A1 + A_TILE_BYTES;
constexpr uint32_t SM_E1 = SM_E0 + E_TILE_BYTES;
constexpr uint32_t SM_W = SM_E1 + E_TILE_BYTES;
constexpr uint32_t SM_TOTAL = SM_W + NUM_WSLOTS * WSLOT_BYTES;  // 229376
static_assert(SM_TOTAL == 224 * 1024, "smem map");

constexpr int MAX_RING = 8;   // CTA pair: eight 8 KB half-slots in the same 64 KB
struct Barriers {
  uint64_t full[MAX_RING];
  uint64_t empty[MAX_RING];
  uint64_t a_ready[2];
  uint64_t d_ready[2];
};

// packed fp32x2 add (Blackwell FADD2): (a.x + b.x, a.y + b.y)
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  float2 r;
  asm("{\n\t.reg .b64 ra, rb, rc;\n\t"
      "mov.b64 ra, {%2, %3};\n\t"
      "mov.b64 rb, {%4, %5};\n\t"
      "add.rn.f32x2 rc, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rc;\n\t}"
      : "=f"(r.x), "=f"(r.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return r;
}

__device__ __noinline__ void load_point(const FwdParams& p, long long s, float& x, float& y,
                                        float& z) {
  if (s >= p.M) s = p.M - 1;
  if (p.src_mode == SRC_POINTS) {
    const float* q = p.points + 3 * s;
    x = __ldg(q);
    y = __ldg(q + 1);
    z = __ldg(q + 2);
  } else if (p.src_mode == SRC_RAYS && s >= p.M_rays) {
    const float* q = p.extra_points + 3 * (s - p.M_rays);   // free points riding behind the ray samples
    x = __ldg(q);
    y = __ldg(q + 1);
    z = __ldg(q + 2);
  } else if (p.src_mode == SRC_RAYS) {
    long long r = s / p.n_per_ray;
    float t = __ldg(p.zvals + s);
    const float* o = p.origins + 3 * r;
    const float* d = p.directions + 3 * r;
    // cast_rays (model_utils.py:97-101): separate multiply and add, no FMA contraction
    x = __fadd_rn(__ldg(o), __fmul_rn(t, __ldg(d)));
    y = __fadd_rn(__ldg(o + 1), __fmul_rn(t, __ldg(d + 1)));
    z = __fadd_rn(__ldg(o + 2), __fmul_rn(t, __ldg(d + 2)));
  } else {
    // extraction grid (octree/extraction.py:296-304): ((i + 0.5)/reso - offset)/scale
    long long plane = (long long)p.g_ny * p.g_nz;
    int ix = int(s / plane) + p.g_x0;
    int rem = int(s % plane);
    int iy = rem / p.g_nz;
    int iz = rem % p.g_nz;
    float inv = 1.0f / float(p.g_reso);  // reso is a power of two in the reference; see host check
    float ax = __fmul_rn(__fadd_rn(float(ix), 0.5f), inv);
    float ay = __fmul_rn(__fadd_rn(float(iy), 0.5f), inv);
    float az = __fmul_rn(__fadd_rn(float(iz), 0.5f), inv);
    x = __fdiv_rn(__fsub_rn(ax, p.g_offset[0]), p.g_scale[0]);
    y = __fdiv_rn(__fsub_rn(ay, p.g_offset[1]), p.g_scale[1]);
    z = __fdiv_rn(__fsub_rn(az, p.g_offset[2]), p.g_scale[2]);
  }
}

// Positional encoding of one sample into the E tile(s).  Feature order (model_utils.py:162-173):
// [x(3), sin(2^j x_c) j-major (30), sin(2^j x_c + pi/2) (30)], column 63 = 1 (bias carrier).
// unit_lo/unit_hi: which 16-byte units (8 features each) this thread stores.
template <int NSPLIT, bool PRECISE>
__device__ __noinline__ void posenc_row(uint8_t* e_hi, uint8_t* e_lo, int row, float x, float y,
                                           float z, int unit_lo, int unit_hi, uint8_t* e_glob = nullptr) {
  float f[64];
  f[0] = x;
  f[1] = y;
  f[2] = z;
  const float xyz[3] = {x, y, z};
  const float half_pi = 1.5707963267948966f;
#pragma unroll
  for (int j = 0; j < 10; ++j) {
    const float sc = float(1 << j);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float xb = __fmul_rn(xyz[c], sc);
      f[3 + 3 * j + c] = posenc_sin<PRECISE>(xb);
      f[33 + 3 * j + c] = posenc_sin<PRECISE>(__fadd_rn(xb, half_pi));
    }
  }
  f[63] = 1.f;   // constant-one column: carries the biases through the tensor cores (common.cuh)
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    if (u < unit_lo || u >= unit_hi) continue;
    uint32_t w[4], wl[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float a = f[8 * u + 2 * i], b = f[8 * u + 2 * i + 1];
      w[i] = pack_f16x2(a, b);
      if (NSPLIT == 3) {
        float2 h = unpack_f16x2(w[i]);
        wl[i] = pack_f16x2(a - h.x, b - h.y);
      }
    }
    const uint32_t off = uint32_t(row) * 128u + (uint32_t(u ^ (row & 7)) << 4);
    *reinterpret_cast<uint4*>(e_hi + off) = make_uint4(w[0], w[1], w[2], w[3]);
    if (NSPLIT == 3) *reinterpret_cast<uint4*>(e_lo + off) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
    if (e_glob) *reinterpret_cast<uint4*>(e_glob + off) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__device__ __forceinline__ void trace_stamp(unsigned long long* tr, int role, uint32_t& n) {
  if (tr && blockIdx.x == 0 && n < 256) tr[role * 256 + n++] = clock64();
}

}  // namespace

// OUTM (= p.out_mode) is a template parameter so that each instantiation carries only its own heads
// epilogue: the fully unrolled 80-column heads loop with all four output modes inlined made the kernel
// 145+ KB of SASS and cost ~8 % of inference throughput in instruction-cache misses.
template <int NSPLIT, int OUTM, bool SAVE>
__device__ __forceinline__ void fwd_body(const FwdParams& p, uint8_t* smem) {
  constexpr bool PAIR = (NSPLIT == 1);   // the single-pass mode runs as CTA pairs, the x3 mode on single CTAs
  constexpr bool PRECISE = (NSPLIT == 3);
  __shared__ __align__(8) Barriers bars;
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) uint4 slot_tab[FWD_TRUNK_SLOTS + FWD_HEAD_SLOTS + 1];   // MMA issue table (see the MMA warp)

  constexpr int NTILES = (NSPLIT == 1) ? 2 : 1;                       // tiles per CTA and iteration
  constexpr int TILES_PER_ITER = PAIR ? 4 : NTILES;                   // tiles per scheduling unit (CTA or pair)
  constexpr int ROWS_PER_ITER = TILES_PER_ITER * TILE_M;
  constexpr int RING = PAIR ? MAX_RING : NUM_WSLOTS;
  constexpr uint32_t RSLOT_BYTES = PAIR ? WSLOT_BYTES / 2 : WSLOT_BYTES;
  const long long num_iters = (p.M + ROWS_PER_ITER - 1) / ROWS_PER_ITER;
  const uint32_t warp = warp_id(), lane = lane_id();
  const uint32_t sbase = smem_u32(smem);
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;                // 0 = leader (issues the MMAs)
  const long long unit = PAIR ? (long long)(blockIdx.x >> 1) : (long long)blockIdx.x;
  const long long nunits = PAIR ? (long long)(gridDim.x >> 1) : (long long)gridDim.x;

  if (threadIdx.x == 0) {
    for (int i = 0; i < RING; ++i) {
      // pair mode, leader: a slot is full when its own half has landed AND the peer has reported its half
      mbar_init(smem_u32(&bars.full[i]), (PAIR && rank == 0) ? 2 : 1);
      mbar_init(smem_u32(&bars.empty[i]), 1);
    }
    for (int g = 0; g < 2; ++g) {
      // one arrival per epilogue warp that writes the operand tile(s) the MMA reads: 8 in the x3 mode (both
      // groups write one tile) and in pair mode (4 own warps, the peer's four arrive remotely)
      mbar_init(smem_u32(&bars.a_ready[g]), 8);
      mbar_init(smem_u32(&bars.d_ready[g]), 1);
    }
    fence_mbar_init();
  }
  if (PAIR) cluster_sync_all();   // both CTAs' barriers exist before any remote arrive / multicast commit
  if (warp == PRODUCER_WARP) {
    if (PAIR) tmem_alloc_pair(smem_u32(&tmem_base_s), 512);
    else tmem_alloc(smem_u32(&tmem_base_s), 512);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const int NH = p.NH;
  auto wait_bar = [&](uint64_t* b, uint32_t parity) {
    mbar_wait(smem_u32(b), parity);   // (arrivals may come from the other CTA; cta-scope acquire is enough)
  };

  if (warp == PRODUCER_WARP) {
    // =============================== weight producer ===================================
    // pair mode: this CTA streams rows [128 rank, +128) of every trunk slot (rows [NH/2 rank, +NH/2) of the
    // heads slots) = the contiguous half `rank` of the slot image
    uint32_t slot = 0, phase = 0;
    for (long long it = unit; it < num_iters; it += nunits) {
      size_t off = 0;
      for (int l = 0; l <= NUM_TRUNK; ++l) {
        const int ns = (l == NUM_TRUNK) ? FWD_HEAD_SLOTS : fwd_slots_of_layer(l);
        const uint32_t bytes = (l == NUM_TRUNK) ? uint32_t(NH) * 64u : uint32_t(WSLOT_BYTES);
        const uint32_t cbytes = PAIR ? bytes / 2 : bytes;
        for (int j = 0; j < ns; ++j) {
#pragma unroll
          for (int part = 0; part < (NSPLIT == 3 ? 2 : 1); ++part) {
            wait_bar(&bars.empty[slot], phase ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(smem_u32(&bars.full[slot]), cbytes);
              bulk_g2s(sbase + SM_W + slot * RSLOT_BYTES, (part == 0 ? p.w.w_hi : p.w.w_lo) + off + rank * cbytes,
                       cbytes, smem_u32(&bars.full[slot]));
            }
            __syncwarp();
            if (++slot == RING) {
              slot = 0;
              phase ^= 1;
            }
          }
          off += bytes;
        }
      }
    }
  } else if (warp == MMA_WARP) {
    // ================================= MMA issuer ======================================
    // The whole warp runs the (warp-uniform) control flow and the mbarrier waits; one elected lane
    // issues tcgen05.mma / tcgen05.commit.  (A single-lane `if (lane == 0)` loop makes the compiler
    // wrap every UTCHMMA in a divergence-handling ELECT loop and slows the issue rate below the
    // tensor pipe's 128 cycles per 128x256x16 MMA.)
    uint32_t slot = 0, phase = 0, aphase = 0, tn = 0;
    if (PAIR && rank != 0) {
      // peer CTA: no MMAs to issue; relay every landed half-slot to the leader's pfull barrier
      const uint32_t pfull0 = mapa_cluster(smem_u32(&bars.full[0]), 0);
      for (long long it = unit; it < num_iters; it += nunits) {
        for (int l = 0; l <= NUM_TRUNK; ++l) {
          const int ns = (l == NUM_TRUNK) ? FWD_HEAD_SLOTS : fwd_slots_of_layer(l);
          for (int j = 0; j < ns; ++j) {
            mbar_wait(smem_u32(&bars.full[slot]), phase);
            if (lane == 0) mbar_arrive_remote(pfull0 + slot * 8u);
            __syncwarp();
            if (++slot == RING) {
              slot = 0;
              phase ^= 1;
            }
          }
        }
      }
    } else {
    const uint32_t idesc_t = make_idesc_f16(PAIR ? 2 * TILE_M : TILE_M, WIDTH);
    const uint32_t idesc_h = make_idesc_f16(PAIR ? 2 * TILE_M : TILE_M, NH);
    constexpr uint64_t A_HI = make_sdesc_hi(1024, LAYOUT_SW128) | (uint64_t(1) << 16);
    constexpr uint64_t W_HI = make_sdesc_hi(512, LAYOUT_SW64) | (uint64_t(1) << 16);
    const uint32_t w_base = sbase + SM_W;
    if (NSPLIT == 1) {
      // Tiles X and Y take turns of TURN weight slots on the tensor core: X's layer ends one turn before Y's,
      // so X's epilogue (accumulator drain, next operand tile) runs under Y's last turn and Y's under the first
      // turn of X's next layer — the tensor pipe no longer idles through every epilogue (lock-step tiles: 4.4 k
      // cycles of MMAs + 1.3 k of epilogue per layer).  Every weight slot is still streamed once: it stays in
      // the ring from X's use to Y's, TURN slots later (5 of the 8 half-slots live, 3 of prefetch).
      // The issue loop must average < 256 cycles per (tile, slot) = two MMAs, so everything that depends on the
      // layer structure (which tile image feeds K-slot j, bias slots, layer ends) is tabulated once per CTA.
      constexpr int TURN = 5;
      for (int n = int(lane); n < FWD_TRUNK_SLOTS + FWD_HEAD_SLOTS; n += 32) {
        int l = 0, j = n;
        while (l < NUM_TRUNK && j >= fwd_slots_of_layer(l)) j -= fwd_slots_of_layer(l++);
        const int ns = (l == NUM_TRUNK) ? FWD_HEAD_SLOTS : fwd_slots_of_layer(l);
        // A operand of K-slot j: the previous layer's activations, or the posenc tile for layer 0, the skip slots
        // of layer 5, and the bias slot (j == 8) of every other layer, which only multiplies the k16 group
        // [48,64) of the posenc tile (column 63 = 1) with its row k = 31.
        const bool bias_slot = (l == NUM_TRUNK || fwd_has_bias_slot(l)) && j == 8;
        const bool from_e = (l == 0) || j >= 8;
        const int kk = bias_slot ? 1 : ((l == SKIP_LAYER && j >= 8) ? j - 8 : j);
        const uint32_t a_off = uint32_t(kk >> 1) * A_CHUNK_BYTES + uint32_t(kk & 1) * 64u;
        uint4 e;
        e.x = ((sbase + (from_e ? SM_E0 : SM_A0) + a_off) >> 4) & 0x3FFF;
        e.y = ((sbase + (from_e ? SM_E1 : SM_A1) + a_off) >> 4) & 0x3FFF;
        e.z = (bias_slot ? 1u : 0u) | (j != 0 ? 2u : 0u) | (j == ns - 1 ? 4u : 0u) | (l == NUM_TRUNK ? 8u : 0u);
        e.w = 0;
        slot_tab[n] = e;
      }
      __syncwarp();
      const uint32_t w_enc0 = (w_base >> 4) & 0x3FFF;
      for (long long it = unit; it < num_iters; it += nunits) {
        int n0 = 0;                               // table index of the layer's first slot
        for (int l = 0; l <= NUM_TRUNK; ++l) {
          const int ns = (l == NUM_TRUNK) ? FWD_HEAD_SLOTS : fwd_slots_of_layer(l);
          for (int j0 = 0; j0 < ns; j0 += TURN) {
            const int j1 = j0 + TURN < ns ? j0 + TURN : ns;
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              uint32_t rs = slot, rph = phase;   // ring position of the turn's first slot
              if (j0 == 0) {
                wait_bar(&bars.a_ready[g], aphase);   // tile g's operand tile written, D drained (both CTAs)
                if (g == 0) trace_stamp(lane == 0 ? p.trace : nullptr, 0, tn);
              }
              uint4 e = slot_tab[n0 + j0];
              for (int j = j0; j < j1; ++j) {
                const uint4 en = slot_tab[n0 + j + 1];   // (one spare entry behind the table)
                if (g == 0) mbar_wait(smem_u32(&bars.full[rs]), rph);   // the slot lands once; Y finds it in place
                tc_fence_after();
                if (elect_one()) {
                  const uint64_t ah0 = A_HI | uint64_t(g ? e.y : e.x);
                  const uint64_t bh0 = W_HI | uint64_t(w_enc0 + rs * (RSLOT_BYTES >> 4));
                  const uint32_t d = tmem + uint32_t(g) * 256u;
                  const uint32_t idesc = (e.z & 8u) ? idesc_h : idesc_t;
                  // M = 256: rows 0-127 = this CTA's tile g, rows 128-255 = the peer's tile g (same offsets)
                  if (!(e.z & 1u)) umma_f16_pair(d, ah0, bh0, idesc, e.z & 2u);
                  umma_f16_pair(d, ah0 + 2, bh0 + 2, idesc, 1u);      // k16 step 1: +32 bytes = +2 encoded
                  if (e.z & 4u) umma_commit_pair(smem_u32(&bars.d_ready[g]), 0x3);
                  if (g == 1) umma_commit_pair(smem_u32(&bars.empty[rs]), 0x3);
                }
                __syncwarp();
                e = en;
                if (++rs == RING) {
                  rs = 0;
                  rph ^= 1;
                }
              }
              if (g == 1) {
                slot = rs;
                phase = rph;
              }
            }
          }
          n0 += ns;
          aphase ^= 1;
          trace_stamp(lane == 0 ? p.trace : nullptr, 0, tn);       // all MMAs of the layer issued
        }
      }
    } else
    for (long long it = unit; it < num_iters; it += nunits) {
      for (int l = 0; l <= NUM_TRUNK; ++l) {
        const int ns = (l == NUM_TRUNK) ? FWD_HEAD_SLOTS : fwd_slots_of_layer(l);
        const uint32_t idesc = (l == NUM_TRUNK) ? idesc_h : idesc_t;
        for (int j = 0; j < ns; ++j) {
          // A operand of K-slot j: the previous layer's activations, or the posenc tile for layer 0,
          // the skip slots of layer 5, and the bias slot (j == 8) of every other layer, which only
          // multiplies the k16 group [48,64) of the posenc tile (column 63 = 1) with its row k = 31.
          const bool bias_slot = (l == NUM_TRUNK || fwd_has_bias_slot(l)) && j == 8;
          const bool from_e = (l == 0) || j >= 8;
          const int kk = bias_slot ? 1 : ((l == SKIP_LAYER && j >= 8) ? j - 8 : j);
          const uint32_t a_off = uint32_t(kk >> 1) * A_CHUNK_BYTES + uint32_t(kk & 1) * 64u;
          const uint32_t s_hi = slot;
          const uint32_t s_lo = slot + 1;  // x3 only; ring depth is even: hi/lo never straddle the wrap
          mbar_wait(smem_u32(&bars.full[s_hi]), phase);
          if (NSPLIT == 3) mbar_wait(smem_u32(&bars.full[s_lo]), phase);
          const uint64_t bh0 = W_HI | uint64_t(((w_base + s_hi * RSLOT_BYTES) >> 4) & 0x3FFF);
          const uint64_t bl0 = W_HI | uint64_t(((w_base + s_lo * RSLOT_BYTES) >> 4) & 0x3FFF);
#pragma unroll
          for (int g = 0; g < NTILES; ++g) {
            if (j == 0) {
              wait_bar(&bars.a_ready[g], aphase);   // tile g's operand tile(s) written, D drained (both CTAs)
              if (g == 0) trace_stamp(lane == 0 ? p.trace : nullptr, 0, tn);
            }
            tc_fence_after();
            if (elect_one()) {
              const uint32_t a_base = sbase + (from_e ? (g ? SM_E1 : SM_E0) : (g ? SM_A1 : SM_A0)) + a_off;
              const uint64_t ah0 = A_HI | uint64_t((a_base >> 4) & 0x3FFF);
              const uint32_t d = tmem + uint32_t(g) * 256u;
              // tile 0 only: hi operand lives in the "tile 0" buffers, lo in the "tile 1" ones
              const uint32_t a_lo_base = sbase + (from_e ? SM_E1 : SM_A1) + a_off;
              const uint64_t al0 = A_HI | uint64_t((a_lo_base >> 4) & 0x3FFF);
              if (!bias_slot) {
                umma_f16(d, al0, bh0, idesc, j != 0);
                umma_f16(d, ah0, bl0, idesc, 1u);
                umma_f16(d, ah0, bh0, idesc, 1u);
              }
              umma_f16(d, al0 + 2, bh0 + 2, idesc, 1u);      // k16 step 1: +32 bytes = +2 encoded
              umma_f16(d, ah0 + 2, bl0 + 2, idesc, 1u);
              umma_f16(d, ah0 + 2, bh0 + 2, idesc, 1u);
              if (j == ns - 1) umma_commit(smem_u32(&bars.d_ready[g]));
              if (g == NTILES - 1) {
                umma_commit(smem_u32(&bars.empty[s_hi]));
                umma_commit(smem_u32(&bars.empty[s_lo]));
              }
            }
            __syncwarp();
          }
          __syncwarp();
          slot += (NSPLIT == 3) ? 2 : 1;
          if (slot == RING) {
            slot = 0;
            phase ^= 1;
          }
        }
        aphase ^= 1;
        trace_stamp(lane == 0 ? p.trace : nullptr, 0, tn);       // all MMAs of the layer issued
      }
    }
    }
  } else {
    // ================================ epilogue warps ====================================
    const int g = warp >> 2;                       // group
    const int row = int((warp & 3) * 32 + lane);   // TMEM lane == tile row
    const int tile_in_iter = (NSPLIT == 1) ? int(rank) * 2 + g : 0;   // pair: leader owns tiles 0,1, peer 2,3
    const int bar_id = (NSPLIT == 1) ? g : 0;
    // column range of the trunk epilogue handled by this thread, in 32-column chunks
    const int c_begin = (NSPLIT == 1) ? 0 : 4 * g;
    const int c_end = (NSPLIT == 1) ? 8 : 4 * g + 4;
    uint8_t* const a_hi = smem + ((NSPLIT == 1 && g == 1) ? SM_A1 : SM_A0);
    uint8_t* const a_lo = smem + SM_A1;
    uint8_t* const e_hi = smem + ((NSPLIT == 1 && g == 1) ? SM_E1 : SM_E0);
    uint8_t* const e_lo = smem + SM_E1;
    const int unit_lo = (NSPLIT == 1) ? 0 : 4 * g, unit_hi = (NSPLIT == 1) ? 8 : 4 * g + 4;
    const uint32_t d_tmem = tmem + (uint32_t((warp & 3) * 32) << 16) + uint32_t(bar_id) * 256u;
    constexpr bool saving = SAVE;   // training launches (NSPLIT == 1): store h_l tiles, posenc tiles and relu masks
    uint32_t dphase = 0, tn = 0;
    const bool tracer = (warp & 3) == 0 && lane == 0;
    unsigned long long* const trp = tracer ? p.trace : nullptr;
    const int trole = 1 + g;

    // the MMA issuer (leader CTA) waits on ITS a_ready barrier: the peer's warps arrive through the cluster map
    const uint32_t a_ready_addr = (PAIR && rank != 0) ? mapa_cluster(smem_u32(&bars.a_ready[bar_id]), 0)
                                                      : smem_u32(&bars.a_ready[bar_id]);
    auto signal_a_ready = [&]() {
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster_any(a_ready_addr, rank != 0);
        else mbar_arrive(a_ready_addr);
      }
    };

    long long it = unit;
    if (it < num_iters) {
      float x, y, z;
      load_point(p, it * ROWS_PER_ITER + tile_in_iter * TILE_M + row, x, y, z);
      posenc_row<NSPLIT, PRECISE>(e_hi, e_lo, row, x, y, z, unit_lo, unit_hi,
                                  saving ? p.save_e + size_t(it * TILES_PER_ITER + tile_in_iter) * E_TILE_BYTES : nullptr);
      signal_a_ready();
    }
    for (; it < num_iters; it += nunits) {
      const long long tile_idx = it * TILES_PER_ITER + tile_in_iter;
      const long long s = tile_idx * TILE_M + row;
      // ------------------------------ trunk layers ------------------------------------
      for (int l = 0; l < NUM_TRUNK; ++l) {
        wait_bar(&bars.d_ready[bar_id], dphase);
        dphase ^= 1;
        tc_fence_after();
        trace_stamp(trp, trole, tn);             // d_ready observed
        constexpr int NCH = (NSPLIT == 1) ? 8 : 4;
        uint32_t va[32], vb[32];
        tmem_ld32(d_tmem + c_begin * 32, va);
#pragma unroll
        for (int cc = 0; cc < NCH; ++cc) {
          const int c = c_begin + cc;
          uint32_t(&v)[32] = (cc & 1) ? vb : va;
          tmem_ld_wait();                                    // chunk cc has landed
          if (cc + 1 < NCH) tmem_ld32(d_tmem + (c + 1) * 32, (cc & 1) ? va : vb);   // prefetch chunk cc+1
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            // bias already accumulated by the tensor cores: ReLU + fp16 pack is all that is left
            uint32_t w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              w[i] = pack_f16x2_relu(__uint_as_float(v[8 * u + 2 * i]), __uint_as_float(v[8 * u + 2 * i + 1]));
            const uint32_t unit = uint32_t((c & 1) * 4 + u);
            const uint32_t off = uint32_t(c >> 1) * A_CHUNK_BYTES + uint32_t(row) * 128u +
                                 ((unit ^ uint32_t(row & 7)) << 4);
            *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(w[0], w[1], w[2], w[3]);
            if (NSPLIT == 3) {
              uint32_t wl[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                float2 h = unpack_f16x2(w[i]);
                wl[i] = pack_f16x2(fmaxf(__uint_as_float(v[8 * u + 2 * i]), 0.f) - h.x,
                                   fmaxf(__uint_as_float(v[8 * u + 2 * i + 1]), 0.f) - h.y);
              }
              *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
            }
          }
          if (cc == 0) trace_stamp(trp, trole, tn);   // first chunk done
        }
        trace_stamp(trp, trole, tn);             // accumulator drained, A tile written
        signal_a_ready();
        trace_stamp(trp, trole, tn);             // a_ready signalled
        if (saving && NSPLIT == 1) {
          // Training saves, AFTER the hand-over (off the MMA -> epilogue -> MMA critical path): every thread reads its
          // own row of the finished tile back from shared memory (the next layer's MMAs only read it too), stores it
          // to global memory in the "T" layout (layouts.py: t_tile_offset; 512 contiguous bytes per warp store) that
          // mlp_wgrad contracts MN-major without swizzle, and derives the ReLU mask of the row from the fp16 values
          // (h > 0 <=> fp16(h) != 0 up to fp16 underflow).  Mask word c covers columns 32c..32c+31: column 32c+2k is
          // bit 15-k, column 32c+2k+1 is bit 31-k (two instructions per fp16 pair; mlp_bwd tests the same bits).
          // The store stream (64 KB per tile and layer against ~25-30 B/clk of SM store bandwidth) is the longest
          // stage of the training forward: it has the whole MMA phase to drain.  Measured alternatives
          // (scripts/overlap_probe.cu, profiles/r2_overlap_probe.json): stores issued from inside the epilogue stall
          // it, because a backed-up st.global queue blocks the warp's later st.shared / fences; a TMA bulk store of the
          // verbatim tile image (no LSU time at all) collides with the weight-slot TMA loads and with the MMA operand
          // reads: 73.5 k vs 63.1 k cycles per iteration (tried in round 2, removed).
          uint8_t* const h_glob = p.save_h + (size_t(tile_idx) * NUM_TRUNK + l) * A_TILE_BYTES;
          uint32_t maskw[8];
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            uint32_t mbits = 0;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const uint32_t unit = uint32_t((c & 1) * 4 + u);
              const uint32_t off = uint32_t(c >> 1) * A_CHUNK_BYTES + uint32_t(row) * 128u +
                                   ((unit ^ uint32_t(row & 7)) << 4);
              const uint4 q = *reinterpret_cast<const uint4*>(a_hi + off);
              *reinterpret_cast<uint4*>(h_glob + uint32_t(warp & 3) * 16384u + uint32_t(c * 4 + u) * 512u + lane * 16u) = q;
              const uint32_t qw[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
              for (int i = 0; i < 4; ++i)   // non-negative fp16 pair -> 0/1 per half (VIMNMX.U16x2), shifted in
                mbits = (mbits << 1) + __vminu2(qw[i], 0x00010001u);
            }
            maskw[c] = mbits;
          }
          const long long mrows = padded_rows(p.M);
          uint4* mp = reinterpret_cast<uint4*>(p.save_mask + (size_t(l) * mrows + s) * 8);
          mp[0] = make_uint4(maskw[0], maskw[1], maskw[2], maskw[3]);
          mp[1] = make_uint4(maskw[4], maskw[5], maskw[6], maskw[7]);
        }
        if (l == SKIP_LAYER) {
          // E is dead until the next iteration: encode the next tile now, in the shadow of the
          // layer-6/7/heads MMAs.
          const long long nit = it + nunits;
          if (nit < num_iters) {
            float x, y, z;
            load_point(p, nit * ROWS_PER_ITER + tile_in_iter * TILE_M + row, x, y, z);
            posenc_row<NSPLIT, PRECISE>(e_hi, e_lo, row, x, y, z, unit_lo, unit_hi,
                                        saving ? p.save_e + size_t(nit * TILES_PER_ITER + tile_in_iter) * E_TILE_BYTES
                                               : nullptr);
            fence_proxy_async_smem();
          }
        }
      }
      // -------------------------------- heads ------------------------------------------
      wait_bar(&bars.d_ready[bar_id], dphase);
      dphase ^= 1;
      tc_fence_after();
      if (NSPLIT == 1 || g == 0) {
        const int K = p.K;
        float sigma_raw = 0.f;
        float pre[3] = {0.f, 0.f, 0.f};
        float basis[25];
        float* stage = nullptr;
        int P = 0;

        if (OUTM == OUT_RGBS) {
          long long sc = s < p.M ? s : p.M - 1;
          long long vi = (p.src_mode == SRC_RAYS) ? (sc < p.M_rays ? sc / p.n_per_ray : 0) : sc;   // free points: any direction
          const float* vd = p.viewdirs + 3 * vi;
          if (p.sh_deg >= 0) sh_basis(p.sh_deg, __ldg(vd), __ldg(vd + 1), __ldg(vd + 2), basis);
          else basis[0] = 1.f;
        } else if (OUTM == OUT_RAW || OUTM == OUT_CELL_MEAN) {
          // per-warp staging area inside this group's (now dead) activation tile
          P = (3 * K + 1) | 1;  // odd pitch -> conflict-free scalar stores
          stage = reinterpret_cast<float*>(a_hi + (warp & 3) * 16384) + lane * P;
        }
#pragma unroll
        for (int q = 0; q < MAX_NH / 16; ++q) {
          if (q * 16 < NH) {
            uint32_t v[16];
            tmem_ld16(d_tmem + q * 16, v);
            tmem_ld_wait();
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
              const int n = q * 16 + jj;
              if (n == 0) {
                sigma_raw = __uint_as_float(v[0]);
              } else {
                const int k = (n - 1) / 3, c = (n - 1) % 3;
                if (k < K) {
                  const float coef = __uint_as_float(v[jj]);
                  if (OUTM == OUT_RGBS) pre[c] = fmaf(basis[k < 25 ? k : 24], coef, pre[c]);
                  else if (OUTM == OUT_RAW) stage[c * K + k] = coef;
                  else if (OUTM == OUT_CELL_MEAN) stage[c * K + k] = coef;
                }
              }
            }
          }
        }
        if (OUTM == OUT_RGBS) {
          if (s < p.M) {
            float4 o;
            o.x = 1.f / (1.f + expf(-pre[0]));
            o.y = 1.f / (1.f + expf(-pre[1]));
            o.z = 1.f / (1.f + expf(-pre[2]));
            if (p.sigma_noise != nullptr && (p.src_mode != SRC_RAYS || s < p.M_rays))
              sigma_raw += __ldg(p.sigma_noise + s);  // add_gaussian_noise
            o.w = fmaxf(sigma_raw, 0.f);
            p.out_rgbs[s] = o;
          }
        } else if (OUTM == OUT_CELL_MEAN) {
          // extraction step 2 (octree/extraction.py:367-394): out[cell] += cat([raw_rgb, raw_sigma]) / S.
          // The warp's 32 rows sit in the staging area; lanes own output columns and sum over rows (one
          // cell per warp when S is a multiple of 32), then one atomicAdd per column.
          stage[3 * K] = sigma_raw;
          __syncwarp();
          const float* wstage = reinterpret_cast<const float*>(a_hi + (warp & 3) * 16384);
          const long long row0 = tile_idx * TILE_M + (warp & 3) * 32;
          const int width = 3 * K + 1;
          const float inv = 1.0f / float(p.cell_S);
          if ((p.cell_S & 31) == 0) {
            if (row0 < p.M) {
              float* dst = p.out_cell + (row0 / p.cell_S) * width;
              for (int i = lane; i < width; i += 32) {
                float acc = 0.f;
                for (int rr = 0; rr < 32; ++rr) acc += wstage[rr * P + i];
                atomicAdd(dst + i, acc * inv);
              }
            }
          } else {
            for (int rr = 0; rr < 32; ++rr) {
              if (row0 + rr >= p.M) break;
              float* dst = p.out_cell + ((row0 + rr) / p.cell_S) * width;
              for (int i = lane; i < width; i += 32) atomicAdd(dst + i, wstage[rr * P + i] * inv);
            }
          }
          __syncwarp();
        } else {
          if (s < p.M) p.out_sigma[s] = sigma_raw;
          if (OUTM == OUT_RAW) {
            __syncwarp();
            const float* wstage = reinterpret_cast<const float*>(a_hi + (warp & 3) * 16384);
            const long long row0 = tile_idx * TILE_M + (warp & 3) * 32;
            const int C3 = 3 * K;
            for (int rr = 0; rr < 32; ++rr) {
              if (row0 + rr >= p.M) break;
              for (int i = lane; i < C3; i += 32)
                p.out_rgb[(row0 + rr) * C3 + i] = wstage[rr * P + i];
            }
            __syncwarp();
          }
        }
      }
      // heads accumulator drained, next E tile already encoded (or this was the last iteration)
      signal_a_ready();
    }
  }

  tc_fence_before();
  if (PAIR) {
    // every epilogue warp has seen the last d_ready = every MMA that reads either CTA's shared memory is done
    cluster_sync_all();
    if (warp == PRODUCER_WARP) tmem_dealloc_pair(tmem, 512);
  } else {
    __syncthreads();
    if (warp == PRODUCER_WARP) tmem_dealloc(tmem, 512);
  }
}

// single-CTA kernel: the x3 mode only (the single-pass mode runs as CTA pairs)
template <int NSPLIT, int OUTM, bool SAVE>
__global__ void __launch_bounds__(FWD_THREADS, 1)
mlp_fwd_kernel(const __grid_constant__ FwdParams p) {
  static_assert(NSPLIT == 3 && !SAVE, "single-CTA kernel: x3 inference only");
  extern __shared__ __align__(1024) uint8_t smem[];
  fwd_body<NSPLIT, OUTM, SAVE>(p, smem);
}

template <int OUTM, bool SAVE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(FWD_THREADS, 1)
mlp_fwd_pair_kernel(const __grid_constant__ FwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  fwd_body<1, OUTM, SAVE>(p, smem);
}

cudaError_t launch_mlp_fwd(const FwdParams& p, int nsplit, int num_sms, cudaStream_t stream) {
  if (p.M <= 0) return cudaSuccess;
  if (nsplit != 1 && nsplit != 3) return cudaErrorInvalidValue;
  const bool pair = nsplit == 1;
  const int rows = pair ? 4 * TILE_M : TILE_M;
  const long long iters = (p.M + rows - 1) / rows;
  const int units = pair ? num_sms / 2 : num_sms;
  const int grid = int(iters < units ? iters : units) * (pair ? 2 : 1);
  auto launch = [&](auto kernel) -> cudaError_t {
    cudaError_t e =
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_TOTAL);
    if (e != cudaSuccess) return e;
    kernel<<<grid, FWD_THREADS, SM_TOTAL, stream>>>(p);
    return cudaGetLastError();
  };
  const bool save = p.save_h != nullptr;
  if (save && (nsplit != 1 || !p.save_e || !p.save_mask ||
               (p.out_mode != OUT_RGBS && p.out_mode != OUT_SIGMA)))
    return cudaErrorInvalidValue;
  if (pair) {
    switch (p.out_mode) {
      case OUT_RAW: return launch(mlp_fwd_pair_kernel<OUT_RAW, false>);
      case OUT_SIGMA: return save ? launch(mlp_fwd_pair_kernel<OUT_SIGMA, true>) : launch(mlp_fwd_pair_kernel<OUT_SIGMA, false>);
      case OUT_RGBS: return save ? launch(mlp_fwd_pair_kernel<OUT_RGBS, true>) : launch(mlp_fwd_pair_kernel<OUT_RGBS, false>);
      case OUT_CELL_MEAN: return launch(mlp_fwd_pair_kernel<OUT_CELL_MEAN, false>);
      default: return cudaErrorInvalidValue;
    }
  }
  switch (p.out_mode) {
    case OUT_RAW: return launch(mlp_fwd_kernel<3, OUT_RAW, false>);
    case OUT_SIGMA: return launch(mlp_fwd_kernel<3, OUT_SIGMA, false>);
    case OUT_RGBS: return launch(mlp_fwd_kernel<3, OUT_RGBS, false>);
    case OUT_CELL_MEAN: return launch(mlp_fwd_kernel<3, OUT_CELL_MEAN, false>);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace pob
