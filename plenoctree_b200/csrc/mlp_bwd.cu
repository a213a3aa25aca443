// mlp_bwd.cu — data-gradient chain of the NeRF-SH MLP (the dgrad half of jax.value_and_grad in
// nerf_sh/train.py:116), fused per iteration like mlp_fwd:
//
//   G' (per-sample d pre_rgb[3], d sigma_raw from render.cu)  --SH basis-->  dO [128 x NH]
//   dH_7 = dO . W_heads ;  dZ_l = dH_l * relu'(h_l) ;  dH_{l-1} = dZ_l . W_l   (l = 7..1)
//
// ReLU masks come from the forward pass (1 bit per activation), the transposed weights from the
// packed `wt_hi` images.  Every dZ_l tile (and dO) is stored to global memory in the same
// swizzled tile-image format as the forward activations; mlp_wgrad contracts them over samples.
// No gradient w.r.t. the inputs is needed (layer 0 and the skip slice of layer 5 stop here).
//
// Warp roles (576 threads): warps 0-3 / 4-7 = epilogue groups of tile X / Y (TMEM lane i <-> sample row i),
// warp 8 = weight producer, warp 9 = MMA issuer (peer CTA: relay), warps 10-13 / 14-17 = copy-out warps of tile
// X / Y.  The finished dZ_l (dO) tile must leave the SM: 64 KB per tile and GEMM against ~25-30 B/clk of SM store
// bandwidth (scripts/overlap_probe.cu) is longer than the GEMM itself, and a warp that issues st.global into a
// full store queue stalls — so the epilogue warps never store.  They hand the tile to the MMA warp AND to their
// copy warps; those pull it into registers half a tile at a time (the shared-memory tile is free again ~2.6 k
// cycles after the hand-over, well before the next epilogue needs it) and let the stores drain from registers.
//
// Two CTAs of a cluster share one tcgen05.mma.cta_group::2 stream over four tiles (512 samples per
// iteration), each CTA holding half of every transposed-weight slot — same protocol as mlp_fwd.cu
// (leader issues, peer relays landed half-slots, commits multicast to both CTAs).
#include "common.cuh"
#include "kernels.h"

namespace pob {

namespace {

constexpr int BWD_THREADS = 576;
constexpr int BWD_COPY_WARP0 = 10;     // first copy-out warp
constexpr int BWD_PRODUCER_WARP = 8;
constexpr int BWD_MMA_WARP = 9;
constexpr int BWD_WSLOTS = 6;            // 16 KB of shared memory each, streamed as two 8 KB half-slots
constexpr int BWD_RING = 2 * BWD_WSLOTS; // ring of 8 KB half-slots: this CTA's half of each weight slot

constexpr uint32_t SB_A0 = 0;
constexpr uint32_t SB_A1 = SB_A0 + A_TILE_BYTES;
constexpr uint32_t SB_W = SB_A1 + A_TILE_BYTES;
constexpr uint32_t SB_TOTAL = SB_W + BWD_WSLOTS * WSLOT_BYTES;  // 128K + 96K = 224K

struct BwdBarriers {
  uint64_t full[BWD_RING];
  uint64_t empty[BWD_RING];
  uint64_t a_ready[2];
  uint64_t d_ready[2];
  uint64_t c_ready[2];   // epilogue group -> copy warps: tile written (4 arrivals)
  uint64_t c_free[2][2]; // copy warps -> epilogue group: first / second half of the tile pulled into registers
};

__device__ __forceinline__ void bwd_stamp(unsigned long long* tr, int role, uint32_t& n) {
  if (tr && blockIdx.x == 0 && n < 256) tr[role * 256 + n++] = clock64();
}

}  // namespace

__device__ __forceinline__ void bwd_body(const BwdParams& p, uint8_t* smem) {
  __shared__ __align__(8) BwdBarriers bars;
  __shared__ uint32_t tmem_base_s;

  constexpr int TILES_PER_ITER = 4;
  constexpr int RING = BWD_RING;
  constexpr uint32_t RSLOT_BYTES = WSLOT_BYTES / 2;
  const long long mrows = padded_rows(p.M);                       // rows of the mask / tile arrays (4-tile units)
  const long long num_iters = mrows / (TILES_PER_ITER * TILE_M);  // padded tiles get zero gradients, not garbage
  const uint32_t warp = warp_id(), lane = lane_id();
  const uint32_t sbase = smem_u32(smem);
  const uint32_t rank = cluster_ctarank();                        // 0 = leader (issues the MMAs)
  const long long unit = (long long)(blockIdx.x >> 1);
  const long long nunits = (long long)(gridDim.x >> 1);
  const int NH = p.NH;
  const int hs = (NH + 31) / 32;            // K slots of the heads dgrad
  const int do_chunks = (NH + 63) / 64;     // 64-wide chunks of the dO tile image

  if (threadIdx.x == 0) {
    for (int i = 0; i < RING; ++i) {
      // leader: a slot is full when its own half has landed AND the peer has reported its half
      mbar_init(smem_u32(&bars.full[i]), rank == 0 ? 2 : 1);
      mbar_init(smem_u32(&bars.empty[i]), 1);
    }
    for (int g = 0; g < 2; ++g) {
      mbar_init(smem_u32(&bars.a_ready[g]), 8);   // 4 own epilogue warps + the peer's 4 (remote)
      mbar_init(smem_u32(&bars.d_ready[g]), 1);
      mbar_init(smem_u32(&bars.c_ready[g]), 4);
      mbar_init(smem_u32(&bars.c_free[g][0]), 4);
      mbar_init(smem_u32(&bars.c_free[g][1]), 4);
    }
    fence_mbar_init();
  }
  cluster_sync_all();   // both CTAs' barriers exist before any remote arrive / multicast commit
  if (warp == BWD_PRODUCER_WARP) tmem_alloc_pair(smem_u32(&tmem_base_s), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  auto wait_bar = [&](uint64_t* b, uint32_t parity) {
    mbar_wait(smem_u32(b), parity);
  };

  if (warp == BWD_PRODUCER_WARP) {
    // whole-warp control flow, one elected lane issues (see mlp_fwd.cu); this CTA's half of every slot
    uint32_t slot = 0, phase = 0;
    const int nslots = hs + 7 * 8;
    for (long long it = unit; it < num_iters; it += nunits) {
      for (int j = 0; j < nslots; ++j) {
        wait_bar(&bars.empty[slot], phase ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(smem_u32(&bars.full[slot]), RSLOT_BYTES);
          bulk_g2s(sbase + SB_W + slot * RSLOT_BYTES, p.w.wt_hi + size_t(j) * WSLOT_BYTES + rank * RSLOT_BYTES,
                   RSLOT_BYTES, smem_u32(&bars.full[slot]));
        }
        __syncwarp();
        if (++slot == RING) {
          slot = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == BWD_MMA_WARP) {
    uint32_t slot = 0, phase = 0, aphase = 0;
    if (rank != 0) {
      // peer CTA: no MMAs to issue; relay every landed half-slot to the leader's full barrier
      const uint32_t pfull0 = mapa_cluster(smem_u32(&bars.full[0]), 0);
      const int nslots = hs + 7 * 8;
      for (long long it = unit; it < num_iters; it += nunits) {
        for (int j = 0; j < nslots; ++j) {
          mbar_wait(smem_u32(&bars.full[slot]), phase);
          if (lane == 0) mbar_arrive_remote(pfull0 + slot * 8u);
          __syncwarp();
          if (++slot == RING) {
            slot = 0;
            phase ^= 1;
          }
        }
      }
    } else {
      // Tile X and tile Y take turns on the tensor core, one whole GEMM at a time: while Y's MMAs run, X's
      // epilogue drains X's accumulator and writes X's next operand tile, and vice versa, so the tensor pipe
      // does not idle through the epilogues (lock-step tiles: MMA 4.4 k + epilogue 1.8 k cycles per GEMM pair).
      // Every weight slot is streamed once and read twice, by X and — one GEMM (ns slots) later — by Y; the
      // ring of 12 half-slots holds the GEMM's 8 slots plus 4 of prefetch.
      const uint32_t idesc = make_idesc_f16(2 * TILE_M, WIDTH);
      constexpr uint64_t A_HI = make_sdesc_hi(1024, LAYOUT_SW128) | (uint64_t(1) << 16);
      constexpr uint64_t W_HI = make_sdesc_hi(512, LAYOUT_SW64) | (uint64_t(1) << 16);
      uint32_t tn = 0;
      unsigned long long* const trm = lane == 0 ? p.trace : nullptr;
      for (long long it = unit; it < num_iters; it += nunits) {
        for (int grp = 0; grp < 8; ++grp) {      // heads, then Dense_7 .. Dense_1
          const int ns = (grp == 0) ? hs : 8;
          constexpr int TURN = 8;   // slots per turn: the whole GEMM (the ring holds it)
          for (int j0 = 0; j0 < ns; j0 += TURN) {
            const int j1 = j0 + TURN < ns ? j0 + TURN : ns;
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              uint32_t rs = slot, rph = phase;   // ring position of the turn's first slot
              if (j0 == 0) {
                wait_bar(&bars.a_ready[g], aphase);
                if (g == 0) bwd_stamp(trm, 0, tn);        // tile X's operand observed
              }
              for (int j = j0; j < j1; ++j) {
                const uint32_t a_off = uint32_t(j >> 1) * A_CHUNK_BYTES + uint32_t(j & 1) * 64u;
                if (g == 0) {                    // the slot lands once; Y finds it in place
                  mbar_wait(smem_u32(&bars.full[rs]), rph);
                }
                const uint64_t bd0 = W_HI | uint64_t(((sbase + SB_W + rs * RSLOT_BYTES) >> 4) & 0x3FFF);
                tc_fence_after();
                if (elect_one()) {
                  const uint32_t a_base = sbase + (g ? SB_A1 : SB_A0) + a_off;
                  const uint64_t ad0 = A_HI | uint64_t((a_base >> 4) & 0x3FFF);
                  const uint32_t d = tmem + uint32_t(g) * 256u;
                  umma_f16_pair(d, ad0, bd0, idesc, j != 0);
                  umma_f16_pair(d, ad0 + 2, bd0 + 2, idesc, 1u);
                  if (j == ns - 1) umma_commit_pair(smem_u32(&bars.d_ready[g]), 0x3);
                  if (g == 1) umma_commit_pair(smem_u32(&bars.empty[rs]), 0x3);
                }
                __syncwarp();
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
          aphase ^= 1;
          bwd_stamp(trm, 0, tn);                        // all MMAs of the GEMM issued
        }
      }
    }
  } else if (warp >= BWD_COPY_WARP0) {
    // ================================ copy-out warps ====================================
    // warp q of tile g copies a quarter of each HALF of every finished tile image (linear: 512 contiguous bytes
    // per warp instruction) through 64 registers: the first half of the image — which the next epilogue rewrites
    // first — is released as soon as it has been read, the second half once the first half's stores are queued.
    const int g = (warp - BWD_COPY_WARP0) >> 2, q = (warp - BWD_COPY_WARP0) & 3;
    const uint8_t* const a_tile = smem + (g ? SB_A1 : SB_A0);
    uint32_t cphase = 0;
    for (long long it = unit; it < num_iters; it += nunits) {
      const long long tile_idx = it * TILES_PER_ITER + int(rank) * 2 + g;
      for (int k = 0; k <= NUM_TRUNK; ++k) {          // dO, dZ_7 .. dZ_0
        const uint32_t half = (k == 0 ? uint32_t(do_chunks) * A_CHUNK_BYTES : uint32_t(A_TILE_BYTES)) / 2;   // 8, 16 or 32 KB
        const uint32_t share = half / 4;                                                                     // 2, 4 or 8 KB
        uint8_t* const dst = (k == 0 ? p.save_do + size_t(tile_idx) * (2 * A_CHUNK_BYTES)
                                     : p.save_dz + (size_t(tile_idx) * NUM_TRUNK + (NUM_TRUNK - k)) * A_TILE_BYTES) +
                             q * share + lane * 16;
        const uint8_t* const src = a_tile + q * share + lane * 16;
        mbar_wait(smem_u32(&bars.c_ready[g]), cphase);
        cphase ^= 1;
        uint4 r[16];
        const int nu = int(share / 512);               // 512-byte rows per batch: 4, 8 or 16
#pragma unroll
        for (int b = 0; b < 2; ++b) {
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (i < nu) r[i] = *reinterpret_cast<const uint4*>(src + b * half + i * 512);
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(&bars.c_free[g][b]));
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (i < nu) *reinterpret_cast<uint4*>(dst + b * half + i * 512) = r[i];
        }
      }
    }
  } else {
    // ================================ epilogue warps ====================================
    const int g = warp >> 2;
    uint32_t tn = 0;
    unsigned long long* const tre = (warp == 0 && lane == 0) ? p.trace : nullptr;
    const int row = int((warp & 3) * 32 + lane);
    uint8_t* const a_tile = smem + (g ? SB_A1 : SB_A0);
    const uint32_t d_tmem = tmem + (uint32_t((warp & 3) * 32) << 16) + uint32_t(g) * 256u;
    uint32_t dphase = 0, fphase = 0;
    bool first_tile = true;
    const uint32_t a_ready_addr = rank != 0 ? mapa_cluster(smem_u32(&bars.a_ready[g]), 0)
                                                      : smem_u32(&bars.a_ready[g]);
    // hand the finished tile to the MMA warp (unless it is dZ_0: no GEMM follows) and to the copy warps
    auto hand_over = [&](bool to_mma) {
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (to_mma) mbar_arrive_cluster_any(a_ready_addr, rank != 0);
        mbar_arrive(smem_u32(&bars.c_ready[g]));
      }
    };
    // before the first write into a half of a_tile: the copy warps have pulled that half of the previous tile
    // into registers (the parity flips after the second half)
    auto wait_half_free = [&](int h) {
      if (!first_tile) mbar_wait(smem_u32(&bars.c_free[g][h]), fphase);
      if (h == 1) {
        if (!first_tile) fphase ^= 1;
        first_tile = false;
      }
    };

    // Global loads of an iteration (per-sample gradient, view direction, ReLU masks) are issued one step ahead
    // of their use.
    auto sample_of = [&](long long it_) { return (it_ * TILES_PER_ITER + int(rank) * 2 + g) * TILE_M + row; };
    auto mask_ptr = [&](int l, long long s_) { return reinterpret_cast<const uint4*>(p.mask + (size_t(l) * mrows + s_) * 8); };
    float4 gq_n = make_float4(0.f, 0.f, 0.f, 0.f);
    float vd_n[3] = {0.f, 0.f, 1.f};
    uint4 mn0 = make_uint4(0, 0, 0, 0), mn1 = mn0;
    auto prefetch_iter = [&](long long it_) {
      const long long s_ = sample_of(it_);
      gq_n = make_float4(0.f, 0.f, 0.f, 0.f);
      if (s_ < p.M) {
        gq_n = p.G[s_];
        const long long vi = p.n_per_ray > 0 ? (s_ < p.M_rays ? s_ / p.n_per_ray : 0) : s_;   // free points: rgb gradient is 0
        const float* vd = p.viewdirs + 3 * vi;
        vd_n[0] = __ldg(vd); vd_n[1] = __ldg(vd + 1); vd_n[2] = __ldg(vd + 2);
      }
      mn0 = __ldg(mask_ptr(NUM_TRUNK - 1, s_));
      mn1 = __ldg(mask_ptr(NUM_TRUNK - 1, s_) + 1);
    };
    if (unit < num_iters) prefetch_iter(unit);

    for (long long it = unit; it < num_iters; it += nunits) {
      const long long tile_idx = it * TILES_PER_ITER + int(rank) * 2 + g;
      const long long s = tile_idx * TILE_M + row;
      // ---- dO row from the per-sample gradient and the SH basis ----
      {
        const float4 gq = gq_n;
        float basis[25];
#pragma unroll
        for (int k = 0; k < 25; ++k) basis[k] = 0.f;   // padded rows: 0 * garbage must not become NaN
        basis[0] = 1.f;
        if (s < p.M && p.sh_deg >= 0) sh_basis(p.sh_deg, vd_n[0], vd_n[1], vd_n[2], basis);
        const float gc[3] = {gq.x, gq.y, gq.z};
        wait_half_free(0);
        wait_half_free(1);
#pragma unroll
        for (int u = 0; u < 16; ++u) {            // 16-byte units of 8 columns, up to 128 columns
          if (u * 8 < do_chunks * 64) {
            uint32_t w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              float f[2];
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const int n = u * 8 + 2 * i + e;
                float v = 0.f;
                if (n == 0) v = gq.w;
                else if (n < 1 + 3 * 25) {
                  const int k = (n - 1) / 3, c = (n - 1) % 3;
                  if (k < p.K) v = gc[c] * basis[k < 25 ? k : 24];
                }
                f[e] = v;
              }
              w[i] = pack_f16x2(f[0], f[1]);
            }
            const uint32_t off = uint32_t(u >> 3) * A_CHUNK_BYTES + uint32_t(row) * 128u +
                                 ((uint32_t(u & 7) ^ uint32_t(row & 7)) << 4);
            *reinterpret_cast<uint4*>(a_tile + off) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
        hand_over(true);
      }
      // ---- dZ_7 .. dZ_0 ----
      for (int l = NUM_TRUNK - 1; l >= 0; --l) {
        // relu mask of h_l (word c: column 32c+2k <-> bit 15-k, column 32c+2k+1 <-> bit 31-k), loaded a step ago
        const uint32_t mw[8] = {mn0.x, mn0.y, mn0.z, mn0.w, mn1.x, mn1.y, mn1.z, mn1.w};
        wait_bar(&bars.d_ready[g], dphase);
        dphase ^= 1;
        tc_fence_after();
        bwd_stamp(tre, 1, tn);                          // d_ready observed
        if (l > 0) {
          mn0 = __ldg(mask_ptr(l - 1, s));
          mn1 = __ldg(mask_ptr(l - 1, s) + 1);
        } else if (it + nunits < num_iters) {
          prefetch_iter(it + nunits);
        }
        // the previous tile is dO for l = 7: its (smaller) image lies entirely inside this tile's first half
        wait_half_free(0);
        if (l == NUM_TRUNK - 1) wait_half_free(1);
        uint32_t va[16], vb[16];
        tmem_ld16(d_tmem, va);
#pragma unroll
        for (int c = 0; c < 16; ++c) {                  // 16 accumulator columns at a time
          uint32_t(&v)[16] = (c & 1) ? vb : va;
          if (c == 8 && l != NUM_TRUNK - 1) wait_half_free(1);   // columns 128.. live in the second half of the image
          tmem_ld_wait();
          if (c + 1 < 16) tmem_ld16(d_tmem + (c + 1) * 16, (c & 1) ? va : vb);   // prefetch next chunk
          const uint32_t m = mw[c >> 1];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            uint32_t w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              // word k of the 32-column group: flags at bits 15-k / 31-k -> shifted to the byte sign bits 15 / 31,
              // replicated over the two halves by PRMT, ANDed onto the packed fp16 pair
              const int k = (c & 1) * 8 + 4 * u + i;
              uint32_t keep;   // bytes 0,1 <- sign of byte 1, bytes 2,3 <- sign of byte 3 (prmt sign-replicate mode)
              asm("prmt.b32 %0, %1, %1, 0xBB99;" : "=r"(keep) : "r"(m << k));
              w[i] = pack_f16x2(__uint_as_float(v[8 * u + 2 * i]), __uint_as_float(v[8 * u + 2 * i + 1])) & keep;
            }
            const uint32_t unit_ = uint32_t((c & 3) * 2 + u);
            const uint32_t off = uint32_t(c >> 2) * A_CHUNK_BYTES + uint32_t(row) * 128u +
                                 ((unit_ ^ uint32_t(row & 7)) << 4);
            *reinterpret_cast<uint4*>(a_tile + off) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
        bwd_stamp(tre, 1, tn);                          // accumulator drained, dZ tile written
        hand_over(l > 0);
        bwd_stamp(tre, 1, tn);                          // handed over
        bwd_stamp(tre, 1, tn);
      }
    }
  }

  tc_fence_before();
  // every epilogue warp has seen the last d_ready = every MMA that reads either CTA's shared memory is done
  cluster_sync_all();
  if (warp == BWD_PRODUCER_WARP) tmem_dealloc_pair(tmem, 512);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(BWD_THREADS, 1)
mlp_bwd_pair_kernel(const __grid_constant__ BwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  bwd_body(p, smem);
}

cudaError_t launch_mlp_bwd(const BwdParams& p, int num_sms, cudaStream_t stream) {
  if (p.M <= 0) return cudaSuccess;
  const long long iters = padded_rows(p.M) / (4 * TILE_M);
  const int pairs = num_sms / 2;
  const int grid = int(iters < pairs ? iters : pairs) * 2;
  cudaError_t e = cudaFuncSetAttribute(mlp_bwd_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SB_TOTAL);
  if (e != cudaSuccess) return e;
  mlp_bwd_pair_kernel<<<grid, BWD_THREADS, SB_TOTAL, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace pob
