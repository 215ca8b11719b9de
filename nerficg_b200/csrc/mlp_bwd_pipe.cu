// mlp_bwd_pipe.cu -- K4 fused: data gradients AND weight gradients of the NeRF MLP in one persistent kernel whose CTA
// pairs are LAYER-STATIONARY pipeline stages.
//
// Why.  In the tile-major chain (mlp_bwd.cu) the per-layer output gradients dY_l leave the SM for HBM (624 KB per
// 128-sample tile) and the layer-major weight-gradient kernel (mlp_wgrad.cu) reads them back together with the activation
// stash (1,424 KB per tile): 10.4 of the step's 23.1 GB are that round trip, and both kernels are bound by memory paths
// (measured, tools/l2_probe.py: an SM's store path to L2 carries 27-32 B/clk whoever issues the store, and a queued 64 KB
// image store delays the weight-ring loads queued behind it).  A weight gradient needs an accumulator per LAYER
// (256 x 256 fp32 = all 512 TMEM columns of one SM), so it cannot live inside a tile-major chain -- but it can if the CHAIN
// is laid across SMs instead of across time:
//
//   pipeline p (8 of them) = 9 CTA pairs: [head] -> [F] -> [L7] -> [L6] -> [L5] -> [L4] -> [L3] -> [L2] -> [L1]
//   head      : dL/d(rgb, sigma_raw) -> dG (CUDA cores, as the chain's prologue), dF = dG W_c0[:, :256]      (tcgen05, 2 slots)
//   stage st  : receives dY_in (dF, dY7, ... dY1), keeps ITS layer's W^T half resident in shared memory and ITS layer's
//               dW half (128 x 256 fp32 = 256 TMEM columns) resident in tensor memory for the whole kernel:
//                 dgrad  acc[256 smp x 256]  = dY_in [K-major A]  x W^T            (cta_group::2, M = 256 samples)
//                 wgrad  dW [256 x 256]     += dY_in^T [MN-major A] x H [MN-major B, activation stash]   (M = 256 features)
//               the epilogue (ReLU mask of the forward, fp16) of group t overlaps the wgrad MMAs of group t, so the tensor
//               pipe never waits for a TMEM drain; dY_out travels to the next pair through a 4-deep ring in L2.
//   Groups of 256 samples (one 128-sample tile per CTA of a pair) are dealt round-robin to the 8 pipelines; the 72 pairs
//   run concurrently (74 two-SM clusters fit on 148 SMs; 2 pairs stay idle) and synchronise through monotone
//   counters in global memory (release/acquire at gpu scope; the producer never overtakes the 4-slot ring).
//
// HBM traffic per tile: the activation stash is read ONCE (H0..H7: 512 KB + masks), and only dG, dY5, dY0 and the head
// panel (176 KB) are still written for the small residual weight-gradient kernel (mlp_wgrad.cu, jobs 8-12: encodings,
// colour head) -- instead of 624 KB written + 1,424 KB read.  Bias gradients are column sums of dY_in on CUDA cores
// (reducer warps), the density head's weight gradient is sum_m dsigma_raw[m] h7[m][:] on the same warps of stage F.
#include "common.cuh"
#include "mlp_layout.cuh"
#include "tc.cuh"
#include "../../include/nerf_b200.h"

namespace nerf {
using namespace tc;

namespace pipe {
constexpr int kThreads = 640;                 // warps 0-3 service, 4-19 epilogue / reducer / store roles
constexpr int kPipelines = 8;
constexpr int kRoles = 9;                     // head + 8 stages
constexpr int kLinks = 8;                     // link k feeds stage k + 1
constexpr int kLinkSlots = 4;
constexpr uint32_t kStageBytes = kPanelBytes128;   // 16 KB ring stage
constexpr uint32_t kHalfPanel = 8192;
constexpr int kRing = 8;
constexpr uint32_t kGroupBytes = 2 * kActBytes;    // one link slot: two tile images
// shared memory map of a stage CTA
constexpr uint32_t kOffW = 0;                                   // 4 x 16 KB: this CTA's half of the layer's W^T panels
constexpr uint32_t kOffRing = kOffW + kActBytes;                // 8 x 16 KB
constexpr uint32_t kOffOut = kOffRing + kRing * kStageBytes;    // 32 KB: two panels of the dY_out image (one 128-column phase)
constexpr uint32_t kOffBars = kOffOut + 2 * kPanelBytes128;
constexpr uint32_t kOffDsig = kOffBars + 512;                   // 128 floats: dsigma_raw of the tile in flight (stage F)
constexpr uint32_t kSmemBytes = kOffDsig + 512;
static_assert(kSmemBytes <= 232448, "shared memory budget exceeded");
// shared memory map of a head CTA: W (2 x 16 KB) | dG operand of slot 0, 1 (2 x 32 KB) | dF image of slot 0, 1 (2 x 64 KB)
constexpr uint32_t kHeadOffA = 2 * kPanelBytes128;
constexpr uint32_t kHeadOffOut = kHeadOffA + 2 * (2 * kPanelBytes128);
static_assert(kHeadOffOut + 2 * kActBytes <= kOffBars, "head layout overlaps the barriers");
constexpr int kRegsEpilogue = 112, kRegsOther = 32;
constexpr size_t kLinkBytes = (size_t)kPipelines * kLinks * kLinkSlots * kGroupBytes;   // 32 MB
constexpr size_t kFlagStride = 32;                                                      // uint32 per flag, 128 B apart
constexpr size_t kFlagBytes = 2 * (size_t)kPipelines * kLinks * kLinkSlots * kFlagStride * 4;
}  // namespace pipe

struct PipeParams {
  float* grads;
  const float4* d_rgbsigma;
  const float4* rgbsigma;
  const uint8_t* stash;
  uint8_t* gstash;
  uint8_t* links;
  uint32_t* flags;          // [2][pipelines][links][slots][kFlagStride]: ready, then freed
  const uint8_t* packed;
  const float* params;
  int64_t n_evals;
  int n_tiles;
  float inv_scale;
  unsigned long long* prof;   // optional stall counters (tools/pipe_timing.py), see the slot list at the end of the kernel
};

// ---- flags (gpu scope) ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// plain (relaxed) add: used to hand a link slot BACK -- the reads it covers have completed (their mbarrier flipped), nothing is published
__device__ __forceinline__ void red_relaxed_gpu(uint32_t* p, uint32_t v) {
  asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void spin_until(const uint32_t* p, uint32_t target) {
  while (ld_acquire_gpu(p) < target) __nanosleep(32);
}
#define PIPE_TIMED(acc, stmt) NERF_TIMED(prof_on, acc, stmt)
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// 16 columns of a dgrad epilogue (as in mlp_bwd.cu): t = acc (+ dsigma_raw * w_sigma), masked by the forward's ReLU bits
template <bool kSig>
__device__ __forceinline__ void pipe_dgrad16(const uint32_t (&v)[16], uint32_t m, int qbase, const float* __restrict__ ws, float dsr,
                                             uint32_t dst0, uint32_t dst1) {
  uint32_t w[8];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float t0 = __uint_as_float(v[4 * q + 0]), t1 = __uint_as_float(v[4 * q + 1]);
    float t2 = __uint_as_float(v[4 * q + 2]), t3 = __uint_as_float(v[4 * q + 3]);
    if (kSig) {
      const float4 wq = __ldg(reinterpret_cast<const float4*>(ws) + q);
      t0 = fmaf(dsr, wq.x, t0);
      t1 = fmaf(dsr, wq.y, t1);
      t2 = fmaf(dsr, wq.z, t2);
      t3 = fmaf(dsr, wq.w, t3);
    }
    t0 = (m & (1u << (qbase + 2 * q))) ? t0 : 0.f;
    t1 = (m & (1u << (16 + qbase + 2 * q))) ? t1 : 0.f;
    t2 = (m & (1u << (qbase + 2 * q + 1))) ? t2 : 0.f;
    t3 = (m & (1u << (16 + qbase + 2 * q + 1))) ? t3 : 0.f;
    w[2 * q] = pack_half2(t0, t1);
    w[2 * q + 1] = pack_half2(t2, t3);
  }
  st_shared_v4(dst0, w[0], w[1], w[2], w[3]);
  st_shared_v4(dst1, w[4], w[5], w[6], w[7]);
}

// accumulator (this warp's 32 lanes x 128 columns at t_acc) -> masked fp16 -> the two panels of this column half at out_h
template <bool kSig>
__device__ __forceinline__ void pipe_drain_acc(uint32_t t_acc, const uint32_t (&mk)[4], const float* __restrict__ wsp, float dsr,
                                               uint32_t out_h, uint32_t xr) {
  uint32_t va[16], vb[16];
  tmem_ld16(t_acc, va);
#pragma unroll
  for (int s = 0; s < 8; s += 2) {
    const uint32_t pbase = out_h + (uint32_t)(s >> 2) * kPanelBytes128;
    const uint32_t c0 = (uint32_t)(s & 3) * 32u;
    tmem_ld_wait16(va);
    tmem_ld16(t_acc + 16 * (s + 1), vb);
    pipe_dgrad16<kSig>(va, mk[s >> 1], 0, wsp + 16 * s, dsr, pbase + (c0 ^ xr), pbase + ((c0 + 16u) ^ xr));
    tmem_ld_wait16(vb);
    if (s + 2 < 8) tmem_ld16(t_acc + 16 * (s + 2), va);
    pipe_dgrad16<kSig>(vb, mk[s >> 1], 8, wsp + 16 * (s + 1), dsr, pbase + ((c0 + 32u) ^ xr), pbase + ((c0 + 48u) ^ xr));
  }
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(pipe::kThreads, 1) mlp_bwd_pipe_kernel(const PipeParams p) {
  using namespace pipe;
  using L = ParamLayout;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = smem_u32(smem_raw);
  if ((smem_base & 1023u) != 0) __trap();
  const uint32_t rank = cluster_ctarank();
  const int cluster_id = (int)blockIdx.x >> 1;
  if (cluster_id >= kPipelines * kRoles) return;          // the two spare pairs
  const int pl = cluster_id / kRoles, role = cluster_id % kRoles;   // role 0 = head, 1..8 = stage st
  const int n_groups = (p.n_tiles + 1) / 2;
  const int n_mine = n_groups > pl ? (n_groups - pl + kPipelines - 1) / kPipelines : 0;   // groups pl, pl + 8, ...
  if (n_mine == 0) return;                                 // (identical in both CTAs and in every role of the pipeline)

  const uint32_t bars = smem_base + kOffBars;
  const uint32_t bar_full = bars;                          // [kRing]
  const uint32_t bar_empty = bars + 8 * kRing;             // [kRing] count 2: MMA commit + reducers
  const uint32_t bar_peer = bars + 16 * kRing;             // [kRing] leader only: the peer's stage has landed
  const uint32_t bar_w_full = bars + 24 * kRing;           // resident weights landed
  const uint32_t bar_w_peer = bar_w_full + 8;              // leader only
  const uint32_t bar_acc_ready = bar_w_peer + 8;           // [2] accumulator complete (multicast commit); stages use [0]
  const uint32_t bar_acc_free = bar_acc_ready + 16;        // leader only, count 16: accumulator drained by both CTAs
  const uint32_t bar_a_ready = bar_acc_free + 8;           // [2] head, leader only, count 16: dG operands written
  const uint32_t bar_img_full = bar_a_ready + 16;          // count 8: dY_out image complete in shared memory
  const uint32_t bar_img_empty = bar_img_full + 8;         // count 4: read out of shared memory by the four store warps
  const uint32_t bar_done = bar_img_empty + 8;             // every MMA of this pair has completed (multicast commit)
  const uint32_t tmem_slot = bar_done + 8;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kRing; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 2);
      mbar_init(bar_peer + 8 * i, 1);
    }
    mbar_init(bar_w_full, 1);
    mbar_init(bar_w_peer, 1);
    mbar_init(bar_acc_ready, 1);
    mbar_init(bar_acc_ready + 8, 1);
    mbar_init(bar_acc_free, 16);
    mbar_init(bar_a_ready, 16);
    mbar_init(bar_a_ready + 8, 16);
    mbar_init(bar_img_full, 8);
    mbar_init(bar_img_empty, 4);
    mbar_init(bar_done, 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc2(tmem_slot, 512);
    tmem_relinquish2();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const uint64_t n_tiles64 = (uint64_t)p.n_tiles;
  const bool prof_on = p.prof != nullptr;
  const uint8_t* wimg = p.packed + kBwdImageOffset;
  auto link_base = [&](int k, int slot) -> uint8_t* { return p.links + ((size_t)(pl * kLinks + k) * kLinkSlots + slot) * kGroupBytes; };
  auto flag_ready = [&](int k, int slot) -> uint32_t* { return p.flags + ((size_t)(pl * kLinks + k) * kLinkSlots + slot) * kFlagStride; };
  auto flag_freed = [&](int k, int slot) -> uint32_t* {
    return p.flags + ((size_t)kPipelines * kLinks * kLinkSlots + (size_t)(pl * kLinks + k) * kLinkSlots + slot) * kFlagStride;
  };

  if (role == 0) {
    // ==================================================================================================================
    // HEAD: prologue on CUDA cores + the C0 dgrad stage, two ping-pong slots (groups t = slot, slot + 2, ...)
    // ==================================================================================================================
    if (warp < 4) {
      setmaxnreg_dec<kRegsOther>();
      if (warp == 0) {
        // resident weights: rows [128 rank, +128) of the two W_c0^T panels (dgrad stage 0 of mlp_layout.cuh)
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_w_full, 2 * kStageBytes);
          for (int pp = 0; pp < 2; ++pp)
            bulk_g2s_hint(smem_base + kOffW + pp * kStageBytes, wimg + (uint32_t)(bwd_first_panel(0) + pp) * kPanelBytes256 + rank * kStageBytes,
                          kStageBytes, bar_w_full, l2_evict_last());
        }
        __syncwarp();
        if (rank == 1) {   // relay: my weights have landed
          mbar_wait(bar_w_full, 0);
          if (elect_one()) mbar_arrive_cluster(mapa(bar_w_peer, 0));
          __syncwarp();
        }
      } else if (warp == 1 && rank == 0) {
        constexpr uint32_t idesc = make_idesc(256, 256, kF16, kF16, 0, 0);
        mbar_wait(bar_w_full, 0);
        mbar_wait_cluster(bar_w_peer, 0);
        uint32_t a_phase[2] = {0, 0};
        for (int t = 0; t < n_mine; ++t) {
          const int slot = t & 1;
          mbar_wait_cluster(bar_a_ready + 8 * slot, a_phase[slot]);
          a_phase[slot] ^= 1;
          tc_fence_after();
          if (elect_one()) {
            const uint32_t a_smem = smem_base + kHeadOffA + slot * (2 * kPanelBytes128);
#pragma unroll
            for (int pp = 0; pp < 2; ++pp) {
              const uint64_t da = make_smem_desc(a_smem + pp * kPanelBytes128, 16u, kAtomBytes);
              const uint64_t db = make_smem_desc(smem_base + kOffW + pp * kStageBytes, 16u, kAtomBytes);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) umma2(tmem_base + slot * 256, da + 2u * ks, db + 2u * ks, idesc, (pp | ks) != 0);
            }
            umma_commit2(bar_acc_ready + 8 * slot, 3);
          }
          __syncwarp();
        }
      }
    } else {
      setmaxnreg_inc<kRegsEpilogue>();
      const int ew = warp - 4;
      const int slot = ew >> 3;
      const int half = (ew >> 2) & 1;
      const int wq = warp & 3;
      const int row = wq * 32 + lane;
      const int tg = threadIdx.x - 128 - slot * 256;
      const uint32_t a_smem = smem_base + kHeadOffA + slot * (2 * kPanelBytes128);
      const uint32_t out_smem = smem_base + kHeadOffOut + slot * kActBytes;
      const uint32_t t_acc = tmem_base + slot * 256 + half * 128 + (static_cast<uint32_t>(wq * 32) << 16);
      const uint32_t bar_id = 1 + slot;
      const uint32_t row_off = (uint32_t)(row >> 3) * kAtomBytes + (uint32_t)(row & 7) * kPanelRowBytes;
      const uint32_t xr = (uint32_t)(row & 7) << 4;
      const uint32_t out_h = out_smem + 2 * half * kPanelBytes128 + row_off;
      const uint32_t a_ready_leader = mapa(bar_a_ready + 8 * slot, 0);
      uint32_t acc_phase = 0;
      long long h_acc = 0, h_freed = 0, h_store = 0;
      const long long h_begin = prof_on ? clock64() : 0;
      for (int t = slot; t < n_mine; t += 2) {
        const int group = pl + kPipelines * t;
        const int tile = group * 2 + (int)rank;
        const bool tile_ok = tile < p.n_tiles;
        const int64_t e = (int64_t)tile * kTile + row;
        const bool valid = tile_ok && e < p.n_evals;
        // ---- prologue (mlp_bwd.cu): dL/dg for this half's 64 colour-layer neurons, masked by the forward's g > 0 bits ----
        uint2 gm = make_uint2(0u, 0u);
        if (tile_ok)
          gm = __ldg(reinterpret_cast<const uint2*>(p.stash + stash_region_offset(kStashMask, n_tiles64) +
                                                    (uint64_t)tile * stash_region_tile_bytes(kStashMask) + 8 * (128 * 32) + row * 32 + half * 8));
        float dp0 = 0.f, dp1 = 0.f, dp2 = 0.f, dsr = 0.f;
        if (valid) {
          const float4 dd = __ldg(p.d_rgbsigma + e);
          const float4 o = __ldg(p.rgbsigma + e);
          dp0 = dd.x * o.x * (1.f - o.x);
          dp1 = dd.y * o.y * (1.f - o.y);
          dp2 = dd.z * o.z * (1.f - o.z);
          dsr = dd.w;
        }
        uint32_t outw[2][16];
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          const int c0 = 64 * half + 32 * ci;
          const uint32_t gbits = ci == 0 ? gm.x : gm.y;
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 w0 = __ldg(reinterpret_cast<const float4*>(p.params + L::kWC1 + c0) + q);
            const float4 w1 = __ldg(reinterpret_cast<const float4*>(p.params + L::kWC1 + 128 + c0) + q);
            const float4 w2 = __ldg(reinterpret_cast<const float4*>(p.params + L::kWC1 + 256 + c0) + q);
            const float d0 = dp0 * w0.x + dp1 * w1.x + dp2 * w2.x;
            const float d1 = dp0 * w0.y + dp1 * w1.y + dp2 * w2.y;
            const float d2 = dp0 * w0.z + dp1 * w1.z + dp2 * w2.z;
            const float d3 = dp0 * w0.w + dp1 * w1.w + dp2 * w2.w;
            const bool m0 = (gbits >> (2 * q)) & 1u, m1 = (gbits >> (16 + 2 * q)) & 1u;
            const bool m2 = (gbits >> (2 * q + 1)) & 1u, m3 = (gbits >> (16 + 2 * q + 1)) & 1u;
            outw[ci][2 * q] = pack_half2(m0 ? d0 : 0.f, m1 ? d1 : 0.f);
            outw[ci][2 * q + 1] = pack_half2(m2 ? d2 : 0.f, m3 ? d3 : 0.f);
          }
        }
        // the previous group's image stores of this slot (dG from a_smem, dF from out_smem) must have left shared memory
        if (tg == 0) bulk_wait_read<0>();
        named_bar_sync(bar_id, 256);
        {
          const uint32_t dpanel = a_smem + half * kPanelBytes128;
#pragma unroll
          for (int ci = 0; ci < 2; ++ci)
#pragma unroll
            for (int q = 0; q < 4; ++q)
              st_shared_v4(dpanel + panel_chunk_offset(row, 4 * ci + q), outw[ci][4 * q], outw[ci][4 * q + 1], outw[ci][4 * q + 2],
                           outw[ci][4 * q + 3]);
        }
        fence_proxy_async_smem();
        named_bar_sync(bar_id, 256);
        if (tg == 0 && tile_ok) {   // dG image for the residual weight-gradient kernel (colour layer 0)
          bulk_s2g_hint(p.gstash + grad_region_offset(kGradC0, n_tiles64) + (uint64_t)tile * grad_region_tile_bytes(kGradC0), a_smem,
                        2 * kPanelBytes128, l2_evict_first());
          bulk_commit();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(a_ready_leader);
        if (tile_ok) {   // head-gradient panel: cols 0..2 = dL/d(rgb pre-sigmoid), col 3 = dL/dsigma_raw, rest zero
          uint8_t* hd = p.gstash + grad_region_offset(kGradHead, n_tiles64) + (uint64_t)tile * grad_region_tile_bytes(kGradHead);
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            uint4 v = make_uint4(0, 0, 0, 0);
            if (ch == 0 && half == 0) {
              v.x = pack_half2(dp0, dp1);
              v.y = pack_half2(dp2, dsr);
            }
            *reinterpret_cast<uint4*>(hd + panel_chunk_offset(row, 4 * half + ch)) = v;
          }
        }
        // ---- dF = dG W_c0[:, :256] (no mask: f is linear) -> fp16 image -> link 0 ----
        PIPE_TIMED(h_acc, mbar_wait(bar_acc_ready + 8 * slot, acc_phase));
        acc_phase ^= 1;
        tc_fence_after();
        {
          const uint32_t mk[4] = {~0u, ~0u, ~0u, ~0u};
          pipe_drain_acc<false>(t_acc, mk, nullptr, 0.f, out_h, xr);
        }
        tc_fence_before();
        fence_proxy_async_smem();
        named_bar_sync(bar_id, 256);
        if (tg == 0) {
          const int ls = t % kLinkSlots, use = t / kLinkSlots;
          PIPE_TIMED(h_freed, spin_until(flag_freed(0, ls), 2u * (uint32_t)use));   // both consumer CTAs have released the slot's previous group
          bulk_s2g(link_base(0, ls) + rank * kActBytes, out_smem, kActBytes);
          bulk_commit();
          PIPE_TIMED(h_store, bulk_wait_all<0>());                      // writes complete (not only read) before the flag
          fence_proxy_async_all();
          __threadfence();
          red_release_gpu(flag_ready(0, ls), 1u);                       // one per CTA: consumers wait for 2 per group
        }
      }
      if (tg == 0) bulk_wait_all<0>();
      if (prof_on && tg == 0) {
        atomicAdd(p.prof + 13, (unsigned long long)(clock64() - h_begin));
        atomicAdd(p.prof + 14, (unsigned long long)h_freed);
        atomicAdd(p.prof + 15, (unsigned long long)h_store);
        atomicAdd(p.prof + 16, (unsigned long long)h_acc);
        atomicAdd(p.prof + 20, 1ull);
        atomicAdd(p.prof + 32 + 0, (unsigned long long)h_freed);
      }
    }
  } else {
    // ==================================================================================================================
    // STAGE st = role: dY_in -> dY_out (dgrad) and dW += dY_in^T H (wgrad), layer-stationary
    // ==================================================================================================================
    const int st = role;                         // 1 = F, 2..8 = hidden layers 7..1 (chain stage numbering of mlp_bwd.cu)
    const int k_in = st - 1;                     // input link
    const int h_region = kStashH0 + (8 - st);    // activations that fed this layer: h7, h6, ..., h0
    // Ring positions of one group (all 16 KB = one whole 128-row panel, ONE bulk copy each: the TMA unit of an SM retires one
    // 1-D bulk copy per ~259 cycles whatever its size up to 16 KB, measured with tools/l2_probe.py):
    //   0..3   A0..A3    this CTA's tile of dY_in, K panels 0..3                                   (dgrad operand, K-major)
    //   4, 5   Xa, Xb    tile 0 of the pair: dY_in panels 2 rank, 2 rank + 1  \  wgrad operands, MN-major, K = the 128 samples
    //   6, 7   Ya, Yb    tile 0: activation panels 2 rank, 2 rank + 1         /  of the tile; (Xa, Xb) and (Ya, Yb) are adjacent
    //   8..11            the same for tile 1                                       ring stages = one 128-column operand each
    if (warp < 4) {
      setmaxnreg_dec<kRegsOther>();
      if (warp != 1) {
        // ------------------------------------------------ loaders (warps 0, 2, 3) ------------------------------------------------
        const int wl = warp == 0 ? 0 : warp - 1;   // 0, 1, 2: in-group positions wl, wl + 3, wl + 6, wl + 9
        if (wl == 0) {
          if (elect_one()) {
            mbar_arrive_expect_tx(bar_w_full, 4 * kStageBytes);
            for (int pp = 0; pp < 4; ++pp)
              bulk_g2s_hint(smem_base + kOffW + pp * kStageBytes, wimg + (uint32_t)(bwd_first_panel(st) + pp) * kPanelBytes256 + rank * kStageBytes,
                            kStageBytes, bar_w_full, l2_evict_last());
          }
          __syncwarp();
        }
        const uint64_t pol_stream = l2_evict_first();
        const long long l_begin = prof_on ? clock64() : 0;
        long long l_flag = 0, l_empty = 0, l_fence = 0, l_issue = 0;
        for (int t = 0; t < n_mine; ++t) {
          const int group = pl + kPipelines * t;
          const int ls = t % kLinkSlots, use = t / kLinkSlots;
          if (elect_one()) {
            PIPE_TIMED(l_flag, spin_until(flag_ready(k_in, ls), 2u * (uint32_t)(use + 1)));
            PIPE_TIMED(l_fence, fence_proxy_async_all());   // the bulk loads below (async proxy) must observe the producer's data
          }
          __syncwarp();
          const uint8_t* lbase = link_base(k_in, ls);
          for (int i = wl; i < 12; i += 3) {
            const uint32_t pos = 12u * (uint32_t)t + (uint32_t)i;
            const uint32_t stage = pos % (uint32_t)kRing, phase = (pos / (uint32_t)kRing) & 1u;
            PIPE_TIMED(l_empty, mbar_wait(bar_empty + 8 * stage, phase ^ 1));
            const long long i0 = prof_on ? clock64() : 0;
            if (elect_one()) {
              mbar_arrive_expect_tx(bar_full + 8 * stage, kStageBytes);
              const uint32_t dst = smem_base + kOffRing + stage * kStageBytes;
              if (i < 4) {
                bulk_g2s(dst, lbase + rank * kActBytes + i * kPanelBytes128, kStageBytes, bar_full + 8 * stage);
              } else {
                const int q = (i - 4) >> 2, xy = ((i - 4) >> 1) & 1, j = i & 1;
                const uint32_t off = (uint32_t)(2 * rank + j) * kPanelBytes128;
                if (xy == 0) {
                  bulk_g2s(dst, lbase + q * kActBytes + off, kStageBytes, bar_full + 8 * stage);
                } else {
                  int tile_q = group * 2 + q;
                  if (tile_q >= p.n_tiles) tile_q = p.n_tiles - 1;   // (its dY is all zero: any finite activations will do)
                  bulk_g2s_hint(dst, p.stash + stash_region_offset(h_region, n_tiles64) + (uint64_t)tile_q * kActBytes + off, kStageBytes,
                                bar_full + 8 * stage, pol_stream);
                }
              }
            }
            __syncwarp();
            if (prof_on) l_issue += clock64() - i0;
          }
        }
        if (prof_on && lane == 0 && rank == 0 && wl == 0) {
          atomicAdd(p.prof + 0, (unsigned long long)l_flag);
          atomicAdd(p.prof + 1, (unsigned long long)l_empty);
          atomicAdd(p.prof + 21, (unsigned long long)l_fence);
          atomicAdd(p.prof + 22, (unsigned long long)(clock64() - l_begin));
          atomicAdd(p.prof + 23, (unsigned long long)l_issue);
          atomicAdd(p.prof + 32 + 3 * role + 0, (unsigned long long)l_flag);
        }
      } else {
        // ------------------------------------------------ MMA issuer (leader) / relay (peer) ------------------------------------------------
        const bool leader = rank == 0;
        constexpr uint32_t idesc_d = make_idesc(256, 256, kF16, kF16, 0, 0);
        constexpr uint32_t idesc_w = make_idesc(256, 256, kF16, kF16, 1, 1);
        const uint32_t acc = tmem_base, dw = tmem_base + 256;
        mbar_wait(bar_w_full, 0);
        if (leader) mbar_wait_cluster(bar_w_peer, 0);
        else {
          if (elect_one()) mbar_arrive_cluster(mapa(bar_w_peer, 0));
          __syncwarp();
        }
        uint32_t stage = 0, phase = 0, free_phase = 0;
        long long m_free = 0, m_full = 0, m_full_w = 0;
        bool in_wgrad = false;
        const long long m_begin = prof_on ? clock64() : 0;
        auto next_stage = [&]() {
          if (++stage == (uint32_t)kRing) {
            stage = 0;
            phase ^= 1;
          }
        };
        // the stage's operands have landed in BOTH CTAs (leader) / in this CTA, announced to the leader (peer)
        auto stage_ready = [&]() {
          const long long w0 = prof_on ? clock64() : 0;
          mbar_wait(bar_full + 8 * stage, phase);
          if (leader) {
            mbar_wait_cluster(bar_peer + 8 * stage, phase);
          } else {
            if (elect_one()) mbar_arrive_cluster(mapa(bar_peer + 8 * stage, 0));
            __syncwarp();
          }
          if (prof_on) (in_wgrad ? m_full_w : m_full) += clock64() - w0;
        };
        for (int t = 0; t < n_mine; ++t) {
          const int ls = t % kLinkSlots;
          if (leader && t > 0) {   // the accumulator of the previous group has been drained by both CTAs
            PIPE_TIMED(m_free, mbar_wait_cluster(bar_acc_free, free_phase));
            free_phase ^= 1;
          }
          in_wgrad = false;
          for (int pp = 0; pp < 4; ++pp) {
            stage_ready();
            if (leader) {
              tc_fence_after();
              if (elect_one()) {
                const uint64_t da = make_smem_desc(smem_base + kOffRing + stage * kStageBytes, 16u, kAtomBytes);
                const uint64_t db = make_smem_desc(smem_base + kOffW + pp * kStageBytes, 16u, kAtomBytes);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) umma2(acc, da + 2u * ks, db + 2u * ks, idesc_d, (pp | ks) != 0);
                umma_commit2(bar_empty + 8 * stage, 3);
                if (pp == 3) umma_commit2(bar_acc_ready, 3);
              }
              __syncwarp();
            }
            next_stage();
          }
          in_wgrad = true;
          for (int q = 0; q < 2; ++q) {
            uint32_t sidx[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {   // Xa, Xb, Ya, Yb
              stage_ready();
              sidx[i] = stage;
              next_stage();
            }
            if (leader) {
              tc_fence_after();
              if (elect_one()) {
                const uint32_t ax = smem_base + kOffRing + sidx[0] * kStageBytes, by = smem_base + kOffRing + sidx[2] * kStageBytes;
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)   // 8 x 16 samples; the two 64-column groups of an operand are one ring stage apart
                  umma2(dw, desc_mnmajor(ax, ks, kStageBytes), desc_mnmajor(by, ks, kStageBytes), idesc_w, (t | q | ks) != 0);
#pragma unroll
                for (int i = 0; i < 4; ++i) umma_commit2(bar_empty + 8 * sidx[i], 3);
              }
              __syncwarp();
            }
            if (q == 1) {   // every load from the input link slot has landed in this CTA: give the slot back to the producer
              if (elect_one()) red_relaxed_gpu(flag_freed(k_in, ls), 1u);
              __syncwarp();
            }
          }
        }
        if (leader) {
          if (elect_one()) umma_commit2(bar_done, 3);
          __syncwarp();
          if (prof_on && lane == 0) {
            atomicAdd(p.prof + 2, (unsigned long long)m_free);
            atomicAdd(p.prof + 3, (unsigned long long)m_full);
            atomicAdd(p.prof + 4, (unsigned long long)m_full_w);
            atomicAdd(p.prof + 5, (unsigned long long)(clock64() - m_begin));
            atomicAdd(p.prof + 19, 1ull);
            atomicAdd(p.prof + 32 + 3 * role + 1, (unsigned long long)(m_full + m_full_w));
          }
        }
      }
    } else if (warp < 12) {
      // ------------------------------------------------ epilogue: acc -> mask -> fp16 image, two 128-column phases ------------------------
      // The image buffer holds two panels (32 KB): phase ph converts accumulator columns [128 ph, +128) -- warp (quarter, hh) takes the
      // 64 columns of panel hh -- and hands them to the store warps, so a group is two image events.
      setmaxnreg_inc<kRegsEpilogue>();
      const int ew = warp - 4;
      const int hh = (ew >> 2) & 1;
      const int wq = warp & 3;
      const int row = wq * 32 + lane;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(wq * 32) << 16);
      const uint32_t row_off = (uint32_t)(row >> 3) * kAtomBytes + (uint32_t)(row & 7) * kPanelRowBytes;
      const uint32_t xr = (uint32_t)(row & 7) << 4;
      const uint32_t out_p = smem_base + kOffOut + hh * kPanelBytes128 + row_off;
      const uint32_t acc_free_leader = mapa(bar_acc_free, 0);
      const int mask_layer = 8 - st;
      uint32_t acc_phase = 0, ev = 0;   // ev = image events handed over so far
      long long e_acc = 0, e_img = 0;
      const long long e_begin = prof_on ? clock64() : 0;
      const bool e_prof = prof_on && rank == 0 && warp == 4 && lane == 0;
      for (int t = 0; t < n_mine; ++t) {
        const int group = pl + kPipelines * t;
        const int tile = group * 2 + (int)rank;
        const bool tile_ok = tile < p.n_tiles;
        const int64_t e = (int64_t)tile * kTile + row;
        // ReLU bits of the row's 256 columns: word w = columns [32 w, 32 w + 32) (tc.cuh relu_mask_bit order); this warp needs words
        // 4 ph + 2 hh, + 1 in phase ph
        uint2 mph[2] = {make_uint2(~0u, ~0u), make_uint2(~0u, ~0u)};
        if (tile_ok) {
          const uint8_t* mp = p.stash + stash_region_offset(kStashMask, n_tiles64) + (uint64_t)tile * stash_region_tile_bytes(kStashMask) +
                              mask_layer * (128 * 32) + row * 32 + 8 * hh;
          mph[0] = __ldg(reinterpret_cast<const uint2*>(mp));
          mph[1] = __ldg(reinterpret_cast<const uint2*>(mp + 16));
        }
        float dsr = 0.f;
        if (st == 1 && tile_ok && e < p.n_evals) dsr = __ldg(p.d_rgbsigma + e).w;
        PIPE_TIMED(e_acc, mbar_wait(bar_acc_ready, acc_phase));
        acc_phase ^= 1;
        tc_fence_after();
#pragma unroll 1
        for (int ph = 0; ph < 2; ++ph) {
          const int col0 = 128 * ph + 64 * hh;                       // first accumulator column of this warp in this phase
          const float* wsp = p.params + L::kWS + col0;
          const uint32_t w0m = ph == 0 ? mph[0].x : mph[1].x, w1m = ph == 0 ? mph[0].y : mph[1].y;
          uint32_t va[16], vb[16];
          tmem_ld16(t_row + col0, va);
          if (ev > 0) PIPE_TIMED(e_img, mbar_wait(bar_img_empty, (ev - 1) & 1u));   // the previous image has left the buffer
          tmem_ld_wait16(va);
          tmem_ld16(t_row + col0 + 16, vb);
          if (st == 1) pipe_dgrad16<true>(va, w0m, 0, wsp, dsr, out_p + (0u ^ xr), out_p + (16u ^ xr));
          else pipe_dgrad16<false>(va, w0m, 0, wsp, dsr, out_p + (0u ^ xr), out_p + (16u ^ xr));
          tmem_ld_wait16(vb);
          tmem_ld16(t_row + col0 + 32, va);
          if (st == 1) pipe_dgrad16<true>(vb, w0m, 8, wsp + 16, dsr, out_p + (32u ^ xr), out_p + (48u ^ xr));
          else pipe_dgrad16<false>(vb, w0m, 8, wsp + 16, dsr, out_p + (32u ^ xr), out_p + (48u ^ xr));
          tmem_ld_wait16(va);
          tmem_ld16(t_row + col0 + 48, vb);
          if (st == 1) pipe_dgrad16<true>(va, w1m, 0, wsp + 32, dsr, out_p + (64u ^ xr), out_p + (80u ^ xr));
          else pipe_dgrad16<false>(va, w1m, 0, wsp + 32, dsr, out_p + (64u ^ xr), out_p + (80u ^ xr));
          tmem_ld_wait16(vb);
          if (ph == 1) {   // the accumulator has been read completely: the next group's dgrad MMAs may overwrite it
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(acc_free_leader);
          }
          if (st == 1) pipe_dgrad16<true>(vb, w1m, 8, wsp + 48, dsr, out_p + (96u ^ xr), out_p + (112u ^ xr));
          else pipe_dgrad16<false>(vb, w1m, 8, wsp + 48, dsr, out_p + (96u ^ xr), out_p + (112u ^ xr));
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_img_full);
          ++ev;
        }
      }
      if (e_prof) {
        atomicAdd(p.prof + 6, (unsigned long long)e_acc);
        atomicAdd(p.prof + 7, (unsigned long long)e_img);
        atomicAdd(p.prof + 8, (unsigned long long)(clock64() - e_begin));
      }
      // ---- flush this CTA's half of dW (rows 128 rank .. +128 = output neurons, 256 columns = input features) ----
      mbar_wait(bar_done, 0);
      tc_fence_after();
      {
        const int layer = 8 - st + 1;   // st = 1 -> feature layer, st = 2..8 -> hidden layers 7..1
        const int64_t w_off = st == 1 ? L::kWF : L::hidden_w(layer);
        const int ld = st == 1 ? 256 : L::hidden_in(layer);
        float* wrow = p.grads + w_off + (int64_t)(128 * rank + row) * ld + 128 * hh;
        const uint32_t t_dw = t_row + 256 + hh * 128;
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(t_dw + c0, v);
          tmem_ld_wait32(v);
#pragma unroll
          for (int j = 0; j < 32; ++j) atomicAdd(wrow + c0 + j, __uint_as_float(v[j]) * p.inv_scale);
        }
      }
      tc_fence_before();
    } else if (warp < 16) {
      // ------------------------------------------------ reducers: bias (and density-head) gradients ------------------------------------------------
      // Every ring position is visited in the loaders' order; the X stages (dY_in: 128 samples x 64 of this CTA's columns) feed
      // the column sums, and in stage F the Y stages (h7) feed dL/dw_sigma.  A consumer arrives on `empty` only after the stage's
      // `full` phase: the barrier counts two arrivals per use (MMA commit + this group) and must never see two of one kind.
      const int tr = threadIdx.x - 12 * 32;      // 0..127
      const int cg = tr & 7;                     // 16-byte chunk = columns [8 cg, 8 cg + 8) of the panel's 64
      const int rg = tr >> 3;                    // rows [8 rg, 8 rg + 8) of the 128
      // (one LDS.128 per row: a first version with 4-byte loads took ~700 cycles per stage -- ~1,000 with the density head -- and,
      //  because `empty` needs this group's arrival, throttled the whole pipeline to stage F's reducers)
      float sb[2][8], sd[2][8], dsum = 0.f;
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int e = 0; e < 8; ++e) sb[j][e] = sd[j][e] = 0.f;
      float* dsig = reinterpret_cast<float*>(smem_raw + kOffDsig);
      uint32_t stage = 0, phase = 0;
      auto next_stage = [&]() {
        if (++stage == (uint32_t)kRing) {
          stage = 0;
          phase ^= 1;
        }
      };
      auto load8 = [&](uint32_t addr, float (&f)[8]) {
        uint32_t w0, w1, w2, w3;
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3) : "r"(addr));
        const float2 a0 = __half22float2(*reinterpret_cast<__half2*>(&w0)), a1 = __half22float2(*reinterpret_cast<__half2*>(&w1));
        const float2 a2 = __half22float2(*reinterpret_cast<__half2*>(&w2)), a3 = __half22float2(*reinterpret_cast<__half2*>(&w3));
        f[0] = a0.x; f[1] = a0.y; f[2] = a1.x; f[3] = a1.y; f[4] = a2.x; f[5] = a2.y; f[6] = a3.x; f[7] = a3.y;
      };
      // The ring (128 KB) cannot cover HBM latency at this operand rate (192 KB per group): measured, every group paid two HBM
      // round trips in series.  The activation panels of the groups ahead are therefore pulled into L2 here (64 KB per group and
      // CTA, one 128-byte line per prefetch), so that every ring load is an L2 hit.
      constexpr int kPrefetchAhead = 3;
      auto prefetch_group = [&](int tt) {
        if (tt >= n_mine) return;
        const int g2 = pl + kPipelines * tt;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          int tile_q = g2 * 2 + q;
          if (tile_q >= p.n_tiles) tile_q = p.n_tiles - 1;
          const uint8_t* hb = p.stash + stash_region_offset(h_region, n_tiles64) + (uint64_t)tile_q * kActBytes + (uint32_t)(2 * rank) * kPanelBytes128;
#pragma unroll
          for (int l = 0; l < 2; ++l) asm volatile("prefetch.global.L2 [%0];" ::"l"(hb + (size_t)(tr + 128 * l) * 128));   // 2 panels = 256 lines
        }
      };
      for (int tt = 0; tt < kPrefetchAhead; ++tt) prefetch_group(tt);
      for (int t = 0; t < n_mine; ++t) {
        const int group = pl + kPipelines * t;
        prefetch_group(t + kPrefetchAhead);
        for (int i = 0; i < 12; ++i) {
          mbar_wait(bar_full + 8 * stage, phase);
          if (i >= 4) {
            const int q = (i - 4) >> 2, xy = ((i - 4) >> 1) & 1, j = i & 1;
            const uint32_t base = smem_base + kOffRing + stage * kStageBytes;
            if (xy == 0) {
#pragma unroll
              for (int r = 0; r < 8; ++r) {
                float f[8];
                load8(base + panel_chunk_offset(8 * rg + r, cg), f);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  if (j == 0) sb[0][e] += f[e]; else sb[1][e] += f[e];
                }
              }
              if (st == 1 && j == 0) {   // dsigma_raw of the tile's 128 samples (zero beyond the batch), used by the Y stages below
                const int64_t em = (int64_t)(group * 2 + q) * kTile + tr;
                dsig[tr] = em < p.n_evals ? __ldg(p.d_rgbsigma + em).w : 0.f;
              }
            } else if (st == 1) {
#pragma unroll
              for (int r = 0; r < 8; ++r) {
                float f[8];
                load8(base + panel_chunk_offset(8 * rg + r, cg), f);
                const float ds = dsig[8 * rg + r];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  if (j == 0) sd[0][e] = fmaf(ds, f[e], sd[0][e]); else sd[1][e] = fmaf(ds, f[e], sd[1][e]);
                }
                if (cg == 0 && j == 0) dsum += ds;
              }
            }
          }
          named_bar_sync(3, 128);
          if (tr == 0) mbar_arrive(bar_empty + 8 * stage);
          next_stage();
        }
      }
      {
        const int layer = 8 - st + 1;
        const int64_t b_off = st == 1 ? L::kBF : L::hidden_b(layer);
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            atomicAdd(p.grads + b_off + 128 * rank + 64 * j + 8 * cg + e, sb[j][e] * p.inv_scale);
            if (st == 1) atomicAdd(p.grads + L::kWS + 128 * rank + 64 * j + 8 * cg + e, sd[j][e] * p.inv_scale);
          }
        if (st == 1 && cg == 0 && rank == 0) atomicAdd(p.grads + L::kBS, dsum * p.inv_scale);   // (both CTAs see all 256 samples)
      }
    } else {
      // ------------------------------------------------ store warps: dY_out image -> next link (and HBM where the residual kernel needs it) -------
      // Four warps through the LSU (the TMA unit of a stage CTA only carries loads): per image event (two panels) warp sw moves the
      // 8 KB half (sw & 1) of panel (sw >> 1).  The buffer is handed back as soon as it has been READ into registers; after the
      // second event of a group the four warps meet and ONE of them (rotating) publishes the group with a gpu-scope release, whose
      // fence (it waits for 64 KB of stores to drain at the SM's 27-32 B/clk store path) then stalls each warp only every 4th group.
      const int sw = warp - 16;
      const uint8_t* src = smem_raw + kOffOut + (sw >> 1) * kPanelBytes128 + (sw & 1) * kHalfPanel;
      const int gregion = st == 3 ? kGradL7 + 2 : (st == 8 ? kGradL0 : -1);   // dY5 (layer-5 encoding columns) / dY0 (layer 0)
      long long s_img = 0, s_freed = 0, s_copy = 0, s_fence = 0;
      const long long s_begin = prof_on ? clock64() : 0;
      uint32_t ev = 0;
      for (int t = 0; t < n_mine; ++t) {
        const int group = pl + kPipelines * t;
        const int tile = group * 2 + (int)rank;
        const bool tile_ok = tile < p.n_tiles;
        const int ls = t % kLinkSlots, use = t / kLinkSlots;
        for (int ph = 0; ph < 2; ++ph, ++ev) {
          PIPE_TIMED(s_img, mbar_wait(bar_img_full, ev & 1u));
          const long long c0 = prof_on ? clock64() : 0;
          uint4 v[16];   // 32 lanes x 16 x 16 B = 8 KB
          const uint4* sp = reinterpret_cast<const uint4*>(src);
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = sp[i * 32 + lane];
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_img_empty);
          const size_t img_off = (size_t)(2 * ph + (sw >> 1)) * kPanelBytes128 + (size_t)(sw & 1) * kHalfPanel;
          if (st < 8) {
            if (ph == 0) {
              if (lane == 0) PIPE_TIMED(s_freed, spin_until(flag_freed(st, ls), 2u * (uint32_t)use));
              __syncwarp();
            }
            uint4* dst = reinterpret_cast<uint4*>(link_base(st, ls) + rank * kActBytes + img_off);
#pragma unroll
            for (int i = 0; i < 16; ++i) dst[i * 32 + lane] = v[i];
          }
          if (gregion >= 0 && tile_ok) {
            uint4* dst = reinterpret_cast<uint4*>(p.gstash + grad_region_offset(gregion, n_tiles64) + (uint64_t)tile * kActBytes + img_off);
#pragma unroll
            for (int i = 0; i < 16; ++i) __stcs(dst + i * 32 + lane, v[i]);
          }
          if (prof_on) s_copy += clock64() - c0;
        }
        if (st < 8) {
          const long long f0 = prof_on ? clock64() : 0;
          named_bar_sync(4, 128);                       // all four warps' stores of this group are ordered before ...
          if (sw == (t & 3) && lane == 0) red_release_gpu(flag_ready(st, ls), 1u);   // ... the (cumulative) release of one lane
          if (prof_on) s_fence += clock64() - f0;
        }
      }
      if (prof_on && lane == 0 && rank == 0 && sw == 0) {
        atomicAdd(p.prof + 9, (unsigned long long)s_img);
        atomicAdd(p.prof + 10, (unsigned long long)s_freed);
        atomicAdd(p.prof + 11, (unsigned long long)(s_copy - s_freed));
        atomicAdd(p.prof + 12, (unsigned long long)(clock64() - s_begin));
        atomicAdd(p.prof + 24, (unsigned long long)s_fence);
        atomicAdd(p.prof + 32 + 3 * role + 2, (unsigned long long)(s_copy - s_freed + s_fence));
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc2(tmem_base, 512);
}

int launch_wgrad_residual(float* grads, const uint8_t* stash, const uint8_t* gstash, int n_tiles, float inv_scale, cudaStream_t stream);

}  // namespace nerf

extern "C" size_t nerf_mlp_backward_pipe_workspace_bytes(void) { return nerf::pipe::kLinkBytes + nerf::pipe::kFlagBytes; }

// Fused backward: `workspace` = gradient stash (nerf_mlp_backward_workspace_bytes) followed by the pipeline's links and flags.
extern "C" int nerf_mlp_backward_pipe(float* grads, const float* d_rgbsigma, const float* rgbsigma, const void* stash, void* workspace,
                                      const void* packed, const float* params, int n_rays, int n_samples, float grad_scale, void* stream) {
  using namespace nerf;
  if (n_rays <= 0) return 0;
  NERF_CHECK_ARG(grads && d_rgbsigma && rgbsigma && stash && workspace && packed && params, "mlp_backward_pipe: null pointer");
  NERF_CHECK_ARG(grad_scale > 0.f, "mlp_backward_pipe: grad_scale must be positive");
  const int64_t n_evals = (int64_t)n_rays * n_samples;
  NERF_CHECK_ARG(n_evals < (int64_t(1) << 31) - kTile, "mlp_backward_pipe: n_rays*n_samples must be < 2^31 per call");
  NERF_CHECK_ARG(((reinterpret_cast<uintptr_t>(stash) | reinterpret_cast<uintptr_t>(workspace) | reinterpret_cast<uintptr_t>(packed)) & 127) == 0,
                 "mlp_backward_pipe: stash, workspace and packed must be 128-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PipeParams p;
  p.grads = grads;
  p.d_rgbsigma = reinterpret_cast<const float4*>(d_rgbsigma);
  p.rgbsigma = reinterpret_cast<const float4*>(rgbsigma);
  p.stash = static_cast<const uint8_t*>(stash);
  p.gstash = static_cast<uint8_t*>(workspace);
  p.n_evals = n_evals;
  p.n_tiles = (int)((n_evals + kTile - 1) / kTile);
  const size_t gbytes = (size_t)(grad_tile_bytes_total() * (uint64_t)p.n_tiles);
  p.links = p.gstash + ((gbytes + 1023) & ~size_t(1023));
  p.flags = reinterpret_cast<uint32_t*>(p.links + pipe::kLinkBytes);
  p.packed = static_cast<const uint8_t*>(packed);
  p.params = params;
  p.inv_scale = 1.f / grad_scale;
  p.prof = reinterpret_cast<unsigned long long*>(timing_buffer());
  // a pipeline whose consumer waits for a producer needs every pair resident at once: 74 clusters on 148 SMs
  static int clusters_ok[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!clusters_ok[dev & 63]) {
    cudaError_t e1 = cudaFuncSetAttribute(mlp_bwd_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pipe::kSmemBytes);
    NERF_CHECK_ARG(e1 == cudaSuccess, "mlp_backward_pipe: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs);
    cfg.blockDim = dim3(pipe::kThreads);
    cfg.dynamicSmemBytes = pipe::kSmemBytes;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    int max_clusters = 0;
    cudaError_t e2 = cudaOccupancyMaxActiveClusters(&max_clusters, mlp_bwd_pipe_kernel, &cfg);
    NERF_CHECK_ARG(e2 == cudaSuccess && max_clusters >= pipe::kPipelines * pipe::kRoles,
                   "mlp_backward_pipe: the device cannot keep %d CTA pairs resident at once (%d): %s", pipe::kPipelines * pipe::kRoles, max_clusters,
                   cudaGetErrorString(e2));
    clusters_ok[dev & 63] = 1;
  }
  cudaError_t em = cudaMemsetAsync(p.flags, 0, pipe::kFlagBytes, s);
  NERF_CHECK_ARG(em == cudaSuccess, "mlp_backward_pipe: cudaMemsetAsync failed: %s", cudaGetErrorString(em));
  mlp_bwd_pipe_kernel<<<kNumSMs, pipe::kThreads, pipe::kSmemBytes, s>>>(p);
  NERF_CHECK_LAUNCH("mlp_bwd_pipe_kernel");
  return launch_wgrad_residual(grads, p.stash, p.gstash, p.n_tiles, p.inv_scale, s);
}
