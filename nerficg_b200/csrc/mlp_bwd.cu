// mlp_bwd.cu -- K4a: the data-gradient ("dgrad") chain of the NeRF MLP as one fused, persistent,
// warp-specialised tcgen05 kernel on a CTA pair (chain.cuh), with the transposed weight images and a 6-stage ring.
//
// Per 128-sample tile, starting from dL/d(r,g,b,sigma_raw) (K6 output, loss-scaled):
//   prologue : sigmoid' and W_c1^T on CUDA cores -> dL/dg (masked by the forward's g > 0 bits)  [128 wide]
//   stage 0  : dL/df   = dG  * W_c0[:, :256]
//   stage 1  : dL/dh7  = (dF * W_f + dsigma_raw (x) w_sigma) . [h7 > 0]
//   stage 2+j: dL/dh_{6-j} = (dY_{7-j} * W_{7-j}[:, :256]) . [h_{6-j} > 0],  j = 0..6
// Every dY image (fp16, 128B-swizzled panels) is bulk-stored to the gradient stash for the
// layer-major weight-gradient kernel (mlp_wgrad.cu).  Gradients are fp16 with a static loss scale:
// mixed bf16 x fp16 UMMA operands are illegal on sm_100a and the stashed activations are fp16.
#include "chain.cuh"
#include "../../include/nerf_b200.h"

namespace nerf {
using namespace tc;

namespace bwd {
constexpr int kRingStages = 6;  // ring stages: this CTA's 128-column half of one W^T panel
constexpr uint32_t kSlotBytes = kActBytes;
constexpr uint32_t kOffRing = 2 * kSlotBytes;
constexpr uint32_t kOffBars = kOffRing + kRingStages * chain::kRingStageBytes;
constexpr uint32_t kSmemBytes = kOffBars + 256 + 1024;  // + 1 KB to align the dynamic window up to 1024 bytes
static_assert(kSmemBytes <= 232448, "shared memory budget exceeded");

struct Stages {
  static constexpr int kStages = kBwdStages, kRingStages = bwd::kRingStages;
  static constexpr int kProfBase = 10;  // stall-counter slots 10..19
  __device__ static constexpr int panels(int st) { return bwd_panels(st); }
  __device__ static constexpr bool shared(int) { return true; }  // every dgrad stage fits the ring
};
}  // namespace bwd

struct BwdParams {
  const float4* d_rgbsigma;
  const float4* rgbsigma;
  const uint8_t* stash;
  uint8_t* gstash;
  const uint8_t* packed;
  const float* params;
  int64_t n_evals;
  int n_tiles;
  unsigned long long* prof;  // optional stall counters (chain.cuh), slots 10..21 and 25
};

// 16 columns of a dgrad epilogue: t = acc (+ dsigma_raw * w_sigma), masked by the forward ReLU bits of half2 words
// qbase..qbase+7 of the enclosing 32-column chunk (tc.cuh relu_mask_bit layout) -> fp16 pairs -> two 16-byte chunks
// of the swizzled A operand of the next stage at dst0 / dst1.
template <bool kSig>
__device__ __forceinline__ void dgrad16(const uint32_t (&v)[16], uint32_t m, int qbase, const float* __restrict__ ws, float dsr,
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

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(chain::kThreads, 1) mlp_dgrad_kernel(const BwdParams p) {
  using namespace bwd;
  using L = ParamLayout;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const chain::Bars bars(smem_base + kOffBars, kRingStages, false);
  const uint32_t rank = cluster_ctarank();  // 0 = leader
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tmem_base = chain::setup(bars, warp);
  const chain::Schedule sch(p.n_tiles);
  const uint8_t* wimg = p.packed + kBwdImageOffset;

  // (the stall counters stay behind this run-time flag here: an instantiation without them -- what the forward does --
  // made THIS kernel 11 % slower, 0.917 -> 1.020 ms, a register-allocation effect measured in round 2)
  const bool prof_on = p.prof != nullptr;
  if (warp < 4) {
    setmaxnreg_dec<chain::kRegsOther>();
    if (warp == 0) {
      // rows [128 * rank, +128) (output columns of dX) of every W^T panel
      chain::producer<Stages>(sch, bars, smem_base + kOffRing, prof_on, p.prof, [&](int st, int pp) {
        return chain::Panel{wimg + (uint32_t)(bwd_first_panel(st) + pp) * kPanelBytes256 + rank * chain::kRingStageBytes,
                            chain::kRingStageBytes};
      });
    } else if (warp == 1 && rank == 0) {
      constexpr uint32_t idesc = make_idesc(256, 256, kF16, kF16, 0, 0);
      chain::issuer<Stages>(sch, bars, smem_base + kOffRing, tmem_base, prof_on, p.prof,
                            [&](int, int slot, int pp, uint32_t d_tmem, uint64_t db) {
        const uint64_t da = make_smem_desc(smem_base + slot * kSlotBytes + pp * kPanelBytes128, 16u, kAtomBytes);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) umma2(d_tmem, da + 2u * ks, db + 2u * ks, idesc, (pp | ks) != 0);
      });
    } else if (warp == 1) {
      chain::relay<Stages>(sch, bars);
    }
  } else {
    setmaxnreg_inc<chain::kRegsEpilogue>();
    const chain::Epilogue epi(warp, lane, smem_base, kSlotBytes, tmem_base, bars);
    const int slot = epi.slot, half = epi.half, row = epi.row, tg = epi.tg;
    const uint32_t act = epi.act, xr = epi.xr;
    const uint32_t t_acc = epi.t_slot + 128 * half;
    uint32_t acc_phase = 0;
    const uint64_t n_tiles64 = (uint64_t)p.n_tiles;
    const bool prof = prof_on && tg == 0 && slot == 0;
    long long t_accw = 0, t_drain = 0, t_pro = 0, t_pro_compute = 0, t_pro_drain = 0, t_maskw = 0;
    const long long t_begin = prof ? clock64() : 0;

    for (int it = 0; it < sch.n_iters; ++it) {
      if (!sch.active(it, slot)) break;
      const int tile = sch.tile(it, slot, rank);
      const bool tile_ok = tile < p.n_tiles;
      const int64_t e = (int64_t)tile * kTile + row;
      const bool valid = tile_ok && e < p.n_evals;

      auto gstash_store = [&](int region, uint32_t src, uint32_t bytes) {
        epi.image_store([&] { return p.gstash + grad_region_offset(region, n_tiles64) + (uint64_t)tile * grad_region_tile_bytes(region); },
                        src, bytes, tile_ok);
      };
      const uint8_t* mask_base = p.stash + stash_region_offset(kStashMask, n_tiles64) +
                                 (uint64_t)tile * stash_region_tile_bytes(kStashMask) + row * 32 + half * 16;

      // ---------------- prologue ----------------
      const long long t_tile = prof ? clock64() : 0;
      // ReLU bits of g (this half's 64 neurons; stash mask slot 8, written by the forward's stage 9)
      uint2 gm = make_uint2(0u, 0u);
      if (tile_ok) gm = __ldg(reinterpret_cast<const uint2*>(mask_base + 8 * (128 * 32) - half * 8));
      float dp0 = 0.f, dp1 = 0.f, dp2 = 0.f, dsr = 0.f;
      if (valid) {
        const float4 dd = __ldg(p.d_rgbsigma + e);
        const float4 o = __ldg(p.rgbsigma + e);
        dp0 = dd.x * o.x * (1.f - o.x);
        dp1 = dd.y * o.y * (1.f - o.y);
        dp2 = dd.z * o.z * (1.f - o.z);
        dsr = dd.w;
      }
      // dL/dg for this half's 64 of the 128 colour-layer neurons -> panel `half` (masked by g > 0).  Everything is computed
      // into registers first: the previous tile's last image store (issued moments ago) still reads act, and waiting for
      // it up front put a full store drain plus the global-load latencies on every tile's critical path.
      uint32_t outw[2][16];
#pragma unroll
      for (int ci = 0; ci < 2; ++ci) {
        const int c0 = 64 * half + 32 * ci;
        const uint32_t gbits = ci == 0 ? gm.x : gm.y;
#pragma unroll
        for (int q = 0; q < 8; ++q) {  // columns 4q..4q+3 of the chunk: half2 words 2q, 2q+1 -> bits (2q, 16+2q), (2q+1, 16+2q+1)
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
      const long long t_mid = prof ? clock64() : 0;
      epi.image_drain(prof, t_drain);  // previous tile's D0 store still reads act
      if (prof) {
        t_pro_compute += t_mid - t_tile;
        t_pro_drain += clock64() - t_mid;
      }
      {
        const uint32_t dpanel = act + half * kPanelBytes128;
#pragma unroll
        for (int ci = 0; ci < 2; ++ci)
#pragma unroll
          for (int q = 0; q < 4; ++q)
            st_shared_v4(dpanel + panel_chunk_offset(row, 4 * ci + q), outw[ci][4 * q], outw[ci][4 * q + 1], outw[ci][4 * q + 2],
                         outw[ci][4 * q + 3]);
      }
      gstash_store(kGradC0, act, 2 * kPanelBytes128);
      epi.hand_off();
      if (prof) t_pro += clock64() - t_tile;
      // (off the critical path: under 4.3 TB/s of stash stores a plain global store can stall its warp for a long time)
      if (tile_ok) {  // head-gradient panel: cols 0..2 = dL/d(rgb pre-sigmoid), col 3 = dL/dsigma_raw, rest zero
        uint8_t* hd = p.gstash + grad_region_offset(kGradHead, n_tiles64) + (uint64_t)tile * grad_region_tile_bytes(kGradHead);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {  // each half of the row writes its four 16-byte chunks
          uint4 v = make_uint4(0, 0, 0, 0);
          if (ch == 0 && half == 0) {
            v.x = pack_half2(dp0, dp1);
            v.y = pack_half2(dp2, dsr);
          }
          *reinterpret_cast<uint4*>(hd + panel_chunk_offset(row, 4 * half + ch)) = v;
        }
      }
      // Pulls the next tile's prologue inputs (upstream gradients, outputs, g bits) into L2.  Called two stages before the
      // end of this tile's chain: issued right after the prologue (a whole tile = 35 us ahead) the lines were evicted
      // again before their use -- the 126 MB L2 turns over every ~27 us under this kernel's 4.3 TB/s of stores -- and the
      // prologue spent 7.4 K cycles per tile waiting for HBM.
      auto prefetch_next_tile = [&]() {
        if (it + 1 < sch.n_iters && sch.active(it + 1, slot)) {
          const int next = sch.tile(it + 1, slot, rank);
          if (next < p.n_tiles) {
            const int64_t en = (int64_t)next * kTile + row;
            if (half == 0 && en < p.n_evals) {
              asm volatile("prefetch.global.L2 [%0];" ::"l"(p.d_rgbsigma + en));
              asm volatile("prefetch.global.L2 [%0];" ::"l"(p.rgbsigma + en));
            }
            if (tg < 32) {  // the next tile's g bits (4 KB)
              const uint8_t* gn = p.stash + stash_region_offset(kStashMask, n_tiles64) + (uint64_t)next * stash_region_tile_bytes(kStashMask) +
                                  8 * (128 * 32) + tg * 128;
              asm volatile("prefetch.global.L2 [%0];" ::"l"(gn));
            }
          }
        }
      };

      // ---------------- chain stages ----------------
#pragma unroll 1
      for (int st = 0; st < kBwdStages; ++st) {
        // stage st produces the gradient w.r.t. the output of: st==0 -> f ; st>=1 -> hidden layer (8 - st)
        const int mask_layer = 8 - st;  // valid for st >= 1
        if (st == kBwdStages - 3) prefetch_next_tile();
        uint4 mk4 = make_uint4(~0u, ~0u, ~0u, ~0u);
        if (st >= 1 && tile_ok)  // ReLU masks of this half of the row (4 words), in flight while the MMAs still run
          mk4 = __ldg(reinterpret_cast<const uint4*>(mask_base + mask_layer * (128 * 32)));
        NERF_TIMED(prof, t_accw, mbar_wait(bars.acc_ready + 8 * slot, acc_phase));
        acc_phase ^= 1;
        tc_fence_after();
        epi.image_drain(prof, t_drain);  // previous image store still reads act
        if (prof) {   // how long the mask words are still in flight once the accumulator is ready
          const long long t0 = clock64();
          asm volatile("mov.b32 %0, %0;" : "+r"(mk4.x));
          t_maskw += clock64() - t0;
        }
        const uint32_t mk[4] = {mk4.x, mk4.y, mk4.z, mk4.w};
        // software pipeline over eight 16-column sub-chunks: the TMEM load of sub-chunk s+1 is in flight while s is processed
        auto run = [&](auto sig_tag) {
          constexpr bool kSig = decltype(sig_tag)::value;  // dL/dh7 also receives dsigma_raw * w_sigma
          const float* wsp = p.params + L::kWS + 128 * half;
          uint32_t va[16], vb[16];
          tmem_ld16(t_acc, va);
#pragma unroll
          for (int s = 0; s < 8; s += 2) {
            const uint32_t pbase = epi.act_h + (uint32_t)(s >> 2) * kPanelBytes128;
            const uint32_t c0 = (uint32_t)(s & 3) * 32u;  // byte offset of sub-chunk s in the (unswizzled) panel row
            tmem_ld_wait16(va);
            tmem_ld16(t_acc + 16 * (s + 1), vb);
            dgrad16<kSig>(va, mk[s >> 1], 0, wsp + 16 * s, dsr, pbase + (c0 ^ xr), pbase + ((c0 + 16u) ^ xr));
            tmem_ld_wait16(vb);
            if (s + 2 < 8) tmem_ld16(t_acc + 16 * (s + 2), va);
            dgrad16<kSig>(vb, mk[s >> 1], 8, wsp + 16 * (s + 1), dsr, pbase + ((c0 + 32u) ^ xr), pbase + ((c0 + 48u) ^ xr));
          }
        };
        if (st == 1) run(chain::BoolTag<true>{}); else run(chain::BoolTag<false>{});
        // operands are handed to the MMA issuer AFTER the slot's warps meet for the image store: the forward's early hand-off
        // measured no faster here (dgrad 0.899 -> 0.900 ms, profiles/r02_store_path_variants.txt)
        gstash_store(kGradF + st, act, kActBytes);  // regions: F, L7, L6, ..., L0
        if (st < kBwdStages - 1) {
          epi.hand_off();
        } else {
          tc_fence_before();  // accumulator drained; released by the next tile's prologue arrive
        }
      }
    }
    if (tg == 0) bulk_wait_all<0>();
    if (prof) {
      chain::epilogue_counters<Stages>(p.prof, t_accw, t_begin, t_drain, t_pro);
      atomicAdd(p.prof + 20, (unsigned long long)t_pro_compute);  // prologue: loads + dL/dg arithmetic
      atomicAdd(p.prof + 21, (unsigned long long)t_pro_drain);    // prologue: wait for the previous tile's last image store
      atomicAdd(p.prof + 25, (unsigned long long)t_maskw);
    }
  }
  chain::teardown(tmem_base, warp);
}

int launch_wgrad(float* grads, const uint8_t* stash, const uint8_t* gstash, int n_tiles, float inv_scale, cudaStream_t stream);

}  // namespace nerf

extern "C" size_t nerf_mlp_backward_workspace_bytes(int64_t n_samples) {
  const uint64_t n_tiles = (uint64_t)((n_samples + nerf::kTile - 1) / nerf::kTile);
  return (size_t)(nerf::grad_tile_bytes_total() * n_tiles);
}

static int run_backward(float* grads, const float* d_rgbsigma, const float* rgbsigma, const void* stash, void* workspace,
                        const void* packed, const float* params, int n_rays, int n_samples, float grad_scale, void* stream,
                        int phases) {
  using namespace nerf;
  if (n_rays <= 0) return 0;
  NERF_CHECK_ARG(stash && workspace, "mlp_backward: null pointer");
  NERF_CHECK_ARG(grad_scale > 0.f, "mlp_backward: grad_scale must be positive");
  const int64_t n_evals = (int64_t)n_rays * n_samples;
  NERF_CHECK_ARG(n_evals < (int64_t(1) << 31) - kTile, "mlp_backward: n_rays*n_samples must be < 2^31 per call");
  NERF_CHECK_ARG(((reinterpret_cast<uintptr_t>(stash) | reinterpret_cast<uintptr_t>(workspace) | reinterpret_cast<uintptr_t>(packed)) & 127) == 0,
                 "mlp_backward: stash, workspace and packed must be 128-byte aligned");
  BwdParams p;
  p.d_rgbsigma = reinterpret_cast<const float4*>(d_rgbsigma);
  p.rgbsigma = reinterpret_cast<const float4*>(rgbsigma);
  p.stash = static_cast<const uint8_t*>(stash);
  p.gstash = static_cast<uint8_t*>(workspace);
  p.packed = static_cast<const uint8_t*>(packed);
  p.params = params;
  p.n_evals = n_evals;
  p.n_tiles = (int)((n_evals + kTile - 1) / kTile);
  p.prof = reinterpret_cast<unsigned long long*>(timing_buffer());
  if (phases & 1) {
    NERF_CHECK_ARG(d_rgbsigma && rgbsigma && packed && params, "mlp_backward: null pointer");
    static bool smem_set[kMaxDevices] = {};
    const cudaError_t e = set_max_dynamic_smem_once(smem_set, {(const void*)mlp_dgrad_kernel}, bwd::kSmemBytes);
    NERF_CHECK_ARG(e == cudaSuccess, "mlp_backward: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
    mlp_dgrad_kernel<<<chain::grid(p.n_tiles), chain::kThreads, bwd::kSmemBytes, static_cast<cudaStream_t>(stream)>>>(p);
    NERF_CHECK_LAUNCH("mlp_dgrad_kernel");
  }
  if (phases & 2) {
    NERF_CHECK_ARG(grads != nullptr, "mlp_backward: null gradient buffer");
    return launch_wgrad(grads, p.stash, p.gstash, p.n_tiles, 1.f / grad_scale, static_cast<cudaStream_t>(stream));
  }
  return 0;
}

extern "C" int nerf_mlp_backward(float* grads, const float* d_rgbsigma, const float* rgbsigma, const void* stash, void* workspace,
                                 const void* packed, const float* params, int n_rays, int n_samples, float grad_scale,
                                 void* stream) {
  return run_backward(grads, d_rgbsigma, rgbsigma, stash, workspace, packed, params, n_rays, n_samples, grad_scale, stream, 3);
}

extern "C" int nerf_mlp_backward_dgrad(const float* d_rgbsigma, const float* rgbsigma, const void* stash, void* workspace,
                                       const void* packed, const float* params, int n_rays, int n_samples, void* stream) {
  return run_backward(nullptr, d_rgbsigma, rgbsigma, stash, workspace, packed, params, n_rays, n_samples, 1.f, stream, 1);
}

extern "C" int nerf_mlp_backward_wgrad(float* grads, const void* stash, const void* workspace, int n_rays, int n_samples,
                                       float grad_scale, void* stream) {
  return run_backward(grads, nullptr, nullptr, stash, const_cast<void*>(workspace), nullptr, nullptr, n_rays, n_samples,
                      grad_scale, stream, 2);
}
