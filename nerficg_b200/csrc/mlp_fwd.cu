// mlp_fwd.cu -- K3: positional encoding + the 8x256 skip-connected NeRF MLP as ONE fused,
// persistent, warp-specialised tcgen05 kernel on a CTA pair (chain.cuh), walking the 10-stage chain of mlp_layout.cuh.
//
// What only the forward does: the epilogues of stages 0..8 add the bias, apply ReLU and write fp16 A operand panels of
// the next stage; the density head (256->1) and the RGB head (128->3, sigmoid) are evaluated on CUDA cores inside the
// epilogues of stages 7 and 9, so the kernel emits packed (r,g,b,sigma) per sample.  Training additionally stashes every
// operand image the backward needs (bulk stores from shared memory, region-major, see mlp_layout.cuh) and per-layer ReLU
// bit masks.
//
// Measured lessons baked into the structure (DESIGN.md "K3"):
//   * N = 256 per instruction halves the instruction count and the re-reads of the A operand;
//   * the epilogue prefetches the next chunk's bias (and density weights) while it processes the
//     current one and takes the registers the producer / MMA warps do not need (setmaxnreg).
#include "chain.cuh"
#include "encoding.cuh"
#include "../../include/nerf_b200.h"

namespace nerf {
using namespace tc;

namespace fwd {
constexpr int kRingStages = 4;
// shared memory map (offsets from the 1024-aligned base)
constexpr uint32_t kSlotBytes = kActBytes + kPanelBytes128;  // act (4 panels) + enc (1 panel)
constexpr uint32_t kOffRing = 2 * kSlotBytes;
constexpr uint32_t kOffBars = kOffRing + kRingStages * chain::kRingStageBytes;
constexpr uint32_t kOffBias = kOffBars + 256;             // [2 slots][256 floats]: the bias vector of the stage in flight
constexpr uint32_t kSmemBytes = kOffBias + 2 * 1024;      // the dynamic window is 1024-byte aligned (checked at kernel entry)
static_assert(kSmemBytes <= 232448, "shared memory budget exceeded");

struct Stages {
  static constexpr int kStages = kFwdStages, kRingStages = fwd::kRingStages;
  static constexpr int kProfBase = 0;  // stall-counter slots 0..9
  __device__ static constexpr int panels(int st) { return fwd_panels(st); }
  // every stage but the two 5-panel ones (skip layer, colour layer).  Measured (profiles/r02_chain_kernel_experiments.txt):
  // the issuer's W-full wait halves and its A-ready wait grows by almost as much -- the epilogue is the critical path --
  // so the gain is 1-2 % (inference 0.674 -> 0.667 ms, training 1.051 -> 1.038).
  __device__ static constexpr bool shared(int st) { return fwd_panels(st) <= kRingStages; }
};
}  // namespace fwd

struct FwdParams {
  float4* rgbsigma;
  uint8_t* stash;  // nullptr for inference
  const uint8_t* packed;
  const float* params;
  const float* origins;
  const float* dirs;
  const float* viewdirs;
  const float* z;
  const float* noise;
  int n_rays;
  int n_samples;    // S
  int64_t n_evals;  // n_rays * S
  int n_tiles;
  unsigned long long* prof;  // optional stall counters (chain.cuh), slots 0..9 and 22..24
};

// ---- per-row input encoding ----------------------------------------------------------------
// 63 position features [x, cos(2^k x_i), sin(2^k x_i)] (reference utils.py:32-36) as 64 halves (encode_axis: encoding.cuh).

// chunks [4 * half, 4 * half + 4) of one panel row: 32 values -> 32 halves (each column half of a row has its own thread)
__device__ __forceinline__ void write_half_row(uint32_t panel_smem, int row, int half, const float* vals /*[32]*/) {
#pragma unroll
  for (int ch = 0; ch < 4; ++ch) {
    st_shared_v4(panel_smem + panel_chunk_offset(row, 4 * half + ch), pack_half2(vals[8 * ch + 0], vals[8 * ch + 1]),
                 pack_half2(vals[8 * ch + 2], vals[8 * ch + 3]), pack_half2(vals[8 * ch + 4], vals[8 * ch + 5]),
                 pack_half2(vals[8 * ch + 6], vals[8 * ch + 7]));
  }
}

// Half (16 columns, kOff = 0 or 16) of a 32-column chunk of a hidden-stage epilogue: x = acc + bias [ReLU] -> fp16
// pairs -> two 16-byte chunks of the swizzled A operand; c0 = byte offset of the 32-column chunk in the (unswizzled)
// panel row.  breg holds the bias of these 16 columns, loaded by the caller from the slot's shared-memory copy (one
// broadcast LDS.128 per four columns; from global memory every ~20th load missed the 28 KB L1 and stalled the warp for
// an L2 round trip).  Returns the ReLU bits of these 16 columns (tc.cuh relu_mask_bit layout); accumulates the density
// head (fp32, weights at ws) when kDens.
template <bool kDens, bool kMask, int kOff>
__device__ __forceinline__ uint32_t hidden16(const uint32_t (&v)[32], const float* __restrict__ ws, bool relu,
                                             uint32_t pbase, uint32_t c0, uint32_t xr, float& dens, const float4* breg) {
  uint32_t m = 0;
  uint32_t w[8];
#pragma unroll
  for (int qq = 0; qq < 4; ++qq) {
    constexpr int kQ0 = kOff / 4;
    const int q = kQ0 + qq;  // index of the 4-column group within the 32-column chunk
    const float4 bq = breg[qq];   // (loaded one 16-column group ahead by the caller)
    float x0 = __uint_as_float(v[4 * q + 0]) + bq.x;
    float x1 = __uint_as_float(v[4 * q + 1]) + bq.y;
    float x2 = __uint_as_float(v[4 * q + 2]) + bq.z;
    float x3 = __uint_as_float(v[4 * q + 3]) + bq.w;
    uint32_t w0, w1;
    if (kDens) {  // the density head reads the fp32 activations (stage 7, always ReLU)
      x0 = fmaxf(x0, 0.f);
      x1 = fmaxf(x1, 0.f);
      x2 = fmaxf(x2, 0.f);
      x3 = fmaxf(x3, 0.f);
      const float4 wq = __ldg(reinterpret_cast<const float4*>(ws) + q);
      dens = fmaf(x0, wq.x, fmaf(x1, wq.y, fmaf(x2, wq.z, fmaf(x3, wq.w, dens))));
      w0 = pack_half2(x0, x1);
      w1 = pack_half2(x2, x3);
    } else {  // ReLU in the fp16 domain: one HMNMX2 per pair, same result as rounding the fp32 ReLU
      w0 = pack_half2(x0, x1);
      w1 = pack_half2(x2, x3);
      if (relu) {
        w0 = half2_relu(w0);
        w1 = half2_relu(w1);
      }
    }
    if (kMask) {
      m |= half2_gt0_mask(w0) & (0x00010001u << (2 * q));
      m |= half2_gt0_mask(w1) & (0x00010001u << (2 * q + 1));
    }
    w[2 * qq] = w0;
    w[2 * qq + 1] = w1;
  }
  st_shared_v4(pbase + ((c0 + 2u * kOff) ^ xr), w[0], w[1], w[2], w[3]);
  st_shared_v4(pbase + ((c0 + 2u * kOff + 16u) ^ xr), w[4], w[5], w[6], w[7]);
  return m;
}

// kProf: the stall counters (nerf_debug_set_timing) are compiled into their own instantiation; in the production one the
// compiler drops every clock read and accumulator (with a run-time flag only, ptxas kept the 64-bit accumulators in local
// memory and their reloads showed up in ncu's hot list)
template <bool kTrain, bool kProf>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(chain::kThreads, 1) mlp_fwd_kernel(const FwdParams p) {
  using namespace fwd;
  using L = ParamLayout;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = smem_u32(smem_raw);
  if ((smem_base & 1023u) != 0) __trap();  // SWIZZLE_128B operands need 1024-byte alignment and there is no slack to re-align
  const chain::Bars bars(smem_base + kOffBars, kRingStages, true);
  const uint32_t rank = cluster_ctarank();  // 0 = leader
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tmem_base = chain::setup(bars, warp);
  const chain::Schedule sch(p.n_tiles);
  const bool prof_on = kProf && p.prof != nullptr;

  if (warp < 4) {
    setmaxnreg_dec<chain::kRegsOther>();
    if (warp == 0) {
      chain::producer<Stages>(sch, bars, smem_base + kOffRing, prof_on, p.prof, [&](int st, int pp) {
        const uint32_t bytes = st == 9 ? chain::kRingStageBytes / 2 : chain::kRingStageBytes;  // colour layer: 64 of 128 neurons
        return chain::Panel{p.packed + fwd_panel_offset(fwd_first_panel(st) + pp) + rank * bytes, bytes};
      });
    } else if (warp == 1 && rank == 0) {
      constexpr uint32_t idesc256 = make_idesc(256, 256, kF16, kF16, 0, 0);
      constexpr uint32_t idesc128 = make_idesc(256, 128, kF16, kF16, 0, 0);
      chain::issuer<Stages>(sch, bars, smem_base + kOffRing, tmem_base, prof_on, p.prof,
                            [&](int st, int slot, int pp, uint32_t d_tmem, uint64_t db) {
        const uint32_t act = smem_base + slot * kSlotBytes;
        const uint32_t enc = act + kActBytes;
        // A: stage 0 reads the encoding panel; panel 4 of stages 5 / 9 is the encoding / direction panel
        const uint64_t da = make_smem_desc((st == 0 || pp == 4) ? enc : act + pp * kPanelBytes128, 16u, kAtomBytes);
        const uint32_t idesc = st == 9 ? idesc128 : idesc256;
        const int ksteps = (st == 9 && pp == 4) ? 2 : 4;  // the direction encoding is 32 wide
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          if (ks < ksteps) umma2(d_tmem, da + 2u * ks, db + 2u * ks, idesc, (pp | ks) != 0);
      });
    } else if (warp == 1) {
      chain::relay<Stages>(sch, bars);
    }
  } else {
    // =============================== epilogue warps ===============================
    setmaxnreg_inc<chain::kRegsEpilogue>();
    const chain::Epilogue epi(warp, lane, smem_base, kSlotBytes, tmem_base, bars);
    const int slot = epi.slot, half = epi.half, row = epi.row, tg = epi.tg;
    const uint32_t act = epi.act, t_slot = epi.t_slot, row_off = epi.row_off, xr = epi.xr;
    const uint32_t enc = act + kActBytes;
    const uint32_t t_acc = t_slot + 128 * half;  // hidden stages: columns [128 * half, +128)
    uint32_t acc_phase = 0, bias_phase = 0;
    const uint64_t n_tiles64 = (uint64_t)p.n_tiles;
    const bool prof = prof_on && tg == 0 && slot == 0;
    // the bias vector of the stage in flight lives in shared memory (one buffer per slot): after the slot's warps have
    // finished a stage (and met at a barrier) one thread bulk-copies the next stage's vector, which lands long before
    // the next accumulator is complete
    const float4* bias_s4 = reinterpret_cast<const float4*>(smem_raw + kOffBias + slot * 1024);
    const uint32_t bias_u32 = smem_base + kOffBias + slot * 1024;
    auto bias_fetch = [&](int stage) {  // one thread; stage 0..7 hidden, 8 feature, 9 colour layer 0
      const float* src = p.params + (stage < 8 ? L::hidden_b(stage) : (stage == 8 ? L::kBF : L::kBC0));
      const uint32_t bytes = stage == 9 ? 512u : 1024u;
      mbar_arrive_expect_tx(bars.bias + 8 * slot, bytes);
      bulk_g2s(bias_u32, src, bytes, bars.bias + 8 * slot);
    };
    if (tg == 0 && sch.active(0, slot)) bias_fetch(0);
    long long t_accw = 0, t_drain = 0, t_pro = 0, t_bias = 0, t_bar = 0, t_mask = 0;
    const long long t_begin = prof ? clock64() : 0;

    for (int it = 0; it < sch.n_iters; ++it) {
      if (!sch.active(it, slot)) break;
      const int tile = sch.tile(it, slot, rank);
      const bool tile_ok = tile < p.n_tiles;
      const long long t_tile = prof ? clock64() : 0;
      const int64_t e = (int64_t)tile * kTile + row;  // sample index
      const bool valid = tile_ok && e < p.n_evals;
      const int ray = valid ? (int)(e / p.n_samples) : 0;

      // training only: the activation stash images
      auto stash_dst = [&](int region) {
        return [&, region] { return p.stash + stash_region_offset(region, n_tiles64) + (uint64_t)tile * stash_region_tile_bytes(region); };
      };
      auto stash_store = [&](int region, uint32_t src, uint32_t bytes) {
        if (kTrain) epi.image_store(stash_dst(region), src, bytes, tile_ok);
      };
      auto stash_drain = [&]() {
        if (kTrain) epi.image_drain(prof, t_drain);
      };

      // ---------------- prologue: position encoding -> enc panel (each half writes its 32 of the 64 columns) ----------------
      // columns: [x y z | enc(x) 3..22 | enc(y) 23..42 | enc(z) 43..62 | 0]; half 0 needs enc(x) and the first nine
      // cosines of enc(y), half 1 the rest of enc(y) and enc(z): two sincos chains per thread instead of three
      float vdx = 0.f, vdy = 0.f, vdz = 0.f;
      {
        float x0 = 0.f, x1 = 0.f, x2 = 0.f;
        if (valid) {
          const float zz = __ldg(p.z + e);
          x0 = __fadd_rn(__ldg(p.origins + 3 * ray + 0), __fmul_rn(__ldg(p.dirs + 3 * ray + 0), zz));
          x1 = __fadd_rn(__ldg(p.origins + 3 * ray + 1), __fmul_rn(__ldg(p.dirs + 3 * ray + 1), zz));
          x2 = __fadd_rn(__ldg(p.origins + 3 * ray + 2), __fmul_rn(__ldg(p.dirs + 3 * ray + 2), zz));
          if (half == 0) {
            vdx = __ldg(p.viewdirs + 3 * ray + 0);
            vdy = __ldg(p.viewdirs + 3 * ray + 1);
            vdz = __ldg(p.viewdirs + 3 * ray + 2);
          }
        }
        float ea[20], eb[20], vals[32];
        encode_axis(half == 0 ? x0 : x1, 10, ea);
        encode_axis(half == 0 ? x1 : x2, 10, eb);
        if (half == 0) {
          vals[0] = x0;
          vals[1] = x1;
          vals[2] = x2;
#pragma unroll
          for (int k = 0; k < 20; ++k) vals[3 + k] = ea[k];
#pragma unroll
          for (int k = 0; k < 9; ++k) vals[23 + k] = eb[k];
        } else {
          vals[0] = ea[9];
#pragma unroll
          for (int k = 0; k < 10; ++k) vals[1 + k] = ea[10 + k];
#pragma unroll
          for (int k = 0; k < 20; ++k) vals[11 + k] = eb[k];
          vals[31] = 0.f;
        }
        stash_drain();  // previous tile's DIR / G stores still reading enc / act
        write_half_row(enc, row, half, vals);
      }
      stash_store(kStashEnc, enc, kPanelBytes128);
      epi.hand_off();
      if (prof) t_pro += clock64() - t_tile;

      // next tile's prologue inputs (depths and the ray of each sample) -> L2, issued two stages before this tile ends
      auto prefetch_next_tile = [&]() {
        if (half == 0 && it + 1 < sch.n_iters && sch.active(it + 1, slot)) {
          const int next = sch.tile(it + 1, slot, rank);
          const int64_t en = (int64_t)next * kTile + row;
          if (next < p.n_tiles && en < p.n_evals) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(p.z + en));
            if ((row & 31) == 0) {  // the 32 samples of a warp span at most two rays
              const int rn = (int)(en / p.n_samples);
              asm volatile("prefetch.global.L2 [%0];" ::"l"(p.origins + 3 * rn));
              asm volatile("prefetch.global.L2 [%0];" ::"l"(p.dirs + 3 * rn));
              asm volatile("prefetch.global.L2 [%0];" ::"l"(p.viewdirs + 3 * rn));
            }
          }
        }
      };
      float dens = 0.f;  // density head, partial sum over this thread's 128 columns (combined in stage 9)
      // ---------------- chain stages 0..8: hidden layers (ReLU) and the feature layer (linear) ----------------
#pragma unroll 1
      for (int st = 0; st < 9; ++st) {
        const bool relu = st < 8;
        if (st == 7) prefetch_next_tile();
        NERF_TIMED(prof, t_accw, mbar_wait(bars.acc_ready + 8 * slot, acc_phase));
        acc_phase ^= 1;
        tc_fence_after();
        uint32_t mw[4] = {0u, 0u, 0u, 0u};  // ReLU bits of this thread's four 32-column chunks
        // software pipeline over the four 32-column chunks of this half (two register buffers).  The load of the next
        // chunk is issued half way through the current one: issued right behind the shared-memory stores that last
        // read the target registers it waits for the store queue, and ptxas then sinks it behind all the arithmetic.
        // (Measured: with the bias in shared memory the exact position no longer matters -- 0.69 ms either way.)
        auto run = [&](auto dens_tag) {
          constexpr bool kDens = decltype(dens_tag)::value;
          const float* wsp = p.params + L::kWS + 128 * half;
          const float4* bsp = bias_s4 + 32 * half;
          uint32_t va[32], vb[32];
          tmem_ld32(t_acc, va);
          stash_drain();  // the act image of the previous stage may still be being stored
          NERF_TIMED(prof, t_bias, mbar_wait(bars.bias + 8 * slot, bias_phase));
          // The bias words of 16-column group g + 1 are loaded BEFORE the (asm volatile, "memory") stores of group g: the compiler
          // cannot move the LDS across them by itself, and ncu's source view showed the first FADD of every group waiting on it
          // (13 % of the epilogue warps' samples).  Measured (round 2, profiles/r02_chain_kernel_experiments.txt): training
          // forward 1.049 -> 0.972 ms, inference 0.703 -> 0.695 ms.
          float4 ba[4], bb[4];
          auto load4 = [&](float4 (&dst)[4], int group) {   // group = 16-column group index within this thread's 128 columns
#pragma unroll
            for (int i = 0; i < 4; ++i) dst[i] = bsp[4 * group + i];
          };
          load4(ba, 0);
#pragma unroll
          for (int c = 0; c < 4; c += 2) {
            const uint32_t pbase = epi.act_h + (uint32_t)(c >> 1) * kPanelBytes128;
            tmem_ld_wait32(va);
            load4(bb, 2 * c + 1);
            mw[c] = hidden16<kDens, kTrain, 0>(va, wsp + 32 * c, relu, pbase, 0u, xr, dens, ba);
            tmem_ld32(t_acc + 32 * (c + 1), vb);
            load4(ba, 2 * c + 2);
            mw[c] |= hidden16<kDens, kTrain, 16>(va, wsp + 32 * c, relu, pbase, 0u, xr, dens, bb);
            tmem_ld_wait32(vb);
            load4(bb, 2 * c + 3);
            mw[c + 1] = hidden16<kDens, kTrain, 0>(vb, wsp + 32 * (c + 1), relu, pbase, 64u, xr, dens, ba);
            if (c + 2 < 4) {
              tmem_ld32(t_acc + 32 * (c + 2), va);
              load4(ba, 2 * c + 4);
            }
            mw[c + 1] |= hidden16<kDens, kTrain, 16>(vb, wsp + 32 * (c + 1), relu, pbase, 64u, xr, dens, bb);
          }
        };
        if (st == 7) run(chain::BoolTag<true>{}); else run(chain::BoolTag<false>{});
        bias_phase ^= 1;
        if (st == 8) {
          // direction encoding -> enc panel (the x encoding was last read by stage 5): 27 values in half 0, zeros beyond
          float vals[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) vals[j] = 0.f;
          if (half == 0) {
            vals[0] = vdx;
            vals[1] = vdy;
            vals[2] = vdz;
            encode_axis(vdx, 4, vals + 3);
            encode_axis(vdy, 4, vals + 11);
            encode_axis(vdz, 4, vals + 19);
          }
          write_half_row(enc, row, half, vals);
          stash_store(kStashDir, enc, kPanelBytes128);
        }
        // operands are handed to the MMA issuer per warp BEFORE the slot's warps meet for the image store / bias refill
        // (measured in round 2: inference 0.689 -> 0.667 ms at 4096 x 192, training unchanged)
        epi.hand_off();
        NERF_TIMED(prof, t_bar, epi.sync());
        if (kTrain) {
          const int region = st < 8 ? kStashH0 + st : kStashF;
          epi.image_issue(stash_dst(region), act, kActBytes, tile_ok);
        }
        if (tg == 0) bias_fetch(st + 1);
        // ReLU bits -> stash, after the hand-off: a plain global store can stall its warp under the stash's HBM write load
        if (kTrain && relu && tile_ok) {
          uint4* md = reinterpret_cast<uint4*>(p.stash + stash_region_offset(kStashMask, n_tiles64) +
                                               (uint64_t)tile * stash_region_tile_bytes(kStashMask) + st * (128 * 32) + row * 32 + half * 16);
          const long long t0 = prof ? clock64() : 0;
          *md = make_uint4(mw[0], mw[1], mw[2], mw[3]);
          if (prof) t_mask += clock64() - t0;
        }
      }
      // ---------------- stage 9: g = ReLU(acc + b) (128 wide); rgb = sigmoid(W_c1 g + b_c1) on CUDA cores ----------------
      {
        const int cb = 64 * half;  // this thread's 64 of the 128 colour-layer neurons
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        uint32_t gm0 = 0u, gm1 = 0u;  // ReLU bits of this thread's two 32-column chunks of g
        NERF_TIMED(prof, t_accw, mbar_wait(bars.acc_ready + 8 * slot, acc_phase));
        acc_phase ^= 1;
        tc_fence_after();
        stash_drain();  // the F image store reads act, which receives g (and the partial sums) below
        mbar_wait(bars.bias + 8 * slot, bias_phase);
        bias_phase ^= 1;
#pragma unroll 1
        for (int s = 0; s < 4; ++s) {
          const int c0 = cb + 16 * s;
          uint32_t v[16];
          tmem_ld16(t_slot + c0, v);
          const float4* b4 = bias_s4 + (c0 >> 2);
          const float4* w0 = reinterpret_cast<const float4*>(p.params + L::kWC1 + c0);
          const float4* w1 = reinterpret_cast<const float4*>(p.params + L::kWC1 + 128 + c0);
          const float4* w2 = reinterpret_cast<const float4*>(p.params + L::kWC1 + 256 + c0);
          tmem_ld_wait16(v);
          uint32_t w[8];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 bq = b4[q], u0 = __ldg(w0 + q), u1 = __ldg(w1 + q), u2 = __ldg(w2 + q);
            const float g0 = fmaxf(__uint_as_float(v[4 * q + 0]) + bq.x, 0.f);
            const float g1 = fmaxf(__uint_as_float(v[4 * q + 1]) + bq.y, 0.f);
            const float g2 = fmaxf(__uint_as_float(v[4 * q + 2]) + bq.z, 0.f);
            const float g3 = fmaxf(__uint_as_float(v[4 * q + 3]) + bq.w, 0.f);
            a0 = fmaf(g0, u0.x, fmaf(g1, u0.y, fmaf(g2, u0.z, fmaf(g3, u0.w, a0))));
            a1 = fmaf(g0, u1.x, fmaf(g1, u1.y, fmaf(g2, u1.z, fmaf(g3, u1.w, a1))));
            a2 = fmaf(g0, u2.x, fmaf(g1, u2.y, fmaf(g2, u2.z, fmaf(g3, u2.w, a2))));
            w[2 * q] = pack_half2(g0, g1);
            w[2 * q + 1] = pack_half2(g2, g3);
            if (kTrain) {  // ReLU bits of g for the dgrad prologue (it no longer has to fetch the 32 KB G image for its signs)
              const uint32_t sh = (uint32_t)((s & 1) * 8 + 2 * q);
              const uint32_t bits = (half2_gt0_mask(w[2 * q]) & (0x00010001u << sh)) | (half2_gt0_mask(w[2 * q + 1]) & (0x00010001u << (sh + 1)));
              if (s < 2) gm0 |= bits; else gm1 |= bits;
            }
          }
          if (kTrain) {  // g image: panel `half`, 16-byte chunks 2s and 2s+1 of the row
            const uint32_t base = act + half * kPanelBytes128 + row_off;
            st_shared_v4(base + (((uint32_t)(2 * s) << 4) ^ xr), w[0], w[1], w[2], w[3]);
            st_shared_v4(base + (((uint32_t)(2 * s + 1) << 4) ^ xr), w[4], w[5], w[6], w[7]);
          }
        }
        if (kTrain && tile_ok)
          *reinterpret_cast<uint2*>(p.stash + stash_region_offset(kStashMask, n_tiles64) + (uint64_t)tile * stash_region_tile_bytes(kStashMask) +
                                    8 * (128 * 32) + row * 32 + half * 8) = make_uint2(gm0, gm1);
        // the two halves of a row meet in act panel 3 (free: F has been consumed, g only fills panels 0 and 1)
        const uint32_t xch = act + 3 * kPanelBytes128 + (uint32_t)row * 16u;
        if (half == 1) st_shared_v4(xch, __float_as_uint(a0), __float_as_uint(a1), __float_as_uint(a2), __float_as_uint(dens));
        stash_store(kStashG, act, 2 * kPanelBytes128);  // (training) its barrier also orders the exchange
        if (!kTrain) {
          fence_proxy_async_smem();
          epi.sync();
        }
        if (tg == 0 && it + 1 < sch.n_iters && sch.active(it + 1, slot)) bias_fetch(0);  // first stage of this slot's next tile
        if (half == 0 && valid) {
          uint32_t r0, r1, r2, r3;
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(xch));
          a0 += __uint_as_float(r0) + __ldg(p.params + L::kBC1 + 0);
          a1 += __uint_as_float(r1) + __ldg(p.params + L::kBC1 + 1);
          a2 += __uint_as_float(r2) + __ldg(p.params + L::kBC1 + 2);
          float raw = dens + __uint_as_float(r3) + __ldg(p.params + L::kBS);
          if (p.noise != nullptr) raw += __ldg(p.noise + e);
          float4 o;
          o.x = 1.f / (1.f + expf(-a0));
          o.y = 1.f / (1.f + expf(-a1));
          o.z = 1.f / (1.f + expf(-a2));
          o.w = fmaxf(raw, 0.f);
          p.rgbsigma[e] = o;
        }
        // the accumulator has been drained; the arrive that releases it is the next tile's prologue
        tc_fence_before();
      }
    }
    if (kTrain && tg == 0) bulk_wait_all<0>();
    if (prof) {
      chain::epilogue_counters<Stages>(p.prof, t_accw, t_begin, t_drain, t_pro);
      atomicAdd(p.prof + 22, (unsigned long long)t_bias);   // (slots 10..21 belong to dgrad) waits the table above counts as busy time
      atomicAdd(p.prof + 23, (unsigned long long)t_bar);
      atomicAdd(p.prof + 24, (unsigned long long)t_mask);
    }
  }
  chain::teardown(tmem_base, warp);
}

}  // namespace nerf

extern "C" size_t nerf_mlp_stash_bytes(int64_t n_samples) {
  const uint64_t n_tiles = (uint64_t)((n_samples + nerf::kTile - 1) / nerf::kTile);
  return (size_t)(nerf::stash_tile_bytes_total() * n_tiles);
}

extern "C" int nerf_mlp_forward(float* rgbsigma, void* stash, const void* packed, const float* params, const float* origins,
                                const float* dirs, const float* viewdirs, const float* z, const float* noise, int n_rays,
                                int n_samples, void* stream) {
  using namespace nerf;
  if (n_rays <= 0) return 0;
  NERF_CHECK_ARG(rgbsigma && packed && params && origins && dirs && viewdirs && z, "mlp_forward: null pointer");
  NERF_CHECK_ARG(n_samples >= 1, "mlp_forward: n_samples must be >= 1");
  const int64_t n_evals = (int64_t)n_rays * n_samples;
  NERF_CHECK_ARG(n_evals < (int64_t(1) << 31) - kTile, "mlp_forward: n_rays*n_samples must be < 2^31 per call");
  NERF_CHECK_ARG((reinterpret_cast<uintptr_t>(packed) & 127) == 0 && (reinterpret_cast<uintptr_t>(rgbsigma) & 15) == 0,
                 "mlp_forward: packed must be 128-byte and rgbsigma 16-byte aligned");
  NERF_CHECK_ARG((reinterpret_cast<uintptr_t>(params) & 15) == 0, "mlp_forward: params must be 16-byte aligned");
  NERF_CHECK_ARG(stash == nullptr || (reinterpret_cast<uintptr_t>(stash) & 127) == 0, "mlp_forward: stash must be 128-byte aligned");
  FwdParams p;
  p.rgbsigma = reinterpret_cast<float4*>(rgbsigma);
  p.stash = static_cast<uint8_t*>(stash);
  p.packed = static_cast<const uint8_t*>(packed);
  p.params = params;
  p.origins = origins;
  p.dirs = dirs;
  p.viewdirs = viewdirs;
  p.z = z;
  p.noise = noise;
  p.n_rays = n_rays;
  p.n_samples = n_samples;
  p.n_evals = n_evals;
  p.n_tiles = (int)((n_evals + kTile - 1) / kTile);
  p.prof = reinterpret_cast<unsigned long long*>(timing_buffer());
  const int grid = chain::grid(p.n_tiles);
  static bool smem_set[kMaxDevices] = {};
  const cudaError_t e = set_max_dynamic_smem_once(
      smem_set, {(const void*)mlp_fwd_kernel<false, false>, (const void*)mlp_fwd_kernel<true, false>,
                 (const void*)mlp_fwd_kernel<false, true>, (const void*)mlp_fwd_kernel<true, true>}, fwd::kSmemBytes);
  NERF_CHECK_ARG(e == cudaSuccess, "mlp_forward: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool with_prof = p.prof != nullptr;
  if (stash != nullptr) {
    if (with_prof) mlp_fwd_kernel<true, true><<<grid, chain::kThreads, fwd::kSmemBytes, st>>>(p);
    else mlp_fwd_kernel<true, false><<<grid, chain::kThreads, fwd::kSmemBytes, st>>>(p);
  } else {
    if (with_prof) mlp_fwd_kernel<false, true><<<grid, chain::kThreads, fwd::kSmemBytes, st>>>(p);
    else mlp_fwd_kernel<false, false><<<grid, chain::kThreads, fwd::kSmemBytes, st>>>(p);
  }
  NERF_CHECK_LAUNCH("mlp_fwd_kernel");
  return 0;
}
