// mlp_dinput.cu -- K4c: gradients of NeRFBlock.forward with respect to its inputs (query positions and view directions),
// read from the gradient stash the dgrad chain (K4a, mlp_bwd.cu) has written.
//
// The encoded position enters the MLP twice (layer 0, and layer 5 behind h4) and the encoded direction once (colour
// layer 0 behind f), so per 128-sample tile
//   dL/d enc(x) = D0 . W0 + D5 . W5[:, 256:319]    one K = 512 contraction into 63 (+1 pad) columns
//   dL/d enc(d) = DC0 . Wc0[:, 256:283]             K = 128 into 27 (+5 pad) columns
// where D0, D5 and DC0 are the fp16 pre-activation gradients of those layers, already stored as K-major panel images
// (mlp_layout.cuh GradRegion).  The chain rule through the frequency encoding then runs in fp32 on CUDA cores.
//
// One persistent CTA per SM, 6 warps:
//   warp 0     producer: streams the tile's A panels (16 KB each) into an 8-stage ring with 1-D bulk copies
//   warp 1     TMEM owner and MMA issuer (one elected lane): M = 128 tcgen05.mma, B = the transposed weight slices,
//              which every CTA builds once in shared memory; two accumulator buffers of 96 columns
//   warps 2-5  epilogue, one sample row per thread (warp w reads TMEM lane quarter w % 4)
#include "common.cuh"
#include "encoding.cuh"
#include "mlp_layout.cuh"
#include "tc.cuh"
#include "../../include/nerf_b200.h"

namespace nerf {
using namespace tc;

namespace dinput {
constexpr int kThreads = 192;
constexpr int kRingStages = 8;
constexpr int kGradL5 = kGradL7 + 2;  // regions D7..D0 follow each other
// A panels of one tile, in issue order: D0 (4), D5 (4) -> position accumulator; DC0 (2) -> direction accumulator
constexpr int kPosPanels = 8, kTilePanels = 10;
// B operands: W0^T and W5[:, 256:319]^T are 64 rows (input feature) x 256 (neuron) = 4 panels of 8 KB each,
// Wc0[:, 256:283]^T is 32 rows x 128 = 2 panels of 4 KB
constexpr uint32_t kPosPanelBytes = 64 * kPanelRowBytes, kDirPanelBytes = 32 * kPanelRowBytes;
constexpr uint32_t kOffW0 = 0, kOffW5 = 4 * kPosPanelBytes, kOffWc0 = 8 * kPosPanelBytes;
constexpr uint32_t kOffRing = kOffWc0 + 2 * kDirPanelBytes;
constexpr uint32_t kOffBars = kOffRing + kRingStages * kPanelBytes128;
constexpr uint32_t kSmemBytes = kOffBars + 256 + 1024;  // + 1 KB to align the dynamic window up to 1024 bytes
static_assert(kSmemBytes <= 232448, "shared memory budget exceeded");
// TMEM: buffer b holds the position accumulator in columns [128 b, +64) and the direction one in [128 b + 64, +32)
constexpr uint32_t kTmemCols = 256, kAccStride = 128, kAccDir = 64;
}  // namespace dinput

struct DinputParams {
  float* d_positions;   // nullptr: skipped
  float* d_directions;  // nullptr: skipped
  const uint8_t* gstash;
  const float* params;
  const float* positions;
  const float* directions;
  int64_t n;
  int n_tiles;
  float inv_scale;
};

// One 16-byte chunk (8 halves) of a transposed weight slice: row `n` (input feature col0 + n of W, zero from `valid` on),
// columns 8 * kc .. 8 * kc + 7 (neurons).  Rounded like nerf_mlp_pack.
__device__ __forceinline__ void build_wt_chunk(uint32_t dst_panels, uint32_t panel_bytes, const float* __restrict__ w, int ld,
                                               int col0, int valid, int n, int kc) {
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = n < valid ? __ldg(w + (int64_t)(8 * kc + e) * ld + col0 + n) : 0.f;
  st_shared_v4(dst_panels + (uint32_t)(kc >> 3) * panel_bytes + panel_chunk_offset(n, kc & 7), pack_half2(v[0], v[1]),
               pack_half2(v[2], v[3]), pack_half2(v[4], v[5]), pack_half2(v[6], v[7]));
}

__global__ void __launch_bounds__(dinput::kThreads, 1) mlp_dinput_kernel(const DinputParams p) {
  using namespace dinput;
  using L = ParamLayout;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = smem_base + kOffBars, bar_empty = bar_full + 8 * kRingStages;
  const uint32_t bar_acc_full = bar_empty + 8 * kRingStages, bar_acc_empty = bar_acc_full + 16, tmem_slot = bar_acc_empty + 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool want_pos = p.d_positions != nullptr, want_dir = p.d_directions != nullptr;
  const int p_begin = want_pos ? 0 : kPosPanels, p_end = want_dir ? kTilePanels : kPosPanels;

  // ---- prologue: the three transposed weight slices (lanes walk the input features: coalesced reads of one W row) ----
  for (int q = threadIdx.x; q < 2 * 2048 + 512; q += kThreads) {
    if (q < 2048) {
      build_wt_chunk(smem_base + kOffW0, kPosPanelBytes, p.params + L::kW0, 63, 0, 63, q & 63, q >> 6);
    } else if (q < 4096) {
      build_wt_chunk(smem_base + kOffW5, kPosPanelBytes, p.params + L::kW5, 319, 256, 63, q & 63, (q - 2048) >> 6);
    } else {
      build_wt_chunk(smem_base + kOffWc0, kDirPanelBytes, p.params + L::kWC0, 283, 256, 27, q & 31, (q - 4096) >> 5);
    }
  }
  fence_proxy_async_smem();
  if (threadIdx.x == 0) {
    for (int i = 0; i < kRingStages; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_acc_full + 8 * b, 1);
      mbar_init(bar_acc_empty + 8 * b, 4);  // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const uint64_t nt = (uint64_t)p.n_tiles;

  if (warp == 0) {
    const uint64_t stream_policy = l2_evict_first();
    const uint8_t* const d0 = p.gstash + grad_region_offset(kGradL0, nt);
    const uint8_t* const d5 = p.gstash + grad_region_offset(kGradL5, nt);
    const uint8_t* const dc0 = p.gstash + grad_region_offset(kGradC0, nt);
    uint32_t stage = 0, phase = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      for (int pp = p_begin; pp < p_end; ++pp) {
        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
        if (elect_one()) {
          const uint8_t* src = pp < kPosPanels ? (pp < 4 ? d0 : d5) + (uint64_t)tile * kActBytes
                                               : dc0 + (uint64_t)tile * grad_region_tile_bytes(kGradC0);
          src += (uint32_t)(pp & 3) * kPanelBytes128;
          mbar_arrive_expect_tx(bar_full + 8 * stage, kPanelBytes128);
          bulk_g2s_hint(smem_base + kOffRing + stage * kPanelBytes128, src, kPanelBytes128, bar_full + 8 * stage, stream_policy);
        }
        __syncwarp();
        if (++stage == kRingStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc_pos = make_idesc(128, 64, kF16, kF16, 0, 0);
    constexpr uint32_t idesc_dir = make_idesc(128, 32, kF16, kF16, 0, 0);
    uint32_t stage = 0, phase = 0, acc_phase[2] = {0, 0};
    int buf = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      mbar_wait(bar_acc_empty + 8 * buf, acc_phase[buf] ^ 1);
      acc_phase[buf] ^= 1;
      tc_fence_after();
      for (int pp = p_begin; pp < p_end; ++pp) {
        mbar_wait(bar_full + 8 * stage, phase);
        tc_fence_after();
        if (elect_one()) {
          const bool pos = pp < kPosPanels;
          const uint32_t d_tmem = tmem_base + buf * kAccStride + (pos ? 0u : kAccDir);
          const uint32_t b_panel = pos ? smem_base + (pp < 4 ? kOffW0 : kOffW5) + (uint32_t)(pp & 3) * kPosPanelBytes
                                       : smem_base + kOffWc0 + (uint32_t)(pp - kPosPanels) * kDirPanelBytes;
          const uint32_t a_panel = smem_base + kOffRing + stage * kPanelBytes128;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma(d_tmem, desc_kmajor(a_panel, ks), desc_kmajor(b_panel, ks), pos ? idesc_pos : idesc_dir,
                 (ks != 0 || (pp != 0 && pp != kPosPanels)) ? 1u : 0u);
          umma_commit(bar_empty + 8 * stage);
          if (pp == p_end - 1) umma_commit(bar_acc_full + 8 * buf);
        }
        __syncwarp();
        if (++stage == kRingStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      buf ^= 1;
    }
  } else {
    const uint32_t wq = (uint32_t)(warp & 3);
    const int row = 32 * (int)wq + lane;
    const uint32_t t_row = tmem_base + (wq * 32u << 16);
    uint32_t acc_phase[2] = {0, 0};
    int buf = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      mbar_wait(bar_acc_full + 8 * buf, acc_phase[buf]);
      acc_phase[buf] ^= 1;
      tc_fence_after();
      // g[c] = dL/d(encoded feature c), times the loss scale
      uint32_t gx0[32], gx1[32], gd[32];
      const uint32_t t_acc = t_row + buf * kAccStride;
      if (want_pos) {
        tmem_ld32(t_acc, gx0);
        tmem_ld32(t_acc + 32, gx1);
        tmem_ld_wait32(gx0);
        tmem_ld_wait32(gx1);
      }
      if (want_dir) {
        tmem_ld32(t_acc + kAccDir, gd);
        tmem_ld_wait32(gd);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty + 8 * buf);
      buf ^= 1;

      const int64_t e = (int64_t)tile * kTile + row;
      if (e >= p.n) continue;
      // d/dv of [v, cos(2^k v), sin(2^k v)] (cos block, then sin block): dv = g_v + sum_k 2^k (cos_k g_sin_k - sin_k g_cos_k)
      if (want_pos) {
        auto g = [&](int c) { return __uint_as_float(c < 32 ? gx0[c] : gx1[c - 32]); };
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          float cs[20];
          encode_axis(__ldg(p.positions + 3 * e + i), 10, cs);
          float dv = g(i);
#pragma unroll
          for (int k = 0; k < 10; ++k)
            dv = fmaf((float)(1 << k), cs[k] * g(3 + 20 * i + 10 + k) - cs[10 + k] * g(3 + 20 * i + k), dv);
          p.d_positions[3 * e + i] = dv * p.inv_scale;
        }
      }
      if (want_dir) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          float cs[8];
          encode_axis(__ldg(p.directions + 3 * e + i), 4, cs);
          float dv = __uint_as_float(gd[i]);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            dv = fmaf((float)(1 << k), cs[k] * __uint_as_float(gd[3 + 8 * i + 4 + k]) - cs[4 + k] * __uint_as_float(gd[3 + 8 * i + k]), dv);
          p.d_directions[3 * e + i] = dv * p.inv_scale;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

}  // namespace nerf

extern "C" int nerf_mlp_backward_inputs(float* d_positions, float* d_directions, const void* workspace, const float* params,
                                        const float* positions, const float* directions, int64_t n_samples, float grad_scale,
                                        void* stream) {
  using namespace nerf;
  NERF_CHECK_ARG(n_samples >= 0, "mlp_backward_inputs: n_samples must be >= 0");
  if (n_samples == 0) return 0;
  NERF_CHECK_ARG(n_samples < (int64_t(1) << 31) - kTile, "mlp_backward_inputs: n_samples must be < 2^31 - 128 per call");
  NERF_CHECK_ARG(workspace && params, "mlp_backward_inputs: null workspace or params");
  NERF_CHECK_ARG(d_positions == nullptr || positions != nullptr, "mlp_backward_inputs: d_positions needs positions");
  NERF_CHECK_ARG(d_directions == nullptr || directions != nullptr, "mlp_backward_inputs: d_directions needs directions");
  NERF_CHECK_ARG(grad_scale > 0.f && grad_scale <= 3.4e38f, "mlp_backward_inputs: grad_scale must be positive and finite");
  NERF_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 127) == 0, "mlp_backward_inputs: workspace must be 128-byte aligned");
  if (d_positions == nullptr && d_directions == nullptr) return 0;
  DinputParams p;
  p.d_positions = d_positions;
  p.d_directions = d_directions;
  p.gstash = static_cast<const uint8_t*>(workspace);
  p.params = params;
  p.positions = positions;
  p.directions = directions;
  p.n = n_samples;
  p.n_tiles = (int)((n_samples + kTile - 1) / kTile);
  p.inv_scale = 1.f / grad_scale;
  static bool smem_set[kMaxDevices] = {};
  const cudaError_t e = set_max_dynamic_smem_once(smem_set, {(const void*)mlp_dinput_kernel}, dinput::kSmemBytes);
  NERF_CHECK_ARG(e == cudaSuccess, "mlp_backward_inputs: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  const int grid = p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs;
  mlp_dinput_kernel<<<grid, dinput::kThreads, dinput::kSmemBytes, static_cast<cudaStream_t>(stream)>>>(p);
  NERF_CHECK_LAUNCH("mlp_dinput_kernel");
  return 0;
}
