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
//
// K4r, the ray-layout instantiation (render_rays): the samples of a pass are laid out as in K3, sample e at depth z[e]
// on ray e / S, and the epilogue rebuilds x = o + d z as K3 does.  Per ray it reduces, over the ray's samples,
//   dL/do = sum_s dL/dx_s,  dL/dd = sum_s z_s dL/dx_s + d / |d|^2 sum_s sigma_s dL/dsigma_s,  dL/dv = sum_s dL/dv_s
// (the last term: sigma and |d| enter compositing only as sigma delta with delta = dz |d|).  The reduction is a segmented
// warp scan over the tile's rows plus the warp-boundary pieces in shared memory, in a fixed order.  A ray that lies in
// one tile is added to the outputs directly; the pieces of a ray cut by tile edges go to a per-tile scratch (head: the
// ray that started in an earlier tile, tail: the one that continues into a later tile), which ray_fixup_kernel adds up
// in tile order.  No float atomics: the result depends neither on gridDim nor on which CTA ran which tile.
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
  // ray mode: positions / directions above are the rays' origins / view directions ([n_rays][3]) and d_positions /
  // d_directions accumulate their gradients
  float* d_dirs;  // nullptr: skipped
  const float* dirs;
  const float* z;
  const float4* rgbsigma;
  const float4* d_rgbsigma;
  float* partials;  // [n_tiles][2][kRayGrads]: head, tail piece
  int n_samples;    // S
};

namespace dinput {
constexpr int kRayGrads = 9;  // dL/do, dL/dd, dL/dv of one ray (or of the piece of it one tile holds)
}

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

// Adds one ray's (dL/do, dL/dd, dL/dv), times the loss scale, to the requested ray-mode outputs.
__device__ __forceinline__ void add_ray_grads(const DinputParams& p, int64_t ray, const float (&g)[dinput::kRayGrads]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    if (p.d_positions) p.d_positions[3 * ray + i] += g[i] * p.inv_scale;
    if (p.d_dirs) p.d_dirs[3 * ray + i] += g[3 + i] * p.inv_scale;
    if (p.d_directions) p.d_directions[3 * ray + i] += g[6 + i] * p.inv_scale;
  }
}

// K4r epilogue of one tile, run by all 128 epilogue threads (rows past the last sample too: they take part in the
// shuffles and the barrier).  gx0 / gx1 / gd: this row's accumulators dL/d enc(x), dL/d enc(v), times the loss scale.
// `parity` alternates from tile to tile, so one barrier per tile keeps a tile's writes of warp_tail apart from the reads
// of the tile before.
__device__ __forceinline__ void ray_tile_epilogue(const DinputParams& p, int tile, int wq, int lane, const uint32_t (&gx0)[32],
                                                  const uint32_t (&gx1)[32], const uint32_t (&gd)[32], bool want_pos,
                                                  bool want_dir, int parity) {
  using namespace dinput;
  __shared__ float warp_tail[2][4][10];  // each warp's scan value at its last row
  const int row = 32 * wq + lane;
  const int64_t e0 = (int64_t)tile * kTile;
  auto ray_of = [&](int r) { return e0 + r < p.n ? (int)(e0 + r) / p.n_samples : INT_MAX; };
  const int64_t e = e0 + row;
  const int ray = ray_of(row);
  // v: dL/dx (0-2), z dL/dx (3-5), dL/dv (6-8), sigma dL/dsigma (9) of this sample
  float v[10];
#pragma unroll
  for (int j = 0; j < 10; ++j) v[j] = 0.f;
  if (e < p.n && want_pos) {
    auto g = [&](int c) { return __uint_as_float(c < 32 ? gx0[c] : gx1[c - 32]); };
    const float zz = __ldg(p.z + e);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      float cs[20];
      encode_axis(ray_point(__ldg(p.positions + 3 * ray + i), __ldg(p.dirs + 3 * ray + i), zz), 10, cs);
      float dv = g(i);
#pragma unroll
      for (int k = 0; k < 10; ++k)
        dv = fmaf((float)(1 << k), cs[k] * g(3 + 20 * i + 10 + k) - cs[10 + k] * g(3 + 20 * i + k), dv);
      v[i] = dv;
      v[3 + i] = zz * dv;
    }
    if (p.d_dirs) v[9] = __ldg(&p.rgbsigma[e].w) * __ldg(&p.d_rgbsigma[e].w);
  }
  if (e < p.n && want_dir) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      float cs[8];
      encode_axis(__ldg(p.directions + 3 * ray + i), 4, cs);
      float dv = __uint_as_float(gd[i]);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        dv = fmaf((float)(1 << k), cs[k] * __uint_as_float(gd[3 + 8 * i + 4 + k]) - cs[4 + k] * __uint_as_float(gd[3 + 8 * i + k]), dv);
      v[6 + i] = dv;
    }
  }
  // segmented inclusive scan over the warp's rows (ray ids do not decrease along the rows)
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int up_ray = __shfl_up_sync(0xffffffffu, ray, off);  // every lane must take part in the shuffle
    const bool same = lane >= off && up_ray == ray;
#pragma unroll
    for (int j = 0; j < 10; ++j) {
      const float u = __shfl_up_sync(0xffffffffu, v[j], off);
      if (same) v[j] += u;
    }
  }
  if (lane == 31) {
#pragma unroll
    for (int j = 0; j < 10; ++j) warp_tail[parity][wq][j] = v[j];
  }
  named_bar_sync(1, 128);
  if (e >= p.n || (row < kTile - 1 && ray_of(row + 1) == ray)) return;
  // this row ends its ray's piece of the tile: add the pieces of the earlier warps, nearest first
  for (int w = wq - 1; w >= 0 && ray_of(32 * w + 31) == ray; --w) {
#pragma unroll
    for (int j = 0; j < 10; ++j) v[j] += warp_tail[parity][w][j];
  }
  float g[kRayGrads];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    g[i] = v[i];
    g[3 + i] = v[3 + i];
    g[6 + i] = v[6 + i];
  }
  if (p.d_dirs) {
    const float dx = __ldg(p.dirs + 3 * ray), dy = __ldg(p.dirs + 3 * ray + 1), dz = __ldg(p.dirs + 3 * ray + 2);
    const float n2 = dx * dx + dy * dy + dz * dz;
    const float c = n2 > 0.f ? v[9] / n2 : 0.f;
    g[3] = fmaf(dx, c, g[3]);
    g[4] = fmaf(dy, c, g[4]);
    g[5] = fmaf(dz, c, g[5]);
  }
  const int64_t first = (int64_t)ray * p.n_samples, last = first + p.n_samples;
  if (first >= e0 && last <= e0 + kTile) {
    add_ray_grads(p, ray, g);
  } else {
    float* dst = p.partials + ((int64_t)tile * 2 + (first < e0 ? 0 : 1)) * kRayGrads;
#pragma unroll
    for (int j = 0; j < kRayGrads; ++j) dst[j] = g[j];
  }
}

// K4r second pass, one thread per ray: a ray cut by tile edges is the tail piece of its first tile plus the head pieces
// of the tiles after it, added in tile order.
__global__ void __launch_bounds__(256) ray_fixup_kernel(const DinputParams p) {
  using namespace dinput;
  const int64_t ray = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (ray >= p.n / p.n_samples) return;
  const int64_t first = ray * p.n_samples;
  const int64_t t0 = first / kTile, t1 = (first + p.n_samples - 1) / kTile;
  if (t0 == t1) return;  // added by mlp_dinput_kernel
  float g[kRayGrads];
#pragma unroll
  for (int j = 0; j < kRayGrads; ++j) g[j] = p.partials[(t0 * 2 + 1) * kRayGrads + j];
  for (int64_t t = t0 + 1; t <= t1; ++t) {
#pragma unroll
    for (int j = 0; j < kRayGrads; ++j) g[j] += p.partials[t * 2 * kRayGrads + j];
  }
  add_ray_grads(p, ray, g);
}

// kRays = false: NeRFBlock layout (K4c), one point per sample; true: render_rays layout (K4r), see the top of the file.
template <bool kRays>
__global__ void __launch_bounds__(dinput::kThreads, 1) mlp_dinput_kernel(const DinputParams p) {
  using namespace dinput;
  using L = ParamLayout;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = smem_base + kOffBars, bar_empty = bar_full + 8 * kRingStages;
  const uint32_t bar_acc_full = bar_empty + 8 * kRingStages, bar_acc_empty = bar_acc_full + 16, tmem_slot = bar_acc_empty + 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool want_pos = p.d_positions != nullptr || (kRays && p.d_dirs != nullptr), want_dir = p.d_directions != nullptr;
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
    int buf = 0, parity = 0;
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

      if constexpr (kRays) {
        ray_tile_epilogue(p, tile, (int)wq, lane, gx0, gx1, gd, want_pos, want_dir, parity);
        parity ^= 1;
        continue;
      }
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
  DinputParams p{};
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
  const cudaError_t e = set_max_dynamic_smem_once(smem_set, {(const void*)mlp_dinput_kernel<false>}, dinput::kSmemBytes);
  NERF_CHECK_ARG(e == cudaSuccess, "mlp_backward_inputs: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  const int grid = p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs;
  mlp_dinput_kernel<false><<<grid, dinput::kThreads, dinput::kSmemBytes, static_cast<cudaStream_t>(stream)>>>(p);
  NERF_CHECK_LAUNCH("mlp_dinput_kernel");
  return 0;
}

extern "C" size_t nerf_mlp_backward_rays_scratch_bytes(int n_rays, int n_samples) {
  if (n_rays <= 0 || n_samples <= 0) return 0;
  const int64_t n_tiles = ((int64_t)n_rays * n_samples + nerf::kTile - 1) / nerf::kTile;
  return (size_t)n_tiles * 2 * nerf::dinput::kRayGrads * sizeof(float);
}

extern "C" int nerf_mlp_backward_rays(float* d_origins, float* d_dirs, float* d_viewdirs, void* scratch, const void* workspace,
                                      const float* params, const float* origins, const float* dirs, const float* viewdirs,
                                      const float* z, const float* rgbsigma, const float* d_rgbsigma, int n_rays,
                                      int n_samples, float grad_scale, void* stream) {
  using namespace nerf;
  NERF_CHECK_ARG(n_rays >= 0 && n_samples >= 0, "mlp_backward_rays: n_rays and n_samples must be >= 0");
  if (n_rays == 0) return 0;
  NERF_CHECK_ARG(n_samples >= 1, "mlp_backward_rays: n_samples must be >= 1");
  const int64_t n = (int64_t)n_rays * n_samples;
  NERF_CHECK_ARG(n < (int64_t(1) << 31) - kTile, "mlp_backward_rays: n_rays * n_samples must be < 2^31 - 128 per call");
  NERF_CHECK_ARG(workspace && params, "mlp_backward_rays: null workspace or params");
  NERF_CHECK_ARG((d_origins == nullptr && d_dirs == nullptr) || (origins && dirs && z),
                 "mlp_backward_rays: d_origins / d_dirs need origins, dirs and z");
  NERF_CHECK_ARG(d_dirs == nullptr || (rgbsigma && d_rgbsigma), "mlp_backward_rays: d_dirs needs rgbsigma and d_rgbsigma");
  NERF_CHECK_ARG(d_viewdirs == nullptr || viewdirs != nullptr, "mlp_backward_rays: d_viewdirs needs viewdirs");
  NERF_CHECK_ARG(grad_scale > 0.f && grad_scale <= 3.4e38f, "mlp_backward_rays: grad_scale must be positive and finite");
  NERF_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 127) == 0, "mlp_backward_rays: workspace must be 128-byte aligned");
  if (d_origins == nullptr && d_dirs == nullptr && d_viewdirs == nullptr) return 0;
  NERF_CHECK_ARG(scratch && (reinterpret_cast<uintptr_t>(scratch) & 3) == 0,
                 "mlp_backward_rays: scratch must be a 4-byte aligned buffer of nerf_mlp_backward_rays_scratch_bytes()");
  DinputParams p{};
  p.d_positions = d_origins;
  p.d_directions = d_viewdirs;
  p.d_dirs = d_dirs;
  p.gstash = static_cast<const uint8_t*>(workspace);
  p.params = params;
  p.positions = origins;
  p.directions = viewdirs;
  p.dirs = dirs;
  p.z = z;
  p.rgbsigma = reinterpret_cast<const float4*>(rgbsigma);
  p.d_rgbsigma = reinterpret_cast<const float4*>(d_rgbsigma);
  p.partials = static_cast<float*>(scratch);
  p.n = n;
  p.n_samples = n_samples;
  p.n_tiles = (int)((n + kTile - 1) / kTile);
  p.inv_scale = 1.f / grad_scale;
  static bool smem_set[kMaxDevices] = {};
  const cudaError_t e = set_max_dynamic_smem_once(smem_set, {(const void*)mlp_dinput_kernel<true>}, dinput::kSmemBytes);
  NERF_CHECK_ARG(e == cudaSuccess, "mlp_backward_rays: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int grid = p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs;
  mlp_dinput_kernel<true><<<grid, dinput::kThreads, dinput::kSmemBytes, s>>>(p);
  NERF_CHECK_LAUNCH("mlp_dinput_kernel<true>");
  if (kTile % n_samples != 0) {  // otherwise no ray crosses a tile edge
    ray_fixup_kernel<<<(unsigned)((n_rays + 255) / 256), 256, 0, s>>>(p);
    NERF_CHECK_LAUNCH("ray_fixup_kernel");
  }
  return 0;
}
