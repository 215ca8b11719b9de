// mlp_wgrad.cu -- K4b: weight and bias gradients of the NeRF MLP, layer-major.
//
// dW_l[n][k] = sum_m dY_l[m][n] * X_l[m][k] is a GEMM whose reduction runs over ALL samples, so it
// cannot live inside the per-tile chain (a 256x256 fp32 dW is the whole TMEM of an SM).  Instead the
// chain kernels stash dY_l (mlp_bwd.cu) and X_l (mlp_fwd.cu) as 128B-swizzled tile images, and this
// kernel re-reads them: the very same bytes that were K-major A operands in the chain are MN-major
// operands here (tc.cuh), so both operands arrive by 1-D bulk copy with no transposition.
// Each CTA owns one (job, tile range): it streams half tiles (64 samples) through a 3-stage
// shared-memory ring, accumulates the full dW block in TMEM (up to 512 columns), sums dY columns on
// CUDA cores for the bias gradient, and flushes once with fp32 atomics into the flat gradient buffer.
// HBM-bound by construction: ~1 KB of operands per sample and layer (DESIGN.md).
#include "common.cuh"
#include "mlp_layout.cuh"
#include "tc.cuh"
#include "../../include/nerf_b200.h"

namespace nerf {
using namespace tc;

namespace wg {
constexpr int kThreads = 256;  // warp 0 producer, warp 1 MMA, warp 2 TMEM alloc, warps 4-7 reduce + flush
constexpr int kMaxStages = 8;
constexpr uint32_t kHalfPanel = 8192;       // 64 rows x 128 B
constexpr uint32_t kRingBytes = 24 * kHalfPanel;  // 192 KB, carved into as many stages as the job's operands allow
constexpr uint32_t kOffBars = kRingBytes;
constexpr uint32_t kSmemBytes = kOffBars + 256 + 1024;
constexpr int kNumJobs = 13;

struct Seg {
  int16_t buf;        // 0 = gradient stash, 1 = activation stash
  int16_t region;
  int16_t panels;     // 64-column panels used (0 = segment absent)
  int16_t valid;      // valid columns
  int32_t out_col;    // first output column of this segment in dW
};
struct Job {
  Seg a;              // dY (rows of dW); for head jobs: the activation (columns of the tiny dW^T)
  Seg b[2];           // X segments
  int64_t w_off;      // dW offset in the flat gradient buffer (floats)
  int32_t ld;         // dW row length
  int64_t bias_off;   // bias gradient offset, or -1
  int32_t head;       // 0 normal; 1 = colour head (dW_c1^T); 2 = density head
  int32_t ctas;       // CTAs assigned to this job
};

using L = ParamLayout;
constexpr Seg seg(int buf, int region, int panels, int valid, int out_col) { return Seg{(int16_t)buf, (int16_t)region, (int16_t)panels, (int16_t)valid, out_col}; }
constexpr Seg none() { return Seg{0, 0, 0, 0, 0}; }
constexpr int gl(int l) { return kGradL7 + (7 - l); }   // gradient-stash region of hidden layer l
constexpr int hx(int l) { return kStashH0 + l; }        // activation-stash region of h_l

__constant__ Job c_jobs[kNumJobs] = {
    {seg(0, gl(1), 4, 256, 0), {seg(1, hx(0), 4, 256, 0), none()}, L::hidden_w(1), 256, L::hidden_b(1), 0, 13},
    {seg(0, gl(2), 4, 256, 0), {seg(1, hx(1), 4, 256, 0), none()}, L::hidden_w(2), 256, L::hidden_b(2), 0, 13},
    {seg(0, gl(3), 4, 256, 0), {seg(1, hx(2), 4, 256, 0), none()}, L::hidden_w(3), 256, L::hidden_b(3), 0, 13},
    {seg(0, gl(4), 4, 256, 0), {seg(1, hx(3), 4, 256, 0), none()}, L::hidden_w(4), 256, L::hidden_b(4), 0, 13},
    {seg(0, gl(5), 4, 256, 0), {seg(1, hx(4), 4, 256, 0), none()}, L::kW5, 319, L::kB5, 0, 13},
    {seg(0, gl(6), 4, 256, 0), {seg(1, hx(5), 4, 256, 0), none()}, L::hidden_w(6), 256, L::hidden_b(6), 0, 13},
    {seg(0, gl(7), 4, 256, 0), {seg(1, hx(6), 4, 256, 0), none()}, L::hidden_w(7), 256, L::hidden_b(7), 0, 13},
    {seg(0, kGradF, 4, 256, 0), {seg(1, hx(7), 4, 256, 0), none()}, L::kWF, 256, L::kBF, 0, 13},
    {seg(0, gl(0), 4, 256, 0), {seg(1, kStashEnc, 1, 63, 0), none()}, L::kW0, 63, L::kB0, 0, 9},
    {seg(0, gl(5), 4, 256, 0), {seg(1, kStashEnc, 1, 63, 256), none()}, L::kW5, 319, -1, 0, 8},
    {seg(0, kGradC0, 2, 128, 0), {seg(1, kStashF, 4, 256, 0), seg(1, kStashDir, 1, 27, 256)}, L::kWC0, 283, L::kBC0, 0, 12},
    {seg(1, kStashG, 2, 128, 0), {seg(0, kGradHead, 1, 4, 0), none()}, L::kWC1, 128, L::kBC1, 1, 6},
    {seg(1, hx(7), 4, 256, 0), {seg(0, kGradHead, 1, 4, 0), none()}, L::kWS, 256, L::kBS, 2, 9},
};
}  // namespace wg

__global__ void __launch_bounds__(wg::kThreads, 1) mlp_wgrad_kernel(float* __restrict__ grads, const uint8_t* __restrict__ stash,
                                                                     const uint8_t* __restrict__ gstash, int n_tiles, float inv_scale) {
  using namespace wg;
  // ---- which (job, part) is this CTA? ----
  int job_idx = 0, part = (int)blockIdx.x;
  while (job_idx < kNumJobs && part >= c_jobs[job_idx].ctas) part -= c_jobs[job_idx++].ctas;
  if (job_idx >= kNumJobs) return;
  const Job& job = c_jobs[job_idx];
  const int parts = job.ctas;
  const int tile_lo = (int)((int64_t)n_tiles * part / parts), tile_hi = (int)((int64_t)n_tiles * (part + 1) / parts);
  const int n_steps = 2 * (tile_hi - tile_lo);  // half tiles
  if (n_steps <= 0) return;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = smem_base + kOffBars;
  const uint32_t bar_full = bars, bar_empty = bars + 8 * kMaxStages, bar_done = bars + 16 * kMaxStages, tmem_slot = bar_done + 8;
  // jobs with small operands (head, encoding) get more, smaller stages: every job keeps ~190 KB of loads in flight,
  // otherwise those CTAs are latency-bound and finish long after the 64 KB-per-stage jobs (measured: SMs 58 % active)
  const uint32_t kStageBytes = (uint32_t)(job.a.panels + job.b[0].panels + job.b[1].panels) * kHalfPanel;
  const int kStages = (int)(kRingBytes / kStageBytes) < kMaxStages ? (int)(kRingBytes / kStageBytes) : kMaxStages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kMaxStages; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 2);  // MMA commit + reducer group
    }
    mbar_init(bar_done, 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const uint64_t nt = (uint64_t)n_tiles;
  const int na = job.a.panels;
  const int nb0 = job.b[0].panels, nb1 = job.b[1].panels;
  const int halves = na / 2;
  const int n_total = 64 * (nb0 + nb1);  // TMEM columns per M' half

  auto region_ptr = [&](const Seg& s, int tile) -> const uint8_t* {
    return s.buf == 0 ? gstash + grad_region_offset(s.region, nt) + (uint64_t)tile * grad_region_tile_bytes(s.region)
                      : stash + stash_region_offset(s.region, nt) + (uint64_t)tile * stash_region_tile_bytes(s.region);
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      const uint64_t stream_policy = l2_evict_first();
      // per-segment source cursors, computed once: the region tables are runtime loops and one thread issues
      // every copy of this CTA (measured: with the lookups inside the loop the producer was 75 % issue-busy and
      // the kernel ran at 4.3 TB/s; DESIGN.md "K4b")
      const Seg* segs[3] = {&job.a, &job.b[0], &job.b[1]};
      const uint8_t* cur[3];
      uint32_t tile_stride[3];
      int panels[3];
      for (int s = 0; s < 3; ++s) {
        panels[s] = segs[s]->panels;
        cur[s] = region_ptr(*segs[s], tile_lo);
        tile_stride[s] = segs[s]->buf == 0 ? grad_region_tile_bytes(segs[s]->region) : stash_region_tile_bytes(segs[s]->region);
      }
      const uint32_t stage_bytes = (uint32_t)(na + nb0 + nb1) * kHalfPanel;
      for (int step = 0; step < n_steps; ++step) {
        const uint32_t half_off = (step & 1) * kHalfPanel;
        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
        mbar_arrive_expect_tx(bar_full + 8 * stage, stage_bytes);
        uint32_t dst = smem_base + stage * kStageBytes;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          const uint8_t* src = cur[s] + half_off;
          for (int pp = 0; pp < panels[s]; ++pp) {
            bulk_g2s_hint(dst, src, kHalfPanel, bar_full + 8 * stage, stream_policy);
            dst += kHalfPanel;
            src += kPanelBytes128;
          }
          if (step & 1) cur[s] += tile_stride[s];
        }
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      const uint32_t idesc_b0 = make_idesc(128, 64 * nb0, kF16, kF16, 1, 1);
      const uint32_t idesc_b1 = make_idesc(128, 64, kF16, kF16, 1, 1);
      for (int step = 0; step < n_steps; ++step) {
        mbar_wait(bar_full + 8 * stage, phase);
        tc_fence_after();
        const uint32_t sa = smem_base + stage * kStageBytes;
        const uint32_t sb0 = sa + na * kHalfPanel, sb1 = sb0 + nb0 * kHalfPanel;
        for (int hm = 0; hm < halves; ++hm) {
          const uint32_t d0 = tmem_base + hm * n_total;
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t da = desc_mnmajor(sa + hm * 2 * kHalfPanel, ks, kHalfPanel);
            umma(d0, da, desc_mnmajor(sb0, ks, kHalfPanel), idesc_b0, (step | ks) != 0);
            if (nb1 > 0) umma(d0 + 64 * nb0, da, desc_mnmajor(sb1, ks, kHalfPanel), idesc_b1, (step | ks) != 0);
          }
        }
        umma_commit(bar_empty + 8 * stage);
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      umma_commit(bar_done);
    }
  } else if (warp >= 4) {
    // ---- bias reduction: column sums of the dY operand over every half tile ----
    const int t = threadIdx.x - 128;  // 0..127
    const bool head = job.head != 0;
    const int bias_cols = head ? 4 : (job.bias_off >= 0 ? 64 * na : 0);
    const uint32_t bias_seg_off = head ? na * kHalfPanel : 0;  // head jobs: dY is operand B
    float s0 = 0.f, s1 = 0.f;
    uint32_t stage = 0, phase = 0;
    for (int step = 0; step < n_steps; ++step) {
      mbar_wait(bar_full + 8 * stage, phase);
      if (2 * t < bias_cols) {
        const int c = 2 * t;
        const uint32_t base = smem_base + stage * kStageBytes + bias_seg_off + (c >> 6) * kHalfPanel;
#pragma unroll 8
        for (int r = 0; r < 64; ++r) {
          uint32_t w;
          asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w) : "r"(base + panel_offset(r, c & 63)));
          const float2 f = __half22float2(*reinterpret_cast<__half2*>(&w));
          s0 += f.x;
          s1 += f.y;
        }
      }
      named_bar_sync(1, 128);
      if (t == 0) mbar_arrive(bar_empty + 8 * stage);
      if (++stage == kStages) {
        stage = 0;
        phase ^= 1;
      }
    }
    if (2 * t < bias_cols) {
      if (!head) {
        atomicAdd(grads + job.bias_off + 2 * t, s0 * inv_scale);
        atomicAdd(grads + job.bias_off + 2 * t + 1, s1 * inv_scale);
      } else if (job.head == 1) {  // colour head: cols 0..2 -> b_c1
        if (t == 0) {
          atomicAdd(grads + job.bias_off + 0, s0 * inv_scale);
          atomicAdd(grads + job.bias_off + 1, s1 * inv_scale);
        } else {
          atomicAdd(grads + job.bias_off + 2, s0 * inv_scale);
        }
      } else if (t == 1) {  // density head: col 3 -> b_sigma
        atomicAdd(grads + job.bias_off, s1 * inv_scale);
      }
    }
    // ---- flush the accumulated dW block ----
    mbar_wait(bar_done, 0);
    tc_fence_after();
    const int wq = warp & 3;
    const int n_local = wq * 32 + lane;
    for (int hm = 0; hm < halves; ++hm) {
      const int n = hm * 128 + n_local;  // row of dW (normal) / input feature k (head)
      const uint32_t t_row = tmem_base + hm * n_total + (static_cast<uint32_t>(wq * 32) << 16);
      if (head) {
        uint32_t v[32];
        tmem_ld32(t_row, v);
        tmem_ld_wait();
        if (job.head == 1) {
#pragma unroll
          for (int j = 0; j < 3; ++j) atomicAdd(grads + job.w_off + j * 128 + n, __uint_as_float(v[j]) * inv_scale);
        } else {
          atomicAdd(grads + job.w_off + n, __uint_as_float(v[3]) * inv_scale);
        }
        continue;
      }
      float* wrow = grads + job.w_off + (int64_t)n * job.ld;
      for (int s = 0; s < 2; ++s) {
        const Seg& sg = job.b[s];
        if (sg.panels == 0) continue;
        const int col_base = s == 0 ? 0 : 64 * nb0;
        for (int c0 = 0; c0 < 64 * sg.panels; c0 += 32) {
          if (c0 >= sg.valid) break;
          uint32_t v[32];
          tmem_ld32(t_row + col_base + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (c0 + j < sg.valid) atomicAdd(wrow + sg.out_col + c0 + j, __uint_as_float(v[j]) * inv_scale);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

int launch_wgrad(float* grads, const uint8_t* stash, const uint8_t* gstash, int n_tiles, float inv_scale, cudaStream_t stream) {
  static bool smem_set[kMaxDevices] = {};
  const cudaError_t e = set_max_dynamic_smem_once(smem_set, {(const void*)mlp_wgrad_kernel}, wg::kSmemBytes);
  NERF_CHECK_ARG(e == cudaSuccess, "mlp_backward: cudaFuncSetAttribute(wgrad) failed: %s", cudaGetErrorString(e));
  mlp_wgrad_kernel<<<kNumSMs, wg::kThreads, wg::kSmemBytes, stream>>>(grads, stash, gstash, n_tiles, inv_scale);
  NERF_CHECK_LAUNCH("mlp_wgrad_kernel");
  return 0;
}

}  // namespace nerf
