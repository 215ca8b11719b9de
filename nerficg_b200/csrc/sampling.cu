// sampling.cu -- K1 stratified sampling and K2 inverse-CDF importance sampling + merge.
// Both are HBM-bound, warp-level kernels (no tensor cores): K1 is elementwise, K2 assigns one
// warp per ray (segmented prefix sum over the ray's weights, binary search per fine sample,
// in-shared-memory bitonic merge of coarse + fine depths).
#include "common.cuh"
#include "../../include/nerf_b200.h"

namespace nerf {

// ---- K1 -------------------------------------------------------------------------------
// t_k follows torch.linspace's two-sided formula so deterministic depths match bit for bit.
__device__ __forceinline__ float linspace_at(int k, int n, float start, float end, float step) {
  return (k < n / 2) ? __fadd_rn(start, __fmul_rn(step, (float)k)) : __fsub_rn(end, __fmul_rn(step, (float)(n - k - 1)));
}

__device__ __forceinline__ float stratified_at(int k, int n, float near_plane, float far_plane, float step, bool randomize, float uk) {
  const float t = n > 1 ? linspace_at(k, n, near_plane, far_plane, step) : near_plane;
  if (!randomize) return t;
  float lo = t, hi = t;
  if (k > 0) lo = __fmul_rn(0.5f, __fadd_rn(t, linspace_at(k - 1, n, near_plane, far_plane, step)));
  if (k < n - 1) hi = __fmul_rn(0.5f, __fadd_rn(linspace_at(k + 1, n, near_plane, far_plane, step), t));
  return __fadd_rn(lo, __fmul_rn(__fsub_rn(hi, lo), uk));
}

// kVec = 4: n_samples % 4 == 0, one float4 of noise in and one float4 of depths out per item.  Every thread owns four
// items a grid stride apart and issues its four loads before any arithmetic (memory-level parallelism: the kernel is a
// 5-20 us streaming pass, so bytes in flight per SM decide its bandwidth); item indices are 32-bit (host-checked).
template <int kVec>
__global__ void __launch_bounds__(256) stratified_kernel(float* __restrict__ z, const float* __restrict__ u, uint32_t n_items,
                                                         int n_samples, float near_plane, float far_plane) {
  const float step = n_samples > 1 ? (far_plane - near_plane) / (float)(n_samples - 1) : 0.f;
  const uint32_t per_ray = (uint32_t)(n_samples / kVec);
  const uint32_t stride = gridDim.x * blockDim.x;
  const bool randomize = u != nullptr;
  for (uint32_t base = blockIdx.x * blockDim.x + threadIdx.x; base < n_items; base += 4u * stride) {
    if (kVec == 4) {
      float4 uv[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t i = base + k * stride;
        uv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (randomize && i < n_items) uv[k] = __ldcs(reinterpret_cast<const float4*>(u) + i);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t i = base + k * stride;
        if (i >= n_items) break;
        const int k0 = (int)(i % per_ray) * 4;
        float4 o;
        o.x = stratified_at(k0 + 0, n_samples, near_plane, far_plane, step, randomize, uv[k].x);
        o.y = stratified_at(k0 + 1, n_samples, near_plane, far_plane, step, randomize, uv[k].y);
        o.z = stratified_at(k0 + 2, n_samples, near_plane, far_plane, step, randomize, uv[k].z);
        o.w = stratified_at(k0 + 3, n_samples, near_plane, far_plane, step, randomize, uv[k].w);
        reinterpret_cast<float4*>(z)[i] = o;
      }
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t i = base + k * stride;
        if (i >= n_items) break;
        z[i] = stratified_at((int)(i % per_ray), n_samples, near_plane, far_plane, step, randomize, randomize ? __ldg(u + i) : 0.f);
      }
    }
  }
}

// ---- K2 -------------------------------------------------------------------------------
// One warp per ray.  The coarse depths arrive ascending, so instead of sorting the concatenated depths (reference
// Renderer.py:70) the warp sorts only the Nf fine depths (bitonic network in shared memory) and merges the two
// ascending lists by rank: position(coarse i) = i + #{fine < z_c[i]}, position(fine j) = j + #{coarse <= z_f[j]}
// (two binary searches).  The cdf itself is summed by one lane in the reference's order (torch.cumsum on the
// CPU oracle is sequential): samples that land in near-empty bins amplify cdf rounding by 1/pdf (SURVEY hard
// part 7), so a parallel scan would break the 1e-5 parity of exactly those samples.
constexpr int kWarpsPerBlock = 8;

__device__ __forceinline__ float invert_cdf(const float* __restrict__ cdf, const float* __restrict__ edges, int nb, float uj) {
  // first index with cdf > u  (searchsorted right=True); cdf[0] = 0 <= u
  int a = 0, b = nb;
  while (a < b) {
    const int mid = (a + b) >> 1;
    if (cdf[mid] <= uj) a = mid + 1; else b = mid;
  }
  const int below = max(a - 1, 0), above = min(a, nb - 1);
  const float c0 = cdf[below], c1 = cdf[above];
  float den = __fsub_rn(c1, c0);
  if (den < 1e-5f) den = 1.f;
  const float t = __fdiv_rn(__fsub_rn(uj, c0), den);
  const float e0 = edges[below], e1 = edges[above];
  return __fadd_rn(e0, __fmul_rn(t, __fsub_rn(e1, e0)));
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32) importance_kernel_smem(
    float* __restrict__ z_merged, float* __restrict__ z_fine_out, const float* __restrict__ z_coarse,
    const float* __restrict__ w_coarse, const float* __restrict__ u, int n_rays, int nc, int nf, int nf_pad) {
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ray = blockIdx.x * kWarpsPerBlock + warp;
  if (ray >= n_rays) return;  // whole warp exits together; only __syncwarp is used below
  const int nb = nc - 1;      // number of bin edges == number of cdf entries
  const int nv = nc - 2;      // interior weights
  const int s = nc + nf;
  float* cdf = sm + warp * (3 * nb + nc + nf_pad + s);
  float* edges = cdf + nb;
  float* pdf = edges + nb;    // nv entries
  float* zcs = pdf + nb;      // nc coarse depths
  float* fine = zcs + nc;     // nf_pad: noise, sorted in place, then the fine depths
  float* merged = fine + nf_pad;
  const float* zc = z_coarse + (int64_t)ray * nc;
  const float* wc = w_coarse + (int64_t)ray * nc;

  // coarse depths, bin edges (midpoints), pdf numerators
  float part = 0.f;
  for (int j = lane; j < nc; j += 32) {
    const float zj = __ldg(zc + j);
    zcs[j] = zj;
    if (j < nb) edges[j] = __fmul_rn(0.5f, __fadd_rn(zj, __ldg(zc + j + 1)));
    if (j < nv) {
      const float v = __fadd_rn(__ldg(wc + j + 1), 1e-5f);
      pdf[j] = v;
      part += v;
    }
  }
  // noise (or torch.linspace(0, 1, nf), two-sided) -> shared memory, +inf padding for the sort
  const float inv_nf1 = nf > 1 ? 1.f / (float)(nf - 1) : 0.f;
  for (int j = lane; j < nf_pad; j += 32) {
    float uj = __int_as_float(0x7f800000);
    if (j < nf) {
      if (u != nullptr) uj = __ldg(u + (int64_t)ray * nf + j);
      else uj = (j < nf / 2) ? __fmul_rn(inv_nf1, (float)j) : __fsub_rn(1.f, __fmul_rn(inv_nf1, (float)(nf - j - 1)));
    }
    fine[j] = uj;
  }
  const float total = warp_sum(part);
  for (int j = lane; j < nv; j += 32) pdf[j] = __fdiv_rn(pdf[j], total);
  __syncwarp();
  if (lane == 0) {  // sequential running sum, the reference's order
    float run = 0.f;
    cdf[0] = 0.f;
    int j = 0;
    for (; j + 4 <= nv; j += 4) {
      const float p0 = pdf[j], p1 = pdf[j + 1], p2 = pdf[j + 2], p3 = pdf[j + 3];
      run = __fadd_rn(run, p0);
      cdf[j + 1] = run;
      run = __fadd_rn(run, p1);
      cdf[j + 2] = run;
      run = __fadd_rn(run, p2);
      cdf[j + 3] = run;
      run = __fadd_rn(run, p3);
      cdf[j + 4] = run;
    }
    for (; j < nv; ++j) {
      run = __fadd_rn(run, pdf[j]);
      cdf[j + 1] = run;
    }
  }
  __syncwarp();
  // invert the cdf for every fine sample (in the caller's noise order), then sort the DEPTHS: they are a monotone
  // function of the noise only up to the last bit at bin boundaries, and the output must be exactly sorted
  for (int j = lane; j < nf; j += 32) {
    const float zf = invert_cdf(cdf, edges, nb, fine[j]);
    fine[j] = zf;
    if (z_fine_out != nullptr) z_fine_out[(int64_t)ray * nf + j] = zf;
  }
  __syncwarp();
  for (int k = 2; k <= nf_pad; k <<= 1) {  // bitonic network, ascending; +inf padding stays at the end
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = lane; t < (nf_pad >> 1); t += 32) {
        const int pos = 2 * t - (t & (j - 1));
        const int partner = pos + j;
        const float x = fine[pos], y = fine[partner];
        const bool up = (pos & k) == 0;
        if ((x > y) == up) {
          fine[pos] = y;
          fine[partner] = x;
        }
      }
      __syncwarp();
    }
  }
  // merge by rank: position(fine j) = j + #{coarse <= z_f[j]}, position(coarse i) = i + #{fine < z_c[i]}
  for (int j = lane; j < nf; j += 32) {
    const float zf = fine[j];
    int a = 0, b = nc;
    while (a < b) {
      const int mid = (a + b) >> 1;
      if (zcs[mid] <= zf) a = mid + 1; else b = mid;
    }
    merged[j + a] = zf;
  }
  __syncwarp();
  for (int i = lane; i < nc; i += 32) {
    const float zi = zcs[i];
    int a = 0, b = nf;  // #{fine < zi}
    while (a < b) {
      const int mid = (a + b) >> 1;
      if (fine[mid] < zi) a = mid + 1; else b = mid;
    }
    merged[i + a] = zi;
  }
  __syncwarp();
  for (int j = lane; j < s; j += 32) z_merged[(int64_t)ray * s + j] = merged[j];
}

// ---- K2, sorted-noise flavour (n_fine <= 512): the production kernel -----------------------------------
// The inverse cdf is a composition of monotone, correctly rounded operations, so SORTING THE NOISE FIRST gives
// the fine depths already in ascending order.  Compared with sorting the depths after the inversion (the
// shared-memory kernel above, kept for n_fine > 512):
//   * one binary search per LANE (for its first key) followed by monotone advances through the cdf, instead
//     of one binary search per SAMPLE;
//   * no search at all to place fine samples among the coarse ones, and none to place coarse among fine: the two
//     ascending lists are merged by MERGE PATH (every lane binary-searches its diagonal once and then emits
//     ceil(S/32) consecutive outputs sequentially);
//   * the noise is sorted in registers in a BLOCKED layout (lane owns K consecutive keys, loaded as float4):
//     compare-exchange distances below K stay inside the lane, so 15 of the 28 stages of a 128-key network need
//     no shuffle.
// Exactness: the fine depths are checked for sortedness (one shuffle) and re-sorted by the same network in the
// (never observed) case of a violation, so the output is bit-identical to sort(cat(z_c, z_f)).  The sequential cdf
// (the reference's summation order) is kept.
template <int K>
__device__ __forceinline__ void bitonic_sort_blocked(float (&x)[K], int lane) {
  // Ascending-only formulation of the bitonic network over the blocked index e = lane * K + r: every merge of size k
  // starts with a FLIP step (partner e ^ (k - 1)) and continues with plain half-cleaners (partner e ^ j, j = k/4 .. 1);
  // the element with the lower index always keeps the minimum, so no direction flags are needed: an in-lane
  // comparator is two FMNMX, a cross-lane one is SHFL + one FMNMX whose min/max select is a lane predicate.
  constexpr int N = 32 * K;
#pragma unroll
  for (int k = 2; k <= N; k <<= 1) {
    // ---- flip: partner index = e ^ (k - 1)
    if (k <= K) {
#pragma unroll
      for (int r = 0; r < K; ++r) {
        const int r2 = r ^ (k - 1);
        if (r < r2) {
          const float lo = fminf(x[r], x[r2]), hi = fmaxf(x[r], x[r2]);
          x[r] = lo;
          x[r2] = hi;
        }
      }
    } else {
      const int lm = k / K - 1;                 // lane mask of the flip; the register index flips completely (r ^ (K - 1))
      const bool keep_min = (lane & ((lm + 1) >> 1)) == 0;   // lower index <=> the top flipped lane bit is clear
      float y[K];
#pragma unroll
      for (int r = 0; r < K; ++r) y[r] = __shfl_xor_sync(0xffffffffu, x[K - 1 - r], lm);
#pragma unroll
      for (int r = 0; r < K; ++r) x[r] = keep_min ? fminf(x[r], y[r]) : fmaxf(x[r], y[r]);
    }
    // ---- half-cleaners
#pragma unroll
    for (int j = k >> 2; j >= 1; j >>= 1) {
      if (j >= K) {
        const int jl = j / K;
        const bool keep_min = (lane & jl) == 0;
#pragma unroll
        for (int r = 0; r < K; ++r) {
          const float other = __shfl_xor_sync(0xffffffffu, x[r], jl);
          x[r] = keep_min ? fminf(x[r], other) : fmaxf(x[r], other);
        }
      } else {
#pragma unroll
        for (int r = 0; r < K; ++r) {
          if ((r & j) == 0) {
            const int r2 = r | j;
            const float lo = fminf(x[r], x[r2]), hi = fmaxf(x[r], x[r2]);
            x[r] = lo;
            x[r2] = hi;
          }
        }
      }
    }
  }
}

// branch-free searchsorted(right=True) over a cdf padded with +inf to kPad entries: number of entries <= u
template <int kPad>
__device__ __forceinline__ int count_le(const float* __restrict__ cdf, float uj) {
  int a = 0;
#pragma unroll
  for (int step = kPad >> 1; step >= 1; step >>= 1)
    if (cdf[a + step - 1] <= uj) a += step;
  return a;
}

template <int K, int kCdfPad>
__global__ void __launch_bounds__(kWarpsPerBlock * 32) importance_kernel_sorted(
    float* __restrict__ z_merged, float* __restrict__ z_fine_out, const float* __restrict__ z_coarse,
    const float* __restrict__ w_coarse, const float* __restrict__ u, int n_rays, int nc, int nf) {
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ray = blockIdx.x * kWarpsPerBlock + warp;
  const bool active = ray < n_rays;
  const int nb = nc - 1, nv = nc - 2, s = nc + nf;
  // per-warp layout (floats): cdf[kCdfPad] (entries >= nb are +inf), edges[nb], pdf[nb], zcs[nc + 1] (+inf sentinel),
  // fine[32 K + 1] (+inf padding and sentinel), merged[s]
  const int per_warp = kCdfPad + 2 * nb + (nc + 1) + (32 * K + 1) + s;
  float* cdf = sm + warp * per_warp;
  float* edges = cdf + kCdfPad;
  float* pdf = edges + nb;
  float* zcs = pdf + nb;
  float* fine = zcs + nc + 1;
  float* merged = fine + 32 * K + 1;
  const float kInf = __int_as_float(0x7f800000);

  float x[K];
  if (active) {
    const float inv_nf1 = nf > 1 ? 1.f / (float)(nf - 1) : 0.f;
    const int e0 = lane * K;
    if (u != nullptr && K % 4 == 0 && (nf & 3) == 0 && ((reinterpret_cast<uintptr_t>(u) & 15) == 0)) {
#pragma unroll
      for (int q = 0; q < K / 4; ++q) {
        float4 v = make_float4(kInf, kInf, kInf, kInf);
        if (e0 + 4 * q < nf) v = __ldcs(reinterpret_cast<const float4*>(u + (int64_t)ray * nf + e0) + q);
        x[4 * q] = v.x;
        x[4 * q + 1] = v.y;
        x[4 * q + 2] = v.z;
        x[4 * q + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int r = 0; r < K; ++r) {
        const int e = e0 + r;
        float uj = kInf;
        if (e < nf) {
          if (u != nullptr) uj = __ldg(u + (int64_t)ray * nf + e);
          else uj = (e < nf / 2) ? __fmul_rn(inv_nf1, (float)e) : __fsub_rn(1.f, __fmul_rn(inv_nf1, (float)(nf - e - 1)));
        }
        x[r] = uj;
      }
    }
    const float* zc = z_coarse + (int64_t)ray * nc;
    const float* wc = w_coarse + (int64_t)ray * nc;
    float part = 0.f;
    for (int j = lane; j < nc; j += 32) {
      const float zj = __ldg(zc + j);
      zcs[j] = zj;
      if (j < nb) edges[j] = __fmul_rn(0.5f, __fadd_rn(zj, __ldg(zc + j + 1)));
      if (j < nv) {
        const float v = __fadd_rn(__ldg(wc + j + 1), 1e-5f);
        pdf[j] = v;
        part += v;
      }
    }
    for (int j = nb + lane; j < kCdfPad; j += 32) cdf[j] = kInf;
    if (lane == 0) {
      zcs[nc] = kInf;
      fine[32 * K] = kInf;
    }
    const float total = warp_sum(part);
    for (int j = lane; j < nv; j += 32) pdf[j] = __fdiv_rn(pdf[j], total);
  }
  __syncthreads();
  if (warp == 0 && lane < kWarpsPerBlock && blockIdx.x * kWarpsPerBlock + lane < n_rays) {
    // sequential running sums (the reference's order) of the block's rays, one lane per ray: 24 warp instructions per ray
    // instead of ~170 when lane 0 of every warp sums its own ray (measured: the kernel is issue-bound, the block barrier is
    // hidden by the other resident blocks)
    float* c = sm + lane * per_warp;
    const float* pd = c + kCdfPad + nb;
    float run = 0.f;
    c[0] = 0.f;
    for (int j = 0; j < nv; ++j) {
      run = __fadd_rn(run, pd[j]);
      c[j + 1] = run;
    }
  }
  // the noise is sorted while warp 0 sums the cdfs (u == nullptr: the linspace is already ascending)
  if (active && u != nullptr) bitonic_sort_blocked<K>(x, lane);
  __syncthreads();
  if (!active) return;

  // (tests only) the fine depths in the CALLER's noise order
  if (z_fine_out != nullptr) {
    const float inv_nf1 = nf > 1 ? 1.f / (float)(nf - 1) : 0.f;
    for (int e = lane; e < nf; e += 32) {
      float uj;
      if (u != nullptr) uj = __ldg(u + (int64_t)ray * nf + e);
      else uj = (e < nf / 2) ? __fmul_rn(inv_nf1, (float)e) : __fsub_rn(1.f, __fmul_rn(inv_nf1, (float)(nf - e - 1)));
      z_fine_out[(int64_t)ray * nf + e] = invert_cdf(cdf, edges, nb, uj);
    }
  }

  // invert the cdf: fixed-trip branch-free searches (the lanes' ascending keys probe neighbouring addresses: few conflicts)
#pragma unroll
  for (int r = 0; r < K; ++r) {
    const float uj = x[r];
    const int a = min(count_le<kCdfPad>(cdf, uj), nb);
    const int below = max(a - 1, 0), above = min(a, nb - 1);
    const float c0 = cdf[below], c1 = cdf[above];
    float den = __fsub_rn(c1, c0);
    if (den < 1e-5f) den = 1.f;
    const float t = __fdiv_rn(__fsub_rn(uj, c0), den);
    const float e0 = edges[below], e1 = edges[above];
    x[r] = (lane * K + r < nf) ? __fadd_rn(e0, __fmul_rn(t, __fsub_rn(e1, e0))) : kInf;
  }
  // ascending by construction; verified (and repaired by the same network) so that the merge below is exact
  {
    bool bad = false;
#pragma unroll
    for (int r = 1; r < K; ++r) bad |= x[r] < x[r - 1];
    const float prev = __shfl_up_sync(0xffffffffu, x[K - 1], 1);
    bad |= lane > 0 && x[0] < prev;
    if (__any_sync(0xffffffffu, bad)) bitonic_sort_blocked<K>(x, lane);
  }
#pragma unroll
  for (int r = 0; r < K; ++r) fine[lane * K + r] = x[r];
  __syncwarp();

  // merge path: this lane emits outputs [o0, o1) of the merged list (coarse first on ties)
  const int per_lane = (s + 31) >> 5;
  const int o0 = min(lane * per_lane, s), o1 = min(o0 + per_lane, s);
  int lo = max(0, o0 - nf), hi = min(o0, nc);
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (zcs[mid] <= fine[o0 - mid - 1]) lo = mid + 1; else hi = mid;
  }
  {
    // sentinels (+inf behind both lists) make the loop body branch-free: one select, one store, one load per output
    const float* pc = zcs + lo;
    const float* pf = fine + (o0 - lo);
    float ci = *pc, fj = *pf;
    for (int o = o0; o < o1; ++o) {
      const bool take_c = ci <= fj;
      merged[o] = take_c ? ci : fj;
      pc += take_c ? 1 : 0;
      pf += take_c ? 0 : 1;
      const float nxt = *(take_c ? pc : pf);
      ci = take_c ? nxt : ci;
      fj = take_c ? fj : nxt;
    }
  }
  __syncwarp();
  for (int q = lane; q < s; q += 32) z_merged[(int64_t)ray * s + q] = merged[q];
}

}  // namespace nerf

extern "C" int nerf_sample_stratified(float* z, const float* u, int n_rays, int n_samples, float near_plane, float far_plane,
                                      void* stream) {
  using namespace nerf;
  if (n_rays <= 0) return 0;
  NERF_CHECK_ARG(z != nullptr && n_samples >= 1, "sample_stratified: bad arguments");
  const int64_t total = (int64_t)n_rays * n_samples;
  NERF_CHECK_ARG(total < (int64_t(1) << 31), "sample_stratified: n_rays*n_samples must be < 2^31 per call");
  const bool vec = n_samples % 4 == 0 && (reinterpret_cast<uintptr_t>(z) & 15) == 0 && (u == nullptr || (reinterpret_cast<uintptr_t>(u) & 15) == 0);
  const uint32_t items = (uint32_t)(vec ? total / 4 : total);
  const int64_t want = ((int64_t)items + 1023) / 1024, cap = (int64_t)kNumSMs * 16;  // four items per thread
  const int blocks = (int)(want < cap ? want : cap);
  if (vec)
    stratified_kernel<4><<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(z, u, items, n_samples, near_plane, far_plane);
  else
    stratified_kernel<1><<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(z, u, items, n_samples, near_plane, far_plane);
  NERF_CHECK_LAUNCH("stratified_kernel");
  return 0;
}

extern "C" int nerf_sample_importance(float* z_merged, float* z_fine, const float* z_coarse, const float* w_coarse,
                                      const float* u, int n_rays, int n_coarse, int n_fine, void* stream) {
  using namespace nerf;
  if (n_rays <= 0) return 0;
  NERF_CHECK_ARG(z_merged && z_coarse && w_coarse, "sample_importance: null pointer");
  NERF_CHECK_ARG(n_coarse >= 3 && n_coarse <= 512, "sample_importance: n_coarse must be in [3,512], got %d", n_coarse);
  NERF_CHECK_ARG(n_fine >= 1 && n_coarse + n_fine <= 2048, "sample_importance: n_coarse+n_fine must be <= 2048");
  if (n_rays == 0) return 0;
  int nf_pad = 32;
  while (nf_pad < n_fine) nf_pad <<= 1;
  const int blocks = (n_rays + kWarpsPerBlock - 1) / kWarpsPerBlock;
  int cdf_pad = 8;   // power of two >= number of cdf entries (n_coarse - 1): the branch-free search probes a padded table
  while (cdf_pad < n_coarse) cdf_pad <<= 1;         // the search covers cdf_pad - 1 entries
  const size_t smem = sizeof(float) * kWarpsPerBlock * (cdf_pad + 2 * (n_coarse - 1) + (n_coarse + 1) + (nf_pad + 1) + n_coarse + n_fine);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define NERF_LAUNCH_K2_FN(FN)                                                                                                \
  do {                                                                                                                       \
    if (smem > 48 * 1024) {                                                                                                  \
      cudaError_t e = cudaFuncSetAttribute(FN, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                      \
      NERF_CHECK_ARG(e == cudaSuccess, "sample_importance: cudaFuncSetAttribute: %s", cudaGetErrorString(e));                \
    }                                                                                                                        \
    FN<<<blocks, kWarpsPerBlock * 32, smem, st>>>(z_merged, z_fine, z_coarse, w_coarse, u, n_rays, n_coarse, n_fine);       \
  } while (0)
#define NERF_LAUNCH_K2(KK)                                                          \
  do {                                                                              \
    switch (cdf_pad) {                                                              \
      case 8: NERF_LAUNCH_K2_FN((importance_kernel_sorted<KK, 8>)); break;          \
      case 16: NERF_LAUNCH_K2_FN((importance_kernel_sorted<KK, 16>)); break;        \
      case 32: NERF_LAUNCH_K2_FN((importance_kernel_sorted<KK, 32>)); break;        \
      case 64: NERF_LAUNCH_K2_FN((importance_kernel_sorted<KK, 64>)); break;        \
      case 128: NERF_LAUNCH_K2_FN((importance_kernel_sorted<KK, 128>)); break;      \
      case 256: NERF_LAUNCH_K2_FN((importance_kernel_sorted<KK, 256>)); break;      \
      default: NERF_LAUNCH_K2_FN((importance_kernel_sorted<KK, 512>)); break;       \
    }                                                                               \
  } while (0)
  switch (nf_pad / 32) {
    case 1: NERF_LAUNCH_K2(1); break;
    case 2: NERF_LAUNCH_K2(2); break;
    case 4: NERF_LAUNCH_K2(4); break;
    case 8: NERF_LAUNCH_K2(8); break;
    case 16: NERF_LAUNCH_K2(16); break;
    default: {  // more than 512 fine samples: shared-memory network
      if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(importance_kernel_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        NERF_CHECK_ARG(e == cudaSuccess, "sample_importance: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      }
      importance_kernel_smem<<<blocks, kWarpsPerBlock * 32, smem, st>>>(z_merged, z_fine, z_coarse, w_coarse, u, n_rays, n_coarse,
                                                                        n_fine, nf_pad);
    }
  }
#undef NERF_LAUNCH_K2
#undef NERF_LAUNCH_K2_FN
  NERF_CHECK_LAUNCH("importance_kernel");
  return 0;
}
