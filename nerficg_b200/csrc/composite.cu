// composite.cu -- K5 / K6: alpha compositing forward and backward.
// HBM-bound per-ray transmittance scans: one warp per ray, lanes stride over the samples so
// every global access is a coalesced 128-bit (rgbsigma) or 32-bit (z, weights) vector per
// lane, the transmittance is a multiplicative warp-shuffle scan with a carry across 32-sample
// chunks, and the backward is the closed form of SURVEY.md A.9 (a reverse additive scan).
// Algorithmic bytes: forward 20 B/sample (+4 when weights are exported) + 32 B/ray;
// backward 20 B read + 16 B written per sample (second read of the ray hits L1/L2).
#include "common.cuh"
#include "../../include/nerf_b200.h"

namespace nerf {

constexpr int kRaysPerBlock = 4;  // measured: 4, 8 and 16 rays per block time the same at config E (+-2 %)
constexpr float kFinalDelta = 1.0e10f;
constexpr int kMaxChunks = 64;  // S <= 2048

struct Chunk {
  float4 cs;   // r, g, b, sigma
  float z;
  float zn;    // z of the next sample (unused for the last one)
};

__device__ __forceinline__ Chunk load_chunk(const float4* __restrict__ rs, const float* __restrict__ z, int i, int s) {
  Chunk c;
  if (i < s) {
    c.cs = __ldg(rs + i);
    c.z = __ldg(z + i);
    c.zn = (i + 1 < s) ? __ldg(z + i + 1) : 0.f;
  } else {
    c.cs = make_float4(0.f, 0.f, 0.f, 0.f);
    c.z = 0.f;
    c.zn = 0.f;
  }
  return c;
}

// alpha of sample i, and the inclusive/exclusive products of (1 - alpha) within the chunk
__device__ __forceinline__ void chunk_scan(const Chunk& c, int i, int s, float dnorm, int lane, float& alpha, float& delta,
                                           float& excl, float& chunk_prod) {
  delta = (i == s - 1) ? kFinalDelta : __fsub_rn(c.zn, c.z);
  delta = __fmul_rn(delta, dnorm);
  alpha = (i < s) ? __fsub_rn(1.f, expf(__fmul_rn(-c.cs.w, delta))) : 0.f;
  float incl = __fsub_rn(1.f, alpha);
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl *= t;
  }
  excl = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) excl = 1.f;
  chunk_prod = __shfl_sync(0xffffffffu, incl, 31);
}

__global__ void __launch_bounds__(kRaysPerBlock * 32) composite_fwd_kernel(
    float* __restrict__ rgb, float* __restrict__ depth, float* __restrict__ alpha_out, float* __restrict__ weights,
    const float* __restrict__ z, const float4* __restrict__ rgbsigma, const float* __restrict__ dirs,
    const float* __restrict__ background, int n_rays, int s) {
  const int lane = threadIdx.x & 31;
  const int ray = blockIdx.x * kRaysPerBlock + (threadIdx.x >> 5);
  if (ray >= n_rays) return;
  const float dx = __ldg(dirs + 3 * ray), dy = __ldg(dirs + 3 * ray + 1), dz = __ldg(dirs + 3 * ray + 2);
  const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
  const float4* rs = rgbsigma + (int64_t)ray * s;
  const float* zr = z + (int64_t)ray * s;
  float carry = 1.f, ar = 0.f, ag = 0.f, ab = 0.f, awz = 0.f;
  Chunk cur = load_chunk(rs, zr, lane, s);
  for (int base = 0; base < s; base += 32) {
    const int i = base + lane;
    Chunk nxt = load_chunk(rs, zr, i + 32, s);  // prefetch: keeps two chunks of loads in flight
    float a, delta, excl, prod;
    chunk_scan(cur, i, s, dnorm, lane, a, delta, excl, prod);
    const float w = a * (carry * excl);
    carry *= prod;
    ar += w * cur.cs.x;
    ag += w * cur.cs.y;
    ab += w * cur.cs.z;
    awz += w * cur.z;
    if (weights != nullptr && i < s) weights[(int64_t)ray * s + i] = w;
    cur = nxt;
  }
  ar = warp_sum(ar);
  ag = warp_sum(ag);
  ab = warp_sum(ab);
  awz = warp_sum(awz);
  if (lane == 0) {
    const float tf = carry, al = 1.f - tf;
    float br = 0.f, bgc = 0.f, bb = 0.f;
    if (background != nullptr) {
      br = __ldg(background);
      bgc = __ldg(background + 1);
      bb = __ldg(background + 2);
    }
    rgb[3 * ray] = ar + tf * br;
    rgb[3 * ray + 1] = ag + tf * bgc;
    rgb[3 * ray + 2] = ab + tf * bb;
    depth[ray] = (tf < 1.f) ? awz / al : 0.f;
    alpha_out[ray] = al;
  }
}

__global__ void __launch_bounds__(kRaysPerBlock * 32) composite_bwd_kernel(
    float4* __restrict__ d_rgbsigma, const float* __restrict__ z, const float4* __restrict__ rgbsigma,
    const float* __restrict__ dirs, const float* __restrict__ background, const float* __restrict__ g_rgb,
    const float* __restrict__ g_depth, const float* __restrict__ g_alpha, int n_rays, int s, int relu_mask,
    float grad_scale) {
  __shared__ float carry_in[kRaysPerBlock][kMaxChunks];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int ray = blockIdx.x * kRaysPerBlock + wid;
  if (ray >= n_rays) return;
  const float dx = __ldg(dirs + 3 * ray), dy = __ldg(dirs + 3 * ray + 1), dz = __ldg(dirs + 3 * ray + 2);
  const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
  const float4* rs = rgbsigma + (int64_t)ray * s;
  const float* zr = z + (int64_t)ray * s;
  const float gr = __ldg(g_rgb + 3 * ray), gg = __ldg(g_rgb + 3 * ray + 1), gb = __ldg(g_rgb + 3 * ray + 2);
  const float gd = g_depth ? __ldg(g_depth + ray) : 0.f;
  const float ga = g_alpha ? __ldg(g_alpha + ray) : 0.f;

  // pass 1: transmittance entering every chunk, final transmittance, sum of w*z
  float carry = 1.f, awz = 0.f;
  const int n_chunks = (s + 31) / 32;
  {
    Chunk cur = load_chunk(rs, zr, lane, s);
    for (int c = 0; c < n_chunks; ++c) {
      const int i = c * 32 + lane;
      Chunk nxt = load_chunk(rs, zr, i + 32, s);
      float a, delta, excl, prod;
      chunk_scan(cur, i, s, dnorm, lane, a, delta, excl, prod);
      if (lane == 0) carry_in[wid][c] = carry;
      awz += a * (carry * excl) * cur.z;
      carry *= prod;
      cur = nxt;
    }
  }
  awz = warp_sum(awz);
  __syncwarp();
  const float tf = carry, al = 1.f - tf;
  const bool has_depth = tf < 1.f;
  const float gd_over_a = has_depth ? gd / al : 0.f;
  float g_t = -ga + (has_depth ? gd * awz / (al * al) : 0.f);  // dL/dT_f (direct)
  if (background != nullptr) g_t += gr * __ldg(background) + gg * __ldg(background + 1) + gb * __ldg(background + 2);
  const float tf_gt = tf * g_t;

  // pass 2: reverse walk with the suffix sum of g_j w_j (re-reads hit L1/L2)
  float suffix = 0.f;
  for (int c = n_chunks - 1; c >= 0; --c) {
    const int i = c * 32 + lane;
    const Chunk cur = load_chunk(rs, zr, i, s);
    float a, delta, excl, prod;
    chunk_scan(cur, i, s, dnorm, lane, a, delta, excl, prod);
    const float t_i = carry_in[wid][c] * excl;
    const float w = a * t_i;
    const float t_next = t_i * (1.f - a);
    const float g = gr * cur.cs.x + gg * cur.cs.y + gb * cur.cs.z + gd_over_a * cur.z;
    const float gw = (i < s) ? g * w : 0.f;
    float incl = gw;  // inclusive suffix within the chunk
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float t = __shfl_down_sync(0xffffffffu, incl, o);
      if (lane + o < 32) incl += t;
    }
    const float after = suffix + (incl - gw);  // sum over j > i
    suffix += __shfl_sync(0xffffffffu, incl, 0);
    if (i < s) {
      float ds = delta * (g * t_next - after - tf_gt);
      if (relu_mask && !(cur.cs.w > 0.f)) ds = 0.f;
      d_rgbsigma[(int64_t)ray * s + i] =
          make_float4(grad_scale * w * gr, grad_scale * w * gg, grad_scale * w * gb, grad_scale * ds);
    }
  }
}

}  // namespace nerf

extern "C" int nerf_composite_forward(float* rgb, float* depth, float* alpha, float* weights, const float* z,
                                      const float* rgbsigma, const float* dirs, const float* background, int n_rays,
                                      int n_samples, void* stream) {
  using namespace nerf;
  if (n_rays <= 0) return 0;
  NERF_CHECK_ARG(rgb && depth && alpha && z && rgbsigma && dirs, "composite_forward: null pointer");
  NERF_CHECK_ARG(n_samples >= 1 && n_samples <= 32 * kMaxChunks, "composite_forward: n_samples must be in [1,%d]", 32 * kMaxChunks);
  NERF_CHECK_ARG((reinterpret_cast<uintptr_t>(rgbsigma) & 15) == 0, "composite_forward: rgbsigma must be 16-byte aligned");
  if (n_rays <= 0) return 0;
  const int blocks = (n_rays + kRaysPerBlock - 1) / kRaysPerBlock;
  composite_fwd_kernel<<<blocks, kRaysPerBlock * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      rgb, depth, alpha, weights, z, reinterpret_cast<const float4*>(rgbsigma), dirs, background, n_rays, n_samples);
  NERF_CHECK_LAUNCH("composite_fwd_kernel");
  return 0;
}

extern "C" int nerf_composite_backward(float* d_rgbsigma, const float* z, const float* rgbsigma, const float* dirs,
                                       const float* background, const float* g_rgb, const float* g_depth,
                                       const float* g_alpha, int n_rays, int n_samples, int relu_mask, float grad_scale,
                                       void* stream) {
  using namespace nerf;
  if (n_rays <= 0) return 0;
  NERF_CHECK_ARG(d_rgbsigma && z && rgbsigma && dirs && g_rgb, "composite_backward: null pointer");
  NERF_CHECK_ARG(n_samples >= 1 && n_samples <= 32 * kMaxChunks, "composite_backward: n_samples must be in [1,%d]", 32 * kMaxChunks);
  NERF_CHECK_ARG(((reinterpret_cast<uintptr_t>(rgbsigma) | reinterpret_cast<uintptr_t>(d_rgbsigma)) & 15) == 0,
                 "composite_backward: rgbsigma buffers must be 16-byte aligned");
  if (n_rays <= 0) return 0;
  const int blocks = (n_rays + kRaysPerBlock - 1) / kRaysPerBlock;
  composite_bwd_kernel<<<blocks, kRaysPerBlock * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<float4*>(d_rgbsigma), z, reinterpret_cast<const float4*>(rgbsigma), dirs, background, g_rgb, g_depth,
      g_alpha, n_rays, n_samples, relu_mask, grad_scale);
  NERF_CHECK_LAUNCH("composite_bwd_kernel");
  return 0;
}
