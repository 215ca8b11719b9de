// encoding.cuh -- the frequency encoding of positions and view directions (reference utils.py:32-36), shared by the
// forward (mlp_fwd.cu), which feeds it to the first layers, and the input-gradient kernel (mlp_dinput.cu), which
// differentiates through it.  Both must see the same sin / cos values.
#pragma once

namespace nerf {

// [cos(2^k v), sin(2^k v)] for k < n_freq, as a cos block followed by a sin block.
// sin/cos of 2^k v are produced by exact sincosf at k = 0 and k = 5 plus double-angle steps
// (<= 4 doublings: error <= 16 ulp, far below the fp16 operand rounding).
__device__ __forceinline__ void encode_axis(float v, int n_freq, float* cs_out /* [2*n_freq]: cos block, sin block */) {
  float s, c;
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    if (k >= n_freq) break;
    if (k == 0 || k == 5) {
      sincosf(v * (float)(1 << k), &s, &c);
    } else {
      const float s2 = 2.f * s * c;
      const float c2 = 1.f - 2.f * s * s;
      s = s2;
      c = c2;
    }
    cs_out[k] = c;
    cs_out[n_freq + k] = s;
  }
}

// Coordinate of the sample at depth z on the ray o + d z, rounded as K3 rounds it (no fused multiply-add): the input
// gradients differentiate cos / sin of 2^9 x, so they must see the forward's x to the last bit.
__device__ __forceinline__ float ray_point(float o, float d, float z) { return __fadd_rn(o, __fmul_rn(d, z)); }

}  // namespace nerf
