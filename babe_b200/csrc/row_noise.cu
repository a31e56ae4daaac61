// k_row_noise: counter-based Gaussian noise keyed by one seed per row, optionally fused into the state update
//   out[b, n] = a[b, n] + eps[b, n] * (mult * scale * row_scale[b])
// (DESIGN.md 4.8).  eps[b, n] is a function of (seeds[b], *draw + slot, n) only (csrc/philox.cuh): not of B, of
// the row's position, of T, of the alignment of the row or of the launch configuration.
#include "common.cuh"
#include "philox.cuh"

namespace babe {

// One thread = one Philox call = the four samples 4j .. 4j+3 of one row.  blockIdx.y strides over the rows,
// blockIdx.x * blockDim.x + threadIdx.x over the groups of four of a row.  Rows whose base addresses are 16-byte
// aligned move full groups with one float4 load / store; the other rows and the tail group go sample by sample
// through the same arithmetic.
__global__ void __launch_bounds__(256) k_row_noise(float* out, const float* a,
                                                   const long long* __restrict__ seeds, int B, int T,
                                                   const int* __restrict__ draw, int slot,
                                                   const float* __restrict__ scale,
                                                   const float* __restrict__ row_scale, float mult) {
  const uint32_t d = (uint32_t)(__ldg(draw) + slot);
  const int groups = (T + 3) >> 2;
  float m0 = mult;
  if (scale != nullptr) m0 = __fmul_rn(m0, __ldg(scale));
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const uint64_t s = (uint64_t)__ldg(seeds + b);
    const float m = row_scale != nullptr ? __fmul_rn(m0, __ldg(row_scale + b)) : m0;
    float* orow = out + (size_t)b * T;
    const float* arow = a != nullptr ? a + (size_t)b * T : nullptr;
    const bool vec = ((reinterpret_cast<uintptr_t>(orow) | reinterpret_cast<uintptr_t>(arow)) & 15) == 0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < groups; j += gridDim.x * blockDim.x) {
      float e[4];
      row_noise4(s, d, (uint32_t)j, e);
      const int n0 = j << 2;
      if (vec && n0 + 4 <= T) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (arow != nullptr) v = *reinterpret_cast<const float4*>(arow + n0);   // may alias out: read first
        v.x = __fadd_rn(v.x, __fmul_rn(e[0], m));
        v.y = __fadd_rn(v.y, __fmul_rn(e[1], m));
        v.z = __fadd_rn(v.z, __fmul_rn(e[2], m));
        v.w = __fadd_rn(v.w, __fmul_rn(e[3], m));
        *reinterpret_cast<float4*>(orow + n0) = v;
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (n0 + q < T) {
            const float base = arow != nullptr ? arow[n0 + q] : 0.f;
            orow[n0 + q] = __fadd_rn(base, __fmul_rn(e[q], m));
          }
        }
      }
    }
  }
}

}  // namespace babe

extern "C" int babe_row_noise(float* out, const float* a, const long long* seeds, int B, int T, const int* draw,
                              int slot, const float* scale, const float* row_scale, float mult, void* stream) {
  BABE_REQUIRE(out != nullptr && seeds != nullptr && draw != nullptr, BABE_EBADARG,
               "babe_row_noise: out, seeds and draw are required");
  BABE_REQUIRE(B >= 0 && T >= 0 && slot >= 0, BABE_EBADARG, "babe_row_noise: B = %d, T = %d, slot = %d", B, T,
               slot);
  if (B == 0 || T == 0) return BABE_OK;
  const int threads = 256;
  const int groups = (T + 3) / 4;
  const int gx = (groups + threads - 1) / threads;
  const int gy = B < 65535 ? B : 65535;
  babe::k_row_noise<<<dim3(gx, gy), threads, 0, (cudaStream_t)stream>>>(out, a, seeds, B, T, draw, slot, scale,
                                                                         row_scale, mult);
  return babe::check_launch("k_row_noise");
}
