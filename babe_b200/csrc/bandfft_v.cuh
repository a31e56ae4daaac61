// Power-of-two FFTs of the constant-Q bands on PACKED complex values (float2 in a 64-bit register pair, Blackwell's
// two-wide FADD2 / FFMA2 / FMUL2: one issue slot per complex add), forward or inverse selected at compile time (no
// conjugation passes), with the window / dual-window multiply folded into the first butterflies.
//
// BandCoreV<R3, INV>: M = 256 R3 points (R3 = 1..16) by TPB = 16 R3 threads, 16 points per thread, three passes
// 16 x 16 x R3 with two exchanges (rows of TPB + 1 float2: conflict-free) -- coalesced on both sides without staging:
//   n = 16 R3 n1 + R3 n2 + n3,   k = k1 + 16 k2 + 256 k3,   t = R3 n2 + n3
//   P1  thread t: FFT16 n1 -> k1, * W_M^{-+ t k1} -> ex[k1][t]            (input slot of register n1: TPB n1 + t)
//   P2  thread (k1 = t & 15, n3 = t >> 4): FFT16 n2 -> k2, in place
//   P3  thread t, pairs (k1 = t & 15, k2 = (t >> 4) + R3 j): * W_{16 R3}^{-+ n3 k2}, FFT_R3 n3 -> k3
//                                                                         (output slot: t + TPB j + 256 k3)
// BandCoreS<R2, INV>: M = 16 R2 points (R2 = 2, 4, 8: the low octaves) by R2 threads:
//   n = R2 n1 + t,  k = k1 + 16 k2;  P1 as above -> ex[k1][t];  P2 thread u: k1 = u + R2 j, FFT_R2 t -> k2
//
// The exchanges are synchronised per BAND (named barrier of TPB threads, __syncwarp for TPB <= 32), never per CTA:
// the bands of a CTA run independently.  Every thread of a band group must call fwd().
// __host__ __device__ passes: tests/host/bandfft_v_host_check.cu.
#pragma once
#include "common.cuh"
#include "fft16v.cuh"

namespace babe {

template <int R, bool INV> BABE_HD void small_fft_v(float2 (&a)[R]) {
  if constexpr (R == 2) { const float2 t = c_sub(a[0], a[1]); a[0] = c_add(a[0], a[1]); a[1] = t; }
  else if constexpr (R == 4) fft4v<INV>(a[0], a[1], a[2], a[3]);
  else if constexpr (R == 8) fft8v<INV, false>(a);
  else if constexpr (R == 16) fft16v<INV>(a);
}

template <int NT> __device__ __forceinline__ void band_sync(int bar_id) {
#ifdef __CUDA_ARCH__
  if (NT <= 32) __syncwarp();
  else asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(NT) : "memory");
#endif
}

template <int R3, bool INV>
struct BandCoreV {
  static constexpr int M = 256 * R3, TPB = 16 * R3, ROW = TPB + 1, EX = 16 * ROW, NP = 16 / R3, NTW = TPB;
  static constexpr int EXP = EX;                                // per-band stride of the exchange buffers
  struct Regs { float2 w[16]; };                                // W_M^{t k1} (forward roots; conjugated on use)
  BABE_HD static void init_regs(Regs& r, const float2* roots_m, int t) {
#pragma unroll
    for (int k1 = 0; k1 < 16; ++k1) r.w[k1] = roots_m[t * k1];
  }
  BABE_HD static float2 twiddle(const float2* roots_m, int i) { return roots_m[16 * i]; }   // W_{16 R3}^i, i < NTW
  BABE_HD static int in_slot(int n1, int t) { return TPB * n1 + t; }
  BABE_HD static int out_slot(int r, int t) { return t + TPB * (r / R3) + 256 * (r % R3); }

  template <bool SCALED>
  BABE_HD static void pass1(float2 (&z)[16], const float (&s)[16], float2* ex, const Regs& rg, int t) {
    fft16v_impl<INV, SCALED>(z, s);
    ex[t] = z[0];
#pragma unroll
    for (int k1 = 1; k1 < 16; ++k1) ex[k1 * ROW + t] = c_tw<INV>(z[k1], rg.w[k1]);
  }
  BABE_HD static void pass2(float2 (&z)[16], float2* ex, int t) {
    float2* col = ex + (t & 15) * ROW + (t >> 4);
#pragma unroll
    for (int n2 = 0; n2 < 16; ++n2) z[n2] = col[R3 * n2];
    fft16v<INV>(z);
    if constexpr (R3 > 1) {
#pragma unroll
      for (int k2 = 0; k2 < 16; ++k2) col[R3 * k2] = z[k2];
    }
  }
  BABE_HD static void pass3(float2 (&z)[16], const float2* ex, const float2* tw, int t) {
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const int k2 = (t >> 4) + R3 * j;
      const float2* row = ex + (t & 15) * ROW + R3 * k2;
      float2 a[R3];
      a[0] = row[0];
#pragma unroll
      for (int n3 = 1; n3 < R3; ++n3) a[n3] = c_tw<INV>(row[n3], tw[n3 * k2]);
      small_fft_v<R3, INV>(a);
#pragma unroll
      for (int k3 = 0; k3 < R3; ++k3) z[j * R3 + k3] = a[k3];
    }
  }
  // z[n1] = input slot TPB n1 + t (times s[n1] if SCALED) -> z[r] = output slot out_slot(r, t)
  // `after_sync` runs right behind the first band-wide synchronisation: every thread of the band has consumed its
  // staged inputs by then (the caller re-arms the staging copy for the next row there)
  template <bool SCALED, class F>
  __device__ static __forceinline__ void fwd(float2 (&z)[16], const float (&s)[16], float2* ex, const float2* tw,
                                             const Regs& rg, int t, int bar_id, F&& after_sync) {
    pass1<SCALED>(z, s, ex, rg, t);
    band_sync<TPB>(bar_id);
    after_sync();
    pass2(z, ex, t);
    if constexpr (R3 > 1) {
      band_sync<TPB>(bar_id);
      pass3(z, ex, tw, t);
    }
  }
};

template <int R2, bool INV>
struct BandCoreS {
  static constexpr int M = 16 * R2, TPB = R2, ROW = R2 + 1, EX = 16 * ROW, NP = 16 / R2, NTW = 1;
  static constexpr int EXP = EX + R2;      // stride = R2 (mod 16 float2): the 16 / R2 bands of a half-warp tile the banks
  struct Regs { float2 w[16]; };
  BABE_HD static void init_regs(Regs& r, const float2* roots_m, int t) {
#pragma unroll
    for (int k1 = 0; k1 < 16; ++k1) r.w[k1] = roots_m[t * k1];
  }
  BABE_HD static float2 twiddle(const float2* roots_m, int i) { return roots_m[0]; }
  BABE_HD static int in_slot(int n1, int t) { return R2 * n1 + t; }
  BABE_HD static int out_slot(int r, int t) { return t + R2 * (r / R2) + 16 * (r % R2); }   // k1 = t + R2 j, k2 = r % R2

  template <bool SCALED>
  BABE_HD static void pass1(float2 (&z)[16], const float (&s)[16], float2* ex, const Regs& rg, int t) {
    fft16v_impl<INV, SCALED>(z, s);
    ex[t] = z[0];
#pragma unroll
    for (int k1 = 1; k1 < 16; ++k1) ex[k1 * ROW + t] = c_tw<INV>(z[k1], rg.w[k1]);
  }
  BABE_HD static void pass2(float2 (&z)[16], const float2* ex, int t) {
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const float2* row = ex + (t + R2 * j) * ROW;
      float2 a[R2];
#pragma unroll
      for (int n2 = 0; n2 < R2; ++n2) a[n2] = row[n2];
      small_fft_v<R2, INV>(a);
#pragma unroll
      for (int k2 = 0; k2 < R2; ++k2) z[j * R2 + k2] = a[k2];
    }
  }
  template <bool SCALED, class F>
  __device__ static __forceinline__ void fwd(float2 (&z)[16], const float (&s)[16], float2* ex, const float2* tw,
                                             const Regs& rg, int t, int bar_id, F&& after_sync) {
    pass1<SCALED>(z, s, ex, rg, t);
    band_sync<TPB>(bar_id);
    after_sync();
    pass2(z, ex, t);
  }
};

}  // namespace babe
