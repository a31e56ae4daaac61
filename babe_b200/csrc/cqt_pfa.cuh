// Third-generation length-Ls transform of the CQT: a PRIME-FACTOR (Good-Thomas) FFT in two passes.
//
// Ls = 184184 = 2 * (4 * 7 * 11) * (13 * 23): all factors of Nc = Ls / 2 are pairwise coprime, so the complex FFT of
// Nc points is a five-dimensional DFT with NO twiddle factors between any two stages (for 132300 = 2 * 2 * 27 * 25 * 49
// and 485100 the prime powers 9, 25, 27, 49 are single digits, transformed by the same mirrored-input odd DFT):
//
//     n = sum_i n_i * (Nc / R_i)  (mod Nc)      input index  (Ruritanian map; n_i = ((n mod R_i) * inv_i) mod R_i)
//     k = k_i  (mod R_i)                        output index (Chinese remainder map)
//     W_Nc^{n k} = prod_i W_{R_i}^{n_i k_i}
//
// Pass 1 transforms the digits of N1 = RA*RB*RC for a tile of S consecutive residues r = n mod N2 (the elements
// n = r + N2 j of S neighbouring residues are S consecutive complex samples: 128-byte runs), pass 2 the digits of
// N2 = RD*RE*RF for the S rows of S/2 residue pairs (k1, N1 - k1) of k mod N1 -- both members of every bin pair
// (k, Nc - k) of the real-FFT post-processing sit in the same tile, and the bins k = k1 + N1 j of consecutive k1 are
// consecutive in the natural-order half spectrum (64-byte runs).  A tile lives in shared memory as [digit index][S]
// float2 and every stage works IN PLACE with compile-time strides (one buffer, no twiddle tables, no Stockham index
// arithmetic); the input / output permutations are two small tables built by every CTA.  The odd-prime DFTs keep the
// (R-1)/2 sums and differences of the mirrored inputs in registers and store every output pair as soon as it is
// complete, which fits the radix-23 butterfly into 64 registers (keeping all R outputs takes 128).
//
// apply_hpf_DC needs 3 launches instead of 5 (pass 2 runs forward, multiplies by H in the r2c / c2r pair processing
// and runs backward without leaving shared memory), analysis 2 + 1, synthesis 1 + 2 (the overlap-add of the band
// spectra is a table-driven gather in the prologue of the inverse pass 2).
//
// All per-thread phases are __host__ __device__: tests/host/pfa_host_check.cu emulates the kernels thread by thread
// against numpy.  Lengths whose factorisation is not instantiated keep the generic passes of cqt_ops.cu.
#pragma once
#include "rfft_pairs.cuh"
#include "fft16v.cuh"

namespace babe {
namespace pfa {

constexpr int THREADS = 256;
constexpr int TW_LO_ = 1024;

BABE_HD constexpr int modinv(int a, int m) {
  a %= m;
  for (int x = 1; x < m; ++x)
    if ((a * x) % m == 1) return x;
  return 0;
}

template <int RA_, int RB_, int RC_, int RD_, int RE_, int RF_>
struct Plan {
  static constexpr int RA = RA_, RB = RB_, RC = RC_, RD = RD_, RE = RE_, RF = RF_;
  static constexpr int N1 = RA * RB * RC, N2 = RD * RE * RF, NC = N1 * N2;
  static constexpr int P2 = (N2 + 1) & ~1;          // row pitch of the intermediate in float2 (even: 16-byte rows)
  // resident CTAs per SM the register budget is sized for: the odd DFTs keep R - 1 float2 in registers
  static constexpr int minb(int a, int b, int c) {
    const int m = a > b ? (a > c ? a : c) : (b > c ? b : c);
    return m <= 23 ? 4 : (m <= 27 ? 3 : 2);
  }
  static constexpr int MINB1 = minb(RA, RB, RC), MINB2 = minb(RD, RE, RF);
  static constexpr int IA = modinv((NC / RA) % RA, RA), IB = modinv((NC / RB) % RB, RB), IC = modinv((NC / RC) % RC, RC);
  static constexpr int ID = modinv((NC / RD) % RD, RD), IE = modinv((NC / RE) % RE, RE), IF_ = modinv((NC / RF) % RF, RF);
  // input side: digit index of residue m = n mod N1 (pass 1) / r = n mod N2 (pass 2)
  BABE_HD static int t1(int m) { return (((m % RA) * IA % RA) * RB + ((m % RB) * IB % RB)) * RC + ((m % RC) * IC % RC); }
  BABE_HD static int t2(int r) { return (((r % RD) * ID % RD) * RE + ((r % RE) * IE % RE)) * RF + ((r % RF) * IF_ % RF); }
  // output side: digit index of k1 = k mod N1 / r2 = k mod N2
  BABE_HD static int q1(int k1) { return ((k1 % RA) * RB + k1 % RB) * RC + k1 % RC; }
  BABE_HD static int d2(int r2) { return ((r2 % RD) * RE + r2 % RE) * RF + r2 % RF; }
};

// exp(-2 pi i m / Ls) from the plan's two-level table
BABE_HD float2 tw_ls(const float2* tab, int m) { return cmul(tab[m & (TW_LO_ - 1)], tab[TW_LO_ + (m >> 10)]); }

// In-place DFT of the R points p[0], p[st], ..., p[(R-1) st]; INV: conjugated roots (no scaling).  All arithmetic on
// float2 register pairs with the two-wide instructions (fft16v.cuh): the odd-prime DFTs are FFMA2 with the root as a
// 32-bit immediate broadcast to both halves -- half the issue slots of the scalar form, no constant registers.
template <int R, bool INV> BABE_HD void dft_io(const float2* q, const int sq, float2* p, const int st);
// Inputs q[0], q[sq], ... and outputs p[0], p[st], ... may be the same array (all inputs are read before the first store)
// or different ones (a stage that reads or writes the global intermediate directly).
template <int R, bool INV>
BABE_HD void dft_inplace(float2* p, const int st) { dft_io<R, INV>(p, st, p, st); }

template <int R, bool INV>
BABE_HD void dft_io(const float2* q, const int sq, float2* p, const int st) {
  if constexpr (R == 1) {
    return;
  } else if constexpr (R == 2) {
    const float2 u = q[0], v = q[sq];
    p[0] = c_add(u, v); p[st] = c_sub(u, v);
  } else if constexpr (R == 4) {
    float2 v0 = q[0], v1 = q[sq], v2 = q[2 * sq], v3 = q[3 * sq];
    fft4v<INV>(v0, v1, v2, v3);
    p[0] = v0; p[st] = v1; p[2 * st] = v2; p[3 * st] = v3;
  } else if constexpr (R == 8 || R == 16) {
    float2 v[R];
#pragma unroll
    for (int t = 0; t < R; ++t) v[t] = q[t * sq];
    if constexpr (R == 8) fft8v<INV, false>(v); else fft16v<INV>(v);
#pragma unroll
    for (int t = 0; t < R; ++t) p[t * st] = v[t];
  } else {
    // odd prime: a_t = v_t + v_{R-t}, b_t = v_t - v_{R-t};  X_u = v_0 + sum a_t cos - i sum b_t sin, X_{R-u} with + i
    constexpr int H = (R - 1) / 2;
    const float2 x0 = q[0];
    float2 a[H], b[H];
    float2 s0 = x0;
#pragma unroll
    for (int t = 1; t <= H; ++t) {
      const float2 u = q[t * sq], v = q[(R - t) * sq];
      a[t - 1] = c_add(u, v);
      b[t - 1] = c_sub(u, v);
      s0 = c_add(s0, a[t - 1]);
    }
    p[0] = s0;
#pragma unroll
    for (int u = 1; u <= H; ++u) {
      float2 A = c_fma(a[0], odd_cos<R>(u % R), x0);
      float2 B = c_scale(b[0], odd_sin<R>(u % R));
#pragma unroll
      for (int t = 2; t <= H; ++t) {
        const int m = (t * u) % R;
        A = c_fma(a[t - 1], odd_cos<R>(m), A);
        B = c_fma(b[t - 1], odd_sin<R>(m), B);
      }
      const float2 lo = c_add_mi(A, B), hi = c_sub_mi(A, B);      // A - iB, A + iB
      p[u * st] = INV ? hi : lo;
      p[(R - u) * st] = INV ? lo : hi;
    }
  }
}

// One stage: digit of radix R with CO digit combinations above it and CI below; element (o, d, i) at ((o R + d) CI + i) S.
template <int R, int CO, int CI, int S, bool INV>
BABE_HD void stage(float2* A, int slot, int col, int nslots) {
  if constexpr (R > 1) {
    constexpr int NB = CO * CI;
    // small butterflies are mostly shared-memory latency: several of them in flight per thread
    constexpr int UNROLL = R <= 4 ? 5 : (R <= 8 ? 2 : 1);
#pragma unroll UNROLL
    for (int idx = slot; idx < NB; idx += nslots) {
      const int o = idx / CI, in = idx - o * CI;
      dft_inplace<R, INV>(A + ((o * R) * CI + in) * S + col, CI * S);
    }
  }
}

#ifdef __CUDA_ARCH__
#define PFA_SYNC() __syncthreads()
#else
#define PFA_SYNC() ((void)0)
#endif

// global -> shared copies that need no registers and no waiting until the tile is complete (LDGSTS); plain copies on the
// host.  All loads of a tile are in flight at once: the load phase of a CTA costs one memory latency.
BABE_HD void copy8_async(float2* dst, const float2* src) {
#ifdef __CUDA_ARCH__
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(src) : "memory");
#else
  *dst = *src;
#endif
}
BABE_HD void copy16_async(float2* dst, const float2* src) {
#ifdef __CUDA_ARCH__
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
#else
  dst[0] = src[0]; dst[1] = src[1];
#endif
}
BABE_HD void copies_wait() {
#ifdef __CUDA_ARCH__
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
#endif
}

// ---------------------------------------------------------------------------------------------------------------------
// pass 1: digits of N1 for a tile of S residues r = n mod N2
// ---------------------------------------------------------------------------------------------------------------------
template <class PL, int S>
struct Pass1 {
  static constexpr int SLOTS = THREADS / S, TILES = (PL::N2 + S - 1) / S;
  static constexpr size_t SMEM = sizeof(float2) * PL::N1 * S + sizeof(unsigned short) * ((PL::N1 + 7) & ~7);
  BABE_HD static unsigned short* table(float2* A) { return reinterpret_cast<unsigned short*>(A + PL::N1 * S); }
  BABE_HD static void tables(unsigned short* T1, int tid) {
    for (int m = tid; m < PL::N1; m += THREADS) T1[m] = (unsigned short)PL::t1(m);
  }
  // z[Nc] (natural order) -> tile, element n = r + N2 j at digit index T1[n mod N1]
  BABE_HD static void load_natural(const float2* z, float2* A, const unsigned short* T1, int tile, int tid) {
    const int col = tid % S, slot = tid / S, r = tile * S + col;
    const bool live = r < PL::N2;
    constexpr int STEP = (PL::N2 * SLOTS) % PL::N1;
    int m = (r + PL::N2 * slot) % PL::N1;
    constexpr int IT = (PL::N1 + SLOTS - 1) / SLOTS, BATCH = 10;
#pragma unroll
    for (int b0 = 0; b0 < IT; b0 += BATCH) {
      float2 v[BATCH];
#pragma unroll
      for (int b = 0; b < BATCH; ++b) {
        const int j = slot + (b0 + b) * SLOTS;
        v[b] = (live && b0 + b < IT && j < PL::N1) ? z[r + PL::N2 * j] : make_float2(0.f, 0.f);
      }
#pragma unroll
      for (int b = 0; b < BATCH; ++b) {
        const int j = slot + (b0 + b) * SLOTS;
        if (b0 + b < IT && j < PL::N1) A[T1[m] * S + col] = v[b];
        m += STEP;
        if (m >= PL::N1) m -= PL::N1;
      }
    }
  }
  BABE_HD static void store_natural(const float2* A, float2* z, const unsigned short* T1, int tile, int tid) {
    const int col = tid % S, slot = tid / S, r = tile * S + col;
    if (r >= PL::N2) return;
    constexpr int STEP = (PL::N2 * SLOTS) % PL::N1;
    int m = (r + PL::N2 * slot) % PL::N1;
#pragma unroll 5
    for (int j = slot; j < PL::N1; j += SLOTS) {
      z[r + PL::N2 * j] = A[T1[m] * S + col];
      m += STEP;
      if (m >= PL::N1) m -= PL::N1;
    }
  }
  // intermediate Y[q][r] (row pitch P2) <-> tile, digit index q in place
  BABE_HD static void store_rows(const float2* A, float2* Y, int tile, int tid) {
    constexpr int HS = S / 2, SL2 = THREADS / HS;
    const int c2 = 2 * (tid % HS), slot = tid / HS, r = tile * S + c2;
    if (r >= PL::N2) return;          // r + 1 == N2 writes the pad element of the row (never read as data)
#pragma unroll 5
    for (int q = slot; q < PL::N1; q += SL2)
      *reinterpret_cast<float4*>(Y + (size_t)q * PL::P2 + r) = *reinterpret_cast<const float4*>(A + q * S + c2);
  }
  // 16 bytes (two residues) per copy: rows of the intermediate and of the tile are 16-byte aligned
  BABE_HD static void load_rows(const float2* Y, float2* A, int tile, int tid) {
    constexpr int HS = S / 2, SL2 = THREADS / HS;
    const int c2 = 2 * (tid % HS), slot = tid / HS, r = tile * S + c2;
    const bool live = r < PL::N2;     // r + 1 == N2: the pad element of the row lands in a dead column
#pragma unroll 4
    for (int q = slot; q < PL::N1; q += SL2) {
      float2* dst = A + q * S + c2;
      if (live) copy16_async(dst, Y + (size_t)q * PL::P2 + r);
      else { dst[0] = make_float2(0.f, 0.f); dst[1] = make_float2(0.f, 0.f); }
    }
    copies_wait();
  }
  // The stages in order (digits A, B, C; radix-1 digits skipped).  MODE 0: in place; MODE 1: inputs straight from the
  // rows of the global intermediate (first stage of the inverse: no separate load pass); MODE 2: outputs straight to
  // the rows of the global intermediate (last stage of the forward: no separate store pass).  Saves two of the eight
  // shared-memory accesses per element and one barrier per tile.
  static constexpr int NST = 1 + (PL::RB > 1) + (PL::RC > 1);
  template <bool INV, int WHICH, int MODE>
  BABE_HD static void run_stage(float2* A, const float2* Yin, float2* Yout, int tile, int tid) {
    constexpr int R = WHICH == 0 ? PL::RA : (WHICH == 1 ? PL::RB : PL::RC);
    constexpr int CO = WHICH == 0 ? 1 : (WHICH == 1 ? PL::RA : PL::RA * PL::RB);
    constexpr int CI = WHICH == 0 ? PL::RB * PL::RC : (WHICH == 1 ? PL::RC : 1);
    constexpr int NB = CO * CI, UNROLL = R <= 4 ? 5 : (R <= 8 ? 2 : 1);
    const int col = tid % S, slot = tid / S, r = tile * S + col;
    const bool live = r < PL::N2;
#pragma unroll UNROLL
    for (int idx = slot; idx < NB; idx += SLOTS) {
      const int o = idx / CI, in = idx - o * CI, e0 = (o * R) * CI + in;
      float2* a = A + e0 * S + col;
      if (MODE == 0) {
        dft_io<R, INV>(a, CI * S, a, CI * S);
      } else if (MODE == 1) {
        if (live) dft_io<R, INV>(Yin + (size_t)e0 * PL::P2 + r, CI * PL::P2, a, CI * S);
        else {
#pragma unroll
          for (int d = 0; d < R; ++d) a[d * CI * S] = make_float2(0.f, 0.f);
        }
      } else {
        if (live) dft_io<R, INV>(a, CI * S, Yout + (size_t)e0 * PL::P2 + r, CI * PL::P2);
        if (PL::P2 > PL::N2 && r == PL::N2 - 1) {     // the pad element of the rows: read (and ignored) as half of a 16-byte load
#pragma unroll
          for (int d = 0; d < R; ++d) Yout[(size_t)(e0 + d * CI) * PL::P2 + PL::N2] = make_float2(0.f, 0.f);
        }
      }
    }
  }
  // n-th executed stage (0 .. NST - 1) -> digit
  static constexpr int which(int n) { return n == 0 ? 0 : (n == 1 ? (PL::RB > 1 ? 1 : 2) : 2); }
  template <bool INV, int N, int MODE>
  BABE_HD static void stage_n(float2* A, const float2* Yin, float2* Yout, int tile, int tid) {
    if constexpr (N < NST) run_stage<INV, which(N), MODE>(A, Yin, Yout, tile, tid);
  }
  // forward: tile (filled by load_natural) -> rows of Y;  device: every thread of the CTA
  BABE_HD static void forward_to_rows(float2* A, float2* Y, int tile, int tid) {
    stage_n<false, 0, NST == 1 ? 2 : 0>(A, nullptr, Y, tile, tid);
    if (NST > 1) { PFA_SYNC(); stage_n<false, 1, NST == 2 ? 2 : 0>(A, nullptr, Y, tile, tid); }
    if (NST > 2) { PFA_SYNC(); stage_n<false, 2, 2>(A, nullptr, Y, tile, tid); }
  }
  // inverse: rows of Y -> tile (then store_natural); ends with a barrier.  The rows are staged by 16-byte cp.async
  // (load_rows): reading them inside the first stage (MODE 1, synchronous 8-byte loads per butterfly) was measured
  // SLOWER (irfft 0.0704 -> 0.0746 ms at B = 64) although it saves a pass over shared memory.
  BABE_HD static void inverse_from_rows(const float2* Y, float2* A, int tile, int tid) {
    load_rows(Y, A, tile, tid); PFA_SYNC();
    stage_n<true, 0, 0>(A, nullptr, nullptr, tile, tid); PFA_SYNC();
    if (NST > 1) { stage_n<true, 1, 0>(A, nullptr, nullptr, tile, tid); PFA_SYNC(); }
    if (NST > 2) { stage_n<true, 2, 0>(A, nullptr, nullptr, tile, tid); PFA_SYNC(); }
  }
};

// ---------------------------------------------------------------------------------------------------------------------
// pass 2: digits of N2 for the rows of S/2 residue pairs (k1, N1 - k1); last tile: the self-mirrored k1 = 0, N1 / 2
// ---------------------------------------------------------------------------------------------------------------------
struct GatherTab {                 // synthesis: overlap-add of the band spectra, <= 3 bands per bin
  const float2* BS;                // this row's band spectra [sum_lg]
  const int4* src;                 // [Nc + 1] offsets into BS (x, y, z); no band: the offset of a zero element
};

template <class PL, int S>
struct Pass2 {
  static constexpr int H = S / 2, SLOTS = THREADS / S, NP = (PL::N1 - 1) / 2, NTP = (NP + H - 1) / H, TILES = NTP + 1;
  static constexpr int NT = (PL::N2 + 7) & ~7;
  static constexpr size_t SMEM = sizeof(float2) * (PL::N2 * S + NT) + 2 * sizeof(unsigned short) * NT;
  // shared memory: tile A [N2][S], TJ[j] = W_Ls^{N1 j} (the bin twiddles of a column are W_Ls^{k1} TJ[j]), T2, D2
  BABE_HD static float2* tab_tj(float2* A) { return A + PL::N2 * S; }
  BABE_HD static unsigned short* tab_t2(float2* A) { return reinterpret_cast<unsigned short*>(A + PL::N2 * S + NT); }
  BABE_HD static unsigned short* tab_d2(float2* A) { return tab_t2(A) + NT; }
  BABE_HD static void tables(float2* A, const float2* twls, int tid) {
    float2* TJ = tab_tj(A);
    unsigned short *T2 = tab_t2(A), *D2 = tab_d2(A);
    for (int r = tid; r < PL::N2; r += THREADS) {
      T2[r] = (unsigned short)PL::t2(r);
      D2[r] = (unsigned short)PL::d2(r);
      TJ[r] = tw_ls(twls, PL::N1 * r);
    }
  }
  BABE_HD static int col_k1(int tile, int col) {               // -1: empty column
    if (tile < NTP) {
      const int lo = 1 + H * tile + (col % H);
      if (lo > NP) return -1;
      return col < H ? lo : PL::N1 - lo;
    }
    if (col == 0) return 0;
    if (col == 1 && PL::N1 % 2 == 0) return PL::N1 / 2;
    return -1;
  }
  // rows of the intermediate (contiguous in r): one lane per row, 16 bytes (two r) per access
  BABE_HD static void load_rows(const float2* Y, float2* A, int tile, int tid) {
    const unsigned short* T2 = tab_t2(A);
    const int col = tid % S, slot = tid / S, k1 = col_k1(tile, col);
    if (k1 < 0) return;
    // 16-byte loads through registers, all of them issued before the first store: LDGSTS from 16 different rows
    // would write shared memory lane by lane as the sectors arrive (measured: twice the wavefronts)
    const float4* row = reinterpret_cast<const float4*>(Y + (size_t)PL::q1(k1) * PL::P2);
    constexpr int NCH = PL::P2 / 2, IT = (NCH + SLOTS - 1) / SLOTS;
    float4 v[IT];
#pragma unroll
    for (int it = 0; it < IT; ++it) {
      const int ch = slot + it * SLOTS;
      if (ch < NCH) v[it] = row[ch];
    }
#pragma unroll
    for (int it = 0; it < IT; ++it) {
      const int ch = slot + it * SLOTS, r = 2 * ch;
      if (ch < NCH) {
        A[T2[r] * S + col] = make_float2(v[it].x, v[it].y);
        if (r + 1 < PL::N2) A[T2[r + 1] * S + col] = make_float2(v[it].z, v[it].w);
      }
    }
  }
  BABE_HD static void store_rows(const float2* A, float2* Y, int tile, int tid) {
    const unsigned short* T2 = tab_t2(const_cast<float2*>(A));
    const int col = tid % S, slot = tid / S, k1 = col_k1(tile, col);
    if (k1 < 0) return;
    float4* row = reinterpret_cast<float4*>(Y + (size_t)PL::q1(k1) * PL::P2);
#pragma unroll 5
    for (int ch = slot; ch < PL::P2 / 2; ch += SLOTS) {
      const int r = 2 * ch;
      const float2 a = A[T2[r] * S + col];
      const float2 b = r + 1 < PL::N2 ? A[T2[r + 1] * S + col] : make_float2(0.f, 0.f);
      row[ch] = make_float4(a.x, a.y, b.x, b.y);
    }
  }
  template <bool INV>
  BABE_HD static void stage_d(float2* A, int tile, int tid) {
    if (col_k1(tile, tid % S) >= 0) stage<PL::RD, 1, PL::RE * PL::RF, S, INV>(A, tid / S, tid % S, SLOTS);
  }
  template <bool INV>
  BABE_HD static void stage_e(float2* A, int tile, int tid) {
    if (col_k1(tile, tid % S) >= 0) stage<PL::RE, PL::RD, PL::RF, S, INV>(A, tid / S, tid % S, SLOTS);
  }
  template <bool INV>
  BABE_HD static void stage_f(float2* A, int tile, int tid) {
    if (col_k1(tile, tid % S) >= 0) stage<PL::RF, PL::RD * PL::RE, 1, S, INV>(A, tid / S, tid % S, SLOTS);
  }
  template <bool INV>
  BABE_HD static void stages(float2* A, int tile, int tid) {
    stage_d<INV>(A, tile, tid); PFA_SYNC();
    if (PL::RE > 1) { stage_e<INV>(A, tile, tid); PFA_SYNC(); }
    if (PL::RF > 1) { stage_f<INV>(A, tile, tid); PFA_SYNC(); }
  }
  // every bin pair (k, Nc - k), k <= Nc - k, whose members live in this tile:
  //   f(k, index of Z[k], index of Z[Nc - k], W_Ls^k)
  // pair tiles: thread = (pair slot i = tid % H, j = tid / H + 32 it); bin k = k1 + N1 j, k mod N2 advanced incrementally
  template <class F>
  BABE_HD static void for_pairs(const float2* A, const float2* twls, int tile, int tid, F&& f) {
    const float2* TJ = tab_tj(const_cast<float2*>(A));
    const unsigned short* D2 = tab_d2(const_cast<float2*>(A));
    if (tile < NTP) {
      static_assert(THREADS % H == 0, "pair slot must be fixed per thread");
      constexpr int JSTEP = THREADS / H, RSTEP = ((PL::N1 % PL::N2) * JSTEP) % PL::N2;
      const int i = tid % H, k1 = 1 + H * tile + i;
      if (k1 > NP) return;
      const float2 W1 = tw_ls(twls, k1);
      int j = tid / H;
      int r2 = (k1 + (PL::N1 % PL::N2) * j) % PL::N2;
#pragma unroll 2
      for (; j < PL::N2; j += JSTEP) {
        f(k1 + PL::N1 * j, D2[r2] * S + i, D2[r2 ? PL::N2 - r2 : 0] * S + i + H, cmul(W1, TJ[j]));
        r2 += RSTEP;
        if (r2 >= PL::N2) r2 -= PL::N2;
      }
    } else {
      constexpr int NCOL = 1 + (PL::N1 % 2 == 0);
      for (int idx = tid; idx < NCOL * PL::N2; idx += THREADS) {
        const int c = idx % NCOL, j = idx / NCOL;
        const int k = (c ? PL::N1 / 2 : 0) + PL::N1 * j;
        if (2 * k > PL::NC) continue;
        const int r2 = k % PL::N2;
        f(k, D2[r2] * S + c, D2[r2 ? PL::N2 - r2 : 0] * S + c, tw_ls(twls, k));
      }
    }
  }
  // r2c: Z (tile) -> X[Nc + 1] natural order, times the optional real bin scale
  BABE_HD static void post_to_x(const float2* A, float2* X, const float2* twls, const float* scale, int tile,
                                int tid) {
    for_pairs(A, twls, tile, tid, [&](int k, int ia, int ib, float2 W) {
      const int kp = PL::NC - k;
      float2 Xk, Xkp;
      if (k == 0) {
        const float2 z0 = A[ia];
        Xk = make_float2(z0.x + z0.y, 0.f);
        Xkp = make_float2(z0.x - z0.y, 0.f);
      } else {
        post_pair(A[ia], A[ib], W, Xk, Xkp);
      }
      if (scale) { const float sk = scale[k], sp = scale[kp]; Xk.x *= sk; Xk.y *= sk; Xkp.x *= sp; Xkp.y *= sp; }
      X[k] = Xk;
      if (kp != k) X[kp] = Xkp;
    });
  }
  // r2c, multiply by the real H, c2r -- in place (apply_hpf_DC)
  BABE_HD static void mid_filter(float2* A, const float2* twls, const float* Hf, int tile, int tid) {
    for_pairs(A, twls, tile, tid, [&](int k, int ia, int ib, float2 W) {
      const int kp = PL::NC - k;
      float2 Xk, Xkp;
      if (k == 0) {
        const float2 z0 = A[ia];
        Xk = make_float2(z0.x + z0.y, 0.f);
        Xkp = make_float2(z0.x - z0.y, 0.f);
      } else {
        post_pair(A[ia], A[ib], W, Xk, Xkp);
      }
      const float hk = Hf[k], hp = Hf[kp];
      Xk.x *= hk; Xk.y *= hk; Xkp.x *= hp; Xkp.y *= hp;
      float2 Zk, Zkp;
      pre_pair(Xk, Xkp, W, 1.0f / (float)PL::NC, Zk, Zkp);          // conj(Z) / Nc
      A[ia] = make_float2(Zk.x, -Zk.y);
      if (k != 0 && kp != k) A[ib] = make_float2(Zkp.x, -Zkp.y);
    });
  }
  // overlap-add of the <= 3 band samples of bin k (GatherTab::src[k].xyz; w unused).  "No band" entries point at a
  // zero element of the row, so the three loads are unconditional and unmasked.
  struct Src3 { float2 t0, t1, t2; };
  BABE_HD static Src3 gather_load(const GatherTab& g, int4 s) {
    Src3 d;
    d.t0 = g.BS[s.x]; d.t1 = g.BS[s.y]; d.t2 = g.BS[s.z];
    return d;
  }
  BABE_HD static float2 gather_sum(const Src3& d, int4) {
    return make_float2(d.t0.x + d.t1.x + d.t2.x, d.t0.y + d.t1.y + d.t2.y);
  }
  BABE_HD static void pre_store(float2* A, int k, int ia, int ib, float2 a, float2 b, float2 W, const float* scale) {
    const int kp = PL::NC - k;
    if (scale) { const float sk = scale[k], sp = scale[kp]; a.x *= sk; a.y *= sk; b.x *= sp; b.y *= sp; }
    if (k == 0) { a.y = 0.f; b.y = 0.f; }
    float2 Zk, Zkp;
    pre_pair(a, b, W, 1.0f / (float)PL::NC, Zk, Zkp);
    A[ia] = make_float2(Zk.x, -Zk.y);
    if (k != 0 && kp != k) A[ib] = make_float2(Zkp.x, -Zkp.y);
  }
  // Gather variant of the c2r prologue for the pair tiles, software-pipelined: the table entries are fetched two
  // iterations ahead and the band samples one iteration ahead, so the dependent chain table -> sample (two L2
  // latencies per pair in the plain loop: long_scoreboard 7.4 of 13 stall cycles per issue) is off the critical path.
  BABE_HD static void pre_gather_pairs(float2* A, const GatherTab& g, const float2* twls, const float* scale, int tile,
                                       int tid) {
    const float2* TJ = tab_tj(A);
    const unsigned short* D2 = tab_d2(A);
    constexpr int JSTEP = THREADS / H, RSTEP = ((PL::N1 % PL::N2) * JSTEP) % PL::N2;
    const int i = tid % H, k1 = 1 + H * tile + i;
    if (k1 > NP) return;
    const float2 W1 = tw_ls(twls, k1);
    int j = tid / H;
    int r2 = (k1 + (PL::N1 % PL::N2) * j) % PL::N2;
    auto table = [&](int jj, int4& sa, int4& sb) {       // past the end: re-read the last pair's entries (unused)
      const int k = k1 + PL::N1 * min(jj, PL::N2 - 1);
      sa = g.src[k]; sb = g.src[PL::NC - k];
    };
    int4 sa0, sb0, sa1, sb1;
    table(j, sa0, sb0);
    table(j + JSTEP, sa1, sb1);
    Src3 da0 = gather_load(g, sa0), db0 = gather_load(g, sb0);
    for (; j < PL::N2; j += JSTEP) {
      int4 sa2, sb2;
      table(j + 2 * JSTEP, sa2, sb2);
      const Src3 da1 = gather_load(g, sa1), db1 = gather_load(g, sb1);
      pre_store(A, k1 + PL::N1 * j, D2[r2] * S + i, D2[r2 ? PL::N2 - r2 : 0] * S + i + H, gather_sum(da0, sa0),
                gather_sum(db0, sb0), cmul(W1, TJ[j]), scale);
      sa0 = sa1; sb0 = sb1; sa1 = sa2; sb1 = sb2; da0 = da1; db0 = db1;
      r2 += RSTEP;
      if (r2 >= PL::N2) r2 -= PL::N2;
    }
  }
  // c2r: X[Nc + 1] (or the gathered band spectra), times the optional bin scale -> Z / Nc (tile)
  template <bool GATHER>
  BABE_HD static void pre_from_x(float2* A, const float2* X, const GatherTab& g, const float2* twls,
                                 const float* scale, int tile, int tid) {
    if (GATHER && tile < NTP) { pre_gather_pairs(A, g, twls, scale, tile, tid); return; }
    for_pairs(A, twls, tile, tid, [&](int k, int ia, int ib, float2 W) {
      float2 a, b;
      if (GATHER) {
        const int4 sa = g.src[k], sb = g.src[PL::NC - k];
        a = gather_sum(gather_load(g, sa), sa); b = gather_sum(gather_load(g, sb), sb);
      } else {
        a = X[k]; b = X[PL::NC - k];
      }
      pre_store(A, k, ia, ib, a, b, W, scale);
    });
  }
};

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------------------------------
// kernels: grid (tiles, rows)
//
// Programmatic dependent launch: every kernel of a CQT chain lets its successor start as soon as all of its own CTAs
// are running (griddepcontrol.launch_dependents first thing) and builds its tables before it waits for the
// predecessor's results (griddepcontrol.wait: returns at once for a plain launch).  The successor's launch latency and
// prologue overlap the predecessor's last wave.  Nothing is read from or written to a buffer of the chain before
// the wait.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <class PL, int S>
__global__ void __launch_bounds__(THREADS, PL::MINB1) k_pfa1_fwd(const float2* __restrict__ x, float2* __restrict__ Y) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  using P = Pass1<PL, S>;
  float2* A = reinterpret_cast<float2*>(smem_raw);
  unsigned short* T1 = P::table(A);
  const int tid = threadIdx.x, tile = blockIdx.x;
  pdl_launch_dependents();
  P::tables(T1, tid);
  __syncthreads();
  pdl_wait();
  P::load_natural(x + (size_t)blockIdx.y * PL::NC, A, T1, tile, tid);
  __syncthreads();
  P::forward_to_rows(A, Y + (size_t)blockIdx.y * PL::N1 * PL::P2, tile, tid);
}

template <class PL, int S>
__global__ void __launch_bounds__(THREADS, PL::MINB1) k_pfa1_inv(const float2* __restrict__ Y, float2* __restrict__ x) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  using P = Pass1<PL, S>;
  float2* A = reinterpret_cast<float2*>(smem_raw);
  unsigned short* T1 = P::table(A);
  const int tid = threadIdx.x, tile = blockIdx.x;
  pdl_launch_dependents();
  P::tables(T1, tid);
  pdl_wait();
  P::inverse_from_rows(Y + (size_t)blockIdx.y * PL::N1 * PL::P2, A, tile, tid);
  P::store_natural(A, x + (size_t)blockIdx.y * PL::NC, T1, tile, tid);
}

struct P2Args {
  const float2* Y;         // intermediate in  [rows][N1][P2]
  float2* Yout;            // intermediate out [rows][N1][P2]
  const float2* X;         // half spectrum in  [rows][Nc + 1]
  float2* Xout;            // half spectrum out [rows][Nc + 1]
  const float2* BS;        // band spectra [rows][sum_lg]
  const int4* src;         // gather table [Nc + 1]
  int sum_lg;
  const float2* tw_ls;
  const float* scale;      // optional bin scale / the filter H
  int xpitch;              // row pitch of X / Xout in float2 (>= Nc + 1; Nc + 2: 16-byte rows, pad element zeroed)
};

// forward pass 2 + r2c -> X
template <class PL, int S>
__global__ void __launch_bounds__(THREADS, PL::MINB2) k_pfa2_fwd(const P2Args a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  using P = Pass2<PL, S>;
  float2* A = reinterpret_cast<float2*>(smem_raw);
  const int tid = threadIdx.x, tile = blockIdx.x;
  pdl_launch_dependents();
  P::tables(A, a.tw_ls, tid);
  __syncthreads();
  pdl_wait();
  P::load_rows(a.Y + (size_t)blockIdx.y * PL::N1 * PL::P2, A, tile, tid);
  __syncthreads();
  P::template stages<false>(A, tile, tid);
  float2* Xrow = a.Xout + (size_t)blockIdx.y * a.xpitch;
  P::post_to_x(A, Xrow, a.tw_ls, a.scale, tile, tid);
  if (tile == 0 && tid == 0 && a.xpitch > PL::NC + 1) Xrow[PL::NC + 1] = make_float2(0.f, 0.f);   // pad: staged by bulk copies
}

// forward pass 2, r2c, * H, c2r, inverse pass 2 (apply_hpf_DC)
template <class PL, int S>
__global__ void __launch_bounds__(THREADS, PL::MINB2) k_pfa2_mid(const P2Args a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  using P = Pass2<PL, S>;
  float2* A = reinterpret_cast<float2*>(smem_raw);
  const int tid = threadIdx.x, tile = blockIdx.x;
  pdl_launch_dependents();
  P::tables(A, a.tw_ls, tid);
  __syncthreads();
  pdl_wait();
  P::load_rows(a.Y + (size_t)blockIdx.y * PL::N1 * PL::P2, A, tile, tid);
  __syncthreads();
  P::template stages<false>(A, tile, tid);
  P::mid_filter(A, a.tw_ls, a.scale, tile, tid);
  __syncthreads();
  P::template stages<true>(A, tile, tid);
  P::store_rows(A, a.Yout + (size_t)blockIdx.y * PL::N1 * PL::P2, tile, tid);
}

// c2r from X (or gathered from the band spectra) + inverse pass 2
template <class PL, int S, bool GATHER>
__global__ void __launch_bounds__(THREADS, PL::MINB2) k_pfa2_inv(const P2Args a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  using P = Pass2<PL, S>;
  float2* A = reinterpret_cast<float2*>(smem_raw);
  const int tid = threadIdx.x, tile = blockIdx.x;
  pdl_launch_dependents();
  P::tables(A, a.tw_ls, tid);
  __syncthreads();
  pdl_wait();
  GatherTab g{GATHER ? a.BS + (size_t)blockIdx.y * a.sum_lg : nullptr, a.src};
  P::template pre_from_x<GATHER>(A, GATHER ? nullptr : a.X + (size_t)blockIdx.y * a.xpitch, g, a.tw_ls, a.scale,
                                 tile, tid);
  __syncthreads();
  P::template stages<true>(A, tile, tid);
  P::store_rows(A, a.Yout + (size_t)blockIdx.y * PL::N1 * PL::P2, tile, tid);
}
#endif  // __CUDACC__

}  // namespace pfa
}  // namespace babe
