// NSGT constant-Q transform kernels for sm_100a.
//
// Real FFT of the whole segment (Ls = 184184 = 2^3*7*11*13*23 in the shipped
// 22.05 kHz configuration -- not a power of two) as a complex FFT of
// Nc = Ls/2 = n1*n2 points in two passes ("four-step"): every CTA transforms a
// tile of 8 interleaved sequences entirely in shared memory with a mixed-radix
// Stockham FFT (smemfft.cuh), so each pass reads and writes the row once with
// >= 64-byte contiguous segments and the intermediate stays in L2.  The
// constant-Q filterbank (window multiply, fold, per-band power-of-two iFFT) is
// one further kernel per direction; overlap-add of the synthesis bands is a
// deterministic gather (no atomics) fused with the c2r pre-processing.
//
// Semantics: oracle/nsgt.py (specification) -- upstream cqt_nsgt_pytorch is not
// available, see DESIGN.md "CQT parity".  Reference call sites:
// networks/cqtdiff+.py:620,743,841; testing/blind_bwe_sampler.py:156.
#include <math.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "bandfft_v.cuh"
#include "tma.cuh"
#include "smemfft.cuh"
#include "rfft_pairs.cuh"
#include "cqt_pfa.cuh"

namespace babe {

constexpr int CQT_THREADS = 256;
constexpr int MAX_TB = 64;          // bands per CTA (tb <= 2048 / 32)
constexpr int BAND_THREADS = 256;   // band kernels: 16 points per thread, 4096-point tiles (bandfft_v.cuh)
constexpr int TILE_SEQ = 8;          // sequences per CTA in the two big-FFT passes
constexpr int TW_LO = 1024;          // low part of the two-level twiddle tables

__device__ __forceinline__ float2 tw2(const float2* tab, int m) {
  // exp(-2 pi i m / n) = lo[m & 1023] * hi[m >> 10]
  return cmul(tab[m & (TW_LO - 1)], tab[TW_LO + (m >> 10)]);
}

static inline int odd_stride(int n) { return padded_len(n); }

// ---------------------------------------------------------------------------
// pass 1: for a tile of n2, FFT over n1 (stride n2), twiddle W_Nc^{n2 k1},
// store as Y[k1][n2]
// ---------------------------------------------------------------------------
struct PassArgs {
  const float2* in; float2* out;
  int Nc, N1, N2;
  FastDiv div_n2;
  FftFactors f;
  const float2* roots;   // n-th roots of this pass
  const float2* tw_nc;   // two-level W_Nc (pass 1 only)
  int conj_out;          // pass 2: conjugate on store (inverse transforms)
};

__global__ void __launch_bounds__(CQT_THREADS, 3) k_fft_cols(const PassArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int S = padded_len(a.N1);
  float2* A = reinterpret_cast<float2*>(smem_raw);
  float2* Bf = A + TILE_SEQ * S;
  float2* roots = Bf + TILE_SEQ * S;
  float2* tw = roots + a.N1;
  const int n_hi = (a.Nc >> 10) + 1;
  const int tid = threadIdx.x;
  for (int i = tid; i < a.N1; i += CQT_THREADS) roots[i] = a.roots[i];
  for (int i = tid; i < TW_LO + n_hi; i += CQT_THREADS) tw[i] = a.tw_nc[i];
  const int n2_0 = blockIdx.x * TILE_SEQ;
  const float2* in = a.in + (size_t)blockIdx.y * a.Nc;
  float2* out = a.out + (size_t)blockIdx.y * a.Nc;
  for (int idx = tid; idx < TILE_SEQ * a.N1; idx += CQT_THREADS) {
    const int n2l = idx % TILE_SEQ, n1 = idx / TILE_SEQ;
    const int n2 = n2_0 + n2l;
    float2 v = make_float2(0.f, 0.f);
    if (n2 < a.N2) v = in[(size_t)a.N2 * n1 + n2];
    A[n2l * S + pad16(n1)] = v;
  }
  __syncthreads();
  const float2* res = smem_fft(A, Bf, a.f, S, TILE_SEQ, roots, tid, CQT_THREADS);
  for (int idx = tid; idx < TILE_SEQ * a.N1; idx += CQT_THREADS) {
    const int n2l = idx % TILE_SEQ, k1 = idx / TILE_SEQ;
    const int n2 = n2_0 + n2l;
    if (n2 < a.N2) out[(size_t)k1 * a.N2 + n2] = cmul(res[n2l * S + pad16(k1)], tw2(tw, n2 * k1));
  }
}

// pass 2: for a tile of k1, FFT over n2 (contiguous), store Z[k1 + N1 k2]
__global__ void __launch_bounds__(CQT_THREADS, 3) k_fft_rows(const PassArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int S = padded_len(a.N2);
  float2* A = reinterpret_cast<float2*>(smem_raw);
  float2* Bf = A + TILE_SEQ * S;
  float2* roots = Bf + TILE_SEQ * S;
  const int tid = threadIdx.x;
  for (int i = tid; i < a.N2; i += CQT_THREADS) roots[i] = a.roots[i];
  const int k1_0 = blockIdx.x * TILE_SEQ;
  const float2* in = a.in + (size_t)blockIdx.y * a.Nc;
  float2* out = a.out + (size_t)blockIdx.y * a.Nc;
  for (int idx = tid; idx < TILE_SEQ * a.N2; idx += CQT_THREADS) {
    const int k1l = a.div_n2.div(idx), n2 = idx - k1l * a.N2;
    const int k1 = k1_0 + k1l;
    float2 v = make_float2(0.f, 0.f);
    if (k1 < a.N1) v = in[(size_t)k1 * a.N2 + n2];
    A[k1l * S + pad16(n2)] = v;
  }
  __syncthreads();
  const float2* res = smem_fft(A, Bf, a.f, S, TILE_SEQ, roots, tid, CQT_THREADS);
  for (int idx = tid; idx < TILE_SEQ * a.N2; idx += CQT_THREADS) {
    const int k1l = idx % TILE_SEQ, k2 = idx / TILE_SEQ;
    const int k1 = k1_0 + k1l;
    if (k1 < a.N1) {
      float2 v = res[k1l * S + pad16(k2)];
      if (a.conj_out) v.y = -v.y;
      out[(size_t)k1 + (size_t)a.N1 * k2] = v;
    }
  }
}

// ---------------------------------------------------------------------------
// r2c post-processing / c2r pre-processing on bin pairs (k, Nc-k)
// ---------------------------------------------------------------------------
__global__ void k_rfft_post(const float2* Z, float2* X, int Nc, const float2* tw_ls,
                            const float* scale) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > Nc / 2) return;
  const float2* z = Z + (size_t)blockIdx.y * Nc;
  float2* x = X + (size_t)blockIdx.y * (Nc + 1);
  if (k == 0) {
    const float2 z0 = z[0];
    const float s0 = scale ? scale[0] : 1.f, sn = scale ? scale[Nc] : 1.f;
    x[0] = make_float2((z0.x + z0.y) * s0, 0.f);
    x[Nc] = make_float2((z0.x - z0.y) * sn, 0.f);
    return;
  }
  const int kp = Nc - k;
  float2 Xk, Xkp;
  post_pair(z[k], z[kp], tw2(tw_ls, k), Xk, Xkp);
  if (scale) { const float sk = scale[k], sp = scale[kp]; Xk.x *= sk; Xk.y *= sk; Xkp.x *= sp; Xkp.y *= sp; }
  x[k] = Xk;
  if (kp != k) x[kp] = Xkp;
}

__global__ void k_irfft_pre(const float2* X, float2* Zc, int Nc, const float2* tw_ls,
                            const float* scale) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > Nc / 2) return;
  const float2* x = X + (size_t)blockIdx.y * (Nc + 1);
  float2* z = Zc + (size_t)blockIdx.y * Nc;
  const int kp = Nc - k;
  float2 a = x[k], b = x[kp];
  if (scale) { const float sk = scale[k], sp = scale[kp]; a.x *= sk; a.y *= sk; b.x *= sp; b.y *= sp; }
  if (k == 0) { a.y = 0.f; b.y = 0.f; }
  float2 Zk, Zkp;
  pre_pair(a, b, tw2(tw_ls, k), 1.0f / (float)Nc, Zk, Zkp);
  z[k] = Zk;
  if (k != 0 && kp != k) z[kp] = Zkp;
}

// rfft post * H * irfft pre in one pass (apply_hpf_DC)
__global__ void k_spectral_mid(const float2* Z, float2* Zc, int Nc, const float2* tw_ls,
                               const float* H) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > Nc / 2) return;
  const float2* zi = Z + (size_t)blockIdx.y * Nc;
  float2* zo = Zc + (size_t)blockIdx.y * Nc;
  const int kp = Nc - k;
  const float2 W = tw2(tw_ls, k);
  float2 Xk, Xkp;
  if (k == 0) {
    const float2 z0 = zi[0];
    Xk = make_float2(z0.x + z0.y, 0.f);
    Xkp = make_float2(z0.x - z0.y, 0.f);
  } else {
    post_pair(zi[k], zi[kp], W, Xk, Xkp);
  }
  const float hk = H[k], hp = H[kp];
  Xk.x *= hk; Xk.y *= hk; Xkp.x *= hp; Xkp.y *= hp;
  float2 Zk, Zkp;
  pre_pair(Xk, Xkp, W, 1.0f / (float)Nc, Zk, Zkp);
  zo[k] = Zk;
  if (k != 0 && kp != k) zo[kp] = Zkp;
}

// ---------------------------------------------------------------------------
// constant-Q bands
// ---------------------------------------------------------------------------
struct BandArgs {
  int Nc, numocts, binsoct, sum_lg;          // sum_lg: row pitch of BS (samples + 2)
  int M[BABE_MAX_OCTAVES];
  int tb[BABE_MAX_OCTAVES];              // bands per CTA in octave o
  int tile0[BABE_MAX_OCTAVES + 1];       // first work item of octave o
  FftFactors fm[BABE_MAX_OCTAVES];
  const float2* rootsm[BABE_MAX_OCTAVES];
  float2* coef[BABE_MAX_OCTAVES];        // per-octave coefficient tensors [B, binsoct, M] complex
  int planar;                            // 1: float [B, 2, binsoct, M] (re plane, im plane) instead
  int B, rows_per_cta, band_variant;
  int xpitch;                            // row pitch of X in float2 (Nc + 1, or Nc + 2 when the slices are bulk-copied)
  const int* band_p; const int* band_lg; const int* band_off;
  const float* win; const float* scale;
  const float2* X;                       // analysis: half spectrum [B, Nc+1]
  float2* BS;                            // synthesis: band spectra [B, sum_lg]
};

__device__ __forceinline__ int find_octave(const BandArgs& a, int item) {
  int o = 0;
  while (o + 1 < a.numocts && item >= a.tile0[o + 1]) ++o;
  return o;
}

// cp.async staging of the band kernels: the 16 input values of a thread for row r+1 (a window slice of the half
// spectrum, or a coefficient row) are copied global -> shared with 8-byte cp.async while row r is transformed.  Loaded
// straight into registers at the top of every row they sat on the scoreboard (long_scoreboard 7.7 of 13 stall cycles
// per issue, profiles/r01_cqt_B64.md).
__device__ __forceinline__ void cp_async8(void* dst, const void* src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4f(void* dst, const void* src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

// --- octaves with M = 32 ... 4096: packed register FFT (bandfft_v.cuh), 4096 / M bands per CTA (M >= 256) ----------
// The transform works on float2 register pairs with the two-wide instructions, runs forward or inverse directly (no
// conjugations), takes the window (and 1 / M) multiply in its first butterflies, and synchronises per band.
// Inputs of a row are staged one row ahead:
//   TMA = true : (analysis only) by the TMA engine -- per band ONE 1-D bulk copy (cp.async.bulk + mbarrier, SASS
//                UBLKCP) of the contiguous window slice X[p - lg/2 .. p + lg/2) (start rounded down / length rounded up
//                to 16 bytes, the row pitch of X is even), issued by one thread per synchronisation group right behind
//                the band's first barrier; no per-thread address / predicate / LDGSTS work in the row loop;
//   TMA = false: by 16 8-byte cp.async per thread: any alignment / pitch.
template <class C, bool SYNTH, bool TMA>
__device__ __forceinline__ void band_tile_v(const BandArgs& a, int o, int tile, int row0, int row_end,
                                            unsigned char* smem_raw) {
  static_assert(!(SYNTH && TMA), "the synthesis stages its coefficient rows with cp.async");
  constexpr int NB = BAND_THREADS / C::TPB, M = C::M, NTWP = (C::NTW + 1) & ~1;
  constexpr int GT = C::TPB < 32 ? 32 : C::TPB;            // threads per synchronisation group (>= one warp)
  constexpr int NG = BAND_THREADS / GT, BPG = GT / C::TPB; // groups per CTA, bands per group
  constexpr int SB = M + 2;                                // staged float2 per band (TMA): slice + alignment pads
  constexpr int STAGE = TMA ? NB * SB : 16 * BAND_THREADS;
  float2* exs = reinterpret_cast<float2*>(smem_raw);
  float2* tw = exs + ((NB * C::EXP + 1) & ~1);
  float2* stage = tw + NTWP;                           // TMA: [NB][SB] natural order; else [16][BAND_THREADS]
  float* wst = reinterpret_cast<float*>(stage + STAGE);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(wst + 16 * BAND_THREADS);      // [NG]
  int* s_src = reinterpret_cast<int*>(mbar + NG);      // [NB] first staged element of the band's slice (analysis)
  int* s_cnt = s_src + NB;                             // [NB] staged elements
  const int tid = threadIdx.x, bl = tid / C::TPB, t = tid % C::TPB, grp = tid / GT;
  const float2* roots_m = a.rootsm[o];
  for (int i = tid; i < C::NTW; i += BAND_THREADS) tw[i] = C::twiddle(roots_m, i);
  typename C::Regs rg;
  C::init_regs(rg, roots_m, t);
  const int band = tile * NB + bl;
  const bool active = band < a.binsoct;
  int p = 0, lg = 0, off = 0;
  if (active) {
    const int j = o * a.binsoct + band;
    p = a.band_p[j]; lg = a.band_lg[j]; off = a.band_off[j];
  }
  const int half = lg / 2;
  float2* ex = exs + bl * C::EXP;
  float2* stage_b = stage + bl * SB;
  unsigned valid = 0;
  int sdelta = 0;                                      // TMA analysis: stage index of window sample i is i + sdelta
  if (!SYNTH) {
    // window sample (times the optional bin scale and 1 / M) of the thread's 16 INPUT slots; 0 = outside the window
    const float inv_m = 1.0f / (float)M;
#pragma unroll
    for (int n1 = 0; n1 < 16; ++n1) {
      int i = C::in_slot(n1, t) + half;
      if (i >= M) i -= M;
      float w = 0.f;
      const int k = p - half + i;
      if (active && i < lg && k >= 0 && k <= a.Nc) {
        w = a.win[off + i] * inv_m;
        if (a.scale) w *= a.scale[k];
        valid |= 1u << n1;
      }
      wst[n1 * BAND_THREADS + tid] = w;
      if (!TMA) stage[n1 * BAND_THREADS + tid] = make_float2(0.f, 0.f);
    }
    if (TMA) {
      // slice [kstart, kend) of the row, widened to 16-byte boundaries; staged slots outside it keep their zeros
      const int start = p - half, kstart = max(start, 0), kend = min(start + lg, a.Nc + 1);
      const int s0 = kstart & ~1, cnt = active && kend > s0 ? ((kend - s0 + 1) & ~1) : 0;
      sdelta = start - s0;
      if (t == 0) { s_src[bl] = s0; s_cnt[bl] = cnt; }
      for (int i = t; i < SB; i += C::TPB) stage_b[i] = make_float2(0.f, 0.f);
    }
  } else {
    // dual-window sample of the thread's 16 OUTPUT slots
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      int i = C::out_slot(r, t) + half;
      if (i >= M) i -= M;
      wst[r * BAND_THREADS + tid] = (active && i < lg) ? a.win[off + i] : 0.f;
    }
  }
  if (TMA && tid < NG) tma::mbar_init(mbar + tid, 1);
  if (TMA) tma::fence_proxy_async();                   // zeros / barrier inits before the first bulk copy
  // ---- staging of one row ------------------------------------------------------------------------------
  auto prefetch = [&](int row) {
    if (TMA) {
      if (tid % GT != 0) return;                       // one thread per synchronisation group
      uint64_t* bar = mbar + grp;
      unsigned total = 0;
#pragma unroll
      for (int b = 0; b < BPG; ++b) total += (unsigned)s_cnt[grp * BPG + b] * 8u;
      if (total == 0) { tma::mbar_arrive(bar); return; }
      tma::mbar_arrive_tx(bar, total);
#pragma unroll
      for (int b = 0; b < BPG; ++b) {
        const int bb = grp * BPG + b, cnt = s_cnt[bb];
        if (cnt == 0) continue;
        tma::bulk_g2s(stage + bb * SB, a.X + (size_t)row * a.xpitch + s_src[bb], cnt * 8u, bar);
      }
      return;
    }
    if (!SYNTH) {
      const float2* X = a.X + (size_t)row * a.xpitch + (p - half);
#pragma unroll
      for (int n1 = 0; n1 < 16; ++n1) {
        int i = C::in_slot(n1, t) + half;
        if (i >= M) i -= M;
        if (valid & (1u << n1)) cp_async8(stage + n1 * BAND_THREADS + tid, X + i);
      }
    } else if (active) {
      if (!a.planar) {
        const float2* in = a.coef[o] + ((size_t)row * a.binsoct + band) * M;
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) cp_async8(stage + n1 * BAND_THREADS + tid, in + C::in_slot(n1, t));
      } else {
        const float* ire = reinterpret_cast<const float*>(a.coef[o]) + (((size_t)row * 2) * a.binsoct + band) * M;
        const float* iim = ire + (size_t)a.binsoct * M;
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
          float* d = reinterpret_cast<float*>(stage + n1 * BAND_THREADS + tid);
          cp_async4f(d, ire + C::in_slot(n1, t));
          cp_async4f(d + 1, iim + C::in_slot(n1, t));
        }
      }
    }
  };
  if (TMA) __syncthreads();                            // barrier inits, slice descriptors, zeroed stage
  pfa::pdl_wait();                                     // everything above read plan constants only
  if (row0 < row_end) prefetch(row0);
  __syncthreads();                                     // twiddle table
  unsigned phase = 0;
  for (int row = row0; row < row_end; ++row) {
    float2 z[16];
    float s[16];
    if (TMA) {
      tma::mbar_wait(mbar + grp, phase);
      phase ^= 1u;
#pragma unroll
      for (int n1 = 0; n1 < 16; ++n1) {
        int i = C::in_slot(n1, t) + half;
        if (i >= M) i -= M;
        i = min(max(i + sdelta, 0), SB - 1);             // slots outside the slice carry weight 0
        z[n1] = stage_b[i];
      }
    } else {
      cp_async_commit_wait();                         // this thread's own copies: no barrier needed to read them
      if (SYNTH && !active) {
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) z[n1] = make_float2(0.f, 0.f);
      } else {
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) z[n1] = stage[n1 * BAND_THREADS + tid];
      }
    }
    if (!SYNTH) {
#pragma unroll
      for (int n1 = 0; n1 < 16; ++n1) s[n1] = wst[n1 * BAND_THREADS + tid];
    }
    const bool more = row + 1 < row_end;
    if (!TMA && more) prefetch(row + 1);              // the staged values are in registers: the slots are free
    C::template fwd<!SYNTH>(z, s, ex, tw, rg, t, 1 + bl, [&]() { if (TMA && more) prefetch(row + 1); });
    if (active) {
      if (!SYNTH) {
        if (!a.planar) {
          float2* out = a.coef[o] + ((size_t)row * a.binsoct + band) * M;
#pragma unroll
          for (int r = 0; r < 16; ++r) out[C::out_slot(r, t)] = z[r];
        } else {   // the layout the denoiser consumes (networks/cqtdiff+.py:750-753) without the transposing copy
          float* ore = reinterpret_cast<float*>(a.coef[o]) + (((size_t)row * 2) * a.binsoct + band) * M;
          float* oim = ore + (size_t)a.binsoct * M;
#pragma unroll
          for (int r = 0; r < 16; ++r) {
            ore[C::out_slot(r, t)] = z[r].x;
            oim[C::out_slot(r, t)] = z[r].y;
          }
        }
      } else {
        float2* BS = a.BS + (size_t)row * a.sum_lg + off;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          int i = C::out_slot(r, t) + half;
          if (i >= M) i -= M;
          if (i < lg) BS[i] = c_scale(z[r], wst[r * BAND_THREADS + tid]);
        }
      }
    }
    band_sync<C::TPB>(1 + bl);                      // the band's exchange buffer is reused by its next row
  }
}

// --- other octave sizes: mixed-radix Stockham in shared memory -------------------------------
template <bool SYNTH>
__device__ __forceinline__ void band_tile_generic(const BandArgs& a, int o, int tile, int row0, int row_end,
                                                  unsigned char* smem_raw) {
  const int M = a.M[o], S = padded_len(M), TB = a.tb[o];
  const int mshift = 31 - __clz(M);              // octave sizes are powers of two
  const int b0 = tile * TB;
  const int nb = min(TB, a.binsoct - b0);
  float2* A = reinterpret_cast<float2*>(smem_raw);
  float2* Bf = A + TB * S;
  float2* roots = Bf + TB * S;
  const int tid = threadIdx.x, nthr = blockDim.x;
  for (int i = tid; i < M; i += nthr) roots[i] = a.rootsm[o][i];
  // band descriptors once per CTA (they would otherwise be chains of dependent global loads)
  __shared__ int s_p[MAX_TB], s_lg[MAX_TB], s_off[MAX_TB];
  for (int i = tid; i < nb; i += nthr) {
    const int j = o * a.binsoct + b0 + i;
    s_p[i] = a.band_p[j]; s_lg[i] = a.band_lg[j]; s_off[i] = a.band_off[j];
  }
  __syncthreads();
  const float inv_m = 1.0f / (float)M;
  for (int row = row0; row < row_end; ++row) {
    if (!SYNTH) {
      const float2* X = a.X + (size_t)row * a.xpitch;
#pragma unroll 4
      for (int idx = tid; idx < nb * M; idx += nthr) {
        const int bl = idx >> mshift, m = idx & (M - 1);
        const int lg = s_lg[bl], half = lg / 2;
        int i = m + half;
        if (i >= M) i -= M;
        float2 v = make_float2(0.f, 0.f);
        if (i < lg) {
          const int k = s_p[bl] - half + i;
          if (k >= 0 && k <= a.Nc) {
            float w = a.win[s_off[bl] + i];
            if (a.scale) w *= a.scale[k];
            const float2 xv = X[k];
            v = make_float2(xv.x * w, -xv.y * w);      // conjugate: inverse FFT via forward
          }
        }
        A[bl * S + pad16(m)] = v;
      }
    } else if (!a.planar) {
      const float2* in = a.coef[o] + ((size_t)row * a.binsoct + b0) * M;
#pragma unroll 4
      for (int idx = tid; idx < nb * M; idx += nthr) {
        const int bl = idx >> mshift, m = idx & (M - 1);
        A[bl * S + pad16(m)] = in[(size_t)bl * M + m];
      }
    } else {
      const float* ire = reinterpret_cast<const float*>(a.coef[o]) + (((size_t)row * 2) * a.binsoct + b0) * M;
      const float* iim = ire + (size_t)a.binsoct * M;
#pragma unroll 4
      for (int idx = tid; idx < nb * M; idx += nthr) {
        const int bl = idx >> mshift, m = idx & (M - 1);
        A[bl * S + pad16(m)] = make_float2(ire[(size_t)bl * M + m], iim[(size_t)bl * M + m]);
      }
    }
    __syncthreads();
    const float2* res = smem_fft(A, Bf, a.fm[o], S, nb, roots, tid, nthr);
    if (!SYNTH) {
      if (!a.planar) {
        float2* out = a.coef[o] + ((size_t)row * a.binsoct + b0) * M;
        for (int idx = tid; idx < nb * M; idx += nthr) {
          const int bl = idx >> mshift, m = idx & (M - 1);
          const float2 v = res[bl * S + pad16(m)];
          out[(size_t)bl * M + m] = make_float2(v.x * inv_m, -v.y * inv_m);
        }
      } else {
        float* ore = reinterpret_cast<float*>(a.coef[o]) + (((size_t)row * 2) * a.binsoct + b0) * M;
        float* oim = ore + (size_t)a.binsoct * M;
        for (int idx = tid; idx < nb * M; idx += nthr) {
          const int bl = idx >> mshift, m = idx & (M - 1);
          const float2 v = res[bl * S + pad16(m)];
          ore[(size_t)bl * M + m] = v.x * inv_m;
          oim[(size_t)bl * M + m] = -v.y * inv_m;
        }
      }
    } else {
      float2* BS = a.BS + (size_t)row * a.sum_lg;
#pragma unroll 4
      for (int idx = tid; idx < nb * M; idx += nthr) {
        const int bl = idx >> mshift, m = idx & (M - 1);
        const int lg = s_lg[bl], half = lg / 2;
        int i = m + half;
        if (i >= M) i -= M;
        if (i < lg) {
          const float w = a.win[s_off[bl] + i];
          const float2 v = res[bl * S + pad16(m)];
          BS[s_off[bl] + i] = make_float2(v.x * w, v.y * w);
        }
      }
    }
    __syncthreads();                             // A / Bf are reused by the next row
  }
}

template <bool SYNTH, bool TMA>
__device__ __forceinline__ void band_segment(const BandArgs& a, int o, int tile, int row0, int row_end,
                                             unsigned char* smem_raw) {
  switch (a.M[o]) {                  // analysis = inverse transform of the windowed slice, synthesis = forward
    case 32: band_tile_v<BandCoreS<2, !SYNTH>, SYNTH, TMA>(a, o, tile, row0, row_end, smem_raw); break;
    case 64: band_tile_v<BandCoreS<4, !SYNTH>, SYNTH, TMA>(a, o, tile, row0, row_end, smem_raw); break;
    case 128: band_tile_v<BandCoreS<8, !SYNTH>, SYNTH, TMA>(a, o, tile, row0, row_end, smem_raw); break;
    case 256: band_tile_v<BandCoreV<1, !SYNTH>, SYNTH, TMA>(a, o, tile, row0, row_end, smem_raw); break;
    case 512: band_tile_v<BandCoreV<2, !SYNTH>, SYNTH, TMA>(a, o, tile, row0, row_end, smem_raw); break;
    case 1024: band_tile_v<BandCoreV<4, !SYNTH>, SYNTH, TMA>(a, o, tile, row0, row_end, smem_raw); break;
    case 2048: band_tile_v<BandCoreV<8, !SYNTH>, SYNTH, TMA>(a, o, tile, row0, row_end, smem_raw); break;
    case 4096: band_tile_v<BandCoreV<16, !SYNTH>, SYNTH, TMA>(a, o, tile, row0, row_end, smem_raw); break;
    default: pfa::pdl_wait(); band_tile_generic<SYNTH>(a, o, tile, row0, row_end, smem_raw); break;
  }
}

template <bool SYNTH, bool TMA>
__device__ __forceinline__ void band_tile(const BandArgs& a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // The successor of a band kernel is triggered when a CTA is DONE, not when it starts: the grid is one wave of
  // 128-register CTAs, and successors started at once sit on the SMs next to the running tiles for the whole kernel
  // (synthesis 0.155 -> 0.178 ms at B = 64 with the early trigger).
  const int o = find_octave(a, blockIdx.x);
  const int row0 = blockIdx.y * a.rows_per_cta, row_end = min(a.B, row0 + a.rows_per_cta);
  band_segment<SYNTH, TMA>(a, o, blockIdx.x - a.tile0[o], row0, row_end, smem_raw);
  pfa::pdl_launch_dependents();
  if (SYNTH && blockIdx.x == 0 && threadIdx.x < 2)          // the "no band" entries of the rows (a.sum_lg = pitch)
    for (int row = row0; row < row_end; ++row)
      a.BS[(size_t)row * a.sum_lg + a.sum_lg - 2 + threadIdx.x] = make_float2(0.f, 0.f);
}

// analysis: window multiply + fold + per-band inverse FFT of the half spectrum X
// synthesis, first half: per-band FFT of the coefficients, dual-window multiply -> band spectra BS
// TMA: window slices staged by bulk copies (default); the cp.async analysis serves spectra that cannot be bulk-copied
template <bool TMA>
__global__ void __launch_bounds__(BAND_THREADS, 2) k_cqt_analysis(const BandArgs a) { band_tile<false, TMA>(a); }
__global__ void __launch_bounds__(BAND_THREADS, 2) k_cqt_synth_bands(const BandArgs a) { band_tile<true, false>(a); }

// overlap-add of the band spectra as a gather, fused with the c2r pre-processing
struct GatherArgs {
  const float2* BS; float2* Zc; int Nc, sum_lg;
  const int* band_p; const int* band_lg; const int* band_off;
  const int* jlo; const int* jhi;
  const float* scale; const float2* tw_ls;
};

__device__ __forceinline__ float2 gather_bin(const GatherArgs& a, const float2* bs, int k) {
  float2 s = make_float2(0.f, 0.f);
  const int hi = a.jhi[k];
  for (int j = a.jlo[k]; j <= hi; ++j) {
    const int lg = a.band_lg[j];
    const int i = k - a.band_p[j] + lg / 2;
    if (i >= 0 && i < lg) {
      const float2 v = bs[a.band_off[j] + i];
      s.x += v.x; s.y += v.y;
    }
  }
  if (a.scale) { const float sc = a.scale[k]; s.x *= sc; s.y *= sc; }
  return s;
}

__global__ void k_cqt_gather_pre(const GatherArgs a) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > a.Nc / 2) return;
  const float2* bs = a.BS + (size_t)blockIdx.y * a.sum_lg;
  float2* z = a.Zc + (size_t)blockIdx.y * a.Nc;
  const int kp = a.Nc - k;
  float2 Xk = gather_bin(a, bs, k);
  float2 Xkp = gather_bin(a, bs, kp);
  if (k == 0) { Xk.y = 0.f; Xkp.y = 0.f; }
  float2 Zk, Zkp;
  pre_pair(Xk, Xkp, tw2(a.tw_ls, k), 1.0f / (float)a.Nc, Zk, Zkp);
  z[k] = Zk;
  if (k != 0 && kp != k) z[kp] = Zkp;
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static inline FftFactors to_dev(const babe_fft_factors& f) {
  FftFactors d;
  d.n = f.n; d.nf = f.nf;
  for (int i = 0; i < MAX_FACTORS; ++i) d.radix[i] = f.radix[i];
  fill_fastdiv(d);
  return d;
}

static bool radix_ok(int r) {
  switch (r) { case 2: case 3: case 4: case 5: case 7: case 8: case 11: case 13: case 16:
    case 17: case 19: case 23: return true; }
  return false;
}

static int validate_factors(const babe_fft_factors& f, const char* what) {
  BABE_REQUIRE(f.n >= 1 && f.nf >= 0 && f.nf <= MAX_FACTORS, BABE_EBADARG, "%s: bad factor list", what);
  long long p = 1;
  for (int i = 0; i < f.nf; ++i) {
    BABE_REQUIRE(radix_ok(f.radix[i]), BABE_EUNSUPPORTED, "%s: unsupported radix %d", what, f.radix[i]);
    p *= f.radix[i];
  }
  BABE_REQUIRE(p == f.n, BABE_EBADARG, "%s: factors multiply to %lld, not %d", what, p, f.n);
  return BABE_OK;
}

static int validate_plan(const babe_cqt_plan* p, bool bands) {
  BABE_REQUIRE(p != nullptr, BABE_EBADARG, "null plan");
  BABE_REQUIRE(p->Ls >= 4 && p->Ls % 2 == 0 && p->Nc == p->Ls / 2, BABE_EUNSUPPORTED,
               "signal length %d must be even", p->Ls);
  int rc = validate_factors(p->f1, "f1");
  if (rc) return rc;
  rc = validate_factors(p->f2, "f2");
  if (rc) return rc;
  BABE_REQUIRE((long long)p->f1.n * p->f2.n == p->Nc, BABE_EBADARG, "n1*n2 != Nc");
  BABE_REQUIRE(p->roots1 && p->roots2 && p->tw_nc && p->tw_ls, BABE_EBADARG, "plan tables missing");
  const size_t smem1 = sizeof(float2) * ((size_t)2 * TILE_SEQ * odd_stride(p->f1.n) + p->f1.n + TW_LO + (p->Nc >> 10) + 1);
  const size_t smem2 = sizeof(float2) * ((size_t)2 * TILE_SEQ * odd_stride(p->f2.n) + p->f2.n);
  BABE_REQUIRE(smem1 <= 220 * 1024 && smem2 <= 220 * 1024, BABE_EUNSUPPORTED,
               "pass lengths %d x %d do not fit shared memory", p->f1.n, p->f2.n);
  if (bands) {
    BABE_REQUIRE(p->numocts >= 1 && p->numocts <= BABE_MAX_OCTAVES && p->binsoct >= 1, BABE_EBADARG,
                 "bad octave layout");
    BABE_REQUIRE(p->band_p && p->band_lg && p->band_off && p->bin_jlo && p->bin_jhi && p->sum_lg > 0,
                 BABE_EBADARG, "band tables missing");
    for (int o = 0; o < p->numocts; ++o) {
      rc = validate_factors(p->fm[o], "fm");
      if (rc) return rc;
      BABE_REQUIRE(p->fm[o].n == p->M[o] && p->rootsm[o] != nullptr, BABE_EBADARG, "octave %d tables", o);
      BABE_REQUIRE(p->M[o] <= 8192, BABE_EUNSUPPORTED, "octave size %d > 8192", p->M[o]);
    }
  }
  return BABE_OK;
}

struct Workspace {
  float2 *bufA, *bufB, *bufX, *bufS;
};

// row pitch of the synthesis band spectra: sum_lg samples + a zero entry (two, for alignment) that the gather table
// of the prime-factor inverse points at for "no band" (bin_src = sum_lg), written by k_cqt_synth_bands
static int bs_pitch(const babe_cqt_plan* p) { return std::max(p->sum_lg, 0) + 2; }
// per-row elements of the two pass buffers: the prime-factor intermediate pads its rows to an even pitch
static size_t pass_row(const babe_cqt_plan* p) { return ((size_t)p->Nc + p->f1.n + 8) & ~(size_t)7; }
static size_t ws_bytes(const babe_cqt_plan* p, int B) {
  return sizeof(float2) * (size_t)B * (2 * pass_row(p) + (((size_t)p->Nc + 8) & ~(size_t)7) +
                                       (size_t)bs_pitch(p)) + 256;
}

static int carve(const babe_cqt_plan* p, int B, void* ws, size_t bytes, Workspace& w) {
  BABE_REQUIRE(B <= 65535, BABE_EBADARG, "batch %d > 65535 rows per call (grid.y); split the batch", B);
  BABE_REQUIRE(ws != nullptr && bytes >= ws_bytes(p, B), BABE_EBADARG, "workspace too small (%zu < %zu)",
               bytes, ws_bytes(p, B));
  w.bufA = static_cast<float2*>(ws);
  w.bufB = w.bufA + (size_t)B * pass_row(p);
  w.bufX = w.bufB + (size_t)B * pass_row(p);
  w.bufS = w.bufX + (size_t)B * (((size_t)p->Nc + 8) & ~(size_t)7);
  return BABE_OK;
}

// complex FFT of B rows of Nc points: in -> tmp (pass 1) -> out (pass 2)
static int big_fft(const babe_cqt_plan* p, const float2* in, float2* tmp, float2* out, int B,
                   int conj_out, cudaStream_t st) {
  PassArgs a{};
  a.Nc = p->Nc; a.N1 = p->f1.n; a.N2 = p->f2.n;
  a.div_n2 = make_fastdiv(a.N2);
  a.tw_nc = reinterpret_cast<const float2*>(p->tw_nc);
  a.in = in; a.out = tmp; a.f = to_dev(p->f1); a.roots = reinterpret_cast<const float2*>(p->roots1);
  a.conj_out = 0;
  const size_t smem1 = sizeof(float2) * ((size_t)2 * TILE_SEQ * odd_stride(a.N1) + a.N1 + TW_LO + (a.Nc >> 10) + 1);
  cudaFuncSetAttribute(k_fft_cols, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1);
  k_fft_cols<<<dim3((a.N2 + TILE_SEQ - 1) / TILE_SEQ, B), CQT_THREADS, smem1, st>>>(a);
  int rc = check_launch("k_fft_cols");
  if (rc) return rc;
  a.in = tmp; a.out = out; a.f = to_dev(p->f2); a.roots = reinterpret_cast<const float2*>(p->roots2);
  a.conj_out = conj_out;
  const size_t smem2 = sizeof(float2) * ((size_t)2 * TILE_SEQ * odd_stride(a.N2) + a.N2);
  cudaFuncSetAttribute(k_fft_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
  k_fft_rows<<<dim3((a.N1 + TILE_SEQ - 1) / TILE_SEQ, B), CQT_THREADS, smem2, st>>>(a);
  return check_launch("k_fft_rows");
}


// 2 (default): prime-factor passes (cqt_pfa.cuh) for the instantiated lengths, round-1 passes otherwise;
// -1: round-1 passes for every length.
static int g_cqt_variant = 2;

// ---- programmatic dependent launch of the kernels of a CQT chain (device side: cqt_pfa.cuh) -------------------------
static int g_cqt_pdl = 15;     // bit mask, A/B: babe_set_cqt_pdl (1: pass-1 kernels, 2: pass-2 kernels, 4: band kernels,
                               // 8: the gathering inverse pass 2 behind the synthesis band kernel)
template <int KIND, class... KArgs, class... Args>
static void launch_chain(void (*kern)(KArgs...), dim3 grid, int block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = (g_cqt_pdl & KIND) ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---- third-generation length-Ls transform: prime-factor passes (cqt_pfa.cuh) -----------------------------------
using Pfa92092 = pfa::Plan<4, 7, 11, 13, 23, 1>;      // Ls = 184184: 22.05 kHz x 8.35 s (BASELINE configs[1])
using Pfa184184 = pfa::Plan<8, 7, 11, 13, 23, 1>;     // Ls = 368368: 44.1 kHz x 8.35 s (conf/exp/maestro44k_8s.yaml)
using Pfa66150 = pfa::Plan<27, 25, 1, 49, 2, 1>;      // Ls = 132300: 22.05 kHz x 6 s (BASELINE configs[0]); prime powers as digits
using Pfa242550 = pfa::Plan<25, 9, 2, 49, 11, 1>;     // Ls = 485100: 44.1 kHz x 11 s (conf/exp/maestro44k_8s.yaml)

static int pfa_id(const babe_cqt_plan* p) {
  if (g_cqt_variant != 2) return 0;
  if (p->Nc == Pfa92092::NC) return 1;
  if (p->Nc == Pfa184184::NC) return 2;
  if (p->Nc == Pfa66150::NC) return 3;
  if (p->Nc == Pfa242550::NC) return 4;
  return 0;
}

// PFA_S: residues / rows per tile (16: 128-byte runs; 8 for small batches: twice the CTAs, half the latency each)
template <class PL, int PFA_S>
struct PfaRun {
  using P1 = pfa::Pass1<PL, PFA_S>;
  using P2 = pfa::Pass2<PL, PFA_S>;
  static int pass1_fwd(const float2* x, float2* Y, int B, cudaStream_t st) {
    cudaFuncSetAttribute(pfa::k_pfa1_fwd<PL, PFA_S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P1::SMEM);
    launch_chain<1>(pfa::k_pfa1_fwd<PL, PFA_S>, dim3(P1::TILES, B), pfa::THREADS, P1::SMEM, st, x, Y);
    return check_launch("k_pfa1_fwd");
  }
  static int pass1_inv(const float2* Y, float2* x, int B, cudaStream_t st) {
    cudaFuncSetAttribute(pfa::k_pfa1_inv<PL, PFA_S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P1::SMEM);
    launch_chain<1>(pfa::k_pfa1_inv<PL, PFA_S>, dim3(P1::TILES, B), pfa::THREADS, P1::SMEM, st, Y, x);
    return check_launch("k_pfa1_inv");
  }
  static pfa::P2Args args(const babe_cqt_plan* p, const float* scale) {
    pfa::P2Args a{};
    a.tw_ls = reinterpret_cast<const float2*>(p->tw_ls);
    a.scale = scale;
    a.xpitch = PL::NC + 1;
    return a;
  }
  // x[B, Ls] -> X[B, Nc + 1] * scale
  static int rfft(const babe_cqt_plan* p, const float2* x, float2* tmp, float2* X, const float* scale, int B,
                  int xpitch, cudaStream_t st) {
    int rc = pass1_fwd(x, tmp, B, st);
    if (rc) return rc;
    pfa::P2Args a = args(p, scale);
    a.Y = tmp; a.Xout = X; a.xpitch = xpitch;
    cudaFuncSetAttribute(pfa::k_pfa2_fwd<PL, PFA_S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2::SMEM);
    launch_chain<2>(pfa::k_pfa2_fwd<PL, PFA_S>, dim3(P2::TILES, B), pfa::THREADS, P2::SMEM, st, a);
    return check_launch("k_pfa2_fwd");
  }
  // X[B, Nc + 1] * scale (or the gathered band spectra) -> x[B, Ls]
  static int irfft(const babe_cqt_plan* p, const float2* X, const float2* BS, float2* tmp, float2* x,
                   const float* scale, int B, cudaStream_t st) {
    pfa::P2Args a = args(p, scale);
    a.X = X; a.Yout = tmp;
    if (BS != nullptr) {
      a.BS = BS; a.src = reinterpret_cast<const int4*>(p->bin_src); a.sum_lg = bs_pitch(p);
      cudaFuncSetAttribute(pfa::k_pfa2_inv<PL, PFA_S, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2::SMEM);
      // its own mask bit: started at the BEGINNING of the band kernel (128 registers, one wave) it measured slower
      // (synthesis 0.155 -> 0.178 ms at B = 64); the band kernels therefore trigger their successor when a CTA is done
      launch_chain<8>(pfa::k_pfa2_inv<PL, PFA_S, true>, dim3(P2::TILES, B), pfa::THREADS, P2::SMEM, st, a);
    } else {
      cudaFuncSetAttribute(pfa::k_pfa2_inv<PL, PFA_S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2::SMEM);
      launch_chain<2>(pfa::k_pfa2_inv<PL, PFA_S, false>, dim3(P2::TILES, B), pfa::THREADS, P2::SMEM, st, a);
    }
    int rc = check_launch("k_pfa2_inv");
    if (rc) return rc;
    return pass1_inv(tmp, x, B, st);
  }
  // y = irfft(rfft(x) H): three launches, the spectrum never leaves shared memory
  static int filter(const babe_cqt_plan* p, const float2* x, float2* tmpA, float2* tmpB, float2* y, const float* H,
                    int B, cudaStream_t st) {
    int rc = pass1_fwd(x, tmpA, B, st);
    if (rc) return rc;
    pfa::P2Args a = args(p, H);
    a.Y = tmpA; a.Yout = tmpB;
    cudaFuncSetAttribute(pfa::k_pfa2_mid<PL, PFA_S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2::SMEM);
    launch_chain<2>(pfa::k_pfa2_mid<PL, PFA_S>, dim3(P2::TILES, B), pfa::THREADS, P2::SMEM, st, a);
    rc = check_launch("k_pfa2_mid");
    if (rc) return rc;
    return pass1_inv(tmpB, y, B, st);
  }
};

// 8-column tiles while 16-column tiles would give fewer than ~2 waves of CTAs (B <= ~60 rows at Ls = 184184;
// measured: apply_hpf_DC 0.046 -> 0.038 ms at B = 16, 0.063 -> 0.060 ms at B = 32; a wash at B = 64)
#define BABE_PFA_DISPATCH_PLAN(PL, call)                                                          \
  do {                                                                                            \
    const bool small = (long long)B * ((PL::N2 + 15) / 16) < 8LL * sm_count();                    \
    return small ? PfaRun<PL, 8>::call : PfaRun<PL, 16>::call;                                    \
  } while (0)
#define BABE_PFA_DISPATCH(call)                                                                   \
  do {                                                                                            \
    switch (pfa_id(p)) {                                                                          \
      case 1: BABE_PFA_DISPATCH_PLAN(Pfa92092, call);                                             \
      case 2: BABE_PFA_DISPATCH_PLAN(Pfa184184, call);                                            \
      case 3: BABE_PFA_DISPATCH_PLAN(Pfa66150, call);                                             \
      default: BABE_PFA_DISPATCH_PLAN(Pfa242550, call);                                           \
    }                                                                                             \
  } while (0)
static int pfa_rfft(const babe_cqt_plan* p, const float2* x, float2* tmp, float2* X, const float* scale, int B,
                    int xpitch, cudaStream_t st) {
  BABE_PFA_DISPATCH(rfft(p, x, tmp, X, scale, B, xpitch, st));
}
static int pfa_irfft(const babe_cqt_plan* p, const float2* X, const float2* BS, float2* tmp, float2* x,
                     const float* scale, int B, cudaStream_t st) {
  BABE_PFA_DISPATCH(irfft(p, X, BS, tmp, x, scale, B, st));
}
static int pfa_filter(const babe_cqt_plan* p, const float2* x, float2* tmpA, float2* tmpB, float2* y,
                      const float* H, int B, cudaStream_t st) {
  BABE_PFA_DISPATCH(filter(p, x, tmpA, tmpB, y, H, B, st));
}
#undef BABE_PFA_DISPATCH
#undef BABE_PFA_DISPATCH_PLAN

// Staging of the analysis band kernel: 1 (default) window slices by TMA bulk copies where the spectrum allows it;
// 2: cp.async.  The synthesis always stages by cp.async.
static int g_band_variant = 1;
static inline int band_r3(int M) {     // M = 256 * R3 handled by BandCoreV<R3>, else 0
  switch (M) { case 256: return 1; case 512: return 2; case 1024: return 4; case 2048: return 8;
               case 4096: return 16; default: return 0; }
}

static int fill_band_args(const babe_cqt_plan* p, BandArgs& a, size_t& smem, int& items, int B) {
  a.Nc = p->Nc; a.numocts = p->numocts; a.binsoct = p->binsoct; a.sum_lg = bs_pitch(p);
  a.band_p = p->band_p; a.band_lg = p->band_lg; a.band_off = p->band_off;
  smem = 0;
  items = 0;
  for (int o = 0; o < p->numocts; ++o) {
    const int M = p->M[o];
    const int r3 = band_r3(M);
    int tb;
    size_t need;
    if (M == 32 || M == 64 || M == 128) {      // BandCoreS<R2>: R2 threads per band
      const int r2 = M / 16;
      tb = BAND_THREADS / r2;
      need = sizeof(float2) * ((size_t)((tb * (16 * (r2 + 1) + r2) + 1) & ~1) + 2 + 16 * BAND_THREADS + 2 * tb) +
             sizeof(float) * 16 * BAND_THREADS + 64 + 8 * tb;   // + TMA: slice pads, mbarriers, slice descriptors
    } else if (r3) {                           // register FFT: 4096 points per CTA
      tb = 16 / r3;
      need = sizeof(float2) * ((size_t)tb * 16 * (16 * r3 + 1) + 16 * r3 + 16 * BAND_THREADS + 2 * tb) +
             sizeof(float) * 16 * BAND_THREADS + 64 + 8 * tb;   // ex + twiddles + stage + window samples (+ TMA extras)
    } else {                                   // shared-memory Stockham: <= 2048 points per CTA
      tb = std::max(1, std::min(std::min(p->binsoct, MAX_TB), 2048 / M));
      need = sizeof(float2) * ((size_t)2 * tb * odd_stride(M) + M);
    }
    a.M[o] = M; a.tb[o] = tb; a.tile0[o] = items;
    a.fm[o] = to_dev(p->fm[o]);
    a.rootsm[o] = reinterpret_cast<const float2*>(p->rootsm[o]);
    items += (p->binsoct + tb - 1) / tb;
    smem = std::max(smem, need);
  }
  a.tile0[p->numocts] = items;
  // rows per CTA: as many as still fill one wave of 2 CTAs per SM -- the per-CTA preamble (twiddles, window samples,
  // band descriptors: ~490 instructions per thread against ~670 per row) is amortised, and there is no partial
  // second wave (measured at B = 64: 1 / 4 / 16 rows per CTA -> 0.181 / 0.142 / 0.136 ms; B = 8: 1 / 2 / 4 ->
  // 0.047 / 0.043 / 0.044 ms, profiles/r02_cqt.md)
  int rpc = 1;
  while (rpc < 16 && (long long)items * ((B + 2 * rpc - 1) / (2 * rpc)) >= (long long)(1.7 * sm_count())) rpc *= 2;
  a.B = B; a.rows_per_cta = rpc; a.band_variant = g_band_variant;
  return BABE_OK;
}

}  // namespace babe

using namespace babe;

extern "C" size_t babe_cqt_workspace(const babe_cqt_plan* plan, int B) {
  if (plan == nullptr || B < 1) return 0;
  return ws_bytes(plan, B);
}

extern "C" int babe_rfft(const babe_cqt_plan* plan, const float* x, float* X, int B,
                         const float* bin_scale, void* workspace, size_t workspace_bytes,
                         void* stream) {
  int rc = validate_plan(plan, false);
  if (rc) return rc;
  BABE_REQUIRE(x && X && B >= 1, BABE_EBADARG, "rfft: bad arguments");
  Workspace w;
  rc = carve(plan, B, workspace, workspace_bytes, w);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (pfa_id(plan))
    return pfa_rfft(plan, reinterpret_cast<const float2*>(x), w.bufA, reinterpret_cast<float2*>(X), bin_scale, B,
                    plan->Nc + 1, st);
  rc = big_fft(plan, reinterpret_cast<const float2*>(x), w.bufA, w.bufB, B, 0, st);
  if (rc) return rc;
  const int n = plan->Nc / 2 + 1;
  k_rfft_post<<<dim3((n + 255) / 256, B), 256, 0, st>>>(w.bufB, reinterpret_cast<float2*>(X), plan->Nc,
                                                        reinterpret_cast<const float2*>(plan->tw_ls),
                                                        bin_scale);
  return check_launch("k_rfft_post");
}

extern "C" int babe_irfft(const babe_cqt_plan* plan, const float* X, float* x, int B,
                          const float* bin_scale, void* workspace, size_t workspace_bytes,
                          void* stream) {
  int rc = validate_plan(plan, false);
  if (rc) return rc;
  BABE_REQUIRE(x && X && B >= 1, BABE_EBADARG, "irfft: bad arguments");
  Workspace w;
  rc = carve(plan, B, workspace, workspace_bytes, w);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (pfa_id(plan))
    return pfa_irfft(plan, reinterpret_cast<const float2*>(X), nullptr, w.bufA, reinterpret_cast<float2*>(x),
                     bin_scale, B, st);
  const int n = plan->Nc / 2 + 1;
  k_irfft_pre<<<dim3((n + 255) / 256, B), 256, 0, st>>>(reinterpret_cast<const float2*>(X), w.bufA,
                                                        plan->Nc,
                                                        reinterpret_cast<const float2*>(plan->tw_ls),
                                                        bin_scale);
  rc = check_launch("k_irfft_pre");
  if (rc) return rc;
  return big_fft(plan, w.bufA, w.bufB, reinterpret_cast<float2*>(x), B, 1, st);
}

extern "C" int babe_spectral_filter(const babe_cqt_plan* plan, const float* x, float* y, int B,
                                    const float* H, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  int rc = validate_plan(plan, false);
  if (rc) return rc;
  BABE_REQUIRE(x && y && H && B >= 1, BABE_EBADARG, "spectral_filter: bad arguments");
  Workspace w;
  rc = carve(plan, B, workspace, workspace_bytes, w);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (pfa_id(plan))
    return pfa_filter(plan, reinterpret_cast<const float2*>(x), w.bufA, w.bufB, reinterpret_cast<float2*>(y), H, B, st);
  rc = big_fft(plan, reinterpret_cast<const float2*>(x), w.bufA, w.bufB, B, 0, st);
  if (rc) return rc;
  const int n = plan->Nc / 2 + 1;
  k_spectral_mid<<<dim3((n + 255) / 256, B), 256, 0, st>>>(w.bufB, w.bufA, plan->Nc,
                                                           reinterpret_cast<const float2*>(plan->tw_ls), H);
  rc = check_launch("k_spectral_mid");
  if (rc) return rc;
  return big_fft(plan, w.bufA, w.bufB, reinterpret_cast<float2*>(y), B, 1, st);
}

extern "C" int babe_cqt_analysis(const babe_cqt_plan* plan, const float* x,
                                 float* const* out_octaves_host, int planar, int B,
                                 const float* win, const float* bin_scale, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  int rc = validate_plan(plan, true);
  if (rc) return rc;
  BABE_REQUIRE(x && out_octaves_host && win && B >= 1, BABE_EBADARG, "cqt_analysis: bad arguments");
  Workspace w;
  rc = carve(plan, B, workspace, workspace_bytes, w);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int xpitch = plan->Nc + 1;
  if (pfa_id(plan)) {
    xpitch = plan->Nc + 2;       // even: rows of the internal spectrum are 16-byte aligned (bulk-copied slices)
    rc = pfa_rfft(plan, reinterpret_cast<const float2*>(x), w.bufA, w.bufX, nullptr, B, xpitch, st);
    if (rc) return rc;
  } else {
    rc = big_fft(plan, reinterpret_cast<const float2*>(x), w.bufA, w.bufB, B, 0, st);
    if (rc) return rc;
    const int n = plan->Nc / 2 + 1;
    k_rfft_post<<<dim3((n + 255) / 256, B), 256, 0, st>>>(w.bufB, w.bufX, plan->Nc,
                                                          reinterpret_cast<const float2*>(plan->tw_ls),
                                                          nullptr);
    rc = check_launch("k_rfft_post");
    if (rc) return rc;
  }
  BandArgs a{};
  size_t smem;
  int items;
  fill_band_args(plan, a, smem, items, B);
  for (int o = 0; o < plan->numocts; ++o) {
    BABE_REQUIRE(out_octaves_host[o] != nullptr, BABE_EBADARG, "cqt_analysis: null octave %d", o);
    a.coef[o] = reinterpret_cast<float2*>(out_octaves_host[o]);
  }
  a.win = win; a.scale = bin_scale; a.X = w.bufX; a.planar = planar ? 1 : 0; a.xpitch = xpitch;
  const dim3 grid(items, (B + a.rows_per_cta - 1) / a.rows_per_cta);
  // bulk-copied window slices need 16-byte aligned rows of X: the internal spectrum buffer of the prime-factor path
  const bool tma_ok = a.band_variant == 1 && (a.xpitch % 2 == 0) && (reinterpret_cast<uintptr_t>(a.X) % 16 == 0);
  if (tma_ok) {
    cudaFuncSetAttribute(k_cqt_analysis<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    launch_chain<4>(k_cqt_analysis<true>, grid, BAND_THREADS, smem, st, a);
  } else {
    cudaFuncSetAttribute(k_cqt_analysis<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    launch_chain<4>(k_cqt_analysis<false>, grid, BAND_THREADS, smem, st, a);
  }
  return check_launch("k_cqt_analysis");
}

extern "C" int babe_cqt_synthesis(const babe_cqt_plan* plan, const float* const* in_octaves_host,
                                  int planar, float* x, int B, const float* win,
                                  const float* bin_scale, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  int rc = validate_plan(plan, true);
  if (rc) return rc;
  BABE_REQUIRE(x && in_octaves_host && win && B >= 1, BABE_EBADARG, "cqt_synthesis: bad arguments");
  Workspace w;
  rc = carve(plan, B, workspace, workspace_bytes, w);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BandArgs a{};
  size_t smem;
  int items;
  fill_band_args(plan, a, smem, items, B);
  for (int o = 0; o < plan->numocts; ++o) {
    BABE_REQUIRE(in_octaves_host[o] != nullptr, BABE_EBADARG, "cqt_synthesis: null octave %d", o);
    a.coef[o] = const_cast<float2*>(reinterpret_cast<const float2*>(in_octaves_host[o]));
  }
  a.win = win; a.scale = nullptr; a.BS = w.bufS; a.planar = planar ? 1 : 0;
  const dim3 grid(items, (B + a.rows_per_cta - 1) / a.rows_per_cta);
  // coefficient rows staged by cp.async: bulk copies measured 68.3 vs 69.8 us at B = 64 but 18.2 vs 16.2 us at B = 8
  // and 20.2 vs 17.1 us for the planar layout the sampler uses (two copies per band) -- profiles/r02_cqt.md
  cudaFuncSetAttribute(k_cqt_synth_bands, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  launch_chain<4>(k_cqt_synth_bands, grid, BAND_THREADS, smem, st, a);
  rc = check_launch("k_cqt_synth_bands");
  if (rc) return rc;
  if (pfa_id(plan) && plan->bin_src != nullptr)   // table-driven overlap-add gather in the prologue of the inverse pass 2
    return pfa_irfft(plan, nullptr, w.bufS, w.bufA, reinterpret_cast<float2*>(x), bin_scale, B, st);
  GatherArgs g{};
  g.BS = w.bufS; g.Zc = w.bufA; g.Nc = plan->Nc; g.sum_lg = bs_pitch(plan);
  g.band_p = plan->band_p; g.band_lg = plan->band_lg; g.band_off = plan->band_off;
  g.jlo = plan->bin_jlo; g.jhi = plan->bin_jhi; g.scale = bin_scale;
  g.tw_ls = reinterpret_cast<const float2*>(plan->tw_ls);
  const int n = plan->Nc / 2 + 1;
  k_cqt_gather_pre<<<dim3((n + 255) / 256, B), 256, 0, st>>>(g);
  rc = check_launch("k_cqt_gather_pre");
  if (rc) return rc;
  return big_fft(plan, w.bufA, w.bufB, reinterpret_cast<float2*>(x), B, 1, st);
}

// profiling / A-B knob (profiles/probe_r02.py): which implementation computes the length-Ls transform
extern "C" int babe_set_cqt_variant(int v) {
  if (v != 2 && v != -1) return BABE_EBADARG;
  babe::g_cqt_variant = v;
  return BABE_OK;
}
extern "C" int babe_get_cqt_variant(void) { return babe::g_cqt_variant; }
extern "C" int babe_set_cqt_pdl(int on) {
  babe::g_cqt_pdl = on;
  return BABE_OK;
}
extern "C" int babe_set_cqt_band_variant(int v) {
  if (v != 1 && v != 2) return BABE_EBADARG;
  babe::g_band_variant = v;
  return BABE_OK;
}
