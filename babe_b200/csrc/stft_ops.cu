// STFT-domain operator kernels for sm_100a.
//
// All kernels share one transform core: a length-N complex FFT computed by a
// "frame group" of threads in two or three in-register passes with
// shared-memory transpositions in between.  Two real frames are carried through
// each complex transform (frame A in the real part, frame B in the imaginary
// part).  Because the lowpass response H is real and symmetric the packed
// spectrum can be multiplied by H directly and inverted without ever
// separating the two frames, so the fused STFT -> H -> iSTFT operator costs one
// forward and one inverse complex FFT per PAIR of frames; window, overlap-add
// and envelope division happen in registers, x is read and y written once.
//
//   Core3 (N = 4096 = 16*16*16): 256 threads per frame pair, 16 points per
//     thread, three radix-16 passes.  ~100 registers/thread -> two 256-thread
//     CTAs per SM (16 warps) and a code footprint that fits the instruction
//     cache.  (Round-1 profile of the earlier 64x64 two-pass core: 255
//     registers, 8 warps/SM, long-scoreboard + no-instruction stalls, 4 % of HBM
//     peak -- profiles/r01_apply_filter_64x64.md.)
//   Core2<R1,R2> (N = R1*R2, R in {16,32,64}): two passes, max(R1,R2) threads
//     per frame pair; used for NFFT 512/1024/2048.
//
// Reference semantics: utils/blind_bwe_utils.py:6-39 of eloimoliner/BABE
// (periodic Hamming window, hop N/2, right zero padding by N, center=False,
// torch.istft envelope normalisation).
#include <math.h>

#include <algorithm>

#include "common.cuh"
#include "filter_design.cuh"
#include "regfft.cuh"
#include "regfft_packed.cuh"
#include "stft_cores.cuh"
#include "stft_fused.cuh"

namespace babe {

// overlap-add envelope at block `blk`, offset r (< HOP) given w^2 of both halves
__device__ __forceinline__ float ola_env(int blk, int frames, float w2lo, float w2hi) {
  float e = 0.f;
  if (blk >= 1 && blk - 1 < frames) e = w2hi;
  if (blk < frames) e = __fadd_rn(e, w2lo);
  return e;
}

// ---------------------------------------------------------------------------
// shared-memory carve-up common to the kernels
// ---------------------------------------------------------------------------
template <class G>
struct Smem {
  float2* tw;    // TW_SMEM
  float* win;    // N
  float* hs;     // F   (H/N, or bin scale)
  float2* ex;    // groups * EX_ELEMS
  __device__ Smem(unsigned char* base, int groups) {
    tw = reinterpret_cast<float2*>(base);
    ex = tw + G::TW_SMEM;
    win = reinterpret_cast<float*>(ex + groups * G::EX_ELEMS);
    hs = win + G::N;
  }
  static size_t bytes(int groups, int extra_floats_per_group = 0) {
    return sizeof(float2) * (G::TW_SMEM + (size_t)groups * G::EX_ELEMS) +
           sizeof(float) * (G::N + G::F + 3 + (size_t)groups * extra_floats_per_group);
  }
};

template <class G>
__device__ __forceinline__ void load_tables(Smem<G>& sm, const float* window, const float2* twiddle) {
  for (int i = threadIdx.x; i < G::N; i += blockDim.x) sm.win[i] = window[i];
  G::load_twiddles(sm.tw, twiddle);
}

// ---------------------------------------------------------------------------
// asynchronous global -> shared staging of one frame pair's input (3 half-frames)
// ---------------------------------------------------------------------------
__device__ __forceinline__ void cp_async4(float* dst, const float* src, int src_bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async16(float* dst, const float* src, int src_bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}
// samples [fA*HOP, fA*HOP + 3*HOP) of the row, zero-filled beyond T
template <class G>
__device__ __forceinline__ void stage_pair(float* stage, const float* xr, int T, int fA, int t, bool vec16) {
  const long long base = (long long)fA * G::HOP;
  if (vec16) {
#pragma unroll 2
    for (int c = t; c < 3 * G::HOP / 4; c += G::TPF) {
      const long long p = base + 4 * c;
      const bool in = p < T;                              // T % 4 == 0: chunk entirely in or out
      cp_async16(stage + 4 * c, xr + (in ? p : 0), in ? 16 : 0);
    }
  } else {
#pragma unroll 4
    for (int c = t; c < 3 * G::HOP; c += G::TPF) {
      const long long p = base + c;
      const bool in = p < T;
      cp_async4(stage + c, xr + (in ? p : 0), in ? 4 : 0);
    }
  }
}

// samples [f*HOP, f*HOP + N) of the row (one frame), zero-filled beyond T
template <class G>
__device__ __forceinline__ void stage_frame(float* stage, const float* xr, int T, int f, int t, bool vec16) {
  const long long base = (long long)f * G::HOP;
  if (vec16) {
#pragma unroll 2
    for (int c = t; c < G::N / 4; c += G::TPF) {
      const long long p = base + 4 * c;
      const bool in = p < T;
      cp_async16(stage + 4 * c, xr + (in ? p : 0), in ? 16 : 0);
    }
  } else {
#pragma unroll 4
    for (int c = t; c < G::N; c += G::TPF) {
      const long long p = base + c;
      const bool in = p < T;
      cp_async4(stage + c, xr + (in ? p : 0), in ? 4 : 0);
    }
  }
}

// ---------------------------------------------------------------------------
// K1: fused STFT -> H -> iSTFT  (forward and adjoint)
// ---------------------------------------------------------------------------
struct FilterArgs {
  const float* x; float* y; int B, T;
  const float* window; const float2* twiddle;
  const float* H; const float* freqs; const float* fc; const float* A; int K;
  int adjoint;
  const float* sub; const float* row_scale; double* row_sumsq; double* item_sumsq;
  int* status;
  int bpi;            // output blocks per work item
  int items_per_row;  // ceil(nblk / bpi)
  int nblk;           // output blocks that contain samples < T
  int frames;         // 1 + T / HOP
};

template <class G, int GROUPS>
__global__ void __launch_bounds__(G::TPF* GROUPS, G::MIN_CTAS) k_apply_filter(const FilterArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem<G> sm(smem_raw, GROUPS);
  __shared__ FilterSegs segs;
  __shared__ double warp_part[GROUPS][G::TPF / 32];

  load_tables(sm, a.window, a.twiddle);
  constexpr float inv_n = 1.0f / G::N;
  if (a.H != nullptr) {
    for (int k = threadIdx.x; k < G::F; k += blockDim.x) sm.hs[k] = a.H[k] * inv_n;
  } else {
    __shared__ float fkf[BABE_MAX_BREAKPOINTS];
    // bin frequencies into shared memory first (the staging area is still free): the K binary
    // searches then cost ~12 shared-memory reads instead of ~12 dependent global loads each
    float* fs = sm.hs + ((G::F + 3) & ~3);
    for (int k = threadIdx.x; k < G::F; k += blockDim.x) fs[k] = a.freqs[k];
    __syncthreads();
    build_segments_coop(segs, fkf, a.fc, a.A, a.K, fs, G::F);
    if (threadIdx.x == 0 && segs.bad && a.status != nullptr && blockIdx.x == 0) *a.status = 1;
    for (int k = threadIdx.x; k < G::F; k += blockDim.x)
      sm.hs[k] = bin_gain(segs, k, fs[k]) * inv_n;
  }
  __syncthreads();

  const int grp = threadIdx.x / G::TPF;
  const int t = threadIdx.x % G::TPF;
  const int bar = 1 + grp;
  float2* ex = sm.ex + grp * G::EX_ELEMS;
  float* stage = sm.hs + ((G::F + 3) & ~3) + (size_t)grp * 3 * G::HOP;   // 16-byte aligned
  // reciprocal overlap-add envelope of interior blocks (two frames overlap), shared by the groups
  float* ienv = sm.hs + ((G::F + 3) & ~3) + (size_t)GROUPS * 3 * G::HOP;
  for (int r = threadIdx.x; r < G::HOP; r += blockDim.x) {
    const float wl = sm.win[r], wh = sm.win[r + G::HOP];
    ienv[r] = __frcp_rn(__fadd_rn(wh * wh, wl * wl));
  }
  __syncthreads();
  typename G::Regs regs;
  G::init_regs(regs, a.twiddle, t);
  const long long n_items = (long long)a.B * a.items_per_row;
  const bool vec16 = (a.T % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.x) & 15) == 0);

  for (long long item = (long long)blockIdx.x * GROUPS + grp; item < n_items;
       item += (long long)gridDim.x * GROUPS) {
    const int row = (int)(item / a.items_per_row);
    const int j0 = (int)(item % a.items_per_row) * a.bpi;
    const int j1 = min(j0 + a.bpi, a.nblk);
    const int fs = max(j0 - 1, 0);
    const int fe = min(j1 - 1, a.frames - 1);
    const float* xr = a.x + (size_t)row * a.T;
    float* yr = a.y + (size_t)row * a.T;
    const float* subr = a.sub ? a.sub + (size_t)row * a.T : nullptr;
    const float rs = a.row_scale ? a.row_scale[row] : 1.0f;
    float carry[G::NT / 2];
#pragma unroll
    for (int i = 0; i < G::NT / 2; ++i) carry[i] = 0.f;
    double acc = 0.0;

    bool staged = false;
    for (int fA = fs; fA <= fe; fA += 2) {
      float ar[G::NT], ai[G::NT], br[G::NF], bi[G::NF];
      // ---- the pair's 3 half-frames come through the cp.async staging buffer: the
      // copy for pair p+1 is issued while pair p is being transformed
      if (!staged) stage_pair<G>(stage, xr, a.T, fA, t, vec16);
      cp_async_wait_all();
      group_sync<G::TPF>(bar);
      if (t < G::TT) {
        float xs[G::NT + G::NT / 2];
        const long long base = (long long)fA * G::HOP + t;
#pragma unroll
        for (int j = 0; j < G::NT + G::NT / 2; ++j) {
          float v = stage[G::TS * j + t];                    // zero beyond T
          if (a.adjoint) {
            const int blk = fA + j / (G::NT / 2);
            const int r = (j % (G::NT / 2)) * G::TS + t;
            if (blk >= 1 && blk < a.frames) {
              v *= ienv[r];                                    // interior block: 1/(w_lo^2 + w_hi^2)
            } else if (v != 0.f) {                             // edge blocks only; zero stays zero
              const float wl = sm.win[r], wh = sm.win[r + G::HOP];
              v = __fdiv_rn(v, ola_env(blk, a.frames, wl * wl, wh * wh));
            }
          }
          xs[j] = v;
        }
        const bool hasB = (fA + 1) < a.frames;
#pragma unroll
        for (int n1 = 0; n1 < G::NT; ++n1) {
          const float w = sm.win[G::TS * n1 + t];
          ar[n1] = xs[n1] * w;
          ai[n1] = hasB ? xs[n1 + G::NT / 2] * w : 0.f;
        }
      }
      G::fwd(ar, ai, br, bi, ex, sm.tw, regs, t, bar);   // its barriers order the stage reads
      staged = (fA + 2 <= fe);
      if (staged) stage_pair<G>(stage, xr, a.T, fA + 2, t, vec16);
      if (t < G::FT) {
#pragma unroll
        for (int k2 = 0; k2 < G::NF; ++k2) {
          const int k = t + G::KS * k2;
          const float h = sm.hs[k <= G::N / 2 ? k : G::N - k];
          br[k2] *= h; bi[k2] *= h;
        }
      }
      group_sync<G::TPF>(bar);            // every thread has finished reading ex
      G::inv(br, bi, ar, ai, ex, sm.tw, regs, t, bar);
      if (t < G::TT) {
        // ---- window, overlap-add, normalise, store
#pragma unroll
        for (int n1 = 0; n1 < G::NT; ++n1) {
          const float w = sm.win[G::TS * n1 + t];
          ar[n1] *= w; ai[n1] *= w;
        }
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int blk = fA + half;
          const bool mine = (blk >= j0) && (blk < j1);
          if (!mine) continue;
          const long long p0 = (long long)blk * G::HOP;
          float* yb = yr + p0;
          // fast path (group-uniform): interior block entirely inside the row -> no per-sample tests
          const bool fast = (blk >= 1) && (blk < a.frames) && (p0 + G::HOP <= a.T);
          if (fast) {
#pragma unroll
            for (int n1 = 0; n1 < G::NT / 2; ++n1) {
              float v = half == 0 ? __fadd_rn(ar[n1], carry[n1])
                                  : __fadd_rn(ar[n1 + G::NT / 2], ai[n1]);
              const int r = G::TS * n1 + t;
              if (!a.adjoint) {
                v *= ienv[r];
                if (subr) v -= subr[p0 + r];
              }
              v *= rs;
              yb[r] = v;
              if (a.item_sumsq != nullptr) acc += (double)v * (double)v;
            }
          } else {
#pragma unroll
            for (int n1 = 0; n1 < G::NT / 2; ++n1) {
              float v = half == 0 ? __fadd_rn(ar[n1], carry[n1])
                                  : __fadd_rn(ar[n1 + G::NT / 2], ai[n1]);
              const int r = G::TS * n1 + t;
              if (p0 + r < a.T) {
                if (!a.adjoint) {
                  const float wl = sm.win[r], wh = sm.win[r + G::HOP];
                  v = __fdiv_rn(v, ola_env(blk, a.frames, wl * wl, wh * wh));
                  if (subr) v -= subr[p0 + r];
                }
                v *= rs;
                yb[r] = v;
                if (a.item_sumsq != nullptr) acc += (double)v * (double)v;
              }
            }
          }
        }
#pragma unroll
        for (int n1 = 0; n1 < G::NT / 2; ++n1) carry[n1] = ai[n1 + G::NT / 2];
      }
      group_sync<G::TPF>(bar);            // ex free for the next pair
    }
    if (a.item_sumsq != nullptr) {
      // one partial per work item; k_row_sumsq adds them in a fixed order
      acc = warp_sum(acc);
      if (G::TPF == 32) {
        if (t == 0) a.item_sumsq[item] = acc;
      } else {
        if ((t & 31) == 0) warp_part[grp][t >> 5] = acc;
        group_sync<G::TPF>(bar);
        if (t == 0) {
          double s = 0.0;
          for (int w = 0; w < G::TPF / 32; ++w) s += warp_part[grp][w];
          a.item_sumsq[item] = s;
        }
        group_sync<G::TPF>(bar);
      }
    }
  }
}

// ---------------------------------------------------------------------------
// K2: STFT statistics.  z = x*w + i*y*w, one frame per transform.
//   mode 0: a += |X|^2, b += |X||Y|, c += |Y|^2
//   mode 1: a += Re(conj(X) G), y divided by the OLA envelope on load
// Per-group partial sums go to workspace[group][3][F]; k_reduce_stats sums
// them in a fixed order (deterministic).
// ---------------------------------------------------------------------------
struct StatsArgs {
  const float* x; const float* y; int B, T;
  const float* window; const float2* twiddle;
  int mode; int frames; int fpi; int items_per_row;
  float* partial;
};

template <class G, int GROUPS>
__global__ void __launch_bounds__(G::TPF* GROUPS, G::MIN_CTAS) k_stft_stats(const StatsArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem<G> sm(smem_raw, GROUPS);
  float* accbase = sm.hs;                 // no filter table in this kernel: reuse its slot
  load_tables(sm, a.window, a.twiddle);
  const int grp = threadIdx.x / G::TPF;
  const int t = threadIdx.x % G::TPF;
  const int bar = 1 + grp;
  float2* ex = sm.ex + grp * G::EX_ELEMS;
  typename G::Regs regs;
  G::init_regs(regs, a.twiddle, t);
  float* acc = accbase + (size_t)grp * 3 * G::F;
  for (int i = t; i < 3 * G::F; i += G::TPF) acc[i] = 0.f;
  // staging buffers (2 N floats per group) follow the accumulators, 16-byte aligned
  float* stage = accbase + (((size_t)GROUPS * 3 * G::F + 3) & ~(size_t)3) + (size_t)grp * 2 * G::N;
  const bool vec16 = (a.T % 4 == 0) && (((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.y)) & 15) == 0);
  __syncthreads();

  const long long n_items = (long long)a.B * a.items_per_row;
  for (long long item = (long long)blockIdx.x * GROUPS + grp; item < n_items;
       item += (long long)gridDim.x * GROUPS) {
    const int row = (int)(item / a.items_per_row);
    const int f0 = (int)(item % a.items_per_row) * a.fpi;
    const int f1 = min(f0 + a.fpi, a.frames);
    const float* xr = a.x + (size_t)row * a.T;
    const float* yr = a.y + (size_t)row * a.T;
    bool staged = false;
    for (int f = f0; f < f1; ++f) {
      float ar[G::NT], ai[G::NT], br[G::NF], bi[G::NF], pr[G::NF], pi[G::NF];
      // both signals' frame goes through the cp.async staging buffer; the copy of
      // frame f+1 overlaps the transform of frame f
      if (!staged) { stage_frame<G>(stage, xr, a.T, f, t, vec16); stage_frame<G>(stage + G::N, yr, a.T, f, t, vec16); }
      cp_async_wait_all();
      group_sync<G::TPF>(bar);
      if (t < G::TT) {
        const long long base = (long long)f * G::HOP + t;
#pragma unroll
        for (int n1 = 0; n1 < G::NT; ++n1) {
          const long long p = base + (long long)G::TS * n1;
          const float w = sm.win[G::TS * n1 + t];
          const float xv = stage[G::TS * n1 + t];             // zero beyond T
          float yv = stage[G::N + G::TS * n1 + t];
          if (a.mode == 1 && p < a.T) {
            const int blk = f + (n1 >= G::NT / 2 ? 1 : 0);
            const int r = (n1 % (G::NT / 2)) * G::TS + t;
            const float wl = sm.win[r], wh = sm.win[r + G::HOP];
            yv = __fdiv_rn(yv, ola_env(blk, a.frames, wl * wl, wh * wh));
          }
          ar[n1] = xv * w; ai[n1] = yv * w;
        }
      }
      G::fwd(ar, ai, br, bi, ex, sm.tw, regs, t, bar);
      staged = (f + 1 < f1);
      if (staged) { stage_frame<G>(stage, xr, a.T, f + 1, t, vec16); stage_frame<G>(stage + G::N, yr, a.T, f + 1, t, vec16); }
      group_sync<G::TPF>(bar);
      G::mirror(br, bi, pr, pi, ex, t, bar);
      if (t < G::FT) {
#pragma unroll
        for (int k2 = 0; k2 <= G::NF / 2; ++k2) {
          if (k2 == G::NF / 2 && t != 0) continue;
          const int k = t + G::KS * k2;
          const float xre = 0.5f * (br[k2] + pr[k2]), xim = 0.5f * (bi[k2] - pi[k2]);
          const float yre = 0.5f * (bi[k2] + pi[k2]), yim = -0.5f * (br[k2] - pr[k2]);
          if (a.mode == 0) {
            const float sx = xre * xre + xim * xim, sy = yre * yre + yim * yim;
            acc[k] += sx;
            acc[G::F + k] += sqrtf(sx) * sqrtf(sy);
            acc[2 * G::F + k] += sy;
          } else {
            acc[k] += xre * yre + xim * yim;
          }
        }
      }
      group_sync<G::TPF>(bar);
    }
  }
  __syncthreads();
  float* out = a.partial + ((size_t)blockIdx.x * GROUPS + grp) * 3 * G::F;
  for (int i = t; i < 3 * G::F; i += G::TPF) out[i] = acc[i];
}

__global__ void k_row_sumsq(const double* item_sumsq, int items_per_row, double* row_sumsq) {
  // single thread per row: deterministic order, items_per_row is small
  const int row = blockIdx.x;
  double s = 0.0;
  for (int i = 0; i < items_per_row; ++i) s += item_sumsq[(size_t)row * items_per_row + i];
  row_sumsq[row] += s;
}

// 32 outputs x 8 slices per CTA: slice s adds partials p = s, s+8, ... in order, the 8 slice
// sums are combined in a fixed order -> deterministic, 8x the parallelism of one thread per output
__global__ void __launch_bounds__(256) k_reduce_stats(const float* partial, int n_partials, int n, double* out) {
  __shared__ double sl[8][33];
  const int o = threadIdx.x & 31, sidx = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + o;
  double s = 0.0;
  if (i < n)
    for (int p = sidx; p < n_partials; p += 8) s += (double)partial[(size_t)p * n + i];
  sl[sidx][o] = s;
  __syncthreads();
  if (sidx == 0 && i < n) {
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sl[k][o];
    out[i] = t;
  }
}

// ---------------------------------------------------------------------------
// K3: standalone STFT   x[B,T] -> X[B,F,frames,2]   (two frames per transform)
// ---------------------------------------------------------------------------
struct StftArgs {
  const float* x; float* X; int B, T;
  const float* window; const float2* twiddle;
  int in_env_div; const float* bin_scale;
  int frames; int ppi; int items_per_row;   // frame pairs per item
};

template <class G, int GROUPS>
__global__ void __launch_bounds__(G::TPF* GROUPS, G::MIN_CTAS) k_stft(const StftArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem<G> sm(smem_raw, GROUPS);
  load_tables(sm, a.window, a.twiddle);
  for (int k = threadIdx.x; k < G::F; k += blockDim.x) sm.hs[k] = a.bin_scale ? a.bin_scale[k] : 1.0f;
  __syncthreads();
  const int grp = threadIdx.x / G::TPF;
  const int t = threadIdx.x % G::TPF;
  const int bar = 1 + grp;
  float2* ex = sm.ex + grp * G::EX_ELEMS;
  typename G::Regs regs;
  G::init_regs(regs, a.twiddle, t);
  const long long n_items = (long long)a.B * a.items_per_row;
  for (long long item = (long long)blockIdx.x * GROUPS + grp; item < n_items;
       item += (long long)gridDim.x * GROUPS) {
    const int row = (int)(item / a.items_per_row);
    const int p0 = (int)(item % a.items_per_row) * a.ppi;
    const float* xr = a.x + (size_t)row * a.T;
    float2* Xr = reinterpret_cast<float2*>(a.X) + (size_t)row * G::F * a.frames;
    for (int pp = p0; pp < p0 + a.ppi && 2 * pp < a.frames; ++pp) {
      const int fA = 2 * pp;
      const bool hasB = fA + 1 < a.frames;
      float ar[G::NT], ai[G::NT], br[G::NF], bi[G::NF], pr[G::NF], pi[G::NF];
      if (t < G::TT) {
        float xs[G::NT + G::NT / 2];
        const long long base = (long long)fA * G::HOP + t;
#pragma unroll
        for (int j = 0; j < G::NT + G::NT / 2; ++j) {
          const long long p = base + (long long)G::TS * j;
          float v = (p < a.T) ? __ldg(xr + p) : 0.f;
          if (a.in_env_div && p < a.T) {
            const int blk = fA + j / (G::NT / 2);
            const int r = (j % (G::NT / 2)) * G::TS + t;
            const float wl = sm.win[r], wh = sm.win[r + G::HOP];
            v = __fdiv_rn(v, ola_env(blk, a.frames, wl * wl, wh * wh));
          }
          xs[j] = v;
        }
#pragma unroll
        for (int n1 = 0; n1 < G::NT; ++n1) {
          const float w = sm.win[G::TS * n1 + t];
          ar[n1] = xs[n1] * w;
          ai[n1] = hasB ? xs[n1 + G::NT / 2] * w : 0.f;
        }
      }
      G::fwd(ar, ai, br, bi, ex, sm.tw, regs, t, bar);
      group_sync<G::TPF>(bar);
      G::mirror(br, bi, pr, pi, ex, t, bar);
      if (t < G::FT) {
#pragma unroll
        for (int k2 = 0; k2 <= G::NF / 2; ++k2) {
          if (k2 == G::NF / 2 && t != 0) continue;
          const int k = t + G::KS * k2;
          const float s = sm.hs[k];
          // frame A = (Z + conj(Zp))/2, frame B = (Z - conj(Zp))/(2i)
          float2 XA, XB;
          XA.x = 0.5f * (br[k2] + pr[k2]) * s; XA.y = 0.5f * (bi[k2] - pi[k2]) * s;
          XB.x = 0.5f * (bi[k2] + pi[k2]) * s; XB.y = -0.5f * (br[k2] - pr[k2]) * s;
          float2* dst = Xr + (size_t)k * a.frames + fA;
          dst[0] = XA;
          if (hasB) dst[1] = XB;
        }
      }
      group_sync<G::TPF>(bar);
    }
  }
}

// ---------------------------------------------------------------------------
// K4: standalone (filter +) iSTFT   X[B,F,frames,2] -> y[B,out_len]
// ---------------------------------------------------------------------------
struct IstftArgs {
  const float* X; float* y; int B; int frames; int out_len;
  const float* window; const float2* twiddle;
  const float* bin_scale; int out_env_div;
  int bpi; int items_per_row; int nblk;
};

template <class G, int GROUPS>
__global__ void __launch_bounds__(G::TPF* GROUPS, G::MIN_CTAS) k_istft(const IstftArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem<G> sm(smem_raw, GROUPS);
  load_tables(sm, a.window, a.twiddle);
  constexpr float inv_n = 1.0f / G::N;
  for (int k = threadIdx.x; k < G::F; k += blockDim.x)
    sm.hs[k] = (a.bin_scale ? a.bin_scale[k] : 1.0f) * inv_n;
  __syncthreads();
  const int grp = threadIdx.x / G::TPF;
  const int t = threadIdx.x % G::TPF;
  const int bar = 1 + grp;
  float2* ex = sm.ex + grp * G::EX_ELEMS;
  typename G::Regs regs;
  G::init_regs(regs, a.twiddle, t);
  const long long n_items = (long long)a.B * a.items_per_row;
  for (long long item = (long long)blockIdx.x * GROUPS + grp; item < n_items;
       item += (long long)gridDim.x * GROUPS) {
    const int row = (int)(item / a.items_per_row);
    const int j0 = (int)(item % a.items_per_row) * a.bpi;
    const int j1 = min(j0 + a.bpi, a.nblk);
    const int fs = max(j0 - 1, 0);
    const int fe = min(j1 - 1, a.frames - 1);
    const float2* Xr = reinterpret_cast<const float2*>(a.X) + (size_t)row * G::F * a.frames;
    float* yr = a.y + (size_t)row * a.out_len;
    float carry[G::NT / 2];
#pragma unroll
    for (int i = 0; i < G::NT / 2; ++i) carry[i] = 0.f;
    for (int fA = fs; fA <= fe; fA += 2) {
      float ar[G::NT], ai[G::NT], br[G::NF], bi[G::NF];
      const bool hasB = fA + 1 < a.frames;
      if (t < G::FT) {
#pragma unroll
        for (int k2 = 0; k2 < G::NF; ++k2) {
          const int k = t + G::KS * k2;
          const bool mir = k > G::N / 2;
          const int kk = mir ? G::N - k : k;
          const float2* src = Xr + (size_t)kk * a.frames + fA;
          float2 XA = src[0];
          float2 XB = hasB ? src[1] : make_float2(0.f, 0.f);
          if (kk == 0 || kk == G::N / 2) { XA.y = 0.f; XB.y = 0.f; }   // c2r ignores these
          if (mir) { XA.y = -XA.y; XB.y = -XB.y; }
          const float h = sm.hs[kk];
          br[k2] = (XA.x - XB.y) * h;
          bi[k2] = (XA.y + XB.x) * h;
        }
      }
      G::inv(br, bi, ar, ai, ex, sm.tw, regs, t, bar);
      if (t < G::TT) {
#pragma unroll
        for (int n1 = 0; n1 < G::NT; ++n1) {
          const float w = sm.win[G::TS * n1 + t];
          ar[n1] *= w; ai[n1] *= w;
        }
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int blk = fA + half;
          const bool mine = (blk >= j0) && (blk < j1);
#pragma unroll
          for (int n1 = 0; n1 < G::NT / 2; ++n1) {
            float v = half == 0 ? __fadd_rn(ar[n1], carry[n1])
                                : __fadd_rn(ar[n1 + G::NT / 2], ai[n1]);
            const int r = G::TS * n1 + t;
            const long long p = (long long)blk * G::HOP + r;
            if (mine && p < a.out_len) {
              if (a.out_env_div) {
                const float wl = sm.win[r], wh = sm.win[r + G::HOP];
                v = __fdiv_rn(v, ola_env(blk, a.frames, wl * wl, wh * wh));
              }
              yr[p] = v;
            }
          }
        }
#pragma unroll
        for (int n1 = 0; n1 < G::NT / 2; ++n1) carry[n1] = ai[n1 + G::NT / 2];
      }
      group_sync<G::TPF>(bar);
    }
  }
}

// ---------------------------------------------------------------------------
// K5: FIR "same" convolution by overlap-save on the Core3 transform (SURVEY 8f-4:
// the non-blind baseline predict_bwe("firwin"), testing/blind_bwe_sampler.py:211-218,
// utils/bandwidth_extension.py:76-95).  torch conv1d is a correlation:
//   y[n] = sum_k b[k] x[n + k - pl],  pl = (L-1)/2 (left "same" padding).
// A block of V = N - L + 1 outputs needs N inputs; two consecutive blocks ride one
// complex transform (real kernel => the packed spectrum is multiplied by the table G
// without separating them).  G = conj(FFT(b zero padded)) / N is prepared by the
// host once per filter; the adjoint is the same kernel with the reversed taps.
// ---------------------------------------------------------------------------
struct FirArgs {
  const float* x; float* y; int B, T;
  const float2* twiddle; const float2* G;
  int L, pl, V;
  int pairs_per_row;
};

template <class G_>
__global__ void __launch_bounds__(G_::TPF, G_::MIN_CTAS) k_fir_filter(const FirArgs a) {
  using G = G_;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* tw = reinterpret_cast<float2*>(smem_raw);
  float2* ex = tw + G::TW_SMEM;
  G::load_twiddles(tw, a.twiddle);
  const int t = threadIdx.x;
  typename G::Regs regs;
  G::init_regs(regs, a.twiddle, t);
  __syncthreads();
  const long long n_items = (long long)a.B * a.pairs_per_row;
  for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int row = (int)(item / a.pairs_per_row);
    const long long s = (long long)(item % a.pairs_per_row) * 2 * a.V;     // first output of block A
    const float* xr = a.x + (size_t)row * a.T;
    float* yr = a.y + (size_t)row * a.T;
    float ar[G::NT], ai[G::NT], br[G::NF], bi[G::NF];
#pragma unroll
    for (int j = 0; j < G::NT; ++j) {
      const long long pa = s - a.pl + G::TS * j + t, pb = pa + a.V;
      ar[j] = (pa >= 0 && pa < a.T) ? __ldg(xr + pa) : 0.f;
      ai[j] = (pb >= 0 && pb < a.T) ? __ldg(xr + pb) : 0.f;
    }
    G::fwd(ar, ai, br, bi, ex, tw, regs, t, 1);
#pragma unroll
    for (int i = 0; i < G::NF; ++i) {
      const float2 g = a.G[t + G::KS * i];
      const float re = br[i] * g.x - bi[i] * g.y;
      bi[i] = br[i] * g.y + bi[i] * g.x;
      br[i] = re;
    }
    group_sync<G::TPF>(1);
    G::inv(br, bi, ar, ai, ex, tw, regs, t, 1);
#pragma unroll
    for (int j = 0; j < G::NT; ++j) {
      const int n = G::TS * j + t;
      if (n < a.V) {
        const long long pa = s + n, pb = pa + a.V;
        if (pa < a.T) yr[pa] = ar[j];
        if (pb < a.T) yr[pb] = ai[j];
      }
    }
    group_sync<G::TPF>(1);
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
template <class G, int GROUPS>
static constexpr int ctas_per_sm() { return G::MIN_CTAS; }

static int pick_chunk(long long rows, int units_per_row, long long capacity, int max_chunk,
                      bool odd_only) {
  // chunk size (units per work item) minimising (rounds * cost per item)
  int best = 1;
  double best_cost = 1e300;
  for (int c = 1; c <= max_chunk; ++c) {
    if (odd_only && (c % 2 == 0)) continue;
    const long long items = rows * ((units_per_row + c - 1) / c);
    const long long rounds = (items + capacity - 1) / capacity;
    const double per_item = odd_only ? (c + 1) * 0.5 : (double)c;  // frame pairs per item
    const double cost = rounds * per_item * (1.0 + 1e-3 / c);
    if (cost < best_cost) { best_cost = cost; best = c; }
  }
  return best;
}

template <class G, int GROUPS>
static int launch_apply_filter(FilterArgs a, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int hop = G::HOP;
  a.frames = 1 + a.T / hop;
  a.nblk = (a.T - 1) / hop + 1;
  const int sms = sm_count();
  a.bpi = pick_chunk(a.B, a.nblk, (long long)sms * GROUPS * ctas_per_sm<G, GROUPS>(), 31, true);
  a.items_per_row = (a.nblk + a.bpi - 1) / a.bpi;
  const long long items = (long long)a.B * a.items_per_row;
  const int grid = (int)std::min<long long>((items + GROUPS - 1) / GROUPS, (long long)sms * ctas_per_sm<G, GROUPS>());
  const size_t smem = Smem<G>::bytes(GROUPS, 3 * G::HOP) + sizeof(float) * G::HOP + 16;   // + staging per group + 1/env
  a.item_sumsq = nullptr;
  if (a.row_sumsq != nullptr) {
    BABE_REQUIRE(ws != nullptr && ws_bytes >= (size_t)items * sizeof(double), BABE_EBADARG,
                 "apply_filter: row_sumsq needs a workspace of babe_apply_filter_workspace() bytes");
    a.item_sumsq = static_cast<double*>(ws);
  }
  auto kern = k_apply_filter<G, GROUPS>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<grid, G::TPF * GROUPS, smem, st>>>(a);
  int rc = check_launch("k_apply_filter");
  if (rc || a.row_sumsq == nullptr) return rc;
  k_row_sumsq<<<a.B, 1, 0, st>>>(a.item_sumsq, a.items_per_row, a.row_sumsq);
  return check_launch("k_row_sumsq");
}

template <class G, int GROUPS>
static int launch_stats(StatsArgs a, double* abc, void* ws, size_t ws_bytes, cudaStream_t st) {
  a.frames = 1 + a.T / G::HOP;
  const int sms = sm_count();
  a.fpi = pick_chunk(a.B, a.frames, (long long)sms * GROUPS * ctas_per_sm<G, GROUPS>(), 32, false);
  a.items_per_row = (a.frames + a.fpi - 1) / a.fpi;
  const long long items = (long long)a.B * a.items_per_row;
  const int grid = (int)std::min<long long>((items + GROUPS - 1) / GROUPS, (long long)sms * ctas_per_sm<G, GROUPS>());
  const size_t need = (size_t)grid * GROUPS * 3 * G::F * sizeof(float);
  BABE_REQUIRE(ws != nullptr && ws_bytes >= need, BABE_EBADARG,
               "stft_stats: workspace too small (%zu < %zu)", ws_bytes, need);
  a.partial = static_cast<float*>(ws);
  const size_t smem = Smem<G>::bytes(GROUPS, 3 * G::F + 2 * G::N) - sizeof(float) * (G::F + 3) + 32;
  auto kern = k_stft_stats<G, GROUPS>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<grid, G::TPF * GROUPS, smem, st>>>(a);
  int rc = check_launch("k_stft_stats");
  if (rc) return rc;
  const int n = 3 * G::F;
  k_reduce_stats<<<(n + 31) / 32, 256, 0, st>>>(a.partial, grid * GROUPS, n, abc);
  return check_launch("k_reduce_stats");
}

template <class G, int GROUPS>
static int launch_stft(StftArgs a, cudaStream_t st) {
  if (a.frames <= 0) a.frames = 1 + a.T / G::HOP;
  const int pairs = (a.frames + 1) / 2;
  const int sms = sm_count();
  a.ppi = pick_chunk(a.B, pairs, (long long)sms * GROUPS * ctas_per_sm<G, GROUPS>(), 16, false);
  a.items_per_row = (pairs + a.ppi - 1) / a.ppi;
  const long long items = (long long)a.B * a.items_per_row;
  const int grid = (int)std::min<long long>((items + GROUPS - 1) / GROUPS, (long long)sms * ctas_per_sm<G, GROUPS>());
  const size_t smem = Smem<G>::bytes(GROUPS);
  auto kern = k_stft<G, GROUPS>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<grid, G::TPF * GROUPS, smem, st>>>(a);
  return check_launch("k_stft");
}

template <class G, int GROUPS>
static int launch_istft(IstftArgs a, cudaStream_t st) {
  a.nblk = (a.out_len - 1) / G::HOP + 1;
  const int sms = sm_count();
  a.bpi = pick_chunk(a.B, a.nblk, (long long)sms * GROUPS * ctas_per_sm<G, GROUPS>(), 31, true);
  a.items_per_row = (a.nblk + a.bpi - 1) / a.bpi;
  const long long items = (long long)a.B * a.items_per_row;
  const int grid = (int)std::min<long long>((items + GROUPS - 1) / GROUPS, (long long)sms * ctas_per_sm<G, GROUPS>());
  const size_t smem = Smem<G>::bytes(GROUPS);
  auto kern = k_istft<G, GROUPS>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<grid, G::TPF * GROUPS, smem, st>>>(a);
  return check_launch("k_istft");
}

// groups per CTA chosen so that one CTA fills an SM's register file / smem
#define BABE_DISPATCH_NFFT(nfft, CALL)                                   \
  switch (nfft) {                                                        \
    case 4096: { using G = Core3; constexpr int GR = 1; CALL; }          \
    case 2048: { using G = Core2<32, 64>; constexpr int GR = 4; CALL; }    \
    case 1024: { using G = Core2<32, 32>; constexpr int GR = 8; CALL; }    \
    case 512:  { using G = Core2<16, 32>; constexpr int GR = 8; CALL; }    \
    default: break;                                                      \
  }

}  // namespace babe

using namespace babe;

extern "C" int babe_stft_supported(int nfft) {
  return nfft == 512 || nfft == 1024 || nfft == 2048 || nfft == 4096;
}

extern "C" int babe_stft_tables_host(int nfft, float* window_host, float* twiddle_host) {
  BABE_REQUIRE(babe_stft_supported(nfft), BABE_EUNSUPPORTED, "unsupported NFFT %d", nfft);
  BABE_REQUIRE(window_host && twiddle_host, BABE_EBADARG, "null table pointer");
  for (int n = 0; n < nfft; ++n) {
    window_host[n] = (float)(0.54 - 0.46 * cos(2.0 * M_PI * (double)n / (double)nfft));
    const double ang = -2.0 * M_PI * (double)n / (double)nfft;
    twiddle_host[2 * n] = (float)cos(ang);
    twiddle_host[2 * n + 1] = (float)sin(ang);
  }
  return BABE_OK;
}

extern "C" int babe_apply_filter(const float* x, float* y, int B, int T, int nfft,
                                 const float* window, const float* twiddle,
                                 const float* H, const float* freqs, const float* fc,
                                 const float* A, int K, int adjoint, const float* sub,
                                 const float* row_scale, double* row_sumsq, void* workspace,
                                 size_t workspace_bytes, int* status, void* stream) {
  BABE_REQUIRE(x && y && window && twiddle, BABE_EBADARG, "apply_filter: null pointer");
  BABE_REQUIRE(B >= 0 && T >= 0, BABE_EBADARG, "apply_filter: bad shape B=%d T=%d", B, T);
  BABE_REQUIRE(H != nullptr || (freqs && fc && A && K >= 1 && K <= BABE_MAX_BREAKPOINTS),
               BABE_EBADARG, "apply_filter: need H or (freqs, fc, A, 1<=K<=%d)", BABE_MAX_BREAKPOINTS);
  BABE_REQUIRE(babe_stft_supported(nfft), BABE_EUNSUPPORTED, "unsupported NFFT %d", nfft);
  if (B == 0 || T == 0) return BABE_OK;
  FilterArgs a{};
  a.x = x; a.y = y; a.B = B; a.T = T; a.window = window;
  a.twiddle = reinterpret_cast<const float2*>(twiddle);
  a.H = H; a.freqs = freqs; a.fc = fc; a.A = A; a.K = K; a.adjoint = adjoint;
  a.sub = adjoint ? nullptr : sub; a.row_scale = row_scale; a.row_sumsq = row_sumsq;
  a.status = status;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (nfft == 4096 && fused_filter_eligible(x, a.sub, T)) {
    // second-generation kernel: TMA-staged frame tiles, Core4k transform (stft_fused.cu)
    FusedArgs f{};
    f.x = x; f.y = y; f.B = B; f.T = T; f.window = window; f.roots = a.twiddle;
    f.H = H; f.freqs = freqs; f.fc = fc; f.A = A; f.K = K; f.adjoint = adjoint;
    f.sub = a.sub; f.row_scale = row_scale; f.status = status;
    if (row_sumsq != nullptr) {
      BABE_REQUIRE(workspace != nullptr && workspace_bytes >= fused_sumsq_slots(B, T) * sizeof(double), BABE_EBADARG,
                   "apply_filter: row_sumsq needs a workspace of babe_apply_filter_workspace() bytes");
      f.item_sumsq = static_cast<double*>(workspace);
    }
    return launch_filter_fused(f, row_sumsq, st);
  }
  BABE_DISPATCH_NFFT(nfft, return (launch_apply_filter<G, GR>(a, workspace, workspace_bytes, st)));
  return BABE_EUNSUPPORTED;
}

extern "C" size_t babe_apply_filter_workspace(int B, int T, int nfft) {
  if (!babe_stft_supported(nfft) || B < 1 || T < 1) return 0;
  return (size_t)B * ((T - 1) / (nfft / 2) + 2) * sizeof(double);   // >= one partial per (CTA, row) segment
}

extern "C" size_t babe_stft_stats_workspace(int B, int T, int nfft) {
  (void)B; (void)T;
  if (!babe_stft_supported(nfft)) return 0;
  const int sms = sm_count();
  return (size_t)sms * 16 * 3 * (nfft / 2 + 1) * sizeof(float);
}

extern "C" int babe_stft_stats(const float* x, const float* y, int B, int T, int nfft,
                               const float* window, const float* twiddle, int mode,
                               double* abc, void* workspace, size_t workspace_bytes,
                               void* stream) {
  BABE_REQUIRE(x && y && window && twiddle && abc, BABE_EBADARG, "stft_stats: null pointer");
  BABE_REQUIRE(B >= 1 && T >= 1, BABE_EBADARG, "stft_stats: bad shape B=%d T=%d", B, T);
  BABE_REQUIRE(mode == 0 || mode == 1, BABE_EBADARG, "stft_stats: bad mode %d", mode);
  BABE_REQUIRE(babe_stft_supported(nfft), BABE_EUNSUPPORTED, "unsupported NFFT %d", nfft);
  StatsArgs a{};
  a.x = x; a.y = y; a.B = B; a.T = T; a.window = window;
  a.twiddle = reinterpret_cast<const float2*>(twiddle); a.mode = mode;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (nfft == 4096 && fused_stats_eligible(x, y, T, mode)) {
    // second-generation kernel: TMA-staged frames, Core4k transform, register accumulators (stft_fused.cu)
    FusedStatsArgs f{};
    f.x = x; f.y = y; f.B = B; f.T = T; f.window = window; f.roots = a.twiddle;
    const size_t need = (size_t)2 * sm_count() * 3 * Core3::F * sizeof(float);
    BABE_REQUIRE(workspace != nullptr && workspace_bytes >= need, BABE_EBADARG,
                 "stft_stats: workspace too small (%zu < %zu)", workspace_bytes, need);
    f.partial = static_cast<float*>(workspace);
    int n_partials = 0;
    int rc = launch_stats_fused(f, &n_partials, st);
    if (rc) return rc;
    const int n = 3 * Core3::F;
    k_reduce_stats<<<(n + 31) / 32, 256, 0, st>>>(f.partial, n_partials, n, abc);
    return check_launch("k_reduce_stats");
  }
  switch (nfft) {
    case 4096: return launch_stats<Core3, 1>(a, abc, workspace, workspace_bytes, st);
    case 2048: return launch_stats<Core2<32, 64>, 4>(a, abc, workspace, workspace_bytes, st);
    case 1024: return launch_stats<Core2<32, 32>, 8>(a, abc, workspace, workspace_bytes, st);
    case 512: return launch_stats<Core2<16, 32>, 8>(a, abc, workspace, workspace_bytes, st);
  }
  return BABE_EUNSUPPORTED;
}

extern "C" int babe_stft(const float* x, float* X, int B, int T, int nfft, int frames,
                         const float* window, const float* twiddle, int in_env_div,
                         const float* bin_scale, void* stream) {
  BABE_REQUIRE(x && X && window && twiddle, BABE_EBADARG, "stft: null pointer");
  BABE_REQUIRE(B >= 0 && T >= 0, BABE_EBADARG, "stft: bad shape B=%d T=%d", B, T);
  BABE_REQUIRE(babe_stft_supported(nfft), BABE_EUNSUPPORTED, "unsupported NFFT %d", nfft);
  if (B == 0) return BABE_OK;
  StftArgs a{};
  a.x = x; a.X = X; a.B = B; a.T = T; a.window = window;
  a.twiddle = reinterpret_cast<const float2*>(twiddle);
  a.in_env_div = in_env_div; a.bin_scale = bin_scale; a.frames = frames;
  BABE_REQUIRE(frames >= 0 && frames <= 1 + T / (nfft / 2), BABE_EBADARG,
               "stft: frames=%d out of range", frames);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BABE_DISPATCH_NFFT(nfft, return (launch_stft<G, GR>(a, st)));
  return BABE_EUNSUPPORTED;
}

extern "C" int babe_istft(const float* X, float* y, int B, int frames, int nfft, int out_len,
                          const float* window, const float* twiddle, const float* bin_scale,
                          int out_env_div, void* stream) {
  BABE_REQUIRE(X && y && window && twiddle, BABE_EBADARG, "istft: null pointer");
  BABE_REQUIRE(babe_stft_supported(nfft), BABE_EUNSUPPORTED, "unsupported NFFT %d", nfft);
  BABE_REQUIRE(B >= 0 && frames >= 1, BABE_EBADARG, "istft: bad shape B=%d frames=%d", B, frames);
  BABE_REQUIRE(out_len >= 1 && out_len <= nfft + (nfft / 2) * (frames - 1), BABE_EBADARG,
               "istft: out_len %d out of range", out_len);
  if (B == 0) return BABE_OK;
  IstftArgs a{};
  a.X = X; a.y = y; a.B = B; a.frames = frames; a.out_len = out_len; a.window = window;
  a.twiddle = reinterpret_cast<const float2*>(twiddle);
  a.bin_scale = bin_scale; a.out_env_div = out_env_div;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BABE_DISPATCH_NFFT(nfft, return (launch_istft<G, GR>(a, st)));
  return BABE_EUNSUPPORTED;
}

extern "C" int babe_fir_filter(const float* x, float* y, int B, int T, const float* twiddle,
                               const float* G, int L, int pad_left, void* stream) {
  BABE_REQUIRE(x && y && twiddle && G, BABE_EBADARG, "fir_filter: null pointer");
  BABE_REQUIRE(B >= 0 && T >= 0, BABE_EBADARG, "fir_filter: bad shape B=%d T=%d", B, T);
  BABE_REQUIRE(L >= 1 && L <= Core3::N / 2 + 1, BABE_EUNSUPPORTED, "fir_filter: %d taps (max %d)", L,
               Core3::N / 2 + 1);
  BABE_REQUIRE(pad_left >= 0 && pad_left < L, BABE_EBADARG, "fir_filter: pad_left=%d", pad_left);
  if (B == 0 || T == 0) return BABE_OK;
  FirArgs a{};
  a.x = x; a.y = y; a.B = B; a.T = T;
  a.twiddle = reinterpret_cast<const float2*>(twiddle);
  a.G = reinterpret_cast<const float2*>(G);
  a.L = L; a.pl = pad_left; a.V = Core3::N - L + 1;
  const int blocks = (T + a.V - 1) / a.V;
  a.pairs_per_row = (blocks + 1) / 2;
  if (fused_fir_eligible(x, T)) {       // second-generation kernel: TMA-staged windows, Core4k (stft_fused.cu)
    FusedFirArgs f{};
    f.x = x; f.y = y; f.B = B; f.T = T; f.roots = a.twiddle; f.G = a.G;
    f.L = L; f.pl = pad_left; f.V = a.V; f.pairs_per_row = a.pairs_per_row;
    return launch_fir_fused(f, static_cast<cudaStream_t>(stream));
  }
  const long long items = (long long)B * a.pairs_per_row;
  const int grid = (int)std::min<long long>(items, (long long)sm_count() * Core3::MIN_CTAS);
  const size_t smem = sizeof(float2) * (Core3::TW_SMEM + Core3::EX_ELEMS);
  cudaFuncSetAttribute(k_fir_filter<Core3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_fir_filter<Core3><<<grid, Core3::TPF, smem, static_cast<cudaStream_t>(stream)>>>(a);
  return check_launch("k_fir_filter");
}

// ---------------------------------------------------------------------------
// one filter per row.  NFFT = 4096 rows that can be bulk-copied take the per-row instantiations of the fused
// kernels (stft_fused.cu); every other case (NFFT 512 / 1024 / 2048, rows that cannot be bulk-copied,
// babe_set_fused_variant(-1)) runs the shared-filter entry point once per row on pointer offsets, which gives each
// row its B = 1 result by construction.
// ---------------------------------------------------------------------------
extern "C" int babe_apply_filter_rows(const float* x, float* y, int B, int T, int nfft,
                                      const float* window, const float* twiddle,
                                      const float* freqs, const float* fc, const float* A, int K,
                                      int adjoint, const float* sub, const float* row_scale, double* row_sumsq,
                                      void* workspace, size_t workspace_bytes, int* status, void* stream) {
  BABE_REQUIRE(x && y && window && twiddle, BABE_EBADARG, "apply_filter_rows: null pointer");
  BABE_REQUIRE(B >= 0 && T >= 0, BABE_EBADARG, "apply_filter_rows: bad shape B=%d T=%d", B, T);
  BABE_REQUIRE(freqs && fc && A && K >= 1 && K <= BABE_MAX_BREAKPOINTS, BABE_EBADARG,
               "apply_filter_rows: need (freqs, fc, A, 1<=K<=%d)", BABE_MAX_BREAKPOINTS);
  BABE_REQUIRE(babe_stft_supported(nfft), BABE_EUNSUPPORTED, "unsupported NFFT %d", nfft);
  if (B == 0 || T == 0) return BABE_OK;
  const float* sub_ = adjoint ? nullptr : sub;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (nfft == 4096 && fused_filter_eligible(x, sub_, T)) {
    FusedArgs f{};
    f.x = x; f.y = y; f.B = B; f.T = T; f.window = window; f.roots = reinterpret_cast<const float2*>(twiddle);
    f.freqs = freqs; f.fc = fc; f.A = A; f.K = K; f.adjoint = adjoint;
    f.sub = sub_; f.row_scale = row_scale; f.status = status; f.per_row = 1;
    if (row_sumsq != nullptr) {
      BABE_REQUIRE(workspace != nullptr && workspace_bytes >= fused_sumsq_slots(B, T) * sizeof(double), BABE_EBADARG,
                   "apply_filter_rows: row_sumsq needs a workspace of babe_apply_filter_workspace() bytes");
      f.item_sumsq = static_cast<double*>(workspace);
    }
    return launch_filter_fused(f, row_sumsq, st);
  }
  for (int b = 0; b < B; ++b) {
    const size_t o = (size_t)b * T;
    const int rc = babe_apply_filter(x + o, y + o, 1, T, nfft, window, twiddle, nullptr, freqs, fc + (size_t)b * K,
                                     A + (size_t)b * K, K, adjoint, sub_ ? sub_ + o : nullptr,
                                     row_scale ? row_scale + b : nullptr, row_sumsq ? row_sumsq + b : nullptr,
                                     workspace, workspace_bytes, status ? status + b : nullptr, stream);
    if (rc) return rc;
  }
  return BABE_OK;
}

extern "C" size_t babe_stft_stats_rows_workspace(int B, int T, int nfft) {
  if (!babe_stft_supported(nfft) || B < 1 || T < 1) return 0;
  const size_t fallback = babe_stft_stats_workspace(1, T, nfft);
  if (nfft != 4096) return fallback;
  return std::max(fallback, fused_stats_rows_slots(B, T) * 3 * Core3::F * sizeof(float));
}

extern "C" int babe_stft_stats_rows(const float* x, const float* y, int B, int T, int nfft,
                                    const float* window, const float* twiddle,
                                    double* abc, void* workspace, size_t workspace_bytes, void* stream) {
  BABE_REQUIRE(x && y && window && twiddle && abc, BABE_EBADARG, "stft_stats_rows: null pointer");
  BABE_REQUIRE(B >= 1 && T >= 1, BABE_EBADARG, "stft_stats_rows: bad shape B=%d T=%d", B, T);
  BABE_REQUIRE(babe_stft_supported(nfft), BABE_EUNSUPPORTED, "unsupported NFFT %d", nfft);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (nfft == 4096 && fused_stats_eligible(x, y, T, 0)) {
    const size_t need = fused_stats_rows_slots(B, T) * 3 * Core3::F * sizeof(float);
    BABE_REQUIRE(workspace != nullptr && workspace_bytes >= need, BABE_EBADARG,
                 "stft_stats_rows: workspace too small (%zu < %zu)", workspace_bytes, need);
    FusedStatsArgs f{};
    f.x = x; f.y = y; f.B = B; f.T = T; f.window = window; f.roots = reinterpret_cast<const float2*>(twiddle);
    f.partial = static_cast<float*>(workspace);
    return launch_stats_rows_fused(f, abc, st);
  }
  const int F = nfft / 2 + 1;
  for (int b = 0; b < B; ++b) {
    const size_t o = (size_t)b * T;
    const int rc = babe_stft_stats(x + o, y + o, 1, T, nfft, window, twiddle, 0, abc + (size_t)b * 3 * F,
                                   workspace, workspace_bytes, stream);
    if (rc) return rc;
  }
  return BABE_OK;
}
