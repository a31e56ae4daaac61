// Fused STFT -> H -> iSTFT operator (forward and adjoint) for NFFT = 4096 on sm_100a, second generation.
//
// Reference semantics: utils/blind_bwe_utils.py:6-39 of eloimoliner/BABE (apply_stft + apply_filter_istft:
// periodic Hamming window, hop N/2, right zero padding by N, center=False, torch.istft envelope division);
// adjoint per SURVEY App. A.1; H designed in the kernel from (fc, A) per utils/blind_bwe_utils.py:82-119.
//
// What changed against round 1's k_apply_filter<Core3,1> (stft_ops.cu), profile profiles/r01_apply_filter.md:
//  * frame tiles are staged by the TMA engine: ONE elected thread per frame-pair group issues one 1-D bulk copy
//    (cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes, SASS UBLKCP) of the pair's three
//    contiguous half-frames (24 KB) and the group waits on an mbarrier; no per-thread address / predicate /
//    LDGSTS work in the loop.  The copy of pair p+1 is in flight while pair p is transformed.
//  * Core4k (core4k.cuh): the second exchange of every transform stays inside a half-warp, so a pair needs
//    3 group barriers instead of 7.
//  * adjoint / epilogue variants are compile-time (the load phase of the old kernel spent 16 % of its issue
//    slots on per-element uniform branches); the envelope division is folded into one of the two window
//    tables (interior blocks) and the tables are stored once (the Hamming window is symmetric);
//    the residual sum of squares is accumulated in fp32 per pair and in fp64 across pairs.
// Rows whose length is not a multiple of 4 samples (or a misaligned base pointer) cannot be bulk-copied and
// take the round-1 kernel.
#include <math.h>

#include <algorithm>

#include "common.cuh"
#include "core4k.cuh"
#include "filter_design.cuh"
#include "stft_fused.cuh"

namespace babe {

// ---------------------------------------------------------------------------
// mbarrier + bulk copy (TMA) wrappers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// samples [base, base + count) of the row, as far as they exist (the readers mask the rest)
__device__ __forceinline__ void issue_copy(float* stage, uint64_t* bar, const float* xr, int T, long long base, int count) {
  const long long left = (long long)T - base;
  const uint32_t bytes = left <= 0 ? 0u : (uint32_t)(left < count ? left : count) * 4u;
  if (bytes) {
    mbar_arrive_tx(bar, bytes);
    bulk_g2s(stage, xr + base, bytes, bar);
  } else {
    mbar_arrive(bar);
  }
}

// ---------------------------------------------------------------------------
// shared-memory layout
// ---------------------------------------------------------------------------
constexpr int TAB = 2052;                                    // 2049 floats, padded to 16 bytes

template <bool SUBSTAGE>
constexpr size_t fused_smem_bytes() {
  return sizeof(float2) * 256 + sizeof(float) * 3 * TAB + sizeof(float2) * Core4k::EX +
         sizeof(float) * (3 + (SUBSTAGE ? 2 : 0)) * Core4k::HOP + 32;
}

// Work distribution: the B * nblk output blocks of the batch, in row-major order, are cut into equal
// contiguous runs of `q` blocks, one per CTA (a run may span several rows; a row may be shared by several
// CTAs).  A run that starts inside a row costs one extra frame (the one whose second half overlaps the
// run's first block); nothing else is computed twice and every CTA does the same amount of work.
//
// EPI: 0 none, 1 subtract + sum of squares (guidance residual), 2 row scale (guidance adjoint),
//      3 any combination decided at run time
// ROWS: one filter per row, fc / A are [B, K] and status is int[B]; H is (re)designed whenever the CTA's
//       segment loop enters a new row, between two segments, when no bulk copy is in flight
// MASK (ROWS only): known-prefix observation model D_b x = m_b x + (1 - m_b) A_b x with m_b[n] = 1[n < kn],
//       kn = known[row] (kn <= 0: no mask, kn >= T: every sample known).  Forward: samples n < kn of the output are
//       x itself; adjoint: D_b^T x = A_b^T (x 1[n >= kn]) + x 1[n < kn].  Only the frame pairs and output blocks of the
//       prefix take a branch (pair- / block-uniform): the adjoint zeroes their staged samples below kn at read time,
//       the epilogues read x from global memory (the stage has been recycled by then).
template <bool ADJ, int EPI, bool ROWS, bool MASK = false>
__global__ void __launch_bounds__(256, 2) k_filter_fused(const FusedArgs a) {
  using C = Core4k;
  constexpr bool SUBSTAGE = EPI == 1 || EPI == 3;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float2* tw3 = reinterpret_cast<float2*>(smem_raw);
  float* wa = reinterpret_cast<float*>(tw3 + 256);                     // analysis window
  float* ws = wa + TAB;                                                // synthesis window
  float* hp = ws + TAB;                                                // H / N, permuted (Core4k::perm_of_bin)
  float2* ex = reinterpret_cast<float2*>(hp + TAB);
  float* stage = reinterpret_cast<float*>(ex + C::EX);
  float* substage = stage + 3 * C::HOP;
  uint64_t* mbar = reinterpret_cast<uint64_t*>(substage + (SUBSTAGE ? 2 * C::HOP : 0));
  uint64_t* mbar_sub = mbar + 1;
  __shared__ FilterSegs segs;
  __shared__ float fkf[BABE_MAX_BREAKPOINTS];
  __shared__ double warp_part[8];

  const int t = threadIdx.x;

  // ---- tables ------------------------------------------------------------------------------------------
  tw3[t] = a.roots[(16 * (t >> 4) * (t & 15)) & (C::N - 1)];
  for (int n = t; n <= C::HOP; n += 256) {
    const int r = n & (C::HOP - 1);
    const float wl = a.window[r], wh = a.window[r + C::HOP];
    const float ienv = __frcp_rn(__fadd_rn(wh * wh, wl * wl));   // interior blocks: two frames overlap
    const float plain = a.window[n], fold = plain * ienv;
    wa[n] = ADJ ? fold : plain;
    ws[n] = ADJ ? plain : fold;
  }
  constexpr float inv_n = 1.0f / C::N;
  if (ROWS) {
    // per-row H: designed in the segment loop
  } else if (a.H != nullptr) {
    for (int k = t; k < C::F; k += 256) hp[C::perm_of_bin(k)] = a.H[k] * inv_n;
  } else {
    float* fs = stage;                                           // the staging area is still free
    for (int k = t; k < C::F; k += 256) fs[k] = a.freqs[k];
    __syncthreads();
    build_segments_coop(segs, fkf, a.fc, a.A, a.K, fs, C::F);
    if (t == 0 && segs.bad && a.status != nullptr && blockIdx.x == 0) *a.status = 1;
    for (int k = t; k < C::F; k += 256) hp[C::perm_of_bin(k)] = bin_gain(segs, k, fs[k]) * inv_n;
  }
  if (t == 0) {
    mbar_init(mbar, 1);
    mbar_init(mbar_sub, 1);
    fence_proxy_async();
  }
  __syncthreads();

  C::TwRegs tw;
  tw.init(a.roots, t);
  const float* wa_lo = wa + t;
  const float* wa_hi = wa + (256 - t);        // window sample 256 n1 + t, n1 >= 8, is entry 256 (15 - n1) + 256 - t
  const float* ws_lo = ws + t;
  const float* ws_hi = ws + (256 - t);
  const float* hp_lo = hp + t;
  const float* hp_hi = hp + C::mirror_base(t);
  const bool has_sub = EPI == 1 || (EPI == 3 && a.sub != nullptr);
  const bool has_scale = EPI == 2 || (EPI == 3 && a.row_scale != nullptr);
  const bool has_sumsq = EPI == 1 || (EPI == 3 && a.item_sumsq != nullptr);
  uint32_t phase = 0, phase_sub = 0;

  const long long total = (long long)a.B * a.nblk;
  long long b0 = (long long)blockIdx.x * a.q;
  const long long b1 = b0 + a.q < total ? b0 + a.q : total;
  int designed = -1;                                             // ROWS: row whose H is in hp
  while (b0 < b1) {
    // ---- one segment: blocks [j0, j1) of one row -------------------------------------------------------
    const int row = (int)(b0 / a.nblk);
    if (ROWS && row != designed) {
      // H of this row.  The staging area is scratch for the bin frequencies, as in the prologue: between two
      // segments no bulk copy is in flight (the last pair's copy was consumed before its closing barrier, which
      // every thread has passed, so hp and segs are no longer read either)
      float* fs = stage;
      for (int k = t; k < C::F; k += 256) fs[k] = a.freqs[k];
      __syncthreads();
      build_segments_coop(segs, fkf, a.fc + (size_t)row * a.K, a.A + (size_t)row * a.K, a.K, fs, C::F);
      if (t == 0 && segs.bad && a.status != nullptr) a.status[row] = 1;
      for (int k = t; k < C::F; k += 256) hp[C::perm_of_bin(k)] = bin_gain(segs, k, fs[k]) * inv_n;
      designed = row;
      __syncthreads();                                           // hp complete, fs read before the copy below
      if (t == 0) fence_proxy_async();                           // generic-proxy writes of the stage before the copy
    }
    const int j0 = (int)(b0 - (long long)row * a.nblk);
    const int j1 = (int)((long long)j0 + (b1 - b0) < a.nblk ? (long long)j0 + (b1 - b0) : a.nblk);
    b0 += j1 - j0;
    const int fs = max(j0 - 1, 0);
    const int fe = min(j1 - 1, a.frames - 1);
    const float* xr = a.x + (size_t)row * a.T;
    float* yr = a.y + (size_t)row * a.T;
    const float* subr = has_sub ? a.sub + (size_t)row * a.T : nullptr;
    const float rs = has_scale ? a.row_scale[row] : 1.0f;
    const int kn = MASK ? a.known[row] : 0;
    float carry[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) carry[i] = 0.f;
    double acc = 0.0;

    if (t == 0) issue_copy(stage, mbar, xr, a.T, (long long)fs * C::HOP, 3 * C::HOP);   // free: barrier at the end of a pair
    for (int fA = fs; fA <= fe; fA += 2) {
      float2 z[16];
      // the residual epilogue's reference samples of output blocks fA, fA+1: in flight during the transforms
      if (SUBSTAGE && has_sub && t == 0) issue_copy(substage, mbar_sub, subr, a.T, (long long)fA * C::HOP, 2 * C::HOP);
      {
        // ---- the pair's 3 half-frames from the staging buffer -------------------------------------------
        float xs[24];
        mbar_wait(mbar, phase);
        phase ^= 1u;
        const long long base = (long long)fA * C::HOP + t;
        if ((long long)(fA + 3) * C::HOP <= a.T) {
#pragma unroll
          for (int j = 0; j < 24; ++j) xs[j] = stage[256 * j + t];
        } else {
#pragma unroll
          for (int j = 0; j < 24; ++j) xs[j] = (base + 256 * j < a.T) ? stage[256 * j + t] : 0.f;
        }
        if (MASK && ADJ && (long long)fA * C::HOP < kn) {
          // D^T: the known samples do not go through the filter
#pragma unroll
          for (int j = 0; j < 24; ++j) xs[j] = (base + 256 * j < kn) ? 0.f : xs[j];
        }
        if (ADJ && fA == 0) {
          // input block 0 is covered by one frame only: divide by w^2 instead of the interior envelope
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float w = ws_lo[256 * j];                      // plain window (synthesis table when ADJ)
            xs[j] = __fdiv_rn(xs[j], w * w) * __fdiv_rn(w, wa_lo[256 * j]);
          }
        }
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) z[n1] = make_float2(xs[n1], xs[n1 + 8]);
      }
      {
        float w[16];
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) w[n1] = n1 < 8 ? wa_lo[256 * n1] : wa_hi[256 * (15 - n1)];
        C::fwd_p1<C::TwRegs, true>(z, ex, tw, t, w);
      }
      group_sync<256>(1);
      if (t == 0 && fA + 2 <= fe)                                // every thread has read the stage
        issue_copy(stage, mbar, xr, a.T, (long long)(fA + 2) * C::HOP, 3 * C::HOP);
      C::fwd_p2_load(z, ex, t);
      __syncwarp();
      C::fwd_p2_store(z, ex, t);
      __syncwarp();
      C::fwd_p3(z, ex, tw3, t);
      {
        float h[16];
#pragma unroll
        for (int k3 = 0; k3 < 16; ++k3) h[k3] = k3 < 8 ? hp_lo[256 * k3] : hp_hi[256 * (15 - k3)];
        C::inv_q1<true>(z, ex, tw3, t, h);   // writes exactly the 16 entries this thread read in fwd_p3
      }
      __syncwarp();
      C::inv_q2_load(z, ex, t);
      __syncwarp();
      C::inv_q2_store(z, ex, t);
      group_sync<256>(1);
      C::inv_q3(z, ex, tw, t);
      // ---- window, overlap-add, (envelope folded into the window), epilogue, store ------------------------
      float o[16];
      if (!ADJ && fA == 0) {
        // output block 0 is covered by frame 0 only: (a w) / (w w)
#pragma unroll
        for (int n1 = 0; n1 < 8; ++n1) {
          const float w = wa_lo[256 * n1];                       // plain window (analysis table when !ADJ)
          o[n1] = __fdiv_rn(z[n1].x * w, w * w);
        }
      } else {
#pragma unroll
        for (int n1 = 0; n1 < 8; ++n1) o[n1] = fmaf(z[n1].x, ws_lo[256 * n1], carry[n1]);
      }
#pragma unroll
      for (int n1 = 0; n1 < 8; ++n1) {
        const float wh = ws_hi[256 * (7 - n1)];                  // window sample 256 (n1 + 8) + t
        o[8 + n1] = fmaf(z[8 + n1].x, wh, z[n1].y * ws_lo[256 * n1]);
        carry[n1] = z[8 + n1].y * wh;
      }
      if (SUBSTAGE && has_sub) {
        mbar_wait(mbar_sub, phase_sub);
        phase_sub ^= 1u;
      }
      float accp = 0.f;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int blk = fA + half;
        if (blk < j0 || blk >= j1) continue;
        const long long p0 = (long long)blk * C::HOP;
        float* yb = yr + p0;
        const bool pre = MASK && p0 < kn;                        // block overlaps the known prefix
        if (p0 + C::HOP <= a.T) {
#pragma unroll
          for (int n1 = 0; n1 < 8; ++n1) {
            float v = o[8 * half + n1];
            const int r = 256 * n1 + t;
            if (pre && p0 + r < kn) v = ADJ ? v + xr[p0 + r] : xr[p0 + r];
            if (SUBSTAGE && has_sub) v -= substage[C::HOP * half + r];
            if (has_scale) v *= rs;
            yb[r] = v;
            if (has_sumsq) accp = fmaf(v, v, accp);
          }
        } else {
#pragma unroll
          for (int n1 = 0; n1 < 8; ++n1) {
            float v = o[8 * half + n1];
            const int r = 256 * n1 + t;
            if (p0 + r < a.T) {
              if (pre && p0 + r < kn) v = ADJ ? v + xr[p0 + r] : xr[p0 + r];
              if (SUBSTAGE && has_sub) v -= substage[C::HOP * half + r];
              if (has_scale) v *= rs;
              yb[r] = v;
              if (has_sumsq) accp = fmaf(v, v, accp);
            }
          }
        }
      }
      if (has_sumsq) acc += (double)accp;
      group_sync<256>(1);                 // ex, the stage (after the last pair) and substage may be overwritten
    }
    if (has_sumsq) {
      // one partial per (CTA, row) segment, slot = CTA + row; k_segment_sumsq adds a row's slots in a fixed order
      acc = warp_sum(acc);
      if ((t & 31) == 0) warp_part[t >> 5] = acc;
      __syncthreads();
      if (t == 0) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += warp_part[w];
        a.item_sumsq[blockIdx.x + row] = s;
      }
      __syncthreads();
    }
  }
}

// row_sumsq[row] += sum of the row's segment partials, in CTA order (deterministic)
__global__ void k_segment_sumsq(const double* seg_sumsq, int nblk, int q, double* row_sumsq) {
  const int row = blockIdx.x;
  const long long g_lo = ((long long)row * nblk) / q, g_hi = ((long long)(row + 1) * nblk - 1) / q;
  double s = 0.0;
  for (long long g = g_lo; g <= g_hi; ++g) s += seg_sumsq[g + row];
  row_sumsq[row] += s;
}

// ---------------------------------------------------------------------------
// Fit statistics (SURVEY App. A.3):  a_k = sum |X|^2, b_k = sum |X||Y|, c_k = sum |Y|^2 over all rows and
// frames, X = STFT(x), Y = STFT(y) (utils/blind_bwe_utils.py:15-26, :250-296).  One frame of x and of y per
// complex transform (z = w x + i w y); X and Y are separated with ONE exchange of the upper half of the
// packed spectrum (thread t's partner is thread 271 - t); the three sums of a thread's 8 bins live in
// registers for the whole run of frames a CTA owns.  Frames are staged by bulk TMA copies like the frame
// pairs of k_filter_fused; the B * frames frames of the batch are cut into equal contiguous runs.
// ---------------------------------------------------------------------------
constexpr size_t stats_smem_bytes() {
  return sizeof(float2) * 256 + sizeof(float) * TAB + sizeof(float2) * Core4k::EX + sizeof(float2) * (8 * 256 + 8) +
         sizeof(float) * 2 * Core4k::N + 32;
}

// ROWS: statistics per group of consecutive rows (a.offsets; NULL: one group per row).  A CTA's run of frames may cross
// group boundaries: its register sums are written out and cleared whenever the next frame starts a new group, one
// partial per (CTA, group) segment at slot CTA + group (as k_segment_sumsq indexes the residual partials), and
// k_reduce_stats_rows adds a group's slots in a fixed order.  Slots stay below grid + G - 1 <= grid + B.
template <bool ROWS>
__global__ void __launch_bounds__(256, 2) k_stats_fused(const FusedStatsArgs a) {
  using C = Core4k;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float2* tw3 = reinterpret_cast<float2*>(smem_raw);
  float* win = reinterpret_cast<float*>(tw3 + 256);
  float2* ex = reinterpret_cast<float2*>(win + TAB);
  float2* mir = ex + C::EX;                       // [8][256] upper-half spectrum + padding
  float* stage = reinterpret_cast<float*>(mir + 8 * 256 + 8);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(stage + 2 * C::N);
  const int t = threadIdx.x;
  tw3[t] = a.roots[(16 * (t >> 4) * (t & 15)) & (C::N - 1)];
  for (int n = t; n <= C::HOP; n += 256) win[n] = a.window[n];
  if (t == 0) {
    mbar_init(mbar, 1);
    fence_proxy_async();
  }
  __syncthreads();
  C::TwRegs tw;
  tw.init(a.roots, t);
  const float* w_lo = win + t;
  const float* w_hi = win + (256 - t);
  // partner thread of the X / Y separation: bins N - k of this thread's bins k < 2048
  const float2* mp = mir + (t == 0 ? 256 : (t < 16 ? 16 - t : 271 - t));
  float sa[8], sb[8], sc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { sa[i] = 0.f; sb[i] = 0.f; sc[i] = 0.f; }
  float na = 0.f, nb = 0.f, nc = 0.f;             // Nyquist bin (thread 0)
  uint32_t phase = 0;

  const long long total = (long long)a.B * a.frames;
  const long long g0 = (long long)blockIdx.x * a.q;
  const long long g1 = g0 + a.q < total ? g0 + a.q : total;
  auto issue = [&](long long g) {
    const int row = (int)(g / a.frames);
    const long long base = (g - (long long)row * a.frames) * C::HOP;
    const long long left = (long long)a.T - base;
    const uint32_t bytes = left <= 0 ? 0u : (uint32_t)(left < C::N ? left : C::N) * 4u;
    if (bytes) {
      mbar_arrive_tx(mbar, 2 * bytes);
      bulk_g2s(stage, a.x + (size_t)row * a.T + base, bytes, mbar);
      bulk_g2s(stage + C::N, a.y + (size_t)row * a.T + base, bytes, mbar);
    } else {
      mbar_arrive(mbar);
    }
  };
  auto flush = [&](long long slot) {
    float* out = a.partial + (size_t)slot * 3 * C::F;
#pragma unroll
    for (int k3 = 0; k3 < 8; ++k3) {
      const int k = C::bin_of(t, k3);
      out[k] = 0.25f * sa[k3];
      out[C::F + k] = 0.25f * sb[k3];
      out[2 * C::F + k] = 0.25f * sc[k3];
    }
    if (t == 0) {
      out[2048] = 0.25f * na;
      out[C::F + 2048] = 0.25f * nb;
      out[2 * C::F + 2048] = 0.25f * nc;
    }
  };
  // ROWS: group of the current frame and the first row past it
  int grp = 0, gend = 0;
  if (ROWS && g0 < g1) {
    const int row0 = (int)(g0 / a.frames);
    if (a.offsets == nullptr) {
      grp = row0;
    } else {
      int hi = a.G;                                   // offsets[grp] <= row0 < offsets[hi]
      while (hi - grp > 1) {
        const int mid = (grp + hi) >> 1;
        if (a.offsets[mid] <= row0) grp = mid; else hi = mid;
      }
    }
    gend = a.offsets == nullptr ? grp + 1 : a.offsets[grp + 1];
  }
  if (t == 0 && g0 < g1) issue(g0);
  for (long long g = g0; g < g1; ++g) {
    float2 z[16];
    {
      const int f = (int)(g % a.frames);
      mbar_wait(mbar, phase);
      phase ^= 1u;
      const long long base = (long long)f * C::HOP + t;
      if ((long long)(f + 2) * C::HOP <= a.T) {
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) z[n1] = make_float2(stage[256 * n1 + t], stage[C::N + 256 * n1 + t]);
      } else {
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
          const bool in = base + 256 * n1 < a.T;
          z[n1] = make_float2(in ? stage[256 * n1 + t] : 0.f, in ? stage[C::N + 256 * n1 + t] : 0.f);
        }
      }
    }
    {
      float w[16];
#pragma unroll
      for (int n1 = 0; n1 < 16; ++n1) w[n1] = n1 < 8 ? w_lo[256 * n1] : w_hi[256 * (15 - n1)];
      C::fwd_p1<C::TwRegs, true>(z, ex, tw, t, w);
    }
    group_sync<256>(1);
    if (t == 0 && g + 1 < g1) issue(g + 1);          // every thread has read the stage
    C::fwd_p2_load(z, ex, t);
    __syncwarp();
    C::fwd_p2_store(z, ex, t);
    __syncwarp();
    C::fwd_p3(z, ex, tw3, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) mir[256 * j + t] = z[8 + j];
    group_sync<256>(1);
#pragma unroll
    for (int k3 = 0; k3 < 8; ++k3) {
      float2 p = mp[256 * (7 - k3)];                  // Z[N - k]
      if (k3 == 0 && t == 0) p = z[0];                // DC is its own mirror
      // X = (Z + conj P) / 2, Y = (Z - conj P) / (2 i); the factors 1/2 are applied once at the end
      const float xre = z[k3].x + p.x, xim = z[k3].y - p.y;
      const float yre = z[k3].y + p.y, yim = p.x - z[k3].x;
      const float sx = fmaf(xre, xre, xim * xim), sy = fmaf(yre, yre, yim * yim);
      sa[k3] += sx;
      sb[k3] += sqrtf(sx * sy);
      sc[k3] += sy;
    }
    if (t == 0) {                                     // Nyquist: Z[2048] is its own mirror
      const float sx = 4.f * z[8].x * z[8].x, sy = 4.f * z[8].y * z[8].y;
      na += sx; nb += sqrtf(sx * sy); nc += sy;
    }
    if (ROWS && (g + 1 == g1 || g + 1 == (long long)gend * a.frames)) {    // last frame of the run or of its group
      flush(blockIdx.x + grp);
#pragma unroll
      for (int i = 0; i < 8; ++i) { sa[i] = 0.f; sb[i] = 0.f; sc[i] = 0.f; }
      na = nb = nc = 0.f;
      if (g + 1 < g1) {
        ++grp;
        gend = a.offsets == nullptr ? grp + 1 : a.offsets[grp + 1];
      }
    }
  }
  if (!ROWS) flush(blockIdx.x);
}

// abc[grp][i] = sum of the group's segment partials (slots g + grp of the CTAs g whose run touches the group's rows
// [r0, r1); offsets NULL: group = row); the same 8-slice fixed-order sum as k_reduce_stats, so one group of all rows
// gives k_reduce_stats' result bit for bit
__global__ void __launch_bounds__(256) k_reduce_stats_rows(const float* partial, int frames, int q, int n, double* abc,
                                                           const int* offsets) {
  __shared__ double sl[8][33];
  const int grp = blockIdx.y;
  const int r0 = offsets == nullptr ? grp : offsets[grp], r1 = offsets == nullptr ? grp + 1 : offsets[grp + 1];
  const int o = threadIdx.x & 31, sidx = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + o;
  const long long g_lo = ((long long)r0 * frames) / q, g_hi = ((long long)r1 * frames - 1) / q;
  double s = 0.0;
  if (i < n)
    for (long long g = g_lo + sidx; g <= g_hi; g += 8) s += (double)partial[(size_t)(g + grp) * n + i];
  sl[sidx][o] = s;
  __syncthreads();
  if (sidx == 0 && i < n) {
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sl[k][o];
    abc[(size_t)grp * n + i] = t;
  }
}

// ---------------------------------------------------------------------------
// FIR "same" convolution by overlap-save on Core4k (SURVEY 8f-4: predict_bwe("firwin"),
// testing/blind_bwe_sampler.py:211-218, utils/bandwidth_extension.py:76-95).  torch conv1d is a correlation:
//   y[n] = sum_k b[k] x[n + k - pl],  pl = (L-1)/2.  A block of V = N - L + 1 outputs needs N inputs; two consecutive
// blocks ride one complex transform and the packed spectrum is multiplied by G = conj(FFT(taps)) / N (host-prepared,
// permuted into the [k3][thread] order of Core4k once per CTA).  Both input windows are staged by bulk TMA copies:
// their starts are arbitrary sample positions, so each copy begins at the 16-byte boundary below the window and
// the readers add the remainder.
// ---------------------------------------------------------------------------
constexpr int FIR_STAGE = Core4k::N + 8;        // floats per staged window (4096 + alignment slack, 16-byte multiple)

constexpr size_t fir_smem_bytes() {
  return sizeof(float2) * (256 + Core4k::N + Core4k::EX) + sizeof(float) * 2 * FIR_STAGE + 32;
}

// window [a0, a0 + N) of a row of length T into `dst` such that sample a0 + n sits at dst[off + n];
// returns off (0..3); positions outside [0, T) are left untouched (the readers mask them)
__device__ __forceinline__ int fir_issue(float* dst, uint64_t* bar, const float* xr, int T, long long a0,
                                         uint32_t* bytes_out) {
  long long lo = a0 >= 0 ? (a0 & ~3LL) : -(((-a0) + 3) & ~3LL);      // 16-byte boundary at or below a0
  const int off = (int)(a0 - lo);
  long long hi = a0 + Core4k::N;                                   // one past the last sample needed
  hi = (hi + 3) & ~3LL;
  long long c0 = lo < 0 ? 0 : lo, c1 = hi > T ? T : hi;              // clipped to the row (T % 4 == 0)
  uint32_t bytes = c1 > c0 ? (uint32_t)(c1 - c0) * 4u : 0u;
  if (bytes) bulk_g2s(dst + (c0 - lo), xr + c0, bytes, bar);
  *bytes_out = bytes;
  return off;
}

__global__ void __launch_bounds__(256, 2) k_fir_fused(const FusedFirArgs a) {
  using C = Core4k;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float2* tw3 = reinterpret_cast<float2*>(smem_raw);
  float2* gp = tw3 + 256;                          // G permuted: entry 256 k3 + t = G[bin_of(t, k3)]
  float2* ex = gp + C::N;
  float* stage = reinterpret_cast<float*>(ex + C::EX);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(stage + 2 * FIR_STAGE);
  const int t = threadIdx.x;
  tw3[t] = a.roots[(16 * (t >> 4) * (t & 15)) & (C::N - 1)];
#pragma unroll
  for (int k3 = 0; k3 < 16; ++k3) gp[256 * k3 + t] = a.G[C::bin_of(t, k3)];
  if (t == 0) {
    mbar_init(mbar, 1);
    fence_proxy_async();
  }
  __syncthreads();
  C::TwRegs tw;
  tw.init(a.roots, t);
  uint32_t phase = 0;
  const long long total = (long long)a.B * a.pairs_per_row;
  const long long i0 = (long long)blockIdx.x * a.q;
  const long long i1 = i0 + a.q < total ? i0 + a.q : total;
  auto issue = [&](long long item) {
    const int row = (int)(item / a.pairs_per_row);
    const long long s0 = (item - (long long)row * a.pairs_per_row) * 2 * a.V;
    const float* xr = a.x + (size_t)row * a.T;
    uint32_t b0, b1;
    // expect the total first: the byte counts are known before either copy is issued
    {
      long long aA = s0 - a.pl, aB = aA + a.V;
      auto nbytes = [&](long long a0) {
        long long lo = a0 >= 0 ? (a0 & ~3LL) : -(((-a0) + 3) & ~3LL);
        long long hi = (a0 + C::N + 3) & ~3LL;
        long long c0 = lo < 0 ? 0 : lo, c1 = hi > a.T ? a.T : hi;
        return c1 > c0 ? (uint32_t)(c1 - c0) * 4u : 0u;
      };
      const uint32_t tot = nbytes(aA) + nbytes(aB);
      if (tot) mbar_arrive_tx(mbar, tot); else mbar_arrive(mbar);
      fir_issue(stage, mbar, xr, a.T, aA, &b0);
      fir_issue(stage + FIR_STAGE, mbar, xr, a.T, aB, &b1);
    }
  };
  if (t == 0 && i0 < i1) issue(i0);
  for (long long item = i0; item < i1; ++item) {
    const int row = (int)(item / a.pairs_per_row);
    const long long s0 = (item - (long long)row * a.pairs_per_row) * 2 * a.V;
    float* yr = a.y + (size_t)row * a.T;
    float2 z[16];
    {
      const long long aA = s0 - a.pl, aB = aA + a.V;
      const long long loA = aA >= 0 ? (aA & ~3LL) : -(((-aA) + 3) & ~3LL);
      const long long loB = aB >= 0 ? (aB & ~3LL) : -(((-aB) + 3) & ~3LL);
      const int offA = (int)(aA - loA), offB = (int)(aB - loB);
      mbar_wait(mbar, phase);
      phase ^= 1u;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const long long pa = aA + 256 * j + t, pb = aB + 256 * j + t;
        const float va = stage[offA + 256 * j + t], vb = stage[FIR_STAGE + offB + 256 * j + t];
        z[j] = make_float2((pa >= 0 && pa < a.T) ? va : 0.f, (pb >= 0 && pb < a.T) ? vb : 0.f);
      }
    }
    C::fwd_p1(z, ex, tw, t);
    group_sync<256>(1);
    if (t == 0 && item + 1 < i1) issue(item + 1);        // every thread has read the stage
    C::fwd_p2_load(z, ex, t);
    __syncwarp();
    C::fwd_p2_store(z, ex, t);
    __syncwarp();
    C::fwd_p3(z, ex, tw3, t);
#pragma unroll
    for (int k3 = 0; k3 < 16; ++k3) z[k3] = c_mul(z[k3], gp[256 * k3 + t]);
    C::inv_q1(z, ex, tw3, t);
    __syncwarp();
    C::inv_q2_load(z, ex, t);
    __syncwarp();
    C::inv_q2_store(z, ex, t);
    group_sync<256>(1);
    C::inv_q3(z, ex, tw, t);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int n = 256 * j + t;
      if (n < a.V) {
        const long long pa = s0 + n, pb = pa + a.V;
        if (pa < a.T) yr[pa] = z[j].x;
        if (pb < a.T) yr[pb] = z[j].y;
      }
    }
    group_sync<256>(1);                                  // ex may be overwritten
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static int g_fused_variant = 0;     // 0: fused kernels (this file); -1: round-1 kernels (stft_ops.cu)

// blocks per CTA: equal runs over at most 2 CTAs per SM; odd, so that a run starting inside a row is a whole
// number of frame pairs
static int fused_run_length(int B, int nblk) {
  const long long total = (long long)B * nblk;
  const long long ctas = 2LL * sm_count();
  long long q = (total + ctas - 1) / ctas;
  if (q < 1) q = 1;
  q |= 1;
  return (int)q;
}

template <bool ADJ, int EPI, bool ROWS, bool MASK>
static int launch_epi(FusedArgs a, cudaStream_t st) {
  const long long total = (long long)a.B * a.nblk;
  const int grid = (int)((total + a.q - 1) / a.q);
  constexpr size_t smem = fused_smem_bytes<EPI == 1 || EPI == 3>();
  auto kern = k_filter_fused<ADJ, EPI, ROWS, MASK>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<grid, 256, smem, st>>>(a);
  return check_launch("k_filter_fused");
}

bool fused_filter_eligible(const float* x, const float* sub, int T) {
  auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return g_fused_variant >= 0 && (T % 4 == 0) && al(x) && al(sub);
}

size_t fused_sumsq_slots(int B, int T) {
  const int nblk = (T - 1) / Core4k::HOP + 1;
  const long long total = (long long)B * nblk;
  const int q = fused_run_length(B, nblk);
  return (size_t)((total + q - 1) / q) + (size_t)B;
}

template <bool ROWS, bool MASK>
static int launch_variant(const FusedArgs& a, cudaStream_t st) {
  const bool sub = a.sub != nullptr, sc = a.row_scale != nullptr, ss = a.item_sumsq != nullptr;
  if (a.adjoint) {
    if (!sub && !sc && !ss) return launch_epi<true, 0, ROWS, MASK>(a, st);
    if (!sub && sc && !ss) return launch_epi<true, 2, ROWS, MASK>(a, st);
    return launch_epi<true, 3, ROWS, MASK>(a, st);
  }
  if (!sub && !sc && !ss) return launch_epi<false, 0, ROWS, MASK>(a, st);
  if (sub && !sc && ss) return launch_epi<false, 1, ROWS, MASK>(a, st);
  return launch_epi<false, 3, ROWS, MASK>(a, st);
}

int launch_filter_fused(FusedArgs a, double* row_sumsq, cudaStream_t st) {
  a.frames = 1 + a.T / Core4k::HOP;
  a.nblk = (a.T - 1) / Core4k::HOP + 1;
  a.q = fused_run_length(a.B, a.nblk);
  const bool ss = a.item_sumsq != nullptr;
  const int rc = !a.per_row ? launch_variant<false, false>(a, st)
                 : a.known != nullptr ? launch_variant<true, true>(a, st) : launch_variant<true, false>(a, st);
  if (rc || !ss) return rc;
  k_segment_sumsq<<<a.B, 1, 0, st>>>(a.item_sumsq, a.nblk, a.q, row_sumsq);
  return check_launch("k_segment_sumsq");
}

bool fused_stats_eligible(const float* x, const float* y, int T, int mode) {
  auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return g_fused_variant >= 0 && mode == 0 && (T % 4 == 0) && al(x) && al(y);
}

static int stats_run_length(int B, int frames) {
  const long long total = (long long)B * frames;
  const long long ctas = 2LL * sm_count();
  long long q = (total + ctas - 1) / ctas;
  if (q < 1) q = 1;
  return (int)q;
}

int launch_stats_fused(FusedStatsArgs a, int* n_partials, cudaStream_t st) {
  a.frames = 1 + a.T / Core4k::HOP;
  const long long total = (long long)a.B * a.frames;
  a.q = stats_run_length(a.B, a.frames);
  const int grid = (int)((total + a.q - 1) / a.q);
  *n_partials = grid;
  constexpr size_t smem = stats_smem_bytes();
  cudaFuncSetAttribute(k_stats_fused<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_stats_fused<false><<<grid, 256, smem, st>>>(a);
  return check_launch("k_stats_fused");
}

size_t fused_stats_rows_slots(int B, int T) {
  const int frames = 1 + T / Core4k::HOP;
  const long long total = (long long)B * frames;
  const int q = stats_run_length(B, frames);
  return (size_t)((total + q - 1) / q) + (size_t)B;
}

int launch_stats_rows_fused(FusedStatsArgs a, double* abc, cudaStream_t st) {
  a.frames = 1 + a.T / Core4k::HOP;
  const long long total = (long long)a.B * a.frames;
  a.q = stats_run_length(a.B, a.frames);
  const int grid = (int)((total + a.q - 1) / a.q);
  constexpr size_t smem = stats_smem_bytes();
  cudaFuncSetAttribute(k_stats_fused<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_stats_fused<true><<<grid, 256, smem, st>>>(a);
  int rc = check_launch("k_stats_fused");
  if (rc) return rc;
  const int n = 3 * Core4k::F;
  const int groups = a.offsets == nullptr ? a.B : a.G;
  k_reduce_stats_rows<<<dim3((n + 31) / 32, groups), 256, 0, st>>>(a.partial, a.frames, a.q, n, abc, a.offsets);
  return check_launch("k_reduce_stats_rows");
}

bool fused_fir_eligible(const float* x, int T) {
  return g_fused_variant >= 0 && (T % 4 == 0) && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
}

int launch_fir_fused(FusedFirArgs a, cudaStream_t st) {
  const long long total = (long long)a.B * a.pairs_per_row;
  const long long ctas = 2LL * sm_count();
  long long q = (total + ctas - 1) / ctas;
  if (q < 1) q = 1;
  a.q = (int)q;
  const int grid = (int)((total + q - 1) / q);
  constexpr size_t smem = fir_smem_bytes();
  cudaFuncSetAttribute(k_fir_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_fir_fused<<<grid, 256, smem, st>>>(a);
  return check_launch("k_fir_fused");
}

}  // namespace babe

// profiling / A-B knob (profiles/probe_r02.py): which implementation serves NFFT = 4096
namespace babe { void set_fit_variant(int v); }
extern "C" int babe_set_fused_variant(int v) {
  if (v < -1 || v > 0) return BABE_EBADARG;
  babe::g_fused_variant = v;
  babe::set_fit_variant(v);
  return BABE_OK;
}
extern "C" int babe_get_fused_variant(void) { return babe::g_fused_variant; }
