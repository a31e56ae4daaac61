// Filter design, its vector-Jacobian product, the device-resident projected
// gradient descent on (fc, A), and spectrogram-domain magnitude statistics.
//
// Reference semantics: design_filter (utils/blind_bwe_utils.py:82-119),
// apply_filter_and_norm_STFTmag_fweighted (:250-296) and
// BlindSampler.fit_params (testing/blind_bwe_sampler.py:533-595) of
// eloimoliner/BABE; analytic gradients per SURVEY Appendix A.2 / A.3.
#include <math.h>
#include <cooperative_groups.h>

#include <algorithm>

#include "common.cuh"
#include "filter_design.cuh"

namespace cg = cooperative_groups;

namespace babe {

constexpr int KMAX = BABE_MAX_BREAKPOINTS;
constexpr int FIT_THREADS = 512;
constexpr int FIT_WARPS = FIT_THREADS / 32;

// ---------------------------------------------------------------------------
__global__ void k_design_filter(const float* fc, const float* A, int K, const float* gain_db,
                                const float* freqs, int F, float* H, int* status) {
  __shared__ FilterSegs segs;
  __shared__ float fkf[BABE_MAX_BREAKPOINTS];
  build_segments_coop(segs, fkf, fc, A, K, freqs, F);
  if (threadIdx.x == 0 && segs.bad && status != nullptr && blockIdx.x == 0) *status = 1;
  float g = 1.0f;
  if (gain_db != nullptr) g = exp10f(__fdiv_rn(gain_db[0], 20.0f));
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < F; k += gridDim.x * blockDim.x) {
    float h = bin_gain(segs, k, freqs[k]);
    if (gain_db != nullptr) h = __fmul_rn(h, g);
    H[k] = h;
  }
}

// Block-wide sum of NV doubles held per thread (v[0..NV)), result valid in
// thread 0 (returned in v).  scratch: FIT_WARPS * NV doubles.
template <int NV>
__device__ __forceinline__ void block_sum(double (&v)[NV], double* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) scratch[warp * NV + i] = v[i];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      double s = 0.0;
      for (int w = 0; w < FIT_WARPS; ++w) s += scratch[w * NV + i];
      v[i] = s;
    }
  }
  __syncthreads();
}

// Accumulate, for the calling thread's bins, per-segment sums
//   s[i] += u_k                (k owned by i)
//   l[i] += u_k log2(f_k/fc_i) (k owned by i)
// where u_k = dL/dH_k * H_k.
// Then (thread 0) the chain rule through the anchors gives dL/dfc, dL/dA.
__global__ void __launch_bounds__(FIT_THREADS, 1)
k_design_filter_vjp(const float* fc, const float* A, int K, const float* gain_db,
                    const float* freqs, int F, const float* gH, float* gfc_out, float* gA_out,
                    float* ggain_out) {
  __shared__ FilterSegs segs;
  __shared__ double scratch[FIT_WARPS * (2 * KMAX + 1)];
  __shared__ float fkf[BABE_MAX_BREAKPOINTS];
  build_segments_coop(segs, fkf, fc, A, K, freqs, F);
  float g = 1.0f;
  if (gain_db != nullptr) g = exp10f(__fdiv_rn(gain_db[0], 20.0f));
  double v[2 * KMAX + 1];
#pragma unroll
  for (int i = 0; i < 2 * KMAX + 1; ++i) v[i] = 0.0;
  for (int k = threadIdx.x; k < F; k += blockDim.x) {
    const float fk = freqs[k];
    const int o = bin_owner(segs, k);
    const float h = bin_gain(segs, k, fk) * g;
    const double u = (double)gH[k] * (double)h;
    v[2 * KMAX] += u;                              // for dL/dG
    if (o >= 0) {
      const double lg = (double)log2f(__fdiv_rn(fk, segs.fc[o]));
#pragma unroll
      for (int i = 0; i < KMAX; ++i) {
        if (i == o) { v[i] += u; v[KMAX + i] += u * lg; }
      }
    }
  }
  block_sum<2 * KMAX + 1>(v, scratch);
  if (threadIdx.x == 0) {
    double gfc[KMAX], gA[KMAX];
    finish_param_grads(segs, freqs, F, v, v + KMAX, gfc, gA);
    for (int i = 0; i < K; ++i) { gfc_out[i] = (float)gfc[i]; gA_out[i] = (float)gA[i]; }
    if (ggain_out != nullptr) ggain_out[0] = (float)(0.11512925464970229 * v[2 * KMAX]);
  }
}

// ---------------------------------------------------------------------------
// device-resident fit loop (single CTA)
// ---------------------------------------------------------------------------
struct FitArgs {
  const double* abc; const float* w; const float* freqs; int F;
  float* params; int K; babe_fit_config cfg; int* iters_out;
};

__global__ void __launch_bounds__(FIT_THREADS, 1) k_fit_params(const FitArgs a) {
  // Per iteration (3 CTA barriers):
  //  (A) every thread evaluates its bins: H_k, the loss term and u_k = (norm dnorm/dH_k) H_k, into
  //      shared memory;
  //  (B) warp (q, s) sums quantity q (segment q's u and u*log2(f/fc_q), or the loss) over bin slice s,
  //      so that all 16 warps work;
  //  (C) warp 0 alone: lane j applies the chain rule through the anchors for breakpoint j, lane 0
  //      takes the fp32 gradient step, the sequential clamps and the stopping test
  //      (testing/blind_bwe_sampler.py:569-588), lanes < K re-locate their breakpoints, lane 0 links
  //      the anchors for the next iteration -- warp-synchronous, no CTA barrier in between.
  // All sums run in a fixed order (bitwise reproducible).
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int F = a.F, K = a.K;
  double* sa = reinterpret_cast<double*>(smem_raw);            // w^2 a
  double* sb = sa + F;                                         // w^2 b
  double* su = sb + F;                                         // u_k
  double* sl = su + F;                                         // u_k log2(f_k/fc_owner)
  double* ss = sl + F;                                         // loss term
  float* sf = reinterpret_cast<float*>(ss + F);                // freqs
  signed char* sown = reinterpret_cast<signed char*>(sf + F);  // owner of bin k
  __shared__ FilterSegs segs;
  __shared__ float fkf[KMAX];
  __shared__ double scratch[FIT_WARPS];
  __shared__ double red[FIT_WARPS + KMAX + 1][2];
  __shared__ double gsum[2 * KMAX + 1];                        // s-sums, l-sums, loss at [2 KMAX]
  __shared__ float cur[2 * KMAX], prev[2 * KMAX];
  __shared__ int stop_flag;
  __shared__ double c_total;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int NQ = K + 1;                                        // K segments + the loss
  const int NS = FIT_WARPS / NQ > 0 ? FIT_WARPS / NQ : 1;      // bin slices per quantity

  {
    double v = 0.0;
    for (int k = threadIdx.x; k < F; k += blockDim.x) {
      const double w2 = (double)a.w[k] * (double)a.w[k];
      sa[k] = w2 * a.abc[k];
      sb[k] = w2 * a.abc[F + k];
      sf[k] = a.freqs[k];
      v += w2 * a.abc[2 * F + k];
    }
    v = warp_sum(v);
    if (lane == 0) scratch[warp] = v;
    if (threadIdx.x < K) { cur[threadIdx.x] = a.params[threadIdx.x]; cur[KMAX + threadIdx.x] = a.params[K + threadIdx.x]; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int w = 0; w < FIT_WARPS; ++w) s += scratch[w];
      c_total = s;
      stop_flag = 0;
    }
  }
  build_segments_coop(segs, fkf, cur, cur + KMAX, K, sf, F);    // ends with a CTA barrier

  int it = 0;
  for (int iter = 0; iter < a.cfg.max_iter; ++iter) {
    for (int k = threadIdx.x; k < F; k += blockDim.x) {                 // (A)
      const float fk = sf[k];
      const int o = bin_owner(segs, k);
      const double h = (double)bin_gain(segs, k, fk);
      const double wa = sa[k], wb = sb[k];
      ss[k] = h * (h * wa - 2.0 * wb);
      double u = 0.0, l = 0.0;
      if (o >= 0) {
        u = (h * wa - wb) * h;
        l = u * (double)log2f(__fdiv_rn(fk, segs.fc[o]));
      }
      su[k] = u; sl[k] = l; sown[k] = (signed char)o;
    }
    __syncthreads();
    for (int job = warp; job < NQ * NS; job += FIT_WARPS) {             // (B)
      const int q = job / NS, s = job - q * NS;
      const int k0 = (int)(((long long)F * s) / NS), k1 = (int)(((long long)F * (s + 1)) / NS);
      double s0 = 0.0, s1 = 0.0;
      if (q < K) {
        for (int k = k0 + lane; k < k1; k += 32)
          if (sown[k] == q) { s0 += su[k]; s1 += sl[k]; }
      } else {
        for (int k = k0 + lane; k < k1; k += 32) s0 += ss[k];
      }
      s0 = warp_sum(s0); s1 = warp_sum(s1);
      if (lane == 0) { red[job][0] = s0; red[job][1] = s1; }
    }
    __syncthreads();
    if (warp == 0) {                                                    // (C)
      if (lane <= K) {                                                  // slice partials, fixed order
        double t0 = 0.0, t1 = 0.0;
        for (int s = 0; s < NS; ++s) { t0 += red[lane * NS + s][0]; t1 += red[lane * NS + s][1]; }
        if (lane < K) { gsum[lane] = t0; gsum[KMAX + lane] = t1; } else { gsum[2 * KMAX] = t0; }
      }
      __syncwarp();
      const double alpha = 0.11512925464970229, ln2 = 0.6931471805599453;
      double gfc = 0.0, gA = 0.0;
      if (lane < K) {
        // dL/dA_j, dL/dfc_j: own segment plus every segment whose anchor chain passes through j
        const int j = lane;
        double ssum = 0.0;
        for (int i = 0; i < K; ++i) {
          if (segs.kf[i] >= F) continue;
          if (i == j) { ssum += gsum[i]; gA += alpha * gsum[KMAX + i]; continue; }
          int c = i;                                  // walk i's ancestors; c = child of j on the path
          while (segs.parent[c] >= 0 && segs.parent[c] != j) c = segs.parent[c];
          if (segs.parent[c] == j) {
            ssum += gsum[i];
            gA += alpha * (double)log2f(__fdiv_rn(sf[segs.kf[c]], segs.fc[j])) * gsum[i];
          }
        }
        gfc = -alpha * (double)segs.A[j] / ((double)segs.fc[j] * ln2) * ssum;
        const double S = gsum[2 * KMAX] + c_total;
        const double inv_norm = 1.0 / sqrt(S > 0.0 ? S : 0.0);
        // gradient step in fp32 like the reference (:569)
        cur[j] = __fsub_rn(cur[j], __fmul_rn(a.cfg.mu_fc, (float)(gfc * inv_norm)));
        cur[KMAX + j] = __fsub_rn(cur[KMAX + j], __fmul_rn(a.cfg.mu_A, (float)(gA * inv_norm)));
      }
      __syncwarp();
      if (lane == 0) {                                                  // sequential clamps (:576-583)
        fit_project(cur, cur + KMAX, K, a.cfg);
        if (iter > 0 && fit_converged(cur, cur + KMAX, prev, prev + KMAX, K, a.cfg)) stop_flag = 1;
        for (int k = 0; k < K; ++k) { prev[k] = cur[k]; prev[KMAX + k] = cur[KMAX + k]; }
      }
      __syncwarp();
      // segments of the next iterate (warp-synchronous version of build_segments_coop)
      if (lane < K) {
        const float c = cur[lane];
        segs.fc[lane] = c;
        segs.A[lane] = cur[KMAX + lane];
        const int k = first_bin_ge(sf, F, c);
        segs.kf[lane] = k;
        fkf[lane] = (k < F) ? sf[k] : 0.f;
      }
      __syncwarp();
      if (lane == 0) {
        segs.K = K;
        segs.bad = 0;
        for (int i = 0; i < K; ++i) {
          int p = -1;
          for (int j = 0; j < i; ++j)
            if (segs.kf[j] <= segs.kf[i]) p = j;
          segs.parent[i] = p;
          if (i > 0 && segs.kf[i] >= F) { segs.bad = 1; segs.anchor[i] = 1.0f; continue; }
          segs.anchor[i] = (i == 0 || p < 0) ? 1.0f
                                             : __fmul_rn(seg_gain(segs.A[p], segs.fc[p], fkf[i]), segs.anchor[p]);
        }
      }
    }
    __syncthreads();
    it = iter + 1;
    if (stop_flag) break;
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < K; ++i) { a.params[i] = cur[i]; a.params[K + i] = cur[KMAX + i]; }
    if (a.iters_out != nullptr) *a.iters_out = it;
  }
}

// ---------------------------------------------------------------------------
// device-resident fit loop, second generation (same arithmetic as k_fit_params above; ~5x less latency per
// iteration).  Round-1 profile (profiles/r01_fit_params.md): 19.8 K cycles per iteration, half of it a serial
// section on one lane (chain rule walk, sequential clamps, 11-step binary searches, a K-step chain of
// log2 / exp10 for the anchors), 40 % the per-bin evaluation with its second log2 and per-bin owner search, the
// rest three CTA barriers and segment-wise shared-memory reductions.  Here
//  * every thread owns <= 5 CONTIGUOUS bins whose static data (f, w^2 a, w^2 b) stay in registers; per-segment sums
//    accumulate in registers and are reduced with one multi-value butterfly per warp (16 double shuffles for 16
//    values instead of 5 per value) + one pass over the 16 warp partials;
//  * warp 0 keeps the breakpoint state in the registers of lanes 0..K-1: chain rule from a precomputed
//    child-of-ancestor table, gradient step, the SEQUENTIAL clamps as shuffle scans (bit-identical to the
//    reference's order, testing/blind_bwe_sampler.py:576-583), closed-form first-bin search with a table fix-up,
//    parents by shuffles, gains in parallel and only the anchor products chained;
//  * two CTA barriers per iteration.
// ---------------------------------------------------------------------------
constexpr int FIT2_NB = 5;            // bins per thread (F <= 2560)

// sum of NV = 16 doubles per lane over the 32 lanes of a warp with 16 shuffles: after the call lane L holds the
// total of value (L >> 1) (both lanes of a pair hold it)
__device__ __forceinline__ double warp_reduce16(double (&v)[16], int lane) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {     // xor 16: lanes with bit 4 clear keep values 0..7, the others 8..15
    const bool up = lane & 16;
    const double send = up ? v[i] : v[i + 8];
    const double keep = up ? v[i + 8] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool up = lane & 8;
    const double send = up ? v[i] : v[i + 4];
    const double keep = up ? v[i + 4] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool up = lane & 4;
    const double send = up ? v[i] : v[i + 2];
    const double keep = up ? v[i + 2] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  {
    const bool up = lane & 2;
    const double send = up ? v[0] : v[1];
    const double keep = up ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
  return v[0];
}
// index of the value lane L holds after warp_reduce16
__device__ __forceinline__ int reduce16_index(int lane) {
  return ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
}

template <int K>      // exact number of breakpoints (1..8): every loop over breakpoints unrolls, lane tests are predicates
__global__ void __launch_bounds__(FIT_THREADS, 1) k_fit_params2(const FitArgs a) {
  constexpr int KP = K;
  const int F = a.F;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sf = reinterpret_cast<float*>(smem_raw);                       // bin frequencies
  __shared__ int s_kf[KMAX];
  __shared__ float s_fc[KMAX], s_A[KMAX], s_anchor[KMAX];
  __shared__ double red[FIT_WARPS][17];
  __shared__ double gS[KMAX], gL[KMAX];
  __shared__ signed char child[KMAX][KMAX];       // child[i][j]: the ancestor-or-self of i whose parent is j (-1: none)
  __shared__ float s_lgc[KMAX];                   // log2(f[kf[c]] / fc[parent[c]]) of breakpoint c
  __shared__ int stop_flag;
  __shared__ double c_total_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ---- static per-bin data of this thread's contiguous bins ----------------------------------------------
  const int base = F / FIT_THREADS, rem = F - base * FIT_THREADS;
  const int nb = base + (tid < rem ? 1 : 0);
  const int k0 = tid * base + min(tid, rem);
  float fk[FIT2_NB];
  double wa[FIT2_NB], wb[FIT2_NB];
  double ct = 0.0;
#pragma unroll
  for (int i = 0; i < FIT2_NB; ++i) {
    fk[i] = 1.0f; wa[i] = 0.0; wb[i] = 0.0;
    if (i < nb) {
      const int k = k0 + i;
      const double w2 = (double)a.w[k] * (double)a.w[k];
      fk[i] = a.freqs[k];
      wa[i] = w2 * a.abc[k];
      wb[i] = w2 * a.abc[F + k];
      ct += w2 * a.abc[2 * F + k];
    }
  }
  for (int k = tid; k < F; k += FIT_THREADS) sf[k] = a.freqs[k];
  ct = warp_sum(ct);
  if (lane == 0) red[warp][16] = ct;
  if (tid == 0) stop_flag = 0;
  __syncthreads();
  // ---- breakpoint state in the registers of warp 0, lanes 0..K-1 --------------------------------------------
  const bool bp = warp == 0 && lane < K;
  float fc = 0.f, A = 0.f, fc_prev = 0.f, A_prev = 0.f;
  if (bp) { fc = a.params[lane]; A = a.params[K + lane]; }
  const float df = F > 1 ? (sf[F - 1] - sf[0]) / (float)(F - 1) : 1.0f;
  const float inv_df = 1.0f / df;
  double c_total = 0.0;

  // segments of the current (fc, A): kf, parent, gains, anchors, child table -> shared memory (warp 0 only)
  auto build = [&]() {
    __syncwarp();                                                // the chain rule has read the previous tables
    int kf = F, par = -1;
    float fkf = 0.f, lgc = 0.f, anchor = 1.0f;
    if (lane < K) {
      if (fc == fc) {                                           // NaN -> F, like first_bin_ge
        int k = (int)fminf(fmaxf((fc - sf[0]) * inv_df, 0.f), (float)F);
        while (k > 0 && sf[k - 1] >= fc) --k;
        while (k < F && sf[k] < fc) ++k;
        kf = k;
      }
      fkf = kf < F ? sf[kf] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < K; ++i) {                                // parent = last earlier breakpoint at or below
      const int kfi = __shfl_sync(0xffffffffu, kf, i);
      if (lane < K && i < lane && kfi <= kf) par = i;
    }
    const float fc_p = __shfl_sync(0xffffffffu, fc, par >= 0 ? par : 0);
    const float A_p = __shfl_sync(0xffffffffu, A, par >= 0 ? par : 0);
    float g = 1.0f;
    const bool chained = lane < K && lane > 0 && par >= 0 && kf < F;
    if (chained) {
      lgc = log2f(rn_div(fkf, fc_p));
      g = exp10f(rn_div(rn_mul(A_p, lgc), 20.0f));               // seg_gain(A_p, fc_p, fkf)
    }
#pragma unroll
    for (int i = 1; i < K; ++i) {                                // anchors along the parent chain, in order
      const float ap = __shfl_sync(0xffffffffu, anchor, par >= 0 ? par : 0);
      if (lane == i && chained) anchor = rn_mul(g, ap);
    }
    if (lane < K) {
      s_kf[lane] = kf; s_fc[lane] = fc; s_A[lane] = A; s_anchor[lane] = anchor; s_lgc[lane] = lgc;
#pragma unroll
      for (int j = 0; j < K; ++j) child[lane][j] = (signed char)(j == lane ? lane : -1);
    }
    __syncwarp();
    int c = lane, q = (lane < K && kf < F) ? par : -1;           // walk this breakpoint's ancestors
#pragma unroll
    for (int s2 = 0; s2 < K - 1; ++s2) {
      if (q >= 0) child[lane][q] = (signed char)c;
      const int nq = __shfl_sync(0xffffffffu, par, q >= 0 ? q : 0);
      if (q >= 0) { c = q; q = nq; }
    }
    return kf;
  };
  int my_kf = F;
  if (warp == 0) {
    double s = 0.0;
    if (lane < FIT_WARPS) s = red[lane][16];
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);     // 16 partials, fixed order
    if (lane == 0) c_total_s = s;
    my_kf = build();
  }
  __syncthreads();
  c_total = c_total_s;

  int it = 0;
  for (int iter = 0; iter < a.cfg.max_iter; ++iter) {
    // ---- (A) per-bin evaluation, per-segment sums in registers ------------------------------------------
    double v[16], loss = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.0;
    int kfr[KP];
#pragma unroll
    for (int i = 0; i < KP; ++i) kfr[i] = i < K ? s_kf[i] : 0x7fffffff;
    // owners are non-decreasing along a thread's contiguous bins: sums of a run of equal owners are flushed into
    // the per-segment accumulators only when the owner changes
    int run_o = -1;
    double run_u = 0.0, run_l = 0.0;
#pragma unroll
    for (int b = 0; b < FIT2_NB; ++b) {
      if (b < nb) {
        const int k = k0 + b;
        int o = -1;
#pragma unroll
        for (int i = 0; i < KP; ++i) if (kfr[i] <= k) o = i;
        float h = 1.0f, lg = 0.f;
        if (o >= 0) {
          lg = log2f(rn_div(fk[b], s_fc[o]));
          const float g = exp10f(rn_div(rn_mul(s_A[o], lg), 20.0f));
          h = (o == 0) ? g : rn_mul(g, s_anchor[o]);
        }
        const double hd = (double)h;
        loss += hd * (hd * wa[b] - 2.0 * wb[b]);
        if (o != run_o) {
#pragma unroll
          for (int i = 0; i < KP; ++i) if (i == run_o) { v[i] += run_u; v[KP + i] += run_l; }
          run_o = o; run_u = 0.0; run_l = 0.0;
        }
        if (o >= 0) {
          const double u = (hd * wa[b] - wb[b]) * hd;
          run_u += u;
          run_l += u * (double)lg;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < KP; ++i) if (i == run_o) { v[i] += run_u; v[KP + i] += run_l; }
    // ---- (B) block reduction: 2 KP segment sums with one butterfly, the loss with a plain warp sum ----------
    const double tot = warp_reduce16(v, lane);
    loss = warp_sum(loss);
    if ((lane & 1) == 0) red[warp][reduce16_index(lane)] = tot;
    if (lane == 0) red[warp][16] = loss;
    __syncthreads();
    // ---- (C) warp 0: totals, chain rule, step, clamps, stopping test, next segments --------------------------
    if (warp == 0) {
      {
        const int q = lane & 15, hhalf = lane >> 4;              // value q, warps [8 hhalf, 8 hhalf + 8)
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += red[8 * hhalf + w][q];
        s += __shfl_xor_sync(0xffffffffu, s, 16);
        if (lane < KP) gS[lane] = s; else if (lane < 2 * KP) gL[lane - KP] = s;
        double ls = lane < FIT_WARPS ? red[lane][16] : 0.0;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) ls += __shfl_xor_sync(0xffffffffu, ls, o);
        loss = __shfl_sync(0xffffffffu, ls, 0);
      }
      __syncwarp();
      const double alpha = 0.11512925464970229, ln2 = 0.6931471805599453;
      if (lane < K) {
        const int j = lane;
        double ssum = 0.0, gA = 0.0;
#pragma unroll
        for (int i = 0; i < K; ++i) {
          const int c = child[i][j];
          if (c < 0 || s_kf[i] >= F) continue;
          const double Si = gS[i];
          ssum += Si;
          gA += (i == j) ? alpha * gL[i] : alpha * (double)s_lgc[c] * Si;
        }
        const double gfc = -alpha * (double)A / ((double)fc * ln2) * ssum;
        const double S = loss + c_total;
        const double inv_norm = 1.0 / sqrt(S > 0.0 ? S : 0.0);
        fc = __fsub_rn(fc, __fmul_rn(a.cfg.mu_fc, (float)(gfc * inv_norm)));       // fp32 step (:569)
        A = __fsub_rn(A, __fmul_rn(a.cfg.mu_A, (float)(gA * inv_norm)));
      }
      // sequential clamps (:576-583) as shuffle scans: lane k needs lane k-1's CLAMPED value
      if (a.cfg.clamp_fc) {
        if (lane == 0) fc = fminf(fmaxf(fc, a.cfg.fcmin), a.cfg.fcmax);
#pragma unroll
        for (int k = 1; k < K; ++k) {
          const float pv = __shfl_sync(0xffffffffu, fc, k - 1);
          if (lane == k) fc = fminf(fmaxf(fc, __fadd_rn(pv, 1.0f)), a.cfg.fcmax);
        }
      }
      if (a.cfg.clamp_A) {
        if (lane == 0) A = fminf(fmaxf(A, a.cfg.Amin), a.cfg.only_negative_A ? -1.0f : a.cfg.Amax);
#pragma unroll
        for (int k = 1; k < K; ++k) {
          const float pv = __shfl_sync(0xffffffffu, A, k - 1);
          if (lane == k) A = fminf(fmaxf(A, a.cfg.Amin), a.cfg.only_negative_A ? pv : a.cfg.Amax);
        }
      }
      // stopping test (:586-588): mean |delta| of fc and of A, summed in breakpoint order like fit_converged
      float d0 = lane < K ? fabsf(fc - fc_prev) : 0.f, d1 = lane < K ? fabsf(A - A_prev) : 0.f;
      float t0 = 0.f, t1 = 0.f;
#pragma unroll
      for (int k = 0; k < K; ++k) { t0 += __shfl_sync(0xffffffffu, d0, k); t1 += __shfl_sync(0xffffffffu, d1, k); }
      if (lane == 0 && iter > 0 && t0 / (float)K < a.cfg.tol_fc && t1 / (float)K < a.cfg.tol_A) stop_flag = 1;
      fc_prev = fc; A_prev = A;
      my_kf = build();
    }
    __syncthreads();
    it = iter + 1;
    if (stop_flag) break;
  }
  if (bp) { a.params[lane] = fc; a.params[K + lane] = A; }
  if (tid == 0 && a.iters_out != nullptr) *a.iters_out = it;
  (void)my_kf;
}

// ---------------------------------------------------------------------------
// device-resident fit loop, third generation: a thread-block CLUSTER of 4 CTAs.  clock64 inside k_fit_params2
// (profiles/r02_summary.md): the per-bin evaluation + reduction of an iteration is ISSUE-bound on its one SM
// (16 warps x ~650 instructions in ~2.6 K cycles), the other half is warp 0's serial section.  Here every CTA
// evaluates a quarter of the bins, the 17 per-CTA sums travel to rank 0 through distributed shared memory, rank 0's
// warp 0 runs the unchanged serial section and writes the next segment tables into every CTA's shared memory; two
// cluster barriers per iteration.  Same arithmetic per bin and per breakpoint; only the association of the fp64 sums
// over bins differs (per CTA, then over the 4 CTAs in rank order -- fixed, bitwise reproducible).
// ---------------------------------------------------------------------------
constexpr int FIT3_NC = 4;            // CTAs per cluster
constexpr int FIT3_NB = 2;            // bins per thread: F <= 4 * 512 * 2

// ROWS: one independent fit per cluster; cluster b reads abc[b] (3 F doubles) and owns params[b] (2 K floats) and
// iters_out[b].  Every exchange stays inside the cluster.
template <int K, bool ROWS>
__global__ void __cluster_dims__(FIT3_NC, 1, 1) __launch_bounds__(FIT_THREADS, 1) k_fit_params3(const FitArgs a) {
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  constexpr int KP = K;
  const int F = a.F;
  const double* abc = a.abc;
  float* params = a.params;
  int* iters_out = a.iters_out;
  if (ROWS) {
    const size_t b = blockIdx.x / FIT3_NC;
    abc += b * 3 * F;
    params += b * 2 * K;
    if (iters_out != nullptr) iters_out += b;
  }
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sf = reinterpret_cast<float*>(smem_raw);                       // bin frequencies
  __shared__ int s_kf[KMAX];
  __shared__ float s_fc[KMAX], s_A[KMAX], s_anchor[KMAX];
  __shared__ double red[FIT_WARPS][17];
  __shared__ double part[FIT3_NC][17];            // per-CTA sums, gathered in rank 0's copy through DSMEM
  __shared__ double gS[KMAX], gL[KMAX];
  __shared__ signed char child[KMAX][KMAX];       // child[i][j]: the ancestor-or-self of i whose parent is j (-1: none)
  __shared__ float s_lgc[KMAX];                   // log2(f[kf[c]] / fc[parent[c]]) of breakpoint c
  __shared__ int stop_flag;
  __shared__ double c_total_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ---- static per-bin data of this thread's contiguous bins ----------------------------------------------
  // bins [rank Fq, (rank + 1) Fq) of the CTA, strided over its threads: bin b of the thread is kb0 + 512 b
  const int Fq = (F + FIT3_NC - 1) / FIT3_NC;
  const int cta_lo = rank * Fq, cta_hi = min(F, cta_lo + Fq);
  const int kb0 = cta_lo + tid;
  const int nb = kb0 < cta_hi ? (cta_hi - kb0 + FIT_THREADS - 1) / FIT_THREADS : 0;
  float fk[FIT3_NB];
  double wa[FIT3_NB], wb[FIT3_NB];
  double ct = 0.0;
#pragma unroll
  for (int i = 0; i < FIT3_NB; ++i) {
    fk[i] = 1.0f; wa[i] = 0.0; wb[i] = 0.0;
    if (i < nb) {
      const int k = kb0 + FIT_THREADS * i;
      const double w2 = (double)a.w[k] * (double)a.w[k];
      fk[i] = a.freqs[k];
      wa[i] = w2 * abc[k];
      wb[i] = w2 * abc[F + k];
      ct += w2 * abc[2 * F + k];
    }
  }
  for (int k = tid; k < F; k += FIT_THREADS) sf[k] = a.freqs[k];
  ct = warp_sum(ct);
  if (lane == 0) red[warp][16] = ct;
  if (tid == 0) stop_flag = 0;
  __syncthreads();
  cluster.sync();          // a peer's shared memory may only be addressed once the peer is known to have started
  // ---- breakpoint state in the registers of warp 0, lanes 0..K-1 --------------------------------------------
  const bool bp = warp == 0 && lane < K;
  float fc = 0.f, A = 0.f, fc_prev = 0.f, A_prev = 0.f;
  if (bp) { fc = params[lane]; A = params[K + lane]; }
  const float f0 = sf[0];
  const float df = F > 1 ? (sf[F - 1] - sf[0]) / (float)(F - 1) : 1.0f;
  const float inv_df = 1.0f / df;
  double c_total = 0.0;

  // segments of the current (fc, A): kf, parent, gains, anchors, child table -> shared memory (warp 0 only)
  auto build = [&]() {
    __syncwarp();                                                // the chain rule has read the previous tables
    int kf = F, par = -1;
    float fkf = 0.f, lgc = 0.f, anchor = 1.0f;
    if (lane < K) {
      if (fc == fc) {                                           // NaN -> F, like first_bin_ge
        int k = (int)fminf(fmaxf((fc - f0) * inv_df, 0.f), (float)F);
        // the closed-form guess is within one bin of the answer: its neighbours are loaded together, the loops of the
        // dependent look-ups only run when that is not enough
        const float sm1 = sf[max(k - 1, 0)], s0 = sf[min(k, F - 1)], sp1 = sf[min(k + 1, F - 1)];
        if (k > 0 && sm1 >= fc) {
          --k;
          while (k > 0 && sf[k - 1] >= fc) --k;
          fkf = sf[k];
        } else if (k < F && s0 < fc) {
          ++k;
          if (k < F && sp1 < fc) { ++k; while (k < F && sf[k] < fc) ++k; fkf = k < F ? sf[k] : 0.f; }
          else fkf = k < F ? sp1 : 0.f;
        } else {
          fkf = k < F ? s0 : 0.f;
        }
        kf = k;
      }
    }
#pragma unroll
    for (int i = 0; i < K; ++i) {                                // parent = last earlier breakpoint at or below
      const int kfi = __shfl_sync(0xffffffffu, kf, i);
      if (lane < K && i < lane && kfi <= kf) par = i;
    }
    const float fc_p = __shfl_sync(0xffffffffu, fc, par >= 0 ? par : 0);
    const float A_p = __shfl_sync(0xffffffffu, A, par >= 0 ? par : 0);
    float g = 1.0f;
    const bool chained = lane < K && lane > 0 && par >= 0 && kf < F;
    if (chained) {
      lgc = log2f(rn_div(fkf, fc_p));
      g = exp10f(rn_div(rn_mul(A_p, lgc), 20.0f));               // seg_gain(A_p, fc_p, fkf)
    }
#pragma unroll
    for (int i = 1; i < K; ++i) {                                // anchors along the parent chain, in order
      const float ap = __shfl_sync(0xffffffffu, anchor, par >= 0 ? par : 0);
      if (lane == i && chained) anchor = rn_mul(g, ap);
    }
    if (lane < K) {
#pragma unroll
      for (int r = 1; r < FIT3_NC; ++r) {     // the segment tables every CTA evaluates its bins with
        cluster.map_shared_rank(s_kf, r)[lane] = kf; cluster.map_shared_rank(s_fc, r)[lane] = fc;
        cluster.map_shared_rank(s_A, r)[lane] = A; cluster.map_shared_rank(s_anchor, r)[lane] = anchor;
      }
      s_kf[lane] = kf; s_fc[lane] = fc; s_A[lane] = A; s_anchor[lane] = anchor; s_lgc[lane] = lgc;
#pragma unroll
      for (int j = 0; j < K; ++j) child[lane][j] = (signed char)(j == lane ? lane : -1);
    }
    __syncwarp();
    int c = lane, q = (lane < K && kf < F) ? par : -1;           // walk this breakpoint's ancestors
#pragma unroll
    for (int s2 = 0; s2 < K - 1; ++s2) {
      if (q >= 0) child[lane][q] = (signed char)c;
      const int nq = __shfl_sync(0xffffffffu, par, q >= 0 ? q : 0);
      if (q >= 0) { c = q; q = nq; }
    }
    return kf;
  };
  int my_kf = F;
  if (warp == 0) {
    double s = 0.0;
    if (lane < FIT_WARPS) s = red[lane][16];
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);     // 16 partials, fixed order
    if (lane == 0) cluster.map_shared_rank(&part[0][0], 0)[rank * 17 + 16] = s;
  }
  cluster.sync();
  if (rank == 0 && warp == 0) {
    double s = 0.0;
#pragma unroll
    for (int r = 0; r < FIT3_NC; ++r) s += part[r][16];
    if (lane == 0) c_total_s = s;
    my_kf = build();
  }
  cluster.sync();
  c_total = c_total_s;                      // meaningful in rank 0 only (the only user)

  int it = 0;
  for (int iter = 0; iter < a.cfg.max_iter; ++iter) {
    // ---- (A) per-bin evaluation, per-segment sums in registers ------------------------------------------
    double v[16], loss = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.0;
    int kfr[KP];
#pragma unroll
    for (int i = 0; i < KP; ++i) kfr[i] = i < K ? s_kf[i] : 0x7fffffff;
#pragma unroll
    for (int b = 0; b < FIT3_NB; ++b) {
      if (b < nb) {
        const int k = kb0 + FIT_THREADS * b;
        int o = -1;
#pragma unroll
        for (int i = 0; i < KP; ++i) if (kfr[i] <= k) o = i;
        float h = 1.0f, lg = 0.f;
        if (o >= 0) {
          lg = log2f(rn_div(fk[b], s_fc[o]));
          const float g = exp10f(rn_div(rn_mul(s_A[o], lg), 20.0f));
          h = (o == 0) ? g : rn_mul(g, s_anchor[o]);
        }
        const double hd = (double)h;
        loss += hd * (hd * wa[b] - 2.0 * wb[b]);
        if (o >= 0) {
          const double u = (hd * wa[b] - wb[b]) * hd, ul = u * (double)lg;
#pragma unroll
          for (int i = 0; i < KP; ++i) if (i == o) { v[i] += u; v[KP + i] += ul; }
        }
      }
    }
    // ---- (B) block reduction: 2 KP segment sums with one butterfly, the loss with a plain warp sum ----------
    const double tot = warp_reduce16(v, lane);
    loss = warp_sum(loss);
    if ((lane & 1) == 0) red[warp][reduce16_index(lane)] = tot;
    if (lane == 0) red[warp][16] = loss;
    __syncthreads();
    // ---- (B2) warp 0 of every CTA: the CTA's 17 sums -> rank 0's `part` (distributed shared memory) --------------
    if (warp == 0) {
      const int q = lane & 15, hhalf = lane >> 4;              // value q, warps [8 hhalf, 8 hhalf + 8)
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < 8; ++w) s += red[8 * hhalf + w][q];
      s += __shfl_xor_sync(0xffffffffu, s, 16);
      double ls = lane < FIT_WARPS ? red[lane][16] : 0.0;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) ls += __shfl_xor_sync(0xffffffffu, ls, o);
      double* dst = cluster.map_shared_rank(&part[0][0], 0) + rank * 17;
      if (lane < 16) dst[q] = s;
      if (lane == 0) dst[16] = ls;             // lanes 0..15 hold the sum of the 16 warp partials
    }
    cluster.sync();
    // ---- (C) rank 0, warp 0: totals, chain rule, step, clamps, stopping test, next segments ----------------------
    if (rank == 0 && warp == 0) {
      {
        double s = 0.0, ls = 0.0;
#pragma unroll
        for (int r = 0; r < FIT3_NC; ++r) { s += part[r][lane & 15]; ls += part[r][16]; }
        if (lane < KP) gS[lane] = s; else if (lane < 2 * KP) gL[lane - KP] = s;
        loss = ls;
      }
      __syncwarp();
      const double alpha = 0.11512925464970229, ln2 = 0.6931471805599453;
      if (lane < K) {
        const int j = lane;
        // branch-free, all look-ups issued before the sums (the version with `continue` ran its K iterations one
        // behind the other: 1.5 K of the serial section's 4.7 K cycles, clock64); same additions in the same order --
        // a skipped term adds +0.0
        int cc[K];
        bool ok[K];
        double Sv[K], Lv[K];
#pragma unroll
        for (int i = 0; i < K; ++i) {
          cc[i] = child[i][j];
          ok[i] = cc[i] >= 0 && s_kf[i] < F;
          Sv[i] = gS[i];
          Lv[i] = gL[i];
        }
        float lgv[K];
#pragma unroll
        for (int i = 0; i < K; ++i) lgv[i] = s_lgc[cc[i] < 0 ? 0 : cc[i]];
        double ssum = 0.0, gA = 0.0;
#pragma unroll
        for (int i = 0; i < K; ++i) {
          const double term = (i == j) ? alpha * Lv[i] : alpha * (double)lgv[i] * Sv[i];
          ssum += ok[i] ? Sv[i] : 0.0;
          gA += ok[i] ? term : 0.0;
        }
        // 1 / (fc ln2) and 1 / sqrt(S): fp32 seeds (MUFU) refined by Newton steps in fp64 to < 1e-15 relative -- the
        // IEEE fp64 division and square root were ~1.2 K of the serial section's 4.4 K cycles (clock64)
        const double S = loss + c_total;
        const double d = (double)fc * ln2;
        double r = (double)__frcp_rn((float)d);
        r = r * (2.0 - d * r);
        r = r * (2.0 - d * r);
        const double gfc = -alpha * (double)A * r * ssum;
        double inv_norm;
        if (S > 0.0 && S < 1e30 && S > 1e-30) {
          double y = (double)rsqrtf((float)S);
          y = y * (1.5 - 0.5 * S * y * y);
          y = y * (1.5 - 0.5 * S * y * y);
          inv_norm = y;
        } else {
          inv_norm = 1.0 / sqrt(S > 0.0 ? S : 0.0);
        }
        fc = __fsub_rn(fc, __fmul_rn(a.cfg.mu_fc, (float)(gfc * inv_norm)));       // fp32 step (:569)
        A = __fsub_rn(A, __fmul_rn(a.cfg.mu_A, (float)(gA * inv_norm)));
      }
      // sequential clamps (:576-583) as shuffle scans: lane k needs lane k-1's CLAMPED value; the fc and A scans are
      // independent chains and run interleaved when both are on
      if (a.cfg.clamp_fc && a.cfg.clamp_A) {
        if (lane == 0) {
          fc = fminf(fmaxf(fc, a.cfg.fcmin), a.cfg.fcmax);
          A = fminf(fmaxf(A, a.cfg.Amin), a.cfg.only_negative_A ? -1.0f : a.cfg.Amax);
        }
#pragma unroll
        for (int k = 1; k < K; ++k) {
          const float pf = __shfl_sync(0xffffffffu, fc, k - 1);
          const float pa = __shfl_sync(0xffffffffu, A, k - 1);
          if (lane == k) {
            fc = fminf(fmaxf(fc, __fadd_rn(pf, 1.0f)), a.cfg.fcmax);
            A = fminf(fmaxf(A, a.cfg.Amin), a.cfg.only_negative_A ? pa : a.cfg.Amax);
          }
        }
      } else {
        if (a.cfg.clamp_fc) {
          if (lane == 0) fc = fminf(fmaxf(fc, a.cfg.fcmin), a.cfg.fcmax);
#pragma unroll
          for (int k = 1; k < K; ++k) {
            const float pv = __shfl_sync(0xffffffffu, fc, k - 1);
            if (lane == k) fc = fminf(fmaxf(fc, __fadd_rn(pv, 1.0f)), a.cfg.fcmax);
          }
        }
        if (a.cfg.clamp_A) {
          if (lane == 0) A = fminf(fmaxf(A, a.cfg.Amin), a.cfg.only_negative_A ? -1.0f : a.cfg.Amax);
#pragma unroll
          for (int k = 1; k < K; ++k) {
            const float pv = __shfl_sync(0xffffffffu, A, k - 1);
            if (lane == k) A = fminf(fmaxf(A, a.cfg.Amin), a.cfg.only_negative_A ? pv : a.cfg.Amax);
          }
        }
      }
      // stopping test (:586-588): mean |delta| of fc and of A, summed in breakpoint order like fit_converged
      float d0 = lane < K ? fabsf(fc - fc_prev) : 0.f, d1 = lane < K ? fabsf(A - A_prev) : 0.f;
      float t0 = 0.f, t1 = 0.f;
#pragma unroll
      for (int k = 0; k < K; ++k) { t0 += __shfl_sync(0xffffffffu, d0, k); t1 += __shfl_sync(0xffffffffu, d1, k); }
      if (lane == 0 && iter > 0 && t0 / (float)K < a.cfg.tol_fc && t1 / (float)K < a.cfg.tol_A) {
#pragma unroll
        for (int r = 0; r < FIT3_NC; ++r) *cluster.map_shared_rank(&stop_flag, r) = 1;
      }
      fc_prev = fc; A_prev = A;
      my_kf = build();
    }
    cluster.sync();
    it = iter + 1;
    if (stop_flag) break;
  }
  if (rank == 0 && bp) { params[lane] = fc; params[K + lane] = A; }
  if (rank == 0 && tid == 0 && iters_out != nullptr) *iters_out = it;
  cluster.sync();                           // no CTA exits while a peer may still address its shared memory
  (void)my_kf;
}

// ---------------------------------------------------------------------------
// spectrogram-domain magnitude statistics: one CTA per frequency bin
// ---------------------------------------------------------------------------
// work item = one 32-frame segment of one (row b, bin k) line of the spectrogram: a warp reads 256 contiguous bytes per
// load and no thread divides 64-bit indices
constexpr int SPEC_THREADS = 256;
constexpr int SPEC_UNROLL = 4;
__global__ void __launch_bounds__(SPEC_THREADS) k_spec_mag_stats(const float2* X, const float2* Xref,
                                                                 const float* H, const float* w, int B,
                                                                 int F, int frames, double* out) {
  const int k = blockIdx.x;
  const float h = H ? H[k] : 1.0f;
  const float wk = w ? w[k] : 1.0f;
  double sa = 0, sb = 0, sc = 0, ss = 0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nseg = (frames + 31) >> 5, items = B * nseg;
  for (int it0 = warp; it0 < items; it0 += SPEC_UNROLL * (SPEC_THREADS / 32)) {
    float2 x[SPEC_UNROLL], y[SPEC_UNROLL];
    bool ok[SPEC_UNROLL];
#pragma unroll
    for (int u = 0; u < SPEC_UNROLL; ++u) {              // all loads of the group in flight before the arithmetic
      const int it = it0 + u * (SPEC_THREADS / 32);
      const int b = it / nseg, m = (it - b * nseg) * 32 + lane;
      ok[u] = it < items && m < frames;
      if (ok[u]) {
        const size_t off = ((size_t)b * F + k) * frames + m;
        x[u] = X[off]; y[u] = Xref[off];
      }
    }
#pragma unroll
    for (int u = 0; u < SPEC_UNROLL; ++u) {
      if (!ok[u]) continue;
      // mirror the reference's fp32 order: sqrt(re^2+im^2), *H, *w, difference
      const float mx = sqrtf(__fadd_rn(__fmul_rn(x[u].x, x[u].x), __fmul_rn(x[u].y, x[u].y)));
      const float my = sqrtf(__fadd_rn(__fmul_rn(y[u].x, y[u].x), __fmul_rn(y[u].y, y[u].y)));
      const float d = __fsub_rn(__fmul_rn(__fmul_rn(mx, h), wk), __fmul_rn(my, wk));
      sa += (double)mx * mx; sb += (double)mx * my; sc += (double)my * my;
      ss += (double)d * d;
    }
  }
  __shared__ double red[SPEC_THREADS / 32][4];
  sa = warp_sum(sa); sb = warp_sum(sb); sc = warp_sum(sc); ss = warp_sum(ss);
  if (lane == 0) { red[warp][0] = sa; red[warp][1] = sb; red[warp][2] = sc; red[warp][3] = ss; }
  __syncthreads();
  if (threadIdx.x < 4) {
    double s = 0;
    for (int wv = 0; wv < SPEC_THREADS / 32; ++wv) s += red[wv][threadIdx.x];
    out[(size_t)threadIdx.x * F + k] = s;
  }
}

// gradient of  norm = || w (H |X| - |Xref|) ||_2  wrt the spectrograms (utils/blind_bwe_utils.py:250-296 under
// autograd):  dnorm/dX = coef w^2 (H|X| - |Xref|) H X/|X|,   dnorm/dXref = -coef w^2 (H|X| - |Xref|) Xref/|Xref|,
// coef = upstream gradient / norm (device scalar).  |X| = 0 gives 0/0 = NaN exactly like the reference's sqrt'.
__global__ void __launch_bounds__(SPEC_THREADS) k_spec_mag_grad(const float2* X, const float2* Xref, const float* H,
                                                                const float* w, const float* coef, int F, int frames,
                                                                int rows, float2* gX, float2* gXref) {
  const float c = coef[0];
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * (SPEC_THREADS / 32);
  for (int r = blockIdx.x * (SPEC_THREADS / 32) + (threadIdx.x >> 5); r < rows; r += nwarps) {   // r = b F + k
    const int k = r % F;
    const float h = H ? H[k] : 1.0f, wk = w ? w[k] : 1.0f;
    const size_t base = (size_t)r * frames;
    for (int m = lane; m < frames; m += 32) {
      const size_t i = base + m;
      const float2 x = X[i], y = Xref[i];
      const float mx = sqrtf(__fadd_rn(__fmul_rn(x.x, x.x), __fmul_rn(x.y, x.y)));
      const float my = sqrtf(__fadd_rn(__fmul_rn(y.x, y.x), __fmul_rn(y.y, y.y)));
      const float d = __fsub_rn(__fmul_rn(__fmul_rn(mx, h), wk), __fmul_rn(my, wk));
      const float e = c * d * wk;
      if (gX) { const float s = e * h / mx; gX[i] = make_float2(s * x.x, s * x.y); }
      if (gXref) { const float s = -e / my; gXref[i] = make_float2(s * y.x, s * y.y); }
    }
  }
}

// ---------------------------------------------------------------------------
// spectrogram distances of the STFT-guidance branches (utils/blind_bwe_utils.py:148-197 complex, :198-248 log-magnitude;
// the plain magnitude distance is k_spec_mag_stats / k_spec_mag_grad with H = 1): one pass over both spectrograms
// instead of the reference's multiply / subtract / norm chain.  MODE 0: s_k = sum |w X - w Xref|^2,
// MODE 2: s_k = sum (log10(w|X| + 1e-8) - log10(w|Xref| + 1e-8))^2; fp32 in the reference's operation order,
// accumulated in double.  MODE 3: s_k = sum Re(conj(X) Xref), the per-bin correlation that is dL/dH of
// apply_filter_istft (utils/blind_bwe_utils.py:28-39) when Xref holds the adjoint spectrogram.
// ---------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(SPEC_THREADS) k_spec_dist_stats(const float2* X, const float2* Xref, const float* w,
                                                                  int B, int F, int frames, double* out) {
  const int k = blockIdx.x;
  const float wk = w ? w[k] : 1.0f;
  double ss = 0;
  float part = 0.0f;                       // fp32 partial over one group of work items, folded into the double sum
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nseg = (frames + 31) >> 5, items = B * nseg;
  for (int it0 = warp; it0 < items; it0 += SPEC_UNROLL * (SPEC_THREADS / 32)) {
    float2 x[SPEC_UNROLL], y[SPEC_UNROLL];
    bool ok[SPEC_UNROLL];
#pragma unroll
    for (int u = 0; u < SPEC_UNROLL; ++u) {              // all loads of the group in flight before the arithmetic
      const int it = it0 + u * (SPEC_THREADS / 32);
      const int b = it / nseg, m = (it - b * nseg) * 32 + lane;
      ok[u] = it < items && m < frames;
      if (ok[u]) {
        const size_t off = ((size_t)b * F + k) * frames + m;
        x[u] = X[off]; y[u] = Xref[off];
      }
    }
#pragma unroll
    for (int u = 0; u < SPEC_UNROLL; ++u) {
      if (!ok[u]) continue;
      if (MODE == 0) {
        const float dr = __fsub_rn(__fmul_rn(x[u].x, wk), __fmul_rn(y[u].x, wk));
        const float di = __fsub_rn(__fmul_rn(x[u].y, wk), __fmul_rn(y[u].y, wk));
        part = fmaf(dr, dr, fmaf(di, di, part));
      } else if (MODE == 3) {
        part = fmaf(x[u].x, y[u].x, fmaf(x[u].y, y[u].y, part));
      } else {
        const float mx = sqrtf(__fadd_rn(__fmul_rn(x[u].x, x[u].x), __fmul_rn(x[u].y, x[u].y)));
        const float my = sqrtf(__fadd_rn(__fmul_rn(y[u].x, y[u].x), __fmul_rn(y[u].y, y[u].y)));
        const float d = __fsub_rn(log10f(__fadd_rn(__fmul_rn(mx, wk), 1e-8f)), log10f(__fadd_rn(__fmul_rn(my, wk), 1e-8f)));
        part = fmaf(d, d, part);
      }
    }
    ss += (double)part; part = 0.0f;
  }
  ss += (double)part;
  __shared__ double red[SPEC_THREADS / 32];
  ss = warp_sum(ss);
  if (lane == 0) red[warp] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0;
    for (int wv = 0; wv < SPEC_THREADS / 32; ++wv) s += red[wv];
    out[k] = s;
  }
}

// gradients of those norms wrt the spectrograms (coef = upstream gradient / norm, device scalar):
// MODE 0: gX = coef w^2 (X - Xref) = -gXref;
// MODE 2: gX = coef d w X / (|X| (w|X| + 1e-8) ln 10), gXref = -coef d w Xref / (|Xref| (w|Xref| + 1e-8) ln 10).
template <int MODE>
__global__ void __launch_bounds__(SPEC_THREADS) k_spec_dist_grad(const float2* X, const float2* Xref, const float* w,
                                                                 const float* coef, int F, int frames, int rows,
                                                                 float2* gX, float2* gXref) {
  const float c = coef[0];
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * (SPEC_THREADS / 32);
  for (int r = blockIdx.x * (SPEC_THREADS / 32) + (threadIdx.x >> 5); r < rows; r += nwarps) {   // r = b F + k
    const float wk = w ? w[r % F] : 1.0f;
    const size_t base = (size_t)r * frames;
    for (int m = lane; m < frames; m += 32) {
      const size_t i = base + m;
      const float2 x = X[i], y = Xref[i];
      if (MODE == 0) {
        const float gr = c * wk * __fsub_rn(__fmul_rn(x.x, wk), __fmul_rn(y.x, wk));
        const float gi = c * wk * __fsub_rn(__fmul_rn(x.y, wk), __fmul_rn(y.y, wk));
        if (gX) gX[i] = make_float2(gr, gi);
        if (gXref) gXref[i] = make_float2(-gr, -gi);
      } else {
        const float mx = sqrtf(__fadd_rn(__fmul_rn(x.x, x.x), __fmul_rn(x.y, x.y)));
        const float my = sqrtf(__fadd_rn(__fmul_rn(y.x, y.x), __fmul_rn(y.y, y.y)));
        const float ax = __fadd_rn(__fmul_rn(mx, wk), 1e-8f), ay = __fadd_rn(__fmul_rn(my, wk), 1e-8f);
        const float e = c * __fsub_rn(log10f(ax), log10f(ay)) * wk * 0.43429448190325176f;
        if (gX) { const float s = e / (ax * mx); gX[i] = make_float2(s * x.x, s * x.y); }
        if (gXref) { const float s = -e / (ay * my); gXref[i] = make_float2(s * y.x, s * y.y); }
      }
    }
  }
}

template <bool ROWS>
static int launch_fit3(const FitArgs& a, int B, cudaStream_t st) {
  const size_t smem3 = (size_t)a.F * sizeof(float) + 16;
  const int grid = FIT3_NC * B;
  switch (a.K) {
    case 1: k_fit_params3<1, ROWS><<<grid, FIT_THREADS, smem3, st>>>(a); break;
    case 2: k_fit_params3<2, ROWS><<<grid, FIT_THREADS, smem3, st>>>(a); break;
    case 3: k_fit_params3<3, ROWS><<<grid, FIT_THREADS, smem3, st>>>(a); break;
    case 4: k_fit_params3<4, ROWS><<<grid, FIT_THREADS, smem3, st>>>(a); break;
    case 5: k_fit_params3<5, ROWS><<<grid, FIT_THREADS, smem3, st>>>(a); break;
    case 6: k_fit_params3<6, ROWS><<<grid, FIT_THREADS, smem3, st>>>(a); break;
    case 7: k_fit_params3<7, ROWS><<<grid, FIT_THREADS, smem3, st>>>(a); break;
    default: k_fit_params3<8, ROWS><<<grid, FIT_THREADS, smem3, st>>>(a); break;
  }
  return check_launch("k_fit_params3");
}

static int g_fit_variant = 0;     // 0: k_fit_params3 (4-CTA cluster), 1: k_fit_params2 (one CTA), -1: round-1 k_fit_params
                                  // (A/B: babe_set_fit_variant; babe_set_fused_variant(-1 / 0) sets it too)
void set_fit_variant(int v) { g_fit_variant = v; }

}  // namespace babe

using namespace babe;

extern "C" int babe_design_filter(const float* fc, const float* A, int K, const float* gain_db,
                                  const float* freqs, int F, float* H, int* status,
                                  void* stream) {
  BABE_REQUIRE(fc && A && freqs && H, BABE_EBADARG, "design_filter: null pointer");
  BABE_REQUIRE(K >= 1 && K <= KMAX, BABE_EBADARG, "design_filter: K=%d outside [1,%d]", K, KMAX);
  BABE_REQUIRE(F >= 1, BABE_EBADARG, "design_filter: F=%d", F);
  const int blocks = (F + 255) / 256;
  k_design_filter<<<blocks < 64 ? blocks : 64, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      fc, A, K, gain_db, freqs, F, H, status);
  return check_launch("k_design_filter");
}

extern "C" int babe_design_filter_vjp(const float* fc, const float* A, int K,
                                      const float* gain_db, const float* freqs, int F,
                                      const float* gH, float* gfc, float* gA, float* ggain,
                                      void* stream) {
  BABE_REQUIRE(fc && A && freqs && gH && gfc && gA, BABE_EBADARG, "design_filter_vjp: null pointer");
  BABE_REQUIRE(K >= 1 && K <= KMAX, BABE_EBADARG, "design_filter_vjp: K=%d outside [1,%d]", K, KMAX);
  BABE_REQUIRE(F >= 1, BABE_EBADARG, "design_filter_vjp: F=%d", F);
  k_design_filter_vjp<<<1, FIT_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      fc, A, K, gain_db, freqs, F, gH, gfc, gA, ggain);
  return check_launch("k_design_filter_vjp");
}

extern "C" int babe_set_fit_variant(int v) {
  if (v < -1 || v > 1) return BABE_EBADARG;
  babe::set_fit_variant(v);
  return BABE_OK;
}
extern "C" int babe_fit_params(const double* abc, const float* w, const float* freqs, int F,
                               float* params, int K, const babe_fit_config* cfg,
                               int* iters_out, void* stream) {
  BABE_REQUIRE(abc && w && freqs && params && cfg, BABE_EBADARG, "fit_params: null pointer");
  BABE_REQUIRE(K >= 1 && K <= KMAX, BABE_EBADARG, "fit_params: K=%d outside [1,%d]", K, KMAX);
  const size_t smem = (size_t)F * (5 * sizeof(double) + sizeof(float) + 1) + 16;
  BABE_REQUIRE(F >= 1 && smem <= 200 * 1024, BABE_EUNSUPPORTED, "fit_params: F=%d too large", F);
  FitArgs a{abc, w, freqs, F, params, K, *cfg, iters_out};
  if (K <= 8 && F <= FIT3_NC * FIT_THREADS * FIT3_NB && g_fit_variant == 0) {     // cluster kernel (default)
    return launch_fit3<false>(a, 1, static_cast<cudaStream_t>(stream));
  }
  if (K <= 8 && F <= FIT_THREADS * FIT2_NB && g_fit_variant >= 0) {     // second-generation kernel
    const size_t smem2 = (size_t)F * sizeof(float) + 16;
    cudaStream_t st2 = static_cast<cudaStream_t>(stream);
    switch (K) {
      case 1: k_fit_params2<1><<<1, FIT_THREADS, smem2, st2>>>(a); break;
      case 2: k_fit_params2<2><<<1, FIT_THREADS, smem2, st2>>>(a); break;
      case 3: k_fit_params2<3><<<1, FIT_THREADS, smem2, st2>>>(a); break;
      case 4: k_fit_params2<4><<<1, FIT_THREADS, smem2, st2>>>(a); break;
      case 5: k_fit_params2<5><<<1, FIT_THREADS, smem2, st2>>>(a); break;
      case 6: k_fit_params2<6><<<1, FIT_THREADS, smem2, st2>>>(a); break;
      case 7: k_fit_params2<7><<<1, FIT_THREADS, smem2, st2>>>(a); break;
      default: k_fit_params2<8><<<1, FIT_THREADS, smem2, st2>>>(a); break;
    }
    return check_launch("k_fit_params2");
  }
  cudaFuncSetAttribute(k_fit_params, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_fit_params<<<1, FIT_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(a);
  return check_launch("k_fit_params");
}

extern "C" int babe_fit_params_rows(const double* abc, const float* w, const float* freqs, int F, float* params,
                                    int B, int K, const babe_fit_config* cfg, int* iters_out, void* stream) {
  BABE_REQUIRE(abc && w && freqs && params && cfg, BABE_EBADARG, "fit_params_rows: null pointer");
  BABE_REQUIRE(B >= 0, BABE_EBADARG, "fit_params_rows: B=%d", B);
  BABE_REQUIRE(K >= 1 && K <= KMAX, BABE_EBADARG, "fit_params_rows: K=%d outside [1,%d]", K, KMAX);
  if (B == 0) return BABE_OK;
  if (K <= 8 && F >= 1 && F <= FIT3_NC * FIT_THREADS * FIT3_NB && g_fit_variant == 0) {   // one cluster per row
    FitArgs a{abc, w, freqs, F, params, K, *cfg, iters_out};
    return launch_fit3<true>(a, B, static_cast<cudaStream_t>(stream));
  }
  for (int b = 0; b < B; ++b) {           // other kernels: one shared-mode fit per row
    const int rc = babe_fit_params(abc + (size_t)b * 3 * F, w, freqs, F, params + (size_t)b * 2 * K, K, cfg,
                                   iters_out == nullptr ? nullptr : iters_out + b, stream);
    if (rc) return rc;
  }
  return BABE_OK;
}

extern "C" int babe_spec_mag_stats(const float* X, const float* Xref, const float* H,
                                   const float* w, int B, int F, int frames, double* out,
                                   void* stream) {
  BABE_REQUIRE(X && Xref && out, BABE_EBADARG, "spec_mag_stats: null pointer");
  BABE_REQUIRE(B >= 1 && F >= 1 && frames >= 1, BABE_EBADARG, "spec_mag_stats: bad shape");
  k_spec_mag_stats<<<F, SPEC_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float2*>(X), reinterpret_cast<const float2*>(Xref), H, w, B, F,
      frames, out);
  return check_launch("k_spec_mag_stats");
}

extern "C" int babe_spec_mag_grad(const float* X, const float* Xref, const float* H, const float* w,
                                  const float* coef, int B, int F, int frames, float* gX, float* gXref,
                                  void* stream) {
  BABE_REQUIRE(X && Xref && coef && (gX || gXref), BABE_EBADARG, "spec_mag_grad: null pointer");
  BABE_REQUIRE(B >= 1 && F >= 1 && frames >= 1, BABE_EBADARG, "spec_mag_grad: bad shape");
  BABE_REQUIRE((long long)B * F <= 0x7fffffffLL, BABE_EUNSUPPORTED, "spec_mag_grad: B*F too large");
  const int rows = B * F;                  // one warp per (row, bin) line of `frames` complex values
  const int grid = std::min((rows + SPEC_THREADS / 32 - 1) / (SPEC_THREADS / 32), sm_count() * 8);
  k_spec_mag_grad<<<grid, SPEC_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float2*>(X), reinterpret_cast<const float2*>(Xref), H, w, coef, F, frames, rows,
      reinterpret_cast<float2*>(gX), reinterpret_cast<float2*>(gXref));
  return check_launch("k_spec_mag_grad");
}

extern "C" int babe_spec_dist_stats(const float* X, const float* Xref, const float* w, int mode, int B, int F,
                                    int frames, double* out, void* stream) {
  BABE_REQUIRE(X && Xref && out, BABE_EBADARG, "spec_dist_stats: null pointer");
  BABE_REQUIRE(B >= 1 && F >= 1 && frames >= 1, BABE_EBADARG, "spec_dist_stats: bad shape");
  BABE_REQUIRE(mode == 0 || mode == 2 || mode == 3, BABE_EBADARG,
               "spec_dist_stats: mode=%d (0 complex, 2 log-magnitude, 3 correlation)", mode);
  const float2* x = reinterpret_cast<const float2*>(X);
  const float2* y = reinterpret_cast<const float2*>(Xref);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (mode == 0) k_spec_dist_stats<0><<<F, SPEC_THREADS, 0, st>>>(x, y, w, B, F, frames, out);
  else if (mode == 3) k_spec_dist_stats<3><<<F, SPEC_THREADS, 0, st>>>(x, y, w, B, F, frames, out);
  else k_spec_dist_stats<2><<<F, SPEC_THREADS, 0, st>>>(x, y, w, B, F, frames, out);
  return check_launch("k_spec_dist_stats");
}

extern "C" int babe_spec_dist_grad(const float* X, const float* Xref, const float* w, const float* coef, int mode,
                                   int B, int F, int frames, float* gX, float* gXref, void* stream) {
  BABE_REQUIRE(X && Xref && coef && (gX || gXref), BABE_EBADARG, "spec_dist_grad: null pointer");
  BABE_REQUIRE(B >= 1 && F >= 1 && frames >= 1, BABE_EBADARG, "spec_dist_grad: bad shape");
  BABE_REQUIRE(mode == 0 || mode == 2, BABE_EBADARG, "spec_dist_grad: mode=%d (0 complex, 2 log-magnitude)", mode);
  BABE_REQUIRE((long long)B * F <= 0x7fffffffLL, BABE_EUNSUPPORTED, "spec_dist_grad: B*F too large");
  const int rows = B * F;
  const int grid = std::min((rows + SPEC_THREADS / 32 - 1) / (SPEC_THREADS / 32), sm_count() * 8);
  const float2* x = reinterpret_cast<const float2*>(X);
  const float2* y = reinterpret_cast<const float2*>(Xref);
  float2* gx = reinterpret_cast<float2*>(gX);
  float2* gy = reinterpret_cast<float2*>(gXref);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (mode == 0) k_spec_dist_grad<0><<<grid, SPEC_THREADS, 0, st>>>(x, y, w, coef, F, frames, rows, gx, gy);
  else k_spec_dist_grad<2><<<grid, SPEC_THREADS, 0, st>>>(x, y, w, coef, F, frames, rows, gx, gy);
  return check_launch("k_spec_dist_grad");
}
