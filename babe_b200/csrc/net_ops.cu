// Element-wise glue of the CQTDiff+ residual layers around the (PyTorch / cuDNN)
// convolutions, one HBM pass each instead of ~8 forward + ~16 backward PyTorch
// kernels per layer (SURVEY 8f-2: the caller on either side of the CQT):
//
//   layer (networks/cqtdiff+.py:470-482):
//     h = gelu( BiasFreeGroupNorm(x) * (affine(sigma) + 1) )          k_gn_stats, k_gn_film_gelu
//     y = (x + conv(h) * gate(sigma)) / sqrt(2)                       k_gate_residual
//   BiasFreeGroupNorm (networks/cqtdiff+.py:137-163): x / (std_g(x) + eps) * gamma_c with the
//   unbiased standard deviation of each (sample, group) -- no mean removal of x itself.
//
// Backward wrt the activations (parameters are frozen while sampling):
//   g_v = g_y * gate / sqrt(2)                                        k_gate_residual (x0 = null), or
//                                                                     k_gn_bwd<true> of the next layer
//   g_x = g_y / sqrt(2) + g_u s - G_r r^2 (x - mean) / ((cnt - 1) std)   k_gn_bwd_reduce, k_gn_bwd
//   with u = x s, s = r gamma (aff + 1), r = 1 / (std + eps), g_u = g_h gelu'(u),
//   G_r = sum_group g_u x gamma (aff + 1).
//
// Layout: contiguous NCHW float32; a "plane" is one (n, c) slice of P = F*T elements, a group
// is gc = C/G consecutive planes.  All reductions run in a fixed order (bitwise reproducible).
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace babe {

constexpr int NET_THREADS = 256;
constexpr int MAX_STAT_SLICES = 64;

__device__ __forceinline__ float gelu_f(float u) {
  return 0.5f * u * (1.0f + erff(u * 0.70710678118654752f));
}
__device__ __forceinline__ float gelu_grad_f(float u) {
  const float cdf = 0.5f * (1.0f + erff(u * 0.70710678118654752f));
  const float pdf = 0.3989422804014327f * __expf(-0.5f * u * u);
  return cdf + u * pdf;
}

__device__ __forceinline__ double block_sum_d(double v, double* scratch /*NET_THREADS/32*/) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0) {
    for (int w = 0; w < NET_THREADS / 32; ++w) s += scratch[w];
  }
  return s;          // valid in thread 0
}

// Elements of one plane handled by one CTA of the streaming kernels (4 float4 per thread).
constexpr long long NET_CHUNK = 4LL * NET_THREADS * 4;

// Called by every thread after thread 0 has stored this CTA's partial sums: true in all threads of the
// CTA that arrives last of `total` CTAs at *ctr, whose partials (and those of all others) are then
// visible.  That CTA also resets the counter, so that every kernel leaves the counters zero -- a graph
// replay or the next launch on the stream finds them as the first one did.  No CTA waits for another.
__device__ __forceinline__ bool arrive_last(unsigned* ctr, unsigned total) {
  __shared__ bool s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned prev = atomicAdd(ctr, 1u);
    s_last = (prev == total - 1);
    if (s_last) *ctr = 0u;
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last;
}

// Finished statistics of one (sample, group) from its S partial (sum, sum of squares) pairs, executed
// by warp 0 in a fixed order: stats = {mean, unbiased std}.
__device__ __forceinline__ void finish_stats(const double* part, int S, long long cnt, float2* stats) {
  const int lane = threadIdx.x & 31;
  double s1 = 0.0, s2 = 0.0;
  for (int s = lane; s < S; s += 32) { s1 += __ldcg(part + 2 * s); s2 += __ldcg(part + 2 * s + 1); }
  s1 = warp_sum(s1); s2 = warp_sum(s2);
  if (lane == 0) {
    const double mean = s1 / (double)cnt;
    double var = (s2 - (double)cnt * mean * mean) / (double)(cnt - 1);
    if (var < 0.0) var = 0.0;
    *stats = make_float2((float)mean, (float)sqrt(var));
  }
}

// (sum, sum of squares) of slice blockIdx.x of group blockIdx.y -> part[group][slice][2]; the last
// slice to finish turns them into stats[group]
__global__ void __launch_bounds__(NET_THREADS) k_gn_stats(const float* __restrict__ x,
                                                          double* __restrict__ part,
                                                          float2* __restrict__ stats,
                                                          unsigned* __restrict__ counters,
                                                          long long cnt, int S) {
  __shared__ double scratch[NET_THREADS / 32];
  const long long per = ((cnt + S - 1) / S + 3) & ~3LL;
  const long long lo = per * blockIdx.x, hi = min(cnt, lo + per);
  const float* g = x + (size_t)blockIdx.y * cnt;
  double s1 = 0.0, s2 = 0.0;
  const bool vec = ((reinterpret_cast<uintptr_t>(g) & 15) == 0);
  if (vec) {
    const long long n4 = (hi > lo) ? (hi - lo) / 4 : 0;
    const float4* g4 = reinterpret_cast<const float4*>(g + lo);
    // <= 32 values per float accumulator between two double updates
    for (long long i = threadIdx.x; i < n4; i += 8LL * NET_THREADS) {
      float a1 = 0.f, a2 = 0.f;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const long long j = i + (long long)u * NET_THREADS;
        if (j < n4) {
          const float4 v = g4[j];
          a1 += (v.x + v.y) + (v.z + v.w);
          a2 += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
        }
      }
      s1 += (double)a1; s2 += (double)a2;
    }
    for (long long i = lo + n4 * 4 + threadIdx.x; i < hi; i += NET_THREADS) {
      const float v = g[i];
      s1 += (double)v; s2 += (double)v * (double)v;
    }
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += NET_THREADS) {
      const float v = g[i];
      s1 += (double)v; s2 += (double)v * (double)v;
    }
  }
  s1 = block_sum_d(s1, scratch);
  s2 = block_sum_d(s2, scratch);
  double* pg = part + (size_t)blockIdx.y * S * 2;
  if (threadIdx.x == 0) { pg[2 * blockIdx.x] = s1; pg[2 * blockIdx.x + 1] = s2; }
  if (arrive_last(counters + blockIdx.y, S) && threadIdx.x < 32)
    finish_stats(pg, S, cnt, stats + blockIdx.y);
}

struct PlaneArgs {
  int N, C, G;
  long long P;             // plane size F*T
  float eps, scale;
  const float2* stats;     // [N*G] {mean, std}
  const float* gamma;      // [C]
  const float* aff;        // [N][C]
  const float* gate;       // [N][C] or null (= 1)
  const float* coef;       // [N*G] G_r r^2 / ((cnt - 1) std)
  const float* gate_prev;  // [N][C]: k_gn_bwd also writes g_v of the preceding layer
  float* gv_prev;
  double* part;            // partial sums of the producing kernels
  float2* stats_out;
  float* coef_out;
  unsigned* counters;      // [N*G] zero on entry, left zero
};

// r * gamma[c] * (aff + 1) of plane pc
__device__ __forceinline__ float film_scale(const PlaneArgs& a, int pc, int c, float r) {
  return r * a.gamma[c] * (a.aff[pc] + 1.0f);
}

// h = gelu(x * r * gamma * (aff + 1));  grid (chunks, N*C)
__global__ void __launch_bounds__(NET_THREADS) k_gn_film_gelu(const float* __restrict__ x,
                                                              float* __restrict__ h, const PlaneArgs a) {
  const int pc = blockIdx.y, n = pc / a.C, c = pc - n * a.C;
  const float2 st = a.stats[n * a.G + c / (a.C / a.G)];
  const float s = film_scale(a, pc, c, 1.0f / (st.y + a.eps));
  const float* xp = x + (size_t)pc * a.P;
  float* hp = h + (size_t)pc * a.P;
  const long long lo = NET_CHUNK * blockIdx.x, hi = min(a.P, lo + NET_CHUNK);
  if (((reinterpret_cast<uintptr_t>(xp) | reinterpret_cast<uintptr_t>(hp)) & 15) == 0) {
    float4 xv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {      // all loads in flight before the first gelu
      const long long i = lo + 4LL * (threadIdx.x + u * NET_THREADS);
      if (i + 3 < hi) xv[u] = *reinterpret_cast<const float4*>(xp + i);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = lo + 4LL * (threadIdx.x + u * NET_THREADS);
      if (i + 3 < hi) {
        float4 v = xv[u];
        v.x = gelu_f(v.x * s); v.y = gelu_f(v.y * s); v.z = gelu_f(v.z * s); v.w = gelu_f(v.w * s);
        *reinterpret_cast<float4*>(hp + i) = v;
      } else {
        for (long long j = i; j < hi; ++j) hp[j] = gelu_f(xp[j] * s);
      }
    }
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += NET_THREADS) hp[i] = gelu_f(xp[i] * s);
  }
}

// out = (x0 + v * gate) * scale   (x0 may be null: out = v * gate * scale); grid (chunks, N*C).
// STATS: also the group statistics of out, as k_gn_stats computes them, into a.stats_out; the partial
// slot of CTA (chunk, plane) is (c mod gc) * chunks + chunk of its group.
template <bool STATS>
__global__ void __launch_bounds__(NET_THREADS, 4) k_gate_residual(const float* __restrict__ x0,
                                                               const float* __restrict__ v,
                                                               float* __restrict__ out, const PlaneArgs a) {
  const int pc = blockIdx.y;
  const float gs = (a.gate ? a.gate[pc] : 1.0f) * a.scale, sc = a.scale;
  const float* vp = v + (size_t)pc * a.P;
  const float* xp = x0 ? x0 + (size_t)pc * a.P : nullptr;
  float* op = out + (size_t)pc * a.P;
  const long long lo = NET_CHUNK * blockIdx.x, hi = min(a.P, lo + NET_CHUNK);
  const bool vec = ((reinterpret_cast<uintptr_t>(vp) | reinterpret_cast<uintptr_t>(op) |
                     reinterpret_cast<uintptr_t>(xp)) & 15) == 0;
  float a1 = 0.f, a2 = 0.f;            // <= 16 values each
  double d1 = 0.0, d2 = 0.0;           // scalar paths
  if (vec) {
    float4 vv[4], xv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {      // all loads in flight before the first store
      const long long i = lo + 4LL * (threadIdx.x + u * NET_THREADS);
      if (i + 3 < hi) {
        vv[u] = *reinterpret_cast<const float4*>(vp + i);
        if (xp) xv[u] = *reinterpret_cast<const float4*>(xp + i);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = lo + 4LL * (threadIdx.x + u * NET_THREADS);
      if (i + 3 < hi) {
        float4 q = vv[u];
        if (xp) {
          const float4 b = xv[u];
          q.x = fmaf(q.x, gs, b.x * sc); q.y = fmaf(q.y, gs, b.y * sc);
          q.z = fmaf(q.z, gs, b.z * sc); q.w = fmaf(q.w, gs, b.w * sc);
        } else {
          q.x *= gs; q.y *= gs; q.z *= gs; q.w *= gs;
        }
        *reinterpret_cast<float4*>(op + i) = q;
        if (STATS) {
          a1 += (q.x + q.y) + (q.z + q.w);
          a2 += (q.x * q.x + q.y * q.y) + (q.z * q.z + q.w * q.w);
        }
      } else {
        for (long long j = i; j < hi; ++j) {
          const float o = xp ? fmaf(vp[j], gs, xp[j] * sc) : vp[j] * gs;
          op[j] = o;
          if (STATS) { d1 += (double)o; d2 += (double)o * (double)o; }
        }
      }
    }
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += NET_THREADS) {
      const float o = xp ? fmaf(vp[i], gs, xp[i] * sc) : vp[i] * gs;
      op[i] = o;
      if (STATS) { d1 += (double)o; d2 += (double)o * (double)o; }
    }
  }
  if (STATS) {
    __shared__ double scratch[NET_THREADS / 32];
    const double s1 = block_sum_d(d1 + (double)a1, scratch);
    const double s2 = block_sum_d(d2 + (double)a2, scratch);
    const int n = pc / a.C, c = pc - n * a.C, gc = a.C / a.G, ng = n * a.G + c / gc;
    const int S = gc * gridDim.x;
    double* pg = a.part + (size_t)ng * S * 2;
    const int slot = (c - (c / gc) * gc) * gridDim.x + blockIdx.x;
    if (threadIdx.x == 0) { pg[2 * slot] = s1; pg[2 * slot + 1] = s2; }
    if (arrive_last(a.counters + ng, S) && threadIdx.x < 32)
      finish_stats(pg, S, (long long)gc * a.P, a.stats_out + ng);
  }
}

// partial sums of g_u * x * gamma (aff + 1) over chunk blockIdx.x of plane blockIdx.y -> part[plane][chunk];
// the last CTA of a group turns its gc * chunks partials into coef_out[group] = G_r r^2 / ((cnt - 1) std)
__global__ void __launch_bounds__(NET_THREADS) k_gn_bwd_reduce(const float* __restrict__ gh,
                                                               const float* __restrict__ x,
                                                               const PlaneArgs a) {
  __shared__ double scratch[NET_THREADS / 32];
  const int pc = blockIdx.y, n = pc / a.C, c = pc - n * a.C;
  const int gc = a.C / a.G, g = c / gc, ng = n * a.G + g;
  const float2 st = a.stats[ng];
  const float r = 1.0f / (st.y + a.eps);
  const float q = a.gamma[c] * (a.aff[pc] + 1.0f), s = r * q;
  const float* xp = x + (size_t)pc * a.P;
  const float* gp = gh + (size_t)pc * a.P;
  const long long lo = NET_CHUNK * blockIdx.x, hi = min(a.P, lo + NET_CHUNK);
  float f = 0.f;                       // <= 16 values
  double acc = 0.0;                    // scalar paths
  if (((reinterpret_cast<uintptr_t>(xp) | reinterpret_cast<uintptr_t>(gp)) & 15) == 0) {
    float4 xv[4], gv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {      // all loads in flight before the first gelu'
      const long long i = lo + 4LL * (threadIdx.x + u * NET_THREADS);
      if (i + 3 < hi) {
        xv[u] = *reinterpret_cast<const float4*>(xp + i);
        gv[u] = *reinterpret_cast<const float4*>(gp + i);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = lo + 4LL * (threadIdx.x + u * NET_THREADS);
      if (i + 3 < hi) {
        f += (gv[u].x * gelu_grad_f(xv[u].x * s) * xv[u].x + gv[u].y * gelu_grad_f(xv[u].y * s) * xv[u].y) +
             (gv[u].z * gelu_grad_f(xv[u].z * s) * xv[u].z + gv[u].w * gelu_grad_f(xv[u].w * s) * xv[u].w);
      } else {
        for (long long j = i; j < hi; ++j) acc += (double)(gp[j] * gelu_grad_f(xp[j] * s) * xp[j]);
      }
    }
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += NET_THREADS)
      acc += (double)(gp[i] * gelu_grad_f(xp[i] * s) * xp[i]);
  }
  acc = block_sum_d(acc + (double)f, scratch);
  const int S2 = gridDim.x;
  double* pg = a.part + ((size_t)n * a.C + (size_t)g * gc) * S2;          // the group's gc * S2 partials
  if (threadIdx.x == 0) pg[(c - g * gc) * S2 + blockIdx.x] = acc * (double)q;
  if (arrive_last(a.counters + ng, gc * S2)) {
    double Gr = 0.0;
    for (int i = threadIdx.x; i < gc * S2; i += NET_THREADS) Gr += __ldcg(pg + i);
    Gr = block_sum_d(Gr, scratch);
    if (threadIdx.x == 0) {
      const long long cnt = (long long)gc * a.P;
      a.coef_out[ng] = (float)(Gr * (double)r * (double)r / ((double)(cnt - 1) * (double)st.y));
    }
  }
}

// g_x = g_y * scale + g_h gelu'(x s) s - coef (x - mean),  coef = G_r r^2 / ((cnt - 1) std);
// GV: also g_v of the preceding layer, gv_prev = g_x * gate_prev * scale (k_gate_residual's product)
template <bool GV>
__global__ void __launch_bounds__(NET_THREADS, 4) k_gn_bwd(const float* __restrict__ gh,
                                                        const float* __restrict__ x,
                                                        const float* __restrict__ gy,
                                                        float* __restrict__ gx, const PlaneArgs a) {
  const int pc = blockIdx.y, n = pc / a.C, c = pc - n * a.C;
  const int ng = n * a.G + c / (a.C / a.G);
  const float2 st = a.stats[ng];
  const float s = film_scale(a, pc, c, 1.0f / (st.y + a.eps));
  const float coef = a.coef[ng], mean = st.x, sc = a.scale;
  const float gs = GV ? a.gate_prev[pc] * a.scale : 0.f;
  const float* xp = x + (size_t)pc * a.P;
  const float* gp = gh + (size_t)pc * a.P;
  const float* yp = gy ? gy + (size_t)pc * a.P : nullptr;
  float* op = gx + (size_t)pc * a.P;
  float* vp = GV ? a.gv_prev + (size_t)pc * a.P : nullptr;
  const long long lo = NET_CHUNK * blockIdx.x, hi = min(a.P, lo + NET_CHUNK);
  auto f = [&](float xv, float gv, float yv) {
    return fmaf(gv * gelu_grad_f(xv * s), s, fmaf(-coef, xv - mean, yv * sc));
  };
  const bool vec = ((reinterpret_cast<uintptr_t>(xp) | reinterpret_cast<uintptr_t>(gp) |
                     reinterpret_cast<uintptr_t>(yp) | reinterpret_cast<uintptr_t>(op) |
                     reinterpret_cast<uintptr_t>(vp)) & 15) == 0;
  if (vec) {
    float4 xa[4], ga[4], ya[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {      // all loads in flight before the first gelu'
      const long long i = lo + 4LL * (threadIdx.x + u * NET_THREADS);
      ya[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i + 3 < hi) {
        xa[u] = *reinterpret_cast<const float4*>(xp + i);
        ga[u] = *reinterpret_cast<const float4*>(gp + i);
        if (yp) ya[u] = *reinterpret_cast<const float4*>(yp + i);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = lo + 4LL * (threadIdx.x + u * NET_THREADS);
      if (i + 3 < hi) {
        const float4 xv = xa[u], gv = ga[u], yv = ya[u];
        float4 o;
        o.x = f(xv.x, gv.x, yv.x); o.y = f(xv.y, gv.y, yv.y);
        o.z = f(xv.z, gv.z, yv.z); o.w = f(xv.w, gv.w, yv.w);
        *reinterpret_cast<float4*>(op + i) = o;
        if (GV) *reinterpret_cast<float4*>(vp + i) = make_float4(o.x * gs, o.y * gs, o.z * gs, o.w * gs);
      } else {
        for (long long j = i; j < hi; ++j) {
          const float o = f(xp[j], gp[j], yp ? yp[j] : 0.f);
          op[j] = o;
          if (GV) vp[j] = o * gs;
        }
      }
    }
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += NET_THREADS) {
      const float o = f(xp[i], gp[i], yp ? yp[i] : 0.f);
      op[i] = o;
      if (GV) vp[i] = o * gs;
    }
  }
}


// ---------------------------------------------------------------------------
// x2 anti-aliased time resampling of UpDownResample (networks/cqtdiff+.py:522-580, mode "T"):
// every (n, c, f) row is filtered independently by the L-tap kernel (the reference builds a dense
// diagonal C x C x L weight per call, :564-570), reflect padding fused, and the two adjoints.
//   down : xp = reflect_pad(x, pad),            y[t] = sum_k w[k] xp[2 t + k]          (T -> T/2)
//   up   : xp = reflect_pad(x, (pad + 1) / 2),  y[j] = sum_k w[k] xp[(j + 2 pad + 1 - k) / 2]
//          over the k of matching parity                                              (T -> 2 T)
// with pad = L/2 - 1.  All four kernels are gathers (deterministic).
// ---------------------------------------------------------------------------
template <int L>
struct Taps { float w[L]; };

__device__ __forceinline__ int reflect_idx(int i, int T) {
  if (i < 0) i = -i;
  if (i >= T) i = 2 * (T - 1) - i;
  return i;
}

// Interior threads of the 8-tap filter use aligned vector loads:
//   corr4  : out[m] = sum_k w[k] v[2 m + 1 + k],  v = in[2 o0 - 4 .. 2 o0 + 11]  4 outputs  (down, grad of up)
//   interp8: out[m] from u = in[o0/2 - 2 .. o0/2 + 5], 4 taps of alternating parity, 8 outputs (up, grad of down)
// (eight outputs of corr would need a 24-float window per thread and leave the short rows of the deep octaves
// to the reflecting path; measured slower).  A thread's outputs o0 .. o0 + OUT - 1 (o0 = OUT * segment) are
// addressed by a 2-D block: threadIdx.x is the segment within the row, threadIdx.y the row, so no thread
// divides to find its row.
constexpr int RS_OUT = 8;

template <int L>
__device__ __forceinline__ void corr4(const float* __restrict__ in, int o0, const Taps<L>& w, float (&o)[4]) {
  float v[16];
  const float4* p = reinterpret_cast<const float4*>(in + 2 * o0 - 4);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float4 q = p[i]; v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w; }
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) a = fmaf(w.w[k], v[2 * m + 1 + k], a);
    o[m] = a;
  }
}
template <int L>
__device__ __forceinline__ void interp8(const float* __restrict__ in, int o0, const Taps<L>& w, float (&o)[RS_OUT]) {
  float u[8];
  const float2* p = reinterpret_cast<const float2*>(in + o0 / 2 - 2);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 q = p[i]; u[2 * i] = q.x; u[2 * i + 1] = q.y; }
#pragma unroll
  for (int m = 0; m < RS_OUT; ++m) {      // even m: odd taps on u[3 + m/2 - kk]; odd m: even taps on u[4 + m/2 - kk]
    float a = 0.f;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
      a = (m & 1) ? fmaf(w.w[2 * kk], u[4 + m / 2 - kk], a) : fmaf(w.w[2 * kk + 1], u[3 + m / 2 - kk], a);
    o[m] = a;
  }
}
template <int OUT>
__device__ __forceinline__ void store_out(float* out, int o0, int n_out, const float (&o)[OUT], bool vec) {
  if (vec && o0 + OUT - 1 < n_out) {
#pragma unroll
    for (int m = 0; m < OUT; m += 4)
      *reinterpret_cast<float4*>(out + o0 + m) = make_float4(o[m], o[m + 1], o[m + 2], o[m + 3]);
  } else {
#pragma unroll
    for (int m = 0; m < OUT; ++m)
      if (o0 + m < n_out) out[o0 + m] = o[m];
  }
}
__device__ __forceinline__ bool aligned16(const void* a, const void* b) {
  return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0;
}
// row and first output of this thread; false past the last row or the row's last output
template <int OUT>
__device__ __forceinline__ bool rs_thread(long long rows, int n_out, long long& row, int& o0) {
  row = (long long)blockIdx.x * blockDim.y + threadIdx.y;
  o0 = OUT * (int)(blockIdx.y * blockDim.x + threadIdx.x);
  return row < rows && o0 < n_out;
}

template <int L>
__global__ void __launch_bounds__(NET_THREADS) k_resample_down(const float* __restrict__ x,
                                                               float* __restrict__ y, int T, int To,
                                                               const Taps<L> w, long long rows) {
  constexpr int PAD = L / 2 - 1;
  long long row;
  int t0;
  if (!rs_thread<4>(rows, To, row, t0)) return;
  const float* xr = x + (size_t)row * T;
  float* yr = y + (size_t)row * To;
  const bool vec = aligned16(xr, yr);
  float o[4];
  if (L == 8 && vec && t0 >= 2 && 2 * t0 + 11 < T) {
    corr4<L>(xr, t0, w, o);
  } else {
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      float acc = 0.f;
      const int q0 = 2 * (t0 + m) - PAD;
      if (t0 + m < To) {
#pragma unroll
        for (int k = 0; k < L; ++k) acc = fmaf(w.w[k], xr[reflect_idx(q0 + k, T)], acc);
      }
      o[m] = acc;
    }
  }
  store_out<4>(yr, t0, To, o, vec);
}

template <int L>
__global__ void __launch_bounds__(NET_THREADS) k_resample_up(const float* __restrict__ x,
                                                             float* __restrict__ y, int T,
                                                             const Taps<L> w, long long rows) {
  constexpr int PAD = L / 2 - 1, PU = (PAD + 1) / 2;
  long long row;
  int j0;
  if (!rs_thread<RS_OUT>(rows, 2 * T, row, j0)) return;
  const float* xr = x + (size_t)row * T;
  float* yr = y + (size_t)row * 2 * T;
  const bool vec = aligned16(xr, yr);
  float o[RS_OUT];
  if (L == 8 && vec && j0 >= 4 && j0 / 2 + 5 < T) {
    interp8<L>(xr, j0, w, o);
  } else {
#pragma unroll
    for (int m = 0; m < RS_OUT; ++m) {
      const int j = j0 + m;
      float acc = 0.f;
      const int par = (j + 2 * PAD + 1) & 1;
      if (j < 2 * T) {
#pragma unroll
        for (int kk = 0; kk < L / 2; ++kk) {
          // k = par + 2 kk (same parity as j + 2 pad + 1); L/2 taps per output
          const int i = (j + 2 * PAD + 1 - par) / 2 - kk;             // index into the padded row
          const float wk = par ? w.w[2 * kk + 1] : w.w[2 * kk];
          acc = fmaf(wk, xr[reflect_idx(i - PU, T)], acc);
        }
      }
      o[m] = acc;
    }
  }
  store_out<RS_OUT>(yr, j0, 2 * T, o, vec);
}

// gradient of `down` wrt x: gy[To] -> gx[T]
template <int L>
__global__ void __launch_bounds__(NET_THREADS) k_resample_down_adj(const float* __restrict__ gy,
                                                                   float* __restrict__ gx, int T, int To,
                                                                   const Taps<L> w, long long rows) {
  constexpr int PAD = L / 2 - 1;
  long long row;
  int i0;
  if (!rs_thread<RS_OUT>(rows, T, row, i0)) return;
  const float* gr = gy + (size_t)row * To;
  float* xr = gx + (size_t)row * T;
  const bool vec = aligned16(gr, xr);
  float o[RS_OUT];
  if (L == 8 && vec && i0 >= 4 && i0 + 12 <= T) {
    interp8<L>(gr, i0, w, o);
  } else {
    // padded-row gradient at q: sum over (t, k) with 2 t + k = q
    auto gxp = [&](int q) {
      float a = 0.f;
#pragma unroll
      for (int kk = 0; kk < L / 2; ++kk) {
        const int k = (q & 1) + 2 * kk, t = (q - k) / 2;
        const float wk = (q & 1) ? w.w[2 * kk + 1] : w.w[2 * kk];
        if (t >= 0 && t < To && q - k >= 0) a = fmaf(wk, gr[t], a);
      }
      return a;
    };
#pragma unroll
    for (int m = 0; m < RS_OUT; ++m) {
      const int i = i0 + m;
      float acc = 0.f;
      if (i < T) {
        acc = gxp(i + PAD);
        if (i >= 1 && i <= PAD) acc += gxp(PAD - i);                        // left reflection
        if (i <= T - 2 && i >= T - 1 - PAD) acc += gxp(2 * (T - 1) - i + PAD);   // right reflection
      }
      o[m] = acc;
    }
  }
  store_out<RS_OUT>(xr, i0, T, o, vec);
}

// gradient of `up` wrt x: gy[2T] -> gx[T]
template <int L>
__global__ void __launch_bounds__(NET_THREADS) k_resample_up_adj(const float* __restrict__ gy,
                                                                 float* __restrict__ gx, int T,
                                                                 const Taps<L> w, long long rows) {
  constexpr int PAD = L / 2 - 1, PU = (PAD + 1) / 2;
  long long row;
  int i0;
  if (!rs_thread<4>(rows, T, row, i0)) return;
  const float* gr = gy + (size_t)row * 2 * T;
  float* xr = gx + (size_t)row * T;
  const bool vec = aligned16(gr, xr);
  float o[4];
  if (L == 8 && vec && i0 >= 4 && i0 + 8 <= T) {
    corr4<L>(gr, i0, w, o);
  } else {
    // padded-row gradient at q: sum_k w[k] gy[2 q + k - (2 pad + 1)]
    auto gxp = [&](int q) {
      float a = 0.f;
      const int j0 = 2 * q - (2 * PAD + 1);
#pragma unroll
      for (int k = 0; k < L; ++k) {
        const int j = j0 + k;
        if (j >= 0 && j < 2 * T) a = fmaf(w.w[k], gr[j], a);
      }
      return a;
    };
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const int i = i0 + m;
      float acc = 0.f;
      if (i < T) {
        acc = gxp(i + PU);
        if (i >= 1 && i <= PU) acc += gxp(PU - i);
        if (i <= T - 2 && i >= T - 1 - PU) acc += gxp(2 * (T - 1) - i + PU);
      }
      o[m] = acc;
    }
  }
  store_out<4>(xr, i0, T, o, vec);
}

template <int L>
static int launch_resample(const float* x, float* y, long long rows, int T, int mode, const float* taps,
                           cudaStream_t st) {
  Taps<L> w;
  for (int k = 0; k < L; ++k) w.w[k] = taps[k];
  const int To = T / 2;
  const int n_out = mode == 0 ? To : (mode == 1 ? 2 * T : T);
  const int out = (mode == 1 || mode == 2) ? RS_OUT : 4;           // outputs per thread
  const int per = (n_out + out - 1) / out;                          // threads per row
  int tx = 1;
  while (tx < per && tx < NET_THREADS) tx *= 2;
  const dim3 block(tx, NET_THREADS / tx);
  const long long gx = (rows + block.y - 1) / block.y;
  const unsigned gy = (unsigned)((per + tx - 1) / tx);
  BABE_REQUIRE(gx < (1LL << 31) && gy <= 65535, BABE_EUNSUPPORTED, "resample2: %lld rows of %d", rows, T);
  const dim3 grid((unsigned)gx, gy);
  switch (mode) {
    case 0: k_resample_down<L><<<grid, block, 0, st>>>(x, y, T, To, w, rows); break;
    case 1: k_resample_up<L><<<grid, block, 0, st>>>(x, y, T, w, rows); break;
    case 2: k_resample_down_adj<L><<<grid, block, 0, st>>>(x, y, T, To, w, rows); break;
    default: k_resample_up_adj<L><<<grid, block, 0, st>>>(x, y, T, w, rows); break;
  }
  return check_launch("k_resample");
}

static int check_dims(int N, int C, int G, long long P, const char* what) {
  BABE_REQUIRE(N >= 1 && C >= 1 && G >= 1 && P >= 1 && C % G == 0, BABE_EBADARG,
               "%s: bad shape N=%d C=%d G=%d P=%lld", what, N, C, G, P);
  BABE_REQUIRE((long long)N * C <= 65535, BABE_EUNSUPPORTED, "%s: N*C = %lld exceeds 65535", what,
               (long long)N * C);
  return BABE_OK;
}
static inline unsigned chunks_of(long long P) { return (unsigned)((P + NET_CHUNK - 1) / NET_CHUNK); }

}  // namespace babe

using namespace babe;

extern "C" int babe_gn_slices(int N, int C, int G, long long P) {
  if (N < 1 || C < 1 || G < 1 || P < 1 || C % G) return 0;
  const long long cnt = (long long)(C / G) * P;
  long long s = (16LL * sm_count() + (long long)N * G - 1) / ((long long)N * G);
  s = std::min<long long>(s, (cnt + 8191) / 8192);
  return (int)std::max<long long>(1, std::min<long long>(s, MAX_STAT_SLICES));
}

extern "C" int babe_net_chunks(long long P) {
  return P < 1 ? 0 : (int)chunks_of(P);
}

extern "C" int babe_gn_stats(const float* x, double* part, float* stats, unsigned* counters, int N, int C, int G,
                             long long P, int slices, void* stream) {
  int rc = check_dims(N, C, G, P, "gn_stats");
  if (rc) return rc;
  BABE_REQUIRE(x && part && stats && counters && slices >= 1 && slices <= MAX_STAT_SLICES, BABE_EBADARG,
               "gn_stats: bad arguments");
  k_gn_stats<<<dim3(slices, N * G), NET_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      x, part, reinterpret_cast<float2*>(stats), counters, (long long)(C / G) * P, slices);
  return check_launch("k_gn_stats");
}

extern "C" int babe_gn_film_gelu(const float* x, float* h, const float* stats, const float* gamma,
                                 const float* aff, int N, int C, int G, long long P, float eps, void* stream) {
  int rc = check_dims(N, C, G, P, "gn_film_gelu");
  if (rc) return rc;
  BABE_REQUIRE(x && h && stats && gamma && aff, BABE_EBADARG, "gn_film_gelu: bad arguments");
  PlaneArgs a{};
  a.N = N; a.C = C; a.G = G; a.P = P; a.eps = eps; a.gamma = gamma; a.aff = aff;
  a.stats = reinterpret_cast<const float2*>(stats);
  k_gn_film_gelu<<<dim3(chunks_of(P), N * C), NET_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(x, h, a);
  return check_launch("k_gn_film_gelu");
}

extern "C" int babe_gate_residual(const float* x0, const float* v, const float* gate, float* out,
                                  int N, int C, long long P, float scale, void* stream) {
  int rc = check_dims(N, C, 1, P, "gate_residual");
  if (rc) return rc;
  BABE_REQUIRE(v && out, BABE_EBADARG, "gate_residual: bad arguments");
  PlaneArgs a{};
  a.N = N; a.C = C; a.G = 1; a.P = P; a.scale = scale; a.gate = gate;
  k_gate_residual<false><<<dim3(chunks_of(P), N * C), NET_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      x0, v, out, a);
  return check_launch("k_gate_residual");
}

extern "C" int babe_gate_residual_stats(const float* x0, const float* v, const float* gate, float* out,
                                        double* part, float* stats, unsigned* counters, int N, int C, int G,
                                        long long P, float scale, void* stream) {
  int rc = check_dims(N, C, G, P, "gate_residual_stats");
  if (rc) return rc;
  BABE_REQUIRE(v && out && part && stats && counters, BABE_EBADARG, "gate_residual_stats: bad arguments");
  PlaneArgs a{};
  a.N = N; a.C = C; a.G = G; a.P = P; a.scale = scale; a.gate = gate;
  a.part = part; a.stats_out = reinterpret_cast<float2*>(stats); a.counters = counters;
  k_gate_residual<true><<<dim3(chunks_of(P), N * C), NET_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      x0, v, out, a);
  return check_launch("k_gate_residual");
}

extern "C" int babe_gn_film_gelu_bwd_reduce(const float* gh, const float* x, const float* stats, double* gr_part,
                                            float* coef, unsigned* counters, const float* gamma, const float* aff,
                                            int N, int C, int G, long long P, float eps, void* stream) {
  int rc = check_dims(N, C, G, P, "gn_film_gelu_bwd_reduce");
  if (rc) return rc;
  BABE_REQUIRE(gh && x && stats && gr_part && coef && counters && gamma && aff, BABE_EBADARG,
               "gn_film_gelu_bwd_reduce: bad arguments");
  PlaneArgs a{};
  a.N = N; a.C = C; a.G = G; a.P = P; a.eps = eps; a.gamma = gamma; a.aff = aff;
  a.stats = reinterpret_cast<const float2*>(stats);
  a.part = gr_part; a.coef_out = coef; a.counters = counters;
  k_gn_bwd_reduce<<<dim3(chunks_of(P), N * C), NET_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(gh, x, a);
  return check_launch("k_gn_bwd_reduce");
}

extern "C" int babe_gn_film_gelu_bwd(const float* gh, const float* x, const float* gy, float* gx,
                                     const float* stats, const float* coef, const float* gamma, const float* aff,
                                     const float* gate_prev, float* gv_prev, int N, int C, int G, long long P,
                                     float eps, float res_scale, void* stream) {
  int rc = check_dims(N, C, G, P, "gn_film_gelu_bwd");
  if (rc) return rc;
  BABE_REQUIRE(gh && x && gx && stats && coef && gamma && aff && (gate_prev == nullptr) == (gv_prev == nullptr),
               BABE_EBADARG, "gn_film_gelu_bwd: bad arguments");
  PlaneArgs a{};
  a.N = N; a.C = C; a.G = G; a.P = P; a.eps = eps; a.scale = res_scale;
  a.stats = reinterpret_cast<const float2*>(stats); a.coef = coef; a.gamma = gamma; a.aff = aff;
  a.gate_prev = gate_prev; a.gv_prev = gv_prev;
  const dim3 grid(chunks_of(P), N * C);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (gv_prev) k_gn_bwd<true><<<grid, NET_THREADS, 0, st>>>(gh, x, gy, gx, a);
  else k_gn_bwd<false><<<grid, NET_THREADS, 0, st>>>(gh, x, gy, gx, a);
  return check_launch("k_gn_bwd");
}

extern "C" int babe_resample2(const float* in, float* out, long long rows, int T, int mode,
                              const float* taps_host, int L, void* stream) {
  BABE_REQUIRE(in && out && taps_host && rows >= 1, BABE_EBADARG, "resample2: bad arguments");
  BABE_REQUIRE(mode >= 0 && mode <= 3, BABE_EBADARG, "resample2: mode %d", mode);
  BABE_REQUIRE(T >= L && T % 2 == 0, BABE_EUNSUPPORTED, "resample2: row length %d (even, >= %d)", T, L);
  BABE_REQUIRE(rows * (long long)T < (1LL << 31), BABE_EUNSUPPORTED, "resample2: more than 2^31 samples");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  switch (L) {
    case 4: rc = launch_resample<4>(in, out, rows, T, mode, taps_host, st); break;
    case 8: rc = launch_resample<8>(in, out, rows, T, mode, taps_host, st); break;
    case 12: rc = launch_resample<12>(in, out, rows, T, mode, taps_host, st); break;
    default: BABE_REQUIRE(false, BABE_EUNSUPPORTED, "resample2: %d taps (4, 8 or 12)", L);
  }
  return rc;
}
