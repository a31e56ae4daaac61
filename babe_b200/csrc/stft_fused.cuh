// Interface between stft_ops.cu (C-ABI entry points, generic kernels) and stft_fused.cu (second-generation
// NFFT-4096 kernels: TMA-staged frame tiles, Core4k transform).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace babe {

struct FusedArgs {
  const float* x; float* y; int B, T;
  const float* window; const float2* roots;            // periodic Hamming window (N), exp(-2 pi i m / N)
  // H: shared filter (NULL: designed from fc, A).  known (per_row only, NULL = none): int[B] known-prefix lengths of
  // the masked operator.  The per-row kernels never read H; sharing its slot keeps the parameter block at 128 bytes
  // (a larger block changes the code ptxas generates for every existing instantiation).
  union { const float* H; const int* known; };
  const float* freqs; const float* fc; const float* A; int K;
  int adjoint;
  const float* sub; const float* row_scale; double* item_sumsq;
  int* status;
  int q, nblk, frames;                                  // filled by the launcher (q: output blocks per CTA)
  int per_row;                                          // 1: fc, A are [B, K], status is int[B] (one filter per row)
};

// rows can be bulk-copied: T % 4 == 0 and a 16-byte aligned base
bool fused_filter_eligible(const float* x, const float* sub, int T);
size_t fused_sumsq_slots(int B, int T);                 // doubles of workspace the residual sum of squares needs
int launch_filter_fused(FusedArgs a, double* row_sumsq, cudaStream_t st);

struct FusedStatsArgs {
  const float* x; const float* y; int B, T;
  const float* window; const float2* roots;
  float* partial;                                       // [CTAs][3][F]
  int q, frames;                                        // filled by the launcher (q: frames per CTA)
  // per-row statistics only: DEVICE int[G + 1] group offsets 0 = o_0 < ... < o_G = B (group g is rows
  // [o_g, o_{g+1})); NULL: every row is its own group (G = B)
  const int* offsets; int G;
};
bool fused_stats_eligible(const float* x, const float* y, int T, int mode);
// launches k_stats_fused; *n_partials = rows of `partial` written (<= 2 * SM count)
int launch_stats_fused(FusedStatsArgs a, int* n_partials, cudaStream_t st);
// per-row (offsets NULL) or per-group statistics: abc[G][3][F]; `partial` needs fused_stats_rows_slots(B, T) rows of
// 3 F floats
size_t fused_stats_rows_slots(int B, int T);
int launch_stats_rows_fused(FusedStatsArgs a, double* abc, cudaStream_t st);

struct FusedFirArgs {
  const float* x; float* y; int B, T;
  const float2* roots; const float2* G;                 // G[N] = conj(FFT(taps zero padded)) / N, natural bin order
  int L, pl, V, pairs_per_row;
  int q;                                                // filled by the launcher (block pairs per CTA)
};
bool fused_fir_eligible(const float* x, int T);
int launch_fir_fused(FusedFirArgs a, cudaStream_t st);

}  // namespace babe
