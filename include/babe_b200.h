/* babe_b200 -- C ABI of the B200-native blind-BWE signal-processing hot path.
 *
 * The reference (eloimoliner/BABE) is pure Python/PyTorch and has no FFI; its
 * plug-in points are Python module functions (utils/blind_bwe_utils.py) and
 * the external class cqt_nsgt_pytorch.CQT_nsgt.  This header is the boundary
 * *beneath* those seams: the Python drop-ins in babe_b200/ bind exactly these
 * symbols with ctypes, and any other host (C, C++, cgo, JNI) can do the same
 * -- see INTEGRATION.md for the reference-side stubs.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host;
 *    the library never allocates, frees or retains caller memory;
 *  - float32 data, row-major, contiguous; `stream` is a cudaStream_t passed as
 *    void* (NULL = legacy default stream); calls are asynchronous;
 *  - return 0 on success, BABE_EBADARG (-1) for an invalid shape/argument,
 *    BABE_EUNSUPPORTED (-2) for an unsupported transform length,
 *    BABE_ECUDA (-3) for a CUDA error; babe_last_error() gives the message
 *    (thread-local);
 *  - thread-safe for distinct streams.
 */
#ifndef BABE_B200_H
#define BABE_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BABE_OK 0
#define BABE_EBADARG (-1)
#define BABE_EUNSUPPORTED (-2)
#define BABE_ECUDA (-3)

#define BABE_MAX_BREAKPOINTS 16

const char* babe_last_error(void);
int babe_version(void);
/* number of SMs of the current device (grid sizing), <0 on error */
int babe_sm_count(void);

/* ---- STFT tables ------------------------------------------------------- */
/* Supported NFFT: 512, 1024, 2048, 4096 (reference configs use 4096,
 * 1024 and 2048: conf/tester/*.yaml). Returns 1/0. */
int babe_stft_supported(int nfft);
/* Fills HOST arrays: window_host[nfft] = periodic Hamming window
 * (utils/blind_bwe_utils.py:19), twiddle_host[2*nfft] = interleaved (re,im) of
 * the nfft-th roots of unity exp(-2*pi*i*m/nfft), m < nfft.
 * The caller uploads them once per NFFT and passes the device copies below. */
int babe_stft_tables_host(int nfft, float* window_host, float* twiddle_host);

/* ---- a4/a5: filter design --------------------------------------------- */
/* Replaces design_filter / design_filter_G (utils/blind_bwe_utils.py:82-119,
 * :41-80).  fc[K], A[K] breakpoints, freqs[F] bin frequencies, gain_db
 * optional 1-element device array (NULL = no gain).  status (optional int*)
 * is set non-zero when some fc_i (i>=1) lies above freqs[F-1], the case in
 * which the reference raises IndexError. */
int babe_design_filter(const float* fc, const float* A, int K, const float* gain_db,
                       const float* freqs, int F, float* H, int* status, void* stream);
/* Vector-Jacobian product of the above: given gH[F] = dL/dH returns
 * gfc[K], gA[K] and (optional) ggain[1]. Replaces the autograd backward the
 * reference runs at testing/blind_bwe_sampler.py:566. */
int babe_design_filter_vjp(const float* fc, const float* A, int K, const float* gain_db,
                           const float* freqs, int F, const float* gH,
                           float* gfc, float* gA, float* ggain, void* stream);

/* ---- kernel selection (profiling / A-B measurements; not needed for normal use) ----------- */
/* Which implementation serves NFFT = 4096 in babe_apply_filter / babe_stft_stats / babe_fir_filter:
 *    0 (default)  second-generation kernels (csrc/stft_fused.cu): frame tiles staged by 1-D bulk TMA copies
 *                 (cp.async.bulk + mbarrier), the batch cut into equal contiguous runs of output blocks;
 *   -1            the round-1 kernels (cp.async staging), which also serve rows that cannot be bulk-copied
 *                 (length not a multiple of 4 samples, misaligned base).
 * Process-wide, not thread-safe against concurrent launches. */
int babe_set_fused_variant(int variant);
int babe_get_fused_variant(void);
/* Which implementation computes the length-Ls real FFT / inverse of the CQT calls (babe_rfft, babe_irfft,
 * babe_spectral_filter, babe_cqt_analysis, babe_cqt_synthesis):
 *    2 (default)  prime-factor passes (csrc/cqt_pfa.cuh) for the instantiated lengths (Ls = 184184, 368368):
 *                 twiddle-free in-place stages, r2c / c2r / filter / synthesis gather fused into pass 2
 *                 (2 launches per transform, 3 for the spectral filter); other lengths run variant -1;
 *    0, 1         round 2's tiled passes (csrc/cqt_fft.cuh), 16 / 8 sequences per CTA -- slower, kept for A/B;
 *   -1            the round-1 generic mixed-radix passes with separate post / pre / gather kernels. */
int babe_set_cqt_variant(int variant);
int babe_get_cqt_variant(void);
/* Band kernels of babe_cqt_analysis / babe_cqt_synthesis: 1 (default) packed register FFTs with per-band
 * synchronisation for every octave size 32 ... 4096 (csrc/bandfft_v.cuh); the analysis stages each band's window slice
 * of the spectrum with one TMA bulk copy per row, the synthesis its coefficient rows with cp.async (faster at the
 * sampler's batch and planar layout); 2: cp.async staging for both (also serves misaligned inputs); 3: TMA staging
 * for both; 0: round 2's cores (A/B). */
int babe_set_cqt_band_variant(int variant);
/* Programmatic dependent launch of the kernels of a CQT call: each kernel lets its successor start while its own last
 * wave runs and waits (griddepcontrol.wait) only before it touches the chain's buffers.  Bit mask of the kernels
 * launched that way: 1 pass-1 kernels, 2 pass-2 kernels, 4 band kernels, 8 the gathering inverse pass 2 behind the
 * synthesis band kernel; default 15, 0 = plain stream-ordered launches (A/B). */
int babe_set_cqt_pdl(int mask);

/* ---- a3/a12: fused STFT -> H -> iSTFT ---------------------------------- */
/* Replaces apply_filter (utils/blind_bwe_utils.py:6-13) and
 * BlindSampler.apply_filter_fcA (testing/blind_bwe_sampler.py:518-520).
 *   x[B,T] -> y[B,T].
 * The filter is either H[F] (H != NULL) or designed on the fly from
 * (freqs, fc, A, K) so that H never exists in HBM.
 * adjoint != 0 computes the transpose wrt x (the autograd backward the
 * reference runs at testing/blind_bwe_sampler.py:120).
 * Optional epilogues (any may be NULL):
 *   sub[B,T]       y <- y - sub                       (forward only)
 *   row_scale[B]   y <- y * row_scale[b]
 *   row_sumsq[B]   row_sumsq[b] += sum_t y[b,t]^2     (double, caller zeroes;
 *                  summed in a fixed order -> bitwise reproducible; needs a
 *                  workspace of babe_apply_filter_workspace() bytes)
 */
size_t babe_apply_filter_workspace(int B, int T, int nfft);
int babe_apply_filter(const float* x, float* y, int B, int T, int nfft,
                      const float* window, const float* twiddle,
                      const float* H, const float* freqs, const float* fc, const float* A, int K,
                      int adjoint, const float* sub, const float* row_scale, double* row_sumsq,
                      void* workspace, size_t workspace_bytes, int* status, void* stream);

/* One filter per row: the same operator with fc[B,K], A[B,K] (row b filtered by the H designed from
 * fc[b], A[b]) and status int[B] (status[b] set like babe_design_filter's for row b).  Epilogues and workspace
 * as above.  Every row's output equals babe_apply_filter on that row alone with its own (fc, A).  NFFT 4096 rows
 * that can be bulk-copied run the per-row variant of the fused kernel (H redesigned where a CTA's run of blocks
 * enters a new row); NFFT 512 / 1024 / 2048, other rows and babe_set_fused_variant(-1) call babe_apply_filter
 * once per row. */
int babe_apply_filter_rows(const float* x, float* y, int B, int T, int nfft,
                           const float* window, const float* twiddle,
                           const float* freqs, const float* fc, const float* A, int K,
                           int adjoint, const float* sub, const float* row_scale, double* row_sumsq,
                           void* workspace, size_t workspace_bytes, int* status, void* stream);

/* ---- a1: STFT, a2: filter + iSTFT (unfused signatures) ------------------ */
/* apply_stft (utils/blind_bwe_utils.py:15-26): x[B,T] -> X[B,F,frames,2].
 * frames = 0 means the reference's 1 + T/(nfft/2) (x is treated as right
 * padded with nfft zeros); an explicit smaller count frames the first
 * nfft + (nfft/2)(frames-1) samples only.  in_env_div: divide the input by
 * the overlap-add envelope of `frames` frames first; bin_scale[F] optional
 * per-bin real factor (both are used by the backward of babe_istft). */
int babe_stft(const float* x, float* X, int B, int T, int nfft, int frames,
              const float* window, const float* twiddle,
              int in_env_div, const float* bin_scale, void* stream);
/* apply_filter_istft (utils/blind_bwe_utils.py:28-39): X[B,F,frames,2], H[F]
 * (NULL = 1) -> y[B,out_len], out_len <= nfft + (nfft/2)(frames-1).
 * out_env_div=1 reproduces torch.istft; 0 with bin_scale = N*c_k gives the
 * adjoint of babe_stft. */
int babe_istft(const float* X, float* y, int B, int frames, int nfft, int out_len,
               const float* window, const float* twiddle,
               const float* bin_scale, int out_env_div, void* stream);

/* ---- classical FIR observation model (SURVEY 8f-4) ------------------------- */
/* Replaces apply_low_pass_firwin (utils/bandwidth_extension.py:76-95) and
 * BlindSampler.apply_FIR_filter (testing/blind_bwe_sampler.py:211-218):
 * torch conv1d(padding="same") with L taps, y[n] = sum_k b[k] x[n + k - pad_left],
 * by overlap-save on the 4096-point transform.  G[4096] (device float2) =
 * conj(FFT_4096(b zero padded)) / 4096; twiddle = the 4096-th roots of
 * babe_stft_tables_host(4096).  The adjoint wrt x is the same call with the
 * reversed taps and pad_left' = L - 1 - pad_left.  L <= 2049. */
int babe_fir_filter(const float* x, float* y, int B, int T, const float* twiddle, const float* G,
                    int L, int pad_left, void* stream);

/* ---- fit statistics (a6 collapsed; SURVEY Appendix A.3) ------------------ */
/* mode 0: abc[0..F) = sum|X|^2, abc[F..2F) = sum|X||Y|, abc[2F..3F) = sum|Y|^2
 *         over batch and frames, X = STFT(x), Y = STFT(y);
 * mode 1: abc[0..F) = sum Re(conj(X) G), G = STFT(y / envelope)  (dL/dH of
 *         apply_filter up to the rfft weights), the rest is zero.
 * abc is double[3F].  workspace: babe_stft_stats_workspace() bytes. */
size_t babe_stft_stats_workspace(int B, int T, int nfft);
int babe_stft_stats(const float* x, const float* y, int B, int T, int nfft,
                    const float* window, const float* twiddle, int mode,
                    double* abc, void* workspace, size_t workspace_bytes, void* stream);
/* Mode-0 statistics per row: abc is double[B,3F], row b's block is what babe_stft_stats gives for row b
 * alone.  NFFT 4096 rows that can be bulk-copied: one launch of the fused statistics kernel with one partial
 * per (CTA, row) segment and a fixed-order fp64 reduction per row (deterministic; a row's result does not
 * depend on the other rows); otherwise babe_stft_stats once per row.  workspace:
 * babe_stft_stats_rows_workspace() bytes. */
size_t babe_stft_stats_rows_workspace(int B, int T, int nfft);
int babe_stft_stats_rows(const float* x, const float* y, int B, int T, int nfft,
                         const float* window, const float* twiddle,
                         double* abc, void* workspace, size_t workspace_bytes, void* stream);
/* Same statistics from precomputed spectrograms X, Xref [B,F,frames,2] as the
 * reference signature apply_filter_and_norm_STFTmag_fweighted(X, Xref, H, w)
 * (utils/blind_bwe_utils.py:250-296) receives them.  out is double[4F]:
 * a, b, c and s_k = sum_{b,t} (w_k (H_k |X| - |Xref|))^2 (H, w may be NULL = 1). */
int babe_spec_mag_stats(const float* X, const float* Xref, const float* H, const float* w,
                        int B, int F, int frames, double* out, void* stream);
/* Gradient of that norm wrt the spectrograms (what autograd gives the reference when X or Xref require grad):
 * gX = coef w^2 (H|X| - |Xref|) H X/|X|, gXref = -coef w^2 (H|X| - |Xref|) Xref/|Xref|; coef is a 1-element
 * DEVICE array holding (upstream gradient / norm); either output may be NULL. */
int babe_spec_mag_grad(const float* X, const float* Xref, const float* H, const float* w, const float* coef,
                       int B, int F, int frames, float* gX, float* gXref, void* stream);

/* a9 / a10: the STFT-distance guidance norms apply_norm_STFT_fweighted (utils/blind_bwe_utils.py:148-197, mode 0:
 * || w X - w Xref ||_2 over re/im) and apply_norm_STFTmag_fweighted(..., logmag=True) (:198-248, mode 2:
 * || log10(w|X| + 1e-8) - log10(w|Xref| + 1e-8) ||_2) from spectrograms [B,F,frames,2]; out is double[F], the per-bin
 * sums of squares (norm = sqrt of their sum).  The plain magnitude distance (:198-248, logmag=False) is
 * babe_spec_mag_stats with H = NULL.  w may be NULL (= 1).  mode 3: out[k] = sum_{b,t} Re(conj(X) Xref) (w unused),
 * the gradient of apply_filter_istft (utils/blind_bwe_utils.py:28-39) wrt H when Xref is the adjoint spectrogram. */
int babe_spec_dist_stats(const float* X, const float* Xref, const float* w, int mode, int B, int F, int frames,
                         double* out, void* stream);
/* Gradients of those norms wrt the spectrograms; coef is a 1-element DEVICE array (upstream gradient / norm);
 * either output may be NULL. */
int babe_spec_dist_grad(const float* X, const float* Xref, const float* w, const float* coef, int mode, int B, int F,
                        int frames, float* gX, float* gXref, void* stream);

/* ---- a7: device-resident filter fit ------------------------------------ */
/* Replaces the Python loop of BlindSampler.fit_params
 * (testing/blind_bwe_sampler.py:562-590): projected gradient descent on
 * params[2,K] (row 0 = fc, row 1 = A; updated IN PLACE like the reference)
 * with the loss sqrt(sum_k w_k^2 (H_k^2 a_k - 2 H_k b_k + c_k)).
 * iters_out (optional int*) receives the number of iterations run. */
typedef struct {
  float mu_fc, mu_A;       /* step sizes, optimization.mu             */
  float fcmin, fcmax;      /* blind_bwe.fcmin, sample_rate//2          */
  float Amin, Amax;        /* blind_bwe.Amin / Amax                    */
  float tol_fc, tol_A;     /* optimization.tol                         */
  int max_iter;            /* optimization.max_iter                    */
  int clamp_fc, clamp_A, only_negative_A;
} babe_fit_config;
/* Which kernel runs the loop: 0 (default) k_fit_params3, a cluster of 4 CTAs (each evaluates a quarter of the bins,
 * sums gathered through distributed shared memory, one serial warp); 1 k_fit_params2 (one CTA); -1 round 1's
 * k_fit_params.  babe_set_fused_variant(-1 / 0) sets it too. */
int babe_set_fit_variant(int variant);
int babe_fit_params(const double* abc, const float* w, const float* freqs, int F,
                    float* params, int K, const babe_fit_config* cfg_host,
                    int* iters_out, void* stream);
/* B independent fits: abc[B,3F] (babe_stft_stats_rows), params[B,2,K] updated in place, iters_out int[B]
 * (optional); clamps and the stopping test apply per row.  Row b's result is bitwise what babe_fit_params gives
 * on abc[b], params[b].  Fit variant 0 with K <= 8 and F <= 4096 launches B clusters of k_fit_params3 (cluster b
 * fits row b); the other variants and sizes call babe_fit_params once per row. */
int babe_fit_params_rows(const double* abc, const float* w, const float* freqs, int F,
                         float* params, int B, int K, const babe_fit_config* cfg_host,
                         int* iters_out, void* stream);

/* ---- a15-a18: NSGT constant-Q transform (cqt_nsgt_pytorch.CQT_nsgt) -------- */
/* Replaces the third-party class the reference imports at
 * networks/cqtdiff+.py:9 and calls at :620 (ctor), :743 (fwd), :841 (bwd) and
 * testing/blind_bwe_sampler.py:156 (apply_hpf_DC).  The plan is a plain
 * struct filled by the host (babe_b200/cqt.py builds it; any host may): the
 * length-Ls real FFT is done as a complex FFT of Nc = Ls/2 = n1*n2 points in
 * two shared-memory passes (four-step), every factor of n1, n2 and of the
 * octave sizes must be in {2,3,4,5,7,8,11,13,16,17,19,23}. */
#define BABE_MAX_FACTORS 12
#define BABE_MAX_OCTAVES 16
typedef struct {
  int n;                       /* transform length                       */
  int nf;                      /* number of stages                       */
  int radix[BABE_MAX_FACTORS]; /* product == n                           */
} babe_fft_factors;

typedef struct {
  int Ls, Nc;                  /* signal length (even), Nc = Ls/2        */
  babe_fft_factors f1, f2;     /* column pass (n1) and row pass (n2)     */
  const float* roots1;         /* device float2[n1]  exp(-2 pi i m/n1)   */
  const float* roots2;         /* device float2[n2]                      */
  const float* tw_nc;          /* device float2[1024 + Nc/1024 + 1]: exp(-2 pi i m/Nc), m<1024,
                                  then exp(-2 pi i 1024 m/Nc)            */
  const float* tw_ls;          /* same two-level table for Ls            */
  /* constant-Q bands (DC and Nyquist bands excluded) */
  int numocts, binsoct;
  int M[BABE_MAX_OCTAVES];     /* coefficients per band in octave o      */
  babe_fft_factors fm[BABE_MAX_OCTAVES];
  const float* rootsm[BABE_MAX_OCTAVES]; /* device float2[M_o]           */
  const int* band_p;           /* device int[nbands]: centre bin         */
  const int* band_lg;          /* device int[nbands]: window length      */
  const int* band_off;         /* device int[nbands]: offset into window tables */
  int sum_lg;                  /* total window samples                   */
  const int* bin_jlo;          /* device int[Nc+1]: first band covering bin k */
  const int* bin_jhi;          /* device int[Nc+1]: last band covering bin k (jhi<jlo: none) */
  const int* bin_src;          /* device int[4*(Nc+1)] (16-byte aligned) or NULL: offsets into one row of the band
                                  spectra (band_off[j] + k - (band_p[j] - band_lg[j]/2)) of the <= 3 bands that cover
                                  bin k in entries 0..2, sum_lg = none (a zero entry the
                                  library keeps behind each row), entry 3 unused.  Lets the synthesis overlap-add
                                  run as a gather inside the inverse transform; NULL (a bin covered by > 3 bands):
                                  separate gather kernel. */
} babe_cqt_plan;

/* bytes of scratch the calls below need for a batch of B rows */
size_t babe_cqt_workspace(const babe_cqt_plan* plan, int B);

/* X[B,Nc+1,2] = rfft(x[B,Ls]) * bin_scale (bin_scale[Nc+1] real, optional). */
int babe_rfft(const babe_cqt_plan* plan, const float* x, float* X, int B, const float* bin_scale,
              void* workspace, size_t workspace_bytes, void* stream);
/* x[B,Ls] = irfft(X[B,Nc+1,2] * bin_scale): imaginary parts of the DC and
 * Nyquist bins are ignored and the 1/Ls normalisation applied, like torch. */
int babe_irfft(const babe_cqt_plan* plan, const float* X, float* x, int B, const float* bin_scale,
               void* workspace, size_t workspace_bytes, void* stream);
/* y = irfft(rfft(x) * H), H[Nc+1] real: CQT_nsgt.apply_hpf_DC (a18) with
 * H = Hhpf.  Self-adjoint, so it is also its own backward. */
int babe_spectral_filter(const babe_cqt_plan* plan, const float* x, float* y, int B,
                         const float* H, void* workspace, size_t workspace_bytes, void* stream);
/* Analysis (a16 CQT_nsgt.fwd, and the backward of bwd):
 *   c_j = IFFT_M(fold(rfft(x)[bins of band j] * win[band_off[j]+i] * bin_scale))
 * out_octaves_host: HOST array of numocts DEVICE pointers, octave o receives
 * [B, binsoct, M[o]] complex64 (lowest octave first), or, planar != 0, float
 * [B, 2, binsoct, M[o]] (real plane, imaginary plane): the layout the denoiser
 * builds with view_as_real + permute + contiguous at networks/cqtdiff+.py:750-753. */
int babe_cqt_analysis(const babe_cqt_plan* plan, const float* x, float* const* out_octaves_host,
                      int planar, int B, const float* win, const float* bin_scale, void* workspace,
                      size_t workspace_bytes, void* stream);
/* Synthesis (a17 CQT_nsgt.bwd, and the backward of fwd):
 *   x = irfft(bin_scale * sum_j unfold(FFT_M(c_j)) * win[band_off[j]+i]) */
int babe_cqt_synthesis(const babe_cqt_plan* plan, const float* const* in_octaves_host, int planar,
                       float* x, int B, const float* win, const float* bin_scale, void* workspace,
                       size_t workspace_bytes, void* stream);   /* planar: networks/cqtdiff+.py:826-830 */

/* ---- denoiser residual-layer glue (SURVEY 8f-2, the caller either side of the CQT) ---- */
/* One layer of ResnetBlock.forward (networks/cqtdiff+.py:470-482) around its convolution, on
 * contiguous NCHW float32 activations x[N,C,F,T] (P = F*T):
 *   h = gelu(BiasFreeGroupNorm_G(x) * gamma[c] * (aff[n,c] + 1))     (norm: networks/cqtdiff+.py:137-163,
 *                                                                     x / (unbiased std of (n, group) + eps))
 *   y = (x0 + v * gate[n,c]) * scale                                 (v = conv(h), scale = 1/sqrt(2))
 * babe_gn_stats writes per-slice (sum, sum of squares) doubles part[N*G][slices][2]
 * (slices = babe_gn_slices(...)); the consumers finish the statistics themselves. */
int babe_gn_slices(int N, int C, int G, long long P);
int babe_gn_stats(const float* x, double* part, int N, int C, int G, long long P, int slices,
                  void* stream);
int babe_gn_film_gelu(const float* x, float* h, const double* part, int slices, const float* gamma,
                      const float* aff, int N, int C, int G, long long P, float eps, void* stream);
/* gate == NULL: gate = 1;  x0 == NULL: out = v * gate * scale (the backward wrt v). */
int babe_gate_residual(const float* x0, const float* v, const float* gate, float* out, int N, int C,
                       long long P, float scale, void* stream);
/* Backward of (babe_gn_stats + babe_gn_film_gelu) wrt x, with the residual branch folded in:
 *   gx = gy * res_scale + d/dx <gh, h(x)>      (gy may be NULL)
 * in two launches: _reduce fills gr_part[N*C][slices2] (slices2 = babe_gn_bwd_slices(...)) with the
 * partial sums of the statistic's gradient, then babe_gn_film_gelu_bwd writes gx. */
int babe_gn_bwd_slices(int N, int C, long long P);
int babe_gn_film_gelu_bwd_reduce(const float* gh, const float* x, const double* part, int slices,
                                 double* gr_part, int slices2, const float* gamma, const float* aff,
                                 int N, int C, int G, long long P, float eps, void* stream);
int babe_gn_film_gelu_bwd(const float* gh, const float* x, const float* gy, float* gx,
                          const double* part, int slices, const double* gr_part, int slices2,
                          const float* gamma, const float* aff, int N, int C, int G, long long P,
                          float eps, float res_scale, void* stream);

/* x2 anti-aliased time resampling of UpDownResample (networks/cqtdiff+.py:522-580, mode "T",
 * reflect padding fused) on `rows` independent rows; T = length of the x-side row (even):
 *   mode 0: down   in[rows][T]   -> out[rows][T/2]     mode 2: gradient of mode 0, in[rows][T/2] -> out[rows][T]
 *   mode 1: up     in[rows][T]   -> out[rows][2T]      mode 3: gradient of mode 1, in[rows][2T]  -> out[rows][T]
 * taps_host: the L = 4, 8 or 12 filter taps (host memory; `_kernels`, networks/cqtdiff+.py:509-521). */
int babe_resample2(const float* in, float* out, long long rows, int T, int mode,
                   const float* taps_host, int L, void* stream);

/* ---- keyed per-row noise (sampler draws with BlindSamplerFused.row_seeds) ---- */
/* out[b,n] = a[b,n] + eps[b,n] * mult * (*scale) * row_scale[b] on B rows of T samples, where eps[b,n] is the
 * standard normal sample n of row seed seeds[b] (int64 read as uint64) at draw index *draw + slot: Philox4x32-10
 * with key (seed low, seed high) and counter (n/4, draw index, 0, 0), uniforms (2 (x >> 9) + 1) 2^-24, Box-Muller
 * (DESIGN.md 4.8).  eps depends on (seed, draw index, n) only, never on B, the row's position, T or alignment.
 * a (may be NULL = 0, may equal out), scale (one device float) and row_scale (B device floats) are optional; draw is
 * one device int, read at run time, so a captured graph replays with the value it holds then. */
int babe_row_noise(float* out, const float* a, const long long* seeds, int B, int T, const int* draw, int slot,
                   const float* scale, const float* row_scale, float mult, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BABE_B200_H */
