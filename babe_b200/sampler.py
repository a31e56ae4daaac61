"""Blind bandwidth-extension posterior sampler on the CUDA operator.

``BlindSamplerFused`` is a drop-in for ``tester.sampler_callable``
('testing.blind_bwe_sampler.BlindSampler' in conf/tester/blind_bwe.yaml:9): same
constructor ``(model, diff_params, args, rid)`` and the same
``predict_blind_bwe`` / ``predict_bwe`` / ``predict_unconditional`` methods and
return tuples (testing/blind_bwe_sampler.py:14,306,366,619).  Differences are
purely in execution:

* the per-step filter re-estimation runs as ONE statistics pass over
  (x_den, y) plus ONE device-resident kernel doing all <=100 projected
  gradient iterations (reference: a Python loop of ~25 launches and >=K+2 host
  syncs per iteration, testing/blind_bwe_sampler.py:562-590);
* the reconstruction-guidance loss and its cotangent are two fused launches
  (filter-design + STFT + multiply + iSTFT + residual + row norms; adjoint)
  and H(fc, A) is never written to HBM;
* noise may be drawn on the device (``device_noise=True``); the default keeps
  the reference's host generator stream so that outputs are comparable for a
  fixed ``torch.manual_seed``;
* with ``row_seeds`` (one 64-bit seed per row) every draw is keyed noise generated on
  the device by ``k_row_noise`` (DESIGN.md 4.8): row r's noise is a function of its seed,
  the draw index and the sample index alone, so a row restores the same whatever the
  batch, its position in it or the number of ranks.

One behaviour goes beyond the reference: with ``filter_per_row`` every row of ``y``
is an independent restoration (its own fit statistics, filter fit, guidance
filter and guidance normaliser), i.e. row r of one call with B rows is what a
call on ``y[r:r+1]`` alone returns with the same noise for that row.  Between the
two, ``filter_groups`` (sizes of consecutive row groups) gives every group one
filter: group g of one call is what a shared-filter call on its rows alone returns.
"""
import types
import warnings

import torch

from . import blind_bwe_utils as bu
from . import ops
from . import profiling
from ._lib import FitConfig


# ---------------------------------------------------------------------------
# args shim (Hydra/OmegaConf are not installed; SURVEY Appendix D / E)
# ---------------------------------------------------------------------------
def _ns(**kw):
    return types.SimpleNamespace(**kw)


def make_args(sample_rate=22050, audio_len=184184, T=35, xi=0.2, start_sigma=0.2,
              NFFT=4096, fc_init=(280, 285, 290, 295, 300), A_init=(-15, -17, -20, -25, -30),
              max_iter=100, Schurn=20, num_octs=7, bins_per_oct=64, filter_per_row=False, **extra):
    """Nested attribute namespace carrying exactly the fields the sampler, EDM
    and the CQTDiff+ constructor read, with the values of
    conf/tester/blind_bwe.yaml, conf/exp/maestro22k_8s.yaml,
    conf/diff_params/edm.yaml and conf/network/cqtdiff+.yaml.  ``filter_per_row`` sets
    ``tester.blind_bwe.filter_per_row`` (one filter estimate per row, see ``BlindSamplerFused``)."""
    args = _ns(
        exp=_ns(sample_rate=sample_rate, audio_len=audio_len, seed=42),
        diff_params=_ns(callable="babe_b200.edm.EDM", sigma_data=0.063, sigma_min=1e-5,
                        sigma_max=10, P_mean=-1.2, P_std=1.2, ro=13, ro_train=13, Schurn=5,
                        Snoise=1, Stmin=0, Stmax=50,
                        aweighting=_ns(use_aweighting=False, ntaps=101)),
        network=_ns(callable="babe_b200.denoiser.CQTDiffPlus", use_fencoding=False, use_norm=True,
                    emb_dim=256, Ns=[64, 96, 96, 128, 128, 256, 256], Ss=[2] * 7,
                    num_dils=[2, 3, 4, 5, 6, 7, 7], attention_layers=[0] * 8,
                    bottleneck_type="res_dil_convs", num_bottleneck_layers=1,
                    cqt=_ns(window="kaiser", beta=1, num_octs=num_octs, bins_per_oct=bins_per_oct),
                    attention_dict=_ns(num_heads=8, attn_dropout=0.0, bias_qkv=False, N=0,
                                       rel_pos_num_buckets=32, rel_pos_max_distance=64,
                                       use_rel_pos=True, Nproj=8)),
        tester=_ns(
            sampler_callable="babe_b200.sampler.BlindSamplerFused",
            T=T, order=2, filter_out_cqt_DC_Nyq=True,
            diff_params=_ns(same_as_training=False, sigma_data=0.063, sigma_min=1e-4, sigma_max=1,
                            ro=8, Schurn=Schurn, Snoise=1.0, Stmin=0, Stmax=50),
            posterior_sampling=_ns(xi=xi, data_consistency=False, norm=2, smoothl1_beta=1,
                                   SNR_observations="None", start_sigma=start_sigma,
                                   freq_weighting="None", freq_weighting_filter="sqrt",
                                   stft_distance=_ns(use=False, mag=False, use_multires=False,
                                                     nfft=2048, logmag=False)),
            blind_bwe=_ns(fcmin=20, fcmax="nyquist", Amin=-50, Amax=30, NFFT=NFFT,
                          sigma_den_estimate=0.0, filter_per_row=bool(filter_per_row),
                          test_filter=_ns(fc=[1000], A=[-20]),
                          initial_conditions=_ns(fc=list(fc_init), A=list(A_init)),
                          optimization=_ns(max_iter=max_iter, tol=[5e-3, 5e-3], mu=[1000, 10],
                                           clamp_fc=True, clamp_A=True, only_negative_A=True)),
            complete_recording=_ns(n_segments_blindstep=2, std=0.1, overlap=0.25, inpaint_DC=True),
        ),
    )
    for k, v in extra.items():
        setattr(args, k, v)
    return args


# ---------------------------------------------------------------------------
# a7: filter fit = one statistics pass + one device-resident loop
# ---------------------------------------------------------------------------
class FilterFit:
    """BlindSampler.fit_params (testing/blind_bwe_sampler.py:533-595)."""

    def __init__(self, nfft=4096, sample_rate=22050, fcmin=20, fcmax="nyquist", Amin=-50, Amax=30,
                 max_iter=100, tol=(5e-3, 5e-3), mu=(1000, 10), clamp_fc=True, clamp_A=True,
                 only_negative_A=True, freq_weighting="sqrt", device="cuda"):
        self.nfft = int(nfft)
        self.sample_rate, self.freq_weighting = sample_rate, str(freq_weighting)
        fcmax_v = sample_rate // 2 if fcmax == "nyquist" else fcmax   # :35-38 (integer division)
        self.cfg = FitConfig(mu_fc=mu[0], mu_A=mu[1], fcmin=fcmin, fcmax=fcmax_v, Amin=Amin, Amax=Amax,
                             tol_fc=tol[0], tol_A=tol[1], max_iter=int(max_iter),
                             clamp_fc=int(bool(clamp_fc)), clamp_A=int(bool(clamp_A)),
                             only_negative_A=int(bool(only_negative_A)))
        self.freqs = torch.fft.rfftfreq(self.nfft, d=1 / sample_rate).to(device)   # :629
        w = bu.freq_weight_vector(freq_weighting, self.nfft // 2 + 1, device)
        self.w = w if w is not None else torch.ones(self.nfft // 2 + 1, device=device)
        self.joint = False
        self.per_row = False           # True: params (B, 2, K), one fit per row on that row's statistics
        self.groups = None             # group sizes: params (G, 2, K), one fit per group of consecutive rows

    @classmethod
    def from_args(cls, args, device):
        b, o = args.tester.blind_bwe, args.tester.blind_bwe.optimization
        return cls(nfft=b.NFFT, sample_rate=args.exp.sample_rate, fcmin=b.fcmin, fcmax=b.fcmax,
                   Amin=b.Amin, Amax=b.Amax, max_iter=o.max_iter, tol=o.tol, mu=o.mu,
                   clamp_fc=o.clamp_fc, clamp_A=o.clamp_A, only_negative_A=o.only_negative_A,
                   freq_weighting=args.tester.posterior_sampling.freq_weighting_filter, device=device)

    def cfg_key(self):
        c = self.cfg
        return (self.nfft, self.sample_rate, self.freq_weighting, c.mu_fc, c.mu_A, c.fcmin, c.fcmax, c.Amin, c.Amax, c.tol_fc, c.tol_A, c.max_iter,
                c.clamp_fc, c.clamp_A, c.only_negative_A)

    def stats(self, x_den, y):
        if self.groups is not None:
            return ops.stft_stats_groups(x_den, y, self.nfft, self.groups)
        if self.per_row:
            return ops.stft_stats_rows(x_den, y, self.nfft)
        return ops.stft_stats(x_den, y, self.nfft, mode=0)

    def __call__(self, x_den, y, params, return_iters=False, abc=None):
        """params (2,K) is updated in place (the reference also mutates it,
        testing/blind_bwe_sampler.py:577-583) and returned; (B,2,K) per row with ``per_row``."""
        if abc is None:
            abc = self.stats(x_den, y)
        if self.per_row or self.groups is not None:
            return ops.fit_params_rows(abc, self.w, self.freqs, params, self.cfg, return_iters=return_iters)
        if self.joint:                 # one filter for the rows of ALL ranks (SURVEY 8e)
            from . import distributed
            distributed.sum_over_ranks_(abc)
        return ops.fit_params(abc, self.w, self.freqs, params, self.cfg, return_iters=return_iters)


# ---------------------------------------------------------------------------
# a8: fused reconstruction-guidance loss
# ---------------------------------------------------------------------------
class _RecGuidanceNorm(torch.autograd.Function):
    """norm_b = || y_b - A_{fc,A}(x_b) ||_2  (testing/blind_bwe_sampler.py:89,117)
    with backward  g_b * A^T((A x_b - y_b) / norm_b)  (what :120 back-propagates
    into the denoiser).  H is designed inside both kernels; fc, A of shape (B, K) give every row its own filter.
    ``known`` (int32[B], per-row filters only) replaces A by the known-prefix operator of the autoregressive windows,
    D_b x = m_b x + (1 - m_b) A_b x with m_b[n] = 1[n < known[b]] (:259-303), and the backward applies D_b^T."""

    @staticmethod
    def forward(ctx, x, y, freqs, fc, A, nfft, known=None):
        ss = torch.zeros(x.shape[0], dtype=torch.float64, device=x.device)
        ctx.masked = {} if known is None else {"known": known}       # unmasked calls keep their exact signature
        if fc.dim() == 2:
            r = ops.apply_filter_rows(x, nfft, freqs, fc, A, sub=y, row_sumsq=ss, **ctx.masked)
        else:
            r = ops.apply_filter(x, nfft, freqs=freqs, fc=fc, A=A, sub=y, row_sumsq=ss)
        norms = torch.sqrt(ss).to(torch.float32)
        ctx.save_for_backward(r, norms, freqs, fc, A)
        ctx.nfft = nfft
        return norms

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        r, norms, freqs, fc, A = ctx.saved_tensors
        scale = (g / norms).contiguous()
        if fc.dim() == 2:
            gx = ops.apply_filter_rows(r, ctx.nfft, freqs, fc, A, adjoint=True, row_scale=scale, **ctx.masked)
        else:
            gx = ops.apply_filter(r, ctx.nfft, freqs=freqs, fc=fc, A=A, adjoint=True, row_scale=scale)
        return gx, None, None, None, None, None, None


def rec_guidance_norms(x, y, freqs, filter_params, nfft, known=None):
    """filter_params (2, K): one filter for all rows; (B, 2, K): row b filtered with filter_params[b].  ``known``
    (int32[B] CUDA tensor, with (B, 2, K) only): the norms of the known-prefix masked operator (``_RecGuidanceNorm``)."""
    fc, A = (filter_params[:, 0], filter_params[:, 1]) if filter_params.dim() == 3 else filter_params
    if known is not None and filter_params.dim() != 3:
        raise ValueError("known-prefix guidance needs per-row (B, 2, K) filter parameters")
    return _RecGuidanceNorm.apply(x, y, freqs, fc.contiguous(), A.contiguous(), int(nfft), known)


def known_prefix_lengths(mask):
    """k_b of a (B, T) mask whose every row is a known prefix (1 for n < k_b, 0 from k_b on; all ones: k_b = T,
    all zeros: 0), as an int32[B] host tensor; None for any other mask."""
    m = mask.detach().cpu()
    k = (m == 1).to(torch.int64).cumprod(-1).sum(-1)
    prefix = torch.arange(m.shape[-1]) < k.unsqueeze(-1)
    return k.to(torch.int32) if torch.equal(m, prefix.to(m.dtype)) else None


_PINNED_NOISE = {}


# ---------------------------------------------------------------------------
class BlindSamplerFused:
    def __init__(self, model, diff_params, args, rid=False, device_noise=False, freeze_model=True,
                 cuda_graph=False):
        """testing/blind_bwe_sampler.py:14-47.  ``freeze_model``: sampling never needs parameter
        gradients (the reference only takes ``autograd.grad(..., inputs=x)``, :120); freezing them lets
        ``babe_b200.denoiser`` run its fused layer glue and skips the parameter-gradient branches."""
        self.model = model
        if freeze_model and isinstance(model, torch.nn.Module):
            model.requires_grad_(False)
        # SURVEY 8f-1: replay the denoiser's forward and backward from two captured CUDA graphs (static
        # shapes, frozen parameters, no host synchronisation inside the network)
        self.cuda_graph = cuda_graph
        self._graphed, self._graph_key, self._graph_launches = None, None, (0, 0)
        # SURVEY 8f-1, whole step: ONE captured CUDA graph per sampler step (stochastic move, denoiser forward and
        # backward, fit statistics + fit loop, fused guidance, Heun correction with its second evaluation, state
        # update); the schedule scalars are device tensors, nothing is launched eagerly between two replays
        self.step_graph = False
        self._step_graphs, self._step_key = {}, None
        self.diff_params = diff_params
        self.args = args
        if not args.tester.diff_params.same_as_training:
            self.update_diff_params()
        self.order = args.tester.order
        self.xi = args.tester.posterior_sampling.xi
        self.data_consistency = args.tester.posterior_sampling.data_consistency
        self.nb_steps = args.tester.T
        self.start_sigma = args.tester.posterior_sampling.start_sigma
        if self.start_sigma == "None":
            self.start_sigma = None
        self.device_noise = device_noise
        self.generator = None          # optional torch.Generator for device noise
        self.noise_fn = None           # optional callable(shape, device) -> tensor (benchmarks, parity runs)
        # one seed per row of the next call (list of ints or an int64 tensor): keyed device noise for every draw,
        # before device_noise / generator; None: the sources above
        self.row_seeds = None
        self._keyed = None             # during a call with row_seeds: the device seeds and the draw-index scalar
        self._eval_slot = 1            # draw slot of the evaluation running (1: first, 4: Heun correction)
        self.joint = False             # True: ranks reproduce ONE reference call on the whole batch
        # True: every row of y is an independent restoration (own filter estimate and guidance scale); Hydra-style
        # configs switch it on with tester.blind_bwe.filter_per_row
        self.filter_per_row = bool(getattr(args.tester.blind_bwe, "filter_per_row", False))
        # None, or the sizes [n_0, ..., n_{G-1}] (sum = B) of consecutive row groups of the next predict_blind_bwe
        # call: group g (rows o_g .. o_g + n_g - 1) is restored with ONE filter, as a shared-filter call on its rows
        # alone would restore it (statistics summed over the group, one fit, the group's guidance normaliser)
        self.filter_groups = None
        self._groups = None            # during a grouped call: sizes and the device row -> group maps
        self._fit = None

    def update_diff_params(self):
        """testing/blind_bwe_sampler.py:50-60."""
        d, s = self.diff_params, self.args.tester.diff_params
        d.sigma_min, d.sigma_max, d.ro, d.sigma_data = s.sigma_min, s.sigma_max, s.ro, s.sigma_data
        d.Schurn, d.Stmin, d.Stmax, d.Snoise = s.Schurn, s.Stmin, s.Stmax, s.Snoise

    # -- noise ---------------------------------------------------------------
    def _randn(self, shape, device):
        if self.noise_fn is not None:
            return self.noise_fn(shape, device)
        if self.device_noise:
            return torch.randn(shape, device=device, generator=self.generator)
        if torch.device(device).type != "cuda":
            return torch.randn(shape).to(device)   # reference: host generator (:513, edm.py:105)
        return self._host_randn_pinned(tuple(shape), device)

    def _host_randn_pinned(self, shape, device):
        """The reference's ``torch.randn(shape).to(device)`` -- same host generator stream, same values --
        drawn into one of two page-locked staging buffers and copied asynchronously (a pageable source makes
        the copy synchronous and ~2x slower)."""
        ring = _PINNED_NOISE                       # process-wide: pinning is expensive, and freeing pinned memory
        slot = ring.get(shape)                     # while a CUDA graph is being captured invalidates the capture
        if slot is None:
            slot = ring[shape] = {"bufs": [torch.empty(shape, pin_memory=True) for _ in range(2)],
                                  "events": [None, None], "i": 0}
        i = slot["i"]
        slot["i"] = 1 - i
        if slot["events"][i] is not None:
            slot["events"][i].synchronize()        # the previous copy out of this buffer has completed
        buf = slot["bufs"][i]
        torch.randn(shape, out=buf)
        out = buf.to(device, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        slot["events"][i] = ev
        return out

    # -- keyed noise (row_seeds) -------------------------------------------------
    # Draw index d of a call: 0 the initial state; schedule step i uses d = 1 + 8 i + slot with slot 0 the stochastic
    # move, 1 / 2 / 3 the first evaluation's SNR observation noise (fit_params), sigma_den_estimate draw and SNR noise
    # (get_rec_grads), 4 / 5 / 6 the same for the Heun evaluation, 7 reserved.  A call resumed at step i therefore
    # draws what the uninterrupted call drew from step i on.
    @staticmethod
    def _seed_tensor(seeds):
        """row_seeds -> int64 tensor (the bits of unsigned 64-bit seeds)."""
        if torch.is_tensor(seeds):
            if seeds.dtype != torch.int64 or seeds.dim() != 1:
                raise ValueError(f"row_seeds must be a 1-D int64 tensor or a list of ints, got a {seeds.dtype} "
                                 f"tensor of shape {tuple(seeds.shape)}")
            return seeds
        vals = []
        for v in seeds:
            if isinstance(v, bool) or not isinstance(v, int) and not hasattr(v, "__index__"):
                raise ValueError(f"row_seeds entries must be ints, got {v!r}")
            v = int(v)
            if not -(1 << 63) <= v < (1 << 64):
                raise ValueError(f"row seed {v} does not fit in 64 bits")
            vals.append(v - (1 << 64) if v >= (1 << 63) else v)
        return torch.tensor(vals, dtype=torch.int64)

    def _keyed_begin(self, B, device):
        """Start a call on B rows: keyed noise if ``row_seeds`` is set (checked here), else the other sources."""
        self._keyed = None
        if self.row_seeds is None:
            return
        if self.noise_fn is not None:
            raise ValueError("row_seeds and noise_fn are both set: choose one noise source")
        seeds = self._seed_tensor(self.row_seeds)
        if seeds.numel() != B:
            raise ValueError(f"row_seeds has {seeds.numel()} seeds for a call on {B} rows")
        self._keyed = types.SimpleNamespace(seeds=seeds.to(device),
                                            draw=torch.zeros(1, dtype=torch.int32, device=device))

    def _keyed_step(self, i):
        """Draw-index base of schedule step i (a device scalar, so captured kernels read it at replay)."""
        if self._keyed is not None:
            self._keyed.draw.fill_(1 + 8 * i)

    def _keyed_noise(self, a_or_shape, slot, scale=None, row_scale=None, mult=1.0, out=None):
        k = self._keyed
        return ops.row_noise(k.seeds, a_or_shape, k.draw, slot, scale=scale, row_scale=row_scale, mult=mult, out=out)

    def _initial_state(self, shape, device, t0, y=None):
        """eps * t0, or y + eps * t0 (:640-644): draw 0."""
        if self._keyed is not None:
            return self._keyed_noise(shape if y is None else y, 0, scale=t0.reshape(1))
        if y is None:
            return self._randn(shape, device) * t0
        return y + self._randn(shape, device) * t0

    def move_timestep(self, x, t, gamma, Snoise=1):
        """testing/blind_bwe_sampler.py:509-516 (always draws).  Keyed noise: draw and update in one launch."""
        t_hat = t + gamma * t
        if self._keyed is not None:
            return self._keyed_noise(x, 0, scale=((t_hat ** 2 - t ** 2) ** (1 / 2)).reshape(1), mult=Snoise), t_hat
        eps = self._randn(x.shape, x.device) * Snoise
        return x + ((t_hat ** 2 - t ** 2) ** (1 / 2)) * eps, t_hat

    # -- pieces of one evaluation -------------------------------------------------
    def get_denoised_estimate(self, x, t_i):
        """testing/blind_bwe_sampler.py:152-157."""
        net = self._graphed_model(x) if self.cuda_graph and x.is_cuda and x.requires_grad else self.model
        x_hat = self.diff_params.denoiser(x, net, t_i.unsqueeze(-1))
        if self.args.tester.filter_out_cqt_DC_Nyq:
            x_hat = self.model.CQTransform.apply_hpf_DC(x_hat)
        return x_hat

    def _graphed_model(self, x):
        """The network as a callable replaying captured CUDA graphs (``torch.cuda.make_graphed_callables``:
        one graph for the forward, one for the backward wrt the input); eager model on any failure."""
        try:      # in-place weight updates (load_state_dict) invalidate what the graphs captured
            ver = sum(p._version for p in self.model.parameters())
        except Exception:                                  # noqa: BLE001 - not an nn.Module
            ver = 0
        key = (tuple(x.shape), x.dtype, x.device, ver)
        if self._graph_key != key:
            self._graph_key, self._graphed = key, None
            try:
                ss = torch.ones(1, 1, device=x.device, dtype=x.dtype)
                s0 = torch.zeros_like(x).requires_grad_(True)
                l0 = profiling.launches()                  # launches of one eager forward / backward
                out = self.model(s0, ss)
                l1 = profiling.launches()
                torch.autograd.grad(out.sum(), s0)
                self._graph_launches = (l1 - l0, profiling.launches() - l1)
                del out, s0                                # no autograd node of the default stream may survive
                torch.cuda.synchronize()
                sx = torch.zeros_like(x).requires_grad_(True)
                model = self.model
                quiet = getattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch", None)
                if quiet is not None:                      # the capture runs on a side stream by design
                    quiet(False)
                self._graphed = torch.cuda.make_graphed_callables(lambda a, b: model(a, b), (sx, ss))
            except Exception as exc:                       # noqa: BLE001 - any capture problem: stay eager
                warnings.warn(f"CUDA-graph capture of the denoiser failed ({exc!r}); running it eagerly")
                self._graphed = None
        if self._graphed is None:
            return self.model
        graphed, (lf, lb) = self._graphed, self._graph_launches

        def net(a, sigma):
            profiling.add_launches(lf + lb)               # replayed kernels of the forward + backward graphs
            return graphed(a.contiguous(), sigma.reshape(1, 1).to(a.dtype))
        return net

    def apply_filter_fcA(self, x, filter_params):
        """testing/blind_bwe_sampler.py:518-520, H designed inside the kernel; filter_params (B, 2, K) filters
        row b with filter_params[b]."""
        if filter_params.dim() == 3:
            return bu.apply_filter_rows(x, self.freqs, filter_params[:, 0], filter_params[:, 1],
                                        self.args.tester.blind_bwe.NFFT)
        H = bu.design_filter(filter_params[0], filter_params[1], self.freqs)
        return bu.apply_filter(x, H, self.args.tester.blind_bwe.NFFT)

    def _maybe_noise_observations(self, y, slot):
        ps = self.args.tester.posterior_sampling
        if ps.SNR_observations != "None":           # :80-86, :542-548 (in place on y)
            snr = 10 ** (ps.SNR_observations / 10)
            sigma = torch.sqrt(torch.var(y, -1) / snr).unsqueeze(-1)
            if self._keyed is None:
                y += sigma * self._randn(y.shape, y.device)
            elif y.is_contiguous():
                self._keyed_noise(y, slot, row_scale=sigma.reshape(-1), out=y)
            else:
                y.copy_(self._keyed_noise(y, slot, row_scale=sigma.reshape(-1)))

    def fit_params(self, denoised_estimate, y, filter_params):
        """testing/blind_bwe_sampler.py:533-595."""
        self._maybe_noise_observations(y, self._eval_slot)
        sde = self.args.tester.blind_bwe.sigma_den_estimate
        if sde and self._keyed is not None:
            denoised_estimate = self._keyed_noise(denoised_estimate, self._eval_slot + 1, mult=sde)
        elif sde:
            denoised_estimate = denoised_estimate + self._randn(denoised_estimate.shape,
                                                                 denoised_estimate.device) * sde
        return self._fit(denoised_estimate, y, filter_params)

    def get_rec_grads(self, x_den, y, x, t_i, filter_params):
        """testing/blind_bwe_sampler.py:75-135."""
        ps = self.args.tester.posterior_sampling
        self._maybe_noise_observations(y, self._eval_slot + 2)
        nfft = self.args.tester.blind_bwe.NFFT
        filter_params = self._row_params(filter_params)
        if ps.norm == 2 and not ps.stft_distance.use:
            norm = rec_guidance_norms(x_den, y, self.freqs, filter_params, nfft)
        else:
            den_rec = self.apply_filter_fcA(x_den, filter_params)
            if ps.norm == "smoothl1":
                norm = torch.nn.functional.smooth_l1_loss(y, den_rec, reduction='sum', beta=ps.smoothl1_beta)
            elif ps.norm == "cosine":
                cos = torch.nn.CosineSimilarity(dim=1, eps=1e-6)
                norm = (1 - cos(den_rec, y)).clamp(min=0)
            elif ps.stft_distance.use:
                if ps.stft_distance.use_multires:
                    raise NotImplementedError("multires STFT distance is dead code in the reference "
                                              "(testing/blind_bwe_sampler.py:108 calls a missing self.norm)")
                if ps.stft_distance.mag:
                    norm = bu.apply_norm_STFTmag_fweighted(y, den_rec, ps.freq_weighting,
                                                           ps.stft_distance.nfft,
                                                           logmag=ps.stft_distance.logmag)
                else:
                    norm = bu.apply_norm_STFT_fweighted(y, den_rec, ps.freq_weighting, ps.stft_distance.nfft)
            else:
                norm = torch.linalg.norm(y - den_rec, dim=1, ord=ps.norm)
        (rec_grads,) = torch.autograd.grad(outputs=norm.sum(), inputs=x)
        if self._groups is not None:   # Frobenius norm over each group's rows, in fp64, gathered back to the rows
            g = self._groups
            sq = (rec_grads.double() ** 2).sum(1)
            gsq = torch.cat((sq, sq.new_zeros(1)))[g.pad].sum(1)       # padding reads the appended zero
            normguide = torch.sqrt(gsq).float()[g.row_group].unsqueeze(1) / self.args.exp.audio_len ** 0.5
        elif self.filter_per_row:      # each row is its own restoration: its own normaliser
            normguide = torch.linalg.norm(rec_grads, dim=1, keepdim=True) / self.args.exp.audio_len ** 0.5
        elif self.joint:               # Frobenius norm over the rows of ALL ranks (:125)
            from . import distributed
            sq = (rec_grads.double() ** 2).sum().reshape(1)
            normguide = torch.sqrt(distributed.sum_over_ranks_(sq))[0].float() / self.args.exp.audio_len ** 0.5
        else:
            normguide = torch.linalg.norm(rec_grads) / self.args.exp.audio_len ** 0.5
        s = self.xi / (normguide + 1e-6)
        return s * rec_grads / t_i

    def data_consistency_step_classic(self, x_hat, y, filter_params):
        """testing/blind_bwe_sampler.py:63-73."""
        return y + x_hat - self.apply_filter_fcA(x_hat, self._row_params(filter_params))

    def _row_params(self, filter_params):
        """Grouped calls: the (B, 2, K) parameters of the rows, row r taking its group's filter; else unchanged."""
        if self._groups is None:
            return filter_params
        return filter_params.index_select(0, self._groups.row_group)

    def _evaluate(self, x_in, t_in, y, filter_params, slot=1):
        """Lines :689-:709 (and :733-:752 for the Heun correction, keyed draw slot 4)."""
        self._eval_slot = slot
        x_in.requires_grad_(True)
        x_den = self.get_denoised_estimate(x_in, t_in)
        x_den_2 = x_den.clone().detach()
        filter_params = self.fit_params(x_den_2, y, filter_params)
        rec_grads = self.get_rec_grads(x_den, y, x_in, t_in, filter_params)
        x_in.detach_()
        score = (x_den_2 - x_in) / t_in ** 2 - rec_grads
        if self.args.tester.posterior_sampling.data_consistency:
            x_den_3 = score * t_in ** 2 + x_in
            x_den_3 = self.data_consistency_step_classic(x_den_3, y, filter_params)
            score = (x_den_3 - x_in) / t_in ** 2
        return score, filter_params, x_den_2

    def _check_per_row(self, compute_sweep):
        """Modes that cannot run with one filter per row."""
        if self.joint:
            raise ValueError("filter_per_row and joint exclude each other: joint shares ONE filter over all rows "
                             "of all ranks, filter_per_row gives every row its own")
        sd = self.args.tester.posterior_sampling.stft_distance
        if sd.use:
            raise NotImplementedError("filter_per_row with the STFT-distance guidance: its norm is one sum over the "
                                      "whole batch, not a per-row quantity" if not sd.use_multires else
                                      "filter_per_row with use_multires: the multi-resolution STFT distance is a "
                                      "batch-wide norm (and dead code in the reference)")
        if compute_sweep:
            raise NotImplementedError("filter_per_row with compute_sweep: the sweep evaluates one loss surface on "
                                      "the statistics of the whole batch")

    def _begin_groups(self, B, device, compute_sweep):
        """Check ``filter_groups`` against a call on B rows and build its device row -> group maps (None: off)."""
        self._groups = None
        if self.filter_groups is None:
            return
        sizes = ops.group_sizes(self.filter_groups, B)
        if self.joint or self.filter_per_row:
            raise ValueError("filter_groups excludes joint and filter_per_row: choose one way of sharing filters "
                             "(joint: one over all ranks, filter_per_row: one per row, filter_groups: one per group)")
        sd = self.args.tester.posterior_sampling.stft_distance
        if sd.use:
            raise NotImplementedError("filter_groups with the STFT-distance guidance: its norm is one sum over the "
                                      "whole batch, not a per-group quantity")
        if compute_sweep:
            raise NotImplementedError("filter_groups with compute_sweep: the sweep evaluates one loss surface on the "
                                      "statistics of the whole batch")
        G, nmax = len(sizes), max(sizes)
        row_group = torch.repeat_interleave(torch.arange(G), torch.tensor(sizes))
        pad = torch.full((G, nmax), B, dtype=torch.int64)              # index B: the zero appended to the rows
        o = 0
        for g, n in enumerate(sizes):
            pad[g, :n] = torch.arange(o, o + n)
            o += n
        self._groups = types.SimpleNamespace(sizes=sizes, row_group=row_group.to(device), pad=pad.to(device))

    def _no_groups(self, what):
        if self.filter_groups is not None:
            raise ValueError(f"{what} does not support filter_groups (set it to None): only predict_blind_bwe "
                             "estimates a filter per group")

    def compute_sweep(self, denoised_estimate, y):
        """testing/blind_bwe_sampler.py:598-616 on the collapsed statistics."""
        abc = self._fit.stats(denoised_estimate, y)
        w2 = self._fit.w.double() ** 2
        grads = torch.zeros(self.fc_s.shape[0], self.A_s.shape[0], 2)
        norms = torch.zeros(self.fc_s.shape[0], self.A_s.shape[0])
        for i in range(self.fc_s.shape[0]):
            for j in range(self.A_s.shape[0]):
                fc, A = self.fc_s[i].reshape(1), self.A_s[j].reshape(1)
                H = ops.design_filter(fc, A, self.freqs, strict=False).double()
                nrm = torch.sqrt((w2 * (H * H * abc[0] - 2 * H * abc[1] + abc[2])).sum())
                gH = (w2 * (H * abc[0] - abc[1]) / nrm).float()
                gfc, gA, _ = ops.design_filter_vjp(fc, A, self.freqs, gH)
                grads[i, j, 0], grads[i, j, 1], norms[i, j] = gfc[0], gA[0], nrm
        return norms, grads

    # -- one sampler step as a pure function of device tensors ----------------------------------------
    def _step_math(self, x, filter_params, eps, t_i, gamma_i, t_next, y, heun):
        """Lines :686-:761 of the reference loop; all scalars are 0-d device tensors.  eps None: keyed noise."""
        t_hat = t_i + gamma_i * t_i
        if eps is None:
            x_hat = self._keyed_noise(x, 0, scale=((t_hat ** 2 - t_i ** 2) ** (1 / 2)).reshape(1))
        else:
            x_hat = x + ((t_hat ** 2 - t_i ** 2) ** (1 / 2)) * eps
        score, filter_params, x_den_2 = self._evaluate(x_hat, t_hat, y, filter_params)
        fp_mid = filter_params.clone()           # what rid logs (:724): the filter after the FIRST evaluation
        d = -t_hat * score
        h = t_next - t_hat
        if heun:
            x_prime = x_hat + h * d
            score, filter_params, _ = self._evaluate(x_prime, t_next, y, filter_params, slot=4)
            x_new = x_hat + h * ((1 / 2) * d + (1 / 2) * (-t_next * score))
        else:
            x_new = x_hat + h * d
        return x_new, filter_params, x_den_2, fp_mid

    def _step_graph_for(self, y, filter_params, heun):
        """Capture (once per shape / variant) and return the replayable step."""
        keyed = self._keyed
        # keyed noise is generated inside the step from the graph's seed and draw-index buffers: the key records that
        # it is on, not the seed values (new seeds are copied into the buffers, no recapture)
        groups = self._groups
        key = (tuple(y.shape), y.device, tuple(filter_params.shape), self.filter_per_row, keyed is not None,
               self._fit.cfg_key(), None if groups is None else groups.sizes)
        if self._step_key != key:
            self._step_key, self._step_graphs = key, {}
        if heun in self._step_graphs:
            st = self._step_graphs[heun]
            st.y.copy_(y)
            return st
        dev = y.device
        # everything the captured kernels read by address is owned by the graph state: the observations are copied
        # into a static buffer, and the fit object (frequency / weight tables) of the capturing call is kept alive
        # and re-installed on replaying calls
        st = types.SimpleNamespace(
            y=y.clone(), fit=self._fit, freqs=self.freqs,
            x=torch.zeros_like(y), fp=filter_params.clone(), eps=None if keyed is not None else torch.zeros_like(y),
            t_i=torch.ones((), device=dev), gamma=torch.zeros((), device=dev), t_next=torch.ones((), device=dev) * 0.5,
            seeds=None, draw=None, graph=None, x_out=None, fp_out=None, den=None, launches=0, groups=groups)
        if keyed is not None:
            st.seeds, st.draw = keyed.seeds.clone(), torch.zeros_like(keyed.draw)
            self._keyed = types.SimpleNamespace(seeds=st.seeds, draw=st.draw)     # what the captured kernels read
        try:
            self._capture_step(st, heun)
        finally:
            self._keyed = keyed
        self._step_graphs[heun] = st
        return st

    def _capture_step(self, st, heun):
        was_prof = profiling._enabled
        profiling.enable(False)                      # no event records inside a capture
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):                       # warm-up: cuDNN autotuning, lazy tables, allocator pools
                fp = st.fp.clone()
                l0 = profiling.launches()
                self._step_math(st.x, fp, st.eps, st.t_i, st.gamma, st.t_next, st.y, heun)
                st.launches = profiling.launches() - l0
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        import gc
        gc.collect()                                 # nothing may be freed behind the capture's back (a pinned
        gc_was = gc.isenabled()                      # buffer released by the collector queries CUDA events)
        gc.disable()
        try:
            with torch.cuda.graph(g, capture_error_mode="relaxed"):
                x_new, fp_new, den, fp_mid = self._step_math(st.x, st.fp, st.eps, st.t_i, st.gamma, st.t_next, st.y, heun)
                st.x.copy_(x_new)                    # the state lives in the static buffers across replays
                if fp_new.data_ptr() != st.fp.data_ptr():
                    st.fp.copy_(fp_new)
                st.den, st.fp_mid = den, fp_mid
        finally:
            if gc_was:
                gc.enable()
        st.graph = g
        profiling.enable(was_prof)

    # -- the sampling loop ---------------------------------------------------
    def predict_blind_bwe(self, y, rid=False, compute_sweep=False, max_steps=None, step_hook=None,
                          start_step=0, init_x=None, init_params=None):
        """testing/blind_bwe_sampler.py:619-769.  ``max_steps`` bounds the loop
        (benchmarks); ``step_hook(i, x, filter_params)`` is called after each
        step.  ``start_step`` / ``init_x`` / ``init_params`` resume the loop from a given state
        (teacher-forced parity tests: one step from each state of a reference run).

        With ``filter_per_row`` the rows of y are independent restorations: the returned filter is (B, 2, K),
        ``init_params`` may be (2, K) (every row) or (B, 2, K), and with ``rid`` the logged filters are
        (T, B, 2, K).  With ``filter_groups`` (G sizes) the same holds per group: (G, 2, K) filters, ``init_params``
        (2, K) or (G, 2, K), logged filters (T, G, 2, K)."""
        args = self.args
        self._begin_groups(y.shape[0], y.device, compute_sweep)
        self._keyed_begin(y.shape[0], y.device)
        if self.filter_per_row:
            self._check_per_row(compute_sweep)
        device = y.device
        self.freqs = torch.fft.rfftfreq(args.tester.blind_bwe.NFFT, d=1 / args.exp.sample_rate).to(device)
        self._fit = FilterFit.from_args(args, device)
        self._fit.joint = self.joint
        self._fit.per_row = self.filter_per_row
        self._fit.groups = None if self._groups is None else self._groups.sizes
        shape = y.shape
        filter_params = torch.Tensor([args.tester.blind_bwe.initial_conditions.fc,
                                      args.tester.blind_bwe.initial_conditions.A]).to(device)
        if len(filter_params.shape) == 1:
            filter_params.unsqueeze_(1)
        if init_params is not None:
            filter_params = init_params.to(device).clone()
        if self.filter_per_row or self._groups is not None:
            n, what = (shape[0], "per-row") if self._groups is None else (len(self._groups.sizes), "per-group")
            if filter_params.dim() == 2:
                filter_params = filter_params.unsqueeze(0).expand(n, -1, -1)
            if filter_params.dim() != 3 or filter_params.shape[0] != n:
                raise ValueError(f"{what} filter parameters must be (2, K) or ({n}, 2, K), "
                                 f"got {tuple(filter_params.shape)}")
            filter_params = filter_params.contiguous().clone()
        if compute_sweep:
            self.fc_s = torch.logspace(2.5, 4, 15).to(device)
            self.A_s = torch.linspace(-80, -5, 12).to(device)
            if rid:
                data_norms = torch.zeros((self.nb_steps, self.fc_s.shape[0], self.A_s.shape[0]))
                data_grads = torch.zeros((self.nb_steps, self.fc_s.shape[0], self.A_s.shape[0], 2))
        if rid:
            data_denoised = torch.zeros((self.nb_steps, shape[0], shape[1]))
            data_filters = torch.zeros((self.nb_steps, *filter_params.shape))

        if self.start_sigma is None:
            t = self.diff_params.create_schedule(self.nb_steps).to(device)
            x = self._initial_state(shape, device, t[0]) if init_x is None else init_x.to(device)
        else:
            t = self.diff_params.create_schedule_from_initial_t(self.start_sigma, self.nb_steps).to(device)
            x = self._initial_state(shape, device, t[0], y) if init_x is None else init_x.to(device)
        gamma = self.diff_params.get_gamma(t).to(device)
        t_host = t.cpu()
        n_steps = self.nb_steps if max_steps is None else min(start_step + max_steps, self.nb_steps)

        use_step_graph = (self.step_graph and y.is_cuda and not compute_sweep and not self.joint
                          and not self.cuda_graph
                          and args.tester.posterior_sampling.SNR_observations == "None"
                          and not args.tester.blind_bwe.sigma_den_estimate)
        if use_step_graph:
            try:
                self._step_graph_for(y, filter_params, True)
                self._step_graph_for(y, filter_params, False)
            except Exception as exc:                       # noqa: BLE001 - any capture problem: stay eager
                warnings.warn(f"CUDA-graph capture of the sampler step failed ({exc!r}); running it eagerly")
                use_step_graph = False
                self._step_graphs = {}
        if use_step_graph:
            Snoise = 1
            for i in range(start_step, n_steps):
                heun = float(t_host[i + 1]) != 0 and self.order == 2
                st = self._step_graphs[heun]
                if i == start_step:
                    for sg in self._step_graphs.values():
                        sg.fp.copy_(filter_params)
                        if self._keyed is not None:
                            sg.seeds.copy_(self._keyed.seeds)
                st.x.copy_(x)
                if self._keyed is not None:
                    st.draw.fill_(1 + 8 * i)               # the noise is generated inside the step
                else:
                    st.eps.copy_(self._randn(shape, device) * Snoise, non_blocking=True)
                st.t_i.copy_(t[i]); st.gamma.copy_(gamma[i]); st.t_next.copy_(t[i + 1])
                st.graph.replay()
                profiling.add_launches(st.launches)
                x, filter_params = st.x, st.fp
                other = self._step_graphs[not heun]
                if other is not st:
                    other.fp.copy_(st.fp)
                if rid:
                    data_denoised[i] = st.den
                    data_filters[i] = st.fp_mid
                if step_hook is not None:
                    step_hook(i, x, filter_params)
            x, filter_params = x.clone(), filter_params.clone()
            n_steps = start_step                           # the eager loop below has nothing left to do

        for i in range(start_step, n_steps):
            self._keyed_step(i)
            x_hat, t_hat = self.move_timestep(x, t[i], gamma[i])
            score, filter_params, x_den_2 = self._evaluate(x_hat, t_hat, y, filter_params)
            if compute_sweep:
                norms, grads = self.compute_sweep(x_den_2, y)
            d = -t_hat * score
            if rid:
                data_denoised[i] = x_den_2
                data_filters[i] = filter_params
                if compute_sweep:
                    data_norms[i] = norms
                    data_grads[i] = grads
            h = t[i + 1] - t_hat
            if float(t_host[i + 1]) != 0 and self.order == 2:
                t_prime = t[i + 1]
                x_prime = x_hat + h * d
                score, filter_params, _ = self._evaluate(x_prime, t_prime, y, filter_params, slot=4)
                d_prime = -t_prime * score
                x = x_hat + h * ((1 / 2) * d + (1 / 2) * d_prime)
            else:
                x = x_hat + h * d
            if step_hook is not None:
                step_hook(i, x, filter_params)

        self._keyed = None
        self._groups = None
        if rid:
            out = (x.detach(), filter_params.detach(), data_denoised.detach(), t.detach(), data_filters.detach())
            if compute_sweep:
                out = out + (data_norms.detach(), data_grads.detach())
            return out
        return x.detach(), filter_params.detach()

    def predict_unconditional(self, shape, device, rid=False):
        """testing/blind_bwe_sampler.py:366-374,406-497 with y = None."""
        self._no_groups("predict_unconditional")
        self._keyed_begin(shape[0], device)
        t = self.diff_params.create_schedule(self.nb_steps).to(device)
        x = self._initial_state(shape, device, t[0])
        gamma = self.diff_params.get_gamma(t).to(device)
        t_host = t.cpu()
        if rid:
            data_denoised = torch.zeros((self.nb_steps, shape[0], shape[1]))
            data_score = torch.zeros((self.nb_steps, shape[0], shape[1]))
        for i in range(self.nb_steps):
            self._keyed_step(i)
            x_hat, t_hat = self.move_timestep(x, t[i], gamma[i], self.diff_params.Snoise)
            with torch.no_grad():
                score = (self.get_denoised_estimate(x_hat, t_hat) - x_hat) / t_hat ** 2
            d = -t_hat * score
            if rid:
                data_denoised[i] = score * t_hat ** 2 + x_hat
                data_score[i] = score
            h = t[i + 1] - t_hat
            if float(t_host[i + 1]) != 0 and self.order == 2:
                t_prime = t[i + 1]
                x_prime = x_hat + h * d
                with torch.no_grad():
                    score = (self.get_denoised_estimate(x_prime, t_prime) - x_prime) / t_prime ** 2
                x = x_hat + h * ((1 / 2) * d + (1 / 2) * (-t_prime * score))
            else:
                x = x_hat + h * d
        self._keyed = None
        if rid:
            return x.detach(), data_denoised.detach(), data_score.detach(), t.detach()
        return x.detach()

    # -- generic (non-blind) conditional sampling: any differentiable degradation ----------------
    @staticmethod
    def denoised2score(x_d0, x, t):
        """testing/blind_bwe_sampler.py:503-505 (Tweedie)."""
        return (x_d0 - x) / t ** 2

    @staticmethod
    def score2denoised(score, x, t):
        """testing/blind_bwe_sampler.py:506-507."""
        return score * t ** 2 + x

    def apply_FIR_filter(self, y):
        """testing/blind_bwe_sampler.py:211-218 on ``k_fir_filter`` (``self.filt``: the taps)."""
        from . import bandwidth_extension as bwe
        return bwe.apply_low_pass_firwin(y, self.filt)

    @staticmethod
    def prepare_smooth_mask(mask, size=10):
        """testing/blind_bwe_sampler.py:232-257: hann ramps of ``size`` samples at every transition of the
        first row's mask (before a gap: falling half, after a gap: rising half); all rows get that mask."""
        hann = torch.hann_window(size * 2)
        left, right = hann[:size].to(mask), hann[size:].to(mask)
        B = mask.shape[0]
        m = mask[0]
        new = m.clone()
        mh = m.detach().cpu()
        change = torch.nonzero(mh[1:] != mh[:-1]).reshape(-1) + 1
        if mh[0] != 1:                                   # the reference starts with prev = 1
            change = torch.cat((torch.zeros(1, dtype=change.dtype), change))
        for i in change.tolist():
            if mh[i] == 0:
                new[i - size:i] = right
            if mh[i] == 1:
                new[i:i + size] = left
        return new.unsqueeze(0).expand(B, -1)

    @classmethod
    def prepare_smooth_mask_rows(cls, mask, size=10):
        """``prepare_smooth_mask`` of every row of a (B, T) mask on its own (the per-row mode's windows differ)."""
        return torch.cat([cls.prepare_smooth_mask(mask[b:b + 1], size) for b in range(mask.shape[0])])

    def _generic_rec_grads(self, x_den, y, x_in, t_in, degradation, fused_params=None, known=None):
        """get_rec_grads (:75-135) for an arbitrary differentiable degradation (2-norm branch); a parametric
        fc_A filter (``fused_params``) takes the fused design + filter + residual-norm kernels, with ``known`` through
        the known-prefix masked operator.  With ``filter_per_row`` every row gets its own normaliser."""
        ps = self.args.tester.posterior_sampling
        if ps.SNR_observations != "None" or ps.stft_distance.use or ps.norm not in (1, 2, "fro"):
            raise NotImplementedError("generic degradations support the plain 1-/2-norm guidance")
        if fused_params is not None and ps.norm == 2:
            norm = rec_guidance_norms(x_den, y, self.freqs, fused_params, self.args.tester.blind_bwe.NFFT, known)
        else:
            norm = torch.linalg.norm(y - degradation(x_den), dim=1, ord=ps.norm)
        (g,) = torch.autograd.grad(outputs=norm.sum(), inputs=x_in)
        if self.filter_per_row:
            normguide = torch.linalg.norm(g, dim=1, keepdim=True) / self.args.exp.audio_len ** 0.5
        else:
            normguide = torch.linalg.norm(g) / self.args.exp.audio_len ** 0.5
        return self.xi / (normguide + 1e-6) * g / t_in

    def get_score(self, x, y, t_i, degradation, dc_step=None, fused_params=None, known=None):
        """testing/blind_bwe_sampler.py:160-209.  ``dc_step(x_hat)``: optional data-consistency step."""
        if y is None:
            with torch.no_grad():
                return self.denoised2score(self.get_denoised_estimate(x, t_i), x, t_i)
        if self.xi > 0:
            x = x.detach().requires_grad_(True)
            x_den = self.get_denoised_estimate(x, t_i)
            rec = self._generic_rec_grads(x_den, y, x, t_i, degradation, fused_params, known)
            x = x.detach()
            score = self.denoised2score(x_den.detach(), x, t_i) - rec
            if dc_step is not None:
                score = self.denoised2score(dc_step(self.score2denoised(score, x, t_i)), x, t_i)
            return score
        with torch.no_grad():
            x_hat = self.diff_params.denoiser(x, self.model, t_i.unsqueeze(-1))     # :192 (no DC/Nyquist filter)
            if dc_step is not None:
                x_hat = dc_step(x_hat)
            return self.denoised2score(x_hat, x, t_i)

    def predict_conditional(self, y, degradation, rid=False, dc_step=None, fused_params=None, known=None):
        """testing/blind_bwe_sampler.py:387-497 (``predict`` with observations y)."""
        self._no_groups("predict_conditional")
        shape, device = y.shape, y.device
        self._keyed_begin(shape[0], device)
        if self.start_sigma is None:
            t = self.diff_params.create_schedule(self.nb_steps).to(device)
            x = self._initial_state(shape, device, t[0])
        else:
            t = self.diff_params.create_schedule_from_initial_t(self.start_sigma, self.nb_steps).to(device)
            x = self._initial_state(shape, device, t[0], y)
        gamma = self.diff_params.get_gamma(t).to(device)
        t_host = t.cpu()
        if rid:
            data_denoised = torch.zeros((self.nb_steps, shape[0], shape[1]))
            data_score = torch.zeros((self.nb_steps, shape[0], shape[1]))
        for i in range(self.nb_steps):
            self._keyed_step(i)
            x_hat, t_hat = self.move_timestep(x, t[i], gamma[i], self.diff_params.Snoise)
            score = self.get_score(x_hat, y, t_hat, degradation, dc_step, fused_params, known)
            d = -t_hat * score
            if rid:
                data_denoised[i] = self.score2denoised(score, x_hat, t_hat)
                data_score[i] = score
            h = t[i + 1] - t_hat
            if float(t_host[i + 1]) != 0 and self.order == 2:
                t_prime = t[i + 1]
                x_prime = x_hat + h * d
                score = self.get_score(x_prime, y, t_prime, degradation, dc_step, fused_params, known)
                x = x_hat + h * ((1 / 2) * d + (1 / 2) * (-t_prime * score))
            else:
                x = x_hat + h * d
        self._keyed = None
        if rid:
            return x.detach(), data_denoised.detach(), data_score.detach(), t.detach()
        return x.detach()

    def predict_bwe_AR(self, ylpf, y_masked, filt, filt_type, rid=False, test_filter_fit=False,
                       compute_sweep=False, mask=None):
        """testing/blind_bwe_sampler.py:259-303: bandwidth extension of a segment whose head (mask = 1)
        is already known from the previous segment: y = mask y_masked + (1 - mask) ylpf, degradation
        x -> mask x + (1 - mask) A(x); with ``complete_recording.inpaint_DC`` the known part is also
        enforced by a data-consistency step through a hann-smoothed mask.

        With ``filter_per_row`` the rows are independent windows: ``filt`` is (2, K) (every row) or (B, 2, K), the
        (B, T) mask may differ per row and each row gets its own smoothed mask and guidance normaliser."""
        assert mask is not None
        self._no_groups("predict_bwe_AR")
        if test_filter_fit or compute_sweep:
            raise NotImplementedError("test_filter_fit / compute_sweep logging on the AR path")
        if self.filter_per_row:
            return self._predict_bwe_AR_rows(ylpf, y_masked, filt, filt_type, rid, mask)
        device = ylpf.device
        mask = mask.to(device)
        if filt_type == "fc_A":
            self.freqs = torch.fft.rfftfreq(self.args.tester.blind_bwe.NFFT, d=1 / self.args.exp.sample_rate).to(device)
            self.params = filt.to(device)
            lowpass = lambda x: self.apply_filter_fcA(x, self.params)
        elif filt_type == "firwin":
            self.filt = filt.to(device)
            lowpass = self.apply_FIR_filter
        else:
            raise NotImplementedError(filt_type)
        y = mask * y_masked + (1 - mask) * ylpf
        degradation = lambda x: mask * x + (1 - mask) * lowpass(x)
        dc_step = None
        if self.args.tester.complete_recording.inpaint_DC:
            smooth = self.prepare_smooth_mask(mask, 50)
            y_smooth = smooth * y_masked
            dc_step = lambda x_hat: y_smooth + x_hat - smooth * x_hat     # data_consistency_step_classic (:63-73)
        return self.predict_conditional(y, degradation, rid, dc_step)

    def _predict_bwe_AR_rows(self, ylpf, y_masked, filt, filt_type, rid, mask):
        """predict_bwe_AR with ``filter_per_row``.  When every mask row is a 0/1 known prefix (what the
        autoregressive driver builds) the 2-norm guidance runs through the masked fused kernel pair; any other mask
        keeps the eager composition on the per-row filter."""
        if filt_type != "fc_A":
            raise NotImplementedError(f"filter_per_row with filt_type {filt_type!r}: only the parametric fc_A filter "
                                      "has per-row kernels (the FIR kernel shares its taps over the rows)")
        device = ylpf.device
        B, T = ylpf.shape
        params = filt.to(device)
        if params.dim() == 2:
            params = params.unsqueeze(0).expand(B, -1, -1)
        if params.dim() != 3 or params.shape[0] != B or params.shape[1] != 2:
            raise ValueError(f"per-row filter parameters must be (2, K) or ({B}, 2, K), got {tuple(filt.shape)}")
        self.freqs = torch.fft.rfftfreq(self.args.tester.blind_bwe.NFFT, d=1 / self.args.exp.sample_rate).to(device)
        self.params = params = params.contiguous()
        mask = mask.to(device).expand(B, T)
        y = mask * y_masked + (1 - mask) * ylpf
        degradation = lambda x: mask * x + (1 - mask) * self.apply_filter_fcA(x, params)
        known = known_prefix_lengths(mask)
        if known is not None:
            known = known.to(device)
        dc_step = None
        if self.args.tester.complete_recording.inpaint_DC:
            smooth = self.prepare_smooth_mask_rows(mask, 50)
            y_smooth = smooth * y_masked
            dc_step = lambda x_hat: y_smooth + x_hat - smooth * x_hat
        return self.predict_conditional(y, degradation, rid, dc_step, fused_params=None if known is None else params,
                                        known=known)

    def predict_bwe(self, ylpf, filt, filt_type, rid=False, test_filter_fit=False, compute_sweep=False):
        """testing/blind_bwe_sampler.py:306-364: non-blind bandwidth extension with a KNOWN observation model,
        routed like the reference through ``predict_conditional`` / ``get_score`` (:160-209, 387-497): with
        ``rid`` the tuple (x, data_denoised, data_score, t) is returned, ``posterior_sampling.data_consistency``
        applies the classic data-consistency step and xi == 0 uses the plain denoiser.  ``fc_A`` (parametric filter,
        fused design + STFT filter guidance) and the FIR models run on the CUDA operators; the IIR / biquad /
        resampling models and the logging-only ``test_filter_fit`` / ``compute_sweep`` flags raise."""
        self._no_groups("predict_bwe")
        if filt_type not in ("fc_A", "firwin", "firwin_hpf"):
            raise NotImplementedError(f"filt_type {filt_type!r}: 'fc_A', 'firwin' and 'firwin_hpf' run on the "
                                      "CUDA operators; the IIR / resampling models are outside this path")
        if test_filter_fit or compute_sweep:
            raise NotImplementedError("test_filter_fit / compute_sweep logging on the non-blind path")
        if self.filter_per_row and filt_type != "fc_A":
            raise NotImplementedError(f"filter_per_row with filt_type {filt_type!r}: only the parametric fc_A filter "
                                      "has per-row kernels (the FIR kernel shares its taps over the rows)")
        args = self.args
        device = ylpf.device
        fused = None
        if filt_type == "fc_A":
            self.freqs = torch.fft.rfftfreq(args.tester.blind_bwe.NFFT, d=1 / args.exp.sample_rate).to(device)
            self.params = filt.to(device)
            degradation = lambda x: self.apply_filter_fcA(x, self.params)
            fused = self.params
        else:
            self.filt = filt.to(device)
            degradation = self.apply_FIR_filter
        dc_step = None
        if self.data_consistency:                     # data_consistency_step_classic (:63-73) inside get_score (:182-204)
            dc_step = lambda x_hat: ylpf + x_hat - degradation(x_hat)
        return self.predict_conditional(ylpf, degradation, rid, dc_step, fused_params=fused)
