"""Test helper: the reference's blind sampling loop written against ``utils.blind_bwe_utils`` BY NAME, the way
testing/blind_bwe_sampler.py:9 imports it -- so that after ``babe_b200.install()`` every operator call lands on the
CUDA drop-ins through the reference's own call pattern (apply_stft on both signals, design_filter inside the
closure, autograd.grad(create_graph=True) on the weighted STFT-magnitude norm, in-place sequential clamps,
apply_filter inside the guidance graph, autograd.grad wrt the noisy input through the denoiser).  Default branches of
conf/tester/blind_bwe.yaml only.  On the CPU the same loop runs on the oracle operators and must reproduce the golden
of the unmodified BlindSampler (tests/test_integration_cpu.py), which is what validates this restatement; with
BABE_REFERENCE set it also runs on the reference's own module."""
import torch


def fit_params(bu, args, freqs, denoised_estimate, y, filter_params):
    """testing/blind_bwe_sampler.py:533-595."""
    o = args.tester.blind_bwe.optimization
    nfft = args.tester.blind_bwe.NFFT
    fcmax = args.exp.sample_rate // 2 if args.tester.blind_bwe.fcmax == "nyquist" else args.tester.blind_bwe.fcmax
    fcmin, Amin, Amax = args.tester.blind_bwe.fcmin, args.tester.blind_bwe.Amin, args.tester.blind_bwe.Amax
    mu = torch.Tensor([o.mu[0], o.mu[1]]).to(y.device)
    Xden = bu.apply_stft(denoised_estimate, nfft)
    Y = bu.apply_stft(y, nfft)
    for i in range(o.max_iter):
        filter_params.requires_grad = True
        H = bu.design_filter(filter_params[0], filter_params[1], freqs)
        norm = bu.apply_filter_and_norm_STFTmag_fweighted(Xden, Y, H, args.tester.posterior_sampling.freq_weighting_filter)
        grad = torch.autograd.grad(norm, filter_params, create_graph=True)
        filter_params = filter_params - mu.unsqueeze(1) * grad[0]
        filter_params.detach_()
        if o.clamp_fc:
            filter_params[0, 0] = torch.clamp(filter_params[0, 0], min=fcmin, max=fcmax)
            for k in range(1, len(filter_params[0])):
                filter_params[0, k] = torch.clamp(filter_params[0, k], min=filter_params[0, k - 1] + 1, max=fcmax)
        if o.clamp_A:
            filter_params[1, 0] = torch.clamp(filter_params[1, 0], min=Amin, max=-1 if o.only_negative_A else Amax)
            for k in range(1, len(filter_params[0])):
                filter_params[1, k] = torch.clamp(filter_params[1, k], min=Amin,
                                                  max=filter_params[1, k - 1] if o.only_negative_A else Amax)
        if i > 0:
            if (torch.abs(filter_params[0] - prev[0]).mean() < o.tol[0]) and \
                    (torch.abs(filter_params[1] - prev[1]).mean() < o.tol[1]):
                break
        prev = filter_params.clone().detach()
    return filter_params


def rec_grads(bu, args, freqs, x_den, y, x, t_i, filter_params):
    """testing/blind_bwe_sampler.py:75-135, norm 2."""
    H = bu.design_filter(filter_params[0], filter_params[1], freqs)
    den_rec = bu.apply_filter(x_den, H, args.tester.blind_bwe.NFFT)
    norm = torch.linalg.norm(y - den_rec, dim=1, ord=2)
    g = torch.autograd.grad(outputs=norm.sum(), inputs=x)[0]
    normguide = torch.linalg.norm(g) / args.exp.audio_len ** 0.5
    return args.tester.posterior_sampling.xi / (normguide + 1e-6) * g / t_i


def predict_blind_bwe(bu, model, diff_params, args, y, randn=torch.randn, trace=None):
    """testing/blind_bwe_sampler.py:619-769 (rid False, no sweep, no data consistency)."""
    device = y.device
    if not args.tester.diff_params.same_as_training:                 # BlindSampler.__init__ / update_diff_params (:28-60)
        d, s = diff_params, args.tester.diff_params
        d.sigma_min, d.sigma_max, d.ro, d.sigma_data = s.sigma_min, s.sigma_max, s.ro, s.sigma_data
        d.Schurn, d.Stmin, d.Stmax, d.Snoise = s.Schurn, s.Stmin, s.Stmax, s.Snoise
    freqs = torch.fft.rfftfreq(args.tester.blind_bwe.NFFT, d=1 / args.exp.sample_rate).to(device)
    filter_params = torch.Tensor([args.tester.blind_bwe.initial_conditions.fc,
                                  args.tester.blind_bwe.initial_conditions.A]).to(device)
    T = args.tester.T
    t = diff_params.create_schedule_from_initial_t(args.tester.posterior_sampling.start_sigma, T).to(device)
    x = y + randn(y.shape).to(device) * t[0]
    gamma = diff_params.get_gamma(t).to(device)

    def evaluate(x_in, t_in, filter_params):
        x_in.requires_grad_(True)
        x_den = diff_params.denoiser(x_in, model, t_in.unsqueeze(-1))
        if args.tester.filter_out_cqt_DC_Nyq:
            x_den = model.CQTransform.apply_hpf_DC(x_den)
        x_den_2 = x_den.clone().detach()
        filter_params = fit_params(bu, args, freqs, x_den_2, y, filter_params)
        rg = rec_grads(bu, args, freqs, x_den, y, x_in, t_in, filter_params)
        x_in.detach_()
        return (x_den_2 - x_in) / t_in ** 2 - rg, filter_params, x_den_2

    for i in range(T):
        t_hat = t[i] + gamma[i] * t[i]
        x_hat = x + ((t_hat ** 2 - t[i] ** 2) ** (1 / 2)) * randn(x.shape).to(device)
        score, filter_params, x_den_2 = evaluate(x_hat, t_hat, filter_params)
        d = -t_hat * score
        h = t[i + 1] - t_hat
        if t[i + 1] != 0 and args.tester.order == 2:
            x_prime = x_hat + h * d
            score, filter_params, _ = evaluate(x_prime, t[i + 1], filter_params)
            x = x_hat + h * ((1 / 2) * d + (1 / 2) * (-t[i + 1] * score))
        else:
            x = x_hat + h * d
        if trace is not None:
            trace.append((x.detach().clone(), filter_params.detach().clone(), x_den_2.clone()))
    return x.detach(), filter_params.detach()
