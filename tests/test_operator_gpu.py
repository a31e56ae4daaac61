"""GPU parity: the CUDA operator (through the C ABI and the drop-in module)
against the oracle on identical seeded inputs, against the golden vectors the
reference produced, and -- at full BASELINE sizes -- through size-independent
properties.  Tolerance: relative L2 <= 1e-5 in fp32 (BASELINE.json north_star)
unless a test states otherwise."""
import numpy as np
import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu

TOL = 1e-5


@pytest.fixture(scope="module")
def bu():
    from babe_b200 import build
    build.build()
    from babe_b200 import blind_bwe_utils
    return blind_bwe_utils


@pytest.fixture(scope="module")
def sf():
    from oracle import stft_filter
    return stft_filter


def cuda(a):
    return torch.as_tensor(np.asarray(a)).cuda()


def make_H(sf, nfft, sr=22050):
    f = torch.fft.rfftfreq(nfft, d=1 / sr)
    return f, sf.design_filter(torch.tensor([500.0, 1500.0, 4000.0]), torch.tensor([-10.0, -25.0, -40.0]), f)


# --------------------------------------------------------------------------- golden
@pytest.mark.parametrize("tag", ["n1024", "n4096"])
def test_golden_forward_and_grads(bu, golden, tag):
    g = golden(f"operator_{tag}.npz")
    nfft = int(g["nfft"])
    x, f, fc, A, H = cuda(g["x"]), cuda(g["f"]), cuda(g["fc"]), cuda(g["A"]), cuda(g["H"])
    assert rel_l2(bu.design_filter(fc, A, f).cpu(), g["H"]) < TOL
    assert rel_l2(bu.design_filter(cuda(g["fc_dup"]), cuda(g["A_dup"]), f).cpu(), g["H_dup"]) < TOL
    assert rel_l2(bu.design_filter(torch.tensor(1000.0).cuda(), torch.tensor(-20.0).cuda(), f).cpu(),
                  g["H_scalar"]) < TOL
    assert rel_l2(bu.design_filter([1000.0], [-20.0], f).cpu(), g["H_list"]) < TOL
    assert rel_l2(bu.design_filter_G(fc, A, torch.tensor(-3.0).cuda(), f).cpu(), g["H_G"]) < TOL
    X = bu.apply_stft(x, nfft)
    assert tuple(X.shape) == g["X"].shape
    assert rel_l2(X.cpu(), g["X"]) < TOL
    assert rel_l2(bu.apply_filter(x, H, nfft).cpu(), g["y"]) < TOL
    y2 = bu.apply_filter_istft(cuda(g["X"]), H, nfft)
    assert tuple(y2.shape) == g["istft"].shape
    assert rel_l2(y2.cpu(), g["istft"]) < TOL
    # gradients of <apply_filter(x,H), r> wrt x and H (autograd of the reference)
    r = cuda(g["r"])
    xg = x.clone().requires_grad_(True)
    Hg = H.clone().requires_grad_(True)
    gx, gH = torch.autograd.grad((bu.apply_filter(xg, Hg, nfft) * r).sum(), (xg, Hg))
    assert rel_l2(gx.cpu(), g["gx"]) < TOL
    assert rel_l2(gH.cpu(), g["gH"]) < 5e-5
    # design_filter VJP
    fcg, Ag = fc.clone().requires_grad_(True), A.clone().requires_grad_(True)
    gfc, gA = torch.autograd.grad((bu.design_filter(fcg, Ag, f) * cuda(g["cotH"])).sum(), (fcg, Ag))
    assert rel_l2(gfc.cpu(), g["gfc"]) < 5e-5
    assert rel_l2(gA.cpu(), g["gA"]) < 5e-5
    # rec-guidance operator part through autograd of the drop-in
    yobs = cuda(g["yobs"])
    xg = x.clone().requires_grad_(True)
    nb = torch.linalg.norm(yobs - bu.apply_filter(xg, H, nfft), dim=1, ord=2)
    (gg,) = torch.autograd.grad(nb.sum(), xg)
    assert rel_l2(nb.detach().cpu(), g["rg_norms"]) < TOL
    assert rel_l2(gg.cpu(), g["rg_grad"]) < 2e-5


@pytest.mark.parametrize("tag", ["n1024", "n4096"])
def test_golden_losses(bu, golden, tag):
    g = golden(f"operator_{tag}.npz")
    nfft = int(g["nfft"])
    x, H, yobs = cuda(g["x"]), cuda(g["H"]), cuda(g["yobs"])
    X, Y = bu.apply_stft(x, nfft), bu.apply_stft(yobs, nfft)
    for wk in ["linear", "None", "log", "sqrt", "cubic", "quadratic", "logcubic", "logquadratic", "squared"]:
        for name, val in (("norm_fw_", bu.apply_filter_and_norm_STFTmag_fweighted(X, Y, H, wk)),
                          ("norm_stft_", bu.apply_norm_STFT_fweighted(yobs, x, wk, nfft)),
                          ("norm_mag_", bu.apply_norm_STFTmag_fweighted(yobs, x, wk, nfft))):
            ref = float(g[name + wk])
            assert abs(float(val) - ref) < 2e-5 * ref, (name, wk)
    ref = float(g["norm_logmag_sqrt"])
    assert abs(float(bu.apply_norm_STFTmag_fweighted(yobs, x, "linear", nfft, logmag=True)) - ref) < 1e-4 * ref
    ref = float(g["norm_plain"])
    assert abs(float(bu.apply_filter_and_norm_STFTmag(X, Y, H)) - ref) < 2e-5 * ref
    assert abs(float(bu.apply_norm_filter(H, cuda(g["H_G"]))) - float(g["norm_filter"])) < 1e-6
    # fit-loss gradients wrt (fc, A) and H exactly as the sampler takes them
    f = cuda(g["f"])
    fcg, Ag = cuda(g["fc"]).requires_grad_(True), cuda(g["A"]).requires_grad_(True)
    Hh = bu.design_filter(fcg, Ag, f)
    Hh.retain_grad()
    nrm = bu.apply_filter_and_norm_STFTmag_fweighted(X, Y, Hh, "sqrt")
    g1, g2, g3 = torch.autograd.grad(nrm, (fcg, Ag, Hh), create_graph=True)
    assert rel_l2(g3.cpu(), g["fit_gH"]) < 5e-5
    assert rel_l2(g1.detach().cpu(), g["fit_gfc"]) < 1e-4
    assert rel_l2(g2.detach().cpu(), g["fit_gA"]) < 1e-4


def test_design_filter_index_error(bu):
    f = torch.fft.rfftfreq(1024, d=1 / 22050).cuda()
    with pytest.raises(IndexError):
        bu.design_filter(torch.tensor([100.0, 20000.0]).cuda(), torch.tensor([-5.0, -9.0]).cuda(), f)
    # fc_0 above the last bin is legal in the reference (H = 1 everywhere)
    H = bu.design_filter(torch.tensor([20000.0]).cuda(), torch.tensor([-5.0]).cuda(), f)
    assert torch.equal(H.cpu(), torch.ones(513))


# --------------------------------------------------------------------------- oracle, seeded
@pytest.mark.parametrize("nfft", [512, 1024, 2048, 4096])
@pytest.mark.parametrize("B,T", [(1, 1), (1, 300), (3, 4096), (2, 12289), (5, 40000)])
def test_apply_filter_vs_oracle(bu, sf, nfft, B, T):
    torch.manual_seed(nfft + B + T)
    x = torch.randn(B, T) * 0.063
    f, H = make_H(sf, nfft)
    y = bu.apply_filter(x.cuda(), H.cuda(), nfft).cpu()
    assert y.shape == x.shape
    assert rel_l2(y, sf.apply_filter(x, H, nfft)) < TOL
    ya = bu._FilterOp.apply(x.cuda(), H.cuda(), nfft, True).cpu()
    assert rel_l2(ya, sf.apply_filter_adjoint(x, H, nfft)) < TOL


@pytest.mark.parametrize("nfft", [1024, 4096])
def test_fused_design_and_epilogues(bu, sf, nfft):
    """In-kernel filter design and the guidance epilogues (residual + sum of squares, adjoint with row scale) against
    the oracle.  At NFFT 4096, T = 30012 runs them on k_filter_fused (<false, 1> and <true, 2>); T = 30011 cannot be
    bulk-copied and runs the round-1 k_apply_filter, as does every NFFT 1024 call."""
    from babe_b200 import ops
    from kernel_trace import assert_path, filter_variants, launched
    for T in (30011, 30012):
        torch.manual_seed(5)
        B = 4
        x, yobs = torch.randn(B, T) * 0.05, torch.randn(B, T) * 0.05
        f = torch.fft.rfftfreq(nfft, d=1 / 22050)
        fc, A = torch.tensor([300.0, 310.0, 900.0, 5000.0]), torch.tensor([-12.0, -14.0, -30.0, -31.0])
        H = sf.design_filter(fc, A, f)
        with launched() as names:
            y = ops.apply_filter(x.cuda(), nfft, freqs=f.cuda(), fc=fc.cuda(), A=A.cuda())
            ss = torch.zeros(B, dtype=torch.float64, device="cuda")
            r = ops.apply_filter(x.cuda(), nfft, freqs=f.cuda(), fc=fc.cuda(), A=A.cuda(), sub=yobs.cuda(),
                                 row_sumsq=ss)
            scale = (1.0 / torch.sqrt(ss)).float()
            g = ops.apply_filter(r, nfft, freqs=f.cuda(), fc=fc.cuda(), A=A.cuda(), adjoint=True, row_scale=scale)
        fused = nfft == 4096 and T % 4 == 0
        assert_path(names, fused=fused, kernel="k_filter_fused" if fused else "k_apply_filter")
        if fused:
            assert filter_variants(names) == {(False, 0, False), (False, 1, False), (True, 2, False)}
        assert rel_l2(y.cpu(), sf.apply_filter(x, H, nfft)) < TOL
        r_ref = sf.apply_filter(x, H, nfft) - yobs
        assert rel_l2(r.cpu(), r_ref) < TOL
        assert rel_l2(ss.cpu(), (r_ref.double() ** 2).sum(1)) < TOL
        n_ref, g_ref = sf.rec_guidance_operator(x, yobs, H, nfft)
        assert rel_l2(torch.sqrt(ss).cpu(), n_ref) < TOL
        assert rel_l2(g.cpu(), g_ref) < 2e-5


@pytest.mark.parametrize("nfft", [512, 1024, 2048, 4096])
def test_stft_istft_stats_vs_oracle(bu, sf, nfft):
    from babe_b200 import ops
    torch.manual_seed(nfft)
    B, T = 3, 5 * nfft + 77
    x, y = torch.randn(B, T), torch.randn(B, T) * 0.3
    f, H = make_H(sf, nfft)
    X = bu.apply_stft(x.cuda(), nfft)
    Xo = sf.apply_stft(x, nfft)
    assert tuple(X.shape) == tuple(Xo.shape)
    assert rel_l2(X.cpu(), Xo) < TOL
    assert rel_l2(bu.apply_filter_istft(Xo.cuda(), H.cuda(), nfft).cpu(), sf.apply_filter_istft(Xo, H, nfft)) < TOL
    abc = ops.stft_stats(x.cuda(), y.cuda(), nfft).cpu()
    a, b, c = sf.stft_mag_stats(x.double(), y.double(), nfft)
    assert rel_l2(abc[0], a) < TOL and rel_l2(abc[1], b) < TOL and rel_l2(abc[2], c) < TOL
    st = ops.spec_mag_stats(X, bu.apply_stft(y.cuda(), nfft)).cpu()
    assert rel_l2(st[0], a) < TOL and rel_l2(st[1], b) < TOL and rel_l2(st[2], c) < TOL
    # autograd of the unfused signatures against autograd of the oracle
    xg = x.clone().requires_grad_(True)
    cot = torch.randn_like(Xo)
    (go,) = torch.autograd.grad((sf.apply_stft(xg, nfft) * cot).sum(), xg)
    xc = x.cuda().requires_grad_(True)
    (gc,) = torch.autograd.grad((bu.apply_stft(xc, nfft) * cot.cuda()).sum(), xc)
    assert rel_l2(gc.cpu(), go) < TOL
    Xg, Hg = Xo.clone().requires_grad_(True), H.clone().requires_grad_(True)
    yo = sf.apply_filter_istft(Xg, Hg, nfft)
    cot = torch.randn_like(yo)
    goX, goH = torch.autograd.grad((yo * cot).sum(), (Xg, Hg))
    Xc, Hc = Xo.cuda().requires_grad_(True), H.cuda().requires_grad_(True)
    gcX, gcH = torch.autograd.grad((bu.apply_filter_istft(Xc, Hc, nfft) * cot.cuda()).sum(), (Xc, Hc))
    # irfft ignores Im of DC/Nyquist; the oracle's autograd agrees
    assert rel_l2(gcX.cpu(), goX) < TOL
    assert rel_l2(gcH.cpu(), goH) < 5e-5
    # H fixed (the guidance case): its response rides in the STFT kernel's per-bin scale
    Xc2 = Xo.cuda().requires_grad_(True)
    (gcX2,) = torch.autograd.grad((bu.apply_filter_istft(Xc2, H.cuda(), nfft) * cot.cuda()).sum(), Xc2)
    assert rel_l2(gcX2.cpu(), goX) < TOL


def test_fit_params_vs_oracle(golden):
    """Short runs against the reference golden (tight); the full 100 iterations
    against the fp64 oracle (tight) and the fp32 golden (loose) -- see
    tests/test_oracle_golden.py::test_fit_params for why."""
    from babe_b200 import ops, sampler
    from oracle import filter_fit as ofit, stft_filter as osf
    g = golden("fit_sampler.npz")
    nfft, sr = int(g["nfft"]), int(g["sr"])
    xden, y, p0 = cuda(g["fit_xden"]), cuda(g["y"]), cuda(g["fit_p0"])
    for iters, tol in ((1, 1e-5), (5, 1e-5), (100, 3e-2)):
        fit = sampler.FilterFit(nfft=nfft, sample_rate=sr, max_iter=iters, device="cuda")
        p = fit(xden, y, p0.clone())
        assert rel_l2(p.cpu(), g[f"fit_p_{iters}"]) < tol, iters
    cfg = ofit.FitConfig(nfft=nfft, sample_rate=sr)
    a, b, c = osf.stft_mag_stats(xden.cpu().double(), y.cpu().double(), nfft)
    s64, it64 = ofit.fit_params_from_stats(a, b, c, p0.cpu().double(), cfg, dtype=torch.float64)
    fit = sampler.FilterFit(nfft=nfft, sample_rate=sr, max_iter=100, device="cuda")
    p, iters = fit(xden, y, p0.clone(), return_iters=True)
    assert int(iters) == it64
    # params are fp32 in the reference and in the kernel: the fp32 trajectory is
    # pinned by the oracle's fp32 run, the fp64 one only bounds the drift
    s32, _ = ofit.fit_params_from_stats(a.float(), b.float(), c.float(), p0.cpu(), cfg)
    assert rel_l2(p.cpu(), s32) < 1e-3
    assert rel_l2(p.cpu(), s64) < 1e-2
    p7 = fit(xden, y, cuda(g["fit7_p0"]).clone())
    assert rel_l2(p7.cpu(), g["fit7_p"]) < 3e-2


def test_fit_kernels_agree_bitwise(golden):
    """The two fit loops -- round 1's k_fit_params (-1), which also serves K > 8 and F > 4096, and the default 4-CTA
    cluster kernel k_fit_params3 (0: bins split over the CTAs, sums through distributed shared memory) -- evaluate the
    same fp32 / fp64 expressions; only the association of the fp64 sums over bins differs.  Their 100-iteration
    trajectories agree to the last bit on the goldens' inputs (K = 5, K = 7, NFFT 1024) and on a 4096-point case."""
    from babe_b200 import ops, sampler
    from babe_b200._lib import lib
    g = golden("fit_sampler.npz")
    nfft, sr = int(g["nfft"]), int(g["sr"])
    xden, y = cuda(g["fit_xden"]), cuda(g["y"])
    cases = [(nfft, xden, y, cuda(g["fit_p0"])), (nfft, xden, y, cuda(g["fit7_p0"]))]
    gen = torch.Generator().manual_seed(5)
    x4 = (torch.randn(2, 60000, generator=gen) * 0.063).cuda()
    f4 = torch.fft.rfftfreq(4096, d=1 / 22050).cuda()
    y4 = ops.apply_filter(x4, 4096, freqs=f4, fc=torch.tensor([1500.0]).cuda(), A=torch.tensor([-25.0]).cuda())
    cases.append((4096, x4, y4, torch.tensor([[280.0, 285, 290, 295, 300], [-15.0, -17, -20, -25, -30]]).cuda()))
    try:
        for n, xd, yy, p0 in cases:
            out = {}
            for v in (-1, 0):
                assert lib().babe_set_fit_variant(v) == 0
                fit = sampler.FilterFit(nfft=n, sample_rate=22050 if n == 4096 else sr, max_iter=100, device="cuda")
                p, its = fit(xd, yy, p0.clone(), return_iters=True)
                out[v] = (p.cpu(), int(its))
            assert out[0][1] == out[-1][1]
            assert torch.equal(out[0][0], out[-1][0])
    finally:
        lib().babe_set_fit_variant(0)


# --------------------------------------------------------------------------- full-size properties
@pytest.mark.parametrize("B,T,nfft", [(8, 184184, 4096), (2, 485100, 4096), (64, 184184, 4096), (3, 132300, 1024)])
def test_full_size_properties(bu, sf, B, T, nfft):
    torch.manual_seed(1)
    x = torch.randn(B, T, device="cuda") * 0.063
    g = torch.randn(B, T, device="cuda")
    f, H = make_H(sf, nfft)
    H = H.cuda()
    # identity filter reconstructs x (window / OLA / envelope bookkeeping)
    assert rel_l2(bu.apply_filter(x, torch.ones_like(H), nfft).cpu(), x.cpu()) < TOL
    # adjoint identity <A x, g> = <x, A^T g>
    Ax = bu.apply_filter(x, H, nfft)
    Atg = bu._FilterOp.apply(g, H, nfft, True)
    lhs, rhs = (Ax.double() * g.double()).sum(), (x.double() * Atg.double()).sum()
    assert abs(float(lhs - rhs)) < 1e-5 * abs(float(lhs))
    # linearity
    x2 = torch.randn(B, T, device="cuda") * 0.063
    lin = bu.apply_filter(0.5 * x - 2.0 * x2, H, nfft)
    assert rel_l2(lin.cpu(), (0.5 * Ax - 2.0 * bu.apply_filter(x2, H, nfft)).cpu()) < TOL
    # one row against the oracle
    assert rel_l2(Ax[:1].cpu(), sf.apply_filter(x[:1].cpu(), H.cpu(), nfft)) < TOL
    # statistics: checksum of checksums (Parseval on the windowed frames)
    from babe_b200 import ops
    abc = ops.stft_stats(x, g, nfft).cpu()
    a1, b1, c1 = sf.stft_mag_stats(x[:1].cpu().double(), g[:1].cpu().double(), nfft)
    abc1 = ops.stft_stats(x[:1], g[:1], nfft).cpu()
    assert rel_l2(abc1[0], a1) < TOL and rel_l2(abc1[1], b1) < TOL and rel_l2(abc1[2], c1) < TOL
    tot = sum(ops.stft_stats(x[i:i + 1], g[i:i + 1], nfft).cpu() for i in range(min(B, 8)))
    if B <= 8:
        assert rel_l2(abc, tot) < TOL


def test_fir_filter_golden_and_properties(golden):
    """SURVEY 8f-4: overlap-save FIR kernel vs the reference's conv1d golden, its autograd,
    and the adjoint identity at a benchmark-size batch."""
    from babe_b200 import bandwidth_extension as bwe, ops
    from oracle import fir
    g = golden("fir.npz")
    x = cuda(g["x"])
    for tag in ("lpf500", "hpf499"):
        taps = cuda(g["taps_" + tag])
        xg = x.clone().requires_grad_(True)
        y = bwe.apply_low_pass_firwin(xg, taps)
        assert rel_l2(y.detach().cpu(), g["y_" + tag]) < TOL
        (gx,) = torch.autograd.grad((y * cuda(g["r_" + tag])).sum(), xg)
        assert rel_l2(gx.cpu(), g["gx_" + tag]) < TOL
    torch.manual_seed(2)
    taps = cuda(g["taps_lpf500"]).reshape(-1)
    for B, T in ((1, 1), (3, 3597), (2, 7195), (8, 184184)):
        xb, gb = torch.randn(B, T, device="cuda"), torch.randn(B, T, device="cuda")
        yb = ops.fir_filter(xb, taps)
        if B * T < 30000:
            assert rel_l2(yb.cpu(), fir.apply_fir_same(xb.cpu(), taps.cpu())) < TOL
        lhs = (yb.double() * gb.double()).sum()
        rhs = (xb.double() * ops.fir_filter(gb, taps, adjoint=True).double()).sum()
        # <Ax, g> of random vectors is a cancelling sum: compare against its natural scale
        assert abs(float(lhs - rhs)) <= 1e-6 * float(yb.double().norm() * gb.double().norm()) + 1e-9


# --------------------------------------------------------------------------- a9 / a10: fused spectrogram distances
@pytest.mark.parametrize("nfft,T", [(1024, 16384), (4096, 65536)])
@pytest.mark.parametrize("wk", ["linear", "None", "sqrt", "logquadratic"])
def test_stft_distance_norms_and_gradients(bu, sf, nfft, T, wk):
    """apply_norm_STFT_fweighted / apply_norm_STFTmag_fweighted (utils/blind_bwe_utils.py:148-248): value and the
    gradient wrt the denoised estimate (what the STFT-guidance branch of get_score differentiates,
    testing/blind_bwe_sampler.py:99-115) -- k_spec_dist_stats / k_spec_dist_grad (+ k_spec_mag_* for the plain
    magnitude) against the oracle's autograd on the same inputs."""
    gen = torch.Generator().manual_seed(nfft + len(wk))
    x = torch.randn(3, T, generator=gen)
    y = x * 0.5 + 0.3 * torch.randn(3, T, generator=gen)
    cases = [("complex", lambda m, a, b: m.apply_norm_STFT_fweighted(a, b, wk, nfft), 2e-5),
             ("mag", lambda m, a, b: m.apply_norm_STFTmag_fweighted(a, b, wk, nfft), 2e-5),
             ("logmag", lambda m, a, b: m.apply_norm_STFTmag_fweighted(a, b, wk, nfft, True), 1e-4)]
    for name, fn, tol in cases:
        xo = x.clone().requires_grad_(True)
        ref = fn(sf, y, xo)
        (gref,) = torch.autograd.grad(ref, xo)
        xc = x.cuda().requires_grad_(True)
        val = fn(bu, y.cuda(), xc)
        (g,) = torch.autograd.grad(val, xc)
        assert abs(float(val.detach()) - float(ref.detach())) < tol * abs(float(ref.detach())), (name, wk)
        if name == "logmag":
            # d log10|X| = X / |X|^2: near-empty bins amplify the fp32 rounding of the STFT itself (the reference's own
            # fp32 gradient is 1e-4 from its fp64 evaluation at NFFT 4096), so the end-to-end gradient gets 1e-3 against
            # fp64 here and the kernels are held to 2e-5 on identical spectrograms in
            # test_spec_dist_kernels_on_given_spectrograms
            xd = x.double().requires_grad_(True)
            (g64,) = torch.autograd.grad(fn(sf, y.double(), xd), xd)
            assert rel_l2(g.cpu(), g64) < 1e-3, (name, wk, rel_l2(g.cpu(), g64), rel_l2(gref, g64))
        else:
            assert rel_l2(g.cpu(), gref) < tol, (name, wk, rel_l2(g.cpu(), gref))
    # gradient wrt the observation as well (both spectrograms require grad)
    yc, xc = y.cuda().requires_grad_(True), x.cuda().requires_grad_(True)
    gy, gx = torch.autograd.grad(bu.apply_norm_STFT_fweighted(yc, xc, wk, nfft), (yc, xc))
    assert rel_l2(gy.cpu(), -gx.cpu()) < 1e-6


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("wk", ["linear", "None", "cubic"])
def test_spec_dist_kernels_on_given_spectrograms(bu, mode, wk):
    """The distance kernels alone: value and both spectrogram gradients from the SAME spectrograms as a float64 torch
    evaluation of the reference's expressions (utils/blind_bwe_utils.py:148-248)."""
    gen = torch.Generator().manual_seed(7 + mode)
    X = torch.randn(2, 513, 31, 2, generator=gen)
    R = 0.7 * X + 0.5 * torch.randn(2, 513, 31, 2, generator=gen)
    w = bu.freq_weight_vector(wk, 513, torch.device("cuda"))
    Xd, Rd = X.double().requires_grad_(True), R.double().requires_grad_(True)
    wd = torch.ones(513, dtype=torch.float64) if w is None else w.cpu().double()
    if mode == 0:
        ref = torch.linalg.norm(((Xd - Rd) * wd[None, :, None, None]).reshape(-1))
    else:
        mx, mr = Xd.pow(2).sum(-1).sqrt() * wd[None, :, None], Rd.pow(2).sum(-1).sqrt() * wd[None, :, None]
        ref = torch.linalg.norm((mx - mr).reshape(-1)) if mode == 1 else \
            torch.linalg.norm((torch.log10(mx + 1e-8) - torch.log10(mr + 1e-8)).reshape(-1))
    gXr, gRr = torch.autograd.grad(ref, (Xd, Rd))
    Xc, Rc = X.cuda().requires_grad_(True), R.cuda().requires_grad_(True)
    from babe_b200.blind_bwe_utils import _SpecDist
    val = _SpecDist.apply(Xc, Rc, w, mode)
    gX, gR = torch.autograd.grad(val, (Xc, Rc))
    assert abs(float(val.detach()) - float(ref.detach())) < 1e-5 * float(ref.detach())
    assert rel_l2(gX.cpu(), gXr) < 2e-5 and rel_l2(gR.cpu(), gRr) < 2e-5, (rel_l2(gX.cpu(), gXr), rel_l2(gR.cpu(), gRr))


def test_spec_dist_abi_rejects_bad_mode(bu):
    from babe_b200 import ops
    from babe_b200._lib import BabeError
    X = torch.zeros(1, 5, 3, 2, device="cuda")
    with pytest.raises(BabeError):
        ops.spec_dist_stats(X, X, mode=1)
