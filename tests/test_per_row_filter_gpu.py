"""GPU: one filter estimate per row of y (``filter_per_row``).  The row operators against their shared-filter
counterparts run on one row at a time, row independence, and the per-row sampler against B = 1 calls, the CPU
oracle, its captured step graph and the segment driver."""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from toy_model import ToyDenoiser

pytestmark = pytest.mark.gpu
SR = 22050


def cuda(a):
    return torch.from_numpy(np.asarray(a)).cuda()


@pytest.fixture(scope="module", autouse=True)
def _built():
    from babe_b200 import build
    build.build()


@pytest.fixture
def fused_variant(request):
    from babe_b200._lib import lib
    assert lib().babe_set_fused_variant(request.param) == 0
    yield request.param
    lib().babe_set_fused_variant(0)


def _signals(B, T, seed=3):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(B, T, generator=g) * 0.063 * torch.linspace(0.2, 3.0, B)[:, None]).cuda()
    y = (torch.randn(B, T, generator=g) * 0.05).cuda()
    return x, y


def _row_filters(B, K=5):
    """Widely different filters, one per row: cutoffs from 300 Hz to 9 kHz, slopes from -5 to -45 dB."""
    fc0 = torch.logspace(np.log10(300.0), np.log10(9000.0), B)
    fc = torch.stack([fc0 * (1.0 + 0.3 * k) for k in range(K)], 1)
    A = torch.stack([torch.linspace(-5.0, -45.0, B) - 3.0 * k for k in range(K)], 1)
    return fc.cuda().contiguous(), A.cuda().contiguous()


# (B, T, nfft): B = 3 at T = 10^6 cuts the batch into runs of 5 frames / output blocks that cross row boundaries
# (489 frames per row); 8 x 184184 is the sampler's batch; T = 50001 cannot be bulk-copied (not a multiple of 4)
CASES = [(3, 1_000_000, 4096), (8, 184184, 4096), (2, 132300, 1024), (3, 50001, 4096)]


@pytest.mark.parametrize("fused_variant", [0, -1], indirect=True)
@pytest.mark.parametrize("B,T,nfft", CASES)
def test_stft_stats_rows_match_single_rows(fused_variant, B, T, nfft):
    from babe_b200 import ops
    x, y = _signals(B, T)
    abc = ops.stft_stats_rows(x, y, nfft)
    assert abc.shape == (B, 3, nfft // 2 + 1) and abc.dtype == torch.float64
    for b in range(B):
        ref = ops.stft_stats(x[b:b + 1], y[b:b + 1], nfft)
        assert rel_l2(abc[b].cpu(), ref.cpu()) < 1e-6, b
    assert torch.equal(ops.stft_stats_rows(x, y, nfft), abc)          # deterministic


@pytest.mark.parametrize("fused_variant", [0, -1], indirect=True)
@pytest.mark.parametrize("B,T,nfft", CASES)
def test_apply_filter_rows_match_single_rows(fused_variant, B, T, nfft):
    from babe_b200 import ops
    x, sub = _signals(B, T)
    f = torch.fft.rfftfreq(nfft, d=1 / SR).cuda()
    fc, A = _row_filters(B)
    scale = torch.linspace(0.5, 2.0, B).cuda()
    ss = torch.zeros(B, dtype=torch.float64, device="cuda")
    out = {
        "fwd": ops.apply_filter_rows(x, nfft, f, fc, A),
        "adj": ops.apply_filter_rows(x, nfft, f, fc, A, adjoint=True),
        "res": ops.apply_filter_rows(x, nfft, f, fc, A, sub=sub, row_sumsq=ss),
        "scaled": ops.apply_filter_rows(x, nfft, f, fc, A, adjoint=True, row_scale=scale),
    }
    for b in range(B):
        xb = x[b:b + 1]
        ss1 = torch.zeros(1, dtype=torch.float64, device="cuda")
        ref = {
            "fwd": ops.apply_filter(xb, nfft, freqs=f, fc=fc[b], A=A[b]),
            "adj": ops.apply_filter(xb, nfft, freqs=f, fc=fc[b], A=A[b], adjoint=True),
            "res": ops.apply_filter(xb, nfft, freqs=f, fc=fc[b], A=A[b], sub=sub[b:b + 1], row_sumsq=ss1),
            "scaled": ops.apply_filter(xb, nfft, freqs=f, fc=fc[b], A=A[b], adjoint=True, row_scale=scale[b:b + 1]),
        }
        for k in out:
            assert rel_l2(out[k][b:b + 1].cpu(), ref[k].cpu()) < 1e-6, (k, b)
        assert abs(float(ss[b]) - float(ss1[0])) <= 1e-6 * float(ss1[0]), b


def test_apply_filter_rows_status_per_row():
    from babe_b200 import ops
    x, _ = _signals(3, 184184)
    f = torch.fft.rfftfreq(4096, d=1 / SR).cuda()
    fc = torch.tensor([[300.0, 900.0], [400.0, 20000.0], [500.0, 2000.0]]).cuda()    # row 1: fc above the last bin
    A = torch.full((3, 2), -20.0).cuda()
    status = torch.zeros(3, dtype=torch.int32, device="cuda")
    ops.apply_filter_rows(x, 4096, f, fc, A, status=status)
    assert status.tolist() == [0, 1, 0]


def test_fit_params_rows_bitwise(golden):
    """Cluster b of the per-row fit kernel fits row b: bitwise the shared-mode fit of that row, iteration counts
    included (rows stop early at different iterations), for every fit kernel generation."""
    from babe_b200 import ops, sampler
    from babe_b200._lib import lib
    tf, g = golden("teacher_forced.npz"), golden("operator_n4096.npz")
    its = tf["fit_iters_n4096"]
    B, T = 3, 184184
    x, _ = _signals(B, T, seed=11)
    f = torch.fft.rfftfreq(4096, d=1 / SR).cuda()
    fc, A = _row_filters(B)
    y = ops.apply_filter_rows(x, 4096, f, fc, A)
    # tolerances under which the reference's late iterates count as converged (with the default 5e-3 its run never
    # stops before 100 iterations), so that rows stop early, at different iterations
    fit = sampler.FilterFit(nfft=int(g["nfft"]), sample_rate=int(g["sr"]), max_iter=100, tol=(1.0, 0.05),
                            device="cuda")
    # rows 0-2: the statistics of the inputs of the reference's own fit run (teacher_forced.npz), started from its
    # iterates 0, 10 and 40; rows 3-5: other recordings, default start
    abc_ref = ops.stft_stats(cuda(g["x"]), cuda(g["yobs"]), 4096)
    abc = torch.cat([abc_ref[None].expand(3, -1, -1), ops.stft_stats_rows(x, y, 4096)]).contiguous()
    p0 = torch.stack([cuda(its[i]) for i in (0, 10, 40)]
                     + [torch.tensor([[280.0, 285, 290, 295, 300], [-15.0, -17, -20, -25, -30]]).cuda()] * B)
    B = 2 * B
    try:
        for v in (0, -1):
            assert lib().babe_set_fit_variant(v) == 0
            p, it = ops.fit_params_rows(abc, fit.w, fit.freqs, p0.clone(), fit.cfg, return_iters=True)
            for b in range(B):
                pb, itb = ops.fit_params(abc[b], fit.w, fit.freqs, p0[b].clone(), fit.cfg, return_iters=True)
                assert torch.equal(p[b], pb), (v, b)
                assert int(it[b]) == int(itb), (v, b)
            if v == 0:
                iters0 = it.cpu().tolist()
        assert len(set(iters0)) > 1, iters0                              # rows stopped at different iterations
    finally:
        lib().babe_set_fit_variant(0)


def test_row_ops_are_row_independent():
    """Perturbing row j's inputs leaves every other row's results bitwise unchanged."""
    from babe_b200 import ops, sampler
    B, T, j = 3, 1_000_000, 1
    x, y = _signals(B, T)
    f = torch.fft.rfftfreq(4096, d=1 / SR).cuda()
    fc, A = _row_filters(B)
    fit = sampler.FilterFit(nfft=4096, sample_rate=SR, max_iter=100, device="cuda")
    p0 = torch.tensor([[280.0, 285, 290, 295, 300], [-15.0, -17, -20, -25, -30]]).cuda().expand(B, -1, -1)

    def run(x, y, fc, A):
        ss = torch.zeros(B, dtype=torch.float64, device="cuda")
        r = ops.apply_filter_rows(x, 4096, f, fc, A, sub=y, row_sumsq=ss)
        adj = ops.apply_filter_rows(r, 4096, f, fc, A, adjoint=True, row_scale=torch.ones(B, device="cuda"))
        abc = ops.stft_stats_rows(x, y, 4096)
        p = ops.fit_params_rows(abc, fit.w, fit.freqs, p0.contiguous().clone(), fit.cfg)
        return r, ss, adj, abc, p

    a = run(x, y, fc, A)
    x2, y2, fc2, A2 = x.clone(), y.clone(), fc.clone(), A.clone()
    x2[j] *= 1.7
    y2[j] = torch.roll(y2[j], 1234)
    fc2[j] *= 0.6
    A2[j] -= 7.0
    b = run(x2, y2, fc2, A2)
    keep = [r for r in range(B) if r != j]
    for u, v in zip(a, b):
        assert torch.equal(u[keep], v[keep])
        assert not torch.equal(u[j], v[j])


# --------------------------------------------------------------------------- the sampler
def _sampler(y, T=4, max_iter=20, nfft=1024, sr=None, per_row=True):
    from babe_b200 import edm, sampler
    args = sampler.make_args(sample_rate=sr or SR, audio_len=y.shape[1], T=T, NFFT=nfft, max_iter=max_iter,
                             filter_per_row=per_row)
    return sampler.BlindSamplerFused(ToyDenoiser().cuda(), edm.EDM(args), args, rid=False)


def _row_noise(seeds):
    """noise_fn drawing row r of every draw from its own host generator (seeded seeds[r])."""
    gens = [torch.Generator().manual_seed(s) for s in seeds]
    return lambda shape, dev: torch.stack([torch.randn(shape[1:], generator=g) for g in gens]).to(dev)


def _three_recordings(golden):
    g = golden("fit_sampler.npz")
    y1 = torch.from_numpy(g["y"])[:1]
    y = torch.cat([y1, 0.5 * y1.roll(777, -1), 2.0 * y1.flip(-1)], 0).cuda()
    return g, y


def test_sampler_rows_are_independent(golden):
    g, y = _three_recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=20)
    s.noise_fn = _row_noise([1, 2, 3])
    x0, p0 = s.predict_blind_bwe(y.clone(), max_steps=2)
    y2 = y.clone()
    y2[1] = 0.3 * y2[1].roll(99)
    s.noise_fn = _row_noise([1, 2, 3])
    x1, p1 = s.predict_blind_bwe(y2, max_steps=2)
    for r in (0, 2):
        assert torch.equal(x0[r], x1[r]) and torch.equal(p0[r], p1[r]), r
    assert not torch.equal(x0[1], x1[1])


def test_sampler_one_step_matches_single_row_calls(golden):
    """One step from given states (the reference run's states, a different one per row) == B = 1 calls."""
    tf = golden("teacher_forced.npz")
    y = cuda(tf["step_y"])
    nfft, sr, mi = int(tf["step_nfft"]), int(tf["step_sr"]), int(tf["step_max_iter"])
    s = _sampler(y, nfft=nfft, sr=sr, max_iter=mi)
    i = 1
    x_in = cuda(tf["step_x_in"][i])
    p_in = torch.stack([cuda(tf["step_p_in"][i]), cuda(tf["step_p_in"][i + 1])])
    s.noise_fn = lambda shape, dev: cuda(tf["step_draws"][i + 1])
    x, p = s.predict_blind_bwe(y.clone(), max_steps=1, start_step=i, init_x=x_in, init_params=p_in)
    s.filter_per_row = False
    for r in range(2):
        s.noise_fn = lambda shape, dev, r=r: cuda(tf["step_draws"][i + 1][r:r + 1])
        xr, pr = s.predict_blind_bwe(y[r:r + 1].clone(), max_steps=1, start_step=i, init_x=x_in[r:r + 1],
                                     init_params=p_in[r])
        assert rel_l2(x[r:r + 1].cpu(), xr.cpu()) < 1e-5, r
        assert rel_l2(p[r].cpu(), pr.cpu()) < 2e-4, r


def test_sampler_full_run_matches_single_row_calls_and_b1_is_shared(golden):
    g, y = _three_recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=20)
    s.noise_fn = _row_noise([21, 22, 23])
    x, p = s.predict_blind_bwe(y.clone())
    assert p.shape == (3, 2, 5)
    for r in range(3):
        s.filter_per_row = False
        s.noise_fn = _row_noise([21 + r])
        xr, pr = s.predict_blind_bwe(y[r:r + 1].clone())
        assert rel_l2(x[r:r + 1].cpu(), xr.cpu()) < 1e-2, r
        assert rel_l2(p[r].cpu(), pr.cpu()) < 1e-2, r
        # B = 1: the per-row mode is the shared mode, bit for bit
        s.filter_per_row = True
        s.noise_fn = _row_noise([21 + r])
        x1, p1 = s.predict_blind_bwe(y[r:r + 1].clone())
        assert torch.equal(x1, xr) and torch.equal(p1[0], pr), r


def test_sampler_rows_match_oracle(golden):
    from oracle import blind_sampler as obs, filter_fit as ofit
    g, y = _three_recordings(golden)
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=3)
    s.noise_fn = _row_noise([7, 8, 9])
    x, p = s.predict_blind_bwe(y.clone())
    cfg = obs.SamplerConfig(T=4, audio_len=y.shape[1])
    cfg.fit = ofit.FitConfig(nfft=int(g["nfft"]), sample_rate=int(g["sr"]), max_iter=3)
    cpu_model = ToyDenoiser()
    for r in range(3):
        gen = torch.Generator().manual_seed(7 + r)
        xo, po = obs.predict_blind_bwe(cfg, cpu_model, cpu_model.CQTransform.apply_hpf_DC, y[r:r + 1].cpu(),
                                       randn=lambda shape: torch.randn(shape, generator=gen))
        assert rel_l2(p[r].cpu(), po) < 1e-4, r
        assert rel_l2(x[r:r + 1].cpu(), xo) < 1e-4, r


def test_per_row_step_graph_matches_eager(golden):
    g, y = _three_recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=3)
    s.noise_fn = _row_noise([5, 6, 7])
    x0, p0, den0, t0, f0 = s.predict_blind_bwe(y.clone(), rid=True)
    assert p0.shape == (3, 2, 5) and f0.shape == (4, 3, 2, 5) and den0.shape == (4, *y.shape)
    s.step_graph = True
    s.noise_fn = _row_noise([5, 6, 7])
    x1, p1, den1, t1, f1 = s.predict_blind_bwe(y.clone(), rid=True)
    assert s._step_graphs, "capture failed"
    assert f1.shape == (4, 3, 2, 5)
    assert rel_l2(x1, x0) < 1e-6 and rel_l2(p1, p0) < 1e-6
    assert rel_l2(den1, den0) < 1e-6 and rel_l2(f1, f0) < 1e-6


def test_restore_recording_batched_matches_sequential():
    from babe_b200 import segments
    torch.backends.cudnn.deterministic = True
    seg_len, L = 16384, 50000
    gen = torch.Generator().manual_seed(4)
    t = torch.arange(L) / SR
    rec = (0.05 * torch.sin(2 * np.pi * 440 * t) * (1 + torch.linspace(0, 2, L)) + 0.01 * torch.randn(L, generator=gen))
    f = torch.fft.rfftfreq(4096, d=1 / SR)
    from oracle import stft_filter as osf
    deg = osf.apply_filter(rec[None], osf.design_filter(torch.tensor([2000.0]), torch.tensor([-30.0]), f), 4096).cuda()
    n_seg = segments.split(deg, seg_len)[0].shape[0]
    s = _sampler(torch.zeros(1, seg_len), T=4, nfft=4096, max_iter=20, per_row=False)
    draws_per_call = s.nb_steps + 1
    gens = [torch.Generator().manual_seed(100 + k) for k in range(n_seg)]
    count = [0]

    def sequential_noise(shape, dev):                 # the loop restores segment 0 completely, then segment 1, ...
        k = count[0] // draws_per_call
        count[0] += 1
        return torch.randn(shape, generator=gens[k]).to(dev)

    s.noise_fn = sequential_noise
    out_seq, fd_seq = segments.restore_recording(s, deg, seg_len)
    assert count[0] == n_seg * draws_per_call
    s.noise_fn = _row_noise([100 + k for k in range(n_seg)])
    out_bat, fd_bat = segments.restore_recording(s, deg, seg_len, batched=True)
    assert s.filter_per_row is False                  # restored after the call
    assert rel_l2(out_bat.cpu(), out_seq.cpu()) < 1e-2
    assert len(fd_bat) == n_seg
    for (sp_b, f_b), (sp_s, f_s) in zip(fd_bat, fd_seq):
        assert sp_b == sp_s and f_b.shape == f_s.shape == (2, 5)
        assert rel_l2(f_b.cpu(), f_s.cpu()) < 1e-2
    filts = torch.stack([f_b for _, f_b in fd_bat])
    assert len({tuple(v.tolist()) for v in filts.reshape(n_seg, -1).cpu()}) == n_seg     # one filter per segment
