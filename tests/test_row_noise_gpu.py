"""GPU: keyed per-row noise (``k_row_noise``, ``BlindSamplerFused.row_seeds``, DESIGN.md 4.8).  The kernel against
the float64 numpy restatement, bitwise invariance of a row's noise under batch size, position, permutation and
length, its distribution, and the sampler and segment drivers with per-row seeds: B rows against B = 1 calls,
reproducibility, resuming, the captured step graph and the absence of host draws."""
import numpy as np
import pytest
import torch

import row_noise_ref as ref
from conftest import rel_l2
from toy_model import ToyDenoiser

pytestmark = pytest.mark.gpu
SR = 22050


@pytest.fixture(scope="module", autouse=True)
def _built():
    from babe_b200 import build
    build.build()


def _seeds(vals):
    from babe_b200.sampler import BlindSamplerFused
    return BlindSamplerFused._seed_tensor(list(vals)).cuda()


# --------------------------------------------------------------------------- the kernel
@pytest.mark.parametrize("B,T", [(3, 1_000_000), (8, 184184), (2, 50001)])
def test_row_noise_matches_numpy(B, T):
    """T = 50001: odd, so row 1 starts misaligned and every row ends in a partial group of four."""
    from babe_b200 import ops, segments
    vals = [segments.row_seed(9, k) for k in range(B)]
    out = ops.row_noise(_seeds(vals), (B, T), 5, slot=2).cpu().numpy()
    for b, s in enumerate(vals):
        want = ref.row_noise(s, 7, T)
        assert np.abs(out[b] - want).max() < 1e-5, b


@pytest.mark.parametrize("T", [184184, 50001])
def test_fused_form(T):
    from babe_b200 import ops
    B = 4
    seeds = _seeds([11, 12, 13, 2 ** 64 - 1])
    g = torch.Generator().manual_seed(0)
    a = torch.randn(B, T, generator=g).cuda()
    scale = torch.tensor([0.37], device="cuda")
    rs = torch.tensor([0.5, 1.0, 2.0, 3.25], device="cuda")
    draw = torch.tensor([17], dtype=torch.int32, device="cuda")
    raw = ops.row_noise(seeds, (B, T), draw, slot=3)
    m = (torch.tensor(0.8, device="cuda") * scale) * rs
    want = a + raw * m[:, None]
    got = ops.row_noise(seeds, a, draw, slot=3, scale=scale, row_scale=rs, mult=0.8)
    assert ((got - want).abs() <= 2.0 ** -23 * (a.abs() + (raw * m[:, None]).abs())).all()
    inplace = a.clone()
    ops.row_noise(seeds, inplace, draw, slot=3, scale=scale, row_scale=rs, mult=0.8, out=inplace)
    assert torch.equal(inplace, got)
    assert torch.equal(ops.row_noise(seeds, (B, T), 20), raw)            # the draw index is *draw + slot


def test_row_noise_invariance_bitwise():
    from babe_b200 import ops
    vals = [101, 2 ** 40 + 7, 3, 2 ** 63 + 5, 99]
    T, d = 10007, 4
    full = ops.row_noise(_seeds(vals), (5, T), d)
    for b, s in enumerate(vals):
        assert torch.equal(ops.row_noise(_seeds([s]), (1, T), d)[0], full[b]), b                # alone
        assert torch.equal(ops.row_noise(_seeds([s]), (1, T + 37), d)[0, :T], full[b]), b       # longer row
        assert torch.equal(ops.row_noise(_seeds([s]), (1, T - 4000), d)[0], full[b, :T - 4000]), b
    perm = [3, 0, 4, 2, 1]
    assert torch.equal(ops.row_noise(_seeds([vals[p] for p in perm]), (5, T), d), full[perm])
    assert torch.equal(ops.row_noise(_seeds([vals[4], vals[1]]), (2, T), d), full[[4, 1]])
    big = ops.row_noise(_seeds(vals * 7), (35, T), d)                                         # another B
    assert torch.equal(big[25:30], full)
    assert not torch.equal(ops.row_noise(_seeds([vals[0] + 1]), (1, T), d)[0], full[0])       # another seed
    assert not torch.equal(ops.row_noise(_seeds([vals[0]]), (1, T), d + 1)[0], full[0])      # another draw


def test_row_noise_distribution():
    from babe_b200 import ops
    B, T = 16, 2 ** 20
    seeds = _seeds(range(1000, 1000 + B))                  # adjacent keys
    x = ops.row_noise(seeds, (B, T), 0).double()
    x2 = ops.row_noise(seeds, (B, T), 1).double()
    N = x.numel()
    assert N >= 2 ** 24
    assert abs(float(x.mean())) < 5 / N ** 0.5
    assert abs(float(x.var()) - 1) < 5 * (2 / N) ** 0.5
    v, _ = torch.sort(x.reshape(-1))
    cdf = torch.special.ndtr(v)
    i = torch.arange(1, N + 1, device=v.device, dtype=torch.float64)
    ks = max(float((i / N - cdf).max()), float((cdf - (i - 1) / N).max()))
    assert ks < 2 / N ** 0.5, ks
    lim = 5 / N ** 0.5
    assert abs(float((x[:, 1:] * x[:, :-1]).mean())) < lim                # lag 1 within a row
    assert abs(float((x[1:] * x[:-1]).mean())) < lim                      # adjacent rows (seeds)
    assert abs(float((x * x2).mean())) < lim                              # adjacent draw indices


# --------------------------------------------------------------------------- the sampler
def _sampler(y, T=4, max_iter=20, nfft=1024, sr=None, per_row=True):
    from babe_b200 import edm, sampler
    args = sampler.make_args(sample_rate=sr or SR, audio_len=y.shape[1], T=T, NFFT=nfft, max_iter=max_iter,
                             filter_per_row=per_row)
    return sampler.BlindSamplerFused(ToyDenoiser().cuda(), edm.EDM(args), args, rid=False)


def _three_recordings(golden):
    g = golden("fit_sampler.npz")
    y1 = torch.from_numpy(g["y"])[:1]
    y = torch.cat([y1, 0.5 * y1.roll(777, -1), 2.0 * y1.flip(-1)], 0).cuda()
    return g, y


SEEDS = [2 ** 63 + 21, 22, 2 ** 40 + 23]


def test_keyed_sampler_one_step_matches_single_row_calls(golden):
    tf = golden("teacher_forced.npz")
    y = torch.from_numpy(tf["step_y"]).cuda()
    nfft, sr, mi = int(tf["step_nfft"]), int(tf["step_sr"]), int(tf["step_max_iter"])
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=nfft, sr=sr, max_iter=mi)
    i = 1
    x_in = torch.from_numpy(tf["step_x_in"][i]).cuda()
    p_in = torch.stack([torch.from_numpy(tf["step_p_in"][i]), torch.from_numpy(tf["step_p_in"][i + 1])]).cuda()
    s.row_seeds = SEEDS[:2]
    x, p = s.predict_blind_bwe(y.clone(), max_steps=1, start_step=i, init_x=x_in, init_params=p_in)
    s.filter_per_row = False
    for r in range(2):
        s.row_seeds = [SEEDS[r]]
        xr, pr = s.predict_blind_bwe(y[r:r + 1].clone(), max_steps=1, start_step=i, init_x=x_in[r:r + 1],
                                     init_params=p_in[r])
        assert rel_l2(x[r:r + 1].cpu(), xr.cpu()) < 1e-5, r
        assert rel_l2(p[r].cpu(), pr.cpu()) < 2e-4, r


def test_keyed_sampler_full_run_matches_single_row_calls_and_repeats(golden):
    g, y = _three_recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=20)
    s.row_seeds = _seeds(SEEDS)                         # an int64 tensor works as well as a list
    x, p = s.predict_blind_bwe(y.clone())
    x2, p2 = s.predict_blind_bwe(y.clone())
    assert torch.equal(x, x2) and torch.equal(p, p2)                      # the same call twice
    s.filter_per_row = False
    for r in range(3):
        s.row_seeds = [SEEDS[r]]
        xr, pr = s.predict_blind_bwe(y[r:r + 1].clone())
        assert rel_l2(x[r:r + 1].cpu(), xr.cpu()) < 1e-2, r
        assert rel_l2(p[r].cpu(), pr.cpu()) < 1e-2, r
    s.filter_per_row = True
    s.row_seeds = [SEEDS[0], SEEDS[1] + 1, SEEDS[2]]
    x3, _ = s.predict_blind_bwe(y.clone())
    assert torch.equal(x3[0], x[0]) and torch.equal(x3[2], x[2]) and not torch.equal(x3[1], x[1])


def test_keyed_sampler_resume_is_bitwise(golden):
    g, y = _three_recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=20)
    s.row_seeds = SEEDS
    state = {}

    def hook(i, x, p):
        if i == 1:
            state["x"], state["p"] = x.clone(), p.clone()
    x, p = s.predict_blind_bwe(y.clone(), step_hook=hook)
    xr, pr = s.predict_blind_bwe(y.clone(), start_step=2, init_x=state["x"], init_params=state["p"])
    assert torch.equal(xr, x) and torch.equal(pr, p)


def test_keyed_observation_and_estimate_noise(golden):
    """The SNR observation noise (in place on y, per-row sigma) and the sigma_den_estimate draw take keyed noise too:
    a call repeats bit for bit, and changing one row's seed changes that row only."""
    g, y = _three_recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=5)
    s.args.tester.posterior_sampling.SNR_observations = 30
    s.args.tester.blind_bwe.sigma_den_estimate = 0.01
    s.row_seeds = SEEDS
    ya = y.clone()
    x, p = s.predict_blind_bwe(ya, max_steps=2)
    assert not torch.equal(ya, y)                                          # the observations were noised in place
    yb = y.clone()
    x2, p2 = s.predict_blind_bwe(yb, max_steps=2)
    assert torch.equal(x, x2) and torch.equal(p, p2) and torch.equal(ya, yb)
    s.row_seeds = [SEEDS[0], SEEDS[1] + 1, SEEDS[2]]
    x3, p3 = s.predict_blind_bwe(y.clone(), max_steps=2)
    for r in (0, 2):
        assert torch.equal(x3[r], x[r]) and torch.equal(p3[r], p[r]), r
    assert not torch.equal(x3[1], x[1])


def test_keyed_step_graph_matches_eager_and_draws_nothing_on_host(golden, monkeypatch):
    from babe_b200 import sampler
    g, y = _three_recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=3)
    s.device_noise = True                          # row_seeds takes precedence over the other sources

    def boom(*a, **k):
        raise AssertionError("keyed noise drew from a generator")
    monkeypatch.setattr(sampler.BlindSamplerFused, "_host_randn_pinned", boom)
    monkeypatch.setattr(torch, "randn", boom)
    s.row_seeds = SEEDS
    x0, p0, den0, _, f0 = s.predict_blind_bwe(y.clone(), rid=True)
    s.step_graph = True
    x1, p1, den1, _, f1 = s.predict_blind_bwe(y.clone(), rid=True)
    assert s._step_graphs, "capture failed"
    assert all(st.eps is None for st in s._step_graphs.values())        # no per-step noise buffer to upload
    assert rel_l2(x1, x0) < 1e-6 and rel_l2(p1, p0) < 1e-6
    assert rel_l2(den1, den0) < 1e-6 and rel_l2(f1, f0) < 1e-6
    graphs = dict(s._step_graphs)
    s.row_seeds = [SEEDS[0], SEEDS[1] + 1, SEEDS[2]]    # new seeds reach the captured steps without a recapture
    x2, _ = s.predict_blind_bwe(y.clone())
    assert all(s._step_graphs[k] is graphs[k] for k in graphs) and len(s._step_graphs) == len(graphs)
    assert torch.equal(x2[0], x1[0]) and torch.equal(x2[2], x1[2]) and not torch.equal(x2[1], x1[1])


def test_keyed_conditional_paths_match_single_rows(golden):
    g, y = _three_recordings(golden)
    y = y[:2].contiguous()
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), per_row=False)
    # xi = 0 with the data-consistency step: the per-row filter enters each row alone (the guidance normaliser of
    # the conditional path is one norm over the batch, as in the reference)
    s.xi = 0
    s.data_consistency = True
    filt = torch.tensor([[[1500.0, 3000.0], [-20.0, -40.0]], [[900.0, 5000.0], [-10.0, -30.0]]]).cuda()
    s.row_seeds = SEEDS[:2]
    xb = s.predict_bwe(y.clone(), filt, "fc_A")
    xu = s.predict_unconditional(tuple(y.shape), y.device)
    for r in range(2):
        s.row_seeds = [SEEDS[r]]
        assert rel_l2(s.predict_bwe(y[r:r + 1].clone(), filt[r:r + 1], "fc_A").cpu(), xb[r:r + 1].cpu()) < 1e-6, r
        assert rel_l2(s.predict_unconditional((1, y.shape[1]), y.device).cpu(), xu[r:r + 1].cpu()) < 1e-6, r


# --------------------------------------------------------------------------- the drivers
def _degraded(L):
    from oracle import stft_filter as osf
    gen = torch.Generator().manual_seed(4)
    t = torch.arange(L) / SR
    rec = (0.05 * torch.sin(2 * np.pi * 440 * t) * (1 + torch.linspace(0, 2, L)) + 0.01 * torch.randn(L, generator=gen))
    f = torch.fft.rfftfreq(4096, d=1 / SR)
    return osf.apply_filter(rec[None], osf.design_filter(torch.tensor([2000.0]), torch.tensor([-30.0]), f), 4096).cuda()


def test_restore_recording_seeded_batched_matches_sequential():
    from babe_b200 import segments
    torch.backends.cudnn.deterministic = True
    seg_len = 16384
    deg = _degraded(50000)
    n_seg = segments.split(deg, seg_len)[0].shape[0]
    s = _sampler(torch.zeros(1, seg_len), T=4, nfft=4096, max_iter=20, per_row=False)
    out_seq, fd_seq = segments.restore_recording(s, deg, seg_len, seed=31337)
    out_bat, fd_bat = segments.restore_recording(s, deg, seg_len, batched=True, seed=31337)
    assert s.row_seeds is None and s.filter_per_row is False
    assert rel_l2(out_bat.cpu(), out_seq.cpu()) < 1e-2
    assert len(fd_bat) == n_seg
    for (sp_b, f_b), (sp_s, f_s) in zip(fd_bat, fd_seq):
        assert sp_b == sp_s and f_b.shape == f_s.shape == (2, 5)
        assert rel_l2(f_b.cpu(), f_s.cpu()) < 1e-2


def test_restore_recording_ar_seeded_is_reproducible():
    from babe_b200 import edm, sampler, segments
    torch.backends.cudnn.deterministic = True
    seg_len = 8192
    deg = _degraded(30000)
    args = sampler.make_args(audio_len=seg_len, T=3, NFFT=1024, max_iter=5)
    s = sampler.BlindSamplerFused(ToyDenoiser().cuda(), edm.EDM(args), args, rid=False)

    def run(seed):
        return segments.restore_recording_ar(s, deg.clone(), seg_len, SR, rng=np.random.RandomState(0), seed=seed)
    a, fa = run(5)
    b, fb = run(5)
    assert torch.equal(a, b) and torch.equal(fa, fb)
    c, _ = run(6)
    assert not torch.equal(a, c)
    assert s.row_seeds is None
