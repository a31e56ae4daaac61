"""GPU: one filter estimate per group of consecutive rows (``filter_groups``).  The grouped statistics against the shared
statistics of each group's rows alone, their two bitwise layouts and group independence, and the grouped sampler
against one shared-filter call per group, its captured step graph, keyed noise and the ``restore_recordings``
driver."""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from kernel_trace import assert_path, launched
from toy_model import ToyDenoiser

pytestmark = pytest.mark.gpu
SR = 22050


@pytest.fixture(scope="module", autouse=True)
def _built():
    from babe_b200 import build
    build.build()


def _signals(B, T, seed=3):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(B, T, generator=g) * 0.063 * torch.linspace(0.2, 3.0, B)[:, None]).cuda()
    y = (torch.randn(B, T, generator=g) * 0.05).cuda()
    return x, y


def _slices(sizes):
    o = 0
    for n in sizes:
        yield o, o + n
        o += n


# (B, T, nfft, sizes): B = 5 at T = 10^6 cuts the batch into runs of frames that cross row and group boundaries;
# 8 and 64 x 184184 are the sampler's batches; T = 50001 cannot be bulk-copied (not a multiple of 4)
CASES = [(5, 1_000_000, 4096, [2, 1, 2]), (8, 184184, 4096, [3, 5]), (64, 184184, 4096, [8] * 8),
         (3, 132300, 1024, [1, 2]), (3, 50001, 4096, [2, 1])]


@pytest.mark.parametrize("B,T,nfft,sizes", CASES)
def test_stft_stats_groups_match_shared_slices(B, T, nfft, sizes):
    from babe_b200 import ops
    x, y = _signals(B, T)
    with launched() as names:
        abc = ops.stft_stats_groups(x, y, nfft, sizes)
    if nfft == 4096:
        assert_path(names, fused=T % 4 == 0, kernel="k_stats_fused" if T % 4 == 0 else None)
    assert abc.shape == (len(sizes), 3, nfft // 2 + 1) and abc.dtype == torch.float64
    for g, (a, b) in enumerate(_slices(sizes)):
        ref = ops.stft_stats(x[a:b], y[a:b], nfft)
        assert rel_l2(abc[g].cpu(), ref.cpu()) < 1e-6, g
    assert torch.equal(ops.stft_stats_groups(x, y, nfft, sizes), abc)          # deterministic


@pytest.mark.parametrize("B,T", [(8, 184184), (5, 1_000_000), (3, 50001)])
def test_stft_stats_groups_bitwise_layouts(B, T):
    """One group of all rows is the shared statistics and singleton groups the per-row statistics, bit for bit."""
    from babe_b200 import ops
    x, y = _signals(B, T, seed=5)
    assert torch.equal(ops.stft_stats_groups(x, y, 4096, [1] * B), ops.stft_stats_rows(x, y, 4096))
    if T % 4 == 0:                                   # fused path: the same grid, flush points and reduction order
        assert torch.equal(ops.stft_stats_groups(x, y, 4096, [B])[0], ops.stft_stats(x, y, 4096))


def test_groups_are_independent():
    """Perturbing one group's rows leaves every other group's statistics and fitted filter bitwise unchanged."""
    from babe_b200 import ops, sampler
    B, T, sizes = 5, 1_000_000, [2, 1, 2]
    x, y = _signals(B, T)
    fit = sampler.FilterFit(nfft=4096, sample_rate=SR, max_iter=100, device="cuda")
    p0 = torch.tensor([[280.0, 285, 290, 295, 300], [-15.0, -17, -20, -25, -30]]).cuda().expand(3, -1, -1)

    def run(x, y):
        abc = ops.stft_stats_groups(x, y, 4096, sizes)
        return abc, ops.fit_params_rows(abc, fit.w, fit.freqs, p0.contiguous().clone(), fit.cfg)

    a = run(x, y)
    x2, y2 = x.clone(), y.clone()
    x2[2] *= 1.7
    y2[2] = torch.roll(y2[2], 1234)
    b = run(x2, y2)
    for u, v in zip(a, b):
        assert torch.equal(u[[0, 2]], v[[0, 2]])
        assert not torch.equal(u[1], v[1])


# --------------------------------------------------------------------------- the sampler
def _sampler(y, T=4, max_iter=20, nfft=1024, sr=None):
    from babe_b200 import edm, sampler
    args = sampler.make_args(sample_rate=sr or SR, audio_len=y.shape[1], T=T, NFFT=nfft, max_iter=max_iter)
    return sampler.BlindSamplerFused(ToyDenoiser().cuda(), edm.EDM(args), args, rid=False)


def _row_noise(seeds):
    """noise_fn drawing row r of every draw from its own host generator (seeded seeds[r])."""
    gens = [torch.Generator().manual_seed(s) for s in seeds]
    return lambda shape, dev: torch.stack([torch.randn(shape[1:], generator=g) for g in gens]).to(dev)


def _recordings(golden):
    """Four different recordings, in two groups of two."""
    g = golden("fit_sampler.npz")
    y1 = torch.from_numpy(g["y"])[:1]
    y = torch.cat([y1, 0.5 * y1.roll(777, -1), 2.0 * y1.flip(-1), 0.8 * y1.flip(-1).roll(3000, -1)], 0).cuda()
    return g, y


SIZES = [2, 2]


def test_grouped_one_step_matches_shared_calls(golden):
    """One step from given states and per-group filters == one shared call per group on its rows."""
    g, y = _recordings(golden)
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=20)
    gen = torch.Generator().manual_seed(9)
    x_in = (y.cpu() + 0.05 * torch.randn(y.shape, generator=gen)).cuda()
    p_in = torch.tensor([[[300.0, 900, 2000, 4000, 8000], [-10.0, -15, -20, -30, -40]],
                         [[500.0, 700, 1500, 3000, 6000], [-5.0, -12, -25, -35, -45]]]).cuda()
    s.filter_groups = SIZES
    s.noise_fn = _row_noise([1, 2, 3, 4])
    x, p = s.predict_blind_bwe(y.clone(), max_steps=1, start_step=1, init_x=x_in, init_params=p_in)
    assert p.shape == (2, 2, 5)
    s.filter_groups = None
    for gi, (a, b) in enumerate(_slices(SIZES)):
        s.noise_fn = _row_noise([1, 2, 3, 4][a:b])
        xg, pg = s.predict_blind_bwe(y[a:b].clone(), max_steps=1, start_step=1, init_x=x_in[a:b], init_params=p_in[gi])
        assert rel_l2(x[a:b].cpu(), xg.cpu()) < 1e-5, gi
        assert rel_l2(p[gi].cpu(), pg.cpu()) < 2e-4, gi


def test_grouped_full_run_matches_shared_calls_and_groups_are_independent(golden):
    g, y = _recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=20)
    s.filter_groups = SIZES
    s.noise_fn = _row_noise([21, 22, 23, 24])
    x, p = s.predict_blind_bwe(y.clone())
    assert p.shape == (2, 2, 5)
    # changing group 1 leaves group 0 bitwise unchanged
    y2 = y.clone()
    y2[3] = 0.3 * y2[3].roll(99)
    s.noise_fn = _row_noise([21, 22, 23, 24])
    x2, p2 = s.predict_blind_bwe(y2)
    assert torch.equal(x[:2], x2[:2]) and torch.equal(p[0], p2[0])
    assert not torch.equal(x[2:], x2[2:])
    s.filter_groups = None
    for gi, (a, b) in enumerate(_slices(SIZES)):
        s.noise_fn = _row_noise([21, 22, 23, 24][a:b])
        xg, pg = s.predict_blind_bwe(y[a:b].clone())
        assert rel_l2(x[a:b].cpu(), xg.cpu()) < 1e-2, gi
        assert rel_l2(p[gi].cpu(), pg.cpu()) < 1e-2, gi
    assert not torch.allclose(p[0], p[1])                                     # the groups got different filters


def test_grouped_step_graph_matches_eager(golden):
    g, y = _recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=3)
    s.filter_groups = SIZES
    s.noise_fn = _row_noise([5, 6, 7, 8])
    x0, p0, den0, t0, f0 = s.predict_blind_bwe(y.clone(), rid=True)
    assert p0.shape == (2, 2, 5) and f0.shape == (4, 2, 2, 5) and den0.shape == (4, *y.shape)
    s.step_graph = True
    s.noise_fn = _row_noise([5, 6, 7, 8])
    x1, p1, den1, t1, f1 = s.predict_blind_bwe(y.clone(), rid=True)
    assert s._step_graphs, "capture failed"
    assert all(st.groups is not None and st.groups.sizes == (2, 2) for st in s._step_graphs.values())
    assert f1.shape == (4, 2, 2, 5)
    assert rel_l2(x1, x0) < 1e-6 and rel_l2(p1, p0) < 1e-6
    assert rel_l2(den1, den0) < 1e-6 and rel_l2(f1, f0) < 1e-6
    # another layout of the same batch is another graph
    s.filter_groups = [1, 3]
    s.noise_fn = _row_noise([5, 6, 7, 8])
    x3, p3 = s.predict_blind_bwe(y.clone())
    assert p3.shape == (2, 2, 5) and s._step_key[-1] == (1, 3)


def test_grouped_row_seeds_give_each_group_its_shared_noise(golden):
    g, y = _recordings(golden)
    torch.backends.cudnn.deterministic = True
    s = _sampler(y, nfft=int(g["nfft"]), sr=int(g["sr"]), max_iter=20)
    seeds = [1001, 1002, 1003, 1004]
    s.filter_groups, s.row_seeds = SIZES, seeds
    x, p = s.predict_blind_bwe(y.clone())
    s.filter_groups = None
    for gi, (a, b) in enumerate(_slices(SIZES)):
        s.row_seeds = seeds[a:b]
        xg, pg = s.predict_blind_bwe(y[a:b].clone())
        assert rel_l2(x[a:b].cpu(), xg.cpu()) < 1e-2, gi
        assert rel_l2(p[gi].cpu(), pg.cpu()) < 1e-2, gi


def test_restore_recordings_matches_restore_recording_joint():
    from babe_b200 import segments
    from oracle import stft_filter as osf
    torch.backends.cudnn.deterministic = True
    seg_len = 16384
    f = torch.fft.rfftfreq(4096, d=1 / SR)
    recs = []
    for k, (L, fc) in enumerate(((50000, 2000.0), (30000, 4000.0))):
        gen = torch.Generator().manual_seed(40 + k)
        t = torch.arange(L) / SR
        rec = 0.05 * torch.sin(2 * np.pi * (330 + 110 * k) * t) * (1 + torch.linspace(0, 2, L)) \
            + 0.01 * torch.randn(L, generator=gen)
        recs.append(osf.apply_filter(rec[None], osf.design_filter(torch.tensor([fc]), torch.tensor([-30.0]), f),
                                     4096).cuda())
    s = _sampler(torch.zeros(1, seg_len), T=4, nfft=4096, max_iter=20)
    seeds = [77, 78]
    out = segments.restore_recordings(s, recs, seg_len, seeds=seeds)
    assert s.filter_groups is None and s.row_seeds is None
    for r, rec in enumerate(recs):
        ref, ref_fd = segments.restore_recording(s, rec, seg_len, joint=True, seed=seeds[r])
        s.joint = False                               # restore_recording(joint=True) leaves it set
        got, fd = out[r]
        assert got.shape == rec.shape
        assert rel_l2(got.cpu(), ref.cpu()) < 1e-2, r
        assert len(fd) == len(ref_fd)
        assert all(torch.equal(fl, fd[0][1]) for _, fl in fd)                 # one filter per recording
        assert rel_l2(fd[0][1].cpu(), ref_fd[0][1].cpu()) < 1e-2, r
    assert not torch.allclose(out[0][1][0][1], out[1][1][0][1])
