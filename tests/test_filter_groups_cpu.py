"""CPU: plumbing of grouped filter estimation (``filter_groups``: one filter per group of consecutive rows).  Argument
checks of ``ops.stft_stats_groups``, the sampler's rejections, the grouped sampler on the oracle operators against one
shared-filter call per group, and the ``restore_recordings`` driver on a stub sampler.  The kernels are checked on the
GPU (tests/test_filter_groups_gpu.py)."""
import pytest
import torch

from conftest import rel_l2
from test_per_row_plumbing_cpu import oracle_row_ops  # noqa: F401 - fixture
from toy_model import ToyDenoiser


# --------------------------------------------------------------------------- argument checks
def test_stft_stats_groups_argument_checks():
    from babe_b200 import ops
    from babe_b200._lib import BabeError
    x = torch.zeros(5, 8192)
    for bad in ([2, 2], [2, 4], [0, 5], [-1, 6], [2.0, 3], [True, 4], [], "23", 5, None):
        with pytest.raises(ValueError):
            ops.stft_stats_groups(x, x, 4096, bad)
    with pytest.raises(ValueError):
        ops.stft_stats_groups(x, x[:4], 4096, [2, 3])
    with pytest.raises(BabeError):                     # CPU tensors: there is no CPU fallback
        ops.stft_stats_groups(x, x, 4096, [2, 3])
    assert ops.group_sizes([2, 1, 2], 5) == (2, 1, 2)


def _sampler(**kw):
    from babe_b200 import edm, sampler
    args = sampler.make_args(audio_len=8192, T=4, NFFT=1024, max_iter=3, **kw)
    return sampler.BlindSamplerFused(ToyDenoiser(), edm.EDM(args), args, rid=False), args


def test_sampler_rejections():
    s, args = _sampler()
    assert s.filter_groups is None
    y = torch.zeros(4, 8192)
    for bad in ([2, 1], [0, 4], [2.5, 1.5], [4, 0]):
        s.filter_groups = bad
        with pytest.raises(ValueError, match="group sizes"):
            s.predict_blind_bwe(y)
    s.filter_groups = [2, 2]
    s.joint = True
    with pytest.raises(ValueError, match="choose one"):
        s.predict_blind_bwe(y)
    s.joint = False
    s.filter_per_row = True
    with pytest.raises(ValueError, match="choose one"):
        s.predict_blind_bwe(y)
    s.filter_per_row = False
    with pytest.raises(NotImplementedError, match="compute_sweep"):
        s.predict_blind_bwe(y, compute_sweep=True)
    args.tester.posterior_sampling.stft_distance.use = True
    with pytest.raises(NotImplementedError, match="STFT-distance"):
        s.predict_blind_bwe(y)
    args.tester.posterior_sampling.stft_distance.use = False
    with pytest.raises(ValueError, match="per-group filter parameters"):
        s.predict_blind_bwe(y, init_params=torch.zeros(4, 2, 5))
    filt = torch.tensor([[500.0], [-20.0]])
    mask = torch.ones(4, 8192)
    for call in (lambda: s.predict_bwe(y, filt, "fc_A"),
                 lambda: s.predict_bwe_AR(y, y, filt, "fc_A", mask=mask),
                 lambda: s.predict_conditional(y, lambda x: x),
                 lambda: s.predict_unconditional((4, 8192), "cpu")):
        with pytest.raises(ValueError, match="filter_groups"):
            call()


# --------------------------------------------------------------------------- sampler bookkeeping on the oracle
@pytest.fixture
def oracle_group_ops(oracle_row_ops, monkeypatch):  # noqa: F811 - the imported fixture
    from babe_b200 import ops

    def stft_stats_groups(x, y, nfft, sizes):
        sizes, out, o = ops.group_sizes(sizes, x.shape[0]), [], 0
        for n in sizes:
            out.append(ops.stft_stats(x[o:o + n], y[o:o + n], nfft))
            o += n
        return torch.stack(out)

    monkeypatch.setattr(ops, "stft_stats_groups", stft_stats_groups)


def _row_noise(gens, rows):
    return lambda shape, dev: torch.stack([torch.randn(shape[1], generator=gens[r]) for r in rows]).to(dev)


@pytest.mark.parametrize("sizes", [[2, 1, 2], [5], [1, 1, 1, 1, 1]])
def test_grouped_sampler_equals_shared_calls_per_group(oracle_group_ops, golden, sizes):
    """Group statistics, one fit per group, the group's filter in the guidance and the group's normaliser: a grouped
    call == one shared call per group on its rows alone (same noise per row), on the oracle operators."""
    from babe_b200 import edm, sampler
    g = golden("fit_sampler.npz")
    y1 = torch.from_numpy(g["y"])[:1]
    y = torch.cat([y1, 0.5 * y1.roll(777, -1), 2.0 * y1.flip(-1), 0.7 * y1.roll(-3000, -1), 1.3 * y1.roll(50, -1)])
    B, G = y.shape[0], len(sizes)
    args = sampler.make_args(sample_rate=int(g["sr"]), audio_len=y.shape[1], T=4, NFFT=int(g["nfft"]), max_iter=5)
    s = sampler.BlindSamplerFused(ToyDenoiser(), edm.EDM(args), args, rid=False)
    s.filter_groups = sizes
    s.noise_fn = _row_noise([torch.Generator().manual_seed(10 + r) for r in range(B)], range(B))
    x, p, den, t, filt = s.predict_blind_bwe(y.clone(), rid=True, max_steps=2)
    assert x.shape == y.shape and p.shape == (G, 2, 5) and filt.shape == (4, G, 2, 5)
    assert s.filter_groups == sizes and s._groups is None
    s.filter_groups = None
    o = 0
    for gi, n in enumerate(sizes):
        rows = range(o, o + n)
        s.noise_fn = _row_noise({r: torch.Generator().manual_seed(10 + r) for r in rows}, rows)
        xg, pg = s.predict_blind_bwe(y[o:o + n].clone(), max_steps=2)
        assert rel_l2(x[o:o + n], xg) < 1e-6, gi
        assert rel_l2(p[gi], pg) < 1e-6, gi
        o += n


# --------------------------------------------------------------------------- the driver
class _GroupStub:
    """Records every call's groups and seeds; 'restoration' = 2 x the input, the filter of group g = (sum of its rows,
    its size) so that a merge error or a group mix-up shows."""
    joint = False

    def __init__(self):
        self.filter_groups, self.filter_per_row, self.row_seeds = None, True, [7]
        self.calls = []

    def predict_blind_bwe(self, y, rid=False):
        assert not self.filter_per_row
        sizes = self.filter_groups if self.filter_groups is not None else [y.shape[0]]
        self.calls.append((list(sizes), None if self.row_seeds is None else list(self.row_seeds)))
        filts, o = [], 0
        for n in sizes:
            filts.append(torch.tensor([[float(y[o:o + n].sum())], [float(n)]]))
            o += n
        f = torch.stack(filts)
        return 2.0 * y, (f if self.filter_groups is not None else f[0])


def _recs(lengths, seed=0):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(1, L, generator=g) for L in lengths]


def test_restore_recordings_packing_groups_and_seeds():
    from babe_b200 import segments
    seg_len = 4096
    recs = _recs([30000, 9000, 20000, 4000, 16000])
    sizes = [segments.split(r, seg_len)[0].shape[0] for r in recs]
    assert sizes == [9, 3, 6, 2, 5]
    s = _GroupStub()
    seeds = [11, 12, 13, 14, 15]
    out = segments.restore_recordings(s, recs, seg_len, seeds=seeds, max_rows=12)
    # greedy, in order, whole recordings: [9, 3] | [6, 2] | [5]
    assert [c[0] for c in s.calls] == [[9, 3], [6, 2], [5]]
    rows_of = [[0, 1], [2, 3], [4]]
    for (groups, got), rs in zip(s.calls, rows_of):
        assert got == [segments.row_seed(seeds[r], k) for r in rs for k in range(sizes[r])]
    # the sampler's settings are restored
    assert s.filter_groups is None and s.filter_per_row is True and s.row_seeds == [7]
    # one call without max_rows, no seeds: the sampler's own noise source stays
    s2 = _GroupStub()
    out2 = segments.restore_recordings(s2, recs, seg_len)
    assert s2.calls == [(sizes, [7])]
    for (a, fa), (b, fb) in zip(out, out2):
        assert torch.equal(a, b) and len(fa) == len(fb)
    with pytest.raises(ValueError, match="max_rows"):
        segments.restore_recordings(_GroupStub(), recs, seg_len, max_rows=8)        # recording 0 has 9 segments
    with pytest.raises(ValueError, match="max_rows"):
        segments.restore_recordings(_GroupStub(), recs, seg_len, max_rows=0)
    with pytest.raises(ValueError, match="seeds"):
        segments.restore_recordings(_GroupStub(), recs, seg_len, seeds=[1, 2])
    assert segments.restore_recordings(_GroupStub(), [], seg_len, max_rows=4) == []
    j = _GroupStub()
    j.joint = True
    with pytest.raises(ValueError, match="joint"):
        segments.restore_recordings(j, recs, seg_len)


def test_restore_recordings_merge_equals_restore_recording_joint():
    from babe_b200 import segments
    seg_len = 4096
    recs = _recs([30000, 9000, 20000], seed=1)
    out = segments.restore_recordings(_GroupStub(), recs, seg_len, max_rows=12)
    for r, rec in enumerate(recs):
        ref_s = _GroupStub()
        ref_s.filter_per_row = False
        ref, ref_fd = segments.restore_recording(ref_s, rec, seg_len, joint=True)
        got, fd = out[r]
        assert got.shape == rec.shape and torch.equal(got, ref)
        assert [sp for sp, _ in fd] == [sp for sp, _ in ref_fd]
        for (_, f), (_, fr) in zip(fd, ref_fd):
            assert f.shape == fr.shape == (2, 1) and torch.equal(f, fd[0][1])       # one filter per recording
            assert rel_l2(f, fr) < 1e-6
