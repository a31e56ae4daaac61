"""GPU: the known-prefix masked operator of the autoregressive windows (``babe_apply_filter_rows_known``: the MASK
instantiations of k_filter_fused and the row-by-row fallback) against a float64 evaluation of D_b / D_b^T built from
the oracle filter, the per-row conditional sampler path (``predict_bwe_AR`` with ``filter_per_row``) and the batched
autoregressive driver ``segments.restore_recordings_ar`` against the sequential one.

D_b x = m_b x + (1 - m_b) A_b x with m_b[n] = 1 for n < known[b]; the residual epilogue subtracts y and sums squares,
the adjoint is D_b^T r = A_b^T (r 1[n >= known[b]]) + r 1[n < known[b]] times the row scale."""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from toy_model import ToyDenoiser

pytestmark = pytest.mark.gpu

SR = 22050
TOL = 1e-5
FILTERS = [([310.7, 905.2, 2200.9], [-6.0, -12.0, -20.0]), ([1500.3, 4000.1, 9000.2], [-3.0, -25.0, -40.0]),
           ([700.3, 1900.8, 5100.2], [-8.0, -15.0, -30.0])]


@pytest.fixture(scope="module", autouse=True)
def _built():
    from babe_b200 import build
    build.build()


@pytest.fixture
def fused_variant(request):
    from babe_b200._lib import lib
    was = lib().babe_get_fused_variant()
    lib().babe_set_fused_variant(request.param)
    yield request.param
    lib().babe_set_fused_variant(was)


def _params(B):
    fc = torch.tensor([FILTERS[b % 3][0] for b in range(B)])
    A = torch.tensor([FILTERS[b % 3][1] for b in range(B)])
    return fc, A


def _known_values(T):
    return [0, 1, 2047, 2048, 2049, 5512, T - 1, T]


def _ref(x, fc, A, known, nfft, adjoint=False, sub=None, scale=None):
    """D_b x (- sub) or D_b^T x (* scale) in float64 from the oracle filter."""
    from oracle import stft_filter as sf
    f = torch.fft.rfftfreq(nfft, d=1 / SR).double()
    B, T = x.shape
    out = []
    for b in range(B):
        H = sf.design_filter(fc[b].double(), A[b].double(), f)
        xb = x[b:b + 1].double()
        pre = torch.arange(T) < int(known[b])
        if adjoint:
            yb = sf.apply_filter_adjoint(xb.masked_fill(pre, 0.0), H, nfft) + xb * pre
            if scale is not None:
                yb = yb * float(scale[b])
        else:
            yb = torch.where(pre, xb, sf.apply_filter(xb, H, nfft))
            if sub is not None:
                yb = yb - sub[b:b + 1].double()
        out.append(yb)
    return torch.cat(out)


# (B, T, nfft): runs that cross row boundaries, the benchmark length, the NFFT-1024 fallback, rows that cannot be
# bulk-copied (fallback); each case gets different known-prefix lengths on its rows, all eight values are covered
CASES = [(3, 1_000_000, 4096, 0), (8, 184184, 4096, 0), (2, 132300, 1024, 3), (3, 50001, 4096, 5)]


@pytest.mark.parametrize("fused_variant", [0, -1], indirect=True)
@pytest.mark.parametrize("B,T,nfft,offset", CASES)
def test_masked_operator_vs_fp64(fused_variant, B, T, nfft, offset):
    from babe_b200 import ops
    g = torch.Generator().manual_seed(B * 7 + T % 1000)
    x = torch.randn(B, T, generator=g) * 0.1
    sub = torch.randn(B, T, generator=g) * 0.05
    scale = torch.rand(B, generator=g) + 0.5
    kv = _known_values(T)
    known = torch.tensor([kv[(b + offset) % 8] for b in range(B)], dtype=torch.int32)
    assert len(set(known.tolist())) == B
    fc, A = _params(B)
    f = torch.fft.rfftfreq(nfft, d=1 / SR).cuda()
    xc, kc, fcc, Ac = x.cuda(), known.cuda(), fc.cuda(), A.cuda()
    ss = torch.zeros(B, dtype=torch.float64, device="cuda")
    fwd = ops.apply_filter_rows(xc, nfft, f, fcc, Ac, known=kc)
    res = ops.apply_filter_rows(xc, nfft, f, fcc, Ac, sub=sub.cuda(), row_sumsq=ss, known=kc)
    adj = ops.apply_filter_rows(xc, nfft, f, fcc, Ac, adjoint=True, known=kc)
    adj_s = ops.apply_filter_rows(xc, nfft, f, fcc, Ac, adjoint=True, row_scale=scale.cuda(), known=kc)
    torch.cuda.synchronize()
    r_fwd = _ref(x, fc, A, known, nfft)
    r_res = _ref(x, fc, A, known, nfft, sub=sub)
    r_adj = _ref(x, fc, A, known, nfft, adjoint=True)
    r_adj_s = _ref(x, fc, A, known, nfft, adjoint=True, scale=scale)
    for name, y, r in (("fwd", fwd, r_fwd), ("res", res, r_res), ("adj", adj, r_adj), ("adj_s", adj_s, r_adj_s)):
        for b in range(B):
            assert rel_l2(y[b].cpu(), r[b]) <= TOL, (name, b, int(known[b]))
    ss_ref = (r_res ** 2).sum(1)
    assert float(((ss.cpu() - ss_ref).abs() / ss_ref).max()) <= 1e-6
    # the known samples pass through exactly (forward) / are added exactly (adjoint, up to the filtered remainder)
    for b in range(B):
        k = int(known[b])
        assert torch.equal(fwd[b, :k].cpu(), x[b, :k])
        assert torch.equal(res[b, :k].cpu(), x[b, :k] - sub[b, :k])


@pytest.mark.parametrize("fused_variant", [0, -1], indirect=True)
def test_masked_operator_limits_are_bitwise(fused_variant):
    """known = 0 everywhere is the unmasked operator bit for bit (on the fused kernel; the fallback adds its prefix
    pass); known = T makes the residual x - sub bit for bit."""
    from babe_b200 import ops
    B, T, nfft = 8, 184184, 4096
    g = torch.Generator().manual_seed(2)
    x = (torch.randn(B, T, generator=g) * 0.1).cuda()
    sub = (torch.randn(B, T, generator=g) * 0.05).cuda()
    scale = (torch.rand(B, generator=g) + 0.5).cuda()
    fc, A = (t.cuda() for t in _params(B))
    f = torch.fft.rfftfreq(nfft, d=1 / SR).cuda()
    zero = torch.zeros(B, dtype=torch.int32, device="cuda")
    full = torch.full((B,), T, dtype=torch.int32, device="cuda")
    ss0, ss1 = (torch.zeros(B, dtype=torch.float64, device="cuda") for _ in range(2))
    r0 = ops.apply_filter_rows(x, nfft, f, fc, A, sub=sub, row_sumsq=ss0, known=zero)
    r1 = ops.apply_filter_rows(x, nfft, f, fc, A, sub=sub, row_sumsq=ss1)
    a0 = ops.apply_filter_rows(x, nfft, f, fc, A, adjoint=True, row_scale=scale, known=zero)
    a1 = ops.apply_filter_rows(x, nfft, f, fc, A, adjoint=True, row_scale=scale)
    if fused_variant == 0:
        assert torch.equal(r0, r1) and torch.equal(ss0, ss1) and torch.equal(a0, a1)
    else:
        assert rel_l2(r0.cpu(), r1.cpu()) < 1e-6 and rel_l2(a0.cpu(), a1.cpu()) < 1e-6
        assert rel_l2(ss0.cpu(), ss1.cpu()) < 1e-6
    ssf = torch.zeros(B, dtype=torch.float64, device="cuda")
    rf = ops.apply_filter_rows(x, nfft, f, fc, A, sub=sub, row_sumsq=ssf, known=full)
    assert torch.equal(rf, x - sub)
    assert rel_l2(ssf.cpu(), ((x - sub).double() ** 2).sum(1).cpu()) < 1e-9
    af = ops.apply_filter_rows(x, nfft, f, fc, A, adjoint=True, row_scale=scale, known=full)
    assert torch.equal(af, x * scale[:, None])


@pytest.mark.parametrize("fused_variant", [0, -1], indirect=True)
def test_masked_operator_adjoint_identity_and_rows(fused_variant):
    """<D x, r> = <x, D^T r> in fp64, and row r of a masked call is the B = 1 call on row r."""
    from babe_b200 import ops
    B, T, nfft = 5, 184184, 4096
    g = torch.Generator().manual_seed(3)
    x = (torch.randn(B, T, generator=g) * 0.1).cuda()
    r = (torch.randn(B, T, generator=g) * 0.1).cuda()
    known = torch.tensor([0, 2049, 5512, 100000, T], dtype=torch.int32, device="cuda")
    fc, A = (t.cuda() for t in _params(B))
    f = torch.fft.rfftfreq(nfft, d=1 / SR).cuda()
    Dx = ops.apply_filter_rows(x, nfft, f, fc, A, known=known).double()
    Dtr = ops.apply_filter_rows(r, nfft, f, fc, A, adjoint=True, known=known).double()
    lhs, rhs = (Dx * r.double()).sum(1), (x.double() * Dtr).sum(1)
    norm = Dx.norm(dim=1) * r.double().norm(dim=1)
    assert float(((lhs - rhs).abs() / norm).max()) <= 1e-6
    res = ops.apply_filter_rows(x, nfft, f, fc, A, sub=r, known=known)
    for b in range(B):
        one = ops.apply_filter_rows(x[b:b + 1], nfft, f, fc[b:b + 1], A[b:b + 1], sub=r[b:b + 1], known=known[b:b + 1])
        assert rel_l2(res[b].cpu(), one[0].cpu()) <= 1e-6, b


# --------------------------------------------------------------------------- the per-row sampler path
SEEDS = [2 ** 63 + 101, 102, 2 ** 40 + 103]


def _ar_sampler(T, nfft=4096, sr=SR, per_row=True):
    from babe_b200 import edm, sampler
    args = sampler.make_args(sample_rate=sr, audio_len=T, T=3, NFFT=nfft, filter_per_row=per_row)
    args.tester.complete_recording = sampler._ns(inpaint_DC=True)
    return sampler.BlindSamplerFused(ToyDenoiser().cuda(), edm.EDM(args), args, rid=False)


def _ar_inputs(T=16384):
    g = torch.Generator().manual_seed(9)
    ylpf = 0.05 * torch.randn(3, T, generator=g)
    y_masked = torch.zeros(3, T)
    mask = torch.zeros(3, T)
    for b, k in enumerate((5512, 2100, 9000)):
        mask[b, :k] = 1
        y_masked[b, :k] = 0.05 * torch.randn(k, generator=g)
    filt = torch.tensor([[FILTERS[b][0], FILTERS[b][1]] for b in range(3)])
    return ylpf.cuda(), y_masked.cuda(), mask.cuda(), filt.cuda()


def test_per_row_predict_bwe_AR(monkeypatch):
    from babe_b200 import sampler
    torch.backends.cudnn.deterministic = True
    ylpf, y_masked, mask, filt = _ar_inputs()
    s = _ar_sampler(ylpf.shape[1])
    s.row_seeds = SEEDS
    x = s.predict_bwe_AR(ylpf, y_masked, filt, "fc_A", mask=mask)
    for r in range(3):
        s.row_seeds = [SEEDS[r]]
        xr = s.predict_bwe_AR(ylpf[r:r + 1], y_masked[r:r + 1], filt[r], "fc_A", mask=mask[r:r + 1])
        assert rel_l2(x[r].cpu(), xr[0].cpu()) <= 1e-5, r
    # another row's input changes nothing in rows 0 and 2
    y2 = ylpf.clone()
    y2[1] = y2[1].flip(-1) * 3
    s.row_seeds = SEEDS
    x2 = s.predict_bwe_AR(y2, y_masked, filt, "fc_A", mask=mask)
    assert torch.equal(x2[0], x[0]) and torch.equal(x2[2], x[2]) and not torch.equal(x2[1], x[1])
    # the fused masked route equals the eager composition D(x) = m x + (1 - m) A x
    monkeypatch.setattr(sampler, "known_prefix_lengths", lambda m: None)
    s.row_seeds = SEEDS
    xe = s.predict_bwe_AR(ylpf, y_masked, filt, "fc_A", mask=mask)
    for r in range(3):
        assert rel_l2(xe[r].cpu(), x[r].cpu()) <= 1e-5, r


def test_per_row_predict_bwe_AR_at_one_row_is_the_default_mode(golden):
    g = golden("sampler_ar.npz")
    torch.backends.cudnn.deterministic = True
    t = lambda k: torch.from_numpy(g[k][:1]).cuda()     # noqa: E731
    nfft, sr = int(g["nfft"]), int(g["sr"])
    filt = torch.from_numpy(g["filt"]).cuda()
    outs = []
    for per_row in (False, True):
        s = _ar_sampler(g["x"].shape[1], nfft=nfft, sr=sr, per_row=per_row)
        s.row_seeds = [SEEDS[0]]
        outs.append(s.predict_bwe_AR(t("ylpf"), t("y_masked"), filt, "fc_A", mask=t("mask")))
    assert rel_l2(outs[1].cpu(), outs[0].cpu()) <= 1e-5


# --------------------------------------------------------------------------- the batched driver
def _recording(L, seed):
    from oracle import stft_filter as osf
    gen = torch.Generator().manual_seed(seed)
    t = torch.arange(L) / SR
    rec = 0.05 * torch.sin(2 * np.pi * (220 + 110 * seed) * t) + 0.01 * torch.randn(L, generator=gen)
    f = torch.fft.rfftfreq(4096, d=1 / SR)
    return osf.apply_filter(rec[None], osf.design_filter(torch.tensor([2000.0]), torch.tensor([-30.0]), f), 4096).cuda()


def test_restore_recordings_ar_matches_sequential():
    from babe_b200 import edm, sampler, segments
    torch.backends.cudnn.deterministic = True
    seg_len = 8192
    recs = [_recording(L, i) for i, L in enumerate((20000, 30000, 45000))]
    seeds = [7, 2 ** 64 - 8, 9]
    args = sampler.make_args(audio_len=seg_len, T=3, NFFT=4096, max_iter=5)
    s = sampler.BlindSamplerFused(ToyDenoiser().cuda(), edm.EDM(args), args, rid=False)
    filters = [torch.tensor([FILTERS[i][0], FILTERS[i][1]]).cuda() for i in range(3)]
    seq = [segments.restore_recording_ar(s, recs[i].clone(), seg_len, SR, estimated_filter=filters[i], seed=seeds[i])
           for i in range(3)]
    bat = segments.restore_recordings_ar(s, [r.clone() for r in recs], seg_len, SR, seeds=seeds,
                                         estimated_filters=filters)
    assert s.row_seeds is None and s.filter_per_row is False
    for i in range(3):
        assert bat[i][0].shape == recs[i].shape
        assert rel_l2(bat[i][0].cpu(), seq[i][0].cpu()) <= 1e-4, i
        assert torch.equal(bat[i][1], filters[i])
    # the blind step on the first windows in one per-row call: the filter fit is chaotic in the last bits (the
    # tolerance of the existing batched blind tests)
    seq_b = [segments.restore_recording_ar(s, recs[i].clone(), seg_len, SR, n_segments_blindstep=1, seed=seeds[i])
             for i in range(3)]
    bat_b = segments.restore_recordings_ar(s, [r.clone() for r in recs], seg_len, SR, n_segments_blindstep=1,
                                           seeds=seeds)
    for i in range(3):
        assert bat_b[i][1].shape == seq_b[i][1].shape == (2, 5)
        assert rel_l2(bat_b[i][1].cpu(), seq_b[i][1].cpu()) <= 1e-2, i
        assert torch.isfinite(bat_b[i][0]).all()
