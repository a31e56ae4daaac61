"""CPU: batched autoregressive restoration of several recordings (``segments.restore_recordings_ar``) and the per-row
conditional path of the sampler (``predict_bwe_AR`` / ``predict_bwe`` with ``filter_per_row``).  The window placement
and the driver run on stub samplers; the sampler runs with the CUDA row operator replaced by a per-row loop over the
oracle, including the known-prefix masked operator.  The kernels are checked on the GPU (tests/test_ar_rows_gpu.py)."""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from toy_model import ToyDenoiser

from babe_b200 import segments


# --------------------------------------------------------------------------- window placement
class _WindowStub:
    """Records the input windows of the AR driver; 'restoration' = 2 x the input outside the mask."""
    filter_per_row, row_seeds, joint = False, None, False

    def __init__(self):
        self.segs = []

    def predict_bwe(self, seg, filt, typefilter, rid=False):
        self.segs.append(seg.clone())
        return 2 * seg

    def predict_bwe_AR(self, seg, y_masked, filt, typefilter, rid=False, mask=None):
        self.segs.append(seg.clone())
        return mask * y_masked + (1 - mask) * 2 * seg


@pytest.mark.parametrize("L", [400, 500, 850, 1730, 5000])
def test_ar_windows_are_the_windows_restore_recording_ar_visits(L):
    # seg_len 400, overlap 50, discard_end 200 -> hop 150.  L = 400 / 500: no autoregressive window; 850: the
    # remainder is exactly one window long (n = seg_len); 1730 / 5000: many windows and a padded last one
    segL, overlap = 400, 50
    x = torch.randn(1, L, generator=torch.Generator().manual_seed(L))
    s = _WindowStub()
    segments.restore_recording_ar(s, x.clone(), segL, 1000, overlap_s=0.05, estimated_filter=torch.zeros(2, 1))
    wins = segments.ar_windows(L, segL, overlap, 200, 0)
    assert len(s.segs) == len(wins)
    assert wins[0] == (0, segL) and all(n == segL for _, n in wins[:-1])
    xn = 0.1 * x / x.std(-1)
    for seg, (ix, n) in zip(s.segs, wins):
        ref = torch.zeros(1, segL)
        ref[:, :n] = xn[:, ix:ix + n]
        assert torch.equal(seg, ref), (ix, n)
    ix, n = wins[-1]
    assert ix + n == L and 0 < n <= segL
    if L == 850:
        assert wins[-1] == (450, segL) and len(wins) == 4
    if L <= 500:
        assert len(wins) == 2


# --------------------------------------------------------------------------- the batched driver
class _RowStub:
    """A row-independent sampler: every output row depends on that row's input, filter and seed alone.  Records
    (method, rows, row seeds) of every call."""
    joint = False

    def __init__(self):
        self.calls, self.filter_per_row, self.row_seeds = [], False, None

    def _seed_term(self, B):
        if self.row_seeds is None:
            return torch.zeros(B, 1)
        return torch.tensor([[(int(s) % 997) * 1e-3] for s in self.row_seeds])

    def _filt_term(self, filt, B):
        f = filt if filt.dim() == 3 else filt.unsqueeze(0).expand(B, -1, -1)
        return f[:, 0, :1] * 1e-4

    def predict_blind_bwe(self, y, rid=False):
        self.calls.append(("blind", y.shape[0], self.row_seeds, self.filter_per_row))
        est = torch.stack([y.std(-1) * 1000, -20 + y.mean(-1)], -1).unsqueeze(-1)      # (B, 2, 1)
        return 1.5 * y + self._seed_term(y.shape[0]), est if self.filter_per_row else est[0]

    def predict_bwe(self, seg, filt, typefilter, rid=False):
        self.calls.append(("bwe", seg.shape[0], self.row_seeds, self.filter_per_row))
        B = seg.shape[0]
        return 2 * seg + self._seed_term(B) + self._filt_term(filt, B)

    def predict_bwe_AR(self, seg, y_masked, filt, typefilter, rid=False, mask=None):
        self.calls.append(("ar", seg.shape[0], self.row_seeds, self.filter_per_row))
        B = seg.shape[0]
        return mask * y_masked + (1 - mask) * (2 * seg + self._seed_term(B) + self._filt_term(filt, B))


def _recordings():
    g = torch.Generator().manual_seed(5)
    return [torch.randn(1, L, generator=g) * a for L, a in ((1000, 1.0), (1730, 0.3), (3100, 2.0))]


@pytest.mark.parametrize("blindstep", [None, 1, 2])
def test_restore_recordings_ar_equals_sequential_calls(blindstep):
    recs, seeds = _recordings(), [11, 22, 2 ** 64 - 5]
    kw = dict(overlap_s=0.05, discard_end=200)
    filters = None if blindstep else [torch.tensor([[500.0 + 100 * r], [-20.0]]) for r in range(3)]
    nb = blindstep or 2
    ref = []
    rng = np.random.RandomState(4)
    for r in range(3):
        ref.append(segments.restore_recording_ar(_RowStub(), recs[r].clone(), 400, 1000, n_segments_blindstep=nb,
                                                 seed=seeds[r], rng=rng, estimated_filter=None if filters is None
                                                 else filters[r], **kw))
    s = _RowStub()
    out = segments.restore_recordings_ar(s, [r.clone() for r in recs], 400, 1000, n_segments_blindstep=nb,
                                         seeds=seeds, rng=np.random.RandomState(4), estimated_filters=filters, **kw)
    assert len(out) == 3
    for r in range(3):
        assert out[r][0].shape == recs[r].shape
        assert rel_l2(out[r][0], ref[r][0]) < 1e-6, r
        assert torch.allclose(out[r][1], ref[r][1]), r
    assert not s.filter_per_row and s.row_seeds is None              # the sampler's settings are restored
    wins = [len(segments.ar_windows(x.shape[-1], 400, 50, 200, 0)) for x in recs]
    calls = [c for c in s.calls if c[0] != "blind"]
    assert len(calls) == max(wins)
    for w, (kind, B, row_seeds, per_row) in enumerate(calls):
        rows = [r for r in range(3) if w < wins[r]]
        assert kind == ("bwe" if w == 0 else "ar") and per_row
        assert B == len(rows)                                        # the batch shrinks as recordings finish
        assert row_seeds == [segments.row_seed(seeds[r], w) for r in rows]
    assert [c[1] for c in calls] == sorted([c[1] for c in calls], reverse=True) and calls[-1][1] == 1
    blind = [c for c in s.calls if c[0] == "blind"]
    if blindstep == 1:
        assert len(blind) == 1 and blind[0][1] == 3 and blind[0][3]
        assert blind[0][2] == [segments.row_seed(sd, 1 << 32) for sd in seeds]
    elif blindstep == 2:
        assert [c[1] for c in blind] == [2, 2, 2] and not any(c[3] for c in blind)
        assert blind[1][2] == [segments.row_seed(seeds[1], (1 << 32) + j) for j in range(2)]


def test_restore_recordings_ar_rejections():
    recs = _recordings()
    s = _RowStub()
    with pytest.raises(ValueError, match="fewer than seg_len"):
        segments.restore_recordings_ar(s, recs, 1200, 1000, estimated_filters=[torch.zeros(2, 1)] * 3)
    with pytest.raises(ValueError, match="one device"):
        segments.restore_recordings_ar(s, [recs[0], torch.zeros(1, 1000, device="meta")], 400, 1000)
    with pytest.raises(NotImplementedError):
        segments.restore_recordings_ar(s, recs, 400, 1000, typefilter="firwin")
    s.joint = True
    with pytest.raises(ValueError, match="joint"):
        segments.restore_recordings_ar(s, recs, 400, 1000)
    assert s.calls == []


# --------------------------------------------------------------------------- masks
def test_known_prefix_lengths():
    from babe_b200.sampler import known_prefix_lengths
    m = torch.zeros(4, 300)
    m[0, :50] = 1
    m[1] = 1
    m[3, :299] = 1
    k = known_prefix_lengths(m)
    assert k.dtype == torch.int32 and k.tolist() == [50, 300, 0, 299]
    holes = m.clone()
    holes[0, 20] = 0                                                 # a gap inside the prefix
    assert known_prefix_lengths(holes) is None
    late = m.clone()
    late[2, 100:110] = 1                                             # known samples after unknown ones
    assert known_prefix_lengths(late) is None
    soft = m.clone()
    soft[1, 5] = 0.5                                                 # not a 0/1 mask
    assert known_prefix_lengths(soft) is None


def test_smooth_mask_rows():
    from babe_b200.sampler import BlindSamplerFused as S
    m = torch.zeros(4, 600)
    for b, k in enumerate((300, 600, 120, 80)):
        m[b, :k] = 1
    m[3, 400:] = 1                                                   # any row pattern, one row at a time
    sm = S.prepare_smooth_mask_rows(m, 50)
    assert sm.shape == m.shape
    for b in range(4):
        assert torch.equal(sm[b], S.prepare_smooth_mask(m[b:b + 1], 50)[0]), b
    assert not torch.equal(sm[0], sm[3])


# --------------------------------------------------------------------------- per-row sampler on the oracle
@pytest.fixture
def oracle_rows(monkeypatch):
    """ops.apply_filter_rows (with ``known``) and the eager per-row filter as loops over the oracle."""
    from babe_b200 import ops, sampler
    from oracle import stft_filter as osf
    calls = []

    def apply_filter_rows(x, nfft, freqs, fc, A, adjoint=False, sub=None, row_scale=None, row_sumsq=None,
                          out=None, status=None, known=None):
        calls.append(known is not None)
        T = x.shape[1]
        rows = []
        for b in range(x.shape[0]):
            H = osf.design_filter(fc[b], A[b], freqs)
            xb = x[b:b + 1]
            pre = torch.arange(T) < (int(known[b]) if known is not None else 0)
            if adjoint:
                yb = osf.apply_filter_adjoint(xb.masked_fill(pre, 0.0), H, nfft) + xb * pre
            else:
                yb = torch.where(pre, xb, osf.apply_filter(xb, H, nfft))
                if sub is not None:
                    yb = yb - sub[b:b + 1]
            if row_scale is not None:
                yb = yb * row_scale[b]
            if row_sumsq is not None:
                row_sumsq[b] += (yb.double() ** 2).sum()
            rows.append(yb)
        return torch.cat(rows)

    def apply_filter_fcA(self, x, p):
        if p.dim() == 3:
            return torch.cat([osf.apply_filter(x[b:b + 1], osf.design_filter(p[b, 0], p[b, 1], self.freqs), 4096)
                              for b in range(x.shape[0])])
        return osf.apply_filter(x, osf.design_filter(p[0], p[1], self.freqs), 4096)

    monkeypatch.setattr(ops, "apply_filter_rows", apply_filter_rows)
    monkeypatch.setattr(sampler.BlindSamplerFused, "apply_filter_fcA", apply_filter_fcA)
    # oneDNN's conv1d rounds the toy denoiser differently at batch 3 and at batch 1 (~1e-7 relative per evaluation,
    # ~2e-6 after a few steps); the native CPU convolution is row-independent to the bit
    with torch.backends.mkldnn.flags(enabled=False):
        yield calls


def _row_noise(seeds):
    gens = [torch.Generator().manual_seed(s) for s in seeds]
    return lambda shape, dev: torch.stack([torch.randn(shape[1], generator=g) for g in gens]).to(dev)


def _ar_inputs(T=8192):
    g = torch.Generator().manual_seed(9)
    ylpf = 0.05 * torch.randn(3, T, generator=g)
    y_masked = torch.zeros(3, T)
    mask = torch.zeros(3, T)
    for b, k in enumerate((1000, 2500, 4096)):
        mask[b, :k] = 1
        y_masked[b, :k] = 0.05 * torch.randn(k, generator=g)
    filt = torch.tensor([[[300.0, 1000.0], [-10.0, -30.0]], [[800.0, 3000.0], [-5.0, -40.0]],
                         [[2000.0, 5000.0], [-20.0, -25.0]]])
    return ylpf, y_masked, mask, filt


def _ar_sampler(T=8192):
    from babe_b200 import edm, sampler
    args = sampler.make_args(audio_len=T, T=3, NFFT=4096)
    args.tester.complete_recording = sampler._ns(inpaint_DC=True)
    s = sampler.BlindSamplerFused(ToyDenoiser(), edm.EDM(args), args)
    s.filter_per_row = True
    return s


def test_per_row_predict_bwe_AR_rows_equal_single_rows(oracle_rows, monkeypatch):
    from babe_b200 import sampler
    ylpf, y_masked, mask, filt = _ar_inputs()
    s = _ar_sampler()
    s.noise_fn = _row_noise([1, 2, 3])
    x = s.predict_bwe_AR(ylpf, y_masked, filt, "fc_A", mask=mask)
    assert oracle_rows and all(oracle_rows)                          # the prefix masks took the masked operator
    for r in range(3):
        s.noise_fn = _row_noise([1 + r])
        xr = s.predict_bwe_AR(ylpf[r:r + 1], y_masked[r:r + 1], filt[r], "fc_A", mask=mask[r:r + 1])
        assert rel_l2(x[r:r + 1], xr) < 1e-6, r
    # the eager composition (any non-prefix mask) computes the same restoration
    monkeypatch.setattr(sampler, "known_prefix_lengths", lambda m: None)
    oracle_rows.clear()
    s.noise_fn = _row_noise([1, 2, 3])
    xe = s.predict_bwe_AR(ylpf, y_masked, filt, "fc_A", mask=mask)
    assert not oracle_rows
    assert rel_l2(xe, x) < 1e-5


def test_per_row_predict_bwe_rows_equal_single_rows(oracle_rows):
    ylpf, _, _, filt = _ar_inputs()
    s = _ar_sampler()
    s.noise_fn = _row_noise([4, 5, 6])
    x = s.predict_bwe(ylpf, filt, "fc_A")
    for r in range(3):
        s.noise_fn = _row_noise([4 + r])
        xr = s.predict_bwe(ylpf[r:r + 1], filt[r:r + 1], "fc_A")
        assert rel_l2(x[r:r + 1], xr) < 1e-6, r


def test_per_row_conditional_rejections():
    ylpf, y_masked, mask, filt = _ar_inputs()
    s = _ar_sampler()
    with pytest.raises(NotImplementedError, match="FIR"):
        s.predict_bwe_AR(ylpf, y_masked, torch.ones(31), "firwin", mask=mask)
    with pytest.raises(NotImplementedError, match="FIR"):
        s.predict_bwe(ylpf, torch.ones(31), "firwin")
    with pytest.raises(ValueError, match="per-row filter parameters"):
        s.predict_bwe_AR(ylpf, y_masked, filt[:2], "fc_A", mask=mask)
