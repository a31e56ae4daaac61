"""CPU: host logic of the non-blind / autoregressive sampling methods of BlindSamplerFused
(predict_conditional, predict_bwe_AR, get_score, prepare_smooth_mask) against trajectories of the
UNMODIFIED reference sampler (tests/golden/make_golden_ar.py).  The CUDA operator is replaced by the
oracle here -- this checks the loop, the masks and the data-consistency step, not the kernels
(tests/test_sampler_gpu.py runs the same comparison on the CUDA operators)."""
import torch

from conftest import rel_l2
from toy_model import ToyDenoiser


def _sampler(g):
    from babe_b200 import edm, sampler
    from oracle import stft_filter as osf
    nfft = int(g["nfft"])

    class CpuSampler(sampler.BlindSamplerFused):
        def apply_filter_fcA(self, x, p):
            return osf.apply_filter(x, osf.design_filter(p[0], p[1], self.freqs), nfft)

    args = sampler.make_args(sample_rate=int(g["sr"]), audio_len=g["x"].shape[1], T=4, NFFT=nfft, max_iter=20)
    args.tester.complete_recording = sampler._ns(inpaint_DC=True)
    return CpuSampler(ToyDenoiser(), edm.EDM(args), args, rid=False), args


def test_predict_bwe_AR_matches_reference(golden):
    g = golden("sampler_ar.npz")
    s, args = _sampler(g)
    t = lambda k: torch.from_numpy(g[k])
    torch.manual_seed(77)
    x = s.predict_bwe_AR(t("ylpf"), t("y_masked"), t("filt"), "fc_A", mask=t("mask"))
    assert rel_l2(x, g["x_ar"]) < 1e-4
    # the known head is reproduced through the data-consistency step
    assert rel_l2(x[:, :1100], g["x"][:, :1100]) < 1e-2


def test_predict_conditional_matches_reference_predict_bwe(golden):
    g = golden("sampler_ar.npz")
    s, args = _sampler(g)
    t = lambda k: torch.from_numpy(g[k])
    s.freqs = torch.fft.rfftfreq(int(g["nfft"]), d=1 / int(g["sr"]))
    filt = t("filt")
    torch.manual_seed(78)
    x = s.predict_conditional(t("ylpf"), lambda v: s.apply_filter_fcA(v, filt))
    assert rel_l2(x, g["x_bwe"]) < 1e-4


def test_smooth_mask_literal():
    """prepare_smooth_mask against the reference's loop (testing/blind_bwe_sampler.py:232-257)."""
    from babe_b200.sampler import BlindSamplerFused as S

    def literal(mask, size):
        hann = torch.hann_window(size * 2)
        m, prev, new = mask[0], 1, mask[0].clone()
        for i in range(len(m)):
            if m[i] != prev:
                if m[i] == 0:
                    new[i - size:i] = hann[size:]
                if m[i] == 1:
                    new[i:i + size] = hann[:size]
            prev = m[i]
        return new.unsqueeze(0).expand(mask.shape[0], -1)

    m = torch.ones(2, 400)
    m[:, 150:250] = 0
    assert torch.equal(S.prepare_smooth_mask(m, 20), literal(m, 20))
    m = torch.ones(3, 300)
    m[:, 120:] = 0
    assert torch.equal(S.prepare_smooth_mask(m, 50), literal(m, 50))


def test_cuda_graph_option_falls_back_to_eager_without_cuda(golden, monkeypatch):
    """``cuda_graph=True`` must never break sampling: any capture problem -> eager model + a warning.  The capture is
    made to fail, as it does without a CUDA device, so that the fallback is exercised on GPU machines too."""
    import pytest

    def no_capture(*a, **k):
        raise RuntimeError("CUDA-graph capture unavailable")
    monkeypatch.setattr(torch.cuda, "make_graphed_callables", no_capture)
    g = golden("sampler_ar.npz")
    s, args = _sampler(g)
    s.cuda_graph = True
    x = torch.zeros(2, 64, requires_grad=True)
    with pytest.warns(UserWarning, match="capture of the denoiser failed"):
        net = s._graphed_model(x)
    assert net is s.model
    assert s._graphed_model(x) is s.model                      # cached decision, no second attempt
