"""GPU: the CUDA constant-Q transform against the oracle NSGT (oracle/nsgt.py,
fp64 on the CPU).  PARITY UNPINNED versus upstream cqt_nsgt_pytorch (not
available offline); these tests pin the CUDA path to the in-repo specification
and check the invariants the reference's call sites rely on.  Tolerance:
relative L2 <= 1e-5 in fp32."""
import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu
TOL = 1e-5

CONFIGS = [(4, 12, 22050, 8192, 3), (5, 24, 44100, 30030, 2), (7, 64, 22050, 184184, 2),
           (7, 64, 22050, 132300, 1), (7, 64, 44100, 368368, 1), (8, 96, 44100, 485100, 1)]


@pytest.fixture(scope="module")
def CQT():
    from babe_b200 import build
    build.build()
    from cqt_nsgt_pytorch import CQT_nsgt
    return CQT_nsgt


def _pair(CQT, numocts, binsoct, fs, Ls):
    from oracle.nsgt import NSGT
    return (CQT(numocts, binsoct, mode="oct", window=("kaiser", 1), fs=fs, audio_len=Ls, device="cuda"),
            NSGT(numocts, binsoct, fs, Ls, ("kaiser", 1)))


@pytest.mark.parametrize("numocts,binsoct,fs,Ls,B", CONFIGS)
def test_fft_and_transform_vs_oracle(CQT, numocts, binsoct, fs, Ls, B):
    cq, ref = _pair(CQT, numocts, binsoct, fs, Ls)
    assert cq.size_per_oct == ref.M
    g = torch.Generator().manual_seed(Ls)
    x = torch.randn(B, Ls, generator=g) * 0.063
    xc = x.cuda()
    # the non-power-of-two real FFT itself
    X = cq.rfft(xc)
    Xr = torch.fft.rfft(x.double(), dim=-1)
    assert rel_l2(torch.view_as_real(X.cpu()), torch.view_as_real(Xr)) < TOL
    assert rel_l2(cq.irfft(Xr.to(torch.complex64).cuda()).cpu(), x) < TOL
    # analysis
    c = cq.fwd(xc.unsqueeze(1))
    cr = ref.fwd(x.double())
    assert len(c) == numocts
    for o in range(numocts):
        assert c[o].shape == (B, 1, binsoct, ref.M[o]) and c[o].dtype == torch.complex64
        assert rel_l2(torch.view_as_real(c[o].cpu().squeeze(1)), torch.view_as_real(cr[o])) < TOL, o
    # synthesis from the oracle's coefficients, and the round trip
    y = cq.bwd([ci.to(torch.complex64).unsqueeze(1).cuda() for ci in cr])
    assert y.shape == (B, 1, Ls)
    assert rel_l2(y.cpu().squeeze(1), ref.bwd(cr)) < TOL
    hp = ref.apply_hpf_DC(x.double())
    assert rel_l2(cq.bwd(c).cpu().squeeze(1), hp) < TOL
    assert rel_l2(cq.apply_hpf_DC(xc).cpu(), hp) < TOL
    assert rel_l2((cq.apply_hpf_DC(xc) + cq.apply_lpf_DC(xc)).cpu(), x) < TOL


@pytest.mark.parametrize("numocts,binsoct,fs,Ls,B", CONFIGS[:3])
def test_gradients_vs_oracle_autograd(CQT, numocts, binsoct, fs, Ls, B):
    cq, ref = _pair(CQT, numocts, binsoct, fs, Ls)
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, Ls, generator=g)
    cots = [torch.randn(B, binsoct, m, 2, generator=g) for m in ref.M]
    # d/dx of <fwd(x), cot>
    xr = x.double().requires_grad_(True)
    lr = sum((torch.view_as_real(c) * ct.double()).sum() for c, ct in zip(ref.fwd(xr), cots))
    (gr,) = torch.autograd.grad(lr, xr)
    xc = x.cuda().requires_grad_(True)
    lc = sum((torch.view_as_real(c.squeeze(1)) * ct.cuda()).sum() for c, ct in zip(cq.fwd(xc.unsqueeze(1)), cots))
    (gc,) = torch.autograd.grad(lc, xc)
    assert rel_l2(gc.cpu(), gr) < TOL
    # d/dc of <bwd(c), r>
    r = torch.randn(B, Ls, generator=g)
    cr = [torch.view_as_complex(ct.double()).requires_grad_(True) for ct in cots]
    grs = torch.autograd.grad((ref.bwd(cr) * r.double()).sum(), cr)
    cc = [torch.view_as_complex(ct.contiguous()).unsqueeze(1).cuda().requires_grad_(True) for ct in cots]
    gcs = torch.autograd.grad((cq.bwd(cc).squeeze(1) * r.cuda()).sum(), cc)
    for o in range(numocts):
        assert rel_l2(torch.view_as_real(gcs[o].cpu().squeeze(1)), torch.view_as_real(grs[o])) < TOL, o
    # hpf is self-adjoint
    xc = x.cuda().requires_grad_(True)
    (gh,) = torch.autograd.grad((cq.apply_hpf_DC(xc) * r.cuda()).sum(), xc)
    assert rel_l2(gh.cpu(), ref.apply_hpf_DC(r.double())) < TOL


def test_full_batch_properties(CQT):
    """Shipped configuration at the benchmark batch: adjoint identities and
    batch independence (size-independent properties, no CPU oracle run)."""
    cq = CQT(7, 64, mode="oct", window=("kaiser", 1), fs=22050, audio_len=184184, device="cuda")
    torch.manual_seed(0)
    B = 8
    x = torch.randn(B, 1, 184184, device="cuda") * 0.063
    c = cq.fwd(x)
    assert [ci.shape[-1] for ci in c] == [32, 64, 128, 256, 512, 1024, 2048]
    rec = cq.bwd(c)
    assert rel_l2(rec.cpu(), cq.apply_hpf_DC(x.squeeze(1)).unsqueeze(1).cpu()) < TOL
    c1 = cq.fwd(x[3:4])
    for a, b in zip(c, c1):
        assert torch.equal(a[3:4], b)
    cot = [torch.randn_like(torch.view_as_real(ci)) for ci in c]
    xg = x.clone().requires_grad_(True)
    loss = sum((torch.view_as_real(ci) * ct).sum() for ci, ct in zip(cq.fwd(xg), cot))
    (gx,) = torch.autograd.grad(loss, xg)
    d = torch.randn_like(x)
    lhs = sum((torch.view_as_real(ci) * ct).double().sum() for ci, ct in zip(cq.fwd(d), cot))
    assert abs(float(lhs - (gx.double() * d.double()).sum())) < 1e-4 * abs(float(lhs))


def test_planar_layout_matches_interleaved(CQT):
    """a21: (B,2,F,T) float planes written/read directly == view_as_real + permute of the complex API
    (networks/cqtdiff+.py:750-753, :826-830), forward values and both gradients."""
    cq = CQT(5, 24, mode="oct", window=("kaiser", 1), fs=44100, audio_len=30030, device="cuda")
    torch.manual_seed(3)
    x = torch.randn(3, 30030, device="cuda")
    c = cq.fwd(x.unsqueeze(1))
    p = cq.fwd_planar(x)
    for ci, pi in zip(c, p):
        ref = torch.view_as_real(ci.squeeze(1)).permute(0, 3, 1, 2).contiguous()
        assert pi.shape == ref.shape and torch.equal(pi, ref)
    assert torch.equal(cq.bwd_planar(p), cq.bwd(c).squeeze(1))
    cots = [torch.randn_like(pi) for pi in p]
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    la = sum((pi * ct).sum() for pi, ct in zip(cq.fwd_planar(xa), cots))
    lb = sum((torch.view_as_real(ci.squeeze(1)).permute(0, 3, 1, 2) * ct).sum()
             for ci, ct in zip(cq.fwd(xb.unsqueeze(1)), cots))
    (ga,), (gb,) = torch.autograd.grad(la, xa), torch.autograd.grad(lb, xb)
    assert rel_l2(ga.cpu(), gb.cpu()) < 1e-6
    pa = [pi.clone().requires_grad_(True) for pi in p]
    r = torch.randn(3, 30030, device="cuda")
    gpa = torch.autograd.grad((cq.bwd_planar(pa) * r).sum(), pa)
    ca = [ci.clone().requires_grad_(True) for ci in c]
    gca = torch.autograd.grad((cq.bwd(ca).squeeze(1) * r).sum(), ca)
    for gp, gc in zip(gpa, gca):
        assert rel_l2(gp.cpu(), torch.view_as_real(gc.squeeze(1)).permute(0, 3, 1, 2).cpu()) < 1e-6


@pytest.mark.parametrize("variant", [-1, 0, 1])
@pytest.mark.parametrize("numocts,binsoct,fs,Ls,B", [(4, 12, 22050, 8192, 3), (7, 64, 22050, 184184, 2),
                                                     (7, 64, 22050, 132300, 1), (8, 96, 44100, 485100, 1)])
def test_tiled_passes_vs_oracle(CQT, variant, numocts, binsoct, fs, Ls, B):
    """The other implementations of the length-Ls transform kept in the library (`babe_set_cqt_variant`: -1 = round 1's
    generic passes, which also serve every length the prime-factor passes are not instantiated for; 0 / 1 = round 2's
    tiled passes of csrc/cqt_fft.cuh) against the same oracle.  The default (2 = prime-factor passes of
    csrc/cqt_pfa.cuh for Ls = 184184 and 368368) is what every other test in this file runs."""
    from babe_b200._lib import lib
    cq, ref = _pair(CQT, numocts, binsoct, fs, Ls)
    g = torch.Generator().manual_seed(Ls + 1)
    x = torch.randn(B, Ls, generator=g) * 0.063
    xc = x.cuda()
    assert lib().babe_set_cqt_variant(variant) == 0
    try:
        X = cq.rfft(xc)
        Xr = torch.fft.rfft(x.double(), dim=-1)
        assert rel_l2(torch.view_as_real(X.cpu()), torch.view_as_real(Xr)) < TOL
        assert rel_l2(cq.irfft(Xr.to(torch.complex64).cuda()).cpu(), x) < TOL
        c = cq.fwd(xc.unsqueeze(1))
        cr = ref.fwd(x.double())
        for o in range(numocts):
            assert rel_l2(torch.view_as_real(c[o].cpu().squeeze(1)), torch.view_as_real(cr[o])) < TOL, o
        assert rel_l2(cq.bwd(c).cpu().squeeze(1), ref.bwd(cr)) < TOL
        assert rel_l2(cq.apply_hpf_DC(xc).cpu(), ref.apply_hpf_DC(x.double())) < TOL
    finally:
        lib().babe_set_cqt_variant(2)


@pytest.mark.parametrize("band_variant", [0, 2, 3])
@pytest.mark.parametrize("numocts,binsoct,fs,Ls,B", [(7, 64, 22050, 184184, 2), (4, 12, 22050, 8192, 3)])
def test_other_band_kernels_vs_oracle(CQT, band_variant, numocts, binsoct, fs, Ls, B):
    """`babe_set_cqt_band_variant`: 0 = round 2's band kernels (BandCore on split re / im registers, CTA-wide barriers,
    generic Stockham for the octaves below 256 points); 2 / 3 = the packed per-band cores of csrc/bandfft_v.cuh with
    cp.async / TMA bulk-copy staging on BOTH directions (the default, 1, stages the analysis slices by TMA and the
    synthesis rows by cp.async and is what every other test runs).  Complex and planar layouts."""
    from babe_b200._lib import lib
    cq, ref = _pair(CQT, numocts, binsoct, fs, Ls)
    g = torch.Generator().manual_seed(Ls + 2)
    x = torch.randn(B, Ls, generator=g) * 0.063
    xc = x.cuda()
    assert lib().babe_set_cqt_band_variant(band_variant) == 0
    try:
        c = cq.fwd(xc.unsqueeze(1))
        cr = ref.fwd(x.double())
        for o in range(numocts):
            assert rel_l2(torch.view_as_real(c[o].cpu().squeeze(1)), torch.view_as_real(cr[o])) < TOL, o
        assert rel_l2(cq.bwd(c).cpu().squeeze(1), ref.bwd(cr)) < TOL
        cp = cq.fwd_planar(xc)
        for o in range(numocts):
            assert rel_l2(cp[o].permute(0, 2, 3, 1).cpu(), torch.view_as_real(cr[o]).float()) < TOL, o
        assert rel_l2(cq.bwd_planar(cp).cpu(), ref.bwd(cr)) < TOL
    finally:
        lib().babe_set_cqt_band_variant(1)


def test_programmatic_launch_is_bitwise_neutral(CQT):
    """`babe_set_cqt_pdl`: the kernels of a CQT call start behind their predecessor's last wave (programmatic dependent
    launch) and wait (`griddepcontrol.wait`) before they touch the chain's buffers.  Back-to-back calls that re-use the
    plan's workspace (the case an early start could corrupt) give bit-identical results with and without it."""
    from babe_b200._lib import lib
    cq = CQT(7, 64, mode="oct", window=("kaiser", 1), fs=22050, audio_len=184184, device="cuda")
    g = torch.Generator().manual_seed(11)
    xs = [(torch.randn(3, 184184, generator=g) * 0.063).cuda() for _ in range(3)]

    def run():
        outs = []
        for _ in range(2):                       # same workspace, different inputs, no host synchronisation in between
            for x in xs:
                c = cq.fwd(x.unsqueeze(1))
                outs.append(cq.bwd(c))
                outs.append(cq.apply_hpf_DC(x))
                outs.extend(c)
        torch.cuda.synchronize()
        return [o.clone() for o in outs]

    try:
        assert lib().babe_set_cqt_pdl(0) == 0
        ref = run()
        assert lib().babe_set_cqt_pdl(15) == 0
        got = run()
    finally:
        lib().babe_set_cqt_pdl(15)
    assert len(ref) == len(got)
    for a, b in zip(ref, got):
        assert torch.equal(torch.view_as_real(a) if a.is_complex() else a, torch.view_as_real(b) if b.is_complex() else b)


@pytest.mark.parametrize("numocts,binsoct,fs,Ls,B", [CONFIGS[0], CONFIGS[2]])
def test_rows_at_odd_float_offset_are_realigned(CQT, numocts, binsoct, fs, Ls, B):
    """The CQT kernels read their input rows as float2 / float4.  A contiguous view that starts at an odd float (a slice
    of a longer buffer) is copied into aligned storage first -- checked before anything is launched on it -- and then
    gives the aligned call's results bit for bit."""
    cq = CQT(numocts, binsoct, mode="oct", window=("kaiser", 1), fs=fs, audio_len=Ls, device="cuda")
    g = torch.Generator().manual_seed(Ls + 1)
    x = (torch.randn(B, Ls, generator=g) * 0.063).cuda()
    buf = torch.empty(B * Ls + 4, device="cuda")
    view = buf[1:1 + B * Ls].view(B, Ls)
    view.copy_(x)
    assert view.is_contiguous() and view.data_ptr() % 8 == 4
    assert cq._rows(view).data_ptr() % 16 == 0
    assert cq._rows(view.unsqueeze(1)).data_ptr() % 16 == 0
    c, c_ref = cq.fwd(view.unsqueeze(1)), cq.fwd(x.unsqueeze(1))
    assert all(torch.equal(a, b) for a, b in zip(c, c_ref))
    assert torch.equal(cq.bwd(c), cq.bwd(c_ref))
    assert torch.equal(cq.apply_hpf_DC(view), cq.apply_hpf_DC(x))
    assert torch.equal(cq.rfft(view), cq.rfft(x))
    assert torch.equal(view, x)                             # the view itself is left alone
