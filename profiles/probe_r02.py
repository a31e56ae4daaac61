"""Round-2 probe of the NFFT-4096 operators: parity of the fused (TMA-staged) kernel variants against the
round-1 kernels, then CUDA-event timings with the L2 flushed between iterations.

    python profiles/probe_r02.py [check] [time] [ncu]
"""
import json
import sys
sys.path.insert(0, ".")
import torch
from babe_b200 import ops
from babe_b200._lib import lib

NFFT, SR = 4096, 22050
dev = torch.device("cuda")
f = torch.fft.rfftfreq(NFFT, d=1 / SR).to(dev)
fc = torch.tensor([300.0, 600.0, 1000.0, 3000.0, 6000.0], device=dev)
A = torch.tensor([-10.0, -15.0, -20.0, -30.0, -40.0], device=dev)
PEAK = 6550.4
VARIANTS = (-1, 0)


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def check():
    worst = 0.0
    for B, T in [(1, 4), (1, 100), (2, 2048), (3, 4096), (2, 6144), (2, 20000), (3, 184184), (2, 132300), (5, 131072),
                 (1, 485100), (70, 20480)]:
        g = torch.Generator(device="cpu").manual_seed(B * 1000 + T)
        x = (torch.randn(B, T, generator=g) * 0.063).to(dev)
        y = (torch.randn(B, T, generator=g) * 0.063).to(dev)
        sc = (torch.rand(B, generator=g) + 0.5).to(dev)
        H = torch.rand(NFFT // 2 + 1, generator=g).to(dev)
        res = {}
        for v in VARIANTS:
            lib().babe_set_fused_variant(v)
            ss = torch.zeros(B, dtype=torch.float64, device=dev)
            res[v] = dict(
                fwd=ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A),
                fwdH=ops.apply_filter(x, NFFT, H=H),
                adj=ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, adjoint=True),
                res=ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, sub=y, row_sumsq=ss),
                ss=ss.clone(),
                adjs=ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, adjoint=True, row_scale=sc),
                subonly=ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, sub=y),
            )
        torch.cuda.synchronize()
        for v in VARIANTS[1:]:
            errs = {k: rel(res[v][k], res[-1][k]) for k in res[v]}
            worst = max(worst, max(errs.values()))
            print(f"B={B} T={T} variant {v}: " + " ".join(f"{k}={e:.1e}" for k, e in errs.items()))
    lib().babe_set_fused_variant(0)
    print("worst", worst)
    assert worst < 2e-6, worst


def timeit(fn, iters=15, flush=None):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.fill_(1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def time_all():
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for B, T in [(512, 1 << 17), (64, 184184), (8, 184184)]:
        x = torch.randn(B, T, device=dev) * 0.063
        y = torch.randn(B, T, device=dev) * 0.063
        out = torch.empty_like(x)
        ss = torch.zeros(B, dtype=torch.float64, device=dev)
        sc = torch.ones(B, device=dev)
        for v in VARIANTS:
            lib().babe_set_fused_variant(v)
            cases = {
                "apply_filter": (lambda: ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, out=out), 8 * B * T),
                "apply_filter_adj": (lambda: ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, adjoint=True, out=out), 8 * B * T),
                "residual+sumsq": (lambda: ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, sub=y, row_sumsq=ss, out=out), 12 * B * T),
                "adj+rowscale": (lambda: ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, adjoint=True, row_scale=sc, out=out), 8 * B * T),
                "stft_stats": (lambda: ops.stft_stats(x, y, NFFT), 8 * B * T),
            }
            for name, (fn, nbytes) in cases.items():
                med, best = timeit(fn, flush=flush)
                print(json.dumps({"B": B, "T": T, "variant": v, "op": name, "ms": round(med, 4), "best_ms": round(best, 4),
                                  "GBps": round(nbytes / med / 1e6, 1), "frac": round(nbytes / med / 1e6 / PEAK, 4)}))
    lib().babe_set_fused_variant(0)


def ncu_driver():
    B, T = 512, 1 << 17
    x = torch.randn(B, T, device=dev) * 0.063
    y = torch.randn(B, T, device=dev) * 0.063
    out = torch.empty_like(x)
    for v in VARIANTS[1:]:
        lib().babe_set_fused_variant(v)
        for _ in range(2):
            ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, out=out)
            ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, adjoint=True, out=out)
            ops.stft_stats(x, y, NFFT)
    torch.cuda.synchronize()
    lib().babe_set_fused_variant(0)


if __name__ == "__main__":
    what = sys.argv[1:] or ["check", "time"]
    if "check" in what:
        check()
    if "time" in what:
        time_all()
    if "ncu" in what:
        ncu_driver()
    print("ok")


def time_cqt():
    from cqt_nsgt_pytorch import CQT_nsgt
    for a in sys.argv:
        if a.startswith("pdl="):
            lib().babe_set_cqt_pdl(int(a[4:]))
    SRc, L = 22050, 184184
    cq = CQT_nsgt(7, 64, mode="oct", window=("kaiser", 1), fs=SRc, audio_len=L, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for B, variant in ((64, 2), (64, -1), (8, 2), (8, -1)):
        lib().babe_set_cqt_variant(variant)
        xc = torch.randn(B, L, device=dev) * 0.063
        cs = cq.fwd(xc.unsqueeze(1))
        Xs = cq.rfft(xc)
        cqb = B * (4 * L + 8 * cq.plan.coef_per_row)
        for name, fn, nb in (("cqt_analysis", lambda: cq.fwd(xc.unsqueeze(1)), cqb),
                             ("cqt_synthesis", lambda: cq.bwd(cs), cqb),
                             ("hpf_DC", lambda: cq.apply_hpf_DC(xc), B * 8 * L),
                             ("rfft", lambda: cq.rfft(xc), B * 8 * L),
                             ("irfft", lambda: cq.irfft(Xs), B * 8 * L)):
            med, best = timeit(fn, flush=flush)
            print(json.dumps({"B": B, "cqt_variant": variant, "op": name, "ms": round(med, 4), "best_ms": round(best, 4),
                              "GBps": round(nb / med / 1e6, 1), "frac": round(nb / med / 1e6 / PEAK, 4)}))


if __name__ == "__main__" and "cqt" in sys.argv[1:]:
    time_cqt()


def time_fit():
    from babe_b200 import sampler
    x8 = torch.randn(8, 184184, device=dev) * 0.063
    y8 = ops.apply_filter(x8, NFFT, freqs=f, fc=torch.tensor([1000.0], device=dev), A=torch.tensor([-20.0], device=dev))
    fit = sampler.FilterFit(nfft=NFFT, sample_rate=SR, device=dev)
    abc = fit.stats(x8, y8)
    for K, p0 in ((5, [[280.0, 285, 290, 295, 300], [-15.0, -17, -20, -25, -30]]),
                  (7, [[200.0, 225, 250, 275, 300, 325, 350], [-15.0, -20, -25, -30, -40, -50, -55]])):
        p0 = torch.tensor(p0, device=dev)
        res = {}
        for v in (-1, 0):
            lib().babe_set_fit_variant(v)
            med, best = timeit(lambda: fit(x8, y8, p0.clone(), abc=abc), iters=20)
            p, its = fit(x8, y8, p0.clone(), abc=abc, return_iters=True)
            res[v] = p.clone()
            print(json.dumps({"op": "fit_params", "K": K, "variant": v, "ms": round(med, 4), "best_ms": round(best, 4),
                              "iters": int(its)}))
        print("  max rel diff cluster kernel vs round-1:", rel(res[0], res[-1]))
    lib().babe_set_fit_variant(0)


if __name__ == "__main__" and "cqt" in sys.argv[1:]:
    lib().babe_set_cqt_variant(2)

if __name__ == "__main__" and "fit" in sys.argv[1:]:
    time_fit()


def time_cqt_lengths():
    """The other segment lengths of the BASELINE configs: prime-factor passes (variant 2) against round 1's generic passes (-1)."""
    from cqt_nsgt_pytorch import CQT_nsgt
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for fs, L, no, bo, B in ((22050, 132300, 7, 64, 64), (44100, 485100, 8, 96, 16), (44100, 368368, 8, 96, 16), (22050, 132300, 7, 64, 1)):
        cq = CQT_nsgt(no, bo, mode="oct", window=("kaiser", 1), fs=fs, audio_len=L, device=dev)
        xc = torch.randn(B, L, device=dev) * 0.063
        for variant in (2, -1):
            lib().babe_set_cqt_variant(variant)
            cs = cq.fwd(xc.unsqueeze(1))
            cqb = B * (4 * L + 8 * cq.plan.coef_per_row)
            for name, fn, nb in (("cqt_analysis", lambda: cq.fwd(xc.unsqueeze(1)), cqb), ("cqt_synthesis", lambda: cq.bwd(cs), cqb),
                                 ("hpf_DC", lambda: cq.apply_hpf_DC(xc), B * 8 * L), ("rfft", lambda: cq.rfft(xc), B * 8 * L)):
                med, best = timeit(fn, flush=flush)
                print(json.dumps({"Ls": L, "B": B, "cqt_variant": variant, "op": name, "ms": round(med, 4),
                                  "GBps": round(nb / med / 1e6, 1), "frac": round(nb / med / 1e6 / PEAK, 4)}))
    lib().babe_set_cqt_variant(2)


if __name__ == "__main__" and "cqtlen" in sys.argv[1:]:
    time_cqt_lengths()


def sweep_cqt():
    """CQT operators over the batch size (Ls = 184184, 7 x 64): profiles/r02_cqt_sweep.jsonl."""
    from cqt_nsgt_pytorch import CQT_nsgt
    SRc, L = 22050, 184184
    cq = CQT_nsgt(7, 64, mode="oct", window=("kaiser", 1), fs=SRc, audio_len=L, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for B in (1, 2, 4, 8, 16, 32, 64, 128, 256):
        xc = torch.randn(B, L, device=dev) * 0.063
        cs = cq.fwd(xc.unsqueeze(1))
        cp = cq.fwd_planar(xc)
        cqb = B * (4 * L + 8 * cq.plan.coef_per_row)
        for name, fn, nb in (("cqt_analysis", lambda: cq.fwd(xc.unsqueeze(1)), cqb), ("cqt_synthesis", lambda: cq.bwd(cs), cqb),
                             ("cqt_analysis_planar", lambda: cq.fwd_planar(xc), cqb), ("cqt_synthesis_planar", lambda: cq.bwd_planar(cp), cqb),
                             ("hpf_DC", lambda: cq.apply_hpf_DC(xc), B * 8 * L)):
            med, best = timeit(fn, flush=flush)
            print(json.dumps({"B": B, "op": name, "ms": round(med, 4), "best_ms": round(best, 4), "GBps": round(nb / med / 1e6, 1),
                              "frac": round(nb / med / 1e6 / PEAK, 4)}))
        del xc, cs, cp


if __name__ == "__main__" and "cqtsweep" in sys.argv[1:]:
    sweep_cqt()
