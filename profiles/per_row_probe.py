"""Per-row filter mode (``filter_per_row``) against the shared filter, on one GPU:

  (a) CUDA-event times of the operator calls (every launch of one ops.* call) per-row vs shared: fit statistics,
      filter forward with the residual epilogue, filter adjoint with the row scale, at B x 184184, B = 8 and 64
      (5.9 / 47 MB per signal: both working sets stay in the 126 MB L2 across the timed repetitions, as they do
      inside a sampler step); fit-loop latency for B = 1, 8, 37, 64
      rows (100 iterations unless a row stops early; the iteration counts are reported);
      plus whether the per-row results equal the shared results of each row alone bit for bit;
  (b) ms per sampler step, per-row vs shared, on the benchmark workload (8 x 184184, random-init CQTDiff+,
      whole-step CUDA graph);
  (c) wall time of segments.restore_recording on the 60 s recording of bench config 5 (8 segments) on one GPU,
      the sequential loop (batched=False) vs one per-row call (batched=True).

    python profiles/per_row_probe.py OUT.json [--steps K] [--skip-restore]
"""
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def event_ms(fn, iters=20, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernels(res):
    from babe_b200 import ops, sampler
    sr, nfft, T = 22050, 4096, 184184
    f = torch.fft.rfftfreq(nfft, d=1 / sr).cuda()
    fit = sampler.FilterFit(nfft=nfft, sample_rate=sr, max_iter=100, device="cuda")
    p_init = torch.tensor([[280.0, 285, 290, 295, 300], [-15.0, -17, -20, -25, -30]]).cuda()
    out = res["a_operators"] = []
    for B in (8, 64):
        g = torch.Generator(device="cuda").manual_seed(B)
        x = torch.randn(B, T, device="cuda", generator=g) * 0.063
        fc1, A1 = torch.tensor([1000.0, 1500, 2000, 2500, 3000]).cuda(), torch.tensor([-20.0, -25, -30, -35, -40]).cuda()
        fcB = (fc1[None] * torch.linspace(0.5, 2.0, B, device="cuda")[:, None]).contiguous()
        AB = A1[None].expand(B, -1).contiguous()
        y = ops.apply_filter_rows(x, nfft, f, fcB, AB)
        ss = torch.zeros(B, dtype=torch.float64, device="cuda")
        scale = torch.ones(B, device="cuda")
        pairs = {
            "stft_stats": (lambda: ops.stft_stats(x, y, nfft), lambda: ops.stft_stats_rows(x, y, nfft)),
            "filter_fwd_residual": (lambda: ops.apply_filter(x, nfft, freqs=f, fc=fc1, A=A1, sub=y, row_sumsq=ss),
                                    lambda: ops.apply_filter_rows(x, nfft, f, fcB, AB, sub=y, row_sumsq=ss)),
            "filter_adj_scaled": (lambda: ops.apply_filter(x, nfft, freqs=f, fc=fc1, A=A1, adjoint=True, row_scale=scale),
                                  lambda: ops.apply_filter_rows(x, nfft, f, fcB, AB, adjoint=True, row_scale=scale)),
        }
        for name, (sh, pr) in pairs.items():
            t_sh, t_pr = [], []
            for _ in range(3):                               # alternate the two, keep the best of three windows
                t_sh.append(event_ms(sh))
                t_pr.append(event_ms(pr))
            out.append({"op": name, "B": B, "T": T, "shared_ms": min(t_sh), "per_row_ms": min(t_pr),
                        "ratio": min(t_pr) / min(t_sh)})
            print(json.dumps(out[-1]), flush=True)
        if B == 8:                                           # bit-for-bit comparison against one row at a time
            abc = ops.stft_stats_rows(x, y, nfft)
            fw = ops.apply_filter_rows(x, nfft, f, fcB, AB)
            ad = ops.apply_filter_rows(x, nfft, f, fcB, AB, adjoint=True)
            eq = {"stft_stats": True, "filter_fwd": True, "filter_adj": True, "fit": True}
            maxrel = {"stft_stats": 0.0, "filter_fwd": 0.0, "filter_adj": 0.0}
            pr = ops.fit_params_rows(abc, fit.w, fit.freqs, p_init.expand(B, -1, -1).contiguous().clone(), fit.cfg)
            for b in range(B):
                r_abc = ops.stft_stats(x[b:b + 1], y[b:b + 1], nfft)
                r_fw = ops.apply_filter(x[b:b + 1], nfft, freqs=f, fc=fcB[b], A=AB[b])
                r_ad = ops.apply_filter(x[b:b + 1], nfft, freqs=f, fc=fcB[b], A=AB[b], adjoint=True)
                for k, u, v in (("stft_stats", abc[b], r_abc), ("filter_fwd", fw[b:b + 1], r_fw),
                                ("filter_adj", ad[b:b + 1], r_ad)):
                    eq[k] &= bool(torch.equal(u, v))
                    maxrel[k] = max(maxrel[k], float((u.double() - v.double()).norm() / v.double().norm()))
                eq["fit"] &= bool(torch.equal(pr[b], ops.fit_params(abc[b], fit.w, fit.freqs, p_init.clone(), fit.cfg)))
            res["bitwise_vs_single_rows_B8"] = {"equal": eq, "max_rel_l2": maxrel}
            print(json.dumps(res["bitwise_vs_single_rows_B8"]), flush=True)
    fits = res["a_fit_latency"] = []
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(64, T, device="cuda", generator=g) * 0.063
    fcB = (torch.tensor([1000.0, 1500, 2000, 2500, 3000]).cuda()[None]
           * torch.linspace(0.5, 2.0, 64, device="cuda")[:, None]).contiguous()
    AB = torch.tensor([-20.0, -25, -30, -35, -40]).cuda()[None].expand(64, -1).contiguous()
    y = ops.apply_filter_rows(x, nfft, f, fcB, AB)
    abc64 = ops.stft_stats_rows(x, y, nfft)
    p64 = p_init.expand(64, -1, -1).contiguous()
    for B in (1, 8, 37, 64):
        abc, p0 = abc64[:B].contiguous(), p64[:B]
        _, its = ops.fit_params_rows(abc, fit.w, fit.freqs, p0.clone(), fit.cfg, return_iters=True)
        t_rows = min(event_ms(lambda: ops.fit_params_rows(abc, fit.w, fit.freqs, p0.clone(), fit.cfg), iters=10)
                     for _ in range(3))
        t_one = min(event_ms(lambda: ops.fit_params(abc[0], fit.w, fit.freqs, p_init.clone(), fit.cfg), iters=10)
                    for _ in range(3))
        fits.append({"B": B, "per_row_ms": t_rows, "shared_B1_fit_ms": t_one, "iters": its.cpu().tolist()})
        print(json.dumps(fits[-1]), flush=True)


def sampler_steps(res, steps):
    import bench
    from babe_b200 import sampler as smod
    cfg = bench.CONFIGS[2]
    out = res["b_sampler_step"] = {}
    torch.backends.cudnn.benchmark = True
    args, net, smp, y, _ = bench.build_world(torch.device("cuda", 0), cfg, cfg["chains"], 0)
    smp.step_graph = True
    for rep in range(2):                                     # alternate the modes twice
        for per_row in (False, True):
            smp.filter_per_row = per_row
            evs = []

            def hook(i, x, p):
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                evs.append(e)
            torch.manual_seed(0)
            smp.predict_blind_bwe(y, max_steps=steps + 2, step_hook=hook)
            torch.cuda.synchronize()
            ms = evs[1].elapsed_time(evs[-1]) / (len(evs) - 2)
            key = "per_row" if per_row else "shared"
            out.setdefault(key + "_ms_per_step", []).append(ms)
            out["graphed"] = bool(smp._step_graphs)
            print(key, ms, flush=True)
    out.update({"B": int(y.shape[0]), "T": int(y.shape[1]), "steps_timed": steps})


def restore(res):
    import bench
    from babe_b200 import blind_bwe_utils as bu, segments
    cfg = bench.CONFIGS[5]
    torch.backends.cudnn.benchmark = True
    args, net, smp, _, _ = bench.build_world(torch.device("cuda", 0), cfg, cfg["chains"], 0)
    smp.step_graph = True
    f = torch.fft.rfftfreq(4096, d=1 / cfg["sr"]).cuda()
    rec = bench.piano_like(1, cfg["recording"], cfg["sr"], 1234 + 5).cuda()
    deg = bu.apply_filter(rec, bu.design_filter([1000.0], [-20.0], f), 4096)
    out = res["c_restore_recording"] = {"L": int(deg.shape[-1]), "seg_len": cfg["T"],
                                        "n_segments": int(segments.split(deg, cfg["T"])[0].shape[0]),
                                        "steps": int(args.tester.T)}
    smp.filter_per_row = False
    torch.manual_seed(0)
    smp.predict_blind_bwe(deg[:, :cfg["T"]].contiguous(), max_steps=1)          # captures the B = 1 step graphs
    for batched in (False, True, False, True):
        torch.manual_seed(0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        final, fd = segments.restore_recording(smp, deg, cfg["T"], batched=batched)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out.setdefault("batched_s" if batched else "sequential_s", []).append(dt)
        out["distinct_filters_" + ("batched" if batched else "sequential")] = len(
            {tuple(v.flatten().tolist()) for _, v in fd})
        print("batched" if batched else "sequential", dt, flush=True)


def main():
    path = sys.argv[1]
    steps = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 6
    from babe_b200 import build
    build.build()
    res = {"card": card(), "torch": torch.__version__}
    print(res, flush=True)
    kernels(res)
    sampler_steps(res, steps)
    if "--skip-restore" not in sys.argv:
        restore(res)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
