"""Batched autoregressive restoration (``segments.restore_recordings_ar``) and the known-prefix masked filter kernels,
on one GPU:

  (a) CUDA-event times of the guidance operator calls with and without the known-prefix mask (every launch of one
      ops.apply_filter_rows call): residual forward (sub + row sums of squares) and scaled adjoint at B x 184184,
      B = 8 and 64, 5512 known samples per row (0.25 s at 22.05 kHz, what every autoregressive window has); 200
      launches per window after warm-up, the two variants alternated three times, the best window kept.  Both working
      sets stay in the 126 MB L2 across the repetitions, as they do inside a sampler step.  GB/s counts the
      algorithmic bytes: x, sub and the output (12 B per sample) for the residual, x and the output (8 B) for the
      adjoint, plus the known prefix read once more by the masked epilogue;
  (b) AR restoration of 8 recordings of 9..30 s (2 to 4 windows of 184184 samples each) with the random-init CQTDiff+
      of ``make_args`` defaults and given filters, ``--steps`` sampler steps per window: 8 sequential
      ``restore_recording_ar`` calls against ``restore_recordings_ar`` on groups of N = 1, 4 and 8 recordings, as
      window-steps per second (each configuration run twice, both runs reported), and the restorations of the
      sequential and the N = 8 runs compared at the same seeds.

    python profiles/ar_rows_probe.py OUT.json [--steps K]
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


def event_ms(fn, iters=200, warmup=10):
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
    from babe_b200 import ops
    sr, nfft, T, kn = 22050, 4096, 184184, 5512
    f = torch.fft.rfftfreq(nfft, d=1 / sr).cuda()
    out = res["a_operators"] = []
    for B in (8, 64):
        g = torch.Generator(device="cuda").manual_seed(B)
        x = torch.randn(B, T, device="cuda", generator=g) * 0.063
        fcB = (torch.tensor([1000.0, 1500, 2000, 2500, 3000]).cuda()[None]
               * torch.linspace(0.5, 2.0, B, device="cuda")[:, None]).contiguous()
        AB = torch.tensor([-20.0, -25, -30, -35, -40]).cuda()[None].expand(B, -1).contiguous()
        y = ops.apply_filter_rows(x, nfft, f, fcB, AB)
        ss = torch.zeros(B, dtype=torch.float64, device="cuda")
        scale = torch.ones(B, device="cuda")
        known = torch.full((B,), kn, dtype=torch.int32, device="cuda")
        pairs = {
            "filter_fwd_residual": (12, lambda k: ops.apply_filter_rows(x, nfft, f, fcB, AB, sub=y, row_sumsq=ss, known=k)),
            "filter_adj_scaled": (8, lambda k: ops.apply_filter_rows(x, nfft, f, fcB, AB, adjoint=True, row_scale=scale,
                                                                     known=k)),
        }
        for name, (bps, call) in pairs.items():
            t_un, t_mk = [], []
            for _ in range(3):
                t_un.append(event_ms(lambda: call(None)))
                t_mk.append(event_ms(lambda: call(known)))
            b_un = bps * B * T
            b_mk = b_un + 4 * B * kn
            out.append({"op": name, "B": B, "T": T, "known": kn, "unmasked_ms": min(t_un), "masked_ms": min(t_mk),
                        "unmasked_GBps": b_un / min(t_un) / 1e6, "masked_GBps": b_mk / min(t_mk) / 1e6,
                        "masked_over_unmasked": min(t_mk) / min(t_un), "windows_ms": {"unmasked": t_un, "masked": t_mk}})
            print(json.dumps(out[-1]), flush=True)


def restoration(res, steps):
    import bench
    from babe_b200 import blind_bwe_utils as bu, denoiser, edm, sampler, segments
    sr, seg_len = 22050, 184184
    torch.backends.cudnn.benchmark = True
    args = sampler.make_args(T=steps)
    torch.manual_seed(0)
    net = denoiser.CQTDiffPlus(args, torch.device("cuda", 0)).cuda()
    for p in net.parameters():
        p.requires_grad_(False)
    smp = sampler.BlindSamplerFused(net, edm.EDM(args), args, rid=False)
    f = torch.fft.rfftfreq(4096, d=1 / sr).cuda()
    H = bu.design_filter([1000.0], [-20.0], f)
    secs = [9, 12, 15, 18, 21, 24, 27, 30]
    recs = [bu.apply_filter(bench.piano_like(1, s * sr, sr, 500 + i).cuda(), H, 4096) for i, s in enumerate(secs)]
    base = torch.tensor([[280.0, 285, 290, 295, 300], [-15.0, -17, -20, -25, -30]])
    filters = [(base * torch.tensor([[1.0 + 0.5 * i], [1.0]])).cuda() for i in range(8)]
    seeds = [1000 + i for i in range(8)]
    n_windows = [len(segments.ar_windows(r.shape[-1], seg_len, int(0.25 * sr), 200, 0)) for r in recs]
    out = res["b_restoration"] = {"recordings_s": secs, "windows": n_windows, "steps": steps, "seg_len": seg_len,
                                  "window_steps": sum(n_windows) * steps}

    def sequential():
        return [segments.restore_recording_ar(smp, recs[i], seg_len, sr, estimated_filter=filters[i], seed=seeds[i])[0]
                for i in range(8)]

    def grouped(n):
        outs = []
        for lo in range(0, 8, n):
            outs += [o for o, _ in segments.restore_recordings_ar(smp, recs[lo:lo + n], seg_len, sr, seeds=seeds[lo:lo + n],
                                                                  estimated_filters=filters[lo:lo + n])]
        return outs

    results = {}
    for rep in range(2):
        for key, fn in (("sequential", sequential), ("N1", lambda: grouped(1)), ("N4", lambda: grouped(4)),
                        ("N8", lambda: grouped(8))):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            results[key] = fn()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            out.setdefault(key + "_s", []).append(dt)
            out.setdefault(key + "_window_steps_per_s", []).append(out["window_steps"] / dt)
            print(key, rep, dt, flush=True)
    rel = []
    for a, b in zip(results["sequential"], results["N8"]):
        rel.append(float((a.double() - b.double()).norm() / b.double().norm()))
    out["rel_l2_sequential_vs_N8"] = rel
    print(json.dumps(out), flush=True)


def main():
    path = sys.argv[1]
    steps = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 4
    from babe_b200 import build
    build.build()
    res = {"card": card(), "torch": torch.__version__}
    print(res, flush=True)
    kernels(res)
    restoration(res, steps)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
