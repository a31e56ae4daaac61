"""Keyed per-row noise (``k_row_noise``, ``BlindSamplerFused.row_seeds``) on one GPU:

  (a) CUDA-event times of ops.row_noise (one launch), raw noise and the fused move x + scale * eps, at
      8 x 184184 (5.9 MB written: stays in the 126 MB L2 across repetitions, as inside a sampler step) and
      512 x 2^17 (268 MB written, 537 MB moved by the fused form: larger than L2); 20 launches per window,
      best of 3 windows; GB/s against the algorithmic bytes (4 B written per sample, plus 4 B read for the fused
      form);
  (b) ms per sampler step on the benchmark workload (8 x 184184, random-init CQTDiff+, whole-step CUDA graph),
      the reference's host noise stream against row_seeds, alternated twice.

    python profiles/row_noise_probe.py OUT.json [--steps K]
"""
import json
import os
import subprocess
import sys

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
    from babe_b200 import ops, segments
    from babe_b200.sampler import BlindSamplerFused
    out = res["a_kernel"] = []
    for B, T in ((8, 184184), (512, 2 ** 17)):
        seeds = BlindSamplerFused._seed_tensor([segments.row_seed(0, k) for k in range(B)]).cuda()
        draw = torch.full((1,), 9, dtype=torch.int32, device="cuda")
        x = torch.zeros(B, T, device="cuda")
        buf = torch.empty(B, T, device="cuda")
        scale = torch.full((1,), 0.3, device="cuda")
        forms = {"raw": (lambda: ops.row_noise(seeds, (B, T), draw, out=buf), 4),
                 "fused_move": (lambda: ops.row_noise(seeds, x, draw, scale=scale, out=buf), 8)}
        best = {k: [] for k in forms}
        for _ in range(3):                                   # alternate the forms, keep the best of three windows
            for name, (fn, _) in forms.items():
                best[name].append(event_ms(fn))
        for name, (_, bps) in forms.items():
            ms = min(best[name])
            out.append({"form": name, "B": B, "T": T, "ms": ms, "windows_ms": best[name],
                        "GBps": bps * B * T / (ms * 1e-3) / 1e9, "bytes": bps * B * T})
            print(json.dumps(out[-1]), flush=True)


def sampler_steps(res, steps):
    import bench
    from babe_b200 import segments
    cfg = bench.CONFIGS[2]
    out = res["b_sampler_step"] = {}
    torch.backends.cudnn.benchmark = True
    args, net, smp, y, _ = bench.build_world(torch.device("cuda", 0), cfg, cfg["chains"], 0)
    smp.step_graph = True
    seeds = [segments.row_seed(0, k) for k in range(y.shape[0])]
    for rep in range(2):                                     # alternate the modes twice
        for keyed in (False, True):
            smp.row_seeds = seeds if keyed else None
            evs = []

            def hook(i, x, p):
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                evs.append(e)
            torch.manual_seed(0)
            smp.predict_blind_bwe(y, max_steps=steps + 2, step_hook=hook)
            torch.cuda.synchronize()
            ms = evs[1].elapsed_time(evs[-1]) / (len(evs) - 2)
            key = "row_seeds" if keyed else "host_stream"
            out.setdefault(key + "_ms_per_step", []).append(ms)
            out["graphed"] = bool(smp._step_graphs)
            print(key, ms, flush=True)
    out.update({"B": int(y.shape[0]), "T": int(y.shape[1]), "steps_timed": steps})


def main():
    path = sys.argv[1]
    steps = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 6
    from babe_b200 import build
    build.build()
    res = {"card": card(), "gpus": torch.cuda.device_count(), "torch": torch.__version__}
    print(res, flush=True)
    kernels(res)
    sampler_steps(res, steps)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
