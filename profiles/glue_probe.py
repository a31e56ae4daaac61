"""The denoiser's residual-layer glue kernels (csrc/net_ops.cu) at the seven octave layer shapes of the
benchmark's CQTDiff+ (N = 8 rows; channels Ns = 64, 96, 96, 128, 128, 256, 256; F = 64 (i + 1) bins;
T = 2048 / 2^i frames), one call at a time with the 126 MB L2 overwritten between calls.  Each
wrapper's own CUDA-event bracket (babe_b200.profiling) gives the kernel time; GB/s is over the
algorithmic bytes the wrapper declares, and the fraction is against MEASURED_PEAKS.json (or bench.py's
fallback).

    python profiles/glue_probe.py OUT.json [--root TREE] [--iters K]

--root imports babe_b200 from another checkout (e.g. the parent commit) so that both builds are
timed by the same script; variants the tree does not have (the statistics-carrying gate_residual,
the g_v-writing gn_film_gelu_bwd) are skipped there.
"""
import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--root", default=os.path.dirname(HERE))
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    root = os.path.abspath(a.root)
    sys.path.insert(0, root)
    import torch
    from babe_b200 import build, denoiser, net_ops, profiling
    build.build()
    sys.path.insert(0, os.path.dirname(HERE))
    from bench import measured_peak
    peak, peak_src = measured_peak()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    card = card[torch.cuda.current_device()] if card else torch.cuda.get_device_name()
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")      # 256 MB > L2

    def measure(fn):
        fn()
        torch.cuda.synchronize()
        profiling.reset()
        profiling.enable(True)
        for _ in range(a.iters):
            flush.add_(1.0)
            fn()
        torch.cuda.synchronize()
        profiling.enable(False)
        return {k: {"ms": round(v["ms_avg"], 4), "GBps": round(v["gbs"], 1), "frac": round(v["gbs"] / peak, 3)}
                for k, v in profiling.summary().items()}

    G, eps = 8, 1e-7
    g = torch.Generator(device="cuda").manual_seed(0)
    rows = []
    for i, C in enumerate([64, 96, 96, 128, 128, 256, 256]):
        shape = (8, C, 64 * (i + 1), 2048 >> i)
        N = shape[0]
        x, v, gh, gy = (torch.randn(shape, device="cuda", generator=g) for _ in range(4))
        gamma = 1 + 0.2 * torch.randn(C, device="cuda", generator=g)
        aff, gate = (0.5 * torch.randn(N, C, device="cuda", generator=g) for _ in range(2))
        rec = net_ops.gn_stats(x, G)
        r = {"shape": list(shape)}
        r.update(measure(lambda: net_ops.gn_stats(x, G)))
        r.update(measure(lambda: net_ops.gn_film_gelu(x, *rec, gamma, aff, G, eps)))
        r.update(measure(lambda: net_ops.gate_residual(x, v, gate)))
        r["gate_residual(gv)"] = measure(lambda: net_ops.gate_residual(None, gy, gate))["gate_residual"]
        r.update(measure(lambda: net_ops.gn_film_gelu_bwd(gh, x, gy, *rec, gamma, aff, G, eps)))
        try:
            r["gate_residual(+stats)"] = measure(lambda: net_ops.gate_residual(x, v, gate, groups=G))["gate_residual"]
            r["gn_film_gelu_bwd(+gv)"] = measure(
                lambda: net_ops.gn_film_gelu_bwd(gh, x, gy, *rec, gamma, aff, G, eps, gate_prev=gate))["gn_film_gelu_bwd"]
        except TypeError:
            pass
        down = net_ops._resample(x, denoiser._CUBIC, 0)
        up = net_ops._resample(x, denoiser._CUBIC, 1)
        for name, inp, mode in (("resample2(down)", x, 0), ("resample2(up)", x, 1),
                                ("resample2(down_adj)", down, 2), ("resample2(up_adj)", up, 3)):
            r[name] = measure(lambda: net_ops._resample(inp, denoiser._CUBIC, mode))["resample2"]
        del down, up
        rows.append(r)
        print(json.dumps(r), flush=True)
        del x, v, gh, gy
    res = {"card": card, "peak_GBps": peak, "peak_source": peak_src, "iters": a.iters,
           "l2": "256 MB buffer rewritten between calls", "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
