#!/usr/bin/env python
"""Benchmark of the blind-BWE sampler hot path (BASELINE.json metric:
"blind-BWE sampler steps/s at 1/2/4/8 B200; operator % of HBM roofline").

    python bench.py --gpus N --steps K --warmup W           # this repo's CUDA path (contract line)
    python bench.py --impl reference --steps K --warmup W   # the reference algorithm on the host cores
    python bench.py --config {1,2,3,5} [--joint]            # the other BASELINE configs (2 = default)
    python bench.py --mode operator [--grid full]           # config 4: operator sweep (table, JSON lines)
    python bench.py --steps K --warmup W --dump-outputs DIR # also write the timed run's outputs as DIR/*.npy

Workload of the contract line (config.workload): BASELINE configs[1] per-GPU slice -- 8 chains of
T=184184 samples at 22.05 kHz per GPU (64 chains over 8 GPUs), random-init CQTDiff+ (44.5 M parameters,
torch.manual_seed(0)), 35-step EDM schedule, 2nd-order sampler, filter fit max_iter=100, NFFT=4096, K=5
breakpoints, synthetic piano-like audio low-passed at 1 kHz / -20 dB/oct.  A "step" is one iteration of
the sampling loop (testing/blind_bwe_sampler.py:685, incl. the Heun correction): 2 x {denoiser fwd+bwd
through both CQTs, hpf, filter fit, reconstruction guidance}.  value = chains * steps / seconds, whole job.

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

NFFT = 4096
# BASELINE.json configs (SURVEY 8d).  "chains" = rows per GPU.
CONFIGS = {
    1: dict(tag="configs[0]", sr=22050, T=132300, chains=1, bins=64, steps_T=35, xi=0.2, start_sigma=0.2, schurn=20,
            fc=(280, 285, 290, 295, 300), A=(-15, -17, -20, -25, -30), only_negative_A=True,
            what="one 6 s segment @ 22.05 kHz, 1 chain"),
    2: dict(tag="configs[1] per-GPU slice", sr=22050, T=184184, chains=8, bins=64, steps_T=35, xi=0.2,
            start_sigma=0.2, schurn=20, fc=(280, 285, 290, 295, 300), A=(-15, -17, -20, -25, -30),
            only_negative_A=True, what="8 chains/GPU (64 over 8 GPUs) @ 22.05 kHz"),
    3: dict(tag="configs[2]", sr=44100, T=485100, chains=2, bins=96, steps_T=50, xi=0.3, start_sigma=0.5, schurn=30,
            fc=(300, 350, 400, 450), A=(-15, -20, -35, -55), only_negative_A=False,
            what="44.1 kHz, 11 s segments, 96 bins/octave, sampler values of conf/tester/blind_bwe_44k.yaml"),
    5: dict(tag="configs[4]", sr=22050, T=184184, chains=8, bins=64, steps_T=35, xi=0.2, start_sigma=0.2, schurn=20,
            fc=(280, 285, 290, 295, 300), A=(-15, -17, -20, -25, -30), only_negative_A=True, recording=1323000,
            what="60 s recording as 8 overlapped segments sharded over the ranks, ONE jointly estimated filter "
                 "(fit statistics and the guidance norm all-reduced over NCCL), gather + hann cross-fade"),
}


def piano_like(B, T, sr, seed):
    """SURVEY 8(d) synthetic input: decaying harmonic notes, std 0.063 (vectorised)."""
    g = torch.Generator().manual_seed(seed)
    n = torch.arange(T, dtype=torch.float32)
    out = torch.zeros(B, T)
    for b in range(B):
        k = torch.randint(20, 76, (24,), generator=g)
        f0 = 27.5 * 2.0 ** (k.float() / 12)
        n0 = torch.randint(0, T, (24,), generator=g).float()
        for p in range(24):
            tt = ((n - n0[p]).clamp(min=0)) / sr
            gate = (n >= n0[p]).float()
            for h in range(1, 13):
                if h * float(f0[p]) >= sr / 2:
                    break
                out[b] += gate * h ** -1.2 * torch.exp(-tt * h / 1.5) * torch.sin(2 * math.pi * h * float(f0[p]) * tt)
    return out / out.std(dim=1, keepdim=True) * 0.063


class ClockSampler:
    """nvidia-smi clocks and throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                    "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in o.strip().split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def fp32_peak_tflops(sm_mhz):
    """SIMT fp32 peak: 148 SMs x 128 lanes x 2 flop (FMA) x clock."""
    return 148 * 128 * 2 * (sm_mhz or 1965.0) * 1e6 / 1e12


# ---------------------------------------------------------------------------
# nominal flop counts of the operators (SURVEY 8d: 5 N log2 N per complex FFT)
# ---------------------------------------------------------------------------
def _fft_flops(n):
    return 5.0 * n * math.log2(n)


def op_flops(name, B, T, cq=None):
    pairs = B * (T / NFFT)                                   # frame pairs of the fused filter: 2 transforms each
    if name.startswith("apply_filter"):
        return pairs * (2 * _fft_flops(NFFT) + 10 * NFFT)
    if name == "stft_stats":
        return B * (T / (NFFT // 2)) * (_fft_flops(NFFT) + 14 * NFFT)
    if cq is not None and name.startswith(("cqt_analysis", "cqt_synthesis")):
        c = cq.plan.c
        bands = sum(c.binsoct * _fft_flops(c.M[o]) for o in range(c.numocts))
        return B * (0.5 * _fft_flops(c.Ls) + bands + 6 * cq.plan.coef_per_row)
    if cq is not None and name.startswith(("spectral_filter", "hpf")):
        return B * (_fft_flops(cq.plan.c.Ls) + 6 * cq.plan.c.Ls)
    return 0.0


SIGNAL_OPS = ("apply_filter", "apply_filter_adj", "stft_stats", "cqt_analysis", "cqt_synthesis", "spectral_filter")


# ---------------------------------------------------------------------------
def build_world(device, cfg, chains, seed, max_iter=100):
    from babe_b200 import blind_bwe_utils as bu, denoiser, edm, sampler
    args = sampler.make_args(sample_rate=cfg["sr"], audio_len=cfg["T"], NFFT=NFFT, max_iter=max_iter, T=cfg["steps_T"],
                             xi=cfg["xi"], start_sigma=cfg["start_sigma"], Schurn=cfg["schurn"],
                             fc_init=cfg["fc"], A_init=cfg["A"], bins_per_oct=cfg["bins"])
    args.tester.blind_bwe.optimization.only_negative_A = cfg["only_negative_A"]
    torch.manual_seed(0)
    net = denoiser.CQTDiffPlus(args, device).to(device)
    for p in net.parameters():
        p.requires_grad_(False)
    f = torch.fft.rfftfreq(NFFT, d=1 / cfg["sr"]).to(device)
    H = bu.design_filter([1000.0], [-20.0], f)                                  # blind_bwe.yaml:135-137
    if cfg.get("recording"):
        from babe_b200 import distributed as bd, segments
        rank, world = (torch.distributed.get_rank(), torch.distributed.get_world_size()) \
            if torch.distributed.is_initialized() else (0, 1)
        rec = piano_like(1, cfg["recording"], cfg["sr"], 1234 + 5)
        segs, spans = segments.split(rec, cfg["T"])
        lo, hi = bd.shard_rows(segs.shape[0], rank, world)
        x = segs[lo:hi].to(device)
        extra = {"spans": spans, "L": cfg["recording"], "n_segments": segs.shape[0]}
    else:
        x = piano_like(chains, cfg["T"], cfg["sr"], 1234 + seed).to(device)
        extra = {}
    y = bu.apply_filter(x, H, NFFT)
    smp = sampler.BlindSamplerFused(net, edm.EDM(args), args, rid=False)
    return args, net, smp, y, extra


def run_ours(a):
    from babe_b200 import build, distributed as bd, profiling
    build.build()
    rank, local, world = bd.init_from_env()
    if world != a.gpus and rank == 0 and a.gpus != 1:
        print(f"warning: --gpus {a.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    torch.backends.cudnn.benchmark = not a.no_autotune
    from babe_b200 import net_ops
    net_ops.AUTOTUNE_CONV = not a.no_autotune
    cfg = CONFIGS[a.config]
    chains = a.chains or cfg["chains"]
    joint = a.joint or bool(cfg.get("recording"))
    args, net, smp, y, extra = build_world(device, cfg, chains, seed=rank)
    chains = y.shape[0]
    smp.joint = joint
    T = cfg["T"]
    K, W = a.steps, a.warmup
    if W + K > args.tester.T:
        raise SystemExit(f"--steps {K} + --warmup {W} exceed the {args.tester.T}-step sampler schedule")
    n_par = len(cfg["fc"])

    def timed_run(mode):
        """mode 'device': inputs resident, device noise, no logging.
        mode 'e2e': the public, reference-compatible call -- y starts in pinned host memory, every step's
        noise is drawn by the host generator into pinned memory and copied (the reference's
        torch.randn(shape).to(device), testing/blind_bwe_sampler.py:513), the step's denoised estimate and
        filter go back to the host (the tester's rid=True logging), and the timed region ends after the
        NCCL gather of the final outputs and filter estimates."""
        ev = {}
        if mode == "device":
            smp.device_noise, smp.noise_fn = True, None
            smp.generator = torch.Generator(device=device).manual_seed(100 + rank)
            y_in = y
            h2d = d2h = 0
        else:
            smp.device_noise, smp.noise_fn = False, None
            torch.manual_seed(100 + rank)
            y_host = y.cpu().pin_memory()
            out_den = torch.empty((chains, T), dtype=torch.float32).pin_memory()
            out_par = torch.empty((2, n_par), dtype=torch.float32).pin_memory()
            h2d = y.numel() * 4            # per step: that step's noise draw
            d2h = y.numel() * 4 + out_par.numel() * 4

        def hook(i, x, p):
            if mode == "e2e":
                out_den.copy_(x, non_blocking=True)     # rid=True logging of the reference tester
                out_par.copy_(p, non_blocking=True)
            if i == W - 1:
                torch.cuda.synchronize()
                bd.barrier()
                torch.cuda.synchronize()
                profiling.reset()
                ev["clk"] = ClockSampler(local).__enter__() if rank == 0 else None
                ev["t0"] = time.perf_counter()
                ev["s"] = torch.cuda.Event(enable_timing=True)
                ev["s"].record()
                # process-wide start/end range (push/pop ranges are per thread and would miss the kernels
                # launched by autograd's backward thread):  ncu --nvtx --nvtx-include "timed_device"
                ev["nvtx"] = torch.cuda.nvtx.range_start("timed_" + mode)
            if i == W + K - 1 and mode == "device":
                finish()

        def finish():
            ev["e"] = torch.cuda.Event(enable_timing=True)
            ev["e"].record()
            torch.cuda.nvtx.range_end(ev["nvtx"])
            ev["host"] = time.perf_counter() - ev["t0"]     # host time to enqueue the K steps
            torch.cuda.synchronize()
            ev["wall"] = time.perf_counter() - ev["t0"]
            ev["launches"] = profiling.launches()
            ev["ops"] = profiling.summary()
            if ev["clk"] is not None:
                ev["clk"].__exit__()
            bd.barrier()

        if mode == "e2e":
            torch.cuda.synchronize()
            y_in = y_host.to(device, non_blocking=True)
        x, p = smp.predict_blind_bwe(y_in, rid=False, max_steps=W + K, step_hook=hook)
        if mode == "e2e":
            # the only collectives of independent mode: final outputs and filter estimates of all ranks
            xg = bd.gather_rows(x)
            pg = bd.gather_params(p)
            if extra:
                from babe_b200 import segments
                xg = segments.merge(xg, extra["spans"], extra["L"])
            ev["gathered"] = [tuple(xg.shape), tuple(pg.shape)]
            finish()
        ev["out"] = (x.clone(), p.clone())         # outside the timed region; later passes must not overwrite it
        ms = ev["s"].elapsed_time(ev["e"])
        ev["ms"] = bd.max_over_ranks(ms, device)
        return ev, h2d, d2h

    # `value`: device-resident run without per-call CUDA events; a second, identical pass with the
    # events on supplies the per-kernel table of `roofline` (the events cost host time only)
    use_graph = not (a.no_cuda_graph or a.single_pass)      # ncu launch lists profile the eager launches
    # whole-step CUDA graph (SURVEY 8f-1) when it captures; else the denoiser-only graphs; else eager
    smp.step_graph, smp.cuda_graph = use_graph and not joint and not a.no_step_graph, False
    dev_run, _, _ = timed_run("device")
    graphed = "step" if smp._step_graphs else False
    if use_graph and not graphed:
        smp.step_graph, smp.cuda_graph = False, True
        dev_run, _, _ = timed_run("device")
        graphed = "denoiser" if smp._graphed is not None else False
    graph_mode = (smp.step_graph, smp.cuda_graph)
    smp.step_graph, smp.cuda_graph = False, False      # the per-kernel pass needs the wrappers to run (eager)
    if a.single_pass:                    # ncu launch lists: exactly K timed steps, no second pass
        prof_run = dev_run
    else:
        profiling.enable(True)
        prof_run, _, _ = timed_run("device")
        profiling.enable(False)
    smp.step_graph, smp.cuda_graph = graph_mode
    if a.skip_e2e:                       # profiling runs (ncu) only need the device-resident leg
        e2e_run, h2d, d2h = dev_run, 0, 0
    else:
        e2e_run, h2d, d2h = timed_run("e2e")

    ct = torch.tensor([float(chains)], dtype=torch.float64, device=device)
    bd.sum_over_ranks_(ct)
    total_chains = int(ct.item())
    dumped = dump_outputs(a.dump_outputs, *dev_run["out"], rank) if a.dump_outputs else None
    value = total_chains * K / (dev_run["ms"] / 1e3)
    e2e_value = total_chains * K / (e2e_run["ms"] / 1e3)

    if rank != 0:
        return
    peak, peak_src = measured_peak()
    clocks = dev_run["clk"].summary() if dev_run.get("clk") else None
    fp32_peak = fp32_peak_tflops(clocks["sm_mhz"] if clocks else None)
    ops = prof_run["ops"]
    cq = net.CQTransform

    def op_entry(k, v):
        fl = op_flops(k, chains, T, cq)
        tf = fl / (v["ms_avg"] / 1e3) / 1e12 if v["ms_avg"] > 0 else 0.0
        return {"ms_avg": round(v["ms_avg"], 4), "GBps": round(v["gbs"], 1), "frac_hbm": round(v["gbs"] / peak, 4),
                "calls": v["calls"], "share": round(v["ms_total"] / prof_run["ms"], 5),
                "algorithmic_bytes": int(v["bytes_avg"]), "gflop": round(fl / 1e9, 3),
                "tflops": round(tf, 3), "frac_fp32_peak": round(tf / fp32_peak, 4) if fl else None}

    # the roofline object names the dominant operator of the SIGNAL path (SURVEY 8a/8d rows: CQT directions,
    # hpf, fused STFT filter and its adjoint, fit statistics).  The fit loop is a latency-bound single-CTA
    # kernel with ~50 KB of traffic (a latency metric, SURVEY 8d); the layer glue of the denoiser body
    # (gn_*, gate_*, resample2: SURVEY 8f-2) is listed under "denoiser_glue", never as the headline.
    sig = {k: v for k, v in ops.items() if k in SIGNAL_OPS}
    dom = max(sig, key=lambda k: sig[k]["ms_total"]) if sig else None
    tj = {}
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    roof = None
    if dom:
        o = ops[dom]
        traffic = None
        if dom in tj and tj[dom].get("B") == chains and tj[dom].get("T", T) == T:
            traffic = tj[dom]["bytes"]
        e = op_entry(dom, o)
        roof = {"bound": "hbm", "kernel": dom, "achieved": round(o["gbs"], 1), "peak": peak, "unit": "GB/s",
                "frac": round(o["gbs"] / peak, 4), "frac_of_nominal_8TBps": round(o["gbs"] / 8000.0, 4),
                "traffic": traffic, "algorithmic_bytes": int(o["bytes_avg"]), "peak_source": peak_src,
                "avg_ms": round(o["ms_avg"], 4), "calls": o["calls"],
                "share_of_step": round(o["ms_total"] / prof_run["ms"], 5),
                "gflop_per_call": e["gflop"], "tflops": e["tflops"], "frac_fp32_peak": e["frac_fp32_peak"],
                "fp32_peak_tflops": round(fp32_peak, 1),
                "note": f"in-sampler call at B={chains} rows: launch/latency-bound at this batch; the same operators "
                        "at a batch that fills the GPU are in operator_roofline",
                "signal_path": {k: op_entry(k, v) for k, v in sig.items()},
                "fit_params": ({"ms_avg": round(ops["fit_params"]["ms_avg"], 4), "calls": ops["fit_params"]["calls"],
                                "share": round(ops["fit_params"]["ms_total"] / prof_run["ms"], 5)}
                               if "fit_params" in ops else None),
                "signal_path_share_of_step": round(sum(v["ms_total"] for k, v in ops.items()
                                                       if k in SIGNAL_OPS or k == "fit_params") / prof_run["ms"], 5),
                "denoiser_glue": {k: {"ms_avg": round(v["ms_avg"], 4), "GBps": round(v["gbs"], 1), "calls": v["calls"],
                                      "share": round(v["ms_total"] / prof_run["ms"], 4)}
                                  for k, v in ops.items() if k not in SIGNAL_OPS and k != "fit_params"},
                "profiled_ms_per_step": round(prof_run["ms"] / K, 3)}
    op_roof = operator_probe(device, peak, fp32_peak) if not a.skip_e2e else None
    cpu = None
    if not a.no_cpu_baseline:
        cpu = cpu_baseline_sample(a.config, steps=1)
    par = f"replicas x{world} (independent chains, no data-path collective; NCCL gather of outputs + filters inside e2e)"
    if joint:
        par = (f"{world} ranks, JOINT filter: all-reduce of the 3F fit statistics per fit and of sum|g|^2 per "
               "guidance call inside every step (NCCL), gather of outputs + filters inside e2e")
    line = {
        "metric": "blind-BWE sampler chain-steps/s", "value": round(value, 4), "unit": "chain-steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": round(dev_run["ms"] / K, 3),
        "higher_is_better": True, "scaling": "weak" if not cfg.get("recording") else "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE {cfg['tag']}: {cfg['what']}; {chains} rows/GPU x T={T} @ {cfg['sr']} Hz, "
                               f"random-init CQTDiff+ (7 octaves x {cfg['bins']} bins), {cfg['steps_T']}-step blind EDM "
                               f"sampler (order 2), NFFT={NFFT}, K={n_par}, fit max_iter=100",
                   "baseline_config": a.config, "joint_filter": joint,
                   "chains_per_gpu": chains, "total_chains": total_chains, "audio_len": T,
                   "sample_rate": cfg["sr"], "nfft": NFFT, "sampler_steps_per_s": round(K / (dev_run["ms"] / 1e3), 4),
                   "parallelism": par,
                   "l2_note": "per-step working set (activations of the 44.5M-param U-Net at B=8, >10 GB) far exceeds the 126 MB L2",
                   "tf32": bool(torch.backends.cudnn.allow_tf32),
                   "cuda_graph": graphed,
                   "host_enqueue_ms_per_step": round(dev_run.get("host", 0.0) * 1e3 / K, 1)},
        "e2e": {"value": round(e2e_value, 4), "unit": "chain-steps/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": round(e2e_run["ms"] / K, 3),
                "includes": "host-generator noise drawn into pinned memory + H2D every step, D2H of the step's estimate "
                            "and filter, final NCCL all-gather of outputs and filter estimates"
                            + (", hann cross-fade of the segments" if extra else ""),
                "gathered_shapes": e2e_run.get("gathered")},
        "gpu_launches": dev_run["launches"],
        "clocks": clocks,
        "roofline": roof, "operator_roofline": op_roof, "cpu_baseline": cpu,
    }
    if dumped is not None:
        line["dumped_outputs"] = dumped
    print(json.dumps(line))


DUMP_BYTES = 64_000_000          # all files of one dump, .npy headers included
NPY_HEADER_BYTES = 4096          # generous bound on one .npy header


def dump_outputs(out_dir, x, p, rank):
    """Write what the timed device-resident run returned after its last step -- the audio estimates of all
    ranks' chains and each rank's filter parameters -- as float32 DIR/<name>.npy, so that two builds can be
    compared output for output on identical inputs.  Estimates above the byte budget are written as every
    k-th element of the flattened rows (x_every_<k>.npy).  Arrays an earlier dump left in DIR are removed
    first.  Returns {name: shape} on rank 0."""
    import glob
    import numpy as np
    from babe_b200 import distributed as bd
    x, p = bd.gather_rows(x), bd.gather_params(p)
    if rank != 0:
        return None
    x, p = x.float().cpu(), p.float().cpu()
    k = -(-x.numel() * 4 // (DUMP_BYTES - 2 * NPY_HEADER_BYTES - p.numel() * 4))
    arrays = {"x" if k == 1 else f"x_every_{k}": x if k == 1 else x.reshape(-1)[::k], "filter_params": p}
    os.makedirs(out_dir, exist_ok=True)
    for old in glob.glob(os.path.join(out_dir, "x_every_*.npy")) + [os.path.join(out_dir, n) for n in
                                                                   ("x.npy", "filter_params.npy")]:
        if os.path.exists(old):
            os.remove(old)
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr.numpy())
    return {name: list(arr.shape) for name, arr in arrays.items()}


# ---------------------------------------------------------------------------
# "library" baseline on the same GPU: the reference's own torch formulation of the operator
# (torch.stft / torch.istft -> cuFFT, masked index ops, autograd) -- measurement only.
def torch_apply_filter(x, H, nfft):
    """utils/blind_bwe_utils.py:6-39 as the reference runs it on a GPU."""
    window = torch.hamming_window(window_length=nfft).to(x.device)
    xp = torch.cat((x, torch.zeros(*x.shape[:-1], nfft).to(x.device)), 1)
    X = torch.stft(xp, nfft, hop_length=nfft // 2, window=window, center=False, onesided=True, return_complex=True)
    X = X * H.unsqueeze(-1)
    return torch.istft(X, nfft, hop_length=nfft // 2, window=window, center=False, return_complex=False)[:, :x.shape[-1]]


def torch_design_filter(fc, A, f):
    """utils/blind_bwe_utils.py:82-119 (multi-slope branch)."""
    H = torch.zeros(f.shape).to(f.device)
    H[f < fc[0]] = 1
    H[f >= fc[0]] = 10 ** (A[0] * torch.log2(f[f >= fc[0]] / fc[0]) / 20)
    for i in range(1, len(fc)):
        H[f >= fc[i]] = 10 ** (A[i] * torch.log2(f[f >= fc[i]] / fc[i]) / 20) * H[f >= fc[i]][0]
    return H


def torch_fit_loop(xden, y, params, f, nfft, sr, iters=100):
    """testing/blind_bwe_sampler.py:556-590 as the reference runs it (Python loop, autograd, host syncs)."""
    window = torch.hamming_window(window_length=nfft).to(y.device)

    def stft(v):
        vp = torch.cat((v, torch.zeros(*v.shape[:-1], nfft).to(v.device)), 1)
        return torch.view_as_real(torch.stft(vp, nfft, hop_length=nfft // 2, window=window, center=False,
                                             onesided=True, return_complex=True))
    Xd, Y = stft(xden), stft(y)
    Xm = torch.sqrt(Xd[..., 0] ** 2 + Xd[..., 1] ** 2)
    Ym = torch.sqrt(Y[..., 0] ** 2 + Y[..., 1] ** 2)
    w = torch.sqrt(torch.linspace(0, 1, Xm.shape[1]).to(y.device)).unsqueeze(-1)
    mu = torch.tensor([1000.0, 10.0], device=y.device)
    p = params.clone()
    for _ in range(iters):
        p.requires_grad = True
        H = torch_design_filter(p[0], p[1], f)
        norm = torch.linalg.norm((Xm * H.unsqueeze(-1) * w).reshape(-1) - (Ym * w).reshape(-1), ord=2)
        g = torch.autograd.grad(norm, p, create_graph=True)
        p = p - mu.unsqueeze(1) * g[0]
        p.detach_()
        p[0, 0] = torch.clamp(p[0, 0], min=20, max=sr // 2)
        for k in range(1, p.shape[1]):
            p[0, k] = torch.clamp(p[0, k], min=p[0, k - 1] + 1, max=sr // 2)
        p[1, 0] = torch.clamp(p[1, 0], min=-50, max=-1)
        for k in range(1, p.shape[1]):
            p[1, k] = torch.clamp(p[1, k], min=-50, max=p[1, k - 1])
    return p


def _time_op(fn, iters, flush):
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
    return sorted(ts)[len(ts) // 2]


def operator_probe(device, peak, fp32_peak):
    """"operator % of HBM roofline" (second half of BASELINE.json's metric): the streaming
    operators alone at a batch that fills the GPU (config 4: B=512 x T=2^17, NFFT=4096; CQT at B=64 x 184184),
    CUDA events, L2 flushed between iterations; GB/s on the algorithmic bytes of SURVEY 8(d), TFLOP/s on the
    nominal flop counts (5 N log2 N per complex FFT)."""
    from babe_b200 import ops, sampler
    from cqt_nsgt_pytorch import CQT_nsgt
    SR, AUDIO_LEN = 22050, 184184
    B, T = 512, 1 << 17
    x = torch.randn(B, T, device=device) * 0.063
    y = torch.randn(B, T, device=device) * 0.063
    out = torch.empty_like(x)
    f = torch.fft.rfftfreq(NFFT, d=1 / SR).to(device)
    fc = torch.tensor([300.0, 600.0, 1000.0, 3000.0, 6000.0], device=device)
    A = torch.tensor([-10.0, -15.0, -20.0, -30.0, -40.0], device=device)
    fp = torch.stack((fc, A))
    cq = CQT_nsgt(7, 64, mode="oct", window=("kaiser", 1), fs=SR, audio_len=AUDIO_LEN, device=device)
    xc = torch.randn(64, AUDIO_LEN, device=device) * 0.063
    coefs = [None]

    def recg():
        xg = x.detach().requires_grad_(True)
        n = sampler.rec_guidance_norms(xg, y, f, fp, NFFT)
        torch.autograd.grad(n.sum(), xg)

    cqb = 64 * (4 * AUDIO_LEN + 8 * cq.plan.coef_per_row)
    cases = {
        "apply_filter": (lambda: ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, out=out), 8 * B * T, op_flops("apply_filter", B, T)),
        "apply_filter_adj": (lambda: ops.apply_filter(x, NFFT, freqs=f, fc=fc, A=A, adjoint=True, out=out), 8 * B * T,
                             op_flops("apply_filter", B, T)),
        "rec_guidance fwd+adj (20BT)": (recg, 20 * B * T, 2 * op_flops("apply_filter", B, T)),
        "stft_stats": (lambda: ops.stft_stats(x, y, NFFT), 8 * B * T, op_flops("stft_stats", B, T)),
        "cqt_analysis_B64": (lambda: coefs.__setitem__(0, cq.fwd(xc.unsqueeze(1))), cqb, op_flops("cqt_analysis", 64, 0, cq)),
        "cqt_synthesis_B64": (lambda: cq.bwd(coefs[0]), cqb, op_flops("cqt_synthesis", 64, 0, cq)),
        "hpf_DC_B64": (lambda: cq.apply_hpf_DC(xc), 64 * 8 * AUDIO_LEN, op_flops("hpf", 64, 0, cq)),
    }
    # a9 / a10: the STFT-distance guidance norm and its gradient on the spectrograms of 64 x 184184 (2049 bins x 88 frames)
    Xs = torch.randn(64, NFFT // 2 + 1, AUDIO_LEN // (NFFT // 2) - 1, 2, device=device)
    Rs = torch.randn_like(Xs)
    wl = torch.linspace(0, 1, NFFT // 2 + 1, device=device)
    c1 = torch.ones(1, device=device)
    cases["stft_distance_B64 (value, both spectrograms read)"] = (lambda: ops.spec_dist_stats(Xs, Rs, wl, 0), 8 * Xs.numel(), 0)
    cases["stft_distance_grad_B64 (both read, one gradient written)"] = (
        lambda: ops.spec_dist_grad(Xs, Rs, wl, c1, 0), 12 * Xs.numel(), 0)
    Hd = ops.design_filter(fc, A, f, strict=False)
    x8, y8 = x[:8, :AUDIO_LEN // 2].contiguous(), y[:8, :AUDIO_LEN // 2].contiguous()
    p0 = torch.tensor([[280.0, 285, 290, 295, 300], [-15.0, -17, -20, -25, -30]], device=device)
    cases["torch+cuFFT apply_filter (library baseline)"] = (lambda: torch_apply_filter(x, Hd, NFFT), 8 * B * T, 0)
    cases["torch+cuFFT hpf (rfft/irfft, library baseline) B64"] = (
        lambda: torch.fft.irfft(torch.fft.rfft(xc) * cq.plan.Hhpf, n=AUDIO_LEN), 64 * 8 * AUDIO_LEN, 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    res = {"shape": f"B={B} x T={T} (STFT ops), B=64 x T={AUDIO_LEN} (CQT ops)", "l2": "flushed between iterations",
           "fp32_peak_tflops": round(fp32_peak, 1)}
    for name, (fn, nbytes, fl) in cases.items():
        ms = _time_op(fn, 7, flush)
        gbs = nbytes / 1e9 / (ms / 1e3)
        r = {"ms": round(ms, 4), "GBps": round(gbs, 1), "frac": round(gbs / peak, 4)}
        if fl:
            r["tflops"] = round(fl / (ms / 1e3) / 1e12, 2)
            r["frac_fp32_peak"] = round(r["tflops"] / fp32_peak, 4)
        res[name] = r
    # filter fit: one launch vs the reference's Python loop on the same GPU (latency, 8 rows)
    fit = sampler.FilterFit(nfft=NFFT, sample_rate=SR, device=device)
    abc = fit.stats(x8, y8)
    for name, fn in (("fit_params 100 it (1 launch, statistics given)", lambda: fit(x8, y8, p0.clone(), abc=abc)),
                     ("fit_params 100 it (stats + 1 launch)", lambda: fit(x8, y8, p0.clone())),
                     ("torch fit loop 100 it (library baseline)", lambda: torch_fit_loop(x8, y8, p0, f, NFFT, SR))):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        res[name] = {"ms": round((time.perf_counter() - t0) * 1e3, 3)}
    return res


# ---------------------------------------------------------------------------
def cpu_world(cfg, chains, seed, max_iter=100):
    """The reference algorithm on the host: oracle operator + oracle CQT + the PyTorch restatement of the
    denoiser body on the CPU (babe_b200.denoiser equals networks/cqtdiff+.py -- tests/test_denoiser_cpu.py; the
    reference tree itself does not travel to the GPU box)."""
    from babe_b200 import denoiser, sampler
    from oracle import blind_sampler as obs, filter_fit as ofit
    from oracle import stft_filter as sf
    from oracle.cqt_shim import OracleCQT
    T = cfg["T"]
    args = sampler.make_args(sample_rate=cfg["sr"], audio_len=T, NFFT=NFFT, max_iter=max_iter, T=cfg["steps_T"],
                             bins_per_oct=cfg["bins"])
    torch.manual_seed(0)
    cqt = OracleCQT(7, cfg["bins"], window=("kaiser", 1), fs=cfg["sr"], audio_len=T, dtype=torch.float32)
    net = denoiser.CQTDiffPlus(args, "cpu", cqt=cqt)
    for p in net.parameters():
        p.requires_grad_(False)
    x = piano_like(chains, T, cfg["sr"], 1234 + seed)
    f = torch.fft.rfftfreq(NFFT, d=1 / cfg["sr"])
    y = sf.apply_filter(x, sf.design_filter([1000.0], [-20.0], f), NFFT)
    scfg = obs.SamplerConfig(T=cfg["steps_T"], audio_len=T)
    scfg.fit = ofit.FitConfig(nfft=NFFT, sample_rate=cfg["sr"], max_iter=max_iter)
    return scfg, net, cqt, y


def cpu_time_steps(config, steps, warmup):
    """Seconds for `steps` sampler steps of ONE full-length chain (no extrapolation)."""
    from oracle import blind_sampler as obs
    torch.set_num_threads(os.cpu_count() or 1)
    scfg, net, cqt, y = cpu_world(CONFIGS[config], 1, 0)
    marks = []

    class Marker(list):
        def append(self, item):
            marks.append(time.perf_counter())

    t0 = time.perf_counter()
    torch.manual_seed(42)
    obs.predict_blind_bwe(scfg, net, cqt.apply_hpf_DC, y, steps=warmup + steps, trace=Marker())
    start = t0 if warmup == 0 else marks[warmup - 1]
    return marks[warmup + steps - 1] - start


def cpu_baseline_sample(config, steps=1):
    cfg = CONFIGS[config]
    dt = cpu_time_steps(config, steps, 0)
    return {"value": round(steps / dt, 5), "unit": "chain-steps/s", "cores": torch.get_num_threads(),
            "kind": "port", "seconds": round(dt, 2),
            "sample": f"1 full-length chain (T={cfg['T']}) x {steps} sampler step(s) (2 denoiser fwd+bwd + 2 filter fits + "
                      "2 guidance evaluations each), measured, not extrapolated; oracle operator/CQT + PyTorch CPU denoiser"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[a.config]
    K, W = a.steps, a.warmup
    # bounded sample: ONE of the GPU arm's chains at full length; main() rejects more timed steps than
    # --ref-max-steps, and the warm-up is capped (the per-step time of the CPU path does not depend on the step index)
    Kc = K
    Wc = min(W, 5)
    dt = cpu_time_steps(a.config, Kc, Wc)
    v = Kc / dt
    cpu = {"value": round(v, 5), "unit": "chain-steps/s", "cores": torch.get_num_threads(), "kind": "port",
           "sample": f"1 chain of the workload at full length T={cfg['T']}, {Kc} timed sampler steps after {Wc} warm-up "
                     f"steps (requested {K}/{W}; warm-up capped to bound the run), measured, not extrapolated; the reference is "
                     "Python: the oracle port restates it"}
    n_par = len(cfg["fc"])
    line = {"impl": "reference", "metric": "blind-BWE sampler chain-steps/s", "value": round(v, 5),
            "unit": "chain-steps/s", "n_gpus": a.gpus, "steps": Kc, "warmup": Wc,
            "ms_per_step": round(dt / Kc * 1e3, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"BASELINE {cfg['tag']}: {cfg['what']}; bounded sample: 1 row x T={cfg['T']} @ {cfg['sr']} Hz, "
                                   f"random-init CQTDiff+ (7 octaves x {cfg['bins']} bins), {cfg['steps_T']}-step blind EDM "
                                   f"sampler (order 2), NFFT={NFFT}, K={n_par}, fit max_iter=100; host cores only",
                       "baseline_config": a.config, "requested_steps": K, "requested_warmup": W},
            "cpu_baseline": cpu,
            "e2e": {"value": round(v, 5), "unit": "chain-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------
def run_operator_sweep(a):
    """Config 4: operator microbenchmark, STFT -> parametric filter -> iSTFT + gradients."""
    from babe_b200 import build, ops, sampler
    build.build()
    dev = torch.device("cuda")
    peak, src = measured_peak()
    fp32_peak = fp32_peak_tflops(None)
    SR, AUDIO_LEN = 22050, 184184
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rows = []
    if a.shapes:
        shapes = [tuple(int(v) for v in s.split("x")) for s in a.shapes.split(",")]
    elif a.grid == "full":
        shapes = [(B, 1 << e) for e in range(14, 21) for B in (1, 2, 4, 8, 16, 32, 64, 128, 256, 512)]
    else:
        shapes = [(1, 1 << 14), (8, 1 << 17), (64, 1 << 17), (8, AUDIO_LEN), (64, AUDIO_LEN), (512, 1 << 17), (512, 1 << 20)]
    nffts = [int(v) for v in a.nffts.split(",")]
    for nfft in nffts:
        f = torch.fft.rfftfreq(nfft, d=1 / SR).to(dev)
        fc = torch.tensor([300.0, 600.0, 1000.0, 3000.0, 6000.0], device=dev)
        A = torch.tensor([-10.0, -15.0, -20.0, -30.0, -40.0], device=dev)
        for B, T in shapes:
            if B * T * 4 > (2 << 30):
                continue
            x = torch.randn(B, T, device=dev) * 0.063
            y = torch.randn(B, T, device=dev) * 0.063
            out = torch.empty_like(x)
            fit = sampler.FilterFit(nfft=nfft, sample_rate=SR, device=dev)
            p = torch.tensor([[280.0, 285, 290, 295, 300], [-15.0, -17, -20, -25, -30]], device=dev)
            fp = torch.stack((fc, A))
            spec_bytes = 8 * B * (nfft // 2 + 1) * ops.num_frames(T, nfft)
            fl_filter = B * (T / nfft) * (2 * _fft_flops(nfft) + 10 * nfft)
            fl_stft = B * (T / nfft) * _fft_flops(nfft)

            def recg(x=x, y=y, fp=fp, f=f, nfft=nfft):
                xg = x.detach().requires_grad_(True)
                n = sampler.rec_guidance_norms(xg, y, f, fp, nfft)
                torch.autograd.grad(n.sum(), xg)

            abc = ops.stft_stats(x, y, nfft)
            X = ops.stft(x, nfft)
            cases = {
                "apply_filter fwd (8BT)": (lambda: ops.apply_filter(x, nfft, freqs=f, fc=fc, A=A, out=out), 8 * B * T, fl_filter),
                "apply_filter adj (8BT)": (lambda: ops.apply_filter(x, nfft, freqs=f, fc=fc, A=A, adjoint=True, out=out),
                                           8 * B * T, fl_filter),
                "fit statistics (8BT)": (lambda: ops.stft_stats(x, y, nfft), 8 * B * T,
                                         B * (T / (nfft // 2)) * (_fft_flops(nfft) + 14 * nfft)),
                "fit loop 100 it": (lambda: fit(x, y, p.clone(), abc=abc), 0, 0),
                "rec-guidance norms + grad (20BT, r materialised)": (recg, 20 * B * T, 2 * fl_filter),
                "apply_stft a1 (4BT + 8BFM)": (lambda: ops.stft(x, nfft), 4 * B * T + spec_bytes, fl_stft),
                "apply_filter_istft a2 (8BFM + 4BT)": (lambda: ops.istft(X, nfft), 4 * B * T + spec_bytes, fl_stft),
            }
            for name, (fn, nbytes, fl) in cases.items():
                ms = _time_op(fn, a.iters, flush if B * T * 8 < (252 << 20) else None)
                gbs = nbytes / 1e9 / (ms / 1e3) if nbytes else 0.0
                tf = fl / (ms / 1e3) / 1e12 if fl else 0.0
                rows.append({"nfft": nfft, "B": B, "T": T, "op": name, "ms": round(ms, 4), "GBps": round(gbs, 1),
                             "frac_of_peak": round(gbs / peak, 4), "tflops": round(tf, 3),
                             "frac_fp32_peak": round(tf / fp32_peak, 4)})
                print(json.dumps(rows[-1]), flush=True)
            del x, y, out, X
    print(json.dumps({"mode": "operator", "peak_GBps": peak, "peak_source": src,
                      "fp32_peak_tflops_at_max_clock": round(fp32_peak, 1), "rows": len(rows)}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="sampler", choices=["sampler", "operator"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS),
                    help="BASELINE.json config: 1 = one 6 s segment, 2 = 64 chains over 8 GPUs (default, the contract "
                         "line), 3 = 44.1 kHz / 11 s / 96 bins per octave, 5 = 60 s recording with a joint filter")
    ap.add_argument("--joint", action="store_true",
                    help="one filter / one guidance norm for the rows of ALL ranks (all-reduces inside every step)")
    ap.add_argument("--chains", type=int, default=0, help="rows per GPU (default: the config's)")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--shapes", default="")
    ap.add_argument("--grid", default="", choices=["", "full"], help="operator mode: the full 2^14..2^20 x 1..512 grid")
    ap.add_argument("--nffts", default="4096", help="operator mode: comma-separated NFFTs (e.g. 4096,1024)")
    ap.add_argument("--ref-max-steps", type=int, default=30,
                    help="reference arm: largest --steps accepted (each step ~7 s of host time at T=184184)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling aid: skip the host-buffer leg")
    ap.add_argument("--no-cuda-graph", action="store_true",
                    help="run everything eagerly instead of replaying captured CUDA graphs")
    ap.add_argument("--no-step-graph", action="store_true",
                    help="capture only the denoiser's forward / backward (round-1 behaviour), not the whole step")
    ap.add_argument("--single-pass", action="store_true",
                    help="profiling aid: skip the second (per-kernel event timing) pass")
    ap.add_argument("--no-autotune", action="store_true", help="profiling aid: cudnn.benchmark off")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the audio estimates and filter parameters of the timed run's last step as DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference" and a.steps > a.ref_max_steps:
        ap.error(f"--impl reference times at most --ref-max-steps ({a.ref_max_steps}) steps; raise it to time more")
    if a.dump_outputs and (a.impl == "reference" or a.mode == "operator"):
        ap.error("--dump-outputs writes the outputs of the CUDA sampler run (--impl ours --mode sampler)")
    if a.impl != "reference":
        a.warmup = max(1, a.warmup)          # the timed region starts after a completed (untimed) step
    if a.impl == "reference":
        return run_reference(a)
    if a.mode == "operator":
        return run_operator_sweep(a)
    return run_ours(a)


if __name__ == "__main__":
    main()
    import torch.distributed as _dist
    if _dist.is_available() and _dist.is_initialized():
        _dist.destroy_process_group()
