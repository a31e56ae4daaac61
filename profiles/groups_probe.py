"""Grouped filter estimation (``filter_groups``) against the shared and per-row modes, on one GPU:

  (a) CUDA-event times of ``ops.stft_stats_groups`` (every launch of one call) against ``ops.stft_stats`` and
      ``ops.stft_stats_rows`` at 8 and 64 x 184184, NFFT 4096, layouts [8], [1]*8, [3, 5] (B = 8) and 8 x 8 (B = 64);
      x and y stay in the 126 MB L2 across the timed repetitions, as they do inside a sampler step;
  (b) ms per sampler step at B = 8 x 184184 (bench config 2, random-init CQTDiff+, whole-step CUDA graph), grouped
      [4, 4] against shared;
  (c) four 60 s recordings of bench config 5 (8 segments of 184184 each, 35 steps) restored three ways: four
      ``restore_recording(joint=True)`` calls (eager: joint mode has no step graph), ``restore_recordings(max_rows=8)``
      (four grouped calls, step graph on) and one ``restore_recordings`` call (B = 32; ``max_rows=16`` instead if
      B = 32 does not fit).  Wall time from the call to a device synchronise, step-graph captures included.

    python profiles/groups_probe.py OUT.json [--steps K] [--skip-restore]
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


def stats(res):
    from babe_b200 import ops
    nfft, T = 4096, 184184
    out = res["a_stats"] = []
    for B, layouts in ((8, ([8], [1] * 8, [3, 5])), (64, ([8] * 8,))):
        g = torch.Generator(device="cuda").manual_seed(B)
        x = torch.randn(B, T, device="cuda", generator=g) * 0.063
        y = torch.randn(B, T, device="cuda", generator=g) * 0.05
        calls = {"stft_stats": lambda: ops.stft_stats(x, y, nfft),
                 "stft_stats_rows": lambda: ops.stft_stats_rows(x, y, nfft)}
        for sizes in layouts:
            calls[f"groups {sizes if len(set(sizes)) > 1 else f'{len(sizes)} x {sizes[0]}'}"] = \
                lambda sizes=sizes: ops.stft_stats_groups(x, y, nfft, sizes)
        best = {k: [] for k in calls}
        for _ in range(3):                                   # alternate the calls, keep the best of three windows
            for k, fn in calls.items():
                best[k].append(event_ms(fn))
        for k, v in best.items():
            out.append({"op": k, "B": B, "T": T, "ms": min(v)})
            print(json.dumps(out[-1]), flush=True)
        if B == 8:
            res["bitwise_B8"] = {
                "[8] == stft_stats": bool(torch.equal(ops.stft_stats_groups(x, y, nfft, [8])[0],
                                                      ops.stft_stats(x, y, nfft))),
                "[1]*8 == stft_stats_rows": bool(torch.equal(ops.stft_stats_groups(x, y, nfft, [1] * 8),
                                                             ops.stft_stats_rows(x, y, nfft)))}
            print(json.dumps(res["bitwise_B8"]), flush=True)


def sampler_steps(res, steps):
    import bench
    cfg = bench.CONFIGS[2]
    out = res["b_sampler_step"] = {}
    torch.backends.cudnn.benchmark = True
    args, net, smp, y, _ = bench.build_world(torch.device("cuda", 0), cfg, cfg["chains"], 0)
    smp.step_graph = True
    for rep in range(2):                                     # alternate the modes twice
        for groups in (None, [4, 4]):
            smp.filter_groups = groups
            evs = []

            def hook(i, x, p):
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                evs.append(e)
            torch.manual_seed(0)
            smp.predict_blind_bwe(y, max_steps=steps + 2, step_hook=hook)
            torch.cuda.synchronize()
            ms = evs[1].elapsed_time(evs[-1]) / (len(evs) - 2)
            key = "shared" if groups is None else "grouped_4_4"
            out.setdefault(key + "_ms_per_step", []).append(ms)
            out["graphed"] = bool(smp._step_graphs)
            print(key, ms, flush=True)
    smp.filter_groups = None
    out.update({"B": int(y.shape[0]), "T": int(y.shape[1]), "steps_timed": steps})


def restore(res):
    import bench
    from babe_b200 import blind_bwe_utils as bu, segments
    cfg = bench.CONFIGS[5]
    torch.backends.cudnn.benchmark = True
    args, net, smp, _, _ = bench.build_world(torch.device("cuda", 0), cfg, cfg["chains"], 0)
    f = torch.fft.rfftfreq(4096, d=1 / cfg["sr"]).cuda()
    recs = []
    for r, fc in enumerate((1000.0, 1500.0, 2500.0, 4000.0)):
        rec = bench.piano_like(1, cfg["recording"], cfg["sr"], 1234 + 5 + r).cuda()
        recs.append(bu.apply_filter(rec, bu.design_filter([fc], [-20.0], f), 4096))
    n_seg = [int(segments.split(d, cfg["T"])[0].shape[0]) for d in recs]
    steps = int(args.tester.T)
    out = res["c_four_recordings"] = {"L": int(recs[0].shape[-1]), "seg_len": cfg["T"], "n_segments": n_seg,
                                      "steps": steps, "runs": []}
    seeds = [11, 12, 13, 14]
    chain_steps = sum(n_seg) * steps

    def joint_calls():
        smp.step_graph = False
        fds = []
        for r, d in enumerate(recs):
            try:
                _, fd = segments.restore_recording(smp, d, cfg["T"], joint=True, seed=seeds[r])
            finally:
                smp.joint = False                            # restore_recording(joint=True) leaves it set
            fds.append(fd)
        return fds

    def grouped(max_rows):
        def run():
            smp.step_graph = True
            return [fd for _, fd in segments.restore_recordings(smp, recs, cfg["T"], seeds=seeds, max_rows=max_rows)]
        return run

    ways = [("4 x restore_recording(joint=True), eager", joint_calls),
            ("restore_recordings(max_rows=8), step graph", grouped(8)),
            ("restore_recordings (B = 32), step graph", grouped(None))]
    for rep in range(2):
        for name, fn in ways:
            # captured step graphs keep their memory pool while the sampler holds them (B = 32: tens of GB); drop them
            # so that every way starts from the same memory state
            smp._step_graphs, smp._step_key = {}, None
            torch.cuda.empty_cache()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            try:
                fds = fn()
            except torch.cuda.OutOfMemoryError as exc:
                out["runs"].append({"way": name, "rep": rep, "error": f"out of memory: {exc}"[:300]})
                print(json.dumps(out["runs"][-1]), flush=True)
                torch.cuda.empty_cache()
                if "B = 32" in name:
                    ways[2] = ("restore_recordings(max_rows=16), step graph", grouped(16))
                continue
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            filts = [fd[0][1] for fd in fds]
            out["runs"].append({"way": name, "rep": rep, "wall_s": dt, "chain_steps_per_s": chain_steps / dt,
                                "filters": [v.flatten().tolist() for v in filts],
                                "max_memory_GB": torch.cuda.max_memory_allocated() / 1e9})
            print(json.dumps({k: v for k, v in out["runs"][-1].items() if k != "filters"}), flush=True)
    # the restorations themselves: one filter per recording, the grouped ways against the joint calls
    ref = {r["way"]: r["filters"] for r in out["runs"] if "filters" in r and r["rep"] == 1}
    base = next(v for k, v in ref.items() if k.startswith("4 x"))
    out["filter_rel_diff_vs_joint"] = {
        k: [float(torch.tensor(a).sub(torch.tensor(b)).norm() / torch.tensor(b).norm()) for a, b in zip(v, base)]
        for k, v in ref.items() if not k.startswith("4 x")}
    print(json.dumps(out["filter_rel_diff_vs_joint"]), flush=True)


def main():
    path = sys.argv[1]
    steps = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 6
    from babe_b200 import build
    build.build()
    res = {"card": card(), "torch": torch.__version__}
    print(res, flush=True)
    stats(res)
    sampler_steps(res, steps)
    if "--skip-restore" not in sys.argv:
        restore(res)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
