"""CPU: the __host__ __device__ FFT building blocks of the kernels (in-register butterflies, the
conjugate-symmetric odd-prime DFTs, the mixed-radix Stockham stages with their skewed buffers and
multiply-shift index arithmetic) compiled for the host with nvcc and checked against a naive
double-precision DFT (tests/host/fft_host_check.cu).  No GPU involved."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_fft_building_blocks_on_host(tmp_path):
    exe = str(tmp_path / "fft_host_check")
    src = os.path.join(ROOT, "tests", "host", "fft_host_check.cu")
    cmd = [NVCC, "-O1", "-std=c++17", "-o", exe, src, "-I", os.path.join(ROOT, "babe_b200", "csrc"),
           "-I", os.path.join(ROOT, "include")]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)
    out = subprocess.run([exe], check=True, capture_output=True, text=True, timeout=600).stdout
    rows = [l.split() for l in out.strip().splitlines()]
    assert len(rows) == 27
    for name, n, err in rows:
        assert float(err) < 2e-6, (name, n, err)        # fp32 transforms of <= 2048 points


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_core3_passes_on_host(tmp_path):
    """Core3 (csrc/stft_cores.cuh): forward / mirror / inverse passes of the 4096-point core of
    k_apply_filter, k_stft_stats and k_fir_filter, emulated thread by thread on the host."""
    exe = str(tmp_path / "core3_host_check")
    src = os.path.join(ROOT, "tests", "host", "core3_host_check.cu")
    cmd = [NVCC, "-O1", "-std=c++17", "-o", exe, src, "-I", os.path.join(ROOT, "babe_b200", "csrc"),
           "-I", os.path.join(ROOT, "include")]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)
    out = subprocess.run([exe], check=True, capture_output=True, text=True, timeout=600).stdout
    vals = dict(l.split() for l in out.strip().splitlines())
    assert float(vals["fwd"]) < 5e-7 and float(vals["roundtrip"]) < 5e-7 and float(vals["mirror"]) == 0.0


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_filter_design_device_logic_on_host(tmp_path, golden):
    """csrc/filter_design.cuh (what k_design_filter and the fused kernels run: breakpoint search, anchor
    chain through the parents, bin ownership, the reference's fp32 operation order) executed on the host
    against H vectors produced by the reference's design_filter (tests/golden/operator_*.npz), including
    the duplicate-bin / last-bin case and the scalar branch."""
    import numpy as np
    exe = str(tmp_path / "filter_design_host_check")
    src = os.path.join(ROOT, "tests", "host", "filter_design_host_check.cu")
    cmd = [NVCC, "-O1", "-std=c++17", "-o", exe, src, "-I", os.path.join(ROOT, "babe_b200", "csrc"),
           "-I", os.path.join(ROOT, "include")]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)

    def run(f, fc, A, gH=None):
        fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
        with open(fin, "wb") as fh:
            np.asarray([f.size, fc.size], dtype=np.int32).tofile(fh)
            f.astype(np.float32).tofile(fh)
            fc.astype(np.float32).tofile(fh)
            A.astype(np.float32).tofile(fh)
            if gH is not None:
                gH.astype(np.float32).tofile(fh)
        subprocess.run([exe, fin, fout], check=True, timeout=60)
        raw = np.fromfile(fout, dtype=np.float32)
        H, bad = raw[:f.size], int(raw[f.size:f.size + 1].view(np.int32)[0])
        if gH is None:
            return H, bad
        K = fc.size
        return H, bad, raw[f.size + 1:f.size + 1 + K], raw[f.size + 1 + K:f.size + 1 + 2 * K]

    for tag in ("operator_n1024.npz", "operator_n4096.npz"):
        g = golden(tag)
        f = g["f"]
        H, bad = run(f, g["fc"], g["A"])
        assert bad == 0 and np.linalg.norm(H - g["H"]) / np.linalg.norm(g["H"]) < 2e-6
        H, bad = run(f, g["fc_dup"], g["A_dup"])
        assert bad == 0 and np.linalg.norm(H - g["H_dup"]) / np.linalg.norm(g["H_dup"]) < 2e-6
        H, bad = run(f, np.asarray([1000.0]), np.asarray([-20.0]))
        assert np.linalg.norm(H - g["H_list"]) / np.linalg.norm(g["H_list"]) < 2e-6
        # analytic gradients wrt (fc, A) through the anchor chain against the reference's autograd
        for cot, kfc, kA, tol in (("cotH", "gfc", "gA", 2e-5), ("fit_gH", "fit_gfc", "fit_gA", 1e-4)):
            _, _, gfc, gA = run(f, g["fc"], g["A"], g[cot])
            assert np.linalg.norm(gfc - g[kfc]) / np.linalg.norm(g[kfc]) < tol
            assert np.linalg.norm(gA - g[kA]) / np.linalg.norm(g[kA]) < tol
    # a breakpoint above the last bin: flagged (the reference raises IndexError there)
    _, bad = run(g["f"], np.asarray([500.0, 1e6]), np.asarray([-10.0, -20.0]))
    assert bad == 1


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_fit_iteration_device_math_on_host(tmp_path, golden):
    """The projected-gradient iteration of k_fit_params assembled on the host from the device functions
    (segments, per-bin gain, chain rule, fp32 step, sequential clamps, stopping test) against the
    trajectories of the reference's own BlindSampler.fit_params (tests/golden/fit_sampler.npz): 1 and 5
    iterations tight, 100 iterations loose (the descent is chaotic in fp32, see DESIGN.md section 2)."""
    import ctypes

    import numpy as np
    import torch
    from babe_b200._lib import FitConfig
    from oracle import stft_filter as osf
    exe = str(tmp_path / "fit_host_check")
    src = os.path.join(ROOT, "tests", "host", "fit_host_check.cu")
    cmd = [NVCC, "-O1", "-std=c++17", "-o", exe, src, "-I", os.path.join(ROOT, "babe_b200", "csrc"),
           "-I", os.path.join(ROOT, "include")]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)
    g = golden("fit_sampler.npz")
    nfft, sr = int(g["nfft"]), int(g["sr"])
    F = nfft // 2 + 1
    a, b, c = osf.stft_mag_stats(torch.from_numpy(g["fit_xden"]).double(), torch.from_numpy(g["y"]).double(), nfft)
    abc = torch.stack((a, b, c)).numpy().astype(np.float64)
    w = osf.freq_weight_vector("sqrt", F).numpy().astype(np.float32)
    f = np.fft.rfftfreq(nfft, d=1 / sr).astype(np.float32)

    def run(p0, iters):
        cfg = FitConfig(mu_fc=1000, mu_A=10, fcmin=20, fcmax=sr // 2, Amin=-50, Amax=30, tol_fc=5e-3, tol_A=5e-3,
                        max_iter=iters, clamp_fc=1, clamp_A=1, only_negative_A=1)
        fin, fout = str(tmp_path / "fit_in.bin"), str(tmp_path / "fit_out.bin")
        K = p0.shape[1]
        with open(fin, "wb") as fh:
            np.asarray([F, K], dtype=np.int32).tofile(fh)
            fh.write(bytes(cfg))
            abc.tofile(fh)
            w.tofile(fh)
            f.tofile(fh)
            p0.astype(np.float32).tofile(fh)
        subprocess.run([exe, fin, fout], check=True, timeout=120)
        raw = np.fromfile(fout, dtype=np.float32)
        return raw[:2 * K].reshape(2, K), int(raw[2 * K:].view(np.int32)[0])

    rel = lambda x, y: np.linalg.norm(x - y) / np.linalg.norm(y)
    for iters, tol in ((1, 1e-5), (5, 1e-5), (100, 3e-2)):
        p, _ = run(g["fit_p0"], iters)
        assert rel(p, g[f"fit_p_{iters}"]) < tol, iters
    p7, _ = run(g["fit7_p0"], 100)
    assert rel(p7, g["fit7_p"]) < 3e-2


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_rfft_pair_processing_on_host(tmp_path):
    """csrc/rfft_pairs.cuh: real FFT of Ls points from the complex FFT of Ls/2 points and back."""
    exe = str(tmp_path / "rfft_pairs_host_check")
    src = os.path.join(ROOT, "tests", "host", "rfft_pairs_host_check.cu")
    cmd = [NVCC, "-O1", "-std=c++17", "-o", exe, src, "-I", os.path.join(ROOT, "babe_b200", "csrc"),
           "-I", os.path.join(ROOT, "include")]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)
    out = subprocess.run([exe], check=True, capture_output=True, text=True, timeout=600).stdout
    vals = dict(l.split() for l in out.strip().splitlines())
    assert float(vals["post"]) < 5e-7 and float(vals["pre"]) < 5e-7


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_core4k_passes_on_host(tmp_path):
    """Core4k (csrc/core4k.cuh) and fft16v (csrc/fft16v.cuh): the 4096-point core of the round-2 fused kernels
    (csrc/stft_fused.cu) -- forward / inverse passes with the half-warp-local second exchange, both twiddle
    sources, the scaled first butterfly stage and the permuted real-symmetric table addressing -- emulated
    thread by thread on the host against naive double-precision DFTs."""
    exe = str(tmp_path / "core4k_host_check")
    src = os.path.join(ROOT, "tests", "host", "core4k_host_check.cu")
    cmd = [NVCC, "-O1", "-std=c++17", "-o", exe, src, "-I", os.path.join(ROOT, "babe_b200", "csrc"),
           "-I", os.path.join(ROOT, "include")]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)
    out = subprocess.run([exe], check=True, capture_output=True, text=True, timeout=600).stdout
    vals = dict(l.split() for l in out.strip().splitlines())
    assert float(vals["fft16"]) < 2e-7 and float(vals["fft16_scaled"]) < 3e-7
    for k in ("fwd_regs", "fwd_smem", "roundtrip_regs", "roundtrip_smem"):
        assert float(vals[k]) < 5e-7, (k, vals[k])
    assert float(vals["perm"]) == 0.0


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
@pytest.mark.parametrize("plan", [0, 1, 2, 3, 4, 6, 7])
def test_prime_factor_passes_on_host(tmp_path, plan):
    """csrc/cqt_pfa.cuh: the prime-factor (Good-Thomas) two-pass transform of the CQT -- index maps, in-place odd-prime
    DFT stages, r2c / c2r pair processing, the fused filter pass and the table-driven gather -- emulated thread by
    thread on the host (tests/host/pfa_host_check.cu) against numpy's rfft / irfft.  Plans: two small ones (even and
    odd N1), Ls = 184184 (BASELINE configs[1]) with 16- and 8-column tiles, Ls = 368368, and the two lengths whose prime
    powers are single digits (Ls = 132300 = 2 * 2 * 27 * 25 * 49, Ls = 485100 = 2 * 2 * 9 * 25 * 49 * 11)."""
    import numpy as np
    exe = str(tmp_path / "pfa_host_check")
    src = os.path.join(ROOT, "tests", "host", "pfa_host_check.cu")
    cmd = [NVCC, "-O1", "-std=c++17", "-o", exe, src, "-I", os.path.join(ROOT, "babe_b200", "csrc"),
           "-I", os.path.join(ROOT, "include")]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)
    d = str(tmp_path)
    subprocess.run([exe, str(plan), d], check=True, capture_output=True, timeout=600)
    ld = lambda n, dt: np.fromfile(os.path.join(d, n), dtype=dt)
    x, H, sc = (ld(n, np.float32).astype(np.float64) for n in ("x.f32", "H.f32", "scale.f32"))
    X, y, xr, xg = ld("X.c64", np.complex64), ld("y.f32", np.float32), ld("xr.f32", np.float32), ld("xg.f32", np.float32)
    BS, src_tab = ld("BS.c64", np.complex64).astype(np.complex128), ld("src.i32", np.int32).reshape(-1, 4)
    rel = lambda a, b: float(np.linalg.norm(a - b) / np.linalg.norm(b))
    Xr = np.fft.rfft(x)
    assert rel(X, Xr * sc) < 5e-7
    assert rel(y, np.fft.irfft(Xr * H, n=len(x))) < 5e-7
    Xin = X.astype(np.complex128) * H
    Xin[0], Xin[-1] = Xin[0].real, Xin[-1].real
    assert rel(xr, np.fft.irfft(Xin, n=len(x))) < 5e-7
    G = np.zeros(len(src_tab), np.complex128)
    for q in range(3):
        G += BS[src_tab[:, q]]                      # "no band" entries point at the pool's zero element
    G *= sc
    G[0], G[-1] = G[0].real, G[-1].real
    assert rel(xg, np.fft.irfft(G, n=len(x))) < 5e-7


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_packed_band_cores_on_host(tmp_path):
    """BandCoreV<R3> / BandCoreS<R2> (csrc/bandfft_v.cuh): the packed forward / inverse band transforms of the CQT
    kernels (M = 32 ... 4096, window multiply folded into the first butterflies) emulated thread by thread."""
    exe = str(tmp_path / "bandfft_v_host_check")
    src = os.path.join(ROOT, "tests", "host", "bandfft_v_host_check.cu")
    cmd = [NVCC, "-O1", "-std=c++17", "-o", exe, src, "-I", os.path.join(ROOT, "babe_b200", "csrc"),
           "-I", os.path.join(ROOT, "include")]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)
    out = subprocess.run([exe], check=True, capture_output=True, text=True, timeout=600).stdout
    rows = [l.split() for l in out.strip().splitlines()]
    assert sorted({int(r[1]) for r in rows}) == [32, 64, 128, 256, 512, 1024, 2048, 4096] and len(rows) == 16
    for r in rows:
        assert float(r[4]) < 5e-7, r
