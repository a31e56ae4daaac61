"""CPU: keyed per-row noise (``BlindSamplerFused.row_seeds``, DESIGN.md 4.8).  The Philox4x32-10 generator of
csrc/philox.cuh compiled for the host against the Random123 known-answer vectors, the numpy restatement the GPU
tests compare with, the seed derivation of the segment drivers, argument checks, and the seeds the drivers hand
to the sampler for every segment, window and rank.  The kernel itself is checked on the GPU
(tests/test_row_noise_gpu.py)."""
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import row_noise_ref as ref
from toy_model import ToyDenoiser

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_philox_header_on_host(tmp_path):
    exe = str(tmp_path / "philox_host_check")
    src = os.path.join(ROOT, "tests", "host", "philox_host_check.cu")
    cmd = [NVCC, "-O1", "-std=c++17", "-o", exe, src, "-I", os.path.join(ROOT, "babe_b200", "csrc"),
           "-I", os.path.join(ROOT, "include")]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)
    out = subprocess.run([exe], check=True, capture_output=True, text=True, timeout=60).stdout
    rows = {l.split()[0]: l.split()[1:] for l in out.strip().splitlines()}
    for i, (_, _, want) in enumerate(ref.KAT):
        assert tuple(int(w, 16) for w in rows[f"kat{i}"]) == want, i
    assert float.fromhex(rows["u0"][0]) == 2.0 ** -24                # never 0
    assert float.fromhex(rows["u1"][0]) == 1.0 - 2.0 ** -24          # never 1


def test_numpy_restatement():
    for c, k, want in ref.KAT:
        assert tuple(int(v) for v in ref.philox4x32_10(*c, *k)) == want
    assert ref.uniform(0) == 2.0 ** -24 and ref.uniform(0xFFFFFFFF) == 1.0 - 2.0 ** -24
    # sample n of a row is word n % 4 of counter n // 4: a shorter row is the prefix of a longer one
    a, b = ref.row_noise(123, 5, 37), ref.row_noise(123, 5, 1001)
    assert np.array_equal(a, b[:37])
    x0, x1, _, _ = ref.philox4x32_10(0, 5, 0, 0, 123, 0)
    r = np.sqrt(-2 * np.log(ref.uniform(x0)))
    assert a[0] == r * np.cos(2 * np.pi * ref.uniform(x1)) and a[1] == r * np.sin(2 * np.pi * ref.uniform(x1))
    assert np.abs(a).max() <= np.sqrt(48 * np.log(2))                  # the 5.77 sigma cut


def test_row_seed_is_splitmix64():
    from babe_b200.segments import row_seed
    # SplitMix64 started at 0: its first three outputs
    assert [row_seed(0, k) for k in range(3)] == [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F]
    mask = (1 << 64) - 1
    z = (42 + 8 * 0x9E3779B97F4A7C15) & mask
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & mask
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & mask
    assert row_seed(42, 7) == z ^ (z >> 31)
    for seed in (0, 1, 2 ** 64 - 1):
        seeds = [row_seed(seed, k) for k in range(10_000)]
        assert len(set(seeds)) == len(seeds) and all(0 <= v < 2 ** 64 for v in seeds)


# --------------------------------------------------------------------------- argument checks
def _sampler():
    from babe_b200 import edm, sampler
    args = sampler.make_args(audio_len=8192, T=4, NFFT=1024, max_iter=3)
    return sampler.BlindSamplerFused(ToyDenoiser(), edm.EDM(args), args, rid=False)


def test_row_seeds_validation():
    s = _sampler()
    assert s.row_seeds is None
    y = torch.zeros(3, 8192)
    for bad in ([1, 2], [1, 2, 3, 4], torch.arange(2), torch.arange(3, dtype=torch.int32),
                torch.zeros(3), [1.0, 2.0, 3.0], [1, 2, 2 ** 64], torch.zeros(3, 1, dtype=torch.int64)):
        s.row_seeds = bad
        with pytest.raises(ValueError):
            s.predict_blind_bwe(y.clone())
    s.row_seeds = [1, 2]
    with pytest.raises(ValueError):
        s.predict_unconditional((3, 8192), "cpu")
    with pytest.raises(ValueError):
        s.predict_bwe(y.clone(), torch.tensor([[500.0], [-20.0]]), "fc_A")
    s.row_seeds = [1, 2, 3]
    s.noise_fn = lambda shape, dev: torch.zeros(shape)
    with pytest.raises(ValueError, match="noise_fn"):
        s.predict_blind_bwe(y.clone())
    assert s._seed_tensor([0, 2 ** 64 - 1, -1, 2 ** 63]).tolist() == [0, -1, -1, -2 ** 63]


def test_ops_row_noise_rejects_cpu_and_bad_arguments():
    from babe_b200 import ops
    from babe_b200._lib import BabeError
    seeds = torch.arange(3, dtype=torch.int64)
    with pytest.raises(BabeError):
        ops.row_noise(seeds, (3, 100), 0)
    with pytest.raises(BabeError):
        ops.row_noise(seeds, torch.zeros(3, 100), 0)
    with pytest.raises(TypeError):
        ops.row_noise([1, 2, 3], (3, 100), 0)


# --------------------------------------------------------------------------- seeds handed out by the drivers
class _SeedRecorder:
    """Records the row seeds of every call; 'restoration' = the input."""

    def __init__(self):
        self.row_seeds, self.filter_per_row, self.joint = None, False, False
        self.calls = []

    def predict_blind_bwe(self, y, rid=False):
        self.calls.append(("blind", list(self.row_seeds) if self.row_seeds is not None else None))
        filt = torch.tensor([[500.0], [-20.0]])
        if self.filter_per_row:
            filt = filt.expand(y.shape[0], -1, -1).contiguous()
        return y.clone(), filt

    def predict_bwe(self, seg, filt, typefilter, rid=False):
        self.calls.append(("bwe", list(self.row_seeds)))
        return seg.clone()

    def predict_bwe_AR(self, seg, y_masked, filt, typefilter, rid=False, mask=None):
        self.calls.append(("ar", list(self.row_seeds)))
        return seg.clone()


@pytest.mark.parametrize("mode", ["sequential", "batched", "joint"])
@pytest.mark.parametrize("world", [1, 2, 3])
def test_restore_recording_hands_segment_s_its_seed(monkeypatch, mode, world):
    import torch.distributed as dist
    from babe_b200 import distributed as bd, segments
    seed, seg_len, L = 2024, 4096, 30000
    n_seg = len(segments.segment_spans(L, seg_len))
    x = torch.randn(1, L)
    seen = {}
    for rank in range(world):
        monkeypatch.setattr(dist, "is_initialized", lambda: True)
        monkeypatch.setattr(dist, "get_rank", lambda rank=rank: rank)
        monkeypatch.setattr(dist, "get_world_size", lambda: world)
        # this rank's rows, zero padded to the whole recording's: what the gathers would return
        monkeypatch.setattr(bd, "gather_rows", lambda t: torch.cat((t, t.new_zeros((n_seg - t.shape[0],) + t.shape[1:]))))
        s = _SeedRecorder()
        segments.restore_recording(s, x, seg_len, batched=mode == "batched", joint=mode == "joint", seed=seed)
        assert s.row_seeds is None                           # restored after the call
        lo, hi = bd.shard_rows(n_seg, rank, world)
        got = [v for _, seeds in s.calls for v in seeds]
        assert len(s.calls) == (hi - lo if mode == "sequential" else 1)
        assert got == [segments.row_seed(seed, k) for k in range(lo, hi)]
        for k, v in zip(range(lo, hi), got):
            seen[k] = v
    assert sorted(seen) == list(range(n_seg))
    # without a seed the sampler's own noise source is left alone
    monkeypatch.setattr(dist, "is_initialized", lambda: False)
    s = _SeedRecorder()
    segments.restore_recording(s, x, seg_len, batched=mode == "batched", joint=mode == "joint")
    assert all(seeds is None for _, seeds in s.calls)


def test_restore_recording_ar_seeds():
    from babe_b200 import segments
    sr, segL, ov_s, L, seed = 1000, 400, 0.05, 1730, 77
    degraded = torch.randn(1, L, generator=torch.Generator().manual_seed(3))
    s = _SeedRecorder()
    segments.restore_recording_ar(s, degraded.clone(), segL, sr, overlap_s=ov_s, n_segments_blindstep=2,
                                  rng=np.random.RandomState(0), seed=seed)
    kinds = [c[0] for c in s.calls]
    assert kinds == ["blind", "bwe"] + ["ar"] * 9
    assert s.calls[0][1] == [segments.row_seed(seed, 2 ** 32 + j) for j in range(2)]
    assert [c[1] for c in s.calls[1:]] == [[segments.row_seed(seed, w)] for w in range(10)]
    assert s.row_seeds is None
