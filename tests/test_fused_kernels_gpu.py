"""GPU: the NFFT-4096 second-generation kernels of babe_b200/csrc/stft_fused.cu -- k_filter_fused (shared and per-row
filters, every epilogue), k_stats_fused and k_fir_fused -- against the fp64 oracle (oracle/stft_filter.py,
oracle/fir.py) at the batch shapes where their work partition matters, and the misaligned inputs that must take the
round-1 kernels of stft_ops.cu instead.

Work partition (restated below from stft_fused.cu): the B * units output blocks (filter), frames (statistics) or
block pairs (FIR) of a batch are cut into equal runs of q units, one run per CTA, over at most two CTAs per SM.  A run
can start inside a row and cross row boundaries, partial sums go to slot CTA + row, and the per-row filter kernel
redesigns H whenever its run enters a new row.  Each test case names a shape class; the shape that serves it is picked
by a classifier from this GPU's SM count, and test_shape_classes_covered fails if some class has no shape, so a
different SM count cannot drop a class silently.

Path check: torch.profiler with CUDA activity (CUPTI) lists the kernels each case launched (tests/kernel_trace.py);
every case asserts that the kernel generation it means to test ran and the other did not.

Error measures against the fp64 oracle, run on the same fp32 inputs with H designed in fp64 from the same (fc, A):
- per row: relative L2 <= TOL = 1e-5, the project's tolerance;
- per 2048-sample output block: the block's RMS error over its row's RMS <= BLOCK_TOL, so that one wrong block at a
  run seam in one row of a large batch cannot hide in a norm over the batch.
"""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from kernel_trace import assert_path, filter_variants, launched, uses

NFFT, HOP, SR = 4096, 2048, 22050
TOL = 1e-5
# Per-block bound.  A correct kernel's block errors are rounding noise.  Measured on a B200: the q = 1 cases (one block
# per CTA, no seams) stay below 5.1e-7 of the row's RMS, a block of a few samples (the 4-sample tail of T = 2052)
# below 2e-6, and rows of 4 samples, whose one block error is their row error, below 5.2e-6.  A lost carry, a frame
# missing at the start of a run or another row's filter in a block is an error of order 1e-2..1, so the bound is the
# row tolerance itself.
BLOCK_TOL = 1e-5

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _built():
    from babe_b200 import build
    build.build()


# --------------------------------------------------------------------------- work partition, restated
def _ctas():
    from babe_b200._lib import lib
    return 2 * lib().babe_sm_count()


def filter_units(T):
    return (T - 1) // HOP + 1                              # output blocks per row (fused_run_length)


def stats_units(T):
    return 1 + T // HOP                                    # frames per row (stats_run_length)


def fir_units(T, L):
    V = NFFT - L + 1
    return (-(-T // V) + 1) // 2                           # block pairs per row (launch_fir_fused)


def run_length(B, units, ctas, odd=False):
    q = max(1, -(-(B * units) // ctas))
    return q | 1 if odd else q


def classify(B, units, q):
    """The partition facts of B rows of `units` units cut into runs of q."""
    total = B * units
    grid = -(-total // q)
    starts = np.arange(grid, dtype=np.int64) * q
    ends = np.minimum(starts + q, total) - 1
    rows = ends // units - starts // units
    return dict(q=q, grid=grid, inside=bool((starts % units != 0).any()), cross1=bool((rows == 1).any()),
                span3=bool((rows >= 2).any()), partial=bool(total % q != 0))


def classes(facts):
    """q1: one unit per CTA.  aligned: runs of q > 1 units that start inside rows but never cross a row boundary.
    inside: some run of q > 1 starts inside a row (it costs one extra frame).  cross1 / span3: some run crosses one
    row boundary / spans three or more rows.  partial: the last run is shorter than q > 1."""
    if facts["q"] == 1:
        return {"q1"}
    c = {k for k in ("inside", "cross1", "span3", "partial") if facts[k]}
    if not (facts["cross1"] or facts["span3"]):
        c.add("aligned")
    return c


PART_CLASSES = ["q1", "aligned", "cross1", "span3"]
ALL_CLASSES = PART_CLASSES + ["inside", "partial"]
# candidates in order of preference (the first that shows a class serves it); at 148 SMs: q = 1 (3, 4096); aligned
# (8, 184184), q = 3; cross1 (3, 10^6), q = 5; span3 (1000, 2048), q = 5
POOL = [(3, 4096), (4, 30012), (8, 184184), (3, 1_000_000), (37, 184184), (64, 184184), (1000, 2048), (300, 4096),
        (512, 16384), (1, 1_000_000), (2, 1_000_000), (16, 184184), (2000, 2048), (6, 184184)]
# the benchmark's batch (q = 21, runs cross rows), one long row cut into many runs, and the row-length tails: shorter
# than one frame, exact multiples of the hop, hop + 4; B = 300 puts several of the short rows into one run
EXTRA = {"bench": (64, 184184), "row1e6": (1, 1_000_000),
         **{f"T{T}": (300, T) for T in (4, 8, 2048, 2052, 4096, 6144)}}
CASES = PART_CLASSES + list(EXTRA)


def pick(cls, units_of, odd):
    if cls in EXTRA:
        return EXTRA[cls]
    ctas = _ctas()
    for B, T in POOL:
        if cls in classes(classify(B, units_of(T), run_length(B, units_of(T), ctas, odd))):
            return B, T
    pytest.fail(f"no shape in the pool shows partition class {cls!r} at {ctas} CTAs")


def filter_shape(cls):
    return pick(cls, filter_units, odd=True)


def stats_shape(cls):
    return pick(cls, stats_units, odd=False)


def test_shape_classes_covered():
    ctas = _ctas()
    print(f"\npartition classes at {ctas // 2} SMs:")
    for name, units_of, odd in (("filter", filter_units, True), ("stats", stats_units, False)):
        seen = set()
        for cls in CASES:
            B, T = pick(cls, units_of, odd)
            f = classify(B, units_of(T), run_length(B, units_of(T), ctas, odd))
            print(f"  {name:6s} {cls:8s} B={B:5d} T={T:8d} {sorted(classes(f))} q={f['q']} grid={f['grid']}")
            seen |= classes(f)
        assert seen >= set(ALL_CLASSES), (name, set(ALL_CLASSES) - seen)
    # FIR: q > 1 with runs that cross rows, q = 1, and rows whose last pair is partial
    facts = [classify(B, fir_units(T, L), run_length(B, fir_units(T, L), ctas)) for B, T in FIR_SHAPES for L in (500, 499)]
    for (B, T), f in zip([s for s in FIR_SHAPES for _ in (0, 1)], facts):
        print(f"  fir    B={B:5d} T={T:8d} {sorted(classes(f))} q={f['q']} grid={f['grid']}")
    seen = set().union(*(classes(f) for f in facts))
    assert seen >= {"q1", "cross1", "span3"}, seen
    assert any(-(-T // (NFFT - L + 1)) % 2 == 1 for _, T in FIR_SHAPES for L in (500, 499))


# --------------------------------------------------------------------------- inputs, oracle, error measures
def signals(B, T, seed, n=1):
    """n (B, T) signals with a different level in every row (so that a row's data or sum in another row's place
    shows)."""
    g = torch.Generator().manual_seed(seed)
    gain = 0.063 * torch.linspace(0.3, 3.0, B)[:, None]
    return [torch.randn(B, T, generator=g) * gain for _ in range(n)]


def freqs():
    return torch.fft.rfftfreq(NFFT, d=1 / SR)              # float32: the kernel and the oracle see the same bins


# (fc, A) of the shared designs; no cutoff sits on a bin frequency, so fp32 and fp64 pick the same segment bins
DESIGNS = {
    "K1": ([1500.3], [-20.0]),
    "K5": ([310.7, 905.2, 2200.9, 4800.4, 8000.6], [-6.0, -12.0, -20.0, -28.0, -35.0]),
    "K16": (np.geomspace(203.1, 9001.7, 16).tolist(), np.linspace(-2.0, -30.0, 16).tolist()),
    "dup": ([700.3, 700.3, 1900.8, 1900.8, 5100.2], [-8.0, -15.0, -22.0, -30.0, -36.0]),
    "above": ([12000.0], [-20.0]),                         # fc_0 above the last bin: H = 1
}


def design64(fc, A):
    from oracle import stft_filter as sf
    return sf.design_filter(torch.tensor(fc, dtype=torch.float32).double(),
                            torch.tensor(A, dtype=torch.float32).double(), freqs().double())


def oracle(x, H, adjoint=False):
    from oracle import stft_filter as sf
    x = x.double()
    return sf.apply_filter_adjoint(x, H, NFFT) if adjoint else sf.apply_filter(x, H, NFFT)


def check(y, ref, what, tol=TOL, block_tol=BLOCK_TOL):
    """Per-row relative L2 and per-block (row-RMS-scaled) errors of y against the fp64 ref; returns their maxima."""
    y = y.detach().cpu().double()
    ref = ref.double()
    assert y.shape == ref.shape, what
    B, T = ref.shape
    d = y - ref
    row = d.norm(dim=1) / ref.norm(dim=1)
    nb = -(-T // HOP)
    d2 = torch.nn.functional.pad(d * d, (0, nb * HOP - T)).view(B, nb, HOP).sum(-1)
    n = torch.full((nb,), float(HOP), dtype=torch.float64)
    n[-1] = T - (nb - 1) * HOP
    blk = (d2 / n).sqrt() / (ref * ref).mean(1).sqrt()[:, None]
    r, (br, bb) = int(row.argmax()), divmod(int(blk.argmax()), nb)
    assert float(row[r]) <= tol, f"{what}: row {r} relative L2 {float(row[r]):.3e}"
    assert float(blk[br, bb]) <= block_tol, f"{what}: row {br} block {bb} error {float(blk[br, bb]):.3e} of the row RMS"
    ERRORS[what] = (float(row.max()), float(blk.max()))
    return float(row.max()), float(blk.max())


ERRORS = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nerrors against the fp64 oracle (largest row relative L2, largest block error / row RMS):")
    for k, (r, b) in ERRORS.items():
        print(f"  {k:52s} {r:.2e}  {b:.2e}")


def cuda(t):
    return t.contiguous().cuda()


# --------------------------------------------------------------------------- 1. apply_filter, shared filter
@pytest.mark.parametrize("cls", CASES)
def test_apply_filter_shared_vs_oracle(cls):
    from babe_b200 import ops
    B, T = filter_shape(cls)
    (x,) = signals(B, T, seed=B + T)
    xc, f = cuda(x), cuda(freqs())
    H64 = {name: design64(*p) for name, p in DESIGNS.items()}
    Hgiven = H64["K5"].float()
    out = {}
    with launched() as names:
        for adj in (False, True):
            out["H", adj] = ops.apply_filter(xc, NFFT, H=cuda(Hgiven), adjoint=adj)
            for name, (fc, A) in DESIGNS.items():
                out[name, adj] = ops.apply_filter(xc, NFFT, freqs=f, fc=cuda(torch.tensor(fc)),
                                                  A=cuda(torch.tensor(A)), adjoint=adj)
    assert_path(names, fused=True, kernel="k_filter_fused")
    assert filter_variants(names) == {(False, 0, False), (True, 0, False)}
    for (name, adj), y in out.items():
        H = Hgiven.double() if name == "H" else H64[name]
        check(y, oracle(x, H, adj), f"apply_filter {'adj' if adj else 'fwd'}: {cls} {name}")


# --------------------------------------------------------------------------- 2. epilogues
EPILOGUES = {
    # name: (adjoint, sub, scale, sumsq, the instantiation launch_variant picks)
    "fwd_sub_sumsq": (False, True, False, True, 1),
    "adj_scale": (True, False, True, False, 2),
    "fwd_scale": (False, False, True, False, 3),
    "fwd_sub": (False, True, False, False, 3),
    "fwd_sumsq": (False, False, False, True, 3),
    "fwd_sub_scale_sumsq": (False, True, True, True, 3),
    "adj_sumsq": (True, False, False, True, 3),
    "adj_scale_sumsq": (True, False, True, True, 3),
}


@pytest.mark.parametrize("cls", ["cross1", "q1", "span3"])
def test_epilogues_vs_oracle(cls):
    """Every branch of launch_variant: y = (A x - sub) * scale (forward) or A^T x * scale (adjoint), and
    row_sumsq += sum_t y^2 per row, against the fp64 oracle."""
    from babe_b200 import ops
    B, T = filter_shape(cls)
    x, sub = signals(B, T, seed=7 + B, n=2)
    fc, A = DESIGNS["K5"]
    H = design64(fc, A)
    kw = dict(freqs=cuda(freqs()), fc=cuda(torch.tensor(fc)), A=cuda(torch.tensor(A)))
    scale = torch.linspace(0.5, 2.0, B)
    fwd, adj = oracle(x, H), oracle(x, H, True)
    for name, (is_adj, has_sub, has_scale, has_ss, epi) in EPILOGUES.items():
        ref = adj if is_adj else fwd
        if has_sub:
            ref = ref - sub.double()
        if has_scale:
            ref = ref * scale.double()[:, None]
        # row_sumsq accumulates: it starts at values of the order of the row sums
        ss0 = (ref * ref).sum(1) * torch.linspace(0.5, 1.5, B, dtype=torch.float64)
        ss = cuda(ss0) if has_ss else None
        with launched() as names:
            y = ops.apply_filter(cuda(x), NFFT, adjoint=is_adj, sub=cuda(sub) if has_sub else None,
                                 row_scale=cuda(scale) if has_scale else None, row_sumsq=ss, **kw)
        assert_path(names, fused=True, kernel="k_filter_fused")
        assert filter_variants(names) == {(is_adj, epi, False)}, (name, names)
        check(y, ref, f"epilogue {name}: {cls}")
        if has_ss:
            # the residual's sum of squares: fp32 squares summed in fp32 per thread and frame pair, in fp64 above
            # that, of outputs within 1e-6 of the oracle's -> 1e-5 relative per row
            got = ss.cpu() - ss0
            want = (ref * ref).sum(1)
            err = ((got - want).abs() / want)
            assert float(err.max()) < 1e-5, (name, int(err.argmax()), float(err.max()))
    # sub is ignored by the adjoint (stft_ops.cu babe_apply_filter / babe_apply_filter_rows)
    plain = ops.apply_filter(cuda(x), NFFT, adjoint=True, **kw)
    with launched() as names:
        with_sub = ops.apply_filter(cuda(x), NFFT, adjoint=True, sub=cuda(sub), **kw)
    assert filter_variants(names) == {(True, 0, False)}
    assert torch.equal(with_sub, plain)
    scaled = ops.apply_filter(cuda(x), NFFT, adjoint=True, row_scale=cuda(scale), **kw)
    assert torch.equal(ops.apply_filter(cuda(x), NFFT, adjoint=True, row_scale=cuda(scale), sub=cuda(sub), **kw), scaled)


# --------------------------------------------------------------------------- 3. apply_filter_rows
def row_bank(B, K=5, n=7):
    """n widely different filters (cutoffs 300 Hz .. 10 kHz, slopes -5 .. -57 dB/oct); row b takes filter b % n, so
    neighbouring rows -- and the rows one run spans -- never share one."""
    fc0 = np.geomspace(300.7, 4500.3, n)
    fcs = np.stack([fc0 * (1.0 + 0.3 * k) for k in range(K)], 1)
    As = np.stack([np.linspace(-5.0, -45.0, n) - 3.0 * k for k in range(K)], 1)
    idx = np.arange(B) % n
    return torch.tensor(fcs[idx], dtype=torch.float32), torch.tensor(As[idx], dtype=torch.float32), fcs, As


def rows_oracle(x, fcs, As, adjoint=False):
    """Each row through the fp64 oracle with its own filter (rows grouped by filter)."""
    out = torch.empty(x.shape, dtype=torch.float64)
    n = len(fcs)
    for i in range(min(n, x.shape[0])):
        sel = torch.arange(i, x.shape[0], n)
        out[sel] = oracle(x[sel], design64(fcs[i].tolist(), As[i].tolist()), adjoint)
    return out


@pytest.mark.parametrize("cls", CASES)
def test_apply_filter_rows_vs_oracle(cls):
    from babe_b200 import ops
    B, T = filter_shape(cls)
    x, sub = signals(B, T, seed=11 + T, n=2)
    fc, A, fcs, As = row_bank(B)
    f = cuda(freqs())
    scale = torch.linspace(0.5, 2.0, B)
    ss = torch.zeros(B, dtype=torch.float64, device="cuda")
    with launched() as names:
        y = ops.apply_filter_rows(cuda(x), NFFT, f, cuda(fc), cuda(A))
        ya = ops.apply_filter_rows(cuda(x), NFFT, f, cuda(fc), cuda(A), adjoint=True)
        r = ops.apply_filter_rows(cuda(x), NFFT, f, cuda(fc), cuda(A), sub=cuda(sub), row_sumsq=ss)
        g = ops.apply_filter_rows(cuda(x), NFFT, f, cuda(fc), cuda(A), adjoint=True, row_scale=cuda(scale))
    assert_path(names, fused=True, kernel="k_filter_fused")
    assert filter_variants(names) == {(False, 0, True), (True, 0, True), (False, 1, True), (True, 2, True)}
    fwd, adj = rows_oracle(x, fcs, As), rows_oracle(x, fcs, As, True)
    check(y, fwd, f"apply_filter_rows fwd: {cls}")
    check(ya, adj, f"apply_filter_rows adj: {cls}")
    res = fwd - sub.double()
    check(r, res, f"apply_filter_rows residual: {cls}")
    err = (ss.cpu() - (res * res).sum(1)).abs() / (res * res).sum(1)
    assert float(err.max()) < 1e-5, (int(err.argmax()), float(err.max()))
    check(g, adj * scale.double()[:, None], f"apply_filter_rows adj scaled: {cls}")


def test_apply_filter_rows_status_inside_a_run():
    """A row whose design the reference rejects (fc_1 above the last bin) is flagged by itself when it is not the
    first row of its CTA's run, and its neighbours in the run keep their own filters."""
    from babe_b200 import ops
    B, T = filter_shape("span3")
    units = filter_units(T)
    q = run_length(B, units, _ctas(), odd=True)
    # a row that starts inside a run that began in an earlier row, and whose run goes on into the next row
    bad = next(r for r in range(1, B - 1) if (r * units) % q and ((r + 1) * units) // q == (r * units) // q)
    x, = signals(B, T, seed=5)
    fc, A, fcs, As = row_bank(B)
    fc[bad] = torch.tensor([400.0, 20000.0, 20001.0, 20002.0, 20003.0])
    status = torch.zeros(B, dtype=torch.int32, device="cuda")
    with launched() as names:
        y = ops.apply_filter_rows(cuda(x), NFFT, cuda(freqs()), cuda(fc), cuda(A), status=status)
    assert_path(names, fused=True, kernel="k_filter_fused")
    flagged = torch.nonzero(status.cpu()).reshape(-1).tolist()
    assert flagged == [bad], (bad, q, flagged)
    keep = torch.tensor([b for b in range(B) if b != bad])
    ref = rows_oracle(x, fcs, As)
    check(y.cpu()[keep], ref[keep], "apply_filter_rows status: span3")


# --------------------------------------------------------------------------- 4. statistics
def mags(x):
    from oracle import stft_filter as sf
    X = sf.apply_stft(x.double(), NFFT)
    return torch.sqrt(X[..., 0] ** 2 + X[..., 1] ** 2)      # (B, F, frames)


@pytest.mark.parametrize("cls", CASES)
def test_stft_stats_vs_oracle(cls):
    from babe_b200 import ops
    from oracle import stft_filter as sf
    B, T = stats_shape(cls)
    x, y = signals(B, T, seed=3 + T, n=2)
    with launched() as names:
        abc = ops.stft_stats(cuda(x), cuda(y), NFFT).cpu()
        rows = ops.stft_stats_rows(cuda(x), cuda(y), NFFT).cpu()
    assert_path(names, fused=True, kernel="k_stats_fused")
    a, b, c = sf.stft_mag_stats(x.double(), y.double(), NFFT)
    for i, ref in enumerate((a, b, c)):
        assert rel_l2(abc[i], ref) < TOL, (cls, i, rel_l2(abc[i], ref))
    mx, my = mags(x), mags(y)
    per_row = torch.stack(((mx * mx).sum(2), (mx * my).sum(2), (my * my).sum(2)), 1)     # (B, 3, F)
    err = (rows - per_row).norm(dim=2) / per_row.norm(dim=2)
    assert float(err.max()) < TOL, (cls, divmod(int(err.argmax()), 3), float(err.max()))
    ERRORS[f"stft_stats_rows: {cls}"] = (float(err.max()), float("nan"))


def test_stft_stats_mode1_vs_oracle():
    """Mode 1 (the filter-gradient cross term sum Re(conj(X) STFT(y / envelope)), row 0) at T % 4 == 0: there is no
    fused kernel for it, the round-1 kernel runs."""
    from babe_b200 import ops
    from oracle import stft_filter as sf
    B, T = filter_shape("cross1")
    x, n = signals(B, T, seed=9, n=2)
    y = 0.7 * x + 0.3 * n
    with launched() as names:
        got = ops.stft_stats(cuda(x), cuda(y), NFFT, mode=1)[0].cpu()
    assert_path(names, fused=False, kernel="k_stft_stats")
    M = sf.num_frames(T, NFFT)
    env = sf.ola_envelope(M, NFFT)[:T]
    X = torch.view_as_complex(sf.apply_stft(x.double(), NFFT))
    G = torch.view_as_complex(sf.apply_stft(y.double() / env, NFFT))
    ref = (X.conj() * G).real.sum((0, 2))
    assert rel_l2(got, ref) < TOL, rel_l2(got, ref)


# --------------------------------------------------------------------------- 5. FIR
def fir_ref(x, taps, adjoint=False):
    """apply_fir_same / apply_fir_same_adjoint of oracle/fir.py as an fp64 FFT convolution (the direct sums cost
    B T L operations; test_fir_ref_is_the_oracle pins the two together)."""
    b = np.asarray(taps, dtype=np.float64).reshape(-1)
    L = b.size
    pl = (L - 1) // 2
    if adjoint:
        b, pl = b[::-1], L - 1 - pl
    x = np.asarray(x, dtype=np.float64)
    T = x.shape[1]
    n = 1 << int(np.ceil(np.log2(T + L - 1)))
    full = np.fft.irfft(np.fft.rfft(x, n, axis=1) * np.fft.rfft(b[::-1], n), n, axis=1)
    return torch.from_numpy(full[:, L - 1 - pl:L - 1 - pl + T].copy())


@pytest.mark.parametrize("L", [500, 499, 31])
def test_fir_ref_is_the_oracle(L):
    """CPU only: the FFT form of the FIR oracle equals its direct sums."""
    from oracle import fir
    g = torch.Generator().manual_seed(L)
    x, taps = torch.randn(3, 9000, generator=g, dtype=torch.float64), torch.randn(L, generator=g, dtype=torch.float64)
    assert rel_l2(fir_ref(x, taps), fir.apply_fir_same(x, taps)) < 1e-12
    assert rel_l2(fir_ref(x, taps, True), fir.apply_fir_same_adjoint(x, taps)) < 1e-12


# q > 1 with runs across rows (64 x 184184: 26 pairs per row, q = 6); rows of 3 blocks, whose second pair is partial;
# one block pair per row, several rows per run; q = 1
FIR_SHAPES = [(64, 184184), (300, 10788), (1000, 2048), (3, 8192)]


def fir_taps(golden):
    g = golden("fir.npz")
    short = torch.tensor([0.05, -0.1, 0.2, 0.7, 0.2, -0.1, 0.05, 0.01, -0.02], dtype=torch.float32)   # 9 taps
    return {"lpf500": torch.from_numpy(g["taps_lpf500"]).float().reshape(-1),
            "hpf499": torch.from_numpy(g["taps_hpf499"]).float().reshape(-1), "short9": short}


@pytest.mark.parametrize("B,T", FIR_SHAPES)
def test_fir_filter_vs_oracle(golden, B, T):
    from babe_b200 import ops
    x, = signals(B, T, seed=T)
    for name, taps in fir_taps(golden).items():
        with launched() as names:
            y = ops.fir_filter(cuda(x), cuda(taps))
            ya = ops.fir_filter(cuda(x), cuda(taps), adjoint=True)
        assert_path(names, fused=True, kernel="k_fir_fused")
        check(y, fir_ref(x, taps), f"fir_filter fwd: {B}x{T} {name}")
        check(ya, fir_ref(x, taps, True), f"fir_filter adj: {B}x{T} {name}")


# --------------------------------------------------------------------------- 6. alignment
def offset_view(t, off):
    """t's values in a contiguous view that starts `off` floats past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 8, dtype=torch.float32, device="cuda")
    v = buf[off:off + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4 * off
    return v


@pytest.fixture
def round1():
    """Runs its callable with the NFFT-4096 entry points switched to the round-1 kernels; the knob is restored
    whatever happens."""
    from babe_b200._lib import lib

    def run(fn):
        assert lib().babe_set_fused_variant(-1) == 0
        try:
            return fn()
        finally:
            lib().babe_set_fused_variant(0)
    return run


@pytest.mark.parametrize("off", [1, 2, 3])
def test_misaligned_inputs_take_round1(round1, off):
    """Rows with T % 4 == 0 but a base that is not 16-byte aligned (e.g. a slice at an odd sample of a longer
    recording) cannot be bulk-copied: every entry point must take the round-1 kernel, meet the oracle, and agree with
    the aligned call under babe_set_fused_variant(-1)."""
    from babe_b200 import ops
    from oracle import stft_filter as sf
    B, T = 6, 30012
    x, sub = signals(B, T, seed=off, n=2)
    fc5, A5 = DESIGNS["K5"]
    H = design64(fc5, A5)
    f, fcc, Ac = cuda(freqs()), cuda(torch.tensor(fc5)), cuda(torch.tensor(A5))
    rfc, rA, fcs, As = row_bank(B)
    taps = torch.from_numpy(np.hanning(501)[1:-1] / np.hanning(501).sum()).float()     # 499 taps
    c = torch.linspace(0.5, 1.5, NFFT // 2 + 1)
    M = sf.num_frames(T, NFFT)
    xv, subv = offset_view(x, off), offset_view(sub, off)
    xa, suba = cuda(x), cuda(sub)
    X = sf.apply_stft(x.double(), NFFT).float()
    Xv = offset_view(X, off)
    env = sf.ola_envelope(M, NFFT)[:T]

    def ss():
        return torch.zeros(B, dtype=torch.float64, device="cuda")

    res64 = oracle(x, H) - sub.double()
    # name: (call on (x, sub, X) views, fp64 reference or None, reference as rows of y)
    cases = {
        "filter_fwd_x": (lambda x_, s_, X_: ops.apply_filter(x_, NFFT, freqs=f, fc=fcc, A=Ac), oracle(x, H)),
        "filter_adj_x": (lambda x_, s_, X_: ops.apply_filter(x_, NFFT, H=cuda(H.float()), adjoint=True),
                         oracle(x, H.float().double(), True)),
        "filter_res_sub": (lambda x_, s_, X_: ops.apply_filter(xa, NFFT, freqs=f, fc=fcc, A=Ac, sub=s_,
                                                               row_sumsq=ss()), res64),
        "rows_fwd_x": (lambda x_, s_, X_: ops.apply_filter_rows(x_, NFFT, f, cuda(rfc), cuda(rA)),
                       rows_oracle(x, fcs, As)),
        "rows_res_sub": (lambda x_, s_, X_: ops.apply_filter_rows(xa, NFFT, f, cuda(rfc), cuda(rA), sub=s_),
                         rows_oracle(x, fcs, As) - sub.double()),
        "fir_fwd_x": (lambda x_, s_, X_: ops.fir_filter(x_, cuda(taps)), fir_ref(x, taps)),
        "fir_adj_x": (lambda x_, s_, X_: ops.fir_filter(x_, cuda(taps), adjoint=True), fir_ref(x, taps, True)),
    }
    for name, (fn, ref) in cases.items():
        with launched() as names:
            y = fn(xv, subv, Xv)
        assert_path(names, fused=False)
        check(y, ref, f"misaligned {name}: off {off}")
        aligned = round1(lambda: fn(xa, suba, cuda(X)))
        assert rel_l2(y.cpu(), aligned.cpu()) < 1e-6, (name, rel_l2(y.cpu(), aligned.cpu()))

    # statistics: x misaligned, then y alone
    a, b, cc = sf.stft_mag_stats(x.double(), sub.double(), NFFT)
    for name, (xx, yy) in {"stats_x": (xv, suba), "stats_y": (xa, subv)}.items():
        with launched() as names:
            abc = ops.stft_stats(xx, yy, NFFT).cpu()
            rows = ops.stft_stats_rows(xx, yy, NFFT).cpu()
        assert_path(names, fused=False, kernel="k_stft_stats")
        for i, ref in enumerate((a, b, cc)):
            assert rel_l2(abc[i], ref) < TOL, (name, i)
        assert rel_l2(rows.sum(0), abc) < TOL, name
        aligned = round1(lambda: (ops.stft_stats(xa, suba, NFFT).cpu(), ops.stft_stats_rows(xa, suba, NFFT).cpu()))
        assert rel_l2(abc, aligned[0]) < 1e-6 and rel_l2(rows, aligned[1]) < 1e-6, name

    # the standalone transforms (round-1 kernels only): STFT of y / envelope with a bin scale, over M frames, and
    # the iSTFT with a bin scale and no envelope division (the adjoint forms of blind_bwe_utils)
    with launched() as names:
        Xs = ops.stft(xv, NFFT, frames=M, in_env_div=True, bin_scale=cuda(c))
        ys = ops.istft(Xv, NFFT, out_len=T, bin_scale=cuda(c), out_env_div=False)
    assert not any(uses(names, k) for k in ("k_filter_fused", "k_stats_fused", "k_fir_fused"))
    assert uses(names, "k_stft") and uses(names, "k_istft")
    ref_X = sf.apply_stft(x.double() / env, NFFT) * c.double()[None, :, None, None]
    assert rel_l2(Xs.cpu(), ref_X) < TOL
    Xc = torch.view_as_complex(X.double().contiguous()) * c.double()[None, :, None]
    fr = torch.fft.irfft(Xc.transpose(1, 2), n=NFFT, dim=-1) * sf.hamming_periodic(NFFT, torch.float64)
    ref_y = torch.zeros(B, NFFT + HOP * (M - 1), dtype=torch.float64)
    for m in range(M):
        ref_y[:, m * HOP:m * HOP + NFFT] += fr[:, m]
    assert rel_l2(ys.cpu(), ref_y[:, :T]) < TOL
    al = round1(lambda: (ops.stft(xa, NFFT, frames=M, in_env_div=True, bin_scale=cuda(c)),
                         ops.istft(cuda(X), NFFT, out_len=T, bin_scale=cuda(c), out_env_div=False)))
    assert rel_l2(Xs.cpu(), al[0].cpu()) < 1e-6 and rel_l2(ys.cpu(), al[1].cpu()) < 1e-6


def test_misaligned_out_keeps_fused_kernel():
    """The fused filter kernel stores its output sample by sample, so `out` may start at any float: it keeps the
    fused path and its results."""
    from babe_b200 import ops
    B, T = filter_shape("cross1")
    x, = signals(B, T, seed=21)
    fc, A = DESIGNS["K5"]
    kw = dict(freqs=cuda(freqs()), fc=cuda(torch.tensor(fc)), A=cuda(torch.tensor(A)))
    ref = ops.apply_filter(cuda(x), NFFT, **kw)
    out = offset_view(torch.zeros(B, T), 1)
    with launched() as names:
        y = ops.apply_filter(cuda(x), NFFT, out=out, **kw)
    assert y is out
    assert_path(names, fused=True, kernel="k_filter_fused")
    assert torch.equal(out, ref)


# --------------------------------------------------------------------------- out= validation
@pytest.mark.parametrize("rows", [False, True])
def test_out_is_validated_before_launch(rows):
    """A wrong `out` raises ValueError before anything runs: the kernels write B * T floats from its base pointer.
    Each bad `out` here lies inside a larger sentinel buffer, so that a write past it would show."""
    from babe_b200 import ops
    B, T = 3, 8192
    x, = signals(B, T, seed=1)
    fc, A = DESIGNS["K5"]
    f = cuda(freqs())
    if rows:
        rfc, rA, _, _ = row_bank(B)
        call = lambda out: ops.apply_filter_rows(cuda(x), NFFT, f, cuda(rfc), cuda(rA), out=out)    # noqa: E731
    else:
        call = lambda out: ops.apply_filter(cuda(x), NFFT, freqs=f, fc=cuda(torch.tensor(fc)),    # noqa: E731
                                            A=cuda(torch.tensor(A)), out=out)
    big = torch.full((2 * B * T + 64,), 7.0, device="cuda")
    bad = {
        "shape": big[:B * (T - 4)].view(B, T - 4),
        "dtype": big.view(torch.int32)[:B * T].view(B, T),
        "strided": big[:2 * B * T].view(B, 2 * T)[:, ::2],
        "cpu": torch.empty(B, T),
    }
    for name, out in bad.items():
        with launched() as names:
            with pytest.raises(ValueError):
                call(out)
        assert not any(uses(names, k) for k in ("k_filter_fused", "k_apply_filter")), (name, names)
        assert torch.all(big == 7.0), name
    good = big[:B * T].view(B, T)
    assert call(good) is good and torch.all(big[B * T:] == 7.0)
