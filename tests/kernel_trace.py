"""Which CUDA kernels a block of code launched, from the CUDA activity that ``torch.profiler`` records (CUPTI).

At NFFT 4096 the filter, statistics and FIR entry points run the second-generation kernels of
``babe_b200/csrc/stft_fused.cu`` when the rows can be bulk-copied and the round-1 kernels of ``stft_ops.cu``
otherwise, with the same results to rounding.  Only the kernel names tell the two paths apart, so the tests that mean
to exercise one of them assert it with::

    with launched() as names:
        ops.apply_filter(...)
    assert_path(names, fused=True)
"""
import contextlib

import torch

FUSED = ("k_filter_fused", "k_stats_fused", "k_fir_fused")
ROUND1 = ("k_apply_filter", "k_stft_stats", "k_fir_filter")


@contextlib.contextmanager
def launched():
    """Yields a list that holds, once the block has run, the names of the kernels it launched."""
    from torch.profiler import ProfilerActivity, profile
    names = []
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        yield names
        torch.cuda.synchronize()
    names.extend(e.name for e in prof.events())


def uses(names, kernel):
    return any(kernel in n for n in names)


def assert_path(names, fused, kernel=None):
    """fused=True: some second-generation kernel ran (``kernel`` if given) and no round-1 one; fused=False: the
    reverse."""
    want, avoid = (FUSED, ROUND1) if fused else (ROUND1, FUSED)
    want = (kernel,) if kernel is not None else want
    assert any(uses(names, k) for k in want), f"expected one of {want}, launched {sorted(set(names))}"
    assert not any(uses(names, k) for k in avoid), f"expected none of {avoid}, launched {sorted(set(names))}"


def filter_variants(names):
    """(adjoint, epilogue, per_row) of every k_filter_fused instantiation that ran."""
    out = set()
    for n in names:
        i = n.find("k_filter_fused<")
        if i < 0:
            continue
        args = n[i + len("k_filter_fused<"):n.index(">", i)].split(",")
        flag = [a.strip().replace("(bool)", "") for a in args]
        out.add((flag[0] in ("true", "1"), int(flag[1].strip("()int ")), flag[2] in ("true", "1")))
    return out
