"""Long recordings as overlapped fixed-length segments (host orchestration).

Restates the non-autoregressive branch of ``BlindTester.formal_test_bwe``
(testing/blind_bwe_tester.py:413-577 of eloimoliner/BABE, ``use_AR: False``,
``OLA: 256`` in the formal configs) without soundfile / wandb: the recording is
cut into ``audio_len`` windows that advance by ``segL - discard_end - OLA``
samples, every window is restored by an independent sampler call (its own
filter estimate, :433,:477,:543) and the predictions are cross-faded with a
``2*OLA`` Hann window.  Segments are independent units, so they shard over
ranks with no data-path collective (SURVEY 8e); ``restore_recording`` gathers
predictions and per-segment filters with NCCL at the end.
"""
import contextlib

import torch

from . import distributed as bd

_MASK64 = (1 << 64) - 1
_GOLDEN64 = 0x9E3779B97F4A7C15


def row_seed(seed, k):
    """Seed of unit ``k`` (segment, window or row) of a run seeded with ``seed``: SplitMix64 of
    ``seed + (k + 1) * 0x9E3779B97F4A7C15`` (mod 2**64), i.e. output k of the SplitMix64 stream started at
    ``seed``.  An unsigned 64-bit int, for ``BlindSamplerFused.row_seeds``.  A pure function: every rank derives
    the seed of a unit from its global index alone."""
    z = (int(seed) + (int(k) + 1) * _GOLDEN64) & _MASK64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _MASK64
    return z ^ (z >> 31)


@contextlib.contextmanager
def _row_seeds(sampler, seeds):
    """Install ``row_seeds`` on the sampler for one call and restore the previous value afterwards
    (``seeds`` None: leave the sampler as it is)."""
    if seeds is None:
        yield
        return
    was = sampler.row_seeds
    sampler.row_seeds = list(seeds)
    try:
        yield
    finally:
        sampler.row_seeds = was


def segment_spans(L, seg_len, ola=256, discard_end=200, discard_start=0):
    """Start indices exactly as the while-loop at testing/blind_bwe_tester.py:469-521
    produces them; the last span is the incomplete tail (:526-533)."""
    step = seg_len - discard_end - ola
    spans, ix = [(0, seg_len)], step
    while ix < L - seg_len - discard_end - discard_start:
        spans.append((ix, ix + seg_len))
        ix += step
    spans.append((ix, ix + seg_len))          # tail, zero padded to seg_len
    return spans


def split(degraded, seg_len, ola=256, discard_end=200):
    """degraded (1, L) -> (segments (S, seg_len), spans)."""
    L = degraded.shape[-1]
    spans = segment_spans(L, seg_len, ola, discard_end)
    segs = degraded.new_zeros((len(spans), seg_len))
    for s, (a, b) in enumerate(spans):
        piece = degraded[0, a:min(b, L)]
        segs[s, :piece.shape[-1]] = piece
    return segs, spans


def merge(preds, spans, L, ola=256, discard_end=200):
    """Cross-fade of the per-segment predictions (:455-461, :493-499, :565-568)."""
    seg_len = preds.shape[-1]
    hann = torch.hann_window(ola * 2, device=preds.device)
    out = preds.new_zeros((1, L))
    last = len(spans) - 1
    for s, (a, _) in enumerate(spans):
        if s == last:
            n = L - a
            w = preds[s, :n].clone()
            w[:ola] *= hann[:ola]
            out[0, a:] += w
            continue
        w = preds[s, :seg_len - discard_end].clone()
        if s > 0:
            w[:ola] *= hann[:ola]
        w[-ola:] *= hann[ola:]
        out[0, a:a + seg_len - discard_end] += w
    return out


def restore_recording(sampler, degraded, seg_len, ola=256, discard_end=200, joint=False, batched=False, seed=None):
    """Blind restoration of a whole recording, segments sharded over the ranks of the
    current process group.  Returns (final_pred (1, L), filter_data) on every rank,
    ``filter_data`` being the list [((ix0, ix1), filter_params), ...] the reference
    pickles (:466-467,:576-577).  ``joint=True`` processes a rank's segments as one
    batch and shares ONE filter across all ranks (testing/blind_bwe_tester.py:758-781).

    ``batched=True`` (with ``joint=False``) restores a rank's segments in ONE sampler call with
    ``filter_per_row``: every segment still gets its own filter estimate and guidance scale, as in
    the sequential loop, but the denoiser and the filter kernels run on all of them at once.  The
    noise is drawn for the whole batch at each step, so the host noise stream is consumed in a
    different order than by the loop of B = 1 calls: the two restorations agree statistically,
    not bitwise (they agree to rounding when every segment gets the same noise either way, e.g.
    through ``sampler.noise_fn``).

    ``seed`` (an int) switches the sampler to keyed per-row noise: segment s, counted over the whole
    recording, draws with ``row_seed(seed, s)`` in all three modes, so the noise each segment sees
    depends neither on the mode nor on how the segments are sharded over ranks (the sequential and
    batched restorations then agree to the rounding of the per-row kernels).  ``seed=None`` keeps the
    sampler's own noise source."""
    import torch.distributed as dist
    if joint and batched:
        raise ValueError("batched=True restores every segment with its own filter; joint=True shares one")
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    segs, spans = split(degraded, seg_len, ola, discard_end)
    if world > segs.shape[0]:
        raise ValueError(f"{world} ranks for {segs.shape[0]} segments: every rank needs at least one segment "
                         "(an empty shard would enter the NCCL gathers with a different shape)")
    lo, hi = bd.shard_rows(segs.shape[0], rank, world)
    mine = segs[lo:hi]
    seeds = None if seed is None else [row_seed(seed, k) for k in range(lo, hi)]
    if joint:
        sampler.joint = True
        with _row_seeds(sampler, seeds):
            pred, filt = sampler.predict_blind_bwe(mine, rid=False)
        filts = filt.unsqueeze(0).expand(mine.shape[0], -1, -1).contiguous()
    elif batched:
        was = sampler.filter_per_row
        sampler.filter_per_row = True
        try:
            with _row_seeds(sampler, seeds):
                pred, filts = sampler.predict_blind_bwe(mine.clone(), rid=False)
        finally:
            sampler.filter_per_row = was
    else:
        preds, fl = [], []
        for s in range(mine.shape[0]):
            with _row_seeds(sampler, None if seeds is None else seeds[s:s + 1]):
                p, f = sampler.predict_blind_bwe(mine[s:s + 1].clone(), rid=False)
            preds.append(p)
            fl.append(f)
        pred = torch.cat(preds, 0) if preds else mine.new_zeros((0, seg_len))
        filts = torch.stack(fl, 0) if fl else mine.new_zeros((0, 2, 1))
    all_pred = bd.gather_rows(pred)
    all_filt = bd.gather_rows(filts)
    final = merge(all_pred, spans, degraded.shape[-1], ola, discard_end)
    return final, [(spans[s], all_filt[s]) for s in range(len(spans))]


def restore_recording_ar(sampler, degraded, seg_len, sample_rate, overlap_s=0.25, n_segments_blindstep=2,
                         ix_start_s=0, std=0.1, typefilter="fc_A", discard_end=200, discard_start=0,
                         rng=None, estimated_filter=None, seed=None):
    """Autoregressive restoration of a whole recording with ONE filter estimated once:
    ``BlindTester.test_real_blind_bwe_complete`` (testing/blind_bwe_tester.py:710-867) without file
    I/O, resampling and wandb.

    1. the recording is normalised to ``std`` (:746-747);
    2. blind step on ``n_segments_blindstep`` randomly placed windows (:757-777) -> filter estimate
       (skipped when ``estimated_filter`` is given);
    3. first window with ``predict_bwe`` (:799-805), then windows advancing by
       ``seg_len - overlap - discard_end`` samples with ``predict_bwe_AR``: the first ``overlap`` samples of
       each window are known from the previous prediction (mask = 1 there, :807-838);
    4. last, zero padded window (:841-859), scale restored (:861).

    Sequential by construction (each window needs the previous prediction): replicas only across
    recordings (SURVEY 8e).  ``degraded``: (1, L) tensor on the sampler's device.  Returns
    (restored (1, L), filter (2, K)).

    ``seed`` (an int) switches the sampler to keyed per-row noise: window w draws with ``row_seed(seed, w)``
    (w = 0 is the first ``predict_bwe`` window, then the autoregressive windows, then the padded last one) and
    row j of the blind step with ``row_seed(seed, 2**32 + j)``, so the restoration is a function of the
    recording and the seed alone.  ``seed=None`` keeps the sampler's own noise source."""
    import numpy as np
    segL = int(seg_len)
    L = degraded.shape[-1]
    scale = degraded.std(-1)
    degraded = std * degraded / scale.unsqueeze(-1)
    ix_first = int(sample_rate * ix_start_s)
    final = torch.zeros_like(degraded)
    if estimated_filter is None:
        if n_segments_blindstep == 1:
            y = degraded[..., ix_first:ix_first + segL]
        else:
            rng = rng if rng is not None else np.random
            y = degraded[..., ix_first:ix_first + segL].repeat(n_segments_blindstep, 1)
            for j in range(n_segments_blindstep):
                ix = int(rng.randint(0, L - segL))
                y[j] = degraded[0, ix:ix + segL]
        blind = None if seed is None else [row_seed(seed, (1 << 32) + j) for j in range(y.shape[0])]
        with _row_seeds(sampler, blind):
            pred, estimated_filter = sampler.predict_blind_bwe(y, rid=False)
        final[0, ix_first:ix_first + segL] = pred[0]
    overlap = int(overlap_s * sample_rate)
    keep = segL - discard_end
    ix = 0
    window = [0]

    def keyed():                                             # the seeds of the next window
        w = window[0]
        window[0] += 1
        return _row_seeds(sampler, None if seed is None else [row_seed(seed, w)])

    seg = degraded[..., ix:ix + segL]
    with keyed():
        pred = sampler.predict_bwe(seg, estimated_filter, typefilter, rid=False)
    previous = pred[..., :keep]
    final[..., ix:ix + keep] = previous
    ix += segL - overlap - discard_end
    y_masked = torch.zeros_like(pred)
    mask = torch.ones_like(seg)
    mask[..., overlap:] = 0
    # the reference stops at ix >= L - segL - discard_end (:820) and then fails on a remainder longer than one
    # window (:852-859); full windows are processed here as long as more than one window is left
    while ix < L - segL - discard_end - discard_start or L - ix > segL:
        y_masked[..., :overlap] = previous[..., segL - overlap - discard_end:]
        seg = degraded[..., ix:ix + segL]
        with keyed():
            pred = sampler.predict_bwe_AR(seg, y_masked, estimated_filter, typefilter, rid=False, mask=mask)
        previous = pred[..., :keep]
        final[..., ix:ix + keep] = previous
        ix += segL - overlap - discard_end
    seg = degraded[..., ix:]
    n = seg.shape[-1]
    y_masked[..., :overlap] = pred[..., -overlap:]          # sic (:842): the tail of the FULL last prediction
    if n < segL:
        seg_zp = torch.cat((seg, seg.new_zeros((1, segL - n))), -1)
        y_masked[..., n:segL] = 0                            # the padding is "observed" silence (:848-850)
        mask[..., n:segL] = 0
    else:
        seg_zp = seg[..., :segL]
    with keyed():
        pred = sampler.predict_bwe_AR(seg_zp, y_masked, estimated_filter, typefilter, rid=False, mask=mask)
    final[..., ix:ix + n] = pred[..., :n]
    return final * scale.unsqueeze(-1) / std, estimated_filter
