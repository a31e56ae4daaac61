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


@contextlib.contextmanager
def _filter_per_row(sampler, on):
    """Set the sampler's ``filter_per_row`` for one call and restore the previous value afterwards."""
    was = sampler.filter_per_row
    sampler.filter_per_row = on
    try:
        yield
    finally:
        sampler.filter_per_row = was


@contextlib.contextmanager
def _filter_groups(sampler, sizes):
    """Set the sampler's ``filter_groups`` for one call and restore the previous value afterwards."""
    was = sampler.filter_groups
    sampler.filter_groups = sizes
    try:
        yield
    finally:
        sampler.filter_groups = was


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


def pack_recordings(sizes, max_rows=None):
    """Consecutive runs of recordings (lists of indices) whose segment counts ``sizes`` add up to at most
    ``max_rows`` each, filled greedily in order; one run of all recordings when ``max_rows`` is None."""
    if max_rows is not None and (isinstance(max_rows, bool) or not isinstance(max_rows, int) or max_rows < 1):
        raise ValueError(f"max_rows must be a positive int, got {max_rows!r}")
    if max_rows is None or not sizes:
        return [list(range(len(sizes)))] if sizes else []
    calls, cur, rows = [], [], 0
    for r, n in enumerate(sizes):
        if n > max_rows:
            raise ValueError(f"recording {r} has {n} segments, more than max_rows = {max_rows}: a recording's "
                             "segments share one filter and cannot be split over calls")
        if rows + n > max_rows:
            calls.append(cur)
            cur, rows = [], 0
        cur.append(r)
        rows += n
    calls.append(cur)
    return calls


def restore_recordings(sampler, recordings, seg_len, ola=256, discard_end=200, seeds=None, max_rows=None):
    """Blind restoration of N recordings with ONE filter each, the segments of many recordings in one sampler call.

    Every recording is cut as ``restore_recording`` cuts it; the segments of consecutive recordings go into one
    ``predict_blind_bwe`` call with ``filter_groups = [S_0, S_1, ...]`` (recording r's S_r segments are one group:
    summed fit statistics, one filter fit, one guidance normaliser), so recording r is restored as
    ``restore_recording(joint=True)`` restores it alone in one process.  ``max_rows`` bounds the rows of a call:
    whole recordings are packed greedily, in order (a recording with more than ``max_rows`` segments raises
    ValueError); None puts every recording into one call.

    ``recordings``: mono (1, L_r) tensors on one device.  ``seeds`` (one int per recording) switches to keyed noise:
    segment s of recording r draws with ``row_seed(seeds[r], s)``, the seed ``restore_recording(seed=seeds[r])``
    gives it.  Single process: sharding recordings over ranks is the caller's.  The sampler's ``filter_groups``,
    ``filter_per_row`` and ``row_seeds`` are restored afterwards.  Returns [(restored (1, L_r), filter_data), ...],
    ``filter_data`` the list [((ix0, ix1), filter (2, K)), ...] of ``restore_recording`` with the recording's one
    filter on every span."""
    if getattr(sampler, "joint", False):
        raise ValueError("restore_recordings gives every recording its own filter; joint=True shares one over all "
                         "rows of all ranks")
    recs = [r.reshape(1, -1) if r.dim() == 1 else r for r in recordings]
    N = len(recs)
    for i, r in enumerate(recs):
        if r.dim() != 2 or r.shape[0] != 1:
            raise ValueError(f"recording {i} must be mono (1, L), got {tuple(r.shape)}")
        if r.device != recs[0].device:
            raise ValueError(f"recording {i} is on {r.device}, recording 0 on {recs[0].device}: one device for all")
    if seeds is not None and len(seeds) != N:
        raise ValueError(f"{len(seeds)} seeds for {N} recordings")
    cuts = [split(r, seg_len, ola, discard_end) for r in recs]
    sizes = [segs.shape[0] for segs, _ in cuts]
    out = [None] * N
    for rows in pack_recordings(sizes, max_rows):
        y = torch.cat([cuts[r][0] for r in rows])
        row_seeds = None if seeds is None else [row_seed(seeds[r], s) for r in rows for s in range(sizes[r])]
        with _filter_groups(sampler, [sizes[r] for r in rows]), _filter_per_row(sampler, False), \
                _row_seeds(sampler, row_seeds):
            pred, filts = sampler.predict_blind_bwe(y, rid=False)
        o = 0
        for g, r in enumerate(rows):
            spans = cuts[r][1]
            final = merge(pred[o:o + sizes[r]], spans, recs[r].shape[-1], ola, discard_end)
            out[r] = (final, [(sp, filts[g]) for sp in spans])
            o += sizes[r]
    return out


def ar_windows(L, seg_len, overlap, discard_end=200, discard_start=0):
    """Windows ``(start, length)`` that the autoregressive restoration of a recording of L samples visits, in order:
    the first window (0, seg_len) (``predict_bwe``), the autoregressive windows advancing by
    ``seg_len - overlap - discard_end`` samples, and the last window (start, n) with n = L - start <= seg_len, which
    is zero padded to seg_len (testing/blind_bwe_tester.py:799-859).  The reference stops at
    ix >= L - seg_len - discard_end (:820) and then fails on a remainder longer than one window (:852-859); full
    windows are placed here as long as more than one window is left."""
    step = seg_len - overlap - discard_end
    windows, ix = [(0, seg_len)], step
    while ix < L - seg_len - discard_end - discard_start or L - ix > seg_len:
        windows.append((ix, seg_len))
        ix += step
    windows.append((ix, L - ix))
    return windows


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
    windows = ar_windows(L, segL, overlap, discard_end, discard_start)
    window = [0]

    def keyed():                                             # the seeds of the next window
        w = window[0]
        window[0] += 1
        return _row_seeds(sampler, None if seed is None else [row_seed(seed, w)])

    seg = degraded[..., :segL]
    with keyed():
        pred = sampler.predict_bwe(seg, estimated_filter, typefilter, rid=False)
    previous = pred[..., :keep]
    final[..., :keep] = previous
    y_masked = torch.zeros_like(pred)
    mask = torch.ones_like(seg)
    mask[..., overlap:] = 0
    for ix, _ in windows[1:-1]:
        y_masked[..., :overlap] = previous[..., segL - overlap - discard_end:]
        seg = degraded[..., ix:ix + segL]
        with keyed():
            pred = sampler.predict_bwe_AR(seg, y_masked, estimated_filter, typefilter, rid=False, mask=mask)
        previous = pred[..., :keep]
        final[..., ix:ix + keep] = previous
    ix, n = windows[-1]
    seg = degraded[..., ix:]
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


def restore_recordings_ar(sampler, recordings, seg_len, sample_rate, overlap_s=0.25, n_segments_blindstep=2,
                          ix_start_s=0, std=0.1, typefilter="fc_A", discard_end=200, discard_start=0, seeds=None,
                          estimated_filters=None, rng=None):
    """``restore_recording_ar`` on N recordings at once: window w of every recording that still has one goes into ONE
    sampler call with ``filter_per_row`` (round 0 ``predict_bwe``, later rounds ``predict_bwe_AR``), so the denoiser
    runs at batch N instead of N times at batch 1.  The batch shrinks as the shorter recordings finish.  Row r of a
    call is independent of the other rows, so recording r is restored as ``restore_recording_ar`` restores it alone:
    the same normalisation, known heads, last padded window and final scale.

    ``recordings``: (1, L_r) tensors on one device, each at least ``seg_len`` long.  ``seeds`` (one int per
    recording) switches to keyed noise with the seeds ``restore_recording_ar(seed=seeds[r])`` uses: window w draws
    with ``row_seed(seeds[r], w)``, blind-step row j with ``row_seed(seeds[r], 2**32 + j)``; the restorations then
    agree to rounding.  ``estimated_filters`` (N filters (2, K)) skips the blind step.  Otherwise
    ``n_segments_blindstep == 1`` estimates the N filters in ONE per-row ``predict_blind_bwe`` call on the first
    windows, and larger counts run one blind call per recording, in recording order, drawing window positions from
    ``rng`` as N sequential ``restore_recording_ar`` calls do.  Single process: sharding recordings over ranks is
    the caller's.  Returns [(restored (1, L_r), filter (2, K)), ...]."""
    import numpy as np
    if getattr(sampler, "joint", False):
        raise ValueError("restore_recordings_ar restores every recording with its own filter; joint=True shares one")
    if typefilter != "fc_A":
        raise NotImplementedError(f"typefilter {typefilter!r}: only the parametric fc_A filter has per-row kernels")
    segL = int(seg_len)
    recs = [r.reshape(1, -1) for r in recordings]
    N = len(recs)
    if N == 0:
        return []
    device = recs[0].device
    for i, r in enumerate(recs):
        if r.device != device:
            raise ValueError(f"recording {i} is on {r.device}, recording 0 on {device}: one device for all")
        if r.shape[-1] < segL:
            raise ValueError(f"recording {i} has {r.shape[-1]} samples, fewer than seg_len = {segL}")
    if seeds is not None and len(seeds) != N:
        raise ValueError(f"{len(seeds)} seeds for {N} recordings")
    if estimated_filters is not None and len(estimated_filters) != N:
        raise ValueError(f"{len(estimated_filters)} filters for {N} recordings")
    scales = [r.std(-1) for r in recs]
    deg = [std * r / sc.unsqueeze(-1) for r, sc in zip(recs, scales)]
    finals = [torch.zeros_like(d) for d in deg]
    ix_first = int(sample_rate * ix_start_s)

    def keyed(rows, k):                                      # seeds of unit k of the given recordings
        return _row_seeds(sampler, None if seeds is None else [row_seed(seeds[r], k) for r in rows])

    if estimated_filters is None:
        if n_segments_blindstep == 1:
            y = torch.cat([d[..., ix_first:ix_first + segL] for d in deg])
            with _filter_per_row(sampler, True), keyed(range(N), 1 << 32):
                pred, filts = sampler.predict_blind_bwe(y, rid=False)
            for r in range(N):
                finals[r][0, ix_first:ix_first + segL] = pred[r]
        else:
            rng = rng if rng is not None else np.random
            fl = []
            for r, d in enumerate(deg):
                L = d.shape[-1]
                y = d[..., ix_first:ix_first + segL].repeat(n_segments_blindstep, 1)
                for j in range(n_segments_blindstep):
                    ix = int(rng.randint(0, L - segL))
                    y[j] = d[0, ix:ix + segL]
                blind = None if seeds is None else [row_seed(seeds[r], (1 << 32) + j) for j in range(y.shape[0])]
                with _filter_per_row(sampler, False), _row_seeds(sampler, blind):
                    pred, f = sampler.predict_blind_bwe(y, rid=False)
                finals[r][0, ix_first:ix_first + segL] = pred[0]
                fl.append(f)
            filts = torch.stack(fl)
    else:
        filts = torch.stack([f.to(device) for f in estimated_filters])
    overlap = int(overlap_s * sample_rate)
    keep = segL - discard_end
    windows = [ar_windows(d.shape[-1], segL, overlap, discard_end, discard_start) for d in deg]
    preds = [None] * N                                       # last prediction of each recording
    previous = [None] * N
    y_masked = [None] * N
    masks = [None] * N
    with _filter_per_row(sampler, True):
        for w in range(max(len(ws) for ws in windows)):
            rows = [r for r in range(N) if w < len(windows[r])]
            segs = []
            for r in rows:
                ix, n = windows[r][w]
                if w == 0:
                    segs.append(deg[r][..., :segL])
                elif w < len(windows[r]) - 1:
                    y_masked[r][..., :overlap] = previous[r][..., segL - overlap - discard_end:]
                    segs.append(deg[r][..., ix:ix + segL])
                else:
                    y_masked[r][..., :overlap] = preds[r][..., -overlap:]     # sic (:842), as restore_recording_ar
                    seg = deg[r][..., ix:]
                    if n < segL:
                        seg = torch.cat((seg, seg.new_zeros((1, segL - n))), -1)
                        y_masked[r][..., n:segL] = 0
                        masks[r][..., n:segL] = 0
                    segs.append(seg[..., :segL])
            with keyed(rows, w):
                if w == 0:
                    out = sampler.predict_bwe(torch.cat(segs), filts, typefilter, rid=False)
                else:
                    out = sampler.predict_bwe_AR(torch.cat(segs), torch.cat([y_masked[r] for r in rows]),
                                                 filts[rows], typefilter, rid=False,
                                                 mask=torch.cat([masks[r] for r in rows]))
            for i, r in enumerate(rows):
                ix, n = windows[r][w]
                preds[r] = pred = out[i:i + 1]
                if w == 0:
                    y_masked[r] = torch.zeros_like(pred)
                    masks[r] = torch.ones_like(pred)
                    masks[r][..., overlap:] = 0
                if w < len(windows[r]) - 1:
                    previous[r] = pred[..., :keep]
                    finals[r][..., ix:ix + keep] = previous[r]
                else:
                    finals[r][..., ix:ix + n] = pred[..., :n]
    return [(f * sc.unsqueeze(-1) / std, filts[r]) for r, (f, sc) in enumerate(zip(finals, scales))]
