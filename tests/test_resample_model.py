"""CPU checks of the resampler (csrc/sed_resample.cu) against the built library and scipy: the filter design of
sed_resample_filter, its frequency response, the indexing formula the kernels follow, and the live plan of
streaming.LiveStreamer (which outputs each tick computes and which inputs -- chunk, history ring, zeros -- they read)."""
import ctypes

import numpy as np
import pytest
import scipy.signal

from sed_b200 import capi, engine, streaming

PAIRS = [(48000, 16000), (44100, 16000), (44100, 32000), (48000, 8000), (8000, 16000), (22050, 16000)]
ROLLOFF, BETA = 0.9475937167399596, 14.769656459379492


def filt(in_rate, out_rate):
    lib = capi.load()
    up, down, n = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    args = (in_rate, out_rate, ctypes.byref(up), ctypes.byref(down), ctypes.byref(n))
    rc = lib.sed_resample_filter(*args, None)
    if rc:
        return rc, None
    taps = np.zeros(n.value, np.float32)
    assert lib.sed_resample_filter(*args, taps.ctypes.data_as(ctypes.c_void_p)) == 0
    return (up.value, down.value, n.value), taps


@pytest.mark.parametrize("in_rate,out_rate", PAIRS + [(96000, 32000), (11025, 16000)])
def test_filter_matches_scipy_firwin(in_rate, out_rate):
    (up, down, n), taps = filt(in_rate, out_rate)
    g = np.gcd(in_rate, out_rate)
    assert (up, down) == (out_rate // g, in_rate // g)
    mx = max(up, down)
    assert n == 2 * 64 * mx + 1
    ref = (up * scipy.signal.firwin(n, ROLLOFF / mx, window=("kaiser", BETA))).astype(np.float32)
    ulps = np.abs(taps.view(np.int32).astype(np.int64) - ref.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1, ulps.max()
    up2, down2, half, taps2 = engine.resample_filter(in_rate, out_rate)
    assert (up2, down2, half) == (up, down, n // 2) and np.array_equal(taps2, taps)


def test_filter_refusals():
    assert filt(48000, 44101)[0] == 2          # max(up, down) = 48000 > 4096: SED_ERR_UNSUPPORTED
    assert filt(384000, 7)[0] == 2
    for a, b in ((0, 16000), (-1, 16000), (16000, 0), (16000, -8000), (384001, 16000), (16000, 400000)):
        assert filt(a, b)[0] == 1, (a, b)      # SED_ERR_BAD_SHAPE
    assert filt(384000, 8000)[0][:2] == (1, 48)
    with pytest.raises(ValueError):
        engine.resample_filter(48000, 44101)


@pytest.mark.parametrize("in_rate,out_rate", PAIRS)
def test_frequency_response(in_rate, out_rate):
    (up, down, n), taps = filt(in_rate, out_rate)
    mx = max(up, down)
    nfft = 1 << 21
    H = np.abs(np.fft.rfft(taps.astype(np.float64) / up, nfft))
    f = np.arange(H.size) / (nfft / 2.0) * mx   # in units of the lower Nyquist frequency
    db = 20 * np.log10(np.maximum(H, 1e-300))
    assert np.abs(db[f <= 0.85]).max() <= 1e-5
    assert np.abs(db[f <= 0.9]).max() <= 0.05
    assert db[f >= 1.05].max() <= -140.0
    assert -60 < np.interp(1.0, f, db) < -50


def poly(x, j, taps, up, down, half, i0=0):
    """float64 y[j] = sum_i x[i] * taps[j*down + half - i*up] over ascending i; x[k] is input i0 + k, zero outside."""
    y = np.zeros(len(j))
    for q, jj in enumerate(j):
        t = jj * down + half
        hi = t // up
        lo = hi - (2 * half - (t - hi * up)) // up
        i = np.arange(lo, hi + 1)
        k = i - i0
        ok = (k >= 0) & (k < len(x))
        y[q] = np.dot(np.where(ok, x[np.clip(k, 0, max(len(x) - 1, 0))] if len(x) else 0.0, 0.0), taps[t - i * up])
    return y


@pytest.mark.parametrize("in_rate,out_rate", [(48000, 16000), (8000, 16000), (22050, 16000), (44100, 32000)])
def test_formula_equals_resample_poly(in_rate, out_rate):
    (up, down, n), taps = filt(in_rate, out_rate)
    half = n // 2
    rng = np.random.RandomState(in_rate + out_rate)
    for n_in in (1, 7, 1001, 3 * n // up + 5):
        x = rng.uniform(-1, 1, n_in)
        h = taps.astype(np.float64) / up
        ref = scipy.signal.resample_poly(x, up, down, window=h)
        n_out = -(-n_in * up // down)
        assert len(ref) == n_out
        got = poly(x, np.arange(n_out), taps.astype(np.float64), up, down, half)
        assert np.abs(got - ref).max() <= 1e-12, (n_in, np.abs(got - ref).max())


# ---------------------------------------------------------------------------------------------------------------
# the live plan: streaming._plan_live_resample through the real _plan_live_push, with sed_live_resample's reads
# ---------------------------------------------------------------------------------------------------------------
class _Plan:
    def __init__(self, in_rate, out_rate):
        (self.up, self.down, n), taps = filt(in_rate, out_rate)
        self.half, self.n_taps, self.taps32 = n // 2, n, taps
        self.taps64 = taps.astype(np.float64)

    n_out = engine.ResamplePlan.n_out
    n_out_live = engine.ResamplePlan.n_out_live
    history_len = engine.ResamplePlan.history_len


def _run_stream_plans(in_rate, out_rate, seed, n_streams=6):
    rs = _Plan(in_rate, out_rate)
    sr, dur, oi, fpw, classes = out_rate, 5, 100, 496, 3
    slack = streaming.LIVE_TICK_SECONDS * sr
    W, ring = sr * dur, sr * dur + slack
    geometry = (sr, dur, W, ring, oi, fpw, classes, slack)
    H = rs.history_len()
    assert H == -(-(rs.n_taps - 1 + rs.down) // rs.up) + 1
    rng = np.random.RandomState(seed)
    slots = 8
    n_in, n_samp, k_run, f_ret = (np.zeros(slots, np.int64) for _ in range(4))
    hist = np.full((slots, H), 1e9)  # history of no stream (or of a slot's previous one): must never be read
    totals = [1, rs.down - 1, int(0.3 * in_rate), int(5.7 * in_rate) + 3, int(7.1 * in_rate)][:n_streams]
    recs = [rng.uniform(-1, 1, t) for t in totals]
    sizes = [0, 1, rs.down - 1, rs.down + 1, 777, in_rate // 3 + 1, 2 * in_rate + 5]
    written = {i: [] for i in range(len(recs))}
    values = {i: {} for i in range(len(recs))}
    min_hist_margin = np.inf
    free = list(range(slots))
    sid_of, fed, open_ = {}, [0] * len(recs), []
    pending = list(range(len(recs)))
    while pending or open_:
        if pending and rng.rand() < 0.6:
            i = pending.pop(0)
            sid_of[i] = free.pop(0)
            n_in[sid_of[i]] = n_samp[sid_of[i]] = k_run[sid_of[i]] = f_ret[sid_of[i]] = 0
            open_.append(i)
        push = [i for i in open_ if rng.rand() < 0.8]
        closing = []
        for i in list(open_):
            if fed[i] == totals[i] and i not in push and rng.rand() < 0.5:
                closing.append(i)
        for group, is_close in ([(push, False)] if push else []) + [([i], True) for i in closing]:
            sids = np.array([sid_of[i] for i in group], np.int64)
            lens = np.zeros(len(group), np.int64) if is_close else np.array(
                [min(int(rng.choice(sizes)), totals[i] - fed[i]) for i in group], np.int64)
            order = rng.permutation(len(group))
            src = np.zeros(len(group), np.int64)
            src[order] = np.cumsum(lens[order]) - lens[order]
            staged = np.zeros(int(lens.sum()))
            for g, i in enumerate(group):
                staged[src[g]:src[g] + lens[g]] = recs[i][fed[i]:fed[i] + lens[g]]
            plan, hist_tab, n_end = streaming._plan_live_resample(
                rs, sids, n_in[sids].copy(), n_samp[sids], k_run[sids], f_ret[sids], lens, src, is_close, *geometry)
            for ing, _, _, _, _ in plan[0]:
                for slot, j0, cnt, off, n_prev, n_e in ing.tolist():
                    i = group[list(sids).index(slot)]
                    assert j0 == len(written[i]), "outputs in order, each once"
                    written[i].extend(range(j0, j0 + cnt))
                    if off < 0:  # zero fill of the closing window 0: beyond the resampled end
                        assert is_close and j0 >= rs.n_out(n_e)
                        continue
                    j = np.arange(j0, j0 + cnt)
                    t = j * rs.down + rs.half
                    i_hi = t // rs.up
                    i_lo = i_hi - (2 * rs.half - (t - i_hi * rs.up)) // rs.up
                    # whole support arrived, or beyond the end at close only
                    assert is_close or i_hi.max() < n_e
                    lo, hi = int(i_lo.min()), int(i_hi.max())
                    span = np.arange(lo, hi + 1)
                    from_hist = (span >= 0) & (span < n_prev)
                    if from_hist.any():
                        margin = int(span[from_hist].min()) - (n_prev - H)
                        assert margin >= 0, ("history read below n_prev - H", margin)
                        min_hist_margin = min(min_hist_margin, margin)
                    x = np.zeros(len(span))  # i < 0 and i >= n_e read zeros
                    x[from_hist] = hist[slot, span[from_hist] % H]
                    cur = (span >= n_prev) & (span < n_e)
                    x[cur] = staged[off + span[cur] - n_prev]
                    y = poly(x, j, rs.taps64, rs.up, rs.down, rs.half, i0=lo)
                    values[i].update(zip(j.tolist(), y.tolist()))
            for slot, off, n_prev, ln in hist_tab.tolist():
                keep = min(ln, H)
                for s in range(ln - keep, ln):
                    hist[slot, (n_prev + s) % H] = staged[off + s]
            for g, i in enumerate(group):
                fed[i] += int(lens[g])
            after = plan[-1]
            n_samp[sids], k_run[sids], f_ret[sids] = after
            n_in[sids] = n_end
            if is_close:
                i = group[0]
                open_.remove(i)
                free.append(sid_of[i])
                free.sort()
                hist[sid_of[i]] = 1e9
                n_out = int(rs.n_out(totals[i]))
                assert written[i][:n_out] == list(range(n_out)) and all(
                    w >= n_out for w in written[i][n_out:]), "outputs 0 .. ceil(n*up/down) - 1, then the window fill"
                ref = poly(recs[i], np.arange(n_out), rs.taps64, rs.up, rs.down, rs.half)
                got = np.array([values[i][j] for j in range(n_out)])
                assert np.array_equal(got, ref), ("live outputs differ from the offline formula", i)
    return min_hist_margin


@pytest.mark.parametrize("in_rate,out_rate", [(48000, 16000), (44100, 16000), (8000, 16000), (22050, 16000)])
def test_live_plan_reads_only_arrived_input_and_recent_history(in_rate, out_rate):
    """Random chunkings (1 sample, down - 1 samples, sizes not a multiple of down, several ticks), streams shorter
    than one window, slot reuse: every tick's outputs have their whole support (or lie beyond the end at close),
    history reads stay within n_prev - H, outputs 0 .. ceil(n*up/down) - 1 are written once each in order, and the
    values the reads produce equal the offline formula on the whole recording exactly."""
    margin = _run_stream_plans(in_rate, out_rate, seed=in_rate + out_rate)
    assert 0 <= margin < np.inf
