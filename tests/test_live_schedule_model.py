"""CPU model of the live (incremental) streaming path: the per-slot merge accumulator with its finality rule, and the
resumable event state machine of csrc/sed_stream.cu (live_merge_kernel / live_events_kernel), restated in numpy and
checked against the pinned oracle (stream_oracle.merge_windows / activity_detection) under random arrival patterns;
and streaming.LiveStreamer's push planner itself, checked against the bounds these kernels rely on."""
import json
import os

import numpy as np
import pytest

import stream_oracle
from conftest import GOLD


# ---------------------------------------------------------------------------------------------------------------
# incremental merge + avg_merge
# ---------------------------------------------------------------------------------------------------------------
def final_frames(windows_run, fpw, oi, dur):
    """Frames of the merged output that no later window and no final length can change once `windows_run` windows
    have been merged: covered by no later window (f < windows_run*oi) and in a block whose avg_merge divisor is the
    same for every total >= (windows_run-1)*oi + fpw."""
    if windows_run <= 0:
        return 0
    K = windows_run - 1
    tmin = K * oi + fpw
    interval = dur * 100 - oi
    b = min(tmin - oi, max(interval, tmin - interval))
    lb = max(oi, -(-b // oi) * oi)
    return min((K + 1) * oi, lb)


class LiveModel:
    """One stream: windows arrive in ascending order, a few per tick; `tick` returns the newly final rows of the merged
    output, `close` the rest.  The accumulator is a ring of `ring` frames, as on the device."""

    def __init__(self, fpw, oi, dur, classes, ring):
        self.fpw, self.oi, self.dur, self.ring = fpw, oi, dur, ring
        self.acc = np.zeros((ring, classes), np.float32)
        self.k = 0     # windows merged
        self.ret = 0   # frames returned
        self.max_live = 0

    def _divide(self, f, v, total):
        oi = self.oi
        if f < oi:
            return v
        i = (f // oi) * oi
        if i >= total - oi:
            return v
        interval = self.dur * 100 - oi
        if i < interval:
            div = i // oi + 1
        elif i >= total - interval:
            div = (total - i) // oi + 1
        else:
            div = self.dur
        return v / np.float32(div)

    def tick(self, windows, closing=False):
        oi, fpw = self.oi, self.fpw
        k0, m = self.k, len(windows)
        if closing and k0 + m == 0:
            raise ValueError("window 0 runs at close: pass it")
        self.k += m
        K = self.k - 1
        tmin = K * oi + fpw
        n_final = tmin if closing else final_frames(self.k, fpw, oi, self.dur)
        hi = tmin if m else n_final
        self.max_live = max(self.max_live, hi - self.ret)
        assert hi - self.ret <= self.ring, (hi, self.ret, self.ring)
        out = []
        for f in range(self.ret, hi):
            r = f % self.ring
            first = not (k0 >= 1 and f < (k0 - 1) * oi + fpw)
            acc = self.acc[r].copy()
            klo = 0 if f - fpw + 1 <= 0 else (f - fpw + oi) // oi
            for k in range(max(k0, klo), min(k0 + m - 1, f // oi) + 1):
                v = windows[k - k0][f - k * oi]
                acc = v.copy() if first else acc + v
                first = False
            if f < n_final:
                out.append(self._divide(f, acc, tmin))
            else:
                self.acc[r] = acc
        self.ret = n_final
        return np.array(out, np.float32).reshape(len(out), self.acc.shape[1])


def ring_frames(fpw, oi, dur, windows_per_tick):
    """Accumulator ring length that the tick can never overrun (streaming.LiveStreamer uses the same bound)."""
    return (windows_per_tick - 1) * oi + max(fpw, 100 * dur) + oi


MERGE_CASES = [(fpw, oi, dur) for fpw in (500, 496, 600) for oi in (100, 50) for dur in (5, 6)]


@pytest.mark.parametrize("fpw,oi,dur", MERGE_CASES)
def test_incremental_merge_equals_offline_merge_bitwise(fpw, oi, dur):
    rng = np.random.RandomState(fpw * 1000 + oi * 10 + dur)
    ov = oi / 100.0
    for trial in range(30):
        nw = int(rng.randint(1, 13))
        frames = rng.rand(nw, fpw, 3).astype(np.float32)
        ref = stream_oracle.merge_windows(frames, dur, ov)[0]
        per_tick = int(rng.choice([1, 2, 3, 4]))
        model = LiveModel(fpw, oi, dur, 3, ring_frames(fpw, oi, dur, per_tick))
        got, k = [], 0
        while k < nw:
            m = int(rng.randint(0, per_tick + 1))
            m = min(m, nw - k)
            got.append(model.tick(list(frames[k:k + m])))
            k += m
            if m and oi <= 100 and fpw > 100 * dur - oi:
                # contract item 3: exactly (k+1)*oi frames after the push in which window k ran
                assert model.ret == k * oi, (k, model.ret)
        got.append(model.tick([], closing=True))
        got = np.concatenate(got)
        assert got.shape == ref.shape
        assert np.array_equal(got, ref), (trial, nw)


def test_streamer_uses_the_same_finality_rule():
    from sed_b200 import streaming
    for fpw, oi, dur in MERGE_CASES:
        k = np.arange(0, 80)
        assert list(streaming.live_final_frames(k, fpw, oi, dur)) == [final_frames(int(v), fpw, oi, dur) for v in k]


def test_final_frames_rule_for_shipped_presets():
    for fpw in (500, 496):
        for k in range(1, 60):
            assert final_frames(k, fpw, 100, 5) == k * 100
    assert final_frames(0, 500, 100, 5) == 0


# ---------------------------------------------------------------------------------------------------------------
# resumable activity_detection
# ---------------------------------------------------------------------------------------------------------------
class LiveEvents:
    """activity_detection (utils/vad.py:11-45) as a state machine over frames that arrive in chunks: the same fields
    and the same order of steps as LiveEventState / live_event_step in csrc/sed_stream.cu."""

    def __init__(self, th, tl, n_smooth, n_salt):
        self.th, self.tl, self.ns, self.salt = float(th), tl, int(n_smooth), int(n_salt)
        self.use_low = tl is not None
        self.n = 0
        self.run_end = -1          # last frame above the high threshold
        self.p_has = False         # the pair of the current run exists
        self.p_b = self.p_s = 0    # its raw onset and extended onset
        self.p_sk = self.p_pushed = self.p_lowend = False
        self.fbr = -1              # first frame after run_end below the low threshold
        self.last_below = -1
        self.q_has, self.q_s = False, 0
        self.s1 = [False, 0, 0]
        self.s2 = [False, 0, 0]
        self.out = []

    def _final(self, b, f):
        if f - b > self.salt:
            self.out.append([b, f])

    def _smooth(self, st, n, b, f, emit):
        if st[0] and b - st[2] > n:
            emit(st[1], st[2])
            st[1] = b
        elif not st[0]:
            st[0], st[1] = True, b
        st[2] = f

    def _s2(self, b, f):
        self._smooth(self.s2, self.ns, b, f, self._final)

    def _s1(self, b, f):
        self._smooth(self.s1, 1, b, f, self._s2)

    def _raw(self, b, f):
        self._s2(b, f)

    def step(self, x):
        i = self.n
        self.n += 1
        x = float(x)
        if not self.use_low:
            if x > self.th:
                if self.p_has and i - self.run_end > 1:
                    self._raw(self.p_b, self.run_end + 1)
                    self.p_b = i + 1
                elif not self.p_has:
                    self.p_has, self.p_b = True, i
                self.run_end = i
            return
        tl = float(self.tl)
        below = x < tl
        if x > self.th:
            if self.p_has and i - self.run_end > 1:
                if not self.p_pushed:
                    if self.fbr >= 0:
                        self._s1(self.p_s, self.fbr)
                    else:
                        self.q_has, self.q_s = True, self.p_s
                self.p_b, self.p_sk, self.p_pushed = i + 1, False, False
            elif not self.p_has:
                self.p_has, self.p_b, self.p_sk, self.p_pushed = True, i, False, False
            self.run_end, self.fbr, self.p_lowend = i, -1, below
        if self.p_has and not self.p_sk and self.p_b == i:
            self.p_s = i + 1 if below else self.last_below + 1
            self.p_sk = True
        if below:
            if self.q_has:
                self._s1(self.q_s, i)
                self.q_has = False
            if self.fbr < 0 and i > self.run_end:
                self.fbr = i
            self.last_below = i
        elif self.q_has and i == self.p_b:
            self.q_has = False  # the pair of the new run extends to the same [S, E]: smooth(1) would collapse them
        if self.p_has and not self.p_pushed and not self.q_has and self.p_sk and not self.p_lowend and self.fbr >= 0:
            self._s1(self.p_s, self.fbr)
            self.p_pushed = True
        if not self.q_has and (not self.p_has or self.p_pushed):
            lb = self.last_below + 1
            if self.s1[0] and lb - self.s1[2] > 1:
                self._s2(self.s1[1], self.s1[2])
                self.s1[0] = False
            if self.s2[0] and not self.s1[0] and lb - self.s2[2] > self.ns:
                self._final(self.s2[1], self.s2[2])
                self.s2[0] = False
        if self.s2[0] and self.s1[0] and self.s1[1] - self.s2[2] > self.ns:
            self._final(self.s2[1], self.s2[2])
            self.s2[0] = False

    def close(self):
        n = self.n
        if not self.use_low:
            if self.p_has:
                self._raw(self.p_b, self.run_end)
        else:
            if self.q_has:
                self._s1(self.q_s, n)
                self.q_has = False
            if self.p_has and not self.p_pushed:
                s = self.p_s if self.p_sk else n + 1
                e = self.run_end if self.p_lowend else (self.fbr if self.fbr >= 0 else n)
                self._s1(s, e)
            if self.s1[0]:
                self._s2(self.s1[1], self.s1[2])
        if self.s2[0]:
            self._final(self.s2[1], self.s2[2])

    def feed(self, xs):
        before = len(self.out)
        for v in xs:
            self.step(v)
        return self.out[before:]


def event_capacity(n_frames):
    """Events one (stream, class) can report for a push that finalizes `n_frames` frames (close included): at most
    one per pending stage (pair of the current run, the one-frame pair queue, smooth(1), smooth(n_smooth)) plus one
    per run that starts in the push, and runs start at least two frames apart."""
    return (n_frames + 1) // 2 + 4


def _sequences(rng):
    n = int(rng.randint(1, 400))
    yield rng.rand(n).astype(np.float32)
    yield (rng.rand(n) > 0.5).astype(np.float32) * np.float32(0.9)             # runs of length 1 and more
    yield np.tile(np.array([0.9, 0.1], np.float32), n // 2 + 1)[:n]           # alternating: every run has length 1
    yield rng.choice(np.array([0.1, 0.3, 0.5, 0.7, 0.9], np.float32), n)      # values exactly at the thresholds
    yield np.repeat(rng.rand(n // 7 + 1).astype(np.float32), 7)[:n]
    yield np.clip(np.cumsum(rng.randn(n)) * 0.05 + 0.5, 0, 1).astype(np.float32)


def _check(x, th, tl, ns, salt, chunk):
    # float64 thresholds: the comparisons are made in float64, as the device kernels make them
    ref = stream_oracle.activity_detection(x, np.float64(th), None if tl is None else np.float64(tl), ns, salt)
    ev = LiveEvents(th, tl, ns, salt)
    got, emitted_at = [], []
    for c0 in range(0, len(x), chunk):
        new = ev.feed(x[c0:c0 + chunk])
        n_done = min(len(x), c0 + chunk)
        assert len(new) <= event_capacity(n_done - c0)
        got += new
        emitted_at += [n_done] * len(new)
    tail = len(ev.out)
    ev.close()
    assert len(ev.out) - tail <= event_capacity(0)
    got += ev.out[tail:]
    emitted_at += [len(x) + 1] * (len(ev.out) - tail)
    assert got == [[int(b), int(f)] for b, f in ref], (th, tl, ns, salt, chunk, got, ref)
    if tl is not None and float(tl) <= float(th):
        # contract item 4: an event with offset F is reported by the push that finalizes frame F + n_smooth + 1 when
        # frames F .. F + n_smooth + 1 are all below the low threshold
        for (b, f), at in zip(got, emitted_at):
            last = f + ns + 1
            if last < len(x) and np.all(x[f:last + 1].astype(np.float64) < float(tl)):
                assert at <= (last // chunk + 1) * chunk, ((b, f), at, last, chunk)


@pytest.mark.parametrize("chunk", [1, 37, 100000])
def test_streaming_events_equal_activity_detection(chunk):
    rng = np.random.RandomState(chunk)
    params = [(0.5, 0.3, 10, 10), (0.5, 0.3, 1, 0), (0.5, 0.3, 0, 0), (0.3, 0.5, 1, 0), (0.3, 0.5, 10, 10),
              (0.5, -0.2, 1, 0), (0.5, -1.0, 0, 10), (0.5, None, 10, 10), (0.5, None, 0, 0), (0.7, 0.7, 1, 0),
              (0.5, 0.5, 0, 0), (0.1, 0.9, 0, 0)]
    for _ in range(6):
        for x in _sequences(rng):
            for th, tl, ns, salt in params:
                _check(x, th, tl, ns, salt, chunk)


def test_streaming_events_with_shipped_thresholds():
    with open(os.path.join(GOLD, "opt_thresholds.json")) as f:
        shipped = json.load(f)
    rng = np.random.RandomState(7)
    for name, p in shipped.items():
        hi, lo = p["sed_high_threshold"], p.get("sed_low_threshold")
        ns, salt = p["n_smooth"], p["n_salt"]
        for c in range(len(hi)):
            for x in _sequences(rng):
                for chunk in (1, 37, len(x)):
                    _check(x, hi[c], None if lo is None else lo[c],
                           ns[c] if np.ndim(ns) else ns, salt[c] if np.ndim(salt) else salt, chunk)


# ---------------------------------------------------------------------------------------------------------------
# the push planner of streaming.LiveStreamer: ring residency, accumulator span, frame and event bookkeeping
# ---------------------------------------------------------------------------------------------------------------
def _check_plan(plan, sids, before, lens, src, closing, geometry):
    """Checks one planned push against the stream counters `before` = (samples, windows run, frames returned) and
    returns the counters after it, as the kernels would leave them."""
    from sed_b200 import streaming
    sr, dur, W, ring, oi, fpw, classes, slack = geometry
    span_max = ring_frames(fpw, oi, dur, streaming.LIVE_TICK_SECONDS)
    ticks, offsets, rows_per_stream, base, n_rows, n_entries, ev_total, after = plan
    n, k_run, f_ret = (v.copy() for v in before)
    taken, rows = np.zeros(len(sids), np.int64), np.zeros(len(sids), np.int64)
    pos = {int(s): j for j, s in enumerate(sids)}
    w0 = ev = entries = 0
    for t, (ing, tab, sel, n_win, span) in enumerate(ticks):
        last = closing and t == len(ticks) - 1
        fill = {}
        for sid, at, piece, n0 in ing.tolist():
            j = pos[sid]
            if at < 0:  # zero fill of the closing window 0 of a stream shorter than one window
                assert last and k_run[j] == 0 and n0 == n[j] < W and piece == W - n0, (t, sid)
                fill[j] = True
                continue
            assert at == src[j] + taken[j] and n0 == n[j] and 0 < piece, (t, sid)
            taken[j] += piece
            n[j] += piece
        ready = np.where(n >= W, n // sr - dur + 1, 0)
        if last:
            ready = np.maximum(ready, 1)
        assert sorted(sel.tolist()) == sorted(set(np.flatnonzero(ready > k_run).tolist()) |
                                              (set(range(len(sids))) if last else set()))
        tick_span = tick_windows = 0
        for sid, k0, m, w_rel, f0, f1, row, ev0, cap, is_last in tab.tolist():
            j = pos[sid]
            assert k0 == k_run[j] and k0 + m == ready[j] and is_last == int(last) and w_rel == tick_windows
            tick_windows += m
            n1 = int(n[j])
            for i, k in enumerate(range(k0, k0 + m)):
                assert offsets[w0 + w_rel + i] == sid * 2 * ring + (k * sr) % ring
                assert k * sr >= n1 - ring, ("window leaves the ring", sid, k, n1)
                assert k * sr + W <= n1 or (last and k == 0 and fill.get(j)), ("window not ready", sid, k, n1)
            # frames: continue where the stream stopped; final_frames after a push, the whole merged length at close
            assert f0 == f_ret[j]
            assert f1 == ((k0 + m - 1) * oi + fpw if last else final_frames(k0 + m, fpw, oi, dur))
            assert row == base[j] + rows[j]
            rows[j] += f1 - f0
            hi = (k0 + m - 1) * oi + fpw if m else f1
            tick_span = max(tick_span, hi - f0)
            assert cap == event_capacity(f1 - f0) and ev0 == ev
            ev += cap * classes
            k_run[j], f_ret[j] = k0 + m, f1
        assert span == tick_span and span <= span_max, (t, span, span_max)
        assert n_win == tick_windows
        w0 += n_win
        entries += len(tab)
    assert list(taken) == list(lens)
    assert (w0, ev, entries, n_rows) == (len(offsets), ev_total, n_entries, int(rows.sum()))
    assert list(rows) == list(rows_per_stream) and list(base) == list(np.cumsum(rows) - rows)
    for got, want in zip(after, (n, k_run, f_ret)):
        assert list(got) == list(want)
    return n, k_run, f_ret


PLAN_GEOMETRIES = [(16000, 500, 100, 5), (16000, 496, 100, 5), (32000, 500, 100, 5), (8000, 496, 100, 5),
                   (16000, 500, 50, 6), (16000, 496, 50, 6), (8000, 600, 100, 5), (8000, 600, 50, 6)]


@pytest.mark.parametrize("sr,fpw,oi,dur", PLAN_GEOMETRIES)
def test_live_push_planner_keeps_windows_in_ring_and_frames_complete(sr, fpw, oi, dur):
    """The real planner driven by random pushes of several streams (chunks of 0 and 1 samples, odd sizes, several
    ticks, a stream that closes before one window): every window it runs is ready and resident in its stream's
    audio ring, no tick spans more frames than the accumulator ring, entries finalize frames contiguously and with
    the finality rule above, their event capacity is event_capacity, and at close a stream has returned the whole
    offline merged length."""
    from sed_b200 import streaming
    classes = 3
    slack = streaming.LIVE_TICK_SECONDS * sr
    W, ring = sr * dur, sr * dur + slack
    geometry = (sr, dur, W, ring, oi, fpw, classes, slack)
    rng = np.random.RandomState(sr + fpw + oi + dur)
    for trial in range(4):
        total = [0, 1, W // 2 + 3, W - 1, W, W + sr - 1, 9 * sr + 123, 31 * sr + 7]
        sid_of = rng.permutation(12)[:len(total)]  # slot ids: not the stream order, not contiguous
        n = np.zeros(12, np.int64)
        k_run, f_ret = n.copy(), n.copy()
        fed = [0] * len(total)
        sizes = [0, 1, 777, sr - 1, sr, 2 * sr, 2 * sr + 5, 5 * sr + 3]
        open_ = list(range(len(total)))
        while open_:
            push = [i for i in open_ if rng.rand() < 0.8]
            lens = np.array([min(int(rng.choice(sizes)), total[i] - fed[i]) for i in push], np.int64)
            sids = sid_of[push].astype(np.int64)
            order = rng.permutation(len(push))  # any disjoint layout of the chunks in the staged audio
            src = np.zeros(len(push), np.int64)
            src[order] = np.concatenate([[0], np.cumsum(lens[order])[:-1]]) if len(push) else []
            before = (n[sids], k_run[sids], f_ret[sids])
            plan = streaming._plan_live_push(sids, *before, lens, src, False, *geometry)
            n[sids], k_run[sids], f_ret[sids] = _check_plan(plan, sids, before, lens, src, False, geometry)
            for i, ln in zip(push, lens):
                fed[i] += int(ln)
            for i in [i for i in open_ if fed[i] == total[i] and rng.rand() < 0.5]:
                sids = sid_of[[i]].astype(np.int64)
                before = (n[sids], k_run[sids], f_ret[sids])
                zero = np.zeros(1, np.int64)
                plan = streaming._plan_live_push(sids, *before, zero, zero, True, *geometry)
                n[sids], k_run[sids], f_ret[sids] = _check_plan(plan, sids, before, zero, zero, True, geometry)
                nw = len(stream_oracle.window_starts(total[i] / float(sr), dur))
                assert k_run[sid_of[i]] == nw and f_ret[sid_of[i]] == (nw - 1) * oi + fpw, (trial, i)
                open_.remove(i)
