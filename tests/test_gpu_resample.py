"""Resampling and downmix on the GPU (csrc/sed_resample.cu): sed_resample against float64 references, the
resampling HostStreamer and LiveStreamer against the offline path on resample()'d audio, the default arguments
against today's path, and the argument checks."""
import numpy as np
import pytest
import scipy.signal
import torch

from sed_b200 import capi, engine, streaming, synth
from test_gpu_streaming import DEV, build

pytestmark = pytest.mark.gpu

ROLLOFF, BETA = 0.9475937167399596, 14.769656459379492
RATE_PAIRS = [(48000, 16000), (48000, 32000), (48000, 8000), (44100, 16000), (44100, 32000), (22050, 16000),
              (96000, 32000), (8000, 16000)]


def source(n, channels, dtype, seed):
    """[n, channels] (or [n] for one channel) CPU waveform with |x| <= 1: events plus full-scale noise."""
    g = torch.Generator().manual_seed(seed)
    w = synth.synthetic_waveform(channels, max(n, 1), seed=seed, kind="events")[:, :n].T.contiguous()
    w = (0.7 * w + 0.3 * (torch.rand(w.shape, generator=g) * 2 - 1)).clamp(-1, 1)
    w = torch.round(w * 32767.0).to(torch.int16) if dtype == torch.int16 else w.float()
    return w[:, 0].contiguous() if channels == 1 else w


def downmix_np(rec):
    """numpy's x.astype(float32).mean(axis=1) (int16: (q / 32767.).astype(float32))."""
    a = rec.numpy()
    a = (a / 32767.).astype(np.float32) if a.dtype == np.int16 else a
    return a if a.ndim == 1 else a.mean(axis=1)


def check_against_references(y, x32, up, down, taps, in_rate, out_rate, what):
    """y: device output (float32 numpy); x32: the float32 downmixed input."""
    x = x32.astype(np.float64)
    t64 = taps.astype(np.float64)
    ref = scipy.signal.resample_poly(x, up, down, window=t64 / up)
    mag = scipy.signal.resample_poly(np.abs(x), up, down, window=np.abs(t64) / up)
    assert y.shape == ref.shape, (what, y.shape, ref.shape)
    rel = np.abs(y - ref) / np.maximum(mag, 1e-30)
    assert rel.max() <= 2.0 ** -18, (what, rel.max())
    h = scipy.signal.firwin(2 * (len(taps) // 2) + 1, ROLLOFF / max(up, down), window=("kaiser", BETA))
    exact = scipy.signal.resample_poly(x, up, down, window=h)
    assert np.abs(y - exact).max() <= 2e-6, (what, np.abs(y - exact).max())
    return float(rel.max()), float(np.abs(y - exact).max())


@pytest.mark.parametrize("in_rate,out_rate", RATE_PAIRS)
def test_resample_against_float64_reference(in_rate, out_rate):
    up, down, half, taps = engine.resample_filter(in_rate, out_rate)
    short = max(1, (2 * half + 1) // up - 3)
    lengths = [1, short, 12345]
    if (in_rate, out_rate) in ((48000, 16000), (44100, 32000)):
        lengths.append(61 * in_rate)
    worst = [0.0, 0.0]
    for C in (1, 2, 6):
        for dtype in (torch.int16, torch.float32):
            recs = [source(n, C, dtype, seed=n + C) for n in lengths]
            got = streaming.resample([r.to(DEV) for r in recs], in_rate, out_rate, channels=C)  # a ragged batch
            assert len(got) == len(recs)
            for r, y in zip(recs, got):
                n = r.shape[0]
                assert y.dtype == torch.float32 and y.shape == (-(-n * up // down),)
                e = check_against_references(y.cpu().numpy(), downmix_np(r), up, down, taps, in_rate, out_rate,
                                             (C, dtype, n))
                worst = [max(a, b) for a, b in zip(worst, e)]
    print("%d -> %d: max error / sum|terms| = 2^%.1f, max |error| vs float64 taps = %.2e"
          % (in_rate, out_rate, np.log2(max(worst[0], 1e-300)), worst[1]))


@pytest.mark.parametrize("C", [1, 2, 6, 8])
def test_downmix_equals_numpy_mean_bitwise(C):
    """Equal rates only downmix: the float32 result is numpy's mean(axis=1), bit for bit (C = 8 included, where numpy
    sums pairwise)."""
    for dtype in (torch.int16, torch.float32):
        rec = source(50001, C, dtype, seed=C)
        if dtype == torch.float32:
            rec = rec * torch.logspace(-6, 3, rec.shape[0])[:, None] if C > 1 else rec
        y = streaming.resample([rec.to(DEV)], 16000, 16000, channels=C)[0].cpu().numpy()
        want = downmix_np(rec)
        assert np.array_equal(y.view(np.int32), want.view(np.int32)), (C, dtype)


def test_table_rows_write_only_their_samples():
    """One launch, ragged rows laid out with gaps: samples outside the rows keep a NaN sentinel."""
    plan = engine.resample_plan(44100, 16000, DEV)
    recs = [source(n, 2, torch.int16, seed=n) for n in (1, 4410, 777, 44100)]
    src = torch.cat([r.reshape(-1) for r in recs]).to(DEV)
    n_in = np.array([r.shape[0] for r in recs])
    n_out = plan.n_out(n_in)
    d0 = np.cumsum(n_out + 13) - n_out
    table = np.stack([np.cumsum(n_in) - n_in, n_in, d0, n_out], 1)
    dst = torch.full((int(d0[-1] + n_out[-1] + 29),), float("nan"), device=DEV)
    engine.resample(src, 2, torch.from_numpy(table).to(DEV), len(recs), int(n_out.max()), plan, dst)
    y = dst.cpu().numpy()
    mask = np.zeros(y.size, bool)
    for a, n, r in zip(d0, n_out, recs):
        mask[a:a + n] = True
        want = streaming.resample([r.to(DEV)], 44100, 16000, channels=2)[0].cpu().numpy()
        assert np.array_equal(y[a:a + n], want)
    assert np.isnan(y[~mask]).all() and not np.isnan(y[mask]).any()


# ---------------------------------------------------------------------------------------------------------------
# the defaults run today's path
# ---------------------------------------------------------------------------------------------------------------
def test_defaults_are_todays_path():
    mt, sr = "Cnn_9layers_Gru_FrameAtt", 16000
    model = build(mt, sr)
    recs = [source(int(d * sr), 1, torch.int16, seed=i) for i, d in enumerate((7.3, 3.1, 12.0))]
    want = [streaming.predict_framewise(model, r.to(DEV), sr).cpu() for r in recs]
    for kw in ({}, {"input_rate": sr, "channels": 1}):
        st = streaming.HostStreamer(model, sr, **kw)
        assert not st.resampling
        st.submit([r.pin_memory() for r in recs], DEV)
        for g, w in zip(st.result(), want):
            assert torch.equal(g, w)
        live = streaming.LiveStreamer(model, sample_rate=sr, max_streams=4, dtype=torch.int16, **kw)
        assert live.arena.dtype == torch.int16 and not live.resampling
        sid = live.open()
        out = [live.push([(sid, recs[2][:5 * sr + 7])])[sid], live.push([(sid, recs[2][5 * sr + 7:])])[sid]]
        out.append(live.close(sid))
        assert torch.equal(torch.cat([o["frames"] for o in out]), want[2][0])


# ---------------------------------------------------------------------------------------------------------------
# HostStreamer with resampling
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("in_rate,C,dtype", [(44100, 2, torch.int16), (48000, 1, torch.float32)])
def test_host_streamer_resampling(in_rate, C, dtype):
    mt, sr = "Cnn_9layers_Gru_FrameAtt", 16000
    model = build(mt, sr)
    recs = [source(int(d * in_rate), C, dtype, seed=30 + i) for i, d in enumerate((7.3, 12.0, 3.1, 5.0))]
    st = streaming.HostStreamer(model, sr, 5, 1, input_rate=in_rate, channels=C)
    st.submit([r.pin_memory() for r in recs], DEV)
    st.submit([r.pin_memory() for r in recs[::-1]], DEV)
    got, got_rev = st.result(), st.result()
    rs = streaming.resample([r.to(DEV) for r in recs], in_rate, sr, channels=C)
    want = streaming.predict_framewise_many(model, rs, sr, 5, 1)
    gap = 0.0
    for i, r in enumerate(recs):
        assert torch.equal(got[i], want[i].cpu()) and torch.equal(got_rev[len(recs) - 1 - i], want[i].cpu()), i
        g = np.gcd(in_rate, sr)
        n_taps, cutoff, window = _firwin_args(in_rate, sr)
        x = scipy.signal.resample_poly(downmix_np(r).astype(np.float64), sr // g, in_rate // g,
                                       window=scipy.signal.firwin(n_taps, cutoff, window=window))
        ref = streaming.predict_framewise(model, torch.from_numpy(x.astype(np.float32)).to(DEV), sr).cpu()
        gap = max(gap, (got[i] - ref).abs().max().item())
        assert gap <= 2e-3, (i, gap)
    print("HostStreamer %d Hz x%d: max |p - p(scipy float64 resampling)| = %.2e" % (in_rate, C, gap))


def _firwin_args(in_rate, out_rate):
    g = np.gcd(in_rate, out_rate)
    mx = max(in_rate // g, out_rate // g)
    return 2 * 64 * mx + 1, ROLLOFF / mx, ("kaiser", BETA)


# ---------------------------------------------------------------------------------------------------------------
# LiveStreamer with resampling
# ---------------------------------------------------------------------------------------------------------------
def drive_frames(live, recs, in_rate, down, seed):
    """drive() of tests/test_gpu_live.py for [n] / [n, C] chunks: positions count frames (shape[0]).  Streams open at
    different pushes, get random chunk sizes (0, 1, down - 1 frames, odd sizes, 1 s, several seconds) and close when
    their audio is in; with fewer slots than streams, slots are reused."""
    rng = np.random.RandomState(seed)
    sizes = [0, 1, down - 1, 777, in_rate, 2 * in_rate + 5, in_rate * 3 // 2]
    pending = list(range(len(recs)))
    active, pos, sid_of, reports = [], {}, {}, {i: [] for i in range(len(recs))}
    while pending or active:
        for _ in range(int(rng.randint(0, 3))):
            if pending and len(active) < live.max_streams:
                i = pending.pop(0)
                sid_of[i] = live.open(name="rec%d" % i)
                active.append(i)
                pos[i] = 0
        items = []
        for i in active:
            if rng.rand() < 0.2:
                continue
            chunk = recs[i][pos[i]:pos[i] + int(rng.choice(sizes))]
            items.append((sid_of[i], chunk.pin_memory() if i % 3 else chunk.to(DEV)))
            pos[i] += chunk.shape[0]
        res = live.push(items)
        for i in active:
            if sid_of[i] in res:
                r = res[sid_of[i]]
                reports[i].append((r["first_frame"], r["frames"].clone(), r["events"]))
        for i in [i for i in active if pos[i] >= recs[i].shape[0] and rng.rand() < 0.7]:
            r = live.close(sid_of[i])
            reports[i].append((r["first_frame"], r["frames"].clone(), r["events"], "close"))
            active.remove(i)
    return reports


def by_label(events):
    out = {}
    for e in events:
        out.setdefault(e["event_label"], []).append((e["onset"], e["offset"]))
    return out


@pytest.mark.parametrize("mt", ["Cnn_9layers_Gru_FrameAtt", "Cnn_9layers_Transformer_FrameAtt"])
@pytest.mark.parametrize("in_rate,C,dtype", [(48000, 2, torch.int16), (44100, 1, torch.float32)])
def test_live_resampling_equals_offline_bitwise(mt, in_rate, C, dtype):
    sr = 16000
    model = build(mt, sr)
    recs = [source(int(d * in_rate) + i, C, dtype, seed=50 + i) for i, d in enumerate((3.1, 5.0, 12.0, 0.2, 13.4, 7.7))]
    live = streaming.LiveStreamer(model, sample_rate=sr, max_streams=3, dtype=dtype, input_rate=in_rate, channels=C)
    assert live.arena.dtype == torch.float32
    reports = drive_frames(live, recs, in_rate, live.rs.down, seed=in_rate + C)
    p = streaming.DEFAULT_SED_PARAMS
    for i, rec in enumerate(recs):
        x = streaming.resample([rec.to(DEV)], in_rate, sr, channels=C)[0]
        ref = streaming.predict_framewise(model, x, sr)
        got = torch.cat([r[1] for r in reports[i]])
        assert torch.equal(got, ref[0].cpu()), (i, got.shape, ref.shape)
        assert [r[0] for r in reports[i]] == list(np.cumsum([0] + [r[1].shape[0] for r in reports[i]])[:-1])
        ref_ev = streaming.frame_prediction_to_event_prediction(ref, p, audio_names=["rec%d" % i])
        assert by_label([e for r in reports[i] for e in r[2]]) == by_label(ref_ev), i


# ---------------------------------------------------------------------------------------------------------------
# argument checks: ValueError before anything is launched
# ---------------------------------------------------------------------------------------------------------------
def test_errors_before_any_launch():
    model = build("Cnn_9layers_Gru_FrameAtt", 16000)
    live = streaming.LiveStreamer(model, sample_rate=16000, max_streams=2, input_rate=48000, channels=2)
    sid = live.open()
    st = streaming.HostStreamer(model, 16000, input_rate=44100, channels=2)
    torch.cuda.synchronize()
    capi.reset_launches()
    stereo = torch.zeros(100, 2, dtype=torch.int16)
    bad = [
        lambda: streaming.resample([stereo.to(DEV)], 48000, 44101, channels=2),      # max(up, down) > 4096
        lambda: streaming.resample([stereo.to(DEV)], 0, 16000, channels=2),          # rate out of range
        lambda: streaming.HostStreamer(model, 16000, input_rate=48000 * 7 + 1),
        lambda: streaming.LiveStreamer(model, sample_rate=16000, input_rate=400000),
        lambda: streaming.resample([stereo.to(DEV)], 48000, 16000, channels=0),
        lambda: streaming.resample([stereo.to(DEV)], 48000, 16000, channels=9),
        lambda: streaming.LiveStreamer(model, sample_rate=16000, channels=9),
        lambda: streaming.HostStreamer(model, 16000, channels=0),
        lambda: streaming.resample([stereo.to(DEV)], 48000, 16000, channels=1),      # trailing dimension
        lambda: streaming.resample([stereo[:, 0].to(DEV)], 48000, 16000, channels=2),
        lambda: streaming.resample([stereo.to(DEV), stereo.float().to(DEV)], 48000, 16000, channels=2),  # dtypes
        lambda: live.push([(sid, torch.zeros(100, 3, dtype=torch.int16))]),
        lambda: live.push([(sid, torch.zeros(100, dtype=torch.int16))]),
        lambda: st.submit([stereo, torch.zeros(100, 3, dtype=torch.int16)], DEV),
        lambda: st.submit([stereo, stereo.float()], DEV),
    ]
    for k, f in enumerate(bad):
        with pytest.raises(ValueError):
            f()
        assert capi.launches() == 0, k
    assert live.n_in[sid] == 0 and live.n_samples[sid] == 0
