"""LiveStreamer on the GPU: audio pushed in arbitrary chunks to many streams at once gives, stream by stream, the
frames of predict_framewise on the whole recording bit for bit and the events of frame_prediction_to_event_prediction
on them, reported push by push as the CPU model of tests/test_live_schedule_model.py reports them."""
import numpy as np
import pytest
import torch

from sed_b200 import streaming, synth
from test_gpu_streaming import DEV, build
from test_live_schedule_model import LiveEvents

pytestmark = pytest.mark.gpu

LENGTHS = (3.1, 5.0, 12.0, 13.4, 60.0)


def recordings(n, sr, dtype, seed):
    recs = []
    for i in range(n):
        L = int(round(LENGTHS[i % len(LENGTHS)] * sr))
        w = synth.synthetic_waveform(1, L, seed=seed + i, kind="events", sample_rate=sr)[0]
        recs.append(torch.round(w * 32767.0).to(torch.int16) if dtype == torch.int16 else w.float())
    return recs


def drive(live, recs, sr, seed, on_device=()):
    """Open the streams at different pushes, feed them in random chunk sizes (1 and 0 samples, odd sizes, 1 s, one
    whole 60 s chunk), close each when its audio is in.  Returns per stream the list of (frames, events) reports."""
    rng = np.random.RandomState(seed)
    sizes = [0, 1, 777, 3333, sr, 2 * sr + 5, sr * 3 // 2]
    pending = list(range(len(recs)))
    active, pos, sid_of, reports = [], {}, {}, {i: [] for i in range(len(recs))}
    whole = {i for i in range(len(recs)) if recs[i].numel() == 60 * sr and i % 2 == 0}
    while pending or active:
        for _ in range(int(rng.randint(0, 4))):
            if pending:
                i = pending.pop(0)
                sid_of[i] = live.open(name="rec%d" % i)
                active.append(i)
                pos[i] = 0
        items = []
        for i in active:
            if rng.rand() < 0.2:
                continue
            n = recs[i].numel() - pos[i] if i in whole else int(rng.choice(sizes))
            chunk = recs[i][pos[i]:pos[i] + n]
            chunk = chunk.to(DEV) if i in on_device else chunk.pin_memory()
            items.append((sid_of[i], chunk))
            pos[i] += chunk.numel()
        res = live.push(items)
        for i in active:
            if sid_of[i] in res:
                r = res[sid_of[i]]
                reports[i].append((r["first_frame"], r["frames"].clone(), r["events"]))
        for i in [i for i in active if pos[i] >= recs[i].numel() and rng.rand() < 0.7]:
            r = live.close(sid_of[i])
            reports[i].append((r["first_frame"], r["frames"].clone(), r["events"], "close"))
            active.remove(i)
    return reports


def by_label(events):
    out = {}
    for e in events:
        out.setdefault(e["event_label"], []).append((e["onset"], e["offset"]))
    return out


CASES = [
    ("Cnn_9layers_Gru_FrameAtt", 16000, torch.int16, 5, 1),
    ("Cnn_9layers_Transformer_FrameAtt", 16000, torch.float32, 5, 1),
    ("Cnn_9layers_Gru_FrameAtt", 32000, torch.float32, 5, 1),
    ("Cnn_9layers_Transformer_FrameAtt", 32000, torch.int16, 5, 1),
    ("Cnn_9layers_Gru_FrameAtt", 8000, torch.int16, 5, 1),
    ("Cnn_9layers_Transformer_FrameAtt", 16000, torch.int16, 5, 0.5),
    ("Cnn_9layers_Gru_FrameAtt", 16000, torch.int16, 6, 1),
]


@pytest.mark.parametrize("mt,sr,dtype,dur,ov", CASES)
def test_live_equals_offline_bitwise(mt, sr, dtype, dur, ov, thresholds):
    model = build(mt, sr)
    recs = recordings(40, sr, dtype, seed=sr + dur)
    params = thresholds["%s/best_logmel_16k.sed.valid.pkl" % mt] if sr == 16000 else None
    live = streaming.LiveStreamer(model, sample_rate=sr, sample_duration=dur, overlap_value=ov, max_streams=48,
                                  dtype=dtype, sed_params=params)
    reports = drive(live, recs, sr, seed=len(mt) + sr, on_device={3, 17})
    p = streaming.DEFAULT_SED_PARAMS if params is None else params
    for i, rec in enumerate(recs):
        ref = streaming.predict_framewise(model, rec.to(DEV), sr, dur, ov)
        got = torch.cat([r[1] for r in reports[i]])
        assert torch.equal(got, ref[0].cpu()), (i, got.shape, ref.shape)
        # frames arrive contiguously, and as soon as they are final
        assert [r[0] for r in reports[i]] == list(np.cumsum([0] + [r[1].shape[0] for r in reports[i]])[:-1])
        # events: label by label equal to the offline extraction on the merged tensor
        ref_ev = streaming.frame_prediction_to_event_prediction(ref, p, audio_names=["rec%d" % i])
        got_ev = [e for r in reports[i] for e in r[2]]
        assert by_label(got_ev) == by_label(ref_ev), i
        assert all(e["filename"] == "rec%d" % i for e in got_ev)
        # push by push: the CPU state machine fed the same finalized frames reports the same events
        fw = ref[0].cpu().numpy()
        hi, lo = p["sed_high_threshold"], p.get("sed_low_threshold")
        for c in range(fw.shape[1]):
            pc = lambda v: v[c] if np.ndim(v) else v
            model_ev = LiveEvents(pc(hi), None if lo is None else pc(lo), pc(p["n_smooth"]), pc(p["n_salt"]))
            for r in reports[i]:
                want = model_ev.feed(fw[r[0]:r[0] + r[1].shape[0], c])
                if len(r) == 4:
                    n = len(model_ev.out)
                    model_ev.close()
                    want = want + model_ev.out[n:]
                lab = streaming.LABELS[c]
                have = [[round(e["onset"] * 100), round(e["offset"] * 100)] for e in r[2] if e["event_label"] == lab]
                assert have == want, (i, c)


def test_live_frames_final_after_each_window():
    """Shipped preset: after the push that runs window k, exactly (k+1)*100 frames have been returned."""
    model = build("Cnn_9layers_Gru_FrameAtt")
    sr = 16000
    rec = recordings(5, sr, torch.int16, seed=3)[4]  # 60 s
    live = streaming.LiveStreamer(model, sample_rate=sr, max_streams=2)
    sid = live.open()
    got = live.push([(sid, rec[:5 * sr])])[sid]
    assert got["frames"].shape[0] == 100
    for k in range(1, 10):
        got = live.push([(sid, rec[(4 + k) * sr:(5 + k) * sr])])[sid]
        assert got["first_frame"] == k * 100 and got["frames"].shape[0] == 100
    live.close(sid)


def test_slot_reuse_equals_fresh_streamer():
    model = build("Cnn_9layers_Gru_FrameAtt")
    sr = 16000
    recs = recordings(5, sr, torch.int16, seed=11)
    long_rec, short_rec = recs[4], recs[0]   # 60 s, then 3.1 s in the same slot

    def run(live, rec):
        sid = live.open()
        out = [live.push([(sid, rec)])[sid]]
        out.append(live.close(sid))
        return sid, torch.cat([o["frames"] for o in out]), [e for o in out for e in o["events"]]

    used = streaming.LiveStreamer(model, sample_rate=sr, max_streams=1)
    run(used, long_rec)
    sid, frames, events = run(used, short_rec)
    fresh = streaming.LiveStreamer(model, sample_rate=sr, max_streams=1)
    sid2, frames2, events2 = run(fresh, short_rec)
    assert sid == sid2 == 0
    assert torch.equal(frames, frames2)
    assert events == events2
    ref = streaming.predict_framewise(model, short_rec.to(DEV), sr)
    assert torch.equal(frames, ref[0].cpu())


def test_live_errors():
    model = build("Cnn_9layers_Gru_FrameAtt")
    live = streaming.LiveStreamer(model, sample_rate=16000, max_streams=2, dtype=torch.int16)
    a = live.open()
    live.open()
    with pytest.raises(RuntimeError, match="all 2 streams"):
        live.open()
    with pytest.raises(TypeError):
        live.push([(a, torch.zeros(10, dtype=torch.float32))])
    with pytest.raises(ValueError, match="1-D"):
        live.push([(a, torch.zeros(2, 10, dtype=torch.int16))])
    live.close(a)
    with pytest.raises(ValueError, match="not open"):
        live.push([(a, torch.zeros(10, dtype=torch.int16))])
    with pytest.raises(ValueError, match="not open"):
        live.push([(7, torch.zeros(10, dtype=torch.int16))])
    with pytest.raises(ValueError, match="not open"):
        live.close(a)
    with pytest.raises(ValueError):
        streaming.LiveStreamer(model, sample_rate=16000, dtype=torch.float64)
