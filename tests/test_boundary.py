"""Drop-in boundary: constructors, state_dict layout, checkpoint format, error behaviour (CPU-only checks)."""
import inspect

import pytest
import torch

from conftest import synthetic_sd
from sed_b200 import models, stft, streaming, synth


@pytest.mark.parametrize("mt", synth.MODEL_TYPES)
def test_state_dict_layout_matches_reference(mt, golden_meta):
    """Keys, order and shapes equal the reference model's state_dict (SURVEY.md 8b; fixture from the reference)."""
    want = golden_meta["state_dict_keys"][mt]
    model = getattr(models, mt)(16000, 512, 160, 64, 25, 7000, 25, "logmel")
    got = {k: list(v.shape) for k, v in model.state_dict().items()}
    assert list(got.keys()) == list(want.keys())
    assert got == want
    assert len(got) == (73 if "Gru" in mt else 75)


@pytest.mark.parametrize("mt", synth.MODEL_TYPES)
def test_constructor_signature(mt):
    sig = inspect.signature(getattr(models, mt).__init__)
    assert list(sig.parameters)[1:] == ["sample_rate", "window_size", "hop_size", "mel_bins", "fmin", "fmax",
                                        "classes_num", "feature_type"]


def test_frontend_constructor_defaults():
    s = inspect.signature(stft.Spectrogram.__init__).parameters
    assert [s[k].default for k in ("n_fft", "hop_length", "win_length", "window", "center", "pad_mode", "power",
                                   "freeze_parameters")] == [2048, None, None, "hann", True, "reflect", 2.0, True]
    m = inspect.signature(stft.LogmelFilterBank.__init__).parameters
    assert [m[k].default for k in ("sr", "n_fft", "n_mels", "fmin", "fmax", "is_log", "ref", "amin", "top_db",
                                   "freeze_parameters")] == [22050, 2048, 64, 0.0, None, True, 1.0, 1e-10, 80.0, True]
    sp = stft.Spectrogram(n_fft=512)
    assert sp.stft.hop_length == 128 and sp.stft.win_length == 512  # stft.py:185-190 defaults
    with pytest.raises(AssertionError):
        stft.Spectrogram(n_fft=512, pad_mode="edge")  # stft.py:175
    assert all(not p.requires_grad for p in sp.parameters())


@pytest.mark.parametrize("mt", synth.MODEL_TYPES)
def test_checkpoint_roundtrip_reference_format(mt, tmp_path):
    """{'iteration','model','optimizer'} file (main_strong.py:326-333) strict-loads (predict.py:232-233)."""
    ck = {"iteration": 0, "model": synthetic_sd(mt), "optimizer": {}}
    path = tmp_path / "best_logmel_16k.pth"
    torch.save(ck, path)
    loaded = torch.load(path, map_location="cpu")
    model = getattr(models, mt)(16000, 512, 160, 64, 25, 7000, 25, "logmel")
    res = model.load_state_dict(loaded["model"])  # strict
    assert not res.missing_keys and not res.unexpected_keys
    bad = dict(loaded["model"])
    bad.pop("bn0.weight")
    with pytest.raises(RuntimeError):
        model.load_state_dict(bad)


def test_refuses_training_mode_and_cpu_inputs():
    model = models.Cnn_9layers_Gru_FrameAtt(16000, 512, 160, 64, 25, 7000, 25, "logmel")
    wave, clips = torch.zeros(16000), torch.zeros(2, 160000)
    streaming_entries = [lambda: streaming.predict_framewise(model, wave, 16000),
                         lambda: streaming.predict_framewise_many(model, [wave, wave], 16000),
                         lambda: streaming.predict_framewise_overlap(model, clips, 16000, 5, 1),
                         lambda: streaming.HostStreamer(model, 16000).submit([wave], "cpu"),
                         lambda: streaming.LiveStreamer(model, 16000),
                         lambda: streaming.LiveStreamer(model, 16000, device="cpu")]
    with pytest.raises(RuntimeError, match="inference only"):
        model(torch.zeros(1, 16000))
    for entry in streaming_entries:
        with pytest.raises(RuntimeError, match="inference only"):
            entry()
    model.eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model(torch.zeros(1, 16000))
    for entry in streaming_entries:
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            entry()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        stft.Spectrogram(n_fft=512, hop_length=160)(torch.zeros(1, 16000))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        stft.LogmelFilterBank(sr=16000, n_fft=512)(torch.zeros(1, 10, 257))
    with pytest.raises(NotImplementedError):
        models.Cnn_9layers_Gru_FrameAtt(16000, 512, 160, 64, 25, 7000, 25, "gamma")


def test_module_names_resolve_like_reference():
    """Callers do `from models import *` then eval(model_type) (main_strong.py:33, 529)."""
    ns = {}
    exec("from sed_b200.models import *", ns)
    for name in synth.MODEL_TYPES:
        assert name in ns


def test_model_can_be_deep_copied_and_pickled():
    import copy
    import pickle
    model = models.Cnn_9layers_Gru_FrameAtt(16000, 512, 160, 64, 25, 7000, 25, "logmel")
    clone = copy.deepcopy(model)
    assert clone._packed == {} and clone._packed is not model._packed
    again = pickle.loads(pickle.dumps(model))
    assert list(again.state_dict().keys()) == list(model.state_dict().keys())


def test_full_state_matches_state_dict_and_survives_replication():
    """DataParallel replicas keep their parameters as plain attributes (state_dict() there has buffers only)."""
    model = models.Cnn_9layers_Transformer_FrameAtt(16000, 512, 160, 64, 25, 7000, 25, "logmel")
    full = model._full_state()
    sd = model.state_dict()
    assert list(full.keys()) == list(sd.keys())
    replica = model._replicate_for_data_parallel()
    replica._former_parameters = dict(replica._parameters)
    replica._parameters = {}
    assert "bn0.weight" in replica._full_state()
    assert replica._packed is model._packed and replica._pack_lock is model._pack_lock
