"""Drop-in `Cnn_9layers_Gru_FrameAtt` / `Cnn_9layers_Transformer_FrameAtt`
(reference: pytorch/models.py:564-688 and :981-1077) running on the B200 kernels.

Same 8-argument constructors, same sub-module names -- hence the same `state_dict` keys/shapes, so
reference checkpoints (`torch.load(path)['model']`) strict-load -- and the same output dict
`{'framewise_output', 'clipwise_output', 'embedding'}`.  Inference only: the training-time branches of
the reference forward (SpecAugment / mixup / timeshift, models.py:647-661) are not built and
`forward` refuses to run in training mode.  Inputs must be CUDA tensors; there is no CPU fallback.
"""
import math
import threading
import weakref

import torch
import torch.nn as nn

from . import engine
from .stft import LogmelFilterBank, Spectrogram

__all__ = ["Cnn_9layers_Gru_FrameAtt", "Cnn_9layers_Transformer_FrameAtt", "Cnn_9layers_FrameMax",
           "Cnn_9layers_FrameAvg", "Cnn_9layers_FrameAtt", "Cnn_9layers_Gru_FrameAvg",
           "Cnn_9layers_Transformer_FrameAvg", "ConvBlock", "AttBlock", "MultiHead", "Spectrogram",
           "LogmelFilterBank"]


def _xavier(layer):
    nn.init.xavier_uniform_(layer.weight)
    if getattr(layer, "bias", None) is not None:
        layer.bias.data.fill_(0.)


class ConvBlock(nn.Module):
    """Parameters of reference ConvBlock (models.py:98-123): two bias-free 3x3 convs, two BatchNorms."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.conv1 = nn.Conv2d(in_channels, out_channels, (3, 3), (1, 1), (1, 1), bias=False)
        self.conv2 = nn.Conv2d(out_channels, out_channels, (3, 3), (1, 1), (1, 1), bias=False)
        self.bn1 = nn.BatchNorm2d(out_channels)
        self.bn2 = nn.BatchNorm2d(out_channels)
        _xavier(self.conv1)
        _xavier(self.conv2)


class AttBlock(nn.Module):
    """Parameters of reference AttBlock (models.py:144-159); `bn_att` exists but is never applied."""

    def __init__(self, n_in, n_out, activation='linear', temperature=1.):
        super().__init__()
        self.activation = activation
        self.temperature = temperature
        self.att = nn.Conv1d(n_in, n_out, 1, bias=True)
        self.cla = nn.Conv1d(n_in, n_out, 1, bias=True)
        self.bn_att = nn.BatchNorm1d(n_out)
        _xavier(self.att)
        _xavier(self.cla)


class MultiHead(nn.Module):
    """Parameters of reference MultiHead (models.py:823-850); `layer_norm` exists but is never applied."""

    def __init__(self, n_head, d_model, d_k, d_v, dropout=0.1):
        super().__init__()
        self.n_head, self.d_k, self.d_v = n_head, d_k, d_v
        self.w_qs = nn.Linear(d_model, n_head * d_k)
        self.w_ks = nn.Linear(d_model, n_head * d_k)
        self.w_vs = nn.Linear(d_model, n_head * d_v)
        for lin, d in ((self.w_qs, d_k), (self.w_ks, d_k), (self.w_vs, d_v)):
            nn.init.normal_(lin.weight, mean=0, std=math.sqrt(2.0 / (d_model + d)))
            lin.bias.data.fill_(0)
        self.layer_norm = nn.LayerNorm(d_model)
        self.fc = nn.Linear(n_head * d_v, d_model)
        nn.init.xavier_normal_(self.fc.weight)
        self.fc.bias.data.fill_(0)


class _Cnn9Base(nn.Module):
    MODEL_TYPE = None

    def __init__(self, sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num, feature_type='logmel'):
        super().__init__()
        if feature_type != 'logmel':
            raise NotImplementedError("feature_type=%r: only 'logmel' is built (SURVEY.md 8a)" % (feature_type,))
        self.feature_type = feature_type
        self.window_size, self.hop_size = window_size, hop_size
        self.spectrogram_extractor = Spectrogram(n_fft=window_size, hop_length=hop_size, win_length=window_size,
                                                 window='hann', center=True, pad_mode='reflect',
                                                 freeze_parameters=True)
        self.logmel_extractor = LogmelFilterBank(sr=sample_rate, n_fft=window_size, n_mels=mel_bins, fmin=fmin,
                                                 fmax=fmax, ref=1.0, amin=1e-10, top_db=None, freeze_parameters=True)
        self.bn0 = nn.BatchNorm2d(64)
        self.conv_block1 = ConvBlock(1, 64)
        self.conv_block2 = ConvBlock(64, 128)
        self.conv_block3 = ConvBlock(128, 256)
        self.conv_block4 = ConvBlock(256, 512)
        # engine state shared (by reference) with DataParallel replicas
        self._packed = {}
        self._generation = [0]
        self._pack_lock = threading.RLock()
        self._master_ref = [weakref.ref(self)]  # DataParallel replicas copy __dict__: they find the master through it
        self.precision = "fp16"   # 16-bit operand type of the tensor-core layers: 'fp16' or 'bf16'
        self.micro_batch = engine.DEFAULT_MICRO_BATCH   # clips per conv-stack launch group (whole waves of the 148 SMs)
        self.conv_variant = 4   # 4 = conv_block1 as one tensor-core kernel (default); 2 = conv_block1 as two kernels
        # (conv1 writes its 64-channel output to memory); every other conv layer runs on CTA pairs either way

    # any parameter movement / reload invalidates the packed copies
    def _invalidate(self):
        self._generation[0] += 1

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self._invalidate()
        return out

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._invalidate()
        return out

    # the engine state (device copies, lock) is not part of the module's value: copy / pickle rebuild it lazily
    def __getstate__(self):
        state = dict(self.__dict__)
        state["_packed"] = {}
        state["_generation"] = [0]
        state.pop("_pack_lock", None)
        state.pop("_master_ref", None)
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self._pack_lock = threading.RLock()
        self._master_ref = [weakref.ref(self)]

    def _full_state(self):
        """state_dict()-like view that also works on DataParallel replicas, whose parameters are plain attributes
        (torch.nn.parallel.replicate keeps them in `_former_parameters`, so `state_dict()` there returns buffers only)."""
        sd = {}
        for prefix, mod in self.named_modules():
            params = dict(mod._parameters)
            params.update(getattr(mod, "_former_parameters", {}))
            for k, v in list(params.items()) + list(mod._buffers.items()):
                if v is not None and k not in mod._non_persistent_buffers_set:
                    sd[(prefix + "." if prefix else "") + k] = v
        return sd

    def _signature(self):
        """Cheap fingerprint of every parameter / buffer: storage pointer and in-place version counter.  In-place edits
        (`p.data.copy_()`, `p.mul_()` under no_grad, manual BatchNorm-statistics updates) bump `_version`, `.to()` /
        `load_state_dict` change pointers or versions: either way the packed copies are rebuilt on the next call."""
        master = self._master_ref[0]() or self  # a replica's own tensors are fresh broadcast copies on every call
        return (self._generation[0],) + tuple((v.data_ptr(), v._version) for v in master._full_state().values())

    def _packed_for(self, device):
        key = (device.type, device.index, self.precision)
        sig = self._signature()
        hit = self._packed.get(key)
        if hit is None or hit[0] != sig:
            with self._pack_lock:  # DataParallel runs one thread per replica; they share _packed by reference
                hit = self._packed.get(key)
                if hit is None or hit[0] != sig:
                    hit = (sig, engine.PackedModel(self._full_state(), self.MODEL_TYPE, self.window_size,
                                                   self.hop_size, device, self.precision))
                    self._packed[key] = hit
        return hit[1]

    def forward(self, input, mixup_lambda=None, timeshift=False, spec_augment=True):
        """input (batch_size, data_length) float32 CUDA tensor -> output dict."""
        if self.training:
            raise RuntimeError("%s: inference only -- call .eval() (training branches models.py:647-661 are "
                               "out of scope)" % type(self).__name__)
        if not input.is_cuda:
            raise RuntimeError("%s: input is on %s; the B200 path has no CPU fallback" % (type(self).__name__,
                                                                                         input.device))
        with torch.no_grad():
            packed = self._packed_for(input.device)
            return packed.forward(input, micro_batch=self.micro_batch, variant=self.conv_variant)


def _make_gru():
    """nn.GRU(512, 256, bidirectional) with the distributions of reference init_gru (models.py:35-60)."""
    gru = nn.GRU(input_size=512, hidden_size=256, num_layers=1, bias=True, batch_first=True, bidirectional=True)
    for name, p in gru.named_parameters():
        if "bias" in name:
            nn.init.constant_(p, 0)
        else:
            fan_in = p.shape[1]
            for g in range(3):
                blk = p.data[g * 256:(g + 1) * 256]
                if "weight_hh" in name and g == 2:
                    nn.init.orthogonal_(blk)
                else:
                    nn.init.uniform_(blk, -math.sqrt(3 / fan_in), math.sqrt(3 / fan_in))
    return gru


def _make_fc(classes_num):
    fc = nn.Linear(512, classes_num, bias=True)
    _xavier(fc)
    return fc


class Cnn_9layers_Gru_FrameAtt(_Cnn9Base):
    MODEL_TYPE = "Cnn_9layers_Gru_FrameAtt"

    def __init__(self, sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num, feature_type):
        super().__init__(sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num, feature_type)
        self.gru = _make_gru()
        self.att_block = AttBlock(n_in=512, n_out=25, activation='sigmoid')  # 25 is hard-coded (models.py:617)


class Cnn_9layers_Transformer_FrameAtt(_Cnn9Base):
    MODEL_TYPE = "Cnn_9layers_Transformer_FrameAtt"

    def __init__(self, sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num, feature_type='logmel'):
        super().__init__(sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num, feature_type)
        self.multihead = MultiHead(8, 512, 64, 64, 0.2)
        self.att_block = AttBlock(n_in=512, n_out=25, activation='sigmoid')


# ---------------------------------------------------------------------------------------------------------
# Sibling heads on the same trunk (SURVEY.md 8f-4).  Constructor signatures as in the reference: the three
# heads without a temporal block take 7 arguments (no feature_type), the Gru / Transformer ones take 8.
# ---------------------------------------------------------------------------------------------------------
class Cnn_9layers_FrameMax(_Cnn9Base):
    """pytorch/models.py:213-295: sigmoid(fc(x)) per frame, x8 interpolation, clipwise = max over frames."""
    MODEL_TYPE = "Cnn_9layers_FrameMax"

    def __init__(self, sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num):
        super().__init__(sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num)
        self.fc = _make_fc(classes_num)


class Cnn_9layers_FrameAvg(_Cnn9Base):
    """pytorch/models.py:298-380: as FrameMax with clipwise = mean over frames."""
    MODEL_TYPE = "Cnn_9layers_FrameAvg"

    def __init__(self, sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num):
        super().__init__(sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num)
        self.fc = _make_fc(classes_num)


class Cnn_9layers_FrameAtt(_Cnn9Base):
    """pytorch/models.py:383-463: AttBlock directly on the conv features; framewise is not padded."""
    MODEL_TYPE = "Cnn_9layers_FrameAtt"

    def __init__(self, sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num):
        super().__init__(sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num)
        self.att_block = AttBlock(n_in=512, n_out=25, activation='sigmoid')


class Cnn_9layers_Gru_FrameAvg(_Cnn9Base):
    """pytorch/models.py:466-561: bi-GRU then the FrameAvg head."""
    MODEL_TYPE = "Cnn_9layers_Gru_FrameAvg"

    def __init__(self, sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num, feature_type):
        super().__init__(sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num, feature_type)
        self.gru = _make_gru()
        self.fc = _make_fc(classes_num)


class Cnn_9layers_Transformer_FrameAvg(_Cnn9Base):
    """pytorch/models.py:880-978: MultiHead then the FrameAvg head."""
    MODEL_TYPE = "Cnn_9layers_Transformer_FrameAvg"

    def __init__(self, sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num, feature_type):
        super().__init__(sample_rate, window_size, hop_size, mel_bins, fmin, fmax, classes_num, feature_type)
        self.multihead = MultiHead(8, 512, 64, 64, 0.2)
        self.fc = _make_fc(classes_num)
