"""Host-side engine: packs a reference-layout `state_dict` once per device and drives the C ABI.

Data layout in HBM (all allocations are torch tensors; the C ABI only sees raw pointers):
  waveform [B, L] f32 -> log-mel(+bn0) [mb, T, 64] f32 -> conv activations NHWC 16-bit
  ([mb,T,64,64] -> [mb,T/2,32,64] -> ... -> [mb,T/8,8,512]) -> freq-mean features [B, T', 512] 16-bit
  -> GRU: gi [B,T',1536] f32 -> h [B,T',512] f32 | MHA: qkv [B,T',1536] f32 -> ctx 16-bit -> fc [B,T',512] f32
  -> clipwise [B,25], framewise [B,frames,25], embedding.
The conv stack runs over micro-batches (default cap 1036 clips = seven per SM: every layer's tile count is then a
multiple of the persistent grid, and fewer launches mean fewer drain / fill gaps between the persistent kernels; a
batch of 1024 is one launch group with a 14.5 GB activation workspace); the temporal block and the head run once over
the batch.
"""
import collections
import ctypes
import functools
import math
import threading

import numpy as np
import torch

from . import capi


def _on_device(fn):
    """Run a PackedModel method with the model's GPU as the current CUDA device: kernels launched through the C ABI,
    `cudaFuncSetAttribute` and the SM-count queries act on the CURRENT device, so a model living on cuda:1 must not
    depend on the caller having selected it (the reference works from any current device)."""
    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)
    return wrapper


def _on_device_of(argname_index):
    """Same guard for the module-level helpers: the device is the one of positional argument `argname_index`."""
    def deco(fn):
        @functools.wraps(fn)
        def wrapper(*args, **kwargs):
            with torch.cuda.device(args[argname_index].device):
                return fn(*args, **kwargs)
        return wrapper
    return deco

CONV_LAYERS = (
    # name, cin, cout, mode
    ("conv_block1.conv2", 64, 64, capi.CONV_POOL),
    ("conv_block2.conv1", 64, 128, capi.CONV_STORE),
    ("conv_block2.conv2", 128, 128, capi.CONV_POOL),
    ("conv_block3.conv1", 128, 256, capi.CONV_STORE),
    ("conv_block3.conv2", 256, 256, capi.CONV_POOL),
    ("conv_block4.conv1", 256, 512, capi.CONV_STORE),
    ("conv_block4.conv2", 512, 512, capi.CONV_FREQMEAN),
)

# clips per conv-stack launch group: 28 x 37 = seven whole waves of 148 persistent CTAs for every layer
DEFAULT_MICRO_BATCH = 1036

_DTYPES = {"fp16": (capi.SED_DTYPE_F16, torch.float16), "bf16": (capi.SED_DTYPE_BF16, torch.bfloat16)}

# model_type -> (temporal block, pooling head); the trunk (front-end + conv stack) is shared.
#   temporal: 'gru' (models.py:614-615) | 'mha' (models.py:1015-1020) | None
#   head: 'att' = AttBlock (models.py:144-175) | 'avg' / 'max' = Linear + sigmoid + mean / max over frames
MODEL_PLANS = {
    "Cnn_9layers_Gru_FrameAtt": ("gru", "att"),            # models.py:564-688
    "Cnn_9layers_Transformer_FrameAtt": ("mha", "att"),    # models.py:981-1077
    "Cnn_9layers_FrameMax": (None, "max"),                 # models.py:213-295
    "Cnn_9layers_FrameAvg": (None, "avg"),                 # models.py:298-380
    "Cnn_9layers_FrameAtt": (None, "att"),                 # models.py:383-463
    "Cnn_9layers_Gru_FrameAvg": ("gru", "avg"),            # models.py:466-561
    "Cnn_9layers_Transformer_FrameAvg": ("mha", "avg"),    # models.py:880-978
}


def fold_bn(sd, prefix, eps=1e-5):
    """Eval-mode BatchNorm as y = x*scale + shift (float64 fold, float32 result)."""
    w = sd[prefix + ".weight"].double()
    b = sd[prefix + ".bias"].double()
    mean = sd[prefix + ".running_mean"].double()
    var = sd[prefix + ".running_var"].double()
    scale = w / torch.sqrt(var + eps)
    shift = b - mean * scale
    return scale.float().contiguous(), shift.float().contiguous()


def _call(name, *args):
    capi.check(getattr(capi.load(), name)(*args), name)


def fold_bn_device(sd, prefix, device, eps=1e-5):
    """fold_bn through the C ABI (sed_fold_bn): raw BatchNorm buffers up, float32 scale / shift on the device."""
    raw = [sd[prefix + k].detach().float().contiguous().to(device)
           for k in (".weight", ".bias", ".running_mean", ".running_var")]
    n = raw[0].numel()
    scale = torch.empty(n, dtype=torch.float32, device=device)
    shift = torch.empty(n, dtype=torch.float32, device=device)
    _call("sed_fold_bn", *[capi.ptr(t) for t in raw], n, float(eps), capi.ptr(scale), capi.ptr(shift),
          capi.current_stream(device))
    return scale, shift


def cast16_device(w, tdtype, dtype_code, device):
    """float32 parameter -> 16-bit operand on the device (sed_cast_16, round to nearest even)."""
    src = w.detach().float().contiguous().to(device)
    dst = torch.empty(src.shape, dtype=tdtype, device=device)
    _call("sed_cast_16", capi.ptr(src), src.numel(), capi.ptr(dst), dtype_code, capi.current_stream(device))
    return dst


def twiddle_table(n_fft):
    k = np.arange(n_fft, dtype=np.float64)
    ang = -2.0 * np.pi * k / n_fft
    return torch.from_numpy(np.stack([np.cos(ang), np.sin(ang)], axis=1).astype(np.float32)).contiguous()


def band_mel(melW):
    """melW [F, M] float32 -> (lo, len, off, val): per mel bin the contiguous span covering all non-zeros."""
    W = melW.detach().cpu().float().numpy()
    F, M = W.shape
    lo = np.zeros(M, np.int32)
    ln = np.zeros(M, np.int32)
    off = np.zeros(M, np.int32)
    vals = []
    pos = 0
    for m in range(M):
        nz = np.nonzero(W[:, m])[0]
        if nz.size:
            lo[m] = nz[0]
            ln[m] = nz[-1] - nz[0] + 1
        off[m] = pos
        vals.append(W[lo[m]:lo[m] + ln[m], m])
        pos += int(ln[m])
    val = np.concatenate(vals) if pos else np.zeros(1, np.float32)
    if val.size == 0:
        val = np.zeros(1, np.float32)
    return (torch.from_numpy(lo), torch.from_numpy(ln), torch.from_numpy(off),
            torch.from_numpy(np.ascontiguousarray(val, dtype=np.float32)))


def band_mel_c(melW):
    """band_mel through the C ABI's host helper (sed_band_mel)."""
    W = melW.detach().cpu().float().contiguous()
    F, M = W.shape
    lo, ln, off = (torch.zeros(M, dtype=torch.int32) for _ in range(3))
    val = torch.zeros(max(1, F * M), dtype=torch.float32)
    n = np.zeros(1, np.int32)
    _call("sed_band_mel", capi.ptr(W), F, M, capi.ptr(lo), capi.ptr(ln), capi.ptr(off), capi.ptr(val), val.numel(),
          n.ctypes.data)
    return lo, ln, off, val[:max(1, int(n[0]))].clone()


def check_windowed_dft(conv_real, conv_imag, n_fft, tol=2e-5):
    """The fused front-end evaluates the loaded Conv1d kernels as window x DFT.  Verify that the
    loaded kernels have that structure (stft.py:207-212) and return the window (row 0 of conv_real)."""
    wr = conv_real.detach().cpu().double().reshape(-1, n_fft)
    wi = conv_imag.detach().cpu().double().reshape(-1, n_fft)
    F = n_fft // 2 + 1
    if wr.shape[0] != F or wi.shape[0] != F:
        raise NotImplementedError("STFT kernels must have n_fft//2+1 output channels")
    win = wr[0].clone()
    kn = (torch.arange(F, dtype=torch.int64)[:, None] * torch.arange(n_fft, dtype=torch.int64)[None, :]) % n_fft
    ang = -2.0 * math.pi * kn.double() / n_fft
    err = max((wr - torch.cos(ang) * win).abs().max().item(), (wi - torch.sin(ang) * win).abs().max().item())
    scale = max(win.abs().max().item(), 1e-30)
    if err > tol * scale:
        raise NotImplementedError(
            "loaded conv_real/conv_imag are not a windowed DFT (max deviation %.3g); the B200 front-end "
            "only supports the reference's frozen STFT kernels" % err)
    return win.float().contiguous()


class FrontendPlan:
    """Device-resident constants of the front-end for one (n_fft, hop, melW) configuration."""

    def __init__(self, conv_real, conv_imag, n_fft, hop, melW, device, amin=1e-10, ref=1.0, is_log=True):
        self.n_fft, self.hop = int(n_fft), int(hop)
        if self.n_fft not in (256, 512, 1024):
            raise NotImplementedError("n_fft=%d: only the reference presets 256/512/1024 are built" % n_fft)
        self.window = check_windowed_dft(conv_real, conv_imag, self.n_fft).to(device)
        tw = torch.empty((self.n_fft, 2), dtype=torch.float32)
        _call("sed_frontend_twiddle", self.n_fft, capi.ptr(tw))
        self.twiddle = tw.to(device)
        self.amin = float(amin)
        self.db_offset = float(10.0 * np.log10(np.maximum(amin, ref)))
        self.is_log = 1 if is_log else 0
        self.n_mels = 0
        if melW is not None:
            lo, ln, off, val = band_mel_c(melW)
            self.mel_lo, self.mel_len, self.mel_off, self.mel_val = (t.to(device) for t in (lo, ln, off, val))
            self.n_mels = int(melW.shape[1])
            self.F = int(melW.shape[0])


def _wave_dtype_code(wave):
    if wave.dtype == torch.float32:
        return 0
    if wave.dtype == torch.int16:
        return 1  # PCM: x = q / 32767 (utils/utilities.py:78-79), converted inside the kernel
    raise TypeError("waveform must be float32 or int16, got %s" % (wave.dtype,))


@_on_device_of(1)
def logmel_forward(plan, wave, bn_scale=None, bn_shift=None, out=None, windows=None):
    """wave [B, L] (f32 or int16 PCM) cuda -> [B, T, n_mels] f32.

    windows=(n_windows, L, stride): `wave` is one 1-D recording; window k = wave[k*stride : k*stride + L], zero
    padded past the end (the slicing of predict.py:302-305) -- read in place, never materialised.
    windows=(n_windows, L, offsets): offsets = int64 CUDA tensor [n_windows] of window starts in samples (the windows
    of many padded clips as one batch, main_strong.py:786-805)."""
    lib = capi.load()
    code = _wave_dtype_code(wave)
    if windows is None:
        if wave.dim() != 2 or not wave.is_contiguous():
            raise ValueError("waveform batch must be a contiguous (batch_size, data_length) tensor")
        B, L = wave.shape
        stride, total = L, B * L
        offsets = None
    else:
        if wave.dim() != 1 or not wave.is_contiguous():
            raise ValueError("windowed input must be a contiguous 1-D recording")
        offsets = None
        if torch.is_tensor(windows[2]):
            B, L, stride = int(windows[0]), int(windows[1]), 0
            offsets = windows[2]
            if offsets.dtype != torch.int64 or offsets.numel() != B or offsets.device != wave.device:
                raise ValueError("window offsets must be an int64 tensor [n_windows] on the waveform's device")
        else:
            B, L, stride = (int(v) for v in windows)
        total = wave.numel()
    T = L // plan.hop + 1
    if out is None:
        out = torch.empty((B, T, plan.n_mels), dtype=torch.float32, device=wave.device)
    rc = lib.sed_frontend_logmel(capi.ptr(wave), code, B, L, max(stride, 1),
                                 capi.ptr(offsets), total, plan.n_fft, plan.hop,
                                 capi.ptr(plan.window), capi.ptr(plan.twiddle), capi.ptr(plan.mel_lo),
                                 capi.ptr(plan.mel_len), capi.ptr(plan.mel_off), capi.ptr(plan.mel_val), plan.n_mels,
                                 plan.amin, plan.db_offset, plan.is_log, capi.ptr(bn_scale), capi.ptr(bn_shift),
                                 capi.ptr(out), capi.current_stream(wave.device))
    capi.check(rc, "sed_frontend_logmel")
    capi._count()
    return out


@_on_device_of(0)
def window_merge_avg(frames, overlap_interval, sample_duration):
    """frames [n_windows, frames_per_window, classes] f32 cuda -> merged [1, total_frames, classes]
    (merge + avg_merge, utils/utilities.py:405-446); a 4-D input [n_recordings, n_windows, fpw, classes] merges every
    recording independently -> [n_recordings, total_frames, classes]."""
    lib = capi.load()
    frames = frames.contiguous()
    nrec = 1 if frames.dim() == 3 else frames.shape[0]
    nw, fpw, ncls = frames.shape[-3:]
    total = (nw - 1) * overlap_interval + fpw
    merged = torch.empty((nrec, total, ncls), dtype=torch.float32, device=frames.device)
    rc = lib.sed_window_merge_avg(capi.ptr(frames), nw, fpw, ncls, int(overlap_interval), int(sample_duration),
                                  nrec, capi.ptr(merged), capi.current_stream(frames.device))
    capi.check(rc, "sed_window_merge_avg")
    capi._count()
    return merged


@_on_device_of(1)
def spectrogram_forward(plan, wave):
    lib = capi.load()
    B, L = wave.shape
    T = L // plan.hop + 1
    out = torch.empty((B, 1, T, plan.n_fft // 2 + 1), dtype=torch.float32, device=wave.device)
    rc = lib.sed_spectrogram_f32(capi.ptr(wave), B, L, plan.n_fft, plan.hop, capi.ptr(plan.window),
                                 capi.ptr(plan.twiddle), capi.ptr(out), capi.current_stream(wave.device))
    capi.check(rc, "sed_spectrogram_f32")
    capi._count()
    return out


@_on_device_of(1)
def logmel_rows_forward(plan, spec):
    lib = capi.load()
    F = spec.shape[-1]
    if F != plan.F:
        raise ValueError("spectrogram has %d bins, mel matrix expects %d" % (F, plan.F))
    spec_c = spec.contiguous()
    rows = spec_c.numel() // F
    out = torch.empty(spec.shape[:-1] + (plan.n_mels,), dtype=torch.float32, device=spec.device)
    rc = lib.sed_logmel_rows_f32(capi.ptr(spec_c), rows, F, capi.ptr(plan.mel_lo), capi.ptr(plan.mel_len),
                                 capi.ptr(plan.mel_off), capi.ptr(plan.mel_val), plan.n_mels, plan.amin,
                                 plan.db_offset, plan.is_log, capi.ptr(out), capi.current_stream(spec.device))
    capi.check(rc, "sed_logmel_rows_f32")
    capi._count()
    return out


def event_params(high, low, n_smooth, n_salt, classes, device):
    """Per-class thresholds (sequences or scalars) -> the device arrays of sed_events / sed_live_events:
    high / low float64 (low may be None), n_smooth / n_salt int32."""
    def per_class(v, dtype):
        if v is None:
            return None
        t = torch.as_tensor(np.asarray(v, dtype=np.float64 if dtype == torch.float64 else np.int64))
        if t.dim() == 0:
            t = t.repeat(classes)
        if t.numel() != classes:
            raise ValueError("expected %d per-class values, got %d" % (classes, t.numel()))
        return t.to(dtype).contiguous().to(device)

    return (per_class(high, torch.float64), per_class(low, torch.float64), per_class(n_smooth, torch.int32),
            per_class(n_salt, torch.int32))


@_on_device_of(0)
def extract_events(frames, high, low, n_smooth, n_salt, max_events=64):
    """frames [n_clips, n_frames, classes] f32 cuda; per-class thresholds (sequences or scalars).
    Returns (events [n_clips, classes, max_events, 2] int32, counts [n_clips, classes] int32) on the device
    (activity_detection, utils/vad.py:11-45, for every clip and class)."""
    lib = capi.load()
    frames = frames.contiguous()
    n_clips, n_frames, classes = frames.shape
    dev = frames.device
    hi, lo, ns, nsalt = event_params(high, low, n_smooth, n_salt, classes, dev)
    while True:
        events = torch.zeros((n_clips, classes, max_events, 2), dtype=torch.int32, device=dev)
        counts = torch.zeros((n_clips, classes), dtype=torch.int32, device=dev)
        rc = lib.sed_events(capi.ptr(frames), n_clips, n_frames, classes, capi.ptr(hi), capi.ptr(lo), capi.ptr(ns),
                            capi.ptr(nsalt), max_events, capi.ptr(events), capi.ptr(counts),
                            capi.current_stream(dev))
        capi.check(rc, "sed_events")
        capi._count()
        most = int(counts.max().item())
        if most <= max_events:
            return events, counts
        max_events = most  # rare: more events than the buffer holds -> rerun once with the exact capacity


@_on_device_of(0)
def live_ingest(src, table, n_entries, max_len, ring_samples, arena):
    """sed_live_ingest: chunks of `src` (packed, arena's dtype) -> their slots' mirrored rings in `arena`;
    table = int64 CUDA tensor [>= n_entries, 4] of (slot, offset in src or -1 for zeros, length, stream position)."""
    _call("sed_live_ingest", capi.ptr(src), _wave_dtype_code(arena), capi.ptr(table), int(n_entries), int(max_len),
          int(ring_samples), capi.ptr(arena), capi.current_stream(arena.device))
    capi._count()


@_on_device_of(0)
def live_merge(window_frames, table, n_entries, max_span, overlap_interval, sample_duration, acc, out):
    """sed_live_merge: window_frames [rows, fpw, classes] of one push -> per-slot accumulators acc [slots, ring,
    classes]; frames that became final -> out rows (table: int32 CUDA tensor [>= n_entries, LIVE_TABLE_COLS])."""
    _, fpw, classes = window_frames.shape
    _call("sed_live_merge", capi.ptr(window_frames), capi.ptr(table), int(n_entries), int(max_span), int(fpw),
          int(classes), int(overlap_interval), int(sample_duration), int(acc.shape[1]), capi.ptr(acc), capi.ptr(out),
          capi.current_stream(acc.device))
    capi._count()


@_on_device_of(0)
def live_events(frames, table, n_entries, params, state, events, counts):
    """sed_live_events over the frames sed_live_merge finalized; params = event_params(...) on the device."""
    hi, lo, ns, nsalt = params
    _call("sed_live_events", capi.ptr(frames), capi.ptr(table), int(n_entries), int(frames.shape[-1]), capi.ptr(hi),
          capi.ptr(lo), capi.ptr(ns), capi.ptr(nsalt), capi.ptr(state), capi.ptr(events), capi.ptr(counts),
          capi.current_stream(frames.device))
    capi._count()


def resample_filter(input_rate, output_rate):
    """sed_resample_filter (host helper): (up, down, half, float32 taps) of the polyphase filter input_rate ->
    output_rate.  ValueError for a rate pair it refuses (rates outside 1 .. 384000, max(up, down) > 4096)."""
    lib = capi.load()
    up, down, n = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    args = (int(input_rate), int(output_rate), ctypes.byref(up), ctypes.byref(down), ctypes.byref(n))
    rc = lib.sed_resample_filter(*args, None)
    if rc == 0:
        taps = np.zeros(n.value, np.float32)
        rc = lib.sed_resample_filter(*args, taps.ctypes.data_as(ctypes.c_void_p))
    if rc != 0:
        raise ValueError("cannot resample %s Hz -> %s Hz: %s" % (input_rate, output_rate,
                                                                 lib.sed_last_error_string().decode("utf-8", "replace")))
    return up.value, down.value, (n.value - 1) // 2, taps


class ResamplePlan:
    """The filter input_rate -> output_rate on one device.  Equal rates keep librosa.load's behaviour (no resampling,
    downmix only): the one-tap filter [1.0], for which y[j] = x[j] exactly."""

    def __init__(self, input_rate, output_rate, device):
        self.input_rate, self.output_rate = int(input_rate), int(output_rate)
        if self.input_rate == self.output_rate and 0 < self.input_rate <= 384000:
            self.up = self.down = 1
            self.half, taps = 0, np.ones(1, np.float32)
        else:
            self.up, self.down, self.half, taps = resample_filter(input_rate, output_rate)
        self.n_taps = 2 * self.half + 1
        self.taps = torch.from_numpy(taps).to(device)

    def n_out(self, n_in):
        """Output samples of a whole recording of n_in input samples: ceil(n_in * up / down)."""
        return -(-np.asarray(n_in, np.int64) * self.up // self.down)

    def n_out_live(self, n_in):
        """Outputs whose whole filter support lies in the first n_in input samples (before a stream's end)."""
        n_in = np.asarray(n_in, np.int64)
        return np.maximum(0, ((n_in - 1) * self.up - self.half) // self.down + 1)

    def history_len(self):
        """Input samples a live stream keeps from earlier pushes (DESIGN.md K7 derives the bound)."""
        return -(-(self.n_taps - 1 + self.down) // self.up) + 1


_RESAMPLE_PLANS = {}


def resample_plan(input_rate, output_rate, device):
    key = (int(input_rate), int(output_rate), torch.device(device))
    if key not in _RESAMPLE_PLANS:
        _RESAMPLE_PLANS[key] = ResamplePlan(input_rate, output_rate, device)
    return _RESAMPLE_PLANS[key]


@_on_device_of(0)
def resample(src, channels, table, n_rows, max_out, plan, dst):
    """sed_resample: the recordings of `src` (interleaved frames of `channels` samples, float32 or int16) -> float32
    `dst`; table = int64 CUDA tensor [>= n_rows, 4] of (first frame in src, n_in, first sample in dst, n_out)."""
    _call("sed_resample", capi.ptr(src), _wave_dtype_code(src), int(channels), capi.ptr(table), int(n_rows),
          int(max_out), capi.ptr(plan.taps), plan.up, plan.down, plan.half, capi.ptr(dst),
          capi.current_stream(src.device))
    capi._count()


@_on_device_of(0)
def live_resample(src, channels, table, n_entries, max_len, plan, ring_samples, arena, hist, history_len, history_table,
                  n_history):
    """sed_live_resample: one tick of live ingest with resampling (table: int64 [>= n_entries, 6]); with n_history > 0
    the push's chunks then go into the slots' history rings hist [slots, history_len] (history_table: int64
    [>= n_history, 4])."""
    _call("sed_live_resample", capi.ptr(src), _wave_dtype_code(src), int(channels), capi.ptr(table), int(n_entries),
          int(max_len), capi.ptr(plan.taps), plan.up, plan.down, plan.half, int(ring_samples), capi.ptr(arena),
          capi.ptr(hist), int(history_len), capi.ptr(history_table),
          int(n_history), capi.current_stream(arena.device))
    capi._count((1 if n_entries and max_len else 0) + (1 if n_history else 0))


def blocks_to_rows(xb, n, T):
    """128-clip transposed blocks [T, nblk, C/4, 128, 4] (float4 column c4 of clip row m of block (t, blk) at
    ((t*nblk + blk)*C/4 + c4)*128 + m) -> ordinary rows [n, T, C]."""
    T_, nblk, c4, _, _ = xb.shape
    return xb.permute(1, 3, 0, 2, 4).reshape(nblk * 128, T_, c4 * 4)[:n]


def clamp_micro_batch(micro_batch, T):
    """Cap of a conv launch group for clips of T STFT frames: the requested cap, scaled down for clips longer than
    10 s so that the activation workspace (14 KB per frame and clip) and the kernels' 32-bit tile arithmetic stay
    where batch 1036 x 10 s puts them; multiples of 37 clips (whole waves of the persistent grids) when possible."""
    if micro_batch < 1:
        raise ValueError("micro_batch must be positive")
    cap = min(int(micro_batch), max(1, DEFAULT_MICRO_BATCH * 1001 // max(int(T), 1)))
    # conv_block1 divides tile indices by multiplication: tiles_per_clip * (tiles + 4096) must stay below 2^32
    per_clip = ((int(T) + 15) // 16) * 8
    cap = max(1, min(cap, ((1 << 32) // per_clip - 4097) // per_clip))
    if cap >= 37 and cap < micro_batch:
        cap -= cap % 37
    return cap


def plan_host_micro_batches(B, int16_input, micro_batch=DEFAULT_MICRO_BATCH, result_parts=1):
    """Micro-batch schedule of forward_host: (parts, plan) with parts = [(begin, end)] clip ranges that each run conv
    stack -> temporal block -> head on their own and plan[i] = the conv micro-batches [(b0, b1)] of part i.

    result_parts=2 cuts the batch in two parts (the last one 185 clips), so that the 100 KB/clip result copy of part 0
    hides behind the conv stack of part 1.  Measured on one box (tools/e2e_ab.py, batch 1024): 23.6 ms either way -- the
    second launch of the latency-bound temporal block + head (1.4 ms) costs what the hidden copy saves (1.7 ms) -- so the
    default is one part.
    Inside a part: a short first micro-batch lets the conv stack start after ~0.4 ms of PCIe traffic; after that a
    micro-batch may only grow as fast as its copy hides behind the previous one's conv stack (~21 us per clip against
    ~12 us of PCIe for float32, ~6 us for int16); sizes are multiples of 37 clips = whole waves of the persistent grids,
    and a short remainder of a part is folded into its last micro-batch."""
    last = 185  # 5 x 37 clips
    parts = [(0, B - last), (B - last, B)] if (result_parts == 2 and B >= 640) else [(0, B)]
    growth = iter((37, 111, 296) if int16_input else (37, 37, 74, 111, 185, 296))
    plan = []
    for (p0, p1) in parts:
        spans, b0 = [], p0
        while b0 < p1:
            size = min(next(growth, micro_batch), micro_batch)
            if p1 - b0 <= min(size + size // 2, micro_batch):
                size = p1 - b0
            spans.append((b0, min(p1, b0 + size)))
            b0 = spans[-1][1]
        plan.append(spans)
    return parts, plan


class PackedModel:
    """Weights of one model repacked for the kernels, resident on one device."""

    def __init__(self, sd, model_type, n_fft, hop, device, precision="fp16"):
        device = torch.device(device)
        if device.type != "cuda":
            raise ValueError("PackedModel needs a CUDA device (no CPU fallback), got %s" % (device,))
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        with torch.cuda.device(device):
            self._init(sd, model_type, n_fft, hop, device, precision)

    def _init(self, sd, model_type, n_fft, hop, device, precision):
        if precision not in _DTYPES:
            raise ValueError("precision must be 'fp16' or 'bf16'")
        if model_type not in MODEL_PLANS:
            raise NotImplementedError("model_type %r is not built" % (model_type,))
        self.model_type = model_type
        self.temporal_kind, self.head_kind = MODEL_PLANS[model_type]
        # only Cnn_9layers_Gru_FrameAtt pads the framewise output to 100-frame blocks (models.py:680-681)
        self.pads_frames = model_type == "Cnn_9layers_Gru_FrameAtt"
        self.device = torch.device(device)
        self.precision = precision
        self.dtype_code, self.tdtype = _DTYPES[precision]
        dev, td = self.device, self.tdtype
        sd = {k: v.detach().to("cpu") for k, v in sd.items()}
        self.front = FrontendPlan(sd["spectrogram_extractor.stft.conv_real.weight"],
                                  sd["spectrogram_extractor.stft.conv_imag.weight"], n_fft, hop,
                                  sd["logmel_extractor.melW"], dev)
        if self.front.n_mels != 64:
            raise NotImplementedError("Cnn_9layers needs mel_bins == 64 (bn0 is BatchNorm2d(64), models.py:607)")
        # weight preparation goes through the C ABI's helpers (sed_fold_bn / sed_pack_* / sed_cast_16), the same calls
        # a torch-free caller makes (examples/sed_infer.c)
        stream = capi.current_stream(dev)
        self.bn0_scale, self.bn0_shift = fold_bn_device(sd, "bn0", dev)
        # conv_block1.conv1 (Cin = 1): float32 weights; bn1 folded
        self.c11_w = sd["conv_block1.conv1.weight"].float().reshape(64, 9).contiguous().to(dev)
        self.c11_scale, self.c11_shift = fold_bn_device(sd, "conv_block1.bn1", dev)
        # fused conv_block1: bn1 scale folded into the nine taps (float64 product, float32 result)
        self.c11_ws = torch.empty((64, 9), dtype=torch.float32, device=dev)
        _call("sed_pack_conv_first", capi.ptr(self.c11_w), capi.ptr(self.c11_scale), capi.ptr(self.c11_ws), stream)
        self.convs = []
        for name, cin, cout, mode in CONV_LAYERS:
            w = sd[name + ".weight"].float()
            if tuple(w.shape) != (cout, cin, 3, 3):
                raise ValueError("%s.weight has shape %s" % (name, tuple(w.shape)))
            w_dev = w.contiguous().to(dev)
            wp = torch.empty((cout, 9 * cin), dtype=td, device=dev)  # [Cout][tap][Cin]
            _call("sed_pack_conv3x3", capi.ptr(w_dev), cout, cin, capi.ptr(wp), self.dtype_code, stream)
            s, b = fold_bn_device(sd, name.replace(".conv", ".bn"), dev)
            self.convs.append((cin, cout, mode, wp, s, b))
        if self.temporal_kind == "gru":
            wih = torch.cat([sd["gru.weight_ih_l0"], sd["gru.weight_ih_l0_reverse"]], 0)
            self.gru_wih = cast16_device(wih, td, self.dtype_code, dev)  # [1536, 512]
            self.gru_bih = torch.cat([sd["gru.bias_ih_l0"], sd["gru.bias_ih_l0_reverse"]], 0).float().contiguous().to(dev)
            # block q of a direction holds hidden units 32q..32q+31 of all three gates (see sed_b200.h: sed_bigru)
            whh = [sd["gru.weight_hh_l0" + suffix].float().contiguous().to(dev) for suffix in ("", "_reverse")]
            self.gru_whh = torch.empty((1536, 256), dtype=td, device=dev)
            _call("sed_pack_gru_whh", capi.ptr(whh[0]), capi.ptr(whh[1]), capi.ptr(self.gru_whh), self.dtype_code, stream)
            self.gru_bhh = torch.stack([sd["gru.bias_hh_l0"], sd["gru.bias_hh_l0_reverse"]], 0).float().contiguous().to(dev)
        elif self.temporal_kind == "mha":
            wqkv = torch.cat([sd["multihead.w_qs.weight"], sd["multihead.w_ks.weight"], sd["multihead.w_vs.weight"]], 0)
            self.mha_wqkv = cast16_device(wqkv, td, self.dtype_code, dev)
            self.mha_bqkv = torch.cat([sd["multihead.w_qs.bias"], sd["multihead.w_ks.bias"],
                                       sd["multihead.w_vs.bias"]], 0).float().contiguous().to(dev)
            self.mha_wfc = cast16_device(sd["multihead.fc.weight"], td, self.dtype_code, dev)
            self.mha_bfc = sd["multihead.fc.bias"].float().contiguous().to(dev)
        if self.head_kind == "att":
            self.classes = 25  # hard-coded in the reference (models.py:617)
            self.att_w = sd["att_block.att.weight"].float().reshape(25, 512).contiguous().to(dev)
            self.att_b = sd["att_block.att.bias"].float().contiguous().to(dev)
            self.cla_w = sd["att_block.cla.weight"].float().reshape(25, 512).contiguous().to(dev)
            self.cla_b = sd["att_block.cla.bias"].float().contiguous().to(dev)
        else:
            self.fc_w = sd["fc.weight"].float().contiguous().to(dev)  # [classes_num, 512]
            self.fc_b = sd["fc.bias"].float().contiguous().to(dev)
            self.classes = int(self.fc_w.shape[0])
            if self.fc_w.shape[1] != 512 or self.classes > 32:
                raise NotImplementedError("fc head: need Linear(512 -> classes_num <= 32)")
        # range guard: packed 16-bit weights that hit the format's limit (fp16: |w| >= 65504) were clipped
        self.weight_saturation = {}
        packed16 = [(CONV_LAYERS[i][0], c[3]) for i, c in enumerate(self.convs)]
        packed16 += [(n, getattr(self, n)) for n in ("gru_wih", "gru_whh", "mha_wqkv", "mha_wfc") if hasattr(self, n)]
        for name, t in packed16:
            self.weight_saturation[name] = self.count_saturated(t)
        if any(self.weight_saturation.values()):
            import warnings
            warnings.warn("sed_b200: %s weights exceed the %s range and were clipped: %s -- outputs will differ from "
                          "the float32 reference" % (model_type, precision,
                                                     {k: v for k, v in self.weight_saturation.items() if v}))
        self._ws = collections.OrderedDict()  # T -> workspace entry, least recently used first
        self._lock = threading.RLock()
        self._pipelines = {}
        self._last_stream = None
        self.conv_events = None  # set to [] to collect (start, end) CUDA events around the tensor-core conv launches

    # ------------------------------------------------------------------ workspaces
    WS_CACHE_ENTRIES = 3          # clip lengths whose activation workspace stays allocated
    WS_CACHE_BYTES = 64 << 30     # ... as long as together they stay below this

    def _workspace(self, mb, T, need_a1=False):
        """Activation buffers of the conv stack for a micro-batch of `mb` clips: views into one allocation per clip
        length T, sized for the largest micro-batch seen (micro-batch sizes vary inside forward_host).  A small LRU of
        clip lengths is kept, so that callers alternating between lengths (10 s evaluation clips and 5 s streaming
        windows) do not re-allocate ~14.5 GB per switch.  a1, the 8.2 MB/clip output of conv_block1.conv1, only exists
        for the two-kernel variants of block 1."""
        ent = self._ws.get(T)
        if ent is None or ent["cap"] < mb or (need_a1 and "a1" not in ent["buf"]):
            cap = mb if ent is None else max(mb, ent["cap"])
            need_a1 = need_a1 or (ent is not None and "a1" in ent["buf"])
            dev, td = self.device, self.tdtype
            H1, H2, H3 = T // 2, T // 4, T // 8
            self._ws.pop(T, None)  # drop this length's old allocation first
            ent = None
            per_clip = 4 * T * 64 + 2 * 64 * (H1 * 32 * 3 + H2 * 16 * 6 + H3 * 8 * 12) + (2 * T * 64 * 64 if need_a1 else 0)
            while self._ws and (len(self._ws) >= self.WS_CACHE_ENTRIES or
                                sum(e["bytes"] for e in self._ws.values()) + cap * per_clip > self.WS_CACHE_BYTES):
                self._ws.popitem(last=False)
            buf = {
                "logmel": torch.empty((cap, T, 64), dtype=torch.float32, device=dev),
                "p1": torch.empty((cap, H1, 32, 64), dtype=td, device=dev),
                "a2": torch.empty((cap, H1, 32, 128), dtype=td, device=dev),
                "p2": torch.empty((cap, H2, 16, 128), dtype=td, device=dev),
                "a3": torch.empty((cap, H2, 16, 256), dtype=td, device=dev),
                "p3": torch.empty((cap, H3, 8, 256), dtype=td, device=dev),
                "a4": torch.empty((cap, H3, 8, 512), dtype=td, device=dev),
            }
            if need_a1:
                buf["a1"] = torch.empty((cap, T, 64, 64), dtype=td, device=dev)
            ent = {"cap": cap, "buf": buf, "bytes": sum(t.numel() * t.element_size() for t in buf.values())}
            self._ws[T] = ent
        self._ws.move_to_end(T)
        return {k: v[:mb] for k, v in ent["buf"].items()}

    def _acquire_stream(self, stream):
        """The activation workspace is shared by every entry point; when the launching stream changes (forward on
        the caller's stream, the host pipeline on its own), the new stream waits for the work queued on the old one."""
        if self._last_stream is not None and self._last_stream != stream:
            stream.wait_stream(self._last_stream)
        self._last_stream = stream

    # ------------------------------------------------------------------ stages
    @_on_device
    def conv_stack(self, wave_mb, feat_out, variant=4, stages=None, windows=None, feat32=None, feat_strides=(0, 0)):
        """wave_mb [mb, L] (f32 / int16) -> feat_out [mb, T', 512] 16-bit (freq-mean of conv_block4).
        windows=(mb, L, stride): wave_mb is a 1-D recording read as overlapping windows.
        feat32: optional [mb, T', 512] f32 copy of the features (models without a temporal block).
        feat_strides=(sn, sh): feature row of (clip n, step h) is n*sn + h*sh rows after feat_out's first element
        ((0, 0) = clip-major [mb, T', 512]; (1, Bp) = time-major [T', Bp, 512] as the GRU wants it)."""
        lib = capi.load()
        if windows is None:
            mb, L = wave_mb.shape
        else:
            mb, L = int(windows[0]), int(windows[1])
        T = L // self.front.hop + 1
        if T // 8 < 1:
            raise ValueError("clip too short: %d frames" % T)
        fused1 = variant in (3, 4)  # conv_block1 as one kernel (its 64-channel intermediate stays on chip)
        ws = self._workspace(mb, T, need_a1=not fused1)
        stream = capi.current_stream(self.device)
        logmel_forward(self.front, wave_mb, self.bn0_scale, self.bn0_shift, out=ws["logmel"], windows=windows)
        producer = 1 if variant == 4 else 0  # conv1 on the tensor cores (split fp16) / on the CUDA cores
        if fused1:
            variant = 2
        else:
            rc = lib.sed_conv_first_f32(capi.ptr(ws["logmel"]), mb, T, 64, capi.ptr(self.c11_w),
                                        capi.ptr(self.c11_scale), capi.ptr(self.c11_shift), capi.ptr(ws["a1"]),
                                        self.dtype_code, stream)
            capi.check(rc, "sed_conv_first_f32")
            capi._count()
        chain = [("a1", "p1"), ("p1", "a2"), ("a2", "p2"), ("p2", "a3"), ("a3", "p3"), ("p3", "a4"), ("a4", None)]
        if self.conv_events is not None:
            ev0 = torch.cuda.Event(enable_timing=True)
            ev0.record(torch.cuda.current_stream(self.device))
        for li, ((cin, cout, mode, wp, s, b), (src, dst)) in enumerate(zip(self.convs, chain)):
            if fused1 and li == 0:
                rc = lib.sed_conv_block1(capi.ptr(ws["logmel"]), mb, T, 64, capi.ptr(self.c11_ws),
                                         capi.ptr(self.c11_shift), capi.ptr(wp), capi.ptr(s), capi.ptr(b),
                                         capi.ptr(ws["p1"]), producer, self.dtype_code, stream)
                capi.check(rc, "sed_conv_block1")
                capi._count()
                continue
            x = ws[src]
            out = feat_out if dst is None else ws[dst]
            rc = lib.sed_conv3x3_bn_relu(capi.ptr(x), mb, x.shape[1], x.shape[2], cin, capi.ptr(wp), capi.ptr(s),
                                         capi.ptr(b), cout, mode, capi.ptr(out),
                                         capi.ptr(feat32) if dst is None else None,
                                         feat_strides[0] if dst is None else 0, feat_strides[1] if dst is None else 0,
                                         self.dtype_code, variant, stream)
            capi.check(rc, "sed_conv3x3_bn_relu(%d->%d)" % (cin, cout))
            capi._count()
        if self.conv_events is not None:
            ev1 = torch.cuda.Event(enable_timing=True)
            ev1.record(torch.cuda.current_stream(self.device))
            self.conv_events.append((ev0, ev1, mb))
        if stages is not None:
            stages["bn0"] = ws["logmel"].clone()
            for k in ("a1", "p1", "a2", "p2", "a3", "p3", "a4"):
                if k in ws and not (fused1 and k == "a1"):  # the fused block never materialises a1
                    stages[k] = ws[k].clone()

    @_on_device
    def linear(self, a16, w16, bias, relu=False, out16=False, out_layout=0, f32=True):
        """out_layout 1: float32 output as 128-row transposed blocks (see sed_b200.h: sed_linear).
        f32=False (with out16=True): only the 16-bit output is written."""
        lib = capi.load()
        M, K = a16.shape
        N = w16.shape[0]
        out = torch.empty((M, N), dtype=torch.float32, device=self.device) if f32 else None
        o16 = torch.empty((M, N), dtype=self.tdtype, device=self.device) if out16 else None
        rc = lib.sed_linear(capi.ptr(a16), M, K, capi.ptr(w16), capi.ptr(bias), N, 1 if relu else 0, capi.ptr(out),
                            capi.ptr(o16), out_layout, self.dtype_code, capi.current_stream(self.device))
        capi.check(rc, "sed_linear")
        capi._count((N + 1535) // 1536)
        if not f32:
            return o16
        return (out, o16) if out16 else out

    @_on_device
    def temporal(self, feat16, stages=None):
        """feat16 [B, T', 512] 16-bit -> [B, T', 512] f32 (GRU or MultiHead output)."""
        lib = capi.load()
        B, Tp, _ = feat16.shape
        stream = capi.current_stream(self.device)
        flat = feat16.view(B * Tp, 512)
        if self.temporal_kind == "gru":
            # clip-major input (tests, tools): repack time-major over the padded batch, then the product path
            feat_t = self.alloc_feat_tmajor(B, Tp)
            feat_t[:, :B].copy_(feat16.transpose(0, 1))
            return blocks_to_rows(self.gru_tmajor(feat_t, B, stages), B, Tp)
        if self.temporal_kind != "mha":
            raise RuntimeError("%s has no temporal block" % self.model_type)
        feat_t = self.alloc_feat_tmajor(B, Tp)
        feat_t[:, :B].copy_(feat16.transpose(0, 1))
        return blocks_to_rows(self.mha_tmajor(feat_t, B, stages), B, Tp)

    def alloc_feat_tmajor(self, B, Tp):
        """[T', Bp, 512] 16-bit feature buffer, Bp = B rounded up to 128 clips (padding rows zero)."""
        Bp = (B + 127) // 128 * 128
        make = torch.empty if Bp == B else torch.zeros
        return make((Tp, Bp, 512), dtype=self.tdtype, device=self.device)

    @_on_device
    def gru_tmajor(self, feat_t, B, stages=None):
        """feat_t [T', Bp, 512] 16-bit (time-major, batch padded to 128) -> bi-GRU output as 128-clip transposed
        blocks (T'*Bp*512 f32, see blocks_to_rows).  The input projection writes gi in the same layout, which the
        recurrence streams with fully coalesced loads (one contiguous 96 KB block per CTA and step)."""
        lib = capi.load()
        Tp, Bp, _ = feat_t.shape
        gi = self.linear(feat_t.view(Tp * Bp, 512), self.gru_wih, self.gru_bih, out_layout=1)
        out = torch.empty((Tp, Bp // 128, 128, 128, 4), dtype=torch.float32, device=self.device)
        ws = torch.empty((max(16, lib.sed_bigru_workspace_bytes(B)),), dtype=torch.uint8, device=self.device)
        rc = lib.sed_bigru(capi.ptr(gi), capi.ptr(self.gru_whh), capi.ptr(self.gru_bhh), B, Tp, capi.ptr(out),
                           capi.ptr(ws), self.dtype_code, capi.current_stream(self.device))
        capi.check(rc, "sed_bigru")
        capi._count()
        if stages is not None:
            stages["gi_blocks"] = gi
        return out

    MHA_TC_MAX_STEPS = 128  # the tensor-core attention kernel holds one 128-step tile of keys per (clip, head)
    mha_split = True        # q, k as split 16-bit operands (hi + lo): float32-grade logits in the tensor-core kernel

    @_on_device
    def mha_tmajor(self, feat_t, B, stages=None, tensor_core=True):
        """feat_t [T', Bp, 512] 16-bit (time-major, batch padded to 128) -> relu(fc(attention)) as 128-clip transposed
        blocks (the layout sed_attpool_blocks consumes).  T' <= 128 (clips up to 10.24 s): q | k | v leave the
        projection as 16-bit rows and feed sed_mha_attention (tcgen05 QK^T / PV, softmax in registers); longer clips
        take the float32 kernel sed_mha_core, which tiles nothing and keeps K / V of a head in shared memory."""
        lib = capi.load()
        Tp, Bp, _ = feat_t.shape
        ctx = torch.empty((Tp * Bp, 512), dtype=self.tdtype, device=self.device)
        if Bp != B:
            ctx.zero_()  # rows of padding clips are not produced by the attention kernels
        if tensor_core and Tp <= self.MHA_TC_MAX_STEPS:
            stream = capi.current_stream(self.device)
            qkv = torch.empty((Tp * Bp, 1536), dtype=self.tdtype, device=self.device)
            qk_lo = torch.empty((Tp * Bp, 1024), dtype=self.tdtype, device=self.device) if self.mha_split else None
            if self.mha_split:
                rc = lib.sed_linear_split16(capi.ptr(feat_t), Tp * Bp, 512, capi.ptr(self.mha_wqkv), capi.ptr(self.mha_bqkv),
                                            1536, capi.ptr(qkv), capi.ptr(qk_lo), 1024, self.dtype_code, stream)
                capi.check(rc, "sed_linear_split16")
            else:
                rc = lib.sed_linear(capi.ptr(feat_t), Tp * Bp, 512, capi.ptr(self.mha_wqkv), capi.ptr(self.mha_bqkv), 1536,
                                    0, None, capi.ptr(qkv), 0, self.dtype_code, stream)
                capi.check(rc, "sed_linear")
            capi._count()
            rc = lib.sed_mha_attention(capi.ptr(qkv), capi.ptr(qk_lo), B, Tp, Bp, capi.ptr(ctx), self.dtype_code, stream)
            capi.check(rc, "sed_mha_attention")
        else:
            qkv = self.linear(feat_t.view(Tp * Bp, 512), self.mha_wqkv, self.mha_bqkv)
            rc = lib.sed_mha_core(capi.ptr(qkv), B, Tp, Bp, 1, capi.ptr(ctx), self.dtype_code,
                                  capi.current_stream(self.device))
            capi.check(rc, "sed_mha_core")
        capi._count()
        out = self.linear(ctx, self.mha_wfc, self.mha_bfc, relu=True, out_layout=1)
        if stages is not None:
            stages["qkv_tmajor"] = qkv
            stages["ctx_tmajor"] = ctx
        return out.view(Tp, Bp // 128, 128, 128, 4)

    def frames_for(self, Tp):
        """Number of framewise rows the model returns for T' pooled steps (x8 interpolation; only
        Cnn_9layers_Gru_FrameAtt pads to the next multiple of 100 when != 1000, models.py:62-63, 680-681)."""
        frames = Tp * 8
        if self.pads_frames and frames != 1000 and frames % 100:
            frames += 100 - frames % 100
        return frames

    @_on_device
    def head(self, x, frames_out, want_cla=True, want_norm_att=False, out=None, n=None, clip0=0):
        """x [B, T', 512] f32 -> (clipwise [B,C], framewise [B,frames_out,C], cla | None, norm_att | None).
        x may also be a 5-D transposed-block tensor (gru_tmajor output) covering n clips."""
        lib = capi.load()
        dev = self.device
        if x.dim() == 5:
            if self.head_kind != "att":
                x = blocks_to_rows(x, n, x.shape[0])
            else:
                return self._head_blocks(x, n, frames_out, want_cla, want_norm_att, out)
        B, Tp, _ = x.shape
        C = self.classes
        if out is not None:
            clip, frame = out  # preallocated [B,C] / [B,frames_out,C] (contiguous slices)
        else:
            clip = torch.empty((B, C), dtype=torch.float32, device=dev)
            frame = torch.empty((B, frames_out, C), dtype=torch.float32, device=dev)
        if self.head_kind == "att":
            cla = torch.empty((B, C, Tp), dtype=torch.float32, device=dev) if want_cla else None
            natt = torch.empty((B, C, Tp), dtype=torch.float32, device=dev) if want_norm_att else None
            rc = lib.sed_attpool(capi.ptr(x), B, Tp, capi.ptr(self.att_w), capi.ptr(self.att_b), capi.ptr(self.cla_w),
                                 capi.ptr(self.cla_b), 8, frames_out, capi.ptr(clip), capi.ptr(frame), capi.ptr(cla),
                                 capi.ptr(natt), capi.current_stream(dev))
            capi.check(rc, "sed_attpool")
            capi._count()
            return clip, frame, cla, natt
        if frames_out != Tp * 8:
            raise ValueError("fc heads return exactly 8 x T' frames")
        rc = lib.sed_fcpool(capi.ptr(x), B, Tp, capi.ptr(self.fc_w), capi.ptr(self.fc_b), C, 8,
                            1 if self.head_kind == "max" else 0, capi.ptr(clip), capi.ptr(frame),
                            capi.current_stream(dev))
        capi.check(rc, "sed_fcpool")
        capi._count()
        return clip, frame, None, None

    @_on_device
    def _head_blocks(self, xb, n, frames_out, want_cla, want_norm_att, out, stage=0, clips=None, scratch=None):
        """Pooling head on a transposed-block input.  stage / clips=(begin, count) / scratch expose the two launches
        of sed_attpool_blocks separately (forward_host overlaps result copies with the per-clip pass); `out` tensors
        always cover all n clips."""
        lib = capi.load()
        dev = self.device
        Tp = xb.shape[0]
        if out is not None:
            clip, frame = out
        else:
            clip = torch.empty((n, 25), dtype=torch.float32, device=dev)
            frame = torch.empty((n, frames_out, 25), dtype=torch.float32, device=dev)
        cla = torch.empty((n, 25, Tp), dtype=torch.float32, device=dev) if want_cla else None
        natt = torch.empty((n, 25, Tp), dtype=torch.float32, device=dev) if want_norm_att else None
        if scratch is None:
            scratch = torch.empty((lib.sed_attpool_blocks_scratch_bytes(n, Tp),), dtype=torch.uint8, device=dev)
        c0, cn = (0, n) if clips is None else clips
        rc = lib.sed_attpool_blocks(capi.ptr(xb), n, Tp, capi.ptr(self.att_w), capi.ptr(self.att_b),
                                    capi.ptr(self.cla_w), capi.ptr(self.cla_b), 8, frames_out, capi.ptr(scratch),
                                    capi.ptr(clip), capi.ptr(frame), capi.ptr(cla), capi.ptr(natt), stage, c0, cn,
                                    capi.current_stream(dev))
        capi.check(rc, "sed_attpool_blocks")
        capi._count(2 if stage == 0 else 1)
        return clip, frame, cla, natt

    def _embedding(self, x, cla, feat32):
        """The reference's 'embedding' entry: cla for the two *_FrameAtt models that expose it (models.py:686, 460),
        else the [B, 512, T'] input of the head (models.py:1075, 288, 553, 970)."""
        if self.model_type in ("Cnn_9layers_Gru_FrameAtt", "Cnn_9layers_FrameAtt"):
            return cla
        if not self.temporal_kind:
            return feat32.transpose(1, 2)
        return x.transpose(1, 2)

    # ------------------------------------------------------------------ whole model
    @_on_device
    def count_saturated(self, t):
        """Number of stored 16-bit values of `t` at the format's +-MAX (= conversions that clipped), via the C ABI."""
        if t.dtype != self.tdtype:
            raise TypeError("expected a %s tensor" % (self.tdtype,))
        t = t.contiguous()
        cnt = torch.zeros(1, dtype=torch.int64, device=self.device)
        _call("sed_count_saturated16", capi.ptr(t), t.numel(), self.dtype_code, capi.ptr(cnt),
              capi.current_stream(self.device))
        capi._count()
        return int(cnt.item())

    def saturation_report(self, wave, micro_batch=DEFAULT_MICRO_BATCH):
        """Debug-mode range check of the 16-bit path on real inputs: runs `wave` through the model with every conv
        activation materialised (block 1 as two kernels, so conv1's output exists in memory) and returns
        {'weights': {name: count}, 'activations': {stage: count}, 'total': n} -- the number of values that hit the
        16-bit format's range limit and were clipped (always 0 for a healthy checkpoint; the float32 reference has no
        such limit, so any non-zero count means the outputs may differ from it).  Weights are checked at pack time
        too (`self.weight_saturation`)."""
        out, stages = self.forward(wave, micro_batch=micro_batch, variant=2, return_stages=True)
        acts = {}
        for k in ("a1", "p1", "a2", "p2", "a3", "p3", "a4", "feat"):
            if k in stages and stages[k] is not None and stages[k].dtype == self.tdtype:
                acts[k] = self.count_saturated(stages[k])
        total = sum(acts.values()) + sum(self.weight_saturation.values())
        return {"weights": dict(self.weight_saturation), "activations": acts, "total": total}

    def host_pipeline(self, depth=2, micro_batch=DEFAULT_MICRO_BATCH, variant=4, head_chunk=256):
        """The cached `pipeline.HostPipeline` of this model for the given options (see that class): asynchronous
        submit / result over host buffers with `depth` batches in flight."""
        from .pipeline import HostPipeline
        key = (depth, micro_batch, variant, head_chunk)
        pipe = self._pipelines.get(key)
        if pipe is None:
            pipe = self._pipelines[key] = HostPipeline(self, depth, micro_batch, variant, head_chunk)
        return pipe

    def forward_host(self, wave_host, micro_batch=DEFAULT_MICRO_BATCH, variant=4, head_chunk=256, result_parts=1,
                     trace=None, copy=False):
        """One synchronous end-to-end call with HOST buffers: `wave_host` [B, L] f32 or int16 (pinned for full
        speed) is copied to the device micro-batch by micro-batch on a copy stream that runs ahead of the compute
        stream, and `clipwise_output` / `framewise_output` come back as host tensors (the reference callers do
        `.data.cpu().numpy()` on exactly these, pytorch_utils.py:57-62).

        Result lifetime: with copy=False (default) the returned tensors are views of pinned staging buffers that
        rotate over THREE calls -- a result stays valid while the next two calls run and is overwritten by the third;
        a loop that keeps results longer must copy them (or pass copy=True, which returns fresh tensors like the
        reference's `.data.cpu()`).  For back-to-back batches use `host_pipeline()`: it overlaps the copies of one
        batch with the kernels of its neighbours."""
        pipe = self.host_pipeline(3, micro_batch, variant, head_chunk)
        pipe.drain()
        pipe.trace = trace
        try:
            ticket = pipe.submit(wave_host, result_parts=result_parts)
            return pipe.result(ticket, copy=copy)
        finally:
            pipe.trace = None

    # shared-memory limits of the temporal / pooling kernels in pooled steps T' (one step = 80 ms at 100 frames/s):
    # mha_core keeps K and V of a head resident (512 T' bytes <= 200 KB); sed_attpool keeps the 100 KB of weights plus
    # [T'][50] f32 (<= 220 KB); sed_attpool_blocks' per-clip pass only the [T'][50] f32
    MAX_POOLED_STEPS = {"mha": 400, "att": 590, "att_blocks": 1100}

    def _check_frames(self, T):
        """Reject clip lengths the kernels cannot take BEFORE anything is launched, naming the limit."""
        if T // 8 < 1:
            raise ValueError("clip too short: %d STFT frames give no pooled time step (need >= 8)" % T)
        Tp = T // 8
        limits = []
        if self.temporal_kind == "mha":
            limits.append(("MultiHead block", self.MAX_POOLED_STEPS["mha"]))
        if self.head_kind == "att":
            limits.append(("frame-attention head", self.MAX_POOLED_STEPS["att_blocks" if self.temporal_kind else "att"]))
        for what, cap in limits:
            if Tp > cap:
                raise ValueError("clip too long for the %s: %d pooled steps, limit %d (= %.0f s of audio at 100 "
                                 "frames/s)" % (what, Tp, cap, cap * 0.08))

    def _alloc_features(self, n, Tp):
        """Feature buffers of the conv stack and slot(b0, b1) -> conv_stack keyword arguments for one micro-batch.
        Models with a temporal block get the features time-major ([T', Bp, 512]: the GRU / MultiHead kernels then
        read and write 128-clip blocks), the others clip-major ([n, T', 512])."""
        if self.temporal_kind is not None:
            feat_t = self.alloc_feat_tmajor(n, Tp)
            Bp = feat_t.shape[1]
            return feat_t, None, (lambda b0, b1: {"feat_out": feat_t[0, b0:b1], "feat_strides": (1, Bp)})
        feat16 = torch.empty((n, Tp, 512), dtype=self.tdtype, device=self.device)
        feat32 = None if self.temporal_kind else torch.empty((n, Tp, 512), dtype=torch.float32, device=self.device)
        return feat16, feat32, (lambda b0, b1: {"feat_out": feat16[b0:b1],
                                                "feat32": None if feat32 is None else feat32[b0:b1]})

    def _temporal_or_features(self, feat16, feat32, n, stages=None):
        if self.temporal_kind is None:
            return feat32
        return (self.gru_tmajor if self.temporal_kind == "gru" else self.mha_tmajor)(feat16, n, stages)

    def _run(self, n, Tp, conv_call, stages=None, want_norm_att=False, out=None):
        """Shared tail of forward / forward_windows: conv stack per micro-batch (conv_call(b0, b1, feat16, feat32,
        stages)), temporal block and head over the whole batch.  out=(clipwise [n, C], framewise [n, frames, C]):
        preallocated destinations -- may be slices of a peer GPU's buffer (dist.PeerGather)."""
        self._acquire_stream(torch.cuda.current_stream(self.device))
        feat16, feat32, slot = self._alloc_features(n, Tp)
        conv_call(slot)
        x = self._temporal_or_features(feat16, feat32, n, stages)
        if x.dim() == 5:
            feat16 = feat16[:, :n].transpose(0, 1)  # clip-major view for the stage dump
        wants_cla = self.model_type in ("Cnn_9layers_Gru_FrameAtt", "Cnn_9layers_FrameAtt")
        clip, frame, cla, natt = self.head(x, self.frames_for(Tp), want_cla=wants_cla, want_norm_att=want_norm_att, n=n,
                                           out=out)
        if x.dim() == 5 and (stages is not None or not wants_cla):
            x = blocks_to_rows(x, n, Tp)  # clip-major view of the GRU output (stage dump / 'embedding' of *_FrameAvg)
        out = {"framewise_output": frame, "clipwise_output": clip, "embedding": self._embedding(x, cla, feat32)}
        return out, feat16, x, natt

    @_on_device
    def forward_windows(self, recording, window_samples, stride_samples, n_windows, micro_batch=DEFAULT_MICRO_BATCH, variant=4,
                        offsets=None):
        """Run the model on `n_windows` overlapping windows of one 1-D recording (f32 or int16, on device):
        window k = recording[k*stride : k*stride + window_samples], zero padded past the end.  Returns the same
        dict as forward() with batch dimension = windows (the per-window calls of predict.py:311-313 as one batch).
        offsets: int64 CUDA tensor [n_windows] of window starts (overrides the constant stride)."""
        if recording.dim() != 1 or recording.device != self.device:
            raise ValueError("recording must be a 1-D tensor on %s" % (self.device,))
        if recording.dtype != torch.int16:
            recording = recording.float()
        recording = recording.contiguous()
        T = window_samples // self.front.hop + 1
        self._check_frames(T)

        def conv_call(slot):
            mb_cap = clamp_micro_batch(micro_batch, T)
            for b0 in range(0, n_windows, mb_cap):
                b1 = min(n_windows, b0 + mb_cap)
                if offsets is not None:
                    self.conv_stack(recording, variant=variant, windows=(b1 - b0, window_samples, offsets[b0:b1]),
                                    **slot(b0, b1))
                else:
                    self.conv_stack(recording[b0 * stride_samples:], variant=variant,
                                    windows=(b1 - b0, window_samples, stride_samples), **slot(b0, b1))

        with self._lock:
            return self._run(n_windows, T // 8, conv_call)[0]

    @_on_device
    def forward(self, wave, micro_batch=DEFAULT_MICRO_BATCH, variant=4, return_stages=False, out=None):
        """wave [B, L] f32 on self.device -> reference output dict (models.py:683-686 / :1072-1075).
        out=(clipwise, framewise): write the two result tensors into these preallocated buffers."""
        if wave.dim() != 2:
            raise ValueError("input must be (batch_size, data_length)")
        if wave.device != self.device:
            raise ValueError("input is on %s, packed weights are on %s" % (wave.device, self.device))
        if wave.dtype != torch.int16:  # int16 PCM is consumed as is (x = q / 32767 inside the front-end)
            wave = wave.float()
        wave = wave.contiguous()
        B, L = wave.shape
        T = L // self.front.hop + 1
        self._check_frames(T)
        stages = {} if return_stages else None

        def conv_call(slot):
            mb_cap = clamp_micro_batch(micro_batch, T)
            for b0 in range(0, B, mb_cap):
                b1 = min(B, b0 + mb_cap)
                self.conv_stack(wave[b0:b1], variant=variant,
                                stages=stages if (return_stages and b0 == 0) else None, **slot(b0, b1))

        with self._lock:
            out, feat16, x, natt = self._run(B, T // 8, conv_call, stages, want_norm_att=return_stages, out=out)
        if return_stages:
            stages["feat"] = feat16
            stages["temporal"] = x
            stages["norm_att"] = natt
            return out, stages
        return out
