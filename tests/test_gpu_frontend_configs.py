"""The front-end (sed_frontend_logmel, sed_spectrogram_f32, sed_logmel_rows_f32) at the launch configurations the
default path runs, against a float64 reference of the same operation on the same float32 samples:

  * production batches (1036 clips at 8 / 16 kHz, 128 at 32 kHz): dozens of work items per persistent block, so the
    claim loop, the double-buffered prefetch and the mbarrier parity run; every clip must equal the same clip launched
    3 at a time (one item per block) bit for bit;
  * frame counts around the frames-per-item boundary, odd frame counts and the shortest clip;
  * strided and offset-table windows, odd and unsorted offsets, windows past total_len in a buffer that holds NaN
    there, and an output that is the leading rows of a larger NaN-filled buffer;
  * an unaligned waveform pointer and hops that turn the bulk copy off, hop > n_fft / 2 and hop > n_fft;
  * power mode per bin (DC and Nyquist included), the mel-rows kernel at 300 007 rows, two launches on two streams;
  * the pair-coupling probe: the kernel transforms frames 2j and 2j + 1 as one complex FFT, so a quiet frame packed
    with a loud one must still meet the log-mel tolerance;
  * a hop too large for the staging buffers is refused with the hop limit in the message.

Error metric of a power bin (or of a mel band's power): |got - ref| / (band weight sum * N * (||w x_a||^2 + ||w x_b||^2))
with a, b the two frames of the kernel's pair -- what a packed float32 FFT can promise.  The log-mel is held to the
tolerance |a - b| <= 1e-4 * max(|b|, 1) dB wherever the float64 band power is well above amin, and to exactly
10 log10(amin) where it is below amin / 2.  Every bound is a small factor above the error measured on a B200; run with
-s to see the measured values.  The reference self-checks at the top need no GPU."""
import re

import numpy as np
import pytest
import torch

import sed_oracle as so
import stream_oracle as sto
from sed_b200 import capi, engine, melbank, stft, synth

gpu = pytest.mark.gpu
DEV = torch.device("cuda:0")
AMIN = 1e-10
FLOOR = np.float32(-100.0)          # 10 log10(amin) - db_offset with amin = 1e-10, ref = 1
SR_OF = {256: 8000, 512: 16000, 1024: 32000}
WELL_ABOVE = 4 * AMIN              # band powers held to the log-mel tolerance
# bounds; the maxima measured over the whole file on a B200 (1000 W power limit) are 6.3e-8, 4.1e-8 and 5.3e-7, and
# the worst log-mel error is 0.70 x the tolerance (frame-count tails, n_fft 1024, int16)
POWER_BOUND = 2.0 ** -21           # power bin error / pair energy
MEL_BOUND = 2.0 ** -22             # mel band power error / (weight sum * pair energy)
ROWS_BOUND = 2.0 ** -19            # sed_logmel_rows_f32: error / sum of |terms|
QUIET = 2.0 ** -10                 # probe: a frame with less than this share of its partner's energy


def report(what, **vals):
    print("\n%s: %s" % (what, ", ".join("%s %s" % (k, ("%.3e" % v) if isinstance(v, float) else v)
                                         for k, v in vals.items())))


def fpb(n_fft, int16):
    """Frames per work item of the shipped kernels (three-pass: 4 warps x 2 pairs; two-pass at 1024: 6 warps x 1 pair),
    doubled for 2-byte samples."""
    return (12 if n_fft == 1024 else 16) * (2 if int16 else 1)


def constants(n_fft, sr=None):
    """(conv_real, conv_imag, melW) of the preset that owns n_fft."""
    sr = sr or SR_OF[n_fft]
    _, _, fmin, fmax = synth.PRESETS[sr]
    wr, wi = melbank.windowed_dft_kernels(n_fft, n_fft, "hann")
    return wr, wi, melbank.mel_filterbank(sr, n_fft, 64, fmin, fmax)


_PLANS = {}


def plan(n_fft, hop=None, is_log=True, mel=True):
    hop = hop or synth.PRESETS[SR_OF[n_fft]][1]
    key = (n_fft, hop, is_log, mel)
    if key not in _PLANS:
        wr, wi, melW = constants(n_fft)
        _PLANS[key] = engine.FrontendPlan(wr, wi, n_fft, hop, melW if mel else None, DEV, is_log=is_log)
    return _PLANS[key]


def as_f32(q):
    """float32 samples of int16 PCM as the kernel converts them: q / 32767, correctly rounded."""
    q = np.asarray(q)
    return q.astype(np.float32) / np.float32(32767) if q.dtype == np.int16 else q.astype(np.float32)


def clips(n, L, seed, sr=16000):
    """int16 [n, L]: noise at a per-clip level (40 dB of spread), a tone in half of the clips, digital silence in some."""
    rng = np.random.default_rng(seed)
    t = np.arange(L) / sr
    x = 0.2 * rng.standard_normal((n, L)) * 10.0 ** -rng.uniform(0, 2, (n, 1))
    f0 = rng.uniform(0.01, 0.45, (n, 1)) * sr
    x += 0.4 * np.sin(2 * np.pi * f0 * t + rng.uniform(0, 6, (n, 1))) * (rng.uniform(size=(n, 1)) < 0.5)
    for i in range(0, n, 3):
        s0 = int(rng.integers(0, L))
        x[i, s0:s0 + int(rng.integers(1, L // 2 + 2))] = 0.0
    return np.round(np.clip(x, -1, 1) * 32767).astype(np.int16)


def ref_windows(rec, offsets, L, total_len):
    """Windows as predict.py slices them: rec[off : off + L], zero past total_len."""
    rec = np.asarray(rec)[:total_len]
    out = np.zeros((len(offsets), L), rec.dtype)
    for i, o in enumerate(offsets):
        seg = rec[o:o + L]
        out[i, :len(seg)] = seg
    return out


class Ref:
    """float64 front-end of clips x [n, L] (float32 or int16 samples): np.pad reflect, frames at hop, float32 window
    as float64, np.fft.rfft, |X|^2, float32 mel matrix as float64, 10 log10(max(., amin)).

    pair [n, T]: N (||w x_a||^2 + ||w x_b||^2) of the kernel's pair (frames 2j, 2j + 1).  For an odd T the last pair's
    second frame lies past the clip; the kernel still transforms it from its staging rule (reflection at L - 1, zero
    where the reflected index is negative), so its energy is computed here by that rule."""

    def __init__(self, x, n_fft, hop, window, melW=None):
        x = as_f32(x).astype(np.float64)
        n, L = x.shape
        pad = n_fft // 2
        win = np.asarray(window, dtype=np.float32).astype(np.float64)
        T = L // hop + 1
        self.T = T
        xp = np.pad(x, ((0, 0), (pad, pad)), mode="reflect")
        idx = np.arange(T)[:, None] * hop + np.arange(n_fft)[None, :]
        power = np.empty((n, T, n_fft // 2 + 1))
        energy = np.empty((n, T + (T & 1)))
        for c in range(n):  # one clip at a time: the frame matrix of a whole batch would not fit comfortably
            fr = xp[c][idx] * win
            X = np.fft.rfft(fr, axis=-1)
            power[c] = X.real ** 2 + X.imag ** 2
            energy[c, :T] = (fr ** 2).sum(-1)
        if T & 1:  # the phantom partner of the last frame
            i = T * hop - pad + np.arange(n_fft)
            i = np.where(i < 0, -i, i)
            i = np.where(i >= L, 2 * (L - 1) - i, i)
            ok = (i >= 0) & (i < L)
            energy[:, T] = ((np.where(ok, x[:, np.clip(i, 0, L - 1)], 0.0) * win) ** 2).sum(-1)
        pe = energy[:, 0::2] + energy[:, 1::2]
        self.pair = n_fft * np.repeat(pe, 2, axis=1)[:, :T]
        self.energy = energy[:, :T]
        self.power = power
        if melW is not None:
            W = np.asarray(melW, dtype=np.float32).astype(np.float64)
            self.mel = power @ W
            self.wsum = W.sum(0)
            self.logmel = 10.0 * np.log10(np.maximum(self.mel, AMIN))


def rel_to_pair(d, denom):
    """|d| / denom, infinite where denom is 0 and d is not (a silent pair must give exactly 0)."""
    d = np.abs(np.asarray(d, dtype=np.float64))
    with np.errstate(divide="ignore", invalid="ignore"):
        r = d / denom
    return np.where(d == 0, 0.0, r)


def power_err(got, ref):
    return rel_to_pair(np.asarray(got, np.float64) - ref.power, ref.pair[..., None]).max()


def mel_err(got, ref):
    return rel_to_pair(np.asarray(got, np.float64) - ref.mel, ref.pair[..., None] * ref.wsum).max()


def logmel_ratio(got, ref, frames=None):
    """Worst |got - ref| / (1e-4 max(|ref|, 1)) over the bands well above amin (of `frames` [n, T], a mask, if given);
    asserts the exact floor below amin / 2."""
    got = np.asarray(got, np.float64)
    low = ref.mel < AMIN / 2
    assert np.all(got[low] == FLOOR), "bands below amin / 2 not at the floor: %s" % got[low][got[low] != FLOOR][:5]
    well = ref.mel > WELL_ABOVE
    if frames is not None:
        well &= frames[..., None]
    if not well.any():
        return 0.0
    return (np.abs(got - ref.logmel)[well] / (1e-4 * np.maximum(np.abs(ref.logmel[well]), 1.0))).max()


def bits(t):
    return t.contiguous().view(torch.int32)


def launch_logmel(p, buf, B, L, total_len, out, stride=1, offsets=None):
    """sed_frontend_logmel through the C ABI, for a total_len smaller than the buffer."""
    lib = capi.load()
    rc = lib.sed_frontend_logmel(capi.ptr(buf), 1 if buf.dtype == torch.int16 else 0, B, L, stride,
                                 capi.ptr(offsets), total_len, p.n_fft, p.hop, capi.ptr(p.window),
                                 capi.ptr(p.twiddle), capi.ptr(p.mel_lo), capi.ptr(p.mel_len), capi.ptr(p.mel_off),
                                 capi.ptr(p.mel_val), p.n_mels, p.amin, p.db_offset, p.is_log, None, None,
                                 capi.ptr(out), capi.current_stream(DEV))
    capi.check(rc, "sed_frontend_logmel")
    return out


def device_wave(q, dtype):
    return torch.from_numpy(q if dtype == "i16" else as_f32(q)).to(DEV)


# ------------------------------------------------------------------------------------------------ reference self-checks
@pytest.mark.parametrize("sr", [8000, 16000, 32000])
def test_reference_matches_the_conv1d_oracle(sr):
    """The float64 reference is sed_oracle.spectrogram + sed_oracle.logmel (the reference's float32 conv1d DFT) within
    float32 accuracy, and its pair energy bounds every frame's own energy."""
    n_fft, hop, _, _ = synth.PRESETS[sr]
    wr, wi, melW = constants(n_fft)
    q = clips(3, 3 * n_fft + 7, seed=sr)
    x = as_f32(q)
    ref = Ref(q, n_fft, hop, wr[0, 0].numpy(), melW.numpy())
    spec = so.spectrogram(torch.from_numpy(x), wr, wi, n_fft, hop)[:, 0]
    lm = so.logmel(spec, melW)
    assert spec.shape == ref.power.shape
    assert power_err(spec.numpy(), ref) < 2.0 ** -19
    assert logmel_ratio(lm.numpy(), ref) < 1.0
    assert np.all(ref.pair >= n_fft * ref.energy)


def test_reference_windows_match_the_stream_oracle():
    """ref_windows slices like stream_oracle (rec[s : s + L] zero padded to L) for strided and offset windows that run
    past the end of the recording, with the recording cut at total_len."""
    rng = np.random.default_rng(5)
    rec = rng.standard_normal(10007).astype(np.float32)
    for total, L, starts in ((10007, 1600, list(range(0, 10007, 997))),
                             (9001, 1601, [5, 0, 1, 3333, 0, 8999, 9000, 9001, 7]),
                             (8000, 1600, [k * 1600 for k in range(6)])):
        want = np.stack([sto.pad_truncate_sequence(rec[:total][s:s + L], L) for s in starts])
        got = ref_windows(rec, starts, L, total)
        assert got.dtype == np.float32 and np.array_equal(got, want.astype(np.float32))
        assert np.all(got[np.array(starts) >= total] == 0)


# ------------------------------------------------------------------------------------------------ production batches
PROD_B = {8000: 1036, 16000: 1036, 32000: 128}


def production_clips(B, L, sr, seed):
    """int16 [B, L] on the device: noise at a per-clip level (1e-2 .. 1 of 0.2 rms), tone bursts, one stretch of digital
    silence per clip starting at an arbitrary sample."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    u = lambda *s: torch.rand(*s, generator=g, device=DEV)  # noqa: E731
    t = torch.arange(L, device=DEV, dtype=torch.float32) / sr
    x = 0.2 * 10.0 ** (-2 * u(B, 1)) * torch.randn(B, L, generator=g, device=DEV)
    f0 = (0.01 + 0.44 * u(B, 1)) * sr
    gate = (torch.sin(2 * np.pi * (0.3 + u(B, 1)) * t) > 0.3).float()
    x += 0.5 * torch.sin(2 * np.pi * f0 * t + 6 * u(B, 1)) * gate
    n = torch.arange(L, device=DEV)
    s0 = (u(B, 1) * 0.8 * L).long()
    s1 = s0 + ((0.02 + 0.2 * u(B, 1)) * L).long()
    x[(n >= s0) & (n < s1)] = 0.0
    return torch.round(x.clamp(-1, 1) * 32767).to(torch.int16)


def in_threes(fn, wave):
    return torch.cat([fn(wave[i:i + 3]) for i in range(0, wave.shape[0], 3)])


@gpu
@pytest.mark.parametrize("sr", [8000, 16000, 32000])
def test_production_batch_equals_small_launches_and_float64(sr):
    """B = 1036 (8 / 16 kHz) and 128 (32 kHz) clips of 10 s: 56 to 110 (16 kHz), 41 to 36 (32 kHz) work items per
    block.  Log-mel and mel power (float32 and int16 input) and the power spectrogram (float32) equal the same clips
    launched 3 at a time bit for bit, int16 equals float32 bit for bit, and the first, the last and 32 random clips
    match float64."""
    n_fft, hop, _, _ = synth.PRESETS[sr]
    B, L = PROD_B[sr], 10 * sr
    q = production_clips(B, L, sr, seed=sr + 1)
    q_cpu = q.cpu().numpy()
    wave = torch.from_numpy(as_f32(q_cpu)).to(DEV)
    rng = np.random.default_rng(sr)
    pick = np.unique(np.concatenate([[0, B - 1], rng.choice(np.arange(1, B - 1), 32, replace=False)]))
    wr, _, melW = constants(n_fft)
    ref = Ref(q_cpu[pick], n_fft, hop, wr[0, 0].numpy(), melW.numpy())
    res = {}
    for is_log in (True, False):
        p = plan(n_fft, is_log=is_log)
        full = engine.logmel_forward(p, wave)
        assert torch.equal(bits(full), bits(in_threes(lambda w: engine.logmel_forward(p, w), wave)))
        full16 = engine.logmel_forward(p, q)
        assert torch.equal(bits(full16), bits(full)), "int16 input differs from its float32 samples"
        got = full[torch.from_numpy(pick).to(DEV)].cpu().numpy()
        res["logmel" if is_log else "mel"] = logmel_ratio(got, ref) if is_log else mel_err(got, ref)
        del full, full16
    p = plan(n_fft, mel=False)
    spec = engine.spectrogram_forward(p, wave)
    assert torch.equal(bits(spec), bits(in_threes(lambda w: engine.spectrogram_forward(p, w), wave)))
    res["power"] = power_err(spec[torch.from_numpy(pick).to(DEV), 0].cpu().numpy(), ref)
    report("production sr %d B %d" % (sr, B), logmel_vs_tol=res["logmel"], mel=res["mel"], power=res["power"])
    assert res["logmel"] <= 1.0 and res["mel"] <= MEL_BOUND and res["power"] <= POWER_BOUND


@gpu
def test_two_streams_equal_their_serial_results():
    """Two production-size launches (16 kHz float32 and 8 kHz int16, 1036 clips each) issued back to back on two
    streams: each equals its serial result bit for bit (each launch owns a claim counter)."""
    p16, p8 = plan(512), plan(256)
    a = production_clips(1036, 160000, 16000, seed=11).float() / 32767.0
    b = production_clips(1036, 80000, 8000, seed=12)
    ra, rb = engine.logmel_forward(p16, a), engine.logmel_forward(p8, b)
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(DEV), torch.cuda.Stream(DEV)
    s1.wait_stream(torch.cuda.current_stream(DEV))
    s2.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(s1):
        oa = engine.logmel_forward(p16, a)
    with torch.cuda.stream(s2):
        ob = engine.logmel_forward(p8, b)
    torch.cuda.synchronize()
    assert torch.equal(bits(oa), bits(ra)) and torch.equal(bits(ob), bits(rb))


# ------------------------------------------------------------------------------------------------ frame-count tails
@gpu
@pytest.mark.parametrize("dtype", ["f32", "i16"])
@pytest.mark.parametrize("n_fft", [256, 512, 1024])
def test_frame_count_tails(n_fft, dtype):
    """T = k FPB, k FPB + 1, k FPB - 1 (odd: the last pair has no second frame), L at both ends of each T, and the
    shortest clip L = n_fft / 2 + 1, against float64."""
    hop = synth.PRESETS[SR_OF[n_fft]][1]
    F = fpb(n_fft, dtype == "i16")
    Ls = [n_fft // 2 + 1, n_fft // 2 + 2]
    for T in (3 * F, 3 * F + 1, 3 * F - 1, F + 1):
        Ls += [(T - 1) * hop, T * hop - 1]
    wr, _, melW = constants(n_fft)
    worst = dict(logmel=0.0, mel=0.0, power=0.0)
    for L in Ls:
        q = clips(5, L, seed=L, sr=SR_OF[n_fft])
        w = device_wave(q, dtype)
        ref = Ref(q, n_fft, hop, wr[0, 0].numpy(), melW.numpy())
        lm = engine.logmel_forward(plan(n_fft), w).cpu().numpy()
        mel = engine.logmel_forward(plan(n_fft, is_log=False), w).cpu().numpy()
        assert lm.shape == (5, ref.T, 64)
        worst["logmel"] = max(worst["logmel"], logmel_ratio(lm, ref))
        worst["mel"] = max(worst["mel"], mel_err(mel, ref))
        if dtype == "f32":
            spec = engine.spectrogram_forward(plan(n_fft, mel=False), w)[:, 0].cpu().numpy()
            worst["power"] = max(worst["power"], power_err(spec, ref))
    report("tails n_fft %d %s" % (n_fft, dtype), logmel_vs_tol=worst["logmel"], mel=worst["mel"], power=worst["power"])
    assert worst["logmel"] <= 1.0 and worst["mel"] <= MEL_BOUND and worst["power"] <= POWER_BOUND


# ------------------------------------------------------------------------------------------------ window layouts
@gpu
@pytest.mark.parametrize("layout", ["stride", "offsets"])
@pytest.mark.parametrize("dtype", ["f32", "i16"])
@pytest.mark.parametrize("n_fft", [256, 512, 1024])
def test_window_layouts(n_fft, dtype, layout):
    """Windows of one recording read in place -- strided (clip_stride < L, odd) or through an unsorted offset table
    with repeated, odd and near-zero starts -- the last ones running past total_len into a buffer that holds NaN
    (float32) or full scale (int16) there.  Equal to the same windows materialised as a dense batch bit for bit and
    to float64; the output is the leading rows of a NaN-filled buffer whose other rows stay NaN."""
    sr = SR_OF[n_fft]
    hop = synth.PRESETS[sr][1]
    L = 23 * hop + 5
    total = 7 * L + 123
    rec = clips(1, total, seed=n_fft + (dtype == "i16"), sr=sr)[0]
    buf = np.concatenate([rec, np.full(4 * L, 32767, np.int16)])
    if dtype == "f32":
        buf = as_f32(buf)
        buf[total:] = np.nan
    if layout == "stride":
        stride = L // 3 + 1
        starts = list(range(0, total + L // 2, stride))
        offs = None
    else:
        stride = 1
        starts = [5, 0, 1, 2 * L + 3, 0, 3, total - L // 2, 7, total - 1, 1, L - 1, total, 4 * L + 1, 2]
        offs = torch.tensor(starts, dtype=torch.int64, device=DEV)
    B = len(starts)
    T = L // hop + 1
    dev_buf = torch.from_numpy(buf).to(DEV)
    dense = ref_windows(buf, starts, L, total)
    dense_dev = torch.from_numpy(dense).to(DEV)
    wr, _, melW = constants(n_fft)
    ref = Ref(dense, n_fft, hop, wr[0, 0].numpy(), melW.numpy())
    res = {}
    for is_log in (True, False):
        p = plan(n_fft, is_log=is_log)
        big = torch.full((B + 3, T, 64), float("nan"), device=DEV)
        launch_logmel(p, dev_buf, B, L, total, big[:B], stride=stride, offsets=offs)
        assert torch.isnan(big[B:]).all(), "rows past B x T were written"
        got = big[:B]
        assert not torch.isnan(got).any(), "a sample past total_len was read"
        assert torch.equal(bits(got), bits(engine.logmel_forward(p, dense_dev)))
        res["logmel" if is_log else "mel"] = (logmel_ratio if is_log else mel_err)(got.cpu().numpy(), ref)
    report("layout %s n_fft %d %s B %d" % (layout, n_fft, dtype, B), logmel_vs_tol=res["logmel"], mel=res["mel"])
    assert res["logmel"] <= 1.0 and res["mel"] <= MEL_BOUND


# ------------------------------------------------------------------------------------------------ alignment and hops
@gpu
@pytest.mark.parametrize("dtype", ["f32", "i16"])
@pytest.mark.parametrize("n_fft", [256, 512, 1024])
def test_unaligned_wave_pointer(n_fft, dtype):
    """A waveform batch that starts one element past an aligned address (rec[1:]): the bulk copy is off for every
    segment; log-mel and power equal the aligned launch bit for bit and match float64."""
    sr = SR_OF[n_fft]
    hop = synth.PRESETS[sr][1]
    B, L = 6, 2 * sr
    q = clips(B, L, seed=3 + n_fft, sr=sr)
    w = device_wave(q, dtype)
    store = torch.zeros(B * L + 1, dtype=w.dtype, device=DEV)
    store[1:] = w.reshape(-1)
    w1 = store[1:].view(B, L)
    assert w1.data_ptr() % 16 != 0
    wr, _, melW = constants(n_fft)
    ref = Ref(q, n_fft, hop, wr[0, 0].numpy(), melW.numpy())
    lm = engine.logmel_forward(plan(n_fft), w1)
    assert torch.equal(bits(lm), bits(engine.logmel_forward(plan(n_fft), w)))
    mel = engine.logmel_forward(plan(n_fft, is_log=False), w1)
    r_lm, r_mel = logmel_ratio(lm.cpu().numpy(), ref), mel_err(mel.cpu().numpy(), ref)
    r_pow = 0.0
    if dtype == "f32":
        spec = engine.spectrogram_forward(plan(n_fft, mel=False), w1)
        assert torch.equal(bits(spec), bits(engine.spectrogram_forward(plan(n_fft, mel=False), w)))
        r_pow = power_err(spec[:, 0].cpu().numpy(), ref)
    report("unaligned n_fft %d %s" % (n_fft, dtype), logmel_vs_tol=r_lm, mel=r_mel, power=r_pow)
    assert r_lm <= 1.0 and r_mel <= MEL_BOUND and r_pow <= POWER_BOUND


HOPS = [(256, 81), (256, 200), (256, 333), (512, 161), (512, 300), (512, 700), (1024, 333), (1024, 700), (1024, 1500)]


@gpu
@pytest.mark.parametrize("dtype", ["f32", "i16"])
@pytest.mark.parametrize("n_fft,hop", HOPS)
def test_non_preset_hops(n_fft, hop, dtype):
    """Hops that break the 16-byte conditions of the bulk copy (161 at 512, every odd hop), hop > n_fft / 2 and
    hop > n_fft (frames skip samples), against float64."""
    sr = SR_OF[n_fft]
    L = 40 * hop + 17
    q = clips(4, L, seed=hop, sr=sr)
    w = device_wave(q, dtype)
    wr, _, melW = constants(n_fft)
    ref = Ref(q, n_fft, hop, wr[0, 0].numpy(), melW.numpy())
    r_lm = logmel_ratio(engine.logmel_forward(plan(n_fft, hop), w).cpu().numpy(), ref)
    r_mel = mel_err(engine.logmel_forward(plan(n_fft, hop, is_log=False), w).cpu().numpy(), ref)
    r_pow = 0.0
    if dtype == "f32":
        r_pow = power_err(engine.spectrogram_forward(plan(n_fft, hop, mel=False), w)[:, 0].cpu().numpy(), ref)
    report("hop %d n_fft %d %s" % (hop, n_fft, dtype), logmel_vs_tol=r_lm, mel=r_mel, power=r_pow)
    assert r_lm <= 1.0 and r_mel <= MEL_BOUND and r_pow <= POWER_BOUND


# ------------------------------------------------------------------------------------------------ power mode, mel rows
@gpu
@pytest.mark.parametrize("n_fft", [256, 512, 1024])
def test_power_mode_per_bin_with_dc_and_nyquist(n_fft):
    """sed_spectrogram_f32 per bin, on signals whose DC and Nyquist bins carry a large share of the energy (offset,
    alternating sign, noise): every bin including k = 0 and k = n_fft / 2 within the pair-energy bound."""
    hop = synth.PRESETS[SR_OF[n_fft]][1]
    B, L = 4, 30 * hop + 3
    rng = np.random.default_rng(n_fft)
    n = np.arange(L)
    x = (rng.uniform(-0.4, 0.4, (B, 1)) + rng.uniform(-0.4, 0.4, (B, 1)) * (-1.0) ** n
         + 0.05 * rng.standard_normal((B, L))).astype(np.float32)
    wr, _, _ = constants(n_fft)
    ref = Ref(x, n_fft, hop, wr[0, 0].numpy())
    got = engine.spectrogram_forward(plan(n_fft, mel=False), torch.from_numpy(x).to(DEV))[:, 0].cpu().numpy()
    F = n_fft // 2 + 1
    err = rel_to_pair(got.astype(np.float64) - ref.power, ref.pair[..., None])
    share = (ref.power[..., [0, F - 1]] / ref.pair[..., None]).min()
    report("power n_fft %d" % n_fft, all_bins=err.max(), dc=err[..., 0].max(), nyquist=err[..., F - 1].max(),
           min_share_of_dc_nyquist=share)
    assert share > 1e-5  # the edge bins are large: a wrong scale there cannot hide below the bound
    assert err.max() <= POWER_BOUND


@gpu
@pytest.mark.parametrize("n_fft", [512, 1024])
def test_logmel_rows_at_300k_rows(n_fft):
    """sed_logmel_rows_f32 on 300 007 rows (9.6 M warps), is_log 0 and 1, against the float64 projection: error
    relative to the sum of |terms|, the log-mel tolerance, exact floor for zero rows."""
    R, F = 300007, n_fft // 2 + 1
    g = torch.Generator(device=DEV).manual_seed(n_fft)
    spec = torch.rand(R, F, generator=g, device=DEV) ** 4 * 10.0 ** (6 * torch.rand(R, 1, generator=g, device=DEV) - 8)
    spec[::997] = 0.0
    _, _, melW = constants(n_fft)
    W = melW.double().to(DEV)
    want = spec.double() @ W
    res = {}
    for is_log in (False, True):
        got = engine.logmel_rows_forward(plan(n_fft, is_log=is_log), spec).double()
        assert got.shape == (R, 64)
        if is_log:
            lw = 10.0 * torch.log10(want.clamp(min=AMIN))
            well, low = want > WELL_ABOVE, want < AMIN / 2
            assert bool((got[low] == float(FLOOR)).all())
            res["logmel_vs_tol"] = ((got - lw).abs() / (1e-4 * lw.abs().clamp(min=1.0)))[well].max().item()
        else:
            res["mel"] = ((got - want).abs() / want.clamp(min=1e-300)).max().item()
    report("logmel rows n_fft %d" % n_fft, **res)
    assert res["mel"] <= ROWS_BOUND and res["logmel_vs_tol"] <= 1.0


# ------------------------------------------------------------------------------------------------ pair-coupling probe
def onset_clips(n_fft, hop, kind, seed):
    """Digital silence, then full-scale noise (or a full-scale sine) from sample s on, with s 0 .. 16 samples before the
    last sample of frame 10 (even: first of its pair) and of frame 11 (odd)."""
    L = 16 * hop + n_fft
    rng = np.random.default_rng(seed)
    rows = []
    for f in (10, 11):
        end = f * hop + n_fft // 2 - 1
        for d in range(17):
            if kind == "noise":
                sig = rng.uniform(-1, 1, L)
            else:
                sig = np.sin(2 * np.pi * 0.1234567 * np.arange(L) + rng.uniform(0, 6))
            sig[:end - d] = 0.0
            rows.append(sig)
    return np.round(np.stack(rows) * 32767).astype(np.int16)


def probe(n_fft, hop, q, spec_fn, lm_fn, window, melW):
    """(kernel's worst log-mel error / tolerance, the same over the quiet frames (less than QUIET of their partner's
    energy), the float32 conv1d's over all frames, power error / pair energy, weakest pair share)"""
    ref = Ref(q, n_fft, hop, window, melW)
    lm = lm_fn()
    r_kernel = logmel_ratio(lm, ref)
    quiet = ref.energy < QUIET * (ref.pair / n_fft - ref.energy)
    assert quiet.sum() >= 20
    r_quiet = logmel_ratio(lm, ref, quiet)
    wr, wi = melbank.windowed_dft_kernels(n_fft, n_fft, "hann")
    conv = so.logmel(so.spectrogram(torch.from_numpy(as_f32(q)), wr, wi, n_fft, hop), torch.as_tensor(melW))[:, 0]
    well = ref.mel > WELL_ABOVE
    r_conv = (np.abs(conv.numpy() - ref.logmel)[well] / (1e-4 * np.maximum(np.abs(ref.logmel[well]), 1.0))).max()
    r_pow = power_err(spec_fn(), ref)
    e = ref.energy
    share = (np.minimum(e[:, 0::2][:, :e.shape[1] // 2], e[:, 1::2]) /
             np.maximum(e[:, 0::2][:, :e.shape[1] // 2], e[:, 1::2]).clip(min=1e-300))
    return r_kernel, r_quiet, r_conv, r_pow, share[share > 0].min()


@gpu
@pytest.mark.parametrize("kind", ["noise", "sine"])
@pytest.mark.parametrize("n_fft", [256, 512, 1024])
def test_pair_coupling_probe(n_fft, kind):
    """A nearly silent frame packed with a full-scale one: the log-mel of the quiet frame meets the tolerance against
    float64, silent bands are exactly the floor, and the power spectrum stays within the pair-energy bound.  With
    noise every band of every frame meets the tolerance, as the reference's float32 conv1d (every frame alone) does.
    A full-scale sine leaves bands 100 dB and more below it in its loud frames, below float32 resolution for the
    conv1d too (1.8 / 4.2 / 6.2 x the tolerance at 256 / 512 / 1024); there the quiet frames are held to it.
    Measured on a B200, worst error / tolerance at n_fft 256 / 512 / 1024: before the second transform of solo_frame
    0.67 / 0.88 / 1.84 (noise); with it 0.13 / 0.18 / 0.027 (noise), quiet frames of the sine 0.12 / 0.14 / 0.0014."""
    sr = SR_OF[n_fft]
    hop = synth.PRESETS[sr][1]
    q = onset_clips(n_fft, hop, kind, seed=n_fft)
    w = torch.from_numpy(as_f32(q)).to(DEV)
    wr, _, melW = constants(n_fft)
    res = {}
    for dtype, wave in (("f32", w), ("i16", torch.from_numpy(q).to(DEV))):
        r = probe(n_fft, hop, q, lambda: engine.spectrogram_forward(plan(n_fft, mel=False), w)[:, 0].cpu().numpy(),
                  lambda: engine.logmel_forward(plan(n_fft), wave).cpu().numpy(), wr[0, 0].numpy(), melW.numpy())
        res[dtype] = r
        report("probe n_fft %d %s %s" % (n_fft, kind, dtype), kernel_vs_tol=r[0], quiet_frames_vs_tol=r[1],
               conv1d_vs_tol=r[2], power=r[3], weakest_pair_share=r[4])
    for r_kernel, r_quiet, r_conv, r_pow, _ in res.values():
        assert r_quiet <= 1.0 and r_pow <= POWER_BOUND
        if kind == "noise":
            assert r_conv <= 1.0 and r_kernel <= 1.0


@gpu
@pytest.mark.parametrize("n_fft", [256, 512, 1024])
def test_pair_coupling_probe_drop_in_hop_equal_to_n_fft(n_fft):
    """stft.Spectrogram with hop = n_fft (frames do not overlap: a silent frame sits next to a loud one) followed by
    stft.LogmelFilterBank (top_db None) against float64.  Worst error / tolerance measured on a B200 at n_fft 256 /
    512 / 1024: 1.36 / 2.31 / 3.27 before the second transform of solo_frame, 0.16 / 0.61 / 0.030 with it."""
    sr = SR_OF[n_fft]
    _, _, fmin, fmax = synth.PRESETS[sr]
    spec_mod = stft.Spectrogram(n_fft=n_fft, hop_length=n_fft, win_length=n_fft, window="hann", center=True,
                                pad_mode="reflect", freeze_parameters=True).to(DEV)
    mel_mod = stft.LogmelFilterBank(sr=sr, n_fft=n_fft, n_mels=64, fmin=fmin, fmax=fmax, ref=1.0, amin=AMIN,
                                    top_db=None, freeze_parameters=True).to(DEV)
    q = onset_clips(n_fft, n_fft, "noise", seed=n_fft + 1)
    w = torch.from_numpy(as_f32(q)).to(DEV)
    window = spec_mod.stft.conv_real.weight[0, 0].detach().cpu().numpy()
    melW = mel_mod.melW.detach().cpu().numpy()
    spec = spec_mod(w)
    r = probe(n_fft, n_fft, q, lambda: spec[:, 0].cpu().numpy(), lambda: mel_mod(spec)[:, 0].cpu().numpy(),
              window, melW)
    report("drop-in hop = n_fft %d" % n_fft, kernel_vs_tol=r[0], quiet_frames_vs_tol=r[1], conv1d_vs_tol=r[2],
           power=r[3], weakest_pair_share=r[4])
    assert r[2] <= 1.0
    assert r[0] <= 1.0 and r[3] <= POWER_BOUND


# ------------------------------------------------------------------------------------------------ staging limit
@gpu
@pytest.mark.parametrize("mode", ["logmel_f32", "logmel_i16", "power"])
@pytest.mark.parametrize("n_fft", [256, 512, 1024])
def test_hop_beyond_the_staging_limit_is_refused(n_fft, mode):
    """A hop whose staging buffers do not fit in shared memory is refused with SED_ERR_UNSUPPORTED, a message that
    names the largest hop, and no launch (the NaN-filled output stays NaN); that largest hop runs and matches
    float64."""
    sr = SR_OF[n_fft]
    wr, wi, melW = constants(n_fft)
    lib = capi.load()

    def run(hop, out):
        L = 6 * hop + 11
        q = clips(2, L, seed=hop, sr=sr)
        p = engine.FrontendPlan(wr, wi, n_fft, hop, None if mode == "power" else melW, DEV)
        w = device_wave(q, "i16" if mode == "logmel_i16" else "f32")
        T = L // hop + 1
        if out is None:
            out = torch.full((2, T, 64 if mode != "power" else n_fft // 2 + 1), float("nan"), device=DEV)
        if mode == "power":
            rc = lib.sed_spectrogram_f32(capi.ptr(w), 2, L, n_fft, hop, capi.ptr(p.window), capi.ptr(p.twiddle),
                                         capi.ptr(out), capi.current_stream(DEV))
            capi.check(rc, "sed_spectrogram_f32")
        else:
            launch_logmel(p, w, 2, L, 2 * L, out, stride=L)
        return q, out, hop

    big = 40000
    out = torch.full((2, (6 * big + 11) // big + 1, 64 if mode != "power" else n_fft // 2 + 1), float("nan"),
                     device=DEV)
    with pytest.raises(NotImplementedError) as e:
        run(big, out)
    torch.cuda.synchronize()
    assert torch.isnan(out).all()
    msg = str(e.value)
    m = re.search(r"hop <= (\d+)", msg)
    assert m and "hop=%d" % big in msg and "shared memory" in msg, msg
    limit = int(m.group(1))
    report("staging limit n_fft %d %s" % (n_fft, mode), largest_hop=limit)
    assert limit > n_fft
    with pytest.raises(NotImplementedError):
        run(limit + 1, None)
    q, got, hop = run(limit, None)
    ref = Ref(q, n_fft, hop, wr[0, 0].numpy(), None if mode == "power" else melW.numpy())
    if mode == "power":
        assert power_err(got.cpu().numpy(), ref) <= POWER_BOUND
    else:
        assert logmel_ratio(got.cpu().numpy(), ref) <= 1.0
