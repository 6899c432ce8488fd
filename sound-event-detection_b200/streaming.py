"""Streaming prediction: the window loop of the reference's `predict.py` as ONE batched call.

Reference behaviour (pytorch/predict.py:297-349 with --overlap): a recording is cut into `sample_duration`-second
windows advancing by a literal 1 s, each window is run through the model with batch size 1 (a host sync per window),
the framewise outputs are overlap-added (`merge`) and block-averaged (`avg_merge`, utils/utilities.py:405-446).
Here the windows become the batch dimension -- the front-end kernel reads them in place from the recording with a
1-second clip stride -- and merge/avg_merge run as one device kernel, bug-compatible with the numpy code.
"""
import numpy as np
import torch

from . import capi, engine


def _resolve(model, device):
    """(packed model, micro_batch, conv variant) that run `model` on `device`.  An engine.PackedModel runs where it was
    packed (`device` is not used); a drop-in model is packed for `device` (a bare 'cuda' is the current device)."""
    if isinstance(model, engine.PackedModel):
        return model, engine.DEFAULT_MICRO_BATCH, 4
    if model.training:
        raise RuntimeError("inference only -- call .eval()")
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("%s is not a CUDA device; the B200 path has no CPU fallback" % (device,))
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return model._packed_for(device), model.micro_batch, model.conv_variant


def _window_starts(duration, sample_duration, stride):
    """The reference's window loop: a window starts at 0 and every `stride` while `end <= duration`, end updated after
    each window.  The start accumulates `stride` (float accumulation for a float stride, as the reference does)."""
    starts = []
    start, end = 0, 0
    while end <= duration:
        starts.append(start)
        start += stride
        end = start + sample_duration
    return starts


def window_starts(audio_duration, sample_duration, overlap=True):
    """Start times (s) of the windows the reference runs: predict.py:279-281, 297, 334-339."""
    return _window_starts(audio_duration, sample_duration, 1 if overlap else sample_duration)


def _layout(lengths, sample_rate, sample_duration):
    """Recordings of `lengths` samples laid out one after another in one flat buffer, each zero padded up to the end
    of its last window (the reference zero-pads the last window, predict.py:302-305).  Returns the window counts, the
    segment lengths and the host list of window start offsets into the buffer."""
    sr, window_samples = int(sample_rate), int(sample_rate * sample_duration)
    counts, seg_len, offsets, base = [], [], [], 0
    for n in lengths:
        starts = window_starts(n / float(sample_rate), sample_duration, overlap=True)
        counts.append(len(starts))
        need = max(n, starts[-1] * sr + window_samples)
        seg_len.append((need + 7) // 8 * 8)  # keep every segment 16-byte aligned for the cp.async staging
        offsets.extend(base + k * sr for k in range(len(starts)))
        base += seg_len[-1]
    return counts, seg_len, offsets


def _merge_groups(frames, counts, overlap_interval, sample_duration):
    """Merge + avg_merge per recording: `frames` holds the windows of every recording in order, recording f has
    counts[f] of them.  Recordings with the same number of windows are merged by one launch; yields (member indices,
    merged [n_members, total_frames, classes]) per window count, in ascending order."""
    groups, first = {}, 0
    for f, nw in enumerate(counts):
        groups.setdefault(nw, []).append((f, first))
        first += nw
    for nw, members in sorted(groups.items()):
        if all(members[i + 1][1] == members[i][1] + nw for i in range(len(members) - 1)):
            group = frames[members[0][1]:members[0][1] + nw * len(members)]  # contiguous rows: a view
        else:
            rows = torch.tensor([fst + k for _, fst in members for k in range(nw)], dtype=torch.int64).to(frames.device)
            group = frames.index_select(0, rows)
        group = group.view(len(members), nw, frames.shape[1], frames.shape[2])
        yield [f for f, _ in members], engine.window_merge_avg(group, int(overlap_interval), int(sample_duration))


def predict_framewise(model, recording, sample_rate, sample_duration=5, overlap_value=1, return_windows=False):
    """model: a sed_b200 drop-in model in eval mode (or an engine.PackedModel); recording: 1-D float32 / int16
    waveform on the model's CUDA device.  Returns merged framewise probabilities [1, total_frames, 25]
    (what `merged` holds after predict.py:349)."""
    packed, micro_batch, variant = _resolve(model, recording.device)
    audio_duration = recording.numel() / float(sample_rate)
    starts = window_starts(audio_duration, sample_duration, overlap=True)
    n_windows = len(starts)
    window_samples = int(sample_rate * sample_duration)
    with torch.no_grad():
        out = packed.forward_windows(recording, window_samples, int(sample_rate), n_windows, micro_batch=micro_batch,
                                     variant=variant)
        _, merged = next(_merge_groups(out["framewise_output"], [n_windows], int(100 * overlap_value), sample_duration))
    if return_windows:
        return merged, out
    return merged


def predict_framewise_many(model, recordings, sample_rate, sample_duration=5, overlap_value=1):
    """predict_framewise for several recordings in ONE batch (the per-file loop of pytorch/predict.py:264 folded into the
    batch dimension): `recordings` is a list of 1-D float32 / int16 CUDA tensors of one dtype.  Every recording is laid
    out in one buffer, zero padded up to the end of its last window (the reference zero-pads the last window,
    predict.py:302-305), the windows of all recordings are read in place through an offset table, and recordings with
    the same number of windows are merged by one launch.  Returns a list of [1, total_frames, classes] tensors equal,
    bit for bit, to calling predict_framewise per recording."""
    packed, micro_batch, variant = _resolve(model, recordings[0].device)
    dev, dtype = recordings[0].device, recordings[0].dtype
    if any(r.dim() != 1 or r.device != dev or r.dtype != dtype for r in recordings):
        raise ValueError("recordings must be 1-D tensors of one dtype on one CUDA device")
    window_samples = int(sample_rate * sample_duration)
    counts, seg_len, offsets = _layout([r.numel() for r in recordings], sample_rate, sample_duration)
    flat = torch.zeros(sum(seg_len), dtype=dtype, device=dev)
    base = 0
    for r, sl in zip(recordings, seg_len):
        flat[base:base + r.numel()].copy_(r)
        base += sl
    offsets = torch.tensor(offsets, dtype=torch.int64, device=dev)
    with torch.no_grad():
        out = packed.forward_windows(flat, window_samples, 0, int(offsets.numel()), micro_batch=micro_batch,
                                     variant=variant, offsets=offsets)
        merged = [None] * len(recordings)
        for idx, m in _merge_groups(out["framewise_output"], counts, int(100 * overlap_value), sample_duration):
            for j, f in enumerate(idx):
                merged[f] = m[j:j + 1]
    return merged


def _check_channels(channels):
    if not isinstance(channels, (int, np.integer)) or not 1 <= channels <= 8:
        raise ValueError("channels must be an int in 1 .. 8, got %r" % (channels,))
    return int(channels)


def _frames(rec, channels, what):
    """Frames of a [n] (mono) or [n, channels] recording or chunk; ValueError for any other shape."""
    if rec.dim() == 2 and rec.shape[1] == channels or rec.dim() == 1 and channels == 1:
        return int(rec.shape[0])
    raise ValueError("%s must be [n, %d]%s, got shape %s" % (what, channels, " or [n]" if channels == 1 else "",
                                                             tuple(rec.shape)))


def resample(recordings, input_rate, sample_rate, channels=1):
    """librosa.load(path, sr=sample_rate, mono=True) (pytorch/predict.py:288-295) for decoded audio on the device:
    `recordings` is a list of CUDA tensors of one dtype (float32, or int16 PCM read as q / 32767), each [n] or
    [n, channels] at `input_rate`.  The channels are averaged, then the polyphase filter of engine.resample_filter
    resamples to `sample_rate`, every recording in ONE launch.  Returns 1-D float32 CUDA tensors of
    ceil(n * up / down) samples.  Equal rates only downmix (librosa does not resample then)."""
    channels = _check_channels(channels)
    if not recordings:
        raise ValueError("no recordings")
    dev, dtype = recordings[0].device, recordings[0].dtype
    if dtype not in (torch.float32, torch.int16) or dev.type != "cuda":
        raise ValueError("recordings must be float32 or int16 CUDA tensors, got %s on %s" % (dtype, dev))
    if any(r.dtype != dtype or r.device != dev for r in recordings):
        raise ValueError("recordings must be tensors of one dtype on one CUDA device")
    n_in = np.array([_frames(r, channels, "recording") for r in recordings], np.int64)
    plan = engine.resample_plan(input_rate, sample_rate, dev)
    n_out = plan.n_out(n_in)
    table = np.stack([np.cumsum(n_in) - n_in, n_in, np.cumsum(n_out) - n_out, n_out], 1)
    src = torch.cat([r.reshape(-1) for r in recordings])
    dst = torch.empty(max(int(n_out.sum()), 1), dtype=torch.float32, device=dev)
    with torch.no_grad():
        engine.resample(src if src.numel() else dst, channels, torch.from_numpy(table).to(dev), len(recordings),
                        int(n_out.max()), plan, dst)
    return list(dst[:int(n_out.sum())].split(n_out.tolist()))


class HostStreamer:
    """predict_framewise_many for recordings that live in HOST memory, end to end: every recording of a call is copied
    by DMA from the caller's (pinned) buffer straight to its place in one flat device buffer (zero padded up to the end
    of its last window by a device memset; nothing is repacked on the host), the window offset table is built on the
    host, and the merged frames of all recordings come back with one device->host copy per window-count group.  Two staging slots alternate, so the copy in of call k+1 can be queued while call k
    computes (`submit` returns at once, `result` blocks for the oldest call).  Replaces the per-file, per-window loop of
    pytorch/predict.py:264-349, which reads each window back to the host before it runs the next one.

    With `input_rate` (Hz) other than `sample_rate`, or `channels` > 1, recordings are [n] or [n, channels] at
    `input_rate`: they are copied as they are into a device staging buffer and sed_resample downmixes and resamples
    all of them in one launch straight into the padded layout -- equal, bit for bit, to
    predict_framewise_many(model, resample(recordings on the device, input_rate, sample_rate, channels))."""

    def __init__(self, model, sample_rate, sample_duration=5, overlap_value=1, input_rate=None, channels=1):
        self.model, self.sr, self.dur, self.ov = model, int(sample_rate), int(sample_duration), overlap_value
        self.channels = _check_channels(channels)
        self.input_rate = self.sr if input_rate is None else int(input_rate)
        self.resampling = self.input_rate != self.sr or self.channels != 1
        if self.resampling and self.input_rate != self.sr:
            engine.resample_filter(self.input_rate, self.sr)  # ValueError now for a rate pair the filter refuses
        self.slots = [dict(), dict()]
        self.calls = 0
        self.pending = []
        self.copy_stream = None

    def submit(self, recordings, device):
        """recordings: list of CPU tensors (float32 or int16 PCM, one dtype), 1-D at sample_rate -- or, when
        resampling, [n] / [n, channels] at input_rate.  Queues the call; returns a ticket."""
        device = torch.device(device)
        packed, micro_batch, variant = _resolve(self.model, device)
        dtype = recordings[0].dtype
        if self.resampling:
            if any(r.is_cuda or r.dtype != dtype for r in recordings) or dtype not in (torch.float32, torch.int16):
                raise ValueError("recordings must be float32 or int16 CPU tensors of one dtype")
            n_in = np.array([_frames(r, self.channels, "recording") for r in recordings], np.int64)
            plan = engine.resample_plan(self.input_rate, self.sr, device)
            lengths = plan.n_out(n_in).tolist()
        elif any(r.dim() != 1 or r.is_cuda or r.dtype != dtype for r in recordings) or dtype not in (torch.float32, torch.int16):
            raise ValueError("recordings must be 1-D float32 or int16 CPU tensors of one dtype")
        else:
            lengths = [r.numel() for r in recordings]
        window_samples = self.sr * self.dur
        counts, seg_len, offs = _layout(lengths, self.sr, self.dur)
        total = sum(seg_len)
        slot = self.slots[self.calls % 2]
        if "done" in slot:
            slot["done"].synchronize()
        with torch.cuda.device(device):
            if self.copy_stream is None:
                self.copy_stream = torch.cuda.Stream(device)
            compute = torch.cuda.current_stream(device)
            cs = self.copy_stream  # the slot's previous call has finished (host-synchronised above): copy at once,
            with torch.cuda.stream(cs):  # under the kernels of the call queued before this one
                key = (total, dtype, len(recordings))
                if slot.get("key") != key:
                    # allocated on the copy stream, which writes them while the compute stream may still run the
                    # previous call: memory that call's temporaries free on the compute stream is never handed out here
                    slot["dev"] = torch.empty(total, dtype=torch.float32 if self.resampling else dtype, device=device)
                    slot["off_host"] = torch.zeros(sum(counts), dtype=torch.int64).pin_memory()
                    slot["off_dev"] = torch.empty(sum(counts), dtype=torch.int64, device=device)
                    for t in (slot["dev"], slot["off_dev"]):
                        t.record_stream(compute)
                    slot["key"] = key
                    slot["out"] = {}
                slot["off_host"].copy_(torch.tensor(offs, dtype=torch.int64))
                slot["src"] = list(recordings)  # keeps pinned sources alive until their asynchronous copies have run
                if self.resampling:
                    self._stage_raw(slot, recordings, n_in, lengths, seg_len, device, compute)
                else:
                    # the DMA engine does the layout: every recording goes straight from the caller's (pinned) buffer to
                    # its place in the flat device buffer -- no host-side repacking; the zero padding is a device memset
                    base = 0
                    for r, sl in zip(recordings, seg_len):
                        slot["dev"][base:base + r.numel()].copy_(r, non_blocking=True)
                        if r.numel() < sl:
                            slot["dev"][base + r.numel():base + sl].zero_()
                        base += sl
                slot["off_dev"].copy_(slot["off_host"], non_blocking=True)
            compute.wait_stream(cs)
            with torch.no_grad():
                if self.resampling:
                    engine.resample(slot["raw"], self.channels, slot["rs_dev"], len(recordings), max(lengths), plan,
                                    slot["dev"])
                out = packed.forward_windows(slot["dev"], window_samples, 0, len(offs), micro_batch=micro_batch,
                                             variant=variant, offsets=slot["off_dev"])
                results = []
                for members, merged in _merge_groups(out["framewise_output"], counts, int(100 * self.ov), self.dur):
                    host_out = slot["out"].get(tuple(merged.shape))
                    if host_out is None:
                        host_out = slot["out"][tuple(merged.shape)] = torch.empty(merged.shape, dtype=torch.float32).pin_memory()
                    host_out.copy_(merged, non_blocking=True)
                    results.append((members, host_out))
            slot["done"] = torch.cuda.Event()
            slot["done"].record(compute)
        self.calls += 1
        self.pending.append((slot, results, len(recordings)))
        return self.calls - 1

    def _stage_raw(self, slot, recordings, n_in, n_out, seg_len, device, compute):
        """Copy stream, resampling call: the raw recordings go as they are into one device staging buffer (DMA from
        the caller's pinned buffers), each recording's padding past its n_out resampled samples is zeroed, and the
        sed_resample table (raw frame offset, n_in, padded-layout offset, n_out) goes up."""
        C, dtype = self.channels, recordings[0].dtype
        total_in = int(n_in.sum()) * C
        if slot.get("raw") is None or slot["raw"].numel() < total_in or slot["raw"].dtype != dtype:
            slot["raw"] = torch.empty(max(total_in, 1), dtype=dtype, device=device)
            slot["raw"].record_stream(compute)
        seg = np.array(seg_len, np.int64)
        n_out = np.array(n_out, np.int64)
        table = np.stack([np.cumsum(n_in) - n_in, n_in, np.cumsum(seg) - seg, n_out], 1)
        slot["rs_host"] = torch.from_numpy(table).pin_memory()
        slot["rs_dev"] = slot["rs_host"].to(device, non_blocking=True)
        slot["rs_dev"].record_stream(compute)
        base = 0
        for r, n in zip(recordings, n_in.tolist()):
            slot["raw"][base:base + n * C].copy_(r.reshape(-1), non_blocking=True)
            base += n * C
        for b, n, sl in zip(table[:, 2].tolist(), n_out.tolist(), seg_len):
            if n < sl:
                slot["dev"][b + n:b + sl].zero_()

    def result(self):
        """Merged frames of the oldest queued call: list of [1, total_frames, classes] CPU tensors, one per recording
        (views of the slot's pinned buffers: valid until two further calls have been submitted)."""
        slot, results, n = self.pending.pop(0)
        slot["done"].synchronize()
        merged = [None] * n
        for members, host_out in results:
            for j, f in enumerate(members):
                merged[f] = host_out[j:j + 1]
        return merged


# predict.py:252-257: the event parameters when no thresholds file is loaded
DEFAULT_SED_PARAMS = {"sed_high_threshold": 0.5, "sed_low_threshold": 0.3, "n_smooth": 10, "n_salt": 10}

LIVE_TICK_SECONDS = 2  # audio one internal tick takes per stream; larger pushes are split into several ticks


def live_final_frames(windows_run, frames_per_window, overlap_interval, sample_duration):
    """Frames of a stream's merged output that are final once `windows_run` windows (numpy int array) have been merged:
    no later window covers them (f < windows_run * oi), and their avg_merge block has the same divisor for every total
    length the stream can still reach (>= (windows_run - 1) * oi + fpw).  0 before the first window."""
    oi, fpw = int(overlap_interval), int(frames_per_window)
    k = np.asarray(windows_run, dtype=np.int64) - 1
    tmin = k * oi + fpw
    interval = int(sample_duration) * 100 - oi
    b = np.minimum(tmin - oi, np.maximum(interval, tmin - interval))
    lb = np.maximum(oi, -(-b // oi) * oi)
    return np.where(k >= 0, np.minimum((k + 1) * oi, lb), 0)


def _plan_live_push(sids, n_samples, windows_run, frames_out, lens, src, closing, sr, sample_duration, W, ring, oi, fpw,
                    classes, slack):
    """The tables of one LiveStreamer push, built from the host counters alone (numpy only, no device round trip).

    sids, n_samples, windows_run, frames_out: the streams of the push and their counters before it; lens, src: each
    stream's chunk length and its first sample in the staged audio; closing: the push closes its (one) stream.
    Geometry: W samples per window, `ring` samples of mirrored audio ring per stream, oi / fpw frames of window stride /
    window, `slack` samples per stream and tick (larger chunks are split into several ticks).  Returns
      * ticks: per tick (ingest table, merge/event table, positions of its streams in `sids`, windows run, merge span
        in frames);
      * offsets: every window's start in the audio arena, ticks in order;
      * rows_per_stream, base: rows of the push's output frames per stream and the first of them;
      * n_rows, n_entries, ev_total: output rows, table entries and event slots of the push;
      * (n_samples, windows_run, frames_out) after the push.
    Every window a tick runs is resident in its stream's ring, no tick spans more frames than the merge accumulator
    holds, and each entry's event capacity bounds what live_events_kernel writes for it."""
    S = len(sids)
    n_ticks = max(1, int(-(-lens.max() // slack)) if S else 1)
    n0, k_run, f_ret = n_samples, windows_run, frames_out
    offsets, ticks, ev_total, rows_per_stream = [], [], 0, np.zeros(S, np.int64)
    for t in range(n_ticks):
        piece = np.clip(lens - t * slack, 0, slack)
        ing = np.stack([sids, src + t * slack, piece, n0], 1)[piece > 0]
        n1 = n0 + piece
        ready = np.where(n1 >= W, n1 // sr - sample_duration + 1, 0)
        last = closing and t == n_ticks - 1
        if last:
            zero = ready == 0  # window 0 runs at close, reading zeros past the end of the stream
            ready = np.maximum(ready, 1)
            fill = np.stack([sids, np.full(S, -1), W - n1, n1], 1)[zero & (n1 < W)]
            ing = np.concatenate([ing, fill])
        m = ready - k_run
        total = (ready - 1) * oi + fpw
        n_final = total if last else live_final_frames(ready, fpw, oi, sample_duration)
        sel = np.flatnonzero((m > 0) | last)
        e = len(sel)
        tab = np.zeros((e, capi.LIVE_TABLE_COLS), np.int64)
        tab[:, 0], tab[:, 1], tab[:, 2] = sids[sel], k_run[sel], m[sel]
        tab[:, 3] = np.concatenate([[0], np.cumsum(m[sel])[:-1]]) if e else []
        tab[:, 4], tab[:, 5] = f_ret[sel], n_final[sel]
        tab[:, 6] = rows_per_stream[sel]  # relative to the stream's block: rebased below
        new = n_final[sel] - f_ret[sel]
        cap = (new + 1) // 2 + 4  # see the output bound of live_events_kernel's state machine
        tab[:, 7] = ev_total + np.concatenate([[0], np.cumsum(cap * classes)[:-1]]) if e else []
        tab[:, 8], tab[:, 9] = cap, int(last)
        ev_total += int((cap * classes).sum())
        win = np.repeat(np.arange(e), m[sel])
        k = np.arange(win.size) - np.repeat(tab[:, 3], m[sel]) + np.repeat(k_run[sel], m[sel])
        offsets.append(sids[sel][win] * 2 * ring + (k * sr) % ring)
        hi = np.where(m[sel] > 0, total[sel], n_final[sel])
        ticks.append((ing, tab, sel, int(win.size), int((hi - f_ret[sel]).max()) if e else 0))
        rows_per_stream[sel] += new
        n0, k_run, f_ret = n1, np.maximum(k_run, ready), np.where((m > 0) | last, n_final, f_ret)
    base = np.concatenate([[0], np.cumsum(rows_per_stream)[:-1]]) if S else np.zeros(0, np.int64)
    for ing, tab, sel, _, _ in ticks:
        tab[:, 6] += base[sel]
    n_rows = int(rows_per_stream.sum())
    n_entries = sum(len(tk[1]) for tk in ticks)
    return ticks, np.concatenate(offsets), rows_per_stream, base, n_rows, n_entries, ev_total, (n0, k_run, f_ret)


def _plan_live_resample(rs, sids, n_in, n_samples, windows_run, frames_out, lens, src, closing, *geometry):
    """_plan_live_push for streams that arrive at another rate: `lens` / `src` are input frames and `n_in` the input
    frames before the push; `rs` is the engine.ResamplePlan.  The planner itself runs unchanged on model-rate counts --
    before close, the outputs whose whole filter support has arrived (rs.n_out_live); at close, the whole resampled
    length -- and each of its ingest rows becomes a sed_live_resample row (slot, j0, outputs, chunk frame or -1, n_prev,
    n_end).  Returns (the planner's result with the rows replaced, history table, input frames after the push)."""
    n_end = n_in + lens
    n_out = rs.n_out(n_end) if closing else rs.n_out_live(n_end)
    out_lens = n_out - n_samples
    out_src = np.cumsum(out_lens) - out_lens
    plan = _plan_live_push(sids, n_samples, windows_run, frames_out, out_lens, out_src, closing, *geometry)
    at = {int(s): j for j, s in enumerate(sids)}
    ticks = []
    for ing, tab, sel, n_win, span in plan[0]:
        j = np.array([at[int(s)] for s in ing[:, 0]], np.int64)
        rows = np.stack([ing[:, 0], ing[:, 3], ing[:, 2], np.where(ing[:, 1] >= 0, src[j], -1), n_in[j], n_end[j]], 1)
        ticks.append((rows.reshape(-1, 6), tab, sel, n_win, span))
    fed = lens > 0
    hist = np.stack([sids, src, n_in, lens], 1)[fed]
    return (ticks,) + plan[1:], hist, n_end


class LiveStreamer:
    """Live detection on many streams at once: audio is pushed as it arrives, every window that becomes ready in any
    stream runs in ONE batch, and each push returns the frames and events that have become final.

    Equivalent, stream by stream, to the offline path on the concatenation `rec` of everything pushed up to `close`:
      * frames: the concatenation of all returned `frames` equals predict_framewise(model, rec, ...)[0] bit for bit;
      * events: label by label, the concatenation of all returned `events` equals frame_prediction_to_event_prediction
        on that merged tensor, in the same order.
    With `input_rate` other than `sample_rate`, or `channels` > 1, chunks are [n] or [n, channels] at input_rate
    (`dtype` is their dtype) and `rec` is resample(everything pushed, input_rate, sample_rate, channels): each push
    resamples on the device the model-rate samples whose whole filter support has arrived, reading earlier input from
    a per-slot history ring (sed_live_resample), into a float32 arena.
    Timeliness:
      * window k runs in the push after which the stream holds (k + sample_duration) * sample_rate samples; window 0
        also runs, zero padded, at close if it never ran (window_starts' rule).  When resampling, a model-rate sample
        is held once the filter's look-ahead has arrived too: half / up input samples more (half = 64 * max(up, down)),
        4 ms of input when downsampling 44.1 or 48 kHz, 8 ms for 8 kHz -> 16 kHz; the last samples come at close;
      * a frame is returned once no later window covers it and its avg_merge block can no longer become a tail block;
        for the shipped presets (frames_per_window 500 / 496, overlap interval <= 100) that is (k + 1) * oi frames after
        the push that ran window k.  The tail blocks, whose divisor depends on the final length, come at close;
      * with a low threshold that is not above the high threshold, an event with offset frame F is returned no later
        than the push that finalizes frame F + n_smooth + 1 when frames F .. F + n_smooth + 1 are all below the low
        threshold;
      * without a low threshold the reference's last pair has no +1 on its offset (find_bgn_fin_pairs), so an event
        stays open until the next run above the high threshold starts, or until close.

    Per slot, the device holds a mirrored audio ring (windows are read in place by the front-end through its offset
    table), a merge accumulator ring and the event state machine; the host holds the counters (samples, windows run,
    frames returned) from which it builds each push's tables without a device round trip.  One device per streamer:
    on several GPUs run one streamer per GPU."""

    def __init__(self, model, sample_rate, sample_duration=5, overlap_value=1, max_streams=4096, dtype=torch.int16,
                 sed_params=None, device=None, labels=None, input_rate=None, channels=1):
        if dtype not in (torch.int16, torch.float32):
            raise ValueError("dtype must be torch.int16 or torch.float32")
        self.channels = _check_channels(channels)
        self.input_rate = int(sample_rate) if input_rate is None else int(input_rate)
        self.resampling = self.input_rate != int(sample_rate) or self.channels != 1
        if self.resampling and self.input_rate != int(sample_rate):
            engine.resample_filter(self.input_rate, sample_rate)  # ValueError for a rate pair the filter refuses
        if device is None and not isinstance(model, engine.PackedModel):
            device = next(model.parameters()).device
        self.packed, self.micro_batch, self.variant = _resolve(model, device)
        self.device = self.packed.device
        self.sr, self.dur, self.dtype = int(sample_rate), int(sample_duration), dtype
        self.oi = int(100 * overlap_value)
        self.W = self.sr * self.dur
        self.fpw = self.packed.frames_for((self.W // self.packed.front.hop + 1) // 8)
        self.classes = int(self.packed.classes)
        self.labels = LABELS if labels is None else labels
        self.max_streams = int(max_streams)
        self.slack = LIVE_TICK_SECONDS * self.sr
        self.ring = self.W + self.slack  # a multiple of sr: every window start is sr-aligned in the ring
        self.ring_frames = (LIVE_TICK_SECONDS - 1) * self.oi + max(self.fpw, 100 * self.dur) + self.oi
        p = DEFAULT_SED_PARAMS if sed_params is None else sed_params
        with torch.cuda.device(self.device):
            self.arena = torch.zeros(self.max_streams * 2 * self.ring, dtype=torch.float32 if self.resampling else dtype,
                                     device=self.device)
            if self.resampling:
                self.rs = engine.resample_plan(self.input_rate, self.sr, self.device)
                self.H = self.rs.history_len()
                self.hist = torch.zeros(self.max_streams * self.H, dtype=torch.float32, device=self.device)
            self.acc = torch.empty((self.max_streams, self.ring_frames, self.classes), dtype=torch.float32,
                                   device=self.device)
            self.ev_state = torch.zeros(self.max_streams * self.classes * capi.LIVE_EVENT_STATE_INTS,
                                        dtype=torch.int32, device=self.device)
            self.ev_params = engine.event_params(p["sed_high_threshold"], p.get("sed_low_threshold"), p["n_smooth"],
                                                 p["n_salt"], self.classes, self.device)
        self.n_samples = np.zeros(self.max_streams, np.int64)  # at sample_rate
        self.n_in = np.zeros(self.max_streams, np.int64)       # at input_rate (frames)
        self.windows_run = np.zeros(self.max_streams, np.int64)
        self.frames_out = np.zeros(self.max_streams, np.int64)
        self.is_open = np.zeros(self.max_streams, bool)
        self.names = [None] * self.max_streams
        self._host = None  # pinned staging (grown on demand, reused)
        self._dev = None

    # ---- slots ----
    def open(self, name=None):
        """Start a stream; returns its slot id (the lowest free one: slots are reused after close)."""
        free = np.flatnonzero(~self.is_open)
        if free.size == 0:
            raise RuntimeError("all %d streams are open" % self.max_streams)
        sid = int(free[0])
        self.is_open[sid] = True
        self.n_samples[sid] = self.n_in[sid] = self.windows_run[sid] = self.frames_out[sid] = 0
        self.names[sid] = name if name is not None else "stream-%d" % sid
        return sid

    def _check_sid(self, sid):
        if not isinstance(sid, (int, np.integer)) or not 0 <= sid < self.max_streams or not self.is_open[sid]:
            raise ValueError("stream %r is not open" % (sid,))
        return int(sid)

    def push(self, items):
        """items: iterable of (sid, chunk), chunk a 1-D CPU (pinned preferred) or CUDA tensor of the streamer's dtype,
        any length (several chunks of one stream are taken in order); [n] or [n, channels] when resampling.  Returns
        {sid: {"first_frame", "frames", "events"}} for every stream of the push: the newly final rows of its merged output (CPU float32
        [n, classes], starting at frame `first_frame`) and its newly decided events."""
        chunks = {}
        for sid, chunk in items:
            sid = self._check_sid(sid)
            if not torch.is_tensor(chunk) or chunk.dtype != self.dtype:
                raise TypeError("chunk for stream %d must be a %s tensor" % (sid, self.dtype))
            if self.resampling:
                _frames(chunk, self.channels, "chunk for stream %d" % sid)
                chunk = chunk.reshape(-1)  # interleaved frames
            elif chunk.dim() != 1:
                raise ValueError("chunk for stream %d must be 1-D, got shape %s" % (sid, tuple(chunk.shape)))
            chunks.setdefault(sid, []).append(chunk)
        sids = np.fromiter(chunks.keys(), np.int64, len(chunks))
        parts = [c[0] if len(c) == 1 else torch.cat([t.to(self.device) for t in c] if any(t.is_cuda for t in c) else c)
                 for c in chunks.values()]
        return self._run(sids, parts, closing=False)

    def close(self, sid):
        """End a stream: runs window 0 (zero padded) if it never ran, returns the remaining frames (the tail blocks)
        and events, in push()'s format for this one stream, and frees the slot."""
        sid = self._check_sid(sid)
        res = self._run(np.array([sid], np.int64), [torch.empty(0, dtype=self.dtype)], closing=True)[sid]
        self.is_open[sid] = False
        return res

    # ---- one push ----
    def _run(self, sids, parts, closing):
        S, W, C, oi, fpw, ncls = len(sids), self.W, self.ring, self.oi, self.fpw, self.classes
        lens = np.fromiter((t.numel() for t in parts), np.int64, S)  # samples (frames x channels when resampling)
        on_dev = np.fromiter((t.is_cuda for t in parts), bool, S)
        # audio layout in the staging buffer: host chunks first (one H2D copy), then device chunks
        order = np.concatenate([np.flatnonzero(~on_dev), np.flatnonzero(on_dev)])
        src = np.zeros(S, np.int64)
        src[order] = np.concatenate([[0], np.cumsum(lens[order])[:-1]]) if S else []
        n_host = int(lens[~on_dev].sum())
        n_audio = int(lens.sum())
        before = (self.n_samples[sids], self.windows_run[sids], self.frames_out[sids])
        geometry = (closing, self.sr, self.dur, W, C, oi, fpw, ncls, self.slack)
        if self.resampling:
            ch = self.channels
            plan, hist_tab, n_in_after = _plan_live_resample(self.rs, sids, self.n_in[sids], *before, lens // ch,
                                                             src // ch, *geometry)
        else:
            plan = _plan_live_push(sids, *before, lens, src, *geometry)
        ticks, offsets, rows_per_stream, base, n_rows, n_entries, ev_total, counters = plan

        # one pinned staging buffer, one host->device copy: audio, then the tables of every tick
        esz = 2 if self.dtype == torch.int16 else 4
        a16 = lambda b: (b + 15) // 16 * 16
        blobs = []
        for ing, tab, _, _, _ in ticks:
            blobs += [ing.astype(np.int64), tab.astype(np.int32)]
        blobs += [offsets.astype(np.int64)]
        i_off = len(blobs) - 1
        if self.resampling:
            blobs += [hist_tab.astype(np.int64)]
        pos, at = [], a16(n_audio * esz)
        for b in blobs:
            pos.append(at)
            at = a16(at + b.nbytes)
        host, dev = self._staging(at)
        if n_host:
            hv = host[:n_host * esz].view(self.dtype)
            torch.cat([parts[i] for i in np.flatnonzero(~on_dev)], out=hv)
        for b, p in zip(blobs, pos):
            host[p:p + b.nbytes].copy_(torch.from_numpy(b.view(np.uint8).reshape(-1)))
        out_words = n_rows * ncls + 2 * ev_total + n_entries * ncls
        with torch.cuda.device(self.device), torch.no_grad():
            dev[:at].copy_(host[:at], non_blocking=True)
            if n_audio > n_host:
                torch.cat([parts[i].to(self.device) for i in np.flatnonzero(on_dev)],
                          out=dev[n_host * esz:n_audio * esz].view(self.dtype))
            audio = dev[:max(n_audio, 1) * esz].view(self.dtype)
            view = lambda j, dt: dev[pos[j]:pos[j] + blobs[j].nbytes].view(dt)
            out = torch.empty(max(out_words, 1), dtype=torch.int32, device=self.device)
            frames = out[:n_rows * ncls].view(torch.float32).view(n_rows, ncls)
            events = out[n_rows * ncls:n_rows * ncls + 2 * ev_total]
            counts_all = out[n_rows * ncls + 2 * ev_total:]
            off_all, e0, w0 = view(i_off, torch.int64), 0, 0
            for j, (ing, tab, sel, n_win, span) in enumerate(ticks):
                if self.resampling:
                    n_hist = len(hist_tab) if j == len(ticks) - 1 else 0  # history: after the push's last reads
                    if len(ing) or n_hist:
                        engine.live_resample(audio, self.channels, view(2 * j, torch.int64), len(ing),
                                             int(ing[:, 2].max()) if len(ing) else 0, self.rs, C, self.arena,
                                             self.hist, self.H, view(i_off + 1, torch.int64), n_hist)
                elif len(ing):
                    engine.live_ingest(audio, view(2 * j, torch.int64), len(ing), int(ing[:, 2].max()), C, self.arena)
                if not len(tab):
                    continue
                if n_win:
                    wf = self.packed.forward_windows(self.arena, W, 0, n_win, micro_batch=self.micro_batch,
                                                     variant=self.variant, offsets=off_all[w0:w0 + n_win])
                    wf = wf["framewise_output"].contiguous()
                    w0 += n_win
                else:
                    wf = torch.empty((1, fpw, ncls), dtype=torch.float32, device=self.device)
                t32 = view(2 * j + 1, torch.int32)
                engine.live_merge(wf, t32, len(tab), span, oi, self.dur, self.acc, frames)
                engine.live_events(frames, t32, len(tab), self.ev_params, self.ev_state, events,
                                   counts_all[e0 * ncls:(e0 + len(tab)) * ncls])
                e0 += len(tab)
            res_host = self._result_buffer(out_words)
            res_host[:out_words].copy_(out[:out_words], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        res = res_host[:out_words].clone()

        self.n_samples[sids], self.windows_run[sids], self.frames_out[sids] = counters
        if self.resampling:
            self.n_in[sids] = n_in_after
        fr = res[:n_rows * ncls].view(torch.float32).view(n_rows, ncls)
        ev = res[n_rows * ncls:n_rows * ncls + 2 * ev_total].numpy()
        cnt = res[n_rows * ncls + 2 * ev_total:].numpy().reshape(n_entries, ncls)
        tab_all = np.concatenate([tk[1] for tk in ticks]) if n_entries else np.zeros((0, capi.LIVE_TABLE_COLS), np.int64)
        if (cnt > tab_all[:, 8:9]).any():
            raise RuntimeError("live event buffer overflow (%d > %d)" % (cnt.max(), tab_all[:, 8].max()))
        first = self.frames_out[sids] - rows_per_stream
        out_res = {}
        for j, sid in enumerate(sids.tolist()):
            out_res[sid] = {"first_frame": int(first[j]), "frames": fr[base[j]:base[j] + rows_per_stream[j]],
                            "events": []}
        # events in the reference's order within a push: class, then time (ticks are in time order)
        for e, c in sorted(zip(*np.nonzero(cnt)), key=lambda ec: (int(tab_all[ec[0], 0]), ec[1], ec[0])):
            sid = int(tab_all[e, 0])
            name = self.names[sid]
            p0 = int(tab_all[e, 7]) + int(c) * int(tab_all[e, 8])
            for q in range(int(cnt[e, c])):
                out_res[sid]["events"].append({"filename": name, "onset": ev[2 * (p0 + q)] / 100.0,
                                               "offset": ev[2 * (p0 + q) + 1] / 100.0,
                                               "event_label": self.labels[c]})
        return out_res

    def _staging(self, nbytes):
        if self._host is None or self._host.numel() < nbytes:
            size = max(nbytes, 1 << 20) * 5 // 4
            self._host = torch.empty(size, dtype=torch.uint8).pin_memory()
            self._dev = torch.empty(size, dtype=torch.uint8, device=self.device)
        return self._host, self._dev

    def _result_buffer(self, words):
        if getattr(self, "_res", None) is None or self._res.numel() < words:
            self._res = torch.empty(max(words, 1 << 18) * 5 // 4, dtype=torch.int32).pin_memory()
        return self._res


def overlap_window_counts(audio_durations, sample_duration, overlap_value):
    """Windows the loop of main_strong.py:786-834 runs per file: start k*overlap_value for k = 0 and every k with
    k*overlap_value + sample_duration <= audio_duration (the `while end <= audio_duration` rule, end updated after
    each window)."""
    return [len(_window_starts(d, sample_duration, overlap_value)) for d in audio_durations]


def predict_framewise_overlap(model, clips, sample_rate, sample_duration, overlap_value, audio_durations=None):
    """The overlap evaluation loop of pytorch/main_strong.py:768-834 for a batch of files at once.

    clips: (n_files, 10 * sample_rate) float32 / int16 CUDA tensor, every file already padded / truncated to 10 s
    (`pad_truncate_sequence`, main_strong.py:785); audio_durations: the files' real durations in seconds (default
    10.0 each) -- they decide how many windows a file gets.  All windows of all files run as ONE batch (the front-end
    reads them in place through an offset table), each file's windows are overlap-added and block-averaged on the
    device.  Returns a list of per-file tensors [1, total_frames, classes] (what `merged` holds after :835)."""
    packed, micro_batch, variant = _resolve(model, clips.device)
    if clips.dim() != 2:
        raise ValueError("clips must be (n_files, samples)")
    n_files, L = clips.shape
    if audio_durations is None:
        audio_durations = [L / float(sample_rate)] * n_files
    counts = overlap_window_counts(audio_durations, sample_duration, overlap_value)
    window_samples = int(sample_duration * sample_rate)
    starts = []
    for f, nw in enumerate(counts):
        for k in range(nw):
            s0 = int(k * overlap_value * sample_rate)  # int(start * sample_rate), main_strong.py:790
            if s0 + window_samples > L:
                raise ValueError("file %d: window %d runs past the padded clip (the reference would feed a short "
                                 "window to the model)" % (f, k))
            starts.append(f * L + s0)
    offsets = torch.tensor(starts, dtype=torch.int64, device=clips.device)
    flat = clips.contiguous().view(-1)
    with torch.no_grad():
        out = packed.forward_windows(flat, window_samples, 0, len(starts), micro_batch=micro_batch, variant=variant,
                                     offsets=offsets)
        merged = [None] * n_files
        for idx, m in _merge_groups(out["framewise_output"], counts, int(100 * overlap_value), sample_duration):
            for j, f in enumerate(idx):
                merged[f] = m[j:j + 1]
    return merged


# Class names of the 25-class strong-label task (utils/config.py:26)
LABELS = ['Applause', 'Breathing', 'Chatter', 'Cheering', 'Child_speech_kid_speaking', 'Clapping', 'Conversation',
          'Cough', 'Crowd', 'Crying_sobbing', 'Female_speech_woman_speaking', 'Laughter',
          'Male_speech_man_speaking', 'Run', 'Screaming', 'Shout', 'Sneeze', 'Walk_footsteps', 'Whispering',
          'Air_horn_truck_horn', 'Car_alarm', 'Emergency_vehicle', 'Explosion', 'Gunshot_gunfire', 'Siren']


def frame_prediction_to_event_prediction(framewise_output, sed_params_dict, frames_per_second=100, audio_names=None,
                                         labels=LABELS):
    """Device version of utils/utilities.py:82-153 (and predict.py:57-121, which uses filename 'test').

    framewise_output: (audios_num, frames_num, classes_num) float32 CUDA tensor; sed_params_dict as loaded from the
    shipped opt_thresholds pickles or the scalar defaults of predict.py:252-257.  Returns the reference's list of
    {'filename', 'onset', 'offset', 'event_label'} dicts in the reference's order (clip-major, class, event)."""
    events, counts = engine.extract_events(framewise_output, sed_params_dict['sed_high_threshold'],
                                           sed_params_dict.get('sed_low_threshold'), sed_params_dict['n_smooth'],
                                           sed_params_dict['n_salt'])
    events = events.cpu().numpy()
    counts = counts.cpu().numpy()
    event_list = []
    for n in range(events.shape[0]):
        name = 'test' if audio_names is None else audio_names[n]
        for k in range(events.shape[1]):
            for e in range(int(counts[n, k])):
                event_list.append({'filename': name, 'onset': events[n, k, e, 0] / float(frames_per_second),
                                   'offset': events[n, k, e, 1] / float(frames_per_second), 'event_label': labels[k]})
    return event_list
