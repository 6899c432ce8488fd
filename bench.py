#!/usr/bin/env python
"""Headline benchmark: clips/sec (10 s, 16 kHz) of logmel + CRNN inference (BASELINE.json `metric`).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # B200 arm (this repo's kernels)
  python bench.py --impl reference [--steps K] [--warmup W]     # reference algorithm on the host CPU

A step = one pass of the whole hot path (waveform -> log-mel -> Cnn9 -> bi-GRU -> frame-attention pooling)
over one batch of synthetic clips: BASELINE.json configs[1], Cnn_9layers_Gru_FrameAtt, 16 kHz, batch 1024 per
GPU.  For N > 1 each rank owns its own 1024-clip shard (weak scaling, no collective on the data path) and the
framewise/clipwise outputs are gathered to rank 0 with NCCL inside the timed step.  One JSON line on stdout.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL_TYPE = "Cnn_9layers_Gru_FrameAtt"
SR, N_FFT, HOP, FMIN, FMAX = 16000, 512, 160, 25, 7000
CLIP_SAMPLES = 160000
CONV_GFLOP_TC = 26.031 - 0.0738  # tensor-core conv layers per clip (SURVEY.md 8d minus conv_block1.conv1)
METRIC = "clips/sec (10 s, 16 kHz) logmel+CRNN inference"
DUMP_BYTES = 64 * 10 ** 6  # what --dump-outputs writes at most, .npy headers included


def config_index():
    """BASELINE.json configs[1] = the GRU model (the headline); configs[2] = the Transformer model, 512 clips per GPU."""
    return 1 if MODEL_TYPE == "Cnn_9layers_Gru_FrameAtt" else 2


def load_conv_traffic():
    """DRAM bytes of the seven conv launches of one 148-clip micro-batch, from the committed ncu --set full capture."""
    path = os.path.join(ROOT, "profiles", "r01_conv_traffic.json")
    if os.path.isfile(path):
        with open(path) as f:
            return json.load(f)
    return None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            pk = json.load(f)
        return {"tflops_sustained": float(pk.get("bf16_tflops_sustained", 1410.6)),
                "tflops_burst": float(pk.get("bf16_tflops", 1678.0)), "hbm_gbs": float(pk.get("hbm_gbs", 6537.6)),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled while the timed regions run.  The sampler is started before the
    warm-up (nvidia-smi needs a few hundred ms to come up); only samples taken between mark_begin() and mark_end()
    -- i.e. under the benchmark's load -- are reported."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []   # (monotonic time, text)
        self.t_begin = None
        self.t_end = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.monotonic(), line.strip()))

    def mark_begin(self):
        self.t_begin = time.monotonic()

    def mark_end(self):
        self.t_end = time.monotonic()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        t0 = self.t_begin if self.t_begin is not None else 0.0
        t1 = (self.t_end if self.t_end is not None else time.monotonic()) + 0.06  # a sample reports the interval before it
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < t0 or ts > t1:
                continue
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "window": "device-resident + end-to-end timed regions"}


def dump_outputs(out, directory, seed=0):
    """Write every tensor of one step's output dict as `directory/<name>.npy` in float32.  When they exceed DUMP_BYTES
    together, each keeps the same seeded sample of clips (rows of the batch dimension, in ascending order) and the
    sampled indices are written as `directory/sampled_clips.npy` (float64).  Returns the names written."""
    import numpy as np
    import torch
    out = {k: v.float() for k, v in out.items() if v is not None}
    n = next(iter(out.values())).shape[0]
    per_clip = sum(v[0].numel() * 4 for v in out.values()) + 8
    keep = min(n, (DUMP_BYTES - 4096) // per_clip)  # 4096: room for the .npy headers
    arrays = {}
    if keep < n:
        idx = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
        sel = torch.from_numpy(idx)
        out = {k: v.index_select(0, sel.to(v.device)) for k, v in out.items()}
        arrays["sampled_clips"] = idx.astype(np.float64)
    arrays.update({k: v.cpu().numpy() for k, v in out.items()})
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a)
    return sorted(arrays)


def reference_modules_available():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_import
    return ref_import.available()


def cpu_reference_throughput(steps, warmup, batch=32, device="cpu", autocast=None, channels_last=False):
    """The reference's own CPU implementation of the path on the host cores, all threads: the UNMODIFIED reference
    modules (`/root/reference/pytorch/models.py` where it lies, else the verbatim snapshot oracle/_ref that
    oracle/snapshot_ref.py wrote -- kind "reference"); without either, the oracle port (kind "port").  With
    device="cuda" (`--ref-device cuda`, extra rows, never the reference arm the driver runs) the same modules run
    eagerly on the GPU -- float32 / TF32, or `--ref-autocast bf16` (+ `--ref-channels-last`): the incumbent a user
    of the reference has today."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import ref_import
    import sed_oracle
    from sed_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = synth.synthetic_state_dict(MODEL_TYPE, SR)
    wave = synth.synthetic_waveform(batch, CLIP_SAMPLES, seed=1234)
    on_gpu = device != "cpu"
    kind = "reference" if ref_import.available() else "port"
    if kind == "reference":
        _, ref_models = ref_import.load()
        model = getattr(ref_models, MODEL_TYPE)(SR, N_FFT, HOP, 64, FMIN, FMAX, 25, "logmel")
        model.load_state_dict(sd, strict=True)
        model = model.eval().to(device)
        if channels_last:
            model = model.to(memory_format=torch.channels_last)
        wave = wave.to(device)

        def run():
            with torch.no_grad():
                if autocast:
                    with torch.autocast("cuda" if on_gpu else "cpu", dtype=getattr(torch, autocast)):
                        return model(wave)
                return model(wave)
    else:
        if on_gpu:
            sd = {k: v.to(device) for k, v in sd.items()}
            wave = wave.to(device)

        def run():
            return sed_oracle.model_forward(sd, wave, MODEL_TYPE, N_FFT, HOP)

    def sync():
        if on_gpu:
            torch.cuda.synchronize()

    for _ in range(warmup):
        run()
    sync()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        out = run()
        if on_gpu:
            out["framewise_output"].float().cpu()
        sync()
        times.append(time.perf_counter() - t0)
    total = sum(times)
    what = "unmodified reference modules" if kind == "reference" else "oracle port of the reference forward"
    if on_gpu:
        where = "%s, torch eager on %s (%s%s, cudnn tf32 %s)" % (
            what, torch.cuda.get_device_name(0), "autocast " + autocast if autocast else "float32",
            ", channels_last" if channels_last else "", torch.backends.cudnn.allow_tf32)
    else:
        where = "%s, float32 torch CPU ops, %d threads" % (what, cores)
    return {"value": batch * steps / total, "unit": "clips/s", "cores": cores, "kind": kind,
            "sample": "%d steps of batch %d x 10 s clips, %s" % (steps, batch, where),
            "ms_per_step": 1e3 * total / steps, "batch": batch}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    warmup = max(0, args.warmup)
    batch = args.ref_batch
    cb = cpu_reference_throughput(steps, warmup, batch, args.ref_device, args.ref_autocast, args.ref_channels_last)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "clips/s", "n_gpus": args.gpus,
        "gpus_used": 0 if args.ref_device == "cpu" else 1, "steps": steps, "warmup": warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32" if not args.ref_autocast else args.ref_autocast, "data": "synthetic",
        "config": {"workload": "%s logmel 16k batch %d per GPU (BASELINE.json configs[%d]), "
                               "10 s clips, seeded synthetic checkpoint" % (MODEL_TYPE, args.batch, config_index()),
                   "batch_per_gpu": args.batch,
                   "sample": "each step is %d clips of that workload on the host CPU (same clips, same checkpoint)"
                             % batch},
        "cpu_baseline": {"value": cb["value"], "unit": "clips/s", "cores": cb["cores"], "kind": cb["kind"],
                         "sample": cb["sample"]},
        "e2e": {"value": cb["value"], "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------------
class Ctx:
    """Rank / device / collectives of one bench process."""

    def __init__(self, torch, dist, dev, world, rank):
        self.torch, self.dist, self.dev, self.world, self.rank = torch, dist, dev, world, rank

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def timed(self, fn, steps, warmup, finish=None):
        """ms per step of fn(i): barrier + synchronize on both sides, CUDA events on the current stream, max over ranks."""
        for i in range(warmup):
            fn(i)
        self.barrier()
        e0 = self.torch.cuda.Event(enable_timing=True)
        e1 = self.torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        if finish is not None:
            finish()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps


class Gatherer:
    """Assembly of every rank's framewise / clipwise on rank 0 inside the step (dist.PeerGather: rank 0 owns one
    buffer for all ranks, mapped everywhere through CUDA IPC; completion = one stream-ordered 4-byte all-reduce).
      push (default)  results are written locally and leave by DMA (sed_peer_copy) on a side stream, so the NVLink
                      transfer of step k overlaps the kernels of step k+1 without occupying an SM; step k is complete
                      on rank 0 after the kernels of step k+1 (one step of latency, no loss of throughput)
      peer            the pooling-head kernels store straight into rank 0's memory over NVLink (fused, no copy)
      nccl            one NCCL gather received in place (also the fallback where peer memory is unavailable)"""

    def __init__(self, ctx, sdist, n, frames, classes, mode):
        self.ctx, self.sdist, self.peer, self.how, self.mode = ctx, sdist, None, "none (1 GPU)", mode
        self.into = None
        t = ctx.torch
        if ctx.world == 1:
            self.mode = "none"
            return
        if mode in ("peer", "push"):
            try:
                self.peer = sdist.PeerGather(n, frames, classes, ctx.dev, dst=0, slots=4)
                done = ("flag words behind the data (stream memory operations; no collective, no per-step lockstep)"
                        if self.peer.use_flags else "4-byte all-reduce")
                self.how = ("results pushed by DMA into rank 0's buffer over NVLink on a side stream (CUDA IPC peer "
                            "memory), overlapping the next step" if mode == "push" else
                            "head kernels store over NVLink into rank 0's buffer (CUDA IPC peer memory)") + "; completion: " + done
            except RuntimeError as e:
                self.mode = "nccl"
                self.how = "nccl gather (peer memory unavailable: %s)" % str(e)[:120]
        elif mode == "none":
            self.how = "NOT assembled (diagnostic: every rank keeps its own outputs)"
        else:
            self.how = "nccl gather received in place"
        if self.mode == "nccl" and ctx.rank == 0:
            self.into = {"framewise_output": t.empty((ctx.world * n, frames, classes), device=ctx.dev),
                         "clipwise_output": t.empty((ctx.world * n, classes), device=ctx.dev)}
        if self.mode == "push":
            self.side = t.cuda.Stream(ctx.dev)
            self.nloc = 4
            self.local = [(t.empty((n, classes), device=ctx.dev), t.empty((n, frames, classes), device=ctx.dev))
                          for _ in range(self.nloc)]
            self.copied = [None] * self.nloc
            self.pending = None   # step whose results are on their way to rank 0

    def step(self, pm, wave, i, **kw):
        t = self.ctx.torch
        if self.mode == "peer":
            self.peer.wait_turn(i)
            pm.forward(wave, out=self.peer.local_out(i), **kw)
            self.peer.signal(i)
            return self.peer.complete(i)
        if self.mode == "push":
            # step i: kernels on the main stream, then its results leave by DMA on the side stream (behind them the
            # completion flag); rank 0 completes step i-1 (whose DMA ran under this step's kernels) on its main stream.
            # No collective kernel ever runs beside the persistent conv kernels and no rank waits for another one
            # except rank 0 for what it consumes.
            main = t.cuda.current_stream(self.ctx.dev)
            loc = self.local[i % self.nloc]
            if self.copied[i % self.nloc] is not None:
                main.wait_event(self.copied[i % self.nloc])  # the DMA of step i - nloc has read this buffer
            pm.forward(wave, out=loc, **kw)
            ready = t.cuda.Event()
            ready.record(main)
            self.side.wait_event(ready)
            with t.cuda.stream(self.side):
                self.peer.push(loc[0], loc[1], i)
                self.copied[i % self.nloc] = t.cuda.Event()
                self.copied[i % self.nloc].record(self.side)
            res = self._complete(self.pending) if self.pending is not None else None
            self.pending = i
            return res
        out = pm.forward(wave, **kw)
        if self.mode == "nccl":
            return self.sdist.gather_outputs(out, dst=0, into=self.into)
        return out

    def _complete(self, i):
        if not self.peer.use_flags:  # the all-reduce fallback needs this rank's transfer ordered before it
            self.ctx.torch.cuda.current_stream(self.ctx.dev).wait_event(self.copied[i % self.nloc])
        return self.peer.complete(i)

    def finish(self):
        """Complete the last step's transfer on the caller's stream (call before the closing timing event)."""
        if self.mode == "push" and self.pending is not None:
            res = self._complete(self.pending)
            self.pending = None
            return res

    def close(self):
        if self.peer is not None:
            self.ctx.torch.cuda.synchronize(self.ctx.dev)
            self.peer.close()


def dp_preflight(torch, models, synth):
    """Untimed: the drop-in model under torch.nn.DataParallel on two GPUs (the reference's own multi-GPU mechanism,
    main_strong.py:541) returns bit for bit what one GPU returns."""
    if torch.cuda.device_count() < 2:
        return "skipped (1 GPU visible)"
    try:
        sd = synth.synthetic_state_dict(MODEL_TYPE, SR)
        model = getattr(models, MODEL_TYPE)(SR, N_FFT, HOP, 64, FMIN, FMAX, 25, "logmel")
        model.load_state_dict(sd)
        model = model.to("cuda:0").eval()
        x = synth.synthetic_waveform(6, 32000, seed=5, kind="events").to("cuda:0")
        one = model(x)
        two = torch.nn.DataParallel(model, device_ids=[0, 1])(x)
        torch.cuda.synchronize()
        same = all(torch.equal(one[k], two[k]) for k in ("framewise_output", "clipwise_output"))
        return "ok" if same else "MISMATCH"
    except Exception as e:  # noqa: BLE001 -- a preflight must not take the benchmark down
        return "error: %s" % str(e)[:160]


def e2e_rate(ctx, pipe, wave_h, steps):
    """clips/s per rank through the host pipeline: K submits + K collected results inside the timed region (every
    step's host->device copy from pinned memory and device->host result copy included; two batches in flight)."""
    for _ in range(2):
        pipe.result(pipe.submit(wave_h))
    ctx.barrier()
    t0 = time.perf_counter()
    pipe.submit(wave_h)
    for _ in range(steps - 1):
        pipe.submit(wave_h)
        res = pipe.result()
    res = pipe.result()
    ctx.torch.cuda.synchronize(ctx.dev)
    dt = ctx.max_over_ranks(time.perf_counter() - t0)
    ctx.barrier()
    return wave_h.shape[0] * steps / dt, res


def bench_config3(ctx, engine, synth, sdist, args):
    """BASELINE configs[2]: Cnn_9layers_Transformer_FrameAtt, 16 kHz, 4096 clips over 8 GPUs = 512 per GPU; timed from
    inputs resident on each rank to framewise + clipwise resident on rank 0 (gather included), and without it."""
    mt = "Cnn_9layers_Transformer_FrameAtt"
    B = 512
    pm = engine.PackedModel(synth.synthetic_state_dict(mt, SR), mt, N_FFT, HOP, ctx.dev, precision=args.precision)
    wave = synth.synthetic_waveform(B, CLIP_SAMPLES, seed=4321, rank=ctx.rank).to(ctx.dev)
    g = Gatherer(ctx, sdist, B, 1000, 25, args.gather)
    ms = ctx.timed(lambda i: g.step(pm, wave, i), steps=4, warmup=2, finish=g.finish)
    ms_nog = ctx.timed(lambda i: pm.forward(wave), steps=4, warmup=1)
    g.close()
    return {"workload": "%s logmel 16k, %d clips per GPU x %d GPUs" % (mt, B, ctx.world), "batch_per_gpu": B,
            "clips_per_s": ctx.world * B / ms * 1e3, "ms_per_step": ms, "gather": g.how,
            "clips_per_s_without_gather": ctx.world * B / ms_nog * 1e3, "steps": 4}


def bench_config4(ctx, engine, streaming, synth, args, with_cpu):
    """BASELINE configs[3]: predict.py streaming path at 32 kHz -- 60 s recordings, 5 s windows, 1 s stride (56 windows
    per recording), frame-wise overlap averaging on the device; recordings sharded over the ranks (no collective).
    e2e: pinned host int16 recordings in -> merged frames on the host."""
    torch = ctx.torch
    sr, files = 32000, 16
    n_fft, hop, fmin, fmax = synth.PRESETS[sr]
    pm = engine.PackedModel(synth.synthetic_state_dict(MODEL_TYPE, sr), MODEL_TYPE, n_fft, hop, ctx.dev,
                            precision=args.precision)
    host = []
    for f in range(files):
        w = synth.synthetic_waveform(1, 60 * sr, seed=100 + f, rank=ctx.rank, kind="events", sample_rate=sr)[0]
        host.append(torch.round(w * 32767.0).to(torch.int16).pin_memory())
    recs = [h.to(ctx.dev) for h in host]
    windows = files * len(streaming.window_starts(60.0, 5, overlap=True))
    ms = ctx.timed(lambda i: streaming.predict_framewise_many(pm, recs, sr, 5, 1), steps=4, warmup=2)

    streamer = streaming.HostStreamer(pm, sr, 5, 1)   # one pinned buffer per call, one copy each way, two calls in flight
    for i in range(2):
        streamer.submit(host, ctx.dev)
        streamer.result()
    ctx.barrier()
    t0 = time.perf_counter()
    streamer.submit(host, ctx.dev)
    for i in range(3):
        streamer.submit(host, ctx.dev)
        out = streamer.result()
    out = streamer.result()
    ms_e2e = 1e3 * ctx.max_over_ranks(time.perf_counter() - t0) / 4
    ctx.barrier()
    res = {"workload": "%s logmel 32k streaming: %d recordings of 60 s per GPU per call x %d GPUs, 5 s windows / 1 s "
                       "stride, merge + avg_merge on the device" % (MODEL_TYPE, files, ctx.world),
           "windows_per_call_per_gpu": windows, "windows_per_s": ctx.world * windows / ms * 1e3,
           "audio_seconds_per_s": ctx.world * files * 60 / ms * 1e3, "ms_per_call": ms,
           "e2e_windows_per_s": ctx.world * windows / ms_e2e * 1e3,
           "e2e_audio_seconds_per_s": ctx.world * files * 60 / ms_e2e * 1e3,
           "e2e_bytes_per_call": {"h2d": files * 60 * sr * 2, "d2h": sum(m.numel() * 4 for m in out)}}
    if with_cpu:
        # the reference's sequential B = 1 window loop (predict.py:297-349) on the host cores: bounded sample
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import stream_oracle
        torch.set_num_threads(os.cpu_count() or 1)
        sd = synth.synthetic_state_dict(MODEL_TYPE, sr)
        audio = (host[0][:15 * sr].float() / 32767.0).numpy()
        nw = len(streaming.window_starts(15.0, 5, overlap=True))
        t0 = time.perf_counter()
        stream_oracle.streaming_predict(sd, audio, MODEL_TYPE, sr, n_fft, hop, 5, 1)
        dt = time.perf_counter() - t0
        res["cpu_b1_loop"] = {"windows_per_s": nw / dt, "audio_seconds_per_s": 15.0 / dt, "cores": os.cpu_count(),
                              "kind": "port", "sample": "one 15 s recording = %d windows of 5 s, batch 1 per window "
                              "(oracle/stream_oracle.streaming_predict, the loop of predict.py:297-349)" % nw}
    return res


def bench_config5(ctx, engine, synth, peaks, total_clips=1000000):
    """BASELINE configs[4]: log-mel front-end alone (waveform f32 -> log-mel f32) at 8k / 16k / 32k; a resident
    592-clip chunk (input + output exceed L2) is looped until `total_clips` clips have gone through all GPUs."""
    torch = ctx.torch
    out = {}
    B = 592
    iters = max(3, -(-total_clips // (ctx.world * B)))
    for sr in (8000, 16000, 32000):
        n_fft, hop, fmin, fmax = synth.PRESETS[sr]
        sd = synth.synthetic_state_dict(MODEL_TYPE, sr)
        plan = engine.FrontendPlan(sd["spectrogram_extractor.stft.conv_real.weight"],
                                   sd["spectrogram_extractor.stft.conv_imag.weight"], n_fft, hop,
                                   sd["logmel_extractor.melW"], ctx.dev)
        L = 10 * sr
        w = synth.synthetic_waveform(B, L, seed=77, rank=ctx.rank).to(ctx.dev)
        o = torch.empty((B, L // hop + 1, 64), dtype=torch.float32, device=ctx.dev)
        for _ in range(3):
            engine.logmel_forward(plan, w, out=o)
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            engine.logmel_forward(plan, w, out=o)
        e1.record()
        ctx.barrier()
        ms = ctx.max_over_ranks(e0.elapsed_time(e1))
        per_clip = 4 * L + 4 * (L // hop + 1) * 64
        rate = ctx.world * B * iters / ms * 1e3
        out["%dk" % (sr // 1000)] = {"clips": ctx.world * B * iters, "clips_per_s": rate,
                                     "algorithmic_GBps_per_gpu": rate / ctx.world * per_clip / 1e9,
                                     "hbm_frac": rate / ctx.world * per_clip / 1e9 / peaks["hbm_gbs"],
                                     "bytes_per_clip": per_clip}
    return {"workload": "log-mel front-end alone, 10 s clips, %d-clip resident chunk looped to >= %d clips over %d "
                        "GPUs" % (B, total_clips, ctx.world), "hbm_peak_GBps": peaks["hbm_gbs"], "presets": out}


def run_b200(args):
    import torch
    import torch.distributed as dist
    from sed_b200 import capi, engine, models, streaming, synth
    from sed_b200 import dist as sdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: everything any library prints to fd 1 (NCCL's version banner, ...) is sent
    # to stderr, the result line is written to the saved descriptor
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the B200 arm)")
    full_affinity = os.sched_getaffinity(0)
    numa = "off" if os.environ.get("SED_NO_NUMA_BIND") else sdist.bind_host_to_gpu(local_rank)  # before pinned buffers
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL banners / warnings never reach stdout (one JSON line)
        dist.init_process_group("nccl", device_id=dev)
    ctx = Ctx(torch, dist, dev, world, rank)
    capi.load()

    B = args.batch
    steps, warmup = args.steps, max(3, args.warmup)
    sd = synth.synthetic_state_dict(MODEL_TYPE, SR)
    pm = engine.PackedModel(sd, MODEL_TYPE, N_FFT, HOP, dev, precision=args.precision)
    wave_host = synth.synthetic_waveform(B, CLIP_SAMPLES, seed=1234, rank=rank).pin_memory()
    wave_i16 = torch.round(wave_host * 32767.0).to(torch.int16).pin_memory()
    wave = wave_host.to(dev)
    frames = pm.frames_for((CLIP_SAMPLES // HOP + 1) // 8)

    # untimed preflight: the reference's own multi-GPU mechanism on the drop-in model
    dp_check = dp_preflight(torch, models, synth) if rank == 0 else None
    ctx.barrier()

    gather = Gatherer(ctx, sdist, B, frames, pm.classes, args.gather)

    def step_device(i):
        return gather.step(pm, wave, i, micro_batch=args.micro_batch, variant=args.variant)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for i in range(warmup):
        step_device(i)
    ctx.barrier()

    # ---------------- timed region 1: inputs resident in HBM ----------------
    if rank == 0:
        sampler.mark_begin()
    capi.reset_launches()
    pm.conv_events = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    e0.record()
    for i in range(steps - 1):
        step_device(warmup + i)
    last = step_device(warmup + steps - 1)  # earlier steps drop their outputs at once, the last one's are kept
    done = gather.finish()  # push: the last step completes here
    if done is not None:
        last = done
    e1.record()
    ctx.barrier()
    # written after the clock samples close (below); region 2 leaves the gather buffers these may alias untouched
    dump = last if args.dump_outputs and rank == 0 else None
    del last, done
    elapsed_ms = e0.elapsed_time(e1)
    launches = capi.launches()
    conv_ms = sum(a.elapsed_time(b) for a, b, _ in pm.conv_events)
    conv_clips = sum(n for _, _, n in pm.conv_events)
    pm.conv_events = None
    elapsed_ms = ctx.max_over_ranks(elapsed_ms)

    # ---------------- timed region 2: end to end with HOST buffers, through the host pipeline ----------------
    # Headline: int16 PCM host input -- the reference's own storage format (utils/utilities.py:78-79); at N = 8 the
    # float32 variant is bound by this platform's host<->device copy ceiling (profiles/r02_h2d_ceiling.json).
    pipe = pm.host_pipeline(depth=2, micro_batch=args.micro_batch, variant=args.variant)
    rate_i16, res = e2e_rate(ctx, pipe, wave_i16, steps)
    d2h = res["clipwise_output"].numel() * 4 + res["framewise_output"].numel() * 4
    rate_f32, _ = e2e_rate(ctx, pipe, wave_host, steps)
    # the synchronous single call (copy in, run, copy out; nothing overlapped across calls), for reference
    for _ in range(4):  # its three rotating result slots are allocated before the clock starts
        pm.forward_host(wave_i16, micro_batch=args.micro_batch, variant=args.variant)
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        pm.forward_host(wave_i16, micro_batch=args.micro_batch, variant=args.variant)
    sync_ms = 1e3 * ctx.max_over_ranks(time.perf_counter() - t0)
    ctx.barrier()
    clocks = None
    if rank == 0:
        sampler.mark_end()
        clocks = sampler.stop()
    if dump is not None:
        dump_outputs(dump, args.dump_outputs)
    del dump

    # ---------------- the other BASELINE configs: short runs outside the headline regions ----------------
    peaks = load_peaks()
    configs = None
    if not args.no_configs:
        del wave
        pm._ws.clear()
        torch.cuda.empty_cache()
        configs = {}
        for name, fn in (("config3_transformer_4096_over_8", lambda: bench_config3(ctx, engine, synth, sdist, args)),
                         ("config4_streaming_32k", lambda: bench_config4(ctx, engine, streaming, synth, args,
                                                                         with_cpu=(world == 1 and rank == 0 and
                                                                                   not args.no_cpu_baseline))),
                         ("config5_frontend_sweep", lambda: bench_config5(ctx, engine, synth, peaks))):
            configs[name] = fn()
            torch.cuda.empty_cache()
    gather.close()

    if rank == 0:
        traffic = load_conv_traffic()
        value = world * B * steps / (elapsed_ms / 1e3)
        # variant 4 runs conv_block1.conv1 inside the first timed launch: the timed group is the whole conv stack
        conv_gflop = 26.031 if args.variant == 4 else CONV_GFLOP_TC
        conv_tflops = conv_gflop * 1e9 * conv_clips / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
        n_conv_launch = 7 * len(pm_spans(B, args.micro_batch)) * steps
        line = {
            "metric": METRIC, "value": value, "unit": "clips/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": elapsed_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": "%s logmel 16k batch %d per GPU (BASELINE.json configs[%d]), "
                                   "10 s clips, seeded synthetic checkpoint" % (MODEL_TYPE, B, config_index()),
                       "batch_per_gpu": B, "micro_batch": args.micro_batch, "parallelism": "dp%d (batch shards, no "
                       "collective on the data path; outputs assembled on rank 0: %s)" % (world, gather.how),
                       "l2": "inputs (%.0f MB/step) and activations (>6 GB/micro-batch) exceed the 126 MB L2" %
                             (B * CLIP_SAMPLES * 4 / 1e6)},
            "e2e": {"value": world * rate_i16, "unit": "clips/s",
                    "h2d_bytes_per_step": B * CLIP_SAMPLES * 2, "d2h_bytes_per_step": d2h,
                    "api": "HostPipeline.submit/result (sed_b200.pipeline; what sed_b200.pytorch_utils.forward drives): "
                           "pinned host int16 PCM waveform in (x = q/32767 in the front-end kernel, the reference's "
                           "HDF5 format), host clipwise/framewise out, two batches in flight",
                    "host_affinity": numa,
                    "f32_input_value": world * rate_f32, "f32_h2d_bytes_per_step": B * CLIP_SAMPLES * 4,
                    "synchronous_forward_host_int16_value": world * B * steps / (sync_ms / 1e3),
                    "platform_ceiling": "profiles/r02_h2d_ceiling.json: 8 ranks doing only these copies reach 344 k "
                                        "clips/s (int16) / 215 k (float32) on this pool's 8-GPU host"},
            "gpu_launches": launches,
            "dp_check": dp_check,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": conv_tflops, "peak": peaks["tflops_sustained"],
                         "unit": "TFLOP/s", "frac": conv_tflops / peaks["tflops_sustained"],
                         "traffic": traffic["dram_bytes_total"] * B / traffic["clips"] if traffic else None,
                         "traffic_note": "DRAM bytes of the 7 conv launches of one step (%d clips): dram__bytes_read+write "
                                         "from ncu --set full of a 148-clip launch group (profiles/r01_ncu_full_conv_umma2"
                                         "_raw.csv, r01_ncu_full_conv_block1_tc_raw.csv: %.3e B), scaled by clips; "
                                         "algorithmic activation bytes (each layer input read once + output written "
                                         "once) for the same launches: %.3e" % (B, traffic["dram_bytes_total"] if traffic
                                                                                else 0.0, B * 21888256.0),
                         "kernel": "conv_block1_tc_kernel + 6 x conv_umma2_kernel (7 tcgen05 cta_group::2 implicit-GEMM "
                                   "launches per micro-batch, %.3f GFLOP/clip algorithmic)" % conv_gflop,
                         "peak_source": peaks["source"] + ", sustained bf16; burst %.1f" % peaks["tflops_burst"],
                         "launches_timed": n_conv_launch, "conv_ms_per_step": conv_ms / steps},
        }
        if configs is not None:
            line["configs"] = configs
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, full_affinity)  # the CPU baseline gets every host core again
            cb = cpu_reference_throughput(steps=3, warmup=1, batch=args.ref_batch)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def pm_spans(B, micro_batch):
    return list(range(0, B, micro_batch))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="clips per GPU per step")
    ap.add_argument("--micro-batch", type=int, default=1036, help="cap of a conv-stack launch group (engine default)")
    ap.add_argument("--variant", type=int, default=4)
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--model-type", default=MODEL_TYPE,
                    choices=["Cnn_9layers_Gru_FrameAtt", "Cnn_9layers_Transformer_FrameAtt"],
                    help="default = the headline config; the Transformer model is BASELINE config 3 (use --batch 512)")
    ap.add_argument("--ref-batch", type=int, default=32)
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"],
                    help="cpu = the reference arm (default); cuda = extra row: the same torch ops eagerly on the GPU")
    ap.add_argument("--ref-autocast", default=None, choices=["bf16", "bfloat16", "fp16", "float16"],
                    help="extra row: run the reference modules under torch.autocast (with --ref-device cuda)")
    ap.add_argument("--ref-channels-last", action="store_true", help="extra row: channels_last reference modules")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the short runs of BASELINE configs 3 / 4 / 5")
    ap.add_argument("--gather", default="push", choices=["push", "peer", "nccl", "none"],
                    help="N > 1: how rank 0 gets every rank's outputs (see class Gatherer)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB: a seeded "
                         "sample of clips when larger, see dump_outputs); the inputs are the same in every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 arm (--impl b200)")
    args.ref_autocast = {"bf16": "bfloat16", "fp16": "float16"}.get(args.ref_autocast, args.ref_autocast)
    globals()["MODEL_TYPE"] = args.model_type
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
