"""Cost of resampling on the device (csrc/sed_resample.cu).

    python tools/resample_time.py [--streams 148,1024,4096] [--ticks 8] [--out result.json]

1. sed_resample alone, CUDA events over many launches (inputs + outputs larger than the 126 MB L2):
   4096 x 1 s of 48 kHz stereo int16 -> 16 kHz, and 16 x 60 s of 44.1 kHz mono float32 -> 32 kHz.  Reports kernel
   time, output samples/s and FMAs (the taps of each output's phase, summed) over the card's FP32 FMA rate at its
   maximum SM clock (SMs x 128 lanes x clocks.max.sm).
2. LiveStreamer median tick (host clock around push(), which ends in a synchronize) with S streams each pushing one
   second per tick: 48 kHz stereo int16 with resampling against native 16 kHz int16, alternated tick by tick.
3. HostStreamer windows/s for 44.1 kHz stereo int16 recordings against the same recordings at 16 kHz mono.
Prints one JSON line with the card's name and power limit; --out also writes it to a file."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from sed_b200 import engine, streaming  # noqa: E402
from live_streams import DUR, build, gpu_info  # noqa: E402


def fma_count(plan, n_out):
    """Taps used by outputs 0 .. n_out-1: output j meets the (2*half - r) // up + 1 taps of its phase r."""
    j = np.arange(n_out, dtype=np.int64)
    r = (j * plan.down + plan.half) % plan.up
    return int(((2 * plan.half - r) // plan.up + 1).sum())


def time_kernel(in_rate, out_rate, n_rec, seconds, channels, dtype, reps=20):
    dev = torch.device("cuda:0")
    plan = engine.resample_plan(in_rate, out_rate, dev)
    n_in = in_rate * seconds
    if dtype == torch.int16:
        src = torch.randint(-20000, 20000, (n_rec * n_in * channels,), dtype=torch.int16, device=dev)
    else:
        src = torch.rand(n_rec * n_in * channels, device=dev) * 2 - 1
    n_out = int(plan.n_out(n_in))
    table = torch.tensor([[k * n_in, n_in, k * n_out, n_out] for k in range(n_rec)], dtype=torch.int64, device=dev)
    dst = torch.empty(n_rec * n_out, device=dev)
    for _ in range(3):
        engine.resample(src, channels, table, n_rec, n_out, plan, dst)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(reps):
        engine.resample(src, channels, table, n_rec, n_out, plan, dst)
    t1.record()
    t1.synchronize()
    ms = t0.elapsed_time(t1) / reps
    fmas = fma_count(plan, n_out) * n_rec
    props = torch.cuda.get_device_properties(0)
    info = gpu_info()
    clock_mhz = float(info.get("clocks.max.sm", "0 MHz").split()[0] or 0)
    peak = props.multi_processor_count * 128 * clock_mhz * 1e6
    return {"case": "%d x %d s, %d Hz x%d %s -> %d Hz" % (n_rec, seconds, in_rate, channels, str(dtype)[6:], out_rate),
            "bytes_in_out_MB": (src.numel() * src.element_size() + dst.numel() * 4) / 1e6,
            "kernel_ms": ms, "output_samples_per_s": n_rec * n_out / (ms * 1e-3), "gfma": fmas / 1e9,
            "fma_per_s": fmas / (ms * 1e-3), "fraction_of_fp32_fma_rate": fmas / (ms * 1e-3) / peak if peak else None}


def live_ticks(model, S, ticks):
    sr, rate, C = 16000, 48000, 2
    g = torch.Generator().manual_seed(S)
    n = DUR + 2 + ticks
    m = min(S, 64)  # streams share m recordings: the cost does not depend on the content
    raw = torch.randint(-8000, 8000, (m, n * rate, C), dtype=torch.int16, generator=g).pin_memory()
    nat = torch.randint(-8000, 8000, (m, n * sr), dtype=torch.int16, generator=g).pin_memory()
    arms = {"native_16k": (streaming.LiveStreamer(model, sample_rate=sr, max_streams=S, dtype=torch.int16), nat, sr),
            "resample_48k_stereo": (streaming.LiveStreamer(model, sample_rate=sr, max_streams=S, dtype=torch.int16,
                                                           input_rate=rate, channels=C), raw, rate)}
    sids = {k: [v[0].open() for _ in range(S)] for k, v in arms.items()}
    for k, (live, buf, r) in arms.items():
        live.push([(s, buf[j % m, :DUR * r]) for j, s in enumerate(sids[k])])
    times = {k: [] for k in arms}
    for t in range(ticks + 1):
        for k, (live, buf, r) in arms.items():
            a = (DUR + t) * r
            items = [(s, buf[j % m, a:a + r]) for j, s in enumerate(sids[k])]
            t0 = time.perf_counter()
            live.push(items)
            if t:
                times[k].append(time.perf_counter() - t0)
    return {k + "_tick_ms_median": float(np.median(v)) * 1e3 for k, v in times.items()}


def host_windows(model, n_rec=256, seconds=30, reps=3):
    sr, rate = 16000, 44100
    g = torch.Generator().manual_seed(1)
    raw = [torch.randint(-8000, 8000, (seconds * rate, 2), dtype=torch.int16, generator=g).pin_memory()
           for _ in range(n_rec)]
    nat = [torch.randint(-8000, 8000, (seconds * sr,), dtype=torch.int16, generator=g).pin_memory()
           for _ in range(n_rec)]
    arms = {"native_16k": (streaming.HostStreamer(model, sr), nat),
            "resample_44k1_stereo": (streaming.HostStreamer(model, sr, input_rate=rate, channels=2), raw)}
    windows = n_rec * len(streaming.window_starts(seconds, DUR))
    out = {}
    for k, (hs, recs) in arms.items():
        hs.submit(recs, "cuda:0")
        hs.result()
    t = {k: [] for k in arms}
    for _ in range(reps):
        for k, (hs, recs) in arms.items():
            t0 = time.perf_counter()
            hs.submit(recs, "cuda:0")
            hs.result()
            t[k].append(time.perf_counter() - t0)
    for k, v in t.items():
        out[k + "_windows_per_s"] = windows / float(np.median(v))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", default="148,1024,4096")
    ap.add_argument("--ticks", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("resample_time.py needs a CUDA device")
    res = {"gpu": gpu_info(), "kernel": [time_kernel(48000, 16000, 4096, 1, 2, torch.int16),
                                         time_kernel(44100, 32000, 16, 60, 1, torch.float32)]}
    model = build(16000)
    res["live"] = [dict(streams=S, **live_ticks(model, S, a.ticks)) for S in [int(v) for v in a.streams.split(",")]]
    res["host"] = host_windows(model)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
