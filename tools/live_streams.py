"""Live multi-stream throughput: S streams of int16 PCM pushed one second per stream per tick through
streaming.LiveStreamer (every stream adds exactly one window per tick), against the same windows run through
streaming.HostStreamer as finished recordings in the same process.

    python tools/live_streams.py [--streams 1,8,148,1024,4096] [--rates 16000,32000] [--ticks 20]
                                 [--out result.json] [--profile trace.txt]

Per (sample rate, S): median / p90 of the tick wall time (host clock around push(), which ends in a synchronize),
windows/s, real-time stream capacity S / median tick seconds, and HostStreamer windows/s on S recordings of
sample_duration + ticks - 1 seconds (the same S * ticks windows).  Prints one JSON line; --out writes it to a file.
--profile writes a torch.profiler table of a few live ticks at the largest S."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from sed_b200 import models, streaming, synth  # noqa: E402

MT = "Cnn_9layers_Gru_FrameAtt"
DUR = 5


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return dict(zip(q.split(","), [v.strip() for v in out.split(",")])) if out else {"name": torch.cuda.get_device_name(0)}


def build(sr):
    n_fft, hop, fmin, fmax = synth.PRESETS[sr]
    model = getattr(models, MT)(sr, n_fft, hop, 64, fmin, fmax, 25, "logmel")
    model.load_state_dict(synth.synthetic_state_dict(MT, sr))
    return model.to("cuda:0").eval()


def audio(S, seconds, sr):
    """S int16 recordings as views of one pinned buffer (random PCM: the model's cost does not depend on content)."""
    buf = torch.randint(-8000, 8000, (S, seconds * sr), dtype=torch.int16).pin_memory()
    return buf


def run_live(model, sr, S, ticks, buf, profile=None):
    live = streaming.LiveStreamer(model, sample_rate=sr, sample_duration=DUR, max_streams=S, dtype=torch.int16)
    sids = [live.open() for _ in range(S)]
    live.push([(s, buf[j, :DUR * sr]) for j, s in enumerate(sids)])  # warm-up: window 0 of every stream
    times = []
    warm = 2
    for t in range(warm + ticks):
        a = (DUR + t) * sr
        items = [(s, buf[j, a:a + sr]) for j, s in enumerate(sids)]
        t0 = time.perf_counter()
        res = live.push(items)
        t1 = time.perf_counter()
        if t >= warm:
            times.append(t1 - t0)
        assert res[sids[0]]["frames"].shape[0] == 100
    if profile:
        from torch.profiler import ProfilerActivity, profile as prof
        a = (DUR + warm + ticks) * sr
        with prof(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as p:
            for t in range(3):
                live.push([(s, buf[j, a + t * sr:a + (t + 1) * sr]) for j, s in enumerate(sids)])
        with open(profile, "a") as f:
            f.write("# live push, S=%d, sr=%d, 3 ticks\n" % (S, sr))
            f.write(p.key_averages().table(sort_by="cuda_time_total", row_limit=30) + "\n")
            f.write(p.key_averages().table(sort_by="cpu_time_total", row_limit=30) + "\n")
    times = np.array(times)
    med, p90 = float(np.median(times)), float(np.percentile(times, 90))
    return {"tick_ms_median": med * 1e3, "tick_ms_p90": p90 * 1e3, "windows_per_s": S / med,
            "realtime_streams": S / med}


def run_host(model, sr, S, ticks, buf, reps=3):
    hs = streaming.HostStreamer(model, sr, DUR, 1)
    recs = [buf[j, :(DUR + ticks - 1) * sr] for j in range(S)]
    hs.submit(recs, "cuda:0")
    hs.result()  # warm-up
    best = []
    for _ in range(reps):
        t0 = time.perf_counter()
        hs.submit(recs, "cuda:0")
        out = hs.result()
        best.append(time.perf_counter() - t0)
        assert out[0].shape[1] == (ticks - 1) * 100 + 500
    med = float(np.median(best))
    return {"host_ms": med * 1e3, "host_windows_per_s": S * ticks / med}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", default="1,8,148,1024,4096")
    ap.add_argument("--rates", default="16000,32000")
    ap.add_argument("--ticks", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("live_streams.py needs a CUDA device")
    streams = [int(v) for v in a.streams.split(",")]
    rows = []
    for sr in [int(v) for v in a.rates.split(",")]:
        model = build(sr)
        buf = audio(max(streams), DUR + 2 + a.ticks + 4, sr)
        for S in streams:
            r = {"sample_rate": sr, "streams": S, "ticks": a.ticks}
            r.update(run_live(model, sr, S, a.ticks, buf[:S],
                              profile=a.profile if (a.profile and S == max(streams)) else None))
            r.update(run_host(model, sr, S, a.ticks, buf[:S]))
            r["live_over_host"] = r["windows_per_s"] / r["host_windows_per_s"]
            rows.append(r)
            print("sr %d S %5d: tick median %.2f ms p90 %.2f ms, %.0f windows/s live, %.0f windows/s HostStreamer "
                  "(%.2fx)" % (sr, S, r["tick_ms_median"], r["tick_ms_p90"], r["windows_per_s"],
                               r["host_windows_per_s"], r["live_over_host"]), flush=True)
        del buf, model
        torch.cuda.empty_cache()
    line = json.dumps({"tool": "live_streams", "model": MT, "sample_duration": DUR, "gpu": gpu_info(), "rows": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
