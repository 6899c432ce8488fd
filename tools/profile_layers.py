"""Per-kernel timing of the hot path on one GPU (CUDA events, median of N) -- developer tool."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from sed_b200 import capi, engine, synth  # noqa: E402


def timeit(fn, n=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mb", type=int, default=148)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--variant", type=int, default=2)
    ap.add_argument("--model", default="Cnn_9layers_Gru_FrameAtt")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    lib = capi.load()
    sd = synth.synthetic_state_dict(args.model, 16000)
    pm = engine.PackedModel(sd, args.model, 512, 160, dev)
    mb = args.mb
    wave = synth.synthetic_waveform(mb, 160000).to(dev)
    T = 1001
    feat = torch.empty((mb, 125, 512), dtype=pm.tdtype, device=dev)
    pm.conv_stack(wave, feat, variant=args.variant)
    ws = pm._workspace(mb, T, need_a1=True)  # after the call: it may re-allocate to add conv1's intermediate
    stream = capi.current_stream(dev)
    rows = []
    t = timeit(lambda: engine.logmel_forward(pm.front, wave, pm.bn0_scale, pm.bn0_shift, out=ws["logmel"]))
    rows.append(("frontend (fft+mel+log+bn0)", t, 0.0, mb * (160000 * 4 + 1001 * 64 * 4)))
    t = timeit(lambda: lib.sed_conv_first_f32(capi.ptr(ws["logmel"]), mb, T, 64, capi.ptr(pm.c11_w), capi.ptr(pm.c11_scale),
                                              capi.ptr(pm.c11_shift), capi.ptr(ws["a1"]), pm.dtype_code, stream))
    rows.append(("conv_block1.conv1 (cuda cores)", t, 2 * 36.9e6 * mb, mb * (1001 * 64 * 4 + 1001 * 64 * 64 * 2)))
    chain = [("a1", "p1"), ("p1", "a2"), ("a2", "p2"), ("p2", "a3"), ("a3", "p3"), ("p3", "a4"), ("a4", None)]
    for (name, _, _, _), (cin, cout, mode, wp, s, b), (src, dst) in zip(engine.CONV_LAYERS, pm.convs, chain):
        x = ws[src]
        out = feat if dst is None else ws[dst]
        t = timeit(lambda: lib.sed_conv3x3_bn_relu(capi.ptr(x), mb, x.shape[1], x.shape[2], cin, capi.ptr(wp),
                                                   capi.ptr(s), capi.ptr(b), cout, mode, capi.ptr(out), None, 0, 0,
                                                   pm.dtype_code, stream))
        flops = 2.0 * mb * x.shape[1] * x.shape[2] * 9 * cin * cout
        rows.append(("%s %d->%d pair" % (name, cin, cout), t, flops, x.numel() * 2 + out.numel() * 2))
    B = args.batch
    featB = torch.randn(B, 125, 512, device=dev).to(pm.tdtype)
    if args.model.endswith("Gru_FrameAtt"):
        t = timeit(lambda: pm.linear(featB.view(-1, 512), pm.gru_wih, pm.gru_bih))
        rows.append(("gru input projection (B=%d)" % B, t * mb / B, 2.0 * mb * 125 * 1536 * 512, 0))
        gi = pm.linear(featB.transpose(0, 1).contiguous().view(-1, 512), pm.gru_wih, pm.gru_bih, out_layout=1)
        out = torch.empty((125, (B + 127) // 128, 128, 128, 4), dtype=torch.float32, device=dev)
        gws = torch.empty((lib.sed_bigru_workspace_bytes(B),), dtype=torch.uint8, device=dev)
        t = timeit(lambda: lib.sed_bigru(capi.ptr(gi), capi.ptr(pm.gru_whh), capi.ptr(pm.gru_bhh), B, 125, capi.ptr(out),
                                         capi.ptr(gws), pm.dtype_code, stream))
        rows.append(("gru recurrence (B=%d)" % B, t * mb / B, 2.0 * mb * 125 * 2 * 768 * 256, 0))
        x = out
    else:
        t = timeit(lambda: pm.temporal(featB))
        rows.append(("multihead (B=%d)" % B, t * mb / B, 2.0 * mb * 147e6, 0))
        x = pm.temporal(featB)
    t = timeit(lambda: pm.head(x, 1000, n=B))
    rows.append(("attpool head (B=%d)" % B, t * mb / B, 2.0 * mb * 3.2e6, 0))
    tot = 0.0
    print("per micro-batch of %d clips (temporal/head rows scaled from B=%d)" % (mb, B))
    for name, t, fl, by in rows:
        tot += t
        print("%-44s %8.3f ms  %8.1f TFLOP/s  %7.1f GB/s" % (name, t, fl / t / 1e9, by / t / 1e6))
    print("sum %.3f ms per %d clips -> %.0f clips/s" % (tot, mb, mb / tot * 1e3))
    t = timeit(lambda: pm.forward(synth_wave_cache(B, dev), micro_batch=mb, variant=args.variant), n=5, warm=2)
    print("whole forward B=%d: %.3f ms -> %.0f clips/s" % (B, t, B / t * 1e3))


_cache = {}


def synth_wave_cache(B, dev):
    if B not in _cache:
        _cache[B] = synth.synthetic_waveform(B, 160000).to(dev)
    return _cache[B]


if __name__ == "__main__":
    main()
