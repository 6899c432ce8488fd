"""Per-kernel GPU diagnostics against the CPU oracle (developer tool beside the graded checks; like them it may use the oracle).

Usage on a GPU box:  python tests/gpu_diag.py            # every stage, each in its own subprocess
                     python tests/gpu_diag.py --stage conv
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

STAGES = ["frontend", "conv_first", "conv", "linear", "gru", "mha", "attpool",
          "model_gru", "model_tr"]


def rel_err(a, b):
    import torch
    a = a.double().cpu()
    b = b.double().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item(), (a - b).abs().max().item()


def conv_ref(x_nhwc, w, scale, shift, mode):
    """x NHWC float (already 16-bit rounded), w [Cout,Cin,3,3] float (rounded)."""
    import torch
    import torch.nn.functional as F
    y = F.conv2d(x_nhwc.permute(0, 3, 1, 2).float(), w.float(), padding=1)
    y = torch.relu(y * scale[None, :, None, None] + shift[None, :, None, None])
    if mode == 1:
        y = F.avg_pool2d(y, 2)
    if mode == 2:
        return y.mean(dim=3).permute(0, 2, 1)  # [N,H,C]
    return y.permute(0, 2, 3, 1)


def run_stage(stage):
    import numpy as np
    import torch
    import sed_oracle as so
    from sed_b200 import capi, engine, synth
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    lib = capi.load()
    stream = capi.current_stream(dev)
    td, code = torch.float16, 0

    if stage == "frontend":
        for sr in (16000, 8000, 32000):
            n_fft, hop, fmin, fmax = synth.PRESETS[sr]
            sd = synth.synthetic_state_dict("Cnn_9layers_Gru_FrameAtt", sr)
            L = sr * 3 + 1
            wave = torch.cat([synth.synthetic_waveform(2, L, kind="events", sample_rate=sr),
                              synth.synthetic_waveform(1, L, kind="noise"), torch.zeros(1, L)])
            tone = 0.8 * torch.sin(2 * np.pi * 440.0 * torch.arange(L) / sr)
            wave = torch.cat([wave, (torch.round(tone * 32767) / 32767)[None].float()])
            plan = engine.FrontendPlan(sd["spectrogram_extractor.stft.conv_real.weight"],
                                       sd["spectrogram_extractor.stft.conv_imag.weight"], n_fft, hop,
                                       sd["logmel_extractor.melW"], dev)
            got = engine.logmel_forward(plan, wave.to(dev)).cpu()
            spec = so.spectrogram(wave, sd["spectrogram_extractor.stft.conv_real.weight"],
                                  sd["spectrogram_extractor.stft.conv_imag.weight"], n_fft, hop)
            ref = so.logmel(spec, sd["logmel_extractor.melW"])[:, 0]
            f64 = torch.from_numpy(so.logmel_float64_fft(wave.numpy(), n_fft, hop, sd["logmel_extractor.melW"].numpy()))
            tol = 1e-4 * torch.clamp(ref.abs(), min=1.0)
            viol = ((got - ref).abs() > tol).float().mean().item()
            print("frontend sr=%d: max|d| vs ref %.3e, viol frac %.3e, ref vs f64 %.3e, got vs f64 %.3e" % (
                sr, (got - ref).abs().max(), viol, (ref.double() - f64).abs().max(), (got.double() - f64).abs().max()))
            for c in range(wave.shape[0]):
                print("     clip %d: vs ref %.3e viol %.3e | got vs f64 %.3e | ref vs f64 %.3e | min dB %.1f" % (
                    c, (got[c] - ref[c]).abs().max(), ((got[c] - ref[c]).abs() > tol[c]).float().mean(),
                    (got[c].double() - f64[c]).abs().max(), (ref[c].double() - f64[c]).abs().max(), ref[c].min()))
            gspec = engine.spectrogram_forward(plan, wave.to(dev)).cpu()
            print("   spectrogram rel err %.3e" % rel_err(gspec, spec)[0])
        return

    if stage == "conv_first":
        x = torch.randn(2, 37, 64)
        w = torch.randn(64, 1, 3, 3) * 0.3
        scale = torch.rand(64) + 0.5
        shift = torch.randn(64) * 0.1
        out = torch.empty(2, 37, 64, 64, dtype=td, device=dev)
        xd, wd, sc, sh = x.to(dev), w.reshape(64, 9).contiguous().to(dev), scale.to(dev), shift.to(dev)
        rc = lib.sed_conv_first_f32(capi.ptr(xd), 2, 37, 64, capi.ptr(wd), capi.ptr(sc), capi.ptr(sh), capi.ptr(out),
                                    code, stream)
        capi.check(rc, "conv_first")
        torch.cuda.synchronize()
        ref = conv_ref(x[..., None], w, scale, shift, 0)
        print("conv_first rel/abs err", rel_err(out.float(), ref))
        return

    if stage == "conv":
        for (name, cin, cout, mode) in engine.CONV_LAYERS:
            W = {64: 64 if cout == 64 else 32, 128: 32 if cout == 128 else 16, 256: 16 if cout == 256 else 8, 512: 8}[cin]
            for (NB, H) in ((1, 16), (3, 37)):
                x = (torch.randn(NB, H, W, cin) * 0.5).to(td)
                w = (torch.randn(cout, cin, 3, 3) * (1.0 / np.sqrt(9 * cin))).to(td)
                scale = torch.rand(cout) + 0.5
                shift = torch.randn(cout) * 0.1
                wp = w.permute(0, 2, 3, 1).reshape(cout, 9 * cin).contiguous().to(dev)
                oshape = {0: (NB, H, W, cout), 1: (NB, H // 2, W // 2, cout), 2: (NB, H, cout)}[mode]
                out = torch.full(oshape, float("nan"), dtype=td, device=dev)
                t0 = time.time()
                xd, sc, sh = x.to(dev), scale.to(dev), shift.to(dev)
                rc = lib.sed_conv3x3_bn_relu(capi.ptr(xd), NB, H, W, cin, capi.ptr(wp), capi.ptr(sc),
                                             capi.ptr(sh), cout, mode, capi.ptr(out), None, 0, 0, code, stream)
                capi.check(rc, name)
                torch.cuda.synchronize()
                ref = conv_ref(x.float(), w.float(), scale, shift, mode)
                r, a = rel_err(out.float(), ref)
                nan = torch.isnan(out.float()).float().mean().item()
                print("%s %s (%d->%d mode %d) NB=%d H=%d W=%d: rel %.3e abs %.3e nan %.3f  [%.3fs]" % (
                    stage, name, cin, cout, mode, NB, H, W, r, a, nan, time.time() - t0), flush=True)
        return

    if stage == "linear":
        for (M, K, N, relu) in ((125 * 3, 512, 1536, 0), (300, 512, 512, 1), (128, 256, 768, 0)):
            a = (torch.randn(M, K) * 0.5).to(td)
            w = (torch.randn(N, K) / np.sqrt(K)).to(td)
            bias = torch.randn(N) * 0.1
            out = torch.full((M, N), float("nan"), dtype=torch.float32, device=dev)
            ad, wd, bd = a.to(dev), w.to(dev), bias.to(dev)
            rc = lib.sed_linear(capi.ptr(ad), M, K, capi.ptr(wd), capi.ptr(bd), N, relu,
                                capi.ptr(out), None, 0, code, stream)
            capi.check(rc, "linear")
            torch.cuda.synchronize()
            ref = a.float() @ w.float().t() + bias
            if relu:
                ref = torch.relu(ref)
            print("linear M=%d K=%d N=%d relu=%d rel/abs" % (M, K, N, relu), rel_err(out, ref),
                  "nan", torch.isnan(out).float().mean().item())
        return

    if stage == "gru":
        sd = synth.synthetic_state_dict("Cnn_9layers_Gru_FrameAtt")
        pm = engine.PackedModel(sd, "Cnn_9layers_Gru_FrameAtt", 512, 160, dev)
        for (B, T) in ((3, 7), (130, 20), (5, 125)):
            x = torch.relu(torch.randn(B, T, 512) * 0.5).to(td)
            t0 = time.time()
            got = pm.temporal(x.to(dev))
            torch.cuda.synchronize()
            ref = so.bigru(x.float(), sd)
            print("gru B=%d T=%d rel/abs" % (B, T), rel_err(got, ref), "[%.3fs]" % (time.time() - t0), flush=True)
        return

    if stage == "mha":
        sd = synth.synthetic_state_dict("Cnn_9layers_Transformer_FrameAtt")
        pm = engine.PackedModel(sd, "Cnn_9layers_Transformer_FrameAtt", 512, 160, dev)
        for (B, T) in ((2, 62), (3, 125)):
            x = torch.relu(torch.randn(B, T, 512) * 0.5).to(td)
            got = pm.temporal(x.to(dev))
            torch.cuda.synchronize()
            ref = so.multihead(x.float(), sd)
            print("mha B=%d T=%d rel/abs" % (B, T), rel_err(got, ref), flush=True)
        return

    if stage == "attpool":
        sd = synth.synthetic_state_dict("Cnn_9layers_Gru_FrameAtt")
        pm = engine.PackedModel(sd, "Cnn_9layers_Gru_FrameAtt", 512, 160, dev)
        for (B, T, frames) in ((3, 125, 1000), (2, 62, 500)):
            x = torch.tanh(torch.randn(B, T, 512))
            clip, frame, cla, natt = pm.head(x.to(dev), frames, True, True)
            torch.cuda.synchronize()
            rclip, rnatt, rcla = so.att_block(x.transpose(1, 2), sd)
            rfw = so.interpolate(rcla.transpose(1, 2), 8)
            if rfw.shape[1] != frames:
                rfw = so.pad_framewise_output(rfw, frames)
            print("attpool B=%d T=%d clip %.3e frame %.3e cla %.3e natt %.3e" % (
                B, T, rel_err(clip, rclip)[1], rel_err(frame, rfw)[1], rel_err(cla, rcla)[1], rel_err(natt, rnatt)[1]))
        return

    if stage in ("model_gru", "model_tr"):
        from sed_b200 import models
        mt = "Cnn_9layers_Gru_FrameAtt" if stage == "model_gru" else "Cnn_9layers_Transformer_FrameAtt"
        sd = synth.synthetic_state_dict(mt)
        wave = torch.cat([synth.synthetic_waveform(2, 160000, kind="events"), synth.synthetic_waveform(1, 160000)])
        ref, rst = so.model_forward(sd, wave, mt, 512, 160, return_stages=True)
        for variant in (4, 2):
            pm = engine.PackedModel(sd, mt, 512, 160, dev)
            t0 = time.time()
            got, st = pm.forward(wave.to(dev), variant=variant, return_stages=True)
            torch.cuda.synchronize()
            print("%s variant %d [%.2fs]" % (mt, variant, time.time() - t0))
            print("   bn0 abs", rel_err(st["bn0"], rst["bn0"][:, 0])[1])
            for k, rk in (("p1", "conv_block1"), ("p2", "conv_block2"), ("p3", "conv_block3")):
                print("   %s rel/abs" % rk, rel_err(st[k].float().permute(0, 3, 1, 2), rst[rk]))
            print("   feat rel/abs", rel_err(st["feat"].float(), rst["feat"]))
            print("   temporal rel/abs", rel_err(st["temporal"], rst["temporal"]))
            for k in ("clipwise_output", "framewise_output", "embedding"):
                print("   %s abs %.3e" % (k, rel_err(got[k], ref[k])[1]))
            flips = ((got["framewise_output"].cpu() > 0.5) != (ref["framewise_output"] > 0.5)).float().mean().item()
            print("   flips@0.5 %.3e" % flips, flush=True)
        return
    raise SystemExit("unknown stage " + stage)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--stage", default=None)
    ap.add_argument("--timeout", type=int, default=240)
    args = ap.parse_args()
    if args.stage:
        run_stage(args.stage)
        return
    for st in STAGES:
        t0 = time.time()
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--stage", st], timeout=args.timeout,
                               capture_output=True, text=True)
            print("===== %s rc=%d (%.1fs)" % (st, r.returncode, time.time() - t0))
            print(r.stdout[-6000:])
            if r.returncode != 0:
                print(r.stderr[-3000:])
        except subprocess.TimeoutExpired as e:
            print("===== %s TIMEOUT after %ds" % (st, args.timeout))
            print((e.stdout or b"").decode("utf-8", "replace")[-3000:] if isinstance(e.stdout, bytes) else (e.stdout or "")[-3000:])
        sys.stdout.flush()


if __name__ == "__main__":
    main()
