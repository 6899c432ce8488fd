"""Fused conv_block1 (engine variant 4) against the two-kernel block 1 (variant 2) -- developer tool."""
import os, sys
sys.path.insert(0, "/root/repo")
import torch
from sed_b200 import capi, engine, synth
from tools.profile_layers import timeit
dev = torch.device("cuda:0")
mt = "Cnn_9layers_Gru_FrameAtt"
pm = engine.PackedModel(synth.synthetic_state_dict(mt, 16000), mt, 512, 160, dev)
wave = synth.synthetic_waveform(148, 160000).to(dev)
feat = torch.empty((148, 125, 512), dtype=pm.tdtype, device=dev)
for v in (2, 4):
    t = timeit(lambda: pm.conv_stack(wave, feat, variant=v))
    print("conv_stack variant %d: %.3f ms per 148 clips" % (v, t))
lib = capi.load(); ws = pm._workspace(148, 1001); stream = capi.current_stream(dev)
cin, cout, mode, wp, s, b = pm.convs[0]
t = timeit(lambda: lib.sed_conv_block1(capi.ptr(ws["logmel"]), 148, 1001, 64, capi.ptr(pm.c11_ws), capi.ptr(pm.c11_shift), capi.ptr(wp), capi.ptr(s), capi.ptr(b), capi.ptr(ws["p1"]), pm.dtype_code, stream))
print("fused conv_block1: %.3f ms" % t)
wv = synth.synthetic_waveform(1024, 160000).to(dev)
for v in (2, 4):
    t = timeit(lambda: pm.forward(wv, variant=v), n=5, warm=2)
    print("forward B=1024 variant %d: %.3f ms -> %.0f clips/s" % (v, t, 1024 / t * 1e3))
