"""Timing decomposition of the conv kernels via SED_CONV_DBG (1 = no stores, 2 = no drain, 4 = no MMA)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from sed_b200 import capi, engine, synth
capi.use_profile_library()  # experiment switches / stamps exist only in the -DSED_PROFILE build
from tools.profile_layers import timeit

dev = torch.device("cuda:0")
lib = capi.load()
sd = synth.synthetic_state_dict("Cnn_9layers_Gru_FrameAtt", 16000)
pm = engine.PackedModel(sd, "Cnn_9layers_Gru_FrameAtt", 512, 160, dev)
mb = 148
wave = synth.synthetic_waveform(mb, 160000).to(dev)
ws = pm._workspace(mb, 1001, need_a1=True)  # conv_block1.conv2 alone reads conv1's output
feat = torch.empty((mb, 125, 512), dtype=pm.tdtype, device=dev)
pm.conv_stack(wave, feat)
stream = capi.current_stream(dev)
chain = [("a1", "p1"), ("p1", "a2"), ("a2", "p2"), ("p2", "a3"), ("a3", "p3"), ("p3", "a4"), ("a4", None)]
print("%-28s %8s %8s %8s %8s %8s" % ("layer", "full", "nostore", "nodrain", "nomma", "nomma+nodrain"))
for (name, _, _, _), (cin, cout, mode, wp, s, b), (src, dst) in zip(engine.CONV_LAYERS, pm.convs, chain):
    x = ws[src]
    out = feat if dst is None else ws[dst]
    res = []
    for flag in (0, 1, 2, 4, 6):
        os.environ["SED_CONV_DBG"] = str(flag)
        res.append(timeit(lambda: lib.sed_conv3x3_bn_relu(capi.ptr(x), mb, x.shape[1], x.shape[2], cin, capi.ptr(wp),
                                                          capi.ptr(s), capi.ptr(b), cout, mode, capi.ptr(out), None, 0, 0,
                                                          pm.dtype_code, stream)))
    os.environ["SED_CONV_DBG"] = "0"
    flops = 2.0 * mb * x.shape[1] * x.shape[2] * 9 * cin * cout
    print("%-28s %8.3f %8.3f %8.3f %8.3f %8.3f   ideal@2.3PF %.3f" % ((name,) + tuple(res) + (flops / 2.3e15 * 1e3,)))
