"""GPU parity of the individual kernels through the C ABI: conv layers (CTA-pair kernels), first conv layer, tensor-core linear, GRU, attention core, frame-attention head."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import sed_oracle as so
from conftest import synthetic_sd
from sed_b200 import capi, engine

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
DTYPES = {"fp16": (0, torch.float16, 2e-3), "bf16": (1, torch.bfloat16, 1.6e-2)}


def conv_ref(x_nhwc, w, scale, shift, mode):
    y = F.conv2d(x_nhwc.permute(0, 3, 1, 2).float(), w.float(), padding=1)
    y = torch.relu(y * scale[None, :, None, None] + shift[None, :, None, None])
    if mode == 1:
        y = F.avg_pool2d(y, 2)
    if mode == 2:
        return y.mean(dim=3).permute(0, 2, 1)
    return y.permute(0, 2, 3, 1)


def run_conv(x, w, scale, shift, mode, code, td):
    lib = capi.load()
    NB, H, W, cin = x.shape
    cout = w.shape[0]
    xd = x.to(DEV)
    wp = w.permute(0, 2, 3, 1).reshape(cout, 9 * cin).contiguous().to(DEV)
    sc, sh = scale.to(DEV), shift.to(DEV)
    oshape = {0: (NB, H, W, cout), 1: (NB, H // 2, W // 2, cout), 2: (NB, H, cout)}[mode]
    out = torch.full(oshape, float("nan"), dtype=td, device=DEV)
    rc = lib.sed_conv3x3_bn_relu(capi.ptr(xd), NB, H, W, cin, capi.ptr(wp), capi.ptr(sc), capi.ptr(sh), cout, mode,
                                 capi.ptr(out), None, 0, 0, code, capi.current_stream(DEV))
    capi.check(rc, "sed_conv3x3_bn_relu")
    torch.cuda.synchronize()
    return out.float().cpu()


@pytest.mark.parametrize("draw", [0, 1, 2])
@pytest.mark.parametrize("layer", engine.CONV_LAYERS, ids=[l[0] for l in engine.CONV_LAYERS])
def test_conv_layers_match_cpu_conv(layer, draw):
    """Every layer's CTA-pair kernel on three independent draws of inputs, weights and BatchNorm."""
    name, cin, cout, mode = layer
    W = {64: 64 if cout == 64 else 32, 128: 32 if cout == 128 else 16, 256: 16 if cout == 256 else 8, 512: 8}[cin]
    code, td, tol = DTYPES["fp16"]
    g = torch.Generator().manual_seed(cin * 7 + cout + 1000 * draw)
    # ragged heights: 1 row, odd rows (pool floors), non-multiples of the 16-row tile, several images
    for NB, H in ((1, 16), (3, 37), (2, 2), (1, 125 if cin >= 256 else 63)):
        if mode == 1 and H < 2:
            continue
        x = (torch.randn(NB, H, W, cin, generator=g) * 0.5).to(td)
        w = (torch.randn(cout, cin, 3, 3, generator=g) / np.sqrt(9 * cin)).to(td)
        scale = torch.rand(cout, generator=g) + 0.5
        shift = torch.randn(cout, generator=g) * 0.1
        got = run_conv(x, w, scale, shift, mode, code, td)
        ref = conv_ref(x.float(), w.float(), scale, shift, mode)
        assert not torch.isnan(got).any()
        err = (got - ref).abs().max().item() / ref.abs().max().item()
        assert err < tol, (name, NB, H, err)


def test_conv_bf16_path():
    code, td, tol = DTYPES["bf16"]
    x = (torch.randn(2, 20, 16, 256) * 0.5).to(td)
    w = (torch.randn(256, 256, 3, 3) / 48).to(td)
    scale, shift = torch.rand(256) + 0.5, torch.randn(256) * 0.1
    got = run_conv(x, w, scale, shift, 1, code, td)
    ref = conv_ref(x.float(), w.float(), scale, shift, 1)
    assert (got - ref).abs().max().item() / ref.abs().max().item() < tol


def test_conv_variants_agree_bitwise():
    """Every output is the same MMAs in the same K order whichever CTA of which pair computes its tile: a batch of
    three images equals the three images launched one at a time, bit for bit (resident and streamed weights)."""
    code, td, _ = DTYPES["fp16"]
    for cin, cout, W in ((128, 128, 32), (256, 256, 16)):
        x = (torch.randn(3, 40, W, cin) * 0.5).to(td)
        w = (torch.randn(cout, cin, 3, 3) / np.sqrt(9 * cin)).to(td)
        scale, shift = torch.rand(cout) + 0.5, torch.randn(cout) * 0.1
        a = run_conv(x, w, scale, shift, 1, code, td)
        b = torch.cat([run_conv(x[i:i + 1], w, scale, shift, 1, code, td) for i in range(3)])
        assert torch.equal(a, b), (cin, cout)


def test_conv_rejects_unsupported_layers():
    lib = capi.load()
    x = torch.zeros(1, 16, 8, 192, dtype=torch.float16, device=DEV)
    with pytest.raises(NotImplementedError):
        rc = lib.sed_conv3x3_bn_relu(capi.ptr(x), 1, 16, 8, 192, capi.ptr(x), capi.ptr(x), capi.ptr(x), 192, 0,
                                     capi.ptr(x), None, 0, 0, 0, capi.current_stream(DEV))
        capi.check(rc, "conv")
    with pytest.raises(ValueError):
        rc = lib.sed_conv3x3_bn_relu(capi.ptr(x), 1, 16, 7, 64, capi.ptr(x), capi.ptr(x), capi.ptr(x), 64, 1,
                                     capi.ptr(x), None, 0, 0, 0, capi.current_stream(DEV))
        capi.check(rc, "conv")


def test_conv_first_layer():
    lib = capi.load()
    for NB, H in ((2, 37), (1, 1001)):
        x = torch.randn(NB, H, 64)
        w = torch.randn(64, 1, 3, 3) * 0.3
        scale, shift = torch.rand(64) + 0.5, torch.randn(64) * 0.1
        out = torch.empty(NB, H, 64, 64, dtype=torch.float16, device=DEV)
        xd, wd, sc, sh = x.to(DEV), w.reshape(64, 9).contiguous().to(DEV), scale.to(DEV), shift.to(DEV)
        rc = lib.sed_conv_first_f32(capi.ptr(xd), NB, H, 64, capi.ptr(wd), capi.ptr(sc), capi.ptr(sh), capi.ptr(out), 0,
                                    capi.current_stream(DEV))
        capi.check(rc, "conv_first")
        ref = conv_ref(x[..., None], w, scale, shift, 0)
        assert (out.float().cpu() - ref).abs().max().item() < 1e-3 * ref.abs().max().item()


@pytest.mark.parametrize("M,K,N,relu", [(375, 512, 1536, 0), (300, 512, 512, 1), (128, 256, 768, 0), (1, 512, 512, 0)])
def test_linear(M, K, N, relu):
    lib = capi.load()
    a = (torch.randn(M, K) * 0.5).half()
    w = (torch.randn(N, K) / np.sqrt(K)).half()
    bias = torch.randn(N) * 0.1
    out = torch.full((M, N), float("nan"), dtype=torch.float32, device=DEV)
    ad, wd, bd = a.to(DEV), w.to(DEV), bias.to(DEV)
    rc = lib.sed_linear(capi.ptr(ad), M, K, capi.ptr(wd), capi.ptr(bd), N, relu, capi.ptr(out), None, 0, 0,
                        capi.current_stream(DEV))
    capi.check(rc, "sed_linear")
    ref = a.float() @ w.float().t() + bias
    if relu:
        ref = torch.relu(ref)
    assert (out.cpu() - ref).abs().max().item() < 2e-4 * max(ref.abs().max().item(), 1.0)


@pytest.mark.parametrize("B,T", [(1, 1), (3, 7), (130, 20), (5, 125), (2, 62)])
def test_bigru_matches_oracle(B, T):
    mt = "Cnn_9layers_Gru_FrameAtt"
    sd = synthetic_sd(mt)
    pm = engine.PackedModel(sd, mt, 512, 160, DEV)
    x = torch.relu(torch.randn(B, T, 512, generator=torch.Generator().manual_seed(B * 131 + T)) * 0.5).half()
    got = pm.temporal(x.to(DEV)).cpu()
    ref = so.bigru(x.float(), sd)
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() < 1.5e-3  # fp16 operands of h W_hh^T over T recurrent steps


@pytest.mark.parametrize("B,T", [(1, 1), (2, 62), (3, 125), (2, 140)])
def test_multihead_matches_oracle(B, T):
    mt = "Cnn_9layers_Transformer_FrameAtt"
    sd = synthetic_sd(mt)
    pm = engine.PackedModel(sd, mt, 512, 160, DEV)
    x = torch.relu(torch.randn(B, T, 512, generator=torch.Generator().manual_seed(B * 17 + T)) * 0.5).half()
    got = pm.temporal(x.to(DEV)).cpu()
    ref = so.multihead(x.float(), sd)
    assert (got - ref).abs().max().item() < 2e-3 * max(ref.abs().max().item(), 1.0)


@pytest.mark.parametrize("B,T", [(3, 125), (130, 62), (2, 128), (1, 1), (5, 17)])
def test_tensor_core_attention_matches_float32_kernel_and_torch(B, T):
    """sed_mha_attention (tcgen05 QK^T / PV, 16-bit q | k | v | P) against softmax(q k^T / 8) v in float64 on the same
    16-bit inputs, and against the float32 kernel sed_mha_core; time-major rows over a batch padded to 128."""
    lib = capi.load()
    Bp = (B + 127) // 128 * 128
    g = torch.Generator().manual_seed(B * 31 + T)
    qkv = (torch.randn(T, Bp, 1536, generator=g) * 1.5).half()
    qkv_d = qkv.to(DEV)
    ctx = torch.full((T * Bp, 512), float("nan"), dtype=torch.float16, device=DEV)
    capi.check(lib.sed_mha_attention(capi.ptr(qkv_d), None, B, T, Bp, capi.ptr(ctx), 0, capi.current_stream(DEV)),
               "sed_mha_attention")
    x = qkv[:, :B].double().permute(1, 0, 2)                              # [B, T, 1536]
    q, k, v = (x[..., i * 512:(i + 1) * 512].reshape(B, T, 8, 64).permute(0, 2, 1, 3) for i in range(3))
    ref = torch.softmax(q @ k.transpose(-1, -2) / 8.0, dim=-1) @ v          # [B, 8, T, 64]
    ref = ref.permute(2, 0, 1, 3).reshape(T, B, 512)
    got = ctx.view(T, Bp, 512)[:, :B].float().cpu()
    assert torch.isfinite(got).all()
    # 16-bit P and the 16-bit store of the context: ~1e-3 relative
    assert (got.double() - ref).abs().max().item() <= 4e-3 * max(1.0, ref.abs().max().item())
    if Bp != B:
        assert torch.isnan(ctx.view(T, Bp, 512)[:, B:].float()).all()       # rows of padding clips are not written
    ctx32 = torch.zeros((T * Bp, 512), dtype=torch.float16, device=DEV)
    qkv32 = qkv_d.float().contiguous()
    capi.check(lib.sed_mha_core(capi.ptr(qkv32), B, T, Bp, 1, capi.ptr(ctx32), 0, capi.current_stream(DEV)), "sed_mha_core")
    old = ctx32.view(T, Bp, 512)[:, :B].float().cpu()
    assert (got - old).abs().max().item() <= 4e-3 * max(1.0, ref.abs().max().item())


def test_split_precision_projection_and_logits():
    """sed_linear_split16: hi + lo reproduce the float32 projection to ~2^-21; with the residual tiles the attention
    kernel's result follows float32 q, k (large logits: the case plain 16-bit operands lose)."""
    lib = capi.load()
    B, T, Bp = 3, 125, 128
    g = torch.Generator().manual_seed(77)
    x = (torch.randn(T * Bp, 512, generator=g)).half()
    w = (torch.randn(1536, 512, generator=g) * 0.2).half()      # logits of magnitude ~ 40
    bias = torch.randn(1536, generator=g)
    hi = torch.empty((T * Bp, 1536), dtype=torch.float16, device=DEV)
    lo = torch.empty((T * Bp, 1024), dtype=torch.float16, device=DEV)
    xd, wd, bd = x.to(DEV), w.to(DEV), bias.to(DEV)
    capi.check(lib.sed_linear_split16(capi.ptr(xd), T * Bp, 512, capi.ptr(wd), capi.ptr(bd), 1536, capi.ptr(hi),
                                      capi.ptr(lo), 1024, 0, capi.current_stream(DEV)), "sed_linear_split16")
    ref = x.double() @ w.double().t() + bias.double()
    assert (hi.double().cpu() - ref).abs().max() <= 1e-3 * ref.abs().max()
    both = hi[:, :1024].double().cpu() + lo.double().cpu()
    assert (both - ref[:, :1024]).abs().max() <= 2e-6 * ref.abs().max()
    r3 = ref.view(T, Bp, 1536)[:, :B].permute(1, 0, 2)
    q, k = (r3[..., i * 512:(i + 1) * 512].reshape(B, T, 8, 64).permute(0, 2, 1, 3) for i in range(2))
    v = hi.view(T, Bp, 1536)[:, :B, 1024:].double().cpu().permute(1, 0, 2).reshape(B, T, 8, 64).permute(0, 2, 1, 3)
    want = (torch.softmax(q @ k.transpose(-1, -2) / 8.0, dim=-1) @ v).permute(2, 0, 1, 3).reshape(T, B, 512)
    errs = []
    for lo_arg in (lo, None):
        ctx = torch.zeros((T * Bp, 512), dtype=torch.float16, device=DEV)
        capi.check(lib.sed_mha_attention(capi.ptr(hi), capi.ptr(lo_arg), B, T, Bp, capi.ptr(ctx), 0,
                                         capi.current_stream(DEV)), "sed_mha_attention")
        errs.append((ctx.view(T, Bp, 512)[:, :B].double().cpu() - want).abs().max().item())
    print("\nattention vs float64 logits: split %.2e, plain 16-bit q/k %.2e" % tuple(errs))
    assert errs[0] <= 4e-3 * max(1.0, want.abs().max().item())
    assert errs[0] < errs[1]


def test_long_clips_take_the_float32_attention_kernel():
    mt = "Cnn_9layers_Transformer_FrameAtt"
    sd = synthetic_sd(mt)
    pm = engine.PackedModel(sd, mt, 512, 160, DEV)
    x = torch.relu(torch.randn(2, 200, 512, generator=torch.Generator().manual_seed(9)) * 0.5).half()
    got = pm.temporal(x.to(DEV)).cpu()
    ref = so.multihead(x.float(), sd)
    assert (got - ref).abs().max().item() < 2e-3 * max(ref.abs().max().item(), 1.0)


@pytest.mark.parametrize("B,T,frames", [(3, 125, 1000), (2, 62, 500), (2, 62, 496), (1, 1, 100)])
def test_attpool_matches_oracle(B, T, frames):
    mt = "Cnn_9layers_Gru_FrameAtt"
    sd = synthetic_sd(mt)
    pm = engine.PackedModel(sd, mt, 512, 160, DEV)
    x = torch.tanh(torch.randn(B, T, 512, generator=torch.Generator().manual_seed(T)))
    clip, frame, cla, natt = pm.head(x.to(DEV), frames, True, True)
    rclip, rnatt, rcla = so.att_block(x.transpose(1, 2), sd)
    rfw = so.interpolate(rcla.transpose(1, 2), 8)
    if rfw.shape[1] != frames:
        rfw = so.pad_framewise_output(rfw, frames)
    assert (clip.cpu() - rclip).abs().max() < 2e-6
    assert (frame.cpu() - rfw).abs().max() < 2e-6
    assert (cla.cpu() - rcla).abs().max() < 2e-6
    assert (natt.cpu() - rnatt).abs().max() < 2e-6


def test_linear_transposed_block_layout_is_a_pure_permutation():
    """sed_linear out_layout=1 (the layout sed_bigru streams): float4 c of row r at ((r/128)*N/4 + c)*128 + r%128."""
    lib = capi.load()
    M, K, N = 384, 512, 1536
    g = torch.Generator().manual_seed(5)
    a = torch.randn(M, K, generator=g).half().to(DEV)
    w = (torch.randn(N, K, generator=g) * 0.05).half().to(DEV)
    b = torch.randn(N, generator=g).to(DEV)
    outs = []
    for layout in (0, 1):
        out = torch.full((M, N), float("nan"), device=DEV)
        rc = lib.sed_linear(capi.ptr(a), M, K, capi.ptr(w), capi.ptr(b), N, 0, capi.ptr(out), None, layout, 0,
                            capi.current_stream(DEV))
        capi.check(rc, "sed_linear")
        outs.append(out)
    torch.cuda.synchronize()
    blocks = outs[1].view(M // 128, N // 4, 128, 4).permute(0, 2, 1, 3).reshape(M, N)
    assert torch.equal(blocks, outs[0])
    with pytest.raises(NotImplementedError):
        rc = lib.sed_linear(capi.ptr(a), 100, K, capi.ptr(w), capi.ptr(b), N, 0, capi.ptr(outs[0]), None, 1, 0,
                            capi.current_stream(DEV))
        capi.check(rc, "sed_linear")


def test_weight_preparation_helpers_match_the_host_statements():
    """sed_fold_bn / sed_pack_conv3x3 / sed_pack_conv_first / sed_pack_gru_whh / sed_cast_16 against the torch
    expressions they replace, bit for bit, for both 16-bit types."""
    from sed_b200 import synth
    sd = synth.synthetic_state_dict("Cnn_9layers_Gru_FrameAtt", 16000)
    for prefix in ("bn0", "conv_block1.bn1", "conv_block4.bn2"):
        s_ref, b_ref = engine.fold_bn(sd, prefix)
        s, b = engine.fold_bn_device(sd, prefix, DEV)
        assert torch.equal(s.cpu(), s_ref) and torch.equal(b.cpu(), b_ref)
    lib = capi.load()
    stream = capi.current_stream(DEV)
    for code, td in ((capi.SED_DTYPE_F16, torch.float16), (capi.SED_DTYPE_BF16, torch.bfloat16)):
        w = sd["conv_block3.conv1.weight"].float()
        ref = w.permute(0, 2, 3, 1).reshape(256, 9 * 128).to(td)
        got = torch.empty((256, 9 * 128), dtype=td, device=DEV)
        wd = w.contiguous().to(DEV)
        assert lib.sed_pack_conv3x3(capi.ptr(wd), 256, 128, capi.ptr(got), code, stream) == 0
        assert torch.equal(got.cpu(), ref)
        packed = []
        for suffix in ("", "_reverse"):
            whh = sd["gru.weight_hh_l0" + suffix].float()
            packed.append(whh.view(3, 8, 32, 256).permute(1, 0, 2, 3).reshape(768, 256))
        ref = torch.cat(packed, 0).to(td)
        got = torch.empty((1536, 256), dtype=td, device=DEV)
        f, r = (sd["gru.weight_hh_l0" + x].float().contiguous().to(DEV) for x in ("", "_reverse"))
        assert lib.sed_pack_gru_whh(capi.ptr(f), capi.ptr(r), capi.ptr(got), code, stream) == 0
        assert torch.equal(got.cpu(), ref)
        x = torch.randn(100003, generator=torch.Generator().manual_seed(1)) * 3
        assert torch.equal(engine.cast16_device(x, td, code, DEV).cpu(), x.to(td))
    s1, _ = engine.fold_bn(sd, "conv_block1.bn1")
    ref = (sd["conv_block1.conv1.weight"].double().reshape(64, 9) * s1.double()[:, None]).float()
    w1 = sd["conv_block1.conv1.weight"].float().reshape(64, 9).contiguous().to(DEV)
    got = torch.empty((64, 9), dtype=torch.float32, device=DEV)
    assert lib.sed_pack_conv_first(capi.ptr(w1), capi.ptr(s1.to(DEV)), capi.ptr(got), stream) == 0
    assert torch.equal(got.cpu(), ref)
    assert lib.sed_pack_conv3x3(capi.ptr(w1), 64, 1, capi.ptr(got), 7, stream) != 0
