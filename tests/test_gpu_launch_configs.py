"""The launch configurations a default forward runs, each against a float64 reference of the same operation computed
from the same 16-bit-rounded operands:

  * conv_block1 as one kernel (sed_conv_block1, engine variant 4) and as two (sed_conv_first_f32 + the conv1_2 pair
    kernel, variant 2), fp16 and bf16, including the 32-bit tile index limit that engine.clamp_micro_batch mirrors;
  * sed_conv3x3_bn_relu 512 -> 512 with the freq-mean epilogue writing time-major feature rows (and its float32 copy);
  * sed_linear / sed_linear_split16 at production row counts (two row tiles per work item, column panels), and the
    temporal blocks that run them at B = 300, T' = 125;
  * sed_attpool_blocks (staged and unstaged) and sed_fcpool.

Every bound is a small factor above the error measured on a B200 and far below what a wrong variant gives; run with
-s to see the measured values.  The reference self-checks at the top need no GPU."""
import pytest
import torch
import torch.nn.functional as F

import sed_oracle as so
from conftest import synthetic_sd
from sed_b200 import capi, engine

gpu = pytest.mark.gpu
DEV = torch.device("cuda:0")
F64 = torch.float64
DTYPES = {"fp16": (capi.SED_DTYPE_F16, torch.float16), "bf16": (capi.SED_DTYPE_BF16, torch.bfloat16)}
GUARD = 4096  # sentinel elements after every output buffer


# ------------------------------------------------------------------------------------------------ helpers
def ulp16(v, td):
    """Spacing of the 16-bit format at |v| (float64): fp16 has 10 fraction bits and emin -14, bf16 7 and -126."""
    p, emin = (10, -14) if td == torch.float16 else (7, -126)
    v = v.double().abs()
    _, e = torch.frexp(v)
    e = torch.where(v == 0, torch.full_like(e, emin + 1), e)
    return torch.ldexp(torch.ones_like(v), (e - 1).clamp(min=emin) - p)


def ulp_distance(a, b):
    """|a - b| in units in the last place of two tensors of the same 16-bit type holding values >= 0."""
    return (a.view(torch.int16).int() - b.view(torch.int16).int()).abs()


def report(what, **vals):
    print("\n%s: %s" % (what, ", ".join("%s %s" % (k, ("%.3e" % v) if isinstance(v, float) else v)
                                         for k, v in vals.items())))


def call(name, *args):
    capi.check(getattr(capi.load(), name)(*args), name)


def stream():
    return capi.current_stream(DEV)


def fold(sd, prefix):
    """Eval-mode BatchNorm of the oracle as scale / shift, in float64."""
    s = sd[prefix + ".weight"] / torch.sqrt(sd[prefix + ".running_var"] + so.BN_EPS)
    return s, sd[prefix + ".bias"] - sd[prefix + ".running_mean"] * s


# ------------------------------------------------------------------------------------------------ conv_block1
def block1_ref(x, w1s, shift1, w2, scale2, shift2, td, r0=0, r1=None):
    """conv_block1 in float64 on the pooled rows [r0, r1) of every image: a1 = relu(conv1(x) * s1 + b1) with zero
    padding (w1s = conv1 weights x s1, shift1 = b1), rounded to `td` (None: not rounded), then conv2 (w2 [64, 64, 3, 3])
    on a1 with zero padding, bn2 (scale2, shift2), ReLU and the 2 x 2 average pool (an odd H floors).
    Returns (p [NB, r1 - r0, W/2, 64], m) with m the same pipeline run on |a1|, |w2|, |scale2|, |shift2|: the
    magnitude the float32 accumulation of the kernel is relative to."""
    NB, H, W = x.shape
    r1 = H // 2 if r1 is None else r1
    if r1 <= r0:
        z = torch.zeros((NB, 0, W // 2, 64), dtype=F64, device=x.device)
        return z, z
    lo, hi = 2 * r0 - 2, 2 * r1 + 2  # input rows the pooled rows read (conv2 and conv1 halos)
    xs = torch.zeros((NB, 1, hi - lo, W), dtype=F64, device=x.device)
    a, b = max(lo, 0), min(hi, H)
    xs[:, 0, a - lo:b - lo] = x[:, a:b].double()
    a1 = F.conv2d(xs, w1s.double().view(64, 1, 3, 3), padding=(0, 1)) + shift1.double().view(1, 64, 1, 1)
    a1 = torch.relu(a1)                                               # rows 2 r0 - 1 .. 2 r1
    rows = torch.arange(lo + 1, hi - 1, device=x.device)
    a1[:, :, (rows < 0) | (rows >= H)] = 0.0                          # conv2's padding is zero, not relu(shift1)
    if td is not None:
        a1 = a1.to(td).double()
    outs = []
    for a_, w_, s_, b_ in ((a1, w2, scale2, shift2), (a1.abs(), w2.abs(), scale2.abs(), shift2.abs())):
        y = F.conv2d(a_, w_.double(), padding=(0, 1))                 # conv rows 2 r0 .. 2 r1 - 1
        y = torch.relu(y * s_.double().view(1, 64, 1, 1) + b_.double().view(1, 64, 1, 1))
        outs.append(F.avg_pool2d(y, 2).permute(0, 2, 3, 1))
    return outs[0], outs[1]


def block1_inputs(NB, H, seed, device, probe=False, W=64):
    """Log-mel scale input (|x| up to 100, as after bn0, so conv1's products need the lo terms), conv1 weights with the
    bn1 scale folded in, a large positive bn1 shift (a padding pixel computed as relu(shift1) instead of 0 shows),
    and conv2 / bn2 parameters.  probe=True: w2 = identity at the centre tap, scale2 = 1, shift2 = 0, so the pooled
    output is the pooled 16-bit a1 and conv1's precision is visible pixel by pixel."""
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(NB, H, W, generator=g) * 30).clamp(-100, 100)
    w1s = torch.randn(64, 9, generator=g) * 0.3
    shift1 = torch.rand(64, generator=g) * 2 + 4
    if probe:
        w2 = torch.zeros(64, 64, 3, 3)
        w2[torch.arange(64), torch.arange(64), 1, 1] = 1.0
        scale2, shift2 = torch.ones(64), torch.zeros(64)
    else:
        w2 = torch.randn(64, 64, 3, 3, generator=g) / 24
        scale2 = torch.rand(64, generator=g) + 0.5
        shift2 = torch.randn(64, generator=g) * 0.1
    return [t.to(device) for t in (x, w1s, shift1, w2, scale2, shift2)]


def test_block1_reference_matches_the_oracle():
    """The reference above without its 16-bit rounding is sed_oracle.conv_block(..., 'conv_block1', (2, 2)) in
    float64, and its row slices are slices of the whole result."""
    g = torch.Generator().manual_seed(3)
    sd = {"conv_block1.conv1.weight": torch.randn(64, 1, 3, 3, generator=g, dtype=F64) * 0.3,
          "conv_block1.conv2.weight": torch.randn(64, 64, 3, 3, generator=g, dtype=F64) / 24}
    for bn in ("bn1", "bn2"):
        sd["conv_block1.%s.weight" % bn] = torch.rand(64, generator=g, dtype=F64) + 0.5
        sd["conv_block1.%s.bias" % bn] = torch.randn(64, generator=g, dtype=F64)
        sd["conv_block1.%s.running_mean" % bn] = torch.randn(64, generator=g, dtype=F64)
        sd["conv_block1.%s.running_var" % bn] = torch.rand(64, generator=g, dtype=F64) + 0.5
    s1, b1 = fold(sd, "conv_block1.bn1")
    s2, b2 = fold(sd, "conv_block1.bn2")
    w1s = sd["conv_block1.conv1.weight"].view(64, 9) * s1[:, None]
    for NB, H, W in ((2, 17, 16), (1, 16, 64), (3, 2, 16)):
        x = torch.randn(NB, H, W, generator=g, dtype=F64) * 30
        want = so.conv_block(x[:, None], sd, "conv_block1", (2, 2)).permute(0, 2, 3, 1)
        got, m = block1_ref(x, w1s, b1, sd["conv_block1.conv2.weight"], s2, b2, None)
        assert got.shape == want.shape
        assert (got - want).abs().max().item() <= 1e-9 * max(1.0, want.abs().max().item())
        assert (m >= got.abs() - 1e-9).all()
        for r0, r1 in ((0, 3), (3, 7), (H // 2 - 2, H // 2)):
            if 0 <= r0 < r1 <= H // 2:
                part, _ = block1_ref(x, w1s, b1, sd["conv_block1.conv2.weight"], s2, b2, None, r0, r1)
                assert (part - got[:, r0:r1]).abs().max().item() <= 1e-9 * max(1.0, want.abs().max().item())


def test_clamp_micro_batch_keeps_conv_block1_tile_indices_in_32_bits():
    """clamp_micro_batch caps a launch group where conv_block1 stops accepting it:
    tiles_per_clip * (NB * tiles_per_clip + 4096) < 2^32, tiles_per_clip = ceil(T / 16) * 8 (W = 64)."""
    def accepted(nb, T):
        per = ((T + 15) // 16) * 8
        return per * (nb * per + 4096) < (1 << 32)
    for T in (1001, 4001, 20001, 65536, 65537, 100001):
        largest = 1
        while accepted(largest + 1, T):
            largest += 1
        for want in (1 << 20, 37, 5):
            cap = engine.clamp_micro_batch(want, T)
            assert accepted(cap, T), (T, want)
            # the activation-workspace cap or the 32-bit limit, whichever is lower (then whole waves of 37 clips)
            expect = min(want, engine.DEFAULT_MICRO_BATCH * 1001 // T, largest)
            if 37 <= expect < want:
                expect -= expect % 37
            assert cap == max(1, expect), (T, want, cap)
    assert engine.clamp_micro_batch(1 << 20, 65536) == 3          # the NB = 3 / NB = 4 boundary tested on the GPU
    assert accepted(3, 65536) and not accepted(4, 65536)


BLOCK1_PATHS = ["fused", "two_kernel"]


def run_block1(x, w1s, shift1, w2_16, scale2, shift2, path, code, td, out=None):
    """conv_block1 through `path`: "fused" = sed_conv_block1, "two_kernel" = sed_conv_first_f32 (bn1 scale 1, as w1s
    carries it) writing a1, then sed_conv3x3_bn_relu 64 -> 64 with the pooling epilogue."""
    NB, H, W = x.shape
    n = NB * (H // 2) * (W // 2) * 64
    if out is None:
        out = torch.full((n + GUARD,), float("nan"), dtype=td, device=DEV)
    wp = w2_16.permute(0, 2, 3, 1).reshape(64, 576).contiguous()
    if path == "fused":
        call("sed_conv_block1", capi.ptr(x), NB, H, W, capi.ptr(w1s), capi.ptr(shift1), capi.ptr(wp), capi.ptr(scale2),
             capi.ptr(shift2), capi.ptr(out), code, stream())
    else:
        a1 = torch.empty((NB, H, W, 64), dtype=td, device=DEV)
        ones = torch.ones(64, device=DEV)
        call("sed_conv_first_f32", capi.ptr(x), NB, H, W, capi.ptr(w1s), capi.ptr(ones), capi.ptr(shift1), capi.ptr(a1),
             code, stream())
        call("sed_conv3x3_bn_relu", capi.ptr(a1), NB, H, W, 64, capi.ptr(wp), capi.ptr(scale2), capi.ptr(shift2), 64,
             capi.CONV_POOL, capi.ptr(out), None, 0, 0, code, stream())
    torch.cuda.synchronize()
    assert torch.isnan(out[n:n + GUARD].float()).all(), "conv_block1 wrote past its output"
    return out[:n].view(NB, H // 2, W // 2, 64)


# Measured on a B200 at 1000 W: the pooled 16-bit a1 equals the float64 rounding on 99.98 % (fp16) / 100 % (bf16) of the
# outputs on both block-1 paths, at most 2 ulps off; a conv1 from the fp16 hi parts alone misses 33 % (fp16) / 6.2 % (bf16),
# 1400-6900 times as often as the kernels.
PROBE_MIN_EXACT = 0.999
PROBE_PLAIN_RATIO = 100.0


@gpu
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
@pytest.mark.parametrize("path", BLOCK1_PATHS)
def test_conv_block1_conv1_precision_probe(path, dt):
    """w2 = identity at the centre tap: p1 is the pooled, rounded a1.  conv1 runs as split 16-bit products
    (hi*hi + lo*hi + hi*lo on the tensor cores, the operands are fp16 whatever the output type), so a1 must round like
    the float64 value nearly everywhere.  Where one a1 of a window rounds the other
    way the window mean moves by a quarter of that a1's ulp: up to two output ulps when that pixel dominates the window.
    A conv1 computed from the fp16 hi parts alone (what a dropped lo term gives) misses far more often."""
    code, td = DTYPES[dt]
    x, w1s, shift1, w2, scale2, shift2 = block1_inputs(3, 37, 11, DEV, probe=True)
    got = run_block1(x, w1s, shift1, w2.to(td), scale2, shift2, path, code, td)
    want = block1_ref(x, w1s, shift1, w2, scale2, shift2, td)[0].to(td)
    d = ulp_distance(got, want)
    exact = (d == 0).double().mean().item()
    h = torch.float16  # the kernel's split type
    plain = block1_ref(x.to(h).float(), w1s.to(h).float(), shift1.to(h).float(), w2, scale2, shift2, td)[0].to(td)
    plain_miss = (ulp_distance(plain, want) != 0).double().mean().item()
    report("conv_block1 probe %s %s" % (path, dt), exact=exact, max_ulp=int(d.max()),
           plain16_miss=plain_miss, miss_ratio=plain_miss / max(1.0 - exact, 1e-9))
    assert int(d.max()) <= 2
    assert exact >= PROBE_MIN_EXACT
    assert plain_miss >= PROBE_PLAIN_RATIO * (1.0 - exact)


# |p1 - ref| <= 0.5 ulp(ref) + BLOCK1_REL[dt] * m: output rounding plus the float32 accumulation over K = 576 and the
# few a1 values whose 16-bit rounding falls on the other side of a tie (one a1 ulp each, 2^-11 / 2^-8 of that term).
# Measured max 1.3e-5 (fp16) / 6.0e-5 (bf16); a padding pixel at relu(shift1) gives O(1).
BLOCK1_REL = {"fp16": 2.0 ** -14, "bf16": 2.0 ** -12}
# With W % 16 == 0 the tile count NB * ceil(H / 16) * W / 8 is always even: every work item of a CTA pair holds two
# tiles.  What varies is the number of items per pair (one each for small NB, several waves for 37 x 37) and whether
# the kernel's two conv1 producer groups, which take alternate items, get equally many.
BLOCK1_SHAPES = [(1, 1), (1, 2), (2, 15), (3, 16), (1, 17), (37, 37), (2, 1001), (3, 501)]


@gpu
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
@pytest.mark.parametrize("path", BLOCK1_PATHS)
@pytest.mark.parametrize("NB,H", BLOCK1_SHAPES, ids=["%dx%d" % s for s in BLOCK1_SHAPES])
def test_conv_block1_matches_float64(NB, H, path, dt):
    """Random conv2 weights, ragged heights (1 row: no output; odd H floors; a partial last 16-row tile), 1-37 images
    (37 x 37 = 444 work items: six waves of the 74 CTA pairs).  A padding pixel computed as relu(shift1) shows at the
    first / last rows and columns."""
    code, td = DTYPES[dt]
    x, w1s, shift1, w2, scale2, shift2 = block1_inputs(NB, H, 100 * NB + H, DEV)
    w2 = w2.to(td)
    got = run_block1(x, w1s, shift1, w2, scale2, shift2, path, code, td).double()
    want, m = block1_ref(x, w1s, shift1, w2, scale2, shift2, td)
    if got.numel() == 0:
        return
    excess = ((got - want).abs() - 0.5 * ulp16(want, td)).clamp(min=0) / m.clamp(min=1e-30)
    edge = torch.zeros_like(got, dtype=torch.bool)
    edge[:, 0] = edge[:, -1] = True
    edge[:, :, 0] = edge[:, :, -1] = True
    report("conv_block1 %dx%d %s %s" % (NB, H, path, dt), rel=excess.max().item(),
           rel_edge=excess[edge].max().item(), max_abs=(got - want).abs().max().item())
    assert excess.max().item() <= BLOCK1_REL[dt]


@gpu
@pytest.mark.parametrize("path", BLOCK1_PATHS)
def test_conv_block1_tile_index_limit(path):
    """NB = 3, H = 65 536 (4096 tiles of 16 rows per image) is the largest launch the 32-bit index arithmetic takes:
    correct in row slices around the image and tile boundaries of every image; NB = 4 is refused before launching."""
    code, td = DTYPES["fp16"]
    H, W = 65536, 64
    x4, w1s, shift1, w2, scale2, shift2 = block1_inputs(4, H, 7, DEV)
    w2 = w2.to(td)
    out = torch.full((4 * (H // 2) * (W // 2) * 64 + GUARD,), float("nan"), dtype=td, device=DEV)
    x = x4[:3]
    got = run_block1(x, w1s, shift1, w2, scale2, shift2, path, code, td, out=out)
    worst = 0.0
    for n in range(3):
        for r0 in (0, H // 4 - 6, H // 2 - 12):
            want, m = block1_ref(x[n:n + 1], w1s, shift1, w2, scale2, shift2, td, r0, r0 + 12)
            g_ = got[n:n + 1, r0:r0 + 12].double()
            excess = ((g_ - want).abs() - 0.5 * ulp16(want, td)).clamp(min=0) / m.clamp(min=1e-30)
            worst = max(worst, excess.max().item())
    report("conv_block1 3x65536 %s" % path, rel=worst)
    assert worst <= BLOCK1_REL["fp16"]
    wp = w2.permute(0, 2, 3, 1).reshape(64, 576).contiguous()
    lib = capi.load()
    if path == "fused":
        rc = lib.sed_conv_block1(capi.ptr(x4), 4, H, W, capi.ptr(w1s), capi.ptr(shift1), capi.ptr(wp), capi.ptr(scale2),
                                 capi.ptr(shift2), capi.ptr(out), code, stream())
    else:  # conv1_2 is where the two-kernel path divides tile indices (its input is any 16-bit buffer: not read)
        rc = lib.sed_conv3x3_bn_relu(capi.ptr(out), 4, H, W, 64, capi.ptr(wp), capi.ptr(scale2), capi.ptr(shift2), 64,
                                     capi.CONV_POOL, capi.ptr(out), None, 0, 0, code, stream())
    assert capi.ERR_NAMES.get(rc) == "SED_ERR_BAD_SHAPE"
    assert engine.clamp_micro_batch(1 << 20, H) == 3


# ------------------------------------------------------------------------------------------------ freq-mean epilogue
def freqmean_ref(x16, w16, scale, shift):
    """relu(bn(conv3x3(x))) averaged over the 8 frequency columns, float64 (im2col + matmul): [H, NB, cout] and the
    magnitude of the same sum over |terms|."""
    NB, H, W, cin = x16.shape
    cols = F.unfold(x16.permute(0, 3, 1, 2).double(), 3, padding=1)          # [NB, 9 cin, H W]
    outs = []
    for c_, w_, s_, b_ in ((cols, w16, scale, shift), (cols.abs(), w16.abs(), scale.abs(), shift.abs())):
        y = w_.double().reshape(w_.shape[0], -1) @ c_                        # [NB, cout, H W]
        y = torch.relu(y * s_.double()[:, None] + b_.double()[:, None])
        outs.append(y.view(NB, -1, H, W).mean(dim=3).permute(2, 0, 1))
    return outs[0], outs[1]


def test_freqmean_reference_is_the_conv():
    g = torch.Generator().manual_seed(4)
    x = torch.randn(2, 5, 8, 64, generator=g, dtype=F64)
    w = torch.randn(32, 64, 3, 3, generator=g, dtype=F64)
    s, b = torch.rand(32, generator=g, dtype=F64), torch.randn(32, generator=g, dtype=F64)
    y = torch.relu(F.conv2d(x.permute(0, 3, 1, 2), w, padding=1) * s[:, None, None] + b[:, None, None])
    got, _ = freqmean_ref(x, w, s, b)
    assert (got - y.mean(dim=3).permute(2, 0, 1)).abs().max().item() < 1e-10


FM_CASES = [(b0, NB, H) for b0, NB in ((0, 3), (37, 5), (296, 3)) for H in (1, 62, 125)] + [(296, 88, 1)]
FREQMEAN_REL = 2.0 ** -19  # float32 accumulation over K = 4608, relative to the sum of |terms| (measured 4.6e-7)


@gpu
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
@pytest.mark.parametrize("b0,NB,H", FM_CASES, ids=["b%d_n%d_h%d" % c for c in FM_CASES])
def test_freqmean_epilogue_writes_time_major_rows(b0, NB, H, dt):
    """conv_block4.conv2 as the models with a temporal block run it: features of clip n, step h go to row
    h * Bp + b0 + n of a [T', Bp, 512] buffer (out_sn = 1, out_sh = Bp), optionally with a float32 copy."""
    code, td = DTYPES[dt]
    Bp = 384
    g = torch.Generator(device=DEV).manual_seed(1000 * b0 + H)
    x = (torch.relu(torch.randn(NB, H, 8, 512, generator=g, device=DEV)) * 0.5).to(td)
    w = (torch.randn(512, 512, 3, 3, generator=g, device=DEV) / 68).to(td)
    scale = torch.rand(512, generator=g, device=DEV) + 0.5
    shift = torch.randn(512, generator=g, device=DEV) * 0.1
    wp = w.permute(0, 2, 3, 1).reshape(512, 9 * 512).contiguous()
    want, m = freqmean_ref(x, w, scale, shift)
    inside = torch.zeros(Bp, dtype=torch.bool, device=DEV)
    inside[b0:b0 + NB] = True
    res = []
    for with_f32 in (False, True):
        o16 = torch.full((H, Bp, 512), float("nan"), dtype=td, device=DEV)
        o32 = torch.full((H, Bp, 512), float("nan"), device=DEV) if with_f32 else None
        call("sed_conv3x3_bn_relu", capi.ptr(x), NB, H, 8, 512, capi.ptr(wp), capi.ptr(scale), capi.ptr(shift), 512,
             capi.CONV_FREQMEAN, capi.ptr(o16[0, b0:]), capi.ptr(None if o32 is None else o32[0, b0:]), 1, Bp, code,
             stream())
        torch.cuda.synchronize()
        assert torch.isnan(o16[:, ~inside].float()).all(), "rows outside [b0, b0 + NB) were written"
        got16 = o16[:, inside]
        err16 = ((got16.double() - want).abs() - 0.5 * ulp16(want, td)).clamp(min=0) / m.clamp(min=1e-30)
        res.append(got16)
        if with_f32:
            assert torch.isnan(o32[:, ~inside]).all()
            got32 = o32[:, inside]
            err32 = (got32.double() - want).abs() / m.clamp(min=1e-30)
            report("freq-mean b0=%d NB=%d H=%d %s" % (b0, NB, H, dt), rel32=err32.max().item(),
                   rel16_beyond_half_ulp=err16.max().item())
            assert err32.max().item() <= FREQMEAN_REL
            assert torch.equal(got32.to(td), got16)  # one rounding apart
        assert err16.max().item() <= FREQMEAN_REL, err16.max().item()
    assert torch.equal(res[0], res[1])


# ------------------------------------------------------------------------------------------------ GEMMs
def sample_rows(M, g):
    """The first and last two 128-row tiles and one random row of every tile."""
    tiles = (M + 127) // 128
    rnd = torch.arange(tiles, device=DEV) * 128 + torch.randint(0, 128, (tiles,), generator=g, device=DEV)
    idx = torch.cat([torch.arange(min(256, M), device=DEV), torch.arange(max(0, M - 256), M, device=DEV),
                     rnd[rnd < M]])
    return torch.unique(idx)


def linear_ref(a, w, bias, rows, relu):
    ar = a[rows].double()
    ref = ar @ w.double().t() + bias.double()
    mag = ar.abs() @ w.double().abs().t() + bias.double().abs()
    return (torch.relu(ref) if relu else ref), mag


def gemm_operands(M, N, td, seed, wscale=None):
    g = torch.Generator(device=DEV).manual_seed(seed)
    a = (torch.randn(M, 512, generator=g, device=DEV) * 0.5).to(td)
    w = (torch.randn(N, 512, generator=g, device=DEV) * (wscale or 512 ** -0.5)).to(td)
    bias = torch.randn(N, generator=g, device=DEV)
    return a, w, bias, g


LINEAR_REL = 2.0 ** -19  # float32 accumulation over K = 512 of exact 16-bit products, relative to sum |a w| + |b|
# (measured 4.0e-7; a column panel with the first panel's bias is off by O(1))
# (M, N, relu, outputs, dtype, out_layout): M = 37 888 is the two-row-tiles threshold, 48 000 = 375 tiles (odd),
# 128 000 = a 1024-clip batch of 10 s clips; M % 128 != 0 only in the row-major layout; N = 2048 runs two column panels
LINEAR_CASES = [
    (37888, 1536, 0, "f32", "fp16", 0), (37888, 512, 1, "both", "bf16", 0), (37889, 1536, 0, "both", "fp16", 0),
    (37889, 2048, 1, "f16", "bf16", 0), (48000, 1536, 0, "f32", "fp16", 0), (48000, 2048, 1, "both", "fp16", 0),
    (48000, 512, 0, "f16", "bf16", 0), (47995, 2048, 0, "f32", "bf16", 0), (47995, 512, 1, "f16", "fp16", 0),
    (128000, 2048, 0, "both", "bf16", 0), (128000, 1536, 1, "f16", "fp16", 0), (128000, 512, 1, "f32", "bf16", 0),
    (48000, 1536, 0, "f32", "fp16", 1), (48000, 2048, 1, "f32", "bf16", 1), (128000, 1536, 0, "f32", "fp16", 1),
    (128000, 2048, 0, "f32", "bf16", 1),
]


@gpu
@pytest.mark.parametrize("M,N,relu,outs,dt,layout", LINEAR_CASES, ids=["-".join(map(str, c)) for c in LINEAR_CASES])
def test_linear_at_production_row_counts(M, N, relu, outs, dt, layout):
    code, td = DTYPES[dt]
    a, w, bias, g = gemm_operands(M, N, td, M + N + relu)
    pad = 0 if layout else 128
    o32 = torch.full(((M + pad) * N + (GUARD if layout else 0),), float("nan"), device=DEV) if outs != "f16" else None
    o16 = torch.full(((M + pad) * N,), float("nan"), dtype=td, device=DEV) if outs != "f32" else None
    call("sed_linear", capi.ptr(a), M, 512, capi.ptr(w), capi.ptr(bias), N, relu, capi.ptr(o32), capi.ptr(o16),
         layout, code, stream())
    torch.cuda.synchronize()
    rows = sample_rows(M, g)
    want, mag = linear_ref(a, w, bias, rows, relu)
    vals, same16 = {}, True
    if o32 is not None:
        assert torch.isnan(o32[M * N:]).all(), "sed_linear wrote past row M"
        got = o32[:M * N].view(M // 128, N // 4, 128, 4).permute(0, 2, 1, 3).reshape(M, N) if layout else \
            o32[:M * N].view(M, N)
        vals["rel32"] = ((got[rows].double() - want).abs() / mag).max().item()
    if o16 is not None:
        assert torch.isnan(o16[M * N:].float()).all(), "sed_linear wrote past row M"
        got16 = o16[:M * N].view(M, N)
        err = ((got16[rows].double() - want).abs() - 0.5 * ulp16(want, td)).clamp(min=0) / mag
        vals["rel16_beyond_half_ulp"] = err.max().item()
        if o32 is not None:
            same16 = torch.equal(o32[:M * N].view(M, N).to(td), got16)  # every row: the 16-bit copy is the rounded f32
    report("sed_linear M=%d N=%d relu=%d %s %s layout %d" % (M, N, relu, outs, dt, layout), **vals)
    assert max(vals.values()) <= LINEAR_REL
    assert same16


@gpu
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
@pytest.mark.parametrize("M", [48000, 128000])
def test_linear_split16_at_production_row_counts(M, dt):
    """The QKV projection of 384 / 1024 clips x 125 steps: hi + lo is the float64 projection to ~2^-21 (fp16)."""
    code, td = DTYPES[dt]
    a, w, bias, g = gemm_operands(M, 1536, td, M + 1, wscale=0.2)
    hi = torch.full(((M + 128) * 1536,), float("nan"), dtype=td, device=DEV)
    lo = torch.full(((M + 128) * 1024,), float("nan"), dtype=td, device=DEV)
    call("sed_linear_split16", capi.ptr(a), M, 512, capi.ptr(w), capi.ptr(bias), 1536, capi.ptr(hi), capi.ptr(lo),
         1024, code, stream())
    torch.cuda.synchronize()
    assert torch.isnan(hi[M * 1536:].float()).all() and torch.isnan(lo[M * 1024:].float()).all()
    rows = sample_rows(M, g)
    want, mag = linear_ref(a, w, bias, rows, False)
    h = hi[:M * 1536].view(M, 1536)[rows].double()
    both = h[:, :1024] + lo[:M * 1024].view(M, 1024)[rows].double()
    scale = want.abs().max().item()
    err_hi = (h - want).abs().max().item() / scale
    err_both = (both - want[:, :1024]).abs().max().item() / scale
    report("sed_linear_split16 M=%d %s" % (M, dt), hi=err_hi, hi_plus_lo=err_both)
    # measured: hi + lo 9.1e-7 (fp16) / 5.4e-6 (bf16), hi alone 3.2e-4 / 2.6e-3
    assert err_both <= (2e-6 if dt == "fp16" else 2e-5)
    assert err_both * 100 < err_hi


# 16-bit operands of the projections and of h W_hh^T; measured 4.0e-4 / 2.9e-3 (GRU), 5.0e-4 / 3.8e-3 (MultiHead)
TEMPORAL_TOL = {("gru", "fp16"): 1.5e-3, ("gru", "bf16"): 1.2e-2, ("mha", "fp16"): 2e-3, ("mha", "bf16"): 1.6e-2}


@gpu
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
@pytest.mark.parametrize("kind", ["gru", "mha"])
def test_temporal_block_at_batch_300(kind, dt):
    """B = 300 clips x T' = 125 steps: the input projection (48 000 rows, an odd 375 tiles) with two row tiles per work
    item, three 128-clip GRU blocks with a partial last one, the split QKV projection of the attention path."""
    mt = "Cnn_9layers_Gru_FrameAtt" if kind == "gru" else "Cnn_9layers_Transformer_FrameAtt"
    sd = synthetic_sd(mt)
    pm = engine.PackedModel(sd, mt, 512, 160, DEV, precision=dt)
    td = DTYPES[dt][1]
    x = torch.relu(torch.randn(300, 125, 512, generator=torch.Generator().manual_seed(300)) * 0.5).to(td)
    got = pm.temporal(x.to(DEV)).double()
    sd64 = {k: v.double().to(DEV) for k, v in sd.items()}
    ref = (so.bigru if kind == "gru" else so.multihead)(x.to(DEV).double(), sd64)
    err = (got - ref).abs().max().item()
    bound = TEMPORAL_TOL[(kind, dt)] * (1.0 if kind == "gru" else max(1.0, ref.abs().max().item()))
    report("%s 300x125 %s" % (kind, dt), max_abs=err, bound=bound)
    assert err <= bound


# ------------------------------------------------------------------------------------------------ pooling heads
def to_blocks(x, garbage):
    """[B, T, 512] rows -> the 128-clip transposed blocks [T, nblk, 128, 128, 4] (engine.blocks_to_rows is the
    inverse); the padding clips of the last block hold `garbage`."""
    B, T, C = x.shape
    Bp = (B + 127) // 128 * 128
    xp = torch.full((Bp, T, C), garbage, dtype=x.dtype, device=x.device)
    xp[:B] = x
    return xp.view(Bp // 128, 128, T, C // 4, 4).permute(2, 0, 3, 1, 4).contiguous()


def test_block_layout_round_trip():
    x = torch.randn(130, 3, 512)
    xb = to_blocks(x, float("nan"))
    assert xb.shape == (3, 2, 128, 128, 4)
    assert torch.equal(engine.blocks_to_rows(xb, 130, 3), x)
    assert torch.isnan(engine.blocks_to_rows(xb, 256, 3)[130:]).all()


def att_ref(x, sd, frames_out):
    """sigmoid / attention head in float64: so.att_block + interpolate (x8) + pad_framewise_output."""
    sd64 = {k: v.double().to(x.device) for k, v in sd.items() if k.startswith("att_block")}
    clip, natt, cla = so.att_block(x.double().transpose(1, 2), sd64)
    fw = so.interpolate(cla.transpose(1, 2), 8)
    if fw.shape[1] != frames_out:
        fw = so.pad_framewise_output(fw, frames_out)
    return clip, fw, cla, natt


ATT_ABS = 5e-6  # float32 projections and sums over T' of probabilities; measured 1.4e-6
ATT_CASES = [(B, T, f) for B in (1, 130, 300) for T in (1, 62, 125, 750)
             for f in sorted({8 * T, so.roundup(8 * T)})]


@gpu
@pytest.mark.parametrize("B,T,frames", ATT_CASES, ids=["b%d_t%d_f%d" % c for c in ATT_CASES])
def test_attpool_blocks_matches_float64_and_stages(B, T, frames):
    """sed_attpool_blocks on the GRU / Transformer output layout; stage 1 + stage 2 over uneven clip ranges (the split
    forward_host runs) gives the stage-0 result bit for bit and writes only the clips of each range."""
    sd = synthetic_sd("Cnn_9layers_Gru_FrameAtt")
    x = torch.tanh(torch.randn(B, T, 512, generator=torch.Generator().manual_seed(B * 7 + T)) * 1.5).to(DEV)
    xb = to_blocks(x, float("nan"))
    wa, wc = (sd["att_block.%s.weight" % k].float().reshape(25, 512).contiguous().to(DEV) for k in ("att", "cla"))
    ba, bc = (sd["att_block.%s.bias" % k].float().to(DEV) for k in ("att", "cla"))
    scratch = torch.empty((capi.load().sed_attpool_blocks_scratch_bytes(B, T),), dtype=torch.uint8, device=DEV)

    def fresh():
        return [torch.full(s, float("nan"), device=DEV) for s in ((B, 25), (B, frames, 25), (B, 25, T), (B, 25, T))]

    def launch(outs, stage, c0, n):
        call("sed_attpool_blocks", capi.ptr(xb), B, T, capi.ptr(wa), capi.ptr(ba), capi.ptr(wc), capi.ptr(bc), 8,
             frames, capi.ptr(scratch), *[capi.ptr(o) for o in outs], stage, c0, n, stream())

    one = fresh()
    launch(one, 0, 0, B)
    torch.cuda.synchronize()
    want = att_ref(x, sd, frames)
    errs = [(g_.double() - w_).abs().max().item() for g_, w_ in zip(one, want)]
    report("attpool_blocks B=%d T=%d frames=%d" % (B, T, frames), clip=errs[0], frame=errs[1], cla=errs[2],
           norm_att=errs[3])
    assert max(errs) <= ATT_ABS
    staged = fresh()
    launch(staged, 1, 0, 0)
    cuts = [c for c in (0, 37, 130, 300) if c < B] + [B]
    for c0, c1 in zip(cuts[:-1], cuts[1:]):
        launch(staged, 2, c0, c1 - c0)
        torch.cuda.synchronize()
        for o in staged:
            assert torch.isnan(o[c1:]).all(), "stage 2 of clips [%d, %d) wrote clips >= %d" % (c0, c1, c1)
    for a, b in zip(one, staged):
        assert torch.equal(a, b)


FC_ABS = 4e-6  # float32 dot products of 512 terms and the mean over T'; measured 1.2e-6


@gpu
@pytest.mark.parametrize("T", [1, 17, 125, 750])
@pytest.mark.parametrize("C", [1, 10, 25, 32])
def test_fcpool_matches_float64(C, T):
    """FrameAvg / FrameMax head: sigmoid(fc(x)) per step, x8 repeat, clipwise mean / max; with the frame output offset
    by one float the kernel takes its scalar store branch and must give the same values."""
    B = 3
    g = torch.Generator(device=DEV).manual_seed(C * 1000 + T)
    x = torch.randn(B, T, 512, generator=g, device=DEV)
    w = torch.randn(C, 512, generator=g, device=DEV) * 0.1
    b = torch.randn(C, generator=g, device=DEV)
    p = torch.sigmoid(x.double() @ w.double().t() + b.double())                    # [B, T, C]
    want_frame = p.repeat_interleave(8, dim=1)
    n = B * T * 8 * C
    for use_max in (0, 1):
        want_clip = p.amax(dim=1) if use_max else p.mean(dim=1)
        frames = []
        for off in (0, 1):
            clip = torch.full((B, C), float("nan"), device=DEV)
            frame = torch.full((n + off + GUARD,), float("nan"), device=DEV)
            call("sed_fcpool", capi.ptr(x), B, T, capi.ptr(w), capi.ptr(b), C, 8, use_max, capi.ptr(clip),
                 capi.ptr(frame[off:]), stream())
            torch.cuda.synchronize()
            assert torch.isnan(frame[:off]).all() and torch.isnan(frame[off + n:]).all()
            got = frame[off:off + n].view(B, T * 8, C)
            e_f = (got.double() - want_frame).abs().max().item()
            e_c = (clip.double() - want_clip).abs().max().item()
            report("fcpool C=%d T=%d max=%d offset %d" % (C, T, use_max, off), frame=e_f, clip=e_c)
            assert e_f <= FC_ABS and e_c <= FC_ABS
            frames.append(got)
        assert torch.equal(frames[0], frames[1])


@gpu
def test_fcpool_rejects_more_than_32_classes():
    x = torch.zeros(1, 4, 512, device=DEV)
    w = torch.zeros(33, 512, device=DEV)
    out = torch.zeros(33 * 32, device=DEV)
    with pytest.raises(ValueError, match="SED_ERR_BAD_SHAPE"):
        call("sed_fcpool", capi.ptr(x), 1, 4, capi.ptr(w), capi.ptr(out), 33, 8, 0, capi.ptr(out), capi.ptr(out),
             stream())
