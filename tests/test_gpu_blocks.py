"""Conv64F blocks 2-3 (csrc/conv3_tc.cu: 64 -> 64 channel 3x3 conv + folded BatchNorm + activation, optionally the
3x3/3 max-pool) against float64 at the batch sizes the benchmark runs, for the TF32 kernel and the separately stated
bf16 kernel.

* Exact arithmetic.  Activations k/4 (|k| <= 7), weights j/32 (|j| <= 7) and shifts m/128 (|m| <= 512) make every
  product a multiple of 2^-7 and every partial sum of the 576 products (plus the shift) a multiple of 2^-7 below 2^8:
  15 significant bits, exact in fp32, and every operand is exact in TF32 and in bf16.  Accumulation order, TF32
  truncation, the host's rounding of the weights and the bf16 operands then change nothing, and both kernels must equal
  the fp64 reference bit for bit: every tile geometry the host can pick, the 4 -> 3 accumulator fallback of the TF32
  kernel, slopes 0, 0.1, 0.2, 0.25 and 2, fp32 and bf16 outputs.  The input sits between two images' worth of sentinel
  pixels and the output is prefilled with NaN between two sentinel guards, so a read outside the input, a skipped
  output element or a write outside the output changes the result.
* Rounding.  Random data against fp64 of the operands as the MMA sees them, per element, in units of 2^-24 of
  maxpool3(conv(|x|, |w|)) + |shift|; the bf16 output is the fp32 output rounded to nearest even, bit for bit.
* Batch independence at the bench batch (3 200 clips, 108-109 tiles per CTA).

Both kernels run every case.  The bf16 kernel runs with two epilogue groups at every shape here, the bench shapes
included (_launch_plan; its one-group fallback needs W > 61, which the entry points reject).  The whole file takes
about 8 s on a B200."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U24 = 2.0 ** -24  # unit roundoff of fp32 (round to nearest)
NUM_SMS = 148     # persistent grid of conv3_tc: min(tiles, kNumSMs)
SENTINEL = 4096.0  # finite (the pooling's fmaxf would drop a NaN) and larger than any output of the exact cases
GUARD = 1024       # sentinel output elements before and after the output (4 KB of fp32: keeps the output 16-byte aligned)
SLOPES = (0.0, 0.1, 0.2, 0.25, 2.0)  # 0.1, 0.2: one fp32 rounding, the same in the kernel and the reference; 2.0: the
                                     # ternary a > 0 ? a : a * slope is LeakyReLU for slopes >= 1 as well

# Per-element bounds, |got - ref| <= C * 2^-24 * (maxpool3(conv(|xq|, |wq|)) + |shift|), xq and wq the operands as the
# MMA multiplies them.  First order, every rounding of the chain is at most 2^-24 of a value bounded by that absolute
# expression: the fp32 accumulator is updated once per MMA (9 taps x 64 / K channels), then the shift add and the slope
# multiply (slope < 1).  The accumulation inside the tensor core is not specified to round to nearest; a truncating
# accumulator doubles each update's error, and the bounds allow for it.
#   TF32 (K = 8): 72 updates + 2 = 74, doubled: 148.  Measured on a B200 (1000 W): at most 12.6 over the cases below.
#   Modelling the activations as rounded to nearest instead of truncated measured 2 513 to 4 190 (17-28 x C_TF32), so
#   the bound tells the two models apart; weights packed truncated instead of rounded measured 2 506 to 3 313.
C_TF32 = 148.0
#   bf16 (K = 16, products exact in fp32): 36 updates + 2 = 38, doubled: 76.  Measured on a B200 (1000 W): at most 5.4.
C_BF16 = 76.0


# ------------------------------------------------------------------------------------------------ geometry
def _conv3_geometry(H, W, pool, max_nm):
    """conv3_geometry: (accumulators NM, image rows of every tile of an image) or None when W does not fit a tile."""
    HP = W + 2
    rows = 3 * (H // 3) if pool else H  # rows below the last complete pooling window are never used
    R = min(max_nm * 128 // HP, rows)
    if pool:
        R -= R % 3
    if R < 1:
        return None
    return -(-R * HP // 128), tuple(min(R, rows - y0) for y0 in range(0, rows, R))


def _acc_tiles(W, geom):
    """conv3_acc_tiles: 128-row accumulator tiles (MMA work) per image."""
    return sum(-(-r * (W + 2) // 128) for r in geom[1])


def _smem_fits(bf16, W, geom, groups):
    """launch_conv3's shared-memory budget: weights, ring stages of the tile's padded pixels, staging tiles, shift."""
    nm, rows = geom
    HP = W + 2
    halo = (nm * 128 + 2 * HP + 2 + 7) & ~7
    ring = (5 if nm == 4 else 6) if bf16 else (3 if nm == 4 else 4)
    stage_pos = (rows[0] * HP + 7) & ~7
    smem = (73728 if bf16 else 147456) + ring * halo * 32 + groups * stage_pos * 12 * 4 + 64 * 4 + 256
    return smem + 256 <= 232448


def _launch_plan(N, H, W, pool, bf16):
    """What afs_conv3x3_c64_bn_act_fwd_{tf32,bf16} launch: conv3_best_geometry (three or four accumulators, whichever
    needs fewer MMAs), then the largest configuration whose shared memory fits -- the bf16 kernel tries two epilogue
    groups, then one; both fall back from four accumulators to three."""
    g3, g4 = _conv3_geometry(H, W, pool, 3), _conv3_geometry(H, W, pool, 4)
    if g3 is None:
        return None
    best = g4 if g4[0] == 4 and _acc_tiles(W, g4) < _acc_tiles(W, g3) else g3
    for geom in (best, g3) if best is g4 else (best,):
        for groups in (2, 1) if bf16 else (1,):
            if _smem_fits(bf16, W, geom, groups):
                tiles = N * len(geom[1])
                ctas = min(tiles, NUM_SMS)
                return dict(nm=geom[0], rows=geom[1], groups=groups, fallback=geom is not best,
                            tiles_per_cta=(tiles // ctas, -(-tiles // ctas)))
    return None


def test_launch_plan_reaches_the_four_to_three_fallback_only_at_w54():
    """The restated host logic over every H <= 129, W <= 61: the TF32 kernel falls back from four accumulators to three
    at W = 54 only, and the bf16 kernel always fits four accumulators and two epilogue groups where it picks them."""
    fallback, one_group = set(), []
    for H in range(1, 130):
        for W in range(1, 62):
            for pool in (False, True) if H >= 3 and W >= 3 else (False,):
                for bf16 in (False, True):
                    plan = _launch_plan(1, H, W, pool, bf16)
                    if plan is None:
                        continue
                    if plan["fallback"]:
                        fallback.add((bf16, W))
                    if plan["groups"] != 2 and bf16:
                        one_group.append((H, W, pool))
    assert fallback == {(False, 54)}
    assert one_group == []


# ------------------------------------------------------------------------------------------------ launches
def _guarded_input(x_nhwc):
    """x [N, H, W, 64] -> a channels-last [N, 64, H, W] view into a buffer that holds one image of SENTINEL pixels on
    each side of it (ops passes such a view to the kernel without a copy)."""
    N, H, W, C = x_nhwc.shape
    pad = H * W * C
    buf = torch.full((2 * pad + x_nhwc.numel(),), SENTINEL, dtype=x_nhwc.dtype, device=x_nhwc.device)
    buf[pad:pad + x_nhwc.numel()].copy_(x_nhwc.reshape(-1))
    return buf.as_strided((N, C, H, W), (H * W * C, 1, W * C, C), pad)


def _run(x, w_packed, shift, slope, pool, out_dtype=torch.float32):
    """One launch through the C ABI: x fp32 -> the TF32 kernel, x bf16 -> the bf16 kernel.  The output is a NaN-filled
    slice of a buffer with GUARD sentinel elements on both sides; the guards must come back unchanged.  Returns the
    output as a channels-last [N, 64, OH, OW] view."""
    from audio_fewshot_b200 import _lib
    assert x.is_contiguous(memory_format=torch.channels_last)
    N, C, H, W = x.shape
    OH, OW = (H // 3, W // 3) if pool else (H, W)
    n = N * OH * OW * C
    buf = torch.full((GUARD + n + GUARD,), SENTINEL, dtype=out_dtype, device=x.device)
    buf[GUARD:GUARD + n] = float("nan")
    out_ptr = buf.data_ptr() + GUARD * buf.element_size()
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    h = _lib.lib()
    if x.dtype == torch.float32:
        assert out_dtype == torch.float32
        rc = h.afs_conv3x3_c64_bn_act_fwd_tf32(x.data_ptr(), N, H, W, w_packed.data_ptr(), shift.data_ptr(), float(slope),
                                               int(pool), out_ptr, stream)
    else:
        rc = h.afs_conv3x3_c64_bn_act_fwd_bf16(x.data_ptr(), N, H, W, w_packed.data_ptr(), shift.data_ptr(), float(slope),
                                               int(pool), out_ptr, int(out_dtype == torch.bfloat16), stream)
    _lib.check(rc, "afs_conv3x3_c64_bn_act_fwd")
    guards = torch.cat([buf[:GUARD], buf[GUARD + n:]])
    assert torch.equal(guards, torch.full_like(guards, SENTINEL)), "write outside the output"
    return buf[GUARD:GUARD + n].view(N, OH, OW, C).permute(0, 3, 1, 2)


def _packed(cuda, w):
    from audio_fewshot_b200 import ops
    tf32 = torch.from_numpy(ops.conv3x3_c64_pack_weights(w)).to(cuda)
    bf16 = torch.from_numpy(ops.conv3x3_c64_pack_weights_bf16(w)).to(cuda).view(torch.bfloat16)
    return tf32, bf16


def _assert_equal(got, want, what):
    if torch.equal(got, want):
        return
    diff = (got.float() != want.float()) | got.float().isnan()
    idx = diff.nonzero()[0].tolist()
    raise AssertionError("%s: %d of %d elements differ (%d NaN, i.e. never written), first at %s: %r vs %r"
                         % (what, int(diff.sum()), diff.numel(), int(got.float().isnan().sum()), idx,
                            got[tuple(idx)].item(), want[tuple(idx)].item()))


def _clip_chunks(N, H, W):
    """Slices of clips whose [n, 64, H, W] float64 tensors stay near 128 MB."""
    step = max(1, (1 << 24) // (64 * H * W))
    return [slice(i, min(N, i + step)) for i in range(0, N, step)]


# ------------------------------------------------------------------------------------------------ exact arithmetic
def _grid_operands(cuda, N, H, W, kind, seed):
    """Activations k/4 as [N, H, W, 64] fp32: "signed" k in [-7, 7]; "relu" k in [1, 7] with 40 % zeros (block 2's
    input is block 1 after ReLU and pooling).  Weights j/32, j in [-7, 7], with an all-zero row; shifts m/128, |m| <= 512."""
    g = torch.Generator(device=cuda).manual_seed(seed)
    shape = (N, H, W, 64)
    if kind == "signed":
        k = torch.randint(-7, 8, shape, generator=g, device=cuda, dtype=torch.int8)
    else:
        k = torch.randint(1, 8, shape, generator=g, device=cuda, dtype=torch.int8)
        k.masked_fill_(torch.rand(shape, generator=g, device=cuda) < 0.4, 0)
    x = k.float().mul_(0.25)
    del k
    w = torch.randint(-7, 8, (64, 64, 3, 3), generator=g, device=cuda).float() / 32
    w[7] = 0.0
    shift = torch.randint(-512, 513, (64,), generator=g, device=cuda).float() / 128
    return x, w, shift


EXACT_CASES = [
    # N, H, W, pool; TF32 kernel: NM, image rows of each tile of an image, tiles per CTA; the bf16 kernel where it differs
    pytest.param(3200, 42, 52, True, (4, (9, 9, 9, 9, 6), (108, 109)), None, id="3200x42x52-pool"),
    # bench block 2: 16 000 tiles, 16 CTAs run a 109th; the last tile of an image leaves accumulator 3 idle
    pytest.param(3200, 14, 17, True, (2, (12,), (21, 22)), None, id="3200x14x17-pool"),
    # bench block 3: rows 12-13 only feed the conv
    pytest.param(3200, 14, 17, False, (3, (14,), (21, 22)), None, id="3200x14x17"),
    # block 3 of the DN4 backbone (maxpool_last2=False)
    pytest.param(37, 42, 52, True, (4, (9, 9, 9, 9, 6), (1, 2)), None, id="37x42x52-pool"),
    # 185 tiles: 37 CTAs run a second tile, the first that uses the second accumulator set
    pytest.param(300, 18, 54, True, (3, (6, 6, 6), (6, 7)), (4, (9, 9), (4, 5)), id="300x18x54-pool"),
    # TF32: four accumulators do not fit shared memory, three do (900 tiles); bf16: four, two epilogue groups
    pytest.param(149, 19, 54, False, (3, (6, 6, 6, 1), (4, 5)), (4, (9, 9, 1), (3, 4)), id="149x19x54"),
    # TF32 after the fallback: the last tile reaches one accumulator of three; bf16: one of four
    pytest.param(64, 16, 61, True, (3, (6, 6, 3), (1, 2)), None, id="64x16x61-pool"),
    pytest.param(2, 10, 61, False, (3, (6, 4), (1, 1)), None, id="2x10x61"),
    # the widest supported row (HP = 63)
    pytest.param(1000, 20, 3, True, (1, (18,), (6, 7)), None, id="1000x20x3-pool"),
    # the narrowest pooled row (PW = 1)
    pytest.param(30, 17, 13, True, (2, (15,), (1, 1)), None, id="30x17x13-pool"),
    # H and W not multiples of 3
    pytest.param(500, 5, 7, True, (1, (3,), (3, 4)), None, id="500x5x7-pool"),
    # 500 one-tile images
    pytest.param(1, 3, 3, True, (1, (3,), (1, 1)), None, id="1x3x3-pool"),
    pytest.param(1, 1, 1, False, (1, (1,), (1, 1)), None, id="1x1x1"),
    # the smallest legal shapes: one tile on one CTA
]


@pytest.mark.parametrize("kind", ["signed", "relu"])
@pytest.mark.parametrize("N,H,W,pool,tf32_plan,bf16_plan", EXACT_CASES)
def test_conv3_is_exact_on_exactly_representable_operands(cuda, N, H, W, pool, tf32_plan, bf16_plan, kind):
    """On the exact grid both kernels equal the fp64 reference bit for bit at every slope: the TF32 kernel (fp32
    output), the bf16 kernel with fp32 output, and with bf16 output (the fp32 reference rounded to nearest even).  The
    reference applies the activation in fp32 as the kernel does, torch.where(v > 0, v, v * slope), then max_pool2d."""
    from audio_fewshot_b200 import ops
    for bf16, (nm, rows, per_cta) in ((False, tf32_plan), (True, bf16_plan or tf32_plan)):
        plan = _launch_plan(N, H, W, pool, bf16)
        assert (plan["nm"], plan["rows"], plan["tiles_per_cta"]) == (nm, rows, per_cta), (bf16, plan)
        assert plan["groups"] == (2 if bf16 else 1) and plan["fallback"] == (not bf16 and W == 54)
    x, w, shift = _grid_operands(cuda, N, H, W, kind, seed=N + 7 * H + W + (kind == "relu"))
    x32 = _guarded_input(x)
    x16 = _guarded_input(x.to(torch.bfloat16))
    del x
    w32, w16 = _packed(cuda, w)
    conv = torch.empty((N, 64, H, W), device=cuda)
    wd, sd = w.double(), shift.double()
    for c in _clip_chunks(N, H, W):
        conv[c] = F.conv2d(x32[c].double(), wd, sd, padding=1).float()  # exact: no rounding anywhere
    for slope in SLOPES:
        want = torch.where(conv > 0, conv, conv * slope)
        if pool:
            want = F.max_pool2d(want, 3, 3)
        got = _run(x32, w32, shift, slope, pool)
        _assert_equal(got, want, "TF32 kernel, slope %g" % slope)
        if slope == 0.0:  # the tensor-level wrapper launches on the same sentinel-guarded view without a copy
            _assert_equal(ops.conv3x3_c64_bn_act(x32, w32, shift, slope, pool=pool), want, "ops, TF32")
        _assert_equal(_run(x16, w16, shift, slope, pool), want, "bf16 kernel, fp32 output, slope %g" % slope)
        _assert_equal(_run(x16, w16, shift, slope, pool, torch.bfloat16), want.to(torch.bfloat16),
                      "bf16 kernel, bf16 output, slope %g" % slope)


# ------------------------------------------------------------------------------------------------ rounding
def _trunc_tf32(t):
    """What the MMA reads of an fp32 activation: the low 13 mantissa bits dropped."""
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def _rna_tf32(t):
    """cvt.rna.tf32.f32 (the host's rounding of the weights): to nearest, ties away from zero."""
    return ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def _random_operands(cuda, N, H, W, kind, seed):
    """randn activations as [N, H, W, 64] fp32: "signed", or "relu": |randn| with 40 % zeros.  Weights randn * 0.06
    (the scale of a folded Conv64F block) with a negated row (a negative BatchNorm scale) and an all-zero row."""
    g = torch.Generator(device=cuda).manual_seed(seed)
    x = torch.randn((N, H, W, 64), generator=g, device=cuda)
    if kind == "relu":
        x.abs_().masked_fill_(torch.rand(x.shape, generator=g, device=cuda) < 0.4, 0.0)
    w = torch.randn((64, 64, 3, 3), generator=g, device=cuda) * 0.06
    w[5] *= -1.0
    w[7] = 0.0
    shift = torch.randn(64, generator=g, device=cuda)
    return x, w, shift


def _worst_ratio(got, x, w, shift, slope, pool):
    """max over elements of |got - ref| / (2^-24 (maxpool3(conv(|x|, |w|)) + |shift|)), ref = fp64 conv2d(x, w) + shift
    -> leaky_relu -> max_pool2d, in chunks of clips."""
    N, _, H, W = x.shape
    wd, sd = w.double(), shift.double().view(1, -1, 1, 1)
    worst = 0.0
    for c in _clip_chunks(N, H, W):
        xc = x[c].double()
        ref = F.leaky_relu(F.conv2d(xc, wd, padding=1) + sd, slope)
        base = F.conv2d(xc.abs(), wd.abs(), padding=1)
        if pool:
            ref, base = F.max_pool2d(ref, 3, 3), F.max_pool2d(base, 3, 3)
        err = (got[c].double() - ref).abs() / ((base + sd.abs()) * U24)
        worst = max(worst, err.max().item())
    return worst


@pytest.mark.parametrize("kind", ["relu", "signed"])
@pytest.mark.parametrize("N,H,W,pool,slope", [
    pytest.param(200, 42, 52, True, 0.0, id="200x42x52-pool"),   # block 2: 1 000 tiles, 6-7 per CTA
    pytest.param(200, 14, 17, True, 0.2, id="200x14x17-pool"),   # block 3
    pytest.param(149, 19, 54, False, 0.1, id="149x19x54"),       # TF32: three accumulators after the fallback
    pytest.param(2, 10, 61, False, 0.2, id="2x10x61"),           # the widest row
])
def test_conv3_matches_fp64_of_the_operands_the_mma_multiplies(cuda, N, H, W, pool, slope, kind):
    """The TF32 kernel against fp64 of trunc_tf32(x) (the MMA ignores the low 13 bits of an fp32 activation) and
    rna_tf32(w) (computed here from w, not read back from the packed buffer): within C_TF32.  The same reference with
    activations rounded to nearest instead of truncated misses the bound by far.  The bf16 kernel against fp64 of the
    bf16 operands: within C_BF16; its bf16 output is its fp32 output rounded to nearest even, bit for bit.  The
    all-zero weight row gives activation(shift) bit for bit in both."""
    x, w, shift = _random_operands(cuda, N, H, W, kind, seed=3 * N + H + W + (kind == "relu"))
    x32 = _guarded_input(x)
    x16 = _guarded_input(x.to(torch.bfloat16))
    del x
    w32, w16 = _packed(cuda, w)
    want7 = torch.tensor(float(shift[7]), device=cuda)
    want7 = torch.where(want7 > 0, want7, want7 * slope)

    got = _run(x32, w32, shift, slope, pool)
    assert torch.equal(got[:, 7], want7.expand_as(got[:, 7]))
    xq, wq = _trunc_tf32(x32), _rna_tf32(w)
    worst = _worst_ratio(got, xq, wq, shift, slope, pool)
    teeth = _worst_ratio(got, _rna_tf32(x32), wq, shift, slope, pool)
    print("TF32 %dx%dx%d %s slope %g: worst error %.2f x 2^-24 x abs (bound %g); activations rounded to nearest: %.1f"
          % (N, H, W, kind, slope, worst, C_TF32, teeth))
    assert worst <= C_TF32
    assert teeth > 5 * C_TF32  # the case has teeth: measured 17-28 x C_TF32

    got16 = _run(x16, w16, shift, slope, pool)
    assert torch.equal(got16[:, 7], want7.expand_as(got16[:, 7]))
    worst16 = _worst_ratio(got16, x16.float(), w.to(torch.bfloat16).float(), shift, slope, pool)
    print("bf16 %dx%dx%d %s slope %g: worst error %.2f x 2^-24 x abs (bound %g)" % (N, H, W, kind, slope, worst16, C_BF16))
    assert worst16 <= C_BF16
    _assert_equal(_run(x16, w16, shift, slope, pool, torch.bfloat16), got16.to(torch.bfloat16), "bf16 output")


@pytest.mark.parametrize("bf16", [False, True], ids=["tf32", "bf16"])
def test_conv3_clip_is_independent_of_its_batch(cuda, bf16):
    """Bench block 2 on 3 200 random clips (16 000 tiles, 108-109 per CTA, the ring wrapping every tile): clips run on
    their own (one CTA, first tile, first ring stage) give the outputs they have inside the batch bit for bit.  The tile
    geometry does not depend on N, so this carries the fp64 bounds checked at 200 clips to the whole bench batch."""
    N, H, W = 3200, 42, 52
    x, w, shift = _random_operands(cuda, N, H, W, "relu", seed=41)
    dtype = torch.bfloat16 if bf16 else torch.float32
    x = _guarded_input(x.to(dtype))
    wp = _packed(cuda, w)[int(bf16)]
    full = _run(x, wp, shift, 0.0, True, dtype)
    for c in (slice(0, 1), slice(1601, 1700), slice(N - 37, N)):
        alone = _guarded_input(x[c].permute(0, 2, 3, 1))
        _assert_equal(_run(alone, wp, shift, 0.0, True, dtype), full[c], "clips %d-%d" % (c.start, c.stop - 1))
