"""The first Conv64F block (the "stem") against float64 at the batch sizes the benchmark runs.

* csrc/conv1_tc.cu (tcgen05 TF32, the default eval path) over its persistent schedule: one CTA per SM (148) walks tiles
  of 128 pooled pixels through four operand buffers and two accumulator sets, so a CTA's fifth tile is the first to
  reuse a buffer.  The reference rounds the operands exactly as the kernel does, which leaves only the fp32
  accumulation, and the bound is per element.
* csrc/conv1.cu (exact fp32, the parity path when torch.backends.cudnn.allow_tf32 is off) at the same shapes.
* csrc/conv1_train.cu (training mode: batch statistics from the 9-tap autocorrelation, fused forward, recomputing
  backward) against float64 autograd of Conv2d -> BatchNorm2d(train) -> activation -> MaxPool2d at the bench training
  size, at strip tails, with exact max-pool ties and with inputs that carry a DC offset.

Every bound is c * 2^-p times an "absolute" evaluation of the same expression (|x| and |w| in place of x and w), the
scale fp32 rounding errors are proportional to.  Each c is stated with the worst ratio measured on a B200."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U23 = 2.0 ** -23  # unit roundoff of TF32 products accumulated in fp32 (one ulp of fp32 at 1.0)
U24 = 2.0 ** -24  # unit roundoff of fp32 (round to nearest)
NUM_SMS = 148     # persistent grid of conv1_tc: min(tiles, kNumSMs)

# conv1_tc against fp64 of TF32-rounded operands: per element
#   |got - ref| <= C_TF32 * 2^-23 * (maxpool3(conv(|xq|, |wq|)) + |shift|).
# Products of TF32 values are exact in fp32; what remains is the accumulation of 15 products inside the MMA and the
# shift add.  Measured on a B200 (1000 W): at most 2.16 over the cases below.  Activations truncated instead of rounded
# (the MMA's own behaviour when the rounding is skipped) measured 278 to 7 918.
C_TF32 = 8.0
# conv1.cu against fp64: a product and eight FMAs (one rounding each), the shift add and the LeakyReLU multiply, each
# at most one rounding of a value bounded by the absolute expression: 11 in first order.  Measured: at most 4.41.
C_FP32 = 11.0
# conv1_train against fp64 autograd, each in units of 2^-24 times the absolute expression of _TrainRef.  Measured on a
# B200 (1000 W), worst over all training cases, DC offsets included:
#   output 5.18 (fp32 conv with folded weights: the same chain as conv1.cu, plus the fp32 scale and shift)
C_TRAIN_OUT = 8.0
#   dW 1.24, dgamma 0.55, dbeta 0.42 (the largest at 5 x 9 x 10, where the sums are shortest)
C_TRAIN_GRAD = 4.0
#   batch variance 1.53 and mean 0.82, running_var 1.58 and running_mean 0.20 (fp32 sums around a pivot, fp64 combine,
#   one fp32 rounding at the store).  The same kernel without the pivot: batch variance 10.9 and running_var 5.2 on
#   10 + randn input (2.7 and 2.5 on the log-mel-like input), 0.9 and 1.6 on zero-mean input.
C_STATS = 4.0


def _train_bound(gate):
    return C_TRAIN_OUT if gate.startswith("out") else C_STATS if gate.startswith("running") else C_TRAIN_GRAD


def _tf32(t):
    """Round finite fp32 values to TF32 the way cvt.rna.tf32.f32 does: to nearest, ties away from zero."""
    return ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def _act32(v, slope):
    """The kernels' activation in fp32: max(v, slope v) for 0 <= slope < 1."""
    return torch.where(v > 0, v, v * slope)


def _clip_chunks(N, H, W, max_clips=None):
    """Slices of clips whose [n, 64, H, W] float64 conv output stays near 128 MB."""
    step = max(1, (1 << 24) // (64 * H * W))
    if max_clips is not None:
        step = min(step, max_clips)
    return [slice(i, min(N, i + step)) for i in range(0, N, step)]


def _tiles_per_cta(N, H, W):
    tiles = -(-N * (H // 3) * (W // 3) // 128)
    return -(-tiles // min(tiles, NUM_SMS))


def _worst(got, ref, base, unit):
    """max |got - ref| / (unit * base) over all elements."""
    err = (got.double() - ref).abs()
    return (err / (base * unit).clamp_min(1e-300)).max().item()


# ------------------------------------------------------------------------------------------------ eval stem
def _stem_input(cuda, N, H, W, seed):
    """randn clips with an exactly constant block (-5.4, the normalised log-mel floor; not a TF32 value) in the top
    left and an all-zero band at the bottom right, so that windows of identical taps and tied maxima occur."""
    g = torch.Generator(device=cuda).manual_seed(seed)
    x = torch.randn((N, 1, H, W), generator=g, device=cuda)
    x[:, :, : (H + 1) // 2, : (W + 1) // 2] = -5.4
    x[:, :, H - max(1, H // 4):, W // 3:] = 0.0
    return x


def _stem_weights(seed):
    rng = np.random.default_rng(seed)
    w = (rng.standard_normal((64, 9)) * 0.3).astype(np.float32)
    w[5] *= -1.0   # a negative BatchNorm scale folded in
    w[7] = 0.0     # an all-zero row: the output is activation(shift) exactly
    shift = rng.standard_normal(64).astype(np.float32)
    return w, shift


def _stem_reference(x, w, shift, slope):
    """float64 conv2d -> + shift -> activation -> max_pool2d(3, 3) of x [N, 1, H, W] with folded weights w [64, 9], and
    the bound scale maxpool3(conv2d(|x|, |w|)) + |shift|; both [N, 64, H/3, W/3], evaluated in chunks of clips."""
    N, _, H, W = x.shape
    wd = w.double().view(64, 1, 3, 3)
    sd = shift.double().view(1, 64, 1, 1)
    outs, bases = [], []
    for c in _clip_chunks(N, H, W):
        xc = x[c].double()
        outs.append(F.max_pool2d(F.leaky_relu(F.conv2d(xc, wd, padding=1) + sd, slope), 3, 3))
        bases.append(F.max_pool2d(F.conv2d(xc.abs(), wd.abs(), padding=1), 3, 3) + sd.abs())
    return torch.cat(outs), torch.cat(bases)


STEM_CASES = [
    # N, H, W, slope                 tiles of 128 pooled pixels; tiles per CTA
    pytest.param(401, 128, 157, 0.0, id="401x128x157"),    # 6 843 tiles: 46-47 per CTA, an uneven last round (35 CTAs
                                                           # run a 47th tile) and a tail tile of 8 pixels
    pytest.param(37, 128, 157, 0.2, id="37x128x157"),      # 632 tiles: CTAs 0-39 run a fifth tile, the first that
                                                           # reuses operand buffer 0 (ring wrap, phase flip)
    pytest.param(20000, 9, 10, 0.99, id="20000x9x10"),     # 9 pooled pixels per image, so a tile straddles ~14
                                                           # images; 1 407 tiles, 9-10 per CTA
    pytest.param(80000, 3, 4, 0.0, id="80000x3x4"),        # one pooled pixel per image: input column 3 is never
                                                           # pooled but feeds the conv's right tap; 625 tiles, 4-5 per CTA
    pytest.param(64, 20, 23, 0.01, id="64x20x23"),         # H, W not multiples of 3 (rows 18-19 and columns 21-22
                                                           # only feed the conv), odd PW = 7; 21 tiles
    pytest.param(1, 3, 3, 0.0, id="1x3x3"),                # a single pooled pixel: one tile, 127 tail rows
    pytest.param(2, 7, 11, 0.2, id="2x7x11"),              # 12 pooled pixels, both dimensions ragged
]


@pytest.mark.parametrize("N,H,W,slope", STEM_CASES)
def test_conv1_tc_matches_fp64_of_tf32_rounded_operands(cuda, N, H, W, slope):
    """conv1_tc rounds the folded weights and every patch value to TF32 (cvt.rna) before the MMA.  Against an fp64
    evaluation of the host-rounded operands (the kernel itself gets the unrounded data) the error per element is
    within C_TF32 * 2^-23 of maxpool3(conv(|xq|, |wq|)) + |shift|; measured on a B200 (1000 W): 1.7 to 2.2 at the
    shapes of more than one tile, 0.6 and 0.9 at the two smallest.  The all-zero weight row gives activation(shift) bit for bit, and the
    bf16 output is the fp32 output rounded to nearest even, bit for bit."""
    from audio_fewshot_b200 import ops
    x = _stem_input(cuda, N, H, W, seed=N + 7 * H + W)
    w, shift = _stem_weights(seed=N * 3 + H)
    got = ops.conv1_bn_act_pool3(x, w, shift, slope, tf32=True)
    assert got.shape == (N, 64, H // 3, W // 3)
    wq = _tf32(torch.from_numpy(w).to(cuda))
    ref, base = _stem_reference(_tf32(x), wq, torch.from_numpy(shift).to(cuda), slope)
    worst = _worst(got, ref, base, U23)
    print("conv1_tc %dx%dx%d slope %g: %d tiles per CTA at most, worst error %.2f x 2^-23 x abs-conv (bound %g)"
          % (N, H, W, slope, _tiles_per_cta(N, H, W), worst, C_TF32))
    assert worst <= C_TF32
    want7 = _act32(torch.tensor(float(shift[7]), device=cuda), slope)
    assert torch.equal(got[:, 7], want7.expand_as(got[:, 7]))
    b16 = ops.conv1_bn_act_pool3(x, w, shift, slope, tf32=True, out_dtype=torch.bfloat16)
    assert b16.dtype == torch.bfloat16 and b16.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(b16, got.to(torch.bfloat16))


@pytest.mark.parametrize("N,H,W,clips", [
    (401, 128, 157, [0, 17, 400]),   # 2 184 pooled pixels per clip: clip 17 starts at pixel 8 of tile 290
    (20000, 9, 10, [0, 14, 19999]),  # 9 per clip: clip 14 spans pixels 126-134, across the boundary of tiles 0 and 1
])
def test_conv1_tc_clip_is_independent_of_its_batch(cuda, N, H, W, clips):
    """A clip's features are bit-identical whether the clip runs alone (one CTA, first tile, first buffer) or inside a
    batch (deep in the persistent schedule, at any offset within a tile)."""
    from audio_fewshot_b200 import ops
    x = _stem_input(cuda, N, H, W, seed=5 * N + W)
    w, shift = _stem_weights(seed=11)
    full = ops.conv1_bn_act_pool3(x, w, shift, 0.2, tf32=True)
    for i in clips:
        alone = ops.conv1_bn_act_pool3(x[i:i + 1].clone(), w, shift, 0.2, tf32=True)
        assert torch.equal(alone, full[i:i + 1]), i


def test_conv1_tc_rejects_slopes_its_activation_cannot_express(cuda):
    """The kernel's activation is max(v, slope v): LeakyReLU only for 0 <= slope < 1."""
    from audio_fewshot_b200 import _lib, ops
    x = torch.zeros((1, 1, 9, 9), device=cuda)
    w, shift = _stem_weights(seed=1)
    for slope in (1.0, 1.5, -0.1):
        with pytest.raises(_lib.AfsError):
            ops.conv1_bn_act_pool3(x, w, shift, slope, tf32=True)


@pytest.mark.parametrize("N,H,W,slope", STEM_CASES)
def test_conv1_fp32_matches_fp64(cuda, N, H, W, slope):
    """conv1.cu (exact fp32) against fp64 of the same operands: per element within C_FP32 * 2^-24 of
    maxpool3(conv(|x|, |w|)) + |shift|, the first-order worst case of its 11 roundings; measured on a B200 (1000 W):
    3.3 to 4.4 at the shapes of more than one tile, 1.3 and 1.8 at the two smallest.  The all-zero weight row gives activation(shift) bit for bit."""
    from audio_fewshot_b200 import ops
    x = _stem_input(cuda, N, H, W, seed=N + 7 * H + W + 1)
    w, shift = _stem_weights(seed=N * 3 + H + 1)
    got = ops.conv1_bn_act_pool3(x, w, shift, slope)
    assert got.shape == (N, 64, H // 3, W // 3)
    ref, base = _stem_reference(x, torch.from_numpy(w).to(cuda), torch.from_numpy(shift).to(cuda), slope)
    worst = _worst(got, ref, base, U24)
    print("conv1 fp32 %dx%dx%d slope %g: worst error %.2f x 2^-24 x abs-conv (bound %g)" % (N, H, W, slope, worst, C_FP32))
    assert worst <= C_FP32
    want7 = _act32(torch.tensor(float(shift[7]), device=cuda), slope)
    assert torch.equal(got[:, 7], want7.expand_as(got[:, 7]))


# ------------------------------------------------------------------------------------------------ training stem
class _TrainRef:
    """float64 Conv2d(1, 64, 3, pad 1) -> BatchNorm2d(batch statistics) -> LeakyReLU(slope) -> MaxPool2d(3, 3) of x, and
    its gradients under autograd, evaluated in chunks of clips so that the bench training size (200 x 128 x 157: 2 GB
    per float64 activation) stays within a few hundred MB of device memory.

    Batch statistics take two passes (mean, then the mean square deviation).  For the gradients, the per-channel mean m
    and variance v are leaves: one pass gives dL/dm and dL/dv, and a second pass adds their chain rule
    (dm/dy = 1/P, dv/dy = 2 (y - m)/P) as an extra gradient on the conv output.  With last_max the max-pool routes the
    gradient of a tied window to its LAST maximum instead of torch's first (H and W must be multiples of 3).

    The bounds of the comparison are "absolute" evaluations of the same quantities (each in units of 2^-24):
      output      |scale| maxpool3(conv(|x|, |w|)) + |shift|
      dW          conv2d_weight(|x|, |dL/dconv|)
      dgamma      sum |dL/dz| invstd (conv(|x|, |w|) + |mean - bias|)  (z: the BatchNorm output)
      dbeta       sum |dL/dz|
      running     |running_mean| + mean |conv|, and running_var."""

    def __init__(self, x, conv, bn, slope, last_max=False, max_clips=None):
        N, _, H, W = x.shape
        assert not last_max or (H % 3 == 0 and W % 3 == 0)
        self.x, self.slope, self.last_max = x, float(slope), last_max
        self.W, self.B = conv.weight.detach().double(), conv.bias.detach().double()
        self.gamma, self.beta = bn.weight.detach().double(), bn.bias.detach().double()
        self.eps = bn.eps
        self.P = N * H * W
        self.parts = _clip_chunks(N, H, W, max_clips)
        s = sa = 0.0
        for c in self.parts:
            y = F.conv2d(x[c].double(), self.W, self.B, padding=1)
            s = s + y.sum((0, 2, 3))
            sa = sa + y.abs().sum((0, 2, 3))
        self.mean, self.mean_abs = s / self.P, sa / self.P
        q = 0.0
        for c in self.parts:
            y = F.conv2d(x[c].double(), self.W, self.B, padding=1)
            q = q + (y - self.mean.view(1, -1, 1, 1)).square().sum((0, 2, 3))
        self.var = q / self.P
        self.invstd = torch.rsqrt(self.var + self.eps)
        self.scale = self.gamma * self.invstd
        self.shift = self.beta - (self.mean - self.B) * self.scale

    def _block(self, xc, W, B, gamma, beta, m, v):
        col = lambda t: t.view(1, -1, 1, 1)  # noqa: E731
        y = F.conv2d(xc, W, B, padding=1)
        z = (y - col(m)) * col(torch.rsqrt(v + self.eps)) * col(gamma) + col(beta)
        a = F.leaky_relu(z, self.slope)
        o = F.max_pool2d(a.flip(2, 3), 3, 3).flip(2, 3) if self.last_max else F.max_pool2d(a, 3, 3)
        return y, z, o

    def running(self, rm, rv, momentum):
        """nn.BatchNorm2d's running-statistics update after this batch (unbiased variance)."""
        return ((1 - momentum) * rm + momentum * self.mean,
                (1 - momentum) * rv + momentum * self.var * self.P / (self.P - 1))

    def forward(self):
        """(output, output bound, gap between the two largest BatchNorm outputs of every pooling window)."""
        outs, bases, gaps = [], [], []
        for c in self.parts:
            xc = self.x[c].double()
            _, z, o = self._block(xc, self.W, self.B, self.gamma, self.beta, self.mean, self.var)
            outs.append(o)
            n, _, H, W = z.shape
            PH, PW = H // 3, W // 3
            win = z[:, :, :3 * PH, :3 * PW].reshape(n, 64, PH, 3, PW, 3).permute(0, 1, 2, 4, 3, 5).reshape(n, 64, PH, PW, 9)
            top = win.topk(2, dim=-1).values
            gaps.append(top[..., 0] - top[..., 1])
            M = F.max_pool2d(F.conv2d(xc.abs(), self.W.abs(), padding=1), 3, 3)
            bases.append(self.scale.abs().view(1, -1, 1, 1) * M + self.shift.abs().view(1, -1, 1, 1))
        return torch.cat(outs), torch.cat(bases), torch.cat(gaps)

    def backward(self, gout):
        """Gradients (dW [64, 1, 3, 3], dbias, dgamma, dbeta) for the upstream gradient gout, and the bounds of dW,
        dgamma, dbeta."""
        m = self.mean.clone().requires_grad_()
        v = self.var.clone().requires_grad_()
        for c in self.parts:
            _, _, o = self._block(self.x[c].double(), self.W, self.B, self.gamma, self.beta, m, v)
            o.backward(gout[c].double())
        gm, gv = m.grad.view(1, -1, 1, 1), v.grad.view(1, -1, 1, 1)
        W, B = self.W.clone().requires_grad_(), self.B.clone().requires_grad_()
        gamma, beta = self.gamma.clone().requires_grad_(), self.beta.clone().requires_grad_()
        base_w = base_g = base_b = 0.0
        mnob = (self.mean - self.B).abs().view(1, -1, 1, 1)
        for c in self.parts:
            xc = self.x[c].double()
            y, z, o = self._block(xc, W, B, gamma, beta, self.mean, self.var)
            y.retain_grad()
            z.retain_grad()
            gy = (gm + 2.0 * gv * (y.detach() - self.mean.view(1, -1, 1, 1))) / self.P
            torch.autograd.backward([o, y], [gout[c].double(), gy])
            base_w = base_w + torch.nn.grad.conv2d_weight(xc.abs(), W.shape, y.grad.abs(), padding=1)
            dz = z.grad.abs()
            base_b = base_b + dz.sum((0, 2, 3))
            base_g = base_g + (dz * (F.conv2d(xc.abs(), self.W.abs(), padding=1) + mnob)).sum((0, 2, 3))
        return (W.grad, B.grad, gamma.grad, beta.grad), (base_w, base_g * self.invstd, base_b)


def _train_block(cuda, seed, integer=False):
    """Conv2d + BatchNorm2d in train mode with a random conv bias, gamma with negative entries, and non-default running
    statistics; integer=True: integer weights, bias 0, gamma 1, beta 0 (for exact ties)."""
    torch.manual_seed(seed)
    conv = torch.nn.Conv2d(1, 64, 3, padding=1).to(cuda)
    bn = torch.nn.BatchNorm2d(64).to(cuda).train()
    with torch.no_grad():
        if integer:
            conv.weight.copy_(torch.randint(-2, 3, conv.weight.shape, device=cuda).float())
            conv.bias.zero_()
        else:
            conv.weight.mul_(2.0)
            conv.bias.copy_(torch.randn(64, device=cuda))
            bn.weight.copy_(torch.randn(64, device=cuda) * 0.5 + 1.0)
            bn.weight[:6] *= -1.0
            bn.bias.copy_(torch.randn(64, device=cuda) * 0.3)
        bn.running_mean.copy_(torch.randn(64, device=cuda) * 0.1)
        bn.running_var.copy_(torch.rand(64, device=cuda) + 0.5)
    return conv, bn


def _train_input(cuda, kind, N, H, W, seed):
    g = torch.Generator(device=cuda).manual_seed(seed)
    x = torch.randn((N, 1, H, W), generator=g, device=cuda)
    if kind == "logmel":  # normalised log-mel: the silent half of every clip sits at the floor
        x[..., : W // 2] = -5.4
    elif kind == "offset10":
        x += 10.0
    elif kind == "integer":  # small integers with zero-padded "silent" blocks: every tie is exact in fp32 and fp64
        x = torch.randint(-2, 3, (N, 1, H, W), generator=g, device=cuda).float()
        x[..., :, 9:18] = 0.0
        x[..., H // 2:, W - 9:] = 0.0
    else:
        assert kind == "randn"
    return x


def _ratio(got, ref, base):
    return _worst(got.reshape(ref.shape), ref, base.reshape(ref.shape), U24)


def _grad_ratios(got, ref, bases):
    return [(key, _ratio(g, r, b)) for key, g, r, b in zip(("dW", "dgamma", "dbeta"), got, ref, bases)]


@pytest.mark.parametrize("N,H,W,slope,kind", [
    pytest.param(200, 128, 157, 0.0, "randn", id="200x128x157-relu"),            # the bench training size: 26.5
    pytest.param(200, 128, 157, 0.2, "randn", id="200x128x157-leaky"),           # positions per autocorrelation thread,
    pytest.param(200, 128, 157, 0.2, "logmel", id="200x128x157-leaky-logmel"),   # ~46 backward strips per warp
    pytest.param(200, 128, 157, 0.0, "offset10", id="200x128x157-relu-offset10"),
    pytest.param(7, 20, 23, 0.2, "randn", id="7x20x23-leaky"),                   # PW = 7: a strip of 3 per row
    pytest.param(5, 9, 10, 0.0, "randn", id="5x9x10-relu"),                      # PW = 3 < 4: one short strip per row
])
def test_conv1_train_matches_fp64_autograd(cuda, N, H, W, slope, kind):
    """Two training steps on different batches (momentum applied twice), then a backward pass, against _TrainRef:
    output of both steps (C_TRAIN_OUT), running_mean / running_var (C_STATS), dW, dgamma, dbeta (C_TRAIN_GRAD), each
    times 2^-24 of its absolute expression, and d(conv bias) exactly 0.

    Windows whose two largest float64 BatchNorm outputs lie within 1e-5 of the output range (but are not equal) get a
    zero upstream gradient in both runs: fp32 and fp64 may route them to different taps.  Exact ties (windows of equal
    taps in the constant half of "logmel") are left in; both route them to the first maximum.

    DC offsets: "logmel" holds half of every clip at -5.4 (mean -2.7, standard deviation 2.8), "offset10" is 10 + randn
    (mean 10, standard deviation 1).  The variance of a tap is then 1/100 of its mean square, so sums of products
    accumulated in fp32 lose two digits when centred; the autocorrelation therefore accumulates around a pivot near the
    mean.  Both meet the zero-mean bounds.  Measured on a B200 (1000 W), worst ratios: see C_TRAIN_OUT, C_TRAIN_GRAD
    and C_STATS; the DC-offset cases reach output 4.88, running_var 1.21, dW 0.09 (zero-mean: 5.18, 1.58, 1.24).  At
    most 0.09 % of the windows are masked as near ties."""
    x1 = _train_input(cuda, kind, N, H, W, seed=2 * N + W)
    x2 = _train_input(cuda, kind, N, H, W, seed=2 * N + W + 1)
    conv, bn = _train_block(cuda, seed=N + H + int(slope * 10))
    rm0, rv0 = bn.running_mean.double(), bn.running_var.double()
    from audio_fewshot_b200 import ops
    gates = []
    ref1 = _TrainRef(x1, conv, bn, slope)
    out1 = ops.conv1_bn_act_pool3_train(x1, conv, bn, slope)
    want1, base1, _ = ref1.forward()
    gates.append(("out step 1", _ratio(out1.detach(), want1, base1)))
    del out1, want1, base1
    ref2 = _TrainRef(x2, conv, bn, slope)
    conv.zero_grad(set_to_none=True)
    bn.zero_grad(set_to_none=True)
    out2 = ops.conv1_bn_act_pool3_train(x2, conv, bn, slope)
    want2, base2, gap = ref2.forward()
    gates.append(("out step 2", _ratio(out2.detach(), want2, base2)))
    rm1, rv1 = ref1.running(rm0, rv0, bn.momentum)
    rm2, rv2 = ref2.running(rm1, rv1, bn.momentum)
    gates.append(("running_mean", _ratio(bn.running_mean, rm2, rm2.abs() + torch.maximum(ref1.mean_abs, ref2.mean_abs))))
    gates.append(("running_var", _ratio(bn.running_var, rv2, rv2)))
    near = (gap > 0) & (gap <= 1e-5 * want2.abs().max())
    n_near = int(near.sum())
    print("%s: %d of %d windows masked as near ties" % (kind, n_near, near.numel()))
    assert n_near < 0.01 * near.numel()
    g = torch.Generator(device=cuda).manual_seed(3 * N + H)
    gout = torch.randn(want2.shape, generator=g, device=cuda, dtype=torch.float64).masked_fill_(near, 0.0).float()
    del want2, base2, gap, near
    out2.backward(gout.contiguous(memory_format=torch.channels_last))
    assert conv.bias.grad is not None and torch.count_nonzero(conv.bias.grad).item() == 0
    ref_grads, bases = ref2.backward(gout)
    got = (conv.weight.grad, bn.weight.grad, bn.bias.grad)
    gates += _grad_ratios(got, (ref_grads[0], ref_grads[2], ref_grads[3]), bases)
    for key, worst in gates:
        print("%dx%dx%d %s slope %g %s: worst error %.2f x 2^-24 x abs (bound %g)" % (N, H, W, kind, slope, key, worst, _train_bound(key)))
    assert all(worst <= _train_bound(key) for key, worst in gates), gates


@pytest.mark.parametrize("slope", [0.0, 0.2])
def test_conv1_train_routes_exact_ties_to_the_first_maximum(cuda, slope):
    """Integer input with silent (zero) blocks and integer weights, bias 0, gamma 1, beta 0: every conv value is an
    integer, exact in fp32 and fp64, so tied windows are tied in both.  Without any masking the gradients match the
    float64 graph, whose max-pool backward routes a tie to the first maximum in row-major order; a graph that routes
    to the last maximum gives different gradients, by far more than the bound."""
    N, H, W = 16, 24, 27
    x = _train_input(cuda, "integer", N, H, W, seed=77)
    conv, bn = _train_block(cuda, seed=78, integer=True)
    ref = _TrainRef(x, conv, bn, slope)
    last = _TrainRef(x, conv, bn, slope, last_max=True)
    from audio_fewshot_b200 import ops
    out = ops.conv1_bn_act_pool3_train(x, conv, bn, slope)
    want, base, gap = ref.forward()
    ties = int((gap == 0).sum())
    print("exact ties: %d of %d windows" % (ties, gap.numel()))
    assert ties > 0.05 * gap.numel()
    gout = torch.randn(want.shape, generator=torch.Generator(device=cuda).manual_seed(79), device=cuda)
    out.backward(gout.contiguous(memory_format=torch.channels_last))
    assert torch.count_nonzero(conv.bias.grad).item() == 0
    (dW, _, dg, db), bases = ref.backward(gout)
    (dW_last, _, dg_last, db_last), _ = last.backward(gout)
    gates = [("out", _ratio(out.detach(), want, base))]
    gates += _grad_ratios((conv.weight.grad, bn.weight.grad, bn.bias.grad), (dW, dg, db), bases)
    teeth = _ratio(dW_last.float(), dW, bases[0])
    print("exact ties slope %g: %s; last-maximum routing: dW off by %.3g x 2^-24 x abs" % (slope, gates, teeth))
    assert all(worst <= _train_bound(key) for key, worst in gates), gates
    # the case has teeth: last-maximum routing moves dW far outside the bound (measured 1.5e6)
    assert teeth > 100 * C_TRAIN_GRAD


@pytest.mark.parametrize("kind", ["randn", "logmel", "offset10"])
def test_conv1_train_batch_statistics_match_fp64(cuda, kind):
    """The batch statistics alone, at the bench training size: with momentum 1 the running statistics ARE the batch mean
    and the unbiased batch variance, computed by the fp64 combine from the fp32 autocorrelation sums.  The variance is
    within C_STATS * 2^-24 of the fp64 variance relative to itself, the mean within C_STATS * 2^-24 of mean |conv|.
    This is what a DC offset attacks: summed as raw x_t x_u, the 10 + randn input's products are ~100x its variance
    and the variance came out 10.9 x 2^-24 off on a B200 (1000 W); summed around the pivot it is 0.9, as for zero-mean
    input (0.96; log-mel-like 1.53)."""
    N, H, W = 200, 128, 157
    x = _train_input(cuda, kind, N, H, W, seed=91)
    conv, bn = _train_block(cuda, seed=92)
    bn.momentum = 1.0
    ref = _TrainRef(x, conv, bn, 0.0)
    from audio_fewshot_b200 import ops
    with torch.no_grad():
        ops.conv1_bn_act_pool3_train(x, conv, bn, 0.0)
    var = ref.var * ref.P / (ref.P - 1)
    e_var = ((bn.running_var.double() - var).abs() / var).max().item() / U24
    e_mean = ((bn.running_mean.double() - ref.mean).abs() / ref.mean_abs).max().item() / U24
    print("batch statistics %s: variance %.2f, mean %.2f x 2^-24 (bound %g)" % (kind, e_var, e_mean, C_STATS))
    assert e_var <= C_STATS and e_mean <= C_STATS


def test_chunked_fp64_reference_matches_the_batch_norm_graph(cuda):
    """_TrainRef in chunks of two clips against F.conv2d -> F.batch_norm(training=True) -> leaky_relu -> max_pool2d in
    float64 on the whole batch, under autograd: output, running statistics and all four gradients to 1e-12."""
    N, H, W, slope = 7, 20, 23, 0.2
    x = _train_input(cuda, "offset10", N, H, W, seed=5)
    conv, bn = _train_block(cuda, seed=6)
    ref = _TrainRef(x, conv, bn, slope, max_clips=2)
    assert len(ref.parts) == 4
    params = [p.detach().double().clone().requires_grad_() for p in (conv.weight, conv.bias, bn.weight, bn.bias)]
    rm, rv = bn.running_mean.double().clone(), bn.running_var.double().clone()
    z = F.batch_norm(F.conv2d(x.double(), params[0], params[1], padding=1), rm, rv, params[2], params[3],
                     training=True, momentum=bn.momentum, eps=bn.eps)
    want = F.max_pool2d(F.leaky_relu(z, slope), 3, 3)
    got, _, _ = ref.forward()
    close = lambda a, b: (a - b).abs().max().item() <= 1e-12 * max(b.abs().max().item(), 1.0)  # noqa: E731
    assert close(got, want)
    rm_ref, rv_ref = ref.running(bn.running_mean.double(), bn.running_var.double(), bn.momentum)
    assert close(rm_ref, rm) and close(rv_ref, rv)
    gout = torch.randn(want.shape, generator=torch.Generator(device=cuda).manual_seed(7), device=cuda, dtype=torch.float64)
    want.backward(gout)
    grads, _ = ref.backward(gout)
    for g, p in zip(grads, params):
        assert close(g, p.grad)
