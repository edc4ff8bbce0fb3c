"""The tensor-core stem (csrc/conv1_tc.cu) bit for bit against float64 on an exact grid.

Inputs k/4 (|k| <= 16), folded weights j/32 (|j| <= 32) and shifts m/128 are TF32 values whose products are multiples
of 2^-7 and whose every partial sum (nine products, the shift, the LeakyReLU slope 1/4) stays below 2^10: exact in
fp32 whatever the order.  The kernel's fp32 output must then equal the float64 evaluation exactly, and its bf16
output must equal that value rounded to nearest even.

The output is written into a NaN-filled buffer between two guard bands of sentinel pixels: every pixel must be
written (no NaN left), none past either end (guards intact).  The kernel stores each EPI warp's 32 pixels x 32
channels as one swizzled TMA box, so a swizzle error moves channels or pixels, and a tail error writes past the last
pixel or leaves its last box unwritten."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

GUARD = 96  # sentinel pixels on each side of the output
SENTINEL = 1234.5


def _grid_case(cuda, N, H, W, seed):
    g = torch.Generator(device=cuda).manual_seed(seed)
    x = torch.randint(-16, 17, (N, 1, H, W), generator=g, device=cuda).float() / 4
    w = torch.randint(-32, 33, (64, 9), generator=g, device=cuda).float() / 32
    w[9] = 0.0  # an all-zero row: activation(shift)
    shift = torch.randint(-512, 513, (64,), generator=g, device=cuda).float() / 128
    return x, w, shift


def _reference(x, w, shift, slope):
    """float64 conv -> + shift -> activation -> max_pool2d(3, 3), channels-last [N, H/3, W/3, 64], in chunks of clips."""
    N, _, H, W = x.shape
    wd = w.double().view(64, 1, 3, 3)
    sd = shift.double().view(1, 64, 1, 1)
    step = max(1, (1 << 24) // (64 * H * W))
    outs = []
    for i in range(0, N, step):
        y = F.conv2d(x[i:i + step].double(), wd, padding=1) + sd
        outs.append(F.max_pool2d(F.leaky_relu(y, slope), 3, 3).permute(0, 2, 3, 1).float())
    return torch.cat(outs)


def _run(cuda, x, w, shift, slope, dtype):
    """The C entry point into the middle of a guarded NaN buffer; returns (output [N, H/3, W/3, 64], whole buffer)."""
    from audio_fewshot_b200 import _lib, ops
    N, _, H, W = x.shape
    total = N * (H // 3) * (W // 3)
    buf = torch.full((GUARD + total + GUARD, 64), float("nan"), dtype=dtype, device=cuda)
    buf[:GUARD] = SENTINEL
    buf[GUARD + total:] = SENTINEL
    out = buf[GUARD:GUARD + total]
    h = _lib.lib()
    fn = h.afs_conv1_bn_act_pool3_fwd_tf32_bf16out if dtype == torch.bfloat16 else h.afs_conv1_bn_act_pool3_fwd_tf32
    wn = w.cpu().numpy()
    sn = shift.cpu().numpy()
    _lib.check(fn(ops._ptr(x.contiguous()), N, H, W, wn.ctypes.data_as(ops.C.c_void_p),
                  sn.ctypes.data_as(ops.C.c_void_p), 64, float(slope), ops._ptr(out), ops._stream()),
               "afs_conv1_bn_act_pool3_fwd")
    torch.cuda.synchronize()
    return out.view(N, H // 3, W // 3, 64), buf


@pytest.mark.parametrize("N,H,W,slope", [
    pytest.param(3200, 128, 157, 0.0, id="3200x128x157-relu"),  # the bench batch: 54 600 tiles, 368-369 per CTA
    pytest.param(37, 128, 157, 0.25, id="37x128x157-leaky"),    # 80 808 pixels: the last tile holds 40, so its second
                                                                # box is 8 pixels and its last two boxes are empty
    pytest.param(2, 7, 11, 0.25, id="2x7x11-leaky"),            # 12 pixels: one partial box, three empty ones
])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_conv1_tc_exact_grid_equals_fp64(cuda, N, H, W, slope, dtype):
    x, w, shift = _grid_case(cuda, N, H, W, seed=N + H + W)
    got, buf = _run(cuda, x, w, shift, slope, dtype)
    total = got.numel() // 64
    assert not torch.isnan(got).any(), "pixels left unwritten"
    assert torch.equal(buf[:GUARD], torch.full_like(buf[:GUARD], SENTINEL)), "written before the output"
    assert torch.equal(buf[GUARD + total:], torch.full_like(buf[GUARD + total:], SENTINEL)), "written past the output"
    want = _reference(x, w, shift, slope).to(dtype)
    bad = (got != want).any(-1)
    assert not bad.any(), "%d of %d pixels differ, first at %s" % (int(bad.sum()), total, tuple(bad.nonzero()[0].tolist()))
    assert torch.equal(got[..., 9], F.leaky_relu(shift[9], slope).to(dtype).expand_as(got[..., 9]))
