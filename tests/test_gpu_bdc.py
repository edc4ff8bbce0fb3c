"""The BDC matrix kernels against a float64 evaluation of the oracle (oracle.heads.bdcovpool + triuvec, plain torch):
csrc/bdc_tc.cu, the persistent tcgen05 forward for C == 64, over every shape its schedule takes; csrc/bdc.cu, the fp32
FMA forward for every other shape and the backward, including the gradient of the log-temperature; both forward paths
at the same shapes; and the full-size DeepBDC step.

afs_bdc_fwd falls back to bdc.cu without a word whenever the tensor-core path declines a shape (C != 64, M % 4 != 0, a
misaligned pointer, a tensor map the driver refuses), so every forward case checks with torch.profiler which kernel
ran: a "tensor-core" case that did not would quietly test the FMA kernel.  Errors are scaled by max|reference|, as in
test_gpu_heads.py."""
import math
import re

import numpy as np
import pytest
import torch

from oracle import heads

pytestmark = pytest.mark.gpu

T200 = math.log(1.0 / 200.0)  # BdcPool's initial log-temperature: log(1 / (2 h w)) of the declared 10 x 10 map
FWD_BAR = 2e-5                # of max|ref|: the bar of test_gpu_heads.py::test_bdc_matches_reference_golden
GRAD_X_BAR = 2e-3             # of max|ref grad|: test_gpu_heads.py::test_bdc_backward_matches_autograd_of_oracle
# grad log_temp = sum over clips and (i, j) of t_ij = dA_ij e^t D_ij / (2 A_ij).  bdc_bwd_kernel sums a clip's C^2
# terms with a rounding depth of 29 (16 serial FMAs per thread, 5 shuffle levels, 8 warp partials) and torch's sum of
# the B <= 300 per-clip values adds at most ~16 more: < 45 fp32 roundings, 45 * 2^-24 = 2.7e-6 of sum|t_ij|.  Each term
# also carries the rounding of the recomputed D, A and of the centred dA (sums of 64 values): a few 2^-24 relative to
# max|dB| per term.  Hence 2e-5 * sum|t_ij|.  A scaled or wrong-signed gradient is off by |sum t_ij|, which for random
# grad_out is ~ sum|t_ij| / sqrt(B C^2): 1/1100 of it at B = 300, C = 64, still 45x the bar.
GRAD_T_BAR = 2e-5


@pytest.fixture(autouse=True)
def _tensor_core_switch_restored(cuda):
    """afs_bdc_set_tensor_core is process-wide: whatever a test sets, the next one starts from the default."""
    from audio_fewshot_b200 import ops
    try:
        yield
    finally:
        ops.bdc_set_tensor_core(True)


def _relu_normal(shape, seed):
    return torch.from_numpy(np.maximum(np.random.default_rng(seed).standard_normal(shape), 0.0).astype(np.float32))


def _bdc_kernels_of(fn):
    """Run fn() once under the CUDA profiler; return its result and the bdc* kernels it launched, in order."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [m.group(1) for e in prof.events() for m in [re.search(r"::(bdc\w*)\(", e.name)] if m]


def _pool(x, log_temp, triu=True, tc=True):
    """ops.bdc_pool with the tensor-core switch set to tc: (output, bdc kernels launched)."""
    from audio_fewshot_b200 import ops
    t = torch.full((1, 1), log_temp, device=x.device)
    ops.bdc_set_tensor_core(tc)
    return _bdc_kernels_of(lambda: ops.bdc_pool(x, t, triu=triu))


def _reference(x, log_temp):
    """float64 BDC matrices [B, C, C] of x [B, C, ...], on x's device."""
    B, C = x.shape[:2]
    t = torch.full((1, 1), log_temp, dtype=torch.float64, device=x.device)
    return heads.bdcovpool(x.double().reshape(B, C, 1, -1), t)


def _assert_close(got, ref, bar=FWD_BAR, what=""):
    scale = ref.abs().max().item()
    err = (got.double() - ref).abs().max().item()
    assert err <= bar * scale, "%s: max error %.3e, max|ref| %.3e, bar %.0e" % (what, err, scale, bar)


def _assert_bdc(got, ref, triu, what=""):
    B = ref.shape[0]
    _assert_close(got, heads.triuvec(ref) if triu else ref.reshape(B, -1), what=what)


# ------------------------------------------------------------------ tensor-core forward over the persistent schedule
# bdc_fwd_tc: tiles = ceil(B / 2) (two clips per tile), grid = min(tiles, kNumSMs = 148); CTA k runs tiles k, k + 148,
# k + 296, ... as its local tiles t = 0, 1, 2, ...  Local tile t goes to epilogue group t & 1 (warps 0-3 / 10-13, TMEM
# columns 0-255 / 256-511, scratch slots 0-1 / 2-3, named barriers 1-2 / 3-4), whose mbarrier phase is (t >> 1) & 1.
# An odd B leaves the second clip of the last tile empty (TMA zero fill, store skipped).
SCHEDULE_B = [
    1, 2, 3,    # one lone clip, one full tile, a full and a lone tile: t = 0 only
    295, 296,   # 148 tiles, the last lone / full: the whole grid busy, still t = 0 only
    297,        # 149 tiles: CTA 0 runs tile 148 as t = 1, the first tile any group 1 sees
    593,        # 297 tiles: CTA 0 runs the lone clip 592 as t = 2, group 0's first phase flip
    1201,       # 601 = 4 * 148 + 9 tiles: every CTA runs t = 0..3, CTAs 0-8 also t = 4; group 1 flips phase at t = 3,
                # the lone clip 1200 is CTA 8's fifth tile
]


@pytest.mark.parametrize("B", SCHEDULE_B)
def test_bdc_tc_forward_over_the_persistent_schedule(cuda, B):
    """C4 maps (64 x 16 x 19, post-ReLU N(0, 1)) at the batch sizes where the schedule changes shape, on both paths:
    within 2e-5 of fp64, the triangle store equal to the full store's upper triangle, symmetric and double-centred."""
    x = _relu_normal((B, 64, 16, 19), seed=B).to(cuda)
    ref = _reference(x, T200)
    scale = ref.abs().max().item()
    for tc, kernel in ((True, "bdc_tc_kernel"), (False, "bdc_kernel")):
        full, ran = _pool(x, T200, triu=False, tc=tc)
        assert ran == [kernel]
        triu, ran = _pool(x, T200, triu=True, tc=tc)
        assert ran == [kernel]
        full = full.reshape(B, 64, 64)
        _assert_bdc(full.reshape(B, -1), ref, triu=False, what=kernel)
        _assert_bdc(triu, ref, triu=True, what=kernel)
        assert torch.equal(heads.triuvec(full), triu), kernel
        assert (full - full.transpose(1, 2)).abs().max().item() <= 1e-5 * scale, kernel
        assert full.double().mean(dim=1).abs().max().item() <= 1e-4 * scale, kernel
        assert full.double().mean(dim=2).abs().max().item() <= 1e-4 * scale, kernel


# M < 32 is one partial 32-wide TMA box (4, 28); 32 exactly one box; 36, 100 and 1028 end on a 4-float chunk; 64 two
# full chunks; 304 the C4 map; 1028 is 33 chunks, eight trips around the 4-stage operand ring
TC_M = [4, 28, 32, 36, 64, 100, 304, 1028]


@pytest.mark.parametrize("M", TC_M)
def test_bdc_tc_forward_over_m_and_temperature(cuda, M):
    """B = 7 clips of 64 x M, log_temp in {log(1 / 2M), -3, 0}: both paths within 2e-5 of fp64."""
    B = 7
    x = _relu_normal((B, 64, M), seed=1000 + M).to(cuda)
    for log_temp in (math.log(1.0 / (2 * M)), -3.0, 0.0):
        ref = _reference(x, log_temp)
        for tc, kernel in ((True, "bdc_tc_kernel"), (False, "bdc_kernel")):
            out, ran = _pool(x, log_temp, tc=tc)
            assert ran == [kernel], (log_temp, tc)
            _assert_bdc(out, ref, triu=True, what="%s log_temp %.3f" % (kernel, log_temp))


@pytest.mark.parametrize("B", [7, 297])
def test_bdc_tc_cancellation_is_no_worse_than_the_fp32_gram(cuda, B):
    """x = 5 + 0.2 relu(N): every channel carries the same large offset, so D_ij = G_ii + G_jj - 2 G_ij is ~1/1000 of
    the Gram entries it is computed from and the fp32 rounding of G is amplified accordingly: neither path can meet
    2e-5.  The 3 x TF32 split keeps 21 bits of each operand and drops lo lo^T, i.e. it computes D of operands within
    2^-21 of x; that must not be worse than the FMA kernel's fp32 Gram."""
    g = np.random.default_rng(500 + B)
    x = torch.from_numpy((5.0 + 0.2 * np.maximum(g.standard_normal((B, 64, 304)), 0.0)).astype(np.float32)).to(cuda)
    ref = heads.triuvec(_reference(x, T200))
    scale = ref.abs().max().item()
    out_tc, ran = _pool(x, T200, tc=True)
    assert ran == ["bdc_tc_kernel"]
    out_fma, ran = _pool(x, T200, tc=False)
    assert ran == ["bdc_kernel"]
    err_tc = (out_tc.double() - ref).abs().max().item()
    err_fma = (out_fma.double() - ref).abs().max().item()
    assert err_tc <= 2.0 * err_fma + 1e-6 * scale, (err_tc / scale, err_fma / scale)


# ------------------------------------------------------------------ fallbacks to bdc.cu
@pytest.mark.parametrize("triu", [True, False])
def test_bdc_misaligned_input_takes_the_fma_kernel_bit_for_bit(cuda, triu):
    """x one float past a 16-byte boundary cannot be a TMA source: with the switch on the call must run bdc.cu and give
    exactly what the switch-off call gives on an aligned copy."""
    B, M = 5, 304
    x = _relu_normal((B, 64, M), seed=3).to(cuda)
    buf = torch.empty(B * 64 * M + 1, device=cuda)
    xm = buf[1:].view(B, 64, M)
    xm.copy_(x)
    assert xm.is_contiguous() and xm.data_ptr() % 16 == 4
    got, ran = _pool(xm, T200, triu=triu, tc=True)
    assert ran == ["bdc_kernel"]
    want, ran = _pool(x, T200, triu=triu, tc=False)
    assert ran == ["bdc_kernel"]
    assert torch.equal(got, want)
    _assert_bdc(got, _reference(x, T200), triu)


@pytest.mark.parametrize("M", [25, 37])
def test_bdc_m_not_a_multiple_of_4_takes_the_fma_kernel_bit_for_bit(cuda, M):
    """A row stride of M floats is not a multiple of 16 bytes, which a tensor map requires."""
    B = 5
    x = _relu_normal((B, 64, M), seed=M).to(cuda)
    got, ran = _pool(x, T200, tc=True)
    assert ran == ["bdc_kernel"]
    want, ran = _pool(x, T200, tc=False)
    assert ran == ["bdc_kernel"]
    assert torch.equal(got, want)
    _assert_bdc(got, _reference(x, T200), triu=True)


@pytest.mark.parametrize("C", [1, 17, 63])
@pytest.mark.parametrize("M", [1, 63, 64, 65, 129])
def test_bdc_fma_kernel_below_64_channels(cuda, C, M):
    """bdc.cu pads C to 64 and streams M in chunks of 64 positions: channel counts off the padding and M on both
    sides of the chunk edges.  C = 1 is identically zero (A - A - A + A) on both sides."""
    B = 3
    x = _relu_normal((B, C, M), seed=100 * C + M).to(cuda)
    ref = _reference(x, T200)
    for triu in (True, False):
        out, ran = _pool(x, T200, triu=triu, tc=True)
        assert ran == ["bdc_kernel"]
        _assert_bdc(out, ref, triu, what="triu=%s" % triu)


def test_bdc_more_than_64_channels_is_refused(cuda):
    from audio_fewshot_b200 import _lib, ops
    x = torch.ones(2, 65, 8, device=cuda)
    t = torch.full((1, 1), T200, device=cuda)
    for tc in (True, False):
        ops.bdc_set_tensor_core(tc)
        with pytest.raises(_lib.AfsError):
            ops.bdc_pool(x, t)


# ------------------------------------------------------------------ schedule independence
# (first, end) of x[first:end] against the 1201-clip call (clip c: tile c // 2, slot c % 2, local tile (c // 2) // 148)
SLICES = [
    (1, 1201),     # every clip changes tile slot
    (296, 1201),   # every clip keeps its slot and changes epilogue group (its tile moves back by one grid)
    (297, 1000),   # both, and clip 999 loses its neighbour: it becomes a lone clip next to zero-filled rows
    (600, 601),    # one clip (group 0, slot 0 in the full call)
    (301, 302),    # one clip that was in group 1, slot 1
]


def test_bdc_tc_rows_do_not_depend_on_slot_group_or_neighbour(cuda):
    """A Gram row depends only on its clip's rows of the operands, and the epilogue's summation order is fixed, so a
    clip's BDC vector must not depend on the clip it shares a tile with, the epilogue group that handles it or the
    zero rows next to a lone clip: bit for bit.  Two identical calls must also agree bit for bit."""
    B = 1201
    x = _relu_normal((B, 64, 16, 19), seed=77).to(cuda)
    full, ran = _pool(x, T200)
    assert ran == ["bdc_tc_kernel"]
    again, _ = _pool(x, T200)
    assert torch.equal(full, again)
    for first, end in SLICES:
        part, ran = _pool(x[first:end], T200)
        assert ran == ["bdc_tc_kernel"]
        assert torch.equal(part, full[first:end]), (first, end)


# ------------------------------------------------------------------ backward, including grad log_temp
def _log_temp_terms(x, log_temp, grad_out, triu):
    """fp64 terms t_ij = dA_ij e^t D_ij / (2 A_ij) [B, C, C] whose sum is grad log_temp; dA is the adjoint of the
    double centring applied to grad_out (zero below the diagonal when triu)."""
    B, C = x.shape[:2]
    x = x.double().reshape(B, C, -1)
    g = x @ x.transpose(1, 2)
    d = g.diagonal(dim1=1, dim2=2)
    D = (d[:, :, None] + d[:, None, :] - 2.0 * g).clamp(min=0.0)
    et = math.exp(log_temp)
    A = torch.sqrt(et * D + 1e-5)
    if triu:
        dB = torch.zeros(B, C, C, dtype=torch.float64, device=x.device)
        r, c = torch.triu_indices(C, C, device=x.device)
        dB[:, r, c] = grad_out.double()
    else:
        dB = grad_out.double().reshape(B, C, C)
    dA = dB - dB.mean(dim=2, keepdim=True) - dB.mean(dim=1, keepdim=True) + dB.mean(dim=(1, 2), keepdim=True)
    return dA * et * D / (2.0 * A)


def _check_backward(x, log_temp, triu, seed):
    from audio_fewshot_b200 import ops
    B, C = x.shape[:2]
    out_dim = C * (C + 1) // 2 if triu else C * C
    g = torch.from_numpy(np.random.default_rng(seed).standard_normal((B, out_dim)).astype(np.float32)).to(x.device)

    xg = x.clone().requires_grad_(True)
    tg = torch.full((1, 1), log_temp, device=x.device, requires_grad=True)
    out = ops.bdc_pool(xg, tg, triu=triu)
    out.backward(g)

    xr = x.double().requires_grad_(True)
    tr = torch.full((1, 1), log_temp, dtype=torch.float64, device=x.device, requires_grad=True)
    full = heads.bdcovpool(xr.reshape(B, C, 1, -1), tr)
    want = heads.triuvec(full) if triu else full.reshape(B, -1)
    want.backward(g.double())

    _assert_close(out.detach(), want.detach(), what="forward")
    _assert_close(xg.grad, xr.grad, bar=GRAD_X_BAR, what="grad x")
    terms = _log_temp_terms(x, log_temp, g, triu)
    mag = terms.abs().sum().item()
    assert abs(terms.sum().item() - tr.grad.item()) <= 1e-9 * mag  # the restatement above is what autograd computes
    assert tg.grad.shape == (1, 1)
    err_t = abs(tg.grad.item() - tr.grad.item())
    assert err_t <= GRAD_T_BAR * mag, "grad log_temp %.9g, fp64 %.9g, sum|t| %.3e" % (tg.grad.item(), tr.grad.item(), mag)


BWD_CASES = [(5, C, M, triu) for C in (1, 17, 64) for M in (1, 63, 64, 65, 304) for triu in (True, False)] + [
    (300, 64, 304, True), (300, 64, 64, False), (300, 17, 65, True)]


@pytest.mark.parametrize("B,C,M,triu", BWD_CASES)
def test_bdc_backward_and_log_temperature_gradient(cuda, B, C, M, triu):
    """afs_bdc_bwd against fp64 autograd through the oracle: grad x within 2e-3 of its range, grad log_temp within
    GRAD_T_BAR of the magnitude of the terms it sums (see above).  M runs over the 64-position chunk edges."""
    x = _relu_normal((B, C, M), seed=10000 * B + 100 * C + M).to(cuda)
    _check_backward(x, T200, triu, seed=C + M)


def test_bdc_backward_where_distances_are_exactly_zero(cuda):
    """Channels that are zero after the ReLU give D_ij = 0 exactly, and so do duplicated channels, where torch.clamp's
    subgradient (passed at D = 0) reaches grad x through H_ij X_j.  Inputs are multiples of 1/4, so every Gram entry
    is exact in fp32 and fp64 whatever the summation order, and both sides see D = 0 on the same pairs."""
    B, C, M = 5, 64, 304
    x = np.round(4.0 * np.maximum(np.random.default_rng(8).standard_normal((B, C, M)), 0.0)) / 4.0
    x[:, [3, 17, 40]] = 0.0
    x[:, [50, 51]] = x[:, [10]]
    x = torch.from_numpy(x.astype(np.float32)).to(cuda)
    for triu in (True, False):
        _check_backward(x, T200, triu, seed=9)


# ------------------------------------------------------------------ full-size DeepBDC step
def test_full_size_deepbdc_step(cuda, monkeypatch):
    """BASELINE's DeepBDC config (resnet12Bdc reduce_dim = 64, 5w5s10q, 128 x 157 images) at 12 episodes = 900 images
    = 450 BDC tiles, so CTAs 0-5 run four tiles.  The features BdcPool hands to the kernel are captured; then (a) the
    kernel's BDC of them is within 2e-5 of fp64; (b) an episode slice of them, starting on an odd clip, gives the full
    batch's rows bit for bit; (c) the logits of a 3-episode slice through the whole model are within 1e-5 of the logit
    range of the full step's, with the same argmax (the trunk is cuDNN, whose algorithm may depend on the batch size);
    (d) a second run is bit-identical; (e) the FMA kernel (switch off) gives every query the same argmax."""
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200 import ops
    from audio_fewshot_b200.synthetic import name_seeded_weights_
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    W, S, Q, E = 5, 5, 10, 12
    per, nq = W * (S + Q), W * Q
    torch.manual_seed(4)
    emb = name_seeded_weights_(arch.resnet12Bdc(reduce_dim=64, num_channels=1))
    model = arch.DeepBDC(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=emb,
                         device=cuda).to(cuda).eval()
    images = (torch.randn(E * per, 1, 128, 157, generator=torch.Generator().manual_seed(6)) * 0.7).to(cuda)

    seen = []
    bdc_pool = ops.bdc_pool

    def spy(x, log_temp, triu=True):
        out = bdc_pool(x, log_temp, triu)
        seen.append((x.contiguous().clone(), log_temp.detach().clone(), out))
        return out

    monkeypatch.setattr(ops, "bdc_pool", spy)

    def run(first, n):
        with torch.no_grad():
            return model.set_forward([images[first * per:(first + n) * per], None,
                                      torch.ones(n * nq, dtype=torch.long), n * W * S])[0]

    logits, ran = _bdc_kernels_of(lambda: run(0, E))
    assert ran == ["bdc_tc_kernel"]
    assert logits.shape == (E * nq, W) and torch.isfinite(logits).all()
    feat, t, bdc = seen[-1]
    assert feat.shape[:2] == (E * per, 64) and feat[0, 0].numel() % 4 == 0  # the tensor-core path's shape
    log_temp = t.item()
    assert log_temp == pytest.approx(T200)

    # (a)
    _assert_bdc(bdc, _reference(feat, log_temp), triu=True, what="captured features")
    # (b) episodes 5-7: clip 375 moves from tile slot 1 to slot 0
    part, ran = _pool(feat[5 * per:8 * per], log_temp)
    assert ran == ["bdc_tc_kernel"]
    assert torch.equal(part, bdc[5 * per:8 * per])
    # (c)
    sliced = run(5, 3)
    ref = logits[5 * nq:8 * nq]
    assert (sliced - ref).abs().max().item() <= 1e-5 * logits.abs().max().item()
    assert torch.equal(sliced.argmax(1), ref.argmax(1))
    # (d)
    assert torch.equal(run(0, E), logits)
    assert torch.equal(seen[-1][0], feat) and torch.equal(seen[-1][2], bdc)
    # (e)
    ops.bdc_set_tensor_core(False)
    fma_logits, ran = _bdc_kernels_of(lambda: run(0, E))
    assert ran == ["bdc_kernel"]
    assert torch.equal(fma_logits.argmax(1), logits.argmax(1))
