"""The BDC kernels at C = 128, 192, ..., 640 (csrc/bdc_wide.cu) against a float64 evaluation of the oracle
(oracle.heads.bdcovpool + triuvec, on the GPU, chunked over clips): forward over C, M and both layouts, cancellation
against the reference's own fp32 op sequence, bit-exact independence of batch size, position and the tensor-core
switch, the size edges of the grid and of 32-bit offsets, refusals, the backward with the log-temperature gradient,
and resnet12Bdc / DeepBDC at the reference's default reduce_dim.  Errors are scaled by max|reference|, as in
test_gpu_bdc.py."""
import ctypes
import math
import re

import numpy as np
import pytest
import torch

from oracle import heads

pytestmark = pytest.mark.gpu

T200 = math.log(1.0 / 200.0)  # BdcPool's initial log-temperature
FWD_BAR = 2e-5                # of max|ref|, as test_gpu_bdc.py
GRAD_X_BAR = 2e-3
# grad log_temp = sum over clips and (i, j) of t_ij = dA_ij e^t D_ij / (2 A_ij).  bdc_wide_bwd_tile sums a pair's terms
# with a rounding depth of at most 32 serial FMAs per thread + 5 shuffle levels + 8 warp partials, bdc_wide_dx adds
# the <= 55 pair partials of a clip in order, and torch's sum of the B <= 75 clip values adds at most 75 more: < 175
# roundings, 175 * 2^-24 = 1.0e-5 of sum|t_ij|.  Each term also carries the rounding of the recomputed D and A and of
# the centred dA (sums of up to 640 values of dB): a few 2^-24 of max|dB| per term.  Hence 2e-5 * sum|t_ij|.  A
# scaled or wrong-signed gradient is off by |sum t_ij|; the backward cases draw grad_out correlated with the output,
# so that |sum t_ij| is a sizeable fraction of sum|t_ij|, and _check_backward asserts it is at least 10x the bar.
GRAD_T_BAR = 2e-5
WIDE_FWD = ["bdc_wide_norms", "bdc_wide_gram", "bdc_wide_center"]
WIDE_BWD = ["bdc_wide_norms", "bdc_wide_dbstats", "bdc_wide_bwd_tile", "bdc_wide_dx"]


@pytest.fixture(autouse=True)
def _tensor_core_switch_restored(cuda):
    from audio_fewshot_b200 import ops
    try:
        yield
    finally:
        ops.bdc_set_tensor_core(True)


def _relu_normal(shape, seed):
    return torch.from_numpy(np.maximum(np.random.default_rng(seed).standard_normal(shape), 0.0).astype(np.float32))


def _bdc_kernels_of(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [m.group(1) for e in prof.events() for m in [re.search(r"::(bdc\w*)\(", e.name)] if m]


def _pool(x, log_temp, triu=True, tc=True):
    from audio_fewshot_b200 import ops
    t = torch.full((1, 1), log_temp, device=x.device)
    ops.bdc_set_tensor_core(tc)
    return ops.bdc_pool(x, t, triu=triu)


def _reference(x, log_temp, triu, chunk=64):
    """float64 BDC [B, C(C+1)/2] (triu) or [B, C*C] of x [B, C, ...], on x's device, chunked over clips."""
    B, C = x.shape[:2]
    t = torch.full((1, 1), log_temp, dtype=torch.float64, device=x.device)
    outs = []
    for s in range(0, B, chunk):
        full = heads.bdcovpool(x[s:s + chunk].double().reshape(-1, C, 1, x[0, 0].numel()), t)
        outs.append(heads.triuvec(full) if triu else full.reshape(full.shape[0], -1))
    return torch.cat(outs)


def _assert_close(got, ref, bar=FWD_BAR, what=""):
    scale = ref.abs().max().item()
    err = (got.double() - ref).abs().max().item()
    assert err <= bar * scale, "%s: max error %.3e, max|ref| %.3e, bar %.0e" % (what, err, scale, bar)


# ------------------------------------------------------------------ forward
@pytest.mark.parametrize("C", [128, 192, 256, 640])
@pytest.mark.parametrize("M", [1, 63, 64, 65, 304])
def test_wide_forward_against_fp64(cuda, C, M):
    """Post-ReLU N(0, 1) maps: within 2e-5 of fp64 in both layouts; the triangle is the full output's upper triangle
    bit for bit; the full output is exactly symmetric and double-centred; only the bdc_wide_* kernels ran.  M runs
    over the 32-position Gram chunks and the 64-position dX tiles."""
    B = 3
    x = _relu_normal((B, C, M), seed=10 * C + M).to(cuda)
    ref_full = _reference(x, T200, triu=False)
    scale = ref_full.abs().max().item()
    full, ran = _bdc_kernels_of(lambda: _pool(x, T200, triu=False))
    assert ran == WIDE_FWD
    triu, ran = _bdc_kernels_of(lambda: _pool(x, T200, triu=True))
    assert ran == WIDE_FWD
    _assert_close(full, ref_full, what="full")
    _assert_close(triu, _reference(x, T200, triu=True), what="triu")
    full = full.reshape(B, C, C)
    assert torch.equal(heads.triuvec(full), triu)
    assert torch.equal(full, full.transpose(1, 2))
    assert full.double().mean(dim=1).abs().max().item() <= 1e-4 * scale
    assert full.double().mean(dim=2).abs().max().item() <= 1e-4 * scale


def test_wide_cancellation_is_no_worse_than_the_reference_fp32_sequence(cuda, monkeypatch):
    """x = 5 + 0.2 relu(N): D_ij = n_i + n_j - 2 G_ij is ~1/1000 of the Gram entries, so fp32 rounding of G is
    amplified and neither side meets 2e-5.  The kernel must be no worse than 2x the reference's own op sequence
    (heads.bdcovpool in float32 on the GPU, TF32 off), plus 1e-6 of scale."""
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    B, C, M = 7, 640, 304
    g = np.random.default_rng(640)
    x = torch.from_numpy((5.0 + 0.2 * np.maximum(g.standard_normal((B, C, M)), 0.0)).astype(np.float32)).to(cuda)
    ref = _reference(x, T200, triu=True)
    scale = ref.abs().max().item()
    t32 = torch.full((1, 1), T200, dtype=torch.float32, device=cuda)
    seq = heads.triuvec(heads.bdcovpool(x.reshape(B, C, 1, M), t32))
    out = _pool(x, T200)
    err = (out.double() - ref).abs().max().item()
    err_seq = (seq.double() - ref).abs().max().item()
    assert err <= 2.0 * err_seq + 1e-6 * scale, (err / scale, err_seq / scale)


# ------------------------------------------------------------------ independence and repeatability
SLICES = [(1, 1201), (600, 601), (1200, 1201), (297, 1000), (0, 55)]


def test_wide_rows_do_not_depend_on_batch_position_switch_or_layout(cuda):
    """1201 clips of 640 x 16 x 19: slices give the full call's rows bit for bit, a second call is bit-identical, the
    tensor-core switch changes nothing, and a channels-last input gives what its contiguous copy gives."""
    B = 1201
    x = _relu_normal((B, 640, 16, 19), seed=77).to(cuda)
    full = _pool(x, T200)
    assert torch.equal(_pool(x, T200), full)
    assert torch.equal(_pool(x, T200, tc=False), full)
    for first, end in SLICES:
        assert torch.equal(_pool(x[first:end], T200), full[first:end]), (first, end)
    xcl = x[:64].contiguous(memory_format=torch.channels_last)
    assert not xcl.is_contiguous()
    assert torch.equal(_pool(xcl, T200), full[:64])
    full_sq = _pool(x[:64], T200, triu=False)
    assert torch.equal(_pool(xcl, T200, triu=False), full_sq)
    _assert_close(full[1190:], _reference(x[1190:], T200, triu=True))


@pytest.mark.parametrize("C,B", [(128, 70000), (640, 10500)])
def test_wide_size_edges(cuda, C, B):
    """C = 128, B = 70 000: 210 000 Gram CTAs, more than 65 535 clips.  C = 640, B = 10 500: the triangle output has
    2.15e9 elements, past 2^31.  The last clips must equal the same clips run alone, bit for bit."""
    M = 4
    x = _relu_normal((B, C, M), seed=B).to(cuda)
    out = _pool(x, T200)
    assert out.shape == (B, C * (C + 1) // 2)
    if C == 640:
        assert out.numel() > 2 ** 31
    tail = x[B - 3:].clone()
    assert torch.equal(out[B - 3:], _pool(tail, T200))
    _assert_close(out[B - 3:], _reference(tail, T200, triu=True))
    del out
    torch.cuda.empty_cache()


def test_wide_empty_batch_is_a_no_op(cuda):
    from audio_fewshot_b200 import ops
    x = torch.empty(0, 640, 16, 19, device=cuda)
    out = _pool(x, T200)
    assert out.shape == (0, 640 * 641 // 2)
    xg = x.clone().requires_grad_(True)
    tg = torch.full((1, 1), T200, device=cuda, requires_grad=True)
    ops.bdc_pool(xg, tg).sum().backward()
    assert xg.grad.shape == x.shape and tg.grad.item() == 0.0


# ------------------------------------------------------------------ refusals
@pytest.mark.parametrize("C", [96, 127, 704, 1024])
def test_wide_other_channel_counts_are_refused(cuda, C):
    from audio_fewshot_b200 import _lib, ops
    x = torch.ones(2, C, 8, device=cuda)
    t = torch.full((1, 1), T200, device=cuda)
    for tc in (True, False):
        ops.bdc_set_tensor_core(tc)
        with pytest.raises(_lib.AfsError):
            ops.bdc_pool(x, t)


def test_wide_short_workspace_is_refused(cuda):
    from audio_fewshot_b200 import _lib, ops
    h = _lib.lib()
    B, C, M = 3, 256, 16
    x = _relu_normal((B, C, M), seed=5).to(cuda)
    t = torch.full((1, 1), T200, device=cuda)
    out = torch.empty(B, C * (C + 1) // 2, device=cuda)
    for backward in (0, 1):
        need = int(h.afs_bdc_wide_workspace_bytes(B, C, backward))
        ws = torch.empty(need, dtype=torch.uint8, device=cuda)
        p = ops._ptr
        if backward:
            gx, gt = torch.empty_like(x), torch.empty(B, device=cuda)
            r = h.afs_bdc_wide_bwd(p(x), B, C, M, p(t), 1, p(out), p(gx), p(gt), p(ws), need - 4, ops._stream())
        else:
            r = h.afs_bdc_wide_fwd(p(x), B, C, M, p(t), 1, p(out), p(ws), need - 4, ops._stream())
        assert r == -4  # AFS_ERR_WORKSPACE
        assert h.afs_bdc_wide_fwd(p(x), B, C, M, p(t), 1, p(out), ctypes.c_void_p(ws.data_ptr() + 4), need,
                                  ops._stream()) == -4


# ------------------------------------------------------------------ backward
def _log_temp_terms(x, log_temp, grad_out, triu):
    """fp64 terms t_ij = dA_ij e^t D_ij / (2 A_ij) [B, C, C] whose sum is grad log_temp."""
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
    with torch.no_grad():
        out0 = ops.bdc_pool(x, torch.full((1, 1), log_temp, device=x.device), triu=triu)
    noise = torch.from_numpy(np.random.default_rng(seed).standard_normal(tuple(out0.shape)).astype(np.float32))
    g = out0 / out0.abs().max() + 0.1 * noise.to(x.device)  # correlated with the output: see GRAD_T_BAR

    xg = x.clone().requires_grad_(True)
    tg = torch.full((1, 1), log_temp, device=x.device, requires_grad=True)
    out, ran = _bdc_kernels_of(lambda: ops.bdc_pool(xg, tg, triu=triu))
    assert ran == WIDE_FWD
    _, ran = _bdc_kernels_of(lambda: out.backward(g))
    assert ran == WIDE_BWD

    xr = x.double().requires_grad_(True)
    tr = torch.full((1, 1), log_temp, dtype=torch.float64, device=x.device, requires_grad=True)
    full = heads.bdcovpool(xr.reshape(B, C, 1, -1), tr)
    want = heads.triuvec(full) if triu else full.reshape(B, -1)
    want.backward(g.double())

    _assert_close(out.detach(), want.detach(), what="forward")
    _assert_close(xg.grad, xr.grad, bar=GRAD_X_BAR, what="grad x")
    terms = _log_temp_terms(x, log_temp, g, triu)
    mag = terms.abs().sum().item()
    assert abs(terms.sum().item() - tr.grad.item()) <= 1e-9 * mag
    assert abs(tr.grad.item()) >= 10 * GRAD_T_BAR * mag, "a sign or scale error would not clear the bar 10x"
    assert tg.grad.shape == (1, 1)
    err_t = abs(tg.grad.item() - tr.grad.item())
    assert err_t <= GRAD_T_BAR * mag, "grad log_temp %.9g, fp64 %.9g, sum|t| %.3e" % (tg.grad.item(), tr.grad.item(), mag)


@pytest.mark.parametrize("B", [5, 75])
@pytest.mark.parametrize("C", [128, 640])
@pytest.mark.parametrize("M", [1, 65, 304])
@pytest.mark.parametrize("triu", [True, False])
def test_wide_backward_and_log_temperature_gradient(cuda, B, C, M, triu):
    x = _relu_normal((B, C, M), seed=10000 * B + 100 * C + M).to(cuda)
    _check_backward(x, T200, triu, seed=C + M)


def test_wide_backward_where_distances_are_exactly_zero(cuda):
    """Zero channels and duplicated channels give D_ij = 0 exactly; multiples of 1/4 keep every Gram entry exact in fp32
    and fp64, so both sides see D = 0 on the same pairs (see test_gpu_bdc.py)."""
    B, C, M = 5, 640, 304
    x = np.round(4.0 * np.maximum(np.random.default_rng(8).standard_normal((B, C, M)), 0.0)) / 4.0
    x[:, [3, 17, 130, 401, 639]] = 0.0
    x[:, [50, 51, 300, 600]] = x[:, [10]]
    x = torch.from_numpy(x.astype(np.float32)).to(cuda)
    for triu in (True, False):
        _check_backward(x, T200, triu, seed=9)


# ------------------------------------------------------------------ model level
def _deepbdc(cuda, reduce_dim=None, E=2, seed=4):
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.synthetic import name_seeded_weights_
    torch.manual_seed(seed)
    kw = {} if reduce_dim is None else {"reduce_dim": reduce_dim}
    emb = name_seeded_weights_(arch.resnet12Bdc(num_channels=1, **kw))
    return arch.DeepBDC(way_num=5, shot_num=5, query_num=10, test_way=5, test_shot=5, test_query=10, emb_func=emb,
                        device=cuda).to(cuda)


def _spy(monkeypatch):
    from audio_fewshot_b200 import ops
    seen = []
    bdc_pool = ops.bdc_pool

    def spy(x, log_temp, triu=True):
        out = bdc_pool(x, log_temp, triu)
        seen.append((x.detach().contiguous().clone(), log_temp.detach().clone(), out))
        return out

    monkeypatch.setattr(ops, "bdc_pool", spy)
    return seen


def _images(n, seed):
    return (torch.randn(n, 1, 128, 157, generator=torch.Generator().manual_seed(seed)) * 0.7)


@pytest.mark.parametrize("reduce_dim", [None, 128, 256])
def test_deepbdc_set_forward_at_wide_reduce_dim(cuda, monkeypatch, reduce_dim):
    """resnet12Bdc(num_channels=1) at the reference's default reduce_dim (640, no conv_dr_block) and at 128, 256:
    DeepBDC.set_forward on 2 episodes of 5w5s10q.  The BDC of the captured features is within the bar of fp64, and
    the logits are within 1e-3 of the fp64 head's on the fp64 BDC, with the same argmax wherever fp64's top two are
    further apart than that."""
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    W, S, Q, E = 5, 5, 10, 2
    C = 640 if reduce_dim is None else reduce_dim
    model = _deepbdc(cuda, reduce_dim).eval()
    seen = _spy(monkeypatch)
    images = _images(E * W * (S + Q), 6).to(cuda)
    with torch.no_grad():
        logits = model.set_forward([images, None, torch.ones(E * W * Q, dtype=torch.long), E * W * S])[0]
    feat, t, bdc = seen[-1]
    assert feat.shape[:2] == (E * W * (S + Q), C) and torch.isfinite(logits).all()
    ref = _reference(feat, t.item(), triu=True)
    _assert_close(bdc, ref, what="captured features")
    want = heads.deepbdc_forward(ref.cpu(), W, S, Q, torch.ones(E * W * Q, dtype=torch.long), E * W * S)[0]
    logits = logits.cpu()
    scale = want.abs().max().item()
    assert (logits.double() - want).abs().max().item() <= 1e-3 * scale
    top2 = want.topk(2, dim=1).values
    clear = (top2[:, 0] - top2[:, 1]) > 2e-3 * scale
    assert torch.equal(logits.argmax(1)[clear], want.argmax(1)[clear])


def test_deepbdc_training_step_at_the_default_reduce_dim(cuda):
    """set_forward_loss + backward at reduce_dim 640 on one episode: the BDC backward runs and the gradients of the
    trunk's last convolution and of the temperature are finite and non-zero."""
    W, S, Q = 5, 5, 10
    model = _deepbdc(cuda).train()
    images = _images(W * (S + Q), 9).to(cuda)
    target = torch.arange(W).repeat_interleave(S + Q)
    _, ran = _bdc_kernels_of(lambda: model.set_forward_loss([images, target])[2].backward())
    assert ran == WIDE_FWD + WIDE_BWD
    last_conv = [m for m in model.emb_func.layer4.modules() if isinstance(m, torch.nn.Conv2d)][-1]
    for name, grad in (("last conv", last_conv.weight.grad), ("temperature", model.emb_func.bdc_pool.temperature.grad)):
        assert grad is not None and torch.isfinite(grad).all() and grad.abs().max().item() > 0, name


def test_full_size_deepbdc_step_at_the_default_reduce_dim(cuda, monkeypatch):
    """BASELINE's DeepBDC shape (5w5s10q, 128 x 157 images) at reduce_dim 640 and 12 episodes = 900 clips = 49 500
    Gram tiles: (a) the kernel's BDC of the captured features is within 2e-5 of fp64; (b) an episode slice of them,
    starting on an odd clip, gives the full batch's rows bit for bit; (c) the logits of a 3-episode slice through the
    whole model are within 1e-5 of the full step's logit range, with the same argmax; (d) a second run is
    bit-identical."""
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    W, S, Q, E = 5, 5, 10, 12
    per, nq = W * (S + Q), W * Q
    model = _deepbdc(cuda).eval()
    images = _images(E * per, 6).to(cuda)
    seen = _spy(monkeypatch)

    def run(first, n):
        with torch.no_grad():
            return model.set_forward([images[first * per:(first + n) * per], None,
                                      torch.ones(n * nq, dtype=torch.long), n * W * S])[0]

    logits, ran = _bdc_kernels_of(lambda: run(0, E))
    assert ran == WIDE_FWD
    assert logits.shape == (E * nq, W) and torch.isfinite(logits).all()
    feat, t, bdc = seen[-1]
    assert feat.shape[:2] == (E * per, 640)
    log_temp = t.item()
    # (a)
    _assert_close(bdc, _reference(feat, log_temp, triu=True), what="captured features")
    # (b) episodes 5-7, first clip 375
    assert torch.equal(_pool(feat[5 * per:8 * per], log_temp), bdc[5 * per:8 * per])
    # (c)
    sliced = run(5, 3)
    ref = logits[5 * nq:8 * nq]
    assert (sliced - ref).abs().max().item() <= 1e-5 * logits.abs().max().item()
    assert torch.equal(sliced.argmax(1), ref.argmax(1))
    # (d)
    assert torch.equal(run(0, E), logits)
    assert torch.equal(seen[-1][0], feat) and torch.equal(seen[-1][2], bdc)
