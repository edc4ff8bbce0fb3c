"""GPU parity of the drop-in classes: backbones (incl. the fused Conv64F inference path) against the
reference's golden features, set_forward / set_forward_loss of ProtoNet, DN4, DeepBDC against the oracle
drivers on identical features, and the waveform -> logits pipeline (plain and CUDA-graph)."""
import math

import numpy as np
import pytest
import torch

from oracle import backbones as obb
from oracle import cases, heads

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _fp32_convs():
    """Backbone parity is asserted with exact-fp32 convolutions (the reference's TF32 default is not bit-stable)."""
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _net(cuda, name):
    from audio_fewshot_b200 import model as arch
    ctor, kwargs = cases.BACKBONE_CASES[name]
    torch.manual_seed(0)
    net = getattr(arch, ctor)(**kwargs).eval()
    cases.perturb_bn_(net)
    return net.to(cuda)


@pytest.mark.parametrize("name", sorted(cases.BACKBONE_CASES))
def test_backbones_match_reference_golden_on_gpu(cuda, golden, name):
    g = golden("backbones.npz")
    net = _net(cuda, name)
    x = torch.from_numpy(cases.backbone_input()).to(cuda)
    with torch.no_grad():
        y = net(x)
    want = g[name + "/out"]
    assert tuple(y.shape) == want.shape
    assert np.abs(y.float().cpu().numpy() - want).max() <= 2e-4 * np.abs(want).max()


@pytest.mark.parametrize("name", ["conv64f_flat", "conv64f_dn4"])
def test_conv64f_inference_path_equals_module_graph(cuda, name):
    """The fused path (conv1 kernel + folded cuDNN blocks) against the plain module graph on a bigger batch."""
    from audio_fewshot_b200 import ops
    net = _net(cuda, name)
    x = torch.from_numpy((np.random.default_rng(5).standard_normal((37, 1, 128, 157)) * 0.7).astype(np.float32)).to(cuda)
    n0 = ops.launch_count()
    with torch.no_grad():
        fast = net(x)
    assert ops.launch_count() > n0  # the conv1 / pooling kernels ran
    n1 = ops.launch_count()
    with torch.enable_grad():  # grad mode -> plain graph (the reference's op sequence)
        slow = net(x).detach()
    assert ops.launch_count() == n1
    assert fast.shape == slow.shape
    assert (fast - slow).abs().max().item() <= 2e-5 * slow.abs().max().item()


def test_conv1_kernel_odd_sizes_and_leaky(cuda):
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(8)
    for (N, H, Wd, slope) in [(3, 128, 157, 0.0), (2, 7, 11, 0.2), (1, 3, 3, 0.0), (130, 9, 10, 0.1)]:
        x = torch.from_numpy(rng.standard_normal((N, 1, H, Wd)).astype(np.float32)).to(cuda)
        w = rng.standard_normal((64, 9)).astype(np.float32) * 0.3
        w[5] *= -1.0  # a negative BatchNorm scale folded in
        b = rng.standard_normal(64).astype(np.float32)
        got = ops.conv1_bn_act_pool3(x, w, b, slope)
        assert got.is_contiguous(memory_format=torch.channels_last) or got.shape[2] * got.shape[3] == 1
        conv = torch.nn.functional.conv2d(x.double(), torch.from_numpy(w).to(cuda).double().view(64, 1, 3, 3),
                                          torch.from_numpy(b).to(cuda).double(), padding=1)
        want = torch.nn.functional.max_pool2d(torch.nn.functional.leaky_relu(conv, slope), 3, 3)
        assert got.shape == want.shape
        assert (got.double() - want).abs().max().item() < 1e-5


def test_conv1_tensor_core_stem_matches_fp32_stem_at_tf32_tolerance(cuda):
    """csrc/conv1_tc.cu (tcgen05 TF32, max-pool over TMEM accumulators) against csrc/conv1.cu (exact fp32)."""
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(18)
    for (N, H, Wd, slope) in [(3, 128, 157, 0.0), (2, 7, 11, 0.2), (1, 3, 3, 0.0), (130, 9, 10, 0.1)]:
        x = torch.from_numpy(rng.standard_normal((N, 1, H, Wd)).astype(np.float32)).to(cuda)
        w = rng.standard_normal((64, 9)).astype(np.float32) * 0.3
        w[5] *= -1.0
        b = rng.standard_normal(64).astype(np.float32)
        exact = ops.conv1_bn_act_pool3(x, w, b, slope)
        tc = ops.conv1_bn_act_pool3(x, w, b, slope, tf32=True)
        assert tc.shape == exact.shape
        assert (tc - exact).abs().max().item() <= 2e-3 * exact.abs().max().item()  # TF32 operands: ~1e-3 relative


@pytest.mark.parametrize("N,H,Wd,slope,pool", [
    (5, 42, 52, 0.0, True),     # Conv64F block 2: 6 rows per tile, three 128-row accumulators
    (3, 14, 17, 0.0, True),     # block 3: two rows of the image fall below the last pooling window
    (2, 14, 17, 0.2, False),    # un-pooled, LeakyReLU, ragged last tile
    (7, 4, 5, 0.0, False),      # block 4 of the DN4 backbone: one tiny tile per image
    (2, 4, 5, 0.0, True),
    (2, 10, 61, 0.1, False),    # widest supported row (HP = 63): 5 rows per tile, ring at the shared-memory limit
    (300, 42, 52, 0.0, True),   # more tiles than SMs: persistent loop, ring wrap-around, both accumulator sets
])
def test_conv3x3_block_tensor_core_kernel(cuda, N, H, Wd, slope, pool):
    """csrc/conv3_tc.cu (tcgen05 TF32 implicit GEMM + folded BN + activation + max-pool) against the fp64 op
    sequence conv2d -> leaky_relu -> max_pool2d.  Tolerance: TF32 operands (weights rounded to nearest,
    activations truncated by the MMA like cuDNN's TF32 convolutions), K = 576 -> <= 2e-3 of the output range."""
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(N * 1000 + H * 10 + Wd)
    x = torch.from_numpy(rng.standard_normal((N, 64, H, Wd)).astype(np.float32)).to(cuda)
    x = x.contiguous(memory_format=torch.channels_last)
    w = torch.from_numpy((rng.standard_normal((64, 64, 3, 3)) * 0.06).astype(np.float32)).to(cuda)
    w[5] *= -1.0
    b = torch.from_numpy(rng.standard_normal(64).astype(np.float32)).to(cuda)
    packed = torch.from_numpy(ops.conv3x3_c64_pack_weights(w)).to(cuda)
    got = ops.conv3x3_c64_bn_act(x, packed, b, slope, pool=pool)
    want = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(x.double(), w.double(), b.double(), padding=1), slope)
    if pool:
        want = torch.nn.functional.max_pool2d(want, 3, 3)
    assert got.shape == want.shape
    assert got.is_contiguous(memory_format=torch.channels_last) or got.shape[2] * got.shape[3] == 1
    err = (got.double() - want).abs().max().item()
    assert err <= 2e-3 * want.abs().max().item(), err
    # the packed weights are exactly the round-to-nearest TF32 values, so with TF32-exact activations the kernel
    # must agree with an fp32-accumulated convolution to fp32 rounding
    xq = (x.view(torch.int32) & ~0x1FFF).view(torch.float32)
    wq = ((w.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)
    got_q = ops.conv3x3_c64_bn_act(xq, packed, b, slope, pool=pool)
    want_q = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(xq.double(), wq.double(), b.double(), padding=1), slope)
    if pool:
        want_q = torch.nn.functional.max_pool2d(want_q, 3, 3)
    assert (got_q.double() - want_q).abs().max().item() <= 2e-5 * want_q.abs().max().item()


@pytest.mark.parametrize("N,H,Wd,slope,pool,out_dtype", [
    (5, 42, 52, 0.0, True, torch.bfloat16),     # Conv64F block 2 of the bf16 path
    (3, 14, 17, 0.0, True, torch.float32),      # block 3: fp32 output for block 4
    (2, 14, 17, 0.2, False, torch.bfloat16),    # un-pooled, LeakyReLU, ragged last tile
    (7, 4, 5, 0.0, False, torch.float32),
    (2, 10, 61, 0.1, False, torch.float32),     # widest supported row
    (300, 42, 52, 0.0, True, torch.bfloat16),   # more tiles than SMs: 8-stage ring wrap-around, both accumulator sets
])
def test_conv3x3_block_bf16_kernel(cuda, N, H, Wd, slope, pool, out_dtype):
    """The separately stated bf16 variant of csrc/conv3_tc.cu (kind::f16 MMAs, K = 16, fp32 accumulation).  With bf16
    inputs every product is exact in fp32, so against an fp64 convolution of the SAME bf16 activations and bf16-rounded
    weights only the accumulation order differs: <= 2e-5 of the output range for the fp32 output, one bf16 rounding
    (2^-8 relative) more for the bf16 output.  Repeated launches are bit-identical."""
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(N * 1000 + H * 10 + Wd + 1)
    x = torch.from_numpy(rng.standard_normal((N, 64, H, Wd)).astype(np.float32)).to(cuda).to(torch.bfloat16)
    x = x.contiguous(memory_format=torch.channels_last)
    w = torch.from_numpy((rng.standard_normal((64, 64, 3, 3)) * 0.06).astype(np.float32)).to(cuda)
    w[5] *= -1.0
    b = torch.from_numpy(rng.standard_normal(64).astype(np.float32)).to(cuda)
    packed = torch.from_numpy(ops.conv3x3_c64_pack_weights_bf16(w)).to(cuda).view(torch.bfloat16)
    got = ops.conv3x3_c64_bn_act_bf16(x, packed, b, slope, pool=pool, out_dtype=out_dtype)
    wq = w.to(torch.bfloat16).double()
    want = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(x.double(), wq, b.double(), padding=1), slope)
    if pool:
        want = torch.nn.functional.max_pool2d(want, 3, 3)
    assert got.shape == want.shape and got.dtype == out_dtype
    assert got.is_contiguous(memory_format=torch.channels_last) or got.shape[2] * got.shape[3] == 1
    err = (got.double() - want).abs().max().item()
    tol = (2e-5 if out_dtype == torch.float32 else 2.0 ** -8) * want.abs().max().item()
    assert err <= tol, (err, tol)
    assert torch.equal(got, ops.conv3x3_c64_bn_act_bf16(x, packed, b, slope, pool=pool, out_dtype=out_dtype))


def test_stem_bf16_output_is_the_rounded_fp32_output(cuda):
    """csrc/conv1_tc.cu with bf16 output does the same TF32 arithmetic and rounds to nearest even at the store."""
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(21)
    for (N, H, Wd, slope) in [(3, 128, 157, 0.0), (130, 9, 10, 0.1)]:
        x = torch.from_numpy(rng.standard_normal((N, 1, H, Wd)).astype(np.float32)).to(cuda)
        w = rng.standard_normal((64, 9)).astype(np.float32) * 0.3
        b = rng.standard_normal(64).astype(np.float32)
        f32 = ops.conv1_bn_act_pool3(x, w, b, slope, tf32=True)
        b16 = ops.conv1_bn_act_pool3(x, w, b, slope, tf32=True, out_dtype=torch.bfloat16)
        assert b16.dtype == torch.bfloat16 and b16.is_contiguous(memory_format=torch.channels_last)
        assert torch.equal(b16, f32.to(torch.bfloat16))


def test_conv64f_bf16_path_is_close_and_keeps_predictions(cuda):
    """Conv64F(precision='bf16') -- stated separately from the parity path: features within 3e-2 of the feature range
    of the TF32 path, and the ProtoNet predictions of well separated synthetic episodes unchanged."""
    from audio_fewshot_b200 import model as arch
    net = _net(cuda, "conv64f_flat")
    x = torch.from_numpy((np.random.default_rng(7).standard_normal((24, 1, 128, 157)) * 0.7).astype(np.float32)).to(cuda)
    with torch.no_grad():
        net.stem_tf32, net.block_tc = True, True
        ref = net(x)
        net.precision = "bf16"
        fast = net(x)
        assert torch.equal(fast, net(x))
    assert fast.dtype == torch.float32 and fast.shape == ref.shape
    assert (fast - ref).abs().max().item() <= 3e-2 * ref.abs().max().item()
    assert not torch.equal(fast, ref)  # the bf16 kernels did run


def test_conv64f_tensor_core_blocks_match_fp32_path(cuda):
    """Whole Conv64F inference path with the tcgen05 stem and blocks (TF32) against the exact-fp32 path."""
    net = _net(cuda, "conv64f_flat")
    x = torch.from_numpy((np.random.default_rng(6).standard_normal((24, 1, 128, 157)) * 0.7).astype(np.float32)).to(cuda)
    with torch.no_grad():
        exact = net(x)
        net.stem_tf32, net.block_tc = True, True
        fast = net(x)
    assert (fast - exact).abs().max().item() <= 5e-3 * exact.abs().max().item()


@pytest.mark.parametrize("name", ["resnet12", "resnet12bdc"])
def test_resnet12_inference_path_equals_module_graph(cuda, name):
    """Folded channels-last trunk (cuDNN convolutions + add_bias_act_pool kernels) against the plain module graph."""
    from audio_fewshot_b200 import ops
    net = _net(cuda, name)
    x = torch.from_numpy((np.random.default_rng(9).standard_normal((5, 1, 128, 157)) * 0.7).astype(np.float32)).to(cuda)
    n0 = ops.launch_count()
    with torch.no_grad():
        fast = net(x)
    assert ops.launch_count() >= n0 + 12  # 3 kernels per BasicBlock
    net.fast_eval = False
    with torch.no_grad():
        slow = net(x)
    assert fast.shape == slow.shape
    assert (fast - slow).abs().max().item() <= 1e-4 * slow.abs().max().item()


def test_add_bias_act_pool_bf16_kernel(cuda):
    """csrc/pool.cu, bf16 operands: fp32 arithmetic on the bf16 inputs, one rounding at the bf16 store, none at the
    fp32 store; in place for k == 1."""
    from audio_fewshot_b200 import ops
    F = torch.nn.functional
    for (shape, k, slope, with_b, with_bias, odt) in [((3, 64, 128, 157), 2, 0.1, True, True, torch.bfloat16),
                                                      ((2, 160, 64, 78), 2, 0.1, True, True, torch.bfloat16),
                                                      ((2, 640, 16, 19), 1, 0.1, True, True, torch.float32),
                                                      ((2, 8, 7, 9), 3, 0.0, False, True, torch.float32),
                                                      ((2, 64, 5, 6), 1, 0.0, False, False, torch.bfloat16)]:
        a = torch.randn(shape, device=cuda).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        b = torch.randn(shape, device=cuda).to(torch.bfloat16).contiguous(memory_format=torch.channels_last) if with_b else None
        bias = torch.randn(shape[1], device=cuda) if with_bias else None
        want = a.float() if b is None else a.float() + b.float()
        if bias is not None:
            want = want + bias.view(1, -1, 1, 1)
        want = F.leaky_relu(want, slope)
        if k > 1:
            want = F.max_pool2d(want, k, k)
        got = ops.add_bias_act_pool_bf16(a, b, bias, slope, k, out_dtype=odt)
        assert got.shape == want.shape and got.dtype == odt
        if odt == torch.float32:
            assert (got - want).abs().max().item() <= 1e-6 * max(want.abs().max().item(), 1.0)
        else:
            assert torch.equal(got, want.to(torch.bfloat16))
        if k == 1 and odt == torch.bfloat16:
            a2 = a.clone(memory_format=torch.channels_last)
            r = ops.add_bias_act_pool_bf16(a2, b, bias, slope, 1, inplace=True)
            assert r.data_ptr() == a2.data_ptr() and torch.equal(r, got)


@pytest.mark.parametrize("name", ["resnet12", "resnet12bdc"])
def test_resnet12_bf16_trunk_is_close_to_the_parity_path(cuda, name):
    """ResNet.precision = 'bf16' (stated separately from the parity path): bf16 cuDNN convolutions + the bf16 tail
    kernel; features stay within 5e-2 of the fp32 path's feature range, fp32 output, our kernels on the path."""
    from audio_fewshot_b200 import ops
    net = _net(cuda, name)
    x = torch.from_numpy((np.random.default_rng(10).standard_normal((5, 1, 128, 157)) * 0.7).astype(np.float32)).to(cuda)
    with torch.no_grad():
        ref = net(x)
        net.precision = "bf16"
        n0 = ops.launch_count()
        fast = net(x)
        assert ops.launch_count() >= n0 + 12
    assert fast.dtype == torch.float32 and fast.shape == ref.shape
    assert not torch.equal(fast, ref)
    assert (fast - ref).abs().max().item() <= 5e-2 * ref.abs().max().item()


def test_add_bias_act_pool_kernel(cuda):
    from audio_fewshot_b200 import ops
    F = torch.nn.functional
    for (shape, k, slope, with_b, with_bias) in [((3, 64, 128, 157), 2, 0.1, True, True), ((2, 160, 64, 78), 2, 0.1, True, True),
                                                 ((2, 640, 16, 19), 1, 0.1, True, True), ((2, 8, 7, 9), 3, 0.0, False, True),
                                                 ((1, 4, 2, 2), 2, 0.3, True, False), ((2, 64, 5, 6), 1, 0.0, False, False)]:
        a = torch.randn(shape, device=cuda).contiguous(memory_format=torch.channels_last)
        b = torch.randn(shape, device=cuda).contiguous(memory_format=torch.channels_last) if with_b else None
        bias = torch.randn(shape[1], device=cuda) if with_bias else None
        want = a if b is None else a + b
        if bias is not None:
            want = want + bias.view(1, -1, 1, 1)
        want = F.leaky_relu(want, slope)
        if k > 1:
            want = F.max_pool2d(want, k, k)
        got = ops.add_bias_act_pool(a, b, bias, slope, k)
        assert got.shape == want.shape and torch.allclose(got, want, atol=1e-6, rtol=1e-6)
        if k == 1:
            a2 = a.clone(memory_format=torch.channels_last)
            r = ops.add_bias_act_pool(a2, b, bias, slope, 1, inplace=True)
            assert r.data_ptr() == a2.data_ptr() and torch.allclose(a2, want, atol=1e-6, rtol=1e-6)


def test_maxpool3_channels_last_matches_torch(cuda):
    from audio_fewshot_b200 import ops
    for shape in [(5, 64, 42, 52), (3, 64, 14, 17), (2, 8, 3, 3), (1, 64, 4, 5)]:
        x = torch.randn(shape, device=cuda).contiguous(memory_format=torch.channels_last)
        got = ops.maxpool3_channels_last(x)
        want = torch.nn.functional.max_pool2d(x, 3, 3)
        assert got.shape == want.shape and torch.equal(got, want)


def test_folded_weights_follow_parameter_updates(cuda):
    net = _net(cuda, "conv64f_flat")
    x = torch.from_numpy(cases.backbone_input()).to(cuda)
    with torch.no_grad():
        a = net(x).clone()
        net.layer1[0].weight.mul_(1.5)
        net.logits[2].bias.add_(1.0)
        b = net(x)
        with torch.enable_grad():
            want = net(x).detach()
    assert not torch.allclose(a, b)
    assert (b - want).abs().max().item() <= 2e-5 * want.abs().max().item()


# ------------------------------------------------------------------------------------------ set_forward
def _ragged(E, W, Q, seed):
    return np.random.default_rng(seed).integers(1, 4, size=E * W * Q).astype(np.int64)


class _Feat(torch.nn.Module):
    """emb_func stand-in: the 'image' rows already are the features (heads are tested on identical inputs)."""

    def forward(self, x):
        return x


@pytest.mark.parametrize("E,W,S,Q,D,distance", [(3, 5, 5, 4, 1600, "euclidean"), (2, 5, 1, 15, 640, "cos_sim")])
def test_protonet_set_forward_matches_oracle(cuda, E, W, S, Q, D, distance):
    from audio_fewshot_b200 import model as arch
    rep = _ragged(E, W, Q, 3)
    N = E * W * S + int(rep.sum())
    feat = torch.from_numpy(np.random.default_rng(1).standard_normal((N, D)).astype(np.float32))
    m = arch.ProtoNet(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=_Feat(),
                      device=cuda, distance=distance).to(cuda).eval()
    with torch.no_grad():
        out, acc = m([feat, torch.zeros(N), torch.from_numpy(rep), E * W * S])
    want, want_acc, _ = heads.proto_forward(feat, W, S, Q, torch.from_numpy(rep), E * W * S, distance)
    assert out.shape == want.shape
    assert (out.cpu() - want).abs().max().item() <= 1e-3 * want.abs().max().item()
    assert torch.equal(out.cpu().argmax(1), want.argmax(1))
    assert acc.item() == pytest.approx(want_acc.item(), abs=1e-4)


def test_dn4_set_forward_matches_oracle(cuda):
    from audio_fewshot_b200 import model as arch
    E, W, S, Q, C, H, Wd = 2, 5, 5, 3, 64, 4, 5
    rep = _ragged(E, W, Q, 4)
    N = E * W * S + int(rep.sum())
    feat = torch.from_numpy(np.abs(np.random.default_rng(2).standard_normal((N, C, H, Wd))).astype(np.float32))
    m = arch.DN4(n_k=3, way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=_Feat(),
                 device=cuda).to(cuda).eval()
    with torch.no_grad():
        out, acc = m([feat, torch.zeros(N), torch.from_numpy(rep), E * W * S])
    want, want_acc, _ = heads.dn4_forward(feat, W, S, Q, torch.from_numpy(rep), E * W * S, 3)
    assert (out.cpu() - want).abs().max().item() <= 1e-3 * want.abs().max().item()
    assert torch.equal(out.cpu().argmax(1), want.argmax(1))
    assert acc.item() == pytest.approx(want_acc.item(), abs=1e-4)


@pytest.mark.parametrize("S", [1, 5])
def test_deepbdc_set_forward_and_energy_match_oracle(cuda, S, tmp_path, monkeypatch):
    from audio_fewshot_b200 import model as arch
    monkeypatch.chdir(tmp_path)  # the energy branch appends to ./test_uncertainty.npy like the reference
    E, W, Q, D = 2, 5, 4, 2080
    rep = _ragged(E, W, Q, 6)
    N = E * W * S + int(rep.sum())
    feat = torch.from_numpy((np.random.default_rng(7).standard_normal((N, D)) * 0.1).astype(np.float32))
    m = arch.DeepBDC(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=_Feat(),
                     device=cuda).to(cuda).eval()
    batch = [feat, torch.zeros(N), torch.from_numpy(rep), E * W * S]
    with torch.no_grad():
        out, acc = m(batch)
        out5 = m.set_forward(batch, update_threshold=True, enhance_classification_via_energy=True)
    want, want_acc, _, _ = heads.deepbdc_forward(feat, W, S, Q, torch.from_numpy(rep), E * W * S)
    assert (out.cpu() - want).abs().max().item() <= 1e-3 * want.abs().max().item()
    assert torch.equal(out.cpu().argmax(1), want.argmax(1))
    assert acc.item() == pytest.approx(want_acc.item(), abs=1e-4)
    assert len(out5) == 5
    en = heads.energy_score(want, torch.from_numpy(rep)).numpy()
    np.testing.assert_allclose(out5[2].cpu().numpy(), en, rtol=1e-4, atol=1e-4)
    assert out5[3].sum() == int(0.2 * len(rep)) and out5[4].sum() == int(rep.sum())
    thr, per_batch = m.get_uncertainty_threshold()
    assert thr is not None and len(per_batch) == 1


def test_protonet_set_forward_loss_gradients_match_autograd_of_oracle(cuda):
    from audio_fewshot_b200 import model as arch
    E, W, S, Q, D = 2, 5, 5, 6, 320
    N = E * W * (S + Q)
    x = np.random.default_rng(11).standard_normal((N, D)).astype(np.float32)
    lin = torch.nn.Linear(D, D, bias=False)
    m = arch.ProtoNet(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=lin,
                      device=cuda).to(cuda)
    m.train()
    out, acc, loss = m([torch.from_numpy(x), torch.zeros(N)])
    loss.backward()
    got = lin.weight.grad.detach().cpu()

    lin2 = torch.nn.Linear(D, D, bias=False)
    with torch.no_grad():
        lin2.weight.copy_(lin.weight.detach().cpu())
    feat = lin2(torch.from_numpy(x))
    sup, qry, _, qt, _ = heads.split_by_episode(feat, W, S, Q)
    ref_out = heads.proto_layer(qry, sup, W, S).reshape(-1, W)
    ref_loss = torch.nn.functional.cross_entropy(ref_out, qt.reshape(-1))
    ref_loss.backward()
    assert loss.item() == pytest.approx(ref_loss.item(), rel=1e-4)
    assert (got - lin2.weight.grad).abs().max().item() <= 2e-3 * lin2.weight.grad.abs().max().item()
    assert isinstance(acc, float)


# ------------------------------------------------------------------------------------------ pipeline
def test_pipeline_waveform_to_logits_and_cuda_graph(cuda):
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.frontend import LogMelFrontEnd
    from audio_fewshot_b200.pipeline import EpisodePipeline
    from oracle import frontend as ofe
    W, S, Q, L, E = 5, 2, 3, 16000, 2
    mean, std = -15.114207, 26.22313
    wav = cases.synthetic_clip_batch(3, 0, E, W, S, Q, L)
    net = _net(cuda, "conv64f_flat")
    model = arch.ProtoNet(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=net,
                          device=cuda).to(cuda).eval()
    front = LogMelFrontEnd(hop_length=102, n_mels=128, mean=mean, std=std).to(cuda).eval()
    repeats = torch.ones(E * W * Q, dtype=torch.long)
    plain = EpisodePipeline(front, model)
    out, acc = plain(torch.from_numpy(wav).pin_memory(), repeats, E * W * S)
    image = torch.from_numpy(ofe.logmel_f64(wav, hop=102, mean=mean, std=std).astype(np.float32))
    sd = {k: v.cpu() for k, v in net.state_dict().items()}
    with torch.no_grad():
        feat = obb.conv64f_forward(sd, image)
    want, want_acc, _ = heads.proto_forward(feat, W, S, Q, repeats, E * W * S)
    assert (out.cpu() - want).abs().max().item() <= 1e-3 * want.abs().max().item()
    assert torch.equal(out.cpu().argmax(1), want.argmax(1))
    assert acc.item() == pytest.approx(want_acc.item(), abs=1e-4)

    graphed = EpisodePipeline(front, model, use_graph=True)
    for _ in range(2):
        out_g, acc_g = graphed(torch.from_numpy(wav).pin_memory(), repeats, E * W * S)
    assert torch.equal(out_g, out) and acc_g.item() == acc.item()
    wav2 = cases.synthetic_clip_batch(4, 0, E, W, S, Q, L)
    out_g2, _ = graphed(torch.from_numpy(wav2).pin_memory(), repeats, E * W * S)
    out_p2, _ = plain(torch.from_numpy(wav2).pin_memory(), repeats, E * W * S)
    assert torch.equal(out_g2, out_p2)


def test_full_size_step_is_episode_separable_and_repeatable(cuda):
    """BASELINE.json's metric configuration at FULL size (32 episodes x 100 clips x 5 s = 1 GB of waveform, the bench
    step), checked through size-independent properties -- the oracle cannot run this size in seconds.  Episodes are
    independent, so (a) the log-mel images of any slice of the batch equal the slice of the full batch's images bit for
    bit (different run boundaries of the persistent pair engine), (b) the logits of two 16-episode steps and of an
    8-episode slice taken in the middle equal the 32-episode step's -- bit for bit through our own kernels (stem tiles
    of 128 pooled pixels crossing clips, four-accumulator block-2 tiles, tail, head); block 4 is a cuDNN call whose
    algorithm may depend on the batch size, hence 1e-5 of the logit range plus identical argmax rather than equality,
    (c) a second run is bit-identical, (d) the separately stated bf16 backbone keeps the argmax of at least 99.9 % of
    the queries on these class-structured episodes, (e) accuracy is what the per-query argmax says."""
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.frontend import LogMelFrontEnd
    from audio_fewshot_b200.synthetic import name_seeded_weights_, synthetic_clip_batch_device
    W, S, Q, L, E = 5, 5, 15, 80000, 32
    mean, std = -15.114207, 26.22313
    torch.manual_seed(0)
    emb = name_seeded_weights_(arch.Conv64F(is_flatten=True, num_channels=1))
    model = arch.ProtoNet(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=emb,
                          device=cuda).to(cuda).eval()
    front = LogMelFrontEnd(sample_rate=16000, hop_length=512, n_mels=128, mean=mean, std=std).to(cuda).eval()
    wav = synthetic_clip_batch_device(11, 0, E, W, S, Q, L, cuda)
    per = W * (S + Q)

    def run(first, n):
        with torch.no_grad():
            image = front(wav[first * per:(first + n) * per], first_clip_index=0)
            out, acc = model.set_forward([image, None, torch.ones(n * W * Q, dtype=torch.long), n * W * S])
        return image, out, acc

    image, full, acc = run(0, E)
    assert image.shape == (E * per, 1, 128, 157)
    assert full.shape == (E * W * Q, W) and torch.isfinite(full).all()
    image2, again, _ = run(0, E)
    assert torch.equal(image, image2) and torch.equal(full, again)
    tol = 1e-5 * full.abs().max().item()
    for first, n in ((0, 16), (16, 16), (13, 8)):
        img, out, _ = run(first, n)
        assert torch.equal(image[first * per:(first + n) * per], img), (first, n)
        ref = full[first * W * Q:(first + n) * W * Q]
        assert (out - ref).abs().max().item() <= tol, (first, n)
        assert torch.equal(out.argmax(1), ref.argmax(1)), (first, n)
    target = torch.arange(W, device=cuda).repeat_interleave(Q).repeat(E)
    assert acc.item() == pytest.approx((full.argmax(1) == target).float().mean().item() * 100.0, abs=1e-3)
    emb.precision = "bf16"
    try:
        _, low, _ = run(0, E)
    finally:
        emb.precision = None
    assert (low.argmax(1) == full.argmax(1)).float().mean().item() >= 0.999
    assert (low - full).abs().max().item() <= 5e-2 * full.abs().max().item()


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_full_size_dn4_step_is_episode_separable(cuda, precision):
    """BASELINE configs[2] (DN4 / Conv64F maps, 5w5s15q, n_k = 3) at the per-config bench size (8 episodes = 800
    images): a 3-episode slice scores as it does inside the full step (both heads are per-episode; own kernels up to
    block 3, then one cuDNN block: 1e-5 of the score range + identical argmax), and a second run is bit-identical."""
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.synthetic import name_seeded_weights_
    W, S, Q, E = 5, 5, 15, 8
    torch.manual_seed(2)
    emb = name_seeded_weights_(arch.Conv64F(is_flatten=False, last_pool=False, num_channels=1))
    model = arch.DN4(n_k=3, precision=precision, way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S,
                     test_query=Q, emb_func=emb, device=cuda).to(cuda).eval()
    per = W * (S + Q)
    g = torch.Generator().manual_seed(5)
    images = (torch.randn(E * per, 1, 128, 157, generator=g) * 0.7).to(cuda)

    def run(first, n):
        with torch.no_grad():
            return model.set_forward([images[first * per:(first + n) * per], None,
                                      torch.ones(n * W * Q, dtype=torch.long), n * W * S])[0]

    full = run(0, E)
    assert full.shape == (E * W * Q, W) and torch.isfinite(full).all()
    assert torch.equal(full, run(0, E))
    part = run(4, 3)
    ref = full[4 * W * Q:7 * W * Q]
    assert (part - ref).abs().max().item() <= 1e-5 * full.abs().max().item()
    assert torch.equal(part.argmax(1), ref.argmax(1))


def test_pipeline_stream_overlaps_copies_and_matches_single_calls(cuda):
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.frontend import LogMelFrontEnd
    from audio_fewshot_b200.pipeline import EpisodePipeline
    W, S, Q, L, E = 5, 1, 2, 16000, 1
    net = _net(cuda, "conv64f_flat")
    model = arch.ProtoNet(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=net,
                          device=cuda).to(cuda).eval()
    front = LogMelFrontEnd(hop_length=102, n_mels=128, mean=-15.0, std=26.0).to(cuda).eval()
    pipe = EpisodePipeline(front, model)
    repeats = torch.ones(E * W * Q, dtype=torch.long)
    batches = [torch.from_numpy(cases.synthetic_clip_batch(9, i, E, W, S, Q, L)).pin_memory() for i in range(5)]
    singles = [pipe(b, repeats, E * W * S) for b in batches]
    got = list(pipe.stream(iter(batches), repeats, E * W * S))
    assert len(got) == 5
    for (o1, a1), (o2, a2) in zip(singles, got):
        assert torch.equal(o1.cpu(), o2) and a1.item() == a2.item()  # stream() returns host tensors


def test_maml_set_forward_on_gpu_matches_cpu_inner_loop(cuda):
    """The CPU inner loop is pinned to the real reference (tests/test_maml.py); here the same class adapts on
    the GPU (dropout disabled so both devices see the same network) and votes with afs_vote_acc."""
    from test_maml import _model
    c = cases.MAML_CASE
    rep = np.ones(c["E"] * c["W"] * c["Q"], dtype=np.int64)
    x = torch.from_numpy(cases.maml_images(c))
    outs = {}
    for dev in ("cpu", cuda):
        m = _model(dev)
        m.emb_func.logits[0].p = 0.0
        m.eval()
        if dev == "cpu":
            tab = m._table(x.shape[0], torch.from_numpy(rep), c["E"] * c["W"] * c["S"])
            sup, qry = tab.episode_rows()
            outs["cpu"] = m._adapt_all(x, tab, sup, qry).detach()
        else:
            with torch.no_grad():  # set_forward re-enables grad for the inner loop itself
                out, acc = m([x, torch.zeros(x.shape[0]), torch.from_numpy(rep), c["E"] * c["W"] * c["S"]])
            outs["gpu"] = out.cpu()
            want_acc = (outs["cpu"].argmax(1) == tab.q_target_long).float().mean().item() * 100
            assert acc.item() == pytest.approx(want_acc, abs=1e-3)
    assert (outs["gpu"] - outs["cpu"]).abs().max().item() <= 5e-3 * outs["cpu"].abs().max().item()


def test_dn4_and_deepbdc_set_forward_loss_train_end_to_end(cuda):
    """set_forward_loss of DN4 (Conv64F maps) and DeepBDC (BdcPool) produce finite losses whose backward
    reaches the backbone through afs_dn4_bwd / afs_bdc_bwd + afs_proto_bwd."""
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.backbone import BdcPool
    E, W, S, Q = 1, 5, 2, 2
    N = E * W * (S + Q)
    x = torch.from_numpy((np.random.default_rng(3).standard_normal((N, 1, 128, 157)) * 0.5).astype(np.float32))
    emb = arch.Conv64F(is_flatten=False, last_pool=False, num_channels=1)
    dn4 = arch.DN4(n_k=3, way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=emb,
                   device=cuda).to(cuda)
    dn4.train()
    out, acc, loss = dn4([x, torch.zeros(N)])
    loss.backward()
    g = emb.layer1[0].weight.grad
    assert out.shape == (E * W * Q, W) and torch.isfinite(loss) and g is not None and g.abs().sum().item() > 0

    class Trunk(torch.nn.Module):  # small stand-in trunk ending in the real BdcPool
        def __init__(self):
            super().__init__()
            self.conv = torch.nn.Conv2d(1, 64, 5, stride=8)
            self.bdc_pool = BdcPool(is_vec=True, input_dim=(64, 10, 10), dimension_reduction=None)

        def forward(self, x):
            return self.bdc_pool(torch.relu(self.conv(x)))

    trunk = Trunk()
    bdc = arch.DeepBDC(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=trunk,
                       device=cuda).to(cuda)
    bdc.train()
    out, acc, loss = bdc([x, torch.zeros(N)])
    loss.backward()
    assert torch.isfinite(loss) and trunk.conv.weight.grad.abs().sum().item() > 0
    assert trunk.bdc_pool.temperature.grad is not None and torch.isfinite(trunk.bdc_pool.temperature.grad).all()


def test_config_to_loader_to_set_forward_on_gpu(cuda):
    """The reference's evaluation loop shape (test.py:362-393): config -> model by name -> loaders -> model(batch)."""
    import os
    from conftest import GOLDEN
    from audio_fewshot_b200.config import Config, build_model
    from audio_fewshot_b200.data import get_dataloader
    cfg = Config(os.path.join(GOLDEN, "config", "proto_fixture.yaml"),
                 {"test_episode": 4, "episode_size": 2, "max_windows": 3, "test_query": 2}).get_config_dict()
    model = build_model(cfg, cuda, mode="test").eval()
    loaders = get_dataloader(cfg, "test", model.model_type, False, cfg["modality"])
    model.reverse_setting_info()
    accs = []
    with torch.no_grad():
        for batch in zip(*loaders):
            flat = [elem for each in batch for elem in each]
            output, acc = model(flat)
            assert output.shape == (int(flat[2].sum()), cfg["test_way"])
            accs.append(acc)
    model.reverse_setting_info()
    assert len(accs) == 2 and all(0.0 <= a.item() <= 100.0 for a in accs)


def test_metabaseline_forward_and_cosine_backward_match_autograd_of_oracle(cuda):
    """MetaBaseline (reference meta_baseline.py): temp * cos(q, proto); gradients through afs_proto_bwd_cos."""
    from audio_fewshot_b200 import model as arch
    E, W, S, Q, D = 2, 5, 3, 4, 192
    N = E * W * (S + Q)
    x = np.random.default_rng(21).standard_normal((N, D)).astype(np.float32)
    lin = torch.nn.Linear(D, D, bias=False)
    m = arch.MetaBaseline(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=lin,
                          device=cuda).to(cuda)
    assert float(m.temp) == 10.0 and "temp" in m.state_dict()
    m.train()
    out, acc, loss = m([torch.from_numpy(x), torch.zeros(N)])
    loss.backward()

    lin2 = torch.nn.Linear(D, D, bias=False)
    with torch.no_grad():
        lin2.weight.copy_(lin.weight.detach().cpu())
    temp = torch.tensor(10.0, requires_grad=True)
    feat = lin2(torch.from_numpy(x))
    sup, qry, _, qt, _ = heads.split_by_episode(feat, W, S, Q)
    ref_out = heads.proto_layer(qry, sup, W, S, "cos_sim").reshape(-1, W) * temp
    ref_loss = torch.nn.functional.cross_entropy(ref_out, qt.reshape(-1))
    ref_loss.backward()
    assert (out.detach().cpu() - ref_out.detach()).abs().max().item() <= 1e-4 * ref_out.abs().max().item()
    assert loss.item() == pytest.approx(ref_loss.item(), rel=1e-4)
    g, gr = lin.weight.grad.detach().cpu(), lin2.weight.grad
    assert (g - gr).abs().max().item() <= 2e-3 * gr.abs().max().item()
    assert m.temp.grad.item() == pytest.approx(temp.grad.item(), rel=1e-3)
    m.eval()
    rep = np.random.default_rng(2).integers(1, 3, size=E * W * Q)
    n2 = E * W * S + int(rep.sum())
    with torch.no_grad():
        out2, acc2 = m([torch.randn(n2, D), torch.zeros(n2), torch.from_numpy(rep), E * W * S])
    assert out2.shape == (int(rep.sum()), W) and 0.0 <= acc2.item() <= 100.0


def test_graphed_train_step_matches_eager_maml(cuda):
    """GraphedTrainStep (one CUDA graph for set_forward_loss + backward + optimizer step) reproduces the eager MAML
    step: from the same weights and the same batch, the same loss and the same parameter update, three batches in a
    row (Dropout disabled so both see the same masks).

    Both models are put on the same weights before every step: a randomly initialised MAML net is chaotic (dead
    channels under batch-statistics BatchNorm amplify a 1e-7 weight difference into a 1e-3 loss difference one step
    later, eager against eager as well -- tools/diag_graphed_maml.py, profiles/r01_maml_step_reproducibility.txt),
    so free-running loss sequences only agree when every kernel is bit-reproducible.  Measured on B200: update
    difference 1e-5 relative with cuDNN's default algorithms, exactly 0 with cudnn.deterministic."""
    import copy
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.graph_step import GraphedTrainStep
    torch.manual_seed(3)
    emb = arch.Conv64F(is_flatten=True, num_channels=1)
    emb.logits[0].p = 0.0
    kw = dict(way_num=3, shot_num=2, query_num=3, test_way=3, test_shot=2, test_query=3, device=cuda)
    m1 = arch.MAML(inner_param={"lr": 0.01, "train_iter": 2, "test_iter": 2}, feat_dim=1600, emb_func=emb, **kw).to(cuda).train()
    m2 = copy.deepcopy(m1)
    m3 = copy.deepcopy(m1)
    E, W, S, Q = 2, 3, 2, 3
    n = E * W * (S + Q)
    target = torch.arange(W).repeat_interleave(S + Q).repeat(E)
    batches = [torch.randn(n, 1, 128, 157, device=cuda) * 0.7 for _ in range(3)]
    ref_state = copy.deepcopy(m1.state_dict())

    def flat(m):
        return torch.cat([p.detach().reshape(-1) for p in m.parameters()])

    old_det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        # (1) SGD: eager and graphed steps from the same weights give the same loss and the same update
        o1 = torch.optim.SGD(m1.parameters(), lr=1e-2)
        o2 = torch.optim.SGD(m2.parameters(), lr=1e-2)
        step = GraphedTrainStep(m2, o2, batches[0].shape, target=target, warmup=1)
        losses1 = []
        for b in batches:
            m2.load_state_dict(m1.state_dict())  # also undoes the warm-up / capture steps on zeros the first time
            w0 = flat(m1).clone()
            o1.zero_grad(set_to_none=True)
            out, acc, loss = m1([b, target])
            loss.backward()
            o1.step()
            out2, acc2, loss2 = step(b)
            l1, l2 = float(loss.detach()), float(loss2.detach())
            losses1.append(l1)
            assert abs(l1 - l2) <= 1e-4 * abs(l1), (l1, l2)
            d1, d2 = flat(m1) - w0, flat(m2) - w0
            assert d1.norm().item() > 1e-3  # the step moved the weights ...
            assert (d2 - d1).norm().item() <= 1e-3 * d1.norm().item()  # ... and the captured step moved them alike
            # accuracy comes back as a 1-element device tensor; its VALUE is not compared: an untrained net has
            # near-tied logits
            assert acc2.numel() == 1 and acc2.is_cuda and 0.0 <= float(acc2) <= 100.0 and 0.0 <= acc <= 100.0
        assert len(set(losses1)) == 3  # three different batches really went through

        # (2) Adam must be capturable, and the captured Adam step really updates the live parameters
        with pytest.raises(ValueError):
            GraphedTrainStep(m3, torch.optim.Adam(m3.parameters(), lr=1e-3), batches[0].shape, target=target)
        o3 = torch.optim.Adam(m3.parameters(), lr=1e-3, capturable=True)
        step3 = GraphedTrainStep(m3, o3, batches[0].shape, target=target, warmup=1)
        m3.load_state_dict(ref_state)
        for st in o3.state.values():
            for k, v in st.items():
                if torch.is_tensor(v):
                    v.zero_()
        for i, b in enumerate(batches):
            _, _, loss3 = step3(b)
            assert math.isfinite(float(loss3.detach()))
            if i == 0:  # identical weights and batch: the same loss as the eager step, whatever the optimizer
                assert abs(float(loss3.detach()) - losses1[0]) <= 1e-4 * abs(losses1[0])
        moved = [(m3.state_dict()[k] - v.to(cuda)).abs().max().item() for k, v in ref_state.items()
                 if v.dtype.is_floating_point and "running" not in k]
        assert 1e-3 <= max(moved) <= 3.5e-3  # three Adam steps of lr 1e-3
    finally:
        torch.backends.cudnn.deterministic = old_det


@pytest.mark.parametrize("N,H,Wd,leaky", [(6, 128, 157, False), (3, 20, 23, True), (2, 9, 10, False)])
def test_fused_training_stem_matches_module_graph(cuda, N, H, Wd, leaky):
    """csrc/conv1_train.cu (batch statistics from the 9-tap autocorrelation, fused forward, recomputing backward)
    against Conv2d -> BatchNorm2d(train) -> activation -> MaxPool2d under autograd: output, running statistics and the
    gradients of all four parameter tensors for a random upstream gradient."""
    from audio_fewshot_b200 import model as arch
    torch.manual_seed(N * 100 + H)
    a = arch.Conv64F(is_flatten=False, leaky_relu=leaky, negative_slope=0.2, num_channels=1).to(cuda).train()
    with torch.no_grad():
        a.layer1[1].weight.copy_(torch.randn(64, device=cuda) * 0.5 + 1.0)  # includes negative scales
        a.layer1[1].bias.copy_(torch.randn(64, device=cuda) * 0.3)
        a.layer1[0].bias.copy_(torch.randn(64, device=cuda))
    import copy
    b = copy.deepcopy(a)
    b.fused_train_stem = False
    x = torch.randn(N, 1, H, Wd, device=cuda) * 0.7 + 0.2
    from audio_fewshot_b200 import ops
    n0 = ops.launch_count()
    out_f = ops.conv1_bn_act_pool3_train(x, a.layer1[0], a.layer1[1], 0.2 if leaky else 0.0)
    assert ops.launch_count() == n0 + 3  # autocorrelation, statistics, forward
    out_r = b.layer1(x)
    assert out_f.shape == out_r.shape
    assert (out_f - out_r).abs().max().item() <= 2e-5 * max(out_r.abs().max().item(), 1.0)
    for name in ("running_mean", "running_var"):
        ra, rb = getattr(a.layer1[1], name), getattr(b.layer1[1], name)
        assert torch.allclose(ra, rb, rtol=1e-4, atol=1e-6), name
    assert int(a.layer1[1].num_batches_tracked) == int(b.layer1[1].num_batches_tracked) == 1
    gout = torch.randn_like(out_r)
    out_f.backward(gout)
    out_r.backward(gout)
    for (na, pa), (_, pb) in zip(a.layer1.named_parameters(), b.layer1.named_parameters()):
        ga, gb = pa.grad, pb.grad
        assert ga is not None and ga.shape == gb.shape, na
        tol = 2e-4 * gb.abs().max().item() + 1e-4 * gout.abs().sum().item() ** 0.5 * 1e-2
        if na == "0.bias":  # the conv bias cancels under batch statistics: autograd gives rounding noise
            assert ga.abs().max().item() == 0.0 and gb.abs().max().item() <= 1e-2 * gout.abs().sum().item() ** 0.5
        else:
            assert (ga - gb).abs().max().item() <= tol, (na, (ga - gb).abs().max().item(), gb.abs().max().item())


def test_protonet_training_step_with_fused_stem_matches_module_graph(cuda):
    import copy
    from audio_fewshot_b200 import model as arch
    torch.manual_seed(4)
    emb = arch.Conv64F(is_flatten=True, num_channels=1)
    emb.logits[0].p = 0.0
    kw = dict(way_num=3, shot_num=2, query_num=3, test_way=3, test_shot=2, test_query=3, device=cuda)
    m1 = arch.ProtoNet(emb_func=emb, **kw).to(cuda).train()
    m2 = copy.deepcopy(m1)
    m2.emb_func.fused_train_stem = False
    E, W, S, Q = 2, 3, 2, 3
    x = torch.randn(E * W * (S + Q), 1, 128, 157, device=cuda) * 0.7
    target = torch.arange(W).repeat_interleave(S + Q).repeat(E)
    out1, acc1, loss1 = m1([x, target])
    out2, acc2, loss2 = m2([x, target])
    assert abs(float(loss1) - float(loss2)) <= 1e-4 * abs(float(loss2))
    loss1.backward()
    loss2.backward()
    top = max(p.grad.abs().max().item() for p in m2.parameters() if p.grad is not None)
    for (n1, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        if p2.grad is None:
            assert p1.grad is None, n1
            continue
        scale = p2.grad.abs().max().item()
        if scale < 1e-5 * top:  # analytically zero gradients (biases cancelled by batch statistics / by q - proto)
            assert p1.grad.abs().max().item() < 1e-4 * top, n1
            continue
        # fp32 rounding of block 1 can flip an arg-max in a later max-pool (18 images, maps down to 1x1), so whole
        # gradients are compared in the L2 sense; the block itself is pinned element-wise by the test above
        rel = (p1.grad - p2.grad).norm().item() / max(p2.grad.norm().item(), 1e-12)
        assert rel <= 5e-2, (n1, rel, scale)


def test_energy_gated_tta_step(cuda, tmp_path, monkeypatch):
    """tta.energy_tta_step (reference test.py:380-414) around DeepBDC: with an identity augmentation and one window per
    query the re-vote over k identical copies cannot change a prediction (with several windows a tied vote may: the
    CUDA torch.mode tie rule depends on the slice length), so the accuracy must be unchanged and the new repeats must
    describe the enlarged batch; with ragged windows and the real noise suppression the step runs end to end."""
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200 import tta
    monkeypatch.chdir(tmp_path)  # the reference appends to ./test_uncertainty.npy (deepbdc.py:326-351)
    torch.manual_seed(0)
    emb = arch.resnet12Bdc(reduce_dim=64, num_channels=1)
    m = arch.DeepBDC(way_num=3, shot_num=2, query_num=4, test_way=3, test_shot=2, test_query=4, emb_func=emb,
                     device=cuda).to(cuda).eval()
    E, W, S, Q = 1, 3, 2, 4
    rng = np.random.default_rng(0)
    ones = torch.ones(E * W * Q, dtype=torch.long)
    x1 = torch.randn(E * W * (S + Q), 1, 128, 157) * 0.7
    repeats = torch.from_numpy(rng.integers(1, 3, size=E * W * Q)).long()
    n = E * W * S + int(repeats.sum())
    x = torch.randn(n, 1, 128, 157) * 0.7
    with torch.no_grad():
        acc, info = tta.energy_tta_step(m, [x1, None, ones, E * W * S], num_augmentations=3, mean=-15.0, std=26.0,
                                        suppression_strength=0.0, noise_percentile=20.0)
        assert info["n_flagged"] == int(0.2 * E * W * Q) >= 1
        assert abs(float(acc) - float(info["acc_before"])) < 1e-4
        rep2 = info["repeats_after"]
        flagged = np.flatnonzero(info["ood_query_mask"])
        assert all(int(rep2[i]) == 3 for i in flagged) and int(rep2.sum()) == E * W * Q + 2 * len(flagged)
        acc2, _ = tta.energy_tta_step(m, [x, None, repeats, E * W * S], num_augmentations=2, mean=-15.0, std=26.0)
        assert 0.0 <= float(acc2) <= 100.0
    assert (tmp_path / "test_uncertainty.npy").exists()


def test_tcgen05_kernels_repeat_bit_identically(cuda):
    """Stand-in for a race detector (compute-sanitizer is not available on the GPU pool): every hand-rolled
    mbarrier / TMEM pipeline must produce bit-identical outputs over repeated launches on a large batch -- a missing
    fence or a barrier phase error shows up as run-to-run differences long before it shows up as a wrong mean."""
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(99)
    # stem: conv1_tc (three TMEM accumulators per window row, double-buffered im2col)
    x = torch.from_numpy(rng.standard_normal((200, 1, 128, 157)).astype(np.float32)).to(cuda)
    w1 = rng.standard_normal((64, 9)).astype(np.float32) * 0.3
    b1 = rng.standard_normal(64).astype(np.float32)
    first = ops.conv1_bn_act_pool3(x, w1, b1, 0.0, tf32=True)
    for _ in range(4):
        assert torch.equal(ops.conv1_bn_act_pool3(x, w1, b1, 0.0, tf32=True), first)
    # blocks 2-3: conv3_tc (producer / three MMA warps / epilogue warps over a 4-stage ring)
    a = first.contiguous(memory_format=torch.channels_last)
    w3 = torch.from_numpy((rng.standard_normal((64, 64, 3, 3)) * 0.06).astype(np.float32)).to(cuda)
    b3 = torch.from_numpy(rng.standard_normal(64).astype(np.float32)).to(cuda)
    packed = torch.from_numpy(ops.conv3x3_c64_pack_weights(w3)).to(cuda)
    ref3 = ops.conv3x3_c64_bn_act(a, packed, b3, 0.0, pool=True)
    for _ in range(4):
        assert torch.equal(ops.conv3x3_c64_bn_act(a, packed, b3, 0.0, pool=True), ref3)


@pytest.mark.parametrize("N,H,W,J", [(3200, 4, 5, 1600), (70, 3, 3, 8), (1, 5, 5, 136)])
def test_pool3_linear_matches_pool_and_addmm(cuda, N, H, W, J):
    """csrc/tail.cu: last max-pool + flatten + Linear of Conv64F (conv_four.py:84,89-92) in one kernel, against
    F.max_pool2d + an fp64 matmul (fp32 FMA over 64 channels: 1e-5 of the output range)."""
    from audio_fewshot_b200 import ops
    g = torch.Generator().manual_seed(N + J)
    x = torch.randn(N, 64, H, W, generator=g).to(cuda).contiguous(memory_format=torch.channels_last)
    w = (torch.randn(J, 64, generator=g) * 0.1).to(cuda)
    b = torch.randn(J, generator=g).to(cuda)
    got = ops.pool3_linear(x, w, b)
    pooled = torch.nn.functional.max_pool2d(x, 3, 3).reshape(N, 64).double()
    want = pooled @ w.double().t() + b.double()
    assert got.shape == (N, J)
    assert (got.double() - want).abs().max().item() < 1e-5 * want.abs().max().item()
    assert torch.equal(got, ops.pool3_linear(x, w, b))
    assert not ops.pool3_linear_supported(torch.empty(1, 64, 6, 5), 1600)  # pooled map larger than one pixel
    with pytest.raises(ValueError):
        ops.pool3_linear(torch.zeros(2, 32, 4, 5, device=cuda), w, b)


def test_bench_dump_outputs_match_the_cpu_reference_arm(cuda, tmp_path):
    """`bench.py --dump-outputs`: the logits and accuracy of the B200 arm's last timed step (default precision) agree
    with those of the CPU oracle arm, which reads the same seeded waveforms at equal --steps and episodes per step."""
    import os
    import subprocess
    import sys

    from conftest import ROOT

    def run(impl):
        out = tmp_path / impl
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", impl, "--steps", "2",
                            "--warmup", "1", "--episodes-per-step", "1", "--no-extras", "--no-cpu-baseline",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        return np.load(out / "logits.npy"), np.load(out / "accuracy_pct.npy")

    got, acc = run("b200")
    want, want_acc = run("reference")
    assert got.dtype == np.float32 and got.shape == want.shape == (5 * 15, 5)
    assert np.abs(got - want).max() < 2e-2 * np.abs(want).max()  # TF32 backbone against the fp32 oracle, as smoke()
    assert (got.argmax(1) == want.argmax(1)).mean() >= 0.97
    assert abs(float(acc) - float(want_acc)) <= 100.0 * 2 / 75
