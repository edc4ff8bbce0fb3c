"""Parity of the CUDA heads (through the C ABI) with the reference goldens and the CPU oracle."""
import numpy as np
import pytest
import torch

from oracle import cases, heads

pytestmark = pytest.mark.gpu


def fixed_table(c, device):
    from audio_fewshot_b200.episode import EpisodeTable
    return EpisodeTable(c["E"], c["W"], c["S"], c["Q"], np.ones(c["E"] * c["W"] * c["Q"], np.int64), device)


def ragged_table(E, W, S, Q, rep, device):
    from audio_fewshot_b200.episode import EpisodeTable
    return EpisodeTable(E, W, S, Q, rep, device)


# ------------------------------------------------------------------ prototype head
@pytest.mark.parametrize("name", sorted(cases.PROTO_CASES))
def test_proto_matches_reference_golden(cuda, golden, name):
    from audio_fewshot_b200 import ops
    c = cases.PROTO_CASES[name]
    feat = torch.from_numpy(cases.proto_features(c)).to(cuda)
    tab = fixed_table(c, cuda)
    logits, pred = ops.proto_logits(feat, tab.cls_row, tab.E, tab.W, tab.S, c["mode"], want_pred=True)
    want = golden("proto_layer.npz")[name]
    got = logits.cpu().numpy()
    # north star: distances/logits within 1e-3 relative; predictions identical
    np.testing.assert_allclose(got, want, rtol=1e-3, atol=1e-3 * np.abs(want).max() * 1e-2)
    assert np.abs(got - want).max() <= 2e-5 * np.abs(want).max()  # what the fp32 path actually achieves
    assert np.array_equal(got.argmax(1), want.argmax(1))
    assert np.array_equal(pred.cpu().numpy(), want.argmax(1))


@pytest.mark.parametrize("name", ["c1_euclid", "c2_euclid_d12800", "c4_euclid_d2080", "bdc_5shot"])
def test_proto_tensor_core_head_is_a_separate_precision_class(cuda, golden, name):
    """csrc/proto_tc.cu: -(|q|^2 - 2 q.p + |p|^2) with q.p as a tcgen05 TF32 GEMM (north star: "one tensor-core GEMM
    epilogue", "stated separately").  Against the reference golden: logits within the absolute error the formulation
    allows (the MMA truncates operands to TF32: ~1e-3 |q| |p| on the cross term, which the expansion does not cancel),
    and the argmax flip rate on these cases is reported and bounded."""
    from audio_fewshot_b200 import ops
    c = cases.PROTO_CASES[name]
    x = cases.proto_features(c)
    feat = torch.from_numpy(x).to(cuda)
    tab = fixed_table(c, cuda)
    logits, pred = ops.proto_logits(feat, tab.cls_row, tab.E, tab.W, tab.S, "euclidean", want_pred=True, precision="tf32")
    want = golden("proto_layer.npz")[name]
    got = logits.cpu().numpy()
    assert np.isfinite(got).all()
    scale = float((np.linalg.norm(x, axis=1) ** 2).max())  # |q| |p| <= max |row|^2
    err = np.abs(got - want).max()
    assert err <= 4e-3 * scale, (err, scale)
    assert err <= 2e-3 * np.abs(want).max()  # for these seeded features also 2e-3 relative to the largest logit
    flips = float((got.argmax(1) != want.argmax(1)).mean())
    print("proto tf32 %s: max abs err %.3e (%.1e of |row|^2), argmax flip rate %.4f" % (name, err, err / scale, flips))
    assert flips <= 0.02
    assert np.array_equal(pred.cpu().numpy(), got.argmax(1))
    fp32 = ops.proto_logits(feat, tab.cls_row, tab.E, tab.W, tab.S, "euclidean")
    assert (logits - fp32).abs().max().item() <= 4e-3 * scale
    for _ in range(3):  # deterministic
        again = ops.proto_logits(feat, tab.cls_row, tab.E, tab.W, tab.S, "euclidean", precision="tf32")
        assert torch.equal(again, logits)


def test_proto_tensor_core_head_large_ragged_batch_and_contract(cuda):
    from audio_fewshot_b200 import ops
    from audio_fewshot_b200._lib import AfsError
    rng = np.random.default_rng(5)
    E, W, S, Q, D = 37, 5, 5, 15, 1600  # 3 700+ rows: many tiles per CTA, tiles straddling episodes
    rep = rng.integers(1, 3, size=E * W * Q)
    n = E * W * S + int(rep.sum())
    feat = torch.from_numpy(rng.standard_normal((n, D)).astype(np.float32)).to(cuda)
    tab = ragged_table(E, W, S, Q, rep, cuda)
    a = ops.proto_logits(feat, tab.cls_row, E, W, S, "euclidean")
    b = ops.proto_logits(feat, tab.cls_row, E, W, S, "euclidean", precision="tf32")
    assert torch.isfinite(b).all()
    assert (a - b).abs().max().item() <= 2e-3 * a.abs().max().item()
    assert (a.argmax(1) != b.argmax(1)).float().mean().item() <= 0.02
    with pytest.raises(AfsError):  # 20 ways: more prototype columns than the kernel's N
        t20 = ragged_table(1, 20, 2, 3, np.ones(60, dtype=np.int64), cuda)
        ops.proto_logits(torch.randn(100, 128, device=cuda), t20.cls_row, 1, 20, 2, "euclidean", precision="tf32")
    with pytest.raises(ValueError):
        ops.proto_logits(feat, tab.cls_row, E, W, S, "cos_sim", precision="tf32")


@pytest.mark.parametrize("mode", ["euclidean", "cos_sim", "dot"])
def test_proto_ragged_layout_matches_oracle(cuda, mode):
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(77)
    E, W, S, Q, D = 3, 5, 2, 4, 320
    rep = rng.integers(0, 4, size=E * W * Q)  # includes zero-window queries
    rep[:Q] = 0  # a class with no query rows at all
    n = E * W * S + int(rep.sum())
    feat = torch.from_numpy(rng.standard_normal((n, D)).astype(np.float32))
    tab = ragged_table(E, W, S, Q, rep, cuda)
    got = ops.proto_logits(feat.to(cuda), tab.cls_row, E, W, S, mode).cpu()
    sup, qry, _, _, _ = heads.split_by_episode(feat, W, S, Q, torch.from_numpy(rep), E * W * S)
    outs = []
    for i in range(E):
        if mode == "dot":
            o = heads.deepbdc_proto_layer(qry[i].unsqueeze(0), sup[i].unsqueeze(0), W, 1) if S == 1 else \
                torch.matmul(qry[i].unsqueeze(0), sup[i].view(1, W, S, D).mean(2).transpose(-1, -2))
        else:
            o = heads.proto_layer(qry[i].unsqueeze(0), sup[i].unsqueeze(0), W, S, mode)
        outs.append(o.reshape(-1, W))
    want = torch.cat(outs)
    assert got.shape == want.shape
    torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-3)
    assert torch.equal(got.argmax(1), want.argmax(1))


def test_proto_strided_rows_and_empty_batch(cuda):
    from audio_fewshot_b200 import ops
    c = dict(E=2, W=5, S=5, Q=3)
    wide = torch.randn(80, 96, device=cuda)
    feat = wide[:, :64]  # row stride 96, not contiguous
    tab = fixed_table(c, cuda)
    a = ops.proto_logits(feat, tab.cls_row, 2, 5, 5)
    b = ops.proto_logits(feat.contiguous(), tab.cls_row, 2, 5, 5)
    assert torch.equal(a, b)
    with pytest.raises(Exception):
        ops.proto_logits(feat.cpu(), tab.cls_row, 2, 5, 5)  # no CPU fallback


def test_proto_many_episodes_is_per_episode_independent(cuda):
    """Full bench size (BASELINE C1, 512 episodes): every episode's logits equal the ones
    computed when that episode is launched alone (a size-independent property)."""
    from audio_fewshot_b200 import ops
    c = dict(E=512, W=5, S=5, Q=15)
    g = torch.Generator(device="cpu").manual_seed(5)
    feat = torch.randn(512 * 100, 1600, generator=g).to(cuda)
    tab = fixed_table(c, cuda)
    full = ops.proto_logits(feat, tab.cls_row, 512, 5, 5)
    one = fixed_table(dict(E=1, W=5, S=5, Q=15), cuda)
    for e in (0, 17, 511):
        part = ops.proto_logits(feat[e * 100:(e + 1) * 100], one.cls_row, 1, 5, 5)
        assert torch.equal(full[e * 75:(e + 1) * 75], part)


@pytest.mark.parametrize("mode,S", [("euclidean", 5), ("euclidean", 1), ("dot", 1), ("dot", 3)])
def test_proto_backward_matches_autograd(cuda, mode, S):
    from audio_fewshot_b200 import ops
    E, W, Q, D = 3, 5, 4, 200
    tab = fixed_table(dict(E=E, W=W, S=S, Q=Q), cuda)
    feat = torch.randn(E * W * (S + Q), D, device=cuda, requires_grad=True)
    gout = torch.randn(E * W * Q, W, device=cuda)
    logits = ops.proto_logits(feat, tab.cls_row, E, W, S, mode)
    logits.backward(gout)
    got = feat.grad.clone()
    ref = feat.detach().clone().requires_grad_(True)
    f = ref.view(E, W, S + Q, D)
    proto = f[:, :, :S].mean(2)
    qry = f[:, :, S:].reshape(E, W * Q, D)
    if mode == "euclidean":
        want_logits = -((qry.unsqueeze(2) - proto.unsqueeze(1)) ** 2).sum(3)
    else:
        want_logits = qry @ proto.transpose(1, 2)
    want_logits.reshape(-1, W).backward(gout)
    torch.testing.assert_close(logits, want_logits.reshape(-1, W), rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(got, ref.grad, rtol=1e-4, atol=1e-4)


# ------------------------------------------------------------------ DN4
def dn4_oracle(c):
    feat = torch.from_numpy(cases.dn4_features(c))
    E, W, S, Q = c["E"], c["W"], c["S"], c["Q"]
    f = feat.view(E, W, S + Q, *feat.shape[1:])
    sup = f[:, :, :S].contiguous().view(E, W * S, *feat.shape[1:])
    qry = f[:, :, S:].contiguous().view(E, W * Q, *feat.shape[1:])
    return heads.dn4_layer(qry, sup, W, S, c["n_k"], return_topk=True)


@pytest.mark.parametrize("name", sorted(cases.DN4_CASES))
def test_dn4_matches_reference_golden_and_topk(cuda, golden, name):
    from audio_fewshot_b200 import ops
    c = cases.DN4_CASES[name]
    feat = torch.from_numpy(cases.dn4_features(c)).to(cuda)
    tab = fixed_table(c, cuda)
    score, topk, pred = ops.dn4_scores(feat, tab.cls_row, tab.E, tab.W, tab.S, c["n_k"], want_topk=True,
                                       want_pred=True)
    want = golden("dn4_layer.npz")[name]
    got = score.cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-3)
    assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()
    assert np.array_equal(got.argmax(1), want.argmax(1))
    assert np.array_equal(pred.cpu().numpy(), want.argmax(1))
    # top-k indices against torch.topk on the oracle's relation tensor (the reference discards
    # them, dn4.py:72).  Identical except where the oracle's own values are within float noise.
    _, topv, topi, relation = dn4_oracle(c)
    E, W, Q = c["E"], c["W"], c["Q"]
    HW = c["H"] * c["Wd"]
    topi = topi.reshape(E * W * Q, W, HW, c["n_k"]).numpy()
    relation = relation.reshape(E * W * Q, W, HW, -1).numpy()
    mine = topk.cpu().numpy()
    diff = np.argwhere(mine != topi)
    for o, w, m, k in diff:
        a, b = relation[o, w, m, mine[o, w, m, k]], relation[o, w, m, topi[o, w, m, k]]
        assert abs(a - b) <= 4e-7, (o, w, m, k, a, b)
    assert len(diff) <= 1e-4 * mine.size


@pytest.mark.parametrize("name", [n for n in sorted(cases.DN4_CASES)
                                  if cases.DN4_CASES[n]["C"] <= 128 or cases.DN4_CASES[n]["C"] % 32 == 0])
def test_dn4_tensor_core_path_matches_reference_golden(cuda, golden, name):
    """tcgen05 TF32 path (csrc/dn4_tc.cu, csrc/dn4_tc2.cu incl. the K-streaming schedule for the ResNet-12 map with
    C = 640): scores within the north star's 1e-3 relative of the reference's
    DN4Layer; selected descriptors are the oracle's top-k except where two cosines differ by less than TF32
    resolution; same argmax."""
    from audio_fewshot_b200 import ops
    c = cases.DN4_CASES[name]
    feat = torch.from_numpy(cases.dn4_features(c)).to(cuda)
    tab = fixed_table(c, cuda)
    score, topk, pred = ops.dn4_scores(feat, tab.cls_row, tab.E, tab.W, tab.S, c["n_k"], want_topk=True,
                                       want_pred=True, precision="tf32")
    want = golden("dn4_layer.npz")[name]
    got = score.cpu().numpy()
    assert np.abs(got - want).max() <= 1e-3 * np.abs(want).max()
    assert np.abs(got - want).max() <= 3e-4 * np.abs(want).max()  # measured ~5e-5 with round-to-nearest operands
    assert np.array_equal(pred.cpu().numpy(), got.argmax(1))
    _, topv, topi, relation = dn4_oracle(c)
    E, W, Q = c["E"], c["W"], c["Q"]
    HW = c["H"] * c["Wd"]
    topi = topi.reshape(E * W * Q, W, HW, c["n_k"]).numpy()
    relation = relation.reshape(E * W * Q, W, HW, -1).numpy()
    mine = topk.cpu().numpy()
    assert mine.min() >= 0 and mine.max() < relation.shape[-1]
    diff = np.argwhere(mine != topi)
    for o, w, m, k in diff:  # a different pick must be a near-tie at TF32 resolution
        a, b = relation[o, w, m, mine[o, w, m, k]], relation[o, w, m, topi[o, w, m, k]]
        assert abs(a - b) <= 2e-3, (o, w, m, k, a, b)
    assert len(diff) <= 0.02 * mine.size


def test_dn4_tensor_core_path_ragged_multi_tile_and_unsupported(cuda):
    from audio_fewshot_b200 import ops
    from audio_fewshot_b200._lib import AfsError
    rng = np.random.default_rng(15)
    for C in (64, 8, 40, 72, 120):  # every width dn4_tc_supported admits below 128 channels has a tensor-core kernel
        assert ops.dn4_tc_supported(C)
        E, W, S, Q, H, Wd, n_k = 3, 5, 8, 3, 4, 5, 3  # S*HW = 160 support descriptors: two column tiles
        rep = rng.integers(1, 4, size=E * W * Q)
        n = E * W * S + int(rep.sum())
        feat = torch.from_numpy(np.abs(rng.standard_normal((n, C, H, Wd))).astype(np.float32)).to(cuda)
        tab = ragged_table(E, W, S, Q, rep, cuda)
        a, _, _ = ops.dn4_scores(feat, tab.cls_row, E, W, S, n_k)
        b, _, _ = ops.dn4_scores(feat, tab.cls_row, E, W, S, n_k, precision="tf32")
        assert (a - b).abs().max().item() <= 3e-4 * a.abs().max().item(), C
    # C = 640 (ResNet-12 maps): K-streaming schedule, ragged windows, three column tiles with a partial last one
    E, W, S, Q, C, H, Wd = 2, 5, 5, 2, 640, 8, 9
    rep = rng.integers(1, 3, size=E * W * Q)
    n = E * W * S + int(rep.sum())
    feat = torch.from_numpy(np.abs(rng.standard_normal((n, C, H, Wd))).astype(np.float32)).to(cuda)
    tab = ragged_table(E, W, S, Q, rep, cuda)
    a, ia, _ = ops.dn4_scores(feat, tab.cls_row, E, W, S, n_k, want_topk=True)
    b, ib, _ = ops.dn4_scores(feat, tab.cls_row, E, W, S, n_k, want_topk=True, precision="tf32")
    assert (a - b).abs().max().item() <= 3e-4 * a.abs().max().item()
    assert (ia != ib).float().mean().item() <= 0.02
    tab2 = ragged_table(2, 5, 1, 2, np.ones(20, dtype=np.int64), cuda)
    for C in (36, 136):  # not a multiple of 8, or > 128 channels and not a multiple of 32: no tensor-core kernel
        assert not ops.dn4_tc_supported(C)
        odd = torch.rand(2 * 5 * 3, C, 2, 2, device=cuda)
        with pytest.raises(AfsError):
            ops.dn4_scores(odd, tab2.cls_row, 2, 5, 1, 2, precision="tf32")


def test_dn4_ragged_matches_oracle(cuda):
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(5)
    E, W, S, Q, C, H, Wd, n_k = 2, 3, 2, 3, 32, 3, 4, 2
    rep = rng.integers(1, 4, size=E * W * Q)
    n = E * W * S + int(rep.sum())
    feat = torch.from_numpy(np.abs(rng.standard_normal((n, C, H, Wd))).astype(np.float32))
    tab = ragged_table(E, W, S, Q, rep, cuda)
    score, _, _ = ops.dn4_scores(feat.to(cuda), tab.cls_row, E, W, S, n_k)
    want, _, _ = heads.dn4_forward(feat, W, S, Q, torch.from_numpy(rep), E * W * S, n_k)
    torch.testing.assert_close(score.cpu(), want, rtol=1e-4, atol=1e-4)


# ------------------------------------------------------------------ BDC
@pytest.mark.parametrize("name", sorted(cases.BDC_CASES))
def test_bdc_matches_reference_golden(cuda, golden, name):
    from audio_fewshot_b200 import ops
    c = cases.BDC_CASES[name]
    x = torch.from_numpy(cases.bdc_features(c)).to(cuda)
    t = torch.full((1, 1), c["log_temp"], device=cuda)
    g = golden("bdc_pool.npz")
    triu = ops.bdc_pool(x, t, triu=True).cpu().numpy()
    full = ops.bdc_pool(x, t, triu=False).cpu().numpy().reshape(c["B"], c["C"], c["C"])
    scale = np.abs(g[name + "/full"]).max()
    assert np.abs(full - g[name + "/full"]).max() <= 1e-3 * scale
    assert np.abs(full - g[name + "/full"]).max() <= 2e-5 * scale
    assert np.abs(triu - g[name + "/triu"]).max() <= 2e-5 * scale
    assert np.abs(full - full.transpose(0, 2, 1)).max() <= 1e-5 * scale  # symmetric
    assert np.abs(full.mean(axis=2)).max() <= 1e-4 * scale               # double-centred


# ------------------------------------------------------------------ vote / accuracy / energy
@pytest.mark.parametrize("name", sorted(cases.SPLIT_CASES))
def test_vote_acc_energy_match_reference_golden(cuda, golden, name):
    from audio_fewshot_b200 import ops
    c = cases.SPLIT_CASES[name]
    g = golden("episode_vote.npz")
    rep = cases.split_repeats(c)
    tab = ragged_table(c["E"], c["W"], c["S"], c["Q"], rep, cuda)
    logits = torch.from_numpy(cases.split_logits(c, int(rep.sum()))).to(cuda)
    assert np.array_equal(tab.q_target.cpu().numpy(), g[name + "/query_target"].reshape(-1))
    # the golden predictions come from the reference run on the CPU: torch.mode's CPU tie rule
    q_pred, acc, stats = ops.vote_acc(logits, tab.q_start, tab.q_target, tie_rule="smallest")
    assert np.array_equal(q_pred.cpu().numpy(), g[name + "/vote_pred"])  # bit-exact predictions
    assert acc.item() == pytest.approx(float(g[name + "/vote_acc"]), rel=1e-6)
    assert stats[1].item() == tab.nq
    en = ops.energy_score(logits, tab.q_start, tab.nq).cpu().numpy()
    np.testing.assert_allclose(en, g[name + "/energy"], rtol=1e-5, atol=1e-5)


def test_vote_matches_measured_torch_mode_cuda_golden(cuda, golden):
    """tests/golden/torch_mode_cuda.npz: torch.mode outputs recorded on a B200 (tools/probe_torch_mode.py)."""
    from audio_fewshot_b200 import ops
    g = golden("torch_mode_cuda.npz")
    n = g["n"].astype(np.int64)
    W = 8
    flat = np.concatenate([row[:k] for row, k in zip(g["labels"], n)]).astype(np.int64)
    logits = torch.zeros(len(flat), W)
    logits[torch.arange(len(flat)), torch.from_numpy(flat)] = 1.0
    q_start = torch.from_numpy(np.concatenate([[0], np.cumsum(n)]).astype(np.int32)).to(cuda)
    target = torch.from_numpy(g["mode"].astype(np.int32)).to(cuda)
    q_pred, acc, stats = ops.vote_acc(logits.to(cuda), q_start, target, tie_rule="torch_cuda")
    assert np.array_equal(q_pred.cpu().numpy(), g["mode"].astype(np.int32))
    assert stats[0].item() == len(n) and acc.item() == 100.0


def test_vote_tie_rule_equals_torch_mode_on_cuda(cuda):
    """The reference calls torch.mode on a CUDA slice (utils.py:443): same tie rule as ours."""
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(3)
    W, nq = 4, 300
    rep = rng.integers(1, 40, size=nq)
    n = int(rep.sum())
    labels = rng.integers(0, W, size=n)
    logits = torch.zeros(n, W)
    logits[torch.arange(n), torch.from_numpy(labels)] = 1.0
    q_start = torch.from_numpy(np.concatenate([[0], np.cumsum(rep)]).astype(np.int32)).to(cuda)
    q_target = torch.zeros(nq, dtype=torch.int32, device=cuda)
    q_pred, acc, _ = ops.vote_acc(logits.to(cuda), q_start, q_target)
    y = logits.to(cuda).argmax(1)
    want, end = [], 0
    for num in rep:
        want.append(torch.mode(y[end:end + int(num)])[0].item())
        end += int(num)
    assert q_pred.cpu().tolist() == want
    assert acc.item() == pytest.approx(100.0 * np.mean(np.asarray(want) == 0), rel=1e-6)


def test_vote_large_batch_counts(cuda):
    from audio_fewshot_b200 import ops
    nq, W = 200_000, 5
    logits = torch.randn(nq, W, device=cuda)
    q_start = torch.arange(nq + 1, dtype=torch.int32, device=cuda)
    target = torch.randint(0, W, (nq,), device=cuda, dtype=torch.int32)
    q_pred, acc, stats = ops.vote_acc(logits, q_start, target)
    want = (logits.argmax(1).int() == target).sum().item()
    assert stats[0].item() == want
    assert torch.equal(q_pred, logits.argmax(1).int())


# ------------------------------------------------------------------------------------------ backward kernels
def test_dn4_backward_matches_autograd_of_oracle(cuda):
    """afs_dn4_bwd against torch autograd through the reference-order DN4 layer (oracle.heads.dn4_layer)."""
    from audio_fewshot_b200 import ops
    from audio_fewshot_b200.episode import EpisodeTable
    E, W, S, Q, C, H, Wd, n_k = 2, 5, 2, 3, 64, 4, 5, 3
    N = E * W * (S + Q)
    x = np.abs(np.random.default_rng(41).standard_normal((N, C, H, Wd))).astype(np.float32) + 0.05
    gs = np.random.default_rng(42).standard_normal((E * W * Q, W)).astype(np.float32)
    tab = EpisodeTable(E, W, S, Q, np.ones(E * W * Q, dtype=np.int64), cuda)

    xg = torch.from_numpy(x).to(cuda).requires_grad_(True)
    score, _, _ = ops.dn4_scores(xg, tab.cls_row, E, W, S, n_k)
    score.backward(torch.from_numpy(gs).to(cuda))

    xc = torch.from_numpy(x).requires_grad_(True)
    sup, qry, _, _, _ = heads.split_by_episode(xc, W, S, Q)
    want = heads.dn4_layer(qry, sup, W, S, n_k).reshape(-1, W)
    want.backward(torch.from_numpy(gs))
    assert (score.detach().cpu() - want.detach()).abs().max().item() <= 1e-4 * want.abs().max().item()
    ref = xc.grad
    assert (xg.grad.cpu() - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()


@pytest.mark.parametrize("B,C,H,Wd,triu", [(3, 64, 16, 19, True), (2, 48, 7, 9, True), (2, 64, 5, 5, False)])
def test_bdc_backward_matches_autograd_of_oracle(cuda, B, C, H, Wd, triu):
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(B * 100 + C)
    x = np.maximum(rng.standard_normal((B, C, H, Wd)), 0.0).astype(np.float32)
    t0 = float(np.log(1.0 / 200.0))
    out_dim = C * (C + 1) // 2 if triu else C * C
    go = rng.standard_normal((B, out_dim)).astype(np.float32)

    xg = torch.from_numpy(x).to(cuda).requires_grad_(True)
    tg = torch.full((1, 1), t0, device=cuda, requires_grad=True)
    out = ops.bdc_pool(xg, tg, triu=triu)
    out.backward(torch.from_numpy(go).to(cuda))

    xc = torch.from_numpy(x).double().requires_grad_(True)
    tc = torch.full((1, 1), t0, dtype=torch.float64, requires_grad=True)
    full = heads.bdcovpool(xc, tc)
    want = heads.triuvec(full).reshape(B, -1) if triu else full.reshape(B, -1)
    want.backward(torch.from_numpy(go).double())
    assert (out.detach().cpu().double() - want.detach()).abs().max().item() <= 1e-4 * want.abs().max().item()
    assert (xg.grad.cpu().double() - xc.grad).abs().max().item() <= 2e-3 * xc.grad.abs().max().item()
    assert tg.grad.shape == (1, 1)
    assert abs(tg.grad.item() - tc.grad.item()) <= 2e-3 * abs(tc.grad.item()) + 1e-6


def test_utils_module_mirrors_reference_helpers(cuda, golden):
    """audio_fewshot_b200.utils: reference-named helpers (accuracy, majority_vote, vote_catagorical_acc,
    average_logits) against the oracle restatements pinned to the reference goldens."""
    from audio_fewshot_b200 import utils as U
    rng = np.random.default_rng(12)
    nums = rng.integers(1, 5, size=37)
    logits = torch.from_numpy(rng.standard_normal((int(nums.sum()), 5)).astype(np.float32))
    want_vote = heads.majority_vote(logits, nums, tie_rule="smallest")
    got_vote = U.majority_vote(logits.to(cuda), torch.from_numpy(nums), tie_rule="smallest")
    assert got_vote.dtype == torch.float32 and not got_vote.is_cuda
    assert np.array_equal(got_vote.numpy(), np.asarray(want_vote, dtype=np.float32))
    want_avg = heads.average_logits(logits, nums)
    got_avg = U.average_logits(logits.to(cuda), nums.tolist())
    assert torch.allclose(got_avg.cpu(), torch.as_tensor(np.asarray(want_avg), dtype=torch.float32), atol=1e-6)
    target = torch.from_numpy(rng.integers(0, 5, size=37)).float()
    acc = U.vote_catagorical_acc(target, got_vote)
    assert abs(float(acc) - 100.0 * float((got_vote == target).float().mean())) < 1e-4
    out = torch.from_numpy(rng.standard_normal((64, 5)).astype(np.float32)).to(cuda)
    tgt = torch.from_numpy(rng.integers(0, 5, size=64)).to(cuda)
    a1 = U.accuracy(out, tgt)
    assert isinstance(a1, float) and abs(a1 - 100.0 * float((out.argmax(1) == tgt).float().mean())) < 1e-4
    a2 = U.accuracy(out, tgt, topk=2)
    assert a2 >= a1
    m, h = U.mean_confidence_interval([80.0, 82.0, 78.0, 85.0])
    assert abs(m - 81.25) < 1e-9 and h > 0


@pytest.mark.parametrize("C,H,Wd,E", [(64, 4, 5, 24), (640, 8, 9, 4)])
def test_dn4_tensor_core_head_repeats_bit_identically(cuda, C, H, Wd, E):
    """dn4_tc2 (TMA + tcgen05 + TMEM double buffering, the K-streaming ring for C = 640): scores, top-k indices and
    predictions of repeated launches are bit-identical -- the stand-in for racecheck on the GPU pool."""
    from audio_fewshot_b200 import ops
    rng = np.random.default_rng(C + E)
    W, S, Q, n_k = 5, 5, 6, 3
    n = E * W * (S + Q)
    feat = torch.from_numpy(np.abs(rng.standard_normal((n, C, H, Wd))).astype(np.float32)).to(cuda)
    tab = ragged_table(E, W, S, Q, np.ones(E * W * Q, dtype=np.int64), cuda)
    s0, i0, p0 = ops.dn4_scores(feat, tab.cls_row, E, W, S, n_k, want_topk=True, want_pred=True, precision="tf32")
    for _ in range(4):
        s, i, p = ops.dn4_scores(feat, tab.cls_row, E, W, S, n_k, want_topk=True, want_pred=True, precision="tf32")
        assert torch.equal(s, s0) and torch.equal(i, i0) and torch.equal(p, p0)
