"""TEST INFRASTRUCTURE ONLY -- never imported by the product path.

CPU restatement (torch CPU ops, fp32, same op order) of the reference's episodic
heads and episode plumbing.  Each function cites the reference file:line it
follows.  Pinned against the real reference classes by tests/test_oracle.py
(when /root/reference is present) and by the committed goldens in tests/golden/
(generated from the reference by oracle/make_golden.py).
"""
import numpy as np
import torch
import torch.nn.functional as F


# ---------------------------------------------------------------- episode plumbing
def class_query_rows(repeats, episode_size, way_num):
    """Query window rows per (episode, class) block.

    reference: hierarchical_cumsum_with_carry, libfewshot_core/model/abstract_model.py:84-121
    (sum of `repeats` over each class's queries; the reference carries the cumsum, we return
    the per-block counts and the carried cumsum)."""
    arr = np.asarray(repeats).reshape(-1)
    if arr.size % (episode_size * way_num) != 0:
        raise ValueError("Length of array must be divisible by %d*%d" % (episode_size, way_num))
    sums = arr.reshape(episode_size, way_num, -1).sum(axis=2)
    return sums, np.cumsum(sums.reshape(-1)).reshape(episode_size, way_num)


def split_by_episode(features, way_num, shot_num, query_num, repeats=None, support_size=0):
    """reference: AbstractModel.split_by_episode modes 1 and 2,
    libfewshot_core/model/abstract_model.py:176-332.

    Returns (support [E, W*S, ...], query: tensor [E, W*Q, ...] or list of [R_i, ...],
    support_target [E, W*S], query_target [E, W*Q], query_mask or None)."""
    W, S, Q = way_num, shot_num, query_num
    if repeats is not None:
        E = (len(repeats) + support_size) // (W * (S + Q))  # :185
        _, carried = class_query_rows(np.asarray(repeats), E, W)  # :187
    else:
        E = features.shape[0] // (W * (S + Q))  # :189-191
    local = torch.arange(W, dtype=torch.long).view(1, -1, 1).repeat(E, 1, S + Q)  # :167-174
    rest = features.shape[1:]
    query_mask = None
    if repeats is None:
        f = features.contiguous().view(E, W, S + Q, *rest)  # :215-229 / :280-296
        support = f[:, :, :S].contiguous().view(E, W * S, *rest)
        query = f[:, :, S:].contiguous().view(E, W * Q, *rest)
    else:
        # :231-258 -- block g = i*W + j starts at row g*S + (query rows of all earlier blocks)
        query_mask = np.zeros(features.shape[0], dtype=bool)
        flat = carried.reshape(-1)
        sup, query = [], []
        for i in range(E):
            q_i = []
            for j in range(W):
                g = i * W + j
                start = g * S + (int(flat[g - 1]) if g > 0 else 0)
                end_q = (g + 1) * S + int(flat[g])
                sup.append(features[start : start + S])
                q_i.append(features[start + S : end_q])
                query_mask[start + S : end_q] = True
            query.append(torch.vstack(q_i))
        support = torch.vstack(sup).contiguous().view(E, W * S, *rest)
    support_target = local[:, :, :S].reshape(E, W * S)
    query_target = local[:, :, S:].reshape(E, W * Q)
    return support, query, support_target, query_target, query_mask


def cls_row_table(repeats, episode_size, way_num, shot_num):
    """int32 [E*W+1] first feature row of every (episode, class) block (the device table the
    kernels consume; derived from the same cumsum as split_by_episode above)."""
    _, carried = class_query_rows(repeats, episode_size, way_num)
    flat = carried.reshape(-1)
    g = np.arange(episode_size * way_num + 1)
    prev = np.concatenate([[0], flat])
    return (g * shot_num + prev).astype(np.int32)


# ---------------------------------------------------------------- heads
def proto_layer(query_feat, support_feat, way_num, shot_num, mode="euclidean"):
    """reference: ProtoLayer.forward, libfewshot_core/model/metric/proto_net.py:34-64.
    query [t, wq, c], support [t, w*s, c] -> [t, wq, w]."""
    t, wq, c = query_feat.shape
    proto = torch.mean(support_feat.reshape(t, way_num, shot_num, c), dim=2)  # :49-50
    if mode == "euclidean":  # :54-57
        return -torch.sum(torch.pow(query_feat.unsqueeze(2) - proto.unsqueeze(1), 2), dim=3)
    if mode == "cos_sim":  # :59-63
        return torch.matmul(F.normalize(query_feat, p=2, dim=-1),
                            torch.transpose(F.normalize(proto, p=2, dim=-1), -1, -2))
    raise KeyError(mode)


def deepbdc_proto_layer(query_feat, support_feat, way_num, shot_num):
    """reference: deepbdc.ProtoLayer.forward, libfewshot_core/model/metric/deepbdc.py:27-53."""
    t = query_feat.shape[0]
    c = support_feat.shape[-1]
    proto = torch.mean(support_feat.reshape(t, way_num, shot_num, c), dim=2)  # :34-35
    if shot_num > 1:  # :37-43
        return -torch.sum(torch.pow(query_feat.unsqueeze(2) - proto.unsqueeze(1), 2), dim=3)
    return torch.matmul(query_feat, torch.transpose(proto, -1, -2))  # :44-53


def dn4_layer(query_feat, support_feat, way_num, shot_num, n_k, return_topk=False):
    """reference: DN4Layer.forward, libfewshot_core/model/metric/dn4.py:39-75.
    query [t, wq, c, h, w], support [t, w*s, c, h, w] -> score [t, wq, w]
    (optionally also the top-k values/indices the reference discards at :72)."""
    t, wq, c, h, w = query_feat.shape
    q = query_feat.reshape(t, wq, c, h * w).permute(0, 1, 3, 2)  # :52-58
    q = F.normalize(q, p=2, dim=-1).unsqueeze(2)  # :59
    s = (support_feat.reshape(t, way_num, shot_num, c, h * w).permute(0, 1, 3, 2, 4)
         .contiguous().view(t, way_num, c, shot_num * h * w))  # :62-67
    s = F.normalize(s, p=2, dim=2).unsqueeze(1)  # :68
    relation = torch.matmul(q, s)  # :71  [t, wq, w, hw, s*hw]
    topv, topi = torch.topk(relation, n_k, dim=-1)  # :72
    score = torch.sum(topv, dim=[3, 4])  # :73
    if return_topk:
        return score, topv, topi, relation
    return score


def bdcovpool(x, t):
    """reference: BDCovpool, libfewshot_core/model/backbone/utils/bdc_pool.py:69-84.
    x [B, dim, h, w], t: log-temperature tensor [1,1].  Runs on x's device and dtype (tests/test_gpu_bdc.py
    evaluates it in float64 on the GPU at batch sizes the CPU would take seconds over)."""
    B, dim, h, w = x.shape
    M = h * w
    x = x.reshape(B, dim, M)
    I = torch.eye(dim, dim, device=x.device).view(1, dim, dim).repeat(B, 1, 1).type(x.dtype)  # :74
    I_M = torch.ones(B, dim, dim, device=x.device).type(x.dtype)  # :75
    x_pow2 = x.bmm(x.transpose(1, 2))  # :76
    dcov = I_M.bmm(x_pow2 * I) + (x_pow2 * I).bmm(I_M) - 2 * x_pow2  # :77
    dcov = torch.clamp(dcov, min=0.0)  # :79
    dcov = torch.exp(t) * dcov  # :80
    dcov = torch.sqrt(dcov + 1e-5)  # :81
    return (dcov - 1.0 / dim * dcov.bmm(I_M) - 1.0 / dim * I_M.bmm(dcov)
            + 1.0 / (dim * dim) * I_M.bmm(dcov).bmm(I_M))  # :82


def triuvec(x):
    """reference: Triuvec, bdc_pool.py:86-93 (row-major upper triangle incl. diagonal).
    The reference's trailing .squeeze() (which drops the batch dim when B == 1) is NOT applied."""
    B, dim, _ = x.shape
    r = x.reshape(B, dim * dim)
    index = torch.ones(dim, dim, device=x.device).triu().reshape(dim * dim).nonzero(as_tuple=False)
    return r[:, index].squeeze(-1)


# ---------------------------------------------------------------- vote / accuracy / CI
def torch_mode_cuda(labels):
    """What torch.mode returns for a 1-D CUDA tensor of <= 2048 integer labels -- the rule the
    reference's CUDA-only set_forward lives by (utils.py:443 called from proto_net.py:116).
    PyTorch's fused small-slice kernel sorts the slice, hands sorted positions (2t, 2t+1) to
    thread t and max-reduces (run count, position) through shuffle-down trees in which the lower
    lane keeps ties, so among equally frequent labels the winner is the one whose run END lies in
    the lane with the smallest bit-reversed (warp id, lane id).  Pinned by measurement on B200 /
    torch 2.11: tools/probe_torch_mode.py -> tests/golden/torch_mode_cuda.npz."""
    y = np.sort(np.asarray(labels).reshape(-1))
    vals, cnt = np.unique(y, return_counts=True)
    mx = cnt.max()
    if mx == 1:
        return int(y[0])
    ends = np.cumsum(cnt) - 1
    rev5 = lambda v: int("{:05b}".format(int(v) & 31)[::-1], 2)
    best = None
    for v, c, e in zip(vals, cnt, ends):
        if c == mx:
            lane = int(e) >> 1
            key = (rev5(lane >> 5), rev5(lane))
            if best is None or key < best[0]:
                best = (key, int(v))
    return best[1]


def majority_vote(logits, query_nums, tie_rule="smallest"):
    """reference: majority_vote, libfewshot_core/utils/utils.py:436-446 (argmax over softmax,
    then torch.mode per query group; returns float32 like the reference).  tie_rule "smallest" is
    torch.mode on this CPU; "torch_cuda" restates what the same call returns on a CUDA slice."""
    y = torch.softmax(torch.as_tensor(logits), dim=1).argmax(dim=1)
    out = torch.zeros(len(query_nums))
    end = 0
    for i, num in enumerate(query_nums):
        sl = y[end : end + int(num)]
        out[i] = torch.mode(sl)[0] if tie_rule == "smallest" else torch_mode_cuda(sl.numpy())
        end += sl.shape[0]
    return out


def vote_categorical_acc(targets, predictions):
    """reference: vote_catagorical_acc, utils.py:432-433."""
    return (predictions == targets).sum().float() / targets.size(0) * 100.0


def average_logits(logits, query_nums):
    """reference: average_logits, utils.py:449-471."""
    out, start = [], 0
    for num in query_nums:
        num = int(num)
        if num == 0:
            out.append(torch.zeros(logits.size(1), dtype=logits.dtype))
            continue
        out.append(logits[start : start + num].mean(dim=0))
        start += num
    return torch.stack(out, dim=0)


def energy_score(logits, query_nums):
    """reference: DeepBDC.set_forward, libfewshot_core/model/metric/deepbdc.py:318-319."""
    return -torch.logsumexp(average_logits(logits, query_nums), dim=1)


def mean_confidence_interval(data, confidence=0.95):
    """reference: mean_confidence_interval, utils.py:148-159."""
    import scipy.stats

    a = np.asarray([1.0 * np.array(d) for d in data])
    n = len(a)
    m, se = np.mean(a), scipy.stats.sem(a)
    h = se * scipy.stats.t.ppf((1 + confidence) / 2.0, n - 1)
    return m, h


# ---------------------------------------------------------------- whole-head drivers
def proto_forward(feat, way_num, shot_num, query_num, repeats, support_size, mode="euclidean",
                  tie_rule="torch_cuda"):
    """reference: ProtoNet.set_forward after emb_func, proto_net.py:103-118.  feat [N, D] (CPU).
    Returns (output [sum R, W], acc, per-query predictions)."""
    support, query, _, query_target, _ = split_by_episode(feat, way_num, shot_num, query_num, repeats, support_size)
    outs = []
    for i in range(len(query)):
        outs.append(proto_layer(query[i].unsqueeze(0), support[i].unsqueeze(0), way_num, shot_num, mode)
                    .reshape(-1, way_num))
    output = torch.cat(outs, dim=0)
    pred = majority_vote(output, repeats, tie_rule).to(torch.long)  # set_forward is CUDA-only: CUDA torch.mode
    acc = vote_categorical_acc(query_target.reshape(-1), pred)
    return output, acc, pred


def dn4_forward(feat, way_num, shot_num, query_num, repeats, support_size, n_k, tie_rule="torch_cuda"):
    """reference: DN4.set_forward after emb_func, dn4.py:100-118.  feat [N, C, H, W]."""
    support, query, _, query_target, _ = split_by_episode(feat, way_num, shot_num, query_num, repeats, support_size)
    outs = []
    for i in range(len(query)):
        outs.append(dn4_layer(query[i].unsqueeze(0), support[i].unsqueeze(0), way_num, shot_num, n_k)
                    .view(-1, way_num))
    output = torch.cat(outs, 0)
    pred = majority_vote(output, repeats, tie_rule).to(torch.long)  # set_forward is CUDA-only: CUDA torch.mode
    acc = vote_categorical_acc(query_target.reshape(-1), pred)
    return output, acc, pred


def deepbdc_forward(feat, way_num, shot_num, query_num, repeats, support_size, tie_rule="torch_cuda"):
    """reference: DeepBDC.set_forward after emb_func, deepbdc.py:291-319.  feat [N, D]."""
    support, query, _, query_target, _ = split_by_episode(feat, way_num, shot_num, query_num, repeats, support_size)
    outs = []
    for i in range(len(query)):
        outs.append(deepbdc_proto_layer(query[i].unsqueeze(0), support[i].unsqueeze(0), way_num, shot_num)
                    .reshape(-1, way_num))
    output = torch.cat(outs, dim=0)
    pred = majority_vote(output, repeats, tie_rule).to(torch.long)  # set_forward is CUDA-only: CUDA torch.mode
    acc = vote_categorical_acc(query_target.reshape(-1), pred)
    return output, acc, pred, energy_score(output, repeats)
