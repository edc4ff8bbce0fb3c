"""DN4 behind the reference's API (libfewshot_core/model/metric/dn4.py:78-155)."""
import torch
from torch import nn

from .. import ops
from .abstract_model import MetricModel
from .proto_net import accuracy_percent


class DN4(MetricModel):
    def __init__(self, n_k=3, precision="fp32", **kwargs):
        """precision (not a reference kwarg): "fp32" keeps the bit-stable head; "tf32" runs the cosine relation
        on the tcgen05 tensor cores in evaluation (Conv64F maps, and ResNet-12 maps through the K-streaming schedule)."""
        super().__init__(**kwargs)
        self.n_k = n_k
        self.precision = precision
        self.loss_func = nn.CrossEntropyLoss()

    def set_forward(self, batch, update_threshold=False, enhance_classification_via_energy=False):
        image, repeats, support_size = self._unpack(batch)
        feat = self.emb_func(image)  # [N, C, H, W]
        tab = self._table(feat.shape[0], repeats, support_size)
        precision = self.precision if ops.dn4_tc_supported(feat.shape[1]) else "fp32"
        output, _, _ = ops.dn4_scores(feat, tab.cls_row, tab.E, tab.W, tab.S, self.n_k, precision=precision)
        _, acc, _ = ops.vote_acc(output, tab.q_start, tab.q_target)
        return output, acc

    def set_forward_loss(self, batch):
        # dn4.py:122-155.  The reference forwards `repeats` to split_by_episode here and then compares
        # per-window scores with per-query targets, which only lines up for one window per query.
        image, repeats, support_size = self._unpack(batch)
        feat = self.emb_func(image)
        tab = self._table(feat.shape[0], repeats, support_size)
        if tab.NQ != tab.nq:
            raise ValueError("DN4.set_forward_loss needs one window per query (dn4.py:141-154)")
        output, _, _ = ops.dn4_scores(feat, tab.cls_row, tab.E, tab.W, tab.S, self.n_k)
        target = tab.q_target_long
        loss = self.loss_func(output, target)
        acc = accuracy_percent(output, target, as_tensor=getattr(self, "acc_on_device", False))
        return output, acc, loss
