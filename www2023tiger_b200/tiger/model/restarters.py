"""Restarters: surrogate models that re-initialise the memory of a node from its raw history
(reference tiger/model/restarters.py:17-114,254-277).

no-grad mode runs the launch sequence of csrc/restart_seq.cu (history and anonymisation come from the
device graph: no host round trip in `restart()`); autograd mode builds the same function with torch
ops so that the mutual-learning loss can train the restarter."""
from typing import Optional, Tuple

import torch
from torch import Tensor, nn
from torch.nn import functional as F

from www2023tiger_b200 import ops
from ._native import f32c, use_kernel
from .basic_modules import MergeLayer
from .feature_getter import FeatureGetter
from .time_encoding import TimeEncode


class Restarter(nn.Module):
    def __init__(self, raw_feat_getter: FeatureGetter, graph):
        super().__init__()
        self.raw_feat_getter = raw_feat_getter
        self.graph = graph
        self.n_nodes = raw_feat_getter.n_nodes
        self.nfeat_dim = raw_feat_getter.nfeat_dim
        self.efeat_dim = raw_feat_getter.efeat_dim
        self.time_encoder = TimeEncode(dim=self.nfeat_dim)
        self.tfeat_dim = self.time_encoder.dim

    def forward(self, nids: Tensor, ts: Tensor, computation_graph=None) -> Tuple[Tensor, Tensor, Tensor]:
        """-> (h(t'-), h(t'+), t') of each node, t' = time of its last event before ts."""
        raise NotImplementedError


class SeqRestarter(Restarter):
    def __init__(self, raw_feat_getter: FeatureGetter, graph, *, hist_len: int = 20, n_head=2, dropout=0.1):
        super().__init__(raw_feat_getter, graph)
        self.hist_len = hist_len
        self.n_head = n_head
        self.dropout = dropout
        self.anony_emb = nn.Embedding(hist_len + 1, self.nfeat_dim)
        self.d_model = self.nfeat_dim * 3 + self.efeat_dim + self.tfeat_dim
        self.mha_fn = nn.MultiheadAttention(self.d_model, n_head, dropout)
        self.out_fn = nn.Linear(self.d_model, self.nfeat_dim)
        self.merger = MergeLayer(self.nfeat_dim, self.d_model - self.tfeat_dim, self.nfeat_dim, self.nfeat_dim,
                                 dropout=dropout)
        self._op, self._op_key = None, None

    # ---- kernel route ----
    def _operator(self, n: int, device) -> ops.SeqRestarterOp:
        if self._op is None or self._op.cap < n or self._op.x.device != device:
            cap = max(256, 1 << (max(n, 1) - 1).bit_length())
            self._op = ops.SeqRestarterOp(self.nfeat_dim, self.efeat_dim, self.hist_len, self.n_head, cap, device)
            self._op_key = None
        key = tuple((p.data_ptr(), p._version) for p in self.parameters())
        if key != self._op_key:
            self._op.set_weights(dict(self.named_parameters()), prefix='')
            self._op_key = key
        return self._op

    def history(self, nids: Tensor, ts: Tensor):
        """get_history + anonymized_reindex on the device graph (reference: host round trip, :67-76)."""
        hn, he, ht, hd = self.graph.find_recent_device(nids.contiguous(), ts.double().contiguous(), self.hist_len)
        return hn, he, ht, hd, ops.anonymized_reindex(hn)

    def fits_kernel(self) -> bool:
        """Whether the kernels take this restarter (ops.seq_restarter_limit_error); past their limits (a history of
        more than 64 events) it runs its torch code, which has none."""
        return ops.seq_restarter_limit_error(self.nfeat_dim, self.efeat_dim, self.hist_len, self.n_head) is None

    def forward(self, nids: Tensor, ts: Tensor, computation_graph=None) -> Tuple[Tensor, Tensor, Tensor]:
        if computation_graph is None:
            hn, he, ht, hd, an = self.history(nids, ts)
        else:
            r = computation_graph.restart_data
            hn, he, ht, hd, an = r.hist_nids, r.hist_eids, r.hist_ts, r.hist_dirs, r.anonymized_ids
        n = nids.numel()
        if use_kernel(self) and hn.is_cuda and self.fits_kernel():
            op = self._operator(n, hn.device)
            fg = self.raw_feat_getter
            hl, hr, pt = op.forward(nids.contiguous(), n, fg.nfeats, fg.efeats,
                                    hist=tuple(t.contiguous() for t in (hn, he, ht, hd, an)))
            return hl.clone(), hr.clone(), pt.clone()
        return self._forward_autograd(nids, hn, he, ht, hd, an)

    # ---- autograd route (training targets of the mutual loss) ----
    def _forward_autograd(self, nids, hn, he, ht, hd, an):
        n, L = hn.shape
        pad = hn == 0
        pad[:, -1] = False                 # set before the emptiness test, so no row is ever "invalid" (:86-88)
        empty = pad.all(1, keepdim=True)
        owner = nids.unsqueeze(1).expand(n, L)
        first = owner * hd + hn * (1 - hd)          # the reference's literal role assignment (:93-94)
        second = owner * (1 - hd) + hn * hd
        fg = self.raw_feat_getter
        tok = torch.cat([fg.get_node_embeddings(first), fg.get_node_embeddings(second), self.anony_emb(an),
                         fg.get_edge_embeddings(he), self.time_encoder(ht[:, -1:] - ht)], 2)
        keep = torch.ones(L, 1, device=tok.device)
        keep[-1] = 0.
        width = self.d_model - self.tfeat_dim
        tok = torch.cat([tok[:, :, :width] * keep, tok[:, :, width:]], 2)    # last token keeps its time code only
        seq = tok.transpose(0, 1)
        out, _ = self.mha_fn(seq, seq, seq, key_padding_mask=pad)
        h_left = self.out_fn(F.relu(out.mean(0)))
        # the merger's second input is the (already zeroed) feature slice of the last token (:103-104)
        h_right = self.merger(h_left, torch.zeros(n, width, device=tok.device))
        return h_left.masked_fill(empty, 0.), h_right.masked_fill(empty, 0.), ht[:, -1]


class StaticRestarter(Restarter):
    def __init__(self, raw_feat_getter: FeatureGetter, graph):
        super().__init__(raw_feat_getter, graph)
        self.left_emb = nn.Embedding(self.n_nodes, self.nfeat_dim)
        self.right_emb = nn.Embedding(self.n_nodes, self.nfeat_dim)
        nn.init.zeros_(self.left_emb.weight)
        nn.init.zeros_(self.right_emb.weight)

    def forward(self, nids: Tensor, ts: Tensor, computation_graph=None) -> Tuple[Tensor, Tensor, Tensor]:
        if computation_graph is None:
            prev_ts = self.graph.find_recent_device(nids.contiguous(), ts.double().contiguous(), 1,
                                                    want_dirs=False)[2][:, 0]
        else:
            prev_ts = computation_graph.restart_data.prev_ts
        if use_kernel() and self.left_emb.weight.is_cuda:
            ids = nids.contiguous()
            return (ops.gather_rows(f32c(self.left_emb.weight), ids)[0],
                    ops.gather_rows(f32c(self.right_emb.weight), ids)[0], prev_ts)
        return self.left_emb(nids), self.right_emb(nids), prev_ts


class WalkRestarter(Restarter):
    """Not constructible from the reference's CLI (init_utils.py:56-57,144-157); name kept for imports."""

    def __init__(self, *a, **k):
        raise NotImplementedError('WalkRestarter is outside the implemented path')
