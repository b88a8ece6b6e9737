"""Temporal graph-attention embedding (reference tiger/model/temporal_agg_modules.py:15-83,173-235).

no-grad mode: one fused kernel per layer (gathers, time encoding, folded single-query attention,
masked softmax, out-projection, merger).  autograd mode: the same math with torch ops."""
from typing import Optional

import torch
from torch import Tensor, nn

from www2023tiger_b200 import ops
from ._native import f32c, use_kernel
from .basic_modules import MergeLayer
from .feature_getter import NumericalFeature
from .time_encoding import TimeEncode


class TemporalAttention(nn.Module):
    def __init__(self, nfeat_dim, efeat_dim, tfeat_dim, n_head=2, dropout=0.1):
        super().__init__()
        if tfeat_dim != nfeat_dim:
            raise NotImplementedError('tfeat_dim must equal nfeat_dim (as everywhere in the reference)')
        self.n_head = n_head
        self.dropout = dropout
        self.nfeat_dim, self.efeat_dim = nfeat_dim, efeat_dim
        self.query_dim = nfeat_dim + tfeat_dim
        self.key_dim = nfeat_dim + efeat_dim + tfeat_dim
        self.merger = MergeLayer(self.query_dim, nfeat_dim, nfeat_dim, nfeat_dim)
        self.mha_fn = nn.MultiheadAttention(embed_dim=self.query_dim, num_heads=self.n_head, dropout=self.dropout,
                                            kdim=self.key_dim, vdim=self.key_dim)
        self._pack, self._pack_key = None, None

    def packed(self, time_encoder: Optional[TimeEncode] = None) -> ops.AttnPack:
        m, g = self.mha_fn, self.merger
        params = [m.q_proj_weight, m.k_proj_weight, m.v_proj_weight, m.in_proj_bias, m.out_proj.weight,
                  m.out_proj.bias, g.fc1.weight, g.fc1.bias, g.fc2.weight, g.fc2.bias]
        if time_encoder is not None:
            params += [time_encoder.basis_freq, time_encoder.phase]
        key = tuple((p.data_ptr(), p._version) for p in params)
        if self._pack is None or key != self._pack_key:
            dev = params[0].device
            if self._pack is None or self._pack.folded.device != dev:
                self._pack = ops.AttnPack(self.nfeat_dim, self.efeat_dim, dev, self.n_head)
            if time_encoder is None:
                zeros = torch.zeros(self.nfeat_dim, device=dev)
                params = params + [zeros, zeros]
            self._pack.refresh(*[f32c(p) for p in params])
            self._pack_key = key
        return self._pack

    def fits_kernel(self, k: int) -> bool:
        """Whether the attention kernel takes this layer with k neighbor slots (ops.attention_limit_error); past its
        limits the layer runs its torch code, which has none."""
        return ops.attention_limit_error(self.nfeat_dim, self.efeat_dim, k, self.n_head) is None

    def forward(self, qx: Tensor, qt: Tensor, kx: Tensor, ky: Tensor, kt: Tensor, padding_mask: Tensor) -> Tensor:
        """qx [n,d] qt [n,d] kx [n,len,d] ky [n,len,de] kt [n,len,d]; padding_mask [n,len], True = padding."""
        if use_kernel(self) and qx.is_cuda and self.fits_kernel(kx.shape[1]):
            return ops.temporal_attention_dense(self.packed(), self.n_head, f32c(qx), f32c(qt), f32c(kx), f32c(ky),
                                                f32c(kt), padding_mask)
        query = torch.cat([qx, qt], 1).unsqueeze(0)
        kv = torch.cat([kx, ky, kt], 2).transpose(0, 1)
        mask = padding_mask.bool().clone()
        empty = mask.all(1, keepdim=True)
        mask[empty.squeeze(1), -1] = False                  # keep the softmax finite for neighbor-less rows
        h, _ = self.mha_fn(query, kv, kv, key_padding_mask=mask)
        h = h.squeeze(0).masked_fill(empty, 0.)             # ... whose attention output is defined as zero
        return self.merger(h, qx)


class GraphEmbedding(nn.Module):
    def __init__(self, raw_feat_getter: NumericalFeature, time_encoder: TimeEncode, graph, n_neighbors=20,
                 n_layers=2):
        super().__init__()
        self.raw_feat_getter = raw_feat_getter
        self.time_encoder = time_encoder
        self.graph = graph
        self.n_neighbors = n_neighbors
        self.n_layers = n_layers

    @property
    def device(self):
        return self.raw_feat_getter.device

    def compute_embedding_with_computation_graph(self, involved_node_reprs: Tensor, center_nids: Tensor, ts: Tensor,
                                                 computation_graph, depth: Optional[int] = None) -> Tensor:
        """h(t-) of `center_nids` at `ts` from the h(t'+) rows of the involved nodes
        (`involved_node_reprs[computation_graph.local_index[u]]`)."""
        depth = self.n_layers if depth is None else depth
        cg = computation_graph
        if (depth == 1 and use_kernel(self) and involved_node_reprs.is_cuda and hasattr(self, 'fns')
                and self.fns[self.n_layers - 1].fits_kernel(cg.layers[1][0].shape[1])):
            nn_, ne_, nt_ = cg.layers[1]
            fn = self.fns[self.n_layers - 1]
            return ops.temporal_attention(fn.packed(self.time_encoder), fn.n_head, center_nids.contiguous(), f32c(ts),
                                          nn_, ne_, nt_, rows_a=None, rows_b=f32c(involved_node_reprs),
                                          sel=cg.local_index, nfeats=self.raw_feat_getter.nfeats,
                                          efeats=self.raw_feat_getter.efeats)
        center = involved_node_reprs[cg.local_index[center_nids]] + self.raw_feat_getter.get_node_embeddings(center_nids)
        if depth == 0:
            return center
        nn_, ne_, nt_ = cg.layers[depth]
        n_center, k = nn_.shape
        neigh = self.compute_embedding_with_computation_graph(
            involved_node_reprs, nn_.flatten(), torch.repeat_interleave(ts, k), cg, depth - 1)   # TGN time convention
        neigh = neigh.reshape(n_center, k, -1)
        delta = ts[:, None] - nt_
        return self.aggregate(depth=depth, center_x=center,
                              center_tx=self.time_encoder(torch.zeros_like(delta[:, 0])), neigh_x=neigh,
                              edge_x=self.raw_feat_getter.get_edge_embeddings(ne_),
                              edge_tx=self.time_encoder(delta), mask=(nn_ == 0))

    def aggregate(self, depth, center_x, center_tx, neigh_x, edge_x, edge_tx, mask) -> Tensor:
        raise NotImplementedError


class GraphAttnEmbedding(GraphEmbedding):
    def __init__(self, raw_feat_getter: NumericalFeature, time_encoder: TimeEncode, graph, n_neighbors=20,
                 n_layers=2, n_head=2, dropout=0.1):
        super().__init__(raw_feat_getter, time_encoder, graph, n_neighbors, n_layers)
        self.n_head = n_head
        self.dropout = dropout
        self.fns = nn.ModuleList([
            TemporalAttention(nfeat_dim=raw_feat_getter.nfeat_dim, efeat_dim=raw_feat_getter.efeat_dim,
                              tfeat_dim=time_encoder.dim, n_head=n_head, dropout=dropout)
            for _ in range(n_layers)])

    def aggregate(self, depth, center_x, center_tx, neigh_x, edge_x, edge_tx, mask) -> Tensor:
        return self.fns[self.n_layers - depth](qx=center_x, qt=center_tx, kx=neigh_x, ky=edge_x, kt=edge_tx,
                                               padding_mask=mask)
