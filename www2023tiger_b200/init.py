"""Random parameters of the TIGER architecture under the reference's state_dict names
(SURVEY.md §8(b)); initialisers follow the reference / torch defaults: nn.GRUCell and nn.Linear
uniform, nn.MultiheadAttention xavier-uniform with zero biases, MergeLayer xavier-normal
(tiger/model/basic_modules.py:13-14), nn.Embedding N(0,1), static restarter embeddings zero
(tiger/model/restarters.py:259-260), TimeEncode 10^(-9 i/(d-1)) (tiger/model/time_encoding.py:12)."""
import math
from typing import Dict, Optional

import numpy as np
import torch


def time_basis(d: int) -> torch.Tensor:
    return torch.from_numpy(1 / 10 ** np.linspace(0, 9, d)).float()


def random_weights(d: int, de: int, *, n_nodes: int = 0, restarter: Optional[str] = None, hist_len: int = 40,
                   seed: int = 0, nonzero_static: bool = False, n_layers: int = 1, msg_tsfm_type: str = 'id',
                   mem_update_type: str = 'gru', hit_type: str = 'bin',
                   n_neighbors: int = 10) -> Dict[str, torch.Tensor]:
    """msg_tsfm_type / mem_update_type as in build_model: 'linear' adds msg_transform_fn.fn.1 (nn.Linear(M, M)),
    'mlp' fn.1 / fn.4 (nn.Linear(M, M/2), nn.Linear(M/2, M)); 'merge' replaces right_mem_updater.cell by
    right_mem_updater.fn (MergeLayer(M, d, d, d), message_modules.py:37-57, update_modules.py:50-56).
    hit_type as in build_model (tiger.py:129-136), K = n_neighbors: 'count' has a hit_embedding [K+1, d], 'vec' none
    and a score_fn.fc1 [d, 2(d+K)] (MergeLayer(d+K, d+K, d, 1)); 'none' has no hit_embedding."""
    if msg_tsfm_type not in ('id', 'linear', 'mlp') or mem_update_type not in ('gru', 'merge'):
        raise NotImplementedError(f'msg_tsfm_type={msg_tsfm_type}, mem_update_type={mem_update_type}')
    if hit_type not in ('none', 'bin', 'vec', 'count'):
        raise NotImplementedError(f'hit_type={hit_type}')
    g = torch.Generator().manual_seed(seed)
    E, C, M = 2 * d, 2 * d + de, 3 * d + de

    def uniform(shape, bound):
        return (torch.rand(shape, generator=g) * 2 - 1) * bound

    def linear(out_f, in_f, prefix, W):
        W[prefix + 'weight'] = uniform((out_f, in_f), 1 / math.sqrt(in_f))
        W[prefix + 'bias'] = uniform((out_f,), 1 / math.sqrt(in_f))

    def xavier_uniform(shape):
        return uniform(shape, math.sqrt(6.0 / (shape[0] + shape[1])))

    def merge_layer(d1, d2, hidden, out, prefix, W):
        linear(hidden, d1 + d2, prefix + 'fc1.', W)
        linear(out, hidden, prefix + 'fc2.', W)
        for n, (o, i) in (('fc1.weight', (hidden, d1 + d2)), ('fc2.weight', (out, hidden))):
            W[prefix + n] = torch.randn((o, i), generator=g) * math.sqrt(2.0 / (o + i))

    W: Dict[str, torch.Tensor] = {}
    W['time_encoder.basis_freq'] = time_basis(d)
    W['time_encoder.phase'] = torch.zeros(d)
    c = 'right_mem_updater.cell.'
    k = 1 / math.sqrt(d)
    W[c + 'weight_ih'], W[c + 'weight_hh'] = uniform((3 * d, M), k), uniform((3 * d, d), k)
    W[c + 'bias_ih'], W[c + 'bias_hh'] = uniform((3 * d,), k), uniform((3 * d,), k)
    def attention_layer(a, W):
        W[a + 'mha_fn.q_proj_weight'] = xavier_uniform((E, E))
        W[a + 'mha_fn.k_proj_weight'] = xavier_uniform((E, C))
        W[a + 'mha_fn.v_proj_weight'] = xavier_uniform((E, C))
        W[a + 'mha_fn.in_proj_bias'] = torch.zeros(3 * E)
        linear(E, E, a + 'mha_fn.out_proj.', W)
        W[a + 'mha_fn.out_proj.bias'] = torch.zeros(E)
        merge_layer(E, d, d, d, a + 'merger.', W)

    attention_layer('temporal_embedding_fn.fns.0.', W)
    W['hit_embedding.weight'] = torch.randn((2, d), generator=g)
    merge_layer(d, d, d, 1, 'score_fn.', W)
    r = 'restarter_fn.'
    if restarter == 'static':
        if nonzero_static:
            W[r + 'left_emb.weight'] = torch.randn((n_nodes, d), generator=g) * 0.5
            W[r + 'right_emb.weight'] = torch.randn((n_nodes, d), generator=g) * 0.5
        else:
            W[r + 'left_emb.weight'] = torch.zeros(n_nodes, d)
            W[r + 'right_emb.weight'] = torch.zeros(n_nodes, d)
    elif restarter == 'seq':
        dm = 4 * d + de
        W[r + 'time_encoder.basis_freq'] = time_basis(d)
        W[r + 'time_encoder.phase'] = torch.zeros(d)
        W[r + 'anony_emb.weight'] = torch.randn((hist_len + 1, d), generator=g)
        W[r + 'mha_fn.in_proj_weight'] = xavier_uniform((3 * dm, dm))
        W[r + 'mha_fn.in_proj_bias'] = torch.zeros(3 * dm)
        linear(dm, dm, r + 'mha_fn.out_proj.', W)
        W[r + 'mha_fn.out_proj.bias'] = torch.zeros(dm)
        linear(d, dm, r + 'out_fn.', W)
        merge_layer(d, dm - d, d, d, r + 'merger.', W)
    # the lower layers' attention (n_layers > 1) is drawn last, so the weights above do not depend on n_layers
    for i in range(1, n_layers):
        attention_layer(f'temporal_embedding_fn.fns.{i}.', W)
    # the updater / message transform variants likewise (a merge model draws the GRU cell too, then drops it)
    if msg_tsfm_type == 'linear':
        linear(M, M, 'msg_transform_fn.fn.1.', W)
    elif msg_tsfm_type == 'mlp':
        linear(M // 2, M, 'msg_transform_fn.fn.1.', W)
        linear(M, M // 2, 'msg_transform_fn.fn.4.', W)
    if mem_update_type == 'merge':
        for n in ('weight_ih', 'weight_hh', 'bias_ih', 'bias_hh'):
            del W[c + n]
        merge_layer(M, d, d, d, 'right_mem_updater.fn.', W)
    # the hit types likewise (the default 'bin' tensors above are drawn for every hit type, then replaced)
    if hit_type != 'bin':
        del W['hit_embedding.weight']
    if hit_type == 'count':
        W['hit_embedding.weight'] = torch.randn((n_neighbors + 1, d), generator=g)
    elif hit_type == 'vec':
        o, i = d, 2 * (d + n_neighbors)
        W['score_fn.fc1.weight'] = torch.randn((o, i), generator=g) * math.sqrt(2.0 / (o + i))
    return W


def perturb_biases(W: Dict[str, torch.Tensor], seed: int = 1, scale: float = 0.2) -> Dict[str, torch.Tensor]:
    """Give every zero-initialised bias / phase a non-trivial value (parity tests only)."""
    g = torch.Generator().manual_seed(seed)
    out = dict(W)
    for k, v in W.items():
        if (k.endswith('bias') or k.endswith('phase')) and float(v.abs().max()) == 0.0:
            out[k] = torch.randn(v.shape, generator=g) * scale
    return out


def build_model(nfeats, efeats, graph, n_nodes: int, n_edges: int, device, *, dim, n_layers=1, n_heads=2, n_neighbors=10,
                hit_type='bin', dropout=0.1, restarter_type='seq', hist_len=40, msg_src='left', upd_src='right',
                msg_tsfm_type='id', mem_update_type='gru'):
    """The drop-in TIGER model wired exactly like the reference's init_utils.init_model (init_utils.py:126-168), from
    this package's classes; `efeats` / `nfeats` may already be device tensors (large tables are generated in HBM)."""
    from .tiger.model.feature_getter import NumericalFeature
    from .tiger.model.restarters import SeqRestarter, StaticRestarter
    from .tiger.model.tiger import TIGER
    as_t = lambda x: None if x is None else torch.as_tensor(x).float()
    nfeats, efeats = as_t(nfeats), as_t(efeats)
    if nfeats is not None:
        dim = nfeats.shape[1] if dim is None else dim
    if efeats is not None:
        dim = efeats.shape[1] if dim is None else dim
    getter = NumericalFeature(nfeats, efeats, dim=dim, register_buffer=True, device=device)
    getter.n_nodes, getter.n_edges = n_nodes, n_edges
    if restarter_type == 'seq':
        restarter = SeqRestarter(raw_feat_getter=getter, graph=graph, hist_len=hist_len, n_head=n_heads, dropout=dropout)
    elif restarter_type == 'static':
        restarter = StaticRestarter(raw_feat_getter=getter, graph=graph)
    else:
        raise NotImplementedError(restarter_type)
    model = TIGER(raw_feat_getter=getter, graph=graph, restarter=restarter, n_neighbors=n_neighbors, hit_type=hit_type,
                  n_layers=n_layers, n_head=n_heads, dropout=dropout, msg_src=msg_src, upd_src=upd_src,
                  msg_tsfm_type=msg_tsfm_type, mem_update_type=mem_update_type, tgn_mode=True, msg_last_only=True)
    return model.to(device)
