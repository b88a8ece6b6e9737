"""Golden fixtures of the TRAINING step: losses and parameter gradients of the UNMODIFIED reference
(a read-only checkout of yzhang1918/www2023tiger) for the loop body of train_self_supervised.py:143-171 (zero_grad ->
contrast_and_mutual_learning -> (contrast + mutual).backward()), on the toy streams of make_golden.py, in train()
mode with dropout = 0 (dropout masks are not reproducible across implementations), no optimizer step (the
parameters stay at their initial values so that every recorded batch is comparable on its own).

    TIGER_REFERENCE=<reference checkout> python tests/golden/make_golden_train.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(HERE, '_shim'))
REFERENCE = os.environ.get('TIGER_REFERENCE', '')
if not os.path.isdir(os.path.join(REFERENCE, 'tiger')):
    sys.exit('set TIGER_REFERENCE to a checkout of the reference (the directory that holds tiger/)')
sys.path.insert(0, REFERENCE)
sys.path.insert(0, ROOT)

from init_utils import init_model                                   # noqa: E402  (reference)
from tiger.data.data_loader import GraphCollator, InteractionData  # noqa: E402  (reference)
from tiger.data.graph import Graph                                 # noqa: E402  (reference)

from www2023tiger_b200.synthetic import StreamShape, make_stream   # noqa: E402

CASES = {
    # name: (shape, nfeat_dim, model kwargs, batch size, n_batches)
    'train_seq_left_right': (StreamShape('t1', 40, 12, 900, 8, None, horizon=5000.), 0,
                             dict(dim=None, restarter_type='seq', msg_src='left', upd_src='right', hist_len=6), 30, 8),
    'train_static_right_right_dim10': (StreamShape('t2', 30, 9, 700, 4, 10, horizon=3000.), 0,
                                       dict(dim=10, restarter_type='static', msg_src='right', upd_src='right', hist_len=6), 25, 8),
    'train_seq_nfeats_left_left': (StreamShape('t3', 30, 10, 600, 6, None, horizon=4000.), 12,
                                   dict(dim=None, restarter_type='seq', msg_src='left', upd_src='left', hist_len=4), 20, 8),
}
N_NEIGHBORS, N_HEADS = 5, 2


def t2n(x):
    return x.detach().cpu().numpy().copy()


def run_case(name, shape, nfeat_dim, mk, bs, n_batches):
    torch.manual_seed(0)
    np.random.seed(0)
    st = make_stream(shape, seed=1, nfeat_dim=nfeat_dim)
    full = InteractionData(st.src, st.dst, st.ts, st.eids, st.labels, seed=0, eval=True)
    g = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=st.n_nodes - 1)
    coll = GraphCollator(g, N_NEIGHBORS, 1, restarter=mk['restarter_type'], hist_len=mk['hist_len'])
    model = init_model(st.nfeats, st.efeats, g, g, full, torch.device('cpu'), feature_as_buffer=True, dim=mk['dim'],
                       n_layers=1, n_heads=N_HEADS, n_neighbors=N_NEIGHBORS, hit_type='bin', dropout=0.0,
                       restarter_type=mk['restarter_type'], hist_len=mk['hist_len'], msg_src=mk['msg_src'],
                       upd_src=mk['upd_src'], msg_tsfm_type='id', mem_update_type='gru')
    with torch.no_grad():
        model.time_encoder.phase.normal_(0, 0.3)
        if mk['restarter_type'] == 'static':
            model.restarter_fn.left_emb.weight.normal_(0, 0.5)
            model.restarter_fn.right_emb.weight.normal_(0, 0.5)
        else:
            model.restarter_fn.time_encoder.phase.normal_(0, 0.3)
    model.train()
    model.reset()
    out = {'meta_bs': bs, 'meta_n_batches': n_batches, 'meta_n_neighbors': N_NEIGHBORS, 'meta_n_heads': N_HEADS,
           'meta_hist_len': mk['hist_len'], 'meta_n_nodes': st.n_nodes, 'meta_dim': model.nfeat_dim,
           'meta_restarter': mk['restarter_type'], 'meta_msg_src': mk['msg_src'], 'meta_upd_src': mk['upd_src'],
           'meta_lazy_restart': 0,
           'stream_src': st.src, 'stream_dst': st.dst, 'stream_ts': st.ts, 'stream_eids': st.eids,
           'stream_neg': full.neg_dst}
    if st.efeats is not None:
        out['stream_efeats'] = st.efeats
    if st.nfeats is not None:
        out['stream_nfeats'] = st.nfeats
    seen = set()
    params = []
    for k, p in model.named_parameters():
        if id(p) in seen:
            continue
        seen.add(id(p))
        params.append((k, p))
        out['w_' + k] = t2n(p)
    for ib in range(n_batches):
        batch = [full[i] for i in range(ib * bs, (ib + 1) * bs)]
        src, dst, neg, ts, eids, _, cg = coll(batch)
        model.zero_grad(set_to_none=True)
        contrast, mutual = model.contrast_and_mutual_learning(src, dst, neg, ts, eids, cg)
        (contrast + mutual).backward()
        p = f'b{ib}_'
        out[p + 'contrast'], out[p + 'mutual'] = t2n(contrast), t2n(mutual)
        if ib >= 3:                                   # histories and memories populated
            for k, prm in params:
                out[p + 'g_' + k] = t2n(prm.grad) if prm.grad is not None else np.zeros(tuple(prm.shape), np.float32)
    out['final_left_vals'], out['final_right_vals'] = t2n(model.left_memory.vals), t2n(model.right_memory.vals)
    out['final_msg_vals'] = t2n(model.msg_store.node_msg_vals)
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print(name, 'written;', len(out), 'arrays;', os.path.getsize(os.path.join(HERE, name + '.npz')) // 1024, 'KB')


if __name__ == '__main__':
    for name, args in CASES.items():
        run_case(name, *args)
