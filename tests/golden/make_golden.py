"""Generate the golden fixtures in this directory by running the UNMODIFIED reference
(a read-only checkout of yzhang1918/www2023tiger) on small seeded synthetic streams:

    TIGER_REFERENCE=<reference checkout> python tests/golden/make_golden.py

Workarounds (SURVEY.md §8(c)): torch_scatter is replaced by tests/golden/_shim
(CPU tie rule of torch_scatter), and load_jodie_data (broken on Python >= 3.11) is
bypassed by constructing InteractionData directly.  Everything else - Graph,
GraphCollator, init_model, TIGER.contrast_learning / restart / flush_msg,
SeqRestarter / StaticRestarter - is the reference's own code.
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
from tiger.model.utils import select_latest_nids, anonymized_reindex  # noqa: E402  (reference)

from www2023tiger_b200.synthetic import StreamShape, make_stream   # noqa: E402

CASES = {
    # name: (shape, nfeat_dim, model kwargs, batch size, n_batches, lazy_restart)
    'seq_left_right': (StreamShape('g1', 40, 12, 900, 8, None, horizon=5000.), 0,
                       dict(dim=None, restarter_type='seq', msg_src='left', upd_src='right', hist_len=6), 30, 14, False),
    'seq_restart_mode': (StreamShape('g2', 40, 12, 900, 8, None, horizon=5000.), 0,
                         dict(dim=None, restarter_type='seq', msg_src='left', upd_src='right', hist_len=6), 30, 14, True),
    'static_right_right_dim10': (StreamShape('g3', 30, 9, 700, 4, 10, horizon=3000.), 0,
                                 dict(dim=10, restarter_type='static', msg_src='right', upd_src='right', hist_len=6), 25, 12, True),
    'seq_noefeat_dim8': (StreamShape('g4', 25, 25, 800, 0, 8, horizon=1.4e8), 0,
                         dict(dim=8, restarter_type='seq', msg_src='left', upd_src='right', hist_len=5), 40, 10, True),
    'seq_nfeats_left_left': (StreamShape('g5', 30, 10, 600, 6, None, horizon=4000.), 12,
                             dict(dim=None, restarter_type='seq', msg_src='left', upd_src='left', hist_len=4), 20, 12, False),
}
# non-default operator variants (SURVEY.md §8(f)3): n_layers = 2 (collator recursion with float32 re-query times,
# data_loader.py:124-131; temporal_agg_modules.py:59-65), hit_type vec | count (tiger.py:261-275), upd_fn merge
# (update_modules.py:40-47), tsfm_fn linear | mlp (message_modules.py:29-55).  Written as var_<name>.npz.
VARIANTS = {
    'var_two_layers': ('seq_left_right', dict(n_layers=2)),
    'var_hit_vec': ('static_right_right_dim10', dict(hit_type='vec')),
    'var_hit_count': ('seq_left_right', dict(hit_type='count')),
    'var_upd_merge': ('seq_left_right', dict(mem_update_type='merge')),
    'var_tsfm_linear': ('static_right_right_dim10', dict(msg_tsfm_type='linear')),
    'var_tsfm_mlp': ('seq_nfeats_left_left', dict(msg_tsfm_type='mlp')),
}
N_NEIGHBORS = 5
N_HEADS = 2


def t2n(x):
    return x.detach().cpu().numpy().copy()   # copy: state tensors are mutated in place later


def run_case(name, shape, nfeat_dim, mk, bs, n_batches, lazy_restart, variant=None):
    variant = {**dict(n_layers=1, hit_type='bin', msg_tsfm_type='id', mem_update_type='gru'), **(variant or {})}
    n_layers = variant['n_layers']
    torch.manual_seed(0)
    np.random.seed(0)
    st = make_stream(shape, seed=1, nfeat_dim=nfeat_dim)
    full = InteractionData(st.src, st.dst, st.ts, st.eids, st.labels, seed=0, eval=True)
    g = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=st.n_nodes - 1)
    coll = GraphCollator(g, N_NEIGHBORS, n_layers, restarter=mk['restarter_type'], hist_len=mk['hist_len'])
    model = init_model(st.nfeats, st.efeats, g, g, full, torch.device('cpu'),
                       feature_as_buffer=True, dim=mk['dim'], n_layers=n_layers, n_heads=N_HEADS,
                       n_neighbors=N_NEIGHBORS, hit_type=variant['hit_type'], dropout=0.1,
                       restarter_type=mk['restarter_type'], hist_len=mk['hist_len'],
                       msg_src=mk['msg_src'], upd_src=mk['upd_src'], msg_tsfm_type=variant['msg_tsfm_type'],
                       mem_update_type=variant['mem_update_type'])
    # non-trivial values for parameters the reference initialises to zero / constants
    with torch.no_grad():
        model.time_encoder.phase.normal_(0, 0.3)
        if mk['restarter_type'] == 'static':
            model.restarter_fn.left_emb.weight.normal_(0, 0.5)
            model.restarter_fn.right_emb.weight.normal_(0, 0.5)
        else:
            model.restarter_fn.time_encoder.phase.normal_(0, 0.3)
    model.eval()
    model.reset()
    out = {'meta_bs': bs, 'meta_n_batches': n_batches, 'meta_lazy_restart': int(lazy_restart),
           'meta_n_neighbors': N_NEIGHBORS, 'meta_n_heads': N_HEADS, 'meta_hist_len': mk['hist_len'],
           'meta_n_nodes': st.n_nodes, 'meta_dim': model.nfeat_dim, 'meta_restarter': mk['restarter_type'],
           'meta_msg_src': mk['msg_src'], 'meta_upd_src': mk['upd_src'],
           'meta_n_layers': n_layers, 'meta_hit_type': variant['hit_type'], 'meta_tsfm': variant['msg_tsfm_type'],
           'meta_upd': variant['mem_update_type'],
           'stream_src': st.src, 'stream_dst': st.dst, 'stream_ts': st.ts, 'stream_eids': st.eids,
           'stream_neg': full.neg_dst}
    if st.efeats is not None:
        out['stream_efeats'] = st.efeats
    if st.nfeats is not None:
        out['stream_nfeats'] = st.nfeats
    for k, v in model.state_dict().items():
        if k.endswith('memory.vals') or k.endswith('update_ts') or k.endswith('active_mask'):
            continue
        out['w_' + k] = t2n(v)
    # adjacency fixtures
    out['adj_lens'] = np.array([len(x) for x in g.node2ts])
    out['adj_nbr'] = np.concatenate([np.asarray(x, dtype=np.int64) for x in g.node2neighbors])
    out['adj_eid'] = np.concatenate([np.asarray(x, dtype=np.int64) for x in g.node2eids])
    out['adj_ts'] = np.concatenate([np.asarray(x, dtype=np.float64) for x in g.node2ts])
    out['adj_flag'] = np.concatenate([np.asarray(x, dtype=np.int64) for x in g.node2flags])

    uptodate = set()
    with torch.no_grad():
        for ib in range(n_batches):
            lo, hi = ib * bs, (ib + 1) * bs
            batch = [full[i] for i in range(lo, hi)]
            src, dst, neg, ts, eids, _, cg = coll(batch)
            p = f'b{ib}_'
            out[p + 'neigh_nids'], out[p + 'neigh_eids'], out[p + 'neigh_ts'] = (t2n(x) for x in cg.layers[1])
            for depth in range(2, n_layers + 1):
                for x, nm in zip(cg.layers[depth], ('neigh_nids', 'neigh_eids', 'neigh_ts')):
                    out[p + f'l{depth}_' + nm] = t2n(x)
            out[p + 'involved'] = cg.np_computation_graph_nodes
            out[p + 'local_index'] = t2n(cg.local_index)
            for hn, hv in zip(('src_hits', 'dst_hits', 'neg_src_hits', 'neg_dst_hits'), cg.hit_data):
                out[p + hn] = t2n(hv)
            rd = cg.restart_data
            out[p + 'r_index'], out[p + 'r_nids'], out[p + 'r_ts'] = t2n(rd.index), t2n(rd.nids), t2n(rd.ts)
            if mk['restarter_type'] == 'seq':
                out[p + 'r_hist_nids'], out[p + 'r_anon'] = t2n(rd.hist_nids), t2n(rd.anonymized_ids)
                out[p + 'r_hist_eids'], out[p + 'r_hist_ts'] = t2n(rd.hist_eids), t2n(rd.hist_ts)
                out[p + 'r_hist_dirs'] = t2n(rd.hist_dirs)
            else:
                out[p + 'r_prev_ts'] = t2n(rd.prev_ts)
            if lazy_restart:                                   # eval_utils.py:37-42
                involved = cg.np_computation_graph_nodes
                restart_nodes = np.array(sorted(set(involved) - uptodate), dtype=np.int64)
                r_nids = torch.from_numpy(restart_nodes).long()
                r_ts = torch.full((len(r_nids),), ts.min().item())
                if len(r_nids):
                    hl, hr, pt = model.restarter_fn(r_nids, r_ts)
                    out[p + 'restart_hl'], out[p + 'restart_hr'], out[p + 'restart_pt'] = t2n(hl), t2n(hr), t2n(pt)
                model.restart(r_nids, r_ts)
                uptodate.update(restart_nodes.tolist())
                out[p + 'restart_nids'] = restart_nodes
            # pending-message nodes before the step (python set -> sorted array)
            out[p + 'pending_before'] = np.array(sorted(int(x) for x in model.msg_store.nodes_with_messages), dtype=np.int64)
            loss, h_left, ps, ns, hpl, hpr = model.contrast_learning(src, dst, neg, ts, eids, cg)
            out[p + 'loss'] = t2n(loss)
            out[p + 'h_left'], out[p + 'pos_scores'], out[p + 'neg_scores'] = t2n(h_left), t2n(ps), t2n(ns)
            out[p + 'h_prev_left'], out[p + 'h_prev_right'] = t2n(hpl), t2n(hpr)
            # restarter on the collated batch + mutual loss (tiger.py:574-590)
            index = rd.index
            sl, sr, _ = model.restarter_fn(torch.cat([src, dst])[index], ts.repeat(2)[index], cg)
            out[p + 'surrogate_left'], out[p + 'surrogate_right'] = t2n(sl), t2n(sr)
            targets = torch.cat([hpl[index], hpr[index]], 0)
            preds = torch.cat([sl, sr], 0)
            valid = torch.where(~(targets == 0).all(1))[0]
            ml = model.mutual_loss_fn(preds[valid], targets[valid]) if len(valid) else torch.tensor(0.)
            out[p + 'mutual_loss'] = t2n(ml)
            # state after the batch
            out[p + 'left_vals'], out[p + 'left_ts'] = t2n(model.left_memory.vals), t2n(model.left_memory.update_ts)
            out[p + 'right_vals'], out[p + 'right_ts'] = t2n(model.right_memory.vals), t2n(model.right_memory.update_ts)
            out[p + 'msg_vals'], out[p + 'msg_ts'] = t2n(model.msg_store.node_msg_vals), t2n(model.msg_store.node_msg_ts)
            out[p + 'pending_after'] = np.array(sorted(int(x) for x in model.msg_store.nodes_with_messages), dtype=np.int64)
        model.flush_msg()
        out['flush_right_vals'], out['flush_right_ts'] = t2n(model.right_memory.vals), t2n(model.right_memory.update_ts)
    # stand-alone known-answer vectors for the index functions
    rng = np.random.RandomState(7)
    ids = rng.randint(1, 15, 60)
    tt = np.floor(rng.uniform(0, 20, 60))
    u, ix = select_latest_nids(torch.from_numpy(ids), torch.from_numpy(tt))
    out['kat_sl_ids'], out['kat_sl_ts'], out['kat_sl_unique'], out['kat_sl_index'] = ids, tt, t2n(u), t2n(ix)
    hh = rng.randint(0, 6, (12, 7))
    hh[:, :2][rng.rand(12, 2) < 0.6] = 0
    out['kat_anon_in'], out['kat_anon_out'] = hh, anonymized_reindex(hh)
    q_n = rng.randint(0, st.n_nodes, 50)
    q_t = np.floor(rng.uniform(0, shape.horizon, 50))
    hn, he_, ht, hd = g.get_history(q_n, q_t, 7)
    out['kat_hist_q_nids'], out['kat_hist_q_ts'] = q_n, q_t
    out['kat_hist_nids'], out['kat_hist_eids'], out['kat_hist_ts'], out['kat_hist_dirs'] = hn, he_, ht, hd
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print(name, 'written;', len(out), 'arrays')


if __name__ == '__main__':
    only = sys.argv[1:]
    for name, args in CASES.items():
        if not only or name in only:
            run_case(name, *args)
    for name, (base, variant) in VARIANTS.items():
        if not only or name in only or 'variants' in only:
            run_case(name, *CASES[base], variant=variant)
