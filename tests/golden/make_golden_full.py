"""Full-dimension golden fixtures: the UNMODIFIED reference (a read-only checkout of yzhang1918/www2023tiger) at the
dimensions of the BASELINE.json configs - d / d_e / K / hist_len / batch = the config values, on the BASELINE-shaped
synthetic streams themselves (not on toy streams):

    TIGER_REFERENCE=<reference checkout> python tests/golden/make_golden_full.py

The streams and the parameters are NOT stored: both are regenerated bit-identically from seeds by
`www2023tiger_b200.synthetic.make_stream` and `www2023tiger_b200.init.random_weights` (+ `perturb_biases`), which
the generator loads into the reference model with `load_state_dict`.  Stored per recorded batch: the complete
integer results (neighbor tables, involved / restart / pending node lists, argmax-by-timestamp winners), the scores
and losses, and for the wide float tensors (embeddings, restarter outputs, the three state tables) a fixed sample
of complete rows plus float64 row / table sums of everything, so that a fixture stays under 1 MB.

Protocol per case (eval_utils.py:29-46 with restart_mode=True): reset at event `start`, WARM lazy-restart batches,
then REC recorded batches; afterwards the restarter on the collated batch + the mutual loss (tiger.py:574-590).
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

from www2023tiger_b200.init import perturb_biases, random_weights  # noqa: E402
from www2023tiger_b200.synthetic import SHAPES, NegativeSampler, make_stream   # noqa: E402

B, K, H, HIST = 200, 10, 2, 40
WARM, REC = 5, 5
N_NODES_KEPT = 16    # state-table rows kept in full per batch
WEIGHT_SEED = 3

# name: (BASELINE shape, restarter, first event of the window, embedding rows kept in full (half src, half dst
# positions), restarter output rows kept in full); the 172-wide cases keep fewer rows to stay under 1 MB
CASES = {
    'full_wikipedia_seq': ('wikipedia', 'seq', 60000, 48, 16),
    'full_reddit_static': ('reddit', 'static', 100000, 48, 16),
    'full_mooc_seq_right_right': ('mooc', 'seq', 60000, 96, 32),
    'full_lastfm_seq_noefeat': ('lastfm', 'seq', 100000, 96, 32),
}


def t2n(x):
    return x.detach().cpu().numpy().copy()


def sums(a):
    a = np.asarray(a, dtype=np.float64)
    return np.array([a.sum(), np.abs(a).sum()])


def case_weights(st, restarter):
    d = st.dim
    de = st.efeats.shape[1] if st.efeats is not None else d
    return perturb_biases(random_weights(d, de, n_nodes=st.n_nodes, restarter=restarter, hist_len=HIST,
                                         seed=WEIGHT_SEED, nonzero_static=True))


def run_case(name, shape_name, restarter, start, n_rows, n_restart_rows):
    shape = SHAPES[shape_name]
    st = make_stream(shape, seed=0)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events, B)
    E = start + (WARM + REC) * B
    data = InteractionData(st.src[:E], st.dst[:E], st.ts[:E], st.eids[:E], st.labels[:E], seed=0, eval=True,
                           neg_dst=neg[:E])
    g = Graph.from_data(data, strategy='recent_edges', seed=0, max_node_id=st.n_nodes - 1)
    coll = GraphCollator(g, K, 1, restarter=restarter, hist_len=HIST)
    torch.manual_seed(0)
    efeats = st.efeats[:E + 1] if st.efeats is not None else None

    class _Len:
        def __len__(self):
            return st.n_events
    model = init_model(None, efeats, g, g, _Len(), torch.device('cpu'), feature_as_buffer=True, dim=shape.dim,
                       n_layers=1, n_heads=H, n_neighbors=K, hit_type='bin', dropout=0.1, restarter_type=restarter,
                       hist_len=HIST, msg_src=shape.msg_src, upd_src=shape.upd_src, msg_tsfm_type='id',
                       mem_update_type='gru')
    W = case_weights(st, restarter)
    missing, unexpected = model.load_state_dict(W, strict=False)
    assert not unexpected, unexpected
    # memories / feature buffers are state, not parameters; the time encoder is one module registered under three
    # names (tiger.py:71-72,121-127), loaded through `time_encoder.*`; the static restarter owns a time encoder it
    # never uses (restarters.py:17-33,254-277), left at its defaults
    sd = model.state_dict()
    for k in missing:
        alias = k.endswith(('time_encoder.basis_freq', 'time_encoder.phase')) and (
            sd[k].data_ptr() == sd['time_encoder.' + k.rsplit('.', 1)[1]].data_ptr()
            or (restarter == 'static' and k.startswith('restarter_fn.')))
        assert 'memory' in k or 'raw_feat_getter' in k or alias, k
    model.eval()
    model.reset()
    out = {'meta_shape': shape_name, 'meta_restarter': restarter, 'meta_start': start, 'meta_warm': WARM,
           'meta_rec': REC, 'meta_bs': B, 'meta_n_neighbors': K, 'meta_n_heads': H, 'meta_hist_len': HIST,
           'meta_weight_seed': WEIGHT_SEED, 'meta_n_rows': n_rows, 'meta_dim': model.nfeat_dim}
    i32 = lambda a: np.asarray(a).astype(np.int32)
    rows_kept = np.concatenate([np.arange(n_rows // 2), B + np.arange(n_rows // 2)])
    uptodate = set()
    with torch.no_grad():
        for ib in range(WARM + REC):
            lo = start + ib * B
            src, dst, negs, ts, eids, _, cg = coll([data[i] for i in range(lo, lo + B)])
            involved = cg.np_computation_graph_nodes
            restart_nodes = np.array(sorted(set(involved) - uptodate), dtype=np.int64)
            r_nids = torch.from_numpy(restart_nodes).long()
            r_ts = torch.full((len(r_nids),), ts.min().item())
            rec = ib >= WARM
            p = f'b{ib - WARM}_'
            if rec and len(r_nids):
                hl, hr, pt = model.restarter_fn(r_nids, r_ts)
                keep = min(n_restart_rows, len(r_nids))
                out[p + 'restart_hl'], out[p + 'restart_hr'] = t2n(hl[:keep]), t2n(hr[:keep])
                out[p + 'restart_hl_rowsum'] = t2n(hl.double().sum(1))
                out[p + 'restart_hr_rowsum'] = t2n(hr.double().sum(1))
                out[p + 'restart_pt'] = t2n(pt)
            model.restart(r_nids, r_ts)
            uptodate.update(restart_nodes.tolist())
            pending_before = np.array(sorted(int(x) for x in model.msg_store.nodes_with_messages), dtype=np.int64)
            loss, h_left, ps, ns, hpl, hpr = model.contrast_learning(src, dst, negs, ts, eids, cg)
            if not rec:
                continue
            out[p + 'neigh_nids'], out[p + 'neigh_eids'] = i32(t2n(cg.layers[1][0])), i32(t2n(cg.layers[1][1]))
            out[p + 'neigh_ts'] = t2n(cg.layers[1][2])
            out[p + 'involved'], out[p + 'restart_nids'] = i32(involved), i32(restart_nodes)
            out[p + 'outdated'] = i32(np.intersect1d(pending_before, involved))
            rd = cg.restart_data
            out[p + 'r_index'] = i32(t2n(rd.index))
            out[p + 'h_left'] = t2n(h_left)[rows_kept]
            out[p + 'h_left_rowsum'] = t2n(h_left.double().sum(1))
            out[p + 'pos_scores'], out[p + 'neg_scores'], out[p + 'loss'] = t2n(ps), t2n(ns), t2n(loss)
            out[p + 'h_prev_left_rowsum'] = t2n(hpl.double().sum(1))
            out[p + 'h_prev_right_rowsum'] = t2n(hpr.double().sum(1))
            index = rd.index
            sl, sr, _ = model.restarter_fn(torch.cat([src, dst])[index], ts.repeat(2)[index], cg)
            out[p + 'surrogate_left_rowsum'] = t2n(sl.double().sum(1))
            out[p + 'surrogate_right_rowsum'] = t2n(sr.double().sum(1))
            out[p + 'surrogate_left'] = t2n(sl[:16])
            targets = torch.cat([hpl[index], hpr[index]], 0)
            preds = torch.cat([sl, sr], 0)
            valid = torch.where(~(targets == 0).all(1))[0]
            ml = model.mutual_loss_fn(preds[valid], targets[valid]) if len(valid) else torch.tensor(0.)
            out[p + 'mutual_loss'] = t2n(ml)
            # state after the batch: complete rows of a fixed sample of this batch's positive nodes, the clocks of
            # all of them, float64 sums of each whole table, the complete pending list
            pos = np.unique(np.concatenate([t2n(src), t2n(dst)]))
            kept = pos[:: max(1, len(pos) // N_NODES_KEPT)][:N_NODES_KEPT]
            out[p + 'kept_nodes'] = i32(kept)
            for tname, tab in (('left_vals', model.left_memory.vals), ('right_vals', model.right_memory.vals),
                               ('msg_vals', model.msg_store.node_msg_vals)):
                out[p + tname + '_rows'] = t2n(tab[kept])
                # rows of nodes that are not pending hold stale message data in the reference too (Q1), so the
                # whole-table sums are well defined
                out[p + tname + '_sums'] = sums(t2n(tab))
            out[p + 'pos_nodes'] = i32(pos)
            out[p + 'left_ts_pos'], out[p + 'right_ts_pos'] = (t2n(model.left_memory.update_ts[pos]),
                                                               t2n(model.right_memory.update_ts[pos]))
            out[p + 'msg_ts_pos'] = t2n(model.msg_store.node_msg_ts[pos])
            out[p + 'pending_after'] = i32(sorted(int(x) for x in model.msg_store.nodes_with_messages))
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print(name, 'written;', len(out), 'arrays;', os.path.getsize(os.path.join(HERE, name + '.npz')) // 1024, 'KB')


if __name__ == '__main__':
    only = sys.argv[1:]
    for name, args in CASES.items():
        if not only or name in only:
            run_case(name, *args)
