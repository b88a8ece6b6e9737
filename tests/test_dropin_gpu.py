"""The drop-in class surface (www2023tiger_b200/tiger) driven exactly like the reference's drivers drive
theirs - DataLoader + GraphCollator -> lazy restart -> contrast_learning / contrast_and_mutual_learning
- and compared with the golden outputs of the unmodified reference on the same streams."""
import numpy as np
import pytest
import torch
from torch.utils.data import DataLoader

from golden_utils import CASES, VAR_CASES, Golden, assert_close
import dropin_utils as D
from tiger.data.data_loader import GraphCollator, InteractionData
from tiger.data.graph import Graph
from tiger.eval_utils import eval_edge_prediction
from tiger.model.utils import anonymized_reindex, select_latest_nids
from tiger.utils import BackgroundThreadGenerator

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = torch.device('cuda')
cpu = lambda t: t.detach().cpu().numpy()


def setup(g, dropout=0.1):
    full = InteractionData(g.src, g.dst, g.ts, g.eids, np.zeros_like(g.src), seed=0, eval=True, neg_dst=g.neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    coll = GraphCollator(graph, g.K, g.n_layers, restarter=g.restarter, hist_len=g.hist_len)
    dl = DataLoader(full, batch_size=g.bs, collate_fn=coll, pin_memory=True)
    model = D.load_golden_weights(D.model_from_golden(g, graph, DEV, dropout=dropout), g)
    return full, graph, coll, dl, model


def to_dev(batch):
    src, dst, neg, ts, eids, _, cg = batch
    return (src.long().to(DEV), dst.long().to(DEV), neg.long().to(DEV), ts.float().to(DEV), eids.long().to(DEV),
            cg.to(DEV))


@pytest.mark.parametrize('name', CASES)
def test_graph_and_index_functions_match_reference(name):
    g = Golden(name)
    full, graph, *_ = setup(g)
    z = g.z
    hn, he, ht, hd = graph.get_history(z['kat_hist_q_nids'], z['kat_hist_q_ts'], 7)
    assert np.array_equal(hn, z['kat_hist_nids']) and np.array_equal(he, z['kat_hist_eids'])
    assert np.array_equal(ht, z['kat_hist_ts']) and np.array_equal(hd, z['kat_hist_dirs'])
    assert ht.dtype == np.float32 and hn.dtype == np.int64
    u, ix = select_latest_nids(torch.from_numpy(z['kat_sl_ids']), torch.from_numpy(z['kat_sl_ts']))
    assert np.array_equal(u.numpy(), z['kat_sl_unique']) and np.array_equal(ix.numpy(), z['kat_sl_index'])
    assert np.array_equal(anonymized_reindex(z['kat_anon_in']), z['kat_anon_out'])
    with pytest.raises(NotImplementedError):
        graph.sample_temporal_neighbor(np.array([1]), np.array([5.0]), 3, strategy='uniform')


def test_graph_from_adjacency_list_equals_from_data():
    g = Golden(CASES[0])
    full, graph, *_ = setup(g)
    adj = [[] for _ in range(g.N)]
    for s, d, t, e in zip(g.src, g.dst, g.ts, g.eids):          # data2adjlist (graph.py:226-241)
        adj[s].append((d, e, t, 0))
        adj[d].append((s, e, t, 1))
    g2 = Graph(adj, strategy='recent_edges', seed=0)
    for a, b in zip((graph.csr.indptr, graph.csr.nbr, graph.csr.eid, graph.csr.ts, graph.csr.flag),
                    (g2.csr.indptr, g2.csr.nbr, g2.csr.eid, g2.csr.ts, g2.csr.flag)):
        assert torch.equal(a, b)


@pytest.mark.parametrize('name', CASES + VAR_CASES)
def test_dropin_replays_reference_golden(name):
    """CASES: the default operators (fused kernel route).  VAR_CASES: the non-default variants of SURVEY.md §8(f)3 -
    n_layers = 2, hit_type vec | count, upd_fn merge, tsfm_fn linear | mlp - whose index / memory operators run the
    same kernels while the variant-specific dense pieces go through the operator modules."""
    g = Golden(name)
    full, graph, coll, dl, model = setup(g)
    model.eval()
    model.reset()
    uptodate = set()
    with torch.no_grad():
        for ib, batch in enumerate(BackgroundThreadGenerator(dl)):
            if ib >= g.n_batches:
                break
            what = f'{name} b{ib} '
            src, dst, neg, ts, eids, cg = to_dev(batch)
            # ---- collator outputs (data_loader.py:77-168) ----
            assert np.array_equal(cpu(cg.layers[1][0]), g.b(ib, 'neigh_nids')), what
            assert np.array_equal(cpu(cg.layers[1][1]), g.b(ib, 'neigh_eids')), what
            assert np.array_equal(cpu(cg.layers[1][2]), g.b(ib, 'neigh_ts')), what
            for depth in range(2, g.n_layers + 1):
                for j, nm in enumerate(('neigh_nids', 'neigh_eids', 'neigh_ts')):
                    assert np.array_equal(cpu(cg.layers[depth][j]), g.b(ib, f'l{depth}_{nm}')), what + f'layer {depth} {nm}'
            assert np.array_equal(cg.np_computation_graph_nodes, g.b(ib, 'involved')), what
            assert np.array_equal(cpu(cg.local_index), g.b(ib, 'local_index')), what
            for got, key in zip(cg.hit_data, ('src_hits', 'dst_hits', 'neg_src_hits', 'neg_dst_hits')):
                assert np.array_equal(cpu(got), g.b(ib, key)), what + key
            rd = cg.restart_data
            assert np.array_equal(cpu(rd.index), g.b(ib, 'r_index')) and np.array_equal(cpu(rd.nids), g.b(ib, 'r_nids'))
            assert np.array_equal(cpu(rd.ts), g.b(ib, 'r_ts'))
            if g.restarter == 'seq':
                for got, key in ((rd.hist_nids, 'r_hist_nids'), (rd.anonymized_ids, 'r_anon'),
                                 (rd.hist_eids, 'r_hist_eids'), (rd.hist_ts, 'r_hist_ts'), (rd.hist_dirs, 'r_hist_dirs')):
                    assert np.array_equal(cpu(got), g.b(ib, key)), what + key
            else:
                assert np.array_equal(cpu(rd.prev_ts), g.b(ib, 'r_prev_ts'))
            # ---- lazy restart exactly as eval_utils.py:37-42 ----
            if g.lazy_restart:
                fresh = set(cg.np_computation_graph_nodes.tolist()) - uptodate
                r_nids = torch.tensor(sorted(fresh), dtype=torch.long, device=DEV)
                r_ts = torch.full((len(r_nids),), ts.min().item(), device=DEV)
                if len(r_nids):
                    hl, hr, pt = model.restarter_fn(r_nids, r_ts)
                    assert_close(cpu(hl), g.b(ib, 'restart_hl'), TOL, what + 'restart_hl')
                    assert_close(cpu(hr), g.b(ib, 'restart_hr'), TOL, what + 'restart_hr')
                    assert np.array_equal(cpu(pt), g.b(ib, 'restart_pt'))
                model.restart(r_nids, r_ts)
                uptodate.update(fresh)
            assert sorted(model.msg_store.nodes_with_messages) == g.b(ib, 'pending_before').tolist(), what
            # ---- the step ----
            loss, h_left, ps, ns, hpl, hpr = model.contrast_learning(src, dst, neg, ts, eids, cg)
            assert_close(cpu(loss).reshape(1), g.b(ib, 'loss').reshape(1), TOL, what + 'loss')
            assert_close(cpu(h_left), g.b(ib, 'h_left'), TOL, what + 'h_left')
            assert_close(cpu(ps), g.b(ib, 'pos_scores'), TOL, what + 'pos')
            assert_close(cpu(ns), g.b(ib, 'neg_scores'), TOL, what + 'neg')
            assert_close(cpu(hpl), g.b(ib, 'h_prev_left'), TOL, what + 'hpl')
            assert_close(cpu(hpr), g.b(ib, 'h_prev_right'), TOL, what + 'hpr')
            # ---- restarter on the collated batch + mutual loss (tiger.py:574-590) ----
            index = rd.index
            sl, sr, _ = model.restarter_fn(torch.cat([src, dst])[index], ts.repeat(2)[index], cg)
            assert_close(cpu(sl), g.b(ib, 'surrogate_left'), TOL, what + 'surrogate_left')
            assert_close(cpu(sr), g.b(ib, 'surrogate_right'), TOL, what + 'surrogate_right')
            targets = torch.cat([hpl[index], hpr[index]], 0)
            valid = torch.where(~(targets == 0).all(1))[0]
            if len(valid):
                ml = model.mutual_loss_fn(torch.cat([sl, sr], 0)[valid], targets[valid])
                assert_close(cpu(ml).reshape(1), g.b(ib, 'mutual_loss').reshape(1), 2e-5, what + 'mutual')
            # ---- state after the batch ----
            assert_close(cpu(model.left_memory.vals), g.b(ib, 'left_vals'), TOL, what + 'left_vals')
            assert_close(cpu(model.right_memory.vals), g.b(ib, 'right_vals'), TOL, what + 'right_vals')
            assert np.array_equal(cpu(model.left_memory.update_ts), g.b(ib, 'left_ts')), what
            assert np.array_equal(cpu(model.right_memory.update_ts), g.b(ib, 'right_ts')), what
            assert_close(cpu(model.msg_store.node_msg_vals), g.b(ib, 'msg_vals'), TOL, what + 'msg_vals')
            assert np.array_equal(cpu(model.msg_store.node_msg_ts), g.b(ib, 'msg_ts')), what
            assert sorted(model.msg_store.nodes_with_messages) == g.b(ib, 'pending_after').tolist(), what
        model.flush_msg()
        assert_close(cpu(model.right_memory.vals), g.z['flush_right_vals'], TOL, name + ' flush vals')
        assert np.array_equal(cpu(model.right_memory.update_ts), g.z['flush_right_ts'])
        assert len(model.msg_store.nodes_with_messages) == 0


def test_fused_route_detaches_the_score_fold_and_left_writeback():
    """The fused route attaches the score fold and the left write-back to the pack of fns.0 for its last attention
    product only.  The step-by-step route's graph-form call uses the same pack: afterwards it must write neither the
    left memory nor pq."""
    g = Golden('seq_left_right')
    full, graph, coll, dl, model = setup(g)
    assert g.n_layers == 1
    src, dst, neg, ts, eids, cg = to_dev(next(iter(dl)))
    model.eval()
    model.reset()
    with torch.no_grad():
        model.contrast_learning(src, dst, neg, ts, eids, cg)
        s = model.temporal_embedding_fn.fns[0].packed(model.time_encoder).struct
        assert s.left_wb is None and s.score_folded is None and s.pq_out is None
        left = model.left_memory
        before = [t.clone() for t in (left.vals, left.update_ts, left.active_mask, model._ws.pq)]
        # representations unlike the fused call's, so that a leaked attachment would change what it writes
        reprs = model.right_memory.vals[cg.computation_graph_nodes] + 1.0
        model.temporal_embedding_fn.compute_embedding_with_computation_graph(
            reprs, torch.cat([src, dst, neg]), ts.repeat(3), cg)
        after = (left.vals, left.update_ts, left.active_mask, model._ws.pq)
        for a, b, what in zip(after, before, ('left vals', 'left ts', 'left active', 'pq')):
            assert torch.equal(a, b), what


@pytest.mark.parametrize('name', ['seq_left_right', 'static_right_right_dim10'])
def test_autograd_route_equals_fused_route_and_trains(name):
    """Training-mode forward (torch autograd ops, dropout 0) must agree with the fused kernel route on the
    same state; backward must reach every trainable part of the path."""
    g = Golden(name)
    full, graph, coll, dl, model = setup(g, dropout=0.0)
    batches = [to_dev(b) for _, b in zip(range(6), dl)]
    snapshots = []
    model.eval()
    model.reset()
    with torch.no_grad():
        for b in batches:
            snapshots.append([cpu(t) for t in model.contrast_learning(*b)])
    final_fused = cpu(model.left_memory.vals), cpu(model.right_memory.vals), cpu(model.msg_store.node_msg_vals)
    model.train()
    model.reset()
    opt = torch.optim.SGD(model.parameters(), lr=0.0)          # lr 0: weights stay fixed, grads still flow
    for ib, b in enumerate(batches):
        opt.zero_grad()
        contrast, mutual = model.contrast_and_mutual_learning(*b)
        outs = None
        (contrast + mutual).backward()
        opt.step()
        assert_close(cpu(contrast).reshape(1), snapshots[ib][0].reshape(1), TOL, f'{name} b{ib} loss')
        assert torch.isfinite(mutual)
    got = cpu(model.left_memory.vals), cpu(model.right_memory.vals), cpu(model.msg_store.node_msg_vals)
    for a, b_, w in zip(got, final_fused, ('left', 'right', 'msg')):
        assert_close(a, b_, TOL, f'{name} final {w}')
    grads = {n: p.grad for n, p in model.named_parameters()}
    for key in ('right_mem_updater.cell.weight_ih', 'temporal_embedding_fn.fns.0.mha_fn.q_proj_weight',
                'temporal_embedding_fn.fns.0.merger.fc2.weight', 'time_encoder.basis_freq', 'score_fn.fc1.weight',
                'hit_embedding.weight'):
        assert grads[key] is not None and torch.isfinite(grads[key]).all() and grads[key].abs().max() > 0, key
    r = 'restarter_fn.out_fn.weight' if g.restarter == 'seq' else 'restarter_fn.left_emb.weight'
    assert grads[r] is not None and grads[r].abs().max() > 0


def test_eval_edge_prediction_ap_matches_oracle():
    """AP/AUC protocol of eval_utils.py:15-68 on our model vs the same protocol on the CPU oracle's scores."""
    from sklearn.metrics import average_precision_score
    from oracle import tiger_oracle as O
    g = Golden('seq_restart_mode')
    full, graph, coll, dl, model = setup(g)
    model.reset()
    ap, auc = eval_edge_prediction(model, dl, DEV, restart_mode=True, mean_over_n_samples=g.bs)
    og = O.OracleGraph(g.src, g.dst, g.ts, g.eids, n_nodes=g.N)
    om = O.OracleTIGER(g.W, og, g.N, g.dim, g.efeats, g.nfeats, n_neighbors=g.K, n_head=g.n_heads,
                       msg_src=g.msg_src, upd_src=g.upd_src, restarter=g.restarter, hist_len=g.hist_len)
    uptodate = np.zeros(g.N, dtype=bool)
    aps = []
    n_b = (len(g.src) + g.bs - 1) // g.bs
    for ib in range(n_b):
        s = slice(ib * g.bs, min((ib + 1) * g.bs, len(g.src)))
        b = O.collate(og, g.src[s], g.dst[s], g.neg[s], g.ts[s], g.eids[s], g.K)
        rn = O.lazy_restart_nodes(b.involved, uptodate)
        om.restart(rn, np.full(len(rn), b.ts.min(), dtype=np.float32))
        o = om.contrast_step(b)
        score = torch.cat([o['pos_scores'], o['neg_scores']]).sigmoid().numpy()
        label = np.concatenate([np.ones(len(b.src)), np.zeros(len(b.src))])
        aps.append(average_precision_score(label, score))
    assert abs(ap - float(np.mean(aps))) <= 0.002
    assert 0.0 <= auc <= 1.0


# ------------------------------------------------------------------------------------------
# BASELINE dimensions (tests/golden/make_golden_full.py): the class surface driven like eval_edge_prediction
# ------------------------------------------------------------------------------------------
from golden_utils import FULL_CASES, FullGolden, check_full_batch   # noqa: E402


@pytest.mark.parametrize('name', FULL_CASES)
def test_dropin_replays_reference_at_baseline_dimensions(name):
    g = FullGolden(name)
    src_, dst_, ts_, eids_ = g.stream_prefix()
    full = InteractionData(src_, dst_, ts_, eids_, np.zeros_like(src_), seed=0, eval=True, neg_dst=g.neg[:g.E])
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    coll = GraphCollator(graph, g.K, 1, restarter=g.restarter, hist_len=g.hist_len)
    model = D.init_model(None, g.efeats, graph, g.N, g.st.n_events, DEV, dim=g.shape.dim, n_layers=1,
                         n_heads=g.n_heads, n_neighbors=g.K, hit_type='bin', dropout=0.1, restarter_type=g.restarter,
                         hist_len=g.hist_len, msg_src=g.msg_src, upd_src=g.upd_src)
    res = model.load_state_dict(g.W, strict=False)
    assert not res.unexpected_keys
    model.eval()
    model.reset()
    uptodate = set()
    with torch.no_grad():
        for ib in range(g.warm + g.rec):
            lo = g.start + ib * g.bs
            src, dst, neg, ts, eids, cg = to_dev(coll([full[i] for i in range(lo, lo + g.bs)]))
            fresh = sorted(set(cg.np_computation_graph_nodes.tolist()) - uptodate)
            r_nids = torch.tensor(fresh, dtype=torch.long, device=DEV)
            r_ts = torch.full((len(r_nids),), ts.min().item(), device=DEV)
            got = {}
            if ib >= g.warm and len(r_nids):
                hl, hr, pt = model.restarter_fn(r_nids, r_ts)
                got.update(restart_hl=cpu(hl), restart_hr=cpu(hr), restart_pt=cpu(pt))
            model.restart(r_nids, r_ts)
            uptodate.update(fresh)
            pending_before = np.array(sorted(model.msg_store.nodes_with_messages), dtype=np.int64)
            loss, h_left, ps, ns, hpl, hpr = model.contrast_learning(src, dst, neg, ts, eids, cg)
            if ib < g.warm:
                continue
            rd = cg.restart_data
            sl, sr, _ = model.restarter_fn(torch.cat([src, dst])[rd.index], ts.repeat(2)[rd.index], cg)
            targets = torch.cat([hpl[rd.index], hpr[rd.index]], 0)
            preds = torch.cat([sl, sr], 0)
            valid = torch.where(~(targets == 0).all(1))[0]
            ml = model.mutual_loss_fn(preds[valid], targets[valid]) if len(valid) else torch.tensor(0.)
            w = np.zeros(2 * g.bs, dtype=np.uint8)
            w[cpu(rd.index)] = 1
            got.update(neigh_nids=cpu(cg.layers[1][0]), neigh_eids=cpu(cg.layers[1][1]), neigh_ts=cpu(cg.layers[1][2]),
                       involved=cg.np_computation_graph_nodes, restart_nids=np.array(fresh),
                       outdated=np.intersect1d(pending_before, cg.np_computation_graph_nodes), winner=w,
                       h_left=cpu(h_left), pos_scores=cpu(ps), neg_scores=cpu(ns), loss=cpu(loss), mutual_loss=cpu(ml),
                       h_prev_left=cpu(hpl), h_prev_right=cpu(hpr), surrogate_left=cpu(sl), surrogate_right=cpu(sr),
                       left_vals=cpu(model.left_memory.vals), right_vals=cpu(model.right_memory.vals),
                       msg_vals=cpu(model.msg_store.node_msg_vals), left_ts=cpu(model.left_memory.update_ts),
                       right_ts=cpu(model.right_memory.update_ts), msg_ts=cpu(model.msg_store.node_msg_ts),
                       pending_after=np.array(sorted(model.msg_store.nodes_with_messages)))
            check_full_batch(g, ib - g.warm, got, TOL, 'dropin ')


# ------------------------------------------------------------------------------------------
# a27: the snapshot API the drivers call around every validation pass (train_self_supervised.py:193-202)
# ------------------------------------------------------------------------------------------
from tiger.eval_utils import warmup   # noqa: E402


def test_save_and_load_memory_state_round_trip():
    """save_memory_state / load_memory_state (tiger.py:465-484): the snapshot restores both memories and the
    message store exactly, later steps run on the restored objects (every buffer on the device - the clone used to
    leave `active_mask` on the host), and Memory.clone drops the activity flags like the reference (Q2)."""
    g = Golden('seq_restart_mode')
    full, graph, coll, dl, model = setup(g)
    batches = [to_dev(b) for _, b in zip(range(8), dl)]
    model.eval()
    model.reset()
    with torch.no_grad():
        for b in batches[:4]:
            model.contrast_learning(*b)
        snap = model.save_memory_state()
        assert all(t.is_cuda for m in snap[:2] for t in (m.vals, m.update_ts, m.active_mask))
        assert int(snap[0].active_mask.sum()) == 0 and int(model.left_memory.active_mask.sum()) > 0     # Q2
        want = [cpu(t).copy() for t in (model.left_memory.vals, model.right_memory.vals, model.left_memory.update_ts,
                                        model.right_memory.update_ts, model.msg_store.node_msg_vals,
                                        model.msg_store.node_msg_ts)]
        pending = sorted(model.msg_store.nodes_with_messages)
        first = [cpu(t) for t in model.contrast_learning(*batches[4])]
        for b in batches[5:]:
            model.contrast_learning(*b)                           # memory modified by "validation"
        model.load_memory_state(snap)
        got = [cpu(t) for t in (model.left_memory.vals, model.right_memory.vals, model.left_memory.update_ts,
                                model.right_memory.update_ts, model.msg_store.node_msg_vals,
                                model.msg_store.node_msg_ts)]
        for a, b_ in zip(got, want):
            assert np.array_equal(a, b_)
        assert sorted(model.msg_store.nodes_with_messages) == pending
        assert model.msg_memory is (model.left_memory if g.msg_src == 'left' else model.right_memory)
        again = [cpu(t) for t in model.contrast_learning(*batches[4])]    # kernels store through the restored buffers
        for a, b_ in zip(again, first):
            assert np.array_equal(a, b_)
        # the snapshot was handed over, not copied: a second restore needs a second snapshot (reference semantics)
        model.flush_msg()
        assert len(model.msg_store.nodes_with_messages) == 0


def test_warmup_equals_eval_loop_without_scoring():
    """warmup (eval_utils.py:102-129) = the lazy-restart loop of eval_edge_prediction without the scores."""
    g = Golden('seq_restart_mode')
    full, graph, coll, dl, model = setup(g)
    model.reset()
    seen = warmup(model, dl, DEV)
    a = [cpu(t).copy() for t in (model.left_memory.vals, model.right_memory.vals, model.msg_store.node_msg_vals)]
    model.reset()
    seen2 = set()
    eval_edge_prediction(model, dl, DEV, restart_mode=True, uptodate_nodes=seen2, mean_over_n_samples=g.bs)
    b = [cpu(t) for t in (model.left_memory.vals, model.right_memory.vals, model.msg_store.node_msg_vals)]
    assert seen == seen2 and len(seen) > 0
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_memory_set_and_flush_with_more_than_2048_ids():
    """Memory.set's duplicate check takes the large-n path of tiger_select_latest in flags-only mode, whose count
    used to stay unwritten; flush_msg hits it after an epoch (ADVICE r1)."""
    from tiger.model.memory import Memory
    n, d = 6000, 12
    mem = Memory(n, d).to(DEV)
    ids = torch.randperm(n, device=DEV)[:5000]
    vals = torch.randn(5000, d, device=DEV)
    ts = torch.rand(5000, device=DEV) + 1
    mem.set(ids, vals, ts)
    assert torch.equal(mem.vals[ids], vals) and torch.equal(mem.update_ts[ids], ts)
    dup = ids.clone()
    dup[4000] = dup[17]
    with pytest.raises(ValueError, match='Duplicate'):
        mem.set(dup, vals, ts + 1)
    with pytest.raises(ValueError, match='past memory'):
        mem.set(ids, vals, ts - 1)
