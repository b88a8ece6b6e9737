"""Two-layer temporal attention (n_layers=2) on the fused path: TigerEngine(n_layers=2) and the drop-in's fused
no-grad route against the golden of the unmodified reference (var_two_layers), and against the drop-in's torch-op
route on seeded streams at BASELINE dimensions."""
import numpy as np
import pytest
import torch
from torch.utils.data import DataLoader

from golden_utils import Golden, assert_close
from www2023tiger_b200.engine import StreamRunner, TigerEngine
from www2023tiger_b200.init import perturb_biases, random_weights
from www2023tiger_b200.synthetic import SHAPES, NegativeSampler, StreamShape, make_stream

TOL = 1e-5
cpu = lambda t: t.detach().cpu().numpy()


def engine2(W, csr, *, N, dim, efeats, nfeats, K, H, B, msg_src, upd_src, restarter=None, lazy_restart=False,
            hist_len=40):
    dev = lambda x: None if x is None else torch.as_tensor(x).float().cuda().contiguous()
    return TigerEngine({k: torch.as_tensor(v) for k, v in W.items()}, csr, n_nodes=N, dim=dim, efeats=dev(efeats),
                       nfeats=dev(nfeats), n_neighbors=K, n_head=H, batch_size=B, msg_src=msg_src, upd_src=upd_src,
                       restarter=restarter, hist_len=hist_len, lazy_restart=lazy_restart, want_restarter_targets=True,
                       n_layers=2)


def test_engine_rejects_three_layers():
    with pytest.raises(NotImplementedError):
        TigerEngine({}, None, n_nodes=10, dim=8, efeats=None, n_layers=3)


# ------------------------------------------------------------------------------------------
# golden of the unmodified reference
# ------------------------------------------------------------------------------------------
def engine_state(e):
    return [t.clone() for t in (e.out_buf, e.emb, e.emb1, e.left_vals, e.right_vals, e.msg_vals, e.left_ts, e.right_ts,
                                e.msg_ts, e.has_msg)]


@pytest.mark.gpu
def test_engine_replays_two_layer_golden_eager_and_captured():
    import gpu_utils as gu
    g = Golden('var_two_layers')
    assert g.n_layers == 2 and not g.lazy_restart
    csr = gu.device_csr(g.src, g.dst, g.ts, g.eids, g.N)
    e = engine2(g.W, csr, N=g.N, dim=g.dim, efeats=g.efeats, nfeats=g.nfeats, K=g.K, H=g.n_heads, B=g.bs,
                msg_src=g.msg_src, upd_src=g.upd_src)
    B = g.bs
    assert e.cap == g.N                       # (3B + 3BK)(K + 1) = 3240 > N = 53
    eager = []
    for ib in range(g.n_batches):
        what = f'var_two_layers batch {ib} '
        e.set_batch(*g.batch(ib))
        e.step()
        e.check_errors()
        U, Oc = (int(x) for x in e.counts[:2])
        for mine, theirs in (('neigh', 'l2_neigh'), ('neigh2', 'neigh')):
            for col in ('nids', 'eids', 'ts'):
                assert np.array_equal(cpu(getattr(e, f'{mine}_{col}')), g.b(ib, f'{theirs}_{col}')), what + mine + col
        assert np.array_equal(cpu(e.involved[:U]), g.b(ib, 'involved')), what + 'involved'
        assert np.array_equal(cpu(e.outdated[:Oc]), np.intersect1d(g.b(ib, 'pending_before'), g.b(ib, 'involved'))), \
            what + 'outdated'
        w = np.zeros(2 * B, dtype=np.uint8)
        w[g.b(ib, 'r_index')] = 1
        assert np.array_equal(cpu(e.winner), w), what + 'winners'
        assert_close(cpu(e.emb[:2 * B]), g.b(ib, 'h_left'), TOL, what + 'h_left')
        assert_close(cpu(e.scores[:B]), g.b(ib, 'pos_scores'), TOL, what + 'pos')
        assert_close(cpu(e.scores[B:]), g.b(ib, 'neg_scores'), TOL, what + 'neg')
        assert_close(cpu(e.loss), g.b(ib, 'loss').reshape(1), TOL, what + 'loss')
        assert_close(cpu(e.hprev_left), g.b(ib, 'h_prev_left'), TOL, what + 'hpl')
        assert_close(cpu(e.hprev_right), g.b(ib, 'h_prev_right'), TOL, what + 'hpr')
        assert_close(cpu(e.left_vals), g.b(ib, 'left_vals'), TOL, what + 'left_vals')
        assert_close(cpu(e.right_vals), g.b(ib, 'right_vals'), TOL, what + 'right_vals')
        assert_close(cpu(e.msg_vals), g.b(ib, 'msg_vals'), TOL, what + 'msg_vals')
        for t in ('left_ts', 'right_ts', 'msg_ts'):
            assert np.array_equal(cpu(getattr(e, t)), g.b(ib, t)), what + t
        assert np.array_equal(np.nonzero(cpu(e.has_msg))[0], g.b(ib, 'pending_after')), what + 'pending'
        eager.append(engine_state(e))
    # the same batches through the captured graphs of the pipeline: bit for bit the eager results
    runner = StreamRunner(e)
    e.set_batch(*g.batch(0))
    runner.capture(warmup=1)
    e.reset()
    # reset() leaves the message table's values to the pending flags; the eager run started from a fresh engine
    e.msg_vals.zero_()
    e.msg_ts.zero_()
    for ib in range(g.n_batches):
        slot = runner.submit_host(*g.batch(ib))
        runner.wait(slot)
        torch.cuda.synchronize()
        e.bind_finder(runner.finder_bufs[slot])
        e.bind_io(runner.d_in[slot], runner.d_out[slot])
        for k, (a, b) in enumerate(zip(eager[ib], engine_state(e))):
            assert torch.equal(a, b), f'graph replay batch {ib} tensor {k}'
    e.check_errors()


# ------------------------------------------------------------------------------------------
# drop-in: the fused no-grad route of TIGER(n_layers=2)
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_dropin_two_layers_takes_fused_route_and_replays_golden(monkeypatch):
    import dropin_utils as D
    from tiger.data.data_loader import GraphCollator, InteractionData
    from tiger.data.graph import Graph
    from tiger.model.tiger import TIGE
    dev = torch.device('cuda')
    g = Golden('var_two_layers')
    full = InteractionData(g.src, g.dst, g.ts, g.eids, np.zeros_like(g.src), seed=0, eval=True, neg_dst=g.neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    coll = GraphCollator(graph, g.K, 2, restarter=g.restarter, hist_len=g.hist_len)
    model = D.load_golden_weights(D.model_from_golden(g, graph, dev), g)
    fused = [0]
    orig = TIGE._contrast_learning_fused

    def spy(self, *a, **kw):
        fused[0] += 1
        return orig(self, *a, **kw)
    monkeypatch.setattr(TIGE, '_contrast_learning_fused', spy)
    model.eval()
    model.reset()
    with torch.no_grad():
        for ib, batch in enumerate(DataLoader(full, batch_size=g.bs, collate_fn=coll)):
            if ib >= g.n_batches:
                break
            what = f'dropin b{ib} '
            src, dst, neg, ts, eids, _, cg = batch
            src, dst, neg, eids = (x.long().cuda() for x in (src, dst, neg, eids))
            ts, cg = ts.float().cuda(), cg.to(dev)
            loss, h_left, ps, ns, hpl, hpr = model.contrast_learning(src, dst, neg, ts, eids, cg)
            assert fused[0] == ib + 1, what + 'fused route not taken'
            assert_close(cpu(loss).reshape(1), g.b(ib, 'loss').reshape(1), TOL, what + 'loss')
            assert_close(cpu(h_left), g.b(ib, 'h_left'), TOL, what + 'h_left')
            assert_close(cpu(ps), g.b(ib, 'pos_scores'), TOL, what + 'pos')
            assert_close(cpu(ns), g.b(ib, 'neg_scores'), TOL, what + 'neg')
            assert_close(cpu(hpl), g.b(ib, 'h_prev_left'), TOL, what + 'hpl')
            assert_close(cpu(hpr), g.b(ib, 'h_prev_right'), TOL, what + 'hpr')
            assert_close(cpu(model.left_memory.vals), g.b(ib, 'left_vals'), TOL, what + 'left_vals')
            assert_close(cpu(model.right_memory.vals), g.b(ib, 'right_vals'), TOL, what + 'right_vals')
            assert_close(cpu(model.msg_store.node_msg_vals), g.b(ib, 'msg_vals'), TOL, what + 'msg_vals')
            assert np.array_equal(cpu(model.left_memory.update_ts), g.b(ib, 'left_ts')), what
            assert np.array_equal(cpu(model.right_memory.update_ts), g.b(ib, 'right_ts')), what
            assert sorted(model.msg_store.nodes_with_messages) == g.b(ib, 'pending_after').tolist(), what


# ------------------------------------------------------------------------------------------
# engine vs the drop-in's torch-op route (grad enabled, eval mode) on seeded streams
# ------------------------------------------------------------------------------------------
def compare_with_torch_route(shape, *, start, n_batches, restarter, lazy, msg_src, upd_src, B=200, K=10, H=2,
                             seed=0, check=None):
    """Runs the same batches through TigerEngine(n_layers=2) (eager launches) and the drop-in TIGER(n_layers=2) on
    its step-by-step torch-op route; integer outputs must agree bit for bit, floats within TOL.  Returns the worst
    relative error seen per quantity."""
    import dropin_utils as D
    import gpu_utils as gu
    from tiger.data.data_loader import GraphCollator, InteractionData
    from tiger.data.graph import Graph
    dev = torch.device('cuda')
    st = make_stream(shape, seed=seed)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    N, d = st.n_nodes, st.dim
    de = st.efeats.shape[1] if st.efeats is not None else d
    W = perturb_biases(random_weights(d, de, n_nodes=N, restarter=restarter, nonzero_static=True, seed=seed + 1,
                                      n_layers=2))
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = engine2(W, csr, N=N, dim=d, efeats=st.efeats, nfeats=None, K=K, H=H, B=B, msg_src=msg_src, upd_src=upd_src,
                restarter=restarter, lazy_restart=lazy)
    full = InteractionData(st.src, st.dst, st.ts, st.eids, np.zeros_like(st.src), seed=0, eval=True, neg_dst=neg)
    graph = Graph.from_csr(csr)
    coll = GraphCollator(graph, K, 2, restarter=restarter, hist_len=40)
    model = D.init_model(None, st.efeats, graph, N, st.n_events, dev, dim=d, n_layers=2, n_heads=H, n_neighbors=K,
                         hit_type='bin', dropout=0.1, restarter_type=restarter, hist_len=40, msg_src=msg_src,
                         upd_src=upd_src)
    res = model.load_state_dict(W, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    model.eval()
    model.reset()
    e.reset()
    uptodate = set()
    worst = {}

    def close(a, b, what, key):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        err = np.abs(a - b).max() / max(np.abs(b).max(), 1e-30) if b.size else 0.0
        worst[key] = max(worst.get(key, 0.0), float(err))
        assert_close(a, b, TOL, what + key)

    for ib in range(n_batches):
        lo = start + ib * B
        what = f'{shape.name} batch {ib} '
        src, dst, ng, ts, eids, _, cg = coll([full[i] for i in range(lo, lo + B)])
        src, dst, ng, eids = (x.long().cuda() for x in (src, dst, ng, eids))
        ts, cg = ts.float().cuda(), cg.to(dev)
        if lazy:
            fresh = sorted(set(cg.np_computation_graph_nodes.tolist()) - uptodate)
            r_nids = torch.tensor(fresh, dtype=torch.long, device=dev)
            model.restart(r_nids, torch.full((len(r_nids),), ts.min().item(), device=dev))
            uptodate.update(fresh)
        pending_before = np.array(sorted(model.msg_store.nodes_with_messages), dtype=np.int64)
        with torch.enable_grad():
            loss, h_left, ps, ns, hpl, hpr = model.contrast_learning(src, dst, ng, ts, eids, cg)
        e.set_batch(st.src[lo:lo + B], st.dst[lo:lo + B], neg[lo:lo + B], st.ts[lo:lo + B], st.eids[lo:lo + B])
        e.step()
        e.check_errors()
        if check is not None:
            check(ib, e, cg)
        U, Oc, R = (int(x) for x in e.counts[:3])
        for j, col in enumerate(('nids', 'eids', 'ts')):
            assert np.array_equal(cpu(getattr(e, f'neigh_{col}')), cpu(cg.layers[2][j])), what + 'hop 1 ' + col
            assert np.array_equal(cpu(getattr(e, f'neigh2_{col}')), cpu(cg.layers[1][j])), what + 'hop 2 ' + col
        assert np.array_equal(cpu(e.involved[:U]), cg.np_computation_graph_nodes), what + 'involved'
        assert np.array_equal(cpu(e.outdated[:Oc]), np.intersect1d(pending_before, cg.np_computation_graph_nodes)), \
            what + 'outdated'
        if lazy:
            assert np.array_equal(cpu(e.restart_nodes[:R]), np.array(fresh, dtype=np.int64)), what + 'restart list'
        w = np.zeros(2 * B, dtype=np.uint8)
        w[cpu(cg.restart_data.index)] = 1
        assert np.array_equal(cpu(e.winner), w), what + 'winners'
        close(cpu(e.emb[:2 * B]), cpu(h_left), what, 'h_left')
        close(cpu(e.scores[:B]), cpu(ps), what, 'pos_scores')
        close(cpu(e.scores[B:]), cpu(ns), what, 'neg_scores')
        close(cpu(e.loss), cpu(loss).reshape(1), what, 'loss')
        close(cpu(e.hprev_left), cpu(hpl), what, 'h_prev_left')
        close(cpu(e.hprev_right), cpu(hpr), what, 'h_prev_right')
        close(cpu(e.left_vals), cpu(model.left_memory.vals), what, 'left_vals')
        close(cpu(e.right_vals), cpu(model.right_memory.vals), what, 'right_vals')
        close(cpu(e.msg_vals), cpu(model.msg_store.node_msg_vals), what, 'msg_vals')
        assert np.array_equal(cpu(e.left_ts), cpu(model.left_memory.update_ts)), what + 'left_ts'
        assert np.array_equal(cpu(e.right_ts), cpu(model.right_memory.update_ts)), what + 'right_ts'
        assert np.array_equal(cpu(e.msg_ts), cpu(model.msg_store.node_msg_ts)), what + 'msg_ts'
        assert np.array_equal(np.nonzero(cpu(e.has_msg))[0], np.array(sorted(model.msg_store.nodes_with_messages))), \
            what + 'pending'
    print(f'{shape.name} {restarter} lazy={lazy} msg_src={msg_src}: max rel err ' +
          ', '.join(f'{k} {v:.2e}' for k, v in worst.items()))
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize('name,restarter,lazy,msg_src', [
    ('wikipedia', 'seq', True, 'left'), ('wikipedia', 'seq', False, 'left'),
    ('reddit', 'static', True, 'left'), ('reddit', 'static', False, 'left'),
    ('wikipedia', 'seq', True, 'right'),
])
def test_engine_matches_torch_route_at_baseline_dimensions(name, restarter, lazy, msg_src):
    """d = d_e = 172, K = 10, B = 200, 30 consecutive batches from the middle of the stream."""
    shape = SHAPES[name]
    assert shape.efeat_dim == 172
    compare_with_torch_route(shape, start=(shape.n_events // 2) // 200 * 200, n_batches=30, restarter=restarter,
                             lazy=lazy, msg_src=msg_src, upd_src='right')


@pytest.mark.gpu
def test_first_batches_after_reset_on_a_graph_below_the_capacity_bound():
    """A stream from its first event: the first batch after reset() finds almost no history, so most hop-2 slots are
    padding; and N = 160 lies below (3B + 3BK)(K + 1), so the involved lists are sized by N."""
    shape = StreamShape('small', 120, 40, 3000, 16, None, horizon=3000.)
    B, K = 50, 10
    padding = []

    def check(ib, e, cg):
        assert e.cap == e.N < (3 * B + 3 * B * K) * (K + 1)
        padding.append(float((e.neigh2_nids == 0).float().mean()))
    compare_with_torch_route(shape, start=0, n_batches=8, restarter='static', lazy=True, msg_src='left',
                             upd_src='right', B=B, K=K, check=check)
    assert padding[0] > 0.5, padding
