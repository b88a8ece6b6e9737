"""The scorer's hit types (--hit_type vec | count) on the fused inference path: the score fold and the folded scorer
against a float64 restatement, TigerEngine (eager and captured) and the drop-in's fused no-grad route against the
goldens of the unmodified reference (var_hit_vec, var_hit_count), the engine against the drop-in's torch-op route at
BASELINE dimensions, the refold after a parameter update, and training, which stays on the torch-op route."""
import numpy as np
import pytest
import torch
from torch.utils.data import DataLoader

from golden_utils import Golden, assert_close
from oracle import tiger_oracle as O
from www2023tiger_b200 import ops
from www2023tiger_b200.engine import StreamRunner, TigerEngine
from www2023tiger_b200.init import perturb_biases, random_weights
from www2023tiger_b200.synthetic import SHAPES, NegativeSampler, make_stream

pytestmark = pytest.mark.gpu
TOL = 1e-5
HIT_GOLDENS = ('var_hit_vec', 'var_hit_count')
cpu = lambda t: t.detach().cpu().numpy()
dev = lambda x: torch.as_tensor(x).cuda().contiguous()


# ------------------------------------------------------------------------------------------
# score fold + folded scorer against float64
# ------------------------------------------------------------------------------------------
def hit_tables(B, K, N, rng):
    """src / dst / neg ids and a [3B, K] neighbor table of [src ; dst ; neg] rows in which the hit counts of the rows
    run through every value 0..K (all-hit and no-hit rows included), with duplicate ids and padding (id 0) in the
    other slots."""
    src = rng.randint(1, N // 2, B)
    dst, neg = rng.randint(N // 2, N, B), rng.randint(N // 2, N, B)
    hit_id = np.concatenate([dst, src, src])               # N(src) holds dst, N(dst) and N(neg) hold src
    counts = rng.permutation(np.arange(3 * B) % (K + 1))
    neigh = np.empty((3 * B, K), dtype=np.int64)
    for r in range(3 * B):
        pool = np.array([u for u in range(0, 8) if u != hit_id[r]] * 2)   # few ids: duplicates, padding slots
        row = rng.choice(pool, K)
        slots = rng.permutation(K)
        row[slots[:counts[r]]] = hit_id[r]
        if r < B and neg[r] != dst[r]:                      # N(src) also holds neg: the negative pair's b flags
            free = slots[counts[r]:]
            row[free[:rng.randint(0, len(free) + 1)]] = neg[r]
        neigh[r] = row
    return src, dst, neg, neigh


def scorer64(z, src, dst, neg, neigh, W, hit_type):
    """tiger.py:259-288 in float64 from the embeddings z [3B, d]: hit flags, hit term, score_fn, BCE mean."""
    B = len(src)
    z = z.astype(np.float64)
    w = {n: W['score_fn.' + n].double().numpy() for n in ('fc1.weight', 'fc1.bias', 'fc2.weight', 'fc2.bias')}
    x, y, ny = z[:B], z[B:2 * B], z[2 * B:]
    flags = lambda ids, rows: (neigh[rows] == ids[:, None]).astype(np.float64)
    pairs = [(x, y, flags(src, slice(B, 2 * B)), flags(dst, slice(0, B))),
             (x, ny, flags(src, slice(2 * B, 3 * B)), flags(neg, slice(0, B)))]
    scores = []
    for xs, ys, a, b in pairs:
        if hit_type == 'vec':
            inp = np.concatenate([xs, a, ys, b], 1)
        else:
            emb = W['hit_embedding.weight'].double().numpy()
            inp = np.concatenate([xs + emb[a.sum(1).astype(int)], ys + emb[b.sum(1).astype(int)]], 1)
        h = np.maximum(inp @ w['fc1.weight'].T + w['fc1.bias'], 0)
        scores.append((h @ w['fc2.weight'].T + w['fc2.bias'])[:, 0])
    s = np.concatenate(scores)
    label = np.r_[np.ones(B), np.zeros(B)]
    loss = np.mean(np.maximum(s, 0) - s * label + np.log1p(np.exp(-np.abs(s))))
    return s, loss


@pytest.mark.parametrize('hit_type', ['vec', 'count'])
@pytest.mark.parametrize('B', [1, 200, 1000])
@pytest.mark.parametrize('K', [5, 10, 33, 64])
@pytest.mark.parametrize('d', [172, 100, 8])
def test_fold_and_scorer_match_float64(d, K, B, hit_type):
    """The batch nodes' attention (gather form) with the hit type's score fold and the left write-back attached writes
    pq; tiger_link_score_folded_hit scores the pairs from it (K > 32: more than one ballot per side)."""
    rng = np.random.RandomState(d * 1000 + K * 10 + B)
    W = perturb_biases(random_weights(d, d, seed=K + B, hit_type=hit_type, n_neighbors=K))
    g = torch.Generator().manual_seed(B)
    N, E, H = 40, 300, 2
    rows, efeats = torch.randn(N, d, generator=g), torch.randn(E, d, generator=g)
    src, dst, neg, neigh_np = hit_tables(B, K, N, rng)
    neigh = torch.from_numpy(neigh_np)
    centers = torch.from_numpy(np.concatenate([src, dst, neg]))
    neigh_e = torch.randint(0, E, (3 * B, K), generator=g)
    ts = torch.rand(B, generator=g) * 100 + 100
    neigh_ts = ts.repeat(3)[:, None] - torch.rand(3 * B, K, generator=g) * 100
    p = 'temporal_embedding_fn.fns.0.'
    tw, tb = W['time_encoder.basis_freq'], W['time_encoder.phase']
    z = O.temporal_attention(W, p, H, rows[centers], O.time_encode(torch.zeros(3 * B), tw, tb), rows[neigh],
                             efeats[neigh_e], O.time_encode(ts.repeat(3)[:, None] - neigh_ts, tw, tb), neigh == 0)
    pack = ops.AttnPack(d, d, 'cuda', H)
    m = p + 'mha_fn.'
    pack.refresh(*(dev(W[n]) for n in (m + 'q_proj_weight', m + 'k_proj_weight', m + 'v_proj_weight',
                                       m + 'in_proj_bias', m + 'out_proj.weight', m + 'out_proj.bias',
                                       p + 'merger.fc1.weight', p + 'merger.fc1.bias', p + 'merger.fc2.weight',
                                       p + 'merger.fc2.bias', 'time_encoder.basis_freq', 'time_encoder.phase')))
    fold, pq = ops.ScoreFold(d, 'cuda', hit_type, K), torch.zeros(3 * B, 2 * d, device='cuda')
    fold.refresh(*(dev(W['score_fn.' + n]) for n in ('fc1.weight', 'fc1.bias', 'fc2.weight', 'fc2.bias')),
                 dev(W[p + 'merger.fc2.weight']), dev(W[p + 'merger.fc2.bias']),
                 dev(W['hit_embedding.weight']) if hit_type == 'count' else None)
    d_centers, d_ts = dev(centers), dev(ts)
    pos = d_centers[:2 * B]
    winner = ops.select_latest(pos, d_ts, want_unique=False, want_count=False)[0]
    left_vals, left_ts = torch.zeros(N, d, device='cuda'), torch.zeros(N, device='cuda')
    left_active = torch.zeros(N, dtype=torch.uint8, device='cuda')
    pack.attach_score_fold(fold, pq)
    pack.attach_left_writeback(pos, winner, d_ts, left_vals, left_ts, left_active)
    out = ops.temporal_attention(pack, H, d_centers, d_ts, dev(neigh), dev(neigh_e), dev(neigh_ts), rows_a=None,
                                 rows_b=dev(rows), sel=torch.arange(N, dtype=torch.int32, device='cuda'), nfeats=None,
                                 efeats=dev(efeats))
    assert_close(cpu(out), z.numpy(), TOL, 'embeddings')
    w = winner.bool()
    assert torch.equal(left_vals[pos[w]], out[:2 * B][w]), 'fused left write-back'
    want_s, want_loss = scorer64(cpu(out), src, dst, neg, neigh_np, W, hit_type)
    for _ in range(2):                    # twice: the done-counter must reset itself
        scores, loss = ops.link_score_folded(fold, pq, dev(src), dev(dst), dev(neg), dev(neigh))
        assert_close(cpu(scores), want_s, TOL, 'scores')
        assert_close(cpu(loss), np.reshape(want_loss, (1,)), TOL, 'loss')


def test_scorer_refuses_a_neighbor_table_of_another_k():
    fold = ops.ScoreFold(8, 'cuda', 'count', 5)
    z = torch.zeros(3, 16, device='cuda')
    ids = torch.ones(1, dtype=torch.int64, device='cuda')
    with pytest.raises(ValueError):
        ops.link_score_folded(fold, z, ids, ids, ids, torch.ones(3, 6, dtype=torch.int64, device='cuda'))


# ------------------------------------------------------------------------------------------
# the reference's goldens through the engine and the drop-in
# ------------------------------------------------------------------------------------------
def engine_for(W, csr, *, N, dim, efeats, nfeats, K, H, B, msg_src, upd_src, restarter, lazy, hit_type,
               hist_len=40, n_layers=1, tsfm='id', upd='gru'):
    f = lambda x: None if x is None else torch.as_tensor(x).float().cuda().contiguous()
    return TigerEngine({k: torch.as_tensor(v) for k, v in W.items()}, csr, n_nodes=N, dim=dim, efeats=f(efeats),
                       nfeats=f(nfeats), n_neighbors=K, n_head=H, batch_size=B, msg_src=msg_src, upd_src=upd_src,
                       restarter=restarter, hist_len=hist_len, lazy_restart=lazy, want_restarter_targets=True,
                       n_layers=n_layers, msg_tsfm_type=tsfm, mem_update_type=upd, hit_type=hit_type)


def engine_state(e):
    return [t.clone() for t in (e.out_buf, e.emb, e.left_vals, e.right_vals, e.msg_vals, e.left_ts, e.right_ts,
                                e.msg_ts, e.has_msg, e.h_new)]


@pytest.mark.parametrize('name', HIT_GOLDENS)
def test_engine_replays_hit_golden_eager_and_captured(name):
    import gpu_utils as gu
    g = Golden(name)
    assert g.hit_type in ('vec', 'count') and g.n_layers == 1
    csr = gu.device_csr(g.src, g.dst, g.ts, g.eids, g.N)
    kw = dict(N=g.N, dim=g.dim, efeats=g.efeats, nfeats=g.nfeats, K=g.K, H=g.n_heads, B=g.bs, msg_src=g.msg_src,
              upd_src=g.upd_src, restarter=g.restarter if g.lazy_restart else None, lazy=g.lazy_restart,
              hist_len=g.hist_len)
    e = engine_for(g.W, csr, hit_type=g.hit_type, **kw)
    de = g.efeats.shape[1] if g.efeats is not None else g.dim
    W_bin = random_weights(g.dim, de, n_nodes=g.N, restarter=g.restarter, hist_len=g.hist_len, nonzero_static=True)
    assert e.launches_per_step() == engine_for(W_bin, csr, hit_type='bin', **kw).launches_per_step()
    B = g.bs
    eager = []
    for ib in range(g.n_batches):
        what = f'{name} batch {ib} '
        e.set_batch(*g.batch(ib))
        e.step()
        e.check_errors()
        U, Oc, R = (int(x) for x in e.counts[:3])
        for col in ('nids', 'eids', 'ts'):
            assert np.array_equal(cpu(getattr(e, f'neigh_{col}')), g.b(ib, f'neigh_{col}')), what + col
        assert np.array_equal(cpu(e.involved[:U]), g.b(ib, 'involved')), what + 'involved'
        if g.lazy_restart:
            assert np.array_equal(cpu(e.restart_nodes[:R]), g.b(ib, 'restart_nids')), what + 'restart list'
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
    # the same batches through the captured graphs of the pipeline (the scorer is a graph of its own): bit for bit
    runner = StreamRunner(e)
    e.set_batch(*g.batch(0))
    runner.capture(warmup=1)
    e.reset()
    e.msg_vals.zero_()
    e.msg_ts.zero_()
    e.h_new.zero_()
    for ib in range(g.n_batches):
        slot = runner.submit_host(*g.batch(ib))
        runner.wait(slot)
        torch.cuda.synchronize()
        e.bind_finder(runner.finder_bufs[slot])
        e.bind_io(runner.d_in[slot], runner.d_out[slot])
        for k, (a, b) in enumerate(zip(eager[ib], engine_state(e))):
            assert torch.equal(a, b), f'graph replay batch {ib} tensor {k}'
    e.check_errors()


def golden_batches(g):
    from tiger.data.data_loader import GraphCollator, InteractionData
    from tiger.data.graph import Graph
    full = InteractionData(g.src, g.dst, g.ts, g.eids, np.zeros_like(g.src), seed=0, eval=True, neg_dst=g.neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    coll = GraphCollator(graph, g.K, 1, restarter=g.restarter, hist_len=g.hist_len)
    return graph, DataLoader(full, batch_size=g.bs, collate_fn=coll)


@pytest.mark.parametrize('name', HIT_GOLDENS)
def test_dropin_hit_type_takes_fused_route_and_replays_golden(name, monkeypatch):
    import dropin_utils as D
    from tiger.model.tiger import TIGE
    device = torch.device('cuda')
    g = Golden(name)
    graph, loader = golden_batches(g)
    model = D.load_golden_weights(D.model_from_golden(g, graph, device), g)
    fused = [0]
    orig = TIGE._contrast_learning_fused

    def spy(self, *a, **kw):
        fused[0] += 1
        return orig(self, *a, **kw)
    monkeypatch.setattr(TIGE, '_contrast_learning_fused', spy)
    model.eval()
    model.reset()
    uptodate = set()
    with torch.no_grad():
        for ib, batch in enumerate(loader):
            if ib >= g.n_batches:
                break
            what = f'dropin {name} b{ib} '
            src, dst, neg, ts, eids, _, cg = batch
            src, dst, neg, eids = (x.long().cuda() for x in (src, dst, neg, eids))
            ts, cg = ts.float().cuda(), cg.to(device)
            if g.lazy_restart:
                fresh = set(cg.np_computation_graph_nodes.tolist()) - uptodate
                r_nids = torch.tensor(sorted(fresh), dtype=torch.long, device=device)
                if len(r_nids):
                    model.restart(r_nids, torch.full((len(r_nids),), ts.min().item(), device=device))
                uptodate.update(fresh)
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


@pytest.mark.parametrize('name', HIT_GOLDENS)
def test_dropin_refolds_after_an_optimizer_step(name):
    """An optimizer step on the hit parameters (score_fn.fc1 for 'vec', hit_embedding for 'count') re-folds the
    scorer; the next fused batches match the torch-op route of the stepped model."""
    import dropin_utils as D
    device = torch.device('cuda')
    g = Golden(name)
    graph, loader = golden_batches(g)
    model = D.load_golden_weights(D.model_from_golden(g, graph, device), g)
    model.eval()
    batches = [b for _, b in zip(range(6), loader)]

    def run(fused):
        model.reset()
        outs = []
        for src, dst, neg, ts, eids, _, cg in batches:
            src, dst, neg, eids = (x.long().cuda() for x in (src, dst, neg, eids))
            ts, cg = ts.float().cuda(), cg.to(device)
            with (torch.no_grad() if fused else torch.enable_grad()):
                outs.append([cpu(t) for t in model.contrast_learning(src, dst, neg, ts, eids, cg)[:4]])
        return outs
    before = run(True)
    param = model.score_fn.fc1.weight if g.hit_type == 'vec' else model.hit_embedding.weight
    opt = torch.optim.SGD([param], lr=0.5)
    param.grad = torch.randn(param.shape, generator=torch.Generator().manual_seed(0)).to(device)
    opt.step()
    after = run(True)
    assert any(not np.array_equal(a[2], b[2]) for a, b in zip(before, after)), 'the step changed no score'
    for a, b in zip(after, run(False)):
        for x, y in zip(a, b):
            assert_close(x.reshape(-1), y.reshape(-1), TOL, 'after the optimizer step')


@pytest.mark.parametrize('name', HIT_GOLDENS)
def test_training_stays_on_the_torch_op_route(name, monkeypatch):
    import dropin_utils as D
    from tiger.model.tiger import TIGE
    device = torch.device('cuda')
    g = Golden(name)
    graph, loader = golden_batches(g)
    model = D.load_golden_weights(D.model_from_golden(g, graph, device), g)
    monkeypatch.setattr(TIGE, '_contrast_learning_fused', lambda *a, **kw: pytest.fail('fused route under autograd'))
    model.train()
    model.reset()
    src, dst, neg, ts, eids, _, cg = next(iter(loader))
    src, dst, neg, eids = (x.long().cuda() for x in (src, dst, neg, eids))
    ts, cg = ts.float().cuda(), cg.to(device)
    with torch.enable_grad():
        assert not model._native_training()
        closs, mloss = model.contrast_and_mutual_learning(src, dst, neg, ts, eids, cg)
        (closs + mloss).backward()
    assert model.score_fn.fc1.weight.grad is not None and bool(model.score_fn.fc1.weight.grad.abs().sum() > 0)
    if g.hit_type == 'count':
        assert model.hit_embedding.weight.grad is not None


# ------------------------------------------------------------------------------------------
# engine vs the drop-in's torch-op route (grad enabled, eval mode) at BASELINE dimensions
# ------------------------------------------------------------------------------------------
def compare_with_torch_route(shape, *, hit_type, restarter, n_batches=30, K=10, n_layers=1, tsfm='id', upd='gru',
                             B=200, H=2, seed=0):
    """The same batches, from mid-stream, lazy restart, through TigerEngine (eager launches) and the drop-in TIGER on
    its step-by-step torch-op route; integer outputs agree bit for bit, floats within TOL."""
    import dropin_utils as D
    import gpu_utils as gu
    from tiger.data.data_loader import GraphCollator, InteractionData
    from tiger.data.graph import Graph
    device = torch.device('cuda')
    st = make_stream(shape, seed=seed)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    N = st.n_nodes
    d = st.nfeats.shape[1] if st.nfeats is not None else st.dim
    de = st.efeats.shape[1] if st.efeats is not None else d
    W = perturb_biases(random_weights(d, de, n_nodes=N, restarter=restarter, nonzero_static=True, seed=seed + 1,
                                      n_layers=n_layers, msg_tsfm_type=tsfm, mem_update_type=upd, hit_type=hit_type,
                                      n_neighbors=K))
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = engine_for(W, csr, N=N, dim=st.dim, efeats=st.efeats, nfeats=st.nfeats, K=K, H=H, B=B,
                   msg_src=shape.msg_src, upd_src=shape.upd_src, restarter=restarter, lazy=True, hit_type=hit_type,
                   n_layers=n_layers, tsfm=tsfm, upd=upd)
    full = InteractionData(st.src, st.dst, st.ts, st.eids, np.zeros_like(st.src), seed=0, eval=True, neg_dst=neg)
    graph = Graph.from_csr(csr)
    coll = GraphCollator(graph, K, n_layers, restarter=restarter, hist_len=40)
    model = D.init_model(st.nfeats, st.efeats, graph, N, st.n_events, device, dim=st.dim, n_layers=n_layers,
                         n_heads=H, n_neighbors=K, hit_type=hit_type, dropout=0.1, restarter_type=restarter,
                         hist_len=40, msg_src=shape.msg_src, upd_src=shape.upd_src, msg_tsfm_type=tsfm,
                         mem_update_type=upd)
    res = model.load_state_dict(W, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    assert not [k for k in res.missing_keys if k.startswith(('score_fn.', 'hit_embedding.'))]
    model.eval()
    model.reset()
    e.reset()
    uptodate = set()
    start = (shape.n_events // 2) // B * B
    for ib in range(n_batches):
        lo = start + ib * B
        what = f'{shape.name} {hit_type} K={K} batch {ib} '
        src, dst, ng, ts, eids, _, cg = coll([full[i] for i in range(lo, lo + B)])
        src, dst, ng, eids = (x.long().cuda() for x in (src, dst, ng, eids))
        ts, cg = ts.float().cuda(), cg.to(device)
        fresh = sorted(set(cg.np_computation_graph_nodes.tolist()) - uptodate)
        model.restart(torch.tensor(fresh, dtype=torch.long, device=device),
                      torch.full((len(fresh),), ts.min().item(), device=device))
        uptodate.update(fresh)
        with torch.enable_grad():
            loss, h_left, ps, ns, hpl, hpr = model.contrast_learning(src, dst, ng, ts, eids, cg)
        e.set_batch(st.src[lo:lo + B], st.dst[lo:lo + B], neg[lo:lo + B], st.ts[lo:lo + B], st.eids[lo:lo + B])
        e.step()
        e.check_errors()
        assert np.array_equal(cpu(e.neigh_nids), cpu(cg.layers[n_layers][0])), what + 'neighbors'
        w = np.zeros(2 * B, dtype=np.uint8)
        w[cpu(cg.restart_data.index)] = 1
        assert np.array_equal(cpu(e.winner), w), what + 'winners'
        assert_close(cpu(e.emb[:2 * B]), cpu(h_left), TOL, what + 'h_left')
        assert_close(cpu(e.scores[:B]), cpu(ps), TOL, what + 'pos_scores')
        assert_close(cpu(e.scores[B:]), cpu(ns), TOL, what + 'neg_scores')
        assert_close(cpu(e.loss), cpu(loss).reshape(1), TOL, what + 'loss')
        assert_close(cpu(e.hprev_left), cpu(hpl), TOL, what + 'h_prev_left')
        assert_close(cpu(e.hprev_right), cpu(hpr), TOL, what + 'h_prev_right')
        assert_close(cpu(e.left_vals), cpu(model.left_memory.vals), TOL, what + 'left_vals')
        assert_close(cpu(e.right_vals), cpu(model.right_memory.vals), TOL, what + 'right_vals')
        assert np.array_equal(cpu(e.left_ts), cpu(model.left_memory.update_ts)), what + 'left_ts'
        assert np.array_equal(cpu(e.right_ts), cpu(model.right_memory.update_ts)), what + 'right_ts'
        assert np.array_equal(np.nonzero(cpu(e.has_msg))[0], np.array(sorted(model.msg_store.nodes_with_messages))), \
            what + 'pending'


@pytest.mark.parametrize('hit_type', ['vec', 'count'])
@pytest.mark.parametrize('name', ['wikipedia', 'reddit'])
def test_engine_matches_torch_route_at_baseline_dimensions(name, hit_type):
    """d = d_e = 172, K = 10, B = 200, lazy restart, 30 batches from mid-stream (Wikipedia: seq restarter,
    Reddit: static)."""
    shape = SHAPES[name]
    compare_with_torch_route(shape, hit_type=hit_type, restarter=shape.restarter)


def test_engine_matches_torch_route_vec_two_layers():
    shape = SHAPES['wikipedia']
    compare_with_torch_route(shape, hit_type='vec', restarter='seq', n_layers=2)


def test_engine_matches_torch_route_count_mlp_merge():
    shape = SHAPES['reddit']
    compare_with_torch_route(shape, hit_type='count', restarter='static', tsfm='mlp', upd='merge')


def test_engine_matches_torch_route_vec_k40():
    """K = 40: two 32-slot ballot chunks per side."""
    shape = SHAPES['reddit']
    compare_with_torch_route(shape, hit_type='vec', restarter='static', K=40)
