"""Read-only one-vs-many candidate queries (TigerEngine.candidate_query): the generalised scorer and its ranks against a
float64 restatement and numpy, the read-only compaction against the normal one, the restart surrogates against the rows
a lazy restart writes, the query's scores against the next ingest step's bit for bit (C = 2, cands = [dst, neg]) on the
goldens and the BASELINE-shaped streams, the state left untouched, arbitrary C against one ingest step per column, the
captured query against the eager one, and the refusals."""
import numpy as np
import pytest
import torch

from golden_utils import CASES, VAR_CASES, Golden
from www2023tiger_b200 import ops
from www2023tiger_b200.engine import TigerEngine
from www2023tiger_b200.init import perturb_biases, random_weights
from www2023tiger_b200.synthetic import SHAPES, NegativeSampler, make_stream

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = 'cuda'
cpu = lambda t: t.detach().cpu().numpy()
dev = lambda x, dt=None: torch.as_tensor(x, dtype=dt).to(DEV).contiguous()


# ------------------------------------------------------------------------------------------
# the generalised scorer and its ranks
# ------------------------------------------------------------------------------------------
def scorer64(pq, nids, neigh, fold, Q, C, K):
    """float64 restatement of tiger_link_score_cands from the folded tables: pair (i, j) scores src[i] (row i) against
    column j's node (row Q + j Q + i) as relu(P[s] + Q[t] + hit term) . w2 + b2."""
    d = fold.d
    pq, cab = pq.astype(np.float64), cpu(fold.cab).astype(np.float64)
    w2, b2 = cpu(fold.fc2_w).astype(np.float64), float(cpu(fold.fc2_b)[0])
    out = np.zeros((C, Q))
    for j in range(C):
        rs, rt = np.arange(Q), Q + j * Q + np.arange(Q)
        s_id, t_id = nids[rs], nids[rt]
        if neigh is not None:
            a = neigh[rt] == s_id[:, None]          # src in N(target)
            b = neigh[rs] == t_id[:, None]          # target in N(src)
        if fold.hit_type == 'none':
            h = np.broadcast_to(cab[:d], (Q, d))
        elif fold.hit_type == 'bin':
            h = cab[:4 * d].reshape(4, d)[2 * a.any(1) + b.any(1)]
        elif fold.hit_type == 'count':
            U, V = cab[:(K + 1) * d].reshape(K + 1, d), cab[(K + 1) * d:2 * (K + 1) * d].reshape(K + 1, d)
            h = U[a.sum(1)] + V[b.sum(1)]
        else:
            Ha, Hb = cab[d:(1 + K) * d].reshape(K, d), cab[(1 + K) * d:(1 + 2 * K) * d].reshape(K, d)
            h = cab[:d] + a @ Ha + b @ Hb
        out[j] = np.maximum(pq[rs, :d] + pq[rt, d:] + h, 0) @ w2 + b2
    return out


def ranks_np(s):
    """s [C, Q] -> 1 + #{j >= 1: s_j > s_0} + 0.5 #{j >= 1: s_j == s_0}, NaN for a NaN s_0."""
    s0 = s[0]
    r = 1 + (s[1:] > s0).sum(0) + 0.5 * (s[1:] == s0).sum(0)
    return np.where(np.isnan(s0), np.nan, r).astype(np.float32)


def make_fold(d, hit_type, K, rng):
    f = lambda *s: torch.from_numpy(rng.standard_normal(s).astype(np.float32) * 0.3).to(DEV)
    fold = ops.ScoreFold(d, DEV, hit_type, K)
    width = 2 * (d + K) if hit_type == 'vec' else 2 * d
    hit_emb = {'bin': f(2, d), 'count': f(K + 1, d)}.get(hit_type)
    fold.refresh(f(d, width), f(d), f(1, d), f(1), f(d, d), f(d), hit_emb)
    return fold


@pytest.mark.parametrize('C', [1, 2, 3, 33, 100])
@pytest.mark.parametrize('K', [1, 5, 10, 32, 40])
@pytest.mark.parametrize('hit_type', ['none', 'bin', 'vec', 'count'])
def test_scorer_and_ranks_against_float64(hit_type, K, C):
    rng = np.random.default_rng(K * 1000 + C)
    d = 24
    Q = 2000 if C <= 3 else 150
    n = (1 + C) * Q
    N = 50
    nids = rng.integers(0, N, n)
    neigh = rng.integers(0, N, (n, K))
    # plant hits: some target rows hold src, some src rows hold the target, some rows are all-hit
    for j in range(C):
        rs, rt = np.arange(Q), Q + j * Q + np.arange(Q)
        m = rng.random((Q, K)) < 0.3
        neigh[rt] = np.where(m, nids[rs][:, None], neigh[rt])
        m = rng.random((Q, K)) < 0.3
        neigh[rs[: Q // 2]] = np.where(m[: Q // 2], nids[rt[: Q // 2]][:, None], neigh[rs[: Q // 2]])
    neigh[rng.integers(0, n, 5)] = 0                 # padding rows
    pq = rng.standard_normal((n, 2 * d)).astype(np.float32)
    # deliberate ties: column j of some rows repeats column 0 (same node, same rows) -> the same score bit for bit
    for j in range(1, C):
        tie = rng.random(Q) < 0.2
        r0, rj = Q + np.arange(Q)[tie], Q + j * Q + np.arange(Q)[tie]
        nids[rj], pq[rj], neigh[rj] = nids[r0], pq[r0], neigh[r0]
    fold = make_fold(d, hit_type, K, rng)
    g_nids, g_neigh = dev(nids), dev(neigh)
    scores = torch.full((C * Q,), float('nan'), device=DEV)
    ranks = torch.full((Q,), -1.0, device=DEV)
    ops.link_score_cands(fold, dev(pq), g_nids[:Q], g_nids[Q:2 * Q], g_nids[2 * Q:],
                         g_neigh if hit_type != 'none' else None, scores, ranks)
    got = cpu(scores).reshape(C, Q)
    want = scorer64(pq, nids, neigh if hit_type != 'none' else None, fold, Q, C, K)
    err = np.abs(got - want).max() / np.abs(want).max()
    assert err <= TOL, f'{hit_type} K={K} C={C}: rel err {err:.3e}'
    np.testing.assert_array_equal(cpu(ranks), ranks_np(got))
    if C > 1:
        assert (cpu(ranks) % 1 == 0.5).any(), 'the planted ties must show as half ranks'
    if C == 2:
        # the batch entry point is this scorer at C = 2 (pos = dst, neg = the second column), loss included
        s2, loss = ops.link_score_folded(fold, dev(pq), g_nids[:Q], g_nids[Q:2 * Q], g_nids[2 * Q:],
                                         g_neigh if hit_type != 'none' else None)
        assert torch.equal(s2, scores)
        y = np.r_[np.ones(Q), np.zeros(Q)]
        x = got.reshape(-1).astype(np.float64)
        bce = np.mean(np.maximum(x, 0) - x * y + np.log1p(np.exp(-np.abs(x))))
        assert abs(float(loss) - bce) <= 1e-5 * max(1.0, abs(bce))


def test_ranks_of_non_finite_scores():
    """NaN true score -> NaN rank; a NaN candidate neither beats nor ties.  A NaN score comes from an infinite first
    layer: relu(inf) times second-layer weights of both signs."""
    rng = np.random.default_rng(3)
    d, Q, C = 8, 6, 4
    n = (1 + C) * Q
    fold = make_fold(d, 'none', 0, rng)
    w2 = cpu(fold.fc2_w)
    assert (w2 > 0).any() and (w2 < 0).any()
    pq = rng.standard_normal((n, 2 * d)).astype(np.float32)
    pq[0, :d] = np.inf                                  # query 0: every score NaN, the true one included
    pq[Q + 2 * Q + 1, d:] = np.inf                      # query 1: column 2 NaN
    pq[Q + 3 * Q + 2] = pq[Q + 2]                       # query 2: column 3 ties column 0
    nids = dev(np.arange(n) % 7)
    scores, ranks = torch.zeros(C * Q, device=DEV), torch.zeros(Q, device=DEV)
    ops.link_score_cands(fold, dev(pq), nids[:Q], nids[Q:2 * Q], nids[2 * Q:], None, scores, ranks)
    s = cpu(scores).reshape(C, Q)
    assert np.isnan(s[:, 0]).all() and np.isnan(s[2, 1]) and np.isfinite(np.delete(s, 0, 1)).sum() == C * (Q - 1) - 1
    r = cpu(ranks)
    assert np.isnan(r[0]) and r[2] % 1 == 0.5
    np.testing.assert_array_equal(r[1:], ranks_np(s)[1:])


# ------------------------------------------------------------------------------------------
# read-only compaction
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('N', [5000, 1_100_000])          # cluster kernel / word-serial kernel (> 8 x 4096 words)
@pytest.mark.parametrize('lazy', [True, False])
def test_read_only_compaction_matches_normal_mode(N, lazy):
    rng = np.random.default_rng(N)
    ids = dev(rng.integers(0, N, 3000))
    has_msg = dev(rng.random(N) < 0.4, torch.uint8)
    uptodate = dev(rng.random(N) < 0.6, torch.uint8)
    cap = 4000
    res = {}
    for ro in (False, True):
        bitmap = torch.zeros(ops.bitmap_words(N), dtype=torch.int32, device=DEV)
        ops.mark_nodes(ids, bitmap, N)
        hm, up = has_msg.clone(), uptodate.clone()
        lists = [torch.full((cap,), -7, dtype=torch.int64, device=DEV) for _ in range(3)]
        gru_row = torch.full((N,), -5, dtype=torch.int32, device=DEV)
        counts = torch.zeros(4, dtype=torch.int32, device=DEV)
        ops.compact_involved(bitmap, N, lists[0], counts, has_msg=hm, uptodate=up if lazy else None,
                             outdated=lists[1], gru_row=gru_row, restart_nodes=lists[2] if lazy else None,
                             read_only=ro, restart_base=cap)
        res[ro] = [cpu(t) for t in (counts, *lists, gru_row, hm, up, bitmap)]
    (cn, inv, out, rst, row, hm, up, bm), (cn_r, inv_r, out_r, rst_r, row_r, hm_r, up_r, bm_r) = res[False], res[True]
    U, O, R = cn[:3]
    assert np.array_equal(cn, cn_r) and np.array_equal(inv[:U], inv_r[:U]) and np.array_equal(out[:O], out_r[:O])
    assert not bm.any() and not bm_r.any()
    assert np.array_equal(hm_r, cpu(has_msg)) and np.array_equal(up_r, cpu(uptodate)), 'read-only mode wrote state'
    inv_nodes = inv[:U]
    if lazy:
        assert R > 0 and np.array_equal(rst[:R], rst_r[:R])
        assert (up[inv_nodes] == 1).all(), 'normal mode marks the involved nodes up to date'
        want = row[inv_nodes].copy()
        want[np.searchsorted(inv_nodes, rst[:R])] = cap + np.arange(R)
        assert np.array_equal(row_r[inv_nodes], want)
        assert (row[rst[:R]] == -1).all()
    else:
        assert np.array_equal(row_r[inv_nodes], row[inv_nodes])
    assert np.array_equal(row[out[:O]], np.arange(O))


# ------------------------------------------------------------------------------------------
# engine-level: the same answer as the step, state untouched
# ------------------------------------------------------------------------------------------
def state_of(e):
    return [t.clone() for t in (e.left_vals, e.left_ts, e.left_active, e.right_vals, e.right_ts, e.right_active,
                                e.msg_vals, e.msg_ts, e.has_msg, e.uptodate, e.err_flags)]


def step_scratch(e):
    return [t.clone() for t in (e.bitmap, e.involved, e.outdated, e.restart_nodes, e.gru_row, e.neigh_nids, e.h_new,
                                e.emb, e.pq)]


def assert_same(a, b, what):
    for k, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), f'{what}: tensor {k} differs'


def stream_with_queries(make_engine, batches, what):
    """Two engines on the same batches, one with a C = 2 query (cands = [dst, neg], the batch's times) before every
    batch: the query equals the step's scores bit for bit and leaves the state bit-identical, the restart surrogates
    equal the rows the step's lazy restart writes, and the two runs agree bit for bit."""
    e, ref = make_engine(), make_engine()
    B = e.B
    q = e.candidate_query(B, 2)
    for ib, (src, dst, neg, ts, eids) in enumerate(batches):
        w = f'{what} batch {ib}'
        before, scratch = state_of(e), step_scratch(e)
        scores, ranks = q.score(src, np.stack([dst, neg], 1), ts)
        scores, ranks = scores.clone(), ranks.clone()
        torch.cuda.synchronize()
        q.check_errors()
        assert_same(before, state_of(e), w + ' state after the query')
        assert_same(scratch, step_scratch(e), w + ' step scratch after the query')
        U, Oc, R = (int(x) for x in q.counts[:3])
        restart_nodes, surrogate = q.restart_nodes[:R].clone(), q.rows_b[q.cap:q.cap + R].clone()
        for eng in (e, ref):
            eng.set_batch(src, dst, neg, ts, eids)
            eng.step()
            eng.check_errors()
        assert [int(x) for x in e.counts[:3]] == [U, Oc, R], w + ' counts'
        assert torch.equal(scores[:, 0], e.scores[:B]), w + ' positive scores'
        assert torch.equal(scores[:, 1], e.scores[B:]), w + ' negative scores'
        s = cpu(scores)
        assert np.array_equal(cpu(ranks), 1 + (s[:, 1] > s[:, 0]) + 0.5 * (s[:, 1] == s[:, 0])), w + ' ranks'
        if e.lazy_restart:
            assert torch.equal(restart_nodes, e.restart_nodes[:R]), w + ' restart list'
            assert torch.equal(surrogate, e.right_vals[restart_nodes]), w + ' restart surrogates'
        assert torch.equal(e.out_buf, ref.out_buf), w + ' step outputs with / without queries'
    assert_same(state_of(e), state_of(ref), what + ' final state with / without queries')
    return e


def golden_engine(g, lazy):
    f = lambda x: None if x is None else dev(x, torch.float32)
    return TigerEngine({k: torch.as_tensor(v) for k, v in g.W.items()}, csr_of(g.src, g.dst, g.ts, g.eids, g.N),
                       n_nodes=g.N, dim=g.dim, efeats=f(g.efeats), nfeats=f(g.nfeats), n_neighbors=g.K,
                       n_head=g.n_heads, batch_size=g.bs, msg_src=g.msg_src, upd_src=g.upd_src,
                       restarter=g.restarter if lazy else None, hist_len=g.hist_len, lazy_restart=lazy,
                       n_layers=g.n_layers, msg_tsfm_type=g.tsfm, mem_update_type=g.upd, hit_type=g.hit_type)


_CSR = {}


def csr_of(src, dst, ts, eids, N):
    key = (id(src), N)
    if key not in _CSR:
        _CSR.clear()
        _CSR[key] = ops.csr_build(dev(src, torch.int64), dev(dst, torch.int64), dev(ts, torch.float64),
                                  dev(eids, torch.int64), N)
    return _CSR[key]


@pytest.mark.parametrize('name', CASES + VAR_CASES)
def test_query_equals_the_next_step_on_goldens(name):
    g = Golden(name)
    for lazy in sorted({g.lazy_restart, False}):
        if lazy and g.restarter not in ('static', 'seq'):
            continue
        stream_with_queries(lambda: golden_engine(g, lazy), [g.batch(ib) for ib in range(g.n_batches)],
                            f'{name} lazy={lazy}')


def full_setup(shape_name, restarter, *, n_layers=1, seed=0):
    shape = SHAPES[shape_name]
    st = make_stream(shape, seed=seed)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    d = st.nfeats.shape[1] if st.nfeats is not None else st.dim
    de = st.efeats.shape[1] if st.efeats is not None else d
    W = perturb_biases(random_weights(d, de, n_nodes=st.n_nodes, restarter=restarter, nonzero_static=True,
                                      seed=seed + 1, n_layers=n_layers))
    csr = csr_of(st.src, st.dst, st.ts, st.eids, st.n_nodes)
    f = lambda x: None if x is None else dev(x, torch.float32)

    def make(lazy=True, B=200):
        return TigerEngine(W, csr, n_nodes=st.n_nodes, dim=st.dim, efeats=f(st.efeats), nfeats=f(st.nfeats),
                           n_neighbors=10, n_head=2, batch_size=B, msg_src=shape.msg_src, upd_src=shape.upd_src,
                           restarter=restarter if lazy else None, lazy_restart=lazy, n_layers=n_layers)
    start = (st.n_events // 2) // 200 * 200

    def batches(n, B=200):
        return [(st.src[lo:lo + B], st.dst[lo:lo + B], neg[lo:lo + B], st.ts[lo:lo + B], st.eids[lo:lo + B])
                for lo in range(start, start + n * B, B)]
    return make, batches, st


@pytest.mark.parametrize('name, restarter', [('wikipedia', 'seq'), ('reddit', 'static')])
@pytest.mark.parametrize('lazy', [True, False])
def test_query_equals_the_next_step_at_baseline_dimensions(name, restarter, lazy):
    make, batches, _ = full_setup(name, restarter)
    stream_with_queries(lambda: make(lazy), batches(12), f'{name}/{restarter} lazy={lazy}')


def test_query_equals_the_next_step_two_layers_at_baseline_dimensions():
    make, batches, _ = full_setup('wikipedia', 'seq', n_layers=2)
    stream_with_queries(lambda: make(True, B=100), batches(6, B=100), 'wikipedia two layers')


# ------------------------------------------------------------------------------------------
# arbitrary C: one ingest step per candidate column, state restored in between
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name, restarter, n_layers', [('wikipedia', 'seq', 1), ('reddit', 'static', 1),
                                                       ('reddit', 'static', 2)])
def test_query_column_equals_one_step_per_column(name, restarter, n_layers):
    B, C = 200 if n_layers == 1 else 50, 20
    make, batches, st = full_setup(name, restarter, n_layers=n_layers)
    e = make(True, B=B)
    bs = batches(11, B=B)
    for b in bs[:10]:
        e.set_batch(*b)
        e.step()
    e.check_errors()
    src, _, neg, ts, eids = bs[10]
    rng = np.random.default_rng(5)
    cands = rng.integers(1, st.n_nodes, (B, C)).astype(np.int64)
    q = e.candidate_query(B, C)
    scores, _ = q.score(src, cands, ts)
    got = cpu(scores)
    q.check_errors()
    saved = state_of(e)
    worst = 0.0
    for j in range(C):
        e.set_batch(src, cands[:, j], neg, ts, eids)
        e.step()
        want = cpu(e.scores[:B])
        worst = max(worst, float(np.abs(got[:, j] - want).max() / np.abs(want).max()))
        restore(e, saved)
    print(f'{name}/{restarter} n_layers={n_layers} C={C}: max rel err of a column vs its step {worst:.3e}')
    assert worst <= TOL


def restore(e, saved):
    for t, s in zip((e.left_vals, e.left_ts, e.left_active, e.right_vals, e.right_ts, e.right_active, e.msg_vals,
                     e.msg_ts, e.has_msg, e.uptodate, e.err_flags), saved):
        t.copy_(s)


# ------------------------------------------------------------------------------------------
# capture, shared weights, refusals
# ------------------------------------------------------------------------------------------
def test_captured_query_equals_eager_query():
    make, batches, st = full_setup('wikipedia', 'seq')
    e = make(True)
    for b in batches(5):
        e.set_batch(*b)
        e.step()
    Q, C = 150, 30
    qe, qc = e.candidate_query(Q, C), e.candidate_query(Q, C)
    qc.capture()
    rng = np.random.default_rng(9)
    for rep in range(4):
        src = rng.integers(1, st.n_nodes, Q).astype(np.int64)
        cands = rng.integers(1, st.n_nodes, (Q, C)).astype(np.int64)
        ts = np.sort(rng.uniform(st.ts[len(st.ts) // 2], st.ts[-1], Q))
        a, ra = qe.score(src, cands, ts)
        b, rb = qc.score(dev(src), dev(cands), dev(ts))          # device inputs into the captured graph
        assert torch.equal(a, b) and torch.equal(ra, rb), f'replay {rep}'
        # fewer queries than captured: eager launches on the same buffers
        a, ra = qe.score(src[:7], cands[:7], ts[:7])
        b, rb = qc.score(src[:7], cands[:7], ts[:7])
        assert torch.equal(a, b) and torch.equal(ra, rb), f'replay {rep}, 7 queries'
    qe.check_errors()
    qc.check_errors()


@pytest.mark.parametrize('name, restarter, n_layers', [('wikipedia', 'seq', 1), ('reddit', 'static', 2)])
def test_capture_below_max_queries_survives_eager_calls_at_max(name, restarter, n_layers):
    """The query's workspaces are sized once for max_queries: a graph captured for fewer queries keeps valid addresses
    after eager calls at max_queries, and its replay equals an eager query bit for bit."""
    make, batches, st = full_setup(name, restarter, n_layers=n_layers)
    B = 200 if n_layers == 1 else 50
    e = make(True, B=B)
    for b in batches(4, B=B):
        e.set_batch(*b)
        e.step()
    Q, n, C = 60, 20, 12
    qe, qc = e.candidate_query(Q, C), e.candidate_query(Q, C)
    works = [p._work.data_ptr() for p in (qc.attn, qc.attn1) if p is not None]
    qc.capture(n)
    rng = np.random.default_rng(11)

    def inputs(m):
        return (rng.integers(1, st.n_nodes, m).astype(np.int64), rng.integers(1, st.n_nodes, (m, C)).astype(np.int64),
                np.sort(rng.uniform(st.ts[len(st.ts) // 2], st.ts[-1], m)))
    for rep in range(3):
        big = inputs(Q)
        a, ra = qe.score(*big)
        b, rb = qc.score(*big)                                   # eager, at max_queries
        assert torch.equal(a, b) and torch.equal(ra, rb), f'eager at max_queries, round {rep}'
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        small = inputs(n)
        a, ra = qe.score(*small)
        b, rb = qc.score(*small)                                 # graph replay
        assert torch.equal(a, b) and torch.equal(ra, rb), f'replay at {n} queries, round {rep}'
    assert [p._work.data_ptr() for p in (qc.attn, qc.attn1) if p is not None] == works
    qe.check_errors()
    qc.check_errors()


def test_graph_captured_before_load_weights_is_not_replayed():
    """load_weights replaces weight tensors a captured query graph reads: the next score() drops the graph and
    launches eagerly on the new weights, and a new capture replays them."""
    make, batches, st = full_setup('reddit', 'static')
    e = make(True)
    bs = batches(3)
    for b in bs[:2]:
        e.set_batch(*b)
        e.step()
    src, dst, neg, ts, eids = bs[2]
    cands = np.stack([dst, neg], 1)
    q = e.candidate_query(200, 2)
    q.capture()
    d = st.nfeats.shape[1] if st.nfeats is not None else st.dim
    de = st.efeats.shape[1] if st.efeats is not None else d
    e.load_weights(perturb_biases(random_weights(d, de, n_nodes=st.n_nodes, restarter='static', nonzero_static=True,
                                                 seed=78)))
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    a = q.score(src, cands, ts)[0].clone()
    assert q.graph is None
    q.capture()
    b = q.score(src, cands, ts)[0].clone()
    assert q.graph is not None and torch.equal(a, b)
    e.set_batch(src, dst, neg, ts, eids)
    e.step()
    assert torch.equal(a[:, 0], e.scores[:200]) and torch.equal(a[:, 1], e.scores[200:])


def test_query_reads_the_engine_weights():
    """No second copy: load_weights on the engine changes the query's scores to the step's under the new weights."""
    make, batches, st = full_setup('reddit', 'static')
    e = make(True)
    bs = batches(3)
    for b in bs[:2]:
        e.set_batch(*b)
        e.step()
    q = e.candidate_query(200, 2)
    src, dst, neg, ts, eids = bs[2]
    before = q.score(src, np.stack([dst, neg], 1), ts)[0].clone()
    d = st.nfeats.shape[1] if st.nfeats is not None else st.dim
    de = st.efeats.shape[1] if st.efeats is not None else d
    W2 = perturb_biases(random_weights(d, de, n_nodes=st.n_nodes, restarter='static', nonzero_static=True, seed=77))
    e.load_weights(W2)
    after = q.score(src, np.stack([dst, neg], 1), ts)[0].clone()
    e.set_batch(src, dst, neg, ts, eids)
    e.step()
    assert not torch.equal(before, after)
    assert torch.equal(after[:, 0], e.scores[:200]) and torch.equal(after[:, 1], e.scores[200:])


def test_refusals_launch_nothing():
    make, _, st = full_setup('reddit', 'static')
    e = make(True)
    q = e.candidate_query(10, 3)
    q.scores.fill_(7.0)
    q.ranks.fill_(7.0)
    ok = dict(src=np.arange(1, 5, dtype=np.int64), cands=np.ones((4, 3), np.int64), ts=np.full(4, 1e6))
    bad = [dict(src=np.arange(1, 12, dtype=np.int64), cands=np.ones((11, 3), np.int64), ts=np.full(11, 1e6)),
           dict(cands=np.ones((4, 2), np.int64)), dict(cands=np.ones((4, 3), np.int32)), dict(ts=np.ones(4, np.float32)),
           dict(src=np.ones((4, 1), np.int64)), dict(cands=np.ones(12, np.int64)),
           dict(cands=np.full((4, 3), st.n_nodes, np.int64)), dict(src=torch.full((4,), -1, dtype=torch.int64,
                                                                                   device=DEV))]
    for b in bad:
        with pytest.raises(ValueError):
            q.score(**{**ok, **b})
    torch.cuda.synchronize()
    assert bool((q.scores == 7.0).all()) and bool((q.ranks == 7.0).all())
    for args in ((0, 2), (5, 0), (2.0, 2)):
        with pytest.raises(ValueError):
            e.candidate_query(*args)
