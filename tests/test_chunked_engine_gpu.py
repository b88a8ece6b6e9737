"""TigerEngine(n_chunks=M): M time chunks of one stream as one batched step, each chunk with its own memory.

The chunked engine against M independent engines each fed its own chunk (neighbor tables, winners and the involved /
outdated / restart sets bit-identical; scores and every state slice within 1e-5; the loss equal to the mean of the
per-chunk losses), eager and under StreamRunner graph replay; n_chunks=1 against the engine without the argument
(bit-identical, same launch list); the chunk modes of tiger_find_recent_ex, tiger_min_time_ex and
tiger_static_restart_ex against numpy / float64; and the isolation of one chunk from the events of another."""
import numpy as np
import pytest
import torch

from golden_utils import assert_close
from oracle import tiger_oracle as O
from www2023tiger_b200 import ops
from www2023tiger_b200.engine import StreamRunner, TigerEngine, chunk_bounds
from www2023tiger_b200.init import perturb_biases, random_weights
from www2023tiger_b200.synthetic import SHAPES, NegativeSampler, StreamShape, make_stream

pytestmark = pytest.mark.gpu
TOL = 1e-5
cpu = lambda t: t.detach().cpu().numpy()
dev = lambda x, dt: torch.as_tensor(x).to(dt).cuda().contiguous()
STATE = ('left_vals', 'left_ts', 'left_active', 'right_vals', 'right_ts', 'right_active', 'msg_vals', 'msg_ts',
         'has_msg', 'uptodate')


class Case:
    """A stream, its CSR and weights, and the chunk windows: batch i of chunk c is events
    [lo_c + i B, lo_c + (i + 1) B) of the ChunkSampler partition."""

    def __init__(self, shape, M, n_batches, *, B=200, K=10, restarter='static', n_layers=1, hit_type='bin',
                 mem_update_type='gru', nfeats=False, seed=0):
        n_events = M * B * (n_batches + 1) + 77
        self.st = st = make_stream(shape, seed=seed, n_events=n_events)
        self.neg = NegativeSampler(st.src, st.dst, seed=seed).pre_sample_neg_dsts(st.n_events, B)
        self.N, self.M, self.B, self.n_batches = st.n_nodes, M, B, n_batches
        d = st.dim
        self.nf = np.random.RandomState(seed).randn(self.N, d).astype(np.float32) if nfeats else None
        self.W = perturb_biases(random_weights(d, d, n_nodes=self.N, restarter=restarter, nonzero_static=True,
                                               n_layers=n_layers, hit_type=hit_type, n_neighbors=K,
                                               mem_update_type=mem_update_type, seed=seed + 1))
        self.csr = ops.csr_build(dev(st.src, torch.int64), dev(st.dst, torch.int64), dev(st.ts, torch.float64),
                                 dev(st.eids, torch.int64), self.N)
        self.kw = dict(n_nodes=self.N, dim=d, efeats=dev(st.efeats, torch.float32),
                       nfeats=None if self.nf is None else dev(self.nf, torch.float32), n_neighbors=K, n_head=2,
                       batch_size=B, msg_src=shape.msg_src, upd_src=shape.upd_src, restarter=restarter,
                       lazy_restart=True, n_layers=n_layers, hit_type=hit_type, mem_update_type=mem_update_type)
        self.bounds = chunk_bounds(st.n_events, M, B, seed=seed)
        assert all(hi - lo >= n_batches * B for lo, hi in self.bounds)

    def engine(self, **kw):
        return TigerEngine(self.W, self.csr, **self.kw, **kw)

    def batch(self, c, i, events=None):
        """(src, dst, neg, ts, eids) of batch i of chunk c (events: a replacement stream window start)."""
        lo = (self.bounds[c][0] if events is None else events) + i * self.B
        s = slice(lo, lo + self.B)
        return self.st.src[s], self.st.dst[s], self.neg[s], self.st.ts[s], self.st.eids[s]

    def chunked(self, i, starts=None, pinned=()):
        """The chunk-major [M, B] arrays of step i (chunks in `pinned` replay their batch 0 at every step)."""
        per = [self.batch(c, 0 if c in pinned else i, None if starts is None else starts[c]) for c in range(self.M)]
        return tuple(np.stack([p[j] for p in per]) for j in range(5))


def lists(e):
    U, O, R = (int(x) for x in cpu(e.counts[:3]))
    return cpu(e.involved[:U]), cpu(e.outdated[:O]), cpu(e.restart_nodes[:R])


def chunk_slice(t, c, N):
    return cpu(t[c * N:(c + 1) * N])


def compare_step(case, eng, refs, worst, *, tables=True, state=True):
    """One step of the chunked engine against the chunk engines; returns nothing, updates worst[name]."""
    M, N, B = case.M, case.N, case.B
    pos, neg = eng.chunk_scores()
    pos, neg = cpu(pos), cpu(neg)
    if tables:
        K = eng.K
        nn = cpu(eng.neigh_nids).reshape(3, M, B, K)
        win = cpu(eng.winner).reshape(2, M, B)
        inv, out, rst = lists(eng)
    losses = []
    for c, r in enumerate(refs):
        if tables:
            got = nn[:, c].reshape(3 * B, K)
            assert np.array_equal(np.where(got == 0, 0, got - c * N), cpu(r.neigh_nids)), f'chunk {c}: neighbors'
            assert np.array_equal(win[:, c].reshape(-1), cpu(r.winner)), f'chunk {c}: winners'
            for got, want, what in zip((inv, out, rst), lists(r), ('involved', 'outdated', 'restart')):
                sel = got[(got >= c * N) & (got < (c + 1) * N)] - c * N
                assert np.array_equal(sel, want), f'chunk {c}: {what} set'
        rs = cpu(r.scores)
        for got, want, what in ((pos[c], rs[:B], 'pos'), (neg[c], rs[B:], 'neg')):
            assert_close(got, want, TOL, f'chunk {c}: {what} scores')
            worst['scores'] = max(worst.get('scores', 0.0), rel(got, want))
        for name in STATE if state else ():
            got, want = chunk_slice(getattr(eng, name), c, N), cpu(getattr(r, name))
            assert_close(got, want, TOL, f'chunk {c}: {name}')
            worst[name] = max(worst.get(name, 0.0), rel(got, want))
        losses.append(float(r.loss))
    assert abs(float(eng.loss) - np.mean(losses)) <= TOL * max(1.0, abs(np.mean(losses))), 'loss'
    worst['loss'] = max(worst.get('loss', 0.0), abs(float(eng.loss) - np.mean(losses)))


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)) if a.size else 0.0


def run_refs(case, refs, i):
    for c, r in enumerate(refs):
        r.set_batch(*case.batch(c, i))
        r.step()


def report(tag, worst, eng, refs):
    caps = (eng.cap, refs[0].cap)
    print(f'\n[chunk parity] {tag}: largest relative deviation ' +
          ', '.join(f'{k} {v:.2e}' for k, v in sorted(worst.items())) + f'; involved capacity {caps[0]} (chunked) '
          f'vs {caps[1]} (per chunk)')


# ------------------------------------------------------------------------------------------
# 1. equivalence with M independent engines
# ------------------------------------------------------------------------------------------
TOY = StreamShape('toy', 70, 25, 0, 16, None, horizon=20000.)
CONFIGS = {
    # name: (shape, restarter, n_layers, extra engine kwargs)
    'toy-static': (TOY, 'static', 1, {}),
    'toy-seq': (TOY, 'seq', 1, {}),
    'toy-static-2l': (TOY, 'static', 2, {}),
    'toy-seq-2l-merge': (TOY, 'seq', 2, {'mem_update_type': 'merge'}),
    'toy-static-vec-nfeats': (TOY, 'static', 1, {'hit_type': 'vec', 'nfeats': True}),
    'wikipedia-seq': (SHAPES['wikipedia'], 'seq', 1, {}),
    'reddit-static': (SHAPES['reddit'], 'static', 1, {}),
}


@pytest.mark.parametrize('M', [1, 2, 3, 5, 6])        # M = 6: 2,400 selection positions, the per-node slot route
@pytest.mark.parametrize('config', list(CONFIGS))
def test_chunked_equals_independent_engines_eager(config, M):
    shape, rst, layers, extra = CONFIGS[config]
    n_batches = 30 if shape is TOY else 31
    case = Case(shape, M, n_batches, restarter=rst, n_layers=layers, **extra)
    eng = case.engine(n_chunks=M)
    assert (eng.sel_scratch is not None) == (M == 6)
    refs = [case.engine() for _ in range(M)]
    for e in [eng] + refs:
        e.reset()
    worst = {}
    for i in range(n_batches):
        eng.set_batch(*case.chunked(i))
        eng.step()
        run_refs(case, refs, i)
        # every state slice after each toy batch; after every 10th and the last at BASELINE sizes
        compare_step(case, eng, refs, worst, state=shape is TOY or i % 10 == 9 or i == n_batches - 1)
    eng.check_errors()
    report(f'{config} M={M} eager', worst, eng, refs)


@pytest.mark.parametrize('M', [2, 3])
def test_seq_chunks_bit_identical_on_the_product_route(M):
    """A chunked engine runs the seq restarter's products for any restarted-row count (its route must not depend on
    the other chunks); independent engines held to that route as well agree with it bit for bit, so the deviation of
    the default engines (matrix-vector tail for <= 64 restarted rows) is that route difference alone."""
    case = Case(SHAPES['wikipedia'], M, 31, restarter='seq')
    eng = case.engine(n_chunks=M)
    assert eng.seq.tail_rows == 0
    refs = [case.engine() for _ in range(M)]
    for r in refs:
        r.seq.tail_rows = 0
    for e in [eng] + refs:
        e.reset()
    small = 0
    for i in range(31):
        eng.set_batch(*case.chunked(i))
        eng.step()
        run_refs(case, refs, i)
        small += sum(int(r.counts[2]) <= 64 for r in refs)
        pos, neg = eng.chunk_scores()
        for c, r in enumerate(refs):
            assert torch.equal(torch.cat([pos[c], neg[c]]), r.scores), f'batch {i} chunk {c}: scores'
            for name in STATE:
                a, b = getattr(eng, name)[c * case.N:(c + 1) * case.N], getattr(r, name)
                assert torch.equal(a, b), f'batch {i} chunk {c}: {name}'
    assert small > 0, 'no chunk restarted <= 64 nodes in a step: the tail route was never in play'


@pytest.mark.parametrize('config,M', [('toy-static', 3), ('toy-seq-2l-merge', 2), ('wikipedia-seq', 5),
                                      ('reddit-static', 5)])
def test_chunked_equals_independent_engines_graph_replay(config, M):
    """StreamRunner: captured graphs fed by submit_host (the first half) and by device_records + submit_device."""
    shape, rst, layers, extra = CONFIGS[config]
    n_batches = 30
    case = Case(shape, M, n_batches, restarter=rst, n_layers=layers, **extra)
    eng = case.engine(n_chunks=M)
    refs = [case.engine() for _ in range(M)]
    runner = StreamRunner(eng)
    eng.set_batch(*case.chunked(0))
    runner.capture(warmup=2)
    for e in [eng] + refs:
        e.reset()
    records = eng.device_records(*(np.stack(x) for x in zip(*(case.chunked(i) for i in range(n_batches)))))
    assert records.shape == (n_batches, 5 * M * case.B)
    worst = {}
    for i in range(n_batches):
        if i < n_batches // 2:
            slot = runner.submit_host(*case.chunked(i))
            pos, neg, loss = runner.wait(slot)
            assert pos.shape == (M, case.B) and neg.shape == (M, case.B)
        else:
            slot = runner.submit_device(records[i])
            runner.join()
            torch.cuda.synchronize()
            res = cpu(runner.d_out[slot])
            pos, neg, loss = res[:M * case.B].reshape(M, -1), res[M * case.B:2 * M * case.B].reshape(M, -1), res[-1]
        torch.cuda.synchronize()
        run_refs(case, refs, i)
        losses = [float(r.loss) for r in refs]
        for c, r in enumerate(refs):
            rs = cpu(r.scores)
            assert_close(np.asarray(pos[c]), rs[:case.B], TOL, f'step {i} chunk {c}: pos')
            assert_close(np.asarray(neg[c]), rs[case.B:], TOL, f'step {i} chunk {c}: neg')
            worst['scores'] = max(worst.get('scores', 0.0), rel(pos[c], rs[:case.B]), rel(neg[c], rs[case.B:]))
            for name in STATE if shape is TOY or i % 10 == 9 or i == n_batches - 1 else ():
                got, want = chunk_slice(getattr(eng, name), c, case.N), cpu(getattr(r, name))
                assert_close(got, want, TOL, f'step {i} chunk {c}: {name}')
                worst[name] = max(worst.get(name, 0.0), rel(got, want))
        assert abs(float(loss) - np.mean(losses)) <= TOL * max(1.0, abs(np.mean(losses))), f'step {i}: loss'
    eng.check_errors()
    report(f'{config} M={M} graph replay', worst, eng, refs)


# ------------------------------------------------------------------------------------------
# 2. n_chunks=1 is the engine
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('config', ['toy-static', 'toy-seq-2l-merge', 'reddit-static'])
def test_one_chunk_is_the_engine(config):
    shape, rst, layers, extra = CONFIGS[config]
    case = Case(shape, 1, 12, restarter=rst, n_layers=layers, **extra)
    a, b = case.engine(), case.engine(n_chunks=1)
    assert a.launches_per_step() == b.launches_per_step() and a.cap == b.cap
    for e in (a, b):
        e.reset()
    for i in range(12):
        for e in (a, b):
            e.set_batch(*case.batch(0, i))
            e.step()
        for name in STATE + ('scores', 'loss', 'neigh_nids', 'winner', 'emb'):
            assert torch.equal(getattr(a, name), getattr(b, name)), f'batch {i}: {name}'


# ------------------------------------------------------------------------------------------
# 3. the chunk modes of the new entry points against numpy / float64
# ------------------------------------------------------------------------------------------
def small_csr(N, E, seed):
    rng = np.random.RandomState(seed)
    src, dst = rng.randint(1, N, E), rng.randint(1, N, E)
    ts = np.sort(rng.randint(0, E // 3, E)).astype(np.float64)      # integer times: ties
    eids = np.arange(1, E + 1)
    src[:5] = dst[:5] = N - 1                                       # self loops at the top id
    csr = ops.csr_build(dev(src, torch.int64), dev(dst, torch.int64), dev(ts, torch.float64), dev(eids, torch.int64), N)
    return csr, O.OracleGraph(src, dst, ts, eids, n_nodes=N)


@pytest.mark.parametrize('M,N,k', [(2, 31, 5), (5, 97, 10), (16, 13, 3)])
def test_find_recent_chunk_neighbors(M, N, k):
    csr, g = small_csr(N, 600, M * N)
    rng = np.random.RandomState(N)
    n_q, period = 3 * 7 * M, 7 * M
    u = rng.randint(0, N, n_q)
    u[:3] = N - 1                                                   # the top id of a chunk ...
    c = rng.randint(0, M, n_q)
    c[:3] = M - 1                                                   # ... of the top chunk
    u[3] = 0                                                        # a node without history
    c[4], u[4] = 0, 0                                               # id 0: the second hop of a padding slot
    qt = rng.randint(0, 250, period).astype(np.float64)
    bitmap = torch.zeros(ops.bitmap_words(M * N), dtype=torch.int32, device='cuda')
    ts32 = torch.zeros(period, device='cuda')
    nn, ne, nt, nd = ops.find_recent(csr, dev(c * N + u, torch.int64), dev(qt, torch.float64), k, ts_period=period,
                                     ts32_out=ts32, bitmap=bitmap, chunk_mode=ops.FIND_CHUNK_NEIGHBORS, node_stride=N)
    wn, we, wt, _ = g.find_recent(u, qt[np.arange(n_q) % period], k)
    virt = wn + (c * N)[:, None]
    assert np.array_equal(cpu(nn), np.where(wn == 0, 0, virt))     # the padding stays 0
    assert np.array_equal(cpu(ne), we) and np.array_equal(cpu(nt), wt)
    assert (cpu(nn[3]) == 0).all()
    live = c * N + u != 0                                           # a query with id 0 marks nothing
    want_bits = np.zeros(M * N, bool)
    want_bits[(c * N + u)[live]] = True
    want_bits[virt[live].ravel()] = True                           # padding marks the chunk's node 0
    assert np.array_equal(cpu(ts32), qt.astype(np.float32))
    bits = np.unpackbits(cpu(bitmap).view(np.uint8), bitorder='little')[:M * N].astype(bool)
    assert np.array_equal(bits, want_bits)


@pytest.mark.parametrize('M,N,L', [(3, 31, 8), (7, 53, 40)])
def test_find_recent_chunk_history(M, N, L):
    csr, g = small_csr(N, 500, M + N)
    rng = np.random.RandomState(M)
    n_q = 4 * M
    u, c = rng.randint(0, N, n_q), rng.randint(0, M, n_q)
    u[0], c[0] = N - 1, M - 1
    tmin = rng.randint(0, 200, M).astype(np.float64)
    count = dev([n_q - 1], torch.int32)                             # the last query is beyond the device count
    out = tuple(torch.full((n_q, L), -7, dtype=dt, device='cuda') for dt in (torch.int64, torch.int64, torch.float32,
                                                                             torch.int64))
    ops.find_recent(csr, dev(c * N + u, torch.int64), dev(tmin, torch.float64), L, out=out, count=count,
                    chunk_mode=ops.FIND_CHUNK_HISTORY, node_stride=N)
    wn, we, wt, wd = g.get_history(u, tmin[c], L)
    for got, want in zip(out, (wn, we, wt, wd)):
        assert np.array_equal(cpu(got[:n_q - 1]), want[:n_q - 1])
    assert (cpu(out[0][n_q - 1]) == -7).all()


@pytest.mark.parametrize('M,B', [(1, 200), (2, 1), (5, 200), (16, 37), (3, 1000)])
def test_min_time_per_chunk(M, B):
    ts = np.random.RandomState(M * B).uniform(-1e6, 1e7, M * B).astype(np.float32)
    out = torch.zeros(M, dtype=torch.float64, device='cuda')
    ops.min_time(dev(ts, torch.float32), out, M)
    assert np.array_equal(cpu(out), ts.reshape(M, B).min(1).astype(np.float64))


@pytest.mark.parametrize('M,N,d', [(2, 31, 16), (5, 97, 172), (9, 13, 7)])
def test_static_restart_chunk_mode(M, N, d):
    csr, g = small_csr(N, 400, d)
    rng = np.random.RandomState(d)
    left_emb, right_emb = rng.randn(N, d).astype(np.float32), rng.randn(N, d).astype(np.float32)
    tmin64 = np.float32(rng.uniform(0, 140, M)).astype(np.float64)
    nodes = rng.choice(M * N, min(M * N, 40), replace=False)
    nodes[0] = M * N - 1
    R = len(nodes)
    z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device='cuda')
    lv, rv, lt, rt = z(M * N, d), z(M * N, d), z(M * N), z(M * N)
    la, ra, hm = z(M * N, dt=torch.uint8), z(M * N, dt=torch.uint8), torch.ones(M * N, dtype=torch.uint8, device='cuda')
    prev = z(R + 3)
    ops.static_restart(dev(nodes, torch.int64), R + 3, csr, dev(left_emb, torch.float32),
                       dev(right_emb, torch.float32), d, count=dev([R], torch.int32), left_vals=lv, left_ts=lt,
                       left_active=la, right_vals=rv, right_ts=rt, right_active=ra, has_msg=hm, out_prev_ts=prev,
                       node_stride=N, chunk_ts=dev(tmin64, torch.float64))
    want_lv, want_rv = np.zeros((M * N, d), np.float32), np.zeros((M * N, d), np.float32)
    want_t, want_hm = np.zeros(M * N, np.float32), np.ones(M * N, np.uint8)
    for i, v in enumerate(nodes):
        c, u = divmod(int(v), N)
        seg = g.ts[g.indptr[u]:g.indptr[u + 1]]
        cut = np.searchsorted(seg, tmin64[c], side='left')
        want_t[v] = np.float32(seg[cut - 1]) if cut > 0 else 0.0
        want_lv[v], want_rv[v], want_hm[v] = left_emb[u], right_emb[u], 0
        assert cpu(prev[i]) == want_t[v], i
    mark = np.zeros(M * N, np.uint8)
    mark[nodes] = 1
    for got, want in ((lv, want_lv), (rv, want_rv), (lt, want_t), (rt, want_t), (la, mark), (ra, mark), (hm, want_hm)):
        assert np.array_equal(cpu(got), want)


# ------------------------------------------------------------------------------------------
# 4. isolation
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('config', ['toy-static', 'toy-seq-2l-merge', 'wikipedia-seq'])
def test_chunk_isolation(config):
    """Replacing every batch of chunk 1 by other events leaves the scores and state slices of the other chunks
    bit-identical.  At the Wikipedia / seq dimensions chunk 1 of the second run replays its first batch at every step,
    so it restarts (almost) nothing after step 0, and the step's restarted-row count (summed over the chunks) lies on
    different sides of the seq restarter's 64-row route threshold in the two runs."""
    shape, rst, layers, extra = CONFIGS[config]
    M, n_batches = (3, 20) if shape is TOY else (2, 40)
    case = Case(shape, M, n_batches, restarter=rst, n_layers=layers, **extra)
    a, b = case.engine(n_chunks=M), case.engine(n_chunks=M)
    starts = [lo for lo, _ in case.bounds]
    pinned = ()
    if shape is TOY:
        starts[1] = starts[2]                                      # chunk 1 replays chunk 2's events
    else:
        pinned = (1,)
    for e in (a, b):
        e.reset()
    N = case.N
    totals = []
    for i in range(n_batches):
        a.set_batch(*case.chunked(i))
        b.set_batch(*case.chunked(i, starts, pinned))
        a.step()
        b.step()
        totals.append((int(a.counts[2]), int(b.counts[2])))
        (pa, na), (pb, nb) = a.chunk_scores(), b.chunk_scores()
        for c in (0, 2)[:M - 1]:
            assert torch.equal(pa[c], pb[c]) and torch.equal(na[c], nb[c]), f'batch {i}: chunk {c} scores'
            for name in STATE:
                assert torch.equal(getattr(a, name)[c * N:(c + 1) * N], getattr(b, name)[c * N:(c + 1) * N]), \
                    f'batch {i}: chunk {c} {name}'
        assert (i == 0 and pinned) or not torch.equal(pa[1], pb[1])      # a pinned chunk 1 differs from step 1
    if rst == 'seq' and shape is not TOY:
        assert any((ra <= 64) != (rb <= 64) for ra, rb in totals), \
            f'the restarted-row totals of the two runs never straddled 64: {totals}'


def test_chunked_engine_refuses_candidate_query():
    case = Case(TOY, 2, 1)
    with pytest.raises(NotImplementedError):
        case.engine(n_chunks=2).candidate_query(4, 3)
