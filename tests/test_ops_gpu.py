"""GPU parity of every C-ABI operator against the CPU oracle (and the reference's golden
vectors).  Index results are compared bit-exactly, fp32 results with max|a-b|/max|b| <= 1e-5."""
import numpy as np
import pytest
import torch

from oracle import tiger_oracle as O
from golden_utils import CASES, Golden, assert_close
from www2023tiger_b200 import ops
from www2023tiger_b200._lib import TigerLibraryError
from www2023tiger_b200.init import perturb_biases, random_weights
from www2023tiger_b200.synthetic import StreamShape, make_stream

pytestmark = pytest.mark.gpu
TOL = 1e-5


@pytest.fixture(scope='module')
def gu():
    import gpu_utils
    return gpu_utils


def small_stream(seed=0, n_events=6000, horizon=4000.):
    return make_stream(StreamShape('t', 300, 40, n_events, 8, None, horizon=horizon), seed=seed)


# ------------------------------------------------------------------ a1: CSR build
@pytest.mark.parametrize('n_events', [0, 1, 37, 6000, 70000])
def test_csr_build_matches_oracle(gu, n_events):
    st = small_stream(n_events=max(n_events, 1))
    src, dst, ts, eids = (x[:n_events] for x in (st.src, st.dst, st.ts, st.eids))
    N = st.n_nodes
    g = O.OracleGraph(src, dst, ts, eids, n_nodes=N)
    c = gu.device_csr(src, dst, ts, eids, N)
    assert np.array_equal(gu.cpu(c.indptr), g.indptr)
    assert np.array_equal(gu.cpu(c.nbr), g.nbr) and np.array_equal(gu.cpu(c.eid), g.eid)
    assert np.array_equal(gu.cpu(c.ts), g.ts) and np.array_equal(gu.cpu(c.flag), g.flag)


def test_csr_build_many_nodes(gu):
    # > 2^16 node ids exercises three radix passes
    rng = np.random.RandomState(0)
    E, N = 50000, 200001
    src = rng.randint(1, 100000, E).astype(np.int64)
    dst = rng.randint(100000, N, E).astype(np.int64)
    ts = np.floor(np.sort(rng.uniform(0, 1e5, E)))
    eids = np.arange(1, E + 1, dtype=np.int64)
    g = O.OracleGraph(src, dst, ts, eids, n_nodes=N)
    c = gu.device_csr(src, dst, ts, eids, N)
    assert np.array_equal(gu.cpu(c.indptr), g.indptr) and np.array_equal(gu.cpu(c.nbr), g.nbr)
    assert np.array_equal(gu.cpu(c.eid), g.eid) and np.array_equal(gu.cpu(c.flag), g.flag)


# ------------------------------------------------------------------ a2: finder
@pytest.mark.parametrize('k', [1, 10, 40])
def test_find_recent_matches_oracle(gu, k):
    st = small_stream(seed=3, n_events=30000, horizon=3000.)   # popular items have > 1000 events: deep search
    N = st.n_nodes
    g = O.OracleGraph(st.src, st.dst, st.ts, st.eids, n_nodes=N)
    c = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    rng = np.random.RandomState(k)
    q_n = np.concatenate([rng.randint(0, N, 3000), st.dst[rng.randint(0, len(st.dst), 2000)]]).astype(np.int64)
    q_t = np.concatenate([np.floor(rng.uniform(-5, 3100, 4000)), st.ts[rng.randint(0, len(st.ts), 1000)]])
    ref = g.find_recent(q_n, q_t, k)
    got = ops.find_recent(c, gu.dev(q_n), gu.dev(q_t, torch.float64), k)
    for a, b in zip(got, ref):
        assert np.array_equal(gu.cpu(a), b)
    assert gu.cpu(got[2]).dtype == np.float32


def test_find_recent_ts_period_and_bitmap(gu):
    st = small_stream(seed=5)
    N = st.n_nodes
    g = O.OracleGraph(st.src, st.dst, st.ts, st.eids, n_nodes=N)
    c = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    B, K = 50, 7
    lo = 3000
    src, dst, ts = st.src[lo:lo + B], st.dst[lo:lo + B], st.ts[lo:lo + B]
    neg = np.random.RandomState(0).randint(301, N, B).astype(np.int64)
    b = O.collate(g, src, dst, neg, ts, st.eids[lo:lo + B], K)
    bitmap = torch.zeros(ops.bitmap_words(N), dtype=torch.int32, device='cuda')
    ts32 = torch.zeros(B, device='cuda')
    nn_, ne_, nt_, _ = ops.find_recent(c, gu.dev(np.concatenate([src, dst, neg])), gu.dev(ts, torch.float64), K,
                                       ts_period=B, want_dirs=False, ts32_out=ts32, bitmap=bitmap)
    assert np.array_equal(gu.cpu(nn_), b.neigh_nids) and np.array_equal(gu.cpu(ne_), b.neigh_eids)
    assert np.array_equal(gu.cpu(nt_), b.neigh_ts) and np.array_equal(gu.cpu(ts32), b.ts)
    # compaction: involved / local_index / outdated
    has_msg = torch.zeros(N, dtype=torch.uint8, device='cuda')
    pend = b.involved[::3]
    has_msg[gu.dev(pend)] = 1
    cap = 3 * B * (K + 1)
    involved = torch.zeros(cap, dtype=torch.int64, device='cuda')
    outdated = torch.zeros(cap, dtype=torch.int64, device='cuda')
    local_index = torch.zeros(N, dtype=torch.int64, device='cuda')
    gru_row = torch.full((N,), -7, dtype=torch.int32, device='cuda')
    counts = torch.zeros(4, dtype=torch.int32, device='cuda')
    ops.compact_involved(bitmap, N, involved, counts, has_msg=has_msg, local_index=local_index, outdated=outdated,
                         gru_row=gru_row)
    U, Oc = int(counts[0]), int(counts[1])
    assert np.array_equal(gu.cpu(involved[:U]), b.involved)
    assert np.array_equal(gu.cpu(local_index), b.local_index)
    assert np.array_equal(gu.cpu(outdated[:Oc]), pend)
    gr = gu.cpu(gru_row)
    assert np.array_equal(gr[pend], np.arange(len(pend))) and (gr[np.setdiff1d(b.involved, pend)] == -1).all()
    assert int(bitmap.abs().sum()) == 0
    # hit windows
    for center, rows, want in ((src, nn_[B:2 * B], b.src_hits), (dst, nn_[:B], b.dst_hits),
                               (src, nn_[2 * B:], b.neg_src_hits), (neg, nn_[:B], b.neg_dst_hits)):
        assert np.array_equal(gu.cpu(ops.hit_window(gu.dev(center), rows.contiguous())), want)


def test_golden_history_known_answers(gu):
    for name in CASES:
        g = Golden(name)
        c = gu.device_csr(g.src, g.dst, g.ts, g.eids, g.N)
        z = g.z
        got = ops.find_recent(c, gu.dev(z['kat_hist_q_nids']), gu.dev(z['kat_hist_q_ts'], torch.float64), 7)
        for a, key in zip(got, ('kat_hist_nids', 'kat_hist_eids', 'kat_hist_ts', 'kat_hist_dirs')):
            assert np.array_equal(gu.cpu(a), z[key]), (name, key)


# ------------------------------------------------------------------ a8 / a22
@pytest.mark.parametrize('n,dtype', [(1, np.float32), (60, np.float32), (400, np.float32), (400, np.float64),
                                     (2048, np.float32), (2049, np.float32), (20000, np.float64)])
def test_select_latest_matches_oracle(gu, n, dtype):
    rng = np.random.RandomState(n)
    n_nodes = 5000
    ids = rng.randint(0, max(2, min(n_nodes, n // 3 + 2)), n).astype(np.int64)
    ts = np.floor(rng.uniform(0, 25, n)).astype(dtype)      # many ties
    if dtype == np.float64:
        ts = ts + 1e-9 * rng.randint(0, 3, n)                # distinct in f64, equal in f32
    u, ix = O.select_latest_scan(ids, ts)
    scratch = ops.SelectScratch(n_nodes, 'cuda')
    winner, du, dix, cnt = ops.select_latest(gu.dev(ids), gu.dev(ts), scratch)
    c = int(cnt)
    assert c == len(u)
    assert np.array_equal(gu.cpu(du[:c]), u) and np.array_equal(gu.cpu(dix[:c]), ix)
    w = np.zeros(n, dtype=np.uint8)
    w[ix] = 1
    assert np.array_equal(gu.cpu(winner), w)
    assert int(scratch.slot_ts.abs().sum()) == 0 and int(scratch.slot_pos.abs().sum()) == 0
    assert int(scratch.bitmap.abs().sum()) == 0
    # flags only (engine form)
    winner2, _, _, _ = ops.select_latest(gu.dev(ids), gu.dev(ts), scratch, want_unique=False)
    assert np.array_equal(gu.cpu(winner2), w)
    assert int(scratch.slot_ts.abs().sum()) == 0 and int(scratch.slot_pos.abs().sum()) == 0


def test_select_latest_golden_and_repeat_semantics(gu):
    z = Golden(CASES[0]).z
    _, du, dix, cnt = ops.select_latest(gu.dev(z['kat_sl_ids']), gu.dev(z['kat_sl_ts']))
    c = int(cnt)
    assert np.array_equal(gu.cpu(du[:c]), z['kat_sl_unique']) and np.array_equal(gu.cpu(dix[:c]), z['kat_sl_index'])
    # ts.repeat(2): ts shorter than ids
    rng = np.random.RandomState(1)
    src, dst = rng.randint(1, 30, 100), rng.randint(30, 40, 100)
    ts = np.floor(np.sort(rng.uniform(0, 40, 100))).astype(np.float32)
    u, ix = O.select_latest(np.concatenate([src, dst]), np.tile(ts, 2))
    _, du, dix, cnt = ops.select_latest(gu.dev(np.concatenate([src, dst])), gu.dev(ts))
    c = int(cnt)
    assert np.array_equal(gu.cpu(du[:c]), u) and np.array_equal(gu.cpu(dix[:c]), ix)


def test_anonymized_reindex(gu):
    z = Golden(CASES[0]).z
    assert np.array_equal(gu.cpu(ops.anonymized_reindex(gu.dev(z['kat_anon_in']))), z['kat_anon_out'])
    rng = np.random.RandomState(0)
    h = rng.randint(0, 9, (300, 40)).astype(np.int64)
    h[:, :10][rng.rand(300, 10) < 0.5] = 0
    assert np.array_equal(gu.cpu(ops.anonymized_reindex(gu.dev(h))), O.anonymized_reindex(h))
    ex = np.array([[0, 0, 5, 7, 5], [3, 4, 3, 3, 9]], dtype=np.int64)     # SURVEY Q14
    assert gu.cpu(ops.anonymized_reindex(gu.dev(ex))).tolist() == [[0, 0, 1, 2, 1], [2, 3, 2, 2, 1]]


# ------------------------------------------------------------------ a10 / a11
def test_time_encode_and_memory_rows(gu):
    d = 172
    W = perturb_biases(random_weights(d, d))
    w, b = W['time_encoder.basis_freq'], W['time_encoder.phase']
    ts = torch.cat([torch.zeros(3), torch.rand(500) * 2.6e6, torch.tensor([2.678e6, 1.0, 86400.])])
    got = ops.time_encode(gu.dev(ts), gu.dev(w), gu.dev(b))
    assert_close(gu.cpu(got), O.time_encode(ts, w, b).numpy(), TOL, 'time_encode')
    table = torch.randn(1000, d)
    tst = torch.rand(1000)
    ids = torch.randint(0, 1000, (333,))
    v, t = ops.gather_rows(gu.dev(table), gu.dev(ids), gu.dev(tst))
    assert torch.equal(v.cpu(), table[ids]) and torch.equal(t.cpu(), tst[ids])
    dt, dts = gu.dev(table), gu.dev(tst)
    uid = torch.randperm(1000)[:200]
    vals, nts = torch.randn(200, d), tst[uid] + 1
    err = torch.zeros(1, dtype=torch.int32, device='cuda')
    act = torch.zeros(1000, dtype=torch.uint8, device='cuda')
    ops.scatter_rows(dt, gu.dev(uid), gu.dev(vals), ts_table=dts, ts=gu.dev(nts), active=act, check=True, err_flags=err)
    table[uid], tst[uid] = vals, nts
    assert torch.equal(dt.cpu(), table) and torch.equal(dts.cpu(), tst) and int(err) == 0
    assert int(act.sum()) == 200
    ops.scatter_rows(dt, gu.dev(uid[:5]), gu.dev(vals[:5]), ts_table=dts, ts=gu.dev(nts[:5] - 5), check=True,
                     err_flags=err)
    assert int(err) == 1       # "not allowed to modify past memory"


# ------------------------------------------------------------------ a13: GRU
@pytest.mark.parametrize('d,de,n', [(172, 172, 1426), (172, 172, 1), (100, 4, 65), (100, 100, 64), (10, 4, 37),
                                    (12, 8, 200), (8, 8, 63)])
def test_gru_update_matches_oracle(gu, d, de, n):
    W = random_weights(d, de, seed=d + n)
    c = 'right_mem_updater.cell.'
    M = 3 * d + de
    g = torch.Generator().manual_seed(n)
    x, h = torch.randn(n, M, generator=g), torch.randn(n, d, generator=g)
    want = O.gru_cell(x, h, W[c + 'weight_ih'], W[c + 'weight_hh'], W[c + 'bias_ih'], W[c + 'bias_hh'])
    pack = ops.GruPack(*(gu.dev(W[c + k]) for k in ('weight_ih', 'weight_hh', 'bias_ih', 'bias_hh')))
    got = ops.gru_update(pack, node_ids=None, x_table=gu.dev(x), h_table=gu.dev(h), n_rows=n)
    assert_close(gu.cpu(got), want.numpy(), TOL, f'gru dense d={d}')
    # gathered form with a device-side count
    N = 3 * n + 5
    xt, ht = torch.randn(N, M, generator=g), torch.randn(N, d, generator=g)
    ids = torch.randperm(N, generator=g)[:n]
    want = O.gru_cell(xt[ids], ht[ids], W[c + 'weight_ih'], W[c + 'weight_hh'], W[c + 'bias_ih'], W[c + 'bias_hh'])
    ids_pad = torch.cat([ids, torch.zeros(100, dtype=torch.int64)])
    out = torch.full((n + 100, d), 7.0, device='cuda')
    cnt = torch.tensor([n], dtype=torch.int32, device='cuda')
    ops.gru_update(pack, node_ids=gu.dev(ids_pad), x_table=gu.dev(xt), h_table=gu.dev(ht), n_rows=n + 100, out=out,
                   count=cnt)
    assert_close(gu.cpu(out[:n]), want.numpy(), TOL, f'gru gathered d={d}')
    assert float(out[n:].min()) == 7.0 and float(out[n:].max()) == 7.0


# ------------------------------------------------------------------ a15/a16: attention
@pytest.mark.parametrize('d,de,n,k,H', [(172, 172, 600, 10, 2), (172, 172, 5, 10, 2), (100, 4, 300, 10, 2),
                                        (100, 100, 151, 10, 2), (10, 4, 75, 5, 2), (12, 8, 90, 5, 2),
                                        (8, 8, 120, 5, 4), (16, 6, 33, 3, 1)])
def test_temporal_attention_dense_matches_oracle(gu, d, de, n, k, H):
    W = perturb_biases(random_weights(d, de, seed=n))
    g = torch.Generator().manual_seed(n)
    qx, qt = torch.randn(n, d, generator=g), torch.randn(n, d, generator=g)
    kx, ky, kt = torch.randn(n, k, d, generator=g), torch.randn(n, k, de, generator=g), torch.randn(n, k, d, generator=g)
    mask = torch.rand(n, k, generator=g) < 0.3
    mask[::7] = True                     # rows where every slot is padding
    mask[1::7, :-1] = True               # exactly one live slot
    p = 'temporal_embedding_fn.fns.0.'
    want = O.temporal_attention(W, p, H, qx, qt, kx, ky, kt, mask)
    pack = ops.AttnPack(d, de, 'cuda', H)
    m = p + 'mha_fn.'
    pack.refresh(*(gu.dev(W[x]) for x in (m + 'q_proj_weight', m + 'k_proj_weight', m + 'v_proj_weight',
                                            m + 'in_proj_bias', m + 'out_proj.weight', m + 'out_proj.bias',
                                            p + 'merger.fc1.weight', p + 'merger.fc1.bias', p + 'merger.fc2.weight',
                                            p + 'merger.fc2.bias', 'time_encoder.basis_freq', 'time_encoder.phase')))
    got = ops.temporal_attention_dense(pack, H, gu.dev(qx), gu.dev(qt), gu.dev(kx), gu.dev(ky), gu.dev(kt),
                                       gu.dev(mask))
    assert_close(gu.cpu(got), want.numpy(), TOL, f'attention dense d={d} de={de} n={n}')


def _dense_attention(gu, d, de, n, k, H, seed):
    W = perturb_biases(random_weights(d, de, seed=seed))
    g = torch.Generator().manual_seed(seed)
    qx, qt = torch.randn(n, d, generator=g), torch.randn(n, d, generator=g)
    kx, ky, kt = torch.randn(n, k, d, generator=g), torch.randn(n, k, de, generator=g), torch.randn(n, k, d, generator=g)
    mask = torch.rand(n, k, generator=g) < 0.3
    mask[::7] = True
    mask[1::7, :-1] = True
    mask[2::7, 1:] = True                # only the first slot live
    p = 'temporal_embedding_fn.fns.0.'
    pack = ops.AttnPack(d, de, 'cuda', H)
    m = p + 'mha_fn.'
    pack.refresh(*(gu.dev(W[x]) for x in (m + 'q_proj_weight', m + 'k_proj_weight', m + 'v_proj_weight',
                                            m + 'in_proj_bias', m + 'out_proj.weight', m + 'out_proj.bias',
                                            p + 'merger.fc1.weight', p + 'merger.fc1.bias', p + 'merger.fc2.weight',
                                            p + 'merger.fc2.bias', 'time_encoder.basis_freq', 'time_encoder.phase')))
    got = lambda: ops.temporal_attention_dense(pack, H, gu.dev(qx), gu.dev(qt), gu.dev(kx), gu.dev(ky), gu.dev(kt),
                                               gu.dev(mask))
    return got, lambda: O.temporal_attention(W, p, H, qx, qt, kx, ky, kt, mask)


@pytest.mark.parametrize('H,d,de', [(1, 16, 6), (2, 16, 6), (4, 16, 6), (3, 12, 8)])
@pytest.mark.parametrize('k', [1, 20, 32, 33, 64])
def test_temporal_attention_dense_matches_oracle_at_every_k(gu, k, H, d, de):
    """K up to ATT_MAXK = 64 (past 32 the softmax holds two values per lane); H = 3 is the generic (HT = 0) launch."""
    got, want = _dense_attention(gu, d, de, 90, k, H, seed=k * 10 + H)
    assert_close(gu.cpu(got()), want().numpy(), TOL, f'attention dense k={k} H={H}')


def test_temporal_attention_dense_at_k64_baseline_width_and_k65_refusal(gu):
    """d = de = 172 at K = 64: the largest shared-memory footprint the kernel takes (about 135 KB, under its 200 KB
    refusal); K = 65 is refused."""
    got, want = _dense_attention(gu, 172, 172, 40, 64, 2, seed=5)
    assert_close(gu.cpu(got()), want().numpy(), TOL, 'attention dense k=64 d=172')
    got, _ = _dense_attention(gu, 16, 6, 10, 65, 2, seed=6)
    with pytest.raises(TigerLibraryError, match='invalid argument'):
        got()


# ------------------------------------------------------------------ step 7: scorer
@pytest.mark.parametrize('hit_type', ['bin', 'none'])
@pytest.mark.parametrize('d,B,k', [(172, 200, 10), (100, 37, 10), (10, 25, 5)])
def test_link_score_folded_matches_oracle(gu, d, B, k, hit_type):
    """The folded scorer: the batch nodes' attention (gather form) with the score fold and the left write-back
    attached writes pq, tiger_link_score_folded scores the pairs from it."""
    W = perturb_biases(random_weights(d, d, seed=B))
    g = torch.Generator().manual_seed(B)
    N, E, H = 40, 300, 2
    rows, efeats = torch.randn(N, d, generator=g), torch.randn(E, d, generator=g)
    src, dst, neg = (torch.randint(1, N, (B,), generator=g) for _ in range(3))
    centers = torch.cat([src, dst, neg])
    neigh = torch.randint(0, N, (3 * B, k), generator=g)            # id 0: padding slot
    neigh[::9] = 0                                                  # rows without a live slot
    neigh_e = torch.randint(0, E, (3 * B, k), generator=g)
    ts = torch.rand(B, generator=g) * 100 + 100
    neigh_ts = ts.repeat(3)[:, None] - torch.rand(3 * B, k, generator=g) * 100
    p = 'temporal_embedding_fn.fns.0.'
    tw, tb = W['time_encoder.basis_freq'], W['time_encoder.phase']
    z = O.temporal_attention(W, p, H, rows[centers], O.time_encode(torch.zeros(3 * B), tw, tb), rows[neigh],
                             efeats[neigh_e], O.time_encode(ts.repeat(3)[:, None] - neigh_ts, tw, tb), neigh == 0)
    x, y, ny = z.reshape(3, B, d)
    emb = W['hit_embedding.weight'] if hit_type == 'bin' else torch.zeros(2, d)
    flag = lambda c, rows: (c[:, None] == rows).any(1).long()
    xp, yp = x + emb[flag(src, neigh[B:2 * B])], y + emb[flag(dst, neigh[:B])]
    xn, yn = x + emb[flag(src, neigh[2 * B:])], ny + emb[flag(neg, neigh[:B])]
    sw = [W['score_fn.' + n] for n in ('fc1.weight', 'fc1.bias', 'fc2.weight', 'fc2.bias')]
    ps, ns = O.merge_layer(xp, yp, *sw).squeeze(1), O.merge_layer(xn, yn, *sw).squeeze(1)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(torch.cat([ps, ns]),
                                                                torch.cat([torch.ones(B), torch.zeros(B)]))
    pack = ops.AttnPack(d, d, 'cuda', H)
    m = p + 'mha_fn.'
    pack.refresh(*(gu.dev(W[n]) for n in (m + 'q_proj_weight', m + 'k_proj_weight', m + 'v_proj_weight',
                                            m + 'in_proj_bias', m + 'out_proj.weight', m + 'out_proj.bias',
                                            p + 'merger.fc1.weight', p + 'merger.fc1.bias', p + 'merger.fc2.weight',
                                            p + 'merger.fc2.bias', 'time_encoder.basis_freq', 'time_encoder.phase')))
    fold, pq = ops.ScoreFold(d, 'cuda'), torch.zeros(3 * B, 2 * d, device='cuda')
    fold.refresh(*(gu.dev(t) for t in sw), gu.dev(W[p + 'merger.fc2.weight']), gu.dev(W[p + 'merger.fc2.bias']),
                 gu.dev(emb) if hit_type == 'bin' else None)
    d_centers, d_ts = gu.dev(centers), gu.dev(ts)
    pos = d_centers[:2 * B]
    winner = ops.select_latest(pos, d_ts, want_unique=False, want_count=False)[0]
    left_vals, left_ts = torch.zeros(N, d, device='cuda'), torch.zeros(N, device='cuda')
    left_active = torch.zeros(N, dtype=torch.uint8, device='cuda')
    pack.attach_score_fold(fold, pq)
    pack.attach_left_writeback(pos, winner, d_ts, left_vals, left_ts, left_active)
    out = ops.temporal_attention(pack, H, d_centers, d_ts, gu.dev(neigh), gu.dev(neigh_e), gu.dev(neigh_ts),
                                 rows_a=None, rows_b=gu.dev(rows), sel=torch.arange(N, dtype=torch.int32, device='cuda'),
                                 nfeats=None, efeats=gu.dev(efeats))
    assert_close(gu.cpu(out), z.numpy(), TOL, 'attention')
    w = winner.bool()
    assert torch.equal(left_vals[pos[w]], out[:2 * B][w]), 'fused left write-back'
    for _ in range(2):                    # twice: the done-counter must reset itself
        scores, dl = ops.link_score_folded(fold, pq, gu.dev(src), gu.dev(dst), gu.dev(neg),
                                           gu.dev(neigh) if hit_type == 'bin' else None)
        assert_close(gu.cpu(scores), torch.cat([ps, ns]).numpy(), TOL, 'scores')
        assert_close(gu.cpu(dl), loss.reshape(1).numpy(), TOL, 'loss')


# ------------------------------------------------------------------ restarter-path GEMM
@pytest.mark.parametrize('m,n,k', [(1, 7, 5), (54, 172, 860), (300, 1720, 860), (2200, 130, 54), (33, 65, 17)])
def test_sgemm_nt_matches_torch(gu, m, n, k):
    g = torch.Generator().manual_seed(m * 1000 + n)
    a = torch.randn(m, k, generator=g)
    w = torch.randn(n, k, generator=g) / k ** 0.5
    b = torch.randn(n, generator=g)
    for relu in (False, True):
        ref = a.double() @ w.double().t() + b.double()
        ref = torch.relu(ref) if relu else ref
        out = torch.empty(m, n, device='cuda')
        ops.sgemm_nt(gu.dev(a), gu.dev(w), gu.dev(b), out, relu=relu)
        assert_close(gu.cpu(out), ref.numpy(), 2e-6, f'sgemm {m}x{n}x{k}')


def test_sgemm_nt_device_count_and_slices(gu):
    g = torch.Generator().manual_seed(0)
    a = torch.randn(400, 96, generator=g)
    w = torch.randn(80, 96, generator=g)
    big = torch.full((400, 200), -7.0, device='cuda')
    count = torch.tensor([9], dtype=torch.int32, device='cuda')
    # rows = count * rows_per_count = 36; output into a column slice of a wider buffer; K = first 50 columns
    ops.sgemm_nt(gu.dev(a), gu.dev(w), None, big[:, 40:120], k_dim=50, count=count, rows_per_count=4)
    ref = a[:36, :50].double() @ w[:, :50].double().t()
    assert_close(gu.cpu(big[:36, 40:120]), ref.numpy(), 2e-6, 'sliced')
    rest = gu.cpu(big)
    assert (rest[36:] == -7).all() and (rest[:, :40] == -7).all() and (rest[:, 120:] == -7).all()


# ------------------------------------------------------------------ a21: SeqRestarter.forward
@pytest.mark.parametrize('name', [c for c in CASES if c.startswith('seq')])
def test_seq_restarter_matches_reference_golden(gu, name):
    """Restarter called with the collated restart data (training-target path, tiger.py:576-581)."""
    g = Golden(name)
    de = g.efeats.shape[1] if g.efeats is not None else g.dim
    op = ops.SeqRestarterOp(g.dim, de, g.hist_len, g.n_heads, 2 * g.bs, 'cuda')
    op.set_weights(g.W)
    nf = None if g.nfeats is None else gu.dev(g.nfeats, torch.float32)
    ef = None if g.efeats is None else gu.dev(g.efeats, torch.float32)
    for ib in range(g.n_batches):
        nids = g.b(ib, 'r_nids')
        n = len(nids)
        hist = tuple(gu.dev(g.b(ib, k)) for k in ('r_hist_nids', 'r_hist_eids', 'r_hist_ts', 'r_hist_dirs', 'r_anon'))
        hl, hr, pt = op.forward(gu.dev(nids), n, nf, ef, hist=hist)
        assert_close(gu.cpu(hl), g.b(ib, 'surrogate_left'), TOL, f'{name} b{ib} left')
        assert_close(gu.cpu(hr), g.b(ib, 'surrogate_right'), TOL, f'{name} b{ib} right')
        assert np.array_equal(gu.cpu(pt), g.b(ib, 'r_hist_ts')[:, -1])


@pytest.mark.parametrize('n_pick', [70, 30, 1])       # > / <= SeqRestarterOp.tail_rows: tensor-core products / fused tail
@pytest.mark.parametrize('d,de,L,with_nf', [(172, 172, 40, False), (100, 4, 40, False), (24, 10, 64, True)])
def test_seq_restarter_matches_oracle(gu, d, de, L, with_nf, n_pick):
    """Restarter with computation_graph=None: history looked up on the device CSR (restart path)."""
    st = make_stream(StreamShape('s', 150, 25, 8000, de, None, horizon=5000.), seed=6, nfeat_dim=d if with_nf else 0)
    N = st.n_nodes
    W = perturb_biases(random_weights(d, de, n_nodes=N, restarter='seq', hist_len=L, seed=3))
    graph = O.OracleGraph(st.src, st.dst, st.ts, st.eids, n_nodes=N)
    model = O.OracleTIGER(W, graph, N, d, st.efeats, st.nfeats, restarter='seq', hist_len=L)
    rng = np.random.RandomState(0)
    nids = np.concatenate([[0], rng.choice(np.arange(1, N), n_pick, replace=False)]).astype(np.int64)
    t = np.float32(3000.0)
    ref_l, ref_r, ref_pt = model.restarter_forward(nids, np.full(len(nids), t, dtype=np.float32))
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    op = ops.SeqRestarterOp(d, de, L, 2, 128, 'cuda')
    op.set_weights(W)
    count = torch.tensor([len(nids)], dtype=torch.int32, device='cuda')
    dn = torch.zeros(128, dtype=torch.int64, device='cuda')
    dn[:len(nids)] = gu.dev(nids)
    ops.min_time(gu.dev(np.array([5000., 3000., 4000.], dtype=np.float32)), op.tmin)
    assert float(op.tmin) == 3000.0
    op.history(csr, dn, op.tmin, 128, ts_period=1, count=count)
    hn, he_, ht, hd = graph.get_history(nids, np.full(len(nids), 3000.0), L)
    n = len(nids)
    assert np.array_equal(gu.cpu(op.hist_nids[:n]), hn) and np.array_equal(gu.cpu(op.hist_dirs[:n]), hd)
    assert np.array_equal(gu.cpu(op.anony[:n]), O.anonymized_reindex(hn))
    hl, hr, pt = op.forward(dn, 128, None if st.nfeats is None else gu.dev(st.nfeats, torch.float32),
                            gu.dev(st.efeats, torch.float32), count=count)
    assert_close(gu.cpu(hl[:n]), ref_l.numpy(), TOL, 'h_left')
    assert_close(gu.cpu(hr[:n]), ref_r.numpy(), TOL, 'h_right')
    assert np.array_equal(gu.cpu(pt[:n]), ref_pt.numpy())
    # rows past the count are not written by either route
    assert op.tail_rows == 64
    hl_a, hr_a = hl.clone(), hr.clone()
    op.tail_rows = 0
    op.h_left.fill_(-3.0), op.h_right.fill_(-3.0)
    hl_b, hr_b, _ = op.forward(dn, 128, None if st.nfeats is None else gu.dev(st.nfeats, torch.float32),
                               gu.dev(st.efeats, torch.float32), count=count)
    assert_close(gu.cpu(hl_a[:n]), gu.cpu(hl_b[:n]), TOL, 'tail vs products, left')
    assert_close(gu.cpu(hr_a[:n]), gu.cpu(hr_b[:n]), TOL, 'tail vs products, right')
    assert (gu.cpu(hl_b[n:]) == -3.0).all() and (gu.cpu(hr_b[n:]) == -3.0).all()
    op.tail_rows = 64
    op.h_left.fill_(-3.0), op.h_right.fill_(-3.0)
    hl_c, hr_c, _ = op.forward(dn, 128, None if st.nfeats is None else gu.dev(st.nfeats, torch.float32),
                               gu.dev(st.efeats, torch.float32), count=count)
    assert (gu.cpu(hl_c[n:]) == -3.0).all() and (gu.cpu(hr_c[n:]) == -3.0).all()
    assert torch.equal(hl_c[:n], hl_a[:n]) and torch.equal(hr_c[:n], hr_a[:n])


# ------------------------------------------------------------------ packed-weight tensor-core GEMM
@pytest.mark.parametrize('m,n,k', [(1, 7, 5), (54, 172, 860), (600, 1040, 344), (600, 172, 1205), (2200, 130, 54)])
def test_sgemm_nt_packed_matches_torch(gu, m, n, k):
    g = torch.Generator().manual_seed(m * 1000 + n)
    a = torch.randn(m, k, generator=g)
    w = torch.randn(n, k, generator=g) / k ** 0.5
    b = torch.randn(n, generator=g)
    pack = ops.WeightPack(gu.dev(w), m_rows_hint=m)
    for relu in (False, True):
        ref = a.double() @ w.double().t() + b.double()
        ref = torch.relu(ref) if relu else ref
        out = torch.full((m, n), float('nan'), device='cuda')
        ops.sgemm_nt_packed(gu.dev(a), pack, gu.dev(b), out, relu=relu)
        assert_close(gu.cpu(out), ref.numpy(), 2e-6, f'packed gemm {m}x{n}x{k}')


@pytest.mark.gpu
@pytest.mark.parametrize('m,n,k', [(7, 40, 172), (600, 704, 172), (333, 96, 100)])
def test_sgemm_nt_packed_gather_matches_torch(gu, m, n, k):
    """A rows looked up by the producers: rows_b[sel[id]] if sel[id] >= 0 else rows_a[id], + add_rows[id]."""
    g = torch.Generator().manual_seed(m + n)
    n_nodes, n_b = 500, 90
    rows_a = torch.randn(n_nodes, k, generator=g)
    rows_b = torch.randn(n_b, k, generator=g)
    add = torch.randn(n_nodes, k, generator=g)
    sel = torch.full((n_nodes,), -1, dtype=torch.int32)
    picked = torch.randperm(n_nodes, generator=g)[:n_b]
    sel[picked] = torch.arange(n_b, dtype=torch.int32)
    ids = torch.randint(0, n_nodes, (m,), generator=g)
    w = torch.randn(n, k, generator=g) / k ** 0.5
    b = torch.randn(n, generator=g)
    pack = ops.WeightPack(gu.dev(w), m_rows_hint=m)
    for with_add in (False, True):
        for sel_dt in (torch.int32, torch.int64):
            x = torch.where((sel[ids] >= 0)[:, None], rows_b[sel[ids].clamp(min=0).long()], rows_a[ids])
            if with_add:
                x = x + add[ids]
            ref = x.double() @ w.double().t() + b.double()
            out = torch.full((m, n), float('nan'), device='cuda')
            ops.sgemm_nt_packed_gather(gu.dev(ids), gu.dev(sel.to(sel_dt)), gu.dev(rows_a), gu.dev(rows_b),
                                       gu.dev(add) if with_add else None, pack, gu.dev(b), out)
            assert_close(gu.cpu(out), ref.numpy(), 2e-6, f'gather gemm {m}x{n}x{k} add={with_add}')


@pytest.mark.gpu
@pytest.mark.parametrize('m,n,k,parts', [(600, 172, 1205, 4), (130, 40, 300, 3), (5, 172, 64, 4), (700, 96, 2048, 8)])
def test_sgemm_nt_packed_splitk_fused_matches_torch(gu, m, n, k, parts):
    g = torch.Generator().manual_seed(m + n + k)
    a = torch.randn(m, k, generator=g)
    w = torch.randn(n, k, generator=g) / k ** 0.5
    b = torch.randn(n, generator=g)
    pack = ops.WeightPack(gu.dev(w), bn=32)
    for relu in (False, True):
        ref = a.double() @ w.double().t() + b.double()
        ref = torch.relu(ref) if relu else ref
        out = torch.full((m, n), float('nan'), device='cuda')
        ops.sgemm_nt_packed_splitk_fused(gu.dev(a), pack, gu.dev(b), out, parts, relu=relu)
        assert_close(gu.cpu(out), ref.numpy(), 2e-6, f'cluster split-K gemm {m}x{n}x{k}/{parts}')
        out2 = torch.full((m, n), float('nan'), device='cuda')
        ops.sgemm_nt_packed_splitk_fused(gu.dev(a), pack, gu.dev(b), out2, parts, relu=relu)
        assert torch.equal(out, out2)       # part order is fixed: bit-identical from run to run


@pytest.mark.gpu
@pytest.mark.parametrize('d', [172, 100, 37])
def test_large_row_sets_take_the_bulk_copy_path(gu, d):
    """>= 64 k rows: gather / scatter / write-backs move rows with one bulk copy per row through shared memory
    (16-byte aligned rows; d = 37 falls back to the register path) - same results as torch indexing."""
    g = torch.Generator().manual_seed(d)
    N, n = 90000, 70001
    table = torch.randn(N, d, generator=g).cuda()
    ts_table = torch.rand(N, generator=g).cuda()
    ids = torch.randperm(N, generator=g)[:n].cuda()
    out, out_ts = ops.gather_rows(table, ids, ts_table)
    assert torch.equal(out, table[ids]) and torch.equal(out_ts, ts_table[ids])
    # scatter (unique ids: a permutation prefix)
    vals = torch.randn(n, d, generator=g).cuda()
    ts = (torch.rand(n, generator=g) + 2).cuda()
    t2, tt2 = table.clone(), ts_table.clone()
    active = torch.zeros(N, dtype=torch.uint8, device='cuda')
    ops.scatter_rows(t2, ids, vals, ts_table=tt2, ts=ts, active=active)
    ref = table.clone(); ref[ids] = vals
    reft = ts_table.clone(); reft[ids] = ts
    assert torch.equal(t2, ref) and torch.equal(tt2, reft) and int(active.sum()) == n
    # left write-back: positions [src ; dst] of a batch, winners only
    B = n // 2
    pos = ids[:2 * B].contiguous()
    winner = (torch.rand(2 * B, generator=g) < 0.7).to(torch.uint8).cuda()
    h_left = torch.randn(2 * B, d, generator=g).cuda()
    bts = (torch.rand(B, generator=g) + 5).cuda()
    lv, lt = table.clone(), ts_table.clone()
    la = torch.zeros(N, dtype=torch.uint8, device='cuda')
    ops.left_writeback(pos, B, winner, h_left, d, bts, lv, lt, la)
    w = winner.bool()
    ref = table.clone(); ref[pos[w]] = h_left[w]
    reft = ts_table.clone(); reft[pos[w]] = bts.repeat(2)[w]
    assert torch.equal(lv, ref) and torch.equal(lt, reft) and torch.equal(la.bool(), torch.zeros(N, dtype=torch.bool, device='cuda').index_fill_(0, pos[w], True))
    # right write-back: winners with a pending message take their GRU row
    has_msg = (torch.rand(N, generator=g) < 0.8).to(torch.uint8).cuda()
    gru_row = torch.full((N,), -1, dtype=torch.int32, device='cuda')
    pend_nodes = torch.nonzero(has_msg).flatten()
    gru_row[pend_nodes] = torch.arange(pend_nodes.numel(), dtype=torch.int32, device='cuda')
    h_new = torch.randn(pend_nodes.numel(), d, generator=g).cuda()
    msg_ts = (ts_table + 1).contiguous()
    rv, rt = table.clone(), ts_table.clone()
    ra = torch.zeros(N, dtype=torch.uint8, device='cuda')
    hm = has_msg.clone()
    ops.right_writeback(pos, winner, gru_row, h_new, d, rv, rt, ra, msg_ts, hm)
    sel = w & has_msg[pos].bool()
    nodes = pos[sel]
    ref = table.clone(); ref[nodes] = h_new[gru_row[nodes].long()]
    reft = ts_table.clone(); reft[nodes] = msg_ts[nodes]
    refm = has_msg.clone(); refm[nodes] = 0
    assert torch.equal(rv, ref) and torch.equal(rt, reft) and torch.equal(hm, refm)


@pytest.mark.parametrize('n', [2049, 5000, 70000])
def test_select_latest_large_flags_only_count(n):
    """flags-only mode (no ordered output) of the large-n path must still report the number of distinct ids."""
    rng = np.random.RandomState(n)
    n_nodes = 3000
    ids = rng.randint(1, n_nodes, n)
    ts = np.floor(rng.uniform(0, 50, n))
    scratch = ops.SelectScratch(n_nodes, 'cuda')
    winner, _, _, count = ops.select_latest(torch.from_numpy(ids).cuda(), torch.from_numpy(ts).cuda(), scratch,
                                            want_unique=False)
    u, ix = O.select_latest(ids, ts)
    assert int(count) == len(u)
    w = np.zeros(n, dtype=np.uint8)
    w[ix] = 1
    assert np.array_equal(winner.cpu().numpy(), w)
    assert int(scratch.slot_ts.abs().sum()) == 0 and int(scratch.slot_pos.abs().sum()) == 0


# ------------------------------------------------------------------ general tensor-core product (training step)
@pytest.mark.parametrize('m,n,k', [(600, 172, 344), (37, 5, 19), (1900, 516, 688), (128, 128, 16), (1, 1, 1)])
@pytest.mark.parametrize('ta,tw', [(False, False), (False, True), (True, True), (True, False)])
def test_sgemm_ex_all_operand_layouts(m, n, k, ta, tw):
    g = torch.Generator(device='cuda').manual_seed(m * 7 + n)
    A = torch.randn((k, m) if ta else (m, k), device='cuda', generator=g)
    W = torch.randn((k, n) if tw else (n, k), device='cuda', generator=g)
    bias = torch.randn(n, device='cuda', generator=g)
    out = torch.empty(m, n, device='cuda')
    ops.sgemm_ex(A, W, out, m=m, n=n, k=k, trans_a=ta, trans_w=tw, bias=bias, relu=True, alpha=0.5)
    opA = (A.t() if ta else A).double()
    opW = (W.t() if tw else W).double()
    want = torch.relu(0.5 * (opA @ opW.t() + bias.double()))
    assert_close(out.cpu().numpy(), want.cpu().numpy(), 2e-6, f'sgemm_ex {m}x{n}x{k} {ta}{tw}')


@pytest.mark.parametrize('rows,count', [(6600, 1900), (6600, 0), (300, 300), (70000, 11200)])
def test_sgemm_ex_weight_gradient_accumulates_with_device_count(rows, count):
    """dW += dY[:count]^T X[:count]: transposed operands, reduction length from device memory, split K, atomic
    accumulation on top of what the buffer already holds."""
    g = torch.Generator(device='cuda').manual_seed(rows + count)
    n_out, n_in = 516, 172
    dY = torch.randn(rows, n_out, device='cuda', generator=g)
    X = torch.randn(rows, n_in, device='cuda', generator=g)
    dW = torch.randn(n_out, n_in, device='cuda', generator=g)
    base = dW.clone()
    cnt = torch.tensor([count], dtype=torch.int32, device='cuda')
    ops.sgemm_ex(dY, X, dW, m=n_out, n=n_in, k=rows, trans_a=True, trans_w=True, accumulate=True,
                 k_parts=max(1, min(64, (rows + 511) // 512)), k_count=cnt)
    want = base.double() + dY[:count].double().t() @ X[:count].double()
    assert_close(dW.cpu().numpy(), want.cpu().numpy(), 2e-6, f'wgrad rows={rows} count={count}')


def test_sgemm_nt_capacity_launch_is_persistent_and_exact():
    """A launch sized for a large row capacity with a small device-side row count (the seq restarter's case)."""
    g = torch.Generator(device='cuda').manual_seed(3)
    cap, rows, k, n = 264000, 920, 860, 1720
    A = torch.randn(cap, k, device='cuda', generator=g)
    W = torch.randn(n, k, device='cuda', generator=g)
    b = torch.randn(n, device='cuda', generator=g)
    out = torch.zeros(cap, n, device='cuda')
    cnt = torch.tensor([rows // 40], dtype=torch.int32, device='cuda')
    ops.sgemm_nt(A, W, b, out, m_rows=cap, count=cnt, rows_per_count=40)
    want = A[:rows].double() @ W.double().t() + b.double()
    assert_close(out[:rows].cpu().numpy(), want.cpu().numpy(), 2e-6, 'capacity launch')
    assert float(out[rows:rows + 4096].abs().max()) == 0.0


@pytest.mark.parametrize('m,n,k', [(344, 516, 6000), (516, 688, 1355), (100, 12, 37), (1720, 860, 11200)])
def test_sgemm_ex_transposed_operands_match_float64(m, n, k):
    """Transposed operands (the scalar transposed loader): weight gradient with both operands transposed, input
    gradient with only W transposed."""
    g = torch.Generator(device='cuda').manual_seed(k)
    A = torch.randn(k, m, device='cuda', generator=g)
    W = torch.randn(k, n, device='cuda', generator=g)
    want = (A.double().t() @ W.double()).cpu().numpy()
    out = torch.zeros(m, n, device='cuda')
    ops.sgemm_ex(A, W, out, m=m, n=n, k=k, trans_a=True, trans_w=True, accumulate=True, k_parts=(k + 255) // 256)
    assert_close(out.cpu().numpy(), want, 3e-6, f'wgrad {m}x{n}x{k}')
    # dgrad: only W transposed
    dY = torch.randn(600, k if k < 2000 else 344, device='cuda', generator=g)
    Wt = torch.randn(dY.shape[1], n, device='cuda', generator=g)
    out = torch.empty(600, n, device='cuda')
    ops.sgemm_ex(dY, Wt, out, m=600, n=n, k=dY.shape[1], trans_w=True)
    assert_close(out.cpu().numpy(), (dY.double() @ Wt.double()).cpu().numpy(), 3e-6, 'dgrad transposed W')


# ------------------------------------------------------------------ pre-packed TMA-fed product (large GEMMs)
@pytest.mark.parametrize('m,n,k,ta,tw,acc', [
    (11240, 1720, 860, False, False, False),     # seq restarter q/k in-projection
    (11240, 860, 1720, False, True, False),      # its input gradient
    (1720, 860, 11240, True, True, True),        # its weight gradient
    (6000, 344, 516, False, False, False),       # attention k projection
    (344, 516, 6000, True, True, True),          # attention weight gradient
    (300, 130, 70, False, False, False),         # ragged edges, small
])
def test_sgemm_pp_matches_float64(m, n, k, ta, tw, acc, monkeypatch):
    monkeypatch.setattr(ops, 'BIG_GEMM_FLOPS', 0.0)
    g = torch.Generator(device='cuda').manual_seed(m + n)
    A = torch.randn((k, m) if ta else (m, k), device='cuda', generator=g)
    W = torch.randn((k, n) if tw else (n, k), device='cuda', generator=g)
    opA, opW = (A.t() if ta else A).double(), (W.t() if tw else W).double()
    if acc:
        out = torch.randn(m, n, device='cuda', generator=g)
        want = out.double() + 0.5 * (opA @ opW.t())
        ops.sgemm_big(A, W, out, m=m, n=n, k=k, trans_a=ta, trans_w=tw, accumulate=True, k_parts=max(1, k // 256), alpha=0.5)
    else:
        bias = torch.randn(n, device='cuda', generator=g)
        out = torch.empty(m, n, device='cuda')
        want = torch.relu(opA @ opW.t() + bias.double())
        ops.sgemm_big(A, W, out, m=m, n=n, k=k, trans_a=ta, trans_w=tw, bias=bias, relu=True)
    assert_close(out.cpu().numpy(), want.cpu().numpy(), 3e-6, f'sgemm_pp {m}x{n}x{k}')


def test_sgemm_pp_device_counts(monkeypatch):
    """Row count (forward / input gradient) and reduction length (weight gradient) from device memory."""
    monkeypatch.setattr(ops, 'BIG_GEMM_FLOPS', 0.0)
    g = torch.Generator(device='cuda').manual_seed(9)
    cap, L, rows, kdim, n = 400, 40, 281, 860, 1720
    X = torch.randn(cap * L, kdim, device='cuda', generator=g)
    Wt = torch.randn(n, kdim, device='cuda', generator=g)
    cnt = torch.tensor([rows], dtype=torch.int32, device='cuda')
    out = torch.zeros(cap * L, n, device='cuda')
    ops.sgemm_big(X, Wt, out, m=cap * L, n=n, k=kdim, m_count=cnt, rows_per_count=L)
    want = X[:rows * L].double() @ Wt.double().t()
    assert_close(out[:rows * L].cpu().numpy(), want.cpu().numpy(), 3e-6, 'pp forward with row count')
    assert float(out[rows * L:].abs().max()) == 0.0
    dY = torch.randn(cap * L, n, device='cuda', generator=g)
    dW = torch.zeros(n, kdim, device='cuda')
    ops.sgemm_big(dY, X, dW, m=n, n=kdim, k=cap * L, trans_a=True, trans_w=True, accumulate=True, k_parts=44, k_count=cnt,
                  rows_per_count=L)
    want = dY[:rows * L].double().t() @ X[:rows * L].double()
    assert_close(dW.cpu().numpy(), want.cpu().numpy(), 3e-6, 'pp weight gradient with reduction count')
