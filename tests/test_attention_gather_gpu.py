"""The gather form of the temporal attention (tiger_temporal_attention_ex, csrc/attention.cu) and its fused last
product, called directly and compared with a float64 restatement of the same operation on the CPU.  The cases sit
where the kernel branches: every head instantiation (HT = 1, 2, 4 and the generic one) at K up to 64, the 16-byte and
the scalar gather, both row sources and both index types of `sel`, node and edge features present or absent, the
depth-1 queries (ts_group = K) and the depth-2 queries (key_rows) of n_layers = 2, rows without a live slot,
misaligned tables, time gaps up to 1e6 s, the split output and the left-memory write-back of the fused product, and
the refusals past the kernel's limits.  Models past those limits must run their torch code instead.

Tolerance: max-norm error relative to the largest entry of the reference, TOL.  The largest error each group reaches
is printed at the end of the module."""
import math

import numpy as np
import pytest
import torch

from oracle import tiger_oracle as O
from www2023tiger_b200 import ops
from www2023tiger_b200._lib import TigerLibraryError, call, ptr
from www2023tiger_b200.init import perturb_biases, random_weights

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda')
TOL = 1e-5
WORST = {}
SENTINEL = 7.25


@pytest.fixture(scope='module', autouse=True)
def report_worst():
    yield
    print('\nlargest relative error per case group:')
    for k in sorted(WORST):
        print(f'  {k:24s} {WORST[k]:.2e}')


def check(group, what, got, want, tol=TOL):
    """max|got - want| / max|want| <= tol; got must hold no NaN."""
    got = got.detach().double().cpu()
    want = want.detach().double().cpu()
    assert got.shape == want.shape, f'{what}: shape {tuple(got.shape)} vs {tuple(want.shape)}'
    if got.numel() == 0:
        return
    assert not torch.isnan(got).any(), f'{what}: NaN in the result'
    scale = float(want.abs().max())
    err = float((got - want).abs().max()) / (scale if scale > 0 else 1.0)
    WORST[group] = max(WORST.get(group, 0.0), err)
    assert err <= tol, f'{what}: rel err {err:.3e} > {tol}'


# ------------------------------------------------------------------------------------------
# parameters and the float64 restatement
# ------------------------------------------------------------------------------------------
P0 = 'temporal_embedding_fn.fns.0.'


def layer_weights(d, de, seed):
    return perturb_biases(random_weights(d, de, seed=seed))


def make_pack(W, d, de, H, prefix=P0):
    pack = ops.AttnPack(d, de, DEV, H)
    m = prefix + 'mha_fn.'
    pack.refresh(*(W[n].to(DEV) for n in (m + 'q_proj_weight', m + 'k_proj_weight', m + 'v_proj_weight',
                                          m + 'in_proj_bias', m + 'out_proj.weight', m + 'out_proj.bias',
                                          prefix + 'merger.fc1.weight', prefix + 'merger.fc1.bias',
                                          prefix + 'merger.fc2.weight', prefix + 'merger.fc2.bias',
                                          'time_encoder.basis_freq', 'time_encoder.phase')))
    return pack


def time_code(dt, w, b):
    """The kernel's time_enc (common.cuh): float32 argument f32(f32(dt * w) + b), no FMA; the cosine in double."""
    arg = (dt.float().unsqueeze(-1) * w.float()) + b.float()     # two separately rounded float32 operations
    return torch.cos(arg.double())


def attention64(W, H, qx, qt, kv, live, prefix=P0):
    """TemporalAttention.forward in float64: qx, qt [n, d], kv [n, K, C], live [n, K] (False = padding slot); a row
    without a live slot has a zero attention output (its merger still sees qx)."""
    g = lambda k: W[prefix + k].double()
    n, K, _ = kv.shape
    E = qx.shape[1] * 2
    hd = E // H
    bq, bk, bv = g('mha_fn.in_proj_bias').chunk(3)
    q = (torch.cat([qx, qt], 1) @ g('mha_fn.q_proj_weight').t() + bq).view(n, H, hd) * math.sqrt(1.0 / hd)
    k = (kv @ g('mha_fn.k_proj_weight').t() + bk).view(n, K, H, hd)
    v = (kv @ g('mha_fn.v_proj_weight').t() + bv).view(n, K, H, hd)
    s = torch.einsum('nhc,nkhc->nhk', q, k)
    any_live = live.any(1)
    s = s.masked_fill(~(live | ~any_live[:, None])[:, None, :], float('-inf'))
    p = torch.softmax(s, -1)
    o = torch.einsum('nhk,nkhc->nhc', p, v).reshape(n, E)
    h = (o @ g('mha_fn.out_proj.weight').t() + g('mha_fn.out_proj.bias')) * any_live[:, None].double()
    hid = torch.relu(torch.cat([h, qx], 1) @ g('merger.fc1.weight').t() + g('merger.fc1.bias'))
    return hid @ g('merger.fc2.weight').t() + g('merger.fc2.bias')


class Case:
    """Inputs of one gather-form call, on the CPU (float32 tables, int64 ids)."""

    def __init__(self, d, de, K, n, *, seed, rows_a=True, sel_dtype=torch.int32, nfeats=True, efeats=True,
                 ts_group=1, period=None, key_rows=False, gap=100.0, n_nodes=50, n_edges=300):
        g = torch.Generator().manual_seed(seed)
        self.d, self.de, self.K, self.n, self.ts_group = d, de, K, n, ts_group
        N, Nb = n_nodes, n_nodes // 2 + 3
        self.rows_b = torch.randn(Nb, d, generator=g)
        self.rows_a = torch.randn(N, d, generator=g) if rows_a else None
        if rows_a:    # the fused routes: -1 = the right-memory row, >= 0 = a GRU-output row
            sel = torch.randint(0, Nb, (N,), generator=g)
            sel[torch.rand(N, generator=g) < 0.5] = -1
        else:         # the class surface: local index into involved_node_reprs
            sel = torch.randint(0, Nb, (N,), generator=g)
        self.sel = sel.to(sel_dtype)
        self.nfeats = torch.randn(N, d, generator=g) * 0.7 if nfeats else None
        self.efeats = torch.randn(n_edges, de, generator=g) if efeats else None
        self.centers = torch.randint(1, N, (n,), generator=g)
        neigh = torch.randint(1, N, (n, K), generator=g)
        neigh[torch.rand(n, K, generator=g) < 0.3] = 0            # id 0: padding slot
        if n >= 3:
            neigh[0] = 0                                          # no live slot
            neigh[1, 1:] = 0                                      # only the first slot live
            neigh[2, :-1] = 0                                     # only the last slot live
            neigh[1, 0] = neigh[2, -1] = 5
        self.neigh = neigh
        self.neigh_e = torch.randint(0, n_edges, (n, K), generator=g)
        self.period = period if period is not None else max(n, 1)
        self.q_ts = (torch.rand(self.period, generator=g) * 1000 + max(gap, 1000.0) + 1000).float()
        qt_of_query = self.q_ts[(torch.arange(n) // ts_group) % self.period]
        self.neigh_ts = (qt_of_query[:, None] - torch.rand(n, K, generator=g) * gap).float()
        self.key_rows = torch.randn(n * K, d, generator=g) * 1.3 if key_rows else None

    def node_rows(self, u):
        s = self.sel.long()[u]
        if self.rows_a is None:
            return self.rows_b.double()[s]
        return torch.where((s >= 0)[..., None], self.rows_b.double()[s.clamp(min=0)], self.rows_a.double()[u])

    def reference(self, W, H, prefix=P0):
        d, de, K, n = self.d, self.de, self.K, self.n
        nf = (lambda u: self.nfeats.double()[u]) if self.nfeats is not None else (lambda u: 0.0)
        qx = self.node_rows(self.centers) + nf(self.centers)
        tw, tb = W['time_encoder.basis_freq'], W['time_encoder.phase']
        qt = time_code(torch.zeros(n), tw, tb)
        if self.key_rows is not None:
            kx = self.key_rows.double().view(n, K, d)
        else:
            kx = self.node_rows(self.neigh) + nf(self.neigh)
        ky = self.efeats.double()[self.neigh_e] if self.efeats is not None else torch.zeros(n, K, de, dtype=torch.float64)
        qt_of_query = self.q_ts[(torch.arange(n) // self.ts_group) % self.period]
        kt = time_code(qt_of_query[:, None] - self.neigh_ts, tw, tb)     # float32 subtraction, as in the kernel
        return attention64(W, H, qx, qt, torch.cat([kx, ky, kt], 2), self.neigh != 0, prefix)

    def device_args(self, lead=0):
        """Device tensors; `lead` floats in front of rows_b and efeats (a lead of d + 1 misaligns them by 4 bytes)."""
        def shifted(t):
            if t is None:
                return None
            buf = torch.full((t.numel() + lead,), -333.0, device=DEV)
            v = buf[lead:].view(t.shape)
            v.copy_(t)
            return v
        # rows_b always keeps a full row of -333 in front: a kernel that indexed it with sel = -1 reads that row
        lead_b = lead if lead >= self.d else self.d
        buf = torch.full((self.rows_b.numel() + lead_b,), -333.0, device=DEV)
        rows_b = buf[lead_b:].view(self.rows_b.shape)
        rows_b.copy_(self.rows_b)
        dv = lambda t: None if t is None else t.to(DEV).contiguous()
        return dict(center_nids=dv(self.centers), q_ts=dv(self.q_ts), neigh_nids=dv(self.neigh),
                    neigh_eids=dv(self.neigh_e), neigh_ts=dv(self.neigh_ts), rows_a=dv(self.rows_a), rows_b=rows_b,
                    sel=dv(self.sel), nfeats=dv(self.nfeats), efeats=shifted(self.efeats) if lead else dv(self.efeats),
                    key_rows=dv(self.key_rows))


def run(pack, H, c, out=None, lead=0):
    a = c.device_args(lead)
    return ops.temporal_attention(pack, H, a['center_nids'], a['q_ts'], a['neigh_nids'], a['neigh_eids'],
                                  a['neigh_ts'], rows_a=a['rows_a'], rows_b=a['rows_b'], sel=a['sel'],
                                  nfeats=a['nfeats'], efeats=a['efeats'], out=out, key_rows=a['key_rows'],
                                  ts_group=c.ts_group)


def test_restatement_matches_the_oracle():
    """attention64 says what O.temporal_attention (the reference's TemporalAttention.forward) says."""
    d, de, K, n, H = 12, 6, 9, 40, 3
    W = layer_weights(d, de, seed=1)
    g = torch.Generator().manual_seed(2)
    qx, qt = torch.randn(n, d, generator=g), torch.randn(n, d, generator=g)
    kx, ky, kt = torch.randn(n, K, d, generator=g), torch.randn(n, K, de, generator=g), torch.randn(n, K, d, generator=g)
    mask = torch.rand(n, K, generator=g) < 0.3
    mask[0] = True
    mask[1, :-1] = True
    want = O.temporal_attention(W, P0, H, qx, qt, kx, ky, kt, mask)
    got = attention64(W, H, qx.double(), qt.double(), torch.cat([kx, ky, kt], 2).double(), ~mask)
    check('restatement', 'float64 restatement vs oracle', got, want, 2e-6)


# ------------------------------------------------------------------------------------------
# K x H at the 16-byte (24, 8) and the scalar (12, 6), (24, 10) gathers; the baseline width
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('d,de', [(24, 8), (12, 6), (24, 10)])
@pytest.mark.parametrize('H', [1, 2, 3, 4, 8])
@pytest.mark.parametrize('K', [1, 7, 32, 33, 64])
def test_gather_at_every_k_and_head_count(K, H, d, de):
    W = layer_weights(d, de, seed=K * 16 + H)
    c = Case(d, de, K, 70, seed=K * 100 + H * 10 + d)
    check('K x H', f'K={K} H={H} d={d} de={de}', run(make_pack(W, d, de, H), H, c), c.reference(W, H))


@pytest.mark.parametrize('K', [10, 20, 64])
def test_gather_at_the_baseline_width(K):
    W = layer_weights(172, 172, seed=K)
    c = Case(172, 172, K, 129, seed=K, n_nodes=400, n_edges=2000)
    check('baseline d=172', f'd=172 K={K}', run(make_pack(W, 172, 172, 2), 2, c), c.reference(W, 2))


# ------------------------------------------------------------------------------------------
# row sources: rows_a + rows_b with both sel types, rows_a = None (class surface); features present or absent
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('source', ['a+b int32', 'a+b int64', 'local int64'])
@pytest.mark.parametrize('nfeats,efeats', [(True, True), (True, False), (False, True), (False, False)])
@pytest.mark.parametrize('d,de', [(24, 8), (12, 6)])
def test_gather_row_sources_and_features(source, nfeats, efeats, d, de):
    W = layer_weights(d, de, seed=3)
    c = Case(d, de, 7, 90, seed=len(source) * 8 + 4 * nfeats + 2 * efeats + d, rows_a=source != 'local int64',
             sel_dtype=torch.int32 if source.endswith('int32') else torch.int64, nfeats=nfeats, efeats=efeats)
    if c.rows_a is not None:
        used = c.sel.long()[torch.cat([c.centers, c.neigh.flatten()])]
        assert (used < 0).any() and (used >= 0).any()
    check('row sources', f'{source} nfeats={nfeats} efeats={efeats} d={d}', run(make_pack(W, d, de, 2), 2, c),
          c.reference(W, 2))


# ------------------------------------------------------------------------------------------
# n_layers = 2: depth-1 queries (query time q_ts[(q / K) % B]) and depth-2 queries keyed by key_rows
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('d,de', [(24, 8), (12, 6)])
def test_depth1_queries_read_their_parent_event_time(d, de):
    B, K = 7, 5
    W = layer_weights(d, de, seed=4)
    c = Case(d, de, K, 3 * B * K, seed=5, ts_group=K, period=B, gap=500.0)
    c.centers = torch.randint(0, 50, (3 * B * K,), generator=torch.Generator().manual_seed(6))   # hop-1 ids, 0 too
    assert len(set(c.q_ts.tolist())) == B
    check('depth-1 form', f'depth 1 d={d}', run(make_pack(W, d, de, 2), 2, c), c.reference(W, 2))


@pytest.mark.parametrize('d,de', [(24, 8), (12, 6)])
def test_depth2_queries_take_key_rows_without_node_features(d, de):
    W = layer_weights(d, de, seed=7)
    c = Case(d, de, 6, 80, seed=8, key_rows=True)
    assert (c.neigh == 0).any()
    want = c.reference(W, 2)
    got = run(make_pack(W, d, de, 2), 2, c)
    check('depth-2 form', f'depth 2 d={d}', got, want)
    # the same call reading the tables instead of key_rows, or adding node features to them, is far off
    rows = Case(d, de, 6, 80, seed=8, key_rows=False)
    assert float((rows.reference(W, 2) - want).abs().max()) > 100 * TOL * float(want.abs().max())


# ------------------------------------------------------------------------------------------
# sizes, untouched rows, misaligned tables, large time gaps
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n', [0, 1, 129, 300])
def test_gather_writes_exactly_its_rows(n):
    d, de, K = 24, 8, 9
    W = layer_weights(d, de, seed=9)
    c = Case(d, de, K, n, seed=n)
    big = torch.full((n + 37, d), SENTINEL, device=DEV)
    pack = make_pack(W, d, de, 2)            # a fresh pack: n = 0 sizes an empty workspace
    got = run(pack, 2, c, out=big[:n])
    check('sizes', f'n={n}', got, c.reference(W, 2))
    assert bool((big[n:] == SENTINEL).all()), 'rows past n_query were written'


@pytest.mark.parametrize('d,de', [(24, 8), (100, 4)])
def test_misaligned_tables(d, de):
    W = layer_weights(d, de, seed=10)
    c = Case(d, de, 11, 150, seed=11)
    pack = make_pack(W, d, de, 2)
    aligned = run(pack, 2, c).clone()
    shifted = run(pack, 2, c, lead=d + 1)        # rows_b and efeats 4 bytes off a 16-byte boundary: scalar gather
    want = c.reference(W, 2)
    check('misaligned', f'aligned d={d}', aligned, want)
    check('misaligned', f'misaligned d={d}', shifted, want)
    check('misaligned', f'misaligned vs aligned d={d}', shifted, aligned.double())


@pytest.mark.parametrize('d,de', [(24, 8), (12, 6)])
def test_time_gaps_up_to_1e6_seconds(d, de):
    W = layer_weights(d, de, seed=12)
    c = Case(d, de, 16, 100, seed=13, gap=1e6)
    assert float((c.q_ts[:, None] - c.neigh_ts).max()) > 5e5
    check('time gaps 1e6', f'gap 1e6 d={d}', run(make_pack(W, d, de, 2), 2, c), c.reference(W, 2))


# ------------------------------------------------------------------------------------------
# fused last product: score fold (split output pq) + left-memory write-back
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('d,key_rows', [(8, False), (20, False), (100, False), (172, False), (20, True)])
def test_fused_last_product(d, key_rows):
    """n_split = d rounded up to 16 (16, 32, 112, 176): pq = [W1a z | W1b z]; winner rows of the first n_pos = 2B
    positions land in the left memory bit-equal to out, with their batch time and the activity flag; nothing else
    changes; TIGER_ERR_PAST_MEMORY is set exactly when a winner's stored clock is later than its batch time."""
    B, K, H, de, N = 40, 6, 2, 8, 100
    W = layer_weights(d, de, seed=d)
    g = torch.Generator().manual_seed(d + 1)
    c = Case(d, de, K, 3 * B, seed=d + 2, key_rows=key_rows, period=B, n_nodes=N)
    c.centers = torch.cat([torch.randint(1, N // 2, (2 * B,), generator=g),        # src, dst
                           torch.randint(N // 2, N, (B,), generator=g)])           # negatives: other ids
    z = c.reference(W, H)
    w1 = W['score_fn.fc1.weight'].double()
    pq_want = torch.cat([z @ w1[:, :d].t(), z @ w1[:, d:].t()], 1)
    pack = make_pack(W, d, de, H)
    sw = [W['score_fn.' + n].to(DEV) for n in ('fc1.weight', 'fc1.bias', 'fc2.weight', 'fc2.bias')]
    fold = ops.ScoreFold(d, DEV)
    fold.refresh(*sw, W[P0 + 'merger.fc2.weight'].to(DEV), W[P0 + 'merger.fc2.bias'].to(DEV),
                 W['hit_embedding.weight'].to(DEV))
    a = c.device_args()
    pos_ids = a['center_nids'][:2 * B]
    # the winner flags and batch times are views of longer buffers whose tails differ: a kernel that read past n_pos
    # or past the batch would see them
    first = np.zeros(3 * B, dtype=np.uint8)
    first[np.unique(c.centers[:2 * B].numpy(), return_index=True)[1]] = 1
    first[2 * B:] = 1
    wbuf = torch.as_tensor(first).to(DEV)
    winner = wbuf[:2 * B]
    tbuf = torch.cat([c.q_ts, c.q_ts + 500]).to(DEV)
    ts = tbuf[:B]
    win_pos = np.nonzero(first[:2 * B])[0]
    win_nodes = c.centers[:2 * B].numpy()[win_pos]
    init_vals = torch.randn(N, d, generator=g)
    init_ts = torch.full((N,), 5.0)
    init_ts[N // 2:] = 1e9          # negatives (and so non-winners) far in the future: no error bit from them
    spare = np.setdiff1d(np.arange(1, N // 2), c.centers[:2 * B].numpy())
    assert len(spare) > 0
    init_ts[spare] = 1e9            # other nodes too
    p_eq = win_pos[0]
    init_ts[win_nodes[0]] = c.q_ts[p_eq % B]            # equal clock: allowed
    for past in (False, True):
        t0 = init_ts.clone()
        if past:
            p1 = win_pos[1]
            t0[win_nodes[1]] = c.q_ts[p1 % B] + 1.0     # one winner's memory is later than its batch time
        left_vals, left_ts = init_vals.to(DEV), t0.to(DEV)
        left_active = torch.zeros(N, dtype=torch.uint8, device=DEV)
        err = torch.zeros(1, dtype=torch.int32, device=DEV)
        pq = torch.full((3 * B, 2 * d), SENTINEL, device=DEV)
        pack.attach_score_fold(fold, pq)
        pack.attach_left_writeback(pos_ids, winner, ts, left_vals, left_ts, left_active, err)
        try:
            out = ops.temporal_attention(pack, H, a['center_nids'], ts, a['neigh_nids'], a['neigh_eids'],
                                         a['neigh_ts'], rows_a=a['rows_a'], rows_b=a['rows_b'], sel=a['sel'],
                                         nfeats=a['nfeats'], efeats=a['efeats'], key_rows=a['key_rows'])
        finally:
            pack.attach_score_fold(None, None)
            pack.attach_left_writeback(None)
        what = f'fused d={d} key_rows={key_rows} past={past}'
        check('fused out', what, out, z)
        check('fused pq', what + ' pq', pq, pq_want)
        assert int(err.item()) == (1 if past else 0), what + ': TIGER_ERR_PAST_MEMORY'
        lv, lt, la = left_vals.cpu(), left_ts.cpu(), left_active.cpu()
        o = out.cpu()
        assert torch.equal(lv[win_nodes], o[win_pos]), what + ': left rows of the winners'
        assert torch.equal(lt[win_nodes], c.q_ts[win_pos % B]), what + ': left clocks'
        assert bool((la[win_nodes] == 1).all()), what + ': left activity'
        rest = np.setdiff1d(np.arange(N), win_nodes)
        assert torch.equal(lv[rest], init_vals[rest]) and torch.equal(lt[rest], t0[rest]), what + ': other rows'
        assert int(la[rest].sum()) == 0, what + ': other activity flags'


# ------------------------------------------------------------------------------------------
# refusals: TigerLibraryError('invalid argument'), out untouched
# ------------------------------------------------------------------------------------------
def raw_call(pack, H, c, out, work, dense=False):
    a = c.device_args()
    if dense:
        n, K, d, de = c.n, c.K, c.d, c.de
        z = lambda *s: torch.zeros(*s, device=DEV)
        mask = (a['neigh_nids'] == 0).to(torch.uint8)
        call('tiger_temporal_attention_dense', ptr(z(n, d)), ptr(z(n, d)), ptr(z(n, K, d)), ptr(z(n, K, de)),
             ptr(z(n, K, d)), ptr(mask), n, K, d, de, H, pack.byref(), ptr(out), ptr(work))
        return
    call('tiger_temporal_attention_ex', ptr(a['center_nids']), ptr(a['q_ts']), c.n, c.period, c.ts_group,
         ptr(a['neigh_nids']), ptr(a['neigh_eids']), ptr(a['neigh_ts']), c.K, ptr(a['rows_a']), ptr(a['rows_b']),
         None, ptr(a['sel']), int(a['sel'].dtype == torch.int64), ptr(a['nfeats']), ptr(a['efeats']), c.d, c.de, H,
         pack.byref(), ptr(out), ptr(work))


@pytest.mark.parametrize('what', ['K=65', 'H=9', 'footprint', 'fold without write-back', 'fused on dense'])
def test_refusals_leave_out_untouched(what):
    d, de, K, H = {'K=65': (16, 8, 65, 2), 'H=9': (18, 6, 10, 9), 'footprint': (258, 258, 64, 2)}.get(
        what, (16, 8, 10, 2))
    W = layer_weights(d, de, seed=14)
    pack = make_pack(W, d, de, H)
    c = Case(d, de, K, 20, seed=15)
    n = c.n
    out = torch.full((n, d), SENTINEL, device=DEV)
    work = torch.zeros(1 << 22, dtype=torch.uint8, device=DEV)    # larger than any of these calls needs
    pq = torch.full((n, 2 * d), SENTINEL, device=DEV)
    left = torch.full((60, d), SENTINEL, device=DEV)
    if what in ('fold without write-back', 'fused on dense'):
        fold = ops.ScoreFold(d, DEV)
        pack.attach_score_fold(fold, pq)
    if what == 'fused on dense':
        a = c.device_args()
        ts = a['q_ts'][:n // 3]
        pack.attach_left_writeback(a['center_nids'][:2 * (n // 3)], torch.ones(2 * (n // 3), dtype=torch.uint8,
                                   device=DEV), ts, left, torch.zeros(60, device=DEV))
    with pytest.raises(TigerLibraryError, match='invalid argument'):
        raw_call(pack, H, c, out, work, dense=what == 'fused on dense')
    torch.cuda.synchronize()
    assert bool((out == SENTINEL).all()) and bool((pq == SENTINEL).all()) and bool((left == SENTINEL).all())
    if what in ('K=65', 'H=9', 'footprint'):
        assert ops.attention_limit_error(d, de, K, H) is not None
        with pytest.raises(TigerLibraryError, match='invalid argument'):
            run(pack, H, c, out=out)
        assert bool((out == SENTINEL).all())


# ------------------------------------------------------------------------------------------
# models past the kernel's limits run on their torch code
# ------------------------------------------------------------------------------------------
def small_stream(de):
    from www2023tiger_b200.synthetic import StreamShape, make_stream
    return make_stream(StreamShape('lim', 60, 20, 1500, de, None, horizon=1500.), seed=0)


LIMIT_CASES = [(65, 2, 8, 1), (65, 2, 8, 2), (10, 9, 18, 1)]     # K, heads, width, n_layers
LIMIT_MATCH = {65: 'at most 64 neighbors', 9: 'at most 8 heads'}


@pytest.mark.parametrize('K,H,de,n_layers', LIMIT_CASES)
def test_engine_refuses_models_past_the_limits(K, H, de, n_layers):
    import gpu_utils as gu
    from www2023tiger_b200.engine import TigerEngine
    st = small_stream(de)
    N = st.n_nodes
    W = random_weights(de, de, n_nodes=N, n_layers=n_layers)
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    efeats = gu.dev(st.efeats, torch.float32)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    with pytest.raises(NotImplementedError, match=LIMIT_MATCH[K if K > 64 else H]):
        TigerEngine(W, csr, n_nodes=N, dim=de, efeats=efeats, n_neighbors=K, n_head=H, batch_size=30,
                    n_layers=n_layers)
    assert torch.cuda.memory_allocated() == before, 'the engine allocated before refusing'


@pytest.mark.parametrize('K,H,de,n_layers', LIMIT_CASES)
def test_dropin_evaluates_models_past_the_limits_on_torch_code(K, H, de, n_layers):
    """No-grad evaluation batches of a model the attention kernel cannot take: no TigerLibraryError, and the same
    scores and memories as the same model with grad enabled, where every operator runs its torch code."""
    import dropin_utils as D
    import gpu_utils as gu
    from tiger.data.data_loader import GraphCollator, InteractionData
    from tiger.data.graph import Graph
    from www2023tiger_b200.synthetic import NegativeSampler
    st = small_stream(de)
    N, B = st.n_nodes, 30
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    full = InteractionData(st.src, st.dst, st.ts, st.eids, np.zeros_like(st.src), seed=0, eval=True, neg_dst=neg)
    graph = Graph.from_csr(gu.device_csr(st.src, st.dst, st.ts, st.eids, N))
    coll = GraphCollator(graph, K, n_layers, restarter='static', hist_len=40)
    models = []
    for _ in range(2):
        torch.manual_seed(0)
        m = D.init_model(None, st.efeats, graph, N, st.n_events, DEV, dim=st.dim, n_layers=n_layers, n_heads=H,
                         n_neighbors=K, hit_type='bin', dropout=0.1, restarter_type='static', hist_len=40,
                         msg_src='left', upd_src='right')
        m.eval()
        m.reset()
        models.append(m)
    kern, ref = models
    ref.load_state_dict(kern.state_dict())
    assert not kern._fusable()
    names = ('loss', 'h_left', 'pos_scores', 'neg_scores', 'h_prev_left', 'h_prev_right')
    for ib in range(4):
        lo = 600 + ib * B
        src, dst, ng, ts, eids, _, cg = coll([full[i] for i in range(lo, lo + B)])
        src, dst, ng, eids = (x.long().to(DEV) for x in (src, dst, ng, eids))
        ts, cg = ts.float().to(DEV), cg.to(DEV)
        with torch.no_grad():
            got = kern.contrast_learning(src, dst, ng, ts, eids, cg)
        with torch.enable_grad():
            want = ref.contrast_learning(src, dst, ng, ts, eids, cg)
        what = f'K={K} H={H} n_layers={n_layers} batch {ib} '
        for name, a, b in zip(names, got, want):
            check('past the limits', what + name, a.reshape(-1), b.reshape(-1))
        for name in ('left_memory', 'right_memory'):
            check('past the limits', what + name, getattr(kern, name).vals, getattr(ref, name).vals)
            assert torch.equal(getattr(kern, name).update_ts, getattr(ref, name).update_ts), what + name
        check('past the limits', what + 'messages', kern.msg_store.node_msg_vals, ref.msg_store.node_msg_vals)
