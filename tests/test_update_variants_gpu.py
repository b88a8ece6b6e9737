"""The message transform (--tsfm_fn linear | mlp) and memory updater (--upd_fn merge) variants on the fused inference
path: the two kernels they add (tiger_merge_update, tiger_gru_update_rows) against a float64 restatement, TigerEngine
and the drop-in's fused no-grad route against the goldens of the unmodified reference (var_tsfm_linear, var_tsfm_mlp,
var_upd_merge), and the engine against the drop-in's torch-op route on seeded streams at BASELINE dimensions."""
import numpy as np
import pytest
import torch
from torch.utils.data import DataLoader

from golden_utils import Golden, assert_close
from www2023tiger_b200 import _lib, ops
from www2023tiger_b200._lib import call, ptr
from www2023tiger_b200.engine import KERNELS_PER_STEP, StreamRunner, TigerEngine
from www2023tiger_b200.init import perturb_biases, random_weights
from www2023tiger_b200.synthetic import SHAPES, NegativeSampler, make_stream

pytestmark = pytest.mark.gpu
TOL = 1e-5
cpu = lambda t: t.detach().cpu().numpy()
VAR_GOLDENS = ('var_tsfm_linear', 'var_tsfm_mlp', 'var_upd_merge')


# ------------------------------------------------------------------------------------------
# the kernels against float64
# ------------------------------------------------------------------------------------------
def sig(x):
    return 1.0 / (1.0 + np.exp(-x))


def gru64(x, h, w_ih, w_hh, b_ih, b_hh):
    d = h.shape[1]
    gi, gh = x @ w_ih.T + b_ih, h @ w_hh.T + b_hh
    r, z = sig(gi[:, :d] + gh[:, :d]), sig(gi[:, d:2 * d] + gh[:, d:2 * d])
    n = np.tanh(gi[:, 2 * d:] + r * gh[:, 2 * d:])
    return (1 - z) * n + z * h


def merge64(x, h, fc1_w, fc1_b, fc2_w, fc2_b):
    return np.maximum(np.concatenate([x, h], 1) @ fc1_w.T + fc1_b, 0) @ fc2_w.T + fc2_b


def strided(a, pad, dev):
    """A [rows, w] float32 view with row stride w + pad (pad 0: contiguous)."""
    buf = torch.zeros(a.shape[0], a.shape[1] + pad, dtype=torch.float32, device=dev)
    buf[:, :a.shape[1]] = torch.from_numpy(a.astype(np.float32))
    return buf[:, :a.shape[1]]


def launch(kind, pack, *, ids, count, n_rows, x, h, out, mid, msg_ts, mem_ts, check_equal, err):
    """The raw entry points, so that x / h may be strided views."""
    if kind == 'gru_rows':
        call('tiger_gru_update_rows', ptr(ids), ptr(count), n_rows, x.data_ptr(), x.stride(0), h.data_ptr(),
             h.stride(0), pack.m_dim, pack.d, ptr(pack.wpack), ptr(pack.b_ih), ptr(pack.b_hh), ptr(out), ptr(msg_ts),
             ptr(mem_ts), int(check_equal), ptr(err))
    else:
        call('tiger_merge_update', ptr(ids), ptr(count), n_rows, x.data_ptr(), x.stride(0), int(kind == 'merge_rows'),
             h.data_ptr(), h.stride(0), pack.m_dim, pack.d, ptr(pack.wpack), ptr(pack.b1), ptr(mid), ptr(msg_ts),
             ptr(mem_ts), int(check_equal), ptr(err))
        ops.sgemm_nt_packed(mid, pack.fc2, pack.b2, out, m_rows=n_rows, count=count)


def kernel_case(kind, d, m, n, pad, seed, *, dev, mem_ts_shift=0.0, check_equal=False):
    """n valid rows (device count) inside a grid of n + 200 rows, over node-indexed tables of N > n + 200 rows;
    `kind`: gru_rows | merge (x by node id) | merge_rows (x by row position)."""
    rng = np.random.default_rng(seed)
    cap = n + 200
    N = cap + 37
    ids_np = rng.permutation(N)[:cap].astype(np.int64)
    x_rows = cap if kind != 'merge' else N
    x_np = rng.standard_normal((x_rows, m))
    h_np = rng.standard_normal((N, d))
    s = 1 / np.sqrt(m + d)
    if kind == 'gru_rows':
        w = [rng.uniform(-s, s, sh) for sh in ((3 * d, m), (3 * d, d), (3 * d,), (3 * d,))]
        pack = ops.GruPack(*(torch.from_numpy(t).float().to(dev) for t in w))
    else:
        w = [rng.standard_normal(sh) * s for sh in ((d, m + d), (d,), (d, d), (d,))]
        pack = ops.MergePack(*(torch.from_numpy(t).float().to(dev) for t in w))
    w32 = [t.astype(np.float32).astype(np.float64) for t in w]
    ids = torch.from_numpy(ids_np).to(dev)
    count = torch.tensor([n], dtype=torch.int32, device=dev)
    x, h = strided(x_np, pad, dev), strided(h_np, pad, dev)
    msg_ts = torch.from_numpy(rng.uniform(0, 100, N).astype(np.float32)).to(dev)
    mem_ts = msg_ts - mem_ts_shift
    out = torch.full((cap, d), float('nan'), device=dev)
    mid = torch.full((cap, d), float('nan'), device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    launch(kind, pack, ids=ids, count=count, n_rows=cap, x=x, h=h, out=out, mid=mid, msg_ts=msg_ts, mem_ts=mem_ts,
           check_equal=check_equal, err=err)
    torch.cuda.synchronize()
    sel = ids_np[:n]
    xr = (x_np[:n] if kind != 'merge' else x_np[sel]).astype(np.float32).astype(np.float64)
    hr = h_np[sel].astype(np.float32).astype(np.float64)
    want = gru64(xr, hr, *w32) if kind == 'gru_rows' else merge64(xr, hr, *w32)
    return cpu(out), want, int(err.item())


@pytest.mark.parametrize('kind', ['gru_rows', 'merge', 'merge_rows'])
@pytest.mark.parametrize('d,m', [(172, 688), (100, 304), (8, 32), (172, 344), (8, 21)])
@pytest.mark.parametrize('n', [0, 1, 127, 128, 129, 2100])
def test_kernel_against_float64(kind, d, m, n):
    """BASELINE widths (M = 3d + d_e = 688 / 304, MLP hidden 344), the fixture widths (d = 8, M = 32, hidden 21);
    row counts around the 128-row tile and past 2,048; rows beyond the device count stay untouched."""
    dev = torch.device('cuda')
    out, want, err = kernel_case(kind, d, m, n, 0, seed=d + m + n, dev=dev)
    assert err == 0
    assert_close(out[:n], want, TOL, f'{kind} d={d} m={m} n={n}')
    assert np.isnan(out[n:]).all(), 'rows past the device count were written'


@pytest.mark.parametrize('kind', ['gru_rows', 'merge', 'merge_rows'])
@pytest.mark.parametrize('pad', [1, 3, 5])
def test_kernel_unaligned_row_strides(kind, pad):
    """x and h tables whose row strides are not a multiple of four floats take the scalar gather."""
    dev = torch.device('cuda')
    out, want, err = kernel_case(kind, 100, 304, 300, pad, seed=pad, dev=dev)
    assert err == 0
    assert_close(out[:300], want, TOL, f'{kind} pad={pad}')


@pytest.mark.parametrize('kind', ['gru_rows', 'merge', 'merge_rows'])
def test_kernel_sets_message_invariant_bits(kind):
    """tiger.py:319-327 from the inputs alone: a memory clock past the message time sets MSG_BEFORE_MEM; with
    check_equal (msg_src = left) any difference sets MSG_TS_MISMATCH."""
    dev = torch.device('cuda')
    _, _, err = kernel_case(kind, 8, 32, 129, 0, seed=1, dev=dev, mem_ts_shift=-1.0)
    assert err & 4 and not err & 8
    _, _, err = kernel_case(kind, 8, 32, 129, 0, seed=1, dev=dev, mem_ts_shift=1.0, check_equal=True)
    assert err == 8
    _, _, err = kernel_case(kind, 8, 32, 129, 0, seed=1, dev=dev, mem_ts_shift=0.0, check_equal=True)
    assert err == 0
    with pytest.raises(ValueError, match='later than memory'):
        _lib.raise_on_err_flags(4)


# ------------------------------------------------------------------------------------------
# goldens of the unmodified reference
# ------------------------------------------------------------------------------------------
def engine_for(W, csr, *, N, dim, efeats, nfeats, K, H, B, msg_src, upd_src, tsfm, upd, restarter=None, lazy=False,
               hist_len=40, n_layers=1):
    dev = lambda x: None if x is None else torch.as_tensor(x).float().cuda().contiguous()
    return TigerEngine({k: torch.as_tensor(v) for k, v in W.items()}, csr, n_nodes=N, dim=dim, efeats=dev(efeats),
                       nfeats=dev(nfeats), n_neighbors=K, n_head=H, batch_size=B, msg_src=msg_src, upd_src=upd_src,
                       restarter=restarter, hist_len=hist_len, lazy_restart=lazy, want_restarter_targets=True,
                       n_layers=n_layers, msg_tsfm_type=tsfm, mem_update_type=upd)


def engine_state(e):
    return [t.clone() for t in (e.out_buf, e.emb, e.left_vals, e.right_vals, e.msg_vals, e.left_ts, e.right_ts,
                                e.msg_ts, e.has_msg, e.h_new)]


@pytest.mark.parametrize('name', VAR_GOLDENS)
def test_engine_replays_variant_golden_eager_and_captured(name):
    import gpu_utils as gu
    g = Golden(name)
    assert g.n_layers == 1
    csr = gu.device_csr(g.src, g.dst, g.ts, g.eids, g.N)
    e = engine_for(g.W, csr, N=g.N, dim=g.dim, efeats=g.efeats, nfeats=g.nfeats, K=g.K, H=g.n_heads, B=g.bs,
                   msg_src=g.msg_src, upd_src=g.upd_src, tsfm=g.tsfm, upd=g.upd,
                   restarter=g.restarter if g.lazy_restart else None, lazy=g.lazy_restart, hist_len=g.hist_len)
    # the variants' extra launches: the MLP's hidden product, the merge updater's fc2 product
    assert e.launches_per_step() == (sum(KERNELS_PER_STEP.values()) + (g.tsfm == 'mlp') + (g.upd == 'merge')
                                     + 1 + (g.lazy_restart and g.restarter == 'static'))
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
    # the same batches through the captured graphs of the pipeline: bit for bit the eager results
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


@pytest.mark.parametrize('name', VAR_GOLDENS)
def test_dropin_variant_takes_fused_route_and_replays_golden(name, monkeypatch):
    import dropin_utils as D
    from tiger.data.data_loader import GraphCollator, InteractionData
    from tiger.data.graph import Graph
    from tiger.model.tiger import TIGE
    dev = torch.device('cuda')
    g = Golden(name)
    full = InteractionData(g.src, g.dst, g.ts, g.eids, np.zeros_like(g.src), seed=0, eval=True, neg_dst=g.neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    coll = GraphCollator(graph, g.K, 1, restarter=g.restarter, hist_len=g.hist_len)
    model = D.load_golden_weights(D.model_from_golden(g, graph, dev), g)
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
        for ib, batch in enumerate(DataLoader(full, batch_size=g.bs, collate_fn=coll)):
            if ib >= g.n_batches:
                break
            what = f'dropin {name} b{ib} '
            src, dst, neg, ts, eids, _, cg = batch
            src, dst, neg, eids = (x.long().cuda() for x in (src, dst, neg, eids))
            ts, cg = ts.float().cuda(), cg.to(dev)
            if g.lazy_restart:
                fresh = set(cg.np_computation_graph_nodes.tolist()) - uptodate
                r_nids = torch.tensor(sorted(fresh), dtype=torch.long, device=dev)
                if len(r_nids):
                    model.restart(r_nids, torch.full((len(r_nids),), ts.min().item(), device=dev))
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


def test_dropin_refolds_after_a_parameter_update():
    """An in-place parameter change (an optimizer step) re-packs the fold; the fused route then matches the torch-op
    route of the changed model."""
    import dropin_utils as D
    from tiger.data.data_loader import GraphCollator, InteractionData
    from tiger.data.graph import Graph
    dev = torch.device('cuda')
    g = Golden('var_tsfm_mlp')
    full = InteractionData(g.src, g.dst, g.ts, g.eids, np.zeros_like(g.src), seed=0, eval=True, neg_dst=g.neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    coll = GraphCollator(graph, g.K, 1, restarter=g.restarter, hist_len=g.hist_len)
    model = D.load_golden_weights(D.model_from_golden(g, graph, dev), g)
    model.eval()
    batches = [b for _, b in zip(range(6), DataLoader(full, batch_size=g.bs, collate_fn=coll))]

    def run(fused):
        model.reset()
        outs = []
        for src, dst, neg, ts, eids, _, cg in batches:
            src, dst, neg, eids = (x.long().cuda() for x in (src, dst, neg, eids))
            ts, cg = ts.float().cuda(), cg.to(dev)
            with (torch.no_grad() if fused else torch.enable_grad()):
                outs.append([cpu(t) for t in model.contrast_learning(src, dst, neg, ts, eids, cg)[:2]])
        return outs
    run(True)
    with torch.no_grad():
        model.msg_transform_fn.fn[4].weight.mul_(1.5)
        model.right_mem_updater.cell.weight_ih.add_(0.01)
    for a, b in zip(run(True), run(False)):
        for x, y in zip(a, b):
            assert_close(x.reshape(-1), y.reshape(-1), TOL, 'after update')


# ------------------------------------------------------------------------------------------
# engine vs the drop-in's torch-op route (grad enabled, eval mode) on seeded streams
# ------------------------------------------------------------------------------------------
def compare_with_torch_route(shape, *, start, n_batches, restarter, lazy, tsfm, upd, n_layers=1, B=200, K=10, H=2,
                             seed=0):
    """The same batches through TigerEngine (eager launches) and the drop-in TIGER on its step-by-step torch-op route;
    integer outputs must agree bit for bit, floats within TOL.  Returns the worst relative error per quantity."""
    import dropin_utils as D
    import gpu_utils as gu
    from tiger.data.data_loader import GraphCollator, InteractionData
    from tiger.data.graph import Graph
    dev = torch.device('cuda')
    st = make_stream(shape, seed=seed)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    N = st.n_nodes
    d = st.nfeats.shape[1] if st.nfeats is not None else st.dim
    de = st.efeats.shape[1] if st.efeats is not None else d
    W = perturb_biases(random_weights(d, de, n_nodes=N, restarter=restarter, nonzero_static=True, seed=seed + 1,
                                      n_layers=n_layers, msg_tsfm_type=tsfm, mem_update_type=upd))
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = engine_for(W, csr, N=N, dim=st.dim, efeats=st.efeats, nfeats=st.nfeats, K=K, H=H, B=B,
                   msg_src=shape.msg_src, upd_src=shape.upd_src, tsfm=tsfm, upd=upd, restarter=restarter, lazy=lazy,
                   n_layers=n_layers)
    full = InteractionData(st.src, st.dst, st.ts, st.eids, np.zeros_like(st.src), seed=0, eval=True, neg_dst=neg)
    graph = Graph.from_csr(csr)
    coll = GraphCollator(graph, K, n_layers, restarter=restarter, hist_len=40)
    model = D.init_model(st.nfeats, st.efeats, graph, N, st.n_events, dev, dim=st.dim, n_layers=n_layers, n_heads=H,
                         n_neighbors=K, hit_type='bin', dropout=0.1, restarter_type=restarter, hist_len=40,
                         msg_src=shape.msg_src, upd_src=shape.upd_src, msg_tsfm_type=tsfm, mem_update_type=upd)
    res = model.load_state_dict(W, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    assert not [k for k in res.missing_keys if k.startswith(('msg_transform_fn.', 'right_mem_updater.'))]
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
        what = f'{shape.name} {tsfm}+{upd} batch {ib} '
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
        U, Oc, R = (int(x) for x in e.counts[:3])
        assert np.array_equal(cpu(e.neigh_nids), cpu(cg.layers[n_layers][0])), what + 'neighbors'
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
    print(f'{shape.name} {restarter} lazy={lazy} {tsfm}+{upd} n_layers={n_layers}: max rel err ' +
          ', '.join(f'{k} {v:.2e}' for k, v in worst.items()))
    return worst


@pytest.mark.parametrize('tsfm,upd', [('linear', 'gru'), ('mlp', 'gru'), ('id', 'merge'), ('mlp', 'merge')])
@pytest.mark.parametrize('name', ['wikipedia', 'reddit'])
def test_engine_matches_torch_route_at_baseline_dimensions(name, tsfm, upd):
    """d = d_e = 172 (M = 688, MLP hidden 344), K = 10, B = 200, lazy restart, 30 batches from mid-stream."""
    shape = SHAPES[name]
    compare_with_torch_route(shape, start=(shape.n_events // 2) // 200 * 200, n_batches=30,
                             restarter=shape.restarter, lazy=True, tsfm=tsfm, upd=upd)


def test_engine_matches_torch_route_mlp_merge_two_layers():
    shape = SHAPES['wikipedia']
    compare_with_torch_route(shape, start=(shape.n_events // 2) // 200 * 200, n_batches=30, restarter='seq',
                             lazy=True, tsfm='mlp', upd='merge', n_layers=2)


@pytest.mark.parametrize('tsfm,upd', [('mlp', 'gru'), ('linear', 'merge')])
def test_engine_matches_torch_route_mooc_shape(tsfm, upd):
    """d_e = 4 with node features (d = 100): M = 304, MLP hidden 152; right / right memory sources."""
    shape = SHAPES['mooc']
    compare_with_torch_route(shape, start=(shape.n_events // 2) // 200 * 200, n_batches=30, restarter='seq',
                             lazy=True, tsfm=tsfm, upd=upd)


# ------------------------------------------------------------------------------------------
# what stays as it was
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('tsfm,upd', [('mlp', 'gru'), ('id', 'merge'), ('linear', 'gru')])
def test_native_trainer_still_refuses_variants(tsfm, upd):
    import dropin_utils as D
    from tiger.data.data_loader import InteractionData
    from tiger.data.graph import Graph
    from www2023tiger_b200.train import NativeTrainer
    g = Golden('var_upd_merge')
    full = InteractionData(g.src, g.dst, g.ts, g.eids, np.zeros_like(g.src), seed=0, eval=True, neg_dst=g.neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    model = D.init_model(None, g.efeats, graph, g.N, len(g.src), torch.device('cuda'), dim=g.dim, n_layers=1,
                         n_heads=2, n_neighbors=g.K, hit_type='bin', dropout=0.1, restarter_type='seq', hist_len=6,
                         msg_src='left', upd_src='right', msg_tsfm_type=tsfm, mem_update_type=upd)
    model.train()
    assert not model._native_training()
    with pytest.raises(NotImplementedError):
        NativeTrainer(model, g.bs)
