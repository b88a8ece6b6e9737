"""End-to-end parity of the fused per-batch path (TigerEngine, through the C ABI) against
(1) the golden fixtures of the unmodified reference and (2) the CPU oracle on seeded streams;
plus size-independent properties at BASELINE stream sizes."""
import numpy as np
import pytest
import torch

from oracle import tiger_oracle as O
from golden_utils import CASES, Golden, assert_close
from www2023tiger_b200 import ops
from www2023tiger_b200.engine import StreamRunner
from www2023tiger_b200.init import perturb_biases, random_weights
from www2023tiger_b200.synthetic import NegativeSampler, SHAPES, StreamShape, make_stream

pytestmark = pytest.mark.gpu
TOL = 1e-5


@pytest.fixture(scope='module')
def gu():
    import gpu_utils
    return gpu_utils


def check_state(gu, e, left_vals, right_vals, left_ts, right_ts, msg_vals, msg_ts, pending, what):
    assert_close(gu.cpu(e.left_vals), left_vals, TOL, what + 'left_vals')
    assert_close(gu.cpu(e.right_vals), right_vals, TOL, what + 'right_vals')
    assert np.array_equal(gu.cpu(e.left_ts), left_ts), what + 'left_ts'
    assert np.array_equal(gu.cpu(e.right_ts), right_ts), what + 'right_ts'
    assert np.array_equal(gu.cpu(e.msg_ts), msg_ts), what + 'msg_ts'
    assert_close(gu.cpu(e.msg_vals), msg_vals, TOL, what + 'msg_vals')
    assert np.array_equal(np.nonzero(gu.cpu(e.has_msg))[0], pending), what + 'pending'


@pytest.mark.parametrize('name', CASES)
def test_engine_replays_reference_golden(gu, name):
    g = Golden(name)
    csr = gu.device_csr(g.src, g.dst, g.ts, g.eids, g.N)
    fused_restart = g.lazy_restart
    e = gu.engine_from(g.W, csr, N=g.N, dim=g.dim, efeats=g.efeats, nfeats=g.nfeats, K=g.K, H=g.n_heads, B=g.bs,
                       msg_src=g.msg_src, upd_src=g.upd_src, restarter=g.restarter if fused_restart else None,
                       lazy_restart=fused_restart, hist_len=g.hist_len)
    B = g.bs
    for ib in range(g.n_batches):
        what = f'{name} batch {ib} '
        e.set_batch(*g.batch(ib))
        e.step()
        e.check_errors()
        U, Oc, R = (int(x) for x in e.counts[:3])
        assert np.array_equal(gu.cpu(e.neigh_nids), g.b(ib, 'neigh_nids')), what
        assert np.array_equal(gu.cpu(e.neigh_eids), g.b(ib, 'neigh_eids')), what
        assert np.array_equal(gu.cpu(e.neigh_ts), g.b(ib, 'neigh_ts')), what
        assert np.array_equal(gu.cpu(e.involved[:U]), g.b(ib, 'involved')), what
        if fused_restart:
            assert np.array_equal(gu.cpu(e.restart_nodes[:R]), g.b(ib, 'restart_nids')), what
            if g.restarter == 'seq' and g.has(ib, 'restart_hl'):
                # the seq restarter's own outputs for the lazily restarted nodes (restarters.py:51-114)
                assert_close(gu.cpu(e.seq.h_left[:R]), g.b(ib, 'restart_hl'), TOL, what + 'restart_hl')
                assert_close(gu.cpu(e.seq.h_right[:R]), g.b(ib, 'restart_hr'), TOL, what + 'restart_hr')
                assert np.array_equal(gu.cpu(e.seq.prev_ts[:R]), g.b(ib, 'restart_pt')), what + 'restart_pt'
        assert np.array_equal(gu.cpu(e.outdated[:Oc]),
                              np.intersect1d(g.b(ib, 'pending_before'), g.b(ib, 'involved'))), what
        assert_close(gu.cpu(e.emb[:2 * B]), g.b(ib, 'h_left'), TOL, what + 'h_left')
        assert_close(gu.cpu(e.scores[:B]), g.b(ib, 'pos_scores'), TOL, what + 'pos')
        assert_close(gu.cpu(e.scores[B:]), g.b(ib, 'neg_scores'), TOL, what + 'neg')
        assert_close(gu.cpu(e.loss), g.b(ib, 'loss').reshape(1), TOL, what + 'loss')
        assert_close(gu.cpu(e.hprev_left), g.b(ib, 'h_prev_left'), TOL, what + 'hpl')
        assert_close(gu.cpu(e.hprev_right), g.b(ib, 'h_prev_right'), TOL, what + 'hpr')
        w = np.zeros(2 * B, dtype=np.uint8)
        w[g.b(ib, 'r_index')] = 1            # collator's select_latest on the same (id, t) pairs
        assert np.array_equal(gu.cpu(e.winner), w), what + 'winners'
        check_state(gu, e, g.b(ib, 'left_vals'), g.b(ib, 'right_vals'), g.b(ib, 'left_ts'), g.b(ib, 'right_ts'),
                    g.b(ib, 'msg_vals'), g.b(ib, 'msg_ts'), g.b(ib, 'pending_after'), what)


def run_oracle(model, graph, st, neg, B, K, n_batches, lazy, start=0):
    uptodate = np.zeros(model.N, dtype=bool)
    outs = []
    for ib in range(n_batches):
        lo = start + ib * B
        b = O.collate(graph, st.src[lo:lo + B], st.dst[lo:lo + B], neg[lo:lo + B], st.ts[lo:lo + B],
                      st.eids[lo:lo + B], K)
        if lazy:
            rn = O.lazy_restart_nodes(b.involved, uptodate)
            model.restart(rn, np.full(len(rn), b.ts.min(), dtype=np.float32))
        outs.append(model.contrast_step(b))
    return outs


@pytest.mark.parametrize('shape,msg_src,upd_src,lazy,restarter', [
    (StreamShape('w', 900, 120, 9000, 172, None), 'left', 'right', False, 'static'),
    (StreamShape('r', 900, 120, 9000, 172, None), 'left', 'right', True, 'static'),
    (StreamShape('m', 700, 30, 9000, 4, 100), 'right', 'right', True, 'static'),
    (StreamShape('l', 200, 200, 9000, 0, 100, horizon=1.4e8), 'left', 'right', False, 'static'),
    (StreamShape('s', 900, 120, 9000, 32, None), 'left', 'right', True, 'seq'),
    (StreamShape('t', 300, 60, 9000, 4, 20), 'right', 'right', True, 'seq'),
])
def test_engine_matches_oracle_on_stream(gu, shape, msg_src, upd_src, lazy, restarter):
    B, K, H, n_batches, start = 200, 10, 2, 30, 2000
    st = make_stream(shape, seed=2)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    N, d = st.n_nodes, st.dim
    de = st.efeats.shape[1] if st.efeats is not None else d
    W = perturb_biases(random_weights(d, de, n_nodes=N, restarter=restarter, nonzero_static=True, seed=1))
    graph, model = gu.oracle_from(W, st.src, st.dst, st.ts, st.eids, N=N, dim=d, efeats=st.efeats, nfeats=None,
                                  K=K, H=H, msg_src=msg_src, upd_src=upd_src, restarter=restarter)
    outs = run_oracle(model, graph, st, neg, B, K, n_batches, lazy, start)
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = gu.engine_from(W, csr, N=N, dim=d, efeats=st.efeats, nfeats=None, K=K, H=H, B=B, msg_src=msg_src,
                       upd_src=upd_src, restarter=restarter, lazy_restart=lazy)
    # graph-captured replay from pinned host buffers (the e2e path)
    runner = StreamRunner(e)
    lo = start
    e.set_batch(st.src[lo:lo + B], st.dst[lo:lo + B], neg[lo:lo + B], st.ts[lo:lo + B], st.eids[lo:lo + B])
    runner.capture(warmup=1)
    e.reset()
    for ib in range(n_batches):
        lo = start + ib * B
        slot = runner.submit_host(st.src[lo:lo + B], st.dst[lo:lo + B], neg[lo:lo + B], st.ts[lo:lo + B],
                                  st.eids[lo:lo + B])
        ps, ns, loss = runner.wait(slot)
        o = outs[ib]
        what = f'{shape.name} batch {ib} '
        assert_close(ps.numpy(), o['pos_scores'].numpy(), TOL, what + 'pos')
        assert_close(ns.numpy(), o['neg_scores'].numpy(), TOL, what + 'neg')
        assert_close(np.array([float(loss)]), o['loss'].reshape(1).numpy(), TOL, what + 'loss')
        assert_close(gu.cpu(e.emb), o['h_left_with_negs'].numpy(), TOL, what + 'emb')
        assert np.array_equal(gu.cpu(e.outdated[:int(e.counts[1])]), o['outdated']), what
    e.check_errors()
    check_state(gu, e, model.left_vals.numpy(), model.right_vals.numpy(), model.left_ts.numpy(),
                model.right_ts.numpy(), model.msg_vals.numpy(), model.msg_ts.numpy(), np.nonzero(model.has_msg)[0],
                shape.name + ' final ')


@pytest.mark.parametrize('K', [20, 40])
def test_engine_matches_oracle_at_wide_neighborhoods(gu, K):
    """K = 20 (the keyword default of TIGE / TIGER) and K = 40 (past one softmax value per lane), eager steps."""
    B, H, n_batches, start = 100, 2, 8, 1500
    st = make_stream(StreamShape('k', 300, 60, 4000, 16, None), seed=K)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    N, d = st.n_nodes, st.dim
    W = perturb_biases(random_weights(d, d, n_nodes=N, restarter='static', nonzero_static=True, seed=1))
    graph, model = gu.oracle_from(W, st.src, st.dst, st.ts, st.eids, N=N, dim=d, efeats=st.efeats, nfeats=None,
                                  K=K, H=H, msg_src='left', upd_src='right', restarter='static')
    outs = run_oracle(model, graph, st, neg, B, K, n_batches, True, start)
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = gu.engine_from(W, csr, N=N, dim=d, efeats=st.efeats, nfeats=None, K=K, H=H, B=B, msg_src='left',
                       upd_src='right', restarter='static', lazy_restart=True)
    for ib in range(n_batches):
        lo = start + ib * B
        e.set_batch(st.src[lo:lo + B], st.dst[lo:lo + B], neg[lo:lo + B], st.ts[lo:lo + B], st.eids[lo:lo + B])
        e.step()
        o, what = outs[ib], f'K={K} batch {ib} '
        assert_close(gu.cpu(e.scores[:B]), o['pos_scores'].numpy(), TOL, what + 'pos')
        assert_close(gu.cpu(e.scores[B:]), o['neg_scores'].numpy(), TOL, what + 'neg')
        assert_close(gu.cpu(e.loss).reshape(1), o['loss'].reshape(1).numpy(), TOL, what + 'loss')
        assert_close(gu.cpu(e.emb), o['h_left_with_negs'].numpy(), TOL, what + 'emb')
    e.check_errors()
    check_state(gu, e, model.left_vals.numpy(), model.right_vals.numpy(), model.left_ts.numpy(),
                model.right_ts.numpy(), model.msg_vals.numpy(), model.msg_ts.numpy(), np.nonzero(model.has_msg)[0],
                f'K={K} final ')


def test_invariant_flags_raise_like_the_reference(gu):
    st = make_stream(StreamShape('e', 100, 20, 2000, 8, None, horizon=1000.), seed=4)
    N, d, B, K = st.n_nodes, 8, 50, 5
    W = random_weights(d, 8, seed=0)
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = gu.engine_from(W, csr, N=N, dim=d, efeats=st.efeats, nfeats=None, K=K, H=2, B=B, msg_src='left', upd_src='right')
    neg = np.full(B, 101, dtype=np.int64)
    e.set_batch(st.src[1000:1050], st.dst[1000:1050], neg, st.ts[1000:1050], st.eids[1000:1050])
    e.step()
    e.check_errors()
    # replaying an EARLIER batch must trip "Events occur before the updated memory" / past-memory checks
    e.set_batch(st.src[:50], st.dst[:50], neg, st.ts[:50], st.eids[:50])
    e.step()
    with pytest.raises(ValueError):
        e.check_errors()


@pytest.mark.parametrize('name', ['wikipedia', 'reddit'])
def test_full_size_stream_properties(gu, name):
    """BASELINE-size tables: determinism (bit-identical reruns), monotone memory clocks, exactly the
    selected positives hold a pending message, no invariant flag."""
    shape = SHAPES[name]
    st = make_stream(shape, seed=0, with_efeats=False)
    N, d, B, K = st.n_nodes, 172, 200, 10
    efeats = torch.randn(st.n_events + 1, 172, generator=torch.Generator().manual_seed(0))
    efeats[0] = 0
    W = random_weights(d, 172, n_nodes=N, restarter='static', seed=0)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    indptr = gu.cpu(csr.indptr)
    assert indptr[-1] == 2 * st.n_events and np.all(np.diff(indptr) >= 0)
    ats = gu.cpu(csr.ts)
    seg = np.repeat(np.arange(N), np.diff(indptr))
    assert np.all((np.diff(ats) >= 0) | (np.diff(seg) > 0))          # per-node time order
    e = gu.engine_from(W, csr, N=N, dim=d, efeats=efeats, nfeats=None, K=K, H=2, B=B, msg_src='left',
                       upd_src='right', restarter='static', lazy_restart=True, want_targets=False)
    runner = StreamRunner(e)
    start, n_batches = st.n_events // 2, 150
    e.set_batch(st.src[:B], st.dst[:B], neg[:B], st.ts[:B], st.eids[:B])
    runner.capture(warmup=1)
    finals = []
    for rep in range(2):
        e.reset()
        prev_l = prev_r = None
        for ib in range(n_batches):
            lo = start + ib * B
            e.set_batch(st.src[lo:lo + B], st.dst[lo:lo + B], neg[lo:lo + B], st.ts[lo:lo + B], st.eids[lo:lo + B])
            runner.run_device()
            if rep == 0 and ib % 25 == 0:
                lt, rt = gu.cpu(e.left_ts), gu.cpu(e.right_ts)
                if prev_l is not None:
                    assert np.all(lt >= prev_l) and np.all(rt >= prev_r)
                prev_l, prev_r = lt, rt
                pos = np.concatenate([st.src[lo:lo + B], st.dst[lo:lo + B]])
                assert gu.cpu(e.has_msg)[pos].all()
                assert torch.isfinite(e.emb).all() and torch.isfinite(e.out_buf).all()
        e.check_errors()
        finals.append([t.clone() for t in (e.left_vals, e.right_vals, e.msg_vals, e.left_ts, e.right_ts, e.out_buf)])
    for a, b in zip(*finals):
        assert torch.equal(a, b)


@pytest.mark.parametrize('name,restarter,start', [('reddit', 'static', 200_000), ('wikipedia', 'seq', 100_000)])
def test_full_size_stream_matches_oracle_for_50_batches(gu, name, restarter, start):
    """BASELINE-size stream, tables and dimensions (d = d_e = 172, K = 10, B = 200, hist_len 40): the pipelined graph
    replay against the CPU oracle for 50 consecutive batches from the middle of the stream (lazy restart from a fresh
    memory, histories from the full graph), every score / embedding / index list and the final state."""
    shape = SHAPES[name]
    st = make_stream(shape, seed=0)
    N, d, B, K, H, n_batches = st.n_nodes, 172, 200, 10, 2, 50
    W = perturb_biases(random_weights(d, 172, n_nodes=N, restarter=restarter, nonzero_static=True, seed=2))
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    graph, model = gu.oracle_from(W, st.src, st.dst, st.ts, st.eids, N=N, dim=d, efeats=st.efeats, nfeats=None, K=K, H=H,
                                  msg_src='left', upd_src='right', restarter=restarter)
    outs = run_oracle(model, graph, st, neg, B, K, n_batches, True, start)
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = gu.engine_from(W, csr, N=N, dim=d, efeats=st.efeats, nfeats=None, K=K, H=H, B=B, msg_src='left',
                       upd_src='right', restarter=restarter, lazy_restart=True)
    cols = lambda ib: tuple(a[start + ib * B:start + (ib + 1) * B] for a in (st.src, st.dst, neg, st.ts, st.eids))
    runner = StreamRunner(e)
    e.set_batch(*cols(0))
    runner.capture(warmup=1)
    e.reset()
    for ib in range(n_batches):
        ps, ns, loss = runner.wait(runner.submit_host(*cols(ib)))
        o, what = outs[ib], f'{name} batch {ib} '
        assert_close(ps.numpy(), o['pos_scores'].numpy(), TOL, what + 'pos')
        assert_close(ns.numpy(), o['neg_scores'].numpy(), TOL, what + 'neg')
        assert_close(np.array([float(loss)]), o['loss'].reshape(1).numpy(), TOL, what + 'loss')
        assert_close(gu.cpu(e.emb), o['h_left_with_negs'].numpy(), TOL, what + 'emb')
        assert np.array_equal(gu.cpu(e.outdated[:int(e.counts[1])]), o['outdated']), what
    e.check_errors()
    check_state(gu, e, model.left_vals.numpy(), model.right_vals.numpy(), model.left_ts.numpy(), model.right_ts.numpy(),
                model.msg_vals.numpy(), model.msg_ts.numpy(), np.nonzero(model.has_msg)[0], name + ' final ')


@pytest.mark.parametrize('name,restarter,start,n_batches', [('reddit', 'static', 200_000, 2000),
                                                            ('wikipedia', 'seq', 20_000, 650)])
def test_graph_pipeline_equals_serial_launches_at_full_size(gu, name, restarter, start, n_batches):
    """The captured pipeline (restarter beside the GRU, write-back beside the attention, tail beside the products,
    finder / scorer of neighbouring batches overlapped, n_slots batches in flight) against eager single-stream
    launches of the same kernels, bit for bit, over thousands of consecutive BASELINE-size batches."""
    shape = SHAPES[name]
    st = make_stream(shape, seed=0)
    N, d, B, K, H = st.n_nodes, 172, 200, 10, 2
    W = perturb_biases(random_weights(d, 172, n_nodes=N, restarter=restarter, nonzero_static=True, seed=5))
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = gu.engine_from(W, csr, N=N, dim=d, efeats=st.efeats, nfeats=None, K=K, H=H, B=B, msg_src='left',
                       upd_src='right', restarter=restarter, lazy_restart=True, want_targets=False)
    assert start + n_batches * B <= st.n_events
    cols = lambda ib: tuple(a[start + ib * B:start + (ib + 1) * B] for a in (st.src, st.dst, neg, st.ts, st.eids))
    state = lambda: [t.clone() for t in (e.left_vals, e.right_vals, e.msg_vals, e.left_ts, e.right_ts, e.msg_ts, e.has_msg)]
    e.reset()
    ref = torch.empty(n_batches, e.out_buf.numel())
    for ib in range(n_batches):
        e.set_batch(*cols(ib))
        e.step()
        ref[ib] = e.out_buf
    e.check_errors()
    final_ref = state()
    runner = StreamRunner(e)
    e.set_batch(*cols(0))
    runner.capture(warmup=1)
    e.reset()
    pending, got = [], []
    for ib in range(n_batches):
        pending.append(runner.submit_host(*cols(ib)))
        if len(pending) >= runner.n_slots:
            ps, ns, loss = runner.wait(pending.pop(0))
            got.append(torch.cat([ps, ns, loss.reshape(1)]).clone())
    while pending:
        ps, ns, loss = runner.wait(pending.pop(0))
        got.append(torch.cat([ps, ns, loss.reshape(1)]).clone())
    e.check_errors()
    bad = [ib for ib in range(n_batches) if not torch.equal(got[ib], ref[ib])]
    assert not bad, f'{len(bad)} batches differ, first {bad[:5]}'
    for a, b in zip(final_ref, state()):
        assert torch.equal(a, b)


def test_pipelined_host_and_device_paths_match_eager_steps(gu):
    """StreamRunner keeps n_slots batches in flight (upload + finder of batch i+1 and download of batch i-1 beside
    the model kernels of batch i, per-slot buffers): the results must be bit-identical to eager, strictly
    sequential steps."""
    shape = StreamShape('p', 700, 90, 12000, 16, None)
    st = make_stream(shape, seed=5)
    B, K, H, n_batches, start = 200, 10, 2, 26, 3000
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    N, d = st.n_nodes, st.dim
    W = perturb_biases(random_weights(d, st.efeats.shape[1], n_nodes=N, restarter='static', nonzero_static=True, seed=3))
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = gu.engine_from(W, csr, N=N, dim=d, efeats=st.efeats, nfeats=None, K=K, H=H, B=B, msg_src='left',
                       upd_src='right', restarter='static', lazy_restart=True)
    cols = lambda ib: tuple(a[start + ib * B:start + (ib + 1) * B] for a in (st.src, st.dst, neg, st.ts, st.eids))
    # eager reference run
    ref = []
    e.reset()
    for ib in range(n_batches):
        e.set_batch(*cols(ib))
        e.step()
        ref.append(e.out_buf.clone())
    final_ref = [t.clone() for t in (e.left_vals, e.right_vals, e.msg_vals, e.left_ts, e.right_ts, e.has_msg)]
    e.check_errors()
    runner = StreamRunner(e)
    e.set_batch(*cols(0))
    runner.capture(warmup=1)
    # host path, n_slots deep
    e.reset()
    pending, got = [], []
    for ib in range(n_batches):
        pending.append(runner.submit_host(*cols(ib)))
        if len(pending) >= runner.n_slots:
            ps, ns, loss = runner.wait(pending.pop(0))
            got.append(torch.cat([ps, ns, loss.reshape(1)]).clone())
    while pending:
        ps, ns, loss = runner.wait(pending.pop(0))
        got.append(torch.cat([ps, ns, loss.reshape(1)]).clone())
    torch.cuda.synchronize()
    e.check_errors()
    for ib in range(n_batches):
        assert torch.equal(got[ib], ref[ib].cpu()), f'host path batch {ib}'
    for a, b in zip(final_ref, (e.left_vals, e.right_vals, e.msg_vals, e.left_ts, e.right_ts, e.has_msg)):
        assert torch.equal(a, b)
    # device-resident path
    e.reset()
    dev_batches = []
    for ib in range(n_batches):
        h = torch.empty(5 * B, dtype=torch.int64)
        runner.fill_host(0, *cols(ib))
        dev_batches.append(runner.h_in[0].clone().cuda())
    outs = []
    for ib in range(n_batches):
        slot = runner.submit_device(dev_batches[ib])
        if ib >= n_batches - runner.n_slots:
            outs.append((ib, slot))
    torch.cuda.synchronize()
    for ib, slot in outs:
        assert torch.equal(runner.d_out[slot], ref[ib]), f'device path batch {ib}'
    for a, b in zip(final_ref, (e.left_vals, e.right_vals, e.msg_vals, e.left_ts, e.right_ts, e.has_msg)):
        assert torch.equal(a, b)


def test_first_batch_after_reset_is_bit_stable_under_graph_replay(gu):
    """The first batch after a reset restarts EVERY involved node while the GRU has no rows: the restarter (a
    parallel branch of the graph) is then far slower than the GRU, the worst case for the join in front of the
    attention chain.  300 resets + replays must reproduce the eager single-stream result bit for bit."""
    shape = StreamShape('r', 300, 40, 4000, 16, None, horizon=4000.)
    st = make_stream(shape, seed=0)
    B, K = 100, 10
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    N, d = st.n_nodes, st.dim
    W = perturb_biases(random_weights(d, d, n_nodes=N, restarter='static', nonzero_static=True, seed=0))
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    e = gu.engine_from(W, csr, N=N, dim=d, efeats=st.efeats, nfeats=None, K=K, H=2, B=B, msg_src='left',
                       upd_src='right', restarter='static', lazy_restart=True, want_targets=False)
    cols = lambda ib: tuple(a[ib * B:(ib + 1) * B] for a in (st.src, st.dst, neg, st.ts, st.eids))
    e.reset()
    e.set_batch(*cols(10))
    e.step()
    ref_out, ref_emb, ref_right = e.out_buf.clone(), e.emb.clone(), e.right_vals.clone()
    runner = StreamRunner(e)
    runner.capture(warmup=1)
    for it in range(300):
        e.reset()
        slot = runner.submit_host(*cols(10))
        ps, ns, loss = runner.wait(slot)
        got = torch.cat([ps, ns, loss.reshape(1)])
        assert torch.equal(got, ref_out.cpu()), f'iteration {it}: scores differ'
        assert torch.equal(e.emb, ref_emb) and torch.equal(e.right_vals, ref_right), f'iteration {it}'
        # single whole-step graph as well
        e.reset()
        e.set_batch(*cols(10))
        runner.run_device()
        torch.cuda.synchronize()
        assert torch.equal(e.emb, ref_emb) and torch.equal(e.out_buf, ref_out), f'iteration {it} (single graph)'


# ------------------------------------------------------------------------------------------
# BASELINE dimensions, fixtures of the unmodified reference (tests/golden/make_golden_full.py)
# ------------------------------------------------------------------------------------------
from golden_utils import FULL_CASES, FullGolden, check_full_batch   # noqa: E402


def engine_results(gu, e, B):
    U, Oc, R = (int(x) for x in e.counts[:3])
    got = dict(neigh_nids=gu.cpu(e.neigh_nids), neigh_eids=gu.cpu(e.neigh_eids), neigh_ts=gu.cpu(e.neigh_ts),
               involved=gu.cpu(e.involved[:U]), outdated=gu.cpu(e.outdated[:Oc]), restart_nids=gu.cpu(e.restart_nodes[:R]),
               winner=gu.cpu(e.winner), h_left=gu.cpu(e.emb[:2 * B]), pos_scores=gu.cpu(e.scores[:B]),
               neg_scores=gu.cpu(e.scores[B:]), loss=gu.cpu(e.loss), h_prev_left=gu.cpu(e.hprev_left),
               h_prev_right=gu.cpu(e.hprev_right), left_vals=gu.cpu(e.left_vals), right_vals=gu.cpu(e.right_vals),
               msg_vals=gu.cpu(e.msg_vals), left_ts=gu.cpu(e.left_ts), right_ts=gu.cpu(e.right_ts),
               msg_ts=gu.cpu(e.msg_ts), pending_after=np.nonzero(gu.cpu(e.has_msg))[0])
    if e.restarter == 'seq' and R:
        got.update(restart_hl=gu.cpu(e.seq.h_left[:R]), restart_hr=gu.cpu(e.seq.h_right[:R]),
                   restart_pt=gu.cpu(e.seq.prev_ts[:R]))
    return got


@pytest.mark.parametrize('replay', ['eager', 'graph'])
@pytest.mark.parametrize('name', FULL_CASES)
def test_engine_replays_reference_at_baseline_dimensions(gu, name, replay):
    """d / d_e / K / hist_len / batch of the BASELINE configs, on the BASELINE-shaped streams, lazy-restart mode:
    eager launches and the captured-graph pipeline (the benchmarked path) against the unmodified reference."""
    g = FullGolden(name)
    csr = gu.device_csr(*g.stream_prefix(), g.N)
    e = gu.engine_from(g.W, csr, N=g.N, dim=g.dim, efeats=g.efeats, nfeats=None, K=g.K, H=g.n_heads, B=g.bs,
                       msg_src=g.msg_src, upd_src=g.upd_src, restarter=g.restarter, lazy_restart=True,
                       hist_len=g.hist_len)
    runner = None
    if replay == 'graph':
        runner = StreamRunner(e)
        e.set_batch(*g.batch(0))
        runner.capture(warmup=1)
        e.reset()
    for ib in range(g.warm + g.rec):
        if runner is None:
            e.set_batch(*g.batch(ib))
            e.step()
        else:
            slot = runner.submit_host(*g.batch(ib))
            runner.wait(slot)
            torch.cuda.synchronize()
            # the pipeline's slot owns the finder outputs and the result buffer of this batch
            e.bind_finder(runner.finder_bufs[slot])
            e.bind_io(runner.d_in[slot], runner.d_out[slot])
        e.check_errors()
        if ib >= g.warm:
            check_full_batch(g, ib - g.warm, engine_results(gu, e, g.bs), TOL, replay + ' ')
