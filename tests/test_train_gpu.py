"""The hand-written training step (www2023tiger_b200/train.py, csrc/train*.cu, tiger_sgemm_ex) against
(1) losses and parameter gradients of the UNMODIFIED reference's training loop body (tests/golden/make_golden_train.py),
(2) the torch-autograd route of the drop-in classes on the same state, (3) torch.optim.Adam, (4) finite differences
with dropout switched on."""
import os

import numpy as np
import pytest
import torch
from torch.utils.data import DataLoader

from golden_utils import CASES, TRAIN_CASES, Golden, assert_close
import dropin_utils as D
from tiger.data.data_loader import GraphCollator, InteractionData
from tiger.data.graph import Graph
from www2023tiger_b200._lib import call, ptr

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda')
cpu = lambda t: t.detach().cpu().numpy()
GRAD_TOL = 2e-5      # max-norm, relative to the largest entry of the gradient tensor


def setup(g, dropout=0.0):
    full = InteractionData(g.src, g.dst, g.ts, g.eids, np.zeros_like(g.src), seed=0, eval=True, neg_dst=g.neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    coll = GraphCollator(graph, g.K, 1, restarter=g.restarter, hist_len=g.hist_len)
    dl = DataLoader(full, batch_size=g.bs, collate_fn=coll)
    model = D.model_from_golden(g, graph, DEV, dropout=dropout)
    res = model.load_state_dict(g.W, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    return dl, model


def to_dev(batch):
    src, dst, neg, ts, eids, _, cg = batch
    return (src.long().to(DEV), dst.long().to(DEV), neg.long().to(DEV), ts.float().to(DEV), eids.long().to(DEV),
            cg.to(DEV))


def unique_named_params(model):
    seen, out = set(), []
    for k, p in model.named_parameters():
        if id(p) not in seen:
            seen.add(id(p))
            out.append((k, p))
    return out


def grad_of(p):
    return cpu(p.grad) if p.grad is not None else np.zeros(tuple(p.shape), np.float32)


def check_grads(got: dict, want: dict, what: str, tol=GRAD_TOL):
    assert set(got) == set(want), set(got) ^ set(want)
    for k in want:
        w = np.asarray(want[k], dtype=np.float64)
        a = np.asarray(got[k], dtype=np.float64)
        scale = np.abs(w).max()
        if scale == 0:
            assert np.abs(a).max() <= 1e-7, f'{what} {k}: expected a zero gradient, got {np.abs(a).max():.2e}'
            continue
        err = np.abs(a - w).max() / scale
        assert err <= tol, f'{what} {k}: rel err {err:.2e} > {tol} (|g|max {scale:.2e})'


@pytest.mark.parametrize('name', TRAIN_CASES)
def test_native_step_matches_reference_gradients(name):
    """Loop body of train_self_supervised.py:143-171 through `loss.backward()` of the drop-in model (one autograd
    node = the native step) vs the reference's own losses and gradients."""
    g = Golden(name)
    dl, model = setup(g)
    model.train()
    model.reset()
    params = unique_named_params(model)
    for ib, batch in zip(range(g.n_batches), dl):
        b = to_dev(batch)
        model.zero_grad(set_to_none=True)
        contrast, mutual = model.contrast_and_mutual_learning(*b)
        assert contrast.grad_fn is not None and type(contrast.grad_fn).__name__.startswith('_NativeStep')
        (contrast + mutual).backward()
        what = f'{name} b{ib}'
        assert_close(cpu(contrast).reshape(1), g.b(ib, 'contrast').reshape(1), 1e-5, what + ' contrast')
        assert_close(cpu(mutual).reshape(1), g.b(ib, 'mutual').reshape(1), 2e-5, what + ' mutual')
        if g.has(ib, 'g_' + params[0][0]):
            got = {k: grad_of(p) for k, p in params}
            want = {k: g.b(ib, 'g_' + k) for k, _ in params}
            check_grads(got, want, what)
    model._trainer.check_errors()
    assert_close(cpu(model.left_memory.vals), g.z['final_left_vals'], 1e-5, name + ' left')
    assert_close(cpu(model.right_memory.vals), g.z['final_right_vals'], 1e-5, name + ' right')
    assert_close(cpu(model.msg_store.node_msg_vals), g.z['final_msg_vals'], 1e-5, name + ' msg')


@pytest.mark.parametrize('name', ['seq_left_right', 'static_right_right_dim10', 'seq_noefeat_dim8'])
def test_native_step_matches_autograd_route(name, monkeypatch):
    """Same state, same batch: the native step vs the torch-op autograd route of the operator modules."""
    g = Golden(name)
    dl, native = setup(g)
    _, ref = setup(g)
    native.train(), ref.train()
    native.reset(), ref.reset()
    for ib, batch in zip(range(7), dl):
        b = to_dev(batch)
        native.zero_grad(set_to_none=True)
        c1, m1 = native.contrast_and_mutual_learning(*b)
        (c1 + 0.5 * m1).backward()
        monkeypatch.setenv('TIGER_AUTOGRAD_ROUTE', '1')
        ref.zero_grad(set_to_none=True)
        c2, m2 = ref.contrast_and_mutual_learning(*b)
        (c2 + 0.5 * m2).backward()
        monkeypatch.delenv('TIGER_AUTOGRAD_ROUTE')
        what = f'{name} b{ib}'
        assert_close(cpu(c1).reshape(1), cpu(c2).reshape(1), 1e-5, what + ' contrast')
        assert_close(cpu(m1).reshape(1), cpu(m2).reshape(1), 2e-5, what + ' mutual')
        got = {k: grad_of(p) for k, p in unique_named_params(native)}
        want = {k: grad_of(p) for k, p in unique_named_params(ref)}
        # tensors without a gradient are the same on both routes (torch optimizers skip them)
        assert [p.grad is None for _, p in unique_named_params(native)] == \
            [p.grad is None for _, p in unique_named_params(ref)], what
        check_grads(got, want, what)
        assert_close(cpu(native.right_memory.vals), cpu(ref.right_memory.vals), 1e-5, what + ' right memory')
        assert_close(cpu(native.left_memory.vals), cpu(ref.left_memory.vals), 1e-5, what + ' left memory')


def test_adam_kernel_equals_torch_adam():
    """Flat segmented Adam vs torch.optim.Adam, including torch's per-tensor step counters: a tensor whose gradient
    is None in a step (here: the gated tensor in steps 1-2) is skipped and its bias correction starts later."""
    gen = torch.Generator(device='cuda').manual_seed(0)
    sizes = [100_003, 517, 4096]
    offs = np.concatenate([[0], np.cumsum([(n + 3) // 4 * 4 for n in sizes])])
    total = int(offs[-1])
    flat = torch.randn(total, device='cuda', generator=gen)
    refs = [torch.nn.Parameter(flat[offs[i]:offs[i] + n].clone()) for i, n in enumerate(sizes)]
    opt = torch.optim.Adam(refs, lr=1e-3)
    gbuf = torch.zeros(total + 4, device='cuda')
    m, v = torch.zeros(total, device='cuda'), torch.zeros(total, device='cuda')
    seg_start = torch.tensor(offs, dtype=torch.int64, device='cuda')
    seg_group = torch.tensor([0, 1, 0], dtype=torch.int32, device='cuda')
    seg_step = torch.zeros(3, dtype=torch.int32, device='cuda')
    seg_bc = torch.zeros(6, device='cuda')
    for step in range(1, 7):
        gate_on = step >= 3
        for i, n in enumerate(sizes):
            grad = torch.randn(n, device='cuda', generator=gen) * 10 ** float(step - 3)
            used = i != 1 or gate_on
            refs[i].grad = grad.clone() if used else None
            gbuf[offs[i]:offs[i] + n] = grad * 4 if used else 0.0     # grad_scale folds the 1 / world_size
        gbuf[total] = 5.0 if gate_on else 0.0
        opt.step()
        call('tiger_train_adam', ptr(flat), ptr(gbuf), ptr(m), ptr(v), ptr(seg_start), ptr(seg_group), ptr(seg_step),
             ptr(seg_bc), 3, ptr(gbuf[total:]), max(sizes), 1e-3, 0.9, 0.999, 1e-8, 0.25, 1)
        assert float(gbuf.abs().max()) == 0.0           # zero_grad (gradients and gates)
        for i, n in enumerate(sizes):
            assert_close(cpu(flat[offs[i]:offs[i] + n]), cpu(refs[i]), 1e-6, f'adam step {step} tensor {i}')
    assert seg_step.tolist() == [6, 4, 6]


def test_training_through_torch_optimizer_and_native_adam_agree():
    """A few optimisation steps: loss.backward() + torch.optim.Adam on the drop-in vs NativeTrainer.step (flat Adam)."""
    g = Golden('seq_left_right')
    dl, a = setup(g)
    _, b_ = setup(g)

    def eval_batch(model, bt):
        """Inference route (weight packs of the kernels, cached per module) from a fresh memory."""
        model.eval()
        model.reset()
        with torch.no_grad():
            out = model.contrast_learning(*bt)
        model.train()
        model.reset()
        return [cpu(t) for t in (out if isinstance(out, (tuple, list)) else (out,))]

    probe = to_dev(next(iter(dl)))
    before = eval_batch(b_, probe)                 # builds the packs from the initial weights
    a.train(), b_.train()
    a.reset(), b_.reset()
    tr = b_.native_trainer(g.bs, lr=1e-3)
    opt = torch.optim.Adam(a.parameters(), lr=1e-3)
    la, lb = [], []
    for ib, batch in zip(range(8), dl):
        bt = to_dev(batch)
        opt.zero_grad()
        c, m = a.contrast_and_mutual_learning(*bt)
        (c + m).backward()
        opt.step()
        la.append(float(c.detach()) + float(m.detach()))
        c2, m2 = tr.step(*bt, mutual_coef=1.0)
        lb.append(float(c2) + float(m2))
    tr.check_errors()
    # same algorithm, same data; Adam normalises gradients, so round-off in near-zero gradients may move single
    # weights differently - the loss trajectories must still agree closely
    assert np.allclose(la, lb, rtol=1e-4), (la, lb)
    # the native Adam kernel writes the parameters through raw pointers: the inference operators must notice (their
    # packs are keyed on the parameters' version counters) and agree with the torch-optimised twin
    ea, eb = eval_batch(a, probe), eval_batch(b_, probe)
    for x, y in zip(ea, eb):
        assert np.allclose(x, y, rtol=2e-3, atol=2e-4), np.abs(x - y).max()
    assert np.abs(eb[1] - before[1]).max() > 1e-3, 'evaluation after training still used the initial weights'


def _mix32(x):
    x = x & 0xffffffff
    x ^= x >> 16
    x = (x * 0x7feb352d) & 0xffffffff
    x ^= x >> 15
    x = (x * 0x846ca68b) & 0xffffffff
    x ^= x >> 16
    return x


def keep_mask(seed: int, stream: int, n: int, p: float) -> np.ndarray:
    """The counter-based dropout decisions of csrc/train.cu (dropout_keep), restated with numpy."""
    idx = np.arange(n, dtype=np.uint64)
    h = _mix32(idx ^ _mix32(np.uint64((seed + 0x9E3779B9 * (stream + 1)) & 0xffffffff)))
    return ((h >> 8).astype(np.float32) * np.float32(1.0 / 16777216.0)) >= np.float32(p)


@pytest.mark.parametrize('name', ['seq_left_right', 'static_right_right_dim10', 'seq_nfeats_left_left'])
def test_dropout_step_matches_autograd_route_with_the_same_masks(name, monkeypatch):
    """Dropout 0.1: the native step (seeded counter-based masks) vs the torch-op autograd route with
    torch.nn.functional.dropout replaced by the SAME masks - losses and every gradient must agree, i.e. forward
    and backward of every dropout site (attention weights, scorer, restarter attention, restarter merger) use one
    consistent mask."""
    import torch.nn.functional as F
    g = Golden(name)
    p = 0.1
    dl, native = setup(g, dropout=p)
    _, ref = setup(g, dropout=p)
    native.train(), ref.train()
    native.reset(), ref.reset()
    tr = native.native_trainer(g.bs)
    H, K, L = g.n_heads, g.K, g.hist_len
    for ib, batch in zip(range(6), dl):
        b = to_dev(batch)
        B = len(b[0])
        d = native.nfeat_dim
        native.zero_grad(set_to_none=True)
        c1, m1 = native.contrast_and_mutual_learning(*b)
        seed = tr.n_steps * 101 & 0x7fffffff                      # NativeTrainer._core with trainer seed 0
        (c1 + m1).backward()
        n_pos = b[5].restart_data.nids.numel()
        queue = [torch.from_numpy(keep_mask(seed, 1, 3 * B * H * K, p)).reshape(3 * B * H, 1, K)]
        score = torch.from_numpy(keep_mask(seed, 2, 2 * B * d, p)).reshape(2 * B, d)
        queue += [score[:B], score[B:]]
        if g.restarter == 'seq':
            queue.append(torch.from_numpy(keep_mask(seed, 3, n_pos * H * L * L, p)).reshape(n_pos * H, L, L))
            queue.append(torch.from_numpy(keep_mask(seed, 4, n_pos * d, p)).reshape(n_pos, d))
        queue = [q.to(DEV) for q in queue]

        def fake_dropout(x, p=0.5, training=True, inplace=False):
            if not training or p == 0.0:
                return x
            mask = queue.pop(0)
            assert mask.shape == x.shape, (mask.shape, x.shape)
            return x * mask.to(x.dtype) / (1.0 - p)

        monkeypatch.setenv('TIGER_AUTOGRAD_ROUTE', '1')
        monkeypatch.setattr(F, 'dropout', fake_dropout)
        ref.zero_grad(set_to_none=True)
        c2, m2 = ref.contrast_and_mutual_learning(*b)
        (c2 + m2).backward()
        monkeypatch.undo()
        assert not queue, f'{len(queue)} dropout sites of the autograd route were not reached'
        what = f'{name} b{ib}'
        assert_close(cpu(c1).reshape(1), cpu(c2).reshape(1), 1e-5, what + ' contrast')
        assert_close(cpu(m1).reshape(1), cpu(m2).reshape(1), 2e-5, what + ' mutual')
        got = {k: grad_of(pp) for k, pp in unique_named_params(native)}
        want = {k: grad_of(pp) for k, pp in unique_named_params(ref)}
        check_grads(got, want, what)
        assert_close(cpu(native.left_memory.vals), cpu(ref.left_memory.vals), 1e-5, what + ' left memory')
    # seeded: the same step number reproduces the same masks, another one does not
    assert np.array_equal(keep_mask(7, 1, 64, p), keep_mask(7, 1, 64, p))
    assert not np.array_equal(keep_mask(7, 1, 64, p), keep_mask(8, 1, 64, p))


# ------------------------------------------------------------------------------------------
# BASELINE dimensions (d = 172 / 100, K = 10, L = 40, B = 200): native step vs the torch-op autograd route
# ------------------------------------------------------------------------------------------
from golden_utils import FULL_CASES, FullGolden   # noqa: E402


@pytest.mark.parametrize('name', FULL_CASES)
def test_native_step_matches_autograd_route_at_baseline_dimensions(name, monkeypatch):
    g = FullGolden(name)
    src_, dst_, ts_, eids_ = g.stream_prefix()
    full = InteractionData(src_, dst_, ts_, eids_, np.zeros_like(src_), seed=0, eval=True, neg_dst=g.neg[:g.E])
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    coll = GraphCollator(graph, g.K, 1, restarter=g.restarter, hist_len=g.hist_len)

    def make():
        m = D.init_model(None, g.efeats, graph, g.N, g.st.n_events, DEV, dim=g.shape.dim, n_layers=1, n_heads=g.n_heads,
                         n_neighbors=g.K, hit_type='bin', dropout=0.0, restarter_type=g.restarter, hist_len=g.hist_len,
                         msg_src=g.msg_src, upd_src=g.upd_src)
        assert not m.load_state_dict(g.W, strict=False).unexpected_keys
        m.train()
        m.reset()
        return m
    native, ref = make(), make()
    for ib in range(4):
        lo = g.start + ib * g.bs
        b = to_dev(coll([full[i] for i in range(lo, lo + g.bs)]))
        native.zero_grad(set_to_none=True)
        c1, m1 = native.contrast_and_mutual_learning(*b)
        (c1 + m1).backward()
        monkeypatch.setenv('TIGER_AUTOGRAD_ROUTE', '1')
        ref.zero_grad(set_to_none=True)
        c2, m2 = ref.contrast_and_mutual_learning(*b)
        (c2 + m2).backward()
        monkeypatch.delenv('TIGER_AUTOGRAD_ROUTE')
        what = f'{name} b{ib}'
        assert_close(cpu(c1).reshape(1), cpu(c2).reshape(1), 1e-5, what + ' contrast')
        assert_close(cpu(m1).reshape(1), cpu(m2).reshape(1), 2e-5, what + ' mutual')
        got = {k: grad_of(p) for k, p in unique_named_params(native)}
        want = {k: grad_of(p) for k, p in unique_named_params(ref)}
        # tensors without a gradient are the same on both routes (torch optimizers skip them)
        assert [p.grad is None for _, p in unique_named_params(native)] == \
            [p.grad is None for _, p in unique_named_params(ref)], what
        check_grads(got, want, what)
    native._trainer.check_errors()


# ------------------------------------------------------------------------------------------
# device-resident stream loop (NativeTrainer.attach_stream / step_stream) and its CUDA-graph replay
# ------------------------------------------------------------------------------------------
def stream_setup(restarter, seed=0, dropout=0.1, B=50):
    import gpu_utils as gu
    from www2023tiger_b200.init import build_model
    from www2023tiger_b200.synthetic import NegativeSampler, StreamShape, make_stream
    st = make_stream(StreamShape('g', 260, 40, 6000, 12, None, horizon=5000.), seed=3)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, st.n_nodes)
    torch.manual_seed(seed)
    model = build_model(None, torch.from_numpy(st.efeats).to(DEV), Graph.from_csr(csr), st.n_nodes, st.n_events, DEV,
                        dim=st.dim, n_layers=1, n_heads=2, n_neighbors=5, hit_type='bin', dropout=dropout,
                        restarter_type=restarter, hist_len=8, msg_src='left', upd_src='right')
    model.train()
    tr = model.native_trainer(B, lr=1e-3, seed=7)
    tr.attach_stream(csr, 8)
    n = 40
    rec = np.empty((n, 5 * B), dtype=np.int64)
    s = slice(1000, 1000 + n * B)
    for k, col in enumerate((st.src, st.dst, neg, st.eids)):
        rec[:, k * B:(k + 1) * B] = col[s].reshape(n, B)
    rec[:, 4 * B:] = st.ts[s].astype(np.float64).reshape(n, B).view(np.int64)
    return model, tr, torch.from_numpy(rec).to(DEV)


@pytest.mark.parametrize('restarter', ['seq', 'static'])
def test_stream_step_graph_replay_matches_eager_launches(restarter):
    """Same model, same batches, dropout ON: eager launches with host seeds vs the captured step whose kernels add
    the device-side step counter to the captured seed - the masks, hence the losses, must follow the same sequence."""
    ma, ta, rec = stream_setup(restarter)
    mb, tb, _ = stream_setup(restarter)
    for (ka, pa), (kb, pb) in zip(unique_named_params(ma), unique_named_params(mb)):
        assert ka == kb and torch.equal(pa, pb)
    ta.reset_stream(), tb.reset_stream()
    tb.capture_stream(mutual_coef=1.0, grad_scale=1.0)
    la, lb = [], []
    try:
        for i in range(rec.shape[0]):
            c, m = ta.step_stream(rec[i], mutual_coef=1.0, grad_scale=1.0)
            la.append((float(c), float(m)))
            if i == 25:                        # an eager step with other arguments in between: the counter re-aligns
                c2, m2 = tb.step_stream(rec[i], mutual_coef=1.0, grad_scale=1.0, sliced=False, allreduce=lambda t: None)
            else:
                c2, m2 = tb.step_stream(rec[i], mutual_coef=1.0, grad_scale=1.0)
            lb.append((float(c2), float(m2)))
        assert tb._graph is not None and tb._g_replays >= rec.shape[0] - 4
        assert int(tb.g_count) == rec.shape[0] - tb._g_base
        ta.check_errors(), tb.check_errors()
    finally:
        tb.release_graph()
    la, lb = np.array(la), np.array(lb)
    assert np.isfinite(la).all() and la[:, 0].std() > 0
    # identical masks and data; the weight gradients are summed with atomics (order differs run to run) and Adam
    # normalises them, so single weights drift at round-off level
    assert np.allclose(la, lb, rtol=2e-3, atol=1e-5), np.abs(la - lb).max()
    for (k, pa), (_, pb) in zip(unique_named_params(ma), unique_named_params(mb)):
        assert torch.allclose(pa, pb, rtol=0, atol=2e-3), k
    # a different mask sequence would not pass: the same run with another seed differs by far more
    mc, tc, _ = stream_setup(restarter)
    tc.seed = 8
    tc.reset_stream()
    lc = np.array([[float(x) for x in tc.step_stream(rec[i], mutual_coef=1.0, grad_scale=1.0)] for i in range(rec.shape[0])])
    assert np.abs(lc - la).max() > 10 * np.abs(lb - la).max()


# ------------------------------------------------------------------------------------------
# neighborhoods and head counts past the goldens', and the sizes the native step refuses
# ------------------------------------------------------------------------------------------
def synthetic_setup(K, H, restarter, hist_len=8):
    from www2023tiger_b200.synthetic import NegativeSampler, StreamShape, make_stream
    st = make_stream(StreamShape('kh', 200, 40, 3000, 16, None, horizon=3000.), seed=K + H)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    full = InteractionData(st.src, st.dst, st.ts, st.eids, np.zeros_like(st.src), seed=0, eval=True, neg_dst=neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=st.n_nodes - 1)
    coll = GraphCollator(graph, K, 1, restarter=restarter, hist_len=hist_len)

    def make():
        m = D.init_model(None, st.efeats, graph, st.n_nodes, st.n_events, DEV, dim=None, n_layers=1, n_heads=H,
                         n_neighbors=K, hit_type='bin', dropout=0.0, restarter_type=restarter, hist_len=hist_len,
                         msg_src='left', upd_src='right')
        m.train()
        return m
    batch = lambda lo, B: to_dev(coll([full[i] for i in range(lo, lo + B)]))
    return make, batch


@pytest.mark.parametrize('restarter', ['seq', 'static'])
@pytest.mark.parametrize('K,H', [(20, 2), (7, 4), (32, 1)])
def test_native_step_matches_autograd_route_at_other_k_and_heads(K, H, restarter, monkeypatch):
    """K = 20 (the keyword default of TIGE / TIGER) runs its own attention-core instantiation, K = 7 and 32 the generic
    one (32: every bit of keep_bits), with 1, 2 and 4 heads."""
    torch.manual_seed(K + H)
    make, batch = synthetic_setup(K, H, restarter)
    native, ref = make(), make()
    ref.load_state_dict(native.state_dict())
    native.reset(), ref.reset()
    B = 80
    for ib in range(4):
        b = batch(1200 + ib * B, B)
        native.zero_grad(set_to_none=True)
        c1, m1 = native.contrast_and_mutual_learning(*b)
        assert type(c1.grad_fn).__name__.startswith('_NativeStep')
        (c1 + m1).backward()
        monkeypatch.setenv('TIGER_AUTOGRAD_ROUTE', '1')
        ref.zero_grad(set_to_none=True)
        c2, m2 = ref.contrast_and_mutual_learning(*b)
        (c2 + m2).backward()
        monkeypatch.delenv('TIGER_AUTOGRAD_ROUTE')
        what = f'K={K} H={H} {restarter} b{ib}'
        assert_close(cpu(c1).reshape(1), cpu(c2).reshape(1), 1e-5, what + ' contrast')
        assert_close(cpu(m1).reshape(1), cpu(m2).reshape(1), 2e-5, what + ' mutual')
        assert [p.grad is None for _, p in unique_named_params(native)] == \
            [p.grad is None for _, p in unique_named_params(ref)], what
        check_grads({k: grad_of(p) for k, p in unique_named_params(native)},
                    {k: grad_of(p) for k, p in unique_named_params(ref)}, what)
    native._trainer.check_errors()


@pytest.mark.parametrize('K,restarter,hist_len', [(40, 'static', 8), (10, 'seq', 70)])
def test_models_past_the_native_limits_train_through_the_torch_op_route(K, restarter, hist_len):
    """More than 32 neighbors, or a seq restarter history longer than 64: the drop-in trains such a model through the
    torch-op route instead of failing inside the native step."""
    from www2023tiger_b200.train import NativeTrainer
    torch.manual_seed(0)
    make, batch = synthetic_setup(K, 2, restarter, hist_len=hist_len)
    model = make()
    model.reset()
    with pytest.raises(NotImplementedError):
        NativeTrainer(model, 80)
    assert not model._native_training()
    model.zero_grad(set_to_none=True)
    c, m = model.contrast_and_mutual_learning(*batch(1200, 80))
    assert c.grad_fn is not None and not type(c.grad_fn).__name__.startswith('_NativeStep')
    (c + m).backward()
    assert getattr(model, '_trainer', None) is None
    grads = [p.grad for p in model.parameters() if p.grad is not None]
    assert grads and all(bool(torch.isfinite(g).all()) for g in grads)
    assert model.time_encoder.basis_freq.grad is not None and float(model.time_encoder.basis_freq.grad.abs().max()) > 0
