"""The native training step at two layers (n_layers=2, the keyword default of TIGE / TIGER): the depth-aware row
builders (tiger_train_attn_build_ex / _bwd_ex) against a float64 restatement, and NativeTrainer against the drop-in's
torch-op autograd route on the var_two_layers golden and at BASELINE dimensions, with and without dropout, in the
device-resident stream loop and its CUDA-graph replay."""
import numpy as np
import pytest
import torch
from torch.utils.data import DataLoader

import dropin_utils as D
from golden_utils import Golden, assert_close
from tiger.data.data_loader import GraphCollator, InteractionData
from tiger.data.graph import Graph
from www2023tiger_b200._lib import call, ptr

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda')
cpu = lambda t: t.detach().cpu().numpy()
GRAD_TOL = 2e-5      # max-norm, relative to the largest entry of the gradient tensor (as in test_train_gpu.py)


def unique_named_params(model):
    seen, out = set(), []
    for k, p in model.named_parameters():
        if id(p) not in seen:
            seen.add(id(p))
            out.append((k, p))
    return out


def grad_of(p):
    return cpu(p.grad) if p.grad is not None else np.zeros(tuple(p.shape), np.float32)


def check_grads(got: dict, want: dict, what: str, tol=GRAD_TOL, worst=None):
    assert set(got) == set(want), set(got) ^ set(want)
    for k in want:
        w = np.asarray(want[k], dtype=np.float64)
        a = np.asarray(got[k], dtype=np.float64)
        scale = np.abs(w).max()
        if scale == 0:
            assert np.abs(a).max() <= 1e-7, f'{what} {k}: expected a zero gradient, got {np.abs(a).max():.2e}'
            continue
        err = np.abs(a - w).max() / scale
        if worst is not None:
            worst['grad'] = max(worst.get('grad', 0.0), float(err))
        assert err <= tol, f'{what} {k}: rel err {err:.2e} > {tol} (|g|max {scale:.2e})'


def to_dev(batch):
    src, dst, neg, ts, eids, _, cg = batch
    return (src.long().to(DEV), dst.long().to(DEV), neg.long().to(DEV), ts.float().to(DEV), eids.long().to(DEV),
            cg.to(DEV))


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


# ------------------------------------------------------------------------------------------
# 1. the row builders of either depth against float64
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('with_keys', [False, True])
@pytest.mark.parametrize('with_nfeats', [False, True])
@pytest.mark.parametrize('depth,d', [(1, 8), (2, 40)])
def test_build_ex_and_bwd_ex_match_float64(with_keys, with_nfeats, depth, d):
    """Both depths the trainer calls, with and without key_rows: depth 1 = 3BK queries at ts[(i / K) % B]
    (ts_group = K), depth 2 = 3B queries at ts[i % B] (ts_group = 1); d = 40 runs the lane loops past 32 columns.
    Padding slots and rows without any neighbor; q_in / kv_in / cat, the gradients onto dh_new, d_key_rows and the
    TimeEncode gradients."""
    gen = torch.Generator().manual_seed(3 + 2 * with_keys + with_nfeats + 4 * depth)
    N, n_e, de, B, K = 40, 90, 6, 3, 4
    g = K if depth == 1 else 1             # ts_group
    nq = 3 * B * K if depth == 1 else 3 * B
    E, C = 2 * d, 2 * d + de
    center = torch.randint(0, N, (nq,), generator=gen)
    nn_ = torch.randint(1, N, (nq, K), generator=gen)
    nn_[torch.rand(nq, K, generator=gen) < 0.3] = 0            # padding slots
    nn_[::7] = 0                                               # rows without any neighbor
    ne_ = torch.randint(0, n_e, (nq, K), generator=gen)
    ts = torch.rand(B, generator=gen) * 10 + 10
    nt_ = torch.rand(nq, K, generator=gen) * 10
    rows_a = torch.randn(N, d, generator=gen)
    n_rows = 15
    sel = torch.full((N,), -1, dtype=torch.int32)
    sel[torch.randperm(N, generator=gen)[:n_rows]] = torch.arange(n_rows, dtype=torch.int32)
    rows_b = torch.randn(n_rows, d, generator=gen)
    nfeats = torch.randn(N, d, generator=gen) if with_nfeats else None
    efeats = torch.randn(n_e, de, generator=gen)
    key_rows = torch.randn(nq * K, d, generator=gen) if with_keys else None
    tw = 1.0 / 10 ** torch.linspace(0, 3, d)
    tb = torch.randn(d, generator=gen) * 0.3
    dkv = torch.randn(nq * K, C, generator=gen)
    dq = torch.randn(nq, E, generator=gen)
    dcat = torch.randn(nq, E + d, generator=gen)

    # ---- float64 restatement under autograd
    f64 = lambda t: None if t is None else t.double()
    rb, w64, b64 = f64(rows_b).requires_grad_(), f64(tw).requires_grad_(), f64(tb).requires_grad_()
    kr = f64(key_rows).requires_grad_() if with_keys else None

    def repr_(ids):
        s = sel[ids].long()
        out = torch.where((s >= 0)[:, None], rb[s.clamp(min=0)], f64(rows_a)[ids])
        return out + (f64(nfeats)[ids] if with_nfeats else 0.0)

    flat = nn_.reshape(-1)
    node = kr if with_keys else repr_(flat)
    q_ts = ts[(torch.arange(nq) // g) % B]
    dt = (q_ts[:, None] - nt_).reshape(-1, 1).double()         # float32 difference, as the model forms it
    kv_ref = torch.cat([node, f64(efeats)[ne_.reshape(-1)], torch.cos(dt * w64 + b64)], 1)
    c_row = repr_(center)
    q_ref = torch.cat([c_row, torch.cos(b64).expand(nq, d)], 1)
    real = (flat != 0).double()[:, None]                       # padding slots carry no gradient
    loss = (kv_ref * f64(dkv) * real).sum() + (q_ref * f64(dq)).sum() + (c_row * f64(dcat)[:, E:]).sum()
    loss.backward()

    # ---- the kernels
    cu = lambda t: None if t is None else t.to(DEV).contiguous()
    q_in, kv_in, cat = torch.zeros(nq, E, device=DEV), torch.zeros(nq * K, C, device=DEV), torch.zeros(nq, E + d,
                                                                                                       device=DEV)
    args = dict(center=cu(center), ts=cu(ts), nn=cu(nn_), ne=cu(ne_), nt=cu(nt_), ra=cu(rows_a), rb=cu(rows_b),
                kr=cu(key_rows), sel=cu(sel), nf=cu(nfeats), ef=cu(efeats), tw=cu(tw), tb=cu(tb))
    a = args
    call('tiger_train_attn_build_ex', ptr(a['center']), nq, ptr(a['ts']), B, g, ptr(a['nn']), ptr(a['ne']),
         ptr(a['nt']), K, ptr(a['ra']), ptr(a['rb']), ptr(a['kr']), ptr(a['sel']), ptr(a['nf']), ptr(a['ef']), d, de,
         ptr(a['tw']), ptr(a['tb']), ptr(q_in), ptr(kv_in), ptr(cat), E + d, E)
    h0 = torch.randn(n_rows, d, generator=gen)
    dh = cu(h0)                                                # accumulated onto
    dkr = torch.full((nq * K, d), 7.0, device=DEV) if with_keys else None       # stored: the 7s must go
    gw, gb = torch.zeros(d, device=DEV), torch.zeros(d, device=DEV)
    dkv_d, dq_d, dcat_d = cu(dkv), cu(dq), cu(dcat)
    call('tiger_train_attn_build_bwd_ex', ptr(dkv_d), ptr(dq_d), ptr(dcat_d), E + d, E, ptr(a['center']), nq,
         ptr(a['ts']), B, g, ptr(a['nn']), ptr(a['nt']), K, ptr(a['sel']), d, de, ptr(a['tw']), ptr(a['tb']), ptr(dh),
         ptr(dkr), ptr(gw), ptr(gb))
    torch.cuda.synchronize()
    assert_close(cpu(kv_in), kv_ref.detach().numpy(), 1e-5, 'kv_in')
    assert_close(cpu(q_in), q_ref.detach().numpy(), 1e-5, 'q_in')
    assert_close(cpu(cat[:, E:]), c_row.detach().numpy(), 1e-5, 'cat')
    assert_close(cpu(dh) - h0.numpy(), rb.grad.numpy(), GRAD_TOL, 'dh_new')
    assert_close(cpu(gw), w64.grad.numpy(), GRAD_TOL, 'time_encoder.basis_freq')
    assert_close(cpu(gb), b64.grad.numpy(), GRAD_TOL, 'time_encoder.phase')
    if with_keys:
        assert_close(cpu(dkr), kr.grad.numpy(), GRAD_TOL, 'd_key_rows')
        assert float(dkr[flat.to(DEV) == 0].abs().max()) == 0.0, 'padding slots must get zeros'


# ------------------------------------------------------------------------------------------
# 2-3. native step vs the torch-op route on the var_two_layers golden's data and weights
# ------------------------------------------------------------------------------------------
def golden_setup(name, dropout, n_layers=2):
    g = Golden(name)
    full = InteractionData(g.src, g.dst, g.ts, g.eids, np.zeros_like(g.src), seed=0, eval=True, neg_dst=g.neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=g.N - 1)
    dl = DataLoader(full, batch_size=g.bs, collate_fn=GraphCollator(graph, g.K, n_layers, restarter=g.restarter,
                                                                   hist_len=g.hist_len))

    def make():
        m = D.init_model(g.nfeats, g.efeats, graph, g.N, len(g.src), DEV, dim=g.dim, n_layers=n_layers,
                         n_heads=g.n_heads, n_neighbors=g.K, hit_type=g.hit_type, dropout=dropout,
                         restarter_type=g.restarter, hist_len=g.hist_len, msg_src=g.msg_src, upd_src=g.upd_src)
        assert not m.load_state_dict(g.W, strict=False).unexpected_keys
        return m
    native = make()
    ref = make()
    ref.load_state_dict(native.state_dict())       # the same fns.1 where the fixture has none
    native.train(), ref.train()
    native.reset(), ref.reset()
    return g, dl, native, ref


def test_native_step_matches_autograd_route_on_two_layer_golden(monkeypatch):
    g, dl, native, ref = golden_setup('var_two_layers', 0.0)
    assert g.n_layers == 2
    for ib, batch in zip(range(7), dl):
        b = to_dev(batch)
        native.zero_grad(set_to_none=True)
        c1, m1 = native.contrast_and_mutual_learning(*b)
        assert type(c1.grad_fn).__name__.startswith('_NativeStep')
        (c1 + 0.5 * m1).backward()
        monkeypatch.setenv('TIGER_AUTOGRAD_ROUTE', '1')
        ref.zero_grad(set_to_none=True)
        c2, m2 = ref.contrast_and_mutual_learning(*b)
        assert c2.grad_fn is not None and not type(c2.grad_fn).__name__.startswith('_NativeStep')
        (c2 + 0.5 * m2).backward()
        monkeypatch.delenv('TIGER_AUTOGRAD_ROUTE')
        what = f'var_two_layers b{ib}'
        assert_close(cpu(c1).reshape(1), cpu(c2).reshape(1), 1e-5, what + ' contrast')
        assert_close(cpu(m1).reshape(1), cpu(m2).reshape(1), 2e-5, what + ' mutual')
        assert [p.grad is None for _, p in unique_named_params(native)] == \
            [p.grad is None for _, p in unique_named_params(ref)], what
        got = {k: grad_of(p) for k, p in unique_named_params(native)}
        want = {k: grad_of(p) for k, p in unique_named_params(ref)}
        assert any(k.startswith('temporal_embedding_fn.fns.1.') and np.abs(v).max() > 0 for k, v in want.items())
        check_grads(got, want, what)
        assert_close(cpu(native.left_memory.vals), cpu(ref.left_memory.vals), 1e-5, what + ' left memory')
        assert_close(cpu(native.right_memory.vals), cpu(ref.right_memory.vals), 1e-5, what + ' right memory')
    native._trainer.check_errors()


@pytest.mark.parametrize('name', ['var_two_layers', 'static_right_right_dim10'])
def test_two_layer_dropout_step_matches_autograd_route_with_the_same_masks(name, monkeypatch):
    """Dropout 0.1: depth 1 draws its attention mask under its own seed (seed + 7919 * 2), then depth 2, the scorer
    and the restarter under the step's seed; the torch-op route replays exactly these masks."""
    import torch.nn.functional as F
    p = 0.1
    g, dl, native, ref = golden_setup(name, p)
    tr = native.native_trainer(g.bs)
    H, K, L = g.n_heads, g.K, g.hist_len
    for ib, batch in zip(range(5), dl):
        b = to_dev(batch)
        B = len(b[0])
        d = native.nfeat_dim
        native.zero_grad(set_to_none=True)
        c1, m1 = native.contrast_and_mutual_learning(*b)
        seed = tr.n_steps * 101 & 0x7fffffff                      # NativeTrainer._core with trainer seed 0
        (c1 + m1).backward()
        n_pos = b[5].restart_data.nids.numel()
        queue = [torch.from_numpy(keep_mask((seed + 7919 * 2) & 0x7fffffff, 1, 3 * B * K * H * K, p))
                 .reshape(3 * B * K * H, 1, K)]
        queue.append(torch.from_numpy(keep_mask(seed, 1, 3 * B * H * K, p)).reshape(3 * B * H, 1, K))
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
        assert not queue, f'{len(queue)} dropout masks were not consumed by the autograd route'
        what = f'{name} b{ib}'
        assert_close(cpu(c1).reshape(1), cpu(c2).reshape(1), 1e-5, what + ' contrast')
        assert_close(cpu(m1).reshape(1), cpu(m2).reshape(1), 2e-5, what + ' mutual')
        got = {k: grad_of(pp) for k, pp in unique_named_params(native)}
        want = {k: grad_of(pp) for k, pp in unique_named_params(ref)}
        check_grads(got, want, what)
        assert_close(cpu(native.left_memory.vals), cpu(ref.left_memory.vals), 1e-5, what + ' left memory')
        assert_close(cpu(native.right_memory.vals), cpu(ref.right_memory.vals), 1e-5, what + ' right memory')


# ------------------------------------------------------------------------------------------
# 4. BASELINE dimensions on seeded streams
# ------------------------------------------------------------------------------------------
class _MaskedReLU(torch.nn.Module):
    """ReLU whose on / off pattern is given (one mask per call, in call order) instead of decided by the sign."""

    def __init__(self, masks):
        super().__init__()
        self.masks = list(masks)

    def forward(self, x):
        return x * self.masks.pop(0).to(x.dtype)


def float64_inputs(model, b):
    """What the differentiable part of the contrast loss reads from `model`'s state before the step: the involved
    nodes' right-memory rows, the pending messages and the memory rows the GRU updates."""
    with torch.no_grad():
        outdated, msgs, _ = model.compute_messages(b[5].np_computation_graph_nodes)
        reprs = model.right_memory.vals[b[5].computation_graph_nodes].double()
        old = model.upd_memory.vals[outdated].double() if len(outdated) else None
    return outdated, None if msgs is None else msgs.double(), reprs, old


def contrast_loss_float64(model, b, inputs, relu_masks=None):
    """The contrast loss restated in float64 with autograd: the torch-op route's steps 1-3 and 7 (GRU on the pending
    messages, both attention depths, hit embedding, scorer, BCE) on float64 copies of `model`'s modules, fed with
    the same collated tables and float64_inputs.  Two decisions are taken from the float32 model rather than made
    again: the argument fl(fl(dt w) + b) of each time code's cos() (both float32 routes compute that same argument;
    its rounding alone moves a code by up to ~1e-2 at dt w ~ 1e5; gradients go through the exact argument, as in both
    routes), and, with relu_masks = {'fns.0': [3B, d], 'fns.1': [3BK, d], 'score': [2B, d]} bool, the on / off
    pattern of the three merger ReLUs.  Returns (loss, {name under unique_named_params: parameter copy})."""
    import copy
    src, dst, neg, ts, eids, cg = b
    B = len(src)
    outdated, msgs, reprs, old = inputs
    upd = copy.deepcopy(model.right_mem_updater).double()
    emb = copy.deepcopy(model.temporal_embedding_fn, memo={id(model.graph): model.graph}).double()
    hit = copy.deepcopy(model.hit_embedding).double()
    score = copy.deepcopy(model.score_fn).double()
    te = emb.time_encoder

    def te_forward(t):
        arg32 = t.unsqueeze(-1) * te.basis_freq.detach().float() + te.phase.detach().float()
        arg = t.unsqueeze(-1).double() * te.basis_freq + te.phase
        return torch.cos(arg + (arg32.double() - arg).detach())
    te.forward = te_forward
    if relu_masks is not None:
        emb.fns[0].merger.act = _MaskedReLU([relu_masks['fns.0']])
        emb.fns[1].merger.act = _MaskedReLU([relu_masks['fns.1']])
        score.act = _MaskedReLU([relu_masks['score'][:B], relu_masks['score'][B:]])
    if len(outdated):
        reprs = reprs.index_copy(0, cg.local_index[outdated], upd.cell(msgs, old))
    h = emb.compute_embedding_with_computation_graph(reprs, torch.cat([src, dst, neg]), ts.repeat(3), cg)
    x, y, ny = h.reshape(3, B, -1)
    code = lambda t: t.max(1).values.long()
    sh, dh, nsh, ndh = cg.hit_data
    pos = score(x + hit(code(sh)), y + hit(code(dh))).squeeze(1)
    negs = score(x + hit(code(nsh)), ny + hit(code(ndh))).squeeze(1)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(
        torch.cat([pos, negs]), torch.cat([torch.ones_like(pos), torch.zeros_like(negs)]))
    if relu_masks is not None:
        assert not (emb.fns[0].merger.act.masks or emb.fns[1].merger.act.masks or score.act.masks)
    params = {'right_mem_updater.' + k: p for k, p in upd.named_parameters()}
    params.update({'temporal_embedding_fn.' + k: p for k, p in emb.named_parameters() if not k.startswith('time_enc')})
    params.update({'time_encoder.' + k: p for k, p in te.named_parameters()})
    params.update({'hit_embedding.' + k: p for k, p in hit.named_parameters()})
    params.update({'score_fn.' + k: p for k, p in score.named_parameters()})
    return loss, params


def float64_grads(model, b, inputs, relu_masks=None):
    loss, params = contrast_loss_float64(model, b, inputs, relu_masks)
    loss.backward()
    return float(loss.detach()), {k: grad_of(p) for k, p in params.items()}


# Weight gradients at two layers and BASELINE dimensions.  The two float32 routes differ by up to ~2e-3 on the GRU,
# time-encoder and attention gradients (relative to each tensor's largest entry), and at some batches each of them
# differs as much from a float64 restatement of the loss.  That gap comes from units of the merger ReLUs whose
# pre-activation lies within round-off of zero, so that they are on in one evaluation and off in another: a switched
# unit of fns.1 moves that layer's fc1 / attention gradients and, through its inputs, the GRU's.  The float64
# restatement therefore takes the on / off pattern of the route it is compared with; against it every gradient of the
# native step is held at 2e-5, the bar of test_train_gpu.py.  The switched units are counted and printed.
@pytest.mark.parametrize('name', ['wikipedia', 'reddit'])
def test_two_layer_native_step_matches_autograd_route_at_baseline_dimensions(name, monkeypatch):
    """d = d_e = 172, K = 10, B = 200, 4 consecutive batches from the middle of the stream.  Losses, memories and the
    restarter's gradients against the torch-op route at the bars of test_train_gpu.py; the gradients the contrast
    loss reaches against the float64 restatement with the native step's ReLU pattern, at 2e-5."""
    import gpu_utils as gu
    from www2023tiger_b200.init import perturb_biases, random_weights
    from www2023tiger_b200.synthetic import SHAPES, NegativeSampler, make_stream
    shape = SHAPES[name]
    B, K, H = 200, 10, 2
    st = make_stream(shape, seed=0)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    N, d = st.n_nodes, st.dim
    de = st.efeats.shape[1]
    W = perturb_biases(random_weights(d, de, n_nodes=N, restarter=shape.restarter, nonzero_static=True, seed=1,
                                      n_layers=2))
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, N)
    full = InteractionData(st.src, st.dst, st.ts, st.eids, np.zeros_like(st.src), seed=0, eval=True, neg_dst=neg)
    graph = Graph.from_csr(csr)
    coll = GraphCollator(graph, K, 2, restarter=shape.restarter, hist_len=40)

    def make():
        m = D.init_model(None, st.efeats, graph, N, st.n_events, DEV, dim=d, n_layers=2, n_heads=H, n_neighbors=K,
                         hit_type='bin', dropout=0.0, restarter_type=shape.restarter, hist_len=40,
                         msg_src=shape.msg_src, upd_src=shape.upd_src)
        assert not m.load_state_dict(W, strict=False).unexpected_keys
        m.train()
        m.reset()
        return m
    native, ref = make(), make()
    # the torch-op route's ReLU patterns (the recursion runs fns.1 before fns.0; the scorer runs twice: pos, neg)
    seen = {'fns.0': [], 'fns.1': [], 'score': []}
    for key, act in (('fns.0', ref.temporal_embedding_fn.fns[0].merger.act),
                     ('fns.1', ref.temporal_embedding_fn.fns[1].merger.act), ('score', ref.score_fn.act)):
        act.register_forward_hook(lambda mod, inp, out, key=key: seen[key].append(out.detach() > 0))
    start = (shape.n_events // 2) // B * B
    worst, flips = {}, []

    def rel(a, w):
        a, w = np.asarray(a, np.float64), np.asarray(w, np.float64)
        scale = np.abs(w).max()
        if scale == 0:                 # no gradient (e.g. no pending message): the other side must have none either
            return 0.0 if np.abs(a).max() <= 1e-7 else float('inf')
        return float(np.abs(a - w).max() / scale)

    def close(a, b, tol, what, key):
        worst[key] = max(worst.get(key, 0.0), rel(a, b))
        assert_close(a, b, tol, what + key)

    for ib in range(4):
        lo = start + ib * B
        b = to_dev(coll([full[i] for i in range(lo, lo + B)]))
        what = f'{name} b{ib} '
        inputs = float64_inputs(ref, b)                  # both models hold the same state before the step
        native.zero_grad(set_to_none=True)
        c1, m1 = native.contrast_and_mutual_learning(*b)
        assert type(c1.grad_fn).__name__.startswith('_NativeStep')
        (c1 + m1).backward()
        tr = native._trainer
        nat_masks = {'fns.0': tr.att.hid[:3 * B] > 0, 'fns.1': tr.att1.hid[:3 * B * K] > 0,
                     'score': tr.hid_s[:2 * B] > 0}
        for v in seen.values():
            v.clear()
        monkeypatch.setenv('TIGER_AUTOGRAD_ROUTE', '1')
        ref.zero_grad(set_to_none=True)
        c2, m2 = ref.contrast_and_mutual_learning(*b)
        (c2 + m2).backward()
        monkeypatch.delenv('TIGER_AUTOGRAD_ROUTE')
        ref_masks = {'fns.0': seen['fns.0'][0], 'fns.1': seen['fns.1'][0], 'score': torch.cat(seen['score'])}
        flips.append(sum(int((nat_masks[k] != ref_masks[k]).sum()) for k in nat_masks))
        close(cpu(c1).reshape(1), cpu(c2).reshape(1), 1e-5, what, 'contrast')
        close(cpu(m1).reshape(1), cpu(m2).reshape(1), 2e-5, what, 'mutual')
        assert [p.grad is None for _, p in unique_named_params(native)] == \
            [p.grad is None for _, p in unique_named_params(ref)], what
        got = {k: grad_of(p) for k, p in unique_named_params(native)}
        want = {k: grad_of(p) for k, p in unique_named_params(ref)}
        l64, g64 = float64_grads(ref, b, inputs, nat_masks)
        close(cpu(c1).reshape(1), np.array([l64]), 1e-5, what, 'contrast vs float64')
        _, g64_ref = float64_grads(ref, b, inputs, ref_masks)
        # the restarter's gradients (mutual loss only): against the torch-op route as in test_train_gpu.py
        check_grads({k: v for k, v in got.items() if k not in g64}, {k: v for k, v in want.items() if k not in g64},
                    what)
        for k, w in g64.items():
            e_nat = rel(got[k], w)
            for key, v in (('grad vs float64, native', e_nat), ('grad vs float64, torch-op', rel(want[k], g64_ref[k])),
                           ('grad native vs torch-op', rel(got[k], want[k]))):
                worst[key] = max(worst.get(key, 0.0), v)
            assert e_nat <= GRAD_TOL, f'{what}{k}: rel err {e_nat:.2e} against float64 > {GRAD_TOL}'
        close(cpu(native.left_memory.vals), cpu(ref.left_memory.vals), 1e-5, what, 'left memory')
        close(cpu(native.right_memory.vals), cpu(ref.right_memory.vals), 1e-5, what, 'right memory')
    native._trainer.check_errors()
    print(f'{name}/{shape.restarter} two layers: ReLU units switched between the routes per batch {flips}; max rel err '
          + ', '.join(f'{k} {v:.2e}' for k, v in worst.items()))


# ------------------------------------------------------------------------------------------
# 5-6. device-resident stream loop
# ------------------------------------------------------------------------------------------
def stream_setup(restarter, n_layers=2, seed=0, dropout=0.1, B=50, n=40):
    import gpu_utils as gu
    from www2023tiger_b200.init import build_model
    from www2023tiger_b200.synthetic import NegativeSampler, StreamShape, make_stream
    st = make_stream(StreamShape('g', 260, 40, 6000, 12, None, horizon=5000.), seed=3)
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    csr = gu.device_csr(st.src, st.dst, st.ts, st.eids, st.n_nodes)
    torch.manual_seed(seed)
    model = build_model(None, torch.from_numpy(st.efeats).to(DEV), Graph.from_csr(csr), st.n_nodes, st.n_events, DEV,
                        dim=st.dim, n_layers=n_layers, n_heads=2, n_neighbors=5, hit_type='bin', dropout=dropout,
                        restarter_type=restarter, hist_len=8, msg_src='left', upd_src='right')
    model.train()
    tr = model.native_trainer(B, lr=1e-3, seed=7)
    tr.attach_stream(csr, 8)
    rec = np.empty((n, 5 * B), dtype=np.int64)
    s = slice(1000, 1000 + n * B)
    for k, col in enumerate((st.src, st.dst, neg, st.eids)):
        rec[:, k * B:(k + 1) * B] = col[s].reshape(n, B)
    rec[:, 4 * B:] = st.ts[s].astype(np.float64).reshape(n, B).view(np.int64)
    return model, tr, torch.from_numpy(rec).to(DEV), csr, st


@pytest.mark.parametrize('n_layers', [1, 2])
def test_sliced_allreduce_hands_off_complete_slices(n_layers):
    """Each slice handed to `allreduce` during backward already holds its final gradients: a clone taken at hand-off
    equals the same range of the gradient buffer once backward has returned (before Adam zeroes it)."""
    model, tr, rec, _, _ = stream_setup('seq', n_layers=n_layers, n=4)
    ranges = tr.fp.comm_ranges()
    assert ranges is not None
    if n_layers == 2:
        lo, hi = ranges['attention']
        fns1 = [o for nm, o in zip(tr.fp.names, tr.fp.offsets) if nm.startswith('temporal_embedding_fn.fns.1.')]
        assert fns1 and all(lo <= o < hi for o in fns1)
    tr.reset_stream()
    for i in range(rec.shape[0]):
        handed, final = [], []
        adam = tr.fp.adam

        def snap(*a, **kw):
            final.append(tr.fp.grad_all.clone())
            return adam(*a, **kw)

        def clone_slice(t):
            handed.append((t.data_ptr(), t.clone()))
        tr.fp.adam = snap
        try:
            tr.step_stream(rec[i], allreduce=clone_slice)
        finally:
            del tr.fp.adam
        torch.cuda.synchronize()
        assert len(handed) == 3
        elt = tr.fp.grad_all.element_size()
        for p_, t in handed:
            lo = (p_ - tr.fp.grad_all.data_ptr()) // elt
            assert torch.equal(t, final[0][lo:lo + t.numel()]), f'step {i}: slice at {lo} handed off incomplete'
        assert float(final[0][ranges['attention'][0]:ranges['attention'][1]].abs().max()) > 0
    tr.check_errors()


@pytest.mark.parametrize('restarter,captured_allreduce', [('seq', False), ('static', False), ('seq', True)])
def test_two_layer_stream_graph_replay_matches_eager_launches(restarter, captured_allreduce):
    """Same model, same batches, dropout ON, two layers: eager launches vs the captured step (with or without the
    sliced all-reduce in the graph); the depth-1 masks follow the step counter like the others."""
    noop = lambda t: None
    ar = noop if captured_allreduce else None
    ma, ta, rec, _, _ = stream_setup(restarter)
    mb, tb, _, _, _ = stream_setup(restarter)
    for (ka, pa), (kb, pb) in zip(unique_named_params(ma), unique_named_params(mb)):
        assert ka == kb and torch.equal(pa, pb)
    ta.reset_stream(), tb.reset_stream()
    tb.capture_stream(mutual_coef=1.0, grad_scale=1.0, allreduce=ar)
    la, lb = [], []
    try:
        for i in range(rec.shape[0]):
            c, m = ta.step_stream(rec[i], mutual_coef=1.0, grad_scale=1.0)
            la.append((float(c), float(m)))
            if i == 25:                        # an eager step with other arguments in between: the counter re-aligns
                other = (lambda t: None) if ar is None else None
                c2, m2 = tb.step_stream(rec[i], mutual_coef=1.0, grad_scale=1.0, sliced=True, allreduce=other)
            else:
                c2, m2 = tb.step_stream(rec[i], mutual_coef=1.0, grad_scale=1.0, allreduce=ar)
            lb.append((float(c2), float(m2)))
        assert tb._graph is not None and tb._g_replays >= rec.shape[0] - 4
        assert int(tb.g_count) == rec.shape[0] - tb._g_base
        ta.check_errors(), tb.check_errors()
    finally:
        tb.release_graph()
    la, lb = np.array(la), np.array(lb)
    assert np.isfinite(la).all() and la[:, 0].std() > 0
    assert np.allclose(la, lb, rtol=2e-3, atol=1e-5), np.abs(la - lb).max()
    for (k, pa), (_, pb) in zip(unique_named_params(ma), unique_named_params(mb)):
        assert torch.allclose(pa, pb, rtol=0, atol=2e-3), k
    mc, tc, _, _, _ = stream_setup(restarter)
    tc.seed = 8
    tc.reset_stream()
    lc = np.array([[float(x) for x in tc.step_stream(rec[i], mutual_coef=1.0, grad_scale=1.0)]
                   for i in range(rec.shape[0])])
    assert np.abs(lc - la).max() > 10 * np.abs(lb - la).max()


@pytest.mark.parametrize('restarter', ['seq', 'static'])
def test_two_layer_forward_stream_matches_engine(restarter):
    """forward_stream(train=False) with lazy restart, no backward, vs TigerEngine(n_layers=2, lazy_restart=True) with
    the same weights: the finder's two hops bit for bit, scores / loss and both memories within 1e-5."""
    from www2023tiger_b200.engine import TigerEngine
    model, tr, rec, csr, st = stream_setup(restarter, dropout=0.0, n=10)
    W = {k: v.detach().clone() for k, v in model.state_dict().items()}
    e = TigerEngine(W, csr, n_nodes=st.n_nodes, dim=st.dim, efeats=torch.from_numpy(st.efeats).float().to(DEV),
                    n_neighbors=5, n_head=2, batch_size=tr.B, msg_src='left', upd_src='right', restarter=restarter,
                    hist_len=8, lazy_restart=True, n_layers=2)
    tr.reset_stream()
    e.reset()
    B = tr.B
    for i in range(rec.shape[0]):
        what = f'{restarter} batch {i} '
        closs, _ = tr.forward_stream(rec[i], lazy_restart=True, train=False)
        e.inp.copy_(rec[i])
        e.step()
        torch.cuda.synchronize()
        for a, b_, nm in ((tr.nn_, e.neigh_nids, 'hop 1 nids'), (tr.ne_, e.neigh_eids, 'hop 1 eids'),
                          (tr.nt_, e.neigh_ts, 'hop 1 ts'), (tr.hop2[0], e.neigh2_nids, 'hop 2 nids'),
                          (tr.hop2[1], e.neigh2_eids, 'hop 2 eids'), (tr.hop2[2], e.neigh2_ts, 'hop 2 ts')):
            assert torch.equal(a, b_), what + nm
        assert_close(cpu(tr.scores[:2 * B]), cpu(e.scores), 1e-5, what + 'scores')
        assert_close(cpu(closs), cpu(e.loss), 1e-5, what + 'loss')
        assert_close(cpu(model.left_memory.vals), cpu(e.left_vals), 1e-5, what + 'left memory')
        assert_close(cpu(model.right_memory.vals), cpu(e.right_vals), 1e-5, what + 'right memory')
    tr.check_errors(), e.check_errors()


# ------------------------------------------------------------------------------------------
# 7. what stays refused
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n_layers,hit_type', [(3, 'bin'), (2, 'vec')])
def test_native_trainer_refuses_other_variants(n_layers, hit_type):
    from www2023tiger_b200.train import NativeTrainer
    g = Golden('var_two_layers')
    model = D.init_model(g.nfeats, g.efeats, None, g.N, len(g.src), DEV, dim=g.dim, n_layers=n_layers,
                         n_heads=g.n_heads, n_neighbors=g.K, hit_type=hit_type, dropout=0.0,
                         restarter_type=g.restarter, hist_len=g.hist_len, msg_src=g.msg_src, upd_src=g.upd_src)
    with pytest.raises(NotImplementedError):
        NativeTrainer(model, g.bs)
