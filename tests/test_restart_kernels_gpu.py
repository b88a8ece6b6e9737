"""The restart path of the no-grad step, called entry point by entry point and compared with a float64 restatement of
the same operation on the CPU: tiger_seq_tokens, tiger_seq_tail (inference and training mode), tiger_seq_gate_count
with ops.SeqRestarterOp.forward on both routes, tiger_min_time (csrc/restart_seq.cu), and tiger_static_restart /
tiger_static_restart_rows (csrc/restart.cu).  The cases sit where the kernels branch: every KREG instantiation of the
tail with its 16-byte and scalar paths and their 256 / 512 / 1024 edges, d % 4 != 0 in the merger layers, 1 to 8
heads, the 64 / 65 row boundary of the gate, d_model > 1024 (products only), the 32-wide and the final step of the
CSR lower bound with ties at the query time, count-bounded tails (rows past *count stay untouched), and the refusals.
A seq restarter with more than 64 history events runs its torch code instead of the kernels.

Tolerances: max-norm error relative to the largest entry of the reference, TOL for outputs that pass through dot
products, TC_TOL for time codes; copies, the gate and prev_ts are compared bit for bit.  The largest error each group
reaches is printed at the end of the module."""
import math

import numpy as np
import pytest
import torch

from oracle import tiger_oracle as O
from test_train_kernels_gpu import (COUNT_FORMS, count_of, inv_keep, keep_mask, seed_word_is_zero,  # noqa: F401
                                    time_arg32)
from www2023tiger_b200 import ops
from www2023tiger_b200._lib import call, load, ptr, stream_ptr
from www2023tiger_b200.init import perturb_biases, random_weights

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda')
TOL = 1e-5           # outputs through dot products
TC_TOL = 1e-6        # time codes
NAN = float('nan')
WORST = {}


@pytest.fixture(scope='module', autouse=True)
def report_worst():
    yield
    print('\nlargest relative error per restart group:')
    for k in sorted(WORST):
        print(f'  {k:28s} {WORST[k]:.2e}')


_ALIVE = []      # device copies made by cu(): a raw pointer does not keep its tensor alive


@pytest.fixture(autouse=True)
def release_device_copies():
    yield
    torch.cuda.synchronize()
    _ALIVE.clear()


def cu(t):
    if t is None:
        return None
    d = torch.as_tensor(t).to(DEV).contiguous()
    _ALIVE.append(d)
    return d


def nan_dev(*shape):
    return torch.full(shape, NAN, dtype=torch.float32, device=DEV)


def placed(t, lead):
    """Device copy of t `lead` floats past the start of its buffer (lead = 1 misaligns it by 4 bytes)."""
    buf = torch.full((t.numel() + lead,), NAN, device=DEV)
    v = buf[lead:].view(t.shape)
    v.copy_(t)
    _ALIVE.append(buf)
    return v


def check(group, what, got, want, tol):
    """max|got - want| / max|want| <= tol (absolute when want is all zero); got must hold no NaN."""
    got = got.detach().double().cpu()
    want = want.detach().double().cpu()
    assert got.shape == want.shape, f'{what}: shape {tuple(got.shape)} vs {tuple(want.shape)}'
    if got.numel() == 0:
        return
    assert not torch.isnan(got).any(), f'{what}: {int(torch.isnan(got).sum())} entries not written'
    scale = float(want.abs().max())
    err = float((got - want).abs().max()) / (scale if scale > 0 else 1.0)
    WORST[group] = max(WORST.get(group, 0.0), err)
    assert err <= tol, f'{what}: rel err {err:.3e} > {tol}'


def untouched(what, t):
    t = t.detach().cpu()
    assert torch.isnan(t).all(), f'{what}: {int((~torch.isnan(t)).sum())} entries past the bound were written'


# ------------------------------------------------------------------------------------------
# the float64 restatement of SeqRestarter.forward (reference restarters.py:51-114)
# ------------------------------------------------------------------------------------------
class SeqCase:
    """Histories of `cap` nodes as the restarter receives them (CPU): ~30 % padding slots (id 0), every fifth row
    padded everywhere, both directions, anonymised ids in [0, L], event times spread over up to 1e6 s."""

    def __init__(self, d, de, L, cap, *, seed, nfeats=True, efeats=True, n_nodes=60, n_edges=400, span=1e6):
        g = torch.Generator().manual_seed(seed)
        self.d, self.de, self.L, self.cap = d, de, L, cap
        self.nids = torch.randint(1, n_nodes, (cap,), generator=g)
        hn = torch.randint(1, n_nodes, (cap, L), generator=g)
        hn[torch.rand(cap, L, generator=g) < 0.3] = 0
        hn[0::5] = 0
        self.hn = hn
        self.he = torch.randint(0, n_edges, (cap, L), generator=g)
        self.ht = torch.sort(torch.rand(cap, L, generator=g) * span, 1).values
        self.hd = torch.randint(0, 2, (cap, L), generator=g)
        self.an = torch.randint(0, L + 1, (cap, L), generator=g)
        self.nfeats = torch.randn(n_nodes, d, generator=g) if nfeats else None
        self.efeats = torch.randn(n_edges, de, generator=g) if efeats else None
        self.anony_emb = torch.randn(L + 1, d, generator=g)
        self.tw = torch.from_numpy((1 / 10 ** np.linspace(0, 9, d)).astype(np.float32))   # TimeEncode's basis
        self.tb = torch.randn(d, generator=g)

    def with_weights(self, W):
        """Time encoder and anonymous embedding taken from a restarter's weights instead."""
        self.anony_emb = W['restarter_fn.anony_emb.weight'].float()
        self.tw, self.tb = W['restarter_fn.time_encoder.basis_freq'].float(), W['restarter_fn.time_encoder.phase'].float()
        return self

    def hist_dev(self):
        return tuple(cu(t) for t in (self.hn, self.he, self.ht, self.hd, self.an))

    def tokens64(self):
        """[src | dst | anony | edge | time] per event in float64 (the last event keeps its time code only) and the
        key-padding mask (True = padded, the last position never)."""
        n, L, d, de = self.cap, self.L, self.d, self.de
        owner = self.nids[:, None].expand(n, L)
        s_id = owner * self.hd + self.hn * (1 - self.hd)          # the reference's literal rule (restarters.py:93-94)
        d_id = owner * (1 - self.hd) + self.hn * self.hd
        zeros = lambda w: torch.zeros(n, L, w, dtype=torch.float64)
        nf = (lambda u: self.nfeats.double()[u]) if self.nfeats is not None else (lambda u: zeros(d))
        ef = self.efeats.double()[self.he] if self.efeats is not None else zeros(de)
        feat = torch.cat([nf(s_id), nf(d_id), self.anony_emb.double()[self.an], ef], 2)
        feat[:, -1] = 0.0
        dt = (self.ht[:, -1:] - self.ht).numpy()[..., None]        # float32 difference, as the kernel forms it
        tcode = torch.cos(time_arg32(dt, self.tw.numpy(), self.tb.numpy()))
        mask = self.hn == 0
        mask[:, -1] = False
        return torch.cat([feat, tcode], 2), mask


def seq64(x, mask, W, H, d):
    """SeqRestarter.forward after the tokens, in float64 and unfolded: self-attention of the tokens under the key
    padding mask, mean over the positions, ReLU, out_fn; the merger on [h_left | 0]."""
    n, L, dm = x.shape
    hd = dm // H
    g = lambda k: W['restarter_fn.' + k].double()
    wi, bi = g('mha_fn.in_proj_weight'), g('mha_fn.in_proj_bias')
    q = (x @ wi[:dm].t() + bi[:dm]).view(n, L, H, hd) * math.sqrt(1.0 / hd)
    k = (x @ wi[dm:2 * dm].t() + bi[dm:2 * dm]).view(n, L, H, hd)
    v = (x @ wi[2 * dm:].t() + bi[2 * dm:]).view(n, L, H, hd)
    s = torch.einsum('nqhc,nkhc->nhqk', q, k).masked_fill(mask[:, None, None, :], float('-inf'))
    o = torch.einsum('nhqk,nkhc->nqhc', torch.softmax(s, -1), v).reshape(n, L, dm)
    o = o @ g('mha_fn.out_proj.weight').t() + g('mha_fn.out_proj.bias')
    h_left = torch.relu(o.mean(1)) @ g('out_fn.weight').t() + g('out_fn.bias')
    hid = torch.relu(h_left @ g('merger.fc1.weight')[:, :d].t() + g('merger.fc1.bias'))
    return h_left, hid @ g('merger.fc2.weight').t() + g('merger.fc2.bias')


def seq_weights(d, de, L, seed):
    return perturb_biases(random_weights(d, de, n_nodes=60, restarter='seq', hist_len=L, seed=seed))


@pytest.mark.parametrize('d,de,L,H,nf', [(12, 6, 9, 3, True), (8, 4, 33, 2, False), (10, 4, 64, 4, True)])
def test_restatement_matches_the_oracle(d, de, L, H, nf):
    """tokens64 + seq64 say what OracleTIGER.seq_restarter (the reference's SeqRestarter.forward) says."""
    W = seq_weights(d, de, L, seed=d)
    c = SeqCase(d, de, L, 40, seed=L, nfeats=nf, span=1e4).with_weights(W)
    model = O.OracleTIGER(W, None, 60, d, c.efeats.numpy(), c.nfeats.numpy() if nf else None, n_head=H,
                          restarter='seq', hist_len=L)
    want_l, want_r, want_pt = model.seq_restarter(c.nids.numpy(), c.hn.numpy(), c.he.numpy(), c.ht.numpy(),
                                                  c.hd.numpy(), c.an.numpy())
    got_l, got_r = seq64(*c.tokens64(), W, H, d)
    check('restatement', 'h_left vs oracle', got_l, want_l, 2e-6)
    check('restatement', 'h_right vs oracle', got_r, want_r, 2e-6)
    assert torch.equal(want_pt, c.ht[:, -1])


# ------------------------------------------------------------------------------------------
# 1. tiger_seq_tokens
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('nf,ef', [(True, True), (False, False), (True, False), (False, True)])
@pytest.mark.parametrize('d,de', [(1, 1), (10, 4), (43, 172), (172, 172)])
@pytest.mark.parametrize('L', [1, 2, 33, 64])
def test_seq_tokens_match_float64(L, d, de, nf, ef):
    """Feature columns bit for bit, the last position zero but for its time code, time codes at dt up to 1e6 s,
    mask[:, -1] = 0 (also in fully padded rows) and prev_ts = hist_ts[:, -1]."""
    cap = 37
    c = SeqCase(d, de, L, cap, seed=L * 7 + d, nfeats=nf, efeats=ef)
    x64, mask = c.tokens64()
    dm, F = 4 * d + de, 3 * d + de
    nids, hist = cu(c.nids), c.hist_dev()
    for form in COUNT_FORMS:
        cnt, m = count_of(form, cap)
        x, mk, pt = nan_dev(cap * L, dm), torch.full((cap, L), 7, dtype=torch.uint8, device=DEV), nan_dev(cap)
        call('tiger_seq_tokens', ptr(nids), ptr(cnt), cap, L, *(ptr(t) for t in hist), ptr(cu(c.nfeats)),
             ptr(cu(c.efeats)), d, de, ptr(cu(c.anony_emb)), ptr(cu(c.tw)), ptr(cu(c.tb)), ptr(x), ptr(mk), ptr(pt))
        x, mk, pt = x.view(cap, L, dm).cpu(), mk.cpu(), pt.cpu()
        what = f'L={L} d={d} de={de} {form}'
        assert torch.equal(x[:m, :, :F].double(), x64[:m, :, :F]), what + ': feature columns'
        check('seq_tokens time codes', what + ': time codes', x[:m, :, F:], x64[:m, :, F:], TC_TOL)
        assert torch.equal(mk[:m].bool(), mask[:m]), what + ': key-padding mask'
        assert not mk[:m, -1].any(), what + ': mask[:, -1] must be 0'
        assert torch.equal(pt[:m], c.ht[:m, -1]), what + ': prev_ts'
        untouched(what + ': x past count', x[m:])
        untouched(what + ': prev_ts past count', pt[m:])
        assert (mk[m:] == 7).all(), what + ': mask past count'


# ------------------------------------------------------------------------------------------
# 2. tiger_seq_tail, inference and training mode
# ------------------------------------------------------------------------------------------
def tail_weights(dm, d, gen):
    """The five layers' weights, scaled so that activations stay O(1).  fc1 is [d, d_model] as the merger stores it;
    only its first d columns take part, the others hold 1e3 (a kernel that read them would be far off)."""
    r = lambda *s: torch.randn(*s, generator=gen) / math.sqrt(s[-1])
    b = lambda k: torch.randn(k, generator=gen) * 0.5
    fc1 = torch.full((d, dm), 1e3)
    fc1[:, :d] = r(d, d)
    return dict(w_v=r(dm, dm), b_v=b(dm), w_out=r(dm, dm), b_out=b(dm), w_fn=r(d, dm), b_fn=b(d), w_fc1=fc1,
                b_fc1=b(d), w_fc2=r(d, d), b_fc2=b(d))


def tail64(xbar, w, H, d, psum=None, p=0.0, seed=0):
    """The five layers after the pooling in float64 on xbar [n, H, d_model]; psum [n, H] scales the value bias, p the
    merger's dropout (mask stream 4, element r * d + c)."""
    n, _, dm = xbar.shape
    hd = dm // H
    g = lambda k: w[k].double()
    scale = psum.double() if psum is not None else torch.ones(n, H, dtype=torch.float64)
    att = (torch.einsum('nhc,hjc->nhj', xbar.double(), g('w_v').view(H, hd, dm))
           + scale[:, :, None] * g('b_v').view(H, hd)).reshape(n, dm)
    o = torch.relu(att @ g('w_out').t() + g('b_out'))
    h_left = o @ g('w_fn').t() + g('b_fn')
    pre = torch.relu(h_left @ g('w_fc1')[:, :d].t() + g('b_fc1'))
    keep = keep_mask(seed, 4, np.arange(n * d), p).reshape(n, d)
    hid = torch.where(keep, pre * inv_keep(p), torch.zeros((), dtype=torch.float64))
    return dict(att=att, o=o, h_left=h_left, hid=hid, h_right=hid @ g('w_fc2').t() + g('b_fc2'), pre=pre, keep=keep)


TAIL_OUTS = ('att', 'o', 'h_left', 'hid', 'h_right')


def run_tail(xbar, w, n, dm, H, d, cnt, *, psum=None, p=0.0, seed=0, lead=0):
    """tiger_seq_tail on xbar [n, H d_model]; `lead` floats in front of xbar and every weight."""
    wd = {k: placed(v.to(DEV), lead) for k, v in w.items()}
    xb = placed(xbar.reshape(n, H * dm).to(DEV), lead)
    out = dict(att=nan_dev(n, dm), o=nan_dev(n, dm), h_left=nan_dev(n, d), hid=nan_dev(n, d), h_right=nan_dev(n, d))
    call('tiger_seq_tail', ptr(xb), ptr(cnt), n, dm, H, d, ptr(wd['w_v']), ptr(wd['b_v']), ptr(wd['w_out']),
         ptr(wd['b_out']), ptr(wd['w_fn']), ptr(wd['b_fn']), ptr(wd['w_fc1']), dm, ptr(wd['b_fc1']), ptr(wd['w_fc2']),
         ptr(wd['b_fc2']), ptr(psum), p, seed, ptr(out['att']), ptr(out['o']), ptr(out['hid']), ptr(out['h_left']),
         ptr(out['h_right']))
    return out


def check_tail(group, got, want, m, what):
    for k in TAIL_OUTS:
        check(group, f'{what}: {k}', got[k][:m], want[k][:m], TOL)
        untouched(f'{what}: {k} past count', got[k][m:])


# d_model = 4 d + d_e.  KREG 8: 106 (scalar), 256 (16-byte, edge); KREG 16: 257 (scalar), 404, 512 (edge); KREG 32: 513
# (scalar), 860, 1024 (edge).  d = 25, 63, 127 put the merger layers on the scalar path.
TAIL_SHAPES = [(106, 25), (256, 60), (257, 63), (404, 100), (512, 127), (513, 128), (860, 172), (1024, 250)]
TAIL_CASES = [(dm, d, H) for dm, d in TAIL_SHAPES for H in (1, 2, 3, 4, 8) if dm % H == 0]


@pytest.mark.parametrize('dm,d,H', TAIL_CASES)
def test_seq_tail_inference_matches_float64(dm, d, H):
    gen = torch.Generator().manual_seed(dm * 10 + H)
    w = tail_weights(dm, d, gen)
    for n in (1, 7, 8, 9, 64):
        xbar = torch.randn(n, H, dm, generator=gen)
        want = tail64(xbar, w, H, d)
        for form in COUNT_FORMS:
            cnt, m = count_of(form, n)
            check_tail('seq_tail', run_tail(xbar, w, n, dm, H, d, cnt), want, m, f'd_model={dm} H={H} n={n} {form}')


@pytest.mark.parametrize('dm,d,H', [(256, 60, 2), (404, 100, 4), (860, 172, 2)])
def test_seq_tail_scalar_path_on_misaligned_rows(dm, d, H):
    """xbar and every weight one float past a 16-byte boundary: the scalar path of each KREG at d_model % 4 == 0."""
    gen = torch.Generator().manual_seed(dm + 1)
    w = tail_weights(dm, d, gen)
    n = 9
    xbar = torch.randn(n, H, dm, generator=gen)
    for form in COUNT_FORMS:
        cnt, m = count_of(form, n)
        check_tail('seq_tail', run_tail(xbar, w, n, dm, H, d, cnt, lead=1), tail64(xbar, w, H, d), m,
                   f'misaligned d_model={dm} {form}')


def products_route(xbar, psum, w, n, dm, H, d, p, seed):
    """The training step's route for many rows (train_seq.py): tensor-core products, tiger_train_seq_vbias, the merger
    dropout as tiger_train_dropout(stream 4)."""
    hd = dm // H
    wd = {k: cu(v) for k, v in w.items()}
    out = dict(att=nan_dev(n, dm), o=nan_dev(n, dm), h_left=nan_dev(n, d), hid=nan_dev(n, d), h_right=nan_dev(n, d))
    for h in range(H):
        ops.sgemm_ex(xbar[:, h * dm:(h + 1) * dm], wd['w_v'][h * hd:(h + 1) * hd], out['att'][:, h * hd:(h + 1) * hd],
                     m=n, n=hd, k=dm)
    call('tiger_train_seq_vbias', ptr(out['att']), ptr(psum), ptr(wd['b_v']), None, n, dm, H)
    ops.sgemm_ex(out['att'], wd['w_out'], out['o'], m=n, n=dm, k=dm, bias=wd['b_out'], relu=True)
    ops.sgemm_ex(out['o'], wd['w_fn'], out['h_left'], m=n, n=d, k=dm, bias=wd['b_fn'])
    ops.sgemm_ex(out['h_left'], wd['w_fc1'][:, :d], out['hid'], m=n, n=d, k=d, bias=wd['b_fc1'], relu=True)
    call('tiger_train_dropout', ptr(out['hid']), None, d, n * d, p, seed, 4)
    ops.sgemm_ex(out['hid'], wd['w_fc2'], out['h_right'], m=n, n=d, k=d, bias=wd['b_fc2'])
    return out


@pytest.mark.parametrize('p', [0.1, 0.5])
@pytest.mark.parametrize('dm,d,H', [(106, 25, 2), (404, 100, 4), (860, 172, 2)])
def test_seq_tail_training_mode_matches_float64_and_the_product_route(dm, d, H, p):
    """psum from a tiger_train_seq_pool call with dropout scales the value bias; the merger's dropout mask must be the
    one tiger_train_dropout(stream 4) draws on the product route, element for element."""
    gen = torch.Generator().manual_seed(dm + int(p * 10))
    w = tail_weights(dm, d, gen)
    L, seed = 6, 4321
    for n in (9, 64):
        qk, x = cu(torch.randn(n * L, 2 * dm, generator=gen)), cu(torch.randn(n * L, dm, generator=gen))
        mask = (torch.rand(n, L, generator=gen) < 0.3).to(torch.uint8)
        mask[:, -1] = 0
        P, pb, psum, xbar = nan_dev(n * H * L * L), nan_dev(n * H * L), nan_dev(n, H), nan_dev(n, H * dm)
        call('tiger_train_seq_pool', ptr(qk), 2 * dm, ptr(x), ptr(cu(mask)), None, n, L, dm, H, p, seed, ptr(P),
             ptr(pb), ptr(psum), ptr(xbar))
        assert float((psum.cpu() - 1).abs().max()) > 0.01, 'attention dropout should move psum away from 1'
        want = tail64(xbar.cpu().view(n, H, dm), w, H, d, psum=psum.cpu(), p=p, seed=seed)
        for form in COUNT_FORMS:
            cnt, m = count_of(form, n)
            check_tail('seq_tail_train', run_tail(xbar.cpu().view(n, H, dm), w, n, dm, H, d, cnt, psum=psum, p=p,
                                                  seed=seed), want, m, f'train d_model={dm} p={p} n={n} {form}')
        tail = run_tail(xbar.cpu().view(n, H, dm), w, n, dm, H, d, None, psum=psum, p=p, seed=seed)
        prod = products_route(xbar, psum, w, n, dm, H, d, p, seed)
        check('seq_tail_train', 'product route h_right', prod['h_right'], want['h_right'], TOL)
        check('seq_tail_train', 'tail vs product route h_right', tail['h_right'], prod['h_right'], TOL)
        pre, keep = want['pre'], want['keep']
        live = pre > 1e-3 * float(pre.abs().max())
        for name, got in (('tail', tail['hid'].cpu()), ('products', prod['hid'].cpu())):
            assert not got[~keep].any(), f'{name}: dropped merger units must be exactly zero'
            assert got[keep & live].ne(0).all(), f'{name}: kept merger units must be live'


# ------------------------------------------------------------------------------------------
# 3. the route gate and ops.SeqRestarterOp.forward
# ------------------------------------------------------------------------------------------
def test_seq_gate_count_splits_at_max_rows():
    cnt, out = torch.zeros(1, dtype=torch.int32, device=DEV), torch.full((2,), -9, dtype=torch.int32, device=DEV)
    for max_rows in (0, 64):
        for c in (0, 1, 63, 64, 65, 1000):
            cnt.fill_(c)
            call('tiger_seq_gate_count', ptr(cnt), max_rows, ptr(out), ptr(out[1:]))
            small, big = out.tolist()
            assert (small, big) == ((c, 0) if c <= max_rows else (0, c)), f'count {c}, max_rows {max_rows}'


def run_op(op, c, nids, n, count):
    """forward on NaN-filled outputs; returns the whole [cap] buffers."""
    for t in (op.h_left, op.h_right, op.prev_ts):
        t.fill_(NAN)
    op.forward(nids, n, cu(c.nfeats), cu(c.efeats), count=count, hist=c.hist_dev())
    return op.h_left.clone(), op.h_right.clone(), op.prev_ts.clone()


def check_op(c, got, want, m, what):
    hl, hr, pt = (t.cpu() for t in got)
    check('seq_restarter_op', what + ': h_left', hl[:m], want[0][:m], TOL)
    check('seq_restarter_op', what + ': h_right', hr[:m], want[1][:m], TOL)
    assert torch.equal(pt[:m], c.ht[:m, -1]), what + ': prev_ts'
    for name, t in (('h_left', hl), ('h_right', hr), ('prev_ts', pt)):
        untouched(f'{what}: {name} past count', t[m:])


@pytest.mark.parametrize('d,de,H', [(24, 10, 2), (24, 8, 1), (24, 8, 4), (256, 100, 2)])
def test_seq_restarter_op_matches_float64_on_both_routes(d, de, H):
    """Device counts 0, 1, 64, 65 and cap, and count = None at n = 64 / 65: both sides of the gate.  d = 256, d_e =
    100 (d_model = 1124 > 1024) has no tail and runs the products alone."""
    cap, L = 130, 5
    W = seq_weights(d, de, L, seed=H)
    c = SeqCase(d, de, L, cap, seed=d + H, span=1e4).with_weights(W)
    want = seq64(*c.tokens64(), W, H, d)
    op = ops.SeqRestarterOp(d, de, L, H, cap, DEV)
    op.set_weights(W)
    assert op.tail_rows == (64 if 4 * d + de <= 1024 else 0)
    nids = cu(c.nids)
    for k in (0, 1, 64, 65, cap):
        cnt = torch.tensor([k], dtype=torch.int32, device=DEV)
        check_op(c, run_op(op, c, nids, cap, cnt), want, k, f'H={H} count {k}')
    for n in (64, 65):
        check_op(c, run_op(op, c, nids, n, None), want, n, f'H={H} n={n} without count')


def test_seq_restarter_op_graph_replay_equals_eager():
    """forward captured once with a device count, replayed with counts 3, 64, 65 and 120 set between replays: the two
    routes are parallel branches of the graph, the gate hands one of them zero rows.  Each replay must equal the eager
    result bit for bit."""
    d, de, H, L, cap = 24, 10, 2, 6, 128
    W = seq_weights(d, de, L, seed=5)
    c = SeqCase(d, de, L, cap, seed=9, span=1e4).with_weights(W)
    want = seq64(*c.tokens64(), W, H, d)
    op = ops.SeqRestarterOp(d, de, L, H, cap, DEV)
    op.set_weights(W)
    nids, nf, ef, hist = cu(c.nids), cu(c.nfeats), cu(c.efeats), c.hist_dev()
    cnt = torch.tensor([3], dtype=torch.int32, device=DEV)
    counts = (3, 64, 65, 120)
    eager = {}
    for k in counts:
        cnt.fill_(k)
        eager[k] = run_op(op, c, nids, cap, cnt)
        check_op(c, eager[k], want, k, f'eager count {k}')
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                        # warm-up off the capturing stream
        op.forward(nids, cap, nf, ef, count=cnt, hist=hist)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = op.forward(nids, cap, nf, ef, count=cnt, hist=hist)
    for k in counts:
        cnt.fill_(k)
        for t in (op.h_left, op.h_right, op.prev_ts):
            t.fill_(NAN)
        graph.replay()
        torch.cuda.synchronize()
        for name, got, ref in zip(('h_left', 'h_right', 'prev_ts'), out, eager[k]):
            assert torch.equal(got[:k], ref[:k]), f'replay with count {k}: {name} differs from the eager result'
            untouched(f'replay with count {k}: {name} past count', got[k:])


# ------------------------------------------------------------------------------------------
# 4. tiger_min_time
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n', [1, 255, 256, 257, 10000])
def test_min_time_is_the_float32_minimum(n):
    rng = np.random.RandomState(n)
    for where in ('first', 'last', 'negative'):
        ts = (rng.rand(n) * 1e6 + 10).astype(np.float32)
        if where == 'first':
            ts[0] = 3.25
        elif where == 'last':
            ts[-1] = 3.25
        else:
            ts[::3] *= -1
        out = torch.full((1,), NAN, dtype=torch.float64, device=DEV)
        ops.min_time(cu(torch.from_numpy(ts)), out)
        assert float(out) == float(np.float64(ts.min())), f'n={n} {where}: {float(out)} vs {ts.min()}'


# ------------------------------------------------------------------------------------------
# 5. tiger_static_restart, tiger_static_restart_rows
# ------------------------------------------------------------------------------------------
DEGREES = (0, 1, 31, 32, 33, 1000, 70000)      # nodes 1..7; fillers 100..199 are the other end of every event
N_RESTART = 200


class RestartGraph:
    """A time-ordered stream whose nodes 1..7 have the degrees above, with many events sharing a time (integer times,
    few distinct values for the small nodes), on the device and in OracleGraph."""

    def __init__(self):
        rng = np.random.RandomState(0)
        src, dst, ts = [], [], []
        self.times = {}
        for u, k in zip(range(1, 8), DEGREES):
            t = 100.0 + rng.randint(0, 10 if k < 100 else 1000, k).astype(np.float64)
            src.append(np.full(k, u)), dst.append(rng.randint(100, N_RESTART, k)), ts.append(t)
        src, dst, ts = np.concatenate(src), np.concatenate(dst), np.concatenate(ts)
        order = np.argsort(ts, kind='stable')
        self.src, self.dst, self.ts = src[order].astype(np.int64), dst[order].astype(np.int64), ts[order]
        self.eids = np.arange(1, len(ts) + 1, dtype=np.int64)
        self.oracle = O.OracleGraph(self.src, self.dst, self.ts, self.eids, n_nodes=N_RESTART)
        dv = lambda a: torch.from_numpy(a).to(DEV)
        self.csr = ops.csr_build(dv(self.src), dv(self.dst), dv(self.ts), dv(self.eids), N_RESTART)
        for u in range(N_RESTART):
            self.times[u] = np.sort(np.concatenate([self.ts[self.src == u], self.ts[self.dst == u]]))

    def prev_ts(self, u, t):
        """float32 time of u's last event strictly before t, 0 without one."""
        ts = self.times[u]
        j = np.searchsorted(ts, t, side='left')
        return np.float32(ts[j - 1]) if j > 0 else np.float32(0.0)


_GRAPH = []


def restart_graph():
    if not _GRAPH:
        _GRAPH.append(RestartGraph())
    return _GRAPH[0]


def restart_list(seed):
    """Nodes 1..7 and twenty fillers, shuffled, without repeats."""
    rng = np.random.RandomState(seed)
    nids = np.concatenate([np.arange(1, 8), rng.choice(np.arange(100, N_RESTART), 20, replace=False)])
    return nids[rng.permutation(len(nids))].astype(np.int64)


class Tables:
    """Node-indexed state before a restart (CPU copies kept for the expected state)."""

    def __init__(self, d, seed, null=()):
        g = torch.Generator().manual_seed(seed)
        N = N_RESTART
        self.emb = dict(left=torch.randn(N, d, generator=g), right=torch.randn(N, d, generator=g))
        self.host = dict(left_vals=torch.randn(N, d, generator=g), right_vals=torch.randn(N, d, generator=g),
                         left_ts=torch.rand(N, generator=g) * 50, right_ts=torch.rand(N, generator=g) * 50,
                         left_active=torch.zeros(N, dtype=torch.uint8), right_active=torch.zeros(N, dtype=torch.uint8),
                         has_msg=torch.ones(N, dtype=torch.uint8))
        self.dev = {k: (None if k in null else v.to(DEV).contiguous()) for k, v in self.host.items()}

    def expected(self, nids, prev):
        want = {k: v.clone() for k, v in self.host.items()}
        for u, p in zip(nids, prev):
            want['left_vals'][u], want['right_vals'][u] = self.emb['left'][u], self.emb['right'][u]
            want['left_ts'][u] = want['right_ts'][u] = float(p)
            want['left_active'][u] = want['right_active'][u] = 1
            want['has_msg'][u] = 0
        return want

    def check(self, nids, prev, what):
        want = self.expected(nids, prev)
        for k, t in self.dev.items():
            if t is not None:
                assert torch.equal(t.cpu(), want[k]), f'{what}: {k}'


def run_static_restart(G, tab, nids, d, cnt, *, batch_ts=None, q_ts=None, with_prev=True):
    out_prev = nan_dev(len(nids)) if with_prev else None
    ops.static_restart(cu(torch.from_numpy(nids)), len(nids), G.csr, cu(tab.emb['left']), cu(tab.emb['right']), d,
                       count=cnt, batch_ts=batch_ts, q_ts=q_ts, out_prev_ts=out_prev, **tab.dev)
    torch.cuda.synchronize()
    return out_prev


def check_prev(G, nids, t, out_prev, m, what):
    want = np.array([G.prev_ts(u, tt) for u, tt in zip(nids, t)], dtype=np.float32)
    ref = G.oracle.get_history(nids, np.asarray(t, dtype=np.float64), 1)[2][:, 0]
    assert np.array_equal(want, ref), 'restatement vs OracleGraph.get_history'
    if out_prev is not None:
        got = out_prev.cpu().numpy()
        assert np.array_equal(got[:m], want[:m]), f'{what}: prev_ts'
        untouched(what + ': prev_ts past count', out_prev[m:])
    return want


# batch query times: before every event, a time many events share, between two event times, after every event
BATCH_TIMES = (50.0, 104.0, 104.5, 5000.0)


@pytest.mark.parametrize('B', [1, 31, 200, 2000])
@pytest.mark.parametrize('d', [1, 10, 100, 172])
def test_static_restart_batch_time_matches_float64(d, B):
    """t = the float32 minimum of batch_ts (found by the warp itself), at the end of the batch for B = 2,000."""
    G = restart_graph()
    nids = restart_list(d + B)
    rng = np.random.RandomState(B)
    for t in BATCH_TIMES:
        bts = (t + rng.rand(B) * 100).astype(np.float32)
        bts[-1 if B == 2000 else rng.randint(B)] = t
        for form in COUNT_FORMS:
            cnt, m = count_of(form, len(nids))
            tab = Tables(d, seed=d)
            what = f'd={d} B={B} t={t} {form}'
            out_prev = run_static_restart(G, tab, nids, d, cnt, batch_ts=cu(torch.from_numpy(bts)))
            prev = check_prev(G, nids, np.full(len(nids), t), out_prev, m, what)
            tab.check(nids[:m], prev[:m], what)


def per_row_times(G, nids, kind):
    """A query time per node: before its first event, at a time several of its events share (its first time when none
    does), between two of its event times, after its last event."""
    out = []
    for u in nids:
        ts = G.times[int(u)]
        if len(ts) == 0:
            out.append(77.0)
            continue
        vals, mult = np.unique(ts, return_counts=True)
        if kind == 'before':
            out.append(ts[0] - 50.0)
        elif kind == 'tie':
            out.append(vals[np.argmax(mult)])
        elif kind == 'between':
            out.append((vals[len(vals) // 2 - 1] + vals[len(vals) // 2]) / 2 if len(vals) > 1 else ts[0] + 0.5)
        else:
            out.append(ts[-1] + 10.0)
    return np.array(out, dtype=np.float64)


@pytest.mark.parametrize('d', [1, 10, 100, 172])
def test_static_restart_per_row_time_matches_float64(d):
    G = restart_graph()
    nids = restart_list(d)
    for kind in ('before', 'tie', 'between', 'after'):
        q = per_row_times(G, nids, kind)
        for form in COUNT_FORMS:
            cnt, m = count_of(form, len(nids))
            tab = Tables(d, seed=d + 1)
            what = f'd={d} {kind} {form}'
            out_prev = run_static_restart(G, tab, nids, d, cnt, q_ts=cu(torch.from_numpy(q)))
            prev = check_prev(G, nids, q, out_prev, m, what)
            tab.check(nids[:m], prev[:m], what)


@pytest.mark.parametrize('null', [('left_vals', 'right_vals', 'left_ts', 'right_ts', 'left_active', 'right_active',
                                   'has_msg'), ('left_vals', 'right_ts', 'has_msg'), ()])
def test_static_restart_optional_outputs(null):
    """Every table may be NULL, and so may out_prev_ts: the given ones are written all the same."""
    G = restart_graph()
    nids, d = restart_list(3), 10
    q = per_row_times(G, nids, 'tie')
    tab = Tables(d, seed=4, null=null)
    out_prev = run_static_restart(G, tab, nids, d, None, q_ts=cu(torch.from_numpy(q)), with_prev=bool(null))
    prev = check_prev(G, nids, q, out_prev, len(nids), 'optional outputs')
    tab.check(nids, prev, f'NULL {null}')


@pytest.mark.parametrize('form', COUNT_FORMS)
@pytest.mark.parametrize('d', [1, 10, 100, 172])
def test_static_restart_rows_match(d, form):
    nids = restart_list(d + 7)
    right = torch.randn(N_RESTART, d, generator=torch.Generator().manual_seed(d))
    cnt, m = count_of(form, len(nids))
    out = nan_dev(len(nids), d)
    ops.static_restart_rows(cu(torch.from_numpy(nids)), len(nids), cu(right), d, out, count=cnt)
    assert torch.equal(out[:m].cpu(), right[torch.from_numpy(nids[:m])]), f'd={d} {form}'
    untouched('rows past count', out[m:])


# ------------------------------------------------------------------------------------------
# 6. refusals: -1 and nothing written
# ------------------------------------------------------------------------------------------
def test_refusals_return_minus_one_and_write_nothing():
    lib, st = load(), stream_ptr()
    z = torch.zeros(1 << 21, device=DEV)          # inputs: never read by a refused call
    outs = [nan_dev(8, 1100) for _ in range(5)]

    def tail(dm, H, d, ld_fc1, p):
        return lib.tiger_seq_tail(ptr(z), None, 4, dm, H, d, *(ptr(z),) * 6, ptr(z), ld_fc1, ptr(z), ptr(z), ptr(z),
                                  ptr(z), p, 1, *(ptr(t) for t in outs), st)
    assert tail(64, 2, 8, 64, 0.0) == 0                            # the same call within the limits runs
    torch.cuda.synchronize()
    for t in outs:
        t.fill_(NAN)
    for what, args in (('d_model > 1024', (1025, 1, 8, 1025, 0.0)), ('d > 1024', (1024, 2, 1025, 1025, 0.0)),
                       ('ld_fc1 < d', (64, 2, 8, 7, 0.0)), ('d_model % n_head', (64, 3, 8, 64, 0.0)),
                       ('p_drop = 1', (64, 2, 8, 64, 1.0)), ('p_drop > 1', (64, 2, 8, 64, 1.5))):
        assert tail(*args) == -1, 'tiger_seq_tail: ' + what
    ids = torch.zeros(64, dtype=torch.int64, device=DEV)
    mask = torch.full((64,), 7, dtype=torch.uint8, device=DEV)
    prev, tmin = nan_dev(8), torch.full((1,), NAN, dtype=torch.float64, device=DEV)
    for L in (0, -1):
        assert lib.tiger_seq_tokens(ptr(ids), None, 4, L, *(ptr(ids),) * 5, ptr(z), ptr(z), 8, 8, ptr(z), ptr(z),
                                    ptr(z), ptr(outs[0]), ptr(mask), ptr(prev), st) == -1, f'tiger_seq_tokens len={L}'
    for n in (0, -1):
        assert lib.tiger_min_time(ptr(z), n, ptr(tmin), st) == -1, f'tiger_min_time n={n}'
    G = restart_graph()
    tab = Tables(4, seed=1)
    args = [ptr(ids), None, 4, None, 0, None, ptr(G.csr.indptr), ptr(G.csr.ts), ptr(z), ptr(z), 4] + \
        [ptr(tab.dev[k]) for k in ('left_vals', 'left_ts', 'left_active', 'right_vals', 'right_ts', 'right_active',
                                   'has_msg')] + [ptr(prev), st]
    assert lib.tiger_static_restart(*args) == -1, 'tiger_static_restart without a time source'
    torch.cuda.synchronize()
    for t in outs + [prev, tmin]:
        untouched('output of a refused call', t)
    assert (mask == 7).all()
    tab.check([], [], 'tables after a refused restart')


# ------------------------------------------------------------------------------------------
# 7. histories past the pooling kernel's limit
# ------------------------------------------------------------------------------------------
def test_pool_limit_is_the_python_limit():
    """tiger_train_seq_pool takes ops.SEQ_MAX_HIST_LEN positions and refuses one more."""
    lib, st = load(), stream_ptr()
    n, dm, H = 2, 8, 1
    L = ops.SEQ_MAX_HIST_LEN
    assert ops.seq_restarter_limit_error(8, 8, L, 2) is None and ops.seq_restarter_limit_error(8, 8, L + 1, 2)
    for length, rc in ((L, 0), (L + 1, -1)):
        qk, x = torch.zeros(n * length, 2 * dm, device=DEV), torch.zeros(n * length, dm, device=DEV)
        mask = torch.zeros(n, length, dtype=torch.uint8, device=DEV)
        P, pb, ps, xb = nan_dev(n * H * length * length), nan_dev(n * H * length), nan_dev(n * H), nan_dev(n * H * dm)
        assert lib.tiger_train_seq_pool(ptr(qk), 2 * dm, ptr(x), ptr(mask), None, n, length, dm, H, 0.0, 0, ptr(P),
                                        ptr(pb), ptr(ps), ptr(xb), st) == rc, f'len={length}'
        torch.cuda.synchronize()
    with pytest.raises(NotImplementedError, match='at most 64 events'):
        ops.SeqRestarterOp(8, 8, L + 1, 2, 4, DEV)


@pytest.mark.parametrize('hist_len', [64, 65, 100])
def test_dropin_restart_with_long_histories_matches_oracle(hist_len):
    """An eval-mode drop-in model restarts nodes under no_grad after a batch left messages pending: memories, clocks
    and the message store equal OracleTIGER.restart.  Past 64 events the restarter runs its torch code (before, the
    pooling kernel refused it after the message store had been cleared); at 64 it stays on the kernels."""
    from torch.utils.data import DataLoader

    import dropin_utils  # noqa: F401  (puts the drop-in package on the path)
    from tiger.data.data_loader import GraphCollator, InteractionData
    from tiger.data.graph import Graph
    from www2023tiger_b200.init import build_model
    from www2023tiger_b200.synthetic import NegativeSampler, StreamShape, make_stream

    st = make_stream(StreamShape('long', 12, 8, 3000, 6, None, horizon=3000.), seed=4)
    N, d, de, K, B, s0 = st.n_nodes, 8, 6, 10, 50, 2000
    neg = NegativeSampler(st.src, st.dst, seed=0).pre_sample_neg_dsts(st.n_events)
    W = perturb_biases(random_weights(d, de, n_nodes=N, restarter='seq', hist_len=hist_len, seed=2))
    full = InteractionData(st.src, st.dst, st.ts, st.eids, np.zeros_like(st.src), seed=0, eval=True, neg_dst=neg)
    graph = Graph.from_data(full, strategy='recent_edges', seed=0, max_node_id=N - 1)
    part = slice(s0, s0 + 2 * B)
    data = InteractionData(st.src[part], st.dst[part], st.ts[part], st.eids[part], np.zeros(2 * B, dtype=np.int64),
                           seed=0, eval=True, neg_dst=neg[part])
    dl = DataLoader(data, batch_size=B, collate_fn=GraphCollator(graph, K, 1, restarter='seq', hist_len=hist_len))
    model = build_model(None, st.efeats, graph, N, len(st.src), DEV, dim=d, n_neighbors=K, restarter_type='seq',
                        hist_len=hist_len)
    res = model.load_state_dict(W, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    model.eval()
    model.reset()
    og = O.OracleGraph(st.src, st.dst, st.ts, st.eids, n_nodes=N)
    om = O.OracleTIGER(W, og, N, d, st.efeats, None, n_neighbors=K, restarter='seq', hist_len=hist_len)
    cpu = lambda t: t.detach().cpu()
    with torch.no_grad():
        for ib, batch in enumerate(dl):
            src, dst, negs, ts, eids, _, cg = batch
            s = slice(s0 + ib * B, s0 + (ib + 1) * B)
            b = O.collate(og, st.src[s], st.dst[s], neg[s], st.ts[s], st.eids[s], K)
            t0 = np.float32(b.ts.min())
            r = b.involved.astype(np.int64)
            assert (og.get_history(r, np.full(len(r), t0), hist_len)[0] != 0).all(1).any(), 'no full history'
            if ib > 0:
                assert om.has_msg[r].any(), 'the restart should clear pending messages'
            om.restart(r, np.full(len(r), t0, dtype=np.float32))
            model.restart(torch.from_numpy(r).to(DEV), torch.full((len(r),), float(t0), device=DEV))
            what = f'hist_len={hist_len} batch {ib}'
            check('dropin_restart', what + ': left memory', cpu(model.left_memory.vals), om.left_vals, TOL)
            check('dropin_restart', what + ': right memory', cpu(model.right_memory.vals), om.right_vals, TOL)
            assert torch.equal(cpu(model.left_memory.update_ts), om.left_ts), what + ': left clocks'
            assert torch.equal(cpu(model.right_memory.update_ts), om.right_ts), what + ': right clocks'
            assert sorted(model.msg_store.nodes_with_messages) == np.flatnonzero(om.has_msg).tolist(), what
            if ib == 0:
                om.contrast_step(b)
                model.contrast_learning(src.long().to(DEV), dst.long().to(DEV), negs.long().to(DEV),
                                        ts.float().to(DEV), eids.long().to(DEV), cg.to(DEV))
    assert (model.restarter_fn._op is not None) == (hist_len <= ops.SEQ_MAX_HIST_LEN), 'route of the restarter'
