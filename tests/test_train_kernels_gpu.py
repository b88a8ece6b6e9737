"""Every kernel of the native training step (csrc/train.cu, csrc/train_seq.cu), called one by one through the C ABI and
compared with a float64 restatement of the same operation on the CPU.  Backward kernels are compared with autograd on
that restatement, not with a re-derivation of their formulas.  The cases sit where kernels go wrong: every
instantiation of the attention core (K = 1..32), rows without any live slot, count-bounded tails (rows past *count must
stay untouched), padded leading dimensions, misaligned views, several column blocks or row slabs of the reductions,
and time codes at arguments up to 1e6 rad.

Tolerances are max-norm errors relative to the largest entry of the reference tensor: EW_TOL for element-wise kernels,
RED_TOL for reductions and atomics.  The largest error each group reaches is printed at the end of the module."""
import re

import numpy as np
import pytest
import torch

from www2023tiger_b200 import train as T
from www2023tiger_b200._lib import TigerLibraryError, call, ptr
from www2023tiger_b200.build import CSRC

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda')
EW_TOL = 1e-6        # element-wise kernels
RED_TOL = 2e-5       # reductions, atomics, dot products
NAN = float('nan')
WORST = {}


@pytest.fixture(scope='module', autouse=True)
def seed_word_is_zero():
    """The dropout kernels add 101 x the registered seed-step word to their seeds; the masks restated below assume
    tiger_step_seed(seed) == seed, i.e. no word registered, or one that is zero (no captured step is replaying)."""
    for idx, word in T._SEED_WORDS.items():
        assert int(word.item()) == 0, f'seed-step word of cuda:{idx} is {int(word.item())}'
    yield
    print('\nlargest relative error per kernel group:')
    for k in sorted(WORST):
        print(f'  {k:28s} {WORST[k]:.2e}')


_ALIVE = []      # device copies made by cu(): a raw pointer does not keep its tensor alive


@pytest.fixture(autouse=True)
def release_device_copies():
    yield
    torch.cuda.synchronize()
    _ALIVE.clear()


def cu(t):
    """Device copy of t, kept alive until the end of the test (the kernels only ever see its pointer)."""
    if t is None:
        return None
    d = t.to(DEV).contiguous()
    _ALIVE.append(d)
    return d


def nan_dev(*shape, dtype=torch.float32):
    return torch.full(shape, NAN, dtype=dtype, device=DEV)


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
# dropout masks, restated with numpy
# ------------------------------------------------------------------------------------------
def test_dropout_mix_functions_are_identical():
    """dropout_keep (train.cu) and seq_keep (common.cuh) must be one function for keep_mask to restate both."""
    def body(path, fn):
        src = open(f'{CSRC}/{path}').read()
        m = re.search(r'uint32_t\s+' + fn + r'\(uint32_t x\)\s*\{(.*?)\}', src, re.S)
        return re.sub(r'\s+', '', m.group(1))

    def keep_body(path, fn, mix):
        src = open(f'{CSRC}/{path}').read()
        m = re.search(r'bool\s+' + fn + r'\((.*?)\)\s*\{(.*?)\n\}', src, re.S)
        return re.sub(r'\s+', '', m.group(1) + m.group(2)).replace(mix, 'MIX')

    assert body('train.cu', 'mix32') == body('common.cuh', 'seq_mix32')
    assert keep_body('train.cu', 'dropout_keep', 'mix32') == keep_body('common.cuh', 'seq_keep', 'seq_mix32')


def _mix32(x):
    x = x & np.uint64(0xffffffff)
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x7feb352d)) & np.uint64(0xffffffff)
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x846ca68b)) & np.uint64(0xffffffff)
    x ^= x >> np.uint64(16)
    return x


def keep_mask(seed: int, stream: int, idx, p: float) -> torch.Tensor:
    """Decision of dropout_keep / seq_keep for element idx of mask stream `stream` under `seed` (True = kept)."""
    idx = np.asarray(idx, dtype=np.uint64)
    if p <= 0:
        return torch.ones(idx.shape, dtype=torch.bool)
    h = _mix32(idx ^ _mix32(np.uint64((seed + 0x9E3779B9 * (stream + 1)) & 0xffffffff)))
    return torch.from_numpy(((h >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)) >= np.float32(p))


def inv_keep(p: float) -> float:
    return float(np.float32(1.0) / (np.float32(1.0) - np.float32(p))) if p > 0 else 1.0


# count forms of the count-bounded kernels: NULL, a device count of 0, one below the capacity, one above it
COUNT_FORMS = ['null', 'zero', 'below', 'above']


def count_of(form: str, cap: int, per: int = 1):
    """(device count or None, rows the kernel must process) for a capacity of `cap` rows, `per` rows per count."""
    if form == 'null':
        return None, cap
    c = {'zero': 0, 'below': max(cap // per - 2, 1), 'above': cap // per + 5}[form]
    return torch.tensor([c], dtype=torch.int32, device=DEV), min(c * per, cap)


def time_arg32(dt, w, b):
    """fp32 argument of the time codes exactly as the kernels form it: __fadd_rn(__fmul_rn(dt, w), b), no FMA."""
    dt, w, b = (np.asarray(x, dtype=np.float32) for x in (dt, w, b))
    return torch.from_numpy(np.add(np.multiply(dt, w, dtype=np.float32), b, dtype=np.float32).astype(np.float64))


def straight_through(arg64, arg32):
    """arg64's gradient with arg32's value: the float64 restatement sees the kernel's float32 argument."""
    return arg64 + (arg32 - arg64).detach()


# ------------------------------------------------------------------------------------------
# 1. attention core (tiger_train_attn_core, _bwd)
# ------------------------------------------------------------------------------------------
def slot_ids(gen, n_q, K):
    """Neighbor ids with ~30 % padding (id 0), rows with exactly one live slot (first / last) and rows with none."""
    nn_ = torch.randint(1, 50, (n_q, K), generator=gen)
    nn_[torch.rand(n_q, K, generator=gen) < 0.3] = 0
    nn_[0::6] = 0                        # no live slot
    nn_[1::6, 1:] = 0                    # only slot 0
    if K > 1:
        nn_[2::6, :-1] = 0               # only slot K - 1
        nn_[2::6, -1] = 7
    return nn_


def attn_core_case(K, H, hd, p, n_q=75, pad=0, seed=11):
    gen = torch.Generator().manual_seed(K * 1000 + H * 100 + hd + int(p * 10))
    E = H * hd
    ldq, ldkv, ld_attn = E + pad, 2 * E + 3 * pad, E + 2 * pad
    Q = torch.randn(n_q, ldq, generator=gen)
    KV = torch.randn(n_q * K, ldkv, generator=gen)
    nn_ = slot_ids(gen, n_q, K)
    dattn = torch.randn(n_q, ld_attn, generator=gen)

    # ---- float64 restatement (temporal_agg_modules.py + torch MHA with need_weights) under autograd
    q = Q[:, :E].double().reshape(n_q, H, hd).requires_grad_()
    k = KV[:, :E].double().reshape(n_q, K, H, hd).requires_grad_()
    v = KV[:, E:2 * E].double().reshape(n_q, K, H, hd).requires_grad_()
    pad_ = nn_ == 0
    empty = pad_.all(1)
    mask = pad_.clone()
    mask[empty, K - 1] = False           # rows without a neighbor keep their last slot
    s = torch.einsum('nhc,nkhc->nhk', q / np.sqrt(hd), k).masked_fill(mask[:, None, :], float('-inf'))
    P = torch.softmax(s, -1)
    keep = keep_mask(seed, 1, np.arange(n_q * H * K), p).reshape(n_q, H, K)
    o = torch.einsum('nhk,nkhc->nhc', P * keep.double() * inv_keep(p), v).reshape(n_q, E)
    (o * dattn[:, :E].double()).sum().backward()

    # ---- the kernels
    Qd, KVd, nnd = cu(Q), cu(KV), cu(nn_)
    attn, Pk = nan_dev(n_q, ld_attn), nan_dev(n_q * H * K)
    bits, emp = torch.full((n_q * H,), -1, dtype=torch.int32, device=DEV), torch.full((n_q,), 9, dtype=torch.uint8,
                                                                                     device=DEV)
    call('tiger_train_attn_core', ptr(Qd), ldq, ptr(KVd), ptr(KVd[:, E:]), ldkv, ptr(nnd), n_q, K, H, hd, p, seed,
         ptr(attn), ld_attn, ptr(Pk), ptr(bits), ptr(emp))
    dQ, dKV = nan_dev(n_q, ldq), nan_dev(n_q * K, ldkv)
    call('tiger_train_attn_core_bwd', ptr(cu(dattn)), ld_attn, ptr(Qd), ldq, ptr(KVd), ptr(KVd[:, E:]), ldkv, ptr(Pk),
         ptr(bits), n_q, K, H, hd, p, ptr(dQ), ptr(dKV), ptr(dKV[:, E:]))
    torch.cuda.synchronize()
    return dict(P=P, o=o, keep=keep, empty=empty, pad=pad_, q=q, k=k, v=v, attn=attn, Pk=Pk, bits=bits, emp=emp,
                dQ=dQ, dKV=dKV, E=E)


@pytest.mark.parametrize('p', [0.0, 0.1, 0.5])
@pytest.mark.parametrize('H,hd', [(1, 8), (2, 100), (2, 172), (3, 33), (4, 25)])
@pytest.mark.parametrize('K', [1, 3, 5, 10, 20, 32])
def test_attn_core_and_bwd_match_float64(K, H, hd, p):
    """K = 5, 10, 20 run their instantiations, 1, 3 and 32 the generic one (K = 32 sets bit 31 of keep_bits)."""
    r = attn_core_case(K, H, hd, p)
    n_q, E = r['empty'].shape[0], r['E']
    bits = r['bits'].cpu().numpy().view(np.uint32).astype(np.uint64).reshape(n_q, H, 1)
    got_keep = torch.from_numpy(((bits >> np.arange(K, dtype=np.uint64)) & np.uint64(1)) == 1)
    assert torch.equal(got_keep, r['keep']), 'keep_bits differ from the stream-1 mask'
    if K < 32:
        assert not (bits >> np.uint64(K)).any(), 'keep_bits set past slot K - 1'
    assert torch.equal(r['emp'].cpu().bool(), r['empty'])
    check('attn_core', 'P', r['Pk'].reshape(n_q, H, K), r['P'], RED_TOL)
    P_empty = r['Pk'].reshape(n_q, H, K)[r['empty'].to(DEV)].cpu()
    assert torch.equal(P_empty, torch.eye(K)[K - 1].expand_as(P_empty)), 'empty rows: P one-hot on slot K - 1'
    check('attn_core', 'attn', r['attn'], r['o'], RED_TOL)
    check('attn_core_bwd', 'dQ', r['dQ'].reshape(n_q, H, -1), r['q'].grad, RED_TOL)
    dKV = r['dKV'].reshape(n_q, K, 2 * E).cpu()
    check('attn_core_bwd', 'dK', dKV[..., :E].reshape(n_q, K, H, -1), r['k'].grad, RED_TOL)
    check('attn_core_bwd', 'dV', dKV[..., E:].reshape(n_q, K, H, -1), r['v'].grad, RED_TOL)
    dead = r['pad'] & ~r['empty'][:, None]             # padding slots of rows with a live slot
    assert not dKV[dead].any(), 'padding slots must get exactly zero dK / dV'


def test_attn_core_padded_leading_dimensions_and_grid_stride():
    """ldq > E, ldkv > 2E, ld_attn > E, with more items than the 148 x 8 CTAs cover at once: the padding columns must
    stay untouched."""
    H, hd, K = 2, 20, 5
    r = attn_core_case(K, H, hd, 0.1, n_q=5003, pad=4)
    E, n_q = r['E'], 5003
    check('attn_core', 'attn', r['attn'][:, :E], r['o'], RED_TOL)
    check('attn_core', 'P', r['Pk'].reshape(n_q, H, K), r['P'], RED_TOL)
    check('attn_core_bwd', 'dQ', r['dQ'][:, :E].reshape(n_q, H, -1), r['q'].grad, RED_TOL)
    check('attn_core_bwd', 'dK', r['dKV'][:, :E].reshape(n_q, K, H, -1), r['k'].grad, RED_TOL)
    check('attn_core_bwd', 'dV', r['dKV'][:, E:2 * E].reshape(n_q, K, H, -1), r['v'].grad, RED_TOL)
    untouched('attn padding columns', r['attn'][:, E:])
    untouched('dQ padding columns', r['dQ'][:, E:])
    untouched('dKV padding columns', r['dKV'][:, 2 * E:])


def test_attn_core_edges():
    Q, KV, nn_ = torch.zeros(4, 8, device=DEV), torch.zeros(4 * 33, 16, device=DEV), torch.ones(4, 33, dtype=torch.int64,
                                                                                                   device=DEV)
    attn, P = nan_dev(4, 8), nan_dev(4 * 33)
    bits, emp = torch.zeros(4, dtype=torch.int32, device=DEV), torch.zeros(4, dtype=torch.uint8, device=DEV)
    # n_q = 0 is a no-op
    call('tiger_train_attn_core', ptr(Q), 8, ptr(KV), ptr(KV[:, 8:]), 16, ptr(nn_), 0, 5, 1, 8, 0.1, 3, ptr(attn), 8,
         ptr(P), ptr(bits), ptr(emp))
    call('tiger_train_attn_core_bwd', ptr(attn), 8, ptr(Q), 8, ptr(KV), ptr(KV[:, 8:]), 16, ptr(P), ptr(bits), 0, 5, 1,
         8, 0.1, ptr(attn), ptr(KV), ptr(KV[:, 8:]))
    torch.cuda.synchronize()
    untouched('attn after n_q = 0', attn)
    untouched('P after n_q = 0', P)
    for k in (0, 33):
        with pytest.raises(TigerLibraryError, match='invalid argument'):
            call('tiger_train_attn_core', ptr(Q), 8, ptr(KV), ptr(KV[:, 8:]), 16, ptr(nn_), 4, k, 1, 8, 0.0, 3,
                 ptr(attn), 8, ptr(P), ptr(bits), ptr(emp))
        with pytest.raises(TigerLibraryError, match='invalid argument'):
            call('tiger_train_attn_core_bwd', ptr(attn), 8, ptr(Q), 8, ptr(KV), ptr(KV[:, 8:]), 16, ptr(P), ptr(bits),
                 4, k, 1, 8, 0.0, ptr(Q), ptr(KV), ptr(KV[:, 8:]))


# ------------------------------------------------------------------------------------------
# 2. GRU (tiger_train_gather_pending, tiger_train_gru_gates, _bwd)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('form', COUNT_FORMS)
@pytest.mark.parametrize('d', [1, 10, 100, 172])
def test_gru_gates_and_bwd_match_float64(d, form):
    cap = 300
    gen = torch.Generator().manual_seed(d)
    Gi, Gh, Hs = torch.randn(cap, 3 * d, generator=gen) * 2, torch.randn(cap, 3 * d, generator=gen) * 2, \
        torch.randn(cap, d, generator=gen)
    dh = torch.randn(cap, d, generator=gen)
    cnt, n = count_of(form, cap)
    # float64 GRUCell gates (torch.nn.GRUCell: r, z, n order), autograd on Gi and Gh
    gi, gh = Gi.double().requires_grad_(), Gh.double().requires_grad_()
    r = torch.sigmoid(gi[:, :d] + gh[:, :d])
    z = torch.sigmoid(gi[:, d:2 * d] + gh[:, d:2 * d])
    nn_ = torch.tanh(gi[:, 2 * d:] + r * gh[:, 2 * d:])
    h_new = (1 - z) * nn_ + z * Hs.double()
    (h_new[:n] * dh[:n].double()).sum().backward()
    Gid, Ghd, Hd = cu(Gi), cu(Gh), cu(Hs)
    out = [nan_dev(cap, d) for _ in range(4)]
    call('tiger_train_gru_gates', ptr(Gid), ptr(Ghd), ptr(Hd), ptr(cnt), cap, d, *(ptr(t) for t in out))
    dGi, dGh = nan_dev(cap, 3 * d), nan_dev(cap, 3 * d)
    call('tiger_train_gru_gates_bwd', ptr(cu(dh)), ptr(out[1]), ptr(out[2]), ptr(out[3]), ptr(Ghd), ptr(Hd), ptr(cnt),
         cap, d, ptr(dGi), ptr(dGh))
    torch.cuda.synchronize()
    for name, got, want in zip(('h_new', 'r', 'z', 'n'), out, (h_new, r, z, nn_)):
        check('gru_gates', name, got[:n], want[:n], EW_TOL)
        untouched(name + ' past count', got[n:])
    check('gru_gates_bwd', 'dGi', dGi[:n], gi.grad[:n], EW_TOL)
    check('gru_gates_bwd', 'dGh', dGh[:n], gh.grad[:n], EW_TOL)
    untouched('dGi past count', dGi[n:])
    untouched('dGh past count', dGh[n:])


def misaligned(rows, cols):
    """A NaN-filled [rows, cols] view 4 bytes past a 16-byte boundary (warp_copy_row's scalar path)."""
    return torch.full((rows * cols + 1,), NAN, device=DEV)[1:].view(rows, cols)


@pytest.mark.parametrize('form', COUNT_FORMS)
@pytest.mark.parametrize('m_dim,d,aligned', [(43, 10, True), (44, 172, False), (400, 100, True), (3, 1, True)])
def test_gather_pending_matches_float64(m_dim, d, aligned, form):
    """Repeated ids, m_dim not a multiple of 4 or misaligned outputs (scalar copies), dh_zero, n_rows_out."""
    N, cap = 90, 700
    gen = torch.Generator().manual_seed(m_dim + d)
    msg_vals, upd_vals = torch.randn(N, m_dim, generator=gen), torch.randn(N, d, generator=gen)
    ids = torch.randint(0, N, (cap,), generator=gen)
    ids[1::3] = ids[0::3][:len(ids[1::3])]          # repeated ids
    msg_ts = torch.rand(N, generator=gen) * 100
    cnt, n = count_of(form, cap)
    X, Hs = (misaligned(cap, m_dim), misaligned(cap, d)) if not aligned else (nan_dev(cap, m_dim), nan_dev(cap, d))
    dh0, err, nrows = nan_dev(cap, d), torch.zeros(1, dtype=torch.int32, device=DEV), nan_dev(1)
    call('tiger_train_gather_pending', ptr(cu(ids)), ptr(cnt), cap, ptr(cu(msg_vals)), m_dim, ptr(cu(msg_ts)),
         ptr(cu(upd_vals)), d, ptr(cu(msg_ts)), 1, ptr(X), ptr(Hs), ptr(dh0), ptr(err), ptr(nrows))
    torch.cuda.synchronize()
    check('gather_pending', 'X', X[:n], msg_vals[ids[:n]], 0.0)
    check('gather_pending', 'H', Hs[:n], upd_vals[ids[:n]], 0.0)
    assert not dh0[:n].any(), 'dh_zero'
    for name, t in (('X', X), ('H', Hs), ('dh_zero', dh0)):
        untouched(name + ' past count', t[n:])
    assert float(nrows) == n
    assert int(err) == 0, 'equal clocks set an error bit'


@pytest.mark.parametrize('check_equal', [0, 1])
@pytest.mark.parametrize('form', ['null', 'below'])
def test_gather_pending_error_bits(check_equal, form):
    """Bit 4 (message older than the memory's clock) always, bit 8 (clocks differ) only with check_equal, and only
    for rows below the count."""
    N, cap, d = 40, 30, 4
    ids = torch.arange(cap) + 5
    msg_ts = torch.full((N,), 10.0)
    mem_ts = msg_ts.clone()
    cnt, n = count_of(form, cap)
    late, early = int(ids[n - 1]), int(ids[n - 2])          # both below the bound
    mem_ts[late] = 11.0                                     # memory clock past the message: bit 4 (and bit 8)
    mem_ts[early] = 9.0                                     # clocks differ: bit 8
    if n < cap:
        mem_ts[int(ids[n])] = 50.0                          # past the bound: must not count
    X, Hs, err = nan_dev(cap, d), nan_dev(cap, d), torch.zeros(1, dtype=torch.int32, device=DEV)
    call('tiger_train_gather_pending', ptr(cu(ids)), ptr(cnt), cap, ptr(cu(torch.zeros(N, d))), d,
         ptr(cu(msg_ts)), ptr(cu(torch.zeros(N, d))), d, ptr(cu(mem_ts)), check_equal, ptr(X), ptr(Hs), None,
         ptr(err), None)
    assert int(err) == 4 | (8 if check_equal else 0)
    if n < cap:                                             # the violation past the bound alone: no bit
        mem_ts[late], mem_ts[early] = 10.0, 10.0
        err.zero_()
        call('tiger_train_gather_pending', ptr(cu(ids)), ptr(cnt), cap, ptr(cu(torch.zeros(N, d))), d,
             ptr(cu(msg_ts)), ptr(cu(torch.zeros(N, d))), d, ptr(cu(mem_ts)), check_equal, ptr(X), ptr(Hs),
             None, ptr(err), None)
        assert int(err) == 0


# ------------------------------------------------------------------------------------------
# 3. shared pieces (zero_rows, relu_bwd, colsum, scatter_add_rows; dropout, axpy of train_seq.cu)
# ------------------------------------------------------------------------------------------
def test_zero_rows_with_ld_past_cols():
    gen = torch.Generator().manual_seed(0)
    rows, ld, cols = 333, 41, 30
    buf = torch.randn(rows, ld, generator=gen)
    flag = (torch.rand(rows, generator=gen) < 0.4).to(torch.uint8)
    want = buf.clone()
    want[flag.bool(), :cols] = 0
    got = cu(buf)
    call('tiger_train_zero_rows', ptr(got), ld, cols, rows, ptr(cu(flag)))
    assert torch.equal(got.cpu(), want)


@pytest.mark.parametrize('form', COUNT_FORMS)
def test_relu_bwd_matches_float64(form):
    """scale != 1, rows_per_count = 3, ld_dy != ld_y; y exactly 0 gives a zero gradient."""
    gen = torch.Generator().manual_seed(1)
    rows, cols, ld_dy, ld_y, per, scale = 301, 37, 45, 39, 3, 1.25
    dy, y = torch.randn(rows, ld_dy, generator=gen), torch.randn(rows, ld_y, generator=gen)
    y[torch.rand(rows, ld_y, generator=gen) < 0.2] = 0.0
    cnt, n = count_of(form, rows, per)
    x = y[:, :cols].double().requires_grad_()       # y = relu(x) with x = y: the ReLU gradient at x = 0 is 0
    (torch.relu(x)[:n] * dy[:n, :cols].double() * scale).sum().backward()
    got = cu(dy)
    call('tiger_train_relu_bwd', ptr(got), ld_dy, ptr(cu(y)), ld_y, cols, rows, ptr(cnt), per, scale)
    got = got.cpu()
    check('relu_bwd', 'dy', got[:n, :cols], x.grad[:n], EW_TOL)
    assert torch.equal(got[n:], dy[n:]) and torch.equal(got[:, cols:], dy[:, cols:]), 'rows / columns past the bound'
    assert not got[:n, :cols][y[:n, :cols] == 0].any(), 'y = 0 must give a zero gradient'


@pytest.mark.parametrize('form', COUNT_FORMS)
@pytest.mark.parametrize('cols', [1, 33, 344])
def test_colsum_matches_float64(cols, form):
    """6,600 rows = 26 slabs of 256; a count of 1,500 x per 4 ends inside a slab; out is accumulated onto."""
    gen = torch.Generator().manual_seed(cols)
    rows, ld, per, scale = 6600, cols + 3, 4, 0.75
    X = torch.randn(rows, ld, generator=gen)
    out0 = torch.randn(cols, generator=gen)
    cnt, n = count_of(form, rows, per)
    if form == 'below':
        cnt.fill_(1500)
        n = 6000
    want = out0.double() + scale * X[:n, :cols].double().sum(0)
    out = cu(out0)
    call('tiger_train_colsum', ptr(cu(X)), ld, rows, ptr(cnt), per, cols, scale, ptr(out))
    check('colsum', 'out', out, want, RED_TOL)


@pytest.mark.parametrize('form', COUNT_FORMS)
def test_scatter_add_rows_matches_float64(form):
    gen = torch.Generator().manual_seed(2)
    n, width, ld_src, n_tab, per, scale = 900, 19, 24, 31, 2, -0.5
    table0 = torch.randn(n_tab, width, generator=gen)
    ids = torch.randint(0, n_tab, (n,), generator=gen)          # many duplicates
    src = torch.randn(n, ld_src, generator=gen)
    cnt, m = count_of(form, n, per)
    want = table0.double().index_add(0, ids[:m], src[:m, :width].double() * scale)
    table = cu(table0)
    call('tiger_train_scatter_add_rows', ptr(table), ptr(cu(ids)), n, ptr(cnt), per, ptr(cu(src)), ld_src, width,
         scale)
    check('scatter_add_rows', 'table', table, want, RED_TOL)


@pytest.mark.parametrize('form', COUNT_FORMS)
@pytest.mark.parametrize('p,stream_id', [(0.0, 4), (0.1, 4), (0.3, 9)])
def test_dropout_and_axpy_match_float64(p, stream_id, form):
    gen = torch.Generator().manual_seed(3)
    n, per, seed, alpha = 5000, 7, 1234567, 0.37
    x0, y0 = torch.randn(n, generator=gen), torch.randn(n, generator=gen)
    cnt, m = count_of(form, n, per)
    x = cu(x0)
    call('tiger_train_dropout', ptr(x), ptr(cnt), per, n, p, seed, stream_id)
    want = x0.clone()
    if p > 0:
        keep = keep_mask(seed, stream_id, np.arange(m), p)
        want[:m] = torch.where(keep, x0[:m] * np.float32(inv_keep(p)), torch.zeros(()))
    check('dropout', 'x', x, want, EW_TOL)
    assert torch.equal(x[m:].cpu(), x0[m:]), 'dropout past the bound'
    y = cu(y0)
    call('tiger_train_axpy', ptr(y), ptr(cu(x0)), ptr(cnt), per, n, alpha)
    want = y0.double().clone()
    want[:m] += alpha * x0[:m].double()
    check('axpy', 'y', y, want, EW_TOL)
    assert torch.equal(y[m:].cpu(), y0[m:]), 'axpy past the bound'


# ------------------------------------------------------------------------------------------
# 4. link scorer (score_build, score_build_bwd, score_head, score_head_bwd)
# ------------------------------------------------------------------------------------------
def hit_codes_from_table(nn_, nids, B):
    """check_in_window's rule (data_loader.py:61-75) on the batch neighbor table [3B, K]: (src, dst, neg_src, neg_dst)."""
    src, dst, neg = nids[:B], nids[B:2 * B], nids[2 * B:]
    ns, nd, nn2 = nn_[:B], nn_[B:2 * B], nn_[2 * B:]
    return torch.cat([(nd == src[:, None]).any(1), (ns == dst[:, None]).any(1), (nn2 == src[:, None]).any(1),
                      (ns == neg[:, None]).any(1)]).long()


@pytest.mark.parametrize('mode,K', [('hits', 10), ('table', 5), ('table', 40), ('none', 10)])
@pytest.mark.parametrize('B,d', [(37, 10), (300, 172)])
def test_score_build_and_bwd_match_float64(mode, K, B, d):
    gen = torch.Generator().manual_seed(B + K)
    z = torch.randn(3 * B, d, generator=gen)
    emb = torch.randn(2, d, generator=gen)
    nids = torch.randint(1, 30, (3 * B,), generator=gen)
    nn_ = torch.randint(0, 30, (3 * B, K), generator=gen)
    hits = (torch.rand(4 * B, K, generator=gen) < 0.08).float()
    if mode == 'hits':
        codes = (hits.max(1).values > 0.5).long()
    elif mode == 'table':
        codes = hit_codes_from_table(nn_, nids, B)
    else:
        codes = torch.zeros(4 * B, dtype=torch.long)
    if mode != 'none':
        assert 0 < int(codes.sum()) < 4 * B, 'both codes should occur'
    # float64 restatement with autograd on z and the hit embedding
    zz, ee = z.double().requires_grad_(), emb.double().requires_grad_()
    he = (lambda c: ee[c]) if mode != 'none' else (lambda c: 0.0)
    x, y, ny = zz[:B], zz[B:2 * B], zz[2 * B:]
    c = codes.reshape(4, B)
    pair = torch.cat([torch.cat([x + he(c[0]), y + he(c[1])], 1), torch.cat([x + he(c[2]), ny + he(c[3])], 1)])
    dpair = torch.randn(2 * B, 2 * d, generator=gen)
    (pair * dpair.double()).sum().backward()
    got_pair = nan_dev(2 * B, 2 * d)
    got_codes = torch.full((4 * B,), 255, dtype=torch.uint8, device=DEV)
    use = mode != 'none'
    call('tiger_train_score_build', ptr(cu(z)), ptr(cu(hits)) if mode == 'hits' else None,
         ptr(cu(nn_)) if mode == 'table' else None, ptr(cu(nids)) if mode == 'table' else None, K,
         ptr(cu(emb)) if use else None, B, d, ptr(got_pair), ptr(got_codes) if use else None)
    check('score_build', 'pair', got_pair, pair, EW_TOL)
    if use:
        assert torch.equal(got_codes.cpu().long(), codes), 'hit codes'
    g_hit0 = torch.randn(2, d, generator=gen)
    dz, g_hit = nan_dev(3 * B, d), cu(g_hit0)
    call('tiger_train_score_build_bwd', ptr(cu(dpair)), ptr(got_codes) if use else None, B, d, ptr(dz), ptr(g_hit))
    check('score_build_bwd', 'dz', dz, zz.grad, EW_TOL)
    if use:
        check('score_build_bwd', 'g_hit', g_hit, g_hit0.double() + ee.grad, RED_TOL)
    else:
        assert torch.equal(g_hit.cpu(), g_hit0), 'codes = NULL must leave the hit gradient alone'


def test_score_build_bwd_grid_strides():
    """B = 2,400: 300 warps of rows over at most 148 CTAs of 8 warps each."""
    gen = torch.Generator().manual_seed(5)
    B, d = 2400, 36
    dpair = torch.randn(2 * B, 2 * d, generator=gen)
    codes = (torch.rand(4 * B, generator=gen) < 0.3).to(torch.uint8)
    zz, ee = torch.zeros(3 * B, d, dtype=torch.float64, requires_grad=True), torch.zeros(2, d, dtype=torch.float64,
                                                                                       requires_grad=True)
    c = codes.long().reshape(4, B)
    x, y, ny = zz[:B], zz[B:2 * B], zz[2 * B:]
    pair = torch.cat([torch.cat([x + ee[c[0]], y + ee[c[1]]], 1), torch.cat([x + ee[c[2]], ny + ee[c[3]]], 1)])
    (pair * dpair.double()).sum().backward()
    g_hit0 = torch.randn(2, d, generator=gen)
    dz, g_hit = nan_dev(3 * B, d), cu(g_hit0)
    call('tiger_train_score_build_bwd', ptr(cu(dpair)), ptr(cu(codes)), B, d, ptr(dz), ptr(g_hit))
    check('score_build_bwd', 'dz', dz, zz.grad, EW_TOL)
    check('score_build_bwd', 'g_hit', g_hit, g_hit0.double() + ee.grad, RED_TOL)


def score_head_inputs(B, d, gen):
    """hid = dropout(relu(x)) as the kernels hold it; fc2 scaled so that the scores spread over about +-60."""
    x = torch.randn(2 * B, d, generator=gen)
    x[torch.rand(2 * B, d, generator=gen) < 0.1] = 0.0
    w = torch.randn(d, generator=gen) * (60.0 / np.sqrt(d))
    b = torch.randn(1, generator=gen)
    return x, w, b


@pytest.mark.parametrize('p', [0.0, 0.1])
@pytest.mark.parametrize('B,d', [(37, 10), (700, 100), (700, 172)])
def test_score_head_and_bwd_match_float64(B, d, p):
    """2B = 1,400 rows (> 1,024) reach the single-CTA mean with several rows per thread; B = 37 is not a multiple of 32;
    d = 100 and 172 span several 32-column blocks of the backward, which must count g_b once."""
    gen = torch.Generator().manual_seed(B + d)
    seed, g = 4242, 0.7
    x, w, b = score_head_inputs(B, d, gen)
    hid_in = torch.relu(x)
    keep = keep_mask(seed, 2, np.arange(2 * B * d), p).reshape(2 * B, d)
    hid_dropped = torch.where(keep, hid_in * np.float32(inv_keep(p)), torch.zeros(()))
    hid = cu(hid_in)
    scores, loss, dscore = nan_dev(2 * B), nan_dev(1), nan_dev(2 * B)
    call('tiger_train_score_head', ptr(hid), ptr(cu(w)), ptr(cu(b)), B, d, p, seed, ptr(scores), ptr(loss),
         ptr(dscore))
    check('score_head', 'hid (dropped out in place)', hid, hid_dropped, EW_TOL)
    # float64 restatement: scores, BCE-with-logits mean, its gradient
    xx, ww, bb = x.double().requires_grad_(), w.double().requires_grad_(), b.double().requires_grad_()
    h = torch.relu(xx) * keep.double() * inv_keep(p)
    s = h @ ww + bb
    labels = torch.cat([torch.ones(B), torch.zeros(B)]).double()
    want_loss = torch.nn.functional.binary_cross_entropy_with_logits(s, labels)
    assert float(s.detach().abs().max()) > 40, 'the scores should reach the saturated range'
    check('score_head', 'scores', scores, s, RED_TOL)
    check('score_head', 'loss', loss, want_loss.reshape(1), RED_TOL)
    # dscore is element-wise given the scores: restate it from the kernel's own scores
    s_k = scores.cpu().double()
    check('score_head', 'dscore', dscore, (torch.sigmoid(s_k) - labels) / (2 * B), EW_TOL)
    # backward against autograd on the restatement: upstream g * dscore on the scores
    (s * g * dscore.cpu().double()).sum().backward()
    gw0, gb0 = torch.randn(d, generator=gen), torch.randn(1, generator=gen)
    dhid, gw, gb = nan_dev(2 * B, d), cu(gw0), cu(gb0)
    call('tiger_train_score_head_bwd', ptr(dscore), g, ptr(hid), ptr(cu(w)), B, d, p, ptr(dhid), ptr(gw), ptr(gb))
    check('score_head_bwd', 'dhid', dhid, xx.grad, EW_TOL)
    check('score_head_bwd', 'g_w', gw, gw0.double() + ww.grad, RED_TOL)
    check('score_head_bwd', 'g_b', gb, gb0.double() + bb.grad, RED_TOL)


# ------------------------------------------------------------------------------------------
# 5. mutual loss (tiger_train_mse)
# ------------------------------------------------------------------------------------------
def mse_case(n, d, form, gen, all_invalid=False, with_grad=True):
    n_t = 60
    pl, pr = torch.randn(n, d, generator=gen), torch.randn(n, d, generator=gen)
    hpl, hpr = torch.randn(n_t, d, generator=gen), torch.randn(n_t, d, generator=gen)
    hpl[::4] = 0.0                                   # never-written memory rows: excluded
    hpr[1::5] = 0.0
    if all_invalid:
        hpl.zero_(), hpr.zero_()
    index = torch.randint(0, n_t, (n,), generator=gen)   # repeated entries
    cnt, m = count_of(form, n)
    # float64 restatement (tiger.py:574-592) with autograd on the predictions
    a, b = pl.double().requires_grad_(), pr.double().requires_grad_()
    t = torch.cat([hpl[index[:m]], hpr[index[:m]]]).double()
    pred = torch.cat([a[:m], b[:m]])
    valid = ~(t == 0).all(1)
    loss = torch.nn.functional.mse_loss(pred[valid], t[valid]) if valid.any() else (pred * 0).sum()
    loss.backward()
    out = dict(loss=nan_dev(1), nv=nan_dev(1), work=nan_dev(2 * n))
    dl, dr = (nan_dev(n, d), nan_dev(n, d)) if with_grad else (None, None)
    call('tiger_train_mse', ptr(cu(pl)), ptr(cu(pr)), ptr(cu(hpl)), ptr(cu(hpr)), ptr(cu(index)), ptr(cnt), n, d,
         ptr(out['loss']), ptr(dl), ptr(dr), ptr(out['nv']), ptr(out['work']))
    torch.cuda.synchronize()
    return dict(m=m, want_loss=loss.detach(), want_nv=int(valid.sum()), ga=a.grad, gb=b.grad, dl=dl, dr=dr, **out)


@pytest.mark.parametrize('form', COUNT_FORMS)
@pytest.mark.parametrize('n,d', [(1, 3), (300, 100), (2048, 172)])
def test_mse_matches_float64(n, d, form):
    """Rows whose target is all zero are excluded; index repeats; the count bounds both halves."""
    r = mse_case(n, d, form, torch.Generator().manual_seed(n + d))
    m = r['m']
    check('mse', 'loss', r['loss'], r['want_loss'].reshape(1), RED_TOL)
    assert float(r['nv']) == r['want_nv']
    check('mse', 'dpred_l', r['dl'][:m], r['ga'][:m], EW_TOL)
    check('mse', 'dpred_r', r['dr'][:m], r['gb'][:m], EW_TOL)
    untouched('dpred_l past count', r['dl'][m:])
    untouched('dpred_r past count', r['dr'][m:])


def test_mse_all_rows_invalid_and_no_gradient_buffers():
    gen = torch.Generator().manual_seed(9)
    r = mse_case(50, 8, 'null', gen, all_invalid=True)
    assert float(r['loss']) == 0.0 and float(r['nv']) == 0.0
    assert float(r['dl'].abs().max()) == 0.0 and float(r['dr'].abs().max()) == 0.0
    r = mse_case(50, 8, 'below', gen, with_grad=False)          # dpred = NULL: the loss alone
    assert r['dl'] is None


def test_mse_row_limit():
    d, n = 4, 2049
    t = torch.zeros(n, d, device=DEV)
    index = torch.zeros(n, dtype=torch.int64, device=DEV)
    loss, work = nan_dev(1), nan_dev(2 * n)
    call('tiger_train_mse', ptr(t), ptr(t), ptr(t), ptr(t), ptr(index), None, n - 1, d, ptr(loss), None, None, None,
         ptr(work))
    with pytest.raises(TigerLibraryError, match='invalid argument'):
        call('tiger_train_mse', ptr(t), ptr(t), ptr(t), ptr(t), ptr(index), None, n, d, ptr(loss), None, None, None,
             ptr(work))


# ------------------------------------------------------------------------------------------
# 6. seq restarter (tiger_train_seq_pool, _bwd, seq_vbias, _bwd, seq_tokens_bwd)
# ------------------------------------------------------------------------------------------
def key_mask(gen, n, L):
    """Key-padding mask as SeqRestarter builds it (restarters.py:86): 1 = padded, the last position always live."""
    mask = (torch.rand(n, L, generator=gen) < 0.3).to(torch.uint8)
    mask[1::3, :] = 1                    # only the last position live
    mask[:, L - 1] = 0
    return mask


def seq_pool_case(n, L, dm, H, p, form='null', seed=777):
    gen = torch.Generator().manual_seed(n * 7 + L * 13 + dm + H + int(p * 10))
    hd = dm // H
    ld_qk = 2 * dm + 5
    qk = torch.randn(n * L, ld_qk, generator=gen)
    x = torch.randn(n * L, dm, generator=gen)
    mask = key_mask(gen, n, L)
    dxbar, dpsum = torch.randn(n, H, dm, generator=gen), torch.randn(n, H, generator=gen)
    cnt, m = count_of(form, n)
    # float64 restatement (SeqRestarter's self-attention, mean-pooled over the query positions) under autograd
    q = qk[:, :dm].double().reshape(n, L, H, hd).requires_grad_()
    k = qk[:, dm:2 * dm].double().reshape(n, L, H, hd).requires_grad_()
    xx = x.double().reshape(n, L, dm).requires_grad_()
    s = torch.einsum('nqhc,nkhc->nhqk', q / np.sqrt(hd), k).masked_fill(mask.bool()[:, None, None, :], float('-inf'))
    P = torch.softmax(s, -1)
    keep = keep_mask(seed, 3, np.arange(n * H * L * L), p).reshape(n, H, L, L)
    pbar = (P * keep.double() * inv_keep(p)).mean(2)
    psum = pbar.sum(-1)
    xbar = torch.einsum('nhj,njc->nhc', pbar, xx)
    ((xbar * dxbar.double())[:m].sum() + (psum * dpsum.double())[:m].sum()).backward()
    # the kernels
    qkd, xd = cu(qk), cu(x)
    Pk, pb, ps, xb = nan_dev(n * H * L * L), nan_dev(n * H * L), nan_dev(n * H), nan_dev(n * H * dm)
    call('tiger_train_seq_pool', ptr(qkd), ld_qk, ptr(xd), ptr(cu(mask)), ptr(cnt), n, L, dm, H, p, seed, ptr(Pk),
         ptr(pb), ptr(ps), ptr(xb))
    dX, dqk = nan_dev(n * L, dm), nan_dev(n * L, ld_qk)
    call('tiger_train_seq_pool_bwd', ptr(cu(dxbar)), ptr(cu(dpsum)), ptr(xd), ptr(qkd), ld_qk, ptr(Pk), ptr(pb),
         ptr(cnt), n, L, dm, H, p, seed, ptr(dX), ptr(dqk))
    torch.cuda.synchronize()
    return dict(m=m, P=P, pbar=pbar, psum=psum, xbar=xbar, q=q, k=k, x=xx, Pk=Pk.reshape(n, H, L, L),
                pb=pb.reshape(n, H, L), ps=ps.reshape(n, H), xb=xb.reshape(n, H, dm), dX=dX.reshape(n, L, dm),
                dqk=dqk.reshape(n, L, ld_qk))


def check_seq_pool(r, dm, H):
    m = r['m']
    hd = dm // H
    check('seq_pool', 'P', r['Pk'][:m], r['P'][:m], RED_TOL)
    check('seq_pool', 'pbar', r['pb'][:m], r['pbar'][:m], RED_TOL)
    check('seq_pool', 'psum', r['ps'][:m], r['psum'][:m], RED_TOL)
    check('seq_pool', 'xbar', r['xb'][:m], r['xbar'][:m], RED_TOL)
    check('seq_pool_bwd', 'dX (value path)', r['dX'][:m], r['x'].grad[:m], RED_TOL)
    n, L = r['x'].shape[:2]
    check('seq_pool_bwd', 'dq (score path)', r['dqk'][:m, :, :dm].reshape(m, L, H, hd), r['q'].grad[:m], RED_TOL)
    check('seq_pool_bwd', 'dk (score path)', r['dqk'][:m, :, dm:2 * dm].reshape(m, L, H, hd), r['k'].grad[:m],
          RED_TOL)
    untouched('dqk columns past 2 d_model', r['dqk'][:, :, 2 * dm:])
    for name in ('Pk', 'pb', 'ps', 'xb', 'dX', 'dqk'):
        untouched(name + ' past count', r[name][m:])


@pytest.mark.parametrize('p', [0.0, 0.1])
@pytest.mark.parametrize('dm,H', [(43, 1), (80, 2), (860, 2)])
@pytest.mark.parametrize('L', [1, 4, 33, 40, 64])
def test_seq_pool_and_bwd_match_float64(L, dm, H, p):
    """d_model 43 = 4 x 10 + 3 (xbar's scalar path), head_dim 40 crosses the 32-column chunks, 860 / 2 heads is the
    BASELINE shape; L = 64 is SP_MAXL.  dpsum is non-zero, so the score path carries the psum gradient too."""
    check_seq_pool(seq_pool_case(5, L, dm, H, p), dm, H)


@pytest.mark.parametrize('form', COUNT_FORMS)
def test_seq_pool_count_forms(form):
    check_seq_pool(seq_pool_case(7, 33, 80, 2, 0.1, form=form), 80, 2)


def test_seq_pool_refuses_long_histories():
    t = torch.zeros(65 * 2, 16, device=DEV)
    mask = torch.zeros(2, 65, dtype=torch.uint8, device=DEV)
    for fn, args in (('tiger_train_seq_pool', (ptr(t), 16, ptr(t), ptr(mask), None, 2, 65, 8, 1, 0.0, 1, ptr(t), ptr(t),
                                               ptr(t), ptr(t))),
                     ('tiger_train_seq_pool_bwd', (ptr(t), ptr(t), ptr(t), ptr(t), 16, ptr(t), ptr(t), None, 2, 65, 8,
                                                   1, 0.0, 1, ptr(t), ptr(t)))):
        with pytest.raises(TigerLibraryError, match='invalid argument'):
            call(fn, *args)


@pytest.mark.parametrize('form', COUNT_FORMS)
@pytest.mark.parametrize('dm,H', [(43, 1), (80, 2), (860, 2)])
def test_seq_vbias_and_bwd_match_float64(dm, H, form):
    gen = torch.Generator().manual_seed(dm + H)
    n = 300
    hd = dm // H
    att0, psum, bv = torch.randn(n, dm, generator=gen), torch.rand(n, H, generator=gen) * 2, torch.randn(dm, generator=gen)
    datt = torch.randn(n, dm, generator=gen)
    cnt, m = count_of(form, n)
    ps, bb = psum.double().requires_grad_(), bv.double().requires_grad_()
    out = att0.double() + (ps[:, :, None] * bb.reshape(H, hd)).reshape(n, dm)
    (out[:m] * datt[:m].double()).sum().backward()
    att = cu(att0)
    call('tiger_train_seq_vbias', ptr(att), ptr(cu(psum)), ptr(cu(bv)), ptr(cnt), n, dm, H)
    check('seq_vbias', 'att', att[:m], out[:m], EW_TOL)
    assert torch.equal(att[m:].cpu(), att0[m:]), 'seq_vbias past count'
    gbv0 = torch.randn(dm, generator=gen)
    gbv, dps = cu(gbv0), nan_dev(n, H)
    call('tiger_train_seq_vbias_bwd', ptr(cu(datt)), ptr(cu(psum)), ptr(cu(bv)), ptr(cnt), n, dm, H, ptr(gbv), ptr(dps))
    check('seq_vbias_bwd', 'g_bv', gbv, gbv0.double() + bb.grad, RED_TOL)
    check('seq_vbias_bwd', 'dpsum', dps[:m], ps.grad[:m], RED_TOL)
    untouched('dpsum past count', dps[m:])


# ------------------------------------------------------------------------------------------
# 7. time-code gradients at large dt (seq_tokens_bwd, attn_build_bwd_ex)
# ------------------------------------------------------------------------------------------
def time_params(gen, d):
    """TimeEncode's initial basis (time_encoding.py): 1 / 10^linspace(0, 9, d), and a random phase."""
    return torch.from_numpy((1 / 10 ** np.linspace(0, 9, d)).astype(np.float32)), torch.randn(d, generator=gen)


@pytest.mark.parametrize('form', COUNT_FORMS)
@pytest.mark.parametrize('L', [1, 4, 33, 64])
def test_seq_tokens_bwd_matches_float64_at_large_dt(L, form):
    """Repeated anonymised ids; the last position gets no embedding gradient; dt up to 1e6 s."""
    gen = torch.Generator().manual_seed(L)
    n, d, de = 9, 10, 3
    dm = 4 * d + de
    dX = torch.randn(n * L, dm, generator=gen)
    anony = torch.randint(0, L + 1, (n * L,), generator=gen)
    hist_ts = torch.sort(torch.rand(n, L, generator=gen) * 1e6, 1).values
    tw, tb = time_params(gen, d)
    cnt, m = count_of(form, n)
    # float64 restatement of the token columns (restarters.py:96-104) under autograd
    an = torch.zeros(L + 1, d, dtype=torch.float64, requires_grad=True)
    w, b = tw.double().requires_grad_(), tb.double().requires_grad_()
    notlast = (torch.arange(n * L) % L != L - 1).double()[:, None]
    dt32 = (hist_ts[:, -1:] - hist_ts).reshape(-1, 1)                  # float32 difference, as the kernel forms it
    arg = straight_through(dt32.double() * w + b, time_arg32(dt32.numpy(), tw.numpy(), tb.numpy()))
    tok_an, tok_tc = an[anony] * notlast, torch.cos(arg)
    rows = slice(0, m * L)
    ((tok_an * dX[:, 2 * d:3 * d].double())[rows].sum() + (tok_tc * dX[:, 3 * d + de:].double())[rows].sum()).backward()
    g_an0, gw0, gb0 = torch.randn(L + 1, d, generator=gen), torch.randn(d, generator=gen), torch.randn(d, generator=gen)
    g_an, gw, gb = cu(g_an0), cu(gw0), cu(gb0)
    call('tiger_train_seq_tokens_bwd', ptr(cu(dX)), ptr(cnt), n, L, ptr(cu(anony)), ptr(cu(hist_ts)), d, de, ptr(cu(tw)),
         ptr(cu(tb)), ptr(g_an), ptr(gw), ptr(gb))
    check('seq_tokens_bwd', 'g_anony_emb', g_an, g_an0.double() + an.grad, RED_TOL)
    check('time_code_grad', 'seq g_time_w', gw, gw0.double() + w.grad, RED_TOL)
    check('time_code_grad', 'seq g_time_b', gb, gb0.double() + b.grad, RED_TOL)


@pytest.mark.parametrize('ts_group', [1, 4])
def test_attn_build_bwd_ex_matches_float64_at_large_dt(ts_group):
    """The TimeEncode gradients of the attention builder at dt up to 1e6 s (the builder test stops at dt <= 20),
    with the representation gradients accumulated onto a non-zero dh_new."""
    gen = torch.Generator().manual_seed(ts_group)
    N, B, K, d, de = 60, 7, 4, 16, 5
    nq = 3 * B * (K if ts_group > 1 else 1)
    E, C = 2 * d, 2 * d + de
    center = torch.randint(0, N, (nq,), generator=gen)
    nn_ = torch.randint(1, N, (nq, K), generator=gen)
    nn_[torch.rand(nq, K, generator=gen) < 0.3] = 0
    nn_[::5] = 0
    ts = torch.rand(B, generator=gen) * 1e6
    q_ts = ts[(torch.arange(nq) // ts_group) % B]
    nt_ = q_ts[:, None] * torch.rand(nq, K, generator=gen)
    n_rows = 25
    sel = torch.full((N,), -1, dtype=torch.int32)
    sel[torch.randperm(N, generator=gen)[:n_rows]] = torch.arange(n_rows, dtype=torch.int32)
    tw, tb = time_params(gen, d)
    dkv, dq, dcat = torch.randn(nq * K, C, generator=gen), torch.randn(nq, E, generator=gen), \
        torch.randn(nq, E + d, generator=gen)
    # float64 restatement with autograd on the GRU rows and the time encoder
    rb = torch.zeros(n_rows, d, dtype=torch.float64, requires_grad=True)
    w, b = tw.double().requires_grad_(), tb.double().requires_grad_()

    def repr_(ids):
        s = sel[ids].long()
        return torch.where((s >= 0)[:, None], rb[s.clamp(min=0)], torch.zeros((), dtype=torch.float64))

    flat = nn_.reshape(-1)
    dt32 = (q_ts[:, None] - nt_).reshape(-1, 1)
    arg = straight_through(dt32.double() * w + b, time_arg32(dt32.numpy(), tw.numpy(), tb.numpy()))
    real = (flat != 0).double()[:, None]
    loss = ((repr_(flat) * dkv[:, :d].double() + torch.cos(arg) * dkv[:, d + de:].double()) * real).sum() + \
        (repr_(center) * (dq[:, :d] + dcat[:, E:]).double()).sum() + (torch.cos(b) * dq[:, d:].double()).sum()
    loss.backward()
    h0, gw0, gb0 = torch.randn(n_rows, d, generator=gen), torch.randn(d, generator=gen), torch.randn(d, generator=gen)
    dh, gw, gb = cu(h0), cu(gw0), cu(gb0)
    call('tiger_train_attn_build_bwd_ex', ptr(cu(dkv)), ptr(cu(dq)), ptr(cu(dcat)), E + d, E, ptr(cu(center)), nq,
         ptr(cu(ts)), B, ts_group, ptr(cu(nn_)), ptr(cu(nt_)), K, ptr(cu(sel)), d, de, ptr(cu(tw)), ptr(cu(tb)), ptr(dh),
         None, ptr(gw), ptr(gb))
    check('attn_build_bwd', 'dh_new', dh, h0.double() + rb.grad, RED_TOL)
    check('time_code_grad', 'attn g_time_w', gw, gw0.double() + w.grad, RED_TOL)
    check('time_code_grad', 'attn g_time_b', gb, gb0.double() + b.grad, RED_TOL)
