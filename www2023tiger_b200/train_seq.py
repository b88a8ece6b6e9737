"""Training step of the seq restarter (SeqRestarter.forward under autograd: reference tiger/model/restarters.py:51-114
as called from TIGER.contrast_and_mutual_learning, tiger.py:574-590) on the kernels of csrc/train_seq.cu and the
tensor-core products of csrc/gemm.cu.  Used by `www2023tiger_b200.train.NativeTrainer`."""
import os

import torch
from torch import Tensor

from . import ops
from ._lib import call, ptr

f32, i64, u8 = torch.float32, torch.int64, torch.uint8


class SeqRestarterTrainer:
    """`cap` rows for forward + backward (the collated unique positives: <= 2B), `cap_fwd` >= cap rows for forward-only
    calls (lazy restart of up to every involved node, in train() mode with the reference's dropout)."""

    def __init__(self, module, fp, cap: int, device, cap_fwd: int = 0):
        self.m, self.fp, self.cap = module, fp, cap
        self.cap_fwd = cf = max(cap, cap_fwd)
        self.d, self.de, self.L, self.H = module.nfeat_dim, module.efeat_dim, module.hist_len, module.n_head
        self.dm = module.d_model
        self.p = float(module.dropout)
        d, L, dm, H = self.d, self.L, self.dm, self.H
        z = lambda *s, dt=f32: torch.zeros(*s, dtype=dt, device=device)
        self.X, self.QK = z(cf * L, dm), z(cf * L, 2 * dm)
        self.mask, self.prev_ts = z(cf, L, dt=u8), z(cf)
        self.P, self.pbar, self.psum = z(cf * H * L * L), z(cf * H * L), z(cf * H)
        self.xbar, self.att, self.o, self.hid = z(cf, H * dm), z(cf, dm), z(cf, dm), z(cf, d)
        self.dX, self.dQK = z(cap * L, dm), z(cap * L, 2 * dm)
        self.dxbar, self.dpsum = z(cap, H * dm), z(cap * H)
        self.datt, self.do = z(cap, dm), z(cap, dm)
        self.dhid, self.dh_left = z(cap, d), z(cap, d)
        # names of this module's parameters inside the flat buffers
        self.prefix = next(n for n, p in zip(fp.names, fp.params) if p is module.anony_emb.weight)[:-len('anony_emb.weight')]
        self._ctx = None
        # few rows (the lazy restart of a steady-state batch) take the matrix-vector tail of csrc/restart_seq.cu, many
        # rows (the collated positives, the first batches of a chunk) the tensor-core products: ops.SeqRestarterOp
        self.tail_rows = int(os.environ.get('TIGER_SEQ_TAIL_ROWS', '64')) if dm <= 1024 else 0
        self.cnt_gate = z(2, dt=torch.int32)

    def _names(self):
        r = self.prefix
        return dict(tw=r + 'time_encoder.basis_freq', tb=r + 'time_encoder.phase', an=r + 'anony_emb.weight',
                    in_w=r + 'mha_fn.in_proj_weight', in_b=r + 'mha_fn.in_proj_bias', out_w=r + 'mha_fn.out_proj.weight',
                    out_b=r + 'mha_fn.out_proj.bias', fn_w=r + 'out_fn.weight', fn_b=r + 'out_fn.bias',
                    fc1_w=r + 'merger.fc1.weight', fc1_b=r + 'merger.fc1.bias', fc2_w=r + 'merger.fc2.weight',
                    fc2_b=r + 'merger.fc2.bias')

    def forward(self, nids: Tensor, hist, fg, pred_l: Tensor, pred_r: Tensor, seed: int, train: bool, *, n: int,
                count: Tensor = None, seed_stream: int = 0):
        """h(t'-), h(t'+) of `nids` into pred_l / pred_r [n, d]; hist = (hist_nids, hist_eids, hist_ts, hist_dirs,
        anonymized_ids), each [n, L].  `count` (device int32) bounds the rows actually processed."""
        assert n <= self.cap_fwd
        d, de, L, dm, H = self.d, self.de, self.L, self.dm, self.H
        hd = dm // H
        P, N = self.fp.p, self._names()
        p = self.p if train else 0.0
        seed = (seed + 7919 * seed_stream) & 0x7fffffff
        hn, he, ht, hdirs, an = hist
        call('tiger_seq_tokens', ptr(nids), ptr(count), n, L, ptr(hn), ptr(he), ptr(ht), ptr(hdirs), ptr(an),
             ptr(fg.nfeats), ptr(fg.efeats), d, de, ptr(P[N['an']]), ptr(P[N['tw']]), ptr(P[N['tb']]), ptr(self.X),
             ptr(self.mask), ptr(self.prev_ts))
        in_w, in_b = P[N['in_w']], P[N['in_b']]
        mc = dict(m_count=count)
        ops.sgemm_big(self.X, in_w[:2 * dm], self.QK, m=n * L, n=2 * dm, k=dm, bias=in_b[:2 * dm], m_count=count,
                      rows_per_count=L)
        call('tiger_train_seq_pool', ptr(self.QK), 2 * dm, ptr(self.X), ptr(self.mask), ptr(count), n, L, dm, H, p, seed,
             ptr(self.P), ptr(self.pbar), ptr(self.psum), ptr(self.xbar))
        ctx = dict(n=n, count=count, p=p, seed=seed, an=an, ht=ht, pred_l=pred_l, keep=(hn, he, hdirs, nids))
        if self.tail_rows > 0 and (count is not None or n <= self.tail_rows):
            small = None
            if count is not None:
                call('tiger_seq_gate_count', ptr(count), self.tail_rows, ptr(self.cnt_gate), ptr(self.cnt_gate[1:]))
                small, count = self.cnt_gate, self.cnt_gate[1:]
                mc = dict(m_count=count)
            fc1_w = P[N['fc1_w']]
            call('tiger_seq_tail', ptr(self.xbar), ptr(small), n, dm, H, d, ptr(in_w[2 * dm:]), ptr(in_b[2 * dm:]),
                 ptr(P[N['out_w']]), ptr(P[N['out_b']]), ptr(P[N['fn_w']]), ptr(P[N['fn_b']]), ptr(fc1_w), fc1_w.stride(0),
                 ptr(P[N['fc1_b']]), ptr(P[N['fc2_w']]), ptr(P[N['fc2_b']]), ptr(self.psum), p, seed, ptr(self.att),
                 ptr(self.o), ptr(self.hid), ptr(pred_l), ptr(pred_r))
            if small is None:
                self._ctx = ctx
                return
        for h in range(H):
            rows = slice(2 * dm + h * hd, 2 * dm + (h + 1) * hd)
            ops.sgemm_ex(self.xbar[:, h * dm:(h + 1) * dm], in_w[rows], self.att[:, h * hd:(h + 1) * hd], m=n, n=hd, k=dm,
                         **mc)
        call('tiger_train_seq_vbias', ptr(self.att), ptr(self.psum), ptr(in_b[2 * dm:]), ptr(count), n, dm, H)
        ops.sgemm_ex(self.att, P[N['out_w']], self.o, m=n, n=dm, k=dm, bias=P[N['out_b']], relu=True, **mc)
        ops.sgemm_ex(self.o, P[N['fn_w']], pred_l, m=n, n=d, k=dm, bias=P[N['fn_b']], **mc)
        # the merger's second input is identically zero (restarters.py:103-104, SURVEY.md Q13): only the first d
        # input columns of fc1 take part
        ops.sgemm_ex(pred_l, P[N['fc1_w']][:, :d], self.hid, m=n, n=d, k=d, bias=P[N['fc1_b']], relu=True, **mc)
        call('tiger_train_dropout', ptr(self.hid), ptr(count), d, n * d, p, seed, 4)
        ops.sgemm_ex(self.hid, P[N['fc2_w']], pred_r, m=n, n=d, k=d, bias=P[N['fc2_b']], **mc)
        self._ctx = ctx

    def backward(self, dpred_l: Tensor, dpred_r: Tensor, g: float):
        ctx = self._ctx
        self._ctx = None
        n, count, p, seed = ctx['n'], ctx['count'], ctx['p'], ctx['seed']
        assert n <= self.cap
        d, de, L, dm, H = self.d, self.de, self.L, self.dm, self.H
        hd = dm // H
        P, G, N = self.fp.p, self.fp.g, self._names()
        inv_keep = 1.0 / (1.0 - p) if p > 0 else 1.0
        wg = dict(trans_a=True, trans_w=True, accumulate=True, k_parts=ops.wgrad_k_parts(n), k_count=count)  # weight gradients
        dg = dict(trans_w=True, m_count=count)                                               # input gradients
        colsum = lambda x, cols, out, scale=1.0, rows=n, per=1: call(
            'tiger_train_colsum', ptr(x), x.stride(0), rows, ptr(count), per, cols, float(scale), ptr(out))
        # merger.fc2 (scaled by the upstream gradient g from here on)
        ops.sgemm_ex(dpred_r, self.hid, G[N['fc2_w']], m=d, n=d, k=n, alpha=g, **wg)
        colsum(dpred_r, d, G[N['fc2_b']], g)
        ops.sgemm_ex(dpred_r, P[N['fc2_w']], self.dhid, m=n, n=d, k=d, alpha=g, **dg)
        call('tiger_train_relu_bwd', ptr(self.dhid), d, ptr(self.hid), d, d, n, ptr(count), 1, float(inv_keep))
        # merger.fc1 (first d input columns)
        ops.sgemm_ex(self.dhid, ctx['pred_l'], G[N['fc1_w']][:, :d], m=d, n=d, k=n, **wg)
        colsum(self.dhid, d, G[N['fc1_b']])
        ops.sgemm_ex(self.dhid, P[N['fc1_w']][:, :d], self.dh_left, m=n, n=d, k=d, **dg)
        call('tiger_train_axpy', ptr(self.dh_left), ptr(dpred_l), ptr(count), d, n * d, float(g))
        # out_fn, ReLU, out-projection
        ops.sgemm_ex(self.dh_left, self.o, G[N['fn_w']], m=d, n=dm, k=n, **wg)
        colsum(self.dh_left, d, G[N['fn_b']])
        ops.sgemm_ex(self.dh_left, P[N['fn_w']], self.do, m=n, n=dm, k=d, **dg)
        call('tiger_train_relu_bwd', ptr(self.do), dm, ptr(self.o), dm, dm, n, ptr(count), 1, 1.0)
        ops.sgemm_ex(self.do, self.att, G[N['out_w']], m=dm, n=dm, k=n, **wg)
        colsum(self.do, dm, G[N['out_b']])
        ops.sgemm_ex(self.do, P[N['out_w']], self.datt, m=n, n=dm, k=dm, **dg)
        # value projection (per head, on the pooled tokens) and its bias term
        in_w, g_in_w, in_b, g_in_b = P[N['in_w']], G[N['in_w']], P[N['in_b']], G[N['in_b']]
        call('tiger_train_seq_vbias_bwd', ptr(self.datt), ptr(self.psum), ptr(in_b[2 * dm:]), ptr(count), n, dm, H,
             ptr(g_in_b[2 * dm:]), ptr(self.dpsum))
        for h in range(H):
            rows = slice(2 * dm + h * hd, 2 * dm + (h + 1) * hd)
            da = self.datt[:, h * hd:(h + 1) * hd]
            ops.sgemm_ex(da, self.xbar[:, h * dm:(h + 1) * dm], g_in_w[rows], m=hd, n=dm, k=n, **wg)
            ops.sgemm_ex(da, in_w[rows], self.dxbar[:, h * dm:(h + 1) * dm], m=n, n=dm, k=hd, **dg)
        # attention probabilities -> q / k, value path -> tokens
        call('tiger_train_seq_pool_bwd', ptr(self.dxbar), ptr(self.dpsum), ptr(self.X), ptr(self.QK), 2 * dm, ptr(self.P),
             ptr(self.pbar), ptr(count), n, L, dm, H, p, seed, ptr(self.dX), ptr(self.dQK))
        ops.sgemm_big(self.dQK, self.X, g_in_w[:2 * dm], m=2 * dm, n=dm, k=n * L, trans_a=True, trans_w=True,
                      accumulate=True, k_parts=ops.wgrad_k_parts(n * L), k_count=count, rows_per_count=L)
        colsum(self.dQK, 2 * dm, g_in_b[:2 * dm], rows=n * L, per=L)
        ops.sgemm_big(self.dQK, in_w[:2 * dm], self.dX, m=n * L, n=dm, k=2 * dm, trans_w=True, accumulate=True,
                      m_count=count, rows_per_count=L)
        call('tiger_train_seq_tokens_bwd', ptr(self.dX), ptr(count), n, L, ptr(ctx['an']), ptr(ctx['ht']), d, de,
             ptr(P[N['tw']]), ptr(P[N['tb']]), ptr(G[N['an']]), ptr(G[N['tw']]), ptr(G[N['tb']]))
