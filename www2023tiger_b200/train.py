"""The training step of the drop-in TIGER model on hand-written kernels: forward that keeps what backward needs,
hand-written backward, Adam - what `loss.backward(); optimizer.step()` of the reference's loops runs through autograd
(train_self_supervised.py:165-171, train_self_supervised_ddp.py:203-208; model function
TIGER.contrast_and_mutual_learning, tiger/model/tiger.py:547-592).

`NativeTrainer` adopts the parameters of a `tiger.model.tiger.TIGER` (this package's mirror of the reference class):
they are re-pointed into ONE flat fp32 buffer (with a flat gradient buffer and flat Adam moments beside it), so the
optimizer is one kernel and the DDP gradient all-reduce is one NCCL call over one bucket.  The module keeps working
as an nn.Module (state_dict, eval route, torch optimizers): only the storage of `p.data` moved.

Step (B events, K neighbors; all data-dependent counts stay on the device):
  forward   compaction of the involved / pending sets -> gather of the pending messages -> GRU (2 tensor-core
            products + gates) -> attention (row builder, q / k / v products, single-query core with dropout,
            out-projection, merger) -> argmax-by-timestamp + right write-back (+ restarter targets) -> link scorer
            (pair rows, first layer, dropout + second layer + BCE) -> restarter on the collated batch + mutual loss
            -> message build + store, left write-back
  backward  scorer -> merger -> out-projection -> attention core -> q / k / v products -> scatter onto the GRU rows
            and TimeEncode gradients -> GRU gates -> GRU weight gradients; restarter backward
With n_layers = 2 the attention is two chains (temporal_agg_modules.py:79-104): depth 1 (fns.1) embeds the 3BK hop-1
neighbors over the second hop, depth 2 (fns.0) the 3B batch nodes over the first hop with its slots keyed by the depth-1
output.  Backward runs depth 2 (slot gradients into the depth-1 output's gradient), then depth 1, then the GRU.
  update    [gradient all-reduce] -> Adam (zeroes the gradient buffer for the next step)
Dense products: ops.sgemm_ex (tcgen05, tf32x3): y = x W^T, dx = dy W, dW += dy^T x on the tensors as stored.
"""
from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from . import _lib, ops
from ._lib import call, ptr, raise_on_err_flags

f32, i32, i64, u8 = torch.float32, torch.int32, torch.int64, torch.uint8


class FlatParams:
    """Parameters of a module re-pointed into one flat buffer (+ gradient and Adam moment buffers of the same
    layout).  Shared parameters (the time encoder is registered under three names, tiger.py:71-72) appear once.

    torch.optim.Adam keeps one step counter per tensor and skips tensors whose gradient is None; which tensors those
    are in a given step is data dependent (no pending message -> the GRU cell is not used, no valid target row -> the
    restarter gets no gradient).  `group_of(name)` puts every tensor into group 0 (always), 1 (GRU cell) or 2
    (restarter); the two gate values sit behind the last tensor of the flat GRADIENT buffer (so they take part in the
    gradient all-reduce) and are written by the step's kernels."""

    ALIGN = 4     # floats: every tensor starts on a 16-byte boundary
    N_GATES = 4

    def __init__(self, module: torch.nn.Module, group_of=lambda name: 0):
        seen, self.names, self.params = set(), [], []
        for name, p in module.named_parameters():
            if id(p) in seen:
                continue
            seen.add(id(p))
            self.names.append(name)
            self.params.append(p)
        dev = self.params[0].device
        self.offsets, off = [], 0
        for p in self.params:
            self.offsets.append(off)
            off += (p.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        self.numel = off
        self.flat = torch.zeros(off, dtype=f32, device=dev)
        self.grad_all = torch.zeros(off + self.N_GATES, dtype=f32, device=dev)     # [gradients | gates]
        self.grad = self.grad_all[:off]
        self.gates = self.grad_all[off:]
        self.exp_avg = torch.zeros(off, dtype=f32, device=dev)
        self.exp_avg_sq = torch.zeros(off, dtype=f32, device=dev)
        self.g: Dict[str, Tensor] = {}
        self.p: Dict[str, Tensor] = {}
        for name, p, o in zip(self.names, self.params, self.offsets):
            view = self.flat[o:o + p.numel()].view(p.shape)
            view.copy_(p.data)
            p.data = view
            self.p[name] = view
            self.g[name] = self.grad[o:o + p.numel()].view(p.shape)
        self.groups = [int(group_of(n)) for n in self.names]
        self.seg_start = torch.tensor(self.offsets + [off], dtype=i64, device=dev)
        self.seg_group = torch.tensor(self.groups, dtype=i32, device=dev)
        self.seg_step = torch.zeros(len(self.names), dtype=i32, device=dev)
        self.seg_bc = torch.zeros(2 * len(self.names), dtype=f32, device=dev)
        self.max_seg = max(p.numel() for p in self.params)

    def comm_ranges(self):
        """Three contiguous slices of the flat gradient buffer, in the order the backward pass completes them:
        restarter (+ the gates), attention / hit embedding / scorer, time encoder + GRU - so that each can be
        all-reduced while the rest of the backward pass still runs.  None when the parameter order differs."""
        first = lambda prefix: next((o for n, o in zip(self.names, self.offsets) if n.startswith(prefix)), None)
        a, r = first('temporal_embedding_fn.'), first('restarter_fn.')
        order_ok = a is not None and r is not None and a < r and all(
            (o < a) == n.startswith(('time_encoder.', 'right_mem_updater.')) and (o >= r) == n.startswith('restarter_fn.')
            for n, o in zip(self.names, self.offsets))
        if not order_ok:
            return None
        total = self.grad_all.numel()
        return {'restarter': (r, total), 'attention': (a, r), 'gru': (0, a)}

    def reset_optimizer(self):
        self.exp_avg.zero_(), self.exp_avg_sq.zero_(), self.grad_all.zero_(), self.seg_step.zero_()

    def adam(self, lr: float, betas=(0.9, 0.999), eps: float = 1e-8, grad_scale: float = 1.0, zero_grad: bool = True):
        call('tiger_train_adam', ptr(self.flat), ptr(self.grad), ptr(self.exp_avg), ptr(self.exp_avg_sq),
             ptr(self.seg_start), ptr(self.seg_group), ptr(self.seg_step), ptr(self.seg_bc), len(self.names),
             ptr(self.gates), self.max_seg, float(lr), float(betas[0]), float(betas[1]), float(eps), float(grad_scale),
             int(zero_grad))
        # the kernel wrote the parameters through raw pointers: bump their version counters so that the weight packs of
        # the inference operators (keyed on (data_ptr, _version) in tiger/model/*.py) are rebuilt before the next eval
        torch._C._increment_version(self.params)


_SEED_WORDS: Dict[int, Tensor] = {}


def _seed_step_word(device) -> Tensor:
    """The device word the dropout kernels add (x 101) to their seeds: one per device, registered with the library once
    and zero except while a captured training step replays (NativeTrainer.capture_stream)."""
    idx = torch.device(device).index
    idx = torch.cuda.current_device() if idx is None else idx
    if idx not in _SEED_WORDS:
        word = torch.zeros(1, dtype=i32, device=torch.device('cuda', idx))
        with torch.cuda.device(idx):
            rc = _lib.load().tiger_train_seed_step(word.data_ptr())
        if rc != 0:
            raise _lib.TigerLibraryError(f'tiger_train_seed_step failed with code {rc}')
        _SEED_WORDS[idx] = word
    return _SEED_WORDS[idx]


# Largest neighborhood the training kernels take: the attention core keeps one dropout bit per slot in a 32-bit word
# (ATT_MAXK, csrc/train.cu).  The seq restarter's limits are the inference kernels' (ops.seq_restarter_limit_error).
# Larger models train through the torch-op route, which has neither limit.
MAX_NEIGHBORS = 32


def native_limit_error(model) -> Optional[str]:
    """Why the native step cannot train `model` at its sizes, or None when it can."""
    if model.n_neighbors > MAX_NEIGHBORS:
        return (f'native training takes at most {MAX_NEIGHBORS} neighbors per query (the attention core keeps one '
                f'dropout bit per slot in a 32-bit word); this model has n_neighbors={model.n_neighbors}')
    r = model.restarter_fn
    if type(r).__name__ == 'SeqRestarter':
        limit = ops.seq_restarter_limit_error(r.nfeat_dim, r.efeat_dim, r.hist_len, r.n_head)
        if limit is not None:
            return 'native training: ' + limit
    return None


def _param_group(name: str) -> int:
    if name.startswith('right_mem_updater.'):
        return 1
    if name.startswith('restarter_fn.'):
        return 2
    return 0


def _linear_fwd(x, w, b, out, *, m, relu=False, m_count=None, per=1):
    ops.sgemm_big(x, w, out, m=m, n=w.shape[0], k=w.shape[1], bias=b, relu=relu, m_count=m_count, rows_per_count=per)


class _AttnLayer:
    """Activations (kept for backward) and gradients of one attention chain of the step: nq queries, K slots each."""

    def __init__(self, nq: int, K: int, H: int, d: int, E: int, C: int, z):
        self.q_in, self.kv_in, self.cat = z(nq, E), z(nq * K, C), z(nq, E + d)
        self.Qp, self.KV, self.attn = z(nq, E), z(nq * K, 2 * E), z(nq, E)
        self.P, self.keep, self.empty = z(nq * H * K), z(nq * H, dt=i32), z(nq, dt=u8)
        self.hid, self.z = z(nq, d), z(nq, d)
        self.dz, self.dhid, self.dcat, self.dattn = z(nq, d), z(nq, d), z(nq, E + d), z(nq, E)
        self.dQ, self.dKV, self.dkv_in, self.dq_in = z(nq, E), z(nq * K, 2 * E), z(nq * K, C), z(nq, E)


def _linear_bwd(dy, x, w, gw, gb, dx, *, m, count=None, per=1, accumulate_dx=False):
    """dy [m, n], x [m, k], w [n, k]: gw += dy^T x, gb += colsum(dy), dx (=|+=) dy w.  `count` bounds m on the device."""
    n, k = w.shape
    if gw is not None:
        ops.sgemm_big(dy, x, gw, m=n, n=k, k=m, trans_a=True, trans_w=True, accumulate=True,
                      k_parts=ops.wgrad_k_parts(m), k_count=count, rows_per_count=per)
    if gb is not None:
        call('tiger_train_colsum', ptr(dy), dy.stride(0), m, ptr(count), per, n, 1.0, ptr(gb))
    if dx is not None:
        ops.sgemm_big(dy, w, dx, m=m, n=k, k=n, trans_w=True, m_count=count, rows_per_count=per,
                      accumulate=accumulate_dx)


class NativeTrainer:
    def __init__(self, model, batch_size: int, *, lr: float = 1e-4, seed: int = 0):
        # class names, not isinstance: the drop-in package is importable both as `tiger` (PYTHONPATH, the way the
        # reference's drivers see it) and as `www2023tiger_b200.tiger`
        kind = lambda o: type(o).__name__
        if not (kind(model.msg_transform_fn) == 'IdentityMessageFunction' and kind(model.right_mem_updater) == 'GRUUpdater'
                and model.n_layers in (1, 2) and model.hit_type in ('bin', 'none')):
            raise NotImplementedError('native training covers the default operator variants '
                                      '(tsfm_fn id, upd_fn gru, n_layers 1|2, hit_type bin|none)')
        limit = native_limit_error(model)
        if limit is not None:
            raise NotImplementedError(limit)
        self.model = model
        # a static restarter owns a time encoder it never uses (restarters.py:17-33,254-277): never stepped (group 3)
        static = type(model.restarter_fn).__name__ == 'StaticRestarter'
        self.fp = FlatParams(model, lambda n: 3 if (static and n.startswith('restarter_fn.time_encoder.'))
                             else _param_group(n))
        self.lr, self.seed, self.n_steps = lr, seed, 0
        dev = self.fp.flat.device
        self.device = dev
        fn = model.temporal_embedding_fn.fns[0]
        self.B, self.K, self.H = batch_size, model.n_neighbors, fn.n_head
        self.d, self.de = model.nfeat_dim, model.efeat_dim
        self.M, self.E, self.C = model.raw_msg_dim, 2 * model.nfeat_dim, 2 * model.nfeat_dim + model.efeat_dim
        self.p_attn = float(fn.dropout)
        self.p_score = float(model.score_fn.dropout.p)
        B, K, d, E, C, M = self.B, self.K, self.d, self.E, self.C, self.M
        N = model.n_nodes
        self.n_layers = model.n_layers
        # involved-node capacity as in TigerEngine / _Workspace: with the second hop the 3BK hop-1 neighbors are
        # queries too, and no list holds more than the N distinct nodes
        self.cap = cap = 3 * B * (K + 1) if self.n_layers == 1 else min((3 * B + 3 * B * K) * (K + 1), N)
        z = lambda *s, dt=f32: torch.zeros(*s, dtype=dt, device=dev)
        # --- compaction scratch
        self.bitmap = z(ops.bitmap_words(N), dt=i32)
        self.involved, self.outdated = z(cap, dt=i64), z(cap, dt=i64)
        self.gru_row = torch.full((N,), -1, dtype=i32, device=dev)
        self.counts = z(4, dt=i32)
        self.err = z(1, dt=i32)
        # --- GRU
        self.X, self.Hs = z(cap, M), z(cap, d)
        self.Gi, self.Gh, self.dGi, self.dGh = z(cap, 3 * d), z(cap, 3 * d), z(cap, 3 * d), z(cap, 3 * d)
        self.h_new, self.dh_new = z(cap, d), z(cap, d)
        self.r, self.zg, self.n = z(cap, d), z(cap, d), z(cap, d)
        # --- attention: fns.0 over the batch nodes; with two layers fns.1 over their 3BK neighbors (depth 1)
        self.att = _AttnLayer(3 * B, K, self.H, d, E, C, z)
        self.att1 = _AttnLayer(3 * B * K, K, self.H, d, E, C, z) if self.n_layers == 2 else None
        # --- steps 4-6
        self.winner = z(2 * B, dt=u8)
        self.hprev_left, self.hprev_right = z(2 * B, d), z(2 * B, d)
        # --- scorer
        self.pair, self.codes, self.hid_s = z(2 * B, 2 * d), z(4 * B, dt=u8), z(2 * B, d)
        self.scores, self.closs, self.dscore = z(2 * B), z(1), z(2 * B)
        self.dhid_s, self.dpair = z(2 * B, d), z(2 * B, 2 * d)
        # --- restarter / mutual loss
        self.mloss = z(1)
        self.mse_work = z(4 * B)
        self.pred_l, self.pred_r = z(2 * B, d), z(2 * B, d)
        self.dpred_l, self.dpred_r = z(2 * B, d), z(2 * B, d)
        self.restarter = model.restarter_fn
        if kind(self.restarter) == 'StaticRestarter':
            self.rkind = 'static'
        elif kind(self.restarter) == 'SeqRestarter':
            self.rkind = 'seq'
            from .train_seq import SeqRestarterTrainer
            self.seq = SeqRestarterTrainer(self.restarter, self.fp, 2 * B, dev)
        else:
            raise NotImplementedError(kind(self.restarter))
        self._ctx = None
        self._graph = self.g_inp = self.g_count = self._g_args = None
        self._g_base = self._g_replays = 0

    # ------------------------------------------------------------------ parameter handles
    def P_(self, name: str) -> Tensor:
        return self.fp.p[name]

    def G_(self, name: str) -> Tensor:
        return self.fp.g[name]

    def check_errors(self):
        v = int(self.err.item()) & 0xffffffff
        if v:
            self.err.zero_()
            raise_on_err_flags(v)

    # ------------------------------------------------------------------ forward
    def forward(self, src: Tensor, dst: Tensor, neg: Tensor, ts: Tensor, eids: Tensor, cg, *, contrast_only: bool = False,
                train: bool = True) -> Tuple[Tensor, Tensor]:
        """The drop-in entry (batch + ComputationGraph from GraphCollator) -> (contrast_loss [1], mutual_loss [1])
        device tensors; memory state advanced like the reference's contrast_and_mutual_learning.  `train=False`
        switches dropout off (eval-mode forward of the same program)."""
        m = self.model
        B = len(src)
        assert B <= self.B
        nn_, ne_, nt_ = cg.layers[self.n_layers]        # the batch nodes' neighbors
        hop2 = cg.layers[1] if self.n_layers == 2 else None
        batch_nids = torch.cat([src, dst, neg]).contiguous()
        ts = ts.to(f32).contiguous()
        # pending set of the involved nodes (tiger.py:206-209)
        ops.mark_nodes(cg.computation_graph_nodes.contiguous(), self.bitmap, m.n_nodes)
        ops.compact_involved(self.bitmap, m.n_nodes, self.involved, self.counts, has_msg=m.msg_store.has_msg,
                             outdated=self.outdated, gru_row=self.gru_row, err_flags=self.err)
        hits = torch.stack(list(cg.hit_data)).to(f32).contiguous() if m.hit_type == 'bin' else None     # [4, B, K]
        rd = cg.restart_data
        targets = None
        if not contrast_only:
            hist = None
            if self.rkind == 'seq':
                hist = tuple(t.contiguous() for t in (rd.hist_nids, rd.hist_eids, rd.hist_ts, rd.hist_dirs,
                                                      rd.anonymized_ids))
            targets = dict(nids=rd.nids.contiguous(), index=rd.index.contiguous(), n=rd.nids.numel(), count=None, hist=hist)
        return self._core(B, batch_nids, ts, eids.contiguous(), nn_, ne_, nt_, hop2, hits=hits, hits_from_table=False,
                          targets=targets, train=train)

    def _core(self, B, batch_nids, ts, eids, nn_, ne_, nt_, hop2, *, hits, hits_from_table, targets, train):
        """Steps 1-7 of TIGE.contrast_learning + the restarter targets, after the involved / pending compaction.
        hop2: (nids, eids, ts) [3BK, K] of the second hop with n_layers = 2, else None."""
        m = self.model
        K, d, de, M, cap = self.K, self.d, self.de, self.M, self.cap
        nq = 3 * B
        P = self.fp.p
        self.n_steps += 1
        seed = (self.seed * 1000003 + self.n_steps * 101) & 0x7fffffff
        p_attn = self.p_attn if train else 0.0
        p_score = self.p_score if train else 0.0
        pos = batch_nids[:2 * B]
        left, right, store = m.left_memory, m.right_memory, m.msg_store
        msg_mem, upd_mem = m.msg_memory, m.upd_memory
        fg = m.raw_feat_getter
        cnt_o = self.counts[1:]
        # ---- steps 1-2: gather of the pending messages, GRU (tiger.py:206-221)
        call('tiger_train_gather_pending', ptr(self.outdated), ptr(cnt_o), cap, ptr(store.node_msg_vals), M,
             ptr(store.node_msg_ts), ptr(upd_mem.vals), d, ptr(msg_mem.update_ts), int(m.msg_src == 'left'),
             ptr(self.X), ptr(self.Hs), ptr(self.dh_new), ptr(self.err), ptr(self.fp.gates))
        c = 'right_mem_updater.cell.'
        _linear_fwd(self.X, P[c + 'weight_ih'], P[c + 'bias_ih'], self.Gi, m=cap, m_count=cnt_o)
        _linear_fwd(self.Hs, P[c + 'weight_hh'], P[c + 'bias_hh'], self.Gh, m=cap, m_count=cnt_o)
        call('tiger_train_gru_gates', ptr(self.Gi), ptr(self.Gh), ptr(self.Hs), ptr(cnt_o), cap, d, ptr(self.h_new),
             ptr(self.r), ptr(self.zg), ptr(self.n))
        # ---- step 3: temporal attention (temporal_agg_modules.py:29-104,210-235)
        tw, tb = P['time_encoder.basis_freq'], P['time_encoder.phase']
        key_rows = None
        if hop2 is not None:
            # depth 1 (fns.1): the 3BK hop-1 neighbors at their parent event's time over the second hop; its own
            # dropout seed (stream 2 of the seed_stream convention, stream 1 is the lazy restart's)
            n2, e2, t2 = hop2
            self._attn_fwd(self.att1, 1, nn_, nq * K, ts, B, K, n2, e2, t2, None, p_attn,
                           (seed + 7919 * 2) & 0x7fffffff)
            key_rows = self.att1.z
        self._attn_fwd(self.att, 0, batch_nids, nq, ts, B, 1, nn_, ne_, nt_, key_rows, p_attn, seed)
        # ---- step 4 + restarter targets (tiger.py:230-251), no grad
        winner = self.winner[:2 * B]
        ops.select_latest(pos, ts, want_unique=False, winner=winner, want_count=False)
        ops.right_writeback(pos, winner, self.gru_row, self.h_new, d, right.vals, right.update_ts, right.active_mask,
                            store.node_msg_ts, store.has_msg, left.vals, self.hprev_left, self.hprev_right, self.err)
        # ---- step 7: link scorer (tiger.py:259-288)
        use_hits = hits is not None or hits_from_table
        call('tiger_train_score_build', ptr(self.att.z), ptr(hits), ptr(nn_) if hits_from_table else None,
             ptr(batch_nids) if hits_from_table else None, K, ptr(P['hit_embedding.weight']) if use_hits else None, B, d,
             ptr(self.pair), ptr(self.codes) if use_hits else None)
        s = 'score_fn.'
        _linear_fwd(self.pair, P[s + 'fc1.weight'], P[s + 'fc1.bias'], self.hid_s, m=2 * B, relu=True)
        call('tiger_train_score_head', ptr(self.hid_s), ptr(P[s + 'fc2.weight']), ptr(P[s + 'fc2.bias']), B, d, p_score,
             seed, ptr(self.scores), ptr(self.closs), ptr(self.dscore))
        # ---- restarter on the collated batch + mutual loss (tiger.py:574-590)
        if targets is not None:
            n_pos, nids, cnt = targets['n'], targets['nids'], targets['count']
            if self.rkind == 'static':
                for side, out in (('left', self.pred_l), ('right', self.pred_r)):
                    call('tiger_gather_rows', ptr(P[f'restarter_fn.{side}_emb.weight']), d, ptr(nids), n_pos, ptr(out),
                         None, None)
            else:
                self.seq.forward(nids, targets['hist'], fg, self.pred_l, self.pred_r, seed, train, n=n_pos, count=cnt)
            call('tiger_train_mse', ptr(self.pred_l), ptr(self.pred_r), ptr(self.hprev_left), ptr(self.hprev_right),
                 ptr(targets['index']), ptr(cnt), n_pos, d, ptr(self.mloss), ptr(self.dpred_l), ptr(self.dpred_r),
                 ptr(self.fp.gates[1:]), ptr(self.mse_work))
        else:
            self.mloss.zero_()
        # ---- steps 5-6 (tiger.py:244-255), no grad
        ops.store_messages(batch_nids[:B], batch_nids[B:2 * B], eids, ts, winner, msg_mem.vals, msg_mem.update_ts,
                           fg.nfeats, fg.efeats, d, de, tw, tb, store.node_msg_vals, store.node_msg_ts, store.has_msg,
                           self.err)
        ops.left_writeback(pos, B, winner, self.att.z, d, ts, left.vals, left.update_ts, left.active_mask, self.err)
        self._ctx = dict(B=B, batch_nids=batch_nids, ts=ts, nn=nn_, nt=nt_, hop2=hop2, hits=use_hits, targets=targets,
                         p_attn=p_attn, p_score=p_score, seed=seed, keepalive=(ne_, hits, eids))
        return self.closs, self.mloss

    def _attn_fwd(self, L: _AttnLayer, fn: int, center, nq, ts, B, ts_group, nn_, ne_, nt_, key_rows, p_attn, seed):
        """One TemporalAttention (temporal_embedding_fn.fns.<fn>) of nq queries with dropout p_attn."""
        m, P = self.model, self.fp.p
        K, H, d, de, E = self.K, self.H, self.d, self.de, self.E
        fg = m.raw_feat_getter
        a = f'temporal_embedding_fn.fns.{fn}.'
        call('tiger_train_attn_build_ex', ptr(center), nq, ptr(ts), B, ts_group, ptr(nn_), ptr(ne_), ptr(nt_), K,
             ptr(m.right_memory.vals), ptr(self.h_new), ptr(key_rows), ptr(self.gru_row), ptr(fg.nfeats),
             ptr(fg.efeats), d, de, ptr(P['time_encoder.basis_freq']), ptr(P['time_encoder.phase']), ptr(L.q_in),
             ptr(L.kv_in), ptr(L.cat), E + d, E)
        in_b = P[a + 'mha_fn.in_proj_bias']
        _linear_fwd(L.q_in, P[a + 'mha_fn.q_proj_weight'], in_b[:E], L.Qp, m=nq)
        _linear_fwd(L.kv_in, P[a + 'mha_fn.k_proj_weight'], in_b[E:2 * E], L.KV[:, :E], m=nq * K)
        _linear_fwd(L.kv_in, P[a + 'mha_fn.v_proj_weight'], in_b[2 * E:], L.KV[:, E:], m=nq * K)
        call('tiger_train_attn_core', ptr(L.Qp), E, ptr(L.KV), ptr(L.KV[:, E:]), 2 * E, ptr(nn_), nq, K, H, E // H,
             p_attn, seed, ptr(L.attn), E, ptr(L.P), ptr(L.keep), ptr(L.empty))
        _linear_fwd(L.attn, P[a + 'mha_fn.out_proj.weight'], P[a + 'mha_fn.out_proj.bias'], L.cat[:, :E], m=nq)
        call('tiger_train_zero_rows', ptr(L.cat), E + d, E, nq, ptr(L.empty))
        _linear_fwd(L.cat, P[a + 'merger.fc1.weight'], P[a + 'merger.fc1.bias'], L.hid, m=nq, relu=True)
        _linear_fwd(L.hid, P[a + 'merger.fc2.weight'], P[a + 'merger.fc2.bias'], L.z, m=nq)

    # ------------------------------------------------------------------ device-resident stream (bench / DDP loop)
    def attach_stream(self, csr: ops.DeviceCSR, hist_len: int = 40):
        """Buffers of the sync-free loop: the temporal neighbor finder, the lazy restart of not-yet-seen nodes and the
        collation of the restarter targets all run on the device from one [5B] int64 batch record (layout of
        TigerEngine.inp: src | dst | neg | eids | ts as float64 bits) - what GraphCollator + the driver's restart
        bookkeeping (train_self_supervised_ddp.py:186-199) do on the host in the reference."""
        m, dev, B, K, cap = self.model, self.device, self.B, self.K, self.cap
        z = lambda *s, dt=f32: torch.zeros(*s, dtype=dt, device=dev)
        self.csr, self.L = csr, hist_len
        self.nn_, self.ne_, self.nt_ = z(3 * B, K, dt=i64), z(3 * B, K, dt=i64), z(3 * B, K)
        self.hop2 = None
        if self.n_layers == 2:        # the second hop: float64 query times of the hop-1 neighbors, the [3BK, K] table
            self.nt64 = z(3 * B * K, dt=torch.float64)
            self.hop2 = (z(3 * B * K, K, dt=i64), z(3 * B * K, K, dt=i64), z(3 * B * K, K))
        self.ts32 = z(B)
        self.uptodate = z(m.n_nodes, dt=u8)
        self.restart_nodes = z(cap, dt=i64)
        self.t_uniq, self.t_index, self.t_count = z(2 * B, dt=i64), z(2 * B, dt=i64), z(1, dt=i32)
        self.t_winner = z(2 * B, dt=u8)
        if self.rkind == 'seq':
            L = hist_len
            from .train_seq import SeqRestarterTrainer
            self.seq = SeqRestarterTrainer(self.restarter, self.fp, 2 * B, dev, cap_fwd=cap)
            self.tmin = z(1, dt=torch.float64)
            mk = lambda n: (z(n, L, dt=i64), z(n, L, dt=i64), z(n, L), z(n, L, dt=i64), z(n, L, dt=i64))
            self.r_hist, self.t_hist = mk(cap), mk(2 * B)
            self.r_left, self.r_right = z(cap, self.d), z(cap, self.d)

    def reset_stream(self):
        self.model.reset()
        self.model.msg_store.has_msg.zero_()
        self.uptodate.zero_()

    def forward_stream(self, inp: Tensor, *, lazy_restart: bool = True, train: bool = True):
        m, B, K, d, cap = self.model, self.B, self.K, self.d, self.cap
        assert inp.numel() == 5 * B and inp.dtype == i64
        batch_nids, pos, eids = inp[:3 * B], inp[:2 * B], inp[3 * B:4 * B]
        ts64 = inp[4 * B:].view(torch.float64)
        left, right, store, fg = m.left_memory, m.right_memory, m.msg_store, m.raw_feat_getter
        # ---- neighbor finder + involved / pending / restart lists (GraphCollator.collate_memory_nodes, the drivers'
        #      restart sets) ----
        ops.find_recent(self.csr, batch_nids, ts64, K, ts_period=B, want_dirs=False, ts32_out=self.ts32,
                        bitmap=self.bitmap, out=(self.nn_, self.ne_, self.nt_, None))
        if self.hop2 is not None:
            ops.find_second_hop(self.csr, self.nn_, self.nt_, K, ts64=self.nt64, bitmap=self.bitmap, out=self.hop2)
        ops.compact_involved(self.bitmap, m.n_nodes, self.involved, self.counts, has_msg=store.has_msg,
                             uptodate=self.uptodate if lazy_restart else None, outdated=self.outdated,
                             gru_row=self.gru_row, restart_nodes=self.restart_nodes if lazy_restart else None,
                             err_flags=self.err)
        seed0 = (self.seed * 1000003 + (self.n_steps + 1) * 101) & 0x7fffffff
        if lazy_restart:                                            # TIGER.restart (tiger.py:594-609)
            R = self.counts[2:]
            if self.rkind == 'static':
                P = self.fp.p
                ops.static_restart(self.restart_nodes, cap, self.csr, P['restarter_fn.left_emb.weight'],
                                   P['restarter_fn.right_emb.weight'], d, count=R, batch_ts=self.ts32,
                                   left_vals=left.vals, left_ts=left.update_ts, left_active=left.active_mask,
                                   right_vals=right.vals, right_ts=right.update_ts, right_active=right.active_mask,
                                   has_msg=store.has_msg)
            else:
                ops.min_time(self.ts32, self.tmin)
                hn, he, ht, hd, an = self.r_hist
                ops.find_recent(self.csr, self.restart_nodes, self.tmin, self.L, ts_period=1, count=R,
                                out=(hn, he, ht, hd))
                ops.anonymized_reindex(hn, out=an, count=R)
                # train() mode: the reference's restart applies the restarter's dropout (the call sits inside the
                # training loop, train_self_supervised_ddp.py:193-199)
                self.seq.forward(self.restart_nodes, self.r_hist, fg, self.r_left, self.r_right, seed0, train, n=cap,
                                 count=R, seed_stream=1)
                ops.scatter_rows(left.vals, self.restart_nodes, self.r_left, ts_table=left.update_ts, ts=self.seq.prev_ts,
                                 active=left.active_mask, count=R)
                ops.scatter_rows(right.vals, self.restart_nodes, self.r_right, ts_table=right.update_ts,
                                 ts=self.seq.prev_ts, active=right.active_mask, count=R)
        # ---- restarter targets: collate_restart_data (data_loader.py:95-168) on the device: unique positives by
        #      float64 time, their histories at those times ----
        call('tiger_select_latest', ptr(pos), ptr(ts64), 1, 2 * B, B, 0, None, None, None, ptr(self.t_winner),
             ptr(self.t_uniq), ptr(self.t_index), ptr(self.t_count))
        hist = None
        if self.rkind == 'seq':
            sel_ts = ts64[self.t_index % B]
            hn, he, ht, hd, an = self.t_hist
            ops.find_recent(self.csr, self.t_uniq, sel_ts, self.L, count=self.t_count, out=(hn, he, ht, hd))
            ops.anonymized_reindex(hn, out=an, count=self.t_count)
            hist = self.t_hist
        targets = dict(nids=self.t_uniq, index=self.t_index, n=2 * B, count=self.t_count, hist=hist)
        return self._core(B, batch_nids, self.ts32, eids, self.nn_, self.ne_, self.nt_, self.hop2, hits=None,
                          hits_from_table=(m.hit_type == 'bin'), targets=targets, train=train)

    # ------------------------------------------------------------------ CUDA-graph replay of the stream step
    def capture_stream(self, *, mutual_coef: float = 1.0, grad_scale: float = 1.0, lr: Optional[float] = None,
                       allreduce=None, sliced: bool = True):
        """Arms the CUDA-graph replay of forward_stream + backward [+ the sliced gradient all-reduce] + Adam; `step_stream`
        then copies the 8 kB batch record into the graph's input buffer and replays.  The eager step is bound by the
        host - 78 (static restarter) to 139 (seq) C-ABI calls from Python per step, ~1.05 ms / ~2.9 ms of issue time
        against 1.08 / 3.03 ms per step (bench.py `host_issue_ms_per_step`) - the replay costs two calls.
        Dropout: the captured kernels carry the capture step's seed and add a device-side step counter
        (csrc/common.cuh: tiger_step_seed): the graph copies its replay count into the registered word at its start
        and clears the word at its end, so replay k draws the masks of eager step k while eager launches between
        replays (of this or any other trainer) see zero.  The first two `step_stream` calls still launch eagerly (they
        create the lazily sized workspaces and, with `allreduce`, the NCCL communicator), the third one captures; calls
        with other arguments than the captured ones (`allreduce` must be the same callable) stay eager.  NCCL
        collectives issued through torch.distributed are capturable: the slices become graph nodes on NCCL's stream
        beside the rest of the backward pass."""
        assert self._graph is None, 'release_graph() first'
        self.g_inp = torch.zeros(5 * self.B, dtype=i64, device=self.device)
        self.g_count = torch.zeros(1, dtype=i32, device=self.device)
        self._g_args = dict(mutual_coef=mutual_coef, grad_scale=grad_scale, lr=lr, allreduce=allreduce, sliced=sliced)
        return self

    def _capture_now(self, inp: Tensor):
        a = self._g_args
        word = _seed_step_word(self.device)
        self.g_inp.copy_(inp)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        base = self.n_steps
        self.g_count.zero_()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            word.copy_(self.g_count)
            closs, mloss = self._step_eager(self.g_inp, **a)
            word.zero_()
            self.g_count.add_(1)
        self.n_steps = base                    # the capture itself ran nothing
        self._graph, self._g_base, self._g_out, self._g_replays = graph, base, (closs, mloss), 0

    def release_graph(self):
        """Back to eager launches."""
        self._graph = self.g_inp = self.g_count = self._g_args = None

    def step_stream(self, inp: Tensor, *, mutual_coef: float = 1.0, grad_scale: float = 1.0, allreduce=None,
                    lr: Optional[float] = None, sliced: bool = True):
        key = dict(mutual_coef=mutual_coef, grad_scale=grad_scale, lr=lr, allreduce=allreduce, sliced=sliced)
        if self._g_args is not None and self._g_args == key and (self._graph is not None or self.n_steps >= 2):
            if self._graph is None:
                self._capture_now(inp)
            if self.n_steps != self._g_base + self._g_replays:      # eager steps in between: re-align the counter
                self.g_count.fill_(self.n_steps - self._g_base)
                self._g_replays = self.n_steps - self._g_base
            self.g_inp.copy_(inp, non_blocking=True)
            self._graph.replay()
            self.n_steps += 1
            self._g_replays += 1
            torch._C._increment_version(self.fp.params)
            return self._g_out
        return self._step_eager(inp, **key)

    def _step_eager(self, inp: Tensor, *, mutual_coef, grad_scale, allreduce, lr, sliced):
        closs, mloss = self.forward_stream(inp)
        if allreduce is None:
            self.backward(1.0, mutual_coef)
        else:
            # one bucket per slice of the flat gradient buffer, started as soon as the backward pass has completed it
            ranges = self.fp.comm_ranges() if sliced else None
            works = []
            if ranges is None:
                self.backward(1.0, mutual_coef)
                works.append(allreduce(self.fp.grad_all))
            else:
                self.backward(1.0, mutual_coef,
                              comm=lambda name: works.append(allreduce(self.fp.grad_all[ranges[name][0]:ranges[name][1]])))
            for w in works:
                if w is not None:
                    w.wait()
        self.fp.adam(self.lr if lr is None else lr, grad_scale=grad_scale)
        return closs, mloss

    # ------------------------------------------------------------------ backward
    def backward(self, g_contrast: float = 1.0, g_mutual: float = 1.0, comm=None):
        """Accumulates d(g_contrast * contrast_loss + g_mutual * mutual_loss)/d(parameters) into the flat gradient
        buffer (call once per forward).  `comm(slice_name)` is called as soon as a slice of the gradient buffer
        (FlatParams.comm_ranges) is complete: the DDP loop starts that slice's all-reduce there, beside the rest of
        the backward pass - the restarter runs first because it is the longest part and depends on nothing else."""
        ctx = self._ctx
        assert ctx is not None, 'backward() needs a forward()'
        self._ctx = None
        B, K, d, cap = ctx['B'], self.K, self.d, self.cap
        nq = 3 * B
        P, G = self.fp.p, self.fp.g
        cnt_o = self.counts[1:]
        s, c = 'score_fn.', 'right_mem_updater.cell.'
        # ---- restarter
        tg = ctx['targets']
        if tg is not None and g_mutual != 0.0:
            if self.rkind == 'static':
                for side, dp in (('left', self.dpred_l), ('right', self.dpred_r)):
                    call('tiger_train_scatter_add_rows', ptr(G[f'restarter_fn.{side}_emb.weight']), ptr(tg['nids']),
                         tg['n'], ptr(tg['count']), 1, ptr(dp), d, d, float(g_mutual))
            else:
                self.seq.backward(self.dpred_l, self.dpred_r, float(g_mutual))
        if comm is not None:
            comm('restarter')
        # ---- scorer
        call('tiger_train_score_head_bwd', ptr(self.dscore), float(g_contrast), ptr(self.hid_s), ptr(P[s + 'fc2.weight']),
             B, d, ctx['p_score'], ptr(self.dhid_s), ptr(G[s + 'fc2.weight']), ptr(G[s + 'fc2.bias']))
        _linear_bwd(self.dhid_s, self.pair, P[s + 'fc1.weight'], G[s + 'fc1.weight'], G[s + 'fc1.bias'], self.dpair,
                    m=2 * B)
        call('tiger_train_score_build_bwd', ptr(self.dpair), ptr(self.codes) if ctx['hits'] else None, B, d,
             ptr(self.att.dz), ptr(G['hit_embedding.weight']) if ctx['hits'] else None)
        # ---- attention weight gradients, then the representation gradients back onto the GRU rows (+ TimeEncode
        #      gradients).  Two layers: depth 2's slot gradients are depth 1's output gradient, and the attention slice
        #      of the gradient buffer is complete only after depth 1's weight gradients
        hop2 = ctx['hop2']
        self._attn_bwd(self.att, 0, nq, ctx['p_attn'])
        if hop2 is None:
            if comm is not None:
                comm('attention')
            self._build_bwd(self.att, ctx['batch_nids'], nq, ctx['ts'], B, 1, ctx['nn'], ctx['nt'], None)
        else:
            self._build_bwd(self.att, ctx['batch_nids'], nq, ctx['ts'], B, 1, ctx['nn'], ctx['nt'], self.att1.dz)
            self._attn_bwd(self.att1, 1, nq * K, ctx['p_attn'])
            if comm is not None:
                comm('attention')
            self._build_bwd(self.att1, ctx['nn'], nq * K, ctx['ts'], B, K, hop2[0], hop2[2], None)
        # ---- GRU (inputs are detached messages / memory buffers: weight gradients only)
        call('tiger_train_gru_gates_bwd', ptr(self.dh_new), ptr(self.r), ptr(self.zg), ptr(self.n), ptr(self.Gh),
             ptr(self.Hs), ptr(cnt_o), cap, d, ptr(self.dGi), ptr(self.dGh))
        _linear_bwd(self.dGi, self.X, P[c + 'weight_ih'], G[c + 'weight_ih'], G[c + 'bias_ih'], None, m=cap,
                    count=cnt_o)
        _linear_bwd(self.dGh, self.Hs, P[c + 'weight_hh'], G[c + 'weight_hh'], G[c + 'bias_hh'], None, m=cap,
                    count=cnt_o)
        if comm is not None:
            comm('gru')

    def _attn_bwd(self, L: _AttnLayer, fn: int, nq: int, p_attn: float):
        """Backward of one TemporalAttention from L.dz: merger (MergeLayer: fc2(relu(fc1([out | c])))),
        out-projection, core, q / k / v products -> weight gradients, L.dq_in, L.dkv_in, L.dcat."""
        K, H, d, E = self.K, self.H, self.d, self.E
        P, G = self.fp.p, self.fp.g
        a = f'temporal_embedding_fn.fns.{fn}.'
        _linear_bwd(L.dz, L.hid, P[a + 'merger.fc2.weight'], G[a + 'merger.fc2.weight'], G[a + 'merger.fc2.bias'],
                    L.dhid, m=nq)
        call('tiger_train_relu_bwd', ptr(L.dhid), d, ptr(L.hid), d, d, nq, None, 1, 1.0)
        _linear_bwd(L.dhid, L.cat, P[a + 'merger.fc1.weight'], G[a + 'merger.fc1.weight'], G[a + 'merger.fc1.bias'],
                    L.dcat, m=nq)
        call('tiger_train_zero_rows', ptr(L.dcat), E + d, E, nq, ptr(L.empty))
        _linear_bwd(L.dcat[:, :E], L.attn, P[a + 'mha_fn.out_proj.weight'], G[a + 'mha_fn.out_proj.weight'],
                    G[a + 'mha_fn.out_proj.bias'], L.dattn, m=nq)
        call('tiger_train_attn_core_bwd', ptr(L.dattn), E, ptr(L.Qp), E, ptr(L.KV), ptr(L.KV[:, E:]), 2 * E, ptr(L.P),
             ptr(L.keep), nq, K, H, E // H, p_attn, ptr(L.dQ), ptr(L.dKV), ptr(L.dKV[:, E:]))
        g_in_b = G[a + 'mha_fn.in_proj_bias']
        _linear_bwd(L.dQ, L.q_in, P[a + 'mha_fn.q_proj_weight'], G[a + 'mha_fn.q_proj_weight'], g_in_b[:E], L.dq_in,
                    m=nq)
        _linear_bwd(L.dKV[:, :E], L.kv_in, P[a + 'mha_fn.k_proj_weight'], G[a + 'mha_fn.k_proj_weight'],
                    g_in_b[E:2 * E], L.dkv_in, m=nq * K)
        _linear_bwd(L.dKV[:, E:], L.kv_in, P[a + 'mha_fn.v_proj_weight'], G[a + 'mha_fn.v_proj_weight'],
                    g_in_b[2 * E:], L.dkv_in, m=nq * K, accumulate_dx=True)

    def _build_bwd(self, L: _AttnLayer, center, nq, ts, B, ts_group, nn_, nt_, d_key_rows):
        """Row-builder backward: representation gradients onto dh_new (slots into d_key_rows when given), TimeEncode
        gradients."""
        P, G, d, E = self.fp.p, self.fp.g, self.d, self.E
        call('tiger_train_attn_build_bwd_ex', ptr(L.dkv_in), ptr(L.dq_in), ptr(L.dcat), E + d, E, ptr(center), nq,
             ptr(ts), B, ts_group, ptr(nn_), ptr(nt_), self.K, ptr(self.gru_row), d, self.de,
             ptr(P['time_encoder.basis_freq']), ptr(P['time_encoder.phase']), ptr(self.dh_new), ptr(d_key_rows),
             ptr(G['time_encoder.basis_freq']), ptr(G['time_encoder.phase']))

    # ------------------------------------------------------------------ whole step
    def step(self, src, dst, neg, ts, eids, cg, *, mutual_coef: float = 1.0, contrast_only: bool = False,
             grad_scale: float = 1.0, allreduce=None):
        """forward + backward + [allreduce(flat gradient)] + Adam.  Returns the two loss tensors (device)."""
        closs, mloss = self.forward(src, dst, neg, ts, eids, cg, contrast_only=contrast_only)
        self.backward(1.0, 0.0 if contrast_only else mutual_coef)
        if allreduce is not None:
            allreduce(self.fp.grad_all)
        self.fp.adam(self.lr, grad_scale=grad_scale)
        return closs, mloss
