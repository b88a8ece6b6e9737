"""Tensor-level wrappers of the C-ABI kernels (one function per entry point).

Every function takes CUDA tensors, allocates its outputs with torch (device memory is the
only thing torch does here), launches on the current stream and never synchronises.
"""
import ctypes
import functools
import os
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import call, check_cuda, ptr

i64, i32, f32, f64, u8 = torch.int64, torch.int32, torch.float32, torch.float64, torch.uint8


def _empty(shape, dtype, like: Tensor) -> Tensor:
    return torch.empty(shape, dtype=dtype, device=like.device)


# ------------------------------------------------------------------------------------------
# graph
# ------------------------------------------------------------------------------------------
class DeviceCSR:
    """Per-node time-sorted adjacency in HBM: indptr int64 [N+1]; nbr/eid int32, ts float64,
    flag uint8, each [2E]."""

    def __init__(self, indptr, nbr, eid, ts, flag):
        self.indptr, self.nbr, self.eid, self.ts, self.flag = indptr, nbr, eid, ts, flag
        self.n_nodes = indptr.numel() - 1

    @property
    def device(self):
        return self.indptr.device


def csr_build(src: Tensor, dst: Tensor, ts: Tensor, eids: Tensor, n_nodes: int) -> DeviceCSR:
    """a1: device CSR from a time-ordered stream (int64 ids, float64 times)."""
    check_cuda(src, dst, ts, eids)
    assert src.dtype == i64 and dst.dtype == i64 and eids.dtype == i64 and ts.dtype == f64
    E = src.numel()
    indptr = _empty(n_nodes + 1, i64, src)
    nbr = _empty(2 * E, i32, src)
    eid = _empty(2 * E, i32, src)
    ats = _empty(2 * E, f64, src)
    flag = _empty(2 * E, u8, src)
    work = _empty(_lib.load().tiger_csr_build_work_bytes(E, n_nodes), u8, src)
    call('tiger_csr_build', ptr(src), ptr(dst), ptr(ts), ptr(eids), E, n_nodes, ptr(indptr), ptr(nbr), ptr(eid),
         ptr(ats), ptr(flag), ptr(work))
    return DeviceCSR(indptr, nbr, eid, ats, flag)


FIND_CHUNK_NEIGHBORS, FIND_CHUNK_HISTORY = 1, 2     # chunk modes of tiger_find_recent_ex (include/tiger_b200.h)


def find_recent(csr: DeviceCSR, q_nids: Tensor, q_ts: Tensor, k: int, *, ts_period: int = 0,
                want_dirs: bool = True, ts32_out: Optional[Tensor] = None, bitmap: Optional[Tensor] = None,
                out: Optional[Tuple[Tensor, Tensor, Tensor, Optional[Tensor]]] = None,
                count: Optional[Tensor] = None, chunk_mode: int = 0, node_stride: int = 0):
    """a2: K most recent events strictly before q_ts, right-aligned and zero-padded.  chunk_mode (FIND_CHUNK_*):
    q_nids are virtual ids c * node_stride + u of a chunked engine (tiger_find_recent_ex)."""
    check_cuda(q_nids, q_ts)
    assert q_nids.dtype == i64 and q_ts.dtype == f64
    n = q_nids.numel()
    if out is None:
        o_n = _empty((n, k), i64, q_nids)
        o_e = _empty((n, k), i64, q_nids)
        o_t = _empty((n, k), f32, q_nids)
        o_d = _empty((n, k), i64, q_nids) if want_dirs else None
    else:
        o_n, o_e, o_t, o_d = out
    args = (ptr(csr.indptr), ptr(csr.nbr), ptr(csr.eid), ptr(csr.ts), ptr(csr.flag), ptr(q_nids), ptr(q_ts), n,
            ts_period or q_ts.numel(), k, ptr(o_n), ptr(o_e), ptr(o_t), ptr(o_d), ptr(ts32_out), ptr(bitmap),
            ptr(count))
    if chunk_mode:
        call('tiger_find_recent_ex', *args, node_stride, chunk_mode)
    else:
        call('tiger_find_recent', *args)
    return o_n, o_e, o_t, o_d


def find_second_hop(csr: DeviceCSR, nn1: Tensor, nt1: Tensor, k: int, *, ts64: Tensor, bitmap: Tensor,
                    out: Tuple[Tensor, Tensor, Tensor], node_stride: int = 0):
    """collate_memory_nodes' second neighbor call for n_layers = 2: the K most recent neighbors of each hop-1 neighbor
    nn1 [n, K] at its own float32 event time nt1, widened to float64 (an exact conversion) in `ts64` [n*K]; marks the
    same involved-node bitmap as the first hop.  node_stride > 0: nn1 holds virtual ids of a chunked engine."""
    ts64.copy_(nt1.view(-1))
    find_recent(csr, nn1.view(-1), ts64, k, want_dirs=False, bitmap=bitmap, out=(*out, None),
                chunk_mode=FIND_CHUNK_NEIGHBORS if node_stride else 0, node_stride=node_stride)


def hit_window(center: Tensor, neigh: Tensor) -> Tensor:
    check_cuda(center, neigh)
    n, k = neigh.shape
    hit = _empty((n, k), f32, neigh)
    call('tiger_hit_window', ptr(center), ptr(neigh), n, k, ptr(hit))
    return hit


def bitmap_words(n_nodes: int) -> int:
    return (n_nodes + 31) // 32


def mark_nodes(ids: Tensor, bitmap: Tensor, n_nodes: int):
    check_cuda(ids, bitmap)
    call('tiger_mark_nodes', ptr(ids), ids.numel(), ptr(bitmap), n_nodes)


def compact_involved(bitmap: Tensor, n_nodes: int, involved: Tensor, counts: Tensor, *,
                     has_msg: Optional[Tensor] = None, uptodate: Optional[Tensor] = None,
                     local_index: Optional[Tensor] = None, outdated: Optional[Tensor] = None,
                     gru_row: Optional[Tensor] = None, restart_nodes: Optional[Tensor] = None,
                     err_flags: Optional[Tensor] = None, read_only: bool = False, restart_base: int = 0):
    """read_only: uptodate / has_msg are only read, restart node r gets gru_row = restart_base + r (its restart
    surrogate's row, tiger_compact_involved_ex)."""
    call('tiger_compact_involved_ex', ptr(bitmap), n_nodes, ptr(has_msg), ptr(uptodate), ptr(involved),
         involved.numel(), ptr(local_index), ptr(outdated), ptr(gru_row), ptr(restart_nodes), ptr(counts),
         ptr(err_flags), int(read_only), restart_base)


# ------------------------------------------------------------------------------------------
# index utilities
# ------------------------------------------------------------------------------------------
class SelectScratch:
    """Per-node scratch of tiger_select_latest (zero on entry and on exit)."""

    def __init__(self, n_nodes: int, device):
        self.n_nodes = n_nodes
        self.slot_ts = torch.zeros(n_nodes, dtype=i64, device=device)
        self.slot_pos = torch.zeros(n_nodes, dtype=i32, device=device)
        self.bitmap = torch.zeros(bitmap_words(n_nodes), dtype=i32, device=device)


def select_latest(nids: Tensor, ts: Tensor, scratch: Optional[SelectScratch] = None, *,
                  want_unique: bool = True, winner: Optional[Tensor] = None, count: Optional[Tensor] = None,
                  want_count: bool = True):
    """a8: returns (winner uint8 [n], unique_ids, index, count) - unique_ids/index have n slots,
    the first `count` (device int32) are valid."""
    check_cuda(nids, ts)
    assert nids.dtype == i64 and ts.dtype in (f32, f64)
    n = nids.numel()
    if winner is None:
        winner = _empty(n, u8, nids)
    uniq = _empty(n, i64, nids) if want_unique else None
    index = _empty(n, i64, nids) if want_unique else None
    if count is None and (want_count or want_unique):
        count = _empty(1, i32, nids)
    if n > 2048 and scratch is None:
        raise _lib.TigerLibraryError('select_latest over more than 2048 positions needs a SelectScratch')
    call('tiger_select_latest', ptr(nids), ptr(ts), int(ts.dtype == f64), n, ts.numel(),
         scratch.n_nodes if scratch else 0, ptr(scratch.slot_ts) if scratch else None,
         ptr(scratch.slot_pos) if scratch else None, ptr(scratch.bitmap) if scratch else None,
         ptr(winner), ptr(uniq), ptr(index), ptr(count))
    return winner, uniq, index, count


def anonymized_reindex(hist_nids: Tensor, out: Optional[Tensor] = None, count: Optional[Tensor] = None) -> Tensor:
    check_cuda(hist_nids)
    n, length = hist_nids.shape
    if out is None:
        out = torch.empty_like(hist_nids)
    call('tiger_anonymized_reindex', ptr(hist_nids), n, length, ptr(out), ptr(count))
    return out


# ------------------------------------------------------------------------------------------
# memory / message store
# ------------------------------------------------------------------------------------------
def gather_rows(table: Tensor, ids: Tensor, ts_table: Optional[Tensor] = None):
    check_cuda(table, ids, ts_table)
    n = ids.numel()
    width = table.shape[1]
    out = _empty((n, width), f32, table)
    out_ts = _empty(n, f32, table) if ts_table is not None else None
    call('tiger_gather_rows', ptr(table), width, ptr(ids), n, ptr(out), ptr(ts_table), ptr(out_ts))
    return out, out_ts


def scatter_rows(table: Optional[Tensor], ids: Tensor, vals: Optional[Tensor], *, ts_table=None, ts=None,
                 active=None, check: bool = False, err_flags=None, count=None, width: Optional[int] = None):
    check_cuda(table, ids, vals, ts_table, ts, active, err_flags, count)
    w = width if width is not None else (table.shape[1] if table is not None else 0)
    call('tiger_scatter_rows', ptr(table), w, ptr(ids), ids.numel(), ptr(count), ptr(vals), ptr(ts_table), ptr(ts),
         ptr(active), int(check), ptr(err_flags))


def time_encode(ts: Tensor, w: Tensor, b: Tensor) -> Tensor:
    check_cuda(ts, w, b)
    dim = w.numel()
    out = _empty((*ts.shape, dim), f32, ts)
    call('tiger_time_encode', ptr(ts), ts.numel(), ptr(w), ptr(b), dim, ptr(out))
    return out


def store_messages(src, dst, eids, ts, winner, mem_vals, mem_ts, nfeats, efeats, d, de, time_w, time_b,
                   msg_vals, msg_ts, has_msg, err_flags=None):
    call('tiger_store_messages', ptr(src), ptr(dst), ptr(eids), ptr(ts), src.numel(), ptr(winner), ptr(mem_vals),
         ptr(mem_ts), ptr(nfeats), ptr(efeats), d, de, ptr(time_w), ptr(time_b), ptr(msg_vals), ptr(msg_ts),
         ptr(has_msg), ptr(err_flags))


def right_writeback(pos_ids, winner, gru_row, h_new, d, right_vals, right_ts, right_active, msg_ts, has_msg,
                    left_vals=None, hprev_left=None, hprev_right=None, err_flags=None):
    check_cuda(pos_ids, winner, gru_row, h_new, right_vals, right_ts, right_active, msg_ts, has_msg, left_vals,
               hprev_left, hprev_right, err_flags)
    call('tiger_right_writeback', ptr(pos_ids), pos_ids.numel(), ptr(winner), ptr(gru_row), ptr(h_new), d,
         ptr(right_vals), ptr(right_ts), ptr(right_active), ptr(msg_ts), ptr(has_msg), ptr(left_vals),
         ptr(hprev_left), ptr(hprev_right), ptr(err_flags))


def left_writeback(pos_ids, batch, winner, h_left, d, ts, left_vals, left_ts, left_active, err_flags=None):
    check_cuda(pos_ids, winner, h_left, ts, left_vals, left_ts, left_active, err_flags)
    call('tiger_left_writeback', ptr(pos_ids), pos_ids.numel(), batch, ptr(winner), ptr(h_left), d, ptr(ts),
         ptr(left_vals), ptr(left_ts), ptr(left_active), ptr(err_flags))


# ------------------------------------------------------------------------------------------
# parameter packing
# ------------------------------------------------------------------------------------------
class GruPack:
    """nn.GRUCell parameters as the kernel reads them: the gate weights pre-split into tf32 head / tail
    planes in the stage layout of tiger_gru_update (tiger_gru_pack), biases as stored."""

    def __init__(self, weight_ih: Tensor, weight_hh: Tensor, bias_ih: Tensor, bias_hh: Tensor):
        self.d = weight_hh.shape[1]
        self.m_dim = weight_ih.shape[1]
        nbytes = _lib.load().tiger_gru_pack_bytes(self.m_dim, self.d)
        self.wpack = torch.empty(nbytes // 4, dtype=f32, device=weight_ih.device)
        self.refresh(weight_ih, weight_hh, bias_ih, bias_hh)

    def refresh(self, weight_ih, weight_hh, bias_ih, bias_hh):
        w_ih = weight_ih.detach().to(f32).contiguous()
        w_hh = weight_hh.detach().to(f32).contiguous()
        check_cuda(w_ih, w_hh)
        call('tiger_gru_pack', ptr(w_ih), ptr(w_hh), self.m_dim, self.d, ptr(self.wpack))
        self.b_ih = bias_ih.detach().to(f32).contiguous()
        self.b_hh = bias_hh.detach().to(f32).contiguous()


def gru_update(pack: GruPack, *, node_ids: Optional[Tensor], x_table: Tensor, h_table: Tensor, n_rows: int,
               out: Optional[Tensor] = None, count: Optional[Tensor] = None, msg_ts: Optional[Tensor] = None,
               check_mem_ts: Optional[Tensor] = None, check_equal: bool = False,
               err_flags: Optional[Tensor] = None, x_by_row: bool = False) -> Tensor:
    """a6+a13: h_new[r] = GRUCell(x_table[ids[r]], h_table[ids[r]]) (ids None => dense rows).  x_by_row: x is
    x_table[r] (tiger_gru_update_rows), h and the checks still read node ids[r]."""
    check_cuda(node_ids, x_table, h_table)
    if out is None:
        out = _empty((n_rows, pack.d), f32, x_table)
    call('tiger_gru_update_rows' if x_by_row else 'tiger_gru_update', ptr(node_ids), ptr(count), n_rows,
         ptr(x_table), x_table.stride(0), ptr(h_table), h_table.stride(0), pack.m_dim, pack.d, ptr(pack.wpack),
         ptr(pack.b_ih), ptr(pack.b_hh), ptr(out), ptr(msg_ts), ptr(check_mem_ts), int(check_equal), ptr(err_flags))
    return out


def fold_linear(w: Tensor, b: Tensor, w_t: Tensor, b_t: Tensor) -> Tuple[Tensor, Tensor]:
    """A layer (w [n, m], b [n]) that consumes the output of a linear map (w_t [m, k], b_t [m]) as one layer on the
    map's input: (w w_t, b + w b_t), accumulated in float64 and rounded once to float32."""
    w64 = w.detach().to(f64)
    return ((w64 @ w_t.detach().to(f64)).to(f32).contiguous(),
            (b.detach().to(f64) + w64 @ b_t.detach().to(f64)).to(f32).contiguous())


class MergePack:
    """MergeLayer(m, d, d, d) of MergeUpdater as tiger_merge_update reads it: fc1 [d, m + d] pre-split into the stage
    layout of the GRU kernel (tiger_merge_pack), fc2 as a WeightPack for the count-bounded second product."""

    def __init__(self, fc1_w: Tensor, fc1_b: Tensor, fc2_w: Tensor, fc2_b: Tensor, m_rows_hint: int = 600):
        self.d = fc2_w.shape[0]
        self.m_dim = fc1_w.shape[1] - self.d
        nbytes = _lib.load().tiger_gru_pack_bytes(self.m_dim, self.d)
        self.wpack = torch.empty(nbytes // 4, dtype=f32, device=fc1_w.device)
        self.fc2 = WeightPack(fc2_w.detach().to(f32).contiguous(), m_rows_hint=m_rows_hint)
        self.refresh(fc1_w, fc1_b, fc2_w, fc2_b)

    def refresh(self, fc1_w, fc1_b, fc2_w, fc2_b):
        w1 = fc1_w.detach().to(f32).contiguous()
        check_cuda(w1)
        assert w1.shape == (self.d, self.m_dim + self.d)
        call('tiger_merge_pack', ptr(w1), self.m_dim, self.d, ptr(self.wpack))
        self.fc2.refresh(fc2_w.detach().to(f32).contiguous())
        self.b1 = fc1_b.detach().to(f32).contiguous()
        self.b2 = fc2_b.detach().to(f32).contiguous()


def merge_update(pack: MergePack, *, node_ids: Tensor, x_table: Tensor, h_table: Tensor, n_rows: int, mid: Tensor,
                 out: Tensor, x_by_row: bool = False, count: Optional[Tensor] = None, msg_ts: Optional[Tensor] = None,
                 check_mem_ts: Optional[Tensor] = None, check_equal: bool = False,
                 err_flags: Optional[Tensor] = None) -> Tensor:
    """MergeUpdater: out[r] = fc2(relu(fc1 [x ; h] + b1)) + b2 with x = x_table[ids[r]] (x_table[r] with x_by_row),
    h = h_table[ids[r]]; mid [>= n_rows, d] holds the first layer."""
    check_cuda(node_ids, x_table, h_table, mid, out)
    call('tiger_merge_update', ptr(node_ids), ptr(count), n_rows, ptr(x_table), x_table.stride(0), int(x_by_row),
         ptr(h_table), h_table.stride(0), pack.m_dim, pack.d, ptr(pack.wpack), ptr(pack.b1), ptr(mid), ptr(msg_ts),
         ptr(check_mem_ts), int(check_equal), ptr(err_flags))
    return sgemm_nt_packed(mid, pack.fc2, pack.b2, out, m_rows=n_rows, count=count)


def gather_linear(ids: Tensor, table: Tensor, pack: 'WeightPack', bias: Optional[Tensor], out: Tensor, *,
                  relu: bool = False, count: Optional[Tensor] = None) -> Tensor:
    """out[m] = act(W table[ids[m]] + bias) for m < count (the plain-row case of tiger_sgemm_nt_packed_gather)."""
    check_cuda(ids, table, bias, out)
    assert ids.dtype == i64 and table.shape[1] == pack.k
    call('tiger_sgemm_nt_packed_gather', ptr(ids), None, 0, ptr(table), None, table.stride(0), None, ptr(pack.data),
         pack.bn, ptr(bias), ptr(out), out.stride(0), ids.numel(), ptr(count), 1, pack.n, pack.k, 1.0, int(relu))
    return out


class MemoryUpdater:
    """Steps 1-2 of the reference (tiger.py:206-221) for every message transform / memory updater pair the reference
    offers (--tsfm_fn id|linear|mlp, --upd_fn gru|merge): h_new[r] = upd(tsfm(msg_vals[ids[r]]), h[ids[r]]) for the
    outdated rows r < count, with the message invariants checked.

      id / linear + gru    one tiger_gru_update; a linear transform is folded into weight_ih / bias_ih
      mlp + gru            the hidden rows relu(W_1 msg + b_1) by row position, then tiger_gru_update_rows on the
                           fold of W_2 into weight_ih / bias_ih
      * + merge            as above with tiger_merge_update (folds into fc1's message columns) + the fc2 product

    Folds are computed in float64 whenever `refresh` runs; the device buffers keep their addresses (captured graphs
    stay valid)."""

    TSFM, UPD = ('id', 'linear', 'mlp'), ('gru', 'merge')

    def __init__(self, tsfm: str, upd: str, d: int, m_dim: int, cap: int, device):
        if tsfm not in self.TSFM:
            raise NotImplementedError(f'msg_tsfm_type={tsfm!r}: expected one of {self.TSFM}')
        if upd not in self.UPD:
            raise NotImplementedError(f'mem_update_type={upd!r}: expected one of {self.UPD}')
        self.tsfm, self.upd, self.d, self.m_dim, self.device = tsfm, upd, d, m_dim, device
        self.cap = 0
        self.gru = self.merge = self.w1 = self.b1 = None
        self.hid = self.mid = None
        self.reserve(cap)

    def scratch(self, cap: int):
        """(hid, mid) for `cap` outdated rows: hidden rows of the MLP, first layer of the merge (None when unused)."""
        z = lambda w: torch.zeros(cap, w, dtype=f32, device=self.device)
        return (z(self.m_dim // 2) if self.tsfm == 'mlp' else None, z(self.d) if self.upd == 'merge' else None)

    def reserve(self, cap: int):
        """Own scratch for `cap` outdated rows."""
        if cap <= self.cap:
            return
        self.cap = cap
        self.hid, self.mid = self.scratch(cap)

    @property
    def launches(self) -> int:
        return 1 + (self.tsfm == 'mlp') + (self.upd == 'merge')

    def param_names(self):
        """The parameters this updater reads, under the reference's state_dict names."""
        t = {'id': (), 'linear': ('fn.1.weight', 'fn.1.bias'),
             'mlp': ('fn.1.weight', 'fn.1.bias', 'fn.4.weight', 'fn.4.bias')}[self.tsfm]
        u = (('cell.weight_ih', 'cell.weight_hh', 'cell.bias_ih', 'cell.bias_hh') if self.upd == 'gru' else
             ('fn.fc1.weight', 'fn.fc1.bias', 'fn.fc2.weight', 'fn.fc2.bias'))
        return ['msg_transform_fn.' + n for n in t] + ['right_mem_updater.' + n for n in u]

    def refresh(self, get):
        """Re-pack from get(name) -> float32 device tensor (names of param_names())."""
        p = {n: get(n) for n in self.param_names()}
        t, u = 'msg_transform_fn.fn.', 'right_mem_updater.'
        fold = None                                      # the linear map in front of the updater's message input
        if self.tsfm == 'linear':
            fold = (p[t + '1.weight'], p[t + '1.bias'])
        elif self.tsfm == 'mlp':
            fold = (p[t + '4.weight'], p[t + '4.bias'])
            w1 = p[t + '1.weight'].detach().to(f32).contiguous()
            if self.w1 is None:
                self.w1 = WeightPack(w1, m_rows_hint=self.cap)
            else:
                self.w1.refresh(w1)
            self.b1 = p[t + '1.bias'].detach().to(f32).contiguous()
        if self.upd == 'gru':
            w_ih, b_ih = p[u + 'cell.weight_ih'], p[u + 'cell.bias_ih']
            if fold is not None:
                w_ih, b_ih = fold_linear(w_ih, b_ih, *fold)
            args = (w_ih, p[u + 'cell.weight_hh'], b_ih, p[u + 'cell.bias_hh'])
            if self.gru is None:
                self.gru = GruPack(*args)
            else:
                self.gru.refresh(*args)
        else:
            fc1, b1 = p[u + 'fn.fc1.weight'], p[u + 'fn.fc1.bias']
            if fold is not None:
                wx, b1 = fold_linear(fc1[:, :self.m_dim], b1, *fold)
                fc1 = torch.cat([wx, fc1[:, self.m_dim:].detach().to(f32)], 1)
            args = (fc1, b1, p[u + 'fn.fc2.weight'], p[u + 'fn.fc2.bias'])
            if self.merge is None:
                self.merge = MergePack(*args, m_rows_hint=self.cap)
            else:
                self.merge.refresh(*args)

    def launch(self, *, node_ids: Tensor, x_table: Tensor, h_table: Tensor, n_rows: int, out: Tensor,
               count: Optional[Tensor], msg_ts: Tensor, check_mem_ts: Optional[Tensor], check_equal: bool,
               err_flags: Optional[Tensor], scratch=None):
        """scratch: (hid, mid) of another caller (`scratch(cap)`), which then runs on these packs beside the owner."""
        hid, mid = (self.hid, self.mid) if scratch is None else scratch
        assert n_rows <= self.cap if scratch is None else all(t is None or n_rows <= t.shape[0] for t in scratch)
        x_by_row = self.tsfm == 'mlp'
        if x_by_row:
            x_table = gather_linear(node_ids[:n_rows], x_table, self.w1, self.b1, hid[:n_rows], relu=True,
                                    count=count)
        kw = dict(node_ids=node_ids, x_table=x_table, h_table=h_table, n_rows=n_rows, out=out, count=count,
                  msg_ts=msg_ts, check_mem_ts=check_mem_ts, check_equal=check_equal, err_flags=err_flags,
                  x_by_row=x_by_row)
        if self.upd == 'gru':
            return gru_update(self.gru, **kw)
        return merge_update(self.merge, mid=mid, **kw)


@functools.lru_cache(maxsize=None)
def _attention_max(which: str) -> int:
    """Largest K ('k', one head) or head count ('h', one slot) the attention kernels take, read off
    tiger_temporal_attention_work_bytes at a width where the shared-memory footprint is far from its limit."""
    fits = lambda v: _lib.load().tiger_temporal_attention_work_bytes(0, v if which == 'k' else 1, 4, 4,
                                                                       v if which == 'h' else 1) >= 0
    v = 1
    while fits(v + 1):
        v += 1
    return v


@functools.lru_cache(maxsize=None)
def attention_limit_error(d: int, de: int, k: int, n_head: int) -> Optional[str]:
    """Why the attention kernels (temporal_attention, temporal_attention_dense) cannot run a layer of node width d,
    edge width de, k neighbor slots and n_head heads, or None when they can.  The limits are the kernels' own
    (tiger_temporal_attention_work_bytes); the reference has none, so callers run such layers through torch."""
    if _lib.load().tiger_temporal_attention_work_bytes(0, k, d, de, n_head) >= 0:
        return None
    if min(d, de, k, n_head) <= 0:
        return f'invalid attention dimensions d={d} de={de} n_neighbors={k} n_head={n_head}'
    max_k, max_h = _attention_max('k'), _attention_max('h')
    if k > max_k:
        return f'the attention kernel takes at most {max_k} neighbors per query; this layer has n_neighbors={k}'
    if n_head > max_h:
        return f'the attention kernel takes at most {max_h} heads; this layer has n_head={n_head}'
    return (f'the attention kernel stages the {k} key rows of a query in shared memory, which does not hold them at '
            f'd={d}, de={de}, n_neighbors={k}, n_head={n_head} (shared-memory footprint over its limit)')


class AttnParamsC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in
                ('wq', 'wk', 'wv', 'wo', 'fc1', 'fc2', 'in_bias', 'out_bias', 'fc1_b', 'fc2_b', 'time_w', 'time_b',
                 'folded', 'score_folded', 'pq_out', 'left_wb')]


class LeftWritebackFusedC(ctypes.Structure):
    """tiger_left_writeback_fused (include/tiger_b200.h)."""
    _fields_ = [('pos_ids', ctypes.c_void_p), ('winner', ctypes.c_void_p), ('n_pos', ctypes.c_int64),
                ('ts', ctypes.c_void_p), ('batch', ctypes.c_int64), ('left_vals', ctypes.c_void_p),
                ('left_ts', ctypes.c_void_p), ('left_active', ctypes.c_void_p), ('err_flags', ctypes.c_void_p),
                ('ready_event', ctypes.c_void_p)]


_ATTN_WEIGHT_FIELDS = tuple(n for n, _ in AttnParamsC._fields_[:13])    # wq .. folded


class AttnPack:
    """TemporalAttention parameters for the kernels: the reference's tensors as stored plus the folded
    weights (tiger_attn_fold: Wqk, bqk, W2f), and a workspace that grows on demand.  A multi-layer embedding
    keeps one pack per layer (temporal_embedding_fn.fns.i); the score fold and the fused left write-back attach
    together, only to the pack of the batch-node layer, whose result they read, and only for the gather form
    (temporal_attention): the kernel refuses a call with one of them alone or with the dense form."""

    def __init__(self, d: int, de: int, device, n_head: int = 2):
        self.d, self.de, self.n_head = d, de, n_head
        self.E, self.C = 2 * d, 2 * d + de
        nbytes = _lib.load().tiger_attn_fold_bytes(d, de, n_head)
        if nbytes <= 0:
            raise _lib.TigerLibraryError(f'invalid attention dims d={d} de={de} heads={n_head}')
        self.folded = torch.zeros(nbytes // 4, dtype=f32, device=device)
        self.struct = AttnParamsC()
        self._keep = None
        self._work = None
        self._work_key = None
        self._base = None

    def share(self) -> 'AttnPack':
        """A pack on this pack's weights and folds (no copy) with its own score-fold attachment and workspace: a
        second caller of the same layer (a candidate query beside the engine's step).  It re-reads the weight pointers
        of this pack at every launch, so refresh() here reaches it."""
        v = AttnPack.__new__(AttnPack)
        v.d, v.de, v.n_head, v.E, v.C = self.d, self.de, self.n_head, self.E, self.C
        v.folded, v.struct, v._keep, v._work, v._work_key, v._base = self.folded, AttnParamsC(), None, None, None, self
        return v

    def refresh(self, q_w, k_w, v_w, in_bias, out_w, out_b, fc1_w, fc1_b, fc2_w, fc2_b, time_w, time_b):
        det = lambda t: t.detach().to(f32).contiguous()
        keep = [det(t) for t in (q_w, k_w, v_w, in_bias, out_w, out_b, fc1_w, fc1_b, fc2_w, fc2_b, time_w, time_b)]
        check_cuda(*keep)
        self._keep = keep
        s = self.struct
        for name, t in zip(('wq', 'wk', 'wv', 'in_bias', 'wo', 'out_bias', 'fc1', 'fc1_b', 'fc2', 'fc2_b', 'time_w',
                            'time_b'), keep):
            setattr(s, name, t.data_ptr())
        s.folded = self.folded.data_ptr()
        call('tiger_attn_fold', self.byref(), self.d, self.de, self.n_head)

    def byref(self):
        if self._base is not None:
            for name in _ATTN_WEIGHT_FIELDS:
                setattr(self.struct, name, getattr(self._base.struct, name))
        return ctypes.addressof(self.struct)

    def attach_score_fold(self, fold: Optional['ScoreFold'], pq_out: Optional[Tensor]):
        """With a ScoreFold (and the left write-back) attached the last attention GEMM also emits the link scorer's
        first layer (pq_out [n_query, 2d]); detach with (None, None)."""
        self._score_fold, self._pq_out = fold, pq_out
        self.struct.score_folded = fold.blob.data_ptr() if fold is not None else None
        self.struct.pq_out = pq_out.data_ptr() if pq_out is not None else None

    def attach_left_writeback(self, pos_ids: Optional[Tensor], winner: Optional[Tensor] = None, ts: Optional[Tensor] = None,
                              left_vals: Optional[Tensor] = None, left_ts: Optional[Tensor] = None,
                              left_active: Optional[Tensor] = None, err_flags: Optional[Tensor] = None,
                              ready_event: Optional[torch.cuda.Event] = None):
        """update_left_memory (tiger.py:408-420) fused into the last attention product: result rows p < len(pos_ids)
        with winner[p] are also stored into left_vals[pos_ids[p]] (+ clock, activity flag).  `ready_event` must
        cover the producer of `winner` and the readers of the old left-memory rows.  None detaches."""
        if pos_ids is None:
            self._left_wb = None
            self.struct.left_wb = None
            return
        check_cuda(pos_ids, winner, ts, left_vals, left_ts, left_active, err_flags)
        w = LeftWritebackFusedC()
        w.pos_ids, w.winner, w.n_pos = pos_ids.data_ptr(), winner.data_ptr(), pos_ids.numel()
        w.ts, w.batch = ts.data_ptr(), ts.numel()
        w.left_vals, w.left_ts = left_vals.data_ptr(), left_ts.data_ptr()
        w.left_active = left_active.data_ptr() if left_active is not None else None
        w.err_flags = err_flags.data_ptr() if err_flags is not None else None
        w.ready_event = ready_event.cuda_event if ready_event is not None else None
        self._left_wb = (w, pos_ids, winner, ts, left_vals, left_ts, left_active, err_flags, ready_event)
        self.struct.left_wb = ctypes.addressof(w)

    def work(self, n_query: int, k: int) -> Tensor:
        key = (n_query, k)
        if self._work is None or self._work_key is None or self._work_key[0] < n_query or self._work_key[1] != k:
            nbytes = _lib.load().tiger_temporal_attention_work_bytes(n_query, k, self.d, self.de, self.n_head)
            if nbytes < 0:
                raise _lib.TigerLibraryError('temporal attention: invalid argument ('
                                             + (attention_limit_error(self.d, self.de, k, self.n_head)
                                                or f'n_query={n_query}') + ')')
            self._work = torch.empty(nbytes, dtype=u8, device=self.folded.device)
            self._work_key = key
        return self._work


def temporal_attention(pack: AttnPack, n_head: int, center_nids: Tensor, q_ts: Tensor, neigh_nids: Tensor,
                       neigh_eids: Tensor, neigh_ts: Tensor, *, rows_a: Optional[Tensor], rows_b: Tensor,
                       sel: Tensor, nfeats: Optional[Tensor], efeats: Optional[Tensor],
                       out: Optional[Tensor] = None, key_rows: Optional[Tensor] = None, ts_group: int = 1,
                       read_only: bool = False) -> Tensor:
    """a15+a16 (gather form).  Query q uses q_ts[(q // ts_group) % len(q_ts)] (ts.repeat semantics; ts_group = K
    gives repeat_interleave(ts.repeat(3), K), the depth-1 queries of n_layers = 2).  key_rows [n * K, d]: slot
    (q, j) takes the lower layer's output row q * K + j as its node representation, without node features.
    read_only: the pack has a score fold attached and no left write-back (tiger_temporal_attention_query)."""
    check_cuda(center_nids, q_ts, neigh_nids, neigh_eids, neigh_ts, rows_a, rows_b, sel, nfeats, efeats, key_rows)
    n, k = neigh_nids.shape
    if out is None:
        out = _empty((n, pack.d), f32, rows_b)
    assert sel.dtype in (i32, i64) and n_head == pack.n_head
    assert key_rows is None or (key_rows.dtype == f32 and key_rows.numel() >= n * k * pack.d)
    entry = 'tiger_temporal_attention_query' if read_only else 'tiger_temporal_attention_ex'
    call(entry, ptr(center_nids), ptr(q_ts), n, q_ts.numel(), ts_group, ptr(neigh_nids),
         ptr(neigh_eids), ptr(neigh_ts), k, ptr(rows_a), ptr(rows_b), ptr(key_rows), ptr(sel), int(sel.dtype == i64),
         ptr(nfeats), ptr(efeats), pack.d, pack.de, n_head, pack.byref(), ptr(out), ptr(pack.work(n, k)))
    return out


def temporal_attention_dense(pack: AttnPack, n_head: int, qx, qt, kx, ky, kt, padding_mask) -> Tensor:
    check_cuda(qx, qt, kx, ky, kt, padding_mask)
    n, k = kx.shape[0], kx.shape[1]
    out = _empty((n, pack.d), f32, qx)
    mask = padding_mask.to(u8).contiguous()
    assert n_head == pack.n_head
    call('tiger_temporal_attention_dense', ptr(qx), ptr(qt), ptr(kx), ptr(ky), ptr(kt), ptr(mask), n, k, pack.d,
         pack.de, n_head, pack.byref(), ptr(out), ptr(pack.work(n, k)))
    return out


HIT_TYPES = ('none', 'bin', 'vec', 'count')      # --hit_type, index = TIGER_HIT_* (include/tiger_b200.h)


class ScoreFold:
    """Link scorer folded into the attention's last GEMM (tiger_score_fold_hit): refresh whenever score_fn,
    the embedding module's merger.fc2 or the hit embedding change.  'bin' also serves 'none' (hit_emb None);
    'vec' and 'count' fold for k = n_neighbors slots (score_fn.fc1 [d, 2(d+k)], hit_embedding [k+1, d])."""

    def __init__(self, d: int, device, hit_type: str = 'bin', k: int = 0):
        if hit_type not in HIT_TYPES:
            raise NotImplementedError(f'hit_type={hit_type}')
        self.d, self.hit_type = d, hit_type
        self.k = k if hit_type in ('vec', 'count') else 0
        lib = _lib.load()
        code = HIT_TYPES.index(hit_type)
        nbytes = lib.tiger_score_fold_hit_bytes(d, code, self.k)
        if nbytes <= 0:
            raise _lib.TigerLibraryError(f'invalid score fold d={d} hit_type={hit_type} k={k}')
        self.blob = torch.zeros(nbytes // 4, dtype=f32, device=device)
        self.cab = self.blob[lib.tiger_score_fold_hit_offset(d, code, self.k):]    # the table the scorer reads
        self.done = torch.zeros(1, dtype=i32, device=device)

    def code(self, with_hits: bool) -> int:
        """TIGER_HIT_* of a fold / score call; for 'bin' / 'none' whether hit data is given decides."""
        if self.hit_type in ('vec', 'count'):
            return HIT_TYPES.index(self.hit_type)
        return HIT_TYPES.index('bin' if with_hits else 'none')

    def refresh(self, fc1_w, fc1_b, fc2_w, fc2_b, merger_fc2_w, merger_fc2_b, hit_emb: Optional[Tensor]):
        det = lambda t: None if t is None else t.detach().to(f32).contiguous()
        self._keep = [det(t) for t in (fc1_w, fc1_b, merger_fc2_w, merger_fc2_b, hit_emb)]
        check_cuda(*self._keep)
        call('tiger_score_fold_hit', *(ptr(t) for t in self._keep), self.d, self.code(hit_emb is not None), self.k,
             ptr(self.blob))
        self.fc2_w = fc2_w.detach().to(f32).reshape(-1).contiguous()
        self.fc2_b = fc2_b.detach().to(f32).contiguous()


def link_score_folded(fold: ScoreFold, pq: Tensor, src: Tensor, dst: Tensor, neg: Tensor,
                      neigh_nids: Optional[Tensor], scores: Optional[Tensor] = None, loss: Optional[Tensor] = None):
    """neigh_nids [3B, K]: the batch nodes' neighbor table (hit flags); None for hit_type 'none'."""
    B = src.numel()
    if scores is None:
        scores = _empty(2 * B, f32, pq)
    if loss is None:
        loss = _empty(1, f32, pq)
    k = neigh_nids.shape[1] if neigh_nids is not None else 0
    if fold.hit_type in ('vec', 'count') and k != fold.k:
        raise ValueError(f'hit_type {fold.hit_type}: the fold holds {fold.k} slots, the neighbor table has {k}')
    call('tiger_link_score_folded_hit', ptr(pq), B, fold.d, ptr(src), ptr(dst), ptr(neg), ptr(neigh_nids), k,
         fold.code(neigh_nids is not None), ptr(fold.cab), ptr(fold.fc2_w), ptr(fold.fc2_b), ptr(scores), ptr(loss),
         ptr(fold.done))
    return scores, loss


def link_score_cands(fold: ScoreFold, pq: Tensor, src: Tensor, pos: Tensor, negs: Tensor,
                     neigh_nids: Optional[Tensor], scores: Tensor, ranks: Optional[Tensor] = None,
                     loss: Optional[Tensor] = None):
    """The scorer over C = scores.numel() / Q candidate columns (tiger_link_score_cands): pq / neigh_nids hold the rows
    of [src | pos | negs], negs [(C-1) Q] candidate-major; scores [C Q] candidate-major, ranks [Q] of column 0."""
    Q = src.numel()
    C = scores.numel() // Q
    k = neigh_nids.shape[1] if neigh_nids is not None else 0
    if fold.hit_type in ('vec', 'count') and k != fold.k:
        raise ValueError(f'hit_type {fold.hit_type}: the fold holds {fold.k} slots, the neighbor table has {k}')
    call('tiger_link_score_cands', ptr(pq), Q, C, fold.d, ptr(src), ptr(pos), ptr(negs), ptr(neigh_nids), k,
         fold.code(neigh_nids is not None), ptr(fold.cab), ptr(fold.fc2_w), ptr(fold.fc2_b), ptr(scores), ptr(ranks),
         ptr(loss), ptr(fold.done) if loss is not None else None)
    return scores, ranks


def static_restart_rows(nids: Tensor, n: int, right_emb: Tensor, d: int, out_rows: Tensor, *, count=None):
    """out_rows[i] = right_emb[nids[i]] for i < min(*count, n): the right-memory rows a static restart writes."""
    check_cuda(nids, right_emb, out_rows, count)
    call('tiger_static_restart_rows', ptr(nids), ptr(count), n, ptr(right_emb), d, ptr(out_rows))


def static_restart(nids: Tensor, n: int, csr: DeviceCSR, left_emb: Tensor, right_emb: Tensor, d: int, *,
                   count=None, batch_ts=None, q_ts=None, left_vals=None, left_ts=None, left_active=None,
                   right_vals=None, right_ts=None, right_active=None, has_msg=None, out_prev_ts=None,
                   node_stride: int = 0, chunk_ts: Optional[Tensor] = None):
    """node_stride > 0: nids are virtual ids of a chunked engine, cut at chunk_ts [M] float64
    (tiger_static_restart_ex)."""
    args = (ptr(nids), ptr(count), n, ptr(batch_ts), batch_ts.numel() if batch_ts is not None else 0, ptr(q_ts),
            ptr(csr.indptr), ptr(csr.ts), ptr(left_emb), ptr(right_emb), d, ptr(left_vals), ptr(left_ts),
            ptr(left_active), ptr(right_vals), ptr(right_ts), ptr(right_active), ptr(has_msg), ptr(out_prev_ts))
    if node_stride:
        call('tiger_static_restart_ex', *args, node_stride, ptr(chunk_ts))
    else:
        call('tiger_static_restart', *args)


# ------------------------------------------------------------------------------------------
# seq restarter (a21, a24)
# ------------------------------------------------------------------------------------------
def sgemm_nt(a: Tensor, w: Tensor, bias: Optional[Tensor], out: Tensor, *, m_rows: Optional[int] = None,
             k_dim: Optional[int] = None, relu: bool = False, count: Optional[Tensor] = None,
             rows_per_count: int = 1) -> Tensor:
    """out[m, n] = act(a[m, :k] @ w[n, :k].T + bias[n]); a/w/out may be column slices of wider buffers.
    Tensor cores (tf32x3)."""
    check_cuda_strided(a, w, out)
    m = a.shape[0] if m_rows is None else m_rows
    k = a.shape[1] if k_dim is None else k_dim
    call('tiger_sgemm_nt', ptr(a), a.stride(0), ptr(w), w.stride(0), ptr(bias), ptr(out), out.stride(0), m,
         ptr(count), rows_per_count, w.shape[0], k, int(relu))
    return out


def wgrad_k_parts(k: int) -> int:
    """K split of a weight-gradient product with reduction length k: at most 256 reduction steps per CTA (the tensor
    core truncates when it adds into its fp32 accumulator, an error that grows with the accumulation length:
    DESIGN.md, Tensor cores)."""
    return max(1, min(128, (k + 255) // 256))


def sgemm_ex(a: Tensor, w: Tensor, out: Tensor, *, m: int, n: int, k: int, trans_a: bool = False,
             trans_w: bool = False, bias: Optional[Tensor] = None, relu: bool = False, alpha: float = 1.0,
             accumulate: bool = False, k_parts: int = 1, m_count: Optional[Tensor] = None,
             k_count: Optional[Tensor] = None, rows_per_count: int = 1) -> Tensor:
    """out[m, n] (+)= act(alpha * (opA @ opW.T + bias)); opA = a[:m, :k] or a[:k, :m].T (trans_a), opW = w[:n, :k] or
    w[:k, :n].T (trans_w).  forward y = x W^T: (False, False); input gradient dx = dy W: (False, True); weight
    gradient dW = dy^T x: (True, True).  `accumulate` adds into `out` (atomic adds; K split over k_parts CTAs)."""
    check_cuda_strided(a, w, out)
    call('tiger_sgemm_ex', ptr(a), a.stride(0), int(trans_a), ptr(w), w.stride(0), int(trans_w), ptr(bias), ptr(out),
         out.stride(0), m, n, k, ptr(m_count), ptr(k_count), rows_per_count, float(alpha), int(relu), int(accumulate),
         k_parts)
    return out


class PPScratch:
    """Two growing scratch buffers for the packed operands of sgemm_big (stream-ordered reuse: a product is always
    launched right behind its two packs on the same stream)."""

    def __init__(self):
        self.bufs = [None, None]

    def get(self, which: int, nbytes: int, device) -> Tensor:
        b = self.bufs[which]
        if b is None or b.numel() * 4 < nbytes or b.device != device:
            b = self.bufs[which] = torch.empty((nbytes + 3) // 4, dtype=f32, device=device)
        return b


_pp_scratch = PPScratch()
BIG_GEMM_FLOPS = float(__import__('os').environ.get('TIGER_BIG_GEMM_FLOPS', 1.5e9))   # products above this many flops (by launch capacity) go through the pre-packed TMA-fed kernel


def sgemm_big(a: Tensor, w: Tensor, out: Tensor, *, m: int, n: int, k: int, trans_a: bool = False,
              trans_w: bool = False, bias: Optional[Tensor] = None, relu: bool = False, alpha: float = 1.0,
              accumulate: bool = False, k_parts: int = 1, m_count: Optional[Tensor] = None,
              k_count: Optional[Tensor] = None, rows_per_count: int = 1) -> Tensor:
    """sgemm_ex for large products: both operands are converted once (tiger_gemm_pp_pack: tf32 head / tail planes in
    stage-image order) and multiplied by the TMA-fed kernel (tiger_sgemm_pp).  Small products (where the two
    conversion passes would cost more than they save) fall through to sgemm_ex."""
    if 2.0 * m * n * k < BIG_GEMM_FLOPS:
        return sgemm_ex(a, w, out, m=m, n=n, k=k, trans_a=trans_a, trans_w=trans_w, bias=bias, relu=relu, alpha=alpha,
                        accumulate=accumulate, k_parts=k_parts, m_count=m_count, k_count=k_count,
                        rows_per_count=rows_per_count)
    check_cuda_strided(a, w, out)
    lib = _lib.load()
    ap = _pp_scratch.get(0, lib.tiger_gemm_pp_pack_bytes(m, k), a.device)
    wp = _pp_scratch.get(1, lib.tiger_gemm_pp_pack_bytes(n, k), a.device)
    call('tiger_gemm_pp_pack', ptr(a), a.stride(0), int(trans_a), m, k, ptr(m_count), ptr(k_count), rows_per_count, ptr(ap))
    call('tiger_gemm_pp_pack', ptr(w), w.stride(0), int(trans_w), n, k, None, ptr(k_count), rows_per_count, ptr(wp))
    call('tiger_sgemm_pp', ptr(ap), ptr(wp), ptr(bias), ptr(out), out.stride(0), m, n, k, ptr(m_count), ptr(k_count),
         rows_per_count, float(alpha), int(relu), int(accumulate), k_parts)
    return out


class WeightPack:
    """tf32 head / tail pack of a weight [N, K] for the tensor-core GEMM (tiger_gemm_pack_weight)."""

    def __init__(self, w: Tensor, bn: Optional[int] = None, m_rows_hint: int = 600):
        check_cuda_strided(w)
        self.n, self.k = w.shape
        lib = _lib.load()
        self.bn = bn if bn is not None else lib.tiger_gemm_pick_bn(m_rows_hint, self.n, 1)
        self.tiles = (self.n + self.bn - 1) // self.bn
        nbytes = lib.tiger_gemm_pack_bytes(self.tiles, self.k, self.bn)
        if self.bn <= 0 or nbytes <= 0:
            raise _lib.TigerLibraryError(f'cannot pack a [{self.n}, {self.k}] weight with bn={self.bn}')
        self.data = torch.empty(nbytes // 4, dtype=f32, device=w.device)
        self.refresh(w)

    def refresh(self, w: Tensor):
        w = w.detach()
        call('tiger_gemm_pack_weight', ptr(w), w.stride(0), None, self.n, self.k, self.bn, self.tiles, ptr(self.data))


def sgemm_nt_packed(a: Tensor, pack: WeightPack, bias: Optional[Tensor], out: Tensor, *, m_rows: Optional[int] = None,
                    relu: bool = False, alpha: float = 1.0, count: Optional[Tensor] = None,
                    rows_per_count: int = 1) -> Tensor:
    """out[m, n] = act(alpha * (a[m, :K] @ W.T + bias)) with W pre-packed (one TMA bulk copy per stage)."""
    check_cuda_strided(a, out)
    m = a.shape[0] if m_rows is None else m_rows
    call('tiger_sgemm_nt_packed', ptr(a), a.stride(0), ptr(pack.data), pack.bn, ptr(bias), ptr(out), out.stride(0), m,
         ptr(count), rows_per_count, pack.n, pack.k, float(alpha), int(relu))
    return out


def sgemm_nt_packed_splitk_fused(a: Tensor, pack: WeightPack, bias: Optional[Tensor], out: Tensor, k_parts: int, *,
                                 relu: bool = False, alpha: float = 1.0, m_rows: Optional[int] = None,
                                 count: Optional[Tensor] = None) -> Tensor:
    """As sgemm_nt_packed with K split over a thread-block cluster of k_parts CTAs per tile (DSMEM reduction)."""
    check_cuda_strided(a, out)
    call('tiger_sgemm_nt_packed_splitk_fused', ptr(a), a.stride(0), ptr(pack.data), pack.bn, ptr(bias), ptr(out),
         out.stride(0), k_parts, a.shape[0] if m_rows is None else m_rows, ptr(count), 1, pack.n, pack.k, float(alpha),
         int(relu))
    return out


def sgemm_nt_packed_gather(ids: Tensor, sel: Tensor, rows_a: Optional[Tensor], rows_b: Tensor, add_rows: Optional[Tensor],
                           pack: WeightPack, bias: Optional[Tensor], out: Tensor, *, relu: bool = False) -> Tensor:
    """out[m] = act(W @ x_m + bias) with x_m the latest representation of node ids[m]: rows_b[sel[ids[m]]] when
    that index is >= 0 (or rows_a is None), else rows_a[ids[m]]; plus add_rows[ids[m]] (node features).  The
    lookup of compute_embedding_with_computation_graph (temporal_agg_modules.py:210-235) inside the GEMM."""
    check_cuda(ids, sel, rows_a, rows_b, add_rows, bias, out)
    assert sel.dtype in (i32, i64) and ids.dtype == i64 and rows_b.stride(0) == pack.k
    call('tiger_sgemm_nt_packed_gather', ptr(ids), ptr(sel), int(sel.dtype == i64), ptr(rows_a), ptr(rows_b),
         rows_b.stride(0), ptr(add_rows), ptr(pack.data), pack.bn, ptr(bias), ptr(out), out.stride(0), ids.numel(),
         None, 1, pack.n, pack.k, 1.0, int(relu))
    return out


def check_cuda_strided(*tensors):
    for t in tensors:
        if not t.is_cuda or t.dtype != f32 or t.dim() != 2 or t.stride(1) != 1:
            raise _lib.TigerLibraryError('sgemm_nt needs 2-D float32 CUDA tensors with unit inner stride')


def min_time(ts: Tensor, out: Tensor, n_chunks: int = 1):
    """out[c] = min of chunk c of the chunk-major ts (float64 [n_chunks]); one chunk: tiger_min_time."""
    if n_chunks == 1:
        call('tiger_min_time', ptr(ts), ts.numel(), ptr(out))
    else:
        call('tiger_min_time_ex', ptr(ts), n_chunks, ts.numel() // n_chunks, ptr(out))


SEQ_MAX_HIST_LEN = 64     # the pooling kernel stages at most this many positions per node (SP_MAXL, csrc/train_seq.cu)


def seq_restarter_limit_error(d: int, de: int, hist_len: int, n_head: int) -> Optional[str]:
    """Why the seq restarter's kernels (SeqRestarterOp, the native training step) cannot run a restarter of node width
    d, edge width de, hist_len events and n_head heads, or None when they can.  The reference has no history limit,
    so callers run such a restarter through torch."""
    if min(d, de, hist_len, n_head) <= 0:
        return f'invalid seq restarter dimensions d={d} de={de} hist_len={hist_len} n_head={n_head}'
    if hist_len > SEQ_MAX_HIST_LEN:
        return (f'the seq restarter kernels take a history of at most {SEQ_MAX_HIST_LEN} events (the pooling kernel '
                f'stages them in shared memory); this restarter has hist_len={hist_len}')
    if (4 * d + de) % n_head != 0:
        return f'd_model = 4 d + de = {4 * d + de} is not a multiple of n_head={n_head}'
    return None


class SeqRestarterOp:
    """SeqRestarter.forward (reference restarters.py:51-114) on device buffers of capacity `cap` rows.

    Weights are used as stored (nn.Linear / in_proj layout), so there is nothing to re-pack when they
    change; `set_weights` only keeps contiguous fp32 views."""

    def __init__(self, d: int, de: int, hist_len: int, n_head: int, cap: int, device):
        limit = seq_restarter_limit_error(d, de, hist_len, n_head)
        if limit is not None:
            raise NotImplementedError(limit)
        self.d, self.de, self.L, self.H, self.cap = d, de, hist_len, n_head, cap
        self.dm = 4 * d + de
        z = lambda *shape, dt=f32: torch.zeros(*shape, dtype=dt, device=device)
        L, dm = hist_len, self.dm
        self.hist_nids, self.hist_eids, self.hist_dirs = z(cap, L, dt=i64), z(cap, L, dt=i64), z(cap, L, dt=i64)
        self.hist_ts = z(cap, L)
        self.anony = z(cap, L, dt=i64)
        self.x = z(cap * L, dm)
        self.qk = z(cap * L, 2 * dm)
        self.mask = z(cap, L, dt=u8)
        self.xbar = z(cap, n_head * dm)
        # attention probabilities of the pooling kernel (kept by the training step; written here as a by-product)
        self.P, self.pbar, self.psum = z(cap * n_head * L * L), z(cap * n_head * L), z(cap * n_head)
        self.att = z(cap, dm)
        self.o = z(cap, dm)
        self.h_left, self.hid, self.h_right = z(cap, d), z(cap, d), z(cap, d)
        self.prev_ts = z(cap)
        self.tmin = z(1, dt=f64)
        # [count if count <= TAIL_ROWS else 0, count if count > TAIL_ROWS else 0]: few restarted rows take the fused
        # matrix-vector tail (tiger_seq_tail), many rows the tensor-core products
        self.tail_rows = int(os.environ.get('TIGER_SEQ_TAIL_ROWS', '64')) if self.dm <= 1024 else 0
        self.cnt_gate = z(2, dt=torch.int32)
        self._aux = self._ev_a = self._ev_b = None

    def set_weights(self, W, prefix: str = 'restarter_fn.'):
        g = lambda k: W[prefix + k].detach().to(self.x.device, f32).contiguous()
        self.time_w, self.time_b = g('time_encoder.basis_freq'), g('time_encoder.phase')
        self.anony_emb = g('anony_emb.weight')
        self.in_w, self.in_b = g('mha_fn.in_proj_weight'), g('mha_fn.in_proj_bias')
        self.out_w, self.out_b = g('mha_fn.out_proj.weight'), g('mha_fn.out_proj.bias')
        self.fn_w, self.fn_b = g('out_fn.weight'), g('out_fn.bias')
        self.fc1_w, self.fc1_b = g('merger.fc1.weight'), g('merger.fc1.bias')
        self.fc2_w, self.fc2_b = g('merger.fc2.weight'), g('merger.fc2.bias')

    def share_weights(self, other: 'SeqRestarterOp'):
        """Read the weights of `other` (no copy): a second workspace for the same restarter."""
        for n in ('time_w', 'time_b', 'anony_emb', 'in_w', 'in_b', 'out_w', 'out_b', 'fn_w', 'fn_b', 'fc1_w', 'fc1_b',
                  'fc2_w', 'fc2_b'):
            setattr(self, n, getattr(other, n))

    def history(self, csr: DeviceCSR, nids: Tensor, q_ts: Tensor, n: int, *, ts_period: int = 0,
                count: Optional[Tensor] = None, node_stride: int = 0):
        """get_history (graph.py:150-155) + anonymized_reindex (utils.py:19-27) for n (or *count) nodes.
        node_stride > 0: nids are virtual ids of a chunked engine and q_ts holds one time per chunk."""
        find_recent(csr, nids[:n], q_ts, self.L, ts_period=ts_period, count=count,
                    out=(self.hist_nids[:n], self.hist_eids[:n], self.hist_ts[:n], self.hist_dirs[:n]),
                    chunk_mode=FIND_CHUNK_HISTORY if node_stride else 0, node_stride=node_stride)
        anonymized_reindex(self.hist_nids[:n], out=self.anony[:n], count=count)

    def forward(self, nids: Tensor, n: int, nfeats: Optional[Tensor], efeats: Optional[Tensor], *,
                count: Optional[Tensor] = None, hist=None):
        """Returns views (h_left [n,d], h_right [n,d], prev_ts [n]) of the workspace.  `hist` =
        (hist_nids, hist_eids, hist_ts, hist_dirs, anonymized_ids) overrides the internal buffers."""
        L, dm, d, H = self.L, self.dm, self.d, self.H
        hd = dm // H
        hn, he, ht, hdirs, an = hist if hist is not None else (self.hist_nids, self.hist_eids, self.hist_ts,
                                                               self.hist_dirs, self.anony)
        call('tiger_seq_tokens', ptr(nids), ptr(count), n, L, ptr(hn), ptr(he), ptr(ht), ptr(hdirs), ptr(an),
             ptr(nfeats), ptr(efeats), d, self.de, ptr(self.anony_emb), ptr(self.time_w), ptr(self.time_b),
             ptr(self.x), ptr(self.mask), ptr(self.prev_ts))
        sgemm_nt(self.x, self.in_w[:2 * dm], self.in_b[:2 * dm], self.qk, m_rows=n * L, count=count,
                 rows_per_count=L)
        # the register-tiled pooling kernel of the training step, with dropout 0
        call('tiger_train_seq_pool', ptr(self.qk), self.qk.stride(0), ptr(self.x), ptr(self.mask), ptr(count), n, L, dm,
             H, 0.0, 0, ptr(self.P), ptr(self.pbar), ptr(self.psum), ptr(self.xbar))
        if self.tail_rows > 0:
            # steady state restarts a few dozen rows per batch: five dependent layers as matrix-vector products (33 us
            # per tensor-core launch x 6 otherwise, profiles/r02_launches.md)
            tail = lambda cnt: call(
                'tiger_seq_tail', ptr(self.xbar), ptr(cnt), n, dm, H, d, ptr(self.in_w[2 * dm:]), ptr(self.in_b[2 * dm:]),
                ptr(self.out_w), ptr(self.out_b), ptr(self.fn_w), ptr(self.fn_b), ptr(self.fc1_w), self.fc1_w.stride(0),
                ptr(self.fc1_b), ptr(self.fc2_w), ptr(self.fc2_b), None, 0.0, 0, ptr(self.att), ptr(self.o), ptr(self.hid),
                ptr(self.h_left), ptr(self.h_right))
            if count is None:
                if n <= self.tail_rows:
                    tail(None)
                    return self.h_left[:n], self.h_right[:n], self.prev_ts[:n]
            else:
                # device-side row count: both routes are launched, the gate gives one of them zero rows.  Under graph
                # capture they are parallel branches (the idle route's launches cost ~2 us each in a serial chain)
                call('tiger_seq_gate_count', ptr(count), self.tail_rows, ptr(self.cnt_gate), ptr(self.cnt_gate[1:]))
                count = self.cnt_gate[1:]
                if os.environ.get('TIGER_SEQ_NO_GEMM') == '1':        # (debug aid: tail route only)
                    tail(self.cnt_gate)
                    return self.h_left[:n], self.h_right[:n], self.prev_ts[:n]
                cur = torch.cuda.current_stream()
                if torch.cuda.is_current_stream_capturing() and os.environ.get('TIGER_SEQ_TAIL_SERIAL') != '1':
                    if self._aux is None:
                        self._aux, self._ev_a, self._ev_b = torch.cuda.Stream(), torch.cuda.Event(), torch.cuda.Event()
                    self._ev_a.record(cur)
                    with torch.cuda.stream(self._aux):
                        self._aux.wait_event(self._ev_a)
                        tail(self.cnt_gate)
                        self._ev_b.record(self._aux)
                    self._products(n, count)
                    cur.wait_event(self._ev_b)
                    return self.h_left[:n], self.h_right[:n], self.prev_ts[:n]
                tail(self.cnt_gate)
        self._products(n, count)
        return self.h_left[:n], self.h_right[:n], self.prev_ts[:n]

    def _products(self, n: int, count: Optional[Tensor]):
        """The layers after the pooling kernel as tensor-core products."""
        dm, d, H = self.dm, self.d, self.H
        hd = dm // H
        for h in range(H):
            rows = slice(2 * dm + h * hd, 2 * dm + (h + 1) * hd)
            sgemm_nt(self.xbar[:, h * dm:(h + 1) * dm], self.in_w[rows], self.in_b[rows],
                     self.att[:, h * hd:(h + 1) * hd], m_rows=n, count=count)
        sgemm_nt(self.att, self.out_w, self.out_b, self.o, m_rows=n, relu=True, count=count)
        sgemm_nt(self.o, self.fn_w, self.fn_b, self.h_left, m_rows=n, count=count)
        sgemm_nt(self.h_left, self.fc1_w, self.fc1_b, self.hid, m_rows=n, k_dim=d, relu=True, count=count)
        sgemm_nt(self.hid, self.fc2_w, self.fc2_b, self.h_right, m_rows=n, count=count)

    LAUNCHES = 5 + 7 + 6   # min_time, find_recent, reindex, tokens, pool + 7 GEMMs + gate_count, 5 tail layers
    TAIL_LAUNCHES = 6      # gate_count + 5 tail layers: not launched when tail_rows == 0


def store_messages_dense(src, dst, eids, ts, winner, src_vals, dst_vals, src_prev_ts, dst_prev_ts, nfeats, efeats,
                         d, de, time_w, time_b, msg_vals, msg_ts, has_msg, err_flags=None):
    """MessageStoreNoGradLastOnly.store_events argument list (memory.py:77-81)."""
    call('tiger_store_messages_dense', ptr(src), ptr(dst), ptr(eids), ptr(ts), src.numel(), ptr(winner),
         ptr(src_vals), ptr(dst_vals), ptr(src_prev_ts), ptr(dst_prev_ts), ptr(nfeats), ptr(efeats), d, de,
         ptr(time_w), ptr(time_b), ptr(msg_vals), ptr(msg_ts), ptr(has_msg), ptr(err_flags))
