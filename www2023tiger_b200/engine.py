"""The per-batch temporal memory path as one fixed, sync-free launch sequence.

`TigerEngine` owns the device state of TIGE/TIGER (both memories, the last-message store, the
pending / up-to-date flags) and runs TIGE.contrast_learning (reference tiger/model/tiger.py:174-290)
as a fixed sequence of kernel launches (13 per batch) whose data-dependent sizes (involved U, outdated O, restarted R) stay on
the device.  `n_layers=2` (the reference's keyword default) adds the second neighbor hop to the finder and a depth-1
attention chain in front of the batch nodes' one.  `StreamRunner` adds the device neighbor finder in front, captures the sequence in a
CUDA graph and feeds it from pinned host buffers.

Launch sequence of one batch (B events, K neighbors):
  1 tiger_find_recent        3B queries -> neighbor tables, involved bitmap, float32 batch times
  2 tiger_compact_involved   involved / outdated / restart lists + gru_row map
  3 tiger_static_restart     (lazy-restart mode only) re-initialise not-yet-seen nodes
  4 tiger_gru_update         h(t'+) for the O outdated nodes      (steps 1-2 of the reference; the message transform
                             and memory updater variants are ops.MemoryUpdater's launches in this position)
  5 tiger_select_latest      argmax-by-timestamp winners of [src;dst]
  6 tiger_right_writeback    persist h(t'+) of outdated positives (step 4) [+ restarter targets]
  7 tiger_store_messages     build + store the new raw messages   (step 5)
  8 tiger_temporal_attention_ex  h(t-) for [src;dst;neg] (step 3); its last product also persists h(t-) of the
                             positives (step 6, tiger_left_writeback_fused) and writes the scorer's first layer pq
  9 tiger_link_score_folded  hit flags, scorer, BCE loss          (step 7)
Under graph capture 5-7 run on a side stream beside 8.

With n_layers = 2 (GraphEmbedding.compute_embedding_with_computation_graph, temporal_agg_modules.py:79-104):
  1  tiger_find_recent hop 1 as above, then the hop-1 times widened to float64 and tiger_find_recent hop 2: the K
     neighbors of each of the 3B*K hop-1 neighbors at that neighbor's own event time (the collator's two calls);
     both mark the involved bitmap, so U, O, R, the GRU and the lazy restart cover the 2-hop nodes
  8a tiger_temporal_attention_ex, fns.1, 3B*K depth-1 queries (center = hop-1 neighbor, time = its parent event's)
     over the hop-2 table -> emb1 [3B*K, d]
  8b tiger_temporal_attention_ex, fns.0, the 3B batch nodes over the hop-1 table, slot (q, j) keyed by emb1[q*K + j]

`CandidateQuery` (TigerEngine.candidate_query) scores one-vs-many candidate lists against the live state with the
same launches, reading the state tables and writing none of them.

With `n_chunks=M` one step ingests one batch of B events from each of M independent chunks of the stream (the DDP
partition of the reference's ChunkSampler, data_loader.py:23-48, on one GPU).  Node u of chunk c has the virtual id
c*N + u: every per-node state table has M*N rows, the launches above run on the M*B events of the step in that id
space, and only the finder (tiger_find_recent_ex), the chunk restart times (tiger_min_time_ex) and the static restart
(tiger_static_restart_ex) map a virtual id back to its real node for the shared CSR and restarter embeddings.
"""
from typing import Dict, Optional

import os

import numpy as np
import torch
from torch import Tensor

from . import _lib, ops
from ._lib import raise_on_err_flags
from .ops import f32, f64, i32, i64, u8

SELECT_SMALL_N = 2048      # tiger_select_latest ranks at most this many positions without per-node scratch
KERNELS_PER_STEP = {  # launches of our kernels per batch (for the bench `gpu_launches` field)
    'find_recent': 1, 'compact_involved': 1, 'gru_update': 1, 'temporal_attention': 4, 'select_latest': 1,
    'right_writeback': 1, 'store_messages': 2, 'left_writeback': 0, 'link_score': 1,
}


class TigerEngine:
    def __init__(self, weights: Dict[str, Tensor], csr: ops.DeviceCSR, *, n_nodes: int, dim: int,
                 efeats: Optional[Tensor], nfeats: Optional[Tensor] = None, n_neighbors: int = 10,
                 n_head: int = 2, batch_size: int = 200, msg_src: str = 'left', upd_src: str = 'right',
                 restarter: Optional[str] = None, hist_len: int = 40, hit_type: str = 'bin',
                 lazy_restart: bool = False, want_restarter_targets: bool = False, n_layers: int = 1,
                 msg_tsfm_type: str = 'id', mem_update_type: str = 'gru', n_chunks: int = 1, device='cuda'):
        """n_chunks = M: each step takes one batch of `batch_size` events from each of M chunks of the stream, and
        each chunk evolves exactly as a separate engine fed only that chunk's batches from reset() would (its own
        memories, message store, pending / up-to-date flags, lazy restart at its own batch minimum); the chunks share
        the weights, the CSR and the feature tables.  Inputs are chunk-major [M, batch_size] arrays of real node ids
        (set_batch, device_records), scores come back as [M, batch_size] (chunk_scores).  With M > 1 node 0 is the
        padding node only (ids of events start at 1, as in the reference's data): the input helpers reject id 0.  M = 1
        is the unchunked engine."""
        if isinstance(n_chunks, bool) or not isinstance(n_chunks, int) or n_chunks < 1:
            raise ValueError(f'n_chunks must be a positive int, got {n_chunks!r}')
        if n_chunks * n_nodes > 2 ** 31 - 1:
            raise ValueError(f'n_chunks * n_nodes = {n_chunks * n_nodes} virtual node ids do not fit the int32 index '
                             f'range of the per-node tables and the CSR')
        if n_chunks > 1 and want_restarter_targets:
            raise NotImplementedError('restarter targets (a training input) on a chunked engine')
        if n_layers not in (1, 2):
            raise NotImplementedError(f'n_layers={n_layers}: the engine runs one or two attention layers')
        if msg_src not in ('left', 'right') or upd_src not in ('left', 'right'):
            raise ValueError(f'Invalid msg_src={msg_src} / upd_src={upd_src}')   # tiger.py:156-160
        if hit_type not in ops.HIT_TYPES:
            raise NotImplementedError(f'hit_type={hit_type}')                  # tiger.py:129-136
        if msg_tsfm_type not in ops.MemoryUpdater.TSFM:
            raise NotImplementedError(f'msg_tsfm_type={msg_tsfm_type}')     # tiger.py:104-108
        if mem_update_type not in ops.MemoryUpdater.UPD:
            raise NotImplementedError(f'mem_update_type={mem_update_type}')   # tiger.py:110-113
        if lazy_restart and restarter not in ('static', 'seq'):
            raise NotImplementedError(f'lazy restart needs a seq or static restarter, got {restarter!r}')
        self.hit_type, self.K = hit_type, n_neighbors
        self.d = nfeats.shape[1] if nfeats is not None else dim              # feature_getter.py:76-77
        self._check_hit_weights(weights)
        dev = torch.device(device)
        self.device, self.csr = dev, csr
        # B: events per step over all chunks (what every launch is sized by); N: real nodes, NV: per-node table rows
        self.n_chunks, self.chunk_batch = n_chunks, batch_size
        self.N, self.H, self.B = n_nodes, n_head, n_chunks * batch_size
        self.NV = n_chunks * n_nodes
        self.n_layers = n_layers
        self.efeats = efeats
        # the attention, the message builder and the seq tokens read node features by (virtual) node id
        self.nfeats = nfeats.repeat(n_chunks, 1) if nfeats is not None and n_chunks > 1 else nfeats
        self.de = efeats.shape[1] if efeats is not None else dim
        # every layer has the same widths, K and heads; models past the attention kernel's limits run on the drop-in's
        # torch route
        limit = ops.attention_limit_error(self.d, self.de, n_neighbors, n_head)
        if limit is not None:
            raise NotImplementedError(limit)
        # the seq restarter's pooling kernel holds at most 64 history events: a longer history would fail at the first
        # restart, after compact_involved has already marked the restarted nodes up to date
        if restarter == 'seq':
            limit = ops.seq_restarter_limit_error(self.d, self.de, hist_len, n_head)
            if limit is not None:
                raise NotImplementedError(limit)
        self.M = 3 * self.d + self.de                                          # tiger.py:62
        self.msg_src, self.upd_src = msg_src, upd_src
        self.restarter, self.lazy_restart = restarter, lazy_restart
        self.want_targets = want_restarter_targets
        N, d, B, K = self.NV, self.d, self.B, self.K
        z = lambda *s, dt=f32: torch.zeros(*s, dtype=dt, device=dev)
        # ---- persistent state (reference: Memory x2, MessageStoreNoGradLastOnly) ----
        self.left_vals, self.left_ts, self.left_active = z(N, d), z(N), z(N, dt=u8)
        self.right_vals, self.right_ts, self.right_active = z(N, d), z(N), z(N, dt=u8)
        self.msg_vals, self.msg_ts, self.has_msg = z(N, self.M), z(N), z(N, dt=u8)
        self.uptodate = z(N, dt=u8)
        # ---- per-batch scratch (fixed capacity) ----
        # involved-node capacity: every query node and its K neighbors (collate_memory_nodes); with the second hop
        # the 3B*K hop-1 neighbors are queries too, and no list can hold more than the N distinct nodes
        self.cap = 3 * B * (K + 1) if n_layers == 1 else min((3 * B + 3 * B * K) * (K + 1), N)
        if n_chunks > 1:
            self.cap = min(self.cap, N)
        self.bitmap = z(ops.bitmap_words(N), dt=i32)
        self.involved, self.outdated, self.restart_nodes = z(self.cap, dt=i64), z(self.cap, dt=i64), z(self.cap, dt=i64)
        self.gru_row = torch.full((N,), -1, dtype=i32, device=dev)
        self.counts = z(4, dt=i32)
        self.err_flags = z(1, dt=i32)
        self.neigh_nids, self.neigh_eids = z(3 * B, K, dt=i64), z(3 * B, K, dt=i64)
        self.neigh_ts = z(3 * B, K)
        self.ts32 = z(B)
        if n_layers == 2:
            # second hop: the hop-1 table's times as float64 queries, the [3BK, K] table, the depth-1 embeddings
            self.neigh_ts64 = z(3 * B * K, dt=f64)
            self.neigh2_nids, self.neigh2_eids = z(3 * B * K, K, dt=i64), z(3 * B * K, K, dt=i64)
            self.neigh2_ts = z(3 * B * K, K)
            self.emb1 = z(3 * B * K, d)
        self.h_new = z(self.cap, d)
        self.emb = z(3 * B, d)
        self.winner = z(2 * B, dt=u8)
        self.sel_count = z(1, dt=i32)
        # M*B events can pass the all-pairs selection's 2,048 positions: the per-node slot route (same winners)
        self.sel_scratch = ops.SelectScratch(N, dev) if n_chunks > 1 and 2 * B > SELECT_SMALL_N else None
        self._stride = n_nodes if n_chunks > 1 else 0          # node stride of the chunk modes, 0: unchunked
        self.chunk_tmin = z(n_chunks, dt=f64) if n_chunks > 1 else None     # restart time of each chunk
        self.out_buf = z(2 * B + 1)                    # [pos scores | neg scores | loss]
        self.hprev_left = z(2 * B, d) if want_restarter_targets else None
        self.hprev_right = z(2 * B, d) if want_restarter_targets else None
        # ---- batch inputs: [src | dst | neg | eids] int64 and ts float64, one contiguous buffer ----
        self.inp = z(5 * B, dt=i64)
        self.bind_io(self.inp, self.out_buf)
        # ---- parameters ----
        self._side = torch.cuda.Stream(device=dev)
        self._serial = int(os.environ.get('TIGER_SERIAL', '0'))   # debug aid, bit mask: branches kept on the main stream
        self._ev_fork, self._ev_side = torch.cuda.Event(), torch.cuda.Event()
        self._ev_fork0, self._ev_rst = torch.cuda.Event(), torch.cuda.Event()
        # steps 1-2: message transform (--tsfm_fn) + memory updater (--upd_fn), scratch sized for `cap` outdated rows
        self.updater = ops.MemoryUpdater(msg_tsfm_type, mem_update_type, self.d, self.M, self.cap, dev)
        self.attn_pack = ops.AttnPack(self.d, self.de, dev, n_head)
        self.attn_pack1 = ops.AttnPack(self.d, self.de, dev, n_head) if n_layers == 2 else None   # fns.1 (depth 1)
        self.score_fold = ops.ScoreFold(self.d, dev, hit_type, K)
        self.pq = torch.zeros(3 * self.B, 2 * self.d, dtype=f32, device=dev)   # [W1a z | W1b z] per query row
        self.hist_len = hist_len
        self.seq = ops.SeqRestarterOp(self.d, self.de, hist_len, n_head, self.cap, dev) if restarter == 'seq' else None
        if self.seq is not None and n_chunks > 1:
            self.seq.tmin = self.chunk_tmin
            # the restarted rows of all chunks share one launch sequence, and the restarter picks its arithmetic route
            # (matrix-vector tail for few rows, tensor-core products otherwise) from their total count: a fixed route
            # keeps a chunk's rounding independent of how many nodes the other chunks restart
            self.seq.tail_rows = 0
        self.weights_version = 0            # counts load_weights calls: a graph captured before one is stale
        self.load_weights(weights)

    # ------------------------------------------------------------------ parameters
    def _check_hit_weights(self, W: Dict[str, Tensor]):
        """The scorer's hit parameters are sized by K (tiger.py:129-136); the fold reads them with this engine's K."""
        d, K = self.d, self.K
        want = {'count': ('hit_embedding.weight', (K + 1, d)), 'vec': ('score_fn.fc1.weight', (d, 2 * (d + K)))}
        if self.hit_type in want:
            name, shape = want[self.hit_type]
            if name not in W or tuple(W[name].shape) != shape:
                got = tuple(W[name].shape) if name in W else 'missing'
                raise ValueError(f'hit_type={self.hit_type} with n_neighbors={K}, dim={d}: {name} must be {shape}, '
                                 f'got {got}')

    def load_weights(self, W: Dict[str, Tensor]):
        """(Re)pack parameters given under the reference's state_dict names."""
        self._check_hit_weights(W)
        g = lambda k: W[k].detach().to(self.device, f32).contiguous()
        self.updater.refresh(g)
        a = 'temporal_embedding_fn.fns.0.'
        self.time_w, self.time_b = g('time_encoder.basis_freq'), g('time_encoder.phase')
        # fns.0 embeds the batch nodes (depth n_layers), fns.1 their neighbors (depth 1); the time encoder is shared
        for pack, fa in ((self.attn_pack, a), (self.attn_pack1, 'temporal_embedding_fn.fns.1.')):
            if pack is not None:
                pack.refresh(g(fa + 'mha_fn.q_proj_weight'), g(fa + 'mha_fn.k_proj_weight'),
                             g(fa + 'mha_fn.v_proj_weight'), g(fa + 'mha_fn.in_proj_bias'),
                             g(fa + 'mha_fn.out_proj.weight'), g(fa + 'mha_fn.out_proj.bias'),
                             g(fa + 'merger.fc1.weight'), g(fa + 'merger.fc1.bias'),
                             g(fa + 'merger.fc2.weight'), g(fa + 'merger.fc2.bias'), self.time_w, self.time_b)
        s = 'score_fn.'
        self.score_fold.refresh(g(s + 'fc1.weight'), g(s + 'fc1.bias'), g(s + 'fc2.weight'), g(s + 'fc2.bias'),
                                g(a + 'merger.fc2.weight'), g(a + 'merger.fc2.bias'),
                                g('hit_embedding.weight') if self.hit_type in ('bin', 'count') else None)
        self.attn_pack.attach_score_fold(self.score_fold, self.pq)
        if self.restarter == 'static':
            self.left_emb = g('restarter_fn.left_emb.weight')
            self.right_emb = g('restarter_fn.right_emb.weight')
        elif self.restarter == 'seq':
            self.seq.set_weights(W)
        self.weights_version += 1

    # ------------------------------------------------------------------ state
    def reset(self):
        """TIGE.reset (tiger.py:457-463) + a fresh up-to-date set."""
        for t in (self.left_vals, self.left_ts, self.left_active, self.right_vals, self.right_ts,
                  self.right_active, self.has_msg, self.uptodate, self.err_flags):
            t.zero_()

    def clear_messages(self):
        """msg_store.clear() + uptodate_nodes = set() of the restart trigger
        (train_self_supervised.py:153-156)."""
        self.has_msg.zero_()
        self.uptodate.zero_()

    def _mem(self, which):
        if which == 'left':
            return self.left_vals, self.left_ts
        return self.right_vals, self.right_ts

    def check_errors(self):
        """Host sync: raise the reference's ValueError if an invariant kernel flag is set."""
        raise_on_err_flags(int(self.err_flags.item()) & 0xffffffff)

    def set_batch(self, src, dst, neg, ts, eids):
        """Copy one batch (numpy or tensors; ts float64) into the device input buffer.  With n_chunks = M > 1 each
        argument is chunk-major [M, batch_size] with real node ids (fill_record)."""
        B = self.B
        host = torch.empty(5 * B, dtype=i64)
        h = host.numpy()
        if self.n_chunks > 1:
            self.fill_record(h, src, dst, neg, ts, eids)
        else:
            h[:B], h[B:2 * B], h[2 * B:3 * B], h[3 * B:4 * B] = src, dst, neg, eids
            h[4 * B:].view(np.float64)[:] = ts
        self.inp.copy_(host)

    def fill_record(self, h: np.ndarray, src, dst, neg, ts, eids):
        """Writes batches into int64 host records h [..., 5 * M * batch_size] (the layout of self.inp) from arrays
        (numpy or CPU tensors) of shape [..., M, batch_size]: real node ids, edge ids, float64 times.  Chunk c's node ids
        are stored as the virtual ids c * n_nodes + u, edge ids and times as given.  Node ids must lie in [0, n_nodes),
        and with M > 1 in [1, n_nodes): a chunked engine keeps id 0 for the padding of the neighbor tables, as the
        reference's data does (ids start at 1), so a real node 0 is rejected (ValueError)."""
        M, Bc = self.n_chunks, self.chunk_batch
        lo = 1 if M > 1 else 0
        rec = h.reshape(-1, 5, M, Bc)
        n = rec.shape[0]
        for i, x in enumerate((src, dst, neg)):
            x = np.asarray(x).reshape(n, M, Bc)
            if x.size and (x.min() < lo or x.max() >= self.N):
                raise ValueError(f'node ids outside [{lo}, {self.N})' + (' (node 0 is the padding node)' if lo else ''))
            np.add(x, np.arange(M, dtype=np.int64)[:, None] * self.N, out=rec[:, i])
        rec[:, 3] = np.asarray(eids).reshape(n, M, Bc)
        rec[:, 4] = np.asarray(ts, dtype=np.float64).reshape(n, M, Bc).view(np.int64)

    def device_records(self, src, dst, neg, ts, eids) -> Tensor:
        """Batch records for StreamRunner.submit_device, resident on the engine's device: arrays of shape
        [n, M, batch_size] give int64 [n, 5 * M * batch_size], arrays of shape [M, batch_size] one record [5 * M *
        batch_size] (fill_record)."""
        one = np.asarray(src).ndim <= 2
        h = np.empty((np.asarray(src).size // self.B, 5 * self.B), dtype=np.int64)
        self.fill_record(h, src, dst, neg, ts, eids)
        out = torch.from_numpy(h).to(self.device)
        return out[0] if one else out

    def chunk_scores(self):
        """(pos, neg) link-scorer logits of the latest step, float32 [M, batch_size] views of the result buffer.  The
        step's loss (self.loss) is the mean BCE over all 2 M batch_size rows; with equal batches per chunk that is the
        mean of the M per-chunk losses."""
        M, Bc = self.n_chunks, self.chunk_batch
        return self.scores[:self.B].view(M, Bc), self.scores[self.B:].view(M, Bc)

    # ------------------------------------------------------------------ the launch sequence
    def launch_finder(self):
        ops.find_recent(self.csr, self.batch_nids, self.ts64, self.K, ts_period=self.B, want_dirs=False,
                        ts32_out=self.ts32, bitmap=self.bitmap,
                        out=(self.neigh_nids, self.neigh_eids, self.neigh_ts, None),
                        chunk_mode=ops.FIND_CHUNK_NEIGHBORS if self._stride else 0, node_stride=self._stride)
        if self.n_layers == 2:
            ops.find_second_hop(self.csr, self.neigh_nids, self.neigh_ts, self.K, ts64=self.neigh_ts64,
                                bitmap=self.bitmap, out=(self.neigh2_nids, self.neigh2_eids, self.neigh2_ts),
                                node_stride=self._stride)

    def launch_model(self, with_scorer: bool = True):
        d, B = self.d, self.B
        # Branches (restarter beside the GRU, write-back / message store beside the attention chain) exist only under
        # graph capture, where they become parallel paths of the graph with explicit edges; eager launches (tests,
        # smoke, debugging) stay on one stream.  TIGER_SERIAL is a debug bit mask (1: restarter, 2: write-back /
        # message branch) that keeps a branch on the main stream under capture as well; TIGER_EAGER_BRANCHES=1
        # re-enables the branches for eager launches (tools/eager_race.py).
        cur = torch.cuda.current_stream()
        serial = self._serial if (torch.cuda.is_current_stream_capturing() or os.environ.get('TIGER_EAGER_BRANCHES') == '1') else 7
        side0 = cur if serial & 1 else self._side
        side1 = cur if serial & 2 else self._side
        msg_vals_mem, msg_ts_mem = self._mem(self.msg_src)
        upd_vals, _ = self._mem(self.upd_src)
        ops.compact_involved(self.bitmap, self.NV, self.involved, self.counts, has_msg=self.has_msg,
                             uptodate=self.uptodate if self.lazy_restart else None, outdated=self.outdated,
                             gru_row=self.gru_row, restart_nodes=self.restart_nodes if self.lazy_restart else None,
                             err_flags=self.err_flags)
        # Fork 0: the restart only writes rows of nodes compact_involved put on the restart list, which it also
        # removed from the outdated list (csrc/graph.cu: pend = member && has_msg && !rst), i.e. rows the GRU
        # neither reads nor writes - the restarter runs next to the GRU on the side stream; the attention and
        # the message builder (same side stream, later) read restarted rows and wait for it.
        main = torch.cuda.current_stream()
        if self.lazy_restart:
            self._ev_fork0.record(main)
            with torch.cuda.stream(side0):
                side0.wait_event(self._ev_fork0)
                if self.restarter == 'static':
                    # chunked: each chunk cuts at the minimum of its own batch times
                    if self._stride:
                        ops.min_time(self.ts32, self.chunk_tmin, self.n_chunks)
                    ops.static_restart(self.restart_nodes, self.cap, self.csr, self.left_emb, self.right_emb, d,
                                       count=self.counts[2:], batch_ts=self.ts32, left_vals=self.left_vals,
                                       left_ts=self.left_ts, left_active=self.left_active, right_vals=self.right_vals,
                                       right_ts=self.right_ts, right_active=self.right_active, has_msg=self.has_msg,
                                       node_stride=self._stride, chunk_ts=self.chunk_tmin)
                else:
                    # TIGER.restart with the seq restarter (tiger.py:594-609, restarters.py:51-114): history at
                    # ts.min() of the batch, surrogate h(t'-) / h(t'+), both memories overwritten without checks
                    # (compact_involved has already dropped the pending-message flags of these nodes)
                    R = self.counts[2:]
                    ops.min_time(self.ts32, self.seq.tmin, self.n_chunks)
                    self.seq.history(self.csr, self.restart_nodes, self.seq.tmin, self.cap, ts_period=1, count=R,
                                     node_stride=self._stride)
                    hl, hr, pt = self.seq.forward(self.restart_nodes, self.cap, self.nfeats, self.efeats, count=R)
                    ops.scatter_rows(self.left_vals, self.restart_nodes, hl, ts_table=self.left_ts, ts=pt,
                                     active=self.left_active, count=R)
                    ops.scatter_rows(self.right_vals, self.restart_nodes, hr, ts_table=self.right_ts, ts=pt,
                                     active=self.right_active, count=R)
                self._ev_rst.record(side0)
        self.updater.launch(node_ids=self.outdated, x_table=self.msg_vals, h_table=upd_vals, n_rows=self.cap,
                            out=self.h_new, count=self.counts[1:], msg_ts=self.msg_ts, check_mem_ts=msg_ts_mem,
                            check_equal=(self.msg_src == 'left'), err_flags=self.err_flags)
        # Fork: the write-back / message branch (argmax-by-timestamp selection -> right write-back -> message
        # build + store) only needs the GRU output and the batch, and touches rows the attention never reads
        # (right-memory rows of nodes WITH a pending message are read from h_new, csrc/attention.cu
        # resolve_row), so it runs on a side stream next to the attention chain.  Captured in a CUDA graph
        # the two branches become parallel paths of the graph.
        if self.lazy_restart and (serial & 2):
            main.wait_event(self._ev_rst)
        self._ev_fork.record(main)
        with torch.cuda.stream(side1):
            side1.wait_event(self._ev_fork)
            ops.select_latest(self.pos, self.ts32, self.sel_scratch, want_unique=False, winner=self.winner,
                              want_count=False)
            ops.right_writeback(self.pos, self.winner, self.gru_row, self.h_new, d, self.right_vals, self.right_ts,
                                self.right_active, self.msg_ts, self.has_msg, self.left_vals, self.hprev_left,
                                self.hprev_right, self.err_flags)
            ops.store_messages(self.src, self.dst, self.eids, self.ts32, self.winner, msg_vals_mem, msg_ts_mem,
                               self.nfeats, self.efeats, d, self.de, self.time_w, self.time_b, self.msg_vals,
                               self.msg_ts, self.has_msg, self.err_flags)
            self._ev_side.record(side1)
        if self.lazy_restart:
            main.wait_event(self._ev_rst)
        key_rows = None
        if self.n_layers == 2:
            # depth 1 (fns.1): one query per entry of the batch nodes' neighbor table, at the parent event's time
            # (repeat_interleave(ts.repeat(3), K)), over the second hop.  It reads node rows through resolve_row only,
            # like depth 2, so the side branch may overlap it (DESIGN.md, "Why the post-GRU branches may overlap").
            # It must stay on this stream right in front of depth 2: depth 2 gathers emb1 before its dependency wait
            # (csrc/attention.cu, attn_score_pool_kernel).
            ops.temporal_attention(self.attn_pack1, self.H, self.neigh_nids.view(-1), self.ts32, self.neigh2_nids,
                                   self.neigh2_eids, self.neigh2_ts, rows_a=self.right_vals, rows_b=self.h_new,
                                   sel=self.gru_row, nfeats=self.nfeats, efeats=self.efeats, out=self.emb1,
                                   ts_group=self.K)
            key_rows = self.emb1
        # update_left_memory is fused into the last attention product, which first waits for the side branch (the
        # message builder reads the OLD left-memory rows, and `winner` comes from the selection kernel)
        self.attn_pack.attach_left_writeback(self.pos, self.winner, self.ts32, self.left_vals, self.left_ts,
                                             self.left_active, self.err_flags, ready_event=self._ev_side)
        ops.temporal_attention(self.attn_pack, self.H, self.batch_nids, self.ts32, self.neigh_nids, self.neigh_eids,
                               self.neigh_ts, rows_a=self.right_vals, rows_b=self.h_new, sel=self.gru_row,
                               nfeats=self.nfeats, efeats=self.efeats, out=self.emb, key_rows=key_rows)
        # the link scorer reads the projections `pq` of the embeddings and changes no state: in the pipelined replay
        # it is a separate graph on the copy-out stream (launch_scorer), beside the next batch's model kernels
        if with_scorer:
            self.launch_scorer()

    def launch_scorer(self):
        ops.link_score_folded(self.score_fold, self.pq, self.src, self.dst, self.neg,
                              self.neigh_nids if self.hit_type != 'none' else None, self.scores, self.loss)

    def bind_pq(self, pq: Tensor):
        """The [3B, 2d] first-layer projections of the link scorer, written by the last attention product and read
        by the scorer: one buffer per pipeline slot, because the scorer of batch i runs beside batch i+1."""
        assert pq.shape == self.pq.shape and pq.dtype == f32
        self.pq = pq
        self.attn_pack.attach_score_fold(self.score_fold, pq)

    def bind_io(self, inp: Tensor, out_buf: Tensor):
        """Points the batch-input views ([src | dst | neg | eids | ts as f64 bits], int64 [5B]) and the result
        views ([pos scores | neg scores | loss], f32 [2B + 1]) at the given device buffers.  Launches issued (or
        captured into a CUDA graph) afterwards read / write them: the host path keeps one buffer pair per
        staging slot so that uploads and downloads of neighbouring batches overlap the kernels."""
        B = self.B
        assert inp.numel() == 5 * B and inp.dtype == i64 and out_buf.numel() == 2 * B + 1 and out_buf.dtype == f32
        self.inp, self.out_buf = inp, out_buf
        self.batch_nids = inp[:3 * B]
        self.src, self.dst, self.neg = inp[:B], inp[B:2 * B], inp[2 * B:3 * B]
        self.pos = inp[:2 * B]
        self.eids = inp[3 * B:4 * B]
        self.ts64 = inp[4 * B:].view(f64)
        self.scores, self.loss = out_buf[:2 * B], out_buf[2 * B:]

    def finder_buffers(self, fresh: bool = False):
        """The finder's outputs (neighbor tables, float32 batch times, involved-node bitmap; with n_layers=2 also the
        float64 hop-1 times and the hop-2 tables).  They depend on the static graph and the batch only, not on the
        memory state, so the finder of batch i+1 may run while batch i is still in its model kernels - provided it
        writes its own set (`fresh=True` allocates one)."""
        bufs = (self.neigh_nids, self.neigh_eids, self.neigh_ts, self.ts32, self.bitmap)
        if self.n_layers == 2:
            bufs += (self.neigh_ts64, self.neigh2_nids, self.neigh2_eids, self.neigh2_ts)
        if not fresh:
            return bufs
        return tuple(torch.zeros_like(t) for t in bufs)

    def bind_finder(self, bufs):
        self.neigh_nids, self.neigh_eids, self.neigh_ts, self.ts32, self.bitmap = bufs[:5]
        if self.n_layers == 2:
            self.neigh_ts64, self.neigh2_nids, self.neigh2_eids, self.neigh2_ts = bufs[5:]

    def launches_per_step(self) -> int:
        n = sum(KERNELS_PER_STEP.values()) + self.updater.launches - KERNELS_PER_STEP['gru_update']
        if self.n_layers == 2:
            # hop-2 finder + the float64 widening of the hop-1 times (a torch copy) + the depth-1 attention chain
            n += 2 + KERNELS_PER_STEP['temporal_attention']
        if self.lazy_restart:
            n += 1 if self.restarter == 'static' else ops.SeqRestarterOp.LAUNCHES + 2
            if self.restarter == 'seq' and self.n_chunks > 1:
                n -= ops.SeqRestarterOp.TAIL_LAUNCHES                             # products only
            n += int(self.restarter == 'static' and self.n_chunks > 1)     # the chunk restart times
        if self.sel_scratch is not None:
            n += 3          # per-node slot selection: max-ts, min-position, flag and reset kernels
        if self.want_targets:
            n += 1
        return n

    def step(self):
        """One batch, eager launches on the current stream (inputs already in self.inp)."""
        self.launch_finder()
        self.launch_model()

    def candidate_query(self, max_queries: int, n_candidates: int) -> 'CandidateQuery':
        """A read-only scorer of up to `max_queries` sources against `n_candidates` candidates each on this engine's
        current state and weights (CandidateQuery)."""
        if self.n_chunks > 1:
            raise NotImplementedError('candidate_query on a chunked engine (n_chunks > 1)')
        return CandidateQuery(self, max_queries, n_candidates)


class CandidateQuery:
    """`scores, ranks = q.score(src [Q], cands [Q, C], ts [Q])`: scores[i, j] is the link-scorer logit the ingest step
    would produce for the event (src[i], cands[i, j]) at ts[i] on the engine's current state - lazy restart of
    not-yet-seen nodes at min(ts) as a surrogate, the updater overlay of nodes with a pending message, the attention
    (one or two layers), the hit flags of cands[i, j] against src[i], the folded scorer - and ranks[i] =
    1 + #{j >= 1: s_ij > s_i0} + 0.5 #{j >= 1: s_ij == s_i0} ranks column 0, the true candidate (ties count half; a
    NaN s_i0 gives a NaN rank, a NaN s_ij neither beats nor ties s_i0).

    Nothing persistent changes: the memories, the message store, `has_msg` and `uptodate` are only read, and the query
    owns all its scratch (finder tables, bitmap, lists, `gru_row`, updater / attention / restarter workspaces, `pq`).
    The weight packs are the engine's own, so `load_weights` reaches both paths; a graph captured before it would read
    replaced weight tensors, so score() drops it and launches eagerly until capture() is called again.  The query's node list is [src | cands[:, 0] | cands[:, 1] | ...], the ingest step's batch layout
    with 3 -> 1 + C rows per event: with C = 2 and cands = [dst, neg] it is that batch, and its scores are the step's.

    Launches go to the current stream, behind the ingest steps issued there before; with a StreamRunner call
    `runner.join()` first.  The results are views of this object's buffers (scores [Q, C] is the transpose of a
    candidate-major [C, Q] buffer), valid until the next score()."""

    def __init__(self, engine: TigerEngine, max_queries: int, n_candidates: int):
        if not (isinstance(max_queries, int) and isinstance(n_candidates, int)) or max_queries < 1 or n_candidates < 1:
            raise ValueError(f'max_queries and n_candidates must be positive ints, got {max_queries!r}, {n_candidates!r}')
        e = self.e = engine
        self.Q, self.C = max_queries, n_candidates
        N, d, K, dev = e.N, e.d, e.K, e.device
        n = (1 + n_candidates) * max_queries
        full = n * (K + 1) if e.n_layers == 1 else (n + n * K) * (K + 1)
        # the lists hold distinct nodes, so never more than N.  A query with at least as many rows as a batch gets at
        # least the engine's own capacity, so that a query shaped like the batch (C = 2, max_queries = B) gets exactly
        # that capacity and runs the step's launch shapes (the GEMMs pick their tiles by capacity)
        self.cap = cap = min(full, max(N, e.cap))
        z = lambda *sh, dt=f32: torch.zeros(*sh, dtype=dt, device=dev)
        # inputs: [src | cands column-major] int64 [(1+C)Q], then the times as float64 bits [Q]
        self.inp = z(n + max_queries, dt=i64)
        self.nids, self.ts64 = self.inp[:n], self.inp[n:].view(f64)
        self.ts32 = z(max_queries)
        self.bitmap = z(ops.bitmap_words(N), dt=i32)
        self.involved, self.outdated, self.restart_nodes = z(cap, dt=i64), z(cap, dt=i64), z(cap, dt=i64)
        self.gru_row = torch.full((N,), -1, dtype=i32, device=dev)
        self.counts, self.err_flags = z(4, dt=i32), z(1, dt=i32)
        self.neigh_nids, self.neigh_eids, self.neigh_ts = z(n, K, dt=i64), z(n, K, dt=i64), z(n, K)
        if e.n_layers == 2:
            self.neigh_ts64 = z(n * K, dt=f64)
            self.neigh2_nids, self.neigh2_eids, self.neigh2_ts = z(n * K, K, dt=i64), z(n * K, K, dt=i64), z(n * K, K)
            self.emb1 = z(n * K, d)
        # node rows the attention reads through gru_row: updater output [0, O), restart surrogates [cap, cap + R)
        self.rows_b = z(2 * cap, d)
        self.emb, self.pq = z(n, d), z(n, 2 * d)
        self.scores, self.ranks = z(n_candidates * max_queries), z(max_queries)
        self.upd_scratch = e.updater.scratch(cap)
        self.attn = e.attn_pack.share()
        self.attn.attach_score_fold(e.score_fold, self.pq)
        self.attn1 = e.attn_pack1.share() if e.attn_pack1 is not None else None
        # both attention workspaces sized once, for max_queries: a captured graph keeps their addresses whatever Q the
        # eager calls in between use
        self.attn.work(n, K)
        if self.attn1 is not None:
            self.attn1.work(n * K, K)
        self.seq = None
        if e.lazy_restart and e.restarter == 'seq':
            self.seq = ops.SeqRestarterOp(d, e.de, e.hist_len, e.H, cap, dev)
            self.seq.h_right = self.rows_b[cap:]        # the restarter writes the surrogates in place
        self.graph = self._graph_key = None

    # ------------------------------------------------------------------ inputs
    def _upload(self, src, cands, ts, Q: int):
        C = self.C
        as_t = lambda x: x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
        src, cands, ts = as_t(src), as_t(cands), as_t(ts)
        self.nids[:Q].copy_(src)
        self.nids[Q:(1 + C) * Q].view(C, Q).copy_(cands.t())
        self.ts64[:Q].copy_(ts)

    # ------------------------------------------------------------------ the launch sequence
    def launch(self, Q: int, ranks: bool = True):
        """The query's launches for the first Q queries already in the input buffer (no host sync)."""
        e, cap, K, C = self.e, self.cap, self.e.K, self.C
        n = (1 + C) * Q
        nids, ts64, ts32 = self.nids[:n], self.ts64[:Q], self.ts32[:Q]
        nn, ne, nt = self.neigh_nids[:n], self.neigh_eids[:n], self.neigh_ts[:n]
        ops.find_recent(e.csr, nids, ts64, K, ts_period=Q, want_dirs=False, ts32_out=ts32, bitmap=self.bitmap,
                        out=(nn, ne, nt, None))
        if e.n_layers == 2:
            n2 = (self.neigh2_nids[:n * K], self.neigh2_eids[:n * K], self.neigh2_ts[:n * K])
            ops.find_second_hop(e.csr, nn, nt, K, ts64=self.neigh_ts64[:n * K], bitmap=self.bitmap, out=n2)
        ops.compact_involved(self.bitmap, e.N, self.involved, self.counts, has_msg=e.has_msg,
                             uptodate=e.uptodate if e.lazy_restart else None, outdated=self.outdated,
                             gru_row=self.gru_row, restart_nodes=self.restart_nodes if e.lazy_restart else None,
                             err_flags=self.err_flags, read_only=True, restart_base=cap)
        if e.lazy_restart:
            R = self.counts[2:]
            if e.restarter == 'static':
                ops.static_restart_rows(self.restart_nodes, cap, e.right_emb, e.d, self.rows_b[cap:], count=R)
            else:
                self.seq.share_weights(e.seq)
                ops.min_time(ts32, self.seq.tmin)
                self.seq.history(e.csr, self.restart_nodes, self.seq.tmin, cap, ts_period=1, count=R)
                self.seq.forward(self.restart_nodes, cap, e.nfeats, e.efeats, count=R)
        msg_ts_mem = e._mem(e.msg_src)[1]
        e.updater.launch(node_ids=self.outdated, x_table=e.msg_vals, h_table=e._mem(e.upd_src)[0], n_rows=cap,
                         out=self.rows_b[:cap], count=self.counts[1:], msg_ts=e.msg_ts, check_mem_ts=msg_ts_mem,
                         check_equal=(e.msg_src == 'left'), err_flags=self.err_flags, scratch=self.upd_scratch)
        rows = dict(rows_a=e.right_vals, rows_b=self.rows_b, sel=self.gru_row, nfeats=e.nfeats, efeats=e.efeats)
        key_rows = None
        if e.n_layers == 2:
            key_rows = self.emb1[:n * K]
            ops.temporal_attention(self.attn1, e.H, nn.view(-1), ts32, *n2, out=key_rows, ts_group=K, **rows)
        ops.temporal_attention(self.attn, e.H, nids, ts32, nn, ne, nt, out=self.emb[:n], key_rows=key_rows,
                               read_only=True, **rows)
        ops.link_score_cands(e.score_fold, self.pq[:n], nids[:Q], nids[Q:2 * Q], nids[2 * Q:],
                             nn if e.hit_type != 'none' else None, self.scores[:C * Q],
                             self.ranks[:Q] if ranks else None)

    def capture(self, n_queries: Optional[int] = None, ranks: bool = True):
        """Record launch(n_queries, ranks) as one CUDA graph; score() replays it for that many queries once it has
        copied the inputs into the input buffer."""
        Q = self.Q if n_queries is None else n_queries
        if not 1 <= Q <= self.Q:
            raise ValueError(f'n_queries={Q}: this CandidateQuery takes 1 to max_queries={self.Q}')
        s = torch.cuda.Stream(device=self.e.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.launch(Q, ranks)               # warm-up: module loads and kernel attributes outside the capture
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.launch(Q, ranks)
        torch.cuda.synchronize()
        self.graph, self._graph_key = graph, (Q, ranks, self.e.weights_version)

    def score(self, src, cands, ts, ranks: bool = True):
        """src int64 [Q], cands int64 [Q, C], ts float64 [Q] (numpy arrays or tensors) -> (scores [Q, C], ranks [Q] or
        None), float32 views of this object's buffers.  ValueError before any launch for a wrong dtype, rank, shape,
        node id or Q > max_queries."""
        Q = check_query_inputs(src, cands, ts, max_queries=self.Q, n_candidates=self.C, n_nodes=self.e.N,
                               device=self.e.device)
        self._upload(src, cands, ts, Q)
        if self.graph is not None and self._graph_key[2] != self.e.weights_version:
            self.graph = self._graph_key = None          # captured on weight tensors load_weights has replaced
        if self.graph is not None and self._graph_key[:2] == (Q, ranks):
            self.graph.replay()
        else:
            self.launch(Q, ranks)
        return self.scores[:self.C * Q].view(self.C, Q).t(), (self.ranks[:Q] if ranks else None)

    def check_errors(self):
        """Host sync: raise the reference's ValueError if an invariant flag of this object's launches is set."""
        raise_on_err_flags(int(self.err_flags.item()) & 0xffffffff)


class StreamRunner:
    """Replays an event stream through a TigerEngine.

    `capture()` records the whole batch as one CUDA graph (`run_device`, inputs in engine.inp) and, per staging
    slot, a finder graph and a model graph bound to the slot's own device input / result buffers and finder
    outputs.  `submit_host` / `submit_device` hand a batch to the native pipeline (csrc/pipe.cu): upload + finder
    on a copy-in stream beside the previous batch's model kernels, model graphs in batch order on the current
    stream, download on a copy-out stream - seven CUDA calls per batch, issued from C."""

    def __init__(self, engine: TigerEngine, n_slots: int = 4):
        self.e = engine
        self.graph = None
        self.pipe = None
        B = engine.B
        self.n_slots = n_slots
        self.h_in = [torch.empty(5 * B, dtype=i64).pin_memory() for _ in range(n_slots)]
        self.h_out = [torch.empty(2 * B + 1, dtype=f32).pin_memory() for _ in range(n_slots)]
        self._h_in_np = [t.numpy() for t in self.h_in]
        dev = engine.inp.device
        self.d_in = [torch.zeros(5 * B, dtype=i64, device=dev) for _ in range(n_slots)]
        self.d_out = [torch.zeros(2 * B + 1, dtype=f32, device=dev) for _ in range(n_slots)]
        self.finder_bufs = [engine.finder_buffers(fresh=True) for _ in range(n_slots)]
        self.pq_bufs = [torch.zeros_like(engine.pq) for _ in range(n_slots)]
        self.slot_busy = [False] * n_slots
        self.check_on_wait = False     # True: wait() also polls the device error word (one more host sync per batch)
        self.slot = 0
        self._lib = _lib.load()

    def __del__(self):
        if getattr(self, 'pipe', None):
            self._lib.tiger_pipe_destroy(self.pipe)
            self.pipe = None

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise _lib.TigerLibraryError(f'{what} failed with code {rc}')

    def capture(self, warmup: int = 2):
        """Warm up (eagerly, state restored afterwards is the caller's business) and capture."""
        e = self.e
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(warmup):
                e.step()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            e.step()
        torch.cuda.synchronize()
        # Per-slot graphs for the pipeline.  The finder (a function of the static graph and the batch only) is
        # captured separately and replayed on the copy-in stream right behind the slot's upload, i.e. beside the
        # model kernels of the previous batch; it writes the slot's own neighbor tables / bitmap, which that
        # slot's model graph reads.
        if self.pipe:
            self._lib.tiger_pipe_destroy(self.pipe)
        self.pipe = self._lib.tiger_pipe_create(self.n_slots)
        if not self.pipe:
            raise _lib.TigerLibraryError('tiger_pipe_create failed')
        inp0, out0, find0, pq0 = e.inp, e.out_buf, e.finder_buffers(), e.pq
        cap = torch.cuda.Stream()
        with torch.cuda.stream(cap):
            for slot in range(self.n_slots):
                e.bind_io(self.d_in[slot], self.d_out[slot])
                e.bind_finder(self.finder_bufs[slot])
                e.bind_pq(self.pq_bufs[slot])
                for kind, launch in ((0, e.launch_finder), (1, lambda: e.launch_model(with_scorer=False)),
                                     (2, e.launch_scorer)):
                    self._check(self._lib.tiger_pipe_capture_begin(cap.cuda_stream), 'capture_begin')
                    try:
                        launch()
                    finally:
                        rc = self._lib.tiger_pipe_capture_end(self.pipe, cap.cuda_stream, slot, kind)
                    self._check(rc, 'capture_end')
        e.bind_io(inp0, out0)
        e.bind_finder(find0)
        e.bind_pq(pq0)
        torch.cuda.synchronize()

    def join(self):
        """Makes the current stream wait for the copy-out stream's work (link scorer, download) of the latest batch."""
        if self.pipe:
            self._check(self._lib.tiger_pipe_join(self.pipe, _lib.stream_ptr()), 'pipe_join')

    def run_device(self):
        """Inputs already resident in engine.inp."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self.e.step()

    def _next_slot(self) -> int:
        slot = self.slot
        self.slot = (slot + 1) % self.n_slots
        return slot

    def submit_device(self, batch: Tensor) -> int:
        """One step on a batch that is already resident in HBM (int64 [5B], layout of engine.inp): staged into the
        next slot's input buffer on the copy-in stream (beside the previous batch's kernels), then that slot's
        graphs.  Results stay in d_out[slot]; returns the slot."""
        if not self.pipe:
            self.e.inp.copy_(batch, non_blocking=True)
            self.run_device()
            return 0
        slot = self._next_slot()
        self._check(self._lib.tiger_pipe_submit(self.pipe, slot, batch.data_ptr(), self.d_in[slot].data_ptr(),
                                                batch.numel() * 8, None, None, 0, _lib.stream_ptr()), 'pipe_submit')
        return slot

    def fill_host(self, slot: int, src, dst, neg, ts, eids):
        if self.e.n_chunks > 1:
            self.e.fill_record(self._h_in_np[slot], src, dst, neg, ts, eids)
            return
        B = self.e.B
        h = self._h_in_np[slot]
        h[:B], h[B:2 * B], h[2 * B:3 * B], h[3 * B:4 * B] = src, dst, neg, eids
        h[4 * B:].view(np.float64)[:] = ts

    def submit_host(self, src, dst, neg, ts, eids) -> int:
        """Host-buffer step: H2D of the batch, the graphs, D2H of scores + loss.  Returns the slot whose
        results become readable after `wait(slot)`.  A chunked engine takes chunk-major [M, batch_size] arrays of
        real node ids (TigerEngine.fill_record)."""
        slot = self._next_slot()
        if self.slot_busy[slot]:
            raise RuntimeError(f'staging slot {slot} still holds unread results: call wait(slot) on every slot returned '
                               f'by submit_host before more than {self.n_slots} batches are in flight')
        self.fill_host(slot, src, dst, neg, ts, eids)
        if not self.pipe:
            e = self.e
            e.inp.copy_(self.h_in[slot], non_blocking=True)
            self.run_device()
            self.h_out[slot].copy_(e.out_buf, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        else:
            self._check(self._lib.tiger_pipe_submit(self.pipe, slot, self.h_in[slot].data_ptr(),
                                                    self.d_in[slot].data_ptr(), self.h_in[slot].numel() * 8,
                                                    self.d_out[slot].data_ptr(), self.h_out[slot].data_ptr(),
                                                    self.h_out[slot].numel() * 4, _lib.stream_ptr()), 'pipe_submit')
        self.slot_busy[slot] = True
        return slot

    def wait(self, slot: int):
        if self.pipe and self.slot_busy[slot]:
            self._check(self._lib.tiger_pipe_wait(self.pipe, slot, 1), 'pipe_wait')
        self.slot_busy[slot] = False
        if self.check_on_wait:
            self.e.check_errors()          # attribute an invariant violation to (at most n_slots batches around) this one
        out = self.h_out[slot]
        B = self.e.B
        if self.e.n_chunks > 1:
            # [M, batch_size] scores; the loss is the mean over all 2 M batch_size rows, which with equal batches is
            # the mean of the M per-chunk losses
            shape = (self.e.n_chunks, self.e.chunk_batch)
            return out[:B].view(shape), out[B:2 * B].view(shape), out[2 * B]
        return out[:B], out[B:2 * B], out[2 * B]

    @property
    def h2d_bytes_per_step(self) -> int:
        return self.h_in[0].numel() * 8

    @property
    def d2h_bytes_per_step(self) -> int:
        return self.h_out[0].numel() * 4


def chunk_bounds(n: int, n_chunks: int, batch_size: int, seed: int = 0, epoch: int = 0):
    """The reference's DDP partition of n events into n_chunks contiguous chunks (ChunkSampler.bounds of every rank,
    data_loader.py:23-48): [(lo_c, hi_c)] with hi_c - lo_c = n // (n_chunks * batch_size) * batch_size, all chunks
    shifted by one draw from Generator(seed + epoch).  Batch i of a chunked engine is events
    [lo_c + i * batch_size, lo_c + (i + 1) * batch_size) of every chunk c."""
    from .tiger.data.data_loader import ChunkSampler
    bounds = []
    for rank in range(n_chunks):
        s = ChunkSampler(n, rank, n_chunks, batch_size, seed=seed)
        s.set_epoch(epoch)
        bounds.append(s.bounds())
    return bounds


def check_query_inputs(src, cands, ts, *, max_queries: int, n_candidates: int, n_nodes: int, device) -> int:
    """The checks CandidateQuery.score runs before it launches anything: src int64 [Q], cands int64
    [Q, n_candidates], ts float64 [Q], numpy arrays or tensors (CUDA tensors on `device`), 1 <= Q <= max_queries, node
    ids in [0, n_nodes).  Raises ValueError; returns Q."""
    def dtype_of(x, what):
        if isinstance(x, torch.Tensor):
            return str(x.dtype).replace('torch.', '')
        if isinstance(x, np.ndarray):
            return str(x.dtype)
        raise ValueError(f'{what} must be a numpy array or a torch tensor, got {type(x).__name__}')
    for x, what, dt, nd in ((src, 'src', 'int64', 1), (cands, 'cands', 'int64', 2), (ts, 'ts', 'float64', 1)):
        if dtype_of(x, what) != dt:
            raise ValueError(f'{what} must be {dt}, got {dtype_of(x, what)}')
        if x.ndim != nd:
            raise ValueError(f'{what} must have {nd} dimension(s), got shape {tuple(x.shape)}')
        if isinstance(x, torch.Tensor) and x.is_cuda:
            want = torch.device(device)
            if want.index is None:
                want = torch.device(want.type, torch.cuda.current_device())
            if x.device != want:
                raise ValueError(f'{what} is on {x.device}, the engine on {want}')
    Q = src.shape[0]
    if Q < 1 or Q > max_queries:
        raise ValueError(f'{Q} queries: this CandidateQuery takes 1 to max_queries={max_queries}')
    if tuple(cands.shape) != (Q, n_candidates):
        raise ValueError(f'cands must be [{Q}, n_candidates={n_candidates}], got {tuple(cands.shape)}')
    if tuple(ts.shape) != (Q,):
        raise ValueError(f'ts must be [{Q}], got {tuple(ts.shape)}')
    for x, what in ((src, 'src'), (cands, 'cands')):
        lo, hi = (x.min(), x.max()) if isinstance(x, np.ndarray) else (int(v) for v in torch.aminmax(x))
        if lo < 0 or hi >= n_nodes:
            raise ValueError(f'{what} holds node ids outside [0, {n_nodes})')
    return Q
