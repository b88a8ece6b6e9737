/*
 * tiger_b200.h - C ABI of libtiger_b200.so: hand-written sm_100a kernels for TIGER's
 * per-batch temporal memory path (reference: yzhang1918/www2023tiger, 100 % Python).
 *
 * The reference has no FFI layer: its "operator API" is the tiger/model + tiger/data class
 * surface (SURVEY.md §8(b)).  Each entry point below replaces the device work of the
 * reference method cited beside it; www2023tiger_b200/ mirrors those classes and calls
 * these functions through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C: raw device pointers + sizes + cudaStream_t (passed as void*); no torch types.
 *   - the CALLER owns every buffer; functions never allocate, never synchronise and are
 *     stream-ordered, so a whole batch is capturable in a CUDA graph.
 *   - node / edge ids are int64 (the reference's LongTensor); the CSR stores int32.
 *   - values fp32; finder timestamps fp64 (reference graph.py:51 compares float64).
 *   - data-dependent counts (involved U, outdated O, restarted R) stay on the device:
 *     kernels take an `int32_t* count` and size their loops from it.
 *   - return 0 on success, TIGER_EINVAL for a rejected argument, TIGER_ECUDA when the launch
 *     failed (cudaGetLastError).  Invariant violations that the reference raises through
 *     `.item()` host syncs are OR-ed into a device word `err_flags` (TIGER_ERR_*).
 */
#ifndef TIGER_B200_H
#define TIGER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TIGER_OK 0
#define TIGER_EINVAL (-1)
#define TIGER_ECUDA (-2)

/* bits of the device-side error word */
#define TIGER_ERR_PAST_MEMORY 1u      /* memory.py:45  "not allowed to modify past memory"      */
#define TIGER_ERR_UNUSED_MSG 2u       /* memory.py:87  "Node has unused messages"               */
#define TIGER_ERR_MSG_BEFORE_MEM 4u   /* message_modules.py:158 "Messages happened later ..."   */
#define TIGER_ERR_MSG_TS_MISMATCH 8u  /* tiger.py:325  msg ts != left update ts                 */
#define TIGER_ERR_EVENT_BEFORE_MEM 16u /* tiger.py:437 "Events occur before the updated memory" */
#define TIGER_ERR_CAPACITY 32u        /* a caller-provided list capacity was exceeded           */

int tiger_abi_version(void);

/* ---------------------------------------------------------------------------------------
 * Temporal graph (tiger/data/graph.py)
 * ------------------------------------------------------------------------------------- */

/* a1  Graph.__init__ / data2adjlist (graph.py:11-36,226-241): per-node time-sorted CSR from
 * a time-ordered stream (src,dst,ts,eid)[n_events].  Entry 2e belongs to src[e] (flag 0), 2e+1
 * to dst[e] (flag 1); per node, entries keep stream order - the stable sort of the reference.
 * Implemented as a stable LSD radix sort of the entry indices by owner id (deterministic).
 * `work` needs tiger_csr_build_work_bytes() bytes.  Output arrays have 2*n_events entries,
 * indptr n_nodes+1. */
int64_t tiger_csr_build_work_bytes(int64_t n_events, int64_t n_nodes);
int tiger_csr_build(const int64_t* src, const int64_t* dst, const double* ts, const int64_t* eid,
                    int64_t n_events, int64_t n_nodes, int64_t* indptr, int32_t* adj_nbr,
                    int32_t* adj_eid, double* adj_ts, uint8_t* adj_flag, void* work, void* stream);

/* a2  Graph.find_before + sample_temporal_neighbor['recent_edges'] + get_history
 * (graph.py:44-53,117-127,150-155).  Eight lanes per query (4 queries per warp), 8-ary cooperative search for the
 * strict-'<' cut, right-aligned zero-padded K most recent entries.
 * q_ts has ts_period entries, query i uses q_ts[i % ts_period] (np.tile of the collator).
 * out_dirs, out_ts32 and mark_bitmap may be NULL.  mark_bitmap (ceil(n_nodes/32) words)
 * receives one bit per query node and per returned neighbor (involved-node marking of
 * collate_memory_nodes, data_loader.py:109-121).  out_ts32 (ts_period floats) receives
 * (float)q_ts - the model-side timestamps of GraphCollator.__call__ (data_loader.py:92).
 * count (device, may be NULL) limits the queries to the first *count. */
int tiger_find_recent(const int64_t* indptr, const int32_t* adj_nbr, const int32_t* adj_eid,
                      const double* adj_ts, const uint8_t* adj_flag, const int64_t* q_nids,
                      const double* q_ts, int64_t n_query, int64_t ts_period, int k,
                      int64_t* out_nids, int64_t* out_eids, float* out_ts, int64_t* out_dirs,
                      float* out_ts32, uint32_t* mark_bitmap, const int32_t* count, void* stream);

/* tiger_find_recent over M chunks of the stream that share one CSR (ChunkSampler, data_loader.py:23-48: every DDP rank
 * keeps its own memory over its own contiguous slice; here the M slices run as one call).  Node u of chunk c has the
 * virtual id v = c * node_stride + u; q_nids hold virtual ids and each query reads the CSR segment of
 * u = v mod node_stride.  mark_bitmap (ceil(M * node_stride / 32) words) is marked with virtual ids.
 *   TIGER_FIND_CHUNK_NEIGHBORS  the neighbor tables of the batch nodes and the second hop
 *       (sample_temporal_neighbor, graph.py:117-127; data_loader.py:105-131): query i at q_ts[i % ts_period] as in
 *       tiger_find_recent, out_nids offset by c * node_stride except id 0: the padding stays 0 (the attention and the
 *       seq restarter key their masks on id 0; node 0 is the padding node, the reference's ids start at 1) and marks
 *       the chunk's own node 0, c * node_stride, as an unchunked call marks node 0.  A query with id 0 - the second
 *       hop of a padding slot, whose chunk the id does not tell - marks nothing (its chunk's node 0 is marked by the
 *       padding slot it comes from).
 *   TIGER_FIND_CHUNK_HISTORY    the seq restarter's get_history (graph.py:150-155) at each chunk's own restart time:
 *       query i at q_ts[v / node_stride] (M chunk times, tiger_min_time_ex), ts_period and out_ts32 unused, out_nids
 *       the real neighbor ids (restarters.py:80-87 masks the padding id 0).
 * mode 0 is tiger_find_recent. */
#define TIGER_FIND_CHUNK_NEIGHBORS 1
#define TIGER_FIND_CHUNK_HISTORY 2
int tiger_find_recent_ex(const int64_t* indptr, const int32_t* adj_nbr, const int32_t* adj_eid,
                         const double* adj_ts, const uint8_t* adj_flag, const int64_t* q_nids,
                         const double* q_ts, int64_t n_query, int64_t ts_period, int k,
                         int64_t* out_nids, int64_t* out_eids, float* out_ts, int64_t* out_dirs,
                         float* out_ts32, uint32_t* mark_bitmap, const int32_t* count,
                         int64_t node_stride, int mode, void* stream);

/* a4  GraphCollator.check_in_window (data_loader.py:61-67): hit[i,k] = (center[i]==neigh[i,k]). */
int tiger_hit_window(const int64_t* center, const int64_t* neigh, int64_t n, int k, float* hit,
                     void* stream);

/* mark ids in a node bitmap (first half of the sorted-unique of collate_memory_nodes). */
int tiger_mark_nodes(const int64_t* ids, int64_t n, uint32_t* bitmap, int64_t n_nodes, void* stream);

/* a3 + a5 + a12  second half: ordered compaction of the bitmap (cleared on exit) into
 *   involved[]      sorted unique involved ids                 (data_loader.py:121)
 *   local_index[u]  = rank of u in involved (may be NULL)       (data_classes.py:163-165)
 *   restart_nodes[] involved nodes not yet up to date; marks them up to date and drops
 *                   their pending-message flag (train_self_supervised.py:158-163,
 *                   tiger.py:603, memory.py:136).  uptodate==NULL disables this list.
 *   outdated[]      involved nodes with a pending message, ascending
 *                   (MessageStoreNoGradLastOnly.get_outdated_node_ids, memory.py:108-126)
 *   gru_row[u]      = rank of u in outdated, -1 for involved nodes without a message (may be NULL)
 * counts[0..2] = U, O, R.  Single CTA; cost O(n_nodes/32). */
int tiger_compact_involved(uint32_t* bitmap, int64_t n_nodes, uint8_t* has_msg, uint8_t* uptodate,
                           int64_t* involved, int64_t cap_involved, int64_t* local_index,
                           int64_t* outdated, int32_t* gru_row, int64_t* restart_nodes,
                           int32_t* counts, uint32_t* err_flags, void* stream);

/* The same compaction with read_only != 0, for a query that scores candidates against the state without advancing it:
 * the lists and counts are those of read_only == 0, but uptodate and has_msg are only read, and restarted node
 * restart_nodes[r] gets gru_row[u] = restart_base + r (r < cap_involved) instead of -1, so the attention reads its
 * restart surrogate from that row of its rows_b (tiger_static_restart_rows / the seq restarter's h_right).  Restart
 * nodes never have a pending message in the lists, so [0, O) and [restart_base, restart_base + R) do not overlap when
 * restart_base >= cap_involved.  tiger_compact_involved is this call with read_only = 0. */
int tiger_compact_involved_ex(uint32_t* bitmap, int64_t n_nodes, uint8_t* has_msg, uint8_t* uptodate,
                              int64_t* involved, int64_t cap_involved, int64_t* local_index,
                              int64_t* outdated, int32_t* gru_row, int64_t* restart_nodes,
                              int32_t* counts, uint32_t* err_flags, int read_only, int restart_base,
                              void* stream);

/* ---------------------------------------------------------------------------------------
 * Index utilities (tiger/model/utils.py)
 * ------------------------------------------------------------------------------------- */

/* a8  select_latest_nids (utils.py:10-16) with torch_scatter's CPU tie rule (lowest position
 * among the maxima).  ts_is_f64 selects float64 (collator) or float32 (model) timestamps;
 * position i uses ts[i % ts_period] (ts.repeat(2) of tiger.py:232,255; 0 means n).
 * slot_ts / slot_pos are caller-owned per-node scratch tables (n_nodes entries, all-zero on
 * entry, all-zero again on exit).  Outputs:
 *   winner[i]   1 when position i is its node's selected position      (n, may be NULL)
 *   unique_ids  ascending distinct ids, index[j] the selected position (may both be NULL)
 *   count       number of distinct ids (device)
 * Four stream-ordered kernels (max-ts atomics, min-pos atomics, flag, ordered compaction). */
int tiger_select_latest(const int64_t* nids, const void* ts, int ts_is_f64, int64_t n,
                        int64_t ts_period, int64_t n_nodes, uint64_t* slot_ts, uint32_t* slot_pos, uint32_t* bitmap,
                        uint8_t* winner, int64_t* unique_ids, int64_t* index, int32_t* count,
                        void* stream);

/* a22  anonymized_reindex (utils.py:19-27): per row rank by last occurrence, 0 stays 0.
 * count (device, may be NULL) limits the rows to the first *count. */
int tiger_anonymized_reindex(const int64_t* hist_nids, int64_t n, int len, int64_t* out,
                             const int32_t* count, void* stream);

/* ---------------------------------------------------------------------------------------
 * Memory / message store (tiger/model/memory.py, time_encoding.py)
 * ------------------------------------------------------------------------------------- */

/* a11 Memory.get (memory.py:36-39): out[i,:] = table[ids[i],:] (+ optional ts gather). */
int tiger_gather_rows(const float* table, int64_t width, const int64_t* ids, int64_t n, float* out,
                      const float* ts_table, float* out_ts, void* stream);

/* a11 Memory.set (memory.py:41-52): table[ids[i],:] = vals[i,:]; ts_table[ids[i]] = ts[i];
 * active[ids[i]] = 1.  With check!=0 sets TIGER_ERR_PAST_MEMORY when ts_table[id] > ts[i].
 * count (device) overrides n when non-NULL. */
int tiger_scatter_rows(float* table, int64_t width, const int64_t* ids, int64_t n,
                       const int32_t* count, const float* vals, float* ts_table, const float* ts,
                       uint8_t* active, int check, uint32_t* err_flags, void* stream);

/* a10 TimeEncode.forward (time_encoding.py:16-27): out[i,:] = cos(ts[i]*w + b), product and
 * sum rounded separately (no FMA contraction) like the CPU reference. */
int tiger_time_encode(const float* ts, int64_t n, const float* w, const float* b, int dim, float* out,
                      void* stream);

/* a9  TIGE.store_events + MessageStoreNoGradLastOnly.store_events (tiger.py:422-442,
 * memory.py:77-106).  For every selected position p (winner[p]!=0) of pos=[src;dst] builds
 *   [mem(self)+nf(self) | mem(other)+nf(other) | ef(eid) | cos((t - mem_ts(self))*w + b)]
 * and writes it to msg_vals[self], msg_ts[self]=t, has_msg[self]=1.  mem = message-source
 * memory (left or right).  nfeats / efeats may be NULL (zeros of width d / de). */
int tiger_store_messages(const int64_t* src, const int64_t* dst, const int64_t* eids, const float* ts,
                         int64_t batch, const uint8_t* winner, const float* mem_vals,
                         const float* mem_ts, const float* nfeats, const float* efeats, int d, int de,
                         const float* time_w, const float* time_b, float* msg_vals, float* msg_ts,
                         uint8_t* has_msg, uint32_t* err_flags, void* stream);

/* Same operator with the argument list of MessageStoreNoGradLastOnly.store_events (memory.py:77-81):
 * src_vals / dst_vals [batch, d] and src_prev_ts / dst_prev_ts [batch] are the copies Memory.get
 * returned for the events' endpoints. */
int tiger_store_messages_dense(const int64_t* src, const int64_t* dst, const int64_t* eids, const float* ts,
                               int64_t batch, const uint8_t* winner, const float* src_vals,
                               const float* dst_vals, const float* src_prev_ts, const float* dst_prev_ts,
                               const float* nfeats, const float* efeats, int d, int de, const float* time_w,
                               const float* time_b, float* msg_vals, float* msg_ts, uint8_t* has_msg,
                               uint32_t* err_flags, void* stream);

/* a17 TIGE.contrast_learning step 4 (tiger.py:230-241,396-406): for selected positions whose
 * node has a pending message: right_vals[u] = h_new[gru_row[u]], right_ts[u] = msg_ts[u],
 * has_msg[u] = 0.  a19: when hprev_left/right are non-NULL also copies left_vals[pos] (before
 * step 6) and right_vals[pos] (after step 4) - hprev_* are written by a second phase launched
 * after the write-back, so the pair of launches honours tiger.py:246-251. */
int tiger_right_writeback(const int64_t* pos_ids, int64_t n_pos, const uint8_t* winner,
                          const int32_t* gru_row, const float* h_new, int d, float* right_vals,
                          float* right_ts, uint8_t* right_active, const float* msg_ts,
                          uint8_t* has_msg, const float* left_vals, float* hprev_left,
                          float* hprev_right, uint32_t* err_flags, void* stream);

/* a18 TIGE.update_left_memory (tiger.py:408-420): left_vals[u] = h_left[p], left_ts[u] = ts[p]
 * for selected positions p (ts indexed modulo batch). */
int tiger_left_writeback(const int64_t* pos_ids, int64_t n_pos, int64_t batch, const uint8_t* winner,
                         const float* h_left, int d, const float* ts, float* left_vals, float* left_ts,
                         uint8_t* left_active, uint32_t* err_flags, void* stream);

/* ---------------------------------------------------------------------------------------
 * Dense operators
 * ------------------------------------------------------------------------------------- */

/* Gate-weight pack of nn.GRUCell for tiger_gru_update: weight_ih [3d][M] and weight_hh [3d][d] (as stored)
 * split into tf32 head / tail planes and laid out as the shared-memory image of every pipeline stage
 * (csrc/gru.cu).  Re-run whenever the weights change. */
int64_t tiger_gru_pack_bytes(int m_dim, int d);
int tiger_gru_pack(const float* w_ih, const float* w_hh, int m_dim, int d, float* out, void* stream);

/* a6 + a13  LastMessageAggregatorNoGradLastOnly.forward gather + GRUUpdater.forward
 * (message_modules.py:150-160, update_modules.py:30-37 = nn.GRUCell, gates r,z,n):
 *   h_new[r,:] = GRUCell(x = msg rows, h = state rows)
 * node_ids==NULL: x/h are dense [n,M]/[n,d]; otherwise row r reads x_table[node_ids[r]] and
 * h_table[node_ids[r]].  count (device, may be NULL) overrides n_rows (n_rows stays the grid
 * bound).  wpack: tiger_gru_pack output; b_ih, b_hh [3d] as stored.  The gate GEMMs run on the
 * tensor cores in tf32x3 (fp32-accurate).  Also checks the message invariants of tiger.py:319-327
 * when check_mem_ts != NULL. */
int tiger_gru_update(const int64_t* node_ids, const int32_t* count, int64_t n_rows,
                     const float* x_table, int64_t x_stride, const float* h_table, int64_t h_stride,
                     int m_dim, int d, const float* wpack,
                     const float* b_ih, const float* b_hh, float* h_new,
                     const float* msg_ts, const float* check_mem_ts, int check_equal,
                     uint32_t* err_flags, void* stream);

/* tiger_gru_update for MLPMessageFunction (message_modules.py:47-57, an MLP transform between the last-message
 * gather and the GRUCell; reference message_modules.py:29-55): x row r is x_table[r] (row position, the hidden
 * rows relu(W_1 msg + b_1) that a plain-row tiger_sgemm_nt_packed_gather wrote for the outdated rows) while h,
 * msg_ts and the invariant checks read node_ids[r] (not NULL).  m_dim is the hidden width; the pack and b_ih are
 * those of weight_ih W_2 and bias_ih + weight_ih b_2 (the second layer folded into the gates). */
int tiger_gru_update_rows(const int64_t* node_ids, const int32_t* count, int64_t n_rows,
                          const float* x_table, int64_t x_stride, const float* h_table, int64_t h_stride,
                          int m_dim, int d, const float* wpack,
                          const float* b_ih, const float* b_hh, float* h_new,
                          const float* msg_ts, const float* check_mem_ts, int check_equal,
                          uint32_t* err_flags, void* stream);

/* First layer of MergeUpdater (update_modules.py:40-47: MergeLayer(msg_dim, d, d, d), basic_modules.py:8-20):
 *   out[r,:] = relu(fc1 [x ; h] + b1)      fc1 [d][m_dim + d] as stored (message columns first)
 * on the tensor cores of tiger_gru_update (tf32x3), with its row gather (x by node id, or by row position with
 * x_by_row), its device row count and its message-invariant checks (tiger.py:319-327).  fc2 follows as a
 * count-bounded tiger_sgemm_nt_packed.  wpack: tiger_merge_pack output, tiger_gru_pack_bytes(m_dim, d) bytes;
 * re-run it whenever fc1 changes.  A linear / MLP message transform folds into the message columns of fc1. */
int tiger_merge_pack(const float* fc1_w, int m_dim, int d, float* out, void* stream);
int tiger_merge_update(const int64_t* node_ids, const int32_t* count, int64_t n_rows,
                       const float* x_table, int64_t x_stride, int x_by_row, const float* h_table,
                       int64_t h_stride, int m_dim, int d, const float* wpack, const float* b1, float* out,
                       const float* msg_ts, const float* check_mem_ts, int check_equal,
                       uint32_t* err_flags, void* stream);

/* temporal-attention parameters (device pointers): the reference's tensors as stored
 * (temporal_embedding_fn.fns.0.*), plus one caller-allocated buffer for the folded weights.
 * E = 2d, C = 2d + de, hd = E / n_head. */
/* Fusion of update_left_memory (tiger.py:408-420, tiger_left_writeback below) into the last product of
 * tiger_temporal_attention_ex: the rows p < n_pos of the result whose winner[p] != 0 are also written to
 * left_vals[pos_ids[p]], with left_ts[...] = ts[p % batch] (error flag if the stored clock is later) and
 * left_active[...] = 1 - the embeddings are persisted by the kernel that produces them.  ready_event (a
 * cudaEvent_t, may be NULL) is waited for on the stream in front of that product: it must cover the producer of
 * `winner` and every reader of the old left-memory rows (the message builder). */
typedef struct {
  const int64_t* pos_ids;
  const uint8_t* winner;
  int64_t n_pos;
  const float* ts;
  int64_t batch;
  float* left_vals;       /* [N][d] */
  float* left_ts;         /* [N] */
  uint8_t* left_active;   /* [N] or NULL */
  uint32_t* err_flags;    /* or NULL */
  void* ready_event;
} tiger_left_writeback_fused;

typedef struct {
  const float* wq;       /* [E][E]    mha_fn.q_proj_weight                                  */
  const float* wk;       /* [E][C]    mha_fn.k_proj_weight                                  */
  const float* wv;       /* [E][C]    mha_fn.v_proj_weight                                  */
  const float* wo;       /* [E][E]    mha_fn.out_proj.weight                                */
  const float* fc1;      /* [d][E+d]  merger.fc1.weight                                     */
  const float* fc2;      /* [d][d]    merger.fc2.weight                                     */
  const float* in_bias;  /* [3E] in_proj_bias (q,k,v)                                       */
  const float* out_bias; /* [E]                                                             */
  const float* fc1_b;    /* [d]                                                             */
  const float* fc2_b;    /* [d]                                                             */
  const float* time_w;   /* [d] time_encoder.basis_freq                                     */
  const float* time_b;   /* [d] time_encoder.phase                                          */
  float* folded;         /* tiger_attn_fold_bytes() bytes, 16-byte aligned, filled by tiger_attn_fold */
  /* The fused last product of the batch-node depth: either all three of the following are set, and only for
   * tiger_temporal_attention_ex, or all three are NULL (TIGER_EINVAL otherwise). */
  float* score_folded;   /* tiger_score_fold blob - the last GEMM then also emits the scorer terms              */
  float* pq_out;         /* per-call output [n_query][2d]: P = W1a z | Q = W1b z                               */
  const tiger_left_writeback_fused* left_wb;   /* see above                                                   */
} tiger_attn_params;

/* Folds the projections that are linear in the per-query vectors (exact by linearity, accumulated in
 * double; see csrc/attention.cu):  Wqk_h = scale [Wk_h | bk_h]^T Wq_h,  bqk_h = scale [Wk_h | bk_h]^T bq_h,
 * W2f = [W1a Wo_h Wv_h .. | W1b | W1a (Wo bv + bo)].  Re-run whenever one of the tensors above changes. */
int64_t tiger_attn_fold_bytes(int d, int de, int n_head);
int tiger_attn_fold(const tiger_attn_params* params, int d, int de, int n_head, void* stream);

/* Link-scorer fold (tiger.py:259-288): the scorer's first layer is linear in the two embeddings, and the
 * embeddings are the output of the merger's last layer, so that layer's GEMM can also emit P = W1a z and
 * Q = W1b z (split output); scoring a pair is then relu(P[s] + Q[t] + c_ab) . w2 + b2 (tiger_link_score_folded).
 * score_fc1 [d][2d], score_fc1_b [d]: score_fn.fc1.*; merger_fc2 [d][d], merger_fc2_b: the embedding
 * module's merger.fc2.*; hit_emb [2][d] or NULL (hit_type 'none').  blob: tiger_score_fold_bytes(d) bytes. */
int64_t tiger_score_fold_bytes(int d);
int64_t tiger_score_fold_cab_offset(int d);   /* float offset of the c_ab table [4][d] inside the blob */
int tiger_score_fold(const float* score_fc1, const float* score_fc1_b, const float* merger_fc2,
                     const float* merger_fc2_b, const float* hit_emb, int d, float* blob, void* stream);

/* the scorer's hit types (--hit_type, tiger.py:129-136,259-288) */
#define TIGER_HIT_NONE 0
#define TIGER_HIT_BIN 1
#define TIGER_HIT_VEC 2
#define TIGER_HIT_COUNT 3

/* The same fold for every hit type, with K = n_neighbors (ignored for 'bin' / 'none', whose blob is exactly
 * tiger_score_fold's).  The head of the blob (W3, b3, c_ab, pack) keeps its layout; 'count' and 'vec' append
 * their hit tables behind it (c_ab stays zero):
 *   count: hit_emb [K+1][d]; tables U [K+1][d] | V [K+1][d], U[c] = b1 + W1a he_c, V[c] = W1b he_c.
 *   vec  : hit_emb NULL, score_fc1 [d][2(d+K)] = [W1a | Ha | W1b | Hb] (score_fn = MergeLayer(d+K, d+K, d, 1));
 *          tables b1 [d] | Ha^T [K][d] | Hb^T [K][d].
 * hit_emb [2][d] for 'bin', NULL for 'none'.  -1 / TIGER_EINVAL for an unknown hit type or K <= 0 ('vec',
 * 'count'). */
int64_t tiger_score_fold_hit_bytes(int d, int hit_type, int k);
int64_t tiger_score_fold_hit_offset(int d, int hit_type, int k);   /* float offset of the scorer's table:
                                                                      c_ab ('bin', 'none') or the hit tables */
int tiger_score_fold_hit(const float* score_fc1, const float* score_fc1_b, const float* merger_fc2,
                         const float* merger_fc2_b, const float* hit_emb, int d, int hit_type, int k, float* blob,
                         void* stream);

/* bytes of caller-provided, 16-byte aligned workspace for n_query queries; -1 for dimensions both attention entry
 * points refuse: k > 64, n_head > 8, or a score-pool shared-memory footprint
 * 4 (k ru4(2d + de) + ru4(n_head k) + n_head ru4(2d + de + 1)) bytes over 200 KiB (ru4: rounded up to a multiple
 * of 4) */
int64_t tiger_temporal_attention_work_bytes(int64_t n_query, int k, int d, int de, int n_head);

/* a15 + a16  one layer of GraphEmbedding.compute_embedding_with_computation_graph +
 * TemporalAttention.forward (temporal_agg_modules.py:29-83,210-235), eval mode: gather (center + K
 * neighbors + edge rows) -> time encoding -> folded single-query attention (score weights through
 * Wqk, masked softmax, pooled keys) -> folded value / out projection + merger MLP on the tensor
 * cores, as the launch sequence described in csrc/attention.cu.
 * Node representations: row(u) = sel[u] >= 0 ? rows_b[sel[u]] : rows_a[u]
 *   fused routes : rows_a = right memory, rows_b = GRU output, sel = gru_row
 *   class surface: rows_a = NULL, rows_b = involved_node_reprs, sel = local_index
 * sel is int32 when sel_is_i64==0, int64 otherwise.  out [n_query, d].  Any depth of a multi-layer embedding
 * (one layer: ts_group = 1, key_rows = NULL):
 *   query q reads q_ts[(q / ts_group) % ts_period]: the depth-1 queries of n_layers = 2 are the K neighbors
 *     of each of the 3B batch nodes at the parent event's time, ts_group = K, ts_period = B
 *     (repeat_interleave(ts.repeat(3), K)).
 *   key_rows [n_query * K][d] (NULL: the rows above): slot (q, j) takes its node representation from
 *     key_rows[q * K + j] with no node features added - the lower layer's output for the depth-2 queries.
 *     Padding slots (neigh_nids == 0) stay masked.  key_rows is gathered before the kernel's programmatic
 *     dependency wait, so its producer must be the previous launch sequence on the same stream. */
int tiger_temporal_attention_ex(const int64_t* center_nids, const float* q_ts, int64_t n_query,
                                int64_t ts_period, int64_t ts_group, const int64_t* neigh_nids,
                                const int64_t* neigh_eids, const float* neigh_ts, int k, const float* rows_a,
                                const float* rows_b, const float* key_rows, const void* sel, int sel_is_i64,
                                const float* nfeats, const float* efeats, int d, int de, int n_head,
                                const tiger_attn_params* params, float* out, void* work, void* stream);

/* tiger_temporal_attention_ex for the batch-node depth of a read-only candidate query: params carries score_folded and
 * pq_out and no left_wb (TIGER_EINVAL otherwise); the last product writes out and pq_out exactly as the fused route of
 * tiger_temporal_attention_ex does and persists nothing. */
int tiger_temporal_attention_query(const int64_t* center_nids, const float* q_ts, int64_t n_query,
                                   int64_t ts_period, int64_t ts_group, const int64_t* neigh_nids,
                                   const int64_t* neigh_eids, const float* neigh_ts, int k, const float* rows_a,
                                   const float* rows_b, const float* key_rows, const void* sel, int sel_is_i64,
                                   const float* nfeats, const float* efeats, int d, int de, int n_head,
                                   const tiger_attn_params* params, float* out, void* work, void* stream);

/* Same operator with the dense argument list of TemporalAttention.forward
 * (temporal_agg_modules.py:210-235): qx [n,d], qt [n,d], kx [n,K,d], ky [n,K,de], kt [n,K,d],
 * padding_mask [n,K] (1 = padding). */
int tiger_temporal_attention_dense(const float* qx, const float* qt, const float* kx, const float* ky,
                                   const float* kt, const uint8_t* padding_mask, int64_t n_query, int k,
                                   int d, int de, int n_head, const tiger_attn_params* params, float* out,
                                   void* work, void* stream);

/* step 7 of TIGE.contrast_learning (tiger.py:259-288), hit_type 'bin' or 'none': hit flags from the neighbor table
 * [3B][K], hit embedding, score_fn MergeLayer on positive / negative pairs, BCE-with-logits mean; scores [2B] = pos
 * then neg.  Folded form (see tiger_score_fold): pq [3B][2d] = [W1a z | W1b z] rows of [src ; dst ; neg]
 * from tiger_temporal_attention_ex, cab = blob + tiger_score_fold_cab_offset(d); neigh_nids NULL = hit_type 'none'. */
int tiger_link_score_folded(const float* pq, int64_t batch, int d, const int64_t* src, const int64_t* dst,
                            const int64_t* neg, const int64_t* neigh_nids, int k, const float* cab,
                            const float* fc2_w, const float* fc2_b, float* scores, float* loss,
                            uint32_t* done_counter, void* stream);

/* The same scorer for every hit type (TIGER_HIT_*); tables = blob + tiger_score_fold_hit_offset(d, hit_type, k).
 * With the hit flags a_j = [N(t)[j] == s], b_j = [N(s)[j] == t] of a pair (s, t) over the K slots of the
 * neighbor table, the first layer is P[s] + Q[t] plus
 *   bin  : c_ab[2 any(a) + any(b)]          count: U[sum a] + V[sum b]
 *   none : c_ab[0] (neigh_nids ignored)     vec  : b1 + sum_{a_j} Ha^T[j] + sum_{b_j} Hb^T[j]
 * One launch per batch, any K >= 1 (neigh_nids required except for 'none'). */
int tiger_link_score_folded_hit(const float* pq, int64_t batch, int d, const int64_t* src, const int64_t* dst,
                                const int64_t* neg, const int64_t* neigh_nids, int k, int hit_type,
                                const float* tables, const float* fc2_w, const float* fc2_b, float* scores,
                                float* loss, uint32_t* done_counter, void* stream);

/* The scorer over C >= 1 candidate columns (tiger_link_score_folded_hit is this call with C = 2, pos = dst, negs = neg,
 * ranks = NULL): pair (i, j), i < n_query, scores src[i] against column j's node - pos[i] for j = 0, negs[(j-1) n_query
 * + i] for j >= 1 - from pq rows i and n_query + j n_query + i, i.e. pq and neigh_nids hold the rows of
 * [src | column 0 | column 1 | ...].  scores [C][n_query] (candidate-major).  loss (may be NULL) is the BCE mean over
 * the C n_query pairs with column 0 as the positive.  ranks (may be NULL) [n_query]:
 * 1 + #{j >= 1 : s_ij > s_i0} + 0.5 #{j >= 1 : s_ij == s_i0}, column 0 the true candidate, ties counted half (the
 * mean of the optimistic and the pessimistic rank), from integer counts (deterministic); a NaN s_i0 gives a NaN rank,
 * a NaN s_ij neither beats nor ties s_i0, infinities compare as values.  One more launch when ranks are wanted. */
int tiger_link_score_cands(const float* pq, int64_t n_query, int n_cands, int d, const int64_t* src,
                           const int64_t* pos, const int64_t* negs, const int64_t* neigh_nids, int k, int hit_type,
                           const float* tables, const float* fc2_w, const float* fc2_b, float* scores, float* ranks,
                           float* loss, uint32_t* done_counter, void* stream);

/* ---------------------------------------------------------------------------------------
 * Restarters (tiger/model/restarters.py, tiger.py:594-609)
 * ------------------------------------------------------------------------------------- */

/* a23 + a24  StaticRestarter.forward + TIGER.restart: for each listed node u:
 *   prev_ts = time of the last event of u strictly before t (0 if none), t = min(batch_ts) when
 *   batch_ts != NULL (restart() is called with ts.min(), train_self_supervised.py:161), else
 *   q_ts[i];  left_vals[u]=left_emb[u], right_vals[u]=right_emb[u], both update_ts = prev_ts,
 *   has_msg[u] = 0.  out_prev_ts (may be NULL) receives prev_ts per listed node. */
int tiger_static_restart(const int64_t* nids, const int32_t* count, int64_t n,
                         const float* batch_ts, int64_t batch, const double* q_ts,
                         const int64_t* indptr, const double* adj_ts, const float* left_emb,
                         const float* right_emb, int d, float* left_vals, float* left_ts,
                         uint8_t* left_active, float* right_vals, float* right_ts,
                         uint8_t* right_active, uint8_t* has_msg, float* out_prev_ts, void* stream);

/* tiger_static_restart in chunk mode (node_stride > 0; virtual ids v = c * node_stride + u as in
 * tiger_find_recent_ex): restart node v of chunk c cuts its history at chunk_ts[c] (the float32 minimum of that
 * chunk's batch times, tiger_min_time_ex: TIGER.restart, tiger.py:594-609, receives the ts.min() of its own rank's
 * batch) and reads its CSR segment and its left_emb / right_emb rows at u (StaticRestarter.forward,
 * restarters.py:254-277); the memories, clocks, flags and has_msg are written at v.  batch_ts and q_ts are unused.
 * node_stride == 0 is tiger_static_restart (chunk_ts unused). */
int tiger_static_restart_ex(const int64_t* nids, const int32_t* count, int64_t n,
                            const float* batch_ts, int64_t batch, const double* q_ts,
                            const int64_t* indptr, const double* adj_ts, const float* left_emb,
                            const float* right_emb, int d, float* left_vals, float* left_ts,
                            uint8_t* left_active, float* right_vals, float* right_ts,
                            uint8_t* right_active, uint8_t* has_msg, float* out_prev_ts,
                            int64_t node_stride, const double* chunk_ts, void* stream);

/* Restart surrogates of a read-only query: out_rows[i] = right_emb[nids[i]] (the right-memory row
 * tiger_static_restart writes) for i < min(*count, n) (count may be NULL); writes nothing node-indexed. */
int tiger_static_restart_rows(const int64_t* nids, const int32_t* count, int64_t n, const float* right_emb, int d,
                              float* out_rows, void* stream);

/* a21 + a24  SeqRestarter.forward (restarters.py:51-114) as a launch sequence; see restart_seq.cu.
 *
 * tiger_min_time: out[0] = (double)min(ts[0..n)) - the float32 ts.min() that restart() receives
 * (train_self_supervised.py:161, eval_utils.py:40), widened for the float64 history search. */
int tiger_min_time(const float* ts, int64_t n, double* out, void* stream);

/* out[c] = (double)min(ts[c*n .. (c+1)*n)) for c < n_chunks: the restart time of each chunk of a chunked batch
 * (chunk-major ts, tiger_find_recent_ex), each chunk's own ts.min() as its DDP rank would compute it
 * (train_self_supervised.py:161).  n_chunks == 1 is tiger_min_time. */
int tiger_min_time_ex(const float* ts, int64_t n_chunks, int64_t n, double* out, void* stream);

/* Event tokens of SeqRestarter.forward (restarters.py:85-104): for node i and history position j
 *   x[i,j,:] = [nf(src) | nf(dst) | anony_emb[anony_ids] | ef(hist_eids) | cos((t_last - hist_ts)*w + b)]
 * (width d_model = 4d + de) with the reference's literal direction rule (:93-94); the last
 * position keeps only its time code (:104).  mask[i,j] = hist_nids==0 with the last column forced
 * valid (:86-87); prev_ts[i] = hist_ts[i,-1].  count (device, may be NULL) overrides n. */
int tiger_seq_tokens(const int64_t* nids, const int32_t* count, int64_t n, int len,
                     const int64_t* hist_nids, const int64_t* hist_eids, const float* hist_ts,
                     const int64_t* hist_dirs, const int64_t* anony_ids, const float* nfeats,
                     const float* efeats, int d, int de, const float* anony_emb, const float* time_w,
                     const float* time_b, float* x, uint8_t* mask, float* prev_ts, void* stream);

/* Small-R tail of SeqRestarter.forward (restarters.py:106-114 after the attention): value projection of the pooled
 * tokens per head, out-projection + ReLU, out_fn, merger (fc1 on its first d input columns + ReLU, fc2) as five
 * matrix-vector layers (one warp per output channel; att [n, d_model], o [n, d_model], hid [n, d] are the intermediate
 * rows).  Training-mode forward (tiger_train_seq_pool with dropout): psum [n, n_head] scales the value bias, p_drop /
 * seed drop the merger's hidden layer exactly like tiger_train_dropout(stream 4); NULL / 0 for inference.
 * Rows: min(n, *count); the caller passes the count gated by
 * tiger_seq_gate_count (count_small = count if count <= max_rows else 0, count_big = the complement), so that few rows
 * take this kernel and many rows the tensor-core products. */
int tiger_seq_gate_count(const int32_t* count, int max_rows, int32_t* count_small, int32_t* count_big, void* stream);
int tiger_seq_tail(const float* xbar, const int32_t* count, int64_t n, int d_model, int n_head, int d, const float* w_v,
                   const float* b_v, const float* w_out, const float* b_out, const float* w_fn, const float* b_fn,
                   const float* w_fc1, int64_t ld_fc1, const float* b_fc1, const float* w_fc2, const float* b_fc2,
                   const float* psum, float p_drop, int seed, float* att, float* o, float* hid, float* h_left,
                   float* h_right, void* stream);

/* Dense products on the tensor cores (csrc/gemm.cu: tcgen05, tf32 head / tail split, fp32-accurate).  Two kernels:
 * tiger_sgemm_nt and tiger_sgemm_ex stage both operands through shared memory; the tiger_sgemm_nt_packed* family
 * takes the weight as a pre-split pack (tiger_gemm_pack_weight) streamed by TMA.
 *
 * C[m,n] = act(sum_k A[m,k] * W[n,k] + bias[n]) on row-major A [M,K] and nn.Linear style weights W [N,K] (bias may
 * be NULL; relu != 0 applies max(.,0)); tiger_sgemm_ex with trans 0 / 0, alpha 1 and no accumulation.  The row count
 * is min(m_rows, *count * rows_per_count) when count (device) is non-NULL.  Replaces the in/out projections of
 * nn.MultiheadAttention, nn.Linear and MergeLayer on the restarter path (restarters.py:45-50,106-111;
 * basic_modules.py:16-19). */
int tiger_sgemm_nt(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, float* C,
                   int64_t ldc, int64_t m_rows, const int32_t* count, int64_t rows_per_count, int n_cols,
                   int k_dim, int relu, void* stream);

/* General product for the training step (the same staging kernel):
 *   C[m,n] (+)= act(alpha * (sum_k opA[m,k] * opW[n,k] + bias[n]))
 * opA[m,k] = A[m*lda + k] (trans_a = 0) or A[k*lda + m] (trans_a = 1), opW likewise, so that the three products of
 * a linear layer use the tensors as stored: y = x W^T (0,0), dx = dy W (0,1), dW = dy^T x (1,1) - what autograd
 * runs for nn.Linear / nn.GRUCell / nn.MultiheadAttention under loss.backward() (train_self_supervised.py:169).
 * accumulate != 0 adds the tile into C with atomic adds (the gradient of a parameter with several uses; bias and
 * relu must be off) and splits K over k_parts CTAs per tile.  m_count / k_count (device, may be NULL) bound the
 * row count / the reduction length by *count * rows_per_count. */
int tiger_sgemm_ex(const float* A, int64_t lda, int trans_a, const float* W, int64_t ldw, int trans_w,
                   const float* bias, float* C, int64_t ldc, int64_t m_rows, int n_cols, int64_t k_dim,
                   const int32_t* m_count, const int32_t* k_count, int64_t rows_per_count, float alpha, int relu,
                   int accumulate, int k_parts, void* stream);

/* Pre-split weight packs for the tensor-core GEMM: W [n_rows][k_dim] (row stride ldw) -> tf32 head / tail
 * planes in the shared-memory image of each (column tile of bn rows, k-block) stage, so the kernel loads
 * a stage of W with one TMA bulk copy.  row_map (device int32 [n_tiles*bn], may be NULL) selects the
 * source row of every tile row (-1 = zeros).  bn: multiple of 16, <= 64 (tiger_gemm_pick_bn proposes
 * one for an expected row count). */
int tiger_gemm_pick_bn(int64_t m_rows, int n_cols, int batch);
int64_t tiger_gemm_pack_bytes(int n_tiles, int k_dim, int bn);
int tiger_gemm_pack_weight(const float* W, int64_t ldw, const int32_t* row_map, int n_rows, int k_dim, int bn,
                           int n_tiles, float* out, void* stream);
/* C = act(alpha * (A Wpack^T + bias)) with a pack of ceil(n_cols / bn) tiles */
int tiger_sgemm_nt_packed(const float* A, int64_t lda, const float* wpack, int bn, const float* bias, float* C,
                          int64_t ldc, int64_t m_rows, const int32_t* count, int64_t rows_per_count, int n_cols,
                          int k_dim, float alpha, int relu, void* stream);

/* Same with a gathered A operand: row m of A is row sel[ids[m]] of rows_b when that index is >= 0 (or rows_a
 * is NULL), else row ids[m] of rows_a, plus row ids[m] of add_rows when given - the "latest representation of
 * node u" lookup of compute_embedding_with_computation_graph (temporal_agg_modules.py:210-235: memory row or
 * the row the GRU just produced, + node features) done by the GEMM's producer warps.  sel is int32 or int64
 * (sel_is_i64); all three tables have row stride ld_rows.  sel == NULL: row m is row ids[m] of rows_a (rows_b
 * unused) - the outdated nodes' pending messages for the first layer of MLPMessageFunction (message_modules.py:47-57). */
int tiger_sgemm_nt_packed_gather(const int64_t* ids, const void* sel, int sel_is_i64, const float* rows_a,
                                 const float* rows_b, int64_t ld_rows, const float* add_rows, const float* wpack,
                                 int bn, const float* bias, float* C, int64_t ldc, int64_t m_rows,
                                 const int32_t* count, int64_t rows_per_count, int n_cols, int k_dim, float alpha,
                                 int relu, void* stream);

/* tiger_sgemm_nt_packed with the fused row scatter described at tiger_left_writeback_fused: result rows are
 * additionally stored into a node-indexed table (wb may be NULL when C2 is given: the split output alone).  With C2
 * (may be NULL) the output is split: the pack has
 * ceil((n_split + n_cols1) / bn) tiles; result columns [0, n_cols0) go to C, columns [n_split, n_split + n_cols1) to
 * C2 (n_split a multiple of 16 >= n_cols0; bias is indexed in the padded column space). */
int tiger_sgemm_nt_packed_scatter(const float* A, int64_t lda, const float* wpack, int bn, const float* bias, float* C,
                                  int64_t ldc, int n_cols0, float* C2, int64_t ldc2, int n_split, int n_cols1,
                                  int64_t m_rows, int k_dim, const tiger_left_writeback_fused* wb, void* stream);

/* Split-K for long reductions with few output tiles, the reduction inside the launch: the k_parts (<= 8; fewer
 * when K has fewer 32-float blocks) CTAs of an output tile form a thread-block cluster, exchange their partial
 * tiles through distributed shared memory, sum them in part order (deterministic) and write
 * act(alpha * (A W^T + bias)) once. */
int tiger_sgemm_nt_packed_splitk_fused(const float* A, int64_t lda, const float* wpack, int bn, const float* bias,
                                       float* C, int64_t ldc, int k_parts, int64_t m_rows, const int32_t* count,
                                       int64_t rows_per_count, int n_cols, int k_dim, float alpha, int relu,
                                       void* stream);

/* ------------------------------------------------------------------------------------------
 * Host-side batch pipeline (csrc/pipe.cu; no device code).  Replaces the synchronous per-batch `.to(device)` /
 * `.item()` traffic of the reference's loop (train_self_supervised.py:140-175): per staging slot a captured
 * finder graph and a captured model graph; tiger_pipe_submit uploads the batch and replays the finder on a
 * copy-in stream (beside the previous batch's model kernels), replays the model graph on main_stream (batch
 * order = call order) and downloads the results on a copy-out stream.  Capture: tiger_pipe_capture_begin(stream),
 * launch the kernels on that stream, tiger_pipe_capture_end(pipe, stream, slot, kind) with kind 0 = finder,
 * 1 = model, 2 = tail (optional: result-only kernels such as the link scorer, replayed on the copy-out stream in
 * front of the download, beside the next batch's model kernels).  src may be pinned host or device memory.
 * tiger_pipe_join makes a stream wait for the copy-out stream's work of the latest submit. */
void* tiger_pipe_create(int n_slots);
void tiger_pipe_destroy(void* pipe);
int tiger_pipe_capture_begin(void* stream);
int tiger_pipe_capture_end(void* pipe, void* stream, int slot, int kind);
int tiger_pipe_submit(void* pipe, int slot, const void* src, void* d_in, int64_t in_bytes, const void* d_out, void* h_out,
                      int64_t out_bytes, void* main_stream);
int tiger_pipe_wait(void* pipe, int slot, int host_results);
int tiger_pipe_join(void* pipe, void* stream);


/* ---------------------------------------------------------------------------------------------------------
 * Training step (csrc/train.cu): forward pieces that keep what backward needs and the hand-written backward of
 * TIGER.contrast_and_mutual_learning (tiger/model/tiger.py:547-592) - what loss.backward() / optimizer.step() of
 * train_self_supervised.py:165-171 and train_self_supervised_ddp.py:203-208 run through autograd.  Dense products
 * go through tiger_sgemm_ex; gradients accumulate into caller-owned buffers that tiger_train_adam zeroes.
 *   gather_pending / gru_gates[_bwd]   compute_messages + GRUUpdater (tiger.py:292-356, update_modules.py:30-37)
 *   attn_build[_bwd]_ex / attn_core[_bwd]   compute_embedding_with_computation_graph + TemporalAttention with
 *                                      dropout (temporal_agg_modules.py:29-104,210-235), either depth of n_layers = 2,
 *                                      TimeEncode gradients
 *   score_build[_bwd] / score_head[_bwd] hit embedding + score_fn + BCE (tiger.py:259-288)
 *   mse                                 mutual loss over valid rows (tiger.py:583-590)
 *   colsum / relu_bwd / zero_rows / scatter_add_rows   bias gradients, ReLU, masked rows, nn.Embedding gradients
 *   adam                                torch.optim.Adam defaults (train_self_supervised.py:116) on a flat buffer
 * --------------------------------------------------------------------------------------------------------- */
int tiger_train_gather_pending(const int64_t* ids, const int32_t* count, int64_t cap, const float* msg_vals, int m_dim, const float* msg_ts, const float* upd_vals, int d, const float* check_mem_ts, int check_equal, float* X, float* H, float* dh_zero, uint32_t* err_flags, float* n_rows_out, void* stream);
int tiger_train_gru_gates(const float* Gi, const float* Gh, const float* H, const int32_t* count, int64_t cap, int d, float* h_new, float* r_out, float* z_out, float* n_out, void* stream);
int tiger_train_gru_gates_bwd(const float* dh, const float* r_in, const float* z_in, const float* n_in, const float* Gh, const float* H, const int32_t* count, int64_t cap, int d, float* dGi, float* dGh, void* stream);
/* attn_build[_bwd]_ex: the builders for either depth of n_layers = 2 (one layer: ts_group = 1 and key_rows / d_key_rows
 * = NULL), the training twins of tiger_temporal_attention_ex:
 *   query i's time is ts[(i / ts_group) % batch] (depth 1: ts_group = K, repeat_interleave(ts.repeat(3), K));
 *   key_rows [n_q * K][d] (NULL: the rows above): slot r takes key_rows[r] as its node part, no node features added
 *     (depth 2: the depth-1 output);
 *   d_key_rows [n_q * K][d] (NULL: onto dh_new through sel): the slots' node-part gradients are STORED there, zeros
 *     for padding slots (neigh_nids == 0).  Query / merger-input gradients still go onto dh_new, and both kinds of
 *     time code accumulate into the TimeEncode gradients. */
int tiger_train_attn_build_ex(const int64_t* center, int64_t n_q, const float* ts, int64_t batch, int64_t ts_group, const int64_t* neigh_nids, const int64_t* neigh_eids, const float* neigh_ts, int k, const float* rows_a, const float* rows_b, const float* key_rows, const int32_t* sel, const float* nfeats, const float* efeats, int d, int de, const float* time_w, const float* time_b, float* q_in, float* kv_in, float* cat, int64_t ld_cat, int cat_off, void* stream);
int tiger_train_attn_core(const float* Q, int64_t ldq, const float* Kp, const float* Vp, int64_t ldkv, const int64_t* neigh_nids, int64_t n_q, int k, int n_head, int head_dim, float p_drop, int seed, float* attn, int64_t ld_attn, float* P, uint32_t* keep_bits, uint8_t* empty, void* stream);
int tiger_train_attn_core_bwd(const float* dattn, int64_t ld_attn, const float* Q, int64_t ldq, const float* Kp, const float* Vp, int64_t ldkv, const float* P, const uint32_t* keep_bits, int64_t n_q, int k, int n_head, int head_dim, float p_drop, float* dQ, float* dKp, float* dVp, void* stream);
int tiger_train_attn_build_bwd_ex(const float* dkv_in, const float* dq_in, const float* dcat, int64_t ld_cat, int cat_off, const int64_t* center, int64_t n_q, const float* ts, int64_t batch, int64_t ts_group, const int64_t* neigh_nids, const float* neigh_ts, int k, const int32_t* sel, int d, int de, const float* time_w, const float* time_b, float* dh_new, float* d_key_rows, float* g_time_w, float* g_time_b, void* stream);
int tiger_train_zero_rows(float* buf, int64_t ld, int cols, int64_t n_rows, const uint8_t* flag, void* stream);
int tiger_train_relu_bwd(float* dy, int64_t ld_dy, const float* y, int64_t ld_y, int cols, int64_t n_rows, const int32_t* count, int64_t rows_per_count, float scale, void* stream);
int tiger_train_colsum(const float* X, int64_t ld, int64_t n_rows, const int32_t* count, int64_t rows_per_count, int cols, float scale, float* out, void* stream);
int tiger_train_scatter_add_rows(float* table, const int64_t* ids, int64_t n, const int32_t* count, int64_t rows_per_count, const float* src, int64_t ld_src, int width, float scale, void* stream);
int tiger_train_score_build(const float* z, const float* hits, const int64_t* neigh_nids, const int64_t* batch_nids, int k, const float* hit_emb, int64_t batch, int d, float* pair, uint8_t* codes, void* stream);
int tiger_train_score_head(float* hid, const float* fc2_w, const float* fc2_b, int64_t batch, int d, float p_drop, int seed, float* scores, float* loss, float* dscore, void* stream);
int tiger_train_score_head_bwd(const float* dscore, float g, const float* hid, const float* fc2_w, int64_t batch, int d, float p_drop, float* dhid, float* g_fc2_w, float* g_fc2_b, void* stream);
int tiger_train_score_build_bwd(const float* dpair, const uint8_t* codes, int64_t batch, int d, float* dz, float* g_hit_emb, void* stream);
int tiger_train_mse(const float* pred_l, const float* pred_r, const float* hprev_left, const float* hprev_right, const int64_t* index, const int32_t* count, int64_t n, int d, float* loss, float* dpred_l, float* dpred_r, float* n_valid_out, float* work /* [2n] scratch */, void* stream);
/* CUDA-graph replay of the training step: registers a device int32 step counter (NULL clears it) that every dropout
 * kernel adds (x 101, the host's per-step seed increment) to the seed it was launched with, so that replays of one
 * captured step draw the masks of consecutive steps.  Process-wide per device; call outside stream capture. */
int tiger_train_seed_step(const int32_t* step);
int tiger_train_adam(float* params, float* grads, float* exp_avg, float* exp_avg_sq, const int64_t* seg_start, const int32_t* seg_group, int32_t* seg_step, float* seg_bc, int n_seg, float* gates, int64_t max_seg, float lr, float beta1, float beta2, float eps, float grad_scale, int zero_grad, void* stream);


/* Large products of the training step with BOTH operands pre-split into tf32 head / tail planes and pre-tiled as the
 * shared-memory image of every pipeline stage (csrc/gemm_pp.cu): tiger_gemm_pp_pack converts an operand once
 * (row-major, or transposed = element (row, k) at src[k*ld + row]; rows / reduction length optionally bounded by
 * *row_count / *k_count times per_count), tiger_sgemm_pp multiplies two packs - TMA bulk copies feed the tensor cores,
 * no thread touches operand data.  Same semantics as tiger_sgemm_ex (accumulate: atomic adds, K split over k_parts). */
int64_t tiger_gemm_pp_pack_bytes(int64_t rows, int64_t k_dim);
int tiger_gemm_pp_pack(const float* src, int64_t ld, int trans, int64_t rows, int64_t k_dim, const int32_t* row_count,
                       const int32_t* k_count, int64_t per_count, float* out, void* stream);
int tiger_sgemm_pp(const float* apack, const float* wpack, const float* bias, float* C, int64_t ldc, int64_t m_rows,
                   int n_cols, int64_t k_dim, const int32_t* m_count, const int32_t* k_count, int64_t per_count,
                   float alpha, int relu, int accumulate, int k_parts, void* stream);

/* Seq-restarter training step (csrc/train_seq.cu): SeqRestarter.forward under autograd (restarters.py:51-114 as
 * called from tiger.py:574-590) - L x L self-attention per (node, head) with dropout, folded through the mean over
 * positions (exact by linearity), forward and backward; value-bias term, token gradients (anony_emb, TimeEncode),
 * dropout, axpy. */
int tiger_train_seq_pool(const float* qk, int64_t ld_qk, const float* x, const uint8_t* mask, const int32_t* count, int64_t n, int len, int d_model, int n_head, float p_drop, int seed, float* P, float* pbar, float* psum, float* xbar, void* stream);
int tiger_train_seq_pool_bwd(const float* dxbar, const float* dpsum, const float* x, const float* qk, int64_t ld_qk, const float* P, const float* pbar, const int32_t* count, int64_t n, int len, int d_model, int n_head, float p_drop, int seed, float* dX, float* dqk, void* stream);
int tiger_train_seq_vbias(float* att, const float* psum, const float* bv, const int32_t* count, int64_t n, int d_model, int n_head, void* stream);
int tiger_train_seq_vbias_bwd(const float* datt, const float* psum, const float* bv, const int32_t* count, int64_t n, int d_model, int n_head, float* g_bv, float* dpsum, void* stream);
int tiger_train_seq_tokens_bwd(const float* dX, const int32_t* count, int64_t n, int len, const int64_t* anony_ids, const float* hist_ts, int d, int de, const float* time_w, const float* time_b, float* g_anony_emb, float* g_time_w, float* g_time_b, void* stream);
int tiger_train_dropout(float* x, const int32_t* count, int64_t per_count, int64_t n, float p_drop, int seed, int stream_id, void* stream);
int tiger_train_axpy(float* y, const float* x, const int32_t* count, int64_t per_count, int64_t n, float alpha, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TIGER_B200_H */
