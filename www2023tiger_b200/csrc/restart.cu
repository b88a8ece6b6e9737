// Restarter re-initialisation path.
// Static: StaticRestarter.forward (tiger/model/restarters.py:254-277) + TIGER.restart
// (tiger/model/tiger.py:594-609): two embedding-row gathers, prev_ts from the temporal CSR,
// both memories and their update_ts overwritten, pending message dropped.
#include "common.cuh"

#define RST_WARPS 8

// CHUNK (tiger_static_restart_ex): virtual node v = c * stride + u cuts at chunk_ts[c] and reads the CSR segment and the
// embedding rows of u; everything node-indexed is written at v
template <bool CHUNK>
__global__ void __launch_bounds__(RST_WARPS * 32)
static_restart_kernel(const int64_t* __restrict__ nids, const int32_t* __restrict__ count, int64_t n,
                      const float* __restrict__ batch_ts, int64_t batch, const double* __restrict__ q_ts,
                      const int64_t* __restrict__ indptr, const double* __restrict__ adj_ts,
                      const float* __restrict__ left_emb, const float* __restrict__ right_emb, int d,
                      float* __restrict__ left_vals, float* __restrict__ left_ts, uint8_t* __restrict__ left_active,
                      float* __restrict__ right_vals, float* __restrict__ right_ts,
                      uint8_t* __restrict__ right_active, uint8_t* __restrict__ has_msg,
                      float* __restrict__ out_prev_ts, int64_t stride, const double* __restrict__ chunk_ts) {
  int64_t total = n;
  if (count != nullptr) {
    const int64_t c = *count;
    total = c < n ? c : n;
  }
  const int lane = lane_id();
  const int64_t first = (int64_t)blockIdx.x * RST_WARPS + warp_id_in_block();
  if (first >= total) return;
  double t_batch = 0.0;
  if (!CHUNK && batch_ts != nullptr) {
    float m = INFINITY;
    for (int64_t j = lane; j < batch; j += 32) m = fminf(m, batch_ts[j]);
    t_batch = (double)warp_min(m);   // restart() receives the float32 ts.min() (train_self_supervised.py:161)
  }
  // grid-stride over the restart list: the list has a device-side length (a few dozen nodes per batch in
  // steady state, up to the whole involved set on the first batches), the grid is capped at one CTA per SM
  for (int64_t i = first; i < total; i += (int64_t)gridDim.x * RST_WARPS) {
    const int64_t u = nids[i];
    const int64_t r = CHUNK ? u % stride : u;        // the real node: CSR segment and embedding rows
    const double t = CHUNK ? chunk_ts[u / stride] : batch_ts != nullptr ? t_batch : q_ts[i];
    const int64_t beg = indptr[r], end = indptr[r + 1];
    const int64_t cut = warp_lower_bound(adj_ts, beg, end, t, lane);
    const float prev = cut > beg ? (float)adj_ts[cut - 1] : 0.f;   // get_history(.., 1): restarters.py:267-270
    if (lane == 0) {
      if (left_ts != nullptr) left_ts[u] = prev;
      if (right_ts != nullptr) right_ts[u] = prev;
      if (left_active != nullptr) left_active[u] = 1;
      if (right_active != nullptr) right_active[u] = 1;
      if (has_msg != nullptr) has_msg[u] = 0;
      if (out_prev_ts != nullptr) out_prev_ts[i] = prev;
    }
    if (left_vals != nullptr) warp_copy_row(left_vals + u * (int64_t)d, left_emb + r * (int64_t)d, d, lane);
    if (right_vals != nullptr) warp_copy_row(right_vals + u * (int64_t)d, right_emb + r * (int64_t)d, d, lane);
  }
}

extern "C" int tiger_static_restart(const int64_t* nids, const int32_t* count, int64_t n, const float* batch_ts,
                                    int64_t batch, const double* q_ts, const int64_t* indptr, const double* adj_ts,
                                    const float* left_emb, const float* right_emb, int d, float* left_vals,
                                    float* left_ts, uint8_t* left_active, float* right_vals, float* right_ts,
                                    uint8_t* right_active, uint8_t* has_msg, float* out_prev_ts, void* stream) {
  if (n < 0 || d <= 0 || (batch_ts == nullptr && q_ts == nullptr)) return TIGER_EINVAL;
  if (n == 0) return TIGER_OK;
  int64_t grid = (n + RST_WARPS - 1) / RST_WARPS;
  grid = grid > 148 ? 148 : grid;
  static_restart_kernel<false><<<(unsigned)grid, RST_WARPS * 32, 0, as_stream(stream)>>>(
      nids, count, n, batch_ts, batch, q_ts, indptr, adj_ts, left_emb, right_emb, d, left_vals, left_ts,
      left_active, right_vals, right_ts, right_active, has_msg, out_prev_ts, 0, nullptr);
  return tiger_launch_status();
}

extern "C" int tiger_static_restart_ex(const int64_t* nids, const int32_t* count, int64_t n, const float* batch_ts,
                                       int64_t batch, const double* q_ts, const int64_t* indptr, const double* adj_ts,
                                       const float* left_emb, const float* right_emb, int d, float* left_vals,
                                       float* left_ts, uint8_t* left_active, float* right_vals, float* right_ts,
                                       uint8_t* right_active, uint8_t* has_msg, float* out_prev_ts,
                                       int64_t node_stride, const double* chunk_ts, void* stream) {
  if (node_stride == 0)
    return tiger_static_restart(nids, count, n, batch_ts, batch, q_ts, indptr, adj_ts, left_emb, right_emb, d,
                                left_vals, left_ts, left_active, right_vals, right_ts, right_active, has_msg,
                                out_prev_ts, stream);
  if (n < 0 || d <= 0 || node_stride < 0 || chunk_ts == nullptr) return TIGER_EINVAL;
  if (n == 0) return TIGER_OK;
  int64_t grid = (n + RST_WARPS - 1) / RST_WARPS;
  grid = grid > 148 ? 148 : grid;
  static_restart_kernel<true><<<(unsigned)grid, RST_WARPS * 32, 0, as_stream(stream)>>>(
      nids, count, n, nullptr, 0, nullptr, indptr, adj_ts, left_emb, right_emb, d, left_vals, left_ts, left_active,
      right_vals, right_ts, right_active, has_msg, out_prev_ts, node_stride, chunk_ts);
  return tiger_launch_status();
}

// Restart surrogates of a read-only query (tiger_compact_involved_ex with read_only): row i of out_rows receives
// right_emb[nids[i]] - the right-memory row tiger_static_restart would write for the i-th restarted node - for
// i < min(*count, n); nothing node-indexed is written.
__global__ void __launch_bounds__(RST_WARPS * 32)
static_restart_rows_kernel(const int64_t* __restrict__ nids, const int32_t* __restrict__ count, int64_t n,
                           const float* __restrict__ right_emb, int d, float* __restrict__ out_rows) {
  int64_t total = n;
  if (count != nullptr) {
    const int64_t c = *count;
    total = c < n ? c : n;
  }
  const int lane = lane_id();
  for (int64_t i = (int64_t)blockIdx.x * RST_WARPS + warp_id_in_block(); i < total; i += (int64_t)gridDim.x * RST_WARPS)
    warp_copy_row(out_rows + i * (int64_t)d, right_emb + nids[i] * (int64_t)d, d, lane);
}

extern "C" int tiger_static_restart_rows(const int64_t* nids, const int32_t* count, int64_t n, const float* right_emb,
                                         int d, float* out_rows, void* stream) {
  if (n < 0 || d <= 0 || nids == nullptr || right_emb == nullptr || out_rows == nullptr) return TIGER_EINVAL;
  if (n == 0) return TIGER_OK;
  int64_t grid = (n + RST_WARPS - 1) / RST_WARPS;
  grid = grid > 148 ? 148 : grid;
  static_restart_rows_kernel<<<(unsigned)grid, RST_WARPS * 32, 0, as_stream(stream)>>>(nids, count, n, right_emb, d,
                                                                                       out_rows);
  return tiger_launch_status();
}
