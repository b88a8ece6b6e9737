// Node memory tables, the last-message store and their write-backs: HBM-bound row gathers and
// scatters, one warp per row, 16-byte vectors where the row alignment allows it.
// Reference: tiger/model/memory.py:12-138, tiger/model/time_encoding.py,
// tiger/model/tiger.py:230-255,396-442.
#include "common.cuh"
#include "umma.cuh"

#define ROW_WARPS 8  // warps (rows) per CTA for the row kernels

static inline unsigned row_grid(int64_t n_rows) {
  const int64_t per_cta = (int64_t)ROW_WARPS * ROWS_PER_WARP;
  return (unsigned)((n_rows + per_cta - 1) / per_cta);
}

// rows one warp resolves and copies (lane-per-row index chain, warp_copy_lane_rows): few rows (a batch of 200
// events) -> 4, so that the rows spread over many warps; many rows -> up to 32, so that the chain of dependent
// index loads is paid once per 32 rows and the warp spends its life streaming
static inline int rows_per_warp(int64_t n_rows) {
  return n_rows >= (1 << 16) ? 32 : n_rows >= (1 << 14) ? 16 : n_rows >= (1 << 12) ? 8 : ROWS_PER_WARP;
}
static inline unsigned row_grid(int64_t n_rows, int rpw) {
  const int64_t per_cta = (int64_t)ROW_WARPS * rpw;
  return (unsigned)((n_rows + per_cta - 1) / per_cta);
}

__device__ __forceinline__ int64_t effective_count(const int32_t* count, int64_t n) {
  if (count == nullptr) return n;
  const int64_t c = *count;
  return c < n ? c : n;
}

// Large row sets (>= 64 k rows): the rows move through shared memory with the bulk-copy engine instead of through
// registers.  Lane l of a warp owns row l of a batch of 32: after the (lane-parallel) index chain every lane issues
// ONE bulk load of its whole row (cp.async.bulk, completion on the warp's mbarrier) - 32 rows = 22 KB per warp and
// 176 KB per SM are in flight at once, far more than the register path can hold - and, once the barrier fires, one
// bulk store of the row to its destination.  No thread touches the payload.  Needs 16-byte aligned rows.
#define ROWS_TMA_MIN (1 << 16)
__device__ __forceinline__ void warp_tma_move_rows(float* my_dst, const float* my_src, uint32_t row_bytes,
                                                   unsigned char* smem_base, int lane) {
  // layout per warp: [32 rows][row_bytes] then one mbarrier (row_bytes is a multiple of 16)
  const int warp = warp_id_in_block();
  unsigned char* rows = smem_base + (size_t)warp * (32u * row_bytes + 16u);
  uint64_t* bar = reinterpret_cast<uint64_t*>(rows + 32u * row_bytes);
  if (lane == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncwarp();
  const bool active = my_dst != nullptr;
  const unsigned n_act = __popc(__ballot_sync(TIGER_FULL_MASK, active));
  if (n_act == 0) return;
  if (lane == 0) mbar_arrive_expect_tx(bar, n_act * row_bytes);
  __syncwarp();
  unsigned char* mine = rows + (size_t)lane * row_bytes;
  if (active) tma_bulk_load(mine, my_src, row_bytes, bar);
  mbar_wait(bar, 0);
  if (active) {
    tma_bulk_store(my_dst, mine, row_bytes);
    tma_store_commit();
    tma_store_wait_read();      // shared memory is released when the CTA exits
  }
}

static inline size_t rows_tma_smem(int64_t width) { return (size_t)ROW_WARPS * (32u * (size_t)width * 4u + 16u); }

// the bulk path applies to a launch when there are many rows, the rows are 16-byte multiples, every base pointer is
// 16-byte aligned and a CTA's staging area fits the shared memory of an SM
template <typename Kernel>
static inline bool rows_tma_ok(Kernel kernel, int64_t n_rows, int64_t width, const void* a, const void* b) {
  if (n_rows < ROWS_TMA_MIN || width <= 0 || (width & 3) != 0 || ((((uintptr_t)a) | ((uintptr_t)b)) & 15) != 0) return false;
  const size_t smem = rows_tma_smem(width);
  if (smem > 200 * 1024) return false;
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
}

// ---------------------------------------------------------------- a11 Memory.get
__global__ void __launch_bounds__(ROW_WARPS * 32, 4)
gather_rows_kernel(const float* __restrict__ table, int64_t width, const int64_t* __restrict__ ids, int64_t n,
                   float* __restrict__ out, const float* __restrict__ ts_table, float* __restrict__ out_ts, int rpw,
                   int tma) {
  extern __shared__ __align__(128) unsigned char row_smem[];
  const int64_t r0 = ((int64_t)blockIdx.x * ROW_WARPS + warp_id_in_block()) * rpw;
  if (r0 >= n) return;
  const int lane = lane_id();
  const int64_t r = r0 + lane;
  float* dst = nullptr;
  const float* src = table;
  if (lane < rpw && r < n) {               // lane l owns row l: index and scalar side
    const int64_t u = ids[r];
    if (out != nullptr) dst = out + r * width;
    src = table + u * width;
    if (out_ts != nullptr) out_ts[r] = ts_table[u];
  }
  if (tma)
    warp_tma_move_rows(dst, src, (uint32_t)width * 4u, row_smem, lane);
  else
    warp_copy_lane_rows(dst, src, rpw, (int)width, lane);
}

extern "C" int tiger_gather_rows(const float* table, int64_t width, const int64_t* ids, int64_t n, float* out,
                                 const float* ts_table, float* out_ts, void* stream) {
  if (n < 0 || width < 0) return TIGER_EINVAL;
  if (n == 0) return TIGER_OK;
  const int rpw = rows_per_warp(n);
  // measured (bench.py --micro, 262,144 rows): the register path is the faster one for the gather direction (0.80 vs
  // 0.785 of the copy peak), the bulk path for the scatter direction (0.69 vs 0.66)
  const bool tma = false;
  gather_rows_kernel<<<row_grid(n, rpw), ROW_WARPS * 32, tma ? rows_tma_smem(width) : 0, as_stream(stream)>>>(
      table, width, ids, n, out, ts_table, out_ts, rpw, tma ? 1 : 0);
  return tiger_launch_status();
}

// ---------------------------------------------------------------- a11 Memory.set
__global__ void __launch_bounds__(ROW_WARPS * 32, 4)
scatter_rows_kernel(float* __restrict__ table, int64_t width, const int64_t* __restrict__ ids, int64_t n,
                    const int32_t* __restrict__ count, const float* __restrict__ vals,
                    float* __restrict__ ts_table, const float* __restrict__ ts, uint8_t* __restrict__ active,
                    int check, uint32_t* __restrict__ err_flags, int rpw, int tma) {
  extern __shared__ __align__(128) unsigned char row_smem[];
  const int64_t r0 = ((int64_t)blockIdx.x * ROW_WARPS + warp_id_in_block()) * rpw;
  const int64_t n_eff = effective_count(count, n);
  if (r0 >= n_eff) return;
  const int lane = lane_id();
  const int64_t r = r0 + lane;
  float* dst = nullptr;
  const float* src = vals;
  if (lane < rpw && r < n_eff) {           // lane l owns row l: index and scalar side
    const int64_t u = ids[r];
    if (ts_table != nullptr) {
      if (check && err_flags != nullptr && ts_table[u] > ts[r]) atomicOr(err_flags, TIGER_ERR_PAST_MEMORY);
      ts_table[u] = ts[r];
    }
    if (active != nullptr) active[u] = 1;
    if (table != nullptr) dst = table + u * width;
    src = vals + r * width;
  }
  if (tma)
    warp_tma_move_rows(dst, src, (uint32_t)width * 4u, row_smem, lane);
  else
    warp_copy_lane_rows(dst, src, rpw, (int)width, lane);
}

extern "C" int tiger_scatter_rows(float* table, int64_t width, const int64_t* ids, int64_t n,
                                  const int32_t* count, const float* vals, float* ts_table, const float* ts,
                                  uint8_t* active, int check, uint32_t* err_flags, void* stream) {
  if (n < 0 || width < 0) return TIGER_EINVAL;
  if (n == 0) return TIGER_OK;
  const int rpw = rows_per_warp(n);
  const bool tma = table != nullptr && rows_tma_ok(scatter_rows_kernel, n, width, table, vals);
  scatter_rows_kernel<<<row_grid(n, rpw), ROW_WARPS * 32, tma ? rows_tma_smem(width) : 0, as_stream(stream)>>>(
      table, width, ids, n, count, vals, ts_table, ts, active, check, err_flags, rpw, tma ? 1 : 0);
  return tiger_launch_status();
}

// ---------------------------------------------------------------- a10 TimeEncode
__global__ void time_encode_kernel(const float* __restrict__ ts, int64_t total, const float* __restrict__ w,
                                   const float* __restrict__ b, int dim, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % dim);
  out[i] = time_enc(ts[i / dim], w[c], b[c]);
}

extern "C" int tiger_time_encode(const float* ts, int64_t n, const float* w, const float* b, int dim, float* out,
                                 void* stream) {
  if (n < 0 || dim <= 0) return TIGER_EINVAL;
  const int64_t total = n * dim;
  if (total == 0) return TIGER_OK;
  time_encode_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(ts, total, w, b, dim, out);
  return tiger_launch_status();
}

// ---------------------------------------------------------------- a9 store_events
// one warp per position p of pos = [src ; dst]; only selected positions build and write a row.
// Table mode: memory rows / update_ts are read from the node-indexed tables (fused engine).
// Dense mode: they are the per-event copies Memory.get returned (class surface, memory.py:77-106).
struct StoreSrc {
  const float* mem_vals;   // [N, d]   table mode
  const float* mem_ts;     // [N]
  const float* src_vals;   // [B, d]   dense mode
  const float* dst_vals;   // [B, d]
  const float* src_prev;   // [B]
  const float* dst_prev;   // [B]
  int dense;
};

__global__ void __launch_bounds__(ROW_WARPS * 32)
store_messages_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                      const int64_t* __restrict__ eids, const float* __restrict__ ts, int64_t batch,
                      const uint8_t* __restrict__ winner, const StoreSrc in, const float* __restrict__ nfeats,
                      const float* __restrict__ efeats, int d, int de, const float* __restrict__ time_w,
                      const float* __restrict__ time_b, float* __restrict__ msg_vals, float* __restrict__ msg_ts,
                      uint8_t* __restrict__ has_msg, uint32_t* __restrict__ err_flags) {
  const int64_t p = (int64_t)blockIdx.x * ROW_WARPS + warp_id_in_block();
  if (p >= 2 * batch) return;
  const int lane = lane_id();
  const bool is_src = p < batch;
  const int64_t e = is_src ? p : p - batch;
  const int64_t self = is_src ? src[e] : dst[e];
  const int64_t other = is_src ? dst[e] : src[e];
  const float t = ts[e];
  const float prev = in.dense ? (is_src ? in.src_prev[e] : in.dst_prev[e]) : in.mem_ts[self];
  if (lane == 0 && err_flags != nullptr) {
    if (prev > t) atomicOr(err_flags, TIGER_ERR_EVENT_BEFORE_MEM);   // tiger.py:436-438
    if (has_msg[self] != 0) atomicOr(err_flags, TIGER_ERR_UNUSED_MSG);  // memory.py:85-87
  }
  if (!winner[p]) return;
  const int64_t m_dim = 3 * (int64_t)d + de;
  float* row = msg_vals + self * m_dim;
  const float* self_row = in.dense ? (is_src ? in.src_vals : in.dst_vals) + e * d : in.mem_vals + self * d;
  const float* other_row = in.dense ? (is_src ? in.dst_vals : in.src_vals) + e * d : in.mem_vals + other * d;
  const float* nf_self = nfeats ? nfeats + self * d : nullptr;
  const float* nf_other = nfeats ? nfeats + other * d : nullptr;
  const float* ef_row = efeats != nullptr ? efeats + eids[e] * de : nullptr;
  const float dt = t - prev;
  float* trow = row + 2 * d + de;
  const int d4 = d >> 2, de4 = de >> 2;
  const bool vec = (d & 3) == 0 && (de & 3) == 0 && d4 <= 64 && de4 <= 64 &&
                   ((((uintptr_t)row | (uintptr_t)self_row | (uintptr_t)other_row | (uintptr_t)nf_self |
                      (uintptr_t)nf_other | (uintptr_t)ef_row | (uintptr_t)time_w | (uintptr_t)time_b) & 15) == 0);
  if (vec) {
    // all gathers of the row are issued before the first store (up to 10 16-byte loads per lane in flight)
    const int c0 = lane, c1 = lane + 32;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 s[2] = {z, z}, o[2] = {z, z}, ns[2] = {z, z}, no[2] = {z, z}, ef[2] = {z, z};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int c = h == 0 ? c0 : c1;
      if (c < d4) {
        s[h] = reinterpret_cast<const float4*>(self_row)[c];
        o[h] = reinterpret_cast<const float4*>(other_row)[c];
        if (nf_self != nullptr) {
          ns[h] = reinterpret_cast<const float4*>(nf_self)[c];
          no[h] = reinterpret_cast<const float4*>(nf_other)[c];
        }
      }
      if (c < de4 && ef_row != nullptr) ef[h] = reinterpret_cast<const float4*>(ef_row)[c];
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int c = h == 0 ? c0 : c1;
      if (c < d4) {
        reinterpret_cast<float4*>(row)[c] = nf_self != nullptr
            ? make_float4(s[h].x + ns[h].x, s[h].y + ns[h].y, s[h].z + ns[h].z, s[h].w + ns[h].w) : s[h];
        reinterpret_cast<float4*>(row + d)[c] = nf_self != nullptr
            ? make_float4(o[h].x + no[h].x, o[h].y + no[h].y, o[h].z + no[h].z, o[h].w + no[h].w) : o[h];
        const float4 w4 = reinterpret_cast<const float4*>(time_w)[c], b4 = reinterpret_cast<const float4*>(time_b)[c];
        reinterpret_cast<float4*>(trow)[c] = make_float4(time_enc(dt, w4.x, b4.x), time_enc(dt, w4.y, b4.y),
                                                        time_enc(dt, w4.z, b4.z), time_enc(dt, w4.w, b4.w));
      }
      if (c < de4) reinterpret_cast<float4*>(row + 2 * d)[c] = ef[h];
    }
  } else {
    warp_add_row(row, self_row, nf_self, d, lane);
    warp_add_row(row + d, other_row, nf_other, d, lane);
    if (ef_row != nullptr) {
      warp_copy_row(row + 2 * d, ef_row, de, lane);
    } else {
      for (int i = lane; i < de; i += 32) row[2 * d + i] = 0.f;
    }
    for (int i = lane; i < d; i += 32) trow[i] = time_enc(dt, time_w[i], time_b[i]);
  }
  if (lane == 0) msg_ts[self] = t;
}

// has_msg is raised by a second launch so that the unused-message check above never observes
// a flag set by another warp of the same batch (a node can occur at several positions)
__global__ void raise_has_msg_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                     int64_t batch, const uint8_t* __restrict__ winner,
                                     uint8_t* __restrict__ has_msg) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= 2 * batch || !winner[p]) return;
  has_msg[p < batch ? src[p] : dst[p - batch]] = 1;
}

static int launch_store(const int64_t* src, const int64_t* dst, const int64_t* eids, const float* ts, int64_t batch,
                        const uint8_t* winner, const StoreSrc& in, const float* nfeats, const float* efeats, int d,
                        int de, const float* time_w, const float* time_b, float* msg_vals, float* msg_ts,
                        uint8_t* has_msg, uint32_t* err_flags, void* stream) {
  if (batch < 0 || d <= 0 || de <= 0) return TIGER_EINVAL;
  if (batch == 0) return TIGER_OK;
  const int64_t n = 2 * batch;
  store_messages_kernel<<<(unsigned)((n + ROW_WARPS - 1) / ROW_WARPS), ROW_WARPS * 32, 0, as_stream(stream)>>>(
      src, dst, eids, ts, batch, winner, in, nfeats, efeats, d, de, time_w, time_b, msg_vals, msg_ts, has_msg,
      err_flags);
  raise_has_msg_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(src, dst, batch, winner,
                                                                                  has_msg);
  return tiger_launch_status();
}

extern "C" int tiger_store_messages(const int64_t* src, const int64_t* dst, const int64_t* eids, const float* ts,
                                    int64_t batch, const uint8_t* winner, const float* mem_vals,
                                    const float* mem_ts, const float* nfeats, const float* efeats, int d, int de,
                                    const float* time_w, const float* time_b, float* msg_vals, float* msg_ts,
                                    uint8_t* has_msg, uint32_t* err_flags, void* stream) {
  StoreSrc in = {mem_vals, mem_ts, nullptr, nullptr, nullptr, nullptr, 0};
  return launch_store(src, dst, eids, ts, batch, winner, in, nfeats, efeats, d, de, time_w, time_b, msg_vals,
                      msg_ts, has_msg, err_flags, stream);
}

extern "C" int tiger_store_messages_dense(const int64_t* src, const int64_t* dst, const int64_t* eids,
                                          const float* ts, int64_t batch, const uint8_t* winner,
                                          const float* src_vals, const float* dst_vals, const float* src_prev_ts,
                                          const float* dst_prev_ts, const float* nfeats, const float* efeats, int d,
                                          int de, const float* time_w, const float* time_b, float* msg_vals,
                                          float* msg_ts, uint8_t* has_msg, uint32_t* err_flags, void* stream) {
  StoreSrc in = {nullptr, nullptr, src_vals, dst_vals, src_prev_ts, dst_prev_ts, 1};
  return launch_store(src, dst, eids, ts, batch, winner, in, nfeats, efeats, d, de, time_w, time_b, msg_vals,
                      msg_ts, has_msg, err_flags, stream);
}

// ---------------------------------------------------------------- a17 right write-back (+ a19)
__global__ void __launch_bounds__(ROW_WARPS * 32, 4)
right_writeback_kernel(const int64_t* __restrict__ pos_ids, int64_t n_pos, const uint8_t* __restrict__ winner,
                       const int32_t* __restrict__ gru_row, const float* __restrict__ h_new, int d,
                       float* __restrict__ right_vals, float* __restrict__ right_ts,
                       uint8_t* __restrict__ right_active, const float* __restrict__ msg_ts,
                       uint8_t* __restrict__ has_msg, uint32_t* __restrict__ err_flags, int rpw, int tma) {
  extern __shared__ __align__(128) unsigned char row_smem[];
  const int64_t p0 = ((int64_t)blockIdx.x * ROW_WARPS + warp_id_in_block()) * rpw;
  if (p0 >= n_pos) return;
  const int lane = lane_id();
  const int64_t p = p0 + lane;
  // lane l resolves position l: position -> node -> {pending flag, GRU row, clocks}; every selected node occurs at
  // one position only (tiger_select_latest), so no two lanes touch the same node
  float* dst = nullptr;
  const float* src = h_new;
  if (lane < rpw && p < n_pos && winner[p]) {
    const int64_t u = pos_ids[p];
    const uint8_t pending = has_msg[u];
    const int32_t r = gru_row[u];
    const float t_msg = msg_ts[u], t_mem = right_ts[u];
    if (pending != 0) {                    // a positive without a pending message has nothing to persist
      if (err_flags != nullptr && t_mem > t_msg) atomicOr(err_flags, TIGER_ERR_PAST_MEMORY);
      right_ts[u] = t_msg;
      if (right_active != nullptr) right_active[u] = 1;
      has_msg[u] = 0;                      // the message is consumed (tiger.py:240)
      dst = right_vals + u * (int64_t)d;
      src = h_new + (int64_t)r * d;
    }
  }
  if (tma)
    warp_tma_move_rows(dst, src, (uint32_t)d * 4u, row_smem, lane);
  else
    warp_copy_lane_rows(dst, src, rpw, d, lane);
}

__global__ void __launch_bounds__(ROW_WARPS * 32)
hprev_copy_kernel(const int64_t* __restrict__ pos_ids, int64_t n_pos, int d, const float* __restrict__ left_vals,
                  const float* __restrict__ right_vals, float* __restrict__ hprev_left,
                  float* __restrict__ hprev_right) {
  const int64_t p0 = ((int64_t)blockIdx.x * ROW_WARPS + warp_id_in_block()) * (ROWS_PER_WARP / 2);
  if (p0 >= n_pos) return;
  const int lane = lane_id();
  float* dst[ROWS_PER_WARP];
  const float* src[ROWS_PER_WARP];
#pragma unroll
  for (int i = 0; i < ROWS_PER_WARP / 2; ++i) {
    const int64_t p = p0 + i;
    const bool live = p < n_pos;
    const int64_t u = live ? pos_ids[p] : 0;
    dst[2 * i] = live ? hprev_left + p * d : nullptr;
    src[2 * i] = left_vals + u * d;
    dst[2 * i + 1] = live ? hprev_right + p * d : nullptr;
    src[2 * i + 1] = right_vals + u * d;
  }
  warp_copy_rows<ROWS_PER_WARP>(dst, src, d, lane);
}

extern "C" int tiger_right_writeback(const int64_t* pos_ids, int64_t n_pos, const uint8_t* winner,
                                     const int32_t* gru_row, const float* h_new, int d, float* right_vals,
                                     float* right_ts, uint8_t* right_active, const float* msg_ts,
                                     uint8_t* has_msg, const float* left_vals, float* hprev_left,
                                     float* hprev_right, uint32_t* err_flags, void* stream) {
  if (n_pos < 0 || d <= 0) return TIGER_EINVAL;
  if ((hprev_left == nullptr) != (hprev_right == nullptr)) return TIGER_EINVAL;
  if (n_pos == 0) return TIGER_OK;
  const int rpw = rows_per_warp(n_pos);
  const bool tma = rows_tma_ok(right_writeback_kernel, n_pos, d, right_vals, h_new);
  right_writeback_kernel<<<row_grid(n_pos, rpw), ROW_WARPS * 32, tma ? rows_tma_smem(d) : 0, as_stream(stream)>>>(
      pos_ids, n_pos, winner, gru_row, h_new, d, right_vals, right_ts, right_active, msg_ts, has_msg, err_flags, rpw,
      tma ? 1 : 0);
  if (hprev_left != nullptr)
    hprev_copy_kernel<<<row_grid(2 * n_pos), ROW_WARPS * 32, 0, as_stream(stream)>>>(pos_ids, n_pos, d, left_vals,
                                                                                    right_vals, hprev_left, hprev_right);
  return tiger_launch_status();
}

// ---------------------------------------------------------------- a18 left write-back
__global__ void __launch_bounds__(ROW_WARPS * 32, 4)
left_writeback_kernel(const int64_t* __restrict__ pos_ids, int64_t n_pos, int64_t batch,
                      const uint8_t* __restrict__ winner, const float* __restrict__ h_left, int d,
                      const float* __restrict__ ts, float* __restrict__ left_vals, float* __restrict__ left_ts,
                      uint8_t* __restrict__ left_active, uint32_t* __restrict__ err_flags, int rpw, int tma) {
  extern __shared__ __align__(128) unsigned char row_smem[];
  const int64_t p0 = ((int64_t)blockIdx.x * ROW_WARPS + warp_id_in_block()) * rpw;
  if (p0 >= n_pos) return;
  const int lane = lane_id();
  const int64_t p = p0 + lane;
  float* dst = nullptr;
  const float* src = h_left;
  if (lane < rpw && p < n_pos && winner[p]) {   // lane l owns position l: index and scalar side
    const int64_t u = pos_ids[p];
    const float t = ts[p % batch];
    if (err_flags != nullptr && left_ts[u] > t) atomicOr(err_flags, TIGER_ERR_PAST_MEMORY);
    left_ts[u] = t;
    if (left_active != nullptr) left_active[u] = 1;
    dst = left_vals + u * (int64_t)d;
    src = h_left + p * d;
  }
  if (tma)
    warp_tma_move_rows(dst, src, (uint32_t)d * 4u, row_smem, lane);
  else
    warp_copy_lane_rows(dst, src, rpw, d, lane);
}

extern "C" int tiger_left_writeback(const int64_t* pos_ids, int64_t n_pos, int64_t batch, const uint8_t* winner,
                                    const float* h_left, int d, const float* ts, float* left_vals, float* left_ts,
                                    uint8_t* left_active, uint32_t* err_flags, void* stream) {
  if (n_pos < 0 || d <= 0 || batch <= 0) return TIGER_EINVAL;
  if (n_pos == 0) return TIGER_OK;
  const int rpw = rows_per_warp(n_pos);
  const bool tma = rows_tma_ok(left_writeback_kernel, n_pos, d, left_vals, h_left);
  left_writeback_kernel<<<row_grid(n_pos, rpw), ROW_WARPS * 32, tma ? rows_tma_smem(d) : 0, as_stream(stream)>>>(
      pos_ids, n_pos, batch, winner, h_left, d, ts, left_vals, left_ts, left_active, err_flags, rpw, tma ? 1 : 0);
  return tiger_launch_status();
}
