// Temporal neighbor finder over a per-node time-sorted CSR, involved-node marking and
// ordered compaction.  Integer / index work: every result is bit-exact with the reference
// (tiger/data/graph.py:44-53,117-127,150-155; tiger/data/data_loader.py:61-67,105-131;
// tiger/data/data_classes.py:163-165; tiger/model/memory.py:108-126).
#include "common.cuh"
#include "umma.cuh"
#ifdef TIGER_TRACE
#include <cstdio>
#endif

// ------------------------------------------------------------------------------------------
// K1  FIND_G lanes per query (4 queries per warp): FIND_G-ary cooperative lower-bound search on the
// float64 timestamps of the node's CSR segment (strict '<', np.searchsorted side='left'), then a gather
// of the K entries that precede the cut, right-aligned, zero-padded on the left.  The kernel is a chain
// of dependent loads (node id -> indptr -> probes -> entries); several queries per warp keep enough of
// those chains in flight to use the memory system.
// ------------------------------------------------------------------------------------------
// Chunk modes (MODE != 0, tiger_find_recent_ex): query ids are virtual ids v = c * stride + u of chunk c; the search
// reads the CSR segment of u.  TIGER_FIND_CHUNK_NEIGHBORS returns the neighbor ids offset by c * stride except the
// padding id 0, which stays 0 (the attention masks slots by id 0) but marks the chunk's own node 0; a query with id 0
// (the second hop of a padding slot) marks nothing.  TIGER_FIND_CHUNK_HISTORY takes the query time from q_ts[c] and
// returns the real neighbor ids.  Both mark the bitmap with virtual ids.
#define FIND_G 8
template <int MODE>
__global__ void __launch_bounds__(256)
find_recent_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ adj_nbr,
                   const int32_t* __restrict__ adj_eid, const double* __restrict__ adj_ts,
                   const uint8_t* __restrict__ adj_flag, const int64_t* __restrict__ q_nids,
                   const double* __restrict__ q_ts, int64_t n_query, const int32_t* __restrict__ count,
                   int64_t ts_period, int k, int64_t* __restrict__ out_nids, int64_t* __restrict__ out_eids,
                   float* __restrict__ out_ts, int64_t* __restrict__ out_dirs,
                   float* __restrict__ out_ts32, uint32_t* __restrict__ bitmap, int64_t stride) {
  const int lane = lane_id(), l = lane & (FIND_G - 1);
  const int64_t q = ((int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block()) * (32 / FIND_G) + lane / FIND_G;
  const bool live = q < n_query && (count == nullptr || q < *count);
  int64_t nid = 0, beg = 0, end = 0, base = 0;
  double t = 0.0;
  if (live) {
    nid = q_nids[q];
    if (MODE != 0) base = nid - nid % stride;
    t = MODE == TIGER_FIND_CHUNK_HISTORY ? q_ts[nid / stride] : q_ts[q % ts_period];
    if (MODE != TIGER_FIND_CHUNK_HISTORY && out_ts32 != nullptr && q < ts_period && l == 0) out_ts32[q] = (float)t;
    beg = indptr[nid - base];
    end = indptr[nid - base + 1];
  }
  const int64_t cut = group_lower_bound<FIND_G>(adj_ts, beg, end, t, lane);
  if (!live) return;
  const bool mark = bitmap != nullptr && (MODE != TIGER_FIND_CHUNK_NEIGHBORS || nid != 0);
  if (mark && l == 0) atomicOr(bitmap + (nid >> 5), 1u << (nid & 31));
  for (int kk = l; kk < k; kk += FIND_G) {
    const int64_t s = cut - k + kk;
    int64_t nb = 0, ei = 0, dr = 0;
    float tv = 0.f;
    if (s >= beg) {
      nb = adj_nbr[s];
      ei = adj_eid[s];
      tv = (float)adj_ts[s];  // float64 -> float32, round-to-nearest (graph.py:91,126)
      dr = adj_flag[s];
    }
    const int64_t o = q * k + kk;
    out_nids[o] = MODE == TIGER_FIND_CHUNK_NEIGHBORS && nb != 0 ? nb + base : nb;
    out_eids[o] = ei;
    out_ts[o] = tv;
    if (out_dirs != nullptr) out_dirs[o] = dr;
    if (MODE != 0) nb += base;
    if (mark) atomicOr(bitmap + (nb >> 5), 1u << (nb & 31));
  }
}

extern "C" int tiger_find_recent(const int64_t* indptr, const int32_t* adj_nbr, const int32_t* adj_eid,
                                 const double* adj_ts, const uint8_t* adj_flag, const int64_t* q_nids,
                                 const double* q_ts, int64_t n_query, int64_t ts_period, int k,
                                 int64_t* out_nids, int64_t* out_eids, float* out_ts, int64_t* out_dirs,
                                 float* out_ts32, uint32_t* mark_bitmap, const int32_t* count, void* stream) {
  if (n_query < 0 || k <= 0 || ts_period < 0) return TIGER_EINVAL;
  if (n_query == 0) return TIGER_OK;
  if (ts_period == 0) ts_period = n_query;
  const int warps = 8, per_cta = warps * (32 / FIND_G);
  const unsigned grid = (unsigned)((n_query + per_cta - 1) / per_cta);
  find_recent_kernel<0><<<grid, warps * 32, 0, as_stream(stream)>>>(
      indptr, adj_nbr, adj_eid, adj_ts, adj_flag, q_nids, q_ts, n_query, count, ts_period, k, out_nids, out_eids,
      out_ts, out_dirs, out_ts32, mark_bitmap, 0);
  return tiger_launch_status();
}

extern "C" int tiger_find_recent_ex(const int64_t* indptr, const int32_t* adj_nbr, const int32_t* adj_eid,
                                    const double* adj_ts, const uint8_t* adj_flag, const int64_t* q_nids,
                                    const double* q_ts, int64_t n_query, int64_t ts_period, int k,
                                    int64_t* out_nids, int64_t* out_eids, float* out_ts, int64_t* out_dirs,
                                    float* out_ts32, uint32_t* mark_bitmap, const int32_t* count,
                                    int64_t node_stride, int mode, void* stream) {
  if (mode == 0)
    return tiger_find_recent(indptr, adj_nbr, adj_eid, adj_ts, adj_flag, q_nids, q_ts, n_query, ts_period, k,
                             out_nids, out_eids, out_ts, out_dirs, out_ts32, mark_bitmap, count, stream);
  if (n_query < 0 || k <= 0 || ts_period < 0 || node_stride <= 0) return TIGER_EINVAL;
  if (mode != TIGER_FIND_CHUNK_NEIGHBORS && mode != TIGER_FIND_CHUNK_HISTORY) return TIGER_EINVAL;
  if (n_query == 0) return TIGER_OK;
  if (ts_period == 0) ts_period = n_query;
  const int warps = 8, per_cta = warps * (32 / FIND_G);
  const unsigned grid = (unsigned)((n_query + per_cta - 1) / per_cta);
  auto kernel = mode == TIGER_FIND_CHUNK_NEIGHBORS ? find_recent_kernel<TIGER_FIND_CHUNK_NEIGHBORS>
                                                   : find_recent_kernel<TIGER_FIND_CHUNK_HISTORY>;
  kernel<<<grid, warps * 32, 0, as_stream(stream)>>>(indptr, adj_nbr, adj_eid, adj_ts, adj_flag, q_nids, q_ts,
                                                     n_query, count, ts_period, k, out_nids, out_eids, out_ts,
                                                     out_dirs, out_ts32, mark_bitmap, node_stride);
  return tiger_launch_status();
}

// ------------------------------------------------------------------------------------------
// hit window (data_loader.py:61-67)
// ------------------------------------------------------------------------------------------
__global__ void hit_window_kernel(const int64_t* __restrict__ center, const int64_t* __restrict__ neigh,
                                  int64_t total, int k, float* __restrict__ hit) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  hit[i] = (center[i / k] == neigh[i]) ? 1.0f : 0.0f;
}

extern "C" int tiger_hit_window(const int64_t* center, const int64_t* neigh, int64_t n, int k, float* hit,
                                void* stream) {
  if (n < 0 || k <= 0) return TIGER_EINVAL;
  const int64_t total = n * k;
  if (total == 0) return TIGER_OK;
  hit_window_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(center, neigh, total, k, hit);
  return tiger_launch_status();
}

// ------------------------------------------------------------------------------------------
// involved-node bitmap: mark + ordered compaction
// ------------------------------------------------------------------------------------------
__global__ void mark_nodes_kernel(const int64_t* __restrict__ ids, int64_t n, uint32_t* __restrict__ bitmap,
                                  int64_t n_nodes) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t u = ids[i];
  if (u >= 0 && u < n_nodes) atomicOr(bitmap + (u >> 5), 1u << (u & 31));
}

extern "C" int tiger_mark_nodes(const int64_t* ids, int64_t n, uint32_t* bitmap, int64_t n_nodes, void* stream) {
  if (n < 0) return TIGER_EINVAL;
  if (n == 0) return TIGER_OK;
  mark_nodes_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(ids, n, bitmap, n_nodes);
  return tiger_launch_status();
}

// exclusive scan of three per-thread counters over a 1024-thread block
__device__ __forceinline__ void block_exscan3(int& a, int& b, int& c, int* total, int (*sm)[32]) {
  const int lane = lane_id(), warp = warp_id_in_block();
  int ia = a, ib = b, ic = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int ta = __shfl_up_sync(TIGER_FULL_MASK, ia, o);
    const int tb = __shfl_up_sync(TIGER_FULL_MASK, ib, o);
    const int tc = __shfl_up_sync(TIGER_FULL_MASK, ic, o);
    if (lane >= o) { ia += ta; ib += tb; ic += tc; }
  }
  if (lane == 31) { sm[0][warp] = ia; sm[1][warp] = ib; sm[2][warp] = ic; }
  __syncthreads();
  if (warp == 0) {
    int va = sm[0][lane], vb = sm[1][lane], vc = sm[2][lane];
    int sa = va, sb = vb, sc = vc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int ta = __shfl_up_sync(TIGER_FULL_MASK, sa, o);
      const int tb = __shfl_up_sync(TIGER_FULL_MASK, sb, o);
      const int tc = __shfl_up_sync(TIGER_FULL_MASK, sc, o);
      if (lane >= o) { sa += ta; sb += tb; sc += tc; }
    }
    sm[0][lane] = sa - va; sm[1][lane] = sb - vb; sm[2][lane] = sc - vc;
    if (lane == 31) { total[0] = sa; total[1] = sb; total[2] = sc; }
  }
  __syncthreads();
  a = ia - a + sm[0][warp];
  b = ib - b + sm[1][warp];
  c = ic - c + sm[2][warp];
}

__global__ void __launch_bounds__(1024)
compact_involved_kernel(uint32_t* __restrict__ bitmap, int64_t n_words, uint8_t* __restrict__ has_msg,
                        uint8_t* __restrict__ uptodate, int64_t* __restrict__ involved, int64_t cap,
                        int64_t* __restrict__ local_index, int64_t* __restrict__ outdated,
                        int32_t* __restrict__ gru_row, int64_t* __restrict__ restart_nodes,
                        int32_t* __restrict__ counts, uint32_t* __restrict__ err_flags, int read_only,
                        int restart_base) {
  __shared__ int sm[3][32];
  __shared__ int total[3];
  const int tid = threadIdx.x;
  const int64_t wpt = (n_words + blockDim.x - 1) / blockDim.x;
  const int64_t w0 = (int64_t)tid * wpt;
  const int64_t w1 = (w0 + wpt < n_words) ? (w0 + wpt) : n_words;
  int c_inv = 0, c_out = 0, c_rst = 0;
  for (int64_t w = w0; w < w1; ++w) {
    uint32_t bits = bitmap[w];
    c_inv += __popc(bits);
    while (bits) {
      const int64_t u = w * 32 + (__ffs(bits) - 1);
      bits &= bits - 1;
      const bool rst = (uptodate != nullptr) && (uptodate[u] == 0);
      c_rst += rst;
      c_out += (has_msg != nullptr) && (has_msg[u] != 0) && !rst;
    }
  }
  int o_inv = c_inv, o_out = c_out, o_rst = c_rst;
  block_exscan3(o_inv, o_out, o_rst, total, sm);
  for (int64_t w = w0; w < w1; ++w) {
    uint32_t bits = bitmap[w];
    if (bits) bitmap[w] = 0u;
    while (bits) {
      const int64_t u = w * 32 + (__ffs(bits) - 1);
      bits &= bits - 1;
      if (o_inv < cap) involved[o_inv] = u;
      if (local_index != nullptr) local_index[u] = o_inv;
      ++o_inv;
      const bool rst = (uptodate != nullptr) && (uptodate[u] == 0);
      const bool pend = (has_msg != nullptr) && (has_msg[u] != 0) && !rst;
      int32_t row = pend ? o_out : -1;
      if (rst) {
        if (o_rst < cap) restart_nodes[o_rst] = u;
        if (read_only) {
          if (o_rst < cap) row = restart_base + o_rst;
        } else {
          uptodate[u] = 1;
          if (has_msg != nullptr) has_msg[u] = 0;  // msg_store.clear(nids): memory.py:136
        }
        ++o_rst;
      }
      if (gru_row != nullptr) gru_row[u] = row;
      if (pend) {
        if (o_out < cap) outdated[o_out] = u;
        ++o_out;
      }
    }
  }
  if (tid == 0) {
    counts[0] = total[0] < cap ? total[0] : (int)cap;
    counts[1] = total[1] < cap ? total[1] : (int)cap;
    counts[2] = total[2] < cap ? total[2] : (int)cap;
    if (total[0] > cap && err_flags != nullptr) atomicOr(err_flags, TIGER_ERR_CAPACITY);
  }
}

// Same operator as a thread-block cluster: COMPACT_CTAS CTAs, each owns a contiguous slice of the bitmap (up to
// COMPACT_FAST_WORDS words, i.e. graphs of up to COMPACT_CTAS * COMPACT_FAST_WORDS * 32 ~ 1 M nodes), one warp per
// bitmap word / lane per bit.  The per-node flag reads (uptodate, has_msg) of a word are 32 parallel loads
// instead of a serial walk over its set bits, the flag ballots are kept in shared memory so the write pass
// re-reads nothing, and the ordered output positions come from per-word popcounts + one block scan + the slice
// totals of the lower-ranked CTAs read through distributed shared memory.  On one SM the kernel spent ~19 k
// cycles (in-kernel trace: 5-7 k in the flag loads, 7 k in the output stores - one SM's load/store path
// serving the whole graph); spread over the cluster each SM handles an eighth of both.
#define COMPACT_FAST_WORDS 4096
#define COMPACT_CTAS 8
__global__ void __launch_bounds__(1024)
compact_involved_cluster_kernel(uint32_t* __restrict__ bitmap, int n_words, int chunk, int64_t n_nodes,
                                uint8_t* __restrict__ has_msg, uint8_t* __restrict__ uptodate,
                                int64_t* __restrict__ involved, int64_t cap, int64_t* __restrict__ local_index,
                                int64_t* __restrict__ outdated, int32_t* __restrict__ gru_row,
                                int64_t* __restrict__ restart_nodes, int32_t* __restrict__ counts,
                                uint32_t* __restrict__ err_flags, int read_only, int restart_base) {
  extern __shared__ uint32_t cw[];           // [3][chunk] masks (member, restart, pending) then [3][chunk] offsets
  uint32_t* m_mem = cw;
  uint32_t* m_rst = cw + chunk;
  uint32_t* m_out = cw + 2 * chunk;
  int* off = reinterpret_cast<int*>(cw + 3 * chunk);   // [3][chunk]
  __shared__ int sm[3][32];
  __shared__ int total[3];                   // this slice's totals (involved, outdated, restart): read by the peers
  __shared__ int peer[COMPACT_CTAS][3];
  const int tid = threadIdx.x, lane = lane_id(), warp = warp_id_in_block();
  const int rank = (int)cluster_cta_rank();
  const int w_begin = rank * chunk < n_words ? rank * chunk : n_words;
  const int nw = (w_begin + chunk < n_words ? w_begin + chunk : n_words) - w_begin;
  pdl_trigger();
  pdl_wait();      // the finder marks the bitmap
  // ---- phase 0: the bitmap slice (one load per thread), so the flag loads below depend on shared memory only ----
  for (int w = tid; w < nw; w += 1024) m_mem[w] = bitmap[w_begin + w];
  __syncthreads();
  // ---- phase 1: flags of every member node, CW words per warp in flight ----
  constexpr int CW = 4;
  for (int w0 = warp * CW; w0 < nw; w0 += 32 * CW) {
    uint32_t bits[CW];
    uint8_t up[CW], hm[CW];
#pragma unroll
    for (int i = 0; i < CW; ++i) {
      const int w = w0 + i;
      bits[i] = w < nw ? m_mem[w] : 0u;
      up[i] = 1;
      hm[i] = 0;
      const int64_t u = (int64_t)(w_begin + w) * 32 + lane;
      if ((bits[i] >> lane) & 1u) {
        if (uptodate != nullptr) up[i] = uptodate[u];
        if (has_msg != nullptr) hm[i] = has_msg[u];
      }
    }
#pragma unroll
    for (int i = 0; i < CW; ++i) {
      const int w = w0 + i;
      const bool member = (bits[i] >> lane) & 1u;
      const bool rst = member && uptodate != nullptr && up[i] == 0;
      const bool pend = member && hm[i] != 0 && !rst;
      const uint32_t br = __ballot_sync(TIGER_FULL_MASK, rst), bp = __ballot_sync(TIGER_FULL_MASK, pend);
      if (lane == 0 && w < nw) {
        m_rst[w] = br;
        m_out[w] = bp;
      }
    }
  }
  __syncthreads();
  // ---- phase 2: ordered output offsets of every word (slice-relative), then the cluster-wide bases ----
  const int wpt = (nw + 1023) / 1024;
  const int a0 = tid * wpt < nw ? tid * wpt : nw, a1 = (a0 + wpt < nw) ? a0 + wpt : nw;
  int c_inv = 0, c_out = 0, c_rst = 0;
  for (int w = a0; w < a1; ++w) {
    c_inv += __popc(m_mem[w]);
    c_rst += __popc(m_rst[w]);
    c_out += __popc(m_out[w]);
  }
  int o_inv = c_inv, o_out = c_out, o_rst = c_rst;
  block_exscan3(o_inv, o_out, o_rst, total, sm);
  for (int w = a0; w < a1; ++w) {
    off[w] = o_inv;
    off[chunk + w] = o_rst;
    off[2 * chunk + w] = o_out;
    o_inv += __popc(m_mem[w]);
    o_rst += __popc(m_rst[w]);
    o_out += __popc(m_out[w]);
  }
  cluster_sync_all();                        // every slice's totals are published (and this CTA's offsets complete)
  if (tid < COMPACT_CTAS * 3) {
    const uint32_t addr = cluster_map_shared(smem_addr_u32(total) + (uint32_t)(tid % 3) * 4u, (uint32_t)(tid / 3));
    int v;
    asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    peer[tid / 3][tid % 3] = v;
  }
  cluster_sync_all();                        // nobody reads a peer's shared memory after this point
  int base[3] = {0, 0, 0}, grand[3] = {0, 0, 0};   // order of total[]: involved, outdated, restart
#pragma unroll
  for (int r = 0; r < COMPACT_CTAS; ++r)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int v = peer[r][k];
      grand[k] += v;
      if (r < rank) base[k] += v;
    }
  // ---- phase 3: independent stores, lane = bit ----
  const uint32_t lt = (1u << lane) - 1u;
  for (int w = warp; w < nw; w += 32) {
    const uint32_t bits = m_mem[w];
    if (bits == 0u) continue;
    const uint32_t br = m_rst[w], bp = m_out[w];
    if (lane == 0) bitmap[w_begin + w] = 0u;
    if (!((bits >> lane) & 1u)) continue;
    const int64_t u = (int64_t)(w_begin + w) * 32 + lane;
    const int r_inv = base[0] + off[w] + __popc(bits & lt);
    if (r_inv < cap) involved[r_inv] = u;
    if (local_index != nullptr) local_index[u] = r_inv;
    const bool rst = (br >> lane) & 1u, pend = (bp >> lane) & 1u;
    const int r_out = base[1] + off[2 * chunk + w] + __popc(bp & lt);
    int32_t row = pend ? r_out : -1;
    if (rst) {
      const int r = base[2] + off[chunk + w] + __popc(br & lt);
      if (r < cap) restart_nodes[r] = u;
      if (read_only) {
        if (r < cap) row = restart_base + r;
      } else {
        uptodate[u] = 1;
        if (has_msg != nullptr) has_msg[u] = 0;  // msg_store.clear(nids): memory.py:136
      }
    }
    if (gru_row != nullptr) gru_row[u] = row;
    if (pend && r_out < cap) outdated[r_out] = u;
  }
  if (rank == 0 && tid == 0) {
    counts[0] = grand[0] < cap ? grand[0] : (int)cap;
    counts[1] = grand[1] < cap ? grand[1] : (int)cap;
    counts[2] = grand[2] < cap ? grand[2] : (int)cap;
    if (grand[0] > cap && err_flags != nullptr) atomicOr(err_flags, TIGER_ERR_CAPACITY);
  }
}

extern "C" int tiger_compact_involved_ex(uint32_t* bitmap, int64_t n_nodes, uint8_t* has_msg, uint8_t* uptodate,
                                         int64_t* involved, int64_t cap_involved, int64_t* local_index,
                                         int64_t* outdated, int32_t* gru_row, int64_t* restart_nodes,
                                         int32_t* counts, uint32_t* err_flags, int read_only, int restart_base,
                                         void* stream) {
  if (n_nodes <= 0 || cap_involved <= 0 || counts == nullptr || involved == nullptr) return TIGER_EINVAL;
  if (has_msg != nullptr && outdated == nullptr) return TIGER_EINVAL;
  if (uptodate != nullptr && restart_nodes == nullptr) return TIGER_EINVAL;
  if (read_only && (restart_base < 0 || (int64_t)restart_base + cap_involved > (int64_t)INT32_MAX)) return TIGER_EINVAL;
  read_only = read_only ? 1 : 0;
  const int64_t n_words = (n_nodes + 31) / 32;
  if (n_words <= (int64_t)COMPACT_CTAS * COMPACT_FAST_WORDS) {
    static bool configured = false;
    if (!configured) {
      if (cudaFuncSetAttribute(compact_involved_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               COMPACT_FAST_WORDS * 6 * (int)sizeof(uint32_t)) != cudaSuccess)
        return TIGER_ECUDA;
      configured = true;
    }
    const int chunk = (int)((n_words + COMPACT_CTAS - 1) / COMPACT_CTAS);
    return tiger_launch_chain(compact_involved_cluster_kernel, dim3(COMPACT_CTAS), dim3(1024),
                              (size_t)chunk * 6 * sizeof(uint32_t), as_stream(stream), dim3(COMPACT_CTAS, 1, 1), bitmap,
                              (int)n_words, chunk, n_nodes, has_msg, uptodate, involved, cap_involved, local_index, outdated,
                              gru_row, restart_nodes, counts, err_flags, read_only, restart_base);
  }
  compact_involved_kernel<<<1, 1024, 0, as_stream(stream)>>>(bitmap, n_words, has_msg, uptodate, involved,
                                                            cap_involved, local_index, outdated, gru_row,
                                                            restart_nodes, counts, err_flags, read_only, restart_base);
  return tiger_launch_status();
}

extern "C" int tiger_compact_involved(uint32_t* bitmap, int64_t n_nodes, uint8_t* has_msg, uint8_t* uptodate,
                                      int64_t* involved, int64_t cap_involved, int64_t* local_index,
                                      int64_t* outdated, int32_t* gru_row, int64_t* restart_nodes,
                                      int32_t* counts, uint32_t* err_flags, void* stream) {
  return tiger_compact_involved_ex(bitmap, n_nodes, has_msg, uptodate, involved, cap_involved, local_index, outdated,
                                   gru_row, restart_nodes, counts, err_flags, 0, 0, stream);
}
