// K2  fused pending-message gather + GRUCell memory update on the tcgen05 tensor cores.
// Reference: LastMessageAggregatorNoGradLastOnly.forward (message_modules.py:150-160) gathers
// msg rows, TIGE.apply_messages (tiger.py:339-356) gathers the update-source memory rows and
// GRUUpdater.forward (update_modules.py:30-37) runs nn.GRUCell (gate order r,z,n):
//   r = s(Wir x + bir + Whr h + bhr)   z = s(Wiz x + biz + Whz h + bhz)
//   n = tanh(Win x + bin + r*(Whn h + bhn))   h' = (h - n)*z + n
//
// One output tile = 128 gathered rows x U = 48 hidden units, computed by a CLUSTER OF TWO CTAs that split the
// K loop in halves (at O ~ 1,900 rows there are only 15 x 4 tiles for 148 SMs, and a CTA's time is its number
// of K stages).  Accumulator set in TMEM: [128 x 4U] fp32 with the column groups [ Win x | r | z | Whn h ].
// The K loop runs over the message columns first (x phase: one MMA of N = 3U per k-step into
// [Win x | r | z], weight tile rows [n | r | z] of weight_ih) and then over the state columns (h phase:
// N = 2U accumulating into [r | z] and N = U into [Whn h], weight tile rows [r | z | n] of weight_hh), in
// tf32x3 (umma.cuh) so the result keeps fp32 accuracy.  Each CTA leaves its partial tile in shared memory;
// after a cluster barrier CTA r adds both partials of rows [64r, 64r + 64) through distributed shared
// memory (fixed order: deterministic) and applies the gates.
//
// Data movement (everything the tensor core reads is produced without shared-memory traffic from the SM):
//   activations  the 16 producer warps (2 groups x 8 warps; two threads per row, 64 bytes each) gather
//                one 128-byte line of every row per stage straight from the node-indexed tables (no
//                [O, M] staging copy in HBM), split it into tf32 head / tail and write it into a 2-stage
//                ring in TENSOR MEMORY (tcgen05.st); the MMAs take A from TMEM and run at the math floor
//                (tools/umma_bench.cu).  A stage is always refilled by the group that filled it before:
//                an mbarrier wait only distinguishes two phases, so a group that skipped a phase of a
//                stage's barrier could run a full round ahead of the tensor core.
//   weights      pre-split once per parameter update (tiger_gru_pack) into the shared-memory image of
//                every stage; one TMA bulk copy per stage into a 6-stage ring
//   MMA issue    two warps (one elected thread each): X issues the cross terms tail*head + head*tail
//                into accumulator set 0, Y the head*head terms into set 1 (the tensor core truncates when
//                it accumulates, a bias that grows with the number of accumulation steps: the K split
//                halves the steps per accumulator); 2 sets x 192 + 2 x 64 activation columns = 512 TMEM columns
//   epilogue     the producer warps add the two sets out of TMEM into the shared-memory partial tile
//
// The same kernel runs the first layer of MergeUpdater (update_modules.py:40-47, MergeLayer, basic_modules.py:8-20):
// relu(fc1 [x | h] + b1) is the n-gate column group without r and z - the x phase multiplies the message columns of
// fc1 into [Win x], the h phase its state columns into [Whn h] (tiger_merge_pack puts them at the n rows of each
// stage), the [r | z] MMAs are skipped and the epilogue is relu(Win x + Whn h + b1).  With x_by_row the message row
// of result row r is x_table row r (the hidden rows of MLPMessageFunction, computed per outdated row upstream)
// instead of x_table row node_ids[r]; h, the message timestamps and the invariant checks stay node-indexed.
#include "common.cuh"
#include "umma.cuh"

#ifdef TIGER_TRACE
#include <cstdio>
#define GTRACE_DECL long long tr_t[48]; int tr_n = 0; const bool tr_on = blockIdx.x == 0 && (blockIdx.y == 0 || blockIdx.y == 7) && lane == 0;
#define GTRACE_MARK() do { if (tr_on && tr_n < 48) tr_t[tr_n++] = clock64(); } while (0)
#define GTRACE_DUMP(tag, id) do { if (tr_on) for (int i_ = 0; i_ < tr_n; ++i_) printf("%s y%d z%d w%d #%d %lld\n", tag, blockIdx.y, blockIdx.z, id, i_, tr_t[i_] - tr_base); } while (0)
#else
#define GTRACE_DECL
#define GTRACE_MARK() do { } while (0)
#define GTRACE_DUMP(tag, id) do { } while (0)
#endif

#define GRU_PRODUCER_WARPS 16
#define GRU_GROUPS 2                   // producer groups: group g fills activation stage g (GROUPS <= A_STAGES, see below)
#define GRU_GROUP_WARPS (GRU_PRODUCER_WARPS / GRU_GROUPS)
#define GRU_ISSUERS 2
#define GRU_THREADS ((GRU_PRODUCER_WARPS + GRU_ISSUERS + 1) * 32)   // + the TMA warp
#define GRU_BM 128
#define GRU_U 48                       // hidden units per tile (multiple of 16)
#define GRU_KPARTS 2                   // CTAs per tile (cluster size): each runs half of the K stages
#define GRU_WROWS (3 * GRU_U)          // weight rows per stage
#define GRU_ACC_COLS (4 * GRU_U)       // one accumulator set: [ Win x | r | z | Whn h ]
#define GRU_SETS 2
#define GRU_A_STAGES 2
#define GRU_W_STAGES 6
#define GRU_A_RING (GRU_SETS * GRU_ACC_COLS)                          // first TMEM column of the activation ring
#define GRU_TMEM_COLS 512
#define GRU_W_STAGE_FLOATS UMMA_PACK_STAGE_FLOATS(GRU_WROWS)
#define GRU_SMEM_BYTES (GRU_W_STAGES * GRU_W_STAGE_FLOATS * 4 + 4 * GRU_U * 4 + 256)
#define GRU_RED_LD (GRU_ACC_COLS + 4)   // row stride of the partial tile parked in the (idle) weight ring
static_assert(GRU_BM * GRU_RED_LD <= GRU_W_STAGES * GRU_W_STAGE_FLOATS, "partial tile must fit the weight ring");
static_assert(GRU_SETS * GRU_ACC_COLS + GRU_A_STAGES * 2 * TS_BK <= GRU_TMEM_COLS, "TMEM budget");

struct GruArgs {
  const int64_t* node_ids;
  const int32_t* count;
  int64_t n_rows;
  const float* x_table;
  int64_t x_stride;
  const float* h_table;
  int64_t h_stride;
  int m_dim, d;
  const float* wpack;  // tiger_gru_pack: pre-split gate weights, one contiguous stage image per (unit tile, k-block)
  const float* b_ih;
  const float* b_hh;
  float* h_new;
  const float* msg_ts;
  const float* check_mem_ts;
  int check_equal;
  uint32_t* err_flags;
  int vec_x, vec_h;
  int x_by_row;        // x row r is x_table[r] instead of x_table[node_ids[r]]
  int merge;           // MergeLayer first layer: out = relu(fc1_x x + fc1_h h + b1), b1 in b_ih
};

__global__ void __launch_bounds__(GRU_THREADS, 1) gru_update_kernel(const GruArgs g) {
  extern __shared__ __align__(128) unsigned char gru_smem[];
  float* wstage0 = reinterpret_cast<float*>(gru_smem);
  float* bias_s = wstage0 + (size_t)GRU_W_STAGES * GRU_W_STAGE_FLOATS;   // [4][GRU_U]: b_r, b_z, b_in, b_hn
  uint64_t* a_full = reinterpret_cast<uint64_t*>(bias_s + 4 * GRU_U);
  uint64_t* a_empty = a_full + GRU_A_STAGES;
  uint64_t* w_full = a_empty + GRU_A_STAGES;
  uint64_t* w_empty = w_full + GRU_W_STAGES;
  uint64_t* done = w_empty + GRU_W_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

#ifdef TIGER_TRACE
  const long long tr_base = clock64();
#endif
  pdl_trigger();
  pdl_wait();      // the row count and the row list come from the compaction kernel
  int64_t n = g.n_rows;
  if (g.count != nullptr) {
    const int64_t c = *g.count;
    n = c < n ? c : n;
  }
  const int64_t row0 = (int64_t)blockIdx.y * GRU_BM;
  if (row0 >= n) return;
  const int j0 = blockIdx.x * GRU_U;
  const int d = g.d, m_dim = g.m_dim;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // producers: the id of this thread's row is in flight while the barriers / TMEM allocation are set up
  int64_t prod_u = 0;
  if (warp < GRU_PRODUCER_WARPS) {
    int64_t r = row0 + (warp & 3) * 32 + lane;
    r = r < n ? r : n - 1;
    prod_u = g.node_ids != nullptr ? g.node_ids[r] : r;
  }
  if (tid < GRU_U && g.merge) {
    const int j = j0 + tid;
    bias_s[tid] = bias_s[GRU_U + tid] = bias_s[3 * GRU_U + tid] = 0.f;
    bias_s[2 * GRU_U + tid] = j < d ? g.b_ih[j] : 0.f;
  } else if (tid < GRU_U) {
    const int j = j0 + tid;
    const bool ok = j < d;
    bias_s[tid] = ok ? g.b_ih[j] + g.b_hh[j] : 0.f;
    bias_s[GRU_U + tid] = ok ? g.b_ih[d + j] + g.b_hh[d + j] : 0.f;
    bias_s[2 * GRU_U + tid] = ok ? g.b_ih[2 * d + j] : 0.f;
    bias_s[3 * GRU_U + tid] = ok ? g.b_hh[2 * d + j] : 0.f;
  }
  if (tid == GRU_PRODUCER_WARPS * 32) {
    for (int s = 0; s < GRU_A_STAGES; ++s) {
      mbar_init(a_full + s, GRU_GROUP_WARPS);
      mbar_init(a_empty + s, GRU_ISSUERS);
    }
    for (int s = 0; s < GRU_W_STAGES; ++s) {
      mbar_init(w_full + s, 1);
      mbar_init(w_empty + s, GRU_ISSUERS);
    }
    mbar_init(done, GRU_ISSUERS);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, GRU_TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t taddr = *tmem_slot;
  GTRACE_DECL
  GTRACE_MARK();   // #0 setup done
  const int nbx = (m_dim + TS_BK - 1) / TS_BK, nbh = (d + TS_BK - 1) / TS_BK;
  const int n_blocks = nbx + nbh;
  // this CTA's share of the K stages: [b0, b1)
  const int part = (int)blockIdx.z;
  const int per_part = (n_blocks + GRU_KPARTS - 1) / GRU_KPARTS;
  const int b0 = part * per_part < n_blocks ? part * per_part : n_blocks;
  const int b1 = b0 + per_part < n_blocks ? b0 + per_part : n_blocks;
  const int n_loc = b1 - b0;
  const bool has_x = n_loc > 0 && b0 < nbx, has_h = n_loc > 0 && b1 > nbx;
  // gate stage (after the cluster barrier): this CTA finishes rows [RB * rank, RB * (rank + 1)) of the tile, one item =
  // one row x 4 units; a thread owns items tid and tid + GRU_THREADS.  The previous state h of an item is fetched
  // before the barrier (gate_prefetch) so that only shared-memory traffic and math remain behind it.
  constexpr int GATE_RB = GRU_BM / GRU_KPARTS, GATE_Q = GRU_U / 4, GATE_ITEMS = 2;
  static_assert(GATE_RB * GATE_Q <= GATE_ITEMS * GRU_THREADS, "gate items per thread");
  const int gate_r0 = (int)cluster_cta_rank() * GATE_RB;
  float4 gate_h[GATE_ITEMS];
  auto gate_prefetch = [&]() {
#pragma unroll
    for (int it = 0; it < GATE_ITEMS; ++it) {
      const int i = tid + it * GRU_THREADS;
      const int rl = gate_r0 + i / GATE_Q, c = (i % GATE_Q) * 4;
      const int64_t r = row0 + rl;
      const int j = j0 + c;
      gate_h[it] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (!g.merge && i < GATE_RB * GATE_Q && r < n && j < d) {
        const int64_t u = g.node_ids != nullptr ? g.node_ids[r] : r;
        gate_h[it] = umma_load_chunk(g.h_table + u * g.h_stride, j, d, g.vec_h != 0);
      }
    }
  };

  if (warp < GRU_PRODUCER_WARPS) {
    // ---------------- producers: two threads per row ----------------
    const int grp = warp / GRU_GROUP_WARPS, wg = warp % GRU_GROUP_WARPS;
    const int q = wg & 3, half = wg >> 2;        // TMEM lane quadrant of this warp, which 16 floats of the stage
    const int rl = q * 32 + lane;
    // rows beyond the count read the last valid row: they only feed accumulator rows nobody stores
    int64_t r = row0 + rl;
    const bool live = r < n;
    r = live ? r : n - 1;
    const int64_t u = prod_u;
    const float* xp = g.x_table + (g.x_by_row ? r : u) * g.x_stride;
    const float* hp = g.h_table + u * g.h_stride;
    if (live && warp < 4 && g.check_mem_ts != nullptr && blockIdx.x == 0 && part == 0 && g.err_flags != nullptr) {
      const float mt = g.msg_ts[u], pt = g.check_mem_ts[u];
      if (pt > mt) atomicOr(g.err_flags, TIGER_ERR_MSG_BEFORE_MEM);                    // message_modules.py:157-159
      if (g.check_equal && mt != pt) atomicOr(g.err_flags, TIGER_ERR_MSG_TS_MISMATCH);  // tiger.py:324-327
    }
    const uint32_t tl = taddr + GRU_A_RING + ((uint32_t)(q * 32) << 16) + 16u * half;
    float4 v[4];
    auto load = [&](int blk) {
      const bool xph = blk < nbx;
      const float* p = xph ? xp : hp;
      const int k0 = (xph ? blk : blk - nbx) * TS_BK + 16 * half, kdim = xph ? m_dim : d;
      if ((xph ? g.vec_x : g.vec_h) != 0 && k0 + 16 <= kdim) {
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = __ldg(reinterpret_cast<const float4*>(p + k0) + i);
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = umma_load_chunk(p, k0 + 4 * i, kdim, false);
      }
    };
    GTRACE_MARK();   // #1 pointers resolved
    if (grp < n_loc) load(b0 + grp);
    for (int lb = grp; lb < n_loc; lb += GRU_GROUPS) {
      const int s = lb % GRU_A_STAGES;
      mbar_wait(a_empty + s, ((lb / GRU_A_STAGES) & 1) ^ 1);
      float hi[16], lo[16];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float4 h, l;
        tf32_split(v[i], h, l);
        hi[4 * i] = h.x; hi[4 * i + 1] = h.y; hi[4 * i + 2] = h.z; hi[4 * i + 3] = h.w;
        lo[4 * i] = l.x; lo[4 * i + 1] = l.y; lo[4 * i + 2] = l.z; lo[4 * i + 3] = l.w;
      }
      const uint32_t ts = tl + (uint32_t)(s * 2 * TS_BK);
      tmem_st16(ts, hi);
      tmem_st16(ts + TS_BK, lo);
      tmem_wait_st();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full + s);
      GTRACE_MARK();   // stage published
      // this group's next line is in flight while the other group's stage is written / consumed
      if (lb + GRU_GROUPS < n_loc) load(b0 + lb + GRU_GROUPS);
    }
    // ---------------- partial tile: TMEM -> shared memory ----------------
    GTRACE_MARK();   // producer loop done
    gate_prefetch();
    mbar_wait(done, 0);
    GTRACE_MARK();   // MMAs done
    tc_fence_after_sync();
    const uint32_t tacc = taddr + ((uint32_t)(q * 32) << 16);   // q == warp & 3: same rows as in the producer role
    float* red = wstage0 + rl * GRU_RED_LD;                       // the weight ring is idle once `done` has fired
    for (int c0 = (warp >> 2) * 16; c0 < GRU_ACC_COLS; c0 += 16 * (GRU_PRODUCER_WARPS / 4)) {
      float a[16], t[16];
      tmem_ld16(tacc + (uint32_t)c0, a);
      tmem_ld16(tacc + (uint32_t)(GRU_ACC_COLS + c0), t);
      // column groups this CTA's stages never touched hold no sum (U is a multiple of 16: a chunk lies in one group)
      const bool valid = c0 < GRU_U ? has_x : (c0 < 3 * GRU_U ? (has_x || has_h) && !g.merge : has_h);
#pragma unroll
      for (int e = 0; e < 16; e += 4)
        *reinterpret_cast<float4*>(red + c0 + e) =
            valid ? make_float4(a[e] + t[e], a[e + 1] + t[e + 1], a[e + 2] + t[e + 2], a[e + 3] + t[e + 3])
                  : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else if (warp == GRU_PRODUCER_WARPS + GRU_ISSUERS) {
    // ---------------- TMA warp: one bulk copy per stage brings both planes of the weight tile ----------------
    if (lane == 0) {
      const uint32_t bytes = (uint32_t)GRU_W_STAGE_FLOATS * 4u;
      const float* src = g.wpack + ((int64_t)blockIdx.x * n_blocks + b0) * GRU_W_STAGE_FLOATS;
      for (int blk = 0; blk < n_loc; ++blk) {
        const int s = blk % GRU_W_STAGES;
        mbar_wait(w_empty + s, ((blk / GRU_W_STAGES) & 1) ^ 1);
        mbar_arrive_expect_tx(w_full + s, bytes);
        tma_bulk_load(wstage0 + (size_t)s * GRU_W_STAGE_FLOATS, src + (int64_t)blk * GRU_W_STAGE_FLOATS, bytes,
                      w_full + s);
      }
    }
    __syncwarp();
    gate_prefetch();
  } else {
    // ---------------- MMA issuers: X (cross terms) and Y (head*head) ----------------
    // The whole warp runs the loop so that every operand stays warp-uniform; only the tcgen05 instructions
    // are issued by the elected lane.
    const bool is_x = uniform_warp_idx() == GRU_PRODUCER_WARPS;
    const uint32_t id3 = umma_idesc_tf32(GRU_BM, 3 * GRU_U), id2 = umma_idesc_tf32(GRU_BM, 2 * GRU_U),
                   id1 = umma_idesc_tf32(GRU_BM, GRU_U);
    const uint32_t tbase = __shfl_sync(0xffffffffu, taddr, 0);
    const uint32_t a_ring = tbase + GRU_A_RING;
    const uint32_t b_hi0 = umma_desc_lo(smem_addr_u32(wstage0), GRU_WROWS);
    const uint32_t b_plane = (uint32_t)(TS_KCH * GRU_WROWS * 16) >> 4;      // head plane -> tail plane, 16-byte units
    const uint32_t b_stage = (uint32_t)(GRU_W_STAGE_FLOATS * 4) >> 4, b_kstep = 2u * GRU_WROWS;
    bool ready_a = mbar_test(a_full, 0), ready_w = mbar_test(w_full, 0);
    const int first_h = b0 > nbx ? b0 : nbx;      // first h-phase block of this part (if it has one)
    for (int lb = 0; lb < n_loc; ++lb) {
      const int blk = b0 + lb;
      const int sa = lb % GRU_A_STAGES, sw = lb % GRU_W_STAGES;
      mbar_wait_probed(ready_a, a_full + sa, (lb / GRU_A_STAGES) & 1);
      mbar_wait_probed(ready_w, w_full + sw, (lb / GRU_W_STAGES) & 1);
      GTRACE_MARK();   // stage ready
      tc_fence_after_sync();
      // probe the next stage now: the probes' latency overlaps the MMA issue below
      const int nb = lb + 1;
      ready_a = nb < n_loc ? mbar_test(a_full + nb % GRU_A_STAGES, (nb / GRU_A_STAGES) & 1) : true;
      ready_w = nb < n_loc ? mbar_test(w_full + nb % GRU_W_STAGES, (nb / GRU_W_STAGES) & 1) : true;
      if (elect_one()) {
        const uint32_t a_hi = a_ring + (uint32_t)(sa * 2 * TS_BK), a_lo = a_hi + TS_BK;
        const uint32_t b_hi = b_hi0 + (uint32_t)sw * b_stage, b_lo = b_hi + b_plane;
        const bool xph = blk < nbx;
        // the first MMA into a column group overwrites it: [Win x] and (with x stages) [r | z] at the first x
        // block, [Whn h] (and [r | z] of a part without x stages) at the first h block
        const bool first = xph ? blk == b0 : blk == first_h;
        const uint32_t acc = tbase + (is_x ? 0u : (uint32_t)GRU_ACC_COLS);   // set 0: cross terms, set 1: head*head
#pragma unroll
        for (int j = 0; j < TS_BK / 8; ++j) {
          const uint32_t ah = a_hi + 8u * j, al = a_lo + 8u * j, bh = b_hi + b_kstep * j, bl = b_lo + b_kstep * j;
          const uint32_t fresh = (first && j == 0) ? 0u : 1u;
          const uint32_t fresh_rz = (first && j == 0 && !has_x) ? 0u : 1u;
          if (g.merge) {
            // [Win x] from the stage's n rows (x phase), [Whn h] likewise (h phase); no r / z products
            const uint32_t acc_n = acc + (xph ? 0u : 3u * GRU_U), b_n = xph ? 0u : 2u * GRU_U;
            if (is_x) {
              umma_tf32_ts(acc_n, al, bh + b_n, id1, fresh);
              umma_tf32_ts(acc_n, ah, bl + b_n, id1, 1u);
            } else {
              umma_tf32_ts(acc_n, ah, bh + b_n, id1, fresh);
            }
          } else if (is_x) {
            if (xph) {
              // weight tile rows [n | r | z] -> columns [0, 3U)
              umma_tf32_ts(acc, al, bh, id3, fresh);
              umma_tf32_ts(acc, ah, bl, id3, 1u);
            } else {
              // weight tile rows [r | z | n] -> [r | z] accumulate at column U, Whn h starts at column 3U
              umma_tf32_ts(acc + GRU_U, al, bh, id2, fresh_rz);
              umma_tf32_ts(acc + GRU_U, ah, bl, id2, 1u);
              umma_tf32_ts(acc + 3 * GRU_U, al, bh + 2 * GRU_U, id1, fresh);
              umma_tf32_ts(acc + 3 * GRU_U, ah, bl + 2 * GRU_U, id1, 1u);
            }
          } else {
            if (xph) {
              umma_tf32_ts(acc, ah, bh, id3, fresh);
            } else {
              umma_tf32_ts(acc + GRU_U, ah, bh, id2, fresh_rz);
              umma_tf32_ts(acc + 3 * GRU_U, ah, bh + 2 * GRU_U, id1, fresh);
            }
          }
        }
        umma_commit(a_empty + sa);
        umma_commit(w_empty + sw);
      }
      __syncwarp();
    }
    if (elect_one()) {
      if (n_loc > 0)
        umma_commit(done);
      else
        mbar_arrive(done);
    }
    __syncwarp();
    gate_prefetch();
  }
  // ---------------- cluster reduction + gates ----------------
  __syncwarp();
  GTRACE_MARK();   // role done
  cluster_sync_all();                         // both partial tiles are in place
  GTRACE_MARK();   // cluster sync 1
  {
    const uint32_t red0 = smem_addr_u32(wstage0);
    const bool vec_out = (d & 3) == 0 && ((((uintptr_t)g.h_new) & 15) == 0);
    float4 acc[GATE_ITEMS][4];                  // Win x, r, z, Whn h
#pragma unroll
    for (int it = 0; it < GATE_ITEMS; ++it) {   // all partial-tile reads of both items are issued before any math
      const int i = tid + it * GRU_THREADS;
      const int rl = gate_r0 + i / GATE_Q, c = (i % GATE_Q) * 4;
      const bool on = i < GATE_RB * GATE_Q && row0 + rl < n && j0 + c < d;
#pragma unroll
      for (int gi = 0; gi < 4; ++gi) {
        acc[it][gi] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (on) {
          const uint32_t off = red0 + (uint32_t)(rl * GRU_RED_LD + gi * GRU_U + c) * 4u;
          acc[it][gi] = cluster_ld_f4(cluster_map_shared(off, 0));
#pragma unroll
          for (int pp = 1; pp < GRU_KPARTS; ++pp) {
            const float4 t = cluster_ld_f4(cluster_map_shared(off, (uint32_t)pp));
            acc[it][gi].x += t.x; acc[it][gi].y += t.y; acc[it][gi].z += t.z; acc[it][gi].w += t.w;
          }
        }
      }
    }
#pragma unroll
    for (int it = 0; it < GATE_ITEMS; ++it) {
      const int i = tid + it * GRU_THREADS;
      const int rl = gate_r0 + i / GATE_Q, c = (i % GATE_Q) * 4;
      const int64_t r = row0 + rl;
      const int j = j0 + c;
      if (i >= GATE_RB * GATE_Q || r >= n || j >= d) continue;
      const float an[4] = {acc[it][0].x, acc[it][0].y, acc[it][0].z, acc[it][0].w};
      const float ar[4] = {acc[it][1].x, acc[it][1].y, acc[it][1].z, acc[it][1].w};
      const float az[4] = {acc[it][2].x, acc[it][2].y, acc[it][2].z, acc[it][2].w};
      const float ah[4] = {acc[it][3].x, acc[it][3].y, acc[it][3].z, acc[it][3].w};
      const float hv[4] = {gate_h[it].x, gate_h[it].y, gate_h[it].z, gate_h[it].w};
      float o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (g.merge) {
          o[e] = fmaxf(an[e] + ah[e] + bias_s[2 * GRU_U + c + e], 0.f);
          continue;
        }
        const float rg = sigmoidf_acc(ar[e] + bias_s[c + e]);
        const float zg = sigmoidf_acc(az[e] + bias_s[GRU_U + c + e]);
        const float nn = tanhf((an[e] + bias_s[2 * GRU_U + c + e]) + rg * (ah[e] + bias_s[3 * GRU_U + c + e]));
        o[e] = (hv[e] - nn) * zg + nn;
      }
      float* dst = g.h_new + r * d + j;
      if (vec_out && j + 4 <= d) {
        *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (j + e < d) dst[e] = o[e];
      }
    }
  }
  GTRACE_MARK();   // gates done
  cluster_sync_all();                         // nobody leaves while its partner still reads its tile
  GTRACE_MARK();   // cluster sync 2
#ifdef TIGER_TRACE
  if (warp == 0 || warp == 8 || warp >= GRU_PRODUCER_WARPS) GTRACE_DUMP(warp < GRU_PRODUCER_WARPS ? "producer" : (warp == GRU_PRODUCER_WARPS + GRU_ISSUERS ? "tma" : "issuer"), warp);
#endif
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(taddr, GRU_TMEM_COLS);
}

// Gate-weight pack: for unit tile t and k-block kb (x phase: kb < nbx over weight_ih, rows [n | r | z]; h phase over
// weight_hh, rows [r | z | n]) the stage image [head plane | tail plane][kc][3U rows][4 floats].  Merge pack (w_hh
// NULL, w_ih = fc1 [d][m_dim + d]): the message columns of fc1 at the x stages' n rows, its state columns at the h
// stages' n rows, zeros elsewhere.
__global__ void gru_pack_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh, int m_dim, int d,
                                int tiles, int nbx, int nbh, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int n_kb = nbx + nbh;
  const int64_t total = (int64_t)tiles * n_kb * TS_KCH * GRU_WROWS;
  if (i >= total) return;
  const int r = (int)(i % GRU_WROWS);
  const int kc = (int)((i / GRU_WROWS) % TS_KCH);
  const int kb = (int)((i / (GRU_WROWS * TS_KCH)) % n_kb);
  const int t = (int)(i / ((int64_t)GRU_WROWS * TS_KCH * n_kb));
  const bool xph = kb < nbx;
  const int gi = r / GRU_U, j = t * GRU_U + r % GRU_U;
  const int gate = xph ? (gi == 0 ? 2 : gi - 1) : gi;   // gate order in the weights: r, z, n
  const int kdim = xph ? m_dim : d;
  const int k = (xph ? kb : kb - nbx) * TS_BK + kc * 4;
  const float* row = nullptr;
  if (j < d && w_hh != nullptr)
    row = (xph ? w_ih : w_hh) + (int64_t)(gate * d + j) * kdim;
  else if (j < d && gate == 2)
    row = w_ih + (int64_t)j * (m_dim + d) + (xph ? 0 : m_dim);
  const float4 v = umma_load_chunk(row, k, kdim, false);
  float4 h, l;
  tf32_split(v, h, l);
  float* stage = out + ((int64_t)t * n_kb + kb) * GRU_W_STAGE_FLOATS;
  *reinterpret_cast<float4*>(stage + (kc * GRU_WROWS + r) * 4) = h;
  *reinterpret_cast<float4*>(stage + TS_KCH * GRU_WROWS * 4 + (kc * GRU_WROWS + r) * 4) = l;
}

extern "C" int64_t tiger_gru_pack_bytes(int m_dim, int d) {
  if (m_dim <= 0 || d <= 0) return -1;
  const int64_t tiles = (d + GRU_U - 1) / GRU_U;
  const int64_t n_kb = (m_dim + TS_BK - 1) / TS_BK + (d + TS_BK - 1) / TS_BK;
  return tiles * n_kb * GRU_W_STAGE_FLOATS * (int64_t)sizeof(float);
}

extern "C" int tiger_gru_pack(const float* w_ih, const float* w_hh, int m_dim, int d, float* out, void* stream) {
  if (w_ih == nullptr || w_hh == nullptr || out == nullptr || tiger_gru_pack_bytes(m_dim, d) < 0 ||
      (((uintptr_t)out) & 15) != 0)
    return TIGER_EINVAL;
  const int tiles = (d + GRU_U - 1) / GRU_U;
  const int nbx = (m_dim + TS_BK - 1) / TS_BK, nbh = (d + TS_BK - 1) / TS_BK;
  const int64_t total = (int64_t)tiles * (nbx + nbh) * TS_KCH * GRU_WROWS;
  gru_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(w_ih, w_hh, m_dim, d, tiles, nbx, nbh,
                                                                                 out);
  return tiger_launch_status();
}

extern "C" int tiger_merge_pack(const float* fc1_w, int m_dim, int d, float* out, void* stream) {
  if (fc1_w == nullptr || out == nullptr || tiger_gru_pack_bytes(m_dim, d) < 0 || (((uintptr_t)out) & 15) != 0)
    return TIGER_EINVAL;
  const int tiles = (d + GRU_U - 1) / GRU_U;
  const int nbx = (m_dim + TS_BK - 1) / TS_BK, nbh = (d + TS_BK - 1) / TS_BK;
  const int64_t total = (int64_t)tiles * (nbx + nbh) * TS_KCH * GRU_WROWS;
  gru_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(fc1_w, nullptr, m_dim, d, tiles, nbx,
                                                                                 nbh, out);
  return tiger_launch_status();
}

static int gru_update_launch(const GruArgs& a, void* stream) {
  if (a.n_rows < 0 || a.m_dim <= 0 || a.d <= 0 || a.wpack == nullptr || (((uintptr_t)a.wpack) & 15) != 0 ||
      a.b_ih == nullptr || (!a.merge && a.b_hh == nullptr) || (a.x_by_row && a.node_ids == nullptr))
    return TIGER_EINVAL;
  if (a.n_rows == 0) return TIGER_OK;
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(gru_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GRU_SMEM_BYTES) !=
        cudaSuccess)
      return TIGER_ECUDA;
    configured = true;
  }
  GruArgs g = a;
  g.vec_x = ((((uintptr_t)g.x_table) & 15) == 0 && (g.x_stride & 3) == 0) ? 1 : 0;
  g.vec_h = ((((uintptr_t)g.h_table) & 15) == 0 && (g.h_stride & 3) == 0) ? 1 : 0;
  return tiger_launch_chain(gru_update_kernel,
                            dim3((unsigned)((g.d + GRU_U - 1) / GRU_U), (unsigned)((g.n_rows + GRU_BM - 1) / GRU_BM),
                                 GRU_KPARTS),
                            dim3(GRU_THREADS), GRU_SMEM_BYTES, as_stream(stream), dim3(1, 1, GRU_KPARTS), g);
}

extern "C" int tiger_gru_update(const int64_t* node_ids, const int32_t* count, int64_t n_rows,
                                const float* x_table, int64_t x_stride, const float* h_table, int64_t h_stride,
                                int m_dim, int d, const float* wpack, const float* b_ih, const float* b_hh,
                                float* h_new, const float* msg_ts, const float* check_mem_ts, int check_equal,
                                uint32_t* err_flags, void* stream) {
  GruArgs g{};
  g.node_ids = node_ids; g.count = count; g.n_rows = n_rows;
  g.x_table = x_table; g.x_stride = x_stride; g.h_table = h_table; g.h_stride = h_stride;
  g.m_dim = m_dim; g.d = d; g.wpack = wpack; g.b_ih = b_ih; g.b_hh = b_hh; g.h_new = h_new;
  g.msg_ts = msg_ts; g.check_mem_ts = check_mem_ts; g.check_equal = check_equal; g.err_flags = err_flags;
  return gru_update_launch(g, stream);
}

extern "C" int tiger_gru_update_rows(const int64_t* node_ids, const int32_t* count, int64_t n_rows,
                                     const float* x_table, int64_t x_stride, const float* h_table, int64_t h_stride,
                                     int m_dim, int d, const float* wpack, const float* b_ih, const float* b_hh,
                                     float* h_new, const float* msg_ts, const float* check_mem_ts, int check_equal,
                                     uint32_t* err_flags, void* stream) {
  GruArgs g{};
  g.node_ids = node_ids; g.count = count; g.n_rows = n_rows;
  g.x_table = x_table; g.x_stride = x_stride; g.h_table = h_table; g.h_stride = h_stride;
  g.m_dim = m_dim; g.d = d; g.wpack = wpack; g.b_ih = b_ih; g.b_hh = b_hh; g.h_new = h_new;
  g.msg_ts = msg_ts; g.check_mem_ts = check_mem_ts; g.check_equal = check_equal; g.err_flags = err_flags;
  g.x_by_row = 1;
  return gru_update_launch(g, stream);
}

extern "C" int tiger_merge_update(const int64_t* node_ids, const int32_t* count, int64_t n_rows,
                                  const float* x_table, int64_t x_stride, int x_by_row, const float* h_table,
                                  int64_t h_stride, int m_dim, int d, const float* wpack, const float* b1, float* out,
                                  const float* msg_ts, const float* check_mem_ts, int check_equal, uint32_t* err_flags,
                                  void* stream) {
  GruArgs g{};
  g.node_ids = node_ids; g.count = count; g.n_rows = n_rows;
  g.x_table = x_table; g.x_stride = x_stride; g.h_table = h_table; g.h_stride = h_stride;
  g.m_dim = m_dim; g.d = d; g.wpack = wpack; g.b_ih = b1; g.h_new = out;
  g.msg_ts = msg_ts; g.check_mem_ts = check_mem_ts; g.check_equal = check_equal; g.err_flags = err_flags;
  g.x_by_row = x_by_row != 0; g.merge = 1;
  return gru_update_launch(g, stream);
}
