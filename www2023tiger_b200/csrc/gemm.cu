// fp32-accurate "NT" GEMM on the 5th-generation tensor cores (tcgen05, kind::tf32, tf32x3 split):
//     C[m, n] = act(alpha * (sum_k A[m, k] * W[n, k] + bias[n]))
// A row-major [M, K] (lda), W row-major [N, K] (ldw) - the layout of nn.Linear / in_proj weights, so
// parameters are used as stored (reference: nn.MultiheadAttention in/out projections, nn.Linear and
// MergeLayer of tiger/model/restarters.py:45-50, temporal_agg_modules.py:203-209, basic_modules.py:5-19).
//
// Why tensor cores, and why three passes: the parity bar is fp32 max-norm 1e-5 against the CPU
// reference.  Single-pass TF32 (10-bit mantissa) cannot meet it; splitting every operand into a tf32
// head and tail and accumulating head*tail + tail*head + head*head in the fp32 TMEM accumulator does
// (error ~2^-22 per product), at 3 MMAs per k-step - still several times the FFMA rate, and the MMAs
// run asynchronously to the threads that stage the operands.
//
// Two kernels:
//   gemm_tf32x3_kernel     (tiger_sgemm_ex, tiger_sgemm_nt) both operands staged through shared memory by
//                          the producer warps; either operand may be read transposed
//   gemm_tf32x3_ts_kernel  (tiger_sgemm_nt_packed*) weights pre-split into a pack (tiger_gemm_pack_weight)
//                          and streamed by TMA, activations staged in tensor memory
// Staging kernel (one CTA = one 128 x BN output tile at a time, BN <= 128, 19 warps):
//   warps 0-15 producers in 4 groups of 4 warps; group g fills stages g, g+4, ...: global (L2) ->
//              registers -> tf32 split -> shared memory in the canonical K-major UMMA layout
//              (umma.cuh), 16 floats of K per stage, up to 8 stages, full/empty mbarriers; a group's
//              next loads are issued before it publishes the current stage, and the four groups keep
//              four stages of loads in flight, which is what hides the L2 latency;
//              afterwards the same warps run the epilogue: tcgen05.ld of the partial accumulators
//              (thread = row, 16 columns at a time), bias / alpha / ReLU, 16-byte stores or atomic adds
//   warps 16-18 MMA issuers: one elected thread each issues one of the three tf32x3 product streams
//              into its own TMEM accumulator and commits each stage back to the producers
//              (tcgen05.commit -> mbarrier); see umma.cuh for why three
//   warp 19    idle: it only takes part in the block barriers.  The block shape, and with it the register
//              budget __launch_bounds__ gives every thread, is the one the kernel was tuned and measured at.
// The row count may live on the device (`count` * rows_per_count), which keeps the restart path free of
// host syncs: CTAs whose row block starts beyond it exit before touching TMEM.
#include "common.cuh"
#include "umma.cuh"

#ifdef TIGER_TRACE
#include <cstdio>
#define TRACE_DECL long long tr_t[40]; int tr_n = 0; const bool tr_on = blockIdx.x == 0 && blockIdx.y == 0 && lane == 0;
#define TRACE_MARK() do { if (tr_on && tr_n < 40) tr_t[tr_n++] = clock64(); } while (0)
#define TRACE_DUMP(tag, id) do { if (tr_on) for (int i_ = 0; i_ < tr_n; ++i_) printf("%s %d #%d %lld\n", tag, id, i_, tr_t[i_] - tr_base); } while (0)
#else
#define TRACE_DECL
#define TRACE_MARK() do { } while (0)
#define TRACE_DUMP(tag, id) do { } while (0)
#endif

#define TCG_PRODUCER_WARPS 16
#define TCG_THREADS ((TCG_PRODUCER_WARPS + UMMA_ISSUERS + 1) * 32)   // + the idle warp
#define TCG_BM 128
#define TCG_GROUPS 4                                    // producer groups, each fills every 4th stage
#define TCG_GROUP_WARPS (TCG_PRODUCER_WARPS / TCG_GROUPS)
#define TCG_MAX_BN 128
#define TCG_MAX_STAGES 8
#define TCG_SMEM_BUDGET (200 * 1024)
#define TCG_NA (TCG_BM / 8 / TCG_GROUP_WARPS)           // A warp-chunks per producer warp
#define TCG_NW (TCG_MAX_BN / 8 / TCG_GROUP_WARPS)       // W warp-chunks per producer warp at the widest tile

// Kernel arguments.  "both": read by both kernels; "staging": gemm_tf32x3_kernel only; "packed":
// gemm_tf32x3_ts_kernel only.
struct GemmArgs {
  const float* A;        // both (packed: may be NULL with a gathered A)
  const float* W;        // staging
  const float* wpack;    // packed: pre-split weight pack (tiger_gemm_pack_weight)
  const float* bias;     // both, may be NULL
  float* C;              // both
  const uint8_t* row_zero;  // staging: always NULL (see the note in gemm_tf32x3_kernel)
  const int32_t* count;  // both: device row count (times rows_per_count) or NULL
  int64_t lda, ldw, ldc; // both (ldw: staging)
  int64_t stride_a, stride_w, stride_bias, stride_c;  // staging: always 0 (see the note in gemm_tf32x3_kernel)
  int64_t M, rows_per_count;  // both
  int N, K;              // both
  float alpha;           // both
  int relu;              // both
  int vec_a, vec_w, vec_c;  // both (vec_w: staging): 16-byte alignment of the rows of A / W / C
  int bn, tiles_n, stages;  // both
  uint32_t tmem_cols;    // both
  // staging: either operand may be read transposed (a template parameter of the kernel) - the dgrad / wgrad
  // products of the training step use the tensors as stored; the reduction length may live on the device
  // (k_count * k_rows_per_count); with `accumulate`, blockIdx.y splits K into parts of kblk_per_part stages whose
  // partial tiles are added into C with atomic adds (gradient accumulation)
  int accumulate;
  const int32_t* k_count;
  int64_t k_rows_per_count;
  int kblk_per_part;
  // packed, split output: columns [0, n_lim0) go to C, columns [n_split, n_split + n_lim1) to C2 (C2 may be NULL)
  float* C2;
  int64_t ldc2;
  int n_split, n_lim0, n_lim1, vec_c2;
  // packed, split-K: blockIdx.y = part; with k_parts > 1 the parts of a tile form a thread-block cluster, exchange
  // their partial tiles through distributed shared memory, sum them in part order (deterministic) and write the
  // biased / activated tile once
  int k_parts;
  int late_trigger;      // packed: programmatic-launch trigger only after this kernel's own dependency wait
  // packed, fused row scatter (tiger_left_writeback_fused): rows m < sc_rows with sc_mask[m] also go to
  // sc_table[sc_ids[m]] (columns of the first output), with the row's clock / activity flag
  const int64_t* sc_ids;
  const uint8_t* sc_mask;
  int64_t sc_rows, sc_period, sc_ld;
  const float* sc_ts;
  float* sc_table;
  float* sc_ts_table;
  uint8_t* sc_active;
  uint32_t* sc_err;
  int vec_sc;
  // packed, gathered A: row m of A is row sel[ids[m]] of a_alt when that is >= 0 (or A is NULL), else row ids[m] of
  // A, plus row ids[m] of a_add - the representation lookup of the embedding module (csrc/attention.cu resolve_row)
  // done by the producer warps instead of a gather kernel in front of the GEMM
  const int64_t* a_ids;
  const void* a_sel;
  int a_sel_i64;
  const float* a_alt;
  const float* a_add;
};

// MODE_A / MODE_W: how the operand is fetched - 0 row-major [rows, K] (vector loads along K), 1 transposed
// (element (row, k) at base[k * ld + row], scalar loads).  Template parameters, not runtime switches: loaders
// selected at run time in one body made the kernel spill heavily.
template <int MODE_A, int MODE_W>
__global__ void __launch_bounds__(TCG_THREADS, 1) gemm_tf32x3_kernel(const GemmArgs g) {
  extern __shared__ __align__(128) unsigned char tcg_smem[];
  const int BN = g.bn, S = g.stages;
  const int a_plane = UMMA_KCH * TCG_BM * 4;  // floats
  const int w_plane = UMMA_KCH * BN * 4;
  const int stage_floats = 2 * a_plane + 2 * w_plane;
  float* stage0 = reinterpret_cast<float*>(tcg_smem);
  uint64_t* full = reinterpret_cast<uint64_t*>(tcg_smem + (size_t)S * stage_floats * sizeof(float));
  uint64_t* empty = full + TCG_MAX_STAGES;
  uint64_t* done = empty + TCG_MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  int64_t M = g.M;
  if (g.count != nullptr) {
    const int64_t c = (int64_t)(*g.count) * g.rows_per_count;
    M = c < M ? c : M;
  }
  // persistent over output tiles: CTA c owns tiles c, c + gridDim.x, ... (row-block major), so a launch sized for
  // a row CAPACITY whose actual row count lives on the device costs at most gridDim.x (<= #SMs) CTAs instead of
  // one (immediately exiting) CTA per capacity tile - at the seq restarter's capacity that was 29k CTAs = 57 us
  const int64_t n_tiles_total = ((g.M + TCG_BM - 1) / TCG_BM) * g.tiles_n;
  if ((int64_t)(blockIdx.x / g.tiles_n) * TCG_BM >= M) return;
  // Note: row_zero and the four strides are never set; every launch leaves them NULL / 0.  They stay because without
  // them ptxas allocates this kernel's registers differently: the transposed-W instantiations spill 20-44 more bytes
  // and the training step measured 0.5-0.7 % slower on a B200 (1000 W power limit).  Drop them together with a change
  // that retunes the producers, and measure it.
  const int b = g.kblk_per_part > 0 ? 0 : blockIdx.y;
  int K_eff = g.K;
  if (g.k_count != nullptr) {
    const int64_t c = (int64_t)(*g.k_count) * g.k_rows_per_count;
    K_eff = c < K_eff ? (int)c : K_eff;
  }
  const int kblk0 = g.kblk_per_part > 0 ? (int)blockIdx.y * g.kblk_per_part : 0;   // first stage of this K part
  {
    const int all_blocks = (K_eff + UMMA_BK - 1) / UMMA_BK;
    if (g.kblk_per_part > 0 && kblk0 >= all_blocks) return;     // nothing to add (also K_eff == 0)
  }
  const float* __restrict__ A = g.A + b * g.stride_a;
  const float* __restrict__ W = g.W + b * g.stride_w;
  const float* __restrict__ bias = g.bias != nullptr ? g.bias + b * g.stride_bias : nullptr;
  float* __restrict__ C = g.C + b * g.stride_c;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  auto init_barriers = [&](bool again) {
    if (tid == TCG_PRODUCER_WARPS * 32) {
      for (int s = 0; s < S; ++s) {
        if (again) { mbar_inval(full + s); mbar_inval(empty + s); }
        mbar_init(full + s, TCG_GROUP_WARPS);
        mbar_init(empty + s, UMMA_ISSUERS);
      }
      if (again) mbar_inval(done);
      mbar_init(done, UMMA_ISSUERS);
      fence_mbar_init();
    }
  };
  init_barriers(false);
  if (warp == 0) tmem_alloc(tmem_slot, g.tmem_cols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t taddr = *tmem_slot;
  for (int64_t tile = blockIdx.x; tile < n_tiles_total; tile += gridDim.x) {
  const int64_t m0 = (tile / g.tiles_n) * TCG_BM;
  if (m0 >= M) break;
  const int n0 = (int)(tile % g.tiles_n) * BN;
  if (tile != (int64_t)blockIdx.x) {
    // every barrier of the previous tile has completed its last phase (the epilogue waited for `done`, which the
    // issuers commit after all MMAs, and the block synchronised): start the next tile from fresh barriers
    init_barriers(true);
    __syncthreads();
  }
  int n_blocks = (K_eff + UMMA_BK - 1) / UMMA_BK;
  if (g.kblk_per_part > 0) {
    n_blocks -= kblk0;
    n_blocks = n_blocks < g.kblk_per_part ? n_blocks : g.kblk_per_part;
  }
#ifdef TIGER_TRACE
  __shared__ long long tr_base_s;
  if (tid == 0) tr_base_s = clock64();
  __syncthreads();
  const long long tr_base = tr_base_s;
#endif
  TRACE_DECL

  if (warp < TCG_PRODUCER_WARPS) {
    // ---------------- producers ----------------
    // group `grp` fills stages grp, grp + GROUPS, ...: while one group waits for its loads the others
    // convert / publish theirs, so GROUPS stages worth of global loads are always in flight
    const int grp = warp / TCG_GROUP_WARPS, wg = warp % TCG_GROUP_WARPS;
    UmmaChunks<TCG_NA> ca;
    UmmaChunks<TCG_NW> cw;
    {
      int row, kc;
      umma_chunk_pos(wg, lane, row, kc);          // chunk 0 = warp-chunk wg; chunk i = warp-chunk wg + 4 i
      const int64_t rows_a = M - m0;
      ca.rows_valid = rows_a < TCG_BM ? (int)rows_a : TCG_BM;
      ca.n_own = TCG_NA;
      ca.row0 = row;
      ca.kq = kc * 4;
      ca.soff0 = (kc * TCG_BM + row) * 4;
      if constexpr (MODE_A == 0) {
        ca.ptr0 = A + (m0 + row) * g.lda + kc * 4;
        ca.step = 32 * g.lda;
      } else {
        ca.ptr0 = A + (int64_t)(kc * 4) * g.lda + m0 + row;
        ca.step = 32;
      }
      const int rows_w = g.N - n0;
      cw.rows_valid = rows_w < BN ? rows_w : BN;
      const int wchunks = BN >> 3;                // warp-chunks of the W tile
      cw.n_own = wchunks > wg ? (wchunks - wg + TCG_GROUP_WARPS - 1) / TCG_GROUP_WARPS : 0;
      cw.row0 = row;
      cw.kq = kc * 4;
      cw.soff0 = (kc * BN + row) * 4;
      if constexpr (MODE_W == 0) {
        cw.ptr0 = W + (int64_t)(n0 + row) * g.ldw + kc * 4;
        cw.step = 32 * g.ldw;
      } else {
        cw.ptr0 = W + (int64_t)(kc * 4) * g.ldw + n0 + row;
        cw.step = 32;
      }
    }
    // two register sets per thread: the loads of this group's next two stages are in flight while the
    // current one is converted and published (the proxy fence would otherwise wait for a stage's loads
    // right after they were issued)
    float4 va0[TCG_NA], vw0[TCG_NW], va1[TCG_NA], vw1[TCG_NW];
    auto load = [&](float4 (&va)[TCG_NA], float4 (&vw)[TCG_NW], int blk) {
      if (blk < n_blocks) {
        const int k0 = (kblk0 + blk) * UMMA_BK;
        if constexpr (MODE_A == 1) umma_chunks_load_t(va, ca, k0, K_eff, g.lda);
        else umma_chunks_load(va, ca, k0, K_eff, g.vec_a != 0);
        if constexpr (MODE_W == 1) umma_chunks_load_t(vw, cw, k0, K_eff, g.ldw);
        else umma_chunks_load(vw, cw, k0, K_eff, g.vec_w != 0);
      }
    };
    auto publish = [&](const float4 (&va)[TCG_NA], const float4 (&vw)[TCG_NW], int blk) {
      const int s = blk % S;
      float* a_hi = stage0 + (size_t)s * stage_floats;
      float* a_lo = a_hi + a_plane;
      float* w_hi = a_lo + a_plane;
      float* w_lo = w_hi + w_plane;
      mbar_wait(empty + s, ((blk / S) & 1) ^ 1);
      TRACE_MARK();
      umma_chunks_store(a_hi, a_lo, ca, va);
      umma_chunks_store(w_hi, w_lo, cw, vw);
      TRACE_MARK();
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(full + s);
      TRACE_MARK();
    };
    load(va0, vw0, grp);
    load(va1, vw1, grp + TCG_GROUPS);
    for (int blk = grp; blk < n_blocks; blk += 2 * TCG_GROUPS) {
      publish(va0, vw0, blk);
      load(va0, vw0, blk + 2 * TCG_GROUPS);
      if (blk + TCG_GROUPS < n_blocks) {
        publish(va1, vw1, blk + TCG_GROUPS);
        load(va1, vw1, blk + 3 * TCG_GROUPS);
      }
    }
    // ---------------- epilogue ----------------
    mbar_wait(done, 0);
    tc_fence_after_sync();
    TRACE_MARK();
    const int q = warp & 3;
    const int64_t m = m0 + q * 32 + lane;
    const bool row_ok = m < M;
    const bool zero = row_ok && g.row_zero != nullptr && g.row_zero[m] != 0;
    const uint32_t tl = taddr + ((uint32_t)(q * 32) << 16);
    for (int c0 = (warp >> 2) * 16; c0 < BN; c0 += 16 * (TCG_PRODUCER_WARPS / 4)) {
      float v[16];
      tmem_ld16(tl + (uint32_t)c0, v);
#pragma unroll
      for (int j = 1; j < UMMA_ACCS; ++j) {
        float t[16];
        tmem_ld16(tl + (uint32_t)(j * BN + c0), t);
#pragma unroll
        for (int e = 0; e < 16; ++e) v[e] += t[e];
      }
      const int nb = n0 + c0;
      if (!row_ok || nb >= g.N) continue;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int n = nb + j;
        float x = (v[j] + ((bias != nullptr && n < g.N) ? __ldg(bias + n) : 0.f)) * g.alpha;
        if (g.relu) x = fmaxf(x, 0.f);
        v[j] = zero ? 0.f : x;
      }
      float* dst = C + m * g.ldc + nb;
      if (g.accumulate) {
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (nb + j < g.N) atomicAdd(dst + j, v[j]);
      } else if (g.vec_c && nb + 16 <= g.N) {
#pragma unroll
        for (int j = 0; j < 16; j += 4)
          *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (nb + j < g.N) dst[j] = v[j];
      }
    }
  } else if (warp < TCG_PRODUCER_WARPS + UMMA_ISSUERS) {
    // ---------------- MMA issuers (one elected thread per role, see umma.cuh) ----------------
    // The whole warp runs the loop so that every operand stays warp-uniform; only the tcgen05 instructions
    // are issued by the elected lane.
    const int role = uniform_warp_idx() - TCG_PRODUCER_WARPS;
    const UmmaRole r = umma_role(role, smem_addr_u32(stage0), (uint32_t)stage_floats * 4u, TCG_BM, BN, (uint32_t)BN);
    const uint32_t idesc = umma_idesc_tf32(TCG_BM, BN);
    const uint32_t tbase = __shfl_sync(0xffffffffu, taddr, 0);
    const uint32_t d_even = tbase + r.acc_even, d_odd = tbase + r.acc_odd;
    int s = 0;
    uint32_t ph = 0, a = r.a_lo, b = r.b_lo;
    for (int blk = 0; blk < n_blocks; ++blk) {
      mbar_wait(full + s, ph);
      tc_fence_after_sync();
      TRACE_MARK();
      if (elect_one()) {
        umma_tf32_lo(d_even, a, b, idesc, blk > 0 ? 1u : 0u);
        umma_tf32_lo(d_odd, a + r.a_kstep, b + r.b_kstep, idesc, (role == 2 && blk == 0) ? 0u : 1u);
        umma_commit(empty + s);
      }
      __syncwarp();
      TRACE_MARK();
      a += r.stage_step;
      b += r.stage_step;
      if (++s == S) {
        s = 0;
        ph ^= 1;
        a = r.a_lo;
        b = r.b_lo;
      }
    }
    if (elect_one()) umma_commit(done);
    __syncwarp();
  }
  TRACE_MARK();
#ifdef TIGER_TRACE
  if (warp % TCG_GROUP_WARPS == 0 || warp >= TCG_PRODUCER_WARPS) TRACE_DUMP(warp < TCG_PRODUCER_WARPS ? "producer" : "issuer", warp);
#endif
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  }  // tile loop
  if (warp == 0) tmem_dealloc(taddr, g.tmem_cols);
}

// ------------------------------------------------------------------------------------------
// Packed-weight variant with the activations in tensor memory ("TS" form).
//   TMEM columns : [0, 4 BN) the four partial accumulators | [4 BN, 4 BN + 64 S) ring of S activation
//                  stages, each 32 head + 32 tail columns (TS_BK = 32 floats of K)
//   shared memory: ring of S weight stages [head plane | tail plane], one TMA bulk copy each
//   warps 0-15   : 4 groups x 4 warps; warp w of a group owns rows 32 w .. 32 w + 31 (its TMEM lanes),
//                  thread = row: one 128-byte line of the row per stage -> tf32 split -> tcgen05.st
//   warps 16-18  : MMA issuers (roles as in umma.cuh), warp 19: TMA
// No shared-memory traffic, no proxy fence and no operand read for the activations: an MMA of this form
// reads only its BN x 32-byte weight tile from shared memory and runs at the math floor (tools/umma_bench.cu).
// ------------------------------------------------------------------------------------------
#define TS_MAX_BN 64
#define TS_MAX_STAGES 6
#define TS_THREADS ((TCG_PRODUCER_WARPS + UMMA_ISSUERS + 1) * 32)

__device__ __forceinline__ void ts_load_row(float4 (&v)[TS_KCH], const float* p, int k0, int k_end, bool vec_ok) {
  if (vec_ok && k0 + TS_BK <= k_end) {
#pragma unroll
    for (int i = 0; i < TS_KCH; ++i) v[i] = __ldg(reinterpret_cast<const float4*>(p + k0) + i);
  } else {
#pragma unroll
    for (int i = 0; i < TS_KCH; ++i) v[i] = umma_load_chunk(p, k0 + 4 * i, k_end, false);
  }
}

// split TS_BK floats and store them as one activation stage [32 head columns | 32 tail columns] of this
// thread's TMEM lane
__device__ __forceinline__ void ts_store_row(uint32_t taddr_stage, const float4 (&v)[TS_KCH]) {
#pragma unroll
  for (int half = 0; half < TS_BK / 16; ++half) {
    float hi[16], lo[16];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float4 h, l;
      tf32_split(v[4 * half + i], h, l);
      hi[4 * i] = h.x; hi[4 * i + 1] = h.y; hi[4 * i + 2] = h.z; hi[4 * i + 3] = h.w;
      lo[4 * i] = l.x; lo[4 * i + 1] = l.y; lo[4 * i + 2] = l.z; lo[4 * i + 3] = l.w;
    }
    tmem_st16(taddr_stage + 16u * half, hi);
    tmem_st16(taddr_stage + TS_BK + 16u * half, lo);
  }
  tmem_wait_st();
}

__global__ void __launch_bounds__(TS_THREADS, 1) gemm_tf32x3_ts_kernel(const GemmArgs g) {
  extern __shared__ __align__(128) unsigned char tcg_smem[];
  const int BN = g.bn, S = g.stages;
  const int w_stage_floats = UMMA_PACK_STAGE_FLOATS(BN);
  float* stage0 = reinterpret_cast<float*>(tcg_smem);
  uint64_t* full = reinterpret_cast<uint64_t*>(tcg_smem + (size_t)S * w_stage_floats * sizeof(float));
  uint64_t* empty = full + TS_MAX_STAGES;
  uint64_t* done = empty + TS_MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  // late_trigger: the kernel behind this one reads, before its own wait, data written upstream of this kernel; it
  // may therefore only be scheduled once this kernel's producers have passed THEIR wait (see below)
  if (!g.late_trigger) pdl_trigger();
  // With a host-side row count the set-up and the weight stream (parameters: nothing the previous kernel
  // writes) run ahead of the previous kernel's completion; only the producers wait, before their first
  // activation load.  A device-side count is itself produced upstream: everybody waits first.
  const bool early = g.count == nullptr;
  if (!early) {
    pdl_wait();
    if (g.late_trigger) pdl_trigger();
  }
  int64_t M = g.M;
  if (g.count != nullptr) {
    const int64_t c = (int64_t)(*g.count) * g.rows_per_count;
    M = c < M ? c : M;
  }
  const int64_t m0 = (int64_t)(blockIdx.x / g.tiles_n) * TCG_BM;
  if (m0 >= M) return;
  const int n_tile = (int)(blockIdx.x % g.tiles_n);
  const int n0 = n_tile * BN;
  const float* __restrict__ A = g.A;
  const float* __restrict__ bias = g.bias;
  float* __restrict__ C = g.C;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == TCG_PRODUCER_WARPS * 32) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full + s, TCG_GROUP_WARPS + 1);
      mbar_init(empty + s, UMMA_ISSUERS);
    }
    mbar_init(done, UMMA_ISSUERS);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, g.tmem_cols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t taddr = *tmem_slot;
  const uint32_t a_ring = taddr + (uint32_t)(UMMA_ACCS * BN);
  const int n_blocks_all = (g.K + TS_BK - 1) / TS_BK;
  const int per_part = (n_blocks_all + g.k_parts - 1) / g.k_parts;
  const int kb0 = (int)blockIdx.y * per_part;                      // first k-block of this part
  const int n_blocks = (kb0 + per_part < n_blocks_all ? kb0 + per_part : n_blocks_all) - kb0;
#ifdef TIGER_TRACE
  __shared__ long long tr_base_s;
  if (tid == 0) tr_base_s = clock64();
  __syncthreads();
  const long long tr_base = tr_base_s;
#endif
  TRACE_DECL

  if (warp < TCG_PRODUCER_WARPS) {
    // ---------------- producers: thread = row ----------------
    const int grp = warp / TCG_GROUP_WARPS, q = warp & 3;
    const int row = q * 32 + lane;
    int64_t m = m0 + row;
    m = m < M ? m : M - 1;                 // rows beyond the edge only feed accumulator rows nobody stores
    if (early) {
      pdl_wait();
      if (g.late_trigger) pdl_trigger();
    }
    const float* rowp = A + m * g.lda;
    const float* addp = nullptr;
    if (g.a_ids != nullptr) {
      const int64_t u = g.a_ids[m];
      const int64_t r = g.a_sel == nullptr ? -1
                        : g.a_sel_i64 ? reinterpret_cast<const int64_t*>(g.a_sel)[u]
                                      : (int64_t) reinterpret_cast<const int32_t*>(g.a_sel)[u];
      rowp = (A == nullptr || r >= 0) ? g.a_alt + r * g.lda : A + u * g.lda;
      if (g.a_add != nullptr) addp = g.a_add + u * g.lda;
    }
    const uint32_t tl = a_ring + ((uint32_t)(q * 32) << 16);
    const bool vec = g.vec_a != 0;
    float4 v[TS_KCH];
    auto load = [&](int blk) {
      const int k0 = (kb0 + blk) * TS_BK;
      ts_load_row(v, rowp, k0, g.K, vec);
      if (g.a_add != nullptr && g.a_ids != nullptr) {
        float4 t[TS_KCH];
        ts_load_row(t, addp, k0, g.K, vec);
#pragma unroll
        for (int i = 0; i < TS_KCH; ++i) {
          v[i].x += t[i].x; v[i].y += t[i].y; v[i].z += t[i].z; v[i].w += t[i].w;
        }
      }
    };
    if (grp < n_blocks) load(grp);
    for (int blk = grp; blk < n_blocks; blk += TCG_GROUPS) {
      const int s = blk % S;
      TRACE_MARK();
      mbar_wait(empty + s, ((blk / S) & 1) ^ 1);
      TRACE_MARK();
      ts_store_row(tl + (uint32_t)(s * 2 * TS_BK), v);
      TRACE_MARK();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(full + s);
      // this group's next stage is loaded while the other groups' stages are converted / consumed
      if (blk + TCG_GROUPS < n_blocks) load(blk + TCG_GROUPS);
    }
    // ---------------- epilogue ----------------
    mbar_wait(done, 0);
    tc_fence_after_sync();
    const int64_t mr = m0 + row;
    const bool row_ok = mr < M;
    const bool sc_row = g.sc_table != nullptr && row_ok && mr < g.sc_rows && g.sc_mask[mr] != 0;
    const int64_t sc_u = sc_row ? g.sc_ids[mr] : 0;
    const uint32_t tacc = taddr + ((uint32_t)(q * 32) << 16);
    for (int c0 = (warp >> 2) * 16; c0 < BN; c0 += 16 * (TCG_PRODUCER_WARPS / 4)) {
      float o[16];
      tmem_ld16(tacc + (uint32_t)c0, o);
#pragma unroll
      for (int j = 1; j < UMMA_ACCS; ++j) {
        float t[16];
        tmem_ld16(tacc + (uint32_t)(j * BN + c0), t);
#pragma unroll
        for (int e = 0; e < 16; ++e) o[e] += t[e];
      }
      if (g.k_parts > 1) {                              // cluster split-K: partial tile to shared memory
        float* dst = stage0 + row * (BN + 4) + c0;       // the weight ring is idle once `done` has fired
#pragma unroll
        for (int j = 0; j < 16; j += 4)
          *reinterpret_cast<float4*>(dst + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
        continue;
      }
      const int nb = n0 + c0;
      if (!row_ok || nb >= g.N) continue;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int n = nb + j;
        float x = (o[j] + ((bias != nullptr && n < g.N) ? __ldg(bias + n) : 0.f)) * g.alpha;
        if (g.relu) x = fmaxf(x, 0.f);
        o[j] = x;
      }
      // destination of this 16-column chunk (n_split is a multiple of 16, so a chunk never straddles it)
      const bool second = g.C2 != nullptr && nb >= g.n_split;
      const int col = second ? nb - g.n_split : nb, lim = second ? g.n_lim1 : g.n_lim0;
      float* dst = second ? g.C2 + mr * g.ldc2 + col : C + mr * g.ldc + col;
      if ((second ? g.vec_c2 : g.vec_c) && col + 16 <= lim) {
#pragma unroll
        for (int j = 0; j < 16; j += 4)
          *reinterpret_cast<float4*>(dst + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (col + j < lim) dst[j] = o[j];
      }
      if (sc_row && !second) {
        // the same values into the node's row of the table (update_left_memory fused into the producing kernel)
        float* d3 = g.sc_table + sc_u * g.sc_ld + col;
        if (g.vec_sc && col + 16 <= lim) {
#pragma unroll
          for (int j = 0; j < 16; j += 4)
            *reinterpret_cast<float4*>(d3 + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (col + j < lim) d3[j] = o[j];
        }
        if (nb == 0) {                         // one thread per row owns the scalar side
          const float t = g.sc_ts[mr % g.sc_period];
          if (g.sc_err != nullptr && g.sc_ts_table[sc_u] > t) atomicOr(g.sc_err, TIGER_ERR_PAST_MEMORY);
          g.sc_ts_table[sc_u] = t;
          if (g.sc_active != nullptr) g.sc_active[sc_u] = 1;
        }
      }
    }
  } else if (warp == TCG_PRODUCER_WARPS + UMMA_ISSUERS) {
    // ---------------- TMA warp ----------------
    if (lane == 0) {
      const uint32_t bytes = (uint32_t)w_stage_floats * 4u;
      const float* src = g.wpack + ((int64_t)n_tile * n_blocks_all + kb0) * w_stage_floats;
      for (int blk = 0; blk < n_blocks; ++blk) {
        const int s = blk % S;
        mbar_wait(empty + s, ((blk / S) & 1) ^ 1);
        TRACE_MARK();
        mbar_arrive_expect_tx(full + s, bytes);
        tma_bulk_load(stage0 + (size_t)s * w_stage_floats, src + (int64_t)blk * w_stage_floats, bytes, full + s);
      }
    }
  } else {
    // ---------------- MMA issuers ----------------
    const int role = uniform_warp_idx() - TCG_PRODUCER_WARPS;
    const uint32_t idesc = umma_idesc_tf32(TCG_BM, BN);
    const uint32_t tbase = __shfl_sync(0xffffffffu, taddr, 0);
    const uint32_t d_even = tbase + (uint32_t)(role * BN), d_odd = role == 2 ? tbase + (uint32_t)(3 * BN) : d_even;
    const uint32_t a_first = tbase + (uint32_t)(UMMA_ACCS * BN) + (role == 0 ? (uint32_t)TS_BK : 0u);   // role 0: tail columns
    const uint32_t b_first = umma_desc_lo(smem_addr_u32(stage0) + (role == 1 ? (uint32_t)(TS_KCH * BN * 16) : 0u),
                                          (uint32_t)BN);
    const uint32_t b_step = (uint32_t)(w_stage_floats * 4) >> 4, b_kstep = 2u * BN;
    int s = 0;
    uint32_t ph = 0, a = a_first, b = b_first;
    bool ready = mbar_test(full, 0);
    for (int blk = 0; blk < n_blocks; ++blk) {
      TRACE_MARK();
      mbar_wait_probed(ready, full + s, ph);
      tc_fence_after_sync();
      TRACE_MARK();
      // probe the next stage now: its latency overlaps the MMA issue below
      int s1 = s + 1;
      uint32_t ph1 = ph;
      if (s1 == S) {
        s1 = 0;
        ph1 ^= 1;
      }
      ready = blk + 1 < n_blocks ? mbar_test(full + s1, ph1) : true;
      if (elect_one()) {
#pragma unroll
        for (int j = 0; j < TS_BK / 8; ++j) {
          const uint32_t fresh = (blk == 0 && (j == 0 || (role == 2 && j == 1))) ? 0u : 1u;
          umma_tf32_ts((j & 1) ? d_odd : d_even, a + 8u * j, b + b_kstep * j, idesc, fresh);
        }
        umma_commit(empty + s);
      }
      __syncwarp();
      a += 2u * TS_BK;
      b += b_step;
      if (s1 == 0) {
        a = a_first;
        b = b_first;
      }
      s = s1;
      ph = ph1;
    }
    if (elect_one()) umma_commit(done);
    __syncwarp();
  }
#ifdef TIGER_TRACE
  TRACE_MARK();
  if (warp % TCG_GROUP_WARPS == 0 || warp >= TCG_PRODUCER_WARPS) TRACE_DUMP(warp < TCG_PRODUCER_WARPS ? "producer" : "issuer", warp);
#endif
  if (g.k_parts > 1) {
    __syncwarp();
    if (early && warp >= TCG_PRODUCER_WARPS) pdl_wait();   // these warps store results below
    cluster_sync_all();                       // every part's tile sits in its CTA's shared memory
    const int kp = g.k_parts, rank = (int)cluster_cta_rank();
    const int rb = (TCG_BM + kp - 1) / kp;    // rows this CTA finishes
    const int r0 = rank * rb, r1 = r0 + rb < TCG_BM ? r0 + rb : TCG_BM;
    const int c4n = BN >> 2;
    const uint32_t red = smem_addr_u32(stage0);
    for (int i = tid; i < (r1 - r0) * c4n; i += TS_THREADS) {
      const int row = r0 + i / c4n, c = (i % c4n) * 4;
      const int64_t mr = m0 + row;
      const int n = n0 + c;
      if (mr >= M || n >= g.N) continue;
      const uint32_t off = (uint32_t)(row * (BN + 4) + c) * 4u;
      float4 acc = cluster_ld_f4(cluster_map_shared(red + off, 0));
      for (int part = 1; part < kp; ++part) {
        const float4 t = cluster_ld_f4(cluster_map_shared(red + off, (uint32_t)part));
        acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
      }
      float o[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float x = (o[j] + ((bias != nullptr && n + j < g.N) ? __ldg(bias + n + j) : 0.f)) * g.alpha;
        o[j] = g.relu ? fmaxf(x, 0.f) : x;
      }
      float* dst = C + mr * g.ldc + n;
      if (g.vec_c && n + 4 <= g.n_lim0) {
        *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (n + j < g.n_lim0) dst[j] = o[j];
      }
    }
    cluster_sync_all();                       // nobody leaves while a peer still reads its tile
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(taddr, g.tmem_cols);
}

static int g_gemm_sms = 0;

// pack kernel: one thread per (tile, k-block, kc, row)
__global__ void gemm_pack_weight_kernel(const float* __restrict__ W, int64_t ldw, const int32_t* __restrict__ row_map,
                                        int n_rows, int k_dim, int bn, int tiles, int n_kb, int vec_ok,
                                        float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)tiles * n_kb * TS_KCH * bn;
  if (i >= total) return;
  const int r = (int)(i % bn);
  const int kc = (int)((i / bn) % TS_KCH);
  const int kb = (int)((i / ((int64_t)bn * TS_KCH)) % n_kb);
  const int t = (int)(i / ((int64_t)bn * TS_KCH * n_kb));
  const int row = row_map != nullptr ? row_map[(int64_t)t * bn + r] : t * bn + r;
  const int k = kb * TS_BK + kc * 4;
  const float4 v = umma_load_chunk((row >= 0 && row < n_rows) ? W + (int64_t)row * ldw : nullptr, k, k_dim, vec_ok != 0);
  float4 h, l;
  tf32_split(v, h, l);
  float* stage = out + ((int64_t)t * n_kb + kb) * UMMA_PACK_STAGE_FLOATS(bn);
  *reinterpret_cast<float4*>(stage + (kc * bn + r) * 4) = h;
  *reinterpret_cast<float4*>(stage + TS_KCH * bn * 4 + (kc * bn + r) * 4) = l;
}

extern "C" int64_t tiger_gemm_pack_bytes(int n_tiles, int k_dim, int bn) {
  if (n_tiles <= 0 || k_dim <= 0 || bn < 16 || bn > TS_MAX_BN || (bn & 15) != 0) return -1;
  const int64_t n_kb = (k_dim + TS_BK - 1) / TS_BK;
  return (int64_t)n_tiles * n_kb * UMMA_PACK_STAGE_FLOATS(bn) * (int64_t)sizeof(float);
}

extern "C" int tiger_gemm_pack_weight(const float* W, int64_t ldw, const int32_t* row_map, int n_rows, int k_dim,
                                      int bn, int n_tiles, float* out, void* stream) {
  if (W == nullptr || out == nullptr || tiger_gemm_pack_bytes(n_tiles, k_dim, bn) < 0 || n_rows <= 0 || ldw < k_dim ||
      (((uintptr_t)out) & 15) != 0)
    return TIGER_EINVAL;
  const int n_kb = (k_dim + TS_BK - 1) / TS_BK;
  const int64_t total = (int64_t)n_tiles * n_kb * TS_KCH * bn;
  const int vec_ok = ((((uintptr_t)W) & 15) == 0 && (ldw & 3) == 0) ? 1 : 0;
  gemm_pack_weight_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(
      W, ldw, row_map, n_rows, k_dim, bn, n_tiles, n_kb, vec_ok, out);
  return tiger_launch_status();
}

// column tile width the packed entry point expects for a weight of n_cols rows used with about m_rows
// activation rows: the widest of 128/64/32 that still yields about one CTA per SM, then balanced
static int gemm_pick_bn(int64_t m_rows, int n_cols, int batch, int sms, int max_bn) {
  const int64_t tiles_m = (m_rows + TCG_BM - 1) / TCG_BM;
  int bn = 32;
  for (int cand = max_bn; cand >= 32; cand >>= 1) {
    const int64_t tiles = tiles_m * ((n_cols + cand - 1) / cand) * batch;
    if (tiles >= (3 * (int64_t)sms) / 4 || cand == 32) {
      bn = cand;
      break;
    }
  }
  const int tiles_n = (n_cols + bn - 1) / bn;
  return (((n_cols + tiles_n - 1) / tiles_n) + 15) & ~15;
}

static int gemm_sms() {
  if (g_gemm_sms == 0) {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
    bool ok = true;
    auto set_smem = [&](auto kernel) {
      ok = ok && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TCG_SMEM_BUDGET + 256) ==
                     cudaSuccess;
    };
    set_smem(gemm_tf32x3_kernel<0, 0>);
    set_smem(gemm_tf32x3_kernel<0, 1>);
    set_smem(gemm_tf32x3_kernel<1, 0>);
    set_smem(gemm_tf32x3_kernel<1, 1>);
    if (!ok ||
        cudaFuncSetAttribute(gemm_tf32x3_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             TS_MAX_STAGES * UMMA_PACK_STAGE_FLOATS(TS_MAX_BN) * 4 + 256) != cudaSuccess)
      return -1;
    g_gemm_sms = sms;
  }
  return g_gemm_sms;
}

extern "C" int tiger_gemm_pick_bn(int64_t m_rows, int n_cols, int batch) {
  const int sms = gemm_sms();
  if (sms < 0 || m_rows <= 0 || n_cols <= 0 || batch <= 0) return TIGER_EINVAL;
  return gemm_pick_bn(m_rows, n_cols, batch, sms, TS_MAX_BN);
}

// A product on the packed kernel: C = act(alpha * (A Wpack^T + bias)) for a pack of ceil(n_cols / bn) column tiles,
// plus the options the attention chain uses.  The tiger_sgemm_nt_packed* entry points fill it by field name; the
// fields they leave out are zero / NULL (or the default given here), which turns every option off.
struct PackedGemm {
  const float* A;                 // NULL allowed with a gathered A
  int64_t lda;
  const float* wpack;
  int bn;
  const float* bias;
  float* C;
  int64_t ldc;
  int n_cols;                     // columns written to C
  int64_t m_rows;
  const int32_t* count;
  int64_t rows_per_count = 1;
  int k_dim;
  float alpha = 1.0f;
  int relu;
  // split output: pack columns [n_split, n_split + n_cols1) go to C2 (n_split a multiple of 16 >= n_cols)
  float* C2;
  int64_t ldc2;
  int n_split, n_cols1;
  int k_parts = 1;                // > 1: K split over a thread-block cluster of up to 8 CTAs per tile
  // gathered A (GemmArgs::a_ids): row m is row sel[ids[m]] of alt when that is >= 0, else row ids[m] of A, + add;
  // without sel always row ids[m] of A
  const int64_t* ids;
  const void* sel;
  int sel_is_i64;
  const float* alt;
  const float* add;
  const tiger_left_writeback_fused* wb;   // fused row scatter into the left memory
};

static int gemm_packed_launch(const PackedGemm& p, void* stream) {
  if (p.wpack == nullptr || p.m_rows < 0 || p.n_cols <= 0 || p.k_dim <= 0 || p.lda < p.k_dim || p.ldc < p.n_cols)
    return TIGER_EINVAL;
  if (p.C2 != nullptr && ((p.n_split & 15) != 0 || p.n_split < p.n_cols || p.n_cols1 <= 0 || p.ldc2 < p.n_cols1))
    return TIGER_EINVAL;
  if (p.k_parts < 1 || p.k_parts > 8 || (p.k_parts > 1 && p.C2 != nullptr)) return TIGER_EINVAL;
  if (p.bn < 16 || p.bn > TS_MAX_BN || (p.bn & 15) != 0 || (((uintptr_t)p.wpack) & 15) != 0) return TIGER_EINVAL;
  if (p.m_rows == 0) return TIGER_OK;
  const int sms = gemm_sms();
  if (sms < 0) return TIGER_ECUDA;
  GemmArgs g{};
  g.A = p.A; g.wpack = p.wpack; g.bias = p.bias; g.C = p.C; g.count = p.count;
  g.lda = p.lda; g.ldc = p.ldc;
  g.M = p.m_rows; g.rows_per_count = p.rows_per_count > 0 ? p.rows_per_count : 1;
  g.N = p.C2 != nullptr ? p.n_split + p.n_cols1 : p.n_cols;   // columns of the (padded) weight / bias space
  g.K = p.k_dim; g.alpha = p.alpha; g.relu = p.relu;
  g.C2 = p.C2; g.ldc2 = p.ldc2; g.n_split = p.n_split; g.n_lim0 = p.n_cols; g.n_lim1 = p.n_cols1;
  g.vec_c2 = (p.C2 != nullptr && (((uintptr_t)p.C2) & 15) == 0 && (p.ldc2 & 3) == 0) ? 1 : 0;
  const int k_blocks = (p.k_dim + TS_BK - 1) / TS_BK;
  g.k_parts = p.k_parts < k_blocks ? p.k_parts : k_blocks;              // every part owns at least one k-block
  g.k_parts = (k_blocks + ((k_blocks + g.k_parts - 1) / g.k_parts) - 1) / ((k_blocks + g.k_parts - 1) / g.k_parts);
  g.late_trigger = p.ids != nullptr ? 1 : 0;
  if (p.wb != nullptr) {
    const tiger_left_writeback_fused* wb = p.wb;
    if (p.k_parts != 1 || wb->pos_ids == nullptr || wb->winner == nullptr || wb->ts == nullptr ||
        wb->left_vals == nullptr || wb->left_ts == nullptr || wb->n_pos < 0 || wb->n_pos > p.m_rows || wb->batch <= 0)
      return TIGER_EINVAL;
    g.sc_table = wb->left_vals; g.sc_ids = wb->pos_ids; g.sc_mask = wb->winner; g.sc_rows = wb->n_pos;
    g.sc_period = wb->batch; g.sc_ld = p.ldc; g.sc_ts = wb->ts; g.sc_ts_table = wb->left_ts;
    g.sc_active = wb->left_active; g.sc_err = wb->err_flags;
    g.vec_sc = ((((uintptr_t)wb->left_vals) & 15) == 0 && (p.ldc & 3) == 0) ? 1 : 0;
  }
  g.a_ids = p.ids; g.a_sel = p.sel; g.a_sel_i64 = p.sel_is_i64; g.a_alt = p.alt; g.a_add = p.add;
  g.vec_a = ((((uintptr_t)p.A) & 15) == 0 && (p.lda & 3) == 0 && ((((uintptr_t)p.alt) | ((uintptr_t)p.add)) & 15) == 0)
                ? 1 : 0;
  g.vec_c = ((((uintptr_t)p.C) & 15) == 0 && (p.ldc & 3) == 0) ? 1 : 0;
  const int64_t tiles_m = (p.m_rows + TCG_BM - 1) / TCG_BM;
  g.bn = p.bn;
  g.tiles_n = (g.N + g.bn - 1) / g.bn;
  // activations in tensor memory: 4 accumulators + a ring of 32-column stages must fit 512 columns
  int stages = (512 - UMMA_ACCS * g.bn) / (2 * TS_BK);
  stages = stages > TS_MAX_STAGES ? TS_MAX_STAGES : stages;
  g.stages = stages;
  g.tmem_cols = tmem_cols_pow2((uint32_t)(UMMA_ACCS * g.bn + stages * 2 * TS_BK));
  const size_t smem = (size_t)stages * UMMA_PACK_STAGE_FLOATS(g.bn) * 4 + 256;
  dim3 grid((unsigned)(tiles_m * g.tiles_n), (unsigned)g.k_parts);
  // the cluster reduction reuses the weight ring for the partial tile
  if (g.k_parts > 1 && (size_t)TCG_BM * (g.bn + 4) * 4 > (size_t)stages * UMMA_PACK_STAGE_FLOATS(g.bn) * 4)
    return TIGER_EINVAL;
  return tiger_launch_chain(gemm_tf32x3_ts_kernel, grid, dim3(TS_THREADS), smem, as_stream(stream),
                            dim3(1, (unsigned)g.k_parts, 1), g);
}

extern "C" int tiger_sgemm_nt_packed(const float* A, int64_t lda, const float* wpack, int bn, const float* bias,
                                     float* C, int64_t ldc, int64_t m_rows, const int32_t* count,
                                     int64_t rows_per_count, int n_cols, int k_dim, float alpha, int relu,
                                     void* stream) {
  return gemm_packed_launch({.A = A, .lda = lda, .wpack = wpack, .bn = bn, .bias = bias, .C = C, .ldc = ldc,
                             .n_cols = n_cols, .m_rows = m_rows, .count = count, .rows_per_count = rows_per_count,
                             .k_dim = k_dim, .alpha = alpha, .relu = relu},
                            stream);
}

extern "C" int tiger_sgemm_nt_packed_scatter(const float* A, int64_t lda, const float* wpack, int bn, const float* bias,
                                             float* C, int64_t ldc, int n_cols0, float* C2, int64_t ldc2, int n_split,
                                             int n_cols1, int64_t m_rows, int k_dim, const tiger_left_writeback_fused* wb,
                                             void* stream) {
  if (wpack == nullptr || (wb == nullptr && C2 == nullptr)) return TIGER_EINVAL;
  if (wb != nullptr && wb->ready_event != nullptr &&
      cudaStreamWaitEvent(as_stream(stream), reinterpret_cast<cudaEvent_t>(wb->ready_event), 0) != cudaSuccess)
    return TIGER_ECUDA;
  return gemm_packed_launch({.A = A, .lda = lda, .wpack = wpack, .bn = bn, .bias = bias, .C = C, .ldc = ldc,
                             .n_cols = n_cols0, .m_rows = m_rows, .k_dim = k_dim, .C2 = C2,
                             .ldc2 = ldc2, .n_split = C2 != nullptr ? n_split : 0,
                             .n_cols1 = C2 != nullptr ? n_cols1 : 0, .wb = wb},
                            stream);
}

extern "C" int tiger_sgemm_nt_packed_splitk_fused(const float* A, int64_t lda, const float* wpack, int bn,
                                                  const float* bias, float* C, int64_t ldc, int k_parts,
                                                  int64_t m_rows, const int32_t* count, int64_t rows_per_count,
                                                  int n_cols, int k_dim, float alpha, int relu, void* stream) {
  if (C == nullptr) return TIGER_EINVAL;
  return gemm_packed_launch({.A = A, .lda = lda, .wpack = wpack, .bn = bn, .bias = bias, .C = C, .ldc = ldc,
                             .n_cols = n_cols, .m_rows = m_rows, .count = count, .rows_per_count = rows_per_count,
                             .k_dim = k_dim, .alpha = alpha, .relu = relu, .k_parts = k_parts},
                            stream);
}

extern "C" int tiger_sgemm_nt_packed_gather(const int64_t* ids, const void* sel, int sel_is_i64, const float* rows_a,
                                            const float* rows_b, int64_t ld_rows, const float* add_rows,
                                            const float* wpack, int bn, const float* bias, float* C, int64_t ldc,
                                            int64_t m_rows, const int32_t* count, int64_t rows_per_count,
                                            int n_cols, int k_dim, float alpha, int relu, void* stream) {
  if (ids == nullptr || (sel != nullptr ? rows_b == nullptr : rows_a == nullptr)) return TIGER_EINVAL;
  return gemm_packed_launch({.A = rows_a, .lda = ld_rows, .wpack = wpack, .bn = bn, .bias = bias, .C = C, .ldc = ldc,
                             .n_cols = n_cols, .m_rows = m_rows, .count = count, .rows_per_count = rows_per_count,
                             .k_dim = k_dim, .alpha = alpha, .relu = relu, .ids = ids, .sel = sel,
                             .sel_is_i64 = sel_is_i64, .alt = rows_b, .add = add_rows},
                            stream);
}

// General product on the staging kernel:
//   C[m, n] (+)= act(alpha * (sum_k opA[m, k] * opW[n, k] + bias[n]))
// opA[m, k] = A[m * lda + k] (trans_a = 0) or A[k * lda + m] (trans_a = 1), opW likewise.  With the three
// combinations the training step needs no transposed copies: forward y = x W^T (0, 0), input gradient
// dx = dy W (0, 1), weight gradient dW = dy^T x (1, 1).  `accumulate` adds the tile into C with atomic adds
// (gradients of a parameter used more than once sum up; bias / relu are not allowed then) and lets the launch
// split K over `k_parts` CTAs per tile; m_count / k_count bound the row count / the reduction length from
// device memory (times rows_per_count).
extern "C" int tiger_sgemm_ex(const float* A, int64_t lda, int trans_a, const float* W, int64_t ldw, int trans_w,
                              const float* bias, float* C, int64_t ldc, int64_t m_rows, int n_cols, int64_t k_dim,
                              const int32_t* m_count, const int32_t* k_count, int64_t rows_per_count, float alpha,
                              int relu, int accumulate, int k_parts, void* stream) {
  if (A == nullptr || W == nullptr || C == nullptr || m_rows < 0 || n_cols <= 0 || k_dim <= 0 || k_dim > 0x7fffffffll ||
      ldc < n_cols || (!trans_a && lda < k_dim) || (trans_a && lda < m_rows) || (!trans_w && ldw < k_dim) ||
      (trans_w && ldw < n_cols) || k_parts < 1 || (accumulate && (bias != nullptr || relu)) ||
      (!accumulate && (k_parts > 1 || k_count != nullptr)))
    return TIGER_EINVAL;
  if (m_rows == 0) return TIGER_OK;
  const int sms = gemm_sms();
  if (sms < 0) return TIGER_ECUDA;
  GemmArgs g{};
  g.A = A; g.W = W; g.bias = bias; g.C = C; g.count = m_count; g.k_count = k_count;
  g.lda = lda; g.ldw = ldw; g.ldc = ldc;
  g.M = m_rows; g.rows_per_count = rows_per_count > 0 ? rows_per_count : 1;
  g.k_rows_per_count = g.rows_per_count;
  g.N = n_cols; g.K = (int)k_dim; g.alpha = alpha; g.relu = relu;
  g.accumulate = accumulate ? 1 : 0;
  g.vec_a = (!trans_a && (((uintptr_t)A) & 15) == 0 && (lda & 3) == 0) ? 1 : 0;
  g.vec_w = (!trans_w && (((uintptr_t)W) & 15) == 0 && (ldw & 3) == 0) ? 1 : 0;
  g.vec_c = ((((uintptr_t)C) & 15) == 0 && (ldc & 3) == 0) ? 1 : 0;
  const int64_t tiles_m = (m_rows + TCG_BM - 1) / TCG_BM;
  g.bn = gemm_pick_bn(m_rows, n_cols, accumulate ? k_parts : 1, sms, TCG_MAX_BN);
  g.tiles_n = (n_cols + g.bn - 1) / g.bn;
  g.tmem_cols = tmem_cols_pow2((uint32_t)(UMMA_ACCS * g.bn));
  const size_t stage_bytes = (size_t)(2 * UMMA_KCH * TCG_BM * 4 + 2 * UMMA_KCH * g.bn * 4) * sizeof(float);
  int stages = (int)(TCG_SMEM_BUDGET / stage_bytes);
  stages = stages > TCG_MAX_STAGES ? TCG_MAX_STAGES : stages;
  if (stages < 2) return TIGER_EINVAL;
  g.stages = stages;
  const int k_blocks = (int)((k_dim + UMMA_BK - 1) / UMMA_BK);
  int parts = accumulate ? (k_parts < k_blocks ? k_parts : k_blocks) : 1;
  g.kblk_per_part = accumulate ? (k_blocks + parts - 1) / parts : 0;
  if (accumulate) parts = (k_blocks + g.kblk_per_part - 1) / g.kblk_per_part;
  const int64_t tiles = tiles_m * g.tiles_n;
  // every (tile, K part) gets its own CTA up to one wave per part: with a device-side reduction length most parts of a
  // capacity-sized launch exit at once, the live ones must not queue behind each other
  dim3 grid((unsigned)(tiles < sms ? tiles : sms), (unsigned)parts);
  const size_t smem = stages * stage_bytes + 256;
  void (*kernel)(GemmArgs) = trans_a ? (trans_w ? gemm_tf32x3_kernel<1, 1> : gemm_tf32x3_kernel<1, 0>)
                                     : (trans_w ? gemm_tf32x3_kernel<0, 1> : gemm_tf32x3_kernel<0, 0>);
  kernel<<<grid, TCG_THREADS, smem, as_stream(stream)>>>(g);
  return tiger_launch_status();
}

extern "C" int tiger_sgemm_nt(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                              float* C, int64_t ldc, int64_t m_rows, const int32_t* count, int64_t rows_per_count,
                              int n_cols, int k_dim, int relu, void* stream) {
  return tiger_sgemm_ex(A, lda, 0, W, ldw, 0, bias, C, ldc, m_rows, n_cols, k_dim, count, nullptr, rows_per_count, 1.0f,
                        relu, 0, 1, stream);
}
