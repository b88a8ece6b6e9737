// Blackwell (sm_100a) tensor-core plumbing for libtiger_b200: mbarriers, TMEM allocation,
// tcgen05.mma (kind::tf32) with shared-memory operand descriptors, tcgen05.ld, and the
// "tf32x3" operand staging (every fp32 value is split into a tf32 head and a tf32 tail; three
// MMAs head*head + head*tail + tail*head reproduce the fp32 product to ~2^-22, which is what lets
// the dense parts of the path (GRU gates, attention / restarter projections) run on the tensor
// cores and still meet the fp32 1e-5 parity bar of the reference's CPU kernels).
//
// Operand tiles live in shared memory in the canonical K-major, non-swizzled UMMA layout:
//     plane[kc][row][4 floats]      kc = k / 4 (one 16-byte chunk), row = 0 .. rows-1
// i.e. a core matrix is 8 consecutive rows x 16 bytes (128 contiguous bytes), core matrices that are
// adjacent in M/N are 128 bytes apart (SBO) and core matrices adjacent in K are rows*16 bytes apart
// (LBO).  One tf32 MMA consumes K = 8 floats = two kc chunks.  A sub-range of rows that starts at a
// multiple of 8 is addressed by moving the start address only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define UMMA_BK 16          // floats of K per pipeline stage (2 MMA k-steps)
#define UMMA_KCH (UMMA_BK / 4)

__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_inval(uint64_t* bar) {
  asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_addr_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_addr_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking probe.  Any phase check costs the issuing thread ~150 cycles of latency (measured,
// tools/issue_bench.cu), so the MMA issuers probe the NEXT stage's barrier before they issue the current
// stage's MMAs: the probe's latency overlaps the issue, and mbar_wait_probed is free when it succeeded.
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_addr_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// Bounded wait: a pipeline that cannot make progress (a malformed descriptor, a lost arrive) traps
// after ~2 s instead of hanging the device.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}
// TMA 1-D bulk copy global -> shared, completion counted in bytes on `bar` (SASS: UBLKCP)
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_addr_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_addr_u32(bar))
               : "memory");
}
// bulk store shared -> global (bulk-group completion); the source must stay valid until tma_store_wait_read
__device__ __forceinline__ void tma_bulk_store(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_addr_u32(smem_src)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait_probed(bool probed_ok, uint64_t* bar, uint32_t parity) {
  if (!probed_ok) mbar_wait(bar, parity);
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy writes to shared memory -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// warp index / elected lane as the compiler can prove them warp-uniform (keeps descriptors in uniform
// registers: UTCHMMA takes uniform-register operands, per-thread values cost an R2UR each)
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// ---- TMEM -----------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_in_smem, uint32_t n_cols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr_u32(dst_in_smem)),
               "r"(n_cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t n_cols) {  // the allocating warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(n_cols) : "memory");
}
// thread-block cluster helpers (split-K partial sums are exchanged through distributed shared memory)
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_map_shared(uint32_t saddr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ float4 cluster_ld_f4(uint32_t cluster_saddr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(cluster_saddr)
               : "memory");
  return v;
}
__device__ __forceinline__ uint32_t cluster_cta_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}

__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

static inline uint32_t tmem_cols_pow2(uint32_t c) {
  uint32_t n = 32;
  while (n < c) n <<= 1;
  return n;
}

// 32 consecutive fp32 accumulator columns of this thread's TMEM lane (lane = 32 * (warp % 4) + lane id)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// 16 consecutive 32-bit columns of this thread's TMEM lane <- registers (whole warp; lane = 32 * (warp % 4) + lane id)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- descriptors ----------------------------------------------------------------------------
// shared-memory matrix descriptor, K-major, SWIZZLE_NONE, descriptor version 1 (sm_100):
//   [0,14) start address >> 4 | [16,30) leading (K) byte offset >> 4 | [32,46) stride (M/N) byte offset >> 4
//   | [46,48) = 1 | [61,64) layout type = 0
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// instruction descriptor, kind::tf32, fp32 accumulate, both operands K-major, M = 128:
//   [4,6) D format = 1 (f32) | [7,10) A format = 2 (tf32) | [10,13) B format = 2 | [17,23) N >> 3 | [24,29) M >> 4
__device__ __forceinline__ uint32_t umma_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]^T, issued by ONE thread
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on `bar` once every tcgen05.mma issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_addr_u32(bar))
               : "memory");
}

// ---- tf32x3 operand staging -----------------------------------------------------------------
// round-to-nearest (ties away from zero) fp32 -> tf32 on the integer pipe: two instructions instead of
// the Inf/NaN-safe cvt.rna.tf32 sequence (operands here are finite model state / parameters)
__device__ __forceinline__ float tf32_rn(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ void tf32_split(const float4& v, float4& hi, float4& lo) {
  hi.x = tf32_rn(v.x); hi.y = tf32_rn(v.y); hi.z = tf32_rn(v.z); hi.w = tf32_rn(v.w);
  lo.x = tf32_rn(v.x - hi.x); lo.y = tf32_rn(v.y - hi.y);
  lo.z = tf32_rn(v.z - hi.z); lo.w = tf32_rn(v.w - hi.w);
}

// four consecutive floats of a row starting at column k, zero beyond k_end / for a missing row
__device__ __forceinline__ float4 umma_load_chunk(const float* row_ptr, int k, int k_end, bool vec_ok) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (row_ptr != nullptr && k < k_end) {
    if (vec_ok && k + 4 <= k_end) {
      v = __ldg(reinterpret_cast<const float4*>(row_ptr + k));
    } else {
      v.x = __ldg(row_ptr + k);
      if (k + 1 < k_end) v.y = __ldg(row_ptr + k + 1);
      if (k + 2 < k_end) v.z = __ldg(row_ptr + k + 2);
      if (k + 3 < k_end) v.w = __ldg(row_ptr + k + 3);
    }
  }
  return v;
}

// A tile of `rows` rows x UMMA_BK floats is moved in warp-chunks of 8 rows x 4 kc chunks
// (lane & 7 -> row, lane >> 3 -> kc): a quarter warp writes 128 contiguous bytes of shared memory
// (conflict-free) and the warp reads 8 x 64 contiguous bytes of global memory.  A thread owns the same N
// (row, kc) positions of every stage it fills - warp-chunks wc0, wc0 + 4, ... , i.e. rows 32 apart - so everything
// about chunk i follows from chunk 0 (kept as scalars, not arrays: the producers also hold two stages of
// operand data in registers):  pointer = ptr0 + i * step,  plane offset = soff0 + 128 i floats,
// tile-relative row = row0 + 32 i.  Rows at or beyond rows_valid (tile edge / device-side row count) read as zero.
template <int N>
struct UmmaChunks {
  const float* ptr0;   // row-major: &A[row, kq];  transposed: &A[kq, row]
  int64_t step;        // row-major: 32 * ld;  transposed: 32
  int soff0;           // (kc * rows + row0) * 4
  int n_own;           // chunks [0, n_own) exist in this tile (narrow W tiles own fewer)
  int row0;            // lane's row inside the tile for chunk 0
  int rows_valid;      // rows of the tile backed by data
  int kq;              // kc * 4
};

template <int N>
__device__ __forceinline__ void umma_chunks_load(float4 (&v)[N], const UmmaChunks<N>& c, int k0, int k_end,
                                                 bool vec_ok) {
  const bool full = vec_ok && k0 + UMMA_BK <= k_end;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < c.n_own && c.row0 + 32 * i < c.rows_valid) {
      const float* p = c.ptr0 + i * c.step + k0;
      if (full) {
        t = __ldg(reinterpret_cast<const float4*>(p));
      } else {
        const int k = k0 + c.kq;
        if (k < k_end) t.x = __ldg(p);
        if (k + 1 < k_end) t.y = __ldg(p + 1);
        if (k + 2 < k_end) t.z = __ldg(p + 2);
        if (k + 3 < k_end) t.w = __ldg(p + 3);
      }
    }
    v[i] = t;
  }
}

// transposed operand: the chunk (row, k .. k+3) is read from base[(k + j) * ld + row] with scalar loads.  Eight
// lanes (rows) share a 32-byte sector per k, so the reads stay sector-efficient.
template <int N>
__device__ __forceinline__ void umma_chunks_load_t(float4 (&v)[N], const UmmaChunks<N>& c, int k0, int k_end,
                                                   int64_t ld) {
#pragma unroll
  for (int i = 0; i < N; ++i) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < c.n_own && c.row0 + 32 * i < c.rows_valid) {
      const int k = k0 + c.kq;
      const float* p = c.ptr0 + i * c.step + (int64_t)k0 * ld;
      if (k < k_end) t.x = __ldg(p);
      if (k + 1 < k_end) t.y = __ldg(p + ld);
      if (k + 2 < k_end) t.z = __ldg(p + 2 * ld);
      if (k + 3 < k_end) t.w = __ldg(p + 3 * ld);
    }
    v[i] = t;
  }
}

template <int N>
__device__ __forceinline__ void umma_chunks_store(float* hi_plane, float* lo_plane, const UmmaChunks<N>& c,
                                                  const float4 (&v)[N]) {
#pragma unroll
  for (int i = 0; i < N; ++i) {
    if (i < c.n_own) {
      float4 h, l;
      tf32_split(v[i], h, l);
      *reinterpret_cast<float4*>(hi_plane + c.soff0 + 128 * i) = h;
      *reinterpret_cast<float4*>(lo_plane + c.soff0 + 128 * i) = l;
    }
  }
}

// (row, kc) of warp-chunk `wc` for this lane
__device__ __forceinline__ void umma_chunk_pos(int wc, int lane, int& row, int& kc) {
  row = wc * 8 + (lane & 7);
  kc = lane >> 3;
}

// ---- pre-split weight packs -------------------------------------------------------------------
// Parameters are split once per update into the exact shared-memory image of the B operand:
//     pack[tile][k-block][plane: head, tail][kc][row 0..bn-1][4 floats]
// so that a pipeline stage of B (both planes, bn * 128 bytes) is ONE contiguous TMA bulk copy and costs
// the SM no instructions.  Rows / columns beyond the matrix are zero.
// (the packed / tensor-memory kernels move TS_BK = 32 floats of K per stage: per-stage costs - barrier
// wait, fence, commit - are paid once per 4 k-steps; measured with tools/umma_bench.cu the MMAs
// themselves run at their math floor of N/2 cycles when issued back to back)
#define TS_BK 32
#define TS_KCH (TS_BK / 4)
#define UMMA_PACK_STAGE_FLOATS(bn) ((bn) * 2 * TS_KCH * 4)

// ---- MMA issue -------------------------------------------------------------------------------
// tf32x3: per k-step three MMAs  tail*head, head*tail (cross terms) and head*head.  They are issued by
// THREE warps (one elected thread each, role 0/1/2), each into its own TMEM accumulator(s):
//   role 0: A tail  x B head -> accumulator 0          role 1: A head x B tail -> accumulator 1
//   role 2: A head  x B head -> accumulator 2 (even k-steps) / 3 (odd k-steps)
// Why three issuers: one tf32 MMA covers only K = 8, so at the tile widths that fill 148 SMs with this
// path's small row counts an MMA lasts 16-64 cycles - less than one thread needs to build and issue
// it; three threads keep the tensor pipe fed.  Why separate accumulators: MMAs of different issuers are
// not ordered, and the tensor core truncates when it adds into the fp32 accumulator (a bias growing
// with the number of accumulation steps), so the large head*head products are also spread over two
// accumulators; the four partial sums are added with round-to-nearest in the epilogue.
#define UMMA_ISSUERS 3
#define UMMA_ACCS 4

// descriptor words: lo = (address >> 4) | (LBO >> 4) << 16 ; hi = (SBO >> 4) | version 1 << 14 (SBO = 128 B)
#define UMMA_DESC_HI ((128u >> 4) | (1u << 14))
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t saddr, uint32_t rows) {
  return ((saddr & 0x3FFFFu) >> 4) | (rows << 16);   // LBO = rows * 16 bytes
}
__device__ __forceinline__ void umma_tf32_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(UMMA_DESC_HI)
      : "memory");
}

// Same with the A operand in tensor memory (128 lanes = rows, 8 consecutive 32-bit columns = one k-step):
// the producers write the split activations straight into TMEM (tcgen05.st), so an MMA reads only its
// B tile from shared memory - at the narrow tiles of this path the A read of the shared-memory form
// costs more than the math.
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], db, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(UMMA_DESC_HI)
      : "memory");
}

// Per-issuer constants of one operand pair (A tile of a_rows rows, B tile of b_rows rows, both
// [hi plane | lo plane] back to back, B directly after A inside a stage).
struct UmmaRole {
  uint32_t a_lo, b_lo;       // descriptor lo words for stage 0, k-step 0
  uint32_t a_kstep, b_kstep; // lo-word increment per k-step (two 16-byte K chunks)
  uint32_t stage_step;       // lo-word increment per stage
  uint32_t acc_even, acc_odd;  // TMEM column offsets of this role's accumulator for even / odd k-steps
};
__device__ __forceinline__ UmmaRole umma_role(int role, uint32_t stage0_addr, uint32_t stage_bytes, int a_rows,
                                              int b_rows, uint32_t acc_stride) {
  const uint32_t a_plane = (uint32_t)UMMA_KCH * a_rows * 16u, b_plane = (uint32_t)UMMA_KCH * b_rows * 16u;
  UmmaRole r;
  r.a_lo = umma_desc_lo(stage0_addr + (role == 0 ? a_plane : 0u), (uint32_t)a_rows);
  r.b_lo = umma_desc_lo(stage0_addr + 2u * a_plane + (role == 1 ? b_plane : 0u), (uint32_t)b_rows);
  r.a_kstep = 2u * a_rows;
  r.b_kstep = 2u * b_rows;
  r.stage_step = stage_bytes >> 4;
  r.acc_even = (uint32_t)role * acc_stride;
  r.acc_odd = role == 2 ? 3u * acc_stride : r.acc_even;
  return r;
}
