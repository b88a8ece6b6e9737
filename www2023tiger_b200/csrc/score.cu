// Link scorer: step 7 of TIGE.contrast_learning (tiger/model/tiger.py:259-288), eval mode:
// hit flags (tiger.py:266-270, data_loader.py:61-75) -> hit term -> score_fn MergeLayer (basic_modules.py:16-19)
// on positive and negative pairs -> BCE-with-logits mean.
//
// Folded form (see tiger_score_fold_hit in attention.cu): the first scorer layer was applied to every
// embedding row by the last attention GEMM (PQ[row] = [W1a z | W1b z]); a pair (s, t) with hit flags a_j = [N(t)[j] == s],
// b_j = [N(s)[j] == t] scores  w2 . relu(P[s] + Q[t] + h(a, b)) + b2  with the hit term h of the hit type
// (compile-time mode HIT):
//   bin / none : c_ab[2 any(a) + any(b)]              (four pre-folded constants; none: c_00, no table read)
//   count      : U[sum a] + V[sum b]                  (hit embedding of the counts folded through W1a / W1b)
//   vec        : b1 + sum_{a_j} Ha^T[j] + sum_{b_j} Hb^T[j]   (the hit vectors' columns of fc1)
// Pairs are candidate-major: pair p = j Q + i of candidate column j (0: the true candidate pos[i], j >= 1: negs[(j-1) Q + i])
// scores row i of [src | column 0 | column 1 | ...] with row Q + p - the batch layout [src ; dst ; neg] at C = 2 and
// the query layout of a one-vs-many candidate query at any C.
// One warp per pair; the flags of 32 slots at a time come from one ballot per side.  The BCE mean (optional) is reduced
// by the last CTA in a fixed order, so the loss does not depend on the order in which the CTAs finish.
#include "common.cuh"

#define SCOREF_WARPS 8
// HIT = TIGER_HIT_BIN also serves 'none' (neigh == NULL); `cab` is the table of the hit type (c_ab, U | V or
// b1 | Ha^T | Hb^T, tiger_score_fold_hit_offset)
template <int HIT>
__global__ void __launch_bounds__(SCOREF_WARPS * 32)
link_score_folded_kernel(const float* __restrict__ pq, int64_t batch, int n_cands, int d,
                         const int64_t* __restrict__ src, const int64_t* __restrict__ pos,
                         const int64_t* __restrict__ negs,
                         const int64_t* __restrict__ neigh, int k, const float* __restrict__ cab,
                         const float* __restrict__ fc2_w, const float* __restrict__ fc2_b,
                         float* __restrict__ scores, float* __restrict__ loss, uint32_t* __restrict__ done_counter) {
  __shared__ float red[SCOREF_WARPS];
  __shared__ bool s_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n_pairs = (int64_t)n_cands * batch;
  const int64_t p = (int64_t)blockIdx.x * SCOREF_WARPS + warp;
  pdl_trigger();
  pdl_wait();      // PQ comes from the last attention product
  if (p < n_pairs) {
    const bool is_neg = p >= batch;
    const int64_t e = is_neg ? p % batch : p;
    const int64_t row_s = e, row_t = batch + p;     // rows of [src | column 0 | column 1 | ...]
    float acc = 0.f;
    if constexpr (HIT == TIGER_HIT_BIN) {
      int fa = 0, fb = 0;
      if (neigh != nullptr) {
        // src_hits: src in N(target) ; dst_hits: target in N(src)   (tiger.py:266-270, data_loader.py:61-75)
        const int64_t s_id = src[e], t_id = is_neg ? negs[p - batch] : pos[e];
        for (int j = lane; j < k; j += 32) {
          fa |= (neigh[row_t * k + j] == s_id);
          fb |= (neigh[row_s * k + j] == t_id);
        }
        fa = __any_sync(TIGER_FULL_MASK, fa);
        fb = __any_sync(TIGER_FULL_MASK, fb);
      }
      const float* P = pq + row_s * 2 * d;
      const float* Q = pq + row_t * 2 * d + d;
      const float* c = cab + (2 * fa + fb) * d;
      for (int j = lane; j < d; j += 32) acc = fmaf(fmaxf(P[j] + Q[j] + c[j], 0.f), fc2_w[j], acc);
    } else {
      const float* P = pq + row_s * 2 * d;
      const float* Q = pq + row_t * 2 * d + d;
      // slot flags a_j (src in N(target)) / b_j (target in N(src)) of slots [c0, c0 + 32), one ballot per side;
      // the loops around the ballots are warp-uniform
      const int64_t s_id = src[e], t_id = is_neg ? negs[p - batch] : pos[e];
      const int64_t *na = neigh + row_t * k, *nb = neigh + row_s * k;
      auto ballots = [&](int c0, uint32_t& ma, uint32_t& mb) {
        const int j = c0 + lane;
        ma = __ballot_sync(TIGER_FULL_MASK, j < k && na[j] == s_id);
        mb = __ballot_sync(TIGER_FULL_MASK, j < k && nb[j] == t_id);
      };
      if constexpr (HIT == TIGER_HIT_COUNT) {
        int ca = 0, cb = 0;
        for (int c0 = 0; c0 < k; c0 += 32) {
          uint32_t ma, mb;
          ballots(c0, ma, mb);
          ca += __popc(ma);
          cb += __popc(mb);
        }
        const float* U = cab + (int64_t)ca * d;
        const float* V = cab + (int64_t)(k + 1 + cb) * d;
        for (int j = lane; j < d; j += 32) acc = fmaf(fmaxf(P[j] + Q[j] + U[j] + V[j], 0.f), fc2_w[j], acc);
      } else {
        static_assert(HIT == TIGER_HIT_VEC, "hit mode");
        const float* Ha = cab + d;                        // Ha^T [K][d], then Hb^T [K][d]
        const float* Hb = cab + (int64_t)(1 + k) * d;
        uint32_t ma0, mb0;
        ballots(0, ma0, mb0);
        for (int j0 = 0; j0 < d; j0 += 32) {
          const int j = j0 + lane;
          float h = 0.f;
          for (int c0 = 0; c0 < k; c0 += 32) {            // K > 32: the later chunks' ballots again per column block
            uint32_t ma = ma0, mb = mb0;
            if (c0 > 0) ballots(c0, ma, mb);
            if (j < d) {
              for (; ma != 0u; ma &= ma - 1u) h += Ha[(int64_t)(c0 + __ffs(ma) - 1) * d + j];
              for (; mb != 0u; mb &= mb - 1u) h += Hb[(int64_t)(c0 + __ffs(mb) - 1) * d + j];
            }
          }
          if (j < d) acc = fmaf(fmaxf(P[j] + Q[j] + cab[j] + h, 0.f), fc2_w[j], acc);
        }
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) scores[p] = acc + fc2_b[0];
  }
  if (loss == nullptr) return;
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = (atomicAdd(done_counter, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  float a = 0.f;
  for (int64_t q = tid; q < n_pairs; q += blockDim.x) {
    const float x = __ldcg(scores + q);
    const float y = q < batch ? 1.f : 0.f;
    a += fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x)));
  }
  a = warp_sum(a);
  if (lane == 0) red[warp] = a;
  __syncthreads();
  if (tid == 0) {
    float s = 0.f;
    for (int w = 0; w < SCOREF_WARPS; ++w) s += red[w];
    *loss = s / (float)n_pairs;
    *done_counter = 0u;
  }
}

// ranks[i] = 1 + #{j >= 1 : s_ij > s_i0} + #{j >= 1 : s_ij == s_i0} / 2 over the candidate-major scores, one warp per
// query row; integer counts, so the result does not depend on the order of the lanes.  A NaN true score gives a NaN
// rank; a NaN candidate score neither beats nor ties the true one.
__global__ void __launch_bounds__(SCOREF_WARPS * 32)
link_rank_kernel(const float* __restrict__ scores, int64_t batch, int n_cands, float* __restrict__ ranks) {
  const int lane = lane_id();
  const int64_t i = (int64_t)blockIdx.x * SCOREF_WARPS + warp_id_in_block();
  pdl_trigger();
  pdl_wait();      // the scores come from the scorer
  if (i >= batch) return;
  const float s0 = scores[i];
  int gt = 0, eq = 0;
  for (int j = 1 + lane; j < n_cands; j += 32) {
    const float s = scores[(int64_t)j * batch + i];
    gt += s > s0;
    eq += s == s0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    gt += __shfl_xor_sync(TIGER_FULL_MASK, gt, o);
    eq += __shfl_xor_sync(TIGER_FULL_MASK, eq, o);
  }
  if (lane == 0) ranks[i] = s0 == s0 ? 1.0f + (float)gt + 0.5f * (float)eq : s0;
}

extern "C" int tiger_link_score_cands(const float* pq, int64_t n_query, int n_cands, int d, const int64_t* src,
                                      const int64_t* pos, const int64_t* negs, const int64_t* neigh_nids, int k,
                                      int hit_type, const float* tables, const float* fc2_w, const float* fc2_b,
                                      float* scores, float* ranks, float* loss, uint32_t* done_counter, void* stream) {
  if (hit_type == TIGER_HIT_NONE) neigh_nids = nullptr;
  else if (hit_type != TIGER_HIT_BIN && hit_type != TIGER_HIT_VEC && hit_type != TIGER_HIT_COUNT) return TIGER_EINVAL;
  else if (neigh_nids == nullptr || k <= 0) return TIGER_EINVAL;
  if (pq == nullptr || tables == nullptr || n_query < 0 || n_cands < 1 || d <= 0 || scores == nullptr) return TIGER_EINVAL;
  if (n_cands > 1 && negs == nullptr) return TIGER_EINVAL;
  if (loss != nullptr && done_counter == nullptr) return TIGER_EINVAL;
  if (n_query == 0) return TIGER_OK;
  const int64_t n_pairs = (int64_t)n_cands * n_query;
  if ((n_pairs + SCOREF_WARPS - 1) / SCOREF_WARPS > 0x7fffffffll) return TIGER_EINVAL;
  const unsigned grid = (unsigned)((n_pairs + SCOREF_WARPS - 1) / SCOREF_WARPS);
  decltype(&link_score_folded_kernel<TIGER_HIT_BIN>) kernel =
      hit_type == TIGER_HIT_VEC     ? link_score_folded_kernel<TIGER_HIT_VEC>
      : hit_type == TIGER_HIT_COUNT ? link_score_folded_kernel<TIGER_HIT_COUNT>
                                    : link_score_folded_kernel<TIGER_HIT_BIN>;
  int rc = tiger_launch_chain(kernel, dim3(grid), dim3(SCOREF_WARPS * 32), 0, as_stream(stream), dim3(1, 1, 1), pq,
                              n_query, n_cands, d, src, pos, negs, neigh_nids, k, tables, fc2_w, fc2_b, scores, loss,
                              done_counter);
  if (rc != TIGER_OK || ranks == nullptr) return rc;
  return tiger_launch_chain(link_rank_kernel, dim3((unsigned)((n_query + SCOREF_WARPS - 1) / SCOREF_WARPS)),
                            dim3(SCOREF_WARPS * 32), 0, as_stream(stream), dim3(1, 1, 1), (const float*)scores, n_query,
                            n_cands, ranks);
}

extern "C" int tiger_link_score_folded_hit(const float* pq, int64_t batch, int d, const int64_t* src,
                                           const int64_t* dst, const int64_t* neg, const int64_t* neigh_nids, int k,
                                           int hit_type, const float* tables, const float* fc2_w, const float* fc2_b,
                                           float* scores, float* loss, uint32_t* done_counter, void* stream) {
  if (batch < 0) return TIGER_EINVAL;
  return tiger_link_score_cands(pq, batch, 2, d, src, dst, neg, neigh_nids, k, hit_type, tables, fc2_w, fc2_b, scores,
                                nullptr, loss, done_counter, stream);
}

extern "C" int tiger_link_score_folded(const float* pq, int64_t batch, int d, const int64_t* src, const int64_t* dst,
                                       const int64_t* neg, const int64_t* neigh_nids, int k, const float* cab,
                                       const float* fc2_w, const float* fc2_b, float* scores, float* loss,
                                       uint32_t* done_counter, void* stream) {
  return tiger_link_score_folded_hit(pq, batch, d, src, dst, neg, neigh_nids, k,
                                     neigh_nids != nullptr ? TIGER_HIT_BIN : TIGER_HIT_NONE, cab, fc2_w, fc2_b, scores,
                                     loss, done_counter, stream);
}
