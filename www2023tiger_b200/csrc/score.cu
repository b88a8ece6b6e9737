// Link scorer: step 7 of TIGE.contrast_learning (tiger/model/tiger.py:259-288), eval mode:
// hit flags ('bin': tiger.py:266-270, data_loader.py:61-75) -> hit embedding -> score_fn
// MergeLayer (basic_modules.py:16-19) on positive and negative pairs -> BCE-with-logits mean.
//
// Folded form (see tiger_score_fold in attention.cu): the first scorer layer was applied to every
// embedding row by the last attention GEMM (PQ[row] = [W1a z | W1b z]); a pair (s, t) with hit flags (a, b)
// scores  w2 . relu(P[s] + Q[t] + c_ab) + b2.  One warp per pair; the BCE mean is reduced by the last CTA
// in a fixed order, so the loss does not depend on the order in which the CTAs finish.
#include "common.cuh"

#define SCOREF_WARPS 8
__global__ void __launch_bounds__(SCOREF_WARPS * 32)
link_score_folded_kernel(const float* __restrict__ pq, int64_t batch, int d, const int64_t* __restrict__ src,
                         const int64_t* __restrict__ dst, const int64_t* __restrict__ neg,
                         const int64_t* __restrict__ neigh, int k, const float* __restrict__ cab,
                         const float* __restrict__ fc2_w, const float* __restrict__ fc2_b,
                         float* __restrict__ scores, float* __restrict__ loss, uint32_t* __restrict__ done_counter) {
  __shared__ float red[SCOREF_WARPS];
  __shared__ bool s_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n_pairs = 2 * batch;
  const int64_t p = (int64_t)blockIdx.x * SCOREF_WARPS + warp;
  pdl_trigger();
  pdl_wait();      // PQ comes from the last attention product
  if (p < n_pairs) {
    const bool is_neg = p >= batch;
    const int64_t e = is_neg ? p - batch : p;
    const int64_t row_s = e, row_t = is_neg ? 2 * batch + e : batch + e;     // rows of [src ; dst ; neg]
    int fa = 0, fb = 0;
    if (neigh != nullptr) {
      // src_hits: src in N(target) ; dst_hits: target in N(src)   (tiger.py:266-270, data_loader.py:61-75)
      const int64_t s_id = src[e], t_id = is_neg ? neg[e] : dst[e];
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
    float acc = 0.f;
    for (int j = lane; j < d; j += 32) acc = fmaf(fmaxf(P[j] + Q[j] + c[j], 0.f), fc2_w[j], acc);
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

extern "C" int tiger_link_score_folded(const float* pq, int64_t batch, int d, const int64_t* src, const int64_t* dst,
                                       const int64_t* neg, const int64_t* neigh_nids, int k, const float* cab,
                                       const float* fc2_w, const float* fc2_b, float* scores, float* loss,
                                       uint32_t* done_counter, void* stream) {
  if (pq == nullptr || cab == nullptr || batch < 0 || d <= 0 || (neigh_nids != nullptr && k <= 0)) return TIGER_EINVAL;
  if (loss != nullptr && done_counter == nullptr) return TIGER_EINVAL;
  if (batch == 0) return TIGER_OK;
  const unsigned grid = (unsigned)((2 * batch + SCOREF_WARPS - 1) / SCOREF_WARPS);
  return tiger_launch_chain(link_score_folded_kernel, dim3(grid), dim3(SCOREF_WARPS * 32), 0, as_stream(stream),
                            dim3(1, 1, 1), pq, batch, d, src, dst, neg, neigh_nids, k, cab, fc2_w, fc2_b, scores, loss,
                            done_counter);
}
