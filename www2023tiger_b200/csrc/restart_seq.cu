// Seq restarter: SeqRestarter.forward (tiger/model/restarters.py:51-114) as a short launch sequence
//   tiger_min_time        restart() is called with ts.min() of the batch (train_self_supervised.py:161)
//   tiger_find_recent     get_history(nids, t, hist_len)                       (graph.cu)
//   tiger_anonymized_reindex                                                   (select.cu)
//   tiger_seq_tokens      event tokens [src | dst | anony | edge | time], key-padding mask, prev_ts
//   tiger_sgemm_nt        packed q,k in-projection of all tokens               (gemm.cu)
//   tiger_train_seq_pool  per (node, head): L x L scores, masked softmax, position-mean of the
//                         attention weights, pooled tokens xbar_h = sum_i pbar_hi x_i  (train_seq.cu, dropout 0)
//   tiger_sgemm_nt x5     value projection of the pooled tokens (per head), out-proj (+ReLU), out_fn,
//                         merger fc1 (+ReLU, first d input columns only), merger fc2
// Folding (exact by linearity, because the reference takes the MEAN over positions of the MHA output
// before anything non-linear): mean_j out_j = W_o [concat_h W_v,h xbar_h + b_v,h] + b_o.  The value
// projection and the out-projection therefore run on n rows instead of n * L.
// last_event_feat is identically zero in the reference (a view that is zeroed in place one line
// later, restarters.py:103-104), so the merger only sees h_prev_left (SURVEY.md Q13).
#include "common.cuh"

// ------------------------------------------------------------------------------------------
__global__ void min_time_kernel(const float* __restrict__ ts, int64_t n, double* __restrict__ out) {
  __shared__ float red[32];
  float m = INFINITY;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) m = fminf(m, ts[i]);
  m = warp_min(m);
  if (lane_id() == 0) red[warp_id_in_block()] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : INFINITY;
    m = warp_min(m);
    if (threadIdx.x == 0) out[0] = (double)m;
  }
}

extern "C" int tiger_min_time(const float* ts, int64_t n, double* out, void* stream) {
  if (n <= 0 || out == nullptr) return TIGER_EINVAL;
  min_time_kernel<<<1, 256, 0, as_stream(stream)>>>(ts, n, out);
  return tiger_launch_status();
}

// ------------------------------------------------------------------------------------------
// tokens: one warp per (node, position)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
seq_tokens_kernel(const int64_t* __restrict__ nids, const int32_t* __restrict__ count, int64_t n, int len,
                  const int64_t* __restrict__ hist_nids, const int64_t* __restrict__ hist_eids,
                  const float* __restrict__ hist_ts, const int64_t* __restrict__ hist_dirs,
                  const int64_t* __restrict__ anony_ids, const float* __restrict__ nfeats,
                  const float* __restrict__ efeats, int d, int de, const float* __restrict__ anony_emb,
                  const float* __restrict__ time_w, const float* __restrict__ time_b, float* __restrict__ x,
                  uint8_t* __restrict__ mask, float* __restrict__ prev_ts) {
  int64_t total = n;
  if (count != nullptr) {
    const int64_t c = *count;
    total = c < n ? c : n;
  }
  total *= len;
  const int lane = lane_id();
  const int64_t dm = 4 * (int64_t)d + de;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); r < total; r += n_warps) {
    const int64_t i = r / len;
    const int j = (int)(r % len);
    const int64_t owner = nids[i];
    const int64_t hn = hist_nids[r], dir = hist_dirs[r];
    const float t_last = hist_ts[i * len + len - 1];
    float* row = x + r * dm;
    const bool last = j == len - 1;
    if (lane == 0) {
      mask[r] = (hn == 0) && !last;                      // mask[:, -1] = False (restarters.py:87)
      if (last) prev_ts[i] = t_last;
    }
    if (last) {
      for (int c = lane; c < 3 * d + de; c += 32) row[c] = 0.f;   // restarters.py:104
    } else {
      // the reference's literal direction rule (restarters.py:93-94, SURVEY.md Q6)
      const int64_t s_id = owner * dir + hn * (1 - dir);
      const int64_t d_id = owner * (1 - dir) + hn * dir;
      if (nfeats != nullptr) {
        warp_copy_row(row, nfeats + s_id * d, d, lane);
        warp_copy_row(row + d, nfeats + d_id * d, d, lane);
      } else {
        for (int c = lane; c < 2 * d; c += 32) row[c] = 0.f;
      }
      warp_copy_row(row + 2 * d, anony_emb + anony_ids[r] * d, d, lane);
      if (efeats != nullptr) {
        warp_copy_row(row + 3 * d, efeats + hist_eids[r] * de, de, lane);
      } else {
        for (int c = lane; c < de; c += 32) row[3 * d + c] = 0.f;
      }
    }
    const float dt = t_last - hist_ts[r];
    float* trow = row + 3 * d + de;
    for (int c = lane; c < d; c += 32) trow[c] = time_enc(dt, time_w[c], time_b[c]);
  }
}

extern "C" int tiger_seq_tokens(const int64_t* nids, const int32_t* count, int64_t n, int len,
                                const int64_t* hist_nids, const int64_t* hist_eids, const float* hist_ts,
                                const int64_t* hist_dirs, const int64_t* anony_ids, const float* nfeats,
                                const float* efeats, int d, int de, const float* anony_emb, const float* time_w,
                                const float* time_b, float* x, uint8_t* mask, float* prev_ts, void* stream) {
  if (n < 0 || len <= 0 || d <= 0 || de <= 0) return TIGER_EINVAL;
  if (n == 0) return TIGER_OK;
  const int64_t rows = n * len;
  int64_t grid = (rows + 7) / 8;
  if (grid > 148 * 8) grid = 148 * 8;
  seq_tokens_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(nids, count, n, len, hist_nids, hist_eids,
                                                                  hist_ts, hist_dirs, anony_ids, nfeats, efeats, d,
                                                                  de, anony_emb, time_w, time_b, x, mask, prev_ts);
  return tiger_launch_status();
}

// ------------------------------------------------------------------------------------------
// Small-R tail of the seq restarter.  After the pooling kernel the path is five dependent layers on the n pooled
// rows - value projection per head, out-projection (+ReLU), out_fn, merger fc1 (+ReLU), fc2 - and in steady state
// n is ~20-50 (the nodes a batch touches for the first time).  As tensor-core products each layer is one CTA per
// tile walking 54 dependent k-steps (K = d_model = 860): 6 launches x 33 us for a few hundred MFLOP.  Here each layer
// is a matrix-vector kernel with one warp per output channel (108 CTAs for the d_model-wide layers), chained by
// programmatic dependent launch so that a layer's weight rows are already in registers when its input arrives.
// (First attempt: all five layers in one CTA per row - 139 us, one row's 6.6 MB of weights through one SM.)  With
// many restarted rows (the first batches of a chunk) the tensor-core products win: tiger_seq_gate_count splits the
// device-side row count into (count if <= max_rows else 0, count if > max_rows else 0) and both routes are launched.
// ------------------------------------------------------------------------------------------
__global__ void seq_gate_count_kernel(const int32_t* __restrict__ count, int32_t max_rows, int32_t* __restrict__ small,
                                      int32_t* __restrict__ big) {
  const int32_t c = *count;
  *small = c <= max_rows ? c : 0;
  *big = c > max_rows ? c : 0;
}

extern "C" int tiger_seq_gate_count(const int32_t* count, int max_rows, int32_t* count_small, int32_t* count_big,
                                    void* stream) {
  if (count == nullptr || count_small == nullptr || count_big == nullptr) return TIGER_EINVAL;
  seq_gate_count_kernel<<<1, 1, 0, as_stream(stream)>>>(count, max_rows, count_small, count_big);
  return tiger_launch_status();
}

// One layer y[r, g*n_out + c] = act(bias[g*n_out + c] + W[g*n_out + c, :k] . x[r, g*x_grp_off : +k]) on the first
// min(n_cap, *count) rows.  One warp per output channel keeps the channel's weight row in registers (fetched before
// the wait on the producing kernel: weights do not depend on it) and walks the rows in groups of TAIL_RT staged in
// shared memory.  Group g (blockIdx.y) is the attention head of the value projection, 0 elsewhere.
#define TAIL_WARPS 8
#define TAIL_RT 8
template <int KREG, bool VEC>
__global__ void __launch_bounds__(TAIL_WARPS * 32)
seq_tail_layer_kernel(const float* __restrict__ x, int64_t ldx, int64_t x_grp_off, const float* __restrict__ W, int64_t ldw,
                      const float* __restrict__ bias, const float* __restrict__ bias_scale, float* __restrict__ y, int64_t ldy,
                      const int32_t* __restrict__ count, int64_t n_cap, int k, int n_out, int relu, float p_drop,
                      uint32_t seed) {
  seed = tiger_step_seed(seed);
  extern __shared__ __align__(16) float tail_xs[];          // [TAIL_RT][32 * KREG]
  constexpr int KP = 32 * KREG;
  constexpr int NT = TAIL_WARPS * 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = blockIdx.y, c = blockIdx.x * TAIL_WARPS + warp;
  const bool live = c < n_out;
  // VEC (16-byte aligned rows, k % 4 == 0): lane l holds elements [4 (l + 32 j), +4) of the weight row, else l + 32 j
  float wr[KREG];
  float b = 0.f;
  {
    const float* w = W + ((int64_t)g * n_out + (live ? c : 0)) * ldw;
    if (VEC) {
      const float4* w4 = reinterpret_cast<const float4*>(w);
#pragma unroll
      for (int j = 0; j < KREG / 4; ++j) {
        const int i4 = lane + 32 * j;
        const float4 v = (live && 4 * i4 < k) ? __ldg(w4 + i4) : make_float4(0.f, 0.f, 0.f, 0.f);
        wr[4 * j] = v.x; wr[4 * j + 1] = v.y; wr[4 * j + 2] = v.z; wr[4 * j + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < KREG; ++j) {
        const int idx = lane + 32 * j;
        wr[j] = (live && idx < k) ? __ldg(w + idx) : 0.f;
      }
    }
    if (live && bias != nullptr) b = __ldg(bias + g * n_out + c);
  }
  pdl_trigger();
  pdl_wait();
  int64_t n = n_cap;
  if (count != nullptr) {
    const int64_t cc = *count;
    n = cc < n ? cc : n;
  }
  const float* xg = x + (int64_t)g * x_grp_off;
  for (int64_t r0 = 0; r0 < n; r0 += TAIL_RT) {
    const int rows = (int)((n - r0) < TAIL_RT ? (n - r0) : TAIL_RT);
    __syncthreads();
    if (VEC) {
      // all loads of the pass first (KREG / 4 independent 16-byte loads per thread), then the stores: the first version
      // walked 32 dependent load -> store iterations per pass and took 38 us per layer under ncu
      constexpr int NV = TAIL_RT * KP / 4 / NT;
      float4 v[NV];
#pragma unroll
      for (int t = 0; t < NV; ++t) {
        const int i = tid + t * NT;
        const int rr = i / (KP / 4), c4 = i % (KP / 4);
        v[t] = (rr < rows && 4 * c4 < k) ? *reinterpret_cast<const float4*>(xg + (r0 + rr) * ldx + 4 * c4)
                                          : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int t = 0; t < NV; ++t) reinterpret_cast<float4*>(tail_xs)[tid + t * NT] = v[t];
    } else {
      for (int i = tid; i < TAIL_RT * KP; i += NT) {
        const int rr = i / KP, col = i % KP;
        tail_xs[i] = (rr < rows && col < k) ? xg[(r0 + rr) * ldx + col] : 0.f;
      }
    }
    __syncthreads();
    float acc[TAIL_RT];
#pragma unroll
    for (int rr = 0; rr < TAIL_RT; ++rr) acc[rr] = 0.f;
    if (VEC) {
#pragma unroll
      for (int j = 0; j < KREG / 4; ++j) {
#pragma unroll
        for (int rr = 0; rr < TAIL_RT; ++rr) {
          const float4 x4 = *reinterpret_cast<const float4*>(&tail_xs[rr * KP + 4 * (lane + 32 * j)]);
          acc[rr] = fmaf(wr[4 * j], x4.x, acc[rr]);
          acc[rr] = fmaf(wr[4 * j + 1], x4.y, acc[rr]);
          acc[rr] = fmaf(wr[4 * j + 2], x4.z, acc[rr]);
          acc[rr] = fmaf(wr[4 * j + 3], x4.w, acc[rr]);
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < KREG; ++j) {
#pragma unroll
        for (int rr = 0; rr < TAIL_RT; ++rr) acc[rr] = fmaf(wr[j], tail_xs[rr * KP + lane + 32 * j], acc[rr]);
      }
    }
    float mine = 0.f;
#pragma unroll
    for (int rr = 0; rr < TAIL_RT; ++rr) {
      const float s = warp_sum(acc[rr]);
      if (lane == rr) mine = s;
    }
    if (live && lane < rows) {
      // bias_scale [n, groups]: the value bias under attention dropout is b * (row sum of the kept probabilities)
      float v = mine + (bias_scale != nullptr ? b * bias_scale[(r0 + lane) * gridDim.y + g] : b);
      if (relu) v = fmaxf(v, 0.f);
      if (p_drop > 0.f)                                      // nn.Dropout of the merger (mask stream 4, element r * n_out + c)
        v = seq_keep(seed, 4u, (uint32_t)((r0 + lane) * n_out + c), p_drop) ? v * (1.0f / (1.0f - p_drop)) : 0.f;
      y[(r0 + lane) * ldy + (int64_t)g * n_out + c] = v;
    }
  }
}

template <int KREG>
static int tail_launch(bool vec, dim3 grid, dim3 block, cudaStream_t st, const float* x, int64_t ldx, int64_t x_grp_off,
                       const float* W, int64_t ldw, const float* bias, const float* bias_scale, float* y, int64_t ldy,
                       const int32_t* count, int64_t n, int k, int n_out, int relu, float p_drop, uint32_t seed) {
  const size_t smem = (size_t)TAIL_RT * 32 * KREG * sizeof(float);
  if (vec)
    return tiger_launch_chain(seq_tail_layer_kernel<KREG, true>, grid, block, smem, st, dim3(1, 1, 1), x, ldx, x_grp_off, W, ldw,
                              bias, bias_scale, y, ldy, count, n, k, n_out, relu, p_drop, seed);
  return tiger_launch_chain(seq_tail_layer_kernel<KREG, false>, grid, block, smem, st, dim3(1, 1, 1), x, ldx, x_grp_off, W, ldw,
                            bias, bias_scale, y, ldy, count, n, k, n_out, relu, p_drop, seed);
}

static int tail_layer(const float* x, int64_t ldx, int64_t x_grp_off, int groups, const float* W, int64_t ldw,
                      const float* bias, const float* bias_scale, float* y, int64_t ldy, const int32_t* count, int64_t n, int k,
                      int n_out, int relu, float p_drop, uint32_t seed, cudaStream_t st) {
  const dim3 grid((unsigned)((n_out + TAIL_WARPS - 1) / TAIL_WARPS), (unsigned)groups), block(TAIL_WARPS * 32);
  const bool vec = (k & 3) == 0 && (ldx & 3) == 0 && (ldw & 3) == 0 && (x_grp_off & 3) == 0 &&
                   (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0;
  if (k <= 256)
    return tail_launch<8>(vec, grid, block, st, x, ldx, x_grp_off, W, ldw, bias, bias_scale, y, ldy, count, n, k, n_out, relu,
                          p_drop, seed);
  if (k <= 512)
    return tail_launch<16>(vec, grid, block, st, x, ldx, x_grp_off, W, ldw, bias, bias_scale, y, ldy, count, n, k, n_out, relu,
                           p_drop, seed);
  return tail_launch<32>(vec, grid, block, st, x, ldx, x_grp_off, W, ldw, bias, bias_scale, y, ldy, count, n, k, n_out, relu,
                         p_drop, seed);
}

extern "C" int tiger_seq_tail(const float* xbar, const int32_t* count, int64_t n, int d_model, int n_head, int d,
                              const float* w_v, const float* b_v, const float* w_out, const float* b_out,
                              const float* w_fn, const float* b_fn, const float* w_fc1, int64_t ld_fc1, const float* b_fc1,
                              const float* w_fc2, const float* b_fc2, const float* psum, float p_drop, int seed, float* att,
                              float* o, float* hid, float* h_left, float* h_right, void* stream) {
  if (xbar == nullptr || w_v == nullptr || w_out == nullptr || w_fn == nullptr || w_fc1 == nullptr || w_fc2 == nullptr ||
      att == nullptr || o == nullptr || hid == nullptr || h_left == nullptr || h_right == nullptr || n < 0 ||
      d_model <= 0 || d_model > 1024 || p_drop < 0.f || p_drop >= 1.f || n_head <= 0 || d_model % n_head != 0 || d <= 0 || d > 1024 || ld_fc1 < d)
    return TIGER_EINVAL;
  if (n == 0) return TIGER_OK;
  cudaStream_t st = as_stream(stream);
  const int dm = d_model, hd = d_model / n_head;
  const uint32_t sd = (uint32_t)seed;
  int rc = tail_layer(xbar, (int64_t)n_head * dm, dm, n_head, w_v, dm, b_v, psum, att, dm, count, n, dm, hd, 0, 0.f, sd, st);
  if (rc == TIGER_OK) rc = tail_layer(att, dm, 0, 1, w_out, dm, b_out, nullptr, o, dm, count, n, dm, dm, 1, 0.f, sd, st);
  if (rc == TIGER_OK) rc = tail_layer(o, dm, 0, 1, w_fn, dm, b_fn, nullptr, h_left, d, count, n, dm, d, 0, 0.f, sd, st);
  if (rc == TIGER_OK)
    rc = tail_layer(h_left, d, 0, 1, w_fc1, ld_fc1, b_fc1, nullptr, hid, d, count, n, d, d, 1, p_drop, sd, st);
  if (rc == TIGER_OK) rc = tail_layer(hid, d, 0, 1, w_fc2, d, b_fc2, nullptr, h_right, d, count, n, d, d, 0, 0.f, sd, st);
  return rc;
}

int tiger_seed_step_set_restart_seq(const int32_t* p) { return tiger_seed_step_set_here(p); }
