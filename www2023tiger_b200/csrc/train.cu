// Training step of the per-batch memory path: the forward pieces that must keep what backward needs, and the
// hand-written backward of every differentiable operator of TIGER.contrast_and_mutual_learning
// (tiger/model/tiger.py:547-592) - what `loss.backward(); optimizer.step()` of the reference's loops
// (train_self_supervised.py:165-171, train_self_supervised_ddp.py:203-208) runs through autograd, cuBLAS and ATen.
//
// The dense products (all nn.Linear / in_proj / GRUCell products and their input / weight gradients) run on the
// tensor-core kernel of gemm.cu (tiger_sgemm_ex: y = x W^T, dx = dy W, dW += dy^T x on the tensors as stored).
// This file holds everything in between, each a bandwidth-bound pass over a few MB that stays in L2:
//   GRU          gather of pending messages + state (kept for the weight gradients), gates forward / backward
//   attention    kv / query row builder (representation lookup, edge features, time codes), single-query
//                multi-head core with dropout forward / backward, scatter of the representation gradients back
//                onto the GRU rows, TimeEncode gradients
//   link scorer  hit-embedding add + pair rows, dropout + second layer + BCE (forward and gradient), pair backward
//   restarter    MSE over valid rows (mutual loss) forward + gradient, row scatter-add for nn.Embedding gradients
//   shared       column sums (bias gradients), ReLU backward, masked-row zeroing, Adam
// Gradients ACCUMULATE (atomic adds into buffers the optimizer kernel zeroes), like autograd's AccumulateGrad: a
// parameter used twice (the time encoder) simply receives two contributions.
#include "common.cuh"

// counter-based dropout mask: the same (seed, stream, index) gives the same decision in forward and backward
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ bool dropout_keep(uint32_t seed, uint32_t stream, uint32_t idx, float p) {
  if (p <= 0.f) return true;
  const uint32_t h = mix32(idx ^ mix32(seed + 0x9E3779B9u * (stream + 1u)));
  return (float)(h >> 8) * (1.0f / 16777216.0f) >= p;
}

__device__ __forceinline__ int64_t bounded_rows(const int32_t* count, int64_t n, int64_t per = 1) {
  if (count == nullptr) return n;
  const int64_t c = (int64_t)(*count) * per;
  return c < n ? c : n;
}

// sin with the double-precision range reduction of cos_reduced (common.cuh): arguments reach 1e6 rad
__device__ __forceinline__ float sin_reduced(float x) {
  const double xd = (double)x;
  const double n = rint(xd * 0.15915494309189535);
  double r = fma(-n, 6.283185307179586, xd);
  r = fma(-n, 2.4492935982947064e-16, r);
  return sinf((float)r);
}

// ------------------------------------------------------------------------------------------
// GRU (tiger.py:292-356, update_modules.py:30-37)
// ------------------------------------------------------------------------------------------
// X[r] = msg_vals[ids[r]], H[r] = upd_vals[ids[r]] for r < *count (copies: steps 4-5 overwrite the table rows before
// backward needs them); the message-clock invariants of compute_messages (message_modules.py:157-159, tiger.py:324-327)
__global__ void __launch_bounds__(256)
train_gather_pending_kernel(const int64_t* __restrict__ ids, const int32_t* __restrict__ count, int64_t cap,
                            const float* __restrict__ msg_vals, int m_dim, const float* __restrict__ msg_ts,
                            const float* __restrict__ upd_vals, int d, const float* __restrict__ check_mem_ts,
                            int check_equal, float* __restrict__ X, float* __restrict__ H, float* __restrict__ dh_zero,
                            uint32_t* __restrict__ err_flags, float* __restrict__ n_rows_out) {
  const int64_t n = bounded_rows(count, cap);
  if (n_rows_out != nullptr && blockIdx.x == 0 && threadIdx.x == 0) n_rows_out[0] = (float)n;
  const int lane = lane_id();
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); r < n; r += n_warps) {
    const int64_t u = ids[r];
    warp_copy_row(X + r * m_dim, msg_vals + u * m_dim, m_dim, lane);
    warp_copy_row(H + r * d, upd_vals + u * d, d, lane);
    if (dh_zero != nullptr)
      for (int c = lane; c < d; c += 32) dh_zero[r * d + c] = 0.f;
    if (lane == 0 && check_mem_ts != nullptr && err_flags != nullptr) {
      const float mt = msg_ts[u], pt = check_mem_ts[u];
      if (pt > mt) atomicOr(err_flags, TIGER_ERR_MSG_BEFORE_MEM);
      if (check_equal && mt != pt) atomicOr(err_flags, TIGER_ERR_MSG_TS_MISMATCH);
    }
  }
}

extern "C" int tiger_train_gather_pending(const int64_t* ids, const int32_t* count, int64_t cap, const float* msg_vals,
                                          int m_dim, const float* msg_ts, const float* upd_vals, int d,
                                          const float* check_mem_ts, int check_equal, float* X, float* H,
                                          float* dh_zero, uint32_t* err_flags, float* n_rows_out, void* stream) {
  if (ids == nullptr || msg_vals == nullptr || upd_vals == nullptr || X == nullptr || H == nullptr || cap < 0 ||
      m_dim <= 0 || d <= 0)
    return TIGER_EINVAL;
  if (cap == 0) return TIGER_OK;
  int64_t grid = (cap + 7) / 8;
  if (grid > 148 * 4) grid = 148 * 4;
  train_gather_pending_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(
      ids, count, cap, msg_vals, m_dim, msg_ts, upd_vals, d, check_mem_ts, check_equal, X, H, dh_zero, err_flags,
      n_rows_out);
  return tiger_launch_status();
}

// Gi = x W_ih^T + b_ih, Gh = h W_hh^T + b_hh (gate order r, z, n): r = s(Gi_r + Gh_r), z = s(Gi_z + Gh_z),
// n = tanh(Gi_n + r * Gh_n), h' = (1 - z) n + z h.  Keeps r, z, n and q = Gh_n for backward.
__global__ void train_gru_gates_kernel(const float* __restrict__ Gi, const float* __restrict__ Gh,
                                       const float* __restrict__ H, const int32_t* __restrict__ count, int64_t cap,
                                       int d, float* __restrict__ h_new, float* __restrict__ r_out,
                                       float* __restrict__ z_out, float* __restrict__ n_out) {
  const int64_t total = bounded_rows(count, cap) * d;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / d;
    const int c = (int)(i % d);
    const float* gi = Gi + row * 3 * d;
    const float* gh = Gh + row * 3 * d;
    const float r = sigmoidf_acc(gi[c] + gh[c]);
    const float z = sigmoidf_acc(gi[d + c] + gh[d + c]);
    const float n = tanhf(gi[2 * d + c] + r * gh[2 * d + c]);
    const float h = H[i];
    h_new[i] = (1.0f - z) * n + z * h;
    r_out[i] = r;
    z_out[i] = z;
    n_out[i] = n;
  }
}

extern "C" int tiger_train_gru_gates(const float* Gi, const float* Gh, const float* H, const int32_t* count,
                                     int64_t cap, int d, float* h_new, float* r_out, float* z_out, float* n_out,
                                     void* stream) {
  if (Gi == nullptr || Gh == nullptr || H == nullptr || h_new == nullptr || cap < 0 || d <= 0) return TIGER_EINVAL;
  if (cap == 0) return TIGER_OK;
  int64_t grid = (cap * d + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  train_gru_gates_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(Gi, Gh, H, count, cap, d, h_new, r_out, z_out,
                                                                       n_out);
  return tiger_launch_status();
}

// dGi = [dr_pre | dz_pre | dn_pre], dGh = [dr_pre | dz_pre | dn_pre * r]; Gh (its n block = q) is read, dGi/dGh written
__global__ void train_gru_gates_bwd_kernel(const float* __restrict__ dh, const float* __restrict__ r_in,
                                           const float* __restrict__ z_in, const float* __restrict__ n_in,
                                           const float* __restrict__ Gh, const float* __restrict__ H,
                                           const int32_t* __restrict__ count, int64_t cap, int d,
                                           float* __restrict__ dGi, float* __restrict__ dGh) {
  const int64_t total = bounded_rows(count, cap) * d;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / d;
    const int c = (int)(i % d);
    const float g = dh[i], r = r_in[i], z = z_in[i], n = n_in[i], h = H[i];
    const float q = Gh[row * 3 * d + 2 * d + c];
    const float dn_pre = g * (1.0f - z) * (1.0f - n * n);
    const float dz_pre = g * (h - n) * z * (1.0f - z);
    const float dr_pre = dn_pre * q * r * (1.0f - r);
    float* gi = dGi + row * 3 * d;
    float* gh = dGh + row * 3 * d;
    gi[c] = dr_pre;
    gi[d + c] = dz_pre;
    gi[2 * d + c] = dn_pre;
    gh[c] = dr_pre;
    gh[d + c] = dz_pre;
    gh[2 * d + c] = dn_pre * r;
  }
}

extern "C" int tiger_train_gru_gates_bwd(const float* dh, const float* r_in, const float* z_in, const float* n_in,
                                         const float* Gh, const float* H, const int32_t* count, int64_t cap, int d,
                                         float* dGi, float* dGh, void* stream) {
  if (dh == nullptr || dGi == nullptr || dGh == nullptr || cap < 0 || d <= 0) return TIGER_EINVAL;
  if (cap == 0) return TIGER_OK;
  int64_t grid = (cap * d + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  train_gru_gates_bwd_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(dh, r_in, z_in, n_in, Gh, H, count, cap, d,
                                                                           dGi, dGh);
  return tiger_launch_status();
}

// ------------------------------------------------------------------------------------------
// temporal attention (temporal_agg_modules.py:29-83,210-235 + torch MHA, need_weights branch)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ const float* resolve_repr(int64_t nid, const float* rows_a, const float* rows_b,
                                                     const int32_t* sel, int d) {
  const int32_t r = sel[nid];
  return r >= 0 ? rows_b + (int64_t)r * d : rows_a + nid * d;
}

// One warp per row.  Rows [0, n_q*K): kv_in[i*K+j] = [repr(nb_ij) + nf | ef(e_ij) | cos((t_i - tau_ij) w + b)];
// rows [n_q*K, n_q*K + n_q): q_in[i] = [repr(center_i) + nf | cos(b)] and the same center row into cat[i, E:E+d]
// (the second input of the merger).  Query i's time is ts[(i / ts_group) % batch]; with key_rows (the lower layer's
// output, [n_q*K, d]) slot r takes key_rows[r] as its node part, with no node features added.
__global__ void __launch_bounds__(256)
train_attn_build_kernel(const int64_t* __restrict__ center, int64_t n_q, const float* __restrict__ ts, int64_t batch,
                        int64_t ts_group, const int64_t* __restrict__ nn, const int64_t* __restrict__ ne,
                        const float* __restrict__ nt, int K, const float* __restrict__ rows_a,
                        const float* __restrict__ rows_b, const float* __restrict__ key_rows,
                        const int32_t* __restrict__ sel, const float* __restrict__ nfeats,
                        const float* __restrict__ efeats, int d, int de, const float* __restrict__ time_w,
                        const float* __restrict__ time_b, float* __restrict__ q_in, float* __restrict__ kv_in,
                        float* __restrict__ cat, int64_t ld_cat, int cat_off) {
  const int lane = lane_id();
  const int C = 2 * d + de;
  const int64_t n_kv = n_q * K, total = n_kv + n_q;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); r < total; r += n_warps) {
    if (r < n_kv) {
      const int64_t i = r / K;
      const int64_t nid = nn[r];
      float* row = kv_in + r * C;
      if (key_rows != nullptr) {
        for (int c = lane; c < d; c += 32) row[c] = key_rows[r * d + c];
      } else {
        const float* src = resolve_repr(nid, rows_a, rows_b, sel, d);
        if (nfeats != nullptr) {
          for (int c = lane; c < d; c += 32) row[c] = src[c] + nfeats[nid * d + c];
        } else {
          for (int c = lane; c < d; c += 32) row[c] = src[c] + 0.0f;
        }
      }
      if (efeats != nullptr) {
        warp_copy_row(row + d, efeats + ne[r] * de, de, lane);
      } else {
        for (int c = lane; c < de; c += 32) row[d + c] = 0.f;
      }
      // (ts_group 1, the one-layer step, skips the 64-bit division)
      const float dt = ts[(ts_group == 1 ? i : i / ts_group) % batch] - nt[r];
      for (int c = lane; c < d; c += 32) row[d + de + c] = time_enc(dt, time_w[c], time_b[c]);
    } else {
      const int64_t i = r - n_kv;
      const int64_t nid = center[i];
      const float* src = resolve_repr(nid, rows_a, rows_b, sel, d);
      float* row = q_in + i * 2 * d;
      float* crow = cat + i * ld_cat + cat_off;
      for (int c = lane; c < d; c += 32) {
        const float v = src[c] + (nfeats != nullptr ? nfeats[nid * d + c] : 0.0f);
        row[c] = v;
        crow[c] = v;
        row[d + c] = time_enc(0.0f, time_w[c], time_b[c]);
      }
    }
  }
}

extern "C" int tiger_train_attn_build_ex(const int64_t* center, int64_t n_q, const float* ts, int64_t batch,
                                         int64_t ts_group, const int64_t* neigh_nids, const int64_t* neigh_eids,
                                         const float* neigh_ts, int k, const float* rows_a, const float* rows_b,
                                         const float* key_rows, const int32_t* sel, const float* nfeats,
                                         const float* efeats, int d, int de, const float* time_w, const float* time_b,
                                         float* q_in, float* kv_in, float* cat, int64_t ld_cat, int cat_off,
                                         void* stream) {
  if (center == nullptr || ts == nullptr || neigh_nids == nullptr || rows_a == nullptr || rows_b == nullptr ||
      sel == nullptr || q_in == nullptr || kv_in == nullptr || cat == nullptr || n_q < 0 || batch <= 0 ||
      ts_group <= 0 || k <= 0 || d <= 0 || de <= 0)
    return TIGER_EINVAL;
  if (n_q == 0) return TIGER_OK;
  int64_t grid = (n_q * (k + 1) + 7) / 8;
  if (grid > 148 * 8) grid = 148 * 8;
  train_attn_build_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(
      center, n_q, ts, batch, ts_group, neigh_nids, neigh_eids, neigh_ts, k, rows_a, rows_b, key_rows, sel, nfeats,
      efeats, d, de, time_w, time_b, q_in, kv_in, cat, ld_cat, cat_off);
  return tiger_launch_status();
}

#define ATT_MAXK 32

// One warp per (query, head).  s_j = (q_h * scale) . k_jh, padding (neighbor id 0) -> -inf, rows without any
// neighbor keep their last slot (and are flagged `empty`: their output is zero-filled downstream), softmax,
// dropout on the probabilities, o_h = sum_j p'_j v_jh.  P keeps the softmax output, keep_bits the dropout decisions.
template <int KT>
__global__ void __launch_bounds__(256)
train_attn_core_kernel(const float* __restrict__ Q, int64_t ldq, const float* __restrict__ Kp, const float* __restrict__ Vp,
                       int64_t ldkv, const int64_t* __restrict__ nn, int64_t n_q, int K, int n_head, int hd,
                       float p_drop, uint32_t seed, float* __restrict__ attn, int64_t ld_attn, float* __restrict__ P,
                       uint32_t* __restrict__ keep_bits, uint8_t* __restrict__ empty) {
  seed = tiger_step_seed(seed);
  // KT > 0: K is a compile-time constant, so the per-neighbor loops below unroll without branches and the K dot
  // products / reductions of one (query, head) overlap instead of forming one dependent chain each
  constexpr int KU = KT > 0 ? KT : ATT_MAXK;
  if (KT > 0) K = KT;
  const int lane = lane_id();
  const float scale = sqrtf(1.0f / (float)hd);
  const float inv_keep = p_drop > 0.f ? 1.0f / (1.0f - p_drop) : 1.0f;
  const int64_t total = n_q * n_head;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t item = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); item < total; item += n_warps) {
    const int64_t i = item / n_head;
    const int h = (int)(item % n_head);
    const float* q = Q + i * ldq + h * hd;
    float s[KU];
    bool any = false;
#pragma unroll
    for (int j = 0; j < KU; ++j) {
      if (j < K) {
        const float* kr = Kp + (i * K + j) * ldkv + h * hd;
        float acc = 0.f;
        for (int c = lane; c < hd; c += 32) acc = fmaf(q[c] * scale, kr[c], acc);
        acc = warp_sum(acc);
        const bool pad = nn[i * K + j] == 0;
        any |= !pad;
        s[j] = pad ? -INFINITY : acc;
      }
    }
    if (!any) {
      // temporal_agg_modules.py:224-225: unmask the last slot so that the softmax stays finite
      const float* kr = Kp + (i * K + K - 1) * ldkv + h * hd;
      float acc = 0.f;
      for (int c = lane; c < hd; c += 32) acc = fmaf(q[c] * scale, kr[c], acc);
      acc = warp_sum(acc);
#pragma unroll
      for (int j = 0; j < KU; ++j)
        if (j == K - 1) s[j] = acc;
    }
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < KU; ++j)
      if (j < K) m = fmaxf(m, s[j]);
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < KU; ++j)
      if (j < K) {
        s[j] = expf(s[j] - m);
        sum += s[j];
      }
    uint32_t bits = 0;
#pragma unroll
    for (int j = 0; j < KU; ++j)
      if (j < K) {
        s[j] = s[j] / sum;
        if (lane == 0) P[item * K + j] = s[j];
        const bool keep = dropout_keep(seed, 1u, (uint32_t)(item * K + j), p_drop);
        bits |= keep ? (1u << j) : 0u;
        s[j] = keep ? s[j] * inv_keep : 0.f;
      }
    if (lane == 0) {
      keep_bits[item] = bits;
      if (h == 0) empty[i] = any ? 0 : 1;
    }
    float* o = attn + i * ld_attn + h * hd;
    for (int c = lane; c < hd; c += 32) {
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < KU; ++j)
        if (j < K) acc = fmaf(s[j], Vp[(i * K + j) * ldkv + h * hd + c], acc);
      o[c] = acc;
    }
  }
}

extern "C" int tiger_train_attn_core(const float* Q, int64_t ldq, const float* Kp, const float* Vp, int64_t ldkv,
                                     const int64_t* neigh_nids, int64_t n_q, int k, int n_head, int head_dim,
                                     float p_drop, int seed, float* attn, int64_t ld_attn, float* P,
                                     uint32_t* keep_bits, uint8_t* empty, void* stream) {
  if (Q == nullptr || Kp == nullptr || Vp == nullptr || neigh_nids == nullptr || attn == nullptr || P == nullptr ||
      keep_bits == nullptr || empty == nullptr || n_q < 0 || k <= 0 || k > ATT_MAXK || n_head <= 0 || head_dim <= 0 ||
      p_drop < 0.f || p_drop >= 1.f)
    return TIGER_EINVAL;
  if (n_q == 0) return TIGER_OK;
  int64_t grid = (n_q * n_head + 7) / 8;
  if (grid > 148 * 8) grid = 148 * 8;
  auto launch = [&](auto kernel) {
    kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(Q, ldq, Kp, Vp, ldkv, neigh_nids, n_q, k, n_head, head_dim,
                                                          p_drop, (uint32_t)seed, attn, ld_attn, P, keep_bits, empty);
  };
  if (k == 10) launch(train_attn_core_kernel<10>);
  else if (k == 5) launch(train_attn_core_kernel<5>);
  else if (k == 20) launch(train_attn_core_kernel<20>);
  else launch(train_attn_core_kernel<0>);
  return tiger_launch_status();
}

// backward of the core: dV_j = p'_j do, dp'_j = do . v_j, dp_j = dp'_j * keep / (1 - p_drop),
// ds_j = p_j (dp_j - sum_l p_l dp_l), dq = scale * sum_j ds_j k_j, dk_j = scale * ds_j q.
template <int KT>
__global__ void __launch_bounds__(256)
train_attn_core_bwd_kernel(const float* __restrict__ dattn, int64_t ld_attn, const float* __restrict__ Q, int64_t ldq,
                           const float* __restrict__ Kp, const float* __restrict__ Vp, int64_t ldkv,
                           const float* __restrict__ P, const uint32_t* __restrict__ keep_bits, int64_t n_q, int K,
                           int n_head, int hd, float p_drop, float* __restrict__ dQ, float* __restrict__ dKp,
                           float* __restrict__ dVp) {
  constexpr int KU = KT > 0 ? KT : ATT_MAXK;
  if (KT > 0) K = KT;
  const int lane = lane_id();
  const float scale = sqrtf(1.0f / (float)hd);
  const float inv_keep = p_drop > 0.f ? 1.0f / (1.0f - p_drop) : 1.0f;
  const int64_t total = n_q * n_head;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t item = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); item < total; item += n_warps) {
    const int64_t i = item / n_head;
    const int h = (int)(item % n_head);
    const float* go = dattn + i * ld_attn + h * hd;
    const float* q = Q + i * ldq + h * hd;
    const uint32_t bits = keep_bits[item];
    float p[KU], ds[KU];
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < KU; ++j)
      if (j < K) {
        p[j] = P[item * K + j];
        const float m = ((bits >> j) & 1u) ? inv_keep : 0.f;
        const float* vr = Vp + (i * K + j) * ldkv + h * hd;
        float* dvr = dVp + (i * K + j) * ldkv + h * hd;
        float acc = 0.f;
        const float pd = p[j] * m;
        for (int c = lane; c < hd; c += 32) {
          const float g = go[c];
          acc = fmaf(g, vr[c], acc);
          dvr[c] = pd * g;
        }
        acc = warp_sum(acc) * m;          // dp_j
        ds[j] = acc;
        dot = fmaf(p[j], acc, dot);
      }
#pragma unroll
    for (int j = 0; j < KU; ++j)
      if (j < K) ds[j] = p[j] * (ds[j] - dot) * scale;
    float* dq = dQ + i * ldq + h * hd;
    for (int c = lane; c < hd; c += 32) {
      float acc = 0.f;
      const float qc = q[c];
#pragma unroll
      for (int j = 0; j < KU; ++j)
        if (j < K) {
          acc = fmaf(ds[j], Kp[(i * K + j) * ldkv + h * hd + c], acc);
          dKp[(i * K + j) * ldkv + h * hd + c] = ds[j] * qc;
        }
      dq[c] = acc;
    }
  }
}

extern "C" int tiger_train_attn_core_bwd(const float* dattn, int64_t ld_attn, const float* Q, int64_t ldq,
                                         const float* Kp, const float* Vp, int64_t ldkv, const float* P,
                                         const uint32_t* keep_bits, int64_t n_q, int k, int n_head, int head_dim,
                                         float p_drop, float* dQ, float* dKp, float* dVp, void* stream) {
  if (dattn == nullptr || Q == nullptr || Kp == nullptr || Vp == nullptr || P == nullptr || keep_bits == nullptr ||
      dQ == nullptr || dKp == nullptr || dVp == nullptr || n_q < 0 || k <= 0 || k > ATT_MAXK || n_head <= 0 ||
      head_dim <= 0)
    return TIGER_EINVAL;
  if (n_q == 0) return TIGER_OK;
  int64_t grid = (n_q * n_head + 7) / 8;
  if (grid > 148 * 8) grid = 148 * 8;
  auto launch = [&](auto kernel) {
    kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(dattn, ld_attn, Q, ldq, Kp, Vp, ldkv, P, keep_bits, n_q, k,
                                                          n_head, head_dim, p_drop, dQ, dKp, dVp);
  };
  if (k == 10) launch(train_attn_core_bwd_kernel<10>);
  else if (k == 5) launch(train_attn_core_bwd_kernel<5>);
  else if (k == 20) launch(train_attn_core_bwd_kernel<20>);
  else launch(train_attn_core_bwd_kernel<0>);
  return tiger_launch_status();
}

// Gradients of the builder's inputs: representation columns of dkv_in / dq_in (+ the merger's second input) are
// added onto the GRU row of the node they were read from (nodes without a pending message read the memory table,
// a buffer: no gradient); with d_key_rows the slots' node parts are stored there instead (zeros for padding slots),
// the gradient of the lower layer's output.  The time-code columns give the TimeEncode gradients
//   d/dw_c = -sin(dt w_c + b_c) dt g,  d/db_c = -sin(dt w_c + b_c) g      (time_encoding.py:16-27)
__global__ void __launch_bounds__(256)
train_attn_build_bwd_kernel(const float* __restrict__ dkv_in, const float* __restrict__ dq_in,
                            const float* __restrict__ dcat, int64_t ld_cat, int cat_off,
                            const int64_t* __restrict__ center, int64_t n_q, const float* __restrict__ ts, int64_t batch,
                            int64_t ts_group, const int64_t* __restrict__ nn, const float* __restrict__ nt, int K,
                            const int32_t* __restrict__ sel, int d, int de, const float* __restrict__ time_w,
                            const float* __restrict__ time_b, float* __restrict__ dh_new,
                            float* __restrict__ d_key_rows, float* __restrict__ g_w, float* __restrict__ g_b) {
  extern __shared__ float acc_smem[];          // [2][d]: block partial sums of g_w, g_b
  float* s_w = acc_smem;
  float* s_b = acc_smem + d;
  for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) acc_smem[c] = 0.f;
  __syncthreads();
  const int lane = lane_id();
  const int C = 2 * d + de;
  const int64_t n_kv = n_q * K, total = n_kv + n_q;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); r < total; r += n_warps) {
    if (r < n_kv) {
      const int64_t i = r / K;
      const int64_t nid = nn[r];
      const float* g = dkv_in + r * C;
      if (d_key_rows != nullptr) {
        for (int c = lane; c < d; c += 32) d_key_rows[r * d + c] = nid == 0 ? 0.f : g[c];
      }
      if (nid == 0) continue;               // padding slot: probability 0, no gradient (and no time gradient)
      if (d_key_rows == nullptr) {
        const int32_t row = sel[nid];
        if (row >= 0)
          for (int c = lane; c < d; c += 32) atomicAdd(dh_new + (int64_t)row * d + c, g[c]);
      }
      const float dt = ts[(ts_group == 1 ? i : i / ts_group) % batch] - nt[r];
      for (int c = lane; c < d; c += 32) {
        const float v = -sin_reduced(__fadd_rn(__fmul_rn(dt, time_w[c]), time_b[c])) * g[d + de + c];
        atomicAdd(s_w + c, v * dt);
        atomicAdd(s_b + c, v);
      }
    } else {
      const int64_t i = r - n_kv;
      const int64_t nid = center[i];
      const float* gq = dq_in + i * 2 * d;
      const float* gc = dcat + i * ld_cat + cat_off;
      const int32_t row = sel[nid];
      for (int c = lane; c < d; c += 32) {
        if (row >= 0) atomicAdd(dh_new + (int64_t)row * d + c, gq[c] + gc[c]);
        atomicAdd(s_b + c, -sin_reduced(time_b[c]) * gq[d + c]);     // query time code cos(0 * w + b)
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    if (s_w[c] != 0.f) atomicAdd(g_w + c, s_w[c]);
    if (s_b[c] != 0.f) atomicAdd(g_b + c, s_b[c]);
  }
}

extern "C" int tiger_train_attn_build_bwd_ex(const float* dkv_in, const float* dq_in, const float* dcat,
                                             int64_t ld_cat, int cat_off, const int64_t* center, int64_t n_q,
                                             const float* ts, int64_t batch, int64_t ts_group,
                                             const int64_t* neigh_nids, const float* neigh_ts, int k,
                                             const int32_t* sel, int d, int de, const float* time_w,
                                             const float* time_b, float* dh_new, float* d_key_rows, float* g_time_w,
                                             float* g_time_b, void* stream) {
  if (dkv_in == nullptr || dq_in == nullptr || dcat == nullptr || center == nullptr || ts == nullptr ||
      neigh_nids == nullptr || neigh_ts == nullptr || sel == nullptr || dh_new == nullptr || g_time_w == nullptr ||
      g_time_b == nullptr || n_q < 0 || batch <= 0 || ts_group <= 0 || k <= 0 || d <= 0 || de <= 0)
    return TIGER_EINVAL;
  if (n_q == 0) return TIGER_OK;
  int64_t grid = (n_q * (k + 1) + 7) / 8;
  if (grid > 148 * 2) grid = 148 * 2;
  train_attn_build_bwd_kernel<<<(unsigned)grid, 256, 2 * d * sizeof(float), as_stream(stream)>>>(
      dkv_in, dq_in, dcat, ld_cat, cat_off, center, n_q, ts, batch, ts_group, neigh_nids, neigh_ts, k, sel, d, de,
      time_w, time_b, dh_new, d_key_rows, g_time_w, g_time_b);
  return tiger_launch_status();
}

// ------------------------------------------------------------------------------------------
// shared element-wise pieces
// ------------------------------------------------------------------------------------------
__global__ void train_zero_rows_kernel(float* __restrict__ buf, int64_t ld, int cols, int64_t n_rows,
                                       const uint8_t* __restrict__ flag) {
  const int64_t total = n_rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols;
    if (flag[r]) buf[r * ld + (i % cols)] = 0.f;
  }
}

extern "C" int tiger_train_zero_rows(float* buf, int64_t ld, int cols, int64_t n_rows, const uint8_t* flag,
                                     void* stream) {
  if (buf == nullptr || flag == nullptr || cols <= 0 || ld < cols || n_rows < 0) return TIGER_EINVAL;
  if (n_rows == 0) return TIGER_OK;
  int64_t grid = (n_rows * cols + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  train_zero_rows_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(buf, ld, cols, n_rows, flag);
  return tiger_launch_status();
}

// dy[r, c] = y[r, c] > 0 ? scale * dy[r, c] : 0  (ReLU backward; with y the dropped-out activation and
// scale = 1 / (1 - p) also the backward of ReLU -> Dropout); rows bounded by *count * rows_per_count
__global__ void train_relu_bwd_kernel(float* __restrict__ dy, int64_t ld_dy, const float* __restrict__ y, int64_t ld_y,
                                      int cols, int64_t n_rows, const int32_t* __restrict__ count, int64_t per,
                                      float scale) {
  const int64_t total = bounded_rows(count, n_rows, per) * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols;
    const int c = (int)(i % cols);
    float* p = dy + r * ld_dy + c;
    *p = y[r * ld_y + c] > 0.f ? *p * scale : 0.f;
  }
}

extern "C" int tiger_train_relu_bwd(float* dy, int64_t ld_dy, const float* y, int64_t ld_y, int cols, int64_t n_rows,
                                    const int32_t* count, int64_t rows_per_count, float scale, void* stream) {
  if (dy == nullptr || y == nullptr || cols <= 0 || n_rows < 0) return TIGER_EINVAL;
  if (n_rows == 0) return TIGER_OK;
  int64_t grid = (n_rows * cols + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  train_relu_bwd_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(dy, ld_dy, y, ld_y, cols, n_rows, count,
                                                                      rows_per_count > 0 ? rows_per_count : 1, scale);
  return tiger_launch_status();
}

// out[c] += scale * sum_r X[r, c]  (bias gradients).  Block = 32 x 8 threads: a warp covers 32 consecutive columns,
// the 8 warps stride over a slab of rows; partial sums meet in shared memory, one atomic add per column and block.
#define COLSUM_ROWS 256
__global__ void __launch_bounds__(256)
train_colsum_kernel(const float* __restrict__ X, int64_t ld, int64_t n_rows, const int32_t* __restrict__ count,
                    int64_t per, int cols, float scale, float* __restrict__ out) {
  __shared__ float part[8][33];
  const int64_t rows = bounded_rows(count, n_rows, per);
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int w = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)blockIdx.y * COLSUM_ROWS;
  if (r0 >= rows) return;
  const int64_t r1 = r0 + COLSUM_ROWS < rows ? r0 + COLSUM_ROWS : rows;
  float acc = 0.f;
  if (c < cols)
    for (int64_t r = r0 + w; r < r1; r += 8) acc += X[r * ld + c];
  part[w][threadIdx.x & 31] = acc;
  __syncthreads();
  if (w == 0 && c < cols) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += part[k][threadIdx.x];
    if (s != 0.f) atomicAdd(out + c, s * scale);
  }
}

extern "C" int tiger_train_colsum(const float* X, int64_t ld, int64_t n_rows, const int32_t* count,
                                  int64_t rows_per_count, int cols, float scale, float* out, void* stream) {
  if (X == nullptr || out == nullptr || cols <= 0 || ld < cols || n_rows < 0) return TIGER_EINVAL;
  if (n_rows == 0) return TIGER_OK;
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((n_rows + COLSUM_ROWS - 1) / COLSUM_ROWS));
  train_colsum_kernel<<<grid, 256, 0, as_stream(stream)>>>(X, ld, n_rows, count, rows_per_count > 0 ? rows_per_count : 1,
                                                          cols, scale, out);
  return tiger_launch_status();
}

// table[ids[r]] += scale * src[r]   (nn.Embedding weight gradient: static restarter, anonymised-id embedding)
__global__ void train_scatter_add_rows_kernel(float* __restrict__ table, const int64_t* __restrict__ ids, int64_t n,
                                              const int32_t* __restrict__ count, int64_t per,
                                              const float* __restrict__ src, int64_t ld_src, int width, float scale) {
  const int64_t total = bounded_rows(count, n, per) * width;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / width;
    const int c = (int)(i % width);
    const float v = src[r * ld_src + c] * scale;
    if (v != 0.f) atomicAdd(table + ids[r] * width + c, v);
  }
}

extern "C" int tiger_train_scatter_add_rows(float* table, const int64_t* ids, int64_t n, const int32_t* count,
                                            int64_t rows_per_count, const float* src, int64_t ld_src, int width,
                                            float scale, void* stream) {
  if (table == nullptr || ids == nullptr || src == nullptr || width <= 0 || ld_src < width || n < 0) return TIGER_EINVAL;
  if (n == 0) return TIGER_OK;
  int64_t grid = (n * width + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  train_scatter_add_rows_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(
      table, ids, n, count, rows_per_count > 0 ? rows_per_count : 1, src, ld_src, width, scale);
  return tiger_launch_status();
}

// ------------------------------------------------------------------------------------------
// link scorer (tiger.py:259-288): hit embedding, MergeLayer with dropout, BCE-with-logits
// ------------------------------------------------------------------------------------------
// pair[i]     = [x_i + he(src_hit_i)     | y_i  + he(dst_hit_i)]        i <  B  (positive pairs)
// pair[B + i] = [x_i + he(neg_src_hit_i) | ny_i + he(neg_dst_hit_i)]           (negative pairs)
// hit codes ('bin': max over the K slots), either from the four [B, K] 0/1 tables of HitData in the order
// (src, dst, neg_src, neg_dst), or straight from the neighbor table of the batch [3B, K] (rows: N(src) | N(dst) |
// N(neg)) with check_in_window's rule (data_loader.py:61-75): src_hit = src in N(dst), dst_hit = dst in N(src),
// neg_src_hit = src in N(neg), neg_dst_hit = neg in N(src)
__global__ void __launch_bounds__(256)
train_score_build_kernel(const float* __restrict__ z, const float* __restrict__ hits, const int64_t* __restrict__ nn,
                         const int64_t* __restrict__ batch_nids, int K, const float* __restrict__ hit_emb, int64_t B,
                         int d, float* __restrict__ pair, uint8_t* __restrict__ codes) {
  const int lane = lane_id();
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const bool use_hits = hits != nullptr || nn != nullptr;
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); r < 2 * B; r += n_warps) {
    const int64_t i = r % B;
    const bool negp = r >= B;
    int code_a = 0, code_b = 0;
    if (hits != nullptr) {
      const float* ha = hits + ((negp ? 2 : 0) * B + i) * K;
      const float* hb = hits + ((negp ? 3 : 1) * B + i) * K;
      float ma = 0.f, mb = 0.f;
      for (int k = lane; k < K; k += 32) {
        ma = fmaxf(ma, ha[k]);
        mb = fmaxf(mb, hb[k]);
      }
      code_a = warp_max(ma) > 0.5f ? 1 : 0;
      code_b = warp_max(mb) > 0.5f ? 1 : 0;
    } else if (nn != nullptr) {
      const int64_t src = batch_nids[i];
      const int64_t other = batch_nids[(negp ? 2 : 1) * B + i];      // dst or neg
      const int64_t* n_other = nn + ((negp ? 2 : 1) * B + i) * K;     // N(dst) or N(neg)
      const int64_t* n_src = nn + i * K;
      bool a = false, b = false;
      for (int k = lane; k < K; k += 32) {
        a |= n_other[k] == src;
        b |= n_src[k] == other;
      }
      code_a = __any_sync(TIGER_FULL_MASK, a) ? 1 : 0;
      code_b = __any_sync(TIGER_FULL_MASK, b) ? 1 : 0;
    }
    if (use_hits && lane == 0) {
      codes[(negp ? 2 : 0) * B + i] = (uint8_t)code_a;
      codes[(negp ? 3 : 1) * B + i] = (uint8_t)code_b;
    }
    const float* xa = z + i * d;
    const float* xb = z + ((negp ? 2 : 1) * B + i) * d;
    float* row = pair + r * 2 * d;
    for (int c = lane; c < d; c += 32) {
      row[c] = xa[c] + (use_hits ? hit_emb[code_a * d + c] : 0.f);
      row[d + c] = xb[c] + (use_hits ? hit_emb[code_b * d + c] : 0.f);
    }
  }
}

extern "C" int tiger_train_score_build(const float* z, const float* hits, const int64_t* neigh_nids,
                                       const int64_t* batch_nids, int k, const float* hit_emb, int64_t batch, int d,
                                       float* pair, uint8_t* codes, void* stream) {
  const bool use_hits = hits != nullptr || neigh_nids != nullptr;
  if (z == nullptr || pair == nullptr || batch <= 0 || d <= 0 ||
      (use_hits && (hit_emb == nullptr || codes == nullptr || k <= 0)) || (neigh_nids != nullptr && batch_nids == nullptr))
    return TIGER_EINVAL;
  int64_t grid = (2 * batch + 7) / 8;
  train_score_build_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(z, hits, neigh_nids, batch_nids, k, hit_emb,
                                                                         batch, d, pair, codes);
  return tiger_launch_status();
}

// hid [2B, d] = relu(fc1(pair)) is overwritten with its dropped-out version; score = hid' . w + b;
// loss = mean BCE-with-logits (labels 1 for rows < B, else 0); dscore = (sigmoid(score) - label) / 2B.
// Two launches: warp per row over the whole grid, then one CTA sums the 2B per-row losses in a fixed order (as a single
// CTA walking all rows the kernel was one latency chain of 13 rows per warp: 27 us, profiles/r02_launches.md).
__global__ void __launch_bounds__(256)
train_score_head_kernel(float* __restrict__ hid, const float* __restrict__ w, const float* __restrict__ b, int64_t B,
                        int d, float p_drop, uint32_t seed, float* __restrict__ scores, float* __restrict__ dscore) {
  seed = tiger_step_seed(seed);
  const int lane = lane_id();
  const float inv_keep = p_drop > 0.f ? 1.0f / (1.0f - p_drop) : 1.0f;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); r < 2 * B; r += n_warps) {
    float* row = hid + r * d;
    float acc = 0.f;
    for (int c = lane; c < d; c += 32) {
      float v = row[c];
      v = dropout_keep(seed, 2u, (uint32_t)(r * d + c), p_drop) ? v * inv_keep : 0.f;
      row[c] = v;
      acc = fmaf(v, w[c], acc);
    }
    acc = warp_sum(acc) + b[0];
    if (lane == 0) {
      const float y = r < B ? 1.f : 0.f;
      scores[r] = acc;
      dscore[r] = (sigmoidf_acc(acc) - y) / (float)(2 * B);
    }
  }
}

__global__ void __launch_bounds__(1024)
train_bce_mean_kernel(const float* __restrict__ scores, int64_t B, float* __restrict__ loss) {
  __shared__ float red[32];
  const int lane = lane_id(), warp = warp_id_in_block(), n_warps = blockDim.x >> 5;
  float local = 0.f;
  for (int64_t r = threadIdx.x; r < 2 * B; r += blockDim.x) {
    const float acc = scores[r], y = r < B ? 1.f : 0.f;
    local += fmaxf(acc, 0.f) - acc * y + log1pf(expf(-fabsf(acc)));
  }
  local = warp_sum(local);
  if (lane == 0) red[warp] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int k = 0; k < n_warps; ++k) t += red[k];      // fixed order: deterministic
    loss[0] = t / (float)(2 * B);
  }
}

extern "C" int tiger_train_score_head(float* hid, const float* fc2_w, const float* fc2_b, int64_t batch, int d,
                                      float p_drop, int seed, float* scores, float* loss, float* dscore,
                                      void* stream) {
  if (hid == nullptr || fc2_w == nullptr || fc2_b == nullptr || scores == nullptr || loss == nullptr ||
      dscore == nullptr || batch <= 0 || d <= 0 || p_drop < 0.f || p_drop >= 1.f)
    return TIGER_EINVAL;
  int64_t grid = (2 * batch + 7) / 8;
  if (grid > 148 * 4) grid = 148 * 4;
  train_score_head_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(hid, fc2_w, fc2_b, batch, d, p_drop,
                                                                        (uint32_t)seed, scores, dscore);
  train_bce_mean_kernel<<<1, 1024, 0, as_stream(stream)>>>(scores, batch, loss);
  return tiger_launch_status();
}

// dhid[r, c] = g dscore_r w_c / (1 - p) where hid'[r, c] > 0 (kept and past the ReLU), else 0;
// g_w[c] += g sum_r dscore_r hid'[r, c];  g_b += g sum_r dscore_r.   CTA (x, y) = 32 columns x one slice of the rows.
#define SHB_ROWS 64
__global__ void __launch_bounds__(256)
train_score_head_bwd_kernel(const float* __restrict__ dscore, float g, const float* __restrict__ hid,
                            const float* __restrict__ w, int64_t B, int d, float p_drop, float* __restrict__ dhid,
                            float* __restrict__ g_w, float* __restrict__ g_b) {
  __shared__ float part[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int wrp = threadIdx.x >> 5;
  const float inv_keep = p_drop > 0.f ? 1.0f / (1.0f - p_drop) : 1.0f;
  const int64_t r0 = (int64_t)blockIdx.y * SHB_ROWS;
  const int64_t r1 = (r0 + SHB_ROWS < 2 * B) ? r0 + SHB_ROWS : 2 * B;
  float acc = 0.f, accb = 0.f;
  for (int64_t r = r0 + wrp; r < r1; r += 8) {
    const float ds = g * dscore[r];
    if (c < d) {
      const float h = hid[r * d + c];
      dhid[r * d + c] = h > 0.f ? ds * w[c] * inv_keep : 0.f;
      acc = fmaf(ds, h, acc);
    }
    accb += ds;
  }
  part[wrp][threadIdx.x & 31] = acc;
  __syncthreads();
  if (wrp == 0 && c < d) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += part[k][threadIdx.x];
    atomicAdd(g_w + c, t);
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    part[wrp][threadIdx.x & 31] = (threadIdx.x & 31) == 0 ? accb : 0.f;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int k = 0; k < 8; ++k) t += part[k][0];
      atomicAdd(g_b, t);
    }
  }
}

extern "C" int tiger_train_score_head_bwd(const float* dscore, float g, const float* hid, const float* fc2_w,
                                          int64_t batch, int d, float p_drop, float* dhid, float* g_fc2_w,
                                          float* g_fc2_b, void* stream) {
  if (dscore == nullptr || hid == nullptr || fc2_w == nullptr || dhid == nullptr || g_fc2_w == nullptr ||
      g_fc2_b == nullptr || batch <= 0 || d <= 0)
    return TIGER_EINVAL;
  const dim3 grid((unsigned)((d + 31) / 32), (unsigned)((2 * batch + SHB_ROWS - 1) / SHB_ROWS));
  train_score_head_bwd_kernel<<<grid, 256, 0, as_stream(stream)>>>(dscore, g, hid, fc2_w, batch, d, p_drop, dhid, g_fc2_w,
                                                                  g_fc2_b);
  return tiger_launch_status();
}

// dz[i] = dpair[i, :d] + dpair[B+i, :d]; dz[B+i] = dpair[i, d:]; dz[2B+i] = dpair[B+i, d:];
// g_hit[code] += the same rows (nn.Embedding(2, d) gradient)
__global__ void __launch_bounds__(256)
train_score_build_bwd_kernel(const float* __restrict__ dpair, const uint8_t* __restrict__ codes, int64_t B, int d,
                             float* __restrict__ dz, float* __restrict__ g_hit) {
  extern __shared__ float s_hit[];       // [2][d]
  for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) s_hit[c] = 0.f;
  __syncthreads();
  const int lane = lane_id();
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); i < B; i += n_warps) {
    const float* gp = dpair + i * 2 * d;
    const float* gn = dpair + (B + i) * 2 * d;
    for (int c = lane; c < d; c += 32) {
      const float a = gp[c], b = gp[d + c], e = gn[c], f = gn[d + c];
      dz[i * d + c] = a + e;
      dz[(B + i) * d + c] = b;
      dz[(2 * B + i) * d + c] = f;
      if (codes != nullptr) {
        atomicAdd(s_hit + codes[i] * d + c, a);
        atomicAdd(s_hit + codes[B + i] * d + c, b);
        atomicAdd(s_hit + codes[2 * B + i] * d + c, e);
        atomicAdd(s_hit + codes[3 * B + i] * d + c, f);
      }
    }
  }
  __syncthreads();
  if (codes != nullptr)
    for (int c = threadIdx.x; c < 2 * d; c += blockDim.x)
      if (s_hit[c] != 0.f) atomicAdd(g_hit + c, s_hit[c]);
}

extern "C" int tiger_train_score_build_bwd(const float* dpair, const uint8_t* codes, int64_t batch, int d, float* dz,
                                           float* g_hit_emb, void* stream) {
  if (dpair == nullptr || dz == nullptr || batch <= 0 || d <= 0 || (codes != nullptr && g_hit_emb == nullptr))
    return TIGER_EINVAL;
  int64_t grid = (batch + 7) / 8;
  if (grid > 148) grid = 148;
  train_score_build_bwd_kernel<<<(unsigned)grid, 256, 2 * d * sizeof(float), as_stream(stream)>>>(dpair, codes, batch, d,
                                                                                                 dz, g_hit_emb);
  return tiger_launch_status();
}

// ------------------------------------------------------------------------------------------
// mutual loss (tiger.py:574-592): MSE between [pred_left; pred_right] and [h_prev_left[index]; h_prev_right[index]]
// over the rows whose target is not all-zero.  dpred = 2 (pred - t) / (n_valid d), 0 for invalid rows (the caller
// scales it with the upstream gradient).  Two grid-wide launches (P <= 2048 rows): warp per row -> validity, the
// row's squared error into `work` (-1 = invalid row) and the unscaled gradient; then every CTA derives n_valid from
// `work` (fixed order), scales its share of the gradient and CTA 0 writes the loss.  (One CTA walking all rows twice
// was 49 us, profiles/r02_launches.md.)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
train_mse_rows_kernel(const float* __restrict__ pred_l, const float* __restrict__ pred_r, const float* __restrict__ hpl,
                      const float* __restrict__ hpr, const int64_t* __restrict__ index, const int32_t* __restrict__ count,
                      int64_t P, int d, float* __restrict__ dpred_l, float* __restrict__ dpred_r, float* __restrict__ work) {
  const int lane = lane_id();
  const int64_t rows = bounded_rows(count, P);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block(); r < 2 * rows; r += n_warps) {
    const bool left = r < rows;
    const int64_t k = left ? r : r - rows;
    const float* t = (left ? hpl : hpr) + index[k] * d;
    const float* p = (left ? pred_l : pred_r) + k * d;
    float* gbase = left ? dpred_l : dpred_r;
    bool nz = false;
    float sse = 0.f;
    for (int c = lane; c < d; c += 32) {
      const float tv = t[c];
      const float e = p[c] - tv;
      nz |= tv != 0.f;
      sse = fmaf(e, e, sse);
      if (gbase != nullptr) gbase[k * d + c] = 2.0f * e;
    }
    nz = __any_sync(TIGER_FULL_MASK, nz);
    sse = warp_sum(sse);
    if (lane == 0) work[r] = nz ? sse : -1.0f;
  }
}

__global__ void __launch_bounds__(256)
train_mse_finish_kernel(const int32_t* __restrict__ count, int64_t P, int d, const float* __restrict__ work,
                        float* __restrict__ loss, float* __restrict__ dpred_l, float* __restrict__ dpred_r,
                        float* __restrict__ n_valid_out) {
  __shared__ float red[8];
  __shared__ int red_n[8];
  const int lane = lane_id(), warp = warp_id_in_block();
  const int64_t rows = bounded_rows(count, P);
  float local = 0.f;
  int nv = 0;
  for (int64_t r = threadIdx.x; r < 2 * rows; r += blockDim.x) {      // same order in every CTA: same n_valid / loss
    const float v = work[r];
    if (v >= 0.f) { local += v; ++nv; }
  }
  local = warp_sum(local);
  nv = __reduce_add_sync(TIGER_FULL_MASK, nv);
  if (lane == 0) { red[warp] = local; red_n[warp] = nv; }
  __syncthreads();
  float total = 0.f;
  int n_valid = 0;
  for (int k = 0; k < 8; ++k) { total += red[k]; n_valid += red_n[k]; }
  const float inv = n_valid > 0 ? 1.0f / ((float)n_valid * (float)d) : 0.f;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    loss[0] = total * inv;
    if (n_valid_out != nullptr) n_valid_out[0] = (float)n_valid;
  }
  if (dpred_l == nullptr) return;
  const int64_t total_e = 2 * rows * d;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total_e; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / d;
    const bool left = r < rows;
    float* gp = (left ? dpred_l : dpred_r) + (e - (left ? 0 : rows * d));
    *gp = work[r] >= 0.f ? *gp * inv : 0.f;
  }
}

extern "C" int tiger_train_mse(const float* pred_l, const float* pred_r, const float* hprev_left,
                               const float* hprev_right, const int64_t* index, const int32_t* count, int64_t n, int d,
                               float* loss, float* dpred_l, float* dpred_r, float* n_valid_out, float* work,
                               void* stream) {
  if (pred_l == nullptr || pred_r == nullptr || hprev_left == nullptr || hprev_right == nullptr || index == nullptr ||
      loss == nullptr || work == nullptr || n < 0 || n > 2048 || d <= 0 || (dpred_l == nullptr) != (dpred_r == nullptr))
    return TIGER_EINVAL;
  int64_t grid = (2 * n + 7) / 8;
  if (grid < 1) grid = 1;
  if (grid > 148 * 2) grid = 148 * 2;
  train_mse_rows_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(pred_l, pred_r, hprev_left, hprev_right, index,
                                                                      count, n, d, dpred_l, dpred_r, work);
  train_mse_finish_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(count, n, d, work, loss, dpred_l, dpred_r,
                                                                        n_valid_out);
  return tiger_launch_status();
}

// ------------------------------------------------------------------------------------------
// Adam (torch.optim.Adam defaults of the reference: train_self_supervised.py:116; no weight decay, no amsgrad) over a
// flat parameter buffer cut into the model's tensors.  torch keeps one step counter PER TENSOR and skips a tensor
// whose gradient is None in a step - the GRU cell when no involved node holds a pending message (tiger.py:215), the
// restarter when contrast_only or no target row is valid (tiger.py:571,586-592) - so every tensor carries a group:
//   0 always stepped | 1 stepped iff gates[0] > 0 | 2 stepped iff gates[1] > 0 | 3 never (gates[2] stays 0)
// with the gates (#GRU rows, #valid target rows) read from device memory - they live at the tail of the flat gradient
// buffer and so take part in the DDP all-reduce: a tensor used on any rank is stepped on every rank.
// gscale folds the 1/world_size of the all-reduce; the gradient (and the gates) are zeroed for the next step
// (optimizer.zero_grad()).
// ------------------------------------------------------------------------------------------
__global__ void train_adam_prepare_kernel(const int32_t* __restrict__ seg_group, int32_t* __restrict__ seg_step,
                                          float* __restrict__ seg_bc, int n_seg, const float* __restrict__ gates,
                                          float b1, float b2) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_seg) return;
  const int grp = seg_group[t];
  const bool active = grp == 0 || (gates != nullptr && gates[grp - 1] > 0.f);
  int step = seg_step[t];
  if (active) seg_step[t] = ++step;
  seg_bc[2 * t] = active ? 1.0f - powf(b1, (float)step) : 0.f;          // 0 marks "skip this tensor"
  seg_bc[2 * t + 1] = active ? sqrtf(1.0f - powf(b2, (float)step)) : 0.f;
}

__global__ void train_adam_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                                  float* __restrict__ v, const int64_t* __restrict__ seg_start,
                                  const float* __restrict__ seg_bc, float lr, float b1, float b2, float eps,
                                  float gscale, int zero_grad) {
  const int t = blockIdx.y;
  const int64_t lo = seg_start[t], hi = seg_start[t + 1];
  const float bc1 = seg_bc[2 * t], bc2_sqrt = seg_bc[2 * t + 1];
  for (int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (int64_t)gridDim.x * blockDim.x) {
    if (bc1 > 0.f) {
      const float gi = g[i] * gscale;
      const float mi = m[i] + (gi - m[i]) * (1.0f - b1);          // exp_avg.lerp_(grad, 1 - beta1)
      const float vi = v[i] * b2 + gi * gi * (1.0f - b2);         // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
      m[i] = mi;
      v[i] = vi;
      const float denom = sqrtf(vi) / bc2_sqrt + eps;
      p[i] = p[i] - (lr / bc1) * (mi / denom);
    }
    if (zero_grad) g[i] = 0.f;
  }
}

__global__ void train_zero_gates_kernel(float* gates, int n) {
  if (threadIdx.x < n) gates[threadIdx.x] = 0.f;
}

extern "C" int tiger_train_adam(float* params, float* grads, float* exp_avg, float* exp_avg_sq, const int64_t* seg_start,
                                const int32_t* seg_group, int32_t* seg_step, float* seg_bc, int n_seg, float* gates,
                                int64_t max_seg, float lr, float beta1, float beta2, float eps, float grad_scale,
                                int zero_grad, void* stream) {
  if (params == nullptr || grads == nullptr || exp_avg == nullptr || exp_avg_sq == nullptr || seg_start == nullptr ||
      seg_group == nullptr || seg_step == nullptr || seg_bc == nullptr || n_seg <= 0 || max_seg < 0)
    return TIGER_EINVAL;
  cudaStream_t st = as_stream(stream);
  train_adam_prepare_kernel<<<(unsigned)((n_seg + 127) / 128), 128, 0, st>>>(seg_group, seg_step, seg_bc, n_seg, gates,
                                                                            beta1, beta2);
  int64_t gx = (max_seg + 255) / 256;
  if (gx < 1) gx = 1;
  if (gx > 512) gx = 512;
  dim3 grid((unsigned)gx, (unsigned)n_seg);
  train_adam_kernel<<<grid, 256, 0, st>>>(params, grads, exp_avg, exp_avg_sq, seg_start, seg_bc, lr, beta1, beta2, eps,
                                          grad_scale, zero_grad);
  if (zero_grad && gates != nullptr) train_zero_gates_kernel<<<1, 32, 0, st>>>(gates, 2);
  return tiger_launch_status();
}

// Registers (or clears, with NULL) the device-side step counter the dropout kernels add to their seeds: see common.cuh.
extern "C" int tiger_train_seed_step(const int32_t* step) {
  int rc = tiger_seed_step_set_here(step);
  if (rc == TIGER_OK) rc = tiger_seed_step_set_train_seq(step);
  if (rc == TIGER_OK) rc = tiger_seed_step_set_restart_seq(step);
  return rc;
}
