// K3  temporal graph attention (one layer per launch sequence; n_layers = 2 chains two of them), eval mode.
// Reference: GraphEmbedding.compute_embedding_with_computation_graph
// (tiger/model/temporal_agg_modules.py:29-83) + TemporalAttention.forward (:210-235) + torch
// F.multi_head_attention_forward (need_weights branch) + MergeLayer (basic_modules.py:16-19).
//
// Math per query (h = head, hd = E / n_head, scale = sqrt(1/hd), E = 2d, C = 2d + de):
//   q    = scale * (Wq [c | qt] + bq)                           c = repr(center) + nf(center), qt = cos(b)
//   s_hj = q_h . (Wk_h kv_j + bk_h)        kv_j = [repr(n_j)+nf | ef(e_j) | cos((t - t_j) w + b)]
//   p_h  = softmax_j(s_hj) over live slots
//   o_h  = Wv_h (sum_j p_hj kv_j) + bv_h                         (sum_j p_hj = 1)
//   out  = Wo [o_1 | o_2 ..] + bo ; 0 if every slot is padding
//   z    = W2 relu(W1 [out | c] + b1) + b2
// All of it is linear in the per-query vectors except the softmax and the ReLU, so the weights are
// folded once per parameter update (tiger_attn_fold, exact by linearity, accumulated in double):
//   Wqk_h = scale [Wk_h | bk_h]^T Wq_h   ([C+1, E])   bqk_h = scale [Wk_h | bk_h]^T bq_h
//       =>  [s-weights qk_h | qb_h] = Wqk_h [c | qt] + bqk_h ,  s_hj = qk_h . kv_j + qb_h
//   W2f   = [ W1a Wo_1 Wv_1 | W1a Wo_2 Wv_2 | W1b | W1a (Wo bv + bo) ]   (W1 = [W1a | W1b])
//       =>  hidden = relu(W2f [kvbar_1 | kvbar_2 | c | live] + b1) ,  live = 0 when every slot is padding
// which needs ~12x fewer flops than projecting all K neighbors of every query and three GEMM
// launches instead of six.
//
// Launch sequence (all queries of the batch at once; workspace provided by the caller):
//   attn_prepare          gather center rows: XQ = [c | qt], KVC[:, c] = c, KVC[:, live]
//   sgemm_nt (tcgen05)    QKF = XQ Wqk^T + bqk                           [n, H (C+1)]
//   attn_score_pool       one CTA per query: gather the K key rows once into shared memory
//                         (memory / GRU-output rows, edge features, time code), scores, masked
//                         softmax, pooled keys -> KVC[:, kvbar]
//   sgemm_nt (tcgen05)    HID = relu(KVC W2f^T + b1)                    [n, d]
//   sgemm_nt (tcgen05)    z = HID W2^T + b2                             [n, d]
#include "common.cuh"
#ifdef TIGER_TRACE
#include <cstdio>
#endif

#define ATT_MAXH 8
#define ATT_MAXK 64                   // the masked softmax holds two slots per lane of one warp
#define ATT_MAX_POOL_SMEM (200 * 1024)  // dynamic shared memory of attn_score_pool: its K key rows stay staged
#ifndef ATT_THREADS
#define ATT_THREADS 256
#endif
#define ATT_BN_QK 64   // column tile of the Wqk pack: H (C+1) ~ 1000 columns -> ~17 tiles per 128 queries
#define ATT_BN_D 64    // column tile of the W2f pack: d columns -> 3 tiles per 128 queries
#ifndef ATT_BN_F3
#define ATT_BN_F3 32   // column tile of the last product (fc2, with the scorer fold 3d columns)
#endif
#define ATT_KPARTS 8   // split-K of the W2f product (K = H C + d + 1 ~ 1200, only ~15 output tiles): the parts of a
                       // tile run as one thread-block cluster and sum their partial tiles through DSMEM

static inline int ru4(int x) { return (x + 3) & ~3; }

struct AttDims {
  int d, de, K, H, E, C, hd;
  int ld_xq, Cq, ld_qkf, Cp, ld_kvc, off_c, off_live, ld_hid;
};

static AttDims att_dims(int d, int de, int k, int n_head) {
  AttDims a;
  a.d = d; a.de = de; a.K = k; a.H = n_head;
  a.E = 2 * d; a.C = 2 * d + de; a.hd = a.E / n_head;
  a.ld_xq = ru4(a.E);
  a.Cq = ru4(a.C + 1); a.ld_qkf = n_head * a.Cq;
  a.Cp = ru4(a.C);
  a.off_c = n_head * a.Cp;               // KVC row: [kvbar_0 .. kvbar_{H-1} | c | live | pad]
  a.off_live = a.off_c + d;
  a.ld_kvc = ru4(a.off_live + 1);
  a.ld_hid = ru4(d);
  return a;
}

struct AttWork {
  float *xq, *qkf, *kvc, *hid;
  int64_t total_floats;
};

static AttWork att_work(const AttDims& a, int64_t n, float* base) {
  AttWork w;
  int64_t off = 0;
  auto take = [&](int64_t cnt) { float* p = base ? base + off : nullptr; off += (cnt + 3) & ~(int64_t)3; return p; };
  w.xq = take(n * a.ld_xq);
  w.qkf = take(n * a.ld_qkf);
  w.kvc = take(n * a.ld_kvc);
  w.hid = take((int64_t)n * a.ld_hid);                // hidden layer of the merger
  w.total_floats = off;
  return w;
}

// dynamic shared memory of attn_score_pool: kv [K][Cp] | scores [H][K] (rounded to 4) | score weights [H][Cq]
static size_t att_pool_smem(const AttDims& a) {
  return ((size_t)a.K * a.Cp + (size_t)((a.H * a.K + 3) & ~3) + (size_t)a.H * a.Cq) * sizeof(float);
}

// the dimensions the kernels take: K, heads and the score-pool footprint within their limits
static bool att_dims_ok(int k, int d, int de, int n_head) {
  if (k <= 0 || d <= 0 || de <= 0 || n_head <= 0 || k > ATT_MAXK || n_head > ATT_MAXH) return false;
  return att_pool_smem(att_dims(d, de, k, n_head)) <= ATT_MAX_POOL_SMEM;
}

// -1 for dimensions the attention refuses (also past ATT_MAXK, ATT_MAXH and ATT_MAX_POOL_SMEM): callers test a model
// against the kernel's limits with it
extern "C" int64_t tiger_temporal_attention_work_bytes(int64_t n_query, int k, int d, int de, int n_head) {
  if (n_query < 0 || !att_dims_ok(k, d, de, n_head)) return -1;
  const AttDims a = att_dims(d, de, k, n_head);
  return att_work(a, n_query, nullptr).total_floats * (int64_t)sizeof(float);
}

// ------------------------------------------------------------------------------------------
// parameter folding (once per parameter update)
// ------------------------------------------------------------------------------------------
struct AttFold {
  float *wqk, *bqk, *w2f, *wov, *bov;   // wqk [H*Cq][E], bqk [H*Cq], w2f [d][ld_kvc] ; temporaries wov [E][H*Cp], bov [E]
  float *pk_wqk, *pk_w2f, *pk_fc2;      // tf32 head / tail packs of wqk, w2f and merger.fc2 for the tensor-core GEMM
  // graph path: the query's time code is the constant cos(time_b) (dt = 0), so its half of Wqk folds into the
  // bias: bqk_c = bqk + Wqk[:, d:] tq ; pk_wqk_c = pack of Wqk[:, :d] (K = d instead of 2d)
  float *tq, *bqk_c, *pk_wqk_c;
  int t_qk, t_d;                        // column tiles of the packs
  int64_t total_floats;
};

static AttFold att_fold(const AttDims& a, float* base) {
  AttFold f;
  int64_t off = 0;
  auto take = [&](int64_t cnt) { float* p = base ? base + off : nullptr; off += (cnt + 3) & ~(int64_t)3; return p; };
  f.wqk = take((int64_t)a.H * a.Cq * a.E);
  f.bqk = take((int64_t)a.H * a.Cq);
  f.w2f = take((int64_t)a.d * a.ld_kvc);
  f.wov = take((int64_t)a.E * a.H * a.Cp);
  f.bov = take(a.E);
  f.t_qk = (a.H * a.Cq + ATT_BN_QK - 1) / ATT_BN_QK;
  f.t_d = (a.d + ATT_BN_D - 1) / ATT_BN_D;
  f.pk_wqk = take(tiger_gemm_pack_bytes(f.t_qk, a.E, ATT_BN_QK) / 4);
  f.pk_w2f = take(tiger_gemm_pack_bytes(f.t_d, a.off_live + 1, ATT_BN_D) / 4);
  f.pk_fc2 = take(tiger_gemm_pack_bytes((a.d + ATT_BN_F3 - 1) / ATT_BN_F3, a.d, ATT_BN_F3) / 4);
  f.tq = take(a.E - a.d);
  f.bqk_c = take((int64_t)a.H * a.Cq);
  f.pk_wqk_c = take(tiger_gemm_pack_bytes(f.t_qk, a.d, ATT_BN_QK) / 4);
  f.total_floats = off;
  return f;
}

__global__ void attn_fold_time0_kernel(const float* __restrict__ w, const float* __restrict__ b, int n,
                                       float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < n) out[c] = time_enc(0.f, w[c], b[c]);
}

extern "C" int64_t tiger_attn_fold_bytes(int d, int de, int n_head) {
  if (d <= 0 || de <= 0 || n_head <= 0 || (2 * d) % n_head != 0) return -1;
  const AttDims a = att_dims(d, de, 1, n_head);
  return att_fold(a, nullptr).total_floats * (int64_t)sizeof(float);
}

// C[m * scm + n] = alpha * sum_k A[m * sam + k * sak] * B[k * sbk + n * sbn] (+ add[m]) ; double accumulation
__global__ void attn_fold_mm_kernel(const float* __restrict__ A, int64_t sam, int64_t sak, const float* __restrict__ B,
                                    int64_t sbk, int64_t sbn, float* C, int64_t scm, int M, int N, int K,
                                    float alpha, const float* add) {   // add may alias C (in-place accumulate)
  const int n = blockIdx.x * blockDim.x + threadIdx.x, m = blockIdx.y;
  if (n >= N || m >= M) return;
  double acc = 0.0;
  for (int k = 0; k < K; ++k) acc += (double)A[m * sam + k * sak] * (double)B[k * sbk + n * sbn];
  acc *= (double)alpha;
  if (add != nullptr) acc += (double)add[m];
  C[m * scm + n] = (float)acc;
}

static void fold_mm(cudaStream_t st, const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbk, int64_t sbn,
                    float* C, int64_t scm, int M, int N, int K, float alpha, const float* add) {
  dim3 grid((unsigned)((N + 127) / 128), (unsigned)M);
  attn_fold_mm_kernel<<<grid, 128, 0, st>>>(A, sam, sak, B, sbk, sbn, C, scm, M, N, K, alpha, add);
}

extern "C" int tiger_attn_fold(const tiger_attn_params* p, int d, int de, int n_head, void* stream) {
  if (p == nullptr || p->folded == nullptr || d <= 0 || de <= 0 || n_head <= 0 || (2 * d) % n_head != 0)
    return TIGER_EINVAL;
  const AttDims a = att_dims(d, de, 1, n_head);
  const AttFold f = att_fold(a, p->folded);
  cudaStream_t st = as_stream(stream);
  const int E = a.E, C = a.C, hd = a.hd, H = a.H;
  const float scale = sqrtf(1.0f / (float)hd);
  const float* bq = p->in_bias;
  const float* bk = p->in_bias + E;
  const float* bv = p->in_bias + 2 * E;
  if (cudaMemsetAsync(p->folded, 0, (size_t)f.total_floats * sizeof(float), st) != cudaSuccess) return TIGER_ECUDA;
  for (int h = 0; h < H; ++h) {
    const float* wk_h = p->wk + (int64_t)h * hd * C;   // [hd][C]
    const float* wq_h = p->wq + (int64_t)h * hd * E;   // [hd][E]
    float* wqk_h = f.wqk + (int64_t)h * a.Cq * E;
    float* bqk_h = f.bqk + (int64_t)h * a.Cq;
    // rows j < C: scale * Wk_h^T Wq_h ; row C: scale * bk_h^T Wq_h
    fold_mm(st, wk_h, 1, C, wq_h, E, 1, wqk_h, E, C, E, hd, scale, nullptr);
    fold_mm(st, bk + h * hd, 0, 1, wq_h, E, 1, wqk_h + (int64_t)C * E, E, 1, E, hd, scale, nullptr);
    fold_mm(st, wk_h, 1, C, bq + h * hd, 1, 0, bqk_h, 1, C, 1, hd, scale, nullptr);
    fold_mm(st, bk + h * hd, 0, 1, bq + h * hd, 1, 0, bqk_h + C, 1, 1, 1, hd, scale, nullptr);
    // Wov_h = Wo[:, h*hd:(h+1)*hd] Wv_h   [E][C]
    fold_mm(st, p->wo + h * hd, E, 1, p->wv + (int64_t)h * hd * C, C, 1, f.wov + h * a.Cp, (int64_t)H * a.Cp, E, C, hd,
            1.0f, nullptr);
  }
  // bov = Wo bv + bo
  fold_mm(st, p->wo, E, 1, bv, 1, 0, f.bov, 1, E, 1, E, 1.0f, p->out_bias);
  // W2f = [ W1a Wov | W1b | W1a bov ]
  const int64_t ld1 = E + d;
  fold_mm(st, p->fc1, ld1, 1, f.wov, (int64_t)H * a.Cp, 1, f.w2f, a.ld_kvc, d, H * a.Cp, E, 1.0f, nullptr);
  if (cudaMemcpy2DAsync(f.w2f + a.off_c, (size_t)a.ld_kvc * sizeof(float), p->fc1 + E, (size_t)ld1 * sizeof(float),
                        (size_t)d * sizeof(float), (size_t)d, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
    return TIGER_ECUDA;
  fold_mm(st, p->fc1, ld1, 1, f.bov, 1, 0, f.w2f + a.off_live, a.ld_kvc, d, 1, E, 1.0f, nullptr);
  if (tiger_launch_status() != TIGER_OK) return TIGER_ECUDA;
  int rc = tiger_gemm_pack_weight(f.wqk, E, nullptr, H * a.Cq, E, ATT_BN_QK, f.t_qk, f.pk_wqk, stream);
  if (rc != TIGER_OK) return rc;
  rc = tiger_gemm_pack_weight(f.w2f, a.ld_kvc, nullptr, d, a.off_live + 1, ATT_BN_D, f.t_d, f.pk_w2f, stream);
  if (rc != TIGER_OK) return rc;
  rc = tiger_gemm_pack_weight(p->fc2, d, nullptr, d, d, ATT_BN_F3, (d + ATT_BN_F3 - 1) / ATT_BN_F3, f.pk_fc2, stream);
  if (rc != TIGER_OK) return rc;
  if (p->time_w == nullptr || p->time_b == nullptr) return TIGER_EINVAL;
  // constant query time code folded into the bias (graph path)
  const int dt = E - d;
  attn_fold_time0_kernel<<<(dt + 127) / 128, 128, 0, st>>>(p->time_w, p->time_b, dt, f.tq);
  fold_mm(st, f.wqk + d, E, 1, f.tq, 1, 0, f.bqk_c, 1, H * a.Cq, 1, dt, 1.0f, f.bqk);
  if (tiger_launch_status() != TIGER_OK) return TIGER_ECUDA;
  return tiger_gemm_pack_weight(f.wqk, E, nullptr, H * a.Cq, d, ATT_BN_QK, f.t_qk, f.pk_wqk_c, stream);
}

// ------------------------------------------------------------------------------------------
// Link-scorer fold (tiger.py:259-288, basic_modules.py:16-19).  The scorer's first layer is linear in the
// two embeddings it concatenates: fc1([x + he_a | y + he_b]) = W1a x + W1b y + (W1a he_a + W1b he_b + b1), and
// the embeddings are themselves z = W2 hid + b2 (the merger's last layer).  So the LAST attention GEMM also
// emits P = W1a z and Q = W1b z for every query row (rows [W2 ; pad ; W1a W2 ; W1b W2] of one packed weight,
// split output), and scoring a pair is an elementwise relu(P[s] + Q[t] + c_ab) . w2 - the 17 us weight-
// streaming scorer kernel becomes a 2 x 688-byte row read per pair.
//   blob: w3 [n_split + 2d][d] | b3 [n_split + 2d] | cab [4][d] (c_ab, index 2a + b) | tf32 pack of w3
// The 'count' and 'vec' hit types (tiger_score_fold_hit) keep this head and append their tables [rows][d]:
//   count: U [K+1][d] | V [K+1][d], U[c] = b1 + W1a he_c, V[c] = W1b he_c (pair term U[ca] + V[cb])
//   vec  : b1 [d] | Ha^T [K][d] | Hb^T [K][d]; fc1 [d][2(d+K)] = [W1a | Ha | W1b | Hb] (pair term
//          b1 + sum of the Ha^T / Hb^T rows of the hit slots)
// ------------------------------------------------------------------------------------------
struct ScoreFold {
  float *w3, *b3, *cab, *pack, *hit;
  int n_split, tiles;
  int64_t total_floats;
};

static ScoreFold score_fold(int d, float* base) {
  ScoreFold f;
  int64_t off = 0;
  auto take = [&](int64_t cnt) { float* p = base ? base + off : nullptr; off += (cnt + 3) & ~(int64_t)3; return p; };
  f.n_split = (d + 15) & ~15;
  const int rows = f.n_split + 2 * d;
  f.tiles = (rows + ATT_BN_F3 - 1) / ATT_BN_F3;
  f.w3 = take((int64_t)rows * d);
  f.b3 = take(rows);
  f.cab = take(4 * d);
  f.pack = take(tiger_gemm_pack_bytes(f.tiles, d, ATT_BN_F3) / 4);
  f.hit = nullptr;
  f.total_floats = off;
  return f;
}

// rows [ ][d] of the hit tables behind the head; -1: not a hit type of tiger_score_fold_hit (or K out of range)
static int score_hit_rows(int hit_type, int k) {
  switch (hit_type) {
    case TIGER_HIT_NONE: case TIGER_HIT_BIN: return 0;
    case TIGER_HIT_VEC: return k > 0 ? 1 + 2 * k : -1;
    case TIGER_HIT_COUNT: return k > 0 ? 2 * (k + 1) : -1;
    default: return -1;
  }
}

static ScoreFold score_fold_hit(int d, int hit_type, int k, float* base) {
  ScoreFold f = score_fold(d, base);
  f.hit = base ? base + f.total_floats : nullptr;
  f.total_floats += ((int64_t)score_hit_rows(hit_type, k) * d + 3) & ~(int64_t)3;
  return f;
}

extern "C" int64_t tiger_score_fold_bytes(int d) {
  if (d <= 0) return -1;
  return score_fold(d, nullptr).total_floats * (int64_t)sizeof(float);
}

// float offset of the c_ab table [4][d] inside the blob (argument of tiger_link_score_folded)
extern "C" int64_t tiger_score_fold_cab_offset(int d) {
  if (d <= 0) return -1;
  float dummy;
  const ScoreFold f = score_fold(d, &dummy);
  return (int64_t)(f.cab - &dummy);
}

extern "C" int64_t tiger_score_fold_hit_bytes(int d, int hit_type, int k) {
  if (d <= 0 || score_hit_rows(hit_type, k) < 0) return -1;
  return score_fold_hit(d, hit_type, k, nullptr).total_floats * (int64_t)sizeof(float);
}

// float offset of the table tiger_link_score_folded_hit reads: c_ab for 'bin' / 'none', the hit tables otherwise
extern "C" int64_t tiger_score_fold_hit_offset(int d, int hit_type, int k) {
  if (d <= 0 || score_hit_rows(hit_type, k) < 0) return -1;
  float dummy;
  const ScoreFold f = score_fold_hit(d, hit_type, k, &dummy);
  return (int64_t)((hit_type == TIGER_HIT_VEC || hit_type == TIGER_HIT_COUNT ? f.hit : f.cab) - &dummy);
}

// hit tables of the 'count' / 'vec' fold (layout above), one thread per (row r, output m), double accumulation
__global__ void score_hit_fold_kernel(const float* __restrict__ fc1, int64_t ld1, const float* __restrict__ b1,
                                      const float* __restrict__ hit_emb, int d, int k, int hit_type,
                                      float* __restrict__ out) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (m >= d) return;
  const float* w = fc1 + (int64_t)m * ld1;
  double acc;
  if (hit_type == TIGER_HIT_COUNT) {
    const int side = r / (k + 1), c = r % (k + 1);        // rows [0, K] = U, [K+1, 2K+1] = V
    const float* wc = w + side * d;                        // W1a / W1b
    const float* e = hit_emb + (int64_t)c * d;
    acc = side == 0 ? (double)b1[m] : 0.0;
    for (int i = 0; i < d; ++i) acc += (double)wc[i] * (double)e[i];
  } else {                                                  // row 0 = b1, 1 + j = Ha[:, j], 1 + K + j = Hb[:, j]
    const int side = (r - 1) / k, j = (r - 1) % k;
    acc = r == 0 ? (double)b1[m] : (double)w[side * (d + k) + d + j];
  }
  out[(int64_t)r * d + m] = (float)acc;
}

extern "C" int tiger_score_fold_hit(const float* score_fc1, const float* score_fc1_b, const float* merger_fc2,
                                    const float* merger_fc2_b, const float* hit_emb, int d, int hit_type, int k,
                                    float* blob, void* stream) {
  const int hit_rows = score_hit_rows(hit_type, k);
  if (score_fc1 == nullptr || score_fc1_b == nullptr || merger_fc2 == nullptr || merger_fc2_b == nullptr ||
      blob == nullptr || d <= 0 || hit_rows < 0 || (((uintptr_t)blob) & 15) != 0)
    return TIGER_EINVAL;
  if ((hit_emb != nullptr) != (hit_type == TIGER_HIT_BIN || hit_type == TIGER_HIT_COUNT)) return TIGER_EINVAL;
  const ScoreFold f = score_fold_hit(d, hit_type, k, blob);
  cudaStream_t st = as_stream(stream);
  // fc1 [d][ld1]: [W1a | W1b] for 'bin' / 'none' / 'count', [W1a | Ha | W1b | Hb] for 'vec'
  const bool vec = hit_type == TIGER_HIT_VEC;
  const int64_t ld1 = vec ? 2 * (d + k) : 2 * d, w1b_col = vec ? d + k : d;
  if (cudaMemsetAsync(blob, 0, (size_t)f.total_floats * sizeof(float), st) != cudaSuccess) return TIGER_ECUDA;
  // rows [0, d): W2 (copy) ; rows [n_split, n_split + d): W1a W2 ; rows [n_split + d, n_split + 2d): W1b W2
  if (cudaMemcpyAsync(f.w3, merger_fc2, (size_t)d * d * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
      cudaMemcpyAsync(f.b3, merger_fc2_b, (size_t)d * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
    return TIGER_ECUDA;
  for (int half = 0; half < 2; ++half) {
    const float* w1 = score_fc1 + half * w1b_col;   // W1a / W1b
    fold_mm(st, w1, ld1, 1, merger_fc2, d, 1, f.w3 + (int64_t)(f.n_split + half * d) * d, d, d, d, d, 1.0f, nullptr);
    fold_mm(st, w1, ld1, 1, merger_fc2_b, 1, 0, f.b3 + f.n_split + half * d, 1, d, 1, d, 1.0f, nullptr);
  }
  if (hit_rows > 0) {
    score_hit_fold_kernel<<<dim3((unsigned)((d + 127) / 128), (unsigned)hit_rows), 128, 0, st>>>(
        score_fc1, ld1, score_fc1_b, hit_emb, d, k, hit_type, f.hit);
  } else {
    // c_ab = b1 + W1a he_a + W1b he_b
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b) {
        float* c = f.cab + (2 * a + b) * d;
        if (hit_emb == nullptr) {
          if (cudaMemcpyAsync(c, score_fc1_b, (size_t)d * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            return TIGER_ECUDA;
        } else {
          fold_mm(st, score_fc1, ld1, 1, hit_emb + a * d, 1, 0, c, 1, d, 1, d, 1.0f, score_fc1_b);
          // second half accumulates onto the first: add = c itself
          fold_mm(st, score_fc1 + d, ld1, 1, hit_emb + b * d, 1, 0, c, 1, d, 1, d, 1.0f, c);
        }
      }
  }
  if (tiger_launch_status() != TIGER_OK) return TIGER_ECUDA;
  return tiger_gemm_pack_weight(f.w3, d, nullptr, f.n_split + 2 * d, d, ATT_BN_F3, f.tiles, f.pack, stream);
}

extern "C" int tiger_score_fold(const float* score_fc1, const float* score_fc1_b, const float* merger_fc2,
                                const float* merger_fc2_b, const float* hit_emb, int d, float* blob, void* stream) {
  return tiger_score_fold_hit(score_fc1, score_fc1_b, merger_fc2, merger_fc2_b, hit_emb, d,
                              hit_emb != nullptr ? TIGER_HIT_BIN : TIGER_HIT_NONE, 0, blob, stream);
}

// ------------------------------------------------------------------------------------------
struct AttArgs {
  // gather mode
  const int64_t* center_nids;
  const float* q_ts;     // query q reads q_ts[(q / ts_group) % ts_period]
  int64_t ts_period;
  int64_t ts_group;
  const int64_t* neigh_nids;
  const int64_t* neigh_eids;
  const float* neigh_ts;
  const float* rows_a;
  const float* rows_b;
  const float* key_rows;   // [n_query * K][d] or NULL: slot (q, j) takes its node row from key_rows[q * K + j]
  const void* sel;
  int sel_is_i64;
  const float* nfeats;
  const float* efeats;
  // dense mode (TemporalAttention.forward signature)
  const float* qx;     // [n,d]
  const float* qt;     // [n,d]
  const float* kx;     // [n,K,d]
  const float* ky;     // [n,K,de]
  const float* kt;     // [n,K,d]
  const uint8_t* pad;  // [n,K]
  int dense;
  int64_t n_query;
  const float* time_w;
  const float* time_b;
  AttDims dm;
  AttWork w;
};

__device__ __forceinline__ const float* resolve_row(const AttArgs& a, int64_t u) {
  int64_t r;
  if (a.sel_is_i64)
    r = reinterpret_cast<const int64_t*>(a.sel)[u];
  else
    r = reinterpret_cast<const int32_t*>(a.sel)[u];
  if (a.rows_a == nullptr || r >= 0) return a.rows_b + r * a.dm.d;
  return a.rows_a + u * a.dm.d;
}

// one warp per query: XQ = [c | time code of dt = 0], KVC[:, c] = c, KVC[:, live] = any live slot
__global__ void __launch_bounds__(256) attn_prepare_kernel(const AttArgs a) {
  const int lane = lane_id();
  const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp_id_in_block();
  if (q >= a.n_query) return;
  const int d = a.dm.d, K = a.dm.K;
  float* xq = a.w.xq + q * a.dm.ld_xq;
  float* cc = a.w.kvc + q * a.dm.ld_kvc + a.dm.off_c;
  int any = 0;
  for (int j = lane; j < K; j += 32) any |= a.dense ? (a.pad[q * K + j] == 0) : (a.neigh_nids[q * K + j] != 0);
  any = __any_sync(TIGER_FULL_MASK, any);
  if (lane == 0) a.w.kvc[q * a.dm.ld_kvc + a.dm.off_live] = any ? 1.f : 0.f;
  if (a.dense) {
    for (int c = lane; c < d; c += 32) {
      const float v = a.qx[q * d + c];
      xq[c] = v;
      cc[c] = v;
      xq[d + c] = a.qt[q * d + c];
    }
  } else {
    const int64_t u = a.center_nids[q];
    const float* rp = resolve_row(a, u);
    const float* nfp = a.nfeats != nullptr ? a.nfeats + u * d : nullptr;
    for (int c = lane; c < d; c += 32) {
      const float v = rp[c] + (nfp != nullptr ? nfp[c] : 0.f);
      xq[c] = v;
      cc[c] = v;
      xq[d + c] = time_enc(0.f, a.time_w[c], a.time_b[c]);
    }
  }
}

// one CTA per query: stage the K key rows in shared memory, scores, masked softmax, pooled keys.
// The gathers of all K slots are issued together (every thread keeps up to 8 independent 16-byte loads in
// flight) - the kernel's time is the latency of those random-row reads, not their volume; the score
// weights of the query are staged in shared memory once.
// exact f / w for 0 <= f < 2^20 with a float reciprocal (the flattened (slot, column) loops below would
// otherwise spend more instructions on integer division than on their loads)
__device__ __forceinline__ int fast_div(int f, float inv_w) { return __float2int_rz(((float)f + 0.5f) * inv_w); }

// HT = number of heads as a compile-time constant (0: any number up to ATT_MAXH, predicated loops)
template <int HT>
__global__ void __launch_bounds__(ATT_THREADS, 5) attn_score_pool_kernel(const AttArgs a) {
  extern __shared__ __align__(16) float att_smem[];
  const int d = a.dm.d, de = a.dm.de, K = a.dm.K, H = HT > 0 ? HT : a.dm.H, C = a.dm.C, Cp = a.dm.Cp, Cq = a.dm.Cq;
  constexpr int HL = HT > 0 ? HT : ATT_MAXH;   // unrolled head loops run over HL, predicated by h < H
  float* kv = att_smem;                 // [K][Cp]
  float* sc = kv + K * Cp;              // [H][K]
  float* qk = sc + ((H * K + 3) & ~3);  // [H][Cq]   score weights of this query
  __shared__ const float* s_row[ATT_MAXK + 1];   // node representation row of slot j (NULL = padding slot)
  __shared__ const float* s_nf[ATT_MAXK + 1];    // entry K: the query's own (center) row, graph path only
  __shared__ const float* s_ef[ATT_MAXK];
  __shared__ float s_dt[ATT_MAXK];
  const int tid = threadIdx.x, lane = lane_id(), warp = warp_id_in_block(), n_warps = ATT_THREADS / 32;
  const int64_t q = blockIdx.x;
#ifdef TIGER_TRACE
  long long tr[10]; int trn = 0;
#define SP_MARK() tr[trn++] = clock64()
#else
#define SP_MARK() do { } while (0)
#endif
  SP_MARK();
  // Everything up to the scores reads what kernels BEFORE the Wqk product wrote (finder tables, GRU rows,
  // memories, and with key_rows the lower layer's output) - the Wqk product (graph path) releases its dependents
  // only after its own dependency wait, so those writes are complete when this CTA starts, and the gathers / time
  // codes below overlap that product.  The dense path's Wqk product triggers at its start: there the wait comes
  // first.  For key_rows this holds only while the lower layer's last product is launched before this layer's
  // Wqk product on the same programmatic-dependent chain (same stream, nothing reordered in between): forking the
  // upper layer's Wqk product onto another stream, or issuing it ahead of the lower layer's last product, needs
  // the key_rows gather moved behind pdl_wait().
  pdl_trigger();
  if (a.dense) pdl_wait();
  const float* qkf = a.w.qkf + q * a.dm.ld_qkf;
  if (tid < K) {
    const int64_t o = q * K + tid;
    const float* rp = nullptr;
    const float* nf = nullptr;
    const float* ef = nullptr;
    float dt = 0.f;
    if (a.dense) {
      if (a.pad[o] == 0) {
        rp = a.kx + o * d;
        ef = a.ky + o * de;
      }
    } else {
      const int64_t u = a.neigh_nids[o];
      if (u != 0) {
        if (a.key_rows != nullptr) {
          rp = a.key_rows + o * d;   // the lower layer's embedding of this slot: no node features on top
        } else {
          rp = resolve_row(a, u);
          nf = a.nfeats != nullptr ? a.nfeats + u * d : nullptr;
        }
        ef = a.efeats != nullptr ? a.efeats + a.neigh_eids[o] * de : nullptr;
        dt = a.q_ts[(q / a.ts_group) % a.ts_period] - a.neigh_ts[o];
      }
    }
    s_row[tid] = rp;
    s_nf[tid] = nf;
    s_ef[tid] = ef;
    s_dt[tid] = dt;
  } else if (tid == K && !a.dense) {
    const int64_t u = a.center_nids[q];
    s_row[K] = resolve_row(a, u);
    s_nf[K] = a.nfeats != nullptr ? a.nfeats + u * d : nullptr;
  }
  __syncthreads();
  SP_MARK();   // metadata
  float* out = a.w.kvc + q * a.dm.ld_kvc;
  // ---- gather: node rows (+ node features) and edge-feature rows of all slots ----
  const bool vec = (d & 3) == 0 && (de & 3) == 0 && (Cp & 3) == 0 &&
                   ((((uintptr_t)a.rows_a | (uintptr_t)a.rows_b | (uintptr_t)a.key_rows | (uintptr_t)a.nfeats |
                      (uintptr_t)a.efeats | (uintptr_t)a.kx | (uintptr_t)a.ky) & 15) == 0);
  const float inv_d = 1.0f / (float)d, inv_de = 1.0f / (float)de;
  if (vec) {
    const int d4 = d >> 2, de4 = de >> 2;
    const float inv_d4 = 1.0f / (float)d4, inv_de4 = 1.0f / (float)de4;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!a.dense) {
      // the query's own representation: the `c` columns of the second-stage operand (attn_prepare does this on
      // the dense path); the loads fly with the slot gathers below
      for (int c = tid; c < d4; c += ATT_THREADS) {
        float4 v = reinterpret_cast<const float4*>(s_row[K])[c];
        if (s_nf[K] != nullptr) {
          const float4 n4 = reinterpret_cast<const float4*>(s_nf[K])[c];
          v = make_float4(v.x + n4.x, v.y + n4.y, v.z + n4.z, v.w + n4.w);
        }
        reinterpret_cast<float4*>(out + a.dm.off_c)[c] = v;
      }
    }
    // first pass: the first 2 * ATT_THREADS node-row vectors and edge-feature vectors (everything at K <= 11,
    // d = 172) are loaded into registers here and stored only after the time codes below have been computed:
    // the cosines (a few thousand instructions per CTA) run while the random-row reads are in flight
    float4 pv[2], pn[2], pe[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int f = tid + u * ATT_THREADS;
      pv[u] = z4; pn[u] = z4; pe[u] = z4;
      if (f < K * d4) {
        const int j = fast_div(f, inv_d4), c = f - j * d4;
        if (s_row[j] != nullptr) {
          pv[u] = reinterpret_cast<const float4*>(s_row[j])[c];
          if (s_nf[j] != nullptr) pn[u] = reinterpret_cast<const float4*>(s_nf[j])[c];
        }
      }
      if (f < K * de4) {
        const int j = fast_div(f, inv_de4), c = f - j * de4;
        if (s_ef[j] != nullptr) pe[u] = reinterpret_cast<const float4*>(s_ef[j])[c];
      }
    }
    // ---- time code of every slot ----
    for (int f = tid; f < K * d; f += ATT_THREADS) {
      const int j = fast_div(f, inv_d), c = f - j * d;
      float v = 0.f;
      if (s_row[j] != nullptr)
        v = a.dense ? a.kt[(q * K + j) * d + c] : time_enc(s_dt[j], a.time_w[c], a.time_b[c]);
      kv[j * Cp + d + de + c] = v;
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int f = tid + u * ATT_THREADS;
      if (f < K * d4) {
        const int j = fast_div(f, inv_d4), c = f - j * d4;
        reinterpret_cast<float4*>(kv + j * Cp)[c] =
            make_float4(pv[u].x + pn[u].x, pv[u].y + pn[u].y, pv[u].z + pn[u].z, pv[u].w + pn[u].w);
      }
      if (f < K * de4) {
        const int j = fast_div(f, inv_de4), c = f - j * de4;
        reinterpret_cast<float4*>(kv + j * Cp + d)[c] = pe[u];
      }
    }
    // remaining vectors (large K): four loads in flight per thread
    for (int f0 = tid + 2 * ATT_THREADS; f0 < K * d4; f0 += 4 * ATT_THREADS) {
      float4 v[4], n4[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int f = f0 + u * ATT_THREADS;
        v[u] = z4;
        n4[u] = z4;
        if (f < K * d4) {
          const int j = fast_div(f, inv_d4), c = f - j * d4;
          if (s_row[j] != nullptr) {
            v[u] = reinterpret_cast<const float4*>(s_row[j])[c];
            if (s_nf[j] != nullptr) n4[u] = reinterpret_cast<const float4*>(s_nf[j])[c];
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int f = f0 + u * ATT_THREADS;
        if (f < K * d4) {
          const int j = fast_div(f, inv_d4), c = f - j * d4;
          reinterpret_cast<float4*>(kv + j * Cp)[c] =
              make_float4(v[u].x + n4[u].x, v[u].y + n4[u].y, v[u].z + n4[u].z, v[u].w + n4[u].w);
        }
      }
    }
    for (int f0 = tid + 2 * ATT_THREADS; f0 < K * de4; f0 += 4 * ATT_THREADS) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int f = f0 + u * ATT_THREADS;
        v[u] = z4;
        if (f < K * de4) {
          const int j = fast_div(f, inv_de4), c = f - j * de4;
          if (s_ef[j] != nullptr) v[u] = reinterpret_cast<const float4*>(s_ef[j])[c];
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int f = f0 + u * ATT_THREADS;
        if (f < K * de4) {
          const int j = fast_div(f, inv_de4), c = f - j * de4;
          reinterpret_cast<float4*>(kv + j * Cp + d)[c] = v[u];
        }
      }
    }
  } else {
    if (!a.dense)
      for (int c = tid; c < d; c += ATT_THREADS)
        out[a.dm.off_c + c] = s_row[K][c] + (s_nf[K] != nullptr ? s_nf[K][c] : 0.f);
    for (int f = tid; f < K * d; f += ATT_THREADS) {
      const int j = fast_div(f, inv_d), c = f - j * d;
      float v = 0.f;
      if (s_row[j] != nullptr) v = s_row[j][c] + (s_nf[j] != nullptr ? s_nf[j][c] : 0.f);
      kv[j * Cp + c] = v;
    }
    for (int f = tid; f < K * de; f += ATT_THREADS) {
      const int j = fast_div(f, inv_de), c = f - j * de;
      kv[j * Cp + d + c] = s_ef[j] != nullptr ? s_ef[j][c] : 0.f;
    }
    for (int f = tid; f < K * d; f += ATT_THREADS) {   // time code of every slot
      const int j = fast_div(f, inv_d), c = f - j * d;
      float v = 0.f;
      if (s_row[j] != nullptr)
        v = a.dense ? a.kt[(q * K + j) * d + c] : time_enc(s_dt[j], a.time_w[c], a.time_b[c]);
      kv[j * Cp + d + de + c] = v;
    }
  }
  SP_MARK();   // gathers + time code
  if (!a.dense) pdl_wait();      // qkf comes from the Wqk product
  for (int i = tid; i < H * Cq; i += ATT_THREADS) qk[i] = qkf[i];
  SP_MARK();
  __syncthreads();
  SP_MARK();   // time code
  // ---- scores: one warp per slot ----
  for (int j = warp; j < K; j += n_warps) {
    const float* row = kv + j * Cp;
    const bool live = s_row[j] != nullptr;
    float s[HL];
#pragma unroll
    for (int h = 0; h < HL; ++h) s[h] = 0.f;
    if (live) {
      for (int c = lane; c < C; c += 32) {
        const float v = row[c];
#pragma unroll
        for (int h = 0; h < HL; ++h)
          if (HT > 0 || h < H) s[h] = fmaf(qk[h * Cq + c], v, s[h]);
      }
    }
#pragma unroll
    for (int h = 0; h < HL; ++h) {
      if (HT > 0 || h < H) {
        const float t = warp_sum(s[h]);
        if (lane == 0) sc[h * K + j] = live ? t + qk[h * Cq + C] : -INFINITY;
      }
    }
  }
  __syncthreads();
  SP_MARK();   // scores
  // ---- masked softmax over the K slots, one warp per head (K <= ATT_MAXK = 64: two values per lane) ----
  for (int h = warp; h < H; h += n_warps) {
    float* row = sc + h * K;
    const float x0 = lane < K ? row[lane] : -INFINITY, x1 = lane + 32 < K ? row[lane + 32] : -INFINITY;
    const float m = warp_max(fmaxf(x0, x1));
    if (h == 0 && lane == 0 && !a.dense) out[a.dm.off_live] = m == -INFINITY ? 0.f : 1.f;
    float e0 = 0.f, e1 = 0.f;                 // every slot padding: the weights stay 0 and the pooled row is zero
    if (m != -INFINITY) {
      e0 = lane < K ? expf(x0 - m) : 0.f;
      e1 = lane + 32 < K ? expf(x1 - m) : 0.f;
      const float sum = warp_sum(e0 + e1);
      e0 = e0 / sum;
      e1 = e1 / sum;
    }
    if (lane < K) row[lane] = e0;
    if (lane + 32 < K) row[lane + 32] = e1;
  }
  __syncthreads();
  SP_MARK();   // softmax
  // ---- pooled keys kvbar[h][c] = sum_j p[h][j] kv[j][c] ----
  for (int c = tid; c < Cp; c += ATT_THREADS) {   // columns C..Cp-1 are alignment padding: written as zeros
    float acc[HL];
#pragma unroll
    for (int h = 0; h < HL; ++h) acc[h] = 0.f;
    for (int j = 0; j < (c < C ? K : 0); ++j) {
      const float v = kv[j * Cp + c];        // padding slots hold zeros and their weights are exactly 0
#pragma unroll
      for (int h = 0; h < HL; ++h)
        if (HT > 0 || h < H) acc[h] = fmaf(sc[h * K + j], v, acc[h]);
    }
#pragma unroll
    for (int h = 0; h < HL; ++h)
      if (HT > 0 || h < H) out[h * Cp + c] = acc[h];
  }
#ifdef TIGER_TRACE
  SP_MARK();
  if ((q == 0 || q == 300) && (tid == 0 || tid == 128))
    printf("pool q%d t%d: meta %lld gather %lld tcode %lld scores %lld softmax %lld pooled %lld\n", (int)q, tid, tr[1] - tr[0],
           tr[2] - tr[1], tr[3] - tr[2], tr[4] - tr[3], tr[5] - tr[4], tr[6] - tr[5]);
#endif
}

template <int HT>
static int launch_score_pool(const AttArgs& a, size_t smem, cudaStream_t st) {
  static size_t configured = 48 * 1024;
  if (smem > configured) {
    if (cudaFuncSetAttribute(attn_score_pool_kernel<HT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
        cudaSuccess)
      return TIGER_ECUDA;
    configured = smem;
  }
  return tiger_launch_chain(attn_score_pool_kernel<HT>, dim3((unsigned)a.n_query), dim3(ATT_THREADS), smem, st,
                            dim3(1, 1, 1), a);
}

static int attention_run(AttArgs& a, const tiger_attn_params* p, float* out, cudaStream_t st) {
  const AttDims& m = a.dm;
  const int64_t n = a.n_query;
  void* s = (void*)st;
  a.time_w = p->time_w;
  a.time_b = p->time_b;
  const AttFold f = att_fold(m, p->folded);
  int rc;
  if (a.dense) {
    attn_prepare_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(a);
    if (tiger_launch_status() != TIGER_OK) return TIGER_ECUDA;
    // [qk_h | qb_h] = XQ Wqk^T + bqk
    rc = tiger_sgemm_nt_packed(a.w.xq, m.ld_xq, f.pk_wqk, ATT_BN_QK, f.bqk, a.w.qkf, m.ld_qkf, n, nullptr, 1,
                               m.H * m.Cq, m.E, 1.0f, 0, s);
  } else {
    // graph path: no gather kernel - the GEMM's producers look the center rows up themselves, and the constant
    // time code of the query sits in the bias (K = d instead of 2d); attn_score_pool fills the c / live columns
    rc = tiger_sgemm_nt_packed_gather(a.center_nids, a.sel, a.sel_is_i64, a.rows_a, a.rows_b, m.d, a.nfeats, f.pk_wqk_c,
                                      ATT_BN_QK, f.bqk_c, a.w.qkf, m.ld_qkf, n, nullptr, 1, m.H * m.Cq, m.d, 1.0f, 0,
                                      s);
  }
  if (rc != TIGER_OK) return rc;
  const size_t smem = att_pool_smem(m);
  rc = m.H == 2 ? launch_score_pool<2>(a, smem, st)
       : m.H == 1 ? launch_score_pool<1>(a, smem, st)
       : m.H == 4 ? launch_score_pool<4>(a, smem, st)
                  : launch_score_pool<0>(a, smem, st);
  if (rc != TIGER_OK) return rc;
  // hidden = relu([kvbar | c | live] W2f^T + b1): the long K is split over a cluster of ATT_KPARTS CTAs per tile whose
  // partial tiles are summed through distributed shared memory ; z = hidden W2^T + b2
  rc = tiger_sgemm_nt_packed_splitk_fused(a.w.kvc, m.ld_kvc, f.pk_w2f, ATT_BN_D, p->fc1_b, a.w.hid, m.ld_hid,
                                          ATT_KPARTS, n, nullptr, 1, m.d, m.off_live + 1, 1.0f, 1, s);
  if (rc != TIGER_OK) return rc;
  if (p->score_folded != nullptr) {
    // batch-node depth of the fused routes: the last GEMM writes z -> out and [W1a z | W1b z] -> pq_out (link-scorer
    // fold) and, with left_wb, persists the winners' embeddings into the left memory (waits for left_wb->ready_event
    // first); a read-only query (tiger_temporal_attention_query) has no left_wb and the same product otherwise
    const ScoreFold sf = score_fold(m.d, p->score_folded);
    return tiger_sgemm_nt_packed_scatter(a.w.hid, m.ld_hid, sf.pack, ATT_BN_F3, sf.b3, out, m.d, m.d, p->pq_out, 2 * m.d,
                                         sf.n_split, 2 * m.d, n, m.d, p->left_wb, s);
  }
  return tiger_sgemm_nt_packed(a.w.hid, m.ld_hid, f.pk_fc2, ATT_BN_F3, p->fc2_b, out, m.d, n, nullptr, 1, m.d, m.d, 1.0f,
                               0, s);
}

static int attention_entry(AttArgs& a, int k, int d, int de, int n_head, const tiger_attn_params* params, float* out,
                           void* work, void* stream, bool query = false) {
  if (params == nullptr || params->folded == nullptr) return TIGER_EINVAL;
  // the fused last product comes whole (score fold, its pq output and the left write-back) and in the gather form only;
  // a query takes the score fold and its pq output without the write-back
  const bool fused = query || params->left_wb != nullptr;
  if ((fused && a.dense) || (params->score_folded != nullptr) != fused || (params->pq_out != nullptr) != fused ||
      (query && params->left_wb != nullptr))
    return TIGER_EINVAL;
  // limits checked before the first launch, so a refused call leaves its outputs and workspace untouched
  if (a.n_query < 0 || !att_dims_ok(k, d, de, n_head)) return TIGER_EINVAL;
  if ((2 * d) % n_head != 0 || (((uintptr_t)work) & 15) != 0) return TIGER_EINVAL;
  if (a.n_query == 0) return TIGER_OK;   // no workspace needed: tiger_temporal_attention_work_bytes(0, ..) is 0
  if (work == nullptr) return TIGER_EINVAL;
  a.dm = att_dims(d, de, k, n_head);
  a.w = att_work(a.dm, a.n_query, reinterpret_cast<float*>(work));
  return attention_run(a, params, out, as_stream(stream));
}

static int attention_gather(const int64_t* center_nids, const float* q_ts, int64_t n_query, int64_t ts_period,
                            int64_t ts_group, const int64_t* neigh_nids, const int64_t* neigh_eids, const float* neigh_ts,
                            int k, const float* rows_a, const float* rows_b, const float* key_rows, const void* sel,
                            int sel_is_i64, const float* nfeats, const float* efeats, int d, int de, int n_head,
                            const tiger_attn_params* params, float* out, void* work, void* stream, bool query) {
  if (rows_b == nullptr || sel == nullptr || ts_group <= 0) return TIGER_EINVAL;
  AttArgs a = {};
  a.center_nids = center_nids; a.q_ts = q_ts; a.ts_period = ts_period > 0 ? ts_period : n_query;
  a.ts_group = ts_group;
  a.neigh_nids = neigh_nids; a.neigh_eids = neigh_eids; a.neigh_ts = neigh_ts;
  a.rows_a = rows_a; a.rows_b = rows_b; a.key_rows = key_rows; a.sel = sel; a.sel_is_i64 = sel_is_i64;
  a.nfeats = nfeats; a.efeats = efeats; a.dense = 0;
  a.n_query = n_query;
  return attention_entry(a, k, d, de, n_head, params, out, work, stream, query);
}

extern "C" int tiger_temporal_attention_ex(const int64_t* center_nids, const float* q_ts, int64_t n_query,
                                           int64_t ts_period, int64_t ts_group, const int64_t* neigh_nids,
                                           const int64_t* neigh_eids, const float* neigh_ts, int k, const float* rows_a,
                                           const float* rows_b, const float* key_rows, const void* sel, int sel_is_i64,
                                           const float* nfeats, const float* efeats, int d, int de, int n_head,
                                           const tiger_attn_params* params, float* out, void* work, void* stream) {
  return attention_gather(center_nids, q_ts, n_query, ts_period, ts_group, neigh_nids, neigh_eids, neigh_ts, k, rows_a,
                          rows_b, key_rows, sel, sel_is_i64, nfeats, efeats, d, de, n_head, params, out, work, stream,
                          false);
}

extern "C" int tiger_temporal_attention_query(const int64_t* center_nids, const float* q_ts, int64_t n_query,
                                              int64_t ts_period, int64_t ts_group, const int64_t* neigh_nids,
                                              const int64_t* neigh_eids, const float* neigh_ts, int k,
                                              const float* rows_a, const float* rows_b, const float* key_rows,
                                              const void* sel, int sel_is_i64, const float* nfeats, const float* efeats,
                                              int d, int de, int n_head, const tiger_attn_params* params, float* out,
                                              void* work, void* stream) {
  return attention_gather(center_nids, q_ts, n_query, ts_period, ts_group, neigh_nids, neigh_eids, neigh_ts, k, rows_a,
                          rows_b, key_rows, sel, sel_is_i64, nfeats, efeats, d, de, n_head, params, out, work, stream,
                          true);
}

extern "C" int tiger_temporal_attention_dense(const float* qx, const float* qt, const float* kx, const float* ky,
                                              const float* kt, const uint8_t* padding_mask, int64_t n_query, int k,
                                              int d, int de, int n_head, const tiger_attn_params* params, float* out,
                                              void* work, void* stream) {
  AttArgs a = {};
  a.qx = qx; a.qt = qt; a.kx = kx; a.ky = ky; a.kt = kt; a.pad = padding_mask; a.dense = 1; a.ts_period = 1;
  a.ts_group = 1;
  a.n_query = n_query;
  return attention_entry(a, k, d, de, n_head, params, out, work, stream);
}
