// a7 + a9 + a10 (K6-K8): the 1-N scorer S = q.E^T + bias (models.py:433-437), the label-smoothed
// sigmoid-BCE (models.py:448-453) and its gradient fused into the scorer epilogue, then the two
// gradient contractions dq = G.E and dE = G^T.q.  The [B,N] logit matrix is never written in training:
// the epilogue turns each accumulator tile straight into loss partials, dbias partials and G.
// Labels are 1-bit rows (coper_csr_to_bits), not the reference's dense fp32 multi-hot (data.py:318-322).
//
// This file holds the exact-fp32 CUDA-core engine (COPER_PREC_FP32) and the precision dispatch; the
// tcgen05/TMEM engine lives in umma_score.cu.
#include "simt_gemm.cuh"

namespace coper {

// implemented in umma_score.cu (tcgen05 path); return COPER_ERR_UNSUPPORTED when not compiled in
int umma_score1n_fwd(const float* q, const float* E, const float* bias, int B, int64_t Ns, int d, float* scores,
                     int64_t ld, void* ws, size_t ws_bytes, int prec, cudaStream_t st);
size_t umma_score1n_workspace_bytes(int B, int64_t Ns, int d, int prec);
// implemented in umma_bce.cu (tcgen05 path)
size_t umma_bce_workspace_bytes(int B, int64_t Ns, int d, int prec);
size_t umma_bce_G_bytes(int B, int64_t Ns, int prec);
int umma_score1n_bce_fwd_bwd(const float* q, const float* E, const void* E_prepared, const float* bias,
                             const uint32_t* label_bits, int B,
                             int64_t Ns, int d, float pos, float neg, float inv_count, double* loss_sum, void* G,
                             int64_t ldG, float* dq, float* dE, float* dbias, void* ws, size_t ws_bytes, int prec,
                             double* dE_sumsq, cudaStream_t st);
int umma_score1n_dE(const void* G, int B, int64_t Ns, int d, float inv_count, float* dE, double* dE_sumsq, float* dbias,
                    void* ws, size_t ws_bytes, int prec, cudaStream_t st);

// implemented in umma_entity.cu (tcgen05 path): softmax cross-entropy over all entities
size_t umma_lse_workspace_bytes(int B, int64_t Ns, int d, int prec);
int umma_score1n_lse(const float* q, const float* E, const void* E_prepared, const float* bias, int B, int64_t Ns, int d,
                     float* ml, void* ws, size_t ws_bytes, int prec, cudaStream_t st);
int lse_reduce(const float* parts, int S, int B, float* ml, float* lse, cudaStream_t st);
float umma_ce_dE_inv_count(float inv_count, int64_t num_ent, int prec);
int umma_score1n_ce_fwd_bwd(const float* q, const float* E, const void* E_prepared, const float* bias,
                            const uint32_t* label_bits_t, const int32_t* rowptr, const float* lse, int B, int64_t Ns,
                            int d, int64_t num_ent, float eps, float inv_count, double* loss_sum, void* G, float* dq,
                            float* dE, float* dbias, void* ws, size_t ws_bytes, int prec, double* dE_sumsq,
                            cudaStream_t st);

using namespace simt;

struct BceArgs {
  const uint32_t* bits;
  int64_t words;
  float pos, neg, inv_count;
  float* loss_partials;  // [gridDim.y * gridDim.x]
  float* dbias_part;     // [gridDim.y, Ns]
};

__device__ __forceinline__ void bce_elem(float s, float z, float inv_count, float& loss, float& g) {
  // tf.nn.sigmoid_cross_entropy_with_logits: max(s,0) - s z + log1p(exp(-|s|))
  float e = expf(-fabsf(s));
  loss = fmaxf(s, 0.f) - s * z + log1pf(e);
  float sig = (s >= 0.f) ? 1.0f / (1.0f + e) : e / (1.0f + e);
  g = (sig - z) * inv_count;
}

template <int MODE>  // 0: write logits, 1: BCE epilogue (write G, loss partial, dbias partial)
__global__ void __launch_bounds__(THREADS) score_kernel(const float* __restrict__ q, const float* __restrict__ E,
                                                        const float* __restrict__ bias, int B, int64_t Ns, int d,
                                                        float* __restrict__ out, int64_t ld, BceArgs bce) {
  pdl_enter();
  __shared__ Smem sm;
  __shared__ float red32[32];
  // entity tiles on x (can be ~80k at 10M entities), batch tiles on y
  int64_t n0 = (int64_t)blockIdx.x * BN;
  int m0 = blockIdx.y * BM;
  SrcK A{q, d, B, d};
  SrcK Bs{E + n0 * d, d, Ns - n0, d};  // rebased so that tile-local column indices stay 32-bit
  float acc[8][8];
  zero_acc(acc);
  mainloop(A, Bs, m0, 0, 0, (d + BK - 1) / BK, acc, sm);

  float bj[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int64_t n = n0 + mt_col(j);
    bj[j] = (n < Ns) ? __ldg(bias + n) : 0.f;
  }
  if (MODE == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int b = m0 + mt_row(i);
      if (b >= B) continue;
      float* orow = out + (int64_t)b * ld + n0;
      // columns come in two contiguous strips of 4
      int c0 = mt_col(0), c1 = mt_col(4);
      if (n0 + c0 + 3 < Ns && ((reinterpret_cast<uintptr_t>(orow + c0) & 15) == 0)) {
        *reinterpret_cast<float4*>(orow + c0) =
            make_float4(acc[i][0] + bj[0], acc[i][1] + bj[1], acc[i][2] + bj[2], acc[i][3] + bj[3]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) if (n0 + c0 + j < Ns) orow[c0 + j] = acc[i][j] + bj[j];
      }
      if (n0 + c1 + 3 < Ns && ((reinterpret_cast<uintptr_t>(orow + c1) & 15) == 0)) {
        *reinterpret_cast<float4*>(orow + c1) =
            make_float4(acc[i][4] + bj[4], acc[i][5] + bj[5], acc[i][6] + bj[6], acc[i][7] + bj[7]);
      } else {
#pragma unroll
        for (int j = 4; j < 8; ++j) if (n0 + c1 + (j - 4) < Ns) orow[c1 + (j - 4)] = acc[i][j] + bj[j];
      }
    }
  } else {
    float lsum = 0.f;
    float cs[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) cs[j] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int b = m0 + mt_row(i);
      if (b >= B) continue;
      const uint32_t* brow = bce.bits + (int64_t)b * bce.words;
      float* grow = out + (int64_t)b * ld + n0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        int64_t n = n0 + mt_col(j);
        if (n >= Ns) continue;
        uint32_t w = __ldg(brow + (n >> 5));
        float z = ((w >> (n & 31)) & 1u) ? bce.pos : bce.neg;
        float l, g;
        bce_elem(acc[i][j] + bj[j], z, bce.inv_count, l, g);
        lsum += l;
        cs[j] += g;
        grow[mt_col(j)] = g;
      }
    }
    // deterministic block reductions: loss partial, per-column dbias partial
    float t = block_sum<float>(lsum, red32);
    if (threadIdx.x == 0) bce.loss_partials[(int64_t)blockIdx.y * gridDim.x + blockIdx.x] = t;
    float(*red)[BN] = reinterpret_cast<float(*)[BN]>(&sm.a[0][0][0]);  // 16 x 128 floats = 8 KB, sm is free now
    int ty = threadIdx.x >> 4;
#pragma unroll
    for (int j = 0; j < 8; ++j) red[ty][mt_col(j)] = cs[j];
    __syncthreads();
    if (threadIdx.x < BN) {
      float s = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) s += red[r][threadIdx.x];
      int64_t n = n0 + threadIdx.x;
      if (n < Ns) bce.dbias_part[(int64_t)blockIdx.y * Ns + n] = s;
    }
  }
}

// ---- softmax cross-entropy (include/coper.h), exact-fp32 engine
// (m, l) = (max, sum exp(s - max)) of the logits of one batch row over one 128-entity tile: per thread over its 8
// columns, then over the 16 threads that share the row in a fixed order
__device__ __forceinline__ void lse_pair_combine(float& m, float& l, float m2, float l2) {
  const float hi = fmaxf(m, m2);
  l = l * expf(m - hi) + l2 * expf(m2 - hi);
  m = hi;
}
__global__ void __launch_bounds__(THREADS, 1) score_lse_kernel(const float* __restrict__ q, const float* __restrict__ E,
                                                            const float* __restrict__ bias, int B, int64_t Ns, int d,
                                                            float2* __restrict__ part) {
  pdl_enter();
  __shared__ Smem sm;
  int64_t n0 = (int64_t)blockIdx.x * BN;
  int m0 = blockIdx.y * BM;
  SrcK A{q, d, B, d};
  SrcK Bs{E + n0 * d, d, Ns - n0, d};
  float acc[8][8];
  zero_acc(acc);
  mainloop(A, Bs, m0, 0, 0, (d + BK - 1) / BK, acc, sm);
  __syncthreads();                                  // the operand tiles are free: per-thread pairs [BM][16]
  float2(*pairs)[16] = reinterpret_cast<float2(*)[16]>(&sm);
  // logits in place; columns past the shard's last entity become -1e30 (exp = 0; the pair of a row without an
  // entity here is (-1e30, 0) after the fixed combine below)
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int64_t n = n0 + mt_col(j);
    const float bj = (n < Ns) ? __ldg(bias + n) : -1e30f;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i][j] += bj;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float m = acc[i][0], l = 0.f;
#pragma unroll
    for (int j = 1; j < 8; ++j) m = fmaxf(m, acc[i][j]);
#pragma unroll
    for (int j = 0; j < 8; ++j) l += (acc[i][j] > -1e30f) ? __expf(acc[i][j] - m) : 0.f;   // x <= 0: abs. error ~1e-7
    pairs[mt_row(i)][threadIdx.x & 15] = make_float2(m, l);
  }
  __syncthreads();
  if (threadIdx.x < BM && m0 + (int)threadIdx.x < B) {   // one thread per batch row: its 16 pairs in a fixed order
    float2 acc2 = pairs[threadIdx.x][0];
    for (int k = 1; k < 16; ++k) lse_pair_combine(acc2.x, acc2.y, pairs[threadIdx.x][k].x, pairs[threadIdx.x][k].y);
    part[(int64_t)blockIdx.x * B + m0 + threadIdx.x] = acc2;
  }
}

struct CeArgs {
  const uint32_t* bits;
  int64_t words;
  const int32_t* rowptr;
  const float* lse;
  float eps, eN, inv_count;
  float* loss_partials;  // [gridDim.y * gridDim.x]
  float* dbias_part;     // [gridDim.y, Ns]
};
// G = (tau exp(s - lse) - t) * inv_count, loss = t (lse - s)
__global__ void __launch_bounds__(THREADS) score_ce_kernel(const float* __restrict__ q, const float* __restrict__ E,
                                                           const float* __restrict__ bias, int B, int64_t Ns, int d,
                                                           float* __restrict__ out, int64_t ld, CeArgs ce) {
  pdl_enter();
  __shared__ Smem sm;
  __shared__ float red32[32];
  int64_t n0 = (int64_t)blockIdx.x * BN;
  int m0 = blockIdx.y * BM;
  SrcK A{q, d, B, d};
  SrcK Bs{E + n0 * d, d, Ns - n0, d};
  float acc[8][8];
  zero_acc(acc);
  mainloop(A, Bs, m0, 0, 0, (d + BK - 1) / BK, acc, sm);
  float bj[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int64_t n = n0 + mt_col(j);
    bj[j] = (n < Ns) ? __ldg(bias + n) : 0.f;
  }
  float lsum = 0.f;
  float cs[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) cs[j] = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int b = m0 + mt_row(i);
    if (b >= B) continue;
    const int nb = __ldg(ce.rowptr + b + 1) - __ldg(ce.rowptr + b);
    const float tau = nb > 0 ? 1.0f : ce.eps;
    const float pw = (1.0f - ce.eps) / (float)max(nb, 1);
    const float lse = __ldg(ce.lse + b);
    const uint32_t* brow = ce.bits + (int64_t)b * ce.words;
    float* grow = out + (int64_t)b * ld + n0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int64_t n = n0 + mt_col(j);
      if (n >= Ns) continue;
      uint32_t w = __ldg(brow + (n >> 5));
      const float t = (((w >> (n & 31)) & 1u) ? pw : 0.f) + ce.eN;
      const float s = acc[i][j] + bj[j];
      const float g = (tau * expf(s - lse) - t) * ce.inv_count;
      lsum += t * (lse - s);
      cs[j] += g;
      grow[mt_col(j)] = g;
    }
  }
  float t = block_sum<float>(lsum, red32);
  if (threadIdx.x == 0) ce.loss_partials[(int64_t)blockIdx.y * gridDim.x + blockIdx.x] = t;
  float(*red)[BN] = reinterpret_cast<float(*)[BN]>(&sm.a[0][0][0]);
  int ty = threadIdx.x >> 4;
#pragma unroll
  for (int j = 0; j < 8; ++j) red[ty][mt_col(j)] = cs[j];
  __syncthreads();
  if (threadIdx.x < BN) {
    float s = 0.f;
#pragma unroll
    for (int r = 0; r < 16; ++r) s += red[r][threadIdx.x];
    int64_t n = n0 + threadIdx.x;
    if (n < Ns) ce.dbias_part[(int64_t)blockIdx.y * Ns + n] = s;
  }
}

// dq partial[split][b][j] = sum_{n in split} G[b,n] E[n,j]
__global__ void __launch_bounds__(THREADS) dq_kernel(const float* __restrict__ G, int64_t ldG,
                                                     const float* __restrict__ E, int B, int64_t Ns, int d,
                                                     int tiles_per_split, float* __restrict__ part) {
  pdl_enter();
  __shared__ Smem sm;
  int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM, split = blockIdx.z;
  int ktiles = (int)((Ns + BK - 1) / BK);
  int t0 = split * tiles_per_split;
  int t1 = min(ktiles, t0 + tiles_per_split);
  SrcK A{G, ldG, B, Ns};
  SrcMN Bs{E, d, d, Ns};
  float acc[8][8];
  zero_acc(acc);
  mainloop(A, Bs, m0, n0, t0, t1, acc, sm);
  float* o = part + (int64_t)split * B * d;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int b = m0 + mt_row(i);
    if (b >= B) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int c = n0 + mt_col(j);
      if (c < d) o[(int64_t)b * d + c] = acc[i][j];
    }
  }
}

// dE[n][j] = sum_b G[b,n] q[b,j]
__global__ void __launch_bounds__(THREADS) dE_kernel(const float* __restrict__ G, int64_t ldG,
                                                     const float* __restrict__ q, int B, int64_t Ns, int d,
                                                     float* __restrict__ dE) {
  pdl_enter();
  __shared__ Smem sm;
  int64_t e0 = (int64_t)blockIdx.x * BM;
  int n0 = blockIdx.y * BN;
  SrcMN A{G + e0, ldG, Ns - e0, B};
  SrcMN Bs{q, d, d, B};
  float acc[8][8];
  zero_acc(acc);
  mainloop(A, Bs, 0, n0, 0, (B + BK - 1) / BK, acc, sm);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int64_t e = e0 + mt_row(i);
    if (e >= Ns) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int c = n0 + mt_col(j);
      if (c < d) dE[e * d + c] = acc[i][j];
    }
  }
}

__global__ void sum_to_double_kernel(const float* __restrict__ in, int64_t n, double* out) {
  pdl_enter();
  __shared__ double smd[32];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += (double)in[i];
  double t = block_sum<double>(acc, smd);
  if (threadIdx.x == 0) *out = t;
}

struct BceLayout {
  int gx, gy, splits, tiles_per_split;
  size_t off_loss, off_dbias, off_dq, total;
};
static BceLayout bce_layout(int B, int64_t Ns, int d) {
  BceLayout L;
  L.gx = ceil_div(Ns, BN);
  L.gy = ceil_div(B, BM);
  int tiles_mn = ceil_div(d, BN) * L.gy;
  int ktiles = ceil_div(Ns, BK);
  int splits = (2 * 148 + tiles_mn - 1) / tiles_mn;
  if (splits > ktiles) splits = ktiles;
  if (splits < 1) splits = 1;
  L.tiles_per_split = (ktiles + splits - 1) / splits;
  L.splits = (ktiles + L.tiles_per_split - 1) / L.tiles_per_split;
  size_t o = 0;
  L.off_loss = o; o = align_up(o + (size_t)L.gx * L.gy * sizeof(float), 256);
  L.off_dbias = o; o = align_up(o + (size_t)L.gy * Ns * sizeof(float), 256);
  L.off_dq = o; o = align_up(o + (size_t)L.splits * B * d * sizeof(float), 256);
  L.total = o;
  return L;
}
}  // namespace coper

using namespace coper;

extern "C" {

size_t coper_score1n_workspace_bytes(int B, int64_t Ns, int d, int prec) {
  if (prec == COPER_PREC_FP32) return 256;
  return umma_score1n_workspace_bytes(B, Ns, d, prec);
}

int coper_score1n_fwd(const float* q, const float* E, const float* bias, int B, int64_t Ns, int d, float* scores,
                      int64_t ld_scores, void* workspace, size_t workspace_bytes, int prec, coper_stream_t stream) {
  COPER_CHECK_ARG(q && E && bias && scores && B > 0 && Ns > 0 && d > 0 && ld_scores >= Ns);
  if (prec != COPER_PREC_FP32)
    return umma_score1n_fwd(q, E, bias, B, Ns, d, scores, ld_scores, workspace, workspace_bytes, prec, as_stream(stream));
  dim3 grid(ceil_div(Ns, BN), ceil_div(B, BM));
  BceArgs none{};
  launch_pdl(score_kernel<0>, grid, THREADS, 0, as_stream(stream), q, E, bias, B, Ns, d, scores, ld_scores, none);
  return check_launch();
}

size_t coper_score1n_bce_workspace_bytes(int B, int64_t Ns, int d, int prec) {
  if (prec != COPER_PREC_FP32) return umma_bce_workspace_bytes(B, Ns, d, prec);
  return bce_layout(B, Ns, d).total;
}
size_t coper_score1n_bce_G_bytes(int B, int64_t Ns, int prec) {
  if (prec != COPER_PREC_FP32) return umma_bce_G_bytes(B, Ns, prec);
  return (size_t)B * ((Ns + 31) / 32 * 32) * sizeof(float);
}

static int fp32_grad_tail(const float* q, const float* E, int B, int64_t Ns, int d, double* loss_sum, const float* G,
                          int64_t ldG, float* dq, float* dE, float* dbias, void* workspace, coper_stream_t stream);

static int score1n_bce_impl(const float* q, const float* E, const void* E_prepared, const float* bias,
                            const uint32_t* label_bits, int B, int64_t Ns, int d, float pos_target, float neg_target,
                            float inv_count, double* loss_sum, void* Gv, int64_t ldG, float* dq, float* dE, float* dbias,
                            void* workspace, size_t workspace_bytes, int prec, double* dE_sumsq, coper_stream_t stream) {
  COPER_CHECK_ARG(q && E && bias && label_bits && loss_sum && Gv && dq && dbias && workspace);
  COPER_CHECK_ARG(B > 0 && Ns > 0 && d > 0 && ldG >= Ns);
  COPER_CHECK_ARG(dE || (prec != COPER_PREC_FP32 && dE_sumsq));   // dE == NULL: split call, see coper_score1n_bce_dE
  if (prec == COPER_PREC_BF16 || prec == COPER_PREC_TF32X3 || prec == COPER_PREC_FP16X3)
    return umma_score1n_bce_fwd_bwd(q, E, E_prepared, bias, label_bits, B, Ns, d, pos_target, neg_target, inv_count, loss_sum, Gv,
                                    ldG, dq, dE, dbias, workspace, workspace_bytes, prec, dE_sumsq, as_stream(stream));
  if (prec != COPER_PREC_FP32) return COPER_ERR_UNSUPPORTED;
  if (dE_sumsq) return COPER_ERR_UNSUPPORTED;         // the CUDA-core engine does not fuse the norm (callers pass NULL)
  float* G = static_cast<float*>(Gv);
  BceLayout L = bce_layout(B, Ns, d);
  if (workspace_bytes < L.total) return COPER_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  char* ws = static_cast<char*>(workspace);
  float* loss_part = reinterpret_cast<float*>(ws + L.off_loss);
  float* dbias_part = reinterpret_cast<float*>(ws + L.off_dbias);
  BceArgs bce{label_bits, (Ns + 31) / 32, pos_target, neg_target, inv_count, loss_part, dbias_part};
  launch_pdl(score_kernel<1>, dim3(L.gx, L.gy), THREADS, 0, st, q, E, bias, B, Ns, d, G, ldG, bce);
  int rc = check_launch();
  if (rc) return rc;
  return fp32_grad_tail(q, E, B, Ns, d, loss_sum, G, ldG, dq, dE, dbias, workspace, stream);
}

// after the fp32 scorer pass (loss / dbias partials in the workspace, G): loss sum, dbias, dq = G.E, dE = G^T.q
static int fp32_grad_tail(const float* q, const float* E, int B, int64_t Ns, int d, double* loss_sum, const float* G,
                          int64_t ldG, float* dq, float* dE, float* dbias, void* workspace, coper_stream_t stream) {
  BceLayout L = bce_layout(B, Ns, d);
  cudaStream_t st = as_stream(stream);
  char* ws = static_cast<char*>(workspace);
  float* loss_part = reinterpret_cast<float*>(ws + L.off_loss);
  float* dbias_part = reinterpret_cast<float*>(ws + L.off_dbias);
  float* dq_part = reinterpret_cast<float*>(ws + L.off_dq);
  int rc;
  launch_pdl(sum_to_double_kernel, 1, 1024, 0, st, loss_part, (int64_t)L.gx * L.gy, loss_sum);
  if ((rc = check_launch())) return rc;
  rc = coper_reduce_partials(dbias_part, L.gy, Ns, 1.0f, 0, dbias, stream);
  if (rc) return rc;
  launch_pdl(dq_kernel, dim3(ceil_div(d, BN), L.gy, L.splits), THREADS, 0, st, G, ldG, E, B, Ns, d,
             L.tiles_per_split, dq_part);
  if ((rc = check_launch())) return rc;
  rc = coper_reduce_partials(dq_part, L.splits, (int64_t)B * d, 1.0f, 0, dq, stream);
  if (rc) return rc;
  launch_pdl(dE_kernel, dim3(ceil_div(Ns, BM), ceil_div(d, BN)), THREADS, 0, st, G, ldG, q, B, Ns, d, dE);
  return check_launch();
}

int coper_score1n_bce_fwd_bwd(const float* q, const float* E, const void* E_prepared, const float* bias,
                              const uint32_t* label_bits, int B, int64_t Ns, int d, float pos_target, float neg_target,
                              float inv_count, double* loss_sum, void* Gv, int64_t ldG, float* dq, float* dE,
                              float* dbias, void* workspace, size_t workspace_bytes, int prec, coper_stream_t stream) {
  return score1n_bce_impl(q, E, E_prepared, bias, label_bits, B, Ns, d, pos_target, neg_target, inv_count, loss_sum, Gv,
                          ldG, dq, dE, dbias, workspace, workspace_bytes, prec, nullptr, stream);
}
int coper_score1n_bce_dE(const void* G, int B, int64_t Ns, int d, float inv_count, float* dE, double* dE_sumsq,
                         float* dbias, void* workspace, size_t workspace_bytes, int prec, coper_stream_t stream) {
  COPER_CHECK_ARG(G && dE && dbias && workspace && B > 0 && Ns > 0 && d > 0);
  if (prec != COPER_PREC_BF16 && prec != COPER_PREC_TF32X3 && prec != COPER_PREC_FP16X3) return COPER_ERR_UNSUPPORTED;
  return umma_score1n_dE(G, B, Ns, d, inv_count, dE, dE_sumsq, dbias, workspace, workspace_bytes, prec, as_stream(stream));
}
int coper_score1n_bce_fwd_bwd_norm(const float* q, const float* E, const void* E_prepared, const float* bias,
                                   const uint32_t* label_bits, int B, int64_t Ns, int d, float pos_target,
                                   float neg_target, float inv_count, double* loss_sum, void* Gv, int64_t ldG, float* dq,
                                   float* dE, float* dbias, double* dE_sumsq, void* workspace, size_t workspace_bytes,
                                   int prec, coper_stream_t stream) {
  COPER_CHECK_ARG(dE_sumsq);
  return score1n_bce_impl(q, E, E_prepared, bias, label_bits, B, Ns, d, pos_target, neg_target, inv_count, loss_sum, Gv,
                          ldG, dq, dE, dbias, workspace, workspace_bytes, prec, dE_sumsq, stream);
}

// ---- softmax cross-entropy over all entities
size_t coper_score1n_lse_workspace_bytes(int B, int64_t Ns, int d, int prec) {
  if (prec == COPER_PREC_FP32) return align_up((size_t)ceil_div(Ns, BN) * B * sizeof(float2), 256);
  if (prec != COPER_PREC_BF16 && prec != COPER_PREC_TF32X3 && prec != COPER_PREC_FP16X3) return 0;
  return umma_lse_workspace_bytes(B, Ns, d, prec);
}
int coper_score1n_lse(const float* q, const float* E, const void* E_prepared, const float* bias, int B, int64_t Ns, int d,
                      float* ml, void* workspace, size_t workspace_bytes, int prec, coper_stream_t stream) {
  COPER_CHECK_ARG(q && E && bias && ml && workspace && B > 0 && Ns > 0 && d > 0);
  if (prec == COPER_PREC_BF16 || prec == COPER_PREC_TF32X3 || prec == COPER_PREC_FP16X3)
    return umma_score1n_lse(q, E, E_prepared, bias, B, Ns, d, ml, workspace, workspace_bytes, prec, as_stream(stream));
  if (prec != COPER_PREC_FP32) return COPER_ERR_UNSUPPORTED;
  if (workspace_bytes < coper_score1n_lse_workspace_bytes(B, Ns, d, prec)) return COPER_ERR_WORKSPACE;
  const int gx = ceil_div(Ns, BN);
  cudaStream_t st = as_stream(stream);
  float2* part = static_cast<float2*>(workspace);
  launch_pdl(score_lse_kernel, dim3(gx, ceil_div(B, BM)), THREADS, 0, st, q, E, bias, B, Ns, d, part);
  int rc = check_launch();
  if (rc) return rc;
  return lse_reduce(reinterpret_cast<const float*>(part), gx, B, ml, nullptr, st);
}
int coper_lse_finalize(const float* parts, int P, int B, float* lse, coper_stream_t stream) {
  COPER_CHECK_ARG(parts && lse && P > 0 && B > 0);
  return lse_reduce(parts, P, B, nullptr, lse, as_stream(stream));
}
float coper_score1n_ce_dE_inv_count(float inv_count, int64_t num_ent, int prec) {
  return umma_ce_dE_inv_count(inv_count, num_ent, prec);
}

static int score1n_ce_impl(const float* q, const float* E, const void* E_prepared, const float* bias,
                           const uint32_t* label_bits, const int32_t* rowptr, const float* lse, int B, int64_t Ns, int d,
                           int64_t num_ent, float eps, float inv_count, double* loss_sum, void* Gv, int64_t ldG, float* dq,
                           float* dE, float* dbias, void* workspace, size_t workspace_bytes, int prec, double* dE_sumsq,
                           coper_stream_t stream) {
  COPER_CHECK_ARG(q && E && bias && label_bits && rowptr && lse && loss_sum && Gv && dq && dbias && workspace);
  COPER_CHECK_ARG(B > 0 && Ns > 0 && d > 0 && ldG >= Ns && num_ent >= Ns && eps >= 0.f && eps <= 1.f);
  COPER_CHECK_ARG(dE || (prec != COPER_PREC_FP32 && dE_sumsq));   // dE == NULL: split call, see coper_score1n_bce_dE
  if (prec == COPER_PREC_BF16 || prec == COPER_PREC_TF32X3 || prec == COPER_PREC_FP16X3)
    return umma_score1n_ce_fwd_bwd(q, E, E_prepared, bias, label_bits, rowptr, lse, B, Ns, d, num_ent, eps, inv_count,
                                   loss_sum, Gv, dq, dE, dbias, workspace, workspace_bytes, prec, dE_sumsq,
                                   as_stream(stream));
  if (prec != COPER_PREC_FP32) return COPER_ERR_UNSUPPORTED;
  if (dE_sumsq) return COPER_ERR_UNSUPPORTED;
  float* G = static_cast<float*>(Gv);
  BceLayout L = bce_layout(B, Ns, d);
  if (workspace_bytes < L.total) return COPER_ERR_WORKSPACE;
  char* ws = static_cast<char*>(workspace);
  CeArgs ce{label_bits, (Ns + 31) / 32, rowptr, lse, eps, (float)((double)eps / (double)num_ent), inv_count,
            reinterpret_cast<float*>(ws + L.off_loss), reinterpret_cast<float*>(ws + L.off_dbias)};
  launch_pdl(score_ce_kernel, dim3(L.gx, L.gy), THREADS, 0, as_stream(stream), q, E, bias, B, Ns, d, G, ldG, ce);
  int rc = check_launch();
  if (rc) return rc;
  return fp32_grad_tail(q, E, B, Ns, d, loss_sum, G, ldG, dq, dE, dbias, workspace, stream);
}
int coper_score1n_ce_fwd_bwd(const float* q, const float* E, const void* E_prepared, const float* bias,
                             const uint32_t* label_bits, const int32_t* rowptr, const float* lse, int B, int64_t Ns, int d,
                             int64_t num_ent, float eps, float inv_count, double* loss_sum, void* G, int64_t ldG,
                             float* dq, float* dE, float* dbias, void* workspace, size_t workspace_bytes, int prec,
                             coper_stream_t stream) {
  return score1n_ce_impl(q, E, E_prepared, bias, label_bits, rowptr, lse, B, Ns, d, num_ent, eps, inv_count, loss_sum, G,
                         ldG, dq, dE, dbias, workspace, workspace_bytes, prec, nullptr, stream);
}
int coper_score1n_ce_fwd_bwd_norm(const float* q, const float* E, const void* E_prepared, const float* bias,
                                  const uint32_t* label_bits, const int32_t* rowptr, const float* lse, int B, int64_t Ns,
                                  int d, int64_t num_ent, float eps, float inv_count, double* loss_sum, void* G,
                                  int64_t ldG, float* dq, float* dE, float* dbias, double* dE_sumsq, void* workspace,
                                  size_t workspace_bytes, int prec, coper_stream_t stream) {
  COPER_CHECK_ARG(dE_sumsq);
  return score1n_ce_impl(q, E, E_prepared, bias, label_bits, rowptr, lse, B, Ns, d, num_ent, eps, inv_count, loss_sum, G,
                         ldG, dq, dE, dbias, workspace, workspace_bytes, prec, dE_sumsq, stream);
}

}  // extern "C"
