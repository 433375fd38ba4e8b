// a3 + a6 (K2 + K3): fused contextual-parameter "generate-and-apply".
//
// Reference: W_b = reshape(c_b . P, [F, d]) is materialised for every query ([B,F,d] fp32 = 1.9 GB at
// FB15k-237, models.py:70-73) and then applied with a batched mat-vec (models.py:412).  Here the
// contraction is evaluated directly as
//     y = (c (x) f) . P^ + cb . Pb ,   P^ = P viewed [dc*F, d]
// with the Khatri-Rao operand (c (x) f) synthesised tile-by-tile in shared memory: P^ is streamed once,
// the per-query weights never exist in HBM.  K = dc*F (36,864 .. 200,704) against an output of only
// [B, d], so the K range is split across CTAs and reduced in a fixed order (deterministic).
//
// Backward (autodiff of the above, models.py:198):
//     T_k = dy . P[k]^T                      (never stored)
//     df  = sum_k c[:,k] * T_k               dc[:,k] = rowsum(f * T_k)         (T kernel, epilogue-reduced)
//     dP[k] = f^T . (c[:,k] * dy)            dPb = cb^T . dy    dcb = dy . Pb^T
//
// This file: exact-fp32 CUDA-core engine (COPER_PREC_FP32) + dispatch + the plain sgemm used by the small
// dense layers.  tcgen05 engine: umma_cpg.cu.
#include "simt_gemm.cuh"

namespace coper {
using namespace simt;

// tcgen05 engine (umma_cpg.cu)
size_t umma_cpg_fwd_workspace_bytes(int B, int dc, int F, int d, int prec);
size_t umma_cpg_bwd_workspace_bytes(int B, int dc, int F, int d, int prec);
int umma_cpg_fwd_partials(const float* c, const float* f, const float* P, const void* P_prepared, int B, int dc, int F,
                          int d, void* ws, size_t ws_bytes, int prec, cudaStream_t st, float** slabs, int* n_slabs);
int umma_cpg_bwd(const float* c, const float* f, const float* P, const void* P_prepared, const float* dy, int B, int dc,
                 int F, int d, float* dP, float* df, float* dc_out, void* ws, size_t ws_bytes, int prec,
                 int flags, cudaStream_t st);

// ---------------------------------------------------------------- sources
struct CpgFwdA {  // (b, kk) -> f[b, i] * c[b, kq],  K-contiguous
  static constexpr bool kKContig = true;
  const float* f;
  const float* c;
  int B, F, dc, nt;
  int kq = 0, i0 = 0;
  __device__ __forceinline__ void tile(int t) { kq = t / nt; i0 = (t - kq * nt) * BK; }
  __device__ __forceinline__ float at(int b, int kk) const {
    int i = i0 + kk;
    return (b < B && i < F) ? __ldg(f + (int64_t)b * F + i) * __ldg(c + (int64_t)b * dc + kq) : 0.f;
  }
};
struct CpgFwdB {  // (j, kk) -> P[kq, i, j],  MN-contiguous
  static constexpr bool kKContig = false;
  const float* P;
  int F, d, nt;
  int kq = 0, i0 = 0;
  __device__ __forceinline__ void tile(int t) { kq = t / nt; i0 = (t - kq * nt) * BK; }
  __device__ __forceinline__ float at(int j, int kk) const {
    int i = i0 + kk;
    return (j < d && i < F) ? __ldg(P + ((int64_t)kq * F + i) * d + j) : 0.f;
  }
};
struct ScaledMN {  // (j, kk) -> x[b, j] * s[b, kq] with b = k index,  MN-contiguous
  static constexpr bool kKContig = false;
  const float* x;
  const float* s;
  int ld, mn_ext, k_ext, lds, kq;
  int k0 = 0;
  __device__ __forceinline__ void tile(int t) { k0 = t * BK; }
  __device__ __forceinline__ float at(int j, int kk) const {
    int b = k0 + kk;
    return (j < mn_ext && b < k_ext) ? __ldg(x + (int64_t)b * ld + j) * __ldg(s + (int64_t)b * lds + kq) : 0.f;
  }
};

// ---------------------------------------------------------------- forward
__global__ void __launch_bounds__(THREADS) cpg_fwd_kernel(const float* __restrict__ c, const float* __restrict__ f,
                                                          const float* __restrict__ P, int B, int dc, int F, int d,
                                                          int tiles_per_split, float* __restrict__ part) {
  pdl_enter();
  __shared__ Smem sm;
  int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM, split = blockIdx.z;
  int nt = (F + BK - 1) / BK;
  int T = dc * nt;
  int t0 = split * tiles_per_split;
  int t1 = min(T, t0 + tiles_per_split);
  CpgFwdA A{f, c, B, F, dc, nt};
  CpgFwdB Bs{P, F, d, nt};
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
      int col = n0 + mt_col(j);
      if (col < d) o[(int64_t)b * d + col] = acc[i][j];
    }
  }
}

// y = sum_s part[s] + cb . Pb, then output dropout (models.py:414-415)
__global__ void cpg_fwd_finalize_kernel(const float* __restrict__ part, int S, const float* __restrict__ cb,
                                        const float* __restrict__ Pb, int B, int d, int dcb, float keep,
                                        float inv_keep, uint32_t thr, const uint64_t* seed_dev, uint64_t salt,
                                        float* __restrict__ y) {
  pdl_enter();
  uint64_t seed = (seed_dev ? *seed_dev : 0ull) + salt;
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t n = (int64_t)B * d;
  if (e >= n) return;
  int b = (int)(e / d), j = (int)(e % d);
  double acc = 0.0;
  // slabs are summed in slab order (deterministic); the loads of 8 slabs are issued together, the adds stay ordered
  int s = 0;
  for (; s + 8 <= S; s += 8) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = __ldg(part + (int64_t)(s + u) * n + e);
#pragma unroll
    for (int u = 0; u < 8; ++u) acc += (double)v[u];
  }
  for (; s < S; ++s) acc += (double)__ldg(part + (int64_t)s * n + e);
  float bias = 0.f;
  for (int k = 0; k < dcb; ++k) bias = fmaf(__ldg(cb + (int64_t)b * dcb + k), __ldg(Pb + (int64_t)k * d + j), bias);
  float v = (float)acc + bias;
  y[e] = v * drop_factor(keep, inv_keep, thr, seed, (uint64_t)e);
}

// float4 form (d % 4 == 0, 16-byte aligned slabs / Pb / y): four adjacent outputs per thread, same slab order and the
// same fmaf chain per output -> same bits as cpg_fwd_finalize_kernel
__global__ void cpg_fwd_finalize_kernel4(const float* __restrict__ part, int S, const float* __restrict__ cb,
                                         const float* __restrict__ Pb, int B, int d, int dcb, float keep, float inv_keep,
                                         uint32_t thr, const uint64_t* seed_dev, uint64_t salt, float* __restrict__ y) {
  pdl_enter();
  const uint64_t seed = (seed_dev ? *seed_dev : 0ull) + salt;
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int64_t n = (int64_t)B * d;
  if (e >= n) return;
  const int b = (int)(e / d), j = (int)(e % d);
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  int s = 0;
  for (; s + 8 <= S; s += 8) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = __ldg(reinterpret_cast<const float4*>(part + (int64_t)(s + u) * n + e));
#pragma unroll
    for (int u = 0; u < 8; ++u) { a0 += (double)v[u].x; a1 += (double)v[u].y; a2 += (double)v[u].z; a3 += (double)v[u].w; }
  }
  for (; s < S; ++s) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(part + (int64_t)s * n + e));
    a0 += (double)v.x; a1 += (double)v.y; a2 += (double)v.z; a3 += (double)v.w;
  }
  float b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
  for (int k = 0; k < dcb; ++k) {
    const float c = __ldg(cb + (int64_t)b * dcb + k);
    const float4 p = __ldg(reinterpret_cast<const float4*>(Pb + (int64_t)k * d + j));
    b0 = fmaf(c, p.x, b0); b1 = fmaf(c, p.y, b1); b2 = fmaf(c, p.z, b2); b3 = fmaf(c, p.w, b3);
  }
  float4 o;
  o.x = ((float)a0 + b0) * drop_factor(keep, inv_keep, thr, seed, (uint64_t)e);
  o.y = ((float)a1 + b1) * drop_factor(keep, inv_keep, thr, seed, (uint64_t)e + 1);
  o.z = ((float)a2 + b2) * drop_factor(keep, inv_keep, thr, seed, (uint64_t)e + 2);
  o.w = ((float)a3 + b3) * drop_factor(keep, inv_keep, thr, seed, (uint64_t)e + 3);
  *reinterpret_cast<float4*>(y + e) = o;
}

// ---------------------------------------------------------------- backward: T kernel -> df, dc partials
__global__ void __launch_bounds__(THREADS) cpg_bwd_T_kernel(const float* __restrict__ c, const float* __restrict__ f,
                                                            const float* __restrict__ P,
                                                            const float* __restrict__ dy, int B, int dc, int F, int d,
                                                            float* __restrict__ df, float* __restrict__ dc_part) {
  pdl_enter();
  __shared__ Smem sm;
  int n0 = blockIdx.x * BN;  // feature tile
  int m0 = blockIdx.y * BM;  // batch tile
  float dfacc[8][8];
  zero_acc(dfacc);
  int kt = (d + BK - 1) / BK;
  for (int kq = 0; kq < dc; ++kq) {
    SrcK A{dy, d, B, d};
    SrcK Bs{P + (int64_t)kq * F * d, d, F, d};
    float acc[8][8];
    zero_acc(acc);
    mainloop(A, Bs, m0, n0, 0, kt, acc, sm);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int b = m0 + mt_row(i);
      float ck = (b < B) ? __ldg(c + (int64_t)b * dc + kq) : 0.f;
      float rp = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        int col = n0 + mt_col(j);
        float fv = (b < B && col < F) ? __ldg(f + (int64_t)b * F + col) : 0.f;
        dfacc[i][j] = fmaf(ck, acc[i][j], dfacc[i][j]);
        rp = fmaf(fv, acc[i][j], rp);
      }
      // reduce over the 16 threads (same half-warp) that share this row
      rp += __shfl_xor_sync(0xffffffffu, rp, 8);
      rp += __shfl_xor_sync(0xffffffffu, rp, 4);
      rp += __shfl_xor_sync(0xffffffffu, rp, 2);
      rp += __shfl_xor_sync(0xffffffffu, rp, 1);
      if ((threadIdx.x & 15) == 0 && b < B) dc_part[((int64_t)blockIdx.x * B + b) * dc + kq] = rp;
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int b = m0 + mt_row(i);
    if (b >= B) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int col = n0 + mt_col(j);
      if (col < F) df[(int64_t)b * F + col] = dfacc[i][j];
    }
  }
}

// dP[kq][i][j] = sum_b f[b,i] c[b,kq] dy[b,j]
__global__ void __launch_bounds__(THREADS) cpg_bwd_dP_kernel(const float* __restrict__ c, const float* __restrict__ f,
                                                             const float* __restrict__ dy, int B, int dc, int F,
                                                             int d, float* __restrict__ dP) {
  pdl_enter();
  __shared__ Smem sm;
  int n0 = blockIdx.x * BN;  // output-dim tile
  int m0 = blockIdx.y * BM;  // feature tile
  int kq = blockIdx.z;
  SrcMN A{f, F, F, B};
  ScaledMN Bs{dy, c, d, d, B, dc, kq};
  float acc[8][8];
  zero_acc(acc);
  mainloop(A, Bs, m0, n0, 0, (B + BK - 1) / BK, acc, sm);
  float* o = dP + (int64_t)kq * F * d;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int row = m0 + mt_row(i);
    if (row >= F) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int col = n0 + mt_col(j);
      if (col < d) o[(int64_t)row * d + col] = acc[i][j];
    }
  }
}

// ---------------------------------------------------------------- bias-generator gradients (tiny: dcb, d <= a few hundred)
// dPb[k, j] = sum_b cb[b,k] dy[b,j] : block = (k, 32-column slab), 8 batch lanes, fixed-order combine
__global__ void __launch_bounds__(256) cpg_dPb_kernel(const float* __restrict__ cb, const float* __restrict__ dy,
                                                      int B, int d, int dcb, float* __restrict__ dPb) {
  pdl_enter();
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int k = blockIdx.y, j = blockIdx.x * 32 + tx;
  float acc = 0.f;
  if (j < d)
    for (int b = ty; b < B; b += 8) acc = fmaf(__ldg(cb + (int64_t)b * dcb + k), __ldg(dy + (int64_t)b * d + j), acc);
  red[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && j < d) {
    float t = red[0][tx];
#pragma unroll
    for (int r = 1; r < 8; ++r) t += red[r][tx];
    dPb[(int64_t)k * d + j] = t;
  }
}
// dcb[b, k] = sum_j dy[b,j] Pb[k,j] : one warp per (b, k)
__global__ void __launch_bounds__(256) cpg_dcb_kernel(const float* __restrict__ dy, const float* __restrict__ Pb, int B,
                                                      int d, int dcb, float* __restrict__ dcb_out, int accumulate) {
  pdl_enter();
  int w = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (w >= B * dcb) return;
  int b = w / dcb, k = w - b * dcb;
  float acc = 0.f;
  for (int j = lane; j < d; j += 32) acc = fmaf(__ldg(dy + (int64_t)b * d + j), __ldg(Pb + (int64_t)k * d + j), acc);
  acc = warp_sum(acc);
  if (lane == 0) dcb_out[w] = accumulate ? dcb_out[w] + acc : acc;
}

// ---------------------------------------------------------------- plain sgemm
template <class SA, class SB>
__global__ void __launch_bounds__(THREADS) sgemm_kernel(SA A, SB Bs, int M, int N, int K, float* __restrict__ C,
                                                        int ldc, int accumulate) {
  pdl_enter();
  __shared__ Smem sm;
  int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
  float acc[8][8];
  zero_acc(acc);
  mainloop(A, Bs, m0, n0, 0, (K + BK - 1) / BK, acc, sm);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int r = m0 + mt_row(i);
    if (r >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int col = n0 + mt_col(j);
      if (col < N) {
        float* p = C + (int64_t)r * ldc + col;
        *p = accumulate ? *p + acc[i][j] : acc[i][j];
      }
    }
  }
}

struct CpgLayout {
  int splits, tiles_per_split;
  size_t total;
};
static CpgLayout cpg_fwd_layout(int B, int dc, int F, int d) {
  CpgLayout L;
  int tiles_mn = ceil_div(d, BN) * ceil_div(B, BM);
  int T = dc * ceil_div(F, BK);
  int splits = (2 * 148 + tiles_mn - 1) / tiles_mn;
  if (splits > T) splits = T;
  if (splits < 1) splits = 1;
  L.tiles_per_split = (T + splits - 1) / splits;
  L.splits = (T + L.tiles_per_split - 1) / L.tiles_per_split;
  L.total = align_up((size_t)L.splits * B * d * sizeof(float), 256);
  return L;
}
}  // namespace coper

using namespace coper;

extern "C" {

int coper_sgemm(int transA, int transB, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                float* C, int ldc, int accumulate, coper_stream_t stream) {
  COPER_CHECK_ARG(A && B && C && M > 0 && N > 0 && K > 0 && lda > 0 && ldb > 0 && ldc >= N);
  dim3 grid(ceil_div(N, BN), ceil_div(M, BM));
  cudaStream_t st = as_stream(stream);
  // operand A(m,k): !transA -> A[m*lda+k] (K-contig); transA -> A[k*lda+m] (MN-contig)
  // operand B(k,n): !transB -> B[k*ldb+n] (MN-contig); transB -> B[n*ldb+k] (K-contig)
  if (!transA && !transB)
    launch_pdl(sgemm_kernel<SrcK, SrcMN>, grid, THREADS, 0, st, SrcK{A, lda, M, K}, SrcMN{B, ldb, N, K}, M, N, K, C, ldc,
               accumulate);
  else if (!transA && transB)
    launch_pdl(sgemm_kernel<SrcK, SrcK>, grid, THREADS, 0, st, SrcK{A, lda, M, K}, SrcK{B, ldb, N, K}, M, N, K, C, ldc,
               accumulate);
  else if (transA && !transB)
    launch_pdl(sgemm_kernel<SrcMN, SrcMN>, grid, THREADS, 0, st, SrcMN{A, lda, M, K}, SrcMN{B, ldb, N, K}, M, N, K, C, ldc,
               accumulate);
  else
    launch_pdl(sgemm_kernel<SrcMN, SrcK>, grid, THREADS, 0, st, SrcMN{A, lda, M, K}, SrcK{B, ldb, N, K}, M, N, K, C, ldc,
               accumulate);
  return check_launch();
}

// The tcgen05 kernels cover F % 32 == 0 and d <= 256 (every shipped configuration); any other shape runs on the
// exact-fp32 CUDA-core engine below whatever `prec` asks for (more accurate, slower - never a host fallback).
static inline bool cpg_on_tensor_pipe(int F, int d, int prec) {
  return (prec == COPER_PREC_BF16 || prec == COPER_PREC_TF32X3 || prec == COPER_PREC_FP16X3) && F % 32 == 0 && d <= 256;
}

size_t coper_cpg_fc_fwd_workspace_bytes(int B, int dc, int F, int d, int prec) {
  if (cpg_on_tensor_pipe(F, d, prec)) return umma_cpg_fwd_workspace_bytes(B, dc, F, d, prec);
  return cpg_fwd_layout(B, dc, F, d).total;
}

int coper_cpg_fc_fwd(const float* c, const float* f, const float* P, const void* P_prepared, const float* cb,
                     const float* Pb, int B, int dc, int F, int d, int dcb, float keep_out, const uint64_t* seed_dev,
                     uint64_t salt_out, float* y, void* workspace, size_t workspace_bytes, int prec,
                     coper_stream_t stream) {
  COPER_CHECK_ARG(c && f && P && cb && Pb && y && workspace && B > 0 && dc > 0 && F > 0 && d > 0 && dcb > 0);
  COPER_CHECK_ARG(keep_out > 0.f);
  cudaStream_t st = as_stream(stream);
  float* part = nullptr;
  int n_slabs = 0;
  int rc;
  if (cpg_on_tensor_pipe(F, d, prec)) {
    if ((rc = umma_cpg_fwd_partials(c, f, P, P_prepared, B, dc, F, d, workspace, workspace_bytes, prec, st, &part, &n_slabs)))
      return rc;
  } else if (prec >= COPER_PREC_FP32 && prec <= COPER_PREC_FP16X3) {
    CpgLayout L = cpg_fwd_layout(B, dc, F, d);
    if (workspace_bytes < L.total) return COPER_ERR_WORKSPACE;
    part = static_cast<float*>(workspace);
    n_slabs = L.splits;
    dim3 grid(ceil_div(d, BN), ceil_div(B, BM), L.splits);
    launch_pdl(cpg_fwd_kernel, grid, THREADS, 0, st, c, f, P, B, dc, F, d, L.tiles_per_split, part);
    if ((rc = check_launch())) return rc;
  } else {
    return COPER_ERR_UNSUPPORTED;
  }
  int64_t n = (int64_t)B * d;
  const bool vec = (d & 3) == 0 && ((reinterpret_cast<uintptr_t>(part) | reinterpret_cast<uintptr_t>(Pb) |
                                     reinterpret_cast<uintptr_t>(y)) & 15) == 0;
  if (vec)
    launch_pdl(cpg_fwd_finalize_kernel4, (unsigned)((n / 4 + 127) / 128), 128, 0, st, part, n_slabs, cb, Pb, B, d,
               dcb, keep_out, 1.0f / keep_out, keep_threshold(keep_out), seed_dev, salt_out, y);
  else
    launch_pdl(cpg_fwd_finalize_kernel, (unsigned)((n + 255) / 256), 256, 0, st, part, n_slabs, cb, Pb, B, d, dcb,
               keep_out, 1.0f / keep_out, keep_threshold(keep_out), seed_dev, salt_out, y);
  return check_launch();
}

size_t coper_cpg_fc_bwd_workspace_bytes(int B, int dc, int F, int d, int prec) {
  if (cpg_on_tensor_pipe(F, d, prec)) return umma_cpg_bwd_workspace_bytes(B, dc, F, d, prec);
  return align_up((size_t)ceil_div(F, BN) * B * dc * sizeof(float), 256);
}

int coper_cpg_fc_bwd(const float* c, const float* f, const float* P, const void* P_prepared, const float* cb,
                     const float* Pb, const float* dy, int B, int dc, int F, int d, int dcb, float* dP, float* dPb, float* df,
                     float* dc_out, float* dcb_out, void* workspace, size_t workspace_bytes, int prec,
                     int flags, coper_stream_t stream) {
  COPER_CHECK_ARG(c && f && P && cb && Pb && dy && dP && dPb && df && dc_out && dcb_out && workspace);
  COPER_CHECK_ARG(B > 0 && dc > 0 && F > 0 && d > 0 && dcb > 0);
  const bool inputs = !(flags & COPER_CPG_BWD_WEIGHT_GRADS_ONLY), weights = !(flags & COPER_CPG_BWD_INPUT_GRADS_ONLY);
  COPER_CHECK_ARG(inputs || weights);
  if (workspace_bytes < coper_cpg_fc_bwd_workspace_bytes(B, dc, F, d, prec)) return COPER_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  int rc;
  if (cpg_on_tensor_pipe(F, d, prec)) {
    if ((rc = umma_cpg_bwd(c, f, P, P_prepared, dy, B, dc, F, d, dP, df, dc_out, workspace, workspace_bytes, prec,
                           flags, st)))
      return rc;
  } else if (prec >= COPER_PREC_FP32 && prec <= COPER_PREC_FP16X3) {
    if (inputs) {
      float* dc_part = static_cast<float*>(workspace);
      int ftiles = ceil_div(F, BN);
      launch_pdl(cpg_bwd_T_kernel, dim3(ftiles, ceil_div(B, BM)), THREADS, 0, st, c, f, P, dy, B, dc, F, d, df,
                 dc_part);
      if ((rc = check_launch())) return rc;
      if ((rc = coper_reduce_partials(dc_part, ftiles, (int64_t)B * dc, 1.0f, 0, dc_out, stream))) return rc;
    }
    if (weights) {
      launch_pdl(cpg_bwd_dP_kernel, dim3(ceil_div(d, BN), ceil_div(F, BM), dc), THREADS, 0, st, c, f, dy, B, dc, F,
                 d, dP);
      if ((rc = check_launch())) return rc;
    }
  } else {
    return COPER_ERR_UNSUPPORTED;
  }
  // dPb [dcb, d] = cb^T . dy ;  dcb [B, dcb] = dy . Pb^T
  if (weights) {
    launch_pdl(cpg_dPb_kernel, dim3(ceil_div(d, 32), dcb), 256, 0, st, cb, dy, B, d, dcb, dPb);
    if ((rc = check_launch())) return rc;
  }
  if (inputs) {
    launch_pdl(cpg_dcb_kernel, ceil_div((int64_t)B * dcb * 32, 256), 256, 0, st, dy, Pb, B, d, dcb, dcb_out,
               (flags & COPER_CPG_BWD_DCB_ACCUMULATE) ? 1 : 0);
    if ((rc = check_launch())) return rc;
  }
  return COPER_OK;
}

}  // extern "C"
