// a3 + a6 (K2 + K3) on the tensor pipe: fused contextual-parameter generate-and-apply and its backward
// (models.py:70-73, 412, 198) for COPER_PREC_BF16 / COPER_PREC_TF32X3.
//
// The Khatri-Rao contraction y = (c (x) f) . P^ is evaluated as a GROUPED GEMM over the context index k:
//     y[b,:] = sum_k c[b,k] * ( f[b,:] . P[k] ),        P[k] = P viewed [F, d]
// Each group's product f.P[k] runs on tcgen05 (A = f K-major, B = P[k] MN-major, both TMA-fed, fp32 accumulators
// in TMEM); the per-row context scale c[b,k] is applied in fp32 while the epilogue warps accumulate the group
// tiles in registers, so neither the per-query weights [B,F,d] nor the Khatri-Rao operand [B, dc*F] ever exist.
// F is split across CTAs (split-K) and the slabs are reduced in a fixed order (deterministic).
//
// Backward:
//   T_k = dy . P[k]^T  (per group, never stored)   df = sum_k c[:,k] * T_k     dc[:,k] = rowsum(f * T_k)
//   dP[k] = f^T . (c[:,k] * dy)                     (grouped GEMM over k with a pre-scaled dy operand)
#include "umma_gemm.cuh"

namespace coper {
using namespace umma;

// ------------------------------------------------------------------------------------------ forward
struct CpgFwdEpi : EpiBase {
  static constexpr bool kAccumulate = true;
  const float* c;       // [M, dc]
  int dc;
  float* out;           // slabs [splits][M, ld]
  long long ld, split_stride;
  __device__ __forceinline__ float group_scale(const GemmProblem& p, const TileCoord& t, int row) const {
    return row < p.M ? __ldg(c + (long long)row * dc + t.group) : 0.f;
  }
  __device__ __forceinline__ void chunk(const GemmProblem& p, const TileCoord& t, int row, int col,
                                        const uint32_t (&r)[32], int) const {
    if (row >= p.M) return;
    float* o = out + t.split * split_stride + (long long)row * ld + col;
    if (col + 31 < p.N && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(o + j) = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                                        __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (col + j < p.N) o[j] = __uint_as_float(r[j]);
    }
  }
};

// N = d <= 256 in one tile.  tf32x3: chains cut every 4 k-blocks (see umma_gemm.cuh)
// fp16x3: 64 k-elements per k-block (two fp16 planes) -> the same chain length is 2 k-blocks
// f does not depend on the context group, but a resident f (RES_A_KB) made this kernel 1-4 us SLOWER at every
// benchmark shape (B200, DESIGN §4.7): both operands stream.
template <int PREC>
using CpgFwdCfg = GemmCfg<PREC, 256, (PREC == PREC_BF16 ? 4 : 2), 8, false, true,
                          (PREC == PREC_BF16 ? 0 : PREC == PREC_FP16X3 ? 2 : 4)>;

struct CpgFwdPlan {
  GemmProblem p;
  size_t off_f, off_P, off_slabs, total;
};
static CpgFwdPlan cpg_fwd_plan(int B, int dc, int F, int d, int prec) {
  CpgFwdPlan L;
  GemmProblem p{};
  p.M = B; p.N = d; p.K = F; p.groups = dc; p.groups_inner = 1;
  p.a_group_mn = 0; p.a_group_k = 0; p.b_group_mn = 0; p.b_group_k = F;
  if (prec == COPER_PREC_BF16) plan_gemm<CpgFwdCfg<PREC_BF16>>(p, true);
  else if (prec == COPER_PREC_FP16X3) plan_gemm<CpgFwdCfg<PREC_FP16X3>>(p, true);
  else plan_gemm<CpgFwdCfg<PREC_TF32X3>>(p, true);
  L.p = p;
  size_t o = 0;
  L.off_f = o; o = align_up(o + prepared_bytes(B, F, prec), 256);
  L.off_P = o; o = align_up(o + prepared_bytes((int64_t)dc * F, d, prec), 256);
  L.off_slabs = o; o = align_up(o + (size_t)p.splits * B * d * sizeof(float), 256);
  L.total = o;
  return L;
}

// ------------------------------------------------------------------------------------------ backward: T kernel
// one 32-column chunk per epilogue warp (BLOCK_N = 128, 16 epilogue warps): the f tile and the df accumulators
// stay in registers across the group loop
struct CpgBwdTEpi : EpiBase {
  static constexpr bool kAccumulate = true;
  const float* c;       // [M, dc]
  const float* f;       // [M, F]
  int dc;
  float* df;            // [M, F]
  float* dc_part;       // [n_tiles * col_groups][M, dc]
  float freg[32];
  float fsum;
  __device__ __forceinline__ void tile_begin(const GemmProblem& p, const TileCoord&, int row, int col0) {
    fsum = 0.f;
    if (row < p.M && col0 < p.N) {           // p.N = F is a multiple of 32
      const float4* src = reinterpret_cast<const float4*>(f + (long long)row * p.N + col0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 v = __ldg(src + j);
        freg[4 * j] = v.x; freg[4 * j + 1] = v.y; freg[4 * j + 2] = v.z; freg[4 * j + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) freg[j] = 0.f;
    }
  }
  __device__ __forceinline__ float group_scale(const GemmProblem& p, const TileCoord& t, int row) const {
    return row < p.M ? __ldg(c + (long long)row * dc + t.group) : 0.f;
  }
  __device__ __forceinline__ void group_vals(const GemmProblem&, const TileCoord&, int, int, const uint32_t (&v)[16],
                                             int half_idx) {
#pragma unroll
    for (int j = 0; j < 16; ++j) fsum = fmaf(freg[(half_idx & 1) * 16 + j], __uint_as_float(v[j]), fsum);
  }
  __device__ __forceinline__ void group_done(const GemmProblem& p, const TileCoord& t, int row, int col_group,
                                             int col_groups) {
    if (row < p.M)
      dc_part[((long long)(t.n_blk * col_groups + col_group) * p.M + row) * dc + t.group] = fsum;
    fsum = 0.f;
  }
  __device__ __forceinline__ void chunk(const GemmProblem& p, const TileCoord&, int row, int col,
                                        const uint32_t (&r)[32], int) const {
    if (row >= p.M) return;
    float4* o = reinterpret_cast<float4*>(df + (long long)row * p.N + col);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      o[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                         __uint_as_float(r[4 * j + 3]));
  }
};
constexpr int kBwdTEpiWarps = 16;
constexpr int kBwdTBlockN = 128;
// The dy tile does not depend on the context group: bf16 / fp16x3 keep its whole K extent (d <= 256: 4 k-blocks) resident
// (64 / 128 KB) and stream only P[k] (8 x 16 KB / 3 x 32 KB stages).  tf32x3 (d = 200: 7 k-blocks x 2 planes x 16 KB)
// does not fit and streams both.
template <int PREC>
using CpgBwdTCfg = GemmCfg<PREC, kBwdTBlockN, (PREC == PREC_BF16 ? 8 : 3), kBwdTEpiWarps, false, false, 0, 0,
                           (PREC == PREC_TF32X3 ? 0 : 4)>;

// fp16x3: max |dy[b,j] * c[b,g]| = max_b (max_j |dy[b,:]| * max_g |c[b,:]|); one warp per row, result in the trailer's
// max word (zeroed before the launch)
__global__ void absmax_scaled_kernel(const float* __restrict__ dy, const float* __restrict__ c, int B, int d, int dc,
                                     uint32_t* __restrict__ trailer) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  for (int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); b < B; b += gridDim.x * (blockDim.x >> 5)) {
    float my = 0.f, mc = 0.f;
    for (int j = lane; j < d; j += 32) my = fmaxf(my, fabsf(__ldg(dy + (int64_t)b * d + j)));
    for (int g = lane; g < dc; g += 32) mc = fmaxf(mc, fabsf(__ldg(c + (int64_t)b * dc + g)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      my = fmaxf(my, __shfl_xor_sync(0xffffffffu, my, o));
      mc = fmaxf(mc, __shfl_xor_sync(0xffffffffu, mc, o));
    }
    if (lane == 0) trailer_max(trailer + kTrMax, my * mc);
  }
}
// dyc[(g*B + b), j] = dy[b,j] * c[b,g] in prepared operand form
__global__ void prepare_scaled_kernel(const float* __restrict__ dy, const float* __restrict__ c, int B, int d, int dc,
                                      int64_t ldp, int prec, void* __restrict__ dst, uint32_t* __restrict__ trailer) {
  pdl_enter();
  int64_t n = (int64_t)dc * B * ldp;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  float sc = 1.0f;
  if (prec == COPER_PREC_FP16X3) sc = fp16x3_publish(trailer, trailer[kTrMax], -1, blockIdx.x == 0 && threadIdx.x == 0);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
    int64_t r = e / ldp;
    int j = (int)(e - r * ldp);
    int g = (int)(r / B), b = (int)(r - (int64_t)g * B);
    float x = j < d ? __ldg(dy + (int64_t)b * d + j) * __ldg(c + (int64_t)b * dc + g) : 0.f;
    emit_prepared(prec, dst, n, e, x, sc);
  }
}

// fp16x3, one batch (B <= a few thousand rows): both backward operands - dy and dy scaled by the context - in ONE launch
// instead of prepare(dy) + absmax_scaled + prepare_scaled.  Every block reduces its rows' maxima into dy's trailer
// (kTrMax: max |dy|, kTrMax2: max |dy| * max |c| per row) and waits at the grid barrier, then the blocks emit the planes.
// tr_dy words 0..7 are zero on entry.  Same maxima, same exponent rule, same rounding as the three kernels it replaces
// -> same bits.
__global__ void __launch_bounds__(256) cpg_bwd_prepare_fp16x3_kernel(const float* __restrict__ dy,
                                                                     const float* __restrict__ c, int B, int d, int dc,
                                                                     int64_t ldp, __half* __restrict__ dyp,
                                                                     __half* __restrict__ dycp,
                                                                     uint32_t* __restrict__ tr_dy,
                                                                     uint32_t* __restrict__ tr_dyc) {
  pdl_enter();
  __shared__ float wmax[2][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float m_dy = 0.f, m_dyc = 0.f;
  for (int b = blockIdx.x * 8 + warp; b < B; b += gridDim.x * 8) {
    float my = 0.f, mc = 0.f;
    for (int j = lane; j < d; j += 32) my = fmaxf(my, fabsf(__ldg(dy + (int64_t)b * d + j)));
    for (int g = lane; g < dc; g += 32) mc = fmaxf(mc, fabsf(__ldg(c + (int64_t)b * dc + g)));
    my = warp_max(my);
    mc = warp_max(mc);
    m_dy = fmaxf(m_dy, my);
    m_dyc = fmaxf(m_dyc, my * mc);
  }
  if (lane == 0) { wmax[0][warp] = m_dy; wmax[1][warp] = m_dyc; }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < 8; ++w) { m_dy = fmaxf(m_dy, wmax[0][w]); m_dyc = fmaxf(m_dyc, wmax[1][w]); }
    trailer_max(tr_dy + kTrMax, m_dy);
    trailer_max(tr_dy + kTrMax2, m_dyc);
    grid_arrive_wait(tr_dy + kTrArrive);
  }
  __syncthreads();
  const bool leader = blockIdx.x == 0 && threadIdx.x == 0;
  const float sc_dy = fp16x3_publish(tr_dy, *reinterpret_cast<volatile uint32_t*>(tr_dy + kTrMax), kTrRunMax, leader);
  const float sc_dyc = fp16x3_publish(tr_dyc, *reinterpret_cast<volatile uint32_t*>(tr_dy + kTrMax2), kTrMax, leader);
  // work unit = one 8-column group of one row of plane-set p (p = 0: dy, p = 1 + g: dy * c[:, g])
  const int gpr = (int)(ldp / 8);
  const int64_t per = (int64_t)B * gpr, units = per * (1 + dc);
  for (int64_t u = (int64_t)blockIdx.x * 256 + threadIdx.x; u < units; u += (int64_t)gridDim.x * 256) {
    const int p = (int)(u / per);
    const int64_t v = u - (int64_t)p * per;
    const int b = (int)(v / gpr), c0 = (int)(v - (int64_t)b * gpr) * 8;
    const float cs = p == 0 ? 1.0f : __ldg(c + (int64_t)b * dc + (p - 1));
    float x[8];
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
      const int j = c0 + k;
      float x0 = j < d ? __ldg(dy + (int64_t)b * d + j) : 0.f, x1 = j + 1 < d ? __ldg(dy + (int64_t)b * d + j + 1) : 0.f;
      if (p != 0) { x0 = j < d ? x0 * cs : 0.f; x1 = j + 1 < d ? x1 * cs : 0.f; }
      x[k] = x0;
      x[k + 1] = x1;
    }
    emit_prepared_vec<COPER_PREC_FP16X3, 8>(p == 0 ? dyp : dycp, p == 0 ? (int64_t)B * ldp : (int64_t)dc * B * ldp,
                                            (p == 0 ? v : (int64_t)(p - 1) * per + v) * 8, x, p == 0 ? sc_dy : sc_dyc);
  }
}

struct CpgBwdPlan {
  size_t off_f, off_P, off_dy, off_dyc, off_dcpart, total;
  int dc_slabs;
};
static CpgBwdPlan cpg_bwd_plan(int B, int dc, int F, int d, int prec) {
  CpgBwdPlan L;
  size_t o = 0;
  // [f][P] first, at the same offsets as the forward plan (so a backward call may reuse them)
  L.off_f = o; o = align_up(o + prepared_bytes(B, F, prec), 256);
  L.off_P = o; o = align_up(o + prepared_bytes((int64_t)dc * F, d, prec), 256);
  L.off_dy = o; o = align_up(o + prepared_bytes(B, d, prec), 256);
  L.off_dyc = o; o = align_up(o + prepared_bytes((int64_t)dc * B, d, prec), 256);
  L.dc_slabs = ((F + kBwdTBlockN - 1) / kBwdTBlockN) * (kBwdTEpiWarps / 4);
  L.off_dcpart = o; o = align_up(o + (size_t)L.dc_slabs * B * dc * sizeof(float), 256);
  L.total = o;
  return L;
}

size_t umma_cpg_fwd_workspace_bytes(int B, int dc, int F, int d, int prec) { return cpg_fwd_plan(B, dc, F, d, prec).total; }
size_t umma_cpg_bwd_workspace_bytes(int B, int dc, int F, int d, int prec) {
  size_t a = cpg_bwd_plan(B, dc, F, d, prec).total, b = cpg_fwd_plan(B, dc, F, d, prec).total;
  return a > b ? a : b;
}

// Computes the split-K slabs of (c (x) f) . P^ into the workspace; *slabs / *n_slabs describe them.
int umma_cpg_fwd_partials(const float* c, const float* f, const float* P, const void* P_prepared, int B, int dc, int F,
                          int d, void* ws, size_t ws_bytes, int prec, cudaStream_t st, float** slabs, int* n_slabs) {
  if (F % 32 != 0 || d > 256) return COPER_ERR_UNSUPPORTED;
  CpgFwdPlan L = cpg_fwd_plan(B, dc, F, d, prec);
  if (!ws || ws_bytes < L.total) return COPER_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(ws) & 255) return COPER_ERR_INVALID_ARG;
  char* w = static_cast<char*>(ws);
  void* fp = w + L.off_f;
  const void* Pp = P_prepared ? P_prepared : w + L.off_P;
  float* out = reinterpret_cast<float*>(w + L.off_slabs);
  int rc;
  if ((rc = tc_prepare(f, B, F, F, prec, fp, st))) return rc;
  if (!P_prepared && (rc = tc_prepare(P, (int64_t)dc * F, d, d, prec, w + L.off_P, st))) return rc;
  CpgFwdEpi epi;
  epi.c = c; epi.dc = dc; epi.out = out; epi.ld = d; epi.split_stride = (long long)B * d;
  TcOperand A = tc_operand(fp, B, F, prec), Bo = tc_operand(Pp, (int64_t)dc * F, d, prec);
  if (prec == COPER_PREC_BF16) rc = launch_gemm<CpgFwdCfg<PREC_BF16>, CpgFwdEpi>(A, Bo, L.p, epi, st);
  else if (prec == COPER_PREC_FP16X3) rc = launch_gemm<CpgFwdCfg<PREC_FP16X3>, CpgFwdEpi>(A, Bo, L.p, epi, st);
  else rc = launch_gemm<CpgFwdCfg<PREC_TF32X3>, CpgFwdEpi>(A, Bo, L.p, epi, st);
  *slabs = out;
  *n_slabs = L.p.splits;
  return rc;
}

// df, dc_out, dP through the tensor pipe.  flags: COPER_CPG_BWD_* (include/coper.h).  REUSE_FWD: the workspace still
// holds the prepared f and P operands written by umma_cpg_fwd_partials for the same (f, P).
int umma_cpg_bwd(const float* c, const float* f, const float* P, const void* P_prepared, const float* dy, int B, int dc,
                 int F, int d, float* dP, float* df, float* dc_out, void* ws, size_t ws_bytes, int prec,
                 int flags, cudaStream_t st) {
  if (F % 32 != 0 || d > 256) return COPER_ERR_UNSUPPORTED;
  const bool inputs = !(flags & COPER_CPG_BWD_WEIGHT_GRADS_ONLY), weights = !(flags & COPER_CPG_BWD_INPUT_GRADS_ONLY);
  CpgBwdPlan L = cpg_bwd_plan(B, dc, F, d, prec);
  if (!ws || ws_bytes < L.total) return COPER_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(ws) & 255) return COPER_ERR_INVALID_ARG;
  char* w = static_cast<char*>(ws);
  void* fp = w + L.off_f;
  const void* Pp = P_prepared ? P_prepared : w + L.off_P;
  void* dyp = w + L.off_dy;
  void* dycp = w + L.off_dyc;
  float* dc_part = reinterpret_cast<float*>(w + L.off_dcpart);
  int rc = COPER_OK;
  if (inputs) {
    // ---- operands: f, P (unless the forward call left them), dy, and dy pre-scaled by the context (for dP)
    if (!(flags & COPER_CPG_BWD_REUSE_FWD)) {
      if ((rc = tc_prepare(f, B, F, F, prec, fp, st))) return rc;
      if (!P_prepared && (rc = tc_prepare(P, (int64_t)dc * F, d, d, prec, w + L.off_P, st))) return rc;
    }
    int64_t ldp = prepared_ld(d, prec);
    int64_t n = (int64_t)dc * B * ldp;
    if (prec == COPER_PREC_FP16X3 && n <= ((int64_t)8 << 20)) {
      // one launch for both operands (grid barrier: <= 2 co-resident blocks per SM)
      uint32_t* tr_dy = fp16x3_trailer(dyp, B, d);
      uint32_t* tr_dyc = fp16x3_trailer(dycp, (int64_t)dc * B, d);
      if ((rc = check_cuda(cudaMemsetAsync(tr_dy, 0, 32, st)))) return rc;
      const int64_t want = ((int64_t)(1 + dc) * B * (ldp / 8) + 256 * 4 - 1) / (256 * 4);
      int g = (int)(want < (int64_t)sm_count() * 2 ? want : (int64_t)sm_count() * 2);
      if (g < 1) g = 1;
      launch_pdl(cpg_bwd_prepare_fp16x3_kernel, g, 256, 0, st, dy, c, B, d, dc, ldp, static_cast<__half*>(dyp),
                 static_cast<__half*>(dycp), tr_dy, tr_dyc);
      if ((rc = check_launch())) return rc;
    } else {
      if ((rc = tc_prepare(dy, B, d, d, prec, dyp, st))) return rc;
      int grid = (int)((n + 255) / 256 < sm_count() * 8 ? (n + 255) / 256 : sm_count() * 8);
      uint32_t* trailer = nullptr;
      if (prec == COPER_PREC_FP16X3) {
        trailer = fp16x3_trailer(dycp, (int64_t)dc * B, d);
        if ((rc = check_cuda(cudaMemsetAsync(trailer, 0, 8, st)))) return rc;
        launch_pdl(absmax_scaled_kernel, (B + 7) / 8, 256, 0, st, dy, c, B, d, dc, trailer);
        if ((rc = check_launch())) return rc;
      }
      launch_pdl(prepare_scaled_kernel, grid, 256, 0, st, dy, c, B, d, dc, ldp, prec, dycp, trailer);
      if ((rc = check_launch())) return rc;
    }
    // ---- T kernel: df, dc partials
    GemmProblem p{};
    p.M = B; p.N = F; p.K = d; p.groups = dc; p.groups_inner = 1;
    p.a_group_mn = 0; p.a_group_k = 0; p.b_group_mn = F; p.b_group_k = 0;
    CpgBwdTEpi epi;
    epi.c = c; epi.f = f; epi.dc = dc; epi.df = df; epi.dc_part = dc_part; epi.fsum = 0.f;
    TcOperand A = tc_operand(dyp, B, d, prec), Bo = tc_operand(Pp, (int64_t)dc * F, d, prec);
    if (prec == COPER_PREC_BF16) {
      plan_gemm<CpgBwdTCfg<PREC_BF16>>(p, false);
      rc = launch_gemm<CpgBwdTCfg<PREC_BF16>, CpgBwdTEpi>(A, Bo, p, epi, st);
    } else if (prec == COPER_PREC_FP16X3) {
      plan_gemm<CpgBwdTCfg<PREC_FP16X3>>(p, false);
      rc = launch_gemm<CpgBwdTCfg<PREC_FP16X3>, CpgBwdTEpi>(A, Bo, p, epi, st);
    } else {
      plan_gemm<CpgBwdTCfg<PREC_TF32X3>>(p, false);
      rc = launch_gemm<CpgBwdTCfg<PREC_TF32X3>, CpgBwdTEpi>(A, Bo, p, epi, st);
    }
    if (rc) return rc;
    if ((rc = coper_reduce_partials(dc_part, L.dc_slabs, (int64_t)B * dc, 1.0f, 0, dc_out, (coper_stream_t)st)))
      return rc;
  }
  // ---- dP[k] = f^T . (c[:,k] * dy): A = f stored [K=B, M=F] (MN-major), B = dyc stored [dc*B, d] (MN-major)
  if (weights) {
    GemmProblem p{};
    p.M = F; p.N = d; p.K = B; p.groups = dc; p.groups_inner = 0;
    p.a_group_mn = 0; p.a_group_k = 0; p.b_group_mn = 0; p.b_group_k = B;
    StoreEpi epi = make_store_epi(dP, d, (long long)F * d, 0);
    rc = tc_gemm_store(prec, true, true, tc_operand(fp, B, F, prec), tc_operand(dycp, (int64_t)dc * B, d, prec), p,
                       false, epi, st);
  }
  return rc;
}

}  // namespace coper
