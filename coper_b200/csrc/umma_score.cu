// a7 / K6 on the tensor pipe: 1-N scorer logits S = q.E^T + bias (models.py:433-437) as a persistent,
// warp-specialised tcgen05 GEMM: TMA-fed 128B-swizzled operand ring, fp32 accumulators double-buffered in
// TMEM, bias add fused into the TMEM->register epilogue.  M = queries (TMEM lanes), N = entities (TMEM
// columns), K = d.  Two arithmetic modes (include/coper.h): COPER_PREC_BF16 and COPER_PREC_TF32X3.
//
// Operands are consumed in "prepared" form (coper_prepare_operand, format: operand.cuh) - the entity table is prepared
// once per evaluation pass / per optimizer step, not per call.
#include "umma_gemm.cuh"

namespace coper {
using namespace umma;

// ------------------------------------------------------------------------------------------ operand preparation
// (format: operand.cuh)  block = (64 column lanes) x (4 rows); grid-stride over rows; each lane converts VEC consecutive
// columns per pass (VEC = 8 bf16 / fp16x3, 4 tf32 -> one 16-byte store per plane); no integer division anywhere.
// fp16x3: max |x| is already in the trailer (absmax_kernel).
template <int PREC>
__global__ void __launch_bounds__(256) prepare_kernel(const float* __restrict__ src, int64_t rows, int cols,
                                                      int64_t ld_src, void* __restrict__ dst, int64_t ldp,
                                                      uint32_t* __restrict__ trailer) {
  pdl_enter();
  constexpr int VEC = PREC == COPER_PREC_TF32X3 ? 4 : 8;
  float sc = 1.0f;
  if (PREC == COPER_PREC_FP16X3) sc = fp16x3_publish(trailer, trailer[kTrMax], kTrRunMax, blockIdx.x == 0 && threadIdx.x == 0);
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  const int nvec = (int)(ldp / VEC);
  const bool vec_src = ((ld_src & 3) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  for (int64_t r = (int64_t)blockIdx.x * 4 + ty; r < rows; r += (int64_t)gridDim.x * 4) {
    const float* srow = src + r * ld_src;
    for (int v = tx; v < nvec; v += 64) {
      const int c0 = v * VEC;
      float x[VEC];
      if (vec_src && c0 + VEC <= cols) {
#pragma unroll
        for (int k = 0; k < VEC; k += 4) {
          float4 t = __ldg(reinterpret_cast<const float4*>(srow + c0 + k));
          x[k] = t.x; x[k + 1] = t.y; x[k + 2] = t.z; x[k + 3] = t.w;
        }
      } else {
#pragma unroll
        for (int k = 0; k < VEC; ++k) x[k] = (c0 + k < cols) ? __ldg(srow + c0 + k) : 0.f;
      }
      emit_prepared_vec<PREC, VEC>(dst, rows * ldp, r * ldp + c0, x, sc);
    }
  }
}

// fp16x3, large operands: max |x| into the trailer, then prepare_kernel<COPER_PREC_FP16X3>
__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ src, int64_t rows, int cols, int64_t ld_src,
                                                     uint32_t* __restrict__ trailer) {
  pdl_enter();
  float m = 0.f;
  if (ld_src == cols) {                                // dense: one flat stream (16-byte loads when aligned)
    const int64_t n = rows * cols;
    if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
      const float4* s4 = reinterpret_cast<const float4*>(src);
      for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n / 4; i += (int64_t)gridDim.x * 256) {
        const float4 v = __ldg(s4 + i);
        m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
      }
      for (int64_t i = (n / 4) * 4 + (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256)
        m = fmaxf(m, fabsf(__ldg(src + i)));
    } else {
      for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256)
        m = fmaxf(m, fabsf(__ldg(src + i)));
    }
  } else {
    for (int64_t r = blockIdx.x; r < rows; r += gridDim.x)
      for (int c = threadIdx.x; c < cols; c += 256) m = fmaxf(m, fabsf(__ldg(src + r * ld_src + c)));
  }
  warp_trailer_max(trailer + kTrMax, m);
}

// Small fp16x3 operands (activations / gradients of one batch: q, f, dy): max |x| and the split in ONE launch.  Every
// block reduces its share of the max into the trailer and waits at the grid barrier, then converts its rows.
__global__ void __launch_bounds__(256) prepare_fp16x3_fused_kernel(const float* __restrict__ src, int64_t rows, int cols,
                                                                   int64_t ld_src, __half* __restrict__ dst, int64_t ldp,
                                                                   uint32_t* __restrict__ trailer) {
  pdl_enter();
  __shared__ float wmax[8];
  // work unit = one 8-column group of one row (ldp / 8 groups per row); consecutive threads take consecutive groups
  const int gpr = (int)(ldp / 8);
  const int64_t units = rows * gpr;
  const bool vec = ((ld_src & 3) == 0) && ((cols & 7) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  auto load8 = [&](int64_t u, float (&x)[8]) {
    const int64_t r = u / gpr;
    const int c0 = (int)(u - r * gpr) * 8;
    const float* p = src + r * ld_src + c0;
    if (vec) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
      x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) x[k] = (c0 + k < cols) ? __ldg(p + k) : 0.f;
    }
  };
  float m = 0.f;
  for (int64_t u = (int64_t)blockIdx.x * 256 + threadIdx.x; u < units; u += (int64_t)gridDim.x * 256) {
    float x[8];
    load8(u, x);
#pragma unroll
    for (int k = 0; k < 8; ++k) m = fmaxf(m, fabsf(x[k]));
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < 8; ++w) m = fmaxf(m, wmax[w]);
    trailer_max(trailer + kTrMax, m);
    grid_arrive_wait(trailer + kTrArrive);
  }
  __syncthreads();
  const uint32_t mbits = *reinterpret_cast<volatile uint32_t*>(trailer + kTrMax);
  const float sc = fp16x3_publish(trailer, mbits, kTrRunMax, blockIdx.x == 0 && threadIdx.x == 0);
  for (int64_t u = (int64_t)blockIdx.x * 256 + threadIdx.x; u < units; u += (int64_t)gridDim.x * 256) {
    float x[8];
    load8(u, x);                                       // second touch of the same addresses: L1 / L2 hits
    emit_prepared_vec<COPER_PREC_FP16X3, 8>(dst, rows * ldp, u * 8, x, sc);        // u * 8 == r * ldp + c0
  }
}

// entity-major scorer kernels: umma_entity.cu
int umma_score1n_fwd_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                              float* scores, int64_t ld, int prec, cudaStream_t st);

size_t umma_score1n_workspace_bytes(int B, int64_t Ns, int d, int prec) {
  return prepared_bytes(B, d, prec) + prepared_bytes(Ns, d, prec) + 256;
}

int tc_prepare(const float* src, int64_t rows, int cols, int64_t ld_src, int prec, void* dst, cudaStream_t st) {
  int64_t ldp = prepared_ld(cols, prec);
  int64_t blocks = (rows + 3) / 4;
  int grid = (int)(blocks < 148 * 8 ? blocks : 148 * 8);
  if (grid < 1) grid = 1;
  uint32_t* trailer = nullptr;
  if (prec == COPER_PREC_BF16)
    launch_pdl(prepare_kernel<COPER_PREC_BF16>, grid, 256, 0, st, src, rows, cols, ld_src, dst, ldp, trailer);
  else if (prec == COPER_PREC_TF32X3)
    launch_pdl(prepare_kernel<COPER_PREC_TF32X3>, grid, 256, 0, st, src, rows, cols, ld_src, dst, ldp, trailer);
  else if (prec == COPER_PREC_FP16X3) {
    trailer = fp16x3_trailer(dst, rows, cols);
    int rc = check_cuda(cudaMemsetAsync(trailer, 0, 16, st));
    if (rc) return rc;
    const int64_t n = rows * cols;
    if (n <= (int64_t)4 << 20) {                          // per-batch operands: one launch (see the kernel)
      // <= 2 blocks of 256 threads per SM: always co-resident (an SM holds 8 of them), which the grid barrier needs
      const int64_t want = (rows * (ldp / 8) + 256 * 4 - 1) / (256 * 4);
      int g = (int)(want < (int64_t)sm_count() * 2 ? want : (int64_t)sm_count() * 2);
      if (g < 1) g = 1;
      launch_pdl(prepare_fp16x3_fused_kernel, g, 256, 0, st, src, rows, cols, ld_src, static_cast<__half*>(dst), ldp,
                 trailer);
      return check_launch();
    }
    int g1 = (int)((n + 2047) / 2048 < sm_count() * 8 ? (n + 2047) / 2048 : sm_count() * 8);
    launch_pdl(absmax_kernel, g1 < 1 ? 1 : g1, 256, 0, st, src, rows, cols, ld_src, trailer);
    if ((rc = check_launch())) return rc;
    launch_pdl(prepare_kernel<COPER_PREC_FP16X3>, grid, 256, 0, st, src, rows, cols, ld_src, dst, ldp, trailer);
  } else
    return COPER_ERR_UNSUPPORTED;
  return check_launch();
}

int umma_score1n_fwd(const float* q, const float* E, const float* bias, int B, int64_t Ns, int d, float* scores,
                     int64_t ld, void* ws, size_t ws_bytes, int prec, cudaStream_t st) {
  if (!ws || ws_bytes < umma_score1n_workspace_bytes(B, Ns, d, prec)) return COPER_ERR_WORKSPACE;
  char* p = static_cast<char*>(ws);
  p = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(p) + 255) & ~uintptr_t(255));
  void* qp = p;
  void* Ep = p + prepared_bytes(B, d, prec);
  int rc;
  if ((rc = tc_prepare(q, B, d, d, prec, qp, st))) return rc;
  if ((rc = tc_prepare(E, Ns, d, d, prec, Ep, st))) return rc;
  return umma_score1n_fwd_prepared(qp, Ep, bias, B, Ns, d, scores, ld, prec, st);
}
}  // namespace coper

using namespace coper;

extern "C" {
size_t coper_prepared_bytes(int64_t rows, int cols, int prec) {
  if (prec != COPER_PREC_BF16 && prec != COPER_PREC_TF32X3 && prec != COPER_PREC_FP16X3) return 0;
  return prepared_bytes(rows, cols, prec);
}
int coper_prepare_operand(const float* src, int64_t rows, int cols, int64_t ld_src, int prec, void* dst,
                          coper_stream_t stream) {
  COPER_CHECK_ARG(src && dst && rows > 0 && cols > 0 && ld_src >= cols);
  COPER_CHECK_ARG((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
  return tc_prepare(src, rows, cols, ld_src, prec, dst, as_stream(stream));
}
int coper_score1n_fwd_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                               float* scores, int64_t ld_scores, int prec, coper_stream_t stream) {
  COPER_CHECK_ARG(q_prep && E_prep && bias && scores && B > 0 && Ns > 0 && d > 0);
  return umma_score1n_fwd_prepared(q_prep, E_prep, bias, B, Ns, d, scores, ld_scores, prec, as_stream(stream));
}
}  // extern "C"
