// a7 / K6 on the tensor pipe: 1-N scorer logits S = q.E^T + bias (models.py:433-437) as a persistent,
// warp-specialised tcgen05 GEMM: TMA-fed 128B-swizzled operand ring, fp32 accumulators double-buffered in
// TMEM, bias add fused into the TMEM->register epilogue.  M = queries (TMEM lanes), N = entities (TMEM
// columns), K = d.  Two arithmetic modes (include/coper.h): COPER_PREC_BF16 and COPER_PREC_TF32X3.
//
// Operands are consumed in "prepared" form (coper_prepare_operand): bf16 copy, or (hi, lo) tf32 planes —
// the entity table is prepared once per evaluation pass / per optimizer step, not per call.
#include <cuda_fp16.h>
#include "umma_gemm.cuh"

namespace coper {
using namespace umma;

// ------------------------------------------------------------------------------------------ operand preparation
static inline int64_t prepared_ld(int cols, int prec) { return prec == COPER_PREC_TF32X3 ? (cols + 3) / 4 * 4 : (cols + 7) / 8 * 8; }

// block = (64 column lanes) x (4 rows); grid-stride over rows; each lane converts VEC consecutive columns per pass
// (VEC = 8 bf16 / 4 tf32 -> one 16-byte store per plane); no integer division anywhere
template <int PREC>
__global__ void __launch_bounds__(256) prepare_kernel(const float* __restrict__ src, int64_t rows, int cols,
                                                      int64_t ld_src, void* __restrict__ dst, int64_t ldp) {
  pdl_enter();
  constexpr int VEC = PREC == COPER_PREC_BF16 ? 8 : 4;
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
      if (PREC == COPER_PREC_BF16) {
        __nv_bfloat162 p0 = __floats2bfloat162_rn(x[0], x[1]), p1 = __floats2bfloat162_rn(x[2], x[3]);
        __nv_bfloat162 p2 = __floats2bfloat162_rn(x[4 % VEC], x[5 % VEC]), p3 = __floats2bfloat162_rn(x[6 % VEC], x[7 % VEC]);
        uint4 u;
        u.x = *reinterpret_cast<uint32_t*>(&p0); u.y = *reinterpret_cast<uint32_t*>(&p1);
        u.z = *reinterpret_cast<uint32_t*>(&p2); u.w = *reinterpret_cast<uint32_t*>(&p3);
        *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(dst) + r * ldp + c0) = u;
      } else {
        float h[4], l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          uint32_t hb;
          asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(x[k]));   // round-to-nearest tf32, low 13 bits zero
          h[k] = __uint_as_float(hb);
          l[k] = x[k] - h[k];                                        // exact in fp32
        }
        float* hi = static_cast<float*>(dst) + r * ldp + c0;
        *reinterpret_cast<float4*>(hi) = make_float4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<float4*>(hi + rows * ldp) = make_float4(l[0], l[1], l[2], l[3]);
      }
    }
  }
}

// ---- COPER_PREC_FP16X3: hi / lo IEEE fp16 planes of x * 2^e with ONE exponent per operand.
// fp16 keeps 11 significand bits per plane (like tf32) but only 5 exponent bits, so the operand is first scaled by a
// power of two (exact) that puts its largest magnitude at [2^10, 2^11): far from the fp16 overflow (2^16) and with
// 12 binades of headroom before the lo plane of an element leaves the normal range (an element 2^12 below the max
// still carries 22 bits; smaller ones lose lo bits they contribute negligibly to any dot product).  e lives in the
// 256-byte trailer of the prepared buffer (int32 at offset 0; the max |x| as float bits at offset 4) and is removed
// from the accumulators by the consuming kernels (umma_gemm.cuh, SCALED).
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
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  // non-negative floats order like their bit patterns; a NaN / Inf input makes the exponent choice fall back to 0
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(trailer + 1, __float_as_uint(m));
}
__device__ __forceinline__ int fp16x3_exponent(uint32_t absmax_bits) { return fp16x3_exponent_of(__uint_as_float(absmax_bits)); }
__global__ void __launch_bounds__(256) prepare_fp16x3_kernel(const float* __restrict__ src, int64_t rows, int cols,
                                                             int64_t ld_src, __half* __restrict__ dst, int64_t ldp,
                                                             uint32_t* __restrict__ trailer) {
  pdl_enter();
  const int e = fp16x3_exponent(trailer[1]);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    reinterpret_cast<int*>(trailer)[0] = e;
    trailer[2] = trailer[1];                           // seeds the optimizer's running max (common.cuh)
  }
  const float sc = exp2f((float)e);
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  const int nvec = (int)(ldp / 8);
  const bool vec_src = ((ld_src & 3) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  __half* lo_plane = dst + rows * ldp;
  for (int64_t r = (int64_t)blockIdx.x * 4 + ty; r < rows; r += (int64_t)gridDim.x * 4) {
    const float* srow = src + r * ld_src;
    for (int v = tx; v < nvec; v += 64) {
      const int c0 = v * 8;
      float x[8];
      if (vec_src && c0 + 8 <= cols) {
#pragma unroll
        for (int k = 0; k < 8; k += 4) {
          float4 t = __ldg(reinterpret_cast<const float4*>(srow + c0 + k));
          x[k] = t.x; x[k + 1] = t.y; x[k + 2] = t.z; x[k + 3] = t.w;
        }
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] = (c0 + k < cols) ? __ldg(srow + c0 + k) : 0.f;
      }
      __half2 h[4], l[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float a = x[2 * k] * sc, b = x[2 * k + 1] * sc;
        h[k] = __floats2half2_rn(a, b);
        const float2 hf = __half22float2(h[k]);
        l[k] = __floats2half2_rn(a - hf.x, b - hf.y);            // the residuals are exact in fp32
      }
      *reinterpret_cast<uint4*>(dst + r * ldp + c0) = *reinterpret_cast<uint4*>(h);
      *reinterpret_cast<uint4*>(lo_plane + r * ldp + c0) = *reinterpret_cast<uint4*>(l);
    }
  }
}

// Small operands (activations / gradients of one batch: q, f, dy): max |x| and the split in ONE launch.  Every block
// reduces its share of the max into the trailer, a grid-wide arrive counter (trailer[3]) tells when all shares are in,
// then each block converts its rows.  The grid is capped so that all blocks are co-resident (the spin cannot wait on a
// block that has not been scheduled); a stuck barrier traps instead of hanging the GPU.
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
    if (m > 0.f) atomicMax(trailer + 1, __float_as_uint(m));
    __threadfence();
    atomicAdd(trailer + 3, 1u);
    const long long t0 = clock64();
    while (*reinterpret_cast<volatile uint32_t*>(trailer + 3) < gridDim.x) {     // plain polling load, no RMW traffic
      if (clock64() - t0 > 4000000000ll) __trap();
    }
    __threadfence();
  }
  __syncthreads();
  const uint32_t mbits = *reinterpret_cast<volatile uint32_t*>(trailer + 1);
  const int e = fp16x3_exponent(mbits);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    reinterpret_cast<int*>(trailer)[0] = e;
    trailer[2] = mbits;
  }
  const float sc = exp2f((float)e);
  __half* lo_plane = dst + rows * ldp;
  for (int64_t u = (int64_t)blockIdx.x * 256 + threadIdx.x; u < units; u += (int64_t)gridDim.x * 256) {
    float x[8];
    load8(u, x);                                       // second touch of the same addresses: L1 / L2 hits
    __half2 h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float a = x[2 * k] * sc, b = x[2 * k + 1] * sc;
      h[k] = __floats2half2_rn(a, b);
      const float2 hf = __half22float2(h[k]);
      l[k] = __floats2half2_rn(a - hf.x, b - hf.y);
    }
    *reinterpret_cast<uint4*>(dst + u * 8) = *reinterpret_cast<uint4*>(h);        // u * 8 == r * ldp + c0
    *reinterpret_cast<uint4*>(lo_plane + u * 8) = *reinterpret_cast<uint4*>(l);
  }
}

// entity-major scorer kernels: umma_entity.cu
int umma_score1n_fwd_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                              float* scores, int64_t ld, int prec, cudaStream_t st);

static size_t prepared_bytes(int64_t rows, int cols, int prec) {
  int64_t ldp = prepared_ld(cols, prec);
  if (prec == COPER_PREC_FP16X3) return align_up((size_t)rows * ldp * 2 * 2, 256) + 256;    // 2 fp16 planes + trailer
  size_t b = prec == COPER_PREC_BF16 ? (size_t)rows * ldp * 2 : (size_t)rows * ldp * 4 * 2;
  return align_up(b, 256);
}
// device address of the 256-byte trailer {int32 e, float-bits max |x|} of an FP16X3 operand
void* tc_fp16x3_trailer(const void* prep, int64_t rows, int cols) {
  return const_cast<char*>(static_cast<const char*>(prep)) + align_up((size_t)rows * prepared_ld(cols, COPER_PREC_FP16X3) * 4, 256);
}

size_t umma_score1n_workspace_bytes(int B, int64_t Ns, int d, int prec) {
  return prepared_bytes(B, d, prec) + prepared_bytes(Ns, d, prec) + 256;
}

static int prepare(const float* src, int64_t rows, int cols, int64_t ld_src, int prec, void* dst, cudaStream_t st) {
  int64_t ldp = prepared_ld(cols, prec);
  int64_t blocks = (rows + 3) / 4;
  int grid = (int)(blocks < 148 * 8 ? blocks : 148 * 8);
  if (grid < 1) grid = 1;
  if (prec == COPER_PREC_BF16)
    launch_pdl(prepare_kernel<COPER_PREC_BF16>, grid, 256, 0, st, src, rows, cols, ld_src, dst, ldp);
  else if (prec == COPER_PREC_TF32X3)
    launch_pdl(prepare_kernel<COPER_PREC_TF32X3>, grid, 256, 0, st, src, rows, cols, ld_src, dst, ldp);
  else if (prec == COPER_PREC_FP16X3) {
    uint32_t* trailer = static_cast<uint32_t*>(tc_fp16x3_trailer(dst, rows, cols));
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
    launch_pdl(prepare_fp16x3_kernel, grid, 256, 0, st, src, rows, cols, ld_src, static_cast<__half*>(dst), ldp,
               trailer);
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
  if ((rc = prepare(q, B, d, d, prec, qp, st))) return rc;
  if ((rc = prepare(E, Ns, d, d, prec, Ep, st))) return rc;
  return umma_score1n_fwd_prepared(qp, Ep, bias, B, Ns, d, scores, ld, prec, st);
}
size_t tc_prepared_bytes(int64_t rows, int cols, int prec) { return prepared_bytes(rows, cols, prec); }
int tc_prepare(const float* src, int64_t rows, int cols, int64_t ld_src, int prec, void* dst, cudaStream_t st) {
  return prepare(src, rows, cols, ld_src, prec, dst, st);
}
int64_t tc_prepared_ld(int cols, int prec) { return prepared_ld(cols, prec); }
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
  return prepare(src, rows, cols, ld_src, prec, dst, as_stream(stream));
}
int coper_score1n_fwd_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                               float* scores, int64_t ld_scores, int prec, coper_stream_t stream) {
  COPER_CHECK_ARG(q_prep && E_prep && bias && scores && B > 0 && Ns > 0 && d > 0);
  return umma_score1n_fwd_prepared(q_prep, E_prep, bias, B, Ns, d, scores, ld_scores, prec, as_stream(stream));
}
}  // extern "C"
