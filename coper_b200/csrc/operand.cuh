// The prepared operand format of the tensor-pipe (tcgen05) kernels: its layout, its roundings and the fp16x3 trailer
// are defined here and nowhere else.  Every kernel that writes an operand in this form (coper_prepare_operand, the
// CPG backward's context-scaled dy, the optimizer's operand copy, the BCE epilogues' dL/dS, the gathered gold rows)
// goes through the functions below.
//
//   COPER_PREC_BF16    one bf16 plane [rows, ldp], ldp = cols rounded up to 8; round to nearest even.
//   COPER_PREC_TF32X3  two fp32 planes [rows, ldp], ldp = cols rounded up to 4: hi = cvt.rna.tf32 (nearest, ties away
//                      from zero, low 13 bits zero), lo = x - hi (exact in fp32).
//   COPER_PREC_FP16X3  two fp16 planes [rows, ldp], ldp = cols rounded up to 8: hi = fp16(x * 2^e), lo = fp16(x * 2^e
//                      - hi), round to nearest even; then a 256-byte trailer of uint32 words (kTr*), 256-byte aligned.
// The lo plane starts right after the hi plane; padding columns hold zero; the buffer is a multiple of 256 bytes.
//
// fp16x3 keeps 11 significand bits per plane (like tf32) but only 5 exponent bits, so the operand is first scaled by a
// power of two (exact) that puts its largest magnitude at [2^10, 2^11): far from the fp16 overflow (2^16) and with 12
// binades of headroom before the lo plane of an element leaves the normal range (an element 2^12 below the max still
// carries 22 bits; smaller ones lose lo bits they contribute negligibly to any dot product).  The consuming kernels
// remove e from the accumulators (umma_gemm.cuh, SCALED).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "common.cuh"

namespace coper {

// ------------------------------------------------------------------------------------------ layout (host and device)
__host__ __device__ constexpr int prepared_planes(int prec) { return prec == COPER_PREC_BF16 ? 1 : 2; }
__host__ __device__ constexpr int prepared_elem_bytes(int prec) { return prec == COPER_PREC_TF32X3 ? 4 : 2; }
__host__ __device__ __forceinline__ int64_t prepared_ld(int cols, int prec) {
  return prec == COPER_PREC_TF32X3 ? (cols + 3) / 4 * 4 : (cols + 7) / 8 * 8;
}
// fp16x3 trailer: after two fp16 planes of plane_elems elements each (rows * ldp; the optimizer's copies have
// pitch == row length, so n), 256-byte aligned
__host__ __device__ __forceinline__ uint32_t* fp16x3_trailer(const void* prep, int64_t plane_elems) {
  return reinterpret_cast<uint32_t*>(const_cast<char*>(static_cast<const char*>(prep)) +
                                     ((size_t)plane_elems * 4 + 255) / 256 * 256);
}
__host__ __device__ __forceinline__ uint32_t* fp16x3_trailer(const void* prep, int64_t rows, int cols) {
  return fp16x3_trailer(prep, rows * prepared_ld(cols, COPER_PREC_FP16X3));
}
inline size_t prepared_bytes(int64_t rows, int cols, int prec) {
  const size_t planes = (size_t)rows * prepared_ld(cols, prec) * prepared_elem_bytes(prec) * prepared_planes(prec);
  return align_up(planes, 256) + (prec == COPER_PREC_FP16X3 ? 256 : 0);
}

// fp16x3 trailer words.  Max words hold float bits: non-negative floats order like their bit patterns (atomicMax).
constexpr int kTrExp = 0;      // e (int32)
constexpr int kTrMax = 1;      // max |x| of the last full preparation
constexpr int kTrRunMax = 2;   // max |x| of what the optimizer re-emits; rolled into kTrExp before its next pass
constexpr int kTrArrive = 3;   // arrive counter of the one-launch preparations' grid barrier
constexpr int kTrMax2 = 4;     // CPG backward, dy's trailer: max |dy * c| for the context-scaled operand

// e such that max |x| lands in [2^10, 2^11); 0 for an all-zero operand or a NaN / Inf max
constexpr int kFp16x3TargetExp = 10;
__host__ __device__ __forceinline__ int fp16x3_exponent_of(float absmax) {
  if (!(absmax > 0.f) || !(absmax < 3.0e38f)) return 0;
  int ex;
  frexpf(absmax, &ex);                       // absmax = f * 2^ex, f in [0.5, 1)  ->  ilogb = ex - 1
  int e = kFp16x3TargetExp - (ex - 1);
  return e < -100 ? -100 : (e > 100 ? 100 : e);
}

// ------------------------------------------------------------------------------------------ element conversions
__device__ __forceinline__ float tf32_hi(float x) {
  uint32_t h;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x));
  return __uint_as_float(h);
}
// hi / lo fp16 of two values already scaled by 2^e, as the 32-bit words of two __half2 (a in the low half)
__device__ __forceinline__ void fp16_split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);          // the residuals are exact in fp32
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// the same split of one value (as fp16x2 with a zero lane it would cost three more instructions per value)
__device__ __forceinline__ void fp16_split(float a, uint16_t& hi, uint16_t& lo) {
  const __half h = __float2half_rn(a);
  hi = __half_as_ushort(h);
  lo = __half_as_ushort(__float2half_rn(a - __half2float(h)));
}
__device__ __forceinline__ uint32_t bf16_pack2(float a, float b) {
  const __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&p);
}
__device__ __forceinline__ uint4 bf16_pack8(const float* x) {
  return make_uint4(bf16_pack2(x[0], x[1]), bf16_pack2(x[2], x[3]), bf16_pack2(x[4], x[5]), bf16_pack2(x[6], x[7]));
}
__device__ __forceinline__ void fp16_split8(const float* x, uint4& hi, uint4& lo) {
  fp16_split2(x[0], x[1], hi.x, lo.x);
  fp16_split2(x[2], x[3], hi.y, lo.y);
  fp16_split2(x[4], x[5], hi.z, lo.z);
  fp16_split2(x[6], x[7], hi.w, lo.w);
}

// N = 4 or 8 consecutive values x to element i of both planes (the lo plane plane_elems elements after the hi plane):
// one 8- / 16-byte store per plane and 4 values.  sc = 2^e for fp16x3, ignored otherwise.
template <int PREC, int N>
__device__ __forceinline__ void emit_prepared_vec(void* dst, int64_t plane_elems, int64_t i, const float* x, float sc) {
  static_assert(N == 4 || N == 8, "4 or 8 values");
  if constexpr (PREC == COPER_PREC_TF32X3) {
    float* hi = static_cast<float*>(dst) + i;
#pragma unroll
    for (int k = 0; k < N; k += 4) {
      float h[4], l[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        h[j] = tf32_hi(x[k + j]);
        l[j] = x[k + j] - h[j];
      }
      *reinterpret_cast<float4*>(hi + k) = make_float4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<float4*>(hi + plane_elems + k) = make_float4(l[0], l[1], l[2], l[3]);
    }
  } else {
    uint32_t h[N / 2], l[N / 2];
#pragma unroll
    for (int k = 0; k < N / 2; ++k) {
      if constexpr (PREC == COPER_PREC_BF16) h[k] = bf16_pack2(x[2 * k], x[2 * k + 1]);
      else fp16_split2(x[2 * k] * sc, x[2 * k + 1] * sc, h[k], l[k]);
    }
    uint16_t* p = static_cast<uint16_t*>(dst) + i;
    if constexpr (N == 8) {
      *reinterpret_cast<uint4*>(p) = make_uint4(h[0], h[1], h[2], h[3]);
      if constexpr (PREC == COPER_PREC_FP16X3) *reinterpret_cast<uint4*>(p + plane_elems) = make_uint4(l[0], l[1], l[2], l[3]);
    } else {
      *reinterpret_cast<uint2*>(p) = make_uint2(h[0], h[1]);
      if constexpr (PREC == COPER_PREC_FP16X3) *reinterpret_cast<uint2*>(p + plane_elems) = make_uint2(l[0], l[1]);
    }
  }
}
// one value x to element i of both planes
__device__ __forceinline__ void emit_prepared(int prec, void* dst, int64_t plane_elems, int64_t i, float x, float sc) {
  if (prec == COPER_PREC_BF16) {
    static_cast<uint16_t*>(dst)[i] = (uint16_t)bf16_pack2(x, 0.f);
  } else if (prec == COPER_PREC_FP16X3) {
    uint16_t h, l;
    fp16_split(x * sc, h, l);
    static_cast<uint16_t*>(dst)[i] = h;
    static_cast<uint16_t*>(dst)[plane_elems + i] = l;
  } else {
    const float h = tf32_hi(x);
    static_cast<float*>(dst)[i] = h;
    static_cast<float*>(dst)[plane_elems + i] = x - h;
  }
}
// 4 values to element i (a multiple of 4).  The lo plane is 16-byte aligned only if plane_elems % 4 == 0: otherwise
// the two-plane formats are emitted one value at a time.
__device__ __forceinline__ void emit_prepared4(int prec, void* dst, int64_t plane_elems, int64_t i, float4 v, float sc) {
  const float x[4] = {v.x, v.y, v.z, v.w};
  if (prec == COPER_PREC_BF16) {
    emit_prepared_vec<COPER_PREC_BF16, 4>(dst, plane_elems, i, x, sc);
  } else if (plane_elems & 3) {
#pragma unroll
    for (int k = 0; k < 4; ++k) emit_prepared(prec, dst, plane_elems, i + k, x[k], sc);
  } else if (prec == COPER_PREC_FP16X3) {
    emit_prepared_vec<COPER_PREC_FP16X3, 4>(dst, plane_elems, i, x, sc);
  } else {
    emit_prepared_vec<COPER_PREC_TF32X3, 4>(dst, plane_elems, i, x, sc);
  }
}

// ------------------------------------------------------------------------------------------ fp16x3 trailer operations
// max m into a max word; nothing is published for 0 (a NaN / Inf max makes the exponent choice fall back to 0)
__device__ __forceinline__ void trailer_max(uint32_t* word, float m) {
  if (m > 0.f) atomicMax(word, __float_as_uint(m));
}
__device__ __forceinline__ void warp_trailer_max(uint32_t* word, float m) {
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) trailer_max(word, m);
}
// the exponent for max bits mbits: the leader writes it to kTrExp and mbits to max_word (< 0: none); returns 2^e
__device__ __forceinline__ float fp16x3_publish(uint32_t* tr, uint32_t mbits, int max_word, bool leader) {
  const int e = fp16x3_exponent_of(__uint_as_float(mbits));
  if (leader) {
    reinterpret_cast<int*>(tr)[kTrExp] = e;
    if (max_word >= 0) tr[max_word] = mbits;
  }
  return exp2f((float)e);
}
// before the optimizer re-emits the operand: the exponent of the magnitude the variable has now, running max restarted
__device__ __forceinline__ void fp16x3_roll(uint32_t* tr) {
  reinterpret_cast<int*>(tr)[kTrExp] = fp16x3_exponent_of(__uint_as_float(tr[kTrRunMax]));
  tr[kTrRunMax] = 0u;
}
// Grid-wide barrier of the one-launch preparations, called by one thread per block after it published the block's
// maxima.  The grid is capped so that all blocks are co-resident (the spin cannot wait on a block that has not been
// scheduled); a barrier that does not complete traps instead of hanging the GPU.
__device__ __forceinline__ void grid_arrive_wait(uint32_t* arrive) {
  __threadfence();
  atomicAdd(arrive, 1u);
  const long long t0 = clock64();
  while (*reinterpret_cast<volatile uint32_t*>(arrive) < gridDim.x) {     // plain polling load, no RMW traffic
    if (clock64() - t0 > 4000000000ll) __trap();
  }
  __threadfence();
}

// ------------------------------------------------------------------------------------------ host (umma_score.cu)
// coper_prepare_operand without the argument checks
int tc_prepare(const float* src, int64_t rows, int cols, int64_t ld_src, int prec, void* dst, cudaStream_t st);

}  // namespace coper
