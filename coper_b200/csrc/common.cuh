// Shared device/host helpers for libcoper_sm100 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/coper.h"

namespace coper {

extern thread_local int g_last_cuda_error;
extern long long g_launch_count;  // kernels launched by this library (every launch is followed by check_launch)

inline int check_launch() {
  ++g_launch_count;
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    g_last_cuda_error = (int)e;
    cudaGetLastError();
    return COPER_ERR_CUDA;
  }
  return COPER_OK;
}
inline int check_cuda(cudaError_t e) {
  if (e != cudaSuccess) {
    g_last_cuda_error = (int)e;
    return COPER_ERR_CUDA;
  }
  return COPER_OK;
}
#define COPER_CHECK_ARG(cond) \
  do {                        \
    if (!(cond)) return COPER_ERR_INVALID_ARG; \
  } while (0)

static inline cudaStream_t as_stream(coper_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// ---- programmatic dependent launch (PDL).  The training / evaluation step is a chain of ~30 short dependent kernels;
// with plain stream order each one is launched only after its predecessor has drained.  Every kernel of this library
// is launched with the programmatic-stream-serialization attribute and starts with pdl_enter(): it releases ITS
// dependent at once (griddepcontrol.launch_dependents - the next kernel's blocks may be scheduled, set up and parked as
// soon as all blocks of this one have started) and then waits for its own predecessor to complete and flush
// (griddepcontrol.wait), before touching any memory.  Correctness never depends on the attribute: without it (or after
// a non-kernel stream operation, an event wait, a kernel of another library) both instructions are no-ops and the
// launch is an ordinary one.  The tcgen05 kernels place the wait after their prologue (barrier init, TMEM allocation,
// descriptor prefetch - nothing that reads a predecessor's output).  coper_set_pdl(0) turns it off.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter() {
  pdl_trigger();
  pdl_wait();
}
bool pdl_enabled();      // elementwise.cu
template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);   // errors surface in check_launch()
}

// Counter-based dropout hash (splitmix64 finaliser): identical on host and device.
__host__ __device__ __forceinline__ uint32_t hash32(uint64_t seed, uint64_t idx) {
  uint64_t z = seed + (idx + 1) * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= (z >> 31);
  return (uint32_t)(z >> 32);
}
// keep threshold: element kept iff hash32 < thr (thr == 0xFFFFFFFF and keep>=1 -> always kept, handled by caller)
__host__ __device__ __forceinline__ uint32_t keep_threshold(float keep) {
  double t = (double)keep * 4294967296.0;
  if (t >= 4294967295.0) return 0xFFFFFFFFu;
  if (t <= 0.0) return 0u;
  return (uint32_t)t;
}
// multiplicative dropout factor for element idx: 0 or 1/keep; keep>=1 -> 1
__device__ __forceinline__ float drop_factor(float keep, float inv_keep, uint32_t thr, uint64_t seed, uint64_t idx) {
  if (keep >= 1.0f) return 1.0f;
  return hash32(seed, idx) < thr ? inv_keep : 0.0f;
}

// dx of batch norm + relu + post-dropout for one element (without the pre-dropout factor): g1 = dout * drop_post *
// relu'(a x + b); dx = a (g1 - c1 - xhat c2).  One definition with explicit roundings, shared by coper_bn_act_bwd_apply and
// the conv backward that consumes dout directly (coper_conv_bwd_bn) - the two give the same bits.
__device__ __forceinline__ float bn_bwd_dx(float dout, float post_factor, float xv, float ac, float bc, float mean,
                                           float invstd, float c1, float c2, int relu) {
  float g = __fmul_rn(dout, post_factor);
  if (relu && !(fmaf(ac, xv, bc) > 0.f)) g = 0.f;
  const float xhat = __fmul_rn(__fsub_rn(xv, mean), invstd);
  return __fmul_rn(ac, fmaf(-xhat, c2, __fsub_rn(g, c1)));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide deterministic sum (all threads must call; result valid in thread 0). blockDim.x multiple of 32, <= 1024.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* smem32) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) smem32[w] = v;
  __syncthreads();
  T r = T(0);
  if (w == 0) {
    int nw = (blockDim.x + 31) >> 5;
    r = lane < nw ? smem32[lane] : T(0);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  }
  __syncthreads();
  return r;
}

// COPER_PREC_FP16X3 operand scaling (umma_score.cu): x is stored as hi / lo fp16 planes of x * 2^e with e chosen so that
// the operand's max |x| lands in [2^10, 2^11).  Trailer of a prepared operand (uint32 words, 256 bytes after the planes):
// [0] e (int32), [1] max |x| of the last full preparation (float bits), [2] max |x| accumulated by the optimizer kernel
// while it re-emits the operand (float bits; rolled into [0] before the next optimizer pass).
constexpr int kFp16x3TargetExp = 10;
__host__ __device__ __forceinline__ int fp16x3_exponent_of(float absmax) {
  if (!(absmax > 0.f) || !(absmax < 3.0e38f)) return 0;
  int ex;
  frexpf(absmax, &ex);                       // absmax = f * 2^ex, f in [0.5, 1)  ->  ilogb = ex - 1
  int e = kFp16x3TargetExp - (ex - 1);
  return e < -100 ? -100 : (e > 100 ? 100 : e);
}

// SMs of the current device (148 on B200), queried once per device: grids of the persistent kernels are sized from it
inline int sm_count() {
  static int cached[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (!cached[dev]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// elementwise.cu: fixed-order reduction of S slabs, optionally with a sum of doubles riding in the same launch
int reduce_partials_and_sum(const float* in, int S, int64_t n, float scale, int accumulate, float* out,
                            const double* dsum_in, int dsum_n, double* dsum_out, cudaStream_t st);

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace coper
