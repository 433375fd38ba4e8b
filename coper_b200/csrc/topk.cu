// Top-k link prediction: selection of the k best entities per query under the total order
//     score descending, then global entity id ascending.
// Every candidate is encoded as one 64-bit key whose unsigned order IS that order:
//     key = ord(score) << 32 | (0x7FFFFFFF - id) << 1 | (score is -0)
// with ord() the monotone map of IEEE floats onto uint32; -0 is folded onto +0 so that equal scores tie on the id, and
// the last bit (never deciding: ids are distinct) gives the score back bit for bit.
// Key 0 is below every real candidate and decodes to the padding pair (-inf, -1).  Keys of real candidates are
// distinct (one per entity), so the k largest keys are unique and any selection order gives the same result.
//
// Selection inside one CTA (BlockTopk): shared memory holds the current top k (sorted, descending) followed by an
// append buffer.  Candidates whose key beats the k-th best key so far are appended (one shared atomic each); when the
// buffer could overflow on the next round it is compacted: one bitonic sort of [top k | buffer], whose first k keys
// are the new top k.  For randomly ordered scores the buffer sees ~k (1 + ln(n / k)) appends, so compactions are rare.
//   coper_topk_scores: logits in HBM [B, ld] -> per (entity chunk, query) top-k lists -> merge.  (fp32 engine)
//   coper_topk_merge:  [n_lists, B, k] (score, id) lists -> [B, k].  (shard merge)
//   topk_merge_keys:   the merge of the fused scorer's per-(CTA, lane quadrant) key lists (umma_entity.cu).
#include "common.cuh"

namespace coper {

constexpr int kTopkThreads = 256;
constexpr int kTopkCap = 4096;                 // shared keys: top k + append buffer (32 KB)
constexpr int kTopkSpan = 16384;               // entities per CTA of coper_topk_scores

__device__ __forceinline__ uint64_t topk_key(float s, int64_t id) {
  if (id < 0) return 0ull;
  uint32_t u = __float_as_uint(s == 0.f ? 0.f : s);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  const uint32_t negz = __float_as_uint(s) == 0x80000000u;
  return ((uint64_t)u << 32) | (uint64_t)(((0x7FFFFFFFu - (uint32_t)id) << 1) | negz);
}
__device__ __forceinline__ void topk_decode(uint64_t key, float* s, int64_t* id) {
  if (key == 0ull) {
    *s = -INFINITY;
    *id = -1;
    return;
  }
  uint32_t u = (uint32_t)(key >> 32);
  u = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
  *s = (key & 1ull) ? -0.f : __uint_as_float(u);
  *id = (int64_t)(0x7FFFFFFFu - ((uint32_t)key >> 1));
}

struct BlockTopk {
  uint64_t* buf;     // [kTopkCap]
  int* n;            // appended keys
  uint64_t* thr;     // k-th best key so far (0 while fewer than k)
  int k;
  __device__ __forceinline__ void init() {
    for (int i = threadIdx.x; i < k; i += blockDim.x) buf[i] = 0ull;
    if (threadIdx.x == 0) { *n = 0; *thr = 0ull; }
    __syncthreads();
  }
  // every thread, after a __syncthreads() that follows init() / compact()
  __device__ __forceinline__ void offer(uint64_t key, uint64_t t) {
    if (key > t) buf[k + atomicAdd(n, 1)] = key;
  }
  // block-uniform call: sort [top k | appended] descending, keep the first k
  __device__ void compact() {
    __syncthreads();
    const int m = k + *n;
    int P = 2;
    while (P < m) P <<= 1;
    for (int i = m + threadIdx.x; i < P; i += blockDim.x) buf[i] = 0ull;
    __syncthreads();
    for (int size = 2; size <= P; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = threadIdx.x; i < P / 2; i += blockDim.x) {
          const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
          const uint64_t a = buf[lo], b = buf[hi];
          const bool desc = (lo & size) == 0;
          if (desc ? a < b : a > b) { buf[lo] = b; buf[hi] = a; }
        }
        __syncthreads();
      }
    }
    if (threadIdx.x == 0) { *n = 0; *thr = buf[k - 1]; }
    __syncthreads();
  }
  // compact if `incoming` more appends could overflow the buffer.  Called by every thread after a __syncthreads() that
  // follows the appends; the second barrier keeps the next round's appends from changing *n before every thread has
  // read it, so the decision (and the barriers inside compact()) is block-uniform.
  __device__ __forceinline__ void maybe_compact(int incoming) {
    const int m = *n;
    __syncthreads();
    if (k + m + incoming > kTopkCap) compact();
  }
};

#define COPER_TOPK_SMEM()                                   \
  __shared__ uint64_t tk_buf[kTopkCap];                     \
  __shared__ int tk_n;                                      \
  __shared__ uint64_t tk_thr;                               \
  BlockTopk bt{tk_buf, &tk_n, &tk_thr, k};

// stage 1 of coper_topk_scores: top k of entities [c * kTopkSpan, +kTopkSpan) of query b -> keys [chunk, B, k]
__global__ void __launch_bounds__(kTopkThreads) topk_scores_chunk_kernel(
    const float* __restrict__ scores, int64_t ld, int B, int64_t Ns, const uint32_t* __restrict__ filt, int64_t ent_lo,
    int k, uint64_t* __restrict__ out) {
  pdl_enter();
  COPER_TOPK_SMEM();
  bt.init();
  const int b = blockIdx.y;
  const int64_t c0 = (int64_t)blockIdx.x * kTopkSpan;
  const int64_t c1 = c0 + kTopkSpan < Ns ? c0 + kTopkSpan : Ns;
  const float* row = scores + (int64_t)b * ld;
  const uint32_t* frow = filt ? filt + (int64_t)b * ((Ns + 31) / 32) : nullptr;
  const bool vec_ok = (reinterpret_cast<uintptr_t>(row) & 15) == 0;
  for (int64_t base = c0; base < c1; base += kTopkThreads * 4) {
    const uint64_t t = *bt.thr;
    const int64_t n = base + (int64_t)threadIdx.x * 4;
    if (n < c1) {
      // 4 consecutive entities per thread (float4), one filter word covers 8 threads
      uint32_t fb = frow ? (__ldg(frow + (n >> 5)) >> (n & 31)) & 0xFu : 0u;
      float v[4];
      if (vec_ok && n + 3 < c1) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(row + n));
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = n + j < c1 ? __ldg(row + n + j) : 0.f;
        if (n + 3 >= c1) fb |= (0xFu << (c1 - n)) & 0xFu;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (!((fb >> j) & 1u)) bt.offer(topk_key(v[j], ent_lo + n + j), t);
    }
    __syncthreads();
    bt.maybe_compact(kTopkThreads * 4);
  }
  if (*bt.n) bt.compact();
  uint64_t* o = out + ((int64_t)blockIdx.x * B + b) * k;
  for (int i = threadIdx.x; i < k; i += blockDim.x) o[i] = bt.buf[i];
}

// Sources of the merge: list L of query b lives at lists + ((slot(L) * B) + b) * k with
//   slot(L) = (first + (L / per) * step) * per + L % per,  first = first_div ? b / first_div : 0
struct KeyLists {
  const uint64_t* lists;
  int per, first_div, step, n_groups;
  __device__ __forceinline__ int64_t count(int, int k) const { return (int64_t)n_groups * per * k; }
  __device__ __forceinline__ uint64_t key(int b, int B, int k, int64_t i) const {
    const int L = (int)(i / k), e = (int)(i - (int64_t)L * k);
    const int first = first_div ? b / first_div : 0;
    const int64_t slot = (int64_t)(first + (L / per) * step) * per + L % per;
    return __ldg(lists + (slot * B + b) * k + e);
  }
};
struct PairLists {
  const float* scores;
  const int64_t* ids;
  int n_lists;
  __device__ __forceinline__ int64_t count(int, int k) const { return (int64_t)n_lists * k; }
  __device__ __forceinline__ uint64_t key(int b, int B, int k, int64_t i) const {
    const int L = (int)(i / k), e = (int)(i - (int64_t)L * k);
    const int64_t o = ((int64_t)L * B + b) * k + e;
    return topk_key(__ldg(scores + o), __ldg(ids + o));
  }
};

template <class Src>
__global__ void __launch_bounds__(kTopkThreads) topk_merge_kernel(Src src, int B, int k, float* __restrict__ out_s,
                                                                  int64_t* __restrict__ out_id) {
  pdl_enter();
  COPER_TOPK_SMEM();
  bt.init();
  const int b = blockIdx.x;
  const int64_t total = src.count(b, k);
  for (int64_t base = 0; base < total; base += kTopkThreads) {
    const uint64_t t = *bt.thr;
    const int64_t i = base + threadIdx.x;
    if (i < total) bt.offer(src.key(b, B, k, i), t);
    __syncthreads();
    bt.maybe_compact(kTopkThreads);
  }
  if (*bt.n) bt.compact();
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    float s;
    int64_t id;
    topk_decode(bt.buf[i], &s, &id);
    out_s[(int64_t)b * k + i] = s;
    out_id[(int64_t)b * k + i] = id;
  }
}

int topk_merge_keys(const uint64_t* lists, int B, int k, int per, int first_div, int step, int n_groups, float* out_s,
                    int64_t* out_id, cudaStream_t st) {
  KeyLists src{lists, per, first_div, step, n_groups};
  launch_pdl(topk_merge_kernel<KeyLists>, B, kTopkThreads, 0, st, src, B, k, out_s, out_id);
  return check_launch();
}

static inline int topk_chunks(int64_t Ns) { return ceil_div(Ns, kTopkSpan); }

}  // namespace coper

using namespace coper;

extern "C" {

size_t coper_topk_scores_workspace_bytes(int B, int64_t Ns, int k) {
  if (B <= 0 || Ns <= 0 || k < 1 || k > COPER_TOPK_MAX) return 0;
  return (size_t)topk_chunks(Ns) * B * k * sizeof(uint64_t);
}

int coper_topk_scores(const float* scores, int64_t ld, int B, int64_t Ns, const uint32_t* filter_bits, int64_t ent_lo,
                      int k, float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                      coper_stream_t stream) {
  COPER_CHECK_ARG(scores && out_scores && out_ids && B > 0 && Ns > 0 && ld >= Ns && B <= 65535);
  COPER_CHECK_ARG(k >= 1 && k <= COPER_TOPK_MAX && ent_lo >= 0);
  if (ent_lo + Ns >= 0x7FFFFFFFll) return COPER_ERR_UNSUPPORTED;           // ids travel as 31-bit key fields
  if (!workspace || workspace_bytes < coper_topk_scores_workspace_bytes(B, Ns, k) ||
      (reinterpret_cast<uintptr_t>(workspace) & 7))
    return COPER_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  uint64_t* lists = static_cast<uint64_t*>(workspace);
  const int chunks = topk_chunks(Ns);
  launch_pdl(topk_scores_chunk_kernel, dim3(chunks, B), kTopkThreads, 0, st, scores, ld, B, Ns, filter_bits, ent_lo, k,
             lists);
  int rc = check_launch();
  if (rc) return rc;
  return topk_merge_keys(lists, B, k, 1, 0, 1, chunks, out_scores, out_ids, st);
}

int coper_topk_merge(const float* in_scores, const int64_t* in_ids, int n_lists, int B, int k, float* out_scores,
                     int64_t* out_ids, coper_stream_t stream) {
  COPER_CHECK_ARG(in_scores && in_ids && out_scores && out_ids && n_lists > 0 && B > 0);
  COPER_CHECK_ARG(k >= 1 && k <= COPER_TOPK_MAX);
  PairLists src{in_scores, in_ids, n_lists};
  launch_pdl(topk_merge_kernel<PairLists>, B, kTopkThreads, 0, as_stream(stream), src, B, k, out_scores, out_ids);
  return check_launch();
}

}  // extern "C"
