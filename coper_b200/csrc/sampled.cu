// a8 / SURVEY §8f-2: the SAMPLED-label scorer of the reference (models.py:438-443: tf.gather of [B, L] entity rows,
// batched mat-vec, + gathered bias), its label-smoothed sigmoid-BCE (models.py:448-453) and the gradients TF's
// autodiff produces for it — what every shipped big-dataset config trains with (num_labels = 100 / 1000).
//
// The path is gather-bound ([B, L, d] rows of the entity table: 410 MB at B=512, L=1000, d=200), not GEMM-shaped:
//   kernel 1 (one CTA per query): q[b] lives in registers, warps stride over the L sampled entities, each row is read
//     ONCE (coalesced 128-byte segments) and used for the logit (warp reduction), the loss, dL/ds and the running
//     dq[b] += g * E_row; per-warp dq accumulators are combined in shared memory in a fixed order.
//   kernel 2: the gradient of the two gathers is an IndexedSlices in TF (values g[b,l]*q[b] at row lookup[b,l]).
//     The optimizer's sparse rule (utils/amsgrad.py:161-189) and tf.clip_by_global_norm need, per entity row, the SUM
//     of its slices and the sum of their SQUARES: (lookup id, position) pairs are radix-sorted (cub) and one warp per
//     segment walks it in sorted order — no atomics, fixed summation order -> deterministic.
#include <cub/device/device_radix_sort.cuh>
#include "common.cuh"

namespace coper {

constexpr int kSampWarps = 8;
constexpr int kSampMaxK = 8;     // d <= 256: up to 8 strided elements per lane

// kShard (coper_score_sampled_bce_fwd_bwd_sharded): E / bias hold the rows [row_lo, row_hi) of the table and only the
// positions whose id falls there are scored; the others read nothing and add nothing.  The arithmetic of a scored
// position is the same in both instantiations, so its score and g are bit-identical to the unsharded call's.
template <bool kShard>
__global__ void __launch_bounds__(kSampWarps * 32) sampled_score_bce_kernel(
    const float* __restrict__ q, const float* __restrict__ E, const float* __restrict__ bias,
    const int32_t* __restrict__ lookup, const float* __restrict__ labels, int L, int64_t N, int d, float one_minus_eps,
    float inv_num_ent, float inv_count, double* __restrict__ loss_part, float* __restrict__ scores,
    float* __restrict__ g_out, float* __restrict__ dq, int64_t row_lo, int64_t row_hi) {
  pdl_enter();
  __shared__ float red[kSampWarps][256];
  __shared__ double lred[kSampWarps];
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float qr[kSampMaxK], acc[kSampMaxK];
#pragma unroll
  for (int k = 0; k < kSampMaxK; ++k) {
    const int c = lane + 32 * k;
    qr[k] = c < d ? __ldg(q + (int64_t)b * d + c) : 0.f;
    acc[k] = 0.f;
  }
  double lsum = 0.0;
  for (int l = warp; l < L; l += kSampWarps) {
    const int64_t p = (int64_t)b * L + l;
    int64_t ent = lookup[p];
    if constexpr (kShard) {
      if (ent < row_lo || ent >= row_hi) continue;       // warp-uniform (one position per warp): another shard's row
      ent -= row_lo;
    }
    const float* row = E + ent * d;
    float er[kSampMaxK];
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < kSampMaxK; ++k) {
      const int c = lane + 32 * k;
      er[k] = c < d ? __ldg(row + c) : 0.f;
      dot = fmaf(qr[k], er[k], dot);
    }
    dot = warp_sum(dot);
    const float s = dot + __ldg(bias + ent);
    const float z = one_minus_eps * __ldg(labels + p) + inv_num_ent;          // models.py:450
    const float e = expf(-fabsf(s));
    const float loss = fmaxf(s, 0.f) - s * z + log1pf(e);
    const float sig = (s >= 0.f) ? 1.0f / (1.0f + e) : e / (1.0f + e);
    const float g = (sig - z) * inv_count;
    if (lane == 0) {
      g_out[p] = g;
      if (scores) scores[p] = s;
      lsum += (double)loss;
    }
#pragma unroll
    for (int k = 0; k < kSampMaxK; ++k) acc[k] = fmaf(g, er[k], acc[k]);
  }
#pragma unroll
  for (int k = 0; k < kSampMaxK; ++k) red[warp][lane + 32 * k] = acc[k];
  if (lane == 0) lred[warp] = lsum;
  __syncthreads();
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kSampWarps; ++w) t += red[w][c];
    dq[(int64_t)b * d + c] = t;
  }
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < kSampWarps; ++w) t += lred[w];
    loss_part[b] = t;
  }
}

__global__ void sum_loss_kernel(const double* __restrict__ in, int n, double* out) {
  pdl_enter();
  __shared__ double smd[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += in[i];
  double t = block_sum<double>(acc, smd);
  if (threadIdx.x == 0) *out = t;
}

__global__ void iota32_kernel(int32_t* p, int n) {
  pdl_enter();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}

// sharded scatter: sort key = local row of an owned position, n_rows (sorts after every owned row) for the others
__global__ void sampled_shard_keys_kernel(const int32_t* __restrict__ lookup, int M, int64_t row_lo, int64_t row_hi,
                                          int32_t* __restrict__ keys, int32_t* __restrict__ pos) {
  pdl_enter();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const int64_t id = lookup[i];
  keys[i] = (int32_t)((id >= row_lo && id < row_hi) ? id - row_lo : row_hi - row_lo);
  pos[i] = i;
}

// one warp per sorted position; segment heads walk their segment: slice value = g[pos] * q[pos / L, :]
// (kShard: keys >= n_rows are the non-owned positions at the end of the sorted order and are skipped)
template <bool kShard>
__global__ void sampled_scatter_kernel(const int32_t* __restrict__ keys, const int32_t* __restrict__ pos, int M, int L,
                                       const float* __restrict__ g, const float* __restrict__ q, int d,
                                       float* __restrict__ dE_sum, float* __restrict__ dE_sq,
                                       float* __restrict__ db_sum, float* __restrict__ db_sq, int n_rows) {
  pdl_enter();
  const int seg = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (seg >= M) return;
  const int32_t key = keys[seg];
  if constexpr (kShard) {
    if (key >= n_rows) return;
  }
  if (seg > 0 && keys[seg - 1] == key) return;   // not a segment head
  int end = seg + 1;
  while (end < M && keys[end] == key) ++end;
  float a1[kSampMaxK], a2[kSampMaxK];
#pragma unroll
  for (int k = 0; k < kSampMaxK; ++k) a1[k] = a2[k] = 0.f;
  float b1 = 0.f, b2 = 0.f;
  for (int i = seg; i < end; ++i) {
    const int p = pos[i];
    const float gv = __ldg(g + p);
    const float* qrow = q + (int64_t)(p / L) * d;
    b1 += gv;
    b2 = fmaf(gv, gv, b2);
#pragma unroll
    for (int k = 0; k < kSampMaxK; ++k) {
      const int c = lane + 32 * k;
      if (c < d) {
        const float v = gv * __ldg(qrow + c);
        a1[k] += v;
        a2[k] = fmaf(v, v, a2[k]);
      }
    }
  }
  float* r1 = dE_sum + (int64_t)key * d;
  float* r2 = dE_sq + (int64_t)key * d;
#pragma unroll
  for (int k = 0; k < kSampMaxK; ++k) {
    const int c = lane + 32 * k;
    if (c < d) {
      r1[c] += a1[k];
      r2[c] += a2[k];
    }
  }
  if (lane == 0) {
    db_sum[key] += b1;
    db_sq[key] += b2;
  }
}

// ---- on-device label sampling (data.py:228-277, _sample_negatives) ------------------------------------------------
// Two keyed random permutations of [0, n):
//   n <= kSampleSmall: ORDER of the n hashes hash32(key, i) (ties broken by i): position of element i = its rank.
//     Uniform over all n! orders for an ideal hash; O(n^2 / threads) per row, n is tiny (a row's positives; the
//     entity set of the toy datasets).
//   larger n: 6-round balanced Feistel network over the next even power of two, restricted to [0, n) by cycle walking
//     (a bijection of the larger domain walked until it lands inside stays a bijection); O(1) per drawn element.
constexpr int kSampleSmall = 1024;
__device__ __forceinline__ uint32_t prp(uint32_t x, uint32_t n, uint64_t key) {
  int bits = 2;
  while (bits < 32 && (1ull << bits) < (uint64_t)n) bits += 2;
  const int half = bits >> 1;
  const uint32_t mask = (1u << half) - 1u;
  do {
    uint32_t l = x >> half, r = x & mask;
#pragma unroll
    for (int round = 0; round < 6; ++round) {
      const uint32_t t = l ^ (hash32(key, ((uint64_t)round << 32) | r) & mask);
      l = r;
      r = t;
    }
    x = (l << half) | r;
  } while (x >= n);
  return x;
}

// rank permutation: every element i < n whose rank is < count writes out(rank, i)
template <class Out>
__device__ __forceinline__ void rank_permute(uint32_t* sh, int n, int count, uint64_t key, Out out) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) sh[i] = hash32(key, (uint64_t)i);
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const uint32_t hi = sh[i];
    int r = 0;
    for (int j = 0; j < n; ++j) {
      const uint32_t hj = sh[j];
      r += (hj < hi) || (hj == hi && j < i);
    }
    if (r < count) out(r, i);
  }
  __syncthreads();
}

constexpr int kSampleThreads = 128;
__global__ void __launch_bounds__(kSampleThreads) sample_labels_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t N, int L, int n_pos_needed,
    const uint64_t* __restrict__ seed_dev, uint64_t salt, int32_t* __restrict__ lookup, float* __restrict__ labels) {
  pdl_enter();
  __shared__ int32_t spos[kSampleSmall];       // the row's positives (membership test)
  __shared__ uint32_t sh[kSampleSmall];        // hashes of the rank permutation
  const int b = blockIdx.x;
  const int p0 = rowptr[b], P = rowptr[b + 1] - p0;
  const int32_t* cols = col + p0;
  for (int i = threadIdx.x; i < P && i < kSampleSmall; i += blockDim.x) spos[i] = cols[i];
  __syncthreads();
  // data.py:244-268: all positives when there are at most n_pos_needed of them, otherwise as many as are left after
  // min(N, L - n_pos_needed) negatives; the rest of the row is the prefix of a random permutation of ALL entities
  int n_pos = P;
  if (P > n_pos_needed) {
    const int64_t want_neg = (int64_t)L - n_pos_needed;
    n_pos = L - (int)(want_neg < N ? want_neg : N);
  }
  n_pos = n_pos < P ? n_pos : P;
  n_pos = n_pos < L ? n_pos : L;
  const int n_neg = L - n_pos;
  const uint64_t seed = *seed_dev + salt;
  const uint64_t key_pos = ((uint64_t)hash32(seed, 2 * (uint64_t)b) << 32) | hash32(seed ^ 0x5bd1e995u, 2 * (uint64_t)b);
  const uint64_t key_neg = ((uint64_t)hash32(seed, 2 * (uint64_t)b + 1) << 32) |
                           hash32(seed ^ 0x5bd1e995u, 2 * (uint64_t)b + 1);
  int32_t* lrow = lookup + (int64_t)b * L;
  // positives: tf.random_shuffle(correct_e2s)[:n_pos]
  if (P <= kSampleSmall) {
    rank_permute(sh, P, n_pos, key_pos, [&](int r, int i) { lrow[r] = spos[i]; });
  } else {
    for (int l = threadIdx.x; l < n_pos; l += blockDim.x) lrow[l] = cols[prp((uint32_t)l, (uint32_t)P, key_pos)];
  }
  // sampled entities: tf.random_shuffle(tf.range(num_ent))[:L - n_pos]
  if (N <= kSampleSmall) {
    rank_permute(sh, (int)N, n_neg, key_neg, [&](int r, int i) { lrow[n_pos + r] = i; });
  } else {
    for (int l = threadIdx.x; l < n_neg; l += blockDim.x)
      lrow[n_pos + l] = (int32_t)prp((uint32_t)l, (uint32_t)N, key_neg);
  }
  __syncthreads();
  // labels = gather(dense multi-hot, ids): a sampled entity that is a true tail keeps its label 1
  for (int l = threadIdx.x; l < L; l += blockDim.x) {
    float lab = l < n_pos ? 1.0f : 0.0f;
    if (l >= n_pos) {
      const int32_t id = lrow[l];
      for (int i = 0; i < P; ++i) {
        const int32_t c = i < kSampleSmall ? spos[i] : cols[i];
        if (c == id) lab = 1.0f;
      }
    }
    labels[(int64_t)b * L + l] = lab;
  }
}

struct SampLayout {
  size_t off_loss, off_keys_in, off_keys_out, off_pos_in, off_pos_out, off_cub, cub_bytes, total;
};
// sharded: + the [B*L] local-row sort keys (the unsharded call sorts the lookup ids themselves)
static SampLayout samp_layout(int B, int L, bool sharded = false) {
  SampLayout S;
  const int M = B * L;
  size_t o = 0;
  S.off_loss = o; o = align_up(o + (size_t)B * sizeof(double), 256);
  S.off_keys_out = o; o = align_up(o + (size_t)M * sizeof(int32_t), 256);
  S.off_pos_in = o; o = align_up(o + (size_t)M * sizeof(int32_t), 256);
  S.off_pos_out = o; o = align_up(o + (size_t)M * sizeof(int32_t), 256);
  size_t cb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cb, (const int32_t*)nullptr, (int32_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, M);
  S.cub_bytes = cb;
  S.off_cub = o; o = align_up(o + cb, 256);
  S.off_keys_in = o;
  if (sharded) o = align_up(o + (size_t)M * sizeof(int32_t), 256);
  S.total = o;
  return S;
}

template <bool kShard>
static int score_sampled(const float* q, const float* E, const float* bias, const int32_t* lookup, const float* labels,
                         int B, int L, int64_t N, int d, float one_minus_eps, float inv_num_ent, float inv_count,
                         double* loss_sum, float* scores, float* g, float* dq, float* dE_sum, float* dE_sq,
                         float* dbias_sum, float* dbias_sq, int64_t row_lo, int64_t row_hi, void* workspace,
                         size_t workspace_bytes, cudaStream_t st) {
  SampLayout S = samp_layout(B, L, kShard);
  if (workspace_bytes < S.total) return COPER_ERR_WORKSPACE;
  char* ws = static_cast<char*>(workspace);
  double* loss_part = reinterpret_cast<double*>(ws + S.off_loss);
  int32_t* keys_out = reinterpret_cast<int32_t*>(ws + S.off_keys_out);
  int32_t* pos_in = reinterpret_cast<int32_t*>(ws + S.off_pos_in);
  int32_t* pos_out = reinterpret_cast<int32_t*>(ws + S.off_pos_out);
  launch_pdl(sampled_score_bce_kernel<kShard>, B, kSampWarps * 32, 0, st, q, E, bias, lookup, labels, L, N, d,
             one_minus_eps, inv_num_ent, inv_count, loss_part, scores, g, dq, row_lo, row_hi);
  int rc = check_launch();
  if (rc) return rc;
  launch_pdl(sum_loss_kernel, 1, 256, 0, st, loss_part, B, loss_sum);
  if ((rc = check_launch())) return rc;
  const int M = B * L;
  // sort keys: the global ids (< N), or the local rows with the sentinel row_hi - row_lo (<= rows)
  const int32_t* keys_in = lookup;
  int64_t key_bound = N;
  if constexpr (kShard) {
    int32_t* keys = reinterpret_cast<int32_t*>(ws + S.off_keys_in);
    launch_pdl(sampled_shard_keys_kernel, ceil_div(M, 256), 256, 0, st, lookup, M, row_lo, row_hi, keys, pos_in);
    keys_in = keys;
    key_bound = row_hi - row_lo + 1;
  } else {
    launch_pdl(iota32_kernel, ceil_div(M, 256), 256, 0, st, pos_in, M);
  }
  if ((rc = check_launch())) return rc;
  int end_bit = 1;
  while (end_bit < 31 && (int64_t(1) << end_bit) < key_bound) ++end_bit;
  size_t cb = S.cub_bytes;
  // (radix sort is stable: the slices of a row are summed in position order, in both forms of the call)
  rc = check_cuda(cub::DeviceRadixSort::SortPairs(ws + S.off_cub, cb, keys_in, keys_out, pos_in, pos_out, M, 0, end_bit,
                                                  st));
  if (rc) return rc;
  launch_pdl(sampled_scatter_kernel<kShard>, ceil_div(M, 8), 256, 0, st, keys_out, pos_out, M, L, g, q, d, dE_sum, dE_sq,
             dbias_sum, dbias_sq, (int)(row_hi - row_lo));
  return check_launch();
}
}  // namespace coper

using namespace coper;

extern "C" {

int coper_sample_labels(const int32_t* rowptr, const int32_t* col, int B, int64_t N, int L, int n_pos_needed,
                        const uint64_t* seed_dev, uint64_t salt, int32_t* lookup, float* labels, coper_stream_t stream) {
  COPER_CHECK_ARG(rowptr && col && seed_dev && lookup && labels && B > 0 && L > 0 && n_pos_needed >= 0);
  COPER_CHECK_ARG(N > 0 && N < (int64_t(1) << 31) && (int64_t)L <= N);
  launch_pdl(sample_labels_kernel, B, kSampleThreads, 0, as_stream(stream), rowptr, col, N, L, n_pos_needed,
             seed_dev, salt, lookup, labels);
  return check_launch();
}

size_t coper_score_sampled_workspace_bytes(int B, int L) { return (B <= 0 || L <= 0) ? 256 : samp_layout(B, L).total; }

int coper_score_sampled_bce_fwd_bwd(const float* q, const float* E, const float* bias, const int32_t* lookup,
                                    const float* labels, int B, int L, int64_t N, int d, float one_minus_eps,
                                    float inv_num_ent, float inv_count, double* loss_sum, float* scores, float* g,
                                    float* dq, float* dE_sum, float* dE_sq, float* dbias_sum, float* dbias_sq,
                                    void* workspace, size_t workspace_bytes, coper_stream_t stream) {
  COPER_CHECK_ARG(q && E && bias && lookup && labels && loss_sum && g && dq && dE_sum && dE_sq && dbias_sum && dbias_sq);
  COPER_CHECK_ARG(B > 0 && L > 0 && N > 0 && d > 0 && workspace);
  if (d > 32 * kSampMaxK) return COPER_ERR_UNSUPPORTED;
  return score_sampled<false>(q, E, bias, lookup, labels, B, L, N, d, one_minus_eps, inv_num_ent, inv_count, loss_sum,
                              scores, g, dq, dE_sum, dE_sq, dbias_sum, dbias_sq, 0, N, workspace, workspace_bytes,
                              as_stream(stream));
}

size_t coper_score_sampled_sharded_workspace_bytes(int B, int L) {
  return (B <= 0 || L <= 0) ? 256 : samp_layout(B, L, true).total;
}

int coper_score_sampled_bce_fwd_bwd_sharded(const float* q, const float* E, const float* bias, const int32_t* lookup,
                                            const float* labels, int B, int L, int64_t N, int d, float one_minus_eps,
                                            float inv_num_ent, float inv_count, double* loss_sum, float* scores,
                                            float* g, float* dq, float* dE_sum, float* dE_sq, float* dbias_sum,
                                            float* dbias_sq, int64_t row_lo, int64_t row_hi, void* workspace,
                                            size_t workspace_bytes, coper_stream_t stream) {
  COPER_CHECK_ARG(q && E && bias && lookup && labels && loss_sum && g && dq && dE_sum && dE_sq && dbias_sum && dbias_sq);
  COPER_CHECK_ARG(B > 0 && L > 0 && N > 0 && N < (int64_t(1) << 31) && (int64_t)B * L < (int64_t(1) << 31) && d > 0 &&
                  workspace);
  COPER_CHECK_ARG(row_lo >= 0 && row_hi > row_lo && row_hi <= N);
  if (d > 32 * kSampMaxK) return COPER_ERR_UNSUPPORTED;
  return score_sampled<true>(q, E, bias, lookup, labels, B, L, N, d, one_minus_eps, inv_num_ent, inv_count, loss_sum,
                             scores, g, dq, dE_sum, dE_sq, dbias_sum, dbias_sq, row_lo, row_hi, workspace,
                             workspace_bytes, as_stream(stream));
}

}  // extern "C"
