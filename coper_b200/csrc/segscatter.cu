// a10 scatter / K8(3): gradient of tf.nn.embedding_lookup (models.py:176-180, IndexedSlices made dense at
// models.py:198).  Duplicate head entities / relations in a batch make this a segmented reduction:
//   1. stable radix sort of (row id, position) pairs (cub::DeviceRadixSort — library plumbing),
//   2. one warp per segment head: lanes stride the embedding width (coalesced 128 B row reads), the warp
//      walks its segment in sorted (= original, the sort is stable) order and issues ONE read-modify-write
//      of the destination row.  No atomics, fixed summation order -> bit-reproducible.
// HBM-bound: M*w*4 B read + 2*rows_touched*w*4 B RMW + 8 M B of indices.
#include <cub/device/device_radix_sort.cuh>
#include "common.cuh"

namespace coper {

__global__ void iota_kernel(int32_t* p, int n) {
  pdl_enter();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}

__global__ void segscatter_kernel(const int64_t* __restrict__ keys, const int32_t* __restrict__ pos, int M,
                                  const float* __restrict__ src, int width, float* __restrict__ dst, int64_t row_lo,
                                  int64_t row_hi) {
  pdl_enter();
  int seg = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // candidate head position
  int lane = threadIdx.x & 31;
  if (seg >= M) return;
  int64_t key = keys[seg];
  if (seg > 0 && keys[seg - 1] == key) return;  // not a segment head
  if (key < row_lo || key >= row_hi) return;    // row owned by another shard
  int end = seg + 1;
  while (end < M && keys[end] == key) ++end;
  float* drow = dst + (key - row_lo) * (int64_t)width;
  for (int c = lane; c < width; c += 32) {
    float acc = 0.f;
    for (int i = seg; i < end; ++i) acc += __ldg(src + (int64_t)pos[i] * width + c);
    drow[c] += acc;
  }
}

// Small-M path (M <= kSegSmallM: the e1 / rel gathers of one batch): no sort at all.  One warp per position i; the
// warp scans the index array (M/32 coalesced steps) to see whether an earlier position holds the same row - then it is
// not a segment head and exits - and otherwise sums every later member of its row in INDEX order (the order a stable
// sort would give): same result bit for bit as the sorted path, one launch, no workspace.
// dst_sq (optional): sum of the SQUARED source rows per destination row (the IndexedSlices bookkeeping).
constexpr int kSegSmallM = COPER_SEGSCATTER_SMALL_M;
// norm_delta (optional, [M] doubles): position i receives sum_c (new_c^2 - old_c^2) of the destination row it updated
// (0 if it is not a segment head / not owned) - the correction that turns a sum of squares taken BEFORE the scatter
// (by the kernel that produced dst) into the sum of squares of the final gradient.
struct SegSmallJob {
  const int64_t* idx;
  int M;
  const float* src;
  int width;
  float* dst;
  float* dst_sq;
  int64_t row_lo, row_hi;
  double* norm_delta;
};
__device__ __forceinline__ void segscatter_small_warp(const int64_t* __restrict__ idx, int M,
                                                      const float* __restrict__ src, int width, float* __restrict__ dst,
                                                      float* __restrict__ dst_sq, int64_t row_lo, int64_t row_hi,
                                                      double* __restrict__ norm_delta, int block) {
  const int i = block * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= M) return;
  if (norm_delta && lane == 0) norm_delta[i] = 0.0;
  const int64_t key = idx[i];
  if (key < row_lo || key >= row_hi) return;
  float* drow = dst + (key - row_lo) * (int64_t)width;
  float* qrow = dst_sq ? dst_sq + (key - row_lo) * (int64_t)width : nullptr;
  double delta = 0.0;
  // ONE scan of the index array per 256-column pass (a single pass for every shipped width): positions before i only
  // decide whether an earlier position owns this row; positions from i on are the members, added in index order.
  // 8 columns per lane, so the source loads of a member and the destination loads are each one round trip.
  for (int c0 = 0; c0 < width; c0 += 32 * 8) {
    float a[8], q[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = q[k] = 0.f;
    for (int j0 = 0; j0 < M; j0 += 32) {
      const int j = j0 + lane;
      uint32_t m = __ballot_sync(0xffffffffu, j < M && __ldg(idx + j) == key);
      if (j0 + 32 <= i) {                              // every position of this group precedes i
        if (m) return;                                 // an earlier position owns this row
        continue;
      }
      if (j0 <= i) {                                   // the group that holds i
        if (m & ((1u << (i - j0)) - 1u)) return;
        m &= ~((1u << (i - j0)) - 1u);
      }
      while (m) {
        const int jj = j0 + __ffs(m) - 1;
        m &= m - 1;
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int c = c0 + lane + 32 * k;
          v[k] = c < width ? __ldg(src + (int64_t)jj * width + c) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          a[k] += v[k];
          q[k] = fmaf(v[k], v[k], q[k]);
        }
      }
    }
    float old[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = c0 + lane + 32 * k;
      old[k] = c < width ? drow[c] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = c0 + lane + 32 * k;
      if (c < width) {
        const float nw = old[k] + a[k];
        drow[c] = nw;
        delta += (double)nw * (double)nw - (double)old[k] * (double)old[k];
        if (qrow) qrow[c] += q[k];
      }
    }
  }
  if (norm_delta) {
    delta = warp_sum_d(delta);
    if (lane == 0) norm_delta[i] = delta;
  }
}
// Small TABLE (the relation embedding: tens to hundreds of rows, each hit by many positions of the batch): one block per
// table row.  The block lists the positions that hold its row in index order (ballot compaction), then every thread owns
// columns and adds the members in that order with the loads of 8 members in flight.  Same sums in the same order as
// segscatter_small_warp - where one warp walks its 20+ members one dependent L2 round trip at a time.
constexpr int kSegRowOwnerRows = 2048;
__device__ __forceinline__ void segscatter_row_block(const SegSmallJob& J, int row, uint16_t* list, int* warp_cnt,
                                                     int* base) {
  const int64_t key = J.row_lo + row;
  const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) *base = 0;
  __syncthreads();
  for (int j0 = 0; j0 < J.M; j0 += 256) {
    const int j = j0 + tid;
    const bool hit = j < J.M && __ldg(J.idx + j) == key;
    const uint32_t m = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) warp_cnt[warp] = __popc(m);
    __syncthreads();
    int off = *base;
    for (int w = 0; w < warp; ++w) off += warp_cnt[w];
    if (hit) list[off + __popc(m & ((1u << lane) - 1u))] = (uint16_t)j;
    __syncthreads();
    if (tid == 0) {
      int t = 0;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += warp_cnt[w];
      *base += t;
    }
    __syncthreads();
  }
  const int cnt = *base;
  if (cnt == 0) return;
  for (int c = tid; c < J.width; c += 256) {
    float a = 0.f, q = 0.f;
    int m = 0;
    for (; m + 8 <= cnt; m += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldg(J.src + (int64_t)list[m + u] * J.width + c);
#pragma unroll
      for (int u = 0; u < 8; ++u) { a += v[u]; q = fmaf(v[u], v[u], q); }
    }
    for (; m < cnt; ++m) {
      const float v = __ldg(J.src + (int64_t)list[m] * J.width + c);
      a += v;
      q = fmaf(v, v, q);
    }
    float* d = J.dst + (int64_t)row * J.width + c;
    *d = *d + a;
    if (J.dst_sq) J.dst_sq[(int64_t)row * J.width + c] += q;
  }
}
// blocks [0, blocks_a) run job A, the rest job B (two independent scatters of one step - head entities and
// relations - in one launch; B.M == 0: single job).  b_row_owner: job B runs one block per table row.
__global__ void __launch_bounds__(256) segscatter_small_kernel(SegSmallJob A, int blocks_a, SegSmallJob Bj,
                                                               int b_row_owner) {
  pdl_enter();
  __shared__ uint16_t list[kSegSmallM];
  __shared__ int warp_cnt[8];
  __shared__ int base;
  if ((int)blockIdx.x < blocks_a)
    segscatter_small_warp(A.idx, A.M, A.src, A.width, A.dst, A.dst_sq, A.row_lo, A.row_hi, A.norm_delta, (int)blockIdx.x);
  else if (b_row_owner)
    segscatter_row_block(Bj, (int)blockIdx.x - blocks_a, list, warp_cnt, &base);
  else
    segscatter_small_warp(Bj.idx, Bj.M, Bj.src, Bj.width, Bj.dst, Bj.dst_sq, Bj.row_lo, Bj.row_hi, Bj.norm_delta,
                          (int)blockIdx.x - blocks_a);
}

struct SegLayout {
  size_t off_keys_out, off_pos_in, off_pos_out, off_cub, cub_bytes, total;
};
static SegLayout seg_layout(int M) {
  SegLayout L;
  size_t o = 0;
  L.off_keys_out = o; o = align_up(o + (size_t)M * sizeof(int64_t), 256);
  L.off_pos_in = o; o = align_up(o + (size_t)M * sizeof(int32_t), 256);
  L.off_pos_out = o; o = align_up(o + (size_t)M * sizeof(int32_t), 256);
  size_t cb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cb, (const int64_t*)nullptr, (int64_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, M);
  L.cub_bytes = cb;
  L.off_cub = o; o = align_up(o + cb, 256);
  L.total = o;
  return L;
}
}  // namespace coper

using namespace coper;

extern "C" {

size_t coper_segscatter_workspace_bytes(int M) { return M <= 0 ? 256 : seg_layout(M).total; }

int coper_segscatter_add_sq(const int64_t* idx, int M, const float* src, int width, float* dst, float* dst_sq,
                            int64_t row_lo, int64_t row_hi, coper_stream_t stream) {
  COPER_CHECK_ARG(idx && src && dst && M >= 0 && width > 0 && row_hi >= row_lo);
  if (M > kSegSmallM) return COPER_ERR_UNSUPPORTED;
  if (M == 0) return COPER_OK;
  SegSmallJob A{idx, M, src, width, dst, dst_sq, row_lo, row_hi, nullptr};
  launch_pdl(segscatter_small_kernel, ceil_div(M, 8), 256, 0, as_stream(stream), A, ceil_div(M, 8), SegSmallJob{}, 0);
  return check_launch();
}

int coper_segscatter_add_pair(const int64_t* idx_a, int M_a, const float* src_a, int width_a, float* dst_a,
                              float* dst_sq_a, int64_t lo_a, int64_t hi_a, double* norm_delta_a, const int64_t* idx_b,
                              int M_b, const float* src_b, int width_b, float* dst_b, float* dst_sq_b, int64_t lo_b,
                              int64_t hi_b, coper_stream_t stream) {
  COPER_CHECK_ARG(idx_a && src_a && dst_a && M_a > 0 && width_a > 0 && hi_a >= lo_a);
  COPER_CHECK_ARG(M_b == 0 || (idx_b && src_b && dst_b && M_b > 0 && width_b > 0 && hi_b >= lo_b));
  if (M_a > kSegSmallM || M_b > kSegSmallM) return COPER_ERR_UNSUPPORTED;
  SegSmallJob A{idx_a, M_a, src_a, width_a, dst_a, dst_sq_a, lo_a, hi_a, norm_delta_a};
  SegSmallJob Bj{idx_b, M_b, src_b, width_b, dst_b, dst_sq_b, lo_b, hi_b, nullptr};
  const int row_owner = M_b > 0 && hi_b - lo_b <= kSegRowOwnerRows && hi_b > lo_b;
  const int ba = ceil_div(M_a, 8), bb = row_owner ? (int)(hi_b - lo_b) : ceil_div(M_b, 8);
  launch_pdl(segscatter_small_kernel, ba + bb, 256, 0, as_stream(stream), A, ba, Bj, row_owner);
  return check_launch();
}

int coper_segscatter_add(const int64_t* idx, int M, const float* src, int width, float* dst, int64_t row_lo,
                         int64_t row_hi, void* workspace, size_t workspace_bytes, coper_stream_t stream) {
  COPER_CHECK_ARG(idx && src && dst && workspace && M >= 0 && width > 0 && row_hi >= row_lo);
  if (M == 0) return COPER_OK;
  if (M <= kSegSmallM) return coper_segscatter_add_sq(idx, M, src, width, dst, nullptr, row_lo, row_hi, stream);
  SegLayout L = seg_layout(M);
  if (workspace_bytes < L.total) return COPER_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  char* ws = static_cast<char*>(workspace);
  int64_t* keys_out = reinterpret_cast<int64_t*>(ws + L.off_keys_out);
  int32_t* pos_in = reinterpret_cast<int32_t*>(ws + L.off_pos_in);
  int32_t* pos_out = reinterpret_cast<int32_t*>(ws + L.off_pos_out);
  launch_pdl(iota_kernel, ceil_div(M, 256), 256, 0, st, pos_in, M);
  int rc = check_launch();
  if (rc) return rc;
  size_t cb = L.cub_bytes;
  rc = check_cuda(cub::DeviceRadixSort::SortPairs(ws + L.off_cub, cb, idx, keys_out, pos_in, pos_out, M, 0, 64, st));
  if (rc) return rc;
  launch_pdl(segscatter_kernel, ceil_div(M, 8), 256, 0, st, keys_out, pos_out, M, src, width, dst, row_lo, row_hi);
  return check_launch();
}

}  // extern "C"
