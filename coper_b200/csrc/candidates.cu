// a8, forward only: the scores of GIVEN candidate entities (models.py:438-443's predictions_lookup for arbitrary
// lookup ids, without the loss and the backward pass of sampled.cu) and the filtered rank of the gold tail among them.
//
// Gather-bound batched mat-vec: every scored position reads one [d] row of E (800 B at d = 200) and q[b] is reused
// across the C candidates of query b.  The grid spreads over (query, candidate chunk); each warp loads the rows of
// kCandGroup candidates before it reduces any of them, so a warp keeps kCandGroup * ceil(d / 32) independent loads in
// flight.  Every dot product is the lane-strided fmaf chain of sampled_score_bce_kernel (element c = lane + 32 k on
// lane `lane`, k = 0..7, zeros beyond d), then warp_sum, then + bias: a scored position is bit-identical to the score
// the sampled-label training step computes for the same q, table and id.
#include "common.cuh"

namespace coper {

constexpr int kCandWarps = 8;
constexpr int kCandGroup = 4;    // candidates per warp in flight
constexpr int kCandMaxK = 8;     // d <= 256: up to 8 strided elements per lane

// The kCandGroup dots of q (qr: this lane's strided elements) with the rows local[0..G) of E; local[g] < 0 reads
// nothing (the dot is then 0 and is not used).  All loads are issued before the first reduction.
__device__ __forceinline__ void group_dots(const float (&qr)[kCandMaxK], const float* __restrict__ E, int d,
                                           const int64_t (&local)[kCandGroup], int lane, float (&dot)[kCandGroup]) {
  float er[kCandGroup][kCandMaxK];
#pragma unroll
  for (int g = 0; g < kCandGroup; ++g) {
    const bool own = local[g] >= 0;                   // warp-uniform
    const float* row = E + (own ? local[g] : 0) * d;
#pragma unroll
    for (int k = 0; k < kCandMaxK; ++k) {
      const int c = lane + 32 * k;
      er[g][k] = (own && c < d) ? __ldg(row + c) : 0.f;
    }
  }
#pragma unroll
  for (int g = 0; g < kCandGroup; ++g) {
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < kCandMaxK; ++k) acc = fmaf(qr[k], er[g][k], acc);
    dot[g] = warp_sum(acc);
  }
}

__device__ __forceinline__ void load_q(const float* __restrict__ q, int b, int d, int lane, float (&qr)[kCandMaxK]) {
#pragma unroll
  for (int k = 0; k < kCandMaxK; ++k) {
    const int c = lane + 32 * k;
    qr[k] = c < d ? __ldg(q + (int64_t)b * d + c) : 0.f;
  }
}

// grid (B, chunks); block nw warps.  Chunk y of query b covers candidate groups y*nw + warp, stepping by
// gridDim.y * nw groups of kCandGroup.
__global__ void __launch_bounds__(kCandWarps * 32, 4) candidate_score_kernel(
    const float* __restrict__ q, const float* __restrict__ E, const float* __restrict__ bias,
    const int32_t* __restrict__ cand, int C, int d, int64_t row_lo, int64_t row_hi, float* __restrict__ scores) {
  pdl_enter();
  const int b = blockIdx.x, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int warp = threadIdx.x >> 5;
  float qr[kCandMaxK];
  load_q(q, b, d, lane, qr);
  const int32_t* crow = cand + (int64_t)b * C;
  float* srow = scores + (int64_t)b * C;
  for (int64_t j0 = ((int64_t)blockIdx.y * nw + warp) * kCandGroup; j0 < C;
       j0 += (int64_t)gridDim.y * nw * kCandGroup) {
    // lane g < G holds candidate j0 + g
    int64_t mine = -1;
    if (lane < kCandGroup && j0 + lane < C) {
      const int64_t id = crow[j0 + lane];
      if (id >= row_lo && id < row_hi) mine = id - row_lo;
    }
    int64_t local[kCandGroup];
#pragma unroll
    for (int g = 0; g < kCandGroup; ++g) local[g] = __shfl_sync(0xffffffffu, mine, g);
    float s = 0.f;                                    // non-owned, padding and out-of-range positions: exactly 0
    // (the vote makes the group's branch visibly warp-uniform, as in candidate_rank_kernel: without it the compiler
    // emits a second, warp-synchronised copy of the loop body and the kernel gathers at half the rank kernel's rate)
    if (__any_sync(0xffffffffu, mine >= 0)) {
      const float bv = mine >= 0 ? __ldg(bias + mine) : 0.f;
      float dot[kCandGroup];
      group_dots(qr, E, d, local, lane, dot);
#pragma unroll
      for (int g = 0; g < kCandGroup; ++g)
        if (lane == g && mine >= 0) s = dot[g] + bv;
    }
    if (lane < kCandGroup && j0 + lane < C) srow[j0 + lane] = s;
  }
}

// Same walk; a position counts when the shard owns it, it is not the gold entity and its filter bit is clear.  Only
// those positions read a row.  bits: query-major [B, ceil(rows/32)] (entity_major = 0) or entity-major
// [rows, ceil(B/32)] (entity_major = 1), NULL = unfiltered.
__global__ void __launch_bounds__(kCandWarps * 32, 4) candidate_rank_kernel(
    const float* __restrict__ q, const float* __restrict__ E, const float* __restrict__ bias,
    const int32_t* __restrict__ cand, const int32_t* __restrict__ e2, int B, int C, int d, int64_t row_lo,
    int64_t row_hi, const float* __restrict__ gold, const uint32_t* __restrict__ bits, int entity_major,
    int32_t* __restrict__ n_greater, int32_t* __restrict__ n_equal) {
  pdl_enter();
  __shared__ int sm_g[kCandWarps], sm_e[kCandWarps];
  const int b = blockIdx.x, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int warp = threadIdx.x >> 5;
  float qr[kCandMaxK];
  load_q(q, b, d, lane, qr);
  const int32_t* crow = cand + (int64_t)b * C;
  const int64_t gold_id = e2[b];
  const float gv = gold[b];
  const int64_t rows = row_hi - row_lo;
  const int64_t words_q = (rows + 31) >> 5, words_e = (B + 31) >> 5;
  int cg = 0, ce = 0;
  for (int64_t j0 = ((int64_t)blockIdx.y * nw + warp) * kCandGroup; j0 < C;
       j0 += (int64_t)gridDim.y * nw * kCandGroup) {
    int64_t mine = -1;
    if (lane < kCandGroup && j0 + lane < C) {
      const int64_t id = crow[j0 + lane];
      if (id >= row_lo && id < row_hi && id != gold_id) {
        const int64_t n = id - row_lo;
        bool filtered = false;
        if (bits) {
          const uint32_t w = entity_major ? __ldg(bits + n * words_e + (b >> 5)) : __ldg(bits + b * words_q + (n >> 5));
          filtered = (w >> (entity_major ? (b & 31) : (int)(n & 31))) & 1u;
        }
        if (!filtered) mine = n;
      }
    }
    int64_t local[kCandGroup];
#pragma unroll
    for (int g = 0; g < kCandGroup; ++g) local[g] = __shfl_sync(0xffffffffu, mine, g);
    if (!__any_sync(0xffffffffu, mine >= 0)) continue;   // nothing of this group counts here
    const float bv = mine >= 0 ? __ldg(bias + mine) : 0.f;
    float dot[kCandGroup];
    group_dots(qr, E, d, local, lane, dot);
#pragma unroll
    for (int g = 0; g < kCandGroup; ++g) {
      if (lane == g && mine >= 0) {
        const float s = dot[g] + bv;
        cg += s > gv;
        ce += s == gv;
      }
    }
  }
  cg = warp_sum_i(cg);
  ce = warp_sum_i(ce);
  if (lane == 0) { sm_g[warp] = cg; sm_e[warp] = ce; }
  __syncthreads();
  if (threadIdx.x == 0) {
    int tg = 0, te = 0;
    for (int w = 0; w < nw; ++w) { tg += sm_g[w]; te += sm_e[w]; }
    if (tg) atomicAdd(n_greater + b, tg);
    if (te) atomicAdd(n_equal + b, te);
  }
}

// Warps per CTA and candidate chunks per query: the largest CTA (<= kCandWarps warps, no more warps than candidate
// groups) that still gives every SM a few CTAs, then as many chunks per query as keep ~32 CTAs per SM in the grid -
// B = 1 spreads over the SMs, B = 512 gives each warp a few groups to amortise its q load.
static void cand_grid(int B, int C, dim3& grid, int& threads) {
  const int64_t groups = (C + kCandGroup - 1) / kCandGroup;
  const int64_t target = 2 * (int64_t)sm_count();
  int nw = kCandWarps;
  while (nw > 1 && (nw / 2 >= groups || (int64_t)B * ((groups + nw - 1) / nw) < target)) nw /= 2;
  const int64_t per_query = (groups + nw - 1) / nw;
  const int64_t want = (16 * target + B - 1) / B;
  int64_t chunks = per_query < want ? per_query : want;
  if (chunks > 65535) chunks = 65535;
  if (chunks < 1) chunks = 1;
  grid = dim3((unsigned)B, (unsigned)chunks);
  threads = nw * 32;
}

static int check_cand_args(int B, int C, int d, int64_t row_lo, int64_t row_hi) {
  if (B < 1 || C < 1 || (int64_t)B * C >= (int64_t(1) << 31)) return COPER_ERR_INVALID_ARG;
  if (row_lo < 0 || row_hi <= row_lo || row_hi >= (int64_t(1) << 31)) return COPER_ERR_INVALID_ARG;
  if (d < 1) return COPER_ERR_INVALID_ARG;
  if (d > 32 * kCandMaxK) return COPER_ERR_UNSUPPORTED;
  return COPER_OK;
}
}  // namespace coper

using namespace coper;

extern "C" {

int coper_score_candidates(const float* q, const float* E, const float* bias, const int32_t* cand, int B, int C, int d,
                           int64_t row_lo, int64_t row_hi, float* scores, coper_stream_t stream) {
  COPER_CHECK_ARG(q && E && bias && cand && scores);
  const int rc = check_cand_args(B, C, d, row_lo, row_hi);
  if (rc) return rc;
  dim3 grid;
  int threads;
  cand_grid(B, C, grid, threads);
  launch_pdl(candidate_score_kernel, grid, threads, 0, as_stream(stream), q, E, bias, cand, C, d, row_lo, row_hi,
             scores);
  return check_launch();
}

int coper_candidate_rank(const float* q, const float* E, const float* bias, const int32_t* cand, const int32_t* e2,
                         int B, int C, int d, int64_t row_lo, int64_t row_hi, const float* gold,
                         const uint32_t* filter_bits, int entity_major, int32_t* n_greater, int32_t* n_equal,
                         coper_stream_t stream) {
  COPER_CHECK_ARG(q && E && bias && cand && e2 && gold && n_greater && n_equal);
  COPER_CHECK_ARG(entity_major == 0 || entity_major == 1);
  const int rc = check_cand_args(B, C, d, row_lo, row_hi);
  if (rc) return rc;
  dim3 grid;
  int threads;
  cand_grid(B, C, grid, threads);
  launch_pdl(candidate_rank_kernel, grid, threads, 0, as_stream(stream), q, E, bias, cand, e2, B, C, d, row_lo,
             row_hi, gold, filter_bits, entity_major, n_greater, n_equal);
  return check_launch();
}

}  // extern "C"
