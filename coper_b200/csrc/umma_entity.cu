// Entity-major tcgen05 scorer family (a7 / a9 / a10 / a11: models.py:433-437, 448-453, 198; metrics.py:44-51).
//
// The 1-N score tile is computed TRANSPOSED:  D[n, b] = E[n,:] . q[b,:]  — the entity table is the A operand (TMEM
// lanes = entities, one entity per epilogue thread), the query block is the B operand (TMEM columns = queries).
// Everything that is per-entity then lives in a register of the thread that owns the entity row:
//   * pred_bias[n] is one register per tile (no per-element load),
//   * dbias[n] = sum_b G[b,n] is a thread-local sum (no cross-lane reduction),
//   * label / filter bits come from the entity-major bit matrix bitsT [Ns, ceil(B/32)] — one word per thread per
//     32-query chunk, prefetched one tile ahead together with the bias,
//   * stores of G[b, n] / S[b, n] are coalesced: for a fixed query column the 32 lanes write 32 consecutive entities.
// Rank counts per query are accumulated across the warp's 32 entities with a ballot + popc per column.
//
// Three epilogues share the pipeline (umma_gemm.cuh):  ScoreEpiT (logits out), BceEpiT (loss + G + dbias partials),
// RankEpiT (filtered-rank counts; logits never leave TMEM) plus DiagEpiT for the bit-identical gold logits.
#include <cuda_fp16.h>
#include "umma_gemm.cuh"
#include "bce_math.cuh"

namespace coper {
using namespace umma;

size_t tc_prepared_bytes(int64_t rows, int cols, int prec);                     // umma_score.cu
int tc_prepare(const float* src, int64_t rows, int cols, int64_t ld_src, int prec, void* dst, cudaStream_t st);
int64_t tc_prepared_ld(int cols, int prec);
TcOperand tc_operand(const void* prep, int64_t rows, int cols, int prec);       // umma_gemm.cu
void* tc_fp16x3_trailer(const void* prep, int64_t rows, int cols);
int tc_gemm_store(int prec, bool a_mn, bool b_mn, const TcOperand& A, const TcOperand& B, const GemmProblem& p,
                  bool split, const StoreEpi& epi, cudaStream_t st);
int tc_plan_splits(int prec, GemmProblem p, bool split);
// fused scorer + BCE + dq kernel (umma_fused.cu)
bool umma_fused_ok(int B, int64_t Ns, int d, int prec);
void umma_fused_plan(int B, int64_t Ns, int* QB, int* R);
int umma_bce_dq_fused(const TcOperand& E, const TcOperand& Q, const float* bias, const uint32_t* bitsT, int B, int64_t Ns,
                      int d, float pos, float neg, float inv_count, void* GT, int64_t ldGT, float* dq_part,
                      float* dbias_part, double* loss_part, int* grid_out, cudaStream_t st);

constexpr int kEntEpiWarps = 16;
constexpr int kBceEpiWarps = 16;   // the BCE epilogue is MUFU / latency bound: 4 warps per scheduler

// ------------------------------------------------------------------------------------------ shared per-row state
// bias + bit words of the current tile, and the same for the next tile (loaded one tile ahead)
template <int NCH>
struct RowState {
  const float* bias;        // [M]
  const uint32_t* bitsT;    // [M, wordsB]  (may be NULL: no bits needed)
  int wordsB;
  float bias_cur, bias_nx;
  uint32_t w_cur[NCH], w_nx[NCH];
  int nx_row, nx_col0;
  __device__ __forceinline__ void load(const GemmProblem& p, int row, int col0, float& b, uint32_t (&w)[NCH]) const {
    // rows >= M are clamped (their values are never used: every consumer masks padded rows itself); the loads are
    // unconditional so that nothing depends on them until the next tile consumes the registers
    const int rc = min(row, p.M - 1);
    b = __ldg(bias + rc);
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int col = min(col0 + i * 32, ((p.N - 1) >> 5) << 5);
      w[i] = bitsT ? __ldg(bitsT + (int64_t)rc * wordsB + (col >> 5)) : 0u;
    }
  }
  __device__ __forceinline__ void begin(const GemmProblem& p, int row, int col0) {
    if (nx_row == row && nx_col0 == col0) {
      bias_cur = bias_nx;
#pragma unroll
      for (int i = 0; i < NCH; ++i) w_cur[i] = w_nx[i];
    } else {
      load(p, row, col0, bias_cur, w_cur);
    }
  }
  __device__ __forceinline__ void prefetch(const GemmProblem& p, int row, int col0) {
    load(p, row, col0, bias_nx, w_nx);
    nx_row = row;
    nx_col0 = col0;
  }
  __host__ void init(const float* bias_, const uint32_t* bitsT_, int wordsB_) {
    bias = bias_; bitsT = bitsT_; wordsB = wordsB_;
    bias_cur = bias_nx = 0.f;
    nx_row = nx_col0 = -1;
    for (int i = 0; i < NCH; ++i) w_cur[i] = w_nx[i] = 0;
  }
};

// ------------------------------------------------------------------------------------------ logits out
template <int NCH>
struct ScoreEpiT : EpiBase {
  RowState<NCH> rs;
  float* out;               // S[b, n]: [N, ld]
  int64_t ld;
  __device__ __forceinline__ void tile_begin(const GemmProblem& p, const TileCoord&, int row, int col0) { rs.begin(p, row, col0); }
  __device__ __forceinline__ void tile_prefetch(const GemmProblem& p, const TileCoord&, int row, int col0) { rs.prefetch(p, row, col0); }
  __device__ __forceinline__ void chunk(const GemmProblem& p, const TileCoord&, int row, int col, const uint32_t (&r)[32],
                                        int) const {
    if (row >= p.M) return;
    float* o = out + (int64_t)col * ld + row;
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (col + j < p.N) o[(int64_t)j * ld] = __uint_as_float(r[j]) + rs.bias_cur;
  }
};

// ------------------------------------------------------------------------------------------ BCE + gradient
// dL/dS is written ENTITY-MAJOR:  GT[n, b]  (bf16 [M, ldGT], or tf32 hi / lo planes fp32 [M, ldGT]) - the thread that
// owns entity n writes its 32 consecutive queries as 16-byte vectors, no per-element address arithmetic.  The dq / dE
// GEMMs read GT through TMA as an MN-major (dq) / K-major (dE) A operand.
// Positives are sparse (a few per query out of N): the dense loop treats every element as a negative (no bit test) and
// chunks that do contain a positive (warp vote) take the general path.
template <int PREC, int NCH>
struct BceEpiT : EpiBase {
  RowState<NCH> rs;
  float pos, neg, inv_count;  // inv_count: factor applied to g (fp16x3: 2^10, the true 1/count is applied downstream)
  float rsum_scale;           // dbias = rsum_scale * sum g  (1 unless fp16x3)
  void* GT;                 // bf16 [M, ldGT] | fp16 hi plane [M, ldGT] + lo plane | fp32 hi plane [N, ldGT] + lo plane
  int64_t ldGT;             // >= N, multiple of 8 (bf16) / 4 (tf32)
  float* dbias_part;        // [n_tiles * col_groups][M]
  double* loss_part;        // [grid * epi_warps]
  double loss_acc;
  float rsum;
  __device__ __forceinline__ void tile_begin(const GemmProblem& p, const TileCoord&, int row, int col0) {
    rs.begin(p, row, col0);
    rsum = 0.f;
  }
  __device__ __forceinline__ void tile_prefetch(const GemmProblem& p, const TileCoord&, int row, int col0) { rs.prefetch(p, row, col0); }

  // GENERAL: label bits and the column-valid mask vm are honoured; otherwise every element is a negative and all 32
  // columns exist.  g[j] = (sigmoid(s) - z') * inv_count, 0 for columns that do not exist; gsum = sum_j g[j];
  // lsum = sum_j of the per-element loss (tf.nn.sigmoid_cross_entropy_with_logits, unscaled).
  template <bool GENERAL>
  __device__ __forceinline__ void body(const uint32_t (&r)[32], uint32_t w, uint32_t vm, float (&g)[32], float& lsum,
                                       float& gsum) const {
    if (GENERAL) {
      bce_chunk_general(r, rs.bias_cur, w, vm, pos, neg, inv_count, g, lsum, gsum);
    } else {
      bce_chunk_dense(r, rs.bias_cur, neg, inv_count, g, lsum, gsum);
    }
  }
  __device__ __forceinline__ void chunk(const GemmProblem& p, const TileCoord&, int row, int col, const uint32_t (&r)[32],
                                        int ci) {
    const bool rowok = row < p.M;
    const int ncol = p.N - col;                        // warp-uniform; < 32 only in the last query chunk
    const uint32_t vm = ncol >= 32 ? 0xFFFFFFFFu : ((1u << ncol) - 1u);
    const uint32_t w = rowok ? (rs.w_cur[ci] & vm) : 0u;
    float g[32];
    float lsum, gsum;
    if (ncol < 32 || __any_sync(0xffffffffu, w != 0u)) body<true>(r, w, vm, g, lsum, gsum);
    else body<false>(r, w, vm, g, lsum, gsum);
    uint4 pk[4];
    uint4 pk2[4];
    if (rowok) {
      loss_acc += (double)lsum;
      rsum += gsum * rsum_scale;
      if (PREC == PREC_FP16X3) {
        // (sigmoid - z') * 2^10 as fp16 hi / lo planes, entity-major like the bf16 path
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float a = g[8 * v + 2 * k], b = g[8 * v + 2 * k + 1];
            const __half2 h = __floats2half2_rn(a, b);
            const float2 hf = __half22float2(h);
            const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
            hw[k] = *reinterpret_cast<const uint32_t*>(&h);
            lw[k] = *reinterpret_cast<const uint32_t*>(&l);
          }
          pk[v] = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          pk2[v] = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      } else if (PREC == PREC_BF16) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          __nv_bfloat162 t0 = __floats2bfloat162_rn(g[8 * v], g[8 * v + 1]);
          __nv_bfloat162 t1 = __floats2bfloat162_rn(g[8 * v + 2], g[8 * v + 3]);
          __nv_bfloat162 t2 = __floats2bfloat162_rn(g[8 * v + 4], g[8 * v + 5]);
          __nv_bfloat162 t3 = __floats2bfloat162_rn(g[8 * v + 6], g[8 * v + 7]);
          pk[v].x = *reinterpret_cast<uint32_t*>(&t0); pk[v].y = *reinterpret_cast<uint32_t*>(&t1);
          pk[v].z = *reinterpret_cast<uint32_t*>(&t2); pk[v].w = *reinterpret_cast<uint32_t*>(&t3);
        }
      } else if (PREC == PREC_TF32X3) {
        // tf32x3: 8 bytes per element in two planes - QUERY-major G[b, n] so that every store instruction of the warp
        // covers 32 consecutive entities (128 B); ldGT is the [N, ld] pitch here
        float* hi = static_cast<float*>(GT) + (int64_t)col * ldGT + row;
        float* lo = hi + (int64_t)p.N * ldGT;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          if (j < ncol) {
            uint32_t hb;
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(g[j]));
            *hi = __uint_as_float(hb);
            *lo = g[j] - __uint_as_float(hb);
          }
          hi += ldGT;
          lo += ldGT;
        }
      }
    }
    if (PREC == PREC_BF16 || PREC == PREC_FP16X3) {
      // stage the warp's [32 entities x 32 queries] 16-bit block (64 B per row) through shared memory so that every
      // store instruction writes 8 rows x 64 contiguous bytes (full sectors) instead of 32 rows x 16 bytes
      __shared__ uint4 stage_g[kBceEpiWarps][128];
      uint4* st = stage_g[(threadIdx.x >> 5) - 4];
      const int lane = threadIdx.x & 31;
      const int row0 = row - lane;
      const int64_t ld16 = ldGT / 8;                    // row pitch in 16-byte units
      const int gq = lane & 3;
#pragma unroll
      for (int plane = 0; plane < (PREC == PREC_FP16X3 ? 2 : 1); ++plane) {
#pragma unroll
        for (int v = 0; v < 4; ++v) st[lane * 4 + (v ^ ((lane >> 1) & 3))] = plane ? pk2[v] : pk[v];
        __syncwarp();
        uint4* o0 = reinterpret_cast<uint4*>(static_cast<uint16_t*>(GT) + ((int64_t)plane * p.M + row0) * ldGT + col);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int rr = 8 * k + (lane >> 2);
          const uint4 x = st[rr * 4 + (gq ^ ((rr >> 1) & 3))];
          if (row0 + rr < p.M) o0[(int64_t)rr * ld16 + gq] = x;   // the pitch is padded to 32 queries: whole chunks writable
        }
        __syncwarp();
      }
    }
  }
  __device__ __forceinline__ void tile_done(const GemmProblem& p, const TileCoord& t, int row, int col_group, int col_groups) {
    if (row < p.M) dbias_part[(int64_t)(t.n_blk * col_groups + col_group) * p.M + row] = rsum;
  }
  __device__ __forceinline__ void finish(int epi_thread, int epi_threads) {
    double t = warp_sum_d(loss_acc);
    if ((epi_thread & 31) == 0) loss_part[(int64_t)blockIdx.x * (epi_threads >> 5) + (epi_thread >> 5)] = t;
  }
};

// ------------------------------------------------------------------------------------------ filtered rank counts
// Per element: s = acc + bias_n, then two compares against the query's gold logit (broadcast from a per-warp shared
// memory copy) set bit j of two 32-bit masks.  The filter word is applied to the masks once per chunk.  The "greater"
// mask is accumulated into BIT-SLICED vertical counters (plane k holds bit k of 32 independent column counters) -
// 2 logic ops per plane per 32 elements - and only converted to per-query integers (ballot + popc) when the counters
// could overflow or the CTA moves to another query block.  Ties are rare: they take a ballot path when any occur.
constexpr int kRankPlanes = 8;
template <int NCH>
struct RankEpiT : EpiBase {
  RowState<NCH> rs;
  const float* gold;        // [N]
  int32_t* n_greater;       // [N] accumulated
  int32_t* n_equal;
  uint32_t planes[NCH][kRankPlanes];
  int ce[NCH];              // lane j: ties of column chunk*32 + j
  int cur_col0, n_queries, adds;
  __device__ __forceinline__ float* gold_smem() {
    __shared__ float gold_s[kEntEpiWarps][NCH * 32];
    return gold_s[(threadIdx.x >> 5) - 4];
  }
  __device__ __forceinline__ void flush() {
    const int lane = threadIdx.x & 31;
    if (cur_col0 >= 0) {
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        // this thread's 32 column counters as integers, then a transposing warp reduction:
        // lane j <- count of column i*32 + j summed over the warp's 32 entity rows
        int v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          int c = 0;
#pragma unroll
          for (int k = 0; k < kRankPlanes; ++k) c |= (int)((planes[i][k] >> j) & 1u) << k;
          v[j] = c;
        }
#pragma unroll
        for (int k = 0; k < kRankPlanes; ++k) planes[i][k] = 0;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
          const bool upper = (lane & off) != 0;
#pragma unroll
          for (int q = 0; q < off; ++q) {
            const int send = upper ? v[q] : v[q + off];
            const int keepv = upper ? v[q + off] : v[q];
            v[q] = keepv + __shfl_xor_sync(0xffffffffu, send, off);
          }
        }
        const int cnt = v[0];
        const int col = cur_col0 + i * 32 + lane;
        if (col < n_queries) {
          if (cnt) atomicAdd(n_greater + col, cnt);
          if (ce[i]) atomicAdd(n_equal + col, ce[i]);
        }
        ce[i] = 0;
      }
    }
    adds = 0;
  }
  __device__ __forceinline__ void tile_begin(const GemmProblem& p, const TileCoord&, int row, int col0) {
    if (col0 != cur_col0 || adds >= (1 << kRankPlanes) - 1) {
      const bool reload = col0 != cur_col0;
      flush();
      cur_col0 = col0;
      if (reload) {
        float* gs = gold_smem();
        const int lane = threadIdx.x & 31;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          const int c = col0 + k * 32 + lane;
          gs[k * 32 + lane] = c < p.N ? __ldg(gold + c) : 0.f;
        }
        __syncwarp();
      }
    }
    rs.begin(p, row, col0);
  }
  __device__ __forceinline__ void tile_prefetch(const GemmProblem& p, const TileCoord&, int row, int col0) { rs.prefetch(p, row, col0); }
  __device__ __forceinline__ void chunk(const GemmProblem& p, const TileCoord&, int row, int, const uint32_t (&r)[32], int ci) {
    const float* gs = gold_smem() + ci * 32;
    // Two mask words per 32 logits with ONE integer-pipe instruction per logit and mask: the comparisons are done as
    // subtractions on the FMA pipe (x = g - s: sign bit set <=> s > g; -|x| + 0: sign bit set <=> s != g, because
    // -0 + +0 = +0) and the sign bits are shifted into the masks by a funnel shift.  FSETP + SEL + IADD3 per logit
    // made this epilogue ALU-pipe bound (64 lanes/clk/SM) at 36 % tensor-active; exact for all finite scores.
    uint32_t mgr = 0, mner = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float s = __uint_as_float(r[j]) + rs.bias_cur;
      const float x = gs[j] - s;                       // warp-wide broadcast read of the gold logit
      float ne;
      asm("add.rn.f32 %0, %1, 0f00000000;" : "=f"(ne) : "f"(-fabsf(x)));
      mgr = __funnelshift_l(__float_as_uint(x), mgr, 1);
      mner = __funnelshift_l(__float_as_uint(ne), mner, 1);
    }
    uint32_t mg = __brev(mgr), me = ~__brev(mner);     // bit j <-> column j
    uint32_t keep = ~rs.w_cur[ci];                     // bit set in w = filtered (true tail, gold entity)
    if (row >= p.M) keep = 0u;                         // padded entity rows
    mg &= keep;
    me &= keep;
    uint32_t carry = mg;
#pragma unroll
    for (int k = 0; k < kRankPlanes; ++k) {
      const uint32_t t = planes[ci][k] & carry;
      planes[ci][k] ^= carry;
      carry = t;
    }
    if (__any_sync(0xffffffffu, me != 0)) {
      const int lane = threadIdx.x & 31;
#pragma unroll 1
      for (int j = 0; j < 32; ++j) {
        const uint32_t be = __ballot_sync(0xffffffffu, (me >> j) & 1u);
        if (lane == j) ce[ci] += __popc(be);
      }
    }
  }
  __device__ __forceinline__ void tile_done(const GemmProblem&, const TileCoord&, int, int, int) { ++adds; }
  __device__ __forceinline__ void finish(int, int) { flush(); }
};

// gold logits: A = gathered gold rows Eg [B, d] (row i = E[e2[i]]), B = q; diagonal (i, i)
struct DiagEpiT : EpiBase {
  const float* bias;        // [Ns]
  const int64_t* e2;
  int64_t ent_lo, Ns;
  float* gold;              // [B]
  __device__ __forceinline__ void chunk(const GemmProblem& p, const TileCoord&, int row, int col, const uint32_t (&r)[32],
                                        int) const {
    if (row >= p.M || row < col || row >= col + 32) return;
    int64_t l = e2[row] - ent_lo;
    float v = 0.f;
    if (l >= 0 && l < Ns) {
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) acc = (col + j == row) ? __uint_as_float(r[j]) : acc;
      v = acc + __ldg(bias + l);
    }
    gold[row] = v;
  }
};

// ------------------------------------------------------------------------------------------ top-k
// One list per (CTA, lane quadrant, query) in global memory: a binary min-heap of k keys (topk.cu: score-then-id
// order as one uint64, 0 = empty slot), written only by the warp that owns the quadrant and the query column - no locks.
// Per query column the warp keeps a threshold tau (the score of the heap's minimum, -inf while the heap has an empty
// slot) in shared memory, laid out like RankEpiT's gold logits.  Dense loop per logit: s = acc + bias, x = s - tau,
// funnel-shift the sign bit (sign clear <=> s >= tau; -inf / +inf thresholds make every / no logit a candidate).
// Chunks with a candidate that survives the filter word take the insert path: per column with candidates, its owner
// lane j pulls the candidate rows' scores by shuffle and pushes them (O(log k) per push), then raises tau.
__device__ __noinline__ void topk_heap_push(uint64_t* h, int k, uint64_t key) {
  if (key <= h[0]) return;
  int i = 0;
  for (;;) {
    const int l = 2 * i + 1;
    if (l >= k) break;
    uint64_t hc = h[l];
    int c = l;
    if (l + 1 < k) {
      const uint64_t hr = h[l + 1];
      if (hr < hc) { hc = hr; c = l + 1; }
    }
    if (hc >= key) break;
    h[i] = hc;
    i = c;
  }
  h[i] = key;
}
// threshold of a heap root: its score, -inf for an empty slot, and -0 for a zero score (so that s - tau keeps its sign
// bit clear for s = +0 and s = -0 alike)
__device__ __forceinline__ float topk_key_score(uint64_t key) {
  if (key == 0ull) return -INFINITY;
  const uint32_t u = (uint32_t)(key >> 32);
  if (u == 0x80000000u) return -0.f;
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}
template <int NCH>
struct TopkEpiT : EpiBase {
  RowState<NCH> rs;
  uint64_t* lists;          // [grid * 4][N][k]
  int k, cur_col0;
  uint32_t id_hi;           // 0x7FFFFFFF - ent_lo: the key's id field of entity row n is id_hi - n (topk.cu)
  __device__ __forceinline__ float* tau_smem() {
    __shared__ float tau_s[kEntEpiWarps][NCH * 32];
    return tau_s[(threadIdx.x >> 5) - 4];
  }
  __device__ __forceinline__ uint64_t* heap(const GemmProblem& p, int col) const {
    return lists + ((int64_t)(blockIdx.x * 4 + ((threadIdx.x >> 5) & 3)) * p.N + col) * k;
  }
  __device__ __forceinline__ void tile_begin(const GemmProblem& p, const TileCoord&, int row, int col0) {
    if (col0 != cur_col0) {                          // new query block: thresholds of its lists
      cur_col0 = col0;
      float* ts = tau_smem();
      const int lane = threadIdx.x & 31;
      __syncwarp();
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = col0 + i * 32 + lane;
        ts[i * 32 + lane] = c < p.N ? topk_key_score(heap(p, c)[0]) : INFINITY;   // (masked in chunk as well)
      }
      __syncwarp();
    }
    rs.begin(p, row, col0);
  }
  __device__ __forceinline__ void tile_prefetch(const GemmProblem& p, const TileCoord&, int row, int col0) { rs.prefetch(p, row, col0); }
  __device__ __forceinline__ void chunk(const GemmProblem& p, const TileCoord&, int row, int col, const uint32_t (&r)[32],
                                        int ci) {
    float* ts = tau_smem() + ci * 32;
    uint32_t msk = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float x = (__uint_as_float(r[j]) + rs.bias_cur) - ts[j];
      msk = __funnelshift_l(__float_as_uint(x), msk, 1);
    }
    uint32_t cand = ~__brev(msk) & ~rs.w_cur[ci];     // bit j <-> column j; filter bit set = excluded
    if (row >= p.M) cand = 0u;                        // padded entity rows
    // columns past the last query: their TMEM words may never have been written by the MMA (it writes n_eff columns),
    // so the +inf threshold alone cannot exclude them (a stale NaN passes the sign test)
    if (p.N - col < 32) cand &= (1u << (p.N - col)) - 1u;
    if (!__any_sync(0xffffffffu, cand != 0u)) return;
    const int lane = threadIdx.x & 31;
    const uint32_t cols = __reduce_or_sync(0xffffffffu, cand);
    const uint32_t key_lo0 = id_hi - (uint32_t)(row - lane);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if ((cols >> j) & 1u) {                         // warp-uniform
        uint32_t rows = __ballot_sync(0xffffffffu, (cand >> j) & 1u);
        const float sj = __uint_as_float(r[j]) + rs.bias_cur;
        uint64_t* h = heap(p, col + j);
        while (rows) {
          const int src = __ffs(rows) - 1;
          rows &= rows - 1;
          const float v = __shfl_sync(0xffffffffu, sj, src);
          if (lane == j) {
            uint32_t u = __float_as_uint(v == 0.f ? 0.f : v);
            u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
            const uint32_t lo = ((key_lo0 - (uint32_t)src) << 1) | (uint32_t)(__float_as_uint(v) == 0x80000000u);
            topk_heap_push(h, k, ((uint64_t)u << 32) | (uint64_t)lo);
          }
        }
        if (lane == j) ts[j] = topk_key_score(h[0]);
      }
    }
    __syncwarp();
  }
};

// rows e2[b] - ent_lo of a prepared operand [Ns, ldp] -> [B, ldp] (zero rows when not owned); 16-byte vectors
__global__ void gather_prepared_kernel(const uint4* __restrict__ src, int64_t Ns, int vec_per_row, int planes,
                                       const int64_t* __restrict__ e2, int64_t ent_lo, int B, uint4* __restrict__ dst,
                                       const int* __restrict__ src_exp, int* __restrict__ dst_exp) {
  pdl_enter();
  int b = blockIdx.x;
  if (src_exp && b == 0 && threadIdx.x == 0) *dst_exp = *src_exp;      // fp16x3: the gathered rows keep E's exponent
  int64_t l = e2[b] - ent_lo;
  bool owned = l >= 0 && l < Ns;
  for (int pl = 0; pl < planes; ++pl) {
    const uint4* s = src + ((int64_t)pl * Ns + (owned ? l : 0)) * vec_per_row;
    uint4* o = dst + ((int64_t)pl * B + b) * vec_per_row;
    for (int v = threadIdx.x; v < vec_per_row; v += blockDim.x) o[v] = owned ? __ldg(s + v) : make_uint4(0, 0, 0, 0);
  }
}

__global__ void sum_doubles_kernel(const double* __restrict__ in, int n, double* out) {
  pdl_enter();
  __shared__ double smd[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += in[i];
  double t = block_sum<double>(acc, smd);
  if (threadIdx.x == 0) *out = t;
}

// ------------------------------------------------------------------------------------------ configurations
// bf16: BLOCK_N = 256 queries per tile with the query block RESIDENT in shared memory (4 k-blocks of 64 = d <= 256):
//       only the 128-entity A tiles stream (16 KB per k-block), 8 epilogue warps x 4 chunks, full TMEM (2 x 256 cols).
// tf32x3 (and bf16 with d > 256): BLOCK_N = 128, both operands stream.
template <int PREC, bool RES>
struct EntSel;
template <>
struct EntSel<PREC_BF16, true> { using Cfg = GemmCfg<PREC_BF16, 256, 5, kEntEpiWarps, false, false, 0, 4>; };
template <>
struct EntSel<PREC_BF16, false> { using Cfg = GemmCfg<PREC_BF16, 128, 6, kEntEpiWarps, false, false, 0, 0>; };
template <>
struct EntSel<PREC_TF32X3, false> { using Cfg = GemmCfg<PREC_TF32X3, 128, 3, kEntEpiWarps, false, false, 0, 0>; };
template <>
struct EntSel<PREC_FP16X3, false> { using Cfg = GemmCfg<PREC_FP16X3, 128, 3, kEntEpiWarps, false, false, 0, 0>; };
// fp16x3 with the 128-query block RESIDENT (2 planes x 4 k-blocks x 16 KB = 128 KB): per 128 x 128 tile only the entity
// planes stream (128 KB instead of 256 KB), which is what bounds the streaming configuration (~42 B/clk/SM of TMA)
template <>
struct EntSel<PREC_FP16X3, true> { using Cfg = GemmCfg<PREC_FP16X3, 128, 2, kEntEpiWarps, false, false, 0, 4>; };   // (3 stages + the rank epilogue's 2 KB would exceed 227 KB by 256 B)
// the BCE epilogue is MUFU / latency bound: 16 epilogue warps (4 per scheduler) hide the TMEM-load and SFU latencies
template <int PREC, bool RES>
struct BceSel;
template <>
struct BceSel<PREC_BF16, true> { using Cfg = GemmCfg<PREC_BF16, 256, 3, kBceEpiWarps, false, false, 0, 4>; };
template <>
struct BceSel<PREC_BF16, false> { using Cfg = GemmCfg<PREC_BF16, 128, 5, kBceEpiWarps, false, false, 0, 0>; };
template <>
struct BceSel<PREC_TF32X3, false> { using Cfg = GemmCfg<PREC_TF32X3, 128, 3, kBceEpiWarps, false, false, 0, 0>; };
template <>
struct BceSel<PREC_FP16X3, false> { using Cfg = GemmCfg<PREC_FP16X3, 128, 3, kBceEpiWarps, false, false, 0, 0>; };
// (2 stages: the BCE epilogue's 32 KB store staging tile shares the 227 KB with the 128 KB resident block)
template <>
struct BceSel<PREC_FP16X3, true> { using Cfg = GemmCfg<PREC_FP16X3, 128, 2, kBceEpiWarps, false, false, 0, 4>; };
template <class Cfg>
constexpr int ent_nch() { return Cfg::BLOCK_N / (Cfg::EPI_WARPS / 4) / 32; }
// the resident-query-block configuration pays a 128 KB fill per CTA: worth it once a CTA processes >= 8 tiles
// (WN18RR: 640 tiles / 148 CTAs -> streaming configuration; 1 M entities: 106 tiles per CTA -> resident)
static inline bool ent_resident(int d, int prec, int64_t Ns, int B) {
  if ((prec != COPER_PREC_BF16 && prec != COPER_PREC_FP16X3) || d > 256) return false;
  const int bn = prec == COPER_PREC_BF16 ? 256 : 128;
  const int64_t tiles = ((Ns + BLOCK_M - 1) / BLOCK_M) * ((B + bn - 1) / bn);
  return tiles >= 8 * (int64_t)sm_count();
}
static inline int ent_block_n(int d, int prec, int64_t Ns, int B) {
  return (prec == COPER_PREC_BF16 && ent_resident(d, prec, Ns, B)) ? 256 : 128;
}

static GemmProblem ent_problem(int B, int64_t Ns, int d, int block_n) {
  GemmProblem p{};
  p.M = (int)Ns; p.N = B; p.K = d; p.groups = 1; p.groups_inner = 0;
  p.m_tiles = (int)((Ns + BLOCK_M - 1) / BLOCK_M);
  p.n_tiles = (B + block_n - 1) / block_n;
  p.splits = 1;
  p.kb_per_split = 1 << 28;   // clamped to the real block count by gemm_decode
  p.n_fastest = 1;            // see GemmProblem: one query block per CTA, entity tiles shared through L2
  return p;
}
// every CTA keeps ONE query block for as long as possible: tiles are enumerated entity-tile fastest, so with
// grid <= m_tiles a CTA changes its query block at most n_tiles - 1 times
static int ent_grid(const GemmProblem& p) {
  long long supers = (long long)p.m_tiles * p.n_tiles;
  const int sms = sm_count();
  int grid = (int)(supers < sms ? supers : sms);
  if (p.n_tiles <= grid) grid = grid / p.n_tiles * p.n_tiles;    // multiple of n_tiles: fixed n-block per CTA
  return grid;
}

// ------------------------------------------------------------------------------------------ logits
template <class Cfg>
static int score_t_impl(const TcOperand& E, const TcOperand& Q, const float* bias, int B, int64_t Ns, int d, float* S,
                        int64_t ld, cudaStream_t st) {
  GemmProblem p = ent_problem(B, Ns, d, Cfg::BLOCK_N);
  ScoreEpiT<ent_nch<Cfg>()> epi;
  epi.rs.init(bias, nullptr, 0);
  epi.out = S; epi.ld = ld;
  return launch_gemm<Cfg, ScoreEpiT<ent_nch<Cfg>()>>(E, Q, p, epi, st, ent_grid(p));
}
// dispatch over (precision, resident query block)
#define ENT_DISPATCH(FN, ...)                                                                              \
  do {                                                                                                     \
    if (prec == COPER_PREC_BF16 && ent_resident(d, prec, Ns, B)) return FN<EntSel<PREC_BF16, true>::Cfg>(__VA_ARGS__);  \
    if (prec == COPER_PREC_BF16) return FN<EntSel<PREC_BF16, false>::Cfg>(__VA_ARGS__);                   \
    if (prec == COPER_PREC_TF32X3) return FN<EntSel<PREC_TF32X3, false>::Cfg>(__VA_ARGS__);               \
    if (prec == COPER_PREC_FP16X3 && ent_resident(d, prec, Ns, B)) return FN<EntSel<PREC_FP16X3, true>::Cfg>(__VA_ARGS__); \
    if (prec == COPER_PREC_FP16X3) return FN<EntSel<PREC_FP16X3, false>::Cfg>(__VA_ARGS__);               \
    return COPER_ERR_UNSUPPORTED;                                                                          \
  } while (0)
int umma_score1n_fwd_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                              float* scores, int64_t ld, int prec, cudaStream_t st) {
  if (ld < Ns || Ns > 0x7fffffff - 512) return COPER_ERR_INVALID_ARG;
  TcOperand Q = tc_operand(q_prep, B, d, prec), E = tc_operand(E_prep, Ns, d, prec);
  ENT_DISPATCH(score_t_impl, E, Q, bias, B, Ns, d, scores, ld, st);
}

// ------------------------------------------------------------------------------------------ gold + rank
size_t umma_rank_workspace_bytes(int B, int d, int prec) { return align_up(tc_prepared_bytes(B, d, prec), 256); }

template <class Cfg>
static int gold_impl(const TcOperand& Eg, const TcOperand& Q, const float* bias, int B, int64_t Ns, int d,
                     const int64_t* e2, int64_t ent_lo, float* gold, cudaStream_t st) {
  GemmProblem p = ent_problem(B, B, d, Cfg::BLOCK_N);
  DiagEpiT epi;
  epi.bias = bias; epi.e2 = e2; epi.ent_lo = ent_lo; epi.Ns = Ns; epi.gold = gold;
  return launch_gemm<Cfg, DiagEpiT>(Eg, Q, p, epi, st);
}
int umma_score1n_gold(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                      const int64_t* e2, int64_t ent_lo, float* gold, void* ws, size_t ws_bytes, int prec,
                      cudaStream_t st) {
  if (!ws || ws_bytes < umma_rank_workspace_bytes(B, d, prec) || (reinterpret_cast<uintptr_t>(ws) & 255))
    return COPER_ERR_WORKSPACE;
  int64_t ldp = tc_prepared_ld(d, prec);
  int elem = prec == COPER_PREC_TF32X3 ? 4 : 2;
  int vec_per_row = (int)(ldp * elem / 16);
  const int* src_exp = nullptr;
  int* dst_exp = nullptr;
  if (prec == COPER_PREC_FP16X3) {
    src_exp = static_cast<const int*>(tc_fp16x3_trailer(E_prep, Ns, d));
    dst_exp = static_cast<int*>(tc_fp16x3_trailer(ws, B, d));
  }
  launch_pdl(gather_prepared_kernel, B, 64, 0, st, static_cast<const uint4*>(E_prep), Ns, vec_per_row, prec ==
             COPER_PREC_BF16 ? 1 : 2, e2, ent_lo, B, static_cast<uint4*>(ws), src_exp, dst_exp);
  int rc = check_launch();
  if (rc) return rc;
  TcOperand Q = tc_operand(q_prep, B, d, prec), Eg = tc_operand(ws, B, d, prec);
  ENT_DISPATCH(gold_impl, Eg, Q, bias, B, Ns, d, e2, ent_lo, gold, st);
}

template <class Cfg>
static int rank_impl(const TcOperand& E, const TcOperand& Q, const float* bias, int B, int64_t Ns, int d,
                     const float* gold, const uint32_t* filtT, int32_t* n_greater, int32_t* n_equal, cudaStream_t st) {
  GemmProblem p = ent_problem(B, Ns, d, Cfg::BLOCK_N);
  constexpr int kEntNCH = ent_nch<Cfg>();
  RankEpiT<kEntNCH> epi;
  epi.rs.init(bias, filtT, (B + 31) / 32);
  epi.gold = gold; epi.n_greater = n_greater; epi.n_equal = n_equal;
  epi.cur_col0 = -1;
  epi.n_queries = B;
  epi.adds = 0;
  for (int i = 0; i < kEntNCH; ++i) {
    epi.ce[i] = 0;
    for (int k = 0; k < kRankPlanes; ++k) epi.planes[i][k] = 0;
  }
  return launch_gemm<Cfg, RankEpiT<kEntNCH>>(E, Q, p, epi, st, ent_grid(p));
}
int umma_score1n_rank(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                      const float* gold, const uint32_t* filtT, int32_t* n_greater, int32_t* n_equal, int prec,
                      cudaStream_t st) {
  if (Ns > 0x7fffffff - 512) return COPER_ERR_UNSUPPORTED;
  TcOperand Q = tc_operand(q_prep, B, d, prec), E = tc_operand(E_prep, Ns, d, prec);
  ENT_DISPATCH(rank_impl, E, Q, bias, B, Ns, d, gold, filtT, n_greater, n_equal, st);
}

// ------------------------------------------------------------------------------------------ fused top-k
int topk_merge_keys(const uint64_t* lists, int B, int k, int per, int first_div, int step, int n_groups, float* out_s,
                    int64_t* out_id, cudaStream_t st);                                                   // topk.cu
// heaps of every (CTA slot, lane quadrant, query); the grid is at most sm_count() CTAs
size_t umma_topk_workspace_bytes(int B, int k) { return align_up((size_t)sm_count() * 4 * B * k * sizeof(uint64_t), 256); }

template <class Cfg>
static int topk_impl(const TcOperand& E, const TcOperand& Q, const float* bias, int B, int64_t Ns, int d,
                     const uint32_t* filtT, int64_t ent_lo, int k, float* out_s, int64_t* out_id, void* ws,
                     cudaStream_t st) {
  GemmProblem p = ent_problem(B, Ns, d, Cfg::BLOCK_N);
  constexpr int kEntNCH = ent_nch<Cfg>();
  const int grid = ent_grid(p);
  uint64_t* lists = static_cast<uint64_t*>(ws);
  int rc = check_cuda(cudaMemsetAsync(lists, 0, (size_t)grid * 4 * B * k * sizeof(uint64_t), st));   // empty heaps
  if (rc) return rc;
  TopkEpiT<kEntNCH> epi;
  epi.rs.init(bias, filtT, (B + 31) / 32);
  epi.lists = lists; epi.k = k; epi.cur_col0 = -1;
  epi.id_hi = 0x7FFFFFFFu - (uint32_t)ent_lo;
  if ((rc = launch_gemm<Cfg, TopkEpiT<kEntNCH>>(E, Q, p, epi, st, grid))) return rc;
  // with a grid that is a multiple of n_tiles, CTA c only ever saw query block c % n_tiles
  if (p.n_tiles <= grid) return topk_merge_keys(lists, B, k, 4, Cfg::BLOCK_N, p.n_tiles, grid / p.n_tiles, out_s, out_id, st);
  return topk_merge_keys(lists, B, k, 4, 0, 1, grid, out_s, out_id, st);
}
int umma_score1n_topk(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                      const uint32_t* filtT, int64_t ent_lo, int k, float* out_s, int64_t* out_id, void* ws,
                      size_t ws_bytes, int prec, cudaStream_t st) {
  if (prec != COPER_PREC_BF16 && prec != COPER_PREC_TF32X3 && prec != COPER_PREC_FP16X3) return COPER_ERR_UNSUPPORTED;
  if (Ns > 0x7fffffff - 512 || ent_lo + Ns >= 0x7FFFFFFFll) return COPER_ERR_UNSUPPORTED;
  if (!ws || ws_bytes < umma_topk_workspace_bytes(B, k) || (reinterpret_cast<uintptr_t>(ws) & 255))
    return COPER_ERR_WORKSPACE;
  TcOperand Q = tc_operand(q_prep, B, d, prec), E = tc_operand(E_prep, Ns, d, prec);
  ENT_DISPATCH(topk_impl, E, Q, bias, B, Ns, d, filtT, ent_lo, k, out_s, out_id, ws, st);
}

// ------------------------------------------------------------------------------------------ training scorer
// dE = G^T . q; with dE_sumsq != NULL the store epilogue also sums the squares of what it writes (per-warp partials,
// fixed-order final sum): the global-norm clip then does not re-read the [Ns, d] gradient (SURVEY §8f-1)
static int dE_gemm(int prec, bool a_mn, const TcOperand& Go, const TcOperand& Qo, const GemmProblem& p, StoreEpi epi,
                   double* dE_sumsq, double* ss_part, cudaStream_t st) {
  int rc;
  const int n_part = sm_count() * 16;
  if (dE_sumsq) {
    if ((rc = check_cuda(cudaMemsetAsync(ss_part, 0, (size_t)n_part * sizeof(double), st)))) return rc;
    epi.sumsq_part = ss_part;
  }
  if ((rc = tc_gemm_store(prec, a_mn, true, Go, Qo, p, false, epi, st))) return rc;
  if (dE_sumsq) {
    launch_pdl(sum_doubles_kernel, 1, 256, 0, st, ss_part, n_part, dE_sumsq);
    rc = check_launch();
  }
  return rc;
}
struct BceTcLayout {
  size_t off_q, off_E, off_dq, off_dbias, off_loss, off_ss, total;
  int splits, dbias_slabs;
};
static BceTcLayout bce_tc_layout(int B, int64_t Ns, int d, int prec) {
  BceTcLayout L;
  GemmProblem p{};
  p.M = B; p.N = d; p.K = (int)Ns; p.groups = 1;
  L.splits = tc_plan_splits(prec, p, true);
  int bn = ent_block_n(d, prec, Ns, B);
  L.dbias_slabs = ((B + bn - 1) / bn) * (kBceEpiWarps / 4);
  size_t dq_rows = (size_t)L.splits * B;
  if (umma_fused_ok(B, Ns, d, prec)) {               // fused kernel: one [128, d] dq block per CTA, QB dbias slabs
    int QB, R;
    umma_fused_plan(B, Ns, &QB, &R);
    if ((size_t)R * B > dq_rows) dq_rows = (size_t)R * B;
    if (QB > L.dbias_slabs) L.dbias_slabs = QB;
  }
  size_t o = 0;
  L.off_q = o; o = align_up(o + tc_prepared_bytes(B, d, prec), 256);
  L.off_E = o; o = align_up(o + tc_prepared_bytes(Ns, d, prec), 256);
  L.off_dq = o; o = align_up(o + dq_rows * d * sizeof(float), 256);
  L.off_dbias = o; o = align_up(o + (size_t)L.dbias_slabs * Ns * sizeof(float), 256);
  L.off_loss = o; o = align_up(o + (size_t)sm_count() * kBceEpiWarps * sizeof(double), 256);
  L.off_ss = o; o = align_up(o + (size_t)sm_count() * 16 * sizeof(double), 256);      // sum-of-squares partials of dE
  L.total = o;
  return L;
}
size_t umma_bce_workspace_bytes(int B, int64_t Ns, int d, int prec) { return bce_tc_layout(B, Ns, d, prec).total; }
// dbias slabs the scorer pass of these arguments writes: QB from the fused kernel, else one per query-block chunk row
static int bce_dbias_slabs_used(const BceTcLayout& L, int B, int64_t Ns, int d, int prec) {
  if (umma_fused_ok(B, Ns, d, prec)) {
    int QB, R;
    umma_fused_plan(B, Ns, &QB, &R);
    return QB;
  }
  int bn = ent_block_n(d, prec, Ns, B);
  (void)L;
  return ((B + bn - 1) / bn) * (kBceEpiWarps / 4);
}
// GT [Ns, ldGT]: ldGT = B rounded up to 32 (whole 16-byte vectors per 32-query chunk)
static inline int64_t gt_pitch(int B) { return (B + 31) / 32 * 32; }
size_t umma_bce_G_bytes(int B, int64_t Ns, int prec) {
  if (prec == COPER_PREC_BF16) return (size_t)Ns * gt_pitch(B) * 2;
  if (prec == COPER_PREC_FP16X3) return (size_t)Ns * gt_pitch(B) * 2 * 2;    // entity-major fp16 hi / lo planes
  return (size_t)B * ((Ns + 31) / 32 * 32) * 8;      // tf32x3: query-major hi / lo planes
}

template <class Cfg>
static int bce_impl(const TcOperand& E, const TcOperand& Q, const float* bias, const uint32_t* bitsT, int B, int64_t Ns,
                    int d, float pos, float neg, float inv_count, void* GT, int64_t ldGT, float* dbias_part,
                    double* loss_part, cudaStream_t st, int* grid_out) {
  GemmProblem p = ent_problem(B, Ns, d, Cfg::BLOCK_N);
  constexpr int kEntNCH = ent_nch<Cfg>();
  constexpr int PREC = Cfg::PREC;
  BceEpiT<PREC, kEntNCH> epi;
  epi.rs.init(bias, bitsT, (B + 31) / 32);
  epi.pos = pos; epi.neg = neg; epi.GT = GT; epi.ldGT = ldGT;
  // fp16x3 carries dL/dS as (sigmoid - z') * 2^10 in fp16 hi / lo planes (values in (-2^10, 2^10)); the true 1/count
  // (far below the fp16 range) is applied by the dq / dE epilogues and to the dbias row sums
  epi.inv_count = PREC == PREC_FP16X3 ? 1024.0f : inv_count;
  epi.rsum_scale = PREC == PREC_FP16X3 ? inv_count * (1.0f / 1024.0f) : 1.0f;
  epi.dbias_part = dbias_part; epi.loss_part = loss_part; epi.loss_acc = 0.0; epi.rsum = 0.f;
  *grid_out = ent_grid(p);
  return launch_gemm<Cfg, BceEpiT<PREC, kEntNCH>>(E, Q, p, epi, st, *grid_out);
}

// dL/dS as a tensor-pipe operand: bf16 / fp16x3 GT stored entity-major [Ns, B]; tf32x3 G stored query-major [B, Ns]
static TcOperand g_operand(const void* G, int B, int64_t Ns, int prec) {
  const bool entity_major = prec != COPER_PREC_TF32X3;
  const int64_t ldGT = entity_major ? gt_pitch(B) : (Ns + 31) / 32 * 32;
  TcOperand Go;
  Go.main = G;
  Go.pitch = (uint64_t)ldGT;
  Go.exp = nullptr;
  if (entity_major) {
    Go.lo = prec == COPER_PREC_FP16X3 ? static_cast<const void*>(static_cast<const uint16_t*>(G) + Ns * ldGT) : nullptr;
    Go.rows = (uint64_t)Ns; Go.cols = (uint64_t)B;
  } else {
    Go.lo = static_cast<const void*>(static_cast<const float*>(G) + (int64_t)B * ldGT);
    Go.rows = (uint64_t)B; Go.cols = (uint64_t)Ns;
  }
  return Go;
}

// Pass 3 on its own: dE = G^T . q from the G and the prepared q that umma_score1n_bce_fwd_bwd (called with dE == NULL)
// left in `G` / `ws`.  Independent of dq and of everything the front-end backward does, so the host may enqueue it on a
// second stream and let the HBM-bound GEMM run under the latency-bound backward chain.
// dbias != NULL: also reduce the dbias slabs the scorer call left in `ws` (it skips that reduction when it is called
// with dE == NULL, so the short dependent chain BCE -> dq on the main stream carries nothing but what dq needs).
int umma_score1n_dE(const void* G, int B, int64_t Ns, int d, float inv_count, float* dE, double* dE_sumsq, float* dbias,
                    void* ws, size_t ws_bytes, int prec, cudaStream_t st) {
  BceTcLayout L = bce_tc_layout(B, Ns, d, prec);
  if (!ws || ws_bytes < L.total) return COPER_ERR_WORKSPACE;
  char* w = static_cast<char*>(ws);
  if (dbias) {
    int rc = coper_reduce_partials(reinterpret_cast<const float*>(w + L.off_dbias), bce_dbias_slabs_used(L, B, Ns, d, prec),
                                   Ns, 1.0f, 0, dbias, (coper_stream_t)st);
    if (rc) return rc;
  }
  TcOperand Qo = tc_operand(w + L.off_q, B, d, prec), Go = g_operand(G, B, Ns, prec);
  GemmProblem p{};
  p.M = (int)Ns; p.N = d; p.K = B; p.groups = 1; p.groups_inner = 0;
  p.post_scale = prec == COPER_PREC_FP16X3 ? inv_count * (1.0f / 1024.0f) : 0.f;
  StoreEpi epi = make_store_epi(dE, d, 0, 0);
  return dE_gemm(prec, prec == COPER_PREC_TF32X3, Go, Qo, p, epi, dE_sumsq, reinterpret_cast<double*>(w + L.off_ss), st);
}

int umma_score1n_bce_fwd_bwd(const float* q, const float* E, const void* E_prepared, const float* bias,
                             const uint32_t* label_bits_t, int B, int64_t Ns, int d, float pos, float neg,
                             float inv_count, double* loss_sum, void* G, int64_t ldG, float* dq, float* dE,
                             float* dbias, void* ws, size_t ws_bytes, int prec, double* dE_sumsq, cudaStream_t st) {
  if (Ns > 0x7fffffff - 512) return COPER_ERR_UNSUPPORTED;
  (void)ldG;                                          // the tensor-pipe engines lay G out entity-major themselves
  if (reinterpret_cast<uintptr_t>(G) & 127) return COPER_ERR_INVALID_ARG;
  const bool entity_major = prec != COPER_PREC_TF32X3;
  const int64_t ldGT = entity_major ? gt_pitch(B) : (Ns + 31) / 32 * 32;
  const float g_post = prec == COPER_PREC_FP16X3 ? inv_count * (1.0f / 1024.0f) : 0.f;   // see bce_impl
  BceTcLayout L = bce_tc_layout(B, Ns, d, prec);
  if (!ws || ws_bytes < L.total) return COPER_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(ws) & 255) return COPER_ERR_INVALID_ARG;
  char* w = static_cast<char*>(ws);
  void* qp = w + L.off_q;
  const void* Ep = E_prepared ? E_prepared : w + L.off_E;
  float* dq_part = reinterpret_cast<float*>(w + L.off_dq);
  float* dbias_part = reinterpret_cast<float*>(w + L.off_dbias);
  double* loss_part = reinterpret_cast<double*>(w + L.off_loss);
  int rc;
  if ((rc = tc_prepare(q, B, d, d, prec, qp, st))) return rc;
  if (!E_prepared && (rc = tc_prepare(E, Ns, d, d, prec, w + L.off_E, st))) return rc;
  TcOperand Qo = tc_operand(qp, B, d, prec), Eo = tc_operand(Ep, Ns, d, prec);
  if (umma_fused_ok(B, Ns, d, prec)) {
    // ---- single pass over E: scores -> loss, dbias, G (TMA store, entity-major) AND dq (G consumed from shared memory)
    int QB, R, grid = 0;
    umma_fused_plan(B, Ns, &QB, &R);
    if ((rc = umma_bce_dq_fused(Eo, Qo, bias, label_bits_t, B, Ns, d, pos, neg, inv_count, G, ldGT, dq_part, dbias_part,
                                loss_part, &grid, st)))
      return rc;
    // dq slabs and the loss partials are reduced by one launch; dbias here only if the caller does not split off dE
    if ((rc = reduce_partials_and_sum(dq_part, R, (int64_t)B * d, 1.0f, 0, dq, loss_part, grid * kBceEpiWarps, loss_sum, st)))
      return rc;
    // ---- dE = G^T . q from the entity-major G the kernel stored (dE == NULL: the caller runs umma_score1n_dE itself)
    if (!dE) return COPER_OK;
    return umma_score1n_dE(G, B, Ns, d, inv_count, dE, dE_sumsq, dbias, ws, ws_bytes, prec, st);
  }
  // ---- pass 1: scores -> loss, G, dbias partials
  int grid = 0;
  auto run_bce = [&]() -> int {
    if (prec == COPER_PREC_BF16 && ent_resident(d, prec, Ns, B))
      return bce_impl<BceSel<PREC_BF16, true>::Cfg>(Eo, Qo, bias, label_bits_t, B, Ns, d, pos, neg, inv_count, G, ldGT,
                                                    dbias_part, loss_part, st, &grid);
    if (prec == COPER_PREC_BF16)
      return bce_impl<BceSel<PREC_BF16, false>::Cfg>(Eo, Qo, bias, label_bits_t, B, Ns, d, pos, neg, inv_count, G, ldGT,
                                                     dbias_part, loss_part, st, &grid);
    if (prec == COPER_PREC_FP16X3 && ent_resident(d, prec, Ns, B))
      return bce_impl<BceSel<PREC_FP16X3, true>::Cfg>(Eo, Qo, bias, label_bits_t, B, Ns, d, pos, neg, inv_count, G, ldGT,
                                                      dbias_part, loss_part, st, &grid);
    if (prec == COPER_PREC_FP16X3)
      return bce_impl<BceSel<PREC_FP16X3, false>::Cfg>(Eo, Qo, bias, label_bits_t, B, Ns, d, pos, neg, inv_count, G, ldGT,
                                                       dbias_part, loss_part, st, &grid);
    return bce_impl<BceSel<PREC_TF32X3, false>::Cfg>(Eo, Qo, bias, label_bits_t, B, Ns, d, pos, neg, inv_count, G, ldGT,
                                                     dbias_part, loss_part, st, &grid);
  };
  if ((rc = run_bce())) return rc;
  TcOperand Go = g_operand(G, B, Ns, prec);
  // ---- pass 2: dq = G . E   (A(b, n): GT is the MN-major form, G the K-major form; B = E stored [K, N] -> MN-major)
  {
    GemmProblem p{};
    p.M = B; p.N = d; p.K = (int)Ns; p.groups = 1; p.groups_inner = 0;
    p.post_scale = g_post;
    StoreEpi epi = make_store_epi(dq_part, d, 0, (long long)B * d);
    if ((rc = tc_gemm_store(prec, entity_major, true, Go, Eo, p, true, epi, st))) return rc;
    // dq slabs and the loss partials of pass 1: one launch
    if ((rc = reduce_partials_and_sum(dq_part, L.splits, (int64_t)B * d, 1.0f, 0, dq, loss_part, grid * kBceEpiWarps,
                                      loss_sum, st)))
      return rc;
  }
  // ---- pass 3: dE = G^T . q (A(n, b): GT is the K-major form, G the MN-major form; B = q stored [K, N] -> MN-major),
  // preceded by the dbias slab reduction
  if (!dE) return COPER_OK;                            // the caller runs umma_score1n_dE itself (second stream)
  return umma_score1n_dE(G, B, Ns, d, inv_count, dE, dE_sumsq, dbias, ws, ws_bytes, prec, st);
}

}  // namespace coper

using namespace coper;

extern "C" {

size_t coper_score1n_rank_workspace_bytes(int B, int d, int prec) {
  if (prec != COPER_PREC_BF16 && prec != COPER_PREC_TF32X3 && prec != COPER_PREC_FP16X3) return 0;
  return umma_rank_workspace_bytes(B, d, prec);
}
int coper_score1n_gold_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                                const int64_t* e2, int64_t ent_lo, float* gold, void* workspace,
                                size_t workspace_bytes, int prec, coper_stream_t stream) {
  COPER_CHECK_ARG(q_prep && E_prep && bias && e2 && gold && B > 0 && Ns > 0 && d > 0);
  return umma_score1n_gold(q_prep, E_prep, bias, B, Ns, d, e2, ent_lo, gold, workspace, workspace_bytes, prec,
                           as_stream(stream));
}
int coper_score1n_rank_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                                const float* gold, const uint32_t* filter_bits_t, int32_t* n_greater,
                                int32_t* n_equal, int prec, coper_stream_t stream) {
  COPER_CHECK_ARG(q_prep && E_prep && bias && gold && filter_bits_t && n_greater && n_equal);
  COPER_CHECK_ARG(B > 0 && Ns > 0 && d > 0);
  return umma_score1n_rank(q_prep, E_prep, bias, B, Ns, d, gold, filter_bits_t, n_greater, n_equal, prec,
                           as_stream(stream));
}

size_t coper_score1n_topk_workspace_bytes(int B, int64_t Ns, int d, int k, int prec) {
  if (prec != COPER_PREC_BF16 && prec != COPER_PREC_TF32X3 && prec != COPER_PREC_FP16X3) return 0;
  if (B <= 0 || Ns <= 0 || d <= 0 || k < 1 || k > COPER_TOPK_MAX) return 0;
  return umma_topk_workspace_bytes(B, k);
}
int coper_score1n_topk_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                                const uint32_t* filter_bits_t, int64_t ent_lo, int k, float* out_scores,
                                int64_t* out_ids, void* workspace, size_t workspace_bytes, int prec,
                                coper_stream_t stream) {
  COPER_CHECK_ARG(q_prep && E_prep && bias && out_scores && out_ids && B > 0 && Ns > 0 && d > 0 && ent_lo >= 0);
  COPER_CHECK_ARG(k >= 1 && k <= COPER_TOPK_MAX);
  return umma_score1n_topk(q_prep, E_prep, bias, B, Ns, d, filter_bits_t, ent_lo, k, out_scores, out_ids, workspace,
                           workspace_bytes, prec, as_stream(stream));
}

}  // extern "C"
