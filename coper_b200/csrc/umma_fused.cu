// Fused 1-N scorer + label-smoothed BCE + query gradient (a7 / a9 / a10: models.py:433-437, 448-453, 198), bf16 engine.
//
// One persistent kernel computes, per 128-entity x 128-query tile,
//     S  = E_t . q_blk^T                      tcgen05.mma #1   (accumulator in TMEM, double-buffered)
//     G  = (sigmoid(S + bias) - z') / count   epilogue warps: TMEM -> registers -> bf16 -> SHARED MEMORY, written in
//                                             the 128-byte-swizzled operand layout
//     dq_blk += G^T . E_t                     tcgen05.mma #2   reads G and the E tile that is still resident from #1;
//                                             the accumulator stays in TMEM for the CTA's whole entity range
//     GT[tile] <- G                           one TMA store (cp.async.bulk.tensor, smem -> HBM) of the same smem tile
// so the dL/dS matrix is written to HBM exactly once (for the dE = G^T.q GEMM that follows) and never read back for
// dq, E is read once, and the logits never exist in memory.  The loss partials, dbias and dq come out of the same pass.
//
// Work split: CTA (qb, r) owns query block qb (128 queries, operand tile resident in shared memory) and entity range
// r (contiguous 128-row tiles); the QB CTAs of one range run side by side, so an entity tile is fetched from HBM once
// and served to the other query blocks from L2.  dq partials (one [128, d] block per CTA) are summed in a fixed order
// by coper_reduce_partials -> deterministic.
//
// Warp roles (640 threads): 0 TMA producer, 1 MMA issuer, 2 TMEM allocator, 3 TMA-store issuer, 4..19 epilogue.
// Shared memory (1 CTA / SM): 2 entity-tile buffers (2 x 64 KB) + query block (64 KB) + G tile (32 KB) = 224 KB.
// TMEM (512 columns): dq accumulator [128 queries x d] in columns 0..255, S buffers at 256 and 384.
#include "umma_gemm.cuh"
#include "bce_math.cuh"

namespace coper {
using namespace umma;

namespace fz {
constexpr int kEpiWarps = 16;
constexpr int kThreads = 128 + kEpiWarps * 32;
constexpr int kKbMax = 4;                        // d <= 256: at most 4 k-blocks of 64 bf16
constexpr int kTile = 128 * 128;                 // bytes of one [128 rows x 128 B] swizzled block
constexpr int kEBuf = kKbMax * kTile;
constexpr int kOffQ = 2 * kEBuf, kOffG = kOffQ + kEBuf, kOffDb = kOffG + 2 * kTile;
constexpr int kOffBar = kOffDb + 3 * 128 * 4;
constexpr int kSmemBytes = kOffBar + 256;
constexpr uint32_t kColS = 256;                  // TMEM column of S buffer 0 (buffer 1 at +128)
enum { B_EFULL = 0, B_EEMPTY = 8, B_QFULL = 10, B_SFULL = 11, B_SEMPTY = 13, B_GFULL = 15, B_GEMPTY = 16, B_DQFULL = 17,
       B_DBFULL = 18, B_DBFREE = 19, B_COUNT = 20 };
static_assert(kSmemBytes <= 232448, "shared memory budget");

struct Params {
  int B, d, KB, Nd;          // Nd = d rounded up to 16 (UMMA N of the dq product)
  int64_t Ns;
  int m_tiles, QB, R;
  const float* bias;         // [Ns]
  const uint32_t* bitsT;     // [Ns, wordsB] entity-major label bits
  int wordsB;
  float pos, neg, ic;
  float* dq_part;            // [R][B][d]
  float* dbias_part;         // [QB][Ns]
  double* loss_part;         // [grid][kEpiWarps]
  long long* trace;          // optional [tiles][8] clock64 stamps of CTA 0 (pipeline timeline, dev tool); NULL = off
};
enum { TR_S_ISSUE = 0, TR_S_ISSUED, TR_G_SEEN, TR_DQ_ISSUED, TR_E_FREE_SEEN, TR_S_SEEN, TR_EPI_MATH_DONE, TR_G_WRITTEN };
}  // namespace fz

__global__ void __launch_bounds__(fz::kThreads, 1)
bce_dq_fused_kernel(const __grid_constant__ CUtensorMap tE, const __grid_constant__ CUtensorMap tQ,
                    const __grid_constant__ CUtensorMap tG, const fz::Params p) {
  using namespace fz;
  coper::pdl_trigger();                          // the next kernel of the stream may be scheduled (common.cuh)
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023u) __trap();          // the swizzled operand tiles need 1024-byte alignment
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bar + B_COUNT);
  float* dbs = reinterpret_cast<float*>(smem + kOffDb);
  uint8_t* smE = smem;
  uint8_t* smQ = smem + kOffQ;
  uint8_t* smG = smem + kOffG;
  const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;

  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 8; ++i) mbar_init(&bar[B_EFULL + i], 1);
    mbar_init(&bar[B_EEMPTY], 1); mbar_init(&bar[B_EEMPTY + 1], 1);
    mbar_init(&bar[B_QFULL], 1);
    mbar_init(&bar[B_SFULL], 1); mbar_init(&bar[B_SFULL + 1], 1);
    mbar_init(&bar[B_SEMPTY], kEpiWarps); mbar_init(&bar[B_SEMPTY + 1], kEpiWarps);
    mbar_init(&bar[B_GFULL], kEpiWarps);
    mbar_init(&bar[B_GEMPTY], 2);                // dq MMAs done (tcgen05.commit) + TMA store has read the tile
    mbar_init(&bar[B_DQFULL], 1);
    mbar_init(&bar[B_DBFULL], kEpiWarps - 4);
    mbar_init(&bar[B_DBFREE], 4);
    fence_barrier_init();
  } else if (warp == 2) {
    tmem_alloc(tmem_ptr, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;
  coper::pdl_wait();                             // barriers / TMEM are set up; from here on the predecessor's output is read

  const int qb = blockIdx.x % p.QB, rr = blockIdx.x / p.QB;
  const int t0 = (int)((int64_t)rr * p.m_tiles / p.R), t1 = (int)((int64_t)(rr + 1) * p.m_tiles / p.R);
  const int T = t1 - t0;

  if (warp == 0) {
    // ===================================================================== TMA producer (warp-uniform loop, one lane issues)
    const bool leader = elect_one();
    if (leader) {
      tma_prefetch_desc(&tE);
      tma_prefetch_desc(&tQ);
      mbar_expect_tx(&bar[B_QFULL], (uint32_t)(p.KB * kTile));
    }
    for (int kb = 0; kb < p.KB; ++kb)
      if (leader) tma_load_2d(smQ + kb * kTile, &tQ, &bar[B_QFULL], kb * 64, qb * 128);
    for (int i = 0; i < T; ++i) {
      const int buf = i & 1, n = i >> 1;
      // only two entity-tile buffers fit beside the resident query block, so the load of tile i cannot be issued before
      // the dq MMAs of tile i-2 have completed; pulling the tile into L2 two tiles ahead turns the exposed part of that
      // load from an HBM round trip into an L2 hit (query block 0 prefetches for the QB CTAs that share the tile)
      if (qb == 0 && i + 2 < T)
        for (int kb = 0; kb < p.KB; ++kb)
          if (leader) tma_prefetch_l2_2d(&tE, kb * 64, (t0 + i + 2) * 128);
      mbar_wait_guarded(&bar[B_EEMPTY + buf], (uint32_t)((n & 1) ^ 1));
      if (p.trace && blockIdx.x == 0 && leader) p.trace[i * 8 + TR_E_FREE_SEEN] = clock64();
      for (int kb = 0; kb < p.KB; ++kb) {
        uint64_t* fb = &bar[B_EFULL + buf * 4 + kb];
        if (leader) {
          mbar_expect_tx(fb, (uint32_t)kTile);
          tma_load_2d(smE + buf * kEBuf + kb * kTile, &tE, fb, kb * 64, (t0 + i) * 128);
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer (warp-uniform loop, one lane issues)
    const bool leader = elect_one();
    const uint32_t idescS = make_idesc(FMT_BF16, 128, 128, 0u, 0u);
    const uint32_t idescD = make_idesc(FMT_BF16, 128, (uint32_t)p.Nd, 1u, 1u);
    // descriptors of the tile bases; k-steps / k-blocks / buffers only add to the 14-bit start-address field (>> 4)
    const uint64_t dQ = make_desc_kmajor(smem_u32(smQ));
    const uint64_t dEk = make_desc_kmajor(smem_u32(smE));
    const uint64_t dGm = make_desc(smem_u32(smG), kTile, 1024);
    const uint64_t dEm = make_desc(smem_u32(smE), kTile, 1024);
    const int nk_last = (min(64, p.d - (p.KB - 1) * 64) + 15) >> 4;
    auto issue_S = [&](int j) {
      const int buf = j & 1, n = j >> 1;
      if (p.trace && blockIdx.x == 0 && leader) p.trace[j * 8 + TR_S_ISSUE] = clock64();
      mbar_wait_guarded(&bar[B_SEMPTY + buf], (uint32_t)((n & 1) ^ 1));
      tc_fence_after();
      const uint32_t tS = tmem + kColS + buf * 128;
      for (int kb = 0; kb < p.KB; ++kb) {
        mbar_wait_guarded(&bar[B_EFULL + buf * 4 + kb], (uint32_t)(n & 1));
        tc_fence_after();
        const uint64_t da = dEk + (uint64_t)((buf * kEBuf + kb * kTile) >> 4), db = dQ + (uint64_t)((kb * kTile) >> 4);
        const int nk = kb == p.KB - 1 ? nk_last : 4;
        if (leader) {
          mma_bf16(tS, da, db, idescS, kb ? 1u : 0u);
          if (nk > 1) mma_bf16(tS, da + 2, db + 2, idescS, 1u);
          if (nk > 2) mma_bf16(tS, da + 4, db + 4, idescS, 1u);
          if (nk > 3) mma_bf16(tS, da + 6, db + 6, idescS, 1u);
        }
        __syncwarp();
      }
      if (leader) mma_commit(&bar[B_SFULL + buf]);
      if (p.trace && blockIdx.x == 0 && leader) p.trace[j * 8 + TR_S_ISSUED] = clock64();
      __syncwarp();
    };
    mbar_wait_guarded(&bar[B_QFULL], 0);
    tc_fence_after();
    issue_S(0);
    for (int i = 0; i < T; ++i) {
      if (i + 1 < T) issue_S(i + 1);             // keeps the tensor pipe busy while the epilogue works on tile i
      mbar_wait_guarded(&bar[B_GFULL], (uint32_t)(i & 1));
      tc_fence_after();
      if (p.trace && blockIdx.x == 0 && leader) p.trace[i * 8 + TR_G_SEEN] = clock64();
      // dq[128 queries, Nd] += G^T[queries, 128 entities] . E_t[128 entities, Nd]: both operands MN-major
      // (A: two 64-query chunks 16 KB apart; B: d/64 column chunks 16 KB apart; 16 entity rows = 2048 B per MMA)
      const uint64_t db = dEm + (uint64_t)(((i & 1) * kEBuf) >> 4);
      if (leader) {
#pragma unroll
        for (int k = 0; k < 8; ++k) mma_bf16(tmem, dGm + (uint64_t)(k * 128), db + (uint64_t)(k * 128), idescD, (i | k) ? 1u : 0u);
        mma_commit(&bar[B_EEMPTY + (i & 1)]);
        mma_commit(&bar[B_GEMPTY]);
        if (p.trace && blockIdx.x == 0) p.trace[i * 8 + TR_DQ_ISSUED] = clock64();
      }
      __syncwarp();
    }
    if (leader) mma_commit(&bar[B_DQFULL]);
    __syncwarp();
  } else if (warp == 3) {
    // ===================================================================== G tile -> HBM (TMA store)
    const bool leader = elect_one();
    if (leader) tma_prefetch_desc(&tG);
    for (int i = 0; i < T; ++i) {
      mbar_wait_guarded(&bar[B_GFULL], (uint32_t)(i & 1));
      if (leader) {
        if (qb * 128 < p.B) tma_store_2d(&tG, smG, qb * 128, (t0 + i) * 128);
        if (qb * 128 + 64 < p.B) tma_store_2d(&tG, smG + kTile, qb * 128 + 64, (t0 + i) * 128);
        tma_store_commit();
        tma_store_wait_read();
        mbar_arrive(&bar[B_GEMPTY]);
      }
      __syncwarp();
    }
    if (leader) tma_store_wait_all();
    __syncwarp();
  } else if (warp >= 4) {
    // ===================================================================== epilogue
    const int ew = warp - 4, quarter = warp & 3, cg = ew >> 2;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const int rit = quarter * 32 + lane;                       // row in tile
    const int qcol0 = qb * 128 + cg * 32;                      // first query of this warp's chunk
    const int ncol = p.B - qcol0;                              // warp-uniform
    const uint32_t vm = ncol >= 32 ? 0xFFFFFFFFu : (ncol > 0 ? ((1u << ncol) - 1u) : 0u);
    const int widx = min(qcol0 >> 5, p.wordsB - 1);
    double loss_acc = 0.0;
    auto load_row = [&](int tile, float& b, uint32_t& w) {
      const int64_t rc = min((int64_t)tile * 128 + rit, p.Ns - 1);
      b = __ldg(p.bias + rc);
      w = __ldg(p.bitsT + rc * p.wordsB + widx);
    };
    float bias_nx;
    uint32_t w_nx;
    load_row(t0, bias_nx, w_nx);
    uint8_t* g_dst = smG + (cg >> 1) * kTile + rit * 128;
    const int u0 = (cg & 1) * 4, sw = rit & 7;
    for (int i = 0; i < T; ++i) {
      const int sb = i & 1, n = i >> 1;
      const float bias = bias_nx;
      const uint32_t wbits = w_nx;
      if (i + 1 < T) load_row(t0 + i + 1, bias_nx, w_nx);
      const int64_t row = (int64_t)(t0 + i) * 128 + rit;
      const bool rowok = row < p.Ns;
      mbar_wait_guarded(&bar[B_SFULL + sb], (uint32_t)(n & 1));
      tc_fence_after();
      const bool tr = p.trace && blockIdx.x == 0 && ew == 0 && lane == 0;
      if (tr) p.trace[i * 8 + TR_S_SEEN] = clock64();
      uint32_t r[32];
      tmem_ld32(tmem + kColS + sb * 128 + cg * 32 + lane_base, r);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[B_SEMPTY + sb]);         // the S buffer is free as soon as it is in registers
      float g[32];
      float lsum = 0.f, gsum = 0.f;
      const uint32_t w = rowok ? (wbits & vm) : 0u;
      if (ncol <= 0) {
#pragma unroll
        for (int j = 0; j < 32; ++j) g[j] = 0.f;
      } else if (ncol < 32 || __any_sync(0xffffffffu, w != 0u)) {
        bce_chunk_general(r, bias, w, vm, p.pos, p.neg, p.ic, g, lsum, gsum);
      } else {
        bce_chunk_dense(r, bias, p.neg, p.ic, g, lsum, gsum);
      }
      if (rowok) loss_acc += (double)lsum;
      const float rsum = rowok ? gsum : 0.f;
      uint4 pk[4];
#pragma unroll
      for (int v = 0; v < 4; ++v) pk[v] = bf16_pack8(g + 8 * v);
      if (tr) p.trace[i * 8 + TR_EPI_MATH_DONE] = clock64();
      // the G tile of the previous entity tile must have been consumed (dq MMAs + TMA store) before it is overwritten
      mbar_wait_guarded(&bar[B_GEMPTY], (uint32_t)((i & 1) ^ 1));
#pragma unroll
      for (int v = 0; v < 4; ++v) *reinterpret_cast<uint4*>(g_dst + (((u0 + v) ^ sw) << 4)) = pk[v];
      fence_proxy_async();                                     // generic-proxy writes -> visible to tcgen05.mma / TMA
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[B_GFULL]);
      if (tr) p.trace[i * 8 + TR_G_WRITTEN] = clock64();
      // dbias[n] = sum over the CTA's 128 queries: column groups 1..3 hand their row sums to group 0
      if (cg > 0) {
        mbar_wait_guarded(&bar[B_DBFREE], (uint32_t)((i & 1) ^ 1));
        dbs[(cg - 1) * 128 + rit] = rsum;
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar[B_DBFULL]);
      } else {
        mbar_wait_guarded(&bar[B_DBFULL], (uint32_t)(i & 1));
        const float tot = ((rsum + dbs[rit]) + dbs[128 + rit]) + dbs[256 + rit];
        if (rowok) p.dbias_part[(int64_t)qb * p.Ns + row] = tot;
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar[B_DBFREE]);
      }
    }
    // ---- drain the dq accumulator: [128 queries x d] fp32 -> this CTA's slab
    mbar_wait_guarded(&bar[B_DQFULL], 0);
    tc_fence_after();
    const int q = qb * 128 + rit;
    for (int cc = cg; cc < 8; cc += 4) {
      const int col = cc * 32;
      if (col < p.d) {                                         // warp-uniform
        uint32_t r[32];
        tmem_ld32(tmem + (uint32_t)col + lane_base, r);
        tmem_ld_wait();
        if (q < p.B) {
          float* o = p.dq_part + ((int64_t)rr * p.B + q) * p.d + col;
          if (col + 32 <= p.d && (p.d & 3) == 0) {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              *reinterpret_cast<float4*>(o + j) = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                                              __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col + j < p.d) o[j] = __uint_as_float(r[j]);
          }
        }
      }
    }
    const double t = warp_sum_d(loss_acc);
    if (lane == 0) p.loss_part[(int64_t)blockIdx.x * kEpiWarps + ew] = t;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// ------------------------------------------------------------------------------------------ host side
static long long* g_fused_trace = nullptr;      // dev tool (tools/fused_trace.py): device buffer [tiles of CTA 0][8]
bool umma_fused_ok(int B, int64_t Ns, int d, int prec) {
  return prec == COPER_PREC_BF16 && d <= 64 * fz::kKbMax && B >= 1 && Ns >= 1 && Ns <= 0x7fffffff - 512;
}
void umma_fused_plan(int B, int64_t Ns, int* QB, int* R) {
  const int qb = (B + 127) / 128;
  const int64_t m_tiles = (Ns + 127) / 128;
  int r = sm_count() / qb;
  if (r < 1) r = 1;
  if (r > m_tiles) r = (int)m_tiles;
  *QB = qb;
  *R = r;
}

// E / q in prepared (bf16) form; GT [Ns, ldGT] bf16 out; dq_part [R][B][d], dbias_part [QB][Ns], loss_part [QB*R][16]
int umma_bce_dq_fused(const TcOperand& E, const TcOperand& Q, const float* bias, const uint32_t* bitsT, int B, int64_t Ns,
                      int d, float pos, float neg, float inv_count, void* GT, int64_t ldGT, float* dq_part,
                      float* dbias_part, double* loss_part, int* grid_out, cudaStream_t st) {
  using namespace fz;
  CUtensorMap tE, tQ, tG;
  int rc;
  if ((rc = make_tmap_2d(&tE, E.main, 2, true, E.rows, E.cols, E.pitch, 64, 128))) return rc;
  if ((rc = make_tmap_2d(&tQ, Q.main, 2, true, Q.rows, Q.cols, Q.pitch, 64, 128))) return rc;
  if ((rc = make_tmap_2d(&tG, GT, 2, true, (uint64_t)Ns, (uint64_t)B, (uint64_t)ldGT, 64, 128))) return rc;
  Params p;
  p.B = B; p.d = d; p.KB = (d + 63) / 64; p.Nd = (d + 15) / 16 * 16; p.Ns = Ns;
  p.m_tiles = (int)((Ns + 127) / 128);
  umma_fused_plan(B, Ns, &p.QB, &p.R);
  p.bias = bias; p.bitsT = bitsT; p.wordsB = (B + 31) / 32;
  p.pos = pos; p.neg = neg; p.ic = inv_count;
  p.dq_part = dq_part; p.dbias_part = dbias_part; p.loss_part = loss_part;
  p.trace = g_fused_trace;
  int dev = 0;
  if ((rc = check_cuda(cudaGetDevice(&dev)))) return rc;
  static bool attr_done[64] = {};
  if (dev < 0 || dev >= 64) return COPER_ERR_UNSUPPORTED;
  if (!attr_done[dev]) {
    if ((rc = check_cuda(cudaFuncSetAttribute(bce_dq_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              kSmemBytes))))
      return rc;
    attr_done[dev] = true;
  }
  const int grid = p.QB * p.R;
  *grid_out = grid;
  launch_pdl(bce_dq_fused_kernel, grid, kThreads, kSmemBytes, st, tE, tQ, tG, p);
  return check_launch();
}

}  // namespace coper

extern "C" void coper_debug_set_fused_trace(long long* device_buffer) { coper::g_fused_trace = device_buffer; }
