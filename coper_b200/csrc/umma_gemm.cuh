// Warp-specialised tcgen05 GEMM building blocks (sm_100a):
//   warp 0  : TMA producer   (one elected lane)  global -> 128B-swizzled smem ring, mbarrier complete_tx
//   warp 1  : MMA issuer     (one elected lane)  tcgen05.mma smem x smem -> fp32 accumulators in TMEM
//   warp 2  : TMEM allocator
//   warps 4+: epilogue       tcgen05.ld TMEM -> registers -> fused epilogue -> HBM
// D[128 x BLOCK_N] = sum_k A[m,k] * B[n,k]; accumulators are double-buffered in TMEM so the epilogue of tile i
// overlaps the MMAs of tile i+1.  Two arithmetic modes:
//   PREC_BF16  : bf16 operands, 1 MMA per k-step (kind::f16)
//   PREC_TF32X3: fp32 operands pre-split into (hi, lo) tf32 planes, 3 MMAs per k-step
//                (lo*hi + hi*lo + hi*hi; kind::tf32) -> fp32-class accuracy on the tensor pipe.
//   PREC_FP16X3: the same 3-term scheme on IEEE fp16 (hi, lo) planes of x * 2^e (kind::f16: twice the MMA rate, half the
//                operand bytes).  fp16 carries tf32's 11-bit significand; the per-operand exponents e (device int32,
//                written by the operand preparation from the operand's max |x|) are removed from the accumulators
//                right after they are read from TMEM (acc * 2^-(ea+eb) * post_scale).
// Operands may be K-major (rows x 128 B tiles) or MN-major (k-rows x 128 B chunks); see umma.cuh.
#pragma once
#include "operand.cuh"
#include "umma.cuh"

namespace coper {
namespace umma {

constexpr int PREC_BF16 = COPER_PREC_BF16, PREC_TF32X3 = COPER_PREC_TF32X3, PREC_FP16X3 = COPER_PREC_FP16X3;
constexpr int BLOCK_M = 128;
constexpr int NUM_NON_EPI_THREADS = 128;

// PROMOTE_KB > 0: the tensor core accumulates in fp32 with truncation, so a long chain of MMAs drifts (~2^-25 per
// accumulate, linear in chain length).  Chains are therefore cut every PROMOTE_KB k-blocks; each partial chain is
// read back from TMEM and added in fp32 registers (round-to-nearest) by the epilogue warps ("promotion").
// RES_KB > 0 ("resident B"): the whole K extent (<= RES_KB k-blocks) of the B tile is loaded ONCE per n-block into
// a dedicated shared-memory region and reused by every tile of the CTA that shares the n-block; only A tiles stream
// through the stage ring.  For the entity-major scorers (B = the query block) this cuts the L2->SM traffic per tile
// from (A + B) to A, which is what bounds a 128 x 128 x 256 bf16 tile on B200 (~42 B/clk/SM of TMA throughput).
// RES_A_KB > 0 ("resident A"): for problems whose A coordinates do not depend on the group (the generator backward's
// T-kernel loops over dc groups with the same dy tile): the A k-blocks of one (m-block, split), at most RES_A_KB of
// them, are loaded ONCE into a dedicated region, one mbarrier per k-block, and serve every group; only B tiles stream
// through the stage ring.  The region is refilled for the next (m-block, split) only after every MMA reading it has
// completed.
template <int PREC_, int BLOCK_N_, int STAGES_, int EPI_WARPS_, bool A_MN_, bool B_MN_, int PROMOTE_KB_ = 0,
          int RES_KB_ = 0, int RES_A_KB_ = 0>
struct GemmCfg {
  static constexpr int PROMOTE_KB = PROMOTE_KB_;
  static constexpr int RES_KB = RES_KB_;
  static constexpr int RES_A_KB = RES_A_KB_;
  static constexpr int PREC = PREC_, BLOCK_N = BLOCK_N_, STAGES = STAGES_, EPI_WARPS = EPI_WARPS_;
  static constexpr bool A_MN = A_MN_, B_MN = B_MN_;
  static constexpr int ELEM = (PREC == PREC_TF32X3) ? 4 : 2;
  static constexpr int CHUNK = 128 / ELEM;          // elements per 128-byte swizzle row: 64 bf16 / 32 tf32
  static constexpr int BLOCK_K = CHUNK;             // k elements per pipeline stage
  static constexpr int UMMA_K = 32 / ELEM;          // 16 bf16 / 8 tf32
  static constexpr int TERMS = (PREC == PREC_BF16) ? 1 : 2;     // operand planes (hi, lo)
  static constexpr bool SCALED = (PREC == PREC_FP16X3);         // accumulators carry 2^(ea+eb)
  static constexpr int A_BYTES = BLOCK_M * 128;     // one plane of the A tile (BLOCK_M x BLOCK_K or BLOCK_K x BLOCK_M)
  static constexpr int B_BYTES = BLOCK_N * 128;
  static constexpr int STAGE_BYTES = RES_KB_ > 0     ? TERMS * A_BYTES
                                     : RES_A_KB_ > 0 ? TERMS * B_BYTES
                                                     : TERMS * (A_BYTES + B_BYTES);
  static constexpr int RES_PLANE_BYTES = RES_KB_ > 0 ? B_BYTES : A_BYTES;
  static constexpr int RES_BYTES = (RES_KB_ + RES_A_KB_) * TERMS * RES_PLANE_BYTES;
  static constexpr int BARRIERS = 2 * STAGES + 2 + 2 + 1 + RES_A_KB_;   // full, empty, tfull, tempty, bfull, afull
  static constexpr int TMEM_COLS = (2 * BLOCK_N <= 32) ? 32 : (2 * BLOCK_N <= 64) ? 64 : (2 * BLOCK_N <= 128) ? 128
                                   : (2 * BLOCK_N <= 256) ? 256 : 512;
  static constexpr int THREADS = NUM_NON_EPI_THREADS + EPI_WARPS * 32;
  static constexpr size_t SMEM_BYTES = (size_t)STAGES * STAGE_BYTES + RES_BYTES + 1024 /*align*/ + 256 /*barriers*/;
  static_assert(RES_KB_ == 0 || RES_A_KB_ == 0, "one resident operand");
  static_assert(BARRIERS * 8 + 4 <= 256, "barriers + TMEM address");
  static_assert(SMEM_BYTES <= 227 * 1024, "dynamic shared memory of one CTA");

  static constexpr uint32_t FMT = (PREC == PREC_BF16) ? FMT_BF16 : (PREC == PREC_FP16X3) ? FMT_F16 : FMT_TF32;
  // MN-major smem layout: 16-bit types use the plain 128B swizzle (8-row k atoms); tf32 must use the
  // 128B swizzle with 32-byte atoms (4-row k atoms)
  static constexpr bool MN_ATOM32 = (PREC == PREC_TF32X3);
  static constexpr uint32_t MN_LAYOUT = MN_ATOM32 ? LAYOUT_SW128_BASE32B : LAYOUT_SW128;
  static constexpr uint32_t MN_SBO = MN_ATOM32 ? 512 : 1024;
  static constexpr uint32_t IDESC = make_idesc(FMT, BLOCK_M, BLOCK_N, A_MN ? 1u : 0u, B_MN ? 1u : 0u);
  static_assert(BLOCK_N % 16 == 0 && BLOCK_N >= 16 && BLOCK_N <= 256, "UMMA N");
  static_assert(2 * BLOCK_N <= 512, "TMEM double buffer");
  static_assert(!A_MN || (BLOCK_M % CHUNK == 0), "MN-major A chunking");
  static_assert(!B_MN || (BLOCK_N % CHUNK == 0), "MN-major B chunking");
};

template <class Cfg>
struct SmemLayout {
  uint8_t* base;        // 1024-aligned
  uint64_t* full;       // [STAGES]
  uint64_t* empty;      // [STAGES]
  uint64_t* tfull;      // [2]
  uint64_t* tempty;     // [2]
  uint64_t* bfull;      // [1] resident B loaded
  uint64_t* afull;      // [RES_A_KB] resident A k-block loaded
  uint32_t* tmem_ptr;
  uint8_t* res;         // resident region: B [RES_KB][TERMS][B_BYTES] or A [RES_A_KB][TERMS][A_BYTES]
  __device__ __forceinline__ explicit SmemLayout(uint8_t* raw) {
    base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~uintptr_t(1023));
    res = base + (size_t)Cfg::STAGES * Cfg::STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(res + Cfg::RES_BYTES);
    full = bars;
    empty = bars + Cfg::STAGES;
    tfull = bars + 2 * Cfg::STAGES;
    tempty = tfull + 2;
    bfull = tempty + 2;
    afull = bfull + 1;
    tmem_ptr = reinterpret_cast<uint32_t*>(afull + Cfg::RES_A_KB);
  }
  __device__ __forceinline__ uint8_t* res_plane(int kb, int term) const {
    return res + ((size_t)kb * Cfg::TERMS + term) * Cfg::RES_PLANE_BYTES;
  }
  __device__ __forceinline__ uint8_t* a_plane(int stage, int term) const {   // streaming-A configurations only
    return base + (size_t)stage * Cfg::STAGE_BYTES + term * Cfg::A_BYTES;
  }
  __device__ __forceinline__ uint8_t* b_plane(int stage, int term) const {   // streaming-B configurations only
    return base + (size_t)stage * Cfg::STAGE_BYTES + (Cfg::RES_A_KB > 0 ? 0 : Cfg::TERMS * Cfg::A_BYTES) +
           term * Cfg::B_BYTES;
  }
};

// One-time CTA setup: barriers + TMEM allocation.  Returns the TMEM base address.
template <class Cfg>
__device__ __forceinline__ uint32_t cta_setup(const SmemLayout<Cfg>& sm) {
  int warp = threadIdx.x >> 5;
  if (warp == 1 && (threadIdx.x & 31) == 0) {
    for (int i = 0; i < Cfg::STAGES; ++i) { mbar_init(&sm.full[i], 1); mbar_init(&sm.empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&sm.tfull[i], 1); mbar_init(&sm.tempty[i], Cfg::EPI_WARPS); }
    mbar_init(sm.bfull, 1);
    for (int i = 0; i < Cfg::RES_A_KB; ++i) mbar_init(&sm.afull[i], 1);
    fence_barrier_init();
  } else if (warp == 2) {
    tmem_alloc(sm.tmem_ptr, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return *sm.tmem_ptr;
}
template <class Cfg>
__device__ __forceinline__ void cta_teardown(uint32_t tmem_base) {
  tc_fence_before();
  __syncthreads();
  if ((threadIdx.x >> 5) == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// One plane of the A tile (a_mn0 = first M index, a_k0 = first k element) into dst, completing on bar.
// K-major operand: tensor map over [rows = MN, cols = K], one box {BLOCK_K, rows}.
// MN-major operand: tensor map over [rows = K, cols = MN], boxes {CHUNK, BLOCK_K} per 128-byte MN chunk.
template <class Cfg>
__device__ __forceinline__ void load_a_plane(uint8_t* dst, const CUtensorMap* ma, uint64_t* bar, int a_mn0, int a_k0,
                                             bool leader) {
  if (!Cfg::A_MN) {
    if (leader) tma_load_2d(dst, ma, bar, a_k0, a_mn0);
  } else {
#pragma unroll
    for (int c = 0; c < BLOCK_M / Cfg::CHUNK; ++c)
      if (leader) tma_load_2d(dst + c * (Cfg::BLOCK_K * 128), ma, bar, a_mn0 + c * Cfg::CHUNK, a_k0);
  }
}

// Producer: fill one stage.  (a_mn0, b_mn0) = first row (M / N index) of the tiles, k0 = first k element.
template <class Cfg>
__device__ __forceinline__ void produce_stage(const SmemLayout<Cfg>& sm, int stage, const CUtensorMap* tA,
                                              const CUtensorMap* tAlo, const CUtensorMap* tB, const CUtensorMap* tBlo,
                                              int a_mn0, int b_mn0, int a_k0, int b_k0, bool leader) {
  // called warp-uniformly; only the leader lane issues (see elect_one in umma.cuh)
  uint64_t* bar = &sm.full[stage];
  if (leader) mbar_expect_tx(bar, Cfg::STAGE_BYTES);
#pragma unroll
  for (int t = 0; t < Cfg::TERMS; ++t) {
    const CUtensorMap* mb = t ? tBlo : tB;
    if (Cfg::RES_A_KB == 0) load_a_plane<Cfg>(sm.a_plane(stage, t), t ? tAlo : tA, bar, a_mn0, a_k0, leader);
    if (Cfg::RES_KB > 0) {
      // B is resident: nothing to stream
    } else if (!Cfg::B_MN) {
      if (leader) tma_load_2d(sm.b_plane(stage, t), mb, bar, b_k0, b_mn0);
    } else {
#pragma unroll
      for (int c = 0; c < Cfg::BLOCK_N / Cfg::CHUNK; ++c)
        if (leader) tma_load_2d(sm.b_plane(stage, t) + c * (Cfg::BLOCK_K * 128), mb, bar, b_mn0 + c * Cfg::CHUNK, b_k0);
    }
  }
}

// same as issue_stage but with a run-time instruction descriptor (N of the last tile may be < BLOCK_N).
// Called warp-uniformly; only the leader lane issues.  The descriptors of the stage bases are built once, a k-step only
// adds to the start-address field (>> 4 units; shared-memory addresses are < 256 KB, so the 14-bit field cannot carry).
template <class Cfg>
__device__ __forceinline__ void issue_stage_rt(const SmemLayout<Cfg>& sm, int stage, uint32_t tmem_d, int kvalid,
                                               bool first, uint32_t idesc, int kb_res, bool leader) {
  const int nk = (kvalid + Cfg::UMMA_K - 1) / Cfg::UMMA_K;
  uint64_t da[2], db[2];
#pragma unroll
  for (int t = 0; t < Cfg::TERMS; ++t) {
    const uint32_t a_addr = smem_u32(Cfg::RES_A_KB > 0 ? sm.res_plane(kb_res, t) : sm.a_plane(stage, t));
    const uint32_t b_addr = smem_u32(Cfg::RES_KB > 0 ? sm.res_plane(kb_res, t) : sm.b_plane(stage, t));
    da[t] = Cfg::A_MN ? make_desc(a_addr, Cfg::BLOCK_K * 128, Cfg::MN_SBO, Cfg::MN_LAYOUT) : make_desc_kmajor(a_addr);
    db[t] = Cfg::B_MN ? make_desc(b_addr, Cfg::BLOCK_K * 128, Cfg::MN_SBO, Cfg::MN_LAYOUT) : make_desc_kmajor(b_addr);
  }
  // K-major: step 32 bytes inside the 128-byte swizzle row; MN-major: step UMMA_K k-rows of 128 bytes
  constexpr uint64_t a_step = (Cfg::A_MN ? Cfg::UMMA_K * 128 : 32) >> 4, b_step = (Cfg::B_MN ? Cfg::UMMA_K * 128 : 32) >> 4;
  constexpr int NK_MAX = Cfg::BLOCK_K / Cfg::UMMA_K;
  if (leader) {
#pragma unroll
    for (int k = 0; k < NK_MAX; ++k) {
      if (k < nk) {
        const uint32_t acc = (first && k == 0) ? 0u : 1u;
        if (Cfg::PREC == PREC_BF16) {
          mma_bf16(tmem_d, da[0] + k * a_step, db[0] + k * b_step, idesc, acc);
        } else if (Cfg::PREC == PREC_FP16X3) {                                    // kind::f16 on fp16 planes
          mma_bf16(tmem_d, da[1] + k * a_step, db[0] + k * b_step, idesc, acc);   // lo * hi
          mma_bf16(tmem_d, da[0] + k * a_step, db[1] + k * b_step, idesc, 1u);    // hi * lo
          mma_bf16(tmem_d, da[0] + k * a_step, db[0] + k * b_step, idesc, 1u);    // hi * hi
        } else {
          mma_tf32(tmem_d, da[1] + k * a_step, db[0] + k * b_step, idesc, acc);   // lo * hi
          mma_tf32(tmem_d, da[0] + k * a_step, db[1] + k * b_step, idesc, 1u);    // hi * lo
          mma_tf32(tmem_d, da[0] + k * a_step, db[0] + k * b_step, idesc, 1u);    // hi * hi
        }
      }
    }
  }
  __syncwarp();
}

struct PipeState {
  int stage = 0;
  uint32_t phase = 0;
  template <int STAGES>
  __device__ __forceinline__ void advance() {
    if (++stage == STAGES) { stage = 0; phase ^= 1; }
  }
};

// Producer, before refilling a resident region: every stage of the ring has been released, i.e. every MMA issued so
// far (all of which may read the resident region) has completed.
template <class Cfg>
__device__ __forceinline__ void wait_ring_drained(const SmemLayout<Cfg>& sm, PipeState q) {
  for (int i = 0; i < Cfg::STAGES; ++i) {
    mbar_wait(&sm.empty[q.stage], q.phase ^ 1);
    q.template advance<Cfg::STAGES>();
  }
}

}  // namespace umma
}  // namespace coper

// ================================================================================================
// Generic persistent kernel: grouped / split-K GEMM with a pluggable epilogue.
// ================================================================================================
namespace coper {
namespace umma {

struct GemmProblem {
  int M, N, K;                  // per-group extents: M -> TMEM lanes (rows), N -> TMEM columns, K reduction
  int m_tiles, n_tiles;
  int splits, kb_per_split;     // split-K in units of BLOCK_K blocks (every split must be non-empty)
  int groups;                   // number of groups (e.g. context index kq)
  int groups_inner;             // 0: groups are independent work items; 1: a CTA loops over all groups of one
                                //    (m_blk, n_blk, split) consecutively (epilogue may accumulate across groups)
  int a_group_mn, a_group_k;    // per-group coordinate offsets into the operand tensor maps
  int b_group_mn, b_group_k;
  const int* exp_a;             // PREC_FP16X3: device exponents of the two operands (NULL = 0) and a host-known
  const int* exp_b;             //   factor: accumulators are multiplied by 2^-(*exp_a + *exp_b) * post_scale
  float post_scale;             //   (0 is read as 1)
  int n_fastest;                // 0: tiles enumerated m-block fastest (default); 1: n-block fastest - with a grid that
                                //    is a multiple of n_tiles every CTA keeps ONE n-block (resident B is loaded once)
                                //    and neighbouring CTAs work on the same m-block at the same time, so the A tile
                                //    is fetched from HBM once and served from L2 to the other n-blocks
};
struct TileCoord {
  int group, split, m_blk, n_blk, kb0, kb1;
};

struct EpiBase {
  static constexpr bool kAccumulate = false;
  __device__ __forceinline__ void tile_begin(const GemmProblem&, const TileCoord&, int, int) {}
  __device__ __forceinline__ void tile_prefetch(const GemmProblem&, const TileCoord&, int, int) {}
  __device__ __forceinline__ float group_scale(const GemmProblem&, const TileCoord&, int) const { return 1.0f; }
  __device__ __forceinline__ void group_vals(const GemmProblem&, const TileCoord&, int, int, const uint32_t (&)[16],
                                             int) {}
  __device__ __forceinline__ void group_done(const GemmProblem&, const TileCoord&, int, int, int) {}
  __device__ __forceinline__ void tile_done(const GemmProblem&, const TileCoord&, int, int, int) {}
  __device__ __forceinline__ void finish(int, int) {}
};

__device__ __forceinline__ long long gemm_supers(const GemmProblem& p) {
  return (long long)p.m_tiles * p.n_tiles * p.splits * (p.groups_inner ? 1 : p.groups);
}
__device__ __forceinline__ TileCoord gemm_decode(const GemmProblem& p, long long s, int g_inner, int block_k) {
  TileCoord t;
  if (p.n_fastest) {
    t.n_blk = (int)(s % p.n_tiles); s /= p.n_tiles;
    t.m_blk = (int)(s % p.m_tiles); s /= p.m_tiles;
  } else {
    t.m_blk = (int)(s % p.m_tiles); s /= p.m_tiles;
    t.n_blk = (int)(s % p.n_tiles); s /= p.n_tiles;
  }
  t.split = (int)(s % p.splits);  s /= p.splits;
  t.group = p.groups_inner ? g_inner : (int)s;
  int kb_total = (p.K + block_k - 1) / block_k;
  t.kb0 = t.split * p.kb_per_split;
  t.kb1 = min(kb_total, t.kb0 + p.kb_per_split);
  return t;
}

// Epi concept (derive from EpiBase for the no-op defaults):
//   static constexpr bool kAccumulate   the output tile is the sum over the inner group loop (groups_inner = 1) of
//                                       group_scale(row, group) * partial tile, accumulated in fp32 registers
//   void tile_begin(p, t, row, col0)    before waiting for the accumulators (issue global prefetches here);
//                                       col0 = first N index of this warp's column range
//   void tile_prefetch(p, t_next, row_next, col0_next)   right after tile_begin, with the coordinates of the tile
//                                       this CTA processes next (issue its global loads here)
//   float group_scale(p, t, row)        kAccumulate: multiplier of this group's partial tile for this row
//   void group_vals(p, t, row, col, const uint32_t (&v)[16], int half_idx)   kAccumulate: raw partial values
//   void group_done(p, t, row, col_group, col_groups)                         kAccumulate: after each group
//   void chunk(p, t, row, col, const uint32_t (&acc)[32], int chunk_idx)
//       row = global M index of this thread's TMEM lane, col = global N index of acc[0]; called for every 32-column
//       chunk this warp owns (warp-uniform), also for rows >= M (mask inside).
//   void tile_done(p, t, row, col_group, col_groups);
//   void finish(int epi_thread, int epi_threads);   // once per CTA, after the last tile
template <class Cfg, class Epi>
__global__ void __launch_bounds__(Cfg::THREADS, 1)
umma_gemm_kernel(const __grid_constant__ CUtensorMap tA, const __grid_constant__ CUtensorMap tAlo,
                 const __grid_constant__ CUtensorMap tB, const __grid_constant__ CUtensorMap tBlo,
                 const GemmProblem p, Epi epi) {
  coper::pdl_trigger();                          // the next kernel of the stream may be scheduled (common.cuh)
  extern __shared__ uint8_t smem_raw[];
  SmemLayout<Cfg> sm(smem_raw);
  uint32_t tmem_base = cta_setup<Cfg>(sm);
  coper::pdl_wait();                             // barriers / TMEM are set up; from here on the predecessor's output is read
  const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;
  const long long supers = gemm_supers(p);
  const int g_loop = p.groups_inner ? p.groups : 1;

  if (warp == 0) {
    // TMA producer: the loop is warp-uniform, only the leader lane issues
    const bool leader = elect_one();
    if (leader) {
      tma_prefetch_desc(&tA);
      tma_prefetch_desc(&tB);
    }
    PipeState ps;
    int res_nblk = -1, res_a_key = -1;
    for (long long s = blockIdx.x; s < supers; s += gridDim.x) {
      for (int g = 0; g < g_loop; ++g) {
        TileCoord t = gemm_decode(p, s, g, Cfg::BLOCK_K);
        int a_mn0 = t.m_blk * BLOCK_M + t.group * p.a_group_mn;
        int b_mn0 = t.n_blk * Cfg::BLOCK_N + t.group * p.b_group_mn;
        bool load_a = false;       // resident A: this group pass also loads the A k-blocks of (m_blk, split)
        if (Cfg::RES_A_KB > 0 && g == 0 && t.split * p.m_tiles + t.m_blk != res_a_key) {
          wait_ring_drained<Cfg>(sm, ps);
          res_a_key = t.split * p.m_tiles + t.m_blk;
          load_a = true;
        }
        if (Cfg::RES_KB > 0 && t.n_blk != res_nblk) {
          // new n-block: wait until every MMA that reads the old resident B has completed (all stages drained),
          // then load the whole K extent of the new B tile
          wait_ring_drained<Cfg>(sm, ps);
          const int kbn = t.kb1 - t.kb0;
          if (leader) mbar_expect_tx(sm.bfull, (uint32_t)(kbn * Cfg::TERMS * Cfg::B_BYTES));
          for (int kb = t.kb0; kb < t.kb1; ++kb)
#pragma unroll
            for (int tm = 0; tm < Cfg::TERMS; ++tm) {
              if (!Cfg::B_MN) {
                if (leader)
                  tma_load_2d(sm.res_plane(kb - t.kb0, tm), tm ? &tBlo : &tB, sm.bfull, kb * Cfg::BLOCK_K, b_mn0);
              } else {
#pragma unroll
                for (int c = 0; c < Cfg::BLOCK_N / Cfg::CHUNK; ++c)
                  if (leader)
                    tma_load_2d(sm.res_plane(kb - t.kb0, tm) + c * (Cfg::BLOCK_K * 128), tm ? &tBlo : &tB, sm.bfull,
                                b_mn0 + c * Cfg::CHUNK, kb * Cfg::BLOCK_K);
              }
            }
          res_nblk = t.n_blk;
        }
        for (int kb = t.kb0; kb < t.kb1; ++kb) {
          if (Cfg::RES_A_KB > 0 && load_a) {
            // issued ahead of the stage's B tile and without waiting for a free stage: the first MMA waits only for
            // its own A k-block
            uint64_t* bar = &sm.afull[kb - t.kb0];
            if (leader) mbar_expect_tx(bar, Cfg::TERMS * Cfg::A_BYTES);
#pragma unroll
            for (int tm = 0; tm < Cfg::TERMS; ++tm)
              load_a_plane<Cfg>(sm.res_plane(kb - t.kb0, tm), tm ? &tAlo : &tA, bar, a_mn0, kb * Cfg::BLOCK_K, leader);
          }
          mbar_wait(&sm.empty[ps.stage], ps.phase ^ 1);
          produce_stage<Cfg>(sm, ps.stage, &tA, &tAlo, &tB, &tBlo, a_mn0, b_mn0,
                             kb * Cfg::BLOCK_K + t.group * p.a_group_k, kb * Cfg::BLOCK_K + t.group * p.b_group_k, leader);
          ps.template advance<Cfg::STAGES>();
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // MMA issuer: warp-uniform loop, the leader lane issues tcgen05.mma / tcgen05.commit
    const bool leader = elect_one();
    PipeState ps;
    int as = 0;
    uint32_t aphase = 0;
    int res_nblk = -1, res_a_key = -1;
    uint32_t bphase = 0;
    uint32_t a_parity = 0;         // bit i: parity of the next completion of afull[i] (a short last split skips some)
    for (long long s = blockIdx.x; s < supers; s += gridDim.x) {
      for (int g = 0; g < g_loop; ++g) {
        TileCoord t = gemm_decode(p, s, g, Cfg::BLOCK_K);
        bool wait_a = false;       // the same decision as the producer's load_a
        if (Cfg::RES_A_KB > 0 && g == 0 && t.split * p.m_tiles + t.m_blk != res_a_key) {
          res_a_key = t.split * p.m_tiles + t.m_blk;
          wait_a = true;
        }
        if (Cfg::RES_KB > 0 && t.n_blk != res_nblk) {
          mbar_wait(sm.bfull, bphase);
          bphase ^= 1;
          res_nblk = t.n_blk;
        }
        int n_rem = p.N - t.n_blk * Cfg::BLOCK_N;
        int n_eff = min(Cfg::BLOCK_N, (n_rem + 15) & ~15);
        uint32_t idesc = make_idesc(Cfg::FMT, BLOCK_M, (uint32_t)n_eff, Cfg::A_MN ? 1u : 0u, Cfg::B_MN ? 1u : 0u);
        const int chain = Cfg::PROMOTE_KB > 0 ? Cfg::PROMOTE_KB : (t.kb1 - t.kb0);
        for (int kc = t.kb0; kc < t.kb1; kc += chain) {
          int kce = min(t.kb1, kc + chain);
          mbar_wait(&sm.tempty[as], aphase ^ 1);
          tc_fence_after();
          for (int kb = kc; kb < kce; ++kb) {
            if (Cfg::RES_A_KB > 0 && wait_a) {
              const int i = kb - t.kb0;
              mbar_wait(&sm.afull[i], (a_parity >> i) & 1u);
              a_parity ^= 1u << i;
            }
            mbar_wait(&sm.full[ps.stage], ps.phase);
            tc_fence_after();
            int kvalid = min(Cfg::BLOCK_K, p.K - kb * Cfg::BLOCK_K);
            issue_stage_rt<Cfg>(sm, ps.stage, tmem_base + as * Cfg::BLOCK_N, kvalid, kb == kc, idesc, kb - t.kb0, leader);
            if (leader) mma_commit(&sm.empty[ps.stage]);
            ps.template advance<Cfg::STAGES>();
          }
          if (leader) mma_commit(&sm.tfull[as]);
          __syncwarp();
          as ^= 1;
          if (as == 0) aphase ^= 1;
        }
      }
    }
  } else if (warp >= 4) {
    const int quarter = warp & 3;
    const int group_c = (warp - 4) >> 2;
    constexpr int GROUPS = Cfg::EPI_WARPS / 4;
    constexpr int COLS = Cfg::BLOCK_N / GROUPS;
    constexpr int NCH = COLS / 32;
    static_assert(COLS % 32 == 0, "epilogue column split");
    int as = 0;
    uint32_t aphase = 0;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    // PREC_FP16X3: the operands were stored as x * 2^e -> every accumulator read from TMEM is multiplied by
    // 2^-(ea+eb) * post_scale before the epilogue sees it
    float acc_scale = 1.0f;
    if (Cfg::SCALED) {
      const int e = (p.exp_a ? __ldg(p.exp_a) : 0) + (p.exp_b ? __ldg(p.exp_b) : 0);
      acc_scale = exp2f((float)-e) * (p.post_scale != 0.f ? p.post_scale : 1.0f);
    }
    for (long long s = blockIdx.x; s < supers; s += gridDim.x) {
      TileCoord t = gemm_decode(p, s, 0, Cfg::BLOCK_K);
      const int row = t.m_blk * BLOCK_M + quarter * 32 + lane;
      const int col0 = t.n_blk * Cfg::BLOCK_N + group_c * COLS;
      epi.tile_begin(p, t, row, col0);
      if (s + gridDim.x < supers) {      // per-row data of the NEXT tile is fetched while this one is processed
        const TileCoord t2 = gemm_decode(p, s + gridDim.x, 0, Cfg::BLOCK_K);
        epi.tile_prefetch(p, t2, t2.m_blk * BLOCK_M + quarter * 32 + lane, t2.n_blk * Cfg::BLOCK_N + group_c * COLS);
      }
      if constexpr (Cfg::PROMOTE_KB == 0 && !Epi::kAccumulate) {
        // one accumulation chain per tile: TMEM -> registers -> epi.chunk
        mbar_wait(&sm.tfull[as], aphase);
        tc_fence_after();
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const int col = col0 + i * 32;
          if (col < p.N) {
            uint32_t r[32];
            tmem_ld32(tmem_base + as * Cfg::BLOCK_N + group_c * COLS + i * 32 + lane_base, r);
            tmem_ld_wait();
            if (Cfg::SCALED) {
#pragma unroll
              for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) * acc_scale);
            }
            epi.chunk(p, t, row, col, r, i);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.tempty[as]);
        as ^= 1;
        if (as == 0) aphase ^= 1;
      } else {
        // several partial chains per output tile (promotion of truncating TMEM chains and / or accumulation
        // over the inner group loop): summed in fp32 registers with round-to-nearest, optionally scaled per group
        float accr[NCH][32];
#pragma unroll
        for (int i = 0; i < NCH; ++i)
#pragma unroll
          for (int j = 0; j < 32; ++j) accr[i][j] = 0.f;
        for (int g = 0; g < g_loop; ++g) {
          t = gemm_decode(p, s, g, Cfg::BLOCK_K);
          const float scale = epi.group_scale(p, t, row);
          const int chain = Cfg::PROMOTE_KB > 0 ? Cfg::PROMOTE_KB : (t.kb1 - t.kb0);
          for (int kc = t.kb0; kc < t.kb1; kc += chain) {
            mbar_wait(&sm.tfull[as], aphase);
            tc_fence_after();
#pragma unroll
            for (int i = 0; i < NCH; ++i) {
              if (col0 + i * 32 < p.N) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                  uint32_t r[16];
                  tmem_ld16(tmem_base + as * Cfg::BLOCK_N + group_c * COLS + i * 32 + h * 16 + lane_base, r);
                  tmem_ld_wait();
                  if (Cfg::SCALED) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) * acc_scale);
                  }
                  epi.group_vals(p, t, row, col0 + i * 32 + h * 16, r, i * 2 + h);
#pragma unroll
                  for (int j = 0; j < 16; ++j) accr[i][h * 16 + j] = fmaf(scale, __uint_as_float(r[j]), accr[i][h * 16 + j]);
                }
              }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.tempty[as]);
            as ^= 1;
            if (as == 0) aphase ^= 1;
          }
          epi.group_done(p, t, row, group_c, GROUPS);
        }
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const int col = col0 + i * 32;
          if (col < p.N) {
            uint32_t r[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(accr[i][j]);
            epi.chunk(p, t, row, col, r, i);
          }
        }
      }
      epi.tile_done(p, t, row, group_c, GROUPS);
    }
    epi.finish(threadIdx.x - NUM_NON_EPI_THREADS, Cfg::EPI_WARPS * 32);
  }
  cta_teardown<Cfg>(tmem_base);
}

// Host-side description of a prepared operand (see coper_prepare_operand)
struct TcOperand {
  const void* main;
  const void* lo;        // tf32x3 / fp16x3 only
  const int* exp;        // fp16x3 only: device exponent e of the stored planes (x * 2^e); NULL = 0
  uint64_t rows, cols;   // extents of the stored row-major matrix (cols contiguous)
  uint64_t pitch;        // elements between rows
};

// Build the 4 tensor maps for a configuration.  K-major operand: stored [MN, K], box {BLOCK_K, tile rows};
// MN-major operand: stored [K, MN], box {CHUNK, BLOCK_K}.
template <class Cfg>
int make_gemm_tmaps(const TcOperand& A, const TcOperand& B, CUtensorMap* tA, CUtensorMap* tAlo, CUtensorMap* tB,
                    CUtensorMap* tBlo) {
  constexpr bool bf16 = Cfg::ELEM == 2;      // any 16-bit plane: TMA only moves bytes
  int rc;
  uint32_t a_box_rows = Cfg::A_MN ? Cfg::BLOCK_K : BLOCK_M;
  uint32_t b_box_rows = Cfg::B_MN ? Cfg::BLOCK_K : Cfg::BLOCK_N;
  const bool a32 = Cfg::A_MN && Cfg::MN_ATOM32, b32 = Cfg::B_MN && Cfg::MN_ATOM32;
  if ((rc = make_tmap_2d(tA, A.main, Cfg::ELEM, bf16, A.rows, A.cols, A.pitch, Cfg::CHUNK, a_box_rows, a32))) return rc;
  if ((rc = make_tmap_2d(tB, B.main, Cfg::ELEM, bf16, B.rows, B.cols, B.pitch, Cfg::CHUNK, b_box_rows, b32))) return rc;
  *tAlo = *tA;
  *tBlo = *tB;
  if (Cfg::TERMS == 2) {
    if (!A.lo || !B.lo) return COPER_ERR_INVALID_ARG;
    if ((rc = make_tmap_2d(tAlo, A.lo, Cfg::ELEM, bf16, A.rows, A.cols, A.pitch, Cfg::CHUNK, a_box_rows, a32))) return rc;
    if ((rc = make_tmap_2d(tBlo, B.lo, Cfg::ELEM, bf16, B.rows, B.cols, B.pitch, Cfg::CHUNK, b_box_rows, b32))) return rc;
  }
  return COPER_OK;
}

template <class Cfg, class Epi>
int launch_gemm(const TcOperand& A, const TcOperand& B, const GemmProblem& p, const Epi& epi, cudaStream_t st,
                int grid_override = 0) {
  if (p.groups_inner && !Epi::kAccumulate) return COPER_ERR_INVALID_ARG;
  if (Cfg::RES_KB > 0 && (p.splits != 1 || p.groups != 1 || (p.K + Cfg::BLOCK_K - 1) / Cfg::BLOCK_K > Cfg::RES_KB))
    return COPER_ERR_UNSUPPORTED;
  if (Cfg::RES_A_KB > 0 && (p.kb_per_split > Cfg::RES_A_KB || p.a_group_mn != 0 || p.a_group_k != 0))
    return COPER_ERR_UNSUPPORTED;
  CUtensorMap tA, tAlo, tB, tBlo;
  int rc = make_gemm_tmaps<Cfg>(A, B, &tA, &tAlo, &tB, &tBlo);
  if (rc) return rc;
  int dev = 0;
  if ((rc = check_cuda(cudaGetDevice(&dev)))) return rc;
  static bool attr_done[64] = {};               // the attribute is per device
  if (dev < 0 || dev >= 64) return COPER_ERR_UNSUPPORTED;
  if (!attr_done[dev]) {
    rc = check_cuda(cudaFuncSetAttribute(umma_gemm_kernel<Cfg, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)Cfg::SMEM_BYTES));
    if (rc) return rc;
    attr_done[dev] = true;
  }
  GemmProblem pp = p;
  if (Cfg::SCALED) {                            // operand exponents travel with the operands
    if (!pp.exp_a) pp.exp_a = A.exp;
    if (!pp.exp_b) pp.exp_b = B.exp;
  }
  const int sms = sm_count();
  long long supers = (long long)p.m_tiles * p.n_tiles * p.splits * (p.groups_inner ? 1 : p.groups);
  int grid = (int)(supers < sms ? supers : sms);
  if (grid_override > 0 && grid_override < grid) grid = grid_override;
  if (grid < 1) return COPER_ERR_INVALID_ARG;
  launch_pdl(umma_gemm_kernel<Cfg, Epi>, grid, Cfg::THREADS, Cfg::SMEM_BYTES, st, tA, tAlo, tB, tBlo, pp, epi);
  return check_launch();
}

// Fill the tiling fields of a problem; split-K chosen so that ~`target_ctas` work items exist.
template <class Cfg>
inline void plan_gemm(GemmProblem& p, bool allow_split, int target_ctas = 0) {
  if (target_ctas <= 0) target_ctas = sm_count();
  p.m_tiles = (p.M + BLOCK_M - 1) / BLOCK_M;
  p.n_tiles = (p.N + Cfg::BLOCK_N - 1) / Cfg::BLOCK_N;
  int kb_total = (p.K + Cfg::BLOCK_K - 1) / Cfg::BLOCK_K;
  long long base = (long long)p.m_tiles * p.n_tiles * (p.groups_inner ? 1 : p.groups);
  int splits = 1;
  if (allow_split && base < target_ctas) {
    splits = (int)((target_ctas + base - 1) / base);
    if (splits > kb_total) splits = kb_total;
  }
  p.kb_per_split = (kb_total + splits - 1) / splits;
  p.splits = (kb_total + p.kb_per_split - 1) / p.kb_per_split;
}

// Warp-cooperative store of a [32 rows x 32 fp32] block held one row per lane.  Writing it straight from the
// registers makes every store instruction touch 32 different rows with 16 bytes each: half-written 32-byte sectors
// that L2 completes with DRAM fill reads (measured: ~1-2 TB/s and +60 % DRAM reads).  Instead the block is staged
// through a 4 KB XOR-swizzled shared-memory tile (conflict-free 16-byte accesses both ways) and written out with
// 8 lanes per row: each instruction stores 4 rows x 128 contiguous bytes.
//   st: this warp's 256-float4 staging tile; out0: address of (row_base, col); rows_valid / cols_valid (multiple of 4)
__device__ __forceinline__ void staged_store_f32(float4* st, const float (&v)[32], float* out0, long long ld,
                                                 int rows_valid, int cols_valid) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int g = 0; g < 8; ++g)
    st[lane * 8 + (g ^ (lane & 7))] = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
  __syncwarp();
  const int g = lane & 7;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int rr = 4 * k + (lane >> 3);
    const float4 x = st[rr * 8 + (g ^ (rr & 7))];
    if (rr < rows_valid && 4 * g < cols_valid) *reinterpret_cast<float4*>(out0 + (long long)rr * ld + 4 * g) = x;
  }
  __syncwarp();
}
constexpr int kStageWarps = 8;
__device__ __forceinline__ float4* stage_tile() {
  __shared__ float4 stage_s[kStageWarps][256];
  return stage_s[((threadIdx.x >> 5) - 4) & (kStageWarps - 1)];
}

// Plain store epilogue: out[(group, split)][row, col] = acc * row_scale[row, group] (+ col_bias[col])
struct StoreEpi : EpiBase {
  float* out;
  long long ld, group_stride, split_stride;
  const float* row_scale;   // optional [M, row_scale_ld]; indexed [row, group]
  int row_scale_ld;
  const float* col_bias;    // optional [N]
  int extra_col;            // if >= 0: column index whose values go to extra_out[row] instead (e.g. dbias)
  float* extra_out;
  double* sumsq_part;       // optional [grid * epilogue warps]: sum of the squares of everything this warp stored
  double ss_acc;            //   (the gradient-norm pass of the optimizer then need not re-read the output)
  __device__ __forceinline__ void chunk(const GemmProblem& p, const TileCoord& t, int row, int col,
                                        const uint32_t (&r)[32], int) {
    const int lane = threadIdx.x & 31;
    const int n_out = extra_col >= 0 ? min(p.N, extra_col) : p.N;
    if (sumsq_part && row < p.M) {           // plain-store uses only (no row scale / bias): squares of the raw values
      float ss = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float v = __uint_as_float(r[j]);
        ss = (col + j < n_out) ? fmaf(v, v, ss) : ss;
      }
      ss_acc += (double)ss;
    }
    float* base = out + t.group * group_stride + t.split * split_stride;
    float* o0 = base + (long long)(row - lane) * ld + col;          // (first row of this warp, col)
    // warp-uniform: whole float4 granules, 16-byte aligned rows
    const bool vec = !col_bias && !row_scale && extra_col < 0 && ((ld & 3) == 0) && ((n_out & 3) == 0) &&
                     ((reinterpret_cast<uintptr_t>(o0) & 15) == 0);
    if (vec) {
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
      staged_store_f32(stage_tile(), v, o0, ld, p.M - (row - lane), n_out - col);
      return;
    }
    if (row >= p.M) return;
    float sc = row_scale ? __ldg(row_scale + (long long)row * row_scale_ld + t.group) : 1.0f;
    float* o = base + (long long)row * ld + col;
    {
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        int cj = col + j;
        if (cj < n_out) o[j] = __uint_as_float(r[j]) * sc + (col_bias ? __ldg(col_bias + cj) : 0.f);
        else if (cj == extra_col && cj < p.N) extra_out[row] = __uint_as_float(r[j]) * sc;
      }
    }
  }
  __device__ __forceinline__ void finish(int epi_thread, int epi_threads) {
    if (!sumsq_part) return;
    const double t = warp_sum_d(ss_acc);
    if ((epi_thread & 31) == 0) sumsq_part[(long long)blockIdx.x * (epi_threads >> 5) + (epi_thread >> 5)] = t;
  }
};

inline StoreEpi make_store_epi(float* out, long long ld, long long group_stride, long long split_stride) {
  StoreEpi e;
  e.out = out; e.ld = ld; e.group_stride = group_stride; e.split_stride = split_stride;
  e.row_scale = nullptr; e.row_scale_ld = 0; e.col_bias = nullptr; e.extra_col = -1; e.extra_out = nullptr;
  e.sumsq_part = nullptr; e.ss_acc = 0.0;
  return e;
}

}  // namespace umma

// ---- host entry points of the generic GEMM (umma_gemm.cu)
// a prepared operand (operand.cuh) of a stored [rows, cols] matrix, as the kernels read it
umma::TcOperand tc_operand(const void* prep, int64_t rows, int cols, int prec);
// p: M, N, K, groups, groups_inner and group offsets filled by the caller; tiling is planned here.  With split == true
// the caller must size `epi.out` for tc_plan_splits() partial slabs.
int tc_gemm_store(int prec, bool a_mn, bool b_mn, const umma::TcOperand& A, const umma::TcOperand& B,
                  const umma::GemmProblem& p, bool split, const umma::StoreEpi& epi, cudaStream_t st);
int tc_plan_splits(int prec, umma::GemmProblem p, bool split);
}  // namespace coper
