// Instantiations of the generic tcgen05 GEMM with the plain store epilogue for every operand layout
// (K-major / MN-major A and B) x {bf16, 3xTF32}, plus coper_tc_gemm: C = op(A).op(B) on the tensor pipe.
#include "umma_gemm.cuh"

namespace coper {
using namespace umma;

// N-is-small configurations (N = d <= 256 in one tile): BLOCK_N = 256
// tf32x3: 8 epilogue warps (128 promoted accumulators per thread), chains cut every 4 k-blocks (48 MMAs)
// fp16x3: a k-block holds 64 k-elements (2 x 16 KB planes per operand tile row block): chains cut every 2 k-blocks
template <int PREC, bool A_MN, bool B_MN>
using StoreCfg = GemmCfg<PREC, 256, (PREC == PREC_BF16 ? 4 : 2), (PREC == PREC_BF16 ? 4 : 8), A_MN, B_MN,
                         (PREC == PREC_BF16 ? 0 : PREC == PREC_FP16X3 ? 2 : 4)>;

template <int PREC>
static int dispatch_layout(bool a_mn, bool b_mn, const TcOperand& A, const TcOperand& B, GemmProblem p, bool split,
                           const StoreEpi& epi, cudaStream_t st) {
  if (!a_mn && !b_mn) { plan_gemm<StoreCfg<PREC, false, false>>(p, split); return launch_gemm<StoreCfg<PREC, false, false>>(A, B, p, epi, st); }
  if (!a_mn && b_mn)  { plan_gemm<StoreCfg<PREC, false, true>>(p, split);  return launch_gemm<StoreCfg<PREC, false, true>>(A, B, p, epi, st); }
  if (a_mn && !b_mn)  { plan_gemm<StoreCfg<PREC, true, false>>(p, split);  return launch_gemm<StoreCfg<PREC, true, false>>(A, B, p, epi, st); }
  plan_gemm<StoreCfg<PREC, true, true>>(p, split);
  return launch_gemm<StoreCfg<PREC, true, true>>(A, B, p, epi, st);
}

// dE-shaped problems (M = entities >> N = d, K = batch <= 512, bf16): the [K, N] operand (q) is kept RESIDENT in shared
// memory per 128-column block, only the A tiles (G) stream -> L2->SM traffic per output tile drops from A + B to A.
using ResBCfg = GemmCfg<PREC_BF16, 128, 4, 8, false, true, 0, 8>;
int tc_gemm_store_resident_b(const TcOperand& A, const TcOperand& B, GemmProblem p, const StoreEpi& epi, cudaStream_t st) {
  plan_gemm<ResBCfg>(p, false);
  return launch_gemm<ResBCfg>(A, B, p, epi, st);
}
bool tc_resident_b_ok(int prec, bool a_mn, bool b_mn, const GemmProblem& p) {
  return prec == COPER_PREC_BF16 && !a_mn && b_mn && p.groups == 1 && p.K <= ResBCfg::RES_KB * ResBCfg::BLOCK_K &&
         p.M >= 16 * BLOCK_M;
}

int tc_gemm_store(int prec, bool a_mn, bool b_mn, const TcOperand& A, const TcOperand& B, const GemmProblem& p,
                  bool split, const StoreEpi& epi, cudaStream_t st) {
  // (the resident-B variant measured slower than the streaming one for dE - the output stores dominate - and is kept
  // for reference only)
  if (prec == COPER_PREC_BF16) return dispatch_layout<PREC_BF16>(a_mn, b_mn, A, B, p, split, epi, st);
  if (prec == COPER_PREC_TF32X3) return dispatch_layout<PREC_TF32X3>(a_mn, b_mn, A, B, p, split, epi, st);
  if (prec == COPER_PREC_FP16X3) return dispatch_layout<PREC_FP16X3>(a_mn, b_mn, A, B, p, split, epi, st);
  return COPER_ERR_UNSUPPORTED;
}
// number of split-K slabs tc_gemm_store will produce for this problem (all StoreCfg share BLOCK_N / BLOCK_K per prec)
int tc_plan_splits(int prec, GemmProblem p, bool split) {
  if (prec == COPER_PREC_BF16) plan_gemm<StoreCfg<PREC_BF16, false, false>>(p, split);
  else if (prec == COPER_PREC_FP16X3) plan_gemm<StoreCfg<PREC_FP16X3, false, false>>(p, split);
  else plan_gemm<StoreCfg<PREC_TF32X3, false, false>>(p, split);
  return p.splits;
}

TcOperand tc_operand(const void* prep, int64_t rows, int cols, int prec) {
  TcOperand o;
  int64_t ldp = prepared_ld(cols, prec);
  o.main = prep;
  o.lo = prec == COPER_PREC_TF32X3 ? static_cast<const void*>(static_cast<const float*>(prep) + rows * ldp)
         : prec == COPER_PREC_FP16X3 ? static_cast<const void*>(static_cast<const uint16_t*>(prep) + rows * ldp)
                                     : nullptr;
  o.exp = prec == COPER_PREC_FP16X3 ? reinterpret_cast<const int*>(fp16x3_trailer(prep, rows, cols) + kTrExp) : nullptr;
  o.rows = (uint64_t)rows;
  o.cols = (uint64_t)cols;
  o.pitch = (uint64_t)ldp;
  return o;
}
}  // namespace coper

using namespace coper;

extern "C" {

size_t coper_tc_gemm_workspace_bytes(int M, int N, int K, int prec) {
  // operands are prepared as stored: [M,K] or [K,M] / [K,N] or [N,K] -> same byte count either way (upper bound)
  size_t a = prepared_bytes(M > K ? M : K, M > K ? K : M, prec) + prepared_bytes(K, M, prec);
  size_t b = prepared_bytes(N > K ? N : K, N > K ? K : N, prec) + prepared_bytes(K, N, prec);
  return a + b + 1024;
}

int coper_tc_gemm(int transA, int transB, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                  float* C, int ldc, int prec, void* workspace, size_t workspace_bytes, coper_stream_t stream) {
  COPER_CHECK_ARG(A && B && C && workspace && M > 0 && N > 0 && K > 0 && ldc >= N);
  if (prec != COPER_PREC_BF16 && prec != COPER_PREC_TF32X3 && prec != COPER_PREC_FP16X3) return COPER_ERR_UNSUPPORTED;
  if (workspace_bytes < coper_tc_gemm_workspace_bytes(M, N, K, prec)) return COPER_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  char* p = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  // operand A(m,k): !transA -> stored [M,K] (K-major); transA -> stored [K,M] (MN-major)
  int64_t a_rows = transA ? K : M, a_cols = transA ? M : K;
  // operand B(k,n): !transB -> stored [K,N] (MN-major); transB -> stored [N,K] (K-major)
  int64_t b_rows = transB ? N : K, b_cols = transB ? K : N;
  void* Ap = p;
  void* Bp = p + prepared_bytes(a_rows, (int)a_cols, prec);
  int rc;
  if ((rc = tc_prepare(A, a_rows, (int)a_cols, lda, prec, Ap, st))) return rc;
  if ((rc = tc_prepare(B, b_rows, (int)b_cols, ldb, prec, Bp, st))) return rc;
  GemmProblem g{};
  g.M = M; g.N = N; g.K = K; g.groups = 1; g.groups_inner = 0;
  StoreEpi epi = make_store_epi(C, ldc, 0, 0);
  return tc_gemm_store(prec, transA != 0, transB == 0, tc_operand(Ap, a_rows, (int)a_cols, prec),
                       tc_operand(Bp, b_rows, (int)b_cols, prec), g, false, epi, st);
}

}  // extern "C"
