// HBM-bound pieces of the CoPER-ConvE hot path: lookups, batch-norm/relu/dropout, label bit rows,
// deterministic reductions, global-norm clip and AMSGrad.  All kernels are streaming: coalesced,
// 128-bit vectorised where the shape allows, grids sized in multiples of the SM count.
#include "operand.cuh"

namespace coper {
thread_local int g_last_cuda_error = 0;
long long g_launch_count = 0;
// programmatic dependent launch: on unless switched off by coper_set_pdl
static int g_pdl = 1;
bool pdl_enabled() { return g_pdl != 0; }
constexpr int kSMs = 148;

// ------------------------------------------------------------------ gather (models.py:176,178)
__global__ void gather_rows_kernel(const float* __restrict__ table, int64_t row_lo, int64_t row_hi, int width,
                                   const int64_t* __restrict__ idx, int n_idx, float* __restrict__ out) {
  pdl_enter();
  int warps_per_block = blockDim.x >> 5;
  int row = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (row >= n_idx) return;
  int64_t id = idx[row];
  bool owned = id >= row_lo && id < row_hi;
  const float* src = table + (id - row_lo) * (int64_t)width;
  float* dst = out + (int64_t)row * width;
  if ((width & 3) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int i = lane; i < (width >> 2); i += 32) d4[i] = owned ? __ldg(s4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
    for (int i = lane; i < width; i += 32) dst[i] = owned ? __ldg(src + i) : 0.f;
  }
}

// Two lookups of one step in ONE launch (blocks [0, blocksA) serve table A, the rest table B); block 0 also advances
// the optimizer / dropout step state when asked to (nothing in this kernel reads it).
struct GatherDesc {
  const float* table;
  int64_t row_lo, row_hi;
  int width;
  const int64_t* idx;
  int n_idx;
  float* out;
};
__device__ __forceinline__ void step_state_advance(float* st, uint64_t* seed_dev, float lr, float b1, float b2) {
  float b1p = st[1], b2p = st[2];
  st[0] = lr * sqrtf(1.0f - b2p) / (1.0f - b1p);  // amsgrad.py:137
  st[1] = b1p * b1;                                // amsgrad.py:234-239
  st[2] = b2p * b2;
  if (seed_dev) *seed_dev += 1ull;
}
__global__ void gather_rows2_kernel(GatherDesc A, GatherDesc Bd, int blocksA, float* step_state, uint64_t* seed_dev,
                                    float lr, float b1, float b2) {
  pdl_enter();
  if (step_state && blockIdx.x == 0 && threadIdx.x == 0) step_state_advance(step_state, seed_dev, lr, b1, b2);
  const bool second = (int)blockIdx.x >= blocksA;
  const GatherDesc& g = second ? Bd : A;
  const int warps_per_block = blockDim.x >> 5;
  const int row = ((int)blockIdx.x - (second ? blocksA : 0)) * warps_per_block + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= g.n_idx) return;
  const int64_t id = g.idx[row];
  const bool owned = id >= g.row_lo && id < g.row_hi;
  const float* src = g.table + (id - g.row_lo) * (int64_t)g.width;
  float* dst = g.out + (int64_t)row * g.width;
  if ((g.width & 3) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int i = lane; i < (g.width >> 2); i += 32) d4[i] = owned ? __ldg(s4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
    for (int i = lane; i < g.width; i += 32) dst[i] = owned ? __ldg(src + i) : 0.f;
  }
}

// ------------------------------------------------------------------ column statistics
// mode 0: (x, x^2); mode 1: backward (g1, g1*xhat) with g1 = dout * drop_post * relu'(a x + b)
// rows per chunk: enough chunks to fill the machine (R = B*OH*OW = 73,728 -> 288 CTAs, two per SM; R = B = 512 -> 8 per
// column slab) and few enough that the finalising block's pass over the chunk partials stays short
__host__ __device__ __forceinline__ int stat_rows(int64_t R) { return R >= 32768 ? 256 : 64; }
struct StatBwdArgs {
  const float* dout;
  const float* a;
  const float* b;
  const float* mean;
  const float* invstd;
  int relu;
  float keep;
  float inv_keep;
  uint32_t thr;
  const uint64_t* seed_dev;
  uint64_t salt;
};
// Per-channel finalisation of the forward / backward statistics: one warp per channel, lanes stride over the chunk
// partials, fixed-order shuffle combine.  Shared by the stand-alone finalize kernels (partials of ALL ranks after the
// all-gather of a data-parallel step) and by the last block of colstats_kernel<_, true> (single-launch statistics).
template <bool CG>
__device__ __forceinline__ float2 ld_partial(const float* partials, int64_t i) {
  const float2* p = reinterpret_cast<const float2*>(partials) + i;
  return CG ? __ldcg(p) : __ldg(p);          // CG: written by other blocks of the SAME launch -> read through L2
}
struct BnFwdFin {
  const float* gamma;
  const float* beta;
  float* moving_mean;
  float* moving_var;
  float momentum, eps;
  int use_batch, update_moving, bessel;
  float* a;
  float* b;
  float* mean;
  float* invstd;
};
struct BnBwdFin {
  int use_batch;
  float* dgamma;
  float* dbeta;
  float* c1;
  float* c2;
};
// (sum, sum of second component) of NC channels' chunk partials at once: lanes stride over the chunks, every lane adds
// its chunks in increasing order (the loads of 4 strides x NC channels are issued together, the adds stay ordered),
// fixed-order shuffle combine -> the result does not depend on NC.
template <bool CG, int NC>
__device__ __forceinline__ void sum_partials(const float* partials, int nchunk, int C, const int (&ch)[NC], int lane,
                                             double (&s)[NC], double (&ss)[NC]) {
#pragma unroll
  for (int i = 0; i < NC; ++i) s[i] = ss[i] = 0.0;
  int k = lane;
  for (; k + 96 < nchunk; k += 128) {
    float2 v[NC][4];
#pragma unroll
    for (int i = 0; i < NC; ++i)
#pragma unroll
      for (int u = 0; u < 4; ++u)
        v[i][u] = ch[i] < C ? ld_partial<CG>(partials, (int64_t)(k + 32 * u) * C + ch[i]) : make_float2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < NC; ++i)
#pragma unroll
      for (int u = 0; u < 4; ++u) { s[i] += (double)v[i][u].x; ss[i] += (double)v[i][u].y; }
  }
  for (; k < nchunk; k += 32) {
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const float2 v = ch[i] < C ? ld_partial<CG>(partials, (int64_t)k * C + ch[i]) : make_float2(0.f, 0.f);
      s[i] += (double)v.x;
      ss[i] += (double)v.y;
    }
  }
#pragma unroll
  for (int i = 0; i < NC; ++i) { s[i] = warp_sum_d(s[i]); ss[i] = warp_sum_d(ss[i]); }
}
// lane 0 of the warp that summed channel c
__device__ __forceinline__ void bn_fwd_finish(double s, double ss, int64_t R, int c, const BnFwdFin& f) {
  float mu, var;
  if (f.use_batch) {
    double m = s / (double)R;
    double v = ss / (double)R - m * m;
    if (v < 0.0) v = 0.0;
    mu = (float)m;
    var = (float)v;
    if (f.update_moving) {
      double vm = f.bessel ? v * ((double)R / (double)(R > 1 ? R - 1 : 1)) : v;
      f.moving_mean[c] = f.moving_mean[c] * f.momentum + mu * (1.0f - f.momentum);
      f.moving_var[c] = f.moving_var[c] * f.momentum + (float)vm * (1.0f - f.momentum);
    }
  } else {
    mu = f.moving_mean[c];
    var = f.moving_var[c];
  }
  float inv = 1.0f / sqrtf(var + f.eps);
  float ac = f.gamma[c] * inv;
  f.a[c] = ac;
  f.b[c] = f.beta[c] - mu * ac;
  f.mean[c] = mu;
  f.invstd[c] = inv;
}
__device__ __forceinline__ void bn_bwd_finish(double s, double ss, int64_t R, int c, const BnBwdFin& f) {
  f.dbeta[c] = (float)s;
  f.dgamma[c] = (float)ss;
  f.c1[c] = f.use_batch ? (float)(s / (double)R) : 0.f;
  f.c2[c] = f.use_batch ? (float)(ss / (double)R) : 0.f;
}

// FIN: the block that arrives LAST at `sync_word` (zero on entry, left zero) finalises every channel from the chunk
// partials of all blocks - statistics + finalize in one launch, same summation order as the two-launch form.
template <int MODE, bool FIN>
__global__ void colstats_kernel(const float* __restrict__ x, int64_t R, int C, float* __restrict__ partials,
                                StatBwdArgs bw, BnFwdFin ff, BnBwdFin fb, unsigned int* sync_word) {
  pdl_enter();
  // block (32, 8): x = column in slab, y = row lane
  __shared__ float s1[8][33], s2[8][33];
  __shared__ int s_last;
  int c = blockIdx.x * 32 + threadIdx.x;
  const int kStatRows = stat_rows(R);
  int64_t r0 = (int64_t)blockIdx.y * kStatRows;
  int64_t r1 = r0 + kStatRows < R ? r0 + kStatRows : R;
  float v1 = 0.f, v2 = 0.f;
  uint64_t seed = 0;
  if (MODE == 1) seed = (bw.seed_dev ? *bw.seed_dev : 0ull) + bw.salt;
  if (c < C) {
    float ac = 0.f, bc = 0.f, mc = 0.f, ic = 0.f;
    if (MODE == 1) { ac = bw.a[c]; bc = bw.b[c]; mc = bw.mean[c]; ic = bw.invstd[c]; }
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
      int64_t e = r * C + c;
      float xv = x[e];
      if (MODE == 0) {
        v1 += xv;
        v2 += xv * xv;
      } else {
        float g = bw.dout[e] * drop_factor(bw.keep, bw.inv_keep, bw.thr, seed, (uint64_t)e);
        if (bw.relu && !(ac * xv + bc > 0.f)) g = 0.f;
        v1 += g;
        v2 += g * ((xv - mc) * ic);
      }
    }
  }
  s1[threadIdx.y][threadIdx.x] = v1;
  s2[threadIdx.y][threadIdx.x] = v2;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float t1 = 0.f, t2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { t1 += s1[i][threadIdx.x]; t2 += s2[i][threadIdx.x]; }
    int64_t o = ((int64_t)blockIdx.y * C + c) * 2;
    partials[o] = t1;
    partials[o + 1] = t2;
  }
  if (FIN) {
    __threadfence();                       // this thread's partials are visible device-wide before the arrival below
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0)
      s_last = atomicAdd(sync_word, 1u) == gridDim.x * gridDim.y - 1u;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // All 256 threads finalise: thread = (channel in round, chunk lane).  Few channels -> up to 8 chunk lanes per
    // channel (each adds its chunks k = lane, lane + lanes, ... in increasing order, the lane sums are added in lane
    // order); every channel of a round is finished by its own thread, so the dependent loads of the finish step
    // (gamma, beta, moving statistics) are paid once per round, not once per channel.
    __shared__ double red[2][256];
    const int nchunk = (int)gridDim.y;
    const int tid = (int)(threadIdx.y * 32 + threadIdx.x);
    const int lanes = C <= 32 ? 8 : C <= 64 ? 4 : C <= 128 ? 2 : 1;
    const int cpr = 256 / lanes;            // channels per round
    const int cl = tid % cpr, kl = tid / cpr;
    for (int c0 = 0; c0 < C; c0 += cpr) {
      const int ch = c0 + cl;
      double sm = 0.0, sq = 0.0;
      if (ch < C) {
        int k = kl;
        for (; k + 7 * lanes < nchunk; k += 8 * lanes) {
          float2 v[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) v[u] = ld_partial<true>(partials, (int64_t)(k + u * lanes) * C + ch);
#pragma unroll
          for (int u = 0; u < 8; ++u) { sm += (double)v[u].x; sq += (double)v[u].y; }
        }
        for (; k < nchunk; k += lanes) {
          const float2 v = ld_partial<true>(partials, (int64_t)k * C + ch);
          sm += (double)v.x;
          sq += (double)v.y;
        }
      }
      if (lanes > 1) {
        red[0][tid] = sm;
        red[1][tid] = sq;
        __syncthreads();
        if (kl == 0) {
          for (int l = 1; l < lanes; ++l) { sm += red[0][l * cpr + cl]; sq += red[1][l * cpr + cl]; }
        }
        __syncthreads();
      }
      if (kl == 0 && ch < C) {
        if (MODE == 0) bn_fwd_finish(sm, sq, R, ch, ff);
        else bn_bwd_finish(sm, sq, R, ch, fb);
      }
    }
    if (tid == 0) *sync_word = 0u;
  }
}

__global__ void bn_finalize_kernel(const float* __restrict__ partials, int nchunk, int64_t R, int C, BnFwdFin f) {
  pdl_enter();
  const int ch[1] = {(int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5)};
  if (ch[0] >= C) return;
  double s[1] = {0.0}, ss[1] = {0.0};
  if (f.use_batch) sum_partials<false, 1>(partials, nchunk, C, ch, threadIdx.x & 31, s, ss);
  if ((threadIdx.x & 31) == 0) bn_fwd_finish(s[0], ss[0], R, ch[0], f);
}

__global__ void bn_act_fwd_kernel(const float* __restrict__ x, int64_t n, int C, const float* __restrict__ a,
                                  const float* __restrict__ b, int relu, float keep, float inv_keep, uint32_t thr,
                                  const uint64_t* seed_dev, uint64_t salt, float* __restrict__ out) {
  pdl_enter();
  uint64_t seed = (seed_dev ? *seed_dev : 0ull) + salt;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
    int c = (int)(e % C);
    float v = a[c] * x[e] + b[c];
    if (relu) v = fmaxf(v, 0.f);
    out[e] = v * drop_factor(keep, inv_keep, thr, seed, (uint64_t)e);
  }
}
// float4 variant (C % 4 == 0, n % 4 == 0)
__global__ void bn_act_fwd_kernel4(const float4* __restrict__ x, int64_t n4, int C, const float* __restrict__ a,
                                   const float* __restrict__ b, int relu, float keep, float inv_keep, uint32_t thr,
                                   const uint64_t* seed_dev, uint64_t salt, float4* __restrict__ out) {
  pdl_enter();
  uint64_t seed = (seed_dev ? *seed_dev : 0ull) + salt;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    int64_t e = i * 4;
    int c = (int)(e % C);
    float4 xv = __ldg(x + i);
    float4 av = *reinterpret_cast<const float4*>(a + c);
    float4 bv = *reinterpret_cast<const float4*>(b + c);
    float4 o;
    o.x = av.x * xv.x + bv.x; o.y = av.y * xv.y + bv.y; o.z = av.z * xv.z + bv.z; o.w = av.w * xv.w + bv.w;
    if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
    if (keep < 1.0f) {
      o.x *= drop_factor(keep, inv_keep, thr, seed, (uint64_t)e);
      o.y *= drop_factor(keep, inv_keep, thr, seed, (uint64_t)e + 1);
      o.z *= drop_factor(keep, inv_keep, thr, seed, (uint64_t)e + 2);
      o.w *= drop_factor(keep, inv_keep, thr, seed, (uint64_t)e + 3);
    }
    out[i] = o;
  }
}

// Inference form (moving statistics, no dropout): coper_bn_finalize(use_batch_stats = 0) + coper_bn_act_fwd in one
// launch - every thread derives the affine pair of its channel with the finalize kernel's expressions (same bits).
__global__ void bn_act_fwd_moving_kernel(const float* __restrict__ x, int64_t n, int C, const float* __restrict__ gamma,
                                         const float* __restrict__ beta, const float* __restrict__ moving_mean,
                                         const float* __restrict__ moving_var, float eps, int relu,
                                         float* __restrict__ out) {
  pdl_enter();
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
    int c = (int)(e % C);
    float inv = 1.0f / sqrtf(__ldg(moving_var + c) + eps);
    float ac = __ldg(gamma + c) * inv;
    float bc = __ldg(beta + c) - __ldg(moving_mean + c) * ac;
    float v = ac * x[e] + bc;
    if (relu) v = fmaxf(v, 0.f);
    out[e] = v;
  }
}

// float4 variant (C % 4 == 0, n % 4 == 0, 16-byte aligned pointers)
__global__ void bn_act_fwd_moving_kernel4(const float4* __restrict__ x, int64_t n4, int C,
                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                          const float* __restrict__ moving_mean, const float* __restrict__ moving_var,
                                          float eps, int relu, float4* __restrict__ out) {
  pdl_enter();
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const int c = (int)((i * 4) % C);
    const float4 xv = __ldg(x + i);
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c)), be = __ldg(reinterpret_cast<const float4*>(beta + c));
    const float4 mu = __ldg(reinterpret_cast<const float4*>(moving_mean + c));
    const float4 va = __ldg(reinterpret_cast<const float4*>(moving_var + c));
    const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {g.x, g.y, g.z, g.w}, bs[4] = {be.x, be.y, be.z, be.w};
    const float ms[4] = {mu.x, mu.y, mu.z, mu.w}, vs[4] = {va.x, va.y, va.z, va.w};
    float o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float inv = 1.0f / sqrtf(vs[k] + eps);
      float ac = gs[k] * inv;
      float bc = bs[k] - ms[k] * ac;
      o[k] = ac * xs[k] + bc;
      if (relu) o[k] = fmaxf(o[k], 0.f);
    }
    out[i] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

__global__ void bn_bwd_finalize_kernel(const float* __restrict__ partials, int nchunk, int64_t R, int C, BnBwdFin f) {
  pdl_enter();
  const int ch[1] = {(int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5)};
  if (ch[0] >= C) return;
  double s[1], ss[1];
  sum_partials<false, 1>(partials, nchunk, C, ch, threadIdx.x & 31, s, ss);
  if ((threadIdx.x & 31) == 0) bn_bwd_finish(s[0], ss[0], R, ch[0], f);
}

__global__ void bn_act_bwd_apply_kernel(const float* __restrict__ dout, const float* __restrict__ x, int64_t n,
                                        int C, const float* __restrict__ a, const float* __restrict__ b,
                                        const float* __restrict__ mean, const float* __restrict__ invstd,
                                        const float* __restrict__ c1, const float* __restrict__ c2, int relu,
                                        float keep_post, float inv_keep_post, uint32_t thr_post,
                                        const uint64_t* seed_dev, uint64_t salt_post, float keep_pre,
                                        float inv_keep_pre, uint32_t thr_pre, uint64_t salt_pre,
                                        float* __restrict__ dx) {
  pdl_enter();
  uint64_t sd = seed_dev ? *seed_dev : 0ull;
  uint64_t seed_post = sd + salt_post, seed_pre = sd + salt_pre;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
    int c = (int)(e % C);
    float d = bn_bwd_dx(dout[e], drop_factor(keep_post, inv_keep_post, thr_post, seed_post, (uint64_t)e), x[e], a[c], b[c],
                        mean[c], invstd[c], c1[c], c2[c], relu);
    dx[e] = d * drop_factor(keep_pre, inv_keep_pre, thr_pre, seed_pre, (uint64_t)e);
  }
}

__global__ void dropout_mask_kernel(int64_t n, uint32_t thr, float keep, const uint64_t* seed_dev, uint64_t salt,
                                    float* mask) {
  pdl_enter();
  uint64_t seed = (seed_dev ? *seed_dev : 0ull) + salt;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride)
    mask[e] = (keep >= 1.0f || hash32(seed, (uint64_t)e) < thr) ? 1.0f : 0.0f;
}
__global__ void dropout_apply_kernel(float* x, int64_t n, float keep, float inv_keep, uint32_t thr,
                                     const uint64_t* seed_dev, uint64_t salt) {
  pdl_enter();
  uint64_t seed = (seed_dev ? *seed_dev : 0ull) + salt;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride)
    x[e] *= drop_factor(keep, inv_keep, thr, seed, (uint64_t)e);
}

// ------------------------------------------------------------------ label / filter bit rows
__global__ void csr_to_bits_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int B,
                                   int64_t lo, int64_t hi, int64_t words, uint32_t* bits) {
  pdl_enter();
  int b = blockIdx.x;
  if (b >= B) return;
  int s = rowptr[b], e = rowptr[b + 1];
  for (int i = s + threadIdx.x; i < e; i += blockDim.x) {
    int64_t n = col[i];
    if (n >= lo && n < hi) {
      int64_t l = n - lo;
      atomicOr(bits + (int64_t)b * words + (l >> 5), 1u << (l & 31));
    }
  }
}
__global__ void dense_to_bits_kernel(const float* __restrict__ dense, int B, int64_t N, int64_t words,
                                     uint32_t* __restrict__ bits) {
  pdl_enter();
  // one warp per output word: lane l tests entity w*32 + l (coalesced 128 B read), ballot packs the word
  int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  int64_t total = (int64_t)B * words;
  if (gw >= total) return;
  int64_t b = gw / words, w = gw % words;
  int64_t n = w * 32 + lane;
  bool on = n < N && dense[b * N + n] == 1.0f;
  uint32_t m = __ballot_sync(0xffffffffu, on);
  if (lane == 0) bits[gw] = m;
}

// entity-major bit matrix bitsT [Ns, wordsB]: bit (b & 31) of word (n, b >> 5) = entity n is a positive of query b
__global__ void csr_to_bits_t_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int B,
                                     int64_t lo, int64_t hi, int wordsB, uint32_t* bitsT) {
  pdl_enter();
  int b = blockIdx.x;
  if (b >= B) return;
  int s = rowptr[b], e = rowptr[b + 1];
  for (int i = s + threadIdx.x; i < e; i += blockDim.x) {
    int64_t n = col[i];
    if (n >= lo && n < hi) atomicOr(bitsT + (n - lo) * wordsB + (b >> 5), 1u << (b & 31));
  }
}
__global__ void bits_t_set_kernel(const int64_t* __restrict__ ent, int B, int64_t lo, int64_t hi, int wordsB,
                                  uint32_t* bitsT) {
  pdl_enter();
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  int64_t n = ent[b];
  if (n >= lo && n < hi) atomicOr(bitsT + (n - lo) * wordsB + (b >> 5), 1u << (b & 31));
}
__global__ void dense_to_bits_t_kernel(const float* __restrict__ dense, int B, int64_t N, int64_t ld, int wordsB,
                                       uint32_t* __restrict__ bitsT) {
  pdl_enter();
  // one warp per output word (n, w): lane l tests query w*32 + l
  int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (gw >= N * wordsB) return;
  int64_t n = gw / wordsB;
  int w = (int)(gw - n * wordsB);
  int b = w * 32 + lane;
  bool on = b < B && dense[(int64_t)b * ld + n] == 1.0f;
  uint32_t m = __ballot_sync(0xffffffffu, on);
  if (lane == 0) bitsT[gw] = m;
}

// ------------------------------------------------------------------ deterministic reductions
// Few slabs (S <= 8), many outputs (dbias of a sharded table, 4 slabs x 10 M floats): one thread per 4 outputs, float4
// loads, slabs added in slab order in fp64 - the same order (and bits) as the general kernel below gives for S <= 8.
__global__ void __launch_bounds__(256) reduce_partials_few_kernel(const float* __restrict__ in, int S, int64_t n,
                                                                  float scale, int accumulate, float* __restrict__ out) {
  pdl_enter();
  const int64_t i4 = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 4;
  if (i4 >= n) return;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  for (int s = 0; s < S; ++s) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(in + (int64_t)s * n + i4));
    a0 += (double)v.x; a1 += (double)v.y; a2 += (double)v.z; a3 += (double)v.w;
  }
  float4 r = make_float4((float)(a0 * (double)scale), (float)(a1 * (double)scale), (float)(a2 * (double)scale),
                         (float)(a3 * (double)scale));
  float4* o = reinterpret_cast<float4*>(out + i4);
  if (accumulate) {
    const float4 p = *o;
    r.x += p.x; r.y += p.y; r.z += p.z; r.w += p.w;
  }
  *o = r;
}
// out[i] = scale * sum_s in[s, i]: block = 32 outputs x 8 slab lanes; every thread sums the slabs s = ty, ty+8, ...
// in fp64, the 8 lane sums are added in a fixed order -> deterministic, and the slab loop is 8x shorter / pipelined
struct ReduceJob {
  const float* in;
  int S;
  int64_t n;
  float scale;
  int accumulate;
  float* out;
};
__device__ __forceinline__ void reduce_job_block(const ReduceJob& j, int block, double (&red)[8][33]) {
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  int64_t i = (int64_t)block * 32 + tx;
  double acc = 0.0;
  if (i < j.n) {
    int s = ty;
    for (; s + 24 < j.S; s += 32) {
      float a0 = __ldg(j.in + (int64_t)s * j.n + i), a1 = __ldg(j.in + (int64_t)(s + 8) * j.n + i);
      float a2 = __ldg(j.in + (int64_t)(s + 16) * j.n + i), a3 = __ldg(j.in + (int64_t)(s + 24) * j.n + i);
      acc += (double)a0; acc += (double)a1; acc += (double)a2; acc += (double)a3;
    }
    for (; s < j.S; s += 8) acc += (double)__ldg(j.in + (int64_t)s * j.n + i);
  }
  red[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && i < j.n) {
    double t = red[0][tx];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += red[k][tx];
    float r = (float)(t * (double)j.scale);
    j.out[i] = j.accumulate ? j.out[i] + r : r;
  }
}
// float4 form of the same reduction (n % 4 == 0, 16-byte aligned): block = 32 x 4 outputs, 8 slab lanes; same slab
// order per output as reduce_job_block -> same bits, a quarter of the load instructions
__device__ __forceinline__ void reduce_job_block4(const ReduceJob& j, int block, double (&red)[8][33], double* red4) {
  (void)red;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t i = ((int64_t)block * 32 + tx) * 4;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  if (i < j.n) {
    int s = ty;
    for (; s + 24 < j.S; s += 32) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldg(reinterpret_cast<const float4*>(j.in + (int64_t)(s + 8 * u) * j.n + i));
#pragma unroll
      for (int u = 0; u < 4; ++u) { a0 += (double)v[u].x; a1 += (double)v[u].y; a2 += (double)v[u].z; a3 += (double)v[u].w; }
    }
    for (; s < j.S; s += 8) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(j.in + (int64_t)s * j.n + i));
      a0 += (double)v.x; a1 += (double)v.y; a2 += (double)v.z; a3 += (double)v.w;
    }
  }
  double* mine = red4 + ((size_t)ty * 32 + tx) * 4;
  mine[0] = a0; mine[1] = a1; mine[2] = a2; mine[3] = a3;
  __syncthreads();
  if (ty == 0 && i < j.n) {
    double t[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) t[c] = red4[(size_t)tx * 4 + c];
#pragma unroll
    for (int k = 1; k < 8; ++k)
#pragma unroll
      for (int c = 0; c < 4; ++c) t[c] += red4[((size_t)k * 32 + tx) * 4 + c];
    float4 r = make_float4((float)(t[0] * (double)j.scale), (float)(t[1] * (double)j.scale),
                           (float)(t[2] * (double)j.scale), (float)(t[3] * (double)j.scale));
    float4* o = reinterpret_cast<float4*>(j.out + i);
    if (j.accumulate) {
      const float4 p = *o;
      r.x = p.x + r.x; r.y = p.y + r.y; r.z = p.z + r.z; r.w = p.w + r.w;
    }
    *o = r;
  }
}
// blocks [0, blocks_a) reduce job A, [blocks_a, blocks_a + blocks_b) job B; one more block (if dsum_in) adds dsum_n
// doubles in the order of sum_doubles_kernel (umma_entity.cu) - three tiny dependent-free reductions, one launch
template <bool VEC_A>
__global__ void __launch_bounds__(256) reduce_partials_kernel(ReduceJob A, int blocks_a, ReduceJob Bj, int blocks_b,
                                                              const double* __restrict__ dsum_in, int dsum_n,
                                                              double* __restrict__ dsum_out) {
  pdl_enter();
  __shared__ double red[8][33];
  __shared__ double red4[VEC_A ? 8 * 32 * 4 : 1];
  const int blk = (int)blockIdx.x;
  if (blk < blocks_a) {
    if (VEC_A) reduce_job_block4(A, blk, red, red4);
    else reduce_job_block(A, blk, red);
  } else if (blk < blocks_a + blocks_b) {
    reduce_job_block(Bj, blk - blocks_a, red);
  } else {
    double acc = 0.0;
    for (int i = threadIdx.x; i < dsum_n; i += blockDim.x) acc += dsum_in[i];
    const double t = block_sum<double>(acc, &red[0][0]);
    if (threadIdx.x == 0) *dsum_out = t;
  }
}

__global__ void sumsq_kernel(const float* __restrict__ x, int64_t n, double* __restrict__ out) {
  pdl_enter();
  __shared__ double sm[32];
  double acc = 0.0;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if ((reinterpret_cast<uintptr_t>(x) & 15) == 0) {
    int64_t n4 = n >> 2;
    const float4* x4 = reinterpret_cast<const float4*>(x);
    float p = 0.f;
    int cnt = 0;
    for (int64_t j = i; j < n4; j += stride) {
      float4 v = __ldg(x4 + j);
      p += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
      if (++cnt == 64) { acc += (double)p; p = 0.f; cnt = 0; }
    }
    acc += (double)p;
    for (int64_t j = (n4 << 2) + i; j < n; j += stride) acc += (double)x[j] * (double)x[j];
  } else {
    for (int64_t j = i; j < n; j += stride) acc += (double)x[j] * (double)x[j];
  }
  double t = block_sum<double>(acc, sm);
  if (threadIdx.x == 0) out[blockIdx.x] = t;
}

__global__ void clip_scale_kernel(const double* __restrict__ partials, int n, float clip, float* out2) {
  pdl_enter();
  __shared__ double sm[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += partials[i];
  double t = block_sum<double>(acc, sm);
  if (threadIdx.x == 0) {
    double norm = sqrt(t);
    double c = (double)clip;
    out2[0] = (float)(c / (norm > c ? norm : c));
    out2[1] = (float)norm;
  }
}

// ------------------------------------------------------------------ AMSGrad (utils/amsgrad.py:130-159)
__global__ void amsgrad_kernel(float* __restrict__ theta, const float* __restrict__ grad, float* __restrict__ m,
                               float* __restrict__ v, float* __restrict__ vhat, int64_t n,
                               const float* __restrict__ step_state, float b1, float b2, float eps,
                               const float* __restrict__ clip_scale, int bug_compat) {
  pdl_enter();
  float lr_t = step_state[0];
  float cs = clip_scale ? *clip_scale : 1.0f;
  float omb1 = 1.0f - b1, omb2 = 1.0f - b2;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float g = grad[i] * cs;
    float mt, vt;
    if (bug_compat) {
      mt = g * omb1;          // slot m == 0 forever (amsgrad.py:142-144)
      vt = (g * g) * omb2;    // slot v == 0 forever (amsgrad.py:149-151)
    } else {
      mt = m[i] * b1 + g * omb1;
      vt = v[i] * b2 + (g * g) * omb2;
      m[i] = mt;
      v[i] = vt;
    }
    float vh = fmaxf(vhat[i], vt);
    vhat[i] = vh;
    theta[i] -= lr_t * mt / (sqrtf(vh) + eps);
  }
}

__global__ void step_state_advance_kernel(float* st, uint64_t* seed_dev, float lr, float b1, float b2) {
  pdl_enter();
  if (threadIdx.x == 0 && blockIdx.x == 0) step_state_advance(st, seed_dev, lr, b1, b2);
}


// ------------------------------------------------------------------ multi-tensor clip + AMSGrad (one launch each)
// work list: chunk c = (tensor id, first element); every chunk covers <= COPER_MT_CHUNK elements of one tensor
__global__ void __launch_bounds__(256) mt_sumsq_kernel(const coper_param_desc* __restrict__ descs,
                                                       const int32_t* __restrict__ chunks,
                                                       double* __restrict__ chunk_partials) {
  pdl_enter();
  __shared__ double sm[32];
  const int t = chunks[2 * blockIdx.x];
  const int64_t start = (int64_t)chunks[2 * blockIdx.x + 1] * COPER_MT_CHUNK;
  const coper_param_desc d = descs[t];
  // the squared norm of this gradient is supplied by its producer (coper_sumsq_combine): nothing to read, and its
  // chunk partials are never summed (mt_tensor_sums_kernel)
  if (d.mode & COPER_GRAD_NORM_EXTERNAL) return;
  const int64_t end = start + COPER_MT_CHUNK < d.n ? start + COPER_MT_CHUNK : d.n;
  const float* x = d.grad;
  float p = 0.f;
  if (d.mode == COPER_GRAD_INDEXED_SLICES) {
    // IndexedSlices: norm over the slice values = sum of the per-row sums of squared slices
    for (int64_t j = start + threadIdx.x; j < end; j += 256) p += d.grad_sq[j];
  } else if (((reinterpret_cast<uintptr_t>(x) & 15) == 0) && end - start == COPER_MT_CHUNK) {
    const float4* x4 = reinterpret_cast<const float4*>(x + start);
#pragma unroll 4
    for (int j = threadIdx.x; j < COPER_MT_CHUNK / 4; j += 256) {
      float4 v = __ldg(x4 + j);
      p += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
  } else {
    for (int64_t j = start + threadIdx.x; j < end; j += 256) { float v = x[j]; p += v * v; }
  }
  double tsum = block_sum<double>((double)p, sm);
  if (threadIdx.x == 0) chunk_partials[blockIdx.x] = tsum;
}
// tensor_sumsq[t] = sum of the chunk partials of tensor t (fixed order); chunk_offsets [n_tensors + 1]
__global__ void mt_tensor_sums_kernel(const coper_param_desc* __restrict__ descs, const double* __restrict__ chunk_partials,
                                      const int32_t* __restrict__ chunk_offsets, int n_tensors,
                                      double* __restrict__ tensor_sumsq) {
  pdl_enter();
  // one warp per tensor: lanes stride over the tensor's chunks, fixed-order shuffle combine.  A tensor whose norm is
  // supplied by its producer (COPER_GRAD_NORM_EXTERNAL) has no partials to add (160 k of them at 10 M entities).
  int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (t >= n_tensors) return;
  double acc = 0.0;
  if (!(descs[t].mode & COPER_GRAD_NORM_EXTERNAL))
    for (int c = chunk_offsets[t] + lane; c < chunk_offsets[t + 1]; c += 32) acc += chunk_partials[c];
  acc = warp_sum_d(acc);
  if (lane == 0) {
    tensor_sumsq[t] = acc;
    // fp16x3 operand copies re-emitted by the update kernel that follows: roll the exponent to the magnitude the
    // variable has NOW (running max of the previous emission / of the full preparation) and restart the running max
    const coper_param_desc d = descs[t];
    if (d.prepared && d.prepared_prec == COPER_PREC_FP16X3) fp16x3_roll(fp16x3_trailer(d.prepared, d.n));
  }
}
// mt_tensor_sums_kernel + sumsq_combine_kernel + clip_scale_kernel in ONE block (same summation orders): per-tensor sums
// of the chunk partials, the producer-supplied squared norm of tensor `ext_tensor` (parts + deltas, < 0: none), and -
// with clip_out != NULL - the clip factor over all tensors.
__global__ void __launch_bounds__(256) mt_sumsq_finish_kernel(const coper_param_desc* __restrict__ descs,
                                                              const double* __restrict__ chunk_partials,
                                                              const int32_t* __restrict__ chunk_offsets, int n_tensors,
                                                              double* tensor_sumsq, int ext_tensor,
                                                              const double* __restrict__ ext_parts, int n_ext_parts,
                                                              const double* __restrict__ ext_deltas, int n_ext_deltas,
                                                              float clip, float* clip_out) {
  pdl_enter();
  __shared__ double smd[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = warp; t < n_tensors; t += 8) {
    const coper_param_desc d = descs[t];
    double acc = 0.0;
    if (!(d.mode & COPER_GRAD_NORM_EXTERNAL))
      for (int c = chunk_offsets[t] + lane; c < chunk_offsets[t + 1]; c += 32) acc += chunk_partials[c];
    acc = warp_sum_d(acc);
    if (lane == 0) {
      if (t != ext_tensor) tensor_sumsq[t] = acc;
      if (d.prepared && d.prepared_prec == COPER_PREC_FP16X3)       // see mt_tensor_sums_kernel
        fp16x3_roll(fp16x3_trailer(d.prepared, d.n));
    }
  }
  if (ext_tensor >= 0) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < n_ext_parts; i += blockDim.x) acc += ext_parts[i];
    for (int i = threadIdx.x; i < n_ext_deltas; i += blockDim.x) acc += ext_deltas[i];
    const double t = block_sum<double>(acc, smd);
    if (threadIdx.x == 0) tensor_sumsq[ext_tensor] = t > 0.0 ? t : 0.0;
  }
  if (!clip_out) return;
  __syncthreads();
  double acc = 0.0;
  for (int i = threadIdx.x; i < n_tensors; i += blockDim.x) acc += tensor_sumsq[i];
  const double t = block_sum<double>(acc, smd);
  if (threadIdx.x == 0) {
    double norm = sqrt(t);
    double c = (double)clip;
    clip_out[0] = (float)(c / (norm > c ? norm : c));
    clip_out[1] = (float)norm;
  }
}
__device__ __forceinline__ void amsgrad_elem(float g, float& th, float* m, float* v, float& vh, int64_t i, float lr_t,
                                             float b1, float b2, float omb1, float omb2, float eps, int bug_compat) {
  float mt, vt;
  if (bug_compat) {
    mt = g * omb1;
    vt = (g * g) * omb2;
  } else {
    mt = m[i] * b1 + g * omb1;
    vt = v[i] * b2 + (g * g) * omb2;
    m[i] = mt;
    v[i] = vt;
  }
  vh = fmaxf(vh, vt);
  th -= lr_t * mt / (sqrtf(vh) + eps);
}
__global__ void __launch_bounds__(256) mt_amsgrad_kernel(const coper_param_desc* __restrict__ descs,
                                                         const int32_t* __restrict__ chunks,
                                                         const float* __restrict__ step_state, float b1, float b2,
                                                         float eps, const float* __restrict__ clip_scale,
                                                         int bug_compat) {
  pdl_enter();
  const int t = chunks[2 * blockIdx.x];
  const int64_t start = (int64_t)chunks[2 * blockIdx.x + 1] * COPER_MT_CHUNK;
  const coper_param_desc d = descs[t];
  const int64_t end = start + COPER_MT_CHUNK < d.n ? start + COPER_MT_CHUNK : d.n;
  const float lr_t = step_state[0];
  const float cs = clip_scale ? *clip_scale : 1.0f;
  const float omb1 = 1.0f - b1, omb2 = 1.0f - b2;
  // fp16x3 operand copy: the exponent was rolled by mt_tensor_sums_kernel; max |theta_new| goes to the running max
  const bool f16x3 = d.prepared && d.prepared_prec == COPER_PREC_FP16X3;
  // the optimizer's operand copies have pitch == row length: planes of n elements
  uint32_t* trailer = f16x3 ? fp16x3_trailer(d.prepared, d.n) : nullptr;
  const float sc = f16x3 ? exp2f((float)reinterpret_cast<const int*>(trailer)[kTrExp]) : 1.0f;
  float amax = 0.f;
  if ((d.mode & 1) == COPER_GRAD_INDEXED_SLICES) {           // utils/amsgrad.py:161-189 (slots accumulate)
    for (int64_t i = start + threadIdx.x; i < end; i += 256) {
      const float g1 = d.grad[i] * cs, g2 = d.grad_sq[i] * cs * cs;
      const float mt = d.m[i] * b1 + g1 * omb1;
      const float vt = d.v[i] * b2 + g2 * omb2;
      d.m[i] = mt;
      d.v[i] = vt;
      const float vh = fmaxf(d.vhat[i], vt);
      d.vhat[i] = vh;
      const float th = d.theta[i] - lr_t * mt / (sqrtf(vh) + eps);
      d.theta[i] = th;
      if (d.prepared) emit_prepared(d.prepared_prec, d.prepared, d.n, i, th, sc);
      amax = fmaxf(amax, fabsf(th));
    }
    if (f16x3) warp_trailer_max(trailer + kTrRunMax, amax);
    return;
  }
  const bool vec = end - start == COPER_MT_CHUNK && bug_compat &&
                   (((reinterpret_cast<uintptr_t>(d.theta) | reinterpret_cast<uintptr_t>(d.grad) |
                      reinterpret_cast<uintptr_t>(d.vhat)) & 15) == 0);
  if (vec) {
    float4* th4 = reinterpret_cast<float4*>(d.theta + start);
    const float4* g4 = reinterpret_cast<const float4*>(d.grad + start);
    float4* vh4 = reinterpret_cast<float4*>(d.vhat + start);
#pragma unroll 4
    for (int j = threadIdx.x; j < COPER_MT_CHUNK / 4; j += 256) {
      float4 g = g4[j], th = th4[j], vh = vh4[j];
      amsgrad_elem(g.x * cs, th.x, nullptr, nullptr, vh.x, 0, lr_t, b1, b2, omb1, omb2, eps, 1);
      amsgrad_elem(g.y * cs, th.y, nullptr, nullptr, vh.y, 0, lr_t, b1, b2, omb1, omb2, eps, 1);
      amsgrad_elem(g.z * cs, th.z, nullptr, nullptr, vh.z, 0, lr_t, b1, b2, omb1, omb2, eps, 1);
      amsgrad_elem(g.w * cs, th.w, nullptr, nullptr, vh.w, 0, lr_t, b1, b2, omb1, omb2, eps, 1);
      th4[j] = th;
      vh4[j] = vh;
      if (d.prepared) {
        emit_prepared4(d.prepared_prec, d.prepared, d.n, start + 4 * (int64_t)j, th, sc);
        if (f16x3) amax = fmaxf(fmaxf(amax, fmaxf(fabsf(th.x), fabsf(th.y))), fmaxf(fabsf(th.z), fabsf(th.w)));
      }
    }
  } else {
    for (int64_t i = start + threadIdx.x; i < end; i += 256) {
      float th = d.theta[i], vh = d.vhat[i];
      amsgrad_elem(d.grad[i] * cs, th, d.m, d.v, vh, i, lr_t, b1, b2, omb1, omb2, eps, bug_compat);
      d.theta[i] = th;
      d.vhat[i] = vh;
      if (d.prepared) emit_prepared(d.prepared_prec, d.prepared, d.n, i, th, sc);
      amax = fmaxf(amax, fabsf(th));
    }
  }
  if (f16x3) warp_trailer_max(trailer + kTrRunMax, amax);
}

// out[0] = sum(parts[0..n_parts)) + sum(deltas[0..n_deltas)) in a fixed order (one block)
__global__ void sumsq_combine_kernel(const double* __restrict__ parts, int n_parts, const double* __restrict__ deltas,
                                     int n_deltas, double* __restrict__ out) {
  pdl_enter();
  __shared__ double smd[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n_parts; i += blockDim.x) acc += parts[i];
  for (int i = threadIdx.x; i < n_deltas; i += blockDim.x) acc += deltas[i];
  const double t = block_sum<double>(acc, smd);
  if (threadIdx.x == 0) *out = t > 0.0 ? t : 0.0;
}

// out = scale * sum of S slabs (+ out), and - in the same launch - *dsum_out = sum of dsum_n doubles (dsum_in may be
// NULL).  Used by the scorer: the split-K slabs of dq and the loss partials of the BCE epilogue.
int reduce_partials_and_sum(const float* in, int S, int64_t n, float scale, int accumulate, float* out,
                            const double* dsum_in, int dsum_n, double* dsum_out, cudaStream_t st) {
  ReduceJob A{in, S, n, scale, accumulate, out};
  const bool vec = n >= 4096 && (n & 3) == 0 &&
                   ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  if (vec) {
    const int ba = (int)((n / 4 + 31) / 32);
    launch_pdl(reduce_partials_kernel<true>, ba + (dsum_in ? 1 : 0), 256, 0, st, A, ba, ReduceJob{}, 0, dsum_in,
               dsum_n, dsum_out);
  } else {
    const int ba = (int)((n + 31) / 32);
    launch_pdl(reduce_partials_kernel<false>, ba + (dsum_in ? 1 : 0), 256, 0, st, A, ba, ReduceJob{}, 0, dsum_in,
               dsum_n, dsum_out);
  }
  return check_launch();
}

static inline int grid_for(int64_t n, int threads, int per_sm = 8) {
  int64_t g = (n + threads - 1) / threads;
  int64_t cap = (int64_t)kSMs * per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}
}  // namespace coper

using namespace coper;

extern "C" {

int coper_version(void) { return 100; }
const char* coper_status_string(int s) {
  switch (s) {
    case COPER_OK: return "ok";
    case COPER_ERR_INVALID_ARG: return "invalid argument";
    case COPER_ERR_CUDA: return "CUDA error";
    case COPER_ERR_UNSUPPORTED: return "unsupported configuration";
    case COPER_ERR_WORKSPACE: return "workspace too small";
    default: return "unknown status";
  }
}
int coper_last_cuda_error(void) { return g_last_cuda_error; }
long long coper_launch_count(void) { return g_launch_count; }
int coper_set_pdl(int on) {
  g_pdl = on ? 1 : 0;
  return COPER_OK;
}
int coper_device_is_sm100(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return COPER_ERR_CUDA;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return COPER_ERR_CUDA;
  return major == 10 ? 1 : 0;
}

int coper_gather_rows(const float* table, int64_t row_lo, int64_t row_hi, int width, const int64_t* idx, int n_idx,
                      float* out, coper_stream_t stream) {
  COPER_CHECK_ARG(table && idx && out && width > 0 && n_idx >= 0 && row_hi >= row_lo);
  if (n_idx == 0) return COPER_OK;
  launch_pdl(gather_rows_kernel, ceil_div(n_idx, 8), 256, 0, as_stream(stream), table, row_lo, row_hi, width, idx,
             n_idx, out);
  return check_launch();
}

int coper_gather_rows2(const float* table_a, int64_t lo_a, int64_t hi_a, int width_a, const int64_t* idx_a, int n_a,
                       float* out_a, const float* table_b, int64_t lo_b, int64_t hi_b, int width_b,
                       const int64_t* idx_b, int n_b, float* out_b, float* step_state, uint64_t* seed_dev, float lr,
                       float beta1, float beta2, coper_stream_t stream) {
  COPER_CHECK_ARG(table_a && idx_a && out_a && width_a > 0 && n_a >= 0 && hi_a >= lo_a);
  COPER_CHECK_ARG(n_b == 0 || (table_b && idx_b && out_b && width_b > 0 && n_b > 0 && hi_b >= lo_b));
  const int blocks_a = ceil_div(n_a, 8), blocks_b = ceil_div(n_b, 8);
  if (blocks_a + blocks_b == 0 && !step_state) return COPER_OK;
  GatherDesc A{table_a, lo_a, hi_a, width_a, idx_a, n_a, out_a}, Bd{table_b, lo_b, hi_b, width_b, idx_b, n_b, out_b};
  const int grid = blocks_a + blocks_b > 0 ? blocks_a + blocks_b : 1;
  launch_pdl(gather_rows2_kernel, grid, 256, 0, as_stream(stream), A, Bd, blocks_a, step_state, seed_dev, lr, beta1,
             beta2);
  return check_launch();
}

int coper_colstats_chunks(int64_t R) { return R <= 0 ? 0 : (int)((R + stat_rows(R) - 1) / stat_rows(R)); }

int coper_colstats(const float* x, int64_t R, int C, float* partials, coper_stream_t stream) {
  COPER_CHECK_ARG(x && partials && R > 0 && C > 0);
  dim3 grid(ceil_div(C, 32), coper_colstats_chunks(R)), block(32, 8);
  launch_pdl(colstats_kernel<0, false>, grid, block, 0, as_stream(stream), x, R, C, partials, StatBwdArgs{},
             BnFwdFin{}, BnBwdFin{}, nullptr);
  return check_launch();
}

int coper_bn_finalize(const float* partials, int nchunk, int64_t R, int C, const float* gamma, const float* beta,
                      float* moving_mean, float* moving_var, float momentum, float eps, int use_batch_stats,
                      int update_moving, int bessel, float* a, float* b, float* mean, float* invstd,
                      coper_stream_t stream) {
  COPER_CHECK_ARG(gamma && beta && moving_mean && moving_var && a && b && mean && invstd && C > 0);
  COPER_CHECK_ARG(!use_batch_stats || (partials && nchunk > 0 && R > 0));
  BnFwdFin f{gamma, beta, moving_mean, moving_var, momentum, eps, use_batch_stats, update_moving, bessel, a, b, mean, invstd};
  launch_pdl(bn_finalize_kernel, ceil_div((int64_t)C * 32, 256), 256, 0, as_stream(stream), partials, nchunk, R, C,
             f);
  return check_launch();
}

int coper_bn_stats_finalize(const float* x, int64_t R, int C, float* partials, unsigned int* sync_word,
                            const float* gamma, const float* beta, float* moving_mean, float* moving_var,
                            float momentum, float eps, int update_moving, int bessel, float* a, float* b, float* mean,
                            float* invstd, coper_stream_t stream) {
  COPER_CHECK_ARG(x && partials && sync_word && R > 0 && C > 0);
  COPER_CHECK_ARG(gamma && beta && moving_mean && moving_var && a && b && mean && invstd);
  dim3 grid(ceil_div(C, 32), coper_colstats_chunks(R)), block(32, 8);
  BnFwdFin f{gamma, beta, moving_mean, moving_var, momentum, eps, 1, update_moving, bessel, a, b, mean, invstd};
  launch_pdl(colstats_kernel<0, true>, grid, block, 0, as_stream(stream), x, R, C, partials, StatBwdArgs{}, f,
             BnBwdFin{}, sync_word);
  return check_launch();
}

int coper_bn_act_fwd(const float* x, int64_t R, int C, const float* a, const float* b, int relu, float keep_post,
                     const uint64_t* seed_dev, uint64_t salt_post, float* out, coper_stream_t stream) {
  COPER_CHECK_ARG(x && a && b && out && R > 0 && C > 0 && keep_post > 0.f);
  int64_t n = R * C;
  float inv = 1.0f / keep_post;
  uint32_t thr = keep_threshold(keep_post);
  bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) |
                               reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0;
  if (vec) {
    int64_t n4 = n / 4;
    launch_pdl(bn_act_fwd_kernel4, grid_for(n4, 256), 256, 0, as_stream(stream), reinterpret_cast<const float4*>(x),
               n4, C, a, b, relu, keep_post, inv, thr, seed_dev, salt_post, reinterpret_cast<float4*>(out));
  } else {
    launch_pdl(bn_act_fwd_kernel, grid_for(n, 256), 256, 0, as_stream(stream), x, n, C, a, b, relu, keep_post, inv,
               thr, seed_dev, salt_post, out);
  }
  return check_launch();
}

int coper_bn_act_fwd_moving(const float* x, int64_t R, int C, const float* gamma, const float* beta,
                            const float* moving_mean, const float* moving_var, float eps, int relu, float* out,
                            coper_stream_t stream) {
  COPER_CHECK_ARG(x && gamma && beta && moving_mean && moving_var && out && R > 0 && C > 0);
  int64_t n = R * C;
  const bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) |
                                     reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta) |
                                     reinterpret_cast<uintptr_t>(moving_mean) | reinterpret_cast<uintptr_t>(moving_var)) & 15) == 0;
  if (vec)
    launch_pdl(bn_act_fwd_moving_kernel4, grid_for(n / 4, 256), 256, 0, as_stream(stream), reinterpret_cast<const
               float4*>(x), n / 4, C, gamma, beta, moving_mean, moving_var, eps, relu,
               reinterpret_cast<float4*>(out));
  else
    launch_pdl(bn_act_fwd_moving_kernel, grid_for(n, 256), 256, 0, as_stream(stream), x, n, C, gamma, beta,
               moving_mean, moving_var, eps, relu, out);
  return check_launch();
}

int coper_bn_act_bwd_stats(const float* dout, const float* x, int64_t R, int C, const float* a, const float* b,
                           const float* mean, const float* invstd, int relu, float keep_post,
                           const uint64_t* seed_dev, uint64_t salt_post, float* partials, coper_stream_t stream) {
  COPER_CHECK_ARG(dout && x && a && b && mean && invstd && partials && R > 0 && C > 0 && keep_post > 0.f);
  dim3 grid(ceil_div(C, 32), coper_colstats_chunks(R)), block(32, 8);
  StatBwdArgs bw{dout, a, b, mean, invstd, relu, keep_post, 1.0f / keep_post, keep_threshold(keep_post), seed_dev,
                 salt_post};
  launch_pdl(colstats_kernel<1, false>, grid, block, 0, as_stream(stream), x, R, C, partials, bw, BnFwdFin{},
             BnBwdFin{}, nullptr);
  return check_launch();
}

int coper_bn_act_bwd_finalize(const float* partials, int nchunk, int64_t R, int C, int use_batch_stats,
                              float* dgamma, float* dbeta, float* c1, float* c2, coper_stream_t stream) {
  COPER_CHECK_ARG(partials && dgamma && dbeta && c1 && c2 && nchunk > 0 && R > 0 && C > 0);
  BnBwdFin f{use_batch_stats, dgamma, dbeta, c1, c2};
  launch_pdl(bn_bwd_finalize_kernel, ceil_div((int64_t)C * 32, 256), 256, 0, as_stream(stream), partials, nchunk, R,
             C, f);
  return check_launch();
}

int coper_bn_act_bwd_stats_finalize(const float* dout, const float* x, int64_t R, int C, const float* a, const float* b,
                                    const float* mean, const float* invstd, int relu, float keep_post,
                                    const uint64_t* seed_dev, uint64_t salt_post, float* partials,
                                    unsigned int* sync_word, int use_batch_stats, float* dgamma, float* dbeta, float* c1,
                                    float* c2, coper_stream_t stream) {
  COPER_CHECK_ARG(dout && x && a && b && mean && invstd && partials && sync_word && R > 0 && C > 0 && keep_post > 0.f);
  COPER_CHECK_ARG(dgamma && dbeta && c1 && c2);
  dim3 grid(ceil_div(C, 32), coper_colstats_chunks(R)), block(32, 8);
  StatBwdArgs bw{dout, a, b, mean, invstd, relu, keep_post, 1.0f / keep_post, keep_threshold(keep_post), seed_dev,
                 salt_post};
  BnBwdFin f{use_batch_stats, dgamma, dbeta, c1, c2};
  launch_pdl(colstats_kernel<1, true>, grid, block, 0, as_stream(stream), x, R, C, partials, bw, BnFwdFin{}, f,
             sync_word);
  return check_launch();
}

int coper_bn_act_bwd_apply(const float* dout, const float* x, int64_t R, int C, const float* a, const float* b,
                           const float* mean, const float* invstd, const float* c1, const float* c2, int relu,
                           float keep_post, const uint64_t* seed_dev, uint64_t salt_post, float keep_pre,
                           uint64_t salt_pre, float* dx, coper_stream_t stream) {
  COPER_CHECK_ARG(dout && x && a && b && mean && invstd && c1 && c2 && dx && R > 0 && C > 0);
  COPER_CHECK_ARG(keep_post > 0.f && keep_pre > 0.f);
  int64_t n = R * C;
  launch_pdl(bn_act_bwd_apply_kernel, grid_for(n, 256), 256, 0, as_stream(stream), dout, x, n, C, a, b, mean, invstd,
             c1, c2, relu, keep_post, 1.0f / keep_post, keep_threshold(keep_post), seed_dev, salt_post, keep_pre,
             1.0f / keep_pre, keep_threshold(keep_pre), salt_pre, dx);
  return check_launch();
}

int coper_dropout_mask(int64_t n, float keep, const uint64_t* seed_dev, uint64_t salt, float* mask,
                       coper_stream_t stream) {
  COPER_CHECK_ARG(mask && n >= 0 && keep > 0.f);
  if (n == 0) return COPER_OK;
  launch_pdl(dropout_mask_kernel, grid_for(n, 256), 256, 0, as_stream(stream), n, keep_threshold(keep), keep,
             seed_dev, salt, mask);
  return check_launch();
}
int coper_dropout_apply(float* x, int64_t n, float keep, const uint64_t* seed_dev, uint64_t salt,
                        coper_stream_t stream) {
  COPER_CHECK_ARG(x && n >= 0 && keep > 0.f);
  if (n == 0 || keep >= 1.0f) return COPER_OK;
  launch_pdl(dropout_apply_kernel, grid_for(n, 256), 256, 0, as_stream(stream), x, n, keep, 1.0f / keep,
             keep_threshold(keep), seed_dev, salt);
  return check_launch();
}

int coper_csr_to_bits(const int32_t* rowptr, const int32_t* col, int B, int64_t ent_lo, int64_t ent_hi,
                      uint32_t* bits, coper_stream_t stream) {
  COPER_CHECK_ARG(rowptr && bits && B > 0 && ent_hi > ent_lo);
  int64_t words = (ent_hi - ent_lo + 31) / 32;
  int rc = check_cuda(cudaMemsetAsync(bits, 0, (size_t)B * words * sizeof(uint32_t), as_stream(stream)));
  if (rc) return rc;
  if (!col) return COPER_OK;
  launch_pdl(csr_to_bits_kernel, B, 64, 0, as_stream(stream), rowptr, col, B, ent_lo, ent_hi, words, bits);
  return check_launch();
}
int coper_dense_to_bits(const float* dense, int B, int64_t N, uint32_t* bits, coper_stream_t stream) {
  COPER_CHECK_ARG(dense && bits && B > 0 && N > 0);
  int64_t words = (N + 31) / 32;
  int64_t threads = (int64_t)B * words * 32;
  launch_pdl(dense_to_bits_kernel, (unsigned)((threads + 255) / 256), 256, 0, as_stream(stream), dense, B, N, words,
             bits);
  return check_launch();
}

int coper_csr_to_bits_t(const int32_t* rowptr, const int32_t* col, int B, int64_t ent_lo, int64_t ent_hi,
                        uint32_t* bits_t, coper_stream_t stream) {
  COPER_CHECK_ARG(rowptr && col && bits_t && B > 0 && ent_hi > ent_lo);
  int wordsB = (B + 31) / 32;
  int rc = check_cuda(cudaMemsetAsync(bits_t, 0, (size_t)(ent_hi - ent_lo) * wordsB * sizeof(uint32_t), as_stream(stream)));
  if (rc) return rc;
  launch_pdl(csr_to_bits_t_kernel, B, 128, 0, as_stream(stream), rowptr, col, B, ent_lo, ent_hi, wordsB, bits_t);
  return check_launch();
}
int coper_bits_t_set(const int64_t* ent, int B, int64_t ent_lo, int64_t ent_hi, uint32_t* bits_t, coper_stream_t stream) {
  COPER_CHECK_ARG(ent && bits_t && B > 0 && ent_hi > ent_lo);
  launch_pdl(bits_t_set_kernel, (B + 127) / 128, 128, 0, as_stream(stream), ent, B, ent_lo, ent_hi, (B + 31) / 32,
             bits_t);
  return check_launch();
}
int coper_dense_to_bits_t(const float* dense, int B, int64_t N, int64_t ld_dense, uint32_t* bits_t, coper_stream_t stream) {
  COPER_CHECK_ARG(dense && bits_t && B > 0 && N > 0 && ld_dense >= N);
  int wordsB = (B + 31) / 32;
  int64_t threads = N * wordsB * 32;
  launch_pdl(dense_to_bits_t_kernel, (unsigned)((threads + 255) / 256), 256, 0, as_stream(stream), dense, B, N,
             ld_dense, wordsB, bits_t);
  return check_launch();
}

int coper_reduce_partials(const float* in, int S, int64_t n, float scale, int accumulate, float* out,
                          coper_stream_t stream) {
  COPER_CHECK_ARG(in && out && S > 0 && n > 0);
  if (S <= 8 && n >= (1 << 16) && (n & 3) == 0 && ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) == 0) {
    launch_pdl(reduce_partials_few_kernel, (unsigned)((n / 4 + 255) / 256), 256, 0, as_stream(stream), in, S, n,
               scale, accumulate, out);
    return check_launch();
  }
  return reduce_partials_and_sum(in, S, n, scale, accumulate, out, nullptr, 0, nullptr, as_stream(stream));
}
int coper_reduce_partials2(const float* in_a, int64_t n_a, float* out_a, const float* in_b, int64_t n_b, float* out_b,
                           int S, float scale, int accumulate, coper_stream_t stream) {
  COPER_CHECK_ARG(in_a && out_a && in_b && out_b && S > 0 && n_a > 0 && n_b > 0);
  ReduceJob A{in_a, S, n_a, scale, accumulate, out_a}, Bj{in_b, S, n_b, scale, accumulate, out_b};
  const int ba = (int)((n_a + 31) / 32), bb = (int)((n_b + 31) / 32);
  launch_pdl(reduce_partials_kernel<false>, ba + bb, 256, 0, as_stream(stream), A, ba, Bj, bb, nullptr, 0, nullptr);
  return check_launch();
}
int coper_sumsq(const float* x, int64_t n, int slot, double* partials, coper_stream_t stream) {
  COPER_CHECK_ARG(x && partials && n >= 0 && slot >= 0);
  launch_pdl(sumsq_kernel, COPER_SUMSQ_BLOCKS, 256, 0, as_stream(stream), x, n, partials + (int64_t)slot *
             COPER_SUMSQ_BLOCKS);
  return check_launch();
}
int coper_clip_scale(const double* partials, int n_slots, float clip_norm, float* out2, coper_stream_t stream) {
  COPER_CHECK_ARG(partials && out2 && n_slots > 0 && clip_norm > 0.f);
  launch_pdl(clip_scale_kernel, 1, 256, 0, as_stream(stream), partials, n_slots * COPER_SUMSQ_BLOCKS, clip_norm,
             out2);
  return check_launch();
}
int coper_clip_scale_n(const double* sums, int n, float clip_norm, float* out2, coper_stream_t stream) {
  COPER_CHECK_ARG(sums && out2 && n > 0 && clip_norm > 0.f);
  launch_pdl(clip_scale_kernel, 1, 256, 0, as_stream(stream), sums, n, clip_norm, out2);
  return check_launch();
}
int coper_mt_sumsq(const coper_param_desc* descs, int n_tensors, const int32_t* chunks, int n_chunks,
                   const int32_t* chunk_offsets, double* chunk_partials, double* tensor_sumsq, coper_stream_t stream) {
  COPER_CHECK_ARG(descs && chunks && chunk_offsets && chunk_partials && tensor_sumsq && n_tensors > 0 && n_chunks > 0);
  launch_pdl(mt_sumsq_kernel, n_chunks, 256, 0, as_stream(stream), descs, chunks, chunk_partials);
  int rc = check_launch();
  if (rc) return rc;
  launch_pdl(mt_tensor_sums_kernel, (n_tensors * 32 + 255) / 256, 256, 0, as_stream(stream), descs, chunk_partials,
             chunk_offsets, n_tensors, tensor_sumsq);
  return check_launch();
}
int coper_mt_sumsq_clip(const coper_param_desc* descs, int n_tensors, const int32_t* chunks, int n_chunks,
                        const int32_t* chunk_offsets, double* chunk_partials, double* tensor_sumsq, int ext_tensor,
                        const double* ext_parts, int n_ext_parts, const double* ext_deltas, int n_ext_deltas,
                        float clip_norm, float* clip_out, coper_stream_t stream) {
  COPER_CHECK_ARG(descs && chunk_offsets && chunk_partials && tensor_sumsq && n_tensors > 0 && n_chunks >= 0);
  COPER_CHECK_ARG(n_chunks == 0 || chunks);
  COPER_CHECK_ARG(ext_tensor < n_tensors && n_ext_parts >= 0 && n_ext_deltas >= 0);
  COPER_CHECK_ARG((ext_parts || n_ext_parts == 0) && (ext_deltas || n_ext_deltas == 0));
  COPER_CHECK_ARG(!clip_out || clip_norm > 0.f);
  int rc;
  if (n_chunks > 0) {
    launch_pdl(mt_sumsq_kernel, n_chunks, 256, 0, as_stream(stream), descs, chunks, chunk_partials);
    if ((rc = check_launch())) return rc;
  }
  launch_pdl(mt_sumsq_finish_kernel, 1, 256, 0, as_stream(stream), descs, chunk_partials, chunk_offsets, n_tensors,
             tensor_sumsq, ext_tensor, ext_parts, n_ext_parts, ext_deltas, n_ext_deltas, clip_norm, clip_out);
  return check_launch();
}
int coper_mt_amsgrad(const coper_param_desc* descs, const int32_t* chunks, int n_chunks, const float* step_state,
                     float beta1, float beta2, float eps, const float* clip_scale, int bug_compat,
                     coper_stream_t stream) {
  COPER_CHECK_ARG(descs && chunks && step_state && n_chunks > 0);
  launch_pdl(mt_amsgrad_kernel, n_chunks, 256, 0, as_stream(stream), descs, chunks, step_state, beta1, beta2, eps,
             clip_scale, bug_compat);
  return check_launch();
}
int coper_sumsq_combine(const double* parts, int n_parts, const double* deltas, int n_deltas, double* out,
                        coper_stream_t stream) {
  COPER_CHECK_ARG(out && n_parts >= 0 && n_deltas >= 0 && (parts || n_parts == 0) && (deltas || n_deltas == 0));
  launch_pdl(sumsq_combine_kernel, 1, 256, 0, as_stream(stream), parts, n_parts, deltas, n_deltas, out);
  return check_launch();
}
int coper_step_state_advance(float* step_state, uint64_t* seed_dev, float lr, float beta1, float beta2,
                             coper_stream_t stream) {
  COPER_CHECK_ARG(step_state);
  launch_pdl(step_state_advance_kernel, 1, 32, 0, as_stream(stream), step_state, seed_dev, lr, beta1, beta2);
  return check_launch();
}
int coper_amsgrad_step(float* theta, const float* grad, float* m, float* v, float* vhat, int64_t n,
                       const float* step_state, float beta1, float beta2, float eps, const float* clip_scale,
                       int bug_compat, coper_stream_t stream) {
  COPER_CHECK_ARG(theta && grad && vhat && step_state && n >= 0);
  COPER_CHECK_ARG(bug_compat || (m && v));
  if (n == 0) return COPER_OK;
  launch_pdl(amsgrad_kernel, grid_for(n, 256, 16), 256, 0, as_stream(stream), theta, grad, m, v, vhat, n, step_state,
             beta1, beta2, eps, clip_scale, bug_compat);
  return check_launch();
}

}  // extern "C"
