// Generic (any k, d) SIMT kernels of the Lloyd loop: exact-fp32 tiled assign, ownership-based
// (atomic-free, deterministic) per-cluster partial sums, fixed-order reductions, finalize.
// These serve every pass b2k_choose_kernel (b2k_api.cu) leaves on the generic path, the update of a chunked Lloyd
// loop, the k-means|| initialiser, and KMeansModel.transform for odd shapes.  sm_100a only; no CPU fallback.
//
// Semantics restated from the reference's backend (EXTERNAL cuML 25.12, called at
// spark_rapids_ml/clustering.py:383-415): argmin over ||c||^2 - 2 x.c with lowest index on ties,
// empty cluster keeps its centroid, convergence on sum_j||dc_j||^2 < tol (SURVEY.md §8a a-6..a-9).
#include <float.h>

#include "b2k_internal.cuh"

#define B2K_EARLY_EXIT(st) \
  if ((st) != nullptr && (st)->done) return;

// ------------------------------------------------------------------------------------------------
// ||c_j||^2 : one warp per center, double accumulation, fp32 result
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_center_norms(const float* __restrict__ C, int k, int d,
                                                      float* __restrict__ cnorm, const B2kLoopState* st) {
  B2K_EARLY_EXIT(st);
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (warp >= k) return;
  const float* c = C + (size_t)warp * d;
  double s = 0.0;
  for (int t = lane; t < d; t += 32) s += (double)c[t] * (double)c[t];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) cnorm[warp] = (float)s;
}

int b2k_launch_center_norms(b2k_ctx* ctx, const float* C, int k, int d, float* cnorm, const B2kLoopState* st,
                            cudaStream_t s) {
  int blocks = (k * 32 + 255) / 256;
  k_center_norms<<<blocks, 256, 0, s>>>(C, k, d, cnorm, st);
  ctx->stats.kernel_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

// ------------------------------------------------------------------------------------------------
// assign: BM x BN register-tiled fp32 FMA contraction, running (min, argmin) over center tiles.
// ------------------------------------------------------------------------------------------------
namespace {
constexpr int BM = 64, BN = 64, BK = 16, PADX = 4;

__global__ void __launch_bounds__(256) k_assign_generic(const float* __restrict__ X, int64_t n, int d,
                                                        const float* __restrict__ C,
                                                        const float* __restrict__ cnorm, int k,
                                                        int32_t* __restrict__ labels,
                                                        float* __restrict__ mindist, const B2kLoopState* st) {
  B2K_EARLY_EXIT(st);
  __shared__ __align__(16) float Xs[BK][BM + PADX];
  __shared__ __align__(16) float Cs[BK][BN + PADX];
  const int tid = threadIdx.x;
  const int tx = tid & 15;   // center group
  const int ty = tid >> 4;   // row group
  const int64_t row0 = (int64_t)blockIdx.x * BM;

  float best[4];
  int bestj[4];
  float xn[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 4; ++i) { best[i] = FLT_MAX; bestj[i] = 0; }

  for (int j0 = 0; j0 < k; j0 += BN) {
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < d; k0 += BK) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int idx = tid + 256 * i;
        int r = idx / BK, c = idx % BK;
        int64_t gr = row0 + r;
        float v = 0.f;
        if (gr < n && k0 + c < d) v = X[(size_t)gr * d + k0 + c];
        Xs[c][r] = v;
        int gj = j0 + r;
        float w = 0.f;
        if (gj < k && k0 + c < d) w = C[(size_t)gj * d + k0 + c];
        Cs[c][r] = w;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) {
        float4 xa = *reinterpret_cast<const float4*>(&Xs[kk][ty * 4]);
        float4 cb = *reinterpret_cast<const float4*>(&Cs[kk][tx * 4]);
        float xv[4] = {xa.x, xa.y, xa.z, xa.w};
        float cv[4] = {cb.x, cb.y, cb.z, cb.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xv[i], cv[j], acc[i][j]);
        }
        if (j0 == 0) {
#pragma unroll
          for (int i = 0; i < 4; ++i) xn[i] = fmaf(xv[i], xv[i], xn[i]);
        }
      }
      __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int gj = j0 + tx * 4 + j;
      if (gj < k) {
        float cn = cnorm[gj];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float dist = fmaf(-2.f, acc[i][j], cn);
          if (dist < best[i]) { best[i] = dist; bestj[i] = gj; }
        }
      }
    }
  }
  // combine the 16 center groups of each row: lexicographic (dist, index) minimum
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      float ob = __shfl_xor_sync(0xffffffffu, best[i], o);
      int oj = __shfl_xor_sync(0xffffffffu, bestj[i], o);
      if (ob < best[i] || (ob == best[i] && oj < bestj[i])) { best[i] = ob; bestj[i] = oj; }
    }
    int64_t gr = row0 + ty * 4 + i;
    if (tx == 0 && gr < n) {
      if (labels) labels[gr] = bestj[i];
      if (mindist) mindist[gr] = fmaxf(xn[i] + best[i], 0.f);
    }
  }
}
}  // namespace

int b2k_launch_assign_generic(b2k_ctx* ctx, const float* X, int64_t n, int d, const float* C,
                              const float* cnorm, int k, int32_t* labels, float* mindist,
                              const B2kLoopState* st, cudaStream_t s) {
  if (n <= 0) return B2K_OK;
  int64_t blocks = (n + BM - 1) / BM;
  if (blocks > 0x7fffffffLL) return b2k_fail(ctx, B2K_ERR_INVALID, "assign_generic: too many rows");
  k_assign_generic<<<(unsigned)blocks, 256, 0, s>>>(X, n, d, C, cnorm, k, labels, mindist, st);
  ctx->stats.kernel_launches++;
  ctx->stats.generic_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

// ------------------------------------------------------------------------------------------------
// update: CTA (p, cc) owns rows chunk p x columns [cc*CW, cc*CW+CW); thread t owns ONE column, so the
// shared-memory accumulators S[k][CW] need no atomics and the result is deterministic.
// ------------------------------------------------------------------------------------------------
__global__ void k_update_smem(const float* __restrict__ X, int64_t n, int d,
                              const int32_t* __restrict__ labels, int k, int64_t rows_per_chunk,
                              float* __restrict__ partials, int32_t* __restrict__ counts,
                              const B2kLoopState* st) {
  B2K_EARLY_EXIT(st);
  extern __shared__ float S[];  // [k][CW] then int cnt[k]
  const int CW = blockDim.x;
  int* cnt = reinterpret_cast<int*>(S + (size_t)k * CW);
  const int t = threadIdx.x;
  const int p = blockIdx.x, cc = blockIdx.y;
  const int col = cc * CW + t;
  const bool col_ok = col < d;
  for (int j = 0; j < k; ++j) S[(size_t)j * CW + t] = 0.f;
  for (int j = t; j < k; j += CW) cnt[j] = 0;
  __syncthreads();
  int64_t r0 = (int64_t)p * rows_per_chunk;
  int64_t r1 = r0 + rows_per_chunk;
  if (r1 > n) r1 = n;
  int64_t r = r0;
  for (; r + 4 <= r1; r += 4) {
    int l0 = labels[r], l1 = labels[r + 1], l2 = labels[r + 2], l3 = labels[r + 3];
    float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
    if (col_ok) {
      v0 = X[(size_t)r * d + col];
      v1 = X[(size_t)(r + 1) * d + col];
      v2 = X[(size_t)(r + 2) * d + col];
      v3 = X[(size_t)(r + 3) * d + col];
    }
    S[(size_t)l0 * CW + t] += v0;
    S[(size_t)l1 * CW + t] += v1;
    S[(size_t)l2 * CW + t] += v2;
    S[(size_t)l3 * CW + t] += v3;
    if (cc == 0 && t == 0) { cnt[l0]++; cnt[l1]++; cnt[l2]++; cnt[l3]++; }
  }
  for (; r < r1; ++r) {
    int l0 = labels[r];
    float v0 = col_ok ? X[(size_t)r * d + col] : 0.f;
    S[(size_t)l0 * CW + t] += v0;
    if (cc == 0 && t == 0) cnt[l0]++;
  }
  __syncthreads();
  if (col_ok) {
    float* out = partials + (size_t)p * k * d;
    for (int j = 0; j < k; ++j) out[(size_t)j * d + col] = S[(size_t)j * CW + t];
  }
  if (cc == 0)
    for (int j = t; j < k; j += CW) counts[(size_t)p * k + j] = cnt[j];
}

// k too large for shared-memory accumulators: warp per row, fp32 atomics into one partial (P == 1).
__global__ void __launch_bounds__(256) k_update_atomic(const float* __restrict__ X, int64_t n, int d,
                                                       const int32_t* __restrict__ labels,
                                                       float* __restrict__ partials,
                                                       int32_t* __restrict__ counts, const B2kLoopState* st) {
  B2K_EARLY_EXIT(st);
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < n; r += nwarps) {
    int l = labels[r];
    const float* x = X + (size_t)r * d;
    float* sdst = partials + (size_t)l * d;
    for (int c = lane; c < d; c += 32) atomicAdd(sdst + c, x[c]);
    if (lane == 0) atomicAdd(counts + l, 1);
  }
}

__global__ void k_zero_f32(float* p, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = 0.f;
}

namespace {
struct UpdatePlan {
  int CW;      // 0 => atomic path
  int P;
  int colchunks;
  size_t smem;
};
UpdatePlan plan_update(const b2k_ctx* ctx, int64_t n, int d, int k) {
  UpdatePlan u{};
  size_t cap = ctx->smem_optin ? ctx->smem_optin : (size_t)48 * 1024;
  cap -= 1024;
  int CW = 0;
  if ((size_t)k * 128 * 4 + (size_t)k * 4 <= cap) CW = 128;
  else if ((size_t)k * 32 * 4 + (size_t)k * 4 <= cap) CW = 32;
  if (d < 64 && CW == 128 && (size_t)k * 32 * 4 + (size_t)k * 4 <= cap) CW = 32;
  u.CW = CW;
  if (CW == 0) { u.P = 1; u.colchunks = 0; u.smem = 0; return u; }
  u.smem = (size_t)k * CW * 4 + (size_t)k * 4;
  u.colchunks = (d + CW - 1) / CW;
  int per_sm = (int)((ctx->smem_optin ? ctx->smem_optin : 48 * 1024) / (u.smem + 1024));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 8) per_sm = 8;
  int64_t target = (int64_t)ctx->sm_count * per_sm * 2;
  int64_t P = (target + u.colchunks - 1) / u.colchunks;
  // bound the partial scratch to 512 MB
  int64_t maxP = ((int64_t)512 << 20) / ((int64_t)k * d * 4 + 1);
  if (maxP < 1) maxP = 1;
  if (P > maxP) P = maxP;
  int64_t min_rows = 256;  // do not split below 256 rows per chunk
  int64_t maxP2 = (n + min_rows - 1) / min_rows;
  if (maxP2 < 1) maxP2 = 1;
  if (P > maxP2) P = maxP2;
  if (P < 1) P = 1;
  u.P = (int)P;
  return u;
}
}  // namespace

int b2k_update_generic_slots(b2k_ctx* ctx, int64_t n, int d, int k) { return plan_update(ctx, n, d, k).P; }

int b2k_launch_update_generic(b2k_ctx* ctx, const float* X, int64_t n, int d, const int32_t* labels, int k,
                              int P, float* partials, int32_t* counts, const B2kLoopState* st,
                              cudaStream_t s) {
  UpdatePlan u = plan_update(ctx, n, d, k);
  if (u.P != P) return b2k_fail(ctx, B2K_ERR_STATE, "update_generic: plan mismatch");
  if (u.CW == 0) {
    size_t tot = (size_t)k * d;
    k_zero_f32<<<(unsigned)((tot + 1023) / 1024 > 4096 ? 4096 : (tot + 1023) / 1024), 256, 0, s>>>(partials, tot);
    B2K_CUDA_OK(ctx, cudaMemsetAsync(counts, 0, (size_t)k * sizeof(int32_t), s));
    k_update_atomic<<<ctx->sm_count * 8, 256, 0, s>>>(X, n, d, labels, partials, counts, st);
    ctx->stats.kernel_launches += 2;
  } else {
    B2K_CUDA_OK(ctx, cudaFuncSetAttribute(k_update_smem, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)u.smem));
    int64_t rows_per_chunk = (n + u.P - 1) / u.P;
    dim3 grid(u.P, u.colchunks);
    k_update_smem<<<grid, u.CW, u.smem, s>>>(X, n, d, labels, k, rows_per_chunk, partials, counts, st);
    ctx->stats.kernel_launches++;
  }
  ctx->stats.generic_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

// ------------------------------------------------------------------------------------------------
// R = fixed-order sum over partials (double): [k*d sums | k counts | cost]
// ------------------------------------------------------------------------------------------------
// sum of m doubles by one warp in a FIXED order (lane-strided chains, then a shuffle tree): deterministic
__device__ __forceinline__ double warp_fold_f64(const double* __restrict__ in, int m) {
  const int lane = threadIdx.x & 31;
  double a = 0.0;
  for (int i = lane; i < m; i += 32) a += in[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  return a;
}

__global__ void __launch_bounds__(256) k_reduce_partials(const float* __restrict__ partials,
                                                         const int32_t* __restrict__ counts, int P,
                                                         const double* __restrict__ cost_partials, int Pc,
                                                         int k, int d, double* __restrict__ R,
                                                         const B2kLoopState* st) {
  B2K_EARLY_EXIT(st);
  size_t kd = (size_t)k * d;
  if (blockIdx.x == gridDim.x - 1) {   // the extra block: the cost partials, one warp
    if (threadIdx.x < 32) {
      const double a = cost_partials ? warp_fold_f64(cost_partials, Pc) : 0.0;
      if (threadIdx.x == 0) R[kd + k] = a;
    }
    return;
  }
  size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < kd) {
    double a = 0.0;
    for (int p = 0; p < P; ++p) a += (double)partials[(size_t)p * kd + e];
    R[e] = a;
  } else if (e < kd + k) {
    int j = (int)(e - kd);
    double a = 0.0;
    for (int p = 0; p < P; ++p) a += (double)counts[(size_t)p * k + j];
    R[e] = a;
  }
}

int b2k_launch_reduce_partials(b2k_ctx* ctx, const float* partials, const int32_t* counts,
                               const double* cost_partials, int P, int Pc, int k, int d, double* R,
                               const B2kLoopState* st, cudaStream_t s) {
  size_t len = b2k_reduced_len(k, d);
  unsigned blocks = (unsigned)((len + 255) / 256) + 1;   // + the cost block
  k_reduce_partials<<<blocks, 256, 0, s>>>(partials, counts, P, cost_partials, Pc, k, d, R, st);
  ctx->stats.kernel_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

// ------------------------------------------------------------------------------------------------
// finalize: one CTA per cluster; the last CTA to finish folds the per-cluster shifts in index order.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_finalize(const double* __restrict__ R, float* __restrict__ C, int k,
                                                  int d, double* __restrict__ shift_scratch,
                                                  B2kLoopState* st) {
  if (st->done) return;
  __shared__ double red[128];
  __shared__ bool is_last;
  const int j = blockIdx.x;
  const size_t kd = (size_t)k * d;
  const double w = R[kd + j];
  double local = 0.0;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float old = C[(size_t)j * d + c];
    float nw = old;
    if (w > 0.0) nw = (float)(R[(size_t)j * d + c] / w);
    double df = (double)nw - (double)old;
    local += df * df;
    C[(size_t)j * d + c] = nw;
  }
  red[threadIdx.x] = local;
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    shift_scratch[j] = red[0];
    __threadfence();
    unsigned int prev = atomicAdd(&st->blocks_done, 1u);
    is_last = (prev == (unsigned)k - 1);
  }
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    __threadfence();
    double sh = 0.0;
    const volatile double* ss = shift_scratch;
    for (int q = 0; q < k; ++q) sh += ss[q];
    st->shift = sh;
    st->cost = R[kd + k];
    st->iter += 1;
    st->blocks_done = 0;
    if (sh < st->tol || st->iter >= st->max_iter) st->done = 1;
    __threadfence();
  }
}

int b2k_launch_finalize(b2k_ctx* ctx, const double* R, float* C, int k, int d, double* shift_scratch,
                        B2kLoopState* st, cudaStream_t s) {
  k_finalize<<<k, 128, 0, s>>>(R, C, k, d, shift_scratch, st);
  ctx->stats.kernel_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

// ------------------------------------------------------------------------------------------------
// deterministic fp32 -> fp64 sum (inertia through the generic path)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_block_sums(const float* __restrict__ v, int64_t n,
                                                    double* __restrict__ block_out) {
  __shared__ double red[256];
  int64_t per = (n + gridDim.x - 1) / gridDim.x;
  int64_t a = (int64_t)blockIdx.x * per, b = a + per;
  if (b > n) b = n;
  double acc = 0.0;
  for (int64_t i = a + threadIdx.x; i < b; i += 256) acc += (double)v[i];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) block_out[blockIdx.x] = red[0];
}
__global__ void k_fold_f64(const double* __restrict__ in, int m, double* __restrict__ out) {
  if (blockIdx.x == 0 && threadIdx.x < 32) {
    const double a = warp_fold_f64(in, m);
    if (threadIdx.x == 0) out[0] = a;
  }
}

int b2k_launch_fold_f64(b2k_ctx* ctx, const double* in, int m, double* out, cudaStream_t s) {
  k_fold_f64<<<1, 32, 0, s>>>(in, m, out);
  ctx->stats.kernel_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

int b2k_launch_sum_f32_to_f64(b2k_ctx* ctx, const float* v, int64_t n, double* out, double* block_scratch,
                              int nblocks, cudaStream_t s) {
  k_block_sums<<<nblocks, 256, 0, s>>>(v, n, block_scratch);
  k_fold_f64<<<1, 32, 0, s>>>(block_scratch, nblocks, out);
  ctx->stats.kernel_launches += 2;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

// ------------------------------------------------------------------------------------------------
// init helpers
// ------------------------------------------------------------------------------------------------
__global__ void k_gather_rows(const float* __restrict__ X, int d, const int64_t* __restrict__ rows, int m,
                              float* __restrict__ out, int64_t out_row0) {
  int i = blockIdx.x;
  if (i >= m) return;
  const float* src = X + (size_t)rows[i] * d;
  float* dst = out + (size_t)(out_row0 + i) * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) dst[c] = src[c];
}
int b2k_launch_gather_rows(b2k_ctx* ctx, const float* X, int d, const int64_t* rows_local, int m, float* out,
                           int64_t out_row0, cudaStream_t s) {
  if (m <= 0) return B2K_OK;
  k_gather_rows<<<m, 128, 0, s>>>(X, d, rows_local, m, out, out_row0);
  ctx->stats.kernel_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

// chunked assign (k > 256): fold one chunk's (min distance, local label) into the running (min distance, global label);
// strict '<' keeps the earlier chunk (= the lower cluster index) on ties
__global__ void k_merge_chunk(float* __restrict__ md_acc, int32_t* __restrict__ lab_acc, const float* __restrict__ md,
                              const int32_t* __restrict__ lab, int base, int64_t n, const B2kLoopState* st) {
  B2K_EARLY_EXIT(st);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    const float v = md[i];
    if (v < md_acc[i]) {
      md_acc[i] = v;
      lab_acc[i] = lab[i] + base;
    }
  }
}
int b2k_launch_merge_chunk(b2k_ctx* ctx, float* md_acc, int32_t* lab_acc, const float* md, const int32_t* lab, int base,
                           int64_t n, const B2kLoopState* st, cudaStream_t s) {
  if (n <= 0) return B2K_OK;
  int64_t blocks = (n + 255) / 256;
  if (blocks > ctx->sm_count * 16) blocks = ctx->sm_count * 16;
  k_merge_chunk<<<(unsigned)blocks, 256, 0, s>>>(md_acc, lab_acc, md, lab, base, n, st);
  ctx->stats.kernel_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

// weighted centroid update of the k-means|| candidate refinement: one CTA per centre scans the (few thousand) candidates
// in index order — fp64 sums, fixed order, identical on every rank
__global__ void __launch_bounds__(256) k_weighted_update(const float* __restrict__ P, const double* __restrict__ w,
                                                         const int32_t* __restrict__ lab, int M, int d,
                                                         float* __restrict__ C) {
  const int j = (int)blockIdx.x;
  for (int t = (int)threadIdx.x; t < d; t += (int)blockDim.x) {
    double S = 0.0, W = 0.0;
    for (int i = 0; i < M; ++i) {
      if (lab[i] == j) {
        const double wi = w[i];
        S += wi * (double)P[(size_t)i * d + t];
        W += wi;
      }
    }
    if (W > 0.0) C[(size_t)j * d + t] = (float)(S / W);
  }
}
int b2k_launch_weighted_update(b2k_ctx* ctx, const float* P, const double* w, const int32_t* lab, int M, int d, int k,
                               float* C, cudaStream_t s) {
  k_weighted_update<<<k, 256, 0, s>>>(P, w, lab, M, d, C);
  ctx->stats.kernel_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// Bernoulli(min(1, scale * mind[i])) keyed on the GLOBAL row index: the sample does not depend on how the
// rows are partitioned across GPUs.
__global__ void k_bernoulli_pick(const float* __restrict__ mind, int64_t n, int64_t row_offset, double scale,
                                 uint64_t seed, int round, int64_t* __restrict__ picked,
                                 int* __restrict__ n_picked, int cap) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    uint64_t g = (uint64_t)(row_offset + i);
    uint64_t h = splitmix64(splitmix64(seed ^ (0xD1B54A32D192ED03ull * (uint64_t)(round + 1))) ^ g);
    double u = (double)(h >> 11) * (1.0 / 9007199254740992.0);
    double p = scale * (double)mind[i];
    if (u < p) {
      int slot = atomicAdd(n_picked, 1);
      if (slot < cap) picked[slot] = (int64_t)g;
    }
  }
}
int b2k_launch_bernoulli_pick(b2k_ctx* ctx, const float* mind, int64_t n, int64_t row_offset, double scale,
                              uint64_t seed, int round, int64_t* picked, int* n_picked, int cap,
                              cudaStream_t s) {
  if (n <= 0) return B2K_OK;
  int64_t blocks = (n + 255) / 256;
  if (blocks > ctx->sm_count * 16) blocks = ctx->sm_count * 16;
  k_bernoulli_pick<<<(unsigned)blocks, 256, 0, s>>>(mind, n, row_offset, scale, seed, round, picked, n_picked,
                                                    cap);
  ctx->stats.kernel_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

__global__ void k_histogram(const int32_t* __restrict__ labels, int64_t n, int m,
                            unsigned long long* __restrict__ hist) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    int l = labels[i];
    if (l >= 0 && l < m) atomicAdd(hist + l, 1ull);
  }
}
__global__ void k_u64_to_f64(const unsigned long long* in, double* out, int m) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) out[i] = (double)in[i];
}
// hist (double[m]) doubles as the u64 accumulation buffer (same width), converted in place at the end.
int b2k_launch_histogram(b2k_ctx* ctx, const int32_t* labels, int64_t n, int m, double* hist, cudaStream_t s) {
  B2K_CUDA_OK(ctx, cudaMemsetAsync(hist, 0, (size_t)m * sizeof(double), s));
  if (n > 0) {
    int64_t blocks = (n + 255) / 256;
    if (blocks > ctx->sm_count * 16) blocks = ctx->sm_count * 16;
    k_histogram<<<(unsigned)blocks, 256, 0, s>>>(labels, n, m, reinterpret_cast<unsigned long long*>(hist));
  }
  k_u64_to_f64<<<(m + 255) / 256, 256, 0, s>>>(reinterpret_cast<unsigned long long*>(hist), hist, m);
  ctx->stats.kernel_launches += 2;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}


// ------------------------------------------------------------------------------------------------
// D2[i][j] = ||p_i - p_j||^2 for the (few thousand) k-means|| candidates: feeds the weighted greedy k-means++ of the
// candidate reduction, which would otherwise recompute M*d-long distances k*trials times on one host thread.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pairwise_sqdist(const float* __restrict__ P, int M, int d, float* __restrict__ D2) {
  __shared__ float a[16][33], b[16][33];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int i = blockIdx.y * 16 + ty, j = blockIdx.x * 16 + tx;
  double acc = 0.0;
  for (int t0 = 0; t0 < d; t0 += 32) {
    for (int e = threadIdx.x; e < 16 * 32; e += 256) {
      const int r = e >> 5, c = e & 31;
      const int gi = blockIdx.y * 16 + r, gj = blockIdx.x * 16 + r;
      a[r][c] = (gi < M && t0 + c < d) ? P[(size_t)gi * d + t0 + c] : 0.f;
      b[r][c] = (gj < M && t0 + c < d) ? P[(size_t)gj * d + t0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int c = 0; c < 32; ++c) {
      const float df = a[ty][c] - b[tx][c];
      acc += (double)df * (double)df;
    }
    __syncthreads();
  }
  if (i < M && j < M) D2[(size_t)i * M + j] = (float)acc;
}

int b2k_launch_pairwise_sqdist(b2k_ctx* ctx, const float* P, int M, int d, float* D2, cudaStream_t s) {
  dim3 grid((M + 15) / 16, (M + 15) / 16);
  k_pairwise_sqdist<<<grid, 256, 0, s>>>(P, M, d, D2);
  ctx->stats.kernel_launches++;
  ctx->stats.generic_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}
