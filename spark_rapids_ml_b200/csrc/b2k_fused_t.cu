// Fused assign + per-cluster partial-sum kernel for LARGE (k, d) on sm_100a — k <= 256, d <= 256 (BASELINE cfg3:
// k = 256, d = 256) — ONE pass over X per Lloyd iteration.  "T" = transposed operand roles with respect to
// b2k_fused_tc.cu: at k = d = 256 neither the centres (256 KB) nor per-CTA [k, d] accumulators (256 KB) fit beside
// a row tile in one SM, and 3xTF32 would be tensor-bound at 2.4x the HBM time.  So:
//
//   * CTA PAIR (cluster of 2, tcgen05 cta_group::2, UMMA M = 256, N = 128, K = 8):
//       A  = the CENTRES, tf32 (round-to-nearest), resident in TMEM for the whole launch: CTA r holds centres
//            [128 r, 128 r + 128) as 128 lanes x DP columns                                   (TMEM cols [0, 256))
//       B  = the X row tile, fed STRAIGHT from the TMA ring (raw fp32 words; the tensor core truncates them to
//            tf32): each CTA supplies 64 of the step's 128 rows — no convert stage, no operand copy in TMEM
//       D  = [cluster, row] partial products, fp32, double buffered                          (TMEM cols [256, 512))
//   * 1xTF32 screening + exact recheck: the epilogue turns D into dist' = ||c||^2 - 2 x~.c~, packs (dist', cluster)
//     into one ordered 32-bit key, and a shuffle butterfly finds the smallest AND second smallest key of every row
//     across the 32 lanes of a warp; 4 warps x 2 CTAs exchange their partials through (distributed) shared memory.
//     A row whose gap is below the PROVEN bound thr = 2E (E: worst-case error of one dist', see k_tables_t) is
//     DEFERRED: the epilogue appends it (row id + the bit mask of every cluster within thr of the best = its
//     candidates) to the CTA pair's segment of a fix-up list and publishes no label for it, so the pass never
//     waits for an exact evaluation.  k_fix_labels_t then decides those rows exactly (fp32 dot products against the
//     fp32 centres, ascending cluster order, strict '<' = lowest index on ties) and k_fix_accum_t adds them to
//     FIX_SLOTS = 4 extra partial-sum slots (slot q: the segments q mod 4, fixed list order: deterministic).  Rows
//     outside the bound provably have the same argmin in exact arithmetic, so labels match the 3xTF32 / fp32 path.
//   * update: per-cluster sums live in REGISTERS, one [256, 256] accumulator set per CTA PAIR (each CTA: 128
//     clusters x 256 columns = 64 registers per update thread).  Each update warp finds its rows itself from the
//     labels the epilogue publishes (through the cluster -> warp table of k_tables_t) and reads them from the local
//     ring or, for the peer's rows, through DSMEM (ld.shared::cluster).  No atomics; static schedule; deterministic.
//   * assign / inertia passes (UPD = false): the same screening + recheck for the labels; the "update" warps
//     compute the exact min distance sum (x - c)^2 of every row from the tile in shared memory.
//
// Replaces (for these shapes) cuML's fusedL2NN + reduce_rows_by_key reached from
// spark_rapids_ml/clustering.py:412-415 (SURVEY.md §8a a-6/a-7).  Algorithmic HBM bytes per launch: 4*n*d (X once)
// + 8*n (row norms) [+ 4*n labels / 4*n mindist when requested] + 78 * (k*d + k) * 4 partials (74 CTA pairs + 4 fix-up slots) + 40 B per deferred row.
#include <float.h>
#include <stdio.h>

#include "b2k_internal.cuh"

namespace {

#include "b2k_ptx.cuh"

constexpr int TN = 128;                      // X rows per step = UMMA N (64 per CTA of the pair)
constexpr int TNH = 64;
constexpr int CHUNK = 32;                    // f32 per 128-byte swizzle row = one TMA box / 4 UMMA K steps
constexpr int SLOT_BYTES = TNH * CHUNK * 4;  // 8 KB: [64 rows x 32 f32], 128B swizzle = K-major SW128 UMMA B operand
constexpr int NSLOT = 24;                    // ring: 192 KB per CTA
constexpr int KH = 128;                      // centres per CTA (TMEM lanes)
constexpr int D_OFF = 256;                   // TMEM column of D buffer 0 (A occupies [0, DP))
constexpr int TMEM_COLS = 512;

constexpr int W_EPI0 = 0;                    // warps 0-3: epilogue (TMEM lane quadrant = warp % 4)
constexpr int W_UPD0 = 4;                    // warps 4-19: update
constexpr int N_UPD = 16;
constexpr int CPW = KH / N_UPD;              // 8 clusters per update warp
constexpr int W_TMA = W_UPD0 + N_UPD;        // 20
constexpr int W_MMA = W_TMA + 1;             // 21
constexpr int NWARPS = 24;                   // 768 threads launched at 80 registers (22 working warps + 2 that pad the last
                                             // warpgroup).  Lloyd pass at d > 128: the TMA/MMA warpgroup drops to 40
                                             // registers (setmaxnreg.dec) and the 16 update warps raise themselves to 88
                                             // from that pool (64 accumulator registers each): 4x32x80 + 4x32x40 + 16x32x88
constexpr int NTHREADS = NWARPS * 32;

// shared memory layout (dynamic, 1 KB aligned base)
constexpr int OFF_RING = 0;
constexpr int OFF_PART = NSLOT * SLOT_BYTES;            // uint2 part[2][8 sources][128 columns]: (best, second) keys
constexpr int OFF_LAB = OFF_PART + 2 * 8 * TN * 8;      // int32 lab[2][128]: final labels of the step
constexpr int OFF_XOFF = OFF_LAB + 2 * TN * 4;          // f32 xoff[128]: per-row key offset ||x||^2 + thr
constexpr int OFF_SORT = OFF_XOFF + TN * 4;             // cluster <-> update-warp key tables, see SortT
struct SortT {
  static constexpr int KEYTAB = 0;                      // u8 [256] cluster -> key (cta*128 + warp*8 + slot)
  static constexpr int KEYINV = KEYTAB + 256;           // u8 [256] key -> cluster
  static constexpr int BYTES = KEYINV + 256;
};
constexpr int OFF_MISC = (OFF_SORT + SortT::BYTES + 15) & ~15;   // flag words [4] u32, tmem ptr, cost doubles [16]
constexpr int MISC_FLAGW = 0, MISC_TMEMPTR = 32, MISC_COST = 48;
constexpr int OFF_BARS = OFF_MISC + 48 + 16 * 8;
constexpr int XG = 4;                        // chunks per x_full barrier: a completed mbarrier wait costs the MMA issuer ~400-500
                                             // cycles (measured), so it waits per half step (4 chunks), not per chunk
constexpr int B_XFULL = 0;                   // [NSLOT / XG used] leader CTA only: both CTAs' TMA boxes of a chunk group landed
constexpr int B_SFREE = B_XFULL + NSLOT;     // [8] step slot may be overwritten (local + remote update roles done)
constexpr int B_DFULL = B_SFREE + 8;         // [2]
constexpr int B_DEMPTY = B_DFULL + 2;        // [2] leader CTA only, count 2
constexpr int B_LFULL = B_DEMPTY + 2;        // [2]
constexpr int B_LEMPTY = B_LFULL + 2;        // [2]
constexpr int B_PX = B_LEMPTY + 2;           // [2] the peer's partial keys of a step landed here (st.async complete_tx)
constexpr int NBARS = B_PX + 2;
constexpr uint32_t PX_BYTES = 4u * (TN / 32) * 32u * 8u;   // 4 warps x 4 chunks x 32 lanes x 8 bytes per step
constexpr int SMEM_BYTES = OFF_BARS + NBARS * 8;
static_assert(SMEM_BYTES <= 227 * 1024, "smem");

// ---- extra PTX for this kernel ----
// TMA load whose completion is signalled on the LEADER CTA's mbarrier (cta_group::2; CUTLASS: SM100_TMA_2SM_LOAD_2D)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar_cluster, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar_cluster), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// remote store that itself signals the destination CTA's mbarrier (complete_tx): no release fence on the producer side
__device__ __forceinline__ void st_async_v2(uint32_t addr_cluster, uint32_t a, uint32_t b, uint32_t bar_cluster) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];" ::"r"(addr_cluster),
               "r"(a), "r"(b), "r"(bar_cluster)
               : "memory");
}
__device__ __forceinline__ void ld_cluster_2(uint32_t addr_cluster, uint64_t& a, uint64_t& b) {
  asm volatile("ld.shared::cluster.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr_cluster));
}

// Bounded wait without a call: a function call inside the update role's setmaxnreg region makes ptxas give up on the
// region's larger register budget (measured: 76 bytes of accumulator spills with mbar_wait's noinline time-out report).
__device__ __forceinline__ void mbar_wait_nocall(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins == (1u << 22)) __trap();
  }
}

__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// Keys: (dist' + ||x||^2 + thr) is a positive float, so its bits order like an unsigned integer; the low 8 bits carry the
// cluster index (2^-15 relative resolution of the key value, part of the proven bound in k_tables_t).
// merge two (smallest, second smallest) pairs of disjoint key sets
__device__ __forceinline__ void merge2(uint32_t& a1, uint32_t& a2, uint32_t b1, uint32_t b2) {
  const uint32_t lo = min(a1, b1), hi = max(a1, b1);
  a2 = min(hi, min(a2, b2));
  a1 = lo;
}
// One level of the transposing butterfly over lane bit LM: on entry a lane holds 2 N columns, on exit the N columns whose
// index bit matches its lane bit, reduced over the lane pair.
template <int N, int LM>
__device__ __forceinline__ void bfly2_level(uint32_t (&m1)[8], uint32_t (&m2)[8], int lane) {
  const bool hi = (lane & LM) != 0;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const uint32_t s1 = hi ? m1[i] : m1[i + N], s2 = hi ? m2[i] : m2[i + N];
    uint32_t k1 = hi ? m1[i + N] : m1[i], k2 = hi ? m2[i + N] : m2[i];
    const uint32_t r1 = __shfl_xor_sync(0xffffffffu, s1, LM), r2 = __shfl_xor_sync(0xffffffffu, s2, LM);
    merge2(k1, k2, r1, r2);
    m1[i] = k1;
    m2[i] = k2;
  }
}

// ------------------------------------------------------------------------------------------------
// prep kernels
// ------------------------------------------------------------------------------------------------
// Ct[256][DP] = centres rounded to nearest tf32, zero padded; cnorm[256] = ||c||^2 (+inf for padding clusters)
__global__ void __launch_bounds__(256) k_prep_centers_t(const float* __restrict__ C, int k, int d, int DP,
                                                        float* __restrict__ Ct, float* __restrict__ cnorm,
                                                        const B2kLoopState* st) {
  if (st != nullptr && st->done) return;
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= 256) return;
  double s = 0.0, e = 0.0;
  for (int t = lane; t < DP; t += 32) {
    const float v = (row < k && t < d) ? C[(size_t)row * d + t] : 0.f;
    const float r = __uint_as_float(rn_tf32_bits(v));
    Ct[(size_t)row * DP + t] = r;
    s += (double)v * (double)v;
    e += ((double)v - (double)r) * ((double)v - (double)r);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    e += __shfl_xor_sync(0xffffffffu, e, o);
  }
  if (lane == 0) {
    cnorm[row] = row < k ? (float)s : __int_as_float(0x7f800000);
    cnorm[256 + row] = row < k ? (float)sqrt(e) : 0.f;   // ||c - c~||: the rounding error of this centre's tf32 operand
  }
}

// One block of 256 threads: (a) cluster -> update-warp key table balanced by the previous iteration's cluster
// sizes (32 "virtual" update warps = 16 per CTA of the pair, 8 slots each; key = vwarp * 8 + slot, so that
// key >> 7 = owning CTA); (b) the coefficients of the recheck threshold thr(x), see "Bound" below.
//
// Bound.  dist'_j = fl(||c_j||^2 - 2 x~.c~_j) with x~ = x cut to tf32 by the tensor core (dx = x~ - x, ||dx|| measured per
// row by k_row_norms) and c~ = RN_tf32(c) (dc_j = c~_j - c_j, ||dc_j|| measured per centre by k_prep_centers_t):
//   |x~.c~ - x.c| = |dx.c~ + x.dc| <= ||dx|| ||c~|| + ||x|| ||dc||                                    (Cauchy-Schwarz)
// tf32 products are exact in fp32; the fp32 accumulation of d <= 256 terms adds at most d * 2^-23 ||x|| ||c||
// <= 2^-15 ||x|| ||c|| (truncating adder assumed); the final fma and add round twice (2^-23 relative) and the key drops
// 8 mantissa bits (2^-15 relative), relative to the key value ||x - c||^2 + thr <= (||x|| + ||c||)^2 + thr.  With
// Cmax = max_j ||c_j|| (1 + 2^-11), dCmax = max_j ||dc_j||:
//   E(x) <= 2 (||dx|| Cmax + ||x|| dCmax) + ||x|| Cmax 2^-14 + (||x|| + Cmax)^2 2^-14
// Two approximate distances can be off by E each in opposite directions, so the argmin is proven whenever the gap exceeds
// 2E.  Shipped with a 1.25x margin (also covers the fp32 rounding of the norms themselves):
//   thr(x) = T0 ||dx|| + T1 ||x|| + T2 ||x||^2 + T3,
//   T0 = 5 Cmax,  T1 = 5 dCmax + Cmax 2^-12 * 1.25 + Cmax 2^-12 * 1.25,  T2 = 2^-13 * 1.25,  T3 = Cmax^2 2^-13 * 1.25
__global__ void __launch_bounds__(256) k_tables_t(const double* __restrict__ counts, int k, const float* __restrict__ cnorm,
                                                  uint8_t* __restrict__ keytab, uint8_t* __restrict__ keyinv,
                                                  float* __restrict__ thr, const B2kLoopState* st) {
  if (st != nullptr && st->done) return;
  __shared__ double w[256];
  __shared__ float cmax2[8];
  __shared__ float dcmax[8];
  const int j = threadIdx.x;
  w[j] = (counts != nullptr && j < k) ? counts[j] : -1.0;   // padding clusters sort last
  float c2 = j < k ? cnorm[j] : 0.f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c2 = fmaxf(c2, __shfl_xor_sync(0xffffffffu, c2, o));
  if ((j & 31) == 0) cmax2[j >> 5] = c2;
  __syncthreads();
  float dc = j < k ? cnorm[256 + j] : 0.f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dc = fmaxf(dc, __shfl_xor_sync(0xffffffffu, dc, o));
  if ((j & 31) == 0) dcmax[j >> 5] = dc;
  __syncthreads();
  if (j == 0) {
    float m = 0.f, dm = 0.f;
    for (int i = 0; i < 8; ++i) { m = fmaxf(m, cmax2[i]); dm = fmaxf(dm, dcmax[i]); }
    const float cmax = sqrtf(m) * 1.0005f;
    thr[0] = 5.f * cmax;
    thr[1] = 5.f * dm + cmax * 0.0006103515625f;          // 2 * 1.25 * 2^-12
    thr[2] = 0.000152587890625f;                          // 1.25 * 2^-13
    thr[3] = cmax * cmax * 0.000152587890625f;
  }
  int key;
  if (counts == nullptr) {
    key = (j & 31) * CPW + (j >> 5);
  } else {
    int rank = 0;   // position in (count desc, index asc) order
    for (int i = 0; i < 256; ++i) rank += (w[i] > w[j]) || (w[i] == w[j] && i < j);
    const int round = rank >> 5, pos = rank & 31;
    const int owner = (round & 1) ? (31 - pos) : pos;
    key = owner * CPW + round;
  }
  keytab[j] = (uint8_t)key;
  keyinv[key] = (uint8_t)j;
}

// xnorm[i] = { ||x_i||, ||x_i - trunc_tf32(x_i)|| } (fp32).  One pass over X, once per fit / lloyd / assign call (X is
// immutable during the call).  The second value is the norm of the error the tensor core makes on this row when it cuts
// the fp32 words to tf32 (an upper bound if the hardware rounds instead: |RN error| <= |truncation error| per element).
__global__ void __launch_bounds__(256) k_row_norms(const float* __restrict__ X, int64_t n, int d, float2* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int d4 = d >> 2;
  for (int64_t row = warp0; row < n; row += nwarps) {
    const float4* p = reinterpret_cast<const float4*>(X + row * d);
    float s = 0.f, e = 0.f;
    for (int t = lane; t < d4; t += 32) {
      const float4 v = __ldcs(p + t);
      s = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, s))));
      const float ex = v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u);
      const float ey = v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u);
      const float ez = v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u);
      const float ew = v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u);
      e = fmaf(ex, ex, fmaf(ey, ey, fmaf(ez, ez, fmaf(ew, ew, e))));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      e += __shfl_xor_sync(0xffffffffu, e, o);
    }
    if (lane == 0) out[row] = make_float2(sqrtf(s) * 1.0000002f, sqrtf(e) * 1.0000002f);   // round up
  }
}

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
struct TArgs {
  int64_t n;
  int nsteps;
  int k;
  int d;
  const float* Ct;         // [256][DP] tf32 centres
  const float* C32;        // [k][d] fp32 centres (recheck, min distance)
  const float* cnorm;      // [256]
  const float* thr;        // [4]
  const float2* xnorm;     // [n] {||x||, ||x - trunc_tf32(x)||}
  const uint8_t* keytab;   // [256]
  const uint8_t* keyinv;   // [256]
  float* partials;         // [npairs][k*d]
  int32_t* counts;         // [npairs][k]
  double* cost_partials;   // [grid]
  int32_t* labels_out;     // [n] or NULL
  float* mind_out;         // [n] or NULL
  int need_cost;
  unsigned long long* rstat;   // [2] deferred (rechecked) rows, candidates evaluated (diagnostics) or NULL
  // deferred rows: CTA pair p appends to fix_list[p * seg_cap ..] in step order (a fixed function of the data) and
  // writes fix_count[p] when it is done; entries below mask_cap also carry their 256-bit candidate mask
  int2* fix_list;              // {row, label (-1 until k_fix_labels_t)}
  uint32_t* fix_masks;         // [npairs][mask_cap][8]
  int32_t* fix_count;          // [npairs]
  int seg_cap;
  int mask_cap;
  const B2kLoopState* st;
};

template <int NCH, bool UPD>
__global__ void __launch_bounds__(NTHREADS, 1) k_fused_t(const __grid_constant__ CUtensorMap mapX, const TArgs args) {
  constexpr int NSTEP = NSLOT / NCH;          // steps resident in the ring (3 at DP = 256)
  constexpr int UPL = NCH / 4;                // float4 units per lane of a row (1 or 2)
  static_assert(NCH == 4 || NCH == 8, "NCH");
  if (args.st != nullptr && args.st->done) return;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = smem_u32(smem_raw);
  uint8_t* gbase = smem_raw;
  if ((base & 1023u) != 0u) {
    if (threadIdx.x == 0) printf("b2k fused_t: dynamic shared memory base %u is not 1 KB aligned\n", base);
    __trap();
  }
  const uint32_t ring = base + OFF_RING;
  const uint32_t bars = base + OFF_BARS;
  auto bar = [&](int i) -> uint32_t { return bars + 8u * (uint32_t)i; };
  uint2* part_s = reinterpret_cast<uint2*>(gbase + OFF_PART);
  float* xoff_s = reinterpret_cast<float*>(gbase + OFF_XOFF);
  int32_t* lab_s = reinterpret_cast<int32_t*>(gbase + OFF_LAB);
  uint8_t* sort_s = gbase + OFF_SORT;
  uint8_t* keytab_s = sort_s + SortT::KEYTAB;
  uint8_t* keyinv_s = sort_s + SortT::KEYINV;
  uint32_t* flagw_s = reinterpret_cast<uint32_t*>(gbase + OFF_MISC + MISC_FLAGW);
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(gbase + OFF_MISC + MISC_TMEMPTR);
  double* cost_s = reinterpret_cast<double*>(gbase + OFF_MISC + MISC_COST);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const uint32_t peer = rank ^ 1u;

  // ---- one-time setup ----
  if (warp == W_TMA && lane == 0) {
    tma_prefetch_desc(&mapX);
    for (int i = 0; i < NSLOT; ++i) mbar_init(bar(B_XFULL + i), 1);
    for (int i = 0; i < 8; ++i) mbar_init(bar(B_SFREE + i), 2 * N_UPD);   // every update warp of both CTAs
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(B_DFULL + i), 1);
      mbar_init(bar(B_DEMPTY + i), 2);
      mbar_init(bar(B_LFULL + i), 1);
      mbar_init(bar(B_LEMPTY + i), N_UPD);
    }
    mbar_init(bar(B_PX + 0), 1);
    mbar_init(bar(B_PX + 1), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == W_MMA) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_s)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  for (int j = threadIdx.x; j < 256; j += NTHREADS) {
    keytab_s[j] = args.keytab[j];
    keyinv_s[j] = args.keyinv[j];
  }
  if (threadIdx.x < 16) cost_s[threadIdx.x] = 0.0;
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // peer barriers initialised / TMEM allocated before any remote signal
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr_s, 0);

  // static schedule: cluster q handles steps q, q + nclusters, ...; CTA `rank` loads rows [128 step + 64 rank, +64)
  const int sched0 = (int)(blockIdx.x >> 1);
  const int sched_step = (int)(gridDim.x >> 1);
  const int nit = sched0 < args.nsteps ? (args.nsteps - sched0 + sched_step - 1) / sched_step : 0;
  auto step_of = [&](int it) -> int { return sched0 + it * sched_step; };

  // A operand: this CTA's 128 centres (tf32) -> TMEM columns [0, 32 NCH), lane = centre
  if (warp < W_UPD0) {
    const int jl = warp * 32 + lane;
    const float4* src = reinterpret_cast<const float4*>(args.Ct + ((size_t)rank * KH + jl) * (NCH * CHUNK));
    const uint32_t lane_field = (uint32_t)(warp * 32) << 16;
#pragma unroll 1
    for (int cb = 0; cb < NCH; ++cb) {
      uint32_t v[32];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 f = __ldg(src + cb * 8 + q);
        v[q * 4 + 0] = __float_as_uint(f.x);
        v[q * 4 + 1] = __float_as_uint(f.y);
        v[q * 4 + 2] = __float_as_uint(f.z);
        v[q * 4 + 3] = __float_as_uint(f.w);
      }
      tmem_st_x32(tmem_base + lane_field + (uint32_t)(cb * 32), v);
    }
    tmem_wait_st();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // both CTAs' A operands are in TMEM before the leader's first MMA
  tc_fence_after();

  if (warp >= W_UPD0 && warp < W_TMA) {
    // ======================= update warps =======================
    const int u = warp - W_UPD0;
    if constexpr (UPD && NCH == 8) asm volatile("setmaxnreg.inc.sync.aligned.u32 88;" ::: "memory");
    uint64_t acc[CPW][UPL][2];
    int cnt = 0;   // lane c < CPW: rows of owned cluster slot c
#pragma unroll
    for (int c = 0; c < CPW; ++c) {
#pragma unroll
      for (int i = 0; i < UPL; ++i) acc[c][i][0] = acc[c][i][1] = 0ull;
    }
    const uint32_t unit_js = (uint32_t)(lane & 7) << 4;
    const int k0 = (int)rank * KH + u * CPW;   // this warp's key range [k0, k0 + CPW)
    double cost = 0.0;
    for (int it = 0; it < nit; ++it) {
      const int b = it & 1;
      const uint32_t bph = (uint32_t)(it >> 1) & 1u;
      const int ss = it % NSTEP;
      // The update warps run decoupled (no per-step barrier among them): rows per warp and step are Poisson(4), and a
      // barrier would make every step wait for its most loaded warp (measured: 5-7 k cycles per step against 2.5 k mean).
      mbar_wait_nocall(bar(B_LFULL + b), bph);
      // The x_full phases of this step completed before the MMA consumed the slots, which happens-before the
      // commit, the epilogue and hence lab_full: the rows are in shared memory (both CTAs).
      const uint32_t slot0 = ring + (uint32_t)((ss * NCH + (lane >> 3)) * SLOT_BYTES);
      if constexpr (UPD) {
        // this warp's rows of the step: labels whose key (cluster -> update warp table) lies in [k0, k0 + 8); processed in
        // column order with two rows in flight whatever their clusters (a fixed function of the labels: deterministic)
        uint32_t keyp = 0, vmask = 0;   // per lane: keys of columns lane + 32 sx (one byte each), validity bits
#pragma unroll
        for (int sx = 0; sx < 4; ++sx) {
          const int lab = lab_s[b * TN + sx * 32 + lane];
          if (lab >= 0) {
            keyp |= (uint32_t)keytab_s[lab] << (8 * sx);
            vmask |= 1u << sx;
          }
        }
        auto load_row = [&](int colr, uint64_t (&v)[UPL][2]) {
          const int lrow = colr & 63;
          const uint32_t a0 = slot0 + (((uint32_t)(lrow * 128 + ((lrow & 7) << 4))) ^ unit_js);
          if ((uint32_t)(colr >> 6) == rank) {
#pragma unroll
            for (int i = 0; i < UPL; ++i) lds128_2(a0 + (uint32_t)(i * 4 * SLOT_BYTES), v[i][0], v[i][1]);
          } else {
            const uint32_t r0 = mapa_u32(a0, peer);
#pragma unroll
            for (int i = 0; i < UPL; ++i) ld_cluster_2(r0 + (uint32_t)(i * 4 * SLOT_BYTES), v[i][0], v[i][1]);
          }
        };
        auto add_row = [&](int c, const uint64_t (&v)[UPL][2]) {
          switch (c) {
#define B2K_ADD_CASE(C_)                                        \
  case C_:                                                      \
    _Pragma("unroll") for (int k2 = 0; k2 < UPL; ++k2) {        \
      acc[C_][k2][0] = add2(acc[C_][k2][0], v[k2][0]);          \
      acc[C_][k2][1] = add2(acc[C_][k2][1], v[k2][1]);          \
    }                                                           \
    break;
            B2K_ADD_CASE(0) B2K_ADD_CASE(1) B2K_ADD_CASE(2) B2K_ADD_CASE(3)
            B2K_ADD_CASE(4) B2K_ADD_CASE(5) B2K_ADD_CASE(6) B2K_ADD_CASE(7)
#undef B2K_ADD_CASE
            default: break;
          }
        };
        // two rows in flight: the load of row i + 1 is issued before row i is added (its latency — 30 cycles local,
        // several hundred through DSMEM under load — is the cost of a row; measured ~700-1000 cycles per row serial)
        uint64_t vA[UPL][2], vB[UPL][2];
        int pend = 0, cP = 0;   // pend: 0 nothing in flight, 1 = vA, 2 = vB (the buffers alternate: no register copies)
#pragma unroll 1
        for (int sx = 0; sx < 4; ++sx) {
          uint32_t m = __ballot_sync(0xffffffffu, ((vmask >> sx) & 1u) != 0u &&
                                                       (((keyp >> (8 * sx)) & 255u) - (uint32_t)k0) < (uint32_t)CPW);
          while (m) {
            const int bit = __ffs(m) - 1;
            m &= m - 1;
            const int cc = (int)((__shfl_sync(0xffffffffu, keyp, bit) >> (8 * sx)) & 255u) - (k0 & 255);
            if (lane == cc) ++cnt;
            if (pend == 0) {
              load_row(sx * 32 + bit, vA);
              pend = 1;
            } else if (pend == 1) {
              load_row(sx * 32 + bit, vB);
              add_row(cP, vA);
              pend = 2;
            } else {
              load_row(sx * 32 + bit, vA);
              add_row(cP, vB);
              pend = 1;
            }
            cP = cc;
          }
        }
        if (pend == 1) add_row(cP, vA);
        else if (pend == 2) add_row(cP, vB);
      } else if (args.need_cost) {
        // exact min distance of this CTA's own rows: sum_t (x_t - c_t)^2 against the row's (final) centre
#pragma unroll 1
        for (int rr = 0; rr < TNH / N_UPD; ++rr) {
          const int lrow = u + N_UPD * rr;
          const int col = (int)rank * TNH + lrow;
          const int64_t grow = (int64_t)step_of(it) * TN + col;
          if (grow >= args.n) continue;
          const int label = lab_s[b * TN + col];
          if (label < 0) continue;   // deferred: k_fix_labels_t writes its min distance
          float s = 0.f;
#pragma unroll
          for (int i = 0; i < UPL; ++i) {
            const int cc = (lane + 32 * i) * 4;
            if (cc < args.d) {
              const float4 xv = lds128(slot0 + (uint32_t)(i * 4 * SLOT_BYTES) +
                                       (((uint32_t)(lrow * 128 + ((lrow & 7) << 4))) ^ unit_js));
              const float4 cv = __ldg(reinterpret_cast<const float4*>(args.C32 + (size_t)label * args.d + cc));
              const float dx = xv.x - cv.x, dy = xv.y - cv.y, dz = xv.z - cv.z, dw = xv.w - cv.w;
              s = fmaf(dx, dx, fmaf(dy, dy, fmaf(dz, dz, fmaf(dw, dw, s))));
            }
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
          if (lane == 0) {
            if (args.mind_out != nullptr) args.mind_out[grow] = s;
            cost += (double)s;
          }
        }
      }
      __syncwarp();
      if (lane == 0) {
        // the rows were consumed (their values fed the adds above) before these arrivals: relaxed is enough for the
        // write-after-read hand-back of the slots to the TMA producers of both CTAs
        mbar_arrive(bar(B_LEMPTY + b));
        mbar_arrive(bar(B_SFREE + ss));
        mbar_arrive_cluster(bar(B_SFREE + ss), peer);
      }
    }
    if constexpr (UPD) {
      // flush: partials[pair][l][col .. col+3] for the owned clusters l = keyinv[rank*128 + u*8 + c]
      float* out = args.partials + (size_t)(blockIdx.x >> 1) * args.k * args.d;
#pragma unroll
      for (int c = 0; c < CPW; ++c) {
        const int l = (int)keyinv_s[(int)rank * KH + u * CPW + c];
        if (l < args.k) {
#pragma unroll
          for (int i = 0; i < UPL; ++i) {
            const int colx = (lane + 32 * i) * 4;
            float e[4];
            unpack2(acc[c][i][0], e[0], e[1]);
            unpack2(acc[c][i][1], e[2], e[3]);
#pragma unroll
            for (int t = 0; t < 4; ++t)
              if (colx + t < args.d) out[(size_t)l * args.d + colx + t] = e[t];
          }
          const int cn_c = __shfl_sync(0xffffffffu, cnt, c);
          if (lane == 0) args.counts[(size_t)(blockIdx.x >> 1) * args.k + l] = cn_c;
        }
      }
    } else {
      if (lane == 0) cost_s[u] = cost;
    }
  } else if (warp >= W_TMA) {
    if constexpr (UPD && NCH == 8) asm volatile("setmaxnreg.dec.sync.aligned.u32 40;" ::: "memory");
   if (warp == W_TMA) {
    // ======================= TMA producer =======================
    const uint32_t xfull_leader0 = mapa_u32(bar(B_XFULL), 0u);   // the leader CTA's x_full[0] (cluster address)
    for (int it = 0; it < nit; ++it) {
      const int step = step_of(it);
      const int ss = it % NSTEP;
      const uint32_t sph = (uint32_t)(it / NSTEP) & 1u;
      // CTA-scope wait: a cluster-scope acquire makes ptxas append CCTL.IVALL (L1 invalidate, ~400 cycles) to every wait
      // (measured: 8 of them per step put 3.6 k cycles on the MMA issuer).  What these barriers order is async-proxy
      // traffic (TMA writes / UMMA reads) and TMEM (tcgen05 fences), not generic-proxy data in the peer's memory.
      mbar_wait_nocall(bar(B_SFREE + ss), sph ^ 1u);
#pragma unroll 1
      for (int c = 0; c < NCH; ++c) {
        const int slot = ss * NCH + c;
        const int xb = slot / XG;
        if (elect_one()) {
          if (rank == 0 && (c % XG) == 0) mbar_expect_tx(bar(B_XFULL + xb), 2u * XG * SLOT_BYTES);
          tma_load_2d_pair(ring + slot * SLOT_BYTES, &mapX, xfull_leader0 + 8u * (uint32_t)xb, c * CHUNK,
                           step * TN + (int)rank * TNH);
        }
        __syncwarp();
      }
    }
  } else if (warp == W_MMA) {
    // ======================= MMA issuer (leader CTA only) =======================
    constexpr uint32_t idesc = make_idesc_tf32(256, TN);
    for (int it = 0; it < (rank != 0 ? 0 : nit); ++it) {
      const int b = it & 1;
      const uint32_t bph = (uint32_t)(it >> 1) & 1u;
      const int ss = it % NSTEP;
      const uint32_t sph = (uint32_t)(it / NSTEP) & 1u;
      mbar_wait_nocall(bar(B_DEMPTY + b), bph ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + D_OFF + b * TN;
#pragma unroll 1
      for (int c = 0; c < NCH; ++c) {
        const int slot = ss * NCH + c;
        if ((c % XG) == 0) {
          mbar_wait_nocall(bar(B_XFULL + slot / XG), sph);
          tc_fence_after();
        }
        if (elect_one()) {
          const uint32_t bx = ring + slot * SLOT_BYTES;
#pragma unroll
          for (int ks = 0; ks < CHUNK / 8; ++ks)
            tc_mma_ts_tf32_pair(d_tmem, tmem_base + (uint32_t)(c * CHUNK + ks * 8), make_kmajor_sw128_desc(bx + ks * 32),
                                idesc, (c | ks) != 0 ? 1u : 0u);
          if (c == NCH - 1) tc_commit_pair(bar(B_DFULL + b));
        }
        __syncwarp();
      }
    }
   }
  } else if (warp < W_UPD0) {
    // ======================= epilogue warps: D -> keys -> (best, second) -> labels =======================
    // tcgen05.ld.16x256b hands thread (t0 = lane & 3, t1 = lane >> 2) the TMEM lanes t1 and t1 + 8 of a 16-lane half and
    // the columns 8 r + 2 t0 + {0, 1}: with both halves a thread owns 4 clusters x 8 columns of a 32-column chunk, reduces
    // its 4 clusters in registers and only 3 shuffle levels (over t1) remain.
    const int w = warp - W_EPI0;
    const int col = w * 32 + lane;                      // the column (row of the step) this thread combines
    const int t0 = lane & 3, t1 = lane >> 2;
    const uint32_t jid0 = rank * KH + (uint32_t)(w * 32 + t1);   // + 16 h + 8 e: the 4 clusters of this thread
    float cn4[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) cn4[q] = args.cnorm[jid0 + 8 * q];   // q = 2 h + e
    const int cidx = (lane & 24) | ((lane & 3) << 1) | ((lane >> 2) & 1);   // column of the chunk this lane ends up with
    const float thr0 = args.thr[0], thr1 = args.thr[1], thr2 = args.thr[2], thr3 = args.thr[3];
    const uint32_t part_peer0 = mapa_u32(base + OFF_PART, peer);
    const uint32_t px_peer0 = mapa_u32(bar(B_PX), peer);
    const uint32_t dempty_leader = mapa_u32(bar(B_DEMPTY), 0u);
    const uint32_t src = rank * 4u + (uint32_t)w;
    const int pairid = (int)(blockIdx.x >> 1);
    int2* const seg_list = args.fix_list + (size_t)pairid * (size_t)args.seg_cap;
    uint32_t* const seg_mask = args.fix_masks + (size_t)pairid * (size_t)args.mask_cap * 8u;
    int seg_cnt = 0;   // deferred rows of this pair so far (identical in all epilogue threads of both CTAs)
    unsigned long long n_flag = 0;
    float2 xn_next = make_float2(0.f, 0.f);
    if (nit > 0) {
      const int64_t g0 = (int64_t)step_of(0) * TN + col;
      if (g0 < args.n) xn_next = __ldg(args.xnorm + g0);
    }
    for (int it = 0; it < nit; ++it) {
      const int step = step_of(it);
      const int b = it & 1;
      const uint32_t bph = (uint32_t)(it >> 1) & 1u;
      const int64_t grow = (int64_t)step * TN + col;
      const bool valid = grow < args.n;
      const float xn = xn_next.x, dxn = xn_next.y;
      if (it + 1 < nit) {   // prefetch the next step's row norms: a global load must not sit on the step's serial chain
        const int64_t gn = (int64_t)step_of(it + 1) * TN + col;
        xn_next = gn < args.n ? __ldg(args.xnorm + gn) : make_float2(0.f, 0.f);
      }
      const float thr = fmaf(dxn, thr0, fmaf(xn, fmaf(xn, thr2, thr1), thr3));
      // per-row key offset ||x||^2 + thr: dist' + offset = ||x - c||^2 + thr +- E > 0, so that the float bits of a key
      // order like unsigned integers, with the key's resolution relative to the true squared distance
      xoff_s[col] = fmaf(xn, xn, thr);
      if (threadIdx.x == 0) mbar_expect_tx(bar(B_PX + b), PX_BYTES);   // the peer's partials of this step
      // two barriers, two warps: even a completed wait costs several hundred cycles, so they are polled in parallel and
      // joined by the hardware barrier below
      if (w == 0) mbar_wait(bar(B_DFULL + b), bph);
      if (w == 1) mbar_wait(bar(B_LEMPTY + b), bph ^ 1u);   // lab[b] of step it - 2 has been consumed by the update role
      asm volatile("bar.sync 1, 128;" ::: "memory");
      tc_fence_after();
#pragma unroll 1
      for (int g = 0; g < TN / 32; ++g) {
        uint32_t v[2][16];
        const uint32_t ta = tmem_base + ((uint32_t)(w * 32) << 16) + (uint32_t)(D_OFF + b * TN + g * 32);
        tmem_ld_16x256b_x4(ta, v[0]);
        tmem_ld_16x256b_x4(ta + (16u << 16), v[1]);
        tmem_wait_ld();
        uint32_t m1[8], m2[8];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const float2 xo = *reinterpret_cast<const float2*>(xoff_s + g * 32 + 8 * r + 2 * t0);
#pragma unroll
          for (int sx = 0; sx < 2; ++sx) {
            uint32_t kk[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {   // q = 2 h + e: cluster jid0 + 8 q
              const float dist = fmaf(-2.f, __uint_as_float(v[q >> 1][4 * r + 2 * (q & 1) + sx]), cn4[q]) + (sx ? xo.y : xo.x);
              kk[q] = (__float_as_uint(dist) & 0xffffff00u) | (jid0 + 8u * (uint32_t)q);
            }
            const uint32_t a = min(kk[0], kk[1]), bb = max(kk[0], kk[1]);
            const uint32_t c = min(kk[2], kk[3]), dd = max(kk[2], kk[3]);
            m1[2 * r + sx] = min(a, c);
            m2[2 * r + sx] = min(max(a, c), min(bb, dd));
          }
        }
        bfly2_level<4, 16>(m1, m2, lane);
        bfly2_level<2, 8>(m1, m2, lane);
        bfly2_level<1, 4>(m1, m2, lane);
        const int pi = (b * 8 + (int)src) * TN + g * 32 + cidx;
        part_s[pi] = make_uint2(m1[0], m2[0]);
        st_async_v2(part_peer0 + (uint32_t)pi * 8u, m1[0], m2[0], px_peer0 + 8u * (uint32_t)b);
      }
      tc_fence_before();
      asm volatile("bar.sync 1, 128;" ::: "memory");   // this CTA's partials
      // D of this parity is drained in this CTA (nothing below reads TMEM)
      if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(dempty_leader + 8u * (uint32_t)b)
                     : "memory");
      }
      mbar_wait(bar(B_PX + b), bph);                    // the peer's partials
      // combine the 8 partials of my column (source s8 = the 32 clusters [32 s8, 32 s8 + 32))
      uint32_t M1 = 0xffffffffu, M2 = 0xffffffffu;
      uint2 pp[8];
#pragma unroll
      for (int s8 = 0; s8 < 8; ++s8) {
        pp[s8] = part_s[(b * 8 + s8) * TN + col];
        merge2(M1, M2, pp[s8].x, pp[s8].y);
      }
      int label = (int)(M1 & 255u);
      const float M1f = __uint_as_float(M1 & 0xffffff00u);
      const bool flag = valid && ((__uint_as_float(M2 & 0xffffff00u) - M1f) < thr);
      const uint32_t fl = __ballot_sync(0xffffffffu, flag);
      if (lane == 0) flagw_s[w] = fl;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      uint32_t fw[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) fw[i] = flagw_s[i];
      const int nflag = __popc(fw[0]) + __popc(fw[1]) + __popc(fw[2]) + __popc(fw[3]);
      if (nflag != 0) {
        // ---- deferred rows (identical flags in both CTAs): entry seg_cnt + (rank of the column among the step's flagged
        // columns), written by the row's owner.  Candidates = every cluster whose approximate distance may be within thr of
        // the best, as a superset read off the 8 partials: a 32-cluster group whose best key is above best + thr has none,
        // one whose second key is above it has exactly its best, otherwise the whole group is tested. ----
        if (flag && (uint32_t)(col >> 6) == rank) {
          int pos = __popc(fl & ((1u << lane) - 1u));
#pragma unroll
          for (int q2 = 0; q2 < 3; ++q2)
            if (q2 < w) pos += __popc(fw[q2]);
          const int e = seg_cnt + pos;
          seg_list[e] = make_int2((int)grow, -1);
          if (e < args.mask_cap) {
            const float T = M1f + thr;
            uint32_t mk[8];
#pragma unroll
            for (int s8 = 0; s8 < 8; ++s8) {
              const bool any = __uint_as_float(pp[s8].x & 0xffffff00u) <= T;
              const bool two = __uint_as_float(pp[s8].y & 0xffffff00u) <= T;
              mk[s8] = any ? (two ? 0xffffffffu : (1u << (pp[s8].x & 31u))) : 0u;
            }
            uint4* dst = reinterpret_cast<uint4*>(seg_mask + (size_t)e * 8u);
            dst[0] = make_uint4(mk[0], mk[1], mk[2], mk[3]);
            dst[1] = make_uint4(mk[4], mk[5], mk[6], mk[7]);
          }
          ++n_flag;
        }
        seg_cnt += nflag;
      }
      if (flag) label = -1;
      // ---- publish the labels: the update warps find their rows themselves (invalid and deferred rows: -1) ----
      lab_s[b * TN + col] = valid ? label : -1;
      if (valid && label >= 0 && (uint32_t)(col >> 6) == rank && args.labels_out != nullptr) args.labels_out[grow] = label;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (threadIdx.x == 0) mbar_arrive(bar(B_LFULL + b));
    }
    if (threadIdx.x == 0 && rank == 0) args.fix_count[pairid] = seg_cnt;
    if (args.rstat != nullptr) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) n_flag += __shfl_xor_sync(0xffffffffu, n_flag, o);
      if (lane == 0 && n_flag != 0ull) atomicAdd(args.rstat + 0, n_flag);
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) {
    double c = 0.0;
    for (int i = 0; i < 16; ++i) c += cost_s[i];
    args.cost_partials[blockIdx.x] = c;
  }
  cluster_sync_all();   // the peer may still receive multicast commits / remote arrivals / DSMEM reads
  if (warp == W_MMA) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// fix-up of the deferred rows
// ------------------------------------------------------------------------------------------------
struct FixArgs {
  const float* X;
  int64_t n;
  int d, k;
  const float* C32;            // [k][d]
  const float* cnorm;          // [256] ||c||^2 (fp32 centres)
  int2* list;
  const uint32_t* masks;
  const int32_t* count;
  int npairs, seg_cap, mask_cap;
  int32_t* labels_out;         // or NULL
  float* mind_out;             // or NULL
  int need_cost;
  double* cost_out;            // [gridDim.x] (always written)
  unsigned long long* rstat;   // or NULL
  float* partial;              // k_fix_accum_t: the extra slot's [k][d] sums
  int32_t* counts_out;         // and its [k] counts
  const B2kLoopState* st;
  B2kLoopState* st_w;          // same object: k_fix_accum_t publishes the cumulative fix-up counters to the host's poll
};
constexpr int FIX_WARPS = 8;
constexpr int FIX_MAXP = 256;

// One warp per deferred row: exact argmin over the row's candidates.  d(j) = ||c_j||^2 - 2 x.c_j with the dot product as
// one fp32 FMA chain per lane (columns lane*4 + 128 i) and a fixed 5-level shuffle tree; candidates in ascending
// cluster order with strict '<' (lowest index wins ties).  Entries beyond the mask capacity test every cluster.
__global__ void __launch_bounds__(FIX_WARPS * 32) k_fix_labels_t(const FixArgs f) {
  if (f.st != nullptr && f.st->done) return;
  __shared__ int pre[FIX_MAXP + 1];
  __shared__ double cost_w[FIX_WARPS];
  if (threadIdx.x == 0) {
    int a = 0;
    for (int p = 0; p < f.npairs; ++p) {
      pre[p] = a;
      a += f.count[p];
    }
    pre[f.npairs] = a;
  }
  __syncthreads();
  const int M = pre[f.npairs];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double cost = 0.0;
  unsigned long long ncand = 0;
  for (int i = (int)blockIdx.x * FIX_WARPS + warp; i < M; i += (int)gridDim.x * FIX_WARPS) {
    int p = 0;   // segment of entry i = the number of segments that end at or before i (ends are non-decreasing)
    for (int b0 = 0; b0 < f.npairs; b0 += 32) {
      const int q = b0 + lane;
      p += __popc(__ballot_sync(0xffffffffu, q < f.npairs && pre[q + 1] <= i));
    }
    const int e = i - pre[p];
    int2* ent = f.list + (size_t)p * (size_t)f.seg_cap + e;
    const int64_t row = (int64_t)ent->x;
    uint32_t mw = 0xffffffffu;
    if (e < f.mask_cap && lane < 8) mw = f.masks[((size_t)p * (size_t)f.mask_cap + (size_t)e) * 8u + (uint32_t)lane];
    float4 xv[2];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int cc = lane * 4 + 128 * t;
      xv[t] = cc < f.d ? __ldg(reinterpret_cast<const float4*>(f.X + (size_t)row * f.d + cc)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float best = __int_as_float(0x7f800000);
    int bj = -1;
    for (int pass = 0; pass < 2 && bj < 0; ++pass) {   // pass 1 (every cluster) only if the mask held no valid candidate
      int wi = -1;
      uint32_t bm = 0;
      auto next_cand = [&]() -> int {   // ascending cluster order, -1 at the end (warp-uniform)
        for (;;) {
          while (bm == 0u && wi < 7) {
            ++wi;
            bm = pass == 0 ? __shfl_sync(0xffffffffu, mw, wi) : 0xffffffffu;
          }
          if (bm == 0u) return -1;
          const int j = wi * 32 + (__ffs(bm) - 1);
          bm &= bm - 1;
          if (j < f.k) return j;
          bm = 0u;   // clusters are ascending: nothing valid is left in this word
        }
      };
      for (;;) {   // two candidates per trip: both centre rows' loads are in flight together
        const int ja = next_cand();
        if (ja < 0) break;
        const int jb = next_cand();
        const int jb2 = jb >= 0 ? jb : ja;
        float dota = 0.f, dotb = 0.f;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const int cc = lane * 4 + 128 * t;
          if (cc < f.d) {
            const float4 ca = __ldg(reinterpret_cast<const float4*>(f.C32 + (size_t)ja * f.d + cc));
            const float4 cb = __ldg(reinterpret_cast<const float4*>(f.C32 + (size_t)jb2 * f.d + cc));
            dota = fmaf(xv[t].x, ca.x, fmaf(xv[t].y, ca.y, fmaf(xv[t].z, ca.z, fmaf(xv[t].w, ca.w, dota))));
            dotb = fmaf(xv[t].x, cb.x, fmaf(xv[t].y, cb.y, fmaf(xv[t].z, cb.z, fmaf(xv[t].w, cb.w, dotb))));
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          dota += __shfl_xor_sync(0xffffffffu, dota, o);
          dotb += __shfl_xor_sync(0xffffffffu, dotb, o);
        }
        const float da = fmaf(-2.f, dota, f.cnorm[ja]);
        if (da < best) { best = da; bj = ja; }
        ++ncand;
        if (jb >= 0) {
          const float db = fmaf(-2.f, dotb, f.cnorm[jb]);
          if (db < best) { best = db; bj = jb; }
          ++ncand;
        }
      }
    }
    if (lane == 0) {
      ent->y = bj;
      if (f.labels_out != nullptr) f.labels_out[row] = bj;
    }
    if (f.need_cost) {   // exact min distance sum (x - c)^2, as the update role computes it for the other rows
      float s2 = 0.f;
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int cc = lane * 4 + 128 * t;
        if (cc < f.d) {
          const float4 cv = __ldg(reinterpret_cast<const float4*>(f.C32 + (size_t)bj * f.d + cc));
          const float dx = xv[t].x - cv.x, dy = xv[t].y - cv.y, dz = xv[t].z - cv.z, dw = xv[t].w - cv.w;
          s2 = fmaf(dx, dx, fmaf(dy, dy, fmaf(dz, dz, fmaf(dw, dw, s2))));
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      if (lane == 0) {
        if (f.mind_out != nullptr) f.mind_out[row] = s2;
        cost += (double)s2;
      }
    }
  }
  if (lane == 0) cost_w[warp] = cost;
  __syncthreads();
  if (threadIdx.x == 0) {
    double c = 0.0;
    for (int w2 = 0; w2 < FIX_WARPS; ++w2) c += cost_w[w2];
    f.cost_out[blockIdx.x] = c;
  }
  if (f.rstat != nullptr && lane == 0 && ncand != 0ull) atomicAdd(f.rstat + 1, ncand);
}

// One CTA per cluster, thread = column: scans the segments in order, compacts the rows labelled with its cluster into
// shared memory (list order) and adds them with eight row loads in flight — the order of the additions is a fixed
// function of the data (segments in pair order, entries in step order), hence deterministic.
constexpr int ACC_CH = 1024;   // entries per scan step (4 per thread)
constexpr int FIX_SLOTS = 4;   // partial-sum slots of the deferred rows: slot q takes the segments p = q (mod 4)
__global__ void __launch_bounds__(256) k_fix_accum_t(const FixArgs f) {
  if (f.st != nullptr && f.st->done) return;
  __shared__ int buf[ACC_CH];
  __shared__ int wsum[8];
  const int j = (int)blockIdx.x;
  const int slot = (int)blockIdx.y;
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float acc = 0.f;
  int cnt = 0;
  for (int p = slot; p < f.npairs; p += FIX_SLOTS) {
    const int c = f.count[p];
    const int2* seg = f.list + (size_t)p * (size_t)f.seg_cap;
    for (int e0 = 0; e0 < c; e0 += ACC_CH) {
      const int eb = e0 + tid * 4;
      int2 en[4];
      if (eb + 3 < c) {   // 32 contiguous bytes (segment bases are 256-byte aligned)
        const int4 a0 = *reinterpret_cast<const int4*>(seg + eb);
        const int4 a1 = *reinterpret_cast<const int4*>(seg + eb + 2);
        en[0] = make_int2(a0.x, a0.y);
        en[1] = make_int2(a0.z, a0.w);
        en[2] = make_int2(a1.x, a1.y);
        en[3] = make_int2(a1.z, a1.w);
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) en[q] = eb + q < c ? seg[eb + q] : make_int2(-1, -1);
      }
      int mine = 0;
#pragma unroll
      for (int q = 0; q < 4; ++q) mine += en[q].y == j ? 1 : 0;
      int incl = mine;   // inclusive scan over the warp, then over the 8 warps
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      if (lane == 31) wsum[warp] = incl;
      __syncthreads();
      int off = incl - mine, total = 0;
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) {
        const int v = wsum[w8];
        if (w8 < warp) off += v;
        total += v;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (en[q].y == j) buf[off++] = en[q].x;
      __syncthreads();
      if (tid < f.d) {
        const float* xc = f.X + tid;
        for (int q = 0; q < total; q += 16) {
          float v[16];
#pragma unroll
          for (int u = 0; u < 16; ++u) v[u] = q + u < total ? __ldg(xc + (size_t)buf[q + u] * f.d) : 0.f;
#pragma unroll
          for (int u = 0; u < 16; ++u) acc += v[u];
        }
      }
      cnt += total;
      __syncthreads();
    }
  }
  if (tid < f.d) f.partial[((size_t)slot * f.k + j) * f.d + tid] = acc;
  if (tid == 0) f.counts_out[(size_t)slot * f.k + j] = cnt;
  if (tid == 0 && j == 0 && slot == 0 && f.st_w != nullptr && f.rstat != nullptr) {
    f.st_w->fix_rows_cum = f.rstat[0];    // complete: the main kernel and k_fix_labels_t have finished
    f.st_w->fix_cands_cum = f.rstat[1];
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
void t_layout(B2kFusedPlan* p, int64_t n, int k, int d, Arena& A) {
  p->ct = A.take<float>((size_t)256 * p->choice.DP, 1024);
  p->cnorm = A.take<float>(512);
  p->thr = A.take<float>(4);
  p->keytab = A.take<uint8_t>(512);
  p->rstat = A.take<unsigned long long>(2);
  p->partials = A.take<float>((size_t)p->P * k * d);
  p->counts = A.take<int32_t>((size_t)p->P * k);
  p->cost_partials = A.take<double>(p->Pc);
  p->xnorm = A.take<float2>(n > 0 ? n : 1);
  // deferred-row segments: a pair can defer every row it sees; candidate masks for the first 1/4 of a segment (entries
  // beyond that are decided against every cluster)
  const int npairs = p->grid / 2;
  const int64_t nsteps = (n + TN - 1) / TN;
  const int64_t nit_max = (nsteps + npairs - 1) / npairs;
  p->seg_cap = (int)(nit_max * TN);
  p->mask_cap = (int)std::min<int64_t>(p->seg_cap, ((nit_max + 3) / 4) * TN);
  p->fix_list = A.take<int2>((size_t)npairs * p->seg_cap);
  p->fix_masks = A.take<uint32_t>((size_t)npairs * p->mask_cap * 8);
  p->fix_count = A.take<int32_t>(npairs);
}

template <int NCH, bool UPD>
int launch_t(b2k_ctx* ctx, int grid, const CUtensorMap& mx, const TArgs& a, cudaStream_t s) {
  auto kern = k_fused_t<NCH, UPD>;
  B2K_CUDA_OK(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  B2K_TRY(b2k_launch_pair(ctx, kern, grid, NTHREADS, SMEM_BYTES, s, mx, a));
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}
}  // namespace

int b2k_fused_t_plan(b2k_ctx* ctx, int64_t n, int d, int k, Arena& A, B2kFusedPlan* plan) {
  const int64_t nsteps = (n + TN - 1) / TN;
  int grid = ctx->sm_count & ~1;
  if (nsteps * 2 < grid) grid = (int)nsteps * 2;
  if (grid < 2) grid = 2;
  plan->grid = grid;
  plan->P = grid / 2 + FIX_SLOTS;             // one slot per CTA pair + the deferred rows' slots (k_fix_accum_t)
  plan->Pc = grid + 8 * ctx->sm_count;        // cost partials: one per CTA + one per k_fix_labels_t CTA
  t_layout(plan, n, k, d, A);
  return B2K_OK;
}

// once per fit / lloyd / assign call: row norms of X into the plan scratch (or, with the fit's norm scope, once per fit
// into the context's cache); clears the recheck counters
int b2k_fused_t_prepare(b2k_ctx* ctx, B2kFusedPlan& plan, const float* X, int64_t n, int d, B2kNormScope* norms,
                        cudaStream_t s) {
  B2K_CUDA_OK(ctx, cudaMemsetAsync(plan.rstat, 0, 16, s));
  int blocks = ctx->sm_count * 8;
  if (norms) {
    if (norms->X != X || norms->n != n) return b2k_fail(ctx, B2K_ERR_STATE, "fused_t: norm scope of another matrix");
    if (ctx->xnorm_cache_rows < n) {
      if (ctx->xnorm_cache) cudaFree(ctx->xnorm_cache);
      ctx->xnorm_cache = nullptr;
      ctx->xnorm_cache_rows = 0;
      B2K_CUDA_OK(ctx, cudaMalloc(&ctx->xnorm_cache, (size_t)n * sizeof(float2)));
      ctx->xnorm_cache_rows = n;
      norms->valid = false;
    }
    plan.xnorm = static_cast<float2*>(ctx->xnorm_cache);
    if (norms->valid) return B2K_OK;
    norms->valid = true;
  }
  k_row_norms<<<blocks, 256, 0, s>>>(X, n, d, plan.xnorm);
  ctx->stats.kernel_launches++;
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

int b2k_launch_fused_t(b2k_ctx* ctx, const B2kFusedPlan& plan, const float* X, int64_t n, int d, const float* C, int k,
                       int32_t* labels_out, float* mindist_out, bool do_update, bool need_cost, const B2kLoopState* st,
                       cudaStream_t s, const double* prev_counts) {
  float* cnorm = plan.cnorm;
  uint8_t* keytab = plan.keytab;
  const int npairs = plan.grid / 2;

  k_prep_centers_t<<<32, 256, 0, s>>>(C, k, d, plan.choice.DP, plan.ct, cnorm, st);
  k_tables_t<<<1, 256, 0, s>>>(do_update ? prev_counts : nullptr, k, cnorm, keytab, keytab + 256, plan.thr, st);
  ctx->stats.kernel_launches += 2;
  B2K_CUDA_OK(ctx, cudaGetLastError());

  CUtensorMap mx;
  B2K_TRY(b2k_encode_2d(ctx, &mx, X, (uint64_t)d, (uint64_t)n, (uint64_t)d * 4, CHUNK, TNH,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B));

  TArgs a{};
  a.n = n;
  a.nsteps = (int)((n + TN - 1) / TN);
  a.k = k;
  a.d = d;
  a.Ct = plan.ct;
  a.C32 = C;
  a.cnorm = cnorm;
  a.thr = plan.thr;
  a.xnorm = plan.xnorm;
  a.keytab = keytab;
  a.keyinv = keytab + 256;
  a.partials = plan.partials;
  a.counts = plan.counts;
  a.cost_partials = plan.cost_partials;
  a.labels_out = labels_out;
  a.mind_out = mindist_out;
  a.need_cost = need_cost ? 1 : 0;
  a.rstat = plan.rstat;
  a.fix_list = plan.fix_list;
  a.fix_masks = plan.fix_masks;
  a.fix_count = plan.fix_count;
  a.seg_cap = plan.seg_cap;
  a.mask_cap = plan.mask_cap;
  a.st = st;
  if (npairs > FIX_MAXP) return b2k_fail(ctx, B2K_ERR_STATE, "fused_t: more CTA pairs than the fix-up kernels index");

  int rc;
  if (plan.choice.DP == 128) rc = do_update ? launch_t<4, true>(ctx, plan.grid, mx, a, s) : launch_t<4, false>(ctx, plan.grid, mx, a, s);
  else rc = do_update ? launch_t<8, true>(ctx, plan.grid, mx, a, s) : launch_t<8, false>(ctx, plan.grid, mx, a, s);
  B2K_TRY(rc);
  ctx->stats.kernel_launches++;
  ctx->stats.fused_tc_launches++;

  // the deferred rows: exact labels (+ min distance / cost), then their contribution to the sums (the last FIX_SLOTS slots)
  FixArgs f{};
  f.X = X;
  f.n = n;
  f.d = d;
  f.k = k;
  f.C32 = C;
  f.cnorm = cnorm;
  f.list = a.fix_list;
  f.masks = a.fix_masks;
  f.count = a.fix_count;
  f.npairs = npairs;
  f.seg_cap = plan.seg_cap;
  f.mask_cap = plan.mask_cap;
  f.labels_out = labels_out;
  f.mind_out = mindist_out;
  f.need_cost = need_cost ? 1 : 0;
  f.cost_out = a.cost_partials + plan.grid;
  f.rstat = a.rstat;
  f.partial = a.partials + (size_t)(plan.P - FIX_SLOTS) * k * d;
  f.counts_out = a.counts + (size_t)(plan.P - FIX_SLOTS) * k;
  f.st = st;
  f.st_w = const_cast<B2kLoopState*>(st);
  k_fix_labels_t<<<plan.Pc - plan.grid, FIX_WARPS * 32, 0, s>>>(f);
  ctx->stats.kernel_launches++;
  if (do_update) {
    k_fix_accum_t<<<dim3((unsigned)k, FIX_SLOTS), 256, 0, s>>>(f);
    ctx->stats.kernel_launches++;
  }
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}
