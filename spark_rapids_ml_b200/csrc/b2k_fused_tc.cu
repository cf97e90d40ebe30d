// Fused assign + per-cluster partial-sum kernel for sm_100a: ONE pass over X per Lloyd iteration.
//
//   TMA (cp.async.bulk.tensor, 128B swizzle)  : X row tiles [128 x 32 f32] HBM -> smem ring (12 slots = 3 tiles)
//   convert warps (4)                          : smem -> split x = hi + lo (both RN to tf32, packed fp32x2 ops)
//                                                 -> TMEM (tcgen05.st)
//   MMA warp (1 thread issues)                 : D[128 x KP] (TMEM, fp32) = hi.Chi^T + lo.Chi^T + hi.Clo^T
//                                                 tcgen05.mma kind::tf32, A from TMEM, B (centers) from smem
//                                                 => "3xTF32": fp32-accurate x.c without an fp32 tensor mode
//   epilogue warps (4)                         : tcgen05.ld D -> dist_j = ||c_j||^2 - 2 x.c_j -> argmin
//                                                 (lowest index on ties) -> labels, min distance, cost
//                                                 + deterministic counting sort of the tile's rows by cluster
//   update warps (16)                          : re-read the SAME smem tile in sorted order, accumulate per-cluster
//                                                 sums in REGISTERS (warp u owns KP/16 clusters dealt by size; lane
//                                                 owns 4 columns): no atomics, deterministic; flushed once per CTA
//
// The step is a latency ring (TMA -> convert -> MMA -> argmin/sort -> update -> slot release) and is sensitive to
// instruction fetch: keep the hot loops rolled and diagnostics out of the product build (DESIGN.md 4.1).
//
// Persistent: one CTA per SM, static round-robin over row tiles (deterministic partial sums).
// What it replaces: cuML's fusedL2NN (minClusterAndDistanceCompute) + reduce_rows_by_key second pass over X,
// reached from spark_rapids_ml/clustering.py:412-415 (SURVEY.md §2a, §8a a-6/a-7).
//
// Algorithmic HBM bytes per launch: 4*n*d (X once) [+ 4*n labels / 4*n mindist when requested]
// + 148 * (k*d + k) * 4 partials (negligible).  See DESIGN.md "Kernels".
#include <float.h>
#include <stdio.h>

#include <type_traits>

#include "b2k_internal.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// configuration
// ------------------------------------------------------------------------------------------------
constexpr int TM = 128;            // rows per tile (UMMA M)
constexpr int CHUNK = 32;          // f32 per 128-byte swizzle row = one TMA box / K chunk
constexpr int SLOT_BYTES = TM * CHUNK * 4;  // 16 KB
constexpr int NA = 4;              // TMEM A-operand ring slots (hi 32 cols + lo 32 cols each)
constexpr int A_COLS = 64;
constexpr int D_OFF = NA * A_COLS; // 256
constexpr int TMEM_COLS = 512;

constexpr int W_CONVERT0 = 0;      // warps 0-3  (lane quadrant = warp % 4)
constexpr int W_EPI0 = 4;          // warps 4-7
constexpr int W_UPD0 = 8;          // warps 8-23: 16 update warps
constexpr int N_UPD = 16;
constexpr int W_TMA = W_UPD0 + N_UPD;   // 24
constexpr int W_MMA = W_TMA + 1;        // 25
constexpr int NWARPS = 26;              // 832 threads -> 72 registers per thread
constexpr int NTHREADS = NWARPS * 32;

constexpr size_t SMEM_LIMIT = 227 * 1024;
// Counting-sort scratch (epilogue -> update hand-off), sized by KP so that the (64, 128, PAIR) instantiation fits a
// 12th ring slot (every byte counts there: see Cfg):
//   CNT     per-warp key histograms, parity buffered: u8 [2][4][KP]
//   ROWS    sorted row list, double buffered: u16 [2][128]; an entry is the row's byte offset inside a ring slot with
//           its swizzle phase folded in: row * 128 + ((row & 7) << 4)
//   START   exclusive start offset per sort key, double buffered: u8 [2][SP], SP = KP + 1 rounded up to 16
//   KEYTAB  u8 [KP]      KEYINV  u8 [KP]
template <int KP>
struct SortLayout {
  static constexpr int SP = (KP + 16) & ~15;
  static constexpr int CNT = 0;
  static constexpr int ROWS = 8 * KP;
  static constexpr int START = ROWS + 512;
  static constexpr int KEYTAB = START + 2 * SP;
  static constexpr int KEYINV = KEYTAB + KP;
  static constexpr int BYTES = KEYINV + KP;
};

template <int KP, int DP, bool PAIR = false>
struct Cfg {
  // PAIR: two CTAs of a cluster issue ONE tcgen05.mma.cta_group::2 (M = 256 = 2 x 128 rows, one row tile per
  // CTA); each CTA keeps only HALF of the centre rows in shared memory (the pair supplies B jointly), which
  // frees KP*DP*4 bytes per CTA for two more ring slots and halves the B-operand shared-memory reads.
  static constexpr int KPS = PAIR ? KP / 2 : KP;               // centre rows resident in this CTA's smem
  static_assert(KP % 16 == 0 && KP >= 16 && KP <= 128, "KP");
  static_assert(DP % CHUNK == 0 && DP >= CHUNK && DP <= 256, "DP");
  static constexpr int NCH = DP / CHUNK;
  static constexpr int C_BYTES = KPS * DP * 4;                 // one of Chi / Clo (this CTA's share)
  using SL = SortLayout<KP>;
  static constexpr int BAR_BYTES = 384;                        // up to 48 mbarriers
  // The dynamic shared memory base is required to be 1 KB aligned (checked at kernel entry; it is: the kernel has no
  // static shared memory), so there is no alignment slack.
  static constexpr int MISC = 1024 /*xnorm*/ + KP * 4 + BAR_BYTES + 64 + SL::BYTES;
  static constexpr int NSLOT_RAW = (int)((SMEM_LIMIT - 2 * C_BYTES - MISC) / SLOT_BYTES);
  static constexpr int NSLOT = NSLOT_RAW > 13 ? 13 : NSLOT_RAW;   // ring depth capped at 13 slots
  static_assert(NSLOT >= NCH + 1, "ring too small");
  static constexpr int OFF_RING = 0;
  static constexpr int OFF_CHI = NSLOT * SLOT_BYTES;
  static constexpr int OFF_CLO = OFF_CHI + C_BYTES;
  static constexpr int OFF_CNORM = OFF_CLO + C_BYTES;
  static constexpr int OFF_XNORM = OFF_CNORM + KP * 4;
  static constexpr int OFF_BARS = OFF_XNORM + 1024;
  // barrier indices (8 bytes each)
  static constexpr int B_XFULL = 0;
  static constexpr int B_XEMPTY = B_XFULL + NSLOT;
  static constexpr int B_AFULL = B_XEMPTY + NSLOT;
  static constexpr int B_AEMPTY = B_AFULL + NA;
  static constexpr int B_DFULL = B_AEMPTY + NA;
  static constexpr int B_DEMPTY = B_DFULL + 2;
  static constexpr int B_LFULL = B_DEMPTY + 2;
  static constexpr int B_LEMPTY = B_LFULL + 2;
  static constexpr int B_NFULL = B_LEMPTY + 2;
  static constexpr int B_NEMPTY = B_NFULL + 2;
  static constexpr int B_CFULL = B_NEMPTY + 2;
  static constexpr int NBARS = B_CFULL + 1;
  static_assert(NBARS * 8 <= BAR_BYTES, "barrier area");
  static constexpr int OFF_TMEMPTR = OFF_BARS + BAR_BYTES;
  static constexpr int OFF_SORT = OFF_TMEMPTR + 64;            // counting-sort scratch (epilogue -> update)
  static constexpr int SMEM_BYTES = OFF_SORT + SL::BYTES;
  static_assert(SMEM_BYTES <= (int)SMEM_LIMIT, "smem");
  static constexpr int UPL = (DP / 4 + 31) / 32;   // float4 units per lane in the update warps
  static constexpr int CPW = (KP + N_UPD - 1) / N_UPD;  // clusters per update warp
  static constexpr int KPL = (KP + 31) / 32;            // sort keys per lane in the epilogue scan
  static_assert(KP % N_UPD == 0, "KP must be a multiple of the update warp count");
};

static_assert(Cfg<64, 128, true>::NSLOT == 12, "the flagship instantiation is laid out for a 12-slot (3-tile) ring");

#include "b2k_ptx.cuh"


// ------------------------------------------------------------------------------------------------
// prep: padded hi/lo split of the centers + ||c||^2
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_prep_centers_tc(const float* __restrict__ C, int k, int d, int KP, int DP,
                                                         float* __restrict__ Chi, float* __restrict__ Clo,
                                                         float* __restrict__ cnorm, const B2kLoopState* st) {
  if (st != nullptr && st->done) return;
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (warp >= KP) return;
  double s = 0.0;
  for (int t = lane; t < DP; t += 32) {
    float v = (warp < k && t < d) ? C[(size_t)warp * d + t] : 0.f;
    uint32_t hb = rn_tf32_bits(v);
    float hi = __uint_as_float(hb);
    float lo = v - hi;
    Chi[(size_t)warp * DP + t] = hi;
    Clo[(size_t)warp * DP + t] = __uint_as_float(rn_tf32_bits(lo));
    s += (double)v * (double)v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) cnorm[warp] = warp < k ? (float)s : __int_as_float(0x7f800000);
}

// ------------------------------------------------------------------------------------------------
// cluster -> (update warp, accumulator slot) table.  The update stage is gated by its most loaded warp, so the
// clusters are dealt to the N_UPD update warps by size (descending, snake order: a deterministic LPT-style packing
// with exactly KP/N_UPD slots per warp).  Sizes = the previous iteration's cluster counts (any positive scaling);
// without them (first pass) the mapping is the identity j -> (j % N_UPD, j / N_UPD).
//   keytab[j]  = owner_warp * CPW + slot        inv[key] = j
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_balance_table(const double* __restrict__ counts, int k, int KP,
                                                       uint8_t* __restrict__ keytab, uint8_t* __restrict__ inv,
                                                       const B2kLoopState* st) {
  if (st != nullptr && st->done) return;
  __shared__ double w[128];
  const int j = threadIdx.x;
  const int CPW = KP / N_UPD;
  if (j < KP) w[j] = (counts != nullptr && j < k) ? counts[j] : -1.0 - (double)0;   // padding clusters sort last
  __syncthreads();
  if (j >= KP) return;
  int key;
  if (counts == nullptr) {
    key = (j % N_UPD) * CPW + j / N_UPD;
  } else {
    int rank = 0;   // position in (count desc, index asc) order
    for (int i = 0; i < KP; ++i) rank += (w[i] > w[j]) || (w[i] == w[j] && i < j);
    const int round = rank / N_UPD, pos = rank % N_UPD;
    const int owner = (round & 1) ? (N_UPD - 1 - pos) : pos;
    key = owner * CPW + round;
  }
  keytab[j] = (uint8_t)key;
  inv[key] = (uint8_t)j;
}

// ------------------------------------------------------------------------------------------------
// the fused kernel
// ------------------------------------------------------------------------------------------------
struct FusedArgs {
  int64_t n;
  int ntiles;
  int k;
  int d;
  const float* cnorm;      // [KP]
  const uint8_t* keytab;   // [KP] cluster -> sort key (owner update warp * CPW + slot)
  const uint8_t* keyinv;   // [KP] sort key -> cluster
  float* partials;         // [grid][k*d]
  int32_t* counts;         // [grid][k]
  double* cost_partials;   // [grid]
  int32_t* labels_out;     // [n] or NULL
  float* mind_out;         // [n] or NULL
  int do_update;
  int need_cost;           // compute ||x||^2, min distance and the cost partial (assign / inertia passes)
  const B2kLoopState* st;
};

// NC: the pass also produces ||x||^2, the min distance and the cost partial (assign / inertia passes); a template
// parameter rather than a run-time flag so that the Lloyd-loop kernel carries none of that code (code size).
template <int KP, int DP, bool PAIR, bool NC>
__global__ void __launch_bounds__(NTHREADS, 1)
k_fused_assign_update(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapChi,
                      const __grid_constant__ CUtensorMap mapClo, const FusedArgs args) {
  using G = Cfg<KP, DP, PAIR>;
  if (args.st != nullptr && args.st->done) return;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = smem_u32(smem_raw);
  uint8_t* gbase = smem_raw;
  if ((base & 1023u) != 0u) {   // 128B-swizzle atoms (TMA boxes, UMMA descriptors) need 1 KB alignment
    if (threadIdx.x == 0) printf("b2k fused: dynamic shared memory base %u is not 1 KB aligned\n", base);
    __trap();
  }
  const uint32_t ring = base + G::OFF_RING;
  const uint32_t chi_s = base + G::OFF_CHI;
  const uint32_t clo_s = base + G::OFF_CLO;
  float* cnorm_s = reinterpret_cast<float*>(gbase + G::OFF_CNORM);
  float* xnorm_s = reinterpret_cast<float*>(gbase + G::OFF_XNORM);   // [2][128]
  const uint32_t bars = base + G::OFF_BARS;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(gbase + G::OFF_TMEMPTR);
  uint8_t* sort_s = gbase + G::OFF_SORT;
  auto bar = [&](int i) -> uint32_t { return bars + 8u * (uint32_t)i; };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr bool need_cost = NC;

  // ---- one-time setup ----
  if (warp == W_TMA && lane == 0) {
    tma_prefetch_desc(&mapX);
    tma_prefetch_desc(&mapChi);
    tma_prefetch_desc(&mapClo);
    for (int i = 0; i < G::NSLOT; ++i) {
      mbar_init(bar(G::B_XFULL + i), 1);
      mbar_init(bar(G::B_XEMPTY + i), 2);                 // convert role + update role
    }
    for (int i = 0; i < NA; ++i) {
      mbar_init(bar(G::B_AFULL + i), PAIR ? 2 : 1);       // PAIR: the convert roles of BOTH CTAs feed the leader
      mbar_init(bar(G::B_AEMPTY + i), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(G::B_DFULL + i), 1);
      mbar_init(bar(G::B_DEMPTY + i), PAIR ? 2 : 1);
      mbar_init(bar(G::B_LFULL + i), 1);
      mbar_init(bar(G::B_LEMPTY + i), 1);
      mbar_init(bar(G::B_NFULL + i), 4);
      mbar_init(bar(G::B_NEMPTY + i), 4);
    }
    mbar_init(bar(G::B_CFULL), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == W_MMA) {
    if constexpr (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_s)),
                   "r"((uint32_t)TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_s)),
                   "r"((uint32_t)TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  for (int j = threadIdx.x; j < KP; j += NTHREADS) cnorm_s[j] = args.cnorm[j];
  using SL = typename G::SL;
  uint8_t* keytab_s = sort_s + SL::KEYTAB;   // [KP]
  uint8_t* keyinv_s = sort_s + SL::KEYINV;   // [KP]
  for (int j = threadIdx.x; j < KP; j += NTHREADS) { keytab_s[j] = args.keytab[j]; keyinv_s[j] = args.keyinv[j]; }
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync_all();   // peer barriers initialised / TMEM allocated before any remote signal
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr_s, 0);   // provably warp-uniform

  // static tile schedule.  PAIR: cluster q handles tile pairs q, q+nclusters, ...; CTA rank r takes tile 2*pair+r
  // (a trailing odd tile leaves the peer an all-out-of-range tile: TMA zero-fills it, every row is invalid).
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const int sched0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int sched_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int sched_n = PAIR ? (args.ntiles + 1) / 2 : args.ntiles;
  const int nit = sched0 < sched_n ? (sched_n - sched0 + sched_step - 1) / sched_step : 0;
  auto tile_of = [&](int it) -> int {
    const int sidx = sched0 + it * sched_step;
    return PAIR ? 2 * sidx + (int)rank : sidx;
  };

  if (warp == W_TMA) {
    // ======================= TMA producer =======================
    if (elect_one()) {
      mbar_expect_tx(bar(G::B_CFULL), 2u * G::C_BYTES);
      for (int c = 0; c < G::NCH; ++c) {   // PAIR: this CTA's half of the centre rows
        tma_load_2d(chi_s + c * (G::KPS * 128), &mapChi, bar(G::B_CFULL), c * CHUNK, (int)rank * G::KPS);
        tma_load_2d(clo_s + c * (G::KPS * 128), &mapClo, bar(G::B_CFULL), c * CHUNK, (int)rank * G::KPS);
      }
    }
    __syncwarp();
    int xs = 0;
    uint32_t xph = 0;
    for (int ti = 0; ti < nit; ++ti) {
      const int tile = tile_of(ti);
#pragma unroll 1
      for (int c = 0; c < G::NCH; ++c) {
        mbar_wait(bar(G::B_XEMPTY + xs), xph ^ 1u);
        if (elect_one()) {
          mbar_expect_tx(bar(G::B_XFULL + xs), SLOT_BYTES);
          tma_load_2d(ring + xs * SLOT_BYTES, &mapX, bar(G::B_XFULL + xs), c * CHUNK, tile * TM);
        }
        __syncwarp();
        if (++xs == G::NSLOT) { xs = 0; xph ^= 1u; }
      }
    }
  } else if (warp == W_MMA) {
    // ======================= MMA issuer =======================
    constexpr uint32_t idesc = make_idesc_tf32(PAIR ? 2 * TM : TM, KP);
    mbar_wait(bar(G::B_CFULL), 0);
    int as = 0;
    uint32_t aph = 0;
    for (int ti = 0; ti < ((PAIR && rank != 0) ? 0 : nit); ++ti) {   // PAIR: only the leader CTA issues
      const int b = ti & 1;
      const uint32_t bph = (uint32_t)(ti >> 1) & 1u;
      // CTA-scope waits, PAIR included: a cluster-scope acquire makes ptxas append CCTL.IVALL (L1 invalidate) to every
      // wait, and what these barriers order is TMEM traffic (tcgen05 fences on both sides)
      mbar_wait(bar(G::B_DEMPTY + b), bph ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + D_OFF + b * KP;
#pragma unroll 1
      for (int c = 0; c < G::NCH; ++c) {
        mbar_wait(bar(G::B_AFULL + as), aph);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_hi = tmem_base + as * A_COLS;
          const uint32_t a_lo = a_hi + CHUNK;
          const uint32_t bhi = chi_s + c * (G::KPS * 128);
          const uint32_t blo = clo_s + c * (G::KPS * 128);
#pragma unroll
          for (int ks = 0; ks < CHUNK / 8; ++ks) {
            const uint64_t dhi = make_kmajor_sw128_desc(bhi + ks * 32);
            const uint64_t dlo = make_kmajor_sw128_desc(blo + ks * 32);
            if constexpr (PAIR) {
              tc_mma_ts_tf32_pair(d_tmem, a_lo + ks * 8, dhi, idesc, (c | ks) != 0 ? 1u : 0u);
              tc_mma_ts_tf32_pair(d_tmem, a_hi + ks * 8, dlo, idesc, 1u);
              tc_mma_ts_tf32_pair(d_tmem, a_hi + ks * 8, dhi, idesc, 1u);
            } else {
              tc_mma_ts_tf32(d_tmem, a_lo + ks * 8, dhi, idesc, (c | ks) != 0 ? 1u : 0u);  // small terms first
              tc_mma_ts_tf32(d_tmem, a_hi + ks * 8, dlo, idesc, 1u);
              tc_mma_ts_tf32(d_tmem, a_hi + ks * 8, dhi, idesc, 1u);
            }
          }
          if constexpr (PAIR) {
            tc_commit_pair(bar(G::B_AEMPTY + as));
            if (c == G::NCH - 1) tc_commit_pair(bar(G::B_DFULL + b));
          } else {
            tc_commit(bar(G::B_AEMPTY + as));
            if (c == G::NCH - 1) tc_commit(bar(G::B_DFULL + b));
          }
        }
        __syncwarp();
        if (++as == NA) { as = 0; aph ^= 1u; }
      }
    }
  } else if (warp < W_EPI0) {
    // ======================= convert warps: smem -> (hi, lo) -> TMEM =======================
    const int q = warp - W_CONVERT0;
    const int r = q * 32 + lane;                       // row within the tile == TMEM lane
    const uint32_t lane_field = (uint32_t)(q * 32) << 16;
    const uint32_t swz = (uint32_t)(r & 7);
    const uint64_t kSplitA = pack2(8193.f, 8193.f), kSplitB = pack2(-8192.f, -8192.f);
    int xs = 0, as = 0;
    uint32_t xph = 0, aph = 0;
    // PAIR: this CTA's centre half must have landed before its first a_full signal reaches the leader
    if constexpr (PAIR) mbar_wait(bar(G::B_CFULL), 0);
    for (int ti = 0; ti < nit; ++ti) {
      const int b = ti & 1;
      const uint32_t bph = (uint32_t)(ti >> 1) & 1u;
      float xn = 0.f;
      // chunks are converted in groups of CG: one tcgen05.wait::st / hardware barrier / signal per group
      constexpr int CG = (G::NCH % 2 == 0) ? 2 : 1;
#pragma unroll 1
      for (int c = 0; c < G::NCH; c += CG) {
        int xs_g[CG], as_g[CG];
        uint32_t xp_g[CG], ap_g[CG];
#pragma unroll
        for (int g = 0; g < CG; ++g) {
          xs_g[g] = xs;
          as_g[g] = as;
          xp_g[g] = xph;
          ap_g[g] = aph ^ 1u;
          if (++xs == G::NSLOT) { xs = 0; xph ^= 1u; }
          if (++as == NA) { as = 0; aph ^= 1u; }
        }
        // The group needs 2*CG barriers (x_full and a_empty per chunk).  Even a completed mbarrier wait costs a few
        // hundred cycles, and one warp polling them in turn put ~1.4 k cycles per tile on the convert role (measured with
        // the event trace): each of the four convert warps polls ONE of them, the hardware barrier joins the results.
        {
          const int p = warp - W_CONVERT0;
          if (p < 2 * CG) {
            const int g = p >> 1;
            if ((p & 1) == 0) mbar_wait(bar(G::B_XFULL + (g == 0 ? xs_g[0] : xs_g[CG - 1])), g == 0 ? xp_g[0] : xp_g[CG - 1]);
            else mbar_wait(bar(G::B_AEMPTY + (g == 0 ? as_g[0] : as_g[CG - 1])), g == 0 ? ap_g[0] : ap_g[CG - 1]);
          }
        }
        asm volatile("bar.sync 6, 128;" ::: "memory");
        tc_fence_after();
        // need_cost is hoisted out of the element loop (two copies of the body): a per-float4 branch costs as
        // much issue bandwidth as a fifth of the split itself
        auto convert_group = [&](auto) {
#pragma unroll 1   // code size (instruction fetch)
        for (int g = 0; g < CG; ++g) {
          const int xsg = (g == 0) ? xs_g[0] : xs_g[CG - 1], asg = (g == 0) ? as_g[0] : as_g[CG - 1];
          const uint32_t rowaddr = ring + xsg * SLOT_BYTES + (uint32_t)r * 128u;
          const uint32_t a_addr = tmem_base + lane_field + (uint32_t)(asg * A_COLS);
          // halves of 16 columns: bounds the live registers (the CTA runs 26 warps at 72 registers/thread)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int j2 = 0; j2 < 4; ++j2) {
              const int j = h * 4 + j2;
              float4 v = lds128(rowaddr + (((uint32_t)j ^ swz) << 4));
              float e[4] = {v.x, v.y, v.z, v.w};
              // Veltkamp split with packed fp32 pairs: t = fl(8193 x); hi = t - 8192 x (one FFMA2, exact) is x rounded
              // to nearest at 11 significant bits = a tf32 value (the tensor core's truncation is then a no-op);
              // l = x - hi is exact.  lo = RN_tf32(l) through the +1/2 ulp word trick (hardware truncates).
              // 2.5 issue slots per element instead of 4 for the unpacked form.
#pragma unroll
              for (int t = 0; t < 4; t += 2) {
                const uint64_t x2 = pack2(e[t], e[t + 1]);
                const uint64_t t2 = mul2(x2, kSplitA);
                const uint64_t h2 = fma2(x2, kSplitB, t2);
                const uint64_t l2 = sub2(x2, h2);
                float h0, h1, l0, l1;
                unpack2(h2, h0, h1);
                unpack2(l2, l0, l1);
                hi[j2 * 4 + t] = __float_as_uint(h0);
                hi[j2 * 4 + t + 1] = __float_as_uint(h1);
                lo[j2 * 4 + t] = __float_as_uint(l0) + 0x1000u;
                lo[j2 * 4 + t + 1] = __float_as_uint(l1) + 0x1000u;
                if constexpr (NC) xn = fmaf(e[t + 1], e[t + 1], fmaf(e[t], e[t], xn));
              }
            }
            tmem_st_x16(a_addr + h * 16, hi);
            tmem_st_x16(a_addr + CHUNK + h * 16, lo);
          }
        }
        };
        convert_group(std::integral_constant<bool, NC>{});
        tmem_wait_st();
        tc_fence_before();
        asm volatile("bar.sync 3, 128;" ::: "memory");   // the 4 convert warps (hardware barrier: no polling)
        if (warp == W_CONVERT0 && lane == 0) {            // one arrival per role keeps the waiters' wake-ups low
#pragma unroll
          for (int g = 0; g < CG; ++g) {
            if constexpr (PAIR) mbar_arrive_cluster(bar(G::B_AFULL + as_g[g]), 0u);
            else mbar_arrive(bar(G::B_AFULL + as_g[g]));
            mbar_arrive(bar(G::B_XEMPTY + xs_g[g]));
          }
        }
      }
      if (need_cost) {
        mbar_wait(bar(G::B_NEMPTY + b), bph ^ 1u);
        xnorm_s[b * TM + r] = xn;
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(G::B_NFULL + b));
      }
    }
  } else if (warp < W_UPD0) {
    // ======================= epilogue warps: TMEM D -> argmin =======================
    const int q = warp - W_EPI0;
    const int r = q * 32 + lane;
    const uint32_t lane_field = (uint32_t)(q * 32) << 16;
    double cost = 0.0;
    for (int ti = 0; ti < nit; ++ti) {
      const int tile = tile_of(ti);
      const int b = ti & 1;
      const uint32_t bph = (uint32_t)(ti >> 1) & 1u;
      if (warp == W_EPI0) mbar_wait(bar(G::B_DFULL + b), bph);
      asm volatile("bar.sync 5, 128;" ::: "memory");
      tc_fence_after();
      float best = __int_as_float(0x7f800000);
      int bj = 0;
      // argmin over j in index order with strict '<' (lowest index wins ties).  Four independent chains of 8
      // consecutive candidates, merged in ascending order, give the same winner with a 12-deep instead of a
      // 32-deep dependent compare/select chain per 32 columns.
#pragma unroll 1   // code size: the kernel is instruction-fetch sensitive (stall_no_inst), see DESIGN.md
      for (int g = 0; g < KP / 32; ++g) {
        uint32_t v[32];
        tmem_ld_x32(tmem_base + lane_field + (uint32_t)(D_OFF + b * KP + g * 32), v);
        tmem_wait_ld();
        float cb[4];
        int ci[4];
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          cb[q4] = __int_as_float(0x7f800000);
          ci[q4] = g * 32 + q4 * 8;
        }
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const int j = q4 * 8 + jj;
            const float dist = fmaf(-2.f, __uint_as_float(v[j]), cnorm_s[g * 32 + j]);
            if (dist < cb[q4]) { cb[q4] = dist; ci[q4] = g * 32 + j; }
          }
        }
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4)
          if (cb[q4] < best) { best = cb[q4]; bj = ci[q4]; }
      }
      if constexpr (KP % 32 != 0) {
        // tail group of 16 columns
        uint32_t v[32];
        constexpr int g = KP / 32;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
              "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
            : "r"(tmem_base + lane_field + (uint32_t)(D_OFF + b * KP + g * 32))
            : "memory");
        tmem_wait_ld();
        float cb[2];
        int ci[2];
#pragma unroll
        for (int q4 = 0; q4 < 2; ++q4) {
          cb[q4] = __int_as_float(0x7f800000);
          ci[q4] = g * 32 + q4 * 8;
        }
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
#pragma unroll
          for (int q4 = 0; q4 < 2; ++q4) {
            const int j = q4 * 8 + jj;
            const float dist = fmaf(-2.f, __uint_as_float(v[j]), cnorm_s[g * 32 + j]);
            if (dist < cb[q4]) { cb[q4] = dist; ci[q4] = g * 32 + j; }
          }
        }
#pragma unroll
        for (int q4 = 0; q4 < 2; ++q4)
          if (cb[q4] < best) { best = cb[q4]; bj = ci[q4]; }
      }
      tc_fence_before();

      const int64_t grow = (int64_t)tile * TM + r;
      const bool valid = grow < args.n;
      // ---- deterministic counting sort of the tile's rows by (owner update warp, owned-cluster slot, row) ----
      // key = keytab[label] (size-balanced, see k_balance_table): update warp u owns the key range [u*CPW, (u+1)*CPW)
      uint8_t* cnt = sort_s + SL::CNT + (ti & 1) * (4 * KP);   // [4 warps][KP] per-warp key histogram (parity buffered)
      uint16_t* rows_sorted = reinterpret_cast<uint16_t*>(sort_s + SL::ROWS) + b * 128;   // [128] rows in key order
      uint8_t* start = sort_s + SL::START + b * SL::SP;    // [KP + 1] exclusive offsets per key
      if (lane < KP / 4) reinterpret_cast<uint32_t*>(cnt + q * KP)[lane] = 0u;
      __syncwarp();
      const int key = valid ? (int)keytab_s[bj] : KP;
      const uint32_t same = __match_any_sync(0xffffffffu, key);
      const int rank = __popc(same & ((1u << lane) - 1u));
      if (valid && rank == 0) cnt[q * KP + key] = (uint8_t)__popc(same);
      asm volatile("bar.sync 1, 128;" ::: "memory");      // the 4 epilogue warps
      if (warp == W_EPI0 && lane == 0) {   // all four have drained D: it may be overwritten by tile ti+2
        if constexpr (PAIR) mbar_arrive_cluster(bar(G::B_DEMPTY + b), 0u);
        else mbar_arrive(bar(G::B_DEMPTY + b));
      }
      int tot[G::KPL];
      int lane_sum = 0;
#pragma unroll
      for (int i = 0; i < G::KPL; ++i) {
        const int kk = lane * G::KPL + i;
        tot[i] = (kk < KP) ? (int)cnt[kk] + (int)cnt[KP + kk] + (int)cnt[2 * KP + kk] + (int)cnt[3 * KP + kk] : 0;
        lane_sum += tot[i];
      }
      int incl = lane_sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      int st[G::KPL];
      st[0] = incl - lane_sum;
#pragma unroll
      for (int i = 1; i < G::KPL; ++i) st[i] = st[i - 1] + tot[i - 1];
      int my_start = 0;
#pragma unroll
      for (int i = 0; i < G::KPL; ++i) {
        const int t = __shfl_sync(0xffffffffu, st[i], (key < KP ? key : 0) / G::KPL);
        if ((key % G::KPL) == i) my_start = t;
      }
      int pos = my_start + rank;
      if (valid) {
#pragma unroll
        for (int q2 = 0; q2 < 3; ++q2)
          if (q2 < q) pos += (int)cnt[q2 * KP + key];
      }
      mbar_wait(bar(G::B_LEMPTY + b), bph ^ 1u);
      if (valid) rows_sorted[pos] = (uint16_t)(r * 128 + ((r & 7) << 4));
      if (q == 0) {
#pragma unroll
        for (int i = 0; i < G::KPL; ++i) {
          const int kk = lane * G::KPL + i;
          if (kk < KP) start[kk] = (uint8_t)st[i];
        }
        if (lane == 31) start[KP] = (uint8_t)incl;
      }
      asm volatile("bar.sync 4, 128;" ::: "memory");      // row list complete
      if (warp == W_EPI0 && lane == 0) mbar_arrive(bar(G::B_LFULL + b));
      // off the critical path: outputs and cost
      if (valid && args.labels_out) args.labels_out[grow] = bj;
      if (need_cost) {
        mbar_wait(bar(G::B_NFULL + b), bph);
        const float xn = xnorm_s[b * TM + r];
        const float md = fmaxf(xn + best, 0.f);
        if (valid) {
          if (args.mind_out) args.mind_out[grow] = md;
          cost += (double)md;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(G::B_NEMPTY + b));
      }
    }
    // per-CTA cost: fixed-order fold (lanes, then the 4 warps through shared memory after the final sync)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cost += __shfl_xor_sync(0xffffffffu, cost, o);
    if (lane == 0) reinterpret_cast<double*>(gbase + G::OFF_TMEMPTR + 16)[q] = cost;
  } else if (warp < W_TMA) {
    // ======================= update warps: per-cluster sums in registers =======================
    const int u = warp - W_UPD0;
    uint64_t acc[G::CPW][G::UPL][2];   // packed fp32 pairs (x,y) (z,w): one FADD2 adds two columns
    int cnt[G::CPW];
#pragma unroll
    for (int c = 0; c < G::CPW; ++c) {
      cnt[c] = 0;
#pragma unroll
      for (int i = 0; i < G::UPL; ++i) acc[c][i][0] = acc[c][i][1] = 0ull;
    }
    // this lane's float4 units of a row: (chunk, 16-B unit inside the 128-B swizzle line) are fixed per lane
    int unit_cc[G::UPL];
    uint32_t unit_js[G::UPL];
#pragma unroll
    for (int i = 0; i < G::UPL; ++i) {
      const int unit = lane + 32 * i;
      unit_cc[i] = unit >> 3;
      unit_js[i] = (uint32_t)(unit & 7) << 4;
    }
    int xs = 0;
    for (int ti = 0; ti < nit; ++ti) {
      const int b = ti & 1;
      const uint32_t bph = (uint32_t)(ti >> 1) & 1u;
      // one warp polls the mbarrier, the other 15 park in a hardware barrier (no issue slots, no wake-ups)
      if (warp == W_UPD0) mbar_wait(bar(G::B_LFULL + b), bph);
      asm volatile("bar.sync 7, 512;" ::: "memory");
      // The x_full phases of this tile's slots completed before the convert warps consumed them, which
      // happens-before the MMA commit, the epilogue and hence this tile's lab_full: no need to poll them again.
      if (args.do_update) {
        const uint16_t* rows_sorted = reinterpret_cast<const uint16_t*>(sort_s + SL::ROWS) + b * 128;
        const uint8_t* start = sort_s + SL::START + b * SL::SP;
        uint32_t unit_base[G::UPL];
#pragma unroll
        for (int i = 0; i < G::UPL; ++i) {
          int s2 = xs + unit_cc[i];
          if (s2 >= G::NSLOT) s2 -= G::NSLOT;
          unit_base[i] = ring + (uint32_t)s2 * SLOT_BYTES;
        }
        // roff = row * 128 + ((row & 7) << 4) (written by the epilogue): address = slot + (roff ^ (unit << 4))
        auto load_row = [&](uint32_t roff, uint64_t (&v)[G::UPL][2]) {
#pragma unroll
          for (int i = 0; i < G::UPL; ++i) {
            if (lane + 32 * i < DP / 4) lds128_2(unit_base[i] + (roff ^ unit_js[i]), v[i][0], v[i][1]);
            else v[i][0] = v[i][1] = 0ull;
          }
        };
        // segment bounds of my CPW owned clusters: start[u*CPW .. u*CPW + CPW]
        const int sv = (lane <= G::CPW) ? (int)start[u * G::CPW + lane] : 0;
#pragma unroll
        for (int c = 0; c < G::CPW; ++c) {
          const int i0 = __shfl_sync(0xffffffffu, sv, c);
          const int i1 = __shfl_sync(0xffffffffu, sv, c + 1);
          cnt[c] += i1 - i0;
#pragma unroll 1   // typical trip count 1-2; ptxas would otherwise unroll it 4x (code size)
          for (int i = i0; i < i1; i += 2) {      // rows of one cluster, ascending row order, two in flight
            const bool two = (i + 1 < i1);
            const uint32_t r0 = rows_sorted[i];
            const uint32_t r1 = rows_sorted[two ? i + 1 : i];
            uint64_t v0[G::UPL][2], v1[G::UPL][2];
            load_row(r0, v0);
            load_row(r1, v1);
#pragma unroll
            for (int k2 = 0; k2 < G::UPL; ++k2) {
              acc[c][k2][0] = add2(acc[c][k2][0], v0[k2][0]);
              acc[c][k2][1] = add2(acc[c][k2][1], v0[k2][1]);
            }
            if (two) {
#pragma unroll
              for (int k2 = 0; k2 < G::UPL; ++k2) {
                acc[c][k2][0] = add2(acc[c][k2][0], v1[k2][0]);
                acc[c][k2][1] = add2(acc[c][k2][1], v1[k2][1]);
              }
            }
          }
        }
      }
      asm volatile("bar.sync 2, 512;" ::: "memory");     // the 16 update warps
      if (warp == W_UPD0 && lane == 0) {
        mbar_arrive(bar(G::B_LEMPTY + b));
        int s2 = xs;
#pragma unroll
        for (int c = 0; c < G::NCH; ++c) {
          mbar_arrive(bar(G::B_XEMPTY + s2));
          if (++s2 == G::NSLOT) s2 = 0;
        }
      }
      xs += G::NCH;
      if (xs >= G::NSLOT) xs -= G::NSLOT;
    }
    // flush: partials[cta][l][col..col+3] for the owned clusters l = keyinv[u*CPW + c]
    if (args.do_update) {
      float* out = args.partials + (size_t)blockIdx.x * args.k * args.d;
#pragma unroll
      for (int c = 0; c < G::CPW; ++c) {
        const int l = (int)keyinv_s[u * G::CPW + c];
        if (l < args.k) {
#pragma unroll
          for (int i = 0; i < G::UPL; ++i) {
            const int col = (lane + 32 * i) * 4;
            float e[4];
            unpack2(acc[c][i][0], e[0], e[1]);
            unpack2(acc[c][i][1], e[2], e[3]);
#pragma unroll
            for (int t = 0; t < 4; ++t)
              if (col + t < args.d) out[(size_t)l * args.d + col + t] = e[t];
          }
          if (lane == 0) args.counts[(size_t)blockIdx.x * args.k + l] = cnt[c];
        }
      }
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) {
    const double* cw = reinterpret_cast<const double*>(gbase + G::OFF_TMEMPTR + 16);
    args.cost_partials[blockIdx.x] = ((cw[0] + cw[1]) + cw[2]) + cw[3];
  }
  if constexpr (PAIR) cluster_sync_all();   // the peer may still receive multicast commits / remote arrivals
  if (warp == W_MMA) {
    tc_fence_after();
    if constexpr (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                   : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_encoder(b2k_ctx* ctx, EncodeTiledFn* fn) {
  if (!ctx->encode_tiled) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p)
      return b2k_fail(ctx, B2K_ERR_CUDA, "cannot resolve cuTensorMapEncodeTiled from the driver");
    ctx->encode_tiled = p;
  }
  *fn = reinterpret_cast<EncodeTiledFn>(ctx->encode_tiled);
  return B2K_OK;
}

}  // namespace

int b2k_encode_2d(b2k_ctx* ctx, CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer,
                  uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer, CUtensorMapL2promotion l2) {
  EncodeTiledFn fn;
  B2K_TRY(get_encoder(ctx, &fn));
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return b2k_fail(ctx, B2K_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
  return B2K_OK;
}

namespace {
// The 3xTF32 instantiations compiled into the library, as <KP, DP>.  b2k_fused_tc_inst searches this list and
// b2k_launch_fused dispatches over it; b2k_tc_pair picks the one that runs on CTA pairs.  There is no <128, 32>:
// d <= 32 with k > 64 runs on the screening kernel (DESIGN.md 4.1).
template <int KP_, int DP_>
struct Inst {
  static constexpr int KP = KP_, DP = DP_;
};
template <typename... I>
struct InstList {};
using Insts = InstList<Inst<16, 32>, Inst<32, 32>, Inst<64, 32>,
                       Inst<16, 64>, Inst<32, 64>, Inst<64, 64>, Inst<128, 64>,
                       Inst<16, 128>, Inst<32, 128>, Inst<64, 128>, Inst<128, 128>>;

template <typename... I>
int smallest_kp(InstList<I...>, int DP, int k) {
  int kp = 0;
  ((I::DP == DP && I::KP >= k && (kp == 0 || I::KP < kp) ? (void)(kp = I::KP) : (void)0), ...);
  return kp;
}

template <int KP, int DP, bool NC>
int launch_inst_nc(b2k_ctx* ctx, int grid, const CUtensorMap& mx, const CUtensorMap& mh, const CUtensorMap& ml,
                const FusedArgs& a, cudaStream_t s) {
  constexpr bool PAIR = b2k_tc_pair(KP, DP);
  using G = Cfg<KP, DP, PAIR>;
  auto kern = k_fused_assign_update<KP, DP, PAIR, NC>;
  B2K_CUDA_OK(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, G::SMEM_BYTES));
  if constexpr (PAIR) B2K_TRY(b2k_launch_pair(ctx, kern, grid, NTHREADS, G::SMEM_BYTES, s, mx, mh, ml, a));
  else kern<<<grid, NTHREADS, G::SMEM_BYTES, s>>>(mx, mh, ml, a);
  B2K_CUDA_OK(ctx, cudaGetLastError());
  return B2K_OK;
}

template <int KP, int DP>
int launch_inst(b2k_ctx* ctx, int grid, const CUtensorMap& mx, const CUtensorMap& mh, const CUtensorMap& ml,
                const FusedArgs& a, cudaStream_t s) {
  return a.need_cost ? launch_inst_nc<KP, DP, true>(ctx, grid, mx, mh, ml, a, s)
                     : launch_inst_nc<KP, DP, false>(ctx, grid, mx, mh, ml, a, s);
}

// launches the listed instantiation <KP, DP>; B2K_ERR_UNSUPPORTED when it is not listed
template <typename... I>
int launch_listed(InstList<I...>, int KP, int DP, b2k_ctx* ctx, int grid, const CUtensorMap& mx,
                  const CUtensorMap& mh, const CUtensorMap& ml, const FusedArgs& a, cudaStream_t s) {
  int rc = B2K_ERR_UNSUPPORTED;
  (void)(((I::KP == KP && I::DP == DP) && (rc = launch_inst<I::KP, I::DP>(ctx, grid, mx, mh, ml, a, s), true)) || ...);
  return rc;
}

void plan_layout(B2kFusedPlan* p, int k, int d, Arena& A) {
  const int KP = p->choice.KP, DP = p->choice.DP;
  p->c_hi = A.take<float>((size_t)KP * DP, 1024);
  p->c_lo = A.take<float>((size_t)KP * DP);
  p->cnorm = A.take<float>(KP);
  p->keytab = A.take<uint8_t>(512);
  p->partials = A.take<float>((size_t)p->grid * k * d);
  p->counts = A.take<int32_t>((size_t)p->grid * k);
  p->cost_partials = A.take<double>(p->grid);
}
}  // namespace

bool b2k_fused_tc_inst(int d, int k, int* KP, int* DP) {
  int dp = (d + CHUNK - 1) / CHUNK * CHUNK;
  if (dp == 96) dp = 128;
  const int kp = smallest_kp(Insts{}, dp, k);
  if (kp == 0) return false;
  *KP = kp;
  *DP = dp;
  return true;
}

int b2k_fused_plan(b2k_ctx* ctx, const B2kChoice& c, int64_t n, int d, int k, Arena& A, B2kFusedPlan* plan) {
  plan->choice = c;
  if (c.variant == 1) return b2k_fused_t_plan(ctx, n, d, k, A, plan);
  int64_t ntiles = (n + TM - 1) / TM;
  int grid = ctx->sm_count;
  if (c.pair) {
    int64_t npairs = (ntiles + 1) / 2;
    grid &= ~1;
    if (npairs * 2 < grid) grid = (int)npairs * 2;
    if (grid < 2) grid = 2;
  } else {
    if (ntiles < grid) grid = (int)ntiles;
    if (grid < 1) grid = 1;
  }
  plan->grid = grid;
  plan->P = grid;
  plan->Pc = grid;
  plan_layout(plan, k, d, A);
  return B2K_OK;
}

int b2k_fused_prepare(b2k_ctx* ctx, B2kFusedPlan& plan, const float* X, int64_t n, int d, B2kNormScope* norms,
                      cudaStream_t s) {
  if (plan.choice.variant == 1) return b2k_fused_t_prepare(ctx, plan, X, n, d, norms, s);
  return B2K_OK;
}

int b2k_fused_recheck_stats(b2k_ctx* ctx, const B2kFusedPlan& plan, unsigned long long out[2], cudaStream_t s) {
  out[0] = out[1] = 0ull;
  if (plan.choice.variant != 1) return B2K_OK;
  B2K_CUDA_OK(ctx, cudaMemcpyAsync(out, plan.rstat, 16, cudaMemcpyDeviceToHost, s));
  B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
  return B2K_OK;
}

int b2k_launch_fused(b2k_ctx* ctx, const B2kFusedPlan& plan, const float* X, int64_t n, int d, const float* C, int k,
                     int32_t* labels_out, float* mindist_out, bool do_update, bool need_cost, const B2kLoopState* st,
                     cudaStream_t s, const double* prev_counts) {
  if (plan.choice.variant == 1)
    return b2k_launch_fused_t(ctx, plan, X, n, d, C, k, labels_out, mindist_out, do_update,
                              !do_update && (mindist_out != nullptr || need_cost), st, s, prev_counts);
  const int KP = plan.choice.KP, DP = plan.choice.DP;
  uint8_t* keytab = plan.keytab;
  k_prep_centers_tc<<<(KP * 32 + 255) / 256, 256, 0, s>>>(C, k, d, KP, DP, plan.c_hi, plan.c_lo, plan.cnorm, st);
  k_balance_table<<<1, 128, 0, s>>>(do_update ? prev_counts : nullptr, k, KP, keytab, keytab + 256, st);
  ctx->stats.kernel_launches += 2;
  B2K_CUDA_OK(ctx, cudaGetLastError());

  CUtensorMap mx, mh, ml;
  B2K_TRY(b2k_encode_2d(ctx, &mx, X, (uint64_t)d, (uint64_t)n, (uint64_t)d * 4, CHUNK, TM,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B));
  const uint32_t cbox = (uint32_t)(plan.choice.pair ? KP / 2 : KP);   // centre rows each CTA keeps in smem
  B2K_TRY(b2k_encode_2d(ctx, &mh, plan.c_hi, (uint64_t)DP, (uint64_t)KP, (uint64_t)DP * 4, CHUNK, cbox,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B));
  B2K_TRY(b2k_encode_2d(ctx, &ml, plan.c_lo, (uint64_t)DP, (uint64_t)KP, (uint64_t)DP * 4, CHUNK, cbox,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B));

  FusedArgs a{};
  a.n = n;
  a.ntiles = (int)((n + TM - 1) / TM);
  a.k = k;
  a.d = d;
  a.cnorm = plan.cnorm;
  a.keytab = keytab;
  a.keyinv = keytab + 256;
  a.partials = plan.partials;
  a.counts = plan.counts;
  a.cost_partials = plan.cost_partials;
  a.labels_out = labels_out;
  a.mind_out = mindist_out;
  a.do_update = do_update ? 1 : 0;
  a.need_cost = (!do_update || mindist_out != nullptr) ? 1 : 0;
  a.st = st;

  const int rc = launch_listed(Insts{}, KP, DP, ctx, plan.grid, mx, mh, ml, a, s);
  if (rc == B2K_ERR_UNSUPPORTED) return b2k_fail(ctx, rc, "fused kernel: instantiation missing");
  B2K_TRY(rc);
  ctx->stats.kernel_launches++;
  ctx->stats.fused_tc_launches++;
  return B2K_OK;
}
