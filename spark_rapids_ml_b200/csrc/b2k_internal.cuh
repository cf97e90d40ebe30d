// Internal declarations shared by the translation units of libb2kmeans.so (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/b2kmeans.h"

// ------------------------------------------------------------------------------------------------
// Device-resident loop state: lets the host enqueue several Lloyd iterations without a D2H sync —
// every hot-loop kernel returns immediately once `done` is set (SURVEY.md §7 step 4).
// ------------------------------------------------------------------------------------------------
struct B2kLoopState {
  int iter;                  // completed iterations
  int done;                  // 1 once shift < tol (or iter == max_iter)
  int max_iter;
  unsigned int blocks_done;  // last-block-done counter of the finalize kernel
  double tol;
  double shift;              // last sum_j ||dc_j||^2
  double cost;               // last sum_i min_j ||x_i - c_j||^2 (w.r.t. the centers of that pass)
  // large-shape kernel: deferred (exactly re-decided) rows / candidate distances evaluated, cumulative over the call
  // (written by k_fix_accum_t; the host's convergence poll reads them to choose the path of the next burst)
  unsigned long long fix_rows_cum;
  unsigned long long fix_cands_cum;
};

// Layout of the reduced buffer R (doubles) that crosses NCCL: [k*d sums | k counts | 1 cost].
static inline size_t b2k_reduced_len(int k, int d) { return (size_t)k * d + k + 1; }

struct B2kNccl;  // opaque (b2k_comm.cu)

struct b2k_ctx {
  int device = 0;
  int sm_count = 0;
  size_t smem_optin = 0;
  std::string err;
  // options
  int kernel_path = B2K_PATH_AUTO;
  int time_kernels = 0;
  int check_every = 4;
  int adaptive_path = 1;         // option "adaptive_path": a Lloyd loop on the large-shape kernel falls back to the generic
                                 // kernels for its remaining iterations when most rows need the exact fix-up
  int collect_recheck = 0;       // option "collect_recheck": fill stats.recheck_* (costs a stream sync per call)
  void* xnorm_cache = nullptr;   // float2 [xnorm_cache_rows]: row norms shared by the passes of one fit (B2kNormScope)
  int64_t xnorm_cache_rows = 0;
  // comm
  B2kNccl* nccl = nullptr;
  int nranks = 1;
  int rank = 0;
  // scratch (device), grown on demand
  void* scratch = nullptr;
  size_t scratch_bytes = 0;
  // pinned staging for ingest (host) + device staging
  void* pinned[2] = {nullptr, nullptr};
  size_t pinned_bytes = 0;
  void* dev_stage[2] = {nullptr, nullptr};
  size_t dev_stage_bytes = 0;
  cudaEvent_t stage_evt[2] = {nullptr, nullptr};
  int stage_next = 0;
  void* copy_pool = nullptr;     // B2kCopyPool (b2k_ingest.cu): helper threads of the pageable -> pinned staging copy
  int ingest_threads = 0;        // option "ingest_threads": threads of that copy (0 = default 4, capped by the CPU quota)
  // pinned host mirror of the loop state (convergence polls)
  B2kLoopState* h_state = nullptr;
  // TMA descriptor encoder (driver entry point, resolved lazily)
  void* encode_tiled = nullptr;
  b2k_stats stats{};
};

// ------------------------------------------------------------------------------------------------
// error helpers
// ------------------------------------------------------------------------------------------------
int b2k_fail(b2k_ctx* ctx, int code, const std::string& msg);
#define B2K_CUDA_OK(ctx, expr)                                                             \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return b2k_fail((ctx), B2K_ERR_CUDA,                                                 \
                      std::string(#expr) + ": " + cudaGetErrorName(_e) + ": " +            \
                          cudaGetErrorString(_e));                                         \
  } while (0)
#define B2K_TRY(expr)            \
  do {                           \
    int _s = (expr);             \
    if (_s != B2K_OK) return _s; \
  } while (0)

int b2k_scratch_reserve(b2k_ctx* ctx, size_t bytes);
void b2k_copy_pool_destroy(b2k_ctx* ctx);

// Bump allocator over device scratch.  A measuring arena (default-constructed: null base, unlimited capacity) only
// counts bytes and hands out null pointers; a scratch user runs its layout on one to size b2k_scratch_reserve, then the
// same layout on Arena(ctx->scratch, ctx->scratch_bytes) to carve its pointers.  A take past the capacity sets
// `overflow`; the owner turns that into B2K_ERR_STATE before it launches anything.
struct Arena {
  char* base = nullptr;
  size_t cap = SIZE_MAX;
  size_t off = 0;
  bool overflow = false;
  Arena() = default;
  Arena(void* b, size_t c) : base(static_cast<char*>(b)), cap(c) {}
  template <typename T>
  T* take(size_t count, size_t align = 256) {
    off = (off + align - 1) / align * align;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    if (off > cap) overflow = true;
    return p;
  }
};

// Row norms of X shared by every large-shape pass of ONE b2k_kmeans_fit (the k-means|| candidate passes, the Lloyd loop
// and the inertia pass all read the same immutable X): the first pass computes them into ctx->xnorm_cache, the rest
// reuse them.  Owned by b2k_kmeans_fit; passes over any other matrix, and standalone lloyd / assign calls, get none.
struct B2kNormScope {
  const float* X;
  int64_t n;
  bool valid = false;   // ctx->xnorm_cache holds the norms of X
};

// Launches `kern` on clusters of two CTAs (the CTA pair of tcgen05 cta_group::2).
template <typename... Params, typename... Args>
int b2k_launch_pair(b2k_ctx* ctx, void (*kern)(Params...), int grid, int threads, size_t smem, cudaStream_t s,
                    const Args&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  B2K_CUDA_OK(ctx, cudaLaunchKernelEx(&cfg, kern, args...));
  return B2K_OK;
}

// ------------------------------------------------------------------------------------------------
// generic (any k, d) kernels — b2k_generic.cu
// ------------------------------------------------------------------------------------------------
// cnorm[j] = ||c_j||^2 (fp32 from a double accumulation)
int b2k_launch_center_norms(b2k_ctx* ctx, const float* C, int k, int d, float* cnorm,
                            const B2kLoopState* st, cudaStream_t s);
// labels/mindist (either may be NULL) + optional per-CTA cost partials
int b2k_launch_assign_generic(b2k_ctx* ctx, const float* X, int64_t n, int d, const float* C,
                              const float* cnorm, int k, int32_t* labels, float* mindist,
                              const B2kLoopState* st, cudaStream_t s);
// per-cluster partial sums from labels: partials [P][k*d] f32, counts [P][k] i32; b2k_update_generic_slots returns P.
int b2k_update_generic_slots(b2k_ctx* ctx, int64_t n, int d, int k);
int b2k_launch_update_generic(b2k_ctx* ctx, const float* X, int64_t n, int d, const int32_t* labels, int k,
                              int P, float* partials, int32_t* counts, const B2kLoopState* st,
                              cudaStream_t s);
// R[k*d+k+1] (double) = fixed-order sum over P partials (+ cost from mindist partial sums)
int b2k_launch_reduce_partials(b2k_ctx* ctx, const float* partials, const int32_t* counts,
                               const double* cost_partials, int P, int Pc, int k, int d, double* R,
                               const B2kLoopState* st, cudaStream_t s);
// C <- R.S / R.w (w == 0 keeps C), shift, iter++, done.  shift_scratch: k doubles.
int b2k_launch_finalize(b2k_ctx* ctx, const double* R, float* C, int k, int d, double* shift_scratch,
                        B2kLoopState* st, cudaStream_t s);
// cost partials: sum of mindist over fixed-size row blocks (deterministic two-level)
int b2k_launch_sum_f32_to_f64(b2k_ctx* ctx, const float* v, int64_t n, double* out /*1*/,
                              double* block_scratch, int nblocks, cudaStream_t s);
int b2k_launch_fold_f64(b2k_ctx* ctx, const double* in, int m, double* out /*1*/, cudaStream_t s);
int b2k_launch_gather_rows(b2k_ctx* ctx, const float* X, int d, const int64_t* rows_local, int m,
                           float* out, int64_t out_row0, cudaStream_t s);
// k-means|| helpers
int b2k_launch_bernoulli_pick(b2k_ctx* ctx, const float* mind, int64_t n, int64_t row_offset,
                              double scale /* l/phi */, uint64_t seed, int round, int64_t* picked,
                              int* n_picked, int cap, cudaStream_t s);
int b2k_launch_histogram(b2k_ctx* ctx, const int32_t* labels, int64_t n, int m, double* hist,
                         cudaStream_t s);
int b2k_launch_weighted_update(b2k_ctx* ctx, const float* P, const double* w, const int32_t* lab, int M, int d, int k,
                               float* C, cudaStream_t s);
int b2k_launch_pairwise_sqdist(b2k_ctx* ctx, const float* P, int M, int d, float* D2, cudaStream_t s);

// ------------------------------------------------------------------------------------------------
// Which kernels one pass over X runs — b2k_choose_kernel (b2k_api.cu)
// ------------------------------------------------------------------------------------------------
// Largest k and d of the 1xTF32 screening kernel (variant 1, b2k_fused_t.cu).
constexpr int kFusedTMaxK = 256;
constexpr int kFusedTMaxD = 256;
// The one 3xTF32 instantiation that runs on CTA pairs (tcgen05 cta_group::2).
constexpr bool b2k_tc_pair(int KP, int DP) { return KP == 64 && DP == 128; }

struct B2kChoice {
  enum Kind { GENERIC, FUSED, CHUNKED };
  Kind kind = GENERIC;
  int ch = 0;                // CHUNKED: centres per chunk; the fields below then describe the kernel of one chunk
  int variant = 0;           // 0: b2k_fused_tc.cu (3xTF32); 1: b2k_fused_t.cu (1xTF32 screening + exact recheck)
  int KP = 0, DP = 0;        // padded cluster count / dimension of the instantiation
  int pair = 0;              // 1: runs on CTA pairs (tcgen05 cta_group::2), the grid is even
  int path() const { return kind == GENERIC ? B2K_PATH_GENERIC : B2K_PATH_TCGEN05; }
};
// Chooses the kernels of one pass over X[n, d] against k centres under kernel path `path` (B2K_PATH_*); `near_tie`: the
// caller expects near-ties.  Fails with B2K_ERR_UNSUPPORTED when path = tcgen05 cannot be honoured.
int b2k_choose_kernel(b2k_ctx* ctx, int path, bool near_tie, int64_t n, int d, int k, const float* X, B2kChoice* out);

// ------------------------------------------------------------------------------------------------
// tcgen05 fused kernel — b2k_fused_tc.cu
// ------------------------------------------------------------------------------------------------
// The smallest 3xTF32 instantiation for (d, k): DP = d rounded up to a multiple of 32 (96 -> 128) and KP >= k.
// Returns false when none is compiled.
bool b2k_fused_tc_inst(int d, int k, int* KP, int* DP);

struct B2kFusedPlan {
  B2kChoice choice;          // the kernel of the pass (of each chunk, for a chunked pass)
  int grid = 0;              // persistent CTAs
  int P = 0;                 // partial-sum slots the pass writes (variant 0: grid; variant 1: CTA pairs + 4 for the deferred rows)
  int Pc = 0;                // cost partials the pass writes (variant 0: grid; variant 1: grid + fix-up CTAs)
  // scratch carved by b2k_fused_plan (null when planned on a measuring arena)
  float* partials = nullptr;         // [P][k*d] partial sums, [P][k] counts, [Pc] cost: b2k_launch_reduce_partials
  int32_t* counts = nullptr;
  double* cost_partials = nullptr;
  float* cnorm = nullptr;            // variant 0: [KP] ||c||^2; variant 1: [512] {||c||^2, ||c - tf32(c)||}
  uint8_t* keytab = nullptr;         // [2][256] cluster -> update slot table and its inverse
  float* c_hi = nullptr;             // variant 0: tf32 split of the centres, [KP][DP] each
  float* c_lo = nullptr;
  float* ct = nullptr;               // variant 1: [256][DP] tf32-rounded centres
  float* thr = nullptr;              // variant 1: [4] screening threshold coefficients
  unsigned long long* rstat = nullptr;  // variant 1: {rows re-decided exactly, candidate distances evaluated}
  float2* xnorm = nullptr;           // variant 1: [n] row norms (b2k_fused_prepare may point it at the fit's cache)
  int2* fix_list = nullptr;          // variant 1: deferred rows, one segment of seg_cap entries per CTA pair
  uint32_t* fix_masks = nullptr;     // variant 1: candidate masks for the first mask_cap entries of a segment
  int32_t* fix_count = nullptr;      // variant 1: entries per segment
  int seg_cap = 0, mask_cap = 0;
};
// Plans a fused pass over X[n, d] against k centres on the kernel `c` names (grid, partial slots) and carves its
// scratch from A.
int b2k_fused_plan(b2k_ctx* ctx, const B2kChoice& c, int64_t n, int d, int k, Arena& A, B2kFusedPlan* plan);
// Once per fit / lloyd / assign call, before the first b2k_launch_fused on this X (variant 1: row norms, into the plan's
// scratch or, with a norm scope, into the fit's cache; variant 0: no-op)
int b2k_fused_prepare(b2k_ctx* ctx, B2kFusedPlan& plan, const float* X, int64_t n, int d, B2kNormScope* norms,
                      cudaStream_t s);
// One fused pass: (labels_out, mindist_out optional) + partial sums/counts/cost into the plan's scratch.
// `do_update` = accumulate partial sums (Lloyd iteration) or labels only (assign/inertia pass).
// `need_cost`: the caller reads plan.cost_partials after an assign pass.  Variant 0 writes them on every assign pass
// (and whenever mindist_out is given); variant 1 on an assign pass that asks for them or writes mindist_out.
int b2k_launch_fused(b2k_ctx* ctx, const B2kFusedPlan& plan, const float* X, int64_t n, int d, const float* C, int k,
                     int32_t* labels_out, float* mindist_out, bool do_update, bool need_cost, const B2kLoopState* st,
                     cudaStream_t s, const double* prev_counts = nullptr);
// variant 1 diagnostics: {rows re-decided exactly, candidate distances evaluated} since the last b2k_fused_prepare
int b2k_fused_recheck_stats(b2k_ctx* ctx, const B2kFusedPlan& plan, unsigned long long out[2], cudaStream_t s);

// Tensor map of a row-major f32 matrix [outer][inner] with 128B swizzle (both fused kernels).
int b2k_encode_2d(b2k_ctx* ctx, CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer,
                  uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer, CUtensorMapL2promotion l2);

// b2k_fused_t.cu (variant 1)
int b2k_fused_t_plan(b2k_ctx* ctx, int64_t n, int d, int k, Arena& A, B2kFusedPlan* plan);
int b2k_fused_t_prepare(b2k_ctx* ctx, B2kFusedPlan& plan, const float* X, int64_t n, int d, B2kNormScope* norms,
                        cudaStream_t s);
int b2k_launch_fused_t(b2k_ctx* ctx, const B2kFusedPlan& plan, const float* X, int64_t n, int d, const float* C, int k,
                       int32_t* labels_out, float* mindist_out, bool do_update, bool need_cost, const B2kLoopState* st,
                       cudaStream_t s, const double* prev_counts);
int b2k_launch_merge_chunk(b2k_ctx* ctx, float* md_acc, int32_t* lab_acc, const float* md, const int32_t* lab, int base,
                           int64_t n, const B2kLoopState* st, cudaStream_t s);

// ------------------------------------------------------------------------------------------------
// comm — b2k_comm.cu
// ------------------------------------------------------------------------------------------------
int b2k_comm_allreduce_f64(b2k_ctx* ctx, double* buf, size_t count, cudaStream_t s);
int b2k_comm_allgather_i64(b2k_ctx* ctx, const int64_t* send_dev, int64_t* recv_dev, size_t count_per_rank,
                           cudaStream_t s);
int b2k_comm_allreduce_f32(b2k_ctx* ctx, float* buf, size_t count, cudaStream_t s);

// ingest — b2k_ingest.cu (entry point is the C ABI itself)
