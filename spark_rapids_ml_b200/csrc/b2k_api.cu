// C-ABI entry points + host-side driver of the Lloyd loop (see include/b2kmeans.h for the reference
// interfaces each one replaces).  The driver enqueues {fused assign+update | generic assign, update} ->
// fixed-order partial reduce -> NCCL allreduce of one fused f64 buffer -> finalize, several iterations ahead
// of the host; convergence lives on the device (B2kLoopState) and is polled every `check_every` iterations.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <random>
#include <vector>

#include "b2k_internal.cuh"

static std::string g_last_error;  // failures of calls that have no context

int b2k_fail(b2k_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  else g_last_error = msg;
  return code;
}

extern "C" int b2k_version(void) { return B2K_VERSION; }

extern "C" const char* b2k_last_error(const b2k_ctx* ctx) {
  return ctx ? ctx->err.c_str() : g_last_error.c_str();
}

extern "C" int b2k_ctx_create(int device, b2k_ctx** out) {
  if (!out) return b2k_fail(nullptr, B2K_ERR_INVALID, "b2k_ctx_create: out is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return b2k_fail(nullptr, B2K_ERR_CUDA,
                    std::string("b2k_ctx_create: no CUDA device (") + cudaGetErrorString(e) +
                        "); libb2kmeans has no CPU fallback");
  }
  if (device < 0 || device >= ndev)
    return b2k_fail(nullptr, B2K_ERR_INVALID, "b2k_ctx_create: device index out of range");
  b2k_ctx* ctx = new b2k_ctx();
  ctx->device = device;
  if ((e = cudaSetDevice(device)) != cudaSuccess) {
    delete ctx;
    return b2k_fail(nullptr, B2K_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  }
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    delete ctx;
    return b2k_fail(nullptr, B2K_ERR_CUDA, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e));
  }
  if (prop.major != 10) {
    delete ctx;
    return b2k_fail(nullptr, B2K_ERR_UNSUPPORTED,
                    "libb2kmeans is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) +
                        std::to_string(prop.minor));
  }
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  if ((e = cudaHostAlloc((void**)&ctx->h_state, 2 * sizeof(B2kLoopState), cudaHostAllocDefault)) != cudaSuccess) {
    delete ctx;
    return b2k_fail(nullptr, B2K_ERR_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
  }
  *out = ctx;
  return B2K_OK;
}

extern "C" int b2k_ctx_destroy(b2k_ctx* ctx) {
  if (!ctx) return B2K_OK;
  cudaSetDevice(ctx->device);
  if (ctx->nccl) b2k_comm_destroy(ctx);
  b2k_copy_pool_destroy(ctx);
  if (ctx->scratch) cudaFree(ctx->scratch);
  if (ctx->xnorm_cache) cudaFree(ctx->xnorm_cache);
  for (int i = 0; i < 2; ++i) {
    if (ctx->pinned[i]) cudaFreeHost(ctx->pinned[i]);
    if (ctx->dev_stage[i]) cudaFree(ctx->dev_stage[i]);
    if (ctx->stage_evt[i]) cudaEventDestroy(ctx->stage_evt[i]);
  }
  if (ctx->h_state) cudaFreeHost(ctx->h_state);
  delete ctx;
  return B2K_OK;
}

extern "C" int b2k_ctx_set_option(b2k_ctx* ctx, const char* key, int64_t value) {
  if (!ctx || !key) return b2k_fail(ctx, B2K_ERR_INVALID, "b2k_ctx_set_option: NULL argument");
  std::string k(key);
  if (k == "kernel_path") {
    if (value < B2K_PATH_AUTO || value > B2K_PATH_TCGEN05)
      return b2k_fail(ctx, B2K_ERR_INVALID, "kernel_path must be 0 (auto), 1 (generic) or 2 (tcgen05)");
    ctx->kernel_path = (int)value;
  } else if (k == "time_kernels") {
    ctx->time_kernels = value < 0 ? 0 : (value > 2 ? 2 : (int)value);
  } else if (k == "check_every") {
    if (value < 1) return b2k_fail(ctx, B2K_ERR_INVALID, "check_every must be >= 1");
    ctx->check_every = (int)value;
  } else if (k == "adaptive_path") {
    ctx->adaptive_path = value ? 1 : 0;
  } else if (k == "ingest_threads") {
    if (value < 0 || value > 64) return b2k_fail(ctx, B2K_ERR_INVALID, "ingest_threads must be in [0, 64]");
    b2k_copy_pool_destroy(ctx);
    ctx->ingest_threads = (int)value;
  } else if (k == "collect_recheck") {
    ctx->collect_recheck = value ? 1 : 0;
  } else {
    return b2k_fail(ctx, B2K_ERR_INVALID, "unknown option: " + k);
  }
  return B2K_OK;
}

extern "C" int b2k_get_stats(const b2k_ctx* ctx, b2k_stats* out) {
  if (!ctx || !out) return B2K_ERR_INVALID;
  *out = ctx->stats;
  return B2K_OK;
}
extern "C" int b2k_reset_stats(b2k_ctx* ctx) {
  if (!ctx) return B2K_ERR_INVALID;
  ctx->stats = b2k_stats{};
  return B2K_OK;
}

// Grows ctx->scratch to at least `bytes`.  Growing frees the old allocation, so no pointer carved before a reserve is
// used after it: each scratch user reserves for its whole layout first and carves afterwards.
int b2k_scratch_reserve(b2k_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->scratch_bytes) return B2K_OK;
  if (ctx->scratch) {
    B2K_CUDA_OK(ctx, cudaDeviceSynchronize());
    B2K_CUDA_OK(ctx, cudaFree(ctx->scratch));
    ctx->scratch = nullptr;
    ctx->scratch_bytes = 0;
  }
  size_t want = bytes + (bytes >> 3) + (1 << 20);
  cudaError_t e = cudaMalloc(&ctx->scratch, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return b2k_fail(ctx, B2K_ERR_NOMEM, "scratch cudaMalloc of " + std::to_string(want) + " bytes failed: " +
                                            cudaGetErrorString(e));
  }
  ctx->scratch_bytes = want;
  return B2K_OK;
}

namespace {
// Runs `layout` (int(Arena&): takes every buffer of one scratch user) on a measuring arena, reserves what it took, then
// runs it again on the scratch to carve the pointers.
template <typename Layout>
int carve_scratch(b2k_ctx* ctx, Layout&& layout) {
  Arena m;
  B2K_TRY(layout(m));
  B2K_TRY(b2k_scratch_reserve(ctx, m.off));
  Arena A(ctx->scratch, ctx->scratch_bytes);
  B2K_TRY(layout(A));
  return A.overflow ? b2k_fail(ctx, B2K_ERR_STATE, "scratch layout outgrew its reserve") : B2K_OK;
}

int check_shape(b2k_ctx* ctx, const char* who, const void* X, int64_t n, int d, int k) {
  if (!ctx) return b2k_fail(nullptr, B2K_ERR_INVALID, std::string(who) + ": ctx is NULL");
  if (!X || n < 0 || d <= 0 || k <= 0)
    return b2k_fail(ctx, B2K_ERR_INVALID, std::string(who) + ": bad X/n/d/k");
  return B2K_OK;
}

// Scratch of one Lloyd loop.
struct LoopBuffers {
  B2kLoopState* st;
  double* R;
  double* shift_scratch;
  float* cnorm;
  // generic
  int32_t* labels;
  float* partials;
  int32_t* counts;
  int P;
  // fused
  B2kFusedPlan plan;
};

}  // namespace

// ------------------------------------------------------------------------------------------------
// Which kernels a pass over X[n, d] against k centres runs.  TMA-ok: d % 4 == 0, X 16-byte aligned and
// 1 <= n <= 0x7fffff00.  tc(d, k): a 3xTF32 instantiation with DP = d rounded up to a multiple of 32 (96 -> 128) and
// KP >= k exists (b2k_fused_tc_inst: DP 32 with KP 16/32/64, DP 64 and 128 with KP 16/32/64/128).
//
//   kernel_path      condition (first match wins)                              pass runs on
//   generic          any                                                       generic
//   auto / tcgen05   TMA-ok, d <= 256, and either k > 256, or (near_tie,       chunks of ch = 128 (d <= 128) or 256
//                    d <= 128, k > 128)                                        centres: each chunk on variant 0 if
//                                                                              tc(d, ch), otherwise variant 1
//   auto / tcgen05   TMA-ok and tc(d, k)                                       variant 0; CTA pairs iff KP = 64, DP = 128
//   auto / tcgen05   TMA-ok, d <= 256, k <= 256                                variant 1, DP = 128 (d <= 128) or 256
//   auto             otherwise (this includes n = 0 in a Lloyd loop)           generic
//   tcgen05          otherwise                                                 B2K_ERR_UNSUPPORTED
//
// Variant 0 is the 3xTF32 kernel (b2k_fused_tc.cu), variant 1 the 1xTF32 screening kernel with its exact fix-up
// (b2k_fused_t.cu).  So d <= 32 with 64 < k <= 128, and 128-centre chunks at d <= 32, run on the screening kernel.
//
// Chunks: the centres are cut into chunks of exactly ch (the last chunk is [k - ch, k): the overlap is harmless for a
// min), each chunk runs one fused assign pass that yields the min distance and label of every row within the chunk, and
// k_merge_chunk keeps the smaller distance (strict '<': lowest cluster index on ties).  A chunked Lloyd loop keeps the
// generic label-driven update.  near_tie is set by the k-means|| candidate passes: candidates drawn from one blob are
// almost equidistant from its rows, which is the worst case of the screening kernel, so they prefer 128-centre chunks.
// ------------------------------------------------------------------------------------------------
int b2k_choose_kernel(b2k_ctx* ctx, int path, bool near_tie, int64_t n, int d, int k, const float* X, B2kChoice* out) {
  B2kChoice c;
  const bool tma_ok = d % 4 == 0 && (reinterpret_cast<uintptr_t>(X) & 15u) == 0 && n >= 1 && n <= (int64_t)0x7fffff00;
  if (path != B2K_PATH_GENERIC && tma_ok && d <= kFusedTMaxD) {
    if (k > kFusedTMaxK || (near_tie && d <= 128 && k > 128)) {
      c.kind = B2kChoice::CHUNKED;
      c.ch = d <= 128 ? 128 : 256;
    } else if (k <= kFusedTMaxK) {
      c.kind = B2kChoice::FUSED;
    }
  }
  if (c.kind != B2kChoice::GENERIC) {
    const int kk = c.kind == B2kChoice::CHUNKED ? c.ch : k;
    if (b2k_fused_tc_inst(d, kk, &c.KP, &c.DP)) {
      c.pair = b2k_tc_pair(c.KP, c.DP) ? 1 : 0;
    } else {
      c.variant = 1;
      c.KP = kFusedTMaxK;
      c.DP = d <= 128 ? 128 : 256;
      c.pair = 1;
    }
  } else if (path == B2K_PATH_TCGEN05) {
    return b2k_fail(ctx, B2K_ERR_UNSUPPORTED,
                    "kernel_path=tcgen05 requested but shape (n=" + std::to_string(n) + ", d=" + std::to_string(d) +
                        ", k=" + std::to_string(k) + ") is outside the fused kernel's instantiations");
  }
  *out = c;
  return B2K_OK;
}

namespace {
struct ChunkedAssign {
  B2kFusedPlan plan;         // the kernel of one chunk (plan.choice.ch centres)
  int32_t* tmp_lab = nullptr;
  float* tmp_md = nullptr;
  int32_t* lab_acc = nullptr;   // used when the caller passes no labels / mindist buffer
  float* md_acc = nullptr;
};
// the caller runs b2k_fused_prepare(ca.plan, ...) before chunked_assign_run
int chunked_assign_layout(b2k_ctx* ctx, const B2kChoice& c, int64_t n, int d, Arena& A, ChunkedAssign* ca) {
  ca->tmp_lab = A.take<int32_t>(n);
  ca->tmp_md = A.take<float>(n);
  ca->lab_acc = A.take<int32_t>(n);
  ca->md_acc = A.take<float>(n);
  return b2k_fused_plan(ctx, c, n, d, c.ch, A, &ca->plan);
}
int chunked_assign_run(b2k_ctx* ctx, const ChunkedAssign& ca, const float* X, int64_t n, int d, const float* C, int k,
                       int32_t* labels, float* mindist, const B2kLoopState* st, cudaStream_t s) {
  int32_t* lab = labels ? labels : ca.lab_acc;
  float* md = mindist ? mindist : ca.md_acc;
  const int ch = ca.plan.choice.ch;
  for (int c0 = 0; c0 < k; c0 += ch) {
    const int base = std::min(c0, k - ch);
    const bool first = c0 == 0;
    // every chunk writes mindist, which makes both variants compute the cost: the merge needs no cost partials
    B2K_TRY(b2k_launch_fused(ctx, ca.plan, X, n, d, C + (size_t)base * d, ch, first ? lab : ca.tmp_lab,
                             first ? md : ca.tmp_md, false, false, st, s));
    if (!first) B2K_TRY(b2k_launch_merge_chunk(ctx, md, lab, ca.tmp_md, ca.tmp_lab, base, n, st, s));
  }
  return B2K_OK;
}
}  // namespace

// ------------------------------------------------------------------------------------------------
// Lloyd loop
// ------------------------------------------------------------------------------------------------
// `norms`: the fit's row-norm scope (null for a standalone call); *path_out: the path the loop ended on (B2K_PATH_*)
static int lloyd_impl(b2k_ctx* ctx, const float* X, int64_t n, int d, int k, float* C, int max_iter, double tol,
                      B2kNormScope* norms, int* n_iter_out, double* shift_out, int* path_out, cudaStream_t s) {
  if (max_iter < 0) return b2k_fail(ctx, B2K_ERR_INVALID, "lloyd: max_iter < 0");
  B2kChoice c;
  B2K_TRY(b2k_choose_kernel(ctx, ctx->kernel_path, false, n, d, k, X, &c));
  const bool fused = c.kind == B2kChoice::FUSED;
  const bool chunked = c.kind == B2kChoice::CHUNKED;
  // The large-shape kernel (1xTF32 screening) hands near-tie rows to an exact fix-up; on data where most rows are
  // near-ties (e.g. uniform noise in 256 dimensions) the generic kernels are several times faster, so the loop may
  // switch to them between bursts.  The choice is local to the rank: both paths fill the same R buffer.
  const bool can_switch = fused && c.variant == 1 && ctx->adaptive_path && ctx->kernel_path == B2K_PATH_AUTO;

  LoopBuffers B{};
  ChunkedAssign ca;
  const size_t rlen = b2k_reduced_len(k, d);
  B2K_TRY(carve_scratch(ctx, [&](Arena& A) -> int {
    B.st = A.take<B2kLoopState>(1);
    B.R = A.take<double>(rlen);
    B.shift_scratch = A.take<double>(k);
    B.cnorm = A.take<float>(k);
    if (fused) B2K_TRY(b2k_fused_plan(ctx, c, n, d, k, A, &B.plan));
    if (!fused || can_switch) {
      B.P = b2k_update_generic_slots(ctx, n, d, k);
      B.labels = A.take<int32_t>(n > 0 ? n : 1);
      B.partials = A.take<float>((size_t)B.P * k * d);
      B.counts = A.take<int32_t>((size_t)B.P * k);
    }
    if (chunked) B2K_TRY(chunked_assign_layout(ctx, c, n, d, A, &ca));
    return B2K_OK;
  }));

  B2kLoopState init{};
  init.iter = 0;
  init.done = max_iter == 0 ? 1 : 0;
  init.max_iter = max_iter;
  init.blocks_done = 0;
  init.tol = tol;
  init.shift = 0.0;
  init.cost = 0.0;
  init.fix_rows_cum = 0;
  init.fix_cands_cum = 0;
  *ctx->h_state = init;
  B2K_CUDA_OK(ctx, cudaMemcpyAsync(B.st, ctx->h_state, sizeof(B2kLoopState), cudaMemcpyHostToDevice, s));
  B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));  // h_state is reused as the D2H mirror below

  // Events are created BEFORE the timed loop (cudaEventCreate inside it showed up in the multi-GPU per-iteration gap).
  // time_kernels = 1: around every fused launch; 2: also after the partial reduce, the allreduce and finalize.
  const int nev_per_it = ctx->time_kernels >= 2 ? 5 : (ctx->time_kernels ? 2 : 0);
  std::vector<cudaEvent_t> ev;
  cudaEvent_t loop0 = nullptr, loop1 = nullptr, poll_ev[2] = {nullptr, nullptr};
  if (ctx->time_kernels) {
    ev.resize((size_t)nev_per_it * (size_t)std::max(max_iter, 0));
    for (auto& e : ev) B2K_CUDA_OK(ctx, cudaEventCreate(&e));
    B2K_CUDA_OK(ctx, cudaEventCreate(&loop0));
    B2K_CUDA_OK(ctx, cudaEventCreate(&loop1));
  }
  B2K_CUDA_OK(ctx, cudaEventCreateWithFlags(&poll_ev[0], cudaEventDisableTiming));
  B2K_CUDA_OK(ctx, cudaEventCreateWithFlags(&poll_ev[1], cudaEventDisableTiming));
  if (fused && max_iter > 0) B2K_TRY(b2k_fused_prepare(ctx, B.plan, X, n, d, norms, s));
  if (chunked && max_iter > 0) B2K_TRY(b2k_fused_prepare(ctx, ca.plan, X, n, d, norms, s));
  if (ctx->time_kernels) B2K_CUDA_OK(ctx, cudaEventRecord(loop0, s));

  // The host stays one burst ahead of the device: burst b + 1 is enqueued BEFORE the convergence flag of burst b is
  // read back, so a poll never drains the stream (every hot-loop kernel returns at once when `done` is set, which
  // makes an over-enqueued burst free).  The read-backs alternate between two pinned mirrors.
  int launched = 0, slot = 0;
  bool done = (max_iter == 0), have_pending = false;
  bool fused_now = fused;
  int burst_iters[2] = {0, 0};
  unsigned long long seen_rows = 0, seen_cands = 0;
  ctx->stats.path_switch_iter = -1;
  B2kLoopState* mirror = ctx->h_state;
  int last_slot = 0;
  while (!done && launched < max_iter) {
    int burst = std::min(ctx->check_every, max_iter - launched);
    for (int b = 0; b < burst; ++b) {
      cudaEvent_t* e = ctx->time_kernels ? &ev[(size_t)launched * nev_per_it] : nullptr;
      if (fused_now) {
        if (e) B2K_CUDA_OK(ctx, cudaEventRecord(e[0], s));
        // cluster sizes of the previous iteration (R = [k*d sums | k counts | cost]) drive the update-warp balancing
        B2K_TRY(b2k_launch_fused(ctx, B.plan, X, n, d, C, k, nullptr, nullptr, true, false, B.st, s,
                                 launched > 0 ? B.R + (size_t)k * d : nullptr));
        if (e) B2K_CUDA_OK(ctx, cudaEventRecord(e[1], s));
        B2K_TRY(b2k_launch_reduce_partials(ctx, B.plan.partials, B.plan.counts, B.plan.cost_partials, B.plan.P,
                                           B.plan.Pc, k, d, B.R, B.st, s));
      } else {
        if (e) B2K_CUDA_OK(ctx, cudaEventRecord(e[0], s));
        if (chunked) {
          B2K_TRY(chunked_assign_run(ctx, ca, X, n, d, C, k, B.labels, nullptr, B.st, s));
        } else {
          B2K_TRY(b2k_launch_center_norms(ctx, C, k, d, B.cnorm, B.st, s));
          B2K_TRY(b2k_launch_assign_generic(ctx, X, n, d, C, B.cnorm, k, B.labels, nullptr, B.st, s));
        }
        B2K_TRY(b2k_launch_update_generic(ctx, X, n, d, B.labels, k, B.P, B.partials, B.counts, B.st, s));
        if (e) B2K_CUDA_OK(ctx, cudaEventRecord(e[1], s));
        B2K_TRY(b2k_launch_reduce_partials(ctx, B.partials, B.counts, nullptr, B.P, 0, k, d, B.R, B.st, s));
      }
      if (e && nev_per_it == 5) B2K_CUDA_OK(ctx, cudaEventRecord(e[2], s));
      if (ctx->nranks > 1) B2K_TRY(b2k_comm_allreduce_f64(ctx, B.R, rlen, s));
      if (e && nev_per_it == 5) B2K_CUDA_OK(ctx, cudaEventRecord(e[3], s));
      B2K_TRY(b2k_launch_finalize(ctx, B.R, C, k, d, B.shift_scratch, B.st, s));
      if (e && nev_per_it == 5) B2K_CUDA_OK(ctx, cudaEventRecord(e[4], s));
      ++launched;
    }
    burst_iters[slot] = fused_now ? burst : 0;
    B2K_CUDA_OK(ctx, cudaMemcpyAsync(&mirror[slot], B.st, sizeof(B2kLoopState), cudaMemcpyDeviceToHost, s));
    B2K_CUDA_OK(ctx, cudaEventRecord(poll_ev[slot], s));
    if (have_pending) {   // the flag of the PREVIOUS burst, while this one is already queued
      B2K_CUDA_OK(ctx, cudaEventSynchronize(poll_ev[slot ^ 1]));
      const B2kLoopState& m = mirror[slot ^ 1];
      done = m.done != 0;
      if (can_switch && fused_now && burst_iters[slot ^ 1] > 0 && n > 0) {
        // measured on B200 (tools/fix_split.py, k = d = 256): the fix-up costs ~0.14 ns per candidate distance + ~0.85 ns
        // per deferred row; the generic kernels ~6.4 ns per row more than the fused pass (scaled here by k d)
        const double it = (double)burst_iters[slot ^ 1];
        const double rows_per_row = (double)(m.fix_rows_cum - seen_rows) / it / (double)n;
        const double cands_per_row = (double)(m.fix_cands_cum - seen_cands) / it / (double)n;
        const double generic_extra_ns = 6.4 * ((double)k * (double)d) / 65536.0;
        if (0.14 * cands_per_row + 0.85 * rows_per_row > generic_extra_ns) {
          fused_now = false;
          ctx->stats.path_switch_iter = launched;
        }
      }
      seen_rows = m.fix_rows_cum;
      seen_cands = m.fix_cands_cum;
    }
    last_slot = slot;
    have_pending = true;
    slot ^= 1;
  }
  B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
  if (have_pending && last_slot != 0) mirror[0] = mirror[last_slot];   // h_state[0] = the final state
  cudaEventDestroy(poll_ev[0]);
  cudaEventDestroy(poll_ev[1]);
  if (ctx->time_kernels) {
    B2K_CUDA_OK(ctx, cudaEventRecord(loop1, s));
    B2K_CUDA_OK(ctx, cudaEventSynchronize(loop1));
    float ms = 0.f;
    B2K_CUDA_OK(ctx, cudaEventElapsedTime(&ms, loop0, loop1));
    ctx->stats.last_loop_ms = ms;
    double acc = 0.0, acc_red = 0.0, acc_comm = 0.0, acc_fin = 0.0;
    int cnt = 0;
    const int iters_done = ctx->h_state->iter;
    for (int i = 0; i < launched && i < iters_done; ++i) {   // launches after convergence are no-ops
      float m = 0.f;
      cudaEvent_t* e = &ev[(size_t)i * nev_per_it];
      cudaEventElapsedTime(&m, e[0], e[1]);
      acc += m;
      if (nev_per_it == 5) {
        cudaEventElapsedTime(&m, e[1], e[2]); acc_red += m;
        cudaEventElapsedTime(&m, e[2], e[3]); acc_comm += m;
        cudaEventElapsedTime(&m, e[3], e[4]); acc_fin += m;
      }
      ++cnt;
    }
    for (auto& e : ev) cudaEventDestroy(e);
    ctx->stats.last_fused_ms = cnt ? acc / cnt : 0.0;
    ctx->stats.last_reduce_ms = cnt ? acc_red / cnt : 0.0;
    ctx->stats.last_allreduce_ms = cnt ? acc_comm / cnt : 0.0;
    ctx->stats.last_finalize_ms = cnt ? acc_fin / cnt : 0.0;
    cudaEventDestroy(loop0);
    cudaEventDestroy(loop1);
  }
  ctx->stats.last_n_iter = ctx->h_state->iter;
  ctx->stats.last_path = ctx->stats.path_switch_iter >= 0 ? B2K_PATH_GENERIC : c.path();
  if (path_out) *path_out = ctx->stats.last_path;
  if (fused && ctx->collect_recheck && max_iter > 0) {
    unsigned long long rs[2];
    B2K_TRY(b2k_fused_recheck_stats(ctx, B.plan, rs, s));
    ctx->stats.recheck_rows = (int64_t)rs[0];
    ctx->stats.recheck_candidates = (int64_t)rs[1];
  }
  if (n_iter_out) *n_iter_out = ctx->h_state->iter;
  if (shift_out) *shift_out = ctx->h_state->shift;
  return B2K_OK;
}

extern "C" int b2k_kmeans_lloyd(b2k_ctx* ctx, const float* X, int64_t n_local, int d, int k, float* centers,
                                int max_iter, double tol, int* n_iter_out, double* shift_out, uintptr_t stream) {
  B2K_TRY(check_shape(ctx, "b2k_kmeans_lloyd", X, n_local, d, k));
  if (!centers) return b2k_fail(ctx, B2K_ERR_INVALID, "b2k_kmeans_lloyd: centers is NULL");
  B2K_CUDA_OK(ctx, cudaSetDevice(ctx->device));
  return lloyd_impl(ctx, X, n_local, d, k, centers, max_iter, tol, nullptr, n_iter_out, shift_out, nullptr,
                    reinterpret_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------------
// assign (+ optional total cost): labels/mindist may be NULL
// ------------------------------------------------------------------------------------------------
namespace {
// per-call choices of an assign pass
struct PassOpts {
  int path;                        // kernel path to honour (B2K_PATH_*): the option, or the path a fit's Lloyd loop ended on
  bool near_tie = false;           // the caller expects near-ties (b2k_choose_kernel)
  B2kNormScope* norms = nullptr;   // the fit's row-norm scope, for passes over the fit's X
};

constexpr int kCostBlocks = 1024;   // block sums of a cost formed from mindist

// One assign pass: chunked, one fused pass, or the generic kernels, and the scratch that route takes.
struct AssignPass {
  B2kChoice c;
  ChunkedAssign ca;
  B2kFusedPlan plan;
  float* cnorm = nullptr;    // generic
  float* md = nullptr;       // generic: mindist of its own, for a cost without the caller's mindist
  double* blocks = nullptr;  // chunked / generic: cost block sums
};

int assign_layout(b2k_ctx* ctx, const PassOpts& o, const float* X, int64_t n, int d, int k, bool own_md, Arena& A,
                  AssignPass* p) {
  B2K_TRY(b2k_choose_kernel(ctx, o.path, o.near_tie, n, d, k, X, &p->c));
  if (p->c.kind == B2kChoice::CHUNKED) {
    B2K_TRY(chunked_assign_layout(ctx, p->c, n, d, A, &p->ca));
    p->blocks = A.take<double>(kCostBlocks);
    return B2K_OK;
  }
  if (p->c.kind == B2kChoice::FUSED) return b2k_fused_plan(ctx, p->c, n, d, k, A, &p->plan);
  p->cnorm = A.take<float>(k);
  if (own_md) p->md = A.take<float>(n > 0 ? n : 1);
  p->blocks = A.take<double>(kCostBlocks);
  return B2K_OK;
}

// Takes room for the largest assign pass over X[n, d] with any centre count in `ks`.  The passes themselves carve from
// a copy of the arena as it was before this call (assign_impl).
int assign_room(b2k_ctx* ctx, const PassOpts& o, const float* X, int64_t n, int d, std::initializer_list<int> ks,
                bool own_md, Arena& A) {
  Arena end = A;
  for (int kk : ks) {
    Arena a = A;
    AssignPass p;
    B2K_TRY(assign_layout(ctx, o, X, n, d, kk, own_md, a, &p));
    if (a.off > end.off) end = a;
  }
  A = end;
  return B2K_OK;
}
}  // namespace

// `A`: the scratch its caller left for the pass (see assign_room)
static int assign_impl(b2k_ctx* ctx, Arena A, const PassOpts& o, const float* X, int64_t n, int d, const float* C,
                       int k, int32_t* labels, float* mindist, double* cost_dev /* device, 1 double, may be NULL */,
                       cudaStream_t s) {
  AssignPass p;
  B2K_TRY(assign_layout(ctx, o, X, n, d, k, cost_dev && !mindist, A, &p));
  if (A.overflow) return b2k_fail(ctx, B2K_ERR_STATE, "assign_impl: the pass outgrows the scratch reserved for it");
  ctx->stats.last_path = p.c.path();
  if (p.c.kind == B2kChoice::CHUNKED) {   // chunks of ch centres through a fused assign pass each
    B2K_TRY(b2k_fused_prepare(ctx, p.ca.plan, X, n, d, o.norms, s));
    B2K_TRY(chunked_assign_run(ctx, p.ca, X, n, d, C, k, labels, mindist, nullptr, s));
    if (cost_dev)
      B2K_TRY(b2k_launch_sum_f32_to_f64(ctx, mindist ? mindist : p.ca.md_acc, n, cost_dev, p.blocks, kCostBlocks, s));
  } else if (p.c.kind == B2kChoice::FUSED) {
    B2K_TRY(b2k_fused_prepare(ctx, p.plan, X, n, d, o.norms, s));
    B2K_TRY(b2k_launch_fused(ctx, p.plan, X, n, d, C, k, labels, mindist, false, cost_dev != nullptr, nullptr, s));
    // fold the per-CTA cost partials in index order
    if (cost_dev) B2K_TRY(b2k_launch_fold_f64(ctx, p.plan.cost_partials, p.plan.Pc, cost_dev, s));
  } else {
    float* md = mindist ? mindist : p.md;
    B2K_TRY(b2k_launch_center_norms(ctx, C, k, d, p.cnorm, nullptr, s));
    B2K_TRY(b2k_launch_assign_generic(ctx, X, n, d, C, p.cnorm, k, labels, md, nullptr, s));
    if (cost_dev) B2K_TRY(b2k_launch_sum_f32_to_f64(ctx, md, n, cost_dev, p.blocks, kCostBlocks, s));
  }
  if (ctx->collect_recheck && p.c.kind != B2kChoice::GENERIC) {
    unsigned long long rs[2];
    B2K_TRY(b2k_fused_recheck_stats(ctx, p.c.kind == B2kChoice::CHUNKED ? p.ca.plan : p.plan, rs, s));
    ctx->stats.recheck_rows = (int64_t)rs[0];
    ctx->stats.recheck_candidates = (int64_t)rs[1];
  }
  return B2K_OK;
}

extern "C" int b2k_kmeans_assign(b2k_ctx* ctx, const float* X, int64_t n, int d, const float* centers, int k,
                                 int32_t* labels_out, float* mindist_out, uintptr_t stream) {
  B2K_TRY(check_shape(ctx, "b2k_kmeans_assign", X, n, d, k));
  if (!centers) return b2k_fail(ctx, B2K_ERR_INVALID, "b2k_kmeans_assign: centers is NULL");
  if (n == 0) return B2K_OK;
  B2K_CUDA_OK(ctx, cudaSetDevice(ctx->device));
  const PassOpts o{ctx->kernel_path};
  Arena pass;
  B2K_TRY(carve_scratch(ctx, [&](Arena& A) -> int {
    pass = A;
    return assign_room(ctx, o, X, n, d, {k}, false, A);
  }));
  return assign_impl(ctx, pass, o, X, n, d, centers, k, labels_out, mindist_out, nullptr,
                     reinterpret_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------------
// initialisers
// ------------------------------------------------------------------------------------------------
namespace {
// global row bookkeeping across ranks
struct Rows {
  std::vector<int64_t> sizes;  // per rank
  int64_t offset = 0;          // this rank's first global row
  int64_t total = 0;
};

int gather_sizes(b2k_ctx* ctx, int64_t n_local, Rows* rows, cudaStream_t s) {
  rows->sizes.assign(ctx->nranks, 0);
  if (ctx->nranks == 1) {
    rows->sizes[0] = n_local;
  } else {
    int64_t *send, *recv;
    B2K_TRY(carve_scratch(ctx, [&](Arena& A) -> int {
      send = A.take<int64_t>(1);
      recv = A.take<int64_t>(ctx->nranks);
      return B2K_OK;
    }));
    B2K_CUDA_OK(ctx, cudaMemcpyAsync(send, &n_local, 8, cudaMemcpyHostToDevice, s));
    B2K_TRY(b2k_comm_allgather_i64(ctx, send, recv, 1, s));
    B2K_CUDA_OK(ctx, cudaMemcpyAsync(rows->sizes.data(), recv, 8 * (size_t)ctx->nranks, cudaMemcpyDeviceToHost, s));
    B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
  }
  rows->offset = 0;
  rows->total = 0;
  for (int r = 0; r < ctx->nranks; ++r) {
    if (r < ctx->rank) rows->offset += rows->sizes[r];
    rows->total += rows->sizes[r];
  }
  return B2K_OK;
}

// out[m,d] (device) <- rows with the given sorted GLOBAL indices, identical on every rank.
int fetch_global_rows(b2k_ctx* ctx, const float* X, int64_t n_local, int d, const Rows& rows,
                      const std::vector<int64_t>& gidx, float* out, int64_t* idx_dev, cudaStream_t s) {
  const int m = (int)gidx.size();
  if (m == 0) return B2K_OK;
  B2K_CUDA_OK(ctx, cudaMemsetAsync(out, 0, (size_t)m * d * sizeof(float), s));
  // contiguous run of indices owned by this rank (gidx is sorted)
  int lo = 0;
  while (lo < m && gidx[lo] < rows.offset) ++lo;
  int hi = lo;
  while (hi < m && gidx[hi] < rows.offset + n_local) ++hi;
  if (hi > lo) {
    std::vector<int64_t> local(hi - lo);
    for (int i = lo; i < hi; ++i) local[i - lo] = gidx[i] - rows.offset;
    B2K_CUDA_OK(ctx, cudaMemcpyAsync(idx_dev, local.data(), local.size() * 8, cudaMemcpyHostToDevice, s));
    B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));  // `local` dies at scope end
    B2K_TRY(b2k_launch_gather_rows(ctx, X, d, idx_dev, hi - lo, out, lo, s));
  }
  if (ctx->nranks > 1) B2K_TRY(b2k_comm_allreduce_f32(ctx, out, (size_t)m * d, s));
  return B2K_OK;
}

std::vector<int64_t> sample_distinct(std::mt19937_64& rng, int64_t total, int m) {
  // Floyd's algorithm: m distinct values in [0,total)
  std::vector<int64_t> chosen;
  chosen.reserve(m);
  for (int64_t j = total - m; j < total; ++j) {
    std::uniform_int_distribution<int64_t> U(0, j);
    int64_t t = U(rng);
    if (std::find(chosen.begin(), chosen.end(), t) == chosen.end()) chosen.push_back(t);
    else chosen.push_back(j);
  }
  std::sort(chosen.begin(), chosen.end());
  return chosen;
}

// Weighted greedy k-means++ on the (small) candidate set — host side, on the candidate-to-candidate squared distances
// D2 [M x M] computed on the device (every k-means++ centre IS a candidate, so the greedy phase is table look-ups:
// k * trials * M instead of k * trials * M * d operations).  Returns the chosen candidate indices; the weighted Lloyd
// refinement that follows runs on the device (init_kmeans_parallel).
void reduce_candidates(const std::vector<float>& D2, const std::vector<double>& wts, int M, int k, std::mt19937_64& rng,
                       std::vector<int64_t>* out) {
  std::vector<double> d2(M), cum(M);
  std::vector<int> chosen;
  chosen.reserve(k);
  // draw i with probability prob[i] / tot from the running sums cum[] (first i with u < cum[i])
  auto pick = [&](double tot) {
    std::uniform_real_distribution<double> U(0.0, tot);
    const double u = U(rng);
    const int i = (int)(std::upper_bound(cum.begin(), cum.end(), u) - cum.begin());
    return std::min(i, M - 1);
  };
  // potential of adding candidate c: sum_i w_i min(d2_i, D2[c][i]); four fixed partial sums (identical on every rank)
  auto potential = [&](int c) {
    const float* row = &D2[(size_t)c * M];
    double p0 = 0, p1 = 0, p2 = 0, p3 = 0;
    int i = 0;
    for (; i + 4 <= M; i += 4) {
      p0 += wts[i] * std::min(d2[i], (double)row[i]);
      p1 += wts[i + 1] * std::min(d2[i + 1], (double)row[i + 1]);
      p2 += wts[i + 2] * std::min(d2[i + 2], (double)row[i + 2]);
      p3 += wts[i + 3] * std::min(d2[i + 3], (double)row[i + 3]);
    }
    for (; i < M; ++i) p0 += wts[i] * std::min(d2[i], (double)row[i]);
    return (p0 + p1) + (p2 + p3);
  };
  double tot = 0;
  for (int i = 0; i < M; ++i) { tot += wts[i]; cum[i] = tot; }
  const int first = pick(tot);
  chosen.push_back(first);
  for (int i = 0; i < M; ++i) d2[i] = (double)D2[(size_t)first * M + i];
  const int trials = 2 + (int)std::log((double)std::max(k, 2));
  for (int j = 1; j < k; ++j) {
    tot = 0;
    for (int i = 0; i < M; ++i) { tot += wts[i] * d2[i]; cum[i] = tot; }
    double best_pot = -1;
    int best_c = 0;
    for (int tr = 0; tr < trials; ++tr) {
      const int c = tot > 0 ? pick(tot) : (int)(rng() % M);
      const double pot = potential(c);
      if (best_pot < 0 || pot < best_pot) { best_pot = pot; best_c = c; }
    }
    chosen.push_back(best_c);
    const float* row = &D2[(size_t)best_c * M];
    for (int i = 0; i < M; ++i) d2[i] = std::min(d2[i], (double)row[i]);
  }
  out->assign(chosen.begin(), chosen.end());
}
}  // namespace

static int init_random(b2k_ctx* ctx, const float* X, int64_t n, int d, int k, uint64_t seed, float* C,
                       cudaStream_t s) {
  Rows rows;
  B2K_TRY(gather_sizes(ctx, n, &rows, s));
  if (rows.total < k)
    return b2k_fail(ctx, B2K_ERR_INVALID, "init=random: fewer rows (" + std::to_string(rows.total) + ") than k");
  std::mt19937_64 rng(seed);
  std::vector<int64_t> gidx = sample_distinct(rng, rows.total, k);
  int64_t* idx_dev;
  B2K_TRY(carve_scratch(ctx, [&](Arena& A) -> int {
    idx_dev = A.take<int64_t>(k);
    return B2K_OK;
  }));
  return fetch_global_rows(ctx, X, n, d, rows, gidx, C, idx_dev, s);
}

// Scalable k-means++ (k-means||): the reference forwards init="scalable-k-means++", oversampling_factor=2.0
// (clustering.py:134-136).  Distributional parity only (the reference's own seeded test is xfail).
static int init_kmeans_parallel(b2k_ctx* ctx, const float* X, int64_t n, int d, int k, uint64_t seed,
                                double oversampling, B2kNormScope* norms, float* C, cudaStream_t s) {
  // the candidate passes are near-tie heavy (see b2k_choose_kernel); only those over X share the fit's row norms
  const PassOpts ox{ctx->kernel_path, true, norms};
  const PassOpts ocand{ctx->kernel_path, true, nullptr};
  const int rounds = 5;
  Rows rows;
  B2K_TRY(gather_sizes(ctx, n, &rows, s));
  if (rows.total < k)
    return b2k_fail(ctx, B2K_ERR_INVALID, "init=k-means||: fewer rows (" + std::to_string(rows.total) + ") than k");
  const double ell = oversampling * k;
  const int cap = (int)std::min<int64_t>(rows.total, (int64_t)(4 * ell) + 64);  // per-round candidate cap
  const int Mmax = 1 + rounds * cap + k;
  const size_t nn = (size_t)(n > 0 ? n : 1);
  const size_t per = (size_t)cap + 1;   // [count | cap indices] per rank in the candidate exchange
  int64_t *idx_dev, *xchg;
  int* n_picked_dev;
  double *phi_dev, *blocks, *hist;
  float *mind, *dn, *cand, *newc;
  int32_t *labels, *lab_new;
  Arena pass;
  B2K_TRY(carve_scratch(ctx, [&](Arena& A) -> int {
    idx_dev = A.take<int64_t>(cap + 8);
    n_picked_dev = A.take<int>(8);
    phi_dev = A.take<double>(4);
    blocks = A.take<double>(1024);
    xchg = A.take<int64_t>(per * (size_t)(ctx->nranks + 1));
    mind = A.take<float>(nn);
    dn = A.take<float>(nn);
    labels = A.take<int32_t>(nn);    // running nearest candidate of every row (global candidate index)
    lab_new = A.take<int32_t>(nn);   // nearest among one round's new candidates
    cand = A.take<float>((size_t)Mmax * d);
    newc = A.take<float>((size_t)cap * d);
    hist = A.take<double>(Mmax);
    pass = A;
    // the assign passes below run with 1 .. Mmax centres: small counts take a fused kernel (its scratch holds per-CTA
    // partial slots and, for the large-shape kernel, the row norms), larger ones chunks or the generic path
    return assign_room(ctx, ox, X, n, d, {1, std::min(cap, 128), std::min(cap, 256), cap, Mmax}, false, A);
  }));

  std::mt19937_64 rng(seed);
  int M = 0;
  {  // first candidate: one uniformly random row
    std::uniform_int_distribution<int64_t> U(0, rows.total - 1);
    std::vector<int64_t> g{U(rng)};
    B2K_TRY(fetch_global_rows(ctx, X, n, d, rows, g, cand, idx_dev, s));
    M = 1;
    B2K_TRY(assign_impl(ctx, pass, ox, X, n, d, cand, 1, nullptr, mind, phi_dev, s));
    B2K_CUDA_OK(ctx, cudaMemsetAsync(labels, 0, nn * 4, s));   // every row is nearest to candidate 0 so far
  }
  std::vector<int64_t> picked_host(cap);
  std::vector<int64_t> counts_host(ctx->nranks);
  for (int r = 0; r < rounds; ++r) {
    double phi = 0;
    if (r > 0) {
      // phi = sum(mind) (deterministic two-level sum)
      B2K_TRY(b2k_launch_sum_f32_to_f64(ctx, mind, n, phi_dev, blocks, 1024, s));
    }
    if (ctx->nranks > 1) B2K_TRY(b2k_comm_allreduce_f64(ctx, phi_dev, 1, s));
    B2K_CUDA_OK(ctx, cudaMemcpyAsync(&phi, phi_dev, 8, cudaMemcpyDeviceToHost, s));
    B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
    if (!(phi > 0)) break;
    // The pick kernel stores at most cap entries and WHICH ones it keeps on overflow depends on atomic slot order, so an
    // overflowing draw (expected ell picks against cap = 4 ell + 64: essentially never) is repeated with a smaller
    // probability scale: the draw is keyed on (seed, round, global row), so the smaller draw is a subset and the
    // candidate set stays a deterministic function of the seed.
    double scale = ell / phi;
    int np = 0;
    for (int attempt = 0; attempt < 8; ++attempt) {
      B2K_CUDA_OK(ctx, cudaMemsetAsync(n_picked_dev, 0, sizeof(int), s));
      B2K_TRY(b2k_launch_bernoulli_pick(ctx, mind, n, rows.offset, scale, seed, r, idx_dev, n_picked_dev, cap, s));
      B2K_CUDA_OK(ctx, cudaMemcpyAsync(&np, n_picked_dev, sizeof(int), cudaMemcpyDeviceToHost, s));
      B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
      if (np <= cap) break;
      scale *= 0.75 * (double)cap / (double)np;
    }
    np = std::min(np, cap);
    if (np > 0) B2K_CUDA_OK(ctx, cudaMemcpy(picked_host.data(), idx_dev, (size_t)np * 8, cudaMemcpyDeviceToHost));
    std::sort(picked_host.begin(), picked_host.begin() + np);   // slot order -> canonical order
    // exchange: every rank learns every rank's picks (global indices), capped in total
    std::vector<int64_t> all;
    if (ctx->nranks == 1) {
      all.assign(picked_host.begin(), picked_host.begin() + np);
    } else {
      // fixed-size allgather of [count | cap indices] per rank through a dedicated exchange buffer
      int64_t* send = xchg;
      int64_t* recv = send + per;
      std::vector<int64_t> pack(per, 0);
      pack[0] = np;
      std::copy(picked_host.begin(), picked_host.begin() + np, pack.begin() + 1);
      B2K_CUDA_OK(ctx, cudaMemcpyAsync(send, pack.data(), per * 8, cudaMemcpyHostToDevice, s));
      B2K_TRY(b2k_comm_allgather_i64(ctx, send, recv, per, s));
      std::vector<int64_t> got(per * ctx->nranks);
      B2K_CUDA_OK(ctx, cudaMemcpyAsync(got.data(), recv, got.size() * 8, cudaMemcpyDeviceToHost, s));
      B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
      for (int q = 0; q < ctx->nranks; ++q) {
        int64_t c = got[q * per];
        for (int64_t i = 0; i < c; ++i) all.push_back(got[q * per + 1 + i]);
      }
      std::sort(all.begin(), all.end());
    }
    if ((int)all.size() > cap) all.resize(cap);
    if (all.empty()) continue;
    const int m = (int)all.size();
    B2K_TRY(fetch_global_rows(ctx, X, n, d, rows, all, newc, idx_dev, s));
    B2K_CUDA_OK(ctx, cudaMemcpyAsync(cand + (size_t)M * d, newc, (size_t)m * d * 4, cudaMemcpyDeviceToDevice, s));
    // nearest among the new candidates, folded into the running (min distance, nearest candidate): strict '<' keeps the
    // earlier candidate on ties, so after the last round `labels` IS the argmin over all candidates — the k-means||
    // weights need no extra pass over X
    B2K_TRY(assign_impl(ctx, pass, ox, X, n, d, newc, m, lab_new, dn, nullptr, s));
    B2K_TRY(b2k_launch_merge_chunk(ctx, mind, labels, dn, lab_new, M, n, nullptr, s));
    M += m;
  }
  if (M < k) {  // top up with distinct random rows so that M >= k (tiny inputs): these need one full assignment
    std::vector<int64_t> extra = sample_distinct(rng, rows.total, k - M + 1);
    B2K_TRY(fetch_global_rows(ctx, X, n, d, rows, extra, cand + (size_t)M * d, idx_dev, s));
    M += (int)extra.size();
    B2K_TRY(assign_impl(ctx, pass, ox, X, n, d, cand, M, labels, nullptr, nullptr, s));
  }
  // weights = #points closest to each candidate (the running argmin of the rounds)
  B2K_TRY(b2k_launch_histogram(ctx, labels, n, M, hist, s));
  if (ctx->nranks > 1) B2K_TRY(b2k_comm_allreduce_f64(ctx, hist, M, s));
  std::vector<float> P((size_t)M * d);
  std::vector<double> wts(M);
  B2K_CUDA_OK(ctx, cudaMemcpyAsync(P.data(), cand, P.size() * 4, cudaMemcpyDeviceToHost, s));
  B2K_CUDA_OK(ctx, cudaMemcpyAsync(wts.data(), hist, (size_t)M * 8, cudaMemcpyDeviceToHost, s));
  B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
  for (auto& w : wts) w = std::max(w, 1e-12);
  // candidate-to-candidate squared distances on the device (identical on every rank: same candidates, same kernel),
  // greedy weighted k-means++ on the host (table look-ups), then 10 weighted Lloyd steps on the device: the assignment
  // of the M candidates through the same kernels as any other assign pass, the weighted update in fixed order (fp64)
  std::vector<float> D2h((size_t)M * M);
  // the scratch may move: only `cand` is needed from here on, and it was copied to P above
  float *candd, *D2d, *Ck_dev;
  double* wts_dev;
  int32_t* lab_dev;
  int64_t* chosen_dev;
  B2K_TRY(carve_scratch(ctx, [&](Arena& A) -> int {
    candd = A.take<float>((size_t)M * d);
    D2d = A.take<float>((size_t)M * M);
    wts_dev = A.take<double>(M);
    Ck_dev = A.take<float>((size_t)k * d);
    lab_dev = A.take<int32_t>(M);
    chosen_dev = A.take<int64_t>(k);
    pass = A;
    return assign_room(ctx, ocand, candd, M, d, {k}, false, A);
  }));
  B2K_CUDA_OK(ctx, cudaMemcpyAsync(candd, P.data(), P.size() * 4, cudaMemcpyHostToDevice, s));
  B2K_CUDA_OK(ctx, cudaMemcpyAsync(wts_dev, wts.data(), (size_t)M * 8, cudaMemcpyHostToDevice, s));
  B2K_TRY(b2k_launch_pairwise_sqdist(ctx, candd, M, d, D2d, s));
  B2K_CUDA_OK(ctx, cudaMemcpyAsync(D2h.data(), D2d, D2h.size() * 4, cudaMemcpyDeviceToHost, s));
  B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
  std::vector<int64_t> chosen;
  reduce_candidates(D2h, wts, M, k, rng, &chosen);  // same seed + same inputs => identical on every rank
  B2K_CUDA_OK(ctx, cudaMemcpyAsync(chosen_dev, chosen.data(), (size_t)k * 8, cudaMemcpyHostToDevice, s));
  B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));  // `chosen` is pageable
  B2K_TRY(b2k_launch_gather_rows(ctx, candd, d, chosen_dev, k, Ck_dev, 0, s));
  for (int it = 0; it < 10; ++it) {
    B2K_TRY(assign_impl(ctx, pass, ocand, candd, M, d, Ck_dev, k, lab_dev, nullptr, nullptr, s));
    B2K_TRY(b2k_launch_weighted_update(ctx, candd, wts_dev, lab_dev, M, d, k, Ck_dev, s));
  }
  B2K_CUDA_OK(ctx, cudaMemcpyAsync(C, Ck_dev, (size_t)k * d * 4, cudaMemcpyDeviceToDevice, s));
  B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
  return B2K_OK;
}

// ------------------------------------------------------------------------------------------------
// fit
// ------------------------------------------------------------------------------------------------
extern "C" int b2k_kmeans_fit(b2k_ctx* ctx, const float* X, int64_t n_local, int d, int k, int init_mode,
                              const float* init_centers, int max_iter, double tol, uint64_t seed,
                              double oversampling, int n_init, float* centers_out, int* n_iter_out,
                              double* inertia_out, uintptr_t stream) {
  B2K_TRY(check_shape(ctx, "b2k_kmeans_fit", X, n_local, d, k));
  if (!centers_out) return b2k_fail(ctx, B2K_ERR_INVALID, "b2k_kmeans_fit: centers_out is NULL");
  if (n_init != 1)
    return b2k_fail(ctx, B2K_ERR_UNSUPPORTED, "b2k_kmeans_fit: n_init must be 1 (the reference forces n_init=1)");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  B2K_CUDA_OK(ctx, cudaSetDevice(ctx->device));
  {
    // reference: core.py:959-962 "A python worker received no data".  With a communicator the decision is taken on the
    // allgathered sizes, so that every rank fails together instead of one rank leaving its peers in a collective.
    Rows rows;
    B2K_TRY(gather_sizes(ctx, n_local, &rows, s));
    for (int r = 0; r < ctx->nranks; ++r)
      if (rows.sizes[r] == 0)
        return b2k_fail(ctx, B2K_ERR_INVALID, "b2k_kmeans_fit: empty partition (rank " + std::to_string(r) +
                                                  " has n_local == 0)");
  }
  B2kNormScope norms{X, n_local};
  switch (init_mode) {
    case B2K_INIT_ARRAY:
      if (!init_centers) return b2k_fail(ctx, B2K_ERR_INVALID, "b2k_kmeans_fit: init_centers is NULL");
      if (init_centers != centers_out)
        B2K_CUDA_OK(ctx, cudaMemcpyAsync(centers_out, init_centers, (size_t)k * d * 4, cudaMemcpyDeviceToDevice, s));
      break;
    case B2K_INIT_RANDOM:
      B2K_TRY(init_random(ctx, X, n_local, d, k, seed, centers_out, s));
      break;
    case B2K_INIT_KMEANS_PARALLEL:
      B2K_TRY(init_kmeans_parallel(ctx, X, n_local, d, k, seed, oversampling > 0 ? oversampling : 2.0, &norms,
                                   centers_out, s));
      break;
    default:
      return b2k_fail(ctx, B2K_ERR_INVALID, "b2k_kmeans_fit: unknown init_mode");
  }
  int lloyd_path;
  B2K_TRY(lloyd_impl(ctx, X, n_local, d, k, centers_out, max_iter, tol, &norms, n_iter_out, nullptr, &lloyd_path, s));
  if (inertia_out) {
    // the inertia pass follows the path the Lloyd loop ended on (see lloyd_impl: adaptive_path)
    const PassOpts o{lloyd_path, false, &norms};
    double* cost_dev;
    Arena pass;
    B2K_TRY(carve_scratch(ctx, [&](Arena& A) -> int {
      cost_dev = A.take<double>(1);
      pass = A;
      return assign_room(ctx, o, X, n_local, d, {k}, true, A);
    }));
    B2K_TRY(assign_impl(ctx, pass, o, X, n_local, d, centers_out, k, nullptr, nullptr, cost_dev, s));
    if (ctx->nranks > 1) B2K_TRY(b2k_comm_allreduce_f64(ctx, cost_dev, 1, s));
    B2K_CUDA_OK(ctx, cudaMemcpyAsync(inertia_out, cost_dev, 8, cudaMemcpyDeviceToHost, s));
    B2K_CUDA_OK(ctx, cudaStreamSynchronize(s));
  }
  return B2K_OK;
}
