/*
 * b2kmeans.h — C ABI of libb2kmeans.so: the B200-native (sm_100a) KMeans Lloyd-loop backend that
 * replaces the cuML calls on spark-rapids-ml's distributed KMeans.fit() path.
 *
 * Reference interfaces each entry point stands in for (paths relative to the reference repo
 * NVIDIA/spark-rapids-ml @ c51743bb, python/src/spark_rapids_ml/):
 *
 *   b2k_ctx_create/destroy      core.py:390-407 (_set_gpu_device) + cuml_context.py:68 (Handle)
 *   b2k_comm_unique_id          cuml_context.py:75-81   (nccl.get_unique_id on rank 0)
 *   b2k_comm_init               cuml_context.py:123-131 (nccl.init + inject_comms_on_handle)
 *   b2k_comm_destroy / _abort   cuml_context.py:158-175 (destroy, or abort when an exception is in flight)
 *   b2k_ingest_append           core.py:907-941 (per-Arrow-batch np.array(list(...))) +
 *                               utils.py:358-400 (_concat_and_free) + utils.py:452-522 (reserved buffer)
 *   b2k_kmeans_fit              clustering.py:383-425 (KMeansMG(handle, **cuml_init).fit(X) and the
 *                               cluster_centers_/n_iter_/inertia_ attribute reads)
 *   b2k_kmeans_lloyd            the Lloyd loop inside the above (EXTERNAL cuML: minClusterAndDistance,
 *                               reduce_rows_by_key, allreduce x2, divide, convergence) — also the unit
 *                               bench.py times as one "step" per iteration
 *   b2k_kmeans_assign           clustering.py:582-602 (KMeans.predict with injected cluster_centers_)
 *
 * Conventions
 *   - Plain C, no exceptions across the boundary: every call returns a b2k_status; the message for the
 *     last failure on a context is b2k_last_error(ctx) (ctx == NULL: last failure of a call that has no
 *     context, e.g. b2k_ctx_create).
 *   - All device pointers are BORROWED from the caller (torch tensors on the Python side); the library owns
 *     only its scratch, TMA descriptors, pinned staging and the NCCL communicator, all inside the ctx.
 *   - `stream` is a cudaStream_t passed as uintptr_t (0 = legacy default stream).  All device work is
 *     enqueued on it.  Calls that return host values (fit, lloyd) synchronise that stream before returning.
 *   - One context per process per GPU; NOT thread-safe (callers are single-threaded Spark Python workers).
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails with B2K_ERR_CUDA.
 */
#ifndef B2KMEANS_H_
#define B2KMEANS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2K_VERSION 100 /* 0.1.0 */
#define B2K_UNIQUE_ID_BYTES 128

typedef struct b2k_ctx b2k_ctx;

typedef enum b2k_status {
  B2K_OK = 0,
  B2K_ERR_INVALID = 1,     /* bad argument */
  B2K_ERR_CUDA = 2,        /* CUDA runtime/driver error (message has the cudaError string) */
  B2K_ERR_NCCL = 3,        /* NCCL error or libnccl not loadable */
  B2K_ERR_UNSUPPORTED = 4, /* shape/dtype/layout not supported by the requested kernel path */
  B2K_ERR_STATE = 5,       /* e.g. comm already initialised / not initialised */
  B2K_ERR_NOMEM = 6
} b2k_status;

/* cuml_init["init"] after the reference's param mapping (clustering.py:86-98,134): "scalable-k-means++"
 * (Spark "k-means||"), "random", or an injected array (used by every parity test). */
typedef enum b2k_init_mode {
  B2K_INIT_ARRAY = 0,
  B2K_INIT_RANDOM = 1,
  B2K_INIT_KMEANS_PARALLEL = 2
} b2k_init_mode;

typedef enum b2k_dtype {
  B2K_F32 = 0,
  B2K_F64 = 1,
  B2K_I8 = 2,
  B2K_I16 = 3,
  B2K_I32 = 4,
  B2K_I64 = 5
} b2k_dtype;

/* Host layouts the Spark->worker Arrow stream delivers (core.py:907-916):
 *   ROWS    : one contiguous [n_b, d] row-major values buffer — the child buffer of an Arrow
 *             list<T>/fixed_size_list<T> column; `offsets` (n_b+1 int32, may be NULL for fixed_size_list)
 *             is validated for a constant row length d.
 *   COLUMNS : d separate scalar columns; `values` is a const void* const[d] array of column buffers. */
typedef enum b2k_layout { B2K_LAYOUT_ROWS = 0, B2K_LAYOUT_COLUMNS = 1 } b2k_layout;

/* Values for the "kernel_path" option. AUTO picks the tcgen05 fused kernel when the shape fits it. */
typedef enum b2k_kernel_path {
  B2K_PATH_AUTO = 0,
  B2K_PATH_GENERIC = 1, /* SIMT fp32 tiles: any (k, d) */
  B2K_PATH_TCGEN05 = 2  /* TMA + tcgen05 fused assign+update (3xTF32 for k, d <= 128; 1xTF32 screening + exact
                           recheck for k, d <= 256); fails with UNSUPPORTED otherwise */
} b2k_kernel_path;

/* Per-fit statistics (b2k_get_stats): what ran, for tests and bench.py's gpu_launches claim. */
typedef struct b2k_stats {
  int64_t kernel_launches;     /* kernels of this library launched since ctx creation / last reset */
  int64_t fused_tc_launches;   /* ... of which the tcgen05 fused assign+update kernel */
  int64_t generic_launches;    /* ... of which generic assign/update kernels */
  int64_t nccl_allreduces;     /* collectives issued */
  int32_t last_path;           /* b2k_kernel_path actually used by the last fit/lloyd/assign */
  int32_t last_n_iter;
  double last_fused_ms;        /* mean device time of the fused kernel over the last lloyd call (CUDA events
                                  on the caller's stream; 0 unless option "time_kernels" is 1) */
  double last_loop_ms;         /* device time of the whole last Lloyd loop (same condition) */
  double last_reduce_ms;       /* option "time_kernels" = 2: mean device time per iteration of the partial fold, ... */
  double last_allreduce_ms;    /* ... of the NCCL allreduce of the [k*d+k+1] buffer (0 on one rank), ... */
  double last_finalize_ms;     /* ... and of finalize */
  int64_t recheck_rows;        /* large-shape kernel (k, d <= 256: 1xTF32 screening): rows of the last lloyd/assign call
                                  whose approximate margin was below the proven error bound and were re-decided
                                  exactly (summed over its passes; 0 unless option "collect_recheck" is 1) */
  int64_t recheck_candidates;  /* ... exact candidate distances evaluated for them */
  int64_t path_switch_iter;    /* iteration from which the last Lloyd loop left the large-shape tcgen05 kernel for the
                                  generic kernels because most rows needed the exact fix-up (option "adaptive_path",
                                  default 1; only with kernel_path = auto); -1 = it did not */
} b2k_stats;

int b2k_version(void);
const char* b2k_last_error(const b2k_ctx* ctx);

int b2k_ctx_create(int device, b2k_ctx** out);
int b2k_ctx_destroy(b2k_ctx* ctx);
/* Options: "kernel_path" (b2k_kernel_path), "time_kernels" (0/1/2: CUDA events around every fused launch; 2 = also
 * around the partial fold, the allreduce and finalize), "check_every" (iterations between host
 * convergence polls, default 4), "collect_recheck"
 * (1 = lloyd/assign synchronise and fill b2k_stats.recheck_*), "adaptive_path" (see b2k_stats.path_switch_iter), "ingest_threads" (host threads of the pageable -> pinned
 * staging copy of b2k_ingest_append; 0 = default: 4, capped by half of the CPUs the process may use).  Any other key
 * fails with B2K_ERR_INVALID. */
int b2k_ctx_set_option(b2k_ctx* ctx, const char* key, int64_t value);
int b2k_get_stats(const b2k_ctx* ctx, b2k_stats* out);
int b2k_reset_stats(b2k_ctx* ctx);

/* ---- communicator (NCCL over NVLink; one rank per process per GPU) ---- */
int b2k_comm_unique_id(char out[B2K_UNIQUE_ID_BYTES]); /* rank 0 only */
int b2k_comm_init(b2k_ctx* ctx, int nranks, int rank, const char uid[B2K_UNIQUE_ID_BYTES]);
int b2k_comm_destroy(b2k_ctx* ctx);
int b2k_comm_abort(b2k_ctx* ctx); /* callable after a CUDA/NCCL error; never blocks on peers */

/* ---- ingest: host Arrow batch -> rows [row0, row0+n_b) of the device matrix dst[n_max, d] (f32, row-major).
 * Stages through pinned memory, converts/transposes on the device (coalesced, vectorised).  Rejects a
 * non-constant row length.  *rows_written receives n_b.  Asynchronous with respect to the host except for
 * the staging copy; ordered on `stream`. ---- */
int b2k_ingest_append(b2k_ctx* ctx, float* dst, int64_t n_max, int d, int64_t row0, const void* values,
                      const int32_t* offsets, int64_t n_b, int src_dtype, int layout, uintptr_t stream,
                      int64_t* rows_written);

/* ---- fit: init + Lloyd loop + (optional) inertia against the final centers.
 *   X              device f32 [n_local, d] row-major (this rank's partition)
 *   init_centers   device f32 [k, d] when init_mode == B2K_INIT_ARRAY (identical on all ranks), else NULL
 *   tol            stop when sum_j ||c_j_new - c_j_old||^2 < tol; the caller maps tol==0 to float32 tiny
 *                  exactly as the reference does (clustering.py:113-123)
 *   n_init         must be 1 (the reference forces n_init=1, clustering.py:316-319)
 *   centers_out    device f32 [k, d]
 *   n_iter_out, inertia_out   host; inertia_out may be NULL (skips the extra assign pass)
 * Collective across the communicator when one is initialised: every rank must call it. ---- */
int b2k_kmeans_fit(b2k_ctx* ctx, const float* X, int64_t n_local, int d, int k, int init_mode,
                   const float* init_centers, int max_iter, double tol, uint64_t seed, double oversampling,
                   int n_init, float* centers_out, int* n_iter_out, double* inertia_out, uintptr_t stream);

/* ---- the Lloyd loop alone, in place on device centers[k,d]: at most max_iter iterations of
 * {assign + per-cluster partial sums (one pass over X), allreduce(sum,count), finalize, convergence}.
 * shift_out (host, may be NULL) receives the last sum_j||dc_j||^2. ---- */
int b2k_kmeans_lloyd(b2k_ctx* ctx, const float* X, int64_t n_local, int d, int k, float* centers,
                     int max_iter, double tol, int* n_iter_out, double* shift_out, uintptr_t stream);

/* ---- assign-only (KMeansModel.transform / predict): labels_out device int32 [n]; mindist_out device f32 [n]
 * or NULL.  Ties -> lowest center index. Asynchronous on `stream`. ---- */
int b2k_kmeans_assign(b2k_ctx* ctx, const float* X, int64_t n, int d, const float* centers, int k,
                      int32_t* labels_out, float* mindist_out, uintptr_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B2KMEANS_H_ */
