"""ctypes binding of libb2kmeans.so (the C ABI declared in include/b2kmeans.h).

PyTorch tensors are used only as device-memory containers: every call hands raw ``data_ptr()``
addresses and the current CUDA stream to the library.  There is NO fallback: if the shared library
is missing or no CUDA device is present, the compute entry points raise.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from typing import Any, Dict, Optional, Sequence, Tuple

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# B2K_LIB selects another build of the same library (e.g. one built from another revision)
LIB_PATH = os.environ.get("B2K_LIB") or os.path.join(_PKG_DIR, "libb2kmeans.so")
CSRC_DIR = os.path.join(_PKG_DIR, "csrc")

B2K_OK = 0
INIT_ARRAY, INIT_RANDOM, INIT_KMEANS_PARALLEL = 0, 1, 2
PATH_AUTO, PATH_GENERIC, PATH_TCGEN05 = 0, 1, 2
LAYOUT_ROWS, LAYOUT_COLUMNS = 0, 1
UNIQUE_ID_BYTES = 128

_DTYPE_CODES = {
    np.dtype("float32"): 0,
    np.dtype("float64"): 1,
    np.dtype("int8"): 2,
    np.dtype("int16"): 3,
    np.dtype("int32"): 4,
    np.dtype("int64"): 5,
}

# every symbol include/b2kmeans.h declares (tests check the library exports exactly these)
EXPORTED_SYMBOLS = (
    "b2k_version",
    "b2k_last_error",
    "b2k_ctx_create",
    "b2k_ctx_destroy",
    "b2k_ctx_set_option",
    "b2k_get_stats",
    "b2k_reset_stats",
    "b2k_comm_unique_id",
    "b2k_comm_init",
    "b2k_comm_destroy",
    "b2k_comm_abort",
    "b2k_ingest_append",
    "b2k_kmeans_fit",
    "b2k_kmeans_lloyd",
    "b2k_kmeans_assign",
)


class B2KError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libb2kmeans error {code}: {msg}")
        self.code = code


class Stats(ctypes.Structure):
    _fields_ = [
        ("kernel_launches", ctypes.c_int64),
        ("fused_tc_launches", ctypes.c_int64),
        ("generic_launches", ctypes.c_int64),
        ("nccl_allreduces", ctypes.c_int64),
        ("last_path", ctypes.c_int32),
        ("last_n_iter", ctypes.c_int32),
        ("last_fused_ms", ctypes.c_double),
        ("last_loop_ms", ctypes.c_double),
        ("last_reduce_ms", ctypes.c_double),
        ("last_allreduce_ms", ctypes.c_double),
        ("last_finalize_ms", ctypes.c_double),
        ("recheck_rows", ctypes.c_int64),
        ("recheck_candidates", ctypes.c_int64),
        ("path_switch_iter", ctypes.c_int64),
    ]


def build(verbose: bool = False) -> str:
    """Compile libb2kmeans.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC_DIR, "-j", "8"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("building libb2kmeans.so failed:\n" + res.stdout + "\n" + res.stderr)
    if verbose:
        print(res.stdout)
    return LIB_PATH


_lib: Optional[ctypes.CDLL] = None


def load_library() -> ctypes.CDLL:
    """Load (never build) the in-tree shared library; raises loudly when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            f"{LIB_PATH} not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C spark_rapids_ml_b200/csrc`). There is no CPU/PyTorch fallback for the KMeans path."
        )
    L = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    vp, i32, i64, u64, f64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double
    L.b2k_version.restype = i32
    L.b2k_last_error.restype = ctypes.c_char_p
    L.b2k_last_error.argtypes = [vp]
    L.b2k_ctx_create.argtypes = [i32, ctypes.POINTER(vp)]
    L.b2k_ctx_destroy.argtypes = [vp]
    L.b2k_ctx_set_option.argtypes = [vp, ctypes.c_char_p, i64]
    L.b2k_get_stats.argtypes = [vp, ctypes.POINTER(Stats)]
    L.b2k_reset_stats.argtypes = [vp]
    L.b2k_comm_unique_id.argtypes = [ctypes.c_char_p]
    L.b2k_comm_init.argtypes = [vp, i32, i32, ctypes.c_char_p]
    L.b2k_comm_destroy.argtypes = [vp]
    L.b2k_comm_abort.argtypes = [vp]
    L.b2k_ingest_append.argtypes = [vp, vp, i64, i32, i64, vp, vp, i64, i32, i32, ctypes.c_size_t,
                                    ctypes.POINTER(i64)]
    L.b2k_kmeans_fit.argtypes = [vp, vp, i64, i32, i32, i32, vp, i32, f64, u64, f64, i32, vp,
                                 ctypes.POINTER(i32), ctypes.POINTER(f64), ctypes.c_size_t]
    L.b2k_kmeans_lloyd.argtypes = [vp, vp, i64, i32, i32, vp, i32, f64, ctypes.POINTER(i32),
                                   ctypes.POINTER(f64), ctypes.c_size_t]
    L.b2k_kmeans_assign.argtypes = [vp, vp, i64, i32, vp, i32, vp, vp, ctypes.c_size_t]
    for name in EXPORTED_SYMBOLS:
        if name not in ("b2k_last_error",):
            getattr(L, name).restype = i32
    _lib = L
    return L


def comm_unique_id() -> bytes:
    """NCCL unique id (rank 0 only) — mirrors nccl.get_unique_id() in cuml_context.py:77."""
    L = load_library()
    buf = ctypes.create_string_buffer(UNIQUE_ID_BYTES)
    rc = L.b2k_comm_unique_id(buf)
    if rc != B2K_OK:
        raise B2KError(rc, (L.b2k_last_error(None) or b"").decode())
    return buf.raw


def _stream_handle(torch_mod: Any, device: Any) -> int:
    return int(torch_mod.cuda.current_stream(device).cuda_stream)


class Context:
    """One library context per process per GPU (reference: one Spark barrier task per GPU)."""

    def __init__(self, device: int = 0):
        import torch

        self._torch = torch
        self._L = load_library()
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        h = ctypes.c_void_p()
        rc = self._L.b2k_ctx_create(self.device_index, ctypes.byref(h))
        if rc != B2K_OK:
            raise B2KError(rc, (self._L.b2k_last_error(None) or b"").decode())
        self._h = h
        self.nranks = 1
        self.rank = 0

    # -- plumbing ---------------------------------------------------------------------------
    def _check(self, rc: int) -> None:
        if rc != B2K_OK:
            raise B2KError(rc, (self._L.b2k_last_error(self._h) or b"").decode())

    def _stream(self) -> int:
        return _stream_handle(self._torch, self.device)

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            self._L.b2k_ctx_destroy(self._h)
            self._h = None

    def __enter__(self) -> "Context":
        return self

    def __exit__(self, *exc: Any) -> None:
        self.close()

    def __del__(self) -> None:  # best effort
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key: str, value: int) -> None:
        self._check(self._L.b2k_ctx_set_option(self._h, key.encode(), int(value)))

    def stats(self) -> Dict[str, Any]:
        st = Stats()
        self._check(self._L.b2k_get_stats(self._h, ctypes.byref(st)))
        return {f: getattr(st, f) for f, _ in Stats._fields_}

    def reset_stats(self) -> None:
        self._check(self._L.b2k_reset_stats(self._h))

    # -- comm -------------------------------------------------------------------------------
    def comm_init(self, nranks: int, rank: int, uid: bytes) -> None:
        assert len(uid) == UNIQUE_ID_BYTES
        self._check(self._L.b2k_comm_init(self._h, int(nranks), int(rank), uid))
        self.nranks, self.rank = int(nranks), int(rank)

    def comm_destroy(self) -> None:
        self._check(self._L.b2k_comm_destroy(self._h))
        self.nranks, self.rank = 1, 0

    def comm_abort(self) -> None:
        self._check(self._L.b2k_comm_abort(self._h))
        self.nranks, self.rank = 1, 0

    # -- ingest -----------------------------------------------------------------------------
    def ingest_rows(self, dst: Any, row0: int, values: np.ndarray, d: int,
                    offsets: Optional[np.ndarray] = None, n_rows: Optional[int] = None) -> int:
        """Append a contiguous [n_b, d] host value buffer (Arrow list child buffer) at dst[row0:]."""
        code = _DTYPE_CODES.get(values.dtype)
        if code is None:
            raise TypeError(f"unsupported source dtype {values.dtype}")
        assert values.flags.c_contiguous
        if offsets is not None:
            offsets = np.ascontiguousarray(offsets, dtype=np.int32)
            n_b = offsets.shape[0] - 1
        else:
            n_b = int(n_rows) if n_rows is not None else values.size // d
            # without offsets nothing downstream can see a wrong row width: a batch whose rows are not `d` wide would make
            # the C side read past the buffer (narrower) or silently re-shape it (wider)
            if values.size != n_b * d:
                raise ValueError(f"feature batch holds {values.size} values for {n_b} rows of width {d}: "
                                 "row width differs from the expected dimension")
        wrote = ctypes.c_int64(0)
        self._check(self._L.b2k_ingest_append(
            self._h, dst.data_ptr(), int(dst.shape[0]), int(d), int(row0), values.ctypes.data,
            offsets.ctypes.data if offsets is not None else None, int(n_b), code, LAYOUT_ROWS,
            self._stream(), ctypes.byref(wrote)))
        return int(wrote.value)

    def ingest_pinned_tensor(self, dst: Any, row0: int, src: Any) -> int:
        """Append a (pinned) host torch tensor [n_b, d] f32."""
        assert src.dtype == self._torch.float32 and src.is_contiguous()
        n_b, d = int(src.shape[0]), int(src.shape[1])
        wrote = ctypes.c_int64(0)
        self._check(self._L.b2k_ingest_append(
            self._h, dst.data_ptr(), int(dst.shape[0]), d, int(row0), src.data_ptr(), None, n_b, 0,
            LAYOUT_ROWS, self._stream(), ctypes.byref(wrote)))
        return int(wrote.value)

    def ingest_columns(self, dst: Any, row0: int, columns: Sequence[np.ndarray]) -> int:
        """Append d scalar host columns (multi-column feature layout, core.py:910)."""
        d = len(columns)
        dt = columns[0].dtype
        code = _DTYPE_CODES.get(dt)
        if code is None:
            raise TypeError(f"unsupported source dtype {dt}")
        n_b = int(columns[0].shape[0])
        cols = [np.ascontiguousarray(c) for c in columns]
        for c in cols:
            if c.dtype != dt or c.shape[0] != n_b:
                raise ValueError("columns must share dtype and length")
        ptrs = (ctypes.c_void_p * d)(*[c.ctypes.data for c in cols])
        wrote = ctypes.c_int64(0)
        self._check(self._L.b2k_ingest_append(
            self._h, dst.data_ptr(), int(dst.shape[0]), d, int(row0), ctypes.addressof(ptrs), None, n_b,
            code, LAYOUT_COLUMNS, self._stream(), ctypes.byref(wrote)))
        self._torch.cuda.current_stream(self.device).synchronize()  # cols/ptrs must outlive the staging copies
        return int(wrote.value)

    # -- compute ----------------------------------------------------------------------------
    def _check_X(self, X: Any) -> Tuple[int, int]:
        t = self._torch
        if not (X.is_cuda and X.dtype == t.float32 and X.dim() == 2 and X.is_contiguous()):
            raise ValueError("X must be a contiguous float32 CUDA tensor [n, d]")
        if X.device.index != self.device_index:
            raise ValueError("X lives on a different device than this context")
        return int(X.shape[0]), int(X.shape[1])

    def kmeans_fit(self, X: Any, k: int, *, init: Any = "scalable-k-means++", max_iter: int = 300,
                   tol: float = 1e-4, seed: int = 0, oversampling_factor: float = 2.0, n_init: int = 1,
                   compute_inertia: bool = True) -> Dict[str, Any]:
        """KMeansMG(**cuml_init).fit(X) equivalent.  Returns dict(cluster_centers_ [k,d] cuda tensor,
        n_iter_, inertia_)."""
        t = self._torch
        n, d = self._check_X(X)
        init_ptr = None
        if isinstance(init, str):
            mode = {"scalable-k-means++": INIT_KMEANS_PARALLEL, "k-means||": INIT_KMEANS_PARALLEL,
                    "random": INIT_RANDOM}.get(init)
            if mode is None:
                raise ValueError(f"unknown init {init!r}")
            keep = None
        else:
            keep = t.as_tensor(init, dtype=t.float32, device=self.device).contiguous()
            if tuple(keep.shape) != (k, d):
                raise ValueError(f"init array must have shape ({k}, {d})")
            mode = INIT_ARRAY
            init_ptr = keep.data_ptr()
        centers = t.empty((k, d), dtype=t.float32, device=self.device)
        n_iter = ctypes.c_int(0)
        inertia = ctypes.c_double(0.0)
        with t.cuda.device(self.device):
            self._check(self._L.b2k_kmeans_fit(
                self._h, X.data_ptr(), n, d, int(k), mode, init_ptr, int(max_iter), float(tol),
                int(seed) & 0xFFFFFFFFFFFFFFFF, float(oversampling_factor), int(n_init), centers.data_ptr(),
                ctypes.byref(n_iter), ctypes.byref(inertia) if compute_inertia else None, self._stream()))
        del keep
        return {"cluster_centers_": centers, "n_iter_": int(n_iter.value),
                "inertia_": float(inertia.value) if compute_inertia else None}

    def kmeans_lloyd(self, X: Any, centers: Any, max_iter: int, tol: float) -> Tuple[int, float]:
        """Lloyd loop in place on `centers` (cuda f32 [k,d]); returns (n_iter, last shift)."""
        t = self._torch
        n, d = self._check_X(X)
        if not (centers.is_cuda and centers.dtype == t.float32 and centers.is_contiguous()
                and centers.shape[1] == d):
            raise ValueError("centers must be a contiguous float32 CUDA tensor [k, d]")
        n_iter = ctypes.c_int(0)
        shift = ctypes.c_double(0.0)
        with t.cuda.device(self.device):
            self._check(self._L.b2k_kmeans_lloyd(
                self._h, X.data_ptr(), n, d, int(centers.shape[0]), centers.data_ptr(), int(max_iter),
                float(tol), ctypes.byref(n_iter), ctypes.byref(shift), self._stream()))
        return int(n_iter.value), float(shift.value)

    def kmeans_assign(self, X: Any, centers: Any, want_mindist: bool = False) -> Tuple[Any, Any]:
        """KMeans.predict equivalent: int32 labels (and optionally squared min distances)."""
        t = self._torch
        n, d = self._check_X(X)
        C = t.as_tensor(centers, dtype=t.float32, device=self.device).contiguous()
        if C.dim() != 2 or C.shape[1] != d:
            raise ValueError("centers must be [k, d]")
        labels = t.empty((n,), dtype=t.int32, device=self.device)
        md = t.empty((n,), dtype=t.float32, device=self.device) if want_mindist else None
        with t.cuda.device(self.device):
            self._check(self._L.b2k_kmeans_assign(
                self._h, X.data_ptr(), n, d, C.data_ptr(), int(C.shape[0]), labels.data_ptr(),
                md.data_ptr() if md is not None else None, self._stream()))
        t.cuda.current_stream(self.device).synchronize()  # C (a temporary) must outlive the kernels
        return labels, md
