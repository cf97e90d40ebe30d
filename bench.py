#!/usr/bin/env python
"""bench.py — KMeans.fit() Lloyd-loop throughput on B200 (BASELINE.json metric), one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (sm_100a kernels via the C ABI)
  python bench.py --impl reference [--gpus N] [--steps K] ...    # CPU arm: the oracle port on host cores
  python bench.py ... --dump-outputs DIR                         # also write the timed loop's results as DIR/*.npy

A "step" is ONE Lloyd iteration over this rank's resident partition: fused assign+partial-sum pass over X,
fixed-order partial reduce, NCCL allreduce of the [k*d sums | k counts | cost] buffer (N>1), finalize.

Headline line (every N, so that the driver's 1/2/4/8 series is one workload): BASELINE.json configs[1] PER GPU
(k=64, n=10M rows/GPU, d=128, float32; weak scaling).  The same run also measures BASELINE configs[2]'s shape
(k=256, d=256, 12.5M rows/GPU — the 8-GPU config of the north star) and reports it under "cfg3" in the same JSON
line, with its own roofline (HBM and tf32 tensor bounds) — see DESIGN.md "Measurement".
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import os



def _usable_host_cores():
    """CPUs this process may actually use: the affinity mask capped by the cgroup CPU quota (this pool's boxes show 128
    CPUs in the mask with cpu.max = 16 cores: 128 OpenMP threads then run 4x SLOWER than 16 — tools/cpu_arm_probe.py)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    note = f"{n} CPUs in the affinity mask"
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            q = max(1, int(int(quota) / int(period)))
            if q < n:
                note = f"cgroup cpu.max = {q} cores of {n} visible CPUs"
                n = q
    except Exception:
        pass
    return n, note


_HOST_CORES, _HOST_CORES_NOTE = _usable_host_cores()   # the CPU arm sets its thread count explicitly (torchrun exports
                                                        # OMP_NUM_THREADS=1, which stays in force for torch itself)

import argparse
import json
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (n_per_gpu, d, k)
    "cfg2": (10_000_000, 128, 64),
    "cfg3": (12_500_000, 256, 256),
    "small": (1_000_000, 128, 64),
}
METRIC = "kmeans_fit_samples_per_sec"
UNIT = "samples/s"
# tcgen05 kind::tf32 peak measured with tools/microbench/mma_rate.cu on this pool's B200 (N = 256: 143 cycles per
# 128 x 256 x 8 MMA per SM = 3666 flop/cycle/SM; x 148 SMs x 1.965 GHz), DESIGN.md 4.1 item 3
TF32_PEAK_TFLOPS = 3666.0 * 148 * 1.965e9 / 1e12


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="Lloyd iterations of each timed region of the headline loop (the cfg3 sub-record and the "
                         "power-capped run have their own --cfg3-steps / --long-steps)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--n-per-gpu", type=int, default=0, help="override rows per GPU")
    ap.add_argument("--kernel-path", default="auto", choices=["auto", "generic", "tcgen05"])
    ap.add_argument("--init", default="auto", choices=["auto", "first_k", "near_true", "kmeans||"],
                    help="initial centres of the timed Lloyd loop: the first k rows of rank 0 (cfg2 default), the "
                         "generating centres + 0.25 sigma noise, or the library's own k-means|| initialiser — the "
                         "estimator's default initMode (cfg3 default)")
    ap.add_argument("--probe", type=int, default=0, help="diagnostic builds only (B2K_LIB=libb2kmeans_probe.so)")
    ap.add_argument("--e2e-iters", type=int, default=20, help="maxIter of the end-to-end fit (Spark default 20)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg3", action="store_true", help="skip the cfg3-shape sub-record")
    ap.add_argument("--cfg3-steps", type=int, default=20)
    ap.add_argument("--long-steps", type=int, default=200, help="second timed loop for the power-capped regime (0 = skip)")
    ap.add_argument("--cpu-sample-rows", type=int, default=1_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed Lloyd loops returned in their last step as "
                         "DIR/<name>.npy (float32 / float64), so that two builds can be compared output for output: "
                         "the headline loop after --steps iterations, cfg3_* after --cfg3-steps")
    return ap.parse_args()


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each array as out_dir/<name>.npy; the inputs are seeded, so the same arguments give the same inputs."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_per_launch(tag: str, workload_rows: int, d: int):
    """dram bytes per launch of the fused kernel from the committed ncu summary (profiles/), scaled to this n.
    NOT measured in this run: the source file is named beside the number."""
    for name in (f"r02_{tag}_ncu_summary.json", "fused_kernel_ncu_summary.json"):
        p = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(p):
            continue
        try:
            j = json.load(open(p))
            if int(j.get("d", d)) != d:
                continue
            return float(j["dram_bytes_per_row"]) * workload_rows, f"profiles/{name} (ncu --set full, scaled by n)"
        except Exception:
            continue
    return None, None


class ClockSampler:
    """Samples SM clock / throttle reasons with NVML during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if bit and (r & bit):
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        if self.ok:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr:
            self._stop.set()
            self._thr.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# CPU arms (reported baselines, never the thing optimised)
# ------------------------------------------------------------------------------------------------
_CPU_SAMPLE = {}


def host_cores() -> int:
    return _HOST_CORES


def cpu_sample(n_rows: int, d: int, k: int, seed: int = 1234):
    """Host blobs of the benchmark's shape (k centres ~ U(-10,10)^d, unit-variance noise), generated once per process."""
    import numpy as np

    key = (n_rows, d, k, seed)
    if key not in _CPU_SAMPLE:
        rng = np.random.default_rng(seed)
        centers = rng.uniform(-10.0, 10.0, size=(k, d)).astype(np.float32)
        X = rng.standard_normal(size=(n_rows, d), dtype=np.float32)
        X += centers[rng.integers(0, k, size=n_rows)]
        _CPU_SAMPLE.clear()
        _CPU_SAMPLE[key] = np.ascontiguousarray(X)
    return _CPU_SAMPLE[key]


def cpu_oracle_run(n_rows: int, d: int, k: int, iters: int, threads: int, repeats: int = 3, seed: int = 1234):
    """Times the oracle's C/OpenMP Lloyd port (oracle/kmeans_oracle.c) on a bounded sample: explicit thread count,
    pages first-touched by the threads that read them, best of `repeats`.  Also returns the last run's result."""
    from oracle import c_oracle

    c_oracle.set_threads(threads)
    X = c_oracle.first_touch_copy(cpu_sample(n_rows, d, k, seed))
    C0 = X[:k].copy()
    c_oracle.lloyd(X[: min(n_rows, 2000)], C0, 1, -1.0, want_labels=False)  # warm the library
    best = None
    for _ in range(max(1, repeats)):
        t0 = time.perf_counter()
        out = c_oracle.lloyd(X, C0, iters, -1.0, want_labels=False)
        dt = time.perf_counter() - t0
        assert out["n_iter"] == iters
        best = dt if best is None else min(best, dt)
    return n_rows * iters / best, best, c_oracle.num_threads(), out


def cpu_sklearn_legs(n_rows: int, d: int, k: int, iters: int, seed: int = 1234):
    """BASELINE.md §3 substitute for pyspark.ml (absent: no pyspark/JVM): scikit-learn Lloyd from the same C0 on the
    same sample with 2 threads (local[2]) and with all cores (reference protocol bench_kmeans.py:196-256)."""
    legs = []
    try:
        import numpy as np
        from sklearn.cluster import KMeans as SkKMeans
        from threadpoolctl import threadpool_limits

        X = cpu_sample(n_rows, d, k, seed)
        C0 = X[:k].copy()
        for threads in (2, host_cores()):
            with threadpool_limits(limits=threads):
                t0 = time.perf_counter()
                import warnings

                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    km = SkKMeans(n_clusters=k, init=C0, n_init=1, algorithm="lloyd", max_iter=iters, tol=0.0).fit(X)
                dt = time.perf_counter() - t0
            legs.append({"kind": "sklearn.cluster.KMeans(algorithm='lloyd')", "threads": threads,
                         "value": n_rows * km.n_iter_ / dt, "unit": UNIT, "seconds": dt,
                         "sample": f"{n_rows} rows x {int(km.n_iter_)} iterations"})
    except Exception as ex:
        legs.append({"kind": "sklearn", "error": repr(ex)[:200]})
    try:
        import pyspark  # noqa: F401

        legs.append({"kind": "pyspark.ml.clustering.KMeans", "note": "pyspark importable: run BASELINE configs[0] separately"})
    except Exception:
        legs.append({"kind": "pyspark.ml.clustering.KMeans", "unavailable": "no pyspark / JVM in this image"})
    return legs


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, d, k = CONFIGS[args.config]
    rows = args.cpu_sample_rows
    threads = host_cores()
    cpu_oracle_run(rows, d, k, max(1, min(args.warmup, 2)), threads, repeats=1)
    val, dt, used, out = cpu_oracle_run(rows, d, k, args.steps, threads, repeats=3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"cluster_centers": out["centers"], "inertia": out["inertia"]})
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.config}: KMeans k={k} d={d} float32 blobs; each step = one Lloyd "
                               f"iteration over a bounded {rows}-row sample on host cores (same sample at every N)",
                   "k": k, "d": d, "sample_rows": rows},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": used, "kind": "port",
                         "sample": f"{rows} rows x {args.steps} Lloyd iterations, oracle/kmeans_oracle.c (OpenMP, "
                                   f"{used} threads set explicitly = {_HOST_CORES_NOTE}, parallel first touch, best of 3)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "pyspark.ml.clustering.KMeans (BASELINE configs[0]) cannot run here: no pyspark/JVM in the image; "
                "the reference's GPU arithmetic (cuML) is absent too, so the CPU arm is the oracle port",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class _DistBarrierContext:
    """BarrierTaskContext facade over torch.distributed for CumlContext's uid exchange (cuml_context.py:75-81)."""

    def __init__(self, dist, rank, world):
        self._dist, self._rank, self._world = dist, rank, world

    def partitionId(self):
        return self._rank

    def allGather(self, message: str = ""):
        out = [None] * self._world
        self._dist.all_gather_object(out, message)
        return out

    def barrier(self):
        self._dist.barrier()


def make_blobs_device(torch, dev, n_local, d, k, rank):
    g = torch.Generator(device=dev).manual_seed(42)
    centers_true = torch.rand((k, d), generator=g, device=dev) * 20.0 - 10.0
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    X = torch.empty((n_local, d), dtype=torch.float32, device=dev)
    chunk = 1_000_000
    for s in range(0, n_local, chunk):
        e = min(n_local, s + chunk)
        z = torch.randint(0, k, (e - s,), generator=g, device=dev)
        X[s:e] = centers_true[z] + torch.randn((e - s, d), generator=g, device=dev)
    return X, centers_true


def timed_lloyd(torch, dist, ctx, X, C0, steps, dev, world, local_rank, sample_clocks=True):
    """K Lloyd iterations, device-timed (CUDA events on the launching stream), max over ranks."""
    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    C = C0.clone()
    ctx.reset_stats()
    sampler = ClockSampler(local_rank) if sample_clocks else None
    barrier()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.set_option("time_kernels", 2)   # CUDA events around every fused launch / fold / allreduce / finalize of THIS loop
    ctx.set_option("collect_recheck", 1)
    if world > 1:
        # synchronised start: the ranks' hosts leave a collective barrier up to milliseconds apart (OS scheduling), and
        # that skew would be charged to the first allreduce; all ranks spin to one wall-clock instant (same host)
        tgt = torch.tensor([time.time() + 0.02], dtype=torch.float64, device=dev)
        dist.broadcast(tgt, 0)
        tgt = float(tgt.item())
        while time.time() < tgt:
            pass
    e0.record()
    t_enter = time.time()
    n_iter, shift = ctx.kmeans_lloyd(X, C, steps, -1.0)
    t_exit = time.time()
    e1.record()
    if os.environ.get("B2K_DEBUG_TIMING"):
        print(f"[bench rank {os.environ.get('RANK', '0')}] enter {t_enter % 100:.6f} exit {t_exit % 100:.6f}", file=sys.stderr, flush=True)
    torch.cuda.synchronize(dev)
    ctx.set_option("time_kernels", 0)
    ctx.set_option("collect_recheck", 0)
    clocks = sampler.stop() if sampler else None
    barrier()
    assert n_iter == steps, (n_iter, steps)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), ctx.stats(), clocks, shift, C


def timed_lloyd_median(torch, dist, ctx, X, C0, steps, dev, world, local_rank, repeats=3):
    """`repeats` back-to-back timed regions of exactly K steps each (every one bracketed by barrier + synchronize, device
    timed, max over ranks); the MEDIAN region is reported and all of them are listed.  A single region on a shared host
    occasionally absorbs a multi-millisecond scheduling hiccup of one rank's process (seen at N=2: 1.19 / 1.63 / 1.19)."""
    runs = [timed_lloyd(torch, dist, ctx, X, C0, steps, dev, world, local_rank) for _ in range(max(1, repeats))]
    order = sorted(range(len(runs)), key=lambda i: runs[i][0])
    mid = order[len(order) // 2]
    return runs[mid], [r[0] / steps for r in runs]


def roofline_record(st, n_local, d, k, kernel, peak, peak_src, tag):
    """Roofline of the dominant kernel from the live per-launch CUDA-event times of the timed loop itself."""
    if st["last_fused_ms"] <= 0:
        return None
    alg_bytes = 4.0 * n_local * d  # X read once (SURVEY.md 8d); partial flush and row norms are < 1 %
    t = st["last_fused_ms"] / 1e3
    hbm = alg_bytes / t / 1e9
    flops = 2.0 * n_local * d * k
    tf = flops / t / 1e12
    traffic, traffic_src = ncu_traffic_per_launch(tag, n_local, d)
    hbm_frac, tf_frac = hbm / peak, tf / TF32_PEAK_TFLOPS
    bound = "hbm" if hbm_frac >= tf_frac else "tensor"
    return {"bound": bound, "kernel": kernel, "achieved": hbm if bound == "hbm" else tf,
            "peak": peak if bound == "hbm" else TF32_PEAK_TFLOPS, "unit": "GB/s" if bound == "hbm" else "TFLOP/s",
            "frac": max(hbm_frac, tf_frac),
            "bounds": {"hbm": {"achieved_gbs": hbm, "peak_gbs": peak, "frac": hbm_frac},
                       "tf32": {"achieved_tflops_1x": tf, "peak_tflops": TF32_PEAK_TFLOPS, "frac": tf_frac,
                                "peak_source": "tools/microbench/mma_rate.cu (tcgen05 kind::tf32, N=256), DESIGN.md 4.1"},
                       "rule": "the kernel's floor is max(t_hbm, t_tf32): frac = max of the two fractions"},
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "kernel_ms": st["last_fused_ms"], "loop_ms_per_iter": st["last_loop_ms"] / max(1, st["last_n_iter"]),
            "step_breakdown_ms": {"fused_pass(+centre prep)": st["last_fused_ms"], "partial_fold": st["last_reduce_ms"],
                                  "allreduce": st["last_allreduce_ms"], "finalize": st["last_finalize_ms"]},
            "algorithmic_bytes_per_launch": alg_bytes, "tensor_flops_per_launch": flops,
            "recheck_rows_per_iter": st["recheck_rows"] / max(1, st["last_n_iter"]),
            "recheck_candidates_per_iter": st["recheck_candidates"] / max(1, st["last_n_iter"])}


def parity_check(torch, dist, ctx, dev, rank, world):
    """N>1: a small sharded problem replayed on all ranks against the single-rank fp64 oracle (rank 0 holds all rows)."""
    import numpy as np

    from oracle import kmeans_oracle as ko

    n, d, k, iters = 4096 * world, 64, 16, 4
    Xall, ctr = ko.make_blobs(n, d, k, seed=5)
    C0 = (ctr + 0.25 * np.random.default_rng(0).normal(size=ctr.shape)).astype(np.float32)
    lo, hi = rank * (n // world), (rank + 1) * (n // world)
    Xd = torch.from_numpy(Xall[lo:hi]).to(dev)
    C = torch.from_numpy(C0).to(dev)
    n_it, _ = ctx.kmeans_lloyd(Xd, C, iters, -1.0)
    ok = n_it == iters
    err = None
    if rank == 0:
        ref = ko.lloyd([Xall], C0, iters, -1.0)
        err = ko.max_center_rel_err(C.cpu().numpy(), ref["centers"])
        ok = ok and err <= 1e-4
    # every rank must hold the same model (core.py:996-1003)
    Cs = [torch.empty_like(C) for _ in range(world)]
    dist.all_gather(Cs, C)
    same = all(torch.equal(Cs[0], c) for c in Cs)
    flag = torch.tensor([1 if (ok and same) else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item()), err


def ingest_record(torch, ctx, dev):
    """GB/s of b2k_ingest_append (source bytes) for the three host layouts Spark delivers, 10 000-row batches."""
    import numpy as np

    out = {}
    n_b, d, nb = 10_000, 128, 40
    rng = np.random.default_rng(0)
    dst = torch.empty((n_b * nb, d), dtype=torch.float32, device=dev)
    off = (np.arange(n_b + 1) * d).astype(np.int32)
    cases = {
        "list<float>": [rng.standard_normal((n_b, d), dtype=np.float32).reshape(-1) for _ in range(4)],
        "list<double>": [rng.standard_normal((n_b, d)).reshape(-1) for _ in range(4)],
    }
    for name, bufs in cases.items():
        for rep in range(2):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for i in range(nb):
                ctx.ingest_rows(dst, i * n_b, bufs[i % 4], d, offsets=off)
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
        out[name] = {"gb_per_s": nb * bufs[0].nbytes / dt / 1e9, "batch_rows": n_b, "d": d}
    cols = [rng.standard_normal(n_b).astype(np.float32) for _ in range(d)]
    for rep in range(2):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for i in range(nb):
            ctx.ingest_columns(dst, i * n_b, cols)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
    out["columnar(float x d)"] = {"gb_per_s": nb * n_b * d * 4 / dt / 1e9, "batch_rows": n_b, "d": d}
    return out


def main():
    # the benchmark leaves the tree it runs from as it found it: no bytecode caches of the modules it imports either
    sys.dont_write_bytecode = True
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch

    from spark_rapids_ml_b200 import _native

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the KMeans path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist  # type: ignore

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    n_local, d, k = CONFIGS[args.config]
    if args.n_per_gpu:
        n_local = args.n_per_gpu
    n_total = n_local * world

    # communicator through the reference's own protocol: CumlContext (uid from rank 0 over the barrier allGather)
    from spark_rapids_ml_b200.common.cuml_context import CumlContext

    cc = CumlContext(rank, world, _DistBarrierContext(dist, rank, world) if world > 1 else None, enable=True,
                     device=local_rank)
    cc.__enter__()
    ctx = cc.handle
    ctx.set_option("kernel_path", {"auto": 0, "generic": 1, "tcgen05": 2}[args.kernel_path])
    if args.probe:
        ctx.set_option("probe", args.probe)
    peak, peak_src = measured_peaks()

    def pick_init(name, cfg, X, centers_true, kk, dd):
        mode = name if name != "auto" else ("kmeans||" if cfg == "cfg3" else "first_k")
        if mode == "near_true":
            g0 = torch.Generator(device=dev).manual_seed(7)
            C0 = (centers_true + 0.25 * torch.randn((kk, dd), generator=g0, device=dev)).contiguous()
        elif mode == "kmeans||":
            # the estimator's default initMode (clustering.py:86-98): the library's k-means|| (collective), not timed
            C0 = ctx.kmeans_fit(X, kk, init="k-means||", max_iter=0, tol=1e-4, seed=1, compute_inertia=False)[
                "cluster_centers_"]
        else:
            C0 = X[:kk].clone()
        if world > 1:
            dist.broadcast(C0, 0)
        return C0.contiguous(), mode

    # ---------------- headline workload ----------------
    X, centers_true = make_blobs_device(torch, dev, n_local, d, k, rank)
    C0, init_mode = pick_init(args.init, args.config, X, centers_true, k, d)
    ctx.kmeans_lloyd(X, C0.clone(), max(args.warmup, 3), -1.0)          # warm-up
    (ms, st, clocks, shift, C_out), rep_ms = timed_lloyd_median(torch, dist, ctx, X, C0, args.steps, dev, world,
                                                                local_rank)
    # every timed region starts from C0, so these are the centres after exactly --steps Lloyd iterations
    outputs = {"cluster_centers": C_out.cpu().numpy(), "shift": shift}
    del C_out
    launches = int(st["kernel_launches"])
    path = {1: "generic", 2: "tcgen05"}.get(st["last_path"], "?")
    value = n_total * args.steps / (ms / 1e3)
    kernel_name = "k_fused_t (1xTF32 + recheck)" if (k > 128 or d > 128) else "k_fused_assign_update (3xTF32)"
    roofline = roofline_record(st, n_local, d, k, kernel_name, peak, peak_src, args.config)
    if roofline is None:  # generic path: time one assign+update iteration as a whole
        ach = 4.0 * n_local * d / (ms / args.steps / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": "generic assign+update (2 passes over X)", "achieved": ach, "peak": peak,
                    "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src}
    if args.long_steps and args.long_steps > args.steps:
        # the power-capped regime: a run long enough to sit at the 1 kW cap (sw_power_cap), same kernel
        ms_l, st_l, clocks_l, _, _ = timed_lloyd(torch, dist, ctx, X, C0, args.long_steps, dev, world, local_rank)
        rl = roofline_record(st_l, n_local, d, k, kernel_name, peak, peak_src, args.config)
        roofline["long_run"] = {"steps": args.long_steps, "ms_per_step": ms_l / args.long_steps,
                                "kernel_ms": rl["kernel_ms"] if rl else None, "frac": rl["frac"] if rl else None,
                                "clocks": clocks_l}

    parity = None
    if world > 1:
        ok, err = parity_check(torch, dist, ctx, dev, rank, world)
        parity = {"parity_ok": ok, "center_rel_err_vs_single_rank_oracle": err,
                  "what": "4096 rows/rank, d=64, k=16, 4 Lloyd iterations: every rank holds the same centres and "
                          "rank 0's match the fp64 oracle run on all rows (<= 1e-4)"}

    # ---------------- end to end ----------------
    e2e = None
    e2e_cabi = None
    ingest = None
    if not args.no_e2e:
        try:
            # (a) C ABI with a pinned host matrix: one H2D copy + fit + centres D2H, every rank (collective fit)
            Xh = torch.empty((n_local, d), dtype=torch.float32, pin_memory=True)
            Xh.copy_(X)
            C0h = C0.cpu().pin_memory()
            torch.cuda.synchronize(dev)
            Xd = torch.empty_like(X)
            del X
            X = None
            times, iters_done = [], 0
            for rep in range(args.e2e_steps + 1):  # first rep is warm-up
                torch.cuda.synchronize(dev)
                if world > 1:
                    dist.barrier()
                t0 = torch.cuda.Event(enable_timing=True)
                t1 = torch.cuda.Event(enable_timing=True)
                t0.record()
                ctx.ingest_pinned_tensor(Xd, 0, Xh)
                C0d = C0h.to(dev, non_blocking=True)
                out = ctx.kmeans_fit(Xd, k, init=C0d, max_iter=args.e2e_iters, tol=1e-30, compute_inertia=False)
                res = out["cluster_centers_"].cpu()  # noqa: F841  D2H of the step's result
                t1.record()
                torch.cuda.synchronize(dev)
                if rep > 0:
                    times.append(t0.elapsed_time(t1))
                    iters_done = out["n_iter_"]
            t = torch.tensor([sum(times) / len(times)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())
            e2e_cabi = {"value": n_total * iters_done / (e2e_ms / 1e3), "unit": UNIT,
                        "h2d_bytes_per_step": int(n_local * d * 4 + k * d * 4), "d2h_bytes_per_step": int(k * d * 4 + 64),
                        "ms_per_fit": e2e_ms, "iterations_per_fit": iters_done,
                        "what": "b2k_ingest_append(one pinned host X) + b2k_kmeans_fit(init=array, maxIter=%d) + centres D2H"
                                % args.e2e_iters}
            del Xd
            torch.cuda.empty_cache()
            # (b) the public API: KMeans(k, maxIter, initMode).fit(df) on a frame of 10 000-row Arrow batches in pageable
            # host memory (what a Spark Python worker receives, core.py:907-941); N=1 in-process, N>1: every rank fits its
            # own shard through the same worker function with the communicator of this run
            from spark_rapids_ml_b200.clustering import KMeans
            from spark_rapids_ml_b200.sparkshim import LocalSession

            Xnp = Xh.numpy()
            if world == 1:
                sess = LocalSession()
                df = sess.from_numpy(Xnp, col="features", num_partitions=1)
                est = KMeans(k=k, maxIter=args.e2e_iters, tol=1e-30, initMode="random", seed=1, num_workers=1)
                est.setFeaturesCol("features")
                times = []
                for rep in range(2):
                    torch.cuda.synchronize(dev)
                    t0 = time.perf_counter()
                    model = est.fit(df)
                    torch.cuda.synchronize(dev)
                    times.append(time.perf_counter() - t0)
                n_it = getattr(model, "n_iter_", None) or args.e2e_iters
                dt = min(times)
                e2e = {"value": n_total * args.e2e_iters / dt, "unit": UNIT,
                       "h2d_bytes_per_step": int(n_local * d * 4), "d2h_bytes_per_step": int(k * d * 8),
                       "ms_per_fit": dt * 1e3, "iterations_per_fit": args.e2e_iters,
                       "what": "spark_rapids_ml_b200.clustering.KMeans(k=%d, maxIter=%d, initMode='random').fit(df): "
                               "LocalSession frame of %d Arrow batches x 10 000 rows (pageable host memory) -> "
                               "b2k_ingest_append per batch -> device concat -> b2k_kmeans_fit -> model rows; "
                               "wall clock, best of 2 (tol ~ 0: all %d iterations run)"
                               % (k, args.e2e_iters, (n_local + 9999) // 10000, args.e2e_iters)}
                # the same fit with the estimator's DEFAULT initMode (k-means||, clustering.py:86-98): the initialiser's
                # candidate passes are part of what a default user call pays
                est2 = KMeans(k=k, maxIter=args.e2e_iters, tol=1e-30, seed=1, num_workers=1)
                est2.setFeaturesCol("features")
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                model = est2.fit(df)
                torch.cuda.synchronize(dev)
                dt2 = time.perf_counter() - t0
                e2e["default_init_kmeans_parallel"] = {"value": n_total * args.e2e_iters / dt2, "unit": UNIT,
                                                       "ms_per_fit": dt2 * 1e3}
                # KMeansModel.transform over the same frame (SURVEY 8 f-2; what the reference benchmark reports as
                # transform_time, bench_kmeans.py:172-177): per batch ingest -> b2k_kmeans_assign -> labels back -> Arrow
                try:
                    t0 = time.perf_counter()
                    out_df = model.transform(df)
                    n_out = out_df.count()
                    torch.cuda.synchronize(dev)
                    dtt = time.perf_counter() - t0
                    e2e["transform"] = {"value": n_out / dtt, "unit": "rows/s", "seconds": dtt, "rows": int(n_out),
                                        "what": "KMeansModel.transform(df) on the same 1000-batch frame, prediction column "
                                                "materialised (count)"}
                    del out_df
                except Exception as ex:   # a side record: never lose the line over it
                    e2e["transform"] = {"error": repr(ex)[:300]}
                del df, model
            else:
                e2e = dict(e2e_cabi)
                e2e["what"] += " [N>1: the Estimator surface needs one Spark barrier stage over all ranks; under torchrun " \
                               "each rank is its own driver, so the C-ABI path is the end-to-end number here]"
            ingest = ingest_record(torch, ctx, dev)
            del Xh
        except Exception as ex:  # pinned allocation can fail on small hosts: report, do not fake
            import traceback

            e2e = {"value": None, "unit": UNIT, "error": (repr(ex) + " | " + traceback.format_exc()[-300:])[:500]}
    if X is not None:
        del X
    torch.cuda.empty_cache()

    # ---------------- BASELINE configs[2] shape (k=256, d=256, 12.5 M rows/GPU) in the same run ----------------
    cfg3 = None
    if not args.no_cfg3 and args.config != "cfg3":
        try:
            n3, d3, k3 = CONFIGS["cfg3"]
            X3, ctr3 = make_blobs_device(torch, dev, n3, d3, k3, rank)
            t_init0 = time.perf_counter()
            C03, mode3 = pick_init(args.init, "cfg3", X3, ctr3, k3, d3)
            torch.cuda.synchronize(dev)
            t_init = time.perf_counter() - t_init0
            ctx.kmeans_lloyd(X3, C03.clone(), 3, -1.0)
            (ms3, st3, clocks3, shift3, C3_out), rep3 = timed_lloyd_median(torch, dist, ctx, X3, C03, args.cfg3_steps, dev,
                                                                           world, local_rank)
            outputs["cfg3_cluster_centers"] = C3_out.cpu().numpy()
            outputs["cfg3_shift"] = shift3
            del C3_out
            cfg3 = {"value": n3 * world * args.cfg3_steps / (ms3 / 1e3), "unit": UNIT, "n_gpus": world,
                    "steps": args.cfg3_steps, "warmup": 3, "ms_per_step": ms3 / args.cfg3_steps,
                    "repeat_ms_per_step": rep3,
                    "config": {"workload": f"cfg3 shape: k={k3}, d={d3}, n={n3}/GPU x {world} GPU, float32 blobs resident in HBM",
                               "k": k3, "d": d3, "n_per_gpu": n3, "kernel_path": {1: "generic", 2: "tcgen05"}.get(st3["last_path"]),
                               "init": mode3, "init_seconds": t_init},
                    "roofline": roofline_record(st3, n3, d3, k3, "k_fused_t (1xTF32 + recheck)", peak, peak_src, "cfg3"),
                    "clocks": clocks3, "gpu_launches": int(st3["kernel_launches"]), "final_shift": shift3}
            del X3
            torch.cuda.empty_cache()
        except Exception as ex:
            cfg3 = {"error": repr(ex)[:300]}

    # ---------------- CPU baselines (rank 0, N=1 only), bounded sample ----------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rows, cpu_iters = args.cpu_sample_rows, 10
        threads = host_cores()
        val, dt, used, _ = cpu_oracle_run(rows, d, k, cpu_iters, threads, repeats=3)
        cpu_baseline = {"value": val, "unit": UNIT, "cores": used, "kind": "port",
                        "sample": f"{rows} rows x {cpu_iters} Lloyd iterations of the same blobs shape (k={k}, d={d}), "
                                  f"oracle/kmeans_oracle.c OpenMP fp64, {used} threads set explicitly = {_HOST_CORES_NOTE}, "
                                  f"parallel first touch, best of 3: {dt:.2f} s",
                        "other_legs": cpu_sklearn_legs(min(rows, 500_000), d, k, 5)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "repeat_ms_per_step": rep_ms,
            "repeats": "3 timed regions of exactly K steps each; the median region is the one reported",
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.config}: KMeans Lloyd iteration, k={k}, n={n_local}/GPU x {world} GPU, d={d}, "
                                   "float32 blobs resident in HBM; fixed 'array' init; tol<0 so every step does full work",
                       "k": k, "d": d, "n_per_gpu": n_local, "n_total": n_total, "kernel_path": path, "init": init_mode,
                       "l2": f"inputs ({n_local * d * 4 / 1e9:.2f} GB/GPU) are larger than the 126 MB L2: no flush needed",
                       "parallelism": f"dp{world} (rows sharded; one f64 allreduce of k*d+k+1 values per step)",
                       "comm_bootstrap": "CumlContext (NCCL uid from rank 0 over the barrier allGather)" if world > 1 else None},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "e2e_cabi_pinned": e2e_cabi, "ingest": ingest,
            "cfg3": cfg3, "parity": parity, "clocks": clocks, "gpu_launches": launches, "final_shift": shift,
        }
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
    cc.__exit__(None, None, None)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
