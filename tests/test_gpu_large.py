"""GPU parity tests of the large-shape fused kernel (csrc/b2k_fused_t.cu: k <= 256, d <= 256 — BASELINE cfg3's shape):
tcgen05 1xTF32 screening + proven-bound exact recheck, through the C ABI, against the fp64 oracle.

Parity rule as in test_gpu_parity.py: labels bit-exact except rows whose fp64 margin is below 1e-6;
centroids within 1e-4 relative.
"""
import numpy as np
import pytest

from oracle import kmeans_oracle as ko

pytestmark = pytest.mark.gpu
TAU = 1e-6
CENTER_RTOL = 1e-4


@pytest.fixture(scope="module")
def ctx():
    from spark_rapids_ml_b200 import _native

    c = _native.Context(0)
    c.set_option("kernel_path", 2)       # tcgen05 or fail: never a silent generic fallback
    c.set_option("collect_recheck", 1)
    yield c
    c.close()


def _dev(x):
    import torch

    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


@pytest.mark.parametrize("n,d,k,gen", [
    (128, 256, 256, "blobs"),
    (20000, 256, 256, "blobs"),          # BASELINE cfg3's (k, d)
    (5000, 256, 256, "uniform"),         # near-tie stress: about half of the rows take the exact recheck
    (3001, 256, 200, "blobs"),           # ragged last step, k < 256 (padding clusters)
    (4096, 192, 130, "uniform"),         # d not a multiple of 256: TMA zero fill
    (1000, 256, 64, "blobs"),            # k <= 128 with d > 128: the peer CTA holds only padding clusters
    (777, 132, 256, "uniform"),          # d % 32 != 0
    (64, 256, 256, "uniform"),           # fewer rows than clusters, half a step
    (1, 256, 3, "uniform"),              # single row
    (5000, 128, 200, "uniform"),         # DP = 128 instantiation (k > 128)
    (3000, 20, 100, "blobs"),            # DP = 128, d % 32 != 0, the peer CTA holds only padding clusters
])
def test_assign_large_matches_oracle(ctx, n, d, k, gen):
    X = ko.make_blobs(n, d, k, seed=7)[0] if gen == "blobs" else ko.make_uniform(n, d, seed=7)
    rng = np.random.default_rng(3)
    C = X[rng.choice(n, size=k, replace=(n < k))].copy() + (0.01 if gen == "uniform" else 0.0)
    ctx.reset_stats()
    labels, md = ctx.kmeans_assign(_dev(X), _dev(C), want_mindist=True)
    st = ctx.stats()
    assert st["last_path"] == 2 and st["fused_tc_launches"] >= 1
    cmp = ko.compare_labels(X, C, labels.cpu().numpy(), tau=TAU)
    assert cmp["n_mismatch_outside_margin"] == 0, cmp
    _, md_o, _ = ko.assign(X, C)
    # the min distance is sum (x - c)^2 in fp32 from the tile in shared memory: ~1e-6 relative
    np.testing.assert_allclose(md.cpu().numpy(), md_o, rtol=1e-4, atol=1e-6)
    if gen == "uniform" and n >= 1000:
        assert st["recheck_rows"] > 0          # the exact path actually ran
        assert st["recheck_candidates"] >= st["recheck_rows"]


def test_large_tie_break_and_duplicates(ctx):
    d, k = 256, 256
    X = ko.make_uniform(512, d, seed=1)
    C = np.repeat(X[:1], k, axis=0).copy()       # all centres identical: every row must pick index 0
    labels, _ = ctx.kmeans_assign(_dev(X), _dev(C))
    assert int(labels.max()) == 0
    C2 = X[:k].copy()
    C2[200] = C2[7]                               # duplicated centre across the two CTAs' halves: 200 never wins
    labels, _ = ctx.kmeans_assign(_dev(X), _dev(C2))
    assert int((labels == 200).sum()) == 0
    C3 = X[:k].copy()
    C3[9] = C3[3]                                 # ... and inside one warp's 32 clusters
    labels, _ = ctx.kmeans_assign(_dev(X), _dev(C3))
    assert int((labels == 9).sum()) == 0


@pytest.mark.parametrize("n,d,k,iters,gen", [
    (20000, 256, 256, 4, "blobs"),
    (6000, 256, 256, 3, "uniform"),
    (30000, 128, 160, 4, "blobs"),
    (5000, 160, 200, 3, "blobs"),
])
def test_lloyd_large_matches_oracle(ctx, n, d, k, iters, gen):
    X, ctr = ko.make_blobs(n, d, k, seed=11)
    if gen == "uniform":
        X = ko.make_uniform(n, d, seed=11)
        C0 = X[:k].copy()
    else:
        C0 = (ctr + 0.25 * np.random.default_rng(0).normal(size=ctr.shape)).astype(np.float32)
    ref = ko.lloyd([X], C0, iters, -1.0)
    C = _dev(C0)
    n_it, _ = ctx.kmeans_lloyd(_dev(X), C, iters, -1.0)
    assert n_it == iters and ctx.stats()["last_path"] == 2
    # an admissible (< 1e-6 margin) tie row may send two trajectories apart on uniform data: check one exact step too
    lab0, _, margin0 = ko.assign(X, C0)
    if gen == "blobs" or margin0.min() > 1e-5:
        assert ko.max_center_rel_err(C.cpu().numpy(), ref["centers"]) <= CENTER_RTOL
    C1, _, _ = ko.lloyd_iteration([X], C0)
    one = _dev(C0)
    ctx.kmeans_lloyd(_dev(X), one, 1, -1.0)
    if margin0.min() > 1e-5:
        assert ko.max_center_rel_err(one.cpu().numpy(), C1) <= CENTER_RTOL


def test_cfg3_shape_properties(ctx):
    """BASELINE cfg3's (k = 256, d = 256) at 1 M rows — beyond what the oracle checks row by row quickly:
    counts sum to n, one Lloyd step == fp64 sums implied by the device labels, bitwise determinism, labels of a
    20 k-row sample against the oracle, zero rechecks on separated blobs with one centre per blob."""
    import torch

    n, d, k = 1_000_003, 256, 256
    g = torch.Generator(device="cuda").manual_seed(5)
    ctr = (torch.rand((k, d), generator=g, device="cuda") * 20 - 10)
    z = torch.randint(0, k, (n,), generator=g, device="cuda")
    X = (ctr[z] + torch.randn((n, d), generator=g, device="cuda")).contiguous()
    C0 = (ctr + 0.25 * torch.randn((k, d), generator=g, device="cuda")).contiguous()
    labels, md = ctx.kmeans_assign(X, C0, want_mindist=True)
    assert ctx.stats()["last_path"] == 2
    assert ctx.stats()["recheck_rows"] == 0      # margins ~ 1.7e4 against a bound of ~70
    assert int(labels.min()) >= 0 and int(labels.max()) < k
    assert torch.equal(labels.long(), z)          # every row goes to its generating centre
    C1 = C0.clone()
    n_it, shift = ctx.kmeans_lloyd(X, C1, 1, 0.0)
    assert n_it == 1
    S = torch.zeros((k, d), dtype=torch.float64, device="cuda").index_add_(0, labels.long(), X.double())
    w = torch.bincount(labels.long(), minlength=k).double()
    exp = torch.where(w[:, None] > 0, S / w.clamp(min=1)[:, None], C0.double()).float()
    rel = ((C1 - exp).double().norm(dim=1) / exp.double().norm(dim=1)).max().item()
    assert rel <= 1e-5, rel
    assert abs(shift - float(((exp - C0).double() ** 2).sum())) <= 1e-4 * shift + 1e-12
    C2 = C0.clone()
    ctx.kmeans_lloyd(X, C2, 1, 0.0)
    assert torch.equal(C1, C2)                    # static schedule, fixed-order sums: bitwise identical reruns
    # a bad start (the first k rows: blobs with two centres, blobs with none) drives ~10 % of the rows through the recheck
    C3 = X[:k].clone()
    ctx.kmeans_lloyd(X, C3, 3, 0.0)
    assert ctx.stats()["recheck_rows"] > 0
    idx = torch.randperm(n, generator=g, device="cuda")[:20000]
    lab, _ = ctx.kmeans_assign(X[idx].contiguous(), C3)
    cmp = ko.compare_labels(X[idx].cpu().numpy(), C3.cpu().numpy(), lab.cpu().numpy(), tau=TAU)
    assert cmp["n_mismatch_outside_margin"] == 0, cmp
    C4 = X[:k].clone()
    ctx.kmeans_lloyd(X, C4, 3, 0.0)
    assert torch.equal(C3, C4)                    # ... deterministic through the recheck path as well


def test_fit_large_inertia_and_estimator_path(ctx):
    """fit() = init + Lloyd + inertia on the cfg3 (k, d): inertia from the exact min distances."""
    X, ctr = ko.make_blobs(30000, 256, 256, seed=3)
    C0 = (ctr + 0.25 * np.random.default_rng(0).normal(size=ctr.shape)).astype(np.float32)
    ref = ko.lloyd([X], C0, 5, 1e-4)
    out = ctx.kmeans_fit(_dev(X), 256, init=C0, max_iter=5, tol=1e-4)
    assert out["n_iter_"] == ref["n_iter"]
    assert ko.max_center_rel_err(out["cluster_centers_"].cpu().numpy(), ref["centers"]) <= CENTER_RTOL
    assert abs(out["inertia_"] - ref["inertia"]) <= 1e-5 * ref["inertia"]


def test_adaptive_path_leaves_the_screening_kernel_on_near_tie_data():
    """A degenerate cloud (every row within 1e-3 of one point): every row is a near-tie between all clusters for 1xTF32
    screening.  With kernel_path = auto the Lloyd loop measures the fix-up load of its first burst and runs the remaining
    iterations on the generic kernels (b2k_stats.path_switch_iter).  Blobs never switch; uniform noise may or may not,
    and stays within the parity tolerance of the oracle either way."""
    from spark_rapids_ml_b200 import _native

    n, d, k, iters = 40000, 256, 256, 12
    rng = np.random.default_rng(5)
    Xd = (1.0 + 1e-3 * rng.random((n, d))).astype(np.float32)
    c = _native.Context(0)
    try:
        c.set_option("collect_recheck", 1)
        res = {}
        for adaptive in (1, 0):
            c.set_option("adaptive_path", adaptive)
            C = _dev(Xd[:k].copy())
            n_it, _ = c.kmeans_lloyd(_dev(Xd), C, iters, -1.0)
            st = c.stats()
            Ch = C.cpu().numpy()
            assert n_it == iters and np.isfinite(Ch).all() and Ch.min() >= Xd.min() - 1e-6 and Ch.max() <= Xd.max() + 1e-6
            res[adaptive] = (st["path_switch_iter"], st["last_path"], st["recheck_rows"])
        # default check_every = 4: the first burst's counters are read after the second burst is queued
        assert res[1][0] == 8 and res[1][1] == 1
        assert res[0][0] == -1 and res[0][1] == 2 and res[0][2] > res[1][2] > 0
        c.set_option("adaptive_path", 1)
        # a fit's inertia pass follows the path its Lloyd loop ended on: the generic kernels after the switch
        out = c.kmeans_fit(_dev(Xd), k, init=Xd[:k].copy(), max_iter=iters, tol=-1.0)
        st = c.stats()
        assert st["path_switch_iter"] >= 0 and st["last_path"] == 1 and np.isfinite(out["inertia_"])
        Xb, ctr = ko.make_blobs(20000, d, k, seed=3)
        Cb = _dev((ctr + 0.25 * np.random.default_rng(0).normal(size=ctr.shape)).astype(np.float32))
        c.kmeans_lloyd(_dev(Xb), Cb, iters, -1.0)
        assert c.stats()["path_switch_iter"] == -1 and c.stats()["last_path"] == 2
        Xu = ko.make_uniform(30000, d, seed=5)
        C0 = Xu[:k].copy()
        Cu = _dev(C0)
        c.kmeans_lloyd(_dev(Xu), Cu, iters, -1.0)
        lab0, _, margin0 = ko.assign(Xu, C0)
        if margin0.min() > 1e-5:   # (an admissible tie row may send trajectories apart on uniform data)
            ref = ko.lloyd([Xu], C0, iters, -1.0)
            assert ko.max_center_rel_err(Cu.cpu().numpy(), ref["centers"]) <= 10 * CENTER_RTOL
    finally:
        c.close()


@pytest.mark.parametrize("n,d,k,gen", [
    (6000, 256, 600, "blobs"),      # 3 chunks, the last one overlapping the second ([344, 600))
    (5000, 64, 257, "uniform"),     # the smallest chunked k; DP = 128 instantiation
    (3000, 128, 1024, "blobs"),
])
def test_assign_and_lloyd_beyond_256_clusters_run_in_chunks(n, d, k, gen):
    """k > 256 (d <= 256): the assignment runs as chunks of 128 (d <= 128, 3xTF32 kernel) or 256 centres (large-shape
    kernel) merged by min distance; Lloyd keeps the generic label-driven update.  Same parity rule as every other path."""
    from spark_rapids_ml_b200 import _native

    X = ko.make_blobs(n, d, k, seed=9)[0] if gen == "blobs" else ko.make_uniform(n, d, seed=9)
    rng = np.random.default_rng(4)
    C0 = X[rng.choice(n, size=k, replace=False)].copy()
    c = _native.Context(0)
    try:
        before = c.stats()["fused_tc_launches"]
        labels, md = c.kmeans_assign(_dev(X), _dev(C0), want_mindist=True)
        st = c.stats()
        ch = 128 if d <= 128 else 256     # d <= 128: exact 3xTF32 chunks; else the large-shape kernel
        assert st["last_path"] == 2 and st["fused_tc_launches"] - before == -(-k // ch)
        cmp = ko.compare_labels(X, C0, labels.cpu().numpy(), tau=TAU)
        assert cmp["n_mismatch_outside_margin"] == 0, cmp
        _, md_o, _ = ko.assign(X, C0)
        xn = (X.astype(np.float64) ** 2).sum(1)
        np.testing.assert_allclose(md.cpu().numpy(), md_o, rtol=2e-4, atol=2e-5 * float(xn.max()) + 1e-6)
        # Lloyd: one exact step, and a few iterations on blobs
        C1, _, _ = ko.lloyd_iteration([X], C0)
        one = _dev(C0)
        c.kmeans_lloyd(_dev(X), one, 1, -1.0)
        lab0, _, margin0 = ko.assign(X, C0)
        if margin0.min() > 1e-5:
            assert ko.max_center_rel_err(one.cpu().numpy(), C1) <= CENTER_RTOL
        if gen == "blobs":
            ref = ko.lloyd([X], C0, 3, -1.0)
            C = _dev(C0)
            n_it, _ = c.kmeans_lloyd(_dev(X), C, 3, -1.0)
            assert n_it == 3 and c.stats()["last_path"] == 2
            assert ko.max_center_rel_err(C.cpu().numpy(), ref["centers"]) <= CENTER_RTOL
        # the generic path still exists and agrees
        c.set_option("kernel_path", 1)
        lg, _ = c.kmeans_assign(_dev(X), _dev(C0))
        assert c.stats()["last_path"] == 1
        assert ko.compare_labels(X, C0, lg.cpu().numpy(), tau=TAU)["n_mismatch_outside_margin"] == 0
    finally:
        c.close()


# Deltas of (kernel_launches, fused_tc_launches, generic_launches) and last_path of one assign pass without min distances,
# or None where kernel_path = tcgen05 must fail.  Per pass: 3 kernels on the 3xTF32 kernel (centre split, update table,
# pass), 5 on the screening kernel (row norms, centre prep, tables, pass, deferred-row labels) and 2 on the generic path
# (centre norms, assign); a chunked pass runs the row norms once, one fused pass per chunk and a merge for every chunk
# after the first.
@pytest.mark.parametrize("d,k,path,misaligned,expect", [
    (64, 32, 0, False, (3, 1, 0, 2)),        # 3xTF32 <32, 64>
    (128, 64, 0, False, (3, 1, 0, 2)),       # 3xTF32 <64, 128> on CTA pairs
    (32, 64, 0, False, (3, 1, 0, 2)),        # 3xTF32 <64, 32>
    (32, 100, 0, False, (5, 1, 0, 2)),       # d <= 32, 64 < k <= 128: no <128, 32>, the screening kernel at DP = 128
    (128, 200, 0, False, (5, 1, 0, 2)),      # screening kernel, DP = 128
    (256, 256, 0, False, (5, 1, 0, 2)),      # screening kernel, DP = 256
    (6, 16, 0, False, (2, 0, 1, 1)),         # d % 4 != 0: no TMA
    (6, 16, 2, False, None),
    (260, 16, 0, False, (2, 0, 1, 1)),       # d > 256
    (260, 16, 2, False, None),
    (64, 32, 0, True, (2, 0, 1, 1)),         # X not 16-byte aligned
    (64, 32, 1, False, (2, 0, 1, 1)),        # kernel_path = generic
    (64, 300, 0, False, (11, 3, 0, 2)),      # 3 chunks of 128 on 3xTF32 <128, 64> + 2 merges
    (200, 600, 0, False, (15, 3, 0, 2)),     # row norms + 3 chunks of 256 on the screening kernel + 2 merges
    (32, 300, 0, False, (15, 3, 0, 2)),      # d <= 32: chunks of 128 on the screening kernel
])
def test_each_shape_takes_its_kernel(d, k, path, misaligned, expect):
    """The kernel each (d, k) runs on (b2k_choose_kernel in csrc/b2k_api.cu), seen through the public stats."""
    import torch
    from spark_rapids_ml_b200 import _native

    n = 4096
    X = torch.from_numpy(ko.make_uniform(n, d, seed=2)).cuda()
    if misaligned:   # a contiguous view starting 4 bytes into its buffer
        X = torch.empty(n * d + 1, dtype=torch.float32, device="cuda")[1:].view(n, d).copy_(X)
        assert X.data_ptr() % 16 == 4
    C = X[:k].clone()
    c = _native.Context(0)
    try:
        c.set_option("kernel_path", path)
        if expect is None:
            with pytest.raises(_native.B2KError) as e:
                c.kmeans_assign(X, C)
            assert e.value.code == 4   # B2K_ERR_UNSUPPORTED
            return
        b = c.stats()
        c.kmeans_assign(X, C)
        a = c.stats()
        got = tuple(a[f] - b[f] for f in ("kernel_launches", "fused_tc_launches", "generic_launches"))
        assert got + (a["last_path"],) == expect
    finally:
        c.close()


def test_baseline_cfg3_full_partition_every_row(ctx):
    """BASELINE configs[2]'s per-GPU partition at its real size (k=256, d=256, 12.5 M rows): every row's label and min
    distance against an fp64 PyTorch restatement on the device, one Lloyd step against the fp64 sums of those labels,
    bitwise determinism — through the screening kernel and its fix-up."""
    import torch
    from _fullsize import check_every_row, check_one_step, make_blobs

    X, C = make_blobs(12_500_000, 256, 256, seed=22)
    r = check_every_row(ctx, X, C, chunk=250_000)
    assert ctx.stats()["last_path"] == 2
    assert r["outside_margin"] == 0, {k: v for k, v in r.items() if k != "labels"}
    assert r["worst_mindist_rel_err"] <= 2e-4, r["worst_mindist_rel_err"]
    rel, same = check_one_step(ctx, X, C, r["labels"])
    assert rel <= 1e-5 and same, (rel, same)
    del X
    torch.cuda.empty_cache()
