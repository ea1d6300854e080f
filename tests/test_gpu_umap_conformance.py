"""Conformance of the UMAP kernels (csrc/umap.cu), stage by stage, against float64 references.

Each stage is driven directly (through _lib.call or the thin stage functions of data/latent_umap.py) with
inputs that isolate it: synthetic kNN lists, CSR graphs and schedules.  oracle/umap_oracle.py is the pin;
its Python loops are too slow at 10^5 rows, so the vectorised restatements below stand in for it there,
and the CPU tests at the top check each restatement against the oracle at small sizes.

kNN: every template (the D pad DP and the candidate count KP, at both edges of KP's k + 8 margin), the
launch shape, and inputs whose scale or offset defeats a plain fp32 selection: power-of-two scale sweeps
(exact, so the result must repeat the unscaled one bit for bit), large offsets, tight clusters far apart,
one far outlier and exact ties.  Outputs start as sentinels, so an unwritten entry shows."""
import importlib
import math

import numpy as np
import pytest
import scipy.sparse
import scipy.sparse.csgraph

from oracle import umap_oracle as uo

lu = importlib.import_module("autoencoded-vocal-analysis_b200.data.latent_umap")
_lib = importlib.import_module("autoencoded-vocal-analysis_b200._lib")

M64 = np.uint64(0xFFFFFFFFFFFFFFFF)
IDX_SENTINEL = -7


# ================================================================ vectorised restatements (CPU)
def _mix(z):
    z = z + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def hash_v(seed, a, b, c):
    """umap_hash over uint64 arrays (wrapping arithmetic)."""
    with np.errstate(over="ignore"):
        s = _mix(np.uint64(seed))
        return _mix(_mix(_mix(s ^ np.asarray(a, np.uint64)) ^ np.asarray(b, np.uint64)) ^ np.asarray(c, np.uint64))


def unit_v(h):
    return ((h >> np.uint64(11)).astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


def kernel_mean(v):
    """The fixed-order mean of mean_kernel: 1024 sequential strided sums, then a halving tree."""
    v = np.asarray(v, np.float64).ravel()
    n = v.size
    pad = np.zeros(-(-n // 1024) * 1024)
    pad[:n] = v
    red = np.add.reduce(pad.reshape(-1, 1024), axis=0)   # along axis 0: row after row, in order
    o = 512
    while o > 0:
        red[:o] = red[:o] + red[o:2 * o]
        o //= 2
    return red[0] / float(n)


def smooth_knn_v(knn_idx, dist, local_connectivity=1.0, n_iter=64):
    """smooth_knn_dist + compute_membership_strengths, vectorised over rows, summing over j in order."""
    dist = np.asarray(dist, np.float64)
    N, k = dist.shape
    target = np.log2(k)
    nz = dist > 0.0
    n_nz = nz.sum(1)
    row_sum = np.zeros(N)
    for j in range(k):
        row_sum = row_sum + dist[:, j]
    # the m-th non-zero distance of each row (0 where there is none)
    order = np.argsort(~nz, axis=1, kind="stable")
    nzs = np.where(np.take_along_axis(nz, order, 1), np.take_along_axis(dist, order, 1), 0.0)
    nzs = np.hstack([nzs, np.zeros((N, 1))])
    rho = np.zeros(N)
    lc = float(local_connectivity)
    full = n_nz >= lc
    if np.isfinite(lc) and full.any():
        index = int(math.floor(lc))
        interp = lc - index
        if index > 0:
            r = nzs[:, index - 1].copy()
            if interp > uo.SMOOTH_K_TOLERANCE:
                r = r + interp * (nzs[:, min(index, k)] - nzs[:, index - 1])
        else:
            r = interp * nzs[:, 0]
        rho[full] = r[full]
    last = np.where(n_nz > 0, nzs[np.arange(N), np.maximum(n_nz - 1, 0)], 0.0)
    rho[~full] = last[~full]
    lo, hi, mid = np.zeros(N), np.full(N, np.inf), np.ones(N)
    done = np.zeros(N, bool)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        for _ in range(n_iter):
            psum = np.zeros(N)
            for j in range(1, k):
                d = dist[:, j] - rho
                psum = psum + np.where(d > 0.0, np.exp(-(d / mid)), 1.0)
            done = done | (np.abs(psum - target) < uo.SMOOTH_K_TOLERANCE)
            act = ~done
            up = act & (psum > target)
            dn = act & ~(psum > target)
            hi = np.where(up, mid, hi)
            lo = np.where(dn, mid, lo)
            mid = np.where(up, (lo + hi) / 2.0, np.where(dn, np.where(np.isinf(hi), mid * 2.0, (lo + hi) / 2.0), mid))
    floor_ref = np.where(rho > 0.0, row_sum / float(k), kernel_mean(dist))
    sigma = np.where(mid < uo.MIN_K_DIST_SCALE * floor_ref, uo.MIN_K_DIST_SCALE * floor_ref, mid)
    with np.errstate(over="ignore", invalid="ignore"):
        w = np.where(dist - rho[:, None] <= 0.0, 1.0, np.exp(-((dist - rho[:, None]) / sigma[:, None])))
    w = np.where(sigma[:, None] == 0.0, 1.0, w)
    w[np.asarray(knn_idx) == np.arange(N)[:, None]] = 0.0
    return rho, sigma, w


def fuzzy_union_v(knn_idx, w):
    """The CSR of P = A + A^T - A.*A^T: (rowptr, cols, vals, rows), vals = (a + b) - a*b."""
    knn_idx = np.asarray(knn_idx, np.int64)
    N, k = knn_idx.shape
    i = np.repeat(np.arange(N, dtype=np.int64), k)
    j = knn_idx.ravel()
    keep = i != j
    i, j, wv = i[keep], j[keep], np.asarray(w, np.float64).ravel()[keep]
    dkeys = i * N + j
    o = np.argsort(dkeys)
    dkeys, wv = dkeys[o], wv[o]
    keys = np.unique(np.concatenate([dkeys, j[o] * N + i[o]]))
    r, c = keys // N, keys % N

    def look(kk):
        if dkeys.size == 0:
            return np.zeros(kk.shape)
        p = np.minimum(np.searchsorted(dkeys, kk), dkeys.size - 1)
        return np.where(dkeys[p] == kk, wv[p], 0.0)

    a, b = look(keys), look(c * N + r)
    vals = (a + b) - a * b
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(r, minlength=N))]).astype(np.int64)
    return rowptr, c.astype(np.int32), vals, r.astype(np.int32)


def _random_knn(N, k, seed, hub=False):
    rng = np.random.default_rng(seed)
    idx = np.empty((N, k), np.int64)
    idx[:, 0] = np.arange(N)
    for i in range(N):
        if k > 1:
            pool = rng.choice(N - 1, size=k - 1, replace=False)
            pool = pool + (pool >= i)
            if hub and i != 0 and 0 not in pool:
                pool[0] = 0
            idx[i, 1:] = pool
    dist = np.sort(rng.uniform(0.1, 3.0, (N, k)), axis=1)
    dist[:, 0] = 0.0
    w = rng.uniform(0.01, 1.0, (N, k))
    w[:, 0] = 0.0
    return idx, dist, w


def _random_knn_fast(N, k, seed):
    """Random kNN lists for large N: distinct columns by rejection of duplicates."""
    rng = np.random.default_rng(seed)
    idx = np.empty((N, k), np.int64)
    idx[:, 0] = np.arange(N)
    cols = rng.integers(0, N, (N, k - 1))
    for _ in range(20):
        bad = (cols == np.arange(N)[:, None])
        s = np.sort(cols, 1)
        dup = np.zeros_like(bad)
        dup_sorted = np.hstack([np.zeros((N, 1), bool), s[:, 1:] == s[:, :-1]])
        if dup_sorted.any():
            rows = np.flatnonzero(dup_sorted.any(1))
            for r in rows:
                _, first = np.unique(cols[r], return_index=True)
                m = np.ones(k - 1, bool)
                m[first] = False
                dup[r] = m
        bad |= dup
        if not bad.any():
            break
        cols[bad] = rng.integers(0, N, int(bad.sum()))
    idx[:, 1:] = cols
    w = rng.uniform(0.01, 1.0, (N, k))
    w[:, 0] = 0.0
    return idx, w


# ------------------------------------------------------------------------ restatements vs oracle
def test_restated_hash_matches_oracle():
    for seed in (0, 42, 2 ** 64 - 1):
        for sid in (0, (3 << 32) | 5, 0xFFFFFFFF00000001):
            i = np.arange(300, dtype=np.uint64)
            h = hash_v(seed, np.uint64(sid), i, np.uint64(1))
            ref = np.array([uo.umap_hash(seed, sid, int(t), 1) for t in range(300)], dtype=np.uint64)
            np.testing.assert_array_equal(h, ref)
            np.testing.assert_array_equal(unit_v(h), [uo.unit(int(t)) for t in ref])


@pytest.mark.parametrize("lc", [0.0, 0.5, 1.0, 1.5, 2.0, 3.25, 19.0, 25.0])
def test_restated_smooth_knn_matches_oracle(lc):
    idx, dist, _ = _random_knn(300, 20, seed=int(lc * 4))
    dist[::7, 1:4] = 0.0                       # duplicates: leading zero distances
    if lc > 0:                                 # (the oracle has no non-zero distance to index at 0)
        dist[::11, :] = 0.0                    # all-zero rows
    dist[5::13, 1:18] = 0.0                    # fewer non-zero distances than local_connectivity
    dist = np.sort(dist, 1)
    rho, sigma, w = smooth_knn_v(idx, dist, lc)
    sref, rref = uo.smooth_knn_dist(dist, 20, local_connectivity=lc)
    np.testing.assert_array_equal(rho, rref)
    np.testing.assert_allclose(sigma, sref, rtol=1e-12, atol=0)
    np.testing.assert_allclose(w, uo.membership_strengths(idx, dist, sref, rref), rtol=1e-12, atol=1e-300)


def test_restated_fuzzy_union_matches_oracle():
    for N, k, hub in ((200, 6, False), (150, 4, True), (50, 1, False)):
        idx, _, w = _random_knn(N, k, seed=N, hub=hub)
        rowptr, cols, vals, _ = fuzzy_union_v(idx, w)
        P = uo.fuzzy_union(idx, w)
        np.testing.assert_array_equal(rowptr, P.indptr)
        np.testing.assert_array_equal(cols, P.indices)
        np.testing.assert_array_equal(vals, P.data)


def test_restated_kernel_mean():
    v = np.random.default_rng(0).uniform(0, 1, 12345)
    assert abs(kernel_mean(v) - v.mean()) <= 1e-15


# ================================================================================ GPU helpers
def _torch():
    import torch
    return torch


def _stream():
    torch = _torch()
    return torch.cuda.current_stream().cuda_stream


def _dev(a, dtype=None):
    torch = _torch()
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def _expect_rejected(name, args, outs, match):
    """Raises AvaB200Error with a message, launches nothing and leaves the outputs as they were."""
    torch = _torch()
    before = [o.clone() for o in outs]
    n0 = _lib.launch_count()
    with pytest.raises(_lib.AvaB200Error, match=match) as e:
        _lib.call(name, *args)
    torch.cuda.synchronize()
    assert str(e.value).split("failed: ", 1)[1].strip()
    assert _lib.launch_count() == n0
    for o, b in zip(outs, before):
        assert torch.equal(o.view(torch.uint8), b.view(torch.uint8))


def run_knn(x, k, ws_bytes=None):
    """ava_b200_umap_knn on a device tensor with sentinel-filled outputs."""
    torch = _torch()
    N, D = x.shape
    need = int(_lib.lib().ava_b200_umap_knn_ws_bytes(N, D, k))
    ws = torch.full((max(need, 1),), 0xA5, dtype=torch.uint8, device=x.device)
    idx = torch.full((N, k), IDX_SENTINEL, dtype=torch.int32, device=x.device)
    dist = torch.full((N, k), float("nan"), dtype=torch.float64, device=x.device)
    _lib.call("ava_b200_umap_knn", x.data_ptr(), 1 if x.dtype == torch.float32 else 0, N, D, k, idx.data_ptr(),
              dist.data_ptr(), ws.data_ptr(), need if ws_bytes is None else ws_bytes, _stream())
    torch.cuda.synchronize()
    return idx, dist


def check_knn(x, k, idx, dist, min_pinned=0.5, exact_ties=True):
    """Every row: valid, unique indices with the row first; the list ordered by (distance, index) after
    the row itself; the j-th listed neighbour's fp64 distance (difference form) equals the j-th smallest
    to 1e-12; the reported distances equal an fp64 recomputation of the listed pairs to 1e-12; and the list
    equals the reference's (distance, not-self, index) order in every row where no two of the first k + 1
    distances are within 1e-12 relative (exact_ties: equal ones, which every summation order reproduces
    for data such as integers, do not count as near)."""
    torch = _torch()
    N = x.shape[0]
    x64 = x.double()
    q = torch.arange(N, device=x.device)
    ii = idx.long()
    assert bool((ii >= 0).all()) and bool((ii < N).all()), "unwritten or invalid indices"
    assert bool(torch.isfinite(dist).all()), "unwritten distances"
    assert bool((ii[:, 0] == q).all()), "the row itself is not first"
    s = torch.sort(ii, 1).values
    assert bool((s[:, 1:] != s[:, :-1]).all()), "repeated neighbour"
    if k > 1:
        d1, d0 = dist[:, 2:], dist[:, 1:-1]
        assert bool((d1 >= d0).all()), "distances out of order"
    rec = torch.sqrt(((x64[:, None, :] - x64[ii]) ** 2).sum(-1))
    assert bool(((dist - rec).abs() <= 1e-12 * rec).all()), float((dist - rec).abs().max())
    kk = min(k + 1, N)
    for b0 in range(0, N, 1024):
        b1 = min(N, b0 + 1024)
        ref = torch.cdist(x64[b0:b1], x64, compute_mode="donot_use_mm_for_euclid_dist")
        ref[torch.arange(b1 - b0), torch.arange(b0, b1)] = -1.0           # the row itself first
        rs, ro = torch.sort(ref, dim=1, stable=True)                           # ties: lower index first
        rs, ro = rs[:, :kk], ro[:, :kk]
        rs[:, 0] = 0.0
        got = rec[b0:b1]
        want = rs[:, :k]
        assert bool(((got - want).abs() <= 1e-12 * want).all()), "a neighbour is not among the k nearest"
        gaps = rs[:, 1:] - rs[:, :-1]
        near = (((gaps > 0) | (not exact_ties)) & (gaps <= 1e-12 * rs[:, 1:]) & (rs[:, 1:] > 0)).any(1)
        pinned = ~near
        assert bool((ii[b0:b1][pinned] == ro[pinned][:, :k]).all()), "order differs from (distance, index)"
        assert float(pinned.float().mean()) >= min_pinned


def knn_case(x, k, **kw):
    torch = _torch()
    idx, dist = run_knn(x, k)
    idx2, dist2 = run_knn(x, k)
    assert torch.equal(idx, idx2) and torch.equal(dist.view(torch.int64), dist2.view(torch.int64))
    check_knn(x, k, idx, dist, **kw)
    return idx, dist


# ===================================================================================== 1. kNN
@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 3, 8, 9, 16, 17, 33, 64])
@pytest.mark.parametrize("k", [1, 2, 8, 9, 24, 25, 56, 57, 100])
@pytest.mark.parametrize("dtype", ["f32", "f64"])
def test_knn_templates(D, k, dtype):
    torch = _torch()
    rng = np.random.default_rng(D * 1000 + k)
    c = rng.standard_normal((12, D)) * 4.0
    x = c[rng.integers(0, 12, 4100)] + rng.standard_normal((4100, D))
    knn_case(_dev(x, torch.float32 if dtype == "f32" else torch.float64), k)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 2, 63, 64, 65, 127, 128, 129])
@pytest.mark.parametrize("dtype", ["f32", "f64"])
def test_knn_launch_shape(N, dtype):
    torch = _torch()
    x = np.random.default_rng(N).standard_normal((N, 5))
    xd = _dev(x, torch.float32 if dtype == "f32" else torch.float64)
    for k in sorted({1, min(2, N), min(20, N), N if N <= 100 else 100}):
        knn_case(xd, k)


SCALES = [-120, -80, -75, -60, 0, 60, 64, 100]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("D", [2, 8, 33])
def test_knn_scale_sweep_is_exact(dtype, D):
    """x 2^s for every s: a power-of-two scale is exact, so the lists repeat the s = 0 ones bit for bit
    and the distances scale by exactly 2^s (fp32 input: the s that keep every value a normal float)."""
    torch = _torch()
    rng = np.random.default_rng(D)
    N, k = 3000, 20
    x = rng.standard_normal((N, D))
    if dtype == "f32":
        x = x.astype(np.float32).astype(np.float64)
    base = None
    for s in sorted(SCALES, key=abs):
        xs = x * 2.0 ** s
        if dtype == "f32":
            a = np.abs(xs[xs != 0])
            if a.min() < 2.0 ** -126 or a.max() >= 2.0 ** 127:
                continue
            xd = _dev(xs.astype(np.float32))
        else:
            xd = _dev(xs)
        idx, dist = run_knn(xd, k)
        assert bool((idx >= 0).all()) and bool(torch.isfinite(dist).all()), "unwritten entries at s=%d" % s
        if s == 0:
            base = (idx, dist)
            check_knn(xd, k, idx, dist)
            continue
        assert torch.equal(idx, base[0]), "s=%d changed the lists" % s
        assert torch.equal(dist * 2.0 ** -s, base[1]), "s=%d changed the distances" % s


@pytest.mark.gpu
@pytest.mark.parametrize("c,sigma", [(1e3, 1.0), (1e3, 1e-3), (1e6, 1e-2)])
@pytest.mark.parametrize("D", [2, 8, 32])
@pytest.mark.parametrize("dtype", ["f32", "f64"])
def test_knn_offset(c, sigma, D, dtype):
    torch = _torch()
    x = c + sigma * np.random.default_rng(D).standard_normal((3000, D))
    xd = _dev(x, torch.float32 if dtype == "f32" else torch.float64)
    knn_case(xd, 20, min_pinned=0.2)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["f32", "f64"])
def test_knn_tight_far_clusters(dtype):
    torch = _torch()
    rng = np.random.default_rng(3)
    x = 1e-3 * rng.standard_normal((3000, 2))
    x[:, 0] += np.where(rng.integers(0, 2, 3000) == 0, -1e3, 1e3)
    knn_case(_dev(x, torch.float32 if dtype == "f32" else torch.float64), 20, min_pinned=0.2)


@pytest.mark.gpu
def test_knn_one_outlier():
    x = 1e-3 * np.random.default_rng(4).standard_normal((3000, 8))
    x[5] = 1e12
    knn_case(_dev(x), 20)


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 1000.1])
@pytest.mark.parametrize("k", [20, 100])
def test_knn_exact_ties(offset, k):
    rng = np.random.default_rng(5)
    lattice = np.stack(np.meshgrid(*[np.arange(6.0)] * 3, indexing="ij"), -1).reshape(-1, 3)
    x = lattice[rng.integers(0, lattice.shape[0], 1500)] + offset
    knn_case(_dev(x), k, min_pinned=0.0 if offset else 0.5, exact_ties=offset == 0.0)


# ============================================================================ 2. smooth kNN
def _smooth_knn_dev(idx, dist, k, lc):
    torch = _torch()
    N = idx.shape[0]
    idx_d, dist_d = _dev(idx.astype(np.int32)), _dev(dist)
    rho = torch.full((N,), float("nan"), dtype=torch.float64, device="cuda")
    sigma = torch.full((N,), float("nan"), dtype=torch.float64, device="cuda")
    w = torch.full((N, k), float("nan"), dtype=torch.float64, device="cuda")
    scratch = torch.empty(1, dtype=torch.float64, device="cuda")
    _lib.call("ava_b200_umap_smooth_knn", idx_d.data_ptr(), dist_d.data_ptr(), N, k, float(lc), rho.data_ptr(),
              sigma.data_ptr(), w.data_ptr(), scratch.data_ptr(), _stream())
    torch.cuda.synchronize()
    return rho.cpu().numpy(), sigma.cpu().numpy(), w.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3, 20, 100])
@pytest.mark.parametrize("lc", [0.0, 0.5, 1.0, 1.5, 2.0, 3.25, "k-1", "k+5"])
def test_smooth_knn(k, lc):
    lc = float(k - 1) if lc == "k-1" else float(k + 5) if lc == "k+5" else lc
    N = 700
    idx, dist, _ = _random_knn(N, k, seed=k * 10 + int(4 * lc))
    rng = np.random.default_rng(k)
    dist[::7, 1:min(4, k)] = 0.0                                    # duplicates
    dist[::11] = 0.0                                                # all-zero rows: the global-mean floor
    dist[3::13, 1:max(1, k - 1)] = 0.0                              # fewer non-zero than local_connectivity
    dist[5::17] = 1e30 * (1.0 + rng.uniform(0, 1e-3, (dist[5::17].shape)))   # the 64-step cap
    dist[:, 0] = 0.0
    dist = np.sort(dist, 1)
    rho, sigma, w = _smooth_knn_dev(idx, dist, k, lc)
    rr, sr, wr = smooth_knn_v(idx, dist, lc)
    np.testing.assert_array_equal(rho, rr)
    np.testing.assert_allclose(sigma, sr, rtol=1e-12, atol=0)
    np.testing.assert_allclose(w, wr, rtol=1e-12, atol=1e-300)
    assert (w[:, 0] == 0.0).all()
    assert (w[(dist <= rho[:, None]) & (idx != np.arange(N)[:, None])] == 1.0).all()


@pytest.mark.gpu
def test_smooth_knn_large_global_mean():
    k, N = 20, 100000
    rng = np.random.default_rng(9)
    idx, w = _random_knn_fast(N, k, 9)
    dist = np.sort(rng.uniform(0.0, 5.0, (N, k)), 1)
    dist[:, 0] = 0.0
    dist[::3] = 0.0                            # a third of the rows take the global-mean floor
    rho, sigma, wt = _smooth_knn_dev(idx, dist, k, 1.0)
    rr, sr, wr = smooth_knn_v(idx, dist, 1.0)
    np.testing.assert_array_equal(rho, rr)
    np.testing.assert_allclose(sigma, sr, rtol=1e-12, atol=0)
    np.testing.assert_array_equal(sigma[::3], np.full(sigma[::3].shape, uo.MIN_K_DIST_SCALE * kernel_mean(dist)))
    np.testing.assert_allclose(wt, wr, rtol=1e-12, atol=1e-300)


@pytest.mark.gpu
def test_latent_umap_local_connectivity_above_k():
    """umap-learn accepts any local_connectivity >= 0; above the non-zero distances rho is the largest."""
    rng = np.random.default_rng(2)
    x = rng.standard_normal((300, 6))
    um = lu.LatentUMAP(n_neighbors=20, local_connectivity=25, random_state=0, n_epochs=20)
    e = um.fit_transform(x)
    assert e.shape == (300, 2) and np.isfinite(e).all()
    np.testing.assert_array_equal(um._graph_dev["rho"].cpu().numpy(), um.knn_dists_.max(1))


# ===================================================================== 3. fuzzy union, schedule
def _graph_dev(idx, w):
    torch = _torch()
    N, k = idx.shape
    idx_d, w_d = _dev(idx.astype(np.int32)), _dev(np.asarray(w, np.float64))
    keys = torch.empty(2 * N * k, dtype=torch.int64, device="cuda")
    _lib.call("ava_b200_umap_edge_keys", idx_d.data_ptr(), N, k, keys.data_ptr(), _stream())
    keys = torch.unique(keys, sorted=True)
    keys = keys[keys >= 0]
    nnz = keys.numel()
    keys = torch.cat([keys, torch.zeros(1, dtype=torch.int64, device="cuda")])   # non-null when nnz = 0
    rows = torch.full((nnz + 1,), -1, dtype=torch.int32, device="cuda")
    cols = torch.full((nnz + 1,), -1, dtype=torch.int32, device="cuda")
    vals = torch.full((nnz + 1,), float("nan"), dtype=torch.float64, device="cuda")
    rowptr = torch.full((N + 1,), -1, dtype=torch.int64, device="cuda")
    _lib.call("ava_b200_umap_graph", keys.data_ptr(), nnz, N, idx_d.data_ptr(), w_d.data_ptr(), k, rows.data_ptr(),
              cols.data_ptr(), vals.data_ptr(), rowptr.data_ptr(), _stream())
    torch.cuda.synchronize()
    assert int(rows[nnz]) == -1 and int(cols[nnz]) == -1 and bool(torch.isnan(vals[nnz]))   # nothing past nnz
    return dict(rows=rows[:nnz], cols=cols[:nnz], vals=vals[:nnz], rowptr=rowptr, n=N)


GRAPHS = ["random", "hub", "k1", "large"]


def _graph_case(name):
    if name == "random":
        idx, _, w = _random_knn(3000, 12, seed=1)
    elif name == "hub":
        idx, _, w = _random_knn(5000, 5, seed=2, hub=True)
    elif name == "k1":
        idx, _, w = _random_knn(50, 1, seed=3)
    else:
        idx, w = _random_knn_fast(200000, 20, 4)
    return idx, w


@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAPHS)
def test_fuzzy_union_and_schedule(name):
    torch = _torch()
    idx, w = _graph_case(name)
    N = idx.shape[0]
    g = _graph_dev(idx, w)
    g2 = _graph_dev(idx, w)
    rowptr, cols, vals, rows = fuzzy_union_v(idx, w)
    for n in ("rows", "cols", "vals", "rowptr"):
        assert torch.equal(g[n], g2[n])
    np.testing.assert_array_equal(g["rowptr"].cpu().numpy(), rowptr)
    np.testing.assert_array_equal(g["cols"].cpu().numpy(), cols)
    np.testing.assert_array_equal(g["rows"].cpu().numpy(), rows)
    gv = g["vals"].cpu().numpy()
    np.testing.assert_array_equal(gv, vals)
    P = scipy.sparse.csr_matrix((gv, g["cols"].cpu().numpy(), g["rowptr"].cpu().numpy()), shape=(N, N))
    PT = P.T.tocsr()
    PT.sort_indices()
    np.testing.assert_array_equal(PT.indptr, P.indptr)
    np.testing.assert_array_equal(PT.indices, P.indices)
    np.testing.assert_array_equal(PT.data, P.data)                       # bitwise symmetric
    if name == "hub":
        assert int(rowptr[1] - rowptr[0]) == N - 1
    if name == "k1":
        assert not rowptr.any() and g["vals"].numel() == 0
    if P.nnz == 0:
        return
    for n_epochs in (1, 2, 7, 200, 500):
        for nsr in (0.5, 1.0, 5.0, 7.3):
            s = lu.edge_schedule(g, n_epochs, nsr)
            ref = uo.prune_and_schedule(P, n_epochs, nsr)
            np.testing.assert_array_equal(s["head"].cpu().numpy(), ref["head"])
            np.testing.assert_array_equal(s["tail"].cpu().numpy(), ref["tail"])
            for n in ("eps", "eps_neg", "next", "next_neg"):
                np.testing.assert_array_equal(s[n].cpu().numpy(), ref[n])


@pytest.mark.gpu
def test_schedule_zero_edges():
    torch = _torch()
    vals = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    vmax = torch.ones(1, dtype=torch.float64, device="cuda")
    n0 = _lib.launch_count()
    _lib.call("ava_b200_umap_epochs_per_sample", vals.data_ptr(), 0, vmax.data_ptr(), 10, 5.0, vals.data_ptr(),
              vals.data_ptr(), vals.data_ptr(), vals.data_ptr(), _stream())
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 and bool(torch.isnan(vals).all())


# ===================================================================== 4. connected components
def _csr_from_edges(N, a, b):
    a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
    P = scipy.sparse.coo_matrix((np.ones(2 * a.size), (np.concatenate([a, b]), np.concatenate([b, a]))),
                                shape=(N, N)).tocsr()
    P.sum_duplicates()
    P.sort_indices()
    P.data = np.random.default_rng(N).uniform(0.1, 1.0, P.nnz)
    P = ((P + P.T) * 0.5).tocsr()
    P.sort_indices()
    return P


def _blob_knn_graph():
    rng = np.random.default_rng(6)
    x = np.concatenate([rng.standard_normal((400, 4)) + c for c in (0.0, 50.0, -50.0)])
    x = x[rng.permutation(x.shape[0])]
    torch = _torch()
    idx, dist = lu.knn(_dev(x), 10)
    g = lu.fuzzy_graph(idx, dist)
    torch.cuda.synchronize()
    return scipy.sparse.csr_matrix((g["vals"].cpu().numpy(), g["cols"].cpu().numpy(), g["rowptr"].cpu().numpy()),
                                   shape=(g["n"], g["n"]))


def _cc_graph(name):
    rng = np.random.default_rng(7)
    if name == "path":
        N = 100000
        p = rng.permutation(N)
        return _csr_from_edges(N, p[:-1], p[1:])
    if name == "star":
        N = 5000
        return _csr_from_edges(N, np.full(N - 1, 1234), np.delete(np.arange(N), 1234))
    if name == "tree":
        N = 2 ** 14 - 1
        c = np.arange(1, N)
        return _csr_from_edges(N, (c - 1) // 2, c)
    if name == "pairs":
        p = rng.permutation(2000)
        return _csr_from_edges(2000, p[0::2], p[1::2])
    if name == "empty":
        return scipy.sparse.csr_matrix((300, 300))
    return _blob_knn_graph()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["path", "star", "tree", "pairs", "empty", "blobs"])
def test_connected_components(name):
    torch = _torch()
    P = _cc_graph(name)
    N = P.shape[0]
    rowptr = _dev(P.indptr.astype(np.int64))
    cols = _dev(P.indices.astype(np.int32)) if P.nnz else torch.zeros(1, dtype=torch.int32, device="cuda")
    labels = torch.arange(N, dtype=torch.int32, device="cuda")
    changed = torch.zeros(1, dtype=torch.int32, device="cuda")
    bound = 3 * math.ceil(math.log2(max(N, 2))) + 10
    rounds = 0
    while True:
        changed.zero_()
        _lib.call("ava_b200_umap_components_step", rowptr.data_ptr(), cols.data_ptr(), N, labels.data_ptr(),
                  changed.data_ptr(), _stream())
        rounds += 1
        if int(changed.item()) == 0:
            break
        assert rounds <= bound, "no fixed point after %d rounds" % rounds
    nc, lab = scipy.sparse.csgraph.connected_components(P, directed=False)
    smallest = np.full(nc, N)
    np.minimum.at(smallest, lab, np.arange(N))
    np.testing.assert_array_equal(labels.cpu().numpy(), smallest[lab])
    print("components %s: N=%d, %d components, %d rounds (bound %d)" % (name, N, nc, rounds, bound))
    if name == "blobs":
        assert nc == 3


# ============================================================== 5. degree and the Laplacian SpMM
def _spmm_graph(name):
    if name in ("random", "hub", "large"):
        idx, w = _graph_case(name)
        rowptr, cols, vals, _ = fuzzy_union_v(idx, w)
        N = idx.shape[0]
        return scipy.sparse.csr_matrix((vals, cols, rowptr), shape=(N, N))
    if name == "k100":
        idx, _, w = _random_knn(3000, 100, seed=8)
        rowptr, cols, vals, _ = fuzzy_union_v(idx, w)
        return scipy.sparse.csr_matrix((vals, cols, rowptr), shape=(3000, 3000))
    return _cc_graph(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["random", "hub", "k100", "path", "star", "tree", "blobs"])
def test_degree_and_spmm(name):
    torch = _torch()
    P = _spmm_graph(name)
    N = P.shape[0]
    rowptr, cols, vals = _dev(P.indptr.astype(np.int64)), _dev(P.indices.astype(np.int32)), _dev(P.data)
    dis = torch.full((N,), float("nan"), dtype=torch.float64, device="cuda")
    _lib.call("ava_b200_umap_degree", rowptr.data_ptr(), vals.data_ptr(), N, dis.data_ptr(), _stream())
    deg = np.array([math.fsum(P.data[P.indptr[i]:P.indptr[i + 1]]) for i in range(N)])
    rl = np.diff(P.indptr)
    dis_h = dis.cpu().numpy()
    assert (np.abs(dis_h - 1.0 / np.sqrt(deg)) <= (rl + 3) * 2.0 ** -52 / np.sqrt(deg)).all()
    nc, lab = scipy.sparse.csgraph.connected_components(P, directed=False)
    c = np.bincount(lab).argmax()
    rng = np.random.default_rng(N)
    verts = rng.permutation(np.flatnonzero(lab == c)).astype(np.int32)
    n = verts.size
    pos = np.full(N, -1, np.int32)
    pos[verts] = np.arange(n, dtype=np.int32)
    Pc = P[verts][:, verts]
    Dm = scipy.sparse.diags(dis_h[verts])
    M = (Dm @ Pc @ Dm).tocsr()
    Mabs = abs(M)
    rlc = np.diff(P.indptr)[verts]
    verts_d, pos_d = _dev(verts), _dev(pos)
    for m in (1, 2, 5, 8, 9, 16, 17, 31, 32):
        X = rng.standard_normal((n, m))
        Xd = _dev(X)
        Y = torch.full((n, m), float("nan"), dtype=torch.float64, device="cuda")
        Y2 = torch.full((n, m), float("nan"), dtype=torch.float64, device="cuda")
        for out in (Y, Y2):
            _lib.call("ava_b200_umap_spmm", rowptr.data_ptr(), cols.data_ptr(), vals.data_ptr(), verts_d.data_ptr(),
                      n, pos_d.data_ptr(), dis.data_ptr(), Xd.data_ptr(), m, out.data_ptr(), _stream())
        torch.cuda.synchronize()
        assert torch.equal(Y, Y2)
        ref = X - M @ X
        bound = (rlc[:, None] + 4) * 2.0 ** -52 * (np.abs(X) + Mabs @ np.abs(X))
        err = np.abs(Y.cpu().numpy() - ref)
        assert (err <= bound).all(), (m, float((err / bound).max()))


# ======================================================================== 6. gram and combine
GRAM_N = [1, 2, 31, 32, 33, 295, 296, 297, 100007]
GRAM_PQ = [(1, 1), (1, 33), (33, 1), (3, 5), (8, 8), (17, 9), (32, 33), (33, 33)]


def _gram_dev(A, B, reps=2):
    torch = _torch()
    n, p = A.shape
    q = B.shape[1]
    wsb = int(_lib.lib().ava_b200_umap_gram_ws_bytes(p, q))
    assert wsb > 0
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    Ad, Bd = _dev(A), _dev(B)
    outs = []
    for _ in range(reps):
        out = torch.full((p, q), float("nan"), dtype=torch.float64, device="cuda")
        _lib.call("ava_b200_umap_gram", Ad.data_ptr(), p, Bd.data_ptr(), q, n, out.data_ptr(), ws.data_ptr(), wsb,
                  _stream())
        outs.append(out)
    torch.cuda.synchronize()
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    return outs[0].cpu().numpy()


def _exact_gram(A, B):
    return np.dot(A.astype(np.longdouble).T, B.astype(np.longdouble))


@pytest.mark.gpu
@pytest.mark.parametrize("n", GRAM_N)
def test_gram_and_combine(n):
    torch = _torch()
    rng = np.random.default_rng(n)
    for p, q in GRAM_PQ:
        A = rng.standard_normal((n, p))
        B = rng.standard_normal((n, q))
        if n >= 2:                               # heavy cancellation: rows in +- pairs plus a small remainder
            h = n // 2
            A[h:2 * h] = A[:h] * (1.0 + 1e-9 * rng.standard_normal((h, p)))
            B[h:2 * h] = -B[:h]
            A[:h] *= 1e6
            A[h:2 * h] *= 1e6
        got = _gram_dev(A, B)
        ref = _exact_gram(A, B)
        bound = max(n, 2) * 2.0 ** -53 * (np.abs(A).T @ np.abs(B))
        err = np.abs(got.astype(np.longdouble) - ref).astype(np.float64)
        assert (err <= bound).all(), (p, q, float((err / np.maximum(bound, 1e-300)).max()))
        if n > 100000:
            continue
        C = rng.standard_normal((p, q))
        Ad, Cd = _dev(A), _dev(C)
        Ys = []
        for _ in range(2):
            Y = torch.full((n, q), float("nan"), dtype=torch.float64, device="cuda")
            _lib.call("ava_b200_umap_combine", Ad.data_ptr(), p, Cd.data_ptr(), q, n, Y.data_ptr(), _stream())
            Ys.append(Y)
        torch.cuda.synchronize()
        assert torch.equal(Ys[0], Ys[1])
        ref = np.dot(A.astype(np.longdouble), C.astype(np.longdouble))
        err = np.abs(Ys[0].cpu().numpy().astype(np.longdouble) - ref).astype(np.float64)
        assert (err <= (p + 1) * 2.0 ** -53 * (np.abs(A) @ np.abs(C))).all()


GRAM_EDGE_OK = [(1, 191), (191, 1), (2, 190), (10, 182), (45, 45), (64, 32), (2048 // 96, 96)]
GRAM_EDGE_BAD = [(200, 1), (1, 192), (96, 97), (46, 45), (2048, 1), (1, 2049), (0, 4), (4, 0)]


@pytest.mark.gpu
def test_gram_shape_limits():
    """Every shape the ABI accepts runs; every shape it refuses is refused before any launch, and the
    workspace query agrees with the check."""
    torch = _torch()
    rng = np.random.default_rng(11)
    for p, q in GRAM_EDGE_OK:
        A, B = rng.standard_normal((297, p)), rng.standard_normal((297, q))
        got = _gram_dev(A, B, reps=1)
        ref = _exact_gram(A, B)
        assert (np.abs(got - ref.astype(np.float64)) <= 297 * 2.0 ** -53 * (np.abs(A).T @ np.abs(B))).all()
    A = torch.zeros(4096, dtype=torch.float64, device="cuda")
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    out = torch.full((4096,), float("nan"), dtype=torch.float64, device="cuda")
    for p, q in GRAM_EDGE_BAD:
        assert int(_lib.lib().ava_b200_umap_gram_ws_bytes(p, q)) == -1, (p, q)
        _expect_rejected("ava_b200_umap_gram", (A.data_ptr(), p, A.data_ptr(), q, 1, out.data_ptr(), ws.data_ptr(),
                                                ws.numel(), _stream()), (out,), r"p \+ q")


# ============================================================================ 7. random draws
@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 42, 2 ** 64 - 1])
def test_random_draws(seed):
    torch = _torch()
    for sid in ((1 << 32), (3 << 32) | 7, 0xFFFFFFFF00000001, 2 ** 64 - 1):
        for n in (1, 255, 256, 257, 1000003):
            i = np.arange(n, dtype=np.uint64)
            u1 = unit_v(hash_v(seed, np.uint64(sid), i, np.uint64(0)))
            out = torch.full((n + 1,), float("nan"), dtype=torch.float64, device="cuda")
            _lib.call("ava_b200_umap_random", seed, sid, n, 0, 2.5, out.data_ptr(), _stream())
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            assert np.isnan(got[n])
            np.testing.assert_array_equal(got[:n], 2.5 * (2.0 * u1 - 1.0))
            out.fill_(float("nan"))
            _lib.call("ava_b200_umap_random", seed, sid, n, 1, 0.5, out.data_ptr(), _stream())
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            assert np.isnan(got[n])
            u2 = unit_v(hash_v(seed, np.uint64(sid), i, np.uint64(1)))
            r = 0.5 * np.sqrt(-2.0 * np.log(u1))
            ref = r * np.cos(6.283185307179586 * u2)
            assert (np.abs(got[:n] - ref) <= 8 * 2.0 ** -52 * r).all()
            if n > 10 ** 6:
                z = got[:n] / 0.5
                assert abs(z.mean()) < 5 / math.sqrt(n) and abs(z.var() - 1.0) < 7 * math.sqrt(2.0 / n)
                assert abs((z ** 4).mean() - 3.0) < 0.05 and abs((z ** 3).mean()) < 0.02


# ============================================================================= 8. init layout
@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 2, 1023, 1024, 1025, 100000])
@pytest.mark.parametrize("dim", [1, 2, 3, 8])
@pytest.mark.parametrize("noise", [False, True])
def test_init_layout(N, dim, noise):
    torch = _torch()
    rng = np.random.default_rng(N * 10 + dim)
    init = rng.standard_normal((N, dim)) * 3.0 + 1.0
    if dim >= 2:
        init[:, 1] = 0.75                       # a constant axis
    nz = 1e-4 * rng.standard_normal((N, dim)) if noise else None
    expansion = 10.0 / np.abs(init).max() if noise else 1.0
    emb = torch.full((N, dim), float("nan"), dtype=torch.float32, device="cuda")
    nzd = _dev(nz) if noise else None
    _lib.call("ava_b200_umap_init_layout", _dev(init).data_ptr(), None if nzd is None else nzd.data_ptr(), expansion,
              N, dim, emb.data_ptr(), _stream())
    torch.cuda.synchronize()
    ref = uo.init_embedding(init, nz) if noise else uo.init_embedding(init)
    np.testing.assert_array_equal(emb.cpu().numpy(), ref)
    if dim >= 2 and not noise:
        assert (emb[:, 1] == 0).all()


# ===================================================================================== 9. SGD
def _sgd_setup(N, dim, seed, n_epochs, nsr):
    idx, _, w = _random_knn(N, 5, seed=seed)
    rowptr, cols, vals, rows = fuzzy_union_v(idx, w)
    P = scipy.sparse.csr_matrix((vals, cols, rowptr), shape=(N, N))
    ref = uo.prune_and_schedule(P, n_epochs, nsr)
    emb = np.random.default_rng(seed).uniform(0, 10, (N, dim)).astype(np.float32)
    return ref, emb


def _sched_dev(ref):
    d = {n: _dev(ref[n].astype(np.int32)) for n in ("head", "tail")}
    d.update({n: _dev(ref[n].copy()) for n in ("eps", "eps_neg", "next", "next_neg")})
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 2, 3, 8])
@pytest.mark.parametrize("gamma", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("nsr", [1.0, 5.0, 12.0])
def test_sgd_sequential_replay(dim, gamma, nsr):
    """One launch per edge replays the sequential oracle; launches over edges not yet due change nothing."""
    torch = _torch()
    N, n_epochs, seed = 24, 6, 77
    ref, emb0 = _sgd_setup(N, dim, seed=dim * 7 + int(nsr), n_epochs=n_epochs, nsr=nsr)
    a, b = lu.find_ab_params(1.0, 0.1)
    s = _sched_dev(ref)
    emb = _dev(emb0.copy())
    E = ref["head"].size
    due_later = np.flatnonzero(ref["next"] > 0)
    for n in range(n_epochs):
        alpha = 1.0 - n / float(n_epochs)
        if n == 0 and due_later.size:           # edges not due at epoch 0: a sub-range launch is a no-op
            e0 = int(due_later[0])
            e1 = e0 + 1
            while e1 < E and ref["next"][e1] > 0:
                e1 += 1
            snap = [emb.clone(), s["next"].clone(), s["next_neg"].clone()]
            lu.sgd_epoch(emb, s, n, a, b, gamma, alpha, seed, e0, e1)
            torch.cuda.synchronize()
            for t, u in zip((emb, s["next"], s["next_neg"]), snap):
                assert torch.equal(t, u)
        for e in range(E):
            lu.sgd_epoch(emb, s, n, a, b, gamma, alpha, seed, e, e + 1)
    torch.cuda.synchronize()
    host = {n: ref[n].copy() for n in ref}
    out = emb0.copy()
    uo.sgd(out, host, n_epochs, a, b, gamma, 1.0, seed)
    np.testing.assert_allclose(emb.cpu().numpy(), out, rtol=1e-5, atol=1e-5)
    np.testing.assert_array_equal(s["next"].cpu().numpy(), host["next"])
    np.testing.assert_allclose(s["next_neg"].cpu().numpy(), host["next_neg"], rtol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [2, 8])
def test_sgd_race_free_epoch(dim):
    """A perfect matching with negative sampling switched off: the edges touch disjoint vertices, so one
    launch over all of them is the sequential epoch, to 1 fp32 ulp (pow and the coefficient in CUDA)."""
    torch = _torch()
    N = 200000
    rng = np.random.default_rng(dim)
    perm = rng.permutation(N)
    head, tail = perm[0::2].astype(np.int64), perm[1::2].astype(np.int64)
    E = head.size
    eps = rng.uniform(1.0, 3.0, E)
    nxt = np.where(rng.uniform(0, 1, E) < 0.2, 2.5, 0.0)   # a fifth not due yet
    ref = dict(head=head, tail=tail, eps=eps, eps_neg=np.full(E, 1e30), next=nxt, next_neg=np.full(E, 1e30))
    emb0 = rng.uniform(0, 10, (N, dim)).astype(np.float32)
    a, b = lu.find_ab_params(1.0, 0.1)
    s = _sched_dev(ref)
    emb = _dev(emb0.copy())
    lu.sgd_epoch(emb, s, 1, a, b, 1.0, 0.9, 5)
    torch.cuda.synchronize()
    host = {n: ref[n].copy() for n in ref}
    out = emb0.copy()
    uo.sgd(out, host, 10, a, b, 1.0, 1.0, 5, epochs=range(1, 2))
    got = emb.cpu().numpy()
    ulp = np.abs(got.view(np.int32).astype(np.int64) - out.view(np.int32).astype(np.int64))
    assert ulp.max() <= 1
    moved = np.zeros(N, bool)
    moved[head[nxt <= 1]] = True
    moved[tail[nxt <= 1]] = True
    np.testing.assert_array_equal(got[~moved], emb0[~moved])
    np.testing.assert_array_equal(s["next"].cpu().numpy(), host["next"])


# ============================================================================== 10. rejections
@pytest.mark.gpu
def test_rejections():
    torch = _torch()
    N, D = 50, 4
    x = _dev(np.random.default_rng(0).standard_normal((N, D)))
    idx = torch.full((N, 101), IDX_SENTINEL, dtype=torch.int32, device="cuda")
    dist = torch.full((N, 101), float("nan"), dtype=torch.float64, device="cuda")
    wsb = int(_lib.lib().ava_b200_umap_knn_ws_bytes(N, 64, 100))
    ws = torch.zeros(wsb, dtype=torch.uint8, device="cuda")

    def knn_args(N=N, D=D, k=5, is_f32=0, ws_bytes=None):
        return (x.data_ptr(), is_f32, N, D, k, idx.data_ptr(), dist.data_ptr(), ws.data_ptr(),
                int(_lib.lib().ava_b200_umap_knn_ws_bytes(N, D, k)) if ws_bytes is None else ws_bytes, _stream())

    for kw, match in ((dict(k=0), "k"), (dict(k=101, ws_bytes=wsb), "k"), (dict(N=4, k=5, ws_bytes=wsb), "k"),
                      (dict(D=0), "D=0"), (dict(D=65), "D=65"), (dict(is_f32=2), "is_f32"),
                      (dict(ws_bytes=int(_lib.lib().ava_b200_umap_knn_ws_bytes(N, D, 5)) - 1), "workspace")):
        _expect_rejected("ava_b200_umap_knn", knn_args(**kw), (idx, dist), match)
    rho = torch.full((N,), float("nan"), dtype=torch.float64, device="cuda")
    _expect_rejected("ava_b200_umap_smooth_knn", (idx.data_ptr(), dist.data_ptr(), N, 1, 1.0, rho.data_ptr(),
                                                  rho.data_ptr(), dist.data_ptr(), rho.data_ptr(), _stream()),
                     (rho, dist), "k >= 2")
    _expect_rejected("ava_b200_umap_smooth_knn", (idx.data_ptr(), dist.data_ptr(), N, 5, -0.5, rho.data_ptr(),
                                                  rho.data_ptr(), dist.data_ptr(), rho.data_ptr(), _stream()),
                     (rho, dist), "local_connectivity")
    P = _cc_graph("star")
    rp, cl, vl = _dev(P.indptr.astype(np.int64)), _dev(P.indices.astype(np.int32)), _dev(P.data)
    verts = _dev(np.arange(10, dtype=np.int32))
    X = torch.zeros(10 * 33, dtype=torch.float64, device="cuda")
    Y = torch.full((10 * 33,), float("nan"), dtype=torch.float64, device="cuda")
    _expect_rejected("ava_b200_umap_spmm", (rp.data_ptr(), cl.data_ptr(), vl.data_ptr(), verts.data_ptr(), 10,
                                            verts.data_ptr(), vl.data_ptr(), X.data_ptr(), 33, Y.data_ptr(), _stream()),
                     (Y,), "m <= 32")
    emb = torch.full((N * 9,), float("nan"), dtype=torch.float32, device="cuda")
    _expect_rejected("ava_b200_umap_init_layout", (X.data_ptr(), None, 1.0, 10, 9, emb.data_ptr(), _stream()), (emb,),
                     "init_layout")
    e = _dev(np.zeros(4, np.int32))
    dd = torch.zeros(4, dtype=torch.float64, device="cuda")
    nx = torch.full((4,), float("nan"), dtype=torch.float64, device="cuda")

    def sgd_args(dim=2, e0=0, e1=4):
        return (emb.data_ptr(), 10, dim, e.data_ptr(), e.data_ptr(), dd.data_ptr(), dd.data_ptr(), nx.data_ptr(),
                nx.data_ptr(), e0, e1, 0, 1.0, 1.0, 1.0, 1.0, 0, _stream())

    _expect_rejected("ava_b200_umap_sgd_epoch", sgd_args(dim=9), (emb, nx), "sgd_epoch")
    _expect_rejected("ava_b200_umap_sgd_epoch", sgd_args(e0=3, e1=2), (emb, nx), "sgd_epoch")
