"""LatentUMAP on the device (csrc/umap.cu) against the CPU restatement oracle/umap_oracle.py: exact kNN,
the fuzzy graph and its schedule element by element, the spectral initialisation by subspace angle,
the SGD by sequential equivalence, the whole fit by quality metrics, and the edge cases."""
import importlib
import warnings

import numpy as np
import pytest
import torch

from oracle import umap_oracle as uo

pytestmark = pytest.mark.gpu
lu = importlib.import_module("autoencoded-vocal-analysis_b200.data.latent_umap")


def blobs(n, d, centers=10, seed=0, spread=10.0):
    rng = np.random.default_rng(seed)
    c = rng.standard_normal((centers, d)) * spread
    lab = rng.integers(0, centers, n)
    return c[lab] + rng.standard_normal((n, d)), lab


def dup_rows(n, d, seed=0):
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((max(n // 3, 1), d))
    return base[rng.integers(0, base.shape[0], n)]


# ----------------------------------------------------------------------------------------- kNN
@pytest.mark.parametrize("N", [37, 4100, 20000])
@pytest.mark.parametrize("D", [8, 32, 64])
@pytest.mark.parametrize("k", [2, 20, 100])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("data", ["blobs", "duplicates"])
def test_knn_exact(N, D, k, dtype, data):
    if k > N:
        pytest.skip("k > N")
    x = blobs(N, D, seed=N + D)[0] if data == "blobs" else dup_rows(N, D, seed=N + D)
    xd = torch.from_numpy(x).to(dtype).cuda()
    idx, dist = lu.knn(xd, k)
    torch.cuda.synchronize()
    x64 = xd.double()
    q = torch.arange(N, device="cuda") if N <= 2000 else torch.randperm(N, generator=torch.Generator().manual_seed(0))[:2000].cuda()
    ref = torch.cdist(x64[q], x64, compute_mode="donot_use_mm_for_euclid_dist")        # difference form, fp64
    ii = idx[q].long()
    assert bool((ii[:, 0] == q).all())                                                  # the row itself first
    assert bool((ii >= 0).all()) and bool((ii < N).all())
    assert all(len(set(r)) == k for r in ii.cpu().numpy().tolist())
    true_d = torch.gather(ref, 1, ii)
    kth = torch.sort(ref, 1).values[:, k - 1:k]
    assert bool((true_d <= kth * (1 + 1e-6)).all())
    got = dist[q]
    assert bool((got - true_d).abs().le(1e-12 * true_d.abs() + 1e-300).all())
    # identical lists where no near-tie: reference order by (distance, not-self, index)
    refn, qn = ref.cpu().numpy(), q.cpu().numpy()
    ii_n = ii.cpu().numpy()
    checked = 0
    rows = range(0, len(qn), max(1, len(qn) // 300))
    for r in rows:
        notself = np.ones(N, dtype=np.int64)
        notself[qn[r]] = 0
        order = np.lexsort((np.arange(N), notself, refn[r]))[:k + 1]
        ds = refn[r, order]
        gaps = np.diff(ds)
        if np.any((gaps > 0) & (gaps <= 1e-9 * np.maximum(ds[1:], 1e-300))):
            continue
        np.testing.assert_array_equal(ii_n[r], order[:k])
        checked += 1
    assert checked >= len(rows) // 2


# ---------------------------------------------------------------------- graph and schedule
@pytest.mark.parametrize("n_epochs", [500, 7])
def test_graph_and_schedule_match_oracle(n_epochs):
    x, _ = blobs(600, 16, centers=4, seed=3, spread=3.0)
    k = 15
    xd = torch.from_numpy(x).cuda()
    out = []
    for _ in range(2):
        idx, dist = lu.knn(xd, k)
        g = lu.fuzzy_graph(idx, dist)
        s = lu.edge_schedule(g, n_epochs)
        torch.cuda.synchronize()
        out.append((idx, dist, g, s))
    (idx, dist, g, s), (idx2, dist2, g2, s2) = out
    for a, b in [(idx, idx2), (dist, dist2)] + [(g[n], g2[n]) for n in ("rho", "sigma", "weights", "rows", "cols",
                                                                          "vals", "rowptr")] + \
            [(s[n], s2[n]) for n in ("head", "tail", "eps", "eps_neg", "next", "next_neg")]:
        assert torch.equal(a, b)                                                         # bitwise repeatable
    I, Dd = idx.cpu().numpy().astype(np.int64), dist.cpu().numpy()
    sig, rho = uo.smooth_knn_dist(Dd, k)
    np.testing.assert_allclose(g["rho"].cpu().numpy(), rho, rtol=1e-9, atol=0)
    np.testing.assert_allclose(g["sigma"].cpu().numpy(), sig, rtol=1e-9, atol=0)
    w = uo.membership_strengths(I, Dd, sig, rho)
    np.testing.assert_allclose(g["weights"].cpu().numpy(), w, rtol=1e-9, atol=1e-12)
    P = uo.fuzzy_union(I, w)
    np.testing.assert_array_equal(g["rowptr"].cpu().numpy(), P.indptr)
    np.testing.assert_array_equal(g["cols"].cpu().numpy(), P.indices)
    np.testing.assert_allclose(g["vals"].cpu().numpy(), P.data, rtol=1e-9, atol=1e-12)
    ref = uo.prune_and_schedule(P, n_epochs)
    np.testing.assert_array_equal(s["head"].cpu().numpy(), ref["head"])
    np.testing.assert_array_equal(s["tail"].cpu().numpy(), ref["tail"])
    for n in ("eps", "eps_neg", "next", "next_neg"):
        np.testing.assert_allclose(s[n].cpu().numpy(), ref[n], rtol=1e-9, atol=0)
    if n_epochs == 7:
        assert ref["head"].size < P.nnz                                                   # pruning happened


# ------------------------------------------------------------------------------- spectral
def _sin_theta(A, B):
    Q1, _ = np.linalg.qr(A)
    Q2, _ = np.linalg.qr(B)
    s = np.linalg.svd(Q1.T @ Q2, compute_uv=False)
    return float(np.sqrt(max(0.0, 1.0 - s.min() ** 2)))


def _graph_of(x, k):
    idx, dist = lu.knn(torch.from_numpy(x).cuda(), k)
    return lu.fuzzy_graph(idx, dist)


def test_spectral_connected_matches_eigsh():
    rng = np.random.default_rng(0)
    n = 4000
    x = np.hstack([rng.uniform(0, 3, (n, 1)), rng.uniform(0, 1, (n, 1)), 0.01 * rng.standard_normal((n, 6))])
    g = _graph_of(x, 15)
    lay, msgs = lu.spectral_layout(torch.from_numpy(x).cuda(), g, 2, 5)
    lay2, _ = lu.spectral_layout(torch.from_numpy(x).cuda(), g, 2, 5)
    assert torch.equal(lay, lay2) and msgs == []
    P = _host_csr(g)
    _, V = uo.laplacian_vectors(P, 2)
    assert _sin_theta(lay.cpu().numpy(), V) <= 1e-3
    emb = lu.init_embedding(lay, 5, True, lay.device)
    emb2 = lu.init_embedding(lay2, 5, True, lay.device)
    assert torch.equal(emb, emb2)
    e = emb.cpu().numpy()
    np.testing.assert_allclose(e.min(0), 0.0, atol=1e-6)
    np.testing.assert_allclose(e.max(0), 10.0, rtol=1e-6)


def _host_csr(g):
    import scipy.sparse
    return scipy.sparse.csr_matrix((g["vals"].cpu().numpy(), g["cols"].cpu().numpy(), g["rowptr"].cpu().numpy()),
                                   shape=(g["n"], g["n"]))


def test_spectral_three_components_placement():
    rng = np.random.default_rng(1)
    centers = np.array([[0.0] * 8, [100.0] + [0.0] * 7, [0.0, 100.0] + [0.0] * 6])
    lab = np.repeat(np.arange(3), [300, 250, 200])
    # anisotropic blobs: the two wanted eigenvectors of each component are separated from the third
    x = centers[lab] + rng.standard_normal((750, 8)) * np.array([3.0, 1.5] + [0.3] * 6)
    x, lab = x[rng.permutation(750)], None
    g = _graph_of(x, 5)
    labels = lu.connected_components(g).cpu().numpy()
    P = _host_csr(g)
    ref_lay, ref_lab, meta, half = uo.spectral_layout(x, P, 2)
    assert len(np.unique(labels)) == 3
    # components numbered by their smallest vertex, as scipy numbers them
    comp = np.searchsorted(np.unique(labels), labels)
    np.testing.assert_array_equal(comp, ref_lab)
    np.testing.assert_array_equal(meta, [[1, 0], [0, 1], [-1, 0]])
    np.testing.assert_allclose(half, [np.sqrt(2) / 2] * 3)
    lay, msgs = lu.spectral_layout(torch.from_numpy(x).cuda(), g, 2, 9)
    lay2, _ = lu.spectral_layout(torch.from_numpy(x).cuda(), g, 2, 9)
    assert torch.equal(lay, lay2) and msgs == []
    lay = lay.cpu().numpy()
    for c in range(3):
        sel = comp == c
        off = lay[sel] - meta[c]
        np.testing.assert_allclose(np.abs(off).max(), half[c], rtol=1e-12)
        assert _sin_theta(off, ref_lay[sel] - meta[c]) <= 1e-3


# ---------------------------------------------------------------------------- SGD, sequential
def test_sgd_edge_by_edge_matches_sequential_oracle():
    x, _ = blobs(30, 8, centers=3, seed=4, spread=4.0)
    n_epochs, seed = 20, 123
    g = _graph_of(x, 5)
    s = lu.edge_schedule(g, n_epochs)
    emb = lu.init_embedding(lu.random_block(seed, 1 << 32, (30, 2), 0, 10.0, "cuda"), seed, False, "cuda")
    host = {n: s[n].cpu().numpy().copy() for n in ("eps", "eps_neg", "next", "next_neg")}
    host["head"] = s["head"].cpu().numpy().astype(np.int64)
    host["tail"] = s["tail"].cpu().numpy().astype(np.int64)
    ref = emb.cpu().numpy().copy()
    a, b = lu.find_ab_params(1.0, 0.1)
    n_edges = s["head"].numel()
    for n in range(n_epochs):
        alpha = 1.0 * (1.0 - n / float(n_epochs))
        for e in range(n_edges):
            lu.sgd_epoch(emb, s, n, a, b, 1.0, alpha, seed, e, e + 1)
    torch.cuda.synchronize()
    uo.sgd(ref, host, n_epochs, a, b, 1.0, 1.0, seed)
    got = emb.cpu().numpy()
    np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(s["next"].cpu().numpy(), host["next"], rtol=1e-12)
    np.testing.assert_allclose(s["next_neg"].cpu().numpy(), host["next_neg"], rtol=1e-12)


# ------------------------------------------------------------------------------ whole fit
def _trust(x, e, n_neighbors=20):
    from sklearn.manifold import trustworthiness
    return trustworthiness(x, e, n_neighbors=n_neighbors)


def _one_nn(e, lab):
    from sklearn.neighbors import NearestNeighbors
    nb = NearestNeighbors(n_neighbors=2).fit(e).kneighbors(e, return_distance=False)
    return float((lab[nb[:, 1]] == lab).mean())


def test_whole_fit_quality():
    x, lab = blobs(20000, 32, centers=10, seed=7)
    um = lu.LatentUMAP(n_neighbors=20, min_dist=0.1, random_state=42)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        e1 = um.fit_transform(x)
        e2 = lu.LatentUMAP(n_neighbors=20, min_dist=0.1, random_state=42).fit_transform(x)
    assert e1.dtype == np.float32 and e1.shape == (20000, 2) and np.isfinite(e1).all()
    assert um.knn_indices_.shape == (20000, 20) and um.knn_dists_.shape == (20000, 20)
    assert um.n_epochs_ == 200 and um.graph_.shape == (20000, 20000)
    assert _one_nn(e1, lab) >= 0.98
    sub = np.random.default_rng(0).choice(20000, 4000, replace=False)   # trustworthiness is O(N^2) in memory
    t1, t2 = _trust(x[sub], e1[sub]), _trust(x[sub], e2[sub])
    assert abs(t1 - t2) <= 0.01
    # the oracle's sequential SGD at N = 20 000 takes minutes on the CPU: compare on the first 3000 rows
    xs, n = x[:3000], 3000
    dev_fit = lu.LatentUMAP(n_neighbors=20, min_dist=0.1, random_state=42)
    es = dev_fit.fit_transform(xs)
    ref = uo.fit(xs, 20, seed=42, knn_lists=(dev_fit.knn_indices_.astype(np.int64), dev_fit.knn_dists_))
    assert np.isfinite(ref).all() and n == es.shape[0]
    assert _trust(xs, es) >= _trust(xs, ref) - 0.02


# ------------------------------------------------------------------------------ edge cases
def test_edge_cases():
    z = lu.LatentUMAP().fit_transform(np.ones((1, 5)))
    np.testing.assert_array_equal(z, np.zeros((1, 2), dtype=np.float32))
    x, _ = blobs(10, 4, centers=2, seed=2)
    with pytest.warns(UserWarning):
        e = lu.LatentUMAP(n_neighbors=15, random_state=0).fit_transform(x)
    assert e.shape == (10, 2) and np.isfinite(e).all()
    xn = x.copy()
    xn[3, 1] = np.nan
    with pytest.raises(ValueError):
        lu.LatentUMAP().fit_transform(xn)
    with pytest.raises(ValueError):
        lu.LatentUMAP().fit_transform(torch.from_numpy(xn).cuda())
    x3, _ = blobs(500, 16, centers=3, seed=5)
    um = lu.LatentUMAP(n_components=3, random_state=1)
    e3 = um.fit_transform_device(torch.from_numpy(x3).float().cuda())
    assert e3.is_cuda and e3.shape == (500, 3) and bool(torch.isfinite(e3).all())
    er = lu.LatentUMAP(init='random', random_state=1, n_epochs=50).fit_transform(x3)
    assert er.shape == (500, 2) and np.isfinite(er).all()
    ea = lu.LatentUMAP(init=np.random.default_rng(0).standard_normal((500, 2)), n_epochs=50).fit_transform(x3)
    assert ea.shape == (500, 2) and np.isfinite(ea).all()
