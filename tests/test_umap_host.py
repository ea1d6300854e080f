"""CPU checks of the UMAP restatement (oracle/umap_oracle.py) and of LatentUMAP's host side: argument
validation, the a/b curve fit, and no CPU fallback."""
import importlib

import numpy as np
import pytest
import scipy.sparse
import torch

from oracle import umap_oracle as uo

lu = importlib.import_module("autoencoded-vocal-analysis_b200.data.latent_umap")
_lib = importlib.import_module("autoencoded-vocal-analysis_b200._lib")


def test_oracle_knn_matches_sklearn_brute():
    from sklearn.neighbors import NearestNeighbors
    rng = np.random.default_rng(0)
    x = rng.standard_normal((300, 12))
    idx, dist = uo.knn(x, 10)
    d_ref, i_ref = NearestNeighbors(n_neighbors=10, algorithm='brute').fit(x).kneighbors(x)
    np.testing.assert_array_equal(idx, i_ref)
    np.testing.assert_allclose(dist, d_ref, rtol=1e-10, atol=1e-12)
    assert (idx[:, 0] == np.arange(300)).all()


def test_oracle_knn_orders_duplicates_self_first():
    x = np.repeat(np.arange(6.0).reshape(3, 2), 4, axis=0)     # every row has three exact copies
    idx, dist = uo.knn(x, 4)
    for i in range(12):
        assert idx[i, 0] == i
        assert sorted(idx[i]) == [j for j in range(12) if j // 4 == i // 4]
        np.testing.assert_array_equal(dist[i], 0.0)


def test_oracle_graph_matches_scipy_restatement():
    rng = np.random.default_rng(1)
    x = rng.standard_normal((200, 6))
    k = 8
    idx, dist = uo.knn(x, k)
    sig, rho = uo.smooth_knn_dist(dist, k)
    w = uo.membership_strengths(idx, dist, sig, rho)
    assert (w[:, 0] == 0).all() and (w[np.arange(200), 1] == 1.0).all()   # self 0; nearest other at rho
    # smooth_knn_dist's target: sum_j>=1 exp(-(d - rho)/sigma) = log2(k)
    psum = np.exp(-np.maximum(dist[:, 1:] - rho[:, None], 0) / sig[:, None]).sum(1)
    np.testing.assert_allclose(psum, np.log2(k), atol=1e-4)
    A = scipy.sparse.coo_matrix((w.ravel(), (np.repeat(np.arange(200), k), idx.ravel())), shape=(200, 200)).tocsr()
    A.eliminate_zeros()
    ref = (A + A.T - A.multiply(A.T)).tocsr()
    ref.sort_indices()
    P = uo.fuzzy_union(idx, w)
    np.testing.assert_array_equal(P.indptr, ref.indptr)
    np.testing.assert_array_equal(P.indices, ref.indices)
    np.testing.assert_allclose(P.data, ref.data, rtol=1e-15)
    s = uo.prune_and_schedule(P, 10)
    assert (s["weights"] >= P.data.max() / 10).all() and s["head"].size == (P.data >= P.data.max() / 10).sum()
    np.testing.assert_allclose(s["eps"] * s["weights"] / s["weights"].max(), 1.0)


@pytest.mark.parametrize("min_dist,a_ref,b_ref", [(0.1, 1.5769, 0.8951), (0.5, 0.5830, 1.3341)])
def test_ab_params(min_dist, a_ref, b_ref):
    from scipy.optimize import curve_fit
    xv = np.linspace(0, 3.0, 300)
    yv = np.where(xv < min_dist, 1.0, np.exp(-(xv - min_dist)))
    (a, b), _ = curve_fit(lambda x, a, b: 1.0 / (1.0 + a * x ** (2 * b)), xv, yv)
    got = lu.find_ab_params(1.0, min_dist)
    np.testing.assert_allclose(got, (a, b), rtol=1e-12)
    np.testing.assert_allclose(got, (a_ref, b_ref), atol=2e-4)


def test_numba_sgd_equals_python_sgd():
    rng = np.random.default_rng(2)
    x = rng.standard_normal((25, 4))
    idx, dist = uo.knn(x, 5)
    sig, rho = uo.smooth_knn_dist(dist, 5)
    P = uo.fuzzy_union(idx, uo.membership_strengths(idx, dist, sig, rho))
    s1 = uo.prune_and_schedule(P, 15)
    s2 = {k: v.copy() for k, v in s1.items()}
    e0 = uo.init_embedding(uo.random_block(3, 1 << 32, (25, 2), 0, 10.0))
    e1, e2 = e0.copy(), e0.copy()
    a, b = lu.find_ab_params(1.0, 0.1)
    uo.sgd(e1, s1, 15, a, b, 1.0, 1.0, 3)
    uo._sgd_py(e2, s2["head"], s2["tail"], s2["eps"], s2["eps_neg"], s2["next"], s2["next_neg"], 15, a, b, 1.0, 1.0,
               3, range(15))
    np.testing.assert_allclose(e1, e2, rtol=1e-6, atol=1e-6)
    assert not np.array_equal(e1, e0)


def test_argument_validation():
    x = np.zeros((20, 4))
    for kw in (dict(metric='cosine'), dict(n_components=0), dict(n_components=9), dict(n_neighbors=1),
               dict(n_neighbors=101), dict(init='pca'), dict(n_epochs=0), dict(min_dist=2.0)):
        with pytest.raises(ValueError):
            lu.LatentUMAP(**kw).fit_transform(x)
    with pytest.raises(ValueError):
        lu.LatentUMAP().fit_transform(np.zeros((20, 65)))
    with pytest.raises(ValueError):
        lu.LatentUMAP().fit_transform(np.zeros((20,)))
    bad = np.zeros((20, 4))
    bad[2, 2] = np.inf
    with pytest.raises(ValueError):
        lu.LatentUMAP().fit_transform(bad)
    with pytest.raises(ValueError):
        lu.LatentUMAP(init=np.zeros((19, 2))).fit_transform(x)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without CUDA")
def test_no_cpu_fallback():
    with pytest.raises(_lib.AvaB200Error):
        lu.LatentUMAP().fit_transform(np.random.default_rng(0).standard_normal((50, 8)))


def test_oracle_meta_positions_many_components():
    """More than 2 * n_components components: the PCA projection of the component centroids, scaled to
    unit minimum spacing (the few-component case is +-unit axes)."""
    from oracle.pca_oracle import pca_fit_transform
    rng = np.random.default_rng(4)
    centers = rng.standard_normal((6, 5)) * 20
    labels = np.repeat(np.arange(6), 30)
    x = centers[labels] + rng.standard_normal((180, 5))
    meta = uo.meta_positions(x, labels, 6, 2)
    assert meta.shape == (6, 2)
    dd = np.sqrt(((meta[:, None] - meta[None]) ** 2).sum(-1))
    np.testing.assert_allclose(dd[~np.eye(6, dtype=bool)].min(), 1.0, rtol=1e-12)
    cent = np.stack([x[labels == c].mean(0) for c in range(6)])
    proj = pca_fit_transform(cent, 2)[0]
    np.testing.assert_allclose(meta * (proj / meta)[0, 0], proj, rtol=1e-9, atol=1e-9)
    np.testing.assert_array_equal(uo.meta_positions(x, labels, 3, 2), [[1, 0], [0, 1], [-1, 0]])
