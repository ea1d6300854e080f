"""LatentUMAP.transform without a GPU: the transform restatement (tests/umap_transform_reference.py) against
scikit-learn and against its own definitions, the argument checks that run before any device work, the
pickled state, and the absence of a CPU fallback."""
import importlib
import pickle

import numpy as np
import pytest
import torch

from tests import umap_transform_reference as uo

lu = importlib.import_module("autoencoded-vocal-analysis_b200.data.latent_umap")
_lib = importlib.import_module("autoencoded-vocal-analysis_b200._lib")


def test_oracle_knn_query_matches_sklearn_brute():
    from sklearn.neighbors import NearestNeighbors
    rng = np.random.default_rng(0)
    x = rng.standard_normal((400, 7))
    q = np.vstack([rng.standard_normal((60, 7)), x[:5], x[:5] + 100.0])
    idx, dist = uo.knn_query(q, x, 12)
    d_ref, i_ref = NearestNeighbors(n_neighbors=12, algorithm='brute').fit(x).kneighbors(q)
    np.testing.assert_array_equal(idx, i_ref)
    np.testing.assert_allclose(dist, d_ref, rtol=1e-9, atol=1e-12)
    np.testing.assert_array_equal(idx[60:65, 0], np.arange(5))   # a query equal to a fitted row: that row first
    assert (dist[60:65, 0] == 0.0).all()


def test_oracle_knn_query_duplicates_lowest_index_first():
    x = np.repeat(np.arange(6.0)[:, None], 3, axis=0)   # each value three times
    idx, dist = uo.knn_query(x[[4, 9, 17]], x, 3)
    np.testing.assert_array_equal(idx, [[3, 4, 5], [9, 10, 11], [15, 16, 17]])
    assert (dist == 0.0).all()


def test_oracle_query_graph_is_bipartite_and_column_sorted():
    rng = np.random.default_rng(1)
    x = rng.standard_normal((200, 4))
    idx, dist = uo.knn_query(x[:30], x, 10)
    rho, sig, cols, w = uo.query_graph(idx, dist, 10, local_connectivity=1.0)
    assert (np.diff(cols, axis=1) > 0).all()
    assert (rho == 0.0).all()                                    # local_connectivity 1 - 1 = 0
    # query i equals fitted row i: its weight there is 1, not zeroed as in the fit's graph
    np.testing.assert_array_equal(w[cols == np.arange(30)[:, None]], 1.0)
    sref, rref = uo.smooth_knn_dist(dist, 10, local_connectivity=0.0)
    np.testing.assert_array_equal(sig, sref)
    np.testing.assert_array_equal(rho, rref)


def test_oracle_init_transform():
    emb = np.array([[0.0, 0.0], [1.0, 2.0], [3.0, -1.0]], dtype=np.float32)
    cols = np.array([[0, 1, 2], [0, 1, 2], [0, 1, 2]])
    w = np.array([[0.5, 0.25, 0.25], [0.5, 1.0, 0.2], [1.0, 1.0, 0.3]])
    out = uo.init_transform(cols, w, emb)
    np.testing.assert_array_equal(out[0], np.float32([0.25 * 1 + 0.25 * 3, 0.25 * 2 - 0.25]))
    np.testing.assert_array_equal(out[1], emb[1])               # a weight of 1 copies that row and stops
    np.testing.assert_array_equal(out[2], emb[0])


def test_oracle_transform_schedule_prunes_and_keeps_row_major_order():
    w = np.array([[1.0, 0.5, 0.001], [0.2, 0.02, 0.9]])
    cols = np.array([[3, 5, 7], [0, 1, 2]])
    s = uo.transform_schedule(cols, w, 10)
    np.testing.assert_array_equal(s["head"], [0, 0, 1, 1])
    np.testing.assert_array_equal(s["tail"], [3, 5, 0, 2])
    np.testing.assert_allclose(s["eps"], [1.0, 2.0, 5.0, 1.0 / 0.9])


def test_transform_n_epochs():
    assert lu.transform_n_epochs(None, 10000) == 100
    assert lu.transform_n_epochs(None, 10001) == 30
    assert lu.transform_n_epochs(200, 5) == 66
    assert lu.transform_n_epochs(2, 5) == 0


def _fitted_on_host(N=20, D=4, dim=2):
    """A model in the state a fit leaves, as unpickling leaves it (tensors on the host)."""
    um = lu.LatentUMAP(n_neighbors=5, random_state=3)
    um.__dict__.update(_fit_x=torch.zeros(N, D, dtype=torch.float64), _fit_emb=torch.zeros(N, dim), _k=5,
                       _seed_=3, a_=1.0, b_=1.0, n_epochs_=200, embedding_=np.zeros((N, dim), np.float32),
                       _graph=None, _graph_dev=None)
    return um


def test_transform_argument_checks():
    with pytest.raises(RuntimeError):
        lu.LatentUMAP().transform(np.zeros((3, 4)))                # not fitted
    um = _fitted_on_host()
    with pytest.raises(ValueError):
        um.transform(np.zeros((3, 5)))                               # wrong column count
    with pytest.raises(ValueError):
        um.transform(np.zeros(4))                                    # not [Nq, D]
    bad = np.zeros((3, 4))
    bad[1, 2] = np.nan
    with pytest.raises(ValueError):
        um.transform(bad)
    bad[1, 2] = -np.inf
    with pytest.raises(ValueError):
        um.transform(torch.from_numpy(bad))


def test_pickle_keeps_the_fitted_state_on_the_host():
    um = _fitted_on_host()
    back = pickle.loads(pickle.dumps(um))
    assert torch.equal(back._fit_x, um._fit_x) and not back._fit_x.is_cuda
    assert back._k == 5 and back._seed_ == 3 and back._graph_dev is None


def test_no_cpu_fallback_in_transform(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    um = _fitted_on_host()
    with pytest.raises(_lib.AvaB200Error):
        um.transform(np.ones((2, 4)))
