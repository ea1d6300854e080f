"""LatentUMAP.transform on the device (csrc/umap.cu) against the CPU restatement in tests/umap_transform_reference.py:
the query kNN (exact, over shapes, scales, offsets and slice counts), the bipartite memberships, the
initialisation (bitwise), the race-free layout (bitwise repeatable, and the sequential oracle), the whole
transform by label agreement, and the edge cases."""
import importlib
import pickle
import warnings

import numpy as np
import pytest
import torch

from tests import umap_transform_reference as uo

pytestmark = pytest.mark.gpu
lu = importlib.import_module("autoencoded-vocal-analysis_b200.data.latent_umap")


def blobs(n, d, centers=10, seed=0, spread=10.0):
    rng = np.random.default_rng(seed)
    c = rng.standard_normal((centers, d)) * spread
    lab = rng.integers(0, centers, n)
    return c[lab] + rng.standard_normal((n, d)), lab


def _check_exact(q, x, k, idx, dist, min_checked=0.5, tie=1e-9):
    """Every returned row is a true k-nearest neighbour with its fp64 distance, and the lists are the
    reference's (distance, index) order wherever no two of the first k + 1 distances are near-ties."""
    q64, x64 = q.double(), x.double()
    ref = torch.cdist(q64, x64, compute_mode="donot_use_mm_for_euclid_dist")
    N = x.shape[0]
    ii = idx.long()
    assert bool((ii >= 0).all()) and bool((ii < N).all())
    if k > 1:
        assert bool((torch.sort(ii, 1).values.diff(dim=1) > 0).all())       # distinct rows
    true_d = torch.gather(ref, 1, ii)
    sd, si = torch.sort(ref, dim=1, stable=True)                     # ties by index
    assert bool((true_d <= sd[:, k - 1:k] * (1 + 1e-12)).all())
    assert bool((dist - true_d).abs().le(1e-12 * true_d.abs() + 1e-300).all())
    m = min(k + 1, N)
    gaps = sd[:, 1:m] - sd[:, :m - 1]
    clean = ~((gaps > 0) & (gaps <= tie * sd[:, 1:m].clamp_min(1e-300))).any(1)
    assert bool((ii[clean] == si[clean, :k]).all())
    assert int(clean.sum()) >= min_checked * q.shape[0]


# ----------------------------------------------------------------------------------- query kNN
@pytest.mark.parametrize("Nq", [1, 63, 64, 65, 3000])
@pytest.mark.parametrize("N", [2, 129, 4100, 20000])
@pytest.mark.parametrize("D", [1, 8, 33, 64])
@pytest.mark.parametrize("k", [1, 2, 20, 100])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_knn_query_exact(Nq, N, D, k, dtype):
    if k > N:
        pytest.skip("k > N")
    x, _ = blobs(N, D, seed=N + D)
    q, _ = blobs(Nq, D, seed=N + D + 1)
    xd, qd = torch.from_numpy(x).to(dtype).cuda(), torch.from_numpy(q).to(dtype).cuda()
    idx, dist = lu.knn_query(qd, xd, k)
    idx2, dist2 = lu.knn_query(qd, xd, k)
    torch.cuda.synchronize()
    assert torch.equal(idx, idx2) and torch.equal(dist, dist2)   # bitwise repeatable
    _check_exact(qd, xd, k, idx, dist, min_checked=0.5 if D > 1 else 0.0)


def test_knn_query_slices_small_queries_large_data():
    """Few queries against many rows split the rows into slices; every slice count gives the exact lists."""
    x, _ = blobs(200000, 32, seed=11)
    q, _ = blobs(257, 32, seed=12)
    xd, qd = torch.from_numpy(x).float().cuda(), torch.from_numpy(q).float().cuda()
    for nq in (1, 5, 128, 257):
        for k in (1, 20, 100):
            idx, dist = lu.knn_query(qd[:nq].contiguous(), xd, k)
            _check_exact(qd[:nq], xd, k, idx, dist)
    # the workspace holds S * KP candidates per query: more than one slice for one query CTA
    lib = lu._lib.lib()
    per_query_1 = lib.ava_b200_umap_knn_query_ws_bytes(2, 200000, 32, 20) - lib.ava_b200_umap_knn_query_ws_bytes(
        1, 200000, 32, 20)
    assert per_query_1 > 32 * 4 + 4 + 4 + 32 * 4 + 8


@pytest.mark.parametrize("s", [-120, -60, -1, 1, 60, 100])
def test_knn_query_scale_sweep(s):
    x, _ = blobs(4100, 8, seed=5)
    q, _ = blobs(300, 8, seed=6)
    xd, qd = torch.from_numpy(x).cuda(), torch.from_numpy(q).cuda()
    idx0, dist0 = lu.knn_query(qd, xd, 20)
    f = 2.0 ** s
    idx, dist = lu.knn_query(qd * f, xd * f, 20)
    assert torch.equal(idx, idx0)
    assert torch.equal(dist, dist0 * f)


@pytest.mark.parametrize("offset", [1e3, 1e6])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_knn_query_offsets(offset, dtype):
    x, _ = blobs(4100, 16, seed=7, spread=3.0)
    q, _ = blobs(500, 16, seed=8, spread=3.0)
    xd = (torch.from_numpy(x) + offset).to(dtype).cuda()
    qd = (torch.from_numpy(q) + offset).to(dtype).cuda()
    idx, dist = lu.knn_query(qd, xd, 20)
    _check_exact(qd, xd, 20, idx, dist)


def test_knn_query_far_queries_and_tight_far_clusters():
    rng = np.random.default_rng(9)
    x = rng.standard_normal((3000, 8))
    q = x[:200] + 1e6                                           # 10^6 away from data near 0
    xd, qd = torch.from_numpy(x).cuda(), torch.from_numpy(q).cuda()
    idx, dist = lu.knn_query(qd, xd, 20)
    # the distances differ by ~1e-10 of themselves: near-ties only below the fp64 rounding of either side
    _check_exact(qd, xd, 20, idx, dist, tie=1e-13)
    c = np.where(rng.random((4000, 1)) < 0.5, -1e3, 1e3)        # tight clusters far apart: the fp64 rescan
    x = c + 1e-3 * rng.standard_normal((4000, 8))
    q = np.where(rng.random((300, 1)) < 0.5, -1e3, 1e3) + 1e-3 * rng.standard_normal((300, 8))
    xd, qd = torch.from_numpy(x).cuda(), torch.from_numpy(q).cuda()
    idx, dist = lu.knn_query(qd, xd, 20)
    _check_exact(qd, xd, 20, idx, dist)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_knn_query_equal_rows_and_duplicates(dtype):
    rng = np.random.default_rng(10)
    base = rng.standard_normal((1500, 12))
    x = base[rng.integers(0, 1500, 5000)]                        # duplicated rows
    sel = rng.choice(5000, 400, replace=False)
    xd = torch.from_numpy(x).to(dtype).cuda()
    idx, dist = lu.knn_query(xd[sel].contiguous(), xd, 10)
    xs = xd.cpu().numpy()
    first = np.array([np.flatnonzero((xs == xs[s]).all(1))[0] for s in sel])
    np.testing.assert_array_equal(idx[:, 0].cpu().numpy(), first)   # lowest index among equal rows
    assert bool((dist[:, 0] == 0).all())
    _check_exact(xd[sel], xd, 10, idx, dist, min_checked=0.0)


@pytest.mark.parametrize("N", [129, 4100, 20000])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_knn_query_of_the_data_equals_fit_knn(N, dtype):
    x, _ = blobs(N, 33, seed=N)
    xd = torch.from_numpy(x).to(dtype).cuda()
    k = min(20, N)
    i1, d1 = lu.knn(xd, k)
    i2, d2 = lu.knn_query(xd, xd, k)
    assert torch.equal(i1, i2) and torch.equal(d1, d2)


# --------------------------------------------------------------------------------- memberships
@pytest.mark.parametrize("lc", [0.0, 1.0, 1.5, 3.0])
def test_query_graph_matches_oracle(lc):
    x, _ = blobs(3000, 16, seed=13, spread=3.0)
    q = np.vstack([blobs(400, 16, seed=14, spread=3.0)[0], x[:50]])
    xd, qd = torch.from_numpy(x).cuda(), torch.from_numpy(q).cuda()
    k = 15
    idx, dist = lu.knn_query(qd, xd, k)
    g = lu.query_graph(idx, dist, lc)
    g2 = lu.query_graph(idx, dist, lc)
    for n in ("rho", "sigma", "cols", "weights"):
        assert torch.equal(g[n], g2[n])
    rho, sig, cols, w = uo.query_graph(idx.cpu().numpy().astype(np.int64), dist.cpu().numpy(), k, lc)
    np.testing.assert_allclose(g["rho"].cpu().numpy(), rho, rtol=1e-9, atol=0)
    np.testing.assert_allclose(g["sigma"].cpu().numpy(), sig, rtol=1e-9, atol=0)
    np.testing.assert_array_equal(g["cols"].cpu().numpy(), cols)
    np.testing.assert_allclose(g["weights"].cpu().numpy(), w, rtol=1e-9, atol=1e-12)
    # the last 50 queries equal fitted rows 0..49: their own column keeps a positive weight
    gw, gc = g["weights"].cpu().numpy()[400:], g["cols"].cpu().numpy()[400:]
    assert (gw[gc == np.arange(50)[:, None]] > 0).all()


# ------------------------------------------------------------------------------ initialisation
def test_init_transform_bitwise():
    x, _ = blobs(3000, 16, seed=15, spread=3.0)
    q = np.vstack([blobs(600, 16, seed=16, spread=3.0)[0], x[100:140]])
    xd, qd = torch.from_numpy(x).cuda(), torch.from_numpy(q).cuda()
    idx, dist = lu.knn_query(qd, xd, 20)
    g = lu.query_graph(idx, dist, 1.0)
    emb = torch.from_numpy(np.random.default_rng(0).uniform(0, 10, (3000, 3)).astype(np.float32)).cuda()
    out = lu.init_transform(g, emb)
    ref = uo.init_transform(g["cols"].cpu().numpy(), g["weights"].cpu().numpy(), emb.cpu().numpy())
    np.testing.assert_array_equal(out.cpu().numpy(), ref)
    assert torch.equal(out[600:], emb[100:140])                  # a query equal to a fitted row starts there


# ------------------------------------------------------------------------------------- layout
@pytest.mark.parametrize("dim", [1, 2, 3, 8])
@pytest.mark.parametrize("gamma", [0.0, 1.0])
@pytest.mark.parametrize("nsr", [1, 5])
def test_sgd_transform_matches_sequential_oracle(dim, gamma, nsr):
    x, _ = blobs(400, 8, centers=4, seed=17, spread=4.0)
    q, _ = blobs(60, 8, centers=4, seed=18, spread=4.0)
    xd, qd = torch.from_numpy(x).cuda(), torch.from_numpy(q).cuda()
    emb = torch.from_numpy(np.random.default_rng(dim).uniform(0, 10, (400, dim)).astype(np.float32)).cuda()
    emb_before = emb.clone()
    idx, dist = lu.knn_query(qd, xd, 10)
    g = lu.query_graph(idx, dist, 1.0)
    init = lu.init_transform(g, emb)
    n_epochs, seed, a, b = 30, 77, *lu.find_ab_params(1.0, 0.1)
    outs = []
    for _ in range(2):
        s = lu.transform_schedule(g, n_epochs, nsr)
        outs.append(lu.sgd_transform(init.clone(), emb, s, n_epochs, a, b, gamma, 0.25, seed))
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])                          # race-free: bitwise repeatable
    assert torch.equal(emb, emb_before)                           # the fitted embedding is only read
    ref_s = uo.transform_schedule(g["cols"].cpu().numpy().astype(np.int64), g["weights"].cpu().numpy(), n_epochs,
                                  nsr)
    np.testing.assert_array_equal(s["tail"].cpu().numpy(), ref_s["tail"])
    np.testing.assert_array_equal(np.diff(s["rowptr"].cpu().numpy()), np.bincount(ref_s["head"], minlength=60))
    ref = uo.sgd_transform(init.cpu().numpy().copy(), emb.cpu().numpy(), ref_s, n_epochs, a, b, gamma, 0.25, seed)
    np.testing.assert_allclose(outs[0].cpu().numpy(), ref, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(s["next"].cpu().numpy(), ref_s["next"], rtol=1e-12)
    np.testing.assert_allclose(s["next_neg"].cpu().numpy(), ref_s["next_neg"], rtol=1e-12)


def test_zero_transform_epochs_return_the_initialisation():
    x, _ = blobs(2000, 8, seed=19)
    q, _ = blobs(100, 8, seed=20)
    um = lu.LatentUMAP(n_neighbors=10, n_epochs=2, random_state=1).fit(x)
    got = um.transform(q)
    xd, qd = torch.from_numpy(x).cuda(), torch.from_numpy(q).cuda()
    idx, dist = lu.knn_query(qd, xd, 10)
    init = lu.init_transform(lu.query_graph(idx, dist, 1.0), torch.from_numpy(um.embedding_).cuda())
    np.testing.assert_array_equal(got, init.cpu().numpy())


# ------------------------------------------------------------------------------ whole transform
def test_whole_transform():
    x, lab = blobs(25000, 32, centers=10, seed=7)
    xf, lf, xq, lq = x[:20000], lab[:20000], x[20000:], lab[20000:]
    um = lu.LatentUMAP(n_neighbors=20, min_dist=0.1, random_state=42)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        assert um.fit(xf) is um
    e = um.transform(xq)
    assert e.dtype == np.float32 and e.shape == (5000, 2) and np.isfinite(e).all()
    from sklearn.neighbors import NearestNeighbors
    nb = NearestNeighbors(n_neighbors=1).fit(um.embedding_).kneighbors(e, return_distance=False)[:, 0]
    assert float((lf[nb] == lq).mean()) >= 0.98
    emb0 = um.embedding_.copy()
    np.testing.assert_array_equal(um.transform(xf), um.embedding_)   # the fitted rows: the embedding itself
    np.testing.assert_array_equal(um.transform(xq), e)               # bitwise repeat
    np.testing.assert_array_equal(um.embedding_, emb0)
    back = pickle.loads(pickle.dumps(um))
    np.testing.assert_array_equal(back.transform(xq), e)
    assert back.graph_.shape == (20000, 20000)
    if torch.cuda.device_count() > 1:
        with torch.cuda.device(1):
            np.testing.assert_array_equal(pickle.loads(pickle.dumps(um)).transform(xq), e)


# ---------------------------------------------------------------------------------- edge cases
def test_transform_edge_cases():
    x, _ = blobs(500, 16, centers=3, seed=21)
    q, _ = blobs(40, 16, centers=3, seed=22)
    with pytest.raises(RuntimeError):
        lu.LatentUMAP().transform(q)
    um = lu.LatentUMAP(random_state=3, n_epochs=60).fit(x)
    with pytest.raises(ValueError):
        um.transform(q[:, :15])
    qn = q.copy()
    qn[0, 0] = np.nan
    with pytest.raises(ValueError):
        um.transform(qn)
    with pytest.raises(ValueError):
        um.transform(torch.from_numpy(qn).cuda())
    z = um.transform(np.zeros((0, 16)))
    assert z.shape == (0, 2) and z.dtype == np.float32
    e_np = um.transform(q)
    np.testing.assert_array_equal(um.transform(torch.from_numpy(q)), e_np)
    np.testing.assert_array_equal(um.transform(torch.from_numpy(q).cuda()), e_np)
    ed = um.transform_device(q)
    assert ed.is_cuda and ed.dtype == torch.float32
    # float32 queries against a float64 fit are converted to float64
    np.testing.assert_array_equal(um.transform(q.astype(np.float32)), um.transform(q.astype(np.float32).astype(np.float64)))
    # a fit on one row maps every query there
    one = lu.LatentUMAP().fit(x[:1])
    np.testing.assert_array_equal(one.transform(q), np.repeat(one.embedding_, 40, 0))
    # N <= n_neighbors: the fit's neighbour count max(N - 1, 2)
    with pytest.warns(UserWarning):
        small = lu.LatentUMAP(n_neighbors=15, random_state=0).fit(x[:8])
    es = small.transform(q)
    assert es.shape == (40, 2) and np.isfinite(es).all()
    for dim in (1, 8):
        m = lu.LatentUMAP(n_components=dim, random_state=4, n_epochs=60).fit(torch.from_numpy(x).float().cuda())
        e = m.transform(q)
        assert e.shape == (40, dim) and np.isfinite(e).all()
