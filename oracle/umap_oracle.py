"""CPU restatement of LatentUMAP (csrc/umap.cu, data/latent_umap.py), stage by stage, in float64
(the layout in float32 with float64 coefficients, as the kernel computes it).  umap-learn is not
installed, so this file is the pin: every formula below is the one umap-learn 0.5 uses for
metric='euclidean' (function names cited), with the project's documented deviations (exact kNN, the
splitmix64 hash for random draws, the PCA meta-layout of many components).  Test infrastructure only.
"""
import math

import numpy as np
import scipy.sparse
import scipy.sparse.csgraph
import scipy.sparse.linalg

M64 = (1 << 64) - 1
SMOOTH_K_TOLERANCE = 1e-5
MIN_K_DIST_SCALE = 1e-3


# ------------------------------------------------------------------------------- the hash
def mix(z):
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def umap_hash(seed, a, b, c):
    return mix(mix(mix(mix(seed & M64) ^ a) ^ b) ^ c)


def unit(h):
    return ((h >> 11) + 0.5) * (1.0 / 9007199254740992.0)


def random_block(seed, stream_id, shape, kind, scale):
    n = int(np.prod(shape))
    out = np.empty(n)
    for i in range(n):
        u1 = unit(umap_hash(seed, stream_id, i, 0))
        if kind == 0:
            out[i] = scale * (2.0 * u1 - 1.0)
        else:
            u2 = unit(umap_hash(seed, stream_id, i, 1))
            out[i] = scale * math.sqrt(-2.0 * math.log(u1)) * math.cos(6.283185307179586 * u2)
    return out.reshape(shape)


# ------------------------------------------------------------------------------- stage 1
def knn(x, k, block=256):
    """Exact kNN in float64, difference form, ordered by (distance, not-self, index)."""
    x = np.asarray(x, dtype=np.float64)
    N = x.shape[0]
    idx = np.empty((N, k), dtype=np.int64)
    dist = np.empty((N, k))
    for b0 in range(0, N, block):
        q = x[b0:b0 + block]
        d2 = ((q[:, None, :] - x[None, :, :]) ** 2).sum(-1)
        for r in range(q.shape[0]):
            i = b0 + r
            notself = np.ones(N, dtype=np.int64)
            notself[i] = 0
            order = np.lexsort((np.arange(N), notself, d2[r]))[:k]
            idx[i] = order
            dist[i] = np.sqrt(d2[r, order])
    return idx, dist


# ------------------------------------------------------------------------------- stage 2
def smooth_knn_dist(distances, k, n_iter=64, local_connectivity=1.0):
    """umap.umap_.smooth_knn_dist (bandwidth 1), in float64."""
    target = np.log2(k)
    N = distances.shape[0]
    rho = np.zeros(N)
    result = np.zeros(N)
    mean_distances = np.mean(distances)
    for i in range(N):
        lo, hi, mid = 0.0, np.inf, 1.0
        ith = distances[i]
        non_zero = ith[ith > 0.0]
        if non_zero.shape[0] >= local_connectivity:
            index = int(np.floor(local_connectivity))
            interpolation = local_connectivity - index
            if index > 0:
                rho[i] = non_zero[index - 1]
                if interpolation > SMOOTH_K_TOLERANCE:
                    rho[i] += interpolation * (non_zero[index] - non_zero[index - 1])
            else:
                rho[i] = interpolation * non_zero[0]
        elif non_zero.shape[0] > 0:
            rho[i] = np.max(non_zero)
        for _ in range(n_iter):
            psum = 0.0
            for j in range(1, distances.shape[1]):
                d = distances[i, j] - rho[i]
                psum += np.exp(-(d / mid)) if d > 0 else 1.0
            if np.fabs(psum - target) < SMOOTH_K_TOLERANCE:
                break
            if psum > target:
                hi = mid
                mid = (lo + hi) / 2.0
            else:
                lo = mid
                mid = mid * 2 if hi == np.inf else (lo + hi) / 2.0
        result[i] = mid
        if rho[i] > 0.0:
            if result[i] < MIN_K_DIST_SCALE * np.mean(ith):
                result[i] = MIN_K_DIST_SCALE * np.mean(ith)
        elif result[i] < MIN_K_DIST_SCALE * mean_distances:
            result[i] = MIN_K_DIST_SCALE * mean_distances
    return result, rho


def membership_strengths(knn_idx, knn_dist, sigmas, rhos):
    """umap.umap_.compute_membership_strengths: weights [N, k]."""
    N, k = knn_idx.shape
    w = np.zeros((N, k))
    for i in range(N):
        for j in range(k):
            if knn_idx[i, j] == i:
                w[i, j] = 0.0
            elif knn_dist[i, j] - rhos[i] <= 0.0 or sigmas[i] == 0.0:
                w[i, j] = 1.0
            else:
                w[i, j] = np.exp(-((knn_dist[i, j] - rhos[i]) / sigmas[i]))
    return w


# ------------------------------------------------------------------------------- stage 3
def fuzzy_union(knn_idx, w):
    """P = A + A^T - A.*A^T over the union of every row's neighbours and reverse neighbours (self
    excluded), as a sorted CSR."""
    N, k = knn_idx.shape
    a = {}
    for i in range(N):
        for j in range(k):
            c = int(knn_idx[i, j])
            if c != i:
                a[(i, c)] = w[i, j]
    entries = {}
    for (i, c) in a:
        for (r, s) in ((i, c), (c, i)):
            if (r, s) not in entries:
                x, y = a.get((r, s), 0.0), a.get((s, r), 0.0)
                entries[(r, s)] = x + y - x * y
    keys = sorted(entries)
    rows = np.array([r for r, _ in keys], dtype=np.int64)
    cols = np.array([c for _, c in keys], dtype=np.int64)
    vals = np.array([entries[key] for key in keys])
    return scipy.sparse.csr_matrix((vals, (rows, cols)), shape=(N, N))


def prune_and_schedule(P, n_epochs, negative_sample_rate=5.0):
    """simplicial_set_embedding's pruning, make_epochs_per_sample and optimize_layout_euclidean's set-up,
    in row-major edge order."""
    coo = P.tocoo()
    keep = coo.data >= coo.data.max() / float(n_epochs)
    head, tail, w = coo.row[keep], coo.col[keep], coo.data[keep]
    n_samples = n_epochs * (w / w.max())
    eps = -1.0 * np.ones(w.shape[0])
    eps[n_samples > 0] = float(n_epochs) / n_samples[n_samples > 0]
    eps_neg = eps / negative_sample_rate
    return dict(head=head.astype(np.int64), tail=tail.astype(np.int64), weights=w, eps=eps, eps_neg=eps_neg,
                next=eps.copy(), next_neg=eps_neg.copy())


# ------------------------------------------------------------------------------- stage 4
def laplacian_vectors(Pc, dim):
    """The dim eigenvectors of I - D^-1/2 P D^-1/2 after the trivial one (scipy eigsh on the shifted
    operator 2I - L, whose largest eigenvalues are L's smallest), signs as in the kernel."""
    deg = np.asarray(Pc.sum(axis=1)).ravel()
    Dm = scipy.sparse.diags(1.0 / np.sqrt(deg))
    n = Pc.shape[0]
    M = Dm @ Pc @ Dm
    if n <= 2000:
        ev, V = np.linalg.eigh(np.eye(n) - M.toarray())
    else:
        ev, V = scipy.sparse.linalg.eigsh(scipy.sparse.identity(n) + M, dim + 1, which='LA', tol=1e-12)
        ev = 2.0 - ev
    order = np.argsort(ev)[1:dim + 1]
    V = V[:, order]
    for c in range(dim):
        if V[np.argmax(np.abs(V[:, c])), c] < 0:
            V[:, c] = -V[:, c]
    return ev[order], V


def meta_positions(x, labels, nc, dim):
    if nc <= 2 * dim:
        k = int(math.ceil(nc / 2.0))
        base = np.hstack([np.eye(k), np.zeros((k, dim - k))])
        return np.vstack([base, -base])[:nc]
    from oracle.pca_oracle import pca_fit_transform
    cent = np.stack([x[labels == c].mean(0) for c in range(nc)])
    K = min(dim, x.shape[1])
    meta = np.zeros((nc, dim))
    meta[:, :K] = pca_fit_transform(cent, K)[0]
    dd = np.sqrt(((meta[:, None] - meta[None]) ** 2).sum(-1))
    dmin = dd[~np.eye(nc, dtype=bool)].min()
    return meta / dmin if dmin > 0 else meta


def spectral_layout(x, P, dim):
    """Before expansion: (layout [N, dim], component labels, meta positions, half distances).
    Components too small for a spectral layout are returned as NaN rows (the kernel fills them from
    the hash generator)."""
    nc, labels = scipy.sparse.csgraph.connected_components(P, directed=False)
    N = P.shape[0]
    out = np.full((N, dim), np.nan)
    if nc == 1:
        meta, half = np.zeros((1, dim)), None
    else:
        meta = meta_positions(np.asarray(x, dtype=np.float64), labels, nc, dim)
        dd = np.sqrt(((meta[:, None] - meta[None]) ** 2).sum(-1))
        dd[np.eye(nc, dtype=bool)] = np.inf
        half = dd.min(1) / 2.0
    for c in range(nc):
        sel = np.flatnonzero(labels == c)
        if sel.size < 2 * dim + 2:
            continue
        _, V = laplacian_vectors(P[sel][:, sel], dim)
        if half is not None:
            V = V * (half[c] / np.abs(V).max())
        out[sel] = V + meta[c]
    return out, labels, meta, half


def init_embedding(init64, noise=None):
    """(float)(init * expansion) + (float)noise, then 10 (v - min) / (max - min) per axis, float32."""
    if noise is not None:
        expansion = 10.0 / np.abs(init64).max()
        v = (init64 * expansion).astype(np.float32) + noise.astype(np.float32)
    else:
        v = init64.astype(np.float32)
    mn, mx = v.min(0), v.max(0)
    rng = (mx - mn).astype(np.float32)
    return np.where(rng > 0, (np.float32(10.0) * (v - mn)) / np.where(rng > 0, rng, 1), 0).astype(np.float32)


# ------------------------------------------------------------------------------- stage 5
def _sgd_py(emb, head, tail, eps, eps_neg, nxt, nxt_neg, n_epochs, a, b, gamma, lr, seed, epochs):
    N, dim = emb.shape
    for n in epochs:
        alpha = lr * (1.0 - n / float(n_epochs))
        for e in range(head.shape[0]):
            if not (nxt[e] <= n):
                continue
            j, k = head[e], tail[e]
            d2 = 0.0
            for d in range(dim):
                t = float(emb[j, d]) - float(emb[k, d])
                d2 = d2 + t * t
            gc = (-2.0 * a * b * d2 ** (b - 1.0)) / (a * d2 ** b + 1.0) if d2 > 0.0 else 0.0
            for d in range(dim):
                g = min(4.0, max(-4.0, gc * (float(emb[j, d]) - float(emb[k, d]))))
                cj = np.float32(float(emb[j, d]) + g * alpha)
                ck = np.float32(float(emb[k, d]) + (-g) * alpha)
                emb[j, d] = cj
                emb[k, d] = ck
            nxt[e] += eps[e]
            n_neg = int((n - nxt_neg[e]) / eps_neg[e])
            for p in range(n_neg):
                kk = umap_hash(seed, n, e, p) % N
                if kk == j:
                    continue
                s = 0.0
                for d in range(dim):
                    t = float(emb[j, d]) - float(emb[kk, d])
                    s = s + t * t
                rc = (2.0 * gamma * b) / ((0.001 + s) * (a * s ** b + 1.0)) if s > 0.0 else 0.0
                for d in range(dim):
                    g = min(4.0, max(-4.0, rc * (float(emb[j, d]) - float(emb[kk, d])))) if rc > 0.0 else 4.0
                    emb[j, d] = np.float32(float(emb[j, d]) + g * alpha)
            nxt_neg[e] = nxt_neg[e] + n_neg * eps_neg[e]


def _make_numba_sgd():
    import numba

    @numba.njit(cache=False)
    def nmix(z):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))

    @numba.njit(cache=False)
    def run(emb, head, tail, eps, eps_neg, nxt, nxt_neg, n_epochs, a, b, gamma, lr, seed, e_lo, e_hi):
        N, dim = emb.shape
        s0 = nmix(seed)
        for n in range(e_lo, e_hi):
            alpha = lr * (1.0 - n / float(n_epochs))
            sn = nmix(s0 ^ np.uint64(n))
            for e in range(head.shape[0]):
                if not (nxt[e] <= n):
                    continue
                j, k = head[e], tail[e]
                d2 = 0.0
                for d in range(dim):
                    t = np.float64(emb[j, d]) - np.float64(emb[k, d])
                    d2 = d2 + t * t
                gc = (-2.0 * a * b * d2 ** (b - 1.0)) / (a * d2 ** b + 1.0) if d2 > 0.0 else 0.0
                for d in range(dim):
                    g = min(4.0, max(-4.0, gc * (np.float64(emb[j, d]) - np.float64(emb[k, d]))))
                    cj = np.float32(np.float64(emb[j, d]) + g * alpha)
                    ck = np.float32(np.float64(emb[k, d]) + (-g) * alpha)
                    emb[j, d] = cj
                    emb[k, d] = ck
                nxt[e] += eps[e]
                n_neg = int((n - nxt_neg[e]) / eps_neg[e])
                se = nmix(sn ^ np.uint64(e))
                for p in range(n_neg):
                    kk = np.int64(nmix(se ^ np.uint64(p)) % np.uint64(N))
                    if kk == j:
                        continue
                    s = 0.0
                    for d in range(dim):
                        t = np.float64(emb[j, d]) - np.float64(emb[kk, d])
                        s = s + t * t
                    rc = (2.0 * gamma * b) / ((0.001 + s) * (a * s ** b + 1.0)) if s > 0.0 else 0.0
                    for d in range(dim):
                        if rc > 0.0:
                            g = min(4.0, max(-4.0, rc * (np.float64(emb[j, d]) - np.float64(emb[kk, d]))))
                        else:
                            g = 4.0
                        emb[j, d] = np.float32(np.float64(emb[j, d]) + g * alpha)
                nxt_neg[e] = nxt_neg[e] + n_neg * eps_neg[e]
    return run


_NUMBA_SGD = None


def sgd(emb, sched, n_epochs, a, b, gamma, lr, seed, epochs=None):
    """Sequential edge-order SGD over `epochs` (default: all), in place on the float32 emb."""
    global _NUMBA_SGD
    epochs = range(n_epochs) if epochs is None else epochs
    args = (emb, sched["head"], sched["tail"], sched["eps"], sched["eps_neg"], sched["next"], sched["next_neg"])
    try:
        if _NUMBA_SGD is None:
            _NUMBA_SGD = _make_numba_sgd()
        _NUMBA_SGD(*args, n_epochs, float(a), float(b), float(gamma), float(lr), np.uint64(seed & M64),
                   epochs.start, epochs.stop)
    except ImportError:
        _sgd_py(*args, n_epochs, a, b, gamma, lr, seed, epochs)
    return emb


def fit(x, k, dim=2, min_dist=0.1, spread=1.0, n_epochs=None, seed=0, knn_lists=None):
    """The whole restatement (spectral init; small components and the noise from the hash)."""
    import importlib
    lu = importlib.import_module("autoencoded-vocal-analysis_b200.data.latent_umap")
    N = x.shape[0]
    n_epochs = n_epochs or lu.default_n_epochs(N)
    idx, dist = knn_lists if knn_lists is not None else knn(x, k)
    sig, rho = smooth_knn_dist(dist, k)
    P = fuzzy_union(idx, membership_strengths(idx, dist, sig, rho))
    sched = prune_and_schedule(P, n_epochs)
    lay, labels, meta, half = spectral_layout(x, P, dim)
    for c in np.unique(labels[np.isnan(lay[:, 0])]):
        sel = np.flatnonzero(labels == c)
        scale = 10.0 if half is None else half[c]
        lay[sel] = random_block(seed, (4 << 32) | int(c), (sel.size, dim), 0, scale) + meta[c]
    emb = init_embedding(lay, random_block(seed, 2 << 32, (N, dim), 1, 1e-4))
    a, b = lu.find_ab_params(spread, min_dist)
    return sgd(emb, sched, n_epochs, a, b, 1.0, 1.0, seed)
