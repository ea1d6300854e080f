"""CPU restatement of LatentUMAP.transform (csrc/umap.cu, data/latent_umap.py), stage by stage: umap-learn
0.5's UMAP.transform for metric='euclidean' (function names cited), with the project's documented deviations
(exact kNN, the splitmix64 hash for random draws, a negative sample never skipped).  It builds on the fit's
restatement in oracle/umap_oracle.py (smooth_knn_dist, the hash).  Test infrastructure only."""
import numpy as np

from oracle.umap_oracle import smooth_knn_dist, umap_hash

TRANSFORM_STREAM = 5 << 32


def knn_query(q, x, k, block=256):
    """Exact kNN of the rows of q among the rows of x in float64, difference form, ordered by
    (distance, index): no row is preferred (umap-learn's transform)."""
    q = np.asarray(q, dtype=np.float64)
    x = np.asarray(x, dtype=np.float64)
    Nq, N = q.shape[0], x.shape[0]
    idx = np.empty((Nq, k), dtype=np.int64)
    dist = np.empty((Nq, k))
    for b0 in range(0, Nq, block):
        d2 = ((q[b0:b0 + block, None, :] - x[None, :, :]) ** 2).sum(-1)
        for r in range(d2.shape[0]):
            order = np.lexsort((np.arange(N), d2[r]))[:k]
            idx[b0 + r] = order
            dist[b0 + r] = np.sqrt(d2[r, order])
    return idx, dist


def membership_strengths_bipartite(knn_dist, sigmas, rhos):
    """compute_membership_strengths(bipartite=True): no entry is zeroed."""
    N, k = knn_dist.shape
    w = np.zeros((N, k))
    for i in range(N):
        for j in range(k):
            if knn_dist[i, j] - rhos[i] <= 0.0 or sigmas[i] == 0.0:
                w[i, j] = 1.0
            else:
                w[i, j] = np.exp(-((knn_dist[i, j] - rhos[i]) / sigmas[i]))
    return w


def query_graph(knn_idx, knn_dist, k, local_connectivity=1.0):
    """UMAP.transform's graph: smooth_knn_dist with local_connectivity max(0, lc - 1), bipartite
    memberships, each row sorted by column (the order of the CSR -> COO conversion).
    Returns (rho, sigma, cols [Nq, k], weights [Nq, k])."""
    sig, rho = smooth_knn_dist(knn_dist, k, local_connectivity=max(0.0, local_connectivity - 1.0))
    w = membership_strengths_bipartite(knn_dist, sig, rho)
    order = np.argsort(knn_idx, axis=1, kind="stable")
    return rho, sig, np.take_along_axis(knn_idx, order, 1), np.take_along_axis(w, order, 1)


def init_transform(cols, w, emb):
    """umap.umap_.init_graph_transform: per row in column order, a weight of exactly 1 copies that
    row's embedding; else out += (w / row_sum) * emb[col], in float64 and rounded to float32 per sum."""
    Nq, k = cols.shape
    out = np.zeros((Nq, emb.shape[1]), dtype=np.float32)
    for i in range(Nq):
        row_sum = 0.0
        for j in range(k):
            row_sum += float(w[i, j])
        for j in range(k):
            e = emb[cols[i, j]].astype(np.float64)
            if w[i, j] == 1.0:
                out[i] = emb[cols[i, j]]
                break
            out[i] = (out[i].astype(np.float64) + (w[i, j] / row_sum) * e).astype(np.float32)
    return out


def transform_schedule(cols, w, n_epochs, negative_sample_rate=5.0):
    """The transform's pruning (below max / n_epochs) and make_epochs_per_sample, row-major."""
    keep = w >= w.max() / float(n_epochs)
    head = np.repeat(np.arange(w.shape[0]), w.shape[1]).reshape(w.shape)[keep]
    tail, wk = cols[keep], w[keep]
    n_samples = n_epochs * (wk / wk.max())
    eps = -1.0 * np.ones(wk.shape[0])
    eps[n_samples > 0] = float(n_epochs) / n_samples[n_samples > 0]
    eps_neg = eps / negative_sample_rate
    return dict(head=head.astype(np.int64), tail=tail.astype(np.int64), weights=wk, eps=eps, eps_neg=eps_neg,
                next=eps.copy(), next_neg=eps_neg.copy())


def _sgd_transform_body(emb_q, emb, head, tail, eps, eps_neg, nxt, nxt_neg, n_epochs, a, b, gamma, alpha0, seed,
                        mixer):
    N, dim = emb.shape
    s0 = mixer(seed)
    for n in range(n_epochs):
        alpha = alpha0 * (1.0 - n / float(n_epochs))
        sn = mixer(s0 ^ np.uint64(n))
        for e in range(head.shape[0]):
            if not (nxt[e] <= n):
                continue
            j, k = head[e], tail[e]
            d2 = 0.0
            for d in range(dim):
                t = np.float64(emb_q[j, d]) - np.float64(emb[k, d])
                d2 = d2 + t * t
            gc = (-2.0 * a * b * d2 ** (b - 1.0)) / (a * d2 ** b + 1.0) if d2 > 0.0 else 0.0
            for d in range(dim):
                g = min(4.0, max(-4.0, gc * (np.float64(emb_q[j, d]) - np.float64(emb[k, d]))))
                emb_q[j, d] = np.float32(np.float64(emb_q[j, d]) + g * alpha)
            nxt[e] += eps[e]
            n_neg = int((n - nxt_neg[e]) / eps_neg[e])
            se = mixer(sn ^ np.uint64(e))
            for p in range(n_neg):
                kk = np.int64(mixer(se ^ np.uint64(p)) % np.uint64(N))
                s = 0.0
                for d in range(dim):
                    t = np.float64(emb_q[j, d]) - np.float64(emb[kk, d])
                    s = s + t * t
                rc = (2.0 * gamma * b) / ((0.001 + s) * (a * s ** b + 1.0)) if s > 0.0 else 0.0
                for d in range(dim):
                    if rc > 0.0:
                        g = min(4.0, max(-4.0, rc * (np.float64(emb_q[j, d]) - np.float64(emb[kk, d]))))
                    else:
                        g = 4.0
                    emb_q[j, d] = np.float32(np.float64(emb_q[j, d]) + g * alpha)
            nxt_neg[e] = nxt_neg[e] + n_neg * eps_neg[e]


_NUMBA_SGD_TRANSFORM = None


def sgd_transform(emb_q, emb, sched, n_epochs, a, b, gamma, initial_alpha, seed):
    """optimize_layout_euclidean(move_other=False), sequential in edge order, in place on the float32
    emb_q; emb is only read.  Negative p of edge e in epoch n: umap_hash(transform seed, n, e, p) mod N
    with the transform seed umap_hash(seed, 5 << 32, 0, 0), never skipped."""
    global _NUMBA_SGD_TRANSFORM
    tseed = np.uint64(umap_hash(seed, TRANSFORM_STREAM, 0, 0))
    args = (emb_q, np.asarray(emb, dtype=np.float32), sched["head"], sched["tail"], sched["eps"], sched["eps_neg"],
            sched["next"], sched["next_neg"], int(n_epochs), float(a), float(b), float(gamma), float(initial_alpha))
    try:
        import numba
        if _NUMBA_SGD_TRANSFORM is None:
            nmix = numba.njit(cache=False)(_mix_u64)
            body = numba.njit(cache=False)(_sgd_transform_body)
            _NUMBA_SGD_TRANSFORM = lambda *a_: body(*a_, nmix)
        _NUMBA_SGD_TRANSFORM(*args, tseed)
    except ImportError:
        with np.errstate(over="ignore"):
            _sgd_transform_body(*args, tseed, _mix_u64)
    return emb_q


def _mix_u64(z):
    z = z + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))
