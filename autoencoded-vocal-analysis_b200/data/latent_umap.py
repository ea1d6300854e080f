"""
LatentUMAP: umap-learn 0.5's ``UMAP(metric='euclidean').fit_transform`` on the device (csrc/umap.cu).

AVA's standard analysis ends in a UMAP of the latent means: the reference's
``DataContainer._make_latent_mean_umap_projection`` (ava/data/data_container.py) calls
``umap.UMAP(n_components=2, n_neighbors=20, min_dist=0.1, metric='euclidean', random_state=42)``.
``LatentUMAP(n_neighbors=20, min_dist=0.1, random_state=42)`` is that projection; the constructor's
defaults are umap-learn's own.

The stages follow umap-learn's algorithm; each is a native kernel, with torch only as plumbing (the
sort that de-duplicates the graph's edge keys, prefix sums, compactions):

1. exact k nearest neighbours by brute force (umap-learn uses NNDescent, an approximation, above
   4096 rows), fp32 selection then fp64 distances, the row itself first;
2. ``smooth_knn_dist`` and ``compute_membership_strengths`` in fp64;
3. the fuzzy union P = A + A^T - A.*A^T as a device CSR, pruned below max(P)/n_epochs for the layout,
   and the ``make_epochs_per_sample`` schedule;
4. the spectral initialisation: connected components, the eigenvectors of the normalised Laplacian
   of each component by LOBPCG (umap-learn: ARPACK ``eigsh``), umap-learn's ``multi_component_layout``
   placement, then the expansion, noise and per-axis rescale of ``simplicial_set_embedding``;
5. the negative-sampling SGD, one launch per epoch with Hogwild updates, like umap-learn's parallel
   mode.

Deviations from umap-learn, all documented in DESIGN.md: exact neighbours; a counter-based hash
(splitmix64 of (seed, epoch, edge, sample)) instead of umap-learn's Tausworthe generator, so the
negative samples can be replayed; with more than 2 * n_components components, the components' meta
positions are the PCA projection of their data-space centroids (umap-learn runs a spectral layout of
the centroids), scaled to unit minimum spacing.  Stages 1-4 are bitwise reproducible from call to
call; the layout is not (Hogwild), as umap-learn's parallel layout is not.

``fit`` keeps the fitted rows and embedding on the device, and ``transform`` places new rows into that
embedding without moving it (umap-learn's ``UMAP.transform``): exact neighbours of each new row among the
fitted rows, the bipartite memberships (local_connectivity - 1), umap-learn's ``init_graph_transform``, and
an SGD in which only the new rows move, one launch for all epochs with a thread per new row.  It has no
races, so a transform repeats bit for bit and equals the sequential algorithm.

``DataContainer`` does not request ``latent_mean_umap`` through this class yet: the field still raises
NotImplementedError there.  Wiring it is a few lines in ``DataContainer._make_field``.

There is no CPU fallback: without CUDA this raises ``_lib.AvaB200Error``.
"""
import math
import warnings

import numpy as np
import torch

from .. import _lib

MAX_D = 64            # the latent widths LatentPCA takes
MAX_NEIGHBORS = 100   # top-k lists live in registers
MAX_COMPONENTS = 8

# streams of the counter-based generator (ava_b200_umap_random): tag << 32 | index; tag 5 is the
# transform's negative sampling (ava_b200_umap_sgd_transform derives its seed from it)
_S_RANDOM_INIT, _S_NOISE, _S_LOBPCG, _S_FILL = 1, 2, 3, 4

_LOBPCG_TOL = 1e-4      # residual norm of a unit eigenvector, relative to the largest wanted eigenvalue
_LOBPCG_MAXITER = 400


def find_ab_params(spread, min_dist):
    """umap.umap_.find_ab_params: fit 1 / (1 + a x^(2b)) to the target membership curve."""
    from scipy.optimize import curve_fit

    def curve(x, a, b):
        return 1.0 / (1.0 + a * x ** (2 * b))

    xv = np.linspace(0, spread * 3, 300)
    yv = np.zeros(xv.shape)
    yv[xv < min_dist] = 1.0
    yv[xv >= min_dist] = np.exp(-(xv[xv >= min_dist] - min_dist) / spread)
    params, _ = curve_fit(curve, xv, yv)
    return float(params[0]), float(params[1])


def default_n_epochs(n):
    """umap-learn's default: 500 epochs up to 10 000 rows, 200 above."""
    return 500 if n <= 10000 else 200


def transform_n_epochs(n_epochs, n_queries):
    """umap-learn's transform epochs: 100 up to 10 000 queries, 30 above, or n_epochs // 3."""
    if n_epochs is None:
        return 100 if n_queries <= 10000 else 30
    return int(n_epochs) // 3


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


# ------------------------------------------------------------------------------ stages 1-3
def knn(x, k):
    """Exact k nearest neighbours of the rows of x [N, D] (float32 or float64, on the device):
    (indices [N, k] int32, Euclidean distances [N, k] float64), the row itself first."""
    N, D = x.shape
    dev = x.device
    ws_bytes = int(_lib.lib().ava_b200_umap_knn_ws_bytes(N, D, k))
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
    idx = torch.empty(N, k, dtype=torch.int32, device=dev)
    dist = torch.empty(N, k, dtype=torch.float64, device=dev)
    _lib.call("ava_b200_umap_knn", x.data_ptr(), 1 if x.dtype == torch.float32 else 0, N, D, k, idx.data_ptr(),
              dist.data_ptr(), ws.data_ptr(), ws_bytes, _stream(dev))
    return idx, dist


def knn_query(q, x, k):
    """Exact k nearest rows of x [N, D] for each row of q [Nq, D] (both float32 or both float64, on the
    device): (indices [Nq, k] int32, Euclidean distances [Nq, k] float64), ranked by (distance, index)."""
    Nq, D = q.shape
    N = x.shape[0]
    dev = x.device
    ws_bytes = int(_lib.lib().ava_b200_umap_knn_query_ws_bytes(Nq, N, D, k))
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
    idx = torch.empty(Nq, k, dtype=torch.int32, device=dev)
    dist = torch.empty(Nq, k, dtype=torch.float64, device=dev)
    _lib.call("ava_b200_umap_knn_query", q.data_ptr() if Nq else None, Nq, x.data_ptr(), N,
              1 if x.dtype == torch.float32 else 0, D, k, idx.data_ptr() if Nq else None,
              dist.data_ptr() if Nq else None, ws.data_ptr(), ws_bytes, _stream(dev))
    return idx, dist


def query_graph(knn_idx, knn_dist, local_connectivity=1.0):
    """The bipartite graph of umap-learn's transform (queries x fitted rows, k entries per row):
    rho, sigma, and cols / weights [Nq, k] with each row sorted by column.  local_connectivity is the
    fitted model's (the kernel uses max(0, local_connectivity - 1))."""
    Nq, k = knn_idx.shape
    dev = knn_idx.device
    rho = torch.empty(Nq, dtype=torch.float64, device=dev)
    sigma = torch.empty(Nq, dtype=torch.float64, device=dev)
    w = torch.empty(Nq, k, dtype=torch.float64, device=dev)
    scratch = torch.empty(1, dtype=torch.float64, device=dev)
    _lib.call("ava_b200_umap_smooth_knn_query", knn_idx.data_ptr(), knn_dist.data_ptr(), Nq, k,
              float(local_connectivity), rho.data_ptr(), sigma.data_ptr(), w.data_ptr(), scratch.data_ptr(),
              _stream(dev))
    cols, order = torch.sort(knn_idx, dim=1)   # the columns of a row are distinct
    return dict(rho=rho, sigma=sigma, cols=cols.contiguous(), weights=torch.gather(w, 1, order).contiguous())


def init_transform(graph, emb):
    """umap-learn's init_graph_transform from the unpruned graph: float32 [Nq, dim] on the device."""
    Nq, k = graph["cols"].shape
    N, dim = emb.shape
    out = torch.empty(Nq, dim, dtype=torch.float32, device=emb.device)
    _lib.call("ava_b200_umap_init_transform", graph["cols"].data_ptr(), graph["weights"].data_ptr(), Nq, k,
              emb.data_ptr(), N, dim, out.data_ptr(), _stream(emb.device))
    return out


def transform_schedule(graph, n_epochs, negative_sample_rate=5.0):
    """The transform's pruned edges (weights below max / n_epochs dropped) as row pointers and tails in
    row-major, column-sorted order, with their SGD schedule."""
    w = graph["weights"]
    dev = w.device
    Nq = w.shape[0]
    vmax = w.max()
    keep = w >= vmax / float(n_epochs)
    rowptr = torch.zeros(Nq + 1, dtype=torch.int64, device=dev)
    rowptr[1:] = torch.cumsum(keep.sum(1), 0)
    vals = w[keep].contiguous()
    out = dict(rowptr=rowptr, tail=graph["cols"][keep].contiguous(), weights=vals)
    n = vals.numel()
    for name in ("eps", "eps_neg", "next", "next_neg"):
        out[name] = torch.empty(n, dtype=torch.float64, device=dev)
    vmax_t = vmax.reshape(1).contiguous()
    _lib.call("ava_b200_umap_epochs_per_sample", vals.data_ptr(), n, vmax_t.data_ptr(), int(n_epochs),
              float(negative_sample_rate), out["eps"].data_ptr(), out["eps_neg"].data_ptr(), out["next"].data_ptr(),
              out["next_neg"].data_ptr(), _stream(dev))
    return out


def sgd_transform(emb_q, emb, sched, n_epochs, a, b, gamma, initial_alpha, seed):
    """All n_epochs of the transform's layout in one launch, in place on emb_q; emb (the fitted
    embedding) is only read."""
    Nq, dim = emb_q.shape
    _lib.call("ava_b200_umap_sgd_transform", emb_q.data_ptr(), Nq, emb.data_ptr(), emb.shape[0], dim,
              sched["rowptr"].data_ptr(), sched["tail"].data_ptr(), sched["eps"].data_ptr(),
              sched["eps_neg"].data_ptr(), sched["next"].data_ptr(), sched["next_neg"].data_ptr(), int(n_epochs),
              float(a), float(b), float(gamma), float(initial_alpha), seed & (2 ** 64 - 1), _stream(emb_q.device))
    return emb_q


def fuzzy_graph(knn_idx, knn_dist, local_connectivity=1.0):
    """rho, sigma, the membership weights and the CSR of P = A + A^T - A.*A^T (unpruned)."""
    N, k = knn_idx.shape
    dev = knn_idx.device
    st = _stream(dev)
    rho = torch.empty(N, dtype=torch.float64, device=dev)
    sigma = torch.empty(N, dtype=torch.float64, device=dev)
    w = torch.empty(N, k, dtype=torch.float64, device=dev)
    scratch = torch.empty(1, dtype=torch.float64, device=dev)
    _lib.call("ava_b200_umap_smooth_knn", knn_idx.data_ptr(), knn_dist.data_ptr(), N, k, float(local_connectivity),
              rho.data_ptr(), sigma.data_ptr(), w.data_ptr(), scratch.data_ptr(), st)
    keys = torch.empty(2 * N * k, dtype=torch.int64, device=dev)
    _lib.call("ava_b200_umap_edge_keys", knn_idx.data_ptr(), N, k, keys.data_ptr(), st)
    keys = torch.unique(keys, sorted=True)
    keys = keys[keys >= 0].contiguous()
    nnz = keys.numel()
    rows = torch.empty(nnz, dtype=torch.int32, device=dev)
    cols = torch.empty(nnz, dtype=torch.int32, device=dev)
    vals = torch.empty(nnz, dtype=torch.float64, device=dev)
    rowptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
    _lib.call("ava_b200_umap_graph", keys.data_ptr(), nnz, N, knn_idx.data_ptr(), w.data_ptr(), k, rows.data_ptr(),
              cols.data_ptr(), vals.data_ptr(), rowptr.data_ptr(), st)
    return dict(rho=rho, sigma=sigma, weights=w, rows=rows, cols=cols, vals=vals, rowptr=rowptr, n=N)


def edge_schedule(graph, n_epochs, negative_sample_rate=5.0):
    """The pruned edge list (row-major) and its SGD schedule, as simplicial_set_embedding and
    optimize_layout_euclidean set them up."""
    vals = graph["vals"]
    dev = vals.device
    vmax = vals.max()
    keep = vals >= vmax / float(n_epochs)
    head = graph["rows"][keep].contiguous()
    tail = graph["cols"][keep].contiguous()
    w = vals[keep].contiguous()
    n = w.numel()
    out = dict(head=head, tail=tail, weights=w)
    for name in ("eps", "eps_neg", "next", "next_neg"):
        out[name] = torch.empty(n, dtype=torch.float64, device=dev)
    vmax_t = vmax.reshape(1).contiguous()
    _lib.call("ava_b200_umap_epochs_per_sample", w.data_ptr(), n, vmax_t.data_ptr(), int(n_epochs),
              float(negative_sample_rate), out["eps"].data_ptr(), out["eps_neg"].data_ptr(), out["next"].data_ptr(),
              out["next_neg"].data_ptr(), _stream(dev))
    return out


# ------------------------------------------------------------------------------ stage 4
def connected_components(graph):
    """labels [N] int32: the smallest vertex of each vertex's component."""
    N = graph["n"]
    dev = graph["vals"].device
    labels = torch.arange(N, dtype=torch.int32, device=dev)
    changed = torch.zeros(1, dtype=torch.int32, device=dev)
    while True:
        changed.zero_()
        _lib.call("ava_b200_umap_components_step", graph["rowptr"].data_ptr(), graph["cols"].data_ptr(), N,
                  labels.data_ptr(), changed.data_ptr(), _stream(dev))
        if int(changed.item()) == 0:
            return labels


def random_block(seed, stream_id, shape, kind, scale, dev):
    """Draws of the counter-based generator: kind 0 uniform(-scale, scale), 1 normal(0, scale)."""
    out = torch.empty(shape, dtype=torch.float64, device=dev)
    _lib.call("ava_b200_umap_random", seed & (2 ** 64 - 1), stream_id, out.numel(), kind, float(scale),
              out.data_ptr(), _stream(dev))
    return out


class _Operator:
    """The normalised Laplacian of one component and the dense block kernels LOBPCG needs."""

    def __init__(self, graph, dis, verts, pos):
        self.g, self.dis, self.verts, self.pos = graph, dis, verts, pos
        self.n = verts.numel()
        self.dev = dis.device

    def lap(self, X):
        Y = torch.empty_like(X)
        _lib.call("ava_b200_umap_spmm", self.g["rowptr"].data_ptr(), self.g["cols"].data_ptr(),
                  self.g["vals"].data_ptr(), self.verts.data_ptr(), self.n, self.pos.data_ptr(), self.dis.data_ptr(),
                  X.data_ptr(), X.shape[1], Y.data_ptr(), _stream(self.dev))
        return Y

    def gram(self, A, B):
        p, q = A.shape[1], B.shape[1]
        ws_bytes = int(_lib.lib().ava_b200_umap_gram_ws_bytes(p, q))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.dev)
        out = torch.empty(p, q, dtype=torch.float64, device=self.dev)
        _lib.call("ava_b200_umap_gram", A.data_ptr(), p, B.data_ptr(), q, self.n, out.data_ptr(), ws.data_ptr(),
                  ws_bytes, _stream(self.dev))
        return out.cpu().numpy()

    def combine(self, A, C):
        C = torch.from_numpy(np.ascontiguousarray(C, dtype=np.float64)).to(self.dev)
        Y = torch.empty(self.n, C.shape[1], dtype=torch.float64, device=self.dev)
        _lib.call("ava_b200_umap_combine", A.data_ptr(), A.shape[1], C.data_ptr(), C.shape[1], self.n, Y.data_ptr(),
                  _stream(self.dev))
        return Y


def _rayleigh_ritz(op, S, AS):
    """Ritz values (ascending) and coefficients of the basis S in float64 on the host; directions the
    basis does not span (Gram eigenvalues below 1e-12 of the largest) are dropped."""
    G = op.gram(S, S)
    H = op.gram(S, AS)
    G = (G + G.T) / 2
    H = (H + H.T) / 2
    d = np.sqrt(np.maximum(np.diag(G), 1e-300))
    G = G / np.outer(d, d)
    H = H / np.outer(d, d)
    eg, vg = np.linalg.eigh(G)
    keep = eg > 1e-12 * eg.max()
    T = vg[:, keep] / np.sqrt(eg[keep])
    th, W = np.linalg.eigh(T.T @ H @ T)
    return th, (T @ W) / d[:, None]


def lobpcg_smallest(op, dim, seed, stream_id, tol=_LOBPCG_TOL, maxiter=_LOBPCG_MAXITER):
    """The dim eigenvectors of the component's normalised Laplacian after the trivial one (which is
    deflated: D^1/2 1 is known exactly), by LOBPCG with block size dim + 3, until every wanted residual
    norm is at most tol times the largest wanted eigenvalue (the eigenvalues of a kNN graph's Laplacian
    start near 1e-3, so an absolute bound would say little about the vectors).  Returns (vectors
    [n, dim] float64 on the device, converged); each vector's largest-magnitude entry is positive."""
    n = op.n
    bs = min(dim + 3, n - 1)
    v0 = (1.0 / op.dis[op.verts.long()]).reshape(n, 1)
    v0 = op.combine(v0, np.array([[1.0 / math.sqrt(op.gram(v0, v0)[0, 0])]]))

    def deflate(X):
        c = op.gram(v0, X)
        return op.combine(torch.cat([X, v0], 1).contiguous(), np.vstack([np.eye(X.shape[1]), -c]))

    X = deflate(random_block(seed, stream_id, (n, bs), 1, 1.0, op.dev))
    AX = op.lap(X)
    th, C = _rayleigh_ritz(op, X, AX)
    C = C[:, :bs]
    th = th[:bs]
    X, AX = op.combine(X, C), op.combine(AX, C)
    P = AP = None
    converged = False
    for _ in range(maxiter):
        m = X.shape[1]
        R = deflate(op.combine(torch.cat([AX, X], 1).contiguous(), np.vstack([np.eye(m), -np.diag(th)])))
        rn = np.sqrt(np.maximum(np.diag(op.gram(R, R)), 0.0))
        if rn[:dim].max() <= max(tol * abs(th[dim - 1]), 1e-12):
            converged = True
            break
        AR = op.lap(R)
        S = [X, R] + ([P] if P is not None else [])
        AS = [AX, AR] + ([AP] if AP is not None else [])
        S = torch.cat(S, 1).contiguous()
        AS = torch.cat(AS, 1).contiguous()
        th_all, C = _rayleigh_ritz(op, S, AS)
        m = min(bs, C.shape[1])
        C = C[:, :m]
        th = th_all[:m]
        Cp = C.copy()
        Cp[:X.shape[1]] = 0.0
        X, AX = op.combine(S, C), op.combine(AS, C)
        P, AP = op.combine(S, Cp), op.combine(AS, Cp)
        if X.shape[1] < dim:
            break
    if X.shape[1] < dim:
        return None, False
    V = X[:, :dim]
    # sign convention: the largest-magnitude entry of every vector positive
    imax = V.abs().argmax(0)
    sign = torch.sign(V[imax, torch.arange(dim, device=op.dev)])
    sign[sign == 0] = 1.0
    return op.combine(V.contiguous(), np.diag(sign.cpu().numpy())), converged


def meta_positions(x, labels_sorted, starts, counts, dim):
    """Positions of the components (umap.spectral.component_layout): +-unit axes for up to 2*dim
    components; above that the PCA projection of the components' data-space centroids scaled to unit
    minimum spacing (umap-learn embeds the centroids spectrally)."""
    nc = len(counts)
    if nc <= 2 * dim:
        k = int(math.ceil(nc / 2.0))
        base = np.hstack([np.eye(k), np.zeros((k, dim - k))])
        return np.vstack([base, -base])[:nc]
    from .data_container import LatentPCA
    xs = x.to(torch.float64)[labels_sorted]
    cs = torch.cat([torch.zeros(1, x.shape[1], dtype=torch.float64, device=x.device), torch.cumsum(xs, 0)])
    st = torch.as_tensor(starts, device=x.device)
    en = st + torch.as_tensor(counts, device=x.device)
    cent = ((cs[en] - cs[st]) / torch.as_tensor(counts, dtype=torch.float64, device=x.device)[:, None]).contiguous()
    K = min(dim, x.shape[1])
    meta = np.zeros((nc, dim))
    meta[:, :K] = LatentPCA(K).fit_transform(cent)
    dd = np.sqrt(((meta[:, None, :] - meta[None, :, :]) ** 2).sum(-1))
    dmin = dd[~np.eye(nc, dtype=bool)].min()
    return meta / dmin if dmin > 0 else meta


def spectral_layout(x, graph, dim, seed):
    """The spectral initialisation before umap-learn's expansion: [N, dim] float64 on the device, and
    the warnings raised (components laid out at random)."""
    N = graph["n"]
    dev = graph["vals"].device
    msgs = []
    dis = torch.empty(N, dtype=torch.float64, device=dev)
    _lib.call("ava_b200_umap_degree", graph["rowptr"].data_ptr(), graph["vals"].data_ptr(), N, dis.data_ptr(),
              _stream(dev))
    labels = connected_components(graph)
    order = torch.argsort(labels, stable=True)
    comp_min, counts = torch.unique_consecutive(labels[order], return_counts=True)
    counts = counts.cpu().numpy()
    nc = len(counts)
    starts = np.concatenate([[0], np.cumsum(counts)[:-1]])
    pos = torch.empty(N, dtype=torch.int32, device=dev)
    comp_of = torch.repeat_interleave(torch.arange(nc, device=dev), torch.as_tensor(counts, device=dev))
    pos[order] = (torch.arange(N, device=dev) - torch.as_tensor(starts, device=dev)[comp_of]).to(torch.int32)
    out = torch.empty(N, dim, dtype=torch.float64, device=dev)
    if nc == 1:
        meta = np.zeros((1, dim))
        half = None
    else:
        meta = meta_positions(x, order, starts, counts, dim)
        dd = np.sqrt(((meta[:, None, :] - meta[None, :, :]) ** 2).sum(-1))
        dd[np.eye(nc, dtype=bool)] = np.inf
        half = dd.min(1) / 2.0
    for c in range(nc):
        verts = order[starts[c]:starts[c] + counts[c]].to(torch.int32).contiguous()
        n = int(counts[c])
        vecs, ok = None, False
        if n >= 2 * dim + 2:
            op = _Operator(graph, dis, verts, pos)
            vecs, ok = lobpcg_smallest(op, dim, seed, (_S_LOBPCG << 32) | c)
        scale = 10.0 if half is None else float(half[c])
        if not ok:
            msgs.append("component %d (%d vertices) %s; laid out at random" %
                        (c, n, "is too small for a spectral layout" if n < 2 * dim + 2
                         else "did not converge in the eigensolver"))
            block = random_block(seed, (_S_FILL << 32) | c, (n, dim), 0, scale, dev)
        elif half is None:
            block = vecs
        else:
            block = vecs * (scale / float(vecs.abs().max()))
        out[verts.long()] = block + torch.as_tensor(meta[c], device=dev)
    return out, msgs


def init_embedding(init64, seed, noise, dev):
    """The float32 embedding the SGD starts from: (float)(init * expansion) + noise, rescaled to
    [0, 10] per axis (umap.umap_.simplicial_set_embedding, umap-learn 0.5)."""
    N, dim = init64.shape
    emb = torch.empty(N, dim, dtype=torch.float32, device=dev)
    if noise:
        expansion = 10.0 / float(init64.abs().max())
        nz = random_block(seed, _S_NOISE << 32, (N, dim), 1, 1e-4, dev)
        _lib.call("ava_b200_umap_init_layout", init64.data_ptr(), nz.data_ptr(), expansion, N, dim, emb.data_ptr(),
                  _stream(dev))
    else:
        _lib.call("ava_b200_umap_init_layout", init64.data_ptr(), None, 1.0, N, dim, emb.data_ptr(), _stream(dev))
    return emb


# ------------------------------------------------------------------------------ stage 5
def sgd_epoch(emb, sched, epoch, a, b, gamma, alpha, seed, e0=0, e1=None):
    """One epoch of the layout over the edges [e0, e1) (default: all)."""
    N, dim = emb.shape
    if e1 is None:
        e1 = sched["head"].numel()
    _lib.call("ava_b200_umap_sgd_epoch", emb.data_ptr(), N, dim, sched["head"].data_ptr(), sched["tail"].data_ptr(),
              sched["eps"].data_ptr(), sched["eps_neg"].data_ptr(), sched["next"].data_ptr(),
              sched["next_neg"].data_ptr(), int(e0), int(e1), int(epoch), float(a), float(b), float(gamma),
              float(alpha), seed & (2 ** 64 - 1), _stream(emb.device))


class LatentUMAP:
    """``umap.UMAP`` restricted to ``metric='euclidean'``, on the device: ``fit``, ``fit_transform`` and
    ``transform``.

    The reference's projection (ava/data/data_container.py, _make_latent_mean_umap_projection) is
    ``LatentUMAP(n_components=2, n_neighbors=20, min_dist=0.1, random_state=42)``.  The defaults here
    are umap-learn's.  ``n_neighbors`` <= 100, ``n_components`` 1..8, at most 64 input dimensions.

    Attributes after a fit: ``embedding_`` (numpy float32 [N, n_components]), ``graph_`` (the fuzzy
    simplicial set as a scipy CSR on the host, built when first read), ``knn_indices_`` and
    ``knn_dists_`` (numpy), ``a_``, ``b_``, ``n_epochs_``.  Same seed, same data: the neighbours, graph
    and initialisation repeat bit for bit; the layout repeats up to the Hogwild races of its SGD.
    ``transform`` places new rows into the fitted embedding without moving it, and repeats bit for bit.
    A fitted model pickles with its state on the host and transforms on any device after unpickling."""

    def __init__(self, n_neighbors=15, n_components=2, min_dist=0.1, spread=1.0, metric='euclidean', n_epochs=None,
                 learning_rate=1.0, init='spectral', negative_sample_rate=5, repulsion_strength=1.0,
                 local_connectivity=1.0, random_state=None, device=None):
        self.n_neighbors = n_neighbors
        self.n_components = n_components
        self.min_dist = min_dist
        self.spread = spread
        self.metric = metric
        self.n_epochs = n_epochs
        self.learning_rate = learning_rate
        self.init = init
        self.negative_sample_rate = negative_sample_rate
        self.repulsion_strength = repulsion_strength
        self.local_connectivity = local_connectivity
        self.random_state = random_state
        self.device = device

    def _validate(self):
        if self.metric != 'euclidean':
            raise ValueError("LatentUMAP supports metric='euclidean' only, got %r" % (self.metric,))
        if not (isinstance(self.n_components, (int, np.integer)) and 1 <= self.n_components <= MAX_COMPONENTS):
            raise ValueError("n_components=%r must be an integer in 1..%d" % (self.n_components, MAX_COMPONENTS))
        if not (isinstance(self.n_neighbors, (int, np.integer)) and 2 <= self.n_neighbors <= MAX_NEIGHBORS):
            raise ValueError("n_neighbors=%r must be an integer in 2..%d" % (self.n_neighbors, MAX_NEIGHBORS))
        if self.n_epochs is not None and not (isinstance(self.n_epochs, (int, np.integer)) and self.n_epochs >= 1):
            raise ValueError("n_epochs=%r must be a positive integer or None" % (self.n_epochs,))
        if not (self.min_dist >= 0 and self.spread > 0 and self.min_dist <= self.spread):
            raise ValueError("need 0 <= min_dist <= spread and spread > 0")
        if not (self.negative_sample_rate > 0 and self.learning_rate >= 0 and self.repulsion_strength >= 0):
            raise ValueError("negative_sample_rate must be > 0, learning_rate and repulsion_strength >= 0")
        if not (0 <= self.local_connectivity):
            raise ValueError("local_connectivity must be >= 0")
        if isinstance(self.init, str) and self.init not in ('spectral', 'random'):
            raise ValueError("init=%r: expected 'spectral', 'random' or an [N, n_components] array" % (self.init,))

    def _device(self, x):
        if torch.is_tensor(x) and x.is_cuda:
            return x.device
        if self.device is not None:
            return torch.device(self.device)
        if not torch.cuda.is_available():
            raise _lib.AvaB200Error("LatentUMAP needs a CUDA device (there is no CPU fallback)")
        return torch.device("cuda", torch.cuda.current_device())

    def _seed(self):
        if self.random_state is None:
            return int(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64))
        if isinstance(self.random_state, np.random.RandomState):
            return int(self.random_state.randint(0, 2 ** 63 - 1, dtype=np.int64))
        return int(self.random_state)

    def _as_rows(self, x):
        if not torch.is_tensor(x):
            x = torch.from_numpy(np.ascontiguousarray(x))
        if x.dim() != 2:
            raise ValueError("expected a [N, D] array, got shape %s" % (tuple(x.shape),))
        if x.dtype not in (torch.float32, torch.float64):
            x = x.to(torch.float64)
        return x

    def fit(self, x):
        """x: [N, D] numpy array or tensor, float32 or float64, D <= 64.  Fits the embedding and keeps
        what ``transform`` needs on the device: the fitted rows (a contiguous device tensor is kept, not
        copied), the float32 embedding, the neighbour count, ``a_``, ``b_`` and the seed.  Returns self."""
        self._validate()
        x = self._as_rows(x)
        N, D = x.shape
        if D > MAX_D or D < 1:
            raise ValueError("LatentUMAP takes 1 to %d input dimensions, got %d" % (MAX_D, D))
        if N < 1:
            raise ValueError("need at least one row")
        dim = int(self.n_components)
        init_arr = None
        if not isinstance(self.init, str):
            init_arr = np.asarray(self.init, dtype=np.float64)
            if init_arr.shape != (N, dim) or not np.isfinite(init_arr).all():
                raise ValueError("init array must be finite with shape (%d, %d)" % (N, dim))
        if not bool(torch.isfinite(x).all()):
            raise ValueError("x contains NaN or inf")
        dev = self._device(x)
        x = x.to(dev).contiguous()
        self.a_, self.b_ = find_ab_params(self.spread, self.min_dist)
        self.n_epochs_ = int(self.n_epochs) if self.n_epochs is not None else default_n_epochs(N)
        self._graph = None
        with torch.cuda.device(dev):
            if N == 1:
                self.knn_indices_ = np.zeros((1, 1), dtype=np.int32)
                self.knn_dists_ = np.zeros((1, 1))
                self._graph_dev = None
                emb = torch.zeros(1, dim, dtype=torch.float32, device=dev)
                self._keep_fit(x, emb, 1, 0)
                return self
            k = int(self.n_neighbors)
            if N <= k:
                warnings.warn("n_neighbors=%d is not smaller than the number of rows %d; using %d neighbours"
                              % (k, N, max(N - 1, 2)))
                k = max(N - 1, 2)
            seed = self._seed()
            idx, dist = knn(x, k)
            graph = fuzzy_graph(idx, dist, self.local_connectivity)
            sched = edge_schedule(graph, self.n_epochs_, self.negative_sample_rate)
            if init_arr is not None:
                emb = init_embedding(torch.from_numpy(init_arr).to(dev), seed, False, dev)
            elif self.init == 'random':
                emb = init_embedding(random_block(seed, _S_RANDOM_INIT << 32, (N, dim), 0, 10.0, dev), seed, False, dev)
            else:
                init64, msgs = spectral_layout(x, graph, dim, seed)
                for m in msgs:
                    warnings.warn(m)
                emb = init_embedding(init64, seed, True, dev)
            for n in range(self.n_epochs_):
                alpha = self.learning_rate * (1.0 - n / float(self.n_epochs_))
                sgd_epoch(emb, sched, n, self.a_, self.b_, self.repulsion_strength, alpha, seed)
            self._graph_dev = graph
            self.knn_indices_ = idx.cpu().numpy()
            self.knn_dists_ = dist.cpu().numpy()
            self._keep_fit(x, emb, k, seed)
        return self

    def _keep_fit(self, x, emb, k, seed):
        self._fit_x, self._fit_emb, self._k, self._seed_ = x, emb, k, seed
        self.embedding_ = emb.cpu().numpy()

    def fit_transform_device(self, x):
        """``fit(x)``, then the float32 [N, n_components] embedding as a tensor on the device."""
        return self.fit(x)._fit_emb

    def fit_transform(self, x):
        """[N, D] -> numpy float32 [N, n_components] (what ``umap.UMAP.fit_transform`` returns)."""
        self.fit(x)
        return self.embedding_

    def transform_device(self, x):
        """Place new rows x [Nq, D] into the fitted embedding without moving it (umap-learn's
        ``transform``): a float32 [Nq, n_components] tensor on the device.  The queries are converted to
        the fitted rows' dtype.  A query set bitwise equal to the fitted rows returns a copy of the
        embedding.  The layout's random draws come from the fit's seed, so repeated transforms of the
        same rows are bitwise equal."""
        if getattr(self, "_fit_x", None) is None:
            raise RuntimeError("LatentUMAP.transform needs a fitted model: call fit first")
        x = self._as_rows(x)
        N, D = self._fit_x.shape
        if x.shape[1] != D:
            raise ValueError("the model was fitted on %d columns, got %d" % (D, x.shape[1]))
        same_dtype = x.dtype == self._fit_x.dtype
        x = x.to(self._fit_x.dtype)
        if not bool(torch.isfinite(x).all()):
            raise ValueError("x contains NaN or inf")
        dev = self._device(x)
        dim = int(self.n_components)
        if x.shape[0] == 0:
            return torch.empty(0, dim, dtype=torch.float32, device=dev)
        # the fitted state follows the device of the latest call (it is on the host after unpickling)
        self._fit_x = self._fit_x.to(dev)
        self._fit_emb = self._fit_emb.to(dev)
        x = x.to(dev).contiguous()
        xf, emb = self._fit_x, self._fit_emb
        with torch.cuda.device(dev):
            if N == 1:
                return emb[:1].repeat(x.shape[0], 1)
            bits = torch.int32 if xf.dtype == torch.float32 else torch.int64
            if same_dtype and x.shape == xf.shape and torch.equal(x.view(bits), xf.view(bits)):
                return emb.clone()
            idx, dist = knn_query(x, xf, self._k)
            graph = query_graph(idx, dist, self.local_connectivity)
            out = init_transform(graph, emb)
            n_epochs = transform_n_epochs(self.n_epochs, x.shape[0])
            if n_epochs > 0:
                sched = transform_schedule(graph, n_epochs, self.negative_sample_rate)
                sgd_transform(out, emb, sched, n_epochs, self.a_, self.b_, self.repulsion_strength,
                              self.learning_rate / 4.0, self._seed_)
        return out

    def transform(self, x):
        """[Nq, D] -> numpy float32 [Nq, n_components] (what ``umap.UMAP.transform`` returns)."""
        return self.transform_device(x).cpu().numpy()

    def __getstate__(self):
        """A fitted model pickles with its state on the host; ``transform`` moves it to the device it runs on."""
        st = self.__dict__.copy()
        if st.get("_graph_dev") is not None:
            st["_graph"] = self.graph_
        st["_graph_dev"] = None
        for name in ("_fit_x", "_fit_emb"):
            if torch.is_tensor(st.get(name)):
                st[name] = st[name].cpu()
        return st

    @property
    def graph_(self):
        """The fuzzy simplicial set P (unpruned) as a scipy.sparse CSR matrix on the host."""
        if getattr(self, "_graph", None) is None:
            import scipy.sparse
            g = getattr(self, "_graph_dev", None)
            if g is None:
                n = getattr(self, "embedding_", np.zeros((0, 0))).shape[0]
                self._graph = scipy.sparse.csr_matrix((n, n))
            else:
                self._graph = scipy.sparse.csr_matrix(
                    (g["vals"].cpu().numpy(), g["cols"].cpu().numpy(), g["rowptr"].cpu().numpy()),
                    shape=(g["n"], g["n"]))
        return self._graph
