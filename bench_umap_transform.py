"""LatentUMAP.transform stage times on the device, with CUDA events: the query kNN, the bipartite graph,
the initialisation, the layout SGD and the total, on held-out rows of the Gaussian blobs of bench_umap.py
(D = 32, n_neighbors=20, min_dist=0.1, random_state=42).

For each fitted size N it fits once, times the fit's own kNN stage at that N in the same run (the rate the
query kNN is compared with), then transforms Nq held-out rows.  Prints one JSON line per (N, Nq) and appends
it to --out: query kNN pairs/s and their share of the card's FP32 FMA peak (2 D pipe operations per pair
against 148 SMs x 128 lanes x the maximum SM clock, read from nvidia-smi in the same run, as bench_umap.py
counts them), the fit kNN's pairs/s, and SGD edge-epochs/s.

    python bench_umap_transform.py [--fit 100000,1000000] [--queries 10000,100000,1000000] [--out FILE]
"""
import argparse
import importlib
import json
import os
import sys
import warnings

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
lu = importlib.import_module("autoencoded-vocal-analysis_b200.data.latent_umap")
bu = importlib.import_module("bench_umap")

D, K = 32, 20


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return out, a.elapsed_time(b) / 1e3


def run(n, nqs, name, watts, clk_mhz):
    x, _ = bu.blobs(n + max(nqs), D)                              # held-out rows come from the same blobs
    xf, xq_all = x[:n].contiguous(), x[n:]
    um = lu.LatentUMAP(n_neighbors=K, min_dist=0.1, random_state=42)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        um.fit(xf)
    _, t_fit_knn = timed(lambda: lu.knn(xf, K))
    fit_pairs_per_s = float(n) * n / t_fit_knn
    peak_fma = 148 * 128 * clk_mhz * 1e6
    emb = um._fit_emb
    lines = []
    for nq in nqs:
        q = xq_all[:nq].contiguous()
        n_epochs = lu.transform_n_epochs(None, nq)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        torch.cuda.synchronize()
        ev[0].record()
        idx, dist = lu.knn_query(q, xf, um._k)
        ev[1].record()
        g = lu.query_graph(idx, dist, um.local_connectivity)
        sched = lu.transform_schedule(g, n_epochs, um.negative_sample_rate)
        ev[2].record()
        out = lu.init_transform(g, emb)
        ev[3].record()
        lu.sgd_transform(out, emb, sched, n_epochs, um.a_, um.b_, 1.0, 0.25, um._seed_)
        ev[4].record()
        torch.cuda.synchronize()
        t = [ev[i].elapsed_time(ev[i + 1]) / 1e3 for i in range(4)]
        pairs = float(nq) * n
        n_edges = sched["tail"].numel()
        lines.append({"what": "LatentUMAP.transform stages, %d held-out rows into a fit of %d x %d float64 blobs, "
                              "n_neighbors=20, min_dist=0.1" % (nq, n, D),
                      "gpu": name, "power_limit_W": watts, "max_sm_clock_MHz": clk_mhz, "N": n, "Nq": nq, "D": D,
                      "knn_s": t[0], "graph_s": t[1], "init_s": t[2], "sgd_s": t[3], "total_s": sum(t),
                      "knn_pairs_per_s": pairs / t[0], "knn_fp32_fma_pipe_share": pairs * 2 * D / t[0] / peak_fma,
                      "fit_knn_s": t_fit_knn, "fit_knn_pairs_per_s": fit_pairs_per_s,
                      "knn_rate_vs_fit": pairs / t[0] / fit_pairs_per_s,
                      "n_epochs": n_epochs, "edges": n_edges, "sgd_edge_epochs_per_s": n_edges * n_epochs / t[3],
                      "finite": bool(torch.isfinite(out).all())})
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fit", default="100000,1000000")
    ap.add_argument("--queries", default="10000,100000,1000000")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_umap_transform.py needs a CUDA device")
    name, watts, clk = bu.card()
    nqs = [int(s) for s in args.queries.split(",")]
    run(3000, [1000], name, watts, clk)                           # warm-up: module load, allocator
    for n in [int(s) for s in args.fit.split(",")]:
        for out in run(n, nqs, name, watts, clk):
            line = json.dumps(out)
            print(line, flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(line + "\n")


if __name__ == "__main__":
    main()
